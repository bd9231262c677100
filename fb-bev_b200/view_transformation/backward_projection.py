"""Backward projection (BEV -> image depth-aware spatial cross-attention)
plugin classes.

Mirror of ``mmdet3d/models/fbbev/view_transformation/backward_projection/``:

==============================  =============================================
class here                      reference
==============================  =============================================
BackwardProjection              backward_projection.py:34-133        (HEADS)
BEVFormer                       bevformer_utils/bevformer.py:23-132  (TRANSFORMER)
bevformer_encoder               bevformer_utils/bevformer_encoder.py:27-203
BEVFormerEncoderLayer           bevformer_utils/bevformer_encoder.py:206-377
MyCustomBaseTransformerLayer    bevformer_utils/custom_base_transformer_layer.py:35-262
DA_SpatialCrossAttention        bevformer_utils/spatial_cross_attention_depth.py:31-223
DA_MSDeformableAttention        bevformer_utils/spatial_cross_attention_depth.py:361-601
CustormLearnedPositionalEncoding  bevformer_utils/positional_encoding.py:11-68
MultiScaleDeformableAttention   mmcv.ops (un-vendored; config :176-180)
FFN                             mmcv.cnn.bricks.transformer.FFN (config :194-201)
==============================  =============================================

Registry names, constructor keywords, ``forward`` signatures and state-dict
keys match, so a FB-OCC checkpoint loads and the detector's call
(``fbocc.py:357-363``) is unchanged.

What runs where: with gradients off (inference), every nn.Linear runs on the
tcgen05 tensor cores through ``fbbev_linear_fwd`` (3xTF32, fp32 in / out) with
the bias, ReLU, residual add and the following LayerNorm in its epilogue; with
gradients on they stay on cuBLAS through PyTorch (``FBBEV_TORCH_LINEAR=1`` forces
that path).  Everything between them -- softmax, sampling-location arithmetic,
the depth look-up, bilinear sampling, the per-camera accumulation and averaging
-- is one hand-written kernel per attention (``fbbev_msda_fused_fwd`` for the
self-attention, ``fbbev_da_sca_fwd`` for the depth-aware cross-attention).  The
reference's per-camera ``nonzero()`` loops, zero-padded re-batching, int64
one-hot tensor and scatter loops (spatial_cross_attention_depth.py:156-216) have
no counterpart here: the kernel iterates cameras per BEV query.
"""
import copy
import math
import os
import warnings

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..ops import linear as _linear_ops
from .forward_projection import inv3x3_many
from ..ops import ms_deform_attn as _msda_ops
from ..ops.ms_deform_attn import (MultiScaleDeformableAttnFunction_fp32,
                                  bev_mask_fold,
                                  da_spatial_cross_attention_core,
                                  da_spatial_cross_attention_core_autograd,
                                  ms_deform_attn_fused, ms_deform_attn_unfused,
                                  needs_grad)
from ..registry import (BaseModule, build_attention,
                        build_feedforward_network, build_positional_encoding,
                        build_transformer, build_transformer_layer,
                        build_transformer_layer_sequence, register)

__all__ = ['BackwardProjection', 'BEVFormer', 'bevformer_encoder',
           'BEVFormerEncoderLayer', 'MyCustomBaseTransformerLayer',
           'DA_SpatialCrossAttention', 'DA_MSDeformableAttention',
           'CustormLearnedPositionalEncoding', 'MultiScaleDeformableAttention',
           'FFN']


_CONST_CACHE = {}
_SIDE_STREAMS = {}  # one side stream per device (module-level: not deep-copied)


def _const_tensor(values, device):
    """Small int64 tensors (spatial shapes, level starts) are constants of the
    configuration: build them once per device instead of a host->device copy
    every forward (the reference re-creates them each call,
    bevformer_encoder.py:337-339, bevformer.py:108-111)."""
    key = (values, str(device))
    t = _CONST_CACHE.get(key)
    if t is None:
        t = torch.tensor(values, dtype=torch.long, device=device)
        _CONST_CACHE[key] = t
    return t


def _fused_linear_on(x, *dropouts):
    """The tensor-core Linear path: CUDA fp32 input, no active dropout.  With
    autograd recording the forward stays on the tcgen05 kernel
    (``ops.linear.LinearTF32Function``; backward = library GEMMs) unless
    ``FBBEV_TRAIN_TORCH_LINEAR=1`` asks for nn.Linear end to end."""
    if os.environ.get('FBBEV_TORCH_LINEAR', '0') == '1':
        return False
    if torch.is_grad_enabled() and \
            os.environ.get('FBBEV_TRAIN_TORCH_LINEAR', '0') == '1':
        return False
    if not x.is_cuda or x.dtype != torch.float32:
        return False
    for d in dropouts:
        if isinstance(d, nn.Dropout) and d.training and d.p > 0:
            return False
    return True


def _linear(mod, x, relu=False, residual=None, norm=None):
    """``norm(act(mod(x)) + residual)`` in one kernel launch per <= 160 output
    columns (``mod`` an nn.Linear, ``norm`` an nn.LayerNorm or None)."""
    n, k = mod.weight.shape
    if k % 4 or n % 4:
        y = mod(x)
        y = F.relu(y) if relu else y
        y = y + residual if residual is not None else y
        return norm(y) if norm is not None else y
    if torch.is_grad_enabled():
        # training: forward on the same kernel, differentiable; LayerNorm as a
        # torch op (its backward needs the row statistics)
        y = _linear_ops.linear_train(x, mod.weight, mod.bias, relu=relu,
                                     residual=residual)
        return norm(y) if norm is not None else y
    if norm is not None and not _linear_ops.ln_supported(n):
        # rows wider than the LayerNorm epilogue keeps in shared memory
        # (n > 80, e.g. embed_dims 256): GEMM + bias + ReLU + residual stay in
        # the tcgen05 kernel, the normalisation is a separate pass
        y = _linear_ops.linear_fused(x, mod.weight, mod.bias, relu=relu,
                                     residual=residual)
        return norm(y)
    return _linear_ops.linear_fused(
        x, mod.weight, mod.bias, relu=relu, residual=residual,
        ln_weight=None if norm is None else norm.weight,
        ln_bias=None if norm is None else norm.bias,
        eps=1e-5 if norm is None else norm.eps)


def _linear_pair(owner, mod_a, mod_b, x, x_add=None):
    """``(mod_a(x + x_add), mod_b(x + x_add))`` for two nn.Linears on the same
    input, one launch when their widths allow (the addition happens in the
    kernel's loader)."""
    if mod_a.weight.shape[1] % 4 == 0 and not torch.is_grad_enabled():
        return _linear_ops.linear_pair(
            x, mod_a.weight, mod_a.bias, mod_b.weight, mod_b.bias,
            owner.__dict__.setdefault('_pair_cache', {}), x_add=x_add)
    if x_add is not None:
        x = x + x_add
    return _linear(mod_a, x), _linear(mod_b, x)


def _xavier_uniform(module, bias=0.):
    if getattr(module, 'weight', None) is not None:
        nn.init.xavier_uniform_(module.weight)
    if getattr(module, 'bias', None) is not None:
        nn.init.constant_(module.bias, bias)


def _constant(module, val, bias=0.):
    if getattr(module, 'weight', None) is not None:
        nn.init.constant_(module.weight, val)
    if getattr(module, 'bias', None) is not None:
        nn.init.constant_(module.bias, bias)


def _ring_offsets(num_heads):
    """Unit offsets on a square ring, one direction per head (the Deformable
    DETR initialisation both attention modules share)."""
    thetas = torch.arange(num_heads, dtype=torch.float32) * (
        2.0 * math.pi / num_heads)
    ring = torch.stack([thetas.cos(), thetas.sin()], -1)
    return ring / ring.abs().max(-1, keepdim=True)[0]


# ---------------------------------------------------------------------------
# positional_encoding.py:11-68
# ---------------------------------------------------------------------------
@register('POSITIONAL_ENCODING')
class CustormLearnedPositionalEncoding(BaseModule):
    """Learned row/column embeddings; ``forward(bs, h, w, device)`` returns
    ``(bs, 2*num_feats, h, w)``."""

    def __init__(self, num_feats, row_num_embed=50, col_num_embed=50,
                 init_cfg=dict(type='Uniform', layer='Embedding')):
        super().__init__(init_cfg)
        self.row_embed = nn.Embedding(row_num_embed, num_feats)
        self.col_embed = nn.Embedding(col_num_embed, num_feats)
        self.num_feats = num_feats
        self.row_num_embed = row_num_embed
        self.col_num_embed = col_num_embed
        # mmcv's `Uniform` initialiser on Embedding layers: U(0, 1)
        nn.init.uniform_(self.row_embed.weight)
        nn.init.uniform_(self.col_embed.weight)

    def forward(self, bs, h, w, device):
        # with gradients off the encoding is a constant of the two embedding
        # tables: build it once per (shape, table version) instead of ~8
        # gather / repeat / cat kernels every forward
        key = None
        if not torch.is_grad_enabled():
            key = (bs, h, w, str(device), self.col_embed.weight._version,
                   self.row_embed.weight._version,
                   self.col_embed.weight.data_ptr(),
                   self.row_embed.weight.data_ptr())
            hit = self.__dict__.get('_pos_cache')
            if hit is not None and hit[0] == key:
                return hit[1]
        x_embed = self.col_embed(torch.arange(w, device=device))
        y_embed = self.row_embed(torch.arange(h, device=device))
        pos = torch.cat((x_embed.unsqueeze(0).repeat(h, 1, 1),
                         y_embed.unsqueeze(1).repeat(1, w, 1)), dim=-1)
        pos = pos.permute(2, 0, 1).unsqueeze(0).repeat(bs, 1, 1, 1)
        if key is not None:
            self.__dict__['_pos_cache'] = (key, pos)
        return pos

    def __repr__(self):
        return (f'{self.__class__.__name__}(num_feats={self.num_feats}, '
                f'row_num_embed={self.row_num_embed}, '
                f'col_num_embed={self.col_num_embed})')


# ---------------------------------------------------------------------------
# mmcv.cnn.bricks.transformer.FFN  (state-dict keys layers.0.0.*, layers.1.*)
# ---------------------------------------------------------------------------
@register('FEEDFORWARD_NETWORK', upstream=False)
class FFN(BaseModule):

    def __init__(self, embed_dims=256, feedforward_channels=1024, num_fcs=2,
                 act_cfg=dict(type='ReLU', inplace=True), ffn_drop=0.,
                 dropout_layer=None, add_identity=True, init_cfg=None,
                 **kwargs):
        super().__init__(init_cfg)
        assert num_fcs >= 2
        act = (act_cfg or {}).get('type', 'ReLU')
        acts = {'ReLU': lambda: nn.ReLU(inplace=True), 'GELU': nn.GELU}
        if act not in acts:
            raise NotImplementedError(f'FFN activation {act}')
        self.embed_dims = embed_dims
        self.feedforward_channels = feedforward_channels
        self.num_fcs = num_fcs
        layers, in_ch = [], embed_dims
        for _ in range(num_fcs - 1):
            layers.append(nn.Sequential(nn.Linear(in_ch, feedforward_channels),
                                        acts[act](), nn.Dropout(ffn_drop)))
            in_ch = feedforward_channels
        layers.append(nn.Linear(feedforward_channels, embed_dims))
        layers.append(nn.Dropout(ffn_drop))
        self.layers = nn.Sequential(*layers)
        p = (dropout_layer or {}).get('drop_prob', 0.) if dropout_layer else 0.
        self.dropout_layer = nn.Dropout(p) if p > 0 else nn.Identity()
        self.add_identity = add_identity

    def forward(self, x, identity=None, post_norm=None):
        drops = [m for m in self.layers.modules() if isinstance(m, nn.Dropout)]
        if (_fused_linear_on(x, self.dropout_layer, *drops) and
                all(isinstance(l[1], nn.ReLU) for l in self.layers[:-2])):
            res = (identity if identity is not None else x) \
                if self.add_identity else None
            fc1, fc2 = self.layers[0][0], self.layers[-2]
            if (self.num_fcs == 2 and
                    _linear_ops.ffn_supported(x, fc1.weight, fc2.weight) and
                    (post_norm is None or
                     _linear_ops.ln_supported(fc2.weight.shape[0]))):
                # both Linears, the ReLU, the identity add and the LayerNorm
                # as one kernel: the hidden activation stays in tensor memory
                return _linear_ops.ffn_fused(
                    x, fc1.weight, fc1.bias, fc2.weight, fc2.bias,
                    residual=res,
                    ln_weight=None if post_norm is None else post_norm.weight,
                    ln_bias=None if post_norm is None else post_norm.bias,
                    eps=1e-5 if post_norm is None else post_norm.eps)
            out = x
            for l in self.layers[:-2]:
                out = _linear(l[0], out, relu=True)
            res = (identity if identity is not None else x) \
                if self.add_identity else None
            return _linear(self.layers[-2], out, residual=res, norm=post_norm)
        out = self.layers(x)
        if self.add_identity:
            out = (x if identity is None else identity) + self.dropout_layer(out)
        else:
            out = self.dropout_layer(out)
        return out if post_norm is None else post_norm(out)


# ---------------------------------------------------------------------------
# mmcv.ops.MultiScaleDeformableAttention (encoder self-attention)
# ---------------------------------------------------------------------------
@register('ATTENTION', upstream=False)
class MultiScaleDeformableAttention(BaseModule):
    """Deformable self-attention over the BEV map.  Same parameters and
    ``forward`` contract as mmcv's module; sampling runs in the fused kernel
    ``fbbev_msda_fused_fwd`` (no ``sampling_locations`` / softmax tensors)."""

    def __init__(self, embed_dims=256, num_heads=8, num_levels=4,
                 num_points=4, im2col_step=64, dropout=0.1, batch_first=False,
                 norm_cfg=None, init_cfg=None):
        super().__init__(init_cfg)
        if embed_dims % num_heads != 0:
            raise ValueError('embed_dims must be divisible by num_heads, '
                             f'but got {embed_dims} and {num_heads}')
        self.norm_cfg = norm_cfg
        self.dropout = nn.Dropout(dropout)
        self.batch_first = batch_first
        self.im2col_step = im2col_step
        self.embed_dims = embed_dims
        self.num_levels = num_levels
        self.num_heads = num_heads
        self.num_points = num_points
        self.sampling_offsets = nn.Linear(
            embed_dims, num_heads * num_levels * num_points * 2)
        self.attention_weights = nn.Linear(
            embed_dims, num_heads * num_levels * num_points)
        self.value_proj = nn.Linear(embed_dims, embed_dims)
        self.output_proj = nn.Linear(embed_dims, embed_dims)
        self.init_weights()

    def init_weights(self):
        _constant(self.sampling_offsets, 0.)
        grid = _ring_offsets(self.num_heads).view(
            self.num_heads, 1, 1, 2).repeat(1, self.num_levels,
                                            self.num_points, 1)
        for i in range(self.num_points):
            grid[:, :, i, :] *= i + 1
        self.sampling_offsets.bias.data = grid.view(-1)
        _constant(self.attention_weights, 0., 0.)
        _xavier_uniform(self.value_proj)
        _xavier_uniform(self.output_proj)
        self._is_init = True

    def forward(self, query, key=None, value=None, identity=None,
                query_pos=None, key_padding_mask=None, reference_points=None,
                spatial_shapes=None, level_start_index=None, post_norm=None,
                **kwargs):
        if value is None:
            value = query
        if identity is None:
            identity = query
        fused = _fused_linear_on(query, self.dropout)
        if query_pos is not None and not fused:
            query = query + query_pos
        if not self.batch_first:
            query = query.permute(1, 0, 2)
            value = value.permute(1, 0, 2)
            if query_pos is not None and fused:
                query_pos = query_pos.permute(1, 0, 2)
        bs, num_query, _ = query.shape
        _, num_value, _ = value.shape
        lin = _linear if fused else (lambda m, x: m(x))
        value = lin(self.value_proj, value)
        if key_padding_mask is not None:
            value = value.masked_fill(key_padding_mask[..., None], 0.0)
        value = value.view(bs, num_value, self.num_heads, -1)
        if fused:
            # query + query_pos is formed in the Linear's loader
            offsets, logits = _linear_pair(self, self.sampling_offsets,
                                           self.attention_weights, query,
                                           x_add=query_pos)
        else:
            offsets = self.sampling_offsets(query)
            logits = self.attention_weights(query)
        offsets = offsets.view(
            bs, num_query, self.num_heads, self.num_levels, self.num_points, 2)
        logits = logits.view(
            bs, num_query, self.num_heads, self.num_levels, self.num_points)
        if reference_points.shape[-1] != 2:
            raise ValueError('Last dim of reference_points must be 2, but get '
                             f'{reference_points.shape[-1]} instead.')
        # the fused sampling kernel is forward-only: with autograd recording,
        # take the differentiable route (mmcv's own op sequence)
        core = ms_deform_attn_unfused if needs_grad(value, offsets, logits) \
            else ms_deform_attn_fused
        output = core(value, spatial_shapes, level_start_index,
                      reference_points, offsets, logits,
                      map_width=kwargs.get('bev_w') or 0)
        if fused:
            res = identity if self.batch_first else identity.permute(1, 0, 2)
            output = _linear(self.output_proj, output, residual=res,
                             norm=post_norm)
            return output if self.batch_first else output.permute(1, 0, 2)
        output = self.output_proj(output)
        if not self.batch_first:
            output = output.permute(1, 0, 2)
        output = self.dropout(output) + identity
        return output if post_norm is None else post_norm(output)


# ---------------------------------------------------------------------------
# spatial_cross_attention_depth.py:361-601
# ---------------------------------------------------------------------------
@register('ATTENTION')
class DA_MSDeformableAttention(BaseModule):
    """Depth-aware deformable attention (one camera batch per row).

    ``forward`` keeps the reference's contract at this class boundary
    (re-batched queries, one-hot ``bev_query_depth``); the enclosing
    ``DA_SpatialCrossAttention`` normally bypasses it and feeds this module's
    three Linears straight into the fused kernel."""

    def __init__(self, embed_dims=256, num_heads=8, num_levels=4,
                 num_points=8, num_Z_anchors=4, im2col_step=64, dropout=0.1,
                 batch_first=True, disable_deformable=False, norm_cfg=None,
                 init_cfg=None):
        super().__init__(init_cfg)
        if embed_dims % num_heads != 0:
            raise ValueError('embed_dims must be divisible by num_heads, '
                             f'but got {embed_dims} and {num_heads}')
        self.norm_cfg = norm_cfg
        self.batch_first = batch_first
        self.output_proj = None
        self.fp16_enabled = False
        self.disable_deformable = disable_deformable
        self.num_Z_anchors = num_Z_anchors
        self.im2col_step = im2col_step
        self.embed_dims = embed_dims
        self.num_levels = num_levels
        self.num_heads = num_heads
        self.num_points = num_points
        self.sampling_offsets = nn.Linear(
            embed_dims, num_heads * num_levels * num_points * 2)
        self.attention_weights = nn.Linear(
            embed_dims, num_heads * num_levels * num_points)
        self.value_proj = nn.Linear(embed_dims, embed_dims)
        self.init_weights()

    def init_weights(self):
        """Offsets bias: ring direction per head, radius (p+1) for the p-th
        point of every Z anchor (:440-462)."""
        _constant(self.sampling_offsets, 0.)
        self.each_anchor_points = self.num_points // self.num_Z_anchors
        grid = _ring_offsets(self.num_heads).view(
            self.num_heads, 1, 1, 1, 2).repeat(
                1, self.num_levels, self.each_anchor_points,
                self.num_Z_anchors, 1)
        for i in range(self.each_anchor_points):
            grid[:, :, i, :, :] *= i + 1
        self.sampling_offsets.bias.data = grid.view(-1)
        _constant(self.attention_weights, 0., 0.)
        _xavier_uniform(self.value_proj)
        self._is_init = True

    # the three input projections, shared by both execution paths
    def project_value(self, value, key_padding_mask=None):
        bs, num_value, _ = value.shape
        lin = _linear if _fused_linear_on(value) else (lambda m, x: m(x))
        value = lin(self.value_proj, value)
        if key_padding_mask is not None:
            value = value.masked_fill(key_padding_mask[..., None], 0.0)
        return value.view(bs, num_value, self.num_heads, -1)

    def project_query(self, query, query_pos=None):
        bs, num_query, _ = query.shape
        if _fused_linear_on(query):
            offsets, logits = _linear_pair(self, self.sampling_offsets,
                                           self.attention_weights, query,
                                           x_add=query_pos)
        else:
            if query_pos is not None:
                query = query + query_pos
            offsets = self.sampling_offsets(query)
            logits = self.attention_weights(query)
        offsets = offsets.view(
            bs, num_query, self.num_heads, self.num_levels, self.num_points, 2)
        logits = logits.view(
            bs, num_query, self.num_heads, self.num_levels, self.num_points)
        if self.disable_deformable:
            offsets = offsets * 0
            logits = logits * 0
        return offsets, logits

    def forward(self, query, key=None, value=None, identity=None,
                query_pos=None, key_padding_mask=None, reference_points=None,
                spatial_shapes=None, level_start_index=None,
                bev_query_depth=None, pred_img_depth=None, **kwargs):
        """query (bs, nq, E); value (bs, n_value, E); reference_points
        (bs, nq, Z, 2); bev_query_depth (bs, nq, Z, DC) one-hot;
        pred_img_depth (bs, H0*W0, DC).  Returns (bs, nq, E)."""
        if value is None:
            value = query
        if query_pos is not None:
            query = query + query_pos
        if not self.batch_first:
            query = query.permute(1, 0, 2)
            value = value.permute(1, 0, 2)
        bs, num_query, _ = query.shape
        value = self.project_value(value, key_padding_mask)
        offsets, logits = self.project_query(query)
        weights = logits.flatten(3).softmax(-1).view_as(logits)
        if reference_points.shape[-1] != 2:
            raise ValueError('Last dim of reference_points must be 2, but get '
                             f'{reference_points.shape[-1]} instead.')
        Z = reference_points.shape[2]
        P = self.num_points
        assert P % Z == 0
        wh = torch.stack([spatial_shapes[..., 1], spatial_shapes[..., 0]], -1)
        offsets = offsets / wh[None, None, None, :, None, :]
        # point index = p*Z + z  (:563-570)
        loc = reference_points[:, :, None, None, None, :, :] + offsets.view(
            bs, num_query, self.num_heads, self.num_levels, P // Z, Z, 2)
        loc = loc.view(bs, num_query, self.num_heads, self.num_levels, P, 2)
        apply = MultiScaleDeformableAttnFunction_fp32.apply
        # depth look-up (:584-591)
        depth_ref = reference_points.reshape(bs, num_query * Z, 1, 1, 1, 2)
        depth_w = apply(pred_img_depth.unsqueeze(2).contiguous(),
                        spatial_shapes[0:1], level_start_index[0:1],
                        depth_ref.contiguous(),
                        torch.ones_like(depth_ref[..., 0]), self.im2col_step)
        depth_w = (depth_w.reshape(bs, num_query, Z, -1) *
                   bev_query_depth).sum(-1)
        depth_w = depth_w.unsqueeze(2).repeat(1, 1, P // Z, 1).reshape(
            bs, num_query, P)
        weights = weights * depth_w[:, :, None, None, :]  # :592
        output = apply(value, spatial_shapes, level_start_index, loc, weights,
                       self.im2col_step)
        if not self.batch_first:
            output = output.permute(1, 0, 2)
        return output


# ---------------------------------------------------------------------------
# spatial_cross_attention_depth.py:31-223
# ---------------------------------------------------------------------------
@register('ATTENTION')
class DA_SpatialCrossAttention(BaseModule):
    """Depth-aware spatial cross-attention of the BEV queries over the camera
    feature maps.

    ``rebatch_bev_mask`` (class attribute, default False): with a ``bev_mask``
    run the reference-shaped per-camera re-batching loops (``nonzero()`` host
    synchronisations) instead of folding the mask on the device and running
    the fused kernel -- kept as the literal restatement the fused route is
    tested against."""

    rebatch_bev_mask = False

    def __init__(self, embed_dims=256, num_cams=6, pc_range=None, dropout=0.1,
                 init_cfg=None, batch_first=False,
                 deformable_attention=dict(type='MSDeformableAttention3D',
                                           embed_dims=256, num_levels=4),
                 layer_scale=None, dbound=None, **kwargs):
        super().__init__(init_cfg)
        self.init_cfg = init_cfg
        self.dropout = nn.Dropout(dropout)
        self.pc_range = pc_range
        self.fp16_enabled = False
        self.deformable_attention = build_attention(deformable_attention)
        self.embed_dims = embed_dims
        self.num_cams = num_cams
        self.dbound = dbound
        self.output_proj = nn.Linear(embed_dims, embed_dims)
        self.batch_first = batch_first
        if layer_scale is not None:
            self.layer_scale = nn.Parameter(
                layer_scale * torch.ones(embed_dims), requires_grad=True)
        else:
            self.layer_scale = None
        self.init_weight()
        self.count = 0

    def init_weight(self):
        _xavier_uniform(self.output_proj)

    def _finish(self, slots, inp_residual, post_norm=None):
        if self.layer_scale is None and _fused_linear_on(slots, self.dropout):
            return _linear(self.output_proj, slots, residual=inp_residual,
                           norm=post_norm)
        slots = self.output_proj(slots)
        if self.layer_scale is None:
            out = self.dropout(slots) + inp_residual
        else:
            out = self.dropout(self.layer_scale * slots) + inp_residual
        return out if post_norm is None else post_norm(out)

    def forward(self, query, key, value, residual=None, query_pos=None,
                key_padding_mask=None, reference_points=None,
                spatial_shapes=None, reference_points_cam=None,
                level_start_index=None, flag='encoder', bev_query_depth=None,
                pred_img_depth=None, bev_mask=None, per_cam_mask_list=None,
                post_norm=None, **kwargs):
        """query (bs, nq, E); key/value (num_cams, n_value, bs, E);
        reference_points_cam (num_cams, bs, nq, Z, 2); bev_query_depth
        (num_cams, bs, nq, Z, 1); pred_img_depth (bs, num_cams, DC, H, W);
        per_cam_mask_list (num_cams, bs, nq, Z) bool.  Returns (bs, nq, E)."""
        query = query.float()
        if key is None:
            key = query
        if value is None:
            value = key
        inp_residual = query if residual is None else residual
        # work the encoder started on its side stream (camera geometry, this
        # module's value projection) must have finished before it is consumed
        side_event = kwargs.get('side_event')
        if side_event is not None and query.is_cuda:
            torch.cuda.current_stream(query.device).wait_event(side_event)
        sca_prepared = (kwargs.get('sca_prepared') or {}).get(id(self))
        if bev_mask is not None:
            if self.rebatch_bev_mask or not query.is_cuda:
                if query_pos is not None:
                    query = query + query_pos.float()
                return self._forward_rebatch(
                    query, value, inp_residual, key_padding_mask,
                    spatial_shapes, reference_points_cam, level_start_index,
                    bev_query_depth, pred_img_depth, bev_mask,
                    per_cam_mask_list, post_norm)
            # the masked list (:156-169) as a device-side pass: the fused
            # kernels then run exactly as without a bev_mask
            per_cam_mask_list = bev_mask_fold(per_cam_mask_list, bev_mask)
            sca_prepared = None    # counts were taken on the unmasked list

        da = self.deformable_attention
        B, N, DC, H, W = pred_img_depth.shape
        depth_prob = pred_img_depth.reshape(B * N, DC, H * W).permute(0, 2, 1)
        v = (kwargs.get('projected_values') or {}).get(id(self))
        if v is None:
            v = self.project_camera_value(value)
        offsets, logits = da.project_query(
            query, None if query_pos is None else query_pos.float())
        if bev_query_depth.dim() == 5:
            bev_query_depth = bev_query_depth[..., 0]
        if needs_grad(v, depth_prob, offsets, logits):
            slots = da_spatial_cross_attention_core_autograd(
                v, depth_prob, reference_points_cam, bev_query_depth,
                per_cam_mask_list, offsets, logits, spatial_shapes,
                level_start_index, self.dbound, da.num_Z_anchors)
        else:
            slots = da_spatial_cross_attention_core(
                v, depth_prob, reference_points_cam, bev_query_depth,
                per_cam_mask_list, offsets, logits, spatial_shapes,
                level_start_index, self.dbound, da.num_Z_anchors,
                prepared=sca_prepared)
        return self._finish(slots, inp_residual, post_norm)

    def project_camera_value(self, value):
        """value (num_cams, n_value, bs, E) -> value_proj(value) as
        (bs * num_cams, n_value, heads, ch) (:188-191, :524-527).
        key_padding_mask is NOT applied: the reference's call of the deformable
        attention omits it (spatial_cross_attention_depth.py:201-206)."""
        num_cams, n_value, bs, E = value.shape
        value = value.permute(2, 0, 1, 3).reshape(bs * num_cams, n_value, E)
        return self.deformable_attention.project_value(value.float())

    def _forward_rebatch(self, query, value, inp_residual, key_padding_mask,
                         spatial_shapes, reference_points_cam,
                         level_start_index, bev_query_depth, pred_img_depth,
                         bev_mask, per_cam_mask_list, post_norm=None):
        """The reference's per-camera re-batching algorithm (:156-216), used
        when a ``bev_mask`` restricts the queries (its empty-camera rule,
        :166-167, has no per-query formulation)."""
        N, B, nq, Z, _ = bev_query_depth.shape
        _, _, DC, H, W = pred_img_depth.shape
        depth_q = bev_query_depth.permute(1, 0, 2, 3, 4)
        depth_prob = pred_img_depth.reshape(B * N, DC, H * W).permute(0, 2, 1)
        bs = query.shape[0]
        masked = per_cam_mask_list & bev_mask[None, :, :, None]
        seen = masked.sum(-1) > 0                      # (N, bs, nq)
        rows = []
        for j in range(bs):
            per_cam = []
            for i in range(self.num_cams):
                idx = seen[i, j].nonzero().squeeze(-1)
                if idx.numel() == 0:
                    idx = (per_cam_mask_list[i, j].sum(-1) > 0).nonzero(
                    ).squeeze(-1)[0:1]
                per_cam.append(idx)
            rows.append(per_cam)
        max_len = max(len(i) for r in rows for i in r)
        q_re = query.new_zeros(bs, self.num_cams, max_len, self.embed_dims)
        ref_re = reference_points_cam.new_zeros(bs, self.num_cams, max_len, Z,
                                                2)
        dep_re = reference_points_cam.new_zeros(bs, self.num_cams, max_len, Z,
                                                1)
        for j in range(bs):
            for i in range(self.num_cams):
                idx = rows[j][i]
                q_re[j, i, :len(idx)] = query[j, idx]
                dep_re[j, i, :len(idx)] = depth_q[j, i, idx]
                ref_re[j, i, :len(idx)] = reference_points_cam[i, j, idx]
        num_cams, n_value, _, E = value.shape
        value = value.permute(2, 0, 1, 3).reshape(bs * num_cams, n_value, E)
        bins = torch.floor((dep_re - self.dbound[0]) / self.dbound[2])
        bins = torch.clip(bins, 0, DC - 1).to(torch.long)
        onehot = F.one_hot(bins.squeeze(-1), num_classes=DC)
        out = self.deformable_attention(
            query=q_re.view(bs * num_cams, max_len, E), key=value, value=value,
            reference_points=ref_re.view(bs * num_cams, max_len, Z, 2),
            spatial_shapes=spatial_shapes, level_start_index=level_start_index,
            bev_query_depth=onehot.view(bs * num_cams, max_len, Z, DC),
            pred_img_depth=depth_prob.contiguous(),
        ).view(bs, num_cams, max_len, E)
        slots = torch.zeros_like(query)
        for j in range(bs):
            for i in range(num_cams):
                idx = rows[j][i]
                slots[j, idx] += out[j, i, :len(idx)]
        count = seen.permute(1, 2, 0).sum(-1)
        count = torch.clamp(count, min=1.0)
        slots = slots / count[..., None]
        return self._finish(slots, inp_residual, post_norm)


# ---------------------------------------------------------------------------
# custom_base_transformer_layer.py:35-262 / bevformer_encoder.py:206-377
# ---------------------------------------------------------------------------
class MyCustomBaseTransformerLayer(BaseModule):
    """Configurable transformer layer: ``operation_order`` over attentions,
    FFNs and LayerNorms built from config dicts."""

    def __init__(self, attn_cfgs=None,
                 ffn_cfgs=dict(type='FFN', embed_dims=256,
                               feedforward_channels=1024, num_fcs=2,
                               ffn_drop=0.,
                               act_cfg=dict(type='ReLU', inplace=True)),
                 operation_order=None, norm_cfg=dict(type='LN'),
                 init_cfg=None, batch_first=True, **kwargs):
        ffn_cfgs = copy.deepcopy(ffn_cfgs)
        deprecated = dict(feedforward_channels='feedforward_channels',
                          ffn_dropout='ffn_drop', ffn_num_fcs='num_fcs')
        for old, new in deprecated.items():
            if old in kwargs:
                warnings.warn(
                    f'The arguments `{old}` in BaseTransformerLayer has been '
                    f'deprecated, now you should set `{new}` and other FFN '
                    'related arguments to a dict named `ffn_cfgs`. ')
                if ffn_cfgs:
                    ffn_cfgs[new] = kwargs[old]
        super().__init__(init_cfg)
        self.batch_first = batch_first
        num_attn = operation_order.count('self_attn') + \
            operation_order.count('cross_attn')
        if isinstance(attn_cfgs, dict):
            attn_cfgs = [copy.deepcopy(attn_cfgs) for _ in range(num_attn)]
        else:
            attn_cfgs = copy.deepcopy(list(attn_cfgs))
            assert num_attn == len(attn_cfgs), (
                f'The length of attn_cfg {num_attn} is not consistent with '
                f'the number of attention in operation_order '
                f'{operation_order}.')
        self.num_attn = num_attn
        self.operation_order = operation_order
        self.norm_cfg = norm_cfg
        self.pre_norm = operation_order[0] == 'norm'
        self.attentions = nn.ModuleList()
        index = 0
        for name in operation_order:
            if name in ('self_attn', 'cross_attn'):
                if 'batch_first' in attn_cfgs[index]:
                    assert self.batch_first == attn_cfgs[index]['batch_first']
                else:
                    attn_cfgs[index]['batch_first'] = self.batch_first
                attention = build_attention(attn_cfgs[index])
                attention.operation_name = name
                self.attentions.append(attention)
                index += 1
        self.embed_dims = self.attentions[0].embed_dims
        self.ffns = nn.ModuleList()
        num_ffns = operation_order.count('ffn')
        if ffn_cfgs:
            if isinstance(ffn_cfgs, dict):
                ffn_cfgs = [copy.deepcopy(ffn_cfgs) for _ in range(num_ffns)]
            assert len(ffn_cfgs) == num_ffns
            for cfg in ffn_cfgs:
                cfg.setdefault('embed_dims', self.embed_dims)
                assert cfg['embed_dims'] == self.embed_dims
                self.ffns.append(build_feedforward_network(cfg))
        self.norms = nn.ModuleList()
        assert (norm_cfg or {}).get('type', 'LN') == 'LN'
        for _ in range(operation_order.count('norm')):
            self.norms.append(nn.LayerNorm(self.embed_dims))


@register('TRANSFORMER_LAYER')
class BEVFormerEncoderLayer(MyCustomBaseTransformerLayer):

    def __init__(self, attn_cfgs, feedforward_channels=512, ffn_dropout=0.0,
                 operation_order=None, act_cfg=dict(type='ReLU', inplace=True),
                 norm_cfg=dict(type='LN'), ffn_num_fcs=2, **kwargs):
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            super().__init__(attn_cfgs=attn_cfgs,
                             feedforward_channels=feedforward_channels,
                             ffn_dropout=ffn_dropout,
                             operation_order=operation_order, act_cfg=act_cfg,
                             norm_cfg=norm_cfg, ffn_num_fcs=ffn_num_fcs,
                             **kwargs)
        self.fp16_enabled = False
        assert len(operation_order) in {2, 4, 6}

    def forward(self, query, key=None, value=None, bev_pos=None,
                query_pos=None, key_pos=None, attn_masks=None,
                query_key_padding_mask=None, key_padding_mask=None,
                ref_2d=None, ref_3d=None, bev_h=None, bev_w=None,
                reference_points_cam=None, mask=None, spatial_shapes=None,
                level_start_index=None, prev_bev=None, debug=False,
                bev_mask=None, bev_query_depth=None, per_cam_mask_list=None,
                lidar_bev=None, pred_img_depth=None, **kwargs):
        """query (bs, nq, E) -> (bs, nq, E); fp32 throughout (the reference
        pins this layer with @force_fp32, bevformer_encoder.py:250)."""
        query = query.float()
        norm_index = attn_index = ffn_index = 0
        identity = query
        if attn_masks is None:
            attn_masks = [None for _ in range(self.num_attn)]
        elif isinstance(attn_masks, torch.Tensor):
            attn_masks = [copy.deepcopy(attn_masks)
                          for _ in range(self.num_attn)]
        else:
            assert len(attn_masks) == self.num_attn
        # a 'norm' that directly follows an attention / FFN runs in that module's
        # last Linear (same arithmetic, one launch less and no extra pass)
        ops = self.operation_order
        skip_norm = False
        for pos, op in enumerate(ops):
            fold = None
            if (op != 'norm' and not self.pre_norm and pos + 1 < len(ops)
                    and ops[pos + 1] == 'norm'
                    and isinstance(self.norms[norm_index], nn.LayerNorm)):
                fold = self.norms[norm_index]
            if op == 'self_attn':
                query = self.attentions[attn_index](
                    query, None, None, identity if self.pre_norm else None,
                    query_pos=bev_pos, key_pos=bev_pos,
                    attn_mask=attn_masks[attn_index],
                    key_padding_mask=bev_mask, reference_points=ref_2d,
                    spatial_shapes=_const_tensor(((bev_h, bev_w),),
                                                 query.device),
                    level_start_index=_const_tensor((0,), query.device),
                    post_norm=fold, bev_w=bev_w, **kwargs)
                attn_index += 1
                identity = query
                skip_norm = fold is not None
            elif op == 'norm':
                if not skip_norm:
                    query = self.norms[norm_index](query)
                skip_norm = False
                norm_index += 1
            elif op == 'cross_attn':
                query = self.attentions[attn_index](
                    query, key, value, identity if self.pre_norm else None,
                    query_pos=bev_pos, key_pos=key_pos,
                    reference_points=ref_3d,
                    reference_points_cam=reference_points_cam,
                    attn_mask=attn_masks[attn_index],
                    key_padding_mask=key_padding_mask,
                    spatial_shapes=spatial_shapes,
                    level_start_index=level_start_index,
                    bev_query_depth=bev_query_depth,
                    pred_img_depth=pred_img_depth, bev_mask=bev_mask,
                    per_cam_mask_list=per_cam_mask_list, post_norm=fold,
                    **kwargs)
                attn_index += 1
                identity = query
                skip_norm = fold is not None
            elif op == 'ffn':
                query = self.ffns[ffn_index](
                    query, identity if self.pre_norm else None,
                    post_norm=fold)
                ffn_index += 1
                skip_norm = fold is not None
        return query


# ---------------------------------------------------------------------------
# bevformer_encoder.py:27-203
# ---------------------------------------------------------------------------
@register('TRANSFORMER_LAYER_SEQUENCE')
class bevformer_encoder(BaseModule):
    """Encoder: builds the voxel-centre reference points, projects them into
    every camera and runs the layer stack.

    ``fused_geometry`` (default True; ``FBBEV_EXACT_GEOMETRY=1`` or setting the
    attribute to False turns it off): ``forward`` projects the reference points
    with one kernel (``fbbev_point_sampling``) instead of ``point_sampling``'s
    ~20 eager ops (8 ms of cuBLAS batched 3x3 products for 200x200x4 points x 6
    cameras on B200).  Same fp32 chain in the same rounding order as the eager
    ops have on this device (3x3 products as torch's broadcast matmul rounds
    them, ``/= scalar`` as the multiplication by a reciprocal torch's CUDA
    kernel performs): reference points, depths and masks are bit-identical to
    ``point_sampling`` (tests/test_backward_gpu.py::
    test_fused_point_sampling_bit_exact), which keeps the reference's exact
    contract."""

    fused_geometry = os.environ.get('FBBEV_EXACT_GEOMETRY', '0') != '1'
    # overlap the geometry / camera-value branch with the self-attention
    side_stream = os.environ.get('FBBEV_SIDE_STREAM', '1') == '1'

    @staticmethod
    def _side(device):
        key = str(device)
        if key not in _SIDE_STREAMS:
            _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
        return _SIDE_STREAMS[key]

    def __init__(self, *args, pc_range=None, grid_config=None,
                 data_config=None, return_intermediate=False,
                 dataset_type='nuscenes', fix_bug=False,
                 transformerlayers=None, num_layers=None, init_cfg=None,
                 **kwargs):
        super().__init__(init_cfg)
        if isinstance(transformerlayers, dict):
            transformerlayers = [copy.deepcopy(transformerlayers)
                                 for _ in range(num_layers)]
        else:
            assert isinstance(transformerlayers, list) and \
                len(transformerlayers) == num_layers
        self.num_layers = num_layers
        self.layers = nn.ModuleList(
            [build_transformer_layer(cfg) for cfg in transformerlayers])
        self.embed_dims = self.layers[0].embed_dims
        self.pre_norm = self.layers[0].pre_norm
        self.return_intermediate = return_intermediate
        self.fix_bug = fix_bug
        self.x_bound = grid_config['x']
        self.y_bound = grid_config['y']
        self.z_bound = grid_config['z']
        self.final_dim = data_config['input_size']
        self.pc_range = pc_range
        self.fp16_enabled = False

    def get_reference_points(self, H, W, Z=8, dim='3d', bs=1, device='cuda',
                             dtype=torch.float):
        """'3d': voxel-centre grid (Y, X, Z, 3) in ego coordinates (:52-75);
        '2d': normalised BEV pixel centres (bs, H*W, 1, 2) (:78-89)."""
        if dim == '3d':
            axes = []
            for bound in (self.x_bound, self.y_bound, self.z_bound):
                axes.append(torch.arange(*bound, dtype=torch.float) +
                            bound[-1] / 2)
            X, Y, Zc = axes
            Yg, Xg, Zg = torch.meshgrid([Y, X, Zc], indexing='ij')
            return torch.stack([Xg, Yg, Zg], dim=-1).to(dtype).to(device)
        ref_y, ref_x = torch.meshgrid(
            torch.linspace(0.5, H - 0.5, H, dtype=dtype, device=device),
            torch.linspace(0.5, W - 0.5, W, dtype=dtype, device=device),
            indexing='ij')
        ref_y = ref_y.reshape(-1)[None] / H
        ref_x = ref_x.reshape(-1)[None] / W
        ref_2d = torch.stack((ref_x, ref_y), -1)
        return ref_2d.repeat(bs, 1, 1).unsqueeze(2)

    def _axes(self, device):
        key = str(device)
        cache = self.__dict__.setdefault('_axes_cache', {})
        if key not in cache:
            cache[key] = tuple(
                (torch.arange(*b, dtype=torch.float) + b[-1] / 2).to(device)
                for b in (self.x_bound, self.y_bound, self.z_bound))
        return cache[key]

    def _token_major(self, bev_pos):
        """``bev_pos`` arrives as a channel-major view of the (bs, E, h, w)
        encoding, and every ``query + query_pos`` of the layers then runs as a
        strided elementwise kernel (~15 us on B200 instead of ~4).  With
        gradients off the encoding is a cached constant (same root tensor every
        forward), so its (bs, nq, E)-contiguous copy is made once."""
        if torch.is_grad_enabled() or bev_pos.is_contiguous():
            return bev_pos
        root = bev_pos._base if bev_pos._base is not None else bev_pos
        key = (root._version, tuple(bev_pos.shape), tuple(bev_pos.stride()),
               bev_pos.storage_offset())
        hit = self.__dict__.get('_pos_tokens')
        if hit is None or hit[0] is not root or hit[1] != key:
            hit = (root, key, bev_pos.contiguous())
            self.__dict__['_pos_tokens'] = hit
        return hit[2]

    def point_sampling_fused(self, cam_params):
        """``point_sampling`` as one kernel.  The small 3x3 products are formed
        with the same torch ops as the reference (inv_ex == torch.inverse
        without the host-side error check)."""
        rots, trans, intrins, post_rots, post_trans, bda = [
            t.float() for t in cam_params]
        inv_k, inv_bda = inv3x3_many(intrins, bda)
        ego2cam, = inv3x3_many(rots.matmul(inv_k))
        return _msda_ops.point_sampling(
            self._axes(rots.device), inv_bda, trans, ego2cam, post_rots,
            post_trans, self.final_dim)

    def point_sampling(self, reference_points, pc_range, img_metas,
                       cam_params=None, gt_bboxes_3d=None):
        """Ego -> camera -> augmented image plane, the inverse of
        ``get_lidar_coor``; same fp32 operation order as :92-120."""
        rots, trans, intrins, post_rots, post_trans, bda = [
            t.float() for t in cam_params]
        reference_points = reference_points.float()
        B, N, _ = trans.shape
        eps = 1e-5
        ogfH, ogfW = self.final_dim
        pts = reference_points[None, None].repeat(B, N, 1, 1, 1, 1)
        pts = torch.inverse(bda).view(B, 1, 1, 1, 1, 3, 3).matmul(
            pts.unsqueeze(-1)).squeeze(-1)
        pts -= trans.view(B, N, 1, 1, 1, 3)
        ego2cam = rots.matmul(torch.inverse(intrins)).inverse()
        cam = ego2cam.view(B, N, 1, 1, 1, 3, 3).matmul(
            pts.unsqueeze(-1)).squeeze(-1)
        z = cam[..., 2:3]
        cam = torch.cat(
            [cam[..., 0:2] / torch.maximum(z, torch.ones_like(z) * eps), z], 5)
        cam = post_rots.view(B, N, 1, 1, 1, 3, 3).matmul(
            cam.unsqueeze(-1)).squeeze(-1)
        cam += post_trans.view(B, N, 1, 1, 1, 3)
        cam[..., 0] /= ogfW
        cam[..., 1] /= ogfH
        mask = (cam[..., 2:3] > eps)
        mask = (mask & (cam[..., 0:1] > eps) & (cam[..., 0:1] < (1.0 - eps)) &
                (cam[..., 1:2] > eps) & (cam[..., 1:2] < (1.0 - eps)))
        B, N, H, W, D, _ = cam.shape
        cam = cam.permute(1, 0, 2, 3, 4, 5).reshape(N, B, H * W, D, 3)
        mask = mask.permute(1, 0, 2, 3, 4, 5).reshape(
            N, B, H * W, D, 1).squeeze(-1)
        return pts, cam[..., :2], mask, cam[..., 2:3]

    def forward(self, bev_query, key, value, *args, bev_h=None, bev_w=None,
                bev_pos=None, spatial_shapes=None, level_start_index=None,
                valid_ratios=None, cam_params=None, gt_bboxes_3d=None,
                pred_img_depth=None, bev_mask=None, prev_bev=None, **kwargs):
        """bev_query / bev_pos (nq, bs, E); key = value (num_cams, n_value,
        bs, E).  Returns (bs, nq, E) (stacked when return_intermediate)."""
        output = bev_query
        intermediate = []
        cache = self.__dict__.setdefault('_ref2d_cache', {})
        ck = (bev_h, bev_w, bev_query.size(1), str(bev_query.device),
              bev_query.dtype)
        if ck not in cache:  # constant for a given BEV size / batch / device
            cache[ck] = self.get_reference_points(
                bev_h, bev_w, dim='2d', bs=bev_query.size(1),
                device=bev_query.device, dtype=bev_query.dtype)
        ref_2d = cache[ck]
        if self.fused_geometry and bev_query.is_cuda:
            ref_3d = None  # only consumed by point_sampling
            if self.side_stream and not torch.is_grad_enabled() and \
                    bev_mask is None:
                # nothing before the first cross-attention depends on the
                # camera geometry or on the projected camera features: run
                # them (~25 small launches + one Linear) on a side stream
                # beside the self-attention; the cross-attention waits on the
                # event.  Also forks / joins correctly under CUDA-graph capture.
                main = torch.cuda.current_stream(bev_query.device)
                side = self._side(bev_query.device)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    reference_points_cam, per_cam_mask_list, bev_query_depth = \
                        self.point_sampling_fused(cam_params)
                    pv, prep = {}, {}
                    n_layers_with_sca = 0
                    for layer in self.layers:
                        for att in layer.attentions:
                            if isinstance(att, DA_SpatialCrossAttention):
                                pv[id(att)] = att.project_camera_value(value)
                                n_layers_with_sca += 1
                    if n_layers_with_sca == 1:
                        # mask-only prologue of the camera-resident kernel
                        # (counts + zero-filled output) off the critical path
                        for layer in self.layers:
                            for att in layer.attentions:
                                if isinstance(att, DA_SpatialCrossAttention):
                                    da = att.deformable_attention
                                    p = _msda_ops.da_sca_prepare(
                                        per_cam_mask_list, bev_query.size(1),
                                        bev_query.size(0), value.shape[1],
                                        da.num_heads,
                                        att.embed_dims // da.num_heads,
                                        da.num_levels, da.num_points,
                                        da.num_Z_anchors)
                                    if p is not None:
                                        prep[id(att)] = p
                    kwargs['projected_values'] = pv
                    kwargs['sca_prepared'] = prep
                    kwargs['side_event'] = side.record_event()
            else:
                reference_points_cam, per_cam_mask_list, bev_query_depth = \
                    self.point_sampling_fused(cam_params)
        else:
            ref_3d = self.get_reference_points(
                bev_h, bev_w, self.pc_range[5] - self.pc_range[2], dim='3d',
                bs=bev_query.size(1), device=bev_query.device,
                dtype=bev_query.dtype)
            ref_3d, reference_points_cam, per_cam_mask_list, \
                bev_query_depth = self.point_sampling(
                    ref_3d, self.pc_range, kwargs.get('img_metas'),
                    cam_params=cam_params, gt_bboxes_3d=gt_bboxes_3d)
        bev_query = bev_query.permute(1, 0, 2)
        bev_pos = self._token_major(bev_pos.permute(1, 0, 2))
        for layer in self.layers:
            output = layer(
                bev_query, key, value, *args, bev_pos=bev_pos, ref_2d=ref_2d,
                ref_3d=ref_3d, bev_h=bev_h, bev_w=bev_w, prev_bev=prev_bev,
                spatial_shapes=spatial_shapes,
                level_start_index=level_start_index,
                reference_points_cam=reference_points_cam,
                per_cam_mask_list=per_cam_mask_list, bev_mask=bev_mask,
                bev_query_depth=bev_query_depth,
                pred_img_depth=pred_img_depth, **kwargs)
            bev_query = output
            if self.return_intermediate:
                intermediate.append(output)
        if self.return_intermediate:
            return torch.stack(intermediate)
        return output


# ---------------------------------------------------------------------------
# bevformer.py:23-132
# ---------------------------------------------------------------------------
@register('TRANSFORMER')
class BEVFormer(BaseModule):

    def __init__(self, num_cams=6, encoder=None, embed_dims=256,
                 output_dims=256, use_cams_embeds=True, **kwargs):
        super().__init__(**kwargs)
        self.encoder = build_transformer_layer_sequence(encoder)
        self.embed_dims = embed_dims
        self.num_cams = num_cams
        self.fp16_enabled = False
        self.output_dims = output_dims
        self.use_cams_embeds = use_cams_embeds
        self.init_layers()

    def init_layers(self):
        # uninitialised in the reference until init_weights(); zeros here so a
        # freshly built module is deterministic
        self.cams_embeds = nn.Parameter(
            torch.zeros(self.num_cams, self.embed_dims))

    def init_weights(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        for m in self.modules():
            if isinstance(m, (DA_MSDeformableAttention,
                              MultiScaleDeformableAttention)):
                m.init_weights()
        nn.init.normal_(self.cams_embeds)

    def forward(self, mlvl_feats, bev_queries, bev_h, bev_w, bev_pos=None,
                cam_params=None, gt_bboxes_3d=None, pred_img_depth=None,
                prev_bev=None, bev_mask=None, **kwargs):
        bev_pos = bev_pos.flatten(2).permute(2, 0, 1)
        feat_flatten, spatial_shapes = [], []
        for feat in mlvl_feats:
            bs, num_cam, c, h, w = feat.shape
            feat = feat.flatten(3).permute(1, 0, 3, 2)
            embed = self.cams_embeds[:, None, None, :].to(feat.dtype)
            feat = feat + (embed if self.use_cams_embeds else embed * 0)
            spatial_shapes.append((h, w))
            feat_flatten.append(feat)
        feat_flatten = torch.cat(feat_flatten, 2)
        starts, acc = [], 0
        for h, w in spatial_shapes:
            starts.append(acc)
            acc += h * w
        spatial_shapes = _const_tensor(tuple(spatial_shapes), bev_pos.device)
        level_start_index = _const_tensor(tuple(starts), bev_pos.device)
        feat_flatten = feat_flatten.permute(0, 2, 1, 3)  # (cam, HW, bs, E)
        return self.encoder(
            bev_queries, feat_flatten, feat_flatten, bev_h=bev_h, bev_w=bev_w,
            bev_pos=bev_pos, spatial_shapes=spatial_shapes,
            level_start_index=level_start_index, cam_params=cam_params,
            gt_bboxes_3d=gt_bboxes_3d, pred_img_depth=pred_img_depth,
            prev_bev=prev_bev, bev_mask=bev_mask, **kwargs)


# ---------------------------------------------------------------------------
# backward_projection.py:34-133
# ---------------------------------------------------------------------------
@register('HEADS')
class BackwardProjection(BaseModule):
    """BEV queries (learned embedding + lift-splat BEV) refined by the
    depth-aware BEVFormer encoder."""

    def __init__(self, *args, transformer=None, positional_encoding=None,
                 pc_range=None, in_channels=64, out_channels=64,
                 use_zero_embedding=False, bev_h=30, bev_w=30, **kwargs):
        super().__init__()
        self.bev_h = bev_h
        self.bev_w = bev_w
        self.fp16_enabled = False
        self.pc_range = pc_range
        self.use_zero_embedding = use_zero_embedding
        self.real_w = self.pc_range[3] - self.pc_range[0]
        self.real_h = self.pc_range[4] - self.pc_range[1]
        self.positional_encoding = build_positional_encoding(
            positional_encoding)
        self.transformer = build_transformer(transformer)
        self.embed_dims = self.transformer.embed_dims
        self._init_layers()

    def _init_layers(self):
        self.bev_embedding = nn.Embedding(self.bev_h * self.bev_w,
                                          self.embed_dims)

    def init_weights(self):
        self.transformer.init_weights()

    def forward(self, mlvl_feats, img_metas, lss_bev=None, gt_bboxes_3d=None,
                cam_params=None, pred_img_depth=None, bev_mask=None, out=None):
        """mlvl_feats: list of (B, N, C, H, W); lss_bev (B, C, bev_h, bev_w);
        pred_img_depth (B, N, DC, H, W).  Returns (B, C, bev_h, bev_w).

        ``out`` (optional, not in the reference): a contiguous (B, C, bev_h,
        bev_w) tensor to write the result into -- e.g. this rank's slot of an
        all-gather buffer (sharding.py), which saves the copy into it."""
        bs = mlvl_feats[0].shape[0]
        dtype = mlvl_feats[0].dtype
        bev_queries = self.bev_embedding.weight.to(dtype)
        if (lss_bev is not None and lss_bev.is_cuda and dtype == torch.float32
                and not needs_grad(bev_queries, lss_bev)):
            # embedding + transposed lift-splat BEV in one kernel
            bev_queries = _msda_ops.bev_query_init(bev_queries, lss_bev)
        else:
            bev_queries = bev_queries.unsqueeze(1).repeat(1, bs, 1)
            if lss_bev is not None:
                bev_queries = bev_queries + lss_bev.flatten(2).permute(2, 0, 1)
        if bev_mask is not None:
            bev_mask = bev_mask.reshape(bs, -1)
        bev_pos = self.positional_encoding(
            bs, self.bev_h, self.bev_w, bev_queries.device).to(dtype)
        bev = self.transformer(
            mlvl_feats, bev_queries, self.bev_h, self.bev_w,
            grid_length=(self.real_h / self.bev_h, self.real_w / self.bev_w),
            bev_pos=bev_pos, img_metas=img_metas, cam_params=cam_params,
            gt_bboxes_3d=gt_bboxes_3d, pred_img_depth=pred_img_depth,
            prev_bev=None, bev_mask=bev_mask)
        if bev.dim() == 3 and not needs_grad(bev):
            # (bs, nq, E) -> (bs, E, h, w) as one transposing kernel
            res = _msda_ops.tokens_to_map(bev, self.bev_h, self.bev_w, out=out) \
                if bev.is_cuda else None
            if res is not None:
                return res
        bev = bev.permute(0, 2, 1).view(bs, -1, self.bev_h, self.bev_w)
        if out is not None:
            return out.copy_(bev)
        return bev.contiguous()
