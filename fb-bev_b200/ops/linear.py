"""Row-wise Linear (+ bias, ReLU, residual, LayerNorm) on the tcgen05 tensor cores.

Host side of ``fbbev_linear_fwd`` / ``fbbev_ffn_fwd`` (include/fbbev_b200.h): the
nn.Linear / LayerNorm / residual chain of the reference's encoder layer
(bevformer_encoder.py:251-377, spatial_cross_attention_depth.py:219, 420-427)
as one kernel per Linear (one for the whole FFN).  With autograd recording,
:class:`LinearTF32Function` keeps the forward on the same kernel and forms the
three gradient products with plain library GEMMs (cuBLAS through torch).
"""
import torch

from .. import _lib

MAX_N = 192  # widest column block of one launch


def _cached(weight, attr, pack):
    """``pack(weight as contiguous fp32)``, cached ON the weight tensor under
    ``attr`` (so it dies with it and can never be mistaken for another
    tensor's) and keyed by storage address and version counter, so an
    optimizer step or ``load_state_dict`` triggers a re-pack."""
    key = (weight.data_ptr(), weight._version, tuple(weight.shape), weight.device)
    hit = getattr(weight, attr, None)
    if hit is not None and hit[0] == key:
        return hit[1]
    packed = pack(weight.detach().contiguous().float())
    try:
        setattr(weight, attr, (key, packed))
    except AttributeError:  # a tensor type without a __dict__: no caching
        pass
    return packed


def _pack_blocks(w):
    L = _lib.lib()
    n, k = w.shape
    blocks = []
    for n0 in range(0, n, MAX_N):
        n1 = min(n, n0 + MAX_N)
        nbytes = L.fbbev_linear_packed_bytes(n1 - n0, k)
        buf = torch.empty(nbytes // 4, dtype=torch.float32, device=w.device)
        _lib.check(L.fbbev_linear_pack(_lib.ptr(w[n0:n1]), n1 - n0, k, _lib.ptr(buf),
                                       _lib.stream_ptr(w.device)), "fbbev_linear_pack")
        blocks.append((n0, n1, buf))
    return blocks


def _pack(weight):
    """hi / lo split image of `weight` (n, k), one block per <= MAX_N columns."""
    return _cached(weight, "_fbbev_packed", _pack_blocks)


def invalidate(obj):
    """Drop the packed-weight images cached for ``obj`` (an nn.Module, walked
    recursively, or a single weight tensor).

    The caches key on ``Tensor._version``, which in-place updates through
    ``param.data`` (EMA hooks, some checkpoint loaders) do NOT bump -- call
    this after such an update.  ``optimizer.step()``, ``load_state_dict`` and
    ordinary in-place ops on the parameter are detected automatically."""
    if isinstance(obj, torch.Tensor):
        for attr in ("_fbbev_packed", "_fbbev_packed_ffn"):
            if hasattr(obj, attr):
                delattr(obj, attr)
        return
    for m in obj.modules():
        m.__dict__.pop("_pair_cache", None)
        for p in m.parameters(recurse=False):
            for attr in ("_fbbev_packed", "_fbbev_packed_ffn"):
                if hasattr(p, attr):
                    delattr(p, attr)


def ln_supported(n):
    """The LayerNorm epilogue keeps whole rows in shared memory beside two
    pipeline stages (linear_tf32.cu): n <= 80 with the 40-float K-block."""
    npad = (n + 15) // 16 * 16
    stage = 2 * 128 * 40 * 4 + 2 * npad * 40 * 4
    return 2 * stage + 256 + 3 * MAX_N * 4 + 2 * 128 * (n + 4) * 4 <= 232448 - 1024


def supported(x, weight):
    n, k = weight.shape
    return (x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32
            and k % 4 == 0 and n % 4 == 0 and not torch.is_grad_enabled())


def linear_fused(x, weight, bias=None, relu=False, residual=None, ln_weight=None,
                 ln_bias=None, eps=1e-5):
    """``LN(act(x @ weight.T + bias) + residual)`` with every part optional."""
    _lib.require_cuda(x)
    n, k = weight.shape
    assert x.shape[-1] == k
    lead = x.shape[:-1]
    x2 = x.reshape(-1, k)
    if x2.stride(-1) != 1 or x2.stride(0) % 4 or x2.data_ptr() % 16:
        x2 = x2.contiguous()
    m = x2.shape[0]
    y = torch.empty((m, n), dtype=torch.float32, device=x.device)
    r2 = None
    if residual is not None:
        r2 = residual.reshape(-1, n)
        if r2.stride(-1) != 1 or r2.stride(0) % 4 or r2.data_ptr() % 16:
            r2 = r2.contiguous()
    blocks = _pack(weight)
    if ln_weight is not None and not ln_supported(n):
        raise _lib.FbbevError("LayerNorm epilogue: n = %d does not fit" % n)
    L = _lib.lib()
    sp = _lib.stream_ptr(x.device)
    b = bias.detach().contiguous() if bias is not None else None
    for n0, n1, buf in blocks:
        _lib.check(L.fbbev_linear_fwd(
            _lib.ptr(x2), x2.stride(0), _lib.ptr(buf),
            _lib.ptr(b[n0:n1]) if b is not None else None,
            _lib.ptr(r2[:, n0:n1]) if r2 is not None else None,
            r2.stride(0) if r2 is not None else 0,
            _lib.ptr(ln_weight) if ln_weight is not None else None,
            _lib.ptr(ln_bias) if ln_bias is not None else None,
            m, k, n1 - n0, int(bool(relu)), float(eps),
            _lib.ptr(y[:, n0:n1]), y.stride(0), sp), "fbbev_linear_fwd")
    return y.view(*lead, n)


def _rows(t, k):
    """(-1, k) view of ``t`` usable by the kernels (dense rows, 16-byte
    aligned), copying only when the layout demands it."""
    t2 = t.reshape(-1, k)
    if t2.stride(-1) != 1 or t2.stride(0) % 4 or t2.data_ptr() % 16:
        t2 = t2.contiguous()
    return t2


def linear_pair(x, weight_a, bias_a, weight_b, bias_b, cache, x_add=None):
    """``(x @ weight_a.T + bias_a, x @ weight_b.T + bias_b)`` as ONE launch when
    both fit a column block (sampling_offsets + attention_weights of an
    attention module: same input, one consumer kernel).  With ``x_add`` the
    input is ``x + x_add`` (``query + query_pos``), added in the kernel's loader.

    ``cache`` is a dict owned by the calling module; it keeps the concatenated
    weight / bias, keyed by the parameters' storage and version counters."""
    _lib.require_cuda(x)
    na, k = weight_a.shape
    nb = weight_b.shape[0]
    if na + nb > MAX_N or na % 4 or nb % 4 or (bias_a is None) != (bias_b is None):
        if x_add is not None:
            x = x + x_add
        return (linear_fused(x, weight_a, bias_a), linear_fused(x, weight_b, bias_b))
    key = tuple((t.data_ptr(), t._version) for t in
                (weight_a, weight_b, bias_a, bias_b) if t is not None)
    hit = cache.get("pair")
    if hit is None or hit[0] != key:
        w = torch.cat((weight_a.detach(), weight_b.detach()), 0).float().contiguous()
        b = None if bias_a is None else torch.cat(
            (bias_a.detach(), bias_b.detach()), 0).float().contiguous()
        hit = (key, w, b)
        cache["pair"] = hit
    _, w, b = hit
    lead = x.shape[:-1]
    x2 = _rows(x, k)
    m = x2.shape[0]
    xa = None
    if x_add is not None:
        if x_add.shape != x.shape:
            x_add = x_add.expand_as(x)
        xa = _rows(x_add, k)
    ya = torch.empty((m, na), dtype=torch.float32, device=x.device)
    yb = torch.empty((m, nb), dtype=torch.float32, device=x.device)
    (_, _, buf), = _pack(w)
    L = _lib.lib()
    _lib.check(L.fbbev_linear_fwd_split(
        _lib.ptr(x2), x2.stride(0), _lib.ptr(xa),
        xa.stride(0) if xa is not None else 0, _lib.ptr(buf), _lib.ptr(b), m, k,
        na + nb, na, 0, _lib.ptr(ya), na, _lib.ptr(yb), nb,
        _lib.stream_ptr(x.device)), "fbbev_linear_fwd_split")
    return ya.view(*lead, na), yb.view(*lead, nb)


def _pack_w1_chunks(w):
    L = _lib.lib()
    hidden, k = w.shape
    assert hidden % 80 == 0
    per = L.fbbev_linear_packed_bytes(80, k) // 4
    buf = torch.empty(per * (hidden // 80), dtype=torch.float32, device=w.device)
    for c in range(hidden // 80):
        _lib.check(L.fbbev_linear_pack(
            _lib.ptr(w[80 * c:80 * c + 80]), 80, k, _lib.ptr(buf[per * c:]),
            _lib.stream_ptr(w.device)), "fbbev_linear_pack")
    return buf


def _pack_ffn_w1(weight):
    """W1 (hidden, embed) as hidden / 80 separately packed 80-row blocks, one
    buffer (the layout ``fbbev_ffn_fwd`` streams)."""
    return _cached(weight, "_fbbev_packed_ffn", _pack_w1_chunks)


def ffn_supported(x, w1, w2):
    hidden, embed = w1.shape
    return (supported(x, w1) and tuple(w2.shape) == (embed, hidden) and
            bool(_lib.lib().fbbev_ffn_supported(embed, hidden)))


def ffn_fused(x, w1, b1, w2, b2, residual=None, ln_weight=None, ln_bias=None,
              eps=1e-5):
    """``LN(residual + relu(x @ w1.T + b1) @ w2.T + b2)`` as ONE kernel
    (``fbbev_ffn_fwd``): the hidden activation never leaves the SM."""
    _lib.require_cuda(x)
    hidden, embed = w1.shape
    assert x.shape[-1] == embed and tuple(w2.shape) == (embed, hidden)
    lead = x.shape[:-1]
    x2 = _rows(x, embed)
    m = x2.shape[0]
    r2 = _rows(residual, embed) if residual is not None else None
    y = torch.empty((m, embed), dtype=torch.float32, device=x.device)
    w1p = _pack_ffn_w1(w1)
    (_, _, w2p), = _pack(w2)
    _lib.check(_lib.lib().fbbev_ffn_fwd(
        _lib.ptr(x2), x2.stride(0), _lib.ptr(w1p),
        _lib.ptr(b1.detach().contiguous()) if b1 is not None else None,
        _lib.ptr(w2p),
        _lib.ptr(b2.detach().contiguous()) if b2 is not None else None,
        _lib.ptr(r2), r2.stride(0) if r2 is not None else 0,
        _lib.ptr(ln_weight) if ln_weight is not None else None,
        _lib.ptr(ln_bias) if ln_bias is not None else None,
        m, embed, hidden, float(eps), _lib.ptr(y), y.stride(0),
        _lib.stream_ptr(x.device)), "fbbev_ffn_fwd")
    return y.view(*lead, embed)


class LinearTF32Function(torch.autograd.Function):
    """``act(x @ weight.T + bias) + residual`` with the forward on the tcgen05
    kernel (``fbbev_linear_fwd``: same 3xTF32 arithmetic as inference) and the
    backward as plain library GEMMs::

        g  = grad * (y > 0)           (ReLU only)
        dx = g @ weight    dW = g^T @ x    db = sum_rows(g)    dresidual = grad

    The reference trains these layers through cuBLAS in both directions
    (nn.Linear); here only the backward is a library call.  LayerNorm stays a
    torch op on this route (its backward needs the row statistics)."""

    @staticmethod
    def forward(ctx, x, weight, bias, relu, residual):
        assert not (relu and residual is not None)
        y = linear_fused(
            x.detach(), weight.detach(),
            None if bias is None else bias.detach(), relu=relu,
            residual=None if residual is None else residual.detach())
        ctx.relu = relu
        ctx.has_bias = bias is not None
        ctx.has_res = residual is not None
        ctx.save_for_backward(x, weight, y if relu else None)
        return y

    @staticmethod
    def backward(ctx, grad):
        x, weight, y = ctx.saved_tensors
        g = grad * (y > 0).to(grad.dtype) if ctx.relu else grad
        n, k = weight.shape
        g2 = g.reshape(-1, n)
        gx = gw = gb = gr = None
        if ctx.needs_input_grad[0]:
            gx = (g2 @ weight).view(x.shape)
        if ctx.needs_input_grad[1]:
            gw = g2.t() @ x.reshape(-1, k)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g2.sum(0)
        if ctx.has_res and ctx.needs_input_grad[4]:
            gr = grad
        return gx, gw, gb, None, gr


def linear_train(x, weight, bias=None, relu=False, residual=None):
    """Differentiable ``act(x @ weight.T + bias) + residual``; forward on the
    tensor-core kernel.  Shapes the kernel does not take (k or n not a multiple
    of 4) must be handled by the caller."""
    if relu and residual is not None:
        return LinearTF32Function.apply(x, weight, bias, True, None) + residual
    return LinearTF32Function.apply(x, weight, bias, relu, residual)
