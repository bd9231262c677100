"""GPU parity tests of the forward (lift-splat) path.  Every CUDA result is
obtained through the C ABI (ctypes -> libfbbev_b200.so) and compared with the
CPU oracle, the committed golden fixtures, the reference's known-answer test
and the recorded outputs of the reference's own CUDA kernels.

Tolerance: integer index path bit-exact; float outputs <= 1e-4 absolute
(BASELINE.json north_star), in practice a few ulp."""
import hashlib

import numpy as np
import pytest
import torch

from conftest import canon_index, load_golden
from test_oracle import (KAT_GRAD_DEPTH, KAT_GRAD_FEAT, kat_inputs)

pytestmark = pytest.mark.gpu
ATOL = 1e-4
DEV = "cuda:0"


def t(a, dtype=None):
    x = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return x if dtype is None else x.to(dtype)


def make_case(name, batch, seed=0):
    """Synthetic rig case -> (vt module on GPU side objects, coor, depth, feat)."""
    from fbbev_b200 import synthetic
    from fbbev_b200.view_transformation.forward_projection import \
        LSSViewTransformerFunction3D
    cfgs = {
        # name: (grid, input_size, downsample, n_cams, C)
        "shipped": ("fbocc_shipped", (256, 704), 16, 6, 80),
        "fbocc_200": ("fbocc_200", (256, 704), 16, 6, 80),
        "unit_128": ("unit_128", (256, 704), 4, 1, 80),
        "unit_128_c64": ("unit_128", (256, 704), 4, 1, 64),
        # BASELINE.json configs[4]: 400x400x32 voxels, 6-cam 512x1408, D = 118
        "fbocc_400": ("fbocc_400", (512, 1408), 16, 6, 80),
    }
    grid, inp, ds, n_cams, C = cfgs[name]
    vt = LSSViewTransformerFunction3D(synthetic.GRID_CONFIGS[grid], inp, ds)
    cam = synthetic.make_cam_params(batch, n_cams, inp, device=DEV,
                                    jitter=1.0 if batch > 1 else 0.0,
                                    seed=seed)
    H, W = inp[0] // ds, inp[1] // ds
    depth, feat = synthetic.make_depth_feat(batch, n_cams, vt.D, H, W, C,
                                            device=DEV, seed=seed)
    return vt, cam, depth, feat


# ---------------------------------------------------------------- KAT ------
def test_kat_forward_and_backward():
    """bev_pool.py:145-176 through the fused op (forward sum 4.4, both grads)."""
    from fbbev_b200.ops.bev_pool_v2 import QuickCumsumCuda, bev_pool_v2
    depth, feat, rd, rf, rb, shape, st, ln = kat_inputs()
    for op in ("fused", "reference-layout"):
        d = t(depth).requires_grad_()
        f = t(feat).requires_grad_()
        args = (d, f, t(rd), t(rf), t(rb), shape, t(st), t(ln))
        if op == "fused":
            out = bev_pool_v2(*args)
            assert out.shape == (1, 2, 1, 2, 2) and out.is_contiguous()
        else:
            out = QuickCumsumCuda.apply(*args)
            assert out.shape == (1, 1, 2, 2, 2)
        loss = out.sum()
        loss.backward()
        assert abs(float(loss) - 4.4) < 1e-6
        np.testing.assert_allclose(d.grad.cpu().numpy().ravel(),
                                   KAT_GRAD_DEPTH, atol=1e-6)
        np.testing.assert_allclose(f.grad.cpu().numpy().ravel(),
                                   KAT_GRAD_FEAT, atol=1e-6)


# ------------------------------------------------------- index preparation --
@pytest.mark.parametrize("case", ["f_small_6cam", "f_unit_1cam",
                                  "f_negative_trunc"])
def test_prepare_vs_reference_golden(case):
    from fbbev_b200.ops.bev_pool_v2 import voxel_pooling_prepare_v2
    g = load_golden(case)
    idx = voxel_pooling_prepare_v2(t(g["coor"]), g["grid_lower_bound"],
                                   g["grid_interval"], g["grid_size"])
    rb, rd, rf, st, ln = (x.cpu().numpy() for x in idx.trimmed())
    np.testing.assert_array_equal(rb, g["ranks_bev"])
    np.testing.assert_array_equal(st, g["interval_starts"])
    np.testing.assert_array_equal(ln, g["interval_lengths"])
    ref = canon_index(g["ranks_bev"], g["ranks_depth"], g["ranks_feat"])
    # device order is already the canonical (stable) one
    for x, y in zip((rb, rd, rf), ref):
        np.testing.assert_array_equal(x, y)


def test_prepare_empty_golden():
    from fbbev_b200.ops.bev_pool_v2 import voxel_pooling_prepare_v2
    g = load_golden("f_empty")
    idx = voxel_pooling_prepare_v2(t(g["coor"]), g["grid_lower_bound"],
                                   g["grid_interval"], g["grid_size"])
    assert idx.counts.tolist() == [0, 0]
    assert all(x is None for x in idx.trimmed())


@pytest.mark.parametrize("name,batch", [("shipped", 1), ("shipped", 2),
                                        ("fbocc_200", 1), ("unit_128", 1)])
def test_prepare_vs_oracle_exact(oracle_cpu, name, batch):
    vt, cam, depth, feat = make_case(name, batch)
    coor = vt.get_lidar_coor(*cam)
    got = [x.cpu().numpy() for x in vt.voxel_pooling_prepare_v2(coor)]
    want = oracle_cpu.voxel_prepare(coor.cpu().numpy(),
                                    vt.grid_lower_bound.numpy(),
                                    vt.grid_interval.numpy(),
                                    vt.grid_size.numpy())
    for a, b, n in zip(got, want, ["rb", "rd", "rf", "st", "ln"]):
        np.testing.assert_array_equal(a, b, err_msg=n)
    # structural invariants (size independent)
    rb, rd, rf, st, ln = got
    assert np.all(np.diff(rb) >= 0)                        # sortedness
    assert ln.sum() == len(rb) and st[0] == 0              # partition
    assert np.all(st[1:] == np.cumsum(ln)[:-1])
    assert np.all(np.diff(rb[st]) > 0)                     # one run per voxel
    assert len(np.unique(rd)) == len(rd)                   # each point once


# ------------------------------------------------------------- pooling ------
@pytest.mark.parametrize("case", ["f_small_6cam", "f_unit_1cam",
                                  "f_negative_trunc", "f_empty"])
def test_plugin_forward_vs_reference_golden(case):
    """LSSViewTransformerFunction3D.forward on the golden camera parameters
    equals the reference module's output (same shape, same view layout)."""
    from test_forward_projection_cpu import build
    g = load_golden(case)
    vt = build(g)
    cam = [t(g[k]) for k in ("rots", "trans", "intrins", "post_rots",
                             "post_trans", "bda")]
    if case in ("f_negative_trunc", "f_empty"):
        bev = vt.voxel_pooling_v2(t(g["coor"]), t(g["depth"]), t(g["feat"]))
    else:
        bev = vt(cam, t(g["feat"]), t(g["depth"]))
    assert tuple(bev.shape) == tuple(g["bev_feat_shape"])
    np.testing.assert_allclose(bev.cpu().numpy(), g["bev_feat"], rtol=0,
                               atol=ATOL)


@pytest.mark.parametrize("name,batch", [("shipped", 1), ("shipped", 3),
                                        ("fbocc_200", 1), ("unit_128", 1),
                                        ("unit_128_c64", 1)])
def test_dense_pool_vs_oracle(oracle_cpu, name, batch):
    from fbbev_b200.ops.bev_pool_v2 import QuickCumsumCuda, bev_pool_v2
    vt, cam, depth, feat = make_case(name, batch)
    coor = vt.get_lidar_coor(*cam)
    rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
    feat_nhwc = feat.permute(0, 1, 3, 4, 2)
    shape = vt._bev_feat_shape(depth, feat_nhwc)
    got = bev_pool_v2(depth, feat_nhwc, rd, rf, rb, shape, st, ln)
    want = oracle_cpu.bev_pool_v2(
        depth.cpu().numpy(), feat_nhwc.contiguous().cpu().numpy(),
        rd.cpu().numpy(), rf.cpu().numpy(), rb.cpu().numpy(), shape,
        st.cpu().numpy(), ln.cpu().numpy())
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=ATOL)
    # reference-layout drop-in kernel: same numbers, (B,Z,Y,X,C)
    ref_layout = QuickCumsumCuda.apply(depth, feat_nhwc, rd, rf, rb, shape, st,
                                       ln)
    np.testing.assert_allclose(ref_layout.cpu().numpy(),
                               want.transpose(0, 2, 3, 4, 1), rtol=0,
                               atol=ATOL)
    # (voxels whose points straddle two warps of the dense kernel are summed
    # as two partials, so the two kernels agree to rounding, not bit for bit)
    assert (ref_layout.permute(0, 4, 1, 2, 3) - got).abs().max().item() <= ATOL
    # sync-free plugin path (padded buffers + device counts) == trimmed path
    vt.fused_geometry = False          # same coordinates as `coor` above
    bev = vt(cam, feat, depth)
    assert torch.equal(bev, got.permute(0, 1, 3, 4, 2))


@pytest.mark.parametrize("name", ["shipped", "fbocc_200", "unit_128",
                                  "fbocc_400"])
def test_vs_reference_cuda_kernel(name):
    """Same inputs as the UNMODIFIED reference kernels were given when
    k_ref_cuda.npz was recorded (tests/golden/gen_golden_ref_kernel.py)."""
    from fbbev_b200.ops.bev_pool_v2 import QuickCumsumCuda, bev_pool_v2
    g = load_golden("k_ref_cuda")
    vt, cam, depth, feat = make_case(name, 1)
    coor = vt.get_lidar_coor(*cam)
    rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
    feat_nhwc = feat.permute(0, 1, 3, 4, 2).contiguous()
    shape = vt._bev_feat_shape(depth, feat_nhwc)
    got = bev_pool_v2(depth, feat_nhwc, rd, rf, rb, shape, st, ln)
    # the drop-in interval kernel keeps the reference's summation order:
    # identical bits, checked on the whole volume through its hash
    same_order = QuickCumsumCuda.apply(depth, feat_nhwc, rd, rf, rb, shape, st,
                                       ln).permute(0, 4, 1, 2, 3).contiguous()
    idx = t(g[name + "__idx"])
    want = g[name + "__val"]
    np.testing.assert_array_equal(same_order.reshape(-1)[idx].cpu().numpy(),
                                  want)
    digest = hashlib.sha256(same_order.cpu().numpy().tobytes()).digest()
    assert digest == g[name + "__sha256"].tobytes()
    # so the fused op is within ATOL of the reference everywhere
    np.testing.assert_allclose(got.reshape(-1)[idx].cpu().numpy(), want,
                               rtol=0, atol=ATOL)
    err = (got - same_order).abs().max().item()
    assert err <= ATOL, err


def test_backward_vs_oracle_and_reference_kernel(oracle_cpu):
    from fbbev_b200.ops.bev_pool_v2 import bev_pool_v2
    vt, cam, depth, feat = make_case("shipped", 1)
    coor = vt.get_lidar_coor(*cam)
    rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
    feat_nhwc = feat.permute(0, 1, 3, 4, 2).contiguous()
    shape = vt._bev_feat_shape(depth, feat_nhwc)
    d = depth.clone().requires_grad_()
    f = feat_nhwc.clone().requires_grad_()
    out = bev_pool_v2(d, f, rd, rf, rb, shape, st, ln)
    go = torch.randn(out.shape, device=DEV,
                     generator=torch.Generator(DEV).manual_seed(5))
    out.backward(go)
    go_zyxc = go.permute(0, 2, 3, 4, 1).contiguous()
    dg, fg = oracle_cpu.bev_pool_v2_bwd(
        go_zyxc.cpu().numpy(), depth.cpu().numpy(), feat_nhwc.cpu().numpy(),
        rd.cpu().numpy(), rf.cpu().numpy(), rb.cpu().numpy())
    np.testing.assert_allclose(d.grad.cpu().numpy(), dg, rtol=0, atol=2e-4)
    np.testing.assert_allclose(f.grad.cpu().numpy(), fg, rtol=0, atol=2e-4)
    # the reference's own backward kernels on these inputs (recorded sample)
    g = load_golden("k_ref_cuda")
    for grad, key in ((d.grad, "depth"), (f.grad, "feat")):
        got = grad.reshape(-1)[t(g[f"bwd__{key}_idx"])].cpu().numpy()
        np.testing.assert_allclose(got, g[f"bwd__{key}_grad"], rtol=0,
                                   atol=2e-4, err_msg=key)


# ----------------------------------- size-independent properties, full size --
@pytest.mark.parametrize("name,batch", [("fbocc_200", 2), ("shipped", 4),
                                        ("fbocc_400", 1)])
def test_properties_full_size(name, batch):
    from fbbev_b200.ops.bev_pool_v2 import bev_pool_v2
    vt, cam, depth, feat = make_case(name, batch)
    coor = vt.get_lidar_coor(*cam)
    idx = vt.prepare_index(coor)
    rb, rd, rf, st, ln = idx.trimmed()
    feat_nhwc = feat.permute(0, 1, 3, 4, 2).contiguous()
    shape = vt._bev_feat_shape(depth, feat_nhwc)
    out = bev_pool_v2(depth, feat_nhwc, rd, rf, rb, shape, st, ln)
    B, C = out.shape[:2]
    flat = out.reshape(B, C, -1)
    # (1) every voxel without an interval is exactly zero, every other written
    occ = torch.zeros(B * flat.shape[2], dtype=torch.bool, device=DEV)
    occ[rb[st.long()].long()] = True
    occ = occ.view(B, 1, -1)
    assert torch.all(flat.masked_select(~occ.expand_as(flat)) == 0)
    # (2) checksum of checksums: sum over voxels of out[b,c] ==
    #     sum over kept points of depth * feat[c]   (float64 accumulation)
    d = depth.reshape(-1)[rd.long()].double()
    fsel = feat_nhwc.reshape(-1, C)[rf.long()].double()
    want = torch.zeros(B, C, dtype=torch.float64, device=DEV)
    bidx = (rb.long() // flat.shape[2])
    want.index_add_(0, bidx, fsel * d[:, None])
    got = flat.double().sum(-1)
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-3)
    # (3) linearity in feat and in depth
    out2 = bev_pool_v2(depth * 2.0, feat_nhwc * 0.5, rd, rf, rb, shape, st, ln)
    assert torch.allclose(out2, out, rtol=1e-6, atol=1e-6)
    # (4) idempotence / determinism: same call, same bits
    out3 = bev_pool_v2(depth, feat_nhwc, rd, rf, rb, shape, st, ln)
    assert torch.equal(out3, out)


def test_odd_grid_scalar_store_path(oracle_cpu):
    """Z*Y*X not a multiple of 4 (no 128-bit stores) and a partial last tile."""
    from fbbev_b200.ops.bev_pool_v2 import bev_pool_v2, \
        voxel_pooling_prepare_v2
    g = torch.Generator().manual_seed(3)
    B, N, D, H, W, C = 2, 2, 5, 6, 7, 13
    lo = torch.tensor([-3.5, -2.5, -1.0])
    iv = torch.tensor([1.0, 1.0, 1.0])
    gs = torch.tensor([7.0, 5.0, 3.0])  # 105 voxels per sample
    coor = (torch.rand(B, N, D, H, W, 3, generator=g) * 9 - 4.5)
    depth = torch.rand(B, N, D, H, W, generator=g)
    feat = torch.randn(B, N, H, W, C, generator=g)
    idx = voxel_pooling_prepare_v2(coor.to(DEV), lo, iv, gs)
    rb, rd, rf, st, ln = idx.trimmed()
    shape = (B, 3, 5, 7, C)
    got = bev_pool_v2(depth.to(DEV), feat.to(DEV), rd, rf, rb, shape, st, ln)
    o = oracle_cpu.voxel_prepare(coor.numpy(), lo.numpy(), iv.numpy(),
                                 gs.numpy())
    for a, b in zip((rb, rd, rf, st, ln), o):
        np.testing.assert_array_equal(a.cpu().numpy(), b)
    want = oracle_cpu.bev_pool_v2(depth.numpy(), feat.numpy(), o[1], o[2],
                                  o[0], shape, o[3], o[4])
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=ATOL)


def test_wide_channels(oracle_cpu):
    """C = 256 (FB-BEV embed width) exercises the 8-channels-per-lane path."""
    from fbbev_b200.ops.bev_pool_v2 import QuickCumsumCuda, bev_pool_v2
    g = torch.Generator().manual_seed(4)
    n_pts, n_vox, C = 5000, 4096, 256
    rb = torch.sort(torch.randint(0, n_vox, (n_pts,), generator=g))[0].int()
    rd = torch.randperm(n_pts, generator=g).int()
    rf = torch.randint(0, 600, (n_pts,), generator=g).int()
    kept = torch.ones(n_pts, dtype=torch.bool)
    kept[1:] = rb[1:] != rb[:-1]
    st = torch.where(kept)[0].int()
    ln = torch.diff(torch.cat([st, torch.tensor([n_pts], dtype=torch.int32)]))
    depth = torch.rand(1, 1, n_pts, 1, 1, generator=g)
    feat = torch.randn(1, 1, 600, 1, C, generator=g)
    shape = (1, 1, 64, 64, C)
    args = [x.to(DEV) for x in (depth, feat, rd, rf, rb)]
    got = bev_pool_v2(*args, shape, st.to(DEV), ln.int().to(DEV))
    want = oracle_cpu.bev_pool_v2(depth.numpy(), feat.numpy(), rd.numpy(),
                                  rf.numpy(), rb.numpy(), shape, st.numpy(),
                                  ln.int().numpy())
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=0, atol=ATOL)
    ref_layout = QuickCumsumCuda.apply(*args, shape, st.to(DEV),
                                       ln.int().to(DEV))
    assert (ref_layout.permute(0, 4, 1, 2, 3) - got).abs().max().item() <= ATOL


def _augment(cam, seed=5):
    """Training-style augmentation so no matrix of the chain is diagonal:
    rotated / flipped post_rots, rotated + scaled bda (loading.py:1064-1105,
    1308-1394)."""
    rots, trans, intr, post_rots, post_trans, bda = [c.clone() for c in cam]
    g = torch.Generator().manual_seed(seed)
    B, N = trans.shape[:2]
    ang = (torch.rand(B, N, generator=g) - 0.5) * 0.2
    c, s_ = torch.cos(ang), torch.sin(ang)
    R = torch.zeros(B, N, 3, 3)
    R[..., 0, 0], R[..., 0, 1], R[..., 1, 0], R[..., 1, 1] = c, -s_, s_, c
    R[..., 2, 2] = 1
    flip = (torch.rand(B, N, generator=g) > 0.5).float() * -2 + 1
    R[..., 0, :] *= flip[..., None]
    post_rots = R.to(DEV).matmul(post_rots)
    post_trans = post_trans + (torch.randn(B, N, 3, generator=g) * 3).to(DEV) * \
        torch.tensor([1.0, 1.0, 0.0], device=DEV)
    a = (torch.rand(B, generator=g) - 0.5) * 0.8
    Rb = torch.zeros(B, 3, 3)
    Rb[:, 0, 0], Rb[:, 0, 1] = torch.cos(a), -torch.sin(a)
    Rb[:, 1, 0], Rb[:, 1, 1] = torch.sin(a), torch.cos(a)
    Rb[:, 2, 2] = 1
    Rb *= (0.95 + 0.1 * torch.rand(B, 1, 1, generator=g))
    return rots, trans, intr, post_rots, post_trans, Rb.to(DEV)


@pytest.mark.parametrize("name,batch,aug", [
    ("unit_128", 1, False),      # configs[0]: one camera (B*N == 1)
    ("fbocc_200", 1, False),     # configs[1], the bench workload
    ("fbocc_200", 16, True),     # configs[2]: 16 frames
    ("fbocc_400", 1, True),      # configs[4]
    ("shipped", 2, True), ("shipped", 1, True), ("unit_128", 1, True),
    ("unit_128", 3, True)])
def test_fused_geometry_bit_exact(name, batch, aug):
    """The plugin's default forward evaluates get_lidar_coor inside the
    voxelisation kernel.  The integer index it produces must be IDENTICAL to
    voxel_pooling_prepare_v2(get_lidar_coor(...)) -- the reference's own eager
    chain on this device (view_transformer.py:458-498, 547-605): no point may
    change voxel, on every BASELINE.json config."""
    vt, cam, depth, feat = make_case(name, batch)
    if aug:
        cam = _augment(cam)
    coor = vt.get_lidar_coor(*cam)
    exact = vt.prepare_index(coor)
    fused = vt.prepare_index_from_cams(*cam)
    assert torch.equal(exact.counts, fused.counts)
    n_kept, n_int = exact.counts.tolist()
    assert n_kept > 0
    for a, b in ((exact.ranks_bev, fused.ranks_bev),
                 (exact.ranks_depth, fused.ranks_depth),
                 (exact.ranks_feat, fused.ranks_feat)):
        assert torch.equal(a[:n_kept], b[:n_kept])
    assert torch.equal(exact.interval_starts[:n_int],
                       fused.interval_starts[:n_int])
    assert torch.equal(exact.interval_lengths[:n_int],
                       fused.interval_lengths[:n_int])
    # the small 3x3 constants feeding the kernel == the reference's own ops
    from fbbev_b200.view_transformation.forward_projection import inv3x3_many
    inv_pr, inv_k = inv3x3_many(cam[3], cam[2])
    assert torch.equal(inv_pr, torch.inverse(cam[3]))
    assert torch.equal(inv_k, torch.inverse(cam[2]))
    if batch <= 2:
        vt.fused_geometry = True
        bev_f = vt(cam, feat, depth)
        vt.fused_geometry = False
        bev_e = vt(cam, feat, depth)
        assert torch.equal(bev_f, bev_e)


# ------------------------------------------- 2-D class / cached index ------
def _vt2d(g, accelerate, cls_name="LSSViewTransformerFunction"):
    from fbbev_b200.view_transformation import forward_projection as fp
    grid = dict(x=list(g["grid_x"]), y=list(g["grid_y"]), z=list(g["grid_z"]),
                depth=list(g["grid_depth"]))
    return getattr(fp, cls_name)(grid, tuple(int(v) for v in g["input_size"]),
                                 int(g["downsample"]), accelerate=accelerate)


@pytest.mark.parametrize("case", ["f2d_z1_6cam", "f2d_z4_6cam"])
@pytest.mark.parametrize("fused", [True, False])
def test_lss_2d_vs_reference_golden(case, fused):
    """LSSViewTransformerFunction (view_transformer.py:24-311), the BEVDet-
    lineage 2-D transformer: Z collapsed into channels (:191); with
    ``accelerate=True`` the index of the FIRST cam_params is cached and Z is
    squeezed instead (:266-283) -- outputs of the reference's own class."""
    g = load_golden(case)
    cam = [t(g[k]) for k in ("rots", "trans", "intrins", "post_rots",
                             "post_trans", "bda")]
    vt = _vt2d(g, accelerate=False)
    vt.fused_geometry = fused
    out = vt(cam, t(g["feat"]), t(g["depth"]))
    assert tuple(out.shape) == g["bev"].shape
    np.testing.assert_allclose(out.cpu().numpy(), g["bev"], rtol=0, atol=ATOL)

    acc = _vt2d(g, accelerate=True)
    acc.fused_geometry = fused
    out = acc(cam, t(g["feat"]), t(g["depth"]))
    assert tuple(out.shape) == g["bev_acc"].shape
    np.testing.assert_allclose(out.cpu().numpy(), g["bev_acc"], rtol=0,
                               atol=ATOL)
    assert acc.initial_flag is False
    # the reference keeps its five index tensors as attributes (:166-170)
    for name in ("ranks_bev", "ranks_depth", "ranks_feat", "interval_starts",
                 "interval_lengths"):
        assert getattr(acc, name).dtype == torch.int32
    # second call: cached index, other cameras must be ignored
    other = [c.clone() for c in cam]
    other[1] = other[1] + 5.0
    out2 = acc(other, t(g["feat2"]), t(g["depth2"]))
    np.testing.assert_allclose(out2.cpu().numpy(), g["bev_acc_second"], rtol=0,
                               atol=ATOL)


def test_lss_3d_accelerate_cached_index():
    """accelerate=True on the 3-D class (the reference's 3-D class asserts out,
    view_transformer.py:628; here it caches the index like the 2-D class):
    same volume as the uncached forward, index computed once."""
    vt, cam, depth, feat = make_case("shipped", 2)
    want = vt(cam, feat, depth)
    from fbbev_b200 import synthetic
    from fbbev_b200.view_transformation.forward_projection import \
        LSSViewTransformerFunction3D
    acc = LSSViewTransformerFunction3D(synthetic.GRID_CONFIGS["fbocc_shipped"],
                                       (256, 704), 16, accelerate=True)
    got = acc(cam, feat, depth)
    assert torch.equal(got, want)
    idx = acc._index
    moved = [c.clone() for c in cam]
    moved[1] = moved[1] + 3.0
    got2 = acc(moved, feat, depth)        # cached: cam change has no effect
    assert acc._index is idx and torch.equal(got2, want)


def test_sixteen_frame_config_full_size(oracle_cpu):
    """BASELINE.json configs[2]: B = 16 frames x 6 cameras into 16 volumes of
    200x200x16 in ONE plugin call (10.24 M voxels, 3.3 GB of output): index
    bit-exact against the oracle on the whole batch, volumes of three frames
    against the oracle, and frame independence -- the batch index is just the
    top term of the voxel rank (view_transformer.py:573-575, 586-587)."""
    vt, cam, depth, feat = make_case("fbocc_200", 16)
    bev = vt(cam, feat, depth)                                # (B,C,Y,X,Z)
    assert tuple(bev.shape) == (16, 80, 200, 200, 16)
    coor = vt.get_lidar_coor(*cam)
    idx = vt.prepare_index(coor)
    n_kept, n_int = idx.counts.tolist()
    rb, rd, rf, st, ln = oracle_cpu.voxel_prepare(
        coor.cpu().numpy(), vt.grid_lower_bound.numpy(),
        vt.grid_interval.numpy(), vt.grid_size.numpy())
    assert n_kept == len(rb) and n_int == len(st)
    assert np.array_equal(idx.ranks_bev[:n_kept].cpu().numpy(), rb)
    assert np.array_equal(idx.interval_starts[:n_int].cpu().numpy(), st)
    assert np.array_equal(idx.interval_lengths[:n_int].cpu().numpy(), ln)
    for b in (0, 7, 15):
        sl = slice(b, b + 1)
        one = vt([c[sl] for c in cam], feat[sl], depth[sl])
        assert (one[0] - bev[b]).abs().max().item() <= 1e-5
        c1 = vt.get_lidar_coor(*[c[sl] for c in cam]).cpu().numpy()
        i1 = oracle_cpu.voxel_prepare(c1, vt.grid_lower_bound.numpy(),
                                      vt.grid_interval.numpy(),
                                      vt.grid_size.numpy())
        f1 = feat[sl].permute(0, 1, 3, 4, 2).contiguous().cpu().numpy()
        want = oracle_cpu.bev_pool_v2(depth[sl].cpu().numpy(), f1, i1[1],
                                      i1[2], i1[0], (1, 16, 200, 200, 80),
                                      i1[3], i1[4])
        got = bev[b].permute(0, 3, 1, 2).cpu().numpy()          # (C,Z,Y,X)
        np.testing.assert_allclose(got, want[0], rtol=0, atol=ATOL)
