"""Generate the committed golden fixtures from the reference's OWN Python.

Run in the build container (needs /root/reference):

    python tests/golden/gen_golden.py

It imports the reference's view-transformation modules through
``tests/golden/ref_import.py`` (mmcv stand-ins, reference files loaded from
/root/reference, nothing copied) and records small seeded input/output pairs as
``tests/golden/*.npz``.  The tests read only the ``.npz`` files, so they run on
the GPU box where the reference checkout does not exist.

What each fixture pins (reference file:line):
  f_*      get_lidar_coor (view_transformer.py:458-498), voxel_pooling_prepare_v2
           (:547-605) and voxel_pooling_v2 glue (:521-545) of
           LSSViewTransformerFunction3D, run on CPU by the reference code itself.
           The bev_pool_v2 CUDA op inside is served by the C oracle (the
           reference has no CPU kernel); its own known-answer test
           (bev_pool.py:145-176) is restated in tests/test_oracle.py.
  b_*      DA_SpatialCrossAttention / DA_MSDeformableAttention / bevformer
           encoder / BackwardProjection forward (spatial_cross_attention_depth.py,
           bevformer_encoder.py, bevformer.py, backward_projection.py), run by
           the reference code with mmcv's `_ext` MSDA op served by the C oracle.
"""
import os
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import ref_import  # noqa: E402
from fbbev_b200 import synthetic  # noqa: E402


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


PART_BYTES = 900_000


def save(name, **arrays):
    """Write ``name.npz``; arrays beyond PART_BYTES go on into
    ``name.part1.npz``, ... so every stored file stays below 1 MB
    (conftest.load_golden merges the parts)."""
    arrays = {k: v for k, v in arrays.items() if v is not None}
    parts, size = [{}], 0
    for k, v in arrays.items():
        if parts[-1] and size + v.nbytes > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += v.nbytes
    for i, part in enumerate(parts):
        path = os.path.join(HERE, name + (f".part{i}" if i else "") + ".npz")
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) < 1_000_000, path
        print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


def gen_forward(ref):
    VT = ref.view_transformer.LSSViewTransformerFunction3D

    def run_case(name, grid_config, input_size, downsample, B, N, C, seed,
                 coor_override=None):
        vt = VT(grid_config=grid_config, input_size=input_size,
                downsample=downsample)
        cam = synthetic.make_cam_params(B, N, input_size=input_size,
                                        jitter=1.0, seed=seed)
        coor = vt.get_lidar_coor(*cam)
        if coor_override is not None:
            coor = coor_override(coor)
        rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
        H, W = input_size[0] // downsample, input_size[1] // downsample
        depth, feat = synthetic.make_depth_feat(B, N, vt.D, H, W, C, seed=seed)
        bev = vt.voxel_pooling_v2(coor, depth, feat)
        save(name,
             grid_x=np.array(grid_config['x'], np.float64),
             grid_y=np.array(grid_config['y'], np.float64),
             grid_z=np.array(grid_config['z'], np.float64),
             grid_depth=np.array(grid_config['depth'], np.float64),
             input_size=np.array(input_size), downsample=np.array(downsample),
             frustum=_np(vt.frustum), grid_size=_np(vt.grid_size),
             grid_interval=_np(vt.grid_interval),
             grid_lower_bound=_np(vt.grid_lower_bound),
             dx=_np(vt.dx), bx=_np(vt.bx), nx=_np(vt.nx),
             rots=_np(cam[0]), trans=_np(cam[1]), intrins=_np(cam[2]),
             post_rots=_np(cam[3]), post_trans=_np(cam[4]), bda=_np(cam[5]),
             coor=_np(coor), ranks_bev=_np(rb), ranks_depth=_np(rd),
             ranks_feat=_np(rf), interval_starts=_np(st),
             interval_lengths=_np(ln), depth=_np(depth), feat=_np(feat),
             bev_feat=_np(bev.contiguous()),
             bev_feat_shape=np.array(bev.shape))

    # scaled-down shipped FB-OCC grid, 2 samples x 6 cameras
    run_case('f_small_6cam',
             dict(x=[-40, 40, 4.0], y=[-40, 40, 4.0], z=[-1, 5.4, 1.6],
                  depth=[2.0, 42.0, 4.0]), (64, 176), 16, B=2, N=6, C=8, seed=3)
    # scaled-down configs[0]: one camera, single-Z BEV
    run_case('f_unit_1cam',
             dict(x=[-51.2, 51.2, 3.2], y=[-51.2, 51.2, 3.2], z=[-5, 3, 8],
                  depth=[1.0, 60.0, 1.0]), (32, 88), 4, B=1, N=1, C=5, seed=5)

    # truncation-toward-zero quirk: coordinates in (-1, 0) are kept in cell 0
    def jitter_box(coor):
        g = torch.Generator().manual_seed(11)
        lo = torch.tensor([-5.0, -5.0, -2.0])
        hi = torch.tensor([5.0, 5.0, 2.0])
        u = torch.rand(coor.shape, generator=g)
        return lo - 1.5 + u * (hi - lo + 3.0)
    run_case('f_negative_trunc',
             dict(x=[-5, 5, 1.0], y=[-5, 5, 1.0], z=[-2, 2, 1.0],
                  depth=[1.0, 5.0, 1.0]), (32, 32), 4, B=2, N=1, C=4, seed=7,
             coor_override=jitter_box)

    # nothing inside the grid -> the reference returns five None + zero volume
    run_case('f_empty',
             dict(x=[-5, 5, 1.0], y=[-5, 5, 1.0], z=[-2, 2, 1.0],
                  depth=[1.0, 5.0, 1.0]), (32, 32), 4, B=1, N=1, C=4, seed=9,
             coor_override=lambda c: c * 0 + 100.0)


def gen_forward_2d(ref):
    """LSSViewTransformerFunction (view_transformer.py:24-311): the 2-D,
    Z-collapsed variant, with and without the cached index
    (``accelerate=True``, :266-283)."""
    VT = ref.view_transformer.LSSViewTransformerFunction

    def run_case(name, grid_config, input_size, downsample, B, N, C, seed):
        cam = synthetic.make_cam_params(B, N, input_size=input_size,
                                        jitter=1.0, seed=seed)
        H, W = input_size[0] // downsample, input_size[1] // downsample
        out = {}
        for acc in (False, True):
            vt = VT(grid_config=grid_config, input_size=input_size,
                    downsample=downsample, accelerate=acc)
            depth, feat = synthetic.make_depth_feat(B, N, vt.D, H, W, C,
                                                    seed=seed)
            out[acc] = vt(cam, feat, depth)
            if acc:     # second call reuses the cached index (initial_flag)
                depth2, feat2 = synthetic.make_depth_feat(B, N, vt.D, H, W, C,
                                                          seed=seed + 50)
                out['second'] = vt(cam, feat2, depth2)
        save(name,
             grid_x=np.array(grid_config['x'], np.float64),
             grid_y=np.array(grid_config['y'], np.float64),
             grid_z=np.array(grid_config['z'], np.float64),
             grid_depth=np.array(grid_config['depth'], np.float64),
             input_size=np.array(input_size), downsample=np.array(downsample),
             rots=_np(cam[0]), trans=_np(cam[1]), intrins=_np(cam[2]),
             post_rots=_np(cam[3]), post_trans=_np(cam[4]), bda=_np(cam[5]),
             depth=_np(depth), feat=_np(feat), depth2=_np(depth2),
             feat2=_np(feat2), bev=_np(out[False]), bev_acc=_np(out[True]),
             bev_acc_second=_np(out['second']))

    # BEVDet-style single-Z grid (accelerate squeezes Z, :283)
    run_case('f2d_z1_6cam',
             dict(x=[-40, 40, 4.0], y=[-40, 40, 4.0], z=[-5, 3, 8],
                  depth=[2.0, 42.0, 4.0]), (64, 176), 16, B=2, N=6, C=8,
             seed=13)
    # several Z slices: Z collapsed into channels (:191)
    run_case('f2d_z4_6cam',
             dict(x=[-40, 40, 4.0], y=[-40, 40, 4.0], z=[-1, 5.4, 1.6],
                  depth=[2.0, 42.0, 4.0]), (64, 176), 16, B=1, N=6, C=8,
             seed=14)


def load_fuse_history():
    """FBOCC.fuse_history / generate_grid / generate_forward_transformation_matrix
    (mmdet3d/models/fbbev/detectors/fbocc.py:37-42, 170-205, 207-319) compiled
    from the reference file WHERE IT LIES: the module itself imports spconv,
    cv2, mmdet ..., so the three function definitions are taken out of its AST
    (decorators dropped: @force_fp32 is an fp32 cast) and executed as they are.
    Nothing is copied into this repository."""
    import ast
    import torch.nn as nn
    import torch.nn.functional as F
    path = os.path.join(ref_import.REF, 'mmdet3d', 'models', 'fbbev',
                        'detectors', 'fbocc.py')
    tree = ast.parse(open(path).read())
    want = {'generate_forward_transformation_matrix', 'generate_grid',
            'fuse_history'}
    nodes = [n for n in ast.walk(tree)
             if isinstance(n, ast.FunctionDef) and n.name in want]
    assert {n.name for n in nodes} == want
    for n in nodes:
        n.decorator_list = []
    mod = ast.Module(body=nodes, type_ignores=[])
    ns = {'torch': torch, 'F': F, 'nn': nn}
    exec(compile(mod, path, 'exec'), ns)
    return ns


def gen_fuse_history():
    """t_fuse_history.npz: four consecutive fuse_history calls of the
    reference (first call, a normal step, a step where one sample starts a new
    sequence, another normal step) on a small voxel grid."""
    import types
    import torch.nn as nn
    from fbbev_b200.view_transformation.forward_projection import gen_dx_bx
    ns = load_fuse_history()
    C, T, Z, H, W, n = 4, 3, 3, 7, 6, 2
    grid = dict(x=[-6, 6, 2.0], y=[-7, 7, 2.0], z=[-1, 5, 2.0])
    dx, bx, nx = gen_dx_bx(grid['x'], grid['y'], grid['z'])
    torch.manual_seed(77)
    time_conv = nn.Sequential(nn.Conv3d(C + 1, C, 1), nn.SyncBatchNorm(C),
                              nn.ReLU(inplace=True))
    cat_conv = nn.Sequential(nn.Conv3d(C * (T + 1), C, 1), nn.SyncBatchNorm(C),
                             nn.ReLU(inplace=True))
    for seq in (time_conv, cat_conv):
        bn = seq[1]
        bn.running_mean.uniform_(-0.2, 0.2)
        bn.running_var.uniform_(0.5, 1.5)
        bn.weight.data.uniform_(0.5, 1.5)
        bn.bias.data.uniform_(-0.2, 0.2)
        seq.eval()
    me = types.SimpleNamespace(
        history_bev=None, history_seq_ids=None, history_forward_augs=None,
        history_sweep_time=None, history_cat_num=T, history_cam_sweep_freq=0.5,
        interpolation_mode='bilinear', single_bev_num_channels=C,
        do_history=True, history_keyframe_time_conv=time_conv,
        history_keyframe_cat_conv=cat_conv,
        forward_projection=types.SimpleNamespace(dx=dx, bx=bx, nx=nx))
    me.generate_grid = lambda *a, **k: ns['generate_grid'](me, *a, **k)
    g = torch.Generator().manual_seed(78)

    def rigid(scale):
        a = (torch.rand((), generator=g) - 0.5) * 0.3 * scale
        m = torch.eye(4)
        m[0, 0], m[0, 1], m[1, 0], m[1, 1] = a.cos(), -a.sin(), a.sin(), a.cos()
        m[:3, 3] = (torch.rand(3, generator=g) - 0.5) * \
            torch.tensor([3.0, 3.0, 0.5]) * scale
        return m

    arrays = dict(C=np.array(C), T=np.array(T), dx=_np(dx), bx=_np(bx),
                  **{'sd_time::' + k: _np(v)
                     for k, v in time_conv.state_dict().items()},
                  **{'sd_cat::' + k: _np(v)
                     for k, v in cat_conv.state_dict().items()})
    seq_ids = [[5, 9], [5, 9], [5, 11], [5, 11]]
    starts = [[True, True], [False, False], [False, True], [False, False]]
    with torch.no_grad():
        for step in range(4):
            curr = torch.randn(n, C, H, W, Z, generator=g)
            bda = torch.stack([rigid(1.0)[:3, :3] *
                               (1.0 if i else -1.0) ** step for i in range(n)])
            metas = [dict(sequence_group_idx=seq_ids[step][i],
                          start_of_sequence=starts[step][i],
                          curr_to_prev_ego_rt=rigid(1.0)) for i in range(n)]
            out = ns['fuse_history'](me, curr, metas, bda)
            arrays[f'curr{step}'] = _np(curr)
            arrays[f'bda{step}'] = _np(bda)
            arrays[f'c2p{step}'] = _np(torch.stack(
                [m['curr_to_prev_ego_rt'] for m in metas]))
            arrays[f'seq{step}'] = np.array(seq_ids[step])
            arrays[f'start{step}'] = np.array(starts[step])
            arrays[f'out{step}'] = _np(out)
            # copies: the reference updates its state tensors in place later
            arrays[f'history{step}'] = _np(me.history_bev).copy()
            arrays[f'sweep{step}'] = _np(me.history_sweep_time).copy()
    save('t_fuse_history', **arrays)


def main():
    if os.environ.get("GOLDEN_ONLY", "") == "fuse":
        ref_import.install_stubs()
        gen_fuse_history()
        return
    if os.environ.get("GOLDEN_ONLY", "") == "lineage":
        import gen_golden_lineage
        gen_golden_lineage.gen_lineage(save)
        return
    ref = ref_import.load_reference()
    torch.manual_seed(0)
    if os.environ.get("GOLDEN_ONLY", "") == "f2d":
        gen_forward_2d(ref)
        return
    if os.environ.get("GOLDEN_ONLY", "") == "backward":
        import gen_golden_backward
        gen_golden_backward.gen_backward(ref, save)
        return
    gen_forward(ref)
    gen_forward_2d(ref)
    gen_fuse_history()
    try:
        import gen_golden_backward
        gen_golden_backward.gen_backward(ref, save)
    except ImportError:
        print("gen_golden_backward.py not present yet; forward fixtures only")


if __name__ == "__main__":
    main()
