"""Golden fixture k_ref_cuda.npz: outputs of the reference's OWN bev_pool_v2
CUDA kernels (bev_pool_cuda.cu, built into oracle/_ref/ by oracle/Makefile) on
the inputs tests/test_forward_gpu.py builds from seeded synthetic rigs.

Run on a GPU, after oracle/Makefile has built oracle/_ref/:

    python tests/golden/gen_golden_ref_kernel.py [OUT_DIR]

What it records, per test_vs_reference_cuda_kernel case ``<name>``:
  <name>__sha256   SHA-256 of the whole (B,C,Z,Y,X) float32 output of the
                   reference op as shipped (bev_pool.py:15-39, 84-90)
  <name>__idx/val  a seeded sample of that output (flat indices, values):
                   three quarters from the written voxels, the rest from the
                   zero ones
and for test_backward_vs_oracle_and_reference_kernel (bev_pool.cpp:72-102):
  bwd__{depth,feat}_{idx,grad}   a seeded sample of both gradients
The volumes are far above the 1 MB a stored file may have; the hash pins every
bit, the samples say where a mismatch is.
"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_cuda  # noqa: E402
from test_forward_gpu import make_case  # noqa: E402

CASES = ("shipped", "fbocc_200", "unit_128", "fbocc_400")
N_SAMPLE = 1024
N_SAMPLE_GRAD = 4096


def sha256(t):
    return np.frombuffer(hashlib.sha256(
        t.contiguous().cpu().numpy().tobytes()).digest(), np.uint8)


def sample(flat, n, rng):
    nz = np.flatnonzero(flat)
    z = np.flatnonzero(flat == 0)
    k = min(len(nz), n * 3 // 4)
    idx = np.concatenate([rng.choice(nz, k, replace=False),
                          rng.choice(z, min(len(z), n - k), replace=False)])
    return np.sort(idx).astype(np.int64)


def gen_forward(rng, arrays):
    for name in CASES:
        vt, cam, depth, feat = make_case(name, 1)
        coor = vt.get_lidar_coor(*cam)
        rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
        feat_nhwc = feat.permute(0, 1, 3, 4, 2).contiguous()
        shape = vt._bev_feat_shape(depth, feat_nhwc)
        want = ref_cuda.bev_pool_v2(depth, feat_nhwc, rd, rf, rb, shape, st,
                                    ln)
        flat = want.reshape(-1).cpu().numpy()
        idx = sample(flat, N_SAMPLE, rng)
        arrays[f"{name}__sha256"] = sha256(want)
        arrays[f"{name}__idx"] = idx
        arrays[f"{name}__val"] = flat[idx]
        print(f"{name}: {tuple(want.shape)}, {np.count_nonzero(flat)} nonzero")
        del want, flat
        torch.cuda.empty_cache()


def gen_backward(rng, arrays):
    """The inputs of test_backward_vs_oracle_and_reference_kernel, step for
    step (same case, same seeded output gradient)."""
    from fbbev_b200.ops.bev_pool_v2 import _feat_intervals
    dev = "cuda:0"
    vt, cam, depth, feat = make_case("shipped", 1)
    coor = vt.get_lidar_coor(*cam)
    rb, rd, rf, st, ln = vt.voxel_pooling_prepare_v2(coor)
    feat_nhwc = feat.permute(0, 1, 3, 4, 2).contiguous()
    B, Z, Y, X, C = vt._bev_feat_shape(depth, feat_nhwc)
    go = torch.randn((B, C, Z, Y, X), device=dev,
                     generator=torch.Generator(dev).manual_seed(5))
    go_zyxc = go.permute(0, 2, 3, 4, 1).contiguous()
    rf2, rd2, rb2, st2, ln2 = _feat_intervals(rf, rd, rb)
    dg, fg = ref_cuda.bev_pool_v2_grad(go_zyxc, depth, feat_nhwc, rd2, rf2,
                                       rb2, st2, ln2)
    for key, grad in (("depth", dg), ("feat", fg)):
        flat = grad.reshape(-1).cpu().numpy()
        idx = np.sort(rng.choice(flat.size, N_SAMPLE_GRAD, replace=False))
        arrays[f"bwd__{key}_idx"] = idx.astype(np.int64)
        arrays[f"bwd__{key}_grad"] = flat[idx]


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    if not ref_cuda.available():
        raise SystemExit(f"{ref_cuda.LIB_PATH} is missing: build it with "
                         "`make -C oracle ref` where the reference checkout "
                         "is present")
    rng = np.random.default_rng(2024)
    arrays = {}
    gen_forward(rng, arrays)
    gen_backward(rng, arrays)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "k_ref_cuda.npz")
    np.savez_compressed(path, **arrays)
    assert os.path.getsize(path) < 1_000_000, path
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
