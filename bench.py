#!/usr/bin/env python
"""bench.py -- headline benchmark of the forward-backward view transformation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--config fbocc200|unit|frames16|bwd_only|large]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic input; every
timed pass runs K of them.  The inputs are seeded, so the same arguments give
the same inputs on every run, and `--dump-outputs DIR` writes what the last
timed step returned (rank 0) as DIR/<name>.npy: two builds of the project
can then be compared output for output.  The
default workload is BASELINE.json configs[1] (FB-OCC R50 single frame: 6
cameras 256x704, feature map 16x44, D = 80 depth bins, C = 80, 200x200x16 voxel
grid, 200x200 BEV queries, 8 heads, 1 level, 8 points, 4 Z anchors), one frame
per GPU:

    F  LSSViewTransformerFunction3D.forward(cam_params, context, depth)
         = get_lidar_coor + voxel_pooling_prepare_v2 + bev_pool_v2
    B  BackwardProjection.forward([context], lss_bev, cam_params, depth)
         = embedding/pos-enc + point_sampling + self-attn + depth-aware
           spatial cross-attention + LayerNorms + FFN

i.e. every row of SURVEY.md section 8(a).  Metric: BEV voxels/s =
frames * Z*Y*X / step time (whole job, all ranks).  `--config` selects the
other BASELINE.json configs (unit = [0], frames16 = [2], bwd_only = [3],
large = [4]); the headline stays configs[1].

Launch contract: `python bench.py --gpus 1 ...` or, for N > 1,
`python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...`
(one rank per GPU, NCCL).  Frames are independent, so ranks shard frames and no
collective sits on the data path (weak scaling: one frame per GPU).  Every
default run also reports BASELINE.json configs[2] as the `frames16` block: 16
frames in total sharded over the N ranks (strong scaling), with and without the
NCCL all-gather of the refined BEV inside the timed step.

`--impl reference` times the reference algorithm's CPU implementation (the
oracle port: the reference ships no CPU kernel for this path) on the host
cores, on the same config.  Rank 0 only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark leaves the tree as it found it (it may be read-only)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

# --------------------------------------------------------------- workloads --
# One entry per BASELINE.json config (SURVEY.md section 8d gives the shapes).
CONFIGS = {
    "unit": dict(
        index=0, workload="bev_pool_v2_unit_1cam_64x176_D59_bev128x128",
        grid="unit_128", input_size=(256, 704), downsample=4, n_cams=1, C=80,
        frames=1, do_f=True, do_b=False),
    "fbocc200": dict(
        index=1, workload="fbocc_r50_single_frame_6cam_256x704_voxel200x200x16",
        grid="fbocc_200", input_size=(256, 704), downsample=16, n_cams=6, C=80,
        bev=(200, 200), dbound=[2.0, 42.0, 0.5], z_step=1.6, frames=1,
        do_f=True, do_b=True),
    "frames16": dict(
        index=2, workload="fbocc_r50_16frame_6x16cam_voxel200x200x16_sharded",
        grid="fbocc_200", input_size=(256, 704), downsample=16, n_cams=6, C=80,
        bev=(200, 200), dbound=[2.0, 42.0, 0.5], z_step=1.6, frames_total=16,
        do_f=True, do_b=True),
    "bwd_only": dict(
        index=3, workload="fbbev_backward_only_200x200q_4scale_8head_e256",
        grid=None, input_size=(512, 1408), downsample=16, n_cams=6, C=256,
        bev=(200, 200), dbound=[2.0, 42.0, 0.5], z_step=1.6, frames=1,
        levels=[(32, 88), (16, 44), (8, 22), (4, 11)], do_f=False, do_b=True),
    "large": dict(
        index=4, workload="fbocc_large_6cam_512x1408_D118_voxel400x400x32",
        grid="fbocc_400", input_size=(512, 1408), downsample=16, n_cams=6,
        C=80, bev=(200, 200), dbound=[1.0, 60.0, 0.5], z_step=1.6, frames=1,
        do_f=True, do_b=True),
}
PC_RANGE = [-40, -40, -1.0, 40, 40, 5.4]


def frames_of(name, world):
    """(frames per rank, frames per step over all ranks, scaling)"""
    c = CONFIGS[name]
    if "frames_total" in c:
        tot = c["frames_total"]
        if tot % world:
            raise SystemExit(f"--config {name}: {tot} frames do not shard "
                             f"evenly over {world} ranks")
        return tot // world, tot, "strong"
    return c["frames"], c["frames"] * world, "weak"


def metric_of(name):
    if CONFIGS[name]["do_f"]:
        return "bev_voxels_per_sec", "voxels/s"
    return "bev_queries_per_sec", "queries/s"


def config_dict(name, world):
    """The `config` object of the JSON line -- IDENTICAL in both arms."""
    c = CONFIGS[name]
    per_rank, total, _ = frames_of(name, world)
    parts = []
    if c["do_f"]:
        parts.append("LSSViewTransformerFunction3D.forward")
    if c["do_b"]:
        parts.append("BackwardProjection.forward")
    return {"workload": c["workload"], "baseline_config_index": c["index"],
            "frames_per_step": total, "frames_per_gpu": per_rank,
            "step": " + ".join(parts),
            "l2": "flushed between timed steps (256 MiB memset)",
            "parallelism": f"dp{world}: frames sharded over ranks, no "
                           "data-path collective"}


def bp_config(c):
    E = c["C"]
    bev_h, bev_w = c["bev"]
    n_levels = len(c.get("levels") or [0])
    grid_bev = dict(x=[-40, 40, 80.0 / bev_w], y=[-40, 40, 80.0 / bev_h],
                    z=[-1, 5.4, c["z_step"]])
    return dict(
        type='BackwardProjection', bev_h=bev_h, bev_w=bev_w, in_channels=E,
        out_channels=E, pc_range=PC_RANGE,
        transformer=dict(
            type='BEVFormer', use_cams_embeds=False, embed_dims=E,
            encoder=dict(
                type='bevformer_encoder', num_layers=1, pc_range=PC_RANGE,
                grid_config=grid_bev,
                data_config=dict(input_size=c["input_size"]),
                return_intermediate=False,
                transformerlayers=dict(
                    type='BEVFormerEncoderLayer',
                    attn_cfgs=[
                        dict(type='MultiScaleDeformableAttention',
                             embed_dims=E, dropout=0.0, num_levels=1),
                        dict(type='DA_SpatialCrossAttention',
                             pc_range=PC_RANGE, dbound=c["dbound"],
                             dropout=0.0,
                             deformable_attention=dict(
                                 type='DA_MSDeformableAttention',
                                 embed_dims=E, num_points=8,
                                 num_levels=n_levels),
                             embed_dims=E)],
                    ffn_cfgs=dict(type='FFN', embed_dims=E,
                                  feedforward_channels=4 * E, ffn_drop=0.0,
                                  act_cfg=dict(type='ReLU', inplace=True)),
                    feedforward_channels=4 * E, ffn_dropout=0.0,
                    operation_order=('self_attn', 'norm', 'cross_attn', 'norm',
                                     'ffn', 'norm')))),
        positional_encoding=dict(type='CustormLearnedPositionalEncoding',
                                 num_feats=E // 2, row_num_embed=bev_h,
                                 col_num_embed=bev_w))


def _pin(t, device):
    return t.pin_memory() if device != "cpu" else t


class Workload:
    """Modules + `frames` frames of seeded synthetic inputs on `device`."""

    def __init__(self, name, device, seed, frames):
        from fbbev_b200 import synthetic
        from fbbev_b200.registry import build_head, build_neck
        c = CONFIGS[name]
        self.name, self.c = name, c
        self.device = device
        self.frames = frames
        H, W = (s // c["downsample"] for s in c["input_size"])
        self.levels = c.get("levels") or [(H, W)]
        self.vt = self.bp = None
        self.voxels_per_frame = 0
        if c["do_f"]:
            self.vt = build_neck(dict(
                type='LSSViewTransformerFunction3D',
                grid_config=synthetic.GRID_CONFIGS[c["grid"]],
                input_size=c["input_size"], downsample=c["downsample"]))
            gs = [int(v) for v in self.vt.grid_size]
            self.voxels_per_frame = gs[0] * gs[1] * gs[2]
            self.D = self.vt.D
        else:
            d0, d1, dd = c["dbound"]
            self.D = int(round((d1 - d0) / dd))
        if c["do_b"]:
            torch.manual_seed(1234)  # identical random-init weights on all ranks
            bp = build_head(bp_config(c))
            bp.init_weights()
            g = torch.Generator().manual_seed(4321)
            with torch.no_grad():
                for p in bp.parameters():  # non-trivial offsets / weights
                    p.add_(torch.randn(p.shape, generator=g) * 0.02)
            self.bp = bp.to(device).eval()
        self.units_per_frame = self.voxels_per_frame if c["do_f"] else \
            c["bev"][0] * c["bev"][1]
        cam = synthetic.make_cam_params(frames, c["n_cams"], c["input_size"],
                                        jitter=1.0, seed=seed)
        H0, W0 = self.levels[0]
        depth, feat = synthetic.make_depth_feat(frames, c["n_cams"], self.D,
                                                H0, W0, c["C"], seed=seed)
        g = torch.Generator().manual_seed(seed + 7)
        more = [torch.randn(frames, c["n_cams"], c["C"], h, w, generator=g)
                for h, w in self.levels[1:]]
        host = dict(cam=[_pin(t, device) for t in cam],
                    depth=_pin(depth, device), feat=_pin(feat, device),
                    more=[_pin(t, device) for t in more])
        if c["do_b"]:
            lss = torch.randn(frames, c["C"], *c["bev"], generator=g) * 0.1
            host["lss"] = _pin(lss, device)
        self.host = host
        self.out_buffer = None  # optional gather slot for the refined BEV
        self.to_device()

    def _host_list(self):
        h = self.host
        return list(h["cam"]) + [h["depth"], h["feat"]] + list(h["more"]) + \
            ([h["lss"]] if "lss" in h else [])

    def to_device(self):
        self._dev = [t.to(self.device, non_blocking=True)
                     for t in self._host_list()]
        self._unpack()

    def _unpack(self):
        d = self._dev
        n_more = len(self.host["more"])
        self.cam = d[:6]
        self.depth, self.feat = d[6], d[7]
        self.more = d[8:8 + n_more]
        self.lss = d[8 + n_more] if "lss" in self.host else None

    def to_device_inplace(self):
        """H2D into the buffers the captured graph reads."""
        for d, s in zip(self._dev, self._host_list()):
            d.copy_(s, non_blocking=True)

    def h2d_bytes(self):
        return int(sum(t.numel() * t.element_size()
                       for t in self._host_list()))

    @torch.no_grad()
    def step(self):
        """-> the step's results, also kept as ``last_out`` (under a CUDA
        graph: the graph's output tensors, which every replay rewrites)."""
        outs = []
        if self.vt is not None:
            outs.append(self.vt(self.cam, self.feat, self.depth))  # (B,C,Y,X,Z)
        if self.bp is not None:
            outs.append(self.bp([self.feat] + list(self.more), None,
                                lss_bev=self.lss, cam_params=self.cam,
                                pred_img_depth=self.depth,
                                out=self.out_buffer))
        self.last_out = tuple(outs)
        return self.last_out

    def out_names(self):
        return (["bev_volume"] if self.vt is not None else []) + \
            (["bev_refined"] if self.bp is not None else [])

    def capture(self, after=None):
        """Capture one step (the plugin forwards, plus `after()` when given --
        the NCCL gather of the with-exchange line) into a CUDA graph: the path
        has no host synchronisation, so the launches of a step replay as one
        submission.  Inputs are read from the same device buffers
        (``to_device_inplace`` copies into them in place)."""
        def body():
            out = self.step()
            if after is not None:
                after()
            return out
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.graph_out = body()
        torch.cuda.synchronize()
        return self.graph


def e2e_streamed(w, steps, barrier, keep=None):
    """K end-to-end steps as a pipeline; returns ms per step (device clock).
    ``keep``: indices of the step's outputs that are copied to the host (None:
    all of them).

    compute stream : wait inputs(i) -> graph replay -> copy results into
                     staging[i % 2] (after the D2H of step i-2 released it)
    H2D stream     : inputs of step i+1 into the graph's input buffers once
                     step i has finished reading them
    D2H stream     : staging[i % 2] -> pinned host[i % 2]
    """
    s_c = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    g_out = list(w.graph_out) if keep is None else \
        [w.graph_out[i] for i in keep]
    stage = [[torch.empty_like(t) for t in g_out] for _ in range(2)]
    host = [[torch.empty(t.shape, dtype=t.dtype).pin_memory()
             for t in g_out] for _ in range(2)]

    def run(n):
        h2d_done = [torch.cuda.Event() for _ in range(n + 1)]
        comp_done = [torch.cuda.Event() for _ in range(n)]
        ready = [torch.cuda.Event() for _ in range(n)]
        d2h_done = [torch.cuda.Event() for _ in range(n)]
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record(s_c)
        s_in.wait_stream(s_c)
        with torch.cuda.stream(s_in):
            w.to_device_inplace()
            h2d_done[0].record(s_in)
        for i in range(n):
            s_c.wait_event(h2d_done[i])
            w.graph.replay()
            comp_done[i].record(s_c)
            with torch.cuda.stream(s_in):          # inputs of the next step
                s_in.wait_event(comp_done[i])
                w.to_device_inplace()
                h2d_done[i + 1].record(s_in)
            if i >= 2:
                s_c.wait_event(d2h_done[i - 2])
            for d, r in zip(stage[i % 2], g_out):
                d.copy_(r, non_blocking=True)
            ready[i].record(s_c)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ready[i])
                for h, d in zip(host[i % 2], stage[i % 2]):
                    h.copy_(d, non_blocking=True)
                d2h_done[i].record(s_out)
        s_c.wait_stream(s_out)
        s_c.wait_stream(s_in)
        t1.record(s_c)
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / n

    run(3)
    barrier()
    ms = run(steps)
    barrier()
    # the last step's results really are on the host
    assert torch.equal(host[(steps - 1) % 2][-1], g_out[-1].cpu())
    return ms


# ------------------------------------------------------------------ clocks --
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,"
         "clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader",
                 "-lms", "20", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                 "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1].split()[0]))
                mx.append(float(r[2].split()[0]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(local):
    """Pin this rank's host threads to the cores next to its GPU (sysfs
    `local_cpulist` of the device) BEFORE any pinned staging buffer is
    allocated, so first-touch places them on the GPU's NUMA node: with 8 ranks
    the per-rank 218 MB D2H otherwise crosses the socket interconnect."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local),
                      "pci_domain_id", 0)
        dev_id = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/"
        with open(path + "local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        with open(path + "numa_node") as f:
            node = int(f.read().strip())
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as ex:  # sysfs layout differs: run unpinned
        return {"numa_node": None, "error": str(ex)[:80]}


# ----------------------------------------------------- per-kernel roofline --
def _call_key(name, a, ctx):
    """Group C-ABI calls into 'kernels' and give their algorithmic bytes.
    Argument positions follow include/fbbev_b200.h."""
    if name == "fbbev_linear_fwd":
        m, k, n = a[8], a[9], a[10]
        extra = m * n if a[4] is not None else 0
        tag = "+res" if a[4] is not None else ""
        tag += "+relu" if a[11] else ""
        tag += "+ln" if a[6] is not None else ""
        return (f"linear_tf32 {m}x{k}->{n}{tag}",
                4 * (m * k + k * n + m * n + extra))
    if name == "fbbev_linear_fwd_split":
        m, k, n = a[6], a[7], a[8]
        add = m * k if a[2] is not None else 0
        tag = ", x+pos" if a[2] is not None else ""
        return (f"linear_tf32 {m}x{k}->{n} (two outputs{tag})",
                4 * (m * k + add + k * n + m * n))
    if name == "fbbev_ffn_fwd":
        m, e, h = a[10], a[11], a[12]
        res = m * e if a[6] is not None else 0
        # x in, y out, residual, both weight matrices (the hidden m x h tile
        # never leaves the SM)
        return (f"ffn_tf32 {m}x{e}->{h}->{e}+res+ln",
                4 * (2 * m * e + res + 2 * e * h))
    if name == "fbbev_msda_fused_fwd":
        bs, n_value, heads, ch, levels, nq, points = a[6:13]
        E = heads * ch
        return (f"msda_fused_fwd ch{ch} L{levels} P{points}",
                4 * (bs * n_value * E + bs * nq * levels * 2 +
                     bs * nq * heads * levels * points * 3 + bs * nq * E))
    if name == "fbbev_da_sca_fwd":
        bs, n_cams, nq, n_value, heads, ch, levels, points, Z, DC = a[10:20]
        E = heads * ch
        # value + depth maps + per-(cam, query, anchor) ref uv / depth / mask +
        # offsets + logits + out (SURVEY.md section 8d, fused boundary)
        return (f"da_sca_fwd ch{ch} L{levels} P{points} Z{Z}",
                4 * (bs * n_cams * n_value * E) + 4 * ctx["depth_elems"] +
                n_cams * bs * nq * Z * 13 +
                4 * (bs * nq * heads * levels * points * 3 + bs * nq * E))
    return name.replace("fbbev_", ""), None


def kernel_table(records, step_us, steps, extra_bytes, ctx):
    """records of a KernelTimer over `steps` steps -> per-kernel rows."""
    groups = {}
    for name, a, e0, e1 in records:
        key, nbytes = _call_key(name, a, ctx)
        if nbytes is None:
            nbytes = extra_bytes.get(key)
        g = groups.setdefault(key, dict(kernel=key, calls=0, us=0.0, bytes=0,
                                        has_bytes=True))
        g["calls"] += 1
        g["us"] += e0.elapsed_time(e1) * 1e3
        if nbytes is None:
            g["has_bytes"] = False
        else:
            g["bytes"] += nbytes
    rows = []
    for g in groups.values():
        us = g["us"] / steps
        row = {"kernel": g["kernel"], "launch_calls_per_step": g["calls"] / steps,
               "us_per_step": us, "share_of_step": us / step_us}
        if g["has_bytes"] and g["us"] > 0:
            row["algorithmic_bytes_per_step"] = int(g["bytes"] / steps)
            row["achieved_gbs"] = g["bytes"] / (g["us"] * 1e-6) / 1e9
        rows.append(row)
    rows.sort(key=lambda r: -r["us_per_step"])
    return rows


# ------------------------------------------------------------ CPU baseline --
class CpuReference:
    """The reference algorithm on the host cores (oracle port).

    F: voxel_pooling_prepare_v2 (C, single thread) + bev_pool_v2 as shipped
       (zero-fill + interval kernel + permute; C, OpenMP over intervals).
    B: BackwardProjection with the reference's re-batching cross-attention
       algorithm (spatial_cross_attention_depth.py:156-216) and MSDA through the
       C oracle; dense layers through torch CPU.
    Geometry through torch CPU ops, as the reference does."""

    def __init__(self, w_cpu):
        from oracle import backward_ref, cpu
        self.cpu = cpu
        self.backward_ref = backward_ref
        self.w = w_cpu
        # all host cores this process may use (torchrun exports
        # OMP_NUM_THREADS=1, which would make the baseline single-threaded)
        try:
            n_cores = len(os.sched_getaffinity(0))
        except AttributeError:
            n_cores = os.cpu_count() or 1
        self._n_cores = n_cores
        cpu.set_num_threads(n_cores)
        self.threads = cpu.num_threads()
        torch.set_num_threads(self.threads)
        if w_cpu.vt is not None:
            gs = [int(v) for v in w_cpu.vt.grid_size]
            self.shape = (w_cpu.frames, gs[2], gs[1], gs[0], w_cpu.c["C"])
            n = int(np.prod(self.shape))
            self.scratch = np.empty(n, np.float32)
            self.out = np.empty((w_cpu.frames, w_cpu.c["C"], gs[2], gs[1],
                                 gs[0]), np.float32)

    def calibrate(self):
        """Pick the thread count the CPU arm is fastest with: all logical
        cores is not it on a 2-way SMT host (measured: 3.5 s per step with 128
        threads against ~0.5 s with 64 on the same box)."""
        best = None
        for n in sorted({self._n_cores, max(1, self._n_cores // 2),
                         max(1, self._n_cores // 4)}, reverse=True):
            self.cpu.set_num_threads(n)
            torch.set_num_threads(n)
            self.step()
            t0 = time.perf_counter()
            self.step()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, n)
        self.threads = best[1]
        self.cpu.set_num_threads(self.threads)
        torch.set_num_threads(self.threads)
        return self.threads

    @torch.no_grad()
    def step(self):
        w = self.w
        out = []
        if w.vt is not None:
            coor = w.vt.get_lidar_coor(*w.cam)
            rb, rd, rf, st, ln = self.cpu.voxel_prepare(
                coor.numpy(), w.vt.grid_lower_bound.numpy(),
                w.vt.grid_interval.numpy(), w.vt.grid_size.numpy())
            feat_nhwc = w.feat.permute(0, 1, 3, 4, 2).contiguous().numpy()
            self.cpu.bev_pool_v2(w.depth.numpy(), feat_nhwc, rd, rf, rb,
                                 self.shape, st, ln, scratch=self.scratch,
                                 out=self.out)
            out.append(self.out)
        if w.bp is not None:
            out.append(self.backward_ref.backward_projection_cpu(
                w.bp, [w.feat] + list(w.more), w.lss, w.cam, w.depth))
        return out


def cpu_sample_note(w):
    parts = []
    if w.vt is not None:
        parts.append("geometry + prepare + bev_pool_v2")
    if w.bp is not None:
        parts.append("BackwardProjection")
    return f"{w.frames} frame(s): " + " + ".join(parts)


# --------------------------------------------------------------------- main --
def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import torch.distributed as dist
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        dist.init_process_group(backend, rank=rank, world_size=world)
    return world, rank, local


def run_reference(args, world, rank):
    """--impl reference: CPU implementation of the same step, rank 0 only."""
    if rank != 0:
        return
    metric, unit = metric_of(args.config)
    w = Workload(args.config, "cpu", seed=0, frames=1)   # bounded sample
    ref = CpuReference(w)
    ref.calibrate()
    for _ in range(args.warmup):
        ref.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.step()
    dt = (time.perf_counter() - t0) / args.steps
    value = w.units_per_frame / dt
    _, _, scaling = frames_of(args.config, world)
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.config, world),
        "cpu_baseline": {"value": value, "unit": unit, "cores": ref.threads,
                         "cores_available": ref._n_cores, "kind": "port",
                         "sample": "each step = " + cpu_sample_note(w) +
                                   " of the workload (throughput per frame is "
                                   "independent of the frame count on the CPU)"},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "details": {"note": "reference algorithm on host cores (CPU port: the "
                            "reference has no CPU kernel for this path)"},
    }
    print(json.dumps(line))


def timed_steps(fn, steps, flush, barrier):
    """K steps bracketed by CUDA events, L2 flushed before each; mean ms."""
    events = []
    barrier()
    for _ in range(steps):
        flush.zero_()
        s = torch.cuda.Event(enable_timing=True)
        e = torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        events.append((s, e))
    barrier()
    return sum(s.elapsed_time(e) for s, e in events) / steps


DUMP_BYTES = 60 << 20


def dump_outputs(outs, names, out_dir):
    """Write each result as out_dir/<name>.npy (float32), DUMP_BYTES in all.
    Smaller results are written whole and first; a result beyond what is left
    of the budget is written as the elements at flat indices drawn by a
    generator seeded with 0 (the same on every run), as <name>_sample.npy."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES // 4
    order = sorted(range(len(outs)), key=lambda i: outs[i].numel())
    for k, i in enumerate(order):
        t, name = outs[i].detach(), names[i]
        cap = left // (len(outs) - k)
        if t.numel() > cap:
            g = torch.Generator().manual_seed(0)
            idx = torch.randint(t.numel(), (cap,), generator=g)
            t, name = t.reshape(-1)[idx.to(t.device)], name + "_sample"
        np.save(os.path.join(out_dir, name + ".npy"),
                t.float().cpu().numpy())
        left -= t.numel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="fbocc200", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true")
    ap.add_argument("--no-frames16", action="store_true",
                    help="skip the configs[2] block of the default run")
    ap.add_argument("--no-graph", action="store_true",
                    help="time eager plugin calls instead of a CUDA graph "
                         "replay of them")
    ap.add_argument("--kernels-only", action="store_true",
                    help="tuning aid: print the per-kernel table of the eager "
                         "pass and stop")
    ap.add_argument("--eager-only", action="store_true",
                    help="profiling aid: stop after the eager pass (what ncu "
                         "captures) and print only its numbers")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the "
                         "last one as DIR/<name>.npy (rank 0; at most 64 MB "
                         "in all, a larger result as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.kernels_only
                              or args.eager_only):
        ap.error("--dump-outputs writes the results of the headline pass: "
                 "not with --impl reference, --kernels-only or --eager-only")
    if args.impl == "reference":
        # CPU arm: rank 0 alone works, the other ranks of a torchrun launch
        # exit at once; no process group is needed
        run_reference(args, int(os.environ.get("WORLD_SIZE", "1")),
                      int(os.environ.get("RANK", "0")))
        return
    world, rank, local = dist_setup(args.gpus)

    assert torch.cuda.is_available(), "bench.py --impl b200 needs a CUDA device"
    import torch.distributed as dist
    from fbbev_b200 import _lib
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    numa = bind_to_gpu_numa(local)
    L = _lib.lib()  # fails loudly if the CUDA library is missing
    metric, unit = metric_of(args.config)
    per_rank, total_frames, scaling = frames_of(args.config, world)
    w = Workload(args.config, dev, seed=rank, frames=per_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        w.step()
    barrier()

    # ---- eager pass: K steps through the plugin calls, L2 flushed between
    # steps --------------------------------------------------------------------
    launches0 = L.fbbev_debug_launch_count()
    eager_ms = timed_steps(w.step, args.steps, flush, barrier)
    launches = (L.fbbev_debug_launch_count() - launches0) / args.steps

    # ---- per-kernel pass: every C-ABI launch bracketed by CUDA events.  A
    # spin kernel keeps the GPU busy while the step's launches queue up, so the
    # intervals are device execution back to back (as in the graph replay), not
    # host launch gaps ---------------------------------------------------------
    ksteps = args.steps
    with _lib.KernelTimer() as kt:
        for _ in range(ksteps):
            flush.zero_()
            torch.cuda._sleep(6_000_000)
            w.step()
        torch.cuda.synchronize()
    krecords = kt.records
    if args.kernels_only:
        if rank == 0:
            rows = kernel_table(krecords, eager_ms * 1e3, ksteps, {},
                                {"depth_elems": w.depth.numel()})
            print(json.dumps({"eager_ms_per_step": eager_ms, "kernels": [
                {"kernel": r["kernel"], "us": round(r["us_per_step"], 1)}
                for r in rows]}))
        if world > 1:
            dist.destroy_process_group()
        return
    if args.eager_only:
        if rank == 0:
            print(json.dumps({"eager_ms_per_step": eager_ms,
                              "gpu_launches": launches}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- headline pass: the same K steps as CUDA-graph replays --------------
    use_graph = not args.no_graph
    if use_graph:
        try:
            w.capture()
            for _ in range(warm):
                w.graph.replay()
        except Exception as ex:  # capture unsupported -> eager numbers stand
            use_graph = False
            print(f"[bench] CUDA graph capture failed: {ex}", file=sys.stderr)
    run_step = w.graph.replay if use_graph else w.step
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    wall0 = time.perf_counter()
    step_ms = timed_steps(run_step, args.steps, flush, barrier)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(w.last_out, w.out_names(), args.dump_outputs)

    # ---- end to end: pinned host inputs -> plugin calls -> host results ----
    outs = w.step()
    host_out = [torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in outs]
    e2e_steps = args.steps

    def e2e_step():
        if use_graph:
            w.to_device_inplace()                       # H2D of every input
            w.graph.replay()
            res = w.graph_out
        else:
            w.to_device()
            res = w.step()
        for h, r in zip(host_out, res):                 # D2H of every result
            h.copy_(r, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    for _ in range(2):
        e2e_step()
    e2e_latency_ms = timed_steps(e2e_step, e2e_steps, flush, barrier)
    e2e_ms = e2e_latency_ms
    e2e_mode = "one step at a time (copy in, compute, copy out)"
    d2h = int(sum(h.numel() * 4 for h in host_out))
    h2d = w.h2d_bytes()

    # the same K steps as a stream: three CUDA streams, step i's results leave
    # over PCIe while step i+1 computes and step i+2's inputs arrive.  Every
    # step still copies all of its inputs in and all of its results out.
    if use_graph:
        try:
            e2e_ms = e2e_streamed(w, e2e_steps, barrier)
            e2e_mode = ("streamed: H2D / compute / D2H of consecutive steps "
                        "overlap on three streams (results double-buffered; "
                        "no L2 flush, the results of a step exceed L2)")
        except Exception as ex:
            print(f"[bench] streamed e2e failed: {ex}", file=sys.stderr)

    # the same pipeline when the consumer of the volume is on the GPU (as in the
    # detector: fuse_history and the occupancy head read it there) and only the
    # refined BEV -- BackwardProjection's output -- goes back to the host
    e2e_small_ms, e2e_small_d2h = 0.0, 0
    if use_graph and len(w.graph_out) > 1:
        try:
            e2e_small_ms = e2e_streamed(w, e2e_steps, barrier,
                                        keep=[len(w.graph_out) - 1])
            e2e_small_d2h = int(w.graph_out[-1].numel() * 4)
        except Exception as ex:
            e2e_small_ms = 0.0
            print(f"[bench] refined-only e2e failed: {ex}", file=sys.stderr)

    # ---- max over ranks ----------------------------------------------------
    t = torch.tensor([step_ms, e2e_ms, eager_ms, e2e_latency_ms,
                      e2e_small_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms, e2e_ms, eager_ms, e2e_latency_ms, e2e_small_ms = (
        float(v) for v in t.tolist())

    extra = {}
    # ---- BASELINE.json configs[2]: 16 frames sharded over the ranks ---------
    if (args.config == "fbocc200" and not args.no_frames16 and 16 % world == 0):
        try:
            extra["frames16"] = frames16_block(world, rank, dev, flush, barrier,
                                               args.steps)
        except Exception as ex:
            extra["frames16"] = {"unavailable": str(ex)[:160]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    units = total_frames * w.units_per_frame
    value = units / (step_ms * 1e-3)

    # ---- roofline -----------------------------------------------------------
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    extra_bytes = {}
    idx = None
    if w.vt is not None:
        idx = w.vt.prepare_index(w.vt.get_lidar_coor(*w.cam))
        n_kept, n_int = (int(v) for v in idx.counts.tolist())
        n_pts = w.depth.numel()
        pool_bytes = 4 * (w.depth.numel() + w.feat.numel() + 3 * n_kept +
                          2 * n_int + w.voxels_per_frame * w.c["C"] * w.frames)
        extra_bytes["bev_pool_v2_fwd_dense_planned"] = pool_bytes
        extra_bytes["voxel_prepare_cams"] = 12 * n_pts + 4 * (3 * n_kept +
                                                               2 * n_int)
        extra_bytes["bev_pool_v2_plan"] = 4 * (n_kept + 4 * n_int)
    if w.bp is not None:
        nq = w.c["bev"][0] * w.c["bev"][1]
        extra_bytes["point_sampling"] = 13 * w.c["n_cams"] * w.frames * nq * 4
    ksum = sum(e0.elapsed_time(e1) for _, _, e0, e1 in krecords) * 1e3 / ksteps
    rows = kernel_table(krecords, step_ms * 1e3, ksteps, extra_bytes,
                        {"depth_elems": w.depth.numel()})
    for r in rows:
        if "achieved_gbs" in r:
            r["frac_of_hbm_peak"] = r["achieved_gbs"] / peak
    dominant = "bev_pool_v2_fwd_dense_planned" if w.vt is not None else \
        rows[0]["kernel"]
    drow = next(r for r in rows if r["kernel"] == dominant)
    d_us = drow["us_per_step"] / drow["launch_calls_per_step"]
    d_bytes = drow.get("algorithmic_bytes_per_step", 0) / \
        drow["launch_calls_per_step"]
    achieved = d_bytes / (d_us * 1e-6) / 1e9
    roofline = {
        "bound": "hbm",
        "kernel": ("interval_sums_kernel + dense_write_kernel (dense "
                   "lift-splat pooling: both launches of "
                   "fbbev_bev_pool_v2_fwd_dense_planned; the kernel the "
                   "voxels/s metric and SURVEY.md section 8(d) are defined on)"
                   if w.vt is not None else dominant),
        "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "peak_source": peak_src, "traffic": None,
        "algorithmic_bytes": int(d_bytes), "kernel_us": d_us,
        "share_of_step": drow["share_of_step"],
        "timed": "CUDA events around the C-ABI call on the launching stream, "
                 f"mean of {ksteps} steps, L2 flushed before each step, "
                 "launches queued behind a spin kernel (device-side back to "
                 "back, as in the graph replay)"}
    prof = os.path.join(ROOT, "profiles", "pool_dense_traffic.json")
    if w.vt is not None and args.config == "fbocc200" and os.path.exists(prof):
        try:
            tr = json.load(open(prof))
            roofline["traffic"] = tr["dram_bytes_per_launch"]
            roofline["traffic_source"] = tr.get(
                "source", "profiles/pool_dense_traffic.json (ncu --set full)")
        except Exception:
            pass
    roofline_kernels = {
        "note": "every C-ABI launch of the step, same timing as `roofline`; "
                "share_of_step is relative to the graph-replay step; "
                "`other_device_time_us` = remaining torch element-wise / copy "
                "/ 3x3 linear-algebra launches",
        "kernels": [r for r in rows if r["share_of_step"] >= 0.02],
        "own_kernels_us_per_step": ksum,
        "other_device_time_us": max(0.0, step_ms * 1e3 - ksum)}

    # ---- the reference on this GPU, for context -----------------------------
    if not args.no_reference_cuda:
        try:
            extra["reference_cuda"] = time_reference_gpu(w, idx, flush, step_ms)
        except Exception as ex:
            extra["reference_cuda"] = {"unavailable": str(ex)[:160]}

    # ---- the detector's glue around the two calls (fbocc.py:339, 357-366) ----
    if world == 1 and args.config == "fbocc200" and not args.no_reference_cuda:
        try:
            extra["pipeline_readd"] = time_pipeline_readd(w, flush)
        except Exception as ex:
            extra["pipeline_readd"] = {"unavailable": str(ex)[:160]}

    # ---- next stage (SURVEY.md section 8 f2): the history warp ----------------
    if world == 1 and args.config == "fbocc200" and not args.no_reference_cuda:
        try:
            extra["fuse_history_warp"] = time_history_warp(dev, flush, peak)
        except Exception as ex:
            extra["fuse_history_warp"] = {"unavailable": str(ex)[:160]}

    # ---- CPU baseline beside it (rank 0, N = 1) ------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        wc = Workload(args.config, "cpu", seed=0, frames=1)
        cr = CpuReference(wc)
        cr.calibrate()
        n, t0 = 0, time.perf_counter()
        while n < 3 or (time.perf_counter() - t0 < 10.0 and n < 50):
            cr.step()
            n += 1
        dt = (time.perf_counter() - t0) / n
        cpu_baseline = {"value": wc.units_per_frame / dt, "unit": unit,
                        "cores": cr.threads, "cores_available": cr._n_cores,
                        "kind": "port",
                        "sample": f"{n} steps of " + cpu_sample_note(wc) +
                                  f" ({dt * 1e3:.1f} ms each); the OpenMP port "
                                  "is fastest on a subset of the logical cores "
                                  "(calibrated at run time)"}

    line = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.config, world),
        "clocks": clocks,
        "e2e": {"value": units / (e2e_ms * 1e-3), "unit": unit,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms, "mode": e2e_mode,
                "latency_ms_one_step": e2e_latency_ms},
        "e2e_refined_only": ({
            "value": units / (e2e_small_ms * 1e-3), "unit": unit,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": e2e_small_d2h,
            "ms_per_step": e2e_small_ms,
            "what": "same streamed pipeline, but only BackwardProjection's "
                    "refined BEV returns to the host; the voxel volume stays "
                    "on the device for its consumer (FBOCC.fuse_history / the "
                    "occupancy head run there).  `e2e` above is the "
                    "conservative number: every result over PCIe"}
            if e2e_small_ms > 0 else None),
        "gpu_launches": launches,
        "roofline": roofline,
        "roofline_kernels": roofline_kernels,
        "cpu_baseline": cpu_baseline,
        "details": {"submission": "cuda graph replay of the plugin calls"
                                  if use_graph else "eager plugin calls",
                    "eager_ms_per_step": eager_ms,
                    "wall_s_timed_region": wall, "host_affinity": numa,
                    "geometry": "fused kernels, bit-identical to the eager "
                                "chain (tests: test_fused_geometry_bit_exact, "
                                "test_fused_point_sampling_bit_exact)"},
    }
    line.update(extra)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def frames16_block(world, rank, dev, flush, barrier, steps):
    """BASELINE.json configs[2]: 16 frames in total, `16 / world` per rank
    (strong scaling), the refined BEV of every frame written straight into the
    rank's slot of the all-gather buffer; timed without and with the NCCL
    all-gather inside the step (device clock, max over ranks)."""
    import torch.distributed as dist
    from fbbev_b200.sharding import GatherBuffer
    per_rank = 16 // world
    w16 = Workload("frames16", dev, seed=100 + rank, frames=per_rank)
    buf = GatherBuffer(per_rank, w16.c["C"], *w16.c["bev"], dev)
    w16.out_buffer = buf.slot
    for _ in range(3):
        w16.step()
    res = {}
    try:
        w16.capture()
        compute, sub = w16.graph.replay, "cuda graph replay"
    except Exception:
        compute, sub = w16.step, "eager"

    def with_gather():
        compute()
        buf.gather()       # NCCL, same stream, in place on the slot's buffer
    for tag, fn in (("compute_only", compute), ("with_gather", with_gather)):
        for _ in range(3):
            fn()
        ms = timed_steps(fn, steps, flush, barrier)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
        res[tag] = {"ms_per_step": ms, "submission": sub,
                    "value": 16 * w16.voxels_per_frame / (ms * 1e-3),
                    "unit": "voxels/s"}
    res["frames_total"] = 16
    res["frames_per_gpu"] = per_rank
    res["scaling"] = "strong"
    res["gather_bytes_per_rank"] = int(buf.slot.numel() * 4)
    res["collective"] = ("nccl all_gather_into_tensor, in place on the buffer "
                         "BackwardProjection.forward(out=slot) wrote into")
    del w16
    torch.cuda.empty_cache()
    return res


def time_pipeline_readd(w, flush):
    """forward -> mean(-1) -> backward -> refined[..., None] + bev_feat, the
    three lines of FBOCC.extract_img_bev_feat around the plugin calls: the
    literal sequence (plugin calls + two torch ops over the 204.8 MB volume)
    against forward_backward_readd (interval sums -> Z-mean -> backward ->
    dense write with the re-add: the volume is written once).  CUDA-graph
    replays of each, L2 flushed, device clock."""
    from fbbev_b200.view_transformation.forward_projection import \
        forward_backward_readd

    @torch.no_grad()
    def literal():
        bev = w.vt(w.cam, w.feat, w.depth)
        ref = w.bp([w.feat], None, lss_bev=bev.mean(-1), cam_params=w.cam,
                   pred_img_depth=w.depth)
        return ref[..., None] + bev

    @torch.no_grad()
    def fused():
        return forward_backward_readd(w.vt, w.bp, w.cam, w.feat, w.depth)[0]

    res = {}
    for name, fn in (("literal_ms", literal), ("fused_ms", fused)):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
        for _ in range(3):
            g.replay()
        ts = []
        for _ in range(10):
            flush.zero_()
            s = torch.cuda.Event(enable_timing=True)
            e = torch.cuda.Event(enable_timing=True)
            s.record()
            g.replay()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        res[name] = statistics.median(ts)
        del g, out
    res["speedup"] = res["literal_ms"] / res["fused_ms"]
    res["what"] = ("F + bev_feat.mean(-1) + B + refined[..., None] + bev_feat "
                   "(fbocc.py:339, 357-366), one frame, graph replay")
    return res


def time_history_warp(dev, flush, peak):
    """The sampling half of FBOCC.fuse_history at the shipped FB-OCC size
    (16 history frames x 80 channels of 8 x 100 x 100 voxels, one sample):
    fbbev_history_warp writing into the concatenation buffer against the
    reference's op sequence (generate_grid matmul + F.grid_sample + torch.cat +
    the history clone, fbocc.py:199-204, 275, 286, 311) on this GPU."""
    from fbbev_b200.view_transformation.temporal_fusion import history_warp
    from oracle.history_ref import history_warp_cpu
    n, T, C, Z, H, W = 1, 16, 80, 8, 100, 100
    g = torch.Generator(device=dev).manual_seed(5)
    hist = torch.randn(n, T * C, Z, H, W, device=dev, generator=g)
    curr = torch.randn(n, C, Z, H, W, device=dev, generator=g)
    out = torch.empty(n, (T + 1) * C, Z, H, W, device=dev)
    flow = torch.eye(4, device=dev)[None].clone()
    flow[0, 0, 0], flow[0, 0, 1] = 0.9994, -0.0349   # 2 degrees of yaw
    flow[0, 1, 0], flow[0, 1, 1] = 0.0349, 0.9994
    flow[0, :3, 3] = torch.tensor([1.7, -0.6, 0.0])

    def ev(fn, iters=10):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            s = torch.cuda.Event(enable_timing=True)
            e = torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) * 1e3)
        return statistics.median(ts)

    def ours():
        out[:, :C].copy_(curr)
        history_warp(hist, flow, out, C)

    def ref():
        tmp = torch.empty(n, T * C, Z, H, W, device=dev)
        history_warp_cpu(hist, flow, tmp, 0)        # grid matmul + grid_sample
        cat = torch.cat([curr, tmp], 1)             # :286
        return cat[:, :-C].detach().clone()         # :311
    us, ref_us = ev(ours), ev(ref)
    nbytes = 4 * (2 * hist.numel() + 2 * curr.numel())
    return {"shape": "1 x (16 x 80) x 8 x 100 x 100", "ours_us": us,
            "reference_eager_us": ref_us, "speedup": ref_us / us,
            "algorithmic_bytes": nbytes,
            "achieved_gbs": nbytes / (us * 1e-6) / 1e9,
            "frac_of_hbm_peak": nbytes / (us * 1e-6) / 1e9 / peak}


def time_reference_gpu(w, idx, flush, our_step_ms):
    """The reference's execution of the same step on THIS GPU: its own
    bev_pool_cuda.cu (oracle/_ref) where it exists, and the eager-PyTorch
    restatement of everything else (oracle/gpu_ref.py; BASELINE.md 2.1-2.2)."""
    from oracle import gpu_ref, ref_cuda

    spread = {}

    def wall(fn, iters=7, warm=4, tag=None):
        """Best of `iters` synchronised calls (us).  The reference path is full
        of host synchronisations, so on a busy host single calls stall by tens
        of ms; the MINIMUM is the reference at its best -- the conservative
        choice for a speed-up -- and the median is recorded beside it."""
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        if tag:
            spread[tag] = statistics.median(ts) * 1e6
        return min(ts) * 1e6

    out = {"timing": "host wall clock around a synchronised call, L2 flushed, "
                     "BEST of 7 after 4 warm-up calls (the reference path has "
                     "host syncs and launches on the legacy default stream; "
                     "medians in `median_us`)",
           "label": "reference (PyTorch restatement; mmcv MSDA kernel "
                    "unavailable -> its documented grid_sample equivalent)"}
    ref_step = 0.0
    if w.vt is not None:
        vt = w.vt
        out["get_lidar_coor_us"] = wall(lambda: vt.get_lidar_coor(*w.cam),
                                        tag="get_lidar_coor")
        coor = vt.get_lidar_coor(*w.cam)
        out["voxel_pooling_prepare_v2_us"] = wall(
            lambda: gpu_ref.voxel_pooling_prepare_v2(
                coor, vt.grid_lower_bound, vt.grid_interval, vt.grid_size),
            tag="voxel_pooling_prepare_v2")
        rb, rd, rf, st, ln = idx.trimmed()
        feat = w.feat.permute(0, 1, 3, 4, 2).contiguous()
        shape = vt._bev_feat_shape(w.depth, feat)
        if ref_cuda.available():
            zo = torch.zeros(shape, device=w.device)
            out["bev_pool_v2_kernel_us"] = wall(
                lambda: ref_cuda.bev_pool_v2_kernel(w.depth, feat, rd, rf, rb,
                                                    st, ln, zo), iters=20)
            out["bev_pool_v2_op_as_shipped_us"] = wall(
                lambda: ref_cuda.bev_pool_v2(w.depth, feat, rd, rf, rb, shape,
                                             st, ln), iters=20)
            del zo
        else:
            out["bev_pool_v2_op_as_shipped_us"] = wall(
                lambda: gpu_ref.bev_pool_v2_index_add(w.depth, feat, rd, rf,
                                                      rb, shape))
            out["bev_pool_v2_note"] = ("oracle/_ref not built: torch "
                                       "index_add_ restatement of the op")
        ref_step += out["get_lidar_coor_us"] + \
            out["voxel_pooling_prepare_v2_us"] + \
            out["bev_pool_v2_op_as_shipped_us"]
        out["forward_projection_us"] = ref_step
    if w.bp is not None:
        enc = w.bp.transformer.encoder

        @torch.no_grad()
        def ref_b():
            with gpu_ref.eager_reference_mode(enc):
                return w.bp([w.feat] + list(w.more), None, lss_bev=w.lss,
                            cam_params=w.cam, pred_img_depth=w.depth)
        out["backward_projection_us"] = wall(ref_b, tag="backward_projection")
        ref_step += out["backward_projection_us"]
    out["median_us"] = spread
    out["step_us"] = ref_step
    out["ours_step_us"] = our_step_ms * 1e3
    out["speedup_vs_reference_gpu"] = ref_step / (our_step_ms * 1e3)
    return out


if __name__ == "__main__":
    main()
