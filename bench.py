#!/usr/bin/env python
"""bench.py -- M query-points/sec of the occupancy query on a dense grid (BASELINE.json's metric).

Usage: `python bench.py --gpus N --steps K --warmup W [--dump-outputs DIR]` prints ONE JSON line on rank 0.
Default workload = BASELINE.json configs[1] (the config the metric is quoted on): icon-filter, dense 256^3
cell-centre lattice, one image per GPU (weak scaling).  A step = one pass of the hot path
(HGPIFuNet.query: SMPL SDF block + feature gather + occupancy MLP + in_cube mask, through query_func) over
every image this rank owns.  `--workload` selects the other BASELINE configs:

    icon-filter-256      config 2   icon prior, c0=13, 256^3, 1 image per GPU               (weak)   DEFAULT
    icon-nofilter-512x8  config 3   icon prior, c0=10, 512^3, 8 images on every GPU          (weak)
    pamir-256            config 4   voxel-aligned prior, 256^3, 32 images sharded over GPUs  (strong)
    pifu-512             config 5   pixel-aligned prior, 512^3, 64 images sharded over GPUs  (strong)

Besides the metric the line carries: `e2e` (same metric through query_func with HOST buffers: pinned H2D of the
points and D2H of the occupancies inside the timed region), `roofline` of the dominant kernel (+ `rooflines` for
the other kernels of the path), `recon` (one full image per rank: filter -> Seg3dLossless engine -> marching cubes
-> NCCL gather of the meshes to rank 0, the only collective of the path), `reference_gpu` (the reference's own
stock-PyTorch/cuDNN encoders timed on the same GPU) and `cpu_baseline`.

`--dump-outputs DIR` writes the occupancies the last timed step computed (see dump_outputs), so that two builds can
be compared output for output: the inputs are seeded and identical from run to run.

`--impl reference` times the reference's CPU path for the same metric: the oracle's port of query_func (oracle/,
brute-force SDF in C with OpenMP + torch CPU MLP) on the host cores, on a bounded sample of the same lattice.
The reference itself cannot be installed here (its hot path needs kaolin / pytorch3d wheels that are not
available offline; see DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: preset, prior, c0, grid, feature map (C, size), images (per GPU | total), scaling, MLP FLOP / point
    "icon-filter-256": dict(preset="icon-filter", prior="icon", c0=13, grid=256, feat=(12, 128), per_gpu=1,
                            total=None, scaling="weak", flop=344602,
                            label="icon-filter, dense 256^3 cell-centre lattice (16,777,216 points), 1 image per GPU"),
    "icon-nofilter-512x8": dict(preset="icon-nofilter", prior="icon", c0=10, grid=512, feat=(6, 512), per_gpu=8,
                                total=None, scaling="weak", flop=340756,
                                label="icon-nofilter, dense 512^3 lattice (134,217,728 points), batch of 8 images per GPU"),
    "pamir-256": dict(preset="pamir", prior="pamir", c0=13, grid=256, feat=(6, 128), per_gpu=None, total=32,
                      scaling="strong", flop=344602,
                      label="pamir (voxel-aligned features), dense 256^3 lattice, batch of 32 images sharded over the GPUs"),
    "pifu-512": dict(preset="pifu", prior="pifu", c0=13, grid=512, feat=(12, 128), per_gpu=None, total=64,
                     scaling="strong", flop=344602,
                     label="pifu, dense 512^3 lattice, batch of 64 images sharded over the GPUs"),
}
DEFAULT_WORKLOAD = "icon-filter-256"
CPU_SAMPLE = 131072
DUMP_BYTES = 60 << 20                # --dump-outputs writes at most this much, over all ranks
DUMP_SEED = 1234


def _peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written).  The tensor figure used is the BURST one: the
    timed region is a fraction of a second at full clocks (VERDICT r1); the sustained figure is reported beside it."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def _measured_traffic():
    """dram bytes per launch of this build's kernels, from the ncu --set full pass committed under profiles/
    (tools/ncu_traffic.py writes the file); None when no pass of the current round exists."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.first = 0

    def mark(self, wait_s=3.0):
        """Call right before the timed region: nvidia-smi was started long before (its start-up takes driver locks and
        can stall kernel launches for tens of ms -- seen as a 2x outlier of the resident figure when it was spawned right
        here); wait until it is in its steady 25 ms polling loop and count only the rows from now on."""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < wait_s:
            time.sleep(0.01)
        self.first = len(self.rows)

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.first:]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------- synthetic cases
def surface_following(sd, c0, prior):
    """Random weights (N(0, 1/fan_in), non-trivial BN statistics) plus one skip-connection term in the last layer so
    that the 0.5 level set is a body-like surface instead of noise: the clipped SDF channel for the icon prior, z for
    pifu / pamir.  Throughput does not depend on the values; the engine's boundary sets and the mesh do."""
    sd = {k: v.clone() for k, v in sd.items()}
    w = sd["filters.3.weight"]                       # [1, 128 + c0, 1]
    w[0, :128, 0] *= 0.2
    if prior == "icon":
        w[0, 128 + (c0 - 7), 0] = 12.0               # point_feat = [local (c0-7), sdf, cmap(3), norm(3)]
        sd["filters.3.bias"] = sd["filters.3.bias"] * 0 + 0.5
    else:
        w[0, 128 + c0 - 1, 0] = -6.0                 # last input channel: z (pifu) / last volume channel (pamir)
        sd["filters.3.bias"] = sd["filters.3.bias"] * 0 + 0.5
    return sd


def build_model(dev, wl, seed=0):
    """The network (one per process, shared by all images): MLP weights + encoders (seeded)."""
    from icon_b200 import config, net, synthetic as S
    cfg = config.preset(wl["preset"])
    netG = net.HGPIFuNet(cfg).to(dev).eval()
    sd = surface_following(S.mlp_state_dict(c0=wl["c0"], seed=seed), wl["c0"], wl["prior"])
    netG.if_regressor.load_state_dict(sd)
    return cfg, netG, sd


def build_image(wl, seed):
    """One synthetic 'image' on the CPU: feature map (+ body mesh | volume feature).  SURVEY.md 8d."""
    import torch
    from icon_b200 import synthetic as S
    C, size = wl["feat"]
    img = {"feat": S.feature_map(C, size, seed=seed)}
    if wl["prior"] == "icon":
        v, f = S.body_mesh(seed=seed)
        cm, vi = S.body_attributes(v, seed=seed)
        img["smpl"] = {"smpl_verts": torch.from_numpy(v)[None], "smpl_faces": torch.from_numpy(f)[None],
                       "smpl_cmap": torch.from_numpy(cm)[None], "smpl_vis": torch.from_numpy(vi)[None]}
    elif wl["prior"] == "pamir":
        g = torch.Generator().manual_seed(seed + 31)
        img["vol_feat"] = torch.randn(1, 7, 32, 32, 32, generator=g)
    return img


class DeviceImage:
    """An image's tensors on the GPU + the per-image state HGPIFuNet.filter() would leave behind."""

    def __init__(self, img, dev):
        self.feat = img["feat"].to(dev)
        self.smpl = {k: t.to(dev) for k, t in img.get("smpl", {}).items()}
        self.vol_feat = img["vol_feat"].to(dev) if "vol_feat" in img else None
        self.body_cache = None

    def bind(self, netG):
        """Point the network at this subject (what filter() does at HGPIFuNet.py:236-245)."""
        from icon_b200 import net
        if self.smpl:
            netG.smpl_feat_dict = self.smpl
            if self.body_cache is None:
                self.body_cache = net._SourceCache()
            netG._body_cache = self.body_cache         # prepared SmplBody is per subject: keep one per image
        if self.vol_feat is not None:
            netG._vol_feat = self.vol_feat


def oracle_threads():
    """Threads the C oracle's OpenMP loop will really use (OMP_NUM_THREADS is fixed before the library loads)."""
    import oracle
    try:
        return int(oracle.lib().oracle_num_threads())
    except Exception:
        return 1


def cpu_port_rate(wl, sd, img, n_sample):
    """Oracle port of query_func on the host cores; returns (M points/s, seconds, threads)."""
    import torch
    from oracle import query as OQ
    from icon_b200 import synthetic as S
    threads = oracle_threads()
    torch.set_num_threads(threads)
    pts = S.lattice_points(min(wl["grid"], 256))
    stride = max(1, pts.shape[1] // n_sample)
    sample = pts[:, ::stride][:, :n_sample].contiguous()
    kw = {"prior": wl["prior"]}
    if wl["prior"] == "icon":
        kw.update(smpl=img["smpl"], sdf_clip=0.05)
    elif wl["prior"] == "pamir":
        kw.update(vol_feat=img["vol_feat"])
    t0 = time.perf_counter()
    OQ.query_func(sd, [img["feat"]], sample, **kw)
    dt = time.perf_counter() - t0
    return sample.shape[1] / dt / 1e6, dt, threads


def _fix_omp_threads():
    """Decide the CPU arm's thread count BEFORE liboracle.so / torch load OpenMP (VERDICT r1 weak #11)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:                                             # cgroup CPU quota, when the box is a container slice
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        try:                                         # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, q // p))
        except Exception:
            pass
    if "TORCHELASTIC_RUN_ID" in os.environ or "LOCAL_RANK" in os.environ:
        # torchrun pins OMP_NUM_THREADS=1 for every rank unless the user set it; the CPU arm runs on rank 0 alone and is
        # specified to use all the host threads it can
        if os.environ.get("OMP_NUM_THREADS", "1") == "1":
            os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.setdefault("OMP_NUM_THREADS", str(n))
    return n


def run_reference(args, wl):
    """Reference arm: the reference's CPU implementation of the path (oracle port), rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    _fix_omp_threads()
    from icon_b200 import synthetic as S
    sd = surface_following(S.mlp_state_dict(c0=wl["c0"], seed=0), wl["c0"], wl["prior"])
    img = build_image(wl, seed=0)
    for _ in range(args.warmup):
        cpu_port_rate(wl, sd, img, 2048)
    t_tot, threads, n = 0.0, 1, CPU_SAMPLE
    for _ in range(args.steps):
        r, dt, threads = cpu_port_rate(wl, sd, img, CPU_SAMPLE)
        t_tot += dt
    value = n * args.steps / t_tot / 1e6
    sample = (f"{n} strided lattice points per step; oracle port of query_func "
              f"(C/OpenMP brute-force SDF + torch CPU MLP), {threads} OpenMP/torch threads")
    line = {
        "impl": "reference", "metric": f"M query-points/sec at {wl['grid']}^3 grid", "value": value, "unit": "Mpoints/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["label"], "sample": f"{n} lattice points per step (strided subset)"},
        "cpu_baseline": {"value": value, "unit": "Mpoints/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- GPU helpers
def timed(fn, reps, flush=None):
    """Median CUDA-event time (ms) of fn() over `reps` runs; `flush` (a > L2 buffer) is rewritten before each."""
    import torch
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def timed_graph(fn, n=8, reps=5):
    """ms per call of fn() with `n` back-to-back calls captured into one CUDA graph (kernels shorter than the host's
    launch latency cannot be timed call by call: the events would measure the CPU)."""
    import torch
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) / n)
    ts.sort()
    return ts[len(ts) // 2]


def encoder_rooflines(dev, peaks, netG):
    """Tensor-bound kernels of the encoders: the ResnetBlock convolution (80 % of NormalNet's FLOPs) and the whole
    forwards, algorithmic FLOPs / time against the measured bf16 burst peak (the kernels execute 3 fp16 MMAs per
    algorithmic one)."""
    import torch
    import torch.nn as nn
    from icon_b200 import nhwc as T, synthetic as S
    out = []
    with torch.no_grad():
        m = nn.Conv2d(1024, 1024, 3, padding=0).to(dev)
        raw = T.raw_from_nchw(torch.randn(1, 1024, 32, 32, device=dev))
        op, _ = T.act(raw, halo=1)
        ms = timed_graph(lambda: T.conv(op, m))
        flop = 2.0 * 1024 * 9 * 1024 * 32 * 32
        out.append({"kernel": "k_conv_nhwc<256,2> + k_splitk_nhwc: ResnetBlock conv 1024->1024 3x3 reflect @32x32 (TMA + tcgen05, "
                              "fp16 hi/lo x3, split-K 4)", "bound": "tensor", "ms": ms, "achieved": flop / ms / 1e9,
                    "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": flop / ms / 1e9 / peaks["bf16_tflops"],
                    "executed_frac": 3 * flop / ms / 1e9 / peaks["bf16_tflops"],
                    "note": "operand traffic L2 -> SM is 96 KB per 64-channel chunk = 59 B/clk/SM at the MMA rate, above the "
                            "~43 B/clk/SM the L2 sustains chip-wide (B300_MICROARCH.md: ~6300 B/clk): L2-bound, not MMA-bound"})
        batch = {k: v.to(dev) for k, v in S.encoder_inputs_512(seed=5).items()}
        for _ in range(3):
            netG.normal_filter(batch)
        ms = timed(lambda: netG.normal_filter(batch), 5)
        out.append({"kernel": "NormalNet.forward 512x512 (2 GlobalGenerators, CUDA-graph replay, all kernels)", "bound": "tensor",
                    "ms": ms, "achieved": 880.0 / ms, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                    "frac": 880.0 / ms / peaks["bf16_tflops"], "executed_frac": 3 * 880.0 / ms / peaks["bf16_tflops"],
                    "flop": 880e9})
        if hasattr(netG, "F_filter"):
            cin = netG.F_filter.conv1.in_channels
            xin = torch.cat([batch["image"], batch["T_normal_F"], batch["T_normal_B"]], 1)[:, :cin].contiguous()
            for _ in range(3):
                netG.F_filter(xin)
            ms = timed(lambda: netG.F_filter(xin), 5)
            gf = 108.3 if cin == 3 else 110.8
            out.append({"kernel": f"HGFilter.forward 512x512 ({cin} input channels, CUDA-graph replay, all kernels)",
                        "bound": "tensor", "ms": ms, "achieved": gf / ms, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                        "frac": gf / ms / peaks["bf16_tflops"], "executed_frac": 3 * gf / ms / peaks["bf16_tflops"],
                        "flop": gf * 1e9})
    return out


def secondary_rooflines(dev, peaks, flush):
    """HBM-bound kernels of the path at their real sizes: algorithmic bytes / CUDA-event time / measured HBM peak."""
    import torch
    from icon_b200 import ops
    out = []
    a = torch.linspace(-1, 1, 257, device=dev)
    z, y, x = torch.meshgrid(a, a, a, indexing="ij")
    occ257 = (0.5 + 2.0 * (0.8 - torch.sqrt((x / 0.45) ** 2 + (y / 0.8) ** 2 + (z / 0.3) ** 2))).contiguous()
    del x, y, z
    # last-level upsample 257^3 -> 513^3 (seg3d_lossless.py:186-203): read R_in^3 * 4, write R_out^3 * 4
    ms = timed(lambda: ops.grid_upsample(occ257, None, 0.5, want_mask=False), 7, flush)
    by = 257 ** 3 * 4 + 513 ** 3 * 4
    out.append({"kernel": "k_grid_upsample (257^3 -> 513^3, last level)", "bound": "hbm", "ms": ms,
                "achieved": by / ms / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": by / ms / 1e6 / peaks["hbm_gbs"],
                "algorithmic_bytes": by})
    # mid-level upsample + boundary mask 129^3 -> 257^3: read 4+1 B, write 4+1+1 B per voxel
    occ129 = occ257[::2, ::2, ::2].contiguous()
    done129 = torch.zeros(129, 129, 129, dtype=torch.uint8, device=dev)
    ms = timed(lambda: ops.grid_upsample(occ129, done129, 0.5), 7, flush)
    by = 129 ** 3 * 5 + 257 ** 3 * 6
    out.append({"kernel": "k_grid_upsample (129^3 -> 257^3 + boundary + done)", "bound": "hbm", "ms": ms,
                "achieved": by / ms / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": by / ms / 1e6 / peaks["hbm_gbs"],
                "algorithmic_bytes": by})
    # marching cubes: read the grid once + 12 B / vertex + 24 B / face written
    for R, occ in ((257, occ257),):
        v, f = ops.marching_cubes(occ, 0.5)
        ms = timed(lambda: ops.marching_cubes(occ, 0.5), 7, flush)
        by = R ** 3 * 4 + v.shape[0] * v.element_size() * 3 + f.shape[0] * 24
        out.append({"kernel": f"marching cubes (k_mc_count + scans + k_mc_verts + k_mc_faces, {R - 1}^3 cells)",
                    "bound": "hbm", "ms": ms, "achieved": by / ms / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": by / ms / 1e6 / peaks["hbm_gbs"], "algorithmic_bytes": by,
                    "verts": int(v.shape[0]), "faces": int(f.shape[0]), "includes": "2 host read-backs (counts)"})
    return out


def recon_stage(dev, cfg, netG, wl, rank, world, reps=3):
    """One full image per rank, the way apps/ICON.py:748-753 drives the path: filter (NormalNet + HGFilter at
    512 x 512 when the config has them) -> Seg3dLossless engine with the real query_func -> marching cubes on the
    device -> gather of the meshes to rank 0 over NCCL (all_gather of headers + grouped send/recv)."""
    import torch
    import torch.distributed as dist
    from icon_b200 import net, ops, synthetic as S, dist as D
    from icon_b200.engine import Seg3dLossless
    mres = wl["grid"]
    res = [2 ** k + 1 for k in range(5, mres.bit_length())]
    eng = Seg3dLossless(query_func=net.query_func, b_min=[[-1.0, 1.0, -1.0]], b_max=[[1.0, -1.0, 1.0]],
                        resolutions=res, align_corners=True, balance_value=0.5, faster=True).to(dev)
    img = build_image(wl, seed=1000 + rank)
    batch = {k: v.to(dev) for k, v in S.encoder_inputs_512(seed=5 + rank).items()}
    if wl["prior"] == "icon":
        batch.update({k: t.to(dev) for k, t in img["smpl"].items()})
    if wl["prior"] == "pamir":
        batch["vol_feat"] = img["vol_feat"].to(dev)
    t = {}
    with torch.no_grad():
        for _ in range(2):                                   # eager + graph capture of the encoders
            feats = netG.filter(batch)
        t["filter"] = timed(lambda: netG.filter(batch), reps)
        feats = netG.filter(batch)
        occ = eng(opt=cfg, netG=netG, features=feats, proj_matrix=None)
        t["engine"] = timed(lambda: eng(opt=cfg, netG=netG, features=feats, proj_matrix=None), reps)
        counts = list(eng.last_query_counts)
        if occ is None:
            verts = torch.zeros(0, 3, device=dev)
            faces = torch.zeros(0, 3, dtype=torch.int64, device=dev)
            t["marching_cubes"] = 0.0
        else:
            verts, faces = ops.marching_cubes(occ, 0.5)
            t["marching_cubes"] = timed(lambda: ops.marching_cubes(occ, 0.5), reps)
    torch.cuda.synchronize()
    if world > 1:                                            # NCCL opens its point-to-point channels on first use: not timed
        D.gather_meshes([(verts[:8].clone(), faces[:8].clone())], [rank], dev)
        torch.cuda.synchronize()
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    got, nbytes = D.gather_meshes([(verts, faces)], [rank], dev)
    e1.record()
    torch.cuda.synchronize()
    t["gather"] = e0.elapsed_time(e1)
    e0.record()
    host = [(v.cpu(), f.cpu()) for v, f in got.values()] if rank == 0 else []
    e1.record()
    torch.cuda.synchronize()
    t["mesh_d2h"] = e0.elapsed_time(e1)
    keys = ["filter", "engine", "marching_cubes", "gather", "mesh_d2h"]
    mx = D.max_over_ranks([t[k] for k in keys], dev)
    out = {k: v for k, v in zip(keys, mx)}
    out.update({"max_over_ranks": True, "resolutions": res, "query_points_per_call": counts,
                "points_evaluated": int(sum(counts)), "fraction_of_dense_grid": sum(counts) / float((mres + 1) ** 3),
                "verts_rank0_image": int(verts.shape[0]), "faces_rank0_image": int(faces.shape[0]),
                "images_gathered": len(got) if rank == 0 else None,
                "gather_payload_bytes": int(nbytes),
                "gather_how": "all_gather(headers) + grouped ncclSend/ncclRecv of verts/faces to rank 0" if world > 1
                              else "single rank: no collective",
                "ms_per_image_device": out["filter"] + out["engine"] + out["marching_cubes"]})
    if rank == 0 and host:
        out["verts_total"] = int(sum(v.shape[0] for v, _ in host))
        out["faces_total"] = int(sum(f.shape[0] for _, f in host))
    return out


def reference_gpu_encoders(dev, netG, reps=3):
    """The reference's own GPU path for the encoders: stock torch ops (cuDNN) on the same weights, same GPU."""
    import torch
    from icon_b200 import synthetic as S
    from tools import torch_encoders as TE
    batch = {k: v.to(dev) for k, v in S.encoder_inputs_512(seed=5).items()}
    cin = netG.F_filter.conv1.in_channels if hasattr(netG, "F_filter") else 3
    xin = torch.cat([batch["image"], batch["T_normal_F"], batch["T_normal_B"]], 1)[:, :cin].contiguous()
    out = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True                     # apps/infer.py:47, apps/ICON.py:32
    try:
        with torch.no_grad():
            for tag, tf32 in (("tf32", True), ("fp32", False)):
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32
                fns = {"normalnet": lambda: TE.normal_net(netG.normal_filter, batch)}
                if hasattr(netG, "F_filter"):
                    fns["hgfilter"] = lambda: TE.hgfilter(netG.F_filter, xin)
                for name, fn in fns.items():
                    for _ in range(3):
                        fn()
                    out[f"{name}_{tag}_ms"] = timed(fn, reps)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    out["note"] = ("stock torch 2.11 ops (cuDNN conv, GroupNorm/InstanceNorm, bicubic interpolate) on this repo's parameter "
                   "containers (tools/torch_encoders.py, pinned to the reference modules' goldens); tf32 = torch default "
                   "for convs (what the reference runs with), fp32 = accuracy-matched to this repo's fp16x3 kernels")
    return out


def dump_outputs(out_dir, preds, image_ids, budget=DUMP_BYTES):
    """preds[k] ([1, 1, N] on the device) of image image_ids[k] -> out_dir/preds_image<id>.npy.  When every point of
    every image does not fit in `budget` bytes, each image keeps the same seeded random sample of its N points, so
    that two runs with the same arguments write comparable arrays."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    if not preds:
        return
    n = preds[0].numel()
    k = min(n, budget // 4 // len(preds))
    idx = None
    if k < n:
        g = torch.Generator().manual_seed(DUMP_SEED)
        idx = torch.randint(0, n, (k,), generator=g).sort().values.to(preds[0].device)
    for i, p in zip(image_ids, preds):
        v = p.reshape(-1)
        v = v if idx is None else v[idx]
        np.save(os.path.join(out_dir, f"preds_image{i:03d}.npy"), v.float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--images", type=int, default=None, help="total images (strong workloads) / per GPU (weak)")
    ap.add_argument("--grid", type=int, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-extras", action="store_true", help="metric + e2e only (skip recon / rooflines / baselines)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the occupancies the last timed step computed to DIR/preds_image<i>.npy (float32; a "
                         "fixed seeded sample of each image's points when all of them would exceed 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    wl = dict(WORKLOADS[args.workload])
    if args.grid:
        wl["grid"] = args.grid
        wl["label"] = f"{wl['preset']}, dense {args.grid}^3 lattice"
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args, wl)
    _fix_omp_threads()

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from icon_b200 import _C, net, synthetic as S, dist as D
    import ctypes
    cfg, netG, sd = build_model(dev, wl, seed=0)
    if wl["scaling"] == "weak":
        per = args.images or wl["per_gpu"]
        mine = [rank * per + j for j in range(per)]
        n_images = per * world
    else:
        n_images = args.images or wl["total"]
        mine = D.shard_images(n_images, rank, world)
    images_cpu = [build_image(wl, seed=i) for i in mine]
    images = [DeviceImage(im, dev) for im in images_cpu]
    grid = wl["grid"]
    pts_cpu = S.lattice_points(grid)                                      # [1, N, 3]: 201 MB at 256^3, 1.6 GB at 512^3
    N = pts_cpu.shape[1]
    pts_dev = pts_cpu.to(dev)                                             # larger than the 126 MB L2
    pts_pin = pts_cpu.pin_memory()
    out_pin = torch.empty(1, 1, N, dtype=torch.float32).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def query(im, pts):
        im.bind(netG)
        return net.query_func(cfg, netG, [im.feat], pts)

    def step_resident(keep=None):
        out = None
        for im in images:
            out = query(im, pts_dev)
            if keep is not None:
                keep.append(out)
        return out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                       # before the warm-up: see ClockSampler.mark
    for _ in range(args.warmup):
        step_resident()
    barrier()

    # ---- timed region 1: inputs resident in HBM
    if rank == 0:
        sampler.mark()
    l0 = _C.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    last_step = []                            # the preds of every image in the last timed step, for --dump-outputs
    e0.record()
    for s in range(args.steps):
        out = step_resident(last_step if args.dump_outputs and s == args.steps - 1 else None)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = _C.launch_count() - l0
    checksum = float(out.double().sum().item()) if out is not None else 0.0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step, mine, DUMP_BYTES // world)
    del last_step

    # ---- timed region 2: end to end through query_func with HOST buffers.  Every image of every step copies its
    #      points from pinned host memory and its result back; the three stages (H2D, query, D2H) of consecutive
    #      images overlap on three streams with double-buffered device tensors, as a serving loop would.
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    s_main = torch.cuda.current_stream()
    d_pts = [torch.empty_like(pts_dev) for _ in range(2)]
    d_out = [None, None]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_outfree = [torch.cuda.Event() for _ in range(2)]

    def run_e2e(nsteps):
        i = 0
        for _ in range(nsteps):
            for im in images:
                b = i & 1
                with torch.cuda.stream(s_in):
                    if i >= 2:
                        s_in.wait_event(ev_free[b])               # query i-2 has consumed d_pts[b]
                    d_pts[b].copy_(pts_pin, non_blocking=True)
                    ev_in[b].record(s_in)
                s_main.wait_event(ev_in[b])
                if i >= 2:
                    s_main.wait_event(ev_outfree[b])              # D2H of query i-2 has drained d_out[b]
                d_out[b] = query(im, d_pts[b])
                ev_free[b].record(s_main)
                ev_done[b].record(s_main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_done[b])
                    out_pin.copy_(d_out[b], non_blocking=True)
                    ev_outfree[b].record(s_out)
                i += 1
        s_main.wait_stream(s_out)
        s_main.wait_stream(s_in)

    if images:
        run_e2e(1 if len(images) > 1 else 2)
    barrier()
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None      # sampled under load through both timed regions
    del d_pts, d_out

    # ---- per-stage timing of the query's kernels (CUDA events inside the library, same stream)
    stage = [0.0, 0.0, 0.0, 0.0]
    if images:
        _C.lib.icon_profile_enable(1)
        buf = (ctypes.c_float * 4)()
        for _ in range(args.steps):
            query(images[0], pts_dev)
            _C.check(_C.lib.icon_profile_last_query(buf), "icon_profile_last_query")
            for i in range(4):
                stage[i] += buf[i] / args.steps
        _C.lib.icon_profile_enable(0)

    ms, ms_e2e = D.max_over_ranks([ms, ms_e2e], dev)             # device-timed, max over ranks
    headers = D.gather_headers([float(rank), float(N * len(images)), checksum], dev)
    assert len(headers) == world

    extras = {}
    if not args.no_extras:
        peaks = _peaks()
        extras["recon"] = recon_stage(dev, cfg, netG, wl, rank, world)
        if rank == 0:
            flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)      # 256 MB > L2
            flush.zero_()
            extras["rooflines"] = secondary_rooflines(dev, peaks, flush) + encoder_rooflines(dev, peaks, netG)
            extras["reference_gpu"] = reference_gpu_encoders(dev, netG)
            del flush

    if rank == 0:
        peaks = _peaks()
        total_pts = N * n_images * args.steps
        value = total_pts / (ms * 1e-3) / 1e6
        e2e = total_pts / (ms_e2e * 1e-3) / 1e6
        mlp_ms, sdf_ms = stage[3], stage[1]
        achieved = N * wl["flop"] / (mlp_ms * 1e-3) / 1e12 if mlp_ms > 0 else 0.0
        traffic = _measured_traffic() or {}
        t_mlp = traffic.get("k_query_mlp_tc", {})
        mlp_roof = {
            "kernel": f"k_query_mlp_tc<{wl['prior']}> (tcgen05, fp16 hi/lo x3)", "bound": "tensor",
            "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": achieved / peaks["bf16_tflops"],
            "traffic": t_mlp.get("dram_bytes_per_launch") if t_mlp.get("points") == N else None,
            "traffic_source": (t_mlp.get("source") if t_mlp.get("points") == N else
                               "no ncu --set full pass of this build at this size under profiles/"),
            "ms": mlp_ms, "executed_tflops": 3.0 * achieved, "executed_frac": 3.0 * achieved / peaks["bf16_tflops"],
            "peak_sustained": peaks["bf16_tflops_sustained"],
            "frac_of_sustained": achieved / peaks["bf16_tflops_sustained"] if peaks["bf16_tflops_sustained"] else None,
            "peak_source": peaks["src"] + ": cuBLAS bf16 BURST figure (the timed region is well under a second at full "
                                          "clocks); the 4-s sustained figure is given beside it",
            "note": "achieved = algorithmic MLP FLOPs (FLOP/pt x points) / kernel time from CUDA events on the launch "
                    "stream; the kernel executes 3 fp16 MMAs per algorithmic one to hold 1e-4 (executed_*)"}
        rooflines = [mlp_roof]
        if wl["prior"] == "icon" and sdf_ms > 0:
            by = N * (16 + 32 + 4)                       # xyz4 in, rec[8] + face-rank out
            t_sdf = traffic.get("k_sdf_warp", {})
            rooflines.append({
                "kernel": "k_sdf_warp<32> (exact nearest face + ray parity, issue-bound tree walk)", "bound": "hbm",
                "ms": sdf_ms, "achieved": by / sdf_ms / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": by / sdf_ms / 1e6 / peaks["hbm_gbs"], "algorithmic_bytes": by,
                "traffic": t_sdf.get("dram_bytes_per_launch") if t_sdf.get("points") == N else None,
                "note": "no clean FLOP count (O(log F)..O(F) triangle tests per point); neither HBM- nor tensor-bound: "
                        "instruction issue (profiles/); the HBM figure is reported because SURVEY 8d asks for bytes"})
        rooflines += extras.get("rooflines", [])
        line = {
            "metric": f"M query-points/sec at {grid}^3 grid", "value": value, "unit": "Mpoints/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": wl["label"], "name": args.workload, "prior": wl["prior"], "c0": wl["c0"],
                       "feature_map": [wl["feat"][0], wl["feat"][1], wl["feat"][1]],
                       "body_mesh": {"V": 6890, "F": 13776} if wl["prior"] == "icon" else None,
                       "points_per_image": N, "images": n_images, "images_per_gpu": [len(D.shard_images(n_images, r, world))
                                                                                     for r in range(world)]
                       if wl["scaling"] == "strong" else [len(images)] * world,
                       "parallelism": f"dp{world} (images sharded, no data-path collective)",
                       "l2_policy": "inputs larger than L2 (>= 201 MB of xyz per query, no flush needed)"},
            "e2e": {"value": e2e, "unit": "Mpoints/s", "h2d_bytes_per_step": N * 12 * len(images),
                    "d2h_bytes_per_step": N * 4 * len(images), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "stages_ms": {"bin_sort": stage[0], "sdf_warp": stage[1], "outlier_rank": stage[2],
                          "gather_mlp": stage[3], "dominant": "k_query_mlp_tc" if mlp_ms >= sdf_ms else "k_sdf_warp",
                          "note": "one query of one image; the query is 9 launches in two phases (the reference's "
                                  "outlier-rank rule, HGPIFuNet.py:303-304, needs a prefix sum over the whole call)"},
            "roofline": mlp_roof, "rooflines": rooflines,
            "checksum": checksum, "image_headers": headers,
        }
        for k in ("recon", "reference_gpu"):
            if k in extras:
                line[k] = extras[k]
        if not args.no_cpu_baseline and world == 1 and not args.no_extras:
            r, dt, threads = cpu_port_rate(wl, sd, images_cpu[0], CPU_SAMPLE * 2)
            line["cpu_baseline"] = {"value": r, "unit": "Mpoints/s", "cores": threads, "kind": "port",
                                    "sample": f"{CPU_SAMPLE * 2} strided lattice points, {dt:.1f} s; oracle port of "
                                              f"query_func (C/OpenMP brute-force SDF + torch CPU MLP), {threads} threads"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
