#!/usr/bin/env python
"""Benchmark of the DUSty-GAN generate-and-evaluate hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline (BASELINE.json): Chamfer pairs/sec. Default workload = configs[2]: 1000 vs 1000 clouds of 2048
FPS-sampled points, full MMD/COV/1-NNA. One "step" is one complete evaluation through the public
API ``compute_cov_mmd_1nna(gen, ref, 512, ("cd",))``: the entries of M_rr, M_rg, M_gg
(3 N^2 = 3 000 000, each a bidirectional Chamfer distance) reduced to the scores.
  value   entries/s with the clouds resident in HBM (device-timed, max over ranks)
  e2e     the same call fed from pinned HOST buffers: H2D copy of both cloud sets + evaluation + D2H
          of the scores inside the timed region
  roofline   the Chamfer kernel against the FP32 FFMA peak; ``frac`` counts the flops the kernel EXECUTES
          (upper triangle of the stacked matrix), ``frac_algorithmic`` the 3 N^2 entries the reference fills
  stages  configs[1] (head + projection, batch 256 of 64x512, HBM roofline, with and without compaction),
          FPS at 888 / 148 / 32 clouds, scan preprocessing, JSD -- compact numbers; the long form goes to stderr
  cpu_baseline   the reference's own compiled CPU path (oracle/_ref) on a bounded sample
--workload cfg3 | cfg4 select BASELINE configs[3] (DUSty-II, 5000 vs 5000 x 2048) and configs[4] (500 vs 500
un-sampled 32 768-point clouds); they are meant for --gpus 8.
With --gpus N > 1 (launched under torchrun) the rows of the stacked matrix are dealt cyclically to
the ranks and the per-cloud (min, arg-min) vectors are combined by one all-gather; total work is fixed, so
scaling is "strong".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL's INFO log proves how many ranks the communicator really has. It goes to stdout by default, which must
# carry only the one JSON line: unless the caller chose a file, every rank logs to its own file and rank 0
# copies the communicator lines to stderr and into the JSON line ("comm").
NCCL_LOG = None
if int(os.environ.get("WORLD_SIZE", "1")) > 1:
    if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
        os.environ["NCCL_DEBUG"] = "INFO"
    os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    if "NCCL_DEBUG_FILE" not in os.environ:
        NCCL_LOG = f"/tmp/dusty_nccl_{os.environ.get('MASTER_PORT', '0')}_rank{os.environ.get('RANK', '0')}.log"
        os.environ["NCCL_DEBUG_FILE"] = NCCL_LOG
        try:
            os.remove(NCCL_LOG)
        except OSError:
            pass

N_CLOUDS = 1000          # per set (configs[2])
N_POINTS = 2048
H, W = 64, 512
HEAD_BATCH = 256         # configs[1]
SM_COUNT, FP32_LANES = 148, 128


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def ncu_traffic(key):
    """DRAM bytes per launch from the committed ncu --set full capture of this round (profiles/)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh).get(key)
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------
# synthetic inputs: backbone-like range images -> (our) head + projection + FPS -> sampled clouds
# ---------------------------------------------------------------------------------------------------
def backbone_like(batch, channels, seed, device):
    """Stand-in for the DCGAN backbone's outputs (the generator stays the reference's PyTorch module and
    /root/reference does not exist on the GPU box): smooth random depth field in tanh space, calibrated
    like SURVEY.md's regime R1 (ranges of a few m ... ~85 m, about half the pixels kept), plus logits."""
    g = torch.Generator(device=device).manual_seed(seed)
    low = torch.randn(batch, 1, 4, 32, generator=g, device=device)
    smooth = torch.nn.functional.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
    z = smooth + 0.35 * torch.randn(batch, 1, H, W, generator=g, device=device)
    z = (z - z.mean()) / z.std()
    # tanh-space inverse depth: q05..q95 of the range = 3.8 m .. 85 m  <=>  atanh(depth) in -0.60 .. -2.83
    depth = torch.tanh(0.68 * z - 1.72)
    conf = 2.0 * torch.randn(batch, channels, H, W, generator=g, device=device)
    return depth.contiguous(), conf.contiguous()


def make_head(kind, device):
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=1.0).to(device).eval()
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    g = torch.Generator(device=device).manual_seed(3)
    gate.fixed_noise = gate._logistic_from_uniform(torch.rand(1, 1, H, W, generator=g, device=device),
                                                   torch.rand(1, 1, H, W, generator=g, device=device))
    return head


def make_lidar(device):
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    return LiDAR(H, W, 0.9, 120.0, angle=synthetic_hdl64e_angles()).to(device)


def make_clouds(n, seed, head, lidar, device, kind=1, full_resolution=False):
    """n clouds through our head + projection (+ FPS unless full_resolution: then the un-sampled
    (H*W,3) clouds with dropped pixels at the origin, configs[4]'s shape)."""
    from dusty_gan_b200 import pipeline
    out = []
    step = 100 if full_resolution else 500
    for i in range(0, n, step):
        b = min(step, n - i)
        depth, conf = backbone_like(b, kind, seed * 1000003 + i, device)      # distinct streams for any n
        if full_resolution:
            out.append(pipeline.maskout_and_project(head, {"depth": depth, "confidence": conf}, lidar, tol=0.0)["points"])
        else:
            out.append(pipeline.generate_points(head, {"depth": depth, "confidence": conf}, lidar, N_POINTS, tol=0.0)[0])
    return torch.cat(out).contiguous()


def time_events(fn, iters, warmup, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


WORKLOADS = {       # BASELINE.json configs[2..4]: (clouds per set, head, un-sampled)
    "cfg2": (1000, 1, False),
    "cfg3": (5000, 2, False),
    "cfg4": (500, 1, True),
}


def resolve_workload(args):
    """(N, head kind, un-sampled, points per cloud, the config.workload string both arms print)."""
    N, kind, full_res = WORKLOADS[args.workload]
    N = args.clouds if args.clouds is not None else N
    kind = args.dusty if args.dusty is not None else kind
    full_res = full_res or args.full_resolution
    P = H * W if full_res else N_POINTS
    names = {"cfg2": "configs[2]", "cfg3": "configs[3]", "cfg4": "configs[4]"}
    text = (f"{names[args.workload]}: {N} vs {N} clouds x {P} points (DUSty-{'II' if kind == 2 else 'I'} head, "
            f"{'un-sampled' if full_res else 'FPS'}), full MMD/COV/1-NNA via Chamfer")
    return N, kind, full_res, P, text


def r4(x):
    """Five significant digits: keeps the one JSON line short enough for the driver's tail."""
    if isinstance(x, float):
        return float(f"{x:.5g}")
    if isinstance(x, dict):
        return {k: r4(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [r4(v) for v in x]
    return x


def bench_head(device, hbm_gbs, kind, compact):
    """configs[1]: batch 256 of 64x512 through the fused head + projection. 20 launches replayed as one CUDA
    graph (a single launch is latency dominated, SURVEY.md 8d) that rotate over 4 independent input AND output
    buffer sets: 4 x 67/101 MB of inputs alone exceed the 126 MB L2, so no launch finds its inputs cached."""
    from dusty_gan_b200 import _lib, pipeline
    lidar = make_lidar(device)
    head = make_head(kind, device)
    nsets, reps = 4, 20
    sets = []
    lib = _lib.load()
    for i in range(nsets):
        depth, conf = backbone_like(HEAD_BATCH, kind, 11 + i, device)
        bufs = {"mask": torch.empty_like(conf), "depth": torch.empty_like(depth),
                "points": torch.empty(HEAD_BATCH, H * W, 3, device=device)}
        if compact:
            bufs.update(valid_count=torch.empty(HEAD_BATCH, device=device, dtype=torch.int32),
                        valid_index=torch.empty(HEAD_BATCH, H * W, device=device, dtype=torch.int32),
                        valid_points=torch.empty(HEAD_BATCH, H * W, 3, device=device),
                        workspace=_lib.workspace(lib.dusty_head_project_workspace_bytes(HEAD_BATCH, H, W), device))
        sets.append((depth, conf, bufs))

    def run(i=0):
        depth, conf, bufs = sets[i % nsets]
        return pipeline.maskout_and_project(head, {"depth": depth, "confidence": conf}, lidar, tol=0.0, compact=compact, buffers=bufs)
    out = run()
    torch.cuda.synchronize()
    valid_frac = float(out["valid_count"].float().mean()) / (H * W) if compact else None
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for i in range(reps):
                run(i)
    t = statistics.median(time_events(graph.replay, 5, 2)) * 1e-3 / reps
    px = HEAD_BATCH * H * W
    bytes_alg = px * (28 if kind == 1 else 36)
    res = {"ms": t * 1e3, "images_per_s": HEAD_BATCH / t, "gbs": bytes_alg / t / 1e9, "frac": bytes_alg / t / 1e9 / hbm_gbs}
    if compact:     # index map + compacted xyz of the valid pixels: real traffic, not algorithmic bytes (SURVEY.md 8d)
        moved = bytes_alg + px * valid_frac * 16
        res.update(valid_frac=valid_frac, gbs_moved=moved / t / 1e9, frac_moved=moved / t / 1e9 / hbm_gbs)
    return res


def bench_fps(device, head, lidar, sm_max_mhz):
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    n_fps = 888                                   # six clouds per SM: the throughput variant of the FPS kernel
    depth, conf = backbone_like(n_fps, 1, 12, device)
    pts = pipeline.maskout_and_project(head, {"depth": depth, "confidence": conf}, lidar, tol=0.0)["points"]
    elig = ((pts.double() ** 2).sum(-1) > 1e-3).sum(1).float()
    res = {"points_in": H * W, "points_out": N_POINTS, "eligible_mean": float(elig.mean()), "eligible_max": float(elig.max())}
    for n in (n_fps, 148, 32):                    # 32 = the reference's batch (evaluate_synthesis.py:152-157)
        sub = pts[:n].contiguous()
        t = statistics.median(time_events(lambda: downsample_point_clouds(sub, N_POINTS), 5, 2)) * 1e-3
        res[f"clouds_per_s_b{n}"] = n / t
        res[f"ms_b{n}"] = t * 1e3
    # real-KITTI-like clouds: ~28 k eligible points (more than fit one SM's shared memory; SURVEY.md H3)
    dense = pts.clone()
    pool = dense[((dense.double() ** 2).sum(-1) > 1e-3)]
    bad = ~((dense.double() ** 2).sum(-1) > 1e-3)
    g = torch.Generator(device=device).manual_seed(5)
    fill = bad & (torch.rand(bad.shape, generator=g, device=device) < 0.75)
    dense[fill] = pool[torch.randint(0, pool.shape[0], (int(fill.sum()),), generator=g, device=device)] * 1.003
    e2 = ((dense.double() ** 2).sum(-1) > 1e-3).sum(1).float()
    res["dense_eligible_mean"] = float(e2.mean())
    for n in (n_fps, 148):
        sub = dense[:n].contiguous()
        t = statistics.median(time_events(lambda: downsample_point_clouds(sub, N_POINTS), 5, 2)) * 1e-3
        res[f"clouds_per_s_dense_b{n}"] = n / t
    t = statistics.median(time_events(lambda: pipeline.generate_points(head, {"depth": depth, "confidence": conf}, lidar, N_POINTS, tol=0.0), 3, 1)) * 1e-3
    res["image_to_cloud_per_s_b888"] = n_fps / t
    return res, depth, conf, pts


def bench_stages(device, hbm_gbs, peak_src, flush, sm_max_mhz=1965.0):
    """configs[1], range image -> FPS, the real-data side and JSD on one GPU. Returns (compact, verbose)."""
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    lidar = make_lidar(device)
    res = {}
    for kind in (1, 2):
        res[f"head_dusty{kind}"] = bench_head(device, hbm_gbs, kind, compact=False)
        res[f"head_dusty{kind}_compact"] = bench_head(device, hbm_gbs, kind, compact=True)
    head = make_head(1, device)
    res["fps"], depth, conf, pts = bench_fps(device, head, lidar, sm_max_mhz)
    res.update(bench_real_side(device, hbm_gbs, peak_src))
    # JSD of the two occupancy histograms (next row 8f-2) on 1000 vs 1000 sampled clouds, as
    # evaluate_synthesis.py:174-177 calls it (clouds halved into the unit sphere)
    from dusty_gan_b200.utils.metrics.jsd import compute_jsd
    sampled = downsample_point_clouds(pts, N_POINTS) / 2.0
    ja, jb = sampled[:444].repeat(3, 1, 1)[:1000].contiguous(), sampled[444:].repeat(3, 1, 1)[:1000].contiguous()
    compute_jsd(ja, jb)
    ms = statistics.median(time_events(lambda: compute_jsd(ja, jb), 5, 1))
    res["jsd"] = {"clouds_per_s": 2000 / (ms * 1e-3), "ms": ms}
    try:
        stage_cpu_baselines(res, head, lidar, depth[:32], conf[:32], pts[:2], sampled[:4])
    except Exception as exc:        # the checker is optional for the measurement
        res["cpu_error"] = repr(exc)[:120]
    notes = {
        "head": f"batch {HEAD_BATCH} of {H}x{W}; 20 launches replayed as a CUDA graph over 4 rotating input+output buffer sets "
                "(inputs alone 4 x 67/101 MB > 126 MB L2); algorithmic bytes 28/36 B/px (SURVEY.md 8d); *_compact also writes "
                "valid_count / valid_index / valid_points (frac_moved counts them)",
        "fps": "32 768 -> 2048 points; b888 = six clouds per SM, b32 = the reference's batch; dense = ~28 k eligible points per cloud",
        "scan": "256 raw scans 64x2048x4 -> inv/mask/points, 10 back-to-back calls, 512 MB of input > L2",
        "peak": f"HBM {hbm_gbs} GB/s {peak_src}"}
    return res, notes


def stage_cpu_baselines(res, head, lidar, depth, conf, pts, jsd_clouds):
    """cpu_baseline leg of the stages (SURVEY.md 8d): the reference's op chains on the host cores, bounded
    samples. The head/projection/real-data chains are the reference's PyTorch/numpy ops (oracle restatement,
    kind "port"); the reference has NO CPU FPS (fps/...cpp:96), so that line is the oracle's C replay."""
    from oracle import head_projection as hp, jsd as ojsd, native, real_data as rd
    threads = torch.get_num_threads()
    d, c = depth.cpu(), conf.cpu()
    noise, angle = head.gumbel.fixed_noise.cpu(), lidar.angle.cpu()

    def head_cpu():
        mask, dout = hp.maskout_dusty1(d, c, noise)
        return hp.project_2d_to_3d_dense(dout, angle, 0.9, 120.0, 0.0)
    head_cpu()
    t0 = time.perf_counter(); head_cpu(); dt = time.perf_counter() - t0
    res["cpu"] = {"head_images_per_s": len(d) / dt, "head_cores": threads}
    p = pts.cpu().numpy()
    t0 = time.perf_counter(); native.fps(p, N_POINTS); dt = time.perf_counter() - t0
    res["cpu"]["fps_clouds_per_s_1core"] = len(p) / dt
    jc = jsd_clouds.cpu().numpy()
    t0 = time.perf_counter(); ojsd.vote(jc); dt = time.perf_counter() - t0
    res["cpu"]["jsd_clouds_per_s_1core"] = len(jc) / dt
    scans = rd.synthetic_scans(4, seed=1)
    t0 = time.perf_counter()
    items = [rd.dataset_item(x, (H, W)) for x in scans]
    rd.preprocess_reals({k: torch.stack([it[k] for it in items]) for k in items[0]})
    dt = time.perf_counter() - t0
    res["cpu"]["scan_per_s_1core"] = len(scans) / dt
    res["cpu"]["kind"] = "port: oracle restatements of the reference's CPU op chains (it has no CPU FPS)"


def bench_real_side(device, hbm_gbs, peak_src):
    """SURVEY.md 8f-4: raw (64,2048,4) scans -> (inv, mask, points) in one kernel (the reference: numpy per
    scan on DataLoader workers + ~12 ATen kernels per batch), at the evaluation's 64x512 and at full width."""
    from dusty_gan_b200.datasets import preprocess_scans
    n = 256
    g = torch.Generator(device=device).manual_seed(21)
    elev = torch.deg2rad(torch.linspace(2.0, -24.8, H, device=device))[:, None]
    azim = torch.linspace(np.pi, -np.pi, 2049, device=device)[:-1][None, :]
    r = (25 + 12 * torch.randn(n, H, 2048, generator=g, device=device)).abs() + 0.3
    r = r * (torch.rand(n, H, 2048, generator=g, device=device) > 0.25)          # empty pixels
    scans = torch.stack([r * torch.cos(elev) * torch.cos(azim), r * torch.cos(elev) * torch.sin(azim),
                         r * torch.sin(elev), torch.rand(n, H, 2048, generator=g, device=device)], dim=-1).contiguous()
    del r
    res = {}
    for w_out in (W, 2048):
        bufs = preprocess_scans(scans, (H, w_out), 0.9, 120.0, -1)
        reps = 10

        def run():
            for _ in range(reps):           # back to back: one launch alone is latency dominated
                preprocess_scans(scans, (H, w_out), 0.9, 120.0, -1, buffers=bufs)
        ms = statistics.median(time_events(run, 5, 2)) / reps
        # algorithmic bytes per output pixel: one (x,y,z,reflectance) source point in, inv + mask + xyz out
        bytes_alg = n * H * w_out * (16 + 4 + 4 + 12)
        res[f"scan_w{w_out}"] = {"scans_per_s": n / (ms * 1e-3), "ms": ms, "gbs": bytes_alg / ms / 1e6,
                                 "frac": bytes_alg / ms / 1e6 / hbm_gbs}
    return res


# ---------------------------------------------------------------------------------------------------
# CPU baseline: the reference's compiled nnsearch driven like reference cov_mmd_1nna.py:24-51
# ---------------------------------------------------------------------------------------------------
def _cpu_rows(args):
    name, a, b, rows = args
    torch.set_num_threads(1)
    from oracle import refload, native
    cd = refload.load(name) if name else None
    tb = torch.from_numpy(b)
    out = np.zeros((len(rows), b.shape[0]), np.float32)
    for r, i in enumerate(rows):
        if cd is None:
            out[r] = native.pairwise_cd(a[i:i + 1], b, rounding="cpu")[0]
            continue
        b1 = torch.from_numpy(a[i:i + 1]).expand(b.shape[0], -1, -1).contiguous()
        d1 = torch.zeros(b.shape[0], a.shape[1]); d2 = torch.zeros(b.shape[0], b.shape[1])
        i1 = torch.zeros(b.shape[0], a.shape[1], dtype=torch.int); i2 = torch.zeros(b.shape[0], b.shape[1], dtype=torch.int)
        cd.forward(b1, tb, d1, d2, i1, i2)
        out[r] = (d1.mean(1) + d2.mean(1)).numpy()
    return out


def cpu_reference_sample(a, b, rows, cols, variant, procs):
    """Time rows x cols entries of the matrix on the host. variant: 'dustyref_cd' (as shipped: g++ -O0),
    'dustyref_cd_o3', or None (oracle port). Returns (entries/s, seconds, kind)."""
    from oracle import refload
    kind = "reference"
    if variant is None or refload.load(variant) is None:
        variant, kind = None, "port"
    a = np.ascontiguousarray(a[:rows]); b = np.ascontiguousarray(b[:cols])
    chunks = [list(range(r, rows, procs)) for r in range(procs)]
    chunks = [c for c in chunks if c]
    t0 = time.perf_counter()
    if procs == 1:
        _cpu_rows((variant, a, b, chunks[0]))
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(len(chunks)) as pool:
            pool.map(_cpu_rows, [(variant, a, b, c) for c in chunks])
    dt = time.perf_counter() - t0
    return rows * cols / dt, dt, kind


# ---------------------------------------------------------------------------------------------------
def run_reference_arm(args):
    """The reference's own CPU implementation of the path (nnsearch, cd/chamfer_distance.cpp:39-62, compiled -O3
    from /root/reference sources into oracle/_ref) on all host cores, on a bounded sample of the SAME workload:
    the same cloud statistics and points per cloud; brute-force nnsearch does the same work for every entry, so
    entries/s of the sample is entries/s of the whole matrix."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, kind, full_res, P, workload_text = resolve_workload(args)
    cores = os.cpu_count() or 1
    rows = max(cores, 16)
    cols = 64 if P <= 4096 else 2     # ~1-4 s per step
    if P > 4096:
        rows = max(cores // 2, 2)
    rng_a = synthetic_cpu_clouds(rows, 1, P, full_res); rng_b = synthetic_cpu_clouds(cols, 2, P, full_res)
    vals = []
    t_all = time.perf_counter()
    kind_ = "reference"
    for s in range(args.warmup + args.steps):
        if s >= 1 and time.perf_counter() - t_all > 150:      # keep the whole arm within a few minutes
            break
        v, dt, kind_ = cpu_reference_sample(rng_a, rng_b, rows, cols, "dustyref_cd_o3", cores)
        if s >= args.warmup or args.warmup + args.steps <= 1:
            vals.append((v, dt))
    if not vals:
        vals.append((v, dt))
    value = statistics.mean(v for v, _ in vals)
    ms = statistics.mean(dt for _, dt in vals) * 1e3
    sample = (f"{rows}x{cols} entries per step of the {N}x{N}x3 entries of this workload, P={P}; reference nnsearch "
              f"(cd/chamfer_distance.cpp:39-62) compiled -O3 from the reference sources, rows over {cores} processes")
    print(json.dumps(r4({
        "impl": "reference", "metric": "chamfer_pairs_per_s", "value": value, "unit": "entries/s", "n_gpus": args.gpus,
        "steps": len(vals), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "entries/s", "cores": cores, "kind": kind_, "sample": sample},
        "e2e": {"value": value, "unit": "entries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})))


def synthetic_cpu_clouds(n, seed, points=N_POINTS, dropped=False):
    """Host-side clouds with the same statistics as the GPU-made ones (only used by the CPU arm, which must not
    touch the GPU kernels): LiDAR-like points, sensor-centred, normalised range; un-sampled clouds keep half of
    their points at the origin (dropped pixels)."""
    rng = np.random.default_rng(seed)
    az = rng.uniform(-np.pi, np.pi, (n, points)); el = np.deg2rad(rng.uniform(-24.8, 2.0, (n, points)))
    r = np.exp(rng.uniform(np.log(0.035), np.log(0.7), (n, points)))
    if dropped:
        r = np.where(rng.uniform(size=r.shape) < 0.5, 0.0, r)
    return np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], -1).astype(np.float32)




def nccl_comm_evidence(world, device):
    """How many ranks the communicator really has: (1) an all-reduce of ones over it, (2) the 'nranks N' lines of
    rank 0's NCCL INFO log (copied to stderr as well: the driver's rank check greps for them)."""
    import glob
    import re
    ones = torch.ones(1, device=device)
    dist.all_reduce(ones)
    ev = {"backend": "nccl", "world_size": world, "allreduce_of_ones": int(ones.item())}
    lines = []
    for path in ([NCCL_LOG] + glob.glob(NCCL_LOG + "*")) if NCCL_LOG else []:
        if os.path.exists(path):
            with open(path, errors="replace") as fh:
                lines += [ln.strip() for ln in fh if "nranks" in ln]
    ev["nranks_seen"] = sorted({int(m.group(1)) for ln in lines for m in [re.search(r"nranks (\d+)", ln)] if m})
    ev["init_line"] = lines[-1][-200:] if lines else None
    for ln in lines[:4]:
        log("[nccl] " + ln)
    if not lines:
        ev["log"] = os.environ.get("NCCL_DEBUG_FILE")
    return ev


def dump_outputs(directory, scores):
    """What compute_cov_mmd_1nna returned to its caller in the last timed step: one 0-d float64 array per score.
    The inputs are made from fixed seeds, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(directory, exist_ok=True)
    for name, value in scores.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.array(value, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS), help="BASELINE.json configs[2] (default), [3] or [4]")
    ap.add_argument("--clouds", type=int, default=None, help="clouds per set (default: the workload's)")
    ap.add_argument("--skip-extras", action="store_true", help="headline only (no stages / cpu baseline)")
    ap.add_argument("--dusty", type=int, default=None, choices=[1, 2], help="head that makes the clouds (default: the workload's)")
    ap.add_argument("--full-resolution", action="store_true", help="un-sampled 64x512 clouds (32768 points each), as cfg4")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores the last timed step returned as DIR/<name>.npy (float64), to compare two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        return run_reference_arm(args)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}"

    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
    hbm_gbs, sm_max_mhz, peak_src = peaks()
    N, kind, full_res, P, workload_text = resolve_workload(args)
    lidar = make_lidar(device); head = make_head(kind, device)
    t0 = time.perf_counter()
    ref = make_clouds(N, 2, head, lidar, device, kind, full_res)
    gen = make_clouds(N, 1, head, lidar, device, kind, full_res)
    torch.cuda.synchronize()
    log(f"[rank {rank}] inputs ready in {time.perf_counter() - t0:.1f}s: 2 x {tuple(ref.shape)}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    entries = N * N * 3
    # ---- resident-in-HBM throughput ----
    for _ in range(args.warmup):
        scores = M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
    M.KERNEL_EVENTS = []
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        flush.zero_()
        scores = M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
    e1.record()
    barrier()
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = e0.elapsed_time(e1)
    kernel_ms = [a.elapsed_time(b) for a, b in M.KERNEL_EVENTS]
    M.KERNEL_EVENTS = None

    # ---- end to end from pinned host buffers ----
    h_gen = gen.cpu().pin_memory(); h_ref = ref.cpu().pin_memory()

    from dusty_gan_b200 import sharding

    def e2e_step():
        # one rank: a plain H2D copy; sharded: every rank uploads 1/G of the clouds and the ranks all-gather them over NVLink
        # (each byte crosses PCIe once), then the evaluation -- which ends with the D2H of the scores
        g = sharding.upload_sharded(h_gen, device); r = sharding.upload_sharded(h_ref, device)
        return M.compute_cov_mmd_1nna(g, r, 512, ("cd",), verbose=False)
    e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        flush.zero_()
        e2e_scores = e2e_step()
    f1.record()
    barrier()
    e2e_ms = f0.elapsed_time(f1)

    # pairs the pruned search really evaluates on this rank: one extra, untimed evaluation with the library's counter on
    # (a collective when sharded: every rank takes part)
    import ctypes as C2
    cnt = C2.c_uint64()
    _lib.check(_lib.load().dusty_chamfer_count_pairs(1, None), "count_pairs")
    M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
    _lib.check(_lib.load().dusty_chamfer_count_pairs(0, C2.byref(cnt)), "count_pairs")
    comm = nccl_comm_evidence(world, device) if world > 1 else None        # collective: every rank takes part
    stats = torch.tensor([dev_ms, e2e_ms, float(launches), statistics.mean(kernel_ms)], device=device, dtype=torch.float64)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, kern_ms = mx[0].item(), mx[1].item(), mx[3].item()
        launches = int(sm[2].item())
    else:
        kern_ms = stats[3].item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, scores)

    ms_per_step = dev_ms / args.steps
    value = entries / (ms_per_step * 1e-3)
    e2e_value = entries / (e2e_ms / args.steps * 1e-3)
    # roofline of the dominant kernel (chamfer nn_kernel): FP32 FFMA
    flops_per_entry = 12.0 * P * P
    alg_flops = entries * flops_per_entry / world                           # per launch, this GPU's share
    exe_entries = (2 * N) * (2 * N + 1) / 2                                 # stacked upper triangle incl. diagonal
    exe_flops = exe_entries * flops_per_entry / world
    # Clouds above 256 points take the sorted search, which skips candidate chunks by an exact box bound: the pairs it
    # really evaluates are data dependent, so the kernel counts them in one extra, untimed evaluation (6 flop each).
    kept = torch.cat([(c != 0).any(-1).sum(1) + ((c == 0).all(-1).any(1)).long() for c in (ref, gen)]).double()
    kept_pairs = float((kept.sum() ** 2 + (kept ** 2).sum()) / 2) * 2 / world       # both directions, this rank's share
    pruned = cnt.value > 0
    merged = None
    if pruned:
        exe_flops = 6.0 * float(cnt.value)
        merged = {"sorted_and_pruned": True, "points_kept_mean": float(kept.mean()), "points_per_cloud": P,
                  "visited_pairs_this_rank": int(cnt.value), "visited_fraction_of_kept_pairs": float(cnt.value) / kept_pairs}
    # the brute-force kernel on the same clouds (what north_star's >= 60 % FFMA bar is about), timed in the same run
    dense = None
    if not full_res and world == 1 and not args.skip_extras:
        thr = M.MERGE_ORIGIN_ABOVE
        M.MERGE_ORIGIN_ABOVE = 1 << 30
        try:
            M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
            dms = statistics.median(time_events(lambda: M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False), 2, 0))
        finally:
            M.MERGE_ORIGIN_ABOVE = thr
        dflops = (2 * N) * (2 * N + 1) / 2 * flops_per_entry
        dense = {"kernel": "nn_kernel<8,1,0,256> (every pair)", "entries_per_s": entries / (dms * 1e-3), "ms_per_step": dms,
                 "achieved": dflops / (dms * 1e-3) / 1e12, "frac": dflops / (dms * 1e-3) / 1e12 / (SM_COUNT * FP32_LANES * 2 * sm_max_mhz * 1e6 / 1e12)}
    peak_nominal = SM_COUNT * FP32_LANES * 2 * sm_max_mhz * 1e6 / 1e12
    sink = torch.zeros(1, device=device)
    import ctypes as C
    flops = C.c_double()
    lib = _lib.load()

    def probe():
        _lib.check(lib.dusty_probe_fp32_peak(64, _lib.ptr(sink), C.byref(flops), _lib.stream_of(sink)), "probe")
    probe_ms = min(time_events(probe, 5, 2))
    peak_probe = flops.value / (probe_ms * 1e-3) / 1e12
    exe_rate = exe_flops / (kern_ms * 1e-3) / 1e12
    alg_rate = alg_flops / (kern_ms * 1e-3) / 1e12
    roofline = {
        "bound": "fp32_ffma",
        "kernel": ("dusty::chamfer::nn_pair_split_kernel (k-d ordered clouds resident in shared memory, best-first pruned walk, 32-row groups)" if pruned and P <= 2048
                   else "dusty::chamfer::nn_walk_split_kernel<1> (k-d ordered clouds, two-level best-first pruned walk from global memory, 32-row groups)" if pruned
                   else "dusty::chamfer::nn_kernel<8,1,0,256>"),
        "achieved": exe_rate, "peak": peak_nominal, "unit": "TFLOP/s",
        "frac": exe_rate / peak_nominal, "achieved_algorithmic": alg_rate, "frac_algorithmic": alg_rate / peak_nominal,
        "peak_source": f"nominal 148x128x2x{sm_max_mhz:.0f} MHz",
        "peak_probe_ffma_only": peak_probe, "kernel_ms": kern_ms, "kernel_share_of_step": kern_ms / ms_per_step,
        "flops_per_entry": flops_per_entry, "entries_per_launch_executed": exe_entries / world,
        "entries_per_launch_algorithmic": entries / world, "pruned_search": merged, "brute_force_kernel_same_run": dense,
        "traffic": ncu_traffic("chamfer_nn_pair_kernel_n1000" if pruned else "chamfer_nn_kernel_n1000")
        if (world == 1 and args.workload == "cfg2" and N == N_CLOUDS) else None,
        "note": "frac = flops EXECUTED (pairs the pruned search evaluated, kernel counter, x 6) / peak; frac_algorithmic = 3 N^2 entries x "
                "12 P^2 (the reference's work; > 1: most pairs are skipped, exactly)"}
    if pruned and dense is not None:
        # the pruned kernel trades FFMA utilisation for pairs not evaluated: put the every-pair kernel's figure (north_star's >= 60 % bar)
        # and the resulting speed-up next to frac, so that nobody reads frac alone as a regression
        roofline["frac_brute_force_kernel"] = dense["frac"]
        roofline["speedup_over_brute_force_kernel"] = dense["ms_per_step"] / ms_per_step
    line = {
        "metric": "chamfer_pairs_per_s", "value": value, "unit": "entries/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text, "entries_per_step": entries, "clouds_from": "synthetic 64x512 range images -> head+projection+FPS kernels",
                   "parallelism": f"row-sharded x{world}, one all-gather of per-cloud (min, arg-min) keys ({24 * 2 * N} B per rank)" if world > 1 else "single GPU",
                   "l2": "256 MB buffer written between timed steps"},
        "e2e": {"value": e2e_value, "unit": "entries/s", "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": int(h_gen.numel() + h_ref.numel()) * 4, "d2h_bytes_per_step": 28,
                "h2d": "plain copy" if world == 1 else f"1/{world} of the clouds per rank over PCIe + one NVLink all-gather per set (bytes = all ranks together)"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
        "scores": {k: scores[k] for k in ("mmd-cd", "cov-cd", "1-nn-accuracy-cd")},
    }
    if comm is not None:
        line["comm"] = comm
    assert e2e_scores == scores, "host-fed and resident runs must agree exactly"

    if world == 1 and not args.skip_extras:
        try:
            stages, notes = bench_stages(device, hbm_gbs, peak_src, flush, sm_max_mhz)
            line["stages"] = stages
            log("[stages] " + json.dumps({"stages": stages, "notes": notes}))
        except Exception as exc:  # the headline line must still be printed
            line["stages"] = {"error": repr(exc)[:300]}
        # bounded CPU sample: 16 x 16 entries of this very workload through the reference as shipped
        a = ref[:16].cpu().numpy(); b = gen[:16].cpu().numpy()
        if full_res:
            a, b = a[:2], b[:2]
        v, dt, kind_ = cpu_reference_sample(a, b, len(a), len(b), "dustyref_cd", 1)
        line["cpu_baseline"] = {
            "value": v, "unit": "entries/s", "cores": 1, "kind": kind_, "seconds": dt,
            "sample": f"{len(a)} x {len(b)} entries of M_rg of this workload (P={P}) through the reference's nnsearch as shipped "
                      "(load() passes no flags => g++ -O0, single thread); --impl reference is the -O3 all-core arm",
            "host_cores_available": os.cpu_count()}
    print(json.dumps(r4(line)))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
