"""EMD timings on the B200; prints one JSON line.

    python tests/perf_emd.py                                   # one GPU: probe, op, 200 vs 200 scores
    torchrun --nproc-per-node 8 tests/perf_emd.py --multi      # the 1000 vs 1000 x 2048 evaluation over 8 GPUs

* the ex2 peak of this card from bench_micro/ex2_probe.cu (built into a temporary directory);
* batch 32 x 2048 forward and backward of earth_mover_distance against the reference's kernels restated in
  oracle/emd_reference.cu, on the same GPU;
* MMD/COV/1-NNA-EMD of 200 vs 200 clouds of 2048 points: time, matrix entries per second, and the share of the ex2
  peak (41 MUFU operations per point pair: 30 ex2 in approxmatch, 10 ex2 + 1 sqrt in the cost pass; counted as ex2).
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import sampled_clouds  # noqa: E402

MUFU_PER_PAIR = 41


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                                       str(torch.cuda.current_device())], text=True)
        return dict(zip(q.split(","), [s.strip() for s in out.strip().split(",")]))
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}


def ex2_peak():
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "ex2_probe")
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe,
                               os.path.join(ROOT, "bench_micro", "ex2_probe.cu")])
        return json.loads(subprocess.check_output([exe, "400"], text=True).strip().splitlines()[-1])


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def op_timings():
    from dusty_gan_b200.utils.metrics.distance.emd.earth_mover_distance import emd_backward, emd_forward
    from oracle import emd_ref
    x1 = torch.from_numpy(sampled_clouds(32, 2048, 1)).cuda()
    x2 = torch.from_numpy(sampled_clouds(32, 2048, 2)).cuda()
    g = torch.ones(32, device="cuda")
    cost, factors = emd_forward(x1, x2)
    match = emd_ref.approxmatch(x1, x2)
    ref_cost = emd_ref.matchcost(x1, x2, match)
    out = {"batch": [32, 2048, 2048], "bit_equal_cost": bool(torch.equal(cost, ref_cost))}
    out["ours_forward_ms"] = timed(lambda: emd_forward(x1, x2), 3)
    out["ours_backward_ms"] = timed(lambda: emd_backward(x1, x2, factors, g), 3)
    out["ref_forward_ms"] = timed(lambda: emd_ref.matchcost(x1, x2, emd_ref.approxmatch(x1, x2)), 2)
    out["ref_backward_ms"] = timed(lambda: emd_ref.matchcost_grad(x1, x2, match, g), 2)
    return out


def scores(n, group_run=False):
    from dusty_gan_b200.utils.metrics import cov_mmd_1nna as C
    ref = torch.from_numpy(sampled_clouds(n, 2048, 10)).cuda()
    gen = torch.from_numpy(sampled_clouds(n, 2048, 11)).cuda()
    C.compute_cov_mmd_1nna(gen[:2], ref[:2], 512, ("emd",), verbose=False)      # load the module, set attributes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = C.compute_cov_mmd_1nna(gen, ref, 512, ("emd",), verbose=False)          # ends in a device read-back
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    entries = 3 * n * n
    return {"clouds": [n, n, 2048], "seconds": dt, "entries": entries, "entries_per_s": entries / dt, "scores": s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--multi", action="store_true", help="1000 vs 1000 x 2048 under torchrun")
    ap.add_argument("--n", type=int, default=None)
    args = ap.parse_args()
    if args.multi:
        import torch.distributed as dist
        rank = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        r = scores(args.n or 1000)
        if dist.get_rank() == 0:
            r.update(world=dist.get_world_size(), card=card())
            print(json.dumps(r))
        dist.destroy_process_group()
        return
    res = {"card": card()}
    res["ex2_probe"] = ex2_peak()
    res["op"] = op_timings()
    res["scores"] = scores(args.n or 200)
    peak = res["ex2_probe"]["ex2_per_s"]
    res["scores"]["ex2_share"] = res["scores"]["entries_per_s"] * 2048 * 2048 * MUFU_PER_PAIR / peak
    print(json.dumps(res))


if __name__ == "__main__":
    main()
