"""SWD timings on the B200; prints one JSON line.

    python tests/perf_swd.py                                   # one GPU: N = 1000 and N = 5000, 64x512, one channel
    torchrun --nproc-per-node 8 tests/perf_swd.py --multi      # N = 5000 with the directions dealt over 8 GPUs

Per N, on DUSty-like images (oracle/swd.py range_images, dropped pixels at -1):
* stage A (dusty_swd_descriptors of both sets) device-timed, and its algorithmic bytes (images read once, descriptors
  written once) over that time against the data-sheet HBM bandwidth of one B200 (7.7 TB/s);
* stage B (dusty_swd_sliced over every level) device-timed, and sorted keys per second (2 sets x rows x directions
  x levels);
* compute_swd end to end (host clock around a synchronised call), and the published op chain (oracle swd_torch) on
  the same GPU and inputs with the same seed, with both scores.
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import swd as oswd  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                                       str(torch.cuda.current_device())], text=True)
        return dict(zip(q.split(","), [s.strip() for s in out.strip().split(",")]))
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}


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


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps, out


def run(n, reference=True):
    from dusty_gan_b200.utils.metrics import swd
    h, w, c, n_desc = 64, 512, 1, 128
    x1 = oswd.range_images(n, c, h, w, 1).cuda()
    x2 = oswd.range_images(n, c, h, w, 2, dropped=0.4).cuda()
    torch.manual_seed(0)
    draws = swd.draw(h, w, c, 2)
    positions, directions = swd.upload_draws(draws, x1.device)
    levels, d, rows = len(draws), directions.shape[2], n * n_desc

    def stage_a():
        return swd.descriptors(x1, positions, levels, n_desc), swd.descriptors(x2, positions, levels, n_desc)
    (desc1, st1), (desc2, st2) = stage_a()
    a_ms = timed(stage_a, 3)
    b_ms = timed(lambda: swd.sliced_sums(desc1, st1, desc2, st2, directions), 3)
    a_bytes = 2 * (x1.numel() * 4 + desc1.numel() * 4)
    keys = 2 * rows * d * levels

    def e2e():
        torch.manual_seed(0)
        return swd.compute_swd(x1, x2)
    e2e_ms, score = wall(e2e, 3)
    out = {"n": n, "rows_per_level": rows, "stage_a_ms": round(a_ms, 3), "stage_a_bytes": a_bytes,
           "stage_a_tb_per_s": round(a_bytes / a_ms / 1e9, 3),
           "stage_a_share_of_hbm_datasheet": round(a_bytes / a_ms / 1e-3 / HBM_BYTES_PER_S, 3),
           "stage_b_ms": round(b_ms, 3), "keys_sorted": keys, "keys_per_s": round(keys / b_ms * 1e3, 1),
           "e2e_ms": round(e2e_ms, 3), "swd": float(score)}
    if reference:
        def ref():
            torch.manual_seed(0)
            return oswd.swd_torch(x1, x2)
        ref_ms, ref_score = wall(ref, 1)
        out.update({"swd_torch_ms": round(ref_ms, 3), "swd_torch": float(ref_score),
                    "speedup_vs_swd_torch": round(ref_ms / e2e_ms, 2)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--multi", action="store_true", help="N = 5000 under torchrun, directions dealt over the ranks")
    args = ap.parse_args()
    if args.multi:
        import torch.distributed as dist
        rank = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl")
        res = run(5000, reference=False)
        if dist.get_rank() == 0:
            print(json.dumps({"card": card(), "world": dist.get_world_size(), "multi": res}))
        dist.destroy_process_group()
        return
    print(json.dumps({"card": card(), "runs": [run(1000), run(5000)]}))


if __name__ == "__main__":
    main()
