"""Saved env records on the GPU: save + load throughput and the batched branching pattern (the worked example of pct_save_envs /
pct_load_envs).  Writes one JSON line to OUT/bench_snapshot.json (and stdout).

  python scratch/bench_snapshot.py --out DIR

* save + load round trip of every env of a setting-1 batch (4096 envs: L2 overwritten before every repetition; 16384 envs: the live bytes of
  records and env state, ~156 MB, exceed the 126 MB L2), timed with CUDA events at steady state (after 60 random steps), against one step of
  the same batch.
  Bytes are the LIVE bytes, computed from the counts in the records (live_bytes below): each of save and load reads and writes them once.
* branching: 1024 sources x 50 children in one 51 200-env handle: save_envs(repeat_interleave(sources, 50)), load_envs(all), one step with
  leaf_idx = child index; child env-steps per second.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pct_b200  # noqa: E402

ITEMS = [(i, j, k) for i in range(1, 6) for j in range(1, 6) for k in range(1, 6)]
HBM_TBS = 7.7  # HGX B200 data sheet, one GPU


def ceil(x, a):
    return (x + a - 1) // a * a


def live_bytes(rec):
    """bytes a save (or a load) copies per record, from the counts in the record's DEnvHot header (pct_discrete.cu, DRec; 64-byte record header
    first): header + hot record + leaf / density / edge-load / polygon prefixes + ALIAS arrays + LSAH footprint"""
    h = rec[:, 64:64 + 80].contiguous().view(torch.int32).long().cpu().numpy()
    n_box, n_leaf, n_edge, n_poly = h[:, 0], h[:, 2], h[:, 11], h[:, 17]
    b = 64 + 3584 + ceil(n_leaf * 12, 16) + ceil(n_box * 8, 16) + ceil(n_edge * 32, 16) + ceil(n_poly * 16, 16)
    b = b + (n_box + 1) * 32 + ceil(n_edge, 8) + 32 + 16
    return b, dict(n_box=float(n_box.mean()), n_leaf=float(n_leaf.mean()), n_edge=float(n_edge.mean()), n_poly=float(n_poly.mean()))


def steady_batch(n):
    b = pct_b200.PctBatch(n, 1, item_set=ITEMS, seed=3)
    b.reset()
    for t in range(60):
        b.step(leaf_idx=b.random_policy(1, t))
    torch.cuda.synchronize()
    return b


def timed(fn, reps, flush=None):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i in range(reps):
        if flush is not None:
            flush.add_(1)
        ev[i][0].record()
        fn()
        ev[i][1].record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return float(np.median(ms)), float(ms.min()), float(ms.max())


def round_trip(n, flush):
    b = steady_batch(n)
    rec = b.save_envs()
    ids = torch.arange(n, dtype=torch.int32, device=b.device)
    per, counts = live_bytes(rec)
    total = float(per.sum())

    def go():
        b.save_envs(ids, out=rec)
        b.load_envs(rec, ids, check=False)
    for _ in range(5):
        go()
    med, lo, hi = timed(go, 40, flush)
    # one step of the same batch (the round trip's yardstick), same flushing
    t = [0]

    def step():
        b.step(leaf_idx=b.random_policy(2, t[0]))
        t[0] += 1
    step_med, _, _ = timed(step, 40, flush)
    moved = 4 * total  # save: read state + write records; load: read records + write state
    gbs = moved / (med * 1e-3) / 1e9
    out = dict(n_envs=n, record_bytes=b.record_bytes, live_bytes_per_env=total / n, mean_counts=counts, l2_flushed=flush is not None,
               round_trip_ms=med, round_trip_ms_min=lo, round_trip_ms_max=hi, bytes_moved=moved, gb_s=gbs, share_of_hbm_peak=gbs / (HBM_TBS * 1e3),
               step_ms=step_med, round_trip_over_step=med / step_med)
    b.close()
    return out


def branching(n_src=1024, k=50):
    n = n_src * k
    b = pct_b200.PctBatch(n, 1, item_set=ITEMS, seed=4)
    b.reset()
    for t in range(30):
        b.step(leaf_idx=b.random_policy(1, t))
    src = torch.arange(0, n, k, device=b.device).repeat_interleave(k)
    rec = torch.empty((n, b.record_bytes), dtype=torch.uint8, device=b.device)
    ids = torch.arange(n, dtype=torch.int32, device=b.device)
    child = torch.arange(k, dtype=torch.int32, device=b.device).repeat(n_src)

    def go():
        b.save_envs(src, out=rec)
        b.load_envs(rec, ids, check=False)
        b.step(leaf_idx=child)
    for _ in range(3):
        go()
    med, lo, hi = timed(go, 20)
    b.close()
    return dict(sources=n_src, children_per_source=k, ms=med, ms_min=lo, ms_max=hi, child_env_steps_per_s=n / (med * 1e-3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_snapshot: needs the GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    flush = torch.zeros(64 << 20, dtype=torch.int32, device="cuda")  # 256 MB, overwritten before every timed repetition
    res = dict(gpu=smi, round_trip=[round_trip(4096, flush), round_trip(16384, None)], branching=branching())
    os.makedirs(a.out, exist_ok=True)
    line = json.dumps(res)
    with open(os.path.join(a.out, "bench_snapshot.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
