#!/usr/bin/env python
"""bench.py — env-steps/s of the batched PCT step (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--setting S] [--envs-per-gpu E] [--continuous] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE batched environment step over all envs of a rank: the synthetic uniform-valid-leaf policy kernel + the PCT step
kernels (action -> placement -> EMS update -> candidate leaves -> feasibility -> observation / reward / done, with auto-reset).

Headline workload (`value`, `e2e`, `roofline`, `vec_env`) = BASELINE.json configs[1]: setting 1 discrete, 10x10x10 bin, items {1..5}^3,
80 internal / 50 leaf holders, EMS scheme, 4096 envs per GPU; weak scaling (env streams keyed by the GLOBAL env index).
The same JSON line carries the other BASELINE configs as sub-records under `configs` (device-timed exactly like `value`):
    N = 1:  "3" setting 2 / 8192 envs, "4" continuous / 4096 envs, "5_shard" setting 1 / 8192 envs (one GPU's shard of config 5)
    N > 1:  "5" setting 1 / 8192 envs per GPU (N = 8: the 65 536 envs of config 5), and `allgather` = the one optional collective
            of the path (NCCL all-gather of the rollout observation buffer), timed separately — the step itself has no collective.

`value`    : device-timed (CUDA events, L2 flushed between steps, max over ranks), inputs resident in HBM.
`e2e`      : the same metric through the C-ABI host-buffer call (pct_step_host): actions come from pinned host memory, observation /
             reward / done / info land in pinned host memory every step and the policy runs on the host from those records.
`vec_env`  : the same metric through the reference-facing VecEnv surface (PctVecEnv.step: device observation, host reward / done / infos).
`roofline` : HBM roofline of the dominant kernel group, algorithmic bytes per launch (DESIGN.md section 5) / its mean duration measured here
             with CUDA events (second pass with events between the kernels).
`--dump-outputs DIR`: after the timed steps, what the last timed step of the headline returned (rank 0) is written as DIR/<name>.npy, so
             that two builds can be compared output for output on identical seeded inputs (see dump_outputs).
`cpu_baseline` / `--impl reference`: the CPU restatement of the reference env (oracle/, C, pthreads over envs like the reference's
             ShmemVecEnv workers) on this box's host cores; >= 3 repeats of >= 1 s each, median reported (min / max beside it).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ITEM_SET = [(i, j, k) for i in range(1, 6) for j in range(1, 6) for k in range(1, 6)]  # givenData.py:7-14
ITEM_SEED, POLICY_SEED = 1234, 4321
METRIC = "env-steps/s (batched PCT step)"
PREROLL = 256  # steps after the synchronised reset before anything is timed: the batch reaches its steady-state episode mix
DUMP_LIMIT = 63 * 10 ** 6  # array bytes written by --dump-outputs at most: under 64 MB with the .npy headers


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--setting", type=int, default=1)
    ap.add_argument("--envs-per-gpu", type=int, default=4096)
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between steps (diagnostic only)")
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="headline only: no sub-records for the other BASELINE configs")
    ap.add_argument("--continuous", action="store_true", help="BASELINE config 4: PctContinuous, sample_from_distribution, bin 1x1x1")
    ap.add_argument("--preroll", type=int, default=PREROLL)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (--impl ours)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def workload_name(setting, continuous, envs_per_gpu, n_gpus):
    if continuous:
        return "setting %d continuous (sample_from_distribution U(0.1,0.5)), bin 1x1x1, 80 internal / 50 leaf, EMS, %d envs/GPU x %d GPU" % (
            setting, envs_per_gpu, n_gpus)
    return "setting %d discrete, bin 10x10x10, items 1-5, 80 internal / 50 leaf, EMS, %d envs/GPU x %d GPU" % (setting, envs_per_gpu, n_gpus)


# ------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx, self.rows, self.stop_flag, self.proc = gpu_index, [], False, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """DRAM bytes per launch of the kernels from the committed ncu captures (profiles/traffic.json: per kernel, with the commit they were taken at)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------------------
def cpu_port_rate(setting, n_envs, min_steps, threads=None, continuous=False, min_seconds=1.0, repeats=3, warm_seconds=0.5):
    """The CPU arm: the C restatement of the reference env (oracle/), one pthread per host core over the envs.  Warm up for >= warm_seconds,
    then `repeats` timed runs of >= min_steps vector steps AND >= min_seconds each (run length adapted from the warm-up rate).
    -> dict(value = median env-steps/s, min, max, runs, steps_per_run, seconds, cores)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pct_oracle  # the ONLY place bench.py touches oracle/: the CPU baseline / reference arm
    if continuous:  # BASELINE config 4: PackingContinuous, sample_from_distribution U(0.1, 0.5), unit container
        b = pct_oracle.OracleBatchContinuous(n_envs, setting, ITEM_SEED, POLICY_SEED, threads=threads)
    else:
        b = pct_oracle.OracleBatch(n_envs, setting, ITEM_SET, ITEM_SEED, POLICY_SEED, threads=threads)
    warm_steps, warm_t = 0, 0.0
    chunk = max(4, min_steps // 4)
    while warm_t < warm_seconds:
        warm_t += b.run(chunk)
        warm_steps += chunk
    per_step = warm_t / warm_steps
    steps = max(int(min_steps), int(min_seconds / per_step) + 1)
    rates, secs = [], []
    for _ in range(repeats):
        dt = b.run(steps)
        rates.append(n_envs * steps / dt)
        secs.append(dt)
    cores = b.threads
    b.close()
    rates_sorted = sorted(rates)
    return {"value": rates_sorted[len(rates_sorted) // 2], "min": rates_sorted[0], "max": rates_sorted[-1], "runs": rates, "steps_per_run": steps,
            "seconds": secs, "cores": cores, "warm_steps": warm_steps}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = a.envs_per_gpu * a.gpus  # whole-job workload of the GPU arm, stepped by all host threads
    r = cpu_port_rate(a.setting, n, max(a.steps, 1), continuous=a.continuous)
    rate = r["value"]
    sample = "%d envs x %d vector steps per run, %d runs of %.2f-%.2f s (median; min %.3g, max %.3g env-steps/s) after %d warm-up steps" % (
        n, r["steps_per_run"], len(r["runs"]), min(r["seconds"]), max(r["seconds"]), r["min"], r["max"], r["warm_steps"])
    line = {"metric": METRIC, "value": rate, "unit": "env-steps/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "timed_steps_per_run": r["steps_per_run"], "warmup_steps_run": r["warm_steps"], "ms_per_step": 1e3 * n / rate, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if a.continuous else "int32+f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(a.setting, a.continuous, a.envs_per_gpu, a.gpus),
                       "note": "reference's CPU env path: C restatement (oracle/, kind=port; the reference itself is pure Python and does not "
                               "travel to the GPU box), pthreads over envs like ShmemVecEnv workers; --steps is the MINIMUM run length: every "
                               "timed run lasts >= 1 s, median of 3"},
            "cpu_baseline": {"value": rate, "unit": "env-steps/s", "cores": r["cores"], "kind": "port", "sample": sample,
                             "min": r["min"], "max": r["max"]},
            "e2e": {"value": rate, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
class Ctx(object):
    pass


def make_batch(setting, continuous, n, rank, local):
    import pct_b200
    if continuous:
        return pct_b200.PctBatch(n, setting, container_size=(1.0, 1.0, 1.0), continuous=True, sample_from_distribution=True,
                                 seed=ITEM_SEED, env_id_base=rank * n, device=local)
    return pct_b200.PctBatch(n, setting, item_set=ITEM_SET, seed=ITEM_SEED, env_id_base=rank * n, device=local)


def measure(cx, setting, continuous, n, K, W, preroll, kernels=True, keep=False, last=None):
    """Device-timed throughput of one configuration on this rank's GPU (all ranks call it together): reset, `preroll` + W untimed steps,
    K timed steps (CUDA events per step, L2 flushed before each, barrier on both sides), then — discrete only — a second pass of K steps
    with events between the kernels for the per-kernel durations.  If `last` is a dict, it receives copies of what the last timed step
    returned (leaf indices of the policy kernel, observation, reward, done, info), taken before the second pass overwrites them."""
    import torch
    batch = make_batch(setting, continuous, n, cx.rank, cx.local)
    batch.reset()
    for t in range(preroll + W):
        batch.step(leaf_idx=batch.random_policy(POLICY_SEED, t))
    torch.cuda.synchronize()
    T0 = preroll + W
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    stats = torch.zeros((4,), dtype=torch.float64, device=cx.dev)  # sums of counter, n_leaf, n_cand, n_ems
    cx.barrier()
    l0 = batch.kernel_launches
    t_wall0 = time.perf_counter()
    for t in range(K):
        if cx.flush is not None:
            cx.flush.zero_()  # L2 flush (256 MiB > 126 MB L2), outside the timed interval of the step
        ev[t][0].record()
        idx = batch.random_policy(POLICY_SEED, T0 + t)
        ev[t][1].record()
        obs, rew, done, info = batch.step(leaf_idx=idx)
        ev[t][2].record()
        if t % 16 == 0:
            stats += torch.stack([info[:, 0].double().mean(), info[:, 5].double().mean(), info[:, 6].double().mean(), info[:, 7].double().mean()])
    cx.barrier()
    wall = time.perf_counter() - t_wall0
    launches = batch.kernel_launches - l0
    if last is not None:
        last.update(zip(("leaf_idx", "obs", "reward", "done", "info"), (x.clone() for x in (idx, obs, rew, done, info))))
    kms, ksteps = {}, 0
    if kernels and not continuous:
        batch.profile(True)
        for t in range(K):
            if cx.flush is not None:
                cx.flush.zero_()
            batch.step(leaf_idx=batch.random_policy(POLICY_SEED, T0 + K + t))
        torch.cuda.synchronize()
        kms, ksteps = batch.profile_read()
        batch.profile(False)
    per_step = sorted(ev[t][0].elapsed_time(ev[t][2]) for t in range(K))
    step_ms = sum(per_step)
    kern_ms = sum(ev[t][1].elapsed_time(ev[t][2]) for t in range(K))
    tt = torch.tensor([step_ms, kern_ms], dtype=torch.float64, device=cx.dev)
    per_rank = None
    if cx.dist is not None:
        allr = [torch.zeros_like(tt) for _ in range(cx.world)]
        cx.dist.all_gather(allr, tt)  # every rank's own device time: the spread attributes the weak-scaling loss (the step has no collective)
        per_rank = [float(x[0]) / K for x in allr]
        cx.dist.all_reduce(tt, op=cx.dist.ReduceOp.MAX)
    step_ms, kern_ms = float(tt[0]), float(tt[1])
    nsamp = len(range(0, K, 16))
    mean_boxes, mean_leaf, mean_cand, mean_ems = [float(x) / nsamp for x in stats.cpu()]
    rec = {"value": cx.world * n * K / (step_ms * 1e-3), "ms_per_step": step_ms / K, "kernel_ms_per_step": kern_ms / K,
           "ms_per_step_p50": per_step[K // 2], "ms_per_step_p99": per_step[min(K - 1, int(K * 0.99))], "wall_s_timed_loop": wall,
           "gpu_launches": int(launches), "mean_boxes": mean_boxes, "mean_ems": mean_ems, "mean_valid_leaves": mean_leaf,
           "mean_candidates": mean_cand, "kernel_ms": {k: v / ksteps for k, v in kms.items()} if ksteps else None, "steps": K, "warmup": W,
           "preroll": preroll, "envs_per_gpu": n}
    if per_rank:
        rec["per_rank_ms_per_step"] = per_rank  # value uses the MAX: a launch lasts as long as its heaviest env, and N ranks sample N times more tails
    if keep:
        return rec, batch
    batch.close()
    return rec


def roofline_of(rec, setting, continuous, n, obs_len, delta_obs):
    """HBM roofline of the dominant kernel group from the per-kernel CUDA-event durations; algorithmic bytes per env as in DESIGN.md section 5."""
    peak, peak_src = measured_peak()
    hot, prefix, stage = 3584, 2576, 1040  # sizeof(DEnvHot), HOT_PREFIX, header + boxes
    stab = setting != 2
    nb_, nl_, nc_ = rec["mean_boxes"], rec["mean_valid_leaves"], rec["mean_candidates"]
    edges = nb_ if stab else 0.0
    loads = (32 * edges + 16 * 0.3 * edges) if stab else 0.0
    walks = 0.45 * nc_ if stab else 0.0  # candidates that need a stability walk (host statistics of the BASELINE streams: 45 %)
    obs_b = (max(nb_, 1.0) + nl_ + 1.0) * 36.0 if delta_obs else obs_len * 4.0
    groups = {
        "apply": 2 * hot + 2 * loads + 4 + 4 + 1 + 32,
        "candidates": prefix + 2 * nc_ + 4 * (nc_ / 32.0 + 1) + 20 * walks,
        "feas_emit": 20 * walks + (hot + loads if stab else 0) + stage + 2 * nc_ + 4 * (nc_ / 32.0 + 1) + 12 * nl_ * 2 + obs_b + 32,
    }
    b_step = sum(groups.values())
    out = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src, "algorithmic_bytes_per_env_step": b_step,
           "step_achieved": b_step * n / (rec["kernel_ms_per_step"] * 1e-3) / 1e9}
    out["step_fraction_of_peak"] = out["step_achieved"] / peak
    km = rec.get("kernel_ms")
    if km:
        dom = max(km, key=lambda k: km[k])
        ach = groups[dom] * n / (km[dom] * 1e-3) / 1e9
        names = {"apply": "pct_apply_kernel", "candidates": "pct_candidates_kernel (+ classify)",
                 "feas_emit": "pct_walk_light_kernel + pct_walk_kernel + pct_emit_kernel"}
        out.update(achieved=ach, frac=ach / peak, kernel=names[dom], kernel_ms=km[dom], algorithmic_bytes_per_env_kernel=groups[dom],
                   all_kernels_ms=km,
                   all_kernels_frac={k: groups[k] * n / (km[k] * 1e-3) / 1e9 / peak for k in km},
                   kernel_timing="second pass of %d steps right after the timed region with CUDA events between the kernel groups; the events "
                                 "serialise the kernels, the timed region itself overlaps apply -> candidates (programmatic dependent launch + "
                                 "per-env hand-over flags), so ms_per_step < sum of these" % rec["steps"])
    else:
        out.update(achieved=out["step_achieved"], frac=out["step_fraction_of_peak"], kernel="whole step (continuous kernels: pctc_apply / pctc_candidates / pctc_feas_emit)",
                   kernel_ms=rec["kernel_ms_per_step"])
    # SURVEY.md 8(d) / BASELINE.md 3.5 figure for the WHOLE step, independent of this implementation's record layout
    b_survey = 5593.0 + 24.0 * nb_ + 48.0 * rec["mean_ems"]
    ach_survey = b_survey * n / (rec["kernel_ms_per_step"] * 1e-3) / 1e9
    out["survey_formula"] = {"bytes_per_env_step": b_survey, "achieved": ach_survey, "frac": ach_survey / peak,
                             "note": "SURVEY 8(d): (5593 + 24 N + 48 E) B x env-steps/s of one GPU / peak, whole step"}
    tr = ncu_traffic()
    out["traffic"] = None
    if tr and not continuous:
        ks = [k for k in tr.get("kernels", {}) if k in out["kernel"]]  # the kernels of the dominant group
        if ks:
            out["traffic"] = sum(tr["kernels"][k]["dram_bytes_per_launch"] for k in ks)
            out["traffic_source"] = "dram__bytes_read + write of %s from the ncu --set full captures of %s (profiles/%s; 4096 envs, setting 1, caches flushed per replay)" % (
                " + ".join(ks), tr.get("commit"), tr.get("file"))
        out["traffic_all_kernels"] = {k: v["dram_bytes_per_launch"] for k, v in tr.get("kernels", {}).items()}
        out["traffic_step_total"] = tr.get("step_total_dram_bytes")
    return out


def dump_outputs(dirname, last):
    """Writes the arrays of `last` (see measure) as DIR/<name>.npy: observation and reward in float32 as returned, done in float32, leaf
    indices and the raw int32 info records (include/pct_b200.h pct_step_info) in float64, both exact.  If they exceed DUMP_LIMIT, the
    same fixed seeded sample of envs is taken from each, and its env indices are written as env_index.npy."""
    import numpy as np
    arrays = {"leaf_idx": last["leaf_idx"].cpu().numpy().astype(np.float64), "obs": last["obs"].float().cpu().numpy(),
              "reward": last["reward"].float().cpu().numpy(), "done": last["done"].cpu().numpy().astype(np.float32),
              "info": last["info"].cpu().numpy().astype(np.float64)}
    n = len(arrays["obs"])
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        rows = np.sort(np.random.default_rng(0).choice(n, n * DUMP_LIMIT // (total + 8 * n), replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), v)


def run_ours(a):
    import numpy as np
    import torch
    import pct_b200

    cx = Ctx()
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local = int(os.environ.get("LOCAL_RANK", "0"))
    cx.dist = None
    if cx.world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(cx.local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", cx.local))
        cx.dist = dist
    torch.cuda.set_device(cx.local)
    cx.dev = torch.device("cuda", cx.local)
    cx.flush = None if a.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=cx.dev)

    def barrier():
        if cx.dist is not None:
            cx.dist.barrier()
        torch.cuda.synchronize()
    cx.barrier = barrier
    world, rank, local, dev = cx.world, cx.rank, cx.local, cx.dev
    n = a.envs_per_gpu
    K, W = a.steps, max(a.warmup, 3)
    switches = {k: v for k, v in sorted(os.environ.items()) if k.startswith("PCT_B200_")}
    delta_obs = os.environ.get("PCT_B200_OBS_DELTA", "1") != "0" and not a.continuous
    zero_copy = os.environ.get("PCT_B200_HOST_ZEROCOPY", "1") != "0"

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    last = {} if a.dump_outputs and rank == 0 else None
    head, batch = measure(cx, a.setting, a.continuous, n, K, W, a.preroll, keep=True, last=last)
    clocks = sampler.finish() if sampler else None
    if last:
        dump_outputs(a.dump_outputs, last)
    ol = batch.obs_len

    # ---- e2e: host buffers through pct_step_host, host policy on the returned records ----
    Ke, We = max(3, min(a.e2e_steps, K)), 5
    obs_h = torch.empty((n, ol), dtype=torch.float32, pin_memory=True).numpy()
    rew_h = torch.empty((n,), dtype=torch.float32, pin_memory=True).numpy()
    done_h = torch.empty((n,), dtype=torch.uint8, pin_memory=True).numpy()
    info_h = torch.empty((n, 8), dtype=torch.int32, pin_memory=True).numpy()
    idx_h = torch.empty((n,), dtype=torch.int32, pin_memory=True).numpy()
    gid = (np.arange(n, dtype=np.uint64) + np.uint64(rank * n))
    GOLD = np.uint64(0x9E3779B97F4A7C15)

    def sm64(x):
        with np.errstate(over="ignore"):
            x = x + GOLD
            z = x
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            return z ^ (z >> np.uint64(31))

    with np.errstate(over="ignore"):
        pol_base = sm64(np.uint64(POLICY_SEED) ^ (gid * GOLD))  # the per-env half of rnd_u64(seed, env, t): constant over the run

    def host_policy(t):
        # uniform choice among the valid leaves, on the HOST from the step's returned records: the number of valid leaf rows
        # is pct_step_info.n_leaf (== the count of 1s in column 8 of the leaf rows of the returned observation)
        nvalid = info_h[:, 5].astype(np.uint64)
        with np.errstate(over="ignore"):
            r = sm64(pol_base + np.uint64(t))
        idx_h[:] = np.where(nvalid > 0, r % np.maximum(nvalid, np.uint64(1)), 0).astype(np.int32)

    batch.reset_host(obs_h)
    info_h[:, 5] = (obs_h.reshape(n, -1, 9)[:, batch.nb:batch.nb + batch.nl, 8] == 1).sum(1)  # first step: count from the observation
    for t in range(We):
        host_policy(t)
        batch.step_host(obs_h, rew_h, done_h, info_h, leaf_idx=idx_h)
    barrier()
    t0 = time.perf_counter()
    for t in range(Ke):
        host_policy(We + t)
        batch.step_host(obs_h, rew_h, done_h, info_h, leaf_idx=idx_h)
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    te = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    if cx.dist is not None:
        cx.dist.all_reduce(te, op=cx.dist.ReduceOp.MAX)
    e2e_value = world * n * Ke / float(te[0])
    h2d = idx_h.nbytes
    rows_changed = (max(head["mean_boxes"], 1.0) + head["mean_valid_leaves"] + 1.0) * 36.0
    d2h_full = obs_h.nbytes + rew_h.nbytes + done_h.nbytes + info_h.nbytes
    d2h = int(n * rows_changed + rew_h.nbytes + done_h.nbytes + info_h.nbytes) if (delta_obs and zero_copy) else d2h_full
    batch.close()

    # ---- the reference-facing VecEnv surface: PctVecEnv.step (device observation; reward / done / infos on the host, one sync per step) ----
    vec = None
    try:
        kw = dict(container_size=(1.0, 1.0, 1.0), continuous=True, sample_from_distribution=True) if a.continuous else dict(item_set=ITEM_SET)
        venv = pct_b200.PctVecEnv(n, a.setting, seed=ITEM_SEED, env_id_base=rank * n, device=local, **kw)
        venv.reset()
        Kv = max(3, min(a.e2e_steps, K))
        n_done = 0
        for t in range(20):
            venv.step(venv.batch.random_policy(POLICY_SEED, t))
        barrier()
        t0 = time.perf_counter()
        for t in range(Kv):
            _, _, d_, infos = venv.step(venv.batch.random_policy(POLICY_SEED, 20 + t))
            if t % 5 == 4:  # train_tools.py:63-79: after every num_steps (= 5, tools.py) steps the trainer reads the LAST step's infos of the finished envs
                for i in np.nonzero(d_)[0]:
                    n_done += 1 if "ratio" in infos[i] else 0
        torch.cuda.synchronize()
        tv = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if cx.dist is not None:
            cx.dist.all_reduce(tv, op=cx.dist.ReduceOp.MAX)
        vec = {"value": world * n * Kv / float(tv[0]), "unit": "env-steps/s", "steps": Kv, "episodes_read": n_done,
               "path": "PctVecEnv.step(leaf indices on the device): device observation (fresh tensor per step), reward / done / lazy infos on the "
                       "host, finished envs' info dicts materialised after every 5th step like the trainer's n-step loop (train_tools.py:63-79); wall clock"}
        venv.close()
    except Exception as ex:  # never fail the headline on the convenience surface
        vec = {"value": None, "error": repr(ex)}

    # ---- the other BASELINE configs, device-timed the same way ----
    configs = {}
    default_head = (a.setting == 1 and not a.continuous and n == 4096)
    Kc, Wc = max(20, min(K, 300)), W
    if not a.skip_configs and default_head:
        if world == 1:
            plan = [("3", 2, False, 8192), ("4", 1, True, 4096), ("5_shard", 1, False, 8192)]
        else:
            plan = [("5", 1, False, 8192)]
        for key, s_, c_, n_ in plan:
            r = measure(cx, s_, c_, n_, Kc, Wc, a.preroll)
            r["workload"] = workload_name(s_, c_, n_, world)
            if rank == 0:
                r["roofline"] = roofline_of(r, s_, c_, n_, ol, (not c_) and os.environ.get("PCT_B200_OBS_DELTA", "1") != "0")
            configs[key] = r

    # ---- the one optional collective of the path: NCCL all-gather of the rollout observation buffer (not part of the step) ----
    allgather = None
    if cx.dist is not None:
        from pct_b200.distributed import gather_observations
        o_loc = torch.zeros((8192 if default_head else n, ol), dtype=torch.float32, device=dev)
        for _ in range(3):
            gather_observations(o_loc)
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        reps = 20
        evs[0].record()
        for _ in range(reps):
            g_all = gather_observations(o_loc)
        evs[1].record()
        barrier()
        tg = torch.tensor([evs[0].elapsed_time(evs[1]) / reps], dtype=torch.float64, device=dev)
        cx.dist.all_reduce(tg, op=cx.dist.ReduceOp.MAX)
        allgather = {"ms": float(tg[0]), "bytes_per_rank": int(o_loc.numel() * 4), "bytes_gathered": int(g_all.numel() * 4),
                     "algbw_GBps": g_all.numel() * 4 / (float(tg[0]) * 1e-3) / 1e9,
                     "note": "optional rollout-buffer gather (pct_b200.distributed.gather_observations); NOT inside `value`: the step has no collective"}

    if rank == 0:
        roof = roofline_of(head, a.setting, a.continuous, n, ol, delta_obs)
        line = {"metric": METRIC, "value": head["value"], "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 geometry and stability, f32 observations" if a.continuous else "int16/int32 geometry + f64 stability, f32 observations",
                "data": "synthetic",
                "config": {"workload": workload_name(a.setting, a.continuous, n, world),
                           "items": "device counter-based RNG seed %d, uniform over 125 sizes" % ITEM_SEED,
                           "policy": "uniform over valid leaves (device kernel)",
                           "launch_mode": os.environ.get("PCT_B200_OVERLAP", "1") != "0" and "overlapped apply -> candidates (PDL + per-env flags), pooled walks"
                                          or "back-to-back kernels",
                           "l2": "not flushed (diagnostic)" if a.no_flush else "flushed between steps (256 MiB memset outside the timed interval)",
                           "phase": "steady-state episode mix: %d pre-roll steps after the synchronised reset, then %d warm-up steps, then the timed steps" % (a.preroll, W),
                           "mean_boxes": head["mean_boxes"], "mean_ems": head["mean_ems"], "mean_valid_leaves": head["mean_valid_leaves"],
                           "mean_candidates": head["mean_candidates"], "switches": switches},
                "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "d2h_bytes_per_step_full_observation": int(d2h_full), "steps": Ke,
                        "path": ("pct_step_host (C ABI, pinned host buffers, zero-copy: the emit kernel writes the changed observation rows straight into the "
                                 "mapped host buffer)" if zero_copy else "pct_step_host (C ABI, pinned host buffers, 4 pipelined env ranges)")
                                + " + numpy policy on the host from the returned step records"},
                "vec_env": vec,
                "gpu_launches": head["gpu_launches"], "kernel_ms_per_step": head["kernel_ms_per_step"],
                "ms_per_step_p50": head["ms_per_step_p50"], "ms_per_step_p99": head["ms_per_step_p99"], "wall_s_timed_loop": head["wall_s_timed_loop"],
                "roofline": roof, "clocks": clocks, "configs": configs}
        if head.get("per_rank_ms_per_step"):
            line["per_rank_ms_per_step"] = head["per_rank_ms_per_step"]
        if allgather:
            line["allgather"] = allgather
        if world == 1 and not a.skip_cpu:
            try:
                r = cpu_port_rate(a.setting, 4096, 50, continuous=a.continuous)
                line["cpu_baseline"] = {"value": r["value"], "unit": "env-steps/s", "cores": r["cores"], "kind": "port", "min": r["min"], "max": r["max"],
                                        "sample": "4096 envs x %d vector steps per run, %d runs of %.2f-%.2f s (median) after %d warm-up steps, same items / policy"
                                                  % (r["steps_per_run"], len(r["runs"]), min(r["seconds"]), max(r["seconds"]), r["warm_steps"])}
            except Exception as ex:  # the oracle is test infrastructure; never fail the GPU number on it
                line["cpu_baseline"] = {"value": None, "error": str(ex)}
        print(json.dumps(line))
    if cx.dist is not None:
        cx.dist.barrier()
        cx.dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
