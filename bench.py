"""bench.py -- scheduling decisions/sec of the batched env on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs C3,C4,C5|none]
                    [--dump-outputs DIR]

Headline (the JSON line's top-level keys) = BASELINE.json configs[1], "C2": 4096 environments per GPU, 50 jobs x 10
executors, fair scheduler (RoundRobinScheduler(10, dynamic_partition=True)), synthetic TPC-H-shaped bank (SURVEY.md
App. D), env seeds 1234 + i, auto-reset with seed + 4096 * reset_count.  One "step" = every environment takes
DECISIONS_PER_STEP scheduling decisions (policy evaluation, step(), observation construction, amortised resets
included).

  value    : decisions/s of the fused on-device rollout (state resident in HBM; one launch per step)
  e2e      : decisions/s through the host-buffer C ABI (ssb_step_fair_host): per decision batch the host's actions go
             H2D, the B observation headers (reward / terminated / ...) and the next actions come back D2H
  e2e_obs  : the same loop with the observation GRAPHS of all envs copied to the host every call (ssb_get_obs_host:
             nodes, edge links, dag_ptr, supplies, packed) -- what a host policy that reads dag_batch pays
  roofline : algorithmic HBM bytes of the rollout kernel (SURVEY.md 8d formula, counters measured by the kernel
             itself) / its CUDA-event duration, against MEASURED_PEAKS.json
  cpu_baseline : the C oracle port (oracle/sim_oracle.c) on the box's host cores, same workload
  --impl reference : only that CPU arm, as its own JSON line
  --dump-outputs DIR : after the headline's timed steps, what a caller of the fused rollout holds after the last of them
             (dump_outputs), as DIR/<name>.npy; inputs depend on the arguments only, so two builds can be compared

"configs" (same JSON line) carries short runs of the other BASELINE.json configurations, each with its own value,
roofline, cpu_baseline and e2e:
  C3 : Decima GNN policy rollouts per config/decima_tpch.yaml (50 executors, 200 jobs, mean time limit 2e7 ms),
       16 384 envs on one GPU, observation adapter + policy + sampling + step on the device          (N = 1 only)
  C4 : continuous Poisson arrivals, 200 jobs x 50 executors, fair scheduler, 8 192 envs per GPU (65 536 on 8 GPUs)
  C5 : C3's rollout collection on every GPU + the learner's exchanges over NCCL: rollout statistics once per
       iteration and the 20 802-float gradient all-reduce of a PPO mini-batch update on the device
"""
from __future__ import annotations

import argparse
import json
import os
import os.path as osp
import subprocess
import sys
import threading
import time

import numpy as np

REPO = osp.dirname(osp.abspath(__file__))
for _p in (REPO, osp.join(REPO, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

ENVS_PER_GPU = 4096
DECISIONS_PER_STEP = 128
E2E_DECISIONS_PER_STEP = 32
ENV_CFG = {"num_executors": 10, "job_arrival_cap": 50, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}  # examples.py:15-23
C3_CFG = {"num_executors": 50, "job_arrival_cap": 200, "job_arrival_rate": 4.0e-5,
          "moving_delay": 2000.0, "warmup_delay": 1000.0}  # config/decima_tpch.yaml:80-87
C3_MEAN_TIME_LIMIT = 2.0e7
C3_ENVS, C4_ENVS = 16384, 8192
METRIC = "scheduling decisions/sec (batched envs)"
WORKLOAD = "C2: 4096 envs/GPU x (50 jobs, 10 executors), fair scheduler, synthetic TPC-H bank"
DTYPE = "f64 event times + integer state"


def peaks():
    path = osp.join(REPO, "MEASURED_PEAKS.json")
    if osp.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tensor": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1402.8))),
                "src": "measured (MEASURED_PEAKS.json hbm_gbs / bf16_tflops_sustained)"}
    return {"hbm": 6650.0, "tensor": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def algorithmic_bytes(st: dict) -> float:
    """SURVEY.md 8(d): B_dec = 80*eps + 20*N*sigma + (12 N + 8 M + 8 Ja + 16), summed over the
    observations / events / schedulability scans the kernel counted."""
    obs = max(st["observations"], 1)
    mean_nodes = st["sum_nodes"] / obs
    return (80.0 * st["events"] + 20.0 * mean_nodes * st["sched_scans"]
            + 12.0 * st["sum_nodes"] + 8.0 * st["sum_edges"] + 8.0 * st["sum_jobs"] + 16.0 * obs)


def _traffic(key=None):
    """DRAM bytes per launch of the rollout kernel from the committed ncu summary (None if absent)."""
    tpath = osp.join(REPO, "profiles", "rollout_traffic.json")
    if not osp.exists(tpath):
        return None
    with open(tpath) as f:
        d = json.load(f)
    return (d.get(key) or {}).get("dram_bytes_per_launch") if key else d.get("dram_bytes_per_launch")


def hbm_roofline(st: dict, kern_ms: float, launches: int, kernel: str, traffic=None) -> dict:
    pk = peaks()
    alg = algorithmic_bytes(st)
    achieved = alg / (kern_ms * 1e-3) / 1e9
    obs = max(st["observations"], 1)
    return {
        "bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": pk["hbm"], "unit": "GB/s",
        "frac": achieved / pk["hbm"], "traffic": traffic, "peak_source": pk["src"],
        "algorithmic_bytes_per_launch": alg / max(launches, 1), "launches": launches,
        "bytes_per_decision": alg / max(st["decisions"], 1),
        "events_per_decision": st["events"] / max(st["decisions"], 1),
        "sched_scans_per_decision": st["sched_scans"] / max(st["decisions"], 1),
        "mean_nodes": st["sum_nodes"] / obs, "mean_edges": st["sum_edges"] / obs,
        "mean_active_jobs": st["sum_jobs"] / obs,
        "note": "latency/dependency-bound event chains: the HBM fraction is expected to be small",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arms
def cpu_arm(seconds: float, threads: int | None = None, cfg: dict | None = None, label: str = "C2") -> dict:
    """The CPU oracle port on host threads: fair episodes of `cfg` back to back, seeds 1234 + i."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import OracleEnv
    from spark_sched_sim_b200.bank import synthetic_bank

    cfg = cfg or ENV_CFG
    bank = synthetic_bank(0)
    P = threads or os.cpu_count() or 1
    envs = [OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                      cfg["job_arrival_rate"]) for _ in range(P)]
    envs[0].run_fair_episode(1234)  # warm-up
    deadline = time.perf_counter() + seconds

    def work(rank):
        dec = ev = eps = 0
        k = 0
        while time.perf_counter() < deadline:
            d, e = envs[rank].run_fair_episode(1234 + rank + P * k)  # ctypes releases the GIL
            dec += d; ev += e; eps += 1; k += 1
        return dec, ev, eps

    t0 = time.perf_counter()
    with ThreadPoolExecutor(P) as ex:
        res = list(ex.map(work, range(P)))
    dt = time.perf_counter() - t0
    dec = sum(r[0] for r in res); ev = sum(r[1] for r in res); eps = sum(r[2] for r in res)
    return {"value": dec / dt, "unit": "decisions/s", "cores": P, "kind": "port",
            "sample": f"{eps} fair {label} episodes ({dec} decisions, {ev} events) in {dt:.1f} s on {P} "
                      f"host threads, oracle/sim_oracle.c incl. reset and observation building",
            "events_per_s": ev / dt}


def _decima_cpu_worker(args):
    """One host process of the Decima CPU arm: the C oracle env + the numpy restatements of DecimaObsWrapper and
    DecimaScheduler.schedule (oracle/decima_obs.py, oracle/decima_policy.py), sampled actions, for `seconds`."""
    rank, seconds, cfg, weights_path = args
    for p in (REPO, osp.join(REPO, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    try:
        import torch

        torch.set_num_threads(1)  # rollout_worker.py:93
    except Exception:
        pass
    import decima_obs
    import decima_policy
    from oracle import OracleEnv
    from spark_sched_sim_b200.bank import synthetic_bank

    E = cfg["num_executors"]
    w = decima_policy.load_weights(weights_path)
    env = OracleEnv(synthetic_bank(0), E, cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                    cfg["job_arrival_rate"])
    rng = np.random.default_rng(1000 + rank)
    dec, k = 0, 0
    t0 = time.perf_counter()
    obs = env.reset_seed(1234 + rank)
    while time.perf_counter() - t0 < seconds:
        d = decima_obs.decima_observation(obs, E)
        h, h_dag, h_glob = decima_policy.encode(w, d["features"], obs["edge_links"], d["edge_bits"], d["depth"],
                                                obs["dag_ptr"])
        ss, jobs = decima_policy.stage_scores(w, d["features"], h, h_dag, h_glob, obs["dag_ptr"], d["stage_mask"])
        pr = np.exp(ss - ss.max()); pr /= pr.sum()
        si = int(rng.choice(len(ss), p=pr))
        job = int(jobs[si])
        cap = int(d["commit_caps"][job])
        es = decima_policy.exec_scores(w, d["features"], h_dag, h_glob, obs["dag_ptr"], job, cap, E)
        pe = np.exp(es - es.max()); pe /= pe.sum()
        ne = int(rng.choice(cap, p=pe))
        rc, _, term = env.step(si, ne + 1)
        assert rc == 0, rc
        dec += 1
        if term:
            k += 1
            obs = env.reset_seed(1234 + rank + 1000 * k)
        else:
            obs = env.obs()
    return dec, time.perf_counter() - t0


def cpu_arm_decima(seconds: float, cfg: dict, label: str, procs: int | None = None) -> dict:
    """Decima decisions/s of the CPU port on all host cores: one process per core (the numpy policy holds the GIL),
    mirroring the reference's one-process-per-env rollout workers (trainers/trainer.py:264-293)."""
    import multiprocessing as mp

    P = procs or os.cpu_count() or 1
    wp = osp.join(REPO, "tests", "golden", "decima_model.npz")
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(P) as pool:
        res = pool.map(_decima_cpu_worker, [(r, seconds, cfg, wp) for r in range(P)])
    wall = time.perf_counter() - t0
    dec = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return {"value": dec / busy, "unit": "decisions/s", "cores": P, "kind": "port",
            "sample": f"{dec} Decima decisions of {label} episodes in {busy:.1f} s on {P} host processes (1 thread "
                      f"each): oracle/sim_oracle.c env + numpy DecimaObsWrapper / DecimaScheduler.schedule "
                      f"(oracle/decima_obs.py, oracle/decima_policy.py), shipped model.pt; {wall:.1f} s incl. spawn"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = 2.0
    vals = []
    for _ in range(args.warmup):
        cpu_arm(0.5)
    t0 = time.perf_counter()
    last = None
    for _ in range(args.steps):
        last = cpu_arm(per_step)
        vals.append(last["value"])
    dt = time.perf_counter() - t0
    v = float(np.mean(vals))
    last["value"] = v
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "decisions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "config": headline_config(ENVS_PER_GPU, args.gpus, None),
        "cpu_baseline": last, "reference_step": f"{per_step} s of CPU episodes",
        "e2e": {"value": v, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference is pure Python and cannot travel to the GPU box; this arm times the C "
                "port of it (oracle/), which is ~250x faster per core than the Python original "
                "(BASELINE.md: 160-210 decisions/s/core)",
    }))


def headline_config(B, world, workspace_mib):
    """`config` of the bench line -- the SAME keys and values for our arm and the reference arm (the driver compares
    them); run-specific details live in other keys of the line."""
    return {"workload": WORKLOAD, "envs_per_gpu": B, "decisions_per_env_per_step": DECISIONS_PER_STEP,
            "policy": "fair", "auto_reset": True,
            "l2": "256 MiB flush write between timed iterations (ours); n/a on the CPU arm",
            "parallelism": "envs sharded over the GPUs; all-reduce of rollout stats only"}


# ------------------------------------------------------------------------------------------ GPU pieces
class Ctx:
    pass


def barrier(cx):
    if cx.world > 1:
        cx.dist.barrier()
    cx.torch.cuda.synchronize()


def reduce_max_sum(cx, ms, counts):
    torch = cx.torch
    t = torch.tensor([ms], dtype=torch.float64, device=cx.dev)
    c = torch.tensor([float(x) for x in counts], dtype=torch.float64, device=cx.dev)
    if cx.world > 1:
        cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MAX)
        cx.dist.all_reduce(c)
    return float(t.item()), [float(x) for x in c.tolist()]


def timed_fair_rollouts(cx, env, seeds, seed_step, W, K, D, pre_decisions=0):
    """W warm-up + K timed steps of the fused fair rollout (D decisions per env and step), each followed on the
    device by ssb_collect_stats into row k of a [K, 8] buffer; the path's only exchange -- the NCCL all-reduce of those
    statistics (the learner's view of rollout_worker.py:122-129) -- is ONE call over the whole buffer after the last
    step, inside the timed region.  (Not overlapped with the rollouts on a side stream: the rollout kernel needs all
    its CTAs resident at once, and a concurrent NCCL kernel pushes its last CTAs into a second wave.)
    Returns per-rank kernel ms, stats dict, launches, the last step's reduced stats vector, wall seconds."""
    torch = cx.torch
    flush = cx.flush
    stats = torch.zeros(K, 8, dtype=torch.float64, device=cx.dev)
    env.reset_host(seeds)
    if pre_decisions:
        env.rollout_fair(pre_decisions, True, True, seed_step)  # into the episodes (see the caller's note)
    for _ in range(W):
        env.rollout_fair(D, True, True, seed_step)
    env.reset_stats()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    barrier(cx)
    t_wall0 = time.perf_counter()
    launches = 0
    for k in range(K):
        flush.fill_(k & 0xFF)  # evict L2 between timed iterations (untimed)
        ev0[k].record()
        env.rollout_fair(D, True, True, seed_step)
        env.collect_stats(stats[k])
        launches += 3  # k_rollout_fair + the two ssb_collect_stats kernels
        ev1[k].record()
    ev0[K].record()
    if cx.world > 1:
        cx.dist.all_reduce(stats)
    ev1[K].record()
    barrier(cx)
    t_wall = time.perf_counter() - t_wall0
    kern_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
    return kern_ms, env.stats(), launches, stats[K - 1], t_wall


DUMP_LIMIT = 64 << 20


def dump_outputs(env, rollout_stats, out_dir: str, limit: int = DUMP_LIMIT) -> list[str]:
    """Writes what a caller of the fused rollout holds after it, as out_dir/<name>.npy: every field of the observation
    headers (reward, wall_time, num_nodes, ...), the observation graphs (nodes, edge_links, dag_ptr, exec_supplies: the
    valid rows of each env, concatenated in env order; the header counts split them), the per-env counters since the
    last reset_stats (stats_<field>) and `rollout_stats`, the collect_stats vector as the caller holds it (with several
    ranks: after the all-reduce, i.e. summed over all ranks, while the other files hold this rank's envs).  Only
    float32 / float64 files: integers are stored as float64 (exact below 2**53).  If all envs at their buffer
    capacities do not fit in `limit` bytes, a fixed sample of them (numpy seed 0) is written, in env order; env_ids
    lists the envs written.  Which envs are written depends on the env count and capacities only, never on what the
    rollout computed, so two builds are compared on the same envs.  Returns the names written."""
    import torch

    from spark_sched_sim_b200 import _native as nat

    h = env.hdr()
    B = len(h)
    n, m, j = (h[f].astype(np.int64) for f in ("num_nodes", "num_edges", "num_active_jobs"))
    S, M, J = env.node_stride, env.edge_stride, env.job_stride
    per_env = 8 * (len(h.dtype.names) + len(nat.STATS_FIELDS) + 1) + 12 * S + 16 * M + 8 * (J + 1) + 8 * J
    fit = (limit - (8 << 10)) // per_env  # less the fixed-size rollout_stats and the .npy headers
    envs = np.arange(B) if fit >= B else np.sort(np.random.default_rng(0).permutation(B)[:fit])

    def rows(view, count):
        a = view[torch.as_tensor(envs, device=view.device)].cpu().numpy()
        return a[np.arange(a.shape[1])[None, :] < count[envs, None]]

    out = {f: h[f][envs] for f in h.dtype.names}
    out.update(nodes=rows(env.nodes, n), edge_links=rows(env.edge_links, m), dag_ptr=rows(env.dag_ptr, j + 1),
               exec_supplies=rows(env.exec_supplies, j))
    st = env.stats_per_env()
    out.update({f"stats_{f}": st[f][envs] for f in nat.STATS_FIELDS})
    out["rollout_stats"] = rollout_stats.cpu().numpy()
    out["env_ids"] = envs
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(osp.join(out_dir, name + ".npy"), v if v.dtype in (np.float32, np.float64) else v.astype(np.float64))
    return sorted(out)


def e2e_step_loop(cx, cfg, seeds, seed_step, Ke, De, budget, with_obs):
    """The caller-facing loop of a vector env through the host-buffer C ABI; with_obs: also the packed observation
    graphs of all envs every call."""
    torch = cx.torch
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B = len(seeds)
    e = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=cx.bank, device=cx.dev)
    a_pin, n_pin, a_nxt, n_nxt = (torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(4))
    e.reset_host(seeds)
    e.set_autoreset(True, seed_step)
    a0, n0 = e.fair_actions(True)   # the first actions; afterwards the step call returns them
    a_pin.copy_(a0); n_pin.copy_(n0)
    torch.cuda.synchronize()
    obs_bytes = [0]

    def steps(n_steps):
        a_h, n_h, a_o, n_o = a_pin.numpy(), n_pin.numpy(), a_nxt.numpy(), n_nxt.numpy()
        for _ in range(n_steps * De):
            # one call per decision batch: H2D of the host's actions, bounded step (envs still simulating come
            # back "pending" and continue next call; finished envs re-seed themselves, ssb_set_autoreset), the
            # fair scheduler's action for the new observation evaluated inside the step kernel, D2H of the B
            # observation headers and of those actions, one synchronisation
            e.step_fair_host(a_h, n_h, a_o, n_o, True, max_events=budget)
            if with_obs:
                po = e.obs_host()
                tn, te, tj = (int(x) for x in po["offsets"][B])
                obs_bytes[0] += 12 * (B + 1) + 12 * tn + 8 * te + 4 * (tj + B) + 4 * tj
            a_h, n_h, a_o, n_o = a_o, n_o, a_h, n_h   # the host feeds the actions it received back in

    steps(2)
    e.reset_stats()
    obs_bytes[0] = 0
    barrier(cx)
    t0 = time.perf_counter()
    steps(Ke)
    barrier(cx)
    dt = time.perf_counter() - t0
    dt, (dec,) = reduce_max_sum(cx, dt, [e.stats()["decisions"]])
    calls = Ke * De
    out = {"value": dec / dt, "unit": "decisions/s", "h2d_bytes_per_step": De * 2 * 4 * B,
           "d2h_bytes_per_step": De * (2 * 4 + 48) * B + obs_bytes[0] // max(Ke, 1),
           "steps": Ke, "calls_per_step": De, "max_events_per_call": budget, "host_threads": 1,
           "gpu_launches": calls * (3 if with_obs else 1)}
    e.close()
    return out


def run_c2(cx, args):
    """The headline: returns the top-level keys of the JSON line."""
    torch = cx.torch
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200 import parallel
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    W, K, B, D = cx.W, cx.K, args.envs, DECISIONS_PER_STEP
    env = BatchedSparkSchedSimEnv(ENV_CFG, num_envs=B, bank=cx.bank, device=cx.dev)
    seeds, seed_step = parallel.shard_seeds(1234, B, cx.rank, cx.world)  # envs shard over ranks: disjoint seeds
    sampler = ClockSampler(cx.local_rank)
    if cx.rank == 0:
        sampler.start()
    kern_ms, st, launches, stats_vec, t_wall = timed_fair_rollouts(cx, env, seeds, seed_step, W, K, D)
    clocks = sampler.stop() if cx.rank == 0 else None
    if args.dump_outputs and cx.rank == 0:
        dump_outputs(env, stats_vec, args.dump_outputs)
    n_err = int((env.hdr()["error"] != 0).sum())
    max_ms, (total_dec, total_ev, total_eps, total_err) = reduce_max_sum(
        cx, kern_ms, [st["decisions"], st["events"], st["episodes"], n_err])
    value = total_dec / (max_ms * 1e-3)
    roofline = hbm_roofline(st, kern_ms, K, "k_rollout_fair<1>", _traffic())  # K launches of the rollout kernel
    roofline["traffic_source"] = ("ncu dram__bytes_read.sum + dram__bytes_write.sum of this kernel over the timed launches "
                                  "of this command (profiles/rollout_traffic.json), mean per launch; 1.2 GB (mid-episode "
                                  "launches) .. 11.8 GB (launches in which most envs reset)")

    e2e = e2e_obs = e2e_rollout = None
    launches_e2e = 0
    if not args.no_e2e:
        Ke = max(2, min(K, 5))
        e2e = e2e_step_loop(cx, ENV_CFG, seeds, seed_step, Ke, E2E_DECISIONS_PER_STEP, args.e2e_budget, False)
        e2e["path"] = ("ssb_step_fair_host per decision batch: H2D of the host's actions -> bounded step with "
                       "auto-reset of finished envs + the fair scheduler's next action (in the step kernel) -> D2H of "
                       "the observation headers and the next actions (pinned) -> host feeds them back; the host never "
                       "reads the graph (the headline e2e: what a caller of the built-in heuristics pays)")
        e2e_obs = e2e_step_loop(cx, ENV_CFG, seeds, seed_step, 2, E2E_DECISIONS_PER_STEP, args.e2e_budget, True)
        e2e_obs["path"] = ("the same loop + ssb_get_obs_host every call: the observation graphs of all envs (nodes, "
                           "edge links, dag_ptr, supplies) packed on the device and copied D2H -- what a host policy "
                           "that consumes dag_batch pays; d2h_bytes_per_step counts the bytes actually copied")
        launches_e2e = e2e["gpu_launches"] + e2e_obs["gpu_launches"]
        # the rollout-collection call (rollout_worker.py:135-157 as ONE call): fused rollout on the device,
        # every transition (wall time, action, reward, flags) copied to pinned host memory per step
        nb = B * D * nat.TRANSITION_DTYPE.itemsize
        traj_dev = torch.empty(nb, dtype=torch.uint8, device=cx.dev)
        traj_pin = torch.empty(nb, dtype=torch.uint8).pin_memory()
        env.reset_host(seeds)
        for _ in range(2):
            env.rollout_fair_traj(D, True, True, seed_step, out=traj_dev, host=traj_pin)
        env.reset_stats()
        barrier(cx)
        t0 = time.perf_counter()
        for _ in range(Ke):
            tr = env.rollout_fair_traj(D, True, True, seed_step, out=traj_dev, host=traj_pin)
        barrier(cx)
        dt, (dd,) = reduce_max_sum(cx, time.perf_counter() - t0, [env.stats()["decisions"]])
        e2e_rollout = {"value": dd / dt, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": nb,
                       "steps": Ke, "path": "ssb_rollout_fair_traj (policy + step fused on the device) -> D2H of the "
                                            "B x 128 transition records to pinned memory",
                       "mean_reward_check": float(tr["reward"].mean())}
        launches_e2e += Ke
    ws = env.workspace_bytes >> 20
    env.close()
    cpu = None
    if cx.rank == 0 and cx.world == 1 and args.cpu_seconds > 0:
        cpu = cpu_arm(args.cpu_seconds)
    return {
        "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": cx.world, "steps": K,
        "warmup": W, "ms_per_step": max_ms / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": headline_config(B, cx.world, ws), "workspace_mib_per_gpu": ws,
        "events_per_s": total_ev / (max_ms * 1e-3), "episodes": total_eps, "env_errors": total_err,
        "rollout_stats": parallel.stats_from_sums(stats_vec),
        "stats_exchange": "ssb_collect_stats after every step on the device into a [steps, 8] buffer; one NCCL "
                          "all-reduce of that buffer after the last step, inside the timed region",
        "wall_s_timed_region": t_wall,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_obs": e2e_obs, "e2e_rollout": e2e_rollout,
        "clocks": clocks, "gpu_launches": launches + launches_e2e,
    }


def run_c4(cx, args):
    """Config 4: continuous Poisson arrivals, 200 jobs x 50 executors long-horizon episodes, 8192 envs per GPU."""
    from spark_sched_sim_b200 import parallel
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, D, K, W = args.c4_envs, 64, max(2, min(cx.K, 4)), 3
    env = BatchedSparkSchedSimEnv(C3_CFG, num_envs=B, bank=cx.bank, device=cx.dev)
    seeds, seed_step = parallel.shard_seeds(4321, B, cx.rank, cx.world)
    # 1500 untimed decisions per env first: the 200-job episodes (~2300 fair decisions each) are then in their long
    # middle part with ~80 active jobs, not in the cheap first minutes after a reset
    kern_ms, st, launches, stats_vec, _ = timed_fair_rollouts(cx, env, seeds, seed_step, W, K, D, pre_decisions=1500)
    n_err = int((env.hdr()["error"] != 0).sum())
    max_ms, (dec, ev, err) = reduce_max_sum(cx, kern_ms, [st["decisions"], st["events"], n_err])
    ws = env.workspace_bytes >> 20
    env.close()
    e2e = None
    if not args.no_e2e:
        e2e = e2e_step_loop(cx, C3_CFG, seeds, seed_step, 2, 16, args.e2e_budget, False)
        e2e["path"] = "ssb_step_fair_host per decision batch (as the headline's e2e), 50 executors / 200 jobs"
    cpu = None
    if cx.rank == 0 and cx.world == 1 and args.cpu_seconds > 0:
        cpu = cpu_arm(min(args.cpu_seconds, 8.0), cfg=C3_CFG, label="C4 (200 jobs x 50 executors)")
    return {
        "workload": f"C4: {B} envs/GPU x (200 jobs, 50 executors), Poisson arrivals 4e-5/ms, fair scheduler "
                    f"({B * cx.world} envs on {cx.world} GPU(s))",
        "value": dec / (max_ms * 1e-3), "unit": "decisions/s", "n_gpus": cx.world, "steps": K, "warmup": W,
        "decisions_per_env_per_step": D, "ms_per_step": max_ms / K, "events_per_s": ev / (max_ms * 1e-3),
        "untimed_decisions_before": 1500 + W * D,
        "env_errors": err, "workspace_mib_per_gpu": ws, "dtype": DTYPE, "scaling": "weak",
        "rollout_stats": parallel.stats_from_sums(stats_vec),
        "roofline": hbm_roofline(st, kern_ms, K, "k_rollout_fair<2> (two executor slots per lane)", _traffic("c4")),
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches + (e2e["gpu_launches"] if e2e else 0),
    }


def run_decima(cx, args, with_update: bool):
    """Configs 3 and 5: Decima rollouts at config/decima_tpch.yaml's env (50 executors, 200 jobs, mean time limit
    2e7 ms) on every GPU.  with_update (C5): + the learner's exchanges -- rollout statistics all-reduce per
    iteration, and one PPO mini-batch update on the device whose 20 802-float gradient is all-reduced over NCCL."""
    torch = cx.torch
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200 import parallel, ppo
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B = args.c3_envs
    chunk, W, K = 25, 3, max(2, min(cx.K, 4))  # decisions per ssb_rollout_decima call (one rollout-buffer slab)
    env = BatchedSparkSchedSimEnv(C3_CFG, num_envs=B, bank=cx.bank, decima_policy=True, device=cx.dev)
    z = np.load(osp.join(REPO, "tests", "golden", "decima_model.npz"))
    env.set_decima_weights({k: z[k] for k in z.files})
    seeds, seed_step = parallel.shard_seeds(1234, B, cx.rank, cx.world)
    env.set_mean_time_limit(C3_MEAN_TIME_LIMIT)
    env.set_autoreset(True, seed_step)
    env.reset_host(seeds)
    nb = B * chunk * nat.TRANSITION_DTYPE.itemsize
    traj_dev = torch.empty(nb, dtype=torch.uint8, device=cx.dev)
    traj_pin = torch.empty(nb, dtype=torch.uint8).pin_memory()
    stats_vec = torch.zeros(8, dtype=torch.float64, device=cx.dev)
    # into the episodes first (untimed): 1500 decisions per env with the cheap fused fair kernel, so that the
    # timed Decima decisions see mid-episode observations (~80 active jobs, ~700 nodes) instead of the small ones
    # right after a reset; then W Decima slabs as warm-up proper
    env.rollout_fair(1500, True, True, seed_step)
    for _ in range(W):
        env.rollout_decima(chunk, max_events=0, out=traj_dev)
    env.reset_stats()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    barrier(cx)
    for k in range(K):
        cx.flush.fill_(k & 0xFF)
        ev0[k].record()
        env.rollout_decima(chunk, max_events=0, out=traj_dev)
        env.collect_stats(stats_vec)
        if cx.world > 1:
            cx.dist.all_reduce(stats_vec)  # once per rollout iteration (rollout_worker.py:122-129)
        ev1[k].record()
    barrier(cx)
    kern_ms = sum(a.elapsed_time(b) for a, b in zip(ev0, ev1))
    st = env.stats()
    hdr = env.hdr()
    n_err = int(((hdr["error"] != 0) & (hdr["error"] != 9)).sum())
    max_ms, (dec, ev, err) = reduce_max_sum(cx, kern_ms, [st["decisions"], st["events"], n_err])
    # the policy call alone (adapter + planning + tile kernels + sampling), CUDA events on the launching stream
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_pol = 10
    env.decima_policy()
    p0.record()
    for _ in range(n_pol):
        env.decima_policy()
    p1.record()
    torch.cuda.synchronize()
    pol_ms = p0.elapsed_time(p1) / n_pol
    work = env.decima_work()
    pk = peaks()
    # useful flops: the MLPs' multiply-adds at the model's real widths (App. E) x 2; the tensor cores execute a
    # multiple of that (operand splitting for fp32 accuracy, padded K / N), stated separately
    useful_tflops = 2.0 * work["macs"] / (pol_ms * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "kernel": "ssb_decima_policy (k_decima_obs_cta, planning, k_tile3<*> x (6 + 2 x depth), sampling)",
        "achieved": useful_tflops, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": useful_tflops / pk["tensor"],
        "traffic": None, "peak_source": pk["src"], "policy_call_ms": pol_ms, "rows": work,
        "useful_macs_per_call": work["macs"], "launches_per_call": "see profiles/ launch list",
        "note": "K <= 64 three-layer MLP chains over gathered rows: bound by the per-layer hand-off and the launch "
                "sequence, not by the tensor pipe; the fraction is reported, not hidden",
    }
    tp = osp.join(REPO, "profiles", "policy_tensor_pipe.json")
    if osp.exists(tp):  # sm__pipe_tensor_cycles_active of the tile kernels, from the committed ncu capture
        with open(tp) as f:
            roofline["tensor_pipe"] = json.load(f)
    # e2e: the rollout-collection call with every slab of transitions copied to pinned host memory (wall clock)
    env.reset_stats()
    barrier(cx)
    t0 = time.perf_counter()
    for _ in range(K):
        env.rollout_decima(chunk, max_events=0, out=traj_dev, host=traj_pin)
    barrier(cx)
    dt, (e2e_dec,) = reduce_max_sum(cx, time.perf_counter() - t0, [env.stats()["decisions"]])
    e2e = {"value": e2e_dec / dt, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": nb,
           "steps": K, "path": f"ssb_rollout_decima ({chunk} decisions per env) -> D2H of the transition slab (pinned)"}
    out = {
        "workload": f"{'C5' if with_update else 'C3'}: {B} envs/GPU x (200 jobs, 50 executors, mean time limit 2e7 "
                    f"ms), Decima policy (shipped model.pt) + sampling + step on the device ({B * cx.world} envs on "
                    f"{cx.world} GPU(s))",
        "value": dec / (max_ms * 1e-3), "unit": "decisions/s", "n_gpus": cx.world, "steps": K, "warmup": W,
        "decisions_per_env_per_step": chunk, "ms_per_step": max_ms / K, "events_per_s": ev / (max_ms * 1e-3),
        "untimed_decisions_before": f"1500 (fair policy) + {W * chunk} (Decima)",
        "mean_nodes": st["sum_nodes"] / max(st["observations"], 1),
        "mean_active_jobs": st["sum_jobs"] / max(st["observations"], 1),
        "env_errors": err, "workspace_mib_per_gpu": env.workspace_bytes >> 20, "scaling": "weak",
        "dtype": "fp32 policy (split-precision tensor-core MMAs, fp32 accumulation); f64 event times + integer state",
        "rollout_stats": parallel.stats_from_sums(stats_vec), "roofline": roofline, "e2e": e2e,
        "gpu_launches": "one CUDA graph of ~50 kernels per decision",
    }
    if with_update:
        # one PPO mini-batch on the device (trainers/ppo.py:72-102): evaluate_actions on a stored observation, clip
        # loss, backward, gradient all-reduce over NCCL (parallel.allreduce_gradients), clip_grad_norm_ + Adam
        snap = env.decima_snapshot()
        env.decima_policy()
        act = env.pol_action.clone()
        old_lg = env.pol_lgprob.clone()
        g = torch.Generator(device="cpu").manual_seed(5 + cx.rank)
        ret = torch.randn(B, generator=g, dtype=torch.float64).to(cx.dev)
        base = torch.zeros(B, dtype=torch.float64, device=cx.dev)
        flat = torch.from_numpy(np.concatenate([z[k].reshape(-1) for k in env.DECIMA_PARAM_ORDER]).astype(np.float32))
        adam = ppo.Adam(flat.to(cx.dev).contiguous(), lr=3e-4, max_grad_norm=0.5)
        loss_fn = ppo.PPOLoss(clip_range=0.2, entropy_coeff=0.04)
        stage_sel, exec_sel = act[:, 0].contiguous(), act[:, 2].contiguous()
        times = []
        for it in range(3):
            barrier(cx)
            u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            u0.record()
            info, stepped = ppo.ppo_minibatch_update(env, snap, stage_sel, exec_sel, old_lg, ret, base, loss_fn, adam,
                                                     target_kl=None, allreduce=parallel.allreduce_gradients)
            u1.record()
            torch.cuda.synchronize()
            times.append(u0.elapsed_time(u1))
        upd_ms, _ = reduce_max_sum(cx, min(times), [0])
        wsum = torch.tensor([float(adam.params.double().sum().item())], dtype=torch.float64, device=cx.dev)
        wmin, wmax = wsum.clone(), wsum.clone()
        if cx.world > 1:
            cx.dist.all_reduce(wmin, op=cx.dist.ReduceOp.MIN)
            cx.dist.all_reduce(wmax, op=cx.dist.ReduceOp.MAX)
        out["ppo_update"] = {
            "ms_per_minibatch": upd_ms, "samples_per_minibatch": B * cx.world,
            "samples_per_s": B * cx.world / (upd_ms * 1e-3),
            "exchange": "one all-reduce of the flat gradient vector (20 802 floats + sample count) per mini-batch "
                        "+ one 2-number all-reduce for the collective KL early stop",
            "weights_identical_across_ranks": bool(wmin.item() == wmax.item()),
            "approx_kl_div": info["approx_kl_div"], "stepped": bool(stepped)}
    env.close()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the headline; the extra configs and the e2e loops run their own short "
                         "windows (2 .. 5 steps), each reported in its entry")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-budget", type=int, default=256,
                    help="max timeline events per env per ssb_step_host call (0 = run to next decision)")
    ap.add_argument("--configs", default="C3,C4,C5", help="extra BASELINE.json configurations to run (or 'none')")
    ap.add_argument("--c3-envs", type=int, default=C3_ENVS)
    ap.add_argument("--c4-envs", type=int, default=C4_ENVS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's outputs after its last timed step to DIR/<name>.npy (rank 0's envs; "
                         "rollout_stats is the all-reduced sum over the ranks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from spark_sched_sim_b200.bank import synthetic_bank

    cx = Ctx()
    cx.torch, cx.dist = torch, dist
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    cx.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(cx.local_rank)
    cx.dev = torch.device("cuda", cx.local_rank)
    if cx.world > 1:
        dist.init_process_group("nccl", device_id=cx.dev)
    cx.W, cx.K = max(args.warmup, 3), args.steps
    cx.bank = synthetic_bank(0)
    cx.flush = torch.empty(256 << 20, dtype=torch.uint8, device=cx.dev)  # > 126 MB L2

    out = run_c2(cx, args)
    want = [c.strip().upper() for c in args.configs.split(",") if c.strip() and c.strip().lower() != "none"]
    configs = {}
    decima_done = False
    for name in want:
        try:
            if name == "C4":
                configs["C4"] = run_c4(cx, args)
            elif name in ("C3", "C5") and not decima_done:
                decima_done = True
                # one GPU: C5 is C3's measurement plus the policy update (the exchanges have no peer); several GPUs:
                # C3 (a one-GPU configuration) is not repeated, C5 is the sweep point
                res = run_decima(cx, args, with_update="C5" in want)
                if cx.rank == 0 and cx.world == 1 and args.cpu_seconds > 0:
                    res["cpu_baseline"] = cpu_arm_decima(min(args.cpu_seconds, 6.0), C3_CFG, "C3")
                if cx.world == 1 and "C3" in want:
                    configs["C3"] = {k: v for k, v in res.items() if k != "ppo_update"}
                    configs["C3"]["workload"] = res["workload"].replace("C5:", "C3:")
                if "C5" in want:
                    configs["C5"] = dict(res, workload=res["workload"].replace("C3:", "C5:"))
        except Exception as exc:  # a failed extra config must not take the headline line with it
            configs[name] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.synchronize()
    if cx.rank == 0:
        out["configs"] = configs
        print(json.dumps(out))
    if cx.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
