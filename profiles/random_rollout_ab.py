"""Fused random-policy rollout (ssb_rollout_random) against the fused fair rollout (ssb_rollout_fair) in one process,
alternating, at two shapes:

    C2: 4096 envs x (50 jobs, 10 executors), 128 decisions per launch, seeds 1234 + i
    C4: 8192 envs x (200 jobs, 50 executors), 64 decisions per launch, seeds 4321 + i, after 1500 untimed decisions

The async pair (--pairs async) times the fixed-duration rollouts instead, ssb_rollout_random_async against
ssb_rollout_fair_async, with the same decisions per launch as max_decisions and a rollout_duration of 6e6 ms at C2 and
5.5e5 ms at C4: about the median simulated time the random policy takes for 128 / 64 decisions at these shapes, so
that the duration stops part of the envs and max_decisions the rest.  Their rate counts the decisions the launches
report in num_steps; each repeat also reports the share of envs the duration stopped (num_steps < max_decisions).

Each policy runs on a handle of its own (auto-reset, seed_step = B, as bench.py).  Every repeat starts over from the
seeds (reset, the untimed decisions, 3 warm-up launches), so the repeats time the same work and their spread is
run-to-run noise, not the episodes moving on.  Timing as bench.py's: CUDA events around each launch, a 256 MiB write
between timed launches to evict L2.  Per repeat and policy: ms per launch, decisions/s and events per decision
(ssb_stats); the summary gives the mean and the spread (max - min over mean) of the repeats.  Random episodes take
other executor counts and other event chains than fair ones, so the two rates are not expected to match.

Usage on a GPU:  python profiles/random_rollout_ab.py [--repeats R] [--iters I] [--shapes C2,C4] [--pairs sync,async]
                 [--out FILE]"""
import argparse
import os.path as osp
import subprocess
import sys

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

SHAPES = {  # B, E, J, decisions per launch, untimed decisions first, first seed, rollout_duration (ms) of the async pair
    "C2": (4096, 10, 50, 128, 0, 1234, 6.0e6),
    "C4": (8192, 50, 200, 64, 1500, 4321, 5.5e5),
}
PAIRS = {"sync": ("random", "fair"), "async": ("random_async", "fair_async")}


def gpu_info() -> str:
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or f"{torch.cuda.get_device_name(0)} (nvidia-smi: {q.stderr.strip()})"


def launch(env, policy, K, B, dur=None):
    """One launch; the async policies return num_steps (device i32[B])."""
    if policy == "random":
        env.rollout_random(K, True, B)
    elif policy == "fair":
        env.rollout_fair(K, True, True, B)
    elif policy == "random_async":
        return env.rollout_random_async(K, dur, B)[1]
    else:
        return env.rollout_fair_async(K, dur, True, B)[1]


def run_shape(name, pair, repeats, iters, log):
    B, E, J, K, pre, seed0, dur = SHAPES[name]
    cfg = {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB of L2
    envs = {policy: BatchedSparkSchedSimEnv(cfg, num_envs=B) for policy in PAIRS[pair]}
    seeds = (seed0 + np.arange(B)).astype(np.uint64)
    res = {p: [] for p in envs}
    for r in range(repeats):
        for policy, env in envs.items():
            env.reset_host(seeds)
            if pre:
                launch(env, policy.removesuffix("_async"), pre, B)
            for _ in range(3):
                launch(env, policy, K, B, dur)
            torch.cuda.synchronize()
            env.reset_stats()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
            nums = []
            for k, (e0, e1) in enumerate(ev):
                flush.fill_(k & 0xFF)
                e0.record()
                nums.append(launch(env, policy, K, B, dur))
                e1.record()
            torch.cuda.synchronize()
            ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) / iters
            st = env.stats()
            err = int((env.hdr()["error"] != 0).sum())
            extra = ""
            if pair == "async":
                num = torch.stack(nums).cpu().numpy()
                decisions = int(num.sum())
                extra = f"  stopped by the duration {100 * (num < K).mean():5.1f} % of envs"
            else:
                decisions = st["decisions"]
            rate = decisions / (ms * iters * 1e-3)
            res[policy].append((ms, rate, st["events"] / st["decisions"]))
            log(f"{name} rep {r} {policy:12s}: {ms:8.2f} ms/launch  {rate / 1e6:7.2f} M decisions/s  "
                f"{st['events'] / st['decisions']:6.2f} events/decision  env_errors={err}{extra}")
    for policy, rows in res.items():
        ms, rate, epd = (np.array(x) for x in zip(*rows))
        log(f"{name} {policy:12s} mean over {repeats} repeats x {iters} launches: {ms.mean():8.2f} ms/launch  "
            f"{rate.mean() / 1e6:7.2f} M decisions/s (spread {100 * (rate.max() - rate.min()) / rate.mean():.2f} %)  "
            f"{epd.mean():6.2f} events/decision")
    for env in envs.values():
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--shapes", default="C2,C4")
    ap.add_argument("--pairs", default="sync", help="sync (rollout_random / rollout_fair), async (the fixed-duration "
                    "rollouts), or both: sync,async")
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# GPU (name, power limit, max SM clock): {gpu_info()}")
    for pair in args.pairs.split(","):
        for name in args.shapes.split(","):
            run_shape(name, pair, args.repeats, args.iters, log)
    log(f"# GPU at the end: {gpu_info()}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
