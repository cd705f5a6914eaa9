"""Cost of an attached episode log (ssb_attach_episode_log) on the fused fair rollout: the same launches with the log
detached and attached, alternating in one process, at two shapes:

    C2: 4096 envs x (50 jobs, 10 executors), fair policy, auto-reset (seed_step = B), 128 decisions per launch,
        seeds 1234 + i -- bench.py's headline rollout
    C4: 8192 envs x (200 jobs, 50 executors), 64 decisions per launch, seeds 4321 + i, after 1500 untimed decisions

Each arm runs on a handle of its own; the attached arm carries a log with a ring of 64 records and a window of 200
durations per env (BatchedSparkSchedSimEnv.attach_episode_log's defaults).  Every repeat starts over from the seeds
(reset, the untimed decisions, 3 warm-up launches), so the repeats time the same work.  Timing as bench.py's: CUDA
events around each launch (the attached arm's k_episode_log launch included), a 256 MiB write between timed launches
to evict L2.  Per repeat and arm: ms per launch and decisions/s; the attached
arm also reports the records and job durations it wrote.  The summary gives the mean and the spread (max - min over
mean) of each arm and the attached arm's cost relative to the detached one.

Usage on a GPU:  python profiles/episode_log_ab.py [--repeats R] [--iters I] [--shapes C2,C4] [--out FILE]"""
import argparse
import os.path as osp
import subprocess
import sys

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

SHAPES = {"C2": (4096, 10, 50, 128, 0, 1234), "C4": (8192, 50, 200, 64, 1500, 4321)}  # B, E, J, K, untimed, seed


def gpu_info() -> str:
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or f"{torch.cuda.get_device_name(0)} (nvidia-smi: {q.stderr.strip()})"


def run_shape(name, repeats, iters, log):
    B, E, J, K, pre, SEED0 = SHAPES[name]
    cfg = {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
           "warmup_delay": 1000.0}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB of L2
    envs = {"detached": BatchedSparkSchedSimEnv(cfg, num_envs=B), "attached": BatchedSparkSchedSimEnv(cfg, num_envs=B)}
    seeds = (SEED0 + np.arange(B)).astype(np.uint64)
    res = {k: [] for k in envs}
    for r in range(repeats):
        for arm, env in envs.items():
            env.reset_host(seeds)
            if arm == "attached":
                env.attach_episode_log(capacity=64, window=200)  # zeroed: a fresh log per repeat
            if pre:
                env.rollout_fair(pre, True, True, B)
            for _ in range(3):
                env.rollout_fair(K, True, True, B)
            torch.cuda.synchronize()
            env.reset_stats()
            c0 = env.episode_cursors()[:, :2].sum(0).cpu().numpy() if arm == "attached" else None
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                  for _ in range(iters)]
            for k, (e0, e1) in enumerate(ev):
                flush.fill_(k & 0xFF)
                e0.record()
                env.rollout_fair(K, True, True, B)
                e1.record()
            torch.cuda.synchronize()
            ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) / iters
            st = env.stats()
            rate = st["decisions"] / (ms * iters * 1e-3)
            err = int((env.hdr()["error"] != 0).sum())
            extra = ""
            if arm == "attached":
                c1 = env.episode_cursors()[:, :2].sum(0).cpu().numpy()
                n_ep, n_jobs = (int(x) for x in c1 - c0)
                extra = (f"  wrote {n_ep} records ({st['decisions'] / max(n_ep, 1):.0f} decisions each) and "
                         f"{n_jobs} job durations")
            res[arm].append((ms, rate))
            log(f"{name} rep {r} {arm:9s}: {ms:8.3f} ms/launch  {rate / 1e6:7.3f} M decisions/s  env_errors={err}{extra}")
    mean = {}
    for arm, rows in res.items():
        ms, rate = (np.array(x) for x in zip(*rows))
        mean[arm] = ms.mean()
        log(f"{name} {arm:9s} mean over {repeats} repeats x {iters} launches: {ms.mean():8.3f} ms/launch  "
            f"{rate.mean() / 1e6:7.3f} M decisions/s (spread {100 * (rate.max() - rate.min()) / rate.mean():.2f} %)")
    log(f"{name} attached / detached time per launch: {mean['attached'] / mean['detached']:.4f}")
    for env in envs.values():
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--shapes", default="C2,C4")
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# GPU (name, power limit, max SM clock): {gpu_info()}")
    for name in args.shapes.split(","):
        run_shape(name, args.repeats, args.iters, log)
    log(f"# GPU at the end: {gpu_info()}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
