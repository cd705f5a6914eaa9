"""Policy evaluation over thousands of episodes with the device episode log: the fair, FIFO, random and Decima
schedulers at the C2 shape, auto-reset on, every finished episode recorded by ssb_attach_episode_log.

    C2: 4096 envs x (50 jobs, 10 executors), seeds 1234 + i, seed_step = 4096 (episode k of env i: 1234 + i + 4096 k)
    Decima: the weights of tests/golden/decima_model.npz, sampled actions (ssb_rollout_decima with auto-reset)

Every policy runs on a handle of its own from the same seeds, so the k-th episodes of the policies play the same job
sequences.  Per policy: the number of finished episodes, the mean and the 10/50/90th percentiles of the per-episode
average job completion time (sum of the completed jobs' durations / their number, in seconds), the episode length in
decisions, and the finished episodes per second of rollout time (host clock around the rollout calls, ending in a
device synchronise).  The reference's behavioural claim is that Decima's average JCT is below the fair scheduler's.

Usage on a GPU:  python profiles/episode_eval.py [--decisions D] [--decima-decisions D] [--out FILE]"""
import argparse
import os.path as osp
import subprocess
import sys
import time

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

B, E, J, SEED0 = 4096, 10, 50, 1234
CFG = {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
       "warmup_delay": 1000.0}


def gpu_info() -> str:
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or f"{torch.cuda.get_device_name(0)} (nvidia-smi: {q.stderr.strip()})"


def run_policy(policy: str, decisions: int, chunk: int):
    env = BatchedSparkSchedSimEnv(CFG, num_envs=B, decima_policy=(policy == "decima"))
    seeds = (SEED0 + np.arange(B)).astype(np.uint64)
    if policy == "decima":
        z = np.load(osp.join(REPO, "tests", "golden", "decima_model.npz"))
        env.set_decima_weights({k: z[k] for k in z.files})
        env.set_autoreset(True, B)
    env.reset_host(seeds)
    env.attach_episode_log(capacity=64, window=200)
    out = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(decisions // chunk):
        if policy in ("fair", "fifo"):
            env.rollout_fair(chunk, policy == "fair", True, B)
        elif policy == "random":
            env.rollout_random(chunk, True, B)
        else:
            out = env.rollout_decima(chunk, out=out)
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    e = env.episodes()
    errors = int((env.hdr()["error"] != 0).sum())
    res = {k: e[k].cpu().numpy() for k in ("avg_job_duration", "decisions", "terminated", "truncated", "env", "episode")}
    res["dropped"] = int(e["dropped"].sum())
    env.close()
    return res, secs, errors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--decisions", type=int, default=4096, help="decisions per env for the heuristics")
    ap.add_argument("--decima-decisions", type=int, default=1536, help="decisions per env for Decima")
    ap.add_argument("--policies", default="fair,fifo,random,decima")
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    args = ap.parse_args()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"# GPU (name, power limit, max SM clock): {gpu_info()}")
    log(f"# C2: {B} envs x ({J} jobs, {E} executors), auto-reset, seeds {SEED0} + i + {B} k")
    jct = {}
    for policy in args.policies.split(","):
        d = args.decima_decisions if policy == "decima" else args.decisions
        res, secs, errors = run_policy(policy, d, 128 if policy != "decima" else 64)
        a = res["avg_job_duration"]
        n = len(a)
        jct[policy] = res
        p10, p50, p90 = np.percentile(a, [10, 50, 90]) if n else (np.nan,) * 3
        log(f"{policy:7s}: {n:6d} finished episodes ({int(res['terminated'].sum())} terminated, "
            f"{int(res['truncated'].sum())} truncated, {res['dropped']} dropped by the ring) in {d} decisions/env, "
            f"{secs:6.2f} s -> {n / secs:9.1f} episodes/s; avg JCT per episode: mean {a.mean():8.2f} s, "
            f"p10 {p10:8.2f}  p50 {p50:8.2f}  p90 {p90:8.2f}; {res['decisions'].mean():6.1f} decisions/episode; "
            f"env_errors={errors}")
    if "decima" in jct and "fair" in jct:
        # the same job sequences: (env, episode index) pairs both policies finished
        f, dm = jct["fair"], jct["decima"]
        kf = {(int(b), int(k)): v for b, k, v in zip(f["env"], f["episode"], f["avg_job_duration"])}
        pairs = [(kf[(int(b), int(k))], v) for b, k, v in zip(dm["env"], dm["episode"], dm["avg_job_duration"])
                 if (int(b), int(k)) in kf]
        if pairs:
            pf, pd = (np.array(x) for x in zip(*pairs))
            log(f"paired episodes (same job sequence) finished by both fair and Decima: {len(pairs)}; mean avg JCT "
                f"fair {pf.mean():.2f} s, Decima {pd.mean():.2f} s; Decima lower in {100 * (pd < pf).mean():.1f} %")
    log(f"# GPU at the end: {gpu_info()}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
