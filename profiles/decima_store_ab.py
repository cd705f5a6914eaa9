"""What recording the observations costs: the fixed-duration Decima rollout (ssb_rollout_decima_async) with and without
an attached rollout store (ssb_decima_attach_rollout_store), in one process, alternating, at two shapes:

    C2: 4096 envs x (50 jobs, 10 executors), the shape of bench.py's C2 with the Decima policy
    C3: 512 envs x (200 jobs, 50 executors, mean time limit 2e7 ms), the environment of config/decima_tpch.yaml with
        fewer envs than bench.py's C3 (the store of 4096 such envs would take most of the card for a few rows)

Both arms run on one handle, the same weights (tests/golden/decima_model.npz) and streams 0 .. B-1; every timed call
starts from the same reset (seeds first_seed + i), so the two arms do the same work -- the store only copies.  One call
= max_decisions rows per env at most, a rollout_duration long enough that max_decisions stops every env.  Timing: a
host clock around the call, which ends in a device synchronise (the loop checks its envs every 8 rounds).  Reported per
shape: ms per call of each arm and the mean of their differences over the repeats, the rounds of a call (the most
rows + in-rollout resets any env had; the loop may run up to 7 rounds past that) and the difference per round, the
stored bytes per row (ssb_decima_snapshot_bytes / B plus the two i32 actions), and the largest K whose store (plus the
RolloutStore's per-row tensors and the transition rows) fits in the memory left free on the card with the handle in
place.  The card's name and power limit come from the same process.

Usage on a GPU:  python profiles/decima_store_ab.py [--repeats R] [--shapes C2,C3] [--out FILE]"""
import argparse
import os.path as osp
import subprocess
import sys
import time

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spark_sched_sim_b200 import _native as nat  # noqa: E402
from spark_sched_sim_b200 import ppo  # noqa: E402
from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

SHAPES = {  # B, E, J, mean time limit (0: none), max_decisions, first seed
    "C2": (4096, 10, 50, 0.0, 64, 1234),
    "C3": (512, 50, 200, 2.0e7, 32, 42),
}
DURATION = 1.0e12  # ms: max_decisions ends every env's call


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return f"{name}, power limit {q}"


def weights():
    z = np.load(osp.join(REPO, "tests", "golden", "decima_model.npz"))
    return {k: z[k] for k in z.files}


def run_shape(label, repeats, log):
    B, E, J, tl, K, seed0 = SHAPES[label]
    cfg = {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
           "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, decima_policy=True)
    env.set_decima_weights(weights())
    if tl:
        env.set_mean_time_limit(tl)
    env.set_policy_streams(np.arange(B, dtype=np.uint32))
    seeds = np.arange(B, dtype=np.uint64) + seed0
    store = ppo.RolloutStore(env, K)
    snap_bytes = env.decima_snapshot_bytes()

    def call(with_store):
        env.reset_host(seeds)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        traj, num, _ = env.rollout_decima_async(K, DURATION, seed_step=B, store=store if with_store else None)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        flags = traj.view(torch.int32).view(B, K, 8)[..., 6]
        resets = ((flags & 4) != 0).sum(1)
        rounds = int((num + resets).max().item())
        return dt * 1e3, rounds

    for w in (False, True, False, True):  # warm-up: module loads, the store's first touch
        call(w)
    plain, stored, diffs, rounds = [], [], [], 0
    for r in range(repeats):
        a, rounds = call(False)
        b, rounds_b = call(True)
        assert rounds_b == rounds  # the store changes no decision
        plain.append(a); stored.append(b); diffs.append(b - a)
        log(f"{label} repeat {r}: plain {a:.2f} ms, with store {b:.2f} ms per call ({rounds} rounds)")
    per_row = snap_bytes / B + 8
    free, total = torch.cuda.mem_get_info()
    per_k = snap_bytes + B * (4 + 4 + 4 + 8 + 8 + 1 + nat.TRANSITION_DTYPE.itemsize)  # RolloutStore tensors + traj
    kmax = int((free + K * per_k) // per_k)  # (this K's store is already allocated)
    m, sd = float(np.mean(diffs)), float(np.std(diffs))
    log(f"{label}: {B} envs x ({J} jobs, {E} executors), max_decisions {K}, {rounds} rounds per call")
    log(f"{label}: plain {np.mean(plain):.2f} ms (spread {np.ptp(plain) / np.mean(plain) * 100:.1f} %), with store "
        f"{np.mean(stored):.2f} ms (spread {np.ptp(stored) / np.mean(stored) * 100:.1f} %) per call")
    log(f"{label}: store overhead {m:.2f} +- {sd:.2f} ms per call = {m / rounds * 1e3:.1f} us per round "
        f"({m / np.mean(plain) * 100:.2f} % of the call)")
    log(f"{label}: {snap_bytes} snapshot bytes per block = {snap_bytes / B:.0f} bytes per env row "
        f"(+ 8 for the actions: {per_row:.0f}); largest K that fits in the {free / 2**30:.1f} GiB left free of "
        f"{total / 2**30:.1f} GiB: {kmax}")
    del store, env
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--shapes", default="C2,C3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log(f"card: {card()}")
    for label in args.shapes.split(","):
        run_shape(label, args.repeats, log)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
