"""The device episode log (ssb_attach_episode_log, BatchedSparkSchedSimEnv.attach_episode_log): one record per
finished episode written by the step that ends it, on every step path, against the CPU oracle replaying each env's
seed sequence and against the transition rows; the job-duration window against the facade's job_duration_buff (the
reference's deque(maxlen=200)); and the edge cases of the attach protocol."""
import os.path as osp

import numpy as np
import pytest
import torch

from helpers import GOLDEN_DIR
from random_policy_spec import random_policy_action

pytestmark = pytest.mark.gpu


def cfg_of(E=10, J=8, beta=0.0):
    return {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
            "warmup_delay": 1000.0, "beta": beta}


def make_env(bank, cfg, B, base=100, mean_time_limit=0.0, **kw):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, **kw)
    if mean_time_limit > 0:
        env.set_mean_time_limit(mean_time_limit)
    seeds = base + np.arange(B, dtype=np.uint64)
    hdr = env.reset_host(seeds)
    assert (hdr["error"] == 0).all()
    return env, seeds


def host_records(env):
    """episodes() as a list (per env) of lists of dicts of python scalars."""
    e = {k: v.cpu().numpy() for k, v in env.episodes().items() if k != "dropped"}
    out = [[] for _ in range(env.num_envs)]
    for i in range(len(e["env"])):
        out[int(e["env"][i])].append({k: e[k][i] for k in e})
    return out


def oracle_episodes(bank, cfg, seed, seed_step, n_episodes, policy="fair", mean_time_limit=0.0):
    """The records of an env's first n_episodes episodes, replayed on the oracle: episode k has seed
    seed + seed_step * k, its StochasticTimeLimit draw when a mean is set, and ends at the first observation that
    reports terminated or truncated.  The sums are restated serially in job-index order."""
    from oracle import OracleEnv
    from philox_ref import time_limit_draw

    orc = OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                    cfg["job_arrival_rate"], cfg.get("beta", 0.0))
    out = []
    for k in range(n_episodes):
        s = int(seed) + seed_step * k
        tl = time_limit_draw(s, mean_time_limit) if mean_time_limit > 0 else np.inf
        orc.reset_seed(s, tl)
        d, term, trunc = 0, False, False
        while not (term or trunc):
            a, n = orc.fair_action(True) if policy == "fair" else random_policy_action(orc.obs(), s, d)
            rc, _, term = orc.step(a, n)
            assert rc == 0
            d += 1
            trunc = orc.wall_time >= tl
        wall = orc.wall_time
        ta, tc, _ = orc.job_times()
        jt, sd, na, nc = 0.0, 0.0, 0, 0
        for j in range(len(ta)):
            if ta[j] > wall:
                continue
            na += 1
            jt += min(tc[j], wall) - ta[j]
            if np.isfinite(tc[j]):
                nc += 1
                sd += tc[j] - ta[j]
        out.append({"seed": s, "wall_time": wall, "time_limit": tl, "job_time": jt, "sum_job_duration": sd,
                    "decisions": d, "jobs_arrived": na, "jobs_completed": nc,
                    "flags": int(term) | 2 * int(trunc), "episode": k})
    return out


def check_against_oracle(bank, cfg, env, seeds, seed_step, policy, mean_time_limit=0.0, min_total=1):
    recs = host_records(env)
    total = 0
    for b in range(env.num_envs):
        got = recs[b]
        total += len(got)
        if not got:
            continue
        assert [int(g["episode"]) for g in got] == list(range(len(got))), b
        want = oracle_episodes(bank, cfg, seeds[b], seed_step, len(got), policy, mean_time_limit)
        for g, w in zip(got, want):
            for k, v in w.items():
                gv = g[k]
                if k == "seed":
                    gv = int(np.int64(gv).view(np.uint64))
                assert gv == v or (isinstance(v, float) and np.isinf(v) and np.isinf(gv)), (b, g["episode"], k, gv, v)
    assert total >= min_total
    return total


@pytest.mark.parametrize("mean_time_limit", [0.0, 2.0e5])
def test_fused_fair_autoreset_bit_exact(bank, mean_time_limit):
    cfg = cfg_of(10, 8)
    B = 64
    env, seeds = make_env(bank, cfg, B, mean_time_limit=mean_time_limit)
    env.attach_episode_log(capacity=1024)  # room for every episode of the 600 decisions (one decision at least each)
    for _ in range(4):
        env.rollout_fair(150, auto_reset=True, seed_step=B)
    n = check_against_oracle(bank, cfg, env, seeds, B, "fair", mean_time_limit, min_total=2 * B)
    e = env.episodes()
    if mean_time_limit > 0:
        assert bool(e["truncated"].any())
    assert int(env.episode_cursors()[:, 0].sum()) == n
    assert int(e["dropped"].sum()) == 0


def test_rollout_random_matches_oracle(bank):
    cfg = cfg_of(10, 8)
    B = 32
    env, seeds = make_env(bank, cfg, B, base=500)
    env.attach_episode_log(capacity=64)
    for _ in range(3):
        env.rollout_random(150, auto_reset=True, seed_step=B)
    check_against_oracle(bank, cfg, env, seeds, B, "random", min_total=B)


def rows_check(env, seeds, seed_step, rows, num_steps=None, skip_flag8=False):
    """Records against transition rows [B, K]: one record per row that ends an episode (flags 1 / 2), with the
    decisions counted since the previous end, the same flags, and the seed of the episode's index."""
    recs = host_records(env)
    total = 0
    for b in range(env.num_envs):
        K = rows.shape[1] if num_steps is None else int(num_steps[b])
        want, d = [], 0
        for r in rows[b, :K]:
            if skip_flag8 and r["flags"] & 8:
                continue
            d += 1
            if r["flags"] & 3:
                want.append((d, int(r["flags"]) & 3))
                d = 0
        got = recs[b]
        assert len(got) == len(want), (b, len(got), len(want))
        for k, (g, (dw, fw)) in enumerate(zip(got, want)):
            assert (int(g["decisions"]), int(g["flags"]), int(g["episode"])) == (dw, fw, k), (b, k)
            assert int(np.int64(g["seed"]).view(np.uint64)) == int(seeds[b]) + seed_step * k
        total += len(got)
    assert total > 0
    return total


def _rows(traj, B, K):
    from spark_sched_sim_b200 import _native as nat

    return traj.cpu().numpy().view(nat.TRANSITION_DTYPE).reshape(B, K)


def test_step_api_autoreset(bank):
    cfg = cfg_of(10, 8)
    B = 16
    env, seeds = make_env(bank, cfg, B, base=900, mean_time_limit=2.0e5)
    env.set_autoreset(True, B)
    env.attach_episode_log(capacity=64)
    flags = []
    for _ in range(300):
        a, n = env.fair_actions()
        env.step(a, n)
        h = env.hdr()
        assert (h["error"] == 0).all()
        flags.append(np.where(h["was_reset"] == 1, 8, h["terminated"].astype(int) | 2 * h["truncated"].astype(int)))
    rows = np.zeros((B, len(flags)), dtype=[("flags", "<i4")])
    rows["flags"] = np.stack(flags, 1)
    rows_check(env, seeds, B, rows, skip_flag8=True)
    check_against_oracle(bank, cfg, env, seeds, B, "fair", 2.0e5)


@pytest.mark.parametrize("path", ["fair_async", "random_async"])
def test_async_rollouts(bank, path):
    cfg = cfg_of(10, 8)
    B, K = 32, 400
    env, seeds = make_env(bank, cfg, B, base=1300, mean_time_limit=2.0e5)
    env.attach_episode_log(capacity=64)
    run = env.rollout_fair_async if path == "fair_async" else env.rollout_random_async
    traj, num, _ = run(K, 4.0e6, seed_step=B)
    rows_check(env, seeds, B, _rows(traj, B, K), num.cpu().numpy())
    check_against_oracle(bank, cfg, env, seeds, B, "fair" if path == "fair_async" else "random", 2.0e5)


def _weights():
    z = np.load(osp.join(GOLDEN_DIR, "decima_model.npz"))
    return {k: z[k] for k in z.files}


def test_rollout_decima_graph_dropped_by_attach(bank):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    cfg = cfg_of(10, 4)
    B, K = 32, 40
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    env.set_decima_weights(_weights())
    seeds = 1700 + np.arange(B, dtype=np.uint64)
    env.reset_host(seeds)
    env.set_autoreset(True, B)
    env.rollout_decima(K)  # captures the decision graph without a log
    env.reset_host(seeds)
    env.attach_episode_log(capacity=64)
    rows = _rows(env.rollout_decima(K), B, K)
    rows_check(env, seeds, B, rows, skip_flag8=True)


def test_rollout_decima_async_rows_and_jobs(bank):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    cfg = cfg_of(10, 4)
    B, K = 16, 120
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    env.set_decima_weights(_weights())
    seeds = 2100 + np.arange(B, dtype=np.uint64)
    env.reset_host(seeds)
    env.attach_episode_log(capacity=64)
    traj, num, _ = env.rollout_decima_async(K, 3.0e6, seed_step=B)
    rows_check(env, seeds, B, _rows(traj, B, K), num.cpu().numpy())
    # with auto-reset off, the last record of an env whose live episode has ended describes the live episode
    h = env.hdr()
    recs = host_records(env)
    for b in range(B):
        if not (h["terminated"][b] or h["truncated"][b]):
            continue
        g = recs[b][-1]
        ta, tc, _, st = env.jobs(b, with_state=True)
        wall = float(h["wall_time"][b])
        jt, sd = 0.0, 0.0
        for j in range(len(ta)):
            if st[j] == 0:
                continue
            jt += min(tc[j], wall) - ta[j]
            if st[j] == 2:
                sd += tc[j] - ta[j]
        assert (g["wall_time"], g["job_time"], g["sum_job_duration"]) == (wall, jt, sd)
        assert g["jobs_completed"] == int((st == 2).sum()) and g["jobs_arrived"] == int((st != 0).sum())


def test_window_matches_facade_and_collect_stats(bank):
    """The window against the facade's job_duration_buff.  Both order jobs that complete at the same wall time by job
    index (the reference appends them in event order), so this checks the values and the order by completion time,
    not the reference's order among ties."""
    from spark_sched_sim_b200 import parallel
    from spark_sched_sim_b200.env import SparkSchedSimEnv

    cfg = cfg_of(10, 8)
    facades, means = [], []
    for f in range(2):
        env = SparkSchedSimEnv(cfg, bank=bank, decima_obs=False)
        env._batched.attach_episode_log(capacity=8, window=200)
        completions = 0
        ep = 0
        while completions <= 260:
            env.reset(seed=3000 + 17 * f + ep)
            done = False
            while not done:
                a, n = env._batched.fair_actions()
                _, _, done, _, _ = env.step({"stage_idx": int(a[0]), "num_exec": int(n[0])})
            completions = env._batched.episode_cursors()[0, 1].item()
            ep += 1
        win, fill = env._batched.job_duration_window()
        assert int(fill[0]) == 200 == len(env.job_duration_buff)
        np.testing.assert_array_equal(win[0].cpu().numpy(), np.asarray(env.job_duration_buff))
        s = env._batched.collect_stats().cpu().numpy()
        ref = np.mean(np.asarray(env.job_duration_buff))
        assert s[7] == 1.0
        assert abs(s[6] - ref) <= 1e-12 * abs(ref)
        facades.append(s)
        means.append(env.avg_job_duration)
    st = parallel.stats_from_sums(np.sum(facades, 0))
    assert abs(st["avg_job_duration"] - np.mean(means)) <= 1e-12 * abs(np.mean(means))


def test_ring_overflow_reset_stats_and_grow(bank):
    cfg = cfg_of(10, 8)
    B = 8
    env, seeds = make_env(bank, cfg, B, base=4000)
    env.attach_episode_log(capacity=2, window=16)
    env.rollout_fair(1500, auto_reset=True, seed_step=B)
    cur = env.episode_cursors().cpu().numpy()
    assert (cur[:, 0] > 2).all()
    e = env.episodes()
    dropped = e["dropped"].cpu().numpy()
    np.testing.assert_array_equal(dropped, cur[:, 0] - 2)
    ep = e["episode"].cpu().numpy().reshape(B, 2)
    np.testing.assert_array_equal(ep, np.stack([cur[:, 0] - 2, cur[:, 0] - 1], 1))
    # an explicit reset mid-episode writes no record and keeps the window; reset_stats keeps the decision count
    env.reset_host(seeds)
    env.rollout_fair(5, auto_reset=False)
    n0, w0 = env.episode_cursors()[:, 0].clone(), env.job_duration_window()[0].clone()
    env.reset_host(seeds)
    assert torch.equal(env.episode_cursors()[:, 0], n0)
    assert torch.equal(torch.nan_to_num(env.job_duration_window()[0]), torch.nan_to_num(w0))
    env.rollout_fair(3, auto_reset=False)
    env.reset_stats()
    env.clear_episodes()
    env.rollout_fair(2000, auto_reset=False)  # every env runs its episode to the end
    recs = host_records(env)
    want = oracle_episodes(bank, cfg, seeds[0], B, 1)[0]
    assert len(recs[0]) == 1 and recs[0][0]["decisions"] == want["decisions"]
    assert recs[0][0]["job_time"] == want["job_time"]
    # grow() keeps the log, the counts and the window
    cur0 = env.episode_cursors().clone()
    win0 = env.job_duration_window()[0].clone()
    env.grow(2 * env.max_jobs)
    assert torch.equal(env.episode_cursors()[:, :2], cur0[:, :2])
    assert torch.equal(torch.nan_to_num(env.job_duration_window()[0]), torch.nan_to_num(win0))
    env.reset_host(seeds)
    env.rollout_fair(2000, auto_reset=False)
    assert (env.episode_cursors()[:, 0] == cur0[:, 0] + 1).all()


def test_detached_and_refusals(bank):
    cfg = cfg_of(10, 8)
    B = 8
    env, seeds = make_env(bank, cfg, B, base=5000)
    env.attach_episode_log(capacity=4, window=8)
    rec, _, dur, _, cur = env._settings["episode_log"]
    env.detach_episode_log()
    env.rollout_fair(400, auto_reset=True, seed_step=B)
    assert int(rec.count_nonzero()) == 0 and int(dur.count_nonzero()) == 0
    assert int(cur.view(torch.int64).view(B, 4)[:, :2].count_nonzero()) == 0
    s = env.collect_stats().cpu().numpy()
    assert s[6] == 0.0 and s[7] == 0.0
    L, h, st = env.L, env._h, env._stream()
    p = cur.data_ptr()
    assert L.ssb_attach_episode_log(None, None, 0, None, 0, p, st) == -1
    for args in ((None, 4, None, 0), (rec.data_ptr(), 0, None, 0), (rec.data_ptr(), -1, None, 0),
                 (None, 0, None, 8), (None, 0, dur.data_ptr(), 0), (None, 0, dur.data_ptr(), -3)):
        assert L.ssb_attach_episode_log(h, args[0], args[1], args[2], args[3], p, st) == -1, args
    assert L.ssb_attach_episode_log(h, None, 0, None, 0, None, st) == 0
