"""Fixed-duration random-policy rollouts (ssb_rollout_random_async, RolloutWorkerAsync.collect_rollout,
rollout_worker.py:160-206) against the worker's loop restated over the CPU oracle driven with the spec's draws
(tests/random_policy_spec.py), against the fused rollout_random where the duration never binds, and at full batch
size against their caps and for determinism."""
import numpy as np
import pytest

from random_policy_spec import random_policy_action

pytestmark = pytest.mark.gpu


def cfg_of(E, J, beta=0.0):
    return {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
            "warmup_delay": 1000.0, "beta": beta}


def make_env(bank, cfg, seeds, mean_time_limit=0.0, **kw):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    env = BatchedSparkSchedSimEnv(cfg, num_envs=len(seeds), bank=bank, **kw)
    if mean_time_limit > 0:
        env.set_mean_time_limit(mean_time_limit)
    hdr = env.reset_host(np.asarray(seeds, np.uint64))
    assert (hdr["error"] == 0).all()
    return env


def async_calls(env, calls, kmax, dur, seed_step):
    """`calls` consecutive rollout_random_async calls -> [(rows [B, kmax], num_steps [B], elapsed [B])]."""
    from spark_sched_sim_b200 import _native as nat

    out = []
    for _ in range(calls):
        traj, num, el = env.rollout_random_async(kmax, dur, seed_step)
        out.append((traj.cpu().numpy().view(nat.TRANSITION_DTYPE).reshape(env.num_envs, kmax), num.cpu().numpy(),
                    el.cpu().numpy()))
    assert (env.hdr()["error"] == 0).all()
    return out


def worker_loop(bank, cfg, seed, calls, kmax, dur, seed_step, mean_time_limit=0.0):
    """RolloutWorkerAsync.collect_rollout over the oracle with the random policy, `calls` times in a row: each call
    steps until its accumulated simulated time reaches dur or kmax rows are stored; a finished episode is re-seeded
    with seed + seed_step * reset_count when the loop comes back around (also in the next call).  The action of
    decision d of an episode is the spec's draw d on the episode seed; with mean_time_limit > 0 every episode's limit
    is the StochasticTimeLimit draw of its seed.  Returns [(rows (elapsed, reward, stage_idx, num_exec, flags),
    elapsed)] per call and the number of episodes ended by truncation."""
    from oracle import OracleEnv
    from philox_ref import time_limit_draw

    orc = OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                    cfg["job_arrival_rate"], cfg.get("beta", 0.0))
    ep, d, done, n_trunc = 0, 0, False, 0
    s = int(seed)
    tl = time_limit_draw(s, mean_time_limit) if mean_time_limit > 0 else np.inf
    orc.reset_seed(s, tl)
    out = []
    for _ in range(calls):
        rows, elapsed = [], 0.0
        while elapsed < dur and len(rows) < kmax:
            if done:
                ep += 1
                s = int(seed) + seed_step * ep
                tl = time_limit_draw(s, mean_time_limit) if mean_time_limit > 0 else np.inf
                orc.reset_seed(s, tl)
                d, done = 0, False
                continue
            wall0 = orc.wall_time
            a, n = random_policy_action(orc.obs(), s, d)
            rc, rew, term = orc.step(a, n)
            assert rc == 0, (seed, ep, d, rc)
            trunc = orc.wall_time >= tl  # StochasticTimeLimit (wrappers/stochastic_time_limit.py:29-30)
            rows.append((elapsed, rew, a, n, int(term) | 2 * int(trunc) | (4 if d == 0 and ep > 0 else 0)))
            elapsed += orc.wall_time - wall0
            n_trunc += trunc
            done = term or trunc
            d += 1
        out.append((rows, elapsed))
    return out, n_trunc


def assert_calls_match(bank, cfg, seeds, got, kmax, dur, seed_step, mean_time_limit=0.0, reward_rtol=0.0):
    """Every row, num_steps and elapsed of every call equal the worker loop's; returns (resets, truncations)."""
    n_resets = n_trunc = 0
    for b in range(len(seeds)):
        want, tr = worker_loop(bank, cfg, seeds[b], len(got), kmax, dur, seed_step, mean_time_limit)
        n_trunc += tr
        for c, ((rows, elapsed), (traj, num, el)) in enumerate(zip(want, got)):
            assert (num[b], el[b]) == (len(rows), elapsed), (b, c, num[b], len(rows))
            for k, (w, rew, a, n, fl) in enumerate(rows):
                r = traj[b, k]
                assert (r["wall_time"], r["stage_idx"], r["num_exec"], r["flags"], r["lgprob"]) == (w, a, n, fl, 0.0), \
                    (b, c, k)
                if reward_rtol:
                    assert abs(r["reward"] - rew) <= reward_rtol * max(abs(rew), 1e-300), (b, c, k, r["reward"], rew)
                else:
                    assert np.float64(r["reward"]).tobytes() == np.float64(rew).tobytes(), (b, c, k)
                n_resets += fl >> 2
    return n_resets, n_trunc


def test_async_rollouts_match_reference_loop(bank):
    """Three consecutive calls at E = 10, J = 5: rows (accumulated time, action, reward, flags), num_steps and elapsed
    equal the worker's loop over the oracle, with resets inside the calls and state carried over to the next."""
    B, KMAX, DUR, STEP = 4, 2000, 2.0e6, 9
    cfg = cfg_of(10, 5)
    seeds = np.arange(80, 80 + B, dtype=np.uint64)
    env = make_env(bank, cfg, seeds)
    got = async_calls(env, 3, KMAX, DUR, STEP)
    n_resets, _ = assert_calls_match(bank, cfg, seeds, got, KMAX, DUR, STEP)
    assert n_resets >= B


@pytest.mark.parametrize("beta", [0.0, 5.0e-3])
def test_async_rollouts_with_truncation(bank, beta):
    """Continuous arrivals under a stochastic time limit: episodes end by truncation (flag 2) and are re-seeded
    inside the rollout; with beta > 0 rewards at 1e-12 relative (device exp vs libm), everything else exact."""
    B, KMAX, DUR, STEP, MEAN = 4, 1500, 1.5e6, 17, 3.0e5
    cfg = cfg_of(10, 0, beta)
    seeds = np.arange(60, 60 + B, dtype=np.uint64)
    env = make_env(bank, cfg, seeds, mean_time_limit=MEAN, max_jobs=128)
    got = async_calls(env, 2, KMAX, DUR, STEP)
    n_resets, n_trunc = assert_calls_match(bank, cfg, seeds, got, KMAX, DUR, STEP, MEAN,
                                           reward_rtol=1e-12 if beta else 0.0)
    assert n_trunc > B and n_resets >= n_trunc - B


@pytest.mark.parametrize("E", [50, 45])
def test_two_slot_kernel_matches_reference_loop(bank, E):
    """E in 33..64 runs k_rollout_random_async<2>: a few hundred decisions per env over two calls."""
    B, KMAX, DUR, STEP = 3, 200, 1.0e6, 5
    cfg = cfg_of(E, 20)
    seeds = np.arange(500, 500 + B, dtype=np.uint64)
    env = make_env(bank, cfg, seeds)
    got = async_calls(env, 2, KMAX, DUR, STEP)
    assert sum(int(num.sum()) for _, num, _ in got) > 200 * B
    assert_calls_match(bank, cfg, seeds, got, KMAX, DUR, STEP)


def step_durations(sync, live_wall):
    """[B, K] duration of every step of a recorded rollout_random: within an episode the wall time before the next
    step minus the wall time before this one, after the last row the live wall time minus it; NaN for a step that
    ended its episode (the wall time after it is not recorded)."""
    w = sync["wall_time"]
    dur = np.empty(w.shape)
    dur[:, :-1] = w[:, 1:] - w[:, :-1]
    dur[:, -1] = live_wall - w[:, -1]
    dur[(sync["flags"] & 3) != 0] = np.nan
    return dur


def assert_time_axis(tr, num, el, dur):
    """The async rows' time axis is the running f64 sum of the step durations in row order, starting at 0, and elapsed
    is the sum over the rows stored; checked wherever the duration is known.  Returns how many envs were checked."""
    B, K = tr.shape
    e = tr["wall_time"]
    assert (e[:, 0] == 0.0).all()
    for b in range(B):
        n = int(num[b])
        known = ~np.isnan(dur[b, :n])
        nxt = np.append(e[b, 1:n], el[b])  # the running sum after each row
        assert np.array_equal(nxt[known], (e[b, :n] + dur[b, :n])[known]), b
        assert (nxt[~known] >= e[b, :n][~known]).all(), b
    return int((~np.isnan(dur)).all(axis=1).sum())


@pytest.mark.parametrize("B,E,J,K", [(4096, 10, 50, 128), (512, 50, 200, 64)])
def test_async_equals_sync_when_the_duration_never_binds(bank, B, E, J, K):
    """C2's shape (and C4's episode shape with fewer envs): with rollout_duration = inf, rollout_random_async(K) takes
    the decisions rollout_random(K, record=True) takes on a second handle from the same seeds -- the same actions,
    rewards and flags, and the same state afterwards -- and its time axis is the running sum of their durations."""
    from spark_sched_sim_b200 import _native as nat

    cfg = cfg_of(E, J)
    seeds = (77 + np.arange(B)).astype(np.uint64)
    STEP = 3
    env_a, env_s = make_env(bank, cfg, seeds), make_env(bank, cfg, seeds)
    sync = env_s.rollout_random(K, seed_step=STEP, record=True).cpu().numpy().view(nat.TRANSITION_DTYPE).reshape(B, K)
    (tr, num, el), = async_calls(env_a, 1, K, np.inf, STEP)
    assert (num == K).all()
    for f in ("stage_idx", "num_exec", "flags", "lgprob"):
        assert np.array_equal(tr[f], sync[f]), f
    assert tr["reward"].tobytes() == sync["reward"].tobytes()
    hs = env_s.hdr()
    assert env_a.hdr().tobytes() == hs.tobytes()
    assert assert_time_axis(tr, num, el, step_durations(sync, hs["wall_time"])) > 0


def test_caps_and_determinism_at_full_size(bank):
    """4096 envs x (50 jobs, 10 executors), a duration that binds for part of the envs: every env stopped at
    max_decisions or at the duration (and not before), elapsed is the f64 sum of its rows' durations in row order
    (durations from a recorded rollout_random on a third handle), envs sharing a seed act identically, and a second
    handle from the same seeds gives byte-identical rows, num_steps and elapsed over two calls."""
    from spark_sched_sim_b200 import _native as nat

    B, KMAX, DUR, STEP = 4096, 128, 5.5e6, 11
    cfg = cfg_of(10, 50)
    seeds = (1234 + np.arange(B) // 2).astype(np.uint64)  # pairs share a seed
    runs = [async_calls(make_env(bank, cfg, seeds), 2, KMAX, DUR, STEP) for _ in range(2)]
    for (t0, n0, e0), (t1, n1, e1) in zip(*runs):
        assert t0.tobytes() == t1.tobytes() and n0.tobytes() == n1.tobytes() and e0.tobytes() == e1.tobytes()
    n_dur = 0
    for tr, num, el in runs[0]:
        assert ((num == KMAX) | (el >= DUR)).all()
        assert (tr["wall_time"][np.arange(B), num - 1] < DUR).all()  # the duration had not run out before the last row
        n_dur += int((num < KMAX).sum())
        for b in range(0, B, 2):
            assert tr[b, :num[b]].tobytes() == tr[b + 1, :num[b]].tobytes(), b
        assert np.array_equal(num[0::2], num[1::2]) and np.array_equal(el[0::2], el[1::2])
    assert 0 < n_dur < 2 * B  # both caps bind somewhere
    tr, num, el = runs[0][0]
    env_s = make_env(bank, cfg, seeds)
    sync = env_s.rollout_random(KMAX, seed_step=STEP, record=True).cpu().numpy().view(
        nat.TRANSITION_DTYPE).reshape(B, KMAX)
    stored = np.arange(KMAX) < num[:, None]
    for f in ("stage_idx", "num_exec", "flags", "reward"):
        assert np.array_equal(tr[f][stored], sync[f][stored]), f
    assert assert_time_axis(tr, num, el, step_durations(sync, env_s.hdr()["wall_time"])) > 0


def test_invalid_arguments_and_null_outputs(bank):
    """Through the raw ABI: max_decisions < 0 and rollout_duration <= 0 (or NaN) are SSB_E_INVALID (-1) and change
    nothing; traj, num_steps and elapsed may all be NULL, and such a call takes the decisions a call with every output
    given takes."""
    import torch

    cfg = cfg_of(10, 5)
    seeds = np.arange(3, dtype=np.uint64)
    env, ref = make_env(bank, cfg, seeds), make_env(bank, cfg, seeds)
    L, h, stream = env.L, env._h, env._stream()
    num = torch.full((3,), 7, dtype=torch.int32, device=env.device)
    el = torch.full((3,), 1.0, dtype=torch.float64, device=env.device)
    h0 = env.hdr().copy()
    for kmax, dur in ((-1, 1.0e5), (10, 0.0), (10, -1.0), (10, float("nan"))):
        assert L.ssb_rollout_random_async(h, kmax, dur, 1, None, num.data_ptr(), el.data_ptr(), stream) == -1
    assert L.ssb_rollout_random_async(None, 10, 1.0e5, 1, None, None, None, stream) == -1
    assert env.hdr().tobytes() == h0.tobytes()
    assert L.ssb_rollout_random_async(h, 0, 1.0e5, 1, None, num.data_ptr(), el.data_ptr(), stream) == 0
    assert (num.cpu().numpy() == 0).all() and (el.cpu().numpy() == 0.0).all()
    assert L.ssb_rollout_random_async(h, 10, 1.0e5, 1, None, None, None, stream) == 0
    _, n_ref, _ = ref.rollout_random_async(10, 1.0e5, 1)
    hdr, taken = env.hdr(), env.stats_per_env()["decisions"]
    assert (hdr["error"] == 0).all() and (taken > 0).all()
    assert np.array_equal(taken, n_ref.cpu().numpy()) and hdr.tobytes() == ref.hdr().tobytes()
