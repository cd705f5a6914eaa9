"""The random scheduler on the device (ssb_random_actions, ssb_rollout_random) against the CPU oracle driven with the
same draws (tests/random_policy_spec.py: the RANDOM stream on the oracle's observation), and at full batch size
against its law.  tests/test_gpu_rollout_deferred_obs.py compares ssb_rollout_random with the eager step path."""
import numpy as np
import pytest
from scipy.stats import chisquare

from random_policy_spec import random_policy_action

pytestmark = pytest.mark.gpu


def cfg_of(E, J, rate=4.0e-5, beta=0.0):
    return {"num_executors": E, "job_arrival_cap": J, "job_arrival_rate": rate, "moving_delay": 2000.0,
            "warmup_delay": 1000.0, "beta": beta}


def make_env(bank, cfg, seeds, time_limit=None, **kw):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    env = BatchedSparkSchedSimEnv(cfg, num_envs=len(seeds), bank=bank, **kw)
    tl = None if time_limit is None else np.full(len(seeds), time_limit)
    hdr = env.reset_host(np.asarray(seeds, np.uint64), time_limits=tl)
    assert (hdr["error"] == 0).all()
    return env


def oracle(bank, cfg, log=False):
    from oracle import OracleEnv

    return OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                     cfg["job_arrival_rate"], cfg.get("beta", 0.0), log=log)


def oracle_loop(bank, cfg, seed, K, seed_step=1, time_limit=np.inf, auto_reset=True):
    """K random-policy decisions of the oracle (auto_reset=False: until the first episode ends), re-seeding finished
    episodes with seed + seed_step * reset_count.  Returns the oracle, the rows (wall before, reward, stage_idx,
    num_exec, flags) and the events of the episodes."""
    orc = oracle(bank, cfg, log=True)
    rows, k, ep, events = [], 0, 0, 0
    while k < K:
        s = int(seed) + seed_step * ep
        orc.reset_seed(s, time_limit)
        d, done = 0, False
        while not done and k < K:
            wall0 = orc.wall_time
            a, n = random_policy_action(orc.obs(), s, d)
            rc, rew, term = orc.step(a, n)
            assert rc == 0, (seed, ep, d, rc)
            trunc = orc.wall_time >= time_limit  # StochasticTimeLimit (wrappers/stochastic_time_limit.py:29-30)
            rows.append((wall0, rew, a, n, int(term) | 2 * int(trunc) | (4 if d == 0 and ep > 0 else 0)))
            done = term or trunc
            d += 1
            k += 1
        events += orc.log_size()
        ep += 1
        if not auto_reset:
            break
    return orc, rows, events


def assert_same_jobs(orc, env, b):
    ta, tc, tm = orc.job_times()
    gta, gtc, gtm = env.jobs(b)
    assert np.array_equal(ta, gta) and np.array_equal(tm, gtm), b
    assert np.asarray(tc).tobytes() == np.asarray(gtc).tobytes(), (b, "job completion times")


def test_random_actions_on_mixed_states(bank):
    """Envs advanced by fair decisions, run to termination, left pending by a budgeted step or masked out:
    random_actions equals the oracle's draw on every served env's observation; done, pending and masked-out envs get
    (-1, 1) and keep their draw counter; a second call without a step gives the next draw."""
    import torch

    cfg = cfg_of(10, 12)
    B = 12
    seeds = 300 + np.arange(B)
    env = make_env(bank, cfg, seeds)
    env.set_autoreset(False)
    n_fair = np.array([0, 1, 2, 5, 9, 3, 0, 4, 7, 1, 0, 6])
    orcs = []
    for b in range(B):
        o = oracle(bank, cfg)
        o.reset_seed(int(seeds[b]))
        orcs.append(o)
    done_set, pend_set, masked = [4, 5], [7, 8, 9], [10, 11]

    def fair_steps(mask, max_events=0):
        a, n = env.fair_actions(True)
        env.step(a, n, mask=torch.as_tensor(mask.astype(np.uint8)), max_events=max_events)
        return a.cpu().numpy(), n.cpu().numpy()

    for r in range(n_fair.max()):
        live = n_fair > r
        a, n = fair_steps(live)
        for b in np.nonzero(live)[0]:
            assert orcs[b].step(int(a[b]), int(n[b]))[0] == 0
    while True:  # done_set to the end of their episodes
        hdr = env.hdr()
        live = np.zeros(B, bool)
        live[done_set] = hdr["terminated"][done_set] == 0
        if not live.any():
            break
        fair_steps(live)
    a_p, n_p = fair_steps(np.isin(np.arange(B), pend_set), max_events=1)
    hdr = env.hdr()
    pending = [b for b in pend_set if hdr["pending"][b]]
    assert pending, "no env left pending by the budgeted step"
    for b in pend_set:
        assert orcs[b].step(int(a_p[b]), int(n_p[b]))[0] == 0
    mask = ~np.isin(np.arange(B), masked)
    served = [b for b in range(B) if mask[b] and b not in done_set and b not in pending]

    def check(got, expect_draw):
        a, n = (x.cpu().numpy() for x in got)
        for b in range(B):
            d = expect_draw.get(b)
            want = (-1, 1) if d is None else random_policy_action(orcs[b].obs(), int(seeds[b]), d)
            assert (a[b], n[b]) == want, (b, d)

    mask_t = torch.as_tensor(mask.astype(np.uint8))
    check(env.random_actions(mask_t), {b: 0 for b in served})
    check(env.random_actions(mask_t), {b: 1 for b in served})
    check(env.random_actions(), {**{b: 2 for b in served}, **{b: 0 for b in masked}})
    fair_steps(np.isin(np.arange(B), pending))  # the pending step ends (its action is ignored)
    assert env.hdr()["pending"].sum() == 0
    check(env.random_actions(torch.as_tensor(np.isin(np.arange(B), pending).astype(np.uint8))),
          {b: 0 for b in pending})


@pytest.mark.parametrize("E,J", [(3, 10), (10, 50), (33, 20), (50, 30), (64, 40), (100, 30), (50, 200)])
def test_episodes_match_oracle(bank, E, J):
    """rollout_random to the end of every episode: every job's arrival and completion time, the final wall time and
    the decision and event counts equal a host loop of the spec's action on the oracle's observation + step from the same seeds (one-slot,
    two-slot and general-only paths; (50, 200) is the C4 episode shape)."""
    cfg = cfg_of(E, J)
    B = 8 if J < 200 else 3
    seeds = 2000 + 17 * np.arange(B)
    env = make_env(bank, cfg, seeds)
    env.rollout_random(10**6, auto_reset=False)
    hdr = env.hdr()
    assert (hdr["error"] == 0).all() and (hdr["terminated"] == 1).all()
    st = env.stats_per_env()
    for b in range(B):
        orc, rows, events = oracle_loop(bank, cfg, seeds[b], 10**9, auto_reset=False)
        assert_same_jobs(orc, env, b)
        assert hdr["wall_time"][b] == orc.wall_time, b
        assert (st["decisions"][b], st["events"][b]) == (len(rows), events), b


def test_episodes_with_discount_and_time_limit(bank):
    """beta > 0 (the reward goes through exp()), and time-limited arrivals that end episodes by truncation."""
    import torch
    from spark_sched_sim_b200 import _native as nat

    cfg = cfg_of(10, 20, beta=5.0e-3)
    seeds = 70 + np.arange(4)
    env = make_env(bank, cfg, seeds)
    K = 300
    host = torch.empty(len(seeds) * K * nat.TRANSITION_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    tr = env.rollout_random(K, auto_reset=True, seed_step=10, record=True, host=host)
    for b in range(len(seeds)):
        _, rows, _ = oracle_loop(bank, cfg, seeds[b], K, seed_step=10)
        for k, (w0, rew, a, n, fl) in enumerate(rows):
            r = tr[b, k]
            assert (r["wall_time"], r["stage_idx"], r["num_exec"], r["flags"]) == (w0, a, n, fl), (b, k)
            assert abs(r["reward"] - rew) <= 1e-12 * max(abs(rew), 1e-300), (b, k)
    TL = 4.0e5
    cfg = cfg_of(10, 0)
    seeds = 900 + np.arange(4)
    env = make_env(bank, cfg, seeds, time_limit=TL, max_jobs=96)
    env.rollout_random(10**6, auto_reset=False)
    hdr = env.hdr()
    assert (hdr["error"] == 0).all() and (hdr["truncated"] == 1).any()
    st = env.stats_per_env()
    for b in range(len(seeds)):
        orc, rows, events = oracle_loop(bank, cfg, seeds[b], 10**9, time_limit=TL, auto_reset=False)
        assert (rows[-1][4] & 3) == int(hdr["terminated"][b]) | 2 * int(hdr["truncated"][b]), b
        assert_same_jobs(orc, env, b)
        assert hdr["wall_time"][b] == orc.wall_time, b
        assert (st["decisions"][b], st["events"][b]) == (len(rows), events), b


TRAJ_CFG = cfg_of(10, 5)


@pytest.mark.parametrize("K", [1, 2, 37, 128])
def test_transitions_across_resets(bank, K):
    """rollout_random(K, record=True, seed_step=100): every row (wall time, reward bytes, action, flags 1/2/4) and the
    live observation afterwards (header, graph, reward) equal the oracle loop across episode boundaries; the same K
    decisions split over several launches give the same rows and state."""
    import torch
    from spark_sched_sim_b200 import _native as nat

    seeds = 40 + np.arange(6)
    B = len(seeds)
    env = make_env(bank, TRAJ_CFG, seeds)
    host = torch.empty(B * K * nat.TRANSITION_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    tr = env.rollout_random(K, seed_step=100, record=True, host=host).copy()
    hdr = env.hdr()
    assert (hdr["error"] == 0).all()
    n_fresh = 0
    for b in range(B):
        orc, rows, _ = oracle_loop(bank, TRAJ_CFG, seeds[b], K, seed_step=100)
        for k, (w0, rew, a, n, fl) in enumerate(rows):
            r = tr[b, k]
            assert (r["wall_time"], r["stage_idx"], r["num_exec"], r["flags"], r["lgprob"]) == (w0, a, n, fl, 0.0), \
                (b, k)
            assert np.float64(r["reward"]).tobytes() == np.float64(rew).tobytes(), (b, k)
            n_fresh += fl >> 2
        h = hdr[b]
        assert h["wall_time"] == orc.wall_time and h["reward"] == rows[-1][1], b
        assert h["terminated"] == rows[-1][4] & 1, b
        o, g = orc.obs(), env.obs(b, hdr)
        for key in ("nodes", "edge_links", "dag_ptr", "exec_supplies"):
            assert np.array_equal(o[key], g[key]), (b, key)
        assert (o["num_committable_execs"], o["source_job_idx"]) == (g["num_committable_execs"], g["source_job_idx"])
    if K == 128:
        assert n_fresh > 0
    if K > 1:
        split = make_env(bank, TRAJ_CFG, seeds)
        parts, done = [], 0
        for k in (K // 3, K // 3 + 1, K - 2 * (K // 3) - 1):
            if k > 0:
                hp = torch.empty(B * k * nat.TRANSITION_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
                parts.append(split.rollout_random(k, seed_step=100, record=True, host=hp).copy())
                done += k
        assert done == K
        assert np.concatenate(parts, axis=1).tobytes() == tr.tobytes()
        assert split.hdr().tobytes() == hdr.tobytes()


def test_full_batch_law_and_determinism(bank):
    """4096 envs x (50 jobs, 10 executors): the first random decision (taken after 40 fair ones, so that several
    jobs are active) picks its job uniformly among the eligible jobs and num_exec uniformly (chi-square per eligible /
    committable count, p > 1e-4 at fixed seeds); envs sharing a seed act identically; two runs are bit-identical; the
    whole batch runs to termination without an env error."""
    B = 4096
    cfg = cfg_of(10, 50)
    seeds = (1234 + np.arange(B) // 2).astype(np.uint64)  # pairs share a seed
    env = make_env(bank, cfg, seeds)
    env.rollout_fair(40, True, auto_reset=False)
    hdr = env.hdr()
    a, n = (x.cpu().numpy() for x in env.random_actions())
    sched = (env.nodes[:, :, 2] != 0).cpu().numpy()
    dag_ptr = env.dag_ptr.cpu().numpy()
    pos_by_k, exec_by_c = {}, {}
    for b in range(0, B, 2):
        Ja, N, c = int(hdr["num_active_jobs"][b]), int(hdr["num_nodes"][b]), int(hdr["num_committable_execs"][b])
        if hdr["terminated"][b] or N == 0:
            continue
        s = sched[b, :N]
        job_of = np.searchsorted(dag_ptr[b, :Ja + 1], np.arange(N), side="right") - 1
        elig = sorted(set(job_of[s].tolist()))
        assert a[b] >= 0, b
        node = np.flatnonzero(s)[a[b]]
        pos_by_k.setdefault(len(elig), []).append(elig.index(job_of[node]))
        exec_by_c.setdefault(c, []).append(n[b] - 1)
        assert 1 <= n[b] <= c
    tested = 0
    for groups in (pos_by_k, exec_by_c):
        for k, xs in groups.items():
            if k >= 2 and len(xs) >= 10 * k:
                assert chisquare(np.bincount(xs, minlength=k)).pvalue > 1e-4, (k, len(xs))
                tested += 1
    assert tested >= 3
    assert np.array_equal(a[0::2], a[1::2]) and np.array_equal(n[0::2], n[1::2])
    finals = []
    for _ in range(2):
        env.reset_stats()
        env.reset_host(seeds)
        env.rollout_random(10**6, auto_reset=False)
        h = env.hdr()
        assert (h["error"] == 0).all() and (h["terminated"] == 1).all()
        finals.append((h.tobytes(), env.stats_per_env().tobytes()))
        assert np.array_equal(h["wall_time"][0::2], h["wall_time"][1::2])
    assert finals[0] == finals[1]
    assert env.stats()["episodes"] == B
    for b in (0, 1, 2049):
        assert env.jobs(b)[1].tobytes() == env.jobs(b ^ 1)[1].tobytes()
