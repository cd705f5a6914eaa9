"""The fused fair rollout (ssb_rollout_fair / _traj) writes the observation graph, and without a trajectory buffer
the reward, only for the observation that is live when the call returns.  These tests run the same seeds through
the eager step path (fair actions + ssb_step, one decision per call, envs masked once they have taken their K
decisions) and require the final state to be bit-identical: every header field, the valid rows of the four graph
slabs, the per-env counters and the job times."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

C2_LIKE = {"num_executors": 10, "job_arrival_cap": 12, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
TWO_SLOT = {"num_executors": 50, "job_arrival_cap": 20, "job_arrival_rate": 4.0e-5,
            "moving_delay": 2000.0, "warmup_delay": 1000.0}
B = 24


def _env(bank, cfg, seeds):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    env = BatchedSparkSchedSimEnv(cfg, num_envs=len(seeds), bank=bank)
    hdr = env.reset_host(np.asarray(seeds, np.uint64))
    assert (hdr["error"] == 0).all()
    return env


def eager(bank, cfg, seeds, K, dynamic=True, auto_reset=True):
    """K decisions per env through ssb_step; returns the env and per-env lists of (reward, wall before, wall after,
    flags) of every decision.  An ssb_step call that only re-seeds a finished env (was_reset) is not a decision."""
    import torch

    env = _env(bank, cfg, seeds)
    env.set_autoreset(auto_reset, 1)
    n_dec = np.zeros(len(seeds), np.int64)
    rows = [[] for _ in seeds]
    hdr = env.hdr()
    while True:
        live = n_dec < K
        if not auto_reset:
            live &= (hdr["terminated"] == 0) & (hdr["truncated"] == 0)
        if not live.any():
            break
        a, n = env.fair_actions(dynamic)
        wall0 = hdr["wall_time"].copy()
        env.step(a, n, mask=torch.as_tensor(live.astype(np.uint8)))
        hdr = env.hdr()
        assert (hdr["error"][live] == 0).all(), hdr["error"][live]
        for b in np.nonzero(live & (hdr["was_reset"] == 0))[0]:
            rows[b].append((hdr["reward"][b], wall0[b], hdr["wall_time"][b],
                            int(hdr["terminated"][b]) | 2 * int(hdr["truncated"][b])))
            n_dec[b] += 1
    return env, rows


def deferred(bank, cfg, seeds, K, dynamic=True, auto_reset=True, traj=False):
    env = _env(bank, cfg, seeds)
    tr = None
    if traj:
        import torch

        pin = torch.empty(len(seeds) * K * 32, dtype=torch.uint8).pin_memory()
        tr = env.rollout_fair_traj(K, dynamic, auto_reset, 1, host=pin).copy()
    else:
        env.rollout_fair(K, dynamic, auto_reset, 1)
    return env, tr


def assert_same_state(ref, got):
    h0, h1 = ref.hdr(), got.hdr()
    assert h0.tobytes() == h1.tobytes(), [f for f in h0.dtype.names if not np.array_equal(h0[f], h1[f])]
    assert ref.stats_per_env().tobytes() == got.stats_per_env().tobytes()
    for b in range(len(h0)):
        o0, o1 = ref.obs(b, h0), got.obs(b, h1)
        for k in ("nodes", "edge_links", "dag_ptr", "exec_supplies"):
            assert o0[k].tobytes() == o1[k].tobytes(), (b, k)
        for x, y in zip(ref.jobs(b), got.jobs(b)):
            assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), b


def assert_same_traj(rows, tr, K):
    for b, r in enumerate(rows):
        assert len(r) == K
        for d, (rew, w0, _, fl) in enumerate(r):
            t = tr[b, d]
            assert np.float64(t["reward"]).tobytes() == np.float64(rew).tobytes(), (b, d)
            assert t["wall_time"] == w0 and (t["flags"] & 3) == fl, (b, d)


SEEDS = 1234 + np.arange(B)


@pytest.mark.parametrize("traj", [False, True])
@pytest.mark.parametrize("K", [1, 2, 37, 128])
def test_fair_matches_eager(bank, K, traj):
    ref, rows = eager(bank, C2_LIKE, SEEDS, K)
    got, tr = deferred(bank, C2_LIKE, SEEDS, K, traj=traj)
    assert_same_state(ref, got)
    if traj:
        assert_same_traj(rows, tr, K)


@pytest.mark.parametrize("traj", [False, True])
def test_fifo_matches_eager(bank, traj):
    ref, rows = eager(bank, C2_LIKE, SEEDS, 37, dynamic=False)
    got, tr = deferred(bank, C2_LIKE, SEEDS, 37, dynamic=False, traj=traj)
    assert_same_state(ref, got)
    if traj:
        assert_same_traj(rows, tr, 37)


@pytest.mark.parametrize("traj", [False, True])
def test_two_slot_matches_eager(bank, traj):
    seeds = 77 + np.arange(8)
    ref, rows = eager(bank, TWO_SLOT, seeds, 50)
    got, tr = deferred(bank, TWO_SLOT, seeds, 50, traj=traj)
    assert_same_state(ref, got)
    if traj:
        assert_same_traj(rows, tr, 50)


def test_episodes_to_the_end_without_auto_reset(bank):
    seeds = 500 + np.arange(8)
    ref, _ = eager(bank, C2_LIKE, seeds, 1 << 30, auto_reset=False)
    got, _ = deferred(bank, C2_LIKE, seeds, 100000, auto_reset=False)
    assert (got.hdr()["terminated"] == 1).all()
    assert_same_state(ref, got)


def test_last_decision_terminates_the_episode(bank):
    """K = the oracle's decision count of env 0's first episode: the rollout ends on the terminal observation, whose
    reward (owed until the loop ends) is not zero; auto-reset is on but never runs."""
    from oracle import OracleEnv

    cfg = C2_LIKE
    orc = OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                    cfg["job_arrival_rate"])
    orc.reset_seed(int(SEEDS[0]))
    K, term = 0, False
    while not term:
        a, n = orc.fair_action(True)
        rc, _, term = orc.step(a, n)
        assert rc == 0
        K += 1
    ref, _ = eager(bank, cfg, SEEDS, K)
    got, _ = deferred(bank, cfg, SEEDS, K)
    h = got.hdr()[0]
    assert h["terminated"] == 1 and h["reward"] != 0.0
    assert_same_state(ref, got)


@pytest.mark.parametrize("traj", [False, True])
def test_last_decision_in_the_same_round(bank, traj):
    """K such that env b's K-th decision continues the commitment round (the wall time does not advance): the owed
    graph is written, the reward stays the 0 of a same-round observation."""
    _, rows = eager(bank, C2_LIKE, SEEDS, 40)
    b, K = next((b, d + 1) for b, r in enumerate(rows) for d, x in enumerate(r) if d >= 2 and x[1] == x[2])
    ref, rows = eager(bank, C2_LIKE, SEEDS, K)
    assert rows[b][-1][1] == rows[b][-1][2]
    got, tr = deferred(bank, C2_LIKE, SEEDS, K, traj=traj)
    assert got.hdr()[b]["reward"] == 0.0
    assert_same_state(ref, got)
    if traj:
        assert_same_traj(rows, tr, K)
