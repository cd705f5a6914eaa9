"""The fused rollouts (ssb_rollout_fair / _traj with the fair or FIFO policy, ssb_rollout_random) write the
observation graph, and without a trajectory buffer the reward, only for the observation that is live when the call
returns.  These tests run the same seeds through the eager step path (the policy's one-decision actions + ssb_step,
one decision per call, envs masked once they have taken their K decisions) and require the final state to be
bit-identical: every header field, the valid rows of the four graph slabs, the per-env counters and the job times;
with a buffer, every transition row equals the eager decision's."""
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


def eager(bank, cfg, seeds, K, policy="fair", auto_reset=True):
    """K decisions per env of `policy` ("fair", "fifo" or "random") through ssb_step; returns the env and per-env
    lists of (reward, wall before, wall after, stage_idx, num_exec, flags) of every decision.  An ssb_step call that
    only re-seeds a finished env (was_reset) is not a decision; the decision after it has flag 4."""
    import torch

    env = _env(bank, cfg, seeds)
    env.set_autoreset(auto_reset, 1)
    n_dec = np.zeros(len(seeds), np.int64)
    fresh = np.zeros(len(seeds), bool)
    rows = [[] for _ in seeds]
    hdr = env.hdr()
    while True:
        live = n_dec < K
        if not auto_reset:
            live &= (hdr["terminated"] == 0) & (hdr["truncated"] == 0)
        if not live.any():
            break
        mask = torch.as_tensor(live.astype(np.uint8))
        # the random policy's draws advance only for the envs it serves
        a, n = env.random_actions(mask) if policy == "random" else env.fair_actions(policy == "fair")
        wall0 = hdr["wall_time"].copy()
        env.step(a, n, mask=mask)
        hdr = env.hdr()
        a, n = a.cpu().numpy(), n.cpu().numpy()
        assert (hdr["error"][live] == 0).all(), hdr["error"][live]
        for b in np.nonzero(live)[0]:
            if hdr["was_reset"][b]:
                fresh[b] = True
                continue
            rows[b].append((hdr["reward"][b], wall0[b], hdr["wall_time"][b], a[b], n[b],
                            int(hdr["terminated"][b]) | 2 * int(hdr["truncated"][b]) | 4 * int(fresh[b])))
            fresh[b] = False
            n_dec[b] += 1
    return env, rows


def deferred(bank, cfg, seeds, K, policy="fair", auto_reset=True, traj=False):
    """The same K decisions per env in one fused rollout; returns the env and, with traj, the transition rows."""
    import torch

    env = _env(bank, cfg, seeds)
    pin = torch.empty(len(seeds) * K * 32, dtype=torch.uint8).pin_memory() if traj else None
    if policy == "random":
        tr = env.rollout_random(K, auto_reset, 1, record=traj, host=pin)
    elif traj:
        tr = env.rollout_fair_traj(K, policy == "fair", auto_reset, 1, host=pin)
    else:
        tr = env.rollout_fair(K, policy == "fair", auto_reset, 1)
    return env, (tr.copy() if traj else None)


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
        for d, (rew, w0, _, a, n, fl) in enumerate(r):
            t = tr[b, d]
            assert np.float64(t["reward"]).tobytes() == np.float64(rew).tobytes(), (b, d)
            assert (t["wall_time"], t["stage_idx"], t["num_exec"], t["flags"], t["lgprob"]) == (w0, a, n, fl, 0.0), \
                (b, d)


def check_matches_eager(bank, cfg, seeds, K, policy, traj):
    ref, rows = eager(bank, cfg, seeds, K, policy)
    got, tr = deferred(bank, cfg, seeds, K, policy, traj=traj)
    assert_same_state(ref, got)
    if traj:
        assert_same_traj(rows, tr, K)
    return got


SEEDS = 1234 + np.arange(B)
TWO_SLOT_SEEDS = 77 + np.arange(8)


@pytest.mark.parametrize("traj", [False, True])
@pytest.mark.parametrize("K", [1, 2, 37, 128])
def test_fair_matches_eager(bank, K, traj):
    check_matches_eager(bank, C2_LIKE, SEEDS, K, "fair", traj)


@pytest.mark.parametrize("traj", [False, True])
@pytest.mark.parametrize("K", [1, 2, 37, 128])
def test_random_matches_eager(bank, K, traj):
    check_matches_eager(bank, C2_LIKE, SEEDS, K, "random", traj)


@pytest.mark.parametrize("traj", [False, True])
def test_fifo_matches_eager(bank, traj):
    check_matches_eager(bank, C2_LIKE, SEEDS, 37, "fifo", traj)


@pytest.mark.parametrize("traj", [False, True])
def test_two_slot_matches_eager(bank, traj):
    check_matches_eager(bank, TWO_SLOT, TWO_SLOT_SEEDS, 50, "fair", traj)


@pytest.mark.parametrize("traj", [False, True])
def test_two_slot_random_matches_eager(bank, traj):
    check_matches_eager(bank, TWO_SLOT, TWO_SLOT_SEEDS, 50, "random", traj)


def test_episodes_to_the_end_without_auto_reset(bank):
    seeds = 500 + np.arange(8)
    ref, _ = eager(bank, C2_LIKE, seeds, 1 << 30, auto_reset=False)
    got, _ = deferred(bank, C2_LIKE, seeds, 100000, auto_reset=False)
    assert (got.hdr()["terminated"] == 1).all()
    assert_same_state(ref, got)


def first_episode_length(bank, cfg, seed, policy):
    """The oracle's decision count of the episode from `seed` under `policy` ("fair" or "random")."""
    from oracle import OracleEnv
    from random_policy_spec import random_policy_action

    orc = OracleEnv(bank, cfg["num_executors"], cfg["job_arrival_cap"], cfg["moving_delay"], cfg["warmup_delay"],
                    cfg["job_arrival_rate"])
    orc.reset_seed(int(seed))
    K, term = 0, False
    while not term:
        a, n = random_policy_action(orc.obs(), int(seed), K) if policy == "random" else orc.fair_action(True)
        rc, _, term = orc.step(a, n)
        assert rc == 0
        K += 1
    return K


def test_last_decision_terminates_the_episode(bank):
    """K = the oracle's decision count of env 0's first episode: the rollout ends on the terminal observation, whose
    reward (owed until the loop ends) is not zero; auto-reset is on but never runs."""
    K = first_episode_length(bank, C2_LIKE, SEEDS[0], "fair")
    got = check_matches_eager(bank, C2_LIKE, SEEDS, K, "fair", False)
    h = got.hdr()[0]
    assert h["terminated"] == 1 and h["reward"] != 0.0


@pytest.mark.parametrize("traj", [False, True])
@pytest.mark.parametrize("E", [10, 50])
def test_random_last_decision_terminates_the_episode(bank, E, traj):
    """As above for the random policy, on the one-slot and the two-slot kernel, without and with a buffer."""
    cfg = {**C2_LIKE, "num_executors": E, "job_arrival_cap": 8}
    K = first_episode_length(bank, cfg, SEEDS[0], "random")
    got = check_matches_eager(bank, cfg, SEEDS, K, "random", traj)
    h = got.hdr()[0]
    assert h["terminated"] == 1 and h["reward"] != 0.0


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
