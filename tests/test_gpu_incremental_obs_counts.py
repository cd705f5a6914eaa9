"""The observation header that the fused rollout writes at every decision takes num_nodes / num_edges from the counts
the simulator keeps as jobs arrive, stages complete and jobs complete (EnvHdr.n_obs_nodes / n_obs_edges), not from a
pass over the graph.  These tests drive ssb_rollout_fair one decision per launch through whole episodes with
auto-reset and require, after every launch, the header to agree with the graph slabs the launch wrote when its loop
ended (nodes: dag_ptr[num_active_jobs]; edges: the edge rows written) and to equal, byte for byte, the header and
graph of a twin env stepped through ssb_step, whose observation counts the graph it builds.  The recorded-trace path
(jobs and task durations from a trace; ssb_step and the fused rollout taking the decisions in turn) is checked
against the counts the reference recorded."""
import numpy as np
import pytest

from helpers import bank_for, load_golden

pytestmark = pytest.mark.gpu

B = 8


def _cfg(E, cap):
    return {"num_executors": E, "job_arrival_cap": cap, "job_arrival_rate": 4.0e-5,
            "moving_delay": 2000.0, "warmup_delay": 1000.0}


def graph_counts(env, hdr):
    """(nodes, edges) per env implied by the graph slabs: dag_ptr[num_active_jobs], and the rows of the edge slab
    written since it was filled with -1 (they must form a prefix)"""
    dag = env.dag_ptr.cpu().numpy()
    written = (env.edge_links[:, :, 0] >= 0).cpu().numpy()
    n = dag[np.arange(len(hdr)), hdr["num_active_jobs"]]
    m = written.sum(1)
    for b in range(len(hdr)):
        assert written[b, :m[b]].all(), b
    return n, m


def eager_decision(env):
    """One fair decision per env through ssb_step; an env the call only re-seeds (was_reset) is stepped again, as the
    fused rollout re-seeds and decides in the same launch."""
    import torch

    a, n = env.fair_actions(True)
    env.step(a, n)
    r = env.hdr()["was_reset"].astype(np.uint8)
    if r.any():
        a, n = env.fair_actions(True)
        env.step(a, n, mask=torch.as_tensor(r))


@pytest.mark.parametrize("kind", ["appd", "wide"])
@pytest.mark.parametrize("E", [3, 10, 50])
def test_counts_match_graph_every_decision(E, kind):
    import spark_sched_sim_b200.bank as bankmod
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    bank = bankmod.synthetic_bank(0, kind)
    cfg = _cfg(E, 6 if kind == "appd" else 4)
    seeds = (40 + 7 * E + np.arange(B)).astype(np.uint64)
    fused = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank)
    eager = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank)
    assert (fused.reset_host(seeds)["error"] == 0).all() and (eager.reset_host(seeds)["error"] == 0).all()
    eager.set_autoreset(True, 1)
    episodes = np.zeros(B, np.int64)
    launches = 0
    while episodes.min() < 2:  # every env through a whole episode after an in-kernel reset
        assert launches < 5000
        fused.edge_links.fill_(-1)
        fused.rollout_fair(1, True, True, 1)
        eager_decision(eager)
        h, he = fused.hdr(), eager.hdr()
        assert (h["error"] == 0).all(), h["error"]
        n, m = graph_counts(fused, h)
        assert np.array_equal(h["num_nodes"], n), (launches, h["num_nodes"], n)
        assert np.array_equal(h["num_edges"], m), (launches, h["num_edges"], m)
        assert h.tobytes() == he.tobytes(), (launches, [f for f in h.dtype.names if not np.array_equal(h[f], he[f])])
        for b in range(B):
            o, oe = fused.obs(b, h), eager.obs(b, he)
            for k in ("nodes", "edge_links", "dag_ptr", "exec_supplies"):
                assert o[k].tobytes() == oe[k].tobytes(), (launches, b, k)
        episodes += h["terminated"]
        launches += 1
    assert fused.stats_per_env().tobytes() == eager.stats_per_env().tobytes()


@pytest.mark.parametrize("name", ["e10_j8_fair_s2_philox", "wide_e10_j6_fair_s31_philox"])
def test_counts_on_a_recorded_trace(name):
    """Jobs and task durations from a recorded trace (k_reset), the recorded fair decisions taken alternately by
    ssb_step and by one-decision fused launches: every header carries the reference's node, edge and job counts."""
    import torch
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    tr = load_golden(name)
    assert tr["policy"] == "fair" and tr["job_arrival_cap"] > 0
    cfg = {"num_executors": tr["num_executors"], "job_arrival_cap": tr["job_arrival_cap"],
           "job_arrival_rate": tr["job_arrival_rate"], "moving_delay": tr["moving_delay"],
           "warmup_delay": tr["warmup_delay"], "beta": tr["beta"]}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=2, bank=bank_for(tr), max_jobs=len(tr["job_template"]) + 2,
                                  tape_capacity=len(tr["tape"]) + 8)
    for b in range(2):
        env.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    h = env.reset_host(np.full(2, tr["seed"], np.uint64)).copy()
    K = len(tr["actions"])
    for k in range(K + 1):
        want = (tr["N"][k], tr["M"][k], tr["Ja"][k])
        for b in range(2):
            assert (h["num_nodes"][b], h["num_edges"][b], h["num_active_jobs"][b]) == want, (k, b)
        if k == K:
            break
        if k % 2 == 0:
            a, n = env.fair_actions(True)
            assert a.tolist() == [tr["actions"][k][0]] * 2 and n.tolist() == [tr["actions"][k][1]] * 2, k
            env.step(a, n)
        else:
            env.rollout_fair(1, True, False, 1)
        h = env.hdr()
        assert (h["error"] == 0).all(), (k, h["error"])
    assert (h["terminated"] == 1).all()
