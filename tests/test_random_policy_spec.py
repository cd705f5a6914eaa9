"""The random scheduler's draw specification (tests/random_policy_spec.py, the RANDOM stream) against the host
schedulers' vectorised find_stage (`job_choices`, pinned to the reference's own preprocess_obs by
tests/test_host_schedulers.py) and against the reference's procedure (the host RandomScheduler: rejection loop over the
jobs on numpy's RandomState).  No GPU needed."""
import numpy as np
import pytest
from scipy.stats import chi2_contingency

from helpers import bank_for, load_golden
from oracle import OracleEnv
from philox_ref import bounded, philox4x32_10
from random_policy_spec import STREAM_RANDOM, random_policy_action
from spark_sched_sim_b200.gym_compat import GraphInstance
from spark_sched_sim_b200.schedulers import RandomScheduler
from spark_sched_sim_b200.schedulers.heuristics import job_choices

# random and fair traces, with 64-bit stage masks (wide_*) and with 3 executors (e3_j5_*)
TRACES = ["e10_j8_random_s5_philox", "e3_j5_random_s12_philox", "wide_e50_j5_random_s32_philox",
          "wide_e10_j6_fair_s31_philox", "e50_j8_fair_s7_philox", "e10_tl_random_s11_philox"]


def replay(name):
    """Every observation of the trace (recorded actions replayed on the oracle from the recorded tape)."""
    tr = load_golden(name)
    env = OracleEnv(bank_for(tr), tr["num_executors"], tr["job_arrival_cap"], tr["moving_delay"],
                    tr["warmup_delay"], tr["job_arrival_rate"], tr["beta"])
    obs = env.reset_trace(tr["job_t_arrival"], tr["job_template"], tr["tape"])
    for a, n in tr["actions"]:
        yield env, obs
        rc, _, _ = env.step(int(a), int(n))
        assert rc == 0
        obs = env.obs()


def eligible_count(obs):
    return sum(1 for j in range(len(obs["dag_ptr"]) - 1)
               if obs["nodes"][obs["dag_ptr"][j]:obs["dag_ptr"][j + 1], 2].any())


@pytest.mark.parametrize("name", TRACES)
def test_spec_matches_find_stage_of_the_host_schedulers(name):
    """On every observation of the trace, several (seed, draw) pairs: the spec's action is the bounded(w0, k)-th of
    the jobs whose find_stage (job_choices) gives a stage, and num_exec = 1 + bounded(w1, num_committable_execs)."""
    for k, (_, obs) in enumerate(replay(name)):
        picks = [int(c) for c in job_choices(host_obs(obs)) if c >= 0]
        assert len(picks) == eligible_count(obs) > 0, k
        ncommit = obs["num_committable_execs"]
        for seed, d in ((0, 0), (7, k), (2**40 + 123, 3 * k + 1), (2**64 - 1, 2**32 - 1 - k)):
            w = philox4x32_10((d, 0, STREAM_RANDOM, 0), (seed & 0xFFFFFFFF, seed >> 32))
            want = (picks[bounded(w[0], len(picks))], 1 + bounded(w[1], ncommit))
            got = random_policy_action(obs, seed, d)
            assert got == want, (k, seed, d)
            assert 1 <= got[1] <= ncommit, (k, got)


def host_obs(obs):
    return {"dag_batch": GraphInstance(obs["nodes"], np.zeros(len(obs["edge_links"]), int),
                                       obs["edge_links"].astype(np.int64)),
            "dag_ptr": obs["dag_ptr"].tolist(), "num_committable_execs": obs["num_committable_execs"],
            "source_job_idx": obs["source_job_idx"], "exec_supplies": obs["exec_supplies"].tolist()}


def test_spec_law_equals_reference_procedure():
    """20 000 draws of the spec and 20 000 of the reference's rejection loop on RandomState, on observations with 1,
    2 and more eligible jobs (some with active jobs that are not eligible): the same distribution of (stage_idx,
    num_exec) by a chi-square two-sample test.  The draws are seeded, so the outcome is fixed; the threshold
    p > 1e-3 is what two samples of one law pass with probability 0.999."""
    picked = {}
    for name in ("e10_j8_random_s5_philox", "wide_e50_j5_random_s32_philox"):
        for _, obs in replay(name):
            k, ja = eligible_count(obs), len(obs["exec_supplies"])
            key = (min(k, 3), ja > k)
            if key not in picked and obs["num_committable_execs"] > 1:
                picked[key] = {x: (v.copy() if isinstance(v, np.ndarray) else v) for x, v in obs.items()}
    assert {(1, True), (2, True), (3, True), (3, False)} <= set(picked), sorted(picked)
    n_draws = 20000
    for key, obs in sorted(picked.items()):
        spec = [random_policy_action(obs, 99, d) for d in range(n_draws)]
        sched = RandomScheduler(seed=5)
        ref = []
        for _ in range(n_draws):
            a, _ = sched.schedule(host_obs(obs))
            ref.append((a["stage_idx"], a["num_exec"]))
        cells = sorted(set(spec) | set(ref))
        assert set(spec) == set(ref), key
        table = np.array([[spec.count(c) for c in cells], [ref.count(c) for c in cells]])
        p = chi2_contingency(table)[1]
        assert p > 1e-3, (key, p, len(cells))


def test_no_eligible_job():
    """An observation without a schedulable node: stage_idx -1, num_exec still uniform on [1, num_committable]."""
    _, obs = next(replay("e10_j8_random_s5_philox"))
    obs = dict(obs, nodes=obs["nodes"].copy(), num_committable_execs=4)
    obs["nodes"][:, 2] = 0
    seen = set()
    for d in range(400):
        a, n = random_policy_action(obs, 3, d)
        assert a == -1 and 1 <= n <= 4
        seen.add(n)
    assert seen == {1, 2, 3, 4}
