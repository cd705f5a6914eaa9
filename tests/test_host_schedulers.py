"""Host-side scheduler plug-ins (same interface as schedulers/heuristics in the reference) against
the observations and actions recorded from the reference run (no GPU needed)."""
import os.path as osp

import numpy as np
import pytest

from helpers import golden_names, load_golden
from spark_sched_sim_b200.gym_compat import GraphInstance
from spark_sched_sim_b200.schedulers import RandomScheduler, RoundRobinScheduler, make_scheduler


def recorded_obs(tr):
    n = e = d = s = 0
    for k in range(len(tr["N"])):
        N, M, Ja = int(tr["N"][k]), int(tr["M"][k]), int(tr["Ja"][k])
        yield {
            "dag_batch": GraphInstance(tr["nodes"][n:n + N], np.zeros(M, int),
                                       tr["edges"][e:e + M].astype(np.int64)),
            "dag_ptr": tr["dag_ptr"][d:d + Ja + 1].tolist(),
            "num_committable_execs": int(tr["ncommit"][k]),
            "source_job_idx": int(tr["src"][k]),
            "exec_supplies": tr["supplies"][s:s + Ja].tolist(),
        }
        n += N; e += M; d += Ja + 1; s += Ja


@pytest.mark.parametrize("name", [n for n in golden_names(slim=False) if not n.startswith("decima_")])
def test_host_policies_reproduce_recorded_actions(name):
    tr = load_golden(name)
    if tr["policy"] in ("fair", "fifo"):
        sched = RoundRobinScheduler(tr["num_executors"], dynamic_partition=(tr["policy"] == "fair"))
    else:
        sched = RandomScheduler(seed=tr["policy_seed"])
    assert sched.env_wrapper_cls is None and sched.name in ("Fair", "FIFO", "Random")
    for k, obs in enumerate(recorded_obs(tr)):
        if k == len(tr["actions"]):
            break
        action, info = sched.schedule(obs)
        assert (int(action["stage_idx"]), int(action["num_exec"])) == tuple(tr["actions"][k]), k
        assert info == {}


SCHEDULER_TRACES = [n for n in golden_names(slim=False) if not n.startswith("decima_")][:8]


@pytest.mark.parametrize("name", SCHEDULER_TRACES)
def test_reference_schedulers_agree_on_the_same_observations(name):
    """The UNMODIFIED reference schedulers, run on every recorded observation of the trace (what they returned and
    left in the observation dict, stored by tests/golden/gen_scheduler_golden.py), and this package's classes on the
    same observations: same action, empty info, and the same `frontier_stages` and `schedulable_stages`.  Together
    with the GPU facade test (the facade's observations equal the recorded ones bit for bit) this is "the reference's
    schedulers run on the facade unchanged"."""
    from helpers import GOLDEN_DIR

    tr = load_golden(name)
    z = np.load(osp.join(GOLDEN_DIR, "scheduler_vectors.npz"))
    act, fr, fr_len = z[f"{name}_action"], z[f"{name}_frontier"], z[f"{name}_frontier_len"]
    sn, si, s_len = z[f"{name}_sched_node"], z[f"{name}_sched_idx"], z[f"{name}_sched_len"]
    assert len(act) == len(tr["actions"]) > 0
    if tr["policy"] in ("fair", "fifo"):
        ours = RoundRobinScheduler(tr["num_executors"], dynamic_partition=(tr["policy"] == "fair"))
    else:
        ours = RandomScheduler(seed=tr["policy_seed"])
    f0 = s0 = 0
    for k, obs in enumerate(recorded_obs(tr)):
        if k == len(act):
            break
        a, info = ours.schedule(obs)
        assert (int(a["stage_idx"]), int(a["num_exec"])) == tuple(act[k]) and info == {}, k
        f1, s1 = f0 + int(fr_len[k]), s0 + int(s_len[k])
        assert sorted(obs["frontier_stages"]) == fr[f0:f1].tolist(), (k, "frontier_stages")
        assert sorted(obs["schedulable_stages"].items()) == list(zip(sn[s0:s1].tolist(), si[s0:s1].tolist())), \
            (k, "schedulable_stages")
        f0, s0 = f1, s1
    assert (f0, s0) == (len(fr), len(sn))


def test_make_scheduler_factory():
    s = make_scheduler({"agent_cls": "RoundRobinScheduler", "num_executors": 10, "dynamic_partition": False})
    assert s.name == "FIFO"
    with pytest.raises(AssertionError):
        make_scheduler({"agent_cls": "Nope"})


def test_decima_scheduler_constructor_contract():
    """schedulers.DecimaScheduler keeps the reference's constructor keywords (schedulers/decima/scheduler.py:22-69)
    and refuses what the device policy does not implement -- no GPU needed for that."""
    import os.path as osp

    from helpers import GOLDEN_DIR
    from spark_sched_sim_b200.decima import DecimaEnvWrapper
    from spark_sched_sim_b200.schedulers import DecimaScheduler, make_scheduler

    agent_cfg = {"agent_cls": "DecimaScheduler", "embed_dim": 16, "gnn_mlp_kwargs": {"hid_dims": [32, 16], "act_cls": "LeakyReLU"},
                 "policy_mlp_kwargs": {"hid_dims": [64, 64], "act_cls": "Tanh"}, "num_executors": 10,
                 "state_dict_path": osp.join(GOLDEN_DIR, "decima_model.npz"), "training_mode": False}
    s = make_scheduler(agent_cfg)
    assert isinstance(s, DecimaScheduler) and s.env_wrapper_cls is DecimaEnvWrapper and s.name.startswith("Decima:")
    assert len(s._state_dict) == 42 and sum(v.size for v in s._state_dict.values()) == 20802
    with pytest.raises(ValueError):
        DecimaScheduler(10, embed_dim=32, state_dict_path=agent_cfg["state_dict_path"])
    with pytest.raises(ValueError):
        DecimaScheduler(10)  # no weights
    with pytest.raises(ValueError):
        s.schedule({"dag_ptr": [0]})  # not an observation of DecimaEnvWrapper


def test_stats_from_sums():
    from spark_sched_sim_b200 import parallel

    d = parallel.stats_from_sums([50.0, 2.0, 30.0, 44.0, 600000.0, 9.0, 0.0, 0.0])
    assert d == {"avg_num_jobs": 25.0, "num_completed_jobs": 15.0, "num_job_arrivals": 22.0, "avg_job_duration": 20.0}
