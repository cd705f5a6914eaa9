"""Generates tests/golden/scheduler_vectors.npz: for every recorded observation of the heuristic-policy golden traces
that test_host_schedulers.py replays, what the reference's schedulers (RoundRobinScheduler fair / FIFO,
RandomScheduler) return and leave in the observation dict -- the action, `frontier_stages` and `schedulable_stages`.

* the action is the one the reference recorded in the trace (tests/golden/gen_golden.py);
* `frontier_stages` / `schedulable_stages` are what the reference's `preprocess_obs` (schedulers/heuristics/utils.py:5-15)
  makes of the recorded observation, restated below with plain loops (independent of this package's vectorised code):
  the nodes that are no edge's destination, and schedulable node id -> its rank among the schedulable nodes.

With a checkout of the original project in $SSB_REFERENCE the UNMODIFIED reference schedulers are also run on every
observation (through oracle/refrun.py) and must return and leave exactly the same before anything is written.

    [SSB_REFERENCE=<checkout of spark-sched-sim>] python tests/golden/gen_scheduler_golden.py [out.npz]
"""
import copy
import os.path as osp
import sys

import numpy as np

HERE = osp.dirname(osp.abspath(__file__))
REPO = osp.dirname(osp.dirname(HERE))
for p in (REPO, osp.join(REPO, "oracle"), osp.dirname(HERE)):
    if p not in sys.path:
        sys.path.insert(0, p)

import refrun  # noqa: E402
from helpers import load_golden  # noqa: E402
from test_host_schedulers import SCHEDULER_TRACES, recorded_obs  # noqa: E402


def reference_preprocess(obs):
    """(frontier node ids, [(schedulable node id, stage_idx)]) of one base observation."""
    nodes, edges = obs["dag_batch"].nodes, obs["dag_batch"].edge_links
    is_dst = [False] * len(nodes)
    for _, dst in edges:
        is_dst[int(dst)] = True
    frontier = [i for i in range(len(nodes)) if not is_dst[i]]
    sched = [i for i in range(len(nodes)) if nodes[i][2]]
    return frontier, [(node, rank) for rank, node in enumerate(sched)]


def main():
    live = refrun.reference_available()
    if live:
        refrun.setup()
    out = {}
    for name in SCHEDULER_TRACES:
        tr = load_golden(name)
        ref = refrun.make_policy(tr["policy"], tr["num_executors"], tr["policy_seed"]) if live else None
        fr, fr_len, sn, si, s_len = [], [], [], [], []
        for k, obs in enumerate(recorded_obs(tr)):
            if k == len(tr["actions"]):
                break
            f, s = reference_preprocess(obs)
            if ref is not None:
                o = copy.deepcopy(obs)
                a, info = ref.schedule(o)
                assert (int(a["stage_idx"]), int(a["num_exec"])) == tuple(tr["actions"][k]) and info == {}, (name, k)
                assert sorted(int(x) for x in o["frontier_stages"]) == f, (name, k)
                assert sorted((int(n), int(i)) for n, i in o["schedulable_stages"].items()) == s, (name, k)
            fr += f
            fr_len.append(len(f))
            sn += [n for n, _ in s]
            si += [i for _, i in s]
            s_len.append(len(s))
        out[f"{name}_action"] = np.asarray(tr["actions"], np.int32).reshape(-1, 2)
        out[f"{name}_frontier"] = np.array(fr, np.int32)
        out[f"{name}_frontier_len"] = np.array(fr_len, np.int32)
        out[f"{name}_sched_node"] = np.array(sn, np.int32)
        out[f"{name}_sched_idx"] = np.array(si, np.int32)
        out[f"{name}_sched_len"] = np.array(s_len, np.int32)
    path = sys.argv[1] if len(sys.argv) > 1 else osp.join(HERE, "scheduler_vectors.npz")
    np.savez_compressed(path, **out)
    print(path, "checked against the reference schedulers" if live else "from the recorded traces",
          {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
