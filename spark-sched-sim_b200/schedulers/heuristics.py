"""Host-side heuristic policies on the base observation dict -- the plug-ins `examples.py --sched fair|fifo|random`
constructs (schedulers/heuristics/round_robin.py:7-49, random_scheduler.py:7-32, utils.py:5-37).  The on-device
equivalent of the fair / FIFO policy is `ssb_rollout_fair` / `ssb_fair_actions`; these classes are the host
compatibility layer for callers that drive the gym facade step by step.

The reference walks the jobs and their nodes in Python loops.  Here one vectorised pass (`job_choices`) answers
"which `stage_idx` would this job get" for every active job at once -- segment minima over the observation's node
arrays -- and the policies are a few array expressions on top of it.  `tests/test_host_schedulers.py` pins the
classes to the actions the reference recorded and to what the reference's classes return and leave in the
observation dict on the same observations (tests/golden/scheduler_vectors.npz)."""
from __future__ import annotations

import numpy as np

from .scheduler import Scheduler

_NONE = np.iinfo(np.int64).max


def job_choices(obs: dict) -> np.ndarray:
    """int64[Ja]: per active job the action index (`stage_idx`, the rank among the schedulable nodes) of the node
    `find_stage` (utils.py:18-37) picks -- its first schedulable node without an incoming edge in the observed graph,
    else its first schedulable node, else -1."""
    g = obs["dag_batch"]
    n = g.nodes.shape[0]
    ptr = np.asarray(obs["dag_ptr"], dtype=np.int64)
    ja = len(ptr) - 1
    if ja <= 0 or n == 0:
        return np.full(max(ja, 0), -1, np.int64)
    sched = g.nodes[:, 2] != 0
    has_parent = np.zeros(n, bool)
    has_parent[g.edge_links[:, 1]] = True
    idx = np.arange(n, dtype=np.int64)
    # candidate node per job: segment minimum of the node index over (schedulable & frontier), then over schedulable;
    # a sentinel row keeps reduceat's "empty segment" rule (it returns the element AT the offset) harmless
    def seg_min(mask):
        key = np.append(np.where(mask, idx, _NONE), _NONE)
        m = np.minimum.reduceat(key, np.minimum(ptr[:-1], n))
        return np.where(ptr[1:] > ptr[:-1], m, _NONE)
    first_frontier, first_any = seg_min(sched & ~has_parent), seg_min(sched)
    node = np.where(first_frontier != _NONE, first_frontier, first_any)
    rank = np.cumsum(sched) - 1  # node id -> rank among the schedulable nodes
    return np.where(node != _NONE, rank[np.minimum(node, n - 1)], -1).astype(np.int64)


def preprocess_obs(obs: dict) -> None:
    """The two keys the reference's heuristics leave in the observation dict (utils.py:5-15), for callers that read
    them: `frontier_stages` and `schedulable_stages` (node id -> `stage_idx`)."""
    g = obs["dag_batch"]
    has_parent = np.zeros(g.nodes.shape[0], bool)
    has_parent[g.edge_links[:, 1]] = True
    sched = np.flatnonzero(g.nodes[:, 2] != 0)
    obs["frontier_stages"] = set(np.flatnonzero(~has_parent).tolist())
    obs["schedulable_stages"] = dict(zip(sched.tolist(), range(len(sched))))


def find_stage(obs: dict, job_idx: int) -> int:
    return int(job_choices(obs)[job_idx])


class RoundRobinScheduler(Scheduler):
    """Fair (dynamic_partition: every active job may hold ceil(E / #jobs) executors) or FIFO (every job may hold
    all of them) round robin over the jobs in arrival order; the job that is releasing executors goes first."""

    def __init__(self, num_executors, dynamic_partition=True, **kwargs):
        self.name = "Fair" if dynamic_partition else "FIFO"
        self.num_executors = num_executors
        self.dynamic_partition = dynamic_partition
        self.env_wrapper_cls = None

    def schedule(self, obs: dict) -> tuple[dict, dict]:
        preprocess_obs(obs)
        supplies = np.asarray(obs["exec_supplies"], dtype=np.int64)
        ja, free, src = len(supplies), obs["num_committable_execs"], obs["source_job_idx"]
        share = -(-self.num_executors // max(1, ja)) if self.dynamic_partition else self.num_executors
        pick = job_choices(obs)
        if src < ja and pick[src] >= 0:
            return {"stage_idx": int(pick[src]), "num_exec": free}, {}
        ok = (pick >= 0) & (supplies < share)
        if src < ja:
            ok[src] = False
        if not ok.any():
            return {"stage_idx": -1, "num_exec": free}, {}
        j = int(np.argmax(ok))
        return {"stage_idx": int(pick[j]), "num_exec": min(free, int(share - supplies[j]))}, {}


class RandomScheduler(Scheduler):
    """A uniformly drawn job that has something to schedule, a uniformly drawn executor count.  The draws follow the
    reference's `RandomState` call sequence (choice over the jobs still in the running, then randint), so a seed
    gives the same actions."""

    def __init__(self, seed=42, **kwargs):
        self.name = "Random"
        self.env_wrapper_cls = None
        self.set_seed(seed)

    def set_seed(self, seed):
        self.np_random = np.random.RandomState(seed)

    def schedule(self, obs: dict) -> tuple[dict, dict]:
        preprocess_obs(obs)
        pick = job_choices(obs)
        running = list(range(len(pick)))
        stage_idx = -1
        while running and stage_idx == -1:
            j = self.np_random.choice(running)
            stage_idx = int(pick[j])
            if stage_idx == -1:
                running.remove(j)
        return {"stage_idx": stage_idx, "num_exec": self.np_random.randint(1, obs["num_committable_execs"] + 1)}, {}
