"""The random scheduler's draw specification (pure Python) -- TEST INFRASTRUCTURE ONLY.

`ssb_random_actions` / `ssb_rollout_random` (csrc/ssb_random.cu) take the reference's `RandomScheduler.schedule`
(schedulers/heuristics/random_scheduler.py:7-32) in law on a Philox stream of their own, in the notation of
oracle/philox_ref.py:

    RANDOM stream  ctr = (policy_draws, 0, 5, 0), key = episode seed
                   w0 -> job:      the bounded(w0, k)-th eligible job in active-job order (k = number of eligible jobs)
                   w1 -> num_exec: 1 + bounded(w1, num_committable_execs)

    policy_draws = decisions the policy has taken so far in the episode (zeroed by reset).  The Decima policy's
    sampling stream (word 2 = 4) counts with the same counter; the streams differ in word 2.

`random_policy_action` restates it on an observation with plain loops, as tests/golden/gen_scheduler_golden.py
restates `preprocess_obs`; the tests drive the CPU oracle (oracle/) with it and compare the device with that loop."""
from __future__ import annotations

from philox_ref import MASK, bounded, philox4x32_10

STREAM_RANDOM = 5


def random_policy_action(obs, seed: int, draw_idx: int) -> tuple[int, int]:
    """RandomScheduler.schedule in law on the RANDOM stream.

    The reference redraws a job uniformly from the jobs still "running" until find_stage (heuristics/utils.py:17-37)
    gives a stage: in law one uniform draw over the "eligible" jobs, those with a schedulable node.  stage_idx is the
    drawn job's find_stage choice -- the rank among the schedulable nodes of its first schedulable node without an
    incoming edge, else of its first schedulable node -- or -1 when no job is eligible; num_exec is uniform on
    [1, num_committable_execs].  `obs`: nodes [N][3], edge_links [M][2], dag_ptr, num_committable_execs;
    draw_idx: the decision's index within the episode."""
    nodes, edges, ptr = obs["nodes"], obs["edge_links"], obs["dag_ptr"]
    n = len(nodes)
    has_parent = [False] * n
    for e in range(len(edges)):
        has_parent[int(edges[e][1])] = True
    rank, r = [-1] * n, 0
    for v in range(n):
        if nodes[v][2] != 0:
            rank[v] = r
            r += 1
    choices = []  # find_stage of every eligible job, in active-job order
    for j in range(len(ptr) - 1):
        sel = -1
        for v in range(int(ptr[j]), int(ptr[j + 1])):
            if rank[v] < 0:
                continue
            if not has_parent[v]:
                sel = rank[v]
                break
            if sel == -1:
                sel = rank[v]
        if sel != -1:
            choices.append(sel)
    seed = int(seed)
    w = philox4x32_10((int(draw_idx) & MASK, 0, STREAM_RANDOM, 0), (seed & MASK, (seed >> 32) & MASK))
    stage_idx = choices[bounded(w[0], len(choices))] if choices else -1
    return stage_idx, 1 + bounded(w[1], int(obs["num_committable_execs"]))
