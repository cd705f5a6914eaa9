"""Shared test helpers: golden fixtures and the trace comparer used for BOTH the CPU oracle
(pinning it to the reference) and the CUDA path (comparing it with the oracle / the fixtures)."""
from __future__ import annotations

import glob
import os.path as osp

import numpy as np

GOLDEN_DIR = osp.join(osp.dirname(osp.abspath(__file__)), "golden")


def golden_names(slim=None):
    names = sorted(osp.basename(p)[:-4] for p in glob.glob(osp.join(GOLDEN_DIR, "*.npz")))
    # fixtures that are not traces
    names = [n for n in names if n not in ("decima_model", "learner_vectors", "scheduler_vectors")
             and not n.startswith("decima_grads_")]
    if slim is None:
        return names
    return [n for n in names if n.startswith(("c2_", "c4_", "decima_c2_", "decima_c3_")) == slim]


def load_golden(name):
    z = np.load(osp.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    tr = {k: z[k] for k in z.files}
    for k in ("num_executors", "job_arrival_cap", "seed", "policy_seed"):
        tr[k] = int(tr[k])
    for k in ("moving_delay", "warmup_delay", "job_arrival_rate", "beta", "time_limit", "final_wall"):
        tr[k] = float(tr[k])
    for k in ("rng", "policy", "bank_checksum"):
        tr[k] = str(tr[k])
    tr["slim"] = "slim" in tr
    tr["bank_kind"] = str(tr["bank_kind"]) if "bank_kind" in tr else "appd"
    tr["bank_seed"] = int(tr["bank_seed"]) if "bank_seed" in tr else 0
    return tr


def bank_for(tr):
    """The template bank the trace was recorded on (App. D workload unless the trace says otherwise)."""
    import spark_sched_sim_b200.bank as bankmod

    b = bankmod.synthetic_bank(tr["bank_seed"], tr["bank_kind"])
    assert b.checksum() == tr["bank_checksum"], "bank differs from the one the fixture was recorded on"
    return b


def decima_digest(feat, caps, depth, edge_bits, stage_mask):
    import hashlib

    h = hashlib.sha256()
    h.update(np.ascontiguousarray(feat, dtype=np.float32).tobytes())
    h.update(np.asarray(caps, dtype=np.int32).tobytes())
    h.update(np.asarray([depth], dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(edge_bits, dtype=np.uint64).tobytes())
    h.update(np.ascontiguousarray(stage_mask, dtype=np.uint8).tobytes())
    return int.from_bytes(h.digest()[:8], "little")


def obs_digest(o):
    import hashlib

    h = hashlib.sha256()
    h.update(np.ascontiguousarray(o["nodes"], dtype=np.float32).tobytes())
    h.update(np.ascontiguousarray(o["edge_links"], dtype=np.int32).tobytes())
    h.update(np.asarray(o["dag_ptr"], dtype=np.int32).tobytes())
    h.update(np.asarray(o["exec_supplies"], dtype=np.int32).tobytes())
    h.update(np.asarray([o["num_committable_execs"], o["source_job_idx"]], dtype=np.int32).tobytes())
    return int.from_bytes(h.digest()[:8], "little")


EV_KEYS = ("ev_t", "ev_type", "ev_job", "ev_stage", "ev_task", "ev_exec", "ev_tacc")


def events_digest(ev, lo, hi):
    import hashlib

    h = hashlib.sha256()
    for k in EV_KEYS:
        h.update(np.ascontiguousarray(ev[k][lo:hi]).tobytes())
    return int.from_bytes(h.digest()[:8], "little")


def replay_and_compare(env, tr, mode, check_policy=None, reward_rtol=0.0):
    """Drives `env` (OracleEnv-like: reset_trace/reset_seed/step/obs/log/job_times/wall_time) with
    the recorded actions and compares everything with the reference trace `tr`.
    mode: "tape" (recorded job sequence + duration tape) or "seed" (Philox streams from the seed)."""
    if mode == "tape":
        obs = env.reset_trace(tr["job_t_arrival"], tr["job_template"], tr["tape"])
    else:
        assert tr["rng"] == "philox"
        obs = env.reset_seed(tr["seed"], tr["time_limit"])
        ta, _, tm = env.job_times()
        assert np.array_equal(ta, tr["job_t_arrival"])
        assert np.array_equal(tm, tr["job_template"])
    off = dict(n=0, e=0, d=0, s=0)

    def chk(o, k):
        N, M, Ja = int(tr["N"][k]), int(tr["M"][k]), int(tr["Ja"][k])
        assert o["nodes"].shape[0] == N and o["edge_links"].shape[0] == M, (k, "sizes")
        assert len(o["exec_supplies"]) == Ja
        assert o["num_committable_execs"] == tr["ncommit"][k], (k, "ncommit")
        assert o["source_job_idx"] == tr["src"][k], (k, "src")
        if tr["slim"]:
            assert obs_digest(o) == int(tr["obs_digest"][k]), (k, "obs digest")
        else:
            assert np.array_equal(o["nodes"], tr["nodes"][off["n"]:off["n"] + N]), (k, "nodes")
            assert np.array_equal(o["edge_links"], tr["edges"][off["e"]:off["e"] + M]), (k, "edges")
            assert np.array_equal(o["dag_ptr"], tr["dag_ptr"][off["d"]:off["d"] + Ja + 1]), (k, "dag_ptr")
            assert np.array_equal(o["exec_supplies"], tr["supplies"][off["s"]:off["s"] + Ja]), (k, "sup")
            off["n"] += N; off["e"] += M; off["d"] += Ja + 1; off["s"] += Ja

    chk(obs, 0)
    for k, (a, n) in enumerate(tr["actions"]):
        if check_policy is not None and tr["policy"] in ("fair", "fifo"):
            assert check_policy(tr["policy"] == "fair") == (a, n), (k, "policy")
        rc, r, term = env.step(int(a), int(n))
        assert rc == 0, (k, rc)
        ref_r = float(tr["reward"][k])
        if reward_rtol == 0.0:
            assert r == ref_r, (k, r, ref_r)
        else:
            assert abs(r - ref_r) <= reward_rtol * max(abs(ref_r), 1e-300), (k, r, ref_r)
        assert env.wall_time == tr["wall"][k], (k, "wall_time")
        assert term == bool(tr["term"][k]), (k, "terminated")
        assert env.log_size() == tr["ev_count"][k + 1], (k, "event count")
        chk(env.obs(), k + 1)
    lg = env.log()
    if tr["slim"]:
        ec = tr["ev_count"]
        lo = np.concatenate([[0], ec[:-1]])
        for k, (a, b) in enumerate(zip(lo, ec)):
            assert events_digest(lg, int(a), int(b)) == int(tr["ev_digest"][k]), (k, "event digest")
    else:
        for key in EV_KEYS:
            assert np.array_equal(lg[key], tr[key]), key
    _, tc, _ = env.job_times()
    assert np.array_equal(tc, tr["job_t_completed"]), "job completion times"
    if "hist_ptr" in tr and hasattr(env, "history"):
        # executor.history (executor.py:25-44): per executor, the add_history calls in order
        hs = env.history()
        for e in range(tr["num_executors"]):
            lo, hi = int(tr["hist_ptr"][e]), int(tr["hist_ptr"][e + 1])
            sel = hs["hist_exec"] == e
            assert np.array_equal(hs["hist_t"][sel], tr["hist_t"][lo:hi]), (e, "history times")
            assert np.array_equal(hs["hist_job"][sel], tr["hist_job"][lo:hi]), (e, "history jobs")
        assert len(hs["hist_t"]) == int(tr["hist_ptr"][-1]), "history length"
