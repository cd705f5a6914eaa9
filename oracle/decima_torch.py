"""Batched torch restatement of DecimaScheduler.evaluate_actions -- TEST INFRASTRUCTURE ONLY.

One function over all environments of a handle at once, in any dtype and on any device, with autograd seeing the 42
weight tensors and, optionally, the node embeddings.  The inputs are the padded per-env tensors a
BatchedSparkSchedSimEnv exposes as device views (or the same layout built on the host, see `stack_observations`):

    features    f32 [B, S, 5]     dec_features          rows [0, num_nodes)
    edge_links  i32 [B, M, 2]     edge_links            rows [0, num_edges)
    edge_bits   i64 [B, M]        dec_edge_bits         bit k: the edge is masked at level k
    depth       i32 [B]           dec_depth
    dag_ptr     i32 [B, J + 1]    dag_ptr               entries [0, num_active_jobs]
    stage_mask  u8  [B, S]        dec_stage_mask
    caps        i32 [B, J]        dec_commit_caps
    action      i32 [B, 4]        pol_action            (stage, job, num_exec, number of candidates)
    num_nodes, num_edges, num_active_jobs i32 [B], live bool [B]   (from the observation headers)

Semantics follow oracle/decima_policy.py (the float32 numpy restatement pinned to the reference's scores) and
schedulers/decima/utils.py's evaluate:
  * NodeEncoder over the disjoint union of the graphs (global node id = b * S + n), levels k = max_depth - 1 .. 0 over
    all envs together, "overwrite" semantics; an env with depth 0 keeps h_init (no sink update).
  * DagEncoder = sum over each job's nodes, GlobalEncoder = sum over the active jobs.
  * stage head over the stage_mask nodes in node order, executor-count head over rows c = 0 .. cap - 1 of the chosen
    job with input c / E rounded to float32 (torch.arange(E) / E is a float32 tensor in the reference).
  * per-env softmax over the candidates, clamped to [eps, 1 - eps] with float32's eps in EVERY dtype (torch's
    clamp_probs would take float64's eps in an fp64 run: a different function from the reference's), lgprob of the
    action, entropy / log(E * num_nodes).
  * envs whose header has `terminated` or `error` set take no part (the device planner's `live` rule).
"""
from __future__ import annotations

import math

import numpy as np
import torch

EPS32 = 1.1920929e-07  # torch.finfo(torch.float32).eps

PARAM_ORDER = tuple(
    f"{net}.{layer}.{kind}"
    for net in ("encoder.node_encoder.mlp_prep", "encoder.node_encoder.mlp_msg", "encoder.node_encoder.mlp_update",
                "encoder.dag_encoder.mlp", "encoder.global_encoder.mlp", "stage_policy_network.mlp_score",
                "exec_policy_network.mlp_score")
    for layer in (0, 2, 4) for kind in ("weight", "bias"))

def weights(state_dict, dtype=torch.float64, device="cpu", requires_grad=True):
    """The 42 tensors of a DecimaScheduler state dict (numpy arrays or tensors) as leaves of the given dtype."""
    out = {}
    for k in PARAM_ORDER:
        v = state_dict[k]
        t = torch.as_tensor(np.asarray(v.detach().cpu() if hasattr(v, "detach") else v, dtype=np.float32))
        out[k] = t.to(device=device, dtype=dtype).requires_grad_(requires_grad)
    return out


def handle_observation(env, hdr=None):
    """What the policy reads of every env of a BatchedSparkSchedSimEnv: the live observation or the snapshot loaded in
    its place, and the actions of its last decima_policy / decima_evaluate call (device tensors, not copies)."""
    if hdr is None:
        hdr = env.hdr()
    dev = env.device
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int32)).to(dev)
    return {
        "features": env.dec_features, "edge_links": env.edge_links, "edge_bits": env.dec_edge_bits,
        "depth": env.dec_depth, "dag_ptr": env.dag_ptr, "stage_mask": env.dec_stage_mask,
        "caps": env.dec_commit_caps, "action": env.pol_action,
        "num_nodes": i32(hdr["num_nodes"]), "num_edges": i32(hdr["num_edges"]),
        "num_active_jobs": i32(hdr["num_active_jobs"]),
        "live": torch.from_numpy((hdr["terminated"] == 0) & (hdr["error"] == 0)).to(dev),
    }


def stack_observations(obs_list, actions):
    """Padded batch (the layout of `handle_observation`, on the host) from per-observation dicts with the keys
    features, edge_links, edge_bits, depth, dag_ptr, stage_mask, caps and actions (stage, job, num_exec, n_cand)."""
    B = len(obs_list)
    S = max(1, max(len(o["features"]) for o in obs_list))
    M = max(1, max(len(o["edge_links"]) for o in obs_list))
    J = max(1, max(len(o["dag_ptr"]) - 1 for o in obs_list))
    f = np.zeros((B, S, 5), np.float32)
    el = np.zeros((B, M, 2), np.int32)
    eb = np.zeros((B, M), np.int64)
    dp = np.zeros((B, J + 1), np.int32)
    sm = np.zeros((B, S), np.uint8)
    caps = np.zeros((B, J), np.int32)
    n_nodes, n_edges, n_jobs, depth = (np.zeros(B, np.int32) for _ in range(4))
    for b, o in enumerate(obs_list):
        N, Mb, Ja = len(o["features"]), len(o["edge_links"]), len(o["dag_ptr"]) - 1
        f[b, :N] = o["features"]
        el[b, :Mb] = np.asarray(o["edge_links"]).reshape(-1, 2)
        eb[b, :Mb] = np.asarray(o["edge_bits"], np.uint64).view(np.int64)
        dp[b, :Ja + 1] = o["dag_ptr"]
        sm[b, :N] = o["stage_mask"]
        caps[b, :Ja] = o["caps"]
        n_nodes[b], n_edges[b], n_jobs[b], depth[b] = N, Mb, Ja, o["depth"]
    t = torch.from_numpy
    return {"features": t(f), "edge_links": t(el), "edge_bits": t(eb), "depth": t(depth), "dag_ptr": t(dp),
            "stage_mask": t(sm), "caps": t(caps), "action": t(np.asarray(actions, np.int32).reshape(B, 4)),
            "num_nodes": t(n_nodes), "num_edges": t(n_edges), "num_active_jobs": t(n_jobs),
            "live": torch.ones(B, dtype=torch.bool)}


def _mlp(x, W, prefix, act):
    for i, k in enumerate((0, 2, 4)):
        x = x @ W[f"{prefix}.{k}.weight"].T + W[f"{prefix}.{k}.bias"]
        if i < 2:
            x = act(x)
    return x


def _leaky(t):
    return torch.nn.functional.leaky_relu(t, 0.2)


class _Batch:
    """Index bookkeeping of a padded batch: compact node rows (live envs' nodes, in (env, node) order), their env and
    job, the edges between them."""

    def __init__(self, obs, dev):
        g = lambda k: obs[k].to(dev)
        self.x = g("features")
        B, S = self.x.shape[:2]
        J = obs["dag_ptr"].shape[1] - 1
        self.B, self.S, self.J = B, S, J
        live = g("live").bool()
        self.live = live
        N = torch.where(live, g("num_nodes").long(), 0)
        Ja = torch.where(live, g("num_active_jobs").long(), 0)
        Me = torch.where(live, g("num_edges").long(), 0)
        self.N, self.Ja = N, Ja
        self.depth = torch.where(live, g("depth").long(), 0)
        ar_s = torch.arange(S, device=dev)
        self.node_valid = ar_s[None, :] < N[:, None]                               # [B, S]
        flat = torch.nonzero(self.node_valid.reshape(-1)).squeeze(1)              # global ids b * S + n
        self.node_g = flat
        self.node_env = flat // S
        self.node_n = flat % S
        cidx = torch.full((B * S,), -1, dtype=torch.long, device=dev)
        cidx[flat] = torch.arange(flat.numel(), device=dev)
        self.cidx = cidx
        # job of every node: last j with dag_ptr[j] <= n (entries past num_active_jobs padded with a large value)
        dp = g("dag_ptr").long()
        ar_j = torch.arange(J + 1, device=dev)
        dp = torch.where(ar_j[None, :] <= Ja[:, None], dp, torch.iinfo(torch.long).max)
        job = torch.searchsorted(dp, ar_s[None, :].expand(B, S).contiguous(), right=True) - 1
        self.node_job = job.reshape(-1)[flat]                                      # job index within its env
        self.node_jobg = self.node_env * J + self.node_job
        self.dag_ptr = dp
        jv = torch.arange(J, device=dev)[None, :] < Ja[:, None]
        self.job_g = torch.nonzero(jv.reshape(-1)).squeeze(1)
        self.job_env = self.job_g // J
        # edges of live envs
        M = obs["edge_links"].shape[1]
        ev = torch.arange(M, device=dev)[None, :] < Me[:, None]
        e_flat = torch.nonzero(ev.reshape(-1)).squeeze(1)
        e_env = e_flat // M
        links = g("edge_links").long().reshape(-1, 2)[e_flat]
        self.u = cidx[e_env * S + links[:, 0]]
        self.v = cidx[e_env * S + links[:, 1]]
        assert (self.u >= 0).all() and (self.v >= 0).all(), "edge to a node outside the observation"
        self.ebits = g("edge_bits").reshape(-1)[e_flat]
        self.e_env = e_env
        d_e = self.depth[e_env]
        above = torch.where(d_e < 63, self.ebits >> d_e.clamp(max=62), torch.zeros_like(self.ebits))
        assert not (above != 0).any(), "edge bits at or above the env's depth"
        self.stage_mask = g("stage_mask").bool() & self.node_valid
        self.caps = g("caps").long()
        self.action = g("action").long()


def encode_nodes(W, obs, device=None):
    """NodeEncoder (scheduler.py:191-241) over the whole batch -> node embeddings, padded [B, S, 16]."""
    dev = torch.device(device) if device is not None else obs["features"].device
    bt = _Batch(obs, dev)
    return _scatter_nodes(bt, _encode(W, bt))


def _scatter_nodes(bt, hc):
    out = torch.zeros(bt.B * bt.S, hc.shape[1], dtype=hc.dtype, device=hc.device)
    return out.index_put((bt.node_g,), hc).reshape(bt.B, bt.S, -1)


def _encode(W, bt):
    dt = W[PARAM_ORDER[0]].dtype
    pre = "encoder.node_encoder"
    X = bt.x.reshape(-1, 5)[bt.node_g].to(dt)
    h_init = _mlp(X, W, f"{pre}.mlp_prep", _leaky)
    n = X.shape[0]
    dev = X.device
    mp = bt.depth[bt.node_env] > 0                      # nodes of envs with message passing
    is_src = torch.zeros(n, dtype=torch.bool, device=dev)
    is_src[bt.u] = True
    sinks = torch.nonzero(mp & ~is_src).squeeze(1)
    h = torch.where(mp[:, None], torch.zeros_like(h_init), h_init)
    h = h.index_put((sinks,), _mlp(h_init[sinks], W, f"{pre}.mlp_update", _leaky))
    max_depth = int(bt.depth.max().item()) if bt.B else 0
    for k in reversed(range(max_depth)):
        m = torch.nonzero((bt.ebits >> k) & 1).squeeze(1)
        if m.numel() == 0:
            continue
        uk, vk = bt.u[m], bt.v[m]
        msg = _mlp(h[vk], W, f"{pre}.mlp_msg", _leaky)   # one row per edge: a child with two parents is sent twice
        recv = torch.unique(uk)
        agg = torch.zeros(n, 16, dtype=dt, device=dev).index_add(0, uk, msg)[recv]
        h = h.index_put((recv,), h_init[recv] + _mlp(agg, W, f"{pre}.mlp_update", _leaky))
    return h


def evaluate_actions(W, obs, coef_lgprob=None, coef_entropy=None, h=None, num_executors=None, device=None):
    """evaluate_actions on the batch `obs` (padded tensors, see the module docstring) for the actions obs["action"].

    W: the 42 tensors (see `weights`); the computation runs in their dtype on their device.  h: optional node
    embeddings [B, S, 16] to use instead of the NodeEncoder's (e.g. a leaf, to get d loss / d h).
    Returns a dict: stage_scores [B, S] and exec_scores [B, E] (-inf outside the candidates), lgprob [B], entropy [B],
    loss = sum_b c1_b lgprob_b + c2_b entropy_b (when coefficients are given), h [B, S, 16]."""
    dt = W[PARAM_ORDER[0]].dtype
    dev = torch.device(device) if device is not None else W[PARAM_ORDER[0]].device
    E = int(num_executors)
    bt = _Batch(obs, dev)
    B, S, J = bt.B, bt.S, bt.J
    if h is None:
        hc = _encode(W, bt)
        h_pad = _scatter_nodes(bt, hc)
    else:
        h_pad = h
        hc = h.reshape(B * S, -1)[bt.node_g]
    X = bt.x.reshape(-1, 5)[bt.node_g].to(dt)
    # DagEncoder, GlobalEncoder
    z = _mlp(torch.cat([X, hc], 1), W, "encoder.dag_encoder.mlp", _leaky)
    h_dag = torch.zeros(B * J, 16, dtype=dt, device=dev).index_add(0, bt.node_jobg, z)
    gj = _mlp(h_dag[bt.job_g], W, "encoder.global_encoder.mlp", _leaky)
    h_glob = torch.zeros(B, 16, dtype=dt, device=dev).index_add(0, bt.job_env, gj)
    # stage head over the schedulable nodes, in node order
    cand_c = torch.nonzero(bt.stage_mask.reshape(-1)[bt.node_g]).squeeze(1)   # compact rows of the candidates
    c_env = bt.node_env[cand_c]
    inp = torch.cat([X[cand_c], hc[cand_c], h_dag[bt.node_jobg[cand_c]], h_glob[c_env]], 1)
    zs = _mlp(inp, W, "stage_policy_network.mlp_score", torch.tanh)[:, 0]
    rank = (torch.cumsum(bt.stage_mask.long(), 1) - 1).reshape(-1)[bt.node_g[cand_c]]
    n_cand = bt.stage_mask.sum(1)
    stage = torch.full((B, S), -math.inf, dtype=dt, device=dev).index_put((c_env, rank), zs)
    act = bt.action
    has = bt.live & (n_cand > 0)
    assert torch.equal(torch.where(has, act[:, 3], 0), torch.where(has, n_cand, 0)), "candidate count differs"
    # the chosen stage's job must be the action's job
    sel_s = act[:, 0].clamp(min=0)
    cand_job = torch.full((B, S), -1, dtype=torch.long, device=dev).index_put((c_env, rank), bt.node_job[cand_c])
    assert torch.equal(torch.where(has, cand_job[torch.arange(B, device=dev), sel_s.clamp(max=S - 1)], -1),
                       torch.where(has, act[:, 1], -1)), "action's job is not the chosen stage's job"
    # executor-count head: rows c = 0 .. cap - 1 of the chosen job
    job = act[:, 1].clamp(min=0)
    cap = torch.where(has & (act[:, 1] >= 0), bt.caps.gather(1, job[:, None])[:, 0], 0)
    assert int(cap.max().item() if B else 0) <= E
    rows = torch.nonzero(torch.arange(E, device=dev)[None, :] < cap[:, None])
    r_env, r_c = rows[:, 0], rows[:, 1]
    # (a slot that takes no part may hold anything in dag_ptr: an empty slot of a gathered batch is not written)
    first = torch.where(has, bt.dag_ptr.gather(1, job[:, None])[:, 0], 0).clamp(min=0, max=S - 1)
    x_dag = bt.x[torch.arange(B, device=dev), first, :3].to(dt)
    cnt = (r_c.double() / E).float().to(dt)[:, None]
    inp = torch.cat([x_dag[r_env], h_dag[r_env * J + job[r_env]], h_glob[r_env], cnt], 1)
    ze = _mlp(inp, W, "exec_policy_network.mlp_score", torch.tanh)[:, 0]
    execs = torch.full((B, E), -math.inf, dtype=dt, device=dev).index_put((r_env, r_c), ze)
    # utils.evaluate per env: clamped softmax, lgprob of the action, entropy
    lgprob = torch.zeros(B, dtype=dt, device=dev)
    ent = torch.zeros(B, dtype=dt, device=dev)
    for scores, valid, sel, on in ((stage, torch.arange(S, device=dev)[None, :] < n_cand[:, None], act[:, 0], has),
                                   (execs, torch.arange(E, device=dev)[None, :] < cap[:, None], act[:, 2], cap > 0)):
        safe = torch.where(on[:, None], scores, torch.zeros_like(scores))
        q = torch.softmax(safe, 1).clamp(min=EPS32, max=1.0 - EPS32)
        lq = q.log()
        lg = lq.gather(1, sel.clamp(min=0, max=scores.shape[1] - 1)[:, None])[:, 0]
        lgprob = lgprob + torch.where(on, lg, torch.zeros_like(lg))
        hq = torch.where(valid & on[:, None], -q * lq, torch.zeros_like(q)).sum(1)
        ent = ent + hq
    norm = torch.log((E * bt.N).clamp(min=2).to(dt))
    entropy = torch.where(has, ent / norm, torch.zeros_like(ent))
    out = {"stage_scores": stage, "exec_scores": execs, "lgprob": lgprob, "entropy": entropy, "h": h_pad,
           "n_cand": n_cand, "cap": cap}
    if coef_lgprob is not None:
        c1 = coef_lgprob.to(device=dev, dtype=dt)
        c2 = coef_entropy.to(device=dev, dtype=dt)
        out["loss"] = (torch.where(bt.live, c1 * lgprob + c2 * entropy, torch.zeros_like(lgprob))).sum()
    return out
