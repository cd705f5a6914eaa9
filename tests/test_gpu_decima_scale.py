"""evaluate_actions' forward and backward passes on the device (ssb_decima_evaluate + ssb_decima_backward) at training
batch sizes, against the batched fp64 restatement of the whole policy (oracle/decima_torch.py, pinned to the reference
DecimaScheduler by test_decima_torch_ref.py) on the same observations and actions.

At these sizes the node-level MLP passes run several 128-row tiles per persistent CTA (the weight-gradient
accumulators and the shared tile matrix of k_mlp_backward carry over between tiles), the message-passing levels go
nine to sixty deep, and the batches mix envs that are live, finished, errored or empty.  Every execution path is
compared: the list-driven tile kernels (mode 0) with the levels replayed by the backward pass, saved by the
evaluation, or recomputed per level (SSB_BACKWARD_RECOMPUTE); the backward stopped above NodeEncoder (d loss / d h);
the fused kernel (mode 1); a shuffled mini-batch gathered from stored observations with empty slots.

Tolerance rule, for every compared quantity Q (scores, lgprob, entropy, each of the 42 gradient tensors, d_h):
    err_dev = max |Q_dev - Q_64|,  err_32 = max |Q_t32 - Q_64|   (Q_t32: the same restatement in float32, TF32 off)
    err_dev <= FP64_FACTOR * err_32 + C * max |Q_64|
i.e. the device must be as close to fp64 as a straightforward float32 evaluation of the same batch, up to a small
floor C relative to the quantity's own scale (float32 atomics over ~1e6 rows, bf16x3 tensor-core products).
For a gradient tensor max |Q_64| is taken over the six tensors of its MLP: a score head's last bias is a sum that
cancels to ~0 (softmax is shift-invariant), and what remains of it on every side is the rounding of that MLP's terms."""
import contextlib
import os.path as osp

import numpy as np
import pytest
import torch

import decima_torch
from helpers import GOLDEN_DIR

pytestmark = pytest.mark.gpu

FP64_FACTOR = 3.0
# Measured on a B200 (1000 W), worst over the paths and shapes: err_dev / err_32 vs fp64 of
#   scores   1.5e-5 / 9.2e-6 of 10.2
#   lgprob   5.4e-6 / 2.6e-6
#   entropy  3.6e-7 / 2.6e-7
#   grad     7.7e-4 / 3.0e-5 of 57.5 (the job summary's MLP at the wide shape, every path alike: float32 sums over
#            1.7e5 rows in per-CTA registers and atomics, torch's in a reduction tree)
#   d_h      2.1e-6 / 3.6e-7 of 1.6
C_FLOOR = {"scores": 1e-6, "lgprob": 1e-6, "entropy": 3e-6, "grad": 3e-5, "d_h": 3e-6}

SHAPES = {
    # name: (env config, bank, envs, fair decisions into the episodes, auto-reset, mean time limit)
    "c2": ({"num_executors": 10, "job_arrival_cap": 50}, "appd", 2048, 1500, True, 0.0),
    "c3": ({"num_executors": 50, "job_arrival_cap": 200}, "appd", 512, 300, True, 2.0e7),
    "wide": ({"num_executors": 10, "job_arrival_cap": 20}, "wide", 256, 300, False, 0.0),
}


def _weights():
    z = np.load(osp.join(GOLDEN_DIR, "decima_model.npz"))
    return {k: z[k] for k in z.files}


@contextlib.contextmanager
def _strict_fp32():
    """float32 matmuls in float32 (no TF32) for the yardstick; the previous settings come back afterwards."""
    tf32, prec = torch.backends.cuda.matmul.allow_tf32, torch.get_float32_matmul_precision()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.set_float32_matmul_precision(prec)


def _make_env(shape, mode, monkeypatch):
    from spark_sched_sim_b200.bank import synthetic_bank
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    cfg, bank_kind, B, warm, auto, time_limit = SHAPES[shape]
    cfg = dict(cfg, job_arrival_rate=4.0e-5, moving_delay=2000.0, warmup_delay=1000.0)
    monkeypatch.setenv("SSB_DECIMA_MODE", mode)  # read when the handle is created
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=synthetic_bank(0, bank_kind), decima_policy=True)
    monkeypatch.delenv("SSB_DECIMA_MODE")
    env.set_decima_weights(_weights())
    if time_limit:
        env.set_mean_time_limit(time_limit)
    env.set_autoreset(auto, B)
    env.reset_host(np.arange(B, dtype=np.uint64) + 4321)
    env.rollout_fair(warm, True, auto, B)  # into mid / late episodes (the fair policy is deterministic)
    return env


def _reference(obs, c1, c2, E, to_h=False):
    """fp64 and float32 runs of the restatement: scores, lgprob, entropy, the 42 gradients (to_h: the gradients of
    the tensors above NodeEncoder and d loss / d h, with the restatement's own h as a leaf)."""
    w = _weights()
    res = {}
    for dt in (torch.float64, torch.float32):
        with _strict_fp32():
            W = decima_torch.weights(w, dt, "cuda")
            if to_h:
                with torch.no_grad():
                    h = decima_torch.encode_nodes(W, obs)
                h.requires_grad_()
                out = decima_torch.evaluate_actions(W, obs, c1, c2, h=h, num_executors=E)
            else:
                out = decima_torch.evaluate_actions(W, obs, c1, c2, num_executors=E)
            out["loss"].backward()
        r = {k: out[k].detach() for k in ("stage_scores", "exec_scores", "lgprob", "entropy")}
        r["grad"] = [W[k].grad if W[k].grad is not None else torch.zeros_like(W[k]) for k in decima_torch.PARAM_ORDER]
        if to_h:
            r["d_h"] = h.grad
        res[dt] = r
    return res[torch.float64], res[torch.float32]


class _Check:
    """Collects err_dev / err_32 per quantity; the bound is asserted once everything has been printed."""

    def __init__(self):
        self.bad = []

    def __call__(self, tag, kind, dev, r64, r32, mask=None, scale=None):
        d, a, b = dev.double(), r64.double(), r32.double()
        if mask is not None:
            d, a, b = d[mask], a[mask], b[mask]
        if a.numel() == 0:
            return 0.0, 0.0, 0.0
        err_dev, err_32 = (float(x) for x in ((d - a).abs().max(), (b - a).abs().max()))
        scale = float(a.abs().max()) if scale is None else scale
        if not err_dev <= FP64_FACTOR * err_32 + C_FLOOR[kind] * scale:
            self.bad.append((tag, kind, err_dev, err_32, scale))
        return err_dev, err_32, scale


def _evaluate(env, snap, act, for_backward, c1, c2, through=True, recompute=False, monkeypatch=None):
    """evaluate + backward of the stored observation `snap` with the actions `act`; returns the device's outputs and
    the observation as the policy saw it (copies)."""
    env.decima_snapshot_load(snap)
    try:
        lg, en = env.decima_evaluate(None, act[:, 0].contiguous(), act[:, 2].contiguous(), for_backward=for_backward)
        out = {"lgprob": lg.clone(), "entropy": en.clone(), "stage": env.pol_stage_logits.clone(),
               "exec": env.pol_exec_logits.clone()}
        out["obs"] = {k: v.clone() for k, v in decima_torch.handle_observation(env).items()}
        out["work"] = env.decima_work()
        if recompute:
            monkeypatch.setenv("SSB_BACKWARD_RECOMPUTE", "1")  # read by every backward call
        gw = torch.zeros(20802, dtype=torch.float32, device="cuda")
        d_h = env.decima_backward(c1, c2, gw, through_node_encoder=through)
        torch.cuda.synchronize()
        if recompute:
            monkeypatch.delenv("SSB_BACKWARD_RECOMPUTE")
        out["grad"], out["d_h"] = gw, (None if through else d_h.clone())
    finally:
        env.decima_snapshot_unload()
    return out


def _compare(check, tag, out, r64, r32, E, to_h=False):
    """Prints and checks one path; returns the per-kind (err_dev, err_32) of the path."""
    stage_mask = torch.isfinite(r64["stage_scores"])
    exec_mask = torch.isfinite(r64["exec_scores"])
    S = stage_mask.shape[1]
    row = {"scores": check(tag, "scores", out["stage"][:, :S], r64["stage_scores"], r32["stage_scores"], stage_mask)}
    e2 = check(tag, "scores", out["exec"][:, :E], r64["exec_scores"], r32["exec_scores"], exec_mask)
    row["scores"] = max(row["scores"], e2)
    row["lgprob"] = check(tag, "lgprob", out["lgprob"], r64["lgprob"], r32["lgprob"])
    row["entropy"] = check(tag, "entropy", out["entropy"], r64["entropy"], r32["entropy"])
    sizes = [int(np.prod(g.shape)) for g in r64["grad"]]
    off = np.concatenate([[0], np.cumsum(sizes)])
    worst, worst_name = (0.0, 0.0, 1.0), ""
    for i, name in enumerate(decima_torch.PARAM_ORDER):
        got = out["grad"][off[i]:off[i + 1]].view(r64["grad"][i].shape)
        if to_h and i < 18:
            assert not got.any(), (tag, name, "NodeEncoder's tensors are not part of this backward")
            continue
        mlp_scale = max(float(t.abs().max()) for t in r64["grad"][6 * (i // 6):6 * (i // 6) + 6])
        e = check(tag + " " + name, "grad", got, r64["grad"][i], r32["grad"][i], scale=mlp_scale)
        if e[0] / max(e[2], 1e-30) > worst[0] / max(worst[2], 1e-30):
            worst, worst_name = e, name
    row["grad"] = worst
    if to_h:
        n = out["obs"]["num_nodes"].long() * out["obs"]["live"].long()
        node_mask = torch.arange(r64["d_h"].shape[1], device="cuda")[None, :] < n[:, None]
        row["d_h"] = check(tag, "d_h", out["d_h"][:, :node_mask.shape[1]], r64["d_h"], r32["d_h"], node_mask)
        assert not out["d_h"][:, :node_mask.shape[1]][~node_mask].any(), (tag, "d_h outside the live nodes")
    txt = "  ".join(f"{k} {v[0]:.2e}/{v[1]:.2e} (of {v[2]:.2e})" for k, v in row.items())
    print(f"  {tag:<26} dev/t32 vs fp64: {txt}  [worst gradient tensor: {worst_name}]")
    return row


def _rows(work):
    return f"nodes {work['nodes']}, senders {work['senders']}, receivers {work['receivers']}, " \
           f"candidates {work['candidates']}, exec rows {work['exec_rows']}"


@pytest.mark.parametrize("shape", list(SHAPES))
def test_evaluate_and_backward_at_training_sizes_against_fp64(shape, monkeypatch):
    """Every execution path on one shape; per path the device's scores, lgprob, entropy, the 42 gradients (and d_h)
    against fp64 under the rule of the module docstring, and the evaluation's lgprob bit-equal to the one stored when
    the action was sampled in the same mode."""
    cfg, _, B, _, _, _ = SHAPES[shape]
    E = cfg["num_executors"]
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    g = torch.Generator(device="cuda").manual_seed(11)
    c1 = torch.randn(B, device="cuda", generator=g)
    c2 = torch.randn(B, device="cuda", generator=g)
    check = _Check()
    print(f"\n{shape}: {B} envs, {E} executors, {torch.cuda.get_device_name(0)}")
    for mode, paths in (("0", ("replay", "to-h", "saved", "recompute")), ("1", ("fused",))):
        env = _make_env(shape, mode, monkeypatch)
        snap = env.decima_snapshot()
        env.decima_policy()
        act, lg_sampled = env.pol_action.clone(), env.pol_lgprob.clone()
        refs = {}
        for path in paths:  # ("replay" first: once a backward has attached its scratch, evaluations save the levels)
            out = _evaluate(env, snap, act, for_backward=path == "saved", c1=c1, c2=c2,
                            through=path != "to-h", recompute=path == "recompute", monkeypatch=monkeypatch)
            assert torch.equal(out["obs"]["action"][:, [0, 2]], act[:, [0, 2]]), (shape, path)
            assert torch.equal(out["lgprob"], lg_sampled), (shape, path, "evaluate's lgprob != the sampled one")
            key = path == "to-h"
            if key not in refs:
                refs[key] = _reference(out["obs"], c1, c2, E, to_h=key)
            if path in ("replay", "fused"):
                obs = out["obs"]
                live = obs["live"]
                depth = int(obs["depth"][live].max()) if live.any() else 0
                no_cand = int((live & (obs["action"][:, 3] == 0)).sum())
                print(f"  mode {mode}: {int(live.sum())} live envs of {B} ({no_cand} without a candidate), max depth "
                      f"{depth}; {_rows(out['work'])}")
                if shape == "wide":
                    assert depth >= 14, depth  # (the bank's deepest template: 16 levels of edges)
                if shape in ("c2", "c3"):
                    # several 128-row tiles per CTA in the node-level passes (grids of num_sms x 4 CTAs and more)
                    assert out["work"]["nodes"] > 2 * 4 * num_sms * 128, out["work"]
                assert live.sum() > B // 2
            _compare(check, f"mode {mode} {path}", out, *refs[key], E, to_h=key)
        env.close()
    assert not check.bad, check.bad


def test_gathered_minibatch_at_training_size_against_fp64(monkeypatch):
    """A PPO mini-batch as ppo_train_samples builds it: RolloutStore.collect() over the C2-shape handle, then a
    shuffled gather of stored samples into the handle's slots with every 8th slot empty (src_step = -1).  Evaluate +
    backward (mode 0) against fp64 on the gathered batch; the evaluation reproduces the stored lgprobs bit for bit
    and the empty slots contribute nothing."""
    from spark_sched_sim_b200 import ppo

    shape = "c2"
    cfg, _, B, _, _, _ = SHAPES[shape]
    E = cfg["num_executors"]
    env = _make_env(shape, "0", monkeypatch)
    store = ppo.RolloutStore(env, 4).collect()
    valid = torch.nonzero(store.valid.reshape(-1)).squeeze(1)
    gen = torch.Generator(device="cuda").manual_seed(5)
    pick = valid[torch.randperm(valid.numel(), device="cuda", generator=gen)[:B]]
    ks = (pick // B).int()
    bs = (pick % B).int()
    ks[::8] = -1  # empty slots
    assert ks.numel() == B
    g = torch.Generator(device="cuda").manual_seed(12)
    c1 = torch.randn(B, device="cuda", generator=g)
    c2 = torch.randn(B, device="cuda", generator=g)
    staging = torch.empty(env.decima_snapshot_bytes(), dtype=torch.uint8, device="cuda")
    lg, en = ppo._evaluate_slots(env, store, staging, ks, bs)
    try:
        out = {"lgprob": lg.clone(), "entropy": en.clone(), "stage": env.pol_stage_logits.clone(),
               "exec": env.pol_exec_logits.clone(), "work": env.decima_work()}
        out["obs"] = {k: v.clone() for k, v in decima_torch.handle_observation(env).items()}
        gw = torch.zeros(20802, dtype=torch.float32, device="cuda")
        env.decima_backward(c1, c2, gw)
        out["grad"], out["d_h"] = gw, None
    finally:
        env.decima_snapshot_unload()
    empty = ks < 0
    real = ~empty
    kk, bb = ks.clamp(min=0).long(), bs.long()
    assert torch.equal(out["lgprob"][real], store.lgprob[kk, bb][real])
    assert not out["lgprob"][empty].any() and not out["entropy"][empty].any()
    assert not out["obs"]["live"][empty].any() and out["obs"]["live"][real].all()
    print(f"\ngathered mini-batch: {int(real.sum())} samples + {int(empty.sum())} empty slots; {_rows(out['work'])}")
    r64, r32 = _reference(out["obs"], c1, c2, E)
    check = _Check()  # (the reference leaves the empty slots out; their coefficients c1, c2 are not zero)
    _compare(check, "gathered mode 0", out, r64, r32, E)
    env.close()
    assert not check.bad, check.bad
