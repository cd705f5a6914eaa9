"""Pins oracle/decima_torch.py (the batched torch restatement of DecimaScheduler.evaluate_actions that the GPU tests
measure the device's forward and backward passes against) to the numpy restatement oracle/decima_policy.py and to what
the reference DecimaScheduler itself recorded: scores and lgprobs on every decision of the Decima goldens, lgprobs,
entropies and all 42 parameter gradients of its own evaluate_actions + loss.backward() on batches of observations."""
import os.path as osp

import numpy as np
import pytest
import torch

import decima_policy
import decima_torch
from helpers import GOLDEN_DIR, golden_names, load_golden
from test_decima_policy_oracle import iter_decisions

SCORE_TOL = 2e-5   # against the reference's recorded float32 scores (as test_decima_policy_oracle)
LGPROB_TOL = 1e-4


def _model():
    z = np.load(osp.join(GOLDEN_DIR, "decima_model.npz"))
    return {k: z[k] for k in z.files}


def _batch(tr, picks=None):
    obs, acts = [], []
    for k, o in iter_decisions(tr):
        if picks is not None and k not in picks:
            continue
        o = dict(o, caps=o["caps"])
        obs.append(o)
        acts.append(list(o["action"]) + [len(o["stage_logits"])])
    return obs, decima_torch.stack_observations(obs, acts)


@pytest.mark.parametrize("name", [n for n in golden_names(slim=False) if n.startswith("decima_")])
def test_batched_reference_matches_the_numpy_oracle_and_the_recorded_scores(name):
    """All decisions of a golden episode in one batch: the fp64 batched restatement equals decima_policy's fp64
    evaluation decision by decision (1e-12: the same arithmetic, summed in another order), and is as close to the
    reference's recorded float32 scores and lgprobs as the numpy oracle is required to be."""
    tr = load_golden(name)
    E = tr["num_executors"]
    w = _model()
    w64 = {k: v.astype(np.float64) for k, v in w.items()}
    obs, batch = _batch(tr)
    with torch.no_grad():
        out = decima_torch.evaluate_actions(decima_torch.weights(w, requires_grad=False), batch, num_executors=E)
    stage, execs = out["stage_scores"].numpy(), out["exec_scores"].numpy()
    lg = out["lgprob"].numpy()
    worst_np = worst_ref = worst_lg = 0.0
    depths = []
    for b, o in enumerate(obs):
        f64 = o["features"].astype(np.float64)
        h, h_dag, h_glob = decima_policy.encode(w64, f64, o["edge_links"], o["edge_bits"], o["depth"], o["dag_ptr"])
        ts, _ = decima_policy.stage_scores(w64, f64, h, h_dag, h_glob, o["dag_ptr"], o["stage_mask"])
        stage_idx, job_idx, num_exec = o["action"]
        te = decima_policy.exec_scores(w64, f64, h_dag, h_glob, o["dag_ptr"], job_idx, int(o["caps"][job_idx]), E)
        ns, ne = len(ts), len(te)
        assert np.isneginf(stage[b, ns:]).all() and np.isneginf(execs[b, ne:]).all(), b
        worst_np = max(worst_np, float(np.abs(stage[b, :ns] - ts).max()), float(np.abs(execs[b, :ne] - te).max()))
        worst_ref = max(worst_ref, float(np.abs(stage[b, :ns] - o["stage_logits"]).max()),
                        float(np.abs(execs[b, :ne] - o["exec_logits"]).max()))
        worst_lg = max(worst_lg, abs(float(lg[b]) - o["lgprob"]))
        depths.append(o["depth"])
    print(f"{name}: {len(obs)} observations, max depth {max(depths)}: |batched - numpy fp64| {worst_np:.3g}, "
          f"|batched - recorded| {worst_ref:.3g}, lgprob {worst_lg:.3g}")
    assert worst_np < 1e-12, worst_np
    assert worst_ref < SCORE_TOL and worst_lg < LGPROB_TOL, (worst_ref, worst_lg)
    assert np.isfinite(out["entropy"].numpy()).all() and (out["entropy"].numpy() > 0).any()


@pytest.mark.parametrize("fixture", ["decima_grads_e10_j8_s5", "decima_grads_e50_j14_s4"])
def test_batched_reference_reproduces_the_reference_models_gradients(fixture):
    """The pick observations of a recorded episode in one batch, the stored coefficients, loss.backward() in fp64:
    lgprobs, entropies and all 42 gradients of the unmodified reference model (recorded in float32) come back to
    float32 rounding -- each tensor within 2e-5 of its largest entry + 1e-6 (the device tests allow 5e-4)."""
    g = np.load(osp.join(GOLDEN_DIR, fixture + ".npz"))
    tr = load_golden(str(g["trace"]))
    picks = [int(k) for k in g["picks"]]
    _, batch = _batch(tr, set(picks))
    W = decima_torch.weights(_model())
    out = decima_torch.evaluate_actions(W, batch, torch.from_numpy(g["coef_lgprob"]), torch.from_numpy(g["coef_entropy"]),
                                        num_executors=tr["num_executors"])
    out["loss"].backward()
    err_lg = float(np.abs(out["lgprob"].detach().numpy() - g["lgprobs"]).max())
    err_en = float(np.abs(out["entropy"].detach().numpy() - g["entropies"]).max())
    assert abs(float(out["loss"].detach()) - float(g["loss"])) < 1e-5 * max(1.0, abs(float(g["loss"])))
    worst, off = 0.0, 0
    for name in decima_torch.PARAM_ORDER:
        got = W[name].grad.numpy().reshape(-1)
        want = g["grad"][off:off + got.size]
        rel = float(np.abs(got - want).max()) / float(np.abs(want).max())
        worst = max(worst, rel if np.abs(want).max() > 1e-3 else 0.0)
        # (a score head's last bias: softmax is shift-invariant, its gradient is a sum that cancels to ~0 -- rounding)
        assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max() + 1e-6, (name, rel)
        off += got.size
    print(f"{fixture}: lgprob {err_lg:.3g}, entropy {err_en:.3g}, worst gradient tensor {worst:.3g} of its largest entry")
    assert off == 20802
    assert err_lg < 2e-5 and err_en < 2e-5, (err_lg, err_en)
