"""GPU parity of the Decima policy kernel (ssb_decima_policy) against the scores the reference's
DecimaScheduler (shipped model.pt) produced on every decision of the recorded Decima-driven episodes.
float32-accurate MLPs with a different summation order than torch's sgemm: the scores are compared with the recorded
ones at the floor two float32 evaluations can agree to, and with an fp64 evaluation of the same weights, to which the
kernel must be as close as the reference's own float32 forward; actions are replayed (the reference samples with
python's `random`, the kernel with Philox), so the trajectory itself must match the golden trace exactly."""
import os.path as osp

import numpy as np
import pytest
import torch

import decima_policy

from helpers import GOLDEN_DIR, bank_for, decima_digest, golden_names, load_golden

pytestmark = pytest.mark.gpu
# Two float32 evaluations of the same network with different summation orders differ by a few 1e-6 relative, so the
# distance to the reference's RECORDED float32 scores has a floor of that size (TOL / REL_TOL below).  The accuracy
# claim proper is made against an fp64 evaluation of the same weights on the same observation ("truth"): the kernel
# must be as close to it as the reference's own float32 forward is (FP64_FACTOR).
TOL = 2.5e-5      # absolute, on scores of magnitude 10 .. 20
REL_TOL = 4e-6    # relative to max(|score|, 1)
LGPROB_TOL = 2e-5
FP64_FACTOR = 3.0   # measured: 1.6 .. 2.1 (8e-6 .. 1.2e-5 absolute on scores of magnitude 10 .. 20, i.e. < 1e-6 relative)
FP64_REL = 2.0e-6   # kernel vs fp64, relative to the largest score of the episode (measured 0.7e-6 .. 1.6e-6; the
                    # reference's own float32 forward: 0.5e-6 .. 1.3e-6)


def env_cfg_of(tr):
    return {"num_executors": tr["num_executors"], "job_arrival_cap": tr["job_arrival_cap"],
            "job_arrival_rate": tr["job_arrival_rate"], "moving_delay": tr["moving_delay"],
            "warmup_delay": tr["warmup_delay"], "beta": tr["beta"]}


def weights():
    z = np.load(osp.join(GOLDEN_DIR, "decima_model.npz"))
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("name", [n for n in golden_names() if n.startswith("decima_")])
def test_policy_scores_match_reference(name):
    """Every Decima golden: the small episodes (all scores kept), the wide-template one (jobs of 30..64 stages), the
    headline shape (50 jobs x 10 executors) and config/decima_tpch.yaml:80-87 (200 jobs x 50 executors; the scores of
    every 8th decision kept, the adapter's outputs as a digest per observation)."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    tr = load_golden(name)
    bank = bank_for(tr)
    B, slot = 2, 1
    kept = {int(k) for k in tr["pol_kept"]} if "pol_kept" in tr else None
    env = BatchedSparkSchedSimEnv(env_cfg_of(tr), num_envs=B, bank=bank, max_jobs=len(tr["job_template"]) + 2,
                                  tape_capacity=len(tr["tape"]) + 8, decima_policy=True)
    env.set_decima_weights(weights())
    for b in range(B):
        env.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    env.reset_host(np.full(B, tr["seed"], np.uint64))
    so = eo = 0
    worst = worst_rel = err_dev = err_ref = scale = 0.0
    w64 = {k: v.astype(np.float64) for k, v in weights().items()}
    n_kept = len(tr["pol_kept"]) if "pol_kept" in tr else len(tr["actions"])
    n_truth, n_seen, truth_stride = 0, 0, max(1, n_kept // 50)
    for k in range(len(tr["actions"])):
        ns, ne = int(tr["pol_stage_count"][k]), int(tr["pol_exec_count"][k])
        stage_idx, job_idx, num_exec = (int(x) for x in tr["pol_actions"][k])
        a, n = env.decima_policy(forced_stage=np.full(B, stage_idx, np.int32),
                                 forced_num_exec=np.full(B, num_exec, np.int32))
        act = env.pol_action[slot].cpu().numpy()
        assert act.tolist() == [stage_idx, job_idx, num_exec, ns], (k, act)
        assert abs(float(env.pol_lgprob[slot].item()) - float(tr["pol_lgprob"][k])) < LGPROB_TOL, k
        if "dec_digest" in tr:  # the adapter ran inside the policy call: its outputs against the reference wrapper's
            d = env.decima_obs_host(slot)
            assert decima_digest(d["features"], d["commit_caps"], d["depth"], d["edge_bits"],
                                 d["stage_mask"].astype(np.uint8)) == int(tr["dec_digest"][k]), (k, "decima obs")
        if kept is not None and k not in kept:  # scores not kept for this decision: replay only
            assert (int(a[slot].item()), int(n[slot].item())) == tuple(tr["actions"][k]), k
            env.step(a, n)
            h = env.hdr()[slot]
            assert h["error"] == 0 and h["wall_time"] == tr["wall"][k] and h["reward"] == tr["reward"][k], k
            continue
        sl = env.pol_stage_logits[slot, :ns].cpu().numpy()
        el = env.pol_exec_logits[slot, :ne].cpu().numpy()
        ref_s, ref_e = tr["pol_stage_logits"][so:so + ns], tr["pol_exec_logits"][eo:eo + ne]
        worst = max(worst, float(np.abs(sl - ref_s).max()), float(np.abs(el - ref_e).max()) if ne else 0.0)
        worst_rel = max(worst_rel, float((np.abs(sl - ref_s) / np.maximum(np.abs(ref_s), 1.0)).max()))
        n_seen += 1
        if n_truth < 60 and n_seen % truth_stride == 0:
            # fp64 evaluation of the policy on the observation the device itself built (bit-equal to the reference
            # wrapper's, checked above / in test_gpu_decima_obs): who is closer to it, the kernel or the reference?
            d = env.decima_obs_host(slot)
            o = env.obs(slot)
            f64 = d["features"].astype(np.float64)
            h, h_dag, h_glob = decima_policy.encode(w64, f64, o["edge_links"], d["edge_bits"], d["depth"], o["dag_ptr"])
            ts, _ = decima_policy.stage_scores(w64, f64, h, h_dag, h_glob, o["dag_ptr"], d["stage_mask"])
            te = decima_policy.exec_scores(w64, f64, h_dag, h_glob, o["dag_ptr"], job_idx, ne, tr["num_executors"])
            err_dev = max(err_dev, float(np.abs(sl - ts).max()), float(np.abs(el - te).max()) if ne else 0.0)
            err_ref = max(err_ref, float(np.abs(ref_s - ts).max()), float(np.abs(ref_e - te).max()) if ne else 0.0)
            scale = max(scale, float(np.abs(ts).max()))
            n_truth += 1
        # evaluate_actions' entropy (scheduler.py:131-137, utils.py:26-42) from the REFERENCE's recorded scores
        def _h(z):
            z = z.astype(np.float64); pr = np.exp(z - z.max()); pr /= pr.sum()
            pr = np.clip(pr, np.finfo(np.float32).eps, 1 - np.finfo(np.float32).eps)
            return float(-(pr * np.log(pr)).sum())
        want_h = (_h(tr["pol_stage_logits"][so:so + ns]) + (_h(tr["pol_exec_logits"][eo:eo + ne]) if ne else 0.0)) \
            / np.log(tr["num_executors"] * int(tr["N"][k]))
        assert abs(float(env.pol_entropy[slot].item()) - want_h) < 2e-4, (k, want_h)
        # env-format action (DecimaActWrapper) and the step it drives
        assert (int(a[slot].item()), int(n[slot].item())) == tuple(tr["actions"][k]), k
        env.step(a, n)
        h = env.hdr()[slot]
        assert h["error"] == 0 and h["wall_time"] == tr["wall"][k] and h["reward"] == tr["reward"][k], k
        so += ns; eo += ne
    print(f"{name}: worst |score - reference| {worst:.3g} abs, {worst_rel:.3g} rel; against fp64 on {n_truth} "
          f"observations (largest score {scale:.3g}): kernel {err_dev:.3g}, reference's float32 forward {err_ref:.3g}")
    assert worst < TOL and worst_rel < REL_TOL, (worst, worst_rel)
    assert n_truth >= 20 and err_dev <= FP64_FACTOR * err_ref and err_dev <= FP64_REL * scale, (err_dev, err_ref, scale)
    assert bool(env.hdr()[slot]["terminated"])
    assert np.array_equal(env.jobs(slot)[1], tr["job_t_completed"])


def test_policy_sampling_rollout_and_distribution(bank):
    """Sampling on the device: (1) many envs in the same state but with different seeds pick stages
    with the softmax frequencies; (2) policy + step loops run whole episodes without errors."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    tr = load_golden("decima_e10_j8_s5_philox")
    B = 2048
    env = BatchedSparkSchedSimEnv(env_cfg_of(tr), num_envs=B, bank=bank, max_jobs=10,
                                  tape_capacity=len(tr["tape"]) + 8, decima_policy=True)
    env.set_decima_weights(weights())
    for b in range(B):
        env.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    # identical episodes (same tape); the seeds only key the Philox policy stream
    env.reset_host(np.arange(B, dtype=np.uint64) + 77)
    checked = 0
    for k in range(60):
        stage_idx, _, num_exec = (int(x) for x in tr["pol_actions"][k])
        ns = int(tr["pol_stage_count"][k])
        if ns >= 3 and checked < 4:  # sample (without stepping) and compare frequencies with softmax
            env.decima_policy()
            acts = env.pol_action.cpu().numpy()
            s = env.pol_stage_logits[0, :ns].cpu().numpy().astype(np.float64)
            p = np.exp(s - s.max()); p /= p.sum()
            assert (acts[:, 3] == ns).all() and (acts[:, 0] >= 0).all() and (acts[:, 0] < ns).all()
            freq = np.bincount(acts[:, 0], minlength=ns) / B
            assert np.abs(freq - p).max() < 0.05, (k, freq, p)
            assert len(np.unique(acts[:, 0])) > 1 or p.max() > 0.97
            checked += 1
        a, n = env.decima_policy(forced_stage=np.full(B, stage_idx, np.int32),
                                 forced_num_exec=np.full(B, num_exec, np.int32))
        env.step(a, n)
    assert checked >= 2
    # (2) whole episodes with sampled actions
    env.reset_host(np.arange(B, dtype=np.uint64) + 5)
    for _ in range(3000):
        a, n = env.decima_policy()
        env.step(a, n)
        h = env.hdr()
        if (h["terminated"] != 0).all():
            break
        assert ((h["error"] == 0) | (h["error"] == 9)).all(), np.unique(h["error"])
    h = env.hdr()
    assert (h["terminated"] != 0).all()
    assert torch.isfinite(env.pol_lgprob).all()


def test_rollout_decima_records_the_python_loop(bank):
    """ssb_rollout_decima == the loop { decima_policy ; step } driven from Python with the same seeds (the
    Philox policy stream makes sampling reproducible): every recorded wall time, action, lgprob, reward and
    flag, across auto-resets."""
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, K = 8, 400
    cfg = {"num_executors": 10, "job_arrival_cap": 5, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    seeds = np.arange(B, dtype=np.uint64) + 21
    envs = []
    for _ in range(2):
        e = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
        e.set_decima_weights(weights())
        e.reset_host(seeds)
        e.set_autoreset(True, 100)
        envs.append(e)
    host = torch.empty(B * K * nat.TRANSITION_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    tr = envs[0].rollout_decima(K, host=host)
    e = envs[1]
    n_reset = n_term = 0
    for d in range(K):
        wall0 = e.hdr()["wall_time"].copy()
        a, n = e.decima_policy()
        lg = e.pol_lgprob.cpu().numpy().copy()
        e.step(a, n)
        h = e.hdr()
        a_h, n_h = a.cpu().numpy(), n.cpu().numpy()
        for b in range(B):
            r = tr[b, d]
            if h["was_reset"][b]:
                assert r["flags"] == 8, (b, d)
                n_reset += 1
                continue
            assert (r["wall_time"], r["stage_idx"], r["num_exec"], r["reward"]) == (wall0[b], a_h[b], n_h[b], h["reward"][b]), (b, d)
            assert r["lgprob"] == lg[b] and (r["flags"] & 1) == int(h["terminated"][b]), (b, d)
            n_term += int(h["terminated"][b])
    assert n_reset >= B and n_term >= B
    assert (envs[0].hdr()["wall_time"] == e.hdr()["wall_time"]).all()


def test_decima_scheduler_plugin_runs_like_examples_py(bank):
    """examples.py:76-102 with the drop-in classes: make_scheduler -> env_wrapper_cls(env) -> schedule/step loop.  The
    episode must equal the batched device rollout from the same seed (same Philox policy stream)."""
    from spark_sched_sim_b200 import metrics
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv
    from spark_sched_sim_b200.env import SparkSchedSimEnv
    from spark_sched_sim_b200.schedulers import make_scheduler

    cfg = {"num_executors": 10, "job_arrival_cap": 6, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    agent_cfg = {"agent_cls": "DecimaScheduler", "embed_dim": 16, "gnn_mlp_kwargs": {"hid_dims": [32, 16]},
                 "policy_mlp_kwargs": {"hid_dims": [64, 64]}, "num_executors": 10,
                 "state_dict_path": osp.join(GOLDEN_DIR, "decima_model.npz")}
    scheduler = make_scheduler(agent_cfg)
    env = scheduler.env_wrapper_cls(SparkSchedSimEnv(cfg, bank=bank))
    obs, _ = env.reset(seed=77, options=None)
    terminated = truncated = False
    steps, lg = 0, []
    while not (terminated or truncated):
        action, info = scheduler.schedule(obs)
        assert set(action) == {"stage_idx", "job_idx", "num_exec"} and np.isfinite(info["lgprob"])
        lg.append(info["lgprob"])
        obs, _, terminated, truncated, _ = env.step(action)
        steps += 1
    assert terminated and steps > 20
    jct = metrics.avg_job_duration(env) * 1e-3
    # the same episode through the batched API
    ref = BatchedSparkSchedSimEnv(cfg, num_envs=1, bank=bank, decima_policy=True)
    ref.set_decima_weights(weights())
    ref.reset_host(np.array([77], np.uint64))
    tr = ref.rollout_decima(steps, host=torch.empty(steps * 32, dtype=torch.uint8).pin_memory())
    assert bool(ref.hdr()[0]["terminated"]) and ref.hdr()[0]["wall_time"] == env.unwrapped.wall_time
    assert np.allclose(tr[0]["lgprob"], np.array(lg, np.float32))
    ta, tc, _ = ref.jobs(0)
    assert jct == pytest.approx(np.mean(tc - ta) * 1e-3)


def test_evaluate_actions_on_stored_observations(bank):
    """RolloutBuffer.obsns + evaluate_actions (forward): observations stored during a sampled rollout are re-evaluated
    later with the stored actions -- lgprobs and entropies come back bit for bit, and neither the envs' state nor
    their sampling stream is disturbed (a twin env that never evaluates stays identical)."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, K = 32, 40
    cfg = {"num_executors": 10, "job_arrival_cap": 8, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    envs = []
    for _ in range(2):
        e = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
        e.set_decima_weights(weights())
        e.reset_host(np.arange(B, dtype=np.uint64) + 400)
        envs.append(e)
    env, twin = envs
    snaps, acts, lgs, ens = [], [], [], []
    for k in range(K):
        snaps.append(env.decima_snapshot())
        a, n = env.decima_policy()
        acts.append(env.pol_action.clone())
        lgs.append(env.pol_lgprob.clone()); ens.append(env.pol_entropy.clone())
        if k % 7 == 3 and k > 3:  # interleave an evaluation of an older observation
            lg, en = env.decima_evaluate(snaps[k - 3], acts[k - 3][:, 0].contiguous(), acts[k - 3][:, 2].contiguous())
            assert torch.equal(lg, lgs[k - 3]) and torch.equal(en, ens[k - 3]), k
        env.step(a, n)
        a2, n2 = twin.decima_policy()
        twin.step(a2, n2)
        assert torch.equal(a, a2) and torch.equal(n, n2), k
    for k in range(K):
        lg, en = env.decima_evaluate(snaps[k], acts[k][:, 0].contiguous(), acts[k][:, 2].contiguous())
        assert torch.equal(lg, lgs[k]) and torch.equal(en, ens[k]), k
    assert np.array_equal(env.hdr()["wall_time"], twin.hdr()["wall_time"])
    assert torch.isfinite(torch.stack(ens)).all() and (torch.stack(ens) >= 0).all()


def test_head_adjoint_matches_torch_autograd(bank):
    """ssb_decima_head_adjoint (first stage of evaluate_actions' backward pass) vs autograd through the reference's
    utils.evaluate written in plain torch fp32 (softmax, clamp_probs, log-prob of the stored action, entropy,
    normalisation by log(num_executors * num_nodes)) on the scores the device produced.  Tolerance: 1e-5 relative
    + 1e-7 absolute on every score gradient; zero outside the candidates."""
    from torch.distributions.utils import clamp_probs

    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, E = 48, 10
    cfg = {"num_executors": E, "job_arrival_cap": 10, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    env.set_decima_weights(weights())
    env.reset_host(np.arange(B, dtype=np.uint64) + 77)
    g = torch.Generator(device="cuda").manual_seed(5)
    for k in range(30):
        a, n = env.decima_policy()
        if k in (0, 12, 29):
            g_lp = torch.randn(B, device="cuda", generator=g)
            g_en = torch.randn(B, device="cuda", generator=g)
            gs, ge = env.decima_head_adjoint(g_lp, g_en)
            act = env.pol_action.cpu().numpy()
            caps = env.dec_commit_caps.cpu().numpy()
            hdr = env.hdr()
            for b in range(B):
                n_cand, job, N = int(act[b, 3]), int(act[b, 1]), int(hdr["num_nodes"][b])
                if n_cand <= 0:
                    assert not gs[b].any() and not ge[b].any()
                    continue
                cap = int(caps[b, job])
                zs = env.pol_stage_logits[b, :n_cand].clone().requires_grad_()
                ze = env.pol_exec_logits[b, :cap].clone().requires_grad_()
                lg = en = 0.0
                for z, sel in ((zs, int(act[b, 0])), (ze, int(act[b, 2]))):
                    q = clamp_probs(torch.softmax(z, 0))
                    lg = lg + q.log()[sel]
                    en = en - (q.log() * q).sum()
                en = en / torch.log(torch.tensor(float(E * N), device="cuda"))
                (g_lp[b] * lg + g_en[b] * en).backward()
                assert torch.allclose(gs[b, :n_cand], zs.grad, rtol=1e-5, atol=1e-7), (k, b)
                assert torch.allclose(ge[b, :cap], ze.grad, rtol=1e-5, atol=1e-7), (k, b)
                assert not gs[b, n_cand:].any() and not ge[b, cap:].any()
        env.step(a, n)


def test_head_mlp_backward_matches_torch_autograd(bank):
    """ssb_decima_head_backward (backward of the stage / executor-count score MLPs on the candidates' rows) vs torch
    autograd through the same MLPs in fp32 on the gathered input rows the kernel reports.  The upstream gradient of a
    score is a function of the score itself (sin(3 s)), so no row order has to be assumed: the recomputed scores
    equal the device's as a multiset (1e-5); d loss / d input rows, weight and bias gradients agree within 2e-4 of
    each tensor's largest entry (the tcgen05 and torch scores differ by ~1e-6, fp32 atomics over ~1e3 rows)."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, E = 48, 10
    cfg = {"num_executors": E, "job_arrival_cap": 10, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    w = weights()
    env.set_decima_weights(w)
    env.reset_host(np.arange(B, dtype=np.uint64) + 91)
    keys = list(w.keys())
    flat_off = np.concatenate([[0], np.cumsum([w[k].size for k in keys])])
    for k in range(25):
        a, n = env.decima_policy()
        if k in (3, 24):
            gs = torch.sin(3.0 * env.pol_stage_logits)
            ge = torch.sin(3.0 * env.pol_exec_logits)
            gw = torch.zeros(20802, device="cuda")
            dxs, dxe, xs, xe = env.decima_head_backward(gs, ge, gw, want_inputs=True)
            act = env.pol_action.cpu().numpy()
            caps = env.dec_commit_caps.cpu().numpy()
            dev_scores = {
                "stage": torch.cat([env.pol_stage_logits[b, :act[b, 3]] for b in range(B)]),
                "exec": torch.cat([env.pol_exec_logits[b, :caps[b, act[b, 1]]] for b in range(B) if act[b, 1] >= 0])}
            for first, X, dX, in_dim, mode in ((30, xs, dxs, 53, "stage"), (36, xe, dxe, 36, "exec")):
                Ws = [torch.from_numpy(w[keys[first + i]]).cuda().requires_grad_() for i in range(6)]
                Xt = X[:, :in_dim].clone().requires_grad_()
                h = torch.tanh(Xt @ Ws[0].T + Ws[1])
                h = torch.tanh(h @ Ws[2].T + Ws[3])
                out = (h @ Ws[4].T + Ws[5]).squeeze(1)
                assert out.numel() == dev_scores[mode].numel() > 0
                assert torch.allclose(torch.sort(out.detach())[0], torch.sort(dev_scores[mode])[0], rtol=1e-5, atol=1e-5)
                (out * torch.sin(3.0 * out.detach())).sum().backward()
                # (the two sides' scores differ by ~1e-6, and so do their sin(3 s): compare against the largest entry)
                tol = 2e-4 * float(Xt.grad.abs().max()) + 1e-6
                assert float((dX[:, :in_dim] - Xt.grad).abs().max()) <= tol, (k, mode)
                assert not dX[:, in_dim:].any()
                for i in range(6):
                    got = gw[flat_off[first + i]:flat_off[first + i + 1]].view(Ws[i].shape)
                    tol = 2e-4 * float(Ws[i].grad.abs().max()) + 3e-6
                    assert float((got - Ws[i].grad).abs().max()) <= tol, (k, mode, keys[first + i])
        env.step(a, n)


def test_backward_down_to_node_embeddings_matches_torch_autograd(bank):
    """ssb_decima_backward vs torch autograd through everything above NodeEncoder, all envs in one batch
    (oracle/decima_torch.py in float32): node embeddings h (the restatement's own, a leaf) -> DagEncoder ->
    GlobalEncoder -> stage / executor-count heads -> utils.evaluate -> loss = sum_b c1_b lgprob_b + c2_b entropy_b.
    Compared: d loss / d h per env and the summed gradients of the four MLPs' 24 tensors, each within 3e-4 of its
    largest entry (device h vs reference h differ by ~1e-6; fp32 atomics)."""
    import decima_torch

    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, E = 24, 10
    cfg = {"num_executors": E, "job_arrival_cap": 8, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    w = weights()
    env.set_decima_weights(w)
    env.reset_host(np.arange(B, dtype=np.uint64) + 301)
    keys = list(w.keys())
    flat_off = np.concatenate([[0], np.cumsum([w[k].size for k in keys])])
    g = torch.Generator(device="cuda").manual_seed(3)
    for k in range(22):
        a, n = env.decima_policy()
        if k in (2, 21):
            c1 = torch.randn(B, device="cuda", generator=g)
            c2 = torch.randn(B, device="cuda", generator=g)
            gw = torch.zeros(20802, device="cuda")
            d_h = env.decima_backward(c1, c2, gw, through_node_encoder=False).cpu()
            assert not gw[:flat_off[18]].any()  # NodeEncoder's tensors: not part of this stage
            hdr = env.hdr().copy()
            env.decima_obs()
            obs = {key: t.cpu() for key, t in decima_torch.handle_observation(env, hdr).items()}
            Wt = decima_torch.weights(w, torch.float32)
            with torch.no_grad():
                h = decima_torch.encode_nodes(Wt, obs)
            h.requires_grad_()
            out = decima_torch.evaluate_actions(Wt, obs, c1.cpu(), c2.cpu(), h=h, num_executors=E)
            out["loss"].backward()
            for b in range(B):
                if hdr["terminated"][b]:
                    continue
                N = int(hdr["num_nodes"][b])
                tol = 3e-4 * float(h.grad[b].abs().max()) + 3e-6
                assert float((d_h[b, :N] - h.grad[b, :N]).abs().max()) <= tol, (k, b)
                assert not d_h[b, N:].any()
            for i in range(18, 42):
                want = Wt[keys[i]].grad
                got = gw[flat_off[i]:flat_off[i + 1]].view(want.shape).cpu()
                tol = 3e-4 * float(want.abs().max()) + 3e-6  # (a last-layer bias gradient is a sum that cancels to ~0: pure rounding)
                assert float((got - want).abs().max()) <= tol, (k, keys[i])
        env.step(a, n)


def test_full_backward_matches_torch_autograd(bank):
    """ssb_decima_backward(through_node_encoder=True): the gradients of all 42 tensors of the shipped model for
    loss = sum_b c1_b lgprob_b + c2_b entropy_b, against torch autograd through oracle/decima_torch.py (the whole
    policy over all envs in one batch: NodeEncoder with its level loop, DagEncoder, GlobalEncoder, both heads,
    utils.evaluate) in float32.  Every tensor within 5e-4 of its largest entry (fp32 atomics; bf16x3 forward vs fp32)."""
    import decima_torch

    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, E = 24, 10
    cfg = {"num_executors": E, "job_arrival_cap": 8, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    w = weights()
    env.set_decima_weights(w)
    env.reset_host(np.arange(B, dtype=np.uint64) + 501)
    keys = list(w.keys())
    flat_off = np.concatenate([[0], np.cumsum([w[k].size for k in keys])])
    g = torch.Generator(device="cuda").manual_seed(9)
    for k in range(22):
        a, n = env.decima_policy()
        if k in (0, 5, 21):
            c1 = torch.randn(B, device="cuda", generator=g)
            c2 = torch.randn(B, device="cuda", generator=g)
            hdr = env.hdr().copy()
            env.decima_obs()
            obs = {key: t.cpu().clone() for key, t in decima_torch.handle_observation(env, hdr).items()}
            gw = torch.zeros(20802, device="cuda")
            env.decima_backward(c1, c2, gw)
            Wt = decima_torch.weights(w, torch.float32)
            decima_torch.evaluate_actions(Wt, obs, c1.cpu(), c2.cpu(), num_executors=E)["loss"].backward()
            if k == 21:
                assert int(obs["depth"][obs["live"]].max()) >= 2  # the level loop was exercised
            for i in range(42):
                want = Wt[keys[i]].grad
                got = gw[flat_off[i]:flat_off[i + 1]].view(want.shape).cpu()
                tol = 5e-4 * float(want.abs().max()) + 3e-6
                assert float((got - want).abs().max()) <= tol, (k, keys[i], float((got - want).abs().max()), tol)
            # the backward pass overwrote the intermediate buffers: the next policy call recomputes everything
        env.step(a, n)


def test_ppo_minibatch_update_on_stored_snapshots(bank):
    """The pieces of PPO._train (trainers/ppo.py:72-102) strung together on the device over stored observations:
    snapshot load -> evaluate -> clip loss -> backward -> clip_grad_norm_ + Adam -> new weights.  Checked: the
    evaluation inside the update reproduces the rollout's lgprobs (ratio 1: approx KL 0, policy loss = -mean of the
    normalised advantages = 0), the gradient of a stored observation equals the gradient of the same observation
    when it was live, the live observation survives the update, repeated updates raise the surrogate objective,
    and the KL early stop skips the step."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv
    from spark_sched_sim_b200.ppo import Adam, PPOLoss, ppo_minibatch_update

    B = 32
    cfg = {"num_executors": 10, "job_arrival_cap": 8, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    w = weights()
    env.set_decima_weights(w)
    env.reset_host(np.arange(B, dtype=np.uint64) + 700)
    g = torch.Generator(device="cuda").manual_seed(1)
    snaps, acts, lgs = [], [], []
    live_grad = None
    for k in range(12):
        snaps.append(env.decima_snapshot())
        a, n = env.decima_policy()
        acts.append(env.pol_action.clone()); lgs.append(env.pol_lgprob.clone())
        if k == 6:  # gradient of this observation while it is the live one
            c1 = torch.randn(B, device="cuda", generator=g); c2 = torch.randn(B, device="cuda", generator=g)
            live_grad = torch.zeros(20802, device="cuda")
            env.decima_backward(c1, c2, live_grad)
        env.step(a, n)
    wall = env.hdr()["wall_time"].copy()
    # the same gradient from the stored observation, many decisions later
    env.decima_snapshot_load(snaps[6])
    lg, _ = env.decima_evaluate(None, acts[6][:, 0].contiguous(), acts[6][:, 2].contiguous())
    assert torch.equal(lg, lgs[6])
    stored_grad = torch.zeros(20802, device="cuda")
    env.decima_backward(c1, c2, stored_grad)
    env.decima_snapshot_unload()
    assert float((stored_grad - live_grad).abs().max()) <= 1e-4 * float(live_grad.abs().max())  # atomics' order only
    # PPO updates on one mini-batch
    flat = torch.from_numpy(np.concatenate([w[k].astype(np.float32).reshape(-1) for k in w])).cuda()
    adam = Adam(flat.clone(), lr=3e-4, max_grad_norm=0.5)
    loss_fn = PPOLoss(0.2, 0.04)
    ret = -1e4 * torch.rand(B, device="cuda", generator=g, dtype=torch.float64)
    base = ret + 2e3 * torch.randn(B, device="cuda", generator=g, dtype=torch.float64)
    k = 4
    args = (snaps[k], acts[k][:, 0].contiguous(), acts[k][:, 2].contiguous(), lgs[k], ret, base, loss_fn, adam)
    info0, stepped = ppo_minibatch_update(env, *args)
    assert stepped and abs(info0["approx_kl_div"]) < 1e-6 and abs(info0["policy_loss"]) < 1e-5
    assert float(adam.grad_norm.item()) > 0 and not torch.equal(adam.params, flat)
    losses = [info0["loss"]]
    for _ in range(5):
        info, stepped = ppo_minibatch_update(env, *args)
        assert stepped
        losses.append(info["loss"])
    assert losses[-1] < losses[0] - 1e-4, losses  # the surrogate loss goes down on the batch it is trained on
    _, stepped = ppo_minibatch_update(env, *args, target_kl=0.0)
    assert not stepped  # approx KL > 0 after six updates: early stop
    # PPO._train over several stored mini-batches: epochs, shuffled order, summary dict, early stop
    from spark_sched_sim_b200.ppo import ppo_train

    batches = [(snaps[j], acts[j][:, 0].contiguous(), acts[j][:, 2].contiguous(), lgs[j], ret, base) for j in (1, 3, 5, 8)]
    env.set_decima_weights(w)  # back to the rollout's policy, so that the first pass has ratio 1
    adam2 = Adam(flat.clone(), lr=3e-4, max_grad_norm=0.5)
    summary = ppo_train(env, batches, loss_fn, adam2, num_epochs=2, target_kl=None,
                        generator=torch.Generator().manual_seed(0))
    assert summary["num_updates"] == 8 and summary["entropy"] > 0 and np.isfinite(summary["policy loss"])
    summary = ppo_train(env, batches, loss_fn, adam2, num_epochs=2, target_kl=1e-9,
                        generator=torch.Generator().manual_seed(0))
    assert summary["num_updates"] == 0 and summary["approx kl div"] > 1.5e-9  # stopped on the first mini-batch
    assert np.array_equal(env.hdr()["wall_time"], wall)  # the live observation came back
    a, n = env.decima_policy()
    env.step(a, n)
    assert (env.hdr()["error"] == 0).all()


def _mlp_fp(x, w, name, tanh, dtype):
    """make_mlp (schedulers/decima/utils.py:45-64) in numpy at the given precision."""
    x = x.astype(dtype)
    for i, k in enumerate((0, 2, 4)):
        x = x @ w[f"{name}.{k}.weight"].astype(dtype).T + w[f"{name}.{k}.bias"].astype(dtype)
        if i < 2:
            x = np.tanh(x) if tanh else np.where(x > 0, x, dtype(0.2) * x)
        x = x.astype(dtype)
    return x


@pytest.mark.parametrize("mlp", range(7))
def test_mlp_rows_accuracy_against_fp64(bank, mlp):
    """Each of the policy's seven MLPs on the tensor-core path (bf16 three-term split, activations in TMEM) against an
    fp64 evaluation of the same weights: the error must be of the size of float32 arithmetic itself -- no larger than
    3x what torch's own float32 forward makes against fp64 on the same rows (plus 2e-7 of the output scale)."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    cfg = {"num_executors": 10, "job_arrival_cap": 4, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    env = BatchedSparkSchedSimEnv(cfg, num_envs=2, bank=bank, decima_policy=True)
    w = weights()
    env.set_decima_weights(w)
    name, (din, dout) = env.MLP_NAMES[mlp], env.MLP_DIMS[mlp]
    rng = np.random.default_rng(100 + mlp)
    n = 1000  # not a multiple of 128: the last tile is ragged
    x = (rng.standard_normal((n, din)) * rng.choice([0.05, 1.0, 4.0], size=(n, 1))).astype(np.float32)
    x[0] = 0.0
    got = env.decima_mlp_rows(mlp, torch.from_numpy(x).cuda()).cpu().numpy().astype(np.float64)
    truth = _mlp_fp(x, w, name, mlp >= 5, np.float64)
    with torch.no_grad():
        t = torch.from_numpy(x)
        for i, k in enumerate((0, 2, 4)):
            t = torch.nn.functional.linear(t, torch.from_numpy(w[f"{name}.{k}.weight"]), torch.from_numpy(w[f"{name}.{k}.bias"]))
            if i < 2:
                t = torch.tanh(t) if mlp >= 5 else torch.nn.functional.leaky_relu(t, 0.2)
        ref32 = t.numpy().astype(np.float64)
    scale = np.abs(truth).max()
    err_ours, err_torch = np.abs(got - truth).max(), np.abs(ref32 - truth).max()
    print(f"mlp {mlp} {name}: scale {scale:.3g}  ours-vs-fp64 {err_ours:.3g}  torch32-vs-fp64 {err_torch:.3g}")
    assert got.shape == (n, dout)
    assert err_ours <= 3.0 * err_torch + 2e-7 * scale, (err_ours, err_torch, scale)


def test_decima_async_rollouts_match_the_workers_loop(bank):
    """ssb_rollout_decima_async == RolloutWorkerAsync.collect_rollout (rollout_worker.py:160-206) with the Decima policy:
    the worker's loop is restated in Python over single-environment handles ({ decima_policy ; step }, reset with
    seed + seed_step * reset_count when an episode ends, time axis = accumulated time, state carried over between
    calls); the Philox policy stream makes the sampled actions reproducible, so every row must agree exactly."""
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, KMAX, DUR, STEP = 5, 700, 1.5e6, 11
    cfg = {"num_executors": 10, "job_arrival_cap": 4, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    seeds = np.arange(B, dtype=np.uint64) + 60
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
    env.set_decima_weights(weights())
    env.reset_host(seeds)
    calls = []
    for _ in range(3):
        traj, num, el = env.rollout_decima_async(KMAX, DUR, STEP)
        calls.append((traj.cpu().numpy().view(nat.TRANSITION_DTYPE).reshape(B, KMAX), num.cpu().numpy(), el.cpu().numpy()))
    assert (env.hdr()["error"] == 0).all()
    n_resets = 0
    for b in range(B):
        one = BatchedSparkSchedSimEnv(cfg, num_envs=1, bank=bank, decima_policy=True)
        one.set_decima_weights(weights())
        hdr = one.reset_host(seeds[b:b + 1]).copy()
        resets, next_wall = 1, 0.0
        for tr, num, el in calls:  # one collect_rollout() each
            elapsed, step = 0.0, 0
            while elapsed < DUR and step < KMAX:
                wall = next_wall
                a, n = one.decima_policy()
                lg = float(one.pol_lgprob[0].item())
                one.step(a, n)
                h = one.hdr()[0]
                assert h["error"] == 0
                next_wall = float(h["wall_time"])
                r = tr[b, step]
                assert (r["wall_time"], r["stage_idx"], r["num_exec"], r["reward"]) == (elapsed, int(a[0]), int(n[0]), h["reward"]), (b, step)
                assert r["lgprob"] == np.float32(lg) and (r["flags"] & 1) == int(h["terminated"]), (b, step)
                elapsed += next_wall - wall
                if h["terminated"]:
                    one.reset_host(np.array([int(seeds[b]) + STEP * resets], np.uint64)); resets += 1
                    next_wall = 0.0
                    n_resets += 1
                    if step + 1 < num[b]:
                        assert tr[b, step + 1]["flags"] & 4  # the next row is the first of the new episode
                step += 1
            assert num[b] == step and el[b] == elapsed, (b, num[b], step, el[b], elapsed)
    assert n_resets >= B


@pytest.mark.parametrize("fixture", ["decima_grads_e10_j8_s5", "decima_grads_e50_j14_s4"])
@pytest.mark.parametrize("mode,for_backward", [(None, False), ("0", False), ("0", True)],
                         ids=["fused-replay", "tiles-replay", "tiles-saved-by-evaluate"])
def test_backward_matches_the_reference_models_gradients(fixture, mode, for_backward, monkeypatch):
    """(mode: the policy's execution mode for this small batch -- default = the fused kernel, "0" = the list-driven tile
    kernels; for_backward: the evaluation leaves the levels' input rows in the attached scratch and the backward pass
    does not replay them.)
    ssb_decima_evaluate + ssb_decima_backward against gradients recorded from the UNMODIFIED reference
    DecimaScheduler (tests/golden/gen_decima_grad_golden.py: its own evaluate_actions, scheduler.py:101-139, and
    loss.backward() on a batch of observations of a recorded episode).  Env i replays the episode up to observation
    picks[i] and stops there; one evaluate / backward over the B live observations must reproduce the reference's
    lgprobs, entropies and all 42 parameter gradients (each tensor within 5e-4 of its largest entry: fp32 atomics)."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    if mode is not None:
        monkeypatch.setenv("SSB_DECIMA_MODE", mode)
    g = np.load(osp.join(GOLDEN_DIR, fixture + ".npz"))
    tr = load_golden(str(g["trace"]))
    picks = [int(k) for k in g["picks"]]
    B = len(picks)
    env = BatchedSparkSchedSimEnv(env_cfg_of(tr), num_envs=B, bank=bank_for(tr), max_jobs=len(tr["job_template"]) + 2,
                                  tape_capacity=len(tr["tape"]) + 8, decima_policy=True)
    assert [str(x) for x in g["param_order"]] == list(env.DECIMA_PARAM_ORDER)  # the ABI's flat order == state_dict order
    env.set_decima_weights(weights())
    for b in range(B):
        env.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    env.reset_host(np.full(B, tr["seed"], np.uint64))
    for k in range(max(picks)):
        a, n = tr["actions"][k]
        mask = np.array([k < picks[i] for i in range(B)], np.uint8)  # env i stops AT observation picks[i]
        hdr = env.step_host(np.full(B, a, np.int32), np.full(B, n, np.int32), mask=mask)
        assert (hdr["error"] == 0).all(), k
    hdr = env.hdr()
    assert [int(x) for x in hdr["num_nodes"]] == [int(tr["N"][k]) for k in picks]
    stage_sel = torch.tensor([int(tr["pol_actions"][k][0]) for k in picks], dtype=torch.int32, device="cuda")
    exec_sel = torch.tensor([int(tr["pol_actions"][k][2]) for k in picks], dtype=torch.int32, device="cuda")
    snap = env.decima_snapshot()
    env.decima_snapshot_load(snap)
    lg, en = env.decima_evaluate(None, stage_sel, exec_sel, for_backward=for_backward)
    assert np.abs(lg.cpu().numpy() - g["lgprobs"]).max() < 2e-5
    assert np.abs(en.cpu().numpy() - g["entropies"]).max() < 2e-5
    grads = torch.zeros(20802, dtype=torch.float32, device="cuda")
    env.decima_backward(torch.from_numpy(g["coef_lgprob"]).cuda(), torch.from_numpy(g["coef_entropy"]).cuda(), grads)
    env.decima_snapshot_unload()
    got, want = grads.cpu().numpy(), g["grad"]
    w = weights()
    off = 0
    for name in env.DECIMA_PARAM_ORDER:
        n = w[name].size
        a, b = got[off:off + n], want[off:off + n]
        tol = 5e-4 * float(np.abs(b).max()) + 3e-6
        assert np.abs(a - b).max() <= tol, (name, float(np.abs(a - b).max()), tol)
        off += n
    assert off == 20802 and np.abs(want).max() > 1.0


def test_decima_rollouts_at_config3_shape_are_deterministic(bank):
    """config/decima_tpch.yaml's env (200 jobs x 50 executors, mean time limit 2e7 ms) with the sampled Decima policy
    on 512 envs: two handles with the same seeds produce identical transitions (Philox policy stream), seed twins
    inside a handle differ only through their sampling streams' keys (= they are identical: same seed), no env
    errors, and the list-driven and the fused policy paths agree bit for bit."""
    import os

    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B, K = 512, 40
    cfg = {"num_executors": 50, "job_arrival_cap": 200, "job_arrival_rate": 4.0e-5,
           "moving_delay": 2000.0, "warmup_delay": 1000.0}
    seeds = (77 + np.arange(B) // 2).astype(np.uint64)
    outs = []
    try:
        for mode in ("0", "1", "0"):
            os.environ["SSB_DECIMA_MODE"] = mode
            env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True)
            env.set_decima_weights(weights())
            env.set_mean_time_limit(2.0e7)
            env.set_autoreset(True, B)
            env.reset_host(seeds)
            env.rollout_fair(300, True, True, B)  # into the episodes
            host = torch.empty(B * K * nat.TRANSITION_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
            tr = env.rollout_decima(K, host=host).copy()
            hdr = env.hdr()
            assert ((hdr["error"] == 0) | (hdr["error"] == 9)).all()
            outs.append(tr)
            env.close()
    finally:
        os.environ.pop("SSB_DECIMA_MODE", None)
    for f in ("wall_time", "reward", "stage_idx", "num_exec", "flags", "lgprob"):
        assert np.array_equal(outs[0][f], outs[1][f]), f   # list-driven == fused
        assert np.array_equal(outs[0][f], outs[2][f]), f   # deterministic
        assert np.array_equal(outs[0][f][0::2], outs[0][f][1::2]), f  # seed twins
    assert (outs[0]["stage_idx"] >= 0).mean() > 0.5
