"""Decima training rollouts on the device: per-env policy sampling streams (ssb_set_policy_streams) so that the members
of a rollout group share a job sequence but not their actions, the stored observations the fused Decima rollouts write
into an attached store (ssb_decima_attach_rollout_store, RolloutStore.collect_fused), and one trainer iteration on
such a store (ppo.train_iteration)."""
import os.path as osp

import numpy as np
import pytest
import torch

from helpers import GOLDEN_DIR, load_golden
from philox_ref import philox4x32_10

pytestmark = pytest.mark.gpu

CFG = {"num_executors": 10, "job_arrival_cap": 4, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0,
       "warmup_delay": 1000.0}
MODES = {"tiles": "0", "fused": "1"}


def _weights():
    z = np.load(osp.join(GOLDEN_DIR, "decima_model.npz"))
    return {k: z[k] for k in z.files}


def _env(bank, B, cfg=CFG, mode=None, monkeypatch=None, **kw):
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    if mode is not None:
        monkeypatch.setenv("SSB_DECIMA_MODE", mode)  # read when the handle is created
    env = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=bank, decima_policy=True, **kw)
    if mode is not None:
        monkeypatch.delenv("SSB_DECIMA_MODE")
    env.set_decima_weights(_weights())
    return env


def _env_cfg_of(tr):
    return {k: tr[k] for k in ("num_executors", "job_arrival_cap", "job_arrival_rate", "moving_delay", "warmup_delay",
                               "beta")}


def _rows(traj, B, K):
    from spark_sched_sim_b200 import _native as nat

    return traj.cpu().numpy().view(nat.TRANSITION_DTYPE).reshape(B, K)


def _u24(w):
    """((float)(w >> 8) + 0.5f) * 2^-24 in float32, as the sampling kernels compute it."""
    return float(np.float32(np.float32(w >> 8) + np.float32(0.5)) * np.float32(1.0 / 16777216.0))


def _inverse_cdf(logits, u):
    """float64 inverse-CDF index of softmax(logits) at u; None when u lies within 1e-6 of a CDF boundary."""
    z = np.asarray(logits, np.float64)
    p = np.exp(z - z.max())
    cdf = np.cumsum(p / p.sum())
    if np.abs(cdf[:-1] - u).min(initial=1.0) < 1e-6:
        return None
    return min(int(np.searchsorted(cdf, u, side="right")), len(z) - 1)


def _slot_bytes(env, block, i):
    """The rows in use of slot i of a snapshot block (ssb_decima_snapshot format of `env`) as bytes per part.  The
    header's was_reset is cleared: an episode started by a rollout's own reset carries it, one started by reset_host
    does not."""
    from spark_sched_sim_b200 import _native as nat

    B, S, M, J = env.num_envs, env.node_stride, env.edge_stride, env.job_stride
    stride = [nat.OBS_HDR_DTYPE.itemsize, M * 8, (J + 1) * 4, S * 20, S, J * 4, M * 8, 4]
    blk = block.cpu().numpy() if isinstance(block, torch.Tensor) else block
    off, parts = 0, []
    for s in stride:
        parts.append(blk[off + i * s: off + (i + 1) * s])
        off += (B * s + 255) & ~255
    parts[0] = parts[0].copy()
    h = parts[0].view(nat.OBS_HDR_DTYPE)[0]
    h["was_reset"] = 0
    N, E, Ja = int(h["num_nodes"]), int(h["num_edges"]), int(h["num_active_jobs"])
    used = [48, E * 8, (Ja + 1) * 4, N * 20, N, Ja * 4, E * 8, 4]
    return [p[:n].tobytes() for p, n in zip(parts, used)]


def _gather_all(env, store, pairs):
    """Gathers the stored observations of the samples `pairs` ((k, b) ...) into zero-filled staging blocks, B at a time;
    yields ((k, b), slot index, block as numpy uint8)."""
    B, dev = env.num_envs, env.device
    nb = env.decima_snapshot_bytes()
    for c in range(0, len(pairs), B):
        chunk = pairs[c:c + B]
        ks = torch.full((B,), -1, dtype=torch.int32, device=dev)
        bs = torch.zeros(B, dtype=torch.int32, device=dev)
        ks[:len(chunk)] = torch.tensor([k for k, _ in chunk], dtype=torch.int32)
        bs[:len(chunk)] = torch.tensor([b for _, b in chunk], dtype=torch.int32)
        staging = torch.zeros(nb, dtype=torch.uint8, device=dev)
        env.decima_snapshot_gather(store.snapshots, ks, bs, out=staging)
        yield chunk, ks, bs, staging


# ---------------------------------------------------------------------------------------------------- default unchanged
@pytest.mark.parametrize("mode", list(MODES))
def test_all_zero_streams_leave_the_rollouts_unchanged(bank, mode, monkeypatch):
    """Streams set explicitly to zero give rows byte-equal to a handle that never called the setter, in the sync and
    the async Decima rollout, in every policy execution mode."""
    B, K = 12, 120
    seeds = np.arange(B, dtype=np.uint64) + 300
    out = []
    for explicit in (False, True):
        env = _env(bank, B, mode=MODES[mode], monkeypatch=monkeypatch)
        if explicit:
            env.set_policy_streams(np.zeros(B, np.uint32))
        env.set_autoreset(True, 5)
        env.reset_host(seeds)
        sync = env.rollout_decima(K).cpu().numpy()
        env.reset_host(seeds)
        traj, num, el = env.rollout_decima_async(K, 1.0e6, seed_step=5)
        out.append((sync, traj.cpu().numpy(), num.cpu().numpy(), el.cpu().numpy()))
    for a, b in zip(*out):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------- counter formula
def test_stream_is_the_second_counter_word(bank):
    """B envs in one state (same trace, tape and seed), streams 0..B-1: every env's sampled stage is the float64
    inverse-CDF index of its scores at u drawn from Philox ctr (draws, b, 4, 0), and the executor count likewise from
    the same counter's second word; over the envs the stage frequencies follow the softmax."""
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    tr = load_golden("decima_e10_j8_s5_philox")
    B, seed = 2048, 91
    env = BatchedSparkSchedSimEnv(_env_cfg_of(tr), num_envs=B, bank=bank, max_jobs=10,
                                  tape_capacity=len(tr["tape"]) + 8, decima_policy=True)
    env.set_decima_weights(_weights())
    for b in range(B):
        env.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    env.set_policy_streams(np.arange(B, dtype=np.uint32))
    env.reset_host(np.full(B, seed, np.uint64))
    key = (seed & 0xFFFFFFFF, seed >> 32)
    checked = freq_checked = skipped = 0
    host_b = list(range(0, B, 16))
    for k in range(40):
        stage_idx, _, num_exec = (int(x) for x in tr["pol_actions"][k])
        ns = int(tr["pol_stage_count"][k])
        env.decima_policy()  # sampled, draw 2k of the episode (the forced call below is draw 2k + 1)
        acts = env.pol_action.cpu().numpy()
        logits = env.pol_stage_logits[:, :ns].cpu().numpy()
        exec_logits = env.pol_exec_logits.cpu().numpy()
        caps = env.dec_commit_caps.cpu().numpy()
        for b in host_b:
            if acts[b, 3] == 0:
                continue
            w = philox4x32_10((2 * k, b, 4, 0), key)
            want = _inverse_cdf(logits[b, :acts[b, 3]], _u24(w[0]))
            if want is None:
                skipped += 1
                continue
            assert acts[b, 0] == want, (k, b, acts[b], want)
            cap = int(caps[b, acts[b, 1]])
            want_n = _inverse_cdf(exec_logits[b, :cap], _u24(w[1])) if cap > 0 else None
            if want_n is not None:
                assert acts[b, 2] == want_n, (k, b, acts[b], want_n)
            checked += 1
        if ns >= 3 and freq_checked < 4:
            s = logits[0].astype(np.float64)
            p = np.exp(s - s.max())
            p /= p.sum()
            freq = np.bincount(acts[:, 0], minlength=ns) / B
            assert np.abs(freq - p).max() < 0.05, (k, freq, p)
            freq_checked += 1
        a, n = env.decima_policy(forced_stage=np.full(B, stage_idx, np.int32),
                                 forced_num_exec=np.full(B, num_exec, np.int32))
        env.step(a, n)
    assert checked > 1000 and skipped < checked // 20 and freq_checked >= 2


# ---------------------------------------------------------------------------------------------------- persistence
def test_streams_persist_through_resets(bank):
    """A one-env handle with stream r reproduces env b (stream r) of a batch exactly: through the auto-resets of the
    sync rollout, the in-rollout resets of the async one, and a reset_host(grow=True) that re-creates the handle."""
    B, K, STEP = 4, 250, 7
    seeds = np.array([40, 41, 40, 43], np.uint64)
    streams = np.array([3, 0, 11, 5], np.uint32)
    env = _env(bank, B)
    env.set_policy_streams(streams)
    env.set_autoreset(True, STEP)
    env.reset_host(seeds)
    sync = _rows(env.rollout_decima(K), B, K)
    env.reset_host(seeds)  # (a reset keeps the streams)
    calls = [env.rollout_decima_async(K, 1.0e6, seed_step=STEP) for _ in range(2)]
    assert (sync["flags"] & 8).any() and (sync["flags"] & 4).any()
    assert any((_rows(t, B, K)["flags"] & 4).any() for t, _, _ in calls)
    assert not np.array_equal(sync[0], sync[2])  # same seed, other stream
    for b in range(B):
        one = _env(bank, 1)
        one.set_policy_streams(streams[b:b + 1])
        one.set_autoreset(True, STEP)
        one.reset_host(seeds[b:b + 1])
        assert one.rollout_decima(K).cpu().numpy().tobytes() == sync[b].tobytes(), b
        one.reset_host(seeds[b:b + 1])
        for traj, num, el in calls:
            t1, n1, e1 = one.rollout_decima_async(K, 1.0e6, seed_step=STEP)
            assert int(n1[0]) == int(num[b]) and float(e1[0]) == float(el[b]), b
            assert t1.cpu().numpy().tobytes() == _rows(traj, B, K)[b].tobytes(), b
    # time-limited arrivals without a job cap: the small handle grows at its reset and keeps its streams
    cfg = {k: v for k, v in CFG.items() if k != "job_arrival_cap"}
    big = _env(bank, B, cfg=cfg, max_jobs=256)
    big.set_mean_time_limit(4.0e5)
    big.set_policy_streams(streams)
    big.reset_host(seeds)
    rows = _rows(big.rollout_decima(60), B, 60)
    for b in range(B):
        one = _env(bank, 1, cfg=cfg, max_jobs=2)
        one.set_mean_time_limit(4.0e5)
        one.set_policy_streams(streams[b:b + 1])
        one.reset_host(seeds[b:b + 1], grow=True)
        assert one.max_jobs > 2 and one.hdr()["error"][0] == 0
        assert one.rollout_decima(60).cpu().numpy().tobytes() == rows[b].tobytes(), b


# ---------------------------------------------------------------------------------------------------- groups
def test_rollout_groups_share_arrivals_not_actions(bank):
    """rollout_groups(4, 4): the members of a group play the same job sequence with their own actions, so the group
    baseline differs from the returns and the advantages are not all zero."""
    from spark_sched_sim_b200 import ppo
    from spark_sched_sim_b200.returns import Baseline, ReturnsCalculator

    seeds, streams, seed_step = ppo.rollout_groups(4, 4, 1000)
    assert seed_step == 4 and seeds.tolist() == [1000 + i // 4 for i in range(16)]
    assert streams.tolist() == [i % 4 for i in range(16)]
    s1, st1, _ = ppo.rollout_groups(4, 4, 1000, rank=1, world=2)
    assert s1.tolist() == seeds[8:].tolist() and st1.tolist() == streams[8:].tolist()
    with pytest.raises(AssertionError):
        ppo.rollout_groups(3, 4, 1000, rank=0, world=2)  # 6 envs per rank: not whole groups
    B, K = 16, 80
    env = _env(bank, B)
    env.set_policy_streams(streams)
    env.reset_host(seeds)
    store = ppo.RolloutStore(env, K).collect_fused()
    for g in range(4):
        jobs = [env.jobs(4 * g + r) for r in range(4)]
        for r in range(1, 4):
            assert np.array_equal(jobs[r][0], jobs[0][0]) and np.array_equal(jobs[r][2], jobs[0][2]), (g, r)
        sel = store.stage_sel[:, 4 * g:4 * g + 4].cpu().numpy(), store.exec_sel[:, 4 * g:4 * g + 4].cpu().numpy()
        assert any(not np.array_equal(x[:, 0], x[:, r]) for x in sel for r in range(1, 4)), g
    ret = ReturnsCalculator(beta=5e-3)(store.traj, store.num_steps, store.final_wall, K)
    base = Baseline(4, 4)(store.traj, ret, store.num_steps)
    valid = store.valid.t()
    adv = (ret - base)[valid]
    assert adv.abs().max().item() > 1e-6


# ---------------------------------------------------------------------------------------------------- store vs loop
@pytest.mark.parametrize("mode", ["tiles", "fused"])
def test_fused_store_matches_the_step_by_step_collect(bank, mode, monkeypatch):
    """collect_fused (sync protocol, auto-reset off) against collect() on a twin handle: the same valid samples,
    actions and lgprobs, and every valid sample's stored observation gathers into a byte-equal block."""
    from spark_sched_sim_b200 import ppo

    B, K = 24, 160
    seeds = np.arange(B, dtype=np.uint64) + 500
    stores = []
    for fused in (True, False):
        env = _env(bank, B, mode=MODES[mode], monkeypatch=monkeypatch)
        env.reset_host(seeds)
        store = ppo.RolloutStore(env, K)
        stores.append((env, store.collect_fused() if fused else store.collect()))
    (ea, sa), (eb, sb) = stores
    valid = sa.valid.cpu().numpy()
    assert np.array_equal(valid, sb.valid.cpu().numpy())
    assert valid.any()
    for name in ("stage_sel", "exec_sel", "lgprob"):
        assert torch.equal(getattr(sa, name)[sa.valid], getattr(sb, name)[sb.valid]), name
    n = valid.sum(0)
    assert np.array_equal(sa.num_steps.cpu().numpy(), n)
    assert torch.equal(sa.wall_time[:K][sa.valid], sb.wall_time[:K][sb.valid])
    assert torch.equal(sa.reward[sa.valid], sb.reward[sb.valid])
    assert torch.equal(sa.final_wall, sb.wall_time[K])
    pairs = [(int(k), int(b)) for k, b in zip(*np.nonzero(valid))]
    ga, gb = _gather_all(ea, sa, pairs), _gather_all(eb, sb, pairs)
    for (chunk, _, _, blk_a), (_, _, _, blk_b) in zip(ga, gb):
        assert torch.equal(blk_a, blk_b), chunk[0]
    _reevaluate(ea, sa)


def test_fused_async_store_matches_the_workers_loop(bank):
    """collect_fused with a rollout duration against RolloutWorkerAsync.collect_rollout restated over one-env handles
    (decima_snapshot + policy + step per decision, re-seeded with seed + seed_step * resets), across three calls: the
    same rows, actions, lgprobs and stored observations."""
    from spark_sched_sim_b200 import ppo

    B, K, DUR, STEP = 3, 300, 1.5e6, 11
    seeds = np.arange(B, dtype=np.uint64) + 60
    streams = np.array([0, 2, 1], np.uint32)
    env = _env(bank, B)
    env.set_policy_streams(streams)
    env.reset_host(seeds)
    calls = []
    for _ in range(3):
        store = ppo.RolloutStore(env, K).collect_fused(rollout_duration=DUR, seed_step=STEP)
        pairs = [(int(k), int(b)) for k, b in zip(*np.nonzero(store.valid.cpu().numpy()))]
        slots = {}
        for chunk, _, _, blk in _gather_all(env, store, pairs):
            blk = blk.cpu().numpy()
            for i, kb in enumerate(chunk):
                slots[kb] = _slot_bytes(env, blk, i)
        calls.append((store.num_steps.cpu().numpy(), store.stage_sel.cpu().numpy(), store.exec_sel.cpu().numpy(),
                      store.lgprob.cpu().numpy(), slots))
    n_resets = 0
    for b in range(B):
        one = _env(bank, 1)
        one.set_policy_streams(streams[b:b + 1])
        one.reset_host(seeds[b:b + 1])
        resets, next_wall = 1, 0.0
        for num, ssel, esel, lgp, slots in calls:
            elapsed, step = 0.0, 0
            while elapsed < DUR and step < K:
                wall = next_wall
                snap = one.decima_snapshot()
                a, n = one.decima_policy()
                act = one.pol_action[0].cpu().numpy()
                assert (ssel[step, b], esel[step, b]) == (act[0], act[2]), (b, step)
                assert lgp[step, b] == np.float32(one.pol_lgprob[0].item()), (b, step)
                assert slots[(step, b)] == _slot_bytes(one, snap, 0), (b, step)
                one.step(a, n)
                h = one.hdr()[0]
                assert h["error"] == 0
                next_wall = float(h["wall_time"])
                elapsed += next_wall - wall
                if h["terminated"]:
                    one.reset_host(np.array([int(seeds[b]) + STEP * resets], np.uint64))
                    resets += 1
                    next_wall = 0.0
                    n_resets += 1
                step += 1
            assert num[b] == step, (b, num[b], step)
    assert n_resets >= B


def _reevaluate(env, store):
    """Every valid sample of the store re-evaluates (decima_evaluate on a gathered batch) to exactly its stored
    lgprob."""
    valid = store.valid.cpu().numpy()
    pairs = [(int(k), int(b)) for k, b in zip(*np.nonzero(valid))]
    for chunk, ks, bs, staging in _gather_all(env, store, pairs):
        kk, bb = ks.clamp(min=0).long(), bs.long()
        lg, _ = env.decima_evaluate(staging, store.stage_sel[kk, bb].contiguous(), store.exec_sel[kk, bb].contiguous())
        n = len(chunk)
        assert torch.equal(lg[:n], store.lgprob[kk[:n], bb[:n]]), chunk[0]


# ---------------------------------------------------------------------------------------------------- iteration
def test_train_iteration_on_a_group_rollout(bank):
    """train_iteration on a 64-env group rollout: the returns / baselines it trains on are ReturnsCalculator /
    Baseline on store.traj, a fixed generator makes it repeatable, the weights move, and the update count is
    epochs x mini-batches without a KL stop and stops early with one."""
    from spark_sched_sim_b200 import ppo
    from spark_sched_sim_b200.returns import Baseline, ReturnsCalculator

    S, R, K = 16, 4, 40
    seeds, streams, seed_step = ppo.rollout_groups(S, R, 77)
    env = _env(bank, S * R)
    env.set_policy_streams(streams)
    env.reset_host(seeds)
    store = ppo.RolloutStore(env, K).collect_fused(rollout_duration=2.0e6, seed_step=seed_step)
    _reevaluate(env, store)
    w0 = torch.from_numpy(np.concatenate([_weights()[k].reshape(-1) for k in env.DECIMA_PARAM_ORDER])).cuda()
    N = int(store.valid.sum().item())
    epochs, batches = 2, 3
    full = epochs * -(-N // (N // batches + 1))

    def run(target_kl):
        env.set_decima_weights(w0)
        adam = ppo.Adam(w0.clone(), lr=3e-4, max_grad_norm=0.5)
        g = torch.Generator().manual_seed(5)
        out = ppo.train_iteration(env, store, ReturnsCalculator(beta=5e-3), Baseline(S, R), ppo.PPOLoss(0.2, 0.01),
                                  adam, epochs, batches, target_kl, generator=g)
        return out, adam.params.clone()

    s1, w1 = run(None)
    ret = ReturnsCalculator(beta=5e-3)(store.traj, store.num_steps, store.final_wall, K)
    assert torch.equal(s1["returns"], ret)
    assert torch.equal(s1["baselines"], Baseline(S, R)(store.traj, ret, store.num_steps))
    assert s1["num_samples"] == N and s1["num_updates"] == full
    assert not torch.equal(w1, w0)
    assert set(s1["collect_stats"]) >= {"avg_num_jobs", "num_completed_jobs"}
    # (the weight gradients are float32 atomic sums, so a repeat is equal up to their rounding; Adam moves a weight by
    # at most ~lr per update whatever its gradient, which bounds how far that rounding can carry)
    s2, w2 = run(None)
    assert s2["num_updates"] == s1["num_updates"] and s2["batch_size"] == s1["batch_size"]
    for k in ("policy loss", "entropy", "approx kl div"):
        assert s2[k] == pytest.approx(s1[k], rel=1e-3, abs=1e-7), k
    assert torch.allclose(w2, w1, rtol=0, atol=2 * 3e-4 * full)
    s3, _ = run(1e-9)
    assert 1 <= s3["num_updates"] < full


# ---------------------------------------------------------------------------------------------------- raw ABI
def test_raw_abi_refusals(bank):
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    L = nat.lib()
    B = 4
    env = _env(bank, B)
    env.reset_host(np.arange(B, dtype=np.uint64))
    nb = env.decima_snapshot_bytes()
    snaps = torch.zeros(5, nb, dtype=torch.uint8, device=env.device)
    sel = torch.zeros(5, B, dtype=torch.int32, device=env.device)
    traj = torch.zeros(B * 10 * 32, dtype=torch.uint8, device=env.device)
    num = torch.zeros(B, dtype=torch.int32, device=env.device)
    el = torch.zeros(B, dtype=torch.float64, device=env.device)
    stream = env._stream()
    assert L.ssb_decima_attach_rollout_store(None, snaps.data_ptr(), 5, sel.data_ptr(), sel.data_ptr()) == -1
    assert L.ssb_set_policy_streams(None, None) == -1
    assert L.ssb_decima_attach_rollout_store(env._h, snaps.data_ptr(), 5, sel.data_ptr(), sel.data_ptr()) == 0
    assert L.ssb_rollout_decima(env._h, 10, 0, traj.data_ptr(), stream) == -1  # capacity too small
    assert L.ssb_rollout_decima_async(env._h, 10, 1e6, 1, traj.data_ptr(), num.data_ptr(), el.data_ptr(), stream) == -1
    assert L.ssb_rollout_decima(env._h, 5, 0, traj.data_ptr(), stream) == 0
    assert L.ssb_decima_attach_rollout_store(env._h, None, 0, None, None) == 0
    snap = env.decima_snapshot()
    env.decima_snapshot_load(snap)
    assert L.ssb_decima_attach_rollout_store(env._h, snaps.data_ptr(), 5, sel.data_ptr(), sel.data_ptr()) == -1
    env.decima_snapshot_unload()
    obs_only = BatchedSparkSchedSimEnv(CFG, num_envs=B, bank=bank, decima_obs=True)
    assert L.ssb_decima_attach_rollout_store(obs_only._h, snaps.data_ptr(), 5, sel.data_ptr(), sel.data_ptr()) == -1
    st = np.zeros(B, np.uint32)
    assert L.ssb_set_policy_streams(obs_only._h, st.ctypes.data) == -1
    torch.cuda.synchronize()
