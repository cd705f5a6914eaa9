"""The reference's PPO trainer (trainers/ppo.py) on the device: the loss head (`_compute_loss`, :104-140: forward values
and the adjoint seeds d loss / d lgprob, d loss / d entropy for the policy's backward pass), the parameter update
(clip_grad_norm_ + Adam), the rollout store and `_train`'s epoch loop over shuffled mini-batches of samples."""
import numpy as np
import torch

from . import _native as nat
from . import parallel
from .returns import _stream


class PPOLoss:
    """clip_range / entropy_coeff as in the trainer's config (ppo.py:43-46).  __call__ takes the flat per-sample
    device arrays (new_lgprob, old_lgprob, entropy: float32; returns, baselines: float64) and an optional int32
    index tensor selecting the mini-batch; returns ({"loss", "policy_loss", "entropy_loss", "approx_kl_div"} as a
    float32 device tensor of 4, grad_lgprob, grad_entropy)."""

    KEYS = ("loss", "policy_loss", "entropy_loss", "approx_kl_div")

    def __init__(self, clip_range=0.2, entropy_coeff=0.0):
        self.clip_range = float(clip_range)
        self.entropy_coeff = float(entropy_coeff)
        self._scratch = None

    def __call__(self, new_lgprob, old_lgprob, entropy, returns, baselines, idx=None):
        for t in (new_lgprob, old_lgprob, entropy):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        for t in (returns, baselines):
            assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
        dev = new_lgprob.device
        if idx is not None:
            assert idx.is_cuda and idx.dtype == torch.int32 and idx.is_contiguous()
        n = int(idx.numel()) if idx is not None else int(new_lgprob.numel())
        if self._scratch is None or self._scratch.device != dev:
            self._scratch = torch.empty(640, dtype=torch.float64, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)
        g_lp = torch.empty(n, dtype=torch.float32, device=dev)
        g_en = torch.empty(n, dtype=torch.float32, device=dev)
        nat.check(nat.lib().ssb_ppo_loss(
            new_lgprob.data_ptr(), old_lgprob.data_ptr(), entropy.data_ptr(), returns.data_ptr(), baselines.data_ptr(),
            idx.data_ptr() if idx is not None else None, n, self.clip_range, self.entropy_coeff,
            self._scratch.data_ptr(), out.data_ptr(), g_lp.data_ptr(), g_en.data_ptr(), _stream(new_lgprob)),
            "ssb_ppo_loss")
        return out, g_lp, g_en


class Loss:
    """What `loss.backward()` needs from the loss head: d loss / d lgprob and d loss / d entropy of the mini-batch's
    samples (the second and third result of PPOLoss.__call__); handed to DecimaScheduler.update_parameters."""

    def __init__(self, grad_lgprob: torch.Tensor, grad_entropy: torch.Tensor):
        self.grad_lgprob, self.grad_entropy = grad_lgprob, grad_entropy


class Adam:
    """clip_grad_norm_ + torch.optim.Adam on one flat float32 device vector (TrainableScheduler.update_parameters,
    schedulers/scheduler.py:37-54; opt_kwargs / max_grad_norm of the trainer's config).  `params` is updated in place;
    hand it to BatchedSparkSchedSimEnv.set_decima_weights afterwards."""

    def __init__(self, params: torch.Tensor, lr=3e-4, betas=(0.9, 0.999), eps=1e-8, max_grad_norm=None,
                 check_finite: bool = True):
        assert params.is_cuda and params.dtype == torch.float32 and params.is_contiguous()
        self.params = params
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.max_grad_norm = float(max_grad_norm) if max_grad_norm else 0.0
        self.exp_avg = torch.zeros_like(params)
        self.exp_avg_sq = torch.zeros_like(params)
        self.grad_norm = torch.zeros(1, dtype=torch.float32, device=params.device)
        self._scratch = torch.empty(128, dtype=torch.float64, device=params.device)
        self.num_steps = 0
        # read the norm back after every step and raise on NaN / Inf as the reference does (one 4-byte D2H per update)
        self.check_finite = bool(check_finite)

    def step(self, grads: torch.Tensor):
        assert grads.is_cuda and grads.dtype == torch.float32 and grads.is_contiguous()
        assert grads.numel() == self.params.numel()
        self.num_steps += 1
        nat.check(nat.lib().ssb_adam_step(
            self.params.data_ptr(), grads.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(),
            int(self.params.numel()), self.num_steps, self.lr, self.betas[0], self.betas[1], self.eps,
            self.max_grad_norm, self._scratch.data_ptr(), self.grad_norm.data_ptr(), _stream(grads)), "ssb_adam_step")
        if self.check_finite and not bool(torch.isfinite(self.grad_norm).item()):
            # clip_grad_norm_(..., error_if_nonfinite=True), schedulers/scheduler.py:46-48; the kernel skipped the update
            self.num_steps -= 1
            raise RuntimeError("The total norm for gradients is non-finite, so it cannot be clipped.")
        return self.grad_norm


def ppo_minibatch_update(env, snapshot, stage_sel, exec_sel, old_lgprob, returns, baselines, loss_fn: PPOLoss,
                         adam: Adam, target_kl=None, allreduce=None):
    """One mini-batch of PPO._train (trainers/ppo.py:72-102) on the device, the mini-batch being the B observations of
    one stored snapshot: evaluate_actions -> clip loss -> backward -> (gradient all-reduce) -> clip_grad_norm_ + Adam
    -> new weights into the policy.  `adam.params` is the flat weight vector (ssb_set_decima_weights layout).
    Returns (info, stepped): info = the loss head's four scalars on the host; stepped is False when the KL early
    stop (approx_kl_div > 1.5 * target_kl) skipped the update, as the trainer does.
    allreduce: optional callable(grads, num_samples) -> (grads, total) for several GPUs
    (parallel.allreduce_gradients).  With it the early stop is decided on the approximate KL averaged over ALL
    ranks' samples (one small all-reduce before the branch), so every rank steps or stops together -- a rank that
    stopped on its local value would leave the others waiting in the gradient all-reduce for ever.  The advantage
    normalisation stays per rank (each rank's mini-batch uses its own mean / std), which is the one place where N
    ranks differ from a single learner over the union of the samples."""
    B = env.num_envs
    env.decima_snapshot_load(snapshot)
    try:
        lg, en = env.decima_evaluate(None, stage_sel, exec_sel, for_backward=True)
        out, g_lp, g_en = loss_fn(lg, old_lgprob, en, returns, baselines)
        info = dict(zip(PPOLoss.KEYS, out.tolist()))
        if allreduce is not None:
            from . import parallel

            info["approx_kl_div_local"] = info["approx_kl_div"]
            info["approx_kl_div"] = parallel.allreduce_weighted_mean(out[3:4], B)
        if target_kl is not None and info["approx_kl_div"] > 1.5 * target_kl:
            return info, False
        grads = torch.zeros_like(adam.params)
        env.decima_backward(g_lp, g_en, grads)
    finally:
        env.decima_snapshot_unload()
    if allreduce is not None:
        grads, _ = allreduce(grads * B, B)
    adam.step(grads)
    env.set_decima_weights(adam.params)
    return info, True


def ppo_train(env, batches, loss_fn: PPOLoss, adam: Adam, num_epochs=3, target_kl=0.01, allreduce=None,
              generator=None):
    """PPO._train (trainers/ppo.py:72-102) over stored rollouts on the device.  `batches`: a list of mini-batches
    (snapshot, stage_sel, exec_sel, old_lgprob, returns, baselines), each the B observations of one stored snapshot
    (the reference draws its mini-batches by shuffling all samples; here the order of the snapshots is shuffled every
    epoch).  Stops for good as soon as a mini-batch's approximate KL exceeds 1.5 * target_kl, before stepping on it,
    as the trainer does.  Returns the trainer's summary: |mean| of the policy losses, entropy losses and approximate
    KL divergences of the mini-batches visited, plus the number of parameter updates."""
    import numpy as np

    policy_losses, entropy_losses, kls = [], [], []
    updates = 0
    go = True
    for _ in range(num_epochs):
        if not go:
            break
        order = torch.randperm(len(batches), generator=generator).tolist()
        for i in order:
            info, stepped = ppo_minibatch_update(env, *batches[i], loss_fn, adam, target_kl=target_kl,
                                                 allreduce=allreduce)
            policy_losses.append(info["policy_loss"]); entropy_losses.append(info["entropy_loss"])
            kls.append(info["approx_kl_div"])
            if not stepped:
                go = False
                break
            updates += 1
    return {"policy loss": float(np.abs(np.mean(policy_losses))), "entropy": float(np.abs(np.mean(entropy_losses))),
            "approx kl div": float(np.abs(np.mean(kls))), "num_updates": updates}


class RolloutStore:
    """RolloutBuffer (trainers/rollout_worker.py:18-46) of ALL environments of a handle for K decisions, on the device:
    per decision k the stored observations of the B envs (one ssb_decima_snapshot block), the Decima-format actions,
    their log-probabilities, rewards, wall times and which (k, b) hold a real transition.  `collect` is the rollout
    loop { snapshot ; policy ; step } (rollout_worker.py:135-157) with the sampled policy, one decision per call;
    `collect_fused` runs the device's Decima rollouts, which write the observations themselves, and also keeps the
    transition rows that ReturnsCalculator / Baseline read (`traj`, `num_steps`, `final_wall`)."""

    def __init__(self, env, num_decisions: int):
        self.env, self.K, self.B = env, int(num_decisions), env.num_envs
        dev = env.device
        self.snapshots = torch.empty(self.K, env.decima_snapshot_bytes(), dtype=torch.uint8, device=dev)
        self.stage_sel = torch.zeros(self.K, self.B, dtype=torch.int32, device=dev)
        self.exec_sel = torch.zeros(self.K, self.B, dtype=torch.int32, device=dev)
        self.lgprob = torch.zeros(self.K, self.B, dtype=torch.float32, device=dev)
        self.reward = torch.zeros(self.K, self.B, dtype=torch.float64, device=dev)
        self.wall_time = torch.zeros(self.K + 1, self.B, dtype=torch.float64, device=dev)
        self.valid = torch.zeros(self.K, self.B, dtype=torch.bool, device=dev)
        self.traj = self.num_steps = self.final_wall = None  # set by collect_fused

    def samples(self, idx: torch.Tensor):
        """The stored observations of dataset indices idx (= k * B + b, at most B of them) for
        DecimaScheduler.evaluate_actions: (store, steps, envs, n) with the B slots padded by empty ones."""
        B, dev = self.B, self.env.device
        idx = torch.as_tensor(idx, device=dev).reshape(-1)
        n = int(idx.numel())
        assert n <= B
        ks = torch.full((B,), -1, dtype=torch.int32, device=dev)
        bs = torch.zeros(B, dtype=torch.int32, device=dev)
        ks[:n], bs[:n] = (idx // B).int(), (idx % B).int()
        return self, ks, bs, n

    def actions(self, idx: torch.Tensor) -> torch.Tensor:
        """(stage_idx, job_idx, num_exec) of dataset indices idx as an int tensor [n, 3] (job_idx is not stored: the
        device policy derives the job from the stage; -1)."""
        idx = torch.as_tensor(idx, device=self.env.device).reshape(-1).long()
        k, b = idx // self.B, idx % self.B
        return torch.stack([self.stage_sel[k, b], torch.full_like(self.stage_sel[k, b], -1), self.exec_sel[k, b]], 1)

    def collect(self, max_events: int = 0):
        env = self.env
        for k in range(self.K):
            env.decima_snapshot(out=self.snapshots[k])
            hdr0 = env.hdr_bytes.clone()  # (device copy of the headers the decision is taken on)
            a, n = env.decima_policy()
            act = env.pol_action
            self.stage_sel[k] = act[:, 0]
            self.exec_sel[k] = act[:, 2]
            self.lgprob[k] = env.pol_lgprob
            env.step(a, n, max_events=max_events)
            h0 = hdr0.cpu().numpy().view(nat.OBS_HDR_DTYPE).reshape(-1)
            h1 = env.hdr()
            ok = (h0["terminated"] == 0) & (h0["error"] == 0) & (h1["error"] == 0) & (h1["was_reset"] == 0)
            self.valid[k] = torch.from_numpy(ok).to(env.device)
            self.wall_time[k] = torch.from_numpy(h0["wall_time"].copy()).to(env.device)
            self.reward[k] = torch.from_numpy(h1["reward"].copy()).to(env.device)
        self.wall_time[self.K] = torch.from_numpy(env.hdr()["wall_time"].copy()).to(env.device)
        return self

    def collect_fused(self, rollout_duration=None, seed_step=1, max_events=0):
        """The store filled by the device's Decima rollouts, without a host round trip per decision.
        rollout_duration None: RolloutWorkerSync (rollout_worker.py:135-157) -- the caller has reset the envs and
        auto-reset is off; rollout_decima(K) runs, a finished env idles, so each env's transitions are its rows
        [0, num_steps) and final_wall is its header's wall time.  Otherwise RolloutWorkerAsync (:160-206):
        rollout_decima_async(K, rollout_duration, seed_step), final_wall = the accumulated time.  `traj` (the
        transition rows, ssb_transition[B][K]), `num_steps` (i32[B]) and `final_wall` (f64[B]) are what
        ReturnsCalculator and Baseline take."""
        env, K, B = self.env, self.K, self.B
        if rollout_duration is None:
            assert not env._settings.get("autoreset", (False,))[0], "the sync protocol runs with auto-reset off"
            traj = env.rollout_decima(K, max_events=max_events, store=self)
            valid = (traj.view(torch.int32).view(B, K, 8)[..., 6] & 8) == 0
            num_steps = valid.sum(1, dtype=torch.int32)
            off = nat.OBS_HDR_DTYPE.fields["wall_time"][1]
            final_wall = env.hdr_bytes[:, off:off + 8].contiguous().view(torch.float64).reshape(B)
        else:
            traj, num_steps, final_wall = env.rollout_decima_async(K, rollout_duration, seed_step, store=self)
            valid = torch.arange(K, device=env.device)[None, :] < num_steps[:, None]
        rows64 = traj.view(torch.float64).view(B, K, 4)
        self.valid.copy_(valid.t())
        self.lgprob.copy_(traj.view(torch.float32).view(B, K, 8)[..., 7].t())
        self.reward.copy_(rows64[..., 1].t())
        self.wall_time[:K] = rows64[..., 0].t()
        self.wall_time[K] = final_wall
        self.traj, self.num_steps, self.final_wall = traj, num_steps, final_wall
        return self


def rollout_groups(num_sequences, num_rollouts, seed, rank=0, world=1):
    """The reference trainer's `num_sequences x num_rollouts` rollout workers (trainer.py:264-293) as this rank's share
    of the envs of BatchedSparkSchedSimEnv handles: worker i (global index) plays the job sequence of seed
    seed + i // num_rollouts and samples its actions from policy stream i % num_rollouts (set_policy_streams), so the
    members of a group share the arrivals but not the actions.  Returns (seeds u64[n], streams u32[n], seed_step =
    num_sequences: the k-th episode of every member of group j is seeded seed + j + num_sequences * k).  A rank holds
    whole groups (Baseline averages within a group), n = num_sequences * num_rollouts / world."""
    total = num_sequences * num_rollouts
    n, rem = divmod(total, world)
    assert rem == 0 and n % num_rollouts == 0, "every rank must hold whole groups of num_rollouts envs"
    seeds, seed_step = parallel.reference_worker_seeds(seed, num_sequences, num_rollouts)
    i = np.arange(rank * n, (rank + 1) * n)
    return seeds[i], (i % num_rollouts).astype(np.uint32), seed_step


def train_iteration(env, store, returns_calc, baseline, loss_fn: PPOLoss, adam: Adam, num_epochs, num_batches, target_kl,
                    allreduce=None, generator=None):
    """One iteration of the reference trainer after collection (trainer.py:172-212 _preprocess_rollouts +
    PPO.train_on_rollouts) on a store filled by RolloutStore.collect_fused: returns_calc (ReturnsCalculator) and
    baseline (Baseline) on the store's transition rows, transposed to the store's [K, B] layout, then
    ppo_train_samples.  Returns ppo_train_samples' summary plus "collect_stats" (the statistics of this handle's envs,
    parallel.stats_from_sums) and the "returns" / "baselines" (f64 [B, K] device tensors) it trained on."""
    assert store.traj is not None, "fill the store with collect_fused first"
    returns = returns_calc(store.traj, store.num_steps, store.final_wall, store.K)
    baselines = baseline(store.traj, returns, store.num_steps)
    summary = ppo_train_samples(env, store, returns.t().contiguous(), baselines.t().contiguous(), loss_fn, adam,
                                num_epochs=num_epochs, num_batches=num_batches, target_kl=target_kl,
                                allreduce=allreduce, generator=generator)
    summary["collect_stats"] = parallel.stats_from_sums(env.collect_stats())
    summary["returns"], summary["baselines"] = returns, baselines
    return summary


def _evaluate_slots(env, store, staging, ks, bs):
    """evaluate_actions on the samples (ks[i], bs[i]) gathered into the handle's B slots (empty where ks < 0);
    leaves the gathered snapshot loaded (the caller unloads)."""
    env.decima_snapshot_gather(store.snapshots, ks, bs, out=staging)
    env.decima_snapshot_load(staging)
    kk, bb = ks.clamp(min=0).long(), bs.clamp(min=0).long()
    stage_sel = store.stage_sel[kk, bb].contiguous()
    exec_sel = store.exec_sel[kk, bb].contiguous()
    return env.decima_evaluate(None, stage_sel, exec_sel, for_backward=True)


def ppo_train_samples(env, store: RolloutStore, returns: torch.Tensor, baselines: torch.Tensor, loss_fn: PPOLoss,
                      adam: Adam, num_epochs=3, num_batches=10, target_kl=0.01, allreduce=None, generator=None):
    """PPO.train_on_rollouts + PPO._train (trainers/ppo.py:52-102) on the device with the reference's mini-batches:
    ALL valid samples (k, b) of the store form the dataset, every epoch they are shuffled and split into mini-batches
    of len(dataset) // num_batches + 1 samples (DataLoader(shuffle=True), :63-68); per mini-batch: evaluate_actions ->
    clip loss over the whole mini-batch -> KL early stop -> backward -> (gradient all-reduce) -> clip_grad_norm_ + Adam
    -> new weights.  returns / baselines: float64 [K, B].  A mini-batch larger than the handle's B slots is evaluated
    in chunks of B (the loss head always sees the whole mini-batch; the backward pass re-evaluates chunk by chunk).
    Returns the trainer's summary plus the number of updates."""
    import numpy as np

    B, dev = env.num_envs, env.device
    flat = torch.nonzero(store.valid.reshape(-1)).reshape(-1)  # dataset: indices k * B + b of the real transitions
    N = int(flat.numel())
    batch_size = N // num_batches + 1
    staging = torch.empty(env.decima_snapshot_bytes(), dtype=torch.uint8, device=dev)
    ret_f, base_f, old_f = returns.reshape(-1), baselines.reshape(-1), store.lgprob.reshape(-1)
    policy_losses, entropy_losses, kls, updates, go = [], [], [], 0, True

    def slots(chunk):  # chunk: up to B dataset indices -> (ks, bs) padded with -1
        ks = torch.full((B,), -1, dtype=torch.int32, device=dev)
        bs = torch.zeros(B, dtype=torch.int32, device=dev)
        ks[:chunk.numel()] = (chunk // B).int()
        bs[:chunk.numel()] = (chunk % B).int()
        return ks, bs

    for _ in range(num_epochs):
        if not go:
            break
        perm = flat[torch.randperm(N, generator=generator).to(dev)]
        for lo in range(0, N, batch_size):
            mb = perm[lo:lo + batch_size]
            n = int(mb.numel())
            chunks = [mb[c:c + B] for c in range(0, n, B)]
            new_lg = torch.empty(n, dtype=torch.float32, device=dev)
            ent = torch.empty(n, dtype=torch.float32, device=dev)
            loaded = False
            try:
                for ci, ch in enumerate(chunks):  # forward over the whole mini-batch
                    lg, en = _evaluate_slots(env, store, staging, *slots(ch))
                    loaded = True
                    new_lg[ci * B:ci * B + ch.numel()] = lg[:ch.numel()]
                    ent[ci * B:ci * B + ch.numel()] = en[:ch.numel()]
                    if len(chunks) > 1:
                        env.decima_snapshot_unload(); loaded = False
                out, g_lp, g_en = loss_fn(new_lg, old_f[mb].contiguous(), ent, ret_f[mb].contiguous(),
                                          base_f[mb].contiguous())
                info = dict(zip(PPOLoss.KEYS, out.tolist()))
                if allreduce is not None:
                    from . import parallel

                    info["approx_kl_div"] = parallel.allreduce_weighted_mean(out[3:4], n)
                policy_losses.append(info["policy_loss"]); entropy_losses.append(info["entropy_loss"])
                kls.append(info["approx_kl_div"])
                if target_kl is not None and info["approx_kl_div"] > 1.5 * target_kl:
                    go = False
                    break
                grads = torch.zeros_like(adam.params)
                for ci, ch in enumerate(chunks):  # backward, chunk by chunk (a single chunk is still loaded)
                    if len(chunks) > 1:
                        _evaluate_slots(env, store, staging, *slots(ch))
                        loaded = True
                    gl = torch.zeros(B, dtype=torch.float32, device=dev)
                    ge = torch.zeros(B, dtype=torch.float32, device=dev)
                    gl[:ch.numel()] = g_lp[ci * B:ci * B + ch.numel()]
                    ge[:ch.numel()] = g_en[ci * B:ci * B + ch.numel()]
                    env.decima_backward(gl, ge, grads)
                    env.decima_snapshot_unload(); loaded = False
            finally:
                if loaded:
                    env.decima_snapshot_unload()
            if allreduce is not None:
                grads, _ = allreduce(grads * n, n)
            adam.step(grads)
            env.set_decima_weights(adam.params)
            updates += 1
    return {"policy loss": float(np.abs(np.mean(policy_losses))), "entropy": float(np.abs(np.mean(entropy_losses))),
            "approx kl div": float(np.abs(np.mean(kls))), "num_updates": updates, "num_samples": N,
            "batch_size": batch_size}
