"""BatchedSparkSchedSimEnv: B independent SparkSchedSimEnv episodes on one GPU.

This replaces the reference's "one CPU process per env" rollout workers
(trainers/trainer.py:264-293, trainers/rollout_worker.py:53-157) by one device-resident batch.
`reset`/`step` keep the reference's per-environment semantics (spark_sched_sim.py:127-221); the
observation comes back as device tensors with a fixed stride per environment:

    nodes          f32 [B, S, 3]   rows [0, num_nodes[b])   (remaining, most-recent duration, schedulable)
    edge_links     i32 [B, M, 2]   rows [0, num_edges[b])   relabelled to observation node ids
    dag_ptr        i32 [B, J+1]    entries [0, num_active_jobs[b]]
    exec_supplies  i32 [B, J]
    hdr            structured [B]  reward, wall_time, counts, num_committable_execs, source_job_idx,
                                   terminated, truncated, error

PyTorch is used for device memory and streams only; all simulation work happens in libssb.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _native as nat
from .bank import TemplateBank, synthetic_bank

ERROR_MESSAGES = {
    1: "invalid action: does not belong to the action space",
    2: "invalid action: stage index out of range of the schedulable stages",
    3: "invalid action: stage is not currently schedulable",
    4: "invalid action: must commit at least one executor",
    5: "invalid action: too many executors requested",
    6: "must either have a limit on job arrivals or time.",
    7: "no task duration data for this stage / executor level",
    8: "duration tape exhausted",
    9: "step() called on a finished episode",
    10: "episode exceeds the configured job/stage capacity",
}


class BatchedSparkSchedSimEnv:
    def __init__(self, env_cfg: dict, num_envs: int, bank: TemplateBank | None = None,
                 device: str | torch.device = "cuda:0", max_jobs: int | None = None,
                 tape_capacity: int = 0, log_capacity: int = 0, decima_obs: bool = False,
                 decima_policy: bool = False, history_capacity: int = 0):
        self.L = nat.lib()
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedSparkSchedSimEnv needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.bank = bank if bank is not None else synthetic_bank(0)
        self.num_envs = int(num_envs)
        self.num_executors = int(env_cfg["num_executors"])
        cap = env_cfg.get("job_arrival_cap")
        self.job_arrival_cap = int(cap) if cap else 0
        if max_jobs is None:
            max_jobs = self.job_arrival_cap if self.job_arrival_cap > 0 else 256
        self.max_jobs = int(max_jobs)
        self._ctor = (env_cfg, int(tape_capacity), int(log_capacity), bool(decima_obs), bool(decima_policy),
                      int(history_capacity))
        self._settings = {}   # what the setters changed on the handle (re-applied by grow())
        self._weights = None
        self._create()

    def _create(self):
        """(Re-)creates the native handle for self.max_jobs and maps its views."""
        env_cfg, tape_capacity, log_capacity, decima_obs, decima_policy, history_capacity = self._ctor
        self.cfg = nat.SsbConfig(
            self.num_envs, self.num_executors, self.job_arrival_cap, self.max_jobs,
            int(tape_capacity), int(log_capacity), float(env_cfg["moving_delay"]),
            float(env_cfg.get("warmup_delay", 0.0)), float(env_cfg["job_arrival_rate"]),
            float(env_cfg.get("beta", 0.0)),
            (nat.FLAG_DECIMA_OBS if (decima_obs or decima_policy) else 0)
            | (nat.FLAG_DECIMA_POLICY if decima_policy else 0), int(history_capacity))
        self.history_capacity = int(history_capacity)
        decima_obs = decima_obs or decima_policy
        self._bank_struct, self._bank_keep = nat.make_bank_struct(self.bank)
        nbytes = C.c_size_t()
        nat.check(self.L.ssb_workspace_bytes(C.byref(self.cfg), C.byref(self._bank_struct),
                                             C.byref(nbytes)), "ssb_workspace_bytes")
        self.workspace_bytes = int(nbytes.value)
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(self.workspace_bytes, dtype=torch.uint8, device=self.device)
        self._h = C.c_void_p()
        nat.check(self.L.ssb_create(C.byref(self.cfg), C.byref(self._bank_struct), self.device.index,
                                    self.workspace.data_ptr(), self.workspace_bytes,
                                    C.byref(self._h)), "ssb_create")
        v = nat.SsbViews()
        nat.check(self.L.ssb_get_views(self._h, C.byref(v)), "ssb_get_views")
        B, S, M, J = self.num_envs, v.node_stride, v.edge_stride, v.job_stride
        self.node_stride, self.edge_stride, self.job_stride = S, M, J
        self.hdr_bytes = self._view(v.hdr, B * nat.OBS_HDR_DTYPE.itemsize, torch.uint8).view(B, -1)
        self.nodes = self._view(v.nodes, B * S * 3 * 4, torch.float32).view(B, S, 3)
        self.edge_links = self._view(v.edge_links, B * M * 2 * 4, torch.int32).view(B, M, 2)
        self.dag_ptr = self._view(v.dag_ptr, B * (J + 1) * 4, torch.int32).view(B, J + 1)
        self.exec_supplies = self._view(v.exec_supplies, B * J * 4, torch.int32).view(B, J)
        sp = C.c_void_p()
        nat.check(self.L.ssb_get_stats(self._h, C.byref(sp)), "ssb_get_stats")
        self.stats_bytes = self._view(sp.value, B * nat.STATS_DTYPE.itemsize, torch.uint8).view(B, -1)
        # pinned: the D2H copy of the headers in the *_host calls is then a true async DMA
        self._hdr_pin = torch.zeros(B * nat.OBS_HDR_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
        self._hdr_host = self._hdr_pin.numpy().view(nat.OBS_HDR_DTYPE).reshape(-1)
        self.has_decima_obs = bool(decima_obs)
        if decima_obs:
            dv = nat.SsbDecimaViews()
            nat.check(self.L.ssb_get_decima_views(self._h, C.byref(dv)), "ssb_get_decima_views")
            self.dec_features = self._view(dv.features, B * S * 5 * 4, torch.float32).view(B, S, 5)
            self.dec_stage_mask = self._view(dv.stage_mask, B * S, torch.uint8).view(B, S)
            self.dec_frontier_mask = self._view(dv.frontier_mask, B * S, torch.uint8).view(B, S)
            self.dec_commit_caps = self._view(dv.commit_caps, B * J * 4, torch.int32).view(B, J)
            self.dec_edge_bits = self._view(dv.edge_bits, B * M * 8, torch.int64).view(B, M)
            self.dec_depth = self._view(dv.depth, B * 4, torch.int32)
        self.has_decima_policy = bool(decima_policy)
        if decima_policy:
            pv = nat.SsbPolicyViews()
            nat.check(self.L.ssb_get_policy_views(self._h, C.byref(pv)), "ssb_get_policy_views")
            Ep = pv.exec_stride
            self.pol_stage_logits = self._view(pv.stage_logits, B * S * 4, torch.float32).view(B, S)
            self.pol_exec_logits = self._view(pv.exec_logits, B * Ep * 4, torch.float32).view(B, Ep)
            self.pol_action = self._view(pv.action, B * 4 * 4, torch.int32).view(B, 4)
            self.pol_lgprob = self._view(pv.lgprob, B * 4, torch.float32)
            self.pol_entropy = self._view(pv.entropy, B * 4, torch.float32)

    # ---------------------------------------------------------------- plumbing
    def _view(self, ptr, nbytes, dtype):
        off = int(ptr) - self.workspace.data_ptr()
        assert 0 <= off and off + nbytes <= self.workspace_bytes
        return self.workspace[off:off + nbytes].view(dtype)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def grow(self, max_jobs: int) -> None:
        """Re-creates the handle with room for `max_jobs` jobs per env (node / edge / pool capacities follow).  The
        capacity is fixed at creation (one workspace, carved once), so growing means a new handle: every env's
        state is lost (reset afterwards); the policy weights, the policy sampling streams, the auto-reset mode,
        the mean time limit and the episode log (attach_episode_log) are carried over.  Time-limited arrivals without a job cap are the case that needs this: an episode that draws
        more jobs than the capacity stops at its reset with SSB_ENV_CAPACITY (`reset_host(..., grow=True)` grows
        and retries; `required_job_capacity` sizes the handle up front)."""
        assert max_jobs > self.max_jobs
        self.close()
        self.max_jobs = int(max_jobs)
        self._create()
        if self._weights is not None:
            self.set_decima_weights(self._weights)
        if "autoreset" in self._settings:
            self.set_autoreset(*self._settings["autoreset"])
        if "mean_time_limit" in self._settings:
            self.set_mean_time_limit(self._settings["mean_time_limit"])
        if "policy_streams" in self._settings:
            self.set_policy_streams(self._settings["policy_streams"])
        if "episode_log" in self._settings:
            self._attach_episode_log()  # the same buffers: the records, counts and window carry over

    @staticmethod
    def required_job_capacity(job_arrival_rate: float, mean_time_limit: float, tail: float = 1e-9) -> int:
        """Jobs per episode that Poisson arrivals (rate per ms) under an Exp(mean) time limit exceed with probability
        `tail`: the count is geometric, P(N > n) = (rate * mean / (1 + rate * mean)) ** n  (+ the job at t = 0)."""
        x = float(job_arrival_rate) * float(mean_time_limit)
        return 2 + int(np.ceil(np.log(tail) / np.log(x / (1.0 + x))))

    def close(self):
        if getattr(self, "_h", None):
            self.L.ssb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _dev(self, x, dtype):
        if x is None:
            return None
        if isinstance(x, torch.Tensor):
            t = x.to(device=self.device, dtype=dtype).contiguous()
        else:
            t = torch.as_tensor(np.asarray(x), dtype=dtype).to(self.device)
        assert t.numel() == self.num_envs
        return t

    # ---------------------------------------------------------------- device-tensor API
    def reset(self, seeds, time_limits=None, mask=None):
        """reset(seed, options={"time_limit"}) per env; arguments are device tensors or arrays."""
        s = self._dev(torch.as_tensor(np.asarray(seeds, dtype=np.uint64).view(np.int64))
                      if not isinstance(seeds, torch.Tensor) else seeds, torch.int64)
        tl = self._dev(time_limits, torch.float64)
        m = self._dev(mask, torch.uint8)
        self._keep = (s, tl, m)
        nat.check(self.L.ssb_reset(self._h, s.data_ptr(), tl.data_ptr() if tl is not None else None,
                                   m.data_ptr() if m is not None else None, self._stream()), "ssb_reset")

    def step(self, stage_idx, num_exec, mask=None, max_events=0):
        """step(action) per env.  max_events > 0: each env processes at most that many timeline
        events; envs that have not reached their next decision come back with hdr["pending"] = 1
        and continue (ignoring their action) at the next call."""
        a = self._dev(stage_idx, torch.int32)
        n = self._dev(num_exec, torch.int32)
        m = self._dev(mask, torch.uint8)
        self._keep = (a, n, m)
        nat.check(self.L.ssb_step(self._h, a.data_ptr(), n.data_ptr(),
                                  m.data_ptr() if m is not None else None, int(max_events),
                                  self._stream()), "ssb_step")

    def fair_actions(self, dynamic_partition=True):
        a = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        n = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        nat.check(self.L.ssb_fair_actions(self._h, int(dynamic_partition), a.data_ptr(), n.data_ptr(),
                                          self._stream()), "ssb_fair_actions")
        return a, n

    def rollout_fair(self, num_decisions, dynamic_partition=True, auto_reset=True, seed_step=1):
        nat.check(self.L.ssb_rollout_fair(self._h, int(num_decisions), int(dynamic_partition),
                                          int(auto_reset), int(seed_step), self._stream()),
                  "ssb_rollout_fair")

    def set_autoreset(self, enable: bool = True, seed_step: int = 1) -> None:
        """Vector-env auto-reset ("next step" mode): a step() on a finished env re-seeds it with
        seed + seed_step * reset_count (rollout_worker.py:118-120), ignores its action and returns the new
        episode's first observation with hdr["was_reset"] = 1."""
        nat.check(self.L.ssb_set_autoreset(self._h, int(bool(enable)), int(seed_step)), "ssb_set_autoreset")
        self._settings["autoreset"] = (bool(enable), int(seed_step))

    def rollout_fair_async(self, max_decisions, rollout_duration, dynamic_partition=True, seed_step=1):
        """Fixed-duration rollouts spanning resets (RolloutWorkerAsync.collect_rollout, rollout_worker.py:160-206).
        Returns (traj uint8 device tensor [B * max_decisions * 32], num_steps i32[B], elapsed f64[B])."""
        return self._async(max_decisions, lambda traj, num, el: nat.check(
            self.L.ssb_rollout_fair_async(self._h, int(max_decisions), float(rollout_duration), int(dynamic_partition),
                                          int(seed_step), traj, num, el, self._stream()), "ssb_rollout_fair_async"))

    def _async(self, max_decisions, launch):
        """Runs launch(traj, num_steps, elapsed) on device pointers to new buffers for a fixed-duration rollout: traj
        for B * max_decisions transition rows, num_steps i32[B] and elapsed f64[B].  Returns the three tensors."""
        nbytes = self.num_envs * int(max_decisions) * nat.TRANSITION_DTYPE.itemsize
        traj = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        num = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        el = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        launch(traj.data_ptr(), num.data_ptr(), el.data_ptr())
        return traj, num, el

    def set_mean_time_limit(self, mean_ms: float) -> None:
        """StochasticTimeLimit on the device: every reset without an explicit limit (and every auto-reset) draws
        the episode's time limit ~ Exp(mean_ms) from the episode seed's Philox LIMIT stream."""
        nat.check(self.L.ssb_set_mean_time_limit(self._h, float(mean_ms)), "ssb_set_mean_time_limit")
        self._settings["mean_time_limit"] = float(mean_ms)

    def rollout_fair_traj(self, num_decisions, dynamic_partition=True, auto_reset=True, seed_step=1,
                          out: "torch.Tensor | None" = None, host: "torch.Tensor | None" = None):
        """Fused rollout that also records every transition (what RolloutBuffer keeps per step besides
        the observation, trainers/rollout_worker.py:18-46).  `out`: uint8 device tensor of
        B * num_decisions * 32 bytes (allocated if None).  With `host` (a pinned uint8 tensor of the same
        size) the records are copied to the host and returned as a structured numpy array
        [B, num_decisions] of _native.TRANSITION_DTYPE; otherwise the device tensor is returned."""
        return self._recorded(num_decisions, out, host, lambda traj: nat.check(
            self.L.ssb_rollout_fair_traj(self._h, int(num_decisions), int(dynamic_partition), int(auto_reset),
                                         int(seed_step), traj, self._stream()), "ssb_rollout_fair_traj"))

    def _recorded(self, num_decisions, out, host, launch):
        """Runs launch(device pointer) on a trajectory buffer for B * num_decisions transition rows: `out` (a uint8
        device tensor of at least that size; allocated if None).  Returns `out`, or with `host` (pinned uint8 of the
        same size) the rows copied to the host as a structured array [B, num_decisions] of _native.TRANSITION_DTYPE."""
        nbytes = self.num_envs * int(num_decisions) * nat.TRANSITION_DTYPE.itemsize
        if out is None:
            out = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        assert out.numel() >= nbytes and out.is_cuda
        launch(out.data_ptr())
        if host is None:
            return out
        host[:nbytes].copy_(out[:nbytes], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return host[:nbytes].numpy().view(nat.TRANSITION_DTYPE).reshape(self.num_envs, int(num_decisions))

    def random_actions(self, mask=None):
        """The random scheduler (RandomScheduler, random_scheduler.py:7-32) on the device: one action per env with
        mask[i] != 0 (None = all), drawn from the env's Philox RANDOM stream (a function of the episode seed and the
        decision's index in the episode).  Envs that are done, pending or masked out get (-1, 1) and keep their
        draws.  Returns device int32 tensors (stage_idx, num_exec)."""
        a = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        n = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        m = self._dev(mask, torch.uint8)
        self._keep = (m,)
        nat.check(self.L.ssb_random_actions(self._h, m.data_ptr() if m is not None else None, a.data_ptr(),
                                            n.data_ptr(), self._stream()), "ssb_random_actions")
        return a, n

    def rollout_random(self, num_decisions, auto_reset=True, seed_step=1, record=False,
                       out: "torch.Tensor | None" = None, host: "torch.Tensor | None" = None):
        """rollout_fair with the random scheduler: `num_decisions` decisions per env in one launch.  With
        record=True every transition is stored (lgprob 0) and returned as rollout_fair_traj returns it: the uint8
        device tensor `out` (allocated if None), or with `host` (pinned, same size) the structured numpy array
        [B, num_decisions] of _native.TRANSITION_DTYPE."""
        if not record:
            nat.check(self.L.ssb_rollout_random(self._h, int(num_decisions), int(auto_reset), int(seed_step), None,
                                                self._stream()), "ssb_rollout_random")
            return None
        return self._recorded(num_decisions, out, host, lambda traj: nat.check(
            self.L.ssb_rollout_random(self._h, int(num_decisions), int(auto_reset), int(seed_step), traj,
                                      self._stream()), "ssb_rollout_random"))

    def rollout_random_async(self, max_decisions, rollout_duration, seed_step=1):
        """rollout_fair_async with the random scheduler: fixed-duration rollouts spanning resets
        (RolloutWorkerAsync.collect_rollout, rollout_worker.py:160-206), every row with lgprob 0.  The draws are those
        of rollout_random from the same seeds.  Returns (traj uint8 device tensor [B * max_decisions * 32], num_steps
        i32[B], elapsed f64[B])."""
        return self._async(max_decisions, lambda traj, num, el: nat.check(
            self.L.ssb_rollout_random_async(self._h, int(max_decisions), float(rollout_duration), int(seed_step), traj,
                                            num, el, self._stream()), "ssb_rollout_random_async"))

    # ---------------------------------------------------------------- host-buffer API (e2e path)
    def reset_host(self, seeds: np.ndarray, time_limits: np.ndarray | None = None,
                   mask: np.ndarray | None = None, grow: bool = False, grow_limit: int = 1 << 16) -> np.ndarray:
        """grow=True (only with mask=None, i.e. when every env is reset): if an episode needs more jobs than the
        handle has room for (hdr["error"] == SSB_ENV_CAPACITY), the handle is re-created with twice the capacity and
        the reset repeated -- resets are functions of the seed, so the result is what a large enough handle gives."""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        tl = None if time_limits is None else np.ascontiguousarray(time_limits, dtype=np.float64)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        while True:
            nat.check(self.L.ssb_reset_host(self._h, seeds.ctypes.data, tl.ctypes.data if tl is not None else None,
                                            m.ctypes.data if m is not None else None,
                                            self._hdr_host.ctypes.data), "ssb_reset_host")
            if not (grow and m is None and (self._hdr_host["error"] == nat.ENV_CAPACITY).any()
                    and 2 * self.max_jobs <= grow_limit):
                return self._hdr_host
            self.grow(2 * self.max_jobs)

    def step_host(self, stage_idx: np.ndarray, num_exec: np.ndarray, mask: np.ndarray | None = None,
                  max_events: int = 0) -> np.ndarray:
        a = np.ascontiguousarray(stage_idx, dtype=np.int32)
        n = np.ascontiguousarray(num_exec, dtype=np.int32)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        nat.check(self.L.ssb_step_host(self._h, self._ptr(a), self._ptr(n),
                                       self._ptr(m) if m is not None else None, int(max_events),
                                       self._ptr(self._hdr_host)), "ssb_step_host")
        return self._hdr_host

    def _ptr(self, arr: np.ndarray) -> int:
        """Address of a host array for the C ABI.  `arr.ctypes.data` builds a ctypes helper object on every access
        (2 us each, five per step call); callers of the host-buffer API pass the same few (pinned) arrays call after call,
        so the addresses of the last arrays seen are kept -- together with the arrays themselves, which keeps an id from
        being reused by another object."""
        c = self.__dict__.setdefault("_ptr_cache", {})
        ent = c.get(id(arr))
        if ent is not None and ent[0] is arr:
            return ent[1]
        if len(c) >= 16:
            c.clear()
        ptr = arr.ctypes.data
        c[id(arr)] = (arr, ptr)
        return ptr

    def step_fair_host(self, stage_idx: np.ndarray, num_exec: np.ndarray, next_stage_idx: np.ndarray,
                       next_num_exec: np.ndarray, dynamic_partition: bool = True, mask: np.ndarray | None = None,
                       max_events: int = 0) -> np.ndarray:
        """step_host that also fills next_stage_idx / next_num_exec (host int32[B], ideally pinned) with the built-in
        fair / FIFO scheduler's action for the new observation (evaluated inside the step kernel)."""
        a = np.ascontiguousarray(stage_idx, dtype=np.int32)
        n = np.ascontiguousarray(num_exec, dtype=np.int32)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        assert next_stage_idx.dtype == np.int32 and next_num_exec.dtype == np.int32
        nat.check(self.L.ssb_step_fair_host(self._h, self._ptr(a), self._ptr(n),
                                            self._ptr(m) if m is not None else None, int(max_events),
                                            int(dynamic_partition), self._ptr(self._hdr_host),
                                            self._ptr(next_stage_idx), self._ptr(next_num_exec)),
                  "ssb_step_fair_host")
        return self._hdr_host

    def obs_host(self, node_capacity: int | None = None, edge_capacity: int | None = None) -> dict:
        """The observation graphs of ALL envs on the host, packed (ssb_get_obs_host): pinned numpy arrays
        offsets i32[B + 1, 3] (first node / edge / job of env b; row B = totals), nodes f32[total, 3],
        edge_links i32[total, 2], dag_ptr i32[total jobs + B], exec_supplies i32[total jobs].  Env b's slices:
        nodes[o[b,0]:o[b+1,0]], edge_links[o[b,1]:o[b+1,1]], exec_supplies[o[b,2]:o[b+1,2]],
        dag_ptr[o[b,2]+b : o[b+1,2]+b+1].  The arrays are reused by the next call."""
        B = self.num_envs
        if getattr(self, "_pack", None) is None:
            n = C.c_size_t()
            nat.check(self.L.ssb_packed_obs_bytes(self._h, C.byref(n)), "ssb_packed_obs_bytes")
            ncap = node_capacity or B * self.node_stride
            ecap = edge_capacity or B * self.edge_stride
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()  # noqa: E731
            self._pack = {
                "scratch": torch.empty(n.value, dtype=torch.uint8, device=self.device),
                "offsets": pin((B + 1, 3), torch.int32), "nodes": pin((ncap, 3), torch.float32),
                "edge_links": pin((ecap, 2), torch.int32), "dag_ptr": pin((B * (self.job_stride + 1),), torch.int32),
                "exec_supplies": pin((B * self.job_stride,), torch.int32)}
            k = self._pack
            self._pack_struct = nat.SsbPackedObs(
                k["offsets"].data_ptr(), k["nodes"].data_ptr(), k["edge_links"].data_ptr(), k["dag_ptr"].data_ptr(),
                k["exec_supplies"].data_ptr(), ncap, ecap, B * self.job_stride)
        k = self._pack
        nat.check(self.L.ssb_get_obs_host(self._h, C.byref(self._pack_struct), k["scratch"].data_ptr(),
                                          k["scratch"].numel()), "ssb_get_obs_host")
        o = k["offsets"].numpy()
        tn, te, tj = (int(x) for x in o[B])
        return {"offsets": o, "nodes": k["nodes"].numpy()[:tn], "edge_links": k["edge_links"].numpy()[:te],
                "dag_ptr": k["dag_ptr"].numpy()[:tj + B], "exec_supplies": k["exec_supplies"].numpy()[:tj]}

    # ---------------------------------------------------------------- results
    def hdr(self) -> np.ndarray:
        """Structured numpy copy of the B observation headers (synchronises)."""
        return self.hdr_bytes.cpu().numpy().view(nat.OBS_HDR_DTYPE).reshape(-1)

    def stats(self) -> dict:
        s = self.stats_bytes.cpu().numpy().view(nat.STATS_DTYPE).reshape(-1)
        return {f: int(s[f].sum()) for f in nat.STATS_FIELDS}

    def stats_per_env(self) -> np.ndarray:
        """The ssb_stats counters of every env (structured array [B])."""
        return self.stats_bytes.cpu().numpy().view(nat.STATS_DTYPE).reshape(-1).copy()

    def collect_stats(self, out: "torch.Tensor | None" = None) -> torch.Tensor:
        """collect_stats (trainers/rollout_worker.py:122-129) over this GPU's envs as a device f64[8] vector of
        sums (see ssb_collect_stats); all-reduce it over ranks, then parallel.stats_from_sums() turns it into
        the reference's dict."""
        if out is None:
            out = torch.zeros(8, dtype=torch.float64, device=self.device)
        nat.check(self.L.ssb_collect_stats(self._h, out.data_ptr(), self._stream()), "ssb_collect_stats")
        return out

    def reset_stats(self):
        nat.check(self.L.ssb_reset_stats(self._h, self._stream()), "ssb_reset_stats")

    # ---------------------------------------------------------------- episode log (ssb_attach_episode_log)
    def attach_episode_log(self, capacity: int = 64, window: int = 200) -> None:
        """Records every finished episode on the device -- a RecordEpisodeStatistics for the batched env -- in a
        ring of `capacity` records per env, and every completed job's duration in a ring of the last `window` per env
        (the reference's job_duration_buff, deque(maxlen=200), which survives resets).  The three buffers are device
        tensors of this object, zeroed here; grow() re-attaches the same ones, so the log and the window carry over.
        Read them with episodes() and job_duration_window(); collect_stats()[6:8] then carries the window's means."""
        B, cap, win = self.num_envs, int(capacity), int(window)
        if cap < 0 or win < 0:
            raise ValueError("capacity and window must be >= 0")
        rec = torch.zeros(max(B * cap * nat.EPISODE_DTYPE.itemsize, 1), dtype=torch.uint8, device=self.device)
        dur = torch.zeros(B, max(win, 1), dtype=torch.float64, device=self.device)
        cur = torch.zeros(B * nat.EPISODE_CURSOR_DTYPE.itemsize, dtype=torch.uint8, device=self.device)
        self._settings["episode_log"] = (rec, cap, dur, win, cur)
        self._attach_episode_log()

    def _attach_episode_log(self) -> None:
        rec, cap, dur, win, cur = self._settings["episode_log"]
        nat.check(self.L.ssb_attach_episode_log(self._h, rec.data_ptr() if cap else None, cap,
                                                dur.data_ptr() if win else None, win, cur.data_ptr(), self._stream()),
                  "ssb_attach_episode_log")

    def detach_episode_log(self) -> None:
        """Stops recording; the buffers are released."""
        nat.check(self.L.ssb_attach_episode_log(self._h, None, 0, None, 0, None, self._stream()),
                  "ssb_attach_episode_log")
        self._settings.pop("episode_log", None)

    def _episode_log(self):
        if "episode_log" not in self._settings:
            raise RuntimeError("no episode log attached (attach_episode_log())")
        return self._settings["episode_log"]

    def episode_cursors(self) -> torch.Tensor:
        """The per-env cursors as an int64 device tensor [B, 4]: episodes recorded, jobs completed, and the two
        library-use words."""
        return self._episode_log()[4].view(torch.int64).view(self.num_envs, 4)

    def episodes(self) -> dict:
        """The stored episode records, flattened env-major and oldest first within an env, as device tensors:
        env, seed (int64 holding the u64 seed), wall_time, time_limit, job_time, sum_job_duration (f64), decisions,
        jobs_arrived, jobs_completed, flags, episode (i32), terminated / truncated (bool), avg_job_duration (seconds,
        sum_job_duration / jobs_completed * 1e-3, nan without a completed job), avg_num_jobs (job_time / wall_time),
        and dropped: per env [B], the records the ring has overwritten.  Synchronises (the count is data-dependent)."""
        rec, cap, _, _, _ = self._episode_log()
        B = self.num_envs
        n_rec = self.episode_cursors()[:, 0]
        stored = n_rec.clamp(max=cap)
        k = torch.arange(max(cap, 1), device=self.device)
        env, kk = (k[None, :] < stored[:, None]).nonzero(as_tuple=True)
        slot = (n_rec[env] - stored[env] + kk) % max(cap, 1)
        rows = rec[:B * cap * nat.EPISODE_DTYPE.itemsize].view(torch.int64).view(B, max(cap, 1) if cap else 0, 8)
        r = rows[env, slot] if cap else torch.zeros(0, 8, dtype=torch.int64, device=self.device)
        f, i = r.view(torch.float64), r.view(torch.int32)
        jc = i[:, 12]
        out = {"env": env.to(torch.int32), "seed": r[:, 0], "wall_time": f[:, 1], "time_limit": f[:, 2],
               "job_time": f[:, 3], "sum_job_duration": f[:, 4], "decisions": i[:, 10], "jobs_arrived": i[:, 11],
               "jobs_completed": jc, "flags": i[:, 13], "episode": i[:, 14]}
        out["terminated"] = (out["flags"] & 1) != 0
        out["truncated"] = (out["flags"] & 2) != 0
        out["avg_job_duration"] = torch.where(jc > 0, out["sum_job_duration"] / jc.clamp(min=1) * 1e-3,
                                              torch.full_like(out["sum_job_duration"], float("nan")))
        out["avg_num_jobs"] = out["job_time"] / out["wall_time"]
        out["dropped"] = n_rec - stored
        return out

    def clear_episodes(self) -> None:
        """Zeroes every env's episode count (stream-ordered); the job-duration window is left as it is."""
        self.episode_cursors()[:, 0].zero_()

    def job_duration_window(self) -> tuple[torch.Tensor, torch.Tensor]:
        """(durations f64 [B, window] in ms, oldest to newest, nan past the fill; fill i64 [B]): env b's last
        min(completions, window) completed-job durations, across resets."""
        _, _, dur, win, _ = self._episode_log()
        n = self.episode_cursors()[:, 1]
        if win == 0:
            return torch.zeros(self.num_envs, 0, dtype=torch.float64, device=self.device), torch.zeros_like(n)
        fill = n.clamp(max=win)
        k = torch.arange(win, device=self.device)
        idx = (n[:, None] - fill[:, None] + k[None, :]) % win
        vals = dur.gather(1, idx)
        return torch.where(k[None, :] < fill[:, None], vals, torch.full_like(vals, float("nan"))), fill

    def obs(self, b: int = 0, hdr: np.ndarray | None = None) -> dict:
        """Observation of environment b as host arrays (the pieces of the reference obs dict)."""
        h = (self.hdr() if hdr is None else hdr)[b]
        N, M, Ja = int(h["num_nodes"]), int(h["num_edges"]), int(h["num_active_jobs"])
        return {
            "nodes": self.nodes[b, :N].cpu().numpy(),
            "edge_links": self.edge_links[b, :M].cpu().numpy(),
            "dag_ptr": self.dag_ptr[b, :Ja + 1].cpu().numpy(),
            "exec_supplies": self.exec_supplies[b, :Ja].cpu().numpy(),
            "num_committable_execs": int(h["num_committable_execs"]),
            "source_job_idx": int(h["source_job_idx"]),
        }

    def decima_obs(self):
        """Launches the Decima observation adapter (env_wrapper.py:69-143, utils.py:238-267) for all
        envs; results land in dec_features / dec_stage_mask / dec_commit_caps / dec_edge_bits /
        dec_depth (device tensors, same node/edge/job order as the base observation)."""
        nat.check(self.L.ssb_decima_obs(self._h, self._stream()), "ssb_decima_obs")

    def decima_obs_host(self, b: int = 0, hdr: np.ndarray | None = None) -> dict:
        """Decima observation of env b as host arrays, in the reference's shapes."""
        h = (self.hdr() if hdr is None else hdr)[b]
        N, M, Ja = int(h["num_nodes"]), int(h["num_edges"]), int(h["num_active_jobs"])
        depth = int(self.dec_depth[b].item())
        bits = self.dec_edge_bits[b, :M].cpu().numpy().view(np.uint64)
        caps = self.dec_commit_caps[b, :Ja].cpu().numpy()
        k = np.arange(depth, dtype=np.uint64)[:, None]
        return {
            "features": self.dec_features[b, :N].cpu().numpy(),
            "stage_mask": self.dec_stage_mask[b, :N].cpu().numpy().astype(bool),
            "frontier_mask": self.dec_frontier_mask[b, :N].cpu().numpy().astype(bool),
            "commit_caps": caps,
            "exec_mask": np.arange(self.num_executors)[None, :] < caps[:, None],
            "edge_bits": bits,
            "depth": depth,
            "edge_masks": ((bits[None, :] >> k) & np.uint64(1)).astype(bool),
        }

    # ---------------------------------------------------------------- Decima policy
    DECIMA_PARAM_ORDER = tuple(
        f"{net}.{layer}.{kind}"
        for net in ("encoder.node_encoder.mlp_prep", "encoder.node_encoder.mlp_msg",
                    "encoder.node_encoder.mlp_update", "encoder.dag_encoder.mlp",
                    "encoder.global_encoder.mlp", "stage_policy_network.mlp_score",
                    "exec_policy_network.mlp_score")
        for layer in (0, 2, 4) for kind in ("weight", "bias"))

    def set_decima_weights(self, state_dict) -> None:
        """Uploads a DecimaScheduler state dict (torch tensors or numpy arrays keyed as in
        models/decima/model.pt): 42 tensors / 20 802 float32 parameters."""
        if isinstance(state_dict, (torch.Tensor, np.ndarray)):  # the flat vector itself (state_dict order)
            flat = np.asarray(state_dict.detach().cpu().numpy() if hasattr(state_dict, "detach") else state_dict,
                              dtype=np.float32).reshape(-1)
        else:
            flat = np.concatenate([np.asarray(state_dict[k].detach().cpu().numpy()
                                              if hasattr(state_dict[k], "detach") else state_dict[k],
                                              dtype=np.float32).reshape(-1)
                                   for k in self.DECIMA_PARAM_ORDER])
        assert flat.size == nat.DECIMA_NUM_PARAMS, flat.size
        flat = np.ascontiguousarray(flat)
        nat.check(self.L.ssb_set_decima_weights(self._h, flat.ctypes.data, flat.size),
                  "ssb_set_decima_weights")
        self._weights = flat

    def set_policy_streams(self, streams) -> None:
        """Each env's Decima sampling stream (uint32 per env, None = all 0): the actions are drawn at Philox counter
        (decision index in the episode, stream, 4, 0) keyed by the episode seed, so envs that share a job sequence
        (same seed) but not a stream sample their own actions, as the reference's rollout workers do with their own
        torch RNGs.  Stream 0 is the default.  Resets keep the streams."""
        st = None if streams is None else np.ascontiguousarray(np.asarray(streams, dtype=np.uint32))
        assert st is None or st.size == self.num_envs
        nat.check(self.L.ssb_set_policy_streams(self._h, st.ctypes.data if st is not None else None),
                  "ssb_set_policy_streams")
        self._settings["policy_streams"] = st

    def _with_store(self, store, run):
        """run() with `store` (a ppo.RolloutStore of this handle) attached to the handle: the Decima rollouts then also
        write every transition row's observation and Decima-format action into it.  Detached again afterwards."""
        if store is None:
            return run()
        assert store.env is self and store.snapshots.shape[1] == self.decima_snapshot_bytes()
        nat.check(self.L.ssb_decima_attach_rollout_store(self._h, store.snapshots.data_ptr(), store.K,
                                                         store.stage_sel.data_ptr(), store.exec_sel.data_ptr()),
                  "ssb_decima_attach_rollout_store")
        try:
            return run()
        finally:
            nat.check(self.L.ssb_decima_attach_rollout_store(self._h, None, 0, None, None),
                      "ssb_decima_attach_rollout_store")

    def decima_policy(self, forced_stage=None, forced_num_exec=None):
        """One Decima decision per env on the device (observation adapter + GNN + sampling).
        Returns (stage_idx, num_exec) device tensors in the env's action format; the scores, the
        Decima-format action and the log-probability are in pol_* tensors."""
        fs = self._dev(forced_stage, torch.int32)
        fn = self._dev(forced_num_exec, torch.int32)
        a = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        n = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        self._keep_pol = (fs, fn)
        nat.check(self.L.ssb_decima_policy(self._h, fs.data_ptr() if fs is not None else None,
                                           fn.data_ptr() if fn is not None else None,
                                           a.data_ptr(), n.data_ptr(), self._stream()), "ssb_decima_policy")
        return a, n

    MLP_NAMES = ("encoder.node_encoder.mlp_prep", "encoder.node_encoder.mlp_msg", "encoder.node_encoder.mlp_update",
                 "encoder.dag_encoder.mlp", "encoder.global_encoder.mlp", "stage_policy_network.mlp_score",
                 "exec_policy_network.mlp_score")
    MLP_DIMS = ((5, 16), (16, 16), (16, 16), (21, 16), (16, 16), (53, 1), (36, 1))

    def decima_mlp_rows(self, mlp: int, x: torch.Tensor) -> torch.Tensor:
        """One of the policy's seven MLPs (index in state_dict order, MLP_NAMES) applied to the rows of x
        (float32 device tensor [n, in]) on the tensor-core path the policy uses -> [n, out]."""
        din, dout = self.MLP_DIMS[mlp]
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.shape[1] == din
        out = torch.empty(x.shape[0], dout, dtype=torch.float32, device=self.device)
        nat.check(self.L.ssb_decima_mlp_rows(self._h, int(mlp), x.data_ptr(), int(x.shape[0]), out.data_ptr(),
                                             self._stream()), "ssb_decima_mlp_rows")
        return out

    def decima_work(self) -> dict:
        """Rows per MLP and multiply-adds of the last decima_policy / decima_evaluate call (measurement)."""
        out = np.zeros(8, np.int64)
        nat.check(self.L.ssb_decima_work(self._h, out.ctypes.data), "ssb_decima_work")
        keys = ("nodes", "sinks", "candidates", "jobs", "exec_rows", "senders", "receivers", "macs")
        return dict(zip(keys, (int(x) for x in out)))

    def decima_snapshot(self, out: "torch.Tensor | None" = None) -> torch.Tensor:
        """Stores what the policy reads of every env's current observation (RolloutBuffer.obsns) in a device
        uint8 tensor."""
        n = C.c_size_t()
        nat.check(self.L.ssb_decima_snapshot_bytes(self._h, C.byref(n)), "ssb_decima_snapshot_bytes")
        if out is None:
            out = torch.empty(n.value, dtype=torch.uint8, device=self.device)
        assert out.numel() >= n.value
        nat.check(self.L.ssb_decima_snapshot(self._h, out.data_ptr(), self._stream()), "ssb_decima_snapshot")
        return out

    def decima_snapshot_bytes(self) -> int:
        n = C.c_size_t()
        nat.check(self.L.ssb_decima_snapshot_bytes(self._h, C.byref(n)), "ssb_decima_snapshot_bytes")
        return int(n.value)

    def decima_snapshot_gather(self, snapshots: torch.Tensor, src_step: torch.Tensor, src_env: torch.Tensor,
                               out: "torch.Tensor | None" = None) -> torch.Tensor:
        """A snapshot whose slot i holds the stored observation of sample (src_step[i], src_env[i]) of `snapshots`
        (uint8 device tensor [num_steps, snapshot_bytes]); src_step[i] < 0 leaves slot i empty.  The mini-batches of
        trainers/ppo.py:52-70 (shuffled over all samples of an iteration) are built with this."""
        nb = self.decima_snapshot_bytes()
        assert snapshots.is_cuda and snapshots.dtype == torch.uint8 and snapshots.dim() == 2 and snapshots.shape[1] == nb
        for t in (src_step, src_env):
            assert t.is_cuda and t.dtype == torch.int32 and t.is_contiguous() and t.numel() == self.num_envs
        if out is None:
            out = torch.empty(nb, dtype=torch.uint8, device=self.device)
        nat.check(self.L.ssb_decima_snapshot_gather(self._h, snapshots.data_ptr(), int(snapshots.shape[0]),
                                                    src_step.data_ptr(), src_env.data_ptr(), out.data_ptr(),
                                                    self._stream()), "ssb_decima_snapshot_gather")
        return out

    def decima_snapshot_load(self, snapshot: torch.Tensor):
        """Puts a stored observation in place (the live one is parked) for decima_evaluate(None, ...) +
        decima_backward; undo with decima_snapshot_unload()."""
        nat.check(self.L.ssb_decima_snapshot_load(self._h, snapshot.data_ptr(), self._stream()),
                  "ssb_decima_snapshot_load")

    def decima_snapshot_unload(self):
        nat.check(self.L.ssb_decima_snapshot_unload(self._h, self._stream()), "ssb_decima_snapshot_unload")

    def _backward_scratch(self) -> torch.Tensor:
        """The backward pass's scratch, allocated once and attached to the handle: evaluations then leave the
        message-passing levels' input rows in it and decima_backward does not have to replay the levels."""
        n = C.c_size_t()
        nat.check(self.L.ssb_decima_backward_bytes(self._h, C.byref(n)), "ssb_decima_backward_bytes")
        if getattr(self, "_bwd_scratch", None) is None or self._bwd_scratch.numel() < n.value:
            self._bwd_scratch = torch.empty(n.value, dtype=torch.uint8, device=self.device)
            self._bwd_attached = None
        if getattr(self, "_bwd_attached", None) != (self._h.value, self._bwd_scratch.data_ptr()):
            nat.check(self.L.ssb_decima_attach_backward_scratch(self._h, self._bwd_scratch.data_ptr()),
                      "ssb_decima_attach_backward_scratch")
            self._bwd_attached = (self._h.value, self._bwd_scratch.data_ptr())
        return self._bwd_scratch

    def decima_evaluate(self, snapshot: "torch.Tensor | None", stage_sel, exec_sel, for_backward: bool = False):
        """DecimaScheduler.evaluate_actions (forward only) on a stored snapshot (None: the one decima_snapshot_load
        put in place): (lgprobs, entropies) f32[B] for the given Decima-format actions; the envs themselves are
        left untouched.  for_backward: a decima_backward call follows (the forward pass keeps what it needs)."""
        if for_backward:
            self._backward_scratch()
        a = self._dev(stage_sel, torch.int32)
        n = self._dev(exec_sel, torch.int32)
        lg = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        en = torch.empty(self.num_envs, dtype=torch.float32, device=self.device)
        nat.check(self.L.ssb_decima_evaluate(self._h, snapshot.data_ptr() if snapshot is not None else None,
                                             a.data_ptr(), n.data_ptr(), lg.data_ptr(),
                                             en.data_ptr(), self._stream()), "ssb_decima_evaluate")
        return lg, en

    def decima_head_adjoint(self, grad_lgprob: torch.Tensor, grad_entropy: torch.Tensor):
        """First stage of evaluate_actions' backward pass: d loss / d scores of the stage head [B, node_stride] and of
        the executor-count head [B, exec_stride] from d loss / d lgprob, d loss / d entropy (f32[B]), for the scores
        and actions of the last decima_evaluate / decima_policy call."""
        for t in (grad_lgprob, grad_entropy):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == self.num_envs
        gs = torch.empty_like(self.pol_stage_logits)
        ge = torch.empty_like(self.pol_exec_logits)
        nat.check(self.L.ssb_decima_head_adjoint(self._h, grad_lgprob.data_ptr(), grad_entropy.data_ptr(),
                                                 gs.data_ptr(), ge.data_ptr(), self._stream()),
                  "ssb_decima_head_adjoint")
        return gs, ge

    def decima_head_backward(self, grad_stage_logits: torch.Tensor, grad_exec_logits: torch.Tensor,
                             grad_weights: torch.Tensor, want_inputs: bool = False):
        """Second stage of the backward pass: the two score heads' MLPs.  Accumulates their weight / bias gradients
        into grad_weights (f32[20802], ABI layout) and returns d loss / d input row of the stage head
        [num candidates, 56] and of the executor-count head [num rows, 40] (list order); with want_inputs also the
        gathered input rows."""
        assert grad_weights.is_cuda and grad_weights.dtype == torch.float32 and grad_weights.numel() == 20802
        B = self.num_envs
        S, Ep = self.pol_stage_logits.shape[1], self.pol_exec_logits.shape[1]
        gxs = torch.zeros(B * S, 56, dtype=torch.float32, device=self.device)
        gxe = torch.zeros(B * Ep, 40, dtype=torch.float32, device=self.device)
        xs = torch.zeros_like(gxs) if want_inputs else None
        xe = torch.zeros_like(gxe) if want_inputs else None
        n = (C.c_int32 * 2)()
        nat.check(self.L.ssb_decima_head_backward(
            self._h, grad_stage_logits.data_ptr(), grad_exec_logits.data_ptr(), grad_weights.data_ptr(),
            gxs.data_ptr(), gxe.data_ptr(), xs.data_ptr() if want_inputs else None,
            xe.data_ptr() if want_inputs else None, n, self._stream()), "ssb_decima_head_backward")
        out = (gxs[:n[0]], gxe[:n[1]])
        return out + (xs[:n[0]], xe[:n[1]]) if want_inputs else out

    def decima_backward(self, grad_lgprob: torch.Tensor, grad_entropy: torch.Tensor, grad_weights: torch.Tensor,
                        through_node_encoder: bool = True):
        """evaluate_actions' backward pass for the last decima_evaluate / decima_policy call: accumulates the
        gradients of all 42 tensors into grad_weights (f32[20802], ABI layout).  through_node_encoder=False stops
        above NodeEncoder (score heads, global and job summaries only) and returns d loss / d node embeddings
        [B, node_stride, 16]; otherwise the returned buffer is working storage."""
        assert grad_weights.is_cuda and grad_weights.dtype == torch.float32 and grad_weights.numel() == 20802
        self._backward_scratch()
        d_h = torch.empty(self.num_envs, self.pol_stage_logits.shape[1], 16, dtype=torch.float32, device=self.device)
        nat.check(self.L.ssb_decima_backward(self._h, grad_lgprob.data_ptr(), grad_entropy.data_ptr(),
                                             grad_weights.data_ptr(), d_h.data_ptr(), int(through_node_encoder),
                                             self._bwd_scratch.data_ptr(), self._stream()), "ssb_decima_backward")
        return d_h

    def rollout_decima(self, num_decisions, max_events=0, out: "torch.Tensor | None" = None,
                       host: "torch.Tensor | None" = None, store=None):
        """Decima rollout collection on the device: num_decisions x { decima_policy ; step } with every call's
        (wall time, action, lgprob, reward, flags) recorded -- the RolloutBuffer of
        trainers/rollout_worker.py:18-46; with `store` (a ppo.RolloutStore of this handle with room for num_decisions)
        also the observations and Decima-format actions, row d in its block d.  Finished envs follow set_autoreset().
        Returns the device tensor, or with `host` (pinned uint8) a structured array [B, num_decisions]."""
        return self._with_store(store, lambda: self._recorded(num_decisions, out, host, lambda traj: nat.check(
            self.L.ssb_rollout_decima(self._h, int(num_decisions), int(max_events), traj, self._stream()),
            "ssb_rollout_decima")))

    def rollout_decima_async(self, max_decisions, rollout_duration, seed_step=1, store=None):
        """Fixed-duration Decima rollouts spanning resets (RolloutWorkerAsync.collect_rollout, rollout_worker.py:160-206).
        With `store` (a ppo.RolloutStore of this handle with room for max_decisions) env b's row d also stores its
        observation and Decima-format action in the store's block d.
        Returns (traj uint8 device tensor [B * max_decisions * 32], num_steps i32[B], elapsed f64[B])."""
        nbytes = self.num_envs * int(max_decisions) * nat.TRANSITION_DTYPE.itemsize
        traj = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        num = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
        el = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        self._with_store(store, lambda: nat.check(self.L.ssb_rollout_decima_async(
            self._h, int(max_decisions), float(rollout_duration), int(seed_step), traj.data_ptr(), num.data_ptr(),
            el.data_ptr(), self._stream()), "ssb_rollout_decima_async"))
        return traj, num, el

    def load_trace(self, b, t_arrival, template, tape=None):
        ta = np.ascontiguousarray(t_arrival, np.float64)
        tm = np.ascontiguousarray(template, np.int32)
        tp = None if tape is None else np.ascontiguousarray(tape, np.float64)
        nat.check(self.L.ssb_load_trace(self._h, int(b), len(ta), ta.ctypes.data, tm.ctypes.data,
                                        tp.ctypes.data if tp is not None else None,
                                        0 if tp is None else len(tp)), "ssb_load_trace")

    def clear_trace(self, b):
        nat.check(self.L.ssb_clear_trace(self._h, int(b)), "ssb_clear_trace")

    def jobs(self, b: int = 0, with_state: bool = False):
        """(t_arrival, t_completed, template[, state]) of every job of environment b."""
        n = C.c_int32()
        cap = self.max_jobs
        ta, tc, tm = np.zeros(cap), np.zeros(cap), np.zeros(cap, np.int32)
        st = np.zeros(cap, np.uint8)
        nat.check(self.L.ssb_get_jobs(self._h, int(b), C.byref(n), ta.ctypes.data, tc.ctypes.data,
                                      tm.ctypes.data, st.ctypes.data, cap), "ssb_get_jobs")
        k = n.value
        if with_state:
            return ta[:k], tc[:k], tm[:k], st[:k]
        return ta[:k], tc[:k], tm[:k]

    def history(self, b: int = 0) -> dict:
        """Every Executor.add_history call of env b's current episode in call order (executor.py:34-44):
        hist_t (wall time), hist_exec, hist_job (-1 = common pool).  Needs history_capacity > 0."""
        if self.history_capacity <= 0:
            raise RuntimeError("executor history is not recorded: construct the env with history_capacity > 0")
        n = C.c_int64()
        cap = max(self.history_capacity, 1)
        t, ex, jb = np.zeros(cap), np.zeros(cap, np.int16), np.zeros(cap, np.int16)
        nat.check(self.L.ssb_get_history(self._h, int(b), C.byref(n), t.ctypes.data, ex.ctypes.data,
                                         jb.ctypes.data, cap), "ssb_get_history")
        if n.value > self.history_capacity:
            raise RuntimeError(f"executor history overflow: {n.value} rows > history_capacity {self.history_capacity}")
        k = int(n.value)
        return {"hist_t": t[:k], "hist_exec": ex[:k].astype(np.int32), "hist_job": jb[:k].astype(np.int32)}

    def executor_histories(self, b: int = 0) -> list:
        """`[executor.history for executor in env.executors]` in the reference's format (spark_sched_sim.py:411):
        per executor [[t_release, job_id], ..., [None, job_id]], job_id -1 = common pool."""
        h = self.history(b)
        out = [[[None, -1]] for _ in range(self.num_executors)]
        for t, e, j in zip(h["hist_t"], h["hist_exec"], h["hist_job"]):
            out[e][-1][0] = float(t)
            out[e].append([None, int(j)])
        return out

    def log_size(self, b: int = 0) -> int:
        n = C.c_int64()
        nat.check(self.L.ssb_get_log(self._h, int(b), 0, 0, C.byref(n), *([None] * 7)), "ssb_get_log")
        return int(n.value)

    def log(self, b: int = 0, lo: int = 0, hi: int | None = None) -> dict:
        n = self.log_size(b)
        hi = n if hi is None else hi
        k = hi - lo
        out = {"ev_t": np.zeros(k), "ev_type": np.zeros(k, np.uint8), "ev_job": np.zeros(k, np.int16),
               "ev_stage": np.zeros(k, np.int16), "ev_task": np.zeros(k, np.int32),
               "ev_exec": np.zeros(k, np.int16), "ev_tacc": np.zeros(k)}
        nn = C.c_int64()
        if k > 0:
            nat.check(self.L.ssb_get_log(
                self._h, int(b), lo, hi, C.byref(nn),
                *[out[x].ctypes.data for x in ("ev_t", "ev_type", "ev_job", "ev_stage", "ev_task",
                                               "ev_exec", "ev_tacc")]), "ssb_get_log")
        return out
