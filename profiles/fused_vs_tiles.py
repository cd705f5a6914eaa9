"""Development aid: the fused policy kernel (MODE_A, default 1) against the list-driven tile path (MODE_B, default 0) on
the same states (two handles driven with the same actions); prints the first step / environments where candidates,
actions or scores differ."""
import os
import os.path as osp
import sys

import numpy as np

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, osp.join(REPO, "tests"))
from helpers import load_golden  # noqa: E402
from spark_sched_sim_b200.bank import synthetic_bank  # noqa: E402
from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

B = int(os.environ.get("REPRO_B", "2048"))
steps = int(os.environ.get("REPRO_STEPS", "400"))
FOLLOW_FUSED = os.environ.get("FOLLOW_FUSED", "0") == "1"
tr = load_golden("decima_e10_j8_s5_philox")
cfg = {"num_executors": 10, "job_arrival_cap": 8, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0, "warmup_delay": 1000.0}
z = np.load(osp.join(REPO, "tests", "golden", "decima_model.npz"))
envs = []
for tiles in (0, 1):
    os.environ["SSB_DECIMA_MODE"] = str(int(os.environ.get("MODE_B", "0")) if tiles else int(os.environ.get("MODE_A", "1")))
    e = BatchedSparkSchedSimEnv(cfg, num_envs=B, bank=synthetic_bank(0), max_jobs=10, tape_capacity=len(tr["tape"]) + 8,
                                decima_policy=True)
    e.set_decima_weights({k: z[k] for k in z.files})
    for b in range(B):
        e.load_trace(b, tr["job_t_arrival"], tr["job_template"], tr["tape"])
    e.reset_host(np.arange(B, dtype=np.uint64) + 5)
    envs.append(e)
f, t = envs
for k in range(steps):
    a, n = f.decima_policy()
    a2, n2 = t.decima_policy()
    fa, ta = f.pol_action.cpu().numpy(), t.pol_action.cpu().numpy()
    hf = f.hdr()
    live = (hf["terminated"] == 0) & (hf["error"] == 0)
    bad = np.flatnonzero(((fa != ta).any(1)) & live)
    sl_f, sl_t = f.pol_stage_logits.cpu().numpy(), t.pol_stage_logits.cpu().numpy()
    worst = 0.0
    for b in np.flatnonzero(live)[:4096]:
        nc = ta[b, 3]
        if nc > 0:
            worst = max(worst, float(np.abs(sl_f[b, :nc] - sl_t[b, :nc]).max()))
    if (len(bad) and not FOLLOW_FUSED) or worst > float(os.environ.get("WORST_TOL", "1e-3")):
        print(f"step {k}: {len(bad)} envs differ, worst score diff {worst:.3g}; first:", bad[:8])
        for b in bad[:3]:
            print("  env", b, "fused", fa[b], "tiles", ta[b], "N", hf["num_nodes"][b], "nsched", hf["num_schedulable"][b])
            nc = max(ta[b, 3], 1)
            print("   fused logits", sl_f[b, :nc][:8], "\n   tiles logits", sl_t[b, :nc][:8])
        break
    av, nv, a2v, n2v = a.cpu().numpy(), n.cpu().numpy(), a2.cpu().numpy(), n2.cpu().numpy()
    if FOLLOW_FUSED:
        if ((av != fa[:, 0]) | (nv != fa[:, 2] + 1)).any():
            w = np.flatnonzero((av != fa[:, 0]) | (nv != fa[:, 2] + 1))
            print(f"step {k}: outputs differ from pol_action in envs", w[:8], av[w[:4]], nv[w[:4]], fa[w[:4]])
            break
        f.step(a, n)
        t.step(a, n)
        hf2, ht2 = f.hdr(), t.hdr()
        if ((hf2["error"] != 0) & (hf2["error"] != 9)).any() or (hf2["wall_time"] != ht2["wall_time"]).any():
            w = np.flatnonzero(((hf2["error"] != 0) & (hf2["error"] != 9)) | (hf2["wall_time"] != ht2["wall_time"]))
            print(f"step {k}: after step, envs", w[:8], "errors fused-handle", hf2["error"][w[:8]], "tiles-handle", ht2["error"][w[:8]],
                  "actions", av[w[:4]], nv[w[:4]], "nsched", hf["num_schedulable"][w[:4]], "ncand", fa[w[:4], 3])
            break
        continue
    f.step(a2, n2)   # both handles follow the tile path's actions
    t.step(a2, n2)
    if not live.any():
        print("all finished at", k)
        break
print("done", k)
