"""One Decima policy call at mid-episode (decision 60) inside a cudaProfilerStart/Stop range, for
    ncu --profile-from-start off --set full --import-source on -k regex:k_tile3 ... python profiles/policy_ncu_target.py"""
import os.path as osp
import sys

REPO = osp.dirname(osp.dirname(osp.abspath(__file__)))
sys.path.insert(0, REPO)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv  # noqa: E402

cfg = {"num_executors": 10, "job_arrival_cap": 50, "job_arrival_rate": 4.0e-5, "moving_delay": 2000.0, "warmup_delay": 1000.0}
B = 4096
env = BatchedSparkSchedSimEnv(cfg, num_envs=B, decima_policy=True)
z = np.load(osp.join(REPO, "tests", "golden", "decima_model.npz"))
env.set_decima_weights({k: z[k] for k in z.files})
env.reset_host((1234 + np.arange(B)).astype(np.uint64))
for _ in range(60):
    a, c = env.decima_policy()
    env.step(a, c)
torch.cuda.synchronize()
torch.cuda.profiler.start()
env.decima_policy()
torch.cuda.synchronize()
torch.cuda.profiler.stop()
