"""bench.py --dump-outputs: the files dump_outputs writes after a fused rollout are what the env's own accessors return,
float32 / float64 only, within the size limit (a sample of the envs when all of them do not fit); through the command
line, two runs with the same arguments write identical files."""
import json
import subprocess
import sys

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("limit", [bench.DUMP_LIMIT, 256 << 10])
def test_dump_outputs_match_the_env(tmp_path, bank, limit):
    from spark_sched_sim_b200 import _native as nat
    from spark_sched_sim_b200.batched_env import BatchedSparkSchedSimEnv

    B = 64
    env = BatchedSparkSchedSimEnv(bench.ENV_CFG, num_envs=B, bank=bank)
    env.reset_host(np.arange(1234, 1234 + B, dtype=np.uint64))
    env.reset_stats()
    env.rollout_fair(40, True, True, B)
    stats = env.collect_stats()
    names = bench.dump_outputs(env, stats, str(tmp_path), limit=limit)
    d = {k: np.load(tmp_path / f"{k}.npy") for k in names}
    assert all(v.dtype in (np.float32, np.float64) for v in d.values())
    assert sum((tmp_path / f"{k}.npy").stat().st_size for k in names) <= limit
    envs = d["env_ids"].astype(np.int64)
    assert 0 < len(envs) and np.all(np.diff(envs) > 0) and (len(envs) == B) == (limit == bench.DUMP_LIMIT)

    h, st = env.hdr(), env.stats_per_env()
    for f in h.dtype.names:
        assert np.array_equal(d[f], h[f][envs].astype(np.float64)), f
    for f in nat.STATS_FIELDS:
        assert np.array_equal(d[f"stats_{f}"], st[f][envs].astype(np.float64)), f
    assert np.array_equal(d["rollout_stats"], stats.cpu().numpy())
    at = dict.fromkeys(("nodes", "edge_links", "dag_ptr", "exec_supplies"), 0)
    for b in envs:
        o = env.obs(int(b), h)
        for k in at:
            n = len(o[k])
            assert np.array_equal(d[k][at[k]:at[k] + n], o[k]), (b, k)
            at[k] += n
    assert all(at[k] == len(d[k]) for k in at)
    assert d["nodes"].dtype == np.float32 and h["num_nodes"][envs].sum() > 0
    env.close()


def test_bench_cli_dump_is_reproducible(tmp_path):
    """bench.py end to end (main -> run_c2 -> dump_outputs): two runs with the same arguments write identical files,
    and --steps sets the timed steps (every env took steps x DECISIONS_PER_STEP decisions after reset_stats)."""
    B, steps = 256, 2
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        r = subprocess.run([sys.executable, bench.__file__, "--gpus", "1", "--steps", str(steps), "--warmup", "0",
                            "--envs", str(B), "--configs", "none", "--no-e2e", "--cpu-seconds", "0",
                            "--dump-outputs", str(d)], cwd=tmp_path, check=True, stdout=subprocess.PIPE, text=True,
                           timeout=900)
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["env_errors"] == 0
    names = sorted(p.name for p in dirs[0].iterdir())
    assert names == sorted(p.name for p in dirs[1].iterdir()) and "nodes.npy" in names
    for f in names:
        assert (dirs[0] / f).read_bytes() == (dirs[1] / f).read_bytes(), f
    assert np.array_equal(np.load(dirs[0] / "env_ids.npy"), np.arange(B))
    assert np.all(np.load(dirs[0] / "stats_decisions.npy") == steps * bench.DECISIONS_PER_STEP)
