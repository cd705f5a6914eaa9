"""parallel.stats_from_sums with the episode log's entries of the ssb_collect_stats vector ([6] sum of the envs'
window means in ms, [7] the number of such envs): the trainer's mean over workers of env.avg_job_duration."""
import numpy as np


def test_stats_from_sums_uses_window_means():
    from spark_sched_sim_b200 import parallel

    windows = [np.array([1500.0, 2500.0, 4000.0]), np.array([800.0]), np.array([12000.0, 3000.0])]
    means = [w.mean() for w in windows]
    vec = [6.0, 3.0, 10.0, 14.0, 50000.0, 9.0e5, sum(means), 3.0]
    st = parallel.stats_from_sums(vec)
    assert abs(st["avg_job_duration"] - np.mean([m * 1e-3 for m in means])) <= 1e-15
    assert st["avg_num_jobs"] == 2.0 and st["num_completed_jobs"] == 10.0 / 3.0


def test_stats_from_sums_without_window_is_unchanged():
    from spark_sched_sim_b200 import parallel

    vec = [6.0, 3.0, 10.0, 14.0, 50000.0, 9.0e5, 0.0, 0.0]
    assert parallel.stats_from_sums(vec)["avg_job_duration"] == 50000.0 / 10.0 * 1e-3
    assert parallel.stats_from_sums(vec[:6])["avg_job_duration"] == 50000.0 / 10.0 * 1e-3
    assert np.isnan(parallel.stats_from_sums([0.0] * 8)["avg_job_duration"])
