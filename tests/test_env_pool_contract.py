"""B200VecEnv's env-pool shape checks run before any CUDA call: a bad envs_per_batch fails on a machine without a GPU."""
import pytest

from nmmo_b200.vecenv import B200VecEnv


@pytest.mark.parametrize("num_envs,envs_per_batch", [(15, 6), (8, 3), (4, 0), (4, 5), (4, -2), (0, 1)])
def test_envs_per_batch_must_divide_num_envs(num_envs, envs_per_batch):
    with pytest.raises(ValueError, match="envs_per_batch"):
        B200VecEnv(num_envs=num_envs, envs_per_batch=envs_per_batch)
