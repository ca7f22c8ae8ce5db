"""float64 references of the rollout statistics (plain helper module of tests/test_gpu_advantage_moments.py and
tests/test_cpu_torque_obs_probe.py): advantage normalisation with torch's unbiased std, two-pass column moments with
the population variance (numpy's np.var, as RunningMeanStd.update takes them), and RunningMeanStd itself
(rsl_rl/rsl_rl/utils/utils.py:79-110, UT) on float64 batches."""
import numpy as np

from oracle import torch_oracle as O


def normalize64(a, ddof=1):
    """(a - mean) / (std + 1e-8) in float64, std with `ddof` (1: torch's default).  One element and ddof 1: 0/0 = NaN,
    as torch's std() of one element."""
    a = np.asarray(a, dtype=np.float64).ravel()
    m = a.size
    mean = a.sum() / m
    with np.errstate(divide="ignore", invalid="ignore"):
        var = np.square(a - mean).sum() / np.float64(m - ddof)
        return (a - mean) / (np.sqrt(var) + 1e-8)


def moments64(x):
    """Two-pass float64 column mean and population variance of a (rows, dim) batch."""
    x = np.asarray(x, dtype=np.float64)
    mean = x.mean(axis=0)
    return mean, np.square(x - mean).mean(axis=0)


class RunningMeanStd64:
    """UT:79-110 with float64 batches: mean 0, var 1, count 1e-4 to start, Chan's parallel merge per update."""

    def __init__(self, dim):
        self.mean, self.var, self.count = np.zeros(dim), np.ones(dim), 1e-4

    def update(self, arr):
        self.mean, self.var, self.count = O.running_moments_update(self.mean, self.var, self.count,
                                                                   np.asarray(arr, dtype=np.float64))
