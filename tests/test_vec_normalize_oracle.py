"""CPU tests of oracle/vec_normalize.py, the NumPy restatement of SB3's VecNormalize / RunningMeanStd that the device
implementation is checked against: the running merge against closed forms, and a two-step example by hand."""
from fractions import Fraction as F

import numpy as np
import pytest

from oracle.vec_normalize import RunningMeanStd, VecNormalize


@pytest.mark.parametrize("k", [1, 2, 7])
def test_merging_batches_equals_closed_form_with_prior(k):
    """Merging k batches through update_from_moments gives the mean / variance of their concatenation, pooled with the
    prior (count 1e-4, mean 0, var 1) as one more group."""
    rng = np.random.default_rng(k)
    batches = [rng.normal(3.0, 2.0, (int(rng.integers(1, 50)), 4)) for _ in range(k)]
    rms = RunningMeanStd(shape=(4,))
    for b in batches:
        rms.update(b)
    x = np.concatenate(batches)
    n, c0 = len(x), 1e-4
    mu = x.mean(axis=0)
    tot = c0 + n
    mean = n * mu / tot
    m2 = c0 * 1.0 + ((x - mu) ** 2).sum(axis=0) + mu ** 2 * c0 * n / tot
    np.testing.assert_allclose(rms.mean, mean, rtol=1e-12)
    np.testing.assert_allclose(rms.var, m2 / tot, rtol=1e-12)
    assert rms.count == pytest.approx(tot, rel=1e-15)


def test_two_step_example_by_hand():
    """Batches [1, 3] then [5] of a one-dimensional observation, in exact rational arithmetic."""
    rms = RunningMeanStd(shape=(1,))
    rms.update(np.array([[1.0], [3.0]]))
    rms.update(np.array([[5.0]]))
    c = F(1, 10000)
    # step 1: batch mean 2, var 1, n 2
    t1 = c + 2
    mean1 = 0 + F(2) * 2 / t1
    var1 = (1 * c + 1 * 2 + F(2) ** 2 * c * 2 / t1) / t1
    # step 2: batch mean 5, var 0, n 1
    d2 = 5 - mean1
    t2 = t1 + 1
    mean2 = mean1 + d2 * 1 / t2
    var2 = (var1 * t1 + 0 + d2 ** 2 * t1 * 1 / t2) / t2
    assert rms.mean[0] == pytest.approx(float(mean2), rel=1e-15)
    assert rms.var[0] == pytest.approx(float(var2), rel=1e-14)
    assert rms.count == pytest.approx(float(t2), rel=1e-15)


class _Venv:
    def __init__(self, batches):
        self.num_envs = batches[0][0].shape[0]
        self._b = list(batches)

    def reset(self):
        return self._b.pop(0)[0]

    def step_async(self, actions):
        pass

    def step_wait(self):
        return self._b.pop(0)


def test_step_wait_order_of_operations():
    """returns = returns*gamma + reward before ret_rms.update; terminal rows use the updated obs statistics; returns of
    finished envs are zeroed after the reward is normalised."""
    obs0 = np.array([[1.0], [2.0]], np.float32)
    obs1 = np.array([[4.0], [0.0]], np.float32)
    rew1 = np.array([1.0, -2.0], np.float32)
    done1 = np.array([False, True])
    term = np.array([7.0], np.float32)
    venv = _Venv([(obs0,), (obs1, rew1, done1, [{}, {"terminal_observation": term}])])
    vn = VecNormalize(venv, obs_shape=(1,), gamma=0.5)
    vn.reset()
    o, r, d, infos = vn.step(None)
    ref = RunningMeanStd(shape=(1,))
    ref.update(obs0)
    ref.update(obs1)
    den = np.sqrt(ref.var + 1e-8)
    np.testing.assert_array_equal(o, np.clip((obs1 - ref.mean) / den, -10, 10).astype(np.float32))
    np.testing.assert_array_equal(infos[1]["terminal_observation"], np.clip((term - ref.mean) / den, -10, 10).astype(np.float32))
    ret = RunningMeanStd()
    ret.update(np.zeros(2) * 0.5 + rew1)
    np.testing.assert_array_equal(r, np.clip(rew1 / np.sqrt(ret.var + 1e-8), -10, 10))
    np.testing.assert_array_equal(vn.returns, [1.0, 0.0])
    np.testing.assert_array_equal(vn.get_original_obs(), obs1)
