"""CPU tests of oracle/rollout_buffer.py, the NumPy restatement of SB3's RolloutBuffer and collect_rollouts loop that the
device implementation is checked against: GAE against its definitions in float64, the env-major sample order, the
minibatch iteration, and the bookkeeping of the collection loop."""
import numpy as np
import pytest

from oracle.rollout_buffer import RolloutBuffer, collect_rollouts


def _filled(T, E, gamma, lam, p_start=0.1, seed=0, D=3, N=2):
    rng = np.random.default_rng(seed)
    buf = RolloutBuffer(T, D, N, gae_lambda=lam, gamma=gamma, n_envs=E)
    for t in range(T):
        start = np.ones(E, bool) if t == 0 else rng.random(E) < p_start
        buf.add(rng.standard_normal((E, D)), rng.standard_normal((E, N)), rng.uniform(0, 1, E).astype(np.float32), start,
                rng.uniform(0, 1, (E, 1)).astype(np.float32), rng.standard_normal(E).astype(np.float32))
    last_values = rng.uniform(0, 1, E).astype(np.float32)
    dones = rng.random(E) < 0.3
    return buf, last_values, dones


def _f64(buf):
    return (buf.rewards.astype(np.float64), buf.values.astype(np.float64), buf.episode_starts.astype(np.float64))


@pytest.mark.parametrize("gamma", [0.99, 0.9, 1.0])
def test_lambda_one_gives_discounted_returns(gamma):
    """gae_lambda = 1: returns are the discounted rewards to the end of each episode, bootstrapped from last_values where
    the episode runs past the buffer."""
    T, E = 20, 7
    buf, lv, dones = _filled(T, E, gamma, 1.0)
    buf.compute_returns_and_advantage(lv, dones)
    r, v, s = _f64(buf)
    want = np.zeros((T, E))
    nxt = lv.astype(np.float64) * (1.0 - dones)
    for t in reversed(range(T)):
        want[t] = r[t] + gamma * nxt
        nxt = want[t] * (1.0 - s[t])
    np.testing.assert_allclose(buf.returns, want, rtol=1e-5)
    np.testing.assert_array_equal(buf.returns, buf.advantages + buf.values)


def test_lambda_zero_gives_td_errors():
    T, E, gamma = 12, 9, 0.95
    buf, lv, dones = _filled(T, E, gamma, 0.0, seed=1)
    buf.compute_returns_and_advantage(lv, dones)
    r, v, s = _f64(buf)
    nv = np.concatenate([v[1:], lv[None].astype(np.float64)])
    nnt = np.concatenate([1.0 - s[1:], (1.0 - dones)[None]])
    np.testing.assert_allclose(buf.advantages, r + gamma * nv * nnt - v, rtol=1e-5, atol=1e-6)


def test_episode_start_cuts_the_bootstrap():
    """An episode start at step k: nothing at or after k reaches the advantages before k, and with gae_lambda = 1 the
    return at k-1 is its reward alone."""
    T, E, k = 16, 4, 9
    a, lv, dones = _filled(T, E, 0.99, 1.0, p_start=0.0, seed=2)
    b, _, _ = _filled(T, E, 0.99, 1.0, p_start=0.0, seed=2)
    for buf in (a, b):
        buf.episode_starts[k, 1] = 1.0
    rng = np.random.default_rng(3)
    b.rewards[k:, 1] = rng.uniform(-5, 5, T - k)
    b.values[k:, 1] = rng.uniform(-5, 5, T - k)
    a.compute_returns_and_advantage(lv, dones)
    b.compute_returns_and_advantage(lv, dones)
    np.testing.assert_array_equal(a.advantages[:k, 1], b.advantages[:k, 1])
    assert a.returns[k - 1, 1] == pytest.approx(a.rewards[k - 1, 1], rel=1e-6)
    assert not np.array_equal(a.advantages[k:, 1], b.advantages[k:, 1])


def test_swap_and_flatten_is_env_major():
    T, E, D = 5, 3, 2
    arr = np.arange(T * E * D).reshape(T, E, D)
    flat = RolloutBuffer.swap_and_flatten(arr)
    for k in range(T * E):
        np.testing.assert_array_equal(flat[k], arr[k % T, k // T])
    flat1 = RolloutBuffer.swap_and_flatten(np.arange(T * E).reshape(T, E))
    assert flat1.shape == (T * E, 1)
    assert [int(x) for x in flat1[:, 0]] == [(k % T) * E + k // T for k in range(T * E)]


def test_get_visits_every_index_once_with_a_short_last_batch():
    T, E, bs = 6, 5, 7
    buf, lv, dones = _filled(T, E, 0.99, 0.95, seed=4)
    buf.compute_returns_and_advantage(lv, dones)
    tagged = np.arange(T * E, dtype=np.float32).reshape(E, T).T     # flat k carries the value k after the flatten
    buf.log_probs[...] = tagged
    np.random.seed(0)
    batches = list(buf.get(bs))
    assert [len(b[0]) for b in batches] == [7, 7, 7, 7, 2]
    seen = np.concatenate([b[3] for b in batches]).astype(np.int64)
    assert sorted(seen.tolist()) == list(range(T * E))
    perm = np.random.default_rng(1).permutation(T * E)
    (whole,) = list(buf.get(None, indices=perm))
    np.testing.assert_array_equal(whole[3], perm.astype(np.float32))


def test_collect_rollouts_loop_bookkeeping():
    """Unclipped actions stored, the env stepped with clipped ones, episode starts = the previous dones, GAE at the end."""
    T, E, D, N = 4, 3, 2, 2
    rng = np.random.default_rng(5)
    stepped, done_seq = [], [rng.random(E) < 0.5 for _ in range(T)]
    acts = [rng.uniform(-3, 3, (E, N)).astype(np.float32) for _ in range(T)]
    k = [0]

    def policy(obs):
        a = acts[k[0]]
        return a, obs[:, :1].astype(np.float32), np.full(E, -1.0, np.float32)

    def env_step(a):
        stepped.append(a)
        d = done_seq[k[0]]
        k[0] += 1
        return np.full((E, D), k[0], np.float32), np.full(E, 0.5, np.float32), d, [{} for _ in range(E)]

    buf = RolloutBuffer(T, D, N, gae_lambda=0.9, gamma=0.9, n_envs=E)
    obs0 = np.zeros((E, D), np.float32)
    last_obs, last_starts = collect_rollouts(env_step, policy, lambda o: o[:, 0].astype(np.float32), buf, T, obs0,
                                             np.ones(E, bool), gamma=0.9)
    assert buf.full
    for t in range(T):
        np.testing.assert_array_equal(buf.actions[t], acts[t])
        np.testing.assert_array_equal(stepped[t], np.clip(acts[t], -1, 1))
        np.testing.assert_array_equal(buf.episode_starts[t], np.ones(E) if t == 0 else done_seq[t - 1])
        np.testing.assert_array_equal(buf.observations[t], np.full((E, D), t, np.float32))
    np.testing.assert_array_equal(last_starts, done_seq[-1])
    ref, lv = RolloutBuffer(T, D, N, gae_lambda=0.9, gamma=0.9, n_envs=E), last_obs[:, 0]
    for name in ("rewards", "values", "episode_starts"):
        setattr(ref, name, getattr(buf, name).copy())
    ref.full = True
    ref.compute_returns_and_advantage(lv, done_seq[-1])
    np.testing.assert_array_equal(buf.advantages, ref.advantages)
