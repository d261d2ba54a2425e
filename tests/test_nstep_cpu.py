"""The n-step target of the oracle (nstep_oracle.nstep_targets, nstep_oracle.loss_and_grads) without a GPU:
n = 1 reproduces the 1-step y bit for bit, and hand-worked windows pin the truncation at a terminal."""
import numpy as np
import pytest

from oracle import nstep_oracle as no

G = 0.99


def _one_step_y(r, term, x, gamma=G):
    """qnet_oracle.loss_and_grads' 1-step target, sample by sample"""
    r = np.array([0.1 if abs(float(v) - 0.1) < 1e-6 else float(v) for v in r], np.float64)
    return np.where(np.asarray(term).astype(bool), r, r + gamma * x).astype(np.float32)


def _nstep_y(R, d, x):
    R, d = np.asarray(R, np.float64), np.asarray(d, np.float64)
    return np.where(d == 0.0, R, R + d * x).astype(np.float32)


def test_n1_equals_the_one_step_target():
    rng = np.random.default_rng(0)
    T, N = 60, 16
    rew = rng.choice(np.array([0.1, 3.0, -3.0, 0.0], np.float32), (T + 1, N), p=[0.7, 0.1, 0.1, 0.1])
    term = (rng.random((T + 1, N)) < 0.15).astype(np.uint8)
    x = rng.standard_normal(T * N).astype(np.float32).astype(np.float64)
    ks = np.repeat(np.arange(1, T + 1), N)
    es = np.tile(np.arange(N), T)
    Rd = [no.nstep_targets(rew, term, e, k, 1, G) for e, k in zip(es, ks)]
    R, d = np.array([a for a, _ in Rd]), np.array([b for _, b in Rd])
    np.testing.assert_array_equal(R, [0.1 if rew[k, e] == np.float32(0.1) else float(rew[k, e]) for e, k in zip(es, ks)])
    np.testing.assert_array_equal(d, np.where(term[ks, es] != 0, 0.0, G))
    y1 = _one_step_y(rew[ks, es], term[ks, es], x)
    yn = _nstep_y(R, d, x)
    assert y1.tobytes() == yn.tobytes()


def test_hand_worked_windows():
    # env 0, steps 1..6: rewards 0.1, 0.1, 3, 0.1, -3, 0.1, terminal at step 5
    rew = np.zeros((8, 1), np.float32)
    rew[1:7, 0] = [0.1, 0.1, 3.0, 0.1, -3.0, 0.1]
    term = np.zeros((8, 1), np.uint8)
    term[5, 0] = 1
    g = 0.5
    # no terminal in the window: R = 0.1 + g 0.1 + g^2 3, disc = g^3
    assert no.nstep_targets(rew, term, 0, 1, 3, g) == (0.1 + 0.5 * 0.1 + 0.25 * 3.0, 0.125)
    # terminal in the middle of the window (k = 3, n = 4: steps 3, 4, 5 | 6 dropped)
    assert no.nstep_targets(rew, term, 0, 3, 4, g) == (3.0 + 0.5 * 0.1 + 0.25 * -3.0, 0.0)
    # terminal at the last step of the window (k = 3, n = 3)
    assert no.nstep_targets(rew, term, 0, 3, 3, g) == (3.0 + 0.5 * 0.1 + 0.25 * -3.0, 0.0)
    # terminal at the first step: the 1-step terminal target whatever n is
    assert no.nstep_targets(rew, term, 0, 5, 2, g) == (-3.0, 0.0)
    # the window starts after the terminal
    assert no.nstep_targets(rew, term, 0, 6, 1, g) == (0.1, 0.5)


def test_forward_accumulation_order():
    """R is accumulated forward with the running product, as the gather kernel does -- not as a closed-form power series"""
    rew = np.full((20, 1), 0.1, np.float32)
    term = np.zeros((20, 1), np.uint8)
    R, d = no.nstep_targets(rew, term, 0, 1, 16, G)
    want_R, g = 0.0, 1.0
    for _ in range(16):
        want_R += g * 0.1
        g *= G
    assert (R, d) == (want_R, g)


@pytest.mark.parametrize("n", [1, 3, 5])
def test_loss_and_grads_takes_the_nstep_target(n):
    """nstep_oracle.loss_and_grads uses y = R (+ disc X): with R = r and disc = gamma * (1 - term) it is qnet_oracle's 1-step
    computation exactly, for every variant and with IS weights"""
    pytest.importorskip("torch")
    from oracle import qnet_oracle as qo
    rng = np.random.default_rng(n)
    B, H = 4, 32
    p = qo.init_params(H, False, seed=1); tg = qo.init_params(H, False, seed=2)
    s = (rng.random((B, 4, 80, 80)) < 0.3).astype(np.uint8) * 255
    s2 = (rng.random((B, 4, 80, 80)) < 0.3).astype(np.uint8) * 255
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = np.array([0.1, 3.0, -3.0, 0.1], np.float32)
    t = np.array([0, 0, 1, 0], np.uint8)
    isw = rng.random(B).astype(np.float32)
    R = np.array([0.1, 3.0, -3.0, 0.1]); d = np.where(t != 0, 0.0, 0.99)
    for variant, w, loss_sum, emulate in ((0, None, True, None), (1, None, False, None), (2, isw, False, None), (1, None, False, "fp16")):
        base = qo.loss_and_grads(variant, p, tg, s, s2, a, r, t, w, 0.99, loss_sum, hidden=H, emulate=emulate)
        same = no.loss_and_grads(variant, p, tg, s, s2, a, R, d, w, loss_sum, hidden=H, emulate=emulate)
        assert base[0] == same[0] and np.array_equal(base[1], same[1]) and np.array_equal(base[3], same[3]), variant
    other = no.loss_and_grads(1, p, tg, s, s2, a, R + 1.0, d * 0.5, hidden=H)
    assert not np.array_equal(base[3], other[3])
