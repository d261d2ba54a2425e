"""The QR-DQN oracle's loss and gradients (oracle/qr_oracle.py) and the C ABI of the quantile head, without a GPU."""
import os
import re
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import qnet_oracle as qo  # noqa: E402
from oracle import qr_oracle as qr  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rows(rng, B, N, spread=3.0):
    th = rng.normal(0.0, spread, (B, N))
    T = rng.normal(0.5, spread, (B, N)).astype(np.float32)
    return th, T


@pytest.mark.parametrize("kappa", [0.0, 0.5, 1.0, 4.0])
@pytest.mark.parametrize("N", [1, 5, 32])
def test_finite_differences_match_the_gradient(N, kappa):
    rng = np.random.default_rng(N)
    th, T = _rows(rng, 6, N)
    g_hand = qr.sample_grad(th, T, kappa)
    t = torch.tensor(th, requires_grad=True)
    qr.sample_loss(t, T, kappa).sum().backward()
    np.testing.assert_allclose(t.grad.numpy(), g_hand, rtol=1e-12, atol=1e-15)
    eps = 1e-6
    for b in range(th.shape[0]):
        for i in range(N):
            # away from the kinks (u = 0, |u| = kappa) the loss is differentiable
            u = T[b].astype(np.float64) - th[b, i]
            if np.min(np.abs(u)) < 1e-3 or (kappa > 0 and np.min(np.abs(np.abs(u) - kappa)) < 1e-3):
                continue
            hi, lo = th.copy(), th.copy()
            hi[b, i] += eps
            lo[b, i] -= eps
            fd = (qr.sample_loss(torch.tensor(hi), T, kappa)[b] - qr.sample_loss(torch.tensor(lo), T, kappa)[b]).item() / (2 * eps)
            assert abs(fd - g_hand[b, i]) <= 1e-6, (b, i, fd, g_hand[b, i])


def test_kappa_zero_is_the_l1_quantile_loss():
    rng = np.random.default_rng(1)
    th, T = _rows(rng, 8, 16)
    u = T.astype(np.float64)[:, None, :] - th[:, :, None]
    check = u * (qr.taus(16)[None, :, None] - (u < 0))           # rho_tau(u) = u (tau - 1{u < 0})
    want = check.sum(-1).sum(-1) / 16
    np.testing.assert_allclose(qr.sample_loss(torch.tensor(th), T, 0.0).numpy(), want, rtol=1e-13)
    assert (want >= 0).all()


@pytest.mark.parametrize("kappa", [0.0, 1.0])
def test_tau_asymmetry_gives_the_sign_of_each_step(kappa):
    """theta_i moves up (negative gradient) exactly when the tau_i-weighted targets above it outweigh the (1 - tau_i)-weighted
    ones below it; with the targets far apart (|u| > kappa everywhere) that is tau_i #above > (1 - tau_i) #below"""
    N = 8
    T = np.arange(N, dtype=np.float32)[None, :] * np.float32(10.0)   # 0, 10, .., 70
    tau = qr.taus(N)
    for v in np.arange(-5.0, 80.0, 10.0):
        th = np.full((1, N), v)
        g = qr.sample_grad(th, T, kappa)[0]
        above, below = (T[0] > v).sum(), (T[0] < v).sum()
        for i in range(N):
            drive = tau[i] * above - (1 - tau[i]) * below
            assert np.sign(-g[i]) == np.sign(drive), (v, i, g[i], drive)
    # the fixed point of quantile i lies between the targets that bracket its fraction: low quantiles below high ones
    th = np.linspace(-5, 75, 81)[:, None].repeat(N, 1)
    g = qr.sample_grad(th, np.repeat(T, 81, 0), kappa)
    zero_cross = [th[np.argmax(g[:, i] > 0), i] for i in range(N)]
    assert all(a <= b for a, b in zip(zero_cross, zero_cross[1:])) and zero_cross[0] < zero_cross[-1]


def test_a_terminal_row_ignores_theta_next():
    rng = np.random.default_rng(3)
    R = np.array([3.0, -3.0, 0.1])
    d = np.array([0.0, 0.0, 0.0])
    T1 = qr.targets(rng.normal(0, 5, (3, 7)).astype(np.float32), R, d)
    T2 = qr.targets(rng.normal(0, 5, (3, 7)).astype(np.float32), R, d)
    assert np.array_equal(T1, T2) and np.array_equal(T1, np.repeat(R.astype(np.float32)[:, None], 7, 1))
    r, dd = qr.one_step_targets(np.float32([0.1, 3.0]), np.uint8([1, 0]), 0.99)
    x = np.float32([[2.0], [1.5]])
    T = qr.targets(x, r, dd)
    assert T[0, 0] == np.float32(0.1) and T[1, 0] == np.float32(3.0 + 0.99 * 1.5)


@pytest.mark.parametrize("kappa", [0.5, 1.0, 16.0])
def test_one_quantile_is_the_scaled_squared_error(kappa):
    """N = 1, every |u| <= kappa: L = (y - Q)^2 / (4 kappa), dL/dQ = -(y - Q) / (2 kappa)"""
    rng = np.random.default_rng(4)
    th = rng.uniform(-0.9, 0.9, (10, 1)) * kappa
    T = np.zeros((10, 1), np.float32)
    u = -th[:, 0]
    np.testing.assert_allclose(qr.sample_loss(torch.tensor(th), T, kappa).numpy(), u * u / (4 * kappa), rtol=1e-13)
    np.testing.assert_allclose(qr.sample_grad(th, T, kappa)[:, 0], -u / (2 * kappa), rtol=1e-13)


def test_loss_and_grads_on_a_small_net():
    """the whole-net oracle: its head gradient is sample_grad routed through the head, Q is the mean of theta, and at N = 1 its
    layout is the expected-value head's"""
    rng = np.random.default_rng(5)
    H, N, B = 32, 6, 5
    params = qr.init_params(H, True, N, seed=1) * np.float32(20.0)
    x = rng.integers(0, 2, (B, 5, 80, 80)).astype(np.uint8) * np.uint8(255)
    acts = rng.integers(0, 2, B).astype(np.uint8)
    R, d = qr.one_step_targets(np.float32([0.1, 3.0, -3.0, 0.1, 0.1]), np.uint8([0, 0, 1, 0, 0]), 0.99)
    loss, g, lb, qt, q, T = qr.loss_and_grads(0, params, None, x[:, 0:4], x[:, 1:5], acts, R, d, None, False, None, H, True, None, N, 1.0)
    th, q2 = qr.forward(params, x[:, 0:4], H, True, N)
    np.testing.assert_allclose(q, q2, rtol=1e-12)
    np.testing.assert_allclose(q, th.mean(-1), rtol=1e-12)
    np.testing.assert_allclose(lb, qr.sample_loss(torch.tensor(th[np.arange(B), acts]), T, 1.0).numpy(), rtol=1e-10)
    assert abs(loss - lb.sum() / B) <= 1e-12 * abs(loss)
    L = qr.layout(H, True, N)
    # dueling: dL/db_v = sum over samples of dL_b/dtheta (both actions' columns share v) / B
    gb = qr.sample_grad(th[np.arange(B), acts], T, 1.0)
    np.testing.assert_allclose(g[L["bv"][0]:L["bv"][0] + N], gb.sum(0) / B, rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(qt, T.astype(np.float64).mean(-1), rtol=1e-6)
    for du in (False, True):
        one, plain = qr.layout(H, du, 1), qo.layout(H, du)
        assert one["total"] == plain["total"] and all(one[k] == plain[k] for k in plain if k != "total")


# ---------------------------------------------------------------------------------------------- the C ABI
_CTYPE = {"int": C.c_int, "double": C.c_double, "long long": C.c_longlong}


def _prototype(hdr, name):
    m = re.search(r"\bint\s+" + name + r"\s*\((.*?)\);", hdr, flags=re.S)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


@pytest.mark.parametrize("name", ["fb_qnet_create_qr", "fb_qnet_forward_quantiles", "fb_debug_qr_loss"])
def test_ctypes_prototypes_match_the_header(name):
    from dqnflappybird_b200 import _lib
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "flappy_b200.h")).read(), flags=re.S)
    params = _prototype(hdr, name)
    argtypes, restype = _lib._SIGNATURES[name]
    assert restype is C.c_int and len(argtypes) == len(params), (name, params)
    for decl, ct in zip(params, argtypes):
        if "*" in decl:
            assert ct is C.c_void_p or (isinstance(ct, type) and issubclass(ct, C._Pointer)), (name, decl, ct)
        else:
            base = " ".join(decl.replace("const ", "").split()[:-1])
            assert ct is _CTYPE[base], (name, decl, ct)
