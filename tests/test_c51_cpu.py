"""The C51 oracle's projection and loss (oracle/c51_oracle.py) and the C ABI of the distributional head, without a GPU."""
import os
import re
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import c51_oracle as c5  # noqa: E402
from oracle import nstep_oracle as no  # noqa: E402
from oracle import qnet_oracle as qo  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUPPORTS = [(51, -10.0, 20.0), (31, -10.0, 20.0), (2, -1.0, 1.0), (64, -3.5, 7.25)]


def _random_p(rng, B, N):
    p = rng.gamma(0.3, size=(B, N)).astype(np.float32) + np.float32(1e-7)
    return (p / p.sum(1, keepdims=True)).astype(np.float32)


def test_support_is_fp32_of_the_float64_grid():
    z = c5.support(51, -10.0, 20.0)
    assert z.dtype == np.float32 and z[0] == -10.0 and z[-1] == 20.0
    np.testing.assert_allclose(z, np.linspace(-10.0, 20.0, 51), rtol=0, atol=1e-5)
    assert np.all(np.diff(z) > 0)


@pytest.mark.parametrize("atoms,v_min,v_max", SUPPORTS)
def test_projection_conserves_mass(atoms, v_min, v_max):
    rng = np.random.default_rng(atoms)
    B = 400
    p = _random_p(rng, B, atoms)
    R = rng.uniform(2 * v_min - 5, 2 * v_max + 5, B)            # targets clipped at both ends included
    d = np.where(rng.random(B) < 0.2, 0.0, rng.choice([0.99, 0.99 ** 3, 0.5], B))
    m = c5.project(p, R, d, atoms, v_min, v_max)
    assert (m >= 0).all()
    np.testing.assert_allclose(m.sum(1), p.astype(np.float64).sum(1), rtol=0, atol=1e-12)


@pytest.mark.parametrize("atoms,v_min,v_max", SUPPORTS)
def test_a_dirac_with_zero_reward_and_unit_discount_projects_to_itself(atoms, v_min, v_max):
    eye = np.eye(atoms, dtype=np.float32)
    m = c5.project(eye, np.zeros(atoms), np.ones(atoms), atoms, v_min, v_max)
    # fp32 atoms of a grid that is not exact in binary land within an fp32 rounding of their own atom
    tol = 0.0 if atoms == 31 else 1e-5
    np.testing.assert_allclose(m, np.eye(atoms), rtol=0, atol=tol)


def test_a_terminal_projects_only_its_reward():
    atoms, v_min, v_max = 51, -10.0, 20.0
    rng = np.random.default_rng(1)
    z = c5.support(atoms, v_min, v_max).astype(np.float64)
    r = np.array([0.1, 3.0, -3.0, 0.1, -3.0, 25.0, -12.0])
    p = _random_p(rng, len(r), atoms)
    m = c5.project(p, r, np.zeros(len(r)), atoms, v_min, v_max)
    for b in range(len(r)):
        nz = np.flatnonzero(m[b])
        assert len(nz) <= 2 and (len(nz) == 1 or nz[1] == nz[0] + 1), (b, nz)
        want = min(max(r[b], v_min), v_max)
        assert abs((m[b] * z).sum() - want) <= 1e-5 * max(1.0, abs(want)), b
    # the 1-step target of a terminal is the same thing: disc 0, the env's 0.1 as a Python float
    R, d = c5.one_step_targets(np.float32([0.1, -3.0]), np.uint8([1, 1]), 0.99)
    assert R[0] == 0.1 and R[1] == -3.0 and (d == 0).all()


def test_n_step_targets_use_nstep_oracle_returns():
    rng = np.random.default_rng(2)
    E, T, n, gamma = 6, 12, 3, 0.99
    rew = rng.choice(np.float32([0.1, 3.0, -3.0]), (T, E), p=[0.8, 0.1, 0.1])
    term = (rew == -3.0).astype(np.uint8)
    pairs = [no.nstep_targets(rew, term, e, k, n, gamma) for e in range(E) for k in range(1, T - n)]
    R = np.array([x[0] for x in pairs]); d = np.array([x[1] for x in pairs])
    assert (d == 0).any() and (d > 0).any()
    p = _random_p(rng, len(R), 51)
    m = c5.project(p, R, d, 51)
    # by hand, atom by atom, from the same R and disc
    z = c5.support(51).astype(np.float64)
    dz = 30.0 / 50
    for b in range(0, len(R), 7):
        want = np.zeros(51)
        for j in range(51):
            tz = min(max(R[b] if d[b] == 0 else R[b] + d[b] * z[j], -10.0), 20.0)
            bb = min((tz + 10.0) / dz, 50.0)
            lo, up = int(np.floor(bb)), int(np.ceil(bb))
            if lo == up:
                want[lo] += float(p[b, j])
            else:
                want[lo] += float(p[b, j]) * (up - bb)
                want[up] += float(p[b, j]) * (bb - lo)
        assert np.array_equal(m[b], want), b
    # at n = 1 the n-step pair is the 1-step target
    r1 = [no.nstep_targets(rew, term, e, 4, 1, gamma) for e in range(E)]
    R1, d1 = c5.one_step_targets(rew[4], term[4], gamma)
    assert np.array_equal(R1, [x[0] for x in r1]) and np.array_equal(d1, [x[1] for x in r1])


@pytest.mark.parametrize("loss_sum", [True, False])
def test_cross_entropy_gradient_is_w_scale_p_minus_m(loss_sum):
    rng = np.random.default_rng(3)
    B, N, gb = 9, 51, 32
    lg = torch.tensor(rng.normal(0, 2, (B, 2, N)), requires_grad=True)
    # autograd gives w scale (p sum(m) - m): the rule the device applies once m sums to 1.  The fp32 probabilities the projection
    # spreads sum to 1 within ~1e-7 (so does m, rounded or not): a relative 1e-7 on the gradient, normalised away here
    m = c5.project(_random_p(rng, B, N), rng.uniform(-5, 25, B), np.full(B, 0.99), N)
    m = torch.tensor(m / m.sum(1, keepdims=True))
    act = torch.tensor(rng.integers(0, 2, B))
    w = torch.tensor(rng.uniform(0.2, 1.0, B))
    scale = 1.0 if loss_sum else 1.0 / gb
    ce = -(m * torch.log_softmax(lg, -1)[torch.arange(B), act]).sum(-1)
    (w * ce * scale).sum().backward()
    want = torch.zeros(B, 2, N, dtype=torch.float64)
    want[torch.arange(B), act] = (w * scale)[:, None] * (torch.softmax(lg.detach(), -1)[torch.arange(B), act] - m)
    torch.testing.assert_close(lg.grad, want, rtol=0, atol=1e-13)


def test_oracle_loss_is_consistent_with_its_parts():
    """one tiny update: the returned CE, q_target and loss follow from the returned m and the oracle forward"""
    rng = np.random.default_rng(4)
    B, H, N = 3, 32, 11
    params = c5.init_params(H, True, N, seed=1) * np.float32(5)
    target = c5.init_params(H, True, N, seed=2) * np.float32(5)
    x = rng.choice(np.uint8([0, 255]), (B, 5, 80, 80))
    acts = np.array([0, 1, 1])
    R, d = c5.one_step_targets(np.float32([0.1, 3.0, -3.0]), np.uint8([0, 0, 1]), 0.99)
    loss, g, ce, qt, q, m = c5.loss_and_grads(1, params, target, x[:, 0:4], x[:, 1:5], acts, R, d, hidden=H, dueling=True, atoms=N,
                                              v_min=-3.0, v_max=4.0)
    p, q2 = c5.forward(params, x[:, 0:4], H, True, N, -3.0, 4.0)
    np.testing.assert_allclose(q, q2, rtol=1e-12)
    np.testing.assert_allclose(ce, -(m * np.log(p[np.arange(B), acts])).sum(-1), rtol=1e-10)
    assert abs(loss - ce.sum() / B) <= 1e-12 * abs(loss)
    np.testing.assert_allclose(qt, (m.astype(np.float64) * c5.support(N, -3.0, 4.0)).sum(-1), rtol=1e-6)
    assert np.isfinite(g).all() and g.shape == (c5.layout(H, True, N)["total"],)
    L = c5.layout(H, True, N)
    assert L["wv"][1] == (H, N) and L["ba"][1] == (2 * N,) and L["wf1"] == qo.layout(H, True)["wf1"]


# ---------------------------------------------------------------------------------------------- the C ABI
_CTYPE = {"int": C.c_int, "double": C.c_double, "long long": C.c_longlong}


def _prototype(hdr, name):
    m = re.search(r"\bint\s+" + name + r"\s*\((.*?)\);", hdr, flags=re.S)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


@pytest.mark.parametrize("name", ["fb_qnet_create_c51", "fb_qnet_forward_dist", "fb_debug_c51_project"])
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
