"""The noisy-network oracle (oracle/noisy_oracle.py) without a GPU: its pieces against each other and against qnet_oracle /
nstep_oracle -- at sigma = 0 the noisy loss and dL/dmu are the plain ones bit for bit, dL/dsigma = dL/dW * eps, the chain rule
agrees with autograd through mu + sigma * eps, and the factor vector has the stated layout and draw ids."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import flappy_oracle as fo  # noqa: E402
from oracle import noisy_oracle as nz  # noqa: E402
from oracle import nstep_oracle as no  # noqa: E402
from oracle import qnet_oracle as qo  # noqa: E402

H = 32


def _batch(B=4, seed=0):
    rng = np.random.default_rng(seed)
    s = (rng.random((B, 4, 80, 80)) < 0.3).astype(np.uint8) * 255
    s2 = (rng.random((B, 4, 80, 80)) < 0.3).astype(np.uint8) * 255
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = np.array([0.1, 3.0, -3.0, 0.1], np.float32)[:B]
    t = np.array([0, 0, 1, 0], np.uint8)[:B]
    return s, s2, a, r, t, rng.random(B).astype(np.float32)


@pytest.mark.parametrize("dueling", [False, True])
def test_layout_of_the_factor_vector(dueling):
    layers, n = nz.noise_layout(H, dueling)
    L = qo.layout(H, dueling)
    names = [("wf1", "bf1")] + ([("wf2", "bf2")] if not dueling else [("wv", "bv"), ("wa", "ba")])
    assert len(layers) == len(names)
    o = 0
    for ly, (w, b) in zip(layers, names):
        assert (ly["w"], ly["b"]) == (L[w][0], L[b][0]) and (ly["p"], ly["q"]) == L[w][1]
        assert (ly["f_in"], ly["f_out"]) == (o, o + ly["p"])
        o += ly["p"] + ly["q"]
    assert n == o == 1600 + H + (H + 2 if not dueling else (H + 1) + (H + 2))
    sig = nz.sigma_init(H, dueling, 0.5)
    mask = nz.noisy_mask(H, dueling)
    assert (sig[~mask] == 0).all() and mask.sum() == sum(ly["p"] * ly["q"] + ly["q"] for ly in layers)
    for ly in layers:
        assert (sig[ly["w"]:ly["b"] + ly["q"]] == np.float32(0.5 / math.sqrt(ly["p"]))).all()


def test_draws_follow_their_definition():
    seed = 123
    fac = nz.factors(seed, "online", 7, H)
    # normal 0 by hand from the Philox words of stream (seed, 5, (7 << 2) | 0)
    w0, w1 = fo.stream_word(seed, 5, 28, 0), fo.stream_word(seed, 5, 28, 1)
    z = np.float32(math.sqrt(-2 * math.log((w0 + 1) / 2 ** 32)) * math.cos(2 * math.pi * w1 / 2 ** 32))
    assert fac[0] == np.float32(math.copysign(math.sqrt(abs(float(z))), z)) == nz.f(z)
    # the same (seed, id) gives the same vector (nothing but seed and id enters: no rank, no env); ids and roles differ
    assert np.array_equal(fac, nz.factors(seed, "online", 7, H))
    for other in (nz.factors(seed, "online", 8, H), nz.factors(seed, "target", 7, H), nz.factors(seed, "act", 7, H),
                  nz.factors(seed + 1, "online", 7, H)):
        assert not np.array_equal(fac, other)
        assert np.mean(fac == other) < 0.01
    zs = nz.normals(seed, "act", 0, 4000)
    assert abs(zs.mean()) < 0.06 and abs(zs.std() - 1) < 0.05 and np.isfinite(zs).all()
    np.testing.assert_array_equal(nz.f(zs), np.sign(zs) * np.sqrt(np.abs(zs)))


def test_weff_is_the_fp32_formula():
    rng = np.random.default_rng(1)
    mu = qo.init_params(H, True, seed=3)
    sigma = nz.sigma_init(H, True) * rng.random(mu.size).astype(np.float32)
    fac = nz.factors(9, "online", 0, H, True)
    w = nz.weff32(mu, sigma, fac, H, True)
    m = torch.from_numpy(mu); sg = torch.from_numpy(sigma)
    ly = nz.noise_layout(H, True)[0][0]
    fin, fout = torch.from_numpy(fac[ly["f_in"]:ly["f_in"] + ly["p"]]), torch.from_numpy(fac[ly["f_out"]:ly["f_out"] + ly["q"]])
    sl = slice(ly["w"], ly["w"] + ly["p"] * ly["q"])
    want = m[sl].view(ly["p"], ly["q"]) + sg[sl].view(ly["p"], ly["q"]) * torch.outer(fin, fout)
    assert torch.equal(torch.from_numpy(w[sl]).view(ly["p"], ly["q"]), want)
    mask = nz.noisy_mask(H, True)
    assert np.array_equal(w[~mask], mu[~mask])


@pytest.mark.parametrize("dueling", [False, True])
def test_sigma_zero_is_the_plain_oracle(dueling):
    s, s2, a, r, t, isw = _batch()
    mu, tmu = qo.init_params(H, dueling, seed=1), qo.init_params(H, dueling, seed=2)
    z = np.zeros_like(mu)
    fac, fac_t = nz.factors(5, "online", 0, H, dueling), nz.factors(5, "target", 0, H, dueling)
    R = r.astype(np.float64) * 1.5; D = np.where(t != 0, 0.0, 0.99 ** 3)
    for variant, w, loss_sum, emulate in ((0, None, True, None), (1, None, False, None), (2, isw, False, None), (1, None, False, "fp16")):
        base = qo.loss_and_grads(variant, mu, tmu, s, s2, a, r, t, w, 0.99, loss_sum, hidden=H, dueling=dueling, emulate=emulate)
        got = nz.loss_and_grads(variant, mu, z, tmu, z, fac, fac_t, s, s2, a, r, t, w, 0.99, loss_sum, hidden=H, dueling=dueling,
                                emulate=emulate)
        assert got[0] == base[0] and np.array_equal(got[1], base[1]) and np.array_equal(got[4], base[3]), variant
        nb = no.loss_and_grads(variant, mu, tmu, s, s2, a, R, D, w, loss_sum, hidden=H, dueling=dueling, emulate=emulate)
        ng = nz.loss_and_grads(variant, mu, z, tmu, z, fac, fac_t, s, s2, a, isw=w, loss_sum=loss_sum, hidden=H, dueling=dueling,
                               emulate=emulate, returns=R, disc=D)
        assert ng[0] == nb[0] and np.array_equal(ng[1], nb[1]) and np.array_equal(ng[4], nb[3]), variant


@pytest.mark.parametrize("variant", [0, 1, 2])
def test_sigma_gradient_is_the_chain_rule(variant):
    """dL/dsigma = dL/dW * eps elementwise, dL/dmu = dL/dW, and both agree with autograd through W = mu + sigma * eps"""
    s, s2, a, r, t, _ = _batch(seed=variant)
    mu, tmu = qo.init_params(H, False, seed=1) * np.float32(3), qo.init_params(H, False, seed=2) * np.float32(3)
    sigma = nz.sigma_init(H, False, 0.5); tsigma = sigma * np.float32(0.5)
    fac, fac_t = nz.factors(5, "online", 3, H), nz.factors(5, "target", 3, H)
    loss, g_mu, g_sigma, _, y, _ = nz.loss_and_grads(variant, mu, sigma, tmu, tsigma, fac, fac_t, s, s2, a, r, t, hidden=H)
    e = nz.eps_flat(fac, H, dtype=np.float64)
    W = mu.astype(np.float64) + sigma.astype(np.float64) * e
    WT = tmu.astype(np.float64) + tsigma.astype(np.float64) * nz.eps_flat(fac_t, H, dtype=np.float64)
    base = qo.loss_and_grads(variant, W, WT if variant else None, s, s2, a, r, t, hidden=H)
    assert loss == base[0] and np.array_equal(g_mu, base[1]) and np.array_equal(g_sigma, base[1] * e)
    assert (g_sigma[~nz.noisy_mask(H)] == 0).all() and np.abs(g_sigma).max() > 0
    # autograd through mu and sigma as leaves, on the same target y
    P = torch.tensor(mu.astype(np.float64), requires_grad=True)
    S = torch.tensor(sigma.astype(np.float64), requires_grad=True)
    q = qo.forward(P + S * torch.from_numpy(e), s, H)
    qa = q[torch.arange(len(a)), torch.from_numpy(a.astype(np.int64))]
    err = torch.from_numpy(y.astype(np.float64)) - qa
    L = (err ** 2).mean()                                         # loss_sum=False above
    L.backward()
    assert abs(L.item() - loss) <= 1e-12 * abs(loss)
    np.testing.assert_allclose(P.grad.numpy(), g_mu, rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(S.grad.numpy(), g_sigma, rtol=1e-9, atol=1e-15)


def test_adam_over_mu_and_sigma_shares_one_alpha():
    n = 10
    rng = np.random.default_rng(0)
    opt = nz.NoisyAdamTF1(n, lr=1e-3)
    mu, sg = rng.standard_normal(n).astype(np.float32), np.full(n, 0.1, np.float32)
    gm, gs = rng.standard_normal(n).astype(np.float32), rng.standard_normal(n).astype(np.float32)
    ref_m, ref_s = qo.AdamTF1(n, lr=1e-3), qo.AdamTF1(n, lr=1e-3)
    for _ in range(3):
        mu_ref, sg_ref = ref_m.step(mu.copy(), gm), ref_s.step(sg.copy(), gs)
        mu, sg = opt.step(mu, sg, gm, gs)
        assert np.array_equal(mu, mu_ref) and np.array_equal(sg, sg_ref)
        mu, sg = mu_ref, sg_ref
