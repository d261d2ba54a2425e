"""Noisy-network oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The definition the device is held to (include/flappy_b200.h, fb_noisy_*; csrc/fb_noisy.cu).  The noisy layers are fc1 and the
head (plain: wf2 / bf2; dueling: wv / bv, then wa / ba); a layer with p inputs and q outputs runs on
    W[i][j] = mu[i][j] + sigma[i][j] * (f(eps_in[i]) * f(eps_out[j])),   b[j] = mu_b[j] + sigma_b[j] * f(eps_out[j]),
f(x) = sgn(x) sqrt|x|, in fp32 with one rounding per operation.  The factor vector of a draw holds, per noisy layer in layer
order, f(eps_in) then f(eps_out); normal k of draw d is Box-Muller in float64 on words 2k, 2k+1 of the Philox stream
(seed, purpose 5, d), d = (counter << 2) | role (0 online net of update `counter`, 1 its target net, 2 acting call `counter`),
rounded to fp32 before f.

Gradients follow from qnet_oracle (or nstep_oracle) by the chain rule: with W = mu + sigma * eps, dL/dmu = dL/dW and
dL/dsigma = dL/dW * eps.  The update is one TF-1 Adam over (mu, sigma) with one pair of beta powers.
"""
from __future__ import annotations

import math

import numpy as np

from . import flappy_oracle as fo
from . import nstep_oracle as no
from . import qnet_oracle as qo

PURPOSE = 5
ROLES = {"online": 0, "target": 1, "act": 2}


def noise_layout(hidden=512, dueling=False):
    """([{w, b, p, q, f_in, f_out}] per noisy layer, factor-vector length): what fb_noisy_layout returns"""
    L = qo.layout(hidden, dueling)
    pairs = [("wf1", "bf1")] + ([("wf2", "bf2")] if not dueling else [("wv", "bv"), ("wa", "ba")])
    out, o = [], 0
    for w, b in pairs:
        wo, (p, q) = L[w]
        out.append(dict(w=wo, b=L[b][0], p=p, q=q, f_in=o, f_out=o + p))
        o += p + q
    return out, o


def draw_id(role, counter):
    return ((int(counter) << 2) | ROLES.get(role, role)) & (2 ** 64 - 1)


def f(z32):
    """sgn(z) sqrt|z| in fp32 (f(0) = +0)"""
    z32 = np.asarray(z32, np.float32)
    s = np.sqrt(np.abs(z32))
    return np.where(z32 < 0, -s, s).astype(np.float32)


def normals(seed, role, counter, n):
    """the n fp32 normals of a draw (before f)"""
    d = draw_id(role, counter)
    z = np.empty(n, np.float32)
    for k in range(n):
        w0, w1 = fo.stream_word(seed, PURPOSE, d, 2 * k), fo.stream_word(seed, PURPOSE, d, 2 * k + 1)
        u1, u2 = (w0 + 1.0) * 2.0 ** -32, w1 * 2.0 ** -32
        z[k] = np.float32(math.sqrt(-2.0 * math.log(u1)) * math.cos(2.0 * math.pi * u2))
    return z


def factors(seed, role, counter, hidden=512, dueling=False):
    """the factor vector of draw (role, counter)"""
    return f(normals(seed, role, counter, noise_layout(hidden, dueling)[1]))


def eps_flat(fac, hidden=512, dueling=False, dtype=np.float32):
    """eps per parameter (0 outside the noisy layers): the fp32 product f_in f_out (dtype float32), or exact (float64)"""
    n = qo.layout(hidden, dueling)["total"]
    e = np.zeros(n, dtype)
    fac = np.asarray(fac, np.float32).astype(dtype)
    for ly in noise_layout(hidden, dueling)[0]:
        fin, fout = fac[ly["f_in"]:ly["f_in"] + ly["p"]], fac[ly["f_out"]:ly["f_out"] + ly["q"]]
        e[ly["w"]:ly["w"] + ly["p"] * ly["q"]] = np.outer(fin, fout).reshape(-1)
        e[ly["b"]:ly["b"] + ly["q"]] = fout
    return e


def noisy_mask(hidden=512, dueling=False):
    m = np.zeros(qo.layout(hidden, dueling)["total"], bool)
    for ly in noise_layout(hidden, dueling)[0]:
        m[ly["w"]:ly["w"] + ly["p"] * ly["q"]] = True
        m[ly["b"]:ly["b"] + ly["q"]] = True
    return m


def weff32(mu, sigma, fac, hidden=512, dueling=False):
    """W_eff in fp32: (f_in f_out) rounded, times sigma rounded, plus mu rounded; mu outside the noisy layers"""
    mu, sigma = np.asarray(mu, np.float32), np.asarray(sigma, np.float32)
    w = mu + sigma * eps_flat(fac, hidden, dueling)
    return np.where(noisy_mask(hidden, dueling), w, mu).astype(np.float32)


def sigma_init(hidden=512, dueling=False, sigma0=0.5):
    """sigma0 / sqrt(fan-in) on every noisy weight and bias, 0 elsewhere (fp32)"""
    s = np.zeros(qo.layout(hidden, dueling)["total"], np.float32)
    for ly in noise_layout(hidden, dueling)[0]:
        v = np.float32(sigma0 / math.sqrt(ly["p"]))
        s[ly["w"]:ly["w"] + ly["p"] * ly["q"]] = v
        s[ly["b"]:ly["b"] + ly["q"]] = v
    return s


def loss_and_grads(variant, mu, sigma, target_mu, target_sigma, fac, fac_target, s, s2, actions, rewards=None, terminals=None,
                   isw=None, gamma=0.99, loss_sum=False, global_batch=None, hidden=512, dueling=False, emulate=None, returns=None,
                   disc=None):
    """The update's loss and gradients in float64 on W = mu + sigma * eps (exact products) for the online draw ``fac`` and, for
    the Nature / Double targets, W_target = target_mu + target_sigma * eps_target of ``fac_target``.  The variant's target, the
    loss and the emulated roundings are qnet_oracle.loss_and_grads' (nstep_oracle's when ``returns`` / ``disc`` are given).
    Returns loss, dL/dmu, dL/dsigma (float64 flat), abs_err, y (fp32 as fed), q(s)."""
    e = eps_flat(fac, hidden, dueling, np.float64)
    W = np.asarray(mu, np.float64) + np.asarray(sigma, np.float64) * e
    if variant != 0:
        WT = np.asarray(target_mu, np.float64) + np.asarray(target_sigma, np.float64) * eps_flat(fac_target, hidden, dueling, np.float64)
    else:
        WT = None
    if returns is not None:
        loss, gW, abs_err, y, q = no.loss_and_grads(variant, W, WT, s, s2, actions, returns, disc, isw, loss_sum, global_batch, hidden,
                                                    dueling, emulate=emulate)
    else:
        loss, gW, abs_err, y, q = qo.loss_and_grads(variant, W, WT, s, s2, actions, rewards, terminals, isw, gamma, loss_sum,
                                                    global_batch, hidden, dueling, emulate=emulate)
    return loss, gW, gW * e, abs_err, y, q


class NoisyAdamTF1:
    """TF-1 Adam over (mu, sigma) as one optimizer: one alpha, one pair of fp32 beta powers (qnet_oracle.AdamTF1 over both)"""

    def __init__(self, n, **kw):
        self.n = n
        self.opt = qo.AdamTF1(2 * n, **kw)

    def step(self, mu32, sigma32, g_mu, g_sigma):
        p = np.concatenate([mu32, sigma32]).astype(np.float32)
        p = self.opt.step(p, np.concatenate([np.asarray(g_mu, np.float32), np.asarray(g_sigma, np.float32)]))
        return p[:self.n].copy(), p[self.n:].copy()
