"""C51 (distributional) head oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The definition the device is held to (include/flappy_b200.h fb_qnet_create_c51; csrc/fb_c51.cu), restated in float64 torch:

  support   dz = (v_max - v_min) / (N - 1) in float64, z_i = fp32(v_min + i dz)
  head      plain: logits l[a][i] = h1 . W_fc2[:, a N + i] + b_fc2[a N + i];
            dueling: l[a][i] = v[i] + (alpha[a][i] - (alpha[0][i] + alpha[1][i]) / 2), v = h1 W_fc2_v + b, alpha = h1 W_fc2_a + b
            p[a] = softmax_i l[a],  Q[a] = sum_i z_i p[a][i]
  target    a* = first argmax of the variant's Q(s') (vanilla: online net; Nature: target net; Double: online argmax, target p);
            m = project(fp32 p[a*](s'), R, disc), rounded to fp32 once
  loss      CE_b = -sum_i m_i log p[a_b][i](s);  loss = sum_b w_b CE_b scale (scale 1 for the sum loss, else 1 / global batch)

The trunk is qnet_oracle.forward (its h1, with the same emulated fp16 / bf16 roundings and gradient scale); the head, the
cross-entropy and every gradient come from autograd.  A noisy net composes through its effective weights (noisy_oracle.weff32):
pass W_eff as the parameters.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from . import qnet_oracle as qo

TRUNK = ("w1", "b1", "w2", "b2", "w3", "b3", "wf1", "bf1")


def layout(hidden=512, dueling=False, atoms=51):
    """{name: (offset, shape)} and "total": the trunk of qnet_oracle.layout, then the head with N outputs per action"""
    base = qo.layout(hidden, dueling)
    out = {k: base[k] for k in TRUNK}
    o = base["bf1"][0] + hidden
    N = atoms
    head = [("wf2", (hidden, 2 * N)), ("bf2", (2 * N,))] if not dueling else \
        [("wv", (hidden, N)), ("bv", (N,)), ("wa", (hidden, 2 * N)), ("ba", (2 * N,))]
    for n, shp in head:
        out[n] = (o, shp)
        o += int(np.prod(shp))
    out["total"] = o
    return out


def init_params(hidden=512, dueling=False, atoms=51, seed=0) -> np.ndarray:
    """truncated_normal(0.01) weights, 0.01 biases (qnet_oracle.init_params' rule on this layout)"""
    g = torch.Generator().manual_seed(seed)
    L = layout(hidden, dueling, atoms)
    flat = np.zeros(L["total"], np.float32)
    for n, v in L.items():
        if n == "total":
            continue
        o, shp = v
        sz = int(np.prod(shp))
        if n.startswith("b"):
            flat[o:o + sz] = 0.01
        else:
            w = torch.randn(sz, generator=g, dtype=torch.float64)
            bad = w.abs() > 2
            while bad.any():
                w[bad] = torch.randn(int(bad.sum()), generator=g, dtype=torch.float64)
                bad = w.abs() > 2
            flat[o:o + sz] = (w * 0.01).numpy().astype(np.float32)
    return flat


def support(atoms=51, v_min=-10.0, v_max=20.0) -> np.ndarray:
    """z_i as fp32: v_min + i dz in float64 (one rounding per operation), then rounded"""
    dz = (float(v_max) - float(v_min)) / (atoms - 1)
    return np.array([np.float32(float(v_min) + i * dz) for i in range(atoms)], np.float32)


def one_step_targets(rewards, terminals, gamma):
    """(R, disc) of the 1-step target: R = r (the env's Python float 0.1), disc = 0 after a terminal, else gamma"""
    r = np.array([0.1 if np.float32(v) == np.float32(0.1) else float(np.float32(v)) for v in np.asarray(rewards).reshape(-1)], np.float64)
    d = np.where(np.asarray(terminals).reshape(-1).astype(bool), 0.0, float(gamma))
    return r, d


def project(p_next, returns, disc, atoms=51, v_min=-10.0, v_max=20.0) -> np.ndarray:
    """the float64 projection m [B][N] of R + disc z under p_next [B][N] (fp32 probabilities, widened), atoms j ascending:
    Tz = clip(disc == 0 ? R : R + disc z_j, v_min, v_max), b = min((Tz - v_min) / dz, N - 1), l = floor(b), u = ceil(b);
    p_j to atom l when l == u, else p_j (u - b) to l and p_j (b - l) to u.  Not yet rounded to fp32."""
    p = np.asarray(p_next, np.float32).astype(np.float64)
    R, d = np.asarray(returns, np.float64).reshape(-1), np.asarray(disc, np.float64).reshape(-1)
    B, N = p.shape
    assert N == atoms
    z = support(atoms, v_min, v_max).astype(np.float64)
    dz = (float(v_max) - float(v_min)) / (atoms - 1)
    m = np.zeros((B, N), np.float64)
    rows = np.arange(B)
    for j in range(N):
        tz = np.where(d == 0.0, R, R + d * z[j])
        tz = np.minimum(np.maximum(tz, float(v_min)), float(v_max))
        b = np.minimum((tz - float(v_min)) / dz, float(N - 1))
        lo, up = np.floor(b), np.ceil(b)
        li, ui = lo.astype(np.int64), up.astype(np.int64)
        whole = li == ui
        m[rows[whole], li[whole]] += p[whole, j]
        part = ~whole
        m[rows[part], li[part]] += p[part, j] * (up[part] - b[part])
        m[rows[part], ui[part]] += p[part, j] * (b[part] - lo[part])
    return m


def _h1(flat, x, hidden, emulate, grad_scale):
    """h1 of qnet_oracle.forward for the trunk of `flat` (the plain head it computes on zeros is discarded)"""
    trunk_end = qo.layout(hidden, False)["bf1"][0] + hidden
    plain = torch.cat([flat[:trunk_end], torch.zeros(2 * hidden + 2, dtype=flat.dtype)])
    _, acts = qo.forward(plain, x, hidden, False, return_all=True, emulate=emulate, grad_scale=grad_scale)
    return acts["h1"]


def logits(flat, x, hidden=512, dueling=False, atoms=51, emulate=None, grad_scale=1.0):
    """l [B][2][N] in float64"""
    L = layout(hidden, dueling, atoms)
    P = {n: flat[o:o + int(np.prod(shp))].reshape(shp) for n, (o, shp) in ((k, v) for k, v in L.items() if k != "total")}
    h1 = _h1(flat, x, hidden, emulate, grad_scale)
    B, N = h1.shape[0], atoms
    if not dueling:
        return (h1 @ P["wf2"] + P["bf2"]).reshape(B, 2, N)
    v = h1 @ P["wv"] + P["bv"]
    a = (h1 @ P["wa"] + P["ba"]).reshape(B, 2, N)
    return v[:, None, :] + (a - a.mean(dim=1, keepdim=True))


def forward(flat, x, hidden=512, dueling=False, atoms=51, v_min=-10.0, v_max=20.0, emulate=None):
    """(p [B][2][N], Q [B][2]) in float64"""
    flat = torch.as_tensor(np.asarray(flat, np.float64))
    p = torch.softmax(logits(flat, x, hidden, dueling, atoms, emulate), dim=-1)
    z = torch.as_tensor(support(atoms, v_min, v_max).astype(np.float64))
    return p.numpy(), (p * z).sum(-1).numpy()


def loss_and_grads(variant, params32, target32, s, s2, actions, returns, disc, isw=None, loss_sum=False, global_batch=None,
                   hidden=512, dueling=False, emulate=None, atoms=51, v_min=-10.0, v_max=20.0):
    """nstep_oracle.loss_and_grads' arguments (the 1-step target is R, disc = one_step_targets(...)) with the C51 head.
    Returns loss, grads (float64 flat), abs_err (= CE_b), q_target (= sum z m, fp32), q(s), m (fp32)."""
    P = torch.tensor(np.asarray(params32).astype(np.float64), requires_grad=True)
    T = torch.tensor(np.asarray(target32 if target32 is not None else params32).astype(np.float64))
    B = len(actions)
    gb = global_batch or B
    gs = qo.fp16_grad_scale(gb, loss_sum) if emulate == "fp16" else 1.0
    z = torch.as_tensor(support(atoms, v_min, v_max).astype(np.float64))
    kw = dict(hidden=hidden, dueling=dueling, atoms=atoms, emulate=emulate, grad_scale=gs)
    with torch.no_grad():
        p_on = torch.softmax(logits(P.detach(), s2, **kw), dim=-1) if variant in (0, 2) else None
        p_tg = torch.softmax(logits(T, s2, **kw), dim=-1) if variant in (1, 2) else None
        p_sel = p_on if variant == 0 else p_tg
        q_arg = ((p_on if variant in (0, 2) else p_tg) * z).sum(-1).numpy().astype(np.float32)    # the device compares fp32 Q
        astar = (q_arg[:, 1] > q_arg[:, 0]).astype(np.int64)                                     # first max on ties
        pn32 = p_sel.numpy()[np.arange(B), astar].astype(np.float32)
        m32 = project(pn32, returns, disc, atoms, v_min, v_max).astype(np.float32)
    lg = logits(P, s, **kw)
    logp = F.log_softmax(lg, dim=-1)
    act = torch.as_tensor(np.asarray(actions).astype(np.int64))
    lp_a = logp[torch.arange(B), act]
    m = torch.as_tensor(m32.astype(np.float64))
    ce = -(m * lp_a).sum(-1)
    w = torch.ones(B, dtype=torch.float64) if isw is None else torch.as_tensor(np.asarray(isw, np.float64))
    loss = (w * ce).sum() if loss_sum else (w * ce).sum() / gb
    loss.backward()
    q_s = (torch.softmax(lg.detach(), dim=-1) * z).sum(-1).numpy()
    q_target = (m * z).sum(-1).numpy().astype(np.float32)
    return float(loss.detach()), P.grad.numpy().copy(), ce.detach().numpy(), q_target, q_s, m32

