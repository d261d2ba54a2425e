"""QR-DQN (quantile-regression) head oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The definition the device is held to (include/flappy_b200.h fb_qnet_create_qr; csrc/fb_qr.cu), restated in float64 torch:

  fractions tau_i = (2 i + 1) / (2 N)
  head      theta[a][i]: c51_oracle.logits on the same layout (plain: h1 . W_fc2[:, a N + i] + b; dueling: v_i + (alpha_{a,i} - mean_a
            alpha_{., i})),  Q[a] = mean_i theta[a][i]
  target    a* = first argmax of the variant's Q(s') (vanilla: online net; Nature: target net; Double: online argmax, target theta);
            T_j = fp32(disc == 0 ? R : R + disc theta[a*][j](s')) -- the expected-value head's td_target per quantile
  loss      u_ij = T_j - theta[a_b][i](s),  L_b = sum_i (1/N) sum_j |tau_i - 1{u_ij < 0}| H(u_ij),
            H(u) = u^2 / (2 kappa) for |u| <= kappa else |u| - kappa / 2 (kappa > 0), H(u) = |u| (kappa = 0, H'(0) = 0);
            loss = sum_b w_b L_b scale (scale 1 for the sum loss, else 1 / global batch)

The trunk is qnet_oracle's (through c51_oracle, with the same emulated fp16 / bf16 roundings and gradient scale); gradients come
from autograd, and sample_grad gives dL_b/dtheta by hand.  A noisy net composes through its effective weights: pass W_eff.
"""
from __future__ import annotations

import numpy as np
import torch

from . import c51_oracle as c5
from . import qnet_oracle as qo

one_step_targets = c5.one_step_targets


def layout(hidden=512, dueling=False, quantiles=32):
    """{name: (offset, shape)} and "total": the C51 layout with N = quantiles outputs per action"""
    return c5.layout(hidden, dueling, quantiles)


def init_params(hidden=512, dueling=False, quantiles=32, seed=0) -> np.ndarray:
    return c5.init_params(hidden, dueling, quantiles, seed=seed)


def taus(quantiles) -> np.ndarray:
    return (2.0 * np.arange(quantiles) + 1.0) / (2.0 * quantiles)


def theta(flat, x, hidden=512, dueling=False, quantiles=32, emulate=None, grad_scale=1.0):
    """theta [B][2][N] in float64 (a torch tensor when flat is one)"""
    return c5.logits(flat, x, hidden, dueling, quantiles, emulate, grad_scale)


def forward(flat, x, hidden=512, dueling=False, quantiles=32, emulate=None):
    """(theta [B][2][N], Q [B][2]) in float64"""
    th = theta(torch.as_tensor(np.asarray(flat, np.float64)), x, hidden, dueling, quantiles, emulate)
    return th.numpy(), th.mean(-1).numpy()


def targets(theta_next_astar, returns, disc) -> np.ndarray:
    """T [B][N] in fp32: R + disc theta (theta fp32, widened) in float64, R alone where disc == 0, rounded once"""
    x = np.asarray(theta_next_astar, np.float32).astype(np.float64)
    R, d = np.asarray(returns, np.float64).reshape(-1, 1), np.asarray(disc, np.float64).reshape(-1, 1)
    return np.where(d == 0.0, R + 0.0 * x, R + d * x).astype(np.float32)


def _huber(u, kappa):
    if kappa == 0:
        return u.abs()
    return torch.where(u.abs() <= kappa, 0.5 * u * u / kappa, u.abs() - 0.5 * kappa)


def sample_loss(theta_a, T, kappa):
    """L_b [B] of theta_a [B][N] (theta[a_b](s), float64 torch, may require grad) against T [B][N]"""
    B, N = theta_a.shape
    tau = torch.as_tensor(taus(N))
    T = torch.as_tensor(np.asarray(T, np.float64))
    u = T[:, None, :] - theta_a[:, :, None]                       # [B][i][j]
    wt = (tau[None, :, None] - (u < 0).to(torch.float64)).abs()
    return (wt * _huber(u, float(kappa))).sum(-1).sum(-1) / N


def sample_grad(theta_a, T, kappa) -> np.ndarray:
    """dL_b/dtheta_i [B][N] by hand: -(1/N) sum_j |tau_i - 1{u_ij < 0}| H'(u_ij)"""
    th, T = np.asarray(theta_a, np.float64), np.asarray(T, np.float64)
    N = th.shape[1]
    u = T[:, None, :] - th[:, :, None]
    wt = np.abs(taus(N)[None, :, None] - (u < 0))
    dh = np.sign(u) if kappa == 0 else np.where(np.abs(u) <= kappa, u / kappa, np.sign(u))
    return -(wt * dh).sum(-1) / N


def loss_and_grads(variant, params32, target32, s, s2, actions, returns, disc, isw=None, loss_sum=False, global_batch=None,
                   hidden=512, dueling=False, emulate=None, quantiles=32, kappa=1.0):
    """nstep_oracle.loss_and_grads' arguments (the 1-step target is R, disc = one_step_targets(...)) with the QR head.
    Returns loss, grads (float64 flat), abs_err (= L_b), q_target (= mean T, fp32), q(s), T (fp32)."""
    P = torch.tensor(np.asarray(params32).astype(np.float64), requires_grad=True)
    Tg = torch.tensor(np.asarray(target32 if target32 is not None else params32).astype(np.float64))
    B = len(actions)
    gb = global_batch or B
    gs = qo.fp16_grad_scale(gb, loss_sum) if emulate == "fp16" else 1.0
    kw = dict(hidden=hidden, dueling=dueling, quantiles=quantiles, emulate=emulate, grad_scale=gs)
    with torch.no_grad():
        th_on = theta(P.detach(), s2, **kw) if variant in (0, 2) else None
        th_tg = theta(Tg, s2, **kw) if variant in (1, 2) else None
        th_sel = th_on if variant == 0 else th_tg
        q_arg = (th_on if variant in (0, 2) else th_tg).mean(-1).numpy().astype(np.float32)    # the device compares fp32 Q
        astar = (q_arg[:, 1] > q_arg[:, 0]).astype(np.int64)                                    # first max on ties
        T32 = targets(th_sel.numpy()[np.arange(B), astar].astype(np.float32), returns, disc)
    th = theta(P, s, **kw)
    act = torch.as_tensor(np.asarray(actions).astype(np.int64))
    lb = sample_loss(th[torch.arange(B), act], T32, kappa)
    w = torch.ones(B, dtype=torch.float64) if isw is None else torch.as_tensor(np.asarray(isw, np.float64))
    loss = (w * lb).sum() if loss_sum else (w * lb).sum() / gb
    loss.backward()
    q_target = T32.astype(np.float64).mean(-1).astype(np.float32)
    return float(loss.detach()), P.grad.numpy().copy(), lb.detach().numpy(), q_target, th.detach().mean(-1).numpy(), T32
