"""n-step return oracle -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The definition the device is held to (include/flappy_b200.h, fb_step_sampling.n_step; csrc/fb_replay.cu): transition k of an
env becomes (s_{k-1}, a_k, R_k, s_{k+n-1}, disc_k).  m is the first i in 1..n whose term_{k+i-1} is set, else n;
R_k = sum_{i<m} gamma^i r_{k+i}, accumulated forward in float64 (R += g r; g *= gamma) with the env's Python float 0.1;
disc_k = 0 when a terminal cut the window, else that running g = gamma^n.  The TD target is y = R if disc == 0 else
R + disc * X, X being the variant's bootstrap value on s_{k+n-1}.  At n = 1, R = r_k and disc = 0 if term_k else gamma, so y is
the 1-step target of qnet_oracle.loss_and_grads bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from .qnet_oracle import forward, fp16_grad_scale


def nstep_targets(rew_rows, term_rows, env, k, n, gamma):
    """(R_k, disc_k) of transition k of env ``env`` in float64.  rew_rows[t][e] / term_rows[t][e]: reward and terminal of step t."""
    R, g = 0.0, 1.0
    for i in range(n):
        rf = np.float32(rew_rows[k + i][env])
        R += g * (0.1 if rf == np.float32(0.1) else float(rf))
        g *= gamma
        if term_rows[k + i][env]:
            return R, 0.0
    return R, g


def loss_and_grads(variant, params32, target32, s, s2, actions, returns, disc, isw=None, loss_sum=False, global_batch=None,
                   hidden=512, dueling=False, emulate=None):
    """qnet_oracle.loss_and_grads with the n-step target y = R if disc == 0 else R + disc * X in place of the 1-step one; s2 is
    s_{k+n-1}.  The rest -- the variant's X (vanilla / Nature / Double), fp32 Q-values into a float64 target fed back as fp32,
    the sum / mean / IS-weighted loss (the intended mean(w_i err_i^2)), the emulated roundings -- is that function's, line for line.
    Returns loss, grads (float64 flat), abs_err, y (fp32 as fed), q(s)."""
    P = torch.tensor(params32.astype(np.float64), requires_grad=True)
    T = torch.tensor((target32 if target32 is not None else params32).astype(np.float64))
    B = len(actions)
    gb = global_batch or B
    gs = fp16_grad_scale(gb, loss_sum) if emulate == "fp16" else 1.0
    with torch.no_grad():
        if variant == 0:
            x = forward(P.detach(), s2, hidden, dueling, emulate=emulate, grad_scale=gs).max(dim=1).values
        elif variant == 1:
            x = forward(T, s2, hidden, dueling, emulate=emulate, grad_scale=gs).max(dim=1).values
        else:
            qt = forward(T, s2, hidden, dueling, emulate=emulate, grad_scale=gs)
            am = forward(P.detach(), s2, hidden, dueling, emulate=emulate, grad_scale=gs).argmax(dim=1)
            x = qt[torch.arange(B), am]
        x32 = x.numpy().astype(np.float32).astype(np.float64)
        R, d = np.asarray(returns, np.float64), np.asarray(disc, np.float64)
        y = np.where(d == 0.0, R, R + d * x32).astype(np.float32)
    q = forward(P, s, hidden, dueling, emulate=emulate, grad_scale=gs)
    onehot = F.one_hot(torch.as_tensor(np.asarray(actions).astype(np.int64)), 2).to(torch.float64)
    q_eval = (q * onehot).sum(dim=1)
    err = torch.as_tensor(y.astype(np.float64)) - q_eval
    w = torch.ones(B, dtype=torch.float64) if isw is None else torch.as_tensor(np.asarray(isw, np.float64))
    loss = (w * err ** 2).sum() if loss_sum else (w * err ** 2).sum() / gb
    loss.backward()
    return float(loss.detach()), P.grad.numpy().copy(), err.detach().abs().numpy(), y, q.detach().numpy()
