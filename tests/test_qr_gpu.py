"""The quantile-regression (QR-DQN) head on the device (csrc/fb_qr.cu, QNetwork(quantile=True), Brain*(quantile=True)) against the
float64 oracle (oracle/qr_oracle.py), against the expected-value head and against itself:

1. fb_debug_qr_loss (the loss kernel's own device function) against the oracle on hand-built rows;
2. forward_quantiles: theta and Q against the oracle, acting picks the first argmax of the Q it returns, chunked acting;
3. loss, every gradient tensor, abs_err and q_target against the oracle (fp32, and fp16 in two tiers);
4. N = 1, kappa = 16 is the plain net's squared TD loss divided by 64, on the same parameters;
5. graph replays are bit-identical to eager steps, and train_step to loss_backward + adam_step;
6. noisy QR: sigma0 = 0 is the plain QR update, and one update against the oracle on the read-back W_eff;
7. every Brain trains; 8. checkpoints; 9. what a QR net refuses; 10. two ranks under NCCL."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import qr_oracle as qr  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = 0.99
VARIANTS = {"vanilla": 0, "nature": 1, "double": 2}
NQ, KAPPA = 32, 1.0


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dqnflappybird_b200 import _lib, brains, game, qnet, replay
    return game, replay, qnet, brains, _lib


def _memory(game, replay, N, C_, n, per, B, steps, seed=3):
    """a memory filled by `steps` random-action env steps (p_flap 0.5: windows straddle crashes); same seed, same contents"""
    ring = torch.zeros((N, C_ + n + 3, 80, 80), dtype=torch.uint8, device="cuda")
    mem = (replay.PrioritizedMemory(ring, C_, seed=7, max_batch=B, mode="rebuild", n_step=n) if per
           else replay.ReplayMemory(ring, C_, seed=7, max_batch=B, n_step=n))
    gs = game.GameState(num_envs=N, seed=seed, history=mem.L, ring=mem.ring)
    gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    for k in range(1, steps + 1):
        a, r, t = mem.rows(k)
        gs.step_random(1, 0.5, 21, a, r, t, None)
        mem.appended(k)
    return mem


def _net(qnet, B, dueling=False, precision="fp16", hidden=512, seed=4, quantiles=NQ, kappa=KAPPA, **kw):
    return qnet.QNetwork(max_batch=B, hidden=hidden, dueling=dueling, seed=seed, precision=precision, quantile=True, quantiles=quantiles,
                         kappa=kappa, **kw)


def _spread_params(dueling, hidden, seed, quantiles=NQ):
    """weights scaled up from the initialisation so that the quantiles of one action differ and the loss sees both sides of kappa"""
    return qr.init_params(hidden, dueling, quantiles, seed=seed) * np.float32(5.0)


def _ring_frames(gs):
    L = gs.ring.shape[1]
    return gs.ring[:, [(gs.slot - 3 + k) % L for k in range(4)]].cpu().numpy()


# ------------------------------------------------------------------------------------------------------ 1. the loss hook
@pytest.mark.parametrize("kappa", [0.0, 1.0])
@pytest.mark.parametrize("N", [1, 32, 64])
def test_debug_loss_matches_the_oracle(mods, N, kappa):
    _, _, qnet, _, _lib = mods
    B = 64
    net = _net(qnet, 8, quantiles=N, kappa=kappa, precision="fp32")
    rng = np.random.default_rng(N)
    th_s = rng.normal(0.0, 2.0, (B, 2, N)).astype(np.float32)
    th_n = rng.normal(0.5, 2.0, (B, N)).astype(np.float32)
    acts = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.float32([0.1, 3.0, -3.0]), B)
    t = (rng.random(B) < 0.3).astype(np.uint8)
    t[:4] = 1
    r[:4] = np.float32(3.0)
    th_s[:4, :, :] = np.float32(3.0)             # terminal rows whose every u is exactly 0
    th_s[4, :, :] = np.float32(0.1)
    t[4], r[4] = 1, np.float32(0.1)
    th_s[5:8, :, :] = np.float32(-40.0)          # far below the targets: |u| > kappa on one side ...
    th_s[8:11, :, :] = np.float32(40.0)          # ... and on the other
    r[11:14], t[11:14] = np.float32(0.1), 0                # theta_i within kappa of its own T_i
    th_s[11:14] = (th_n[11:14, None, :] * np.float32(0.99) + np.float32(0.1)
                   + rng.uniform(-0.9, 0.9, (3, 2, N)).astype(np.float32) * np.float32(kappa))
    R = rng.uniform(-6.0, 8.0, B)
    d = np.where(rng.random(B) < 0.25, 0.0, GAMMA ** 3)
    d[:3] = 0.0
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    ts, tn, ta = dev(th_s), dev(th_n), dev(acts)
    dth, lb = torch.empty(B, N, device="cuda"), torch.empty(B, device="cuda")
    tr, tt = dev(r), dev(t)
    for n_step in (1, 3):
        if n_step == 1:
            rc = net._L.fb_debug_qr_loss(net._h, ts.data_ptr(), tn.data_ptr(), ta.data_ptr(), tr.data_ptr(), tt.data_ptr(), None, None,
                                         GAMMA, B, dth.data_ptr(), lb.data_ptr(), net._stream())
            Rr, dd = qr.one_step_targets(r, t, GAMMA)
        else:
            rt, dt = dev(R), dev(d)
            rc = net._L.fb_debug_qr_loss(net._h, ts.data_ptr(), tn.data_ptr(), ta.data_ptr(), None, None, rt.data_ptr(), dt.data_ptr(),
                                         GAMMA, B, dth.data_ptr(), lb.data_ptr(), net._stream())
            Rr, dd = R, d
        _lib.check(rc, "fb_debug_qr_loss")
        torch.cuda.synchronize()
        T = qr.targets(th_n, Rr, dd)
        th_a = th_s[np.arange(B), acts].astype(np.float64)
        want_l = qr.sample_loss(torch.tensor(th_a), T, kappa).numpy()
        want_g = qr.sample_grad(th_a, T, kappa)
        got_l, got_g = lb.cpu().numpy(), dth.cpu().numpy()
        print(f"\n[N={N} kappa={kappa} n={n_step}] loss {np.abs(got_l - want_l).max():.2e}  grad {np.abs(got_g - want_g).max():.2e}")
        np.testing.assert_allclose(got_l, want_l, rtol=2e-5, atol=1e-6)
        np.testing.assert_allclose(got_g, want_g, rtol=2e-5, atol=1e-6)
        if n_step == 1:                          # u = 0 exactly: no loss and no step (H'(0) = 0 at kappa = 0 too)
            assert (got_l[:5] == 0).all() and (got_g[:5] == 0).all()


# ----------------------------------------------------------------------------------------------------------- 2. forward
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
def test_forward_and_acting(mods, dueling, precision):
    game, _, qnet, _, _ = mods
    N = 200
    net = _net(qnet, N, dueling, precision)
    W = _spread_params(dueling, 512, 2)
    net.params.copy_(torch.from_numpy(W))
    gs = game.GameState(num_envs=N, seed=1, history=7)
    gs.step_random(20, 0.4, 3)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    theta, q = net.forward_quantiles(fb)
    torch.cuda.synchronize()
    th, q = theta.cpu().numpy(), q.cpu().numpy()
    acc = np.zeros(th.shape[:2], np.float32)
    for i in range(NQ):                                                   # Q: fp32 adds in ascending i, then / N
        acc = (acc + th[:, :, i]).astype(np.float32)
    assert np.array_equal(q, (acc / np.float32(NQ)).astype(np.float32))
    x = _ring_frames(gs)
    th_ref, q_ref = qr.forward(W, x, 512, dueling, NQ, emulate=None if precision == "fp32" else "fp16")
    tol = (2e-5 if precision == "fp32" else 5e-4) * np.abs(th_ref).max()
    print(f"\n[{precision}] theta {np.abs(th - th_ref).max():.2e}  Q {np.abs(q - q_ref).max():.2e}  scale {np.abs(th_ref).max():.2e}")
    assert np.abs(th - th_ref).max() <= tol and np.abs(q - q_ref).max() <= tol
    assert th.std(-1).mean() > 1e-3                                       # the quantiles of an action differ: the head is exercised
    assert torch.equal(net.forward(fb), torch.from_numpy(q).cuda())
    rng_pos = torch.zeros(N, dtype=torch.int32, device="cuda")
    acts, q_out = torch.zeros(N, dtype=torch.uint8, device="cuda"), torch.zeros(N, 2, device="cuda")
    net.act(fb, 0.0, 11, 0, rng_pos, acts, q_out)
    qa = q_out.cpu().numpy()
    assert np.array_equal(qa, q) and np.array_equal(acts.cpu().numpy(), (qa[:, 1] > qa[:, 0]).astype(np.uint8))


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_chunked_acting_matches_per_chunk_forwards(mods, precision):
    game, _, qnet, _, _ = mods
    MB = 64
    N = 3 * MB + 5
    net = _net(qnet, MB, True, precision)
    net.params.copy_(torch.from_numpy(_spread_params(True, 512, 3)))
    gs = game.GameState(num_envs=N, seed=2, history=7)
    gs.step_random(15, 0.4, 5)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    theta, q = net.forward_quantiles(fb)
    rng_pos = torch.zeros(N, dtype=torch.int32, device="cuda")
    acts, q_out = torch.zeros(N, dtype=torch.uint8, device="cuda"), torch.zeros(N, 2, device="cuda")
    net.act(fb, 0.0, 3, 0, rng_pos, acts, q_out)
    L = gs.ring.shape[1]
    for c0 in range(0, N, MB):
        n = min(MB, N - c0)
        part = qnet.FrameBatch(gs.ring, L * 6400, [((gs.slot - 3 + k) % L) * 6400 for k in range(4)], n, base_offset=c0 * L * 6400)
        tc, qc = net.forward_quantiles(part)
        assert torch.equal(tc, theta[c0:c0 + n]) and torch.equal(qc, q[c0:c0 + n]) and torch.equal(q_out[c0:c0 + n], qc), c0
    assert torch.equal(acts, (q_out[:, 1] > q_out[:, 0]).to(torch.uint8))


# -------------------------------------------------------------------------------------------------------- 3. the oracle
CASES = [  # variant, dueling, loss_sum, per, n
    ("vanilla", False, True, False, 1), ("nature", False, False, False, 1), ("double", False, False, False, 1),
    ("nature", True, False, False, 1), ("double", True, False, True, 1), ("nature", False, False, True, 3), ("double", False, False, False, 3)]
HEAD = {False: ["wf2", "bf2"], True: ["wv", "bv", "wa", "ba"]}
CONV = ("w1", "b1", "w2", "b2", "w3", "b3")


def _per_tensor(g, g_ref, dueling, hidden, quantiles=NQ):
    out = {}
    for name, (o, shp) in ((k, v) for k, v in qr.layout(hidden, dueling, quantiles).items() if k != "total"):
        sz = int(np.prod(shp))
        out[name] = float(np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) / np.linalg.norm(g_ref[o:o + sz]))
    return out


def _oracle_targets(mb, n):
    if n > 1:
        return mb.returns.cpu().numpy(), mb.disc.cpu().numpy()
    return qr.one_step_targets(mb.rewards.cpu().numpy(), mb.terminals.cpu().numpy(), GAMMA)


def _check_against_oracle(net, mb, per, n, variant, dueling, loss_sum, hidden, precision, W, WT, abs_err, y):
    """The tiers of test_c51_gpu: fp32, loss and every tensor 2e-4.  fp16, tier A (oracle with the same roundings): loss 5e-4, each
    head tensor 1.5e-3 and the whole gradient vector 1.5e-3 (5e-3 with prioritized replay, whose IS weights put the gradient on a
    few samples so that the convolution backward's rounding-decision flips are not averaged out); tier B (exact oracle): loss 4e-3,
    every tensor 4.5e-2.  abs_err and q_target (relative norm of the vector) at the loss tolerance."""
    x = mb.frames.cpu().numpy()
    m = min(n, 4)
    R, d = _oracle_targets(mb, n)
    isw = mb.is_weights_f32.cpu().numpy() if per else None
    g = net.grads.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    tiers = [(None, 2e-4, 2e-4)] if precision == "fp32" else [("fp16", 5e-4, 1.5e-3), (None, 4e-3, 4.5e-2)]
    for emulate, tol_loss, tol_g in tiers:
        loss, r, lb, qt, _, _ = qr.loss_and_grads(VARIANTS[variant], W, WT, x[:, 0:4], x[:, m:m + 4], mb.actions.cpu().numpy(), R, d, isw,
                                                  loss_sum, None, hidden, dueling, emulate, NQ, KAPPA)
        rep = _per_tensor(g, r, dueling, hidden)
        whole = float(np.linalg.norm(g - r) / np.linalg.norm(r))
        lo = abs(net.loss.item() - loss) / abs(loss)
        print(f"\n[{precision}/{emulate}] loss {lo:.2e}  grads {whole:.2e}  " + " ".join(f"{k} {v:.1e}" for k, v in rep.items()))
        assert lo <= tol_loss, (net.loss.item(), loss)
        assert np.linalg.norm(abs_err.cpu().numpy() - lb) <= tol_loss * np.linalg.norm(lb)
        assert np.linalg.norm(y.cpu().numpy() - qt) <= tol_loss * np.linalg.norm(qt)
        if precision == "fp16" and emulate == "fp16":
            assert whole <= (5e-3 if per else tol_g) and all(rep[k] <= tol_g for k in HEAD[dueling]), (whole, rep)
        else:
            assert all(v <= tol_g for v in rep.values()), (emulate, rep)


@pytest.mark.parametrize("precision,hidden", [("fp32", 512), ("fp16", 512), ("fp16", 256)])
@pytest.mark.parametrize("B", [32, 256])
@pytest.mark.parametrize("variant,dueling,loss_sum,per,n", CASES)
def test_loss_and_gradients_match_the_oracle(mods, variant, dueling, loss_sum, per, n, B, precision, hidden):
    if hidden == 256 and (B, variant, dueling, per, n) != (32, "double", True, True, 1):
        pytest.skip("hidden 256 runs one case")
    if B == 256 and (precision, variant, dueling, per, n) not in (("fp16", "nature", False, False, 1), ("fp32", "double", True, True, 1),
                                                                  ("fp16", "double", False, False, 3)):
        pytest.skip("minibatch 256 runs a representative subset (the float64 oracle is slow at that size)")
    game, replay, qnet, _, _ = mods
    net = _net(qnet, B, dueling, precision, hidden)
    W, WT = _spread_params(dueling, hidden, 1), _spread_params(dueling, hidden, 2)
    net.params.copy_(torch.from_numpy(W)); net.target.copy_(torch.from_numpy(WT))
    mem = _memory(game, replay, 64, 30, n, per, B, 60)
    abs_err, y = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
    sp, mb = mem.step_sampling(B)
    isw = mb.is_weights_f32 if per else None
    net.loss_backward(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, isw, GAMMA, loss_sum, None, abs_err, y, sampling=sp)
    torch.cuda.synchronize()
    _check_against_oracle(net, mb, per, n, variant, dueling, loss_sum, hidden, precision, W, WT if variant != "vanilla" else None, abs_err, y)


# ------------------------------------------------------------------------------ 4. against the expected-value head
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
@pytest.mark.parametrize("per", [False, True])
@pytest.mark.parametrize("variant", ["vanilla", "nature", "double"])
def test_one_quantile_is_the_squared_td_loss_over_64(mods, variant, per, dueling, precision):
    """N = 1 has the plain head's layout and initial parameters; with every |u| <= kappa = 16 the quantile-Huber loss of one
    quantile is u^2 / (4 kappa) = u^2 / 64, so loss, gradients and q_target equal the plain net's (abs_err: its square / 64)
    up to the order of the sums.  Rewards are the env's (|r| <= 3) and the weights the initialisation's (|Q| < 1).
    fp32: every tensor.  fp16: the loss, the head and fc1 (whose gradients are formed in fp32); the convolution gradients are
    not compared there, because they run on fp16 operands scaled for the plain loss (fp16_grad_scale), and at 1/64 of that loss
    the deepest of them reach fp16's subnormal range: a B200 measured conv1's weight gradient 0.4e-2 .. 2.3e-2 away, conv3's
    below 2e-4, fc1 and the head below 1.3e-5."""
    game, replay, qnet, _, _ = mods
    B, n = 32, (3 if per else 1)
    kw = dict(max_batch=B, hidden=512, dueling=dueling, seed=5, precision=precision)
    plain, one = qnet.QNetwork(**kw), qnet.QNetwork(quantile=True, quantiles=1, kappa=16.0, **kw)
    assert torch.equal(plain.params, one.params) and torch.equal(plain.target, one.target) and plain.offsets == one.offsets
    outs = []
    for net in (plain, one):
        mem = _memory(game, replay, 48, 20, n, per, B, 30)
        ae, qt = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
        sp, mb = mem.step_sampling(B)
        net.loss_backward(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32 if per else None, GAMMA, False, None, ae,
                          qt, sampling=sp)
        torch.cuda.synchronize()
        outs.append((net.loss.item(), net.grads.cpu().numpy().astype(np.float64), ae.cpu().numpy().astype(np.float64),
                     qt.cpu().numpy().astype(np.float64)))
    (l0, g0, e0, y0), (l1, g1, e1, y1) = outs
    assert np.abs(e0).max() <= 16.0
    tol = 1e-5 if precision == "fp32" else 1e-4
    rep = {k: float(np.linalg.norm(g1[o:o + int(np.prod(s))] - g0[o:o + int(np.prod(s))] / 64) / np.linalg.norm(g0[o:o + int(np.prod(s))] / 64))
           for k, (o, s) in ((k, v) for k, v in qr.layout(512, dueling, 1).items() if k != "total")}
    print(f"\n[{variant} per={per} dueling={dueling} {precision}] loss {abs(l1 - l0 / 64) / (l0 / 64):.1e} " +
          " ".join(f"{k} {v:.1e}" for k, v in rep.items()))
    assert abs(l1 - l0 / 64) <= tol * l0 / 64
    assert all(v <= tol for k, v in rep.items() if precision == "fp32" or k not in CONV), rep
    np.testing.assert_allclose(e1, e0 * e0 / 64, rtol=1e-4, atol=1e-8)
    np.testing.assert_allclose(y1, y0, rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------- 5. determinism and graphs
@pytest.mark.parametrize("variant,dueling,per,n", [("nature", False, True, 3), ("double", True, False, 1)])
def test_graph_replay_is_bit_identical_to_eager(mods, variant, dueling, per, n):
    game, replay, qnet, _, _lib = mods
    B = 32
    nets = [_net(qnet, B, dueling, "fp16", lr=1e-4) for _ in range(2)]
    _lib.check(nets[1]._L.fb_qnet_use_graphs(nets[1]._h, 0), "fb_qnet_use_graphs")
    mems = [_memory(game, replay, 48, 20, n, per, B, 30) for _ in range(2)]
    bufs = [[torch.zeros(B, device="cuda") for _ in range(2)] for _ in range(2)]
    for u in range(20):
        for net, mem, (ae, qt) in zip(nets, mems, bufs):
            if u % 7 == 6:
                net.sync_target()
            sp, mb = mem.step_sampling(B)
            net.train_step(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32 if per else None, GAMMA, False, None,
                           ae, qt, sampling=sp)
        torch.cuda.synchronize()
        for x, y in ((nets[0].loss, nets[1].loss), (nets[0].grads, nets[1].grads), (nets[0].params, nets[1].params),
                     (nets[0].adam_m, nets[1].adam_m), (nets[0].adam_v, nets[1].adam_v), (bufs[0][0], bufs[1][0]), (bufs[0][1], bufs[1][1])):
            assert torch.equal(x, y), u
    assert torch.isfinite(nets[0].params).all() and nets[0].adam_steps == 20


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_train_step_is_loss_backward_plus_adam(mods, precision):
    game, replay, qnet, _, _ = mods
    B = 32
    nets = [_net(qnet, B, True, precision, lr=1e-4) for _ in range(2)]
    mems = [_memory(game, replay, 48, 20, 1, True, B, 30) for _ in range(2)]
    bufs = [[torch.zeros(B, device="cuda") for _ in range(2)] for _ in range(2)]
    for u in range(4):
        for k, (net, mem) in enumerate(zip(nets, mems)):
            sp, mb = mem.step_sampling(B)
            args = ("nature", mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32, GAMMA, False, None, *bufs[k])
            if k == 0:
                net.train_step(*args, sampling=sp)
            else:
                net.loss_backward(*args, sampling=sp)
                net.adam_step()
        torch.cuda.synchronize()
        for name in ("loss", "grads", "params", "adam_m", "adam_v"):
            assert torch.equal(getattr(nets[0], name), getattr(nets[1], name)), (u, name)
        assert torch.equal(bufs[0][0], bufs[1][0]) and torch.equal(bufs[0][1], bufs[1][1])


# -------------------------------------------------------------------------------------------------------- 6. noisy QR
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
def test_noisy_sigma_zero_is_the_plain_qr_update(mods, dueling, precision):
    game, replay, qnet, _, _ = mods
    B = 32
    nets = [_net(qnet, B, dueling, precision, lr=1e-4, noisy=noisy, sigma0=0.0) for noisy in (True, False)]
    outs = []
    for net in nets:
        mem = _memory(game, replay, 48, 20, 3, True, B, 30)
        ae, qt = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
        sp, mb = mem.step_sampling(B)
        net.train_step("double", mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32, GAMMA, False, None, ae, qt, sampling=sp)
        outs.append((net.loss, net.grads, ae, qt, net.params, net.adam_m, net.adam_v))
    torch.cuda.synchronize()
    lay = nets[0].noise_layout
    assert lay[-1]["q"] == 2 * NQ and (not dueling or lay[1]["q"] == NQ)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_noisy_qr_update_matches_the_oracle_on_weff(mods, precision):
    game, replay, qnet, _, _ = mods
    B, n, dueling = 32, 3, True
    net = _net(qnet, B, dueling, precision, noisy=True)
    W, WT = _spread_params(dueling, 512, 1), _spread_params(dueling, 512, 2)
    net.params.copy_(torch.from_numpy(W)); net.target.copy_(torch.from_numpy(WT))
    net.sigma.mul_(4.0); net.target_sigma.mul_(4.0)
    mem = _memory(game, replay, 64, 30, n, False, B, 60)
    abs_err, y = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
    sp, mb = mem.step_sampling(B)
    net.loss_backward("double", mb.frames, mb.actions, mb.rewards, mb.terminals, None, GAMMA, False, None, abs_err, y, sampling=sp)
    torch.cuda.synchronize()
    weff, weff_t = net.weff.cpu().numpy(), net.weff_target.cpu().numpy()
    assert not np.array_equal(weff, W)
    _check_against_oracle(net, mb, False, n, "double", dueling, False, 512, precision, weff, weff_t, abs_err, y)


# -------------------------------------------------------------------------------------------------------------- 7. Brains
@pytest.mark.parametrize("name,extra", [("dqn", {}), ("dqnnature", {}), ("ddqn", {}), ("duelingdqn", {}), ("prioritydqn", {}),
                                        ("ddqn", {"noisy": True, "n_step": 3, "initial_epsilon": 0.0})])
def test_every_brain_trains(mods, name, extra):
    game, _, _, brains, _ = mods
    N, C_, steps = 64, 12, 207
    brain = brains.MODELS[name](2, "bird", num_envs=N, replay_memory_per_env=C_, observe=6., batch_size=32, seed=1, lr=1e-4,
                                replace_target_iter=20, quantile=True, **extra)
    assert brain.net.quantile and brain.net.quantiles == 32 and brain.net.kappa == 1.0 and not brain.net.distributional
    gs = game.GameState(num_envs=N, seed=2, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    p0 = brain.net.params.clone()
    losses = []
    for _ in range(steps):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
        brain.setPerception(obs, a, r, t, s)
        losses.append(brain.net.loss.clone())
    gs.check_errors()
    assert brain.net.adam_steps == steps - 7
    assert torch.isfinite(torch.cat(losses)).all() and torch.isfinite(brain.net.params).all()
    assert not torch.equal(brain.net.params, p0)


# ---------------------------------------------------------------------------------------------------------- 8. checkpoint
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_checkpoint_round_trip(mods, tmp_path, precision):
    game, _, qnet, _, _ = mods
    B = 32
    gs = game.GameState(num_envs=B, seed=7, history=5)
    gs.step_random(45, 0.3, 11)
    frames = gs.ring[:, [(gs.slot - 4 + k) % 5 for k in range(5)]].contiguous()
    rng = np.random.default_rng(0)
    a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
    r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
    t = (r == -3.0).to(torch.uint8)
    fb = qnet.FrameBatch.from_stack(frames)
    A = _net(qnet, B, precision=precision, seed=3, lr=1e-4)
    for _ in range(3):
        A.train_step("nature", frames, a, r, t)
    A.sync_target()
    torch.save(A.state_dict(), tmp_path / "ck.pt")

    def step(net):
        net.train_step("double", frames, a, r, t)
        th, q = net.forward_quantiles(fb)
        torch.cuda.synchronize()
        return [x.clone() for x in (net.loss, net.grads, net.params, net.target, net.adam_m, net.adam_v, th, q)]
    want = step(A)
    Bn = _net(qnet, B, precision=precision, seed=99, lr=1e-4)
    Bn.load_state_dict(torch.load(tmp_path / "ck.pt", map_location="cuda"))
    got = step(Bn)
    for i, (x, y) in enumerate(zip(want, got)):
        assert torch.equal(x, y), i
    others = [qnet.QNetwork(max_batch=B, seed=3, precision=precision),
              qnet.QNetwork(max_batch=B, seed=3, precision=precision, distributional=True, atoms=NQ),
              _net(qnet, B, precision=precision, quantiles=16),
              _net(qnet, B, precision=precision, kappa=0.0),
              _net(qnet, B, precision=precision, quantiles=1)]
    for o in others:
        with pytest.raises(AssertionError):
            o.load_state_dict(A.state_dict())
        with pytest.raises(AssertionError):
            A.load_state_dict(o.state_dict())


# ----------------------------------------------------------------------------------------------------------- 9. refusals
def test_what_a_qr_net_refuses(mods):
    game, _, qnet, brains, _lib = mods
    L = _lib.lib()
    h = C.c_void_p()
    for args in ((512, 0, 8, 0, 1.0), (512, 0, 8, 65, 1.0), (512, 0, 8, 32, -0.5), (512, 0, 8, 32, float("inf")),
                 (512, 0, 8, 32, float("nan")), (500, 0, 8, 32, 1.0), (4096, 0, 8, 32, 1.0), (512, 0, 0, 32, 1.0)):
        assert L.fb_qnet_create_qr(*args, C.byref(h)) == -1, args
    gs = game.GameState(num_envs=8, seed=1, history=5)
    gs.step_random(6, 0.3, 1)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    th, q = torch.empty(8, 2, 64, device="cuda"), torch.empty(8, 2, device="cuda")
    plain = qnet.QNetwork(max_batch=8, seed=1, precision="fp16")
    c51 = qnet.QNetwork(max_batch=8, seed=1, precision="fp16", distributional=True, atoms=NQ)
    for other in (plain, c51):
        assert L.fb_qnet_forward_quantiles(other._h, other.params.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, 8, th.data_ptr(),
                                           q.data_ptr(), other._stream()) == -1
        with pytest.raises(ValueError):
            other.forward_quantiles(fb)
    with pytest.raises(ValueError):
        qnet.QNetwork(max_batch=8, precision="fp16", distributional=True, quantile=True)
    for precision in ("fp32", "fp16"):
        net = _net(qnet, 8, precision=precision)
        assert L.fb_qnet_forward_dist(net._h, net.params.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, 8, th.data_ptr(), q.data_ptr(),
                                      net._stream()) == -1
        with pytest.raises(ValueError):
            net.forward_dist(fb)
        assert L.fb_debug_qr_loss(plain._h, th.data_ptr(), th.data_ptr(), th.data_ptr(), th.data_ptr(), th.data_ptr(), None, None, GAMMA, 8,
                                  th.data_ptr(), q.data_ptr(), net._stream()) == -1
        net.set_per_broadcast(True)
        frames = gs.ring[:, [(gs.slot - 4 + k) % 5 for k in range(5)]].contiguous()
        z8 = torch.zeros(8, dtype=torch.uint8, device="cuda")
        with pytest.raises(_lib.FlappyError):
            net.loss_backward("nature", frames, z8, torch.zeros(8, device="cuda"), z8, torch.ones(8, device="cuda"))
        from dqnflappybird_b200.dist import PeerGradExchange
        x = PeerGradExchange(net.n_params, "cuda:0", rank=0, world=2, connect=False)
        assert L.fb_qnet_attach_exchange(net._h, x._h) == -1
        assert L.fb_qnet_attach_exchange(net._h, None) == 0
        with pytest.raises(ValueError):
            net.enable_peer_exchange(x)
    for kw in ({"reference_quirks": True}, {"peer_exchange": True}, {"distributional": True}):
        with pytest.raises(ValueError):
            brains.BrainPrioritizedReplyDQN(2, "bird", num_envs=8, replay_memory_per_env=4, quantile=True, **kw)


# -------------------------------------------------------------------------------------------------------- 10. two ranks
def test_two_ranks_under_nccl():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "qr_two_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "QR_TWO_RANK_OK" in r.stdout
