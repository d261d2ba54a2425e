"""Noisy networks on the device (csrc/fb_noisy.cu, QNetwork(noisy=True), Brain*(noisy=True)) against the oracle
(oracle/noisy_oracle.py) and against a recomposition from the library's existing calls:

1. factor vectors within 1 fp32 ulp of the oracle's Box-Muller; W_eff bit-identical to torch's mu + sigma * outer(f_in, f_out);
2. sigma0 = 0: one update bit-identical to the plain net's;
3. 20 graph-replayed updates bit-identical to: the read-back factors -> W_eff in torch -> the plain gradient-only step ->
   fb_qnet_adam on (mu, g) and on (sigma, g * eps);
4. loss, dL/dmu and dL/dsigma against the float64 oracle;
5. acting: noise=False is the plain act bit for bit, with noise Q is the oracle forward on the acting draw's W_eff;
6. every Brain trains; 7. a checkpoint round trip is invisible; 8. replicas stay bit-identical on the all-reduce path."""
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import noisy_oracle as nz  # noqa: E402
from oracle import qnet_oracle as qo  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAMMA = 0.99


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dqnflappybird_b200 import _lib, brains, game, qnet, replay
    return game, replay, qnet, brains, _lib


def _memory(game, replay, N, C, n, per, B, steps, seed=3):
    """a memory filled by `steps` random-action env steps (p_flap 0.5: windows straddle crashes); same seed, same contents"""
    ring = torch.zeros((N, C + n + 3, 80, 80), dtype=torch.uint8, device="cuda")
    mem = (replay.PrioritizedMemory(ring, C, seed=7, max_batch=B, mode="rebuild", n_step=n) if per
           else replay.ReplayMemory(ring, C, seed=7, max_batch=B, n_step=n))
    gs = game.GameState(num_envs=N, seed=seed, history=mem.L, ring=mem.ring)
    gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    for k in range(1, steps + 1):
        a, r, t = mem.rows(k)
        gs.step_random(1, 0.5, 21, a, r, t, None)
        mem.appended(k)
    return mem


def _eps(net, fac):
    """eps per parameter in torch float32 (one rounding per product), 0 outside the noisy layers; and the noisy mask"""
    e = torch.zeros(net.n_params, dtype=torch.float32, device="cuda")
    mask = torch.zeros(net.n_params, dtype=torch.bool, device="cuda")
    for ly in net.noise_layout:
        p, q = ly["p"], ly["q"]
        fin, fout = fac[ly["f_in"]:ly["f_in"] + p], fac[ly["f_out"]:ly["f_out"] + q]
        e[ly["w"]:ly["w"] + p * q] = (fin[:, None] * fout[None, :]).reshape(-1)
        e[ly["b"]:ly["b"] + q] = fout
        mask[ly["w"]:ly["w"] + p * q] = True
        mask[ly["b"]:ly["b"] + q] = True
    return e, mask


def _weff(mu, sigma, e, mask):
    return torch.where(mask, mu + sigma * e, mu)


def _ulps(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia); ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


# ------------------------------------------------------------------------------------------------------------ 1. draws
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
def test_draws_match_the_oracle_and_weff_is_torch_fp32(mods, dueling, precision):
    game, replay, qnet, _, _ = mods
    net = qnet.QNetwork(max_batch=8, dueling=dueling, seed=3, precision=precision, noisy=True)
    layers, n = nz.noise_layout(512, dueling)
    assert net.n_factors == n and net.noise_layout == layers
    seen = []
    for seed, role, counter in ((0, "online", 0), (3, "target", 0), (3, "act", 5), (12345, "online", 2 ** 40 + 7)):
        net.noise_seed = seed
        fac = net.draw_noise(role, counter).cpu().numpy()
        want = nz.factors(seed, role, counter, 512, dueling)
        assert _ulps(fac, want).max() <= 1, (seed, role, counter, _ulps(fac, want).max())
        seen.append(fac)
    assert all(not np.array_equal(seen[i], seen[j]) for i in range(4) for j in range(i))
    # W_eff from the device's own factors, at a sigma with varied entries
    fac = net.draw_noise("online", 3)
    g = torch.Generator(device="cuda").manual_seed(1)
    net.sigma.mul_(torch.rand(net.n_params, device="cuda", generator=g) * 4)
    w = net.noisy_weights(net.params, net.sigma, fac, torch.empty_like(net.params))
    e, mask = _eps(net, fac)
    assert torch.equal(w, _weff(net.params, net.sigma, e, mask))
    assert torch.equal(w[~mask], net.params[~mask]) and not torch.equal(w, net.params)


# --------------------------------------------------------------------------------------------- 2. sigma0 = 0 is the plain net
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("variant,dueling,per", [("nature", False, False), ("double", False, False), ("nature", True, False),
                                                 ("nature", False, True)])
def test_sigma_zero_update_is_the_plain_update(mods, variant, dueling, per, precision):
    game, replay, qnet, _, _ = mods
    B = 32
    nets = [qnet.QNetwork(max_batch=B, dueling=dueling, seed=4, lr=1e-4, precision=precision, noisy=noisy, sigma0=0.0)
            for noisy in (True, False)]
    outs = []
    for net in nets:
        mem = _memory(game, replay, 48, 20, 1, per, B, 30)
        abs_err, y = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
        sp, mb = mem.step_sampling(B)
        net.train_step(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32 if per else None, GAMMA, False,
                       None, abs_err, y, sampling=sp)
        outs.append((net.loss, net.grads, abs_err, y, net.params, net.adam_m, net.adam_v))
    torch.cuda.synchronize()
    assert nets[0].update_draws == 1
    for a, b in zip(*outs):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------------- 3. composition
COMPOSE = [  # variant, dueling, loss_sum, per, n
    ("vanilla", False, True, False, 1), ("nature", False, False, False, 1), ("double", False, False, False, 1),
    ("nature", True, False, False, 1), ("nature", False, False, True, 1), ("double", False, False, False, 3)]


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("variant,dueling,loss_sum,per,n", COMPOSE)
def test_noisy_update_is_its_recomposition(mods, variant, dueling, loss_sum, per, n, precision):
    game, replay, qnet, _, _lib = mods
    B, lr = 32, 1e-4
    net = qnet.QNetwork(max_batch=B, dueling=dueling, seed=4, lr=lr, precision=precision, noisy=True)
    ref = qnet.QNetwork(max_batch=B, dueling=dueling, seed=4, lr=lr, precision=precision)
    mem_a, mem_b = (_memory(game, replay, 48, 20, n, per, B, 30) for _ in range(2))
    mu, tmu, sg, tsg = net.params.clone(), net.target.clone(), net.sigma.clone(), net.target_sigma.clone()
    m, v, sm, sv = (torch.zeros_like(mu) for _ in range(4))
    b1p, b2p = np.float32(0.9), np.float32(0.999)
    L, st = ref._L, ref._stream()
    bufs = [torch.zeros(B, device="cuda") for _ in range(4)]
    for u in range(20):
        if variant != "vanilla" and u % 5 == 4:
            net.sync_target(); tmu.copy_(mu); tsg.copy_(sg)
        sp, mb = mem_a.step_sampling(B)
        net.train_step(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32 if per else None, GAMMA, loss_sum,
                       None, bufs[0], bufs[1], sampling=sp)
        e, mask = _eps(net, net.noise_online.clone())
        ref.params.copy_(_weff(mu, sg, e, mask))
        if variant != "vanilla":
            et, _ = _eps(net, net.noise_target.clone())
            ref.target.copy_(_weff(tmu, tsg, et, mask))
        sp, mb = mem_b.step_sampling(B)
        ref.loss_backward(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, mb.is_weights_f32 if per else None, GAMMA, loss_sum,
                          None, bufs[2], bufs[3], sampling=sp)
        alpha = float(np.float32(np.float32(lr) * np.sqrt(np.float32(1) - b2p) / (np.float32(1) - b1p)))
        _lib.check(L.fb_qnet_adam(ref._h, mu.data_ptr(), ref.grads.data_ptr(), m.data_ptr(), v.data_ptr(), alpha, 0.9, 0.999, 1e-8, 1.0, st))
        g_sigma = ref.grads * e
        _lib.check(L.fb_qnet_adam(ref._h, sg.data_ptr(), g_sigma.data_ptr(), sm.data_ptr(), sv.data_ptr(), alpha, 0.9, 0.999, 1e-8, 1.0, st))
        b1p, b2p = np.float32(b1p * np.float32(0.9)), np.float32(b2p * np.float32(0.999))
        assert torch.equal(net.loss, ref.loss) and torch.equal(net.grads, ref.grads), u
        assert torch.equal(bufs[0], bufs[2]) and torch.equal(bufs[1], bufs[3]), u
    net.sync_target(); tmu.copy_(mu); tsg.copy_(sg)
    torch.cuda.synchronize()
    assert net.update_draws == net.adam_steps == 20
    for a, b in ((net.params, mu), (net.sigma, sg), (net.target, tmu), (net.target_sigma, tsg), (net.adam_m, m), (net.adam_v, v),
                 (net.sigma_m, sm), (net.sigma_v, sv)):
        assert torch.equal(a, b)
    assert (sv[mask] > 0).float().mean() > 0.5 and (sm[~mask] == 0).all()
    assert not torch.equal(sg, torch.from_numpy(nz.sigma_init(512, dueling)).cuda())       # sigma has moved


# ---------------------------------------------------------------------------------------------------------- 4. the oracle
CASES = [  # variant, dueling, loss_sum, per, n
    ("vanilla", False, True, False, 1), ("nature", False, False, False, 1), ("double", False, False, False, 1),
    ("nature", True, False, False, 1), ("double", True, False, True, 1), ("nature", False, False, True, 3), ("double", False, False, False, 3)]


def _per_tensor(g, g_ref, dueling, names=None):
    out = {}
    for name, (o, shp) in ((k, v) for k, v in qo.layout(512, dueling).items() if k != "total"):
        if names is not None and name not in names:
            continue
        sz = int(np.prod(shp))
        out[name] = float(np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) / np.linalg.norm(g_ref[o:o + sz]))
    return out


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("B", [32, 256])
@pytest.mark.parametrize("variant,dueling,loss_sum,per,n", CASES)
def test_loss_and_gradients_match_the_oracle(mods, variant, dueling, loss_sum, per, n, B, precision):
    """fp32: loss, dL/dmu per tensor and dL/dsigma per noisy tensor to 2e-4.  fp16, the two tiers of tests/test_nstep_gpu.py:
    (A) against the oracle with the same roundings, loss 5e-4 and 1.5e-3 on the whole dL/dsigma and on dL/dmu of the noisy layers;
    (B) against the exact oracle, loss 4e-3 and every tensor of dL/dmu and dL/dsigma 4.5e-2.
    Tier A is not asserted on the convolution gradients: with prioritized replay (IS weights put the gradient on a few samples) a B200
    measured conv1 .. conv3 6e-3 .. 8e-3 from the emulating oracle (the whole dL/dmu 4.9e-3) while every dL/dsigma tensor stayed
    within 3e-4, the loss within 2e-5, and the same cases in fp32 within 3e-6.  Those gradients are bit-identical to the plain fp16
    step's on the same W_eff (test_noisy_update_is_its_recomposition): it is the convolution backward's rounding-decision flips that
    tests/test_nstep_gpu.py describes, not the noise."""
    if B == 256 and (precision, variant, dueling, per, n) not in (("fp16", "nature", False, False, 1), ("fp32", "double", True, True, 1),
                                                                  ("fp16", "double", False, False, 3)):
        pytest.skip("minibatch 256 runs a representative subset (the float64 oracle is slow at that size)")
    game, replay, qnet, _, _ = mods
    net = qnet.QNetwork(max_batch=B, dueling=dueling, seed=4, precision=precision, noisy=True)
    mu = qo.init_params(512, dueling, seed=1) * np.float32(3.0)
    tmu = qo.init_params(512, dueling, seed=2) * np.float32(3.0)
    rng = np.random.default_rng(5)
    sg = nz.sigma_init(512, dueling) * rng.uniform(0.5, 4.0, mu.size).astype(np.float32)
    tsg = nz.sigma_init(512, dueling) * rng.uniform(0.5, 4.0, mu.size).astype(np.float32)
    for t, a in ((net.params, mu), (net.target, tmu), (net.sigma, sg), (net.target_sigma, tsg)):
        t.copy_(torch.from_numpy(a))
    net.update_draws = 11
    mem = _memory(game, replay, 64, 30, n, per, B, 60)
    abs_err, y = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
    sp, mb = mem.step_sampling(B)
    isw = mb.is_weights_f32 if per else None
    net.loss_backward(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, isw, GAMMA, loss_sum, None, abs_err, y, sampling=sp)
    torch.cuda.synchronize()
    fac, fac_t = net.noise_online.cpu().numpy(), net.noise_target.cpu().numpy()
    assert _ulps(fac, nz.factors(4, "online", 11, 512, dueling)).max() <= 1
    x = mb.frames.cpu().numpy()
    m = min(n, 4)                                                         # s' = frames m..m+3 of a minibatch row
    kw = dict(returns=mb.returns.cpu().numpy(), disc=mb.disc.cpu().numpy()) if n > 1 else \
        dict(rewards=mb.rewards.cpu().numpy(), terminals=mb.terminals.cpu().numpy(), gamma=GAMMA)
    g_mu = net.grads.cpu().numpy().astype(np.float64)
    e32 = nz.eps_flat(fac, 512, dueling)
    g_sg = (net.grads.cpu().numpy() * e32).astype(np.float64)              # what the noisy Adam feeds sigma
    noisy_names = ["wf1", "bf1"] + (["wf2", "bf2"] if not dueling else ["wv", "bv", "wa", "ba"])
    assert np.isfinite(g_mu).all()
    for emulate, tol_loss, tol_g in ([(None, 2e-4, 2e-4)] if precision == "fp32" else [("fp16", 5e-4, 1.5e-3), (None, 4e-3, 4.5e-2)]):
        loss, r_mu, r_sg, _, y_ref, _ = nz.loss_and_grads(qnet.VARIANTS[variant], mu, sg, tmu, tsg, fac, fac_t, x[:, 0:4], x[:, m:m + 4],
                                                          mb.actions.cpu().numpy(), isw=isw.cpu().numpy() if per else None,
                                                          loss_sum=loss_sum, dueling=dueling, emulate=emulate, **kw)
        rep_mu, rep_sg = _per_tensor(g_mu, r_mu, dueling), _per_tensor(g_sg, r_sg, dueling, noisy_names)
        whole_mu = float(np.linalg.norm(g_mu - r_mu) / np.linalg.norm(r_mu))
        whole_sg = float(np.linalg.norm(g_sg - r_sg) / np.linalg.norm(r_sg))
        print(f"\n[{emulate}] loss {abs(net.loss.item() - loss) / abs(loss):.2e}  dmu {whole_mu:.2e} (worst {max(rep_mu.values()):.2e})  "
              f"dsigma {whole_sg:.2e} (worst {max(rep_sg.values()):.2e})")
        assert abs(net.loss.item() - loss) <= tol_loss * abs(loss), (net.loss.item(), loss)
        assert np.abs(y.cpu().numpy() - y_ref).max() <= tol_loss * np.abs(y_ref).max()
        if precision == "fp16" and emulate == "fp16":
            sel = np.zeros(g_mu.size, bool)
            for ly in nz.noise_layout(512, dueling)[0]:
                sel[ly["w"]:ly["b"] + ly["q"]] = True
            noisy_mu = float(np.linalg.norm(g_mu[sel] - r_mu[sel]) / np.linalg.norm(r_mu[sel]))
            assert noisy_mu <= tol_g and whole_sg <= tol_g, (noisy_mu, whole_sg, rep_mu, rep_sg)
        else:
            assert all(v <= tol_g for v in rep_mu.values()), (emulate, rep_mu)
            assert all(v <= tol_g for v in rep_sg.values()), (emulate, rep_sg)


# ------------------------------------------------------------------------------------------------------------- 5. acting
def _ring_frames(gs):
    L = gs.ring.shape[1]
    return gs.ring[:, [(gs.slot - 3 + k) % L for k in range(4)]].cpu().numpy()


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
def test_acting(mods, dueling, precision):
    game, _, qnet, _, _ = mods
    N = 300
    gs = game.GameState(num_envs=N, seed=1, history=7)
    gs.step_random(20, 0.4, 3)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    noisy = qnet.QNetwork(max_batch=N, dueling=dueling, seed=3, precision=precision, noisy=True)
    plain = qnet.QNetwork(max_batch=N, dueling=dueling, seed=3, precision=precision)
    z = lambda dt, *s: torch.zeros(*s, dtype=dt, device="cuda")
    rp, rq = z(torch.int32, N), z(torch.int32, N)
    a1, a2, q1, q2 = z(torch.uint8, N), z(torch.uint8, N), z(torch.float32, N, 2), z(torch.float32, N, 2)
    plain.act(fb, 0.3, 11, 5, rp, a1, q1)
    noisy.act(fb, 0.3, 11, 5, rq, a2, q2, noise=False)
    assert torch.equal(a1, a2) and torch.equal(q1, q2) and torch.equal(rp, rq) and noisy.act_draws == 0
    # with noise: the acting draw's W_eff; the epsilon-greedy stream advances exactly as the plain net's
    noisy.act(fb, 0.3, 11, 5, rq, a2, q2)
    plain.act(fb, 0.3, 11, 5, rp, a1, q1)
    assert torch.equal(rp, rq) and noisy.act_draws == 1
    fac = noisy.noise_act.clone()
    assert torch.equal(fac, noisy.draw_noise("act", 0))
    e, mask = _eps(noisy, fac)
    W = _weff(noisy.params, noisy.sigma, e, mask)
    assert torch.equal(W, noisy.weff_act)
    x = _ring_frames(gs)
    q = q2.cpu().numpy()
    if precision == "fp32":
        ref = qo.forward(torch.tensor(W.cpu().numpy().astype(np.float64)), x, dueling=dueling).numpy()
        np.testing.assert_allclose(q, ref, rtol=1e-4, atol=1e-5)
    else:
        emu = qo.forward(torch.tensor(W.cpu().numpy().astype(np.float64)), x, dueling=dueling, emulate="fp16").numpy()
        assert np.abs(q - emu).max() <= 5e-4 * np.abs(emu).max()
    assert not torch.equal(q2, q1)
    q_first = q2.clone()
    noisy.act(fb, 0.3, 11, 5, rq, a2, q2)                                 # acting call 1: the next draw id
    assert noisy.act_draws == 2 and torch.equal(noisy.noise_act, noisy.draw_noise("act", 1)) and not torch.equal(q2, q_first)
    noisy.act_draws = 0                                                   # id 0 again: the same Q
    noisy.act(fb, 0.3, 11, 5, rq, a2, q2)
    assert torch.equal(q2, q_first)
    assert torch.equal(noisy.forward(fb, noise=False), plain.forward(fb))


# -------------------------------------------------------------------------------------------------------------- 6. Brains
@pytest.mark.parametrize("name,n_step", [("dqn", 1), ("dqnnature", 1), ("ddqn", 1), ("duelingdqn", 1), ("prioritydqn", 1), ("prioritydqn", 3),
                                         ("ddqn", 3)])
def test_every_brain_trains_with_noise(mods, name, n_step):
    game, _, _, brains, _ = mods
    N, C, steps = 64, 12, 300
    brain = brains.MODELS[name](2, "bird", num_envs=N, replay_memory_per_env=C, observe=6., batch_size=32, seed=1, lr=1e-4,
                                replace_target_iter=20, n_step=n_step, noisy=True, initial_epsilon=0.0)
    gs = game.GameState(num_envs=N, seed=2, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    mu0, sg0 = brain.net.params.clone(), brain.net.sigma.clone()
    losses = []
    for _ in range(steps):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
        brain.setPerception(obs, a, r, t, s)
        losses.append(brain.net.loss.clone())
    gs.check_errors()
    net = brain.net
    assert net.adam_steps == net.update_draws == steps - 7 and net.act_draws == steps
    assert torch.isfinite(torch.cat(losses)).all() and torch.isfinite(net.params).all() and torch.isfinite(net.sigma).all()
    assert not torch.equal(net.params, mu0) and not torch.equal(net.sigma, sg0)
    _, mask = _eps(net, net.noise_online)
    assert torch.equal(net.sigma[~mask], sg0[~mask])                      # zero outside the noisy layers, and it stays so


# ----------------------------------------------------------------------------------------------------------- 7. checkpoint
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
    A = qnet.QNetwork(max_batch=B, seed=3, lr=1e-4, precision=precision, noisy=True)
    for _ in range(3):
        A.train_step("nature", frames, a, r, t)
        A.forward(fb)
    A.sync_target()
    torch.save(A.state_dict(), tmp_path / "ck.pt")

    def step(net):
        net.train_step("double", frames, a, r, t)
        q = net.forward(fb)
        torch.cuda.synchronize()
        return [x.clone() for x in (net.loss, net.grads, net.params, net.sigma, net.target, net.target_sigma, net.adam_m, net.adam_v,
                                    net.sigma_m, net.sigma_v, q)] + [net.update_draws, net.act_draws]
    want = step(A)
    Bn = qnet.QNetwork(max_batch=B, seed=99, lr=1e-4, precision=precision, noisy=True, sigma0=0.1)
    Bn.load_state_dict(torch.load(tmp_path / "ck.pt", map_location="cuda"))
    got = step(Bn)
    for i, (x, y) in enumerate(zip(want, got)):
        assert (torch.equal(x, y) if torch.is_tensor(x) else x == y), i
    plain = qnet.QNetwork(max_batch=B, seed=3, precision=precision)
    with pytest.raises(AssertionError):
        plain.load_state_dict(A.state_dict())
    with pytest.raises(AssertionError):
        A.load_state_dict(plain.state_dict())


# ---------------------------------------------------------------------------------------------------------- 8. two ranks
def test_replicas_stay_identical_on_the_all_reduce_path(mods):
    """two replicas on two env shards, the NCCL path's arithmetic in one process: loss_backward on each shard (global mean loss),
    the gradient sum, the noisy Adam -- the draws do not depend on the rank, so mu and sigma stay bit-identical"""
    game, replay, qnet, brains, _ = mods
    B = 16
    nets = [qnet.QNetwork(max_batch=B, seed=5, lr=1e-4, precision="fp16", noisy=True) for _ in range(2)]
    mems = [_memory(game, replay, 32, 10, 1, False, B, 20, seed=3 + r) for r in range(2)]
    for u in range(6):
        for net, mem in zip(nets, mems):
            sp, mb = mem.step_sampling(B)
            net.loss_backward("nature", mb.frames, mb.actions, mb.rewards, mb.terminals, None, GAMMA, False, 2 * B, sampling=sp)
        assert torch.equal(nets[0].noise_online, nets[1].noise_online) and torch.equal(nets[0].noise_target, nets[1].noise_target)
        total = nets[0].grads + nets[1].grads
        for net in nets:
            net.grads.copy_(total)
            net.adam_step()
    for k in ("params", "sigma", "adam_m", "adam_v", "sigma_m", "sigma_v"):
        assert torch.equal(getattr(nets[0], k), getattr(nets[1], k)), k
    with pytest.raises(ValueError):
        brains.BrainDQNNature(2, "bird", num_envs=8, replay_memory_per_env=4, noisy=True, peer_exchange=True)
    with pytest.raises(ValueError):
        nets[0].enable_peer_exchange()


def test_two_ranks_under_nccl():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tests", "noisy_two_rank_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "NOISY_TWO_RANK_OK" in r.stdout
