"""The distributional (C51) head on the device (csrc/fb_c51.cu, QNetwork(distributional=True), Brain*(distributional=True)) against
the float64 oracle (oracle/c51_oracle.py) and against itself:

1. the projection of fb_debug_c51_project is bit-identical to the oracle's float64 projection rounded to fp32;
2. forward: p sums to 1, p and Q against the oracle, acting picks the first argmax of the Q it returns, chunked acting;
3. loss, every gradient tensor, abs_err and q_target against the oracle (fp32, and fp16 in two tiers);
4. graph replays are bit-identical to eager steps, and train_step to loss_backward + adam_step;
5. noisy C51: sigma0 = 0 is the plain C51 update, and one update against the oracle on the read-back W_eff;
6. every Brain trains; 7. checkpoints; 8. what a C51 net refuses."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import c51_oracle as c5  # noqa: E402

GAMMA = 0.99
VARIANTS = {"vanilla": 0, "nature": 1, "double": 2}
N_ATOMS, V_MIN, V_MAX = 51, -10.0, 20.0


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


def _net(qnet, B, dueling=False, precision="fp16", hidden=512, seed=4, **kw):
    return qnet.QNetwork(max_batch=B, hidden=hidden, dueling=dueling, seed=seed, precision=precision, distributional=True, atoms=N_ATOMS,
                         v_min=V_MIN, v_max=V_MAX, **kw)


def _spread_params(dueling, hidden, seed):
    """weights scaled up from the initialisation so that the distributions are far from uniform"""
    return c5.init_params(hidden, dueling, N_ATOMS, seed=seed) * np.float32(3.0)


def _ring_frames(gs):
    L = gs.ring.shape[1]
    return gs.ring[:, [(gs.slot - 3 + k) % L for k in range(4)]].cpu().numpy()


# -------------------------------------------------------------------------------------------------------- 1. projection
def test_projection_is_bit_exact(mods):
    game, replay, qnet, _, _lib = mods
    B = 96
    net = _net(qnet, B)
    net.params.copy_(torch.from_numpy(_spread_params(False, 512, 1)))
    gs = game.GameState(num_envs=B, seed=5, history=7)
    gs.step_random(20, 0.4, 3)
    probs, _ = net.forward_dist(qnet.FrameBatch.from_ring(gs.ring, gs.slot))
    p = probs[:, 1].contiguous()                                             # the device's own fp32 probabilities
    rng = np.random.default_rng(0)
    # 1-step rows (0.1 / 3 / -3, some terminal), and n = 3 rows whose targets clip at both ends
    r = torch.from_numpy(rng.choice(np.float32([0.1, 3.0, -3.0]), B)).cuda()
    t = torch.from_numpy((rng.random(B) < 0.3).astype(np.uint8)).cuda()
    R = rng.uniform(-25.0, 40.0, B)
    R[:8] = [25.0, -15.0, 30.0, -30.0, 19.999, -9.999, 0.1, 3.0]
    d = np.where(rng.random(B) < 0.25, 0.0, GAMMA ** 3)
    d[:6] = [0.0, 0.0, GAMMA ** 3, GAMMA ** 3, 0.0, 0.0]
    out = torch.empty(B, N_ATOMS, device="cuda")
    L, st = net._L, net._stream()
    pn = p.cpu().numpy()
    for ret, disc in ((None, None), (R, d)):
        if ret is None:
            rc = L.fb_debug_c51_project(net._h, p.data_ptr(), r.data_ptr(), t.data_ptr(), None, None, GAMMA, B, out.data_ptr(), st)
            Rr, dd = c5.one_step_targets(r.cpu().numpy(), t.cpu().numpy(), GAMMA)
        else:
            rt, dt = torch.from_numpy(ret).cuda(), torch.from_numpy(disc).cuda()
            rc = L.fb_debug_c51_project(net._h, p.data_ptr(), None, None, rt.data_ptr(), dt.data_ptr(), GAMMA, B, out.data_ptr(), st)
            Rr, dd = ret, disc
        _lib.check(rc, "fb_debug_c51_project")
        torch.cuda.synchronize()
        want = c5.project(pn, Rr, dd, N_ATOMS, V_MIN, V_MAX).astype(np.float32)
        got = out.cpu().numpy()
        assert np.array_equal(got, want), np.abs(got - want).max()
        assert (dd == 0).any()
    top, bottom = np.eye(N_ATOMS, dtype=bool)[-1], np.eye(N_ATOMS, dtype=bool)[0]     # clipped above / below: one end atom
    assert all(np.array_equal(got[b] > 0, e) for b, e in ((0, top), (1, bottom), (2, top), (3, bottom)))


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
    probs, q = net.forward_dist(fb)
    torch.cuda.synchronize()
    p, q = probs.cpu().numpy(), q.cpu().numpy()
    assert np.abs(p.astype(np.float64).sum(-1) - 1.0).max() <= 1e-6
    x = _ring_frames(gs)
    p_ref, q_ref = c5.forward(W, x, 512, dueling, N_ATOMS, V_MIN, V_MAX, emulate=None if precision == "fp32" else "fp16")
    # p to `tol`; Q = sum z p carries p's error times the atoms, so Q is held to `tol` of the support's width
    tol = 2e-5 if precision == "fp32" else 5e-4
    print(f"\n[{precision}] p {np.abs(p - p_ref).max():.2e}  Q {np.abs(q - q_ref).max():.2e}")
    assert np.abs(p - p_ref).max() <= tol and np.abs(q - q_ref).max() <= tol * (V_MAX - V_MIN)
    assert p.std(-1).mean() > 1e-3                                        # not uniform: the head is exercised
    assert torch.equal(net.forward(fb), torch.from_numpy(q).cuda())
    # epsilon = 0 acting: the first argmax of the Q it returns
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
    probs, q = net.forward_dist(fb)
    rng_pos = torch.zeros(N, dtype=torch.int32, device="cuda")
    acts, q_out = torch.zeros(N, dtype=torch.uint8, device="cuda"), torch.zeros(N, 2, device="cuda")
    net.act(fb, 0.0, 3, 0, rng_pos, acts, q_out)
    L = gs.ring.shape[1]
    for c0 in range(0, N, MB):
        n = min(MB, N - c0)
        part = qnet.FrameBatch(gs.ring, L * 6400, [((gs.slot - 3 + k) % L) * 6400 for k in range(4)], n, base_offset=c0 * L * 6400)
        pc, qc = net.forward_dist(part)
        assert torch.equal(pc, probs[c0:c0 + n]) and torch.equal(qc, q[c0:c0 + n]) and torch.equal(q_out[c0:c0 + n], qc), c0
    assert torch.equal(acts, (q_out[:, 1] > q_out[:, 0]).to(torch.uint8))


# -------------------------------------------------------------------------------------------------------- 3. the oracle
CASES = [  # variant, dueling, loss_sum, per, n
    ("vanilla", False, True, False, 1), ("nature", False, False, False, 1), ("double", False, False, False, 1),
    ("nature", True, False, False, 1), ("double", True, False, True, 1), ("nature", False, False, True, 3), ("double", False, False, False, 3)]
HEAD = {False: ["wf2", "bf2"], True: ["wv", "bv", "wa", "ba"]}


def _per_tensor(g, g_ref, dueling, hidden):
    out = {}
    for name, (o, shp) in ((k, v) for k, v in c5.layout(hidden, dueling, N_ATOMS).items() if k != "total"):
        sz = int(np.prod(shp))
        out[name] = float(np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) / np.linalg.norm(g_ref[o:o + sz]))
    return out


def _oracle_targets(mb, n):
    if n > 1:
        return mb.returns.cpu().numpy(), mb.disc.cpu().numpy()
    return c5.one_step_targets(mb.rewards.cpu().numpy(), mb.terminals.cpu().numpy(), GAMMA)


def _check_against_oracle(net, mb, per, n, variant, dueling, loss_sum, hidden, precision, W, WT, abs_err, y):
    """fp32: loss and every tensor 2e-4.  fp16, tier A (oracle with the same roundings): loss 5e-4, each head tensor 1.5e-3 and the
    whole gradient vector 1.5e-3; tier B (exact oracle): loss 4e-3, every tensor 4.5e-2.  abs_err and q_target (relative norm of the
    vector) at the loss tolerance.
    Tier A is not asserted per tensor on the trunk: the n-step and noisy work measured the convolution backward's rounding-decision
    flips at 1.5e-3 .. 8e-3 against the emulating oracle.  With prioritized replay (IS weights put the gradient on a few samples) those
    flips are not averaged out and the whole vector is held to 5e-3 instead: a B200 measured it at 2.6e-3 .. 2.9e-3, conv1 .. conv3
    at 2.3e-3 .. 4.1e-3 (fc1 2.3e-3 at hidden 256), while every head tensor stayed within 1e-4 and the loss within 1e-5."""
    x = mb.frames.cpu().numpy()
    m = min(n, 4)
    R, d = _oracle_targets(mb, n)
    isw = mb.is_weights_f32.cpu().numpy() if per else None
    g = net.grads.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    tiers = [(None, 2e-4, 2e-4)] if precision == "fp32" else [("fp16", 5e-4, 1.5e-3), (None, 4e-3, 4.5e-2)]
    for emulate, tol_loss, tol_g in tiers:
        loss, r, ce, qt, _, _ = c5.loss_and_grads(VARIANTS[variant], W, WT, x[:, 0:4], x[:, m:m + 4], mb.actions.cpu().numpy(), R, d, isw,
                                                  loss_sum, None, hidden, dueling, emulate, N_ATOMS, V_MIN, V_MAX)
        rep = _per_tensor(g, r, dueling, hidden)
        whole = float(np.linalg.norm(g - r) / np.linalg.norm(r))
        lo = abs(net.loss.item() - loss) / abs(loss)
        print(f"\n[{precision}/{emulate}] loss {lo:.2e}  grads {whole:.2e}  " + " ".join(f"{k} {v:.1e}" for k, v in rep.items()))
        assert lo <= tol_loss, (net.loss.item(), loss)
        assert np.linalg.norm(abs_err.cpu().numpy() - ce) <= tol_loss * np.linalg.norm(ce)
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


# ------------------------------------------------------------------------------------------- 4. determinism and graphs
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


# ------------------------------------------------------------------------------------------------------- 5. noisy C51
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("dueling", [False, True])
def test_noisy_sigma_zero_is_the_plain_c51_update(mods, dueling, precision):
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
    assert lay[-1]["q"] == 2 * N_ATOMS and (not dueling or lay[1]["q"] == N_ATOMS)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_noisy_c51_update_matches_the_oracle_on_weff(mods, precision):
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


# -------------------------------------------------------------------------------------------------------------- 6. Brains
@pytest.mark.parametrize("name,extra", [("dqn", {}), ("dqnnature", {}), ("ddqn", {}), ("duelingdqn", {}), ("prioritydqn", {}),
                                        ("ddqn", {"noisy": True, "n_step": 3, "initial_epsilon": 0.0})])
def test_every_brain_trains(mods, name, extra):
    game, _, _, brains, _ = mods
    N, C_, steps = 64, 12, 207
    brain = brains.MODELS[name](2, "bird", num_envs=N, replay_memory_per_env=C_, observe=6., batch_size=32, seed=1, lr=1e-4,
                                replace_target_iter=20, distributional=True, **extra)
    assert brain.net.distributional and brain.net.atoms == 51 and (brain.net.v_min, brain.net.v_max) == (-10.0, 20.0)
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


# ---------------------------------------------------------------------------------------------------------- 7. checkpoint
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
        pr, q = net.forward_dist(fb)
        torch.cuda.synchronize()
        return [x.clone() for x in (net.loss, net.grads, net.params, net.target, net.adam_m, net.adam_v, pr, q)]
    want = step(A)
    Bn = _net(qnet, B, precision=precision, seed=99, lr=1e-4)
    Bn.load_state_dict(torch.load(tmp_path / "ck.pt", map_location="cuda"))
    got = step(Bn)
    for i, (x, y) in enumerate(zip(want, got)):
        assert torch.equal(x, y), i
    plain = qnet.QNetwork(max_batch=B, seed=3, precision=precision)
    with pytest.raises(AssertionError):
        plain.load_state_dict(A.state_dict())
    with pytest.raises(AssertionError):
        A.load_state_dict(plain.state_dict())
    other = qnet.QNetwork(max_batch=B, seed=3, precision=precision, distributional=True, atoms=N_ATOMS, v_min=-10.0, v_max=10.0)
    with pytest.raises(AssertionError):
        other.load_state_dict(A.state_dict())


# ----------------------------------------------------------------------------------------------------------- 8. refusals
def test_what_a_c51_net_refuses(mods):
    game, _, qnet, brains, _lib = mods
    L = _lib.lib()
    h = C.c_void_p()
    for args in ((512, 0, 8, 1, -10.0, 20.0), (512, 0, 8, 65, -10.0, 20.0), (512, 0, 8, 51, 20.0, 20.0), (512, 0, 8, 51, 5.0, -5.0),
                 (512, 0, 8, 51, float("-inf"), 20.0), (512, 0, 8, 51, -10.0, float("nan")), (500, 0, 8, 51, -10.0, 20.0)):
        assert L.fb_qnet_create_c51(*args, C.byref(h)) == -1, args
    plain = qnet.QNetwork(max_batch=8, seed=1, precision="fp16")
    gs = game.GameState(num_envs=8, seed=1, history=5)
    gs.step_random(6, 0.3, 1)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    pr, q = torch.empty(8, 2, 51, device="cuda"), torch.empty(8, 2, device="cuda")
    assert L.fb_qnet_forward_dist(plain._h, plain.params.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, 8, pr.data_ptr(), q.data_ptr(),
                                  plain._stream()) == -1
    with pytest.raises(ValueError):
        plain.forward_dist(fb)
    for precision in ("fp32", "fp16"):
        net = _net(qnet, 8, precision=precision)
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
    for kw in ({"reference_quirks": True}, {"peer_exchange": True}):
        with pytest.raises(ValueError):
            brains.BrainPrioritizedReplyDQN(2, "bird", num_envs=8, replay_memory_per_env=4, distributional=True, **kw)
