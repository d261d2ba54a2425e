"""n-step returns on the device (fb_step_sampling.n_step; csrc/fb_replay.cu, the TD target of fb_qnet*.cu) against the oracle:
the drawn indices, the F gathered frames and R / disc bit for bit while the step's graph is replayed, n = 1 through the new path
bit-identical to the 1-step path, loss and gradients at the stated tolerances, and every Brain training with n_step = 3."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import nstep_oracle as no  # noqa: E402
from oracle import qnet_oracle as qo  # noqa: E402
from oracle import replay_oracle as ro  # noqa: E402

GAMMA = 0.99


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dqnflappybird_b200 import brains, game, qnet, replay
    return game, replay, qnet, brains


class Rollout:
    """random actions at p_flap 0.5 (every env crashes about every 50 steps, so windows straddle terminals) into the memory's
    ring and rows; the recorded history is what the oracle reads"""

    def __init__(self, game, mem, seed=5):
        self.mem = mem
        self.gs = game.GameState(num_envs=mem.N, seed=seed, history=mem.L, ring=mem.ring)
        self.gs.frame_step(torch.zeros(mem.N, dtype=torch.uint8, device="cuda"))           # f_0
        self.f = [mem.ring[:, self.gs.slot].cpu().numpy().copy()]
        self.a, self.r, self.t = [None], [None], [None]

    def step(self):
        k = len(self.f)
        a_row, r_row, t_row = self.mem.rows(k)
        self.gs.step_random(1, 0.5, 21, a_row, r_row, t_row, None)
        self.mem.appended(k)
        self.f.append(self.mem.ring[:, self.gs.slot].cpu().numpy().copy())
        self.a.append(a_row.cpu().numpy().copy()); self.r.append(r_row.cpu().numpy().copy()); self.t.append(t_row.cpu().numpy().copy())
        return k

    def frame(self, time, e):
        return self.f[max(time, 0)][e]


def _frame_times(k, n):
    m = min(n, 4)
    return [k - 4 + f if f < 4 else k - 4 + n + (f - m) for f in range(4 + m)]


def _memory(replay, N, C, n, prioritized, batch, lib_n_step=None):
    ring = torch.zeros((N, C + n + 3, 80, 80), dtype=torch.uint8, device="cuda")
    mem = (replay.PrioritizedMemory(ring, C, seed=7, max_batch=batch, mode="rebuild", n_step=n) if prioritized
           else replay.ReplayMemory(ring, C, seed=7, max_batch=batch, n_step=n))
    if lib_n_step is not None:
        mem.lib_n_step = lib_n_step
    return mem


def _draw(net, mem, batch, abs_err):
    """one gradient-only training step whose graph draws and gathers the minibatch (the sampling head under test)"""
    sp, mb = mem.step_sampling(batch)
    isw = mb.is_weights_f32 if mem.prioritized else None
    net.loss_backward("nature", mb.frames, mb.actions, mb.rewards, mb.terminals, isw, GAMMA, False, None, abs_err[:batch], None, sampling=sp)
    return mb


@pytest.mark.parametrize("prioritized", [False, True])
@pytest.mark.parametrize("n", [1, 2, 4, 5, 8])
def test_draw_and_gather_match_the_oracle(mods, n, prioritized):
    """from the first complete horizon (t_eff = 1: every frame clamps to f_0 at first) through 70 steps with crashes, one draw per
    step, consecutive steps replaying the captured graph with t_eff patched in: indices = CPython's random.sample over the t_eff
    population / the oracle Memory with the delayed store, frames = the recorded history, R and disc = the oracle's float64 bits"""
    game, replay, qnet, _ = mods
    N, C, B = 48, 40, 32
    mem = _memory(replay, N, C, n, prioritized, B, lib_n_step=n)
    net = qnet.QNetwork(hidden=512, max_batch=B, precision="fp16")
    abs_err = torch.zeros(B, device="cuda")
    ro_uni = ro.UniformSampler(mem.seed)
    orc = ro.Memory(N, C, mem.seed, mode="rebuild")
    roll = Rollout(game, mem)
    draws = terminal_windows = clamped = 0
    for _ in range(n + 70):
        if prioritized:                                        # the tree after the previous step's batch_update (|err| of the net)
            orc.sum_tree.tree[:] = mem.tree().cpu().numpy()
        k_now = roll.step()
        if prioritized:                                        # Memory.store of transition k - n + 1, none before it exists
            if k_now - n + 1 >= 1:
                orc.store_step(k_now - n + 1)
            np.testing.assert_array_equal(mem.tree().cpu().numpy(), orc.sum_tree.tree, err_msg=f"store at t={k_now}")
        t_eff = mem.t - n + 1
        if t_eff < 1:
            assert len(mem) == 0
            continue
        assert len(mem) == N * min(t_eff, C)
        if prioritized:
            idx_want, data_want, w_want = orc.sample(B)
            e_want, k_want = ro.data_index_to_transition(data_want, t_eff, C)
        else:
            ro_uni.pos = mem.rng_positions()[0]
            data_want = np.array(ro_uni.sample(len(mem), B))
            e_want, k_want = ro.population_to_transition(data_want, t_eff, N, C)
        mb = _draw(net, mem, B, abs_err)
        torch.cuda.synchronize()
        draws += 1
        np.testing.assert_array_equal(mb.idx.cpu().numpy(), data_want, err_msg=f"t={mem.t}")
        if prioritized:
            np.testing.assert_array_equal(mb.tree_idx.cpu().numpy(), idx_want)
            np.testing.assert_allclose(mb.is_weights.cpu().numpy(), w_want, rtol=1e-12)
        else:
            assert mem.rng_positions()[0] == ro_uni.pos
        np.testing.assert_array_equal(mb.env.cpu().numpy(), e_want)
        np.testing.assert_array_equal(mb.k.cpu().numpy(), k_want)
        frames = mb.frames.cpu().numpy()
        R, D = mb.returns.cpu().numpy(), mb.disc.cpu().numpy()
        a, r, t = mb.actions.cpu().numpy(), mb.rewards.cpu().numpy(), mb.terminals.cpu().numpy()
        assert frames.shape[1] == 4 + min(n, 4)
        for b, (e, k) in enumerate(zip(e_want, k_want)):
            times = _frame_times(int(k), n)
            clamped += times[0] < 0
            for f, tf in enumerate(times):
                np.testing.assert_array_equal(frames[b, f], roll.frame(tf, e), err_msg=f"t={mem.t} sample {b} env {e} k {k} frame {f}")
            assert (a[b], r[b], t[b]) == (roll.a[k][e], roll.r[k][e], roll.t[k][e])
            want_R, want_d = no.nstep_targets(roll.r, roll.t, int(e), int(k), n, GAMMA)
            assert R[b].tobytes() == np.float64(want_R).tobytes() and D[b].tobytes() == np.float64(want_d).tobytes(), (b, e, k)
            terminal_windows += want_d == 0.0 and not roll.t[k][e]
    assert draws >= 70 and clamped > 0
    if n > 1:
        assert terminal_windows > 0                   # some windows were cut by a terminal after their first step


def _brain_run(brains, game, model, precision, lib_n_step, steps=24, N=48):
    brain = brains.MODELS[model](2, "bird", num_envs=N, replay_memory_per_env=10, batch_size=32, observe=3, seed=6, lr=1e-4,
                                 replace_target_iter=5, precision=precision)
    brain.replayMemory.lib_n_step = lib_n_step
    gs = game.GameState(num_envs=N, seed=2, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    trace = []
    for _ in range(steps):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
        brain.setPerception(obs, a, r, t, s)
        trace.append((brain.net.loss.clone(), brain.net.grads.clone()))
    return brain, trace


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("model", ["dqnnature", "ddqn", "duelingdqn", "prioritydqn"])
def test_n1_through_the_nstep_path_equals_the_one_step_path(mods, model, precision):
    """n_step = 1 handed to the library (gather writes R = r, disc = gamma or 0; the head reads them) against n_step = 0 (the
    original path): 20 fused updates with bit-identical loss, gradients and parameters"""
    game, _, _, brains = mods
    (b1, tr1), (b0, tr0) = (_brain_run(brains, game, model, precision, 1), _brain_run(brains, game, model, precision, 0))
    assert b1.net.adam_steps == b0.net.adam_steps == 20
    for (l1, g1), (l0, g0) in zip(tr1, tr0):
        assert torch.equal(l1, l0) and torch.equal(g1, g0)
    assert torch.equal(b1.net.params, b0.net.params) and torch.equal(b1.net.adam_m, b0.net.adam_m)
    assert torch.equal(b1.replayMemory._frames, b0.replayMemory._frames)
    if model == "prioritydqn":
        assert torch.equal(b1.replayMemory.tree(), b0.replayMemory.tree())


CASES = [  # variant, dueling, loss_sum, per
    ("vanilla", False, True, False), ("nature", False, False, False), ("double", False, False, False),
    ("nature", True, False, False), ("double", True, False, False), ("nature", False, False, True), ("double", True, False, True)]


def _per_tensor(g, g_ref, dueling):
    out = {}
    for name, (o, shp) in ((k, v) for k, v in qo.layout(512, dueling).items() if k != "total"):
        sz = int(np.prod(shp))
        out[name] = float(np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) / np.linalg.norm(g_ref[o:o + sz]))
    return out


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("n,B", [(3, 32), (5, 32), (3, 256), (5, 256)])
@pytest.mark.parametrize("variant,dueling,loss_sum,per", CASES)
def test_loss_and_gradients_match_the_oracle(mods, variant, dueling, loss_sum, per, n, B, precision):
    """the n-step TD target inside the fused head against nstep_oracle.loss_and_grads on the very minibatch the
    step drew.  fp32: loss and per-tensor gradients to 2e-4.  fp16, two tiers: (A) against the oracle with the same roundings,
    loss 5e-4 and the whole gradient vector 1.5e-3 (the form smoke() states); (B) against the exact oracle, loss 4e-3 and every
    tensor 4.5e-2.  Tier A is not asserted per tensor: on a B200 some of these minibatches put conv1 / conv2's gradients 1.5e-3 ..
    1.8e-3 from the emulating oracle (others 1e-4 .. 2e-4) while the loss agreed to 2e-5 and the same cases in fp32 stayed inside
    2e-4 -- rounding-decision flips in the convolution backward (tests/test_qnet_tc_gpu.py), not the n-step target."""
    if B == 256 and (precision, variant, dueling, per) not in (("fp16", "nature", False, False), ("fp32", "double", True, True),
                                                               ("fp16", "vanilla", False, False), ("fp16", "double", True, True)):
        pytest.skip("minibatch 256 runs a representative subset (the float64 oracle is slow at that size)")
    game, replay, qnet, _ = mods
    N, C = 64, 30
    mem = _memory(replay, N, C, n, per, B)
    net = qnet.QNetwork(hidden=512, dueling=dueling, max_batch=B, precision=precision)
    p = qo.init_params(512, dueling, seed=1) * np.float32(3.0)
    tg = qo.init_params(512, dueling, seed=2) * np.float32(3.0)
    net.params.copy_(torch.from_numpy(p)); net.target.copy_(torch.from_numpy(tg))
    roll = Rollout(game, mem, seed=3)
    for _ in range(60):
        roll.step()
    abs_err = torch.zeros(B, device="cuda"); y = torch.zeros(B, device="cuda")
    sp, mb = mem.step_sampling(B)
    isw = mb.is_weights_f32 if per else None
    net.loss_backward(variant, mb.frames, mb.actions, mb.rewards, mb.terminals, isw, GAMMA, loss_sum, None, abs_err, y, sampling=sp)
    torch.cuda.synchronize()
    x = mb.frames.cpu().numpy()
    m = min(n, 4)
    R, D = mb.returns.cpu().numpy(), mb.disc.cpu().numpy()
    assert (D > 0).any()
    w = isw.cpu().numpy() if per else None
    g = net.grads.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    # fp32: the strict tier; fp16: (A) the oracle with the same roundings, (B) the exact oracle (tests/test_qnet_tc_gpu.py)
    tiers = [(None, 2e-4, 2e-4)] if precision == "fp32" else [("fp16", 5e-4, 1.5e-3), (None, 4e-3, 4.5e-2)]
    for emulate, tol_loss, tol_g in tiers:
        loss, g_ref, _, y_ref, _ = no.loss_and_grads(qnet.VARIANTS[variant], p, tg, x[:, 0:4], x[:, m:m + 4], mb.actions.cpu().numpy(),
                                                     R, D, w, loss_sum, None, 512, dueling, emulate=emulate)
        report = _per_tensor(g, g_ref, dueling)
        whole = float(np.linalg.norm(g - g_ref) / np.linalg.norm(g_ref))
        print(f"\n[{emulate}] loss {abs(net.loss.item() - loss) / abs(loss):.2e}  gradient {whole:.2e}, worst tensor {max(report.values()):.2e}")
        assert abs(net.loss.item() - loss) <= tol_loss * abs(loss), (emulate, net.loss.item(), loss)
        assert np.abs(y.cpu().numpy() - y_ref).max() <= tol_loss * np.abs(y_ref).max(), emulate
        if precision == "fp16" and emulate == "fp16":
            assert whole <= tol_g, (whole, report)
        else:
            assert all(v <= tol_g for v in report.values()), (emulate, report)


@pytest.mark.parametrize("name", ["dqn", "dqnnature", "ddqn", "duelingdqn", "prioritydqn"])
def test_every_brain_trains_with_n_step_3(mods, name):
    game, _, _, brains = mods
    N, C, n = 64, 12, 3
    brain = brains.MODELS[name](2, "bird", num_envs=N, replay_memory_per_env=C, observe=6., batch_size=32, seed=1,
                                replace_target_iter=4, n_step=n)
    assert brain.ring.shape[1] == C + n + 3
    gs = game.GameState(num_envs=N, seed=2, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    p0 = brain.net.params.clone()
    for step in range(25):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
        brain.setPerception(obs, a, r, t, s)
        assert len(brain.replayMemory) == N * max(0, min(step + 1 - n + 1, C))
    gs.check_errors()
    assert brain.net.adam_steps == 25 - 7
    assert torch.isfinite(brain.net.params).all() and not torch.equal(brain.net.params, p0)
    if name == "prioritydqn":
        cap = N * C
        tree = brain.replayMemory.tree()
        assert abs(tree[0].item() - tree[cap - 1:].sum().item()) < 1e-9
        stored = min(25 - n + 1, C)
        assert int((tree[cap - 1:] > 0).sum()) == N * stored
    brain.fuse_sampling = False
    with pytest.raises(ValueError):
        brain._trainQNetwork()


def test_nstep_arguments_are_checked(mods):
    game, replay, qnet, brains = mods
    ring = torch.zeros((4, 20, 80, 80), dtype=torch.uint8, device="cuda")
    for bad in (0, 17):
        with pytest.raises(ValueError):
            replay.ReplayMemory(ring, 10, n_step=bad)
    with pytest.raises(ValueError):
        replay.ReplayMemory(ring, 15, n_step=3)                   # 15 + 3 + 3 > 20 frames
    mem = replay.ReplayMemory(ring, 14, n_step=3)
    assert mem.C == 14 and replay.ReplayMemory(ring, n_step=3).C == 14
    with pytest.raises(ValueError):
        mem.sample(4)                                            # n-step draws ride inside the step only
    # the library's own checks: ring too short for the horizon, n out of range, missing R / disc
    mem.t = 12
    net = qnet.QNetwork(max_batch=8, precision="fp32")
    from dqnflappybird_b200 import _lib
    for field, value in (("n_step", 7), ("n_step", 17), ("ret_out_dev", None)):
        sp, mb = mem.step_sampling(8)
        setattr(sp, field, value)
        with pytest.raises(_lib.FlappyError):
            net.loss_backward("nature", mb.frames, mb.actions, mb.rewards, mb.terminals, None, GAMMA, sampling=sp)
