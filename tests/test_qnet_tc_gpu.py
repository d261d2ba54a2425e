"""GPU parity of the tensor-core Q-network path (csrc/fb_qnet_tc.cu: TMA + tcgen05, bf16 operands, fp32 accumulate).

Oracle: oracle/qnet_oracle.py (float64 restatement of the TF-1.12 graph, PARITY UNPINNED -- see its header).
Two comparisons, two tolerances (operands and stored activations / gradients are bf16: 8 significant bits, unit
round-off 2^-9 = 0.2 %; sums, head, TD loss and Adam are fp32):

  (A) implementation -- against the oracle run with emulate_bf16=True (the same float64 graph with the bf16
      roundings placed where this path has them).  What is left is fp32-vs-float64 summation and the rare
      ReLU / max-pool decision that flips on it:
        Q-values   |dq| <= 3e-3 * max|q_ref|        loss  relative 3e-3       y  |dy| <= 3e-3 * max|y_ref|
        gradients  per tensor ||g - g_ref||_2 <= 1.5e-2 ||g_ref||_2
  (B) precision of the format -- against the exact float64 oracle:
        Q-values   |dq| <= 2e-2 * max|q_ref|        loss  relative 3e-2
        gradients  per tensor ||g - g_ref||_2 <= 1.2e-1 ||g_ref||_2 at minibatch 32 (measured 5-7 %: rounded
                   activations flip ReLU masks of individual samples; the error averages down with the batch,
                   measured < 4 % at minibatch 256)
  raw GEMM self-test: exact bf16 inputs, fp32 accumulation: |d - ref| <= 9e-3 * sqrt(K)
The strict-fp32 path (tests/test_qnet_gpu.py, 2e-4) remains the anchor.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import qnet_oracle as qo  # noqa: E402


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dqnflappybird_b200 import _lib, game, qnet
    return _lib, game, qnet


def _gemm(_lib, mode, bn, a, b, M, N, K, strides=None):
    d = torch.full((M, N), float("nan"), dtype=torch.float32, device="cuda")
    st = (C.c_uint32 * 6)(*strides) if strides is not None else None
    _lib.check(_lib.lib().fb_debug_tc_gemm(mode, bn, M, N, K, a.data_ptr(), b.data_ptr(), d.data_ptr(), st,
                                           torch.cuda.current_stream().cuda_stream), "fb_debug_tc_gemm")
    torch.cuda.synchronize()
    return d


@pytest.mark.parametrize("bn,M,N,K", [(32, 300, 32, 256), (64, 128, 64, 576), (128, 256, 512, 1600), (64, 77, 128, 64)])
def test_raw_gemm_k_major(mods, bn, M, N, K):
    """D = A Bt^T through the kernel the forward and data-gradient layers use (both operands K-major, SWIZZLE_128B)"""
    _lib, _, _ = mods
    g = torch.Generator(device="cuda").manual_seed(bn + M)
    a = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    b = torch.randn((N, K), device="cuda", generator=g).to(torch.bfloat16)
    d = _gemm(_lib, 0, bn, a, b, M, N, K)
    ref = a.double() @ b.double().T
    err = (d.double() - ref).abs().max().item()
    assert err <= 1e-3 * np.sqrt(K) * 9, (err, bn, M, N, K)


@pytest.mark.parametrize("bn,M,N,K", [(64, 128, 64, 64), (64, 256, 64, 1000), (32, 256, 32, 1536), (128, 1600, 512, 256), (64, 576, 64, 333)])
def test_raw_gemm_mn_major(mods, bn, M, N, K):
    """D = A^T B with the contraction over ROWS of both row-major operands (weight gradients): MN-major descriptors"""
    _lib, _, _ = mods
    g = torch.Generator(device="cuda").manual_seed(bn + K)
    a = torch.randn((K, M), device="cuda", generator=g).to(torch.bfloat16)
    b = torch.randn((K, N), device="cuda", generator=g).to(torch.bfloat16)
    d = _gemm(_lib, 1, bn, a, b, M, N, K)
    ref = a.double().T @ b.double()
    err = (d.double() - ref).abs().max().item()
    assert err <= 1e-3 * np.sqrt(K) * 9, (err, bn, M, N, K)


@pytest.mark.parametrize("shift", [0, 1, 7, 8, 21, 22, 100, 128])
def test_slab_descriptor_shift(mods, shift):
    """tcgen05 swizzles on absolute shared-memory address bits: a K-major SWIZZLE_128B descriptor started `shift` rows
    into a TMA-written slab reads rows shift..shift+127 (base_offset 0) -- the property the slab convolutions rely on"""
    _lib, _, _ = mods
    g = torch.Generator(device="cuda").manual_seed(shift)
    a = torch.randn((256, 64), device="cuda", generator=g).to(torch.bfloat16)
    b = torch.randn((64, 64), device="cuda", generator=g).to(torch.bfloat16)
    d = torch.full((128, 64), float("nan"), device="cuda")
    _lib.check(_lib.lib().fb_debug_tc_slab(shift, 0, a.data_ptr(), b.data_ptr(), d.data_ptr(), torch.cuda.current_stream().cuda_stream), "slab")
    torch.cuda.synchronize()
    ref = a[shift:shift + 128].double() @ b.double().T
    assert (d.double() - ref).abs().max().item() <= 1e-4


def _env_frames(game, B, seed):
    gs = game.GameState(num_envs=B, seed=seed, history=5)
    gs.step_random(40 + seed % 7, 0.3, 99 + seed)
    gs.step_random(5, 0.3, 99 + seed)
    torch.cuda.synchronize()
    order = [(gs.slot - 4 + k) % 5 for k in range(5)]
    return gs.ring[:, order].contiguous()


def _set_params(net, flat, target=None):
    net.params.copy_(torch.from_numpy(flat))
    net.target.copy_(torch.from_numpy(target if target is not None else flat))


@pytest.mark.parametrize("dueling", [False, True])
def test_forward_matches_oracle_bf16(mods, dueling):
    _lib, game, qnet = mods
    B = 37
    frames = _env_frames(game, B, 3)
    net = qnet.QNetwork(hidden=512, dueling=dueling, max_batch=16, precision="bf16")     # 37 > 16: chunking
    flat = qo.init_params(512, dueling, seed=5) * np.float32(4.0)
    _set_params(net, flat)
    q = net.forward(qnet.FrameBatch.from_stack(frames, 0)).cpu().numpy()
    q2 = net.forward(qnet.FrameBatch.from_stack(frames, 1)).cpu().numpy()
    x = frames.cpu().numpy()
    ref = qo.forward(torch.tensor(flat.astype(np.float64)), x[:, 0:4], 512, dueling).numpy()
    ref2 = qo.forward(torch.tensor(flat.astype(np.float64)), x[:, 1:5], 512, dueling).numpy()
    emu = qo.forward(torch.tensor(flat.astype(np.float64)), x[:, 0:4], 512, dueling, emulate_bf16=True).numpy()
    assert np.abs(q - emu).max() <= 3e-3 * np.abs(emu).max(), np.abs(q - emu).max() / np.abs(emu).max()          # (A)
    assert np.abs(q - ref).max() <= 2e-2 * np.abs(ref).max(), np.abs(q - ref).max() / np.abs(ref).max()          # (B)
    assert np.abs(q2 - ref2).max() <= 2e-2 * np.abs(ref2).max()
    noise = (torch.rand((9, 5, 80, 80), device="cuda") < 0.3).to(torch.uint8) * 255
    qn = net.forward(qnet.FrameBatch.from_stack(noise.contiguous(), 0)).cpu().numpy()
    refn = qo.forward(torch.tensor(flat.astype(np.float64)), noise.cpu().numpy()[:, 0:4], 512, dueling).numpy()
    assert np.abs(qn - refn).max() <= 2e-2 * np.abs(refn).max()
    # and the strict path agrees with it to the same bound
    net32 = qnet.QNetwork(hidden=512, dueling=dueling, max_batch=64, precision="fp32")
    _set_params(net32, flat)
    q32 = net32.forward(qnet.FrameBatch.from_stack(frames, 0)).cpu().numpy()
    assert np.abs(q - q32).max() <= 2e-2 * np.abs(q32).max()


def test_conv1_paths_are_bit_identical(mods):
    """conv1 of the training forward on s has two data paths: built from the u8 frames, with X2 (which then only the conv1 weight
    gradient reads) packed beside it -- when the step draws its own minibatch, up to minibatch 512 -- or from X2 materialised
    first and read by TMA -- on a minibatch the caller passes.  The same arithmetic on different data paths: a step that draws its
    minibatch and a twin net's step on that same minibatch, passed by the caller, give identical gradients and loss, bit for bit
    (bf16, an odd minibatch)"""
    _lib, game, qnet = mods
    from dqnflappybird_b200 import replay
    B = 70
    mem = _memory(game, replay, 48, 20, B, 30)
    nets = [qnet.QNetwork(max_batch=128, seed=2, precision="bf16") for _ in range(2)]
    for n in nets:
        n.params.mul_(4.0); n.target.mul_(4.0)
    for rep in range(3):                            # eager, eager, graph replay
        sp, mb = mem.step_sampling(B)
        nets[0].loss_backward("double", mb.frames, mb.actions, mb.rewards, mb.terminals, sampling=sp)     # conv1 from the u8 frames
        nets[1].loss_backward("double", mb.frames, mb.actions, mb.rewards, mb.terminals)                  # conv1 from X2
        assert torch.isfinite(nets[0].grads).all()
        assert torch.equal(nets[0].grads, nets[1].grads) and nets[0].loss.item() == nets[1].loss.item(), rep
    assert nets[0].grads.abs().max().item() > 0


def test_forward_from_ring_view_bf16(mods):
    _lib, game, qnet = mods
    N = 300
    gs = game.GameState(num_envs=N, seed=1, history=7)
    gs.step_random(23, 0.4, 5)
    net = qnet.QNetwork(max_batch=256, precision="bf16")
    net.params.mul_(4.0)
    q = net.forward(qnet.FrameBatch.from_ring(gs.ring, gs.slot)).cpu().numpy()
    st = gs.stacked_state().permute(0, 3, 1, 2).contiguous().cpu().numpy()
    ref = qo.forward(torch.tensor(net.params.cpu().numpy().astype(np.float64)), st).numpy()
    assert np.abs(q - ref).max() <= 2e-2 * np.abs(ref).max()


@pytest.mark.parametrize("N,chunk", [(2500, 2048), (4500, 4096)])
def test_forward_large_chunks_and_single_sample_bf16(mods, N, chunk):
    """acting-sized batches: 2,500 envs through workspaces of 2,048 / 4,500 through 4,096 (fc1 forward then runs 2 / 1
    K-splits instead of 5, the conv1 slab is built from the u8 ring in the kernel, chunks alternate between two streams)
    and a batch of one"""
    _lib, game, qnet = mods
    gs = game.GameState(num_envs=N, seed=8, history=6)
    gs.step_random(31, 0.45, 11)
    fb = qnet.FrameBatch.from_ring(gs.ring, gs.slot)
    net = qnet.QNetwork(max_batch=chunk, precision="bf16")
    net.params.mul_(4.0)
    q = net.forward(fb)
    small = qnet.QNetwork(max_batch=128, precision="bf16")           # same weights, 20 chunks of 128 (5 K-splits)
    small.params.copy_(net.params)
    qs = small.forward(fb)
    scale = q.abs().max().item()
    assert (q - qs).abs().max().item() <= 2e-5 * scale               # only the fp32 summation order of fc1 differs
    st = gs.stacked_state().permute(0, 3, 1, 2).contiguous().cpu().numpy()
    pick = np.r_[0:24, chunk - 8:chunk + 8, N - 24:N]                # both chunks and their seam
    ref = qo.forward(torch.tensor(net.params.cpu().numpy().astype(np.float64)), st[pick]).numpy()
    assert np.abs(q.cpu().numpy()[pick] - ref).max() <= 2e-2 * np.abs(ref).max()
    one = game.GameState(num_envs=1, seed=8, history=6)
    one.step_random(31, 0.45, 11)
    q1 = net.forward(qnet.FrameBatch.from_ring(one.ring, one.slot))
    assert (q1[0] - q[0]).abs().max().item() <= 2e-5 * scale         # env 0 of the batch = the same env alone


CASES = [("vanilla", False, True, False, 32), ("nature", False, False, False, 32), ("double", False, False, False, 32),
         ("nature", True, False, False, 32), ("nature", False, False, True, 32), ("double", True, False, True, 32),
         ("nature", False, False, False, 256), ("nature", False, False, False, 100)]


@pytest.mark.parametrize("variant,dueling,loss_sum,per,B", CASES)
def test_loss_and_gradients_match_oracle_bf16(mods, variant, dueling, loss_sum, per, B):
    _lib, game, qnet = mods
    frames = _env_frames(game, B, 11)
    net = qnet.QNetwork(hidden=512, dueling=dueling, max_batch=256, precision="bf16")
    p = qo.init_params(512, dueling, seed=1) * np.float32(3.0)
    t = qo.init_params(512, dueling, seed=2) * np.float32(3.0)
    _set_params(net, p, t)
    rng = np.random.default_rng(0)
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B, p=[0.8, 0.1, 0.1])
    term = (r == -3.0).astype(np.uint8)
    isw = rng.random(B).astype(np.float32) if per else None
    abs_err = torch.zeros(B, device="cuda"); y = torch.zeros(B, device="cuda")
    net.loss_backward(variant, frames, torch.from_numpy(a).cuda(), torch.from_numpy(r).cuda(), torch.from_numpy(term).cuda(),
                      torch.from_numpy(isw).cuda() if per else None, 0.99, loss_sum, None, abs_err, y)
    x = frames.cpu().numpy()
    g = net.grads.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    L = qo.layout(512, dueling)
    for emulate, tol_loss, tol_y, tol_g in ((True, 3e-3, 3e-3, 1.5e-2), (False, 3e-2, 2e-2, 1.2e-1)):
        loss, g_ref, ae_ref, y_ref, _ = qo.loss_and_grads(qnet.VARIANTS[variant], p, t, x[:, 0:4], x[:, 1:5], a, r, term, isw, 0.99,
                                                          loss_sum, None, 512, dueling, emulate_bf16=emulate)
        assert abs(net.loss.item() - loss) <= tol_loss * abs(loss), (emulate, net.loss.item(), loss)
        assert np.abs(y.cpu().numpy() - y_ref).max() <= tol_y * np.abs(y_ref).max(), emulate
        report = {}
        for name, v in L.items():
            if name == "total":
                continue
            o, shp = v
            sz = int(np.prod(shp))
            num = np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]); den = np.linalg.norm(g_ref[o:o + sz])
            assert den > 0, name
            report[name] = float(num / den)
        assert all(v <= tol_g for v in report.values()), (emulate, report)


def test_training_steps_track_the_strict_path(mods):
    """ten Nature-DQN updates on the same minibatches: bf16 and fp32 paths stay together (Adam lr 1e-6)"""
    _lib, game, qnet = mods
    B = 64
    frames = _env_frames(game, B, 7)
    nets = [qnet.QNetwork(max_batch=B, seed=3, precision=pr) for pr in ("bf16", "fp32")]
    for n in nets:
        n.params.mul_(3.0); n.target.mul_(3.0)
    rng = np.random.default_rng(4)
    p0 = nets[0].params.clone()
    for step in range(10):
        a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
        r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
        term = (r == -3.0).to(torch.uint8)
        for n in nets:
            n.loss_backward("nature", frames, a, r, term)
            n.adam_step()
        if step == 4:
            for n in nets:
                n.sync_target()
    u0, u1 = (nets[0].params - p0).double(), (nets[1].params - p0).double()     # Adam normalises: compare directions
    cos = (u0 @ u1 / (u0.norm() * u1.norm())).item()
    assert u1.abs().max().item() > 5e-6 and cos > 0.95, cos
    assert abs(nets[0].loss.item() - nets[1].loss.item()) <= 3e-2 * abs(nets[1].loss.item())


@pytest.mark.parametrize("precision,variant,dueling", [("bf16", "nature", False), ("bf16", "double", True), ("bf16", "vanilla", False),
                                                       ("fp32", "nature", False)])
def test_train_step_is_loss_backward_plus_adam(mods, precision, variant, dueling):
    """fb_qnet_step with Adam (inside the step's last kernel, alpha from beta powers in device memory, one CUDA graph) is
    bit-identical to the gradient-only fb_qnet_step + fb_qnet_adam, over graph capture / replay and when the two forms are mixed"""
    _lib, game, qnet = mods
    B = 64
    frames = _env_frames(game, B, 21)
    rng = np.random.default_rng(5)
    a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
    r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
    term = (r == -3.0).to(torch.uint8)
    fused, split = [qnet.QNetwork(max_batch=B, seed=3, dueling=dueling, precision=precision, lr=1e-3) for _ in range(2)]
    for n in (fused, split):
        n.params.mul_(4.0); n.target.mul_(4.0)
    plan = ["f", "f", "f", "f", "s", "f", "f", "s", "s", "f"]          # what `fused` does; `split` always takes the two calls
    for k, how in enumerate(plan):
        if how == "f":
            lf = fused.train_step(variant, frames, a, r, term, loss_sum=(variant == "vanilla")).clone()
        else:
            lf = fused.loss_backward(variant, frames, a, r, term, loss_sum=(variant == "vanilla")).clone(); fused.adam_step()
        ls = split.loss_backward(variant, frames, a, r, term, loss_sum=(variant == "vanilla")).clone(); split.adam_step()
        assert torch.equal(lf, ls), (k, how)
        assert torch.equal(fused.grads, split.grads), (k, how)
        for name in ("params", "adam_m", "adam_v"):
            assert torch.equal(getattr(fused, name), getattr(split, name)), (k, how, name)
        assert fused.beta1_power == split.beta1_power and fused.beta2_power == split.beta2_power and fused.adam_steps == k + 1
        if k == 5:
            fused.sync_target(); split.sync_target()
    # the updated parameters are what the next forward uses (the bf16 operand copies were refreshed by the fused Adam)
    qf = fused.forward(qnet.FrameBatch.from_stack(frames, 0)); qs = split.forward(qnet.FrameBatch.from_stack(frames, 0))
    assert torch.equal(qf, qs)
    # resume: the powers come back from a checkpoint and re-seed the device copy
    sd = split.state_dict()
    fresh = qnet.QNetwork(max_batch=B, seed=9, dueling=dueling, precision=precision, lr=1e-3)
    fresh.load_state_dict(sd)
    fresh.train_step(variant, frames, a, r, term, loss_sum=(variant == "vanilla"))
    split.loss_backward(variant, frames, a, r, term, loss_sum=(variant == "vanilla")); split.adam_step()
    assert torch.equal(fresh.params, split.params)


def test_pack_then_forward_never_reads_stale_operands(mods):
    """The pack kernel writes the bf16 operand copies that its stream successor (a conv kernel launched with programmatic
    dependent launch) TMA-loads in its prologue, before its own griddepcontrol.wait: the pack kernel must therefore not
    release its dependents early.  Poison the copies (NaN bit patterns, NOT marked stale), mark them stale, run
    pack + forward back to back many times: a conv kernel that fetched weights before the pack finished shows as NaN /
    different Q-values.  Both operand slots: the online net (acting) and the target net (first update after a sync)."""
    _lib, game, qnet = mods
    L = _lib.lib()
    B = 48
    frames = _env_frames(game, B, 13)
    net = qnet.QNetwork(max_batch=64, seed=4, precision="bf16")
    net.params.mul_(4.0); net.target.mul_(3.0)
    fb = qnet.FrameBatch.from_stack(frames, 0)
    st = torch.cuda.current_stream().cuda_stream
    for use_target in (False, True):
        good = net.forward(fb, target=use_target).clone()
        assert torch.isfinite(good).all()
        for rep in range(40):
            for slot in (0, 1):
                _lib.check(L.fb_debug_poison_packed(net._h, slot, st), "fb_debug_poison_packed")
            _lib.check(L.fb_qnet_invalidate(net._h), "fb_qnet_invalidate")
            q = net.forward(fb, target=use_target)
            assert torch.equal(q, good), (use_target, rep)
    # the training step: Q(s') on the second stream right after the target operands were re-packed
    rng = np.random.default_rng(6)
    a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
    r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
    term = (r == -3.0).to(torch.uint8)
    ref_loss = net.loss_backward("nature", frames, a, r, term).clone()
    ref_grads = net.grads.clone()
    for rep in range(20):
        for slot in (0, 1):
            _lib.check(L.fb_debug_poison_packed(net._h, slot, st), "fb_debug_poison_packed")
        _lib.check(L.fb_qnet_invalidate(net._h), "fb_qnet_invalidate")
        loss = net.loss_backward("nature", frames, a, r, term)
        assert torch.equal(loss, ref_loss) and torch.equal(net.grads, ref_grads), rep


@pytest.mark.parametrize("precision,tol_g", [("fp32", 2e-4), ("bf16", 1.5e-2)])
def test_per_broadcast_loss_is_what_the_reference_graph_computes(mods, precision, tol_g):
    """BrainPrioritizedReplyDQN.py:243-251: ISWeights is a [B,1] placeholder, tf.square(q_target - q_eval) a [B] vector; their
    product broadcasts to [B,B] and reduce_mean gives mean(w) * mean(err^2).  fb_qnet_set_per_broadcast(1) (what
    reference_quirks=True selects) reproduces that; the default is the intended mean(w_i err_i^2).  Both against the oracle."""
    _lib, game, qnet = mods
    B = 32
    frames = _env_frames(game, B, 17)
    net = qnet.QNetwork(max_batch=B, precision=precision)
    p = qo.init_params(512, False, seed=1) * np.float32(3.0)
    t = qo.init_params(512, False, seed=2) * np.float32(3.0)
    _set_params(net, p, t)
    rng = np.random.default_rng(2)
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B, p=[0.8, 0.1, 0.1])
    term = (r == -3.0).astype(np.uint8)
    isw = (0.05 + rng.random(B)).astype(np.float32)
    x = frames.cpu().numpy()
    emulate = precision == "bf16"
    got = {}
    for on in (False, True):
        net.set_per_broadcast(on)
        abs_err = torch.zeros(B, device="cuda")
        net.loss_backward("nature", frames, torch.from_numpy(a).cuda(), torch.from_numpy(r).cuda(), torch.from_numpy(term).cuda(),
                          torch.from_numpy(isw).cuda(), 0.99, False, None, abs_err, None)
        loss, g_ref, ae_ref, _, _ = qo.loss_and_grads(1, p, t, x[:, 0:4], x[:, 1:5], a, r, term, isw, emulate_bf16=emulate, isw_broadcast=on)
        g = net.grads.cpu().numpy().astype(np.float64)
        assert abs(net.loss.item() - loss) <= (3e-3 if emulate else 1e-4) * abs(loss), (on, net.loss.item(), loss)
        assert np.linalg.norm(g - g_ref) <= tol_g * np.linalg.norm(g_ref), (on, np.linalg.norm(g - g_ref) / np.linalg.norm(g_ref))
        assert np.abs(abs_err.cpu().numpy() - ae_ref).max() <= (2e-2 if emulate else 1e-4) * np.abs(ae_ref).max()      # |delta| is not weighted
        got[on] = (net.loss.item(), g)
    # the two forms really differ on this minibatch (so the switch is observable), and relate as the algebra says
    assert abs(got[True][0] - got[False][0]) > 1e-3 * abs(got[False][0])


def test_loss_and_gradients_other_hidden_width_bf16(mods):
    """hidden = 256 (north_star's "fc256" as a configuration): the head runs as the two-kernel form instead of the fused
    fc1_head_train_kernel<16> (hidden = 512); same tolerances against the oracle with the bf16 roundings emulated"""
    _lib, game, qnet = mods
    B, H = 48, 256
    frames = _env_frames(game, B, 19)
    net = qnet.QNetwork(hidden=H, max_batch=64, precision="bf16")
    p = qo.init_params(H, False, seed=1) * np.float32(3.0)
    t = qo.init_params(H, False, seed=2) * np.float32(3.0)
    _set_params(net, p, t)
    rng = np.random.default_rng(8)
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B, p=[0.8, 0.1, 0.1])
    term = (r == -3.0).astype(np.uint8)
    net.loss_backward("nature", frames, torch.from_numpy(a).cuda(), torch.from_numpy(r).cuda(), torch.from_numpy(term).cuda())
    x = frames.cpu().numpy()
    loss, g_ref, *_ = qo.loss_and_grads(1, p, t, x[:, 0:4], x[:, 1:5], a, r, term, hidden=H, emulate_bf16=True)
    g = net.grads.cpu().numpy().astype(np.float64)
    assert abs(net.loss.item() - loss) <= 3e-3 * abs(loss)
    Lo = qo.layout(H, False)
    for name, v in Lo.items():
        if name == "total":
            continue
        o, shp = v
        sz = int(np.prod(shp))
        assert np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) <= 1.5e-2 * np.linalg.norm(g_ref[o:o + sz]), name


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("B,variant,dueling", [(33, "nature", False), (70, "double", True), (300, "nature", False), (700, "vanilla", False)])
def test_fused_backward_is_bit_identical(mods, B, variant, dueling, precision):
    """tc_bwd23_kernel (conv3 data gradient + ReLU mask + conv2 data gradient + un-pool in one kernel, dZ2 handed from the
    first GEMM's epilogue to the second through a hand-swizzled shared-memory slab) against the three separate kernels:
    identical gradients, bit for bit, in both 16-bit operand formats (fp16: gradient tensors scaled by a power of two).  Odd
    minibatch (last tile = one sample), one tile per CTA, and several tiles per CTA (the slab ring and both accumulators are
    reused: 350 tiles on 148 CTAs)."""
    _lib, game, qnet = mods
    frames = _env_frames(game, B, 23)
    nets = [qnet.QNetwork(max_batch=B, seed=2, dueling=dueling, precision=precision) for _ in range(2)]
    for n in nets:
        n.params.mul_(4.0); n.target.mul_(4.0)
    _lib.check(_lib.lib().fb_debug_tc_separate_kernels(nets[1]._h, 1), "fb_debug_tc_separate_kernels")
    # (the hook also turns off the forward twin, tc_fwd23_kernel: conv2 + conv3 as one kernel)
    q = [n.forward(qnet.FrameBatch.from_stack(frames, 1)) for n in nets]
    assert torch.isfinite(q[0]).all() and torch.equal(q[0], q[1])
    rng = np.random.default_rng(3)
    a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
    r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
    term = (r == -3.0).to(torch.uint8)
    for rep in range(3):                       # eager, eager, graph replay
        for n in nets:
            n.loss_backward(variant, frames, a, r, term, loss_sum=(variant == "vanilla"))
        assert torch.isfinite(nets[0].grads).all()
        assert torch.equal(nets[0].grads, nets[1].grads) and nets[0].loss.item() == nets[1].loss.item(), rep
    assert nets[0].grads.abs().max().item() > 0


FP16_CASES = [("vanilla", False, True, False, 32), ("nature", False, False, False, 32), ("double", True, False, True, 32),
              ("nature", False, False, False, 256), ("nature", True, False, False, 100)]


@pytest.mark.parametrize("variant,dueling,loss_sum,per,B", FP16_CASES)
def test_loss_and_gradients_match_oracle_fp16(mods, variant, dueling, loss_sum, per, B):
    """precision="fp16": the same tcgen05 kernels with IEEE fp16 operands -- an 11-bit significand, exactly TF32's -- and the
    gradient tensors scaled by a power of two (removed where weight / bias gradients are finalised).  Two tiers as for bf16:
      (A) against the oracle with the same roundings emulated (emulate="fp16", gradient scale included):
            Q 5e-4 of max|q|, loss 5e-4, gradients per tensor 1.5e-3 (measured 1e-4 .. 4e-4)
      (B) against the exact float64 oracle: Q 3e-3, loss 4e-3, gradients per tensor 4.5e-2 (measured 1-3 %: the error of a
          per-tensor gradient is dominated by the rare ReLU / max-pool decisions that flip under rounding, ~ sqrt(unit
          round-off); the oracle's emulate="tf32" gives the same figures, so a kind::tf32 path would not do better)."""
    _lib, game, qnet = mods
    frames = _env_frames(game, B, 11)
    net = qnet.QNetwork(hidden=512, dueling=dueling, max_batch=256, precision="fp16")
    p = qo.init_params(512, dueling, seed=1) * np.float32(3.0)
    t = qo.init_params(512, dueling, seed=2) * np.float32(3.0)
    _set_params(net, p, t)
    rng = np.random.default_rng(0)
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B, p=[0.8, 0.1, 0.1])
    term = (r == -3.0).astype(np.uint8)
    isw = rng.random(B).astype(np.float32) if per else None
    abs_err = torch.zeros(B, device="cuda"); y = torch.zeros(B, device="cuda")
    for rep in range(3):                                                  # eager, eager, graph replay
        net.loss_backward(variant, frames, torch.from_numpy(a).cuda(), torch.from_numpy(r).cuda(), torch.from_numpy(term).cuda(),
                          torch.from_numpy(isw).cuda() if per else None, 0.99, loss_sum, None, abs_err, y)
    x = frames.cpu().numpy()
    g = net.grads.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    L = qo.layout(512, dueling)
    worst = {}
    for emulate, tol_loss, tol_y, tol_g in (("fp16", 5e-4, 5e-4, 1.5e-3), (None, 4e-3, 3e-3, 4.5e-2)):
        loss, g_ref, ae_ref, y_ref, _ = qo.loss_and_grads(qnet.VARIANTS[variant], p, t, x[:, 0:4], x[:, 1:5], a, r, term, isw, 0.99,
                                                          loss_sum, None, 512, dueling, emulate=emulate)
        assert abs(net.loss.item() - loss) <= tol_loss * abs(loss), (emulate, net.loss.item(), loss)
        assert np.abs(y.cpu().numpy() - y_ref).max() <= tol_y * np.abs(y_ref).max(), emulate
        report = {}
        for name, v in L.items():
            if name == "total":
                continue
            o, shp = v
            sz = int(np.prod(shp))
            report[name] = float(np.linalg.norm(g[o:o + sz] - g_ref[o:o + sz]) / np.linalg.norm(g_ref[o:o + sz]))
        worst[emulate] = max(report.values())
        assert all(v <= tol_g for v in report.values()), (emulate, report)
    print("fp16 worst per-tensor gradient error: emulated %.2e, exact %.2e" % (worst["fp16"], worst[None]))


def test_fp16_forward_and_training_step(mods):
    """fp16 operands: Q-values against the exact oracle to 3e-3 (bf16: 2e-2), acting from the ring, and ten training steps that
    stay with the strict fp32 path (direction of the Adam update, loss)"""
    _lib, game, qnet = mods
    B = 64
    frames = _env_frames(game, B, 7)
    flat = qo.init_params(512, False, seed=5) * np.float32(4.0)
    net = qnet.QNetwork(max_batch=16, precision="fp16")
    _set_params(net, flat)
    x = frames.cpu().numpy()
    q = net.forward(qnet.FrameBatch.from_stack(frames, 0)).cpu().numpy()
    ref = qo.forward(torch.tensor(flat.astype(np.float64)), x[:, 0:4]).numpy()
    emu = qo.forward(torch.tensor(flat.astype(np.float64)), x[:, 0:4], emulate="fp16").numpy()
    assert np.abs(q - emu).max() <= 5e-4 * np.abs(emu).max(), np.abs(q - emu).max() / np.abs(emu).max()
    assert np.abs(q - ref).max() <= 3e-3 * np.abs(ref).max(), np.abs(q - ref).max() / np.abs(ref).max()
    nets = [qnet.QNetwork(max_batch=B, seed=3, precision=pr) for pr in ("fp16", "fp32")]
    for n in nets:
        n.params.mul_(3.0); n.target.mul_(3.0)
    rng = np.random.default_rng(4)
    p0 = nets[0].params.clone()
    for step in range(10):
        a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
        r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
        term = (r == -3.0).to(torch.uint8)
        nets[0].train_step("nature", frames, a, r, term)                  # one graph launch, Adam inside
        nets[1].loss_backward("nature", frames, a, r, term); nets[1].adam_step()
        if step == 4:
            for n in nets:
                n.sync_target()
    u0, u1 = (nets[0].params - p0).double(), (nets[1].params - p0).double()
    cos = (u0 @ u1 / (u0.norm() * u1.norm())).item()
    assert u1.abs().max().item() > 5e-6 and cos > 0.995, cos
    assert abs(nets[0].loss.item() - nets[1].loss.item()) <= 4e-3 * abs(nets[1].loss.item())


def _memory(game, replay, N, C, B, steps, prioritized=False):
    """a replay memory filled by `steps` random-action env steps: the same arguments give the same contents and the same draws"""
    ring = torch.zeros((N, C + 4, 80, 80), dtype=torch.uint8, device="cuda")
    mem = replay.PrioritizedMemory(ring, C, seed=7, max_batch=B) if prioritized else replay.ReplayMemory(ring, C, seed=7, max_batch=B)
    gs = game.GameState(num_envs=N, seed=3, history=mem.L, ring=mem.ring)
    gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    for k in range(1, steps + 1):
        a, r, t = mem.rows(k)
        gs.step_random(1, 0.5, 21, a, r, t, None)
        mem.appended(k)
    return mem


# one argument of the training step changed from BASE at a time: a captured graph that ignored it would be replayed for it
BASE = dict(variant="nature", gamma=0.99, loss_sum=False, global_batch=None, outputs=True, grad_scale=1.0)
CHANGES = [dict(gamma=0.9), dict(loss_sum=True), dict(global_batch=64), dict(variant="double"), dict(outputs=False),
           dict(grad_scale=0.5)]


@pytest.mark.parametrize("sampled", [False, True])
def test_graph_replay_honours_every_argument(mods, sampled):
    """fp16, graphs on: every configuration is called three times (eager, capture, replay), then once more each after all were
    captured (replay), and after every call the net is bit-identical to a twin that never uses graphs -- the captured step is
    keyed on all of its arguments, so a changed argument never replays a graph captured for another value"""
    _lib, game, qnet = mods
    from dqnflappybird_b200 import replay
    B = 32
    graph, eager = nets = [qnet.QNetwork(max_batch=B, seed=3, precision="fp16", lr=1e-4) for _ in range(2)]
    _lib.check(_lib.lib().fb_qnet_use_graphs(eager._h, 0), "fb_qnet_use_graphs")
    for n in nets:
        n.params.mul_(3.0); n.target.mul_(3.0)
    if sampled:
        mems = [_memory(game, replay, 48, 20, B, 30) for _ in nets]
    else:
        frames = _env_frames(game, B, 21)
        rng = np.random.default_rng(5)
        a = torch.from_numpy(rng.integers(0, 2, B).astype(np.uint8)).cuda()
        r = torch.from_numpy(rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B)).cuda()
        term = (r == -3.0).to(torch.uint8)
    outs = [(torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")) for _ in nets]
    p0 = graph.params.clone()
    bits = lambda x: x.view(torch.int32)                               # bitwise, NaN included
    configs = [BASE] + [{**BASE, **c} for c in CHANGES]
    calls = [cfg for cfg in configs for _ in range(3)] + configs
    for k, cfg in enumerate(calls):
        for i, n in enumerate(nets):
            sp = None
            if sampled:
                sp, mb = mems[i].step_sampling(B)
                frames, a, r, term = mb.frames, mb.actions, mb.rewards, mb.terminals
            abs_err, y = outs[i] if cfg["outputs"] else (None, None)
            n.train_step(cfg["variant"], frames, a, r, term, None, cfg["gamma"], cfg["loss_sum"], cfg["global_batch"], abs_err, y,
                         cfg["grad_scale"], sampling=sp)
        for name in ("loss", "grads", "params", "adam_m", "adam_v"):
            assert torch.equal(bits(getattr(graph, name)), bits(getattr(eager, name))), (k, cfg, name)
        # (without outputs the buffers keep the last call's values: a replay that still wrote them would show here)
        assert torch.equal(bits(outs[0][0]), bits(outs[1][0])) and torch.equal(bits(outs[0][1]), bits(outs[1][1])), (k, cfg)
        if sampled:
            assert torch.equal(mems[0]._idx[:B], mems[1]._idx[:B]), (k, cfg)
    assert graph.adam_steps == len(calls) and torch.isfinite(graph.params).all() and not torch.equal(graph.params, p0)


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_step_rejects_bad_arguments(mods, precision):
    """fb_qnet_step validates its descriptor once, for both precisions: FB_ERR_INVALID for a missing pointer, a batch outside
    1..max_batch, a bad variant or a missing target, half of the Adam slots, prioritized replay without abs_err_out_dev, and
    caller-minibatch fields set together with `sampling`"""
    _lib, game, qnet = mods
    from dqnflappybird_b200 import replay
    L = _lib.lib()
    B = 8
    net = qnet.QNetwork(max_batch=B, precision=precision)
    frames = torch.zeros((B, 5, 80, 80), dtype=torch.uint8, device="cuda")
    a, r, t = torch.zeros(B, dtype=torch.uint8, device="cuda"), torch.zeros(B, device="cuda"), torch.zeros(B, dtype=torch.uint8, device="cuda")
    abs_err = torch.zeros(B, device="cuda")

    def step(sampling=None, **kw):
        d = _lib.QnetStepArgs(variant=1, gamma=0.99, params_dev=net.params.data_ptr(), target_params_dev=net.target.data_ptr(),
                              grads_dev=net.grads.data_ptr(), loss_out_dev=net.loss.data_ptr())
        if sampling is None:
            d.batch, d.frames_dev, d.sample_stride = B, frames.data_ptr(), 5 * 6400
            d.chan_off_s[:] = (0, 6400, 12800, 19200)
            d.chan_off_next[:] = (6400, 12800, 19200, 25600)
            d.actions_dev, d.rewards_dev, d.terminals_dev = a.data_ptr(), r.data_ptr(), t.data_ptr()
        else:
            d.sampling = C.addressof(sampling)
        for k, v in kw.items():
            setattr(d, k, v)
        rc = L.fb_qnet_step(net._h, C.byref(d), net._stream())
        assert rc == 0 or b"fb_qnet_step" in L.fb_last_error(), L.fb_last_error()
        return rc

    assert step() == 0 and step(variant=0, target_params_dev=None) == 0
    assert step(m_dev=net.adam_m.data_ptr(), v_dev=net.adam_v.data_ptr(), lr=1e-6, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0,
                beta1_power=0.9, beta2_power=0.999) == 0
    for bad in (dict(params_dev=None), dict(grads_dev=None), dict(frames_dev=None), dict(actions_dev=None), dict(rewards_dev=None),
                dict(terminals_dev=None), dict(batch=0), dict(batch=B + 1), dict(variant=3), dict(variant=-1),
                dict(target_params_dev=None), dict(variant=2, target_params_dev=None), dict(m_dev=net.adam_m.data_ptr()),
                dict(v_dev=net.adam_v.data_ptr())):
        assert step(**bad) == -1, bad
    mem = _memory(game, replay, 4, 8, B, 6)
    sp, _ = mem.step_sampling(B)
    assert step(sp) == 0 and step(sp, batch=B) == 0
    for bad in (dict(frames_dev=frames.data_ptr()), dict(sample_stride=5 * 6400), dict(actions_dev=a.data_ptr()),
                dict(rewards_dev=r.data_ptr()), dict(terminals_dev=t.data_ptr()), dict(is_weights_dev=r.data_ptr()),
                dict(chan_off_next=(C.c_int32 * 4)(0, 0, 0, 6400)), dict(batch=B - 1)):
        assert step(sp, **bad) == -1, bad
    pmem = _memory(game, replay, 4, 8, B, 6, prioritized=True)
    psp, _ = pmem.step_sampling(B)
    assert step(psp) == -1 and step(psp, abs_err_out_dev=abs_err.data_ptr()) == 0
    torch.cuda.synchronize()
