"""End-to-end: the reference's driver loop (FlappyBirdDQN.py:60-76) on the batched GameState + Brain*."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import qnet_oracle as qo  # noqa: E402
from oracle import replay_oracle as ro  # noqa: E402


@pytest.fixture(scope="module")
def mods():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dqnflappybird_b200 import brains, game
    return game, brains


def test_reference_driver_loop_single_env(mods):
    """the five-line loop of FlappyBirdDQN.py:60-76, call shapes unchanged (numpy in / numpy out for one env)"""
    game, brains = mods
    brain = brains.BrainDQNNature(2, "bird", replay_memory_per_env=200, observe=40., replace_target_iter=7)
    flappyBird = game.GameState(num_envs=1, seed=3, history=204, ring=brain.ring)
    action0 = np.array([1, 0])
    observation0, reward0, terminal, curScore = flappyBird.frame_step(action0)
    brain.setInitState(observation0[:, :, 0])
    p0 = brain.net.params.clone(); t0 = brain.net.target.clone()
    assert not torch.equal(p0, t0)                       # target net is initialised independently (SURVEY Q4)
    eps = 0.03
    for step in range(80):
        action = brain.getAction()
        assert action.shape == (2,) and action.sum() == 1
        if brain.onlineTimeStep > 40 and eps > 0:        # the decrement happens inside getAction (BrainDQN.py:112-114)
            eps -= 0.03 / 1000000.
        assert brain.epsilon == eps
        nextObserv, reward, terminal, curScore = flappyBird.frame_step(action)
        assert nextObserv.shape == (80, 80, 1)
        brain.setPerception(nextObserv, action, reward, terminal, curScore)
        if step < 41:
            assert torch.equal(brain.net.params, p0)     # observing: no training until onlineTimeStep > OBSERVE
    assert brain.timeStep == 80 and brain.onlineTimeStep == 80 and len(brain.replayMemory) == 80
    assert not torch.equal(brain.net.params, p0) and brain.net.adam_steps == 80 - 41
    assert torch.isfinite(brain.net.params).all()
    assert not torch.equal(brain.net.target, t0)         # synced at timeStep % 7 == 0
    cs = brain.currentState
    assert cs.shape == (1, 80, 80, 4) and torch.equal(cs[0, :, :, 3], flappyBird.ring[0, flappyBird.slot])


def test_training_step_matches_oracle_on_the_sampled_minibatch(mods):
    """one BrainDQNNature update, batched envs: the minibatch is what CPython's random.sample picks from the same
    word stream, and the gradient equals the float64 oracle's on exactly those transitions"""
    game, brains = mods
    N, C = 16, 28
    brain = brains.BrainDQNNature(2, "bird", num_envs=N, replay_memory_per_env=C, observe=1e9, batch_size=32, seed=5, precision="fp32")
    gs = game.GameState(num_envs=N, seed=9, history=C + 4, ring=brain.ring)
    hist = []
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    hist.append((obs.cpu().numpy().copy(), None, None, None))
    rng = np.random.default_rng(0)
    for k in range(1, 41):
        a = torch.from_numpy((rng.random(N) < 0.2).astype(np.uint8)).cuda()
        obs, r, t, s = gs.frame_step(a)
        brain.setPerception(obs, a, r, t, s)
        hist.append((obs.cpu().numpy().copy(), a.cpu().numpy(), r.cpu().numpy().copy(), t.cpu().numpy().copy()))
    mem = brain.replayMemory
    assert mem.t == 40 and len(mem) == N * C
    pos = mem.rng_positions()[0]
    orc = ro.UniformSampler(mem.seed); orc.pos = pos
    want = orc.sample(N * C, 32)
    p = brain.net.params.cpu().numpy().copy(); tg = brain.net.target.cpu().numpy().copy()
    brain.timeStep = 3                                   # not a multiple of 500: no target sync in this step
    brain._trainQNetwork()
    env, ks = ro.population_to_transition(np.array(want), 40, N, C)
    x = np.stack([[hist[max(k - 4 + f, 0)][0][e] for f in range(5)] for e, k in zip(env, ks)])
    a = np.array([hist[k][1][e] for e, k in zip(env, ks)]); r = np.array([hist[k][2][e] for e, k in zip(env, ks)])
    t = np.array([hist[k][3][e] for e, k in zip(env, ks)]).astype(np.uint8)
    loss, g_ref, *_ = qo.loss_and_grads(1, p, tg, x[:, 0:4], x[:, 1:5], a, r, t)
    g = brain.net.grads.cpu().numpy().astype(np.float64)
    assert abs(brain.net.loss.item() - loss) <= 1e-4 * abs(loss)
    assert np.linalg.norm(g - g_ref) <= 3e-4 * np.linalg.norm(g_ref)
    ref = qo.AdamTF1(len(p)); want_p = ref.step(p.copy(), g_ref.astype(np.float32))
    np.testing.assert_allclose(brain.net.params.cpu().numpy(), want_p, rtol=0, atol=3e-7)


@pytest.mark.parametrize("name", ["dqn", "dqnnature", "ddqn", "duelingdqn", "prioritydqn"])
def test_every_brain_trains_batched(mods, name):
    """FlappyBirdDQN.py:41-50 model table: each agent runs the batched loop past OBSERVE and updates its weights"""
    game, brains = mods
    N = 64
    brain = brains.MODELS[name](2, "bird", num_envs=N, replay_memory_per_env=12, observe=6., batch_size=32, seed=1,
                                replace_target_iter=4)
    assert brain.net.dueling == (name == "duelingdqn")
    gs = game.GameState(num_envs=N, seed=2, history=16, ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    p0 = brain.net.params.clone()
    for _ in range(25):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a)
        brain.setPerception(obs, a, r, t, s)
    gs.check_errors()
    assert brain.net.adam_steps == 25 - 7
    assert torch.isfinite(brain.net.params).all() and not torch.equal(brain.net.params, p0)
    assert torch.isfinite(brain.net.loss).all()
    if name == "prioritydqn":
        tree = brain.replayMemory.tree()
        assert tree[0].item() > 0 and abs(tree[0].item() - tree[N * 12 - 1:].sum().item()) < 1e-9
    sd = brain.state_dict()
    brain.load_state_dict(sd)
    assert brain.timeStep == 25


def test_quirk_switches(mods):
    game, brains = mods
    b = brains.BrainDoubleDQN(2, "bird", num_envs=4, replay_memory_per_env=8, reference_quirks=True)
    assert b._trainQNetwork.__func__ is not brains.BrainDoubleDQN.trainQNetwork
    d = brains.BrainDuelingDQN(2, "bird", num_envs=4, replay_memory_per_env=8, reference_quirks=True)
    assert d.net.dueling is False and d.net.n_params == 898722       # Q2: the shipped code builds the plain net
    d2 = brains.BrainDuelingDQN(2, "bird", num_envs=4, replay_memory_per_env=8)
    assert d2.net.dueling is True and d2.net.n_params == 899235


def test_logging_surface_and_disk_checkpoint(mods, tmp_path):
    """Rows N2/N3 of SURVEY 8(f): the five log lists / text files of BrainDQN.py:49-58,270-294 fed from device-side
    accumulators, and save/restore in the layout of BrainDQN.py:176-192,226-233 (weights + the three pickles)."""
    import pickle
    game, brains = mods
    N = 64
    kw = dict(num_envs=N, replay_memory_per_env=12, batch_size=32, observe=5, record=True, root_dir=str(tmp_path), save_every=10, seed=4)
    brain = brains.BrainDQNNature(2, "bird", **kw)
    assert brain.logs_path.endswith("logs_bird/dqn_nature/") and brain.save_path.endswith("saved_parameters/dqn_nature/")
    gs = game.GameState(num_envs=N, seed=2, history=16, ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    want_steps, want_envs, want_scores, want_rewards = [], [], [], []
    for step in range(60):
        a = torch.zeros(N, dtype=torch.uint8, device="cuda") if step % 3 else brain.getAction()
        obs, r, t, s = gs.frame_step(a)
        tt, ss = t.cpu().numpy(), s.cpu().numpy()
        for e in np.nonzero(tt)[0]:
            want_steps.append(brain.timeStep); want_envs.append(int(e)); want_scores.append(int(ss[e]))
        want_rewards.append(float(r.mean().item()))
        brain.setPerception(obs, a, r, t, s)
    assert len(want_steps) > 0                        # all-no-op episodes hit the ground on their 19th step
    # saved at timeStep 10, 20, ... 50 (inside _trainQNetwork, BrainDQN.py:227): the lists were emptied into the files then
    brain.flush_logs()
    n_file = len(brain._get_loss_score_timestep_reward_qtarget_from_file()[1])
    brain._save_loss_score_timestep_reward_qtarget_to_file()
    loss, scores, steps, rewards, q = brain._get_loss_score_timestep_reward_qtarget_from_file()
    assert n_file <= len(scores)
    assert [int(x) for x in steps] == want_steps and [int(x) for x in scores] == want_scores
    np.testing.assert_allclose(rewards, want_rewards, rtol=1e-6)
    assert len(loss) == brain.net.adam_steps == 60 - 6 and len(q) == 32 * len(loss)
    assert np.isfinite(loss).all() and brain.gameTimes == len(want_steps)
    # the three pickles, readable the way BrainDQN.py:186-189 reads them
    with open(brain.saved_parameters_file_path, "rb") as f:
        g, ts, eps = pickle.load(f), pickle.load(f), pickle.load(f)
    assert ts == 50 and isinstance(eps, float) and g <= brain.gameTimes
    # a new brain on the same directory resumes from the newest checkpoint: timeStep and epsilon restored, onlineTimeStep not (Q12)
    ref_params = torch.load(brain.save_path + "bird-50.pt")["params"]
    b2 = brains.BrainDQNNature(2, "bird", **kw)
    assert b2.timeStep == 50 and b2.onlineTimeStep == 0 and b2.epsilon == eps and b2.gameTimes == g
    assert torch.equal(b2.net.params.cpu(), ref_params.cpu())
    # without a checkpoint directory nothing is restored and save() says why it cannot run
    b3 = brains.BrainDQN(2, "bird", num_envs=4, replay_memory_per_env=8)
    assert b3.timeStep == 0
    with pytest.raises(RuntimeError):
        b3.save()


@pytest.mark.parametrize("model", ["dqn", "ddqn", "dqnnature", "duelingdqn", "prioritydqn"])
def test_driver_loop_every_model(mods, model):
    """FlappyBirdDQN.py:36-79, batched (row N4): --model picks the Brain, the env draws into its ring, the loop trains."""
    from dqnflappybird_b200 import play
    brain, gs, stats = play.playFlappyBird(model, num_envs=32, steps=20, replay_memory_per_env=12, batch_size=32, observe=3)
    assert stats == {"steps": 20, "envs": 32, "updates": 20 - 4}
    assert brain.timeStep == 20 and gs.steps == 21                  # one no-op step for the initial state (:63-69)
    assert gs.ring.data_ptr() == brain.ring.data_ptr()
    assert torch.isfinite(brain.net.params).all()


def test_driver_loop_single_env_and_bad_model(mods):
    from dqnflappybird_b200 import play
    brain, gs, stats = play.playFlappyBird("dqnnature", num_envs=1, steps=12, replay_memory_per_env=40, batch_size=4, observe=5)
    assert stats["updates"] == 12 - 6 and brain.timeStep == 12
    with pytest.raises(SystemExit):
        play.playFlappyBird("actorcritic")                         # outside the DQN hot path, like an unknown model (:51-54)


@pytest.mark.parametrize("model", ["dqn", "ddqn", "duelingdqn", "prioritydqn"])
def test_sampling_inside_the_step_is_identical_to_separate_launches(mods, model):
    """fb_qnet_step with `sampling`: random.sample + gather as the first two kernels of the update's CUDA graph (their `t`
    patched into the graph nodes every step) -- same minibatches, same parameters, same stream positions as
    fb_replay_sample_uniform + fb_replay_gather + fb_qnet_step on that minibatch, while the replay fills, wraps and the graph
    replays"""
    game, brains = mods
    N = 48
    runs = []
    for fuse in (True, False):
        brain = brains.MODELS[model](2, "bird", num_envs=N, replay_memory_per_env=10, batch_size=32, observe=3, seed=6, lr=1e-4)
        brain.fuse_sampling = fuse
        gs = game.GameState(num_envs=N, seed=2, history=14, ring=brain.ring)
        obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device="cuda"))
        brain.setInitState(obs)
        picked = []
        for _ in range(30):
            a = brain.getAction()
            obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
            brain.setPerception(obs, a, r, t, s)
            picked.append(brain.replayMemory._idx[:32].clone())
        runs.append((brain, picked))
    (b1, p1), (b0, p0) = runs
    assert b1.net.adam_steps == b0.net.adam_steps == 30 - 4
    for x, y in zip(p1[4:], p0[4:]):              # (no minibatch is drawn during the first OBSERVE + 1 steps)
        assert torch.equal(x, y)
    assert torch.equal(b1.net.params, b0.net.params) and torch.equal(b1.net.adam_v, b0.net.adam_v)
    assert b1.replayMemory.rng_positions() == b0.replayMemory.rng_positions()
    assert torch.equal(b1.net.loss, b0.net.loss)
    # inside the step the convolutions read the drawn frames in place from the ring (offsets left by the sampler) and the gather
    # runs beside them: the caller-visible minibatch buffers are filled all the same
    m1, m0 = b1.replayMemory, b0.replayMemory
    assert torch.equal(m1._frames[:32], m0._frames[:32]) and torch.equal(m1._a[:32], m0._a[:32])
    assert torch.equal(m1._r[:32], m0._r[:32]) and torch.equal(m1._t[:32], m0._t[:32])
    if model == "prioritydqn":                    # Memory.sample at the head, Memory.batch_update at the tail of the same graph
        assert torch.equal(b1.replayMemory.tree(), b0.replayMemory.tree()) and b1.replayMemory.beta == b0.replayMemory.beta
        assert torch.equal(b1.replayMemory._isw[:32], b0.replayMemory._isw[:32])


def test_sampling_inside_the_step_raises_like_random_sample(mods):
    game, brains = mods
    brain = brains.BrainDQNNature(2, "bird", num_envs=2, replay_memory_per_env=8, batch_size=32, observe=0)
    gs = game.GameState(num_envs=2, seed=2, history=12, ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(2, dtype=torch.uint8, device="cuda"))
    brain.setInitState(obs)
    a = brain.getAction()
    obs, r, t, s = gs.frame_step(a)
    brain.setPerception(obs, a, r, t, s)          # onlineTimeStep 0: no training yet
    a = brain.getAction()
    obs, r, t, s = gs.frame_step(a)
    with pytest.raises(ValueError):               # 2 envs x 2 transitions < 32 (random.sample's ValueError, BrainDQN.py:197)
        brain.setPerception(obs, a, r, t, s)
