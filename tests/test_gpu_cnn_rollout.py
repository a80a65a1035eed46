"""CNNModel trained on device-resident Atari frames of another size and stack depth: RawFrameMultiEnv /
DeviceAtariMultiEnv(size=64, num_stacked_frames=2) -> MultiEnvAgent (rollout buffers [E, T, 64, 64, 2] on the device,
acting through CNNModel's engine) -> A2CObjective.optimize_shared through Session.run."""
import numpy as np
import pytest
import torch

from oracle import preprocess_sq as PS
from test_gpu_raw_env import FakeAtari, _lengths

pytestmark = pytest.mark.gpu

SIZE, K = 64, 2


class HostChainSq:
    """The reference's wrapper chain for one environment at SIZE x SIZE x K, array work by the oracle."""

    def __init__(self, env, frameskip):
        self.env, self.frameskip = env, frameskip
        self.stack = PS.FrameStackSq((SIZE, SIZE, 1), K)
        self.terminated = False

    def reset(self):
        self.terminated = False
        return self.stack.reset(PS.preprocess_frame_sq(self.env.reset(), SIZE)).copy()

    def step(self, action):
        if self.terminated:                             # multi_env.py:128-129
            self.stack.reset(PS.preprocess_frame_sq(self.env.reset(), SIZE))
        frames, total, terminal, info = [], 0.0, False, None
        for _ in range(self.frameskip):                 # wrappers.py:52-62
            f, r, terminal, info = self.env.step(action)
            frames.append(f)
            total += r
            if terminal:
                break
        frame = np.amax((frames[-2], frames[-1]), axis=0) if len(frames) >= 2 else frames[0]
        obs = self.stack.step(PS.preprocess_frame_sq(frame, SIZE), terminal).copy()
        self.terminated = terminal
        return obs, total, terminal, info


def test_raw_frame_multi_env_at_64_by_2_matches_the_host_chain():
    from actorcritic_b200.envs.atari.raw_env import RawFrameMultiEnv
    e_count = 5
    env = RawFrameMultiEnv([FakeAtari(40 + i, _lengths(i)) for i in range(e_count)], size=SIZE, num_stacked_frames=K)
    assert env.observation_space.shape == (SIZE, SIZE, K) and not env.pre.kpre
    chains = [HostChainSq(FakeAtari(40 + i, _lengths(i)), 4) for i in range(e_count)]
    got = env.reset()
    assert tuple(got.shape) == (e_count, SIZE, SIZE, K)
    assert np.array_equal(got.cpu().numpy(), np.stack([c.reset() for c in chains]))
    rng = np.random.default_rng(1)
    saw_terminal = False
    for t in range(30):
        actions = rng.integers(0, 4, e_count).tolist()
        obs, rew, term = env.step_device(torch.tensor(actions, dtype=torch.int32, device="cuda"))
        ref = [c.step(a) for c, a in zip(chains, actions)]
        assert np.array_equal(obs.cpu().numpy(), np.stack([r[0] for r in ref])), "step %d" % t
        assert rew.cpu().tolist() == [r[1] for r in ref]
        assert term.bool().cpu().tolist() == [r[2] for r in ref]
        saw_terminal |= any(r[2] for r in ref)
    assert saw_terminal
    env.close()


def _setup(seed=0, use_graphs=True):
    import actorcritic_b200 as ac
    from actorcritic_b200 import kfac, nn, objectives, spaces
    from actorcritic_b200.cnn import CNNModel
    from actorcritic_b200.kfac_utils import ColdStartPeriodicInvUpdateKfacOpt
    model = CNNModel(spaces.Box(low=0, high=255, shape=(SIZE, SIZE, K), dtype=np.uint8), spaces.Discrete(4),
                     conv_layers=((16, 8, 4), (32, 4, 2), (32, 3, 1)), hidden_sizes=(128,), random_seed=seed)
    model.engine_options["use_graphs"] = use_graphs
    objective = objectives.A2CObjective(model, discount_factor=0.99, entropy_regularization_strength=0.01)
    global_step = ac.GlobalStep()
    lr = nn.linear_decay(0.25, 0.025, global_step, 1e6)
    lc = kfac.LayerCollection()
    model.register_layers(lc)
    model.register_predictive_distributions(lc)
    cold = nn.ClipGlobalNormOptimizer(nn.MomentumOptimizer(learning_rate=0.0003, momentum=0.9), clip_norm=0.5)
    optimizer = ColdStartPeriodicInvUpdateKfacOpt(num_cold_updates=4, cold_optimizer=cold, invert_every=4, learning_rate=lr,
                                                  cov_ema_decay=0.99, damping=0.01, layer_collection=lc, momentum=0.9,
                                                  norm_constraint=0.0001)
    optimize_op = objective.optimize_shared(optimizer, baseline_loss_weight=0.5, global_step=global_step)
    return ac, model, optimize_op


def _feed(model, obs, act, rew, term, nxt):
    return {model.observations_placeholder: obs, model.bootstrap_observations_placeholder: nxt,
            model.actions_placeholder: act, model.rewards_placeholder: rew, model.terminals_placeholder: term}


def test_acktr_from_device_rollouts_equals_the_same_arrays_from_the_host():
    """Ten ACKTR updates (the cold phase, covariance updates and an inverse refresh) trained from the agent's device
    tensors leave the same parameters, bit for bit, as the same rollouts fed as host numpy arrays."""
    from actorcritic_b200 import agents
    from actorcritic_b200.envs.atari.raw_env import RawFrameMultiEnv
    e_count, steps, updates = 4, 5, 10
    ac, model, optimize_op = _setup()
    env = RawFrameMultiEnv([FakeAtari(60 + i, _lengths(i)) for i in range(e_count)], size=SIZE, num_stacked_frames=K)
    agent = agents.MultiEnvAgent(env, model, num_steps=steps)
    rollouts = []
    with ac.Session() as session:
        for _ in range(updates):
            obs, act, rew, term, nxt, infos = agent.interact(session)
            assert all(isinstance(x, torch.Tensor) and x.is_cuda for x in (obs, act, rew, term, nxt))
            assert tuple(obs.shape) == (e_count, steps, SIZE, SIZE, K) and obs.dtype == torch.uint8
            assert tuple(nxt.shape) == (e_count, SIZE, SIZE, K)
            assert len(infos) == e_count and len(infos[0]) == steps
            rollouts.append(tuple(x.cpu().numpy().copy() for x in (obs, act, rew, term, nxt)))
            session.run(optimize_op, feed_dict=_feed(model, obs, act, rew, term, nxt))
        assert model.engine.is_learner and model.engine.get_state()["inverses_valid"]
        device_params = model.get_variables()
    env.close()
    assert any(r[3].any() for r in rollouts)                          # episodes ended inside the rollouts

    ac, host_model, optimize_op = _setup()
    with ac.Session() as session:
        for obs, act, rew, term, nxt in rollouts:
            session.run(optimize_op, feed_dict=_feed(host_model, obs, act, rew, term, nxt))
        host_params = host_model.get_variables()
    for name, v in device_params.items():
        assert np.isfinite(v).all() and np.array_equal(v, host_params[name]), name
    assert any(not np.array_equal(v, _setup()[1].get_variables()[n]) for n, v in device_params.items())   # it trained


def test_graph_replayed_device_rollout_equals_the_eager_one():
    """DeviceAtariMultiEnv(size=64, num_stacked_frames=2) rollouts replayed as one CUDA graph (from the third call on)
    equal step-by-step ones: observations, actions, rewards, terminals, next observations."""
    from actorcritic_b200 import agents
    from actorcritic_b200.envs.atari.device_env import DeviceAtariMultiEnv

    def run(use_graphs):
        ac, model, _ = _setup(seed=3, use_graphs=use_graphs)
        env = DeviceAtariMultiEnv(6, pool_frames=8, terminal_prob=0.2, seed=5, size=SIZE, num_stacked_frames=K)
        agent = agents.MultiEnvAgent(env, model, 8)
        outs = []
        with ac.Session() as session:
            for _ in range(5):
                o, a, r, t, nxt, _ = agent.interact(session)
                torch.cuda.synchronize()
                outs.append(tuple(x.cpu().numpy().copy() for x in (o, a, r, t, nxt)))
        return outs, getattr(agent, "_graph_state", 0)

    eager, st0 = run(False)
    graph, st1 = run(True)
    assert st0 == 0 and st1 == 2
    assert eager[0][0].shape == (6, 8, SIZE, SIZE, K)
    for i, (x, y) in enumerate(zip(eager, graph)):
        for j, name in enumerate(("observations", "actions", "rewards", "terminals", "next_observations")):
            assert np.array_equal(x[j], y[j]), (i, name)
    assert len({tuple(x[1].ravel()) for x in eager}) > 1


def test_atari_model_with_default_raw_frame_env_still_runs_k_pre():
    from torch.profiler import ProfilerActivity, profile
    from actorcritic_b200 import agents
    from actorcritic_b200.envs.atari.raw_env import RawFrameMultiEnv
    from test_gpu_api import _build
    ac, model, *_ = _build(True, 4, 5)
    env = RawFrameMultiEnv([FakeAtari(80 + i, _lengths(i)) for i in range(4)])
    assert env.observation_space.shape == (84, 84, 4) and env.pre.kpre
    agent = agents.MultiEnvAgent(env, model, num_steps=5)
    with ac.Session() as session:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            obs, *_ = agent.interact(session)
            torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert any("preprocess_kernel" in n or "preprocess_persistent_kernel" in n for n in names), sorted(names)
    assert not any("preprocess_sq_kernel" in n for n in names)
    assert tuple(obs.shape) == (4, 5, 84, 84, 4)
    env.close()
