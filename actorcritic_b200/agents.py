"""actorcritic/agents.py: agents that sample rollouts.  `interact()` keeps the reference's contract - the 6-tuple
(observations, actions, rewards, terminals, next_observations, infos) in batch-major [environment][step] order
(agents.py:26-45,157-228) - for any `MultiEnv`.  When the environment is device resident
(envs.atari.device_env.DeviceAtariMultiEnv) the rollout stays on the GPU: K-PRE writes each step's frame stacks
straight into a [E,T,*observation_shape] rollout buffer (sized from the environment's observation space: [E,T,84,84,4]
for AtariModel, [E,T,S,S,k] for a CNNModel on other frames) and the tuple holds torch tensors instead of nested lists
(the replacement for the reference's Python list shuffling, SURVEY 8(a) a4).  The acting engine is the model's own
(`_build_engine`), so any model with an engine (AtariModel, CNNModel) rolls out this way."""
from abc import ABCMeta, abstractmethod

import numpy as np
import torch


class Agent(object, metaclass=ABCMeta):
    """agents.py:6-47."""

    @abstractmethod
    def interact(self, session):
        pass


def transpose_list(values):
    """agents.py:231-257: [[a1, a2], [b1, b2], [c1, c2]] -> [[a1, b1, c1], [a2, b2, c2]]."""
    return list(map(list, zip(*values)))


class MultiEnvAgent(Agent):
    """agents.py:134-228."""

    def __init__(self, multi_env, model, num_steps):
        self._env = multi_env
        self._model = model
        self._num_steps = num_steps
        self._observations = None   # kept between calls to reuse `next_observations` (agents.py:155,198-200,219)

    def interact(self, session):
        if getattr(self._env, "device_resident", False):
            return self._interact_device(session)
        observation_steps, action_steps, reward_steps, terminal_steps, info_steps = [], [], [], [], []
        next_observations = self._observations
        if next_observations is None:
            next_observations = self._env.reset()
        for _ in range(self._num_steps):
            observation_steps.append(next_observations)
            batch_next_observations = transpose_list([next_observations])          # [env] -> [env, 1]
            actions = self._model.sample_actions(batch_next_observations, session)
            next_observations, rewards, terminals, infos = self._env.step(actions)
            action_steps.append(actions)
            reward_steps.append(rewards)
            terminal_steps.append(terminals)
            info_steps.append(infos)
        self._observations = next_observations
        return (transpose_list(observation_steps), transpose_list(action_steps), transpose_list(reward_steps),
                transpose_list(terminal_steps), next_observations, transpose_list(info_steps))

    def _interact_device(self, session):
        env, t_count = self._env, self._num_steps
        engine = self._model.engine
        if engine is None:
            engine = self._model._build_engine(session, env.num_envs, t_count, None)
        if self._observations is None:
            self._observations = env.reset()                                       # uint8 [E,S,S,k] on the device
        # A device environment whose rollouts of this length always touch the same buffers (rollout_repeats) is replayed as
        # ONE CUDA graph: T x (K-PRE, acting forward, sample, bookkeeping copies) = ~14 T launches become one.  The first
        # rollout runs eagerly (one-time host work of the library), the second is captured, later ones are replayed.
        repeat = getattr(env, "rollout_repeats", None)
        if engine.config.use_graphs and repeat is not None and repeat(t_count):
            return self._interact_device_graph(session, engine)
        return self._rollout_eager(engine)

    def _rollout_buffers(self, engine):
        env, t_count = self._env, self._num_steps
        e_count, dev = env.num_envs, env.device
        space = env.observation_space
        obs_shape = tuple(int(d) for d in space.shape)
        obs_dtype = torch.from_numpy(np.zeros(0, space.low.dtype)).dtype
        if getattr(self, "_step_actions", None) is None or self._step_actions.shape != (t_count, e_count):
            self._step_actions = torch.empty((t_count, e_count), dtype=torch.int32, device=dev)
            self._obs_buf = torch.empty((e_count, t_count) + obs_shape, dtype=obs_dtype, device=dev)
            self._next_obs_buf = torch.empty((e_count,) + obs_shape, dtype=obs_dtype, device=dev)
            self._act_buf = torch.empty((e_count, t_count), dtype=torch.uint8, device=dev)
            self._rew_buf = torch.empty((e_count, t_count), dtype=torch.float32, device=dev)
            self._term_buf = torch.empty((e_count, t_count), dtype=torch.uint8, device=dev)

    def _rollout_steps(self, engine):
        """T steps into the agent's own buffers (stable pointers: the library replays each acting step as a CUDA graph;
        per-step results are gathered step-major and turned batch-major once at the end)."""
        env, t_count = self._env, self._num_steps
        e_count = env.num_envs
        self._rollout_buffers(engine)
        cur = self._observations
        reward_steps, terminal_steps, info_steps = [], [], []
        for t in range(t_count):
            self._obs_buf[:, t].copy_(cur)
            a = engine.act(cur, out=self._step_actions[t])                         # int32 [E]
            cur, r, term = env.step_device(a)
            reward_steps.append(r)
            terminal_steps.append(term)
            # environments hosted on the CPU (envs.atari.raw_env.RawFrameMultiEnv) report their info dicts per step
            info_steps.append(list(getattr(env, "last_infos", None) or [{} for _ in range(e_count)]))
        self._act_buf.copy_(self._step_actions.t())
        torch.stack(reward_steps, dim=1, out=self._rew_buf)
        torch.stack(terminal_steps, dim=1, out=self._term_buf)
        self._next_obs_buf.copy_(cur)      # the environment reuses its stack buffer; the tuple must not alias it
        return info_steps

    def _result(self, info_steps):
        self._observations = self._next_obs_buf.clone()
        return (self._obs_buf.clone(), self._act_buf.clone(), self._rew_buf.clone(), self._term_buf.bool(),
                self._next_obs_buf.clone(), transpose_list(info_steps))

    def _rollout_eager(self, engine):
        with engine.on_stream():
            info_steps = self._rollout_steps(engine)
            return self._result(info_steps)

    def _interact_device_graph(self, session, engine):
        env, t_count = self._env, self._num_steps
        state = getattr(self, "_graph_state", 0)
        if state == 0:                     # first rollout: eager
            self._graph_state = 1
            return self._rollout_eager(engine)
        with engine.on_stream():
            if state == 1:                 # second rollout: capture (the captured launches also execute on replay only)
                # the rollout must start from the agent's persistent observation buffer
                self._cur_buf = self._observations.clone()
                self._observations = self._cur_buf
                t0 = env.t
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=engine.stream):
                    self._graph_infos = self._rollout_steps(engine)
                    self._cur_buf.copy_(self._next_obs_buf)
                env.t = t0                 # capture does not execute: the environment's host-side clock is advanced per replay
                self._graph, self._graph_state = graph, 2
                self._observations = self._cur_buf
            # replay: the environment's own stack buffer and the agent's `_cur_buf` carry the state between rollouts
            self._graph.replay()
            env.t += t_count
            out = (self._obs_buf.clone(), self._act_buf.clone(), self._rew_buf.clone(), self._term_buf.bool(),
                   self._next_obs_buf.clone(), transpose_list(self._graph_infos))
            self._observations = self._cur_buf
            return out


class SingleEnvAgent(Agent):
    """agents.py:50-131: same contract with one environment ([1][step])."""

    def __init__(self, env, model, num_steps):
        self._env = env
        self._model = model
        self._num_steps = num_steps
        self._observation = None

    def interact(self, session):
        observations, actions, rewards, terminals, infos = [], [], [], [], []
        next_observation = self._observation
        if next_observation is None:
            next_observation = self._env.reset()
        for _ in range(self._num_steps):
            observations.append(next_observation)
            action = self._model.sample_actions([[next_observation]], session)[0]
            action = action[0] if isinstance(action, list) else action
            next_observation, reward, terminal, info = self._env.step(action)
            actions.append(action)
            rewards.append(reward)
            terminals.append(terminal)
            infos.append(info)
            if terminal:
                next_observation = self._env.reset()
        self._observation = next_observation
        return [observations], [actions], [rewards], [terminals], [next_observation], [infos]
