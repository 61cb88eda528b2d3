"""Multi-agent environments: the reference's dict-of-agents API over the batched B200 simulator.

Mirrors zombsole/gym/multiagent_env.py:
  * ``MultiagentZombsoleEnv`` / ``MultiagentZombsoleEnvDiscreteAction``: the reference's constructor
    arguments and return types (dicts keyed by agent id; observation ``(3, w, w)`` per agent); one world.
  * ``MultiagentZombsoleVectorEnv``: the same arguments plus ``num_envs``; ``step(actions [N, A])`` ->
    ``(obs [N, A, 3, w, w] int32, reward [N, A] float64, terminated [N] bool, truncated [N] bool,
    {"agent_mask": [N, A] bool})`` as CUDA tensors.  ``agent_mask`` marks the agents that were alive
    before the step, i.e. the keys the reference's per-agent dicts would carry
    (multiagent_env.py:88-97,156-166); rewards of the others are 0 and their windows are centred on
    the position where they died.
"""
import numpy as np
import torch

from .. import abi
from ..engine import ZsEngine
from ..gym_env import CompactHostOutputs, FinalObservation, NextStepAutoreset, check_final_observation, encode_action
from ..spaces import Box, Dict, Discrete, Text
from ..things import Game


class MultiagentZombsoleVectorEnv(CompactHostOutputs, FinalObservation, NextStepAutoreset):
    metadata = {"render.modes": ["human"]}
    reward_range = (-float("inf"), float("inf"))
    game_actions = [
        {"action_type": "move", "parameter": [0, 1]},
        {"action_type": "move", "parameter": [-1, 0]},
        {"action_type": "move", "parameter": [0, -1]},
        {"action_type": "move", "parameter": [1, 0]},
        {"action_type": "attack_closest"},
        {"action_type": "heal"},
        {"action_type": "heal_closest"},
    ]

    def __init__(self, rules_name, player_names, map_name, agent_ids, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_surroundings_width=21, observation_position_encoding_style="channels",
                 agent_weapons="rifle", debug=False, *, num_envs=1, device="cuda", seed=0, env_index_base=0,
                 max_episode_steps=None, auto_reset=True, host_outputs=False, host_threads=0, compact_words=0,
                 final_observation=False, autoreset_mode="same_step"):
        if render_mode is not None:
            if render_mode not in self.metadata["render.modes"]:
                raise ValueError("render_mode={} is not supported".format(render_mode))
            raise NotImplementedError("rendering is outside the batched simulator's scope (render_mode=None only)")
        self.render_mode = None
        check_final_observation(final_observation, auto_reset, host_outputs)
        abi.check_autoreset_mode(autoreset_mode, auto_reset, final_observation)
        width = observation_surroundings_width
        if (width % 2 == 0) or (width <= 1):  # observation.py:206-207
            raise ValueError("surroundings width must be an odd number greater than 1")
        lpes = observation_position_encoding_style.lower()
        if lpes not in ["simple", "channels"]:
            raise ValueError(f"{lpes} must be \"simple\" or \"channels\"")
        if lpes != "channels":
            # the reference's get_observation needs get_observation_at_position, which only the channels
            # handler has (multiagent_env.py:92 vs observation.py:145-156): "simple" raises AttributeError there
            raise AttributeError("'SurroundingsSimpleObservation' object has no attribute 'get_observation_at_position'")
        self.surroundings_width = width
        self.position_encoding_style = observation_position_encoding_style
        self.possible_agents = list(agent_ids)
        self.cfg = abi.make_config(rules_name, list(player_names), list(agent_ids), agent_weapons, initial_zombies,
                                   minimum_zombies, abi.OBS_SURROUNDINGS, abi.OBS_CHANNELS, width, True, num_envs,
                                   seed=seed, env_index_base=env_index_base, max_episode_steps=max_episode_steps,
                                   auto_reset=auto_reset, autoreset_mode=autoreset_mode)
        self.engine = ZsEngine(self.cfg, map_name, device=device)
        self.num_envs = num_envs
        self.num_agents = len(agent_ids)
        self.device = self.engine.device
        self.debug = debug
        self._ctor = (rules_name, list(player_names), list(agent_ids), initial_zombies, minimum_zombies)
        self.action_spaces = {aid: Discrete(len(self.game_actions)) for aid in self.possible_agents}
        self.observation_spaces = {aid: Box(low=0, high=128, shape=(3, width, width), dtype=np.int32)
                                   for aid in self.possible_agents}
        # host_outputs: the kernel writes observations, rewards, flags and the agent mask straight into pinned host memory and
        # reads the actions from there; step() synchronises the stream once and also leaves the agents' lives after the step
        # in `agent_life_host` (what a host loop needs to know who is still playing, multiagent_env.py:169)
        # host_outputs="compact": the same host tensors, but what crosses PCIe every step is one small record per env (the
        # agents' window centres and lives, the rewards, the mask, the flags and the cells any window shows that differ from
        # the map's pristine layer) which the library's host threads expand into the windows (zs_step_host_agents);
        # "compact-copy" is the same with explicit copies and a stream synchronisation between the stages
        # (zs_step_compact_agents / zs_expand_compact_agents, include/zs_b200.h)
        if isinstance(host_outputs, str) and host_outputs not in ("compact", "compact-copy"):
            raise ValueError("host_outputs must be False, True, 'compact' or 'compact-copy'")
        self.compact = host_outputs in ("compact", "compact-copy")
        self.streamed = host_outputs == "compact"
        self.host_outputs = bool(host_outputs)
        self.host_threads = int(host_threads)
        if self.compact and not self.engine.agent_compact_words():
            raise ValueError("host_outputs=%r needs at most 32 things per env (one lane per thing in the step kernel); this game "
                             "has %d (bots + agents + zombies)" % (host_outputs, self.engine.M))
        if self.host_outputs:
            self.obs, self.reward, self._term, self._trunc = self.engine.new_host_outputs()
            self._mask = torch.ones((num_envs, self.num_agents), dtype=torch.uint8).pin_memory()
            self._actions = torch.zeros((num_envs, self.num_agents, 3), dtype=torch.int32).pin_memory()
            self.agent_life_host = torch.zeros((num_envs, self.num_agents), dtype=torch.int16).pin_memory()
            if self.compact:
                self._dev_obs = self.engine.new_obs()  # full rows of the rare envs a record cannot hold
                self._overflow = torch.zeros(num_envs, dtype=torch.int32)
                self.compact_overflows = 0
                self._act_pin = torch.zeros((num_envs, self.num_agents), dtype=torch.int32).pin_memory()
                self._actions_pin = self._actions
                self._size_records(int(compact_words) if compact_words else self.engine.agent_compact_words())
        else:
            self.obs = self.engine.new_obs()
            self.reward, self._term, self._trunc = self.engine.new_outputs()
            self._mask = torch.ones((num_envs, self.num_agents), dtype=torch.uint8, device=self.device)
            self._actions = torch.zeros((num_envs, self.num_agents, 3), dtype=torch.int32, device=self.device)
        self._h2d_done, self._h2d_pending = None, False
        FinalObservation.__init__(self, final_observation)
        NextStepAutoreset.__init__(self, autoreset_mode)

    def game(self, env=0):
        rules_name, player_names, agent_ids, iz, mz = self._ctor
        return Game(self.engine, env, rules_name, player_names, agent_ids, iz, mz)

    def get_observation(self):
        self.engine.encode_obs(self.obs)
        if self.host_outputs:
            torch.cuda.current_stream(self.device).synchronize()
        if self.compact:
            self._compact_first = True  # the rows are complete again: the next step's records start from scratch
        return self.obs

    def _action_rows(self, actions):
        """One dict per env, keyed by agent id -> (type, dx, dy) rows [N, A, 3]; a missing key is ZS_ACT_ABSENT (heal self,
        multiagent_env.py:129-131)."""
        rows = np.zeros((self.num_envs, self.num_agents, 3), np.int32)
        for n, d in enumerate(actions):
            for i, aid in enumerate(self.possible_agents):
                rows[n, i] = encode_action(dict(d[aid], parameter=d[aid].get("parameter", [0, 0]))) \
                    if aid in d else (abi.ACT_ABSENT, 0, 0)
        return rows

    def _stage_actions(self, actions):
        N, A = self.num_envs, self.num_agents
        if isinstance(actions, (list, tuple)) and len(actions) and isinstance(actions[0], dict):
            self._actions.copy_(torch.from_numpy(self._action_rows(actions)), non_blocking=not self.host_outputs)
            return self._actions, abi.ACTIONS_FULL
        t = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
        if self.host_outputs and t.dtype == torch.int32 and t.device.type == "cpu" and t.is_pinned():
            pass  # the kernel reads a pinned host action tensor in place
        elif t.dtype != torch.int32 or t.device != self.device:
            pinned_src = t.device.type == "cpu" and t.is_pinned()
            t = t.to(device=self.device, dtype=torch.int32, non_blocking=True)
            if pinned_src:  # the copy is in flight: step() waits for it before the caller may refill the buffer
                self._h2d_done = self._h2d_done or torch.cuda.Event()
                self._h2d_done.record(torch.cuda.current_stream(self.device))
                self._h2d_pending = True
        t = t.contiguous()
        if t.numel() == N * A:
            return t.view(N, A), abi.ACTIONS_DISCRETE
        if t.numel() == 3 * N * A:
            return t.view(N, A, 3), abi.ACTIONS_FULL
        raise ValueError("actions must hold %d discrete ids or (type, dx, dy) rows" % (N * A))

    def step(self, actions):
        """One transition of every world (multiagent_env.py:111-171); discrete id -1 = key missing."""
        if self.streamed:
            return self._step_streamed(actions)
        a, fmt = self._stage_actions(actions)
        if self.compact:
            return self._step_compact(a, fmt)
        if self.final_observation:
            self.engine.step_final(a, fmt, self.obs, self.final_obs, self.reward, self._term, self._trunc, self._mask)
        else:
            self.engine.step(a, fmt, self.obs, self.reward, self._term, self._trunc, self._mask)
        if self.host_outputs:  # the host owns the results (and any pinned action buffer) when step() returns
            P = self.cfg.n_bots
            self.agent_life_host.copy_(self.engine.fields["life"][:, P:P + self.num_agents], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            self._h2d_pending = False
        if self._h2d_pending:  # a pinned host action buffer is the caller's again when step() returns
            self._h2d_done.synchronize()
            self._h2d_pending = False
        info = {"agent_mask": self._mask.view(torch.bool)}  # (0/1 bytes: views, no kernels)
        if self.final_observation:
            self._final_info(info)
        return self.obs, self.reward, self._term.view(torch.bool), self._trunc.view(torch.bool), info

    # (CompactHostOutputs)
    def _max_words(self):
        return self.engine.agent_compact_max_words()

    def _host_stepper(self):
        return self.engine.host_stepper(self._records_host, self._records_prev, self._dev_obs, self.obs, self.reward, self._term,
                                        self._trunc, self._overflow, self.host_threads, self._mask, self.agent_life_host)

    def _info(self):
        return {"agent_mask": self._mask.view(torch.bool)}

    def _step_compact(self, a, fmt):
        eng = self.engine
        eng.step_compact_agents(a, fmt, self._records, self._dev_obs)
        self._records_host.copy_(self._records, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        self._h2d_pending = False
        over = eng.expand_compact_agents(self._records_host, self._records_prev, self.obs, self.reward, self._term, self._trunc,
                                         self._mask, self.agent_life_host, self._overflow, self._compact_first, self.host_threads)
        self._compact_first = False
        if len(over):
            self._fetch_overflow_rows(over)
        return (self.obs, self.reward, self._term.view(torch.bool), self._trunc.view(torch.bool), self._info())

    def reset(self, seed=None, options=None, mask=None):
        if self.compact:
            return self._compact_reset(mask)
        self.engine.reset(mask, self.obs)
        if self.host_outputs:
            torch.cuda.current_stream(self.device).synchronize()
        return self.obs, {}

    def rollout(self, n_steps, actions=None, first_step_index=0, obs=None, reward=None, terminated=None, truncated=None,
                final_obs=None):
        """As ZombsoleVectorEnv.rollout; ``final_obs`` is a ring shaped like ``obs``."""
        fmt = abi.ACTIONS_DISCRETE
        if actions is not None and actions.dim() == 4:
            fmt = abi.ACTIONS_FULL
        self.engine.rollout(n_steps, first_step_index, actions, fmt, self.obs if obs is None else obs, reward,
                            terminated, truncated, final_obs=final_obs)
        return self.obs if obs is None else obs

    def close(self):
        self.engine.close()

    def __enter__(self):
        return self

    def __exit__(self, *args):
        self.close()
        return False


class MultiagentZombsoleEnv(object):
    """Drop-in for the reference's MultiagentZombsoleEnv (multiagent_env.py:15-216): one world, dicts."""

    metadata = {"render.modes": ["human"]}
    reward_range = (-float("inf"), float("inf"))

    def __init__(self, rules_name, player_names, map_name, agent_ids, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_surroundings_width=21, observation_position_encoding_style="channels",
                 agent_weapons="rifle", debug=False, *, device="cuda", seed=0, env_index_base=0):
        self.vec = MultiagentZombsoleVectorEnv(
            rules_name, player_names, map_name, agent_ids, initial_zombies, minimum_zombies, render_mode,
            observation_surroundings_width, observation_position_encoding_style, agent_weapons, debug,
            num_envs=1, device=device, seed=seed, env_index_base=env_index_base, max_episode_steps=None,
            auto_reset=False, host_outputs=True)
        self.position_encoding_style = observation_position_encoding_style
        self.surroundings_width = observation_surroundings_width
        self.agents = list(agent_ids)
        self.possible_agents = list(agent_ids)
        self.action_spaces = {aid: Dict({"action_type": Text(15),
                                         "parameter": Box(low=-10, high=10, shape=(2,), dtype=np.int32)})
                              for aid in self.possible_agents}
        self.observation_spaces = dict(self.vec.observation_spaces)
        self.render_mode = render_mode
        self.game = self.vec.game(0)

    def get_observation(self):
        obs = self.vec.get_observation()[0].numpy().copy()  # (host memory; the caller gets arrays of its own)
        return {aid: obs[i] for i, aid in enumerate(self.possible_agents) if aid in self.agents}

    def step(self, action):
        # one launch whose outputs land in pinned host memory, one synchronisation (the vector env's host_outputs mode)
        obs, reward, term, trunc, info = self.vec.step([action])
        obs, reward = obs[0].numpy().copy(), reward[0].numpy()
        doneflag, truncatedflag = bool(term[0]), bool(trunc[0])
        before = self.agents
        observations = {aid: obs[i] for i, aid in enumerate(self.possible_agents) if aid in before}
        rewards = {aid: float(reward[i]) for i, aid in enumerate(self.possible_agents) if aid in before}
        done = {aid: doneflag for aid in before}
        truncated = {aid: truncatedflag for aid in before}
        life = self.vec.agent_life_host[0].numpy()
        self.agents = [aid for i, aid in enumerate(self.possible_agents) if life[i] > 0]  # multiagent_env.py:169
        return observations, rewards, done, truncated, {}

    def reset(self, seed=None, options=None):
        self.agents = list(self.possible_agents)
        self.vec.reset()
        return self.get_observation(), {}

    def render(self):
        raise ValueError("mode={} is not supported".format(self.render_mode))

    def close(self):
        self.vec.close()

    def __str__(self):
        return "<{} instance>".format(type(self).__name__)

    def __enter__(self):
        return self

    def __exit__(self, *args):
        self.close()
        return False


class MultiagentZombsoleEnvDiscreteAction(object):
    """Drop-in for the reference's discrete wrapper (multiagent_env.py:258-319): Discrete(7) per agent."""

    game_actions = MultiagentZombsoleVectorEnv.game_actions

    def __init__(self, rules_name, player_names, map_name, agent_ids, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_surroundings_width=21, agent_weapons="rifle", debug=False,
                 **device_kwargs):
        self.env = MultiagentZombsoleEnv(rules_name, player_names, map_name, agent_ids,
                                         initial_zombies=initial_zombies, minimum_zombies=minimum_zombies,
                                         render_mode=render_mode,
                                         observation_surroundings_width=observation_surroundings_width,
                                         agent_weapons=agent_weapons, debug=debug, **device_kwargs)
        self.action_spaces = {aid: Discrete(len(self.game_actions)) for aid in self.env.possible_agents}
        self.observation_spaces = self.env.observation_spaces
        self.reward_range = self.env.reward_range
        self.metadata = self.env.metadata
        self.render_mode = self.env.render_mode

    def step(self, actions):
        return self.env.step(self.actions(actions))

    def reset(self, seed=None, options=None):
        return self.env.reset(seed=seed, options=options)

    def actions(self, actions):
        return {agent_id: self.game_actions[action] for agent_id, action in actions.items()}

    def reverse_actions(self, actions):
        return {agent_id: self.game_actions.index(action) for agent_id, action in actions.items()}

    def close(self):
        self.env.close()
