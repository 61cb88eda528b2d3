"""Single-agent environments: the reference's Gymnasium API over the batched B200 simulator.

Mirrors zombsole/gym_env.py:
  * ``ZombsoleGymEnv`` / ``ZombsoleGymEnvDiscreteAction`` take the reference's constructor
    arguments and return the reference's types (numpy observation ``(C, H, W)`` int32, float
    reward, bool flags) — a drop-in for code written against the reference; one world (num_envs=1).
  * ``ZombsoleVectorEnv`` takes the same arguments plus ``num_envs`` and keeps everything on the
    device: ``step(actions)`` -> ``(obs [N, C, H, W] int32, reward [N] float64, terminated [N] bool,
    truncated [N] bool, info)`` as CUDA tensors, with same-step auto-reset by default.
All randomness comes from the counter-based draw contract (philox.py): a given ``seed`` and global
env index reproduce the reference driven by the same injected draws bit for bit.
"""
import numpy as np
import torch

from . import abi
from .engine import ZsEngine
from .spaces import Box, Dict, Discrete, Text
from .things import Game

try:  # pragma: no cover - depends on the image
    from gymnasium.core import Env as _GymEnv
except ImportError:
    class _GymEnv(object):
        metadata = {}
        spec = None


def _observation_space(engine, cfg):
    """zombsole/gym/observation.py:130-131,141-142,155-156,168-169"""
    c, h, w = engine.obs_shape[-3:]
    high = 8 * 16 * 16 if cfg.obs_encoding == abi.OBS_SIMPLE else 128
    return Box(low=0, high=high, shape=(c, h, w), dtype=np.int32)


def encode_action(action):
    """The reference's action dict -> (type, dx, dy) (players/agent.py:22-96).  A missing or empty
    ``parameter`` is (0, 0), which ``heal`` reads as "self" exactly as the reference does."""
    atype = action.get("action_type", None)
    code = abi.ACTION_TYPES.get(atype, abi.ACT_NONE) if (atype is None or isinstance(atype, str)) else abi.ACT_NONE
    param = action.get("parameter", None)
    if param is None or len(param) == 0:
        dx, dy = 0, 0
        if code in (abi.ACT_MOVE, abi.ACT_ATTACK):
            code = abi.ACT_NONE  # the reference raises inside next_step and the thing idles (core.py:96-99)
    else:
        dx, dy = int(param[0]), int(param[1])
    return code, dx, dy


class CompactHostOutputs(object):
    """What host_outputs="compact" / "compact-copy" share between the vector envs: the record buffers, the streamed step's
    action staging, the full rows of envs a record cannot hold and the resets.  A subclass sets ``obs`` / ``reward`` /
    ``_term`` / ``_trunc`` (host), ``_dev_obs``, ``_overflow``, ``_act_pin`` (discrete ids) / ``_actions_pin`` ((type, dx, dy)
    rows) and provides ``_max_words()``, ``_host_stepper()``, ``_action_rows(dicts)`` and ``_info()``."""

    def _size_records(self, words):
        """(Re)allocate the record buffers: ``words`` 32-bit words per env (header + entries)."""
        words = min(int(words), self._max_words())
        self.compact_words = words
        self._records_host = torch.zeros((self.num_envs, words), dtype=torch.int32).pin_memory()
        self._records_prev = torch.zeros((self.num_envs, words), dtype=torch.int32)
        self._compact_first = True
        self._overflows_since_resize = 0
        if self.streamed:
            torch.cuda.current_stream(self.device).synchronize()  # (nothing in flight still writes the old records)
            self._host_step = self._host_stepper()
            self._host_step_raw = self._host_step.raw
            # (what step() returns never changes: the env's own buffers, the flag bytes as bool views)
            self._step_result = (self.obs, self.reward, self._term.view(torch.bool), self._trunc.view(torch.bool))
        else:
            self._records = torch.zeros((self.num_envs, words), dtype=torch.int32, device=self.device)

    def _step_streamed(self, actions):
        """host_outputs="compact": the actions go over from host memory as they are, the kernel writes the pinned records in
        place (zs_step_host)."""
        n = self._act_pin.numel()  # discrete ids per step
        if isinstance(actions, torch.Tensor) and actions.dtype == torch.int32 and actions.device.type == "cpu" \
                and actions.is_contiguous() and actions.numel() in (n, 3 * n):
            a = actions  # the caller's own buffer, in place: it is free again when step() returns
        elif isinstance(actions, (list, tuple)) and len(actions) and isinstance(actions[0], dict):
            a = self._actions_pin
            a.copy_(torch.from_numpy(self._action_rows(actions)))
        else:
            t = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
            if t.numel() == n:
                a = self._act_pin
            elif t.numel() == 3 * n:
                a = self._actions_pin
            else:
                raise ValueError("actions must hold %d discrete ids or %d (type, dx, dy) rows" % (n, n))
            a.copy_(t.reshape(a.shape))  # (any dtype / device: converted into the env's pinned buffer)
        over = self._host_step_raw(a.data_ptr(), abi.ACTIONS_DISCRETE if a.numel() == n else abi.ACTIONS_FULL, self._compact_first)
        self._compact_first = False
        if over is not None:
            self._fetch_overflow_rows(over)
        return self._step_result + (self._info(),)

    def _fetch_overflow_rows(self, over):
        """Rare: more differing cells than a record holds — those rows come over as they are."""
        stream = torch.cuda.current_stream(self.device)
        stream.synchronize()
        self.compact_overflows += len(over)
        if len(over) > 16:  # many: one gather on the device, one copy
            idx = over.to(self.device, dtype=torch.long)
            self.obs[over.long()] = self._dev_obs[idx].cpu()
        else:
            for e in over.tolist():
                self.obs[e].copy_(self._dev_obs[e], non_blocking=True)
            stream.synchronize()
        # box/wall damage persists across episodes, so the differing cells of long-running envs creep up: when more
        # than one env in 64 no longer fits, or full rows keep being fetched, the records double (up to the size nothing
        # can overflow)
        self._overflows_since_resize += len(over)
        if ((len(over) * 64 > self.num_envs or self._overflows_since_resize > 64)
                and self.compact_words < self._max_words()):
            self._size_records(2 * self.compact_words)

    def _compact_reset(self, mask):
        """(resets are rare next to steps: the full rows come over, and the next step starts afresh)"""
        self.engine.reset(mask, self._dev_obs)
        if mask is None:
            self.obs.copy_(self._dev_obs, non_blocking=True)
        else:
            sel = torch.as_tensor(mask).to(torch.bool).cpu()
            self.obs[sel] = self._dev_obs.cpu()[sel]
        torch.cuda.current_stream(self.device).synchronize()
        self._compact_first = True
        return self.obs, {}


def check_final_observation(final_observation, auto_reset, host_outputs):
    """The argument combinations final_observation=True cannot serve."""
    if not final_observation:
        return
    if not auto_reset:
        raise ValueError("final_observation=True needs auto_reset=True: without auto-reset step() returns the final "
                         "observation itself")
    if host_outputs in ("compact", "compact-copy"):
        raise ValueError("final_observation=True is not available with host_outputs=%r" % (host_outputs,))


class FinalObservation(object):
    """final_observation=True (gymnasium's SAME_STEP autoreset): an env whose step ends its episode is re-initialised in the
    same step and ``obs`` shows the new episode; the observation of the world it ended in goes to ``final_obs`` (shaped like
    ``obs``, written by the step kernel in place, also into pinned host memory) and step()'s info carries it as
    ``"final_obs"`` with the mask ``"_final_obs"`` (bool [N] = terminated | truncated).  Rows outside the mask are
    unspecified."""

    def __init__(self, final_observation):
        self.final_observation = bool(final_observation)
        if self.final_observation:
            if self.host_outputs:
                self.final_obs = torch.empty(self.obs.shape, dtype=torch.int32).pin_memory()
            else:
                self.final_obs = self.engine.new_obs()
            self._final_mask = torch.zeros(self.num_envs, dtype=torch.bool, device=self._term.device)
            if self._term.is_pinned():
                self._final_mask = self._final_mask.pin_memory()

    def _final_info(self, info):
        torch.logical_or(self._term, self._trunc, out=self._final_mask)
        info["final_obs"] = self.final_obs
        info["_final_obs"] = self._final_mask
        return info


def _next_step_mode():
    """gymnasium's AutoresetMode.NEXT_STEP where gymnasium has it, else its value."""
    try:
        from gymnasium.vector import AutoresetMode
        return AutoresetMode.NEXT_STEP
    except ImportError:
        return "next_step"


class NextStepAutoreset(object):
    """autoreset_mode="next_step" (gymnasium's AutoresetMode.NEXT_STEP; include/zs_b200.h: ZS_AUTORESET_NEXT_STEP): the step
    that ends an episode returns its terminal observation, reward and flags and leaves the world as it is; the env's next
    step ignores its action, re-initialises the world and returns the new episode's first observation with reward 0 and
    both flags false.  Works with every host_outputs value.  ``metadata["autoreset_mode"]`` says so (an instance copy);
    ``autoreset_envs`` (bool [N] on the device, read-only) marks the envs whose next step is such a reset step."""

    def __init__(self, autoreset_mode):
        self.autoreset_mode = autoreset_mode
        if autoreset_mode == "next_step":
            self.metadata = dict(type(self).metadata, autoreset_mode=_next_step_mode())

    @property
    def autoreset_envs(self):
        return self.engine.autoreset_pending()


class ZombsoleVectorEnv(CompactHostOutputs, FinalObservation, NextStepAutoreset):
    """``num_envs`` independent ZombsoleGymEnv worlds on one GPU (constructor: gym_env.py:49-53)."""

    metadata = {"render.modes": ["human"]}
    reward_range = (-float("inf"), float("inf"))
    game_actions = [
        {"action_type": "move", "parameter": [0, 1]},
        {"action_type": "move", "parameter": [-1, 0]},
        {"action_type": "move", "parameter": [0, -1]},
        {"action_type": "move", "parameter": [1, 0]},
        {"action_type": "attack_closest"},
        {"action_type": "heal"},
    ]

    def __init__(self, rules_name, player_names, map_name, agent_id, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_scope="world", observation_position_encoding="simple",
                 agent_weapon="rifle", debug=False, *, num_envs=1, device="cuda", seed=0, env_index_base=0,
                 max_episode_steps=None, auto_reset=True, host_outputs=False, host_threads=0, compact_words=0,
                 final_observation=False, autoreset_mode="same_step"):
        if render_mode is not None:
            if render_mode not in self.metadata["render.modes"]:
                raise ValueError("render_mode={} is not supported".format(render_mode))
            raise NotImplementedError("rendering is outside the batched simulator's scope (render_mode=None only)")
        self.render_mode = None
        check_final_observation(final_observation, auto_reset, host_outputs)
        abi.check_autoreset_mode(autoreset_mode, auto_reset, final_observation)
        scope, enc, width = abi.parse_observation_scope(observation_scope, observation_position_encoding)
        self.cfg = abi.make_config(rules_name, list(player_names), [agent_id], [agent_weapon], initial_zombies,
                                   minimum_zombies, scope, enc, width, False, num_envs, seed=seed,
                                   env_index_base=env_index_base, max_episode_steps=max_episode_steps,
                                   auto_reset=auto_reset, autoreset_mode=autoreset_mode)
        self.engine = ZsEngine(self.cfg, map_name, device=device)
        self.num_envs = num_envs
        self.device = self.engine.device
        self.debug = debug
        self._ctor = (rules_name, list(player_names), [agent_id], initial_zombies, minimum_zombies)
        self.single_observation_space = _observation_space(self.engine, self.cfg)
        self.observation_space = self.single_observation_space
        self.single_action_space = Discrete(len(self.game_actions))
        self.action_space = self.single_action_space
        # host_outputs: step() returns tensors in pinned host memory that the kernel wrote directly (zero-copy over
        # PCIe, overlapped with the transition) and has synchronised on — for loops whose policy runs on the host
        # host_outputs="compact": the same host tensors, but what crosses PCIe every step is one small record per env
        # (the cells that differ from the map's pristine layer, the reward, the flags: about 0.5 KB instead of the
        # 5-16 KB observation row) which a threaded host routine of the library expands in place into the env's host
        # observation tensor — byte-identical results.  "compact" is ONE library call per step: the kernel writes the pinned
        # records itself and the host threads, already waiting, expand them the moment a flag kernel behind it says they
        # are complete (zs_step_host); "compact-copy" is the same with explicit copies and a stream
        # synchronisation between the stages (zs_step_compact / zs_expand_compact, include/zs_b200.h)
        if isinstance(host_outputs, str) and host_outputs not in ("compact", "compact-copy", "compact-if-available"):
            raise ValueError("host_outputs must be False, True, 'compact', 'compact-copy' or 'compact-if-available'")
        if host_outputs == "compact-if-available":  # (device outputs where the configuration has no compact record form)
            host_outputs = "compact" if self.engine.compact_words() and not final_observation else False
        self.compact = host_outputs in ("compact", "compact-copy")
        self.streamed = host_outputs == "compact"
        self.host_outputs = bool(host_outputs)
        self.host_threads = int(host_threads)
        if self.compact:
            words = self.engine.compact_words()
            if not words:
                raise ValueError("host_outputs='compact' needs a world-scope observation")
            self.obs, self.reward, self._term, self._trunc = self.engine.new_host_outputs()
            self._dev_obs = self.engine.new_obs()  # full rows of the rare envs a record cannot hold
            self._overflow = torch.zeros(num_envs, dtype=torch.int32)
            self.compact_overflows = 0
            self._act_pin = torch.zeros((num_envs, 1), dtype=torch.int32).pin_memory()
            self._actions_pin = torch.zeros((num_envs, 1, 3), dtype=torch.int32).pin_memory()
            self._size_records(int(compact_words) if compact_words else words)
        elif self.host_outputs:
            self.obs, self.reward, self._term, self._trunc = self.engine.new_host_outputs()
        else:
            self.obs = self.engine.new_obs()
            self.reward, self._term, self._trunc = self.engine.new_outputs()
        self._actions = torch.zeros((num_envs, 1, 3), dtype=torch.int32, device=self.device)
        self._act_dev = torch.zeros((num_envs, 1), dtype=torch.int32, device=self.device)
        self._h2d_done, self._h2d_pending = None, False
        FinalObservation.__init__(self, final_observation)
        NextStepAutoreset.__init__(self, autoreset_mode)

    # -- the reference's object protocol for one world of the batch
    def game(self, env=0):
        rules_name, player_names, agent_ids, iz, mz = self._ctor
        return Game(self.engine, env, rules_name, player_names, agent_ids, iz, mz)

    def get_observation(self):
        self.engine.encode_obs(self.obs)
        if self.host_outputs:  # (pinned host tensor written by the kernel: the host owns it when this returns)
            torch.cuda.current_stream(self.device).synchronize()
        if self.compact:
            self._compact_first = True  # the rows are complete again: the next step's records start from scratch
        return self.obs

    def get_frame_size(self):
        return tuple(self.observation_space.shape[1:3])

    def _stage_actions(self, actions):
        """-> (device int32 tensor, format).  Accepts discrete ids [N], (type, dx, dy) rows [N, 3],
        or a list of N reference action dicts."""
        if isinstance(actions, (list, tuple)) and len(actions) and isinstance(actions[0], dict):
            rows = np.array([encode_action(a) for a in actions], dtype=np.int32).reshape(self.num_envs, 1, 3)
            self._actions.copy_(torch.from_numpy(rows), non_blocking=True)
            return self._actions, abi.ACTIONS_FULL
        t = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions))
        if self.compact and t.dtype == torch.int32 and t.device.type == "cpu" and t.numel() == self.num_envs:
            # the host loop's hot path: one copy into the env's own device buffer; step() synchronises the stream before it
            # returns, so the caller's buffer is free again by then
            self._act_dev.copy_(t.view(self.num_envs, 1), non_blocking=True)
            return self._act_dev, abi.ACTIONS_DISCRETE
        if self.host_outputs and not self.compact and t.dtype == torch.int32 and t.device.type == "cpu" and t.is_pinned():
            pass  # the kernel reads a pinned host action tensor in place
        elif t.dtype != torch.int32 or t.device != self.device:
            pinned_src = t.device.type == "cpu" and t.is_pinned()
            t = t.to(device=self.device, dtype=torch.int32, non_blocking=True)
            if pinned_src:  # the copy is in flight: step() waits for it before the caller may refill the buffer
                self._h2d_done = self._h2d_done or torch.cuda.Event()
                self._h2d_done.record(torch.cuda.current_stream(self.device))
                self._h2d_pending = True
        t = t.contiguous()
        if t.numel() == self.num_envs:
            return t.view(self.num_envs, 1), abi.ACTIONS_DISCRETE
        if t.numel() == 3 * self.num_envs:
            return t.view(self.num_envs, 1, 3), abi.ACTIONS_FULL
        raise ValueError("actions must hold %d discrete ids or %d (type, dx, dy) rows" % (self.num_envs, self.num_envs))

    def step(self, actions):
        """One transition of every world (gym_env.py:99-145).  The returned tensors are the env's own
        output buffers: they are overwritten by the next call."""
        if self.compact and self.streamed:
            return self._step_streamed(actions)
        a, fmt = self._stage_actions(actions)
        if self.compact:
            return self._step_compact(a, fmt)
        if self.final_observation:
            self.engine.step_final(a, fmt, self.obs, self.final_obs, self.reward, self._term, self._trunc)
        else:
            self.engine.step(a, fmt, self.obs, self.reward, self._term, self._trunc)
        if self._h2d_pending:  # a pinned host action buffer is the caller's again when step() returns
            self._h2d_done.synchronize()
            self._h2d_pending = False
        if self.host_outputs:
            torch.cuda.current_stream(self.device).synchronize()  # the host owns the results when step() returns
        info = self._final_info({}) if self.final_observation else {}
        return self.obs, self.reward, self._term.view(torch.bool), self._trunc.view(torch.bool), info  # (0/1 bytes: a view, no kernel)

    # (CompactHostOutputs)
    def _max_words(self):
        return self.engine.compact_max_words()

    def _host_stepper(self):
        return self.engine.host_stepper(self._records_host, self._records_prev, self._dev_obs, self.obs, self.reward, self._term,
                                        self._trunc, self._overflow, self.host_threads)

    def _action_rows(self, actions):
        return np.array([encode_action(x) for x in actions], dtype=np.int32).reshape(self.num_envs, 1, 3)

    def _info(self):
        return {}

    def _step_compact(self, a, fmt):
        eng = self.engine
        eng.step_compact(a, fmt, self._records, self._dev_obs)
        self._records_host.copy_(self._records, non_blocking=True)
        stream = torch.cuda.current_stream(self.device)
        stream.synchronize()
        self._h2d_pending = False
        over = eng.expand_compact(self._records_host, self._records_prev, self.obs, self.reward, self._term, self._trunc,
                                  self._overflow, self._compact_first, self.host_threads)
        self._compact_first = False
        if len(over):
            self._fetch_overflow_rows(over)
        return self.obs, self.reward, self._term.view(torch.bool), self._trunc.view(torch.bool), {}

    def reset(self, seed=None, options=None, mask=None):
        """Re-initialise every world (or those selected by ``mask``); gym_env.py:148-164.  ``seed`` is
        accepted for API compatibility and ignored, as in the reference (it only seeds gymnasium's unused
        np_random): the draw stream is fixed by the constructor's ``seed``."""
        if self.compact:
            return self._compact_reset(mask)
        self.engine.reset(mask, self.obs)
        if self.host_outputs:
            torch.cuda.current_stream(self.device).synchronize()
        return self.obs, {}

    def rollout(self, n_steps, actions=None, first_step_index=0, obs=None, reward=None, terminated=None, truncated=None,
                final_obs=None):
        """``n_steps`` transitions in one kernel launch with same-step auto-reset (next-step with autoreset_mode="next_step").  ``actions`` is an int32
        tensor [n_steps, N] of discrete ids or None for the synthetic uniform stream.  ``final_obs``: a ring shaped like
        ``obs`` (or like the env's observation when ``obs`` is None) that receives, in step i's slot, the observation each env
        whose episode step i ended had before it was re-initialised (the rows where terminated | truncated)."""
        fmt = abi.ACTIONS_DISCRETE
        if actions is not None and actions.dim() == 3 and actions.shape[-1] == 3:
            fmt = abi.ACTIONS_FULL
        self.engine.rollout(n_steps, first_step_index, actions, fmt, self.obs if obs is None else obs, reward,
                            terminated, truncated, final_obs=final_obs)
        return self.obs if obs is None else obs

    def render(self):
        raise ValueError("mode={} is not supported".format(self.render_mode))

    def render_text(self, env=0, use_basic_icons=True):
        """Text frame of world ``env`` laid out like the reference's terminal renderer (renderer.py:45-88); debugging aid."""
        return self.game(env).draw_text(use_basic_icons)

    def render_image(self, env=0, with_text=True):
        """RGB frame (uint8 [height, width, 3]) of world ``env`` with the geometry and shapes of the reference's OpenCV
        renderer (renderer.py:97-277); debugging aid."""
        return self.game(env).draw_image(with_text)

    def close(self):
        self.engine.close()

    def __enter__(self):
        return self

    def __exit__(self, *args):
        self.close()
        return False


class ZombsoleGymEnv(_GymEnv):
    """Drop-in for the reference's ZombsoleGymEnv (gym_env.py:16-240): one world, numpy/python outputs."""

    metadata = {"render.modes": ["human"]}
    reward_range = (-float("inf"), float("inf"))
    action_space = Dict({"action_type": Text(15), "parameter": Box(low=-10, high=10, shape=(2,), dtype=np.int32)})

    def __init__(self, rules_name, player_names, map_name, agent_id, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_scope="world", observation_position_encoding="simple",
                 agent_weapon="rifle", debug=False, *, device="cuda", seed=0, env_index_base=0):
        kw = dict(num_envs=1, device=device, seed=seed, env_index_base=env_index_base, max_episode_steps=None, auto_reset=False)
        args = (rules_name, player_names, map_name, agent_id, initial_zombies, minimum_zombies, render_mode, observation_scope,
                observation_position_encoding, agent_weapon, debug)
        # one world answers a host caller: where the configuration has a compact record form the whole step is ONE library
        # call that leaves observation, reward and flags in host memory (zs_step_host) instead of a launch and four copies
        self.vec = ZombsoleVectorEnv(*args, host_outputs="compact-if-available", host_threads=1, **kw)
        self.render_mode = render_mode
        self.observation_space = self.vec.single_observation_space
        self.game = self.vec.game(0)

    @staticmethod
    def _fresh(row):
        """The caller gets an array of its own, as from the reference (the env's buffers are overwritten by the next call)."""
        return row.cpu().numpy() if row.is_cuda else row.numpy().copy()

    def get_observation(self):
        return self._fresh(self.vec.get_observation()[0])

    def get_frame_size(self):
        return self.vec.get_frame_size()

    def step(self, action):
        obs, reward, terminated, truncated, info = self.vec.step([action])
        return (self._fresh(obs[0]), float(reward[0].item()), bool(terminated[0].item()), bool(truncated[0].item()), {})

    def reset(self, seed=None, options=None):
        obs, _ = self.vec.reset()
        return self._fresh(obs[0]), {}

    def render(self):
        raise ValueError("mode={} is not supported".format(self.render_mode))

    def close(self):
        self.vec.close()

    @property
    def unwrapped(self):
        return self

    def __str__(self):
        return "<{} instance>".format(type(self).__name__)

    def __enter__(self):
        return self

    def __exit__(self, *args):
        self.close()
        return False


class ZombsoleGymEnvDiscreteAction(object):
    """Drop-in for the reference's discrete-action wrapper (gym_env.py:327-379): Discrete(6)."""

    game_actions = ZombsoleVectorEnv.game_actions

    def __init__(self, rules_name, player_names, map_name, agent_id, initial_zombies=0, minimum_zombies=0,
                 render_mode=None, observation_scope="world", observation_position_encoding="simple", debug=False,
                 **device_kwargs):
        self.env = ZombsoleGymEnv(rules_name, player_names, map_name, agent_id, initial_zombies=initial_zombies,
                                  minimum_zombies=minimum_zombies, render_mode=render_mode,
                                  observation_scope=observation_scope,
                                  observation_position_encoding=observation_position_encoding, debug=debug,
                                  **device_kwargs)
        self.action_space = Discrete(len(self.game_actions))
        self.observation_space = self.env.observation_space
        self.reward_range = self.env.reward_range
        self.metadata = self.env.metadata
        self.render_mode = self.env.render_mode

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError("attempted to get missing private attribute '{}'".format(name))
        return getattr(self.env, name)

    def reset(self, **kwargs):
        return self.env.reset(**kwargs)

    def step(self, action):
        return self.env.step(self.action(action))

    def action(self, action):
        return self.game_actions[action]

    def reverse_action(self, action):
        return self.game_actions.index(action)

    def close(self):
        return self.env.close()

    @property
    def unwrapped(self):
        return self.env.unwrapped


#: the ids the reference registers with gymnasium (gym_env.py:382-414) and their kwargs
REGISTERED = {
    "jvstinian/Zombsole-v0": dict(rules_name="extermination", player_names=[], map_name="bridge", agent_id=0,
                                  initial_zombies=10, minimum_zombies=0, debug=False),
    "jvstinian/Zombsole-SurroundingsView-v0": dict(rules_name="extermination", player_names=[], map_name="bridge",
                                                   agent_id=0, initial_zombies=10, minimum_zombies=0,
                                                   observation_scope="surroundings:21",
                                                   observation_position_encoding="simple", debug=False),
}
MAX_EPISODE_STEPS = 1000


def make_vector(env_id, num_envs, **overrides):
    """Batched equivalent of ``gym.make(env_id)``: the registered kwargs, TimeLimit(1000) included."""
    kwargs = dict(REGISTERED[env_id])
    kwargs.update(overrides)
    kwargs.setdefault("max_episode_steps", MAX_EPISODE_STEPS)
    return ZombsoleVectorEnv(num_envs=num_envs, **kwargs)


try:  # pragma: no cover - only when gymnasium is installed
    from gymnasium.envs.registration import register as _register
    for _id, _kw in REGISTERED.items():
        _register(id=_id.replace("jvstinian/", "jvstinian/B200-"),
                  entry_point="libzombsole_b200.gym_env:ZombsoleGymEnvDiscreteAction",
                  max_episode_steps=MAX_EPISODE_STEPS, nondeterministic=False, kwargs=_kw)
except ImportError:
    pass
