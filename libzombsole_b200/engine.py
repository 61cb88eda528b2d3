"""ZsEngine: N worlds resident in HBM, driven through the C ABI (include/zs_b200.h).

PyTorch is the plumbing here — it owns the device memory (state buffer, action / observation /
reward tensors) and the stream; every transition is computed by the hand-written sm_100a
kernels in csrc/.
"""
import ctypes as C

import numpy as np
import torch

from . import abi
from ._native import lib, check, ZsError

_TORCH_DTYPES = {np.int16: torch.int16, np.int32: torch.int32, np.uint8: torch.uint8, np.uint32: torch.int32}


def _ptr(t):
    return None if t is None else t.data_ptr()


# (torch.cuda.current_stream() builds a Stream object per call: 1.5 us on the step path; the raw accessor is 0.2 us)
_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)

class ZsEngine(object):
    def __init__(self, cfg, map_, device="cuda"):
        if not torch.cuda.is_available():
            raise ZsError("no CUDA device: the batched zombsole simulator has no CPU path")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ZsError("device must be a CUDA device, got %r" % (device,))
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.L = lib()
        self.cfg = cfg
        self.map_arg = abi.MapArg(abi.resolve_map(map_))
        self.map = self.map_arg.map
        self.layout = abi.ZsLayout()
        check(self.L.zs_layout(C.byref(cfg), C.byref(self.map_arg.struct), C.byref(self.layout)))
        self.N = cfg.num_envs
        self.A = cfg.n_agents
        self.P = cfg.n_bots
        self.M = self.layout.n_slots
        self.S = len(self.map.statics)
        self.cells = self.layout.cells
        self.obs_elems = int(self.layout.obs_elems_per_env)
        self.per_agent = bool(cfg.obs_per_agent)
        self.R = self.A if self.per_agent else 1
        lay = self.layout
        if self.per_agent:
            self.obs_shape = (self.A, lay.obs_channels, lay.obs_height, lay.obs_width)
        else:
            self.obs_shape = (lay.obs_channels, lay.obs_height, lay.obs_width)
        self.n_discrete_actions = lay.n_discrete_actions
        self.h = C.c_void_p()
        with torch.cuda.device(self.device):
            torch.cuda.current_stream()  # make sure the primary context exists
            check(self.L.zs_set_device(self.device.index))
            check(self.L.zs_create(C.byref(cfg), C.byref(self.map_arg.struct), C.byref(self.h)))
            self.state = torch.zeros(int(lay.state_bytes), dtype=torch.uint8, device=self.device)
            check(self.L.zs_bind_state(self.h, self.state.data_ptr(), int(lay.state_bytes)))
            check(self.L.zs_init_static_life(self.h, self._stream()))
        self.fields = {}
        for f, name in abi.FIELD_NAMES.items():
            dt = abi.FIELD_DTYPES[f]
            nbytes = lay.row_bytes[f] * self.N
            flat = self.state[lay.offset[f]: lay.offset[f] + nbytes]
            self.fields[name] = flat.view(_TORCH_DTYPES[dt]).view(self.N, -1)
        self.reset_draws = torch.zeros(self.N, dtype=torch.int32, device=self.device)
        self.reset()  # world initialisation #0: what the reference's constructor does (game.py:138)

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        """The caller's current stream on this engine's device, as the raw handle the C ABI takes."""
        if _RAW_STREAM is not None:
            return _RAW_STREAM(self.device.index)
        return torch.cuda.current_stream(self.device).cuda_stream

    def state_written(self):
        """Call after writing into ``fields`` (the views are the live state buffer): the engine keeps a parked on-chip
        image of every env next to the state and starts launches from it; this marks the images stale, so the next
        launch re-derives everything from the state buffer (zs_state_written)."""
        check(self.L.zs_state_written(self.h))

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.L.zs_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def new_obs(self, slots=None):
        shape = (self.N,) + self.obs_shape if slots is None else (slots, self.N) + self.obs_shape
        return torch.empty(shape, dtype=torch.int32, device=self.device)

    def new_outputs(self, steps=None):
        lead = (self.N,) if steps is None else (steps, self.N)
        rshape = lead + ((self.A,) if self.per_agent else ())
        return (torch.empty(rshape, dtype=torch.float64, device=self.device),
                torch.empty(lead, dtype=torch.uint8, device=self.device),
                torch.empty(lead, dtype=torch.uint8, device=self.device))

    def new_host_outputs(self):
        """Observation / reward / flag buffers in PINNED HOST memory.  Under unified addressing the device reaches
        pinned host memory at the same address, so the step kernel can write its outputs there directly (the
        device-to-host transfer happens inside the kernel, overlapped with the transition, instead of as separate
        copies afterwards)."""
        rshape = (self.N,) + ((self.A,) if self.per_agent else ())
        return (torch.empty((self.N,) + self.obs_shape, dtype=torch.int32).pin_memory(),
                torch.empty(rshape, dtype=torch.float64).pin_memory(),
                torch.empty((self.N,), dtype=torch.uint8).pin_memory(),
                torch.empty((self.N,), dtype=torch.uint8).pin_memory())

    # ------------------------------------------------------------------ the ABI boundary: what the kernels may be handed
    _FLAG_DTYPES = (torch.uint8, torch.bool)

    def _arg(self, t, dtypes, numel, name):
        """Pointer of a tensor argument after checking that the kernels can take it as it is: on this engine's device
        (or pinned host memory, which the device reaches at the same address), the right element type, contiguous, and
        at least as large as what the launch reads or writes.  The C ABI sees raw pointers; a wrong tensor would be
        misread or overrun."""
        if t is None:
            return None
        if not isinstance(t, torch.Tensor):
            raise ValueError("%s must be a torch tensor, got %s" % (name, type(t).__name__))
        if not isinstance(dtypes, tuple):
            dtypes = (dtypes,)
        if t.dtype not in dtypes:
            raise ValueError("%s must be %s, got %s" % (name, " or ".join(str(d) for d in dtypes), t.dtype))
        if t.device != self.device and not (t.device.type == "cpu" and t.is_pinned()):
            raise ValueError("%s must live on %s (or in pinned host memory), got %s" % (name, self.device, t.device))
        if not t.is_contiguous():
            raise ValueError("%s must be contiguous" % name)
        if t.numel() < numel:
            raise ValueError("%s must hold at least %d elements, got %d (shape %s)" % (name, numel, t.numel(), tuple(t.shape)))
        return t.data_ptr()

    def _action_arg(self, actions, fmt, n_steps):
        if fmt not in (abi.ACTIONS_DISCRETE, abi.ACTIONS_FULL):
            raise ValueError("bad action format %r" % (fmt,))
        per = 3 if fmt == abi.ACTIONS_FULL else 1
        return self._arg(actions, torch.int32, n_steps * self.N * self.A * per, "actions")

    # ------------------------------------------------------------------ the ABI calls
    def reset(self, mask=None, obs=None):
        """zs_reset: re-initialise the masked worlds (all if mask is None)."""
        if mask is not None:
            mask = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        check(self.L.zs_reset(self.h, self._arg(mask, torch.uint8, self.N, "mask"),
                              self._arg(obs, torch.int32, self.N * self.obs_elems, "obs"), _ptr(self.reset_draws),
                              self._stream()))
        return obs

    def step(self, actions, fmt, obs, reward, terminated, truncated, agent_mask=None, draws=None):
        N = self.N
        check(self.L.zs_step(self.h, self._action_arg(actions, fmt, 1), fmt,
                             self._arg(obs, torch.int32, N * self.obs_elems, "obs"),
                             self._arg(reward, torch.float64, N * self.R, "reward"),
                             self._arg(terminated, self._FLAG_DTYPES, N, "terminated"),
                             self._arg(truncated, self._FLAG_DTYPES, N, "truncated"),
                             self._arg(agent_mask, self._FLAG_DTYPES, N * self.A, "agent_mask"),
                             self._arg(draws, torch.int32, N, "draws"), self._stream()))

    def step_final(self, actions, fmt, obs, final_obs, reward, terminated, truncated, agent_mask=None, draws=None):
        """zs_step_final: ``step`` that also writes, for every env whose episode the step ends (and re-initialises), the
        observation of the world it ended in to its row of ``final_obs`` (shaped like ``obs``); the other rows are
        unspecified.  Needs an engine built with auto_reset."""
        N = self.N
        check(self.L.zs_step_final(self.h, self._action_arg(actions, fmt, 1), fmt,
                                   self._arg(obs, torch.int32, N * self.obs_elems, "obs"),
                                   self._arg(final_obs, torch.int32, N * self.obs_elems, "final_obs"),
                                   self._arg(reward, torch.float64, N * self.R, "reward"),
                                   self._arg(terminated, self._FLAG_DTYPES, N, "terminated"),
                                   self._arg(truncated, self._FLAG_DTYPES, N, "truncated"),
                                   self._arg(agent_mask, self._FLAG_DTYPES, N * self.A, "agent_mask"),
                                   self._arg(draws, torch.int32, N, "draws"), self._stream()))

    def step_masked(self, mask, actions, fmt, obs, reward, terminated, truncated, agent_mask=None):
        """zs_step_masked: one transition of the worlds selected by ``mask`` (uint8 [N]); the others are not touched."""
        N = self.N
        mask = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        check(self.L.zs_step_masked(self.h, self._arg(mask, torch.uint8, N, "mask"), self._action_arg(actions, fmt, 1), fmt,
                                    self._arg(obs, torch.int32, N * self.obs_elems, "obs"),
                                    self._arg(reward, torch.float64, N * self.R, "reward"),
                                    self._arg(terminated, self._FLAG_DTYPES, N, "terminated"),
                                    self._arg(truncated, self._FLAG_DTYPES, N, "truncated"),
                                    self._arg(agent_mask, self._FLAG_DTYPES, N * self.A, "agent_mask"), self._stream()))

    # ---- compact host outputs (include/zs_b200.h: zs_step_compact / zs_expand_compact)
    def compact_words(self):
        """Words per compact observation record, 0 if this configuration has no compact form."""
        return int(self.L.zs_compact_words(self.h))

    def compact_max_words(self):
        return int(self.L.zs_compact_max_words(self.h))

    def step_compact(self, actions, fmt, records, obs=None):
        """One transition whose observation / reward / flags come out as one small record per env (device tensor
        ``records`` int32 [N, words]); ``obs`` receives the full row of the rare env a record cannot hold."""
        words = int(records.shape[-1])
        check(self.L.zs_step_compact(self.h, self._action_arg(actions, fmt, 1), fmt,
                                     self._arg(records, torch.int32, self.N * words, "records"), words,
                                     self._arg(obs, torch.int32, self.N * self.obs_elems, "obs"), self._stream()))

    def expand_compact(self, records_host, prev_host, obs_host, reward_host, term_host, trunc_host, overflow_host,
                       first_call, n_threads=0):
        """HOST side: records (already copied to host memory) -> the reference's observation tensor, reward, flags.
        Returns the indices of the envs whose rows must be fetched from the device observation tensor."""
        n_over = C.c_int32(0)
        check(self.L.zs_expand_compact(self.h, records_host.data_ptr(), prev_host.data_ptr(), obs_host.data_ptr(),
                                       reward_host.data_ptr(), term_host.data_ptr(), trunc_host.data_ptr(),
                                       overflow_host.data_ptr(), C.addressof(n_over), int(records_host.shape[-1]),
                                       1 if first_call else 0, int(n_threads)))
        return overflow_host[:n_over.value]

    def host_stepper(self, records, prev_host, obs_dev, obs_host, reward_host, term_host, trunc_host, overflow_host, n_threads=0,
                     agent_mask_host=None, agent_life_host=None):
        """zs_step_host bound to one set of buffers: ``step(actions, fmt, first_call)`` runs one transition whose actions
        come from host memory and whose records are written to pinned host memory by the kernel itself, the host
        threads expanding each env as its record arrives.  Returns the envs whose rows must be fetched from ``obs_dev``, or None.
        With ``agent_mask_host`` (uint8 [N, A]) and ``agent_life_host`` (int16 [N, A]) it is zs_step_host_agents: per-agent
        surroundings records, rewards [N, A]."""
        words = int(records.shape[-1])
        for name, t in (("records", records),):
            if not (t.device.type == "cpu" and t.is_pinned()):
                raise ValueError("%s must be pinned host memory" % name)
        N, agents = self.N, agent_mask_host is not None or agent_life_host is not None
        ptrs = (self._arg(records, torch.int32, N * words, "records"), self._host_arg(prev_host, torch.int32, N * words, "prev"), words,
                self._arg(obs_dev, torch.int32, N * self.obs_elems, "obs_dev"),
                self._host_arg(obs_host, torch.int32, N * self.obs_elems, "obs_host"),
                self._host_arg(reward_host, torch.float64, N * self.R, "reward"), self._host_arg(term_host, self._FLAG_DTYPES, N, "terminated"),
                self._host_arg(trunc_host, self._FLAG_DTYPES, N, "truncated"), self._host_arg(overflow_host, torch.int32, N, "overflow"))
        n_over = C.c_int32(0)
        n_over_p = C.addressof(n_over)
        call, h, A, nthr = self.L.zs_step_host, self.h, self.A, int(n_threads)
        keep = (records, prev_host, obs_dev, obs_host, reward_host, term_host, trunc_host, overflow_host, n_over,
                agent_mask_host, agent_life_host)

        stream_of = self._stream

        if agents:
            call = self.L.zs_step_host_agents
            mask_p = self._host_arg(agent_mask_host, self._FLAG_DTYPES, N * A, "agent_mask")
            life_p = self._host_arg(agent_life_host, torch.int16, N * A, "agent_life")

            def raw(actions_ptr, fmt, first_call):
                """(no checks: ``actions_ptr`` addresses N * A (* 3) int32 in host memory)"""
                rc = call(h, actions_ptr, fmt, ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], ptrs[6], ptrs[7], mask_p, life_p,
                          ptrs[8], n_over_p, 1 if first_call else 0, nthr, stream_of())
                if rc:
                    check(rc)
                return overflow_host[:n_over.value] if n_over.value else None
        else:
            def raw(actions_ptr, fmt, first_call):
                """(no checks: ``actions_ptr`` addresses N * A (* 3) int32 in host memory)"""
                rc = call(h, actions_ptr, fmt, ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], ptrs[6], ptrs[7], ptrs[8],
                          n_over_p, 1 if first_call else 0, nthr, stream_of())
                if rc:
                    check(rc)
                return overflow_host[:n_over.value] if n_over.value else None

        def step(actions, fmt, first_call):
            per = 3 if fmt == abi.ACTIONS_FULL else 1
            if (not isinstance(actions, torch.Tensor) or actions.dtype != torch.int32 or actions.device.type != "cpu"
                    or not actions.is_contiguous() or actions.numel() < N * A * per):
                raise ValueError("actions must be a contiguous int32 host tensor of %d elements" % (N * A * per))
            return raw(actions.data_ptr(), fmt, first_call)
        step.raw = raw
        step.keep = keep
        return step

    # ---- compact host outputs for per-agent surroundings observations (include/zs_b200.h: zs_step_compact_agents)
    def agent_compact_words(self):
        """Words per per-agent compact record, 0 if this configuration has no such form."""
        return int(self.L.zs_agent_compact_words(self.h))

    def agent_compact_max_words(self):
        return int(self.L.zs_agent_compact_max_words(self.h))

    def step_compact_agents(self, actions, fmt, records, obs=None):
        """One transition whose per-agent windows, rewards, agent mask, lives and flags come out as one small record per env
        (device tensor ``records`` int32 [N, words]); ``obs`` receives the full rows of the rare env a record cannot hold."""
        words = int(records.shape[-1])
        check(self.L.zs_step_compact_agents(self.h, self._action_arg(actions, fmt, 1), fmt,
                                            self._arg(records, torch.int32, self.N * words, "records"), words,
                                            self._arg(obs, torch.int32, self.N * self.obs_elems, "obs"), self._stream()))

    def expand_compact_agents(self, records_host, prev_host, obs_host, reward_host, term_host, trunc_host, mask_host, life_host,
                              overflow_host, first_call, n_threads=0):
        """HOST side: per-agent records (already in host memory) -> observation [N, A, C, w, w], reward [N, A], flags, agent
        mask [N, A] and lives [N, A].  Returns the indices of the envs whose rows must be fetched from the device."""
        N, A, words = self.N, self.A, int(records_host.shape[-1])
        n_over = C.c_int32(0)
        check(self.L.zs_expand_compact_agents(
            self.h, self._host_arg(records_host, torch.int32, N * words, "records"),
            self._host_arg(prev_host, torch.int32, N * words, "prev"),
            self._host_arg(obs_host, torch.int32, N * self.obs_elems, "obs_host"),
            self._host_arg(reward_host, torch.float64, N * self.R, "reward"),
            self._host_arg(term_host, self._FLAG_DTYPES, N, "terminated"), self._host_arg(trunc_host, self._FLAG_DTYPES, N, "truncated"),
            self._host_arg(mask_host, self._FLAG_DTYPES, N * A, "agent_mask"), self._host_arg(life_host, torch.int16, N * A, "agent_life"),
            self._host_arg(overflow_host, torch.int32, N, "overflow"), C.addressof(n_over), words, 1 if first_call else 0,
            int(n_threads)))
        return overflow_host[:n_over.value]

    def step_host_stats(self):
        """(calls, mean us from entry to: launches issued, previous cells restored, flag seen = records in host memory,
        return) since the last read."""
        out = (C.c_double * 5)()
        check(self.L.zs_step_host_stats(self.h, out))
        return tuple(out)

    def _host_arg(self, t, dtypes, numel, name):
        """Pointer of a HOST tensor argument (read or written by the library's host threads)."""
        if not isinstance(dtypes, tuple):
            dtypes = (dtypes,)
        if not isinstance(t, torch.Tensor) or t.device.type != "cpu" or t.dtype not in dtypes or not t.is_contiguous() or t.numel() < numel:
            raise ValueError("%s must be a contiguous host tensor of %s with at least %d elements" % (
                name, " or ".join(str(d) for d in dtypes), numel))
        return t.data_ptr()

    def encode_obs(self, obs):
        check(self.L.zs_encode_obs(self.h, self._arg(obs, torch.int32, self.N * self.obs_elems, "obs"), self._stream()))
        return obs

    def rollout(self, n_steps, first_step_index=0, actions=None, fmt=abi.ACTIONS_DISCRETE, obs=None, reward=None,
                terminated=None, truncated=None, final_obs=None):
        """``n_steps`` transitions in one launch with same-step auto-reset.  ``obs`` is [N, ...] or a ring [slots, N, ...];
        step i writes slot i % slots.  ``final_obs`` (zs_rollout_final; needs ``obs``): a ring of the same shape that receives,
        in step i's slot, the observation each env whose episode step i ended had before its re-initialisation."""
        n_steps, N = int(n_steps), self.N
        slots = 0 if obs is None else (obs.shape[0] if obs.dim() == len(self.obs_shape) + 2 else 1)
        args = (self._arg(reward, torch.float64, n_steps * N * self.R, "reward"),
                self._arg(terminated, self._FLAG_DTYPES, n_steps * N, "terminated"),
                self._arg(truncated, self._FLAG_DTYPES, n_steps * N, "truncated"), self._stream())
        head = (self.h, n_steps, int(first_step_index), self._action_arg(actions, fmt, n_steps), fmt,
                self._arg(obs, torch.int32, max(1, slots) * N * self.obs_elems, "obs"))
        if final_obs is None:
            check(self.L.zs_rollout(*head, slots, *args))
            return
        if obs is None:
            raise ValueError("final_obs needs obs: the final observations go to the slots of the observation ring")
        if tuple(final_obs.shape) != tuple(obs.shape):
            raise ValueError("final_obs must be shaped like obs %s, got %s" % (tuple(obs.shape), tuple(final_obs.shape)))
        check(self.L.zs_rollout_final(*head, self._arg(final_obs, torch.int32, max(1, slots) * N * self.obs_elems, "final_obs"),
                                      slots, *args))

    def fill_synthetic_actions(self, step_index, actions):
        check(self.L.zs_fill_synthetic_actions(self.h, int(step_index),
                                               self._arg(actions, torch.int32, self.N * self.A, "actions"), self._stream()))
        return actions

    def fill_synthetic_tape(self, first_step_index, actions):
        """actions int32 [n_steps, N, A]: the synthetic action stream of n_steps consecutive steps, one launch."""
        n_steps = int(actions.shape[0])
        check(self.L.zs_fill_synthetic_tape(self.h, int(first_step_index), n_steps,
                                            self._arg(actions, torch.int32, n_steps * self.N * self.A, "actions"), self._stream()))
        return actions

    def episode_stats(self, reset=False):
        out = torch.zeros(4, dtype=torch.int64, device=self.device)
        check(self.L.zs_episode_stats(self.h, _ptr(out), 1 if reset else 0, self._stream()))
        return out

    def launch_count(self):
        return int(self.L.zs_launch_count(self.h))

    def lanes_per_env(self):
        return int(self.L.zs_lanes_per_env(self.h))

    def autoreset_pending(self):
        """Next-step autoreset engines (zs_autoreset_pending): the handle's marks as a bool [N] device tensor, True = the env's
        episode has ended and its next step re-initialises it (gymnasium's ``_autoreset_envs``).  A view of memory the library
        owns and writes, valid while the engine is open: read it, do not write it.  Raises on other engines."""
        if getattr(self, "_pending", None) is None:
            ptr = C.c_void_p()
            check(self.L.zs_autoreset_pending(self.h, C.byref(ptr)))

            class _Marks(object):
                __cuda_array_interface__ = dict(shape=(self.N,), typestr="|u1", data=(ptr.value, False), version=3, strides=None)
            self._pending = torch.as_tensor(_Marks(), device=self.device).view(torch.bool)
        return self._pending
