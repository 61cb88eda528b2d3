"""Adapter giving ZsEngine (the CUDA path, through the C ABI) the same test-facing methods as
oracle.oracle.OracleEnv, so parity_util.replay_traces can drive either."""
import numpy as np
import torch

from libzombsole_b200 import abi
from libzombsole_b200.engine import ZsEngine


class CudaEngine(object):
    def __init__(self, cfg, map_, device="cuda"):
        self.eng = ZsEngine(cfg, map_, device=device)
        e = self.eng
        self.N, self.A, self.M, self.S, self.cells = e.N, e.A, e.M, e.S, e.cells
        self.obs = e.new_obs()
        self.reward, self.term, self.trunc = e.new_outputs()
        self.mask = torch.zeros((e.N, e.A), dtype=torch.uint8, device=e.device)
        self.draws = torch.zeros(e.N, dtype=torch.int32, device=e.device)
        self._cache = None

    @classmethod
    def of(cls, eng):
        """The adapter around an engine made elsewhere (a vector env's): export() and fields() only."""
        self = cls.__new__(cls)
        self.eng, self._cache = eng, None
        self.N, self.A, self.M, self.S, self.cells = eng.N, eng.A, eng.M, eng.S, eng.cells
        return self

    def close(self):
        self.eng.close()

    def _np(self, t):
        return t.detach().cpu().numpy()

    def reset(self, mask=None):
        m = None if mask is None else torch.as_tensor(np.ascontiguousarray(mask, dtype=np.uint8))
        self.eng.reset(m, self.obs)
        self._cache = None
        return self._np(self.obs).reshape(self.N, -1)

    def encode_obs(self):
        self.eng.encode_obs(self.obs)
        return self._np(self.obs).reshape(self.N, -1)

    def step(self, actions, fmt):
        a = torch.as_tensor(np.ascontiguousarray(actions, dtype=np.int32)).to(self.eng.device)
        self.eng.step(a, fmt, self.obs, self.reward, self.term, self.trunc, self.mask, self.draws)
        self._cache = None
        return (self._np(self.obs).reshape(self.N, -1), self._np(self.reward).reshape(self.N, -1), self._np(self.term),
                self._np(self.trunc), self._np(self.mask), self._np(self.draws))

    def fields(self):
        if self._cache is None:
            torch.cuda.synchronize(self.eng.device)
            self._cache = {k: self._np(v) for k, v in self.eng.fields.items()}
            self._cache["reset_draws"] = self._np(self.eng.reset_draws)
        return self._cache

    def export(self, env):
        f = self.fields()
        M, S = self.M, self.S
        meta = f["meta"][env, :M]
        in_world = (meta >> 7).astype(np.uint8)
        stamp = f["stamp"][env, :M]
        order = np.full(M, -1, np.int16)
        live = np.nonzero(in_world)[0]
        live = live[np.argsort(stamp[live], kind="stable")]
        order[:len(live)] = live
        sc = f["scalars"][env]
        slife = f["static_life"][env, :S].copy()
        fresh = bool(sc[abi.S_FLAGS] & 1)
        dead_bytes = f["dead_body"][env].view(np.uint8)[: (self.cells + 7) // 8].copy()
        return {
            "x": f["x"][env, :M].copy(), "y": f["y"][env, :M].copy(), "life": f["life"][env, :M].copy(),
            "in_world": in_world, "weapon": (meta & 15).astype(np.uint8), "order": order,
            "static_life": slife, "static_present": ((slife > 0) | fresh).astype(np.uint8),
            "dead_body": dead_bytes,
            "counters": np.array([sc[abi.S_T], sc[abi.S_DEATHS], sc[abi.S_ZOMBIE_DEATHS]], np.int32),
            "episode": int(sc[abi.S_EPISODE]), "episode_steps": int(sc[abi.S_EPISODE_STEPS]),
            "reset_draws": int(f["reset_draws"][env]),
        }
