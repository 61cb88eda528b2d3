"""The largest map zs_create accepts at the batch sizes a user runs, and a map no CTA can hold.

wide_max (2,047 x 32 = 65,504 cells) needs about 75 KB of shared memory per env of the bench game: at 4,096 envs the
default two-warp CTA of two-env warps would need four of them (about 300 KB), more than a CTA can have, and zs_create
falls back to narrower CTAs.  Each batch size runs a fused rollout of the bench game against the oracle."""
import numpy as np
import pytest
import torch

import parity_util as pu
from libzombsole_b200 import abi
from libzombsole_b200.maps import Map

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,K,want_obs", [(64, 48, True), (1024, 32, True), (4096, 16, False)])
def test_wide_max_rollout_matches_oracle(N, K, want_obs):
    """(At 4,096 envs the oracle's observations would take 1 GB: reward bits, flags and episode statistics are compared;
    the kernel still writes its observations, so the standard rollout shape runs.)"""
    from oracle import oracle as orc
    from test_cuda_properties import engine
    eng, cfg, m = engine("bench_wide_max", N, seed=61, base=3, mes=12)
    obs = eng.new_obs()
    rew, term, trunc = eng.new_outputs(K)
    eng.rollout(K, 0, None, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)
    ref = orc.OracleEnv(cfg, m)
    o, r, te, tr = ref.rollout_synthetic(K, 0, want_obs=want_obs)
    if want_obs:
        assert np.array_equal(obs.cpu().numpy().reshape(N, -1), o)
    assert np.array_equal(rew.cpu().numpy().view(np.uint64).reshape(K, N, -1), r.view(np.uint64).reshape(K, N, -1))
    assert np.array_equal(term.cpu().numpy(), te) and np.array_equal(trunc.cpu().numpy(), tr)
    stats = eng.episode_stats().cpu().numpy()
    assert np.array_equal(stats, ref.stats())
    assert stats[0] > 0  # episodes ended (TimeLimit 12) and worlds were re-initialised inside the rollout
    eng.close()
    ref.close()


def test_map_beyond_any_cta_is_refused():
    """65,535 cells with 30,000 walls: one env alone needs more shared memory than a CTA has.  zs_create refuses the map
    with its message (and the library stays usable)."""
    from libzombsole_b200._native import ZsError
    from libzombsole_b200.engine import ZsEngine
    W, H = 255, 257
    rows = []
    for y in range(H):
        row = ["w" if (y * W + x) % 2 == 1 and (y * W + x) // 2 < 30000 else "." for x in range(W)]
        rows.append("".join(row))
    rows[H - 1] = "p" * 3 + "z" * 10 + rows[H - 1][13:]
    m = Map.from_text("\n".join(rows), name="walls")
    assert m.size == (W, H) and W * H == 65535 and len(m.statics) == 30000
    cfg, _ = pu.build(pu.CONFIGS["c1_bridge_ext"], 64, 1)
    with pytest.raises(ZsError, match="more shared memory than one CTA has"):
        ZsEngine(cfg, m)
    # a fitting handle afterwards still works
    eng = ZsEngine(cfg, "bridge")
    obs = eng.new_obs()
    rew, term, trunc = eng.new_outputs(4)
    eng.rollout(4, 0, None, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)
    torch.cuda.synchronize()
    eng.close()
