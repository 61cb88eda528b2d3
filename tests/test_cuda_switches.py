"""The tuning switches of zs_create (INTEGRATION.md §5) select among kernel variants and data placements; none of
them may change a result.  Each case runs a fused rollout with same-step auto-resets under one switch and compares
observations, float64 reward bits, flags and episode statistics with the oracle."""
import numpy as np
import pytest

from libzombsole_b200 import abi
from test_cuda_properties import engine

pytestmark = pytest.mark.gpu

CASES = [
    # switch, value, config, envs, steps
    ("ZS_NO_TMA", "1", "c1_bridge_ext", 2048, 48),
    ("ZS_NO_TMA_PAIR", "1", "c1_bridge_ext", 2048, 48),
    ("ZS_SMEM_SKEW", "0", "c1_bridge_ext", 2048, 48),
    ("ZS_OCC", "4", "c1_bridge_ext", 1024, 48),
    # (6 is accepted for two-env warps only: 4,096 envs is an even batch of more than 16 envs per SM)
    ("ZS_OCC", "6", "c1_bridge_ext", 4096, 48),
    ("ZS_OCC", "7", "c1_bridge_ext", 1024, 48),
    ("ZS_WARPS_PER_CTA", "1", "c5_bridge_channels", 512, 48),
    ("ZS_WARPS_PER_CTA", "4", "c1_bridge_ext", 1024, 48),
    ("ZS_NO_FAST_INIT", "1", "c1_bridge_ext", 512, 64),
    ("ZS_NO_SL_GLOBAL", "1", "c4_maze_safehouse", 128, 24),
    ("ZS_WARPS_PER_CTA", "2", "c4_maze_safehouse", 128, 24),
    ("ZS_NO_WINDOW_TABLE", "1", "c3_city_evac", 256, 40),
    # without the parked images every launch re-derives ranks, grid and lists from the state buffer (large batches)
    ("ZS_IMAGE_MB", "0", "c1_bridge_ext", 2048, 48),
    ("ZS_IMAGE_MB", "0", "c3_city_evac", 256, 40),
    ("ZS_IMAGE_MB", "0", "c4_maze_safehouse", 128, 24),
    # groups without spawn cells: candidates by compaction of all cells instead of from the map's free-cell table
    ("ZS_NO_FREE_TABLE", "1", "c4_maze_safehouse", 128, 24),
    ("ZS_NO_FREE_TABLE", "1", "c3_city_evac", 256, 40),
    ("ZS_NO_FREE_TABLE", "1", "minz_allcells", 256, 40),
    # one launch shape for everything / single steps with two envs per warp
    ("ZS_ONE_SHAPE", "1", "c1_bridge_ext", 4000, 48),
    ("ZS_SHORT_STEPS", "1000", "c1_bridge_ext", 4000, 48),
    ("ZS_PDL", "1", "c1_bridge_ext", 2048, 48),
    ("ZS_PDL", "0", "c1_bridge_ext", 2048, 5),
    ("ZS_TMA_PAIR", "1", "c1_bridge_ext", 4000, 48),
    # observations written by a producer warp per CTA instead of by the game warps themselves (an experiment kept correct)
    ("ZS_PRODUCER", "1", "c1_bridge_ext", 4000, 48),
    ("ZS_PRODUCER", "1", "c5_bridge_channels", 3000, 48),
    # the same placements on the maps at the edges of the accepted geometry (tests/maps)
    ("ZS_NO_WINDOW_TABLE", "1", "surr255_strip_col", 64, 24),
    ("ZS_NO_WINDOW_TABLE", "1", "surr3_channels_strip_row", 256, 40),
    ("ZS_NO_WINDOW_TABLE", "1", "multi_strip_col", 256, 40),
    ("ZS_IMAGE_MB", "0", "bench_odd_cells", 1024, 48),
    ("ZS_IMAGE_MB", "0", "bench_wide_max", 64, 24),
    ("ZS_IMAGE_MB", "0", "general_odd_cells", 256, 40),
    ("ZS_IMAGE_MB", "0", "minz_few_spawns", 256, 40),
    ("ZS_NO_FREE_TABLE", "1", "minz_no_player_spawns", 256, 40),
    ("ZS_NO_FREE_TABLE", "1", "crowded", 256, 40),
]


@pytest.mark.parametrize("switch,value,name,N,K", CASES)
def test_switch_does_not_change_results(monkeypatch, switch, value, name, N, K):
    from oracle import oracle as orc
    monkeypatch.setenv(switch, value)
    eng, cfg, m = engine(name, N, seed=23)
    obs = eng.new_obs()
    rew, term, trunc = eng.new_outputs(K)
    eng.rollout(K, 0, None, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)
    ref = orc.OracleEnv(cfg, m)
    o, r, te, tr = ref.rollout_synthetic(K, 0)
    assert np.array_equal(obs.cpu().numpy().reshape(N, -1), o)
    assert np.array_equal(rew.cpu().numpy().view(np.uint64).reshape(K, N, -1), r.view(np.uint64).reshape(K, N, -1))
    assert np.array_equal(term.cpu().numpy(), te) and np.array_equal(trunc.cpu().numpy(), tr)
    assert np.array_equal(eng.episode_stats().cpu().numpy(), ref.stats())
    eng.close()


def test_prefetch_switch_single_steps(monkeypatch):
    """ZS_NO_PREFETCH only concerns launches of fewer than four steps: single steps with and without it land in the same state."""
    import torch
    from test_cuda_properties import state_snapshot, assert_same_state
    snaps = []
    for off in ("", "1"):
        if off:
            monkeypatch.setenv("ZS_NO_PREFETCH", off)
        eng, cfg, m = engine("c1_bridge_ext", 40000, seed=3)
        obs = eng.new_obs()
        rew, term, trunc = eng.new_outputs()
        acts = torch.zeros((eng.N, 1), dtype=torch.int32, device=eng.device)
        for t in range(6):
            eng.fill_synthetic_actions(t, acts)
            eng.step(acts, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)
        snaps.append((state_snapshot(eng), obs.clone()))
        M = eng.M
        eng.close()
    assert_same_state(snaps[0][0], snaps[1][0], M)
    assert torch.equal(snaps[0][1], snaps[1][1])
