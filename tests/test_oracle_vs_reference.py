"""Live check of the C oracle against the UNMODIFIED reference (needs /root/reference; skipped on
the GPU box).  Fresh seeds / action tapes, longer than the committed fixtures."""
import pytest

import parity_util as pu
from oracle import oracle as orc
from oracle import ref_harness

pytestmark = pytest.mark.skipif(not ref_harness.reference_available(), reason="reference tree not present")

CASES = [
    ("c1_bridge_ext", 220, 0), ("c1_bridge_ext", 120, 17), ("c5_bridge_channels", 60, 0), ("gym_v0_alone", 120, 0),
    ("gym_surroundings", 80, 0), ("surroundings_channels", 120, 0), ("c3_city_evac", 150, 0),
    ("village_evac_mixed", 120, 0), ("c4_maze_safehouse", 40, 0), ("safehouse_small", 150, 0),
    ("multi_boxed_2p", 120, 0), ("multi_fort_32p", 30, 0), ("survival_minz", 150, 33), ("minz_allcells", 100, 0), ("bots_mixed", 80, 0), ("bots_hamsters", 150, 0), ("fort_max_slots", 12, 0), ("no_zombies", 30, 0),
    ("box_arena", 50, 0),
    # map geometry at the edges of what zs_create accepts (tests/maps)
    ("bench_odd_cells", 80, 0), ("bench_strip_row", 80, 0), ("bench_wide_max", 30, 0), ("fort_world", 60, 0),
    ("odd_cells_channels", 80, 0), ("surr3_odd_cells", 80, 0), ("surr3_channels_strip_row", 80, 0),
    ("surr255_strip_col", 30, 0), ("surr255_channels_strip_col", 30, 0), ("surr255_odd_cells", 30, 0),
    ("surr255_channels_odd_cells", 30, 0), ("multi_strip_col", 80, 0), ("multi_wide_max", 30, 0),
    ("general_wide_max", 30, 0), ("general_odd_cells", 60, 0), ("minz_no_player_spawns", 80, 0), ("minz_few_spawns", 80, 0),
    ("crowded", 60, 0), ("safehouse_edges", 80, 0),
]


@pytest.mark.parametrize("name,T,mes", CASES)
def test_oracle_matches_live_reference(name, T, mes):
    cfgd = pu.CONFIGS[name]
    seed, base, E = 991 + T, 40, 2
    if name in ("no_zombies", "gym_v0_alone"):
        seed += 0x9E3779B97F4A7C15  # 64-bit seed: both Philox key words in use
    traces = [ref_harness.run_trace(cfgd, base + e, seed, pu.action_tape(cfgd, T, 7 * T + e), max_episode_steps=mes)
              for e in range(E)]
    cfg, m = pu.build(cfgd, E, seed, env_index_base=base, max_episode_steps=mes)
    eng = orc.OracleEnv(cfg, m)
    errs = pu.replay_traces(eng, cfgd, traces)
    eng.close()
    assert not errs, "\n".join(errs[:3])
