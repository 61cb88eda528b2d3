"""The maps of tests/maps/ that put the kernels at the edges of the geometry zs_create accepts (width or height 1, cell counts
not a multiple of 4, more than 32,768 cells, maps without spawn cells or with too few, objectives on the outermost row
and column).  Each map is asserted to have the property it is there for, so that an edit of a map cannot quietly take it
out of the case it covers, and every configuration on it runs through the oracle with episodes ending where the rules let
them end.  (The CUDA kernels are compared with the oracle on these configurations by the GPU tests.)"""
import numpy as np
import pytest

import parity_util as pu
from libzombsole_b200 import abi
from libzombsole_b200.maps import Map

# the configurations on the edge maps (parity_util.CONFIGS)
EDGE_CONFIGS = ["bench_odd_cells", "bench_strip_row", "bench_wide_max", "fort_world", "odd_cells_channels", "surr3_odd_cells",
                "surr3_channels_strip_row", "surr255_strip_col", "surr255_channels_strip_col", "surr255_odd_cells",
                "surr255_channels_odd_cells", "multi_strip_col", "multi_wide_max", "general_wide_max", "general_odd_cells",
                "minz_no_player_spawns", "minz_few_spawns", "crowded", "safehouse_edges"]


def _map(name):
    return Map.from_map_name(pu._edge_map(name) if name != "fort" else name)


def _cells(m):
    return m.size[0] * m.size[1]


def _slots(cfgd):
    return len(cfgd["player_names"]) + len(cfgd["agent_ids"]) + max(cfgd["initial_zombies"], cfgd["minimum_zombies"])


def _window_table_bytes(m, width, channels):
    """zs_create's per-cell window table (zs_b200.cu): cells x round_up(planes * width^2, 32) ints."""
    ints = (2 if channels else 1) * width * width
    return _cells(m) * ((ints + 31) // 32 * 32) * 4


def _bench_lean_init(m):
    """zs_create's lean world init (and so the bench roster kernel) for 3 players and 10 zombies."""
    ps, zs = len(m.player_spawns), len(m.zombie_spawns)
    return ps >= 3 and zs >= 10 and ps + zs <= 256


def test_cell_counts_mod_4():
    """The world observation's template is copied by TMA only when the cell count is a multiple of 4: these maps are not."""
    assert _cells(_map("strip_row")) % 4 == 1 and _cells(_map("fort")) % 4 == 1
    assert _cells(_map("strip_col")) % 4 == 2 and _cells(_map("no_player_spawns")) % 4 == 2
    assert _cells(_map("odd_cells")) % 4 == 3


def test_strips():
    r, c = _map("strip_row"), _map("strip_col")
    assert r.size[1] == 1 and r.size[0] >= 64
    assert c.size[0] == 1 and c.size[1] >= 32
    for m in (r, c):
        assert m.statics and _bench_lean_init(m)


def test_wide_max():
    m = _map("wide_max")
    W, H = m.size
    assert (W, H) == (2047, 32) and W * H <= 65535
    # everything stands at cells of 32,768 or more, near both ends of the rows
    things = [s[:2] for s in m.statics] + m.player_spawns + m.zombie_spawns
    assert min(y * W + x for x, y in things) >= 32768
    xs = [x for x, _ in m.player_spawns + m.zombie_spawns]
    assert min(xs) == 0 and max(xs) == W - 1
    assert any(y * W + x == W * H - 1 for x, y, _ in m.statics)  # the last cell holds a box
    assert 0 < len(m.statics) < 32 and _bench_lean_init(m)
    # more zombie spawn cells than the general-kernel game has zombies, player spawn cells for the multi-agent game
    assert len(m.zombie_spawns) >= pu.CONFIGS["general_wide_max"]["initial_zombies"]
    assert len(m.player_spawns) >= pu.n_fixed_slots(pu.CONFIGS["multi_wide_max"])


def test_odd_cells():
    m = _map("odd_cells")
    assert _bench_lean_init(m) and _cells(m) % 4 == 3
    # width 255 windows: too many cells for the window table in either encoding (32 MB) ...
    assert _window_table_bytes(m, 255, False) > 32 << 20 and _window_table_bytes(m, 255, True) > 32 << 20
    # ... while strip_col keeps it in both
    c = _map("strip_col")
    assert _window_table_bytes(c, 255, False) <= 32 << 20 and _window_table_bytes(c, 255, True) <= 32 << 20
    assert _slots(pu.CONFIGS["general_odd_cells"]) > 32 and len(m.zombie_spawns) >= 32


def test_spawn_shortages():
    n = _map("no_player_spawns")
    assert not n.player_spawns and n.zombie_spawns
    f, cfgd = _map("few_spawns"), pu.CONFIGS["minz_few_spawns"]
    # exactly one player spawn cell per player (the reference raises when a player finds none), fewer zombie spawn cells
    # than zombies: the lean init is off through the spawn counts alone
    assert len(f.player_spawns) == pu.n_fixed_slots(cfgd)
    assert len(f.zombie_spawns) < cfgd["initial_zombies"] < cfgd["minimum_zombies"]
    c, cfgd = _map("crowded"), pu.CONFIGS["crowded"]
    assert not c.player_spawns and not c.zombie_spawns
    free = _cells(c) - len(c.statics)
    assert pu.n_fixed_slots(cfgd) <= free < _slots(cfgd)


def test_edge_objectives():
    m = _map("edge_objectives")
    W, H = m.size
    assert any(y == H - 1 for _, y in m.objectives) and any(x == W - 1 for x, _ in m.objectives)
    assert (W - 1, H - 1) in m.objectives


@pytest.mark.parametrize("name", EDGE_CONFIGS)
def test_config_runs_through_the_oracle(name):
    """Each configuration steps through the oracle with random actions and manual resets; where the rules let episodes end
    (all of them here) at least one ends, and for the configurations with too few cells or spawn cells the things that
    cannot be placed are left out of the world."""
    from oracle import oracle as orc
    cfgd = pu.CONFIGS[name]
    N, T = 8, 150
    cfg, m = pu.build(cfgd, N, 77)
    env = orc.OracleEnv(cfg, m)
    multi = cfgd["kind"] == "multi"
    rs = np.random.RandomState(0)
    ends = 0
    placed_max = 0
    for _ in range(T):
        acts = rs.randint(-1 if multi else 0, 7 if multi else 6, size=(N, cfg.n_agents)).astype(np.int32)
        obs, rew, term, trunc, _, _ = env.step(acts, abi.ACTIONS_DISCRETE)
        assert obs.shape == (N, env.obs_elems)
        done = (term | trunc).astype(np.uint8)
        ends += int(done.sum())
        if name == "crowded":
            placed_max = max(placed_max, max(int(env.export(e)["in_world"].sum()) for e in range(N)))
        if done.any():
            env.reset(done)
    env.close()
    assert ends > 0
    if name == "crowded":
        mp = Map.from_map_name(cfgd["map_name"])
        assert placed_max == _cells(mp) - len(mp.statics)  # the map was full
