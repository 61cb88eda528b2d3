"""GPU parity tests: the CUDA path, called through the C ABI, against
  (1) the committed golden traces of the unmodified reference (bit-exact, every field), and
  (2) the C oracle on fresh seeded inputs at sizes the oracle finishes in seconds.
All comparisons are bit-exact (integer state, observation tensors, float64 reward bits)."""
import numpy as np
import pytest

import parity_util as pu
from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", golden_names())
def test_cuda_reproduces_reference_trace(name):
    from cuda_engine import CudaEngine
    meta, traces = load_golden(name)
    cfgd = pu.CONFIGS[name]
    cfg, m = pu.build(cfgd, meta["E"], meta["seed"], env_index_base=meta["base"],
                      max_episode_steps=meta["max_episode_steps"])
    eng = CudaEngine(cfg, m)
    errs = pu.replay_traces(eng, cfgd, traces)
    eng.close()
    assert not errs, "\n".join(errs[:3])


def lockstep(cfgd, N, T, seed, base=0, mes=0, wild=0.25, discrete=False, auto_reset=False, seen=None):
    """CUDA vs oracle, N envs, T ticks, manual masked resets; compares every output and the state.  With auto_reset both
    re-initialise an ended env inside its step (same-step auto-reset) and the episode statistics are compared at the end.
    `seen` (a dict) receives the number of episodes that ended."""
    from cuda_engine import CudaEngine
    from oracle import oracle as orc
    from libzombsole_b200 import abi
    cfg, m = pu.build(cfgd, N, seed, env_index_base=base, max_episode_steps=mes, auto_reset=auto_reset)
    cu, orc_env = CudaEngine(cfg, m), orc.OracleEnv(cfg, m)
    nf = pu.n_fixed_slots(cfgd)
    rs = np.random.RandomState(seed & 0xFFFFFFFF)
    multi = cfgd["kind"] == "multi"
    A = cfg.n_agents
    tapes = [pu.action_tape(cfgd, T, rs.randint(1 << 30), wild=wild) for _ in range(min(N, 8))]
    errs = []
    ended = 0
    assert np.array_equal(cu.encode_obs(), orc_env.encode_obs())
    for t in range(T):
        if discrete:
            actions = rs.randint(-1 if multi else 0, 7 if multi else 6, size=(N, A)).astype(np.int32)
            fmt = abi.ACTIONS_DISCRETE
        else:
            actions = np.stack([tapes[(e + t) % len(tapes)][(t * 7 + e) % T] for e in range(N)])
            fmt = abi.ACTIONS_FULL
        got = cu.step(actions, fmt)
        want = orc_env.step(actions, fmt)
        names = ["obs", "reward", "terminated", "truncated", "agent_mask", "draws"]
        for nme, g, w in zip(names, got, want):
            if nme == "obs" and multi:
                mk = np.repeat(want[4].astype(bool), g.shape[1] // A, axis=1)
                g, w = np.where(mk, g, 0), np.where(mk, w, 0)
            if nme == "reward":
                g, w = g.view(np.uint64), w.view(np.uint64)
            if not np.array_equal(g, w):
                bad = np.argwhere(g != w)[:4].tolist()
                errs.append("tick %d: %s differs at %s" % (t, nme, bad))
        for e in range(0, N, max(1, N // 16)):
            errs += pu.compare_record("env%d tick%d" % (e, t), orc_env.export(e), cu.export(e), nf, check_obs=False)
        if errs:
            break
        done = (want[2] | want[3]).astype(np.uint8)
        ended += int(done.sum())
        if done.any() and not auto_reset:
            ro_c, ro_o = cu.reset(done), orc_env.reset(done)
            sel = done.astype(bool)
            if not np.array_equal(ro_c[sel], ro_o[sel]):
                errs.append("tick %d: reset obs differs" % t)
                break
    if auto_reset and not errs:
        got, want = cu.eng.episode_stats().cpu().numpy(), orc_env.stats()
        if not np.array_equal(got, want):
            errs.append("episode statistics differ: %s vs %s" % (got, want))
    if seen is not None:
        seen["ended"] = ended
    cu.close()
    orc_env.close()
    return errs


CASES = [
    ("c1_bridge_ext", 64, 120, 0), ("c1_bridge_ext", 257, 60, 13), ("c5_bridge_channels", 32, 60, 0),
    ("gym_v0_alone", 64, 80, 0), ("gym_surroundings", 32, 60, 0), ("surroundings_channels", 32, 80, 0),
    ("c3_city_evac", 32, 120, 0), ("village_evac_mixed", 16, 100, 0), ("c4_maze_safehouse", 8, 40, 0),
    ("safehouse_small", 32, 120, 0), ("multi_boxed_2p", 64, 80, 0), ("multi_fort_32p", 4, 30, 0),
    ("survival_minz", 32, 120, 25), ("minz_allcells", 16, 80, 0), ("bots_mixed", 16, 60, 0), ("bots_hamsters", 32, 120, 0), ("fort_max_slots", 3, 25, 0), ("no_zombies", 16, 30, 0),
    ("bots_randoman", 64, 150, 0), ("randoman_crowd", 12, 60, 0), ("box_arena", 96, 60, 0),
    # map geometry at the edges of what zs_create accepts (tests/maps, test_map_edges.py)
    ("bench_odd_cells", 128, 80, 0), ("bench_strip_row", 128, 80, 0), ("bench_wide_max", 24, 60, 0), ("fort_world", 64, 60, 0),
    ("odd_cells_channels", 96, 80, 0), ("surr3_odd_cells", 96, 80, 0), ("surr3_channels_strip_row", 96, 80, 0),
    ("surr255_strip_col", 16, 40, 0), ("surr255_channels_strip_col", 16, 40, 0), ("surr255_odd_cells", 16, 40, 0),
    ("surr255_channels_odd_cells", 16, 40, 0), ("multi_strip_col", 96, 80, 0), ("multi_wide_max", 16, 40, 0),
    ("general_wide_max", 16, 40, 0), ("general_odd_cells", 96, 60, 0), ("minz_no_player_spawns", 96, 80, 0),
    ("minz_few_spawns", 96, 80, 0), ("crowded", 96, 60, 0), ("safehouse_edges", 96, 80, 20),
    # single-agent world scope with 17-32 things (the 32-slot world-scope kernels)
    ("bridge_world_32", 64, 80, 0), ("fort_world_32", 64, 60, 0),
]


@pytest.mark.parametrize("name,N,T,mes", CASES)
def test_cuda_matches_oracle_lockstep(name, N, T, mes):
    seed = 1000 + N + T + (0xC0FFEE0000000000 if name in ("no_zombies", "gym_v0_alone", "c3_city_evac") else 0)  # some with 64-bit seeds
    errs = lockstep(pu.CONFIGS[name], N, T, seed=seed, base=5, mes=mes)
    assert not errs, "\n".join(errs[:3])


@pytest.mark.parametrize("name", ["c1_bridge_ext", "c3_city_evac"])
def test_cuda_matches_oracle_discrete_actions(name):
    errs = lockstep(pu.CONFIGS[name], 48, 100, seed=4242, discrete=True)
    assert not errs, "\n".join(errs[:3])


SURROUNDINGS_CASES = ["gym_surroundings", "surroundings_channels", "c3_city_evac"]


@pytest.mark.parametrize("name", SURROUNDINGS_CASES)
def test_surroundings_without_window_table(name, monkeypatch):
    """The surroundings observation has two pristine-layer paths: a straight copy from the per-cell window table
    (the default, as long as the table is small) and windows cut from the wall-padded template planes.  The
    other cases run the first; this one forces the second."""
    monkeypatch.setenv("ZS_NO_WINDOW_TABLE", "1")
    errs = lockstep(pu.CONFIGS[name], 24, 60, seed=5, base=1)
    assert not errs, "\n".join(errs[:3])
