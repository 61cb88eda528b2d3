"""Box/wall damage over long horizons and at the edges of its encoding.

Boxes and walls keep their damage across episodes (game.py:154-155), so the static patch list (csrc/zs_device.cuh: SPL)
and the compact host records only grow with how long an env has run.  These tests run the CUDA path far enough to reach
the states that growth produces, and write the extreme box/wall lives the public setter allows, and compare with the
oracle bit for bit.  Every test first asserts, from the oracle, that it reached the state it is meant to test:

* the bench game at the bench's horizon (K = 2,000, auto-reset at 1,000 steps) in one fused launch per lane layout, in
  launches of mixed length through the parked images, and with every launch rebuilding its lists from the state;
* the maze past the far index of the patch list (more than 254 entries: SIDX_FAR, spl_find_far), four ways;
* compact host outputs over 2,000 steps of play, and records that outgrow their default size;
* box/wall lives far below zero (written into the state and put back by a masked reset: a fresh world holds them again),
  on both sides of every value where the 16-bit payload used to wrap or read as "gone", in every encoder.
"""
import numpy as np
import pytest
import torch

import parity_util as pu
from cuda_engine import CudaEngine
from libzombsole_b200 import abi
from libzombsole_b200.maps import LABEL_BOX

pytestmark = pytest.mark.gpu


def _labels(cfgd):
    return np.array([s[2] for s in abi.resolve_map(cfgd["map_name"]).statics])


def _simple(cfgd):
    return cfgd["kind"] == "single" and cfgd["observation_position_encoding"] == "simple"


def _listed(cfgd, lives):
    """[..., S] bool: the boxes/walls whose observation differs from the pristine layer (what the patch list holds)."""
    lab = _labels(cfgd)
    mx = np.where(lab == LABEL_BOX, 10, 200)
    if _simple(cfgd):
        val = lambda life: 256 * lab + np.floor_divide(15 * np.minimum(life, 100), 100)
        return val(np.asarray(lives, np.int64)) != val(mx)
    return np.asarray(lives) != mx


def _lives(ref):
    return np.stack([ref.export(e)["static_life"] for e in range(ref.N)]).astype(np.int64)


def _cmp_outputs(tag, got, want):
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError("%s differs at %d places, first %s: %s vs oracle %s" % (
            tag, len(bad), bad[0].tolist(), got[tuple(bad[0])], want[tuple(bad[0])]))


def _rollout_vs_oracle(monkeypatch, cfgd, ref, launches, env, synthetic, envs_checked):
    """Run the whole horizon on the device in the given launches; compare with the oracle's outputs and states."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cu = CudaEngine(ref["cfg"], ref["map"])
    eng = cu.eng
    if "ZS_LANES_PER_ENV" in env:
        assert eng.lanes_per_env() == int(env["ZS_LANES_PER_ENV"])
    K, N = sum(launches), eng.N
    tape = None
    if not synthetic:
        tape = torch.empty((K, N, eng.A), dtype=torch.int32, device=eng.device)
        eng.fill_synthetic_tape(0, tape)
    obs = eng.new_obs()
    rew, term, trunc = eng.new_outputs(K)
    t = 0
    for n in launches:
        eng.rollout(n, t, None if tape is None else tape[t:t + n], abi.ACTIONS_DISCRETE, obs, rew[t:t + n], term[t:t + n],
                    trunc[t:t + n])
        t += n
    torch.cuda.synchronize()
    _cmp_outputs("reward bits", rew.cpu().numpy().view(np.uint64).reshape(ref["rew"].shape), ref["rew"].view(np.uint64))
    _cmp_outputs("terminated", term.cpu().numpy(), ref["term"])
    _cmp_outputs("truncated", trunc.cpu().numpy(), ref["trunc"])
    _cmp_outputs("final observation", obs.cpu().numpy().reshape(N, -1), ref["obs"])
    assert np.array_equal(eng.episode_stats().cpu().numpy(), ref["stats"])
    nf = pu.n_fixed_slots(cfgd)
    errs = []
    for e in envs_checked:
        errs += pu.compare_record("env%d" % e, ref["records"][e], cu.export(e), nf, check_obs=False)
    assert not errs, "\n".join(errs[:3])
    cu.close()


# ------------------------------------------------------------------ a. the bench game at the bench's horizon
BENCH = pu.CONFIGS["c1_bridge_ext"]
BENCH_N, BENCH_K = 4096, 2000
# launches of mixed length through the parked images (one boundary at t = 1000)
MIXED = [1, 3, 8, 20, 64, 500, 1, 7, 396, 1000]
BENCH_SAMPLE = list(range(0, BENCH_N, 97))


@pytest.fixture(scope="module")
def bench_ref():
    from oracle import oracle as orc
    cfg, m = pu.build(BENCH, BENCH_N, 0, max_episode_steps=1000, auto_reset=True)
    ref = orc.OracleEnv(cfg, m)
    o, r, te, tr = ref.rollout_synthetic(BENCH_K, 0)
    out = dict(cfg=cfg, map=m, obs=o, rew=r, term=te, trunc=tr, stats=ref.stats(),
               records={e: ref.export(e) for e in BENCH_SAMPLE}, lives=_lives(ref))
    ref.close()
    return out


@pytest.mark.parametrize("launches,env", [
    ([BENCH_K], {"ZS_LANES_PER_ENV": "16"}), ([BENCH_K], {"ZS_LANES_PER_ENV": "32"}),
    (MIXED, {}), (MIXED, {"ZS_IMAGE_MB": "0"})], ids=["fused-16", "fused-32", "mixed", "mixed-no-image"])
def test_bench_game_at_the_bench_horizon(monkeypatch, bench_ref, launches, env):
    """4,096 bench envs, 2,000 steps of the bench's action tape with auto-reset at 1,000 steps: every reward bit, flag, the
    final observation, the episode statistics and the final state of a sample of envs equal the oracle's."""
    assert sum(MIXED) == BENCH_K
    n = _listed(BENCH, bench_ref["lives"]).sum(axis=1)
    # (the oracle's counts for seed 0: about 60 boxes/walls differ per env, up to 68; some lives are below zero)
    assert n.mean() >= 55 and n.max() >= 64, (n.mean(), n.max())
    assert bench_ref["lives"].min() < 0
    assert bench_ref["trunc"].sum() > 0 and bench_ref["term"].sum() > BENCH_N  # time limits and episode ends
    _rollout_vs_oracle(monkeypatch, BENCH, bench_ref, launches, env, False, BENCH_SAMPLE)


# ------------------------------------------------------------------ b. the maze past the far index
# The simple encoding lists a wall only below 100 life (the value saturates above), and the maze's envs stay under 100
# such entries in 3,000 steps; with the channels encoding every damaged box/wall is listed, and some envs pass 254.
MAZE = dict(pu.CONFIGS["c4_maze_safehouse"], observation_position_encoding="channels")
MAZE_N, MAZE_K, MAZE_SEED = 32, 3000, 5
MAZE_MIXED = [1, 3, 8, 20, 64, 500, 1, 7, 396, 1000, 1000]


@pytest.fixture(scope="module")
def maze_ref():
    from oracle import oracle as orc
    cfg, m = pu.build(MAZE, MAZE_N, MAZE_SEED, max_episode_steps=1000, auto_reset=True)
    ref = orc.OracleEnv(cfg, m)
    _, r0, te0, tr0 = ref.rollout_synthetic(MAZE_K - 500, 0, want_obs=False)
    before = _lives(ref)
    o, r1, te1, tr1 = ref.rollout_synthetic(500, MAZE_K - 500)
    out = dict(cfg=cfg, map=m, obs=o, rew=np.concatenate([r0, r1]), term=np.concatenate([te0, te1]),
               trunc=np.concatenate([tr0, tr1]), stats=ref.stats(), records={e: ref.export(e) for e in range(MAZE_N)},
               before=before, lives=_lives(ref))
    ref.close()
    return out


@pytest.mark.parametrize("launches,env", [
    ([MAZE_K], {}), (MAZE_MIXED, {}), (MAZE_MIXED, {"ZS_IMAGE_MB": "0"}), ([MAZE_K], {"ZS_NO_SL_GLOBAL": "1"})],
    ids=["fused", "mixed", "mixed-no-image", "no-sl-global"])
def test_maze_past_the_far_index(monkeypatch, maze_ref, launches, env):
    assert sum(MAZE_MIXED) == MAZE_K
    listed = _listed(MAZE, maze_ref["lives"])
    far = np.nonzero(listed.sum(axis=1) >= 255)[0]
    assert len(far) > 0, listed.sum(axis=1).max()
    # in such an env, boxes/walls that were listed 500 steps before the end were hit again since (spl_find_far)
    again = _listed(MAZE, maze_ref["before"]) & (maze_ref["lives"] != maze_ref["before"])
    assert again[far].sum(axis=1).max() > 0
    assert maze_ref["trunc"].sum() > 0  # the time limit at 1,000 steps ended episodes
    _rollout_vs_oracle(monkeypatch, MAZE, maze_ref, launches, env, True, range(MAZE_N))


# ------------------------------------------------------------------ c. compact records over a long run
COMPACT_KW = dict(rules_name="extermination", player_names=["terminator", "terminator"], map_name="bridge", agent_id=0,
                  initial_zombies=10, minimum_zombies=0, observation_scope="world", agent_weapon="rifle")


@pytest.mark.parametrize("enc", ["simple", "channels"])
def test_compact_records_over_a_long_run(monkeypatch, enc):
    """2,000 steps at 512 envs with the default record size, auto-reset at 1,000 steps: "compact" (restore + write, and the
    difference of records) and "compact-copy" equal the device-output env every step while damage piles up.  On this game
    the differing cells level off below a default record (the oracle's count of entries per env with the bench's action
    stream: simple about 76, at most 80 of 92, from 3,000 to 6,000 steps; channels about 75, at most 79 of 94, at 3,000
    steps), so no env overflows; records that outgrow their size are reached by written lives
    (test_extreme_static_lives_in_compact_world_records)."""
    from libzombsole_b200.gym_env import ZombsoleVectorEnv
    N, T = 512, 2000
    kw = dict(COMPACT_KW, num_envs=N, seed=9, max_episode_steps=1000, observation_position_encoding=enc)
    plain = ZombsoleVectorEnv(**kw)
    comps = [ZombsoleVectorEnv(host_outputs=mode, **kw) for mode in ("compact", "compact", "compact-copy")]
    words0 = [c.compact_words for c in comps]
    rs = np.random.RandomState(0)
    for t in range(T):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32)).pin_memory()
        o, r, te, tr, _ = plain.step(a.cuda())
        o, r, te, tr = o.cpu(), r.cpu().view(torch.int64), te.cpu(), tr.cpu()
        for i, c in enumerate(comps):
            if t == 0 and i < 2:  # the expansion of zs_step_host is chosen on its first call
                monkeypatch.setenv("ZS_HOST_DIFF", str(i))
            co, cr, cte, ctr, _ = c.step(a)
            assert torch.equal(o, co), "mode %d: observation differs at step %d" % (i, t)
            assert torch.equal(r, cr.view(torch.int64)) and torch.equal(te, cte) and torch.equal(tr, ctr), (i, t)
    # the run reached the damage of a long horizon: about 60 boxes/walls per env differ from the pristine layer
    lives = plain.engine.fields["static_life"][:, :len(_labels(pu.CONFIGS["c1_bridge_ext"]))].cpu().numpy()
    listed = _listed(pu.CONFIGS["c1_bridge_ext" if enc == "simple" else "c5_bridge_channels"], lives).sum(axis=1)
    assert listed.mean() >= 50, listed.mean()
    for c, w0 in zip(comps, words0):
        assert c.compact_overflows == 0 and c.compact_words == w0
    for e in comps + [plain]:
        e.close()


# ------------------------------------------------------------------ d. extreme box/wall lives
# each value on both sides of an edge of the old payload: simple boxes read as "gone" at -1701..-1706 and wrapped below;
# simple walls the same at -6821..-6826; the channels encoding kept 12 bits of life.  -32000 leaves room for the hits
# of the test itself (int16 wrap is out of scope).
SIMPLE_BOX = [-1700, -1701, -1706, -1707, -1800, -4000, -32000]
SIMPLE_WALL = [-6820, -6821, -6826, -6827, -9000, -32000]
CHANNELS = [-2048, -2049, -5000, -32000]


# the lives at which the old simple payload was 0, the "gone" value: the box/wall is present but was taken off the grid,
# which only a move into it or a hit on it in the fresh world's first step shows (the observation value is 0 either way)
GONE_BOX = [-1701, -1702, -1703, -1704, -1705, -1706]
GONE_WALL = [-6821, -6822, -6823, -6824, -6825, -6826]
# one agent with a knife on box_arena's checkerboard of boxes, simple encoding: the adjacent tape moves into, hits and heals
# the neighbouring boxes every step
ARENA_SIMPLE = dict(pu.CONFIGS["box_arena"], kind="single", agent_ids=[0], agent_weapons="knife",
                    observation_scope="world", observation_position_encoding="simple")
CONFIGS = dict(pu.CONFIGS, box_arena_simple=ARENA_SIMPLE)


def _extreme_lives(cfgd, N, S):
    """{(env, static): life}: every other box/wall of every env (every one on box_arena_simple, with the "gone" values),
    the values in turn."""
    lab = _labels(cfgd)[:S]
    gone = cfgd is ARENA_SIMPLE
    out = {}
    for e in range(N):
        for i in range(S):
            if (i + e) % 2 and not gone:
                continue
            if gone:
                vals = GONE_BOX if lab[i] == LABEL_BOX else GONE_WALL
            else:
                vals = (SIMPLE_BOX if lab[i] == LABEL_BOX else SIMPLE_WALL) if _simple(cfgd) else CHANNELS
            out[(e, i)] = vals[(i // 2 + e) % len(vals)]
    return out


@pytest.mark.parametrize("name,N,env", [
    ("c1_bridge_ext", 16, {}), ("c5_bridge_channels", 16, {}),                      # world scope
    ("gym_surroundings", 16, {}), ("village_evac_mixed", 16, {}),                   # surroundings
    ("village_evac_mixed", 16, {"ZS_NO_WINDOW_TABLE": "1"}), ("bots_mixed", 8, {}),
    ("c4_maze_safehouse", 4, {}), ("box_arena", 8, {}),                             # more slots than lanes
    ("c1_bridge_ext", 16, {"ZS_IMAGE_MB": "0"}), ("box_arena_simple", 64, {})])
def test_extreme_static_lives_match_oracle(monkeypatch, name, N, env):
    """Lives far below zero written into boxes/walls, put back into a fresh world by a masked reset (every 4 ticks), then
    stepped in lockstep: observation, reward bits, flags and every env's state equal the oracle's every tick."""
    from oracle import oracle as orc
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cfgd = CONFIGS[name]
    cfg, m = pu.build(cfgd, N, 3)
    cu, ref = CudaEngine(cfg, m), orc.OracleEnv(cfg, m)
    S, nf, T = ref.S, pu.n_fixed_slots(cfgd), 12
    writes = _extreme_lives(cfgd, N, S)
    sl = cu.eng.fields["static_life"]
    for (e, i), v in writes.items():
        sl[e, i] = v
        ref.set_static_life(e, i, v)
    cu.eng.state_written()
    written = np.zeros((N, S), bool)
    for (e, i) in writes:
        written[e, i] = True
    tapes = np.stack([pu.action_tape(cfgd, T, 40 + e) for e in range(N)], axis=1)  # [T, N, A, 3]
    hits = 0
    fresh = np.ones(N, np.uint8)
    for t in range(T):
        if fresh.any():
            _cmp_outputs("reset observation (tick %d)" % t, cu.reset(fresh)[fresh.astype(bool)], ref.reset(fresh)[fresh.astype(bool)])
            if t == 0:  # the written lives are in the fresh worlds, every box/wall present
                lives = _lives(ref)
                assert all(lives[e, i] == v for (e, i), v in writes.items())
                assert all(ref.export(e)["static_present"][written[e]].all() for e in range(N))
        lives0 = _lives(ref)
        got, want = cu.step(tapes[t], abi.ACTIONS_FULL), ref.step(tapes[t], abi.ACTIONS_FULL)
        _cmp_outputs("observation at tick %d" % t, got[0], want[0])
        _cmp_outputs("reward bits at tick %d" % t, got[1].view(np.uint64), want[1].reshape(N, -1).view(np.uint64))
        assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3]), t
        lives1 = _lives(ref)
        hits += int((written & (lives1 != lives0) & fresh.astype(bool)[:, None]).sum())  # hit or healed in a fresh world
        errs = []
        for e in range(N):
            errs += pu.compare_record("env%d tick%d" % (e, t), ref.export(e), cu.export(e), nf, check_obs=False)
        assert not errs, "\n".join(errs[:3])
        fresh = (want[2] | want[3]).astype(np.uint8)
        if t % 4 == 3:
            fresh[:] = 1
    assert lives1.min() > -32700  # no hit came near the int16 wrap
    if name.startswith("box_arena"):  # the agents' hits and heals reach the written boxes on a fresh world's first step
        assert hits > 0
    cu.close()
    ref.close()


def _write_extreme(env, cfgd):
    sl = env.engine.fields["static_life"]
    for (e, i), v in _extreme_lives(cfgd, env.num_envs, len(_labels(cfgd))).items():
        sl[e, i] = v
    env.engine.state_written()


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
@pytest.mark.parametrize("cfg_name", ["c1_bridge_ext", "c5_bridge_channels"])
def test_extreme_static_lives_in_compact_world_records(cfg_name, mode):
    """The world record carries the simple value / the life as signed 16 bits; the host expander reads them back.  Episodes
    of 3 steps with auto-reset: every third step's record holds a fresh world, in which the written boxes/walls are present
    with their lives.  Half of every env's boxes/walls differ, more than a default record holds: on the first step every
    env comes over as a full row (the gather path) and the records grow; after that the records carry the envs."""
    from libzombsole_b200.gym_env import ZombsoleVectorEnv
    cfgd = pu.CONFIGS[cfg_name]
    simple = _simple(cfgd)
    N = 64
    kw = dict(COMPACT_KW, num_envs=N, seed=4, max_episode_steps=3, observation_position_encoding=cfgd["observation_position_encoding"])
    plain, comp = ZombsoleVectorEnv(**kw), ZombsoleVectorEnv(host_outputs=mode, **kw)
    words0 = comp.compact_words
    for env in (plain, comp):
        _write_extreme(env, cfgd)
    m = abi.resolve_map(cfgd["map_name"])
    cells = np.array([y * m.size[0] + x for (x, y, _) in m.statics])
    rs = np.random.RandomState(2)
    most = carried = 0
    for t in range(12):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        before = comp.compact_overflows
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a.pin_memory())
        most = max(most, comp.compact_overflows - before)
        assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
        assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64)) and torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
        if comp.compact_overflows == before:  # every env of this step came in its record
            rows = co.reshape(N, 1 if simple else 3, -1).numpy()[:, 0 if simple else 1, cells]
            # below what the old record could carry: a negative simple value (box <= -1707, wall <= -6827), a life < -2048
            carried += int((rows < (0 if simple else -2048)).sum())
    assert most > 16 and comp.compact_words > words0  # the gather path, then the records grew
    assert carried > 0
    plain.close()
    comp.close()


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
def test_extreme_static_lives_in_compact_agent_records(mode):
    """The same for the per-agent surroundings record: episodes of 3 steps, and the windows of the fresh worlds show
    written boxes/walls with lives below -2048, carried by records (no env of that step overflowed)."""
    from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
    cfgd = pu.CONFIGS["village_evac_mixed"]
    N = 32
    kw = dict(rules_name="evacuation", player_names=["terminator"], map_name="village_for_evacuation",
              agent_ids=["0", "1", "2"], initial_zombies=15, minimum_zombies=0, num_envs=N, seed=5, max_episode_steps=3,
              observation_surroundings_width=9, agent_weapons=["axe", "shotgun", "knife"])
    plain, comp = MultiagentZombsoleVectorEnv(**kw), MultiagentZombsoleVectorEnv(host_outputs=mode, **kw)
    for env in (plain, comp):
        _write_extreme(env, cfgd)
    g = torch.Generator().manual_seed(3)
    carried = 0
    for t in range(12):
        a = torch.randint(-1, 7, (N, 3), generator=g, dtype=torch.int32)
        before = comp.compact_overflows
        o, r, te, tr, info = plain.step(a.cuda())
        co, cr, cte, ctr, cinfo = comp.step(a.pin_memory())
        assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
        assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64)) and torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
        assert torch.equal(info["agent_mask"].cpu(), cinfo["agent_mask"])
        if comp.compact_overflows == before:
            carried += int((co[:, :, 1] < -2048).sum())  # (only a written box/wall has such a life)
    assert carried > 0
    plain.close()
    comp.close()
