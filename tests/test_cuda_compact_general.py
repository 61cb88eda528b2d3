"""Compact host outputs (host_outputs="compact" | "compact-copy") for world-scope games of more than 32 things: the general
step kernels (more slots than lanes) build the record themselves (zs_sim_kernel SHAPE 5).  Everything must be
byte-identical to the device tensors of a plain env on the same seed and inputs, step after step: observations, reward
bits and flags — across auto-resets, masked resets, the minimum-zombie respawn, every placement of the env's state, box/wall
lives far below zero, and envs whose records overflow (the full rows are fetched).  Every test first asserts that its
handle really has more than 32 slots."""
import numpy as np
import pytest
import torch

import parity_util as pu
from libzombsole_b200 import abi
from libzombsole_b200.engine import ZsEngine
from libzombsole_b200.gym_env import ZombsoleGymEnv, ZombsoleVectorEnv
from test_cuda_long_horizon import _labels, _write_extreme

pytestmark = pytest.mark.gpu

# BASELINE config 4's game: 1 agent + 100 zombies, world observation (1, 39, 72)
C4 = dict(rules_name="safehouse", player_names=[], map_name="maze_for_safehouse", agent_id=0, initial_zombies=100,
          minimum_zombies=0, observation_scope="world", agent_weapon="rifle")
# 1 agent + 4 bots + 200 zombies: 256 slots, and the minimum-zombie respawn runs before the record is built
FORT_256 = dict(rules_name="survival", player_names=["sniper", "troll", "hamster", "terminator"], map_name="fort", agent_id=0,
                initial_zombies=200, minimum_zombies=195, observation_scope="world", agent_weapon="gun")

# as in test_cuda_compact.py: zs_step_host restores ahead and writes after the flag, or (":diff") takes the difference of two
# records; left alone (":auto") the handle times both and switches between them
MODES = ["compact", "compact:diff", "compact:auto", "compact-copy"]


def _mode(monkeypatch, mode):
    if mode.endswith(":diff"):
        monkeypatch.setenv("ZS_HOST_DIFF", "1")
        return mode[:-5]
    if mode.endswith(":auto"):
        monkeypatch.delenv("ZS_HOST_DIFF", raising=False)
        return mode[:-5]
    monkeypatch.setenv("ZS_HOST_DIFF", "0")
    return mode


def _slots(env, at_least=33):
    slots = env.engine.fields["life"].shape[1]
    assert slots >= at_least, slots
    return slots


def _same(t, o, r, te, tr, co, cr, cte, ctr):
    assert co.device.type == "cpu"
    assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
    assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64)), "reward bits differ at step %d" % t
    assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr), "flags differ at step %d" % t


def _lockstep(kw, N, mode, threads=0, steps=70, seed=9, max_episode_steps=30, compact_words=0, each_step=None):
    """plain and compact env in lockstep on the same random discrete ids; a masked reset at step 40 and an observation refresh
    at step 55.  Returns the compact env (closed)."""
    plain = ZombsoleVectorEnv(num_envs=N, seed=seed, max_episode_steps=max_episode_steps, **kw)
    comp = ZombsoleVectorEnv(num_envs=N, seed=seed, max_episode_steps=max_episode_steps, host_outputs=mode,
                             host_threads=threads, compact_words=compact_words, **kw)
    _slots(comp)
    assert comp.compact
    o0, _ = plain.reset()
    c0, _ = comp.reset()
    assert torch.equal(o0.cpu(), c0)
    rs = np.random.RandomState(0)
    acts = torch.from_numpy(rs.randint(0, 6, size=(steps, N)).astype(np.int32))
    for t in range(steps):
        o, r, te, tr, _ = plain.step(acts[t].cuda())
        co, cr, cte, ctr, _ = comp.step(acts[t].pin_memory())
        _same(t, o, r, te, tr, co, cr, cte, ctr)
        if each_step:
            each_step(t, plain)
        if t == 40:
            mask = torch.from_numpy((rs.rand(N) < 0.25).astype(np.uint8))
            ro, _ = plain.reset(mask=mask)
            rc, _ = comp.reset(mask=mask)
            sel = mask.bool()
            assert torch.equal(ro.cpu()[sel], rc[sel])
        if t == 55:
            assert torch.equal(plain.get_observation().cpu(), comp.get_observation())
    plain.close()
    comp.close()
    return comp


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("enc,N,threads", [("simple", 1024, 0), ("simple", 333, 3), ("channels", 1024, 0), ("channels", 333, 3)])
def test_config4_game(monkeypatch, enc, N, threads, mode):
    """BASELINE config 4's game (101 slots, 128-slot kernels): no env overflows a default record."""
    comp = _lockstep(dict(C4, observation_position_encoding=enc), N, _mode(monkeypatch, mode), threads)
    assert comp.compact_overflows == 0


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
@pytest.mark.parametrize("enc", ["simple", "channels"])
def test_256_slot_game_with_respawn(enc, mode):
    """Scripted bots and 200 zombies on the fort (256-slot kernels), with the minimum-zombie respawn: zombies die and are
    replaced in the step before its record is built."""
    N = 256
    deaths = []

    def respawned(t, plain):
        P, M = 5, 205  # bots + agent, slots in use
        eng = plain.engine
        assert eng.fields["life"].shape[1] > 128
        in_world = (eng.fields["meta"][:, P:M].to(torch.int32) & 0x80) != 0
        assert int(in_world.sum(dim=1).min()) >= FORT_256["minimum_zombies"], t
        deaths.append(int(eng.fields["scalars"][:, abi.S_ZOMBIE_DEATHS].sum()))

    comp = _lockstep(dict(FORT_256, observation_position_encoding=enc), N, mode, each_step=respawned)
    assert max(deaths) > 0
    assert comp.compact_overflows == 0


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
@pytest.mark.parametrize("placement", [{"ZS_IMAGE_MB": "0"}, {"ZS_NO_SL_GLOBAL": "1"}])
def test_placements(monkeypatch, placement, mode):
    """ZS_IMAGE_MB=0: every launch loads the state and a single step walks the dead-body bitmap (FL_DEAD_LAUNCH), so the
    records come from the bitmap branch.  ZS_NO_SL_GLOBAL=1: the box/wall lives stay in shared memory."""
    for k, v in placement.items():
        monkeypatch.setenv(k, v)
    comp = _lockstep(dict(C4, observation_position_encoding="simple"), 256, mode, steps=60)
    assert comp.compact_overflows == 0


def _damage_walls(env, envs, n):
    """The first n boxes/walls of the given envs lose most of their life: n more differing cells in those envs."""
    sl = env.engine.fields["static_life"]
    part = sl[envs, :n]
    sl[envs, :n] = torch.where(part > 60, torch.full_like(part, 55), part)
    env.engine.state_written()


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
def test_overflow_fetches_the_full_rows_and_grows(mode):
    """300 damaged walls in every fifth env: more than a default record holds.  Those envs come over as full rows, then the
    records grow and hold them."""
    N = 64
    plain = ZombsoleVectorEnv(num_envs=N, seed=2, **C4)
    comp = ZombsoleVectorEnv(num_envs=N, seed=2, host_outputs=mode, **C4)
    _slots(comp)
    words0 = comp.compact_words
    for env in (plain, comp):
        _damage_walls(env, slice(None, None, 5), 300)
    rs = np.random.RandomState(1)
    for t in range(12):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a)
        _same(t, o, r, te, tr, co, cr, cte, ctr)
    assert comp.compact_overflows >= len(range(0, N, 5)) and comp.compact_words > words0
    plain.close()
    comp.close()


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
def test_overflow_without_growth(mode):
    """Records held at 160 words: the two damaged envs overflow on every step and come over as full rows each time (too few
    to make the records grow)."""
    N = 256
    plain = ZombsoleVectorEnv(num_envs=N, seed=4, **C4)
    comp = ZombsoleVectorEnv(num_envs=N, seed=4, host_outputs=mode, compact_words=160, **C4)
    _slots(comp)
    for env in (plain, comp):
        _damage_walls(env, [7, 100], 200)
    rs = np.random.RandomState(5)
    for t in range(10):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a)
        _same(t, o, r, te, tr, co, cr, cte, ctr)
    assert comp.compact_overflows >= 20 and comp.compact_words == 160
    plain.close()
    comp.close()


@pytest.mark.parametrize("mode", ["compact", "compact-copy"])
@pytest.mark.parametrize("enc", ["simple", "channels"])
def test_extreme_static_lives(enc, mode):
    """Lives far below zero written into every other box/wall of the maze (test_cuda_long_horizon.py), put back by 3-step
    episodes with auto-reset: the records carry simple values below zero / channel lives below -2048 in steps where no env
    overflowed."""
    cfgd = dict(pu.CONFIGS["c4_maze_safehouse"], observation_position_encoding=enc)
    simple = enc == "simple"
    N = 32
    kw = dict(C4, num_envs=N, seed=4, max_episode_steps=3, observation_position_encoding=enc)
    plain, comp = ZombsoleVectorEnv(**kw), ZombsoleVectorEnv(host_outputs=mode, **kw)
    _slots(comp)
    for env in (plain, comp):
        _write_extreme(env, cfgd)
    m = abi.resolve_map(cfgd["map_name"])
    assert len(_labels(cfgd)) == len(m.statics)
    cells = np.array([y * m.size[0] + x for (x, y, _) in m.statics])
    rs = np.random.RandomState(2)
    carried = 0
    for t in range(12):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        before = comp.compact_overflows
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a.pin_memory())
        _same(t, o, r, te, tr, co, cr, cte, ctr)
        if comp.compact_overflows == before:  # every env of this step came in its record
            rows = co.reshape(N, 1 if simple else 3, -1).numpy()[:, 0 if simple else 1, cells]
            carried += int((rows < (0 if simple else -2048)).sum())
    assert carried > 0
    plain.close()
    comp.close()


def test_long_run():
    """512 envs for 2,000 steps with auto-reset at 1,000: "compact" equals the device-output env every step while box/wall
    damage and dead bodies pile up."""
    N, T = 512, 2000
    kw = dict(C4, num_envs=N, seed=9, max_episode_steps=1000)
    plain, comp = ZombsoleVectorEnv(**kw), ZombsoleVectorEnv(host_outputs="compact", **kw)
    _slots(comp)
    rs = np.random.RandomState(0)
    resets = 0
    for t in range(T):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32)).pin_memory()
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a)
        _same(t, o, r, te, tr, co, cr, cte, ctr)
        resets += int((te | tr).sum())
    assert resets >= N  # every env reset at least once (the time limit, if nothing else)
    plain.close()
    comp.close()


def test_drop_in_class_takes_the_compact_path():
    """ZombsoleGymEnv asks for "compact-if-available": on config 4's game it now steps through zs_step_host, and equals a
    one-env device-output vector env over two episodes (each until the game ends, at most 600 steps)."""
    g = ZombsoleGymEnv(**C4, seed=3)
    assert g.vec.compact and g.vec.streamed
    _slots(g.vec)
    plain = ZombsoleVectorEnv(num_envs=1, seed=3, max_episode_steps=None, auto_reset=False, **C4)
    rs = np.random.RandomState(7)
    steps = 0
    for ep in range(2):
        go, _ = g.reset()
        po, _ = plain.reset()
        assert np.array_equal(go, po[0].cpu().numpy())
        for t in range(600):
            steps += 1
            i = int(rs.randint(0, 6))
            go, gr, gte, gtr, _ = g.step(ZombsoleVectorEnv.game_actions[i])
            po, pr, pte, ptr, _ = plain.step(torch.tensor([i], dtype=torch.int32, device=plain.device))
            assert np.array_equal(go, po[0].cpu().numpy()), (ep, t)
            assert np.float64(gr).view(np.int64) == pr.cpu().view(torch.int64).item()
            assert gte == bool(pte[0].item()) and gtr == bool(ptr[0].item())
            if gte or gtr:
                break
    assert steps > 2
    g.close()
    plain.close()


def test_abi():
    """The maze's world handle has a record form; surroundings and per-agent handles of more than 32 slots still have none."""
    cfg, m = pu.build(pu.CONFIGS["c4_maze_safehouse"], 8, 0)
    world = ZsEngine(cfg, m)
    assert world.fields["life"].shape[1] > 32
    assert world.compact_words() > 0 and world.compact_max_words() >= world.compact_words()
    assert world.agent_compact_words() == 0
    surr = ZsEngine(*pu.build(dict(pu.CONFIGS["c4_maze_safehouse"], observation_scope="surroundings:11"), 8, 0))
    assert surr.fields["life"].shape[1] > 32
    assert surr.compact_words() == 0 and surr.compact_max_words() == 0 and surr.agent_compact_words() == 0
    multi = ZsEngine(*pu.build(pu.CONFIGS["fort_max_slots"], 8, 0))
    assert multi.fields["life"].shape[1] > 32
    assert multi.compact_words() == 0 and multi.agent_compact_words() == 0 and multi.agent_compact_max_words() == 0
    for e in (world, surr, multi):
        e.close()
    with pytest.raises(ValueError, match="world-scope"):
        ZombsoleVectorEnv(num_envs=4, host_outputs="compact", **dict(C4, observation_scope="surroundings:11"))


def test_streamed_step_takes_any_action_container():
    """host_outputs="compact" on config 4's game takes an int32 host tensor as it is; device tensors, numpy arrays, int64
    and lists of reference action dicts go through the env's own pinned buffer — the same transition either way."""
    N = 96
    envs = [ZombsoleVectorEnv(num_envs=N, seed=11, host_outputs="compact", **C4) for _ in range(5)]
    _slots(envs[0])
    plain = ZombsoleVectorEnv(num_envs=N, seed=11, **C4)
    rs = np.random.RandomState(3)
    for t in range(15):
        ids = rs.randint(0, 6, size=N)
        a32 = torch.from_numpy(ids.astype(np.int32))
        o, r, te, tr, _ = plain.step(a32.cuda())
        outs = [envs[0].step(a32.pin_memory()), envs[1].step(a32.cuda()), envs[2].step(ids.astype(np.int64)),
                envs[3].step([ZombsoleVectorEnv.game_actions[i] for i in ids]), envs[4].step(a32)]
        for co, cr, cte, ctr, _ in outs:
            _same(t, o, r, te, tr, co, cr, cte, ctr)
    for e in envs + [plain]:
        e.close()
