"""MultiagentZombsoleVectorEnv(host_outputs="compact" | "compact-copy"): one small record per env crosses PCIe (the agents'
window centres and lives, rewards, agent mask, flags, and the cells any window shows that differ from the map's pristine
layer); the library's host threads expand the records into the per-agent windows.  Everything must be byte-identical to the
device tensors of a plain env on the same inputs, step after step: observations, reward bits, flags, the agent mask, and
the agents' lives after the step (against the state buffer) — across auto-resets, masked resets, dead agents' windows,
windows reaching past the map edge, and envs whose records overflow (the full rows are fetched)."""
import numpy as np
import pytest
import torch

import parity_util as pu
from libzombsole_b200 import abi
from libzombsole_b200._native import ZsError
from libzombsole_b200.engine import ZsEngine
from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv

pytestmark = pytest.mark.gpu

MODES = ["compact", "compact-copy"]


def _kwargs(name):
    c = pu.CONFIGS[name]
    return dict(rules_name=c["rules_name"], player_names=c["player_names"], map_name=c["map_name"], agent_ids=c["agent_ids"],
                initial_zombies=c["initial_zombies"], minimum_zombies=c["minimum_zombies"],
                observation_surroundings_width=c["surroundings_width"], agent_weapons=c["agent_weapons"])


def _check(plain, comp, step, o, r, te, tr, info, co, cr, cte, ctr, cinfo):
    assert co.device.type == "cpu"
    assert torch.equal(o.cpu(), co), "observation differs at step %d" % step
    assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64)), "reward bits differ at step %d" % step
    assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr), "flags differ at step %d" % step
    assert torch.equal(info["agent_mask"].cpu(), cinfo["agent_mask"]), "agent mask differs at step %d" % step
    P, A = plain.cfg.n_bots, plain.num_agents
    assert torch.equal(plain.engine.fields["life"][:, P:P + A].cpu(), comp.agent_life_host), "agent lives differ at step %d" % step


def _run(name, N, mode, threads=0, steps=70, seed=9, max_episode_steps=30, compact_words=0):
    kw = _kwargs(name)
    plain = MultiagentZombsoleVectorEnv(num_envs=N, seed=seed, max_episode_steps=max_episode_steps, **kw)
    comp = MultiagentZombsoleVectorEnv(num_envs=N, seed=seed, max_episode_steps=max_episode_steps, host_outputs=mode,
                                       host_threads=threads, compact_words=compact_words, **kw)
    A = plain.num_agents
    o0, _ = plain.reset()
    c0, _ = comp.reset()
    assert torch.equal(o0.cpu(), c0)
    rs = np.random.RandomState(0)
    acts = torch.from_numpy(rs.randint(-1, 7, size=(steps, N, A)).astype(np.int32))  # (-1: the agent's key is missing)
    dead_windows = 0
    for t in range(steps):
        o, r, te, tr, info = plain.step(acts[t].cuda())
        co, cr, cte, ctr, cinfo = comp.step(acts[t].pin_memory())
        _check(plain, comp, t, o, r, te, tr, info, co, cr, cte, ctr, cinfo)
        dead_windows += int((comp.agent_life_host <= 0).sum())
        if t == 40:  # a masked reset in the middle, then an observation refresh
            mask = torch.from_numpy((rs.rand(N) < 0.25).astype(np.uint8))
            ro, _ = plain.reset(mask=mask)
            rc, _ = comp.reset(mask=mask)
            sel = mask.bool()
            assert torch.equal(ro.cpu()[sel], rc[sel])
        if t == 55:
            assert torch.equal(plain.get_observation().cpu(), comp.get_observation())
    plain.close()
    comp.close()
    return comp, dead_windows


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("N,threads", [(1024, 0), (333, 3)])
def test_config3_game(N, threads, mode):
    """BASELINE config 3's game: city_for_evacuation, 4 agents, 20 zombies, 21-wide windows (they reach past the map edge)."""
    comp, dead_windows = _run("c3_city_evac", N, mode, threads)
    assert comp.compact_overflows == 0
    assert dead_windows > 0  # windows centred where an agent died were compared too


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["village_evac_mixed", "bots_hamsters"])
def test_more_games(name, mode):
    """A bot and mixed weapons on 9-wide windows; hamsters with the minimum-zombie respawn and decide-phase draws."""
    _run(name, 256, mode)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,N", [("multi_strip_col", 256), ("multi_wide_max", 64)])
def test_edge_maps(name, N, mode):
    """Maps at the edges of the accepted geometry (tests/maps): one cell wide (every window mostly past the map edge) and
    65,504 cells (window centres and record cells past 32,767)."""
    _run(name, N, mode)


@pytest.mark.parametrize("mode", MODES)
def test_two_envs_per_warp(monkeypatch, mode):
    monkeypatch.setenv("ZS_LANES_PER_ENV", "16")
    kw = _kwargs("multi_boxed_2p")
    probe = MultiagentZombsoleVectorEnv(num_envs=512, seed=3, **kw)
    assert probe.engine.lanes_per_env() == 16
    probe.close()
    _run("multi_boxed_2p", 512, mode, seed=3)


@pytest.mark.parametrize("mode", MODES)
def test_without_window_table(monkeypatch, mode):
    """ZS_NO_WINDOW_TABLE=1: the overflow rows and the plain env's windows come from the other device encoder."""
    monkeypatch.setenv("ZS_NO_WINDOW_TABLE", "1")
    _run("c3_city_evac", 256, mode, compact_words=64)


def _damage(env, every=5):
    """Damage every box/wall of every fifth env: on the city map many of them lie in the agents' windows."""
    sl = env.engine.fields["static_life"]
    sl[::every] = torch.where(sl[::every] > 1, sl[::every] - 1, sl[::every])
    env.engine.state_written()


@pytest.mark.parametrize("mode", MODES)
def test_overflow_fetches_the_full_rows_and_grows(mode):
    N = 128
    kw = _kwargs("c3_city_evac")
    plain = MultiagentZombsoleVectorEnv(num_envs=N, seed=2, **kw)
    comp = MultiagentZombsoleVectorEnv(num_envs=N, seed=2, host_outputs=mode, **kw)
    for env in (plain, comp):
        _damage(env)
    words0 = comp.compact_words
    rs = np.random.RandomState(1)
    for t in range(12):
        a = torch.from_numpy(rs.randint(-1, 7, size=(N, plain.num_agents)).astype(np.int32))
        o, r, te, tr, info = plain.step(a.cuda())
        co, cr, cte, ctr, cinfo = comp.step(a)
        _check(plain, comp, t, o, r, te, tr, info, co, cr, cte, ctr, cinfo)
    # the first steps could not fit those envs (their full rows were fetched), then the records grew and held them
    assert comp.compact_overflows >= len(range(0, N, 5)) and comp.compact_words > words0
    plain.close()
    comp.close()


@pytest.mark.parametrize("mode", MODES)
def test_overflow_without_growth(mode):
    """Records held small on purpose: a few envs overflow on every step and come over as full rows each time."""
    N = 256
    kw = _kwargs("c3_city_evac")
    plain = MultiagentZombsoleVectorEnv(num_envs=N, seed=4, **kw)
    comp = MultiagentZombsoleVectorEnv(num_envs=N, seed=4, host_outputs=mode, compact_words=96, **kw)
    for env in (plain, comp):
        _damage(env, every=100)
    rs = np.random.RandomState(5)
    for t in range(10):
        a = torch.from_numpy(rs.randint(-1, 7, size=(N, plain.num_agents)).astype(np.int32))
        o, r, te, tr, info = plain.step(a.cuda())
        co, cr, cte, ctr, cinfo = comp.step(a)
        _check(plain, comp, t, o, r, te, tr, info, co, cr, cte, ctr, cinfo)
    assert comp.compact_overflows >= 20 and comp.compact_words == 96
    plain.close()
    comp.close()


def test_streamed_step_takes_any_action_container():
    """host_outputs="compact" takes an int32 host tensor as it is; device tensors, numpy arrays and lists of per-agent action
    dicts go through the env's own pinned buffer — the same transition either way."""
    N = 64
    kw = _kwargs("c3_city_evac")
    envs = [MultiagentZombsoleVectorEnv(num_envs=N, seed=11, host_outputs="compact", **kw) for _ in range(5)]
    plain = MultiagentZombsoleVectorEnv(num_envs=N, seed=11, **kw)
    ids_ = plain.possible_agents
    rs = np.random.RandomState(3)
    for t in range(15):
        ids = rs.randint(0, 7, size=(N, plain.num_agents))
        a32 = torch.from_numpy(ids.astype(np.int32))
        o, r, te, tr, info = plain.step(a32.cuda())
        dicts = [{aid: MultiagentZombsoleVectorEnv.game_actions[ids[n, i]] for i, aid in enumerate(ids_)} for n in range(N)]
        outs = [envs[0].step(a32.pin_memory()), envs[1].step(a32.cuda()), envs[2].step(ids.astype(np.int64)),
                envs[3].step(dicts), envs[4].step(a32)]
        for co, cr, cte, ctr, cinfo in outs:
            assert torch.equal(o.cpu(), co) and torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64))
            assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
            assert torch.equal(info["agent_mask"].cpu(), cinfo["agent_mask"])
    for e in envs + [plain]:
        e.close()


def test_refusals():
    with pytest.raises(ValueError, match="at most 32 things"):  # 32 agents + 100 zombies
        MultiagentZombsoleVectorEnv(num_envs=4, host_outputs="compact", **_kwargs("multi_fort_32p"))
    # the per-agent record exists for per-agent surroundings handles only, the world record for world-scope handles only
    cfg, m = pu.build(pu.CONFIGS["c1_bridge_ext"], 8, 0)
    world = ZsEngine(cfg, m)
    assert world.agent_compact_words() == 0 and world.agent_compact_max_words() == 0
    rec = torch.zeros((8, 128), dtype=torch.int32, device=world.device)
    acts = torch.zeros((8, 1), dtype=torch.int32, device=world.device)
    with pytest.raises(ZsError, match="per-agent compact"):
        world.step_compact_agents(acts, abi.ACTIONS_DISCRETE, rec)
    cfg, m = pu.build(pu.CONFIGS["c3_city_evac"], 8, 0)
    multi = ZsEngine(cfg, m)
    assert multi.compact_words() == 0 and multi.agent_compact_words() > 0
    assert multi.agent_compact_max_words() >= multi.agent_compact_words()
    world.close()
    multi.close()
