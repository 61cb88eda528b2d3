"""host_outputs="compact": what crosses PCIe per step is one small record per env (the cells that differ from the map's
pristine layer, reward, flags); a threaded host routine of the library expands the records into the reference's
observation tensor.  The result must be byte-identical to the device tensors of a plain env on the same inputs, step
after step (the expansion is incremental: it undoes the previous record's cells), across auto-resets, masked resets,
and for envs whose differing cells do not fit a record (overflow: the full row is fetched).  Both flavours: "compact"
(zs_step_host: the records in pinned host memory, written by the kernel in place, every env expanded as its record
arrives) and "compact-copy" (zs_step_compact, copies, zs_expand_compact)."""
import numpy as np
import pytest
import torch

from libzombsole_b200.gym_env import ZombsoleVectorEnv

pytestmark = pytest.mark.gpu

KW = dict(rules_name="extermination", player_names=["terminator", "terminator"], map_name="bridge", agent_id=0,
          initial_zombies=10, minimum_zombies=0, observation_scope="world", agent_weapon="rifle")


# zs_step_host expands an env either by restoring the previous record's cells ahead of the flag and writing the new ones
# after it, or (":diff") as the difference of its two records; left alone (":auto") the handle times both and switches
# between them — sixteen calls of one, sixteen of the other, then the faster — which must never show in a result
MODES = ["compact", "compact-copy", "compact:diff", "compact:auto"]


def _mode(monkeypatch, mode):
    if mode.endswith(":diff"):
        monkeypatch.setenv("ZS_HOST_DIFF", "1")
        return mode[:-5]
    if mode.endswith(":auto"):
        monkeypatch.delenv("ZS_HOST_DIFF", raising=False)
        return mode[:-5]
    monkeypatch.setenv("ZS_HOST_DIFF", "0")
    return mode


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("enc,N,threads", [("simple", 4096, 0), ("simple", 333, 3), ("channels", 1024, 0)])
def test_compact_outputs_equal_device_outputs(monkeypatch, enc, N, threads, mode):
    assert _compare(monkeypatch, mode, N, threads, observation_position_encoding=enc, **KW) == 0


# maps at the edges of the accepted geometry (tests/maps): 143 cells (rows not 16-byte aligned) and 65,504 cells (record
# cells past 32,767), with at most 32 things and with more (the general kernel's record)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,N", [("bench_odd_cells", 512), ("bench_wide_max", 48), ("general_odd_cells", 256),
                                    ("general_wide_max", 32)])
def test_compact_outputs_on_edge_maps(monkeypatch, name, N, mode):
    import parity_util as pu
    c = pu.CONFIGS[name]
    _compare(monkeypatch, mode, N, 0, rules_name=c["rules_name"], player_names=c["player_names"], map_name=c["map_name"],
             agent_id=0, initial_zombies=c["initial_zombies"], minimum_zombies=c["minimum_zombies"],
             observation_scope=c["observation_scope"], agent_weapon=c["agent_weapons"],
             observation_position_encoding=c["observation_position_encoding"])


def _compare(monkeypatch, mode, N, threads, **kw):
    mode = _mode(monkeypatch, mode)
    plain = ZombsoleVectorEnv(num_envs=N, seed=9, max_episode_steps=30, **kw)
    comp = ZombsoleVectorEnv(num_envs=N, seed=9, max_episode_steps=30, host_outputs=mode, host_threads=threads, **kw)
    o0, _ = plain.reset()
    c0, _ = comp.reset()
    assert torch.equal(o0.cpu(), c0)
    rs = np.random.RandomState(0)
    acts = torch.from_numpy(rs.randint(0, 6, size=(70, N)).astype(np.int32))
    for t in range(70):
        o, r, te, tr, _ = plain.step(acts[t].cuda())
        co, cr, cte, ctr, _ = comp.step(acts[t].pin_memory())
        assert co.device.type == "cpu"
        assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
        assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64)), "reward bits differ at step %d" % t
        assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
        if t == 40:  # a masked reset in the middle, then an observation refresh
            mask = torch.from_numpy((rs.rand(N) < 0.25).astype(np.uint8))
            ro, _ = plain.reset(mask=mask)
            rc, _ = comp.reset(mask=mask)
            sel = mask.bool()
            assert torch.equal(ro.cpu()[sel], rc[sel])
        if t == 55:
            assert torch.equal(plain.get_observation().cpu(), comp.get_observation())
    overflows = comp.compact_overflows
    plain.close()
    comp.close()
    return overflows


@pytest.mark.parametrize("mode", MODES)
def test_compact_overflow_fetches_the_full_row(monkeypatch, mode):
    mode = _mode(monkeypatch, mode)
    """More differing cells than a record holds (here: 150 damaged walls in some envs): those envs come over as full rows."""
    N = 64
    plain = ZombsoleVectorEnv(num_envs=N, seed=2, **KW)
    comp = ZombsoleVectorEnv(num_envs=N, seed=2, host_outputs=mode, **KW)
    for env in (plain, comp):
        sl = env.engine.fields["static_life"]
        sl[::5, :150] = torch.where(sl[::5, :150] == 200, torch.full_like(sl[::5, :150], 55), sl[::5, :150])
        env.engine.state_written()
    rs = np.random.RandomState(1)
    for t in range(12):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a)
        assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
        assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64))
        assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
    # the first step could not fit those envs (their full rows were fetched), then the records grew and held them
    assert comp.compact_overflows >= len(range(0, N, 5)) and comp.compact_words > 128
    plain.close()
    comp.close()


@pytest.mark.parametrize("mode", MODES)
def test_compact_overflow_without_growth(monkeypatch, mode):
    mode = _mode(monkeypatch, mode)
    """Records at the size nothing can grow beyond... here held small on purpose: a few envs overflow on every step and
    come over as full rows each time (few enough not to trigger the growth)."""
    N = 256
    plain = ZombsoleVectorEnv(num_envs=N, seed=4, **KW)
    comp = ZombsoleVectorEnv(num_envs=N, seed=4, host_outputs=mode, compact_words=48, **KW)
    for env in (plain, comp):
        sl = env.engine.fields["static_life"]
        sl[7, :60] = 77
        sl[100, :60] = 12
        env.engine.state_written()
    rs = np.random.RandomState(5)
    for t in range(10):
        a = torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32))
        o, r, te, tr, _ = plain.step(a.cuda())
        co, cr, cte, ctr, _ = comp.step(a)
        assert torch.equal(o.cpu(), co), "observation differs at step %d" % t
        assert torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64))
    assert comp.compact_overflows >= 20 and comp.compact_words == 48
    plain.close()
    comp.close()


def test_compact_needs_a_world_observation():
    with pytest.raises(ValueError):
        ZombsoleVectorEnv(num_envs=8, host_outputs="compact", **dict(KW, observation_scope="surroundings:11"))


def test_streamed_step_takes_any_action_container():
    """host_outputs="compact" takes an int32 host tensor as it is; everything else (device tensors, numpy arrays, int64,
    lists of reference action dicts) goes through the env's own pinned buffer — the same transition either way."""
    N = 96
    envs = [ZombsoleVectorEnv(num_envs=N, seed=11, host_outputs="compact", **KW) for _ in range(5)]
    plain = ZombsoleVectorEnv(num_envs=N, seed=11, **KW)
    rs = np.random.RandomState(3)
    for t in range(15):
        ids = rs.randint(0, 6, size=N)
        a32 = torch.from_numpy(ids.astype(np.int32))
        o, r, te, tr, _ = plain.step(a32.cuda())
        outs = [envs[0].step(a32.pin_memory()), envs[1].step(a32.cuda()), envs[2].step(ids.astype(np.int64)),
                envs[3].step([ZombsoleVectorEnv.game_actions[i] for i in ids]), envs[4].step(a32)]
        for co, cr, cte, ctr, _ in outs:
            assert torch.equal(o.cpu(), co) and torch.equal(r.cpu().view(torch.int64), cr.view(torch.int64))
            assert torch.equal(te.cpu(), cte) and torch.equal(tr.cpu(), ctr)
    for e in envs + [plain]:
        e.close()


def test_step_host_rejects_pageable_buffers():
    env = ZombsoleVectorEnv(num_envs=32, seed=1, host_outputs="compact", **KW)
    with pytest.raises(ValueError):
        env._host_step(torch.zeros((32, 1), dtype=torch.int64), 1, True)  # not int32
    with pytest.raises(ValueError):  # records the device cannot reach
        env.engine.host_stepper(torch.zeros((32, env.compact_words), dtype=torch.int32), env._records_prev, env._dev_obs, env.obs,
                                env.reward, env._term, env._trunc, env._overflow)
    env.close()
