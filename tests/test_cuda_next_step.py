"""Next-step autoreset (include/zs_b200.h: ZS_AUTORESET_NEXT_STEP; gymnasium's AutoresetMode.NEXT_STEP).  The step that ends an
episode is a step of an auto_reset = 0 handle; the env's next step ignores its action, re-initialises the world as zs_reset
does and returns the new world's observation with reward +0.0, no flags, every agent in the mask and the init's draws.

* lockstep against a twin (same seed and env indices, auto_reset = 0) that runs zs_step_masked on the envs that are not
  pending and zs_reset on those that are: observations, reward bits, flags, agent masks, draws, the state, the marks and the
  episode statistics agree after every step, on nine configurations and TimeLimits 1, 2 and 9, and at the BASELINE size;
* fused rollouts (K = 1, 7, 64, and launches of mixed length, an episode ending on the last step of a launch) equal single
  steps, starting from the parked images and without them;
* every output path of the vector envs (device, pinned host, both compact record paths, record overflow) gives the same bytes;
* reset(mask), masked steps and encode_obs of pending envs; the refusals; the kernel a bench-shaped rollout launches.
"""
import re

import numpy as np
import pytest
import torch

import parity_util as pu
from libzombsole_b200 import abi
from test_cuda_properties import assert_same_state, state_snapshot

gpu = pytest.mark.gpu


def _engine(name, N, seed, mes, next_step, base=11):
    from libzombsole_b200.engine import ZsEngine
    cfg, m = pu.build(pu.CONFIGS[name], N, seed, env_index_base=base, max_episode_steps=mes, auto_reset=next_step)
    if next_step:
        cfg.auto_reset = abi.AUTORESET_NEXT_STEP
    return ZsEngine(cfg, m), cfg


def _bits(t):
    return t.view(torch.int64)


class Twin(object):
    """An auto_reset = 0 engine composed into next-step autoreset from calls the oracle tests pin: zs_step_masked on the envs
    that are not pending, zs_reset on those that are (their outputs: reward +0.0, no flags, every agent, the init's draws).
    Keeps the episode statistics a next-step handle counts at the ending steps."""

    def __init__(self, eng, cfg):
        self.e, self.cfg = eng, cfg
        self.pending = torch.zeros(eng.N, dtype=torch.bool, device=eng.device)
        self.stats = np.zeros(4, np.int64)

    def step(self, acts, fmt, obs, rew, term, trunc, mask, draws, select=None):
        e, N = self.e, self.e.N
        sel = torch.ones(N, dtype=torch.bool, device=e.device) if select is None else select
        run, rst = sel & ~self.pending, sel & self.pending
        if bool(run.all()):
            e.step(acts, fmt, obs, rew, term, trunc, mask, draws)
        elif bool(run.any()):
            e.step_masked(run.to(torch.uint8), acts, fmt, obs, rew, term, trunc, mask)
        if bool(rst.any()):
            e.reset(rst.to(torch.uint8), obs)
            rew[rst] = 0.0
            term[rst] = 0
            trunc[rst] = 0
            mask[rst] = 1
            draws[rst] = e.reset_draws[rst]
        ended = run & (term | trunc).bool()
        if bool(ended.any()):
            self._count(ended, term, rew)
        self.pending = (self.pending & ~sel) | ended
        return run, rst

    def _count(self, ended, term, rew):
        """What the ending steps add to zs_episode_stats: episodes, won episodes, their lengths, their zombie deaths.  A won
        episode is a termination whose end reward was +10: some agent still alive gained more than it could by the step
        alone (-10 plus what a step gives is below 0)."""
        sc = self.e.fields["scalars"]
        P, A = self.cfg.n_bots, self.cfg.n_agents
        alive = self.e.fields["life"][:, P:P + A] > 0
        r = rew.view(self.e.N, -1)
        gained = ((r > 0) & (alive if r.shape[1] == A else alive.any(dim=1, keepdim=True))).any(dim=1)
        self.stats += np.array([int(ended.sum()), int((ended & term.bool() & gained).sum()),
                                int(sc[ended, abi.S_EPISODE_STEPS].sum()), int(sc[ended, abi.S_ZOMBIE_DEATHS].sum())])

    def reset(self, mask, obs):
        self.e.reset(mask, obs)
        self.pending &= ~mask.bool()


class Pair(object):
    """A next-step engine and its twin, with one set of outputs each."""

    def __init__(self, name, N, seed, mes):
        self.a, self.cfg = _engine(name, N, seed, mes, True)
        b, _ = _engine(name, N, seed, mes, False)
        self.t = Twin(b, self.cfg)
        self.N, self.A = N, self.cfg.n_agents
        dev = self.a.device
        self.out = []
        for eng in (self.a, b):
            rew, term, trunc = eng.new_outputs()
            self.out.append(dict(obs=eng.new_obs(), rew=rew, term=term, trunc=trunc,
                                 mask=torch.zeros((N, self.A), dtype=torch.uint8, device=dev),
                                 draws=torch.zeros(N, dtype=torch.int32, device=dev)))
        self.acts = torch.zeros((N, self.A), dtype=torch.int32, device=dev)
        self.n_reset_steps = 0

    def step(self, t, select=None):
        """Step t (synthetic actions of step t) on both; compares everything."""
        self.a.fill_synthetic_actions(t, self.acts)
        oa, ob = self.out
        for o in self.out:
            o["draws"].fill_(-1)
        if select is None:
            self.a.step(self.acts, abi.ACTIONS_DISCRETE, oa["obs"], oa["rew"], oa["term"], oa["trunc"], oa["mask"], oa["draws"])
        else:
            self.a.step_masked(select.to(torch.uint8), self.acts, abi.ACTIONS_DISCRETE, oa["obs"], oa["rew"], oa["term"],
                               oa["trunc"], oa["mask"])
        run, rst = self.t.step(self.acts, abi.ACTIONS_DISCRETE, ob["obs"], ob["rew"], ob["term"], ob["trunc"], ob["mask"],
                               ob["draws"], select)
        self.n_reset_steps += int(rst.sum())
        sel = run | rst
        assert torch.equal(oa["term"][sel], ob["term"][sel]) and torch.equal(oa["trunc"][sel], ob["trunc"][sel]), \
            "flags differ at step %d" % t
        assert torch.equal(_bits(oa["rew"][sel]), _bits(ob["rew"][sel])), "reward bits differ at step %d" % t
        assert torch.equal(oa["mask"][sel], ob["mask"][sel]), "agent mask differs at step %d" % t
        assert torch.equal(oa["obs"][sel], ob["obs"][sel]), "observation differs at step %d" % t
        if select is None:
            # (zs_step_masked has no draws output: the twin's are known where it stepped all envs, and on its reset steps)
            known = sel if bool(run.all()) or not bool(run.any()) else rst
            assert torch.equal(oa["draws"][known], ob["draws"][known]), "draws differ at step %d" % t
        self.check_state(t)
        return run, rst

    def check_state(self, t):
        assert torch.equal(self.a.autoreset_pending(), self.t.pending), "pending marks differ after step %d" % t
        assert_same_state(state_snapshot(self.a), state_snapshot(self.t.e), self.a.M)

    def check_stats(self):
        got = self.a.episode_stats().cpu().numpy()
        assert np.array_equal(got, self.t.stats), (got, self.t.stats)

    def close(self):
        self.a.close()
        self.t.e.close()


# (config, envs): both encodings and scopes, per-agent windows, 128 slots, boxes, the minimum-zombie respawn, and a game
# whose every episode ends on its first step (a reset step is followed at once by another ending step)
LOCKSTEP = [("c1_bridge_ext", 512), ("c5_bridge_channels", 256), ("gym_surroundings", 256), ("surroundings_channels", 256),
            ("c3_city_evac", 128), ("c4_maze_safehouse", 64), ("box_arena", 128), ("survival_minz", 128), ("no_zombies", 64)]


@gpu
@pytest.mark.parametrize("mes", [1, 2, 9])
@pytest.mark.parametrize("name,N", LOCKSTEP)
def test_lockstep_with_the_composed_twin(name, N, mes):
    pr = Pair(name, N, 71, mes)
    assert pr.a.lanes_per_env() == 32
    T = 30
    for t in range(T):
        pr.step(t)
    assert pr.n_reset_steps > 0
    if mes == 1:  # every other step of every env is a reset step
        assert pr.n_reset_steps == N * (T // 2)
    pr.check_stats()
    pr.close()


@gpu
def test_baseline_size_lockstep():
    """BASELINE configs[1]'s size: 4,096 bridge envs (two envs per warp on a same-step handle) x 64 steps."""
    pr = Pair("c1_bridge_ext", 4096, 73, 9)
    assert pr.a.lanes_per_env() == 32
    for t in range(64):
        pr.step(t)
    assert pr.n_reset_steps > 4096
    pr.check_stats()
    pr.close()


def _rollouts_vs_single_steps(name, N, lengths, mes, seed=79):
    a, cfg = _engine(name, N, seed, mes, True)
    c, _ = _engine(name, N, seed, mes, True)
    A, T = cfg.n_agents, sum(lengths)
    tape = torch.zeros((T, N, A), dtype=torch.int32, device=a.device)
    for s in range(T):
        a.fill_synthetic_actions(500 + s, tape[s])
    obs_c = c.new_obs()
    rc, tc, uc = c.new_outputs()
    s0 = 0
    ended_last = reset_first = False
    for K in lengths:
        ring = a.new_obs(K)
        ra, ta, ua = a.new_outputs(K)
        pend_before = a.autoreset_pending().clone()
        a.rollout(K, 0, tape[s0:s0 + K].contiguous(), abi.ACTIONS_DISCRETE, ring, ra, ta, ua)
        reset_first |= bool(pend_before.any())
        for s in range(K):
            c.step(tape[s0 + s], abi.ACTIONS_DISCRETE, obs_c, rc, tc, uc)
            assert torch.equal(ta[s], tc) and torch.equal(ua[s], uc), "flags differ at step %d" % (s0 + s)
            assert torch.equal(_bits(ra[s]), _bits(rc)), "reward bits differ at step %d" % (s0 + s)
            assert torch.equal(ring[s], obs_c), "observation of step %d differs" % (s0 + s)
        ended_last |= bool((ta[K - 1] | ua[K - 1]).any())
        assert torch.equal(a.autoreset_pending(), c.autoreset_pending())
        assert_same_state(state_snapshot(a), state_snapshot(c), a.M)
        s0 += K
    assert torch.equal(a.episode_stats(), c.episode_stats())
    a.close()
    c.close()
    return ended_last, reset_first


@gpu
@pytest.mark.parametrize("images", [True, False])
@pytest.mark.parametrize("K,mes", [(1, 1), (7, 3), (64, 4)])
@pytest.mark.parametrize("name,N", [("c1_bridge_ext", 1024), ("gym_surroundings", 256), ("c3_city_evac", 128),
                                    ("c4_maze_safehouse", 48)])
def test_rollouts_equal_single_steps(monkeypatch, name, N, K, mes, images):
    """Two launches of K steps; the TimeLimit (mes + 1 divides K + 1 or K) ends the episodes of the TimeLimit on the last step
    of the first launch, and their reset steps are the first of the second."""
    if not images:
        monkeypatch.setenv("ZS_IMAGE_MB", "0")
    ended_last, reset_first = _rollouts_vs_single_steps(name, N, [K, K], mes)
    assert ended_last and reset_first


@gpu
@pytest.mark.parametrize("images", [True, False])
@pytest.mark.parametrize("name,N", [("c1_bridge_ext", 1024), ("survival_minz", 128), ("c4_maze_safehouse", 48)])
def test_mixed_launch_lengths_equal_single_steps(monkeypatch, name, N, images):
    if not images:
        monkeypatch.setenv("ZS_IMAGE_MB", "0")
    # TimeLimit 3: the TimeLimit ends episodes on steps 2, 6, 10, 14, ...; launches end on steps 2, 6, 7, 10, 11, 14, 22
    ended_last, reset_first = _rollouts_vs_single_steps(name, N, [3, 4, 1, 3, 1, 3, 8, 1, 9], 3)
    assert ended_last and reset_first


# ---------------------------------------------------------------- control calls
@gpu
@pytest.mark.parametrize("name,N", [("c1_bridge_ext", 256), ("c3_city_evac", 64), ("c4_maze_safehouse", 32)])
def test_reset_masked_step_and_encode_of_pending_envs(name, N):
    pr = Pair(name, N, 83, 4)
    rs = np.random.RandomState(7)
    enc = pr.a.new_obs()
    for t in range(24):
        if t % 3 == 1:
            # a masked step: unselected envs stay pending, selected pending envs take their reset step
            sel = torch.from_numpy(rs.rand(N) < 0.5).to(pr.a.device)
            pend = pr.t.pending.clone()
            pr.step(t, select=sel)
            still = pend & ~sel
            assert bool(pr.a.autoreset_pending()[still].all())
        else:
            pr.step(t)
        pend = pr.t.pending.clone()
        if bool(pend.any()):
            # encode_obs of a pending env shows the world it ended in: the observation of its ending step
            pr.a.encode_obs(enc)
            assert torch.equal(enc[pend], pr.out[0]["obs"][pend])
        if t % 4 == 2 and bool(pend.any()):
            # reset(mask) of pending envs clears their marks: their next step is a transition
            m = (pend & torch.from_numpy(rs.rand(N) < 0.5).to(pr.a.device)).to(torch.uint8)
            pr.a.reset(m, pr.out[0]["obs"])
            pr.t.reset(m, pr.out[1]["obs"])
            assert torch.equal(pr.out[0]["obs"], pr.out[1]["obs"])
            assert not bool(pr.a.autoreset_pending()[m.bool()].any())
            pr.check_state(t)
    pr.close()


# ---------------------------------------------------------------- the Python layer
def _host_action_tapes(N, A, n, T, seed):
    rs = np.random.RandomState(seed)
    return [torch.from_numpy(rs.randint(0, n, size=(N, A) if A > 1 else N).astype(np.int32)) for _ in range(T)]


def _env_paths_vs_twin(make, paths, N, A, n_actions, T=24):
    """Every env of `paths` (kwargs) against the twin, step after step: outputs as host bytes."""
    envs = [make(autoreset_mode="next_step", **kw) for kw in paths]
    twin_env = make(auto_reset=False)
    tw = Twin(twin_env.engine, twin_env.cfg)
    for env in envs:
        assert env.engine.lanes_per_env() == 32 and env.cfg.auto_reset == abi.AUTORESET_NEXT_STEP
        env.reset()
    twin_env.reset()
    dev = twin_env.device
    rew, term, trunc = twin_env.engine.new_outputs()
    obs = twin_env.engine.new_obs()
    mask = torch.ones((N, A), dtype=torch.uint8, device=dev)
    draws = torch.zeros(N, dtype=torch.int32, device=dev)
    n_reset = 0
    for t, a in enumerate(_host_action_tapes(N, A, n_actions, T, 13)):
        _, rst = tw.step(a.to(dev).view(N, A), abi.ACTIONS_DISCRETE, obs, rew, term, trunc, mask, draws)
        n_reset += int(rst.sum())
        for env, kw in zip(envs, paths):
            o, r, te, tr, info = env.step(a)
            what = "%s at step %d" % (kw, t)
            assert torch.equal(o.cpu(), obs.cpu()), "observation differs: " + what
            assert torch.equal(_bits(r.cpu()), _bits(rew.cpu())), "reward bits differ: " + what
            assert torch.equal(te.cpu(), term.bool().cpu()) and torch.equal(tr.cpu(), trunc.bool().cpu()), "flags differ: " + what
            if "agent_mask" in info:
                assert torch.equal(info["agent_mask"].cpu(), mask.bool().cpu()), "agent mask differs: " + what
            assert torch.equal(env.autoreset_envs, tw.pending), "marks differ: " + what
    assert n_reset > N
    overflows = [getattr(env, "compact_overflows", 0) for env in envs]
    for env in envs:
        env.close()
    twin_env.close()
    return overflows


@gpu
def test_vector_env_every_output_path(monkeypatch):
    from libzombsole_b200.gym_env import make_vector
    N = 256

    def make(**kw):
        return make_vector("jvstinian/Zombsole-v0", N, seed=89, max_episode_steps=5, **kw)

    paths = [dict(host_outputs=False), dict(host_outputs=True), dict(host_outputs="compact-copy"),
             dict(host_outputs="compact-copy", compact_words=12), dict(host_outputs="compact", compact_words=12)]
    overflows = _env_paths_vs_twin(make, paths, N, 1, 6)
    assert overflows[3] > 0 and overflows[4] > 0  # the record-overflow path ran
    for diff in ("0", "1"):  # zs_step_host's two expansions (read when the handle takes its first host step)
        monkeypatch.setenv("ZS_HOST_DIFF", diff)
        _env_paths_vs_twin(make, [dict(host_outputs="compact")], N, 1, 6)


@gpu
def test_multiagent_env_every_output_path():
    from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
    cfgd = pu.CONFIGS["c3_city_evac"]
    args = (cfgd["rules_name"], cfgd["player_names"], cfgd["map_name"], cfgd["agent_ids"], cfgd["initial_zombies"],
            cfgd["minimum_zombies"])
    N, A = 64, len(cfgd["agent_ids"])

    def make(**kw):
        return MultiagentZombsoleVectorEnv(*args, num_envs=N, seed=97, max_episode_steps=4, **kw)

    paths = [dict(host_outputs=False), dict(host_outputs=True), dict(host_outputs="compact"),
             dict(host_outputs="compact-copy"), dict(host_outputs="compact", compact_words=2 + 3 * A + 8)]
    overflows = _env_paths_vs_twin(make, paths, N, A, 7)
    assert overflows[4] > 0


@gpu
def test_make_vector_passes_the_mode():
    from libzombsole_b200.gym_env import ZombsoleVectorEnv, _next_step_mode, make_vector
    env = make_vector("jvstinian/Zombsole-v0", 8, autoreset_mode="next_step")
    same = make_vector("jvstinian/Zombsole-v0", 8)
    assert env.cfg.auto_reset == abi.AUTORESET_NEXT_STEP and same.cfg.auto_reset == abi.AUTORESET_SAME_STEP
    assert env.metadata["autoreset_mode"] == _next_step_mode() and "autoreset_mode" not in same.metadata
    assert "autoreset_mode" not in ZombsoleVectorEnv.metadata  # (an instance copy)
    assert env.autoreset_envs.dtype == torch.bool and env.autoreset_envs.shape == (8,) and not bool(env.autoreset_envs.any())
    with pytest.raises(Exception, match="next-step"):
        same.autoreset_envs
    env.close()
    same.close()


# ---------------------------------------------------------------- refusals
@pytest.mark.parametrize("kw,match", [(dict(autoreset_mode="next-step"), "autoreset_mode must be"),
                                      (dict(autoreset_mode=None), "autoreset_mode must be"),
                                      (dict(autoreset_mode="next_step", auto_reset=False), "needs auto_reset=True"),
                                      (dict(autoreset_mode="next_step", final_observation=True), "final_observation")])
def test_refusals(kw, match):
    """The argument combinations next-step autoreset cannot serve are refused before anything is allocated (no GPU needed)."""
    from libzombsole_b200.gym_env import ZombsoleVectorEnv, make_vector
    from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
    with pytest.raises(ValueError, match=match):
        make_vector("jvstinian/Zombsole-v0", 4, **kw)
    with pytest.raises(ValueError, match=match):
        ZombsoleVectorEnv("extermination", [], "bridge", 0, 10, num_envs=4, **kw)
    with pytest.raises(ValueError, match=match):
        MultiagentZombsoleVectorEnv("evacuation", [], "city_for_evacuation", ["0", "1"], 20, num_envs=4, **kw)


def test_make_config_modes():
    cfgd = pu.CONFIGS["c1_bridge_ext"]
    for auto_reset, mode, want in [(False, "same_step", 0), (True, "same_step", 1), (True, "next_step", 2)]:
        cfg, _ = pu.build(cfgd, 4, 0, auto_reset=auto_reset)
        cfg2 = abi.make_config(cfgd["rules_name"], cfgd["player_names"], cfgd["agent_ids"], cfgd["agent_weapons"],
                               cfgd["initial_zombies"], cfgd["minimum_zombies"], abi.OBS_WORLD, abi.OBS_SIMPLE, 0, False, 4,
                               auto_reset=auto_reset, autoreset_mode=mode)
        assert cfg2.auto_reset == want and cfg.auto_reset == min(want, 1)
    with pytest.raises(ValueError, match="auto_reset=True"):
        abi.make_config("extermination", [], [0], "rifle", 1, 0, abi.OBS_WORLD, abi.OBS_SIMPLE, 0, False, 4,
                        auto_reset=False, autoreset_mode="next_step")


@gpu
def test_engine_refuses_final_observations():
    eng, cfg = _engine("c1_bridge_ext", 64, 0, 10, True)
    obs, fin = eng.new_obs(), eng.new_obs()
    rew, term, trunc = eng.new_outputs()
    acts = torch.zeros((64, 1), dtype=torch.int32, device=eng.device)
    with pytest.raises(Exception, match="next-step autoreset"):
        eng.step_final(acts, abi.ACTIONS_DISCRETE, obs, fin, rew, term, trunc)
    with pytest.raises(Exception, match="next-step autoreset"):
        eng.rollout(2, 0, None, abi.ACTIONS_DISCRETE, eng.new_obs(2), None, None, None, final_obs=eng.new_obs(2))
    eng.close()


# ---------------------------------------------------------------- kernel selection
# (in an interpreter of its own, as in tests/test_cuda_final_obs.py: profiler sessions in the pytest process disturb later ones)
_PROFILED_BENCH_LAUNCH = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import torch
from libzombsole_b200 import abi
from libzombsole_b200.engine import ZsEngine
import parity_util as pu
from test_cuda_roster import _kernels_launched
N, K = 4096, 20
cfg, m = pu.build(pu.CONFIGS["c1_bridge_ext"], N, 5, auto_reset=True, max_episode_steps=1000)
if sys.argv[2] == "1":
    cfg.auto_reset = abi.AUTORESET_NEXT_STEP
eng = ZsEngine(cfg, m)
obs = eng.new_obs()
rew, term, trunc = eng.new_outputs(K)
acts = torch.zeros((K, N, eng.A), dtype=torch.int32, device=eng.device)
names = _kernels_launched(lambda: eng.rollout(K, 0, acts, abi.ACTIONS_DISCRETE, obs, rew, term, trunc))
eng.close()
print(json.dumps(names))
"""


@gpu
@pytest.mark.parametrize("next_step", [False, True])
def test_bench_rollout_kernel(next_step):
    """bench.py's workload on a next-step handle runs the next-step world-scope kernel (SHAPE 8, one env per warp), never the
    standard rollout shape or a roster kernel; on a same-step handle it still runs the roster kernel."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    flags = ["-I"] if sys.flags.isolated else (["-s"] if sys.flags.no_user_site else [])
    run = subprocess.run([sys.executable] + flags + ["-c", _PROFILED_BENCH_LAUNCH, root, "1" if next_step else "0"], cwd=root,
                         capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stderr[-3000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    ros = 1 + abi.RULES["extermination"] + 4 * 3
    pat = re.compile(r"zs_sim_kernel<0, 16, 32, 8, \d+, 0>" if next_step else r"zs_sim_kernel<0, 16, (16|32), 1, \d+, %d>" % ros)
    assert names and all(pat.search(n) for n in names), names
