"""Final observations of auto-reset episodes (include/zs_b200.h: zs_step_final, zs_rollout_final; gymnasium's SAME_STEP
autoreset, info["final_obs"] / info["_final_obs"]).  An env whose step ends its episode is re-initialised in that step; the
observation of the world it ended in must be exactly what zs_step writes for that step on a handle without auto-reset.

* lockstep against a twin (same seed and env indices, auto_reset=False, stepped with step and then reset(mask)): final rows,
  observations, reward bits, flags, agent masks, draws and the state agree after every step;
* fused rollouts (K = 1, 7, 64, one ring slot per step) equal that twin stepped one step at a time, starting from the parked
  images and without them;
* asking for final observations changes nothing else: outputs, state and episode statistics are bit-identical;
* the final rows equal the oracle's observation taken after its step and before its reset;
* the vector envs' info keys (device and pinned host outputs), the multi-agent env, the refusals, and the kernel a
  bench-shaped rollout launches.
"""
import re

import numpy as np
import pytest
import torch

import parity_util as pu
from libzombsole_b200 import abi
from test_cuda_properties import assert_same_state, engine, state_snapshot

gpu = pytest.mark.gpu

# (config, envs): the lane layouts, both encodings and scopes, 128 and 256 slots, the respawn, randoman bots
LOCKSTEP = [("c1_bridge_ext", 512), ("c5_bridge_channels", 256), ("gym_surroundings", 256), ("surroundings_channels", 256),
            ("c3_city_evac", 128), ("c4_maze_safehouse", 64), ("fort_max_slots", 32), ("survival_minz", 128),
            ("bots_randoman", 128), ("bench_odd_cells", 256), ("bench_wide_max", 32), ("surr255_odd_cells", 16)]


def _twins(name, N, seed, mes):
    a, cfg, _ = engine(name, N, seed=seed, base=11, mes=mes, auto_reset=True)
    b, _, _ = engine(name, N, seed=seed, base=11, mes=mes, auto_reset=False)
    return a, b, cfg


def _bits(t):
    return t.view(torch.int64)


def _lockstep(a, b, cfg, T, first_action_step=0):
    """Steps a (step_final) and b (step + reset(mask)) T times; returns (terminations, time-limit truncations, other
    truncations) seen."""
    N, A = a.N, cfg.n_agents
    obs_a, fin_a, obs_b = a.new_obs(), a.new_obs(), b.new_obs()
    ra, ta, ua = a.new_outputs()
    rb, tb, ub = b.new_outputs()
    ma, mb = (torch.zeros((N, A), dtype=torch.uint8, device=a.device) for _ in range(2))
    da, db = (torch.zeros(N, dtype=torch.int32, device=a.device) for _ in range(2))
    acts = torch.zeros((N, A), dtype=torch.int32, device=a.device)
    n_term = n_limit = n_death = 0
    for t in range(T):
        a.fill_synthetic_actions(first_action_step + t, acts)
        fin_a.fill_(-7)
        a.step_final(acts, abi.ACTIONS_DISCRETE, obs_a, fin_a, ra, ta, ua, ma, da)
        b.step(acts, abi.ACTIONS_DISCRETE, obs_b, rb, tb, ub, mb, db)
        assert torch.equal(ta, tb) and torch.equal(ua, ub), "flags differ at step %d" % t
        assert torch.equal(_bits(ra), _bits(rb)), "reward bits differ at step %d" % t
        assert torch.equal(ma, mb) and torch.equal(da, db), "agent mask / draws differ at step %d" % t
        ended = (tb | ub).bool()
        assert torch.equal(fin_a[ended], obs_b[ended]), "final observation differs at step %d" % t
        if ended.any():
            steps = b.fields["scalars"][:, abi.S_EPISODE_STEPS]
            limit = ub.bool() & (steps >= cfg.max_episode_steps)
            n_term += int(tb.sum())
            n_limit += int(limit.sum())
            n_death += int((ub.bool() & ~limit).sum())
            b.reset(ended.to(torch.uint8), obs_b)
        assert torch.equal(obs_a, obs_b), "observation after the auto-reset differs at step %d" % t
        assert_same_state(state_snapshot(a), state_snapshot(b), a.M)
    return n_term, n_limit, n_death


@gpu
@pytest.mark.parametrize("mes", [9, 1000])
@pytest.mark.parametrize("name,N", LOCKSTEP)
def test_step_final_equals_step_then_masked_reset(name, N, mes):
    a, b, cfg = _twins(name, N, 41, mes)
    n_term, n_limit, n_death = _lockstep(a, b, cfg, 40 if mes == 9 else 80)
    if mes == 9:
        assert n_limit > 0, "no TimeLimit truncation happened"
    else:
        assert n_limit == 0
    a.close()
    b.close()


@gpu
@pytest.mark.parametrize("lanes", ["16", "32"])
def test_step_final_both_lane_layouts_all_endings(monkeypatch, lanes):
    """Config 1's game in each lane layout; terminations, TimeLimit truncations and truncations by the agent's death all
    occur (two envs per warp: one env of a warp ends while its partner goes on)."""
    monkeypatch.setenv("ZS_LANES_PER_ENV", lanes)
    a, b, cfg = _twins("c1_bridge_ext", 1024, 43, 60)
    assert a.lanes_per_env() == int(lanes) and b.lanes_per_env() == int(lanes)
    n_term, n_limit, n_death = _lockstep(a, b, cfg, 130)
    assert n_term > 0 and n_limit > 0 and n_death > 0, (n_term, n_limit, n_death)
    a.close()
    b.close()


def _rollout_vs_twin(name, N, K, seed=47, mes=9):
    a, b, cfg = _twins(name, N, seed, mes)
    A = cfg.n_agents
    tape = torch.zeros((K, N, A), dtype=torch.int32, device=a.device)
    for s in range(K):
        a.fill_synthetic_actions(200 + s, tape[s])
    ring, fin = a.new_obs(K), a.new_obs(K)
    fin.fill_(-7)
    ra, ta, ua = a.new_outputs(K)
    a.rollout(K, 0, tape, abi.ACTIONS_DISCRETE, ring, ra, ta, ua, final_obs=fin)
    obs_b = b.new_obs()
    rb, tb, ub = b.new_outputs()
    ended_any = False
    for s in range(K):
        b.step(tape[s], abi.ACTIONS_DISCRETE, obs_b, rb, tb, ub)
        assert torch.equal(ta[s], tb) and torch.equal(ua[s], ub), "flags differ at step %d" % s
        assert torch.equal(_bits(ra[s]), _bits(rb)), "reward bits differ at step %d" % s
        ended = (tb | ub).bool()
        assert torch.equal(fin[s][ended], obs_b[ended]), "final observation of step %d differs" % s
        if ended.any():
            ended_any = True
            b.reset(ended.to(torch.uint8), obs_b)
        assert torch.equal(ring[s], obs_b), "observation of step %d differs" % s
    assert_same_state(state_snapshot(a), state_snapshot(b), a.M)
    a.close()
    b.close()
    return ended_any


@gpu
@pytest.mark.parametrize("images", [True, False])
@pytest.mark.parametrize("K", [1, 7, 64])
@pytest.mark.parametrize("name,N,lanes", [("c1_bridge_ext", 1024, "16"), ("c1_bridge_ext", 1024, "32"),
                                          ("gym_surroundings", 256, "32"), ("c3_city_evac", 128, "32"),
                                          ("c4_maze_safehouse", 48, "32"), ("bench_odd_cells", 256, "16"),
                                          ("bench_wide_max", 32, "32")])
def test_rollout_final_equals_single_steps(monkeypatch, name, N, lanes, K, images):
    monkeypatch.setenv("ZS_LANES_PER_ENV", lanes)
    if not images:
        monkeypatch.setenv("ZS_IMAGE_MB", "0")
    # (TimeLimits shorter than the rollout: every env ends in it at least once)
    assert _rollout_vs_twin(name, N, K, mes={1: 1, 7: 4, 64: 9}[K])


@gpu
@pytest.mark.parametrize("name,N", [("c1_bridge_ext", 4096), ("c5_bridge_channels", 512), ("c3_city_evac", 256),
                                    ("c4_maze_safehouse", 64), ("fort_max_slots", 32), ("gym_surroundings", 512)])
def test_asking_for_final_observations_changes_nothing_else(name, N):
    """The same launches with and without final observations: observations, reward bits, flags, state and episode
    statistics are bit-identical.  (Config 1 at 4,096 envs is bench.py's shape: the roster kernel against SHAPE 6.)"""
    K, mes = 24, 10
    outs = []
    for final in (False, True):
        eng, cfg, _ = engine(name, N, seed=53, mes=mes)
        A = cfg.n_agents
        tape = torch.zeros((K, N, A), dtype=torch.int32, device=eng.device)
        for s in range(K):
            eng.fill_synthetic_actions(300 + s, tape[s])
        ring, fin = eng.new_obs(4), eng.new_obs(4)
        rew, term, trunc = eng.new_outputs(K)
        eng.rollout(K, 0, tape, abi.ACTIONS_DISCRETE, ring, rew, term, trunc, final_obs=fin if final else None)
        obs = eng.new_obs()
        r1, t1, u1 = eng.new_outputs(8)
        mask = torch.zeros((8, N, A), dtype=torch.uint8, device=eng.device)
        for s in range(8):
            if final:
                eng.step_final(tape[s], abi.ACTIONS_DISCRETE, obs, fin[0], r1[s], t1[s], u1[s], mask[s])
            else:
                eng.step(tape[s], abi.ACTIONS_DISCRETE, obs, r1[s], t1[s], u1[s], mask[s])
        outs.append(dict(ring=ring.clone(), obs=obs.clone(), rew=_bits(torch.cat([rew.flatten(), r1.flatten()])),
                         flags=torch.cat([term.flatten(), trunc.flatten(), t1.flatten(), u1.flatten()]), mask=mask.clone(),
                         stats=eng.episode_stats().clone(), state=state_snapshot(eng)))
        M = eng.M
        eng.close()
    a, b = outs
    for k in ("ring", "obs", "rew", "flags", "mask", "stats"):
        assert torch.equal(a[k], b[k]), k
    assert int(a["stats"][0]) > 0  # episodes ended (and were re-initialised) in these launches
    assert_same_state(a["state"], b["state"], M)


@gpu
@pytest.mark.parametrize("name,N", [("c1_bridge_ext", 256), ("c3_city_evac", 64)])
def test_final_rows_equal_the_oracle_before_its_reset(name, N):
    from oracle import oracle as orc
    cfgd = pu.CONFIGS[name]
    eng, cfg, m = engine(name, N, seed=59, base=5, mes=12)
    rcfg, _ = pu.build(cfgd, N, 59, env_index_base=5, max_episode_steps=12, auto_reset=False)
    ref = orc.OracleEnv(rcfg, m)
    A = cfg.n_agents
    obs, fin = eng.new_obs(), eng.new_obs()
    rew, term, trunc = eng.new_outputs()
    acts = torch.zeros((N, A), dtype=torch.int32, device=eng.device)
    n_ended = 0
    for t in range(40):
        eng.fill_synthetic_actions(t, acts)
        a = acts.cpu().numpy()
        eng.step_final(acts, abi.ACTIONS_DISCRETE, obs, fin, rew, term, trunc)
        _, r, te, tr, _, _ = ref.step(a, abi.ACTIONS_DISCRETE)
        assert np.array_equal(term.cpu().numpy(), te) and np.array_equal(trunc.cpu().numpy(), tr), "flags differ at step %d" % t
        ended = (te | tr).astype(bool)
        want = ref.encode_obs()
        assert np.array_equal(fin.cpu().numpy().reshape(N, -1)[ended], want[ended]), "final observation differs at step %d" % t
        if ended.any():
            n_ended += int(ended.sum())
            ref.reset(ended.astype(np.uint8))
        assert np.array_equal(obs.cpu().numpy().reshape(N, -1), ref.encode_obs()), "observation differs at step %d" % t
    assert n_ended > N  # every env ended at least once on average (TimeLimit 12 over 40 steps)
    eng.close()
    ref.close()


# ---------------------------------------------------------------- the Python layer
def _single_env(**kw):
    from libzombsole_b200.gym_env import make_vector
    return make_vector("jvstinian/Zombsole-v0", 256, seed=61, max_episode_steps=7, **kw)


@gpu
@pytest.mark.parametrize("host_outputs", [False, True])
def test_vector_env_info_keys(host_outputs):
    env = _single_env(final_observation=True, host_outputs=host_outputs)
    twin = _single_env(auto_reset=False, host_outputs=host_outputs)
    want_dev = "cpu" if host_outputs else "cuda"
    assert env.final_obs.shape == env.obs.shape and env.final_obs.device.type == want_dev
    if host_outputs:
        assert env.final_obs.is_pinned()
    env.reset()
    twin.reset()
    rs = np.random.RandomState(3)
    seen = 0
    for t in range(20):
        a = torch.from_numpy(rs.randint(0, 6, size=256).astype(np.int32))
        obs, rew, term, trunc, info = env.step(a)
        tobs, trew, tterm, ttrunc, _ = twin.step(a)
        assert set(info) == {"final_obs", "_final_obs"}
        fo, fm = info["final_obs"], info["_final_obs"]
        assert fo is env.final_obs and fo.dtype == torch.int32 and fo.device.type == want_dev
        assert fm.dtype == torch.bool and fm.shape == (256,) and fm.device.type == want_dev
        assert torch.equal(fm, term | trunc) and torch.equal(term, tterm) and torch.equal(trunc, ttrunc)
        assert torch.equal(fo[fm], tobs[fm]), "final observation differs at step %d" % t
        seen += int(fm.sum())
        if fm.any():
            twin.reset(mask=fm.to(torch.uint8))
        assert torch.equal(obs, tobs)
        assert torch.equal(_bits(rew), _bits(trew))
    assert seen > 256  # the TimeLimit of 7 steps ended every env at least twice
    # a fused rollout into a caller ring
    K = 9
    ring = torch.empty((K,) + tuple(env.obs.shape), dtype=torch.int32, device=env.device)
    fin = torch.empty_like(ring)
    rew, term, trunc = env.engine.new_outputs(K)
    env.rollout(K, obs=ring, reward=rew, terminated=term, truncated=trunc, final_obs=fin)
    torch.cuda.synchronize()
    assert bool((term | trunc).any())
    env.close()
    twin.close()


@gpu
@pytest.mark.parametrize("host_outputs", [False, True])
def test_multiagent_env_final_obs(host_outputs):
    from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
    cfgd = pu.CONFIGS["c3_city_evac"]
    args = (cfgd["rules_name"], cfgd["player_names"], cfgd["map_name"], cfgd["agent_ids"], cfgd["initial_zombies"],
            cfgd["minimum_zombies"])
    kw = dict(num_envs=64, seed=67, max_episode_steps=6, host_outputs=host_outputs)
    env = MultiagentZombsoleVectorEnv(*args, final_observation=True, **kw)
    twin = MultiagentZombsoleVectorEnv(*args, auto_reset=False, **kw)
    assert env.final_obs.shape == (64, 4, 3, 21, 21)
    rs = np.random.RandomState(5)
    seen = 0
    for t in range(15):
        a = torch.from_numpy(rs.randint(0, 7, size=(64, 4)).astype(np.int32))
        obs, rew, term, trunc, info = env.step(a)
        tobs, trew, tterm, ttrunc, tinfo = twin.step(a)
        assert set(info) == {"agent_mask", "final_obs", "_final_obs"}
        fm = info["_final_obs"]
        assert torch.equal(fm, term | trunc) and torch.equal(info["agent_mask"], tinfo["agent_mask"])
        assert torch.equal(info["final_obs"][fm], tobs[fm]), "final observation differs at step %d" % t
        seen += int(fm.sum())
        if fm.any():
            twin.reset(mask=fm.to(torch.uint8))
        assert torch.equal(obs, tobs) and torch.equal(_bits(rew), _bits(trew))
    assert seen >= 64
    env.close()
    twin.close()


@pytest.mark.parametrize("kw", [dict(auto_reset=False), dict(host_outputs="compact"), dict(host_outputs="compact-copy")])
def test_refusals(kw):
    """The argument combinations final observations cannot serve are refused before anything is allocated (no GPU needed)."""
    from libzombsole_b200.gym_env import ZombsoleVectorEnv, make_vector
    from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
    with pytest.raises(ValueError, match="final_observation"):
        make_vector("jvstinian/Zombsole-v0", 4, final_observation=True, **kw)
    with pytest.raises(ValueError, match="final_observation"):
        ZombsoleVectorEnv("extermination", [], "bridge", 0, 10, num_envs=4, final_observation=True, **kw)
    with pytest.raises(ValueError, match="final_observation"):
        MultiagentZombsoleVectorEnv("evacuation", [], "city_for_evacuation", ["0", "1"], 20, num_envs=4, final_observation=True, **kw)


@gpu
def test_engine_refusals():
    eng, cfg, _ = engine("c1_bridge_ext", 64, mes=10, auto_reset=False)
    obs, fin = eng.new_obs(), eng.new_obs()
    rew, term, trunc = eng.new_outputs()
    acts = torch.zeros((64, 1), dtype=torch.int32, device=eng.device)
    with pytest.raises(Exception, match="auto_reset"):
        eng.step_final(acts, abi.ACTIONS_DISCRETE, obs, fin, rew, term, trunc)
    with pytest.raises(ValueError, match="final_obs"):
        eng.rollout(2, 0, None, abi.ACTIONS_DISCRETE, None, None, None, None, final_obs=fin)
    with pytest.raises(ValueError, match="final_obs"):
        eng.rollout(2, 0, None, abi.ACTIONS_DISCRETE, eng.new_obs(2), None, None, None, final_obs=fin)
    eng.close()


# The profiled launch runs in an interpreter of its own: with this test's two torch.profiler sessions in the pytest process,
# the session of tests/test_cuda_roster.py that followed them in the same process recorded no kernels at all.
_PROFILED_BENCH_LAUNCH = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import torch
from libzombsole_b200 import abi
from test_cuda_properties import engine
from test_cuda_roster import _kernels_launched
final = sys.argv[2] == "1"
N, K = 4096, 20
eng, cfg, m = engine("c1_bridge_ext", N, seed=5)
obs, fin = eng.new_obs(), eng.new_obs()
rew, term, trunc = eng.new_outputs(K)
acts = torch.zeros((K, N, eng.A), dtype=torch.int32, device=eng.device)
names = _kernels_launched(lambda: eng.rollout(K, 0, acts, abi.ACTIONS_DISCRETE, obs, rew, term, trunc,
                                               final_obs=fin if final else None))
eng.close()
print(json.dumps(names))
"""


@gpu
@pytest.mark.parametrize("final", [False, True])
def test_bench_rollout_kernel(final):
    """bench.py's workload without final observations still runs the roster kernel; with them, the generic SHAPE 6 kernel."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    flags = ["-I"] if sys.flags.isolated else (["-s"] if sys.flags.no_user_site else [])  # (as this interpreter was started)
    run = subprocess.run([sys.executable] + flags + ["-c", _PROFILED_BENCH_LAUNCH, root, "1" if final else "0"], cwd=root,
                         capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stderr[-3000:]
    names = json.loads(run.stdout.strip().splitlines()[-1])
    ros = 1 + abi.RULES["extermination"] + 4 * 3
    pat = re.compile(r"zs_sim_kernel<0, 16, (16|32), 6, \d+, 0>" if final else r"zs_sim_kernel<0, 16, (16|32), 1, \d+, %d>" % ros)
    assert names and all(pat.search(n) for n in names), names
