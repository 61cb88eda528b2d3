"""One row per zs_sim_kernel instantiation launch_sim can launch: its template arguments <MODE, MPC, G, SHAPE, OCC, ROS> and a
recipe that reaches it (a CONFIGS game, a batch size, the zs_create switches that force the lane layout and the occupancy,
and the calls).

* the table equals the instantiations compiled into the library (cuobjdump; no GPU needed): a kernel added without a row,
  or a row without a kernel, fails here;
* each recipe launches its row's kernel and no other of its mode (torch.profiler, one interpreter for the whole table);
* each row agrees with the oracle bit for bit at every step: observations (every slot of a fused rollout's ring), float64
  reward bits, flags, agent masks, draws, final observations, expanded compact records, episode statistics and the state
  of a sample of envs; next-step rows against the composed twin of test_cuda_next_step.py, whose calls are rows here;
* every row reaches what it exists for: episodes end and worlds are re-initialised inside the launch, next-step reset steps
  happen, compact records are expanded (and, for one row per record kind, overflow);
* zs_create's own choices at the BASELINE per-GPU sizes, with no switches, are rows of the table.
"""
import collections
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import parity_util as pu
from libzombsole_b200 import abi

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MODE_STEP, MODE_RESET, MODE_ENCODE = 0, 1, 2
ROS_BENCH = 1 + abi.RULES["extermination"] + 4 * 3  # the bench game's roster (zs_world.cuh: ZS_ROSTER_BENCH)
KERNEL = re.compile(r"zs_sim_kernel<(\d+), (\d+), (\d+), (\d+), (\d+), (\d+)>")

# calls: "step" (CudaEngine.step with draws and agent mask, same-step auto-reset), "rollout" (one fused launch on a discrete
# tape, a ring slot per step), "compact" (a vector env with host_outputs="compact"), "final" (zs_step_final), "next"
# (next-step autoreset, zs_step), "next_compact" (a next-step vector env with host_outputs="compact"), "manual" (zs_step, then
# zs_reset of the ended envs; zs_encode_obs first).  over: a second compact env whose records are too small for most envs.
Recipe = collections.namedtuple("Recipe", "config N calls env T mes over")


def _recipe(config, N, calls, env=(), T=32, mes=11, over=False):
    return Recipe(config, N, tuple(calls.split("+")), tuple(sorted(env)), T, mes, over)


def _occ_env(G, occ):
    env = [("ZS_OCC", str(occ))]
    if G == 16 and occ != 4:
        env.append(("ZS_WARPS_PER_CTA", "4"))  # the CTA shape these kernels get at the batch sizes zs_create gives them
    return env


def _table():
    rows = []

    def add(mode, mpc, g, shape, occ, ros, recipe):
        rows.append(((mode, mpc, g, shape, occ, ros), recipe))

    # 16 slots, one env per warp (ZS_LANES_PER_ENV=32) and two (16)
    for g, occs in ((32, (4, 7)), (16, (4, 6, 7))):
        for occ in occs:
            env = [("ZS_LANES_PER_ENV", str(g))] + _occ_env(g, occ)
            first = occ == 4
            world = "c1_bridge_ext" if first else "c5_bridge_channels"
            surr = "gym_surroundings" if first else "surroundings_channels"
            add(0, 16, g, 0, occ, 0, _recipe(world, 256, "step+compact", env, over=first and g == 32))
            add(0, 16, g, 1, occ, 0, _recipe(world, 256, "rollout", env + [("ZS_NO_ROSTER", "1")]))
            add(0, 16, g, 1, occ, ROS_BENCH, _recipe(world, 256, "rollout", env))
            add(0, 16, g, 2, occ, 0, _recipe(surr, 128, "step", env))
            add(0, 16, g, 4, occ, 0, _recipe("multi_boxed_2p", 128, "compact", env))
            add(0, 16, g, 6, occ, 0, _recipe(world, 256, "final", env))
            add(0, 16, g, 7, occ, 0, _recipe(surr, 128, "final", env))
            if g == 32:  # (next-step autoreset runs one env per warp)
                add(0, 16, g, 8, occ, 0, _recipe(world, 256, "next", env))
                add(0, 16, g, 9, occ, 0, _recipe(surr, 128, "next", env))
                add(0, 16, g, 10, occ, 0, _recipe("multi_boxed_2p", 128, "next_compact", env))
    # the producer-warp variant (ZS_PRODUCER=1): two-env warps, four game warps and a producer per CTA
    add(0, 16, 16, 3, 4, 0, _recipe("c1_bridge_ext", 512, "rollout", [("ZS_LANES_PER_ENV", "16"), ("ZS_PRODUCER", "1")]))
    # 32 slots
    for occ in (4, 7):
        env = _occ_env(32, occ)
        first = occ == 4
        world = "bridge_world_32" if first else "fort_world_32"
        surr = "c3_city_evac" if first else "bots_mixed"
        agents = "c3_city_evac" if first else "village_evac_mixed"
        add(0, 32, 32, 0, occ, 0, _recipe(world, 128, "step+compact", env, over=first))
        add(0, 32, 32, 1, occ, 0, _recipe(world, 128, "rollout", env))
        add(0, 32, 32, 2, occ, 0, _recipe(surr, 64, "step", env))
        add(0, 32, 32, 4, occ, 0, _recipe(agents, 64, "compact", env, over=first))
        add(0, 32, 32, 6, occ, 0, _recipe(world, 128, "final", env))
        add(0, 32, 32, 7, occ, 0, _recipe(surr, 64, "final", env))
        add(0, 32, 32, 8, occ, 0, _recipe(world, 128, "next", env))
        add(0, 32, 32, 9, occ, 0, _recipe(surr, 64, "next", env))
        add(0, 32, 32, 10, occ, 0, _recipe(agents, 64, "next_compact", env, over=first))
    # more slots than lanes: the general kernels, at the one occupancy launch_sim runs them at
    for mpc, world, surr, n_w, n_s in ((128, "c4_maze_safehouse", "box_arena", 64, 64), (256, "fort_world_256", "fort_max_slots", 32, 16)):
        add(0, mpc, 32, 0, 6, 0, _recipe(world, n_w, "step", T=24, mes=9))
        add(0, mpc, 32, 2, 6, 0, _recipe(surr, n_s, "step", T=24, mes=9))
        add(0, mpc, 32, 5, 6, 0, _recipe(world, n_w, "compact", T=24, mes=9, over=mpc == 128))
        add(0, mpc, 32, 6, 6, 0, _recipe("general_odd_cells" if mpc == 128 else world, 96 if mpc == 128 else n_w, "final", T=24, mes=9))
        add(0, mpc, 32, 7, 6, 0, _recipe("randoman_crowd" if mpc == 128 else surr, 48 if mpc == 128 else n_s, "final", T=24, mes=9))
        add(0, mpc, 32, 8, 6, 0, _recipe(world, n_w, "next", T=24, mes=9))
        add(0, mpc, 32, 9, 6, 0, _recipe(surr, n_s, "next", T=24, mes=9))
        add(0, mpc, 32, 11, 6, 0, _recipe(world, n_w, "next_compact", T=24, mes=5, over=mpc == 128))
    # zs_reset / zs_encode_obs: one kernel per slot count and lane layout, world scope and surroundings
    for mpc, g, world, surr, n in ((16, 16, "c1_bridge_ext", "gym_surroundings", 128), (16, 32, "c1_bridge_ext", "gym_surroundings", 128),
                                   (32, 32, "bridge_world_32", "c3_city_evac", 64), (128, 32, "c4_maze_safehouse", "box_arena", 32),
                                   (256, 32, "fort_world_256", "fort_max_slots", 16)):
        env = [("ZS_LANES_PER_ENV", str(g))] if mpc == 16 else []
        for shape, name in ((0, world), (2, surr)):
            r = _recipe(name, n, "manual", env, T=24, mes=7)
            add(MODE_RESET, mpc, g, shape, 7, 0, r)
            add(MODE_ENCODE, mpc, g, shape, 7, 0, r)
    return rows


TABLE = _table()
ROWS = [args for args, _ in TABLE]
RECIPES = dict(TABLE)


def _row_id(args):
    return "<%s>" % ",".join(str(v) for v in args)


def _parse(names):
    out = []
    for n in names:
        m = KERNEL.search(n)
        assert m, n
        out.append(tuple(int(v) for v in m.groups()))
    return out


# ---------------------------------------------------------------- a. the table equals the library
def test_table_equals_the_library():
    from tools import compiler_report
    if not os.path.exists(compiler_report.CUOBJDUMP) or shutil.which("c++filt") is None:
        pytest.skip("cuobjdump / c++filt not available")
    from libzombsole_b200 import build
    lib = build.build_native()
    mangled = sorted(compiler_report.res_usage(lib))
    pretty = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.splitlines()
    compiled = _parse([p for p in pretty if "zs_sim_kernel" in p])
    assert len(set(ROWS)) == len(ROWS), "a row appears twice"
    assert len(compiled) == len(set(compiled))
    missing = sorted(set(compiled) - set(ROWS))
    extra = sorted(set(ROWS) - set(compiled))
    assert not missing, "compiled kernels without a row: %s" % [_row_id(a) for a in missing]
    assert not extra, "rows without a compiled kernel: %s" % [_row_id(a) for a in extra]
    assert sum(1 for a in ROWS if a[0] == MODE_STEP) == 76 and len(ROWS) == 96


def test_every_recipe_forces_its_dimensions():
    """(no GPU) The switches of each recipe are the ones that select its row: ZS_OCC where the occupancy is a choice, the
    lane layout at 16 slots, ZS_NO_ROSTER / ZS_PRODUCER for those variants, an even batch for two envs per warp."""
    for args, r in TABLE:
        mode, mpc, g, shape, occ, ros = args
        env = dict(r.env)
        cfgd = pu.CONFIGS[r.config]
        assert {"ZS_LANES_PER_ENV": str(g)}.items() <= env.items() if mpc == 16 else "ZS_LANES_PER_ENV" not in env, args
        if mode == MODE_STEP and mpc <= 32 and shape != 3:
            assert env.get("ZS_OCC") == str(occ), args
        assert ("ZS_NO_ROSTER" in env) == (shape == 1 and mpc == 16 and ros == 0), args
        assert ("ZS_PRODUCER" in env) == (shape == 3), args
        if g == 16:
            assert r.N % 2 == 0, args
        multi = cfgd["kind"] == "multi"
        surr = multi or cfgd["observation_scope"].startswith("surroundings")
        assert surr == ((mode == MODE_STEP and shape in (2, 4, 7, 9, 10)) or (mode != MODE_STEP and shape == 2)), args
        if shape in (4, 10):
            assert multi, args


# ---------------------------------------------------------------- the recipes
def _actions(rs, N, A, multi):
    return rs.randint(-1 if multi else 0, 7 if multi else 6, size=(N, A)).astype(np.int32)


def _obs_mask(obs, mask, A):
    """Multi-agent rows: the windows of agents alive before the step (as test_cuda_parity.lockstep compares them)."""
    return np.where(np.repeat(mask.astype(bool), obs.shape[1] // A, axis=1), obs, 0)


def _same(errs, what, got, want):
    if not np.array_equal(got, want):
        errs.append("%s differs at %s" % (what, np.argwhere(got != want)[:4].tolist() if got.shape == want.shape else "shape"))


def _records_agree(cu, ref, cfgd, tag):
    nf = pu.n_fixed_slots(cfgd)
    errs = []
    for e in range(0, cu.N, max(1, cu.N // 16)):
        errs += pu.compare_record("env%d %s" % (e, tag), ref.export(e), cu.export(e), nf, check_obs=False)
    return errs


def _call_step(r, seed, check):
    if check:
        from test_cuda_parity import lockstep
        seen = {}
        errs = lockstep(pu.CONFIGS[r.config], r.N, r.T, seed, base=5, mes=r.mes, auto_reset=True, seen=seen)
        assert not errs, "\n".join(errs[:3])
        assert seen["ended"] > 0  # episodes ended, and were re-initialised inside the step launch
        return
    from cuda_engine import CudaEngine
    cfg, m = pu.build(pu.CONFIGS[r.config], r.N, seed, max_episode_steps=r.mes, auto_reset=True)
    cu = CudaEngine(cfg, m)
    rs = np.random.RandomState(seed)
    for _ in range(3):
        cu.step(_actions(rs, r.N, cfg.n_agents, cfg.obs_per_agent), abi.ACTIONS_DISCRETE)
    cu.close()


def _call_rollout(r, seed, check):
    """One fused launch of T steps on a discrete tape with a ring of T observation slots, against the oracle stepped one step
    at a time (same-step auto-reset): every slot, reward bits and flags of every step, then the episode statistics and the
    state of a sample of envs."""
    import torch
    from cuda_engine import CudaEngine
    from oracle import oracle as orc
    cfgd = pu.CONFIGS[r.config]
    cfg, m = pu.build(cfgd, r.N, seed, env_index_base=3, max_episode_steps=r.mes, auto_reset=True)
    cu = CudaEngine(cfg, m)
    eng, N, A, K = cu.eng, r.N, cfg.n_agents, r.T
    multi = cfgd["kind"] == "multi"
    rs = np.random.RandomState(seed)
    tape = np.stack([_actions(rs, N, A, multi) for _ in range(K)])
    ring = eng.new_obs(K)
    rew, term, trunc = eng.new_outputs(K)
    eng.rollout(K, 0, torch.from_numpy(tape).to(eng.device), abi.ACTIONS_DISCRETE, ring, rew, term, trunc)
    if not check:
        cu.close()
        return
    ref = orc.OracleEnv(cfg, m)
    ring, rew = ring.cpu().numpy().reshape(K, N, -1), rew.cpu().numpy().reshape(K, N, -1)
    term, trunc = term.cpu().numpy(), trunc.cpu().numpy()
    errs = []
    for s in range(K):
        o, rw, te, tr, mk, _ = ref.step(tape[s], abi.ACTIONS_DISCRETE)
        got = _obs_mask(ring[s], mk, A) if multi else ring[s]
        _same(errs, "observation of step %d" % s, got, _obs_mask(o, mk, A) if multi else o)
        _same(errs, "reward bits of step %d" % s, rew[s].view(np.uint64), rw.view(np.uint64))
        _same(errs, "terminated of step %d" % s, term[s], te)
        _same(errs, "truncated of step %d" % s, trunc[s], tr)
        if errs:
            break
    stats = eng.episode_stats().cpu().numpy()
    if not errs:
        _same(errs, "episode statistics", stats, ref.stats())
        errs += _records_agree(cu, ref, cfgd, "after the rollout")
    cu.close()
    ref.close()
    assert not errs, "\n".join(errs[:3])
    assert (term | trunc).any() and stats[0] > 0  # episodes ended and were re-initialised inside the launch


def _vector_env(cfgd, N, seed, mes, **kw):
    if cfgd["kind"] == "multi":
        from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv
        return MultiagentZombsoleVectorEnv(cfgd["rules_name"], cfgd["player_names"], cfgd["map_name"], cfgd["agent_ids"],
                                           cfgd["initial_zombies"], cfgd["minimum_zombies"],
                                           observation_surroundings_width=cfgd["surroundings_width"],
                                           agent_weapons=cfgd["agent_weapons"], num_envs=N, seed=seed, max_episode_steps=mes, **kw)
    from libzombsole_b200.gym_env import ZombsoleVectorEnv
    return ZombsoleVectorEnv(cfgd["rules_name"], cfgd["player_names"], cfgd["map_name"], cfgd["agent_ids"][0],
                             cfgd["initial_zombies"], cfgd["minimum_zombies"], observation_scope=cfgd["observation_scope"],
                             observation_position_encoding=cfgd["observation_position_encoding"],
                             agent_weapon=cfgd["agent_weapons"], num_envs=N, seed=seed, max_episode_steps=mes, **kw)


def _small_words(cfgd):
    """Records with room for 8 entries: most envs overflow and have their full rows fetched."""
    return 2 + 3 * len(cfgd["agent_ids"]) + 8 if cfgd["kind"] == "multi" else 4 + 8


def _call_compact(r, seed, check):
    """Vector envs with host_outputs="compact" (zs_step_host / zs_step_host_agents) against the oracle, step after step: the
    expanded observations, reward bits, flags and agent masks, then the episode statistics and the state of a sample."""
    import torch
    from cuda_engine import CudaEngine
    from oracle import oracle as orc
    cfgd = pu.CONFIGS[r.config]
    multi = cfgd["kind"] == "multi"
    kws = [dict(host_outputs="compact")] + ([dict(host_outputs="compact", compact_words=_small_words(cfgd))] if r.over else [])
    envs = [_vector_env(cfgd, r.N, seed, r.mes, **kw) for kw in kws]
    N, A = r.N, envs[0].cfg.n_agents
    ref = orc.OracleEnv(envs[0].cfg, cfgd["map_name"]) if check else None
    rs = np.random.RandomState(seed)
    errs = []
    for env in envs:
        o0, _ = env.reset()
        if check:
            _same(errs, "reset observation", o0.numpy().reshape(N, -1), ref.encode_obs() if env is not envs[0] else ref.reset())
    ended = 0
    for t in range(r.T if check else 3):
        a = _actions(rs, N, A, multi)
        want = ref.step(a, abi.ACTIONS_DISCRETE) if check else None
        for i, env in enumerate(envs):
            o, rw, te, tr, info = env.step(torch.from_numpy(a.reshape(N) if not multi else a).contiguous())
            if not check:
                continue
            tag = " of step %d (env %d)" % (t, i)
            o = o.numpy().reshape(N, -1)
            if multi:
                _same(errs, "agent mask" + tag, info["agent_mask"].numpy().astype(np.uint8), want[4])
            _same(errs, "observation" + tag, _obs_mask(o, want[4], A) if multi else o, _obs_mask(want[0], want[4], A) if multi else want[0])
            _same(errs, "reward bits" + tag, rw.numpy().reshape(N, -1).view(np.uint64), want[1].view(np.uint64))
            _same(errs, "flags" + tag, np.stack([te.numpy(), tr.numpy()]).astype(np.uint8), np.stack([want[2], want[3]]))
        if errs:
            break
        if check:
            ended += int((want[2] | want[3]).sum())
    if check and not errs:
        for env in envs:
            _same(errs, "episode statistics", env.engine.episode_stats().cpu().numpy(), ref.stats())
        errs += _records_agree(CudaEngine.of(envs[0].engine), ref, cfgd, "after the steps")
    overflows = [env.compact_overflows for env in envs]
    for env in envs:
        env.close()
    if not check:
        return
    ref.close()
    assert not errs, "\n".join(errs[:3])
    assert ended > 0
    assert overflows[0] < N * r.T  # records were expanded (an env-step whose record overflowed is fetched instead)
    if r.over:
        assert 0 < overflows[1] < N * r.T  # the overflow path ran, next to expanded records


def _call_final(r, seed, check):
    """zs_step_final against the oracle without auto-reset: the final rows of the envs a step ended are the oracle's
    observation after its step and before its reset (test_cuda_final_obs.test_final_rows_equal_the_oracle_before_its_reset)."""
    import torch
    from libzombsole_b200.engine import ZsEngine
    from oracle import oracle as orc
    cfgd = pu.CONFIGS[r.config]
    N = r.N
    cfg, m = pu.build(cfgd, N, seed, env_index_base=5, max_episode_steps=r.mes, auto_reset=True)
    eng = ZsEngine(cfg, m)
    rcfg, _ = pu.build(cfgd, N, seed, env_index_base=5, max_episode_steps=r.mes, auto_reset=False)
    ref = orc.OracleEnv(rcfg, m) if check else None
    obs, fin = eng.new_obs(), eng.new_obs()
    rew, term, trunc = eng.new_outputs()
    mask = torch.zeros((N, cfg.n_agents), dtype=torch.uint8, device=eng.device)
    draws = torch.zeros(N, dtype=torch.int32, device=eng.device)
    acts = torch.zeros((N, cfg.n_agents), dtype=torch.int32, device=eng.device)
    n_ended = 0
    for t in range(r.T if check else 3):
        eng.fill_synthetic_actions(t, acts)
        fin.fill_(-7)
        eng.step_final(acts, abi.ACTIONS_DISCRETE, obs, fin, rew, term, trunc, mask, draws)
        if not check:
            continue
        o, rw, te, tr, mk, dr = ref.step(acts.cpu().numpy(), abi.ACTIONS_DISCRETE)
        assert np.array_equal(term.cpu().numpy(), te) and np.array_equal(trunc.cpu().numpy(), tr), "flags differ at step %d" % t
        assert np.array_equal(rew.cpu().numpy().reshape(N, -1).view(np.uint64), rw.view(np.uint64)), "reward bits differ at step %d" % t
        assert np.array_equal(mask.cpu().numpy(), mk) and np.array_equal(draws.cpu().numpy(), dr), "agent mask / draws differ at step %d" % t
        ended = (te | tr).astype(bool)
        want = ref.encode_obs()
        assert np.array_equal(fin.cpu().numpy().reshape(N, -1)[ended], want[ended]), "final observation differs at step %d" % t
        if ended.any():
            n_ended += int(ended.sum())
            ref.reset(ended.astype(np.uint8))
        assert np.array_equal(obs.cpu().numpy().reshape(N, -1), ref.encode_obs()), "observation differs at step %d" % t
    eng.close()
    if check:
        ref.close()
        assert n_ended > 0  # episodes ended, and their worlds were re-initialised inside the step launch


def _call_next(r, seed, check):
    """Next-step autoreset against the composed twin (zs_step_masked / zs_reset of an auto_reset = 0 handle)."""
    import torch
    from test_cuda_next_step import Pair, _engine
    if not check:
        eng, cfg = _engine(r.config, r.N, seed, r.mes, True)
        o = eng.new_obs()
        rew, term, trunc = eng.new_outputs()
        acts = torch.zeros((r.N, cfg.n_agents), dtype=torch.int32, device=eng.device)
        for t in range(3):
            eng.fill_synthetic_actions(t, acts)
            eng.step(acts, abi.ACTIONS_DISCRETE, o, rew, term, trunc)
        eng.close()
        return
    pr = Pair(r.config, r.N, seed, r.mes)
    for t in range(r.T):
        pr.step(t)
    pr.check_stats()
    n = pr.n_reset_steps
    pr.close()
    assert n > 0  # reset steps happened


def _call_next_compact(r, seed, check):
    from test_cuda_next_step import _env_paths_vs_twin
    cfgd = pu.CONFIGS[r.config]
    multi = cfgd["kind"] == "multi"
    A = len(cfgd["agent_ids"])

    def make(**kw):
        return _vector_env(cfgd, r.N, seed, r.mes, **kw)

    paths = [dict(host_outputs="compact")] + ([dict(host_outputs="compact", compact_words=_small_words(cfgd))] if r.over else [])
    if not check:
        import torch
        env = make(autoreset_mode="next_step", **paths[0])
        env.reset()
        for t in range(3):
            env.step(torch.zeros((r.N, A) if multi else (r.N,), dtype=torch.int32))
        env.close()
        return
    overflows = _env_paths_vs_twin(make, paths, r.N, A, 7 if multi else 6, T=r.T)
    assert overflows[0] < r.N * r.T  # records were expanded
    if r.over:
        assert 0 < overflows[1] < r.N * r.T


def _call_manual(r, seed, check):
    """zs_encode_obs of the fresh worlds, then zs_step and zs_reset of the envs each step ended."""
    if check:
        from test_cuda_parity import lockstep
        seen = {}
        errs = lockstep(pu.CONFIGS[r.config], r.N, r.T, seed, base=9, mes=r.mes, seen=seen)
        assert not errs, "\n".join(errs[:3])
        assert seen["ended"] > 0  # worlds were re-initialised by zs_reset
        return
    from cuda_engine import CudaEngine
    cfg, m = pu.build(pu.CONFIGS[r.config], r.N, seed, max_episode_steps=r.mes)
    cu = CudaEngine(cfg, m)
    cu.encode_obs()
    cu.reset(np.arange(r.N) % 2)
    cu.close()


CALLS = dict(step=_call_step, rollout=_call_rollout, compact=_call_compact, final=_call_final, next=_call_next,
             next_compact=_call_next_compact, manual=_call_manual)


def _seed(args):
    return 1 + ROWS.index(args) * 7919


def run_recipe(args, check):
    r = RECIPES[args]
    for call in r.calls:
        CALLS[call](r, _seed(args), check)


# ---------------------------------------------------------------- b. each recipe launches its kernel
ZS_SWITCHES = ("ZS_OCC", "ZS_LANES_PER_ENV", "ZS_WARPS_PER_CTA", "ZS_NO_ROSTER", "ZS_PRODUCER")

# zs_create's choices at the BASELINE per-GPU sizes, no switches: (config, envs, compact host step?) -> kernels of each call
PRODUCTION = {
    "config2": ("c1_bridge_ext", 4096, False),
    "config3": ("c3_city_evac", 65536, True),
    "config4": ("c4_maze_safehouse", 131072, True),
    "config5": ("c1_bridge_ext", 1048576, False),
}


def _production_launches(kernels_launched):
    import torch
    from libzombsole_b200.engine import ZsEngine
    out = {}
    for key, (name, N, compact) in PRODUCTION.items():
        cfgd = pu.CONFIGS[name]
        cfg, m = pu.build(cfgd, N, 1, max_episode_steps=1000, auto_reset=True)
        eng = ZsEngine(cfg, m)
        K, A = 2, cfg.n_agents
        ring = eng.new_obs(K)
        rew, term, trunc = eng.new_outputs(K)
        tape = torch.zeros((K, N, A), dtype=torch.int32, device=eng.device)
        eng.fill_synthetic_tape(0, tape)
        out[key + " rollout"] = kernels_launched(lambda: eng.rollout(K, 0, tape, abi.ACTIONS_DISCRETE, ring, rew, term, trunc))
        del ring
        obs = eng.new_obs()
        r1, t1, u1 = eng.new_outputs()
        out[key + " step"] = kernels_launched(lambda: eng.step(tape[0], abi.ACTIONS_DISCRETE, obs, r1, t1, u1))
        eng.close()
        del obs
        if compact:
            env = _vector_env(cfgd, N, 1, 1000, host_outputs="compact")
            env.reset()
            a = torch.zeros((N, A) if cfgd["kind"] == "multi" else (N,), dtype=torch.int32)
            out[key + " compact"] = kernels_launched(lambda: env.step(a))
            env.close()
        torch.cuda.empty_cache()
    return out


def launch_sweep():
    """Every recipe once, without the oracle, under torch.profiler: {row id: [kernel names]}; then the production choices."""
    from test_cuda_roster import _kernels_launched
    for k in list(os.environ):
        if k.startswith("ZS_"):
            del os.environ[k]
    out = {}
    for args in ROWS:
        env = dict(RECIPES[args].env)
        os.environ.update(env)
        try:
            out[_row_id(args)] = _kernels_launched(lambda: run_recipe(args, check=False))
        finally:
            for k in env:
                del os.environ[k]
    out["production"] = _production_launches(_kernels_launched)
    return out


_SWEEP = r"""
import json, sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import test_cuda_kernel_matrix as km
print(json.dumps(km.launch_sweep()))
"""


@pytest.fixture(scope="module")
def launched():
    """(in an interpreter of its own, as in tests/test_cuda_final_obs.py: profiler sessions in the pytest process disturb later ones)"""
    flags = ["-I"] if sys.flags.isolated else (["-s"] if sys.flags.no_user_site else [])
    env = {k: v for k, v in os.environ.items() if not k.startswith("ZS_")}
    run = subprocess.run([sys.executable] + flags + ["-c", _SWEEP, ROOT], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=1800)
    assert run.returncode == 0, run.stderr[-3000:]
    return json.loads(run.stdout.strip().splitlines()[-1])


@gpu
@pytest.mark.parametrize("args", ROWS, ids=_row_id)
def test_recipe_launches_its_kernel(launched, args):
    got = [a for a in _parse(launched[_row_id(args)]) if a[0] == args[0]]
    assert got and all(a == args for a in got), sorted(set(_row_id(a) for a in got))


# what zs_create picks at the BASELINE sizes (one env per warp for the short launches of 4,096 bridge envs, two per warp
# and 6 CTAs per SM at 1,048,576; the occupancy of batches of three rounds or more at 65,536 city envs)
PRODUCTION_KERNELS = {
    "config2 rollout": (0, 16, 32, 1, 7, ROS_BENCH), "config2 step": (0, 16, 32, 1, 7, ROS_BENCH),
    "config3 rollout": (0, 32, 32, 2, 7, 0), "config3 step": (0, 32, 32, 2, 7, 0), "config3 compact": (0, 32, 32, 4, 7, 0),
    "config4 rollout": (0, 128, 32, 0, 6, 0), "config4 step": (0, 128, 32, 0, 6, 0), "config4 compact": (0, 128, 32, 5, 6, 0),
    "config5 rollout": (0, 16, 16, 1, 6, ROS_BENCH), "config5 step": (0, 16, 16, 1, 6, ROS_BENCH),
}


@gpu
@pytest.mark.parametrize("key", sorted(PRODUCTION_KERNELS))
def test_production_choices_are_rows(launched, key):
    got = _parse(launched["production"][key])
    steps = [a for a in got if a[0] == MODE_STEP]
    assert got and all(a in RECIPES for a in got), [_row_id(a) for a in got]
    assert steps and all(a == PRODUCTION_KERNELS[key] for a in steps), sorted(set(_row_id(a) for a in steps))


# ---------------------------------------------------------------- c. each row agrees with the oracle
@gpu
@pytest.mark.parametrize("args", ROWS, ids=_row_id)
def test_row_matches_the_oracle(monkeypatch, args):
    for k in list(os.environ):
        if k.startswith("ZS_"):
            monkeypatch.delenv(k)
    for k, v in RECIPES[args].env:
        monkeypatch.setenv(k, v)
    run_recipe(args, check=True)
