"""What next-step autoreset costs: the same launches on a same-step handle and on a next-step handle (ZS_AUTORESET_NEXT_STEP),
alternating, CUDA events, median milliseconds per fused step; and microseconds per ZombsoleVectorEnv.step() from host actions
to host outputs with host_outputs="compact" (zs_step_host), alternating blocks of steps.

A next-step handle runs one env per warp in every launch.  For the bench game (config 1: bridge, extermination, agent + 2
terminators; at most 16 slots, so a same-step handle of 4,096 envs packs two per warp in fused rollouts) the rows separate
the two parts of the cost: same-step with two envs per warp (SHAPE 0, G = 16), same-step with one env per warp
(ZS_LANES_PER_ENV=32, SHAPE 0, G = 32), next-step (SHAPE 8, G = 32), all with actions drawn in the kernel; and a bench-shaped
launch (an action tape in HBM), which on a same-step handle runs the roster kernel.

usage: python tools/probe_next_step.py [reps]"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import parity_util as pu
from libzombsole_b200 import abi
from libzombsole_b200.engine import ZsEngine

CASES = [("c1_bridge_ext", 4096, 20), ("c1_bridge_ext", 4096, 512), ("c3_city_evac", 65536, 20),
         ("c4_maze_safehouse", 131072, 20)]


def make(name, N, next_step, lanes=None):
    if lanes:
        os.environ["ZS_LANES_PER_ENV"] = lanes
    cfg, m = pu.build(pu.CONFIGS[name], N, 0, auto_reset=True, max_episode_steps=1000)
    if next_step:
        cfg.auto_reset = abi.AUTORESET_NEXT_STEP
    eng = ZsEngine(cfg, m)
    os.environ.pop("ZS_LANES_PER_ENV", None)
    return eng


def fused(name, N, K, reps):
    engines = {"same-step": make(name, N, False), "next-step": make(name, N, True)}
    bench = name == "c1_bridge_ext"
    if bench:
        engines["same-step, one env per warp"] = make(name, N, False, "32")
    first = engines["same-step"]
    tape = torch.zeros((K, N, first.A), dtype=torch.int32, device=first.device)
    first.fill_synthetic_tape(3, tape)
    bufs = {}
    for key, eng in engines.items():
        obs = eng.new_obs()
        rew, term, trunc = eng.new_outputs(K)
        eng.rollout(3, 0, None, abi.ACTIONS_DISCRETE, obs, None, None, None)  # worlds in mid-episode
        bufs[key] = (obs, rew, term, trunc)
    # (engine, action tape)
    modes = [(key, False) for key in engines]
    if bench:
        modes += [("same-step", True), ("next-step", True)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {m: [] for m in modes}
    ends = []
    for r in range(reps + 1):  # (round 0 warms every mode up)
        for key, with_tape in modes:
            obs, rew, term, trunc = bufs[key]
            torch.cuda.synchronize()
            ev[0].record()
            engines[key].rollout(K, 3, tape if with_tape else None, abi.ACTIONS_DISCRETE, obs, rew, term, trunc)
            ev[1].record()
            torch.cuda.synchronize()
            if r:
                times[(key, with_tape)].append(ev[0].elapsed_time(ev[1]) / K)
                if key == "next-step":
                    ends.append(float((term | trunc).float().mean()))
    med = {m: float(np.median(v)) for m, v in times.items()}

    def fmt(m):
        return "%.4f [%.4f, %.4f]" % (med[m], min(times[m]), max(times[m]))

    lanes = {key: eng.lanes_per_env() for key, eng in engines.items()}
    base = ("same-step", False)
    print("%-18s N=%7d K=%4d  ms per fused step, actions drawn in the kernel:" % (name, N, K), flush=True)
    for m in modes:
        if not m[1]:
            print("    %-30s %d lanes per env  %s  %+.2f %%" % (m[0], lanes[m[0]], fmt(m), 100.0 * (med[m] / med[base] - 1.0)), flush=True)
    if bench:
        a, b = ("same-step", True), ("next-step", True)
        print("    bench-shaped (action tape): same-step (roster kernel) %s, next-step %s: %+.2f %%" % (
            fmt(a), fmt(b), 100.0 * (med[b] / med[a] - 1.0)), flush=True)
    print("    next-step env-steps ending an episode: 1 in %.1f" % (1.0 / max(1e-9, float(np.mean(ends)))), flush=True)
    for eng in engines.values():
        eng.close()


def host_steps(N, reps, block=200):
    from libzombsole_b200.gym_env import ZombsoleVectorEnv
    cfgd = pu.CONFIGS["c1_bridge_ext"]
    args = (cfgd["rules_name"], cfgd["player_names"], cfgd["map_name"], cfgd["agent_ids"][0], cfgd["initial_zombies"],
            cfgd["minimum_zombies"])
    envs = {mode: ZombsoleVectorEnv(*args, num_envs=N, seed=1, max_episode_steps=1000, host_outputs="compact",
                                    autoreset_mode=mode) for mode in ("same_step", "next_step")}
    rs = np.random.RandomState(0)
    acts = [torch.from_numpy(rs.randint(0, 6, size=N).astype(np.int32)) for _ in range(block)]
    times = {mode: [] for mode in envs}
    for env in envs.values():
        env.reset()
    for r in range(reps + 1):
        for mode, env in envs.items():
            per = []
            for a in acts:
                t0 = time.perf_counter()
                env.step(a)
                per.append(time.perf_counter() - t0)
            if r:
                times[mode].extend(per)
    med = {m: 1e6 * float(np.median(v)) for m, v in times.items()}
    print("ZombsoleVectorEnv.step(), host_outputs='compact', bridge game, %d envs: median us per step over %d steps each, "
          "blocks of %d alternating" % (N, len(times["same_step"]), block), flush=True)
    for m in envs:
        print("    %-10s %.1f us" % (m, med[m]), flush=True)
    print("    next-step %+.2f %%" % (100.0 * (med["next_step"] / med["same_step"] - 1.0)), flush=True)
    for env in envs.values():
        env.close()


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print("%s, power limit %s" % (torch.cuda.get_device_name(0), os.popen(
        "nvidia-smi --query-gpu=power.limit --format=csv,noheader").read().strip() or "not read"), flush=True)
    print("median [min, max] of %d launches per mode, alternating" % reps, flush=True)
    for name, N, K in CASES:
        fused(name, N, K, reps)
    host_steps(4096, reps)


if __name__ == "__main__":
    main()
