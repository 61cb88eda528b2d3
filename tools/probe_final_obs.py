"""What final observations cost in fused rollouts: zs_rollout_final against zs_rollout on the same engine, launches
alternating, CUDA events, milliseconds per fused step.  An env writes its final row only in the step that ends its episode,
so the measured share of env-steps that end one is printed beside the times.

For the bench game (config 1: bridge, extermination, agent + 2 terminators) a rollout with final observations runs the
generic world-scope kernel (SHAPE 6), not the standard-shape kernel (SHAPE 1, with the game's roster compiled in unless
ZS_NO_ROSTER=1).  So the cost of the final rows is timed on launches that take the generic kernel either way (actions drawn
inside the kernel: SHAPE 0 against SHAPE 6), and what a bench-shaped launch (an action tape in HBM) pays for asking is timed
against the roster kernel and against the standard-shape kernel without the roster (ZS_NO_ROSTER=1).

usage: python tools/probe_final_obs.py [reps]"""
import os
import sys

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


def make(name, N, roster):
    if roster:
        os.environ.pop("ZS_NO_ROSTER", None)
    else:
        os.environ["ZS_NO_ROSTER"] = "1"
    cfg, m = pu.build(pu.CONFIGS[name], N, 0, auto_reset=True, max_episode_steps=1000)
    return ZsEngine(cfg, m)


def run(name, N, K, reps):
    engines = {"roster": make(name, N, True)} if name == "c1_bridge_ext" else {}
    engines["plain"] = make(name, N, False)
    os.environ.pop("ZS_NO_ROSTER", None)
    first = next(iter(engines.values()))
    tape = torch.zeros((K, N, first.A), dtype=torch.int32, device=first.device)
    first.fill_synthetic_tape(3, tape)
    bufs = {}
    for key, eng in engines.items():
        obs, fin = eng.new_obs(), eng.new_obs()
        rew, term, trunc = eng.new_outputs(K)
        eng.rollout(3, 0, None, abi.ACTIONS_DISCRETE, obs, None, None, None)  # worlds in mid-episode
        bufs[key] = (obs, fin, rew, term, trunc)
    bench = "roster" in engines
    # (engine, final observations, action tape): the bench game's isolated comparison draws its actions in the kernel
    modes = [("plain", False, not bench), ("plain", True, not bench)]
    if bench:
        modes += [("plain", True, True), ("plain", False, True), ("roster", False, True)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {m: [] for m in modes}
    ends = []
    for r in range(reps + 1):  # (round 0 warms every mode up)
        for key, final, with_tape in modes:
            obs, fin, rew, term, trunc = bufs[key]
            torch.cuda.synchronize()
            ev[0].record()
            engines[key].rollout(K, 3, tape if with_tape else None, abi.ACTIONS_DISCRETE, obs, rew, term, trunc,
                                 final_obs=fin if final else None)
            ev[1].record()
            torch.cuda.synchronize()
            if r:
                times[(key, final, with_tape)].append(ev[0].elapsed_time(ev[1]) / K)
                if final:
                    ends.append(float((term | trunc).float().mean()))
    med = {m: float(np.median(v)) for m, v in times.items()}

    def fmt(m):
        return "%.4f [%.4f, %.4f]" % (med[m], min(times[m]), max(times[m]))

    a, b = modes[0], modes[1]
    line = "%-18s N=%7d K=%4d  ms/step: without %s  with %s  cost of the final rows %+.2f %%" % (
        name, N, K, fmt(a), fmt(b), 100.0 * (med[b] / med[a] - 1.0))
    if bench:
        w, s1, ros = ("plain", True, True), ("plain", False, True), ("roster", False, True)
        line += ("\n    bench-shaped (action tape): with final observations %s, standard kernel without the roster %s, roster "
                 "kernel %s: asking costs %+.2f %% against the roster kernel" % (fmt(w), fmt(s1), fmt(ros), 100.0 * (med[w] / med[ros] - 1.0)))
    line += "\n    env-steps ending an episode: 1 in %.1f" % (1.0 / max(1e-9, float(np.mean(ends))))
    print(line, flush=True)
    for eng in engines.values():
        eng.close()


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print("%s, power limit %s" % (torch.cuda.get_device_name(0), os.popen(
        "nvidia-smi --query-gpu=power.limit --format=csv,noheader").read().strip() or "not read"), flush=True)
    print("median [min, max] of %d launches per mode, alternating" % reps, flush=True)
    for name, N, K in CASES:
        run(name, N, K, reps)


if __name__ == "__main__":
    main()
