"""End-to-end host step of the multi-agent env at BASELINE config 3 (city_for_evacuation, 4 agents with rifles, 20 zombies,
channels, 21-wide windows): host_outputs=True (the kernel writes every agent's full window into pinned host memory) against
"compact-copy" and "compact" (one record per env crosses PCIe, the library's host threads expand it).

usage: python tools/probe_e2e_multi.py [N ...]   (default 4096 65536)
Per size and mode: microseconds per step() from box to box (host clock; step() returns synchronised, the host owns the
results), 50 warm-up and 300 timed steps of random discrete ids; mean and max entries per record; device-to-host bytes per
env and step (True: the rows, rewards, flags, mask and lives; "compact-copy": the whole record buffer; "compact": the words
the kernel writes, header and entries).  The device name and power limit are printed in the same run."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from libzombsole_b200.gym.multiagent_env import MultiagentZombsoleVectorEnv  # noqa: E402

KW = dict(rules_name="evacuation", player_names=[], map_name="city_for_evacuation", agent_ids=["0", "1", "2", "3"],
          initial_zombies=20, minimum_zombies=0, observation_surroundings_width=21, agent_weapons="rifle")
WARMUP, TIMED = 50, 300


def run(N, mode):
    env = MultiagentZombsoleVectorEnv(num_envs=N, seed=0, max_episode_steps=1000, host_outputs=mode, **KW)
    A = env.num_agents
    acts = torch.from_numpy(np.random.RandomState(0).randint(0, 7, size=(WARMUP + TIMED, N, A)).astype(np.int32)).pin_memory()
    for s in range(WARMUP):
        env.step(acts[s])
    torch.cuda.synchronize()
    ent_sum, ent_max, dt = 0.0, 0, 0.0
    over0 = getattr(env, "compact_overflows", 0)
    for s in range(TIMED):
        t0 = time.perf_counter()
        env.step(acts[WARMUP + s])
        dt += time.perf_counter() - t0
        if env.compact:  # (outside the clock)
            e = (env._records_host[:, 0] & 0xffff).float()
            ent_sum += e.mean().item()
            ent_max = max(ent_max, int(e.max().item()))
    us = dt / TIMED * 1e6
    row = env.engine.obs_elems * 4 + A * 8 + 2 + A + 2 * A
    if env.compact:
        hdr = 2 + 3 * A
        e_mean = ent_sum / TIMED
        d2h = env.compact_words * 4 if mode == "compact-copy" else (hdr + 2 * e_mean) * 4  # (channels: two words per entry)
        extra = "entries/record mean %.1f max %d  words %d  overflows %d" % (e_mean, ent_max, env.compact_words,
                                                                             env.compact_overflows - over0)
    else:
        d2h = row
        extra = ""
    print("N %6d  %-13s %9.1f us/step  %.3e env-steps/s  D2H %8.0f B/env/step  %s" % (N, repr(mode), us, N / us * 1e6, d2h, extra),
          flush=True)
    env.close()


def main():
    sizes = [int(v) for v in sys.argv[1:]] or [4096, 65536]
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print("device:", q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0))
    print("host threads available:", len(os.sched_getaffinity(0)))
    row = 4 * 3 * 21 * 21 * 4
    print("config 3 observation row: %d B per env (4 agents x 3 x 21 x 21 int32)" % row)
    for N in sizes:
        for mode in (True, "compact-copy", "compact"):
            run(N, mode)


if __name__ == "__main__":
    main()
