"""End-to-end host step of BASELINE config 4's game (safehouse on maze_for_safehouse, 1 agent with a rifle, 100 zombies,
world observation (1, 39, 72) — 101 slots, so the general step kernels): host_outputs=True (the kernel writes every full
observation row into pinned host memory) against "compact-copy" and "compact" (one record per env crosses PCIe, the
library's host threads expand it).

usage: python tools/probe_e2e_world.py [N:enc ...]   (default 4096:simple 131072:simple 4096:channels)
Per size, encoding and mode: microseconds per step() from box to box (host clock; step() returns synchronised, the host owns
the results), warm-up and timed steps of random discrete ids; mean and max entries per record; record words and overflows;
device-to-host bytes per env and step (True: the row, reward and flags; "compact-copy": the whole record buffer; "compact":
the words the kernel writes, header and entries); for "compact", where zs_step_host's time goes (zs_step_host_stats: the
flag is the moment the last record is in host memory, what follows it is the host threads' expansion).  The device name and
power limit are printed in the same run."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from libzombsole_b200.gym_env import ZombsoleVectorEnv  # noqa: E402

KW = dict(rules_name="safehouse", player_names=[], map_name="maze_for_safehouse", agent_id=0, initial_zombies=100,
          minimum_zombies=0, observation_scope="world", agent_weapon="rifle")


def run(N, enc, mode):
    warmup, timed = (50, 300) if N <= 16384 else (20, 100)
    env = ZombsoleVectorEnv(num_envs=N, seed=0, max_episode_steps=1000, host_outputs=mode,
                            observation_position_encoding=enc, **KW)
    assert env.engine.fields["life"].shape[1] > 32
    acts = torch.from_numpy(np.random.RandomState(0).randint(0, 6, size=(warmup + timed, N)).astype(np.int32)).pin_memory()
    for s in range(warmup):
        env.step(acts[s])
    torch.cuda.synchronize()
    ent_sum, ent_max, dt = 0.0, 0, 0.0
    over0 = getattr(env, "compact_overflows", 0)
    if env.streamed:
        env.engine.step_host_stats()  # (read and cleared: the stats below cover the timed steps only)
    for s in range(timed):
        t0 = time.perf_counter()
        env.step(acts[warmup + s])
        dt += time.perf_counter() - t0
        if env.compact:  # (outside the clock)
            e = (env._records_host[:, 0] & 0xffff).float()
            ent_sum += e.mean().item()
            ent_max = max(ent_max, int(e.max().item()))
    us = dt / timed * 1e6
    wpe = 1 if enc == "simple" else 2
    if env.compact:
        e_mean = ent_sum / timed
        d2h = env.compact_words * 4 if mode == "compact-copy" else (4 + wpe * e_mean) * 4
        extra = "entries/record mean %.1f max %d  words %d  overflows %d" % (e_mean, ent_max, env.compact_words,
                                                                             env.compact_overflows - over0)
        if env.streamed:
            _, launched, restored, flag, ret = env.engine.step_host_stats()
            extra += "\n          zs_step_host, us from entry: launches issued %.0f, previous cells restored %.0f, records in host " \
                     "memory (flag) %.0f, return %.0f" % (launched, restored, flag, ret)
    else:
        d2h = env.engine.obs_elems * 4 + 8 + 2
        extra = ""
    print("N %6d  %-8s %-14s %10.1f us/step  %.3e env-steps/s  D2H %8.0f B/env/step  %s" % (
        N, enc, repr(mode), us, N / us * 1e6, d2h, extra), flush=True)
    env.close()


def main():
    runs = [(int(a.split(":")[0]), a.split(":")[1]) for a in sys.argv[1:]] or [(4096, "simple"), (131072, "simple"),
                                                                             (4096, "channels")]
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print("device:", q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0))
    print("host threads available:", len(os.sched_getaffinity(0)))
    print("config 4 observation row: 11232 B per env in the simple encoding (1 x 39 x 72 int32), 33696 B in channels")
    for N, enc in runs:
        for mode in (True, "compact-copy", "compact"):
            run(N, enc, mode)


if __name__ == "__main__":
    main()
