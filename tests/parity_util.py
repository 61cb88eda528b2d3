"""Shared helpers of the parity tests: config dicts, action tapes, record comparison."""
import os

import numpy as np

from libzombsole_b200 import abi

#: test-only maps (the reference takes an absolute path as map_name: os.path.join keeps it, gym_env.py:54-56)
MAPS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "maps")

#: parity configurations: BASELINE.json's five configs at small N, plus edge-case variants
CONFIGS = {
    # config 1/2/5: bridge, extermination, 10 zombies, agent + 2 terminators
    "c1_bridge_ext": dict(kind="single", rules_name="extermination", player_names=["terminator", "terminator"],
                          map_name="bridge", agent_ids=[0], agent_weapons="rifle", initial_zombies=10,
                          minimum_zombies=0, observation_scope="world", observation_position_encoding="simple"),
    "c5_bridge_channels": dict(kind="single", rules_name="extermination", player_names=["terminator", "terminator"],
                               map_name="bridge", agent_ids=[0], agent_weapons="rifle", initial_zombies=10,
                               minimum_zombies=0, observation_scope="world", observation_position_encoding="channels"),
    # the registered gym ids: agent alone (gym_env.py:382-414)
    "gym_v0_alone": dict(kind="single", rules_name="extermination", player_names=[], map_name="bridge", agent_ids=[0],
                         agent_weapons="rifle", initial_zombies=10, minimum_zombies=0, observation_scope="world",
                         observation_position_encoding="simple"),
    "gym_surroundings": dict(kind="single", rules_name="extermination", player_names=[], map_name="bridge",
                             agent_ids=[0], agent_weapons="rifle", initial_zombies=10, minimum_zombies=0,
                             observation_scope="surroundings:21", observation_position_encoding="simple"),
    "surroundings_channels": dict(kind="single", rules_name="extermination", player_names=["terminator"],
                                  map_name="boxed", agent_ids=["3"], agent_weapons="gun", initial_zombies=6,
                                  minimum_zombies=0, observation_scope="surroundings:11",
                                  observation_position_encoding="channels"),
    # config 3: multi-agent evacuation, 4 agents
    "c3_city_evac": dict(kind="multi", rules_name="evacuation", player_names=[], map_name="city_for_evacuation",
                         agent_ids=["0", "1", "2", "3"], agent_weapons="rifle", initial_zombies=20, minimum_zombies=0,
                         surroundings_width=21),
    "village_evac_mixed": dict(kind="multi", rules_name="evacuation", player_names=["terminator"],
                               map_name="village_for_evacuation", agent_ids=["0", "1", "2"],
                               agent_weapons=["axe", "shotgun", "knife"], initial_zombies=15, minimum_zombies=0,
                               surroundings_width=9),
    # config 4: safehouse, 100 zombies on the obstacle-dense maze
    "c4_maze_safehouse": dict(kind="single", rules_name="safehouse", player_names=[], map_name="maze_for_safehouse",
                              agent_ids=[0], agent_weapons="rifle", initial_zombies=100, minimum_zombies=0,
                              observation_scope="world", observation_position_encoding="simple"),
    "safehouse_small": dict(kind="single", rules_name="safehouse", player_names=["terminator"], map_name="easy_exit",
                            agent_ids=[0], agent_weapons="shotgun", initial_zombies=8, minimum_zombies=0,
                            observation_scope="world", observation_position_encoding="simple"),
    # reference test fixtures (tests/test_multiagent_env.py): boxed / fort
    "multi_boxed_2p": dict(kind="multi", rules_name="extermination", player_names=[], map_name="boxed",
                           agent_ids=["0", "1"], agent_weapons="rifle", initial_zombies=1, minimum_zombies=0,
                           surroundings_width=21),
    "multi_fort_32p": dict(kind="multi", rules_name="extermination", player_names=[], map_name="fort",
                           agent_ids=[str(i) for i in range(32)], agent_weapons="rifle", initial_zombies=100,
                           minimum_zombies=0, surroundings_width=21),
    # minimum-zombie flow + survival rules + random weapons (SURVEY 8f rank 1)
    "survival_minz": dict(kind="single", rules_name="survival", player_names=["terminator"], map_name="arduino",
                          agent_ids=[0], agent_weapons="random", initial_zombies=5, minimum_zombies=8,
                          observation_scope="world", observation_position_encoding="simple"),
    # the other scripted players (SURVEY 8f rank 2): sniper, troll, hamster (random default weapons, decide-phase draws)
    "bots_mixed": dict(kind="single", rules_name="extermination", player_names=["sniper", "troll", "hamster", "terminator"],
                       map_name="fort", agent_ids=[0], agent_weapons="gun", initial_zombies=25, minimum_zombies=0,
                       observation_scope="surroundings:15", observation_position_encoding="channels"),
    "bots_hamsters": dict(kind="multi", rules_name="survival", player_names=["hamster", "hamster", "sniper"],
                          map_name="hallway", agent_ids=["0", "1"], agent_weapons="knife", initial_zombies=6,
                          minimum_zombies=4, surroundings_width=11),
    # randoman (players/randoman.py): attack / heal ANY thing of World.things by dict index (boxes and walls included),
    # 2 or 3 decide-phase draws per bot
    "bots_randoman": dict(kind="single", rules_name="extermination", player_names=["randoman", "randoman", "hamster"],
                          map_name="boxed", agent_ids=[0], agent_weapons="gun", initial_zombies=6, minimum_zombies=0,
                          observation_scope="world", observation_position_encoding="simple"),
    "randoman_crowd": dict(kind="multi", rules_name="survival", player_names=["randoman", "terminator", "randoman"],
                           map_name="fort", agent_ids=["0", "1"], agent_weapons="shotgun", initial_zombies=40,
                           minimum_zombies=30, surroundings_width=9),
    # slot capacity 256: 8 agents + 2 bots + 236 zombies on the biggest stock map with zombie spawns
    "fort_max_slots": dict(kind="multi", rules_name="extermination", player_names=["terminator", "sniper"], map_name="fort",
                           agent_ids=[str(i) for i in range(8)], agent_weapons=["shotgun", "axe"], initial_zombies=236,
                           minimum_zombies=0, surroundings_width=7),
    # edge: no zombies at all (extermination ends on the first step; every episode is one step long)
    "no_zombies": dict(kind="single", rules_name="extermination", player_names=["terminator"], map_name="hallway",
                       agent_ids=[0], agent_weapons="axe", initial_zombies=0, minimum_zombies=0,
                       observation_scope="world", observation_position_encoding="channels"),
    # boxes destroyed and healed back in the middle of execute_actions with more than 32 actions per step (two chunks of
    # the general kernel): 24 agents with knives (a box survives a hit or two), axes and shotguns on a checkerboard of boxes
    # and spawn cells, 30 zombies; the tape is attacks / moves / heals at adjacent offsets (tape="adjacent").  A destroyed
    # box stays in World.things until clean_dead_things (core.py:121-138): later movers bump into it, a heal revives it.
    "box_arena": dict(kind="multi", rules_name="survival", player_names=[], map_name=os.path.join(MAPS_DIR, "box_arena.txt"),
                      agent_ids=[str(i) for i in range(24)], agent_weapons=["knife", "axe", "knife", "shotgun"],
                      initial_zombies=30, minimum_zombies=0, surroundings_width=5, tape="adjacent"),
    "minz_allcells": dict(kind="multi", rules_name="extermination", player_names=[], map_name="village_for_evacuation",
                          agent_ids=["0", "1"], agent_weapons="random", initial_zombies=4, minimum_zombies=6,
                          surroundings_width=21),
}


def _edge_map(name):
    return os.path.join(MAPS_DIR, name + ".txt")


def _single(map_name, scope="world", enc="simple", rules="extermination", players=("terminator", "terminator"), weapon="rifle",
            zombies=10, minimum=0):
    return dict(kind="single", rules_name=rules, player_names=list(players), map_name=map_name, agent_ids=[0],
                agent_weapons=weapon, initial_zombies=zombies, minimum_zombies=minimum, observation_scope=scope,
                observation_position_encoding=enc)


# map geometry at the edges of what zs_create accepts (tests/maps/*.txt; test_map_edges.py asserts the fact each map is for)
CONFIGS.update({
    # the bench game (agent + 2 terminators, extermination, rifle, 10 zombies, world/simple): with few enough spawn cells the
    # standard rollout shape runs the roster kernel.  odd_cells: 13 x 11 = 143 cells (3 mod 4): the world observation's
    # rows are not 16-byte aligned, so the template is copied cell by cell (no TMA template)
    "bench_odd_cells": _single(_edge_map("odd_cells")),
    # strip_row: 81 x 1 (height 1; 81 cells, 1 mod 4): every neighbour above or below is outside the map
    "bench_strip_row": _single(_edge_map("strip_row")),
    # wide_max: 2,047 x 32 = 65,504 cells, everything in rows 17-31 (cells >= 34,799) near both ends: moves, hits and
    # closest-target searches at the largest cell indices and distances; one env needs ~75 KB of shared memory
    "bench_wide_max": _single(_edge_map("wide_max")),
    # world observations on a 1,533-cell stock map (1 mod 4)
    "fort_world": _single("fort", players=["terminator"], weapon="shotgun", zombies=12),
    # world/channels on odd_cells: three planes of 143 cells each
    "odd_cells_channels": _single(_edge_map("odd_cells"), enc="channels", players=["sniper"], weapon="gun", zombies=8),
    # surroundings width 3 (the narrowest window) on a 3-mod-4 map and on a map one cell high
    "surr3_odd_cells": _single(_edge_map("odd_cells"), scope="surroundings:3", players=["terminator"], zombies=8),
    "surr3_channels_strip_row": _single(_edge_map("strip_row"), scope="surroundings:3", enc="channels", zombies=4),
    # surroundings width 255, far wider than the map: 260 KB (simple) / 520 KB (channels) per window.  strip_col (1 x 42)
    # keeps the per-cell window table under its 32 MB limit (10.9 / 21.9 MB); odd_cells (143 cells: 37 / 74 MB) does not,
    # so its windows are cut from the padded template planes
    "surr255_strip_col": _single(_edge_map("strip_col"), scope="surroundings:255", players=["terminator"], zombies=6),
    "surr255_channels_strip_col": _single(_edge_map("strip_col"), scope="surroundings:255", enc="channels", zombies=4),
    "surr255_odd_cells": _single(_edge_map("odd_cells"), scope="surroundings:255", players=["terminator"], zombies=8),
    "surr255_channels_odd_cells": _single(_edge_map("odd_cells"), scope="surroundings:255", enc="channels",
                                          players=["sniper"], weapon="shotgun", zombies=8),
    # multi-agent surroundings on a map one cell wide (strip_col: 1 x 42, 42 cells, 2 mod 4) and on wide_max
    "multi_strip_col": dict(kind="multi", rules_name="extermination", player_names=["terminator"],
                            map_name=_edge_map("strip_col"), agent_ids=["0", "1", "2"], agent_weapons=["rifle", "knife", "gun"],
                            initial_zombies=6, minimum_zombies=0, surroundings_width=5),
    "multi_wide_max": dict(kind="multi", rules_name="extermination", player_names=["terminator"],
                           map_name=_edge_map("wide_max"), agent_ids=["0", "1", "2", "3"], agent_weapons="shotgun",
                           initial_zombies=12, minimum_zombies=0, surroundings_width=9),
    # more than 32 slots (the general kernel) on wide_max and odd_cells
    "general_wide_max": _single(_edge_map("wide_max"), players=["terminator"], zombies=40),
    "general_odd_cells": _single(_edge_map("odd_cells"), enc="channels", zombies=32),
    # survival with a zombie minimum: no_player_spawns (players stand anywhere free), few_spawns (3 player spawn cells for
    # 3 players, 4 zombie spawn cells for up to 8 zombies: the lean init is off, most respawns find no free spawn cell)
    "minz_no_player_spawns": _single(_edge_map("no_player_spawns"), enc="channels", rules="survival", players=["terminator"],
                                     weapon="knife", zombies=4, minimum=6),
    "minz_few_spawns": _single(_edge_map("few_spawns"), rules="survival", players=["terminator", "sniper"], weapon="axe",
                               zombies=6, minimum=8),
    # crowded: no spawn cells at all and 12 things for 10 free cells (the last two zombies find no cell)
    "crowded": _single(_edge_map("crowded"), players=["terminator"], weapon="knife", zombies=10),
    # safehouse with its objectives on the map's last row and last column
    "safehouse_edges": _single(_edge_map("edge_objectives"), rules="safehouse", players=["terminator"], zombies=6),
})

# single-agent world scope with 17-32 things: 32 slots, the world-scope kernels compiled for 32 slots per env
CONFIGS.update({
    # the bench game with 20 zombies: agent + 2 terminators + 20 zombies = 23 things
    "bridge_world_32": _single("bridge", zombies=20),
    # channels on fort (1,533 cells): agent + terminator + sniper + 24 zombies = 27 things
    "fort_world_32": _single("fort", enc="channels", players=["terminator", "sniper"], weapon="shotgun", zombies=24),
    # world scope at 256 slots: agent + 4 bots + 200 zombies, the minimum-zombie respawn
    "fort_world_256": _single("fort", rules="survival", players=["sniper", "troll", "hamster", "terminator"], weapon="gun",
                              zombies=200, minimum=195),
})


DISCRETE = [(abi.ACT_MOVE, 0, 1), (abi.ACT_MOVE, -1, 0), (abi.ACT_MOVE, 0, -1), (abi.ACT_MOVE, 1, 0),
            (abi.ACT_ATTACK_CLOSEST, 0, 0), (abi.ACT_HEAL, 0, 0), (abi.ACT_HEAL_CLOSEST, 0, 0)]


def build(cfgd, num_envs, seed, env_index_base=0, max_episode_steps=0, auto_reset=False):
    """config dict -> (ZsConfig, Map)."""
    multi = cfgd["kind"] == "multi"
    if multi:
        scope, enc, width = abi.OBS_SURROUNDINGS, abi.OBS_CHANNELS, cfgd["surroundings_width"]
    else:
        scope, enc, width = abi.parse_observation_scope(cfgd["observation_scope"], cfgd["observation_position_encoding"])
    cfg = abi.make_config(cfgd["rules_name"], cfgd["player_names"], cfgd["agent_ids"], cfgd["agent_weapons"],
                          cfgd["initial_zombies"], cfgd["minimum_zombies"], scope, enc, width, multi, num_envs,
                          seed=seed, env_index_base=env_index_base, max_episode_steps=max_episode_steps,
                          auto_reset=auto_reset)
    return cfg, abi.resolve_map(cfgd["map_name"])


def action_tape(cfgd, T, seed, wild=0.25):
    """[T, A, 3] actions: mostly the discrete set, plus `wild` fraction of parametrised edge cases
    (targeted attack/heal at offsets, diagonal / two-cell / null moves, idle, absent keys)."""
    rs = np.random.RandomState(seed)
    multi = cfgd["kind"] == "multi"
    A = len(cfgd["agent_ids"])
    acts = np.zeros((T, A, 3), np.int32)
    if cfgd.get("tape") == "adjacent":
        adj = [(0, 1), (0, -1), (1, 0), (-1, 0)]
        for t in range(T):
            for a in range(A):
                u = rs.rand()
                dx, dy = adj[rs.randint(0, 4)]
                if u < 0.35:
                    acts[t, a] = (abi.ACT_ATTACK, dx, dy)
                elif u < 0.70:
                    acts[t, a] = (abi.ACT_MOVE, dx, dy)
                elif u < 0.90:
                    k = rs.randint(1, 3)  # heal reaches three cells (core.py:8): the box next door or the one behind it
                    acts[t, a] = (abi.ACT_HEAL, k * dx, k * dy)
                else:
                    acts[t, a] = (abi.ACT_ATTACK_CLOSEST, 0, 0)
        return acts
    for t in range(T):
        for a in range(A):
            if rs.rand() < wild:
                kind = rs.randint(0, 6)
                dx, dy = rs.randint(-3, 4, size=2)
                if kind == 0:
                    acts[t, a] = (abi.ACT_ATTACK, dx, dy)
                elif kind == 1:
                    acts[t, a] = (abi.ACT_HEAL, dx, dy)
                elif kind == 2:
                    acts[t, a] = (abi.ACT_MOVE, rs.randint(-2, 3), rs.randint(-2, 3))
                elif kind == 3:
                    acts[t, a] = (abi.ACT_NONE, 0, 0)
                elif kind == 4:
                    acts[t, a] = (abi.ACT_HEAL_CLOSEST, 0, 0)
                else:
                    acts[t, a] = (abi.ACT_ABSENT, 0, 0) if multi else (abi.ACT_ATTACK, rs.randint(-1, 2), rs.randint(-1, 2))
            else:
                acts[t, a] = DISCRETE[rs.randint(0, 7 if multi else 6)]
    return acts


def n_fixed_slots(cfgd):
    return len(cfgd["player_names"]) + len(cfgd["agent_ids"])


def compare_record(tag, ref, got, n_fixed, check_obs=True):
    """Bit-exact comparison of one state record (dict of arrays).  Dead zombie slots carry no
    state in the reference (the object is gone), so x/y/life/weapon are compared only where
    in_world is set or the slot belongs to a bot/agent."""
    errs = []

    def chk(name, a, b):
        a, b = np.asarray(a), np.asarray(b)
        if a.shape != b.shape or not np.array_equal(a, b):
            where = np.argwhere(a != b)[:5].tolist() if a.shape == b.shape else "shape %s vs %s" % (a.shape, b.shape)
            errs.append("%s: %s differs at %s\n  ref=%s\n  got=%s" % (tag, name, where, a.ravel()[:40], b.ravel()[:40]))

    chk("in_world", ref["in_world"], got["in_world"])
    M = len(ref["in_world"])
    keep = np.asarray(ref["in_world"]).astype(bool) | (np.arange(M) < n_fixed)
    for k in ("x", "y", "life", "weapon"):
        chk(k, np.where(keep, ref[k], 0), np.where(keep, got[k], 0))
    chk("order", ref["order"], got["order"])
    chk("static_life", ref["static_life"], got["static_life"])
    chk("static_present", ref["static_present"], got["static_present"])
    chk("dead_body", ref["dead_body"], got["dead_body"])
    chk("counters", np.asarray(ref["counters"])[:3], np.asarray(got["counters"])[:3])
    for k in ("draws", "reward_bits", "terminated", "truncated", "alive_before"):
        if k in ref and k in got:
            chk(k, ref[k], got[k])
    if check_obs and "obs" in ref and "obs" in got:
        chk("obs", np.asarray(ref["obs"]).ravel(), np.asarray(got["obs"]).ravel())
    return errs


def trace_record(trace, prefix, t=None):
    out = {}
    for k, v in trace.items():
        if k.startswith(prefix + "_"):
            out[k[len(prefix) + 1:]] = v if t is None else v[t]
    return out


def replay_traces(engine, cfgd, traces, max_errors=3):
    """Replay E reference traces (global env indices engine.base .. base+E-1) on `engine`
    (an OracleEnv or a CUDA engine adapter with the same methods) in lock-step and compare
    everything after the constructor, every step and every reset.  Returns a list of error strings."""
    E = len(traces)
    multi = cfgd["kind"] == "multi"
    nf = n_fixed_slots(cfgd)
    errs = []
    T = traces[0]["actions"].shape[0]
    obs0 = engine.encode_obs()
    for e in range(E):
        got = engine.export(e)
        got["obs"] = obs0[e]
        got["draws"] = got["reset_draws"]
        ref = trace_record(traces[e], "init")
        if multi:
            ref.pop("obs_mask", None)
        errs += compare_record("env%d init" % e, ref, got, nf)
    if errs:
        return errs
    for t in range(T):
        actions = np.stack([tr["actions"][t] for tr in traces])  # [E, A, 3]
        obs, reward, term, trunc, mask, draws = engine.step(actions, abi.ACTIONS_FULL)
        for e in range(E):
            ref = trace_record(traces[e], "step", t)
            got = engine.export(e)
            got.update(draws=draws[e], terminated=term[e], truncated=trunc[e],
                       reward_bits=np.ascontiguousarray(reward[e]).view(np.uint64))
            if multi:
                om = ref.pop("obs_mask").astype(bool)
                got["alive_before"] = mask[e]
                per = obs[e].reshape(len(om), -1)
                ref["obs"] = np.asarray(ref["obs"]).reshape(len(om), -1)[om]
                got["obs"] = per[om]
                got["reward_bits"] = np.where(ref["alive_before"].astype(bool), got["reward_bits"], 0)
            else:
                got["obs"] = obs[e]
            errs += compare_record("env%d step%d" % (e, t), ref, got, nf)
        if len(errs) >= max_errors:
            return errs
        rmask = np.array([tr["did_reset"][t] for tr in traces], np.uint8)
        want = (term | trunc).astype(np.uint8)
        if not np.array_equal(rmask, want):
            errs.append("tick %d: reset mask %s vs reference %s" % (t, want, rmask))
            return errs
        if rmask.any():
            robs = engine.reset(rmask)
            for e in range(E):
                if not rmask[e]:
                    continue
                ref = trace_record(traces[e], "reset", t)
                if multi:
                    ref.pop("obs_mask", None)
                got = engine.export(e)
                got["obs"] = robs[e]
                got["draws"] = got["reset_draws"]
                errs += compare_record("env%d reset@%d" % (e, t), ref, got, nf)
            if len(errs) >= max_errors:
                return errs
    return errs
