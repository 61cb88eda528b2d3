"""ctypes mirror of include/zs_b200.h (structs, enums, prototypes) and the env-kwargs -> ZsConfig
translation.  Importing this module loads no shared library."""
import ctypes as C

import numpy as np

from .maps import Map

ZS_ABI_VERSION = 1
ZS_MAX_BOTS = 32
ZS_MAX_AGENTS = 32
ZS_MAX_SLOTS = 250

RULES = {"extermination": 0, "survival": 1, "evacuation": 2, "safehouse": 3}
KIND_ZOMBIE, KIND_TERMINATOR, KIND_AGENT, KIND_SNIPER, KIND_TROLL, KIND_HAMSTER, KIND_RANDOMAN = 0, 1, 2, 3, 4, 5, 6
BOT_KINDS = {"terminator": KIND_TERMINATOR, "sniper": KIND_SNIPER, "troll": KIND_TROLL, "hamster": KIND_HAMSTER,
             "randoman": KIND_RANDOMAN}
WEAPONS = {"knife": 10, "axe": 11, "gun": 12, "rifle": 13, "shotgun": 14, "random": 255}
WEAPON_CLAWS = 1
ACT_NONE, ACT_MOVE, ACT_ATTACK_CLOSEST, ACT_ATTACK, ACT_HEAL, ACT_HEAL_CLOSEST, ACT_ABSENT = range(7)
ACTION_TYPES = {None: ACT_NONE, "": ACT_NONE, "move": ACT_MOVE, "attack_closest": ACT_ATTACK_CLOSEST,
                "attack": ACT_ATTACK, "heal": ACT_HEAL, "heal_closest": ACT_HEAL_CLOSEST}
ACTIONS_FULL, ACTIONS_DISCRETE = 0, 1
OBS_WORLD, OBS_SURROUNDINGS = 0, 1
OBS_SIMPLE, OBS_CHANNELS = 0, 1
#: ZsConfig.auto_reset values: the caller resets, same-step autoreset, next-step autoreset (ZS_AUTORESET_NEXT_STEP)
AUTORESET_OFF, AUTORESET_SAME_STEP, AUTORESET_NEXT_STEP = 0, 1, 2
AUTORESET_MODES = ("same_step", "next_step")

(F_X, F_Y, F_LIFE, F_STAMP, F_META, F_PREV_LIFE, F_STATIC_LIFE, F_DEAD_BODY, F_SCALARS, F_COUNT) = range(10)
(S_T, S_EPISODE, S_DEATHS, S_ZOMBIE_DEATHS, S_STAMP_COUNTER, S_FLAGS, S_PREV_ZOMBIE_DEATHS, S_EPISODE_STEPS) = range(8)
FIELD_DTYPES = {F_X: np.int16, F_Y: np.int16, F_LIFE: np.int16, F_STAMP: np.int32, F_META: np.uint8,
                F_PREV_LIFE: np.int16, F_STATIC_LIFE: np.int16, F_DEAD_BODY: np.uint32, F_SCALARS: np.int32}
FIELD_NAMES = {F_X: "x", F_Y: "y", F_LIFE: "life", F_STAMP: "stamp", F_META: "meta", F_PREV_LIFE: "prev_life",
               F_STATIC_LIFE: "static_life", F_DEAD_BODY: "dead_body", F_SCALARS: "scalars"}


class ZsMap(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("n_statics", C.c_int32), ("static_xy", C.c_void_p), ("static_label", C.c_void_p),
        ("n_player_spawns", C.c_int32), ("player_spawn_xy", C.c_void_p),
        ("n_zombie_spawns", C.c_int32), ("zombie_spawn_xy", C.c_void_p),
        ("n_objectives", C.c_int32), ("objective_xy", C.c_void_p),
    ]


class ZsConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32), ("env_index_base", C.c_int64), ("seed", C.c_uint64),
        ("rules", C.c_int32), ("n_bots", C.c_int32), ("bot_kinds", C.c_uint8 * ZS_MAX_BOTS),
        ("n_agents", C.c_int32), ("agent_weapons", C.c_uint8 * ZS_MAX_AGENTS), ("agent_obs_ids", C.c_int32 * ZS_MAX_AGENTS),
        ("initial_zombies", C.c_int32), ("minimum_zombies", C.c_int32),
        ("obs_scope", C.c_int32), ("obs_encoding", C.c_int32), ("surroundings_width", C.c_int32),
        ("obs_per_agent", C.c_int32), ("max_episode_steps", C.c_int32), ("auto_reset", C.c_int32),
    ]


class ZsLayout(C.Structure):
    _fields_ = [
        ("state_bytes", C.c_int64), ("offset", C.c_int64 * F_COUNT), ("row_bytes", C.c_int32 * F_COUNT),
        ("n_slots", C.c_int32), ("slot_pitch", C.c_int32), ("agent_pitch", C.c_int32), ("static_pitch", C.c_int32),
        ("dead_words", C.c_int32), ("cells", C.c_int32),
        ("obs_channels", C.c_int32), ("obs_height", C.c_int32), ("obs_width", C.c_int32), ("obs_count", C.c_int32),
        ("obs_elems_per_env", C.c_int64), ("n_discrete_actions", C.c_int32),
    ]


#: name -> (restype, argtypes); every symbol include/zs_b200.h declares
PROTOTYPES = {
    "zs_abi_version": (C.c_int, []),
    "zs_last_error": (C.c_char_p, []),
    "zs_set_device": (C.c_int, [C.c_int32]),
    "zs_layout": (C.c_int, [C.POINTER(ZsConfig), C.POINTER(ZsMap), C.POINTER(ZsLayout)]),
    "zs_create": (C.c_int, [C.POINTER(ZsConfig), C.POINTER(ZsMap), C.POINTER(C.c_void_p)]),
    "zs_destroy": (C.c_int, [C.c_void_p]),
    "zs_bind_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "zs_state_written": (C.c_int, [C.c_void_p]),
    "zs_step_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_compact_words": (C.c_int32, [C.c_void_p]),
    "zs_compact_max_words": (C.c_int32, [C.c_void_p]),
    "zs_step_compact": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "zs_expand_compact": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "zs_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "zs_step_host_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zs_agent_compact_words": (C.c_int32, [C.c_void_p]),
    "zs_agent_compact_max_words": (C.c_int32, [C.c_void_p]),
    "zs_step_compact_agents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "zs_expand_compact_agents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "zs_step_host_agents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int32, C.c_void_p]),
    "zs_init_static_life": (C.c_int, [C.c_void_p, C.c_void_p]),
    "zs_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_step_final": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_encode_obs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_rollout": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_rollout_final": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "zs_fill_synthetic_actions": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "zs_fill_synthetic_tape": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "zs_episode_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "zs_launch_count": (C.c_int64, [C.c_void_p]),
    "zs_lanes_per_env": (C.c_int32, [C.c_void_p]),
    "zs_autoreset_pending": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
}


class MapArg(object):
    """Keeps the numpy tables alive next to the ZsMap that points into them."""

    def __init__(self, map_):
        self.map = map_
        self.tables = map_.tables()
        t = self.tables
        self.struct = ZsMap(
            width=map_.size[0], height=map_.size[1],
            n_statics=len(map_.statics), static_xy=t["static_xy"].ctypes.data, static_label=t["static_label"].ctypes.data,
            n_player_spawns=len(map_.player_spawns), player_spawn_xy=t["player_spawn_xy"].ctypes.data,
            n_zombie_spawns=len(map_.zombie_spawns), zombie_spawn_xy=t["zombie_spawn_xy"].ctypes.data,
            n_objectives=len(map_.objectives), objective_xy=t["objective_xy"].ctypes.data)


def parse_observation_scope(scope, position_encoding):
    """zombsole/gym/observation.py:176-203 (same errors)."""
    lscope = scope.lower()
    width = 0
    if lscope in ["world", "map"]:
        obs_scope = OBS_WORLD
    elif lscope.startswith("surroundings"):
        obs_scope = OBS_SURROUNDINGS
        width = int(lscope[len("surroundings:"):])
        if (width % 2 == 0) or (width <= 1):
            raise ValueError("surroundings width must be an odd number greater than 1")
    else:
        raise ValueError(f"{scope} is not a valid observation scope, must be \"world\", \"map\", or of the form "
                         f"\"surroundings:i\" where i is an integer")
    lpes = position_encoding.lower()
    if lpes not in ["simple", "channels"]:
        raise ValueError(f"{lpes} must be \"simple\" or \"channels\"")
    return obs_scope, (OBS_SIMPLE if lpes == "simple" else OBS_CHANNELS), width


def weapon_code(weapon_name):
    """zombsole/weapons.py:28-45 (same error)."""
    code = WEAPONS.get(weapon_name.lower())
    if code is None:
        raise ValueError(f"{weapon_name} is not a valid player weapon name.  Valid options are knife, axe, gun, "
                         f"rifle, shotgun, and random.")
    return code


def agent_weapon_list(agent_weapons, agent_count):
    """zombsole/game.py:142-149 (same error)."""
    if isinstance(agent_weapons, str):
        return [agent_weapons] * agent_count
    if isinstance(agent_weapons, list):
        from itertools import cycle, islice
        return list(islice(cycle(agent_weapons), agent_count))
    raise ValueError(f"{agent_weapons} is not a valid value for argument agent_weapons.  Value must be the weapon "
                     f"name as a string or a list of weapon names.")


def check_autoreset_mode(autoreset_mode, auto_reset=True, final_observation=False):
    """The autoreset_mode values and the argument combinations next-step autoreset cannot serve."""
    if autoreset_mode not in AUTORESET_MODES:
        raise ValueError("autoreset_mode must be 'same_step' or 'next_step', got %r" % (autoreset_mode,))
    if autoreset_mode == "next_step" and not auto_reset:
        raise ValueError("autoreset_mode='next_step' needs auto_reset=True: without auto-reset the caller resets ended envs")
    if autoreset_mode == "next_step" and final_observation:
        raise ValueError("autoreset_mode='next_step' does not take final_observation=True: the observation of the step that "
                         "ends an episode already is its final observation")


def make_config(rules_name, player_names, agent_ids, agent_weapons, initial_zombies, minimum_zombies,
                obs_scope, obs_encoding, surroundings_width, obs_per_agent, num_envs, seed=0, env_index_base=0,
                max_episode_steps=0, auto_reset=False, autoreset_mode="same_step"):
    if rules_name not in RULES:
        # zombsole/rules/factory.py:19
        raise ValueError(f"{rules_name} is not a valid rule name.  Valid options are extermination, survival, "
                         f"evacuation, and safehouse")
    cfg = ZsConfig()
    cfg.abi_version = ZS_ABI_VERSION
    cfg.num_envs = int(num_envs)
    cfg.env_index_base = int(env_index_base)
    cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    cfg.rules = RULES[rules_name]
    if len(player_names) > ZS_MAX_BOTS:
        raise ValueError("at most %d scripted players are supported" % ZS_MAX_BOTS)
    cfg.n_bots = len(player_names)
    for i, name in enumerate(player_names):
        if name not in BOT_KINDS:
            raise NotImplementedError("scripted player %r is not available in the batched simulator "
                                      "(available: %s)" % (name, ", ".join(sorted(BOT_KINDS))))
        cfg.bot_kinds[i] = BOT_KINDS[name]
    if not 1 <= len(agent_ids) <= ZS_MAX_AGENTS:
        raise ValueError("between 1 and %d agents are supported" % ZS_MAX_AGENTS)
    cfg.n_agents = len(agent_ids)
    for i, (aid, w) in enumerate(zip(agent_ids, agent_weapon_list(agent_weapons, len(agent_ids)))):
        cfg.agent_weapons[i] = weapon_code(w)
        try:
            cfg.agent_obs_ids[i] = int(aid)  # observation.py:74: 8 + int(thing.agent_id)
        except (TypeError, ValueError):
            if obs_encoding == OBS_CHANNELS:
                raise
            cfg.agent_obs_ids[i] = i
    cfg.initial_zombies = int(initial_zombies)
    cfg.minimum_zombies = int(minimum_zombies)
    cfg.obs_scope, cfg.obs_encoding, cfg.surroundings_width = obs_scope, obs_encoding, surroundings_width
    cfg.obs_per_agent = 1 if obs_per_agent else 0
    cfg.max_episode_steps = int(max_episode_steps or 0)
    check_autoreset_mode(autoreset_mode, auto_reset)
    cfg.auto_reset = (AUTORESET_NEXT_STEP if autoreset_mode == "next_step" else AUTORESET_SAME_STEP) if auto_reset else AUTORESET_OFF
    return cfg


def resolve_map(map_name):
    return map_name if isinstance(map_name, Map) else Map.from_map_name(map_name)
