/*
 * zs_b200.h — C ABI of the B200-native batched zombsole simulator.
 *
 * The reference (jvstinian/libzombsole, pure Python) has no FFI; the boundary
 * this library sits behind is the reference's Python env API and the object
 * protocol underneath it.  Each entry point below names the reference code it
 * replaces (paths relative to the reference tree):
 *
 *   zs_create        Map.from_file + Game.__init__ (static part)      zombsole/game.py:44-97,115-140
 *   zs_reset         ZombsoleGymEnv.reset / MultiagentZombsoleEnv.reset
 *                      -> Game.__initialize_world__ -> World.spawn_in_random
 *                                                                      zombsole/gym_env.py:148-164,
 *                                                                      zombsole/gym/multiagent_env.py:173-184,
 *                                                                      zombsole/game.py:151-201, zombsole/core.py:40-66
 *   zs_step          ZombsoleGymEnv.step / MultiagentZombsoleEnv.step  zombsole/gym_env.py:99-145,
 *                      -> Agent.set_action/next_step, World.step,      zombsole/gym/multiagent_env.py:111-171,
 *                         reward tracker, rules, observation           zombsole/core.py:72-208, zombsole/things.py:70-105,
 *                                                                      zombsole/players/agent.py:22-96,
 *                                                                      zombsole/players/terminator.py:9-37,
 *                                                                      zombsole/gym/reward.py:19-98, zombsole/rules/ (all files)
 *   zs_encode_obs    observation_handler.get_observation(game)         zombsole/gym/observation.py:36-173
 *   zs_rollout       a K-step loop of the above with same-step auto-reset (what an RL rollout does
 *                    around gym_env.py:99-164); one launch, state stays on chip between steps
 *   zs_step_final / zs_rollout_final   zs_step / zs_rollout that also return the observation an auto-reset episode
 *                    ended with (gym_env.py:99-164)
 *   ZS_AUTORESET_NEXT_STEP   gymnasium's NEXT_STEP autoreset around the reference's step and reset
 *                    (gym_env.py:99-164, zombsole/gym/multiagent_env.py:111-184)
 *   zs_fill_synthetic_actions   Discrete(6|7).sample() for synthetic rollouts (gym_env.py:367)
 *   zs_step_compact_agents / zs_expand_compact_agents / zs_step_host_agents
 *                    MultiagentZombsoleEnv.step with its per-agent windows  zombsole/gym/multiagent_env.py:111-171,
 *                    returned to a caller on the host                         zombsole/gym/observation.py:99-119
 *
 * Conventions: every `*_dev` / output pointer is a DEVICE pointer owned by the
 * caller (torch allocates); ZsConfig/ZsMap and the pointers inside them are HOST
 * memory read only during the call; `stream` is a cudaStream_t passed as void*;
 * no call synchronises the host except zs_create/zs_destroy; return value 0 = OK,
 * non-zero = error (text from zs_last_error(), thread-local).  One handle per
 * GPU; the caller serialises calls on a handle.  There is no CPU fallback: with
 * no usable CUDA device zs_create fails.
 */
#ifndef ZS_B200_H
#define ZS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZS_ABI_VERSION 1
#define ZS_MAX_BOTS 32
#define ZS_MAX_AGENTS 32
#define ZS_MAX_SLOTS 250 /* bots + agents + zombie slots per env */

/* rules (zombsole/rules/factory.py:7-19) */
enum { ZS_RULES_EXTERMINATION = 0, ZS_RULES_SURVIVAL = 1, ZS_RULES_EVACUATION = 2, ZS_RULES_SAFEHOUSE = 3 };
/* mobile thing kinds; the bots mirror zombsole/players/{terminator,sniper,troll,hamster,randoman}.py */
enum { ZS_KIND_ZOMBIE = 0, ZS_KIND_TERMINATOR = 1, ZS_KIND_AGENT = 2, ZS_KIND_SNIPER = 3, ZS_KIND_TROLL = 4,
       ZS_KIND_HAMSTER = 5, ZS_KIND_RANDOMAN = 6 };
/* observation thing labels (zombsole/gym/observation.py:18-26) */
enum { ZS_LABEL_BOX = 1, ZS_LABEL_DEAD_BODY = 2, ZS_LABEL_OBJECTIVE = 3, ZS_LABEL_WALL = 4,
       ZS_LABEL_ZOMBIE = 5, ZS_LABEL_PLAYER = 6, ZS_LABEL_AGENT = 7 };
/* weapon codes = observation weapon labels (zombsole/gym/observation.py:27-34, zombsole/weapons.py:18-25) */
enum { ZS_WEAPON_NONE = 0, ZS_WEAPON_CLAWS = 1, ZS_WEAPON_KNIFE = 10, ZS_WEAPON_AXE = 11, ZS_WEAPON_GUN = 12,
       ZS_WEAPON_RIFLE = 13, ZS_WEAPON_SHOTGUN = 14, ZS_WEAPON_RANDOM = 255 };
/* agent action types (zombsole/players/agent.py:28-96); ABSENT = key missing from a multi-agent
 * action dict, which the reference turns into "heal self" (zombsole/gym/multiagent_env.py:129-131) */
enum { ZS_ACT_NONE = 0, ZS_ACT_MOVE = 1, ZS_ACT_ATTACK_CLOSEST = 2, ZS_ACT_ATTACK = 3, ZS_ACT_HEAL = 4,
       ZS_ACT_HEAL_CLOSEST = 5, ZS_ACT_ABSENT = 6 };
/* action tensor formats */
enum {
    ZS_ACTIONS_FULL = 0,     /* int32 [N, A, 3] = (type, dx, dy) */
    ZS_ACTIONS_DISCRETE = 1  /* int32 [N, A] ids of ZombsoleGymEnvDiscreteAction.game_actions (gym_env.py:328-351)
                                / MultiagentZombsoleEnvDiscreteAction.game_actions (multiagent_env.py:259-285) */
};
/* observation scope / encoding (zombsole/gym/observation.py:176-203) */
enum { ZS_OBS_WORLD = 0, ZS_OBS_SURROUNDINGS = 1 };
enum { ZS_OBS_SIMPLE = 0, ZS_OBS_CHANNELS = 1 };

typedef struct ZsMap {
    int32_t width, height;          /* Map.size (game.py:88-93) */
    int32_t n_statics;              /* boxes + walls, in file (row-major) order (game.py:76-79) */
    const int16_t* static_xy;       /* [n_statics, 2] */
    const uint8_t* static_label;    /* [n_statics] ZS_LABEL_BOX | ZS_LABEL_WALL */
    int32_t n_player_spawns;        /* 'p' cells in file order (game.py:80-81) */
    const int16_t* player_spawn_xy; /* [n, 2] */
    int32_t n_zombie_spawns;        /* 'z' cells (game.py:82-83) */
    const int16_t* zombie_spawn_xy;
    int32_t n_objectives;           /* 'o' cells (game.py:84-86) */
    const int16_t* objective_xy;
} ZsMap;

typedef struct ZsConfig {
    int32_t abi_version;       /* ZS_ABI_VERSION */
    int32_t num_envs;          /* N environments on this handle */
    int64_t env_index_base;    /* global index of local env 0 (draw counters use the global index) */
    uint64_t seed;
    int32_t rules;             /* ZS_RULES_* */
    int32_t n_bots;            /* len(player_names) */
    uint8_t bot_kinds[ZS_MAX_BOTS];
    int32_t n_agents;          /* 1 for ZombsoleGymEnv, len(agent_ids) for the multi-agent env */
    uint8_t agent_weapons[ZS_MAX_AGENTS]; /* ZS_WEAPON_* (RANDOM draws at every world init, weapons.py:43) */
    int32_t agent_obs_ids[ZS_MAX_AGENTS]; /* int(agent_id): channels thing code is 8 + this (observation.py:73-74) */
    int32_t initial_zombies;
    int32_t minimum_zombies;
    int32_t obs_scope;         /* ZS_OBS_WORLD | ZS_OBS_SURROUNDINGS */
    int32_t obs_encoding;      /* ZS_OBS_SIMPLE | ZS_OBS_CHANNELS */
    int32_t surroundings_width;/* odd, > 1 (observation.py:185) */
    int32_t obs_per_agent;     /* 0: one observation per env (agent 0); 1: one per agent [N, A, ...] */
    int32_t max_episode_steps; /* 0 = none; gymnasium TimeLimit of the registered ids (gym_env.py:385) */
    int32_t auto_reset;        /* 0: the caller resets ended envs (zs_reset); 1: same-step autoreset, zs_step re-initialises
                                  an env in the same call when it ends; ZS_AUTORESET_NEXT_STEP: next-step autoreset (below) */
} ZsConfig;

/* ---- next-step autoreset (ZsConfig.auto_reset = ZS_AUTORESET_NEXT_STEP; gymnasium 1.x's AutoresetMode.NEXT_STEP, the
 * default of its vector envs)
 * The step that ends an episode (rules, all agents dead, or the TimeLimit) is a step of an auto_reset = 0 handle: its
 * observation, reward (with the +-10 end reward), flags, agent mask and draws, the world left as it ended, the episode
 * counted in zs_episode_stats.  The env is then marked pending.  Its next step runs no transition and ignores its action:
 * it performs the world init zs_reset would perform (the same draws; episode + 1; box/wall damage kept; gym_env.py:148-164,
 * zombsole/gym/multiagent_env.py:173-184) and returns the new world's observation with reward +0.0 in every reward slot,
 * terminated = truncated = 0, every agent in the agent mask and, as draws, the init's draw count.  That step clears the
 * mark and does not count toward the TimeLimit.  Other envs of the launch step normally.
 * zs_step, zs_step_masked (unselected envs stay pending), zs_rollout, zs_step_compact, zs_step_host, zs_step_compact_agents
 * and zs_step_host_agents follow it on such a handle; zs_step_final / zs_rollout_final refuse it (the observation of the
 * ending step already is the final observation).  zs_reset clears the marks of the envs it re-initialises, zs_bind_state
 * and zs_init_static_life clear all of them; zs_encode_obs of a pending env shows the world it ended in.
 * Such a handle runs one env per warp in every launch (zs_lanes_per_env = 32, whatever ZS_LANES_PER_ENV says). */
#define ZS_AUTORESET_NEXT_STEP 2

/* Layout of the caller-owned state buffer: structure-of-arrays, one row per env per field.
 * Field f of env e starts at byte  offset[f] + e * row_bytes[f]. */
enum {
    ZS_F_X = 0,          /* int16 [N, slot_pitch]   */
    ZS_F_Y,              /* int16 [N, slot_pitch]   */
    ZS_F_LIFE,           /* int16 [N, slot_pitch]   */
    ZS_F_STAMP,          /* int32 [N, slot_pitch]   dict-order stamp: any values whose ORDER among the slots in the world is
                            the World.things iteration order (smaller = earlier); the library writes ranks 0..n-1 */
    ZS_F_META,           /* uint8 [N, slot_pitch]   bit7 = in World.things, bits0-3 = weapon code */
    ZS_F_PREV_LIFE,      /* int16 [N, agent_pitch]  reward tracker's agents_life (reward.py:21,27,33) */
    ZS_F_STATIC_LIFE,    /* int16 [N, static_pitch] persists across resets (game.py:154-155) */
    ZS_F_DEAD_BODY,      /* uint32 [N, dead_words]  bit c = DeadBody decoration on cell c */
    ZS_F_SCALARS,        /* int32 [N, 8]  see ZS_S_* */
    ZS_F_COUNT
};
enum {
    ZS_S_T = 0,          /* World.t (core.py:17,74) */
    ZS_S_EPISODE,        /* world initialisations so far (0 = constructor) */
    ZS_S_DEATHS,         /* World.deaths */
    ZS_S_ZOMBIE_DEATHS,  /* World.zombie_deaths */
    ZS_S_STAMP_COUNTER,  /* number of mobile things in World.things (= the next dict-order rank) */
    ZS_S_FLAGS,          /* bit0: fresh world (statics with life<=0 still present until the first clean) */
    ZS_S_PREV_ZOMBIE_DEATHS, /* reward tracker's zombie_deaths (reward.py:22,28,34) */
    ZS_S_EPISODE_STEPS,  /* steps since the last world init (TimeLimit) */
    ZS_S_COUNT           /* = 8 */
};

typedef struct ZsLayout {
    int64_t state_bytes;
    int64_t offset[ZS_F_COUNT];
    int32_t row_bytes[ZS_F_COUNT];
    int32_t n_slots;       /* bots + agents + zombie slots */
    int32_t slot_pitch;
    int32_t agent_pitch;
    int32_t static_pitch;
    int32_t dead_words;
    int32_t cells;
    int32_t obs_channels;  /* C */
    int32_t obs_height;    /* H (map height or surroundings width) */
    int32_t obs_width;     /* W */
    int32_t obs_count;     /* observations per env: 1 or n_agents */
    int64_t obs_elems_per_env; /* obs_count * C * H * W (int32 elements) */
    int32_t n_discrete_actions; /* 6 single-agent, 7 multi-agent */
} ZsLayout;

typedef struct ZsHandle ZsHandle;

int zs_abi_version(void);
const char* zs_last_error(void);

/* Pure host arithmetic: validates cfg/map and fills the layout.  Needs no GPU. */
int zs_layout(const ZsConfig* cfg, const ZsMap* map, ZsLayout* out);

/* Select the CUDA device for the calling thread inside this library's own CUDA runtime instance
 * (the library links cudart statically; call it with the ordinal of the device the caller's
 * tensors live on before zs_create). */
int zs_set_device(int32_t device);

/* Uploads the map tables (handle-owned device memory) on the current device. */
int zs_create(const ZsConfig* cfg, const ZsMap* map, ZsHandle** out);
int zs_destroy(ZsHandle* h);

/* Bind the caller-allocated state buffer (>= layout.state_bytes, 16-byte aligned, device). */
int zs_bind_state(ZsHandle* h, void* state_dev, int64_t bytes);

/* The caller has written into the state buffer (imported a state, edited a life, ...): the handle's parked on-chip
 * images of the envs (a launch leaves them in device memory and the next one starts from them) are stale, the next
 * launch re-derives everything from the state buffer.  Not needed after zs_bind_state / zs_init_static_life.
 * (The reference's counterpart is mutating World.things / thing.life between steps, as its tests do:
 * tests/test_game.py:41-66.) */
int zs_state_written(ZsHandle* h);

/* zs_init_static_life: what constructing a new env does before its first world init — every
 * box/wall gets its MAX_LIFE (Map.from_file builds the objects once, game.py:76-79) and the
 * episode counter is set so that the next zs_reset is world initialisation #0 (game.py:138).
 * The state buffer must have been zero-filled by the caller.
 *
 * zs_reset: (re)initialise the worlds selected by env_mask_dev (uint8 [N], NULL = all) and, if
 * obs_dev is not NULL, write their observation; draws_dev (int32 [N], may be NULL) receives the
 * number of draws each init consumed.  Static lives are NOT restored: wall/box damage persists
 * across resets exactly as in the reference (game.py:154-155). */
int zs_init_static_life(ZsHandle* h, void* stream);
int zs_reset(ZsHandle* h, const uint8_t* env_mask_dev, int32_t* obs_dev, int32_t* draws_dev, void* stream);

/* One env transition for all N envs.
 *   actions_dev     per action_format
 *   obs_dev         int32 [N, obs_elems_per_env]
 *   reward_dev      float64 [N] (obs_per_agent=0) or [N, n_agents]
 *   terminated_dev, truncated_dev   uint8 [N]
 *   agent_mask_dev  uint8 [N, n_agents] agents alive before the step (keys of the reference's
 *                   per-agent dicts, multiagent_env.py:88-97,156-166); may be NULL
 *   draws_dev       int32 [N] number of draws the step consumed (parity diagnostics); may be NULL */
int zs_step(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev,
            double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
            uint8_t* agent_mask_dev, int32_t* draws_dev, void* stream);

/* zs_step for the worlds selected by env_mask_dev (uint8 [N], NULL = all) only: the others are not touched — no
 * transition, no outputs written.  This is what serving N independent clients from one batch needs (one client's
 * GameAction advances that client's world, zombsole/interactive_json.py:317-325).  Needs a handle with one warp per
 * env (zs_lanes_per_env == 32). */
int zs_step_masked(ZsHandle* h, const uint8_t* env_mask_dev, const int32_t* actions_dev, int32_t action_format,
                   int32_t* obs_dev, double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                   uint8_t* agent_mask_dev, void* stream);

/* Encode the observation of the current state only. */
int zs_encode_obs(ZsHandle* h, int32_t* obs_dev, void* stream);

/* n_steps transitions in ONE launch with same-step auto-reset (regardless of cfg.auto_reset), or with next-step autoreset on
 * a handle created with auto_reset = ZS_AUTORESET_NEXT_STEP.
 *   actions_dev  int32 [n_steps, N, A(,3)] or NULL: discrete ids drawn in-kernel from the
 *                synthetic action stream (same values as zs_fill_synthetic_actions with
 *                step_index = first_step_index + i)
 *   obs_dev      int32 [obs_slots, N, obs_elems_per_env]; step i writes slot i % obs_slots
 *   reward_dev   float64 [n_steps, N(, A)];  terminated_dev/truncated_dev uint8 [n_steps, N]
 *   any of reward/terminated/truncated may be NULL */
int zs_rollout(ZsHandle* h, int32_t n_steps, int64_t first_step_index, const int32_t* actions_dev,
               int32_t action_format, int32_t* obs_dev, int32_t obs_slots, double* reward_dev,
               uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream);

/* ---- final observations of auto-reset episodes (gymnasium's SAME_STEP autoreset: info["final_obs"], info["_final_obs"])
 * An env whose step ends its episode (terminated or truncated, TimeLimit included) is re-initialised in the same step, and
 * obs_dev receives the first observation of the new episode.  These two calls also write, for each such env, the
 * observation of the world the episode ended in to its row of final_obs_dev: exactly what zs_step writes for that step on a
 * handle with auto_reset = 0 — taken after the transition, the reward and the minimum-zombie respawn, before the world init
 * (zombsole/gym_env.py:99-164, zombsole/gym/multiagent_env.py:111-184).  final_obs_dev has the layout of obs_dev.  The rows
 * of envs whose step did not end an episode are unspecified: terminated | truncated says which rows hold a final
 * observation.  Everything else (outputs, state, episode statistics) is what zs_step / zs_rollout compute.  Both calls need
 * non-NULL obs_dev and final_obs_dev.
 * zs_step_final: zs_step on a handle with auto_reset = 1 (it fails on another: nothing would be re-initialised).
 * zs_rollout_final: zs_rollout; final_obs_dev int32 [obs_slots, N, obs_elems_per_env], step i writes slot i % obs_slots. */
int zs_step_final(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev,
                  int32_t* final_obs_dev, double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                  uint8_t* agent_mask_dev, int32_t* draws_dev, void* stream);
int zs_rollout_final(ZsHandle* h, int32_t n_steps, int64_t first_step_index, const int32_t* actions_dev,
                     int32_t action_format, int32_t* obs_dev, int32_t* final_obs_dev, int32_t obs_slots,
                     double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream);

/* ---- compact host outputs (world-scope observation, one agent's reward per env)
 * The world observation of an env is the map's pristine layer (the same for every env and step) plus a few dozen cells
 * that differ: the mobile things, damaged or destroyed boxes/walls, dead bodies.  zs_step_compact runs one transition
 * like zs_step but emits, instead of the int32 [N, C, H, W] observation, one fixed-size RECORD per env:
 *   word 0      bits 0-15 number of entries, bit 16 terminated, bit 17 truncated, bit 18 overflow
 *   word 1      reserved
 *   words 2-3   the reward (float64 bits, little endian)
 *   words 4..   the entries: simple encoding — cell | value << 16; channels — two words: cell | thing << 16, then
 *               (life & 0xffff) | weapon << 16 (value and life are signed 16-bit: a box/wall's may be negative)
 * so that a step costs about 0.5 KB per env over PCIe instead of 5-16 KB.  An env with more differing cells than a
 * record holds (or a value that does not fit) sets the overflow bit and gets its full row written to obs_dev, which the
 * caller fetches for that env alone.  zs_expand_compact (HOST code, threaded) turns the records the caller copied to
 * host memory into the reference's observation tensor, byte-identical to what zs_step writes: it keeps the previous
 * records in `prev_host` and only rewrites the cells that changed.  (Reference: observation.py:83-89, 122-142 builds
 * the same tensor cell by cell; gym_env.py:99-145 returns it with reward and flags.) */
#define ZS_COMPACT_HEADER 4
/* zs_compact_words: a good record size for this handle in words (0 if the configuration has no compact form:
 * surroundings scope, per-agent observations); zs_compact_max_words: the size no env overflows by count.  Games of at
 * most 32 slots default to 96 words (simple) / 192 (channels); games of more slots to room for every slot plus as many
 * entries again as a small game gets (224 / 416 words for 101 slots).  The caller picks compact_words (the same value for
 * zs_step_compact and zs_expand_compact of a step) and may grow it when overflows become frequent: box/wall damage
 * persists across episodes (game.py:154-155), so the number of differing cells of a long-running env creeps up. */
int32_t zs_compact_words(const ZsHandle* h);
int32_t zs_compact_max_words(const ZsHandle* h);
int zs_step_compact(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, uint32_t* compact_dev,
                    int32_t compact_words, int32_t* obs_dev, void* stream);
/* compact_host, prev_host: uint32 [N, compact_words]; obs_host int32 [N, obs_elems_per_env]; reward_host float64 [N];
 * terminated_host / truncated_host uint8 [N]; overflow_envs_host int32 [N] receives the indices of the envs whose rows
 * the caller must copy from obs_dev, *n_overflow their number.  first_call != 0: prev_host / obs_host hold nothing yet.
 * n_threads <= 0: all the host threads of the process. */
int zs_expand_compact(const ZsHandle* h, const uint32_t* compact_host, uint32_t* prev_host, int32_t* obs_host,
                      double* reward_host, uint8_t* terminated_host, uint8_t* truncated_host,
                      int32_t* overflow_envs_host, int32_t* n_overflow, int32_t compact_words, int32_t first_call,
                      int32_t n_threads);

/* zs_step_host: zs_step_compact + zs_expand_compact in one call for a caller whose buffers live in HOST memory.
 * `actions_host` (int32 [N, A(,3)], any host memory; pinned avoids a staging copy) goes to the device with the copy engine
 * ahead of the launch.  The kernel writes `compact_pinned` (uint32 [N, compact_words]) in place — it must be page-locked
 * host memory the device can address (cudaHostAlloc / cudaHostRegister / torch pin_memory) — as coalesced rows, and the
 * warp that completes the batch raises a flag in pinned memory behind one system-scope fence; n_threads host threads,
 * which have meanwhile put the cells of the previous records back to the pristine layer and are spinning on that flag
 * inside their parallel region, expand the records into obs_host / reward_host / terminated_host / truncated_host (ordinary
 * host memory, as for zs_expand_compact) the moment it shows.  No device-to-host copy, no stream synchronisation and no
 * thread wake-up are on the way of a step; when the call returns every env has been expanded, the action buffer is the
 * caller's again, and obs_dev holds the rows of the envs listed in overflow_envs_host (as for zs_expand_compact; the
 * call synchronises the stream when there are any).  prev_host / first_call as for zs_expand_compact (one prev_host per
 * record buffer).  How the threads expand — previous cells restored ahead of the flag and the new ones written after it, or
 * every env as the difference of its two records, which suits a host bound by memory traffic — is timed and chosen by
 * the handle (ZS_HOST_DIFF=0/1 forces one); the results are the same.  Fails after ten seconds if the flag does not show.  (Reference: the same transition as gym_env.py:99-145 returns to a caller
 * on the host.) */
int zs_step_host(ZsHandle* h, const int32_t* actions_host, int32_t action_format, uint32_t* compact_pinned,
                 uint32_t* prev_host, int32_t compact_words, int32_t* obs_dev, int32_t* obs_host, double* reward_host,
                 uint8_t* terminated_host, uint8_t* truncated_host, int32_t* overflow_envs_host, int32_t* n_overflow,
                 int32_t first_call, int32_t n_threads, void* stream);
/* ---- compact host outputs for per-agent surroundings observations (the multi-agent env)
 * Every agent's observation is the (w, w) window of the map around it: MultiagentZombsoleEnv.step builds one per agent
 * (zombsole/gym/multiagent_env.py:111-171) from observation.py:99-119.  Most of a window is the map's pristine layer
 * (out-of-bounds cells are a fresh Wall), so one fixed-size record per env carries the agents' window centres and the
 * cells any window shows that differ from that layer.  With A = n_agents, H = ZS_AGENT_COMPACT_HEADER(A) words:
 *   word 0          bits 0-15 number of entries, bit 16 terminated, bit 17 truncated, bit 18 overflow
 *   word 1          agent mask: bit a = agent a was alive before the step (zs_step's agent_mask_dev)
 *   words 2..2+2A-1 the reward of agent a as float64 bits, two words each, little endian
 *   words 2+2A..H-1 per agent: bits 0-15 the cell (y * width + x) its window is centred on (the agent slot's position,
 *                   where it died if it is dead), bits 16-31 its life after the step (and after the step's auto-reset)
 *                   as int16
 *   words H..       the entries, encoded as in the world record: box/wall patches, dead bodies, mobile things, each one
 *                   only if its cell lies inside at least one agent's window
 * Overflow follows the world record's rules (too many entries, or a value outside its field): the env's full rows
 * [A, C, w, w] are written to obs_dev for the caller to fetch.  Available for obs_scope = ZS_OBS_SURROUNDINGS with
 * obs_per_agent = 1, at most 32 slots and fewer than 65,536 cells; both encodings.
 * zs_agent_compact_words: a good record size for this handle (0 outside that scope); zs_agent_compact_max_words: the
 * size no env overflows by count.  As for the world record, the caller may grow compact_words between steps. */
#define ZS_AGENT_COMPACT_HEADER(A) (2 + 3 * (A))
int32_t zs_agent_compact_words(const ZsHandle* h);
int32_t zs_agent_compact_max_words(const ZsHandle* h);
int zs_step_compact_agents(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, uint32_t* compact_dev,
                           int32_t compact_words, int32_t* obs_dev, void* stream);
/* HOST code, threaded: records -> obs_host int32 [N, A, C, w, w], byte-identical to what zs_step writes, reward_host
 * float64 [N, A], terminated_host / truncated_host uint8 [N], agent_mask_host uint8 [N, A], agent_life_host int16 [N, A].
 * Incremental per env and agent: a window whose centre moved (or on the first call, or after the env's previous record
 * overflowed) is copied from the pristine layer; otherwise only the previous record's cells inside it are restored.  Then
 * the new entries are written into every window that shows them.  prev_host, overflow_envs_host, n_overflow, first_call
 * and n_threads as for zs_expand_compact. */
int zs_expand_compact_agents(const ZsHandle* h, const uint32_t* compact_host, uint32_t* prev_host, int32_t* obs_host,
                             double* reward_host, uint8_t* terminated_host, uint8_t* truncated_host,
                             uint8_t* agent_mask_host, int16_t* agent_life_host, int32_t* overflow_envs_host,
                             int32_t* n_overflow, int32_t compact_words, int32_t first_call, int32_t n_threads);
/* zs_step_compact_agents + zs_expand_compact_agents in one call for a caller whose buffers live in host memory: the same
 * transport as zs_step_host (actions copied ahead of the launch, records written by the kernel into compact_pinned, a flag
 * in pinned memory, host threads waiting for it, ten seconds until it gives up).  The threads expand every env after the
 * flag: whether a window is restored cell by cell or copied whole depends on the new record.  ZS_HOST_DIFF has no effect
 * here. */
int zs_step_host_agents(ZsHandle* h, const int32_t* actions_host, int32_t action_format, uint32_t* compact_pinned,
                        uint32_t* prev_host, int32_t compact_words, int32_t* obs_dev, int32_t* obs_host, double* reward_host,
                        uint8_t* terminated_host, uint8_t* truncated_host, uint8_t* agent_mask_host,
                        int16_t* agent_life_host, int32_t* overflow_envs_host, int32_t* n_overflow, int32_t first_call,
                        int32_t n_threads, void* stream);
/* diagnostics: out[5] = zs_step_host calls since the last read, and the mean microseconds from entry until the launches
 * were issued / thread 0 had restored the cells of its previous records / the flag showed (every record in host memory) /
 * the call returned (every env expanded) */
int zs_step_host_stats(ZsHandle* h, double* out);

/* actions_dev int32 [N, A]: uniform discrete ids for step `step_index` (Philox action stream). */
int zs_fill_synthetic_actions(ZsHandle* h, int64_t step_index, int32_t* actions_dev, void* stream);
/* the same for n_steps consecutive steps in one launch: actions_dev int32 [n_steps, N, A] (an action tape for zs_rollout) */
int zs_fill_synthetic_tape(ZsHandle* h, int64_t first_step_index, int32_t n_steps, int32_t* actions_dev, void* stream);

/* Episode statistics accumulated on the device since the last call with reset=1:
 * out_dev int64 [4] = episodes finished, episodes won, sum of episode lengths, sum of zombie deaths. */
int zs_episode_stats(ZsHandle* h, int64_t* out_dev, int32_t reset, void* stream);

/* Number of kernel launches issued through this handle so far (bench.py's gpu_launches). */
int64_t zs_launch_count(const ZsHandle* h);

/* Lanes of a warp that work on one env on this handle: 32, or 16 (two envs per warp) for worlds of at
 * most 16 things in batches larger than one resident wave (diagnostics / tests). */
int32_t zs_lanes_per_env(const ZsHandle* h);

/* Next-step autoreset handles: *dev = the handle's marks, device uint8 [N], 1 = the env's next step is its reset step
 * (gymnasium's _autoreset_envs).  Owned by the handle; read them on the handle's stream.  Fails on other handles. */
int zs_autoreset_pending(const ZsHandle* h, const uint8_t** dev);

#ifdef __cplusplus
}
#endif
#endif /* ZS_B200_H */
