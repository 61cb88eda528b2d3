// zs_device.cuh — device-side data model and helpers of the batched zombsole simulator (sm_100a).
//
// Execution model: ONE LANE GROUP PER ENVIRONMENT.  A group is a full warp (G = 32) or, when an
// env has at most 16 mobile slots (bridge: 13), a HALF warp (G = 16, two envs per warp, every sync /
// vote / reduce carries the group's member mask).  The world of an env lives in shared memory while
// its group works on it:
//   * EnvS<MPC>: the mobile things as structure-of-arrays (packed x/y, life, dict-order rank, meta)
//     and the per-step scratch, in a struct templated on the slot capacity MPC so that every field has
//     a COMPILE-TIME offset (LDS [base + imm]);
//   * after it, at run-time offsets: the occupancy grid, one byte per map cell (0 empty, 1..250 mobile
//     slot+1, 255 box or wall, 254 dead-body decoration) — the shared-memory-staged stand-in for
//     the reference's position-keyed dicts World.things / World.decoration (zombsole/core.py:15-16) —
//     the dead-body bitmap, the static lives and the spawn candidate list.
// Phases that are parallel in the reference's semantics (every actor decides against the pre-step
// world; observation cells are independent) are spread over the group's lanes; the phases that the
// reference defines sequentially (execute_actions) are run by the group's lane 0 on shared memory.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/zs_b200.h"

#define ZS_WPC 4              // warps per CTA
#define ZS_MIN_CTAS 7         // 7 CTAs x 4 warps resident per SM: 4,096 full-warp envs fit the 148 SMs in one wave
#define ZS_MIN_CTAS_LOWOCC 4  // small (latency-bound) batches: 4 CTAs x 4 warps per SM, 128 registers
#define ZS_PROD_ENVS 8        // envs of a producer-warp CTA (four two-env game warps + the producer warp)
#ifndef ZS_OCC_GENERAL
#define ZS_OCC_GENERAL 6      // step kernels with more slots than lanes: shared memory allows six CTAs at best (80 registers)
#endif
#ifndef ZS_MIN_CTAS_G16
#define ZS_MIN_CTAS_G16 6     // two envs per warp: 6 CTAs (80 registers) measured slightly ahead of 7 (72) and of 5 (96)
#endif

// occupancy-grid byte codes (a box/wall is on the grid while it is in World.things, whatever its life)
#define G_EMPTY 0
#define G_MAX_SLOT 250        // 1..250: mobile slot + 1
#define G_DEAD 254            // DeadBody decoration and no thing
#define G_STATIC 255          // pristine box/wall present

// decided action types (the 2-tuples things return from next_step, core.py:87-90)
#define D_IDLE 0
#define D_MOVE 1
#define D_ATTACK 2
#define D_HEAL 3
#define D_WANDER 4            // zombie with no humans: destination drawn in dict order (things.py:101-103)
#define D_RANDOM 5            // randoman: action, target / direction drawn in dict order (players/randoman.py:9-21)

#define RK_NONE 255           // rank of a slot that is not in the world
#define ZS_DEAD_CAP 38        // dead-body cells tracked individually (one-lane-per-slot kernels); more -> bitmap scan
#define ZS_NP_MAX (ZS_MAX_BOTS + ZS_MAX_AGENTS)

struct ZsParams {
    // (kernel parameters live in the constant bank: what the step loop reads every step comes first, packed, so that it
    // takes few constant-cache lines; what only world inits, other scopes or other kernels read follows)
    // ---- configuration, hot
    int32_t N;
    uint32_t env_base;        // low 32 bits of the global index of env 0
    int32_t rules, P, A, Z, M, Mp, Ap, S, Sp, W, H, cells, cells_pad, dead_words;
    int32_t initial_zombies, minimum_zombies;
    int32_t obs_scope, obs_enc, sw, obs_count, obs_C;
    int32_t obs_per_agent, max_steps, auto_reset, n_discrete;
    int32_t has_randoman;     // some bot is a randoman: decide-phase draws are resolved sequentially in dict order
    int32_t fast_init;        // world inits take initialize_world_lists (spawn cells for everybody, fixed weapons)
    int64_t obs_elems;
    uint32_t rkey0[10], rkey1[10];  // Philox round keys (key + r * Weyl constants), so the key schedule costs no instructions
    // ---- shared memory: run-time sized tail behind EnvS<MPC> (byte offsets from the end of the struct)
    int32_t off_dead, off_sl, off_cand, off_spl, off_sidx;
    int32_t smem_per_env;          // sizeof(EnvS<MPC>) + tail, multiple of 16
    int32_t tmpl_smem_off;         // CTA-shared copy of the pristine observation planes (TMA source), -1 if unused
    int32_t tmpl_planes;           // planes staged there: 1 (simple) or 3 (channels: label, life, zeros)
    int32_t tmpl_pair;             // the planes are staged twice back to back: one bulk copy serves both envs of a warp
    int32_t tmpl_bytes;            // bytes of one staged copy of the planes (tmpl_planes * cells * 4)
    // ---- map tables (device, read-only), hot
    const int16_t* cell_static;    // [cells] static index or -1
    const uint16_t* static_cell;   // [Sp] cell of static i
    const int16_t* static_max;     // [Sp] MAX_LIFE of static i (0 in the padding)
    const int32_t* tmpl_obs;       // [2][cells] world-scope observation of the pristine static layer
    unsigned long long* stats;     // [4]
    uint8_t bot_kinds[ZS_MAX_BOTS];
    uint8_t agent_weapons[ZS_MAX_AGENTS];
    // ---- the parked images
    unsigned char* img;            // the parked on-chip images [N, img_pitch bytes] (EnvS: "the IMAGE"), NULL = not kept
    int32_t img_pitch, img_bytes;  // bytes between two envs' images / bytes of one (multiples of 16)
    int32_t img_load;              // the images are current: a launch starts from them instead of load_state + build_grid
    int32_t mpc;                   // slot capacity the kernels are instantiated for (16, 32, 128 or 256)
    // ---- state (device, caller-owned buffer; see ZsLayout)
    int16_t* X; int16_t* Y; int16_t* LIFE; int32_t* STAMP; uint8_t* META;
    int16_t* PREV; int16_t* SLIFE; uint32_t* DEAD; int32_t* SCAL;
    // ---- world init, other scopes, other kernels
    uint32_t key0, key1;      // Philox key = seed
    int32_t n_ps, n_zs;
    const uint16_t* ps_cells;      // [n_ps] player spawn cells, file order
    const uint16_t* zs_cells;      // [n_zs]
    const uint8_t* static_label;   // [Sp]
    const uint8_t* tmpl_grid;      // [cells_pad] G_STATIC on box/wall cells, else 0
    const uint16_t* tmpl_pad;      // surroundings scope: the same planes with a border of fresh Walls sw/2 cells wide,
    int32_t pad_w, pad_plane;      // [1 or 2][H + sw - 1][pad_w = W + sw - 1]; pad_plane = elements per plane
    uint32_t sw_magic;             // ceil(2^32 / sw): i / sw == umulhi(i, sw_magic) for i < 65536
    int32_t win_ints, win_pitch;   // agent standing on the cell, laid out like the output; rows start on 128-byte
                                   // boundaries (L2-resident; NULL when it would be too large)
    const int32_t* win_table;      // [cells][win_pitch] pristine window planes (label / label+life; win_ints words) of an
    const uint32_t* objective_bits;// [dead_words]
    const uint16_t* free_xm;       // [n_free0] the cells without a box/wall in x-major order: World.spawn_in_random's candidates
    const uint16_t* free_index;    // [cells] position of a cell in free_xm (maps where some group has no spawn cells; else NULL)
    int32_t n_free0;
    int32_t cand_cap;
    uint32_t* spl_global;          // static patch lists + SIDX bytes in device memory [N, spl_pitch words] for the kernels with
    int32_t spl_pitch;             // more slots than lanes on maps with many boxes/walls (keeps CTAs resident); NULL = shared
    int32_t prefetch_ahead;        // load_state also prefetches the state of env + prefetch_ahead into the L2 (0 = off)
    uint16_t* cand_global;         // spawn candidate lists in device memory [N, cand_cap] when they are too long for shared
                                   // memory (maps without spawn cells: every cell is a candidate); NULL = in shared memory
    int32_t sl_global;             // same kernels, same maps: box/wall lives are used where they are, in the state buffer
    int32_t prod_off;              // producer-warp launches: CTA-shared mailboxes (ObsMail + record) of the CTA's envs, -1 if unused
    int32_t prod_cap;              // entries one record holds
    int32_t agent_obs_ids[ZS_MAX_AGENTS];
};

struct ZsIO {
    const int32_t* actions;   // [n_steps, N, A(,3)] or NULL (synthetic)
    int32_t fmt;
    int32_t* obs;             // [obs_slots, N, obs_elems] or NULL
    int32_t obs_slots;
    double* reward;           // [n_steps, N(,A)] or NULL
    uint8_t* terminated;      // [n_steps, N] or NULL
    uint8_t* truncated;
    uint8_t* agent_mask;      // [n_steps, N, A] or NULL
    int32_t* draws;           // [n_steps, N] or NULL
    uint32_t* compact;        // [N, compact_words] compact observation records (zs_obs.cuh: obs_world_compact) or NULL
    int32_t compact_words;    // words per record: ZS_COMPACT_HEADER + entry words
    // zs_step_host, records streamed to pinned HOST memory in groups of group_envs consecutive envs: the warp that completes a
    // group raises that group's flag (host_flags + 16 * group, one cache line each) to `ticket` behind a system-scope fence
    uint32_t* host_flags;     // or NULL
    int32_t* group_count;     // device counters, zero between steps
    int32_t group_envs;
    uint32_t ticket;
    const uint8_t* env_mask;  // reset only
    int32_t n_steps;
    int64_t first_step;
    int32_t force_auto_reset;
    // [obs_slots, N, obs_elems] or NULL: the observation of the world an episode ended in, for the envs the step re-initialises
    // (zs_step_final, zs_rollout_final; only the kernels with FIN compiled in write it).  Last, so that the fields every
    // other kernel reads keep their parameter offsets.
    int32_t* final_obs;
    // [N] next-step autoreset (ZS_AUTORESET_NEXT_STEP): 1 = the env's episode has ended and its next step re-initialises it.
    // Handle-owned; only the kernels with NXT compiled in read or write it.  After final_obs for the same reason.
    uint8_t* pending;
};

// weapon tables indexed by weapon code (zombsole/weapons.py:18-25); range2 = floor(max_range^2)
__constant__ int16_t c_range2[16] = {0, 2, 0, 0, 0, 0, 0, 0, 0, 0, 2, 2, 36, 100, 9, 0};
__constant__ int16_t c_dmg_lo[16] = {0, 5, 0, 0, 0, 0, 0, 0, 0, 0, 5, 75, 10, 25, 75, 0};
__constant__ int16_t c_dmg_n[16] = {1, 6, 1, 1, 1, 1, 1, 1, 1, 1, 6, 26, 41, 51, 26, 1};  // hi - lo + 1

// ---------------------------------------------------------------- Philox4x32-10
__device__ __noinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1;
        c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// the env draw stream: key = seed, round keys straight from the kernel parameters (constant-bank operands: inline only —
// behind a call the parameter struct is reached through a generic pointer and every key becomes a load)
__device__ __forceinline__ uint4 philox_draws(const ZsParams& p, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ p.rkey0[r]; c1 = lo1;
        c2 = hi0 ^ c3 ^ p.rkey1[r]; c3 = lo0;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ uint32_t word_of(const uint4& o, int w) { return w == 0 ? o.x : w == 1 ? o.y : w == 2 ? o.z : o.w; }

// ---------------------------------------------------------------- shared-memory image of one env
extern __shared__ __align__(16) unsigned char zs_smem[];

template <int MPC>
struct alignas(16) EnvS {
    static constexpr int GEN = MPC > 32 ? MPC : 1;  // arrays only the general (more slots than lanes) kernels use
    // ---- scratch: lives for a step (or a launch)
    unsigned long long act[MPC];            // the step's action list (packed, see pack_action): actor order, then shuffled in place
    uint32_t bk[MPC];                       // per step: closest-player key of a zombie / heal_closest agent
    // per step: the draws, 4 per Philox block (stored as uint4).  One-lane kernels: up to 3 per slot (a randoman's decision)
    // plus shuffle and hit; general kernels: a slot draws for wandering or for a hit, never both, so 2 per slot plus the
    // randomans' (bots only: at most ZS_MAX_BOTS of them)
    static constexpr int NDRAWS = MPC > 32 ? 2 * MPC + 3 * ZS_MAX_BOTS + 4 : 3 * MPC + 4;
    alignas(16) uint32_t draws[NDRAWS];
    uint32_t zb[GEN < ZS_NP_MAX ? GEN : ZS_NP_MAX];  // per step: closest-zombie key of a player slot
    int32_t scal[8];                        // scalar hand-off around out-of-line functions
    int16_t acts[3 * (GEN < ZS_MAX_AGENTS ? GEN : ZS_MAX_AGENTS) + 1];  // agent actions of the step (type, dx, dy), narrowed
    uint32_t masks[2 * ((MPC + 31) / 32) + 2];  // rank bit-masks: stayers, then movers
    alignas(8) unsigned long long mbar;     // mbarrier of the image load (one phase per launch)
    int16_t da[GEN];
    int16_t db[GEN];
    uint16_t list[MPC];
    uint8_t dtype[MPC];
    uint8_t mvp[GEN];                       // general kernels: list position of the slot's successful move, RK_NONE if none
    uint8_t mpos[GEN];                      // general kernels: list position of the slot's (valid) move action, RK_NONE if none
    alignas(16) uint8_t fyj[MPC > 32 ? 16 : MPC];  // per step: Fisher-Yates partner of every list position (one-lane-per-slot kernels)
    // ---- the IMAGE: everything from here to the end of the struct, and the run-time tail behind it up to the spawn
    // candidate list, is what an env needs on chip between two steps.  A launch leaves it in device memory as one
    // contiguous block next to the canonical state (ZsParams::img) and the next launch brings it back with ONE bulk copy
    // (cp.async.bulk global -> shared behind `mbar`) instead of re-deriving ranks, grid and lists from the state.
    alignas(16) uint32_t txy[MPC];          // x | y << 16 (int16 each)
    int32_t pscal[8];                       // the scalars (ZS_S_*; flags with the launch-lifetime bits) while the env is parked
    int16_t tl[MPC];                        // life
    int16_t prev[MPC < ZS_MAX_AGENTS ? MPC : ZS_MAX_AGENTS];  // reward tracker's agents_life
    uint16_t spn[8];                        // spn[0] = entries of the static patch list (SPL, in the run-time tail)
    uint16_t dbl[ZS_DEAD_CAP + 2];          // dbl[0] = count, dbl[1..] = cells that got a dead body in this world (repeats allowed)
    uint8_t tm[MPC];                        // bit7 in world, bits0-3 weapon code
    uint8_t rk[MPC];                        // dict-order rank among the things in the world (RK_NONE if absent)
    uint8_t sor[MPC];                       // slot of a rank
    uint8_t mvq[MPC];                       // order of this step's successful moves, RK_NONE if none
};
template <int MPC> __host__ __device__ constexpr int img_off() { return (int)offsetof(EnvS<MPC>, txy); }

// Producer-warp launches (zs_sim_kernel SHAPE 3): the game warps hand the observation of every step to a third warp of
// the CTA through one mailbox per env — the cells that differ from the pristine planes as (cell, value) entries — and go on
// with the next transition; the producer warp sends the pristine planes (bulk copy), waits for them, stores the entries.
struct alignas(16) ObsMail {
    unsigned long long full;    // mbarrier: the game warp has filled the record of a step
    unsigned long long empty;   // mbarrier: the producer warp is done with it
    int32_t count;              // entries, or -1: the producer encodes from the env's own shared-memory block (the game warp waits)
    int32_t flags;              // Env::flags of the env at that moment (for the -1 case)
    int32_t pad[2];
    // uint32_t rec[2 * prod_cap] follows
};
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}

// The env a lane group is working on (warp-uniform within the group).
struct Env {
    uint32_t b;       // byte offset of this env's EnvS in zs_smem
    int32_t t, episode, deaths, zd, nlive, flags, prev_zd, ep_steps;
    int32_t env; uint32_t env_global;
    int32_t gl;       // lane within the group
    uint32_t gm;      // member mask of the group
    int32_t gshift;   // first lane of the group within the warp
    uint32_t tmpl_saddr;  // shared-space address of the CTA's observation template (TMA source), computed once per launch
#ifdef ZS_PHASE_CLOCKS
    long long ph_last;
#endif
};
// Env::flags: bit0 is state (ZS_S_FLAGS); the others live for one launch only
#define FL_FRESH 1       // first step of a world: boxes/walls with life <= 0 are still present
#define FL_DMG 2         // the static patch list is not empty
#define FL_SL_DIRTY 4    // static lives changed during this launch: write them back
#define FL_DEAD_OVER 16  // the dead-body list is not complete (overflow, or a kernel that does not keep it): scan the bitmap
#define FL_DEAD_LAUNCH 32  // ... for the whole launch (single-step launches do not build the list), also across world inits

// Bind the shared-memory views of `e` in the current scope (S: the struct; GRIDP/DEADP/SLP/CANDP: the tail).
#define ZS_VIEWS                                                                                   \
    EnvS<MPC>& S = *reinterpret_cast<EnvS<MPC>*>(zs_smem + e.b);                                     \
    uint8_t* const GRIDP = zs_smem + e.b + sizeof(EnvS<MPC>);                                        \
    uint32_t* const DEADP = reinterpret_cast<uint32_t*>(GRIDP + p.off_dead);                         \
    int16_t* const SLP = (MPC > 32 && p.sl_global) ? p.SLIFE + (size_t)e.env * p.Sp                    \
                                                   : reinterpret_cast<int16_t*>(GRIDP + p.off_sl);      \
    uint16_t* const CANDP = p.cand_global ? p.cand_global + (size_t)e.env * p.cand_cap                 \
                                          : reinterpret_cast<uint16_t*>(GRIDP + p.off_cand);             \
    uint32_t* const SPLP = (MPC > 32 && p.spl_global) ? p.spl_global + (size_t)e.env * p.spl_pitch       \
                                                      : reinterpret_cast<uint32_t*>(GRIDP + p.off_spl);  \
    uint8_t* const SIDXP = (MPC > 32 && p.spl_global) ? reinterpret_cast<uint8_t*>(SPLP + p.Sp)          \
                                                      : GRIDP + p.off_sidx;                              \
    (void)S; (void)GRIDP; (void)DEADP; (void)SLP; (void)CANDP; (void)SPLP; (void)SIDXP
// -DZS_CHECKS (development builds, tools/checked_build.sh): every access through these views is bounds-checked on the
// device and a violation traps the kernel (the launch then fails with an error instead of corrupting a neighbour env).
// compute-sanitizer is closed on the GPU pool this was developed on; this is the in-house substitute.
#ifdef ZS_CHECKS
template <typename T> __device__ __forceinline__ T& zs_chk(T* base, long long i, long long n, int what) {
    if (i < 0 || i >= n) { printf("ZS_CHECKS: view %d index %lld outside [0, %lld) (block %d thread %d)\n", what, i, n, blockIdx.x, threadIdx.x); __trap(); }
    return base[i];
}
#define ZS_AT(base, i, n, what) zs_chk(base, (long long)(i), (long long)(n), what)
#else
#define ZS_AT(base, i, n, what) (base)[i]
#endif
#define GRID(i) ZS_AT(GRIDP, i, p.cells_pad, 1)
#define DEADW(i) ZS_AT(DEADP, i, p.dead_words, 2)
#define SL(i) ZS_AT(SLP, i, p.Sp, 3)
#define CAND(i) ZS_AT(CANDP, i, p.cand_cap, 4)
#define TXY(i) ZS_AT(S.txy, i, MPC, 5)
#define TL(i) ZS_AT(S.tl, i, MPC, 6)
#define TM(i) ZS_AT(S.tm, i, MPC, 7)
#define RK(i) ZS_AT(S.rk, i, MPC, 8)
#define SOR(i) ZS_AT(S.sor, i, MPC, 9)
#define MVQ(i) ZS_AT(S.mvq, i, MPC, 10)
#define DTYPE(i) ZS_AT(S.dtype, i, MPC, 11)
#define DA(i) S.da[i]
#define DB(i) S.db[i]
#define ACT(i) ZS_AT(S.act, i, MPC, 12)
#define DRAWS(i) ZS_AT(S.draws, i, EnvS<MPC>::NDRAWS, 13)
#define LIST(i) ZS_AT(S.list, i, MPC, 14)
#define PREVL(i) S.prev[i]
#define ACTS(i) S.acts[i]
#define BK(i) ZS_AT(S.bk, i, MPC, 15)
#define ZB(i) S.zb[i]
#define SCALW(i) S.scal[i]
#define MASKW(i) S.masks[i]
#define SPN S.spn[0]
#define SPL(i) ZS_AT(SPLP, i, p.Sp, 16)
#define SIDX(i) ZS_AT(SIDXP, i, p.Sp, 17)
#define DBL(i) ZS_AT(S.dbl, i, ZS_DEAD_CAP + 2, 18)

// ---------------------------------------------------------------- TMA bulk copies (shared -> global)
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes) : "memory");
}
// the same with the shared-space address already at hand (kept opaque so it is not recomputed at every use)
__device__ __forceinline__ void bulk_store_s(void* gdst, uint32_t saddr, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(saddr), "r"(bytes) : "memory");
}
// ---------------------------------------------------------------- TMA bulk copies (global -> shared) behind an mbarrier
__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // (visible to the async proxy before a copy names it)
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, uint32_t bytes, unsigned long long* bar) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(sdst), a = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(d), "l"(gsrc), "r"(bytes), "r"(a) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "ZS_MBAR_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra ZS_MBAR_DONE_%=;\n"
        "bra ZS_MBAR_WAIT_%=;\n"
        "ZS_MBAR_DONE_%=:\n"
        "}\n" ::"r"(a), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* g) { asm volatile("prefetch.global.L2 [%0];" ::"l"(g)); }
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// generic-proxy stores to global memory (observation patches) before later async-proxy stores to the same addresses
// (the next bulk copy of the pristine planes into that row): without it the bulk copy can overtake them
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

// ---------------------------------------------------------------- phase clocks (development builds only)
// -DZS_PHASE_CLOCKS: thread 0 of CTA 0 accumulates the cycles it spends in each phase of the step loop and prints
// them at the end of the launch (tools/phase_clocks.sh) — the latency chain of one warp, which is what bounds
// small batches.
#ifdef ZS_PHASE_CLOCKS
__device__ unsigned long long zs_ph[24];  // 0-19: the step loop; 20-23: staging, load_state, build_grid, store_state
#define PH(i)                                                                         \
    do {                                                                              \
        if (blockIdx.x == 0 && threadIdx.x == 0) {                                    \
            const long long _c = clock64();                                           \
            atomicAdd(&zs_ph[i], (unsigned long long)(_c - e.ph_last));               \
            e.ph_last = clock64();                                                    \
        }                                                                             \
    } while (0)
#else
#define PH(i) do { } while (0)
#endif

// ---------------------------------------------------------------- launch trace (development builds only)
// -DZS_TRACE: lane 0 of every warp of a step launch records the global timer at kernel entry, after each part of the
// prologue, after each of the first 24 steps and at exit (tools/trace_launch.sh): where a launch's fixed cost goes.
#ifdef ZS_TRACE
#define ZS_TRACE_WARPS 8192
#define ZS_TRACE_SLOTS 40
__device__ unsigned long long zs_trace_buf[ZS_TRACE_WARPS * ZS_TRACE_SLOTS];
__device__ __forceinline__ unsigned long long zs_globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned zs_smid() { unsigned r; asm volatile("mov.u32 %0, %%smid;" : "=r"(r)); return r; }
#define TR(i)                                                                                         \
    do {                                                                                              \
        const int _w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);                           \
        if ((threadIdx.x & 31) == 0 && _w < ZS_TRACE_WARPS && (i) < ZS_TRACE_SLOTS)                   \
            zs_trace_buf[_w * ZS_TRACE_SLOTS + (i)] = (i) == 31 ? (unsigned long long)zs_smid() : zs_globaltimer(); \
    } while (0)
// which of the less common paths a warp took during the launch (slot 28, one bit each)
#define TRF(bit)                                                                                      \
    do {                                                                                              \
        const int _w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);                           \
        if ((threadIdx.x & 31) == 0 && _w < ZS_TRACE_WARPS) {                                         \
            zs_trace_buf[_w * ZS_TRACE_SLOTS + 28] |= (1ull << (bit));                                \
            zs_trace_buf[_w * ZS_TRACE_SLOTS + 34] |= (1ull << (bit));                                \
        }                                                                                             \
    } while (0)
// the warp's slowest step of the launch: its duration (slot 32), the paths it took (slot 33) and its index (slot 35); slot 34
// collects the paths of the step in progress.  TR_STEP_BEGIN / TR_STEP_END bracket a step of the step loops.
#define TR_STEP_BEGIN()                                                                               \
    unsigned long long _tr_t0 = 0;                                                                    \
    do {                                                                                              \
        const int _w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);                           \
        if ((threadIdx.x & 31) == 0 && _w < ZS_TRACE_WARPS) { zs_trace_buf[_w * ZS_TRACE_SLOTS + 34] = 0; _tr_t0 = zs_globaltimer(); } \
    } while (0)
#define TR_STEP_END(step)                                                                             \
    do {                                                                                              \
        const int _w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);                           \
        if ((threadIdx.x & 31) == 0 && _w < ZS_TRACE_WARPS) {                                         \
            const unsigned long long _d = zs_globaltimer() - _tr_t0;                                  \
            if (_d > zs_trace_buf[_w * ZS_TRACE_SLOTS + 32]) {                                        \
                zs_trace_buf[_w * ZS_TRACE_SLOTS + 32] = _d;                                          \
                zs_trace_buf[_w * ZS_TRACE_SLOTS + 33] = zs_trace_buf[_w * ZS_TRACE_SLOTS + 34];      \
                zs_trace_buf[_w * ZS_TRACE_SLOTS + 35] = (unsigned long long)(step);                  \
            }                                                                                         \
        }                                                                                             \
    } while (0)
#else
#define TR(i) do { } while (0)
#define TRF(bit) do { } while (0)
#define TR_STEP_BEGIN() do { } while (0)
#define TR_STEP_END(step) do { } while (0)
#endif

// ---------------------------------------------------------------- lane-group primitives
// G = lanes per env.  With G == 16 a *.sync primitive on the half warp's own member mask costs a convergence
// check (MATCH.ANY + REDUX + VOTEU + branch) in front of every use, which made two envs per warp slower than one.
// CV = true ("converged") instead promises that BOTH halves of the warp reach every primitive together: the
// primitives run on the full mask and are segmented by hand (ballot bits shifted to the half, reductions done
// per half or on values shifted into the half's own 16 bits, shuffles with width 16).  Every branch of the hot
// loop that contains a primitive is therefore taken on a WARP-level condition (wany) and predicated per env
// inside.  CV = false is the divergent flavour (member mask e.gm): the rare out-of-line paths (world init, respawn,
// sequential execute) that one env of a warp may take alone, and the reset / encode kernels.
template <int G, bool CV> __device__ __forceinline__ unsigned gmask(const Env& e) { return (G == 32 || CV) ? 0xffffffffu : e.gm; }
template <int G, bool CV> __device__ __forceinline__ void gsync(const Env& e) { __syncwarp(gmask<G, CV>(e)); }
template <int G, bool CV> __device__ __forceinline__ unsigned gballot(const Env& e, bool pred) {
    const unsigned m = __ballot_sync(gmask<G, CV>(e), pred);
    return G == 32 ? m : ((m >> e.gshift) & ((1u << (G & 31)) - 1u));
}
// any over the env's lanes
template <int G, bool CV> __device__ __forceinline__ bool gany(const Env& e, bool pred) {
    if (G == 32 || !CV) return __any_sync(gmask<G, CV>(e), pred);
    return gballot<G, CV>(e, pred) != 0u;
}
// any over everybody who has to take a branch together: the whole warp when converged, else the env's lanes
template <int G, bool CV> __device__ __forceinline__ bool wany(const Env& e, bool pred) { return __any_sync(gmask<G, CV>(e), pred); }
template <int G, bool CV> __device__ __forceinline__ int gbcast(const Env& e, int v, int src) { return __shfl_sync(gmask<G, CV>(e), v, src, G); }
template <int G, bool CV> __device__ __forceinline__ int gadd(const Env& e, int v) {
    if (G == 32 || !CV) return __reduce_add_sync(gmask<G, CV>(e), v);
    const int lo = __reduce_add_sync(0xffffffffu, e.gshift ? 0 : v), hi = __reduce_add_sync(0xffffffffu, e.gshift ? v : 0);
    return e.gshift ? hi : lo;
}
template <int G, bool CV> __device__ __forceinline__ uint32_t gminu(const Env& e, uint32_t v) {
    if (G == 32 || !CV) return __reduce_min_sync(gmask<G, CV>(e), v);
    const uint32_t lo = __reduce_min_sync(0xffffffffu, e.gshift ? 0xffffffffu : v), hi = __reduce_min_sync(0xffffffffu, e.gshift ? v : 0xffffffffu);
    return e.gshift ? hi : lo;
}
// OR of bit-masks whose set bits are all below G (rank / position masks): one reduction serves both halves
template <int G, bool CV> __device__ __forceinline__ unsigned gor_bits(const Env& e, unsigned v) {
    if (G == 32 || !CV) return __reduce_or_sync(gmask<G, CV>(e), v);
    return (__reduce_or_sync(0xffffffffu, v << e.gshift) >> e.gshift) & ((1u << (G & 31)) - 1u);
}
// lanes of the env holding the same value (value < 2^20), as a mask of group lanes
template <int G, bool CV> __device__ __forceinline__ unsigned gmatch(const Env& e, uint32_t v) {
    if (G == 32) return __match_any_sync(0xffffffffu, v);
    if (!CV) return __match_any_sync(e.gm, v) >> e.gshift;
    return (__match_any_sync(0xffffffffu, v | ((uint32_t)e.gshift << 20)) >> e.gshift) & ((1u << (G & 31)) - 1u);
}
// the larger of a value that is uniform within each env, over the envs that share control flow
template <int G, bool CV> __device__ __forceinline__ int wmax(const Env& e, int v) {
    if (G == 32 || !CV) return v;
    const int o = __shfl_xor_sync(0xffffffffu, v, 16);
    return v > o ? v : o;
}

__device__ __forceinline__ int xy_x(uint32_t xy) { return (int)(int16_t)(xy & 0xffffu); }
__device__ __forceinline__ int xy_y(uint32_t xy) { return (int)xy >> 16; }
__device__ __forceinline__ uint32_t xy_pack(int x, int y) { return (uint32_t)(uint16_t)x | ((uint32_t)y << 16); }

__device__ __forceinline__ uint32_t draw_at(const ZsParams& p, const Env& e, uint32_t t_word, int k) {
    return word_of(philox4x32_10(e.env_global, (uint32_t)e.episode, t_word, (uint32_t)(k >> 2), p.key0, p.key1), k & 3);
}
__device__ __forceinline__ int below(uint32_t u, int n) { return (int)__umulhi(u, (uint32_t)n); }

__device__ __forceinline__ bool g_is_thing(int g) { return g != G_EMPTY && g != G_DEAD; }
__device__ __forceinline__ bool g_is_static(int g) { return g == G_STATIC; }

// World.things.get((x, y)) as a grid byte; positions outside the map hold nothing
__device__ __forceinline__ int grid_at(const ZsParams& p, const uint8_t* GRIDP, int x, int y) {
    if ((unsigned)x >= (unsigned)p.W || (unsigned)y >= (unsigned)p.H) return G_EMPTY;
    return GRIDP[y * p.W + x];
}
__device__ __forceinline__ int dist2(int x1, int y1, int x2, int y2) {
    const int dx = x1 - x2, dy = y1 - y2;
    return dx * dx + dy * dy;
}
__device__ __forceinline__ bool objective_bit(const ZsParams& p, int c) {
    return (__ldg(p.objective_bits + (c >> 5)) >> (c & 31)) & 1u;
}
// adjacent_positions order (zombsole/utils.py:34-44): (0,+1), (0,-1), (+1,0), (-1,0)
__device__ __forceinline__ int adj_dx(int a) { return a == 2 ? 1 : a == 3 ? -1 : 0; }
__device__ __forceinline__ int adj_dy(int a) { return a == 0 ? 1 : a == 1 ? -1 : 0; }

__device__ __forceinline__ int floordiv100(int a) { return a >= 0 ? a / 100 : -((-a + 99) / 100); }
__device__ __forceinline__ int max_life_of_label(int label) { return label == ZS_LABEL_BOX ? 10 : 200; }

// ---------------------------------------------------------------- the static patch list (SPL)
// Boxes and walls keep their damage across episodes (game.py:154-155), so over a long run more and more cells
// differ from the pristine observation template.  SPL holds one 32-bit entry per box/wall whose OBSERVATION differs
// (cell | payload << 16): the world-scope observation patches them every step straight from the list, the first
// clean_dead_things of a world and the grid rebuild walk it instead of all the statics, and SIDX (one byte per static:
// 0 not listed, entry + 1, or 255 = listed further back, found by searching for the cell) finds the entry when the
// box/wall is hit again.  Payload (16 bits): 0 — the box/wall is gone from World.things; simple encoding — the cell
// value v << 1 | 1 (box/wall lives are int16 here, so v lies in [-4660, 1039]; an arithmetic shift of the entry by 17
// gives v, and 0 for "gone", which shows an empty cell); channels — the life, a life of 0 stored as SPL_LIFE0 (the label
// is the pristine template's at the cell).  SPL_LIFE0 is -32768: a channels life of exactly -32768 reads back as 0, the
// one int16 life that does not come out as it is (reserved).  Entries are never removed.
#define SPL_GONE 0
#define SPL_LIFE0 (-32768)
__device__ __forceinline__ int static_payload(const ZsParams& p, int max_life, int life, bool present) {
    if (!present) return SPL_GONE;
    if (p.obs_enc != ZS_OBS_SIMPLE) return life != 0 ? life : SPL_LIFE0;
    const int label = max_life == 10 ? ZS_LABEL_BOX : ZS_LABEL_WALL;
    const int adj = life < 100 ? life : 100;
    return (256 * label + floordiv100(15 * adj)) * 2 + 1;
}
__device__ __forceinline__ uint32_t spl_entry(int cell, int pay) { return (uint32_t)cell | ((uint32_t)pay << 16); }
__device__ __forceinline__ bool spl_gone(uint32_t w) { return (w >> 16) == 0u; }
// What the observation shows on an entry's cell (a gone box/wall leaves it empty): simple — v0 = the value; channels —
// v0 = label, v1 = life.
__device__ __forceinline__ void spl_cell_obs(const ZsParams& p, uint32_t w, int& v0, int& v1) {
    if (p.obs_enc == ZS_OBS_SIMPLE) { v0 = (int)w >> 17; v1 = 0; return; }
    const int pay = (int)w >> 16;
    v0 = spl_gone(w) ? 0 : __ldg(p.tmpl_obs + (w & 0xffffu));
    v1 = pay == SPL_LIFE0 ? 0 : pay;
}
#define SIDX_FAR 255
