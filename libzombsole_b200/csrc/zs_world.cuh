// zs_world.cuh — the world transition, rules, rewards and world (re)initialisation, one lane group per env.
// Reference line numbers are relative to the reference tree (jvstinian/libzombsole v0.13.2).
// Everything is templated on the slot capacity MPC (16, 32, 128, 256), the lanes per env G (32, or 16 for
// MPC == 16) and CV (see zs_device.cuh: full-mask warp primitives); ONE = "every slot has its own lane".
#pragma once
#include "zs_device.cuh"

#define ZS_TPL template <int MPC, int G, bool CV>
#define ZS_CONSTS                                   \
    constexpr bool ONE = MPC <= G;                  \
    (void)ONE

// A game roster compiled into the standard rollout kernel: the rules, the player count NP (bots + ONE agent) and every
// bot a terminator.  ROS = 0 reads the game from ZsParams instead.  Under a roster the player loops, the lane tests and
// the bot-kind predicates of the step fold to constants, and the randoman path and the rules dispatch drop out.
// launch_sim picks a roster kernel when the handle's game is one (ZsHandle::roster, set by zs_create).
constexpr int zs_roster(int rules, int np) { return 1 + rules + 4 * np; }
template <int ROS> struct Roster {
    static constexpr bool on = ROS != 0;
    static constexpr int rules = on ? (ROS - 1) & 3 : -1, NP = on ? (ROS - 1) >> 2 : -1, P = NP - 1;
};
#define ZS_ROSTER_BENCH zs_roster(ZS_RULES_EXTERMINATION, 3)  // the bench game: agent + 2 terminators, extermination

// identity of a lane group, passed by value to the out-of-line functions (keeps the caller's Env in registers)
struct GrpId { uint32_t b; int32_t env; int32_t gl; uint32_t gm; int32_t gshift; };
__device__ __forceinline__ Env env_of(const ZsParams& p, const GrpId& id) {
    Env e;
    e.b = id.b; e.env = id.env; e.env_global = p.env_base + (uint32_t)id.env; e.gl = id.gl; e.gm = id.gm; e.gshift = id.gshift;
    e.t = e.episode = e.deaths = e.zd = e.nlive = e.flags = e.prev_zd = e.ep_steps = 0;
    e.tmpl_saddr = 0;
    return e;
}
__device__ __forceinline__ GrpId id_of(const Env& e) { GrpId id; id.b = e.b; id.env = e.env; id.gl = e.gl; id.gm = e.gm; id.gshift = e.gshift; return id; }

template <int G, bool CV> __device__ __forceinline__ void scalars_from_lane(Env& e, int sc) {
    e.t = gbcast<G, CV>(e, sc, ZS_S_T); e.episode = gbcast<G, CV>(e, sc, ZS_S_EPISODE);
    e.deaths = gbcast<G, CV>(e, sc, ZS_S_DEATHS); e.zd = gbcast<G, CV>(e, sc, ZS_S_ZOMBIE_DEATHS);
    e.nlive = gbcast<G, CV>(e, sc, ZS_S_STAMP_COUNTER); e.flags = gbcast<G, CV>(e, sc, ZS_S_FLAGS);
    e.prev_zd = gbcast<G, CV>(e, sc, ZS_S_PREV_ZOMBIE_DEATHS); e.ep_steps = gbcast<G, CV>(e, sc, ZS_S_EPISODE_STEPS);
}
__device__ __forceinline__ int scalar_of_lane(const Env& e) {
    const int l = e.gl;
    return l == ZS_S_T ? e.t : l == ZS_S_EPISODE ? e.episode : l == ZS_S_DEATHS ? e.deaths
         : l == ZS_S_ZOMBIE_DEATHS ? e.zd : l == ZS_S_STAMP_COUNTER ? e.nlive
         : l == ZS_S_FLAGS ? e.flags : l == ZS_S_PREV_ZOMBIE_DEATHS ? e.prev_zd : e.ep_steps;
}
// hand-off through shared memory around the out-of-line functions
ZS_TPL __device__ __forceinline__ void scalars_from_smem(const ZsParams& p, Env& e) {
    ZS_CONSTS; ZS_VIEWS;
    gsync<G, CV>(e);
    e.t = SCALW(ZS_S_T); e.episode = SCALW(ZS_S_EPISODE); e.deaths = SCALW(ZS_S_DEATHS); e.zd = SCALW(ZS_S_ZOMBIE_DEATHS);
    e.nlive = SCALW(ZS_S_STAMP_COUNTER); e.flags = SCALW(ZS_S_FLAGS); e.prev_zd = SCALW(ZS_S_PREV_ZOMBIE_DEATHS);
    e.ep_steps = SCALW(ZS_S_EPISODE_STEPS);
}

// Dict-order ranks from arbitrary order-preserving stamps (state import / start of a launch): the rank of
// a thing in the world is the number of things in the world with a smaller stamp (A.2 of SURVEY.md).
// store_state writes the ranks themselves as stamps, so in a state this library left behind the stamps of the n
// things in the world are a permutation of 0 .. n-1 and ARE the ranks: that is checked first (every stamp below n,
// all n bits set), the counting loop is for imported states.
ZS_TPL __device__ __noinline__ int ranks_from_stamps(const ZsParams& p, GrpId id, int stamp0) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    const int env = id.env, lane = e.gl;
    const int32_t* st = p.STAMP + (size_t)env * p.Mp;
    constexpr int rw = (MPC + 31) / 32;
    int n = 0;
    bool bad = false;
    if (lane < rw) MASKW(lane) = 0u;
#pragma unroll 1
    for (int s0 = 0; s0 < (ONE ? 1 : (p.Mp)); s0 += G) {
        const int s = s0 + lane;
        n += __popc(gballot<G, CV>(e, s < p.Mp && (TM(s) & 0x80)));
    }
    gsync<G, CV>(e);
#pragma unroll 1
    for (int s0 = 0; s0 < (ONE ? 1 : (p.Mp)); s0 += G) {
        const int s = s0 + lane;
        const bool live = s < p.Mp && (TM(s) & 0x80);
        const int mine = live ? (s0 == 0 ? stamp0 : st[s]) : 0;  // (the first round's stamps came with the state, load_state)
        if (live) {
            if ((unsigned)mine < (unsigned)n) atomicOr(&MASKW(mine >> 5), 1u << (mine & 31));
            else bad = true;
        }
        if (s < p.Mp) {  // (provisional: the stamp as the rank)
            RK(s) = live ? (uint8_t)mine : (uint8_t)RK_NONE;
            MVQ(s) = RK_NONE;
        }
    }
    gsync<G, CV>(e);
    if (lane < rw) {
        const int full = n - 32 * lane;
        const uint32_t want = full >= 32 ? 0xffffffffu : full <= 0 ? 0u : (1u << full) - 1u;
        bad |= MASKW(lane) != want;
    }
    if (!gany<G, CV>(e, bad)) {
#pragma unroll 1
        for (int s0 = 0; s0 < (ONE ? 1 : (p.Mp)); s0 += G) {
            const int s = s0 + lane;
            if (s < p.Mp && (TM(s) & 0x80)) SOR(RK(s)) = (uint8_t)s;
        }
        gsync<G, CV>(e);
        return n;
    }
#pragma unroll 1
    for (int s0 = 0; s0 < (ONE ? 1 : (p.Mp)); s0 += G) {
        const int s = s0 + lane;
        const bool live = s < p.Mp && (TM(s) & 0x80);
        const int mine = live ? st[s] : 0;
        int r = 0;
#pragma unroll 1
        for (int j = 0; j < p.M; ++j) r += ((TM(j) & 0x80) && st[j] < mine);
        if (s < p.Mp) {
            RK(s) = live ? (uint8_t)r : (uint8_t)RK_NONE;
            if (live) SOR(r) = (uint8_t)s;
        }
    }
    gsync<G, CV>(e);
    return n;
}

// Build the static patch list (zs_device.cuh) from the static lives: state import / start of a launch.  Eight
// boxes/walls per lane (one 128-bit word of lives against one of MAX_LIFEs): almost all are pristine, the few lanes
// that find a difference list theirs behind the lanes before them (prefix sum of the counts).
ZS_TPL __device__ __noinline__ int scan_damaged_statics(const ZsParams& p, GrpId id, int fresh) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    const uint4* life4 = reinterpret_cast<const uint4*>(SLP);
    const uint4* max4 = reinterpret_cast<const uint4*>(p.static_max);
    const uint4* cell4 = reinterpret_cast<const uint4*>(p.static_cell);
    const int n8 = p.Sp >> 3;
    int n = 0;
#pragma unroll 1
    for (int i0 = 0; i0 < n8; i0 += G) {
        const int i8 = i0 + e.gl;
        uint4 lv = make_uint4(0u, 0u, 0u, 0u), mv = lv;
        uint4 cv = lv;  // the cells of the eight (issued with the lives: an entry then needs no trip of its own)
        if (i8 < n8) { lv = life4[i8]; mv = __ldg(max4 + i8); cv = __ldg(cell4 + i8); }
        const bool differs = ((lv.x ^ mv.x) | (lv.y ^ mv.y) | (lv.z ^ mv.z) | (lv.w ^ mv.w)) != 0u;
        uint32_t sx0 = 0u, sx1 = 0u;  // the eight SIDX bytes of this lane's boxes/walls
        if (gany<G, CV>(e, differs)) {
            const unsigned long long l0 = (unsigned long long)lv.x | ((unsigned long long)lv.y << 32), l1 = (unsigned long long)lv.z | ((unsigned long long)lv.w << 32);
            const unsigned long long m0 = (unsigned long long)mv.x | ((unsigned long long)mv.y << 32), m1 = (unsigned long long)mv.z | ((unsigned long long)mv.w << 32);
            auto pay_of = [&](int k, bool& listed) {
                const int sh = 16 * (k & 3);
                const int life = (int)(int16_t)((k & 4 ? l1 : l0) >> sh), mx = (int)(int16_t)((k & 4 ? m1 : m0) >> sh);
                const int pay = static_payload(p, mx, life, life > 0 || fresh);
                listed = life != mx && pay != static_payload(p, mx, mx, true);
                return pay;
            };
            // the boxes/walls whose life differs (one bit per 16-bit field), then the ones among them that show
            const uint32_t x0 = lv.x ^ mv.x, x1 = lv.y ^ mv.y, x2 = lv.z ^ mv.z, x3 = lv.w ^ mv.w;
            unsigned dm = ((x0 & 0xffffu) ? 1u : 0u) | ((x0 >> 16) ? 2u : 0u) | ((x1 & 0xffffu) ? 4u : 0u) | ((x1 >> 16) ? 8u : 0u) |
                          ((x2 & 0xffffu) ? 16u : 0u) | ((x2 >> 16) ? 32u : 0u) | ((x3 & 0xffffu) ? 64u : 0u) | ((x3 >> 16) ? 128u : 0u);
            unsigned lm = 0u;
#pragma unroll 1
            for (; dm; dm &= dm - 1u) {
                const int k = __ffs(dm) - 1;
                bool listed;
                pay_of(k, listed);
                if (listed && i8 * 8 + k < p.S) lm |= 1u << k;
            }
            const int c = __popc(lm);
            int inc = c;
#pragma unroll
            for (int d = 1; d < G; d <<= 1) { const int t = __shfl_up_sync(gmask<G, CV>(e), inc, d, G); if (e.gl >= d) inc += t; }
            int pos = n + inc - c;
            n += gbcast<G, CV>(e, inc, G - 1);
#pragma unroll 1
            for (unsigned mm = lm; mm; mm &= mm - 1u) {
                const int k = __ffs(mm) - 1;
                bool listed;
                const int pay = pay_of(k, listed);
                const uint32_t cw = k < 2 ? cv.x : k < 4 ? cv.y : k < 6 ? cv.z : cv.w;
                SPL(pos) = ((cw >> (16 * (k & 1))) & 0xffffu) | ((uint32_t)pay << 16);
                const uint32_t sb = (uint32_t)(pos + 1 < SIDX_FAR ? pos + 1 : SIDX_FAR) << (8 * (k & 3));
                if (k < 4) sx0 |= sb; else sx1 |= sb;
                ++pos;
            }
        }
        if (i8 < n8) *reinterpret_cast<uint2*>(SIDXP + 8 * i8) = make_uint2(sx0, sx1);
    }
    if (e.gl == 0) SPN = (uint16_t)n;
    gsync<G, CV>(e);
    return n == 0 ? 0 : FL_DMG;
}

// entry + 1 of a cell listed at or beyond entry SIDX_FAR - 1
ZS_TPL __device__ __forceinline__ int spl_find_far(const ZsParams& p, const Env& e, int cell) {
    ZS_VIEWS;
    int i = SIDX_FAR - 1;
    while ((int)(SPL(i) & 0xffffu) != cell) ++i;
    return i + 1;
}

// One box/wall changed (single-lane contexts): refresh or create its entry.
ZS_TPL __device__ __forceinline__ void spl_update_one(const ZsParams& p, const Env& e, int si, int cell, int life, bool present) {
    ZS_VIEWS;
    const int mx = __ldg(p.static_max + si);
    const int pay = static_payload(p, mx, life, present);
    int idx = SIDX(si);
    if (idx == 0) {
        if (pay == static_payload(p, mx, mx, true)) return;
        idx = (int)SPN + 1;
        SPN = (uint16_t)idx;
        SIDX(si) = (uint8_t)(idx < SIDX_FAR ? idx : SIDX_FAR);
    } else if (idx == SIDX_FAR) idx = spl_find_far<MPC, G, CV>(p, e, cell);
    SPL(idx - 1) = spl_entry(cell, pay);
}

// A new world: every box/wall is back in World.things, also the ones with life <= 0 (game.py:154-155).
// (An entry with a payload already shows its box/wall as present with its current life: only the entries of boxes/walls
// that were gone — SPL_GONE — change, so the map tables are only read for those.)  restore_grid: the grid is not
// rebuilt from the template by the caller; the returning boxes/walls are put back on it here.
ZS_TPL __device__ __forceinline__ void spl_refresh_present(const ZsParams& p, const Env& e, bool restore_grid = false) {
    ZS_VIEWS;
    const int n = SPN;
#pragma unroll 1
    for (int i = e.gl; i < n; i += G) {
        const uint32_t w = SPL(i);
        if (!spl_gone(w)) continue;
        const int cell = w & 0xffffu;
        const int si = __ldg(p.cell_static + cell);
        SPL(i) = spl_entry(cell, static_payload(p, __ldg(p.static_max + si), SL(si), true));
        if (restore_grid) GRID(cell) = G_STATIC;
    }
}

// First clean_dead_things of a world (core.py:121-138): every box/wall with life <= 0 leaves now.  Returns this
// lane's count.
ZS_TPL __device__ __forceinline__ int spl_clean_fresh(const ZsParams& p, const Env& e) {
    ZS_VIEWS;
    const int n = SPN;
    int gone = 0;
#pragma unroll 1
    for (int i = e.gl; i < n; i += G) {
        const int cell = SPL(i) & 0xffffu;
        if (!g_is_static(GRID(cell))) continue;
        if (SL(__ldg(p.cell_static + cell)) <= 0) { GRID(cell) = G_EMPTY; SPL(i) = spl_entry(cell, SPL_GONE); ++gone; }
    }
    return gone;
}

// The cells that carry a dead body, as a short list (or, past ZS_DEAD_CAP, a flag for bitmap scans).
ZS_TPL __device__ __noinline__ int scan_dead_bodies(const ZsParams& p, GrpId id) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    int n = 0;
#pragma unroll 1
    for (int w0 = 0; w0 < p.dead_words; w0 += G) {
        const int w = w0 + e.gl;
        uint32_t bits = w < p.dead_words ? DEADW(w) : 0u;
        // lanes take turns appending their word's cells (rare: once per launch)
#pragma unroll 1
        for (int l = 0; l < G; ++l) {
            const int cnt = gbcast<G, CV>(e, __popc(bits), l);
            if (e.gl == l) {
                int m = n;
                while (bits) {
                    const int b = __ffs(bits) - 1;
                    bits &= bits - 1;
                    if (m < ZS_DEAD_CAP) DBL(1 + m) = (uint16_t)(w * 32 + b);
                    ++m;
                }
            }
            n += cnt;
        }
    }
    if (e.gl == 0) DBL(0) = (uint16_t)(n < ZS_DEAD_CAP ? n : ZS_DEAD_CAP);
    gsync<G, CV>(e);
    return n <= ZS_DEAD_CAP ? 0 : FL_DEAD_OVER;
}

// with_lists: also build the dead-body list (worth it when the launch runs several steps; a single step walks the bitmap)
// for_reset: the world is about to be re-initialised — the dead-body bitmap, the tracker lives and the dict order are all
// set anew by the world init, so they are neither loaded nor derived (the slots are: one that is not placed again keeps
// what it holds, and the store writes every slot).
ZS_TPL __device__ __forceinline__ void load_state(const ZsParams& p, Env& e, bool with_lists, bool for_reset = false) {
    ZS_CONSTS; ZS_VIEWS;
    const size_t row = (size_t)e.env * p.Mp;
    // A launch starts with a handful of dependent round trips to memory unless the loads are issued together: the first
    // round of every field goes out back to back (all a small world has), then the values go to shared memory.
    const int s0 = e.gl;
    const bool has_slot = s0 < p.Mp;
    int x0 = 0, y0 = 0, l0 = 0, m0 = 0;
    int st0 = 0;
    if (has_slot) { x0 = p.X[row + s0]; y0 = p.Y[row + s0]; l0 = p.LIFE[row + s0]; m0 = p.META[row + s0]; st0 = p.STAMP[row + s0]; }
    const uint32_t* dead = p.DEAD + (size_t)e.env * p.dead_words;
    constexpr int DR = 96 / G;  // rounds of the dead-body bitmap issued up front (96 words = 3,072 cells)
    uint32_t dw[DR];
#pragma unroll
    for (int r = 0; r < DR; ++r) dw[r] = (!for_reset && e.gl + r * G < p.dead_words) ? dead[e.gl + r * G] : 0u;
    const int pv = (!for_reset && e.gl < p.Ap) ? (int)p.PREV[(size_t)e.env * p.Ap + e.gl] : 0;
    const bool sl_here = !(MPC > 32 && p.sl_global);
    const uint4* sl4 = (const uint4*)(p.SLIFE + (size_t)e.env * p.Sp);
    constexpr int SR = 32 / G;  // rounds of box/wall lives issued up front (32 words = 256 boxes/walls)
    uint4 sv[SR];
#pragma unroll
    for (int r = 0; r < SR; ++r) sv[r] = (sl_here && e.gl + r * G < (p.Sp >> 3)) ? sl4[e.gl + r * G] : make_uint4(0u, 0u, 0u, 0u);
    const int sc = e.gl < 8 ? p.SCAL[(size_t)e.env * 8 + e.gl] : 0;
    // ... and the same lines of the env a later CTA will work on are pulled into the L2 (the launch is a stream of
    // short-lived CTAs: without this every one of them starts with a trip to DRAM behind the observation writes)
    if (p.prefetch_ahead > 0 && e.env + p.prefetch_ahead < p.N) {
        const size_t pe = (size_t)(e.env + p.prefetch_ahead), prow = pe * p.Mp;
        if (has_slot) { prefetch_l2(p.X + prow + s0); prefetch_l2(p.Y + prow + s0); prefetch_l2(p.LIFE + prow + s0); prefetch_l2(p.META + prow + s0); prefetch_l2(p.STAMP + prow + s0); }
#pragma unroll
        for (int r = 0; r < DR; ++r) if (e.gl + r * G < p.dead_words) prefetch_l2(p.DEAD + pe * p.dead_words + e.gl + r * G);
        if (e.gl < p.Ap) prefetch_l2(p.PREV + pe * p.Ap + e.gl);
        if (sl_here) {
#pragma unroll
            for (int r = 0; r < SR; ++r) if (e.gl + r * G < (p.Sp >> 3)) prefetch_l2((const uint4*)(p.SLIFE + pe * p.Sp) + e.gl + r * G);
        }
        if (e.gl < 8) prefetch_l2(p.SCAL + pe * 8 + e.gl);
    }
    if (has_slot) { TXY(s0) = xy_pack(x0, y0); TL(s0) = (int16_t)l0; TM(s0) = (uint8_t)m0; }
#pragma unroll 1
    for (int s = s0 + G; s < p.Mp; s += G) {
        TXY(s) = xy_pack(p.X[row + s], p.Y[row + s]);
        TL(s) = p.LIFE[row + s]; TM(s) = p.META[row + s];
    }
#pragma unroll
    for (int r = 0; r < DR; ++r) if (e.gl + r * G < p.dead_words) DEADW(e.gl + r * G) = dw[r];
#pragma unroll 1
    for (int w = e.gl + DR * G; w < p.dead_words; w += G) DEADW(w) = for_reset ? 0u : dead[w];
    if (e.gl < p.Ap) PREVL(e.gl) = (int16_t)pv;
#pragma unroll 1
    for (int a = e.gl + G; a < p.Ap; a += G) PREVL(a) = for_reset ? (int16_t)0 : p.PREV[(size_t)e.env * p.Ap + a];
    if (sl_here) {
#pragma unroll
        for (int r = 0; r < SR; ++r) if (e.gl + r * G < (p.Sp >> 3)) reinterpret_cast<uint4*>(SLP)[e.gl + r * G] = sv[r];
#pragma unroll 1
        for (int i = e.gl + SR * G; i < (p.Sp >> 3); i += G) reinterpret_cast<uint4*>(SLP)[i] = sl4[i];
    }
    scalars_from_lane<G, CV>(e, sc);
    gsync<G, CV>(e);
    if (for_reset) e.nlive = 0;
    else e.nlive = ranks_from_stamps<MPC, G, false>(p, id_of(e), st0);
    e.flags = (e.flags & FL_FRESH) | scan_damaged_statics<MPC, G, false>(p, id_of(e), e.flags & FL_FRESH);
    if (ONE && with_lists) e.flags |= scan_dead_bodies<MPC, G, false>(p, id_of(e));
    else e.flags |= FL_DEAD_OVER;
}

ZS_TPL __device__ __forceinline__ void store_state(const ZsParams& p, Env& e) {
    ZS_CONSTS; ZS_VIEWS;
    gsync<G, CV>(e);
    const size_t row = (size_t)e.env * p.Mp;
#pragma unroll 1
    for (int s = e.gl; s < p.Mp; s += G) {
        const uint32_t xy = TXY(s);
        p.X[row + s] = (int16_t)xy_x(xy); p.Y[row + s] = (int16_t)xy_y(xy); p.LIFE[row + s] = TL(s);
        p.STAMP[row + s] = RK(s); p.META[row + s] = TM(s);
    }
#pragma unroll 1
    for (int w = e.gl; w < p.dead_words; w += G) p.DEAD[(size_t)e.env * p.dead_words + w] = DEADW(w);
#pragma unroll 1
    for (int a = e.gl; a < p.Ap; a += G) p.PREV[(size_t)e.env * p.Ap + a] = PREVL(a);
    if ((e.flags & FL_SL_DIRTY) && !(MPC > 32 && p.sl_global)) {
        uint4* sl4 = (uint4*)(p.SLIFE + (size_t)e.env * p.Sp);
#pragma unroll 1
        for (int i = e.gl; i < (p.Sp >> 3); i += G) sl4[i] = reinterpret_cast<const uint4*>(SLP)[i];
    }
    const int keep = e.flags;
    e.flags &= FL_FRESH;
    if (e.gl < 8) p.SCAL[(size_t)e.env * 8 + e.gl] = scalar_of_lane(e);
    e.flags = keep;
}

// ---------------------------------------------------------------- the parked image (zs_device.cuh: EnvS, "the IMAGE")
// Start of a launch: the group's lane 0 arms the env's mbarrier and issues ONE bulk copy of the whole image; the wait
// comes later (the caller puts independent work in between).  The canonical state is not read at all.
ZS_TPL __device__ __forceinline__ void load_image_issue(const ZsParams& p, const Env& e) {
    ZS_VIEWS;
    if (e.gl == 0) {
        mbar_init(&S.mbar, 1);
        mbar_expect_tx(&S.mbar, (uint32_t)p.img_bytes);
        bulk_load(zs_smem + e.b + img_off<MPC>(), p.img + (size_t)e.env * p.img_pitch, (uint32_t)p.img_bytes, &S.mbar);
    }
}
ZS_TPL __device__ __forceinline__ void load_image_wait(const ZsParams& p, Env& e) {
    ZS_VIEWS;
    __syncwarp(e.gm);  // (lane 0's mbarrier.init comes before anybody's wait)
    mbar_wait(&S.mbar, 0u);
    e.t = S.pscal[ZS_S_T]; e.episode = S.pscal[ZS_S_EPISODE]; e.deaths = S.pscal[ZS_S_DEATHS]; e.zd = S.pscal[ZS_S_ZOMBIE_DEATHS];
    e.nlive = S.pscal[ZS_S_STAMP_COUNTER]; e.prev_zd = S.pscal[ZS_S_PREV_ZOMBIE_DEATHS]; e.ep_steps = S.pscal[ZS_S_EPISODE_STEPS];
    e.flags = (S.pscal[ZS_S_FLAGS] & (FL_FRESH | FL_DEAD_OVER)) | (SPN ? FL_DMG : 0);
}
// End of a launch: the scalars join the image, the lanes' shared-memory writes are handed to the async proxy and lane 0
// sends the block back with one bulk copy (it must have been READ before the CTA may go: image_store_drain).
ZS_TPL __device__ __forceinline__ void store_image(const ZsParams& p, Env& e) {
    ZS_VIEWS;
    const int keep = e.flags;
    e.flags &= FL_FRESH | FL_DEAD_OVER;
    if (e.gl < 8) S.pscal[e.gl] = scalar_of_lane(e);
    e.flags = keep;
    fence_proxy_async_smem();
    __syncwarp(e.gm);
    if (e.gl == 0) {
        bulk_store(p.img + (size_t)e.env * p.img_pitch, zs_smem + e.b + img_off<MPC>(), (uint32_t)p.img_bytes);
        bulk_commit();
    }
}
__device__ __forceinline__ void image_store_drain(const Env& e) { if (e.gl == 0) bulk_wait_read_all(); }

// Rebuild the occupancy grid from the compact state.  FL_FRESH = first step after a world init:
// boxes/walls whose life is already <= 0 are still in World.things (game.py:154-155) until the
// first clean_dead_things.
ZS_TPL __device__ __noinline__ void build_grid(const ZsParams& p, GrpId id, int flags) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    const uint4* tg = (const uint4*)p.tmpl_grid;
#pragma unroll 4
    for (int i = e.gl; i < (p.cells_pad >> 4); i += G) reinterpret_cast<uint4*>(GRIDP)[i] = __ldg(tg + i);
    gsync<G, CV>(e);
    if (flags & FL_DMG) {  // boxes/walls that are gone from World.things (SPL_GONE in the static patch list)
        const int n = SPN;
#pragma unroll 1
        for (int i = e.gl; i < n; i += G) { const uint32_t w = SPL(i); if (spl_gone(w)) GRID(w & 0xffffu) = G_EMPTY; }
        gsync<G, CV>(e);
    }
#pragma unroll 1
    for (int w = e.gl; w < p.dead_words; w += G) {
        uint32_t bits = DEADW(w);
        while (bits) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            const int c = w * 32 + b;
            if (GRID(c) == G_EMPTY) GRID(c) = G_DEAD;
        }
    }
    gsync<G, CV>(e);
#pragma unroll 1
    for (int s = e.gl; s < p.M; s += G)
        if (TM(s) & 0x80) { const uint32_t xy = TXY(s); GRID(xy_y(xy) * p.W + xy_x(xy)) = (uint8_t)(s + 1); }
    gsync<G, CV>(e);
}

// ---------------------------------------------------------------- decide phase
// target id: mobile slot s -> s, static i -> M + i
__device__ __forceinline__ int target_of_cell(const ZsParams& p, int g, int cell) {
    return g <= G_MAX_SLOT ? g - 1 : p.M + (int)__ldg(p.cell_static + cell);
}

// A decided action, packed into one 64-bit word so that the sequential execute loop touches as little as
// possible; everything that cannot change before the actor acts is resolved when the word is built.
//   bits 0-2 kind, then per kind:
//   X_NOP       an action that can no longer have an effect but still takes part in the shuffle
//   X_MOVE      3-10 actor | 11 restore (dead body under the actor) | 16-31 destination cell | 32-47 current cell;
//               the destination is already known to be in bounds and one step away; its packed x/y is in BK(actor)
//   X_ATTACK_M / X_HEAL_M   3-10 mobile target slot | 11-17 range^2 | 18-24 lo | 25-30 n | 32-63 the actor's packed
//               x/y (it cannot move before it acts); the range is checked against the target's CURRENT position
//   X_ATTACK_S / X_HEAL_S   3-10 unused | 18-24 lo | 25-30 n | 32-47 static index; already known to be in range
//   The draw of an attack / heal is lo + randbelow(n).
#define X_NOP 0
#define X_MOVE 1
#define X_ATTACK_M 2
#define X_HEAL_M 3
#define X_ATTACK_S 4
#define X_HEAL_S 5
__device__ __forceinline__ unsigned long long pack_move(int actor, int restore, int c, int old) {
    // (the cell in uint32_t: on maps of 32,768 cells or more an int shift overflows, and the sign extension of the low word
    // would overwrite the old cell in the high word)
    return (unsigned long long)((uint32_t)(X_MOVE | (actor << 3) | (restore << 11)) | ((uint32_t)c << 16)) |
           ((unsigned long long)(uint32_t)old << 32);
}
__device__ __forceinline__ unsigned long long pack_hit(int kind, int target, int r2, int lo, int n, uint32_t hi) {
    return (unsigned long long)(uint32_t)(kind | (target << 3) | (r2 << 11) | (lo << 18) | (n << 25)) | ((unsigned long long)hi << 32);
}

// number of set bits below `bit` in the rank bit-mask starting at word `word0`
ZS_TPL __device__ __forceinline__ int prefix_popc(const ZsParams& p, const Env& e, int word0, int bit) {
    ZS_VIEWS;
    int n = 0;
#pragma unroll 1
    for (int w = 0; w < (bit >> 5); ++w) n += __popc(MASKW(word0 + w));
    return n + __popc(MASKW(word0 + (bit >> 5)) & ((1u << (bit & 31)) - 1u));
}

// ---------------------------------------------------------------- decide-phase draws with a randoman around
// A decision that draws is handed over as DTYPE(s) = D_WANDER (free adjacent cells as a bit-mask in BK(s)) or D_RANDOM
// and comes back packed in BK(s): type << 29 | (b + 1) << 15 | (a + 1) for a move to (a, b), type << 29 | target for a hit.
__device__ __forceinline__ uint32_t pack_decision(int type, int a, int b) {
    return ((uint32_t)type << 29) | ((uint32_t)(b + 1) << 15) | (uint32_t)(a + (type == D_MOVE ? 1 : 0));
}
__device__ __forceinline__ void unpack_decision(uint32_t w, int& type, int& a, int& b) {
    type = (int)(w >> 29);
    a = (int)(w & 0x7fffu) - (type == D_MOVE ? 1 : 0);
    b = (int)((w >> 15) & 0x3fffu) - 1;
}
// The draws of wandering zombies / hamsters (one each) and randomans (two or three each: what the second one means and
// whether there is a third depends on the first) are consumed in actor (dict) order, so with a randoman in the game the
// drawing actors are walked one after the other.  RandoMan.next_step (players/randoman.py:9-21): random.choice(('move',
// 'attack', 'heal')); attack / heal: random.choice(list(things.values())) — any thing of World.things by dict index:
// the boxes/walls still in the world in file order, then the mobile things in dict order; move: coordinate
// random.choice((0, 1)) changes by random.choice((-1, 1)), drawn in that order.  Returns the draws consumed.
ZS_TPL __device__ __noinline__ int decide_draws_seq(const ZsParams& p, GrpId id, int episode, uint32_t t_word, int nlive, int flags) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    e.episode = episode;
    const int lane = e.gl;
    const bool fresh = flags & FL_FRESH;
    int n_sp = 0;  // boxes/walls in World.things
#pragma unroll 1
    for (int i0 = 0; i0 < p.S; i0 += G) n_sp += __popc(gballot<G, CV>(e, i0 + lane < p.S && (SL(i0 + lane) > 0 || fresh)));
    int k = 0;
#pragma unroll 1
    for (int r = 0; r < nlive; ++r) {
        const int s = SOR(r);
        const int ty = DTYPE(s);
        if (ty != D_WANDER && ty != D_RANDOM) continue;
        const uint32_t xy = TXY(s);
        const int x = xy_x(xy), y = xy_y(xy);
        uint32_t out;
        if (ty == D_WANDER) {
            const unsigned fm = BK(s);
            int pick = below(draw_at(p, e, t_word, k), __popc(fm));
            k += 1;
            int d = 0;
            for (int q = 0; q < 4; ++q) if ((fm >> q) & 1u) { if (pick == 0) { d = q; break; } --pick; }
            out = pack_decision(D_MOVE, x + adj_dx(d), y + adj_dy(d));
        } else {
            const int action = below(draw_at(p, e, t_word, k), 3);
            if (action == 0) {
                const int axis = below(draw_at(p, e, t_word, k + 1), 2);
                const int sign = below(draw_at(p, e, t_word, k + 2), 2) ? 1 : -1;
                k += 3;
                out = pack_decision(D_MOVE, x + (axis == 0 ? sign : 0), y + (axis == 1 ? sign : 0));
            } else {
                const int idx = below(draw_at(p, e, t_word, k + 1), n_sp + nlive);
                k += 2;
                int target;
                if (idx >= n_sp) target = SOR(idx - n_sp);
                else {  // the idx-th box/wall that is still in the world, in file order
                    int base = 0, found = -1;
#pragma unroll 1
                    for (int i0 = 0; i0 < p.S && found < 0; i0 += G) {
                        unsigned m = gballot<G, CV>(e, i0 + lane < p.S && (SL(i0 + lane) > 0 || fresh));
                        const int c = __popc(m);
                        if (idx < base + c) {
                            for (int q = idx - base; q > 0; --q) m &= m - 1;
                            found = i0 + __ffs(m) - 1;
                        }
                        base += c;
                    }
                    target = p.M + found;
                }
                out = pack_decision(action == 1 ? D_ATTACK : D_HEAL, target, 0);
            }
        }
        gsync<G, CV>(e);  // (everybody has read BK(s))
        if (lane == 0) BK(s) = out;
    }
    gsync<G, CV>(e);
    return k;
}

// ---------------------------------------------------------------- World.step (core.py:72-78)
// General version: more slots than lanes (round loops over the slots).  Returns the draws consumed so far in this step.
ZS_TPL __device__ __forceinline__ int world_step(const ZsParams& p, Env& e) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl;
    constexpr int rw = (MPC + 31) / 32;
    const int NP = p.P + p.A;
    e.t += 1;
    const uint32_t t_word = (uint32_t)(e.t + 1);

    // ---- which players are in the world, and which of them look for their closest zombie
    // (terminators and snipers always, terminator.py:10-14, sniper.py:10-16; agents for attack_closest, agent.py:41-47)
    bool humans = false;
    unsigned needz0 = 0, needz1 = 0;  // slots < NP <= 64
#pragma unroll 1
    for (int s0 = 0; s0 < NP; s0 += G) {
        const int s = s0 + lane;
        bool needz = false;
        if (s < NP && (TM(s) & 0x80)) {
            humans = true;
            needz = s < p.P ? (p.bot_kinds[s] == ZS_KIND_TERMINATOR || p.bot_kinds[s] == ZS_KIND_SNIPER)
                            : ACTS(3 * (s - p.P)) == ZS_ACT_ATTACK_CLOSEST;
        }
        const unsigned m = gballot<G, CV>(e, needz);
        if (s0 == 0) needz0 = m; else needz1 = m;
        if (s < NP) ZB(s) = 0xffffffffu;
    }
    const bool has_humans = gany<G, CV>(e, humans);
    gsync<G, CV>(e);
    // ---- closest(self, others) (utils.py:23-31) for everybody from ONE pass over the (thing, player) distances:
    // a zombie (things.py:73-82) or a heal_closest agent (agent.py:79-86) takes the minimum over the players in
    // its own lane; a player's closest zombie is the minimum of the same distances across the zombie lanes
    // (redux.sync).  Key = (d^2 << 8) | dict rank: sorted() is stable, so ties go to the earlier thing.
#pragma unroll 1
    for (int s0 = 0; s0 < p.M; s0 += G) {
        const int s = s0 + lane;
        const uint32_t myrank = s < p.M ? RK(s) : RK_NONE;
        const bool live = myrank != RK_NONE;
        const bool zombie = s >= NP;
        const uint32_t xy = live ? TXY(s) : 0u;
        const int x = xy_x(xy), y = xy_y(xy);
        const bool wantp = live && (zombie ? has_humans : (s >= p.P && ACTS(3 * (s - p.P)) == ZS_ACT_HEAL_CLOSEST));
        const uint32_t zkey = (live && zombie) ? myrank : 0xffffffffu;
        uint32_t bestp = 0xffffffffu;
#pragma unroll 1
        for (int q = 0; q < NP; ++q) {
            const uint32_t rq = RK(q);
            if (rq == RK_NONE) continue;  // player q is not in the world (warp-uniform)
            const uint32_t qxy = TXY(q);
            const uint32_t d = (uint32_t)dist2(x, y, xy_x(qxy), xy_y(qxy)) << 8;
            if (wantp && q != s) bestp = min(bestp, d | rq);
            if (((q < 32 ? needz0 : needz1) >> (q & 31)) & 1u) {
                const uint32_t m = gminu<G, CV>(e, d | zkey);
                if (lane == 0 && m < ZB(q)) ZB(q) = m;
            }
        }
        if (s < p.Mp) BK(s) = bestp;
    }
    gsync<G, CV>(e);

    // ---- get_actions (core.py:80-101): every actor decides against the pre-step world
    bool any_wander = false;
    int n_idle = 0;
#pragma unroll 1
    for (int s0 = 0; s0 < p.M; s0 += G) {
        const int s = s0 + lane;
        const bool live = s < p.M && RK(s) != RK_NONE;
        const uint32_t xy = live ? TXY(s) : 0u;
        const int x = xy_x(xy), y = xy_y(xy);
        const bool zombie = s >= NP, agent = !zombie && s >= p.P;
        int at = ZS_ACT_NONE, adx = 0, ady = 0;
        if (live && agent) {
            at = ACTS(3 * (s - p.P)); adx = ACTS(3 * (s - p.P) + 1); ady = ACTS(3 * (s - p.P) + 2);
            if (at == ZS_ACT_ABSENT) { at = ZS_ACT_HEAL; adx = 0; ady = 0; }  // multiagent_env.py:129-131
        }
        uint32_t key = 0xffffffffu;
        if (live) key = (zombie || at == ZS_ACT_HEAL_CLOSEST) ? BK(s) : ZB(s);
        const int tg = key == 0xffffffffu ? -1 : (int)SOR(key & 255u);
        const int d2 = (int)(key >> 8);
        int type = D_IDLE, a = 0, b = 0;
        if (live) {
            const uint32_t gxy = tg >= 0 ? TXY(tg) : 0u;
            const int gx = xy_x(gxy), gy = xy_y(gxy);
            if (!agent) {
                // the four adjacent cells (utils.py:34-44): what is on them and how far they are from the target
                unsigned freemask = 0, gs[4];
                int dd[4];
#pragma unroll
                for (int d = 0; d < 4; ++d) {  // no bounds check: cells outside the map hold nothing (utils.py:47-52)
                    gs[d] = grid_at(p, GRIDP, x + adj_dx(d), y + adj_dy(d));
                    dd[d] = dist2(gx, gy, x + adj_dx(d), y + adj_dy(d));
                    if (!g_is_thing(gs[d])) freemask |= 1u << d;
                }
                if (zombie) {  // Zombie.next_step (things.py:70-105)
                    if (!has_humans) {
                        if (freemask) { type = D_WANDER; a = (int)freemask; any_wander = true; }
                    } else if (d2 <= 2) { type = D_ATTACK; a = tg; }  // distance < 1.5 (things.py:83)
                    else {
                        // free cells: closest(target, positions), first minimum in adjacency order; boxed in: the first
                        // Box/Wall among the adjacent cells stably sorted by distance to the target (things.py:88-99)
                        int bdir = -1, bdist = 0x7fffffff;
#pragma unroll
                        for (int d = 0; d < 4; ++d) {
                            const bool cand = freemask ? ((freemask >> d) & 1u) : g_is_static(gs[d]);
                            if (cand && dd[d] < bdist) { bdir = d; bdist = dd[d]; }
                        }
                        if (bdir >= 0) {
                            const int cx = x + adj_dx(bdir), cy = y + adj_dy(bdir);
                            if (freemask) { type = D_MOVE; a = cx; b = cy; }
                            else { type = D_ATTACK; a = p.M + (int)__ldg(p.cell_static + cy * p.W + cx); }
                        }
                    }
                } else if (p.bot_kinds[s] == ZS_KIND_SNIPER) {  // Sniper.next_step (players/sniper.py:9-19)
                    if (tg >= 0) { type = D_ATTACK; a = tg; }
                } else if (p.bot_kinds[s] == ZS_KIND_TROLL) {   // Troll.next_step (players/troll.py:10-12)
                    type = D_HEAL; a = s;
                } else if (p.bot_kinds[s] == ZS_KIND_HAMSTER) { // Hamster.next_step (players/hamster.py:10-14)
                    if (freemask) { type = D_WANDER; a = (int)freemask; any_wander = true; }
                } else if (p.bot_kinds[s] == ZS_KIND_RANDOMAN) { // RandoMan.next_step: resolved in decide_draws_seq
                    type = D_RANDOM; any_wander = true;
                } else {  // Terminator.next_step (players/terminator.py:9-37)
                    if (tg < 0) { type = D_HEAL; a = s; }
                    else if (d2 > c_range2[TM(s) & 15]) {
                        int bdir = 0, bdist = 0x7fffffff, g = 0;
#pragma unroll
                        for (int d = 0; d < 4; ++d)  // closest(target, adjacent_positions(self)): out-of-bounds cells included
                            if (dd[d] < bdist) { bdir = d; bdist = dd[d]; g = (int)gs[d]; }
                        const int bx = x + adj_dx(bdir), by = y + adj_dy(bdir);
                        if (g_is_thing(g)) {
                            type = (g <= G_MAX_SLOT && (g - 1) < NP) ? D_HEAL : D_ATTACK;
                            a = target_of_cell(p, g, by * p.W + bx);
                        } else { type = D_MOVE; a = bx; b = by; }
                    } else { type = D_ATTACK; a = tg; }
                }
            } else {  // Agent.next_step (players/agent.py:28-96)
                // (a step of two cells or more fails whatever its length, core.py:149-153: deltas are clamped to +-2 so
                // that an unchecked user value can neither overflow nor wrap in the 16-bit hand-off below)
                if (at == ZS_ACT_MOVE) { type = D_MOVE; a = x + max(-2, min(2, adx)); b = y + max(-2, min(2, ady)); }
                else if (at == ZS_ACT_ATTACK_CLOSEST) { if (tg >= 0) { type = D_ATTACK; a = tg; } }
                else if (at == ZS_ACT_HEAL_CLOSEST) { type = D_HEAL; a = tg >= 0 ? tg : s; }
                else if (at == ZS_ACT_ATTACK || at == ZS_ACT_HEAL) {
                    if (at == ZS_ACT_HEAL && adx == 0 && ady == 0) { type = D_HEAL; a = s; }
                    else {
                        adx = max(-4096, min(4096, adx)); ady = max(-4096, min(4096, ady));  // (off the map either way)
                        const int g = grid_at(p, GRIDP, x + adx, y + ady);
                        // attack: any thing; heal: Player / Box / Wall only (agent.py:69-75)
                        const bool ok = at == ZS_ACT_ATTACK ? g_is_thing(g)
                                                            : (g_is_static(g) || (g_is_thing(g) && (g - 1) < NP));
                        if (ok) { type = at == ZS_ACT_ATTACK ? D_ATTACK : D_HEAL; a = target_of_cell(p, g, (y + ady) * p.W + (x + adx)); }
                    }
                }
            }
            n_idle += type == D_IDLE;
        }
        if (s < p.Mp) { DTYPE(s) = (uint8_t)type; DA(s) = (int16_t)a; DB(s) = (int16_t)b; }
    }
    n_idle = gadd<G, CV>(e, n_idle);
    gsync<G, CV>(e);
    int nd = 0;
    if (p.has_randoman) {
        if (gany<G, CV>(e, any_wander)) {
#pragma unroll 1
            for (int s = e.gl; s < p.M; s += G) if (DTYPE(s) == D_WANDER) BK(s) = (uint32_t)DA(s);
            gsync<G, CV>(e);
            nd = decide_draws_seq<MPC, G, false>(p, id_of(e), e.episode, t_word, e.nlive, e.flags);
#pragma unroll 1
            for (int s = e.gl; s < p.M; s += G) {
                if (DTYPE(s) != D_WANDER && DTYPE(s) != D_RANDOM) continue;
                int ty, a, b;
                unpack_decision(BK(s), ty, a, b);
                DTYPE(s) = (uint8_t)ty; DA(s) = (int16_t)a; DB(s) = (int16_t)b;
            }
            gsync<G, CV>(e);
        }
    } else if (gany<G, CV>(e, any_wander)) {
        // wandering zombies and hamsters draw random.choice(positions) in dict order (things.py:101-103, hamster.py:12-14)
        int mine = 0;
#pragma unroll 1
        for (int s = e.gl; s < p.M; s += G) {
            if (DTYPE(s) != D_WANDER) continue;
            int rank = 0;
#pragma unroll 1
            for (int j = 0; j < p.M; ++j) rank += (DTYPE(j) == D_WANDER && RK(j) < RK(s));
            const unsigned fm = (unsigned)DA(s);
            int pick = below(draw_at(p, e, t_word, rank), __popc(fm));
            int d = 0;
            for (int q = 0; q < 4; ++q) if ((fm >> q) & 1u) { if (pick == 0) { d = q; break; } --pick; }
            const uint32_t xy = TXY(s);
            DA(s) = (int16_t)(xy_x(xy) + adj_dx(d)); DB(s) = (int16_t)(xy_y(xy) + adj_dy(d));
            ++mine;
        }
        nd = gadd<G, CV>(e, mine);
        gsync<G, CV>(e);
#pragma unroll 1
        for (int s = e.gl; s < p.M; s += G) if (DTYPE(s) == D_WANDER) DTYPE(s) = D_MOVE;
        gsync<G, CV>(e);
    }
    // actions list in actor (dict) order (core.py:83-90): the position of an acting thing is its dict rank minus
    // the idle things before it (idle things are rare: usually the rank is the position).
    // Everything that cannot change before the actor acts is resolved here, in parallel.
    int cnt = 0, n_ah = 0;
#pragma unroll 1
    for (int s0 = 0; s0 < p.M; s0 += G) {
        const int s = s0 + lane;
        const int type = s < p.M ? DTYPE(s) : D_IDLE;  // D_IDLE for everything that is not in the world
        int pos = s < p.M ? RK(s) : 0;
        if (n_idle) {
            const int mine = pos;
#pragma unroll 1
            for (int j = 0; j < p.M; ++j) pos -= (RK(j) < mine && DTYPE(j) == D_IDLE);
        }
        unsigned long long word = X_NOP;
        bool acting = type != D_IDLE;
        if (acting) {
            const int a = DA(s), b = DB(s);
            const uint32_t xy = TXY(s);
            const int x = xy_x(xy), y = xy_y(xy);
            if (type == D_MOVE) {  // in bounds and at most one step (core.py:149-153); occupancy is checked when it runs
                if ((unsigned)a < (unsigned)p.W && (unsigned)b < (unsigned)p.H && dist2(x, y, a, b) <= 1) {
                    const int old = y * p.W + x;
                    word = pack_move(s, (DEADW(old >> 5) >> (old & 31)) & 1u, b * p.W + a, old);
                    BK(s) = xy_pack(a, b);
                }
            } else {
                const bool is_static = a >= p.M;
                int mx = 100, r2, dlo, dn;
                if (type == D_ATTACK) { const int w = TM(s) & 15; r2 = c_range2[w]; dlo = c_dmg_lo[w]; dn = c_dmg_n[w]; }
                else {  // heal: randint(MAX_LIFE // 10, MAX_LIFE // 4) of the target's class, range 3 (core.py:194-198)
                    if (is_static) mx = max_life_of_label(__ldg(p.static_label + (a - p.M)));
                    r2 = 9; dlo = mx / 10; dn = mx / 4 - mx / 10 + 1;
                }
                if (is_static) {
                    const int cell = __ldg(p.static_cell + (a - p.M));
                    const int gy = cell / p.W, gx = cell - gy * p.W;
                    if (dist2(x, y, gx, gy) <= r2) { word = pack_hit(type == D_ATTACK ? X_ATTACK_S : X_HEAL_S, 0, 0, dlo, dn, (uint32_t)(a - p.M)); ++n_ah; }
                } else { word = pack_hit(type == D_ATTACK ? X_ATTACK_M : X_HEAL_M, a, r2, dlo, dn, xy); ++n_ah; }
            }
            ++cnt;
        }
        if (acting) ACT(pos) = word;
    }
    const int L = gadd<G, CV>(e, cnt);
    n_ah = gadd<G, CV>(e, n_ah);
    // ---- draws of this step, generated 4 per lane (counter-based: any k is available directly)
    const int n_need = nd + (L > 1 ? L - 1 : 0) + n_ah;
#pragma unroll 1
    for (int blk = lane; blk * 4 < n_need; blk += G)
        reinterpret_cast<uint4*>(S.draws)[blk] = philox_draws(p, e.env_global, (uint32_t)e.episode, t_word, (uint32_t)blk);
    gsync<G, CV>(e);
    // Fisher-Yates partner of every iteration (random.shuffle: for i = L-1 .. 1: j = randbelow(i + 1))
#pragma unroll 1
    for (int i = 1 + e.gl; i < L; i += G) DTYPE(i) = (uint8_t)below(DRAWS(nd + (L - 1 - i)), i + 1);
    gsync<G, CV>(e);

    // ---- random.shuffle (core.py:76): the swaps are a fixed sequence once the partners are known, and where an element
    // ends up can be read off them without running it.  Iteration i (i = L-1 .. 1) swaps positions i and j_i <= i and
    // is the last one to touch position i.  So an element at position q: the largest iteration i > q with j_i == q takes
    // it to its final position i; if there is none, iteration q takes it to j_q (final if j_q == q, or q == 0), where
    // the next smaller iteration with the same partner j_q finds it, and so on.  The iterations that hit a position are
    // chained in shared memory (head = the largest, next = the next smaller one with the same partner), built 32
    // iterations at a time with match.any; every lane then follows its own elements (lane, lane + 32, ...), two hops
    // on average, instead of all L swaps.
    int k = nd + (L > 1 ? L - 1 : 0);
    int nmv = 0;
    {
        static_assert(G == 32, "the general step function runs one env per warp");
        constexpr int R = MPC / 32;
        uint8_t* const HITH = S.mpos;   // both arrays are (re)initialised for their own purpose right below
        uint8_t* const HITN = S.mvp;
#pragma unroll 1
        for (int q = lane; q < L; q += 32) HITH[q] = 0;  // 0 = none (an iteration that hits q is > q >= 0)
        gsync<G, CV>(e);
#pragma unroll 1
        for (int i0 = 1; i0 < L; i0 += 32) {  // ascending, so that the head ends up the largest
            const int i = i0 + lane;
            const int j = i < L ? (int)DTYPE(i) : i;
            const bool hit = j != i;  // (a swap with itself moves nothing)
            const unsigned grp = __match_any_sync(0xffffffffu, hit ? (uint32_t)j : 0xffffu);
            const unsigned lower = grp & ((1u << lane) - 1u), higher = grp & ~((2u << lane) - 1u);
            int prev = 0;
            if (hit) prev = lower ? i0 + 31 - __clz(lower) : (int)HITH[j];
            gsync<G, CV>(e);
            if (hit) { HITN[i] = (uint8_t)prev; if (!higher) HITH[j] = (uint8_t)i; }
            gsync<G, CV>(e);
        }
        int fp[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            int q = lane + 32 * r;
            if (q < L) {
                int h = HITH[q];
#pragma unroll 1
                while (h == 0 && q != 0) {  // nobody takes it from q: iteration q moves it to j_q ...
                    const int nq = DTYPE(q);
                    if (nq == q) break;
                    h = HITN[q];            // ... where the next iteration below q that hits j_q finds it
                    q = nq;
                }
                if (h) q = h;
            }
            fp[r] = q;
        }
        gsync<G, CV>(e);
#pragma unroll 1
        for (int s = lane; s < p.Mp; s += G) { S.mpos[s] = RK_NONE; S.mvp[s] = RK_NONE; }
        gsync<G, CV>(e);
        // the words move to their places within the one list (through registers)
        unsigned long long wr[R];
#pragma unroll
        for (int r = 0; r < R; ++r) wr[r] = lane + 32 * r < L ? ACT(lane + 32 * r) : 0ull;
        gsync<G, CV>(e);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (lane + 32 * r < L) {
                ACT(fp[r]) = wr[r];
                if (((uint32_t)wr[r] & 7u) == X_MOVE) S.mpos[((uint32_t)wr[r] >> 3) & 0xffu] = (uint8_t)fp[r];
            }
        }
        gsync<G, CV>(e);
    }
    // ---- execute_actions (core.py:103-119) in chunks of 32 list positions: within a chunk the resolution of
    // world_step_one (first mover per free destination by match.any, hits grouped per target, ballot-prefix draw
    // indices); a chunk sees the world the chunks before it left.  A move into a cell whose occupant moves earlier in
    // the SAME chunk sends that chunk through the sequential loop.
    const unsigned below_l = (1u << lane) - 1u;
    int16_t* const KILL = S.da;  // boxes/walls whose life fell to <= 0 during this step (DA is free once the words are built;
    int nk = 0;                  // at most one entry per hit: <= L <= MPC; repeats allowed)
#pragma unroll 1
    for (int base = 0; base < L; base += 32) {
        const int q = base + lane;  // list position
        const unsigned long long pk = q < L ? ACT(q) : 0ull;
        const uint32_t lo32 = (uint32_t)pk, hi32 = (uint32_t)(pk >> 32);
        int kind = lo32 & 7;
        const int who = (lo32 >> 3) & 0xff;  // the actor of a move, the mobile target of a hit
        const int c = lo32 >> 16;
        const int g0 = kind == X_MOVE ? (int)GRID(c) : G_STATIC;
        bool need_seq = false;
        if (kind == X_MOVE && g0 >= 1 && g0 <= G_MAX_SLOT) { const int mp = S.mpos[g0 - 1]; need_seq = mp >= base && mp < q; }
        if (gany<G, CV>(e, need_seq)) {
            if (lane == 0) {  // this chunk in list order on shared memory
                int fl = e.flags, n_touched = 0;
                const int end = base + 32 < L ? base + 32 : L;
#pragma unroll 1
                for (int i = base; i < end; ++i) {
                    const unsigned long long w = ACT(i);
                    const uint32_t l32 = (uint32_t)w, h32 = (uint32_t)(w >> 32);
                    const int kd = l32 & 7;
                    if (kd == X_NOP) continue;
                    if (kd == X_MOVE) {  // World.thing_move (core.py:140-166)
                        const int cc = l32 >> 16;
                        if (!g_is_thing(GRID(cc))) {
                            const int actor = (l32 >> 3) & 0xff;
                            GRID(h32 & 0xffffu) = (l32 & 0x800u) ? G_DEAD : G_EMPTY;
                            GRID(cc) = (uint8_t)(actor + 1);
                            TXY(actor) = BK(actor);
                            S.mvp[actor] = (uint8_t)i;
                            MVQ(actor) = (uint8_t)nmv++;  // things[dest] = thing; del things[old]: goes last in the dict
                        }
                        continue;
                    }
                    const int dlo = (l32 >> 18) & 127, dn = (l32 >> 25) & 63;
                    if (kd <= X_HEAL_M) {  // mobile target: distance between CURRENT positions (core.py:176,194)
                        const int a = (l32 >> 3) & 0xff;
                        const uint32_t gxy = TXY(a);
                        if (dist2(xy_x(h32), xy_y(h32), xy_x(gxy), xy_y(gxy)) > (int)((l32 >> 11) & 127)) continue;
                        const int amount = dlo + below(DRAWS(k++), dn);
                        if (kd == X_ATTACK_M) TL(a) = (int16_t)(TL(a) - amount);
                        else { const int nl = TL(a) + amount; TL(a) = (int16_t)(nl < 100 ? nl : 100); }
                    } else {
                        const int a = h32 & 0xffffu;
                        const int amount = dlo + below(DRAWS(k++), dn);
                        if (kd == X_ATTACK_S) SL(a) = (int16_t)(SL(a) - amount);
                        else {
                            const int mx = __ldg(p.static_max + a);
                            const int nl = SL(a) + amount;
                            SL(a) = (int16_t)(nl < mx ? nl : mx);
                        }
                        LIST(n_touched++) = (uint16_t)a;
                        fl |= FL_SL_DIRTY;
                    }
                }
                // the boxes/walls hit in this chunk: their patch-list entries.  A box/wall destroyed now stays in
                // World.things — later movers still bump into it, a heal may bring it back — until clean_dead_things
                // (core.py:121-138): it is only remembered here (KILL) and leaves in the clean phase below.
#pragma unroll 1
                for (int i = 0; i < n_touched; ++i) {
                    const int si = LIST(i);
                    const int cell = __ldg(p.static_cell + si);
                    const int life = SL(si);
                    const bool fresh = fl & FL_FRESH;
                    if (life <= 0 && !fresh && g_is_static(GRID(cell))) KILL[nk++] = (int16_t)si;
                    spl_update_one<MPC, G, CV>(p, e, si, cell, life, life > 0 || fresh);
                }
                if (SPN) fl |= FL_DMG;
                e.flags = fl;
            }
            k = gbcast<G, CV>(e, k, 0);
            nmv = gbcast<G, CV>(e, nmv, 0);
            nk = gbcast<G, CV>(e, nk, 0);
            e.flags = gbcast<G, CV>(e, e.flags, 0);
            gsync<G, CV>(e);
            continue;
        }
        // ---- moves (World.thing_move, core.py:140-166)
        const bool dest_free = kind == X_MOVE && !g_is_thing(g0);
        const unsigned want = gmatch<G, CV>(e, dest_free ? (uint32_t)c : 0x10000u);
        const bool success = dest_free && !(want & below_l);
        const unsigned succ_m = gballot<G, CV>(e, success);
        if (success) {
            GRID(hi32 & 0xffffu) = (lo32 & 0x800u) ? G_DEAD : G_EMPTY;
            GRID(c) = (uint8_t)(who + 1);
            S.mvp[who] = (uint8_t)q;
            MVQ(who) = (uint8_t)(nmv + __popc(succ_m & below_l));  // things[dest] = thing; del things[old]: goes last in the dict
        }
        nmv += __popc(succ_m);
        gsync<G, CV>(e);
        // ---- hits (World.thing_attack / thing_heal, core.py:168-208)
        const bool on_static = kind >= X_ATTACK_S;
        bool inrange = on_static;  // boxes/walls do not move: their range was checked when the word was built
        if (kind == X_ATTACK_M || kind == X_HEAL_M) {  // distance between CURRENT positions (core.py:176,194)
            uint32_t txy = TXY(who);
            const int mp = S.mvp[who];
            if (mp >= base && mp < q) txy = BK(who);  // (moves of earlier chunks are in TXY already)
            inrange = dist2(xy_x(hi32), xy_y(hi32), xy_x(txy), xy_y(txy)) <= (int)((lo32 >> 11) & 127);
        }
        if (gany<G, CV>(e, inrange)) {
            const unsigned hit_m = gballot<G, CV>(e, inrange);
            const int si = hi32 & 0xffffu;
            const bool heal = kind == X_HEAL_M || kind == X_HEAL_S;
            if (inrange) {
                const int amount = (int)((lo32 >> 18) & 127) + below(DRAWS(k + __popc(hit_m & below_l)), (int)((lo32 >> 25) & 63));
                LIST(lane) = (uint16_t)(amount | (heal ? 0x8000 : 0));
            }
            k += __popc(hit_m);
            const uint32_t tid = on_static ? 0x100u + (uint32_t)si : (uint32_t)who;
            const unsigned grp = gmatch<G, CV>(e, inrange ? tid : 0x20000u);
            const bool lead = inrange && !(grp & below_l);  // the first hit on a target applies all of them, in order
            gsync<G, CV>(e);
            int life = 0;
            if (lead) {
                life = on_static ? (int)SL(si) : (int)TL(who);
                const int mx = on_static ? (int)__ldg(p.static_max + si) : 100;
                unsigned bits = grp;
                while (bits) {
                    const int v = LIST(__ffs(bits) - 1);
                    bits &= bits - 1;
                    if (v & 0x8000) { life += v & 0x7fff; life = life < mx ? life : mx; }
                    else life -= v;
                }
                if (on_static) SL(si) = (int16_t)life; else TL(who) = (int16_t)life;
            }
            const bool slead = lead && on_static;
            if (gany<G, CV>(e, slead)) {
                bool is_new = false, gone = false;
                int cell = 0, pay = 0, idx = 0;
                if (slead) {
                    const int mx = __ldg(p.static_max + si);
                    const bool fresh = e.flags & FL_FRESH;
                    cell = __ldg(p.static_cell + si);
                    gone = life <= 0 && !fresh && g_is_static(GRID(cell));  // (leaves in the clean phase: see KILL above)
                    pay = static_payload(p, mx, life, life > 0 || fresh);
                    idx = SIDX(si);
                    is_new = idx == 0 && pay != static_payload(p, mx, mx, true);
                }
                const unsigned gone_m = gballot<G, CV>(e, gone);
                if (gone) KILL[nk + __popc(gone_m & below_l)] = (int16_t)si;
                nk += __popc(gone_m);
                e.flags |= FL_SL_DIRTY;
                const unsigned new_m = gballot<G, CV>(e, is_new);
                const int n0 = SPN;
                gsync<G, CV>(e);  // (everybody has read the count before lane 0 rewrites it)
                if (is_new) { idx = n0 + __popc(new_m & below_l) + 1; SIDX(si) = (uint8_t)(idx < SIDX_FAR ? idx : SIDX_FAR); }
                else if (idx == SIDX_FAR) idx = spl_find_far<MPC, G, CV>(p, e, cell);
                if (slead && idx) SPL(idx - 1) = spl_entry(cell, pay);
                if (new_m) {
                    if (lane == 0) SPN = (uint16_t)(n0 + __popc(new_m));
                    e.flags |= FL_DMG;
                }
            }
        }
        gsync<G, CV>(e);
        if (success) TXY(who) = BK(who);  // the chunk's movers arrive (the hits above needed both positions)
        gsync<G, CV>(e);
    }

    // ---- clean_dead_things (core.py:121-138)
    int nd_all = 0, nd_z = 0;
    if (e.flags & FL_FRESH) {  // first step of this world: every box/wall with life <= 0 leaves now
        if (e.flags & FL_DMG) nd_all = spl_clean_fresh<MPC, G, CV>(p, e);
        e.flags &= ~FL_FRESH;
    } else if (nk > 0) {
        // the boxes/walls destroyed during execute_actions leave now, unless a later heal brought them back (rare: one
        // lane walks the few candidates; a box/wall listed twice is gone from the grid the second time)
        if (lane == 0) {
#pragma unroll 1
            for (int i = 0; i < nk; ++i) {
                const int si = KILL[i];
                const int cell = __ldg(p.static_cell + si);
                const int life = SL(si);
                if (life <= 0 && g_is_static(GRID(cell))) { GRID(cell) = G_EMPTY; ++nd_all; }
                // (the patch-list payload follows the final life: a hit wrote "gone" while the life was <= 0)
                else if (life > 0) spl_update_one<MPC, G, CV>(p, e, si, cell, life, true);
            }
        }
        gsync<G, CV>(e);
    }
    for (int w = e.gl; w < 2 * rw; w += G) MASKW(w) = 0u;
    gsync<G, CV>(e);
#pragma unroll 1
    for (int s = e.gl; s < p.M; s += G) {
        const int r = RK(s);
        if (r == RK_NONE) continue;
        if (TL(s) <= 0) {
            const uint32_t xy = TXY(s);
            const int c = xy_y(xy) * p.W + xy_x(xy);
            GRID(c) = G_DEAD;                         // DeadBody overwrites any decoration (core.py:30-31,126-128)
            atomicOr(&DEADW(c >> 5), 1u << (c & 31));
            TM(s) &= 0x7f;
            ++nd_all;
            nd_z += s >= NP;
        } else {  // survivors: the ones that did not move keep their relative order, the movers follow in move order
            const int q = MVQ(s);
            if (q == RK_NONE) atomicOr(&MASKW(r >> 5), 1u << (r & 31));
            else atomicOr(&MASKW(rw + (q >> 5)), 1u << (q & 31));
        }
    }
    nd_all = gadd<G, CV>(e, nd_all);
    e.deaths += nd_all;
    e.zd += gadd<G, CV>(e, nd_z);
    gsync<G, CV>(e);
    // ---- new dict order: World.things after the moves (re-inserted at the end, core.py:158-159) and the deletions
    if (nmv > 0 || nd_all > 0) {
        int stayers = 0;
#pragma unroll 1
        for (int w = 0; w < rw; ++w) stayers += __popc(MASKW(w));
        int nl = 0;
#pragma unroll 1
        for (int s0 = 0; s0 < p.M; s0 += G) {
            const int s = s0 + lane;
            int r = s < p.M ? RK(s) : RK_NONE;
            if (r != RK_NONE) {
                if (!(TM(s) & 0x80)) r = RK_NONE;
                else {
                    const int q = MVQ(s);
                    r = q == RK_NONE ? prefix_popc<MPC, G, CV>(p, e, 0, r) : stayers + prefix_popc<MPC, G, CV>(p, e, rw, q);
                    SOR(r) = (uint8_t)s;
                }
                RK(s) = (uint8_t)r;
                MVQ(s) = RK_NONE;
            }
            nl += __popc(gballot<G, CV>(e, r != RK_NONE));
        }
        e.nlive = nl;
        gsync<G, CV>(e);
    }
    return k;
}

// ---------------------------------------------------------------- World.step when every slot has its own lane
// (MPC <= G).  Same semantics as world_step above, organised for short dependent chains and no divergence
// between the two envs of a warp in half-warp mode:
//   * SLOT SPACE (lane = slot): everything an actor decides stays in registers; closest-zombie keys land in the
//     player's own lane straight from redux.sync.min; wander / idle bookkeeping uses rank bit-masks from redux.sync.or.
//   * the Fisher-Yates partners are exchanged with shuffles, every lane follows its own action to its position.
//   * POSITION SPACE (lane = position in the shuffled action list): execute_actions (core.py:103-119) is sequential
//     by definition, but its dependencies are few and can be decided up front:
//       - a move succeeds iff its destination holds no thing when it runs.  A destination that is free before the
//         step goes to the FIRST mover that wants it (match.any on the cell, lowest position wins; the winner can
//         not leave again); a box/wall never leaves during execute; a mobile thing only leaves through its own
//         move, so the move fails unless that move comes EARLIER in the list — the one case that needs the
//         sequential loop (execute_sequential), an agent walking into a cell somebody is just leaving;
//       - a hit on a mobile target checks the range against the target's position at that time: its destination
//         if its successful move comes earlier in the list, else its old position;
//       - the draw index of a hit is the number of in-range hits before it (ballot prefix);
//       - the hits on one target (match.any on the target) are applied in list order by the first of them.
#define MVP(i) S.mvq[i]      // position of the slot's successful move in this step's list, RK_NONE if none
#define MPOS(i) S.dtype[i]   // position of the slot's (valid) move action in the list, RK_NONE if none
#define AMT(i) S.list[i]     // amount drawn by the hit at a position, bit 15 = heal

// The sequential loop over the shuffled list, for the steps the parallel resolution cannot decide.  Scalars go
// through SCALW: in [0] k, [1] flags, [2] deaths; out the same plus [3] = bit-mask of the positions whose move succeeded.
ZS_TPL __device__ __noinline__ void execute_sequential(const ZsParams& p, GrpId id, int L) {
    Env e = env_of(p, id);
    ZS_VIEWS;
    if (e.gl == 0) {
        int k = SCALW(0), fl = SCALW(1), deaths = SCALW(2), n_touched = 0;
        unsigned succ = 0;
#pragma unroll 1
        for (int i = 0; i < L; ++i) {
            const unsigned long long pk = ACT(i);
            const uint32_t lo32 = (uint32_t)pk, hi32 = (uint32_t)(pk >> 32);
            const int kind = lo32 & 7;
            if (kind == X_NOP) continue;
            if (kind == X_MOVE) {  // World.thing_move (core.py:140-166)
                const int c = lo32 >> 16;
                if (!g_is_thing(GRID(c))) {
                    const int actor = (lo32 >> 3) & 0xff;
                    GRID(hi32 & 0xffffu) = (lo32 & 0x800u) ? G_DEAD : G_EMPTY;
                    GRID(c) = (uint8_t)(actor + 1);
                    TXY(actor) = BK(actor);
                    MVP(actor) = (uint8_t)i;
                    succ |= 1u << i;
                }
                continue;
            }
            const int dlo = (lo32 >> 18) & 127, dn = (lo32 >> 25) & 63;
            if (kind <= X_HEAL_M) {  // mobile target: distance between CURRENT positions (core.py:176,194)
                const int a = (lo32 >> 3) & 0xff;
                const uint32_t gxy = TXY(a);
                if (dist2(xy_x(hi32), xy_y(hi32), xy_x(gxy), xy_y(gxy)) > (int)((lo32 >> 11) & 127)) continue;
                const int amount = dlo + below(DRAWS(k++), dn);
                if (kind == X_ATTACK_M) TL(a) = (int16_t)(TL(a) - amount);
                else { const int nl = TL(a) + amount; TL(a) = (int16_t)(nl < 100 ? nl : 100); }
            } else {
                const int a = hi32 & 0xffffu;
                const int amount = dlo + below(DRAWS(k++), dn);
                if (kind == X_ATTACK_S) SL(a) = (int16_t)(SL(a) - amount);
                else {
                    const int mx = __ldg(p.static_max + a);
                    const int nl = SL(a) + amount;
                    SL(a) = (int16_t)(nl < mx ? nl : mx);
                }
                LIST(n_touched++) = (uint16_t)a;
                fl |= FL_SL_DIRTY;
            }
        }
        // the boxes/walls hit this step: their patch-list entries, and clean_dead_things (core.py:121-138) for the
        // ones destroyed now (on the first step of a world the clean phase below covers them)
#pragma unroll 1
        for (int i = 0; i < n_touched; ++i) {
            const int si = LIST(i);
            const int cell = __ldg(p.static_cell + si);
            const int life = SL(si);
            const bool fresh = fl & FL_FRESH;
            if (life <= 0 && !fresh && g_is_static(GRID(cell))) { GRID(cell) = G_EMPTY; deaths++; }
            spl_update_one<MPC, G, CV>(p, e, si, cell, life, life > 0 || fresh);
        }
        if (SPN) fl |= FL_DMG;
        SCALW(0) = k; SCALW(1) = fl; SCALW(2) = deaths; SCALW(3) = (int)succ;
    }
    gsync<G, CV>(e);
}

// (at, adx, ady): the action of the agent whose slot this lane is (Agent.set_action, agent.py:22-25).
template <int MPC, int G, bool CV, int ROS = 0>
__device__ __forceinline__ int world_step_one(const ZsParams& p, Env& e, int at, int adx, int ady) {
    ZS_VIEWS;
    static_assert(MPC <= G, "one lane per slot");
    using R = Roster<ROS>;
    const int s = e.gl;  // slot in slot space, list position in position space
    const int P = R::on ? R::P : p.P, NP = R::on ? R::NP : p.P + p.A;
    const unsigned below_s = (1u << s) - 1u;
    e.t += 1;
    const uint32_t t_word = (uint32_t)(e.t + 1);

    // ================= slot space
    const bool in_cap = G == MPC || s < MPC;
    const uint32_t rk = in_cap ? RK(s) : RK_NONE;
    const bool live = rk != RK_NONE;
    const uint32_t xy = live ? TXY(s) : 0u;
    const int x = xy_x(xy), y = xy_y(xy);
    const bool zombie = s >= NP, agent = !zombie && s >= P;
    const int bkind = s < P ? (R::on ? (int)ZS_KIND_TERMINATOR : (int)p.bot_kinds[s]) : -1;
    if (!(live && agent)) at = ZS_ACT_NONE;
    else if (at == ZS_ACT_ABSENT) { at = ZS_ACT_HEAL; adx = 0; ady = 0; }  // multiagent_env.py:129-131
    // what is on the four adjacent cells (utils.py:34-44) does not depend on the target: read it now, so the loads
    // are back by the time the closest things are known.  No bounds check: cells outside the map hold nothing
    // (utils.py:47-52)
    unsigned gs[4];
    unsigned freemask = 0;
    {
        // (0,+1), (0,-1), (+1,0), (-1,0) from ONE cell index: a thing in the world stands inside the map, so a neighbour is
        // outside exactly at the map's edges — four compares instead of a bounds check per neighbour
        // (every lane reads: a lane without a thing in the world stands at (0, 0), inside the map; only the scripted actors use the result)
        const int c0 = y * p.W + x;
        gs[0] = y + 1 < p.H ? (unsigned)GRIDP[c0 + p.W] : (unsigned)G_EMPTY;
        gs[1] = y > 0 ? (unsigned)GRIDP[c0 - p.W] : (unsigned)G_EMPTY;
        gs[2] = x + 1 < p.W ? (unsigned)GRIDP[c0 + 1] : (unsigned)G_EMPTY;
        gs[3] = x > 0 ? (unsigned)GRIDP[c0 - 1] : (unsigned)G_EMPTY;
    }
    const int my_tm = in_cap ? (int)TM(s) : 0;
    bool has_humans = false;  // any player (bot or agent) in the world: every lane sees all of them in the pass below

    // ---- closest(self, others) (utils.py:23-31) for everybody from ONE pass over the (thing, player) distances:
    // a zombie (things.py:73-82) or a heal_closest agent (agent.py:79-86) takes the minimum over the players in its
    // own lane; a player's closest zombie is the minimum of the same distances across the zombie lanes (redux.sync)
    // and lands in the player's lane.  Key = (d^2 << 8) | dict rank: sorted() is stable, ties go to the earlier thing.
    // (bestp is only read by a live zombie or heal_closest agent)
    const uint32_t zkey = (live && zombie) ? rk : 0xffffffffu;
    uint32_t bestp = 0xffffffffu, zb = 0xffffffffu;
    auto one_player = [&](int q) {
        const uint32_t rq = RK(q), qxy = TXY(q);
        const bool hq = rq != RK_NONE;  // player q is in the world
        const uint32_t d = (uint32_t)dist2(x, y, xy_x(qxy), xy_y(qxy)) << 8;
        has_humans |= hq;
        if (hq && q != s) bestp = min(bestp, d | rq);
        const uint32_t m = gminu<G, CV>(e, hq ? (d | zkey) : 0xffffffffu);
        if (q == s) zb = m;
    };
    // (the first four players unrolled: their loads and reductions are independent and overlap)
#pragma unroll
    for (int q = 0; q < 4; ++q) if (q < NP) one_player(q);
#pragma unroll 1
    for (int q = 4; q < NP; ++q) one_player(q);

    PH(1);
    // ---- get_actions (core.py:80-101): every actor decides against the pre-step world
    int type = D_IDLE, a = 0, b = 0;
    if (live) {
        const uint32_t key = (zombie || at == ZS_ACT_HEAL_CLOSEST) ? bestp : zb;
        const int tg = key == 0xffffffffu ? -1 : (int)SOR(key & 255u);
        const int d2 = (int)(key >> 8);
        const uint32_t gxy = tg >= 0 ? TXY(tg) : 0u;
        const int gx = xy_x(gxy), gy = xy_y(gxy);
        if (!agent) {
            // The scripted actors decide with as little divergence as possible: the lanes of a warp are zombies, terminators
            // and others side by side, and every branch one kind takes is issued for the whole warp.
            // the four adjacent cells: how far they are from the target, which are free, which hold a box/wall
            // (with e = target - self, the squared distance from the cell at (0,+1), (0,-1), (+1,0), (-1,0) is |e|^2 + 1 plus
            // -2ey, +2ey, -2ex, +2ex: the order of the four, ties included, is the order of these)
            const int dd[4] = {y - gy, gy - y, x - gx, gx - x};
            unsigned staticmask = 0;
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                if (!g_is_thing(gs[d])) freemask |= 1u << d;
                if (g_is_static(gs[d])) staticmask |= 1u << d;
            }
            const bool term = bkind == ZS_KIND_TERMINATOR;
            // Zombie.next_step (things.py:70-105): a human out of reach (distance >= 1.5) is chased — to the free adjacent
            // cell closest to it (first minimum in adjacency order), or, boxed in, the first Box/Wall among the adjacent
            // cells stably sorted by distance to the target is attacked (things.py:88-99).
            // Terminator.next_step (players/terminator.py:9-37): a zombie out of range is approached through the adjacent
            // cell closest to it, out-of-bounds cells included; what stands there is healed (a player) or attacked.
            const bool z_chase = zombie && has_humans && d2 > 2;
            const bool t_chase = term && tg >= 0 && d2 > c_range2[my_tm & 15];
            const unsigned cand = t_chase ? 0xfu : (freemask ? freemask : staticmask);
            int bdir = -1, bdist = 0x7fffffff;
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (((cand >> d) & 1u) && dd[d] < bdist) { bdir = d; bdist = dd[d]; }
            if ((z_chase || t_chase) && bdir >= 0) {
                const int cx = x + adj_dx(bdir), cy = y + adj_dy(bdir);
                const int g = (int)(bdir == 0 ? gs[0] : bdir == 1 ? gs[1] : bdir == 2 ? gs[2] : gs[3]);
                if (g_is_thing(g)) {
                    type = (g <= G_MAX_SLOT && (g - 1) < NP) ? D_HEAL : D_ATTACK;
                    a = target_of_cell(p, g, cy * p.W + cx);
                } else { type = D_MOVE; a = cx; b = cy; }
            } else {
                // zombie next to its human: attack it (distance < 1.5, things.py:83); no humans: wander (things.py:101-103);
                // terminator: in range attack, no zombies heal self; Sniper (players/sniper.py:9-19): attack the closest
                // zombie; Troll (troll.py:10-12): heal self; Hamster (hamster.py:10-14): wander; RandoMan: decide_draws_seq
                const bool attack_tg = (zombie && has_humans && d2 <= 2) || (term && tg >= 0 && !t_chase) ||
                                       (bkind == ZS_KIND_SNIPER && tg >= 0);
                const bool heal_self = (term && tg < 0) || bkind == ZS_KIND_TROLL;
                const bool wander = freemask != 0u && ((zombie && !has_humans) || bkind == ZS_KIND_HAMSTER);
                type = attack_tg ? D_ATTACK : heal_self ? D_HEAL : wander ? D_WANDER : bkind == ZS_KIND_RANDOMAN ? D_RANDOM : D_IDLE;
                a = attack_tg ? tg : heal_self ? s : 0;
            }
        }
        // Agent.next_step (players/agent.py:28-96), by selects: `at` is ZS_ACT_NONE in every lane that is not a live agent, so
        // the two or so agent lanes of a warp do not cost the others a divergent branch
        // (a step of two cells or more fails whatever its length, core.py:149-153: clamped, so nothing can overflow)
        {
            const bool mv = at == ZS_ACT_MOVE, ac = at == ZS_ACT_ATTACK_CLOSEST && tg >= 0, hc = at == ZS_ACT_HEAL_CLOSEST;
            const bool hs = at == ZS_ACT_HEAL && adx == 0 && ady == 0;
            type = mv ? D_MOVE : ac ? D_ATTACK : (hc || hs) ? D_HEAL : type;
            a = mv ? x + max(-2, min(2, adx)) : (ac || (hc && tg >= 0)) ? tg : (hc || hs) ? s : a;
            b = mv ? y + max(-2, min(2, ady)) : b;
            if (at == ZS_ACT_ATTACK || (at == ZS_ACT_HEAL && !hs)) {  // a target named by its offset: rare
                adx = max(-4096, min(4096, adx)); ady = max(-4096, min(4096, ady));  // (off the map either way)
                const int g = grid_at(p, GRIDP, x + adx, y + ady);
                // attack: any thing; heal: Player / Box / Wall only (agent.py:69-75)
                const bool ok = at == ZS_ACT_ATTACK ? g_is_thing(g)
                                                    : (g_is_static(g) || (g_is_thing(g) && (g - 1) < NP));
                if (ok) { type = at == ZS_ACT_ATTACK ? D_ATTACK : D_HEAL; a = target_of_cell(p, g, (y + ady) * p.W + (x + adx)); }
            }
        }
    }
    PH(2);
    // wandering zombies and hamsters draw random.choice(positions) in dict order (things.py:101-103, hamster.py:12-14)
    int nd = 0;
    if (!R::on && p.has_randoman) {
        if (wany<G, CV>(e, type == D_WANDER || type == D_RANDOM)) {
            if (in_cap) { MPOS(s) = (uint8_t)type; BK(s) = freemask; }  // (MPOS = DTYPE, free until the list is built)
            gsync<G, CV>(e);
            nd = decide_draws_seq<MPC, G, false>(p, id_of(e), e.episode, t_word, e.nlive, e.flags);
            if (type == D_WANDER || type == D_RANDOM) unpack_decision(BK(s), type, a, b);
        }
    } else if (wany<G, CV>(e, type == D_WANDER)) {
        TRF(0);
        const unsigned wm = gor_bits<G, CV>(e, type == D_WANDER ? (1u << rk) : 0u);
        if (type == D_WANDER) {
            int pick = below(draw_at(p, e, t_word, __popc(wm & ((1u << rk) - 1u))), __popc(freemask));
            int d = 0;
            for (int q = 0; q < 4; ++q) if ((freemask >> q) & 1u) { if (pick == 0) { d = q; break; } --pick; }
            type = D_MOVE; a = x + adj_dx(d); b = y + adj_dy(d);
        }
        nd = __popc(wm);
    }
    // actions list in actor (dict) order (core.py:83-90): the position of an acting thing is its dict rank minus
    // the idle things before it.  Everything that cannot change before the actor acts is resolved here.
    int pos = (int)rk;
    if (wany<G, CV>(e, live && type == D_IDLE)) {
        TRF(1);
        const unsigned im = gor_bits<G, CV>(e, (live && type == D_IDLE) ? (1u << rk) : 0u);
        pos -= __popc(im & ((1u << (rk & 31u)) - 1u));
    }
    unsigned long long my_word = X_NOP;
    const bool acting = type != D_IDLE;
    bool is_hit = false;
    if (acting) {
        if (type == D_MOVE) {  // in bounds and at most one step (core.py:149-153); occupancy is checked when it runs
            if ((unsigned)a < (unsigned)p.W && (unsigned)b < (unsigned)p.H && dist2(x, y, a, b) <= 1) {
                const int old = y * p.W + x;
                my_word = pack_move(s, (DEADW(old >> 5) >> (old & 31)) & 1u, b * p.W + a, old);
                BK(s) = xy_pack(a, b);
            }
        } else {
            const bool is_static = a >= p.M;
            int mx = 100, r2, dlo, dn;
            if (type == D_ATTACK) { const int w = my_tm & 15; r2 = c_range2[w]; dlo = c_dmg_lo[w]; dn = c_dmg_n[w]; }
            else {  // heal: randint(MAX_LIFE // 10, MAX_LIFE // 4) of the target's class, range 3 (core.py:194-198)
                if (is_static) mx = __ldg(p.static_max + (a - p.M));
                r2 = 9; dlo = mx / 10; dn = mx / 4 - mx / 10 + 1;
            }
            if (is_static) {
                const int cell = __ldg(p.static_cell + (a - p.M));
                const int gy = cell / p.W, gx = cell - gy * p.W;
                if (dist2(x, y, gx, gy) <= r2) { my_word = pack_hit(type == D_ATTACK ? X_ATTACK_S : X_HEAL_S, 0, 0, dlo, dn, (uint32_t)(a - p.M)); is_hit = true; }
            } else { my_word = pack_hit(type == D_ATTACK ? X_ATTACK_M : X_HEAL_M, a, r2, dlo, dn, xy); is_hit = true; }
        }
    }
    const int L = __popc(gballot<G, CV>(e, acting));
    const int n_ah = __popc(gballot<G, CV>(e, is_hit));
    PH(3);
    // ---- draws of this step, 4 per lane (counter-based: any k is available directly)
    const int n_need = nd + (L > 1 ? L - 1 : 0) + n_ah;
    if (s * 4 < n_need)
        reinterpret_cast<uint4*>(S.draws)[s] = philox_draws(p, e.env_global, (uint32_t)e.episode, t_word, (uint32_t)s);
    gsync<G, CV>(e);
    // ---- random.shuffle (core.py:76): for i = L-1 .. 1: j = randbelow(i + 1); swap.  The swaps are a fixed sequence
    // once the partners are known: every lane follows its own action through them in registers.
    PH(4);
    // The partners go through shared memory as bytes and come back as broadcast 128-bit loads, so the swap loop is
    // pure register arithmetic with compile-time indices (iterations at or beyond L change nothing).
    if (in_cap) S.fyj[s] = (uint8_t)((s >= 1 && s < L) ? below(DRAWS(nd + (L - 1 - s)), s + 1) : s);
    gsync<G, CV>(e);
    int my_pos = acting ? pos : -1;
    {
        uint32_t jw[MPC / 4];
#pragma unroll
        for (int q = 0; q < MPC / 16; ++q) {
            const uint4 v = reinterpret_cast<const uint4*>(S.fyj)[q];
            jw[4 * q] = v.x; jw[4 * q + 1] = v.y; jw[4 * q + 2] = v.z; jw[4 * q + 3] = v.w;
        }
        // iterations at or beyond the list's length swap nothing: enter the unrolled sequence at the longest list of the
        // warp (one indexed branch; the cases fall through down to iteration 1)
#define ZS_FY(i)                                                                        \
    case (i) + 1:                                                                       \
        if constexpr ((i) < MPC) {                                                      \
            const int j = (int)((jw[(i) >> 2] >> (8 * ((i) & 3))) & 0xffu);             \
            my_pos = my_pos == (i) ? j : (my_pos == j ? (i) : my_pos);                  \
        }
        const int Lw = wmax<G, CV>(e, L);
        switch (Lw < MPC ? Lw : MPC) {
            ZS_FY(31) ZS_FY(30) ZS_FY(29) ZS_FY(28) ZS_FY(27) ZS_FY(26) ZS_FY(25) ZS_FY(24)
            ZS_FY(23) ZS_FY(22) ZS_FY(21) ZS_FY(20) ZS_FY(19) ZS_FY(18) ZS_FY(17) ZS_FY(16)
            ZS_FY(15) ZS_FY(14) ZS_FY(13) ZS_FY(12) ZS_FY(11) ZS_FY(10) ZS_FY(9) ZS_FY(8)
            ZS_FY(7) ZS_FY(6) ZS_FY(5) ZS_FY(4) ZS_FY(3) ZS_FY(2) ZS_FY(1)
            default: break;
        }
#undef ZS_FY
    }
    if (my_pos >= 0) ACT(my_pos) = my_word;
    if (in_cap) { MPOS(s) = (uint8_t)(((uint32_t)my_word & 7u) == X_MOVE ? my_pos : RK_NONE); MVP(s) = RK_NONE; }
    gsync<G, CV>(e);

    PH(5);
    // ================= position space: execute_actions (core.py:103-119)
    int k = nd + (L > 1 ? L - 1 : 0);
    unsigned succ_m = 0;
    {
        const unsigned long long pk = s < L ? ACT(s) : 0ull;
        const uint32_t lo32 = (uint32_t)pk, hi32 = (uint32_t)(pk >> 32);
        int kind = lo32 & 7;
        const int who = (lo32 >> 3) & 0xff;  // the actor of a move, the mobile target of a hit
        const int c = lo32 >> 16;
        const int g0 = kind == X_MOVE ? (int)GRID(c) : G_STATIC;
        bool need_seq = false;
        if (kind == X_MOVE && g0 >= 1 && g0 <= G_MAX_SLOT) need_seq = MPOS(g0 - 1) < s;
        // an env that needs the sequential loop sits out the parallel resolution (all its actions read as no-ops)
        const bool seq = gany<G, CV>(e, need_seq);
        if (seq) kind = X_NOP;
        // ---- moves (World.thing_move, core.py:140-166)
        const bool dest_free = kind == X_MOVE && !g_is_thing(g0);
        // (match.any takes time per DISTINCT value: everybody who does not take part shares one dummy)
        const unsigned want = gmatch<G, CV>(e, dest_free ? (uint32_t)c : 0x10000u);
        const bool success = dest_free && !(want & below_s);
        succ_m = gballot<G, CV>(e, success);
        if (success) {
            GRID(hi32 & 0xffffu) = (lo32 & 0x800u) ? G_DEAD : G_EMPTY;
            GRID(c) = (uint8_t)(who + 1);
            MVP(who) = (uint8_t)s;  // things[dest] = thing; del things[old]: goes last in the dict
        }
        gsync<G, CV>(e);
        PH(6);
        // ---- hits (World.thing_attack / thing_heal, core.py:168-208)
        const bool on_static = kind >= X_ATTACK_S;
        bool inrange = on_static;  // boxes/walls do not move: their range was checked when the word was built
        if (kind == X_ATTACK_M || kind == X_HEAL_M) {  // distance between CURRENT positions (core.py:176,194)
            uint32_t txy = TXY(who);
            if (MVP(who) < s) txy = BK(who);
            inrange = dist2(xy_x(hi32), xy_y(hi32), xy_x(txy), xy_y(txy)) <= (int)((lo32 >> 11) & 127);
        }
        if (wany<G, CV>(e, inrange)) {
            TRF(2);
            const unsigned hit_m = gballot<G, CV>(e, inrange);
            const int si = hi32 & 0xffffu;
            const bool heal = kind == X_HEAL_M || kind == X_HEAL_S;
            if (inrange) {
                const int amount = (int)((lo32 >> 18) & 127) + below(DRAWS(k + __popc(hit_m & below_s)), (int)((lo32 >> 25) & 63));
                AMT(s) = (uint16_t)(amount | (heal ? 0x8000 : 0));
            }
            k += __popc(hit_m);
            const uint32_t tid = on_static ? 0x100u + (uint32_t)si : (uint32_t)who;
            const unsigned grp = gmatch<G, CV>(e, inrange ? tid : 0x20000u);
            const bool lead = inrange && !(grp & below_s);  // the first hit on a target applies all of them, in order
            gsync<G, CV>(e);
            int life = 0;
            if (lead) {
                life = on_static ? (int)SL(si) : (int)TL(who);
                const int mx = on_static ? (int)__ldg(p.static_max + si) : 100;
                unsigned bits = grp;
                while (bits) {
                    const int v = AMT(__ffs(bits) - 1);
                    bits &= bits - 1;
                    if (v & 0x8000) { life += v & 0x7fff; life = life < mx ? life : mx; }
                    else life -= v;
                }
                if (on_static) SL(si) = (int16_t)life; else TL(who) = (int16_t)life;
            }
            const bool slead = lead && on_static;
            if (wany<G, CV>(e, slead)) {
                TRF(3);
                // a box/wall changed: clean_dead_things (core.py:121-138) for the ones destroyed now (on the first step of
                // a world the clean phase covers them), and their entries in the static patch list
                bool is_new = false, gone = false;
                int cell = 0, pay = 0, idx = 0;
                if (slead) {
                    const int mx = __ldg(p.static_max + si);
                    const bool fresh = e.flags & FL_FRESH;
                    cell = __ldg(p.static_cell + si);
                    gone = life <= 0 && !fresh && g_is_static(GRID(cell));
                    if (gone) GRID(cell) = G_EMPTY;
                    pay = static_payload(p, mx, life, life > 0 || fresh);
                    idx = SIDX(si);
                    is_new = idx == 0 && pay != static_payload(p, mx, mx, true);
                }
                e.deaths += __popc(gballot<G, CV>(e, gone));
                if (gany<G, CV>(e, slead)) e.flags |= FL_SL_DIRTY;
                const unsigned new_m = gballot<G, CV>(e, is_new);
                const int n0 = SPN;
                gsync<G, CV>(e);  // (everybody has read the count before lane 0 rewrites it)
                if (is_new) { idx = n0 + __popc(new_m & below_s) + 1; SIDX(si) = (uint8_t)(idx < SIDX_FAR ? idx : SIDX_FAR); }
                else if (idx == SIDX_FAR) idx = spl_find_far<MPC, G, CV>(p, e, cell);
                if (slead && idx) SPL(idx - 1) = spl_entry(cell, pay);
                if (new_m) {
                    if (s == 0) SPN = (uint16_t)(n0 + __popc(new_m));
                    e.flags |= FL_DMG;
                }
            }
        }
        gsync<G, CV>(e);
        if (wany<G, CV>(e, seq)) TRF(4);
        if (seq) {  // rare, and possibly only one env of the warp: the divergent flavour from here
            if (s == 0) { SCALW(0) = k; SCALW(1) = e.flags; SCALW(2) = e.deaths; }
            gsync<G, false>(e);
            execute_sequential<MPC, G, false>(p, id_of(e), L);
            k = SCALW(0); e.flags = SCALW(1); e.deaths = SCALW(2); succ_m = (unsigned)SCALW(3);
        }
    }

    PH(7);
    // ================= slot space: clean_dead_things (core.py:121-138)
    int nd_all = 0;
    const bool fresh_scan = (e.flags & FL_FRESH) && (e.flags & FL_DMG);
    if (e.flags & FL_FRESH) {  // first step of this world: every box/wall with life <= 0 leaves now
        TRF(7);
        if (e.flags & FL_DMG) nd_all = spl_clean_fresh<MPC, G, CV>(p, e);
        e.flags &= ~FL_FRESH;
    }
    // deaths, dead bodies and the new dict order in one pass.  Survivors that did not move keep their relative
    // order, the movers follow in move order (re-inserted at the end, core.py:158-159).
    const int mvp = in_cap ? (int)MVP(s) : RK_NONE;
    const bool moved = mvp != RK_NONE;
    uint32_t nxy = xy;
    if (moved) { nxy = BK(s); TXY(s) = nxy; }
    const bool dead = live && TL(s) <= 0;
    if (dead) {
        const int c = xy_y(nxy) * p.W + xy_x(nxy);
        GRID(c) = G_DEAD;                         // DeadBody overwrites any decoration (core.py:30-31,126-128)
        atomicOr(&DEADW(c >> 5), 1u << (c & 31));
        TM(s) &= 0x7f;
    }
    const unsigned dead_m = gballot<G, CV>(e, dead);
    if (wany<G, CV>(e, dead)) {  // remember the cells for the observation patches (the bitmap stays the state)
        TRF(5);
        const int n0 = DBL(0), idx = n0 + __popc(dead_m & below_s), tot = n0 + __popc(dead_m);
        gsync<G, CV>(e);  // (everybody has read the count before lane 0 rewrites it)
        if (dead && idx < ZS_DEAD_CAP) DBL(1 + idx) = (uint16_t)(xy_y(nxy) * p.W + xy_x(nxy));
        if (dead_m) {
            if (tot > ZS_DEAD_CAP) e.flags |= FL_DEAD_OVER;
            if (s == 0) DBL(0) = (uint16_t)(tot < ZS_DEAD_CAP ? tot : ZS_DEAD_CAP);
        }
    }
    e.deaths += __popc(dead_m);
    if (wany<G, CV>(e, fresh_scan)) e.deaths += gadd<G, CV>(e, nd_all);  // (nd_all is 0 for an env that did not scan)
    e.zd += __popc(dead_m >> NP);
    if (wany<G, CV>(e, succ_m || dead_m)) {  // (an env without changes gets its old ranks back)
        TRF(6);
        const bool alive = live && !dead;
        const unsigned stay_m = gor_bits<G, CV>(e, (alive && !moved) ? (1u << rk) : 0u);
        const unsigned move_m = gor_bits<G, CV>(e, (alive && moved) ? (1u << mvp) : 0u);
        if (live) {
            int nr = RK_NONE;
            if (alive) {
                nr = !moved ? __popc(stay_m & ((1u << rk) - 1u)) : __popc(stay_m) + __popc(move_m & ((1u << mvp) - 1u));
                SOR(nr) = (uint8_t)s;
            }
            RK(s) = (uint8_t)nr;
        }
        e.nlive = __popc(stay_m) + __popc(move_m);
    }
    gsync<G, CV>(e);
    PH(8);
    return k;
}

// Draws k0 .. k0 + count - 1 of the env's stream, staged in shared memory (the per-step draw array): consecutive draw
// indices share Philox blocks of four, so ONE evaluation per lane yields up to 4 * G draws.  Returns how many of the
// `count` it staged (what the staging area holds); draw k is then at STAGE[k - 4 * (k0 >> 2)].
ZS_TPL __device__ __forceinline__ int stage_draws(const ZsParams& p, const Env& e, uint32_t t_word, int k0, int count) {
    ZS_VIEWS;
    constexpr int NB = EnvS<MPC>::NDRAWS / 4 < G ? EnvS<MPC>::NDRAWS / 4 : G;  // blocks the array holds / lanes there are
    const int off = k0 & 3;
    const int chunk = min(count, 4 * NB - off);
    gsync<G, CV>(e);  // (whatever used the array before has been read)
    if (e.gl < NB && e.gl * 4 < off + chunk)
        reinterpret_cast<uint4*>(S.draws)[e.gl] = philox4x32_10(e.env_global, (uint32_t)e.episode, t_word, (uint32_t)((k0 >> 2) + e.gl), p.key0, p.key1);
    gsync<G, CV>(e);
    return chunk;
}

// ---------------------------------------------------------------- World.spawn_in_random (core.py:40-66)
// Places the `count` slots listed in LIST[0..count) on shuffled free cells of the player (which = 0) or
// zombie (which = 1) spawn cells, or of the whole map, x-major, when the map has no such spawn cells.  Only
// the first `count` Fisher-Yates iterations decide placements (spawns.pop() takes from the end); the rest of
// the shuffle only advances the draw counter.  New things are appended to the dict order (rank0 + i).
// all_free: the caller knows that nothing stands on any cell of the spawn list (a new world: spawn cells never
// carry boxes/walls, and player and zombie spawn cells are different cells — as long as the players stood on player spawn
// cells), so the list is taken as it is.
// Returns the new draw index; the new number of things in the world is left in SCALW(ZS_S_STAMP_COUNTER).
ZS_TPL __device__ __noinline__ int spawn_in_random(const ZsParams& p, GrpId id, int episode,
                                                   uint32_t t_word, int k, int count, int which, int rank0, bool all_free,
                                                   bool new_world) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    const int lane = e.gl;
    e.episode = episode;
    const uint16_t* spawn = which ? p.zs_cells : p.ps_cells;
    const int n_spawn = which ? p.n_zs : p.n_ps;
    const int n_src = n_spawn > 0 ? n_spawn : p.cells;
    int n = 0;
    // A group without spawn cells of its own may stand on any cell that holds no thing, taken in x-major order
    // (core.py:44-52).  In a NEW world those are the cells without a box/wall — a constant of the map, tabulated once
    // (free_xm) — minus the cells of the things placed so far, which all stand on such cells: the candidate list is not
    // materialised at all.  Candidate i is entry x of the table, x the smallest index with x - #{taken <= x} == i; the
    // taken entries (TAKEN, at most the players) are noted as the groups are placed.
    uint16_t* const TAKEN = reinterpret_cast<uint16_t*>(S.bk);
    const bool virt = new_world && n_spawn == 0 && p.free_xm != nullptr && rank0 <= ZS_NP_MAX && rank0 <= 2 * MPC;
    if (all_free && n_spawn > 0) {
#pragma unroll 4
        for (int i = lane; i < n_spawn; i += G) CAND(i) = __ldg(spawn + i);
        n = n_spawn;
    } else if (virt) {
        n = p.n_free0 - rank0;
    } else {
#pragma unroll 1
        for (int b0 = 0; b0 < n_src; b0 += G) {
            const int i = b0 + lane;
            bool ok = false;
            int c = 0;
            if (i < n_src) {
                if (n_spawn > 0) c = __ldg(spawn + i);
                else { const int x = i / p.H; const int y = i - x * p.H; c = y * p.W + x; }
                ok = !g_is_thing(GRID(c));
            }
            const unsigned m = gballot<G, CV>(e, ok);
            if (ok) CAND(n + __popc(m & ((1u << e.gl) - 1u))) = (uint16_t)c;
            n += __popc(m);
        }
    }
    gsync<G, CV>(e);
    const int placed = count < n ? count : n;
    // random.shuffle + spawns.pop() (core.py:54-61): only the first `placed` Fisher-Yates iterations decide anything, and
    // they touch at most 2 * placed positions of the list.  Iteration `it` swaps positions i = n - 1 - it and j = draw:
    // it takes what is at j and leaves there what was at i.  What an iteration finds at a position is what the LAST
    // earlier iteration with that j left there, else the list's own entry.  All of it is resolved in parallel:
    //   * the draws: consecutive draw indices share Philox blocks of four, so one evaluation per lane yields the draws of
    //     128 iterations (staged through shared memory);
    //   * PI[it], the last earlier iteration that wrote position i_it: only an iteration q with j_q >= n - placed can
    //     have hit one of the i's, and it names the iteration it hits (n - 1 - j_q) itself — an atomic max, no search;
    //   * PJ[it], the last earlier iteration with the same j: equal draws are rare, so a hashed bitmap of the j's says
    //     which iterations have a partner at all and only those search (short groups: one match.any);
    //   * what iteration q left at j_q is the list entry at the root of q's PI chain, so every lane follows its own.
    uint16_t* const Bi = reinterpret_cast<uint16_t*>(S.act);  // [MPC] list entry at i
    uint16_t* const Bj = Bi + MPC;                            // [MPC] list entry at j
    uint16_t* const Jp = Bj + MPC;                            // [MPC] j
    uint16_t* const Ch = Jp + MPC;                            // [MPC] the cell the it-th thing gets
    int32_t* const PI = reinterpret_cast<int32_t*>(S.draws);  // [MPC] see above, or -1
    int16_t* const PJ = reinterpret_cast<int16_t*>(PI + MPC); // [MPC] see above, or -1
    uint32_t* const STAGE = reinterpret_cast<uint32_t*>(S.draws);  // [4 * G] draws of one chunk (before PI / PJ are written)
    auto cand_at = [&](int i) -> uint16_t {
        if (!virt) return CAND(i);
        int x = i;
#pragma unroll 1
        for (;;) {
            int c = 0;
#pragma unroll 1
            for (int t = 0; t < rank0; ++t) c += (int)TAKEN[t] <= x;
            if (i + c == x) break;
            x = i + c;
        }
        return __ldg(p.free_xm + x);
    };
#pragma unroll 1
    for (int it0 = 0; it0 < placed;) {  // a chunk of draws k + it0 ..: as many blocks of four as the staging area holds
        const int chunk = stage_draws<MPC, G, CV>(p, e, t_word, k + it0, placed - it0);
        const int kb = (k + it0) >> 2;
#pragma unroll 1
        for (int it = it0 + lane; it < it0 + chunk; it += G) {
            const int i = n - 1 - it;
            const int j = i >= 1 ? below(STAGE[(k + it) - 4 * kb], i + 1) : i;
            Jp[it] = (uint16_t)j; Bi[it] = cand_at(i); Bj[it] = cand_at(j);
        }
        gsync<G, CV>(e);
        it0 += chunk;
    }
#pragma unroll 1
    for (int it = lane; it < placed; it += G) { PI[it] = -1; PJ[it] = -1; }
    gsync<G, CV>(e);
#pragma unroll 1
    for (int q = lane; q < placed; q += G) {  // the iterations whose partner position is one of the i's
        const int hit = n - 1 - (int)Jp[q];
        if (hit > q && hit < placed) atomicMax(&PI[hit], q);
    }
    if (placed <= G) {  // one round: equal draws by match.any, the partner is the nearest lower lane
        const bool on = lane < placed;
        const unsigned grp = gmatch<G, CV>(e, on ? (uint32_t)Jp[on ? lane : 0] : 0x80000u + (uint32_t)lane) & ((1u << lane) - 1u);
        if (on && grp) PJ[lane] = (int16_t)(31 - __clz(grp));
    } else if constexpr (MPC > 32) {
        // hashed bitmaps over the j's, in the decide phase's per-slot arrays DA and DB (free here): 16 bits per slot each
        uint32_t* const SEEN = reinterpret_cast<uint32_t*>(S.da);  // [HB / 32]
        constexpr int HB = 16 * EnvS<MPC>::GEN;
        static_assert((HB & (HB - 1)) == 0 && offsetof(EnvS<MPC>, db) == offsetof(EnvS<MPC>, da) + sizeof(int16_t) * EnvS<MPC>::GEN, "DA and DB are adjacent");
        uint32_t* const DUP = SEEN + HB / 32;
#pragma unroll 1
        for (int w = lane; w < 2 * (HB / 32); w += G) SEEN[w] = 0u;
        gsync<G, CV>(e);
#pragma unroll 1
        for (int it = lane; it < placed; it += G) {
            const uint32_t hsh = ((uint32_t)Jp[it] * 0x9E3779B1u) >> 16 & (uint32_t)(HB - 1);
            const uint32_t old = atomicOr(&SEEN[hsh >> 5], 1u << (hsh & 31));
            if ((old >> (hsh & 31)) & 1u) atomicOr(&DUP[hsh >> 5], 1u << (hsh & 31));
        }
        gsync<G, CV>(e);
#pragma unroll 1
        for (int it = lane; it < placed; it += G) {
            const int j = Jp[it];
            const uint32_t hsh = ((uint32_t)j * 0x9E3779B1u) >> 16 & (uint32_t)(HB - 1);
            if (!((DUP[hsh >> 5] >> (hsh & 31)) & 1u)) continue;
            int pj = -1;
#pragma unroll 1
            for (int q = 0; q < it; ++q) if ((int)Jp[q] == j) pj = q;
            PJ[it] = (int16_t)pj;
        }
    }
    gsync<G, CV>(e);
    auto left_by = [&](int q) -> int {  // what iteration q left at its position j: the list entry at the root of its PI chain
        int r = q;
#pragma unroll 1
        while (PI[r] >= 0) r = PI[r];
        return (int)Bi[r];
    };
#pragma unroll 1
    for (int it = lane; it < placed; it += G) {
        const int pj = PJ[it];
        int vj;
        if ((int)Jp[it] == n - 1 - it) vj = left_by(it);   // (a swap with itself: what is at i)
        else vj = pj >= 0 ? left_by(pj) : (int)Bj[it];
        Ch[it] = (uint16_t)vj;  // position i (never read again) holds what was at j: the it-th thing's cell
    }
    if (lane == 0) SCALW(ZS_S_STAMP_COUNTER) = rank0 + placed;
    gsync<G, CV>(e);
#pragma unroll 1
    for (int it = e.gl; it < placed; it += G) {  // spawns.pop() for the it-th thing: place it, append it to the dict order
        const int c = (int)Ch[it];
        const int s = LIST(it);
        const int y = c / p.W;
        TXY(s) = xy_pack(c - y * p.W, y);
        TM(s) |= 0x80;
        RK(s) = (uint8_t)(rank0 + it);
        SOR(rank0 + it) = (uint8_t)s;
        MVQ(s) = RK_NONE;
        GRID(c) = (uint8_t)(s + 1);
        // (a later group of this world init may take its candidates from the table: see TAKEN above)
        if (new_world && p.free_index != nullptr && which == 0 && rank0 + it < ZS_NP_MAX && rank0 + it < 2 * MPC)
            TAKEN[rank0 + it] = __ldg(p.free_index + c);
    }
    gsync<G, CV>(e);
    return k + (n > 1 ? n - 1 : 0);
}

// Game.spawn_zombies (game.py:189-194): `count` Zombie() constructions (life draws, things.py:62)
// followed by spawn_in_random on the zombie spawn cells; free zombie slots are taken in ascending order.
ZS_TPL __device__ __noinline__ int spawn_zombies(const ZsParams& p, GrpId id, int episode,
                                                 uint32_t t_word, int k, int count, int rank0, bool all_free, bool new_world) {
    ZS_CONSTS;
    Env e = env_of(p, id);
    ZS_VIEWS;
    const int lane = e.gl;
    e.episode = episode;
    const int NP = p.P + p.A;
    int n = 0;
#pragma unroll 1
    for (int b0 = NP; b0 < p.M; b0 += G) {
        const int s = b0 + lane;
        const bool free_slot = s < p.M && !(TM(s) & 0x80);
        const unsigned m = gballot<G, CV>(e, free_slot);
        const int pos = n + __popc(m & ((1u << e.gl) - 1u));
        if (free_slot && pos < count) LIST(pos) = (uint16_t)s;
        n += __popc(m);
    }
    const int made = count < n ? count : n;
    gsync<G, CV>(e);
#pragma unroll 1
    for (int i0 = 0; i0 < made;) {  // Zombie.__init__: life = randint(50, 100) (things.py:62), one draw each
        const int chunk = stage_draws<MPC, G, CV>(p, e, t_word, k + i0, made - i0);
        const int kb = (k + i0) >> 2;
#pragma unroll 1
        for (int i = i0 + e.gl; i < i0 + chunk; i += G) {
            const int s = LIST(i);
            TL(s) = (int16_t)(50 + below(S.draws[(k + i) - 4 * kb], 51));
            TM(s) = ZS_WEAPON_CLAWS;
        }
        i0 += chunk;
    }
    gsync<G, CV>(e);
    return spawn_in_random<MPC, G, false>(p, id, episode, t_word, k + count, made, 1, rank0, all_free, new_world);
}

// Game.__initialize_world__ for the common shape (p.fast_init, decided in zs_create): one lane per slot, a map with
// player AND zombie spawn cells and room for everybody, fixed weapons.  Nothing can stand on a spawn cell of a new
// world (boxes/walls never do, and the two kinds of spawn cells are different cells), so World.spawn_in_random's
// filter (core.py:47-52) keeps the whole list for the bots and the zombies, and the list minus the bots' cells for
// the agents; every draw index is known up front.  Lane = slot = dict rank of the new thing, and everything stays in
// registers:
//   * each lane evaluates Philox for its own placement draw (and its life draw: zombies, things.py:62);
//   * random.shuffle + spawns.pop() (core.py:54-61): iteration `it` of a group takes the candidate at position
//     j_it = randbelow(n - it) and leaves the one from position n - 1 - it there.  What iteration `it` finds at j_it is
//     read off the earlier iterations' partners with shuffles: walking t = it-1 .. 0, a t with j_t == q means the
//     content of q came from position n - 1 - t at iteration t, so the search goes on for that position (one
//     descending pass, the three groups at once);
//   * the agents' candidates are the player spawn cells the bots did not take, in list order: the f-th of them is the
//     smallest x with x - #{bot picks <= x} == f.
// Runs CONVERGED (CV): both envs of a warp go through it when either ends an episode, the writes predicated on
// `need`.  Same results as the general initialize_world below.  Returns the draws consumed; the scalars of the new
// world go straight into e.
// Under a roster (ROS) the group sizes but the zombies' are constants: the trace-back runs for a constant count and the
// agents' candidates come from the bots' picks broadcast once, with the fixpoint in registers.
template <int MPC, int G, bool CV, int ROS = 0>
__device__ __forceinline__ int initialize_world_fast(const ZsParams& p, Env& e, bool need) {
    ZS_VIEWS;
    using R = Roster<ROS>;
    const int s = e.gl;
    const int P = R::on ? R::P : p.P, A = R::on ? 1 : p.A, NP = P + A, Z0 = p.initial_zombies;
    const uint32_t episode = (uint32_t)(e.episode + 1);
    // draw indices (A.7 of SURVEY.md): players shuffle, agents shuffle, zombie lives, zombies shuffle; a shuffle of n
    // candidates consumes n - 1 draws whatever is placed
    const int n1 = p.n_ps, n2 = p.n_ps - P, n3 = p.n_zs;
    const int K1 = n1 > 1 ? n1 - 1 : 0, K2 = K1 + (n2 > 1 ? n2 - 1 : 0), K3 = K2 + Z0, K4 = K3 + (n3 > 1 ? n3 - 1 : 0);
    TR(20);
    const bool in_cap = G == MPC || s < MPC;
    const bool is_bot = s < P, is_agent = !is_bot && s < NP, placed = s < NP + Z0;
    const int base = is_bot ? 0 : is_agent ? P : NP;
    const int it = placed ? s - base : 0;
    const int n = is_bot ? n1 : is_agent ? n2 : n3;
    const int kp = (is_bot ? 0 : is_agent ? K1 : K3) + it;  // this thing's placement draw: randbelow(n - it)
    const int kl = K2 + it;                                  // a zombie's life draw
    const uint4 o1 = philox_draws(p, e.env_global, episode, 0u, (uint32_t)(kp >> 2));
    const uint4 o2 = philox_draws(p, e.env_global, episode, 0u, (uint32_t)(kl >> 2));
    const int j = n - it > 1 ? below(word_of(o1, kp & 3), n - it) : 0;
    const int life = s < NP ? 100 : 50 + below(word_of(o2, kl & 3), 51);
    int q = placed ? j : -1;
    const int tmax = max(max(P, A), Z0);
    if constexpr (R::on) {
        // a group of n things needs iterations t < n - 1 only (t < it): the bots have P, the zombies at most MPC - NP
        constexpr int TB = R::P > MPC - R::NP ? R::P : MPC - R::NP;
#pragma unroll
        for (int t = TB - 2; t >= 0; --t) {
            const int jt = gbcast<G, CV>(e, j, (base + t) & (G - 1));
            if (t < it && jt == q) q = n - 1 - t;
        }
    } else if constexpr (MPC <= 16 && CV) {
        // (the step loop's converged call, which is latency-bound: unrolled, the shuffles do not depend on one another and go
        // out back to back, only the compare-select chain is serial.  The reset kernel, which is throughput-bound and runs the
        // member-mask flavour, is 8 % faster with the loop)
#pragma unroll
        for (int t = MPC - 1; t >= 0; --t) {
            if (t < tmax) {
                const int jt = gbcast<G, CV>(e, j, (base + t) & (G - 1));
                if (t < it && jt == q) q = n - 1 - t;
            }
        }
    } else {
#pragma unroll 1
        for (int t = tmax - 1; t >= 0; --t) {
            const int jt = gbcast<G, CV>(e, j, base + t);
            if (t < it && jt == q) q = n - 1 - t;
        }
    }
    if constexpr (R::on) {
        if constexpr (R::P > 0) {
            int qb[R::P > 0 ? R::P : 1];
#pragma unroll
            for (int b = 0; b < R::P; ++b) qb[b] = gbcast<G, CV>(e, q, b);
            int x = q;
#pragma unroll
            for (int r = 0; r < R::P; ++r) {
                int c = 0;
#pragma unroll
                for (int b = 0; b < R::P; ++b) c += qb[b] <= x;
                x = q + c;
            }
            if (is_agent) q = x;
        }
    } else if (P > 0) {  // (an agent's q counts the player spawn cells the bots left)
        int x = q;
#pragma unroll 1
        for (int r = 0; r < P; ++r) {
            int c = 0;
#pragma unroll 1
            for (int b = 0; b < P; ++b) c += gbcast<G, CV>(e, q, b) <= x;
            x = q + c;
        }
        if (is_agent) q = x;
    }
    // (one gather from the map's spawn lists, L1-resident; the copy in the kernel parameters costs a constant-cache access per
    // distinct index: a dozen in a row here)
    const int c = placed ? (int)__ldg((s < NP ? p.ps_cells : p.zs_cells) + q) : 0;
    const int flags_in = e.flags;
    TR(21);
    // The grid of a new world is the pristine template: every box/wall is back, nothing else is on it.  It is reached from
    // the old world's grid by taking off what the lists name — the things in the world, the dead bodies — and putting
    // back the boxes/walls that were gone; all of it in shared memory (the template copy was a trip to the L2).
    const bool by_lists = !(flags_in & FL_DEAD_OVER);
    if (need) {
        if (by_lists) {
            if (in_cap && (TM(s) & 0x80)) { const uint32_t oxy = TXY(s); GRID(xy_y(oxy) * p.W + xy_x(oxy)) = G_EMPTY; }
            const int nb = DBL(0);
#pragma unroll 1
            for (int i = s; i < nb; i += G) { const int dc = DBL(1 + i); GRID(dc) = G_EMPTY; DEADW(dc >> 5) = 0u; }
        } else {  // the dead-body list is not complete: the template, and the whole bitmap
            const uint4* tg = (const uint4*)p.tmpl_grid;
#pragma unroll 6
            for (int i = s; i < (p.cells_pad >> 4); i += G) reinterpret_cast<uint4*>(GRIDP)[i] = __ldg(tg + i);
#pragma unroll 1
            for (int w = s; w < p.dead_words; w += G) DEADW(w) = 0;
        }
    }
    gsync<G, CV>(e);
    if (need) {
        if (s == 0) DBL(0) = 0;
        if (flags_in & FL_DMG) spl_refresh_present<MPC, G, CV>(p, e, by_lists);
    }
    gsync<G, CV>(e);
    TR(22);
    if (need && in_cap) {
        int w = ZS_WEAPON_CLAWS;
        if (is_bot) w = !R::on && p.bot_kinds[s] == ZS_KIND_SNIPER ? ZS_WEAPON_RIFLE : ZS_WEAPON_SHOTGUN;  // sniper.py:23-24, terminator.py:41-42
        else if (is_agent) w = p.agent_weapons[R::on ? 0 : s - P];
        TM(s) = (uint8_t)(placed ? (w | 0x80) : w);
        RK(s) = placed ? (uint8_t)s : (uint8_t)RK_NONE;
        MVQ(s) = RK_NONE;
        if (placed) {  // spawns.pop() for every thing: thing s of the new world gets dict rank s
            const int y = c / p.W;
            TXY(s) = xy_pack(c - y * p.W, y);
            TL(s) = (int16_t)life;
            SOR(s) = (uint8_t)s;
            GRID(c) = (uint8_t)(s + 1);
            if (is_agent) PREVL(s - P) = 100;  // reward_tracker.reset (reward.py:26-28)
        }
    }
    if (need) {
        e.t = -1; e.episode = (int)episode; e.deaths = 0; e.zd = 0; e.nlive = NP + Z0; e.prev_zd = 0; e.ep_steps = 0;
        e.flags = (flags_in & (FL_DMG | FL_SL_DIRTY)) | FL_FRESH | ((flags_in & FL_DEAD_LAUNCH) ? (FL_DEAD_OVER | FL_DEAD_LAUNCH) : 0);
    }
    gsync<G, CV>(e);
    TR(23);
    return K4;
}

// Game.__initialize_world__ (game.py:151-169) + reward_tracker.reset (reward.py:26-28).  Out of line and
// with its own binding of the env's shared memory, so the hot loop's registers stay registers: the new
// scalars are left in SCALW (read back with scalars_from_smem).  `flags_in`: the launch-lifetime static
// damage flags survive a world init (the damage itself does, game.py:154-155).  Returns the draws consumed.
ZS_TPL __device__ __noinline__ int initialize_world(const ZsParams& p, GrpId id, int episode, int flags_in) {
    ZS_CONSTS;
    if constexpr (ONE) {
        if (p.fast_init) {
            Env e = env_of(p, id);
            ZS_VIEWS;
            e.episode = episode - 1; e.flags = flags_in;
            const int k = initialize_world_fast<MPC, G, CV>(p, e, true);
            if (e.gl < 8) SCALW(e.gl) = scalar_of_lane(e);
            gsync<G, CV>(e);
            return k;
        }
    }
    Env e = env_of(p, id);
    ZS_VIEWS;
    const int lane = e.gl;
    const int NP = p.P + p.A;
    const int flags = (flags_in & (FL_DMG | FL_SL_DIRTY)) | FL_FRESH | ((ONE && !(flags_in & FL_DEAD_LAUNCH)) ? 0 : (FL_DEAD_OVER | (flags_in & FL_DEAD_LAUNCH)));
    e.episode = episode;
#ifdef ZS_PHASE_CLOCKS
    e.ph_last = clock64();
#endif
#pragma unroll 1
    for (int w = e.gl; w < p.dead_words; w += G) DEADW(w) = 0;
    if (lane == 0) DBL(0) = 0;  // a new world has no dead bodies
    int k = 0;
#pragma unroll 1
    for (int s = e.gl; s < p.Mp; s += G) {
        int w = 0;
        if (s < p.P) w = p.bot_kinds[s] == ZS_KIND_SNIPER ? ZS_WEAPON_RIFLE : ZS_WEAPON_SHOTGUN;  // sniper.py:23-24, terminator.py:41-42
        else if (s < NP) w = p.agent_weapons[s - p.P];
        else w = ZS_WEAPON_CLAWS;
        TM(s) = (uint8_t)(w == ZS_WEAPON_RANDOM ? 15 : w);
        RK(s) = RK_NONE; MVQ(s) = RK_NONE;
        if (s < NP) TL(s) = 100;
    }
    gsync<G, CV>(e);
    // trolls, hamsters and randomans are created without a weapon: Player.__init__ draws random.choice([Gun, Shotgun, Rifle,
    // Knife, Axe]) (things.py:115-116), in player_names order, before the agents are created (game.py:157-165)
#pragma unroll 1
    for (int b = 0; b < p.P; ++b) {
        if (p.bot_kinds[b] == ZS_KIND_TROLL || p.bot_kinds[b] == ZS_KIND_HAMSTER || p.bot_kinds[b] == ZS_KIND_RANDOMAN) {
            const int pick = below(draw_at(p, e, 0u, k), 5);
            ++k;
            if (lane == 0) TM(b) = (uint8_t)(pick == 0 ? ZS_WEAPON_GUN : pick == 1 ? ZS_WEAPON_SHOTGUN
                                             : pick == 2 ? ZS_WEAPON_RIFLE : pick == 3 ? ZS_WEAPON_KNIFE : ZS_WEAPON_AXE);
        }
    }
    // agent_weapon="random": one random.choice per agent, in agent order (weapons.py:43)
#pragma unroll 1
    for (int a = 0; a < p.A; ++a) {
        if (p.agent_weapons[a] == ZS_WEAPON_RANDOM) {
            const int pick = below(draw_at(p, e, 0u, k), 5);
            ++k;
            if (lane == 0) TM(p.P + a) = (uint8_t)(pick == 0 ? ZS_WEAPON_KNIFE : pick == 1 ? ZS_WEAPON_AXE
                                                   : pick == 2 ? ZS_WEAPON_GUN : pick == 3 ? ZS_WEAPON_RIFLE : ZS_WEAPON_SHOTGUN);
        }
    }
    PH(13);
    if (flags & FL_DMG) spl_refresh_present<MPC, G, CV>(p, e);
    gsync<G, CV>(e);
    build_grid<MPC, G, false>(p, id, flags);  // every slot is out of the world here: statics (all present) only
    PH(14);
#pragma unroll 1
    for (int s = e.gl; s < p.P; s += G) LIST(s) = (uint16_t)s;
    if (lane == 0) SCALW(ZS_S_STAMP_COUNTER) = 0;
    gsync<G, CV>(e);
    k = spawn_in_random<MPC, G, false>(p, id, episode, 0u, k, p.P, 0, 0, true, true);
    PH(15);
#pragma unroll 1
    for (int a = e.gl; a < p.A; a += G) LIST(a) = (uint16_t)(p.P + a);
    gsync<G, CV>(e);
    k = spawn_in_random<MPC, G, false>(p, id, episode, 0u, k, p.A, 0, SCALW(ZS_S_STAMP_COUNTER), p.P == 0, true);
    PH(16);
    // (the zombie spawn cells are all free unless the players, lacking spawn cells of their own, stood anywhere: on them too)
    k = spawn_zombies<MPC, G, false>(p, id, episode, 0u, k, p.initial_zombies, SCALW(ZS_S_STAMP_COUNTER),
                                     p.n_ps > 0 || p.P + p.A == 0, true);
    PH(17);
#pragma unroll 1
    for (int a = e.gl; a < p.A; a += G) PREVL(a) = TL(p.P + a);
    if (lane == 0) {
        SCALW(ZS_S_T) = -1; SCALW(ZS_S_EPISODE) = episode; SCALW(ZS_S_DEATHS) = 0; SCALW(ZS_S_ZOMBIE_DEATHS) = 0;
        SCALW(ZS_S_FLAGS) = flags; SCALW(ZS_S_PREV_ZOMBIE_DEATHS) = 0; SCALW(ZS_S_EPISODE_STEPS) = 0;
    }
    gsync<G, CV>(e);
    return k;
}

// ---------------------------------------------------------------- rules (zombsole/rules/*.py)
template <int MPC, int G, bool CV, int ROS = 0>
__device__ __forceinline__ void rules_eval(const ZsParams& p, Env& e, bool& ended, bool& won, bool& agents_alive) {
    ZS_CONSTS; ZS_VIEWS;
    using R = Roster<ROS>;
    static_assert(!R::on || ONE, "a roster kernel has one lane per slot");
    const int lane = e.gl;
    const int P = R::on ? R::P : p.P, NP = R::on ? R::NP : p.P + p.A;
    const int rules = R::on ? R::rules : p.rules;
    int alive = 0, ag = 0;
#pragma unroll 1
    for (int s0 = 0; s0 < (ONE ? 1 : (NP)); s0 += G) {
        const int s = s0 + lane;
        const bool al = s < NP && TL(s) > 0;
        alive += __popc(gballot<G, CV>(e, al));
        ag += __popc(gballot<G, CV>(e, al && s >= P));
    }
    agents_alive = ag > 0;                    // rules/rules.py:13-18
    const bool players_alive = alive > 0;     // rules/rules.py:6-11
    won = players_alive;
    if (rules == ZS_RULES_EXTERMINATION) {  // extermination.py:12-26
        bool z = false;
        if constexpr (R::on) {  // (one lane per slot: every zombie slot is NP + lane of some lane)
            const int s = NP + e.gl;
            z = s < p.M && (TM(s) & 0x80) && TL(s) > 0;
        } else {
#pragma unroll 1
            for (int s = NP + e.gl; s < p.M; s += G) z |= (TM(s) & 0x80) && TL(s) > 0;
        }
        const bool any_z = gany<G, CV>(e, z);  // (every lane of the warp votes: no short-circuit around a primitive)
        ended = !players_alive || !any_z;
    } else if (rules == ZS_RULES_SURVIVAL) {  // survival.py:5-7
        ended = !players_alive;
    } else if (rules == ZS_RULES_SAFEHOUSE) {  // safehouse.py:10-32
        bool out = false;
#pragma unroll 1
        for (int s = e.gl; s < NP; s += G) {
            const uint32_t xy = TXY(s);
            out |= TL(s) > 0 && !objective_bit(p, xy_y(xy) * p.W + xy_x(xy));
        }
        const bool any_out = gany<G, CV>(e, out);
        ended = players_alive ? !any_out : true;
    } else {  // evacuation.py:13-57: at least half the team alive and the living form one 4-connected cluster
        const bool half = 2 * alive >= NP;  // len(alive) >= len(all) / 2.0
        won = half;
        ended = true;
        {
            int together = 0;
            if (half && lane == 0) {
                unsigned long long seen = 0, pending = 0;
                int first = 0;
                while (TL(first) <= 0) ++first;
                pending = 1ull << first;
                while (pending) {
                    const int s = __ffsll((long long)pending) - 1;
                    pending &= pending - 1;
                    seen |= 1ull << s;
                    ++together;
                    const uint32_t xy = TXY(s);
#pragma unroll 1
                    for (int d = 0; d < 4; ++d) {
                        const int g = grid_at(p, GRIDP, xy_x(xy) + adj_dx(d), xy_y(xy) + adj_dy(d));
                        if (g >= 1 && g <= NP && TL(g - 1) > 0 && !((seen | pending) >> (g - 1) & 1ull)) pending |= 1ull << (g - 1);
                    }
                }
            }
            together = gbcast<G, CV>(e, together, 0);
            if (half) ended = together == alive;
        }
    }
}

// life / 100.0, correctly rounded like the reference's float division.  For the integers that occur (|life sum| is
// a few thousand at most) one Newton correction of the product with RN(1/100) is exact — checked exhaustively for
// |a| <= 200,000 against exact rational arithmetic (tests/test_reward_division.py); anything larger takes the division.
__device__ __forceinline__ double div100(int a) {
    const double x = __int2double_rn(a);
    if (a > 200000 || a < -200000) return __ddiv_rn(x, 100.0);
    const double r = 0.01;  // RN(1/100)
    const double q0 = __dmul_rn(x, r);
    return __fma_rn(__fma_rn(-100.0, q0, x), r, q0);
}
__device__ __forceinline__ double total_reward(int zombie_deaths, int life_sum) {
    // reward.py:37-41 / 90-92: int + float, the division first
    return __dadd_rn(__int2double_rn(zombie_deaths), div100(life_sum));
}
