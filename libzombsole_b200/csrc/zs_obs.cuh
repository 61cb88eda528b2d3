// zs_obs.cuh — observation encoder (zombsole/gym/observation.py:36-173), lanes over cells.
//
// World scope: template stream + ordered patches (obs_world_template / obs_world_patch below).
// Surroundings scope: per-cell encoding of the agent-centred window from the occupancy grid.
#pragma once
#include "zs_world.cuh"

struct CellInfo { int label, life, weapon, agent; };

ZS_TPL __device__ __forceinline__ CellInfo cell_info(const ZsParams& p, const Env& e, int c, int g) {
    ZS_VIEWS;
    CellInfo ci;
    ci.life = 0; ci.weapon = 0; ci.agent = -1;
    if (g == G_EMPTY) ci.label = objective_bit(p, c) ? ZS_LABEL_OBJECTIVE : 0;
    else if (g == G_DEAD) ci.label = ZS_LABEL_DEAD_BODY;
    else if (g > G_MAX_SLOT) {
        const int i = __ldg(p.cell_static + c);
        ci.label = __ldg(p.static_label + i);
        ci.life = SL(i);
    } else {
        const int s = g - 1;
        ci.life = TL(s);
        ci.weapon = TM(s) & 15;
        ci.label = s < p.P ? ZS_LABEL_PLAYER : s < p.P + p.A ? ZS_LABEL_AGENT : ZS_LABEL_ZOMBIE;
        ci.agent = s - p.P;
    }
    return ci;
}
// encode_position_simple (observation.py:36-55)
__device__ __forceinline__ int encode_simple(const CellInfo& ci) {
    if (ci.label == 0) return 0;
    const int adj = ci.life < 100 ? ci.life : 100;
    return 256 * ci.label + 16 * ci.weapon + floordiv100(15 * adj);
}
// encode_position_as_channels (observation.py:57-81): thing code of an agent is 8 + int(agent_id)
__device__ __forceinline__ int channel_label(const ZsParams& p, const CellInfo& ci) {
    return ci.label == ZS_LABEL_AGENT ? 8 + p.agent_obs_ids[ci.agent] : ci.label;
}

// World scope, pass 1: the observation of the pristine static layer (boxes, walls, objectives) is the
// same for every env and every step.  It is staged once per CTA in shared memory and copied to the env's
// observation row by the TMA (cp.async.bulk shared -> global, one instruction per plane per step); when the
// row is not 16-byte aligned (cell count not a multiple of 4) or the template does not fit, it is streamed
// from the L1-resident template with 128-bit loads/stores instead.  Either way it is issued BEFORE the
// world transition and drains underneath the latency-bound game logic.
ZS_TPL __device__ __forceinline__ void obs_world_template(const ZsParams& p, Env& e, int32_t* __restrict__ obs) {
    ZS_CONSTS;
    const int lane = e.gl;
    const int cells = p.cells;
    const bool channels = p.obs_enc == ZS_OBS_CHANNELS;
    if (p.tmpl_smem_off >= 0) {
        // TMA: the group's lane 0 issues one bulk copy per plane from the CTA-shared template to the env's row —
        // no per-lane loads/stores at all.  obs_world_patch waits for the group before it patches cells.
        // (issuing a bulk copy costs the lane about a thousand cycles, and the two halves of a warp cannot issue together:
        // small batches of two envs per warp, which are latency-bound, stage the planes twice and send both rows — they
        // are neighbours in the output — with one copy)
        const uint32_t row = (uint32_t)(p.tmpl_planes * cells) * 4u;
        if (G == 16 && CV && p.tmpl_pair) {
            if (e.gshift == 0 && lane == 0) { bulk_store_s(obs, e.tmpl_saddr, 2u * row); bulk_commit(); }
        } else if (lane == 0) { bulk_store_s(obs, e.tmpl_saddr, row); bulk_commit(); }
        return;
    }
    if ((cells & 3) == 0) {
        const int n4 = cells >> 2;
        const uint4* to4 = (const uint4*)p.tmpl_obs;
        uint4* o4 = (uint4*)obs;
#pragma unroll 4
        for (int i = lane; i < n4; i += G) __stcs(o4 + i, __ldg(to4 + i));
        if (channels) {
#pragma unroll 4
            for (int i = lane; i < n4; i += G) {
                __stcs(o4 + n4 + i, __ldg(to4 + n4 + i));
                __stcs(o4 + 2 * n4 + i, make_uint4(0, 0, 0, 0));
            }
        }
        return;
    }
    // maps whose cell count is not a multiple of 4 (an env's row is then not 16-byte aligned)
#pragma unroll 1
    for (int c = lane; c < cells; c += G) {
        __stcs(obs + c, __ldg(p.tmpl_obs + c));
        if (channels) { __stcs(obs + cells + c, __ldg(p.tmpl_obs + cells + c)); __stcs(obs + 2 * cells + c, 0); }
    }
}

__device__ __forceinline__ void obs_store_cell(const ZsParams& p, int32_t* obs, int c, const CellInfo& ci) {
    if (p.obs_enc == ZS_OBS_SIMPLE) obs[c] = encode_simple(ci);
    else { obs[c] = channel_label(p, ci); obs[p.cells + c] = ci.life; obs[2 * p.cells + c] = ci.weapon; }
}

// World scope, pass 2: the cells that differ from the pristine layer are patched with scalar stores.  The
// reference shows the thing on a cell, else its decoration (observation.py:41-42); the occupancy grid says which
// one that is, so every patched cell is written by exactly one lane and the three kinds of patches (damaged or
// destroyed boxes/walls, dead bodies, mobile things) need no ordering among themselves — only after pass 1.
__device__ __forceinline__ void obs_store_static(const ZsParams& p, int32_t* obs, uint32_t w) {
    const int cell = w & 0xffffu;
    int v0, v1;
    spl_cell_obs(p, w, v0, v1);
    if (p.obs_enc == ZS_OBS_SIMPLE) obs[cell] = v0;
    else { obs[cell] = v0; obs[p.cells + cell] = v1; obs[2 * p.cells + cell] = 0; }
}
__device__ __forceinline__ CellInfo thing_info(const ZsParams& p, int s, int life, int meta) {
    CellInfo ci;
    ci.life = life; ci.weapon = meta & 15; ci.agent = s - p.P;
    ci.label = s < p.P ? ZS_LABEL_PLAYER : s < p.P + p.A ? ZS_LABEL_AGENT : ZS_LABEL_ZOMBIE;
    return ci;
}

ZS_TPL __device__ __forceinline__ void obs_world_patch(const ZsParams& p, Env& e, int32_t* obs) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl;
    CellInfo body;
    body.label = ZS_LABEL_DEAD_BODY; body.life = 0; body.weapon = 0; body.agent = -1;
    // The first round of every kind of patch is read from shared memory BEFORE waiting for pass 1: the reads do
    // not depend on it, and issued together their latencies overlap.
    const int n_spl = (e.flags & FL_DMG) ? (int)SPN : 0;                 // boxes/walls whose observation differs
    const int n_dead = (e.flags & FL_DEAD_OVER) ? 0 : (int)DBL(0);        // dead bodies of this world, from the list
    const uint32_t w0 = lane < n_spl ? SPL(lane) : 0xffff0000u;
    const int cell0 = w0 & 0xffffu;
    const int dc0 = lane < n_dead ? (int)DBL(1 + lane) : 0;
    // gone from World.things (SPL_GONE): whatever took the cell patches it itself; a thing on a dead body hides it
    const bool do_static0 = lane < n_spl && (!spl_gone(w0) || GRID(cell0) == G_EMPTY);
    const bool do_dead0 = lane < n_dead && GRID(dc0) == G_DEAD;
    int tm0 = 0, tl0 = 0;
    uint32_t txy0 = 0;
    if (ONE && (G == MPC || lane < MPC)) { tm0 = TM(lane); tl0 = TL(lane); txy0 = TXY(lane); }
    if (p.tmpl_smem_off >= 0 && lane == 0) bulk_wait_all();  // pass 1 (TMA) has landed before any cell is patched
    gsync<G, CV>(e);
    PH(12);
    if (do_static0) obs_store_static(p, obs, w0);
    if (do_dead0) obs_store_cell(p, obs, dc0, body);
    if (ONE) {
        if (tm0 & 0x80) obs_store_cell(p, obs, xy_y(txy0) * p.W + xy_x(txy0), thing_info(p, lane, tl0, tm0));
    } else {
#pragma unroll 1
        for (int s = lane; s < p.M; s += G) {
            const int m = TM(s);
            if (!(m & 0x80)) continue;
            const uint32_t xy = TXY(s);
            obs_store_cell(p, obs, xy_y(xy) * p.W + xy_x(xy), thing_info(p, s, TL(s), m));
        }
    }
    // further rounds (long lists are rare)
#pragma unroll 1
    for (int i = lane + G; i < n_spl; i += G) {
        const uint32_t w = SPL(i);
        if (spl_gone(w) && GRID(w & 0xffffu) != G_EMPTY) continue;
        obs_store_static(p, obs, w);
    }
#pragma unroll 1
    for (int i = lane + G; i < n_dead; i += G) {
        const int c = DBL(1 + i);
        if (GRID(c) == G_DEAD) obs_store_cell(p, obs, c, body);
    }
    if (e.flags & FL_DEAD_OVER) {  // the list is not complete: walk the dead-body bitmap
#pragma unroll 1
        for (int w = lane; w < p.dead_words; w += G) {
            uint32_t bits = DEADW(w);
            while (bits) {
                const int c = w * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                if (GRID(c) == G_DEAD) obs_store_cell(p, obs, c, body);
            }
        }
    }
    // These patches went through the generic proxy; the next write to this row may be a bulk copy (async proxy: a later
    // step of this launch reusing the ring slot).  Each lane orders its own stores before whatever the async proxy does
    // later; the sync at the end of the step then puts them before lane 0's next issue.
    if (p.tmpl_smem_off >= 0) fence_proxy_async_global();
}

// World scope as a compact record (include/zs_b200.h: zs_step_compact): the cells pass 2 would patch, as entries of the
// env's record instead of stores into its observation row.  Every patched cell has exactly one writer, so the entries
// need no order; their positions come from ballot prefix sums (all rounds run on warp-level bounds: the primitives are
// full-mask when two envs share a warp).  Returns true when the record cannot hold the env (too many entries, or a
// value outside the entry's fields): the caller then writes the full row.  n_out: the entry count (0 on overflow).
// The words are STAGED in the env's per-step scratch (EnvS: act / bk / draws, dead by now) and leave as coalesced rows at the end
// (compact_flush): written to pinned host memory piece by piece as the rounds produce them they took 12 us longer to drain
// over PCIe than the same bytes in 128-byte rows (profiles/r02_e2e_host_step.txt).  Words beyond the scratch go out directly.
template <int MPC> __host__ __device__ constexpr int compact_stage_words() { return (int)(offsetof(EnvS<MPC>, zb) / sizeof(uint32_t)); }
ZS_TPL __device__ __forceinline__ void compact_flush(Env& e, uint32_t* __restrict__ rec, int n_words) {
    const uint32_t* const stage = reinterpret_cast<const uint32_t*>(zs_smem + e.b);  // (EnvS::act is the struct's first member)
    const int n = n_words < compact_stage_words<MPC>() ? n_words : compact_stage_words<MPC>();
    gsync<G, CV>(e);
    for (int i = e.gl; i < n; i += G) rec[i] = stage[i];
}
// WIN: keep only the items whose cell lies in at least one agent's surroundings window (obs_surroundings_compact);
// hdr: the record's header words, in front of the entries.
template <int MPC, int G, bool CV, bool WIN>
__device__ __forceinline__ bool obs_compact_entries(const ZsParams& p, Env& e, uint32_t* __restrict__ rec, int hdr, int cap_words, int& n_out) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl;
    // the window test of encode_surroundings (into_windows), windows centred on every agent slot's (possibly stale) position
    auto seen = [&](int cell) {
        if (!WIN) return true;
        const int half = p.sw >> 1, y = cell / p.W, x = cell - y * p.W;
#pragma unroll 1
        for (int a = 0; a < p.A; ++a) {
            const uint32_t axy = TXY(p.P + a);
            if ((unsigned)(x - (xy_x(axy) - half)) < (unsigned)p.sw && (unsigned)(y - (xy_y(axy) - half)) < (unsigned)p.sw) return true;
        }
        return false;
    };
    const unsigned below_l = (1u << lane) - 1u;
    const bool simple = p.obs_enc == ZS_OBS_SIMPLE;
    const int cap = simple ? cap_words : (cap_words >> 1);
    int n = 0;
    bool bad = false;
    uint32_t* const stage = reinterpret_cast<uint32_t*>(&S.act[0]);
    auto put = [&](int w, uint32_t v) { if (w < compact_stage_words<MPC>()) stage[w] = v; else rec[w] = v; };
    auto emit = [&](bool on, int cell, int v0, int v1, int v2) {
        if (WIN) on = on && seen(cell);
        const unsigned m = gballot<G, CV>(e, on);
        const int pos = n + __popc(m & below_l);
        if (on) {
            if (simple) {
                bad |= v0 < -32768 || v0 > 32767;
                if (pos < cap) put(hdr + pos, (uint32_t)cell | ((uint32_t)v0 << 16));
            } else {
                bad |= v0 < -32768 || v0 > 32767 || (unsigned)v2 > 0xffffu || v1 < -32768 || v1 > 32767;
                if (pos < cap) {
                    put(hdr + 2 * pos, (uint32_t)cell | ((uint32_t)v0 << 16));
                    put(hdr + 2 * pos + 1, ((uint32_t)v1 & 0xffffu) | ((uint32_t)v2 << 16));
                }
            }
        }
        n += __popc(m);
    };
    const int n_spl = (e.flags & FL_DMG) ? (int)SPN : 0;
    const int r_spl = wmax<G, CV>(e, n_spl);
#pragma unroll 1
    for (int i0 = 0; i0 < r_spl; i0 += G) {
        const int i = i0 + lane;
        const uint32_t w = i < n_spl ? SPL(i) : 0u;
        const int cell = w & 0xffffu;
        // gone from World.things (SPL_GONE): whatever took the cell shows itself; else the cell reads as empty
        const bool on = i < n_spl && (!spl_gone(w) || GRID(cell) == G_EMPTY);
        int v0 = 0, v1 = 0;
        if (on) spl_cell_obs(p, w, v0, v1);
        emit(on, cell, v0, v1, 0);
    }
    const int body0 = simple ? 256 * ZS_LABEL_DEAD_BODY : ZS_LABEL_DEAD_BODY;
    const bool dead_over = (e.flags & FL_DEAD_OVER) != 0;
    const int n_dead = dead_over ? 0 : (int)DBL(0);
    const int r_dead = wmax<G, CV>(e, n_dead);
#pragma unroll 1
    for (int i0 = 0; i0 < r_dead; i0 += G) {
        const int i = i0 + lane;
        const int c = i < n_dead ? (int)DBL(1 + i) : 0;
        emit(i < n_dead && GRID(c) == G_DEAD, c, body0, 0, 0);  // (a cell listed twice makes two equal entries)
    }
    if (wany<G, CV>(e, dead_over)) {  // the list is not complete: walk the dead-body bitmap
        const int words = dead_over ? p.dead_words : 0;
        const int r_w = wmax<G, CV>(e, words);
#pragma unroll 1
        for (int w0 = 0; w0 < r_w; w0 += G) {
            const int w = w0 + lane;
            uint32_t bits = w < words ? DEADW(w) : 0u;
            int left = (int)__reduce_max_sync(gmask<G, CV>(e), (unsigned)__popc(bits));
#pragma unroll 1
            for (; left > 0; --left) {
                const int c = bits ? w * 32 + __ffs(bits) - 1 : 0;
                const bool on = bits != 0u && GRID(c) == G_DEAD;
                bits &= bits - 1u;
                emit(on, c, body0, 0, 0);
            }
        }
    }
    if constexpr (MPC > G) {  // more slots than lanes (step_loop_general): a ballot round per G slots
#pragma unroll 1
        for (int s0 = 0; s0 < p.M; s0 += G) {
            const int s = s0 + lane;
            const int m = s < p.M ? (int)TM(s) : 0;
            const bool on = (m & 0x80) != 0;
            const uint32_t xy = on ? TXY(s) : 0u;
            const CellInfo ci = thing_info(p, s, on ? (int)TL(s) : 0, m);
            if (simple) emit(on, xy_y(xy) * p.W + xy_x(xy), encode_simple(ci), 0, 0);
            else emit(on, xy_y(xy) * p.W + xy_x(xy), channel_label(p, ci), ci.life, ci.weapon);
        }
    } else {
        const bool in_cap = G == MPC || lane < MPC;
        const int m = in_cap ? (int)TM(lane) : 0;
        const bool on = (m & 0x80) != 0;
        const uint32_t xy = in_cap ? TXY(lane) : 0u;
        const CellInfo ci = thing_info(p, lane, in_cap ? (int)TL(lane) : 0, m);
        if (simple) emit(on, xy_y(xy) * p.W + xy_x(xy), encode_simple(ci), 0, 0);
        else emit(on, xy_y(xy) * p.W + xy_x(xy), channel_label(p, ci), ci.life, ci.weapon);
    }
    const bool over = gany<G, CV>(e, bad) || n > cap;
    n_out = over ? 0 : n;
    return over;
}
ZS_TPL __device__ __forceinline__ bool obs_world_compact(const ZsParams& p, Env& e, uint32_t* __restrict__ rec, int cap_words, int& n_out) {
    return obs_compact_entries<MPC, G, CV, false>(p, e, rec, ZS_COMPACT_HEADER, cap_words, n_out);
}
// Surroundings scope, one window per agent, as a compact record (include/zs_b200.h: zs_step_compact_agents): the items pass 2
// of encode_surroundings patches, in the world record's entry encoding, behind a header of ZS_AGENT_COMPACT_HEADER(A) words
// (the caller stages it).  An item no window shows is left out: that keeps the records of large maps small.  Returns the entry
// count, -1 on overflow.  (Out of line: inlined into the step loop it made the surroundings kernels spill more.)
ZS_TPL __device__ __noinline__ int obs_surroundings_compact(const ZsParams& p, GrpId id, int flags, uint32_t* __restrict__ rec, int cap_words) {
    Env e = env_of(p, id);
    e.flags = flags;
    int n = 0;
    return obs_compact_entries<MPC, G, CV, true>(p, e, rec, ZS_AGENT_COMPACT_HEADER(p.A), cap_words, n) ? -1 : n;
}

// World scope as a record for the producer warp (zs_device.cuh: ObsMail): the cells pass 2 would patch as two-word entries
// in shared memory — simple encoding: cell, value; channels: cell | thing << 16, (life & 0xffff) | weapon << 16.  Returns
// the number of entries, or -1 when the record cannot describe the env (the dead-body list is not complete, more entries
// than it holds, a channel value outside 16 bits): the producer then encodes from the env's block itself.
ZS_TPL __device__ __forceinline__ int obs_world_record(const ZsParams& p, Env& e, uint32_t* __restrict__ rec, int cap) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl;
    const unsigned below_l = (1u << lane) - 1u;
    const bool simple = p.obs_enc == ZS_OBS_SIMPLE;
    int n = 0;
    bool bad = (e.flags & FL_DEAD_OVER) != 0;
    auto emit = [&](bool on, int cell, int v0, int v1, int v2) {
        const unsigned m = gballot<G, CV>(e, on);
        const int pos = n + __popc(m & below_l);
        if (on && pos < cap) {
            if (simple) { rec[2 * pos] = (uint32_t)cell; rec[2 * pos + 1] = (uint32_t)v0; }
            else {
                bad |= (unsigned)v0 > 0xffffu || (unsigned)v2 > 0xffffu || v1 < -32768 || v1 > 32767;
                rec[2 * pos] = (uint32_t)cell | ((uint32_t)v0 << 16);
                rec[2 * pos + 1] = ((uint32_t)v1 & 0xffffu) | ((uint32_t)v2 << 16);
            }
        }
        n += __popc(m);
    };
    const int n_spl = (e.flags & FL_DMG) ? (int)SPN : 0;
    const int r_spl = wmax<G, CV>(e, n_spl);
#pragma unroll 1
    for (int i0 = 0; i0 < r_spl; i0 += G) {
        const int i = i0 + lane;
        const uint32_t w = i < n_spl ? SPL(i < n_spl ? i : 0) : 0u;
        const int cell = w & 0xffffu;
        // gone from World.things (SPL_GONE): whatever took the cell shows itself; else the cell reads as empty
        const bool on = i < n_spl && (!spl_gone(w) || GRID(cell) == G_EMPTY);
        int v0 = 0, v1 = 0;
        if (on) spl_cell_obs(p, w, v0, v1);
        emit(on, cell, v0, v1, 0);
    }
    const int body0 = simple ? 256 * ZS_LABEL_DEAD_BODY : ZS_LABEL_DEAD_BODY;
    const int n_dead = (e.flags & FL_DEAD_OVER) ? 0 : (int)DBL(0);
    const int r_dead = wmax<G, CV>(e, n_dead);
#pragma unroll 1
    for (int i0 = 0; i0 < r_dead; i0 += G) {
        const int i = i0 + lane;
        const int c = i < n_dead ? (int)DBL(1 + i) : 0;
        emit(i < n_dead && GRID(c) == G_DEAD, c, body0, 0, 0);
    }
    {
        const bool in_cap = G == MPC || lane < MPC;
        const int m = in_cap ? (int)TM(in_cap ? lane : 0) : 0;
        const bool on = (m & 0x80) != 0;
        const uint32_t xy = in_cap ? TXY(in_cap ? lane : 0) : 0u;
        const CellInfo ci = thing_info(p, lane, in_cap ? (int)TL(in_cap ? lane : 0) : 0, m);
        if (simple) emit(on, xy_y(xy) * p.W + xy_x(xy), encode_simple(ci), 0, 0);
        else emit(on, xy_y(xy) * p.W + xy_x(xy), channel_label(p, ci), ci.life, ci.weapon);
    }
    return (gany<G, CV>(e, bad) || n > cap) ? -1 : n;
}

// The producer warp of a CTA (zs_sim_kernel SHAPE 3): for every step, the pristine planes go to the rows of the CTA's envs,
// then the entries the game warps left in the mailboxes are stored.  One warp, 32 lanes, no env of its own.
template <int MPC>
__device__ __forceinline__ void obs_producer(const ZsParams& p, const ZsIO& io, int envs_per_cta, uint32_t tmpl_saddr) {
    const int lane = threadIdx.x & 31;
    const int env0 = blockIdx.x * envs_per_cta;
    const int mail_stride = (int)sizeof(ObsMail) + 8 * p.prod_cap;
    const int n4 = (p.tmpl_planes * p.cells) >> 2;  // 128-bit words per row
    const uint4* const t4 = reinterpret_cast<const uint4*>(zs_smem + p.tmpl_smem_off);
    const bool simple = p.obs_enc == ZS_OBS_SIMPLE;
    int n_act = p.N - env0;
    if (n_act > envs_per_cta) n_act = envs_per_cta;
    const size_t obs_stride = (size_t)p.N * p.obs_elems;
    // pass 1 for one row: the pristine planes straight from the staged copy with 128-bit stores (a bulk copy per row,
    // issued by one thread, cost more than the whole step it was meant to relieve: measured)
    auto pristine = [&](int32_t* row) {
        uint4* const o4 = reinterpret_cast<uint4*>(row);
#pragma unroll 4
        for (int c = lane; c < n4; c += 32) __stcs(o4 + c, t4[c]);
    };
    // The envs are served as their records arrive, each at its own pace (lane i keeps env i's step and ring slot): a
    // producer that waited for all its envs every step would tie the four game warps of the CTA to the slowest of them.
    int my_step = 0, my_slot = 0;
#pragma unroll 1
    for (int i = 0; i < n_act; ++i) pristine(io.obs + (size_t)(env0 + i) * p.obs_elems);  // step 0's rows
    __syncwarp();
    int left = n_act * io.n_steps;
#pragma unroll 1
    while (left > 0) {
        // which envs have a record waiting (one test per lane, no blocking)
        bool ready = false;
        if (lane < n_act && my_step < io.n_steps) {
            const uint32_t a = (uint32_t)__cvta_generic_to_shared(&reinterpret_cast<ObsMail*>(zs_smem + p.prod_off + lane * mail_stride)->full);
            uint32_t ok;
            asm volatile("{\n.reg .pred q;\nmbarrier.test_wait.parity.shared::cta.b64 q, [%1], %2;\nselp.u32 %0, 1, 0, q;\n}\n"
                         : "=r"(ok) : "r"(a), "r"((uint32_t)(my_step & 1)) : "memory");
            ready = ok != 0u;
        }
        unsigned todo = __ballot_sync(0xffffffffu, ready);
        if (todo == 0u) { __nanosleep(64); continue; }
#pragma unroll 1
        for (; todo; todo &= todo - 1u) {
            const int i = __ffs(todo) - 1;
            const int slot_i = __shfl_sync(0xffffffffu, my_slot, i), step_i = __shfl_sync(0xffffffffu, my_step, i);
            ObsMail* const mail = reinterpret_cast<ObsMail*>(zs_smem + p.prod_off + i * mail_stride);
            const uint32_t* rec = reinterpret_cast<const uint32_t*>(mail + 1);
            int32_t* const obs = io.obs + (size_t)slot_i * obs_stride + (size_t)(env0 + i) * p.obs_elems;
            const int cnt = mail->count;
            if (cnt >= 0) {  // pass 2: the entries
#pragma unroll 1
                for (int k = lane; k < cnt; k += 32) {
                    const uint32_t w0 = rec[2 * k], w1 = rec[2 * k + 1];
                    if (simple) obs[w0] = (int32_t)w1;
                    else {
                        const int cell = (int)(w0 & 0xffffu);
                        obs[cell] = (int32_t)(w0 >> 16);
                        obs[p.cells + cell] = (int32_t)(int16_t)(w1 & 0xffffu);
                        obs[2 * p.cells + cell] = (int32_t)(w1 >> 16);
                    }
                }
            } else {  // rare: straight from the env's block (its game warp waits for `empty`)
                Env e2;
                e2.b = (uint32_t)(i * p.smem_per_env); e2.env = env0 + i; e2.env_global = p.env_base + (uint32_t)(env0 + i);
                e2.gl = lane; e2.gm = 0xffffffffu; e2.gshift = 0; e2.flags = mail->flags; e2.tmpl_saddr = tmpl_saddr;
                e2.t = e2.episode = e2.deaths = e2.zd = e2.nlive = e2.prev_zd = e2.ep_steps = 0;
                obs_world_patch<MPC, 32, false>(p, e2, obs);
            }
            __syncwarp();  // (the record has been read; these stores come before this warp's next stores into the same row)
            if (lane == 0) mbar_arrive(&mail->empty);
            // the next step's row of this env gets its pristine planes right away, long before its record arrives
            if (step_i + 1 < io.n_steps) {
                const int ns = slot_i + 1 >= io.obs_slots ? 0 : slot_i + 1;
                pristine(io.obs + (size_t)ns * obs_stride + (size_t)(env0 + i) * p.obs_elems);
                __syncwarp();
            }
            if (lane == i) { my_step += 1; my_slot = my_slot + 1 >= io.obs_slots ? 0 : my_slot + 1; }
            left -= 1;
        }
    }
}

// surroundings window (observation.py:99-119): rows = y, columns = x, centred on the agent's (possibly stale, if
// dead) position; out-of-bounds cells are a fresh Wall (observation.py:43-44,64-65).  Like the world scope it is
// written in two passes: the pristine layer of every window from the (L1-resident) padded template planes, then
// the cells that differ — static patch list, dead bodies, mobile things — stored into the windows they fall in.
// The occupancy grid says what is on top of a cell, so every patched cell has exactly one writer; one __syncwarp
// orders the patches after pass 1.
// One plane of one window, pristine layer: ww = sw*sw consecutive int32 whose first element is only 4-byte aligned
// (a plane is 441 elements at the default width).  The elements up to the first 16-byte boundary and behind the last
// one go out as one scalar store from a few lanes; the body is 128-bit stores, each lane gathering its four cells
// from the padded template plane (uint16, out-of-bounds cells are the fresh Wall of observation.py:43-44,64-65, so
// there is no bounds check): one division per store (multiply by the reciprocal of sw, exact for i < 65536), the
// row wrap of the three following cells by compare.  src == nullptr: the plane is zero (weapons of the static layer).
template <int G>
__device__ __forceinline__ void window_plane(const ZsParams& p, int lane, int32_t* __restrict__ o, const uint16_t* __restrict__ src) {
    const int w = p.sw, ww = w * w, skip = p.pad_w - w;
    int head = (int)(((0u - (uint32_t)(uintptr_t)o) >> 2) & 3u);
    if (head > ww) head = ww;
    const int nb = (ww - head) >> 2, tail = ww - head - 4 * nb;
    if (lane < head + tail) {
        const int i = lane < head ? lane : ww - tail + (lane - head);
        const int r = (int)__umulhi((uint32_t)i, p.sw_magic);
        __stcs(o + i, src ? (int)__ldg(src + i + r * skip) : 0);
    }
    uint4* o4 = reinterpret_cast<uint4*>(o + head);
    if (src == nullptr) {
#pragma unroll 2
        for (int q = lane; q < nb; q += G) __stcs(o4 + q, make_uint4(0u, 0u, 0u, 0u));
        return;
    }
#pragma unroll 2
    for (int q = lane; q < nb; q += G) {
        const int i0 = head + 4 * q;
        const int r0 = (int)__umulhi((uint32_t)i0, p.sw_magic);
        const int c0 = i0 - r0 * w;
        const uint16_t* s0 = src + i0 + r0 * skip;  // == src + r0 * pad_w + c0
        uint4 v;
        v.x = __ldg(s0);
        v.y = __ldg(s0 + 1 + (c0 + 1 >= w ? skip : 0));
        v.z = __ldg(s0 + 2 + (c0 + 2 >= w ? skip : 0));
        v.w = __ldg(s0 + 3 + (c0 + 3 >= w ? skip : 0));
        __stcs(o4 + q, v);
    }
}
// The pristine window block of one agent as a straight copy: win_table holds, for every cell an agent can stand on,
// the n_copy = (1 or 2) * sw * sw int32 of its label (and life) planes exactly as they go out (rows of the table start
// on 128-byte boundaries); the rest of the block (the weapon plane) is zero.  A block in the output is only 4-byte
// aligned, so the copy is word by word with consecutive lanes on consecutive words: every load is one aligned
// 128-byte line from the L2, every store at most two — cheaper in the L1 than wider accesses that straddle lines.
// Eight loads per lane are issued back to back.
template <int G>
__device__ __forceinline__ void window_block(int lane, int32_t* __restrict__ o, const int32_t* __restrict__ src, int n_copy, int n_all) {
#pragma unroll 1
    for (int i0 = lane; i0 < n_copy; i0 += 8 * G) {
        int v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) if (i0 + k * G < n_copy) v[k] = __ldg(src + i0 + k * G);
#pragma unroll
        for (int k = 0; k < 8; ++k) if (i0 + k * G < n_copy) __stcs(o + i0 + k * G, v[k]);
    }
#pragma unroll 4
    for (int i = n_copy + lane; i < n_all; i += G) __stcs(o + i, 0);
}
__device__ __forceinline__ void window_store(const ZsParams& p, int32_t* o, int ww, int idx, int v0, int v1, int v2) {
    if (p.obs_enc == ZS_OBS_SIMPLE) o[idx] = v0;
    else { o[idx] = v0; o[ww + idx] = v1; o[2 * ww + idx] = v2; }
}
ZS_TPL __device__ __forceinline__ void encode_surroundings(const ZsParams& p, Env& e, int32_t* __restrict__ obs) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl;
    const int w = p.sw, half = p.sw >> 1, ww = p.sw * p.sw;
    const bool simple = p.obs_enc == ZS_OBS_SIMPLE;
    const int A = p.obs_count;
    // ---- pass 1
#pragma unroll 1
    for (int a = 0; a < A; ++a) {
        const uint32_t axy = TXY(p.P + a);
        int32_t* o = obs + (size_t)a * p.obs_C * ww;
        if (p.win_table) {
            window_block<G>(lane, o, p.win_table + (size_t)(xy_y(axy) * p.W + xy_x(axy)) * p.win_pitch, p.win_ints, p.obs_C * ww);
            continue;
        }
        // top-left corner of the window in the padded planes (the padding is `half` cells wide)
        const uint16_t* src = p.tmpl_pad + xy_y(axy) * p.pad_w + xy_x(axy);
        window_plane<G>(p, lane, o, src);
        if (!simple) { window_plane<G>(p, lane, o + ww, src + p.pad_plane); window_plane<G>(p, lane, o + 2 * ww, nullptr); }
    }
    gsync<G, CV>(e);
    // ---- pass 2: one item (box/wall entry, dead body, mobile thing) per lane, stored into every window that shows it
    auto into_windows = [&](int cell, int v0, int v1, int v2) {
        const int y = cell / p.W, x = cell - y * p.W;
#pragma unroll 1
        for (int a = 0; a < A; ++a) {
            const uint32_t axy = TXY(p.P + a);
            const int wx = x - (xy_x(axy) - half), wy = y - (xy_y(axy) - half);
            if ((unsigned)wx < (unsigned)w && (unsigned)wy < (unsigned)w)
                window_store(p, obs + (size_t)a * p.obs_C * ww, ww, wy * w + wx, v0, v1, v2);
        }
    };
    if (e.flags & FL_DMG) {
        const int n_spl = SPN;
#pragma unroll 1
        for (int i = lane; i < n_spl; i += G) {
            const uint32_t wd = SPL(i);
            const int cell = wd & 0xffffu;
            if (spl_gone(wd) && GRID(cell) != G_EMPTY) continue;  // gone: whatever took the cell shows itself
            int v0, v1;
            spl_cell_obs(p, wd, v0, v1);
            into_windows(cell, v0, v1, 0);
        }
    }
    const int body0 = simple ? 256 * ZS_LABEL_DEAD_BODY : ZS_LABEL_DEAD_BODY;
    if (!(e.flags & FL_DEAD_OVER)) {
        const int n_dead = DBL(0);
#pragma unroll 1
        for (int i = lane; i < n_dead; i += G) {
            const int c = DBL(1 + i);
            if (GRID(c) == G_DEAD) into_windows(c, body0, 0, 0);
        }
    } else {
#pragma unroll 1
        for (int wd = lane; wd < p.dead_words; wd += G) {
            uint32_t bits = DEADW(wd);
            while (bits) {
                const int c = wd * 32 + __ffs(bits) - 1;
                bits &= bits - 1;
                if (GRID(c) == G_DEAD) into_windows(c, body0, 0, 0);
            }
        }
    }
#pragma unroll 1
    for (int s = lane; s < p.M; s += G) {
        const int m = TM(s);
        if (!(m & 0x80)) continue;
        const CellInfo ci = thing_info(p, s, TL(s), m);
        const uint32_t xy = TXY(s);
        const int cell = xy_y(xy) * p.W + xy_x(xy);
        if (simple) into_windows(cell, encode_simple(ci), 0, 0);
        else into_windows(cell, channel_label(p, ci), ci.life, ci.weapon);
    }
}

template <int MPC, int G, bool CV, bool SURR>
__device__ __forceinline__ void encode_obs(const ZsParams& p, Env& e, int32_t* obs) {
    if constexpr (!SURR) { obs_world_template<MPC, G, CV>(p, e, obs); obs_world_patch<MPC, G, CV>(p, e, obs); }
    else encode_surroundings<MPC, G, CV>(p, e, obs);
}
