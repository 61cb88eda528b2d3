// zs_b200.cu — kernels and C ABI (include/zs_b200.h) of the B200-native batched zombsole simulator.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
// No CPU fallback: every entry point that computes launches CUDA kernels.
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <omp.h>
#include <algorithm>
#include <vector>

#include "zs_device.cuh"
#include "zs_world.cuh"
#include "zs_obs.cuh"

// ================================================================ kernels
enum { MODE_STEP = 0, MODE_RESET = 1, MODE_ENCODE = 2 };

__device__ __forceinline__ int synthetic_action(const ZsParams& p, uint32_t env_global, uint32_t step_index, int agent) {
    const uint4 o = philox4x32_10(env_global, step_index, 0u, (uint32_t)(agent >> 2), p.key0, p.key1 ^ 0xAC710115u);
    return below(word_of(o, agent & 3), p.n_discrete);
}

// discrete id -> (type, dx, dy): ZombsoleGymEnvDiscreteAction.game_actions (gym_env.py:328-351),
// MultiagentZombsoleEnvDiscreteAction.game_actions (multiagent_env.py:259-285)
// (a table: type | (dx + 1) << 8 | (dy + 1) << 16 per id — one constant-bank load instead of a chain of selects)
__constant__ uint32_t c_discrete[8] = {
    ZS_ACT_MOVE | (1u << 8) | (2u << 16), ZS_ACT_MOVE | (0u << 8) | (1u << 16), ZS_ACT_MOVE | (1u << 8) | (0u << 16),
    ZS_ACT_MOVE | (2u << 8) | (1u << 16), ZS_ACT_ATTACK_CLOSEST | (1u << 8) | (1u << 16), ZS_ACT_HEAL | (1u << 8) | (1u << 16),
    ZS_ACT_HEAL_CLOSEST | (1u << 8) | (1u << 16), ZS_ACT_NONE | (1u << 8) | (1u << 16)};
__device__ __forceinline__ void discrete_to_action(const ZsParams& p, int id, int& type, int& dx, int& dy) {
    uint32_t w = c_discrete[(unsigned)id < (unsigned)p.n_discrete ? id : 7];
    if (id < 0 && p.obs_per_agent) w = ZS_ACT_ABSENT | (1u << 8) | (1u << 16);
    type = (int)(w & 0xffu); dx = (int)((w >> 8) & 0xffu) - 1; dy = (int)(w >> 16) - 1;
}

// zs_step_host: the env's record is complete.  ONE system-scope fence per group of envs, by whoever completes the group (a fence
// per warp takes 8-34 us when 4,096 warps fence at once): the others order their record words before the counter at gpu scope.
template <int G, bool CV>
__device__ __forceinline__ void compact_signal(const ZsParams& p, const ZsIO& io, const Env& e, int env) {
    __threadfence();
    gsync<G, CV>(e);
    if (e.gl == 0) {
        const int grp = env / io.group_envs;
        const int size = min(io.group_envs, p.N - grp * io.group_envs);
        if (atomicAdd(io.group_count + grp, 1) == size - 1) {
            io.group_count[grp] = 0;
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t*>(io.host_flags + 16 * grp) = io.ticket;
        }
    }
}

// ---------------------------------------------------------------- the K-step loop, more slots than lanes
// REC: world scope with the compact record compiled in (zs_sim_kernel SHAPE 5): every step leaves as a record (zs_step_compact,
// zs_step_host), the full row only for an env the record cannot hold.
// FIN: the final observation compiled in (zs_sim_kernel SHAPE 6 / 7): an env that the step re-initialises first writes the
// observation of the world it ended in to its row of io.final_obs, in the ring slot of the step's own observation.
// NXT: next-step autoreset compiled in (zs_sim_kernel SHAPE 8 / 9 / 11; one env per warp): an env whose step ends its episode
// keeps the world it ended in and is marked in io.pending; its next step is the world init instead of a transition, with the
// outputs of a new episode (reward +0.0, no flags, every agent in the mask, the init's draws).
template <int MPC, int G, bool CV, bool SURR, bool REC = false, bool FIN = false, bool NXT = false>
__device__ __forceinline__ void step_loop_general(const ZsParams& p, const ZsIO& io, Env& e) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl, env = e.env;
    const int A = p.A, NP = p.P + p.A;
    const int R = p.obs_per_agent ? A : 1;
    constexpr bool world_obs = !SURR;  // (the observation scope is compiled in: see zs_sim_kernel)
    // agent actions for the coming step, fetched one step ahead (Agent.set_action, agent.py:22-25);
    // agent a is handled by lanes a, a + G, ... of the group
    constexpr int AR = ZS_MAX_AGENTS / G > 0 ? ZS_MAX_AGENTS / G : 1;  // agents per lane (1 or 2)
    int at[AR], adx[AR], ady[AR];
    auto fetch_action = [&](int step) {
#pragma unroll
        for (int r = 0; r < AR; ++r) {
            const int a = lane + r * G;
            at[r] = ZS_ACT_NONE; adx[r] = 0; ady[r] = 0;
            if (a >= A) continue;
            const size_t sn = (size_t)step * p.N + env;
            if (io.actions == nullptr) discrete_to_action(p, synthetic_action(p, e.env_global, (uint32_t)(io.first_step + step), a), at[r], adx[r], ady[r]);
            else if (io.fmt == ZS_ACTIONS_DISCRETE) discrete_to_action(p, io.actions[sn * A + a], at[r], adx[r], ady[r]);
            else { const int32_t* q = io.actions + (sn * A + a) * 3; at[r] = q[0]; adx[r] = q[1]; ady[r] = q[2]; }
        }
    };
    fetch_action(0);
    int oslot = 0;
    bool pend = NXT && io.pending[env] != 0;
#pragma unroll 1
    for (int step = 0; step < io.n_steps; ++step) {
        const size_t sn = (size_t)step * p.N + env;
        int32_t* obs_out = nullptr;
        if (io.obs) {
            obs_out = io.obs + ((size_t)oslot * p.N + env) * p.obs_elems;
            if (++oslot >= io.obs_slots) oslot = 0;
            // pass 1 of the world observation does not depend on the transition: issue its stores now
            if constexpr (world_obs && !REC) obs_world_template<MPC, G, CV>(p, e, obs_out);
        }
        // agents alive before the step: the keys of the reference's per-agent dicts (multiagent_env.py:88-97)
        unsigned alive_before = 0;
        int life_before[AR];
#pragma unroll
        for (int r = 0; r < AR; ++r) {
            const int a = lane + r * G;
            // (narrowed to 16 bits: an unknown action type stays unknown, an offset beyond +-4097 is off any map either way)
            if (a < A) {
                ACTS(3 * a) = (int16_t)max(-1, min(127, at[r]));
                ACTS(3 * a + 1) = (int16_t)max(-4097, min(4097, adx[r])); ACTS(3 * a + 2) = (int16_t)max(-4097, min(4097, ady[r]));
            }
            alive_before |= gballot<G, CV>(e, a < A && TL(p.P + (a < A ? a : 0)) > 0) << (r * G);
            life_before[r] = a < A ? PREVL(a) : 0;
        }
        const int zd_before = e.prev_zd;
        const int life_prev0 = PREVL(0);
        gsync<G, CV>(e);
        if (step + 1 < io.n_steps) fetch_action(step + 1);

        int k;
        int life_now[AR];
        double rew[AR];
        bool ended = false, won = false, agents_alive = true;
        if (NXT && pend) {
            // ---- the reset step of next-step autoreset: the world init zs_reset performs (gym_env.py:148-164,
            // multiagent_env.py:173-184) instead of the transition; a new world's outputs
            k = initialize_world<MPC, G, false>(p, id_of(e), e.episode + 1, e.flags);
            scalars_from_smem<MPC, G, false>(p, e);
            pend = false;
            alive_before = 0;
#pragma unroll
            for (int r = 0; r < AR; ++r) {
                const int a = lane + r * G;
                life_now[r] = a < A ? TL(p.P + a) : 0;
                rew[r] = 0.0;
                alive_before |= gballot<G, CV>(e, a < A) << (r * G);
            }
        } else {
            k = world_step<MPC, G, CV>(p, e);
            e.ep_steps += 1;

            // ---- reward tracker update (reward.py:30-41, 77-92), float64 in the reference's operation order.
            // A tracker whose inputs did not change yields exactly +0.0.
            int sum_prev = 0, sum_new = 0;
#pragma unroll
            for (int r = 0; r < AR; ++r) {
                const int a = lane + r * G;
                life_now[r] = a < A ? TL(p.P + a) : 0;
                rew[r] = 0.0;
                if (!p.obs_per_agent) {
                    if (A > 1) { sum_prev += gadd<G, CV>(e, life_before[r]); sum_new += gadd<G, CV>(e, life_now[r]); }
                } else if (a < A && (life_before[r] != life_now[r] || zd_before != e.zd))
                    rew[r] = __dsub_rn(total_reward(e.zd, life_now[r]), total_reward(zd_before, life_before[r]));
            }
            if (!p.obs_per_agent) {
                if (A == 1) { sum_prev = life_prev0; sum_new = TL(p.P); }  // one agent: every lane reads the same two words
                if (sum_prev != sum_new || zd_before != e.zd)
                    rew[0] = __dsub_rn(total_reward(e.zd, sum_new), total_reward(zd_before, sum_prev));
            }
#pragma unroll
            for (int r = 0; r < AR; ++r) { const int a = lane + r * G; if (a < A) PREVL(a) = (int16_t)life_now[r]; }
            e.prev_zd = e.zd;
            gsync<G, CV>(e);

            // ---- Game.spawn_zombies_to_maintain_minimum (game.py:196-201)
            if (p.minimum_zombies > 0) {
                int zc = 0;
#pragma unroll 1
                for (int s0 = NP; s0 < p.M; s0 += G) zc += __popc(gballot<G, CV>(e, s0 + lane < p.M && (TM(s0 + lane) & 0x80)));
                if (zc < p.minimum_zombies) {
                    k = spawn_zombies<MPC, G, false>(p, id_of(e), e.episode, (uint32_t)(e.t + 1), k, p.minimum_zombies - zc, e.nlive, false, false);
                    e.nlive = SCALW(ZS_S_STAMP_COUNTER);
                }
            }

            // ---- rules and end reward (gym_env.py:130-141, multiagent_env.py:143-162)
            rules_eval<MPC, G, CV>(p, e, ended, won, agents_alive);
        }
        bool done = false, trunc = false;
        double end_reward = 0.0;
        if (ended) { done = true; end_reward = won ? 10.0 : -10.0; }
        else if (!agents_alive) { trunc = true; end_reward = -10.0; }
        if (!p.obs_per_agent) {
            if (done || trunc) rew[0] = __dadd_rn(rew[0], end_reward);
            if (io.reward && lane == 0) io.reward[sn] = rew[0];
        } else {
#pragma unroll
            for (int r = 0; r < AR; ++r) {
                const int a = lane + r * G;
                if (a >= A) continue;
                if (!((alive_before >> a) & 1u)) rew[r] = 0.0;
                else if (life_now[r] > 0) rew[r] = __dadd_rn(rew[r], end_reward);
                if (io.reward) io.reward[sn * R + a] = rew[r];
                if (io.agent_mask) io.agent_mask[sn * A + a] = (alive_before >> a) & 1u;
            }
        }
        if (p.max_steps > 0 && e.ep_steps >= p.max_steps) trunc = true;  // gymnasium TimeLimit
        if (lane == 0) {
            if (io.terminated) io.terminated[sn] = done;
            if (io.truncated) io.truncated[sn] = trunc;
            if (io.draws) io.draws[sn] = k;
        }
        if (!p.obs_per_agent && io.agent_mask && lane < A) io.agent_mask[sn * A + lane] = (alive_before >> lane) & 1u;

        // ---- same-step auto-reset (next-step: the world stays as it ended, its next step re-initialises it)
        if ((done || trunc) && (p.auto_reset || io.force_auto_reset)) {
            if (lane == 0) {
                atomicAdd(p.stats + 0, 1ull);
                if (done && won) atomicAdd(p.stats + 1, 1ull);
                atomicAdd(p.stats + 2, (unsigned long long)e.ep_steps);
                atomicAdd(p.stats + 3, (unsigned long long)e.zd);
            }
            // the terminal world, after the transition, the reward and the respawn: what zs_step writes without auto-reset
            // (gym_env.py:99-145)
            if constexpr (FIN) encode_obs<MPC, G, CV, SURR>(p, e, io.final_obs + (obs_out - io.obs));
            if constexpr (NXT) pend = true;
            else {
                // rare, and possibly only one env of the warp: the divergent flavour
                initialize_world<MPC, G, false>(p, id_of(e), e.episode + 1, e.flags);
                scalars_from_smem<MPC, G, false>(p, e);
            }
        }
        if constexpr (REC) {
            // the observation as a compact record with the reward and flags in its header (include/zs_b200.h: zs_step_compact),
            // staged in the step's scratch (EnvS::act .. zb): the respawn and the world init above were its last users, and the
            // next step writes it only after the sync at the end of this one
            uint32_t* const rec = io.compact + (size_t)env * io.compact_words;
            uint32_t* const stage = reinterpret_cast<uint32_t*>(zs_smem + e.b);
            int n_ent = 0;
            const bool over = obs_world_compact<MPC, G, CV>(p, e, rec, io.compact_words - ZS_COMPACT_HEADER, n_ent);
            if (lane == 0) {
                stage[0] = (uint32_t)n_ent | (done ? 1u << 16 : 0u) | (trunc ? 1u << 17 : 0u) | (over ? 1u << 18 : 0u); stage[1] = 0u;
                stage[2] = (uint32_t)__double2loint(rew[0]); stage[3] = (uint32_t)__double2hiint(rew[0]);
            }
            compact_flush<MPC, G, CV>(e, rec, ZS_COMPACT_HEADER + n_ent * (p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2));
            if (over && obs_out) {  // rare: the full row, for the caller to fetch
                obs_world_template<MPC, G, CV>(p, e, obs_out);
                obs_world_patch<MPC, G, CV>(p, e, obs_out);
            }
            if (io.host_flags) compact_signal<G, CV>(p, io, e, env);
        } else if (obs_out) {
            if constexpr (world_obs) obs_world_patch<MPC, G, CV>(p, e, obs_out);
            else encode_surroundings<MPC, G, CV>(p, e, obs_out);
        }
        gsync<G, CV>(e);
    }
    if constexpr (NXT) { if (lane == 0) io.pending[env] = pend; }
}

// ---------------------------------------------------------------- the K-step loop, one lane per slot
// Agent a is handled by the lane of its slot (P + a): its action, its tracker life and its reward never leave
// that lane's registers.  Output cursors advance by one step's stride instead of being recomputed.
// FAST = the standard rollout shape, fixed at compile time: one agent, one reward per env, world-scope observation,
// no minimum-zombie respawn, a discrete action tape in, observation / reward / terminated / truncated out and no
// diagnostics outputs (zs_launch picks it when a launch has that shape).
// PROD: the observation of every step is handed to the CTA's producer warp (zs_obs.cuh: obs_producer) instead of being
// written by the game warp: no bulk-copy issue, no wait for it, no global stores on the game warps' dependent chain.
// ROS: a game roster compiled in (zs_world.cuh: Roster; the standard rollout shape only), 0 = the game from ZsParams.
// REC: surroundings scope with the per-agent compact record compiled in (zs_sim_kernel SHAPE 4).
// FIN: the final observation compiled in (zs_sim_kernel SHAPE 6 / 7, as for step_loop_general).
// NXT: next-step autoreset compiled in (zs_sim_kernel SHAPE 8 / 9 / 10, one env per warp; as for step_loop_general).
template <int MPC, int G, bool CV, bool FAST, bool SURR, bool PROD = false, int ROS = 0, bool REC = false, bool FIN = false,
          bool NXT = false>
__device__ __forceinline__ void step_loop_one(const ZsParams& p, const ZsIO& io, Env& e) {
    ZS_CONSTS; ZS_VIEWS;
    const int lane = e.gl, env = e.env;
    ObsMail* const mail = PROD ? reinterpret_cast<ObsMail*>(zs_smem + p.prod_off + (int)(e.b / (uint32_t)p.smem_per_env) * ((int)sizeof(ObsMail) + 8 * p.prod_cap)) : nullptr;
    using R = Roster<ROS>;
    static_assert(!R::on || (FAST && !PROD), "rosters are compiled into the standard rollout shape");
    static_assert(!NXT || (G == 32 && !FAST && !FIN), "next-step autoreset runs one env per warp, in the generic shapes");
    const int A = FAST ? 1 : p.A, P = R::on ? R::P : p.P, NP = P + A;
    const int aidx = lane - P;
    const bool is_agent = aidx >= 0 && aidx < A;
    const bool per_agent = FAST ? false : p.obs_per_agent != 0;
    const bool lane_sum = FAST ? false : (!per_agent && A > 1);  // one reward from the sum of several agents' lives (reward.py:37-41)
    const bool want_mask = FAST ? false : (per_agent || io.agent_mask != nullptr);
    constexpr bool world_obs = !SURR;
    const bool auto_reset = p.auto_reset || io.force_auto_reset;
    // The agent's action for the coming step is LOADED one step ahead and decoded when its step starts, so the load's
    // latency hides under the previous transition (Agent.set_action, agent.py:22-25).
    int raw0 = -1, raw1 = 0, raw2 = 0;
    auto load_action = [&](int step) {
        if (!is_agent) return;
        const size_t ia = ((size_t)step * p.N + env) * A + aidx;
        if (FAST) { raw0 = io.actions[ia]; return; }
        if (io.actions == nullptr) raw0 = synthetic_action(p, e.env_global, (uint32_t)(io.first_step + step), aidx);
        else if (io.fmt == ZS_ACTIONS_DISCRETE) raw0 = io.actions[ia];
        else { const int32_t* q = io.actions + ia * 3; raw0 = q[0]; raw1 = q[1]; raw2 = q[2]; }
    };
    load_action(0);
    const size_t obs_stride = (size_t)p.N * p.obs_elems;
    int32_t* const obs_first = (FAST || io.obs) ? io.obs + (size_t)env * p.obs_elems : nullptr;
    int32_t* obs_cur = obs_first;
    int oslot = 0;
    size_t sn = env;  // step * N + env
    bool pend = NXT && io.pending[env] != 0;
#pragma unroll 1
    for (int step = 0; step < io.n_steps; ++step, sn += p.N) {
        TR_STEP_BEGIN();
        int32_t* const obs_out = obs_cur;
        if (FAST || obs_out) {
            { const bool wrap = ++oslot >= io.obs_slots; oslot = wrap ? 0 : oslot; obs_cur = wrap ? obs_first : obs_cur + obs_stride; }
            // pass 1 of the world observation does not depend on the transition: issue its stores now
            if constexpr (world_obs && !PROD) { if (FAST || io.compact == nullptr) obs_world_template<MPC, G, CV>(p, e, obs_out); }
        }
        PH(18);
        if (step == io.n_steps - 1) TR(24);
        // agents alive before the step: the keys of the reference's per-agent dicts (multiagent_env.py:88-97)
        unsigned alive_before = 0;
        if (want_mask) alive_before = gballot<G, CV>(e, is_agent && TL(is_agent ? lane : 0) > 0) >> P;
        const int life_before = is_agent ? (int)PREVL(aidx) : 0;
        const int zd_before = e.prev_zd;
        int my_at = ZS_ACT_NONE, my_dx = 0, my_dy = 0;
        if (is_agent) {
            if (FAST || io.actions == nullptr || io.fmt == ZS_ACTIONS_DISCRETE) discrete_to_action(p, raw0, my_at, my_dx, my_dy);
            else { my_at = raw0; my_dx = raw1; my_dy = raw2; }
        }
        if (step + 1 < io.n_steps) load_action(step + 1);
        PH(19);
        PH(0);

        int k, life_now;
        double rew = 0.0;
        bool ended = false, won = false, agents_alive = true;
        if (NXT && pend) {
            // ---- the reset step of next-step autoreset: the world init zs_reset performs (gym_env.py:148-164,
            // multiagent_env.py:173-184) instead of the transition; a new world's outputs.  (One env per warp: the branch is
            // warp-uniform.)
            if (p.fast_init) k = initialize_world_fast<MPC, G, CV>(p, e, true);
            else {
                k = initialize_world<MPC, G, false>(p, id_of(e), e.episode + 1, e.flags);
                scalars_from_smem<MPC, G, false>(p, e);
            }
            pend = false;
            life_now = is_agent ? (int)TL(lane) : 0;
            if (want_mask) alive_before = gballot<G, CV>(e, is_agent) >> P;
        } else {
            k = world_step_one<MPC, G, CV, ROS>(p, e, my_at, my_dx, my_dy);
            e.ep_steps += 1;
            if (step == io.n_steps - 1) TR(25);

            // ---- reward tracker update (reward.py:30-41, 77-92), float64 in the reference's operation order.
            // A tracker whose inputs did not change yields exactly +0.0.
            life_now = is_agent ? (int)TL(lane) : 0;
            if (lane_sum) {
                const int sum_prev = gadd<G, CV>(e, life_before), sum_new = gadd<G, CV>(e, life_now);
                if (sum_prev != sum_new || zd_before != e.zd) rew = __dsub_rn(total_reward(e.zd, sum_new), total_reward(zd_before, sum_prev));
            } else if (is_agent && (life_before != life_now || zd_before != e.zd)) {
                rew = __dsub_rn(total_reward(e.zd, life_now), total_reward(zd_before, life_before));
            }
            if (is_agent) PREVL(aidx) = (int16_t)life_now;
            e.prev_zd = e.zd;

            // ---- Game.spawn_zombies_to_maintain_minimum (game.py:196-201)
            if (!FAST && p.minimum_zombies > 0) {
                const int zc = __popc(gballot<G, CV>(e, lane >= NP && lane < p.M && (TM(lane < p.M ? lane : 0) & 0x80)));
                if (zc < p.minimum_zombies) {  // rare, and possibly only one env of the warp: the divergent flavour
                    k = spawn_zombies<MPC, G, false>(p, id_of(e), e.episode, (uint32_t)(e.t + 1), k, p.minimum_zombies - zc, e.nlive, false, false);
                    e.nlive = SCALW(ZS_S_STAMP_COUNTER);
                }
            }

            // ---- rules and end reward (gym_env.py:130-141, multiagent_env.py:143-162)
            rules_eval<MPC, G, CV, ROS>(p, e, ended, won, agents_alive);
        }
        bool done = false, trunc = false;
        double end_reward = 0.0;
        if (ended) { done = true; end_reward = won ? 10.0 : -10.0; }
        else if (!agents_alive) { trunc = true; end_reward = -10.0; }
        if (!per_agent) {
            if (done || trunc) rew = __dadd_rn(rew, end_reward);
            if ((FAST || io.reward) && (lane_sum ? lane == 0 : aidx == 0)) io.reward[sn] = rew;
            if (!FAST && io.agent_mask && is_agent) io.agent_mask[sn * A + aidx] = (alive_before >> aidx) & 1u;
        } else if (is_agent) {
            if (!((alive_before >> aidx) & 1u)) rew = 0.0;
            else if (life_now > 0) rew = __dadd_rn(rew, end_reward);
            if (io.reward) io.reward[sn * A + aidx] = rew;
            if (io.agent_mask) io.agent_mask[sn * A + aidx] = (alive_before >> aidx) & 1u;
        }
        if (p.max_steps > 0 && e.ep_steps >= p.max_steps) trunc = true;  // gymnasium TimeLimit
        if (lane == 0) {
            if (FAST || io.terminated) io.terminated[sn] = done;
            if (FAST || io.truncated) io.truncated[sn] = trunc;
            if (!FAST && io.draws) io.draws[sn] = k;
        }

        PH(9);
        if (step == io.n_steps - 1) TR(26);
        // ---- same-step auto-reset
        const bool need_init = (done || trunc) && auto_reset;
        if (wany<G, CV>(e, need_init)) {
            TRF(8);
            if (need_init && lane == 0) {
                atomicAdd(p.stats + 0, 1ull);
                if (done && won) atomicAdd(p.stats + 1, 1ull);
                atomicAdd(p.stats + 2, (unsigned long long)e.ep_steps);
                atomicAdd(p.stats + 3, (unsigned long long)e.zd);
            }
            // the terminal world, after the transition, the reward and the respawn: what zs_step writes without auto-reset
            // (gym_env.py:99-145).  The encoders are group-collective, so both envs of a warp write their row: the row of an
            // env that did not end is not flagged to the caller.
            if constexpr (FIN) encode_obs<MPC, G, CV, SURR>(p, e, io.final_obs + (obs_out - io.obs));
            if constexpr (NXT) pend = true;  // next-step autoreset: the world stays as it ended, its next step re-initialises it
            else if (R::on || p.fast_init) initialize_world_fast<MPC, G, CV, ROS>(p, e, need_init);  // both envs of the warp, converged
            else if (need_init) {  // possibly only one env of the warp: the divergent flavour
                initialize_world<MPC, G, false>(p, id_of(e), e.episode + 1, e.flags);
                scalars_from_smem<MPC, G, false>(p, e);
            }
        }
        PH(10);
        if (step == io.n_steps - 1) TR(27);
        bool compacted = false;
        if constexpr (!FAST && (world_obs || REC)) {
            // the observation as a compact record (include/zs_b200.h: zs_step_compact, zs_step_compact_agents), with the
            // reward(s) and flags in its header
            if (io.compact) {
                compacted = true;
                uint32_t* const rec = io.compact + (size_t)env * io.compact_words;
                uint32_t* const stage = reinterpret_cast<uint32_t*>(zs_smem + e.b);  // (EnvS::act: see obs_world_compact)
                int n_ent = 0;
                bool over;
                int hdr;
                if constexpr (world_obs) {
                    hdr = ZS_COMPACT_HEADER;
                    over = obs_world_compact<MPC, G, CV>(p, e, rec, io.compact_words - hdr, n_ent);
                    if (lane == 0) { stage[0] = (uint32_t)n_ent | (done ? 1u << 16 : 0u) | (trunc ? 1u << 17 : 0u) | (over ? 1u << 18 : 0u); stage[1] = 0u; }
                    if (lane_sum ? lane == 0 : aidx == 0) { stage[2] = (uint32_t)__double2loint(rew); stage[3] = (uint32_t)__double2hiint(rew); }
                } else {
                    hdr = ZS_AGENT_COMPACT_HEADER(A);
                    n_ent = obs_surroundings_compact<MPC, G, CV>(p, id_of(e), e.flags, rec, io.compact_words - hdr);
                    over = n_ent < 0;
                    if (over) n_ent = 0;
                    if (lane == 0) { stage[0] = (uint32_t)n_ent | (done ? 1u << 16 : 0u) | (trunc ? 1u << 17 : 0u) | (over ? 1u << 18 : 0u); stage[1] = alive_before; }
                    if (is_agent) {  // reward, window centre and life after the step (and after its auto-reset)
                        stage[2 + 2 * aidx] = (uint32_t)__double2loint(rew); stage[3 + 2 * aidx] = (uint32_t)__double2hiint(rew);
                        const uint32_t xy = TXY(lane);
                        stage[2 + 2 * A + aidx] = (uint32_t)(xy_y(xy) * p.W + xy_x(xy)) | ((uint32_t)(uint16_t)TL(lane) << 16);
                    }
                }
                compact_flush<MPC, G, CV>(e, rec, hdr + n_ent * (p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2));
                if (wany<G, CV>(e, over) && obs_out) {  // rare: the full row, for the caller to fetch
                    if constexpr (world_obs) {
                        obs_world_template<MPC, G, CV>(p, e, obs_out);
                        obs_world_patch<MPC, G, CV>(p, e, obs_out);
                    } else encode_surroundings<MPC, G, CV>(p, e, obs_out);
                }
                if (io.host_flags) compact_signal<G, CV>(p, io, e, env);
            }
        }
        if constexpr (PROD) {
            // hand the observation over: the mailbox is free again once the producer is done with the previous step's
            // record (long ago, normally), the record is filled, the group's lane 0 tells the producer
            if (step > 0) mbar_wait(&mail->empty, (uint32_t)((step - 1) & 1));
            const int cnt = obs_world_record<MPC, G, CV>(p, e, reinterpret_cast<uint32_t*>(mail + 1), p.prod_cap);
            if (lane == 0) { mail->count = cnt; mail->flags = e.flags; }
            gsync<G, CV>(e);
            if (lane == 0) mbar_arrive(&mail->full);
            // (the record could not describe the env: the producer reads the env's block itself, which must not change meanwhile)
            if (cnt < 0) mbar_wait(&mail->empty, (uint32_t)(step & 1));
        } else if (!compacted && (FAST || obs_out)) {
            if constexpr (world_obs) obs_world_patch<MPC, G, CV>(p, e, obs_out);
            else encode_surroundings<MPC, G, CV>(p, e, obs_out);
        }
        gsync<G, CV>(e);
        PH(11);
        if (step < 16) TR(4 + step);
        TR_STEP_END(step);
    }
    if constexpr (NXT) { if (lane == 0) io.pending[env] = pend; }
#ifdef ZS_PHASE_CLOCKS
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long tot = 0;
        for (int i = 0; i < 13; ++i) tot += zs_ph[i];  // (13.. are inside [10])
        printf("phase cycles/step over %d steps (total %.0f):", io.n_steps, (double)tot / io.n_steps);
        for (int i = 0; i < 24; ++i) { printf(" [%d] %.0f", i, (double)zs_ph[i] / io.n_steps); zs_ph[i] = 0; }
        printf("\n");
    }
#endif
}

// OCC = resident 4-warp CTAs per SM the kernel is compiled for.  A rollout keeps an env in its CTA for all K steps, so a
// batch runs in ceil(warps / resident warps) rounds: zs_create picks the OCC with the fewest rounds, and among those the
// one with the most registers — 4 (128 registers, nothing spilled or re-derived in the step loop: +10 % at 4,096 envs,
// which are latency-bound), 6 (80) or 7 (72); large batches are issue-bound and take 6 (two envs per warp) or 7.
// SHAPE: what is compiled in — 0 = world-scope observation, 1 = the standard rollout shape (FAST, world scope),
// 2 = surroundings observation.  (With both observation encoders in one kernel the step loop of the kernels that
// never run the window code spilled more registers: 5-8 % on large world-scope batches.)
// SHAPE 3 = the standard rollout shape with a producer warp: CTAs of four game warps (eight envs) plus one warp that writes
// the observations (160 threads; compiled for 4 CTAs per SM: 20 warps, five per scheduler = 96 registers, and 4,096 envs
// are one wave.  Three-warp CTAs at seven per SM would put six warps on one scheduler: 80 registers and spills).
// SHAPE 4 = surroundings observation with the per-agent compact record (zs_step_compact_agents / zs_step_host_agents; step
// launches of at most 32 slots only): a kernel of its own, since with the record compiled into SHAPE 2 that kernel spilled more
// and its device-output steps of config 3's game at 65,536 envs took 6 % longer (profiles/r04_ab_surroundings.txt).
// SHAPE 5 = world-scope observation with the compact record, more slots than lanes (zs_step_compact / zs_step_host; step
// launches of 128 and 256 slots only): a kernel of its own, so that the device-output general kernels stay as they are.
// SHAPE 6 / 7 = world-scope / surroundings observation with the final observation of every env the step re-initialises
// (zs_step_final / zs_rollout_final; step launches only): kernels of their own, so that the kernels without it stay as they
// are (the record of SHAPE 4 compiled into SHAPE 2 made it spill more and slowed config 3 by 6 %).
// SHAPE 8 / 9 / 10 / 11 = next-step autoreset (ZS_AUTORESET_NEXT_STEP handles, one env per warp; step launches only): the
// counterparts of SHAPE 0 (world scope, with its run-time compact-record branch), 2 (surroundings), 4 (surroundings with the
// per-agent record) and 5 (world scope with the record, more slots than lanes), so that the kernels of the other handles
// stay as they are.
// ROS: the game roster compiled into a standard-rollout-shape kernel (zs_world.cuh: Roster), 0 = read from ZsParams.
template <int MODE, int MPC, int G, int SHAPE, int OCC, int ROS = 0>
__global__ void __launch_bounds__(SHAPE == 3 ? 160 : ZS_WPC * 32, OCC) zs_sim_kernel(const __grid_constant__ ZsParams p, const __grid_constant__ ZsIO io) {
    ZS_CONSTS;
    constexpr bool PROD = SHAPE == 3;
    constexpr bool FAST = SHAPE == 1 || PROD, SURR = SHAPE == 2 || SHAPE == 4 || SHAPE == 7 || SHAPE == 9 || SHAPE == 10;
    constexpr bool FIN = SHAPE == 6 || SHAPE == 7;
    constexpr bool NXT = SHAPE >= 8;
    // the step kernel keeps both envs of a warp converged (zs_device.cuh); masked resets and encodes may not
    constexpr bool CV = MODE == MODE_STEP;
    constexpr int EPW = 32 / G;  // envs per warp
    const int wlane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    Env e;
    e.gl = wlane & (G - 1);
    e.gshift = wlane & ~(G - 1);
    e.gm = G == 32 ? 0xffffffffu : (0xffffu << e.gshift);
    const int slot = wid * EPW + (wlane / G);
#ifdef ZS_PHASE_CLOCKS
    e.ph_last = clock64();
#endif
    if (MODE == MODE_STEP) { TR(0); TR(31); }
    // (programmatic dependent launch, launch_sim: the next kernel of the stream may start scheduling its CTAs now; it
    // waits for this grid's completion in its own griddepcontrol.wait)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const int game_warps = (int)(blockDim.x >> 5) - (PROD ? 1 : 0);
    const int env = blockIdx.x * (game_warps * EPW) + slot;  // (a CTA has ZS_WPC warps, or fewer for small batches)
    unsigned long long* const tmpl_bar = reinterpret_cast<unsigned long long*>(zs_smem + p.tmpl_smem_off + (p.tmpl_pair ? 2 : 1) * p.tmpl_bytes);
    if (p.tmpl_smem_off >= 0) {
        // stage the pristine observation planes once per CTA, the source of the per-step TMA bulk copies: one thread
        // asks the TMA for them (global -> shared behind an mbarrier) and the launch goes on; whoever issues the first
        // observation copy waits for the barrier first
        if (threadIdx.x == 0) {
            mbar_init(tmpl_bar, 1);
            mbar_expect_tx(tmpl_bar, (uint32_t)((p.tmpl_pair ? 2 : 1) * p.tmpl_bytes));
            bulk_load(zs_smem + p.tmpl_smem_off, p.tmpl_obs, (uint32_t)p.tmpl_bytes, tmpl_bar);
            if (p.tmpl_pair) bulk_load(zs_smem + p.tmpl_smem_off + p.tmpl_bytes, p.tmpl_obs, (uint32_t)p.tmpl_bytes, tmpl_bar);
            if (PROD) {
                for (int i = 0; i < game_warps * EPW; ++i) {
                    ObsMail* m = reinterpret_cast<ObsMail*>(zs_smem + p.prod_off + i * ((int)sizeof(ObsMail) + 8 * p.prod_cap));
                    mbar_init(&m->full, 1); mbar_init(&m->empty, 1);
                }
            }
        }
        __syncthreads();  // (the barriers exist before anybody waits on them)
    }
    // everything below reads what earlier work of the stream wrote (state, images, actions, masks)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if constexpr (PROD) {
        if (wid == game_warps) {  // the producer warp
            uint32_t sa = (uint32_t)__cvta_generic_to_shared(zs_smem + p.tmpl_smem_off);
            if (wlane == 0) mbar_wait(tmpl_bar, 0u);
            __syncwarp();
            obs_producer<MPC>(p, io, game_warps * EPW, sa);
            return;
        }
    }
    if (env >= p.N) return;
    e.tmpl_saddr = 0;
    if (p.tmpl_smem_off >= 0) {
        const uint32_t a = (uint32_t)__cvta_generic_to_shared(zs_smem + p.tmpl_smem_off);
        asm volatile("mov.u32 %0, %1;" : "=r"(e.tmpl_saddr) : "r"(a));
    }
    PH(20);
    if (MODE == MODE_STEP) TR(1);
    e.b = (uint32_t)slot * (uint32_t)p.smem_per_env;
    e.env = env; e.env_global = p.env_base + (uint32_t)env;
    const int lane = e.gl;
    ZS_VIEWS;
    // the dead-body list is kept (instead of scanning the bitmap) when it lives on: in the parked image, or for a
    // launch of several steps
    const bool keep_lists = p.img != nullptr || (MODE == MODE_STEP && io.n_steps >= 4);

    if (MODE == MODE_RESET) {
        if (io.env_mask && !io.env_mask[env]) return;
        // slots keep their last position/life until re-placed; bring them in so the store is complete
        if (p.img_load) { load_image_issue<MPC, G, CV>(p, e); load_image_wait<MPC, G, CV>(p, e); }
        else load_state<MPC, G, CV>(p, e, false, true);
        if (!p.img) e.flags |= FL_DEAD_LAUNCH;
        const int k = initialize_world<MPC, G, false>(p, id_of(e), e.episode + 1, e.flags);
        scalars_from_smem<MPC, G, CV>(p, e);
        if (io.draws && lane == 0) io.draws[env] = k;
        if (io.obs) encode_obs<MPC, G, CV, SURR>(p, e, io.obs + (size_t)env * p.obs_elems);
        store_state<MPC, G, CV>(p, e);
        if (p.img) { store_image<MPC, G, CV>(p, e); image_store_drain(e); }
        return;
    }
    // a masked step (zs_step_masked: one lane group = one whole warp) leaves the other worlds exactly as they are
    if (MODE == MODE_STEP && io.env_mask && !io.env_mask[env]) return;
    if (p.img_load) {
        load_image_issue<MPC, G, CV>(p, e);
        load_image_wait<MPC, G, CV>(p, e);
        PH(21);
        if (MODE == MODE_STEP) { TR(2); TR(3); }
    } else {
        load_state<MPC, G, CV>(p, e, keep_lists);
        PH(21);
        if (MODE == MODE_STEP) TR(2);
        if (!keep_lists) e.flags |= FL_DEAD_LAUNCH;
        build_grid<MPC, G, false>(p, id_of(e), e.flags);
        PH(22);
        if (MODE == MODE_STEP) TR(3);
    }
    if (MODE == MODE_ENCODE) {
        encode_obs<MPC, G, CV, SURR>(p, e, io.obs + (size_t)env * p.obs_elems);
        return;
    }
    // the staged observation planes have landed before the first bulk copy out of them is issued
    if (p.tmpl_smem_off >= 0 && lane == 0) mbar_wait(tmpl_bar, 0u);
    if (MODE == MODE_STEP) TR(29);

#ifdef ZS_PHASE_CLOCKS
    e.ph_last = clock64();
#endif
    if constexpr (ONE) step_loop_one<MPC, G, CV, FAST, SURR, PROD, ROS, SHAPE == 4 || SHAPE == 10, FIN, NXT>(p, io, e);
    else step_loop_general<MPC, G, CV, SURR, SHAPE == 5 || SHAPE == 11, FIN, NXT>(p, io, e);
#ifdef ZS_PHASE_CLOCKS
    e.ph_last = clock64();
#endif
    if (p.img) store_image<MPC, G, CV>(p, e);
    store_state<MPC, G, CV>(p, e);
    if (p.img) image_store_drain(e);
    PH(23);
    TR(30);
}

__global__ void zs_init_static_life_kernel(const __grid_constant__ ZsParams p) {
    const size_t n = (size_t)p.N * p.Sp;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p.SLIFE[i] = __ldg(p.static_max + (i % p.Sp));
    // the next zs_reset is world initialisation #0 (what Game.__init__ does, game.py:138)
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (size_t)p.N; i += (size_t)gridDim.x * blockDim.x)
        p.SCAL[i * 8 + ZS_S_EPISODE] = -1;
}

// win_table (zs_obs.cuh: window_block): the pristine label (and life) planes of the window centred on every cell
__global__ void zs_build_window_table_kernel(const __grid_constant__ ZsParams p, int32_t* table) {
    const int ww = p.sw * p.sw;
    for (int cell = blockIdx.x; cell < p.cells; cell += gridDim.x) {
        const int y = cell / p.W, x = cell - y * p.W;
        for (int i = threadIdx.x; i < p.win_ints; i += blockDim.x) {
            const int pl = i / ww, k = i - pl * ww, r = k / p.sw, c = k - r * p.sw;
            table[(size_t)cell * p.win_pitch + i] = p.tmpl_pad[(size_t)pl * p.pad_plane + (y + r) * p.pad_w + x + c];
        }
    }
}

// actions [n_steps, N, A] of the synthetic action stream, steps step_index .. step_index + n_steps - 1
__global__ void zs_fill_actions_kernel(const __grid_constant__ ZsParams p, uint32_t step_index, int32_t n_steps, int32_t* actions) {
    const long long per = (long long)p.N * p.A, n = per * n_steps;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int step = (int)(i / per);
        const int r = (int)(i - step * per);
        const int env = r / p.A, a = r - env * p.A;
        actions[i] = synthetic_action(p, p.env_base + (uint32_t)env, step_index + (uint32_t)step, a);
    }
}

// next-step autoreset: the envs zs_reset re-initialises (env_mask NULL = all) have no reset step pending any more
__global__ void zs_clear_pending_kernel(uint8_t* pending, const uint8_t* env_mask, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (env_mask == nullptr || env_mask[i]) pending[i] = 0;
}

__global__ void zs_stats_kernel(unsigned long long* stats, int64_t* out, int reset) {
    const int i = threadIdx.x;
    if (i < 4) {
        out[i] = (int64_t)stats[i];
        if (reset) stats[i] = 0ull;
    }
}

// zs_step_host with ZS_HOST_GROUPS=0 (a diagnostic setting): runs behind the step kernel in the stream — that kernel's writes to
// host memory are complete and visible when this one starts — and tells the waiting host threads so.  The default is a flag
// raised by the step kernel itself (ZsIO::host_flags): 3-5 us earlier.
#define ZS_HOST_GROUPS_MAX 256
__global__ void zs_host_flag_kernel(volatile uint32_t* flag, uint32_t ticket) { *flag = ticket; }

// ================================================================ host side
static thread_local char g_err[512] = "";
static int fail(const char* fmt, const char* a = "") {
    snprintf(g_err, sizeof(g_err), fmt, a);
    return 1;
}
#define CU(call)                                                                  \
    do {                                                                          \
        cudaError_t _e = (call);                                                  \
        if (_e != cudaSuccess) {                                                  \
            snprintf(g_err, sizeof(g_err), "%s: %s", #call, cudaGetErrorString(_e)); \
            return 2;                                                             \
        }                                                                         \
    } while (0)

struct ZsHandle {
    int device;  // the CUDA device the handle was created on: every entry point runs there, whatever is current
    ZsConfig cfg;
    ZsLayout lay;
    ZsParams p;
    std::vector<void*> dev_allocs;
    int64_t launches;
    int64_t bound_bytes;
    int sm_count;
    // How a launch is cut into lane groups, CTAs and shared memory.  shape[0] serves fused rollouts; shape[1] the short
    // launches (single steps, resets, encodes).  They differ for small worlds in mid-sized batches: two envs per warp halve
    // the instructions of a long rollout, one env per warp gives a short launch the shorter critical path (fewer slow
    // paths per warp, no waiting for the partner env).  Both work on the same state and the same parked images.
    struct Shape {
        int lanes_per_env, warps_per_cta, envs_per_cta, smem_per_env, smem_bytes, occ;
        int tmpl_smem_off, tmpl_planes, tmpl_pair, tmpl_bytes;
        int prod_off, prod_cap, prod_smem_bytes;  // the producer-warp variant of the standard rollout shape (0 bytes = not available)
    } shape[2];
    int short_steps;       // launches of fewer steps than this take shape[1]
    int use_pdl;           // launch with programmatic stream serialization (launch_sim): 0 never, 1 always, 2 short step launches
    int compact_words;     // words per compact observation record, 0 = this configuration has no compact form
    int agent_compact_words;  // the same for the per-agent surroundings record (zs_step_compact_agents)
    int32_t* host_actions_dev = nullptr;  // zs_step_host: this step's actions on the device
    uint32_t host_ticket = 0;  // zs_step_host: the value that marks the current step's records as arrived
    volatile uint32_t* host_flag = nullptr;  // pinned, one cache line each: [0] zs_host_flag_kernel's, [1 + g] group g's (the step kernel's)
    int32_t* host_group_count = nullptr;     // device: envs of each group done in this step
    int host_groups = 0;
    int host_diff = -1;                      // zs_step_host's expansion: -1 timed and chosen by the handle, 0 restore ahead + write, 1 difference of the records (ZS_HOST_DIFF)
    struct HostTune { int mode = 0; bool exploring = true; int left = 32; int n[2] = {0, 0}; double last[2][16]; } host_tune;
    const void* host_records_checked = nullptr;
    double host_stats[5] = {0, 0, 0, 0, 0};  // zs_step_host: calls, and summed us from entry to: launched / previous cells restored / flag seen / return
    std::vector<int32_t> tmpl_obs_host;  // the pristine observation planes [obs_C][cells] (zs_expand_compact)
    std::vector<int32_t> pad_host;       // surroundings scope: the padded pristine planes p.tmpl_pad as int32 (zs_expand_compact_agents)
    int tmpl_single_step;  // launches of fewer than four steps stage the observation template for the TMA as well
    int roster;            // the game as a roster (zs_world.cuh: Roster) when the standard rollout kernel has it compiled in, else 0
    bool img_valid;  // the parked images (ZsParams::img) match the canonical state of every env
    uint8_t* pending = nullptr;  // next-step autoreset handles only: device uint8 [N], ZsIO::pending
};

// Makes the handle's device current for the duration of an entry point and puts the caller's back afterwards: the
// stream, the map tables, the kernels' function attributes and the state buffer all belong to that device.
struct DeviceGuard {
    int prev = -1, cur = -1;
    explicit DeviceGuard(const ZsHandle* h) {
        if (!h) return;
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; return; }
        cur = h->device;
        if (prev != cur) cudaSetDevice(cur);
    }
    ~DeviceGuard() { if (prev >= 0 && prev != cur) cudaSetDevice(prev); }
};

static int round_up(int v, int m) { return (v + m - 1) / m * m; }
// the compact record size that no env can overflow by count: every thing, every box/wall, every listed dead body
static int compact_max_words(const ZsParams& p) {
    const int wpe = p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2;
    const int entries = p.M + p.S + p.cells;  // (dead bodies: at most every cell; far more than ever occurs)
    const int cap = p.M + p.S + 64;
    return round_up(ZS_COMPACT_HEADER + wpe * (cap < entries ? cap : entries), 32);
}

extern "C" __attribute__((visibility("default"))) int zs_abi_version(void) { return ZS_ABI_VERSION; }
extern "C" __attribute__((visibility("default"))) int zs_set_device(int32_t device) {
    CU(cudaSetDevice(device));
    return 0;
}
extern "C" __attribute__((visibility("default"))) const char* zs_last_error(void) { return g_err; }

static int validate(const ZsConfig* cfg, const ZsMap* map) {
    if (!cfg || !map) return fail("null config or map");
    if (cfg->abi_version != ZS_ABI_VERSION) return fail("ABI version mismatch");
    if (cfg->num_envs < 1) return fail("num_envs must be >= 1");
    if (cfg->rules < 0 || cfg->rules > ZS_RULES_SAFEHOUSE) return fail("unknown rules id");
    if (cfg->n_bots < 0 || cfg->n_bots > ZS_MAX_BOTS) return fail("n_bots out of range");
    for (int i = 0; i < cfg->n_bots; ++i)
        if (cfg->bot_kinds[i] != ZS_KIND_TERMINATOR && cfg->bot_kinds[i] != ZS_KIND_SNIPER &&
            cfg->bot_kinds[i] != ZS_KIND_TROLL && cfg->bot_kinds[i] != ZS_KIND_HAMSTER &&
            cfg->bot_kinds[i] != ZS_KIND_RANDOMAN) return fail("unsupported bot kind");
    if (cfg->n_agents < 1 || cfg->n_agents > ZS_MAX_AGENTS) return fail("n_agents out of range");
    for (int i = 0; i < cfg->n_agents; ++i) {
        int w = cfg->agent_weapons[i];
        if (!(w == ZS_WEAPON_RANDOM || (w >= ZS_WEAPON_KNIFE && w <= ZS_WEAPON_SHOTGUN))) return fail("bad agent weapon code");
    }
    if (cfg->initial_zombies < 0 || cfg->minimum_zombies < 0) return fail("negative zombie count");
    int Z = cfg->initial_zombies > cfg->minimum_zombies ? cfg->initial_zombies : cfg->minimum_zombies;
    if (cfg->n_bots + cfg->n_agents + Z > ZS_MAX_SLOTS) return fail("too many things per env (ZS_MAX_SLOTS)");
    if (map->width < 1 || map->height < 1 || map->width > 2048 || map->height > 2048 ||
        (int64_t)map->width * map->height > 65535) return fail("map size out of range");
    if (map->n_statics < 0 || map->n_statics > 30000) return fail("too many statics");
    if (cfg->obs_scope == ZS_OBS_SURROUNDINGS) {
        if (cfg->surroundings_width <= 1 || cfg->surroundings_width % 2 == 0) return fail("surroundings width must be an odd number greater than 1");
    } else if (cfg->obs_scope != ZS_OBS_WORLD) return fail("bad obs_scope");
    if (cfg->obs_encoding != ZS_OBS_SIMPLE && cfg->obs_encoding != ZS_OBS_CHANNELS) return fail("bad obs_encoding");
    if (cfg->obs_per_agent && cfg->obs_scope != ZS_OBS_SURROUNDINGS) return fail("per-agent observations need the surroundings scope");
    if (cfg->rules == ZS_RULES_SAFEHOUSE && map->n_objectives == 0) return fail("Safe house game requires objectives defined.");
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_layout(const ZsConfig* cfg, const ZsMap* map, ZsLayout* out) {
    if (int rc = validate(cfg, map)) return rc;
    if (!out) return fail("null layout");
    memset(out, 0, sizeof(*out));
    const int64_t N = cfg->num_envs;
    const int Z = cfg->initial_zombies > cfg->minimum_zombies ? cfg->initial_zombies : cfg->minimum_zombies;
    out->n_slots = cfg->n_bots + cfg->n_agents + Z;
    out->slot_pitch = round_up(out->n_slots, 16);
    out->agent_pitch = round_up(cfg->n_agents, 8);
    out->static_pitch = round_up(map->n_statics > 0 ? map->n_statics : 1, 8);
    out->cells = map->width * map->height;
    out->dead_words = round_up((out->cells + 31) / 32, 4);
    const int elem[ZS_F_COUNT] = {2, 2, 2, 4, 1, 2, 2, 4, 4};
    const int pitch[ZS_F_COUNT] = {out->slot_pitch, out->slot_pitch, out->slot_pitch, out->slot_pitch, out->slot_pitch,
                                   out->agent_pitch, out->static_pitch, out->dead_words, 8};
    int64_t off = 0;
    for (int f = 0; f < ZS_F_COUNT; ++f) {
        out->offset[f] = off;
        out->row_bytes[f] = elem[f] * pitch[f];
        off += (int64_t)out->row_bytes[f] * N;
        off = (off + 255) / 256 * 256;
    }
    out->state_bytes = off;
    out->obs_channels = cfg->obs_encoding == ZS_OBS_CHANNELS ? 3 : 1;
    if (cfg->obs_scope == ZS_OBS_WORLD) { out->obs_height = map->height; out->obs_width = map->width; }
    else { out->obs_height = out->obs_width = cfg->surroundings_width; }
    out->obs_count = cfg->obs_per_agent ? cfg->n_agents : 1;
    out->obs_elems_per_env = (int64_t)out->obs_count * out->obs_channels * out->obs_height * out->obs_width;
    out->n_discrete_actions = cfg->obs_per_agent ? 7 : 6;
    return 0;
}

template <int MODE>
static void launch_sim(const ZsHandle* h, const ZsIO& io_in, cudaStream_t st) {
    ZsIO io = io_in;
    io.pending = h->pending;
    // staging the observation template for the TMA pays off when a launch runs several steps
    ZsParams pp = h->p;
    const ZsHandle::Shape& sh = h->shape[(MODE == MODE_STEP && io.n_steps >= h->short_steps && io.env_mask == nullptr) ? 0 : 1];
    pp.smem_per_env = sh.smem_per_env; pp.tmpl_smem_off = sh.tmpl_smem_off; pp.tmpl_planes = sh.tmpl_planes;
    pp.tmpl_pair = sh.tmpl_pair; pp.tmpl_bytes = sh.tmpl_bytes; pp.prod_off = -1; pp.prod_cap = 0;
    int smem = sh.smem_bytes;
    // envs in flight chip-wide, roughly: the distance load_state prefetches ahead (a launch of many short-lived CTAs)
    pp.prefetch_ahead = (MODE != MODE_STEP || io.n_steps < 4) && !getenv("ZS_NO_PREFETCH") ? h->sm_count * 7 * sh.envs_per_cta : 0;
    if (MODE != MODE_STEP || (io.n_steps < 4 && h->tmpl_single_step == 0)) {  // (and without the template a CTA more fits an SM)
        if (pp.tmpl_smem_off >= 0) smem = pp.tmpl_smem_off;
        pp.tmpl_smem_off = -1;
    }
    // start from the parked images when they are current; a launch that goes through every env leaves them current
    pp.img_load = pp.img != nullptr && h->img_valid;
    const dim3 grid((pp.N + sh.envs_per_cta - 1) / sh.envs_per_cta), block(sh.warps_per_cta * 32);
    // next-step autoreset handles step with the kernels that have it compiled in (zs_sim_kernel: SHAPE 8 to 11)
    const bool next_step = MODE == MODE_STEP && h->pending != nullptr;
    // the standard rollout shape gets the kernel with that shape compiled in (step_loop_one)
    const bool fast = MODE == MODE_STEP && pp.mpc <= 32 && pp.A == 1 && !pp.obs_per_agent && pp.minimum_zombies == 0 &&
                      pp.obs_scope == ZS_OBS_WORLD && io.actions && io.fmt == ZS_ACTIONS_DISCRETE && io.obs && io.reward &&
                      io.terminated && io.truncated && !io.draws && !io.agent_mask && !io.final_obs && !next_step;
    // ... and with the handle's game compiled in when it is an instantiated roster (only the bench game's, at 16 slots)
    const bool roster = fast && h->roster == ZS_ROSTER_BENCH && pp.mpc == 16;
    const int occ = MODE == MODE_STEP ? sh.occ : ZS_MIN_CTAS;
    const bool surr = pp.obs_scope == ZS_OBS_SURROUNDINGS;
    // the standard rollout shape of a batch that one wave of producer-warp CTAs holds: observations through a third warp
    const bool prod = fast && MODE == MODE_STEP && sh.prod_smem_bytes > 0 && pp.tmpl_smem_off >= 0 && io.env_mask == nullptr;
    // SH_: 0 world scope, 1 the standard rollout shape (step launches only), 2 surroundings, 4 surroundings with the per-agent
    // record, 5 world scope with the record and more slots than lanes, 6 / 7 world scope / surroundings with the final
    // observation, 8 to 11 next-step autoreset (one env per warp: compiled for G = 32 only) (4 to 11: step launches only)
    // (zs_sim_kernel: SHAPE)
    // Programmatic dependent launch: the kernel's CTAs may be scheduled while the previous kernel of the stream is still
    // draining (they stage the observation template and then wait in griddepcontrol.wait for that kernel to have
    // completed, all its writes visible) — the launch latency and the ramp hide under the predecessor's tail.
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = (size_t)smem; lc.stream = st;
    cudaLaunchAttribute la[1];
    la[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    la[0].val.programmaticStreamSerializationAllowed = 1;
    // (measured, profiles/r02_pdl.txt: back-to-back single steps 16.4 -> 14.5 us per launch, nothing lost on an idle stream; fused
    // rollouts lose 1-1.5 % — the early CTAs of the next launch sit on the SMs — so only short step launches ask for it)
    const bool pdl = h->use_pdl == 1 || (h->use_pdl == 2 && MODE == MODE_STEP && io.n_steps < h->short_steps);
    lc.attrs = la; lc.numAttrs = pdl ? 1 : 0;
#define ZS_LAUNCH_R(MPC_, G_, SH_, O_, R_) cudaLaunchKernelEx(&lc, zs_sim_kernel<MODE, MPC_, G_, MODE == MODE_STEP ? (SH_) : (SH_) == 1 || (SH_) == 5 || (SH_) == 6 || (SH_) == 8 || (SH_) == 11 ? 0 : (SH_) == 4 || (SH_) == 7 || (SH_) == 9 || (SH_) == 10 ? 2 : (SH_), MODE == MODE_STEP ? (O_) : ZS_MIN_CTAS, MODE == MODE_STEP ? (R_) : 0>, pp, io)
#define ZS_LAUNCH(MPC_, G_, SH_, O_) ZS_LAUNCH_R(MPC_, G_, SH_, O_, 0)
#define ZS_LAUNCH_F(MPC_, G_, O_) do { if (next_step && (G_) == 32) { if (surr && io.compact) ZS_LAUNCH(MPC_, G_, ((G_) == 32 ? 10 : 4), O_); \
                                                                      else if (surr) ZS_LAUNCH(MPC_, G_, ((G_) == 32 ? 9 : 2), O_); \
                                                                      else ZS_LAUNCH(MPC_, G_, ((G_) == 32 ? 8 : 0), O_); } \
                                       else if (roster) ZS_LAUNCH_R(MPC_, G_, 1, O_, (MPC_) == 16 ? ZS_ROSTER_BENCH : 0); else if (fast) ZS_LAUNCH(MPC_, G_, 1, O_); \
                                       else if (surr && io.compact) ZS_LAUNCH(MPC_, G_, 4, O_); else if (surr && io.final_obs) ZS_LAUNCH(MPC_, G_, 7, O_); \
                                       else if (surr) ZS_LAUNCH(MPC_, G_, 2, O_); else if (io.final_obs) ZS_LAUNCH(MPC_, G_, 6, O_); \
                                       else ZS_LAUNCH(MPC_, G_, 0, O_); } while (0)
#define ZS_LAUNCH_G(MPC_, G_, O_) do { if (next_step) { if (surr) ZS_LAUNCH(MPC_, G_, 9, O_); else if (io.compact) ZS_LAUNCH(MPC_, G_, 11, O_); \
                                                        else ZS_LAUNCH(MPC_, G_, 8, O_); } \
                                       else if (surr && io.final_obs) ZS_LAUNCH(MPC_, G_, 7, O_); else if (surr) ZS_LAUNCH(MPC_, G_, 2, O_); \
                                       else if (io.compact) ZS_LAUNCH(MPC_, G_, 5, O_); else if (io.final_obs) ZS_LAUNCH(MPC_, G_, 6, O_); \
                                       else ZS_LAUNCH(MPC_, G_, 0, O_); } while (0)
    if (prod) {
        pp.prod_off = sh.prod_off; pp.prod_cap = sh.prod_cap; pp.tmpl_smem_off = ZS_PROD_ENVS * sh.smem_per_env;
        lc.gridDim = dim3((pp.N + ZS_PROD_ENVS - 1) / ZS_PROD_ENVS); lc.blockDim = dim3(32 * (ZS_PROD_ENVS / 2 + 1));
        lc.dynamicSmemBytes = (size_t)sh.prod_smem_bytes;
        if constexpr (MODE == MODE_STEP) cudaLaunchKernelEx(&lc, zs_sim_kernel<MODE_STEP, 16, 16, 3, ZS_MIN_CTAS_LOWOCC>, pp, io);
        if (pp.img != nullptr) const_cast<ZsHandle*>(h)->img_valid = true;
        return;
    }
    switch (pp.mpc) {
        case 16:
            if (sh.lanes_per_env == 16) {
                if (occ == ZS_MIN_CTAS_LOWOCC) ZS_LAUNCH_F(16, 16, ZS_MIN_CTAS_LOWOCC);
                else if (occ == ZS_MIN_CTAS_G16) ZS_LAUNCH_F(16, 16, ZS_MIN_CTAS_G16);
                else ZS_LAUNCH_F(16, 16, ZS_MIN_CTAS);
            } else {
                if (occ == ZS_MIN_CTAS_LOWOCC) ZS_LAUNCH_F(16, 32, ZS_MIN_CTAS_LOWOCC); else ZS_LAUNCH_F(16, 32, ZS_MIN_CTAS);
            }
            break;
        case 32:
            if (occ == ZS_MIN_CTAS_LOWOCC) ZS_LAUNCH_F(32, 32, ZS_MIN_CTAS_LOWOCC); else ZS_LAUNCH_F(32, 32, ZS_MIN_CTAS);
            break;
        case 128: ZS_LAUNCH_G(128, 32, ZS_OCC_GENERAL); break;
        default: ZS_LAUNCH_G(256, 32, ZS_OCC_GENERAL); break;
    }
#undef ZS_LAUNCH_G
#undef ZS_LAUNCH_F
#undef ZS_LAUNCH
#undef ZS_LAUNCH_R
    if (pp.img != nullptr && (MODE == MODE_STEP || MODE == MODE_RESET) && io.env_mask == nullptr) const_cast<ZsHandle*>(h)->img_valid = true;
}
template <int MPC, int G, int OCC>
static cudaError_t set_smem_attr_step(int bytes) {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    cudaError_t e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, 0, OCC>, attr, bytes);
    if (e == cudaSuccess && MPC <= 32) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (MPC <= 32 ? 1 : 0), OCC>, attr, bytes);
    if (e == cudaSuccess && MPC == 16) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (MPC == 16 ? 1 : 0), OCC, (MPC == 16 ? ZS_ROSTER_BENCH : 0)>, attr, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, 2, OCC>, attr, bytes);
    if (e == cudaSuccess && MPC <= 32) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (MPC <= 32 ? 4 : 2), OCC>, attr, bytes);
    constexpr bool rec_g = MPC > 32 && OCC == ZS_OCC_GENERAL;  // (the only occupancy launch_sim runs them at)
    if (e == cudaSuccess && rec_g) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (rec_g ? 5 : 0), OCC>, attr, bytes);
    // the final-observation kernels: every occupancy launch_sim runs the world-scope and surroundings kernels at
    constexpr bool fin = MPC <= 32 || OCC == ZS_OCC_GENERAL;
    if (e == cudaSuccess && fin) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (fin ? 6 : 0), OCC>, attr, bytes);
    if (e == cudaSuccess && fin) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (fin ? 7 : 2), OCC>, attr, bytes);
    // the next-step autoreset kernels: one env per warp, at the same occupancies
    constexpr bool nxt = fin && G == 32;
    if (e == cudaSuccess && nxt) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (nxt ? 8 : 0), OCC>, attr, bytes);
    if (e == cudaSuccess && nxt) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (nxt ? 9 : 2), OCC>, attr, bytes);
    if (e == cudaSuccess && nxt) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, MPC, G, (!nxt ? 2 : MPC <= 32 ? 10 : 11), OCC>, attr, bytes);
    return e;
}
template <int MPC, int G>
static cudaError_t set_smem_attr_for(int bytes) {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    cudaError_t e = cudaSuccess;
    // only the occupancies launch_sim runs: the kernels with more slots than lanes step at ZS_OCC_GENERAL alone (compiling
    // them for the others too would leave step kernels in the library that nothing can launch)
    if constexpr (MPC <= 32) {
        e = set_smem_attr_step<MPC, G, ZS_MIN_CTAS>(bytes);
        if (e == cudaSuccess) e = set_smem_attr_step<MPC, G, ZS_MIN_CTAS_LOWOCC>(bytes);
    }
    if constexpr (G == 16) if (e == cudaSuccess) e = set_smem_attr_step<MPC, G, ZS_MIN_CTAS_G16>(bytes);
    if (e == cudaSuccess && G == 16 && MPC == 16) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_STEP, 16, 16, 3, ZS_MIN_CTAS_LOWOCC>, attr, bytes);
    if (e == cudaSuccess && MPC > 32) e = set_smem_attr_step<MPC, G, (MPC > 32 ? ZS_OCC_GENERAL : ZS_MIN_CTAS)>(bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_RESET, MPC, G, 0, ZS_MIN_CTAS>, attr, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_ENCODE, MPC, G, 0, ZS_MIN_CTAS>, attr, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_RESET, MPC, G, 2, ZS_MIN_CTAS>, attr, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(zs_sim_kernel<MODE_ENCODE, MPC, G, 2, ZS_MIN_CTAS>, attr, bytes);
    return e;
}
// resident warps per SM of the step kernel compiled for OCC CTAs, at this block size and shared-memory footprint
template <int MPC, int G, int OCC>
static int resident_warps_of(int block_threads, int smem) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, zs_sim_kernel<MODE_STEP, MPC, G, 0, OCC>, block_threads, smem) != cudaSuccess) n = 0;
    return n * (block_threads / 32);
}
static int resident_warps(int mpc, int lanes, int occ, int block_threads, int smem) {
    if (mpc == 16 && lanes == 16)
        return occ == ZS_MIN_CTAS_LOWOCC ? resident_warps_of<16, 16, ZS_MIN_CTAS_LOWOCC>(block_threads, smem)
             : occ == ZS_MIN_CTAS_G16 ? resident_warps_of<16, 16, ZS_MIN_CTAS_G16>(block_threads, smem)
                                      : resident_warps_of<16, 16, ZS_MIN_CTAS>(block_threads, smem);
    if (mpc == 16)
        return occ == ZS_MIN_CTAS_LOWOCC ? resident_warps_of<16, 32, ZS_MIN_CTAS_LOWOCC>(block_threads, smem)
                                         : resident_warps_of<16, 32, ZS_MIN_CTAS>(block_threads, smem);
    return occ == ZS_MIN_CTAS_LOWOCC ? resident_warps_of<32, 32, ZS_MIN_CTAS_LOWOCC>(block_threads, smem)
                                     : resident_warps_of<32, 32, ZS_MIN_CTAS>(block_threads, smem);
}
static int set_smem_attr(int mpc, int lanes, int bytes) {
    cudaError_t e;
    if (mpc == 16) e = lanes == 16 ? set_smem_attr_for<16, 16>(bytes) : set_smem_attr_for<16, 32>(bytes);
    else if (mpc == 32) e = set_smem_attr_for<32, 32>(bytes);
    else if (mpc == 128) e = set_smem_attr_for<128, 32>(bytes);
    else e = set_smem_attr_for<256, 32>(bytes);
    CU(e);
    return 0;
}

template <typename T>
static int upload(ZsHandle* h, const std::vector<T>& v, const T** out) {
    void* d = nullptr;
    size_t bytes = (v.size() ? v.size() : 1) * sizeof(T);
    bytes = (bytes + 15) / 16 * 16;
    CU(cudaMalloc(&d, bytes));
    h->dev_allocs.push_back(d);
    CU(cudaMemset(d, 0, bytes));
    if (v.size()) CU(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = (const T*)d;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_create(const ZsConfig* cfg, const ZsMap* map, ZsHandle** out) {
    if (!out) return fail("null out");
    *out = nullptr;
    ZsLayout lay;
    if (int rc = zs_layout(cfg, map, &lay)) return rc;
    int dev = 0;
    cudaDeviceProp prop;
    CU(cudaGetDevice(&dev));
    CU(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) return fail("this library is built for sm_100a (B200) only");
    ZsHandle* h = new ZsHandle();
    h->device = dev; h->cfg = *cfg; h->lay = lay; h->launches = 0; h->bound_bytes = 0; h->sm_count = prop.multiProcessorCount;
    ZsParams& p = h->p;
    memset(&p, 0, sizeof(p));
    p.N = cfg->num_envs; p.env_base = (uint32_t)cfg->env_index_base;
    p.key0 = (uint32_t)cfg->seed; p.key1 = (uint32_t)(cfg->seed >> 32);
    for (int r = 0; r < 10; ++r) { p.rkey0[r] = p.key0 + (uint32_t)r * 0x9E3779B9u; p.rkey1[r] = p.key1 + (uint32_t)r * 0xBB67AE85u; }
    p.rules = cfg->rules; p.P = cfg->n_bots; p.A = cfg->n_agents;
    p.Z = cfg->initial_zombies > cfg->minimum_zombies ? cfg->initial_zombies : cfg->minimum_zombies;
    p.M = lay.n_slots; p.Mp = lay.slot_pitch; p.Ap = lay.agent_pitch; p.S = map->n_statics; p.Sp = lay.static_pitch;
    p.W = map->width; p.H = map->height; p.cells = lay.cells; p.cells_pad = round_up(lay.cells, 16); p.dead_words = lay.dead_words;
    p.initial_zombies = cfg->initial_zombies; p.minimum_zombies = cfg->minimum_zombies;
    p.obs_scope = cfg->obs_scope; p.obs_enc = cfg->obs_encoding; p.sw = cfg->surroundings_width;
    p.obs_count = lay.obs_count; p.obs_C = lay.obs_channels; p.obs_per_agent = cfg->obs_per_agent;
    p.max_steps = cfg->max_episode_steps; p.auto_reset = cfg->auto_reset; p.n_discrete = lay.n_discrete_actions;
    p.n_ps = map->n_player_spawns; p.n_zs = map->n_zombie_spawns; p.obs_elems = lay.obs_elems_per_env;
    memcpy(p.agent_weapons, cfg->agent_weapons, sizeof(p.agent_weapons));
    memcpy(p.bot_kinds, cfg->bot_kinds, sizeof(p.bot_kinds));
    for (int i = 0; i < cfg->n_bots; ++i) if (cfg->bot_kinds[i] == ZS_KIND_RANDOMAN) p.has_randoman = 1;
    memcpy(p.agent_obs_ids, cfg->agent_obs_ids, sizeof(p.agent_obs_ids));

    // ---- map tables
    const int cells = p.cells, S = p.S;
    std::vector<int16_t> cell_static(cells, -1), static_max(p.Sp, 0);
    std::vector<uint16_t> static_cell(p.Sp, 0), ps(p.n_ps), zs(p.n_zs);
    std::vector<uint8_t> static_label(p.Sp, 0), tmpl_grid(p.cells_pad, 0);
    std::vector<int32_t> tmpl_obs(3 * (size_t)cells, 0);  // label (or simple value), life, weapon (zeros) planes
    std::vector<uint32_t> objective_bits(p.dead_words, 0);
    auto cell_of = [&](const int16_t* xy, int i, int* c) {
        int x = xy[2 * i], y = xy[2 * i + 1];
        if (x < 0 || x >= p.W || y < 0 || y >= p.H) return false;
        *c = y * p.W + x;
        return true;
    };
    int c = 0;
    for (int i = 0; i < map->n_objectives; ++i) {
        if (!cell_of(map->objective_xy, i, &c)) { delete h; return fail("objective outside the map"); }
        objective_bits[c >> 5] |= 1u << (c & 31);
        tmpl_obs[c] = cfg->obs_encoding == ZS_OBS_SIMPLE ? 256 * ZS_LABEL_OBJECTIVE : ZS_LABEL_OBJECTIVE;
    }
    for (int i = 0; i < S; ++i) {
        if (!cell_of(map->static_xy, i, &c)) { delete h; return fail("static thing outside the map"); }
        const int label = map->static_label[i];
        if (label != ZS_LABEL_BOX && label != ZS_LABEL_WALL) { delete h; return fail("static label must be box or wall"); }
        if (cell_static[c] >= 0) { delete h; return fail("two static things on one cell"); }
        const int mx = label == ZS_LABEL_BOX ? 10 : 200;
        cell_static[c] = (int16_t)i; static_cell[i] = (uint16_t)c; static_max[i] = (int16_t)mx; static_label[i] = (uint8_t)label;
        tmpl_grid[c] = G_STATIC;
        if (cfg->obs_encoding == ZS_OBS_SIMPLE) tmpl_obs[c] = 256 * label + (15 * (mx < 100 ? mx : 100)) / 100;
        else { tmpl_obs[c] = label; tmpl_obs[cells + c] = mx; }
    }
    for (int i = 0; i < p.n_ps; ++i) { if (!cell_of(map->player_spawn_xy, i, &c)) { delete h; return fail("spawn outside the map"); } ps[i] = (uint16_t)c; }
    for (int i = 0; i < p.n_zs; ++i) { if (!cell_of(map->zombie_spawn_xy, i, &c)) { delete h; return fail("spawn outside the map"); } zs[i] = (uint16_t)c; }
    int rc = 0;
    if (cfg->obs_scope == ZS_OBS_SURROUNDINGS) {
        // the planes the windows are cut from (zs_obs.cuh: window_plane): out-of-bounds cells are a fresh Wall
        const int sw = p.sw, half = sw >> 1, pw = p.W + sw - 1, ph = p.H + sw - 1;
        if (sw < 1 || sw * sw > 65535) { delete h; return fail("surroundings width out of range"); }
        const bool simple = cfg->obs_encoding == ZS_OBS_SIMPLE;
        std::vector<uint16_t> pad((size_t)(simple ? 1 : 2) * pw * ph);
        for (int y = 0; y < ph; ++y)
            for (int x = 0; x < pw; ++x) {
                const int mx = x - half, my = y - half;
                const bool inb = mx >= 0 && mx < p.W && my >= 0 && my < p.H;
                const size_t at = (size_t)y * pw + x;
                if (simple) pad[at] = (uint16_t)(inb ? tmpl_obs[my * p.W + mx] : 256 * ZS_LABEL_WALL + 15);
                else {
                    pad[at] = (uint16_t)(inb ? tmpl_obs[my * p.W + mx] : ZS_LABEL_WALL);
                    pad[(size_t)pw * ph + at] = (uint16_t)(inb ? tmpl_obs[cells + my * p.W + mx] : 200);
                }
            }
        p.pad_w = pw; p.pad_plane = pw * ph;
        p.sw_magic = (uint32_t)((0x100000000ull + (unsigned)sw - 1) / (unsigned)sw);
        rc |= upload(h, pad, &p.tmpl_pad);
        h->pad_host.assign(pad.begin(), pad.end());
        // one pristine window block per cell, as long as the table stays a small part of the L2
        p.win_ints = (simple ? 1 : 2) * sw * sw;
        p.win_pitch = round_up(p.win_ints, 32);
        const size_t table_bytes = (size_t)cells * p.win_pitch * sizeof(int32_t);
        if (!rc && table_bytes <= (32u << 20) && !getenv("ZS_NO_WINDOW_TABLE")) {
            void* d = nullptr;
            if (cudaMalloc(&d, table_bytes) != cudaSuccess) { zs_destroy(h); return fail("out of device memory (window table)"); }
            h->dev_allocs.push_back(d);
            zs_build_window_table_kernel<<<cells < 1024 ? cells : 1024, 256>>>(p, (int32_t*)d);
            if (cudaDeviceSynchronize() != cudaSuccess) { zs_destroy(h); return fail("window table build failed"); }
            p.win_table = (const int32_t*)d;
        }
    }
    rc |= upload(h, cell_static, &p.cell_static); rc |= upload(h, static_cell, &p.static_cell);
    rc |= upload(h, static_max, &p.static_max); rc |= upload(h, static_label, &p.static_label);
    rc |= upload(h, tmpl_grid, &p.tmpl_grid); rc |= upload(h, tmpl_obs, &p.tmpl_obs);
    h->tmpl_obs_host = tmpl_obs;
    rc |= upload(h, objective_bits, &p.objective_bits); rc |= upload(h, ps, &p.ps_cells); rc |= upload(h, zs, &p.zs_cells);
    if (p.n_ps == 0 || p.n_zs == 0) {  // some group may stand anywhere: the cells without a box/wall, x-major (core.py:44-46)
        std::vector<uint16_t> free_xm, free_index(cells, 0xffff);
        for (int x = 0; x < p.W; ++x)
            for (int y = 0; y < p.H; ++y) {
                const int cc = y * p.W + x;
                if (cell_static[cc] < 0) { free_index[cc] = (uint16_t)free_xm.size(); free_xm.push_back((uint16_t)cc); }
            }
        p.n_free0 = (int)free_xm.size();
        if (!getenv("ZS_NO_FREE_TABLE")) { rc |= upload(h, free_xm, &p.free_xm); rc |= upload(h, free_index, &p.free_index); }
    }
    std::vector<unsigned long long> zero(4, 0ull);
    const unsigned long long* st = nullptr;
    rc |= upload(h, zero, &st);
    p.stats = (unsigned long long*)st;
    if (rc) { zs_destroy(h); return rc; }

    // ---- shared memory per env: EnvS<MPC> (compile-time layout) + run-time sized tail (grid, dead bits, static lives, candidates)
    p.mpc = p.Mp <= 16 ? 16 : p.Mp <= 32 ? 32 : p.Mp <= 128 ? 128 : 256;
    const int struct_bytes = p.mpc == 16 ? (int)sizeof(EnvS<16>) : p.mpc == 32 ? (int)sizeof(EnvS<32>)
                           : p.mpc == 128 ? (int)sizeof(EnvS<128>) : (int)sizeof(EnvS<256>);
    int off = p.cells_pad;  // the grid starts right behind the struct
    auto take = [&](int bytes) { int o = off; off = round_up(off + bytes, 16); return o; };
    p.off_dead = take(p.dead_words * 4);
    // maps with many boxes/walls under the general kernels: their lives (touched by the odd hit only) stay in the state
    // buffer instead of costing resident CTAs (zs_device.cuh: SLP)
    p.sl_global = p.mpc > 32 && p.Sp > 512 && !getenv("ZS_NO_SL_GLOBAL");
    p.off_sl = take(p.sl_global ? 16 : p.Sp * 2);
    if (p.mpc > 32 && p.Sp > 512) {  // (only the general kernels look at spl_global)
        p.spl_pitch = p.Sp + (p.Sp + 3) / 4;  // Sp entries, then Sp index bytes
        void* d = nullptr;
        if (cudaMalloc(&d, (size_t)p.N * p.spl_pitch * sizeof(uint32_t)) != cudaSuccess) { zs_destroy(h); return fail("out of device memory (static patch lists)"); }
        h->dev_allocs.push_back(d);
        p.spl_global = (uint32_t*)d;
        p.off_spl = take(16); p.off_sidx = take(16);
    } else {
        p.off_spl = take(p.Sp * 4);
        p.off_sidx = take(p.Sp);
    }
    // (the spawn candidate list comes last: everything in front of it is the parked image, zs_device.cuh: EnvS)
    int cand = 1;
    if (p.P + p.A > 0) cand = p.n_ps > 0 ? p.n_ps : cells;
    if (p.Z > 0) { int zc = p.n_zs > 0 ? p.n_zs : cells; if (zc > cand) cand = zc; }
    // the lean world init (initialize_world_lists): one lane per slot, spawn cells for everybody, fixed weapons
    p.fast_init = p.Mp <= 32 && p.n_ps >= p.P + p.A && p.n_ps > 0 && p.n_zs > 0 && p.n_zs >= p.initial_zombies &&
                  p.n_ps + p.n_zs <= 256 && p.initial_zombies > 0;
    for (int i = 0; i < p.P; ++i) if (p.bot_kinds[i] != ZS_KIND_TERMINATOR && p.bot_kinds[i] != ZS_KIND_SNIPER) p.fast_init = 0;
    for (int i = 0; i < p.A; ++i) if (p.agent_weapons[i] == ZS_WEAPON_RANDOM) p.fast_init = 0;
    if (getenv("ZS_NO_FAST_INIT")) p.fast_init = 0;
    // the game as a roster (launch_sim: the standard rollout kernel with it compiled in); ZS_NO_ROSTER keeps the kernel that
    // reads the game from the parameters (the reference the roster kernels are tested against)
    bool all_terminators = true;
    for (int i = 0; i < p.P; ++i) all_terminators &= p.bot_kinds[i] == ZS_KIND_TERMINATOR;
    h->roster = p.fast_init && p.A == 1 && all_terminators && !getenv("ZS_NO_ROSTER") ? zs_roster(p.rules, p.P + p.A) : 0;
    if (p.fast_init) {
        cand = p.n_ps + p.n_zs;  // both index lists side by side
    }
    p.cand_cap = cand;
    // the candidate list is only touched while things are being placed: long ones (a map without spawn cells offers every
    // cell) live in device memory, so they do not cost resident CTAs
    if (cand > 256) {
        void* d = nullptr;
        if (cudaMalloc(&d, (size_t)p.N * cand * sizeof(uint16_t)) != cudaSuccess) { zs_destroy(h); return fail("out of device memory (spawn candidate lists)"); }
        h->dev_allocs.push_back(d);
        p.cand_global = (uint16_t*)d;
        p.off_cand = take(16);
    } else p.off_cand = take(cand * 2);
    p.smem_per_env = round_up(struct_bytes + off, 16);
    // the parked images: kept when all of them together stay a modest part of the L2 (a launch then starts with one bulk
    // copy per env out of the L2 instead of re-deriving ranks, grid and lists; larger batches hide that latency behind
    // their other CTAs and would pay for the extra bytes in HBM bandwidth)
    {
        const int img_off_bytes = p.mpc == 16 ? img_off<16>() : p.mpc == 32 ? img_off<32>() : p.mpc == 128 ? img_off<128>() : img_off<256>();
        p.img_bytes = struct_bytes - img_off_bytes + p.off_cand;
        p.img_pitch = round_up(p.img_bytes, 128);
        long long budget = 64ll << 20;
        if (const char* force = getenv("ZS_IMAGE_MB")) budget = (long long)atoll(force) << 20;
        if ((long long)p.N * p.img_pitch <= budget) {
            void* d = nullptr;
            if (cudaMalloc(&d, (size_t)p.N * p.img_pitch) != cudaSuccess) { zs_destroy(h); return fail("out of device memory (parked images)"); }
            h->dev_allocs.push_back(d);
            p.img = (unsigned char*)d;
        }
        h->img_valid = false;
    }
    // lanes per env: a half warp (two envs per warp, in lock-step) when an env has at most 16 slots, the env count is
    // even and the batch is large enough that the halved instruction count matters more than the few extra cycles a
    // two-env warp needs per step (measured cross-over: about 16 envs per SM)
    int lanes0 = (p.mpc == 16 && p.N % 2 == 0 && p.N > prop.multiProcessorCount * 16) ? 16 : 32;
    // ... for fused rollouts.  A short launch of such a batch runs one env per warp as long as all its warps are resident
    // at once (measured at 4,096 bridge envs: a single step takes 16.6 us with one env per warp, 21.8 us with two; from
    // about eight fused steps on two envs per warp win)
    int lanes1 = lanes0;
    if (lanes0 == 16 && p.N <= prop.multiProcessorCount * 28 && !getenv("ZS_ONE_SHAPE")) lanes1 = 32;
    if (const char* force = getenv("ZS_LANES_PER_ENV")) {
        const int v = atoi(force);
        if ((v == 16 && p.mpc == 16 && p.N % 2 == 0) || v == 32) lanes0 = lanes1 = v;
    }
    // next-step autoreset: an env's reset step skips the transition its partner in a two-env warp would run, which the step
    // loop's converged primitives cannot do per half warp: one env per warp in every launch
    if (cfg->auto_reset == ZS_AUTORESET_NEXT_STEP) {
        lanes0 = lanes1 = 32;
        void* d = nullptr;
        if (cudaMalloc(&d, (size_t)p.N) != cudaSuccess) { zs_destroy(h); return fail("out of device memory (autoreset marks)"); }
        h->dev_allocs.push_back(d);
        if (cudaMemset(d, 0, (size_t)p.N) != cudaSuccess) { zs_destroy(h); return fail("autoreset marks: cudaMemset failed"); }
        h->pending = (uint8_t*)d;
    }
    h->short_steps = 8;
    h->use_pdl = 2;  // programmatic dependent launch: 2 = short step launches only (launch_sim), ZS_PDL=1 every launch, ZS_PDL=0 none
    if (const char* force = getenv("ZS_PDL")) h->use_pdl = atoi(force) ? 1 : 0;
    if (const char* force = getenv("ZS_SHORT_STEPS")) h->short_steps = atoi(force);
    h->tmpl_single_step = getenv("ZS_NO_TMA_SINGLE") ? 0 : 1;
    // header + 92 entries; with more slots than lanes, room for every slot on top (config 4's maze game: 224 / 416 words).  The
    // caller grows them.
    h->compact_words = 0;
    if (p.obs_scope == ZS_OBS_WORLD && !p.obs_per_agent) {
        const int wpe = p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2;
        h->compact_words = p.mpc <= 32 ? (wpe == 1 ? 96 : 192) : std::min(round_up(ZS_COMPACT_HEADER + wpe * (p.M + 92), 32), compact_max_words(p));
    }
    // (the entry count and the window centres are 16-bit fields: fewer than 65,536 cells is what zs_layout accepts)
    h->agent_compact_words = (p.mpc <= 32 && p.obs_scope == ZS_OBS_SURROUNDINGS && p.obs_per_agent)
                                 ? round_up(ZS_AGENT_COMPACT_HEADER(p.A) + (p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2) * 92, 32) : 0;
    const int smem_per_env_base = p.smem_per_env;
    for (int si = 0; si < 2; ++si) {
        ZsHandle::Shape& sh = h->shape[si];
        if (si == 1 && lanes1 == lanes0) { sh = h->shape[0]; break; }
        sh.lanes_per_env = si == 0 ? lanes0 : lanes1;
        sh.smem_per_env = smem_per_env_base;
        // two envs per warp: the halves touch the same fields of neighbouring env blocks with the same instruction, so the
        // blocks are placed half a bank row apart (an odd multiple of 64 bytes): 16 lanes x 4 bytes of one env and of the
        // other then fall on different banks.  (Swept on the bridge map, ZS_SMEM_SKEW = 0 .. 112: no measurable difference
        // either way — the step is bound by dependent latency, not by shared-memory wavefronts; it fixes the layout so that
        // a change of sizeof(EnvS) cannot move the two halves onto the same banks.)
        if (sh.lanes_per_env == 16) {
            int skew = 64;
            if (const char* force = getenv("ZS_SMEM_SKEW")) skew = atoi(force) & 0x70;
            while ((sh.smem_per_env & 127) != skew) sh.smem_per_env += 16;
        }
        // warps per CTA: ZS_WPC, or 2 when the batch is small enough that 4-warp CTAs would spread unevenly over the SMs
        // (a small batch is latency-bound: the most loaded SM sets the pace)
        const int epw = 32 / sh.lanes_per_env;
        sh.warps_per_cta = ZS_WPC;
        if ((p.N + ZS_WPC * epw - 1) / (ZS_WPC * epw) < prop.multiProcessorCount * 5) sh.warps_per_cta = 2;
        if (const char* force = getenv("ZS_WARPS_PER_CTA")) { const int v = atoi(force); if (v == 1 || v == 2 || v == 4) sh.warps_per_cta = v; }
        // large maps: narrower CTAs (4 -> 2 -> 1 warps) when the envs of the chosen one do not fit in a CTA's shared memory
        while (sh.warps_per_cta > 1 && (long long)sh.smem_per_env * sh.warps_per_cta * epw > (long long)prop.sharedMemPerBlockOptin)
            sh.warps_per_cta >>= 1;
        sh.envs_per_cta = sh.warps_per_cta * epw;
        sh.smem_bytes = sh.smem_per_env * sh.envs_per_cta;
        sh.tmpl_smem_off = -1; sh.tmpl_planes = 0; sh.tmpl_pair = 0; sh.tmpl_bytes = 0;
        if (p.obs_scope == ZS_OBS_WORLD && (p.cells & 3) == 0) {
            const int planes = p.obs_enc == ZS_OBS_CHANNELS ? 3 : 1;
            int bytes = planes * p.cells * 4;
            // two envs per warp: ONE bulk copy can serve both envs of a warp (their rows are neighbours) from planes staged
            // twice back to back.  Off by default since the staging itself became an asynchronous bulk copy: measured
            // slightly behind one copy per env (ZS_TMA_PAIR=1 turns it on)
            const bool pair = sh.lanes_per_env == 16 && getenv("ZS_TMA_PAIR") && !getenv("ZS_NO_TMA_PAIR") &&
                              p.N / 2 <= prop.multiProcessorCount * ZS_MIN_CTAS_LOWOCC * ZS_WPC &&
                              (sh.smem_bytes + 2 * bytes + 1024) * (16 / sh.warps_per_cta) <= (int)prop.sharedMemPerMultiprocessor;
            if (pair) bytes *= 2;
            // keep at least 6 CTAs per SM resident (2-warp CTAs are only chosen for batches that need no more)
            if ((sh.smem_bytes + bytes + 1024) * 6 <= (int)prop.sharedMemPerMultiprocessor && !getenv("ZS_NO_TMA")) {
                sh.tmpl_smem_off = sh.smem_bytes; sh.tmpl_planes = planes; sh.tmpl_pair = pair; sh.tmpl_bytes = planes * p.cells * 4;
                sh.smem_bytes += bytes + 16;  // (+ the mbarrier of the staging copy)
            }
        }
        // the producer-warp variant (four game warps + one producer per CTA, 4 CTAs per SM): for two-env warps whose whole
        // batch is one wave of such CTAs, with the TMA template; one record of every thing, every box/wall and every listed
        // dead body per env
        sh.prod_off = -1; sh.prod_cap = 0; sh.prod_smem_bytes = 0;
        // OFF by default (ZS_PRODUCER=1): measured at 4,096 bridge envs it is SLOWER — 7.8 us per fused step with a producer
        // that issues the rows as bulk copies, 8.1 us with 128-bit stores, 9.2 us with a producer that polls its envs one by
        // one, against 5.6 us with the game warps writing their own observations (and 4.9 us with no observation at all).
        // More resident warps slow every warp on the SM down (the same shows with 4-warp CTAs): the step is bound by how
        // its dependent chain interleaves with the other warps' chains, not by the observation's own instructions.
        if (sh.lanes_per_env == 16 && p.mpc == 16 && sh.tmpl_smem_off >= 0 && !sh.tmpl_pair && getenv("ZS_PRODUCER") &&
            (p.N + ZS_PROD_ENVS - 1) / ZS_PROD_ENVS <= 4 * prop.multiProcessorCount) {
            const int cap = round_up(p.M + p.S + ZS_DEAD_CAP, 8);
            const int off = round_up(ZS_PROD_ENVS * sh.smem_per_env + sh.tmpl_bytes + 16, 16);
            const int total = off + ZS_PROD_ENVS * ((int)sizeof(ObsMail) + 8 * cap);
            if ((total + 1024) * 4 <= (int)prop.sharedMemPerMultiprocessor) { sh.prod_off = off; sh.prod_cap = cap; sh.prod_smem_bytes = total; }
        }
        if (sh.smem_bytes > (int)prop.sharedMemPerBlockOptin) { zs_destroy(h); return fail("map/thing count needs more shared memory than one CTA has"); }
        // (the attribute belongs to the kernel, not to the handle: every handle asks for all a CTA can have, so that handles
        // of different maps can live side by side)
        if (int rc2 = set_smem_attr(p.mpc, sh.lanes_per_env, (int)prop.sharedMemPerBlockOptin)) { zs_destroy(h); return rc2; }
        // resident CTAs per SM the step kernel is compiled for (zs_sim_kernel: OCC): fewest rounds first, then most
        // registers; batches of three rounds or more are issue-bound and take the occupancy
        sh.occ = ZS_MIN_CTAS;
        if (p.mpc <= 32) {
            const long long warps = ((long long)p.N + epw - 1) / epw;
            const int cands16[3] = {ZS_MIN_CTAS_LOWOCC, ZS_MIN_CTAS_G16, ZS_MIN_CTAS}, cands32[2] = {ZS_MIN_CTAS_LOWOCC, ZS_MIN_CTAS};
            const int* cands = sh.lanes_per_env == 16 ? cands16 : cands32;
            const int nc = sh.lanes_per_env == 16 ? 3 : 2;
            long long rounds[3], best = 0;
            for (int i = 0; i < nc; ++i) {
                long long cap = (long long)resident_warps(p.mpc, sh.lanes_per_env, cands[i], sh.warps_per_cta * 32, sh.smem_bytes) * prop.multiProcessorCount;
                if (cap < 1) cap = 1;
                rounds[i] = (warps + cap - 1) / cap;
                if (i == 0 || rounds[i] < best) best = rounds[i];
            }
            if (best >= 3) sh.occ = sh.lanes_per_env == 16 ? ZS_MIN_CTAS_G16 : ZS_MIN_CTAS;
            else for (int i = 0; i < nc; ++i) if (rounds[i] == best) { sh.occ = cands[i]; break; }
            if (const char* force = getenv("ZS_OCC")) {
                const int v = atoi(force);
                if (v == ZS_MIN_CTAS_LOWOCC || v == ZS_MIN_CTAS || (v == ZS_MIN_CTAS_G16 && sh.lanes_per_env == 16)) sh.occ = v;
            }
        }
    }
    p.smem_per_env = h->shape[0].smem_per_env;

    *out = h;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_destroy(ZsHandle* h) {
    if (!h) return 0;
    DeviceGuard guard(h);
    cudaDeviceSynchronize();
    for (void* d : h->dev_allocs) cudaFree(d);
    if (h->host_flag) cudaFreeHost((void*)h->host_flag);
    delete h;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_bind_state(ZsHandle* h, void* state_dev, int64_t bytes) {
    if (!h) return fail("null handle");
    if (!state_dev || bytes < h->lay.state_bytes) return fail("state buffer too small");
    if (((uintptr_t)state_dev & 15) != 0) return fail("state buffer must be 16-byte aligned");
    unsigned char* b = (unsigned char*)state_dev;
    ZsParams& p = h->p;
    p.X = (int16_t*)(b + h->lay.offset[ZS_F_X]); p.Y = (int16_t*)(b + h->lay.offset[ZS_F_Y]);
    p.LIFE = (int16_t*)(b + h->lay.offset[ZS_F_LIFE]); p.STAMP = (int32_t*)(b + h->lay.offset[ZS_F_STAMP]);
    p.META = (uint8_t*)(b + h->lay.offset[ZS_F_META]); p.PREV = (int16_t*)(b + h->lay.offset[ZS_F_PREV_LIFE]);
    p.SLIFE = (int16_t*)(b + h->lay.offset[ZS_F_STATIC_LIFE]); p.DEAD = (uint32_t*)(b + h->lay.offset[ZS_F_DEAD_BODY]);
    p.SCAL = (int32_t*)(b + h->lay.offset[ZS_F_SCALARS]);
    h->bound_bytes = bytes;
    h->img_valid = false;
    if (h->pending) {  // (a new state: no env has a reset step pending)
        DeviceGuard guard(h);
        CU(cudaMemset(h->pending, 0, (size_t)p.N));
    }
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_state_written(ZsHandle* h) {
    if (!h) return fail("null handle");
    h->img_valid = false;
    return 0;
}

static int check_bound(ZsHandle* h) {
    if (!h) return fail("null handle");
    if (!h->bound_bytes) return fail("no state buffer bound (zs_bind_state)");
    return 0;
}
static int launched(ZsHandle* h) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "kernel launch: %s", cudaGetErrorString(e)); return 2; }
    h->launches++;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_init_static_life(ZsHandle* h, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    h->img_valid = false;
    if (h->pending) CU(cudaMemsetAsync(h->pending, 0, (size_t)h->p.N, (cudaStream_t)stream));
    zs_init_static_life_kernel<<<h->sm_count * 4, 256, 0, (cudaStream_t)stream>>>(h->p);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int zs_reset(ZsHandle* h, const uint8_t* env_mask_dev, int32_t* obs_dev, int32_t* draws_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.env_mask = env_mask_dev; io.obs = obs_dev; io.obs_slots = 1; io.draws = draws_dev;
    launch_sim<MODE_RESET>(h, io, (cudaStream_t)stream);
    if (h->pending) {
        if (int rc = launched(h)) return rc;
        zs_clear_pending_kernel<<<(h->p.N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(h->pending, env_mask_dev, h->p.N);
    }
    return launched(h);
}

// zs_step and zs_step_final
static int step_launch(ZsHandle* h, const char* who, const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev,
                       int32_t* final_obs_dev, double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                       uint8_t* agent_mask_dev, int32_t* draws_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (!actions_dev) return fail("%s needs an action tensor", who);
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = 1; io.reward = reward_dev;
    io.terminated = terminated_dev; io.truncated = truncated_dev; io.agent_mask = agent_mask_dev; io.draws = draws_dev;
    io.final_obs = final_obs_dev;
    io.n_steps = 1;
    launch_sim<MODE_STEP>(h, io, (cudaStream_t)stream);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int zs_step(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev, double* reward_dev,
                       uint8_t* terminated_dev, uint8_t* truncated_dev, uint8_t* agent_mask_dev, int32_t* draws_dev, void* stream) {
    return step_launch(h, "zs_step", actions_dev, action_format, obs_dev, nullptr, reward_dev, terminated_dev, truncated_dev,
                       agent_mask_dev, draws_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int zs_step_final(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev,
                                                                     int32_t* final_obs_dev, double* reward_dev, uint8_t* terminated_dev,
                                                                     uint8_t* truncated_dev, uint8_t* agent_mask_dev, int32_t* draws_dev,
                                                                     void* stream) {
    if (int rc = check_bound(h)) return rc;
    if (!h->p.auto_reset) return fail("zs_step_final needs a handle with auto_reset = 1: without it no step re-initialises an env");
    if (h->pending) return fail("zs_step_final needs a handle with auto_reset = 1: under next-step autoreset the observation of the step that ends an episode already is its final observation");
    if (!obs_dev || !final_obs_dev) return fail("zs_step_final needs an observation and a final observation tensor");
    return step_launch(h, "zs_step_final", actions_dev, action_format, obs_dev, final_obs_dev, reward_dev, terminated_dev,
                       truncated_dev, agent_mask_dev, draws_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int zs_step_masked(ZsHandle* h, const uint8_t* env_mask_dev, const int32_t* actions_dev, int32_t action_format,
                                                                      int32_t* obs_dev, double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                                                                      uint8_t* agent_mask_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (!actions_dev) return fail("zs_step_masked needs an action tensor");
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    if (env_mask_dev && h->shape[1].lanes_per_env != 32)
        return fail("masked steps need one warp per env: this handle packs two envs per warp in every launch (very large batches "
                    "of at most 16 things per env, or ZS_LANES_PER_ENV=16)");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = 1; io.reward = reward_dev;
    io.terminated = terminated_dev; io.truncated = truncated_dev; io.agent_mask = agent_mask_dev; io.env_mask = env_mask_dev;
    io.n_steps = 1;
    launch_sim<MODE_STEP>(h, io, (cudaStream_t)stream);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int32_t zs_compact_words(const ZsHandle* h) { return h ? h->compact_words : 0; }
extern "C" __attribute__((visibility("default"))) int32_t zs_compact_max_words(const ZsHandle* h) {
    return h && h->compact_words ? compact_max_words(h->p) : 0;
}

extern "C" __attribute__((visibility("default"))) int zs_step_compact(ZsHandle* h, const int32_t* actions_dev, int32_t action_format, uint32_t* compact_dev,
                                                                       int32_t compact_words, int32_t* obs_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (!h->compact_words) return fail("this configuration has no compact observation form (world scope, one reward per env)");
    if (!actions_dev || !compact_dev) return fail("zs_step_compact needs an action tensor and a record buffer");
    if (compact_words < ZS_COMPACT_HEADER + 8 || compact_words > 65535) return fail("compact_words out of range");
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = 1;
    io.compact = compact_dev; io.compact_words = compact_words;
    io.n_steps = 1;
    launch_sim<MODE_STEP>(h, io, (cudaStream_t)stream);
    return launched(h);
}

static int host_threads(int n_threads, int N) {
    if (n_threads <= 0) {
        cpu_set_t set;
        n_threads = sched_getaffinity(0, sizeof(set), &set) == 0 ? CPU_COUNT(&set) : 1;
    }
    return n_threads > N ? N : n_threads;
}

// HOST code: one env's record -> its row of the observation tensor, reward and flags.  Returns true when the record could not
// hold the env (overflow bit): the caller copies that row from the device.
struct ExpandCtx {
    const int32_t* T;  // the pristine observation planes [C][cells]
    int cells, C, wpe, words;
    bool first_call;
    int32_t* obs; double* reward; uint8_t* terminated; uint8_t* truncated;
};
// The two halves of an env's expansion.  expand_restore needs the PREVIOUS record only: the cells it patched go back to the
// pristine value (the whole row when there is no usable previous record) — zs_step_host runs it while the device is still
// working on the step.  expand_write applies the new record.
static inline void expand_restore(const ExpandCtx& cx, int e, const uint32_t* pv) {
    const int cells = cx.cells, C = cx.C, wpe = cx.wpe;
    const int32_t* T = cx.T;
    const size_t row = (size_t)C * cells;
    int32_t* o = cx.obs + (size_t)e * row;
    if (cx.first_call || ((pv[0] >> 18) & 1u)) { memcpy(o, T, row * sizeof(int32_t)); return; }
    const int pn = (int)(pv[0] & 0xffffu);
    for (int i = 0; i < pn; ++i) {
        const int cell = (int)(pv[ZS_COMPACT_HEADER + i * wpe] & 0xffffu);
        for (int c = 0; c < C; ++c) o[(size_t)c * cells + cell] = T[(size_t)c * cells + cell];
    }
}
static inline bool expand_write(const ExpandCtx& cx, int e, const uint32_t* r, uint32_t* pv) {
    const int cells = cx.cells, wpe = cx.wpe;
    int32_t* o = cx.obs + (size_t)e * cx.C * cells;
    const uint32_t h0 = r[0];
    const int n = (int)(h0 & 0xffffu);
    if (cx.terminated) cx.terminated[e] = (uint8_t)((h0 >> 16) & 1u);
    if (cx.truncated) cx.truncated[e] = (uint8_t)((h0 >> 17) & 1u);
    if (cx.reward) memcpy(cx.reward + e, r + 2, sizeof(double));
    if ((h0 >> 18) & 1u) { pv[0] = h0; return true; }  // the record could not hold this env: the caller copies its row from the device
    if (wpe == 1) {
        for (int i = 0; i < n; ++i) { const uint32_t w = r[ZS_COMPACT_HEADER + i]; o[w & 0xffffu] = (int32_t)(int16_t)(w >> 16); }
    } else {
        for (int i = 0; i < n; ++i) {
            const uint32_t w0 = r[ZS_COMPACT_HEADER + 2 * i], w1 = r[ZS_COMPACT_HEADER + 2 * i + 1];
            const int cell = (int)(w0 & 0xffffu);
            o[cell] = (int32_t)(int16_t)(w0 >> 16);
            o[(size_t)cells + cell] = (int32_t)(int16_t)(w1 & 0xffffu);
            o[2 * (size_t)cells + cell] = (int32_t)(w1 >> 16);
        }
    }
    memcpy(pv, r, (size_t)(ZS_COMPACT_HEADER + n * wpe) * sizeof(uint32_t));
    return false;
}
// One env's expansion as a DIFFERENCE of its two records: only the cells whose entry changed are touched.  For a host that
// is bound by memory traffic (several ranks' observation rows do not fit its caches, so every scattered store is a DRAM line
// fill and write-back) this is a third of the lines of restore + write; where the rows are cache-resident the comparisons
// cost what the stores save, and restoring ahead of the flag (expand_restore) is the better half.
// Records of equal length are compared position by position, others up to their first difference (entries keep their list
// order: boxes/walls, dead bodies, mobile things).  Untouched entries keep their cells because a record names a cell once —
// except a cell with several dead bodies, whose equal entries come and go together, so that an untouched one always has a
// twin among the rewritten ones (new dead bodies only append; the list empties only with the world).
static inline bool expand_diff(const ExpandCtx& cx, int e, const uint32_t* r, uint32_t* pv) {
    const uint32_t h0 = r[0];
    if (cx.first_call || ((pv[0] >> 18) & 1u) || ((h0 >> 18) & 1u)) {  // no usable previous record / the row comes from the device
        if (!((h0 >> 18) & 1u)) expand_restore(cx, e, pv);
        return expand_write(cx, e, r, pv);
    }
    const int cells = cx.cells, C = cx.C, wpe = cx.wpe;
    const int32_t* T = cx.T;
    int32_t* o = cx.obs + (size_t)e * C * cells;
    const int n = (int)(h0 & 0xffffu), pn = (int)(pv[0] & 0xffffu);
    if (cx.terminated) cx.terminated[e] = (uint8_t)((h0 >> 16) & 1u);
    if (cx.truncated) cx.truncated[e] = (uint8_t)((h0 >> 17) & 1u);
    if (cx.reward) memcpy(cx.reward + e, r + 2, sizeof(double));
    const uint32_t* re = r + ZS_COMPACT_HEADER;
    uint32_t* pe = pv + ZS_COMPACT_HEADER;
    auto same = [&](int i) { return wpe == 1 ? pe[i] == re[i] : (pe[2 * i] == re[2 * i] && pe[2 * i + 1] == re[2 * i + 1]); };
    auto restore = [&](int i) {
        const int cell = (int)(pe[i * wpe] & 0xffffu);
        for (int c = 0; c < C; ++c) o[(size_t)c * cells + cell] = T[(size_t)c * cells + cell];
    };
    auto write = [&](int i) {
        if (wpe == 1) { const uint32_t w = re[i]; o[w & 0xffffu] = (int32_t)(int16_t)(w >> 16); }
        else {
            const uint32_t w0 = re[2 * i], w1 = re[2 * i + 1];
            const int cell = (int)(w0 & 0xffffu);
            o[cell] = (int32_t)(int16_t)(w0 >> 16);
            o[(size_t)cells + cell] = (int32_t)(int16_t)(w1 & 0xffffu);
            o[2 * (size_t)cells + cell] = (int32_t)(w1 >> 16);
        }
    };
    if (n == pn) {
        for (int i = 0; i < n; ++i) if (!same(i)) restore(i);
        for (int i = 0; i < n; ++i) if (!same(i)) { write(i); for (int w = 0; w < wpe; ++w) pe[i * wpe + w] = re[i * wpe + w]; }
    } else {
        const int m = n < pn ? n : pn;
        int k = 0;
        while (k < m && same(k)) ++k;
        for (int i = k; i < pn; ++i) restore(i);
        for (int i = k; i < n; ++i) write(i);
        memcpy(pe + k * wpe, re + k * wpe, (size_t)(n - k) * wpe * sizeof(uint32_t));
    }
    pv[0] = h0; pv[1] = r[1]; pv[2] = r[2]; pv[3] = r[3];
    return false;
}
static inline bool expand_one(const ExpandCtx& cx, int e, const uint32_t* r, uint32_t* pv) {
    if (!((r[0] >> 18) & 1u)) expand_restore(cx, e, pv);
    return expand_write(cx, e, r, pv);
}

// every env's record through expand(e, record, prev) on n_threads host threads; returns the number of envs whose record
// overflowed, their indices in overflow_envs_host
template <class Expand>
static int expand_records(int N, int n_threads, int words, const uint32_t* compact_host, uint32_t* prev_host,
                          int32_t* overflow_envs_host, const Expand& expand) {
    n_threads = host_threads(n_threads, N);
    int n_over = 0;
#pragma omp parallel for num_threads(n_threads) schedule(static)
    for (int e = 0; e < N; ++e) {
        if (expand(e, compact_host + (size_t)e * words, prev_host + (size_t)e * words)) {
            int at;
#pragma omp atomic capture
            at = n_over++;
            overflow_envs_host[at] = e;
        }
    }
    return n_over;
}

// HOST code: records -> the reference's observation tensor (include/zs_b200.h).  Incremental: the cells the previous
// record of an env patched go back to the pristine value, the new record's cells are written; a full row is only
// rewritten on the first call and after an overflow.
extern "C" __attribute__((visibility("default"))) int zs_expand_compact(const ZsHandle* h, const uint32_t* compact_host, uint32_t* prev_host, int32_t* obs_host,
                                                                         double* reward_host, uint8_t* terminated_host, uint8_t* truncated_host,
                                                                         int32_t* overflow_envs_host, int32_t* n_overflow, int32_t compact_words,
                                                                         int32_t first_call, int32_t n_threads) {
    if (!h) return fail("null handle");
    if (!h->compact_words) return fail("this configuration has no compact observation form");
    if (!compact_host || !prev_host || !obs_host || !overflow_envs_host || !n_overflow) return fail("null argument");
    if (compact_words < ZS_COMPACT_HEADER + 8) return fail("compact_words out of range");
    const int N = h->p.N, words = compact_words, cells = h->p.cells, C = h->p.obs_C;
    const bool simple = h->p.obs_enc == ZS_OBS_SIMPLE;
    const ExpandCtx cx{h->tmpl_obs_host.data(), cells, C, simple ? 1 : 2, words, first_call != 0, obs_host, reward_host, terminated_host,
                       truncated_host};
    *n_overflow = expand_records(N, n_threads, words, compact_host, prev_host, overflow_envs_host,
                                 [&](int e, const uint32_t* r, uint32_t* pv) { return expand_one(cx, e, r, pv); });
    return 0;
}

// One transition with HOST buffers (include/zs_b200.h): the actions go over with the copy engine, the kernel writes the
// pinned record buffer itself (coalesced rows staged in shared memory) and whoever completes the batch raises a flag in
// pinned memory behind ONE system-scope fence; the host threads are already spinning on that flag inside their parallel
// region and expand the records the moment it shows.  No device-to-host copy, no stream synchronisation, no thread
// wake-up on the way.  What was measured on the way here (profiles/r02_e2e_host_step.txt): a fence + ticket per warp, so
// that envs could be expanded as they arrive, costs 8-34 us per warp with 4,096 warps fencing at once; a flag per group
// of envs does not arrive earlier than the last one either (a system-scope fence waits for the whole burst to drain), so
// one group is the default (ZS_HOST_GROUPS).
// The transport of zs_step_host and zs_step_host_agents: `ahead(e)` (when use_ahead) runs for every env while the device works
// on the step, `expand(e, record, prev)` after the flag; it returns true when the env's record overflowed.  *us_total: the
// microseconds from entry to return.
template <class Ahead, class Expand>
static int host_step_run(ZsHandle* h, const int32_t* actions_host, int32_t action_format, uint32_t* compact_pinned,
                         uint32_t* prev_host, int32_t compact_words, int32_t* obs_dev, int32_t* overflow_envs_host,
                         int32_t* n_overflow, int32_t n_threads, void* stream, bool use_ahead, const Ahead& ahead,
                         const Expand& expand, double* us_total) {
    struct timespec ts0;
    clock_gettime(CLOCK_MONOTONIC, &ts0);
    auto us_since = [&ts0]() {
        struct timespec t;
        clock_gettime(CLOCK_MONOTONIC, &t);
        return (double)(t.tv_sec - ts0.tv_sec) * 1e6 + (double)(t.tv_nsec - ts0.tv_nsec) * 1e-3;
    };
    if (compact_pinned != h->host_records_checked) {  // the device must reach the record buffer in place (checked once per buffer)
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, compact_pinned) != cudaSuccess || (at.type != cudaMemoryTypeHost && at.type != cudaMemoryTypeManaged)) {
            cudaGetLastError();
            return fail("zs_step_host needs the records in pinned (page-locked) host memory");
        }
        h->host_records_checked = compact_pinned;
    }
    const cudaStream_t st = (cudaStream_t)stream;
    // the actions go over with the copy engine: 4,096 warps each reading its own word of host memory in place is 4,096 PCIe
    // read round trips
    const size_t act_bytes = (size_t)h->p.N * h->p.A * (action_format == ZS_ACTIONS_FULL ? 3 : 1) * sizeof(int32_t);
    if (!h->host_actions_dev) {
        void* d = nullptr;
        if (cudaMalloc(&d, (size_t)h->p.N * h->p.A * 3 * sizeof(int32_t)) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory (action buffer)"); }
        h->dev_allocs.push_back(d);
        h->host_actions_dev = (int32_t*)d;
        CU(cudaHostAlloc((void**)&h->host_flag, 64 * (ZS_HOST_GROUPS_MAX + 1), cudaHostAllocMapped | cudaHostAllocPortable));
        memset((void*)h->host_flag, 0, 64 * (ZS_HOST_GROUPS_MAX + 1));
        if (cudaMalloc(&d, ZS_HOST_GROUPS_MAX * sizeof(int32_t)) != cudaSuccess) { cudaGetLastError(); return fail("out of device memory (group counters)"); }
        h->dev_allocs.push_back(d);
        h->host_group_count = (int32_t*)d;
        CU(cudaMemsetAsync(d, 0, ZS_HOST_GROUPS_MAX * sizeof(int32_t), st));
        const char* force = getenv("ZS_HOST_GROUPS");
        h->host_groups = force ? atoi(force) : 1;
        if (h->host_groups > ZS_HOST_GROUPS_MAX) h->host_groups = ZS_HOST_GROUPS_MAX;
        if (h->host_groups > h->p.N) h->host_groups = h->p.N;
    }
    CU(cudaMemcpyAsync(h->host_actions_dev, actions_host, act_bytes, cudaMemcpyHostToDevice, st));
    const int N = h->p.N, words = compact_words;
    uint32_t ticket = ++h->host_ticket;
    if (ticket == 0) ticket = ++h->host_ticket;
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = h->host_actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = 1;
    io.compact = compact_pinned; io.compact_words = compact_words;
    io.n_steps = 1;
    const int groups = h->host_groups;  // 0: one flag for everything, raised by a kernel behind the step kernel
    const int group_envs = groups > 0 ? (N + groups - 1) / groups : N;
    if (groups > 0) { io.host_flags = (uint32_t*)h->host_flag + 16; io.group_count = h->host_group_count; io.group_envs = group_envs; io.ticket = ticket; }
    launch_sim<MODE_STEP>(h, io, st);
    if (groups <= 0) { zs_host_flag_kernel<<<1, 1, 0, st>>>(h->host_flag, ticket); h->launches++; }
    if (int rc = launched(h)) return rc;
    const double us_launched = us_since();
    double us_flag = 0, us_restored = 0;
    n_threads = host_threads(n_threads, N);
    int n_over = 0, gave_up = 0;
    const volatile uint32_t* const flags = h->host_flag;
    const int n_flags = groups > 0 ? (N + group_envs - 1) / group_envs : 1;
#pragma omp parallel num_threads(n_threads)
    {
        // every thread waits for the flags itself (nobody has to be woken when one shows) and expands its share of each
        // group as the group arrives, while the records of later groups are still on their way
        // (shares cut by hand: a thread that gave up must not leave the others stuck in a work-sharing construct)
        const int nt = omp_get_num_threads(), tid = omp_get_thread_num();
        // while the device works on the step: what the previous records patched goes back to the pristine layer (half of an
        // expansion's stores need nothing from the new records)
        if (use_ahead)
        for (int g = 0; g < n_flags; ++g) {
            const int g0 = g * group_envs, gn = (g0 + group_envs < N ? g0 + group_envs : N) - g0;
            const int e0 = g0 + (int)((long long)gn * tid / nt), e1 = g0 + (int)((long long)gn * (tid + 1) / nt);
            for (int e = e0; e < e1; ++e) ahead(e);
        }
        if (tid == 0) us_restored = us_since();
        struct timespec t0;
        clock_gettime(CLOCK_MONOTONIC, &t0);
        for (int g = 0; g < n_flags; ++g) {
            const volatile uint32_t* const flag = flags + (groups > 0 ? 16 * (g + 1) : 0);
            for (unsigned spins = 1; *flag != ticket; ++spins) {
                __builtin_ia32_pause();
                if ((spins & 0xfffffu) == 0) {  // a launch that died never delivers: give up after ten seconds
                    struct timespec t1;
                    clock_gettime(CLOCK_MONOTONIC, &t1);
                    if (t1.tv_sec - t0.tv_sec > 10) break;
                }
            }
            __atomic_thread_fence(__ATOMIC_ACQUIRE);
            if (*flag != ticket) {
#pragma omp atomic write
                gave_up = 1;
                break;
            }
            if (tid == 0 && g == 0) us_flag = us_since();
            const int g0 = g * group_envs, gn = (g0 + group_envs < N ? g0 + group_envs : N) - g0;
            const int e0 = g0 + (int)((long long)gn * tid / nt), e1 = g0 + (int)((long long)gn * (tid + 1) / nt);
            for (int e = e0; e < e1; ++e) {
                if (expand(e, compact_pinned + (size_t)e * words, prev_host + (size_t)e * words)) {
                    int at;
#pragma omp atomic capture
                    at = n_over++;
                    overflow_envs_host[at] = e;
                }
            }
        }
    }
    *n_overflow = n_over;
    if (gave_up) {
        const cudaError_t err = cudaStreamSynchronize(st);
        return err != cudaSuccess ? fail("zs_step_host: %s", cudaGetErrorString(err)) : fail("zs_step_host: the records did not arrive");
    }
    // rows of overflowing envs: obs_dev is complete when the launch is (the caller reads them next)
    if (n_over > 0) CU(cudaStreamSynchronize(st));
    *us_total = us_since();
    h->host_stats[0] += 1; h->host_stats[1] += us_launched; h->host_stats[2] += us_restored; h->host_stats[3] += us_flag; h->host_stats[4] += *us_total;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_step_host(ZsHandle* h, const int32_t* actions_host, int32_t action_format,
                                                                    uint32_t* compact_pinned, uint32_t* prev_host, int32_t compact_words,
                                                                    int32_t* obs_dev, int32_t* obs_host, double* reward_host,
                                                                    uint8_t* terminated_host, uint8_t* truncated_host,
                                                                    int32_t* overflow_envs_host, int32_t* n_overflow, int32_t first_call,
                                                                    int32_t n_threads, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (!h->compact_words) return fail("this configuration has no compact observation form (world scope, one reward per env)");
    if (!actions_host || !compact_pinned || !prev_host || !obs_host || !overflow_envs_host || !n_overflow) return fail("null argument");
    if (compact_words < ZS_COMPACT_HEADER + 8 || compact_words > 65535) return fail("compact_words out of range");
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    const ExpandCtx cx{h->tmpl_obs_host.data(), h->p.cells, h->p.obs_C, h->p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2, compact_words, first_call != 0,
                       obs_host, reward_host, terminated_host, truncated_host};
    // restore ahead + write, or every env as the difference of its two records after the flag (expand_diff).
    // Which of the two is faster depends on the host (its caches, how many ranks share it, the threads this rank got): the
    // handle times both — 32 calls alternating between them, then the faster one for 512 calls, then the next sample.
    // (Both leave the same rows and the same previous records, so the choice never shows in a result.)
    if (!h->host_actions_dev) { if (const char* v = getenv("ZS_HOST_DIFF")) h->host_diff = atoi(v) != 0; }  // (read on the first call)
    bool diff = h->host_diff != 0;
    if (h->host_diff < 0) {
        // a sample is 32 calls that ALTERNATE between the two (the records grow over the first steps of a batch: sixteen calls of
        // one and then sixteen of the other would compare different work); the medians decide (one hiccup of the host must not
        // decide 512 calls)
        ZsHandle::HostTune& t = h->host_tune;
        if (t.left <= 0) {
            if (t.exploring) {
                double med[2];
                for (int m = 0; m < 2; ++m) {
                    const int n = t.n[m] < 16 ? t.n[m] : 16;
                    std::sort(t.last[m], t.last[m] + n);
                    med[m] = n ? t.last[m][n / 2] : 1e30;
                }
                t.mode = med[1] < med[0] ? 1 : 0; t.exploring = false; t.left = 512;
            } else { t.exploring = true; t.left = 32; }
            t.n[0] = t.n[1] = 0;
        }
        if (t.exploring) t.mode = t.left & 1;
        diff = t.mode != 0;
    }
    double us_total = 0;
    const int rc = host_step_run(h, actions_host, action_format, compact_pinned, prev_host, compact_words, obs_dev, overflow_envs_host,
                                 n_overflow, n_threads, stream, !diff, [&](int e) { expand_restore(cx, e, prev_host + (size_t)e * compact_words); },
                                 [&](int e, const uint32_t* r, uint32_t* pv) { return diff ? expand_diff(cx, e, r, pv) : expand_write(cx, e, r, pv); },
                                 &us_total);
    if (rc) return rc;
    if (h->host_diff < 0) {
        ZsHandle::HostTune& t = h->host_tune;
        if (t.exploring && !first_call && *n_overflow == 0 && t.left <= 28) { t.last[t.mode][t.n[t.mode] & 15] = us_total; t.n[t.mode] += 1; }  // (the first four settle the caches)
        t.left -= 1;
    }
    return 0;
}

// ---------------------------------------------------------------- per-agent surroundings records (include/zs_b200.h)
extern "C" __attribute__((visibility("default"))) int32_t zs_agent_compact_words(const ZsHandle* h) { return h ? h->agent_compact_words : 0; }
// the record size that no env can overflow by count: every thing, every box/wall, every listed dead body
extern "C" __attribute__((visibility("default"))) int32_t zs_agent_compact_max_words(const ZsHandle* h) {
    if (!h || !h->agent_compact_words) return 0;
    const int wpe = h->p.obs_enc == ZS_OBS_SIMPLE ? 1 : 2;
    const int entries = h->p.M + h->p.S + h->p.cells;
    const int cap = h->p.M + h->p.S + 64;
    return round_up(ZS_AGENT_COMPACT_HEADER(h->p.A) + wpe * (cap < entries ? cap : entries), 32);
}
static int check_agent_words(const ZsHandle* h, int32_t compact_words) {
    if (!h->agent_compact_words)
        return fail("this configuration has no per-agent compact observation form (surroundings scope, one observation per agent, "
                    "at most 32 slots)");
    if (compact_words < ZS_AGENT_COMPACT_HEADER(h->p.A) + 8 || compact_words > 65535) return fail("compact_words out of range");
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_step_compact_agents(ZsHandle* h, const int32_t* actions_dev, int32_t action_format,
                                                                              uint32_t* compact_dev, int32_t compact_words, int32_t* obs_dev,
                                                                              void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (int rc = check_agent_words(h, compact_words)) return rc;
    if (!actions_dev || !compact_dev) return fail("zs_step_compact_agents needs an action tensor and a record buffer");
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = 1;
    io.compact = compact_dev; io.compact_words = compact_words;
    io.n_steps = 1;
    launch_sim<MODE_STEP>(h, io, (cudaStream_t)stream);
    return launched(h);
}

// HOST code: one env's agent record -> its A windows, rewards, flags, mask and lives.  Returns true on overflow (the caller
// copies the env's rows from the device).
struct AgentExpandCtx {
    const int32_t* T;  // the padded pristine planes [Cp][ph][pw] (Cp = 1 simple, 2 channels: label, life; weapons are 0)
    int pw, plane, W, w, half, C, Cp, A, hdr, wpe;
    bool first_call;
    int32_t* obs; double* reward; uint8_t* terminated; uint8_t* truncated; uint8_t* mask; int16_t* life;
};
static inline bool expand_agents(const AgentExpandCtx& cx, int e, const uint32_t* r, uint32_t* pv) {
    const int A = cx.A, w = cx.w, ww = w * w, half = cx.half, W = cx.W, wpe = cx.wpe;
    const uint32_t h0 = r[0];
    const int n = (int)(h0 & 0xffffu);
    if (cx.terminated) cx.terminated[e] = (uint8_t)((h0 >> 16) & 1u);
    if (cx.truncated) cx.truncated[e] = (uint8_t)((h0 >> 17) & 1u);
    for (int a = 0; a < A; ++a) {
        if (cx.reward) memcpy(cx.reward + (size_t)e * A + a, r + 2 + 2 * a, sizeof(double));
        if (cx.mask) cx.mask[(size_t)e * A + a] = (uint8_t)((r[1] >> a) & 1u);
        if (cx.life) cx.life[(size_t)e * A + a] = (int16_t)(r[2 + 2 * A + a] >> 16);
    }
    if ((h0 >> 18) & 1u) { pv[0] = h0; return true; }  // the record could not hold this env: the caller copies its rows from the device
    const bool prev_ok = !cx.first_call && !((pv[0] >> 18) & 1u);
    const int pn = prev_ok ? (int)(pv[0] & 0xffffu) : 0;
    int32_t* const o = cx.obs + (size_t)e * A * cx.C * ww;
    auto pristine = [&](int32_t* oa, int idx, int x, int y) {  // cell (x, y) of the map at index idx of window oa
        for (int pl = 0; pl < cx.Cp; ++pl) oa[pl * ww + idx] = cx.T[(size_t)pl * cx.plane + (size_t)(y + half) * cx.pw + x + half];
        if (cx.C == 3) oa[2 * ww + idx] = 0;
    };
    for (int a = 0; a < A; ++a) {
        const int c = (int)(r[2 + 2 * A + a] & 0xffffu), cy = c / W, cx0 = c - cy * W;
        int32_t* const oa = o + (size_t)a * cx.C * ww;
        if (!prev_ok || (pv[2 + 2 * A + a] & 0xffffu) != (uint32_t)c) {  // a new window: its rows from the padded planes
            for (int pl = 0; pl < cx.Cp; ++pl)
                for (int y = 0; y < w; ++y) memcpy(oa + pl * ww + y * w, cx.T + (size_t)pl * cx.plane + (size_t)(cy + y) * cx.pw + cx0, w * sizeof(int32_t));
            if (cx.C == 3) memset(oa + 2 * ww, 0, ww * sizeof(int32_t));
            continue;
        }
        // the same window: the cells the previous record patched in it go back to the pristine layer (the previous record
        // holds every patched cell this window showed)
        for (int i = 0; i < pn; ++i) {
            const int cell = (int)(pv[cx.hdr + i * wpe] & 0xffffu), y = cell / W, x = cell - y * W;
            const int wx = x - (cx0 - half), wy = y - (cy - half);
            if ((unsigned)wx < (unsigned)w && (unsigned)wy < (unsigned)w) pristine(oa, wy * w + wx, x, y);
        }
    }
    for (int i = 0; i < n; ++i) {
        const uint32_t w0 = r[cx.hdr + i * wpe], w1 = wpe == 2 ? r[cx.hdr + 2 * i + 1] : 0u;
        const int cell = (int)(w0 & 0xffffu), y = cell / W, x = cell - y * W;
        for (int a = 0; a < A; ++a) {
            const int c = (int)(r[2 + 2 * A + a] & 0xffffu), cy = c / W, cx0 = c - cy * W;
            const int wx = x - (cx0 - half), wy = y - (cy - half);
            if ((unsigned)wx >= (unsigned)w || (unsigned)wy >= (unsigned)w) continue;
            int32_t* const oa = o + (size_t)a * cx.C * ww;
            const int idx = wy * w + wx;
            oa[idx] = (int32_t)(int16_t)(w0 >> 16);
            if (wpe == 2) { oa[ww + idx] = (int32_t)(int16_t)(w1 & 0xffffu); oa[2 * ww + idx] = (int32_t)(w1 >> 16); }
        }
    }
    memcpy(pv, r, (size_t)(cx.hdr + n * wpe) * sizeof(uint32_t));
    return false;
}
static AgentExpandCtx agent_ctx(const ZsHandle* h, int32_t first_call, int32_t* obs_host, double* reward_host, uint8_t* terminated_host,
                                uint8_t* truncated_host, uint8_t* agent_mask_host, int16_t* agent_life_host) {
    const ZsParams& p = h->p;
    const bool simple = p.obs_enc == ZS_OBS_SIMPLE;
    return AgentExpandCtx{h->pad_host.data(), p.pad_w, p.pad_plane, p.W, p.sw, p.sw >> 1, p.obs_C, simple ? 1 : 2, p.A,
                          ZS_AGENT_COMPACT_HEADER(p.A), simple ? 1 : 2, first_call != 0, obs_host, reward_host, terminated_host,
                          truncated_host, agent_mask_host, agent_life_host};
}

extern "C" __attribute__((visibility("default"))) int zs_expand_compact_agents(const ZsHandle* h, const uint32_t* compact_host, uint32_t* prev_host,
                                                                                int32_t* obs_host, double* reward_host, uint8_t* terminated_host,
                                                                                uint8_t* truncated_host, uint8_t* agent_mask_host,
                                                                                int16_t* agent_life_host, int32_t* overflow_envs_host,
                                                                                int32_t* n_overflow, int32_t compact_words, int32_t first_call,
                                                                                int32_t n_threads) {
    if (!h) return fail("null handle");
    if (int rc = check_agent_words(h, compact_words)) return rc;
    if (!compact_host || !prev_host || !obs_host || !overflow_envs_host || !n_overflow) return fail("null argument");
    const AgentExpandCtx cx = agent_ctx(h, first_call, obs_host, reward_host, terminated_host, truncated_host, agent_mask_host, agent_life_host);
    *n_overflow = expand_records(h->p.N, n_threads, compact_words, compact_host, prev_host, overflow_envs_host,
                                 [&](int e, const uint32_t* r, uint32_t* pv) { return expand_agents(cx, e, r, pv); });
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_step_host_agents(ZsHandle* h, const int32_t* actions_host, int32_t action_format,
                                                                           uint32_t* compact_pinned, uint32_t* prev_host, int32_t compact_words,
                                                                           int32_t* obs_dev, int32_t* obs_host, double* reward_host,
                                                                           uint8_t* terminated_host, uint8_t* truncated_host,
                                                                           uint8_t* agent_mask_host, int16_t* agent_life_host,
                                                                           int32_t* overflow_envs_host, int32_t* n_overflow, int32_t first_call,
                                                                           int32_t n_threads, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (int rc = check_agent_words(h, compact_words)) return rc;
    if (!actions_host || !compact_pinned || !prev_host || !obs_host || !overflow_envs_host || !n_overflow) return fail("null argument");
    if (action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    const AgentExpandCtx cx = agent_ctx(h, first_call, obs_host, reward_host, terminated_host, truncated_host, agent_mask_host, agent_life_host);
    double us_total = 0;
    return host_step_run(h, actions_host, action_format, compact_pinned, prev_host, compact_words, obs_dev, overflow_envs_host, n_overflow,
                         n_threads, stream, false, [](int) {}, [&](int e, const uint32_t* r, uint32_t* pv) { return expand_agents(cx, e, r, pv); },
                         &us_total);
}

// diagnostics: out[5] = zs_step_host calls since the last read, and the mean microseconds from entry until the launches were
// issued / thread 0 had restored its previous cells / the flag showed (all records in host memory) / the call returned
extern "C" __attribute__((visibility("default"))) int zs_step_host_stats(ZsHandle* h, double* out) {
    if (!h || !out) return fail("null argument");
    const double n = h->host_stats[0] > 0 ? h->host_stats[0] : 1;
    out[0] = h->host_stats[0];
    for (int i = 1; i < 5; ++i) out[i] = h->host_stats[i] / n;
    for (double& v : h->host_stats) v = 0;
    return 0;
}

extern "C" __attribute__((visibility("default"))) int zs_encode_obs(ZsHandle* h, int32_t* obs_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (!obs_dev) return fail("null obs");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.obs = obs_dev; io.obs_slots = 1;
    launch_sim<MODE_ENCODE>(h, io, (cudaStream_t)stream);
    return launched(h);
}

// zs_rollout and zs_rollout_final: auto-reset whatever cfg.auto_reset says — same-step, or next-step on a handle created for it
// (the kernels of those handles have it compiled in, launch_sim)
static int rollout_launch(ZsHandle* h, int32_t n_steps, int64_t first_step_index, const int32_t* actions_dev, int32_t action_format,
                          int32_t* obs_dev, int32_t* final_obs_dev, int32_t obs_slots, double* reward_dev, uint8_t* terminated_dev,
                          uint8_t* truncated_dev, void* stream) {
    if (int rc = check_bound(h)) return rc;
    DeviceGuard guard(h);
    if (n_steps < 1) return fail("n_steps must be >= 1");
    if (obs_dev && obs_slots < 1) return fail("obs_slots must be >= 1");
    if (actions_dev && action_format != ZS_ACTIONS_FULL && action_format != ZS_ACTIONS_DISCRETE) return fail("bad action format");
    ZsIO io;
    memset(&io, 0, sizeof(io));
    io.actions = actions_dev; io.fmt = action_format; io.obs = obs_dev; io.obs_slots = obs_slots; io.reward = reward_dev;
    io.terminated = terminated_dev; io.truncated = truncated_dev; io.n_steps = n_steps; io.first_step = first_step_index;
    io.final_obs = final_obs_dev;
    io.force_auto_reset = 1;
    launch_sim<MODE_STEP>(h, io, (cudaStream_t)stream);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int zs_rollout(ZsHandle* h, int32_t n_steps, int64_t first_step_index, const int32_t* actions_dev,
                          int32_t action_format, int32_t* obs_dev, int32_t obs_slots, double* reward_dev,
                          uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream) {
    return rollout_launch(h, n_steps, first_step_index, actions_dev, action_format, obs_dev, nullptr, obs_slots, reward_dev,
                          terminated_dev, truncated_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int zs_rollout_final(ZsHandle* h, int32_t n_steps, int64_t first_step_index,
                                                                        const int32_t* actions_dev, int32_t action_format, int32_t* obs_dev,
                                                                        int32_t* final_obs_dev, int32_t obs_slots, double* reward_dev,
                                                                        uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream) {
    if (h && h->pending) return fail("zs_rollout_final needs a handle with auto_reset = 0 or 1: under next-step autoreset the observation of the step that ends an episode already is its final observation");
    if (!obs_dev || !final_obs_dev) return fail("zs_rollout_final needs an observation and a final observation ring");
    return rollout_launch(h, n_steps, first_step_index, actions_dev, action_format, obs_dev, final_obs_dev, obs_slots, reward_dev,
                          terminated_dev, truncated_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int zs_fill_synthetic_actions(ZsHandle* h, int64_t step_index, int32_t* actions_dev, void* stream) {
    if (!h) return fail("null handle");
    if (!actions_dev) return fail("null actions");
    DeviceGuard guard(h);
    const int n = h->p.N * h->p.A;
    int blocks = (n + 255) / 256;
    if (blocks > h->sm_count * 8) blocks = h->sm_count * 8;
    zs_fill_actions_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(h->p, (uint32_t)step_index, 1, actions_dev);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int zs_fill_synthetic_tape(ZsHandle* h, int64_t first_step_index, int32_t n_steps, int32_t* actions_dev, void* stream) {
    if (!h) return fail("null handle");
    if (!actions_dev) return fail("null actions");
    if (n_steps < 1) return fail("n_steps must be >= 1");
    DeviceGuard guard(h);
    const long long n = (long long)h->p.N * h->p.A * n_steps;
    long long blocks = (n + 255) / 256;
    if (blocks > h->sm_count * 16) blocks = h->sm_count * 16;
    zs_fill_actions_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(h->p, (uint32_t)first_step_index, n_steps, actions_dev);
    return launched(h);
}

extern "C" __attribute__((visibility("default"))) int zs_episode_stats(ZsHandle* h, int64_t* out_dev, int32_t reset, void* stream) {
    if (!h) return fail("null handle");
    if (!out_dev) return fail("null out");
    DeviceGuard guard(h);
    zs_stats_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(h->p.stats, out_dev, reset);
    return launched(h);
}

#ifdef ZS_TRACE
// development builds: copy the launch trace (zs_device.cuh: TR) to host memory [ZS_TRACE_WARPS][ZS_TRACE_SLOTS] uint64
extern "C" __attribute__((visibility("default"))) int zs_debug_trace(unsigned long long* out_host, int32_t clear) {
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(out_host, zs_trace_buf, sizeof(unsigned long long) * ZS_TRACE_WARPS * ZS_TRACE_SLOTS));
    if (clear) { void* d = nullptr; CU(cudaGetSymbolAddress(&d, zs_trace_buf)); CU(cudaMemset(d, 0, sizeof(unsigned long long) * ZS_TRACE_WARPS * ZS_TRACE_SLOTS)); }
    return 0;
}
#endif

extern "C" __attribute__((visibility("default"))) int64_t zs_launch_count(const ZsHandle* h) { return h ? h->launches : 0; }
extern "C" __attribute__((visibility("default"))) int32_t zs_lanes_per_env(const ZsHandle* h) { return h ? h->shape[0].lanes_per_env : 0; }
extern "C" __attribute__((visibility("default"))) int zs_autoreset_pending(const ZsHandle* h, const uint8_t** dev) {
    if (!h || !dev) return fail("null argument");
    *dev = h->pending;
    return h->pending ? 0 : fail("the handle has no next-step autoreset (auto_reset = ZS_AUTORESET_NEXT_STEP)");
}
