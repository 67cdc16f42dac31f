// mpe_kernels.cu -- the hot path of multiagent-particle-envs for a batch of worlds, sm_100a.
//
//   kFusedStep  MultiAgentEnv.step            environment.py:80-104   (one launch)
//   kSetAction  MultiAgentEnv._set_action     environment.py:144-192
//   kWorldStep  World.step                    core.py:117-131
//   kObserve    scenario.observation/reward + step glue (also used by reset)
//
// All four are the same kernel template with phases compiled in or out, so the fused step is
// bit-identical to set_action -> world_step -> observe.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <type_traits>
#include <utility>

#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: ranges cost a few ns unless a profiler is attached

#include "mpe_scenarios.cuh"
#include "mpe_spread_lanes.cuh"

namespace mpe {

template <int... I, class F>
__device__ __forceinline__ void static_for_impl(std::integer_sequence<int, I...>, F &&f) {
    (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
    static_for_impl(std::make_integer_sequence<int, N>{}, static_cast<F &&>(f));
}

template <class P>
struct Shape {
    // warp-private staging, in floats: [mbarrier: 4][action tiles of all agents][observation tiles]
    // Dense observation tiles (exact images of the global rows) each get their own slot, so that the
    // rows of all agents are written first and then streamed out after ONE __syncwarp; padded tiles
    // share one slot.
    static constexpr int kBarFloats = 4;
    __host__ __device__ static constexpr int act_floats(int i) { return 32 * (P::act_dim(i) | 1); }
    __host__ __device__ static constexpr int act_off(int i) { int s = kBarFloats; for (int j = 0; j < i; ++j) s += act_floats(j); return s; }
    __host__ __device__ static constexpr bool act_dense(int i) { return (P::act_dim(i) | 1) == P::act_dim(i); }
    __host__ __device__ static constexpr bool all_act_dense() { for (int i = 0; i < P::A; ++i) if (!act_dense(i)) return false; return true; }
    __host__ __device__ static constexpr int act_bytes_total() { int s = 0; for (int i = 0; i < P::A; ++i) s += 32 * P::act_dim(i) * 4; return s; }
    __host__ __device__ static constexpr int obs_pitch(int i) {
        const int od = P::obs_dim(i), unit = (od % 2 == 0) ? 2 : 1;
        return ((od / unit) | 1) * unit;
    }
    __host__ __device__ static constexpr bool obs_dense(int i) { return obs_pitch(i) == P::obs_dim(i); }
    // Every observation tile of a warp shares ONE slot (write rows, sync, stream out, sync) -- MPE_COMPACT_OBS=1, the
    // default since round 2.  With a private slot per dense tile (-DMPE_COMPACT_OBS=0, round 1: all rows written first,
    // one sync, then streamed) the staging of world_comm was 22 KB per warp and shared memory capped residency at 10
    // warps per SM; shared it is 6 KB (spread N=3: 8.8 -> 4.3 KB) and registers are the limit (16 warps per SM).
    // Measured (profiles/r2f_sweep_{default,compact}.jsonl): world_comm 65 536 worlds 20.3 -> 15.7 us (0.58 -> 0.75 of
    // the HBM peak), 32 768: 11.0 -> 10.0 us, 262 144: 58.6 -> 53.0 us; spread N=3 262 144: 18.7 -> 18.1 us; tag unchanged.
#ifndef MPE_COMPACT_OBS
#define MPE_COMPACT_OBS 1
#endif
    __host__ __device__ static constexpr bool obs_private(int i) { return obs_dense(i) && !MPE_COMPACT_OBS; }
    __host__ __device__ static constexpr int obs_floats(int i) { return (32 * obs_pitch(i) + 3) & ~3; }
    __host__ __device__ static constexpr int obs_base() { return act_off(P::A); }
    __host__ __device__ static constexpr int shared_obs_floats() { int m = 0; for (int i = 0; i < P::A; ++i) if (!obs_private(i)) m = obs_floats(i) > m ? obs_floats(i) : m; return m; }
    __host__ __device__ static constexpr int obs_off(int i) {
        if (!obs_private(i)) return obs_base();
        int s = obs_base() + shared_obs_floats();
        for (int j = 0; j < i; ++j) if (obs_private(j)) s += obs_floats(j);
        return s;
    }
    __host__ __device__ static constexpr int warp_floats() {
        int s = obs_base() + shared_obs_floats();
        for (int j = 0; j < P::A; ++j) if (obs_private(j)) s += obs_floats(j);
        return (s + 3) & ~3;
    }
    static constexpr int kWarpFloats = warp_floats();
    static constexpr int kWarpBytes = kWarpFloats * 4;
    // K-step rollout: a second set of action tiles behind the regular staging (step t+1 is prefetched while step t runs)
    static constexpr int kRolloutWarpFloats = kWarpFloats + ((obs_base() + 3) & ~3);
    static constexpr int kRolloutWarpBytes = kRolloutWarpFloats * 4;
    // software-pipelined persistent step (mpe_pipe_kernel): per warp [regular staging incl. obs tiles][second action
    // region][2 x state image: pv float4 [A][32], lm float2 [L][32], goal int [G][32]]
    static constexpr int kStateFloats = (4 * P::A + 2 * P::L + P::G) * 32;
    static constexpr int kPipeAct1 = kWarpFloats;
    static constexpr int kPipeState0 = kPipeAct1 + ((obs_base() + 3) & ~3);
    static constexpr int kPipeWarpFloats = kPipeState0 + 2 * kStateFloats;
    static constexpr int kPipeWarpBytes = kPipeWarpFloats * 4;
    static constexpr int kNC = P::NS * P::DIMC;
};

// World.step physics for one world held in registers (core.py:134-169)
template <class P>
__device__ __forceinline__ void physics(const DevDesc &d, typename P::W &w, const float (&ux)[P::A],
                                        const float (&uy)[P::A]) {
    constexpr int A = P::A, L = P::L;
    float2 F[A];   // (x, y) force pairs: accumulated with packed FADD2 (bit-identical to two scalar adds)
#pragma unroll
    for (int i = 0; i < A; ++i) F[i] = make_float2(ux[i], uy[i]);  // apply_action_force (core.py:134-140)
    const float k = d.contact_margin, cf = d.contact_force;
    // apply_environment_force (core.py:143-155): pairs (a, b), a < b, agents then landmarks.
    // Landmark-landmark pairs move nothing and are dropped at compile time.
#pragma unroll
    for (int a = 0; a < A; ++a) {
#pragma unroll
        for (int b = a + 1; b < A + L; ++b) {
            const bool b_agent = b < A;
            const int bi = b_agent ? b : 0, bl = b_agent ? 0 : b - A;
            // get_collision_force (core.py:181-182): the collide flags are structural constants of the
            // scenario program, so non-colliding pairs vanish at compile time and the remaining pairs form
            // one straight-line block that the scheduler interleaves freely
            if (!(P::agent_collides(a) && (b_agent ? P::agent_collides(bi) : P::landmark_collides(bl)))) continue;
            const float bx = b_agent ? w.px[bi] : w.lx[bl];
            const float by = b_agent ? w.py[bi] : w.ly[bl];
            const float sb = b_agent ? d.a_size[bi] : d.l_size[bl];
            const float2 dl = sub2(make_float2(w.px[a], w.py[a]), make_float2(bx, by));
            const float2 f = pair_force(dl.x, dl.y, __fadd_rn(d.a_size[a], sb), cf, k, d.inv_margin);   // :186-193
            if (P::movable(a)) F[a] = __fadd2_rn(F[a], f);                  // :194, 149-151
            if (b_agent && P::movable(bi)) F[bi] = sub2(F[bi], f);          // :195, 152-154
        }
    }
    // integrate_state (core.py:158-169)
#pragma unroll
    for (int i = 0; i < A; ++i) {
        if (!P::movable(i)) continue;
        const float4 r = integrate_entity<P::kSpeedLimit>(w.px[i], w.py[i], w.vx[i], w.vy[i], F[i].x, F[i].y, d.keep,
                                                          d.a_dt_over_mass[i], d.dt, d.a_max_speed[i]);
        w.px[i] = r.x; w.py[i] = r.y; w.vx[i] = r.z; w.vy[i] = r.w;
    }
}


// ---- warp-pair physics (SPLIT) ------------------------------------------------------------------------------------
// The active (colliding) pairs of apply_environment_force, numbered in the reference's (a, b) order.
template <class P>
__host__ __device__ constexpr bool pair_active(int a, int b) {
    return b > a && P::agent_collides(a) && (b < P::A ? P::agent_collides(b) : P::landmark_collides(b - P::A));
}
template <class P>
__host__ __device__ constexpr int pair_index(int a, int b) {   // number of active pairs before (a, b)
    int k = 0;
    for (int aa = 0; aa < P::A; ++aa)
        for (int bb = aa + 1; bb < P::A + P::L; ++bb) {
            if (aa == a && bb == b) return k;
            if (pair_active<P>(aa, bb)) ++k;
        }
    return k;
}
template <class P>
__host__ __device__ constexpr int pair_count() { return pair_index<P>(P::A, P::A + P::L); }

__device__ __forceinline__ void pair_sync(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

// Same result as physics<P>, bit for bit, computed by TWO warps that hold the same 32 worlds: warp `half` evaluates the
// contact forces of the pairs with index % 2 == half (the MUFU-heavy part) and publishes them in the pair's exchange
// buffer `ex` ([pair][lane] float2); after the pair barrier both warps read ALL pair forces back and accumulate them in
// the reference's order, then integrate.  The barrier also orders the partner's state loads before the in-place store.
template <class P>
__device__ __forceinline__ void physics_split(const DevDesc &d, typename P::W &w, const float (&ux)[P::A],
                                              const float (&uy)[P::A], int half, float2 *ex, int lane, int bar_id) {
    constexpr int A = P::A, L = P::L;
    const float k = d.contact_margin, cf = d.contact_force;
    static_for<A>([&](auto ac) {
        static_for<A + L>([&](auto bc) {
            constexpr int a = decltype(ac)::value, b = decltype(bc)::value;
            if constexpr (pair_active<P>(a, b)) {
                constexpr int idx = pair_index<P>(a, b);
                if ((idx & 1) == half) {   // warp-uniform
                    constexpr bool b_agent = b < A;
                    constexpr int bi = b_agent ? b : 0, bl = b_agent ? 0 : b - A;
                    const float bx = b_agent ? w.px[bi] : w.lx[bl];
                    const float by = b_agent ? w.py[bi] : w.ly[bl];
                    const float sb = b_agent ? d.a_size[bi] : d.l_size[bl];
                    const float2 dl = sub2(make_float2(w.px[a], w.py[a]), make_float2(bx, by));
                    ex[idx * 32 + lane] = pair_force(dl.x, dl.y, __fadd_rn(d.a_size[a], sb), cf, k, d.inv_margin);
                }
            }
        });
    });
    pair_sync(bar_id);
    float fx[A], fy[A];
#pragma unroll
    for (int i = 0; i < A; ++i) {  // apply_action_force (core.py:134-140)
        fx[i] = ux[i];
        fy[i] = uy[i];
    }
    static_for<A>([&](auto ac) {
        static_for<A + L>([&](auto bc) {
            constexpr int a = decltype(ac)::value, b = decltype(bc)::value;
            if constexpr (pair_active<P>(a, b)) {
                constexpr int idx = pair_index<P>(a, b);
                const float2 f = ex[idx * 32 + lane];
                if (P::movable(a)) {
                    fx[a] = __fadd_rn(fx[a], f.x);
                    fy[a] = __fadd_rn(fy[a], f.y);
                }
                if constexpr (b < A) {
                    if (P::movable(b)) {
                        fx[b] = __fsub_rn(fx[b], f.x);
                        fy[b] = __fsub_rn(fy[b], f.y);
                    }
                }
            }
        });
    });
#pragma unroll
    for (int i = 0; i < A; ++i) {
        if (!P::movable(i)) continue;
        const float4 r = integrate_entity<P::kSpeedLimit>(w.px[i], w.py[i], w.vx[i], w.vy[i], fx[i], fy[i], d.keep,
                                                          d.a_dt_over_mass[i], d.dt, d.a_max_speed[i]);
        w.px[i] = r.x; w.py[i] = r.y; w.vx[i] = r.z; w.vy[i] = r.w;
    }
}

// MultiAgentEnv._set_action (environment.py:144-192) for this lane's world, from the warp's staged action tiles
// (s_act = the warp's staging base; tile i starts at Shape<P>::act_off(i))
template <class P, bool ALLOW_FORCE_DISCRETE = true>
__device__ __forceinline__ void decode_rows(const float *s_act, int lane, const DevDesc &d, uint32_t flags,
                                            float (&ux)[P::A], float (&uy)[P::A], float *cact) {
    static_for<P::A>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        constexpr int AD = P::act_dim(i);
        constexpr int OFF = Shape<P>::act_off(i);
        const float *row = s_act + OFF + lane * Tile<AD>::kStride;
        int off = 0;
        float x = 0.0f, y = 0.0f;                                       // :145
        if constexpr (P::movable(i)) {
            float p0 = row[0], p1 = row[1], p2 = row[2], p3 = row[3], p4 = row[4];
            if (ALLOW_FORCE_DISCRETE && (flags & MPE_FLAG_FORCE_DISCRETE_ACTION)) {   // :169-172 (first arg-max)
                int best = 0;
                float bv = p0;
                if (p1 > bv) { bv = p1; best = 1; }
                if (p2 > bv) { bv = p2; best = 2; }
                if (p3 > bv) { bv = p3; best = 3; }
                if (p4 > bv) { bv = p4; best = 4; }
                p1 = best == 1 ? 1.0f : 0.0f; p2 = best == 2 ? 1.0f : 0.0f;
                p3 = best == 3 ? 1.0f : 0.0f; p4 = best == 4 ? 1.0f : 0.0f;
            }
            x += p1 - p2;                                               // :174
            y += p3 - p4;                                               // :175
            // explicit multiplies: must not be contracted into the force accumulation, or the fused
            // step would round differently from set_action -> world_step
            x = __fmul_rn(x, d.a_sens[i]);                              // :178-181
            y = __fmul_rn(y, d.a_sens[i]);
            off = 5;
        }
        ux[i] = x;
        uy[i] = y;
        if constexpr (i < P::NS) {                                      // :183-190 speakers come first
#pragma unroll
            for (int q = 0; q < P::DIMC; ++q) cact[i * P::DIMC + q] = row[off + q];
        }
    });
}

// observation rows of one 32-world tile into obs[i] + (row0 + world) * obs_dim_i: with `tile` (a full warp whose rows
// start 16-byte aligned) the rows go through the warp-private tiles and stream out as coalesced 16-byte stores;
// otherwise (the batch's last, partial warp) each lane writes its row straight to global memory.
// `half` < 0: every agent; 0: agents [0, split_point); 1: agents [split_point, A) (warp pairs; the second warp also
// computes the rewards, so it gets the smaller share: split_point = ceil(2A/3)).
template <class P>
__host__ __device__ constexpr int split_point() { return (2 * P::A + 2) / 3; }
template <class P>
__host__ __device__ constexpr int agent_half(int i) { return i < split_point<P>() ? 0 : 1; }
template <class P>
__device__ __forceinline__ void write_observations(float *const *obs, int64_t row0, const DevDesc &d, const typename P::W &w,
                                                   float *s_warp, int lane, bool tile, bool active, int64_t w0, int64_t wi,
                                                   int half) {
    constexpr int A = P::A;
    if (tile) {
        // Tiles are private per agent (dense ones), so no barrier is needed between agents: all rows are
        // written, one __syncwarp, then the warp streams every tile out as 16-byte stores and retires.
        // (A TMA bulk store was measured slower here: the warp has to stay resident until the copy
        // engine has read its shared memory, ~1.7 us at 13 warps/SM; see profiles/.)
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int OD = P::obs_dim(i);
            if (half >= 0 && agent_half<P>(i) != half) return;     // warp-uniform: the partner warp writes this agent
            TileWriter<OD> o(s_warp + Shape<P>::obs_off(i), lane);
            P::template observe<i>(d, w, o);
            if constexpr (!Shape<P>::obs_private(i)) {  // tiles without a slot of their own share one
                __syncwarp();
                obs_tile_store<OD>(obs[i] + (row0 + w0) * OD, s_warp + Shape<P>::obs_off(i), lane);
                __syncwarp();
            }
        });
        __syncwarp();
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int OD = P::obs_dim(i);
            if (half >= 0 && agent_half<P>(i) != half) return;
            if constexpr (Shape<P>::obs_private(i)) obs_tile_store<OD>(obs[i] + (row0 + w0) * OD, s_warp + Shape<P>::obs_off(i), lane);
        });
    } else if (active) {
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            if (half >= 0 && agent_half<P>(i) != half) return;
            RowWriter o{obs[i] + (row0 + wi) * P::obs_dim(i)};
            P::template observe<i>(d, w, o);
        });
    }
}

#ifndef MPE_BOUND_THREADS
#define MPE_BOUND_THREADS kMaxThreads   // register-budget experiments: -DMPE_BOUND_THREADS=128 lifts the cap from 128 to 255
#endif
#ifndef MPE_MIN_BLOCKS
#define MPE_MIN_BLOCKS 1   // 512-thread bound x 1 block = the same 128-register budget that measured best
#endif

// SPLIT (fused step only): TWO warps share a 32-world tile.  Both load the state and the actions; each evaluates half
// of the contact forces (exchanged through shared memory, accumulated by both in the reference's order: bit-identical
// state); warp 2k writes the new state and the observations of the first ceil(2A/3) agents, warp 2k+1 computes and
// writes the rewards / dones / info and the remaining observations.  It doubles the warps in flight and nearly halves
// each warp's instruction stream: batches too small to fill the machine with one lane per world (world_comm at 32 768
// worlds = 1.7 warps per scheduler, ~2500 dependent instructions each) are bound by instruction latency, not by HBM.
//
// HOT (fused step only): the specialisation the launcher uses whenever it can -- whole 32-world tiles, 16-byte aligned
// action rows, float action vectors without force_discrete_action, cp.async staging.  It contains none of the cold
// alternatives (partial-tile scalar paths, TMA staging, integer decode, arg-max), i.e. about half the static code of
// the general kernel: with ~3 resident warps per scheduler the step is bound by each warp's own instruction stream,
// and instruction-fetch stalls across the skipped cold blocks were ~8 % of it (profiles/).  Same arithmetic, same
// order: bit-identical.  A ragged tail and every other flag combination run on the general kernel.
//
// DENSE (HOT only): the same code compiled for an 80-register budget (__launch_bounds__(128, 6): 24 instead of 16
// resident warps per SM).  Only instantiated for programs that fit 80 registers without spilling (P::kLowRegVariant:
// the tag family up to 6 agents, spread N=4) and only launched when the batch has more tiles than the 128-register
// kernel keeps resident (> 148 x 16 warps): there occupancy wins (tag, 131 072 worlds: 13.1 -> 11.3 us, 0.75 -> 0.87
// of the HBM peak; 262 144: 23.1 -> 22.0 us), below it the register-rich version is faster (65 536: 7.5 vs 7.8 us)
// (profiles/r2g_sweep_{default,regs80}.jsonl).
template <class P, int MODE, bool SPLIT = false, bool HOT = false, bool DENSE = false>
__global__ void __launch_bounds__(DENSE ? 128 : MPE_BOUND_THREADS, DENSE ? 6 : MPE_MIN_BLOCKS) mpe_kernel(const __grid_constant__ StepArgs a) {
    static_assert(!DENSE || HOT, "the low-register build exists for the HOT fused step only");
    static_assert(!SPLIT || MODE == kFusedStep, "warp pairs exist for the fused step only");
    static_assert(!HOT || (MODE == kFusedStep && !SPLIT && Shape<P>::all_act_dense()), "HOT = plain fused step, dense tiles");
    static_assert(!SPLIT || pair_count<P>() * 64 <= Shape<P>::kWarpFloats - Shape<P>::obs_base(), "pair exchange must fit the obs tiles");
    constexpr int A = P::A, L = P::L, NC = Shape<P>::kNC;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int half = SPLIT ? (warp & 1) : 0;
    const int64_t n = a.n;
    const int64_t end = a.begin + a.count;
    const int64_t tile = SPLIT ? static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 6) + (warp >> 1)
                               : static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const int64_t w0 = a.begin + tile * 32;
    // Programmatic dependent launch (MPE_B200_PDL, see launch()): the index arithmetic and the first touches of the
    // parameter block (constant-bank misses) run before the wait; no global memory is touched before the previous
    // grid has completed and flushed.  A warp that exits early counts as having released the dependent grid.
    if (a.flags & kFlagPdlEarly) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (w0 >= end) return;  // whole warp exits together
    const int rows = HOT ? 32 : ((end - w0) < 32 ? static_cast<int>(end - w0) : 32);
    const bool active = HOT ? true : (lane < rows);
    const int64_t wi = w0 + (active ? lane : 0);  // inactive lanes shadow row 0 and never store
    float *s_warp = smem + warp * Shape<P>::kWarpFloats;
    uint64_t *bar = reinterpret_cast<uint64_t *>(s_warp);
    const DevDesc &d = a.d;
    {   // pull the parameter lines that the load phase needs into registers / the constant cache now
        uintptr_t touch = reinterpret_cast<uintptr_t>(a.pv) ^ reinterpret_cast<uintptr_t>(a.lm) ^
                          reinterpret_cast<uintptr_t>(a.obs[0]) ^ reinterpret_cast<uintptr_t>(a.rew) ^ a.flags ^
                          __float_as_uint(d.dt) ^ __float_as_uint(d.a_size[0]);
        asm volatile("" ::"l"(touch));
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // ---- action tiles: asynchronous copies (cp.async, or TMA bulk) issued FIRST, so that they fly together
    //      with the state loads -------------------------------------------------------------------------
    bool bulk = false;
    if constexpr (HOT) {
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int AD = P::act_dim(i), kVec = 32 * AD / 4;
            const float *g = a.act[i] + w0 * AD;
            float *sdst = s_warp + Shape<P>::act_off(i);
#pragma unroll
            for (int q0 = 0; q0 < kVec; q0 += 32)
                if (q0 + 32 <= kVec || q0 + lane < kVec) cp_async16(sdst + 4 * (q0 + lane), g + 4 * (q0 + lane));
        });
    } else if constexpr ((MODE == kFusedStep || MODE == kSetAction) && Shape<P>::all_act_dense()) {
        uintptr_t bits = 0;
#pragma unroll
        for (int i = 0; i < A; ++i) bits |= reinterpret_cast<uintptr_t>(a.act[i]);
        // warp-uniform; integer actions (discrete_action_input) are one or two words per world and need no tile
        bulk = (rows == 32) && ((bits & 15u) == 0) && !(a.flags & MPE_FLAG_DISCRETE_ACTION_INPUT);
        if (bulk && (a.flags & kFlagCpAsync)) {
            // every lane copies 16-byte pieces of the (contiguous) tiles straight into shared memory
            static_for<A>([&](auto ic) {
                constexpr int i = decltype(ic)::value;
                constexpr int AD = P::act_dim(i), kVec = 32 * AD / 4;
                const float *g = a.act[i] + w0 * AD;
                float *sdst = s_warp + Shape<P>::act_off(i);
#pragma unroll
                for (int q0 = 0; q0 < kVec; q0 += 32)
                    if (q0 + 32 <= kVec || q0 + lane < kVec) cp_async16(sdst + 4 * (q0 + lane), g + 4 * (q0 + lane));
            });
        } else if (bulk && lane == 0) {
            // one UBLKCP per agent tile (32 rows x act_dim floats, contiguous in global memory)
            mbar_init(bar, 1);
            mbar_expect_tx(bar, Shape<P>::act_bytes_total());
            static_for<A>([&](auto ic) {
                constexpr int i = decltype(ic)::value;
                constexpr int AD = P::act_dim(i);
                bulk_g2s(s_warp + Shape<P>::act_off(i), a.act[i] + w0 * AD, 32 * AD * 4, bar);
            });
        }
    }

    typename P::W w;
    // ---- state loads (issued first so they overlap the action staging) ---------------------
    if constexpr (MODE != kSetAction) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
            const float4 v = state_load(a.pv + i * n + wi);
            w.px[i] = v.x; w.py[i] = v.y; w.vx[i] = v.z; w.vy[i] = v.w;
        }
#pragma unroll
        for (int l = 0; l < L; ++l) {
            const float2 v = state_load(a.lm + l * n + wi);
            w.lx[l] = v.x; w.ly[l] = v.y;
        }
        if constexpr (MODE == kObserve && NC > 0) {
#pragma unroll
            for (int q = 0; q < NC; ++q) w.c[q] = a.comm[q * n + wi];
        }
        if constexpr ((MODE == kObserve || MODE == kFusedStep) && P::G > 0) {
#pragma unroll
            for (int q = 0; q < P::G; ++q) w.g[q] = a.goal[q * n + wi];
        }
    }

    if (a.flags & kFlagPdlAfterIssue) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    float ux[A], uy[A];
    float cact[NC > 0 ? NC : 1];
    // ---- MultiAgentEnv._set_action (environment.py:144-192) --------------------------------
    if constexpr (HOT) {
        cp_async_wait_all();
        __syncwarp();
        decode_rows<P, false>(s_warp, lane, d, a.flags, ux, uy, cact);
    } else if constexpr (MODE == kFusedStep || MODE == kSetAction) {
        if (a.flags & MPE_FLAG_DISCRETE_ACTION_INPUT) {
            // env.discrete_action_input (environment.py:161-167, 185-187): act_n[i] is int32 [n_env][n_sub_i], one index
            // per sub-action (movement 0..4, then the utterance 0..dim_c-1); consecutive lanes read consecutive words
            static_for<A>([&](auto ic) {
                constexpr int i = decltype(ic)::value;
                constexpr int NSUB = (P::movable(i) ? 1 : 0) + (i < P::NS ? 1 : 0);
                const int32_t *row = reinterpret_cast<const int32_t *>(a.act[i]) + wi * NSUB;
                float x = 0.0f, y = 0.0f;                                       // :145, 162
                int off = 0;
                if constexpr (P::movable(i)) {
                    const int k = row[0];
                    x = k == 1 ? -1.0f : (k == 2 ? 1.0f : 0.0f);                // :164-165
                    y = k == 3 ? -1.0f : (k == 4 ? 1.0f : 0.0f);                // :166-167
                    x = __fmul_rn(x, d.a_sens[i]);                              // :178-181
                    y = __fmul_rn(y, d.a_sens[i]);
                    off = 1;
                }
                ux[i] = x;
                uy[i] = y;
                if constexpr (i < P::NS) {                                      // :186-187 one-hot utterance
                    const int k = row[off];
#pragma unroll
                    for (int q = 0; q < P::DIMC; ++q) cact[i * P::DIMC + q] = (k == q) ? 1.0f : 0.0f;
                }
            });
        } else {
        if (bulk && (a.flags & kFlagCpAsync)) {
            cp_async_wait_all();
            __syncwarp();
        } else if (bulk) {
            __syncwarp();
            mbar_wait(bar, 0);
        } else {
            static_for<A>([&](auto ic) {
                constexpr int i = decltype(ic)::value;
                constexpr int AD = P::act_dim(i);
                constexpr int OFF = Shape<P>::act_off(i);
                tile_load<AD>(s_warp + OFF, a.act[i] + w0 * AD, rows, lane);
            });
            __syncwarp();
        }
        decode_rows<P>(s_warp, lane, d, a.flags, ux, uy, cact);
        }   // float action vectors
        if constexpr (MODE == kSetAction) {
            if (active) {
#pragma unroll
                for (int i = 0; i < A; ++i) a.u[i * n + wi] = make_float2(ux[i], uy[i]);
#pragma unroll
                for (int q = 0; q < NC; ++q) a.c[q * n + wi] = cact[q];
            }
            return;
        }
    }
    if constexpr (MODE == kWorldStep) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
            const float2 v = a.u[i * n + wi];
            ux[i] = v.x; uy[i] = v.y;
        }
#pragma unroll
        for (int q = 0; q < NC; ++q) cact[q] = a.c[q * n + wi];
    }

    if (a.flags & kFlagPdlAfterLoads) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // ---- World.step (core.py:117-131) --------------------------------------------------------
    if constexpr (MODE == kFusedStep || MODE == kWorldStep) {
        if constexpr (SPLIT) {
            // exchange buffer = the observation-tile area of the pair's even warp (idle until the observations are
            // written; the second barrier below keeps it intact until the partner has read every pair force)
            float2 *ex = reinterpret_cast<float2 *>(smem + (warp & ~1) * Shape<P>::kWarpFloats + Shape<P>::obs_base());
            physics_split<P>(d, w, ux, uy, half, ex, lane, 1 + (warp >> 1));
        } else {
            physics<P>(d, w, ux, uy);
        }
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = cact[q];  // update_agent_state (core.py:171-177)
        if (active && half == 0) {
#pragma unroll
            for (int i = 0; i < A; ++i)
                if (P::movable(i)) a.pv[i * n + wi] = make_float4(w.px[i], w.py[i], w.vx[i], w.vy[i]);
#pragma unroll
            for (int q = 0; q < NC; ++q) a.comm[q * n + wi] = w.c[q];
        }
        if constexpr (MODE == kWorldStep) return;
    }

    // ---- observation / reward / done / info (environment.py:92-102) -------------------------
    float rew[A];
    float info[(P::INFO > 0 ? P::INFO : 1) * A];
    P::prepare(d, w);   // per-world predicates shared by all agents' observations (world_comm: forest membership)
    if (!SPLIT || half == 1) {   // warp pairs: only the warp that stores the rewards computes them
        P::reward(d, w, rew, (P::INFO > 0 && a.info != nullptr) ? info : nullptr);
        if (a.flags & MPE_FLAG_SHARED_REWARD) {                                  // :100-102 np.sum(reward_n)
            float s = 0.0f;
#pragma unroll
            for (int i = 0; i < A; ++i) s += rew[i];
#pragma unroll
            for (int i = 0; i < A; ++i) rew[i] = s;
        }
    }
    if constexpr (SPLIT) pair_sync(1 + (warp >> 1));   // the partner has consumed the exchange buffer (= obs tiles of the even warp)
    if (!(a.flags & (kFlagPdlEarly | kFlagPdlAfterLoads | kFlagPdlAtExit | kFlagPdlAfterIssue))) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    write_observations<P>(a.obs, 0, d, w, s_warp, lane, rows == 32, active, w0, wi, SPLIT ? half : -1);
    if (active && (!SPLIT || half == 1)) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
            a.rew[i * n + wi] = rew[i];
            a.done[i * n + wi] = 0;  // done_callback is None (make_env.py:41-43, environment.py:132-135)
        }
        if (P::INFO > 0 && a.info != nullptr) {
#pragma unroll
            for (int q = 0; q < P::INFO * A; ++q) a.info[q * n + wi] = info[q];
        }
    }
}



// ---- software-pipelined persistent fused step (MPE_B200_PIPE=1; VERDICT r1 item 3(i)) -------------------------
// A grid of (tiles / tiles-per-warp) warps; every warp walks its 32-world tiles with a two-deep pipeline: ALL inputs
// of tile k+1 (action tiles, agent state, landmarks, goal indices) are fetched with cp.async into the second half of
// the warp's staging while tile k is decoded, integrated, observed and streamed out.  Load, compute and store phases
// of different tiles overlap inside one strictly ordered launch.  Same arithmetic functions as mpe_kernel: results
// are bit-identical (tests/test_gpu_parity.py).  Full tiles only; the launcher sends a ragged tail to mpe_kernel.
template <class P>
__global__ void __launch_bounds__(MPE_BOUND_THREADS, MPE_MIN_BLOCKS) mpe_pipe_kernel(const __grid_constant__ StepArgs a) {
    constexpr int A = P::A, L = P::L, NC = Shape<P>::kNC;
    using S = Shape<P>;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n = a.n;
    const int64_t n_tiles = a.count >> 5;
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
    int64_t t = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    float *s_warp = smem + warp * S::kPipeWarpFloats;
    const DevDesc &d = a.d;
    {
        uintptr_t touch = reinterpret_cast<uintptr_t>(a.pv) ^ reinterpret_cast<uintptr_t>(a.lm) ^
                          reinterpret_cast<uintptr_t>(a.obs[0]) ^ reinterpret_cast<uintptr_t>(a.rew) ^ a.flags ^
                          __float_as_uint(d.dt) ^ __float_as_uint(d.a_size[0]);
        asm volatile("" ::"l"(touch));
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (t >= n_tiles) return;

    auto act_base = [&](int b) { return s_warp + b * S::kPipeAct1; };
    auto state_base = [&](int b) { return s_warp + S::kPipeState0 + b * S::kStateFloats; };
    auto prefetch = [&](int64_t tile, int b) {
        const int64_t w0 = a.begin + tile * 32;
        float *ab = act_base(b);
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int AD = P::act_dim(i), kVec = 32 * AD / 4;
            const float *g = a.act[i] + w0 * AD;
            float *sdst = ab + S::act_off(i);
#pragma unroll
            for (int q0 = 0; q0 < kVec; q0 += 32)
                if (q0 + 32 <= kVec || q0 + lane < kVec) cp_async16(sdst + 4 * (q0 + lane), g + 4 * (q0 + lane));
        });
        float *sb = state_base(b);
#pragma unroll
        for (int i = 0; i < A; ++i) cp_async16(sb + (i * 32 + lane) * 4, a.pv + i * n + w0 + lane);
#pragma unroll
        for (int l = 0; l < L; ++l) cp_async8(sb + A * 128 + (l * 32 + lane) * 2, a.lm + l * n + w0 + lane);
#pragma unroll
        for (int q = 0; q < P::G; ++q) cp_async4(sb + A * 128 + L * 64 + q * 32 + lane, a.goal + q * n + w0 + lane);
    };

    prefetch(t, 0);
    cp_async_commit();
    bool first = true;
#pragma unroll 1
    for (int b = 0; t < n_tiles; t += nwarps, b ^= 1) {
        const int64_t w0 = a.begin + t * 32, wi = w0 + lane;
        if (t + nwarps < n_tiles) prefetch(t + nwarps, b ^ 1);
        cp_async_commit();
        cp_async_wait_group<1>();
        __syncwarp();
        if (first && (a.flags & kFlagPdlAfterLoads)) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        first = false;
        typename P::W w;
        const float *sb = state_base(b);
#pragma unroll
        for (int i = 0; i < A; ++i) {
            const float4 v = *reinterpret_cast<const float4 *>(sb + (i * 32 + lane) * 4);
            w.px[i] = v.x; w.py[i] = v.y; w.vx[i] = v.z; w.vy[i] = v.w;
        }
#pragma unroll
        for (int l = 0; l < L; ++l) {
            const float2 v = *reinterpret_cast<const float2 *>(sb + A * 128 + (l * 32 + lane) * 2);
            w.lx[l] = v.x; w.ly[l] = v.y;
        }
        if constexpr (P::G > 0) {
#pragma unroll
            for (int q = 0; q < P::G; ++q) w.g[q] = reinterpret_cast<const int *>(sb + A * 128 + L * 64)[q * 32 + lane];
        }
        float ux[A], uy[A];
        float cact[NC > 0 ? NC : 1];
        decode_rows<P>(act_base(b), lane, d, a.flags, ux, uy, cact);
        physics<P>(d, w, ux, uy);
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = cact[q];
#pragma unroll
        for (int i = 0; i < A; ++i)
            if (P::movable(i)) a.pv[i * n + wi] = make_float4(w.px[i], w.py[i], w.vx[i], w.vy[i]);
#pragma unroll
        for (int q = 0; q < NC; ++q) a.comm[q * n + wi] = w.c[q];
        float rew[A];
        float info[(P::INFO > 0 ? P::INFO : 1) * A];
        P::prepare(d, w);
        P::reward(d, w, rew, (P::INFO > 0 && a.info != nullptr) ? info : nullptr);
        if (a.flags & MPE_FLAG_SHARED_REWARD) {
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < A; ++i) sum += rew[i];
#pragma unroll
            for (int i = 0; i < A; ++i) rew[i] = sum;
        }
        write_observations<P>(a.obs, 0, d, w, s_warp, lane, true, true, w0, wi, -1);
#pragma unroll
        for (int i = 0; i < A; ++i) {
            a.rew[i * n + wi] = rew[i];
            a.done[i * n + wi] = 0;
        }
        if (P::INFO > 0 && a.info != nullptr) {
#pragma unroll
            for (int q = 0; q < P::INFO * A; ++q) a.info[q * n + wi] = info[q];
        }
        __syncwarp();   // every lane is done with buffer b (inputs) and the obs tiles before they are reused
    }
}

// ---- K-step open-loop rollout (SURVEY.md 8(f) rank 3: the persistent multi-step form) --------------------------
// T consecutive MultiAgentEnv.step calls on pre-generated actions act[i] : [T][n_env][act_dim_i] in ONE launch: a
// world's state is loaded once, lives in registers for all T steps and is written once; per step only the actions are
// read (the next step's tiles are prefetched with cp.async while this step computes) and, optionally, the per-step
// rewards written.  Observations are produced for the final state only.  This is what sampling-based planners (CEM /
// MPPI: score many candidate action sequences by their return) and policy evaluation on recorded actions need; HBM
// traffic per env-step drops from 411 B to 60 (+12) B for simple_spread N=3.  Bit-identical to T launches of the
// fused step with rewards summed in step order (tests/test_gpu_api.py).
struct RolloutArgs {
    StepArgs s;
    int32_t T;
    float *rew_steps;   // [T][A][n] per-step rewards (after the shared-reward sum), or null
};

template <class P>
__global__ void __launch_bounds__(MPE_BOUND_THREADS, MPE_MIN_BLOCKS) mpe_rollout_kernel(const __grid_constant__ RolloutArgs ra) {
    constexpr int A = P::A, L = P::L, NC = Shape<P>::kNC;
    const StepArgs &a = ra.s;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n = a.n;
    const int64_t end = a.begin + a.count;
    const int64_t w0 = a.begin + (static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp) * 32;
    if (w0 >= end) return;
    const int rows = (end - w0) < 32 ? static_cast<int>(end - w0) : 32;
    const bool active = lane < rows;
    const int64_t wi = w0 + (active ? lane : 0);
    float *s_warp = smem + warp * Shape<P>::kRolloutWarpFloats;
    const DevDesc &d = a.d;
    uintptr_t bits = 0;
#pragma unroll
    for (int i = 0; i < A; ++i) bits |= reinterpret_cast<uintptr_t>(a.act[i]) | static_cast<uintptr_t>((n * P::act_dim(i) * 4) & 15);
    const bool fast = Shape<P>::all_act_dense() && rows == 32 && (bits & 15u) == 0;   // warp-uniform

    auto stage = [&](int t, float *base) {   // action tiles of step t -> base (asynchronously on the fast path)
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            constexpr int AD = P::act_dim(i), kVec = 32 * AD / 4;
            const float *g = a.act[i] + (static_cast<int64_t>(t) * n + w0) * AD;
            float *sdst = base + Shape<P>::act_off(i);
            if (fast) {
#pragma unroll
                for (int q0 = 0; q0 < kVec; q0 += 32)
                    if (q0 + 32 <= kVec || q0 + lane < kVec) cp_async16(sdst + 4 * (q0 + lane), g + 4 * (q0 + lane));
            } else {
                tile_load<AD>(sdst, g, rows, lane);
            }
        });
    };
    stage(0, s_warp);
    cp_async_commit();

    typename P::W w;
#pragma unroll
    for (int i = 0; i < A; ++i) {
        const float4 v = state_load(a.pv + i * n + wi);
        w.px[i] = v.x; w.py[i] = v.y; w.vx[i] = v.z; w.vy[i] = v.w;
    }
#pragma unroll
    for (int l = 0; l < L; ++l) {
        const float2 v = state_load(a.lm + l * n + wi);
        w.lx[l] = v.x; w.ly[l] = v.y;
    }
    if constexpr (NC > 0) {   // only matters for T == 0; every step overwrites it (update_agent_state)
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = a.comm[q * n + wi];
    }
    if constexpr (P::G > 0) {
#pragma unroll
        for (int q = 0; q < P::G; ++q) w.g[q] = a.goal[q * n + wi];
    }

    float rsum[A];
#pragma unroll
    for (int i = 0; i < A; ++i) rsum[i] = 0.0f;
#pragma unroll 1
    for (int t = 0; t < ra.T; ++t) {
        float *cur = s_warp + (t & 1) * Shape<P>::kWarpFloats;           // tiles of step t; step t+1 goes to the other half
        if (t + 1 < ra.T) stage(t + 1, s_warp + ((t + 1) & 1) * Shape<P>::kWarpFloats);
        cp_async_commit();                 // possibly empty: keeps "all but the newest group" == "step t has landed"
        cp_async_wait_group<1>();
        __syncwarp();
        float ux[A], uy[A];
        float cact[NC > 0 ? NC : 1];
        decode_rows<P>(cur, lane, d, a.flags, ux, uy, cact);
        __syncwarp();                      // every lane has read `cur` before step t+2 is staged into it
        physics<P>(d, w, ux, uy);
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = cact[q];
        float rew[A];
        P::reward(d, w, rew, nullptr);
        if (a.flags & MPE_FLAG_SHARED_REWARD) {
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < A; ++i) sum += rew[i];
#pragma unroll
            for (int i = 0; i < A; ++i) rew[i] = sum;
        }
#pragma unroll
        for (int i = 0; i < A; ++i) rsum[i] = __fadd_rn(rsum[i], rew[i]);
        if (ra.rew_steps != nullptr && active) {
#pragma unroll
            for (int i = 0; i < A; ++i) ra.rew_steps[(static_cast<int64_t>(t) * A + i) * n + wi] = rew[i];
        }
    }
    cp_async_wait_all();
    if (active) {
#pragma unroll
        for (int i = 0; i < A; ++i)
            if (P::movable(i)) a.pv[i * n + wi] = make_float4(w.px[i], w.py[i], w.vx[i], w.vy[i]);
#pragma unroll
        for (int q = 0; q < NC; ++q) a.comm[q * n + wi] = w.c[q];
    }
    P::prepare(d, w);
    write_observations<P>(a.obs, 0, d, w, s_warp, lane, rows == 32, active, w0, wi, -1);
    if (active) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
            a.rew[i * n + wi] = rsum[i];
            a.done[i * n + wi] = 0;
        }
    }
}


// ---- K-step CLOSED-LOOP rollout with an in-kernel policy (SURVEY.md 8(f) rank 3, the persistent form with a device-
// resident policy; VERDICT r1 item 9) -------------------------------------------------------------------------------
// T consecutive MultiAgentEnv.step calls in ONE launch where every agent's action is produced inside the kernel by its
// own perceptron.  DEPTH 1:  logits_i = W2_i . relu(W1_i^T . obs_i + b1_i) + b2_i  (obs_dim_i -> H -> act_dim_i);
// DEPTH 2, the MADDPG actor:  logits_i = W3_i . relu(W2_i . relu(W1_i^T . obs_i + b1_i) + b2_i) + b3_i
// (obs_dim_i -> H -> H -> act_dim_i).  The logits split into the heads of the reference's action space
// (environment.py:58-64, MADDPG samples each head on its own): 5 movement logits if the agent moves, then dim_c
// communication logits if it speaks; each head gets its own softmax.  A world's state lives in registers for all T
// steps; an agent's observation is produced straight into registers, pushed through the perceptron (weights of all
// agents sit in shared memory once per block, read as broadcast LDS.128), decoded and integrated.  Per step NOTHING is
// read from HBM and only the optional records (rewards, actions, observations) are written; observations are always
// written for the final state.
// With MPE_FLAG_SAMPLE_ACTIONS the action is MADDPG's exploration sample softmax(logits + g), g = -log(-log u) Gumbel
// noise from a Philox stream keyed by (seed, global world, step, agent, logit), so trajectories do not depend on
// sharding.  The physics / reward / observation arithmetic is the fused step's: feeding the recorded actions to T fused
// steps reproduces the final state, the communication state, the observations and the reward sums bit for bit; the
// perceptron matches a float64 evaluation to ~1e-6 (tests).
struct PolicyArgs {
    StepArgs s;
    int32_t T;
    float *rew_steps;               // [T][A][n] or null
    float *act_rec[kMaxA];          // [T][n][act_dim_i] per agent, or null
    float *obs_rec[kMaxA];          // [T][n][obs_dim_i] per agent (row t: the observation acted on at step t), or all null
    const float *w1[kMaxA];         // [obs_dim_i][H]  (input-major: W1^T of a torch Linear(obs_dim_i, H))
    const float *b1[kMaxA];         // [H]
    const float *w2[kMaxA];         // depth 1: [act_dim_i][H] (torch Linear(H, act_dim_i).weight); depth 2: [H][H]
    const float *b2[kMaxA];         // depth 1: [act_dim_i]; depth 2: [H]
    const float *w3[kMaxA];         // depth 2: [act_dim_i][H] (torch Linear(H, act_dim_i).weight); depth 1: unused
    const float *b3[kMaxA];         // depth 2: [act_dim_i]
    uint2 sample_key;               // Philox key of the exploration noise (MPE_FLAG_SAMPLE_ACTIONS)
    uint64_t world_offset;          // global index of world 0 of this batch
    uint32_t sample_step;           // global step index of step 0 of this launch
};

__host__ __device__ constexpr int pad4(int x) { return (x + 3) & ~3; }
__host__ __device__ constexpr int ilog2(int x) { return x > 1 ? 1 + ilog2(x >> 1) : 0; }

// shared-memory image of one agent's actor (floats, every part 16-byte aligned), AD = act_dim_i, AP = pad4(AD):
//   depth 1: [W1: OD x H][b1: H][W2: AD x H][b2: AD, padded to AP]
//   depth 2: [W1: OD x H][b1: H][W2: H x H][b2: H][W3: H x AP, input-major, outputs AD..AP-1 zero][b3: AD, padded to AP]
template <class P, int H, int DEPTH>
struct PolicyShape {
    __host__ __device__ static constexpr int agent_floats(int i) {
        const int AD = P::act_dim(i), AP = pad4(AD);
        return P::obs_dim(i) * H + H + (DEPTH == 1 ? AD * H + AP : H * H + H + AP * H + AP);
    }
    __host__ __device__ static constexpr int agent_off(int i) { int s = 0; for (int j = 0; j < i; ++j) s += agent_floats(j); return s; }
    static constexpr int kWeightFloats = (agent_off(P::A) + 3) & ~3;
};

// observation writer into registers (every index is a compile-time constant after unrolling)
template <int DIM>
struct RegWriter {
    float v[DIM];
    int k = 0;
    __device__ __forceinline__ void put(float x) { v[k++] = x; }
    __device__ __forceinline__ void put2(float a, float b) { v[k] = a; v[k + 1] = b; k += 2; }
    __device__ __forceinline__ void put2(float2 a) { put2(a.x, a.y); }
};

// Philox counter word 3 of the exploration noise: bit 30 set keeps it apart from the reset stream (small block numbers
// and 0x80000000).  Movement logits: two blocks per (world, step, agent), 5 of their 8 words used.  Communication
// logit q: word q & 3 of block q >> 2 under 0x40000100 | agent << 2 | block (dim_c <= 16), which no movement tag
// (at most 0x4000000f) reaches.
__host__ __device__ constexpr uint32_t sample_tag(int agent, int block) { return 0x40000000u | (static_cast<uint32_t>(agent) << 1) | block; }
__host__ __device__ constexpr uint32_t comm_sample_tag(int agent, int block) {
    return 0x40000100u | (static_cast<uint32_t>(agent) << 2) | block;
}

// (2 k + 1) 2^-24, k < 2^23: exact in fp32 and strictly inside (0, 1), so both logarithms of the Gumbel term are finite
__device__ __forceinline__ float gumbel(uint32_t bits) {
    const float u = static_cast<float>(2u * (bits >> 9) + 1u) * 5.9604644775390625e-8f;
    return -logf(-logf(u));
}

// in-place softmax of one action head: max-subtracted, exponentials summed in ascending order
template <int N>
__device__ __forceinline__ void head_softmax(float *v) {
    float m = v[0];
#pragma unroll
    for (int c = 1; c < N; ++c) m = fmaxf(m, v[c]);
    float sum = 0.0f;
#pragma unroll
    for (int c = 0; c < N; ++c) { v[c] = expf(__fsub_rn(v[c], m)); sum = __fadd_rn(sum, v[c]); }
#pragma unroll
    for (int c = 0; c < N; ++c) v[c] = __fdiv_rn(v[c], sum);
}

// one agent of the in-kernel policy: observation -> registers -> perceptron -> (+ Gumbel noise) -> per-head softmax ->
// decoded (u.x, u.y) of the movement head (zero for an immovable agent) and, for a speaker, the communication head's
// probabilities in cact[I * dim_c ...] (action.c).  A plain force-inlined function with unrolled loops (not a lambda:
// arrays captured by reference by a lambda that the compiler declines to inline end up in local memory).  W = the
// agent's PolicyShape image in shared memory.
// Summation order (fixed; the float64 tests rely on it): every unit starts from its bias and adds its inputs in
// ascending order with FMAs -- layer 1 over j = observation index, layer 2 over j = layer-1 unit, the output layer over
// q = last hidden unit.
template <class P, int H, int DEPTH, int I, int NC>
__device__ __forceinline__ float2 policy_agent(const DevDesc &d, const typename P::W &w, const float *__restrict__ W,
                                               float *__restrict__ record, bool sample, uint2 key, uint64_t gw, uint32_t step,
                                               float (&cact)[NC]) {
    constexpr int OD = P::obs_dim(I), AD = P::act_dim(I), AP = pad4(AD);
    constexpr bool MOVE = P::movable(I), SPEAK = I < P::NS;
    constexpr int C0 = MOVE ? 5 : 0;                       // first communication logit
    static_assert(AD == C0 + (SPEAK ? P::DIMC : 0) && AD > 0 && P::DIMC <= 16, "policy rollout: action heads");
    const float *W1 = W, *B1 = W1 + OD * H, *W2 = B1 + H;
    RegWriter<OD> o;
    P::template observe<I>(d, w, o);                       // scenario.observation(agent I) -> registers
    float h[H];
#pragma unroll
    for (int q = 0; q < H; q += 4) {
        const float4 b = *reinterpret_cast<const float4 *>(B1 + q);
        h[q] = b.x; h[q + 1] = b.y; h[q + 2] = b.z; h[q + 3] = b.w;
    }
#pragma unroll
    for (int j = 0; j < OD; ++j) {                         // h += obs[j] * W1[j][:]   (ascending j, FMA)
        const float oj = o.v[j];
#pragma unroll
        for (int q = 0; q < H; q += 4) {
            const float4 wv = *reinterpret_cast<const float4 *>(W1 + j * H + q);
            h[q] = __fmaf_rn(oj, wv.x, h[q]);
            h[q + 1] = __fmaf_rn(oj, wv.y, h[q + 1]);
            h[q + 2] = __fmaf_rn(oj, wv.z, h[q + 2]);
            h[q + 3] = __fmaf_rn(oj, wv.w, h[q + 3]);
        }
    }
#pragma unroll
    for (int q = 0; q < H; ++q) h[q] = fmaxf(h[q], 0.0f);  // ReLU
    float lg[AD];
    if constexpr (DEPTH == 1) {
        const float *B2 = W2 + AD * H;
#pragma unroll
        for (int c = 0; c < AD; ++c) {                     // logits[c] = b2[c] + sum_q h[q] * W2[c][q]  (ascending q)
            float acc = B2[c];
#pragma unroll
            for (int q = 0; q < H; q += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(W2 + c * H + q);
                acc = __fmaf_rn(h[q], wv.x, acc);
                acc = __fmaf_rn(h[q + 1], wv.y, acc);
                acc = __fmaf_rn(h[q + 2], wv.z, acc);
                acc = __fmaf_rn(h[q + 3], wv.w, acc);
            }
            lg[c] = acc;
        }
    } else {
        // The second hidden layer is never materialised: unit q is computed, rectified and immediately folded into the
        // logits, so only h[H] and lg[AD] stay live (the register profile of depth 1).  The q loop stays rolled
        // (H x H unrolled FMAs per agent would overflow the instruction cache); the j loop is unrolled because h needs
        // compile-time indices.  h2_q = relu(b2[q] + sum_j h[j] W2[q][j]) (ascending j), then
        // logits[c] = b3[c] + sum_q h2_q W3[c][q] (ascending q).
        const float *B2 = W2 + H * H, *W3 = B2 + H, *B3 = W3 + AP * H;
#pragma unroll
        for (int c = 0; c < AD; ++c) lg[c] = B3[c];
#pragma unroll 1
        for (int q = 0; q < H; ++q) {
            const float *row = W2 + q * H;
            float acc = B2[q];
#pragma unroll
            for (int j = 0; j < H; j += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(row + j);
                acc = __fmaf_rn(h[j], wv.x, acc);
                acc = __fmaf_rn(h[j + 1], wv.y, acc);
                acc = __fmaf_rn(h[j + 2], wv.z, acc);
                acc = __fmaf_rn(h[j + 3], wv.w, acc);
            }
            acc = fmaxf(acc, 0.0f);
            float4 wv[AP / 4];                             // row q of W3: AP / 4 broadcast LDS.128
            static_for<AP / 4>([&](auto vc) {              // straight-line code: an inner loop, even unrolled, changes
                constexpr int v = decltype(vc)::value;     // how the rolled q loop is compiled
                wv[v] = *reinterpret_cast<const float4 *>(W3 + AP * q + 4 * v);
            });
            static_for<AD>([&](auto cc) {
                constexpr int c = decltype(cc)::value;
                const float4 &u = wv[c >> 2];
                lg[c] = __fmaf_rn(acc, (c & 3) == 0 ? u.x : (c & 3) == 1 ? u.y : (c & 3) == 2 ? u.z : u.w, lg[c]);
            });
        }
    }
    if (sample) {   // MADDPG's exploration: softmax(logits - log(-log u)), u uniform in (0, 1)
        const uint4 ctr = make_uint4(static_cast<uint32_t>(gw), static_cast<uint32_t>(gw >> 32), step, sample_tag(I, 0));
        if constexpr (MOVE) {
            const uint4 r0 = philox4x32_10(ctr, key);
            const uint4 r1 = philox4x32_10(make_uint4(ctr.x, ctr.y, ctr.z, sample_tag(I, 1)), key);
            const uint32_t bits[5] = {r0.x, r0.y, r0.z, r0.w, r1.x};
#pragma unroll
            for (int c = 0; c < 5; ++c) lg[c] = __fadd_rn(lg[c], gumbel(bits[c]));
        }
        if constexpr (SPEAK) {
#pragma unroll
            for (int b = 0; b < (P::DIMC + 3) / 4; ++b) {
                const uint4 r = philox4x32_10(make_uint4(ctr.x, ctr.y, ctr.z, comm_sample_tag(I, b)), key);
                const uint32_t bits[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                for (int q = 4 * b; q < P::DIMC && q < 4 * b + 4; ++q) lg[C0 + q] = __fadd_rn(lg[C0 + q], gumbel(bits[q & 3]));
            }
        }
    }
    float pr[AD];                                          // per-head softmax: the action vector [movement | comm]
    if constexpr (MOVE) {
        const float m = fmaxf(fmaxf(fmaxf(lg[0], lg[1]), fmaxf(lg[2], lg[3])), lg[4]);
        float e[5], sum = 0.0f;
#pragma unroll
        for (int c = 0; c < 5; ++c) { e[c] = expf(__fsub_rn(lg[c], m)); sum = __fadd_rn(sum, e[c]); }
#pragma unroll
        for (int c = 0; c < 5; ++c) pr[c] = __fdiv_rn(e[c], sum);
    }
    if constexpr (SPEAK) {
#pragma unroll
        for (int q = 0; q < P::DIMC; ++q) pr[C0 + q] = lg[C0 + q];
        head_softmax<P::DIMC>(pr + C0);
#pragma unroll
        for (int q = 0; q < P::DIMC; ++q) cact[I * P::DIMC + q] = pr[C0 + q];   // action.c (environment.py:183-190)
    }
    if (record != nullptr) {
#pragma unroll
        for (int c = 0; c < AD; ++c) record[c] = pr[c];
    }
    if constexpr (MOVE) {
        // _set_action (environment.py:173-181), the arithmetic of decode_rows
        float x = 0.0f, y = 0.0f;
        x += pr[1] - pr[2];
        y += pr[3] - pr[4];
        return make_float2(__fmul_rn(x, d.a_sens[I]), __fmul_rn(y, d.a_sens[I]));
    } else {
        return make_float2(0.0f, 0.0f);
    }
}

// block sizes: depth 1 as it always was (1, 2 or 4 warps); depth 2 up to 8 warps, because its weights (70-92 KB at
// H = 64) are staged once per block and only larger blocks let an SM hold as many warps as its registers allow
template <int DEPTH>
constexpr int kPolicyMaxWarps = DEPTH == 1 ? 4 : 8;

// EXTRAS = false: the plain closed loop (no exploration noise, no observation records) compiled without those paths.
// With them the depth-1 tag kernel at H = 64 needs 189 registers instead of 160 and takes 40.4 instead of 34.2 us per
// step at 65 536 worlds (B200, 1000 W), so depth 1 keeps the plain build for plain calls.
template <class P, int H, int DEPTH, bool EXTRAS>
__global__ void __launch_bounds__(32 * kPolicyMaxWarps<DEPTH>) mpe_policy_rollout_kernel(const __grid_constant__ PolicyArgs pa) {
    static_assert(H % 4 == 0, "policy rollout: hidden width a multiple of 4");
    static_assert(DEPTH == 1 || DEPTH == 2, "policy rollout: one or two hidden layers");
    constexpr int A = P::A, L = P::L, NC = Shape<P>::kNC;
    using PS = PolicyShape<P, H, DEPTH>;
    const StepArgs &a = pa.s;
    extern __shared__ __align__(16) float smem[];
    float *s_w = smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // ---- all agents' weights -> shared memory, once per block ------------------------------------------------
    static_for<A>([&](auto ic) {
        constexpr int i = decltype(ic)::value;
        constexpr int OD = P::obs_dim(i), AD = P::act_dim(i), AP = pad4(AD);
        float *base = s_w + PS::agent_off(i);
        for (int q = threadIdx.x; q < OD * H; q += blockDim.x) base[q] = pa.w1[i][q];
        for (int q = threadIdx.x; q < H; q += blockDim.x) base[OD * H + q] = pa.b1[i][q];
        base += OD * H + H;
        if constexpr (DEPTH == 1) {
            for (int q = threadIdx.x; q < AD * H; q += blockDim.x) base[q] = pa.w2[i][q];
            for (int q = threadIdx.x; q < AD; q += blockDim.x) base[AD * H + q] = pa.b2[i][q];
        } else {
            for (int q = threadIdx.x; q < H * H; q += blockDim.x) base[q] = pa.w2[i][q];
            for (int q = threadIdx.x; q < H; q += blockDim.x) base[H * H + q] = pa.b2[i][q];
            base += H * H + H;
            constexpr bool POW2 = (AP & (AP - 1)) == 0;   // every built program: AP = 4, 8 or 16
            for (int q = threadIdx.x; q < AP * H; q += blockDim.x) {     // W3 [AD][H] -> [H][AP]
                const int c = POW2 ? (q & (AP - 1)) : q % AP, r = POW2 ? (q >> ilog2(AP)) : q / AP;
                base[q] = c < AD ? pa.w3[i][c * H + r] : 0.0f;
            }
            for (int q = threadIdx.x; q < AP; q += blockDim.x) base[AP * H + q] = q < AD ? pa.b3[i][q] : 0.0f;
        }
    });
    __syncthreads();

    const int64_t n = a.n;
    const int64_t end = a.begin + a.count;
    const int64_t w0 = a.begin + (static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp) * 32;
    if (w0 >= end) return;
    const int rows = (end - w0) < 32 ? static_cast<int>(end - w0) : 32;
    const bool active = lane < rows;
    const int64_t wi = w0 + (active ? lane : 0);
    float *s_warp = smem + PS::kWeightFloats + warp * Shape<P>::kWarpFloats;
    const DevDesc &d = a.d;
    const bool sample = EXTRAS && (a.flags & MPE_FLAG_SAMPLE_ACTIONS) != 0;
    const bool rec_obs = EXTRAS && pa.obs_rec[0] != nullptr;
    const uint64_t gw = pa.world_offset + static_cast<uint64_t>(wi);

    typename P::W w;
#pragma unroll
    for (int i = 0; i < A; ++i) {
        const float4 v = state_load(a.pv + i * n + wi);
        w.px[i] = v.x; w.py[i] = v.y; w.vx[i] = v.z; w.vy[i] = v.w;
    }
#pragma unroll
    for (int l = 0; l < L; ++l) {
        const float2 v = state_load(a.lm + l * n + wi);
        w.lx[l] = v.x; w.ly[l] = v.y;
    }
    if constexpr (NC > 0) {   // the speakers' utterances of the previous step: what listeners observe at step 0
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = a.comm[q * n + wi];
    }
    if constexpr (P::G > 0) {
#pragma unroll
        for (int q = 0; q < P::G; ++q) w.g[q] = a.goal[q * n + wi];
    }

    float rsum[A];
#pragma unroll
    for (int i = 0; i < A; ++i) rsum[i] = 0.0f;
#pragma unroll 1
    for (int t = 0;; ++t) {
        P::prepare(d, w);
        const bool last = t == pa.T;
        if (last || rec_obs) {
            // the observations of step t go to record row t, and after the last step to obs_n: one call site for both
            // keeps a single inlined copy of every agent's observation code.  The tile path needs every row block
            // 16-byte aligned, which fails for odd t when n * obs_dim_i is not a multiple of 4: such rows go direct.
            float *const *obs = last ? a.obs : pa.obs_rec;
            const int64_t row0 = last ? 0 : static_cast<int64_t>(t) * n;
            bool tile = rows == 32;
#pragma unroll
            for (int i = 0; i < A; ++i)
                tile = tile && ((reinterpret_cast<uintptr_t>(obs[i] + (row0 + w0) * P::obs_dim(i)) & 15u) == 0);
            write_observations<P>(obs, row0, d, w, s_warp, lane, tile, active, w0, wi, -1);
            if (last) break;
            __syncwarp();   // every lane has streamed the tiles out before any lane refills them
        }
        float ux[A], uy[A];
        float cact[NC > 0 ? NC : 1];
        static_for<A>([&](auto ic) {
            constexpr int i = decltype(ic)::value, AD = P::act_dim(i);
            const float2 u = policy_agent<P, H, DEPTH, i>(d, w, s_w + PS::agent_off(i),
                                                          (pa.act_rec[i] != nullptr && active)
                                                              ? pa.act_rec[i] + (static_cast<int64_t>(t) * n + wi) * AD : nullptr,
                                                          sample, pa.sample_key, gw, pa.sample_step + static_cast<uint32_t>(t),
                                                          cact);
            ux[i] = u.x;
            uy[i] = u.y;
        });
        physics<P>(d, w, ux, uy);
        // update_agent_state (core.py:172-178) after every agent has acted on the step-t utterances, as the fused step
#pragma unroll
        for (int q = 0; q < NC; ++q) w.c[q] = cact[q];
        float rew[A];
        P::reward(d, w, rew, nullptr);
        if (a.flags & MPE_FLAG_SHARED_REWARD) {
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < A; ++i) sum += rew[i];
#pragma unroll
            for (int i = 0; i < A; ++i) rew[i] = sum;
        }
#pragma unroll
        for (int i = 0; i < A; ++i) rsum[i] = __fadd_rn(rsum[i], rew[i]);
        if (pa.rew_steps != nullptr && active) {
#pragma unroll
            for (int i = 0; i < A; ++i) pa.rew_steps[(static_cast<int64_t>(t) * A + i) * n + wi] = rew[i];
        }
    }
    if (active) {
#pragma unroll
        for (int i = 0; i < A; ++i)
            if (P::movable(i)) a.pv[i * n + wi] = make_float4(w.px[i], w.py[i], w.vx[i], w.vy[i]);
#pragma unroll
        for (int q = 0; q < NC; ++q) a.comm[q * n + wi] = w.c[q];
    }
    if (active) {
#pragma unroll
        for (int i = 0; i < A; ++i) {
            a.rew[i * n + wi] = rsum[i];
            a.done[i * n + wi] = 0;
        }
    }
}

template <class P>
constexpr bool policy_rollout_ok() {     // every agent moves, nobody speaks: the action is the 5-vector of probabilities
    bool ok = P::NS == 0;
    for (int i = 0; i < P::A; ++i) ok = ok && P::movable(i) && P::act_dim(i) == 5;
    return ok;
}
// Worlds the closed loop is built for (each instantiation unrolls obs_dim x H FMAs per agent: compile time): the
// BASELINE.json worlds (`baseline`: also the plain depth-1 kernel, and the opt-in step alternatives of make_program)
// and the other scenarios of the MADDPG benchmark suite at their reference entity counts.
template <class P> struct PolicyBuilt { static constexpr bool value = false, baseline = false; };
template <> struct PolicyBuilt<Simple<1, 1>> { static constexpr bool value = true, baseline = true; };
template <> struct PolicyBuilt<Spread<3>> { static constexpr bool value = true, baseline = true; };
template <> struct PolicyBuilt<Tag<3, 1, 2>> { static constexpr bool value = true, baseline = true; };
template <> struct PolicyBuilt<Adversary<1, 2, 2>> { static constexpr bool value = true, baseline = false; };
template <> struct PolicyBuilt<Push<1, 1, 2>> { static constexpr bool value = true, baseline = false; };
template <> struct PolicyBuilt<SpeakerListener> { static constexpr bool value = true, baseline = false; };
template <> struct PolicyBuilt<Reference> { static constexpr bool value = true, baseline = false; };
template <> struct PolicyBuilt<Crypto> { static constexpr bool value = true, baseline = false; };

// ---- generic program for user scenarios (MPE_SCN_CUSTOM) ------------------------------------------
// Any entity table, flags read at run time; same arithmetic primitives and the same (a, b) pair order as
// the compiled programs, so for a table that matches a built-in scenario the state is bit-identical.
// Loops are unrolled to the maximum counts with run-time guards, which keeps every array in registers.
__global__ void __launch_bounds__(128) generic_set_action_kernel(const __grid_constant__ StepArgs a) {
    const int64_t w = a.begin + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= a.begin + a.count) return;
    const DevDesc &d = a.d;
    const int64_t n = a.n;
    const int C = d.g_dim_c;
#pragma unroll
    for (int i = 0; i < kMaxA; ++i) {
        if (i >= d.g_agents) break;
        const bool movable = (d.g_movable >> i) & 1u, silent = (d.g_silent >> i) & 1u;
        const int adim = (movable ? 5 : 0) + (silent ? 0 : C);
        float x = 0.0f, y = 0.0f;
        int off = 0;
        if (a.flags & MPE_FLAG_DISCRETE_ACTION_INPUT) {            // environment.py:161-167, 185-187
            const int nsub = (movable ? 1 : 0) + (silent ? 0 : 1);
            const int32_t *irow = reinterpret_cast<const int32_t *>(a.act[i]) + w * nsub;
            if (movable) {
                const int k = irow[0];
                x = __fmul_rn(k == 1 ? -1.0f : (k == 2 ? 1.0f : 0.0f), d.a_sens[i]);
                y = __fmul_rn(k == 3 ? -1.0f : (k == 4 ? 1.0f : 0.0f), d.a_sens[i]);
                off = 1;
            }
            a.u[i * n + w] = make_float2(x, y);
            if (!silent) {
                const int k = irow[off];
                for (int q = 0; q < C; ++q) a.c[(d.g_slot[i] * C + q) * n + w] = (k == q) ? 1.0f : 0.0f;
            }
            continue;
        }
        const float *row = a.act[i] + w * adim;
        if (movable) {                                             // environment.py:157-181
            float p0 = row[0], p1 = row[1], p2 = row[2], p3 = row[3], p4 = row[4];
            if (a.flags & MPE_FLAG_FORCE_DISCRETE_ACTION) {
                int best = 0;
                float bv = p0;
                if (p1 > bv) { bv = p1; best = 1; }
                if (p2 > bv) { bv = p2; best = 2; }
                if (p3 > bv) { bv = p3; best = 3; }
                if (p4 > bv) { bv = p4; best = 4; }
                p1 = best == 1 ? 1.0f : 0.0f; p2 = best == 2 ? 1.0f : 0.0f;
                p3 = best == 3 ? 1.0f : 0.0f; p4 = best == 4 ? 1.0f : 0.0f;
            }
            x = __fmul_rn(p1 - p2, d.a_sens[i]);
            y = __fmul_rn(p3 - p4, d.a_sens[i]);
            off = 5;
        }
        a.u[i * n + w] = make_float2(x, y);
        if (!silent)                                               // environment.py:183-190
            for (int q = 0; q < C; ++q) a.c[(d.g_slot[i] * C + q) * n + w] = row[off + q];
    }
}

__global__ void __launch_bounds__(128) generic_world_step_kernel(const __grid_constant__ StepArgs a) {
    const int64_t w = a.begin + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= a.begin + a.count) return;
    const DevDesc &d = a.d;
    const int64_t n = a.n;
    const int A = d.g_agents, L = d.g_landmarks, C = d.g_dim_c;
    float px[kMaxA], py[kMaxA], vx[kMaxA], vy[kMaxA], fx[kMaxA], fy[kMaxA], lx[kMaxL], ly[kMaxL];
#pragma unroll
    for (int i = 0; i < kMaxA; ++i) {
        px[i] = py[i] = vx[i] = vy[i] = fx[i] = fy[i] = 0.0f;
        if (i < A) {
            const float4 v = a.pv[i * n + w];
            const float2 u = a.u[i * n + w];
            px[i] = v.x; py[i] = v.y; vx[i] = v.z; vy[i] = v.w;
            fx[i] = u.x; fy[i] = u.y;                               // apply_action_force (core.py:134-140)
        }
    }
#pragma unroll
    for (int l = 0; l < kMaxL; ++l) {
        lx[l] = ly[l] = 0.0f;
        if (l < L) {
            const float2 v = a.lm[l * n + w];
            lx[l] = v.x; ly[l] = v.y;
        }
    }
    // apply_environment_force (core.py:143-155), pairs (a, b), a < b, agents then landmarks
#pragma unroll
    for (int i = 0; i < kMaxA; ++i) {
        if (i >= A || !((d.g_collide >> i) & 1u)) continue;
#pragma unroll
        for (int j = i + 1; j < kMaxA; ++j) {
            if (j >= A || !((d.g_collide >> j) & 1u)) continue;
            const float2 f = pair_force(__fsub_rn(px[i], px[j]), __fsub_rn(py[i], py[j]), __fadd_rn(d.a_size[i], d.a_size[j]),
                                        d.contact_force, d.contact_margin, d.inv_margin);
            if ((d.g_movable >> i) & 1u) { fx[i] = __fadd_rn(fx[i], f.x); fy[i] = __fadd_rn(fy[i], f.y); }
            if ((d.g_movable >> j) & 1u) { fx[j] = __fsub_rn(fx[j], f.x); fy[j] = __fsub_rn(fy[j], f.y); }
        }
#pragma unroll
        for (int l = 0; l < kMaxL; ++l) {
            if (l >= L || !((d.g_lcollide >> l) & 1u)) continue;
            const float2 f = pair_force(__fsub_rn(px[i], lx[l]), __fsub_rn(py[i], ly[l]), __fadd_rn(d.a_size[i], d.l_size[l]),
                                        d.contact_force, d.contact_margin, d.inv_margin);
            if ((d.g_movable >> i) & 1u) { fx[i] = __fadd_rn(fx[i], f.x); fy[i] = __fadd_rn(fy[i], f.y); }
        }
    }
    // integrate_state (core.py:158-169)
#pragma unroll
    for (int i = 0; i < kMaxA; ++i) {
        if (i >= A || !((d.g_movable >> i) & 1u)) continue;
        float4 r;
        if (d.a_max_speed[i] >= 0.0f)
            r = integrate_entity<true>(px[i], py[i], vx[i], vy[i], fx[i], fy[i], d.keep, d.a_dt_over_mass[i], d.dt, d.a_max_speed[i]);
        else
            r = integrate_entity<false>(px[i], py[i], vx[i], vy[i], fx[i], fy[i], d.keep, d.a_dt_over_mass[i], d.dt, 0.0f);
        a.pv[i * n + w] = r;
    }
    // update_agent_state (core.py:171-177): state.c = action.c for the speakers
    for (int q = 0; q < d.g_comm_rows; ++q) a.comm[q * n + w] = a.c[q * n + w];
    (void)C;
}

// ---- reset: i.i.d. uniform positions (e.g. simple_spread.py:38-45) -----------------------------
struct ResetArgs {
    int64_t n;
    int A, L, NC, G;
    float4 *pv;
    float2 *lm;
    float *comm;
    int32_t *goal;
    const uint8_t *mask;
    uint64_t seed, world_offset, epoch;
    const unsigned long long *epoch_dev;   // when non-null the epoch is read from device memory
    float agent_range, landmark_range[kMaxL];
    int goal_mod[4];
};

__global__ void __launch_bounds__(256) reset_kernel(const __grid_constant__ ResetArgs a) {
    const int64_t w = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= a.n) return;
    if (a.mask != nullptr && a.mask[w] == 0) return;
    const uint64_t epoch = a.epoch_dev ? *a.epoch_dev : a.epoch;
    const uint64_t gw = a.world_offset + static_cast<uint64_t>(w);
    const uint2 key = make_uint2(static_cast<uint32_t>(a.seed), static_cast<uint32_t>(a.seed >> 32));
    // one Philox block = 4 x 32 bits = two entities' (x, y); counter = (world lo, world hi, epoch, block)
    const int E = a.A + a.L;
    for (int e = 0; e < E; e += 2) {
        const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(gw), static_cast<uint32_t>(gw >> 32),
                                                 static_cast<uint32_t>(epoch), static_cast<uint32_t>(e >> 1)), key);
        const uint32_t bits[4] = {r.x, r.y, r.z, r.w};
        for (int k = 0; k < 2 && e + k < E; ++k) {
            const int ent = e + k;
            if (ent < a.A) {
                const float x = uniform_from_bits(bits[2 * k], -a.agent_range, a.agent_range);
                const float y = uniform_from_bits(bits[2 * k + 1], -a.agent_range, a.agent_range);
                a.pv[ent * a.n + w] = make_float4(x, y, 0.0f, 0.0f);
            } else {
                const float rg = a.landmark_range[ent - a.A];
                a.lm[(ent - a.A) * a.n + w] = make_float2(uniform_from_bits(bits[2 * k], -rg, rg),
                                                           uniform_from_bits(bits[2 * k + 1], -rg, rg));
            }
        }
    }
    for (int q = 0; q < a.NC; ++q) a.comm[q * a.n + w] = 0.0f;
    if (a.G > 0) {
        const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(gw), static_cast<uint32_t>(gw >> 32),
                                                 static_cast<uint32_t>(epoch), 0x80000000u), key);
        const uint32_t bits[4] = {r.x, r.y, r.z, r.w};
        for (int g = 0; g < a.G && g < 4; ++g) a.goal[g * a.n + w] = static_cast<int32_t>(bits[g] % static_cast<uint32_t>(a.goal_mod[g]));
    }
}

__global__ void bump_epoch_kernel(unsigned long long *epoch) { *epoch += 1ull; }

// ---- diagnostics: a pure streaming kernel with a step's byte counts (bench.py's size-matched ceiling) ------
// Reads n_read4 float4, then writes n_write4 float4 that depend on what was read (like a step: stores follow the
// loads), same launch path (programmatic dependent launch) and the same evict-first stores as the step kernel.
__global__ void __launch_bounds__(256) stream_probe_kernel(const float4 *__restrict__ src, long long n_read4,
                                                           float4 *__restrict__ dst, long long n_write4) {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long nth = static_cast<long long>(gridDim.x) * blockDim.x;
    float acc = 0.0f;
#pragma unroll 8
    for (long long i = tid; i < n_read4; i += nth) {
        const float4 v = src[i];
        acc += (v.x + v.y) + (v.z + v.w);
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const float4 o = make_float4(acc, acc, acc, acc);
#pragma unroll 8
    for (long long i = tid; i < n_write4; i += nth) __stcs(dst + i, o);
}

// ---- program table -----------------------------------------------------------------------------
typedef void (*KernelFn)(StepArgs);

struct Program {
    int scenario;
    bool (*validate)(const mpe_desc &);
    KernelFn fn[4];
    int smem_bytes;  // dynamic shared memory per WARP
    KernelFn hot_fn;    // fused step specialised for whole tiles / float actions / cp.async staging (null: no such program)
    KernelFn hot_dense_fn;   // the same compiled for 80 registers (large batches of programs that fit without spilling)
    KernelFn split_fn;  // fused step with a warp PAIR per 32-world tile (small batches of heavy scenarios)
    KernelFn pipe_fn;   // software-pipelined persistent fused step (null unless every action tile is dense)
    int pipe_smem;      // dynamic shared memory per WARP of the pipelined kernel
    void (*policy_fn[2][2])(PolicyArgs);  // K-step closed-loop rollout [depth - 1][hidden 32 / 64] (null: not built)
    void (*policy_plain_fn[2])(PolicyArgs);  // the same at depth 1 without exploration noise and observation records
                                             // (null: policy_fn serves plain calls too)
    int policy_weight_floats[2][2];
    bool policy_move_only;   // every agent moves and is silent: actions are the 5 movement probabilities (mpe_rollout_policy)
    void (*rollout_fn)(RolloutArgs);   // K-step open-loop rollout
    int rollout_smem;   // dynamic shared memory per WARP of the rollout kernel
    KernelFn lanes_fn;  // lane-per-agent fused step (simple_spread only), else null
    int lanes_smem, lanes_wpw;
    int A, L, NS, DIMC, INFO, G;
    int obs_dim[kMaxA], act_dim[kMaxA];
    int unread_state_floats;   // state floats per world that this scenario's step never needs (not compulsory traffic)
};

template <class P>
static Program make_program() {
    Program p{};
    p.scenario = P::kScenario;
    p.validate = &P::validate;
    p.fn[kFusedStep] = mpe_kernel<P, kFusedStep>;
    p.fn[kSetAction] = mpe_kernel<P, kSetAction>;
    p.fn[kWorldStep] = mpe_kernel<P, kWorldStep>;
    p.fn[kObserve] = mpe_kernel<P, kObserve>;
    // the two restructurings that measurements rejected (warp pairs, software-pipelined persistent grid) stay available as
    // opt-in, bit-identical alternatives for the BASELINE.json worlds only (compile time)
    constexpr bool kAlternatives = PolicyBuilt<P>::baseline || std::is_same<P, Spread<6>>::value ||
                                   std::is_same<P, WorldComm<4, 2, 1, 2>>::value;
    if constexpr (kAlternatives && P::A >= 2 && pair_count<P>() * 64 <= Shape<P>::kWarpFloats - Shape<P>::obs_base())
        p.split_fn = mpe_kernel<P, kFusedStep, true>;     // (the pair exchange must fit the observation tiles)
    if constexpr (Shape<P>::all_act_dense()) p.hot_fn = mpe_kernel<P, kFusedStep, false, true>;
    if constexpr (Shape<P>::all_act_dense() && P::kLowRegVariant) p.hot_dense_fn = mpe_kernel<P, kFusedStep, false, true, true>;
    if constexpr (kAlternatives && Shape<P>::all_act_dense()) p.pipe_fn = mpe_pipe_kernel<P>;
    p.pipe_smem = Shape<P>::kPipeWarpBytes;
    p.rollout_fn = mpe_rollout_kernel<P>;
    p.rollout_smem = Shape<P>::kRolloutWarpBytes;
    // the closed-loop rollout; only the BASELINE.json worlds also get the plain depth-1 build (compile time)
    if constexpr (PolicyBuilt<P>::value) {
        if constexpr (PolicyBuilt<P>::baseline) {
            p.policy_plain_fn[0] = mpe_policy_rollout_kernel<P, 32, 1, false>;
            p.policy_plain_fn[1] = mpe_policy_rollout_kernel<P, 64, 1, false>;
        }
        p.policy_fn[0][0] = mpe_policy_rollout_kernel<P, 32, 1, true>;
        p.policy_fn[0][1] = mpe_policy_rollout_kernel<P, 64, 1, true>;
        p.policy_fn[1][0] = mpe_policy_rollout_kernel<P, 32, 2, true>;
        p.policy_fn[1][1] = mpe_policy_rollout_kernel<P, 64, 2, true>;
        p.policy_weight_floats[0][0] = PolicyShape<P, 32, 1>::kWeightFloats;
        p.policy_weight_floats[0][1] = PolicyShape<P, 64, 1>::kWeightFloats;
        p.policy_weight_floats[1][0] = PolicyShape<P, 32, 2>::kWeightFloats;
        p.policy_weight_floats[1][1] = PolicyShape<P, 64, 2>::kWeightFloats;
    }
    p.policy_move_only = policy_rollout_ok<P>();
    p.smem_bytes = Shape<P>::kWarpBytes;  // per warp
    p.A = P::A; p.L = P::L; p.NS = P::NS; p.DIMC = P::DIMC; p.INFO = P::INFO; p.G = P::G;
    for (int i = 0; i < P::A; ++i) { p.obs_dim[i] = P::obs_dim(i); p.act_dim[i] = P::act_dim(i); }
    // simple_crypto never looks at a position (nobody moves, observations and rewards are about utterances only);
    // simple_speaker_listener never looks at the immovable speaker's position
    p.unread_state_floats = P::kScenario == MPE_SCN_CRYPTO ? 4 * P::A + 2 * P::L
                          : (P::kScenario == MPE_SCN_SPEAKER_LISTENER ? 4 : 0);
    return p;
}

// MPE_SCN_CUSTOM: shapes come from the descriptor at create time (see mpe_create)
static Program make_generic_program() {
    Program p{};
    p.scenario = MPE_SCN_CUSTOM;
    p.validate = [](const mpe_desc &) { return true; };
    p.fn[kSetAction] = generic_set_action_kernel;
    p.fn[kWorldStep] = generic_world_step_kernel;
    p.smem_bytes = 0;
    return p;
}

template <int N>
static Program make_spread_program() {
    Program p = make_program<Spread<N>>();
    p.lanes_fn = spread_lanes_kernel<N>;
    p.lanes_smem = SpreadLanes<N>::kWarpBytes;
    p.lanes_wpw = SpreadLanes<N>::WPW;
    return p;
}

static const Program *programs(int *count) {
    static const Program table[] = {
        make_generic_program(),
        make_program<Simple<1, 1>>(),
        make_spread_program<2>(), make_spread_program<3>(), make_spread_program<4>(),
        make_spread_program<5>(), make_spread_program<6>(),
        make_program<Tag<3, 1, 2>>(), make_program<Tag<1, 1, 2>>(), make_program<Tag<2, 1, 2>>(),
        make_program<Tag<4, 2, 2>>(), make_program<Tag<6, 2, 3>>(),
        make_program<WorldComm<4, 2, 1, 2>>(),
        make_program<Adversary<1, 2, 2>>(), make_program<Adversary<1, 3, 3>>(),
        make_program<Push<1, 1, 2>>(),
        make_program<SpeakerListener>(),
        make_program<Reference>(),
        make_program<Crypto>(),
    };
    *count = static_cast<int>(sizeof(table) / sizeof(table[0]));
    return table;
}

}  // namespace mpe

// =================================================================================================
// C ABI
// =================================================================================================
using namespace mpe;

namespace {
struct NvtxRange {   // RAII range around the C-ABI entry points (visible in nsys / ncu --nvtx)
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
}  // namespace

// largest block (in warps) whose warp-private staging fits the 227 KB of dynamic shared memory of an SM
static int max_warps_per_block(int smem_per_warp) {
    const int fit = (227 * 1024) / (smem_per_warp > 0 ? smem_per_warp : 1);
    return fit < 1 ? 1 : (fit > kMaxWarpsPerBlock ? kMaxWarpsPerBlock : fit);
}

// dynamic shared memory of a closed-loop rollout block: the actors of all agents once, one staging slot per warp;
// capped to what an SM offers (larger blocks are then never launched: policy_warps_per_block)
static int policy_smem_bytes(const Program *prog, int di, int k, int wpb) {
    const long long b = static_cast<long long>(prog->policy_weight_floats[di][k]) * 4 + static_cast<long long>(prog->smem_bytes) * wpb;
    return b < 227 * 1024 ? static_cast<int>(b) : 227 * 1024;
}

static_assert(sizeof(mpe_desc) == 480, "mpe_desc layout is part of the ABI (mirrored by _lib.MpeDesc)");

struct mpe_env {
    mpe_desc desc;
    DevDesc dev;
    Program custom;        // MPE_SCN_CUSTOM: the generic program with this handle's shapes
    const Program *prog;
    int64_t n;
    int device;
    // mpe_step_host pipelines chunks of the batch over two internal streams so that the H2D copy of one
    // chunk overlaps the D2H copy of the previous one (PCIe is full duplex)
    cudaStream_t aux[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    int policy2_wpb[2] = {0, 0};   // depth-2 closed-loop rollout: warps per block of most residency (0: not yet asked)
};

static thread_local char g_cuda_err[256] = "";
static long long g_launches = 0;

static int cuda_fail(cudaError_t e, const char *what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
    return MPE_ERR_CUDA;
}
#define CUDA_TRY(expr)                                     \
    do {                                                   \
        cudaError_t e_ = (expr);                           \
        if (e_ != cudaSuccess) return cuda_fail(e_, #expr); \
    } while (0)

extern "C" int mpe_create(const mpe_desc *desc, int64_t n_env, int device, mpe_handle *out) {
    if (!desc || !out || n_env <= 0) return MPE_ERR_BAD_ARG;
    if (desc->abi_version != MPE_ABI_VERSION) return MPE_ERR_BAD_DESC;
    if (desc->n_agents < 1 || desc->n_agents > MPE_MAX_AGENTS || desc->n_landmarks < 0 ||
        desc->n_landmarks > MPE_MAX_LANDMARKS)
        return MPE_ERR_BAD_DESC;
    int count = 0;
    const Program *tab = programs(&count);
    const Program *prog = nullptr;
    bool scenario_known = false;
    for (int i = 0; i < count; ++i) {
        if (tab[i].scenario != desc->scenario) continue;
        scenario_known = true;
        if (tab[i].validate(*desc)) { prog = &tab[i]; break; }
    }
    if (!prog) return scenario_known ? MPE_ERR_BAD_DESC : MPE_ERR_UNSUPPORTED;
    if (device != -1) {  // device == -1: shape-only handle (no CUDA call is made; launches are refused)
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return MPE_ERR_NO_DEVICE;
        int major = 0;
        CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
        if (major != 10) return MPE_ERR_NO_DEVICE;  // sm_100a cubin only
        int prev = 0;
        CUDA_TRY(cudaGetDevice(&prev));
        CUDA_TRY(cudaSetDevice(device));
        for (int m = 0; m < 4; ++m)
            if (prog->fn[m] && prog->smem_bytes > 0)
                CUDA_TRY(cudaFuncSetAttribute(prog->fn[m], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              prog->smem_bytes * max_warps_per_block(prog->smem_bytes)));
        if (prog->lanes_fn)
            CUDA_TRY(cudaFuncSetAttribute(prog->lanes_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, prog->lanes_smem * 4));
        if (prog->hot_fn && prog->smem_bytes > 0)
            CUDA_TRY(cudaFuncSetAttribute(prog->hot_fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          prog->smem_bytes * max_warps_per_block(prog->smem_bytes)));
        if (prog->hot_dense_fn && prog->smem_bytes > 0)
            CUDA_TRY(cudaFuncSetAttribute(prog->hot_dense_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, prog->smem_bytes * 4));
        if (prog->pipe_fn)
            CUDA_TRY(cudaFuncSetAttribute(prog->pipe_fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          prog->pipe_smem * max_warps_per_block(prog->pipe_smem)));
        for (int dk = 0; dk < 4; ++dk)
            if (prog->policy_fn[dk >> 1][dk & 1])
                CUDA_TRY(cudaFuncSetAttribute(prog->policy_fn[dk >> 1][dk & 1], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              policy_smem_bytes(prog, dk >> 1, dk & 1, dk < 2 ? kPolicyMaxWarps<1> : kPolicyMaxWarps<2>)));
        for (int k = 0; k < 2; ++k)
            if (prog->policy_plain_fn[k])
                CUDA_TRY(cudaFuncSetAttribute(prog->policy_plain_fn[k], cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              policy_smem_bytes(prog, 0, k, kPolicyMaxWarps<1>)));
        if (prog->rollout_fn)
            CUDA_TRY(cudaFuncSetAttribute(prog->rollout_fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          prog->rollout_smem * max_warps_per_block(prog->rollout_smem)));
        if (prog->split_fn && prog->smem_bytes > 0)
            CUDA_TRY(cudaFuncSetAttribute(prog->split_fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          prog->smem_bytes * max_warps_per_block(prog->smem_bytes)));
        CUDA_TRY(cudaSetDevice(prev));
    }

    mpe_env *h = new (std::nothrow) mpe_env();
    if (!h) return MPE_ERR_BAD_ARG;
    if (device != -1) {
        int prev = 0;
        cudaGetDevice(&prev);
        cudaSetDevice(device);
        cudaError_t e = cudaSuccess;
        for (int k = 0; k < 2 && e == cudaSuccess; ++k) {
            e = cudaStreamCreateWithFlags(&h->aux[k], cudaStreamNonBlocking);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join[k], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
        cudaSetDevice(prev);
        if (e != cudaSuccess) { delete h; return cuda_fail(e, "mpe_create: streams/events"); }
    }
    h->desc = *desc;
    h->prog = prog;
    if (desc->scenario == MPE_SCN_CUSTOM) {   // shapes of a user scenario come from its descriptor
        h->custom = *prog;
        Program &c = h->custom;
        c.A = desc->n_agents; c.L = desc->n_landmarks; c.DIMC = desc->dim_c; c.INFO = 0; c.G = 0; c.NS = 0;
        for (int i = 0; i < c.A; ++i) {
            c.NS += desc->agent_silent[i] ? 0 : 1;
            c.act_dim[i] = (desc->agent_movable[i] ? 5 : 0) + (desc->agent_silent[i] ? 0 : desc->dim_c);
            c.obs_dim[i] = 0;   // defined by the caller's observation code
        }
        h->prog = &h->custom;
    }
    h->n = n_env;
    h->device = device;
    DevDesc &d = h->dev;
    memset(&d, 0, sizeof(d));
    d.dt = static_cast<float>(desc->dt);
    d.keep = static_cast<float>(1.0 - desc->damping);
    d.contact_force = static_cast<float>(desc->contact_force);
    d.contact_margin = static_cast<float>(desc->contact_margin);
    d.inv_margin = static_cast<float>(1.0 / desc->contact_margin);
    for (int i = 0; i < desc->n_agents; ++i) {
        d.a_size[i] = static_cast<float>(desc->agent_size[i]);
        d.a_dt_over_mass[i] = static_cast<float>(desc->dt / desc->agent_mass[i]);
        d.a_sens[i] = static_cast<float>(desc->agent_sens[i]);
        d.a_max_speed[i] = desc->agent_max_speed[i] < 0 ? -1.0f : static_cast<float>(desc->agent_max_speed[i]);
    }
    for (int l = 0; l < desc->n_landmarks; ++l) d.l_size[l] = static_cast<float>(desc->landmark_size[l]);
    d.g_agents = desc->n_agents; d.g_landmarks = desc->n_landmarks; d.g_dim_c = desc->dim_c;
    int slot = 0;
    for (int i = 0; i < desc->n_agents; ++i) {
        if (desc->agent_movable[i]) d.g_movable |= 1u << i;
        if (desc->agent_collide[i]) d.g_collide |= 1u << i;
        if (desc->agent_silent[i]) d.g_silent |= 1u << i;
        d.g_slot[i] = desc->agent_silent[i] ? static_cast<int8_t>(-1) : static_cast<int8_t>(slot++);
    }
    for (int l = 0; l < desc->n_landmarks; ++l)
        if (desc->landmark_collide[l]) d.g_lcollide |= 1u << l;
    d.g_comm_rows = slot * desc->dim_c;
    *out = h;
    return MPE_OK;
}

extern "C" int mpe_destroy(mpe_handle h) {
    if (!h) return MPE_ERR_BAD_ARG;
    for (int k = 0; k < 2; ++k) {
        if (h->aux[k]) cudaStreamDestroy(h->aux[k]);
        if (h->ev_join[k]) cudaEventDestroy(h->ev_join[k]);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    delete h;
    return MPE_OK;
}

extern "C" int mpe_num_agents(mpe_handle h) { return h ? h->prog->A : MPE_ERR_BAD_ARG; }
extern "C" int64_t mpe_num_envs(mpe_handle h) { return h ? h->n : static_cast<int64_t>(MPE_ERR_BAD_ARG); }
extern "C" int mpe_obs_dim(mpe_handle h, int i) {
    if (!h || i < 0 || i >= h->prog->A) return MPE_ERR_BAD_ARG;
    return h->prog->scenario == MPE_SCN_CUSTOM ? MPE_ERR_UNSUPPORTED : h->prog->obs_dim[i];
}
extern "C" int mpe_act_dim(mpe_handle h, int i) { return (h && i >= 0 && i < h->prog->A) ? h->prog->act_dim[i] : MPE_ERR_BAD_ARG; }
extern "C" int mpe_num_speakers(mpe_handle h) { return h ? h->prog->NS : MPE_ERR_BAD_ARG; }
extern "C" int mpe_num_goals(mpe_handle h) { return h ? h->prog->G : MPE_ERR_BAD_ARG; }
extern "C" int mpe_info_dim(mpe_handle h) { return h ? h->prog->INFO : MPE_ERR_BAD_ARG; }

extern "C" int64_t mpe_bytes_per_env_step(mpe_handle h) {
    if (!h) return MPE_ERR_BAD_ARG;
    // SURVEY.md 8(d): read agent pos+vel, landmark pos, goal indices, actions; write pos+vel of the movable
    // agents, observations, rewards, speaker comm state, 1 done byte per agent
    const Program *p = h->prog;
    int64_t f = 4 * p->A + 2 * p->L + p->G + p->A + p->NS * p->DIMC - p->unread_state_floats;
    for (int i = 0; i < p->A; ++i) f += p->act_dim[i] + p->obs_dim[i] + (h->desc.agent_movable[i] ? 4 : 0);
    return 4 * f + p->A;
}

constexpr int64_t kLanesMaxWorlds = 0;  // set from measurements (see profiles/)

// Programmatic dependent launch between consecutive step kernels.  MPE_B200_PDL: 0 = off, 1 = release the next grid
// before our stores, 2 = at entry, 3 = once our inputs have arrived (DEFAULT: measured best, 5.88 vs 6.56 us per step at
// 65536 worlds), 4 = implicitly at exit, 5 = as soon as our loads are issued
static int pdl_mode() {
    static const int m = [] { const char *e = getenv("MPE_B200_PDL"); return (e && e[0] >= '0' && e[0] <= '5') ? e[0] - '0' : 3; }();
    return m;
}

static int launch(mpe_handle h, int mode, StepArgs &args, void *stream, int64_t begin = 0, int64_t count = -1) {
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    args.d = h->dev;
    args.n = h->n;
    args.begin = begin;
    args.count = count < 0 ? h->n - begin : count;
    // simple_spread fused steps may run on the lane-per-agent kernel (mpe_spread_lanes.cuh): MPE_B200_SPREAD_LANES
    // = 0 never, 1 always, unset: up to kLanesMaxWorlds worlds, where the lane-per-world kernel has too few warps
    static const int lanes_env = [] { const char *e = getenv("MPE_B200_SPREAD_LANES"); return e ? atoi(e) : -1; }();
    const bool lanes = mode == kFusedStep && h->prog->lanes_fn != nullptr &&
                       (lanes_env == 1 || (lanes_env < 0 && args.count <= kLanesMaxWorlds));
    if (lanes) {
        const int64_t lw = (args.count + h->prog->lanes_wpw - 1) / h->prog->lanes_wpw;
        constexpr int kLanesWpb = 4;
        const int64_t lb = (lw + kLanesWpb - 1) / kLanesWpb;
        int prev = 0;
        CUDA_TRY(cudaGetDevice(&prev));
        if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
        void *params[] = {&args};
        cudaError_t e = cudaLaunchKernel(reinterpret_cast<const void *>(h->prog->lanes_fn), dim3(static_cast<unsigned>(lb)),
                                         dim3(32 * kLanesWpb), params, static_cast<size_t>(h->prog->lanes_smem) * kLanesWpb,
                                         static_cast<cudaStream_t>(stream));
        if (prev != h->device) cudaSetDevice(prev);
        if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernel(spread_lanes)");
        __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
        return MPE_OK;
    }
    if (h->prog->scenario == MPE_SCN_CUSTOM) {   // generic program: one thread per world, no staging
        if (h->prog->fn[mode] == nullptr) return MPE_ERR_UNSUPPORTED;
        int prev = 0;
        CUDA_TRY(cudaGetDevice(&prev));
        if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
        void *params[] = {&args};
        cudaError_t e = cudaLaunchKernel(reinterpret_cast<const void *>(h->prog->fn[mode]),
                                         dim3(static_cast<unsigned>((args.count + 127) / 128)), dim3(128), params, 0,
                                         static_cast<cudaStream_t>(stream));
        if (prev != h->device) cudaSetDevice(prev);
        if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernel(generic)");
        __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
        return MPE_OK;
    }
    // Software-pipelined persistent kernel (mpe_pipe_kernel): MPE_B200_PIPE=1, MPE_B200_PIPE_TPW tiles per warp (default 2)
    static const int pipe_env = [] { const char *e = getenv("MPE_B200_PIPE"); return e ? atoi(e) : 0; }();
    static const int pipe_tpw = [] { const char *e = getenv("MPE_B200_PIPE_TPW"); int v = e ? atoi(e) : 2; return v < 1 ? 1 : v; }();
    if (pipe_env == 1 && mode == kFusedStep && h->prog->pipe_fn != nullptr && args.count >= 32 &&
        !(args.flags & MPE_FLAG_DISCRETE_ACTION_INPUT)) {
        bool aligned = true;
        for (int i = 0; i < h->prog->A; ++i)
            aligned = aligned && ((reinterpret_cast<uintptr_t>(args.act[i]) + static_cast<uintptr_t>(begin) * h->prog->act_dim[i] * 4) & 15u) == 0;
        if (aligned && (begin % 32) == 0 && (h->n % 4) == 0) {
            const int64_t tiles = args.count / 32, tail = args.count - tiles * 32;
            static const int pwpb_env = [] { const char *e = getenv("MPE_B200_WPB"); int v = e ? atoi(e) : 0; return (v >= 1 && v <= kMaxWarpsPerBlock) ? v : 0; }();
            int pwpb = pwpb_env ? pwpb_env : 2;
            if (pwpb > max_warps_per_block(h->prog->pipe_smem)) pwpb = max_warps_per_block(h->prog->pipe_smem);
            const int64_t pwarps = (tiles + pipe_tpw - 1) / pipe_tpw;
            const int64_t pblocks = (pwarps + pwpb - 1) / pwpb;
            int prev = 0;
            CUDA_TRY(cudaGetDevice(&prev));
            if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(static_cast<unsigned>(pblocks));
            cfg.blockDim = dim3(32 * pwpb);
            cfg.dynamicSmemBytes = static_cast<size_t>(h->prog->pipe_smem) * pwpb;
            cfg.stream = static_cast<cudaStream_t>(stream);
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr;
            cfg.numAttrs = pdl_mode() ? 1 : 0;
            StepArgs pa = args;
            pa.count = tiles * 32;
            if (pdl_mode() == 3) pa.flags |= kFlagPdlAfterLoads;
            void *params[] = {&pa};
            cudaError_t e = cudaLaunchKernelExC(&cfg, reinterpret_cast<const void *>(h->prog->pipe_fn), params);
            if (prev != h->device) cudaSetDevice(prev);
            if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernelExC(pipe)");
            __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
            if (tail == 0) return MPE_OK;
            args.begin = begin + tiles * 32;      // the ragged tail goes through the regular kernel below
            args.count = tail;
        }
    }
    int64_t warps = (args.count + 31) / 32;
    // Warp pairs (see mpe_kernel<..., SPLIT>): MPE_B200_SPLIT = 1 always, 2 = for small batches of >= 4-agent scenarios,
    // unset / 0 never.  MEASURED SLOWER than one warp per tile at every size but 8192 worlds (profiles/r2a_sweep_split*:
    // world_comm 32768 worlds 15.2 vs 11.2 us, spread 65536 worlds 9.8 vs 5.8 us): the duplicated physics + reward cost
    // more than the extra warps hide.  Kept as an opt-in, bit-identical alternative.
    static const int split_env = [] { const char *e = getenv("MPE_B200_SPLIT"); return e ? atoi(e) : -1; }();
    static const int64_t split_max_warps = [] { const char *e = getenv("MPE_B200_SPLIT_MAX_WARPS"); return e ? atoll(e) : 148LL * 10; }();
    const bool split = mode == kFusedStep && h->prog->split_fn != nullptr &&
                       (split_env == 1 || (split_env == 2 && h->prog->A >= 4 && warps <= split_max_warps));
    if (split) warps *= 2;
    static const int wpb_env = [] { const char *e = getenv("MPE_B200_WPB"); int v = e ? atoi(e) : 0; return (v >= 1 && v <= kMaxWarpsPerBlock) ? v : 0; }();
    // action tiles: cp.async (LDGSTS) by default -- measured 1-5 % faster than the TMA bulk copy + mbarrier at every
    // batch size (no barrier init / proxy fence in the prologue); MPE_B200_ACT_STAGING=tma selects the TMA path
    static const bool cpasync = [] { const char *e = getenv("MPE_B200_ACT_STAGING"); return !(e && e[0] == 't'); }();
    static const bool hot_env = [] { const char *e = getenv("MPE_B200_HOT"); return !(e && e[0] == '0'); }();   // 0 = general kernel only
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
    if (pdl_mode() == 2) args.flags |= kFlagPdlEarly;
    if (pdl_mode() == 3) args.flags |= kFlagPdlAfterLoads;
    if (pdl_mode() == 4) args.flags |= kFlagPdlAtExit;
    if (pdl_mode() == 5) args.flags |= kFlagPdlAfterIssue;
    if (cpasync) args.flags |= kFlagCpAsync;
    // one grid of autonomous warps over [sa.begin, sa.begin + sa.count)
    auto launch_grid = [&](KernelFn fn, StepArgs &sa, bool pairs, int max_wpb = kMaxWarpsPerBlock) -> int {
        int64_t nw = (sa.count + 31) / 32;
        if (pairs) nw *= 2;
        // Warps are autonomous, so the block size only sets scheduling granularity.  While every warp of the batch is
        // resident at once (<= 16 per SM) one warp per block balances the SMs best (world_comm, 32 768 worlds = 6.9
        // warps per SM: 9.03 vs 9.60 us with two; spread N=3 and tag at 65 536 worlds: 1 and 2 tie, 4 loses 10 %,
        // profiles/r2f_geometry_*, r2j_*); mid-size batches use two, large ones four.
        int wpb = wpb_env ? wpb_env : (nw <= 148 * 16 ? 1 : (nw <= 148 * 64 ? 2 : 4));
        if (wpb > max_warps_per_block(h->prog->smem_bytes)) wpb = max_warps_per_block(h->prog->smem_bytes);
        if (wpb > max_wpb) wpb = max_wpb;
        if (pairs) wpb = (wpb < 2) ? 2 : (wpb & ~1);      // a pair lives in one block
        const int64_t blocks = (nw + wpb - 1) / wpb;
        if (blocks > 0x7fffffffLL) return MPE_ERR_BAD_ARG;
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(static_cast<unsigned>(blocks));
        cfg.blockDim = dim3(32 * wpb);
        cfg.dynamicSmemBytes = static_cast<size_t>(h->prog->smem_bytes) * wpb;
        cfg.stream = static_cast<cudaStream_t>(stream);
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = pdl_mode() ? 1 : 0;
        void *params[] = {&sa};
        cudaError_t e = cudaLaunchKernelExC(&cfg, reinterpret_cast<const void *>(fn), params);
        if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernelExC");
        __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
        return MPE_OK;
    };
    int rc = MPE_OK;
    // the specialised fused step (mpe_kernel<..., HOT>) takes every whole tile it is eligible for
    bool hot = hot_env && cpasync && !split && mode == kFusedStep && h->prog->hot_fn != nullptr && args.count >= 32 &&
               !(args.flags & (MPE_FLAG_DISCRETE_ACTION_INPUT | MPE_FLAG_FORCE_DISCRETE_ACTION));
    for (int i = 0; hot && i < h->prog->A; ++i)
        hot = ((reinterpret_cast<uintptr_t>(args.act[i]) + static_cast<uintptr_t>(args.begin) * h->prog->act_dim[i] * 4) & 15u) == 0;
    if (hot) {
        StepArgs ha = args;
        ha.count = args.count / 32 * 32;
        // more tiles than the 128-register kernel keeps resident (16 warps per SM): the 80-register build, if there is one
        static const int dense_env = [] { const char *e = getenv("MPE_B200_DENSE"); return e ? atoi(e) : -1; }();   // 0 never, 1 always
        const bool dense = h->prog->hot_dense_fn != nullptr &&
                           (dense_env == 1 || (dense_env < 0 && ha.count / 32 > 148LL * 16));
        rc = dense ? launch_grid(h->prog->hot_dense_fn, ha, false, 4) : launch_grid(h->prog->hot_fn, ha, false);
        args.begin += ha.count;
        args.count -= ha.count;
    }
    if (rc == MPE_OK && args.count > 0) rc = launch_grid(split ? h->prog->split_fn : h->prog->fn[mode], args, split);
    if (prev != h->device) cudaSetDevice(prev);
    return rc;
}

static bool ok16(const void *p) { return p != nullptr && (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static bool ok8(const void *p) { return p != nullptr && (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }
static bool ok4(const void *p) { return p != nullptr && (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

static int fill_state(mpe_handle h, StepArgs &a, void *pv, const void *lm, float *comm, const int32_t *goal,
                      bool need_goal = true) {
    const Program *p = h->prog;
    if (!ok16(pv)) return MPE_ERR_BAD_ARG;
    if (p->L > 0 && !ok8(lm)) return MPE_ERR_BAD_ARG;
    if (p->NS * p->DIMC > 0 && !ok4(comm)) return MPE_ERR_BAD_ARG;
    if (need_goal && p->G > 0 && !ok4(goal)) return MPE_ERR_BAD_ARG;
    a.pv = static_cast<float4 *>(pv);
    a.lm = static_cast<const float2 *>(lm);
    a.comm = comm;
    a.goal = goal;
    return MPE_OK;
}

static int fill_outputs(mpe_handle h, StepArgs &a, float *const *obs_n, float *rew, uint8_t *done, float *info) {
    const Program *p = h->prog;
    if (!obs_n || !ok4(rew) || !done) return MPE_ERR_BAD_ARG;
    for (int i = 0; i < p->A; ++i) {
        if (!ok16(obs_n[i])) return MPE_ERR_BAD_ARG;   // observation rows are written as 16-byte stores
        a.obs[i] = obs_n[i];
    }
    a.rew = rew;
    a.done = done;
    a.info = p->INFO > 0 ? info : nullptr;
    return MPE_OK;
}

static int fill_actions(mpe_handle h, StepArgs &a, const float *const *act_n) {
    if (!act_n) return MPE_ERR_BAD_ARG;
    for (int i = 0; i < h->prog->A; ++i) {
        if (!ok4(act_n[i])) return MPE_ERR_BAD_ARG;
        a.act[i] = act_n[i];
    }
    return MPE_OK;
}

extern "C" int mpe_set_action(mpe_handle h, const float *const *act_n, float *u, float *c, uint32_t flags, void *stream) {
    if (!h || !ok8(u)) return MPE_ERR_BAD_ARG;
    if (h->prog->NS * h->prog->DIMC > 0 && !ok4(c)) return MPE_ERR_BAD_ARG;
    StepArgs a{};
    int r = fill_actions(h, a, act_n);
    if (r) return r;
    a.u = reinterpret_cast<float2 *>(u);
    a.c = c;
    a.flags = flags;
    return launch(h, kSetAction, a, stream);
}

extern "C" int mpe_world_step(mpe_handle h, void *pv, const void *lm, float *comm, const float *u, const float *c, void *stream) {
    if (!h || !ok8(u)) return MPE_ERR_BAD_ARG;
    if (h->prog->NS * h->prog->DIMC > 0 && !ok4(c)) return MPE_ERR_BAD_ARG;
    StepArgs a{};
    int r = fill_state(h, a, pv, lm, comm, nullptr, false);
    if (r) return r;
    a.u = reinterpret_cast<float2 *>(const_cast<float *>(u));
    a.c = const_cast<float *>(c);
    return launch(h, kWorldStep, a, stream);
}

extern "C" int mpe_observe(mpe_handle h, const void *pv, const void *lm, const float *comm, const int32_t *goal,
                           float *const *obs_n, float *rew, uint8_t *done, float *info, uint32_t flags, void *stream) {
    if (!h) return MPE_ERR_BAD_ARG;
    if (h->prog->scenario == MPE_SCN_CUSTOM) return MPE_ERR_UNSUPPORTED;
    StepArgs a{};
    int r = fill_state(h, a, const_cast<void *>(pv), lm, const_cast<float *>(comm), goal);
    if (r) return r;
    r = fill_outputs(h, a, obs_n, rew, done, info);
    if (r) return r;
    a.flags = flags;
    return launch(h, kObserve, a, stream);
}

extern "C" int mpe_step(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal,
                        const float *const *act_n, float *const *obs_n, float *rew, uint8_t *done, float *info,
                        uint32_t flags, void *stream) {
    if (!h) return MPE_ERR_BAD_ARG;
    NvtxRange range("mpe_step");
    StepArgs a{};
    int r = fill_state(h, a, pv, lm, comm, goal);
    if (r) return r;
    r = fill_actions(h, a, act_n);
    if (r) return r;
    r = fill_outputs(h, a, obs_n, rew, done, info);
    if (r) return r;
    a.flags = flags;
    return launch(h, kFusedStep, a, stream);
}

extern "C" int mpe_rollout(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal,
                           const float *const *act_seq, int32_t n_steps, float *const *obs_n, float *rew_sum,
                           float *rew_steps, uint8_t *done, uint32_t flags, void *stream) {
    if (!h || n_steps < 0) return MPE_ERR_BAD_ARG;
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    if (h->prog->scenario == MPE_SCN_CUSTOM || h->prog->rollout_fn == nullptr) return MPE_ERR_UNSUPPORTED;
    if (flags & MPE_FLAG_DISCRETE_ACTION_INPUT) return MPE_ERR_UNSUPPORTED;
    if (rew_steps != nullptr && !ok4(rew_steps)) return MPE_ERR_BAD_ARG;
    NvtxRange range("mpe_rollout");
    RolloutArgs ra{};
    StepArgs &a = ra.s;
    int r = fill_state(h, a, pv, lm, comm, goal);
    if (r) return r;
    r = fill_actions(h, a, act_seq);
    if (r) return r;
    r = fill_outputs(h, a, obs_n, rew_sum, done, nullptr);
    if (r) return r;
    a.info = nullptr;
    a.flags = flags;
    a.d = h->dev;
    a.n = h->n;
    a.begin = 0;
    a.count = h->n;
    ra.T = n_steps;
    ra.rew_steps = rew_steps;
    const int64_t warps = (h->n + 31) / 32;
    int wpb = warps <= 148 * 4 ? 1 : (warps <= 148 * 64 ? 2 : 4);
    if (wpb > max_warps_per_block(h->prog->rollout_smem)) wpb = max_warps_per_block(h->prog->rollout_smem);
    const int64_t blocks = (warps + wpb - 1) / wpb;
    if (blocks > 0x7fffffffLL) return MPE_ERR_BAD_ARG;
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
    void *params[] = {&ra};
    cudaError_t e = cudaLaunchKernel(reinterpret_cast<const void *>(h->prog->rollout_fn), dim3(static_cast<unsigned>(blocks)),
                                     dim3(32 * wpb), params, static_cast<size_t>(h->prog->rollout_smem) * wpb,
                                     static_cast<cudaStream_t>(stream));
    if (prev != h->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernel(rollout)");
    __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
    return MPE_OK;
}

// Depth 1 keeps its original block sizes.  Depth 2 stages 70-92 KB of weights per block (H = 64), so one-warp blocks
// would leave an SM 2-3 warps: it takes the block size of 1-8 warps with the most resident warps per SM (registers and
// shared memory, from the occupancy calculator; the smaller on ties), and small batches shrink it until every SM has a
// block.
static int policy_warps_per_block(mpe_handle h, int di, int k, int64_t warps) {
    if (di == 0) return warps <= 148 * 16 ? 1 : (warps <= 148 * 64 ? 2 : 4);
    int &best = h->policy2_wpb[k];
    if (best == 0) {
        int most = 0;
        best = 1;
        for (int wpb = 1; wpb <= kPolicyMaxWarps<2>; ++wpb) {
            const long long smem = static_cast<long long>(h->prog->policy_weight_floats[di][k]) * 4 +
                                   static_cast<long long>(h->prog->smem_bytes) * wpb;
            if (smem > 227 * 1024) break;
            int blocks = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, h->prog->policy_fn[di][k], 32 * wpb,
                                                              static_cast<size_t>(smem)) != cudaSuccess)
                break;
            if (blocks * wpb > most) { most = blocks * wpb; best = wpb; }
        }
    }
    int wpb = best;
    if (warps < 148LL * wpb) wpb = warps >= 148 ? static_cast<int>(warps / 148) : 1;
    return wpb;
}

extern "C" int mpe_collect_supported(mpe_handle h, int32_t depth, int32_t hidden) {
    if (!h || (depth != 1 && depth != 2) || (hidden != 32 && hidden != 64)) return MPE_ERR_BAD_ARG;
    const bool built = h->prog->scenario != MPE_SCN_CUSTOM && h->prog->policy_fn[depth - 1][hidden == 32 ? 0 : 1] != nullptr;
    return built ? MPE_OK : MPE_ERR_UNSUPPORTED;
}

extern "C" int mpe_collect(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal, int32_t depth,
                           int32_t hidden, const float *const *w1_n, const float *const *b1_n, const float *const *w2_n,
                           const float *const *b2_n, const float *const *w3_n, const float *const *b3_n, int32_t n_steps,
                           uint64_t sample_seed, uint32_t sample_step, uint64_t world_offset, float *const *obs_n,
                           float *rew_sum, float *rew_steps, float *const *act_record_n, float *const *obs_record_n,
                           uint8_t *done, uint32_t flags, void *stream) {
    if (!h || n_steps < 0 || !w1_n || !b1_n || !w2_n || !b2_n) return MPE_ERR_BAD_ARG;
    if ((depth != 1 && depth != 2) || (hidden != 32 && hidden != 64)) return MPE_ERR_BAD_ARG;
    if ((depth == 2) != (w3_n != nullptr) || (depth == 2) != (b3_n != nullptr)) return MPE_ERR_BAD_ARG;
    if (static_cast<uint64_t>(sample_step) + static_cast<uint64_t>(n_steps) > (1ull << 32)) return MPE_ERR_BAD_ARG;
    if (rew_steps != nullptr && !ok4(rew_steps)) return MPE_ERR_BAD_ARG;
    const int A = h->prog->A;
    for (int i = 0; i < A; ++i) {
        if (!ok16(w1_n[i]) || !ok16(b1_n[i]) || !ok16(w2_n[i]) || !ok4(b2_n[i])) return MPE_ERR_BAD_ARG;
        if (depth == 2 && (!ok16(w3_n[i]) || !ok4(b3_n[i]))) return MPE_ERR_BAD_ARG;
        if (act_record_n && act_record_n[i] != nullptr && !ok4(act_record_n[i])) return MPE_ERR_BAD_ARG;
        if (obs_record_n && !ok16(obs_record_n[i])) return MPE_ERR_BAD_ARG;
    }
    if (h->prog->NS * h->prog->DIMC > 0 && !ok4(comm)) return MPE_ERR_BAD_ARG;
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    const int di = depth - 1, k = hidden == 32 ? 0 : 1;
    if (mpe_collect_supported(h, depth, hidden) != MPE_OK) return MPE_ERR_UNSUPPORTED;
    if (flags & (MPE_FLAG_DISCRETE_ACTION_INPUT | MPE_FLAG_FORCE_DISCRETE_ACTION)) return MPE_ERR_UNSUPPORTED;
    NvtxRange range("mpe_collect");
    PolicyArgs pa{};
    StepArgs &a = pa.s;
    int r = fill_state(h, a, pv, lm, comm, goal);
    if (r) return r;
    r = fill_outputs(h, a, obs_n, rew_sum, done, nullptr);
    if (r) return r;
    for (int i = 0; i < A; ++i) {
        pa.w1[i] = w1_n[i]; pa.b1[i] = b1_n[i]; pa.w2[i] = w2_n[i]; pa.b2[i] = b2_n[i];
        pa.w3[i] = depth == 2 ? w3_n[i] : nullptr;
        pa.b3[i] = depth == 2 ? b3_n[i] : nullptr;
        pa.act_rec[i] = act_record_n ? act_record_n[i] : nullptr;
        pa.obs_rec[i] = obs_record_n ? obs_record_n[i] : nullptr;
    }
    a.info = nullptr;
    a.flags = flags;
    a.d = h->dev;
    a.n = h->n;
    a.begin = 0;
    a.count = h->n;
    pa.T = n_steps;
    pa.rew_steps = rew_steps;
    pa.sample_key = make_uint2(static_cast<uint32_t>(sample_seed), static_cast<uint32_t>(sample_seed >> 32));
    pa.world_offset = world_offset;
    pa.sample_step = sample_step;
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
    const int64_t warps = (h->n + 31) / 32;
    const int wpb = policy_warps_per_block(h, di, k, warps);
    const int64_t blocks = (warps + wpb - 1) / wpb;
    cudaError_t e = cudaErrorInvalidValue;
    if (blocks <= 0x7fffffffLL) {
        void *params[] = {&pa};
        const bool plain = depth == 1 && !(flags & MPE_FLAG_SAMPLE_ACTIONS) && obs_record_n == nullptr &&
                           h->prog->policy_plain_fn[k] != nullptr;
        e = cudaLaunchKernel(reinterpret_cast<const void *>(plain ? h->prog->policy_plain_fn[k] : h->prog->policy_fn[di][k]),
                             dim3(static_cast<unsigned>(blocks)),
                             dim3(32 * wpb), params, static_cast<size_t>(policy_smem_bytes(h->prog, di, k, wpb)),
                             static_cast<cudaStream_t>(stream));
    }
    if (prev != h->device) cudaSetDevice(prev);
    if (blocks > 0x7fffffffLL) return MPE_ERR_BAD_ARG;
    if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernel(collect)");
    __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
    return MPE_OK;
}

extern "C" int mpe_rollout_policy(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal,
                                  const float *const *w1_n, const float *const *b1_n, const float *const *w2_n,
                                  const float *const *b2_n, int32_t hidden, int32_t n_steps, float *const *obs_n,
                                  float *rew_sum, float *rew_steps, float *const *act_record_n, uint8_t *done,
                                  uint32_t flags, void *stream) {
    if (!h || n_steps < 0 || !w1_n || !b1_n || !w2_n || !b2_n) return MPE_ERR_BAD_ARG;
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    const int k = hidden == 32 ? 0 : (hidden == 64 ? 1 : -1);
    if (k < 0 || mpe_collect_supported(h, 1, hidden) != MPE_OK || !h->prog->policy_move_only) return MPE_ERR_UNSUPPORTED;
    return mpe_collect(h, pv, lm, comm, goal, 1, hidden, w1_n, b1_n, w2_n, b2_n, nullptr, nullptr, n_steps, 0, 0, 0,
                       obs_n, rew_sum, rew_steps, act_record_n, nullptr, done, flags & ~MPE_FLAG_SAMPLE_ACTIONS, stream);
}

// adjacent (dst, src, bytes) copies with equal small gaps on both sides are issued as one DMA
struct CopySeg { char *dst; const char *src; size_t bytes; };
static int issue_copies(CopySeg *seg, int n, cudaMemcpyKind kind, cudaStream_t s, const char *what, bool coalesce) {
    int i = 0;
    while (i < n) {
        CopySeg cur = seg[i++];
        while (coalesce && i < n) {
            const ptrdiff_t gd = seg[i].dst - (cur.dst + cur.bytes), gs = seg[i].src - (cur.src + cur.bytes);
            if (gd != gs || gd < 0 || gd >= 512) break;
            cur.bytes += static_cast<size_t>(gd) + seg[i].bytes;
            ++i;
        }
        cudaError_t e = cudaMemcpyAsync(cur.dst, cur.src, cur.bytes, kind, s);
        if (e != cudaSuccess) return cuda_fail(e, what);
    }
    return MPE_OK;
}

static int step_range(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal,
                      const float *const *act_n, float *const *obs_n, float *rew, uint8_t *done, float *info,
                      uint32_t flags, void *stream, int64_t begin, int64_t count) {
    if (h->prog->scenario == MPE_SCN_CUSTOM) return MPE_ERR_UNSUPPORTED;
    StepArgs a{};
    int r = fill_state(h, a, pv, lm, comm, goal);
    if (r) return r;
    r = fill_actions(h, a, act_n);
    if (r) return r;
    r = fill_outputs(h, a, obs_n, rew, done, info);
    if (r) return r;
    a.flags = flags;
    return launch(h, kFusedStep, a, stream, begin, count);
}

// floats (4-byte words) per world in act_n[i]: the action vector, or one index per sub-action (discrete_action_input)
static size_t act_row_words(const mpe_env *h, int i, uint32_t flags) {
    if (flags & MPE_FLAG_DISCRETE_ACTION_INPUT) return (h->desc.agent_movable[i] ? 1 : 0) + (h->desc.agent_silent[i] ? 0 : 1);
    return static_cast<size_t>(h->prog->act_dim[i]);
}

static int64_t host_chunk_min() {  // MPE_B200_HOST_CHUNK_MIN: smallest batch that is pipelined (default 262144)
    static const int64_t m = [] { const char *e = getenv("MPE_B200_HOST_CHUNK_MIN"); return e ? atoll(e) : 262144LL; }();
    return m;
}
static int host_chunks() {  // MPE_B200_HOST_CHUNKS: 1 disables the pipeline (default 4)
    static const int c = [] { const char *e = getenv("MPE_B200_HOST_CHUNKS"); int v = e ? atoi(e) : 4; return v < 1 ? 1 : (v > 16 ? 16 : v); }();
    return c;
}

extern "C" int mpe_step_host(mpe_handle h, void *pv, const void *lm, float *comm, const int32_t *goal,
                             const float *const *act_n_host, float *const *act_n_dev, float *const *obs_n_dev,
                             float *rew_dev, uint8_t *done_dev, float *info_dev, float *const *obs_n_host,
                             float *rew_host, uint8_t *done_host, float *info_host, uint32_t flags, void *stream) {
    if (!h || !act_n_host || !act_n_dev || !obs_n_host || !obs_n_dev || !rew_host || !done_host) return MPE_ERR_BAD_ARG;
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    NvtxRange range("mpe_step_host");
    const Program *p = h->prog;
    cudaStream_t user = static_cast<cudaStream_t>(stream);
    const size_t n = static_cast<size_t>(h->n);
    for (int i = 0; i < p->A; ++i)
        if (!act_n_host[i] || !act_n_dev[i] || !obs_n_host[i] || !obs_n_dev[i]) return MPE_ERR_BAD_ARG;
    const bool want_info = info_host && info_dev && p->INFO > 0;
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
    int rc = MPE_OK;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(user, &cap);
    // measured on B200 (PCIe Gen5): below ~256k worlds the extra copy calls cost more than the overlap gains
    const int chunks = (h->n >= host_chunk_min() && cap == cudaStreamCaptureStatusNone) ? host_chunks() : 1;
    if (chunks == 1) {
        // small batches: one H2D per agent, one launch, one coalesced D2H
        CopySeg seg[kMaxA + 3];
        int ns = 0;
        for (int i = 0; i < p->A; ++i)
            seg[ns++] = {reinterpret_cast<char *>(act_n_dev[i]), reinterpret_cast<const char *>(act_n_host[i]),
                         sizeof(float) * n * act_row_words(h, i, flags)};
        rc = issue_copies(seg, ns, cudaMemcpyHostToDevice, user, "cudaMemcpyAsync(H2D actions)", false);
        if (rc == MPE_OK)
            rc = step_range(h, pv, lm, comm, goal, act_n_dev, obs_n_dev, rew_dev, done_dev, want_info ? info_dev : nullptr,
                            flags, stream, 0, h->n);
        if (rc == MPE_OK) {
            ns = 0;
            for (int i = 0; i < p->A; ++i)
                seg[ns++] = {reinterpret_cast<char *>(obs_n_host[i]), reinterpret_cast<const char *>(obs_n_dev[i]),
                             sizeof(float) * n * p->obs_dim[i]};
            seg[ns++] = {reinterpret_cast<char *>(rew_host), reinterpret_cast<const char *>(rew_dev), sizeof(float) * n * p->A};
            seg[ns++] = {reinterpret_cast<char *>(done_host), reinterpret_cast<const char *>(done_dev), n * p->A};
            if (want_info)
                seg[ns++] = {reinterpret_cast<char *>(info_host), reinterpret_cast<const char *>(info_dev),
                             sizeof(float) * n * p->A * p->INFO};
            rc = issue_copies(seg, ns, cudaMemcpyDeviceToHost, user, "cudaMemcpyAsync(D2H obs/rew/done/info)",
                              (flags & MPE_FLAG_HOST_SLAB) != 0);
        }
    } else {
        // Large batches: the worlds are cut into `chunks` ranges (multiples of 128 worlds, so every tile stays
        // 16-byte aligned) that alternate between two internal streams: while chunk c drains over the D2H copy
        // engine, chunk c+1 uploads its actions and computes.  The caller's stream forks into and joins the two.
        cudaError_t e = cudaEventRecord(h->ev_fork, user);
        for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaStreamWaitEvent(h->aux[k], h->ev_fork, 0);
        if (e != cudaSuccess) rc = cuda_fail(e, "mpe_step_host: fork");
        const int64_t per = ((h->n + chunks - 1) / chunks + 127) / 128 * 128;
        for (int c = 0; c < chunks && rc == MPE_OK; ++c) {
            const int64_t begin = c * per;
            if (begin >= h->n) break;
            const int64_t count = (begin + per <= h->n) ? per : h->n - begin;
            cudaStream_t s = h->aux[c & 1];
            for (int i = 0; i < p->A && e == cudaSuccess; ++i)
                e = cudaMemcpyAsync(act_n_dev[i] + begin * act_row_words(h, i, flags), act_n_host[i] + begin * act_row_words(h, i, flags),
                                    sizeof(float) * count * act_row_words(h, i, flags), cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync(H2D actions)"); break; }
            rc = step_range(h, pv, lm, comm, goal, act_n_dev, obs_n_dev, rew_dev, done_dev, want_info ? info_dev : nullptr,
                            flags, s, begin, count);
            if (rc != MPE_OK) break;
            for (int i = 0; i < p->A && e == cudaSuccess; ++i)
                e = cudaMemcpyAsync(obs_n_host[i] + begin * p->obs_dim[i], obs_n_dev[i] + begin * p->obs_dim[i],
                                    sizeof(float) * count * p->obs_dim[i], cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess)   // rew / done / info are [rows][n_env]: one strided copy per array
                e = cudaMemcpy2DAsync(rew_host + begin, sizeof(float) * n, rew_dev + begin, sizeof(float) * n,
                                      sizeof(float) * count, p->A, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess)
                e = cudaMemcpy2DAsync(done_host + begin, n, done_dev + begin, n, count, p->A, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess && want_info)
                e = cudaMemcpy2DAsync(info_host + begin, sizeof(float) * n, info_dev + begin, sizeof(float) * n,
                                      sizeof(float) * count, static_cast<size_t>(p->A) * p->INFO, cudaMemcpyDeviceToHost, s);
            if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync(D2H chunk)");
        }
        for (int k = 0; k < 2; ++k) {   // join, even after an error, so that the caller's stream stays ordered
            cudaError_t j = cudaEventRecord(h->ev_join[k], h->aux[k]);
            if (j == cudaSuccess) j = cudaStreamWaitEvent(user, h->ev_join[k], 0);
            if (j != cudaSuccess && rc == MPE_OK) rc = cuda_fail(j, "mpe_step_host: join");
        }
    }
    if (prev != h->device) cudaSetDevice(prev);
    return rc;
}

static int reset_impl(mpe_handle h, void *pv, void *lm, float *comm, int32_t *goal, const uint8_t *mask,
                      uint64_t seed, uint64_t world_offset, uint64_t epoch, unsigned long long *epoch_dev, void *stream) {
    if (!h) return MPE_ERR_BAD_ARG;
    if (h->device < 0) return MPE_ERR_NO_DEVICE;
    NvtxRange range("mpe_reset");
    StepArgs tmp{};
    int r = fill_state(h, tmp, pv, lm, comm, goal);
    if (r) return r;
    const Program *p = h->prog;
    ResetArgs a{};
    a.n = h->n; a.A = p->A; a.L = p->L; a.NC = p->NS * p->DIMC; a.G = p->G;
    a.pv = static_cast<float4 *>(pv); a.lm = static_cast<float2 *>(lm); a.comm = comm; a.goal = goal; a.mask = mask;
    a.seed = seed; a.world_offset = world_offset; a.epoch = epoch; a.epoch_dev = epoch_dev;
    a.agent_range = 1.0f;  // every scenario: agents ~ U(-1, +1)^2
    // landmarks: U(-1,+1) (simple.py:37, simple_spread.py:44) or U(-0.9,+0.9) (simple_tag.py:53, simple_world_comm.py:105-113)
    const bool narrow = (p->scenario == MPE_SCN_TAG || p->scenario == MPE_SCN_WORLD_COMM);
    for (int l = 0; l < kMaxL; ++l) a.landmark_range[l] = narrow ? 0.9f : 1.0f;
    for (int g = 0; g < 4; ++g) a.goal_mod[g] = p->L > 0 ? p->L : 1;
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != h->device) CUDA_TRY(cudaSetDevice(h->device));
    const unsigned blocks = static_cast<unsigned>((h->n + 255) / 256);
    reset_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && epoch_dev) {
        bump_epoch_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(epoch_dev);
        e = cudaGetLastError();
        __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
    }
    if (prev != h->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(e, "reset_kernel");
    __atomic_add_fetch(&g_launches, 1, __ATOMIC_RELAXED);
    return MPE_OK;
}

extern "C" int mpe_reset(mpe_handle h, void *pv, void *lm, float *comm, int32_t *goal, const uint8_t *mask,
                         uint64_t seed, uint64_t world_offset, uint64_t epoch, void *stream) {
    return reset_impl(h, pv, lm, comm, goal, mask, seed, world_offset, epoch, nullptr, stream);
}

extern "C" int mpe_reset_dev_epoch(mpe_handle h, void *pv, void *lm, float *comm, int32_t *goal, const uint8_t *mask,
                                   uint64_t seed, uint64_t world_offset, unsigned long long *epoch_dev, void *stream) {
    if (!epoch_dev) return MPE_ERR_BAD_ARG;
    return reset_impl(h, pv, lm, comm, goal, mask, seed, world_offset, 0, epoch_dev, stream);
}

extern "C" int mpe_probe_stream(int device, const void *src, int64_t read_bytes, void *dst, int64_t write_bytes,
                                int64_t threads, void *stream) {
    if (!ok16(src) || !ok16(dst) || read_bytes < 0 || write_bytes < 0 || threads < 256) return MPE_ERR_BAD_ARG;
    int prev = 0;
    CUDA_TRY(cudaGetDevice(&prev));
    if (prev != device) CUDA_TRY(cudaSetDevice(device));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>((threads + 255) / 256));
    cfg.blockDim = dim3(256);
    cfg.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_mode() ? 1 : 0;
    const float4 *s4 = static_cast<const float4 *>(src);
    float4 *d4 = static_cast<float4 *>(dst);
    long long nr = read_bytes / 16, nw = write_bytes / 16;
    void *params[] = {&s4, &nr, &d4, &nw};
    cudaError_t e = cudaLaunchKernelExC(&cfg, reinterpret_cast<const void *>(stream_probe_kernel), params);
    if (prev != device) cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaLaunchKernelExC(stream_probe)");
    return MPE_OK;
}

extern "C" const char *mpe_strerror(int err) {
    switch (err) {
    case MPE_OK: return "ok";
    case MPE_ERR_BAD_ARG: return "bad argument (null or misaligned pointer, bad size or index)";
    case MPE_ERR_BAD_DESC: return "descriptor does not fit its scenario program";
    case MPE_ERR_UNSUPPORTED: return "no compiled sm_100a program for this scenario / shape / flag";
    case MPE_ERR_CUDA: return "CUDA runtime error (see mpe_last_cuda_error)";
    case MPE_ERR_NO_DEVICE: return "no sm_100 (B200) device with that index, or shape-only handle (device -1)";
    default: return "unknown error";
    }
}
extern "C" const char *mpe_last_cuda_error(void) { return g_cuda_err; }
extern "C" int mpe_abi_version(void) { return MPE_ABI_VERSION; }
extern "C" int64_t mpe_kernel_launches(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }
