// nig_kernels.cuh -- the sm_100a kernels of the batched IndustrialEnv step path.
//
//  step_core_impl    one env step in registers (environments/base.py:157-213): clip, constraints on the pre-step
//                    state, dynamics, reward, penalties, counters, termination, critical shutdown. One basic
//                    block: the divisions are guarded fast paths with ONE deferred guard per step (nig_math.cuh).
//  step_kernel       one IndustrialEnv.step for every env (+ auto-reset). HBM-bound: SoA fp32 state, VEC consecutive
//                    envs per thread (64-/128-bit LDG/STG); teacher-forced noise / reset states, AoS layouts,
//                    observation copies and host-evaluated constraint masks as runtime-uniform branches.
//                    Algorithmic traffic 122 B / env-step (reactor).
//  step_pipe_kernel  the plain SoA step of large populations: persistent CTAs, every input row of a 256-env tile
//                    staged in shared memory by 1-D bulk copies (cp.async.bulk -> UBLKCP) on a 3-stage mbarrier
//                    ring. 0.93 of the measured HBM copy bandwidth at 16.7M reactor envs.
//  rollout_kernel    K fused steps with the state in registers (the reset/step loops of
//                    performance_benchmark.py:106-133, utils.py:82-125, chemical_reactor.py:355-405): actions from a
//                    TMA-staged [K][A][pitch] tensor (cp.async.bulk.tensor.3d) or from register-prefetched LDGs, or
//                    generated in-kernel (uniform, get_dataset P-controllers, the benchmark baseline controllers),
//                    Philox process noise, REDUX / shuffle reductions for the violation / return statistics.
//                    FP32-issue bound.
//  dataset_kernel    get_dataset on the device: length-probe pass, scan, write pass (D4RL layout).
//  reset_kernel      IndustrialEnv.reset (base.py:133-155) for masked envs; coop_reset / coop_reset_blocks are the
//                    warp-cooperative in-kernel auto-resets.
#pragma once
#include <cuda.h>
#include "../../include/nig_b200.h"
#include "nig_envs.cuh"

namespace nig {

constexpr int kThreads = 128;
// how a kernel instantiation evaluates the safety constraints (see step_core_impl)
// CONS_BOUNDS1 / CONS_BOUNDS2: the built-ins plus exactly one / two pure state bounds (lo <= s[i] <= hi: the temperature /
// pressure bands of a SafetyWrapper) as straight-line code -- fused rollout kernels only, everything else treats them as
// CONS_PREFIX (cons_for_step). The guarded descriptor loop of CONS_PREFIX splits the step into several basic blocks and
// measured +56 % for the first extra constraint (tools/wrapper_cost.py).
enum : int { CONS_GENERIC = 0, CONS_DEFAULT = 1, CONS_PREFIX = 2, CONS_BOUNDS1 = 3, CONS_BOUNDS2 = 4 };
__host__ __device__ constexpr int cons_fast_extras(int cons) { return cons == CONS_BOUNDS1 ? 1 : cons == CONS_BOUNDS2 ? 2 : 0; }
inline int cons_for_step(int cons) { return cons > CONS_PREFIX ? CONS_PREFIX : cons; }

struct ConsParams {
    int32_t n;
    int32_t is_default;        // CONS_GENERIC / CONS_DEFAULT / CONS_PREFIX / CONS_BOUNDS* (host-side dispatch only)
    nig_constraint_t c[NIG_MAX_CONSTRAINTS];
    // NIG_CON_BOUND one-hot masks in DEVICE memory (kept out of the kernel parameters: 1.3 KB of them made every launch
    // measurably slower): row k = [NIG_MAX_STATE_DIM words: all-ones at si][NIG_MAX_ACTION_DIM words: all-ones at ai >= 0]
    const uint32_t* masks;
};
constexpr int kConsMaskRow = NIG_MAX_STATE_DIM + NIG_MAX_ACTION_DIM;

// ---- vector access helpers -----------------------------------------------------------------------
template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

template <int VEC>
__device__ __forceinline__ void ldvec(const float* p, float (&v)[VEC])
{
    using T = typename VecT<VEC>::type;
    const T t = *reinterpret_cast<const T*>(p);
    if constexpr (VEC == 1) { v[0] = t; }
    else if constexpr (VEC == 2) { v[0] = t.x; v[1] = t.y; }
    else { v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
}
template <int VEC>
__device__ __forceinline__ void stvec(float* p, const float (&v)[VEC])
{
    using T = typename VecT<VEC>::type;
    T t;
    if constexpr (VEC == 1) { t = v[0]; }
    else if constexpr (VEC == 2) { t.x = v[0]; t.y = v[1]; }
    else { t.x = v[0]; t.y = v[1]; t.z = v[2]; t.w = v[3]; }
    *reinterpret_cast<T*>(p) = t;
}

// s[i] for a runtime (warp-uniform) index i out of a register array, exact and branch-free: OR of the bit patterns
// under host-built one-hot masks (device memory, warp-uniform loads)
template <int S>
__device__ __forceinline__ float pick(const float (&s)[S], const uint32_t* __restrict__ onehot)
{
    uint32_t b = 0u;
#pragma unroll
    for (int k = 0; k < S; ++k) b |= __float_as_uint(s[k]) & onehot[k];
    return __uint_as_float(b);
}

// one runtime constraint descriptor (SafetyConstraint, core/types.py:56-64) on the pre-step state / clipped action
template <class Env>
__device__ __forceinline__ bool eval_constraint(const ConsParams& cp, int k, const float (&s)[Env::S], const float (&a)[Env::A], uint32_t hostmask)
{
    const nig_constraint_t& c = cp.c[k];
    if (c.kind == NIG_CON_BUILTIN) return Env::builtin(c.id, s, a);
    if (c.kind == NIG_CON_BOUND) {
        float v = pick<Env::S>(s, cp.masks + k * kConsMaskRow);
        if (c.ai >= 0) v = add(v, mul(c.coef, pick<Env::A>(a, cp.masks + k * kConsMaskRow + NIG_MAX_STATE_DIM)));
        return (c.lo <= v) && (v <= c.hi);
    }
    return !((hostmask >> c.id) & 1u);
}

// ep_word: bits 0..15 episode step, bits 16..30 episode violation count (saturating), bit 31 done latch
__device__ __forceinline__ uint32_t epw_step(uint32_t w) { return w & 0xffffu; }
__device__ __forceinline__ uint32_t epw_viol(uint32_t w) { return (w >> 16) & 0x7fffu; }
__device__ __forceinline__ uint32_t epw_make(uint32_t step, uint32_t viol, uint32_t done)
{
    return (step & 0xffffu) | ((viol > 0x7fffu ? 0x7fffu : viol) << 16) | (done << 31);
}

// ---- one env step in registers (base.py:157-213) --------------------------------------------------
// `div` carries out the divisions (DivExact = IEEE; DivFast = guarded fast path, see nig_math.cuh). With DivFast
// the outputs are only valid if div.ok() afterwards -- the callers redo the step with DivExact otherwise.
template <class Env, int CONS, class Div, bool CLIP = true>
__device__ __forceinline__ void step_core_impl(const ConsParams& cp, int max_steps,
                                               const float (&s)[Env::S], const float (&a_raw)[Env::A],
                                               const float (&nz)[Env::NZ > 0 ? Env::NZ : 1], uint32_t hostmask,
                                               uint32_t ep_step_in, uint32_t ep_viol_in, uint32_t& ep_step, uint32_t& ep_viol,
                                               float (&ns)[Env::S],
                                               typename Env::acc_t& reward, uint32_t& flags, uint32_t& vmask, Div& div)
{
    using acc_t = typename Env::acc_t;
    float a[Env::A];
#pragma unroll
    for (int j = 0; j < Env::A; ++j) {               // base.py:167 np.clip(action, -1, 1)
        float v = a_raw[j];
        if constexpr (CLIP) {                        // CLIP = false: the caller generated a in [-1, 1] itself (policy_uniform)
            v = v < -1.0f ? -1.0f : v;
            v = v > 1.0f ? 1.0f : v;
        }
        a[j] = v;
    }
    // base.py:170 -- constraints on the PRE-step state (the reference calls every check_fn twice with
    // identical arguments, :102 and :180; evaluated once here)
    // NOTE: `crit` is carried as a predicate of its own, never derived from the integer mask: ptxas 12.9
    // (sm_100a) mis-folds `((p ? 0 : 2) | (q ? 1 : 0)) != 0` into a PLOP3 with the polarity of q inverted
    // (found by the oracle parity tests on RobotAssembly; PTX correct, SASS wrong -- see DESIGN.md).
    uint32_t vm = 0;
    bool crit = false;
    // CONS_DEFAULT: exactly the env's built-ins with their default penalties (the env as registered upstream): compile-time
    // code, no loop. CONS_PREFIX: the built-ins first, then extra descriptors (a SafetyWrapper that ADDS constraints): the
    // built-ins stay compile-time code, the loop walks only the extras. CONS_GENERIC: every descriptor at run time.
    constexpr bool DEFCONS = CONS != CONS_GENERIC, EXTRAS = CONS == CONS_GENERIC || CONS == CONS_PREFIX;
    constexpr int NXF = cons_fast_extras(CONS);
    constexpr int K0 = DEFCONS ? Env::NB : 0;
    if constexpr (DEFCONS) {
#pragma unroll
        for (int k = 0; k < Env::NB; ++k) {
            const bool ok = Env::builtin(k, s, a);
            vm |= ok ? 0u : (1u << k);
            if ((Env::CRIT_MASK >> k) & 1u) crit = crit || !ok;
        }
    }
    if constexpr (NXF > 0) {                // exactly NXF pure state bounds after the built-ins: no guards, no kind dispatch
#pragma unroll
        for (int k = Env::NB; k < Env::NB + NXF; ++k) {
            const float v = pick<Env::S>(s, cp.masks + k * kConsMaskRow);
            const bool ok = (cp.c[k].lo <= v) && (v <= cp.c[k].hi);
            vm |= ok ? 0u : (1u << k);
            crit = crit || (!ok && cp.c[k].critical != 0);
        }
    }
    if constexpr (EXTRAS) {
#pragma unroll
        for (int k = K0; k < NIG_MAX_CONSTRAINTS; ++k) {
            if (k < cp.n) {                 // uniform: the descriptor count is a kernel parameter
                const bool ok = eval_constraint<Env>(cp, k, s, a, hostmask);
                vm |= ok ? 0u : (1u << k);
                crit = crit || (!ok && cp.c[k].critical != 0);
            }
        }
    }
    Env::dynamics(s, a, nz, ns, div);                 // base.py:173
    acc_t r = Env::reward(ns, a, div);                // base.py:176
    if constexpr (DEFCONS) {                          // base.py:179-183, in constraint order
#pragma unroll
        for (int k = 0; k < Env::NB; ++k)
            if ((vm >> k) & 1u) r = r + (acc_t)Env::penalty(k);
    }
    if constexpr (NXF > 0) {
#pragma unroll
        for (int k = Env::NB; k < Env::NB + NXF; ++k) {
            const acc_t rp = r + (acc_t)cp.c[k].penalty;      // same sum as the guarded form, selected instead of branched
            r = ((vm >> k) & 1u) ? rp : r;
        }
    }
    if constexpr (EXTRAS) {
#pragma unroll
        for (int k = K0; k < NIG_MAX_CONSTRAINTS; ++k)
            if (k < cp.n && ((vm >> k) & 1u)) r = r + (acc_t)cp.c[k].penalty;
    }
    const uint32_t step = ep_step_in + 1u;            // base.py:187
    const uint32_t viol = ep_viol_in + (uint32_t)__popc(vm);
    bool terminated = Env::is_done(ns);               // base.py:190
    const bool truncated = step >= (uint32_t)max_steps;   // base.py:191
    uint32_t f = 0;
    if (crit) { terminated = true; r = r - (acc_t)1000.0f; f |= NIG_F_CRITICAL; }   // base.py:195-198
    if (terminated) f |= NIG_F_TERMINATED;
    if (truncated) f |= NIG_F_TRUNCATED;
    ep_step = step; ep_viol = viol;
    reward = r; flags = f; vmask = vm;
}

// one step with the fast divisions and the deferred guard: the common path is a single basic block.
// Episode step / violation counters unpacked (the fused rollout keeps them in separate registers across K steps).
template <class Env, int CONS, bool CLIP = true, bool WARP_REDO = false>
__device__ __forceinline__ void step_core_unpacked(const ConsParams& cp, int max_steps,
                                                   const float (&s)[Env::S], const float (&a_raw)[Env::A],
                                                   const float (&nz)[Env::NZ > 0 ? Env::NZ : 1], uint32_t hostmask,
                                                   uint32_t ep_step_in, uint32_t ep_viol_in, uint32_t& ep_step, uint32_t& ep_viol,
                                                   float (&ns)[Env::S], typename Env::acc_t& reward, uint32_t& flags, uint32_t& vmask)
{
    if constexpr (Env::FAST_DIV) {
        DivFast df;
        step_core_impl<Env, CONS, DivFast, CLIP>(cp, max_steps, s, a_raw, nz, hostmask, ep_step_in, ep_viol_in, ep_step, ep_viol,
                                                 ns, reward, flags, vmask, df);
        // WARP_REDO (convergent call sites only): the redo decision is a warp vote, i.e. a uniform branch without a
        // divergence barrier; lanes whose guard held recompute the same IEEE-exact values
        if constexpr (WARP_REDO) { if (__builtin_expect(!__any_sync(0xffffffffu, !df.ok()), 1)) return; }
        else { if (__builtin_expect(df.ok(), 1)) return; }
    }
    DivExact de;
    step_core_impl<Env, CONS, DivExact, CLIP>(cp, max_steps, s, a_raw, nz, hostmask, ep_step_in, ep_viol_in, ep_step, ep_viol,
                                              ns, reward, flags, vmask, de);
}

// the same with the packed episode word of the HBM layout (single-step and dataset kernels)
template <class Env, int CONS, bool CLIP = true>
__device__ __forceinline__ void step_core(const ConsParams& cp, int max_steps,
                                          const float (&s)[Env::S], const float (&a_raw)[Env::A],
                                          const float (&nz)[Env::NZ > 0 ? Env::NZ : 1], uint32_t hostmask,
                                          uint32_t& ep_word, float (&ns)[Env::S],
                                          typename Env::acc_t& reward, uint32_t& flags, uint32_t& vmask)
{
    uint32_t st, vi;
    step_core_unpacked<Env, CONS, CLIP>(cp, max_steps, s, a_raw, nz, hostmask, epw_step(ep_word), epw_viol(ep_word), st, vi,
                                        ns, reward, flags, vmask);
    ep_word = epw_make(st, vi, 0u);
}

// ---- warp-cooperative auto-reset ---------------------------------------------------------------------------------
// A finished env needs Env::RESET_NORMALS fresh Gaussians (reactor: 2 Philox blocks + 8 table normals, ~150
// instructions) and on average only 1 lane in 12 warp-steps finishes: instead of the whole warp walking the full draw
// for one lane, every resetting lane in turn broadcasts its env id, lanes 0..3 each produce ONE pair of normals of its
// draw, and the 8 normals are shuffled back. Same counters, same values as Env::reset(). Must be called convergently.
template <class Env>
__device__ __forceinline__ void coop_reset(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, bool need, float (&s)[Env::S])
{
    unsigned m = __ballot_sync(0xffffffffu, need);
    const uint32_t lane = threadIdx.x & 31u;
    while (m) {
        const int src = __ffs(m) - 1;
        m &= m - 1;
        const uint32_t e_src = __shfl_sync(0xffffffffu, env, src);
        float z0, z1;
        Env::reset_pair(key, e_src, tick, epoch, lane & 3u, z0, z1);
        float z[Env::RESET_NORMALS];
#pragma unroll
        for (int q = 0; q < Env::RESET_NORMALS / 2; ++q) {
            z[2 * q] = __shfl_sync(0xffffffffu, z0, q);
            z[2 * q + 1] = __shfl_sync(0xffffffffu, z1, q);
        }
        if ((int)lane == src) Env::reset_from_normals(z, s);
    }
}

// Block-granular flavour for envs whose draw is long AND whose episodes are short (PowerGrid: 8 Philox blocks, 26
// Gaussians + 8 uniforms per reset, ~18 % of the envs reset every step under random actions, i.e. ~6 lanes of every
// warp): the work items (resetting lane, block) of the whole warp are dealt round-robin to the 32 lanes, the raw values
// go through a per-warp shared-memory buffer [32 resetting lanes][COOP_BLOCKS * 4], the owners rebuild their state.
constexpr int kFkRanks = 8, kFkWarpFloats = kFkRanks * 8 * 3 * 2 + 32;       // coop_reset_fk: 8 ranks x 8 slots x {q, sin, cos} fp64 + the rank list
template <class Env>
struct CoopSmem {
    static constexpr int floats = Env::COOP_BLOCKS > 0 ? (kThreads / 32) * 32 * Env::COOP_BLOCKS * 4
                                : (Env::COOP_FK ? (kThreads / 32) * kFkWarpFloats : 1);
};

// RobotAssembly-v0: a fresh state is seven uniform joint angles and the forward kinematics of them -- seven binary64
// sin / cos pairs, ~430 instructions that the whole warp walks for the 2 - 3 lanes that finished (episodes are short under
// random actions: 58 % of the warp-steps have a resetting lane). Here the (resetting lane, joint) items are dealt to the
// lanes -- four ranks per round, lane l takes joint l mod 8 (slot 7 idles) --, each producer draws the joint's angle from the
// reset stream, evaluates ONE sin / cos pair and leaves {q, sin q, cos q} in the warp's shared-memory buffer; the owners sum the
// link contributions in the reference's order (:94-111). Same counters, same bits as Env::reset(). Must be called convergently.
template <class Env>
__device__ __forceinline__ void coop_reset_fk(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, bool need,
                                              float (&s)[Env::S], float* cta_buf)
{
    const unsigned m = __ballot_sync(0xffffffffu, need);
    if (m == 0u) return;                                        // warp-uniform
    const uint32_t lane = threadIdx.x & 31u;
    double* const buf = reinterpret_cast<double*>(cta_buf + (threadIdx.x >> 5) * kFkWarpFloats);       // [kFkRanks][8][3]
    uint32_t* const list = reinterpret_cast<uint32_t*>(buf + kFkRanks * 8 * 3);
    const int cnt = __popc(m);
    const int rk = __popc(m & ((1u << lane) - 1u));
    if (need) list[rk] = lane;
    __syncwarp();
    const uint32_t j = lane & 7u;
    const int q4 = (int)(lane >> 3);
#pragma unroll 1
    for (int c0 = 0; c0 < cnt; c0 += kFkRanks) {
#pragma unroll 1
        for (int r0 = c0; r0 < cnt && r0 < c0 + kFkRanks; r0 += 4) {
            const int r = r0 + q4;
            const bool live = r < cnt && j < 7u;
            const int src = (int)list[r < cnt ? r : 0];
            const uint32_t e_src = __shfl_sync(0xffffffffu, env, src);
            const uint4 w = rng_words(key, e_src, tick, STREAM_RESET, (epoch << 8) | (j >> 2));
            const uint32_t word = (j & 2u) ? ((j & 1u) ? w.w : w.z) : ((j & 1u) ? w.y : w.x);
            const double q = (double)mul(0x1.921fb6p+0f, u_sym(word));
            double sn, cs;
            spec_sincos_f64(q, sn, cs);
            if (live) {
                double* d = buf + ((r - c0) * 8 + (int)j) * 3;
                d[0] = q; d[1] = sn; d[2] = cs;
            }
        }
        __syncwarp();
        const int row = rk - c0;
        if (need && row >= 0 && row < kFkRanks) {
            const double* d = buf + row * 8 * 3;
            double x = 0.0, y = 0.0, z = 0.0;
#pragma unroll
            for (int i = 0; i < Env::S; ++i) s[i] = 0.0f;
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                const double q = d[i * 3], sn = d[i * 3 + 1], cs = d[i * 3 + 2];
                if ((i & 1) == 0) { x = dadd(x, dmul(Env::link(i), cs)); z = dadd(z, dmul(Env::link(i), sn)); }
                else y = dadd(y, dmul(Env::link(i), sn));
                s[7 + i] = (float)q;
            }
            s[0] = (float)x; s[1] = (float)y; s[2] = (float)z;
            s[6] = 1.0f;
        }
        __syncwarp();
    }
}

template <class Env>
__device__ __forceinline__ void coop_reset_blocks(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, bool need,
                                                  float (&s)[Env::S], float* cta_buf)
{
    constexpr int RB = Env::COOP_BLOCKS, NV = RB * 4;
    const unsigned m = __ballot_sync(0xffffffffu, need);
    if (m == 0u) return;                                        // warp-uniform
    const uint32_t lane = threadIdx.x & 31u;
    float* buf = cta_buf + (threadIdx.x >> 5) * 32 * NV;
    const int items = __popc(m) * RB;
    for (int base = 0; base < items; base += 32) {
        const int it = base + (int)lane;
        const bool live = it < items;
        const int r = live ? it / RB : 0;                       // rank of the resetting lane this item belongs to
        const uint32_t j = (uint32_t)(it % RB);
        const int src = (int)__fns(m, 0u, r + 1);               // lane index of the r-th set bit
        const uint32_t e_src = __shfl_sync(0xffffffffu, env, src);
        float v[4];
        Env::reset_block(key, e_src, tick, epoch, j, v);
        if (live) {
#pragma unroll
            for (int q = 0; q < 4; ++q) buf[r * NV + (int)j * 4 + q] = v[q];
        }
    }
    __syncwarp();
    if (need) {
        const int r = __popc(m & ((1u << lane) - 1u));
        float v[NV];
#pragma unroll
        for (int q = 0; q < NV; ++q) v[q] = buf[r * NV + q];
        Env::reset_from_values(v, s);
    }
    __syncwarp();
}

// ---- device-resident tick (CUDA-graph capture) --------------------------------------------------------------------
// The batched-step counter that keys the random streams is normally a kernel argument (host-side state of the handle).
// A captured graph replays the SAME arguments, so in device-tick mode the kernels read the counter from tick_dev[0]
// instead, and the last CTA of a launch to finish (tick_dev[1] counts finished CTAs) advances it for the next launch.
__device__ __forceinline__ uint32_t load_tick(const uint32_t* tick_dev, uint32_t host_tick)
{
    return tick_dev ? *reinterpret_cast<const volatile uint32_t*>(tick_dev) : host_tick;
}
// Third way of supplying the counters (captured host-buffer pipelines, nig_rollout_host): tick_base -> {tick, epoch} in device
// memory, refreshed by the graph's first node from a pinned host word on every replay; the kernel arguments then hold
// OFFSETS from that base (the slices of one call run concurrently, so the device tick above cannot serve them).
__device__ __forceinline__ uint32_t base_tick(const uint32_t* tick_base) { return tick_base ? __ldg(tick_base) : 0u; }
__device__ __forceinline__ uint32_t base_epoch(const uint32_t* tick_base) { return tick_base ? __ldg(tick_base + 1) : 0u; }
__device__ __forceinline__ void advance_device_tick(uint32_t* tick_dev, uint32_t by)
{
    if (tick_dev == nullptr) return;                // uniform
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(tick_dev + 1, 1u) == gridDim.x * gridDim.y - 1u) {
            tick_dev[1] = 0u;
            tick_dev[0] += by;
            __threadfence();
        }
    }
}

// ---- extrema of finished-episode returns (evaluate_with_safety's return_min / return_max, utils.py:131-132) -------------
// Kept outside the summable stats block: two order-preserving integer keys combined with atomicMax (0 = no episode
// yet), so that ranks combine them with ONE max all-reduce. key(x) is monotone in x; slot 0 holds key(-x) (the minimum),
// slot 1 key(x). The last mantissa bit is dropped to keep the keys non-negative as int64 (NCCL max on int64).
__device__ __forceinline__ unsigned long long extremum_key(double x)
{
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    const unsigned long long k = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
    return k >> 1;                   // 0 only for a NaN bit pattern
}

template <class T> __device__ __forceinline__ T warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- block-level statistics: per-thread counts -> REDUX -> shared atomics -> one global atomic per slot
struct BlockStats {
    unsigned int* sh;   // [NIG_STATS_SLOTS] shared counters
    __device__ __forceinline__ void init(unsigned int* smem)
    {
        sh = smem;
        if (threadIdx.x < NIG_STATS_SLOTS) sh[threadIdx.x] = 0u;
        __syncthreads();
    }
    __device__ __forceinline__ void warp_add(int slot, unsigned int v)
    {
        const unsigned int t = __reduce_add_sync(0xffffffffu, v);
        if ((threadIdx.x & 31) == 0 && t) atomicAdd(&sh[slot], t);
    }
    __device__ __forceinline__ void flush(unsigned long long* g)
    {
        __syncthreads();
        if (threadIdx.x < 24 && sh[threadIdx.x]) atomicAdd(&g[threadIdx.x], (unsigned long long)sh[threadIdx.x]);
    }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "NIG_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra NIG_DONE_%=;\n\t"
        "bra NIG_WAIT_%=;\n\t"
        "NIG_DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}

// 1-D bulk copy global -> shared through the TMA unit (UBLKCP), completion counted on an mbarrier
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ================================================================================================
// single-step kernel
// ================================================================================================
struct StepArgs {
    float* state;            // [S][pitch]
    uint32_t* ep_word;       // [pitch]
    double* ep_return;       // [pitch] running episode return (shared with the rollout kernel), or null: not tracked (nig_track_returns)
    int64_t n, pitch;
    uint32_t env0, tick, epoch;
    uint32_t* tick_dev;      // non-null: device-resident tick (graph capture), see load_tick()
    const uint32_t* tick_base;   // non-null: tick / epoch above are offsets from tick_base[0] (sequence-tick graphs, see base_tick())
    RngKey key;
    int32_t max_steps, auto_reset;
    const float* actions;
    const float* noise;
    const float* reset_states;
    const uint8_t* hostmask;
    float* obs;
    float* next_obs;
    float* reward;
    uint8_t* flags;
    uint8_t* viol_mask;
    uint8_t* terminated;     // optional 0/1 arrays (torch bool views): unpacked flags
    uint8_t* truncated;
    int32_t action_aos, aux_aos;
    unsigned long long* stats;
    // PLAIN flavour: kStatsShards copies of the stats block; CTA b adds to copy b % kStatsShards. At 65,536 envs the 512
    // CTAs' ~1,600 reductions on the three hot addresses of ONE block kept every launch waiting 1.25 us for the L2 atomic unit
    // (4.07 -> 2.82 us per replayed launch without them); the copies are folded into `stats` whenever it is read (fold_stats_kernel)
    unsigned long long* stats_shards;
    ConsParams cons;
};
constexpr int kStatsShards = 128;

// finished-episode statistics of the single-step kernels (the same slots the fused rollout fills: evaluate_with_safety's
// return / length aggregates, utils.py:128-152), so that a handle driven through nig_step reports them too and a
// nig_rollout that follows continues every running episode's return from the right value
struct StepEpisodeStats {
    unsigned int c_succ = 0;
    unsigned long long len_sum = 0, len_sq = 0;
    double ret_sum = 0.0, ret_sq = 0.0;
    __device__ __forceinline__ void episode(double ret, unsigned long long len)
    {
        c_succ += ret > 0.0 ? 1u : 0u;
        len_sum += len; len_sq += len * len;
        ret_sum += ret; ret_sq += ret * ret;
    }
};

// finished-episode return / length sums of a warp -> per-CTA shared staging (EpisodeStaging) -> one global atomic per slot
// per CTA (PowerGrid finishes an episode in ~18 % of its envs every step: per-warp global atomics on four addresses cost the
// 1M-env single step 48 us)
struct EpisodeStaging {
    unsigned long long len[2];      // EP_LEN_SUM, EP_LEN_SQ
    double ret[2];                  // RETURN_SUM, RETURN_SQ
};
__device__ __forceinline__ void episode_staging_init(EpisodeStaging* st)
{
    if (threadIdx.x < 2) { st->len[threadIdx.x] = 0ull; st->ret[threadIdx.x] = 0.0; }      // (before a __syncthreads of the caller)
}
__device__ __forceinline__ void stage_episode_stats(BlockStats& bs, EpisodeStaging* st, const StepEpisodeStats& eps)
{
    bs.warp_add(NIG_ST_SUCCESSES, eps.c_succ);
    const unsigned long long ls = warp_sum(eps.len_sum), lq = warp_sum(eps.len_sq);
    const double rs_ = warp_sum(eps.ret_sum), rq = warp_sum(eps.ret_sq);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&st->len[0], ls); atomicAdd(&st->len[1], lq);
        atomicAdd(&st->ret[0], rs_); atomicAdd(&st->ret[1], rq);
    }
}
// after a __syncthreads that follows the last stage_episode_stats of the CTA (BlockStats::flush has one)
__device__ __forceinline__ void flush_episode_staging(unsigned long long* stats, const EpisodeStaging* st)
{
    if (threadIdx.x < 2) {
        if (st->len[threadIdx.x]) atomicAdd(&stats[threadIdx.x == 0 ? NIG_ST_EP_LEN_SUM : NIG_ST_EP_LEN_SQ], st->len[threadIdx.x]);
        if (st->ret[threadIdx.x] != 0.0) atomicAdd(reinterpret_cast<double*>(stats) + NIG_ST_F_RETURN_SUM + threadIdx.x, st->ret[threadIdx.x]);
    }
}

template <int D, int VEC>
__device__ __forceinline__ void load_rows(const float* base, int64_t pitch, int64_t n, int64_t i0, bool aos, float (&v)[D][VEC])
{
    if (!aos) {
#pragma unroll
        for (int k = 0; k < D; ++k) ldvec<VEC>(base + k * pitch + i0, v[k]);
    } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e)
#pragma unroll
            for (int k = 0; k < D; ++k) v[k][e] = (i0 + e < n) ? base[(i0 + e) * D + k] : 0.0f;
    }
}
template <int D, int VEC>
__device__ __forceinline__ void store_rows(float* base, int64_t pitch, int64_t n, int64_t i0, bool aos, const float (&v)[D][VEC])
{
    if (!aos) {
#pragma unroll
        for (int k = 0; k < D; ++k) stvec<VEC>(base + k * pitch + i0, v[k]);
    } else {
#pragma unroll
        for (int e = 0; e < VEC; ++e)
            if (i0 + e < n) {
#pragma unroll
                for (int k = 0; k < D; ++k) base[(i0 + e) * D + k] = v[k][e];
            }
    }
}

// AoS rows ([n][D] row-major: the layout of the host and torch APIs) through a per-warp shared-memory transpose, so
// that the global accesses of a warp are D fully coalesced 128-byte requests instead of D requests that each touch 32
// sectors (measured at 4M envs with obs + next_obs outputs, tools/aos_vs_soa.py: reactor 340 -> 197 us, grid 1553 -> 652 us).
// One env per lane. STREAM: evict-first stores (__stcs) for outputs nothing in the kernel reads again (nig_rollout_record).
template <int D, bool STREAM = false>
__device__ __forceinline__ void store_aos_warp(float* base, int64_t n, int64_t i, const float (&v)[D], float* tile)
{
    const int lane = threadIdx.x & 31;
    const int64_t env0 = i - lane;
#pragma unroll
    for (int k = 0; k < D; ++k) tile[lane * (D + 1) + k] = v[k];
    __syncwarp();
#pragma unroll
    for (int it = 0; it < D; ++it) {
        const int j = it * 32 + lane;           // float index inside the warp's [32][D] block
        const int e = j / D, k = j - e * D;
        if (env0 + e < n) {
            if constexpr (STREAM) __stcs(base + env0 * D + j, tile[e * (D + 1) + k]);
            else base[env0 * D + j] = tile[e * (D + 1) + k];
        }
    }
    __syncwarp();
}
// PLAIN: the caller guarantees the plain SoA step (no teacher-forced noise / reset states, no host-evaluated constraint mask,
// no observation copies, no unpacked flag arrays, SoA actions): every run-time-uniform option branch below folds away at
// compile time -- ~400 of PowerGrid's 1,923 issued instructions per step were those branches and their address arithmetic.
template <class Env, int VEC, int CONS, bool PLAIN = false>
__global__ void __launch_bounds__(kThreads, VEC == 1 ? Env::STEP_MIN_CTAS : 1) step_kernel(const __grid_constant__ StepArgs p0)
{
    // (a by-value copy of the option fields with the PLAIN ones pinned to "absent"; everything else is read from p0 directly)
    struct Opt {
        const float* noise; const float* reset_states; const uint8_t* hostmask; float* obs; float* next_obs;
        uint8_t* terminated; uint8_t* truncated; int32_t action_aos, aux_aos;
    };
    const Opt o = PLAIN ? Opt{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0}
                        : Opt{p0.noise, p0.reset_states, p0.hostmask, p0.obs, p0.next_obs, p0.terminated, p0.truncated, p0.action_aos, p0.aux_aos};
    const StepArgs& p = p0;
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    using acc_t = typename Env::acc_t;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ EpisodeStaging estage;
    __shared__ alignas(16) float coop_buf[CoopSmem<Env>::floats];
    __shared__ float aos_tile[(VEC == 1 && !PLAIN) ? (kThreads / 32) * 32 * (S + 1) : 1];      // AoS transposes (VEC == 1 only)
    float* my_tile = aos_tile + ((VEC == 1 && !PLAIN) ? (threadIdx.x >> 5) * 32 * (S + 1) : 0);
    BlockStats bs;
    episode_staging_init(&estage);
    bs.init(sstat);
    const Rng key(p.key, g_normal_tab);        // one-tile CTA: the L1-cached global table
    // PLAIN + a tick that does not depend on the previous launch (a kernel argument, or base + sequence offset): this step's
    // process noise is a function of (env, tick) alone and is drawn BEFORE waiting for the previous step (below)
    const bool early = PLAIN && VEC == 1 && NZ > 0 && p.tick_dev == nullptr && (p.tick_base == nullptr || p.tick != 0u);
    float nz_pre[NZA];
    uint32_t tick_pre = 0u;
    if (early) {
        tick_pre = p.tick + base_tick(p.tick_base);
        const int64_t ie = (int64_t)blockIdx.x * kThreads + threadIdx.x;
        Env::NoiseGen::get_single(key, p.env0 + (uint32_t)ie, tick_pre, nz_pre);
    }
    if constexpr (PLAIN) {
        // programmatic dependent launch (the launcher sets cudaLaunchAttributeProgrammaticStreamSerialization on this flavour):
        // the CTAs of step t + 1 are scheduled while step t drains, set up their shared memory and (see above) draw their
        // noise, and wait HERE until step t has completed and flushed -- before the first read of anything it writes (device
        // tick, state, episode words). Their own dependents may be scheduled at once: they will wait in the same place.
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }
    const uint32_t tick0 = early ? tick_pre : load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);

    const int64_t i0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
    unsigned int c_steps = 0, c_ep = 0, c_term = 0, c_trunc = 0, c_crit = 0, c_viol = 0, c_con = 0;  // c_con: 4 bits/constraint
    // an env finishes at most one episode per launch: its return / length are kept per element and only summed in the
    // epilogue, where nothing else is live (a running StepEpisodeStats cost PowerGrid 40 B of spills and 30 % of its rate)
    double fin_ret[VEC];
    uint32_t fin_len[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) { fin_ret[e] = 0.0; fin_len[e] = 0u; }
    if (i0 < p.pitch) {
        float sv[S][VEC], av[A][VEC], nzv[NZA][VEC], rs[S][VEC];
        load_rows<S, VEC>(p.state, p.pitch, p.n, i0, false, sv);
        load_rows<A, VEC>(p.actions, p.pitch, p.n, i0, o.action_aos != 0, av);   // (a transposed AoS load measured 5 % slower)
        float wv[VEC];
        ldvec<VEC>(reinterpret_cast<const float*>(p.ep_word) + i0, wv);
        if (NZ > 0 && o.noise) load_rows<NZA, VEC>(o.noise, p.pitch, p.n, i0, o.aux_aos != 0, nzv);
        if (o.reset_states) load_rows<S, VEC>(o.reset_states, p.pitch, p.n, i0, o.aux_aos != 0, rs);

        float nsv[S][VEC], rw[VEC];
        uint32_t fl[VEC], vmk[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const int64_t i = i0 + e;
            const uint32_t env = p.env0 + (uint32_t)i;
            uint32_t w = __float_as_uint(wv[e]);
            float s[S], a[A], nz[NZA], ns[S];
#pragma unroll
            for (int k = 0; k < S; ++k) s[k] = sv[k][e];
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = av[k][e];
            const bool valid = i < p.n;
            const bool active = valid && !(w >> 31);
            acc_t er = (acc_t)0;                       // running episode return (the accumulator the fused rollout continues)
            if (p.ep_return && active) er = (acc_t)p.ep_return[i];
            if (NZ > 0) {
                if (o.noise) {
#pragma unroll
                    for (int k = 0; k < NZA; ++k) nz[k] = nzv[k][e];
                } else if (early) {
#pragma unroll
                    for (int k = 0; k < NZA; ++k) nz[k] = nz_pre[k];
                } else {
                    Env::NoiseGen::get_single(key, env, tick0, nz);
                }
            } else nz[0] = 0.0f;
            acc_t r; uint32_t f, vm;
            const uint32_t hm = o.hostmask && valid ? o.hostmask[i] : 0u;
            step_core<Env, CONS>(p.cons, p.max_steps, s, a, nz, hm, w, ns, r, f, vm);
            if (!active) {            // finished env without auto-reset (or padding lane): nothing happens
#pragma unroll
                for (int k = 0; k < S; ++k) ns[k] = s[k];
                r = (acc_t)0; f = NIG_F_INACTIVE; vm = 0; w = __float_as_uint(wv[e]);
            }
            const bool done = active && (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED));
            bool need_reset = false;
            if (p.ep_return && active) {
                er = er + r;
                if (done) { fin_ret[e] = (double)er; fin_len[e] = epw_step(w); }
                p.ep_return[i] = (done && p.auto_reset) ? 0.0 : (double)er;
            }
#pragma unroll
            for (int k = 0; k < S; ++k) nsv[k][e] = ns[k];     // s' of the transition (pre-reset)
            if (done) {
                if (p.auto_reset) {
                    if (o.reset_states) {
#pragma unroll
                        for (int k = 0; k < S; ++k) s[k] = rs[k][e];
                    } else {
                        if constexpr (Env::COOP_RESET || Env::COOP_BLOCKS > 0 || Env::COOP_FK) need_reset = true;
                        else Env::reset(key, env, tick0 + 1u, p.epoch, s);
                    }
                    w = 0u; f |= NIG_F_RESET;
                } else {
#pragma unroll
                    for (int k = 0; k < S; ++k) s[k] = ns[k];
                    w |= 0x80000000u;
                }
            } else {
#pragma unroll
                for (int k = 0; k < S; ++k) s[k] = ns[k];
            }
            if constexpr (Env::COOP_RESET) coop_reset<Env>(key, env, tick0 + 1u, p.epoch, need_reset, s);
            else if constexpr (Env::COOP_BLOCKS > 0) coop_reset_blocks<Env>(key, env, tick0 + 1u, p.epoch, need_reset, s, coop_buf);
            else if constexpr (Env::COOP_FK) coop_reset_fk<Env>(key, env, tick0 + 1u, p.epoch, need_reset, s, coop_buf);
#pragma unroll
            for (int k = 0; k < S; ++k) sv[k][e] = s[k];
            wv[e] = __uint_as_float(w);
            rw[e] = (float)r; fl[e] = f; vmk[e] = vm;
            if (active) {
                c_steps += 1; c_viol += __popc(vm);
                c_crit += (f & NIG_F_CRITICAL) ? 1u : 0u;
                if (done) { c_ep += 1; c_term += (f & NIG_F_TERMINATED) ? 1u : 0u; c_trunc += (f & NIG_F_TRUNCATED) ? 1u : 0u; }
#pragma unroll
                for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) c_con += ((vm >> k) & 1u) << (4 * k);
            }
        }
        store_rows<S, VEC>(p.state, p.pitch, p.n, i0, false, sv);
        stvec<VEC>(reinterpret_cast<float*>(p.ep_word) + i0, wv);
        if constexpr (VEC == 1) {
            if (o.aux_aos) {
                float row[S];
                if (o.obs) {
#pragma unroll
                    for (int k = 0; k < S; ++k) row[k] = sv[k][0];
                    store_aos_warp<S>(o.obs, p.n, i0, row, my_tile);
                }
                if (o.next_obs) {
#pragma unroll
                    for (int k = 0; k < S; ++k) row[k] = nsv[k][0];
                    store_aos_warp<S>(o.next_obs, p.n, i0, row, my_tile);
                }
            } else {
                if (o.obs) store_rows<S, VEC>(o.obs, p.pitch, p.n, i0, false, sv);
                if (o.next_obs) store_rows<S, VEC>(o.next_obs, p.pitch, p.n, i0, false, nsv);
            }
        } else {
            if (o.obs) store_rows<S, VEC>(o.obs, p.pitch, p.n, i0, o.aux_aos != 0, sv);
            if (o.next_obs) store_rows<S, VEC>(o.next_obs, p.pitch, p.n, i0, o.aux_aos != 0, nsv);
        }
        // VEC == 1 serves the exact-size [n] arrays of the host-buffer (zero-copy) and torch APIs: no store past env n - 1
        // (the vector flavours require pitch-capacity device arrays, include/nig_b200.h)
        const bool in_n = VEC > 1 || i0 < p.n;
        if (p.reward && in_n) stvec<VEC>(p.reward + i0, rw);
        if (p.flags && in_n) {
            if constexpr (VEC == 4) *reinterpret_cast<uchar4*>(p.flags + i0) = make_uchar4(fl[0], fl[1], fl[2], fl[3]);
            else if constexpr (VEC == 2) *reinterpret_cast<uchar2*>(p.flags + i0) = make_uchar2(fl[0], fl[1]);
            else p.flags[i0] = (uint8_t)fl[0];
        }
        if (p.viol_mask && in_n) {
            if constexpr (VEC == 4) *reinterpret_cast<uchar4*>(p.viol_mask + i0) = make_uchar4(vmk[0], vmk[1], vmk[2], vmk[3]);
            else if constexpr (VEC == 2) *reinterpret_cast<uchar2*>(p.viol_mask + i0) = make_uchar2(vmk[0], vmk[1]);
            else p.viol_mask[i0] = (uint8_t)vmk[0];
        }
        if (o.terminated || o.truncated) {
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                if (i0 + e < (VEC == 1 ? p.n : p.pitch)) {
                    if (o.terminated) o.terminated[i0 + e] = (uint8_t)((fl[e] & NIG_F_TERMINATED) ? 1 : 0);
                    if (o.truncated) o.truncated[i0 + e] = (uint8_t)((fl[e] & NIG_F_TRUNCATED) ? 1 : 0);
                }
            }
        }
    }
    if (p.stats == nullptr) {             // nig_track_step_stats(env, 0): no device counters for single steps (the per-env outputs are complete)
        advance_device_tick(p.tick_dev, 1u);
        return;
    }
    if constexpr (PLAIN) {
        if (p.stats_shards) {
            // per-WARP flush straight into a shard copy of the stats block: no CTA barrier and no shared staging, so the
            // reductions leave right behind the warp's stores instead of one L2 round trip after the slowest warp of the CTA
            // (the kernel cannot retire before they are acknowledged: 3.97 -> see DESIGN 3.1 us per replayed 65,536-env launch)
            unsigned long long* const row = p.stats_shards +
                (size_t)((blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) % kStatsShards) * NIG_STATS_SLOTS;
            const bool lead = (threadIdx.x & 31) == 0;
            auto red = [&](int slot, unsigned int v) {
                const unsigned int t = __reduce_add_sync(0xffffffffu, v);
                if (lead && t) atomicAdd(&row[slot], (unsigned long long)t);
            };
            red(NIG_ST_STEPS, c_steps);
            if (__any_sync(0xffffffffu, (c_ep | c_viol | c_crit) != 0u)) {
                red(NIG_ST_EPISODES, c_ep); red(NIG_ST_TERMINATED, c_term); red(NIG_ST_TRUNCATED, c_trunc);
                red(NIG_ST_CRITICAL, c_crit); red(NIG_ST_VIOLATIONS, c_viol);
                for (int k = 0; k < p.cons.n; ++k) red(NIG_ST_CON0 + k, (c_con >> (4 * k)) & 0xfu);
                if (p.ep_return && __any_sync(0xffffffffu, c_ep != 0u)) {
                    StepEpisodeStats eps;
#pragma unroll
                    for (int e = 0; e < VEC; ++e)
                        if (fin_len[e]) eps.episode(fin_ret[e], (unsigned long long)fin_len[e]);
                    red(NIG_ST_SUCCESSES, eps.c_succ);
                    const unsigned long long ls = warp_sum(eps.len_sum), lq = warp_sum(eps.len_sq);
                    const double rs_ = warp_sum(eps.ret_sum), rq = warp_sum(eps.ret_sq);
                    if (lead) {
                        atomicAdd(&row[NIG_ST_EP_LEN_SUM], ls); atomicAdd(&row[NIG_ST_EP_LEN_SQ], lq);
                        atomicAdd(reinterpret_cast<double*>(row) + NIG_ST_F_RETURN_SUM, rs_);
                        atomicAdd(reinterpret_cast<double*>(row) + NIG_ST_F_RETURN_SQ, rq);
                    }
                }
            }
            advance_device_tick(p.tick_dev, 1u);
            return;
        }
    }
    bs.warp_add(NIG_ST_STEPS, c_steps);
    if (__any_sync(0xffffffffu, (c_ep | c_viol | c_crit) != 0u)) {
        bs.warp_add(NIG_ST_EPISODES, c_ep);
        bs.warp_add(NIG_ST_TERMINATED, c_term);
        bs.warp_add(NIG_ST_TRUNCATED, c_trunc);
        bs.warp_add(NIG_ST_CRITICAL, c_crit);
        bs.warp_add(NIG_ST_VIOLATIONS, c_viol);
        for (int k = 0; k < p.cons.n; ++k) bs.warp_add(NIG_ST_CON0 + k, (c_con >> (4 * k)) & 0xfu);
        if (p.ep_return && __any_sync(0xffffffffu, c_ep != 0u)) {
            StepEpisodeStats eps;
#pragma unroll
            for (int e = 0; e < VEC; ++e)
                if (fin_len[e]) eps.episode(fin_ret[e], (unsigned long long)fin_len[e]);
            stage_episode_stats(bs, &estage, eps);
        }
    }
    unsigned long long* const stats_out = (PLAIN && p.stats_shards) ? p.stats_shards + (blockIdx.x % kStatsShards) * NIG_STATS_SLOTS : p.stats;
    bs.flush(stats_out);
    if (p.ep_return) flush_episode_staging(stats_out, &estage);
    advance_device_tick(p.tick_dev, 1u);
}

// ================================================================================================
// single-step kernel, persistent + TMA-pipelined (the production fast path: SoA actions, in-kernel noise and reset draws)
// ================================================================================================
// step_kernel above keeps one tile per CTA in registers, so the bytes in flight per SM are bounded by the
// register-limited occupancy (4 CTAs x 15 KB at 100 registers) -- short of the ~52 KB/SM that 6.4 TB/s x ~1.2 us
// of loaded latency needs. Here each CTA is persistent (grid = SMs x resident CTAs), walks tiles of kThreads x VEC
// envs with stride gridDim.x, and stages every input row of a tile (S state rows, A action rows, the episode word)
// in shared memory with 1-D bulk copies (cp.async.bulk -> UBLKCP) on a kStepStages-deep mbarrier ring, issued by
// one thread two tiles ahead: loads in flight no longer depend on occupancy. Arithmetic and stores are those of
// step_kernel (same step_core, bit-identical results).
constexpr int kStepStages = 3;

template <class Env, int VEC>
constexpr size_t step_pipe_smem() { return (size_t)kStepStages * (Env::S + Env::A + 1) * kThreads * VEC * sizeof(float); }

template <class Env, int VEC, int CONS>
__global__ void __launch_bounds__(kThreads, 4) step_pipe_kernel(const __grid_constant__ StepArgs p)
{
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    constexpr int TILE = kThreads * VEC, ROWS = S + A + 1;
    using acc_t = typename Env::acc_t;
    extern __shared__ __align__(128) float stage_smem[];     // [kStepStages][ROWS][TILE]
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ EpisodeStaging estage;
    __shared__ alignas(8) uint64_t full[kStepStages];
    __shared__ alignas(16) float coop_buf[CoopSmem<Env>::floats];
    // persistent CTAs amortise a shared copy of the normal table where the env draws many normals per step (PowerGrid);
    // for the reactor it would cost the fourth resident CTA its stage ring (measured: 0.90 -> 0.85 of the HBM peak)
    __shared__ float4 s_tab[Env::TAB_SMEM ? NIG_NORMAL_TAB_N : 1];
    if constexpr (Env::TAB_SMEM) normal_table_to_smem(s_tab);
    BlockStats bs;
    episode_staging_init(&estage);
    bs.init(sstat);
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const Rng key(p.key, Env::TAB_SMEM ? s_tab : g_normal_tab);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kStepStages; ++k) mbar_init(&full[k], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int64_t n_tiles = (p.pitch + TILE - 1) / TILE;
    auto issue = [&](int64_t tile, int stage) {            // thread 0 only
        const int64_t i0 = tile * TILE;
        const int64_t left = p.pitch - i0;
        const uint32_t bytes = (uint32_t)(left < TILE ? left : TILE) * (uint32_t)sizeof(float);
        float* dst = stage_smem + (size_t)stage * ROWS * TILE;
        mbar_expect_tx(&full[stage], bytes * ROWS);
#pragma unroll
        for (int r = 0; r < S; ++r) bulk_load(dst + r * TILE, p.state + r * p.pitch + i0, bytes, &full[stage]);
#pragma unroll
        for (int r = 0; r < A; ++r) bulk_load(dst + (S + r) * TILE, p.actions + r * p.pitch + i0, bytes, &full[stage]);
        bulk_load(dst + (S + A) * TILE, p.ep_word + i0, bytes, &full[stage]);
    };
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < kStepStages; ++k) {
            const int64_t tile = (int64_t)blockIdx.x + (int64_t)k * gridDim.x;
            if (tile < n_tiles) issue(tile, k);
        }
    }

    unsigned int c_steps = 0, c_ep = 0, c_term = 0, c_trunc = 0, c_crit = 0, c_viol = 0;
    unsigned int c_con[NIG_MAX_CONSTRAINTS];
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) c_con[k] = 0;
    StepEpisodeStats eps;

    for (int it = 0;; ++it) {
        const int64_t tile = (int64_t)blockIdx.x + (int64_t)it * gridDim.x;
        if (tile >= n_tiles) break;
        const int stage = it % kStepStages;
        mbar_wait(&full[stage], (uint32_t)((it / kStepStages) & 1));
        const float* src = stage_smem + (size_t)stage * ROWS * TILE + threadIdx.x * VEC;
        float sv[S][VEC], av[A][VEC], wv[VEC];
#pragma unroll
        for (int k = 0; k < S; ++k) ldvec<VEC>(src + k * TILE, sv[k]);
#pragma unroll
        for (int k = 0; k < A; ++k) ldvec<VEC>(src + (S + k) * TILE, av[k]);
        ldvec<VEC>(src + (S + A) * TILE, wv);
        __syncthreads();                                    // every thread has its tile in registers: the stage is free
        if (threadIdx.x == 0) {
            const int64_t next = tile + (int64_t)kStepStages * gridDim.x;
            if (next < n_tiles) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue(next, stage);
            }
        }
        const int64_t i0 = tile * TILE + (int64_t)threadIdx.x * VEC;
        if (i0 >= p.pitch) continue;
        float rw[VEC];
        uint32_t fl[VEC], vmk[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const int64_t i = i0 + e;
            const uint32_t env = p.env0 + (uint32_t)i;
            uint32_t w = __float_as_uint(wv[e]);
            float s[S], a[A], nz[NZA], ns[S];
#pragma unroll
            for (int k = 0; k < S; ++k) s[k] = sv[k][e];
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = av[k][e];
            const bool valid = i < p.n;
            const bool active = valid && !(w >> 31);
            acc_t er = (acc_t)0;                       // running episode return (plain LDG / STG beside the staged rows)
            if (p.ep_return && active) er = (acc_t)p.ep_return[i];
            if constexpr (NZ > 0) Env::NoiseGen::get_single(key, env, tick0, nz);
            else nz[0] = 0.0f;
            acc_t r; uint32_t f, vm;
            step_core<Env, CONS>(p.cons, p.max_steps, s, a, nz, 0u, w, ns, r, f, vm);
            if (!active) {            // finished env without auto-reset (or padding lane): nothing happens
#pragma unroll
                for (int k = 0; k < S; ++k) ns[k] = s[k];
                r = (acc_t)0; f = NIG_F_INACTIVE; vm = 0; w = __float_as_uint(wv[e]);
            }
            const bool done = active && (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED));
            bool need_reset = false;
            if (p.ep_return && active) {
                er = er + r;
                if (done) eps.episode((double)er, (unsigned long long)epw_step(w));
                p.ep_return[i] = (done && p.auto_reset) ? 0.0 : (double)er;
            }
            if (done) {
                if (p.auto_reset) {
                    if constexpr (Env::COOP_RESET || Env::COOP_BLOCKS > 0 || Env::COOP_FK) need_reset = true;
                    else Env::reset(key, env, tick0 + 1u, p.epoch, ns);
                    w = 0u; f |= NIG_F_RESET;
                } else w |= 0x80000000u;
            }
            if constexpr (Env::COOP_RESET) coop_reset<Env>(key, env, tick0 + 1u, p.epoch, need_reset, ns);
            else if constexpr (Env::COOP_BLOCKS > 0) coop_reset_blocks<Env>(key, env, tick0 + 1u, p.epoch, need_reset, ns, coop_buf);
            else if constexpr (Env::COOP_FK) coop_reset_fk<Env>(key, env, tick0 + 1u, p.epoch, need_reset, ns, coop_buf);
#pragma unroll
            for (int k = 0; k < S; ++k) sv[k][e] = ns[k];
            wv[e] = __uint_as_float(w);
            rw[e] = (float)r; fl[e] = f; vmk[e] = vm;
            if (active) {
                c_steps += 1; c_viol += __popc(vm);
                c_crit += (f & NIG_F_CRITICAL) ? 1u : 0u;
                if (done) { c_ep += 1; c_term += (f & NIG_F_TERMINATED) ? 1u : 0u; c_trunc += (f & NIG_F_TRUNCATED) ? 1u : 0u; }
#pragma unroll
                for (int k = 0; k < Env::NB; ++k) c_con[k] += (vm >> k) & 1u;
                if constexpr (CONS != CONS_DEFAULT) {
#pragma unroll
                    for (int k = Env::NB; k < NIG_MAX_CONSTRAINTS; ++k) c_con[k] += (vm >> k) & 1u;
                }
            }
        }
        store_rows<S, VEC>(p.state, p.pitch, p.n, i0, false, sv);
        stvec<VEC>(reinterpret_cast<float*>(p.ep_word) + i0, wv);
        if (p.reward) stvec<VEC>(p.reward + i0, rw);
        if (p.flags) {
            if constexpr (VEC == 4) *reinterpret_cast<uchar4*>(p.flags + i0) = make_uchar4(fl[0], fl[1], fl[2], fl[3]);
            else if constexpr (VEC == 2) *reinterpret_cast<uchar2*>(p.flags + i0) = make_uchar2(fl[0], fl[1]);
            else p.flags[i0] = (uint8_t)fl[0];
        }
        if (p.viol_mask) {
            if constexpr (VEC == 4) *reinterpret_cast<uchar4*>(p.viol_mask + i0) = make_uchar4(vmk[0], vmk[1], vmk[2], vmk[3]);
            else if constexpr (VEC == 2) *reinterpret_cast<uchar2*>(p.viol_mask + i0) = make_uchar2(vmk[0], vmk[1]);
            else p.viol_mask[i0] = (uint8_t)vmk[0];
        }
    }
    bs.warp_add(NIG_ST_STEPS, c_steps);
    if (__any_sync(0xffffffffu, (c_ep | c_viol | c_crit) != 0u)) {
        bs.warp_add(NIG_ST_EPISODES, c_ep);
        bs.warp_add(NIG_ST_TERMINATED, c_term);
        bs.warp_add(NIG_ST_TRUNCATED, c_trunc);
        bs.warp_add(NIG_ST_CRITICAL, c_crit);
        bs.warp_add(NIG_ST_VIOLATIONS, c_viol);
#pragma unroll
        for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k)
            if (k < p.cons.n) bs.warp_add(NIG_ST_CON0 + k, c_con[k]);
        if (p.ep_return && __any_sync(0xffffffffu, c_ep != 0u)) stage_episode_stats(bs, &estage, eps);
    }
    if (p.stats != nullptr) {
        bs.flush(p.stats);
        if (p.ep_return) flush_episode_staging(p.stats, &estage);
    }
    advance_device_tick(p.tick_dev, 1u);
}

// ================================================================================================
// reset kernel
// ================================================================================================
struct ResetArgs {
    float* state; uint32_t* ep_word; double* ep_return;
    int64_t n, pitch;
    uint32_t env0, tick, epoch;
    uint32_t* tick_dev;
    RngKey key;
    const uint8_t* mask;
    const float* init_states;
    int32_t init_aos;
    const uint32_t* tick_base;      // see base_tick(): tick / epoch above are offsets from it when non-null
};

template <class Env>
__global__ void __launch_bounds__(kThreads) reset_kernel(const __grid_constant__ ResetArgs p)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.n) return;
    if (p.mask && !p.mask[i]) return;
    const Rng key(p.key, g_normal_tab);
    float s[Env::S];
    if (p.init_states) {
#pragma unroll
        for (int k = 0; k < Env::S; ++k) s[k] = p.init_aos ? p.init_states[i * Env::S + k] : p.init_states[k * p.pitch + i];
    } else {
        Env::reset(key, p.env0 + (uint32_t)i, load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base), p.epoch + base_epoch(p.tick_base), s);
    }
#pragma unroll
    for (int k = 0; k < Env::S; ++k) p.state[k * p.pitch + i] = s[k];
    p.ep_word[i] = 0u;
    p.ep_return[i] = 0.0;
}

// stats[k] += sum over the shard copies, shards zeroed (slots 0..23 int64 counters, 24.. fp64 sums); one warp
static __global__ void __launch_bounds__(32) fold_stats_kernel(unsigned long long* __restrict__ shards, unsigned long long* __restrict__ stats)
{
    const int k = threadIdx.x;
    if (k >= NIG_STATS_SLOTS) return;
    if (k < 24) {
        unsigned long long sum = 0;
        for (int r = 0; r < kStatsShards; ++r) { sum += shards[r * NIG_STATS_SLOTS + k]; shards[r * NIG_STATS_SLOTS + k] = 0ull; }
        stats[k] += sum;
    } else {
        double* sh = reinterpret_cast<double*>(shards);
        double sum = 0.0;
        for (int r = 0; r < kStatsShards; ++r) { sum += sh[r * NIG_STATS_SLOTS + k]; sh[r * NIG_STATS_SLOTS + k] = 0.0; }
        reinterpret_cast<double*>(stats)[k] += sum;
    }
}

// sequence-tick mode: the launches of a captured sequence carry tick offsets 0 .. n-1 from tick_base[0]; this one-thread
// kernel, captured at the end of the sequence, moves the base on by n so that the next replay draws fresh noise
static __global__ void commit_ticks_kernel(uint32_t* tick_base, uint32_t by) { tick_base[0] += by; }
static __global__ void set_ticks_kernel(uint32_t* tick_base, uint32_t tick, uint32_t epoch) { tick_base[0] = tick; tick_base[1] = epoch; }

// SoA <-> AoS / ep_word <-> (step, viol, done) conversion for get/set_state
struct StateIoArgs {
    float* state; uint32_t* ep_word;
    int64_t n, pitch;
    float* ext_state; int32_t* ext_step; int32_t* ext_viol; uint8_t* ext_done;
    int32_t S, aos, to_ext;
    double* ep_return;       // import with an episode step counter: the episode's return accumulator restarts (else null)
};
static __global__ void __launch_bounds__(kThreads) state_io_kernel(const __grid_constant__ StateIoArgs p)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.n) return;
    if (p.ext_state) {
        for (int k = 0; k < p.S; ++k) {
            float* ext = p.ext_state + (p.aos ? i * p.S + k : (int64_t)k * p.pitch + i);
            float* in = p.state + (int64_t)k * p.pitch + i;
            if (p.to_ext) *ext = *in; else *in = *ext;
        }
    }
    if (p.to_ext) {
        const uint32_t w = p.ep_word[i];
        if (p.ext_step) p.ext_step[i] = (int32_t)epw_step(w);
        if (p.ext_viol) p.ext_viol[i] = (int32_t)epw_viol(w);
        if (p.ext_done) p.ext_done[i] = (uint8_t)(w >> 31);
    } else if (p.ext_step || p.ext_viol || p.ext_done) {
        // imported counters are clamped to what the word holds: step to [0, 65535], violations to [0, 32767] (epw_make)
        const uint32_t w = p.ep_word[i];
        const uint32_t st = p.ext_step ? (uint32_t)min(max(p.ext_step[i], 0), 65535) : epw_step(w);
        const uint32_t vi = p.ext_viol ? (uint32_t)max(p.ext_viol[i], 0) : epw_viol(w);
        const uint32_t dn = p.ext_done ? (uint32_t)(p.ext_done[i] != 0) : (w >> 31);
        p.ep_word[i] = epw_make(st, vi, dn);
        if (p.ep_return) p.ep_return[i] = 0.0;
    }
}

// ---- nig_rollout_host without staging copies: the slice's kernels read / write the caller's page-locked arrays themselves ----
// ingest: IndustrialEnv.reset(options = initial states) of one env slice straight from the mapped host array [n][S]
// (every warp instruction reads 512 contiguous bytes over PCIe; the AoS -> SoA transposition goes through shared memory);
// export: final observations [n][S] + per-env reward sums / violation counts / episode counts straight into the mapped host
// arrays (posted 512-byte writes). One kernel per slice replaces a copy node + a kernel on the way in and a kernel + four
// copy nodes on the way out. Requires 16-byte aligned rows (S % 4 == 0, slices start at multiples of 128 envs).
struct HostIoArgs {
    float* state; uint32_t* ep_word; double* ep_return;
    int64_t n, pitch;
    int32_t S;
    const float* in_aos;                          // ingest: mapped host [n][S]
    float* out_aos;                               // export (each may be null)
    const float* d_reward; const int32_t* d_viol; const int32_t* d_done;
    float* h_reward; int32_t* h_viol; int32_t* h_done;
};
static __global__ void __launch_bounds__(kThreads) host_ingest_kernel(const __grid_constant__ HostIoArgs p)
{
    __shared__ alignas(16) float tile[kThreads * NIG_MAX_STATE_DIM];
    const int64_t i0 = (int64_t)blockIdx.x * kThreads;
    const int64_t cnt = p.n - i0 < kThreads ? p.n - i0 : kThreads;          // envs of this CTA
    const int nvec = (int)(cnt * p.S / 4);
    const float4* src = reinterpret_cast<const float4*>(p.in_aos + i0 * p.S);
    for (int j = threadIdx.x; j < nvec; j += kThreads) reinterpret_cast<float4*>(tile)[j] = src[j];
    __syncthreads();
    const int64_t i = i0 + threadIdx.x;
    if (i >= p.n) return;
    for (int k = 0; k < p.S; ++k) p.state[(int64_t)k * p.pitch + i] = tile[threadIdx.x * p.S + k];
    p.ep_word[i] = 0u;
    p.ep_return[i] = 0.0;
}
static __global__ void __launch_bounds__(kThreads) host_export_kernel(const __grid_constant__ HostIoArgs p)
{
    __shared__ alignas(16) float tile[kThreads * NIG_MAX_STATE_DIM];
    const int64_t i0 = (int64_t)blockIdx.x * kThreads;
    const int64_t i = i0 + threadIdx.x;
    const bool valid = i < p.n;
    if (valid) {
        if (p.h_reward) p.h_reward[i] = p.d_reward[i];
        if (p.h_viol) p.h_viol[i] = p.d_viol[i];
        if (p.h_done) p.h_done[i] = p.d_done[i];
    }
    if (!p.out_aos) return;
    if (valid)
        for (int k = 0; k < p.S; ++k) tile[threadIdx.x * p.S + k] = p.state[(int64_t)k * p.pitch + i];
    __syncthreads();
    const int64_t cnt = p.n - i0 < kThreads ? p.n - i0 : kThreads;
    const int nvec = (int)(cnt * p.S / 4);
    float4* dst = reinterpret_cast<float4*>(p.out_aos + i0 * p.S);
    for (int j = threadIdx.x; j < nvec; j += kThreads) dst[j] = reinterpret_cast<const float4*>(tile)[j];
}

// ================================================================================================
// fused K-step rollout kernel
// ================================================================================================
// steps of actions staged per TMA box. Two boxes of [chunk][A][128] floats per CTA: with 16 steps the reactor kernel needed 48 KB
// + 9.5 KB static = 3 resident CTAs per SM, i.e. a second wave for the 512 CTAs of 65,536 envs (PowerGrid: 131 KB, one CTA per SM)
__host__ __device__ constexpr int tma_chunk(int action_dim) { return action_dim <= 4 ? 8 : 4; }

// Programmatic dependent launch of the fused rollout kernels (the launchers set cudaLaunchAttributeProgrammaticStreamSerialization):
// the K-step launches of an env slice follow each other on one stream; the CTAs of launch c + 1 are scheduled while launch c
// drains, copy the normal table and zero their shared counters, and wait HERE -- before the first read of anything launch c
// writes (device tick words, state, episode words, per-env sums, statistics). A no-op when launched without the attribute.
__device__ __forceinline__ void rollout_pdl_sync()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

struct RolloutArgs {
    float* state; uint32_t* ep_word; double* ep_return;
    int64_t n, pitch;
    uint32_t env0, tick, epoch;
    uint32_t* tick_dev;
    RngKey key;
    int32_t max_steps, auto_reset, n_steps;
    const float* actions;      // [K][A][pitch]
    const float* noise;        // [K][NZ][pitch] or null
    nig_policy_params_t pp;
    float* reward_sum; int32_t* viol_count; int32_t* done_count;
    int32_t accumulate;        // per-env outputs: out[i] += this launch's value instead of out[i] = ...
    unsigned long long* extrema;   // [2] keys of the min / max finished-episode return (see extremum_key); EXTREMA kernels
    double* pid_state;         // [2][A][pitch] fp64: PID integral rows, then previous-error rows (POLICY_BASELINE / PID)
    unsigned long long* stats;
    const uint32_t* tick_base; // see base_tick(): tick / epoch are offsets from it when non-null
    ConsParams cons;
};

// in-kernel policies ---------------------------------------------------------------------------------
template <class Env>
__device__ __forceinline__ void policy_uniform(const Rng& key, uint32_t env, uint32_t tick, float (&a)[Env::A])
{
    Env::uniform_actions(key, env, tick, a);
}

// get_dataset mixes (chemical_reactor.py:364-390, power_grid.py:216-232, robot_assembly.py:266-291):
// block 0 word 0 of the POLICY stream is the np.random.random() coin; the controller branch gets 8
// normals (blocks 1, 2) and 4 words (block 3); the random branch uses words 1..3 of block 0 and blocks 8..
template <class Env>
__device__ __forceinline__ void policy_pctrl(const Rng& key, const nig_policy_params_t& pp, uint32_t env, uint32_t tick,
                                             const float (&s)[Env::S], float (&a)[Env::A])
{
    const uint4 w0 = rng_words(key, env, tick, STREAM_POLICY, 0u);
    const float coin = u_open(w0.x);                       // (0, 1]
    if (coin <= pp.p_ctrl) {
        Env::policy_ctrl(key, pp, env, tick, s, a);
    } else {
        const uint32_t ww[3] = {w0.y, w0.z, w0.w};
#pragma unroll
        for (int k = 0; k < Env::A; ++k) {
            if (k < 3) a[k] = mul(pp.uniform_scale, u_sym(ww[k]));
        }
        if constexpr (Env::A > 3) {
#pragma unroll
            for (int j = 0; j < (Env::A - 3 + 3) / 4; ++j) {
                const uint4 w = rng_words(key, env, tick, STREAM_POLICY, (uint32_t)(8 + j));
                const uint32_t wq[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (3 + 4 * j + q < Env::A) a[3 + 4 * j + q] = mul(pp.uniform_scale, u_sym(wq[q]));
            }
        }
    }
}

// policy_pctrl with every random input supplied by the caller (coin in (0, 1], 8 standard normals, 8 uniforms in
// [-1, 1]): the arithmetic of the get_dataset branches without the draws, for the teacher-forced replay of the
// reference's own get_dataset transitions (selftest_policy_kernel, tests/golden/policy_forced.npz)
template <class Env>
__device__ __forceinline__ void policy_pctrl_forced(const nig_policy_params_t& pp, const float (&s)[Env::S], float coin,
                                                    const float (&z)[8], const float (&u)[8], float (&a)[Env::A])
{
    if (coin <= pp.p_ctrl) {
        const float u4[4] = {u[0], u[1], u[2], u[3]};
        Env::policy_ctrl_from(pp, s, z, u4, a);
    } else {
#pragma unroll
        for (int k = 0; k < Env::A; ++k) a[k] = mul(pp.uniform_scale, u[k]);
    }
}

// benchmarks/baseline_agents.py controllers in fp64 like numpy computes them; integ / prev are the PID agent's state
template <class Env>
__device__ __forceinline__ void policy_baseline(const Rng& key, const nig_baseline_t& b, uint32_t env, uint32_t tick,
                                                const float (&s)[Env::S], float (&a)[Env::A],
                                                double (&integ)[Env::A], double (&prev)[Env::A])
{
    constexpr int A = Env::A;
    if (b.kind == NIG_BASELINE_PID) {
#pragma unroll
        for (int k = 0; k < A; ++k) {
            const double e = dsub(b.setpoint[k], (double)s[k]);                    // :67 (first action_dim states)
            const double prop = dmul(b.kp, e);                                     // :70
            integ[k] = dadd(integ[k], e);                                          // :71
            const double it = dmul(b.ki, integ[k]);                                // :72
            const double der = dmul(b.kd, dsub(e, prev[k]));                       // :73
            double u = dadd(dadd(prop, it), der);                                  // :76
            u = u < -1.0 ? -1.0 : u;                                               // :77 np.clip
            u = u > 1.0 ? 1.0 : u;
            prev[k] = e;                                                           // :79
            a[k] = (float)u;
        }
    } else if (b.kind == NIG_BASELINE_MPC) {
#pragma unroll
        for (int k = 0; k < A; ++k) {
            double u = dmul(0.5, dsub(0.0, (double)s[k]));                         // :93-97
            u = u < -1.0 ? -1.0 : u;
            u = u > 1.0 ? 1.0 : u;
            a[k] = (float)u;
        }
    } else if (b.kind == NIG_BASELINE_CONSTANT) {
#pragma unroll
        for (int k = 0; k < A; ++k) a[k] = (float)b.setpoint[k];                   // :112
    } else {
        float u[A];
        policy_uniform<Env>(key, env, tick, u);                                    // :38-42
        const float mid = (float)(0.5 * (b.setpoint[0] + b.setpoint[1])), half = (float)(0.5 * (b.setpoint[1] - b.setpoint[0]));
#pragma unroll
        for (int k = 0; k < A; ++k) a[k] = add(mid, mul(half, u[k]));
    }
}

// ================================================================================================
// ChemicalReactor-v0: the invariant-specialised step loop of the fused rollout (uniform-random policy, default
// constraints, auto-reset -- BASELINE config #2, the loop of performance_benchmark.py:106-133)
// ================================================================================================
// Inside a free-running rollout almost everything step_core evaluates is decided before the step starts:
//   * e-stop latch s8 is 0 at every step start -- a step that sets it (T' > 350 or P' > 506625, :199-201) ends the episode
//     (_is_done, :283) and the env is re-initialised in the same step -> the PLC is always in manual mode (:126-129),
//     `estop > 0.5` is simply "tripped this step";
//   * for the same reason T <= 350 and P <= 506625 hold at every step start (fresh states are N(320, 2) / N(253312.5, 1e4)
//     with |z| < 6.4) -> the two critical constraints (:292-299) are satisfied, only `level_limits` can be violated, no
//     critical shutdown, no -1000;
//   * the alarm latch s9 is 0 or 1 -> carried as a predicate; cat / 100 of the next step is this step's reward term.
// The loop below carries these as invariants (checked once at entry by the caller, re-established by every step) and
// drops the work they decide: 9 of 12 division-guard compares (the ranges are implied: |T' - 320| <= 120 is checked on the
// value the exp argument needs anyway), the e-stop / alarm float selects and compares, the constraint mask, the penalty
// and critical-shutdown logic of constraints 0 / 1. Every arithmetic operation that remains is the one step_core performs,
// in the same order -> bit-identical results (tests/test_gpu_parity.py compares with the oracle, which knows nothing of
// this). If a guard fails (never observed: it takes |T' - 320| > 120 K, a pressure outside [1e3, 1e7] Pa or a denormal
// heat balance) the warp leaves the loop WITHOUT committing the step and the generic loop carries on from there.
__device__ __forceinline__ float cdiv_noguard(float x, float c, float rc)
{
    const float q = __fmul_rn(x, rc);
    const float r = __fmaf_rn(-q, c, x);
    return __fmaf_rn(r, rc, q);
}
#define NIG_CDIV_NG(x, c) cdiv_noguard((x), (c), 1.0f / (c))

struct RolloutAcc {            // episode / launch statistics of one thread (shared by the fast and the generic loop)
    unsigned int c_steps = 0, c_ep = 0, c_term = 0, c_trunc = 0, c_crit = 0, c_viol = 0, c_succ = 0, c_done = 0;
    unsigned int c_con[NIG_MAX_CONSTRAINTS];
    unsigned long long len_sum = 0, len_sq = 0;
    double ret_sum = 0.0, ret_sq = 0.0, rew_sum = 0.0;
};

// The six values of a step that depend on nothing but the random streams: the manual-mode actuator commands
// hp = a0 * 50000, cadj = a1 * 0.1, fadj = a2 * 0.1 (:127-129), the action penalty ((|a0| + |a1|) + |a2|) * 0.1 (:267-268)
// and the two scaled process-noise normals (:149, :159).
struct StepDraw { float hp, cadj, fadj, apen, nz0, nz1; };

__device__ __forceinline__ StepDraw reactor_step_draw(const Rng& key, uint32_t env, uint32_t tick)
{
    const uint4 w = rng_words(key, env, tick, STREAM_NOISE, 0u);
    float za, zb, a[Reactor::A];
    normal_pair(key.tab, w.x, w.y, za, zb);
    Reactor::uniform_from_words(w.z, w.w, a);
    StepDraw d;
    d.nz0 = mul(0.1f, za); d.nz1 = mul(500.0f, zb);
    d.hp = mul(a[0], 50000.0f); d.cadj = mul(a[1], 0.1f); d.fadj = mul(a[2], 0.1f);
    d.apen = mul(add(add(fabsf(a[0]), fabsf(a[1])), fabsf(a[2])), 0.1f);
    return d;
}

// where the fast loop gets a step's draw from: computed in place ...
struct DrawInKernel {
    static constexpr bool kPure = true;        // get(t) is a pure function of t: may be called one step ahead
    static constexpr bool kUserActions = false;
    const Rng& key; uint32_t env, tick0;
    __device__ __forceinline__ StepDraw get(int t, int) const { return reactor_step_draw(key, env, tick0 + (uint32_t)t); }
    __device__ __forceinline__ void done(int, int) const {}
};
struct DrawInKernel2 {         // two envs per thread: lane 0 / 1 of the value type
    static constexpr bool kPure = true, kUserActions = false;
    const Rng& key; uint32_t env[2], tick0;
    __device__ __forceinline__ StepDraw get(int t, int lane) const { return reactor_step_draw(key, env[lane], tick0 + (uint32_t)t); }
    __device__ __forceinline__ void done(int, int) const {}
};

// ... or built from caller-supplied actions (NIG_POLICY_ACTIONS): np.clip(action, -1, 1) (base.py:167), then the same derived
// values; the process noise still comes from words x, y of the step's Philox block (Reactor::NoiseGen)
__device__ __forceinline__ StepDraw reactor_draw_from_actions(const Rng& key, uint32_t env, uint32_t tick, const float (&a_raw)[Reactor::A])
{
    float a[Reactor::A];
#pragma unroll
    for (int j = 0; j < Reactor::A; ++j) {
        float v = a_raw[j];
        v = v < -1.0f ? -1.0f : v;
        v = v > 1.0f ? 1.0f : v;
        a[j] = v;
    }
    const uint4 w = rng_words(key, env, tick, STREAM_NOISE, 0u);
    float za, zb;
    normal_pair(key.tab, w.x, w.y, za, zb);
    StepDraw d;
    d.nz0 = mul(0.1f, za); d.nz1 = mul(500.0f, zb);
    d.hp = mul(a[0], 50000.0f); d.cadj = mul(a[1], 0.1f); d.fadj = mul(a[2], 0.1f);
    d.apen = mul(add(add(fabsf(a[0]), fabsf(a[1])), fabsf(a[2])), 0.1f);
    return d;
}
// action rows [K][A][pitch] read one step ahead into registers (the LDG flavour of rollout_kernel; a_pf holds step t's
// actions whenever get(t) is called and step t + 1's afterwards)
struct DrawActionsLdg {
    static constexpr bool kPure = false, kUserActions = true;
    const Rng& key; uint32_t env, tick0; const float* actions; int64_t pitch, ic; int n_steps; float (&a_pf)[Reactor::A];
    __device__ __forceinline__ StepDraw get(int t, int)
    {
        float a[Reactor::A];
#pragma unroll
        for (int k = 0; k < Reactor::A; ++k) a[k] = a_pf[k];
        const int tn = t + 1 < n_steps ? t + 1 : t;
#pragma unroll
        for (int k = 0; k < Reactor::A; ++k) a_pf[k] = __ldcs(actions + ((int64_t)tn * Reactor::A + k) * pitch + ic);
        return reactor_draw_from_actions(key, env, tick0 + (uint32_t)t, a);
    }
    __device__ __forceinline__ void done(int, int) const {}
    __device__ __forceinline__ void rewind(int t)           // the loop left at step t without committing it: a_pf = step t again
    {
#pragma unroll
        for (int k = 0; k < Reactor::A; ++k) a_pf[k] = __ldcs(actions + ((int64_t)t * Reactor::A + k) * pitch + ic);
    }
};

// action boxes [kTmaChunk][A][kThreads] staged in shared memory by cp.async.bulk.tensor.3d (the TMA flavour): the same
// double-buffer protocol as the generic loop of rollout_kernel -- wait for the box at its first step, one CTA barrier and a
// refill at its last -- so warps of one CTA may run either loop (and change over on a failed guard) without losing count
struct DrawActionsTma {
    static constexpr bool kPure = false, kUserActions = true;
    static constexpr int kTmaChunk = tma_chunk(Reactor::A);
    const Rng& key; uint32_t env, tick0; float* act_smem; uint64_t* bars; const CUtensorMap* amap; int n_chunks;
    __device__ __forceinline__ StepDraw get(int t, int) const
    {
        const int c = t / kTmaChunk, tt = t % kTmaChunk, b = c & 1;
        if (tt == 0) mbar_wait(&bars[b], (uint32_t)((c >> 1) & 1));
        const float* src = act_smem + ((size_t)b * kTmaChunk + tt) * Reactor::A * kThreads;
        float a[Reactor::A];
#pragma unroll
        for (int k = 0; k < Reactor::A; ++k) a[k] = src[k * kThreads + threadIdx.x];
        return reactor_draw_from_actions(key, env, tick0 + (uint32_t)t, a);
    }
    __device__ __forceinline__ void done(int t, int n_steps) const
    {
        const int c = t / kTmaChunk, tt = t % kTmaChunk, b = c & 1;
        if (tt == kTmaChunk - 1 || t == n_steps - 1) {
            __syncthreads();                       // everyone finished reading buffer b
            if (threadIdx.x == 0 && c + 2 < n_chunks) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(&bars[b], kTmaChunk * Reactor::A * kThreads * (uint32_t)sizeof(float));
                tma_load_3d(act_smem + (size_t)b * kTmaChunk * Reactor::A * kThreads, amap, (int)(blockIdx.x * kThreads), 0, (c + 2) * kTmaChunk, &bars[b]);
            }
        }
    }
};

// ---- one or two envs per thread -------------------------------------------------------------------------------------
// The loop below is written once over a value type V: float (one env per thread) or F2 (two envs per thread, every
// add / mul / fma of the physics issued as ONE packed instruction -- add.rn.f32x2 / mul.rn.f32x2 / fma.rn.f32x2, SASS FADD2 /
// FMUL2 / FFMA2, IEEE round-to-nearest per lane, so the results are the scalar ones bit for bit). Compares, selects, min / max
// and conversions have no packed form and stay per lane; so do the RNG and the table normals.
struct F2 { float x, y; };
struct B2 { bool x, y; };
__device__ __forceinline__ float2 f2v(F2 a) { return make_float2(a.x, a.y); }
__device__ __forceinline__ F2 v2f(float2 a) { return F2{a.x, a.y}; }
template <class V> struct VT;
template <> struct VT<float> {
    static constexpr int N = 1; using M = bool;
    __device__ static __forceinline__ float bc(float c) { return c; }
    __device__ static __forceinline__ float get(float v, int) { return v; }
    __device__ static __forceinline__ void set(float& v, int, float x) { v = x; }
    __device__ static __forceinline__ bool getm(bool m, int) { return m; }
    __device__ static __forceinline__ void setm(bool& m, int, bool x) { m = x; }
};
template <> struct VT<F2> {
    static constexpr int N = 2; using M = B2;
    __device__ static __forceinline__ F2 bc(float c) { return F2{c, c}; }
    __device__ static __forceinline__ float get(F2 v, int k) { return k ? v.y : v.x; }
    __device__ static __forceinline__ void set(F2& v, int k, float x) { if (k) v.y = x; else v.x = x; }
    __device__ static __forceinline__ bool getm(B2 m, int k) { return k ? m.y : m.x; }
    __device__ static __forceinline__ void setm(B2& m, int k, bool x) { if (k) m.y = x; else m.x = x; }
};
// packed arithmetic (the scalar add / mul / sub are in nig_envs.cuh).
// TOOLCHAIN: ptxas 12.9 contracts `mul.rn.f32x2` followed by `add.rn.f32x2` into ONE FFMA2 -- despite the explicit .rn on
// both (the PTX is right: cicc keeps them apart) and despite -fmad=false, also when the add is written fma(m, 1, c) or the
// product fma(a, b, -0), and through an empty asm volatile on the halves (scalar mul.rn + add.rn are never contracted). A
// single rounding instead of two changes the last bit: the first packed build differed from the oracle in 12 % of the
// pressure / concentration values after 70 steps. Work-around: packed sums are written a * ONE + b and b * MINUS_ONE + a with
// the +-1 read from constant memory, which ptxas cannot fold (FFMA2 R, R, UR.F32, R: same issue cost as FADD2, exact: RN(a+b)).
static __device__ __constant__ float g_f2_one = 1.0f, g_f2_mone = -1.0f;
__device__ __forceinline__ F2 add(F2 a, F2 b) { const float o = g_f2_one; return v2f(__ffma2_rn(f2v(a), make_float2(o, o), f2v(b))); }
__device__ __forceinline__ F2 mul(F2 a, F2 b) { return v2f(__fmul2_rn(f2v(a), f2v(b))); }
__device__ __forceinline__ F2 sub(F2 a, F2 b) { const float o = g_f2_mone; return v2f(__ffma2_rn(f2v(b), make_float2(o, o), f2v(a))); }
__device__ __forceinline__ float vfma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ F2 vfma(F2 a, F2 b, F2 c) { return v2f(__ffma2_rn(f2v(a), f2v(b), f2v(c))); }
__device__ __forceinline__ float vneg(float a) { return -a; }
__device__ __forceinline__ F2 vneg(F2 a) { return F2{-a.x, -a.y}; }
__device__ __forceinline__ float vabs(float a) { return fabsf(a); }
__device__ __forceinline__ F2 vabs(F2 a) { return F2{fabsf(a.x), fabsf(a.y)}; }
__device__ __forceinline__ float rcp_approx(float a) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(a)); return y; }
__device__ __forceinline__ F2 rcp_approx(F2 a) { return F2{rcp_approx(a.x), rcp_approx(a.y)}; }
// comparisons against a constant / selects, per lane
#define NIG_CMP(name, op) \
    __device__ __forceinline__ bool name(float a, float c) { return a op c; } \
    __device__ __forceinline__ B2 name(F2 a, float c) { return B2{a.x op c, a.y op c}; }
NIG_CMP(vgt, >) NIG_CMP(vlt, <) NIG_CMP(vge, >=) NIG_CMP(vle, <=)
__device__ __forceinline__ bool mand(bool a, bool b) { return a && b; }
__device__ __forceinline__ B2 mand(B2 a, B2 b) { return B2{a.x && b.x, a.y && b.y}; }
__device__ __forceinline__ bool mor(bool a, bool b) { return a || b; }
__device__ __forceinline__ B2 mor(B2 a, B2 b) { return B2{a.x || b.x, a.y || b.y}; }
__device__ __forceinline__ bool mnot(bool a) { return !a; }
__device__ __forceinline__ B2 mnot(B2 a) { return B2{!a.x, !a.y}; }
__device__ __forceinline__ bool mall(bool a) { return a; }
__device__ __forceinline__ bool mall(B2 a) { return a.x && a.y; }
__device__ __forceinline__ bool many(bool a) { return a; }
__device__ __forceinline__ bool many(B2 a) { return a.x || a.y; }
__device__ __forceinline__ float vsel(bool m, float a, float b) { return m ? a : b; }
__device__ __forceinline__ F2 vsel(B2 m, F2 a, F2 b) { return F2{m.x ? a.x : b.x, m.y ? a.y : b.y}; }
__device__ __forceinline__ float vselc(bool m, float a, float b) { return m ? a : b; }                 // constants
__device__ __forceinline__ F2 vselc(B2 m, float a, float b) { return F2{m.x ? a : b, m.y ? a : b}; }
__device__ __forceinline__ F2 py_clamp(F2 v, float lo, float hi) { return F2{py_clamp(v.x, lo, hi), py_clamp(v.y, lo, hi)}; }

template <class V>
__device__ __forceinline__ V cdiv_noguard_v(V x, float c, float rc)
{
    using T = VT<V>;
    const V q = mul(x, T::bc(rc));
    const V r = vfma(vneg(q), T::bc(c), x);
    return vfma(r, T::bc(rc), q);
}
#define NIG_CDIV_V(x, c) cdiv_noguard_v((x), (c), 1.0f / (c))

// spec_expf (nig_math.cuh) over V on the fast loop's range |x| <= 6, bit for bit: the exp argument -(T' - 320) / 20 of a
// committed step, since the loop's guard requires |T' - 320| <= 120 (a lane outside it fails the guard and the step is
// redone by the generic loop, so whatever this returns there is discarded). On that range
//   * spec_expf's clamps to [-104, 89] never act;
//   * t = x * log2e is in [-8.66, 8.66]: m = RN(t + 1.5 * 2^23) lies in [2^23, 2^24), where the float spacing is 1, so
//     m - 1.5 * 2^23 is rint(t), ties to even (exact for |t| < 2^22), and the bit pattern of m is 0x4b400000 + n;
//     (pattern + 127) << 23 is then the pattern of 2^n (0x4b400000 << 23 wraps to 0), instead of FRND + F2I;
//   * p is in [0.70, 1.42] and |n| <= 9, so p * 2^n is a normal float and one multiply by 2^n equals spec_expf's two
//     multiplies by 2^(n >> 1) and 2^(n - (n >> 1)).
// n is +0 where rintf gives -0 (t in (-0.5, -0]); r = fma(n, -c, x) is x either way, and every Horner step then adds a
// nonzero constant. Cody-Waite and Horner are spec_expf's. tests/test_fast_exp_cpu.py checks all 2.2e9 binary32 in [-6, 6]
// against the oracle's spec_expf.
template <class V>
__device__ __forceinline__ V spec_expf_small_v(V x)
{
    using T = VT<V>;
    const V t = mul(x, T::bc(0x1.715476p+0f));
    const V m = add(t, T::bc(0x1.8p23f));
    const V n = add(m, T::bc(-0x1.8p23f));
    V r = vfma(n, T::bc(-0x1.62e4p-1f), x);
    r = vfma(n, T::bc(-0x1.7f7d1cp-20f), r);
    V p = T::bc(0x1.a17e08p-13f);
    p = vfma(p, r, T::bc(0x1.6d7548p-10f));
    p = vfma(p, r, T::bc(0x1.1110a6p-7f));
    p = vfma(p, r, T::bc(0x1.5554acp-5f));
    p = vfma(p, r, T::bc(0x1.555556p-3f));
    p = vfma(p, r, T::bc(0x1.0p-1f));
    p = vfma(p, r, T::bc(1.0f));
    p = vfma(p, r, T::bc(1.0f));
    V s;
#pragma unroll
    for (int k = 0; k < T::N; ++k) T::set(s, k, __uint_as_float((__float_as_uint(T::get(m, k)) + 127u) << 23));
    return mul(p, s);
}

// returns the number of steps committed (== n_steps unless a guard failed). V = float: one env (env[0]); V = F2: two envs.
// NX appended SafetyWrapper bounds (CONS_BOUNDS1 / 2: non-critical lo <= T <= hi or lo <= P <= hi on the PRE-step state, the
// temperature / pressure bands of BASELINE config 4) ride along as straight-line code: one select of the bounded value, two
// compares, a selected penalty add after the built-ins' penalties (base.py:179-183 walks the constraints in order), counters.
struct FastBounds { float lo[2], hi[2], pen[2]; bool use_p[2]; };

// the appended bounds of p.cons the fast loop can carry (warp-uniform): pure, non-critical, on state component 0 (T) or 1 (P)
template <int NX>
__device__ __forceinline__ bool fast_bounds_from(const ConsParams& cp, FastBounds& fb)
{
    bool ok = true;
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        const nig_constraint_t& c = cp.c[Reactor::NB + j];
        ok = ok && c.kind == NIG_CON_BOUND && c.ai < 0 && c.critical == 0 && (c.si == 0 || c.si == 1);
        fb.lo[j] = c.lo; fb.hi[j] = c.hi; fb.pen[j] = c.penalty; fb.use_p[j] = c.si == 1;
    }
    return ok;
}

template <class V, bool EXTREMA, class Src, int NX = 0>
__device__ __forceinline__ int reactor_fast_steps_v(Src& src, const Rng& key, const uint32_t (&env)[VT<V>::N], uint32_t tick0, uint32_t epoch,
                                                    int n_steps, int max_steps, float (&s)[VT<V>::N][Reactor::S],
                                                    uint32_t (&ep_st)[VT<V>::N], uint32_t (&ep_vi)[VT<V>::N], float (&ep_ret_)[VT<V>::N],
                                                    float (&rsum_)[VT<V>::N], RolloutAcc (&acc)[VT<V>::N], float& r_lo, float& r_hi,
                                                    const FastBounds& fb = FastBounds{})
{
    using T_ = VT<V>;
    using M = typename T_::M;
    constexpr int N = T_::N;
    static_assert(NX == 0 || N == 1, "appended bounds: one env per thread only");
    unsigned int c_x[NX > 0 ? NX : 1] = {0u};
    bool xbad[NX > 0 ? NX : 1] = {false};
    V T, P, cool, feed, conc, cat, hx, rv, level, bt, catd, ep_ret, rsum;
    M alarm;
    int t_trunc[N];
    unsigned int c_lvl[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        T_::set(T, k, s[k][0]); T_::set(P, k, s[k][1]); T_::set(cool, k, s[k][2]); T_::set(feed, k, s[k][3]); T_::set(conc, k, s[k][4]);
        T_::set(cat, k, s[k][5]); T_::set(hx, k, s[k][6]); T_::set(rv, k, s[k][7]); T_::set(level, k, s[k][10]); T_::set(bt, k, s[k][11]);
        T_::setm(alarm, k, __float_as_uint(s[k][9]) != 0u);
        T_::set(catd, k, __fdiv_rn(s[k][5], 100.0f));
        T_::set(ep_ret, k, ep_ret_[k]); T_::set(rsum, k, rsum_[k]);
        t_trunc[k] = max_steps - (int)ep_st[k] - 1;      // loop index of the step at which the running episode is truncated (base.py:191)
        c_lvl[k] = 0u;
    }
    int t = 0;
    // the draw of step t + 1 is computed during step t (it depends on nothing but the counters): the Philox block, the table
    // normals and the action scaling leave the head of the step's dependency chain and fill the physics' issue gaps instead.
    // Measured +6.3 % at 65,536 envs (3.5 warps per sub-partition: latency shows), -12 % in the two-env flavour (12 more live
    // registers), so one env per thread only (profiles/r02_h_draw_ahead_ab.txt)
    constexpr bool kAhead = Src::kPure && N == 1;
    StepDraw nxt[N];
    if constexpr (kAhead) {
#pragma unroll
        for (int k = 0; k < N; ++k) nxt[k] = src.get(0, k);
    }
#pragma unroll 1
    for (; t < n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        V nz0, nz1, hp, cadj, fadj, apen;
#pragma unroll
        for (int k = 0; k < N; ++k) {
            StepDraw dr;
            if constexpr (kAhead) { dr = nxt[k]; nxt[k] = src.get(t + 1, k); }
            else dr = src.get(t, k);
            T_::set(nz0, k, dr.nz0); T_::set(nz1, k, dr.nz1); T_::set(hp, k, dr.hp); T_::set(cadj, k, dr.cadj); T_::set(fadj, k, dr.fadj);
            T_::set(apen, k, dr.apen);
        }
        const M lvl_bad = mnot(mand(vge(level, 20.0f), vle(level, 90.0f)));     // :302-305 on the pre-step state
        // _dynamics (:109-226), manual mode
        const V c01 = mul(T_::bc(0.1f), conc);
        const V kca = mul(c01, catd);
        const V rh = mul(kca, T_::bc(10000.0f));
        const V ch = mul(mul(mul(cool, T_::bc(100.0f)), sub(T, hx)), T_::bc(0.1f));
        const V num = sub(add(hp, rh), ch);
        M ok = vge(vabs(num), 0x1.0p-120f);
        // caller-supplied actions may be NaN (np.clip keeps it): |a0| + |a1| + |a2| <= 3 fails then and the step is the generic loop's
        if constexpr (Src::kUserActions) ok = mand(ok, vle(apen, 1.0f));
        const V dT = add(NIG_CDIV_V(num, 418000.0f), nz0);
        const V nT = add(T, mul(dT, T_::bc(0.1f)));
        const V d = sub(nT, T_::bc(320.0f));
        ok = mand(ok, vle(vabs(d), 120.0f));            // 200 <= T' <= 440: T' / T and -(T' - 320) / 20 are in the proven domain
        const V y0 = rcp_approx(T);
        const V e0 = vfma(vneg(T), y0, T_::bc(1.0f));
        const V y1 = vfma(y0, e0, y0);
        const V q0 = vfma(nT, y1, T_::bc(0.0f));
        const V q = vfma(y1, vfma(vneg(T), q0, nT), q0);                        // == __fdiv_rn(nT, T) (DivFast::vdiv)
        const V pfr = mul(c01, T_::bc(1000.0f));                               // mul(mul(conc, 0.1f), 1000.0f)
        V nP = add(add(mul(P, q), mul(pfr, T_::bc(0.1f))), nz1);
        const V nrv = py_clamp(add(rv, mul(sub(nP, T_::bc(506625.0f)), T_::bc(0.001f))), 0.0f, 100.0f);
        {
            const V x = sub(nP, mul(mul(nrv, T_::bc(0.01f)), T_::bc(10000.0f)));
            const V xr = vsel(vgt(x, 101325.0f), x, T_::bc(101325.0f));
            nP = vsel(vgt(nrv, 0.0f), xr, nP);
        }
        ok = mand(ok, vle(vabs(sub(nP, T_::bc(5.0e6f))), 4.999e6f));   // 1e3 <= P' < 1e7: |P' - 253312.5| is 0 or >= 2^-14, finite
        const V ex = spec_expf_small_v(NIG_CDIV_V(vneg(d), 20.0f));
        const V rr = mul(kca, ex);
        if (__builtin_expect(!__all_sync(0xffffffffu, mall(ok)), 0)) break;     // (uniform) redo this step in the generic loop
        src.done(t, n_steps);
        // the rest of the step after the vote: the values it replaces are dead from here on (a failed guard leaves the loop
        // with the pre-step state), so each new value can take its old value's register instead of a copy at the commit
        const V ncool = py_clamp(add(cool, cadj), 10.0f, 100.0f);
        const V feed_v = add(feed, fadj);
        const V nfeed = py_clamp(feed_v, 5.0f, 50.0f);
        V fdil = mul(nfeed, T_::bc(0.001f));
        fdil = vsel(vgt(feed_v, 5.0f), fdil, T_::bc(0x1.47ae14p-8f));
        fdil = vsel(vlt(feed_v, 50.0f), fdil, T_::bc(0x1.99999ap-5f));
        const V cv = add(conc, mul(sub(rr, fdil), T_::bc(0.1f)));
        const V nconc = vsel(vgt(cv, 0.0f), cv, T_::bc(0.0f));
        const V catv = sub(cat, vselc(vgt(nT, 340.0f), 0.001f, 0.0001f));
        const V ncat = vsel(vgt(catv, 50.0f), catv, T_::bc(50.0f));
        const V nhx = add(hx, mul(mul(T_::bc(0.1f), sub(add(T_::bc(290.0f), mul(cool, T_::bc(0.1f))), hx)), T_::bc(0.1f)));
        const M trip = mor(vgt(nT, 350.0f), vgt(nP, 506625.0f));                // :199 -> estop' = alarm' = 1
        const M nalarm = mor(alarm, mor(vgt(nT, 345.0f), vgt(nP, 480000.0f)));  // :197
        const V nlevel = py_clamp(add(level, mul(mul(sub(nfeed, T_::bc(20.0f)), T_::bc(0.1f)), T_::bc(0.1f))), 0.0f, 100.0f);
        const V nbt = add(bt, T_::bc(0.1f));
        // _compute_reward (:228-270) on the new state, then the level penalty (base.py:179-183)
        V r = mul(nconc, T_::bc(100.0f));                // (0 + x of step_core: x >= +0, never -0, so the add is the identity)
        r = sub(r, mul(vabs(d), T_::bc(0.5f)));
        r = sub(r, mul(NIG_CDIV_V(vabs(sub(nP, T_::bc(253312.5f))), 1000.0f), T_::bc(0.1f)));
        const V ncatd = NIG_CDIV_V(ncat, 100.0f);
        r = add(r, mul(ncatd, T_::bc(10.0f)));
        const M band = mand(vge(nlevel, 30.0f), vle(nlevel, 80.0f));
        r = vsel(band, add(r, T_::bc(5.0f)), sub(r, mul(vabs(sub(nlevel, T_::bc(55.0f))), T_::bc(0.2f))));
        r = vsel(nalarm, sub(r, T_::bc(50.0f)), r);
        r = vsel(trip, sub(r, T_::bc(200.0f)), r);
        r = sub(r, apen);
        r = vsel(lvl_bad, add(r, T_::bc(-25.0f)), r);
        if constexpr (NX > 0) {
#pragma unroll
            for (int j = 0; j < NX; ++j) {
                const float v = fb.use_p[j] ? T_::get(P, 0) : T_::get(T, 0);           // pre-step value (committed below)
                xbad[j] = !((fb.lo[j] <= v) && (v <= fb.hi[j]));
                const float rp = add(T_::get(r, 0), fb.pen[j]);
                T_::set(r, 0, xbad[j] ? rp : T_::get(r, 0));
            }
        }
        rsum = add(rsum, r);
        ep_ret = add(ep_ret, r);
        T = nT; P = nP; cool = ncool; feed = nfeed; conc = nconc; cat = ncat; hx = nhx; rv = nrv; level = nlevel; bt = nbt;
        alarm = nalarm; catd = ncatd;
        const M term = mor(mor(trip, vlt(nlevel, 5.0f)), mor(vgt(nlevel, 95.0f), vgt(nbt, 50.0f)));   // _is_done (:272-290)
        M fin;
#pragma unroll
        for (int k = 0; k < N; ++k) {
            const unsigned int bad = T_::getm(lvl_bad, k) ? 1u : 0u;
            c_lvl[k] += bad; ep_vi[k] += bad;
            if constexpr (NX > 0) {
#pragma unroll
                for (int j = 0; j < NX; ++j) { const unsigned int b = xbad[j] ? 1u : 0u; c_x[j] += b; ep_vi[k] += b; }
            }
            T_::setm(fin, k, T_::getm(term, k) || t >= t_trunc[k]);
        }
        if (__any_sync(0xffffffffu, many(fin))) {
#pragma unroll
            for (int k = 0; k < N; ++k) {
                const bool fk = T_::getm(fin, k);
                if (fk) {
                    const float ret = T_::get(ep_ret, k);
                    const unsigned long long len = (unsigned long long)(max_steps - (t_trunc[k] - t));
                    acc[k].c_ep += 1; acc[k].c_done += 1;
                    acc[k].c_term += T_::getm(term, k) ? 1u : 0u;
                    acc[k].c_trunc += (t >= t_trunc[k]) ? 1u : 0u;
                    acc[k].c_succ += (ret > 0.0f) ? 1u : 0u;
                    acc[k].len_sum += len; acc[k].len_sq += len * len;
                    acc[k].ret_sum += (double)ret; acc[k].ret_sq += (double)ret * (double)ret;
                    if constexpr (EXTREMA) { r_lo = ret < r_lo ? ret : r_lo; r_hi = ret > r_hi ? ret : r_hi; }
                }
                // the fresh state (Reactor::reset: 2 Philox blocks, 8 table normals) drawn by the whole warp for its finished
                // lane(s): one pair of normals per helper lane instead of the full draw under a one-lane mask
                float f[Reactor::S];
                coop_reset<Reactor>(key, env[k], tick + 1u, epoch, fk, f);
                if (fk) {
                    T_::set(T, k, f[0]); T_::set(P, k, f[1]); T_::set(cool, k, f[2]); T_::set(feed, k, f[3]); T_::set(conc, k, f[4]);
                    T_::set(cat, k, f[5]); T_::set(hx, k, f[6]); T_::set(rv, k, f[7]); T_::set(level, k, f[10]); T_::set(bt, k, f[11]);
                    T_::setm(alarm, k, false);
                    // a reset draws cat = 95 + 2 z with |z| <= 6.34 (all of the table normal's range), i.e. cat in [82.3, 107.7],
                    // where the constant division is the IEEE quotient (tests/test_fast_exp_cpu.py checks every such cat)
                    T_::set(catd, k, NIG_CDIV_V(f[5], 100.0f));
                    ep_vi[k] = 0u; T_::set(ep_ret, k, 0.0f);
                    t_trunc[k] = t + max_steps;
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < N; ++k) {
        s[k][0] = T_::get(T, k); s[k][1] = T_::get(P, k); s[k][2] = T_::get(cool, k); s[k][3] = T_::get(feed, k); s[k][4] = T_::get(conc, k);
        s[k][5] = T_::get(cat, k); s[k][6] = T_::get(hx, k); s[k][7] = T_::get(rv, k);
        s[k][8] = 0.0f; s[k][9] = T_::getm(alarm, k) ? 1.0f : 0.0f; s[k][10] = T_::get(level, k); s[k][11] = T_::get(bt, k);
        ep_st[k] = (uint32_t)(max_steps - (t_trunc[k] - t + 1));
        ep_ret_[k] = T_::get(ep_ret, k); rsum_[k] = T_::get(rsum, k);
        acc[k].c_steps += (unsigned int)t;
        acc[k].c_viol += c_lvl[k];
        acc[k].c_con[2] += c_lvl[k];
        if constexpr (NX > 0) {
#pragma unroll
            for (int j = 0; j < NX; ++j) { acc[k].c_viol += c_x[j]; acc[k].c_con[Reactor::NB + j] += c_x[j]; }
        }
    }
    return t;
}

// one env per thread: the scalar instantiation behind the interface the one-env kernels use
template <bool EXTREMA, class Src, int NX = 0>
__device__ __forceinline__ int reactor_fast_steps(Src& src, const Rng& key, uint32_t env, uint32_t tick0, uint32_t epoch, int n_steps, int max_steps,
                                                  float (&s)[Reactor::S], uint32_t& ep_st, uint32_t& ep_vi, float& ep_ret, float& rsum,
                                                  RolloutAcc& acc, float& r_lo, float& r_hi, const FastBounds& fb = FastBounds{})
{
    const uint32_t envs[1] = {env};
    auto& s1 = reinterpret_cast<float (&)[1][Reactor::S]>(s);
    auto& st1 = reinterpret_cast<uint32_t (&)[1]>(ep_st);
    auto& vi1 = reinterpret_cast<uint32_t (&)[1]>(ep_vi);
    auto& er1 = reinterpret_cast<float (&)[1]>(ep_ret);
    auto& rs1 = reinterpret_cast<float (&)[1]>(rsum);
    auto& ac1 = reinterpret_cast<RolloutAcc (&)[1]>(acc);
    return reactor_fast_steps_v<float, EXTREMA, Src, NX>(src, key, envs, tick0, epoch, n_steps, max_steps, s1, st1, vi1, er1, rs1, ac1, r_lo, r_hi, fb);
}

// ================================================================================================
// PowerGrid-v0: the lean step loop of the fused rollout (uniform-random policy, default constraints, auto-reset --
// BASELINE config #3). The generic loop costs 1,390 instructions per step for 228 algorithmic operations; 200 of them
// are register moves (ns -> s under the `active` / `done` selects), 100 are compares. This loop
//   * updates the 32 state values IN PLACE, block of noise by block of noise (a Philox block's four normals are consumed
//     as soon as they are drawn: no ns[32], no nz[23]);
//   * carries, like the reactor loop above, the invariants a free-running env satisfies at every step start -- the
//     frequency deviation is finite with |f| <= 1 and the voltages are in [0.9, 1.1] (else the previous step ended the
//     episode and the state is fresh: V = 1 + 0.01 z with |z| < 6.4), generation is in [+0, 100] (a clamp result or
//     N(base, 2)), loads are finite and >= +0 -- checked once per warp at entry, re-established by every step. Under them
//       - V' - 1 is exact (Sterbenz), so the sixteen range compares of `voltage_limits` (:17-21) and the sixteen of `_is_done`
//         (:179-192) become min / max trees (FMNMX3) of e_i = V_i - 1 compared with the exactly representable
//         0.95f - 1, 1.05f - 1, 0.9f - 1, 1.1f - 1; the reward's |V' - 1| is the same e_i;
//       - np.clip(gen + a, 0, 100) is max(min(g, 100), 0) (finite g, never -0.0), `generation_limits` (:24-30) is
//         "the clamp changed nothing"; the load clamp is max(l, +0) (finite l);
//       - frequency_stability / voltage_limits violations are critical: they end the episode, so their counters (and the
//         critical-shutdown counter) are bumped in the episode-end branch, only generation_limits counts per step;
//   * checks the one division guard (|f_dot numerator| in [2^-120, 2^100]) BEFORE anything is committed: a warp whose
//     guard fails leaves the loop and the generic loop redoes the step with the IEEE division.
// Every arithmetic operation that remains is the one step_core performs, in the same order -> bit-identical results
// (tests/test_gpu_parity.py, tests/test_gpu_round2.py compare with the oracle, which knows nothing of this).
// ================================================================================================
__device__ __forceinline__ bool grid_fast_invariants(const float (&s)[Grid::S])
{
    bool inv = fabsf(s[0]) <= 1.0f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        inv = inv && s[1 + i] >= 0.9f && s[1 + i] <= 1.1f;
        inv = inv && __float_as_uint(s[9 + i]) <= 0x42c80000u;       // +0 <= gen <= 100, not -0, not NaN
        inv = inv && __float_as_uint(s[17 + i]) <= 0x7f7fffffu;      // load finite, >= +0
    }
    return inv;
}

// ---- the normal table, replicated 8 x in shared memory ---------------------------------------------------------------
// 23 table normals per step (+ 4 per step for the resets) are 39 LDS.128 per warp-step; the draws concentrate on the ~50 rows
// of the first octaves of p, so the lanes of a quarter-warp hit different rows of the same four banks all the time: ncu counts
// 8.4 shared-memory wavefronts per LDS.128 (4 is the minimum for 32 x 16 B) and the SM's shared-memory data pipe 64 % busy --
// at 1.8e10 env-steps/s; it would saturate at 2.9e10. The dedicated PowerGrid kernel therefore keeps EIGHT interleaved copies of
// the table, row r of copy c at float4 index 8 r + c, and lane l reads copy l mod 8: the eight lanes of a quarter-warp always
// touch eight different bank groups -> exactly 4 wavefronts per LDS.128, whatever the rows. 65.7 KB per CTA (dynamic).
constexpr int kTabRep = 8;                     // the fused rollout kernel; the single-step kernel also runs with 4 (two lanes per copy)
template <int REP>
__device__ __forceinline__ void normal_table_to_smem_rep(float4* dst)
{
    static_assert(REP == 8 || REP == 4, "copies per bank-group set");
    for (int i = threadIdx.x; i < NIG_NORMAL_TAB_N * REP; i += blockDim.x) dst[i] = g_normal_tab[i / REP];
}
// spec_normal with the replicated table; tabl = table base + (lane & (REP - 1))
template <int REP>
__device__ __forceinline__ float spec_normal_rep(const float4* tabl, uint32_t w)
{
    constexpr int SH = REP == 8 ? 16 : 17;
    constexpr uint32_t MASK = REP == 8 ? 0xfff8u : 0x7ffcu;
    const uint32_t v = w * 2u + 1u;
    const float f = __uint2float_rn(v);
    const float4 c = tabl[((__float_as_uint(f) >> SH) & MASK) - 2032u * REP];
    const float z = __fmaf_rn(__fmaf_rn(__fmaf_rn(c.w, f, c.z), f, c.y), f, c.x);
    return __uint_as_float(__float_as_uint(z) ^ (w & 0x80000000u));
}
template <int REP>
__device__ __forceinline__ void rng_normals4_rep(const Rng& key, const float4* tabl, uint32_t env, uint32_t tick, uint32_t stream, uint32_t j, float (&z)[4])
{
    const uint4 w = rng_words(key, env, tick, stream, j);
    z[0] = spec_normal_rep<REP>(tabl, w.x); z[1] = spec_normal_rep<REP>(tabl, w.y);
    z[2] = spec_normal_rep<REP>(tabl, w.z); z[3] = spec_normal_rep<REP>(tabl, w.w);
}

// ---- block-granular cooperative reset of the dedicated PowerGrid kernel (same draws as coop_reset_blocks / Grid::reset) ----
// The lanes of a warp own consecutive envs. Resetting lanes publish their lane index in rank order (list), the (rank, block)
// work items are dealt four ranks per round to the four quarter-warps -- lane l always draws block l mod 8 --, each producer
// stores its four raw values with one STS.128 into row `rank` of the warp's buffer (rows padded to 36 floats: the owners'
// LDS.128 of different rows fall into different banks), the owners rebuild their state from their row.
constexpr int kGridResetRow = 36;
constexpr int kGridResetRanks = 8;                 // rows of a warp's buffer: the resetting lanes are served eight ranks at a time
template <int REP>
__device__ __forceinline__ void grid_coop_reset(const Rng& key, const float4* tab8l, uint32_t env, uint32_t tick, uint32_t epoch, bool need,
                                                float (&s)[Grid::S], float* wbuf, uint32_t* list)
{
    const unsigned m = __ballot_sync(0xffffffffu, need);
    const uint32_t lane = threadIdx.x & 31u;
    const int cnt = __popc(m);
    const int rk = __popc(m & ((1u << lane) - 1u));
    if (need) list[rk] = lane;
    __syncwarp();
    const uint32_t j = lane & 7u;
    const int q4 = (int)(lane >> 3);                                 // this lane's rank within a round of four
    const uint32_t env_w = env - lane;                               // env id of lane 0
    const bool uni = (j == 4u) || (j == 5u);
    float4* const slot = reinterpret_cast<float4*>(wbuf + q4 * kGridResetRow + (int)j * 4);
    // one round: ranks r0 .. r0 + 3, one Philox block (4 raw values) per lane, stored at row (r0 - c0) + q4 of the buffer
    auto round = [&](int r0, int row0) {
        const int r = r0 + q4;
        const bool live = r < cnt;
        const uint32_t src = list[live ? r : 0];
        const uint4 w = rng_words(key, env_w + src, tick, STREAM_RESET, (epoch << 8) | j);
        float4 v;
        v.x = uni ? u_sym(w.x) : spec_normal_rep<REP>(tab8l, w.x);
        v.y = uni ? u_sym(w.y) : spec_normal_rep<REP>(tab8l, w.y);
        v.z = uni ? u_sym(w.z) : spec_normal_rep<REP>(tab8l, w.z);
        v.w = uni ? u_sym(w.w) : spec_normal_rep<REP>(tab8l, w.w);
        if (live) slot[row0 * (kGridResetRow / 4)] = v;
    };
#pragma unroll 1
    for (int c0 = 0; c0 < cnt; c0 += kGridResetRanks) {              // (8 or fewer resetting lanes: one pass)
        round(c0, 0);
        if (cnt - c0 > 4) round(c0 + 4, 4);                          // (uniform)
        __syncwarp();
        const int row = rk - c0;
        if (need && row >= 0 && row < kGridResetRanks) {
            float v[32];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float4 x = *reinterpret_cast<const float4*>(wbuf + row * kGridResetRow + q * 4);
                v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
            }
            Grid::reset_from_values(v, s);
        }
        __syncwarp();
    }
}

__device__ __forceinline__ float fmax3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }
__device__ __forceinline__ float fmin3(float a, float b, float c) { return fminf(fminf(a, b), c); }

// returns the number of steps committed (== n_steps unless the division guard failed)
template <bool EXTREMA>
__device__ __forceinline__ int grid_fast_steps(const Rng& key, uint32_t env, uint32_t tick0, uint32_t epoch, int n_steps, int max_steps,
                                               float (&s)[Grid::S], uint32_t& ep_st, uint32_t& ep_vi, double& ep_ret, float& rsum,
                                               RolloutAcc& acc, double& r_lo, double& r_hi, const float4* tab8l, float* wbuf, uint32_t* list)
{
    constexpr float kE90 = (float)((double)0.9f - 1.0), kE95 = (float)((double)0.95f - 1.0);
    constexpr float kE105 = (float)((double)1.05f - 1.0), kE110 = (float)((double)1.1f - 1.0);
    static_assert((double)kE90 == (double)0.9f - 1.0 && (double)kE95 == (double)0.95f - 1.0 &&
                  (double)kE105 == (double)1.05f - 1.0 && (double)kE110 == (double)1.1f - 1.0, "thresholds must be exact in binary32");
    int t_trunc = max_steps - (int)ep_st - 1;      // loop index of the step at which the running episode is truncated (base.py:191)
    unsigned int c_gen = 0u, vi = ep_vi;
    const double ret_sum0 = acc.ret_sum, ep_ret0 = ep_ret;
    const unsigned int con0_0 = acc.c_con[0], con1_0 = acc.c_con[1];
    int t = 0;
#pragma unroll 1
    for (; t < n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        // action_space.sample(); np.clip(gen + a, 0, 100) (:124); generation_limits on the pre-step state (:24-30)
        float gen[8], ap;
        bool gen_bad = false;
        {
            float a[8], a2[8];
            Grid::uniform_actions(key, env, tick, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                a2[i] = mul(a[i], a[i]);                                         // :173
                const float g = add(s[9 + i], a[i]);
                gen[i] = fmaxf(fminf(g, 100.0f), 0.0f);
                gen_bad = gen_bad || (gen[i] != g);
            }
            ap = mul(-5.0f, pairwise8(a2));
        }
        float sum_load;
        {
            const float ld[8] = {s[17], s[18], s[19], s[20], s[21], s[22], s[23], s[24]};
            sum_load = pairwise8(ld);
        }
        const float imb = sub(pairwise8(gen), sum_load);                          // :127-129
        const float x = add(-s[0], imb);                                          // mul(-1.0f, f) == -f
        const bool ok = fabsf(x) >= 0x1.0p-120f && fabsf(x) <= 0x1.0p+100f;
        // frequency_stability (:10-14), voltage_limits (:17-21) on the pre-step state
        const bool f_bad = !(fabsf(s[0]) < 0.5f);
        bool v_bad;
        {
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) e[i] = sub(s[1 + i], 1.0f);
            const float emax = fmax3(fmax3(e[0], e[1], e[2]), fmax3(e[3], e[4], e[5]), fmaxf(e[6], e[7]));
            const float emin = fmin3(fmin3(e[0], e[1], e[2]), fmin3(e[3], e[4], e[5]), fminf(e[6], e[7]));
            v_bad = emin < kE95 || emax > kE105;
        }
        // _dynamics (:112-153), in place
        {   // outside the proven domain of the constant division (a zero / denormal / huge / NaN imbalance): the IEEE division,
            // for that lane only -- no warp vote, no way out of the loop (+1 % over the vote + break)
            float q5 = NIG_CDIV_NG(x, 5.0f);
            if (__builtin_expect(!ok, 0)) q5 = __fdiv_rn(x, 5.0f);
            s[0] = add(s[0], mul(q5, 0.1f));                                      // :132-133
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) s[9 + i] = gen[i];
#pragma unroll
        for (int j = 0; j < 6; ++j) {                                             // V(8) sigma .005, load(8) sigma 1, flow(7) sigma 2
            float z[4];
            rng_normals4_rep<kTabRep>(key, tab8l, env, tick, STREAM_NOISE, (uint32_t)j, z);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = 4 * j + q;
                if (k < 8) s[1 + k] = add(s[1 + k], mul(0.005f, z[q]));           // :136-137
                else if (k < 16) s[9 + k] = fmaxf(add(s[9 + k], z[q]), 0.0f);     // :140-141 (mul(1.0f, z) == z)
                else if (k < 23) s[9 + k] = add(s[9 + k], mul(2.0f, z[q]));       // :144
            }
        }
        // _compute_reward (:155-177) on the new state; _is_done (:179-192)
        const float fr = mul(-100.0f, mul(s[0], s[0]));
        float vr;
        bool term;
        {
            float e[8], d2[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { e[i] = sub(s[1 + i], 1.0f); d2[i] = mul(e[i], e[i]); }
            vr = mul(-50.0f, pairwise8(d2));
            const float emax = fmax3(fmax3(e[0], e[1], e[2]), fmax3(e[3], e[4], e[5]), fmaxf(e[6], e[7]));
            const float emin = fmin3(fmin3(e[0], e[1], e[2]), fmin3(e[3], e[4], e[5]), fminf(e[6], e[7]));
            term = fabsf(s[0]) > 1.0f || emin < kE90 || emax > kE110;
        }
        double cg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) cg[i] = dmul(Grid::gen_cost(i), (double)gen[i]);   // :169
        const double ec = ddiv_const(-pairwise8d(cg), 1000.0, 1.0 / 1000.0);     // :170
        double r = dadd(dadd((double)add(fr, vr), ec), (double)ap);              // :175
        if (f_bad) r = r + (double)Grid::penalty(0);                              // base.py:179-183, in constraint order
        if (v_bad) r = r + (double)Grid::penalty(1);
        if (gen_bad) r = r + (double)Grid::penalty(2);
        const bool crit = f_bad || v_bad;
        if (crit) r = r - 1000.0;                                                 // base.py:195-198
        term = term || crit;
        rsum = add(rsum, (float)r);
        ep_ret = ep_ret + r;
        c_gen += gen_bad ? 1u : 0u;
        vi += gen_bad ? 1u : 0u;
        const bool fin = term || t >= t_trunc;
        if (__any_sync(0xffffffffu, fin)) {
            if (fin) {
                const unsigned long long len = (unsigned long long)(max_steps - (t_trunc - t));
                acc.c_ep += 1; acc.c_done += 1;
                acc.c_term += term ? 1u : 0u;
                acc.c_trunc += (t >= t_trunc) ? 1u : 0u;
                acc.c_succ += (ep_ret > 0.0) ? 1u : 0u;
                acc.c_crit += crit ? 1u : 0u;
                acc.c_con[0] += f_bad ? 1u : 0u;
                acc.c_con[1] += v_bad ? 1u : 0u;
                acc.len_sq += len * len;
                acc.ret_sum += ep_ret; acc.ret_sq += ep_ret * ep_ret;
                if constexpr (EXTREMA) { r_lo = ep_ret < r_lo ? ep_ret : r_lo; r_hi = ep_ret > r_hi ? ep_ret : r_hi; }
                ep_ret = 0.0; vi = 0u;
                t_trunc = t + max_steps;
            }
            grid_coop_reset<kTabRep>(key, tab8l, env, tick + 1u, epoch, fin, s, wbuf, list);
        }
    }
    // every step belongs to an episode: the lengths of the episodes finished here add up to the steps taken, plus the part of
    // the first episode that was there at entry, minus the part of the running one
    const uint32_t ep_st_exit = (uint32_t)(max_steps - (t_trunc - t + 1));
    acc.len_sum += (unsigned long long)((uint32_t)t + ep_st - ep_st_exit);
    ep_st = ep_st_exit;
    ep_vi = vi;
    acc.c_steps += (unsigned int)t;
    acc.c_con[2] += c_gen;
    acc.c_viol += c_gen + (acc.c_con[0] - con0_0) + (acc.c_con[1] - con1_0);
    // per-launch reward statistic: (returns of the episodes finished here) + (running return at exit - at entry)
    acc.rew_sum += (acc.ret_sum - ret_sum0) + (ep_ret - ep_ret0);
    return t;
}

// ---- the common tail of the fused rollout kernels: state / episode word / return accumulator back to HBM, per-env
// outputs, then the violation / episode statistics: warp REDUX + shuffle trees -> one global atomic per slot per block
// per-env outputs of a launch (reward sum, violation / finished-episode counts)
__device__ __forceinline__ void rollout_env_outputs(const RolloutArgs& p, int64_t i, float rsum, const RolloutAcc& acc)
{
    if (p.accumulate) {
        if (p.reward_sum) p.reward_sum[i] = add(p.reward_sum[i], rsum);
        if (p.viol_count) p.viol_count[i] += (int32_t)acc.c_viol;
        if (p.done_count) p.done_count[i] += (int32_t)acc.c_done;
    } else {
        if (p.reward_sum) p.reward_sum[i] = rsum;
        if (p.viol_count) p.viol_count[i] = (int32_t)acc.c_viol;
        if (p.done_count) p.done_count[i] = (int32_t)acc.c_done;
    }
}

template <class Env, bool EXTREMA>
__device__ __forceinline__ void rollout_stats_flush(const RolloutArgs& p, BlockStats& bs, double* sfl, unsigned long long* sext, RolloutAcc& acc,
                                                    typename Env::acc_t r_lo, typename Env::acc_t r_hi);

template <class Env, bool EXTREMA>
__device__ __forceinline__ void rollout_epilogue(const RolloutArgs& p, BlockStats& bs, double* sfl, unsigned long long* sext,
                                                 bool valid, int64_t i, const float (&s)[Env::S], uint32_t ep_st, uint32_t ep_vi, bool latched,
                                                 typename Env::acc_t ep_ret, float rsum, RolloutAcc& acc,
                                                 typename Env::acc_t r_lo, typename Env::acc_t r_hi)
{
    constexpr int S = Env::S;
    using acc_t = typename Env::acc_t;
    // fp32-reward envs (reactor): the reward statistic of this launch is the fp32 per-env sum (K <= a few hundred
    // terms) widened once, instead of an F2F + DADD per step on the XU / FP64 pipes
    if constexpr (sizeof(acc_t) == 4) acc.rew_sum = (double)rsum;
    if (valid) {
#pragma unroll
        for (int k = 0; k < S; ++k) p.state[k * p.pitch + i] = s[k];
        p.ep_word[i] = epw_make(ep_st, ep_vi, latched ? 1u : 0u);
        p.ep_return[i] = (double)ep_ret;
        rollout_env_outputs(p, i, rsum, acc);
    }
    rollout_stats_flush<Env, EXTREMA>(p, bs, sfl, sext, acc, r_lo, r_hi);
}

template <class Env, bool EXTREMA>
__device__ __forceinline__ void rollout_stats_flush(const RolloutArgs& p, BlockStats& bs, double* sfl, unsigned long long* sext, RolloutAcc& acc,
                                                    typename Env::acc_t r_lo, typename Env::acc_t r_hi)
{
    using acc_t = typename Env::acc_t;
    if (blockDim.x == 32) {
        // one-warp CTA (the env slices of a small population): no shared staging, no CTA barrier -- lane l ends up holding the warp
        // total of statistics slot l and ONE atomic-add instruction per warp sends the non-zero ones to the global block
        const int lane = threadIdx.x;
        unsigned long long mine = 0ull;
        double dmine = 0.0;
        auto put = [&](int slot, unsigned int v) {
            const unsigned int t = __reduce_add_sync(0xffffffffu, v);
            if (lane == slot) mine = t;
        };
        put(NIG_ST_STEPS, acc.c_steps);
        put(NIG_ST_VIOLATIONS, acc.c_viol);
        put(NIG_ST_CRITICAL, acc.c_crit);
#pragma unroll
        for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k)
            if (k < p.cons.n) put(NIG_ST_CON0 + k, acc.c_con[k]);
        if (__any_sync(0xffffffffu, acc.c_ep != 0u)) {
            put(NIG_ST_EPISODES, acc.c_ep);
            put(NIG_ST_TERMINATED, acc.c_term);
            put(NIG_ST_TRUNCATED, acc.c_trunc);
            put(NIG_ST_SUCCESSES, acc.c_succ);
            const unsigned long long ls = warp_sum(acc.len_sum), lq = warp_sum(acc.len_sq);
            const double rs_ = warp_sum(acc.ret_sum), rq = warp_sum(acc.ret_sq);
            if (lane == NIG_ST_EP_LEN_SUM) mine = ls;
            if (lane == NIG_ST_EP_LEN_SQ) mine = lq;
            if (lane == NIG_ST_F_RETURN_SUM) dmine = rs_;
            if (lane == NIG_ST_F_RETURN_SQ) dmine = rq;
            if constexpr (EXTREMA) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const acc_t a_ = __shfl_xor_sync(0xffffffffu, r_lo, o), b_ = __shfl_xor_sync(0xffffffffu, r_hi, o);
                    r_lo = a_ < r_lo ? a_ : r_lo; r_hi = b_ > r_hi ? b_ : r_hi;
                }
                if (lane == 0) {
                    atomicMax(&p.extrema[0], extremum_key(-(double)r_lo));
                    atomicMax(&p.extrema[1], extremum_key((double)r_hi));
                }
            }
        }
        {
            const double rw_ = warp_sum(acc.rew_sum);
            if (lane == NIG_ST_F_REWARD_SUM) dmine = rw_;
        }
        if (lane < 24) { if (mine != 0ull) atomicAdd(&p.stats[lane], mine); }
        else if (lane <= NIG_ST_F_REWARD_SUM && dmine != 0.0) atomicAdd(reinterpret_cast<double*>(p.stats) + lane, dmine);
        advance_device_tick(p.tick_dev, (uint32_t)p.n_steps);
        return;
    }
    bs.warp_add(NIG_ST_STEPS, acc.c_steps);
    bs.warp_add(NIG_ST_VIOLATIONS, acc.c_viol);
    bs.warp_add(NIG_ST_CRITICAL, acc.c_crit);
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k)
        if (k < p.cons.n) bs.warp_add(NIG_ST_CON0 + k, acc.c_con[k]);
    if (__any_sync(0xffffffffu, acc.c_ep != 0u)) {
        bs.warp_add(NIG_ST_EPISODES, acc.c_ep);
        bs.warp_add(NIG_ST_TERMINATED, acc.c_term);
        bs.warp_add(NIG_ST_TRUNCATED, acc.c_trunc);
        bs.warp_add(NIG_ST_SUCCESSES, acc.c_succ);
        const unsigned long long ls = warp_sum(acc.len_sum), lq = warp_sum(acc.len_sq);
        const double rs_ = warp_sum(acc.ret_sum), rq = warp_sum(acc.ret_sq);
        if constexpr (EXTREMA) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const acc_t a_ = __shfl_xor_sync(0xffffffffu, r_lo, o), b_ = __shfl_xor_sync(0xffffffffu, r_hi, o);
                r_lo = a_ < r_lo ? a_ : r_lo; r_hi = b_ > r_hi ? b_ : r_hi;
            }
        }
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&p.stats[NIG_ST_EP_LEN_SUM], ls);
            atomicAdd(&p.stats[NIG_ST_EP_LEN_SQ], lq);
            atomicAdd(&sfl[0], rs_);
            atomicAdd(&sfl[1], rq);
            if constexpr (EXTREMA) {
                atomicMax(&sext[0], extremum_key(-(double)r_lo));
                atomicMax(&sext[1], extremum_key((double)r_hi));
            }
        }
    }
    {
        const double rw_ = warp_sum(acc.rew_sum);
        if ((threadIdx.x & 31) == 0) atomicAdd(&sfl[2], rw_);
    }
    bs.flush(p.stats);
    if (threadIdx.x < 3 && sfl[threadIdx.x] != 0.0)
        atomicAdd(reinterpret_cast<double*>(p.stats) + NIG_ST_F_RETURN_SUM + threadIdx.x, sfl[threadIdx.x]);
    if constexpr (EXTREMA) {
        if (threadIdx.x < 2 && sext[threadIdx.x] != 0ull) atomicMax(&p.extrema[threadIdx.x], sext[threadIdx.x]);
    }
    advance_device_tick(p.tick_dev, (uint32_t)p.n_steps);
}

// TFNOISE: process noise teacher-forced from p.noise (POLICY_ACTIONS only). The LDG flavour of POLICY_ACTIONS
// prefetches the next step's actions / noise into registers one step ahead, so the L2 latency of the loads is
// hidden behind a whole step of arithmetic. Block size is a launch parameter (blockDim.x <= kThreads; TMA launches
// use kThreads).
// EXTREMA (NIG_ROLLOUT_EXTREMA): also track the smallest / largest finished-episode return. A template flag rather
// than a run-time one: two more live registers in the step loop moved ptxas' schedule of the throughput kernel by 2 %.
template <class Env, int CONS, int POLICY, bool TMA, bool TFNOISE, bool EXTREMA = false>
__global__ void __launch_bounds__(kThreads, Env::ROLLOUT_MIN_CTAS) rollout_kernel(const __grid_constant__ RolloutArgs p, const __grid_constant__ CUtensorMap amap)
{
    static_assert(!TFNOISE || POLICY == NIG_POLICY_ACTIONS, "teacher-forced noise comes with teacher-forced actions");
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    constexpr int kTmaChunk = tma_chunk(A);
    constexpr bool PREFETCH = (POLICY == NIG_POLICY_ACTIONS) && !TMA;
    using acc_t = typename Env::acc_t;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ double sfl[4];
    __shared__ unsigned long long sext[2];       // extremum keys of the episodes this CTA finished
    __shared__ float4 s_tab[Env::ROLLOUT_TAB_SMEM ? NIG_NORMAL_TAB_N : 1];   // this CTA's copy of the normal table (8 KB, read K * draws times)
    __shared__ alignas(8) uint64_t bars[2];
    __shared__ alignas(16) float coop_buf[CoopSmem<Env>::floats];
    extern __shared__ __align__(128) float act_smem[];     // [2][kTmaChunk][A][kThreads] when TMA
    BlockStats bs;
    if (threadIdx.x < 4) sfl[threadIdx.x] = 0.0;
    if constexpr (EXTREMA) { if (threadIdx.x < 2) sext[threadIdx.x] = 0ull; }
    if constexpr (Env::ROLLOUT_TAB_SMEM) normal_table_to_smem(s_tab);
    const Rng key(p.key, Env::ROLLOUT_TAB_SMEM ? s_tab : g_normal_tab);
    bs.init(sstat);                              // (synchronises the CTA)
    rollout_pdl_sync();

    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < p.n;
    const int64_t ic = valid ? i : 0;      // padding lanes shadow env 0 without side effects
    const uint32_t env = p.env0 + (uint32_t)ic;
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);

    constexpr uint32_t kChunkBytes = kTmaChunk * A * kThreads * sizeof(float);
    int n_chunks = 0;
    if constexpr (TMA) {
        n_chunks = (p.n_steps + kTmaChunk - 1) / kTmaChunk;
        if (threadIdx.x == 0) {
            mbar_init(&bars[0], 1);
            mbar_init(&bars[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int c = 0; c < 2 && c < n_chunks; ++c) {
                mbar_expect_tx(&bars[c], kChunkBytes);
                tma_load_3d(act_smem + (size_t)c * kTmaChunk * A * kThreads, &amap, (int)(blockIdx.x * kThreads), 0, c * kTmaChunk, &bars[c]);
            }
        }
    }

    float s[S];
#pragma unroll
    for (int k = 0; k < S; ++k) s[k] = p.state[k * p.pitch + ic];
    const uint32_t w0 = p.ep_word[ic];
    uint32_t ep_st = epw_step(w0), ep_vi = epw_viol(w0);      // unpacked across the K steps
    bool latched = (w0 >> 31) != 0u;
    acc_t ep_ret = (acc_t)p.ep_return[ic];
    typename Env::NoiseGen ng;

    float rsum = 0.0f;
    RolloutAcc acc;
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) acc.c_con[k] = 0;
    acc_t r_lo = (acc_t)INFINITY, r_hi = -(acc_t)INFINITY;     // extrema of this thread's finished-episode returns

    double pid_i[A], pid_e[A];             // POLICY_BASELINE: the PID agent's integral and previous error
    if constexpr (POLICY == NIG_POLICY_BASELINE) {
        const bool pid = p.pp.baseline.kind == NIG_BASELINE_PID && p.pid_state != nullptr;
#pragma unroll
        for (int k = 0; k < A; ++k) {
            pid_i[k] = pid ? p.pid_state[(int64_t)k * p.pitch + ic] : 0.0;
            pid_e[k] = pid ? p.pid_state[(int64_t)(A + k) * p.pitch + ic] : 0.0;
        }
    }
    float a_pf[A], nz_pf[NZA];             // PREFETCH: the values of step t, loaded during step t - 1
    if constexpr (PREFETCH) {
#pragma unroll
        for (int k = 0; k < A; ++k) a_pf[k] = __ldcs(p.actions + (int64_t)k * p.pitch + ic);
        if constexpr (TFNOISE) {
#pragma unroll
            for (int k = 0; k < NZA; ++k) nz_pf[k] = __ldcs(p.noise + (int64_t)k * p.pitch + ic);
        }
    }

    // ChemicalReactor-v0 under the benchmark's own configuration (uniform-random policy, the env's default constraints,
    // auto-reset): warps whose envs all satisfy the loop invariants of reactor_fast_steps run the specialised loop; whatever
    // it does not commit (nothing, normally) is left to the generic loop below
    int t_begin = 0;
    if constexpr (Env::KIND == NIG_ENV_CHEMICAL_REACTOR && (CONS == CONS_DEFAULT || cons_fast_extras(CONS) > 0) && !TFNOISE &&
                  ((POLICY == NIG_POLICY_UNIFORM && !TMA) || POLICY == NIG_POLICY_ACTIONS)) {
        constexpr int NX = cons_fast_extras(CONS);
        FastBounds fb;
        const bool fb_ok = fast_bounds_from<NX>(p.cons, fb);       // else (critical / other components): the generic loop
        const bool inv = fb_ok && valid && !latched && p.auto_reset != 0 && __float_as_uint(s[8]) == 0u &&
                         (__float_as_uint(s[9]) == 0u || __float_as_uint(s[9]) == 0x3f800000u) &&
                         s[0] >= 200.0f && s[0] <= 350.0f && s[1] <= 506625.0f && s[5] >= 1e-30f && s[5] <= 1e30f &&
                         ep_st < (uint32_t)p.max_steps;
        if (__all_sync(0xffffffffu, inv))
        {
            if constexpr (POLICY == NIG_POLICY_UNIFORM) {
                DrawInKernel src{key, env, tick0};
                t_begin = reactor_fast_steps<EXTREMA, DrawInKernel, NX>(src, key, env, tick0, epoch, p.n_steps, p.max_steps, s, ep_st, ep_vi, ep_ret, rsum,
                                                                        acc, r_lo, r_hi, fb);
            } else if constexpr (TMA) {
                DrawActionsTma src{key, env, tick0, act_smem, bars, &amap, n_chunks};
                t_begin = reactor_fast_steps<EXTREMA, DrawActionsTma, NX>(src, key, env, tick0, epoch, p.n_steps, p.max_steps, s, ep_st, ep_vi, ep_ret, rsum,
                                                                          acc, r_lo, r_hi, fb);
            } else {
                DrawActionsLdg src{key, env, tick0, p.actions, p.pitch, ic, p.n_steps, a_pf};
                t_begin = reactor_fast_steps<EXTREMA, DrawActionsLdg, NX>(src, key, env, tick0, epoch, p.n_steps, p.max_steps, s, ep_st, ep_vi, ep_ret, rsum,
                                                                          acc, r_lo, r_hi, fb);
                if (t_begin < p.n_steps) src.rewind(t_begin);
            }
        }
    }

#pragma unroll 1      // measured: unrolling by 2 (to drop the 12 state moves per step) is 4 % slower
    for (int t = t_begin; t < p.n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        float a[A], nz[NZA], ns[S];
        if constexpr (POLICY == NIG_POLICY_ACTIONS) {
            if constexpr (TMA) {
                const int c = t / kTmaChunk, tt = t % kTmaChunk, b = c & 1;
                if (tt == 0) mbar_wait(&bars[b], (uint32_t)((c >> 1) & 1));
                const float* src = act_smem + ((size_t)b * kTmaChunk + tt) * A * kThreads;
#pragma unroll
                for (int k = 0; k < A; ++k) a[k] = src[k * kThreads + threadIdx.x];
                if (tt == kTmaChunk - 1 || t == p.n_steps - 1) {
                    __syncthreads();                       // everyone finished reading buffer b
                    if (threadIdx.x == 0 && c + 2 < n_chunks) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        mbar_expect_tx(&bars[b], kChunkBytes);
                        tma_load_3d(act_smem + (size_t)b * kTmaChunk * A * kThreads, &amap, (int)(blockIdx.x * kThreads), 0, (c + 2) * kTmaChunk, &bars[b]);
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < A; ++k) a[k] = a_pf[k];
                const int tn = t + 1 < p.n_steps ? t + 1 : t;     // last step re-reads its own row (in bounds, unused)
#pragma unroll
                for (int k = 0; k < A; ++k) a_pf[k] = __ldcs(p.actions + ((int64_t)tn * A + k) * p.pitch + ic);
            }
        } else if constexpr (POLICY == NIG_POLICY_UNIFORM) {
            policy_uniform<Env>(key, env, tick, a);
        } else if constexpr (POLICY == NIG_POLICY_PCTRL) {
            policy_pctrl<Env>(key, p.pp, env, tick, s, a);
        } else if constexpr (POLICY == NIG_POLICY_BASELINE) {
            policy_baseline<Env>(key, p.pp.baseline, env, tick, s, a, pid_i, pid_e);
        } else {
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = 0.0f;
        }
        if constexpr (NZ > 0) {
            if constexpr (TFNOISE) {
                if constexpr (PREFETCH) {
#pragma unroll
                    for (int k = 0; k < NZA; ++k) nz[k] = nz_pf[k];
                    const int tn = t + 1 < p.n_steps ? t + 1 : t;
#pragma unroll
                    for (int k = 0; k < NZA; ++k) nz_pf[k] = __ldcs(p.noise + ((int64_t)tn * NZA + k) * p.pitch + ic);
                } else {
#pragma unroll
                    for (int k = 0; k < NZA; ++k) nz[k] = __ldcs(p.noise + ((int64_t)t * NZA + k) * p.pitch + ic);
                }
            } else ng.get(key, env, tick, nz);
        } else nz[0] = 0.0f;

        // this step-and-bookkeeping block is repeated statement for statement in rollout_step_generic (nig_mlp.cuh, the
        // kernels of the MLP policy and of nig_rollout_record) and, for the uniform policy, in rollout_generic_uniform_step: a change here goes there too
        // (moving it into a shared function changed ptxas' schedule of this kernel's reactor instantiations)
        const bool active = valid && !latched;
        uint32_t st2, vi2, f, vm;
        acc_t r;
        bool need_reset = false;
        step_core_unpacked<Env, CONS, POLICY != NIG_POLICY_UNIFORM, true>(p.cons, p.max_steps, s, a, nz, 0u, ep_st, ep_vi, st2, vi2, ns, r, f, vm);
        if (active) {
            const bool done = (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED)) != 0;
            rsum = add(rsum, (float)r);
            ep_ret = ep_ret + r;
            if constexpr (sizeof(acc_t) == 8) acc.rew_sum += r;      // fp32-reward envs: derived from rsum after the loop
            acc.c_steps += 1; acc.c_viol += __popc(vm);
            acc.c_crit += (f & NIG_F_CRITICAL) ? 1u : 0u;
#pragma unroll
            for (int k = 0; k < Env::NB; ++k) acc.c_con[k] += (vm >> k) & 1u;
            if constexpr (cons_fast_extras(CONS) > 0) {
#pragma unroll
                for (int k = Env::NB; k < Env::NB + cons_fast_extras(CONS); ++k) acc.c_con[k] += (vm >> k) & 1u;
            } else if constexpr (CONS != CONS_DEFAULT) {
#pragma unroll
                for (int k = Env::NB; k < NIG_MAX_CONSTRAINTS; ++k) acc.c_con[k] += (vm >> k) & 1u;
            }
            ep_st = st2; ep_vi = vi2;
            if (done) {
                const unsigned long long len = st2;
                acc.c_ep += 1; acc.c_done += 1;
                acc.c_term += (f & NIG_F_TERMINATED) ? 1u : 0u;
                acc.c_trunc += (f & NIG_F_TRUNCATED) ? 1u : 0u;
                acc.c_succ += (ep_ret > (acc_t)0) ? 1u : 0u;
                acc.len_sum += len; acc.len_sq += len * len;
                acc.ret_sum += (double)ep_ret; acc.ret_sq += (double)ep_ret * (double)ep_ret;
                if constexpr (EXTREMA) { r_lo = ep_ret < r_lo ? ep_ret : r_lo; r_hi = ep_ret > r_hi ? ep_ret : r_hi; }
                if (p.auto_reset) {
                    if constexpr (Env::COOP_BLOCKS > 0 || Env::COOP_FK) need_reset = true;
                    else Env::reset(key, env, tick + 1u, epoch, s);
                    ep_st = 0u; ep_vi = 0u; ep_ret = (acc_t)0;
                } else {
#pragma unroll
                    for (int k = 0; k < S; ++k) s[k] = ns[k];
                    latched = true;
                }
            } else {
#pragma unroll
                for (int k = 0; k < S; ++k) s[k] = ns[k];
            }
        }
        if constexpr (Env::COOP_BLOCKS > 0) coop_reset_blocks<Env>(key, env, tick + 1u, epoch, need_reset, s, coop_buf);
        else if constexpr (Env::COOP_FK) coop_reset_fk<Env>(key, env, tick + 1u, epoch, need_reset, s, coop_buf);
    }

    if (valid) {
        if constexpr (POLICY == NIG_POLICY_BASELINE) {
            if (p.pp.baseline.kind == NIG_BASELINE_PID && p.pid_state != nullptr) {
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    p.pid_state[(int64_t)k * p.pitch + i] = pid_i[k];
                    p.pid_state[(int64_t)(A + k) * p.pitch + i] = pid_e[k];
                }
            }
        }
    }
    rollout_epilogue<Env, EXTREMA>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
}

// one generic step of the uniform-random rollout with in-place draws: the loop body of rollout_kernel for POLICY_UNIFORM
// (envs without a block-cooperative reset), used by rollout_grid_kernel and rollout_reactor_pair_kernel where a warp cannot
// take the fast loop
template <class Env, int CONS, bool EXTREMA>
__device__ __forceinline__ void rollout_generic_uniform_step(const RolloutArgs& p, const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, bool valid,
                                                             float (&s)[Env::S], uint32_t& ep_st, uint32_t& ep_vi, bool& latched,
                                                             typename Env::acc_t& ep_ret, float& rsum, RolloutAcc& acc,
                                                             typename Env::acc_t& r_lo, typename Env::acc_t& r_hi)
{
    // (envs with a block-cooperative reset -- PowerGrid -- reset per lane here: this is their fallback path only)
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    using acc_t = typename Env::acc_t;
    float a[A], nz[NZA], ns[S];
    policy_uniform<Env>(key, env, tick, a);
    if constexpr (NZ > 0) { typename Env::NoiseGen ng; ng.get(key, env, tick, nz); } else nz[0] = 0.0f;
    const bool active = valid && !latched;
    uint32_t st2, vi2, f, vm;
    acc_t r;
    step_core_unpacked<Env, CONS, false, true>(p.cons, p.max_steps, s, a, nz, 0u, ep_st, ep_vi, st2, vi2, ns, r, f, vm);
    if (active) {
        const bool done = (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED)) != 0;
        rsum = add(rsum, (float)r);
        ep_ret = ep_ret + r;
        if constexpr (sizeof(acc_t) == 8) acc.rew_sum += r;
        acc.c_steps += 1; acc.c_viol += __popc(vm);
        acc.c_crit += (f & NIG_F_CRITICAL) ? 1u : 0u;
#pragma unroll
        for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k)
            if (k < Env::NB || CONS != CONS_DEFAULT) acc.c_con[k] += (vm >> k) & 1u;
        ep_st = st2; ep_vi = vi2;
        if (done) {
            const unsigned long long len = st2;
            acc.c_ep += 1; acc.c_done += 1;
            acc.c_term += (f & NIG_F_TERMINATED) ? 1u : 0u;
            acc.c_trunc += (f & NIG_F_TRUNCATED) ? 1u : 0u;
            acc.c_succ += (ep_ret > (acc_t)0) ? 1u : 0u;
            acc.len_sum += len; acc.len_sq += len * len;
            acc.ret_sum += (double)ep_ret; acc.ret_sq += (double)ep_ret * (double)ep_ret;
            if constexpr (EXTREMA) { r_lo = ep_ret < r_lo ? ep_ret : r_lo; r_hi = ep_ret > r_hi ? ep_ret : r_hi; }
            if (p.auto_reset) {
                Env::reset(key, env, tick + 1u, epoch, s);
                ep_st = 0u; ep_vi = 0u; ep_ret = (acc_t)0;
            } else {
#pragma unroll
                for (int k = 0; k < S; ++k) s[k] = ns[k];
                latched = true;
            }
        } else {
#pragma unroll
            for (int k = 0; k < S; ++k) s[k] = ns[k];
        }
    }
}

// ================================================================================================
// fused K-step rollout of PowerGrid-v0 under the benchmark's configuration (uniform-random policy, default constraints,
// auto-reset): grid_fast_steps with the 8 x replicated normal table. THREADS x CTAS resident threads per SM share
// CTAS x (65.7 KB table + 4.6 KB of reset buffer per warp) of dynamic shared memory. Warps whose envs do not all satisfy
// the loop invariants (and warps whose division guard failed) step through the generic path (global-memory table).
// ================================================================================================
template <int THREADS, int REP = kTabRep> __host__ __device__ constexpr size_t grid_rollout_smem()
{
    return (size_t)NIG_NORMAL_TAB_N * REP * sizeof(float4) + (size_t)(THREADS / 32) * (kGridResetRanks * kGridResetRow * sizeof(float) + 32 * sizeof(uint32_t));
}
template <bool EXTREMA, int THREADS, int MAXREG>
__global__ void __launch_bounds__(THREADS) __maxnreg__(MAXREG) rollout_grid_kernel(const __grid_constant__ RolloutArgs p)
{
    using Env = Grid;
    constexpr int S = Env::S;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ double sfl[4];
    __shared__ unsigned long long sext[2];
    extern __shared__ __align__(128) float4 dyn_smem4[];
    float4* tab8 = dyn_smem4;
    float* wbuf_all = reinterpret_cast<float*>(tab8 + NIG_NORMAL_TAB_N * kTabRep);
    uint32_t* list_all = reinterpret_cast<uint32_t*>(wbuf_all + (THREADS / 32) * kGridResetRanks * kGridResetRow);
    BlockStats bs;
    if (threadIdx.x < 4) sfl[threadIdx.x] = 0.0;
    if constexpr (EXTREMA) { if (threadIdx.x < 2) sext[threadIdx.x] = 0ull; }
    normal_table_to_smem_rep<kTabRep>(tab8);
    const Rng key(p.key, g_normal_tab);          // (the generic fallback and nothing else reads the table through `key`)
    bs.init(sstat);                              // (synchronises the CTA)
    rollout_pdl_sync();

    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < p.n;
    const int64_t ic = valid ? i : 0;
    const uint32_t env = p.env0 + (uint32_t)ic;
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);
    float s[S];
#pragma unroll
    for (int k = 0; k < S; ++k) s[k] = p.state[k * p.pitch + ic];
    const uint32_t w0 = p.ep_word[ic];
    uint32_t ep_st = epw_step(w0), ep_vi = epw_viol(w0);
    bool latched = (w0 >> 31) != 0u;
    double ep_ret = p.ep_return[ic];
    float rsum = 0.0f;
    double r_lo = INFINITY, r_hi = -INFINITY;
    RolloutAcc acc;
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) acc.c_con[k] = 0;

    int t_begin = 0;
    {
        const bool inv = valid && !latched && p.auto_reset != 0 && ep_st < (uint32_t)p.max_steps && grid_fast_invariants(s);
        if (__all_sync(0xffffffffu, inv)) {
            const int warp = threadIdx.x >> 5;
            t_begin = grid_fast_steps<EXTREMA>(key, env, tick0, epoch, p.n_steps, p.max_steps, s, ep_st, ep_vi, ep_ret, rsum, acc, r_lo, r_hi,
                                               tab8 + (threadIdx.x & 7), wbuf_all + warp * kGridResetRanks * kGridResetRow, list_all + warp * 32);
        }
    }
#pragma unroll 1
    for (int t = t_begin; t < p.n_steps; ++t)
        rollout_generic_uniform_step<Env, CONS_DEFAULT, EXTREMA>(p, key, env, tick0 + (uint32_t)t, epoch, valid, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
    rollout_epilogue<Env, EXTREMA>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
}

// ================================================================================================
// PowerGrid-v0 single step, dedicated persistent kernel (plain SoA step, default constraints): the lean step of the fused
// rollout above applied to ONE step per launch. gridDim = resident CTAs; each CTA copies the 8 x replicated normal table
// once and walks tiles of THREADS envs. The state is updated in place in registers; instead of entry invariants (there is no
// previous step to establish them) every step carries its own guards, all evaluated before anything is stored:
//   * bits(gen + a) <= bits(100.0f) for the eight generators: gen + a is in [+0, 100] (no generation_limits violation, the
//     np.clip is the identity, not NaN, not -0.0) -- so the lean path has no clamp and no third constraint at all;
//   * |f_dot numerator| in [2^-120, 2^100]: the fast division is exact; a NaN / inf frequency, generation or load ends up here;
//   * the voltage reward term is not NaN (a NaN voltage would be dropped by the FMNMX trees);
//   * 0 * a stays 0 for the raw actions (a NaN action would be hidden by the min / max clip; an infinite one only costs the
//     fallback).
// A warp in which any lane fails a guard (or is inactive: padding, done latch) reloads its inputs and takes step_core, the
// generic path. Same outputs, flags, counters and episode statistics as step_kernel<Grid, 1, CONS_DEFAULT, PLAIN>.
// The inputs of the NEXT tile (32 state rows, 8 action rows, the episode words, the episode returns: 42 contiguous row
// segments) are fetched by cp.async.bulk into one shared-memory stage while the current tile, already in registers, is
// stepped: with few warps per scheduler the loads of a tile (2 us under load) would otherwise serialise with its arithmetic
// (measured, 384-thread CTAs, 1M envs: 103 us per step without the stage -- no better than the one-tile kernel --, 90 us with
// it; a per-warp stage fed by 128-byte copies: 102 us).
// ================================================================================================
template <int THREADS> __host__ __device__ constexpr size_t grid_step_stage_bytes() { return (size_t)(Grid::S + Grid::A + 1) * THREADS * sizeof(float) + (size_t)THREADS * sizeof(double); }
template <int THREADS, int REP> __host__ __device__ constexpr size_t grid_step_smem() { return grid_rollout_smem<THREADS, REP>() + grid_step_stage_bytes<THREADS>(); }

template <int THREADS, int MAXREG, int REP>
__global__ void __launch_bounds__(THREADS) __maxnreg__(MAXREG) step_grid_kernel(const __grid_constant__ StepArgs p)
{
    using Env = Grid;
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ;
    constexpr float kE90 = (float)((double)0.9f - 1.0), kE95 = (float)((double)0.95f - 1.0);
    constexpr float kE105 = (float)((double)1.05f - 1.0), kE110 = (float)((double)1.1f - 1.0);
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ EpisodeStaging estage;
    __shared__ alignas(8) uint64_t full_bar;
    extern __shared__ __align__(128) float4 dyn_smem4[];
    float4* tab8 = dyn_smem4;
    float* wbuf = reinterpret_cast<float*>(tab8 + NIG_NORMAL_TAB_N * REP) + (threadIdx.x >> 5) * kGridResetRanks * kGridResetRow;
    uint32_t* list = reinterpret_cast<uint32_t*>(reinterpret_cast<float*>(tab8 + NIG_NORMAL_TAB_N * REP) + (THREADS / 32) * kGridResetRanks * kGridResetRow) + (threadIdx.x >> 5) * 32;
    const float4* tab8l = tab8 + (threadIdx.x & (REP - 1));
    float* stage = reinterpret_cast<float*>(reinterpret_cast<char*>(dyn_smem4) + grid_rollout_smem<THREADS, REP>());   // [S + A + 1][THREADS] floats
    double* stage_er = reinterpret_cast<double*>(stage + (S + A + 1) * THREADS);                                   // [THREADS]
    BlockStats bs;
    episode_staging_init(&estage);
    normal_table_to_smem_rep<REP>(tab8);
    if (threadIdx.x == 0) {
        mbar_init(&full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    bs.init(sstat);                              // (synchronises the CTA)
    const Rng key(p.key, g_normal_tab);          // (the generic fallback reads the global table)
    // programmatic dependent launch: everything above overlaps the tail of the previous step (see step_kernel)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch;
    const int64_t n_tiles = (p.pitch + THREADS - 1) / THREADS;
    // one elected thread issues the 42 row copies of a tile
    auto fetch = [&](int64_t tile) {
        const int64_t e0 = tile * THREADS;
        const uint32_t cnt = (uint32_t)((p.pitch - e0 < THREADS) ? (p.pitch - e0) : THREADS);        // (a multiple of 128)
        const bool with_er = p.ep_return != nullptr;
        mbar_expect_tx(&full_bar, cnt * (uint32_t)sizeof(float) * (S + A + 1) + (with_er ? cnt * (uint32_t)sizeof(double) : 0u));
        for (int k = 0; k < S; ++k) bulk_load(stage + k * THREADS, p.state + k * p.pitch + e0, cnt * (uint32_t)sizeof(float), &full_bar);
        for (int k = 0; k < A; ++k) bulk_load(stage + (S + k) * THREADS, p.actions + k * p.pitch + e0, cnt * (uint32_t)sizeof(float), &full_bar);
        bulk_load(stage + (S + A) * THREADS, p.ep_word + e0, cnt * (uint32_t)sizeof(float), &full_bar);
        if (with_er) bulk_load(stage_er, p.ep_return + e0, cnt * (uint32_t)sizeof(double), &full_bar);
    };
    if (threadIdx.x == 0 && (int64_t)blockIdx.x < n_tiles) fetch(blockIdx.x);
    uint32_t phase = 0u;

    unsigned int c_steps = 0, c_ep = 0, c_term = 0, c_trunc = 0, c_crit = 0, c_viol = 0, c_con0 = 0, c_con1 = 0, c_con2 = 0;
    StepEpisodeStats eps;
#pragma unroll 1
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t i = tile * THREADS + threadIdx.x;
        const bool in_pitch = i < p.pitch, valid = i < p.n;
        const int64_t ic = in_pitch ? i : 0;            // lanes past the pitch shadow another env and store nothing
        const uint32_t env = p.env0 + (uint32_t)i;
        float s[S], a_raw[A];
        mbar_wait(&full_bar, phase);
        phase ^= 1u;
        const int tl = in_pitch ? (int)threadIdx.x : 0;
#pragma unroll
        for (int k = 0; k < S; ++k) s[k] = stage[k * THREADS + tl];
#pragma unroll
        for (int k = 0; k < A; ++k) a_raw[k] = stage[(S + k) * THREADS + tl];
        uint32_t w = __float_as_uint(stage[(S + A) * THREADS + tl]);
        const bool active = valid && !(w >> 31);
        double er = 0.0;
        if (p.ep_return && active) er = stage_er[tl];
        __syncthreads();                                 // everyone has its tile in registers: the stage is free
        // (letting the last warp to arrive -- a shared counter instead of the barrier -- issue the refill: 92 instead of 87 us)
        if (threadIdx.x == 0 && tile + gridDim.x < n_tiles) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            fetch(tile + gridDim.x);
        }

        double r = 0.0;
        uint32_t f = NIG_F_INACTIVE, vm = 0u;
        bool lean = false;
        if (__all_sync(0xffffffffu, active)) {
            // ---- the lean step (see grid_fast_steps for the derivation) ----
            float a[A], poison = 0.0f, ap;
            bool ok = true;
            float gsum;
            {
                float a2[A], g[A];
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    poison = __fmaf_rn(0.0f, a_raw[k], poison);
                    a[k] = fmaxf(fminf(a_raw[k], 1.0f), -1.0f);                   // base.py:167 (finite or infinite a; NaN -> poison)
                    a2[k] = mul(a[k], a[k]);
                    g[k] = add(s[9 + k], a[k]);
                    ok = ok && __float_as_uint(g[k]) <= 0x42c80000u;
                }
                ap = mul(-5.0f, pairwise8(a2));
                gsum = pairwise8(g);
#pragma unroll
                for (int k = 0; k < A; ++k) s[9 + k] = g[k];                      // np.clip(gen + a, 0, 100) == gen + a here
            }
            float lsum;
            {
                const float ld[8] = {s[17], s[18], s[19], s[20], s[21], s[22], s[23], s[24]};
                lsum = pairwise8(ld);
            }
            const float x = add(-s[0], sub(gsum, lsum));
            ok = ok && fabsf(x) >= 0x1.0p-120f && fabsf(x) <= 0x1.0p+100f && poison == 0.0f;
            const bool f_bad = !(fabsf(s[0]) < 0.5f);
            bool v_bad;
            {
                float e[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) e[k] = sub(s[1 + k], 1.0f);
                const float emax = fmax3(fmax3(e[0], e[1], e[2]), fmax3(e[3], e[4], e[5]), fmaxf(e[6], e[7]));
                const float emin = fmin3(fmin3(e[0], e[1], e[2]), fmin3(e[3], e[4], e[5]), fminf(e[6], e[7]));
                v_bad = emin < kE95 || emax > kE105;
            }
            s[0] = add(s[0], mul(NIG_CDIV_NG(x, 5.0f), 0.1f));
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                float z[4];
                rng_normals4_rep<REP>(key, tab8l, env, tick0, STREAM_NOISE, (uint32_t)j, z);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int k = 4 * j + q;
                    if (k < 8) s[1 + k] = add(s[1 + k], mul(0.005f, z[q]));
                    else if (k < 16) s[9 + k] = fmaxf(add(s[9 + k], z[q]), 0.0f);
                    else if (k < 23) s[9 + k] = add(s[9 + k], mul(2.0f, z[q]));
                }
            }
            const float fr = mul(-100.0f, mul(s[0], s[0]));
            float vr;
            bool term;
            {
                float e[8], d2[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { e[k] = sub(s[1 + k], 1.0f); d2[k] = mul(e[k], e[k]); }
                vr = mul(-50.0f, pairwise8(d2));
                const float emax = fmax3(fmax3(e[0], e[1], e[2]), fmax3(e[3], e[4], e[5]), fmaxf(e[6], e[7]));
                const float emin = fmin3(fmin3(e[0], e[1], e[2]), fmin3(e[3], e[4], e[5]), fminf(e[6], e[7]));
                term = fabsf(s[0]) > 1.0f || emin < kE90 || emax > kE110;
            }
            ok = ok && vr == vr;
            double cg[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) cg[k] = dmul(Grid::gen_cost(k), (double)s[9 + k]);
            const double ec = ddiv_const(-pairwise8d(cg), 1000.0, 1.0 / 1000.0);
            r = dadd(dadd((double)add(fr, vr), ec), (double)ap);
            if (f_bad) r = r + (double)Grid::penalty(0);
            if (v_bad) r = r + (double)Grid::penalty(1);
            const bool crit = f_bad || v_bad;
            if (crit) r = r - 1000.0;
            lean = __all_sync(0xffffffffu, ok);
            if (lean) {
                const uint32_t step = epw_step(w) + 1u;
                vm = (f_bad ? 1u : 0u) | (v_bad ? 2u : 0u);
                f = (crit ? (uint32_t)NIG_F_CRITICAL : 0u) | ((term || crit) ? (uint32_t)NIG_F_TERMINATED : 0u) |
                    (step >= (uint32_t)p.max_steps ? (uint32_t)NIG_F_TRUNCATED : 0u);
                w = epw_make(step, epw_viol(w) + (uint32_t)__popc(vm), 0u);
            } else {                                     // (uniform) reload: the lean path has updated s in place
#pragma unroll
                for (int k = 0; k < S; ++k) s[k] = p.state[k * p.pitch + ic];
            }
        }
        if (!lean && active) {
            float nz[NZ], ns[S];
            Env::NoiseGen::get_single(key, env, tick0, nz);
            step_core<Env, CONS_DEFAULT>(p.cons, p.max_steps, s, a_raw, nz, 0u, w, ns, r, f, vm);
#pragma unroll
            for (int k = 0; k < S; ++k) s[k] = ns[k];
        }
        // (an inactive env keeps its state and episode word: r = 0, f = NIG_F_INACTIVE, vm = 0)
        const bool done = active && (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED));
        if (p.ep_return && active) {
            er = er + r;
            if (done) eps.episode(er, (unsigned long long)epw_step(w));
            p.ep_return[i] = (done && p.auto_reset) ? 0.0 : er;
        }
        bool need_reset = false;
        if (done) {
            if (p.auto_reset) { need_reset = true; w = 0u; f |= NIG_F_RESET; }
            else w |= 0x80000000u;
        }
        if (__any_sync(0xffffffffu, need_reset)) grid_coop_reset<REP>(key, tab8l, env, tick0 + 1u, epoch, need_reset, s, wbuf, list);
        if (in_pitch) {
#pragma unroll
            for (int k = 0; k < S; ++k) p.state[k * p.pitch + i] = s[k];
            p.ep_word[i] = w;
        }
        if (valid) {
            if (p.reward) p.reward[i] = (float)r;
            if (p.flags) p.flags[i] = (uint8_t)f;
            if (p.viol_mask) p.viol_mask[i] = (uint8_t)vm;
        }
        if (active) {
            c_steps += 1; c_viol += __popc(vm);
            c_crit += (f & NIG_F_CRITICAL) ? 1u : 0u;
            if (done) { c_ep += 1; c_term += (f & NIG_F_TERMINATED) ? 1u : 0u; c_trunc += (f & NIG_F_TRUNCATED) ? 1u : 0u; }
            c_con0 += vm & 1u; c_con1 += (vm >> 1) & 1u; c_con2 += (vm >> 2) & 1u;
        }
    }
    bs.warp_add(NIG_ST_STEPS, c_steps);
    if (__any_sync(0xffffffffu, (c_ep | c_viol | c_crit) != 0u)) {
        bs.warp_add(NIG_ST_EPISODES, c_ep);
        bs.warp_add(NIG_ST_TERMINATED, c_term);
        bs.warp_add(NIG_ST_TRUNCATED, c_trunc);
        bs.warp_add(NIG_ST_CRITICAL, c_crit);
        bs.warp_add(NIG_ST_VIOLATIONS, c_viol);
        bs.warp_add(NIG_ST_CON0, c_con0); bs.warp_add(NIG_ST_CON0 + 1, c_con1); bs.warp_add(NIG_ST_CON0 + 2, c_con2);
        if (p.ep_return && __any_sync(0xffffffffu, c_ep != 0u)) stage_episode_stats(bs, &estage, eps);
    }
    if (p.stats != nullptr) {
        unsigned long long* const stats_out = p.stats_shards ? p.stats_shards + (blockIdx.x % kStatsShards) * NIG_STATS_SLOTS : p.stats;
        bs.flush(stats_out);
        if (p.ep_return) flush_episode_staging(stats_out, &estage);
    }
    advance_device_tick(p.tick_dev, 1u);
}

// ================================================================================================
// fused K-step rollout, two envs per thread with packed f32x2 arithmetic (ChemicalReactor-v0, the benchmark's configuration)
// ================================================================================================
// Thread j owns envs 2j and 2j + 1 (adjacent: 64-bit loads / stores of the SoA rows) and runs reactor_fast_steps_v<F2>: the
// add / mul / fma instructions of the physics are issued once for both envs (FADD2 / FMUL2 / FFMA2), the per-lane rest twice.
// Warps whose 64 envs do not all satisfy the loop invariants step both envs through the generic path.
template <bool EXTREMA>
__global__ void __launch_bounds__(kThreads, 1) rollout_reactor_pair_kernel(const __grid_constant__ RolloutArgs p)
{
    using Env = Reactor;
    constexpr int S = Env::S;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ double sfl[4];
    __shared__ unsigned long long sext[2];
    __shared__ float4 s_tab[NIG_NORMAL_TAB_N];
    BlockStats bs;
    if (threadIdx.x < 4) sfl[threadIdx.x] = 0.0;
    if constexpr (EXTREMA) { if (threadIdx.x < 2) sext[threadIdx.x] = 0ull; }
    normal_table_to_smem(s_tab);
    const Rng key(p.key, s_tab);
    bs.init(sstat);                              // (synchronises the CTA)
    rollout_pdl_sync();

    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i0 = 2 * j;
    const bool valid[2] = {i0 < p.n, i0 + 1 < p.n};
    const int64_t ib = valid[0] ? i0 : 0;           // (pitch is even: a valid first env has an in-bounds partner row slot)
    const uint32_t env[2] = {p.env0 + (uint32_t)ib, p.env0 + (uint32_t)ib + 1u};
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);

    float s[2][S];
#pragma unroll
    for (int k = 0; k < S; ++k) {
        const float2 v = *reinterpret_cast<const float2*>(p.state + k * p.pitch + ib);
        s[0][k] = v.x; s[1][k] = v.y;
    }
    const uint2 w0 = *reinterpret_cast<const uint2*>(p.ep_word + ib);
    uint32_t ep_st[2] = {epw_step(w0.x), epw_step(w0.y)}, ep_vi[2] = {epw_viol(w0.x), epw_viol(w0.y)};
    bool latched[2] = {(w0.x >> 31) != 0u, (w0.y >> 31) != 0u};
    const double2 er0 = *reinterpret_cast<const double2*>(p.ep_return + ib);
    float ep_ret[2] = {(float)er0.x, (float)er0.y}, rsum[2] = {0.0f, 0.0f};
    float r_lo = INFINITY, r_hi = -INFINITY;
    RolloutAcc acc[2];
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) acc[e].c_con[k] = 0;

    bool inv = p.auto_reset != 0;
#pragma unroll
    for (int e = 0; e < 2; ++e)
        inv = inv && valid[e] && !latched[e] && __float_as_uint(s[e][8]) == 0u &&
              (__float_as_uint(s[e][9]) == 0u || __float_as_uint(s[e][9]) == 0x3f800000u) &&
              s[e][0] >= 200.0f && s[e][0] <= 350.0f && s[e][1] <= 506625.0f && s[e][5] >= 1e-30f && s[e][5] <= 1e30f &&
              ep_st[e] < (uint32_t)p.max_steps;
    int t_begin = 0;
    if (__all_sync(0xffffffffu, inv)) {
        DrawInKernel2 src{key, {env[0], env[1]}, tick0};
        t_begin = reactor_fast_steps_v<F2, EXTREMA>(src, key, env, tick0, epoch, p.n_steps, p.max_steps, s, ep_st, ep_vi, ep_ret, rsum, acc, r_lo, r_hi);
    }
#pragma unroll 1
    for (int t = t_begin; t < p.n_steps; ++t) {
#pragma unroll
        for (int e = 0; e < 2; ++e)
            rollout_generic_uniform_step<Env, CONS_DEFAULT, EXTREMA>(p, key, env[e], tick0 + (uint32_t)t, epoch, valid[e], s[e], ep_st[e], ep_vi[e],
                                                                     latched[e], ep_ret[e], rsum[e], acc[e], r_lo, r_hi);
    }
    if (valid[0]) {                                  // rows are written pairwise; an invalid partner (odd n) keeps what it loaded
#pragma unroll
        for (int k = 0; k < S; ++k) *reinterpret_cast<float2*>(p.state + k * p.pitch + i0) = make_float2(s[0][k], s[1][k]);
        *reinterpret_cast<uint2*>(p.ep_word + i0) = make_uint2(epw_make(ep_st[0], ep_vi[0], latched[0] ? 1u : 0u),
                                                               valid[1] ? epw_make(ep_st[1], ep_vi[1], latched[1] ? 1u : 0u) : w0.y);
        *reinterpret_cast<double2*>(p.ep_return + i0) = make_double2((double)ep_ret[0], valid[1] ? (double)ep_ret[1] : er0.y);
        rollout_env_outputs(p, i0, rsum[0], acc[0]);
        if (valid[1]) rollout_env_outputs(p, i0 + 1, rsum[1], acc[1]);
    }
    // one statistics flush for both envs of the thread
    acc[0].rew_sum = (double)rsum[0] + (double)rsum[1];
    acc[0].c_steps += acc[1].c_steps; acc[0].c_ep += acc[1].c_ep; acc[0].c_term += acc[1].c_term; acc[0].c_trunc += acc[1].c_trunc;
    acc[0].c_crit += acc[1].c_crit; acc[0].c_viol += acc[1].c_viol; acc[0].c_succ += acc[1].c_succ; acc[0].c_done += acc[1].c_done;
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) acc[0].c_con[k] += acc[1].c_con[k];
    acc[0].len_sum += acc[1].len_sum; acc[0].len_sq += acc[1].len_sq; acc[0].ret_sum += acc[1].ret_sum; acc[0].ret_sq += acc[1].ret_sq;
    rollout_stats_flush<Env, EXTREMA>(p, bs, sfl, sext, acc[0], r_lo, r_hi);
}

// ================================================================================================
// dataset writer (get_dataset: chemical_reactor.py:324-420, power_grid.py:194-249, robot_assembly.py:246-308)
// ================================================================================================
// One thread = one episode (an independent env with global id env0 + e): reset, then up to n_steps
// policy/step iterations, stopping at done. WRITE=false only records the episode length (pass 1); after an
// exclusive scan of the lengths WRITE=true replays the identical counter-based random streams and stores every
// transition at row offsets[e] + t, so the arrays come out episode-contiguous like the reference's lists.
struct DatasetArgs {
    int64_t n_episodes;
    int32_t n_steps, max_steps, policy, terminals_include_truncation;
    uint32_t env0, epoch;
    RngKey key;
    nig_policy_params_t pp;
    ConsParams cons;
    int64_t* lengths;          // pass 1 out
    const int64_t* offsets;    // pass 2 in (exclusive scan of lengths)
    float* observations; float* actions; float* rewards; uint8_t* terminals; uint8_t* timeouts;
    float* next_observations; uint8_t* safety;
};

template <class Env, int CONS, bool WRITE>
__global__ void __launch_bounds__(kThreads) dataset_kernel(const __grid_constant__ DatasetArgs p)
{
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    using acc_t = typename Env::acc_t;
    __shared__ float4 s_tab[NIG_NORMAL_TAB_N];
    normal_table_to_smem(s_tab);
    __syncthreads();
    const Rng key(p.key, s_tab);
    const int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (e >= p.n_episodes) return;
    const uint32_t env = p.env0 + (uint32_t)e;
    float s[S];
    Env::reset(key, env, 0u, p.epoch, s);
    typename Env::NoiseGen ng;
    uint32_t w = 0u;
    int64_t row = WRITE ? p.offsets[e] : 0;
    int32_t len = 0;
    for (int t = 0; t < p.n_steps; ++t) {
        float a[A], nz[NZA], ns[S];
        if (p.policy == NIG_POLICY_UNIFORM) policy_uniform<Env>(key, env, (uint32_t)t, a);
        else if (p.policy == NIG_POLICY_PCTRL) policy_pctrl<Env>(key, p.pp, env, (uint32_t)t, s, a);
        else {
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = 0.0f;
        }
        if (p.pp.store_clip > 0.0f) {        // np.clip(action, -c, c) BEFORE env.step and before storing
#pragma unroll
            for (int k = 0; k < A; ++k) {
                float v = a[k];
                v = v < -p.pp.store_clip ? -p.pp.store_clip : v;
                v = v > p.pp.store_clip ? p.pp.store_clip : v;
                a[k] = v;
            }
        }
        if (NZ > 0) ng.get(key, env, (uint32_t)t, nz); else nz[0] = 0.0f;
        acc_t r; uint32_t f, vm;
        step_core<Env, CONS>(p.cons, p.max_steps, s, a, nz, 0u, w, ns, r, f, vm);
        const bool done = (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED)) != 0;
        if constexpr (WRITE) {
#pragma unroll
            for (int k = 0; k < S; ++k) p.observations[row * S + k] = s[k];
#pragma unroll
            for (int k = 0; k < A; ++k) p.actions[row * A + k] = a[k];
            p.rewards[row] = (float)r;
            p.terminals[row] = (uint8_t)(p.terminals_include_truncation ? done : ((f & NIG_F_TERMINATED) != 0));
            if (p.timeouts) p.timeouts[row] = 0;      // chemical_reactor.py:419
            if (p.next_observations) {
#pragma unroll
                for (int k = 0; k < S; ++k) p.next_observations[row * S + k] = ns[k];
            }
            if (p.safety) p.safety[row] = (uint8_t)vm;
            row += 1;
        }
        len = t + 1;
        if (done) break;
#pragma unroll
        for (int k = 0; k < S; ++k) s[k] = ns[k];
    }
    if constexpr (!WRITE) p.lengths[e] = len;
}

// exclusive scan of n int64 lengths (one 1024-thread block; n is a few thousand .. a few million episodes)
static __global__ void __launch_bounds__(1024) scan_lengths_kernel(const int64_t* __restrict__ len, int64_t* __restrict__ off, int64_t n, int64_t* total)
{
    __shared__ long long part[1024];
    const int t = threadIdx.x;
    const int64_t chunk = (n + 1023) / 1024;
    const int64_t lo = (int64_t)t * chunk, hi = lo + chunk < n ? lo + chunk : n;
    long long sum = 0;
    for (int64_t i = lo; i < hi; ++i) sum += len[i];
    part[t] = sum;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const long long v = t >= d ? part[t - d] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    long long run = part[t] - sum;      // exclusive prefix of this thread's chunk
    for (int64_t i = lo; i < hi; ++i) { off[i] = run; run += len[i]; }
    if (t == 1023) *total = part[1023];
}

// ---- self-test of the guarded fast divisions (nig_math.cuh) against the IEEE division -------------------------
// mode 0: x, y = raw Philox words (all exponents, ~22 % inside the vdiv guard); mode 1: the physics regime
// (y ~ 300, x = y * (1 + small)); mode 2: x = raw word divided by each constant the kernels use.
static __global__ void __launch_bounds__(256) selftest_division_kernel(RngKey key, int iters, unsigned long long* out)
{
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long bad = 0, acc = 0;
    for (int it = 0; it < iters; ++it) {
        const uint4 w = philox4x32<10>(tid, (uint32_t)it, 7u, 0u, key.k0, key.k1);
        {   // mode 0
            DivFast d;
            const float x = __uint_as_float(w.x), y = __uint_as_float(w.y);
            const float q = d.vdiv(x, y);
            if (d.ok()) { acc++; bad += __float_as_uint(q) != __float_as_uint(__fdiv_rn(x, y)); }
        }
        {   // mode 1
            DivFast d;
            const float y = __fadd_rn(250.0f, __fmul_rn(150.0f, u_open(w.z)));
            const float x = __fmul_rn(y, __fadd_rn(1.0f, __fmul_rn(0.01f, u_sym(w.w))));
            const float q = d.vdiv(x, y);
            if (d.ok()) { acc++; bad += __float_as_uint(q) != __float_as_uint(__fdiv_rn(x, y)); }
        }
        {   // mode 2
            const float x = __uint_as_float(w.x ^ w.z);
            const float cs[6] = {5.0f, 20.0f, 50.0f, 100.0f, 1000.0f, 418000.0f};
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                DivFast d;
                const float q = d(x, cs[k], 1.0f / cs[k]);
                if (d.ok()) { acc++; bad += __float_as_uint(q) != __float_as_uint(__fdiv_rn(x, cs[k])); }
            }
        }
        {   // mode 3: the binary64 constant division of PowerGrid's cost term (ddiv_const), operands across +-2^+-40
            const double m = (double)(int)w.y + (double)w.z * 0x1.0p-32;
            const double x = ldexp(m, (int)(w.w % 81u) - 40);
            const double q = ddiv_const(x, 1000.0, 1.0 / 1000.0);
            acc++; bad += __double_as_longlong(q) != __double_as_longlong(__ddiv_rn(x, 1000.0));
        }
    }
    atomicAdd(&out[0], bad);
    atomicAdd(&out[1], acc);
}

// checksums of spec_normal over the words first + k * stride, k < count (the oracle computes the same two sums on the CPU)
static __global__ void __launch_bounds__(256) selftest_normal_kernel(uint32_t first, uint32_t stride, unsigned long long count, unsigned long long* out)
{
    unsigned long long s0 = 0, s1 = 0;
    for (unsigned long long k = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t w = first + (uint32_t)k * stride;
        const unsigned long long bits = __float_as_uint(spec_normal(g_normal_tab, w));
        s0 += bits;
        s1 += bits * (k + 1ull);
    }
    atomicAdd(&out[0], s0);
    atomicAdd(&out[1], s1);
}

// ---- teacher-forced policy replay: the in-kernel policies on caller-supplied states and random inputs ------------------
// One thread = one env walking T steps (the PID controller's integral / previous error persist across the steps like the
// agent object's, benchmarks/baseline_agents.py:58-60). Layouts: states [T][n][S], coin [T][n], z / u [T][n][8],
// actions out [T][n][A] (the value the dataset stores: clipped to +-store_clip when that is positive).
struct PolicyTestArgs {
    int32_t policy, T;
    int64_t n;
    nig_policy_params_t pp;
    const float* states; const float* coin; const float* z; const float* u;
    float* actions;
};
template <class Env>
__global__ void __launch_bounds__(kThreads) selftest_policy_kernel(const __grid_constant__ PolicyTestArgs p)
{
    constexpr int S = Env::S, A = Env::A;
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= p.n) return;
    const Rng key(RngKey{0u, 0u}, g_normal_tab);
    double pid_i[A], pid_e[A];
#pragma unroll
    for (int k = 0; k < A; ++k) { pid_i[k] = 0.0; pid_e[k] = 0.0; }
    for (int t = 0; t < p.T; ++t) {
        const int64_t row = (int64_t)t * p.n + i;
        float s[S], a[A], z[8], u[8];
#pragma unroll
        for (int k = 0; k < S; ++k) s[k] = p.states[row * S + k];
#pragma unroll
        for (int k = 0; k < 8; ++k) { z[k] = p.z ? p.z[row * 8 + k] : 0.0f; u[k] = p.u ? p.u[row * 8 + k] : 0.0f; }
        if (p.policy == NIG_POLICY_PCTRL) policy_pctrl_forced<Env>(p.pp, s, p.coin ? p.coin[row] : 0.5f, z, u, a);
        else policy_baseline<Env>(key, p.pp.baseline, (uint32_t)i, (uint32_t)t, s, a, pid_i, pid_e);
        if (p.pp.store_clip > 0.0f) {
#pragma unroll
            for (int k = 0; k < A; ++k) {
                float v = a[k];
                v = v < -p.pp.store_clip ? -p.pp.store_clip : v;
                v = v > p.pp.store_clip ? p.pp.store_clip : v;
                a[k] = v;
            }
        }
#pragma unroll
        for (int k = 0; k < A; ++k) p.actions[row * A + k] = a[k];
    }
}

// ---- measured-peak probe: independent unfused FADD/FMUL chains (what the physics is made of) ------
static __global__ void __launch_bounds__(256) fp32_probe_kernel(float* out, int iters)
{
    float x[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = 1.0f + 1e-3f * (float)(threadIdx.x + k);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { x[k] = __fmul_rn(x[k], 1.0000001f); x[k] = __fadd_rn(x[k], 1e-7f); }
    }
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc += x[k];
    if (acc == 123.456f) out[0] = acc;
}

} // namespace nig
