// nig_mlp.cuh -- device code shared by the fused rollouts of nig_rollout_mlp.cu (NIG_POLICY_MLP) and
// nig_rollout_record.cu (nig_rollout_record): the tcgen05 MLP forward pass, rollout_kernel's generic step as a function, and
// the launch-side sizing of the MLP kernels' dynamic shared memory.
#pragma once
#include <mutex>
#include <vector>
#include <cuda_bf16.h>
#include "nig_launch.h"

namespace nig {

// ---- tcgen05 / UMMA helpers --------------------------------------------------------------------------------------------
// shared-memory matrix descriptor (sm_100): start >> 4 [0,14), LBO >> 4 [16,30), SBO >> 4 [32,46), version 1 [46,48),
// base offset 0, layout SWIZZLE_NONE (0) [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// instruction descriptor of kind::f16: fp32 accumulator [4,6) = 1, A = B = bf16 [7,10) / [10,13) = 1, both K-major,
// N >> 3 at [17,23), M >> 4 at [24,29); M = 128
__device__ __forceinline__ uint32_t umma_idesc_bf16(int n)
{
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accumulate)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(accumulate));
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] = __uint_as_float(r[q]);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi)
{
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);        // round to nearest even, NaN stays NaN
    return *reinterpret_cast<const uint32_t*>(&h);
}
// generic-proxy stores to shared memory -> visible to the MMA (async proxy), then the CTA barrier
__device__ __forceinline__ void mlp_publish_smem()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
}

// Per-CTA state of the network: shared-memory copy of the blob, tensor-memory accumulators, the MMA-completion mbarrier.
struct MlpCta {
    uint8_t* sm;
    uint32_t sm_addr, tmem, lane_off, phase;
    uint64_t* bar;               // [0] weights landed, [1] MMA done
    MlpLayout L;
};

// prologue of both kernels: weights -> shared memory (cp.async.bulk), tensor memory allocated by warp 0. The blob is
// written only by nig_set_mlp_policy, which synchronises the device first, so this may run before griddepcontrol.wait;
// a CTA whose columns are still held by a CTA of the previous launch (programmatic dependent launch) blocks in
// tcgen05.alloc until that CTA deallocates -- those CTAs are all resident and do not wait for this launch.
__device__ __forceinline__ void mlp_setup(MlpCta& c, const MlpParams& m, int S, uint8_t* sm, uint64_t* bars, uint32_t* tmem_slot)
{
    c.sm = sm; c.sm_addr = smem_u32(sm); c.bar = bars; c.phase = 0u;
    c.L = mlp_layout(S, m);
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bars[0], m.blob_bytes);
        for (uint32_t off = 0; off < m.blob_bytes; off += 32768u) {
            const uint32_t len = m.blob_bytes - off < 32768u ? m.blob_bytes - off : 32768u;
            bulk_load(sm + off, static_cast<const uint8_t*>(m.blob) + off, len, &bars[0]);
        }
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(c.L.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    c.tmem = *tmem_slot;
    c.lane_off = (uint32_t)(threadIdx.x & ~31u) << 16;          // warp w reads TMEM lanes 32w .. 32w + 31
    mbar_wait(&bars[0], 0u);
}

__device__ __forceinline__ void mlp_teardown(const MlpCta& c)
{
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(c.tmem), "r"(c.L.tmem_cols) : "memory");
    }
}

// issue (one thread) the MMAs of one K range of a layer: D[128][n] (+)= X[128][k0 .. k0 + kc) . W[n][k0 .. k0 + kc)^T, with X a
// 128-row tile in shared memory and W the layer's [n][kw] weights; then wait for them on every thread
__device__ __forceinline__ void mlp_mma(MlpCta& c, uint32_t d_col, uint32_t x_off, uint32_t w_off, int n, int k0, int kc, bool acc0)
{
    if (threadIdx.x == 0) {
        tc_fence_after();
        const uint32_t idesc = umma_idesc_bf16(n);
#pragma unroll 1
        for (int k = 0; k < kc; k += 16) {
            const uint64_t a = umma_desc(c.sm_addr + x_off + (uint32_t)(k / 8) * 2048u, 2048u, 128u);
            const uint64_t b = umma_desc(c.sm_addr + w_off + (uint32_t)((k0 + k) / 8) * (uint32_t)(n * 16), (uint32_t)(n * 16), 128u);
            umma_bf16(c.tmem + d_col, a, b, idesc, (acc0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&c.bar[1]);
    }
    mbar_wait(&c.bar[1], c.phase);
    c.phase ^= 1u;
    tc_fence_after();
}

// one hidden-to-next layer: activation rows of the k-wide accumulator at src_col (bias, ReLU, bf16) -> staging tile, MMA
// with the [n][k] weights at w_off into the accumulator at dst_col; at most 128 input columns per pass
__device__ __forceinline__ void mlp_hidden_layer(MlpCta& c, uint32_t src_col, int k, uint32_t b_off, uint32_t dst_col, uint32_t w_off, int n)
{
    const float* bias = reinterpret_cast<const float*>(c.sm + b_off);
    uint8_t* stage = c.sm + c.L.stage + threadIdx.x * 16u;
#pragma unroll 1
    for (int c0 = 0; c0 < k; c0 += c.L.kc) {
        const int kc = k - c0 < c.L.kc ? k - c0 : c.L.kc;
#pragma unroll 1
        for (int j = 0; j < kc; j += 16) {
            float v[16];
            tmem_ld16(c.tmem + c.lane_off + src_col + (uint32_t)(c0 + j), v);
            uint32_t w[8];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                float x = __fadd_rn(v[q], bias[c0 + j + q]);
                v[q] = x < 0.0f ? 0.0f : x;                         // ReLU; NaN stays NaN like torch.relu
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) w[q] = pack_bf16x2(v[2 * q], v[2 * q + 1]);
            *reinterpret_cast<uint4*>(stage + (uint32_t)(j / 8) * 2048u) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(stage + (uint32_t)(j / 8 + 1) * 2048u) = make_uint4(w[4], w[5], w[6], w[7]);
        }
        mlp_publish_smem();
        mlp_mma(c, dst_col, c.L.stage, w_off, n, c0, kc, c0 > 0);
    }
}

// the forward pass of this thread's env row: observation s -> action a (before the env's clip). Convergent: every thread
// of the CTA calls it the same number of times.
template <int S, int A>
__device__ __forceinline__ void mlp_forward(MlpCta& c, const MlpParams& m, const float (&s)[S], float (&a)[A])
{
    constexpr int SP = mlp_in_pad(S);
    const MlpLayout& L = c.L;
    const float* mean = reinterpret_cast<const float*>(c.sm + L.mean);
    const float* istd = reinterpret_cast<const float*>(c.sm + L.istd);
    uint32_t w[SP / 2];
#pragma unroll
    for (int k = 0; k < SP / 2; ++k) {
        const float x0 = 2 * k < S ? __fmul_rn(__fsub_rn(s[2 * k], mean[2 * k]), istd[2 * k]) : 0.0f;
        const float x1 = 2 * k + 1 < S ? __fmul_rn(__fsub_rn(s[2 * k + 1], mean[2 * k + 1]), istd[2 * k + 1]) : 0.0f;
        w[k] = pack_bf16x2(x0, x1);
    }
    uint8_t* x0 = c.sm + L.x0 + threadIdx.x * 16u;
#pragma unroll
    for (int q = 0; q < SP / 8; ++q)
        *reinterpret_cast<uint4*>(x0 + q * 2048) = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
    mlp_publish_smem();
    // accumulators: layer 1 -> columns [0, h1), layer 2 -> [h1, h1 + h2) ... alternating, the output layer -> the free one
    const uint32_t acc_a = 0u, acc_b = (uint32_t)(L.tmem_cols / 2);
    mlp_mma(c, acc_a, L.x0, L.w1, m.h1, 0, SP, false);
    uint32_t src = acc_a, dst = acc_b;
    int width = m.h1;
    if (m.layers == 2) {
        mlp_hidden_layer(c, acc_a, m.h1, L.b1, acc_b, L.w2, m.h2);
        src = acc_b; dst = acc_a; width = m.h2;
    }
    mlp_hidden_layer(c, src, width, m.layers == 2 ? L.b2 : L.b1, dst, L.w3, kMlpOut);
    float v[16];
    tmem_ld16(c.tmem + c.lane_off + dst, v);
    const float* b3 = reinterpret_cast<const float*>(c.sm + L.b3);
#pragma unroll
    for (int k = 0; k < A; ++k) {
        const float y = __fadd_rn(v[k], b3[k]);
        a[k] = m.out_tanh ? tanhf(y) : y;
    }
}

// one step of rollout_kernel's generic loop after the policy: step_core, the per-thread statistics, the episode bookkeeping
// and the (cooperative) auto-reset, statement for statement; must be called convergently (coop resets). `extrema` is the
// run-time switch of nig_track_extrema. rollout_kernel keeps its inline copy: calling this function from it changed ptxas'
// instruction schedule of 24 of its reactor instantiations (the benchmark's among them), and existing kernels stay as measured.
// REC (nig_rollout_record's kernels; off for the MLP rollout, whose code it leaves as it was) also hands out in *rec what
// nig_step writes for the env in this step.
template <class Env>
struct StepRecord {
    float ns[Env::S];          // s' of the transition, before the auto-reset; an inactive env's unchanged state
    float r;                   // reward; 0 for an inactive env
    uint32_t f, vm;            // NIG_F_* flags with NIG_F_RESET / NIG_F_INACTIVE as nig_step sets them; violation mask (0 inactive)
};
template <class Env, int CONS, bool CLIP, bool REC = false>
__device__ __forceinline__ void rollout_step_generic(const RolloutArgs& p, const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch,
                                                     bool valid, bool extrema, const float (&a)[Env::A],
                                                     const float (&nz)[Env::NZ > 0 ? Env::NZ : 1], float (&s)[Env::S],
                                                     uint32_t& ep_st, uint32_t& ep_vi, bool& latched, typename Env::acc_t& ep_ret,
                                                     float& rsum, RolloutAcc& acc, typename Env::acc_t& r_lo, typename Env::acc_t& r_hi,
                                                     float* coop_buf, StepRecord<Env>* rec = nullptr)
{
    constexpr int S = Env::S;
    using acc_t = typename Env::acc_t;
    float ns[S];
    const bool active = valid && !latched;
    uint32_t st2, vi2, f, vm;
    acc_t r;
    bool need_reset = false;
    step_core_unpacked<Env, CONS, CLIP, true>(p.cons, p.max_steps, s, a, nz, 0u, ep_st, ep_vi, st2, vi2, ns, r, f, vm);
    if constexpr (REC) {
        // step_kernel's outputs: the rollout computes r / f / vm for inactive lanes too, nig_step reports them as nothing happened
        const bool done = (f & (NIG_F_TERMINATED | NIG_F_TRUNCATED)) != 0;
#pragma unroll
        for (int k = 0; k < S; ++k) rec->ns[k] = active ? ns[k] : s[k];
        rec->r = active ? (float)r : 0.0f;
        rec->f = !active ? (uint32_t)NIG_F_INACTIVE : (done && p.auto_reset) ? (f | (uint32_t)NIG_F_RESET) : f;
        rec->vm = active ? vm : 0u;
    }
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
            if (extrema) { r_lo = ep_ret < r_lo ? ep_ret : r_lo; r_hi = ep_ret > r_hi ? ep_ret : r_hi; }
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

// dynamic shared memory of a launch: the blob and the activation tiles, raised where needed so that no more CTAs fit on an SM
// than its 512 tensor-memory columns serve at once (a CTA beyond that would wait inside tcgen05.alloc)
inline size_t mlp_smem_bytes(int S, const MlpParams& m)
{
    const MlpLayout L = mlp_layout(S, m);
    const size_t per_sm = 228u * 1024u, ctas = 512u / (size_t)L.tmem_cols;
    const size_t floor_ = per_sm / (ctas + 1) + 16;
    return ((size_t)L.bytes > floor_ ? (size_t)L.bytes : floor_ + 15) / 16 * 16;
}

// the opt-in dynamic shared memory of a kernel on the current device, set once per (kernel, device) and raised only when a
// larger network needs it -- not a host call per launch of the sliced nig_rollout_steps / nig_rollout_host sequences
template <class Kern>
cudaError_t mlp_prepare(Kern kern, size_t smem)
{
    struct Entry { const void* fn; int dev; size_t bytes; };
    static std::mutex mu;
    static std::vector<Entry> set;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    for (Entry& x : set)
        if (x.fn == (const void*)kern && x.dev == dev) {
            if (x.bytes >= smem) return cudaSuccess;
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) x.bytes = smem;
            return e;
        }
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) set.push_back(Entry{(const void*)kern, dev, smem});
    return e;
}

} // namespace nig
