// nig_rollout_mlp.cu -- NIG_POLICY_MLP: the fused K-step rollout with a learned MLP actor evaluated by the sm_100a tensor
// cores (tcgen05.mma, accumulators in tensor memory), and the selftest kernel that runs the same forward pass on given
// observations. See include/nig_b200.h (nig_mlp_t) for the numeric contract and DESIGN.md §3.6 for the budgets.
//
// One CTA = 128 threads = one 128-env tile; thread t owns env row t of every activation tile and accumulator lane t, so
// `tcgen05.ld .32x32b` hands each thread its own env's row. Per step and layer: every thread writes its bf16 input row to
// shared memory (canonical no-swizzle K-major layout), one thread issues the layer's MMAs and commits them to an mbarrier,
// every thread loads its accumulator row, applies bias and activation in fp32 and writes the next layer's bf16 input.
// Hidden activations are staged through one tile of at most 128 columns (two K chunks at width 256), which keeps the
// PowerGrid kernel at H = 256 inside the 227 KB of shared memory. Two H-wide accumulators alternate between layers.
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
template <class Env, int CONS, bool CLIP>
__device__ __forceinline__ void rollout_step_generic(const RolloutArgs& p, const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch,
                                                     bool valid, bool extrema, const float (&a)[Env::A],
                                                     const float (&nz)[Env::NZ > 0 ? Env::NZ : 1], float (&s)[Env::S],
                                                     uint32_t& ep_st, uint32_t& ep_vi, bool& latched, typename Env::acc_t& ep_ret,
                                                     float& rsum, RolloutAcc& acc, typename Env::acc_t& r_lo, typename Env::acc_t& r_hi,
                                                     float* coop_buf)
{
    constexpr int S = Env::S;
    using acc_t = typename Env::acc_t;
    float ns[S];
    const bool active = valid && !latched;
    uint32_t st2, vi2, f, vm;
    acc_t r;
    bool need_reset = false;
    step_core_unpacked<Env, CONS, CLIP, true>(p.cons, p.max_steps, s, a, nz, 0u, ep_st, ep_vi, st2, vi2, ns, r, f, vm);
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

// ---- the fused rollout with the MLP policy: rollout_kernel's generic loop (rollout_step_generic above) with the action from
// mlp_forward. 128 threads per CTA, one env per thread; CONS_DEFAULT and CONS_GENERIC (which also runs the CONS_PREFIX and
// CONS_BOUNDS* sets, bit-identically); return extrema as a run-time switch (m.extrema).
template <class Env, int CONS>
__global__ void __launch_bounds__(kThreads, 1) rollout_mlp_kernel(const __grid_constant__ RolloutArgs p, const __grid_constant__ MlpParams m)
{
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    using acc_t = typename Env::acc_t;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ double sfl[4];
    __shared__ unsigned long long sext[2];
    __shared__ float4 s_tab[Env::ROLLOUT_TAB_SMEM ? NIG_NORMAL_TAB_N : 1];
    __shared__ alignas(8) uint64_t bars[2];
    __shared__ uint32_t tmem_slot;
    __shared__ alignas(16) float coop_buf[CoopSmem<Env>::floats];
    extern __shared__ __align__(128) uint8_t mlp_smem[];
    BlockStats bs;
    if (threadIdx.x < 4) sfl[threadIdx.x] = 0.0;
    if (threadIdx.x < 2) sext[threadIdx.x] = 0ull;
    if constexpr (Env::ROLLOUT_TAB_SMEM) normal_table_to_smem(s_tab);
    const Rng key(p.key, Env::ROLLOUT_TAB_SMEM ? s_tab : g_normal_tab);
    bs.init(sstat);
    MlpCta mc;
    mlp_setup(mc, m, S, mlp_smem, bars, &tmem_slot);
    rollout_pdl_sync();

    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < p.n;
    const int64_t ic = valid ? i : 0;      // padding lanes shadow env 0 without side effects
    const uint32_t env = p.env0 + (uint32_t)ic;
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);
    const bool extrema = m.extrema != 0;

    float s[S];
#pragma unroll
    for (int k = 0; k < S; ++k) s[k] = p.state[k * p.pitch + ic];
    const uint32_t w0 = p.ep_word[ic];
    uint32_t ep_st = epw_step(w0), ep_vi = epw_viol(w0);
    bool latched = (w0 >> 31) != 0u;
    acc_t ep_ret = (acc_t)p.ep_return[ic];
    typename Env::NoiseGen ng;
    float rsum = 0.0f;
    RolloutAcc acc;
#pragma unroll
    for (int k = 0; k < NIG_MAX_CONSTRAINTS; ++k) acc.c_con[k] = 0;
    acc_t r_lo = (acc_t)INFINITY, r_hi = -(acc_t)INFINITY;

#pragma unroll 1
    for (int t = 0; t < p.n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        float a[A], nz[NZA];
        mlp_forward<S, A>(mc, m, s, a);
        if constexpr (NZ > 0) ng.get(key, env, tick, nz);
        else nz[0] = 0.0f;
        rollout_step_generic<Env, CONS, true>(p, key, env, tick, epoch, valid, extrema, a, nz, s, ep_st, ep_vi, latched, ep_ret, rsum,
                                              acc, r_lo, r_hi, coop_buf);
    }
    mlp_teardown(mc);
    if (extrema) rollout_epilogue<Env, true>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
    else rollout_epilogue<Env, false>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
}

// nig_selftest_mlp: the same forward pass and tiling on observations [n][S] -> actions [n][A]
template <class Env>
__global__ void __launch_bounds__(kThreads, 1) selftest_mlp_kernel(const __grid_constant__ MlpParams m, const float* __restrict__ obs,
                                                                   float* __restrict__ act, int64_t n)
{
    constexpr int S = Env::S, A = Env::A;
    __shared__ alignas(8) uint64_t bars[2];
    __shared__ uint32_t tmem_slot;
    extern __shared__ __align__(128) uint8_t mlp_smem[];
    MlpCta mc;
    mlp_setup(mc, m, S, mlp_smem, bars, &tmem_slot);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t ic = i < n ? i : 0;
    float s[S], a[A];
#pragma unroll
    for (int k = 0; k < S; ++k) s[k] = obs[ic * S + k];
    mlp_forward<S, A>(mc, m, s, a);
    if (i < n) {
#pragma unroll
        for (int k = 0; k < A; ++k) act[i * A + k] = a[k];
    }
    mlp_teardown(mc);
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

template <class Env>
cudaError_t rollout_mlp_env(const RolloutLaunch& c, int64_t pitch, const RolloutArgs& a, cudaStream_t st)
{
    const size_t smem = mlp_smem_bytes(Env::S, c.mlp);
    auto kern = c.cons == CONS_DEFAULT ? rollout_mlp_kernel<Env, CONS_DEFAULT> : rollout_mlp_kernel<Env, CONS_GENERIC>;
    const cudaError_t e = mlp_prepare(kern, smem);
    if (e != cudaSuccess) return e;
    return launch_pdl(kern, grid_for(pitch), (unsigned)kThreads, smem, st, a, c.mlp);
}

cudaError_t launch_rollout_mlp(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, cudaStream_t st)
{
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: return rollout_mlp_env<Reactor>(cfg, pitch, a, st);
    case NIG_ENV_POWER_GRID: return rollout_mlp_env<Grid>(cfg, pitch, a, st);
    default: return rollout_mlp_env<Robot>(cfg, pitch, a, st);
    }
}

template <class Env>
cudaError_t selftest_mlp_env(const MlpParams& m, const float* obs, float* act, int64_t n, cudaStream_t st)
{
    const size_t smem = mlp_smem_bytes(Env::S, m);
    const cudaError_t e = mlp_prepare(selftest_mlp_kernel<Env>, smem);
    if (e != cudaSuccess) return e;
    selftest_mlp_kernel<Env><<<grid_for(n), kThreads, smem, st>>>(m, obs, act, n);
    return cudaGetLastError();
}

cudaError_t launch_selftest_mlp(int kind, const MlpParams& m, const float* obs, float* act, int64_t n, cudaStream_t st)
{
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: return selftest_mlp_env<Reactor>(m, obs, act, n, st);
    case NIG_ENV_POWER_GRID: return selftest_mlp_env<Grid>(m, obs, act, n, st);
    default: return selftest_mlp_env<Robot>(m, obs, act, n, st);
    }
}

} // namespace nig
