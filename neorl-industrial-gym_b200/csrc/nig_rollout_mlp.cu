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
#include "nig_mlp.cuh"

namespace nig {

// ---- the fused rollout with the MLP policy: rollout_kernel's generic loop (rollout_step_generic, nig_mlp.cuh) with the action from
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
