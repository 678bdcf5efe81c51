// nig_rollout_record.cu -- nig_rollout_record: the fused K-step rollout that also writes every step's (obs, action, reward,
// flags, violation mask, terminated, truncated, next_obs) into time-major device arrays [K][n][dim]. Two kernels:
//  - rollout_record_kernel: teacher-forced actions (with or without teacher-forced noise) and the in-kernel policies UNIFORM,
//    ZERO, PCTRL and BASELINE -- rollout_kernel's generic loop with the policy a run-time switch;
//  - rollout_mlp_record_kernel: NIG_POLICY_MLP -- rollout_mlp_kernel's loop (same mlp_forward, tiling and tensor memory).
// Both step through rollout_step_generic (nig_kernels.cuh) with its record outputs, so that dynamics, statistics and episode
// bookkeeping are nig_rollout's, and both end in rollout_epilogue. 128 threads per CTA, one env per thread; CONS_DEFAULT and
// CONS_GENERIC (which runs every other constraint set bit-identically). AoS rows leave through the per-warp shared-memory
// transpose (store_aos_warp) with streaming stores. See DESIGN.md §3.7 for the budgets.
#include "nig_mlp.cuh"

namespace nig {

// per-warp transpose tile of the AoS rows: 32 rows of S + 1 floats (S >= A for every env)
template <class Env>
__host__ __device__ constexpr uint32_t rec_tile_floats() { return 32u * (uint32_t)(Env::S + 1); }

// the rows known before the step: s_t and the action. Convergent (every lane of the warp; padding lanes store nothing).
template <class Env>
__device__ __forceinline__ void record_pre(const nig_trajectory_t& o, int64_t row0, int64_t n, int64_t i, const float (&s)[Env::S],
                                           const float (&a)[Env::A], float* tile)
{
    if (o.obs) store_aos_warp<Env::S, true>(o.obs + row0 * Env::S, n, i, s, tile);
    if (o.actions) store_aos_warp<Env::A, true>(o.actions + row0 * Env::A, n, i, a, tile);
}

// the rows of the transition; the [K][n] rows are one contiguous 32- or 128-byte segment per warp already
template <class Env>
__device__ __forceinline__ void record_post(const nig_trajectory_t& o, int64_t row0, int64_t n, int64_t i, bool valid,
                                            const StepRecord<Env>& rc, float* tile)
{
    if (o.next_obs) store_aos_warp<Env::S, true>(o.next_obs + row0 * Env::S, n, i, rc.ns, tile);
    if (valid) {
        const int64_t j = row0 + i;
        if (o.rewards) __stcs(o.rewards + j, rc.r);
        if (o.flags) __stcs(o.flags + j, (unsigned char)rc.f);
        if (o.viol_mask) __stcs(o.viol_mask + j, (unsigned char)rc.vm);
        if (o.terminated) __stcs(o.terminated + j, (unsigned char)((rc.f & NIG_F_TERMINATED) ? 1 : 0));
        if (o.truncated) __stcs(o.truncated + j, (unsigned char)((rc.f & NIG_F_TRUNCATED) ? 1 : 0));
    }
}

struct RecordPolicy {
    int32_t policy;            // NIG_POLICY_* other than MLP: a run-time switch (uniform across the grid)
    int32_t extrema;           // nig_track_extrema
};

template <class Env, int CONS>
__global__ void __launch_bounds__(kThreads) rollout_record_kernel(const __grid_constant__ RolloutArgs p, const __grid_constant__ nig_trajectory_t o,
                                                                  const RecordPolicy rp)
{
    constexpr int S = Env::S, A = Env::A, NZ = Env::NZ, NZA = NZ > 0 ? NZ : 1;
    using acc_t = typename Env::acc_t;
    __shared__ unsigned int sstat[NIG_STATS_SLOTS];
    __shared__ double sfl[4];
    __shared__ unsigned long long sext[2];
    __shared__ float4 s_tab[Env::ROLLOUT_TAB_SMEM ? NIG_NORMAL_TAB_N : 1];
    __shared__ alignas(16) float coop_buf[CoopSmem<Env>::floats];
    __shared__ float rec_tile[(kThreads / 32) * rec_tile_floats<Env>()];
    float* tile = rec_tile + (threadIdx.x >> 5) * rec_tile_floats<Env>();
    BlockStats bs;
    const Rng key = rollout_cta_init<Env>(p, bs, sstat, sfl, sext, s_tab, true);
    rollout_pdl_sync();

    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < p.n;
    const int64_t ic = valid ? i : 0;      // padding lanes shadow env 0 without side effects
    const uint32_t env = p.env0 + (uint32_t)ic;
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);
    const bool extrema = rp.extrema != 0;
    const bool pid = rp.policy == NIG_POLICY_BASELINE && p.pp.baseline.kind == NIG_BASELINE_PID && p.pid_state != nullptr;

    float s[S];
    uint32_t ep_st, ep_vi;
    bool latched;
    acc_t ep_ret;
    rollout_load<Env>(p, ic, s, ep_st, ep_vi, latched, ep_ret);
    typename Env::NoiseGen ng;
    float rsum = 0.0f;
    RolloutAcc acc;
    acc_t r_lo = (acc_t)INFINITY, r_hi = -(acc_t)INFINITY;
    double pid_i[A], pid_e[A];             // POLICY_BASELINE: the PID agent's integral and previous error
#pragma unroll
    for (int k = 0; k < A; ++k) {
        pid_i[k] = pid ? p.pid_state[(int64_t)k * p.pitch + ic] : 0.0;
        pid_e[k] = pid ? p.pid_state[(int64_t)(A + k) * p.pitch + ic] : 0.0;
    }

#pragma unroll 1
    for (int t = 0; t < p.n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        const int64_t row0 = (int64_t)t * p.n;
        float a[A], nz[NZA];
        if (rp.policy == NIG_POLICY_ACTIONS) {
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = __ldcs(p.actions + ((int64_t)t * A + k) * p.pitch + ic);
        } else if (rp.policy == NIG_POLICY_UNIFORM) {
            policy_uniform<Env>(key, env, tick, a);
        } else if (rp.policy == NIG_POLICY_PCTRL) {
            policy_pctrl<Env>(key, p.pp, env, tick, s, a);
        } else if (rp.policy == NIG_POLICY_BASELINE) {
            policy_baseline<Env>(key, p.pp.baseline, env, tick, s, a, pid_i, pid_e);
        } else {
#pragma unroll
            for (int k = 0; k < A; ++k) a[k] = 0.0f;
        }
        if constexpr (NZ > 0) {
            if (p.noise) {
#pragma unroll
                for (int k = 0; k < NZA; ++k) nz[k] = __ldcs(p.noise + ((int64_t)t * NZA + k) * p.pitch + ic);
            } else ng.get(key, env, tick, nz);
        } else nz[0] = 0.0f;
        record_pre<Env>(o, row0, p.n, i, s, a, tile);
        // (the clip is the identity on the uniform policy's actions: CLIP = true for every policy gives rollout_kernel's values)
        StepRecord<Env> rc;
        rollout_step_generic<Env, CONS, true, true>(p, key, env, tick, epoch, valid, extrema, a, nz, s, ep_st, ep_vi, latched, ep_ret,
                                                    rsum, acc, r_lo, r_hi, coop_buf, &rc);
        record_post<Env>(o, row0, p.n, i, valid, rc, tile);
    }

    if (valid && pid) {
#pragma unroll
        for (int k = 0; k < A; ++k) {
            p.pid_state[(int64_t)k * p.pitch + i] = pid_i[k];
            p.pid_state[(int64_t)(A + k) * p.pitch + i] = pid_e[k];
        }
    }
    if (extrema) rollout_epilogue<Env, true>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
    else rollout_epilogue<Env, false>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
}

// NIG_POLICY_MLP: rollout_mlp_kernel's loop with the record rows. The transpose tiles live in the hidden-activation staging
// tile of the MLP's shared memory (L.stage): it is free from the wait for a step's last MMA to the first hidden-activation
// write of the next step's forward pass, which comes after that forward pass's publish barrier (mlp_publish_smem: the
// proxy fence orders the hand-back to the tensor cores, the CTA barrier keeps every warp's transposes ahead of it).
template <class Env, int CONS>
__global__ void __launch_bounds__(kThreads, 1) rollout_mlp_record_kernel(const __grid_constant__ RolloutArgs p,
                                                                         const __grid_constant__ nig_trajectory_t o,
                                                                         const __grid_constant__ MlpParams m)
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
    const Rng key = rollout_cta_init<Env>(p, bs, sstat, sfl, sext, s_tab, true);
    MlpCta mc;
    mlp_setup(mc, m, S, mlp_smem, bars, &tmem_slot);
    rollout_pdl_sync();
    float* tile = reinterpret_cast<float*>(mlp_smem + mc.L.stage) + (threadIdx.x >> 5) * rec_tile_floats<Env>();

    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < p.n;
    const int64_t ic = valid ? i : 0;
    const uint32_t env = p.env0 + (uint32_t)ic;
    const uint32_t tick0 = load_tick(p.tick_dev, p.tick) + base_tick(p.tick_base);
    const uint32_t epoch = p.epoch + base_epoch(p.tick_base);
    const bool extrema = m.extrema != 0;

    float s[S];
    uint32_t ep_st, ep_vi;
    bool latched;
    acc_t ep_ret;
    rollout_load<Env>(p, ic, s, ep_st, ep_vi, latched, ep_ret);
    typename Env::NoiseGen ng;
    float rsum = 0.0f;
    RolloutAcc acc;
    acc_t r_lo = (acc_t)INFINITY, r_hi = -(acc_t)INFINITY;

#pragma unroll 1
    for (int t = 0; t < p.n_steps; ++t) {
        const uint32_t tick = tick0 + (uint32_t)t;
        const int64_t row0 = (int64_t)t * p.n;
        float a[A], nz[NZA];
        mlp_forward<S, A>(mc, m, s, a);
        if constexpr (NZ > 0) ng.get(key, env, tick, nz);
        else nz[0] = 0.0f;
        record_pre<Env>(o, row0, p.n, i, s, a, tile);
        StepRecord<Env> rc;
        rollout_step_generic<Env, CONS, true, true>(p, key, env, tick, epoch, valid, extrema, a, nz, s, ep_st, ep_vi, latched, ep_ret,
                                                    rsum, acc, r_lo, r_hi, coop_buf, &rc);
        record_post<Env>(o, row0, p.n, i, valid, rc, tile);
    }
    mlp_teardown(mc);
    if (extrema) rollout_epilogue<Env, true>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
    else rollout_epilogue<Env, false>(p, bs, sfl, sext, valid, i, s, ep_st, ep_vi, latched, ep_ret, rsum, acc, r_lo, r_hi);
}

template <class Env>
cudaError_t rollout_record_env(const RolloutLaunch& c, int64_t pitch, const RolloutArgs& a, const nig_trajectory_t& o, cudaStream_t st)
{
    if (c.policy == NIG_POLICY_MLP) {
        // the MLP rollout's shared memory, widened where the staging tile is smaller than the four warps' transpose tiles
        // (a hidden width of 64 with PowerGrid's 32-float rows)
        const MlpLayout L = mlp_layout(Env::S, c.mlp);
        const size_t tiles = (size_t)L.stage + (kThreads / 32) * rec_tile_floats<Env>() * sizeof(float);
        size_t smem = mlp_smem_bytes(Env::S, c.mlp);
        if (tiles > smem) smem = (tiles + 15) / 16 * 16;
        auto kern = c.cons == CONS_DEFAULT ? rollout_mlp_record_kernel<Env, CONS_DEFAULT> : rollout_mlp_record_kernel<Env, CONS_GENERIC>;
        const cudaError_t e = mlp_prepare(kern, smem);
        if (e != cudaSuccess) return e;
        return launch_pdl(kern, grid_for(pitch), (unsigned)kThreads, smem, st, a, o, c.mlp);
    }
    const RecordPolicy rp{c.policy, c.extrema ? 1 : 0};
    auto kern = c.cons == CONS_DEFAULT ? rollout_record_kernel<Env, CONS_DEFAULT> : rollout_record_kernel<Env, CONS_GENERIC>;
    return launch_pdl(kern, grid_for(pitch), (unsigned)kThreads, 0, st, a, o, rp);
}

cudaError_t launch_rollout_record(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const nig_trajectory_t& out,
                                  cudaStream_t st)
{
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: return rollout_record_env<Reactor>(cfg, pitch, a, out, st);
    case NIG_ENV_POWER_GRID: return rollout_record_env<Grid>(cfg, pitch, a, out, st);
    default: return rollout_record_env<Robot>(cfg, pitch, a, out, st);
    }
}

} // namespace nig
