// fused K-step rollout kernels of Grid (see nig_kernels.cuh)
#include "nig_rollout_launch.cuh"
namespace nig {
// 192 threads per CTA x 168 registers per thread: two CTAs / SM, 12 warps, no spills, the fastest of the CTA shapes measured
// at 1M envs (profiles/r02_f_grid_rollout_ab.txt)
template <bool EXTREMA>
static cudaError_t grid_fast(int64_t pitch, const RolloutArgs& a, cudaStream_t st)
{
    constexpr int THREADS = 192, MAXREG = 168;
    auto kern = rollout_grid_kernel<EXTREMA, THREADS, MAXREG>;
    constexpr size_t smem = grid_rollout_smem<THREADS>();
    static bool attr_set[64] = {false};           // the attribute is per function and per device: set once for each
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (!attr_set[dev]) {
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    return launch_pdl(kern, grid_for(pitch, THREADS), (unsigned)THREADS, smem, st, a);
}
cudaError_t launch_rollout_grid(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st)
{
    if (cfg.grid_fast && cfg.policy == NIG_POLICY_UNIFORM && cfg.cons == CONS_DEFAULT && !cfg.tma && !cfg.tf_noise)
        return cfg.extrema ? grid_fast<true>(pitch, a, st) : grid_fast<false>(pitch, a, st);
    return rollout_env<Grid>(cfg, pitch, a, map, st);
}
} // namespace nig
