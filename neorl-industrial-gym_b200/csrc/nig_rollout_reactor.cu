// fused K-step rollout kernels of Reactor (see nig_kernels.cuh)
#include "nig_rollout_launch.cuh"
namespace nig {
cudaError_t launch_rollout_reactor(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st)
{
    if (cfg.pair && cfg.policy == NIG_POLICY_UNIFORM && cfg.cons == CONS_DEFAULT && !cfg.tma && !cfg.tf_noise) {
        const unsigned grid = grid_for(pitch / 2, cfg.block);
        return cfg.extrema ? launch_pdl(rollout_reactor_pair_kernel<true>, grid, (unsigned)cfg.block, 0, st, a)
                           : launch_pdl(rollout_reactor_pair_kernel<false>, grid, (unsigned)cfg.block, 0, st, a);
    }
    return rollout_env<Reactor>(cfg, pitch, a, map, st);
}
} // namespace nig
