// reset, state import/export and the fp32 issue-rate probe (see nig_kernels.cuh)
#include "nig_launch.h"
namespace nig {
cudaError_t launch_reset(int kind, const ResetArgs& a, cudaStream_t st)
{
    const unsigned g = grid_for(a.n);
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: reset_kernel<Reactor><<<g, kThreads, 0, st>>>(a); break;
    case NIG_ENV_POWER_GRID: reset_kernel<Grid><<<g, kThreads, 0, st>>>(a); break;
    default: reset_kernel<Robot><<<g, kThreads, 0, st>>>(a); break;
    }
    return cudaGetLastError();
}
cudaError_t launch_state_io(const StateIoArgs& a, cudaStream_t st)
{
    state_io_kernel<<<grid_for(a.n), kThreads, 0, st>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_fold_stats(unsigned long long* shards, unsigned long long* stats, cudaStream_t st)
{
    fold_stats_kernel<<<1, 32, 0, st>>>(shards, stats);
    return cudaGetLastError();
}
cudaError_t launch_commit_ticks(uint32_t* tick_base, uint32_t by, cudaStream_t st)
{
    commit_ticks_kernel<<<1, 1, 0, st>>>(tick_base, by);
    return cudaGetLastError();
}
cudaError_t launch_set_ticks(uint32_t* tick_base, uint32_t tick, uint32_t epoch, cudaStream_t st)
{
    set_ticks_kernel<<<1, 1, 0, st>>>(tick_base, tick, epoch);
    return cudaGetLastError();
}
cudaError_t launch_host_ingest(const HostIoArgs& a, cudaStream_t st)
{
    host_ingest_kernel<<<(unsigned)((a.n + kThreads - 1) / kThreads), kThreads, 0, st>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_host_export(const HostIoArgs& a, cudaStream_t st)
{
    host_export_kernel<<<(unsigned)((a.n + kThreads - 1) / kThreads), kThreads, 0, st>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_fp32_probe(float* sink, int iters, int blocks, cudaStream_t st)
{
    fp32_probe_kernel<<<blocks, 256, 0, st>>>(sink, iters);
    return cudaGetLastError();
}
cudaError_t launch_selftest_normal(uint32_t first, uint32_t stride, unsigned long long count, unsigned long long* out, cudaStream_t st)
{
    selftest_normal_kernel<<<148 * 8, 256, 0, st>>>(first, stride, count, out);
    return cudaGetLastError();
}
cudaError_t launch_selftest_division(RngKey key, int iters, int blocks, unsigned long long* out, cudaStream_t st)
{
    selftest_division_kernel<<<blocks, 256, 0, st>>>(key, iters, out);
    return cudaGetLastError();
}
cudaError_t launch_selftest_policy(int kind, const PolicyTestArgs& a, cudaStream_t st)
{
    const unsigned g = grid_for(a.n);
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: selftest_policy_kernel<Reactor><<<g, kThreads, 0, st>>>(a); break;
    case NIG_ENV_POWER_GRID: selftest_policy_kernel<Grid><<<g, kThreads, 0, st>>>(a); break;
    default: selftest_policy_kernel<Robot><<<g, kThreads, 0, st>>>(a); break;
    }
    return cudaGetLastError();
}
cudaError_t launch_rollout(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st)
{
    if (cfg.policy == NIG_POLICY_MLP) return launch_rollout_mlp(kind, cfg, pitch, a, st);
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: return launch_rollout_reactor(cfg, pitch, a, map, st);
    case NIG_ENV_POWER_GRID: return launch_rollout_grid(cfg, pitch, a, map, st);
    default: return launch_rollout_robot(cfg, pitch, a, map, st);
    }
}
} // namespace nig
