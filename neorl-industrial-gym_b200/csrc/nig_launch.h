// nig_launch.h -- kernel launchers, one translation unit per kernel family so the library builds in parallel
// (nig_step.cu, nig_rollout_{reactor,grid,robot}.cu, nig_dataset.cu, nig_misc.cu). nig_api.cu holds no kernels.
#pragma once
#include "nig_kernels.cuh"

namespace nig {

struct RolloutLaunch {
    int policy;        // NIG_POLICY_*
    int cons;          // CONS_GENERIC / CONS_DEFAULT / CONS_PREFIX
    bool tma;          // stage POLICY_ACTIONS through cp.async.bulk.tensor
    bool tf_noise;     // teacher-forced process noise (POLICY_ACTIONS only)
    int block;         // threads per CTA: 32, 64 or 128
    bool extrema;      // nig_track_extrema: the kernel flavour that also keeps return_min / return_max
    bool pair;         // ChemicalReactor-v0, uniform policy, default constraints: two envs per thread, packed f32x2 arithmetic
    bool grid_fast;    // PowerGrid-v0, uniform policy, default constraints, auto-reset: rollout_grid_kernel instead of the generic kernel
};

cudaError_t launch_step(int kind, int vec, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool plain);
cudaError_t launch_step_pipelined(int kind, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used);
cudaError_t launch_rollout(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_reactor(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_grid(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_robot(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_dataset(int kind, int cons, bool write, const DatasetArgs& a, cudaStream_t st);
cudaError_t launch_reset(int kind, const ResetArgs& a, cudaStream_t st);
cudaError_t launch_state_io(const StateIoArgs& a, cudaStream_t st);
cudaError_t launch_host_ingest(const HostIoArgs& a, cudaStream_t st);
cudaError_t launch_host_export(const HostIoArgs& a, cudaStream_t st);
cudaError_t launch_scan_lengths(const int64_t* len, int64_t* off, int64_t n, int64_t* total, cudaStream_t st);
cudaError_t launch_fp32_probe(float* sink, int iters, int blocks, cudaStream_t st);
cudaError_t launch_commit_ticks(uint32_t* tick_base, uint32_t by, cudaStream_t st);
cudaError_t launch_set_ticks(uint32_t* tick_base, uint32_t tick, uint32_t epoch, cudaStream_t st);
cudaError_t launch_fold_stats(unsigned long long* shards, unsigned long long* stats, cudaStream_t st);
cudaError_t launch_selftest_normal(uint32_t first, uint32_t stride, unsigned long long count, unsigned long long* out, cudaStream_t st);
cudaError_t launch_selftest_policy(int kind, const PolicyTestArgs& a, cudaStream_t st);
cudaError_t launch_selftest_division(RngKey key, int iters, int blocks, unsigned long long* out, cudaStream_t st);

inline unsigned grid_for(int64_t items, int block = kThreads) { return (unsigned)((items + block - 1) / block); }

// launch of a kernel that executes griddepcontrol.wait before its first dependent read (rollout_pdl_sync): programmatic
// stream serialisation lets its prologue overlap the tail of the previous launch on the stream
template <class Kern, class... Args>
cudaError_t launch_pdl(Kern kern, unsigned grid, unsigned block, size_t smem, cudaStream_t st, const Args&... args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}

} // namespace nig
