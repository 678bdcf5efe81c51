// nig_launch.h -- kernel launchers, one translation unit per kernel family so the library builds in parallel
// (nig_step.cu, nig_rollout_{reactor,grid,robot,mlp,record}.cu, nig_dataset.cu, nig_misc.cu). nig_api.cu holds no kernels.
#pragma once
#include "nig_kernels.cuh"

namespace nig {

// NIG_POLICY_MLP: the network of nig_set_mlp_policy, packed by the library into one device blob that every CTA copies to
// shared memory verbatim (see nig_rollout_mlp.cu). Weights are bf16 in the no-swizzle K-major canonical layout of the
// tcgen05 shared-memory descriptors: element (n, k) of an [N][K] matrix at byte (k / 8) * N * 16 + n * 16 + (k % 8) * 2,
// i.e. 8 x 16-byte core matrices, rows 16 bytes apart (SBO = 128), K-neighbour core matrices N * 16 bytes apart (LBO).
struct MlpParams {
    const void* blob;
    uint32_t blob_bytes;
    int32_t layers;            // hidden layers: 1 or 2
    int32_t h1, h2;            // hidden widths (64, 128 or 256); h2 = h1 when layers == 1
    int32_t out_tanh;          // output activation: 1 tanh, 0 identity
    int32_t extrema;           // rollout only: nig_track_extrema (return_min / return_max), a run-time switch here
};
constexpr int kMlpOut = 16;    // output rows of the last MMA (A <= 8 padded to the smallest N of a 128-row MMA)
__host__ __device__ constexpr int mlp_in_pad(int s) { return (s + 15) / 16 * 16; }
// byte offsets of the blob (weights, fp32 biases, fp32 observation mean / inverse std) and, behind it, of the per-CTA
// activation tiles: the 128-row input tile and one staging tile of up to 128 columns for the hidden activations
struct MlpLayout {
    uint32_t w1, w2, w3, b1, b2, b3, mean, istd, blob, x0, stage, bytes;
    int sp, kc, tmem_cols;
};
__host__ __device__ inline MlpLayout mlp_layout(int S, const MlpParams& m)
{
    MlpLayout L{};
    L.sp = mlp_in_pad(S);
    const int hl = m.layers == 2 ? m.h2 : m.h1;                   // width feeding the output layer
    L.w1 = 0;
    L.w2 = L.w1 + (uint32_t)(m.h1 * L.sp * 2);
    L.w3 = L.w2 + (m.layers == 2 ? (uint32_t)(m.h2 * m.h1 * 2) : 0u);
    L.b1 = L.w3 + (uint32_t)(kMlpOut * hl * 2);
    L.b2 = L.b1 + (uint32_t)(m.h1 * 4);
    L.b3 = L.b2 + (m.layers == 2 ? (uint32_t)(m.h2 * 4) : 0u);
    L.mean = L.b3 + kMlpOut * 4;
    L.istd = L.mean + (uint32_t)(L.sp * 4);
    L.blob = L.istd + (uint32_t)(L.sp * 4);
    L.x0 = (L.blob + 127u) / 128u * 128u;
    L.stage = L.x0 + (uint32_t)(128 * L.sp * 2);
    const int hmax = m.h1 > m.h2 ? m.h1 : m.h2;
    L.kc = hmax < 128 ? hmax : 128;
    L.bytes = L.stage + (uint32_t)(128 * L.kc * 2);
    int cols = 32;                                                 // two accumulators: layer outputs alternate between them
    while (cols < 2 * hmax) cols *= 2;
    L.tmem_cols = cols;
    return L;
}

struct RolloutLaunch {
    int policy;        // NIG_POLICY_*
    int cons;          // CONS_GENERIC / CONS_DEFAULT / CONS_PREFIX
    bool tma;          // stage POLICY_ACTIONS through cp.async.bulk.tensor
    bool tf_noise;     // teacher-forced process noise (POLICY_ACTIONS only)
    int block;         // threads per CTA: 32, 64 or 128
    bool extrema;      // nig_track_extrema: the kernel flavour that also keeps return_min / return_max
    bool pair;         // ChemicalReactor-v0, uniform policy, default constraints: two envs per thread, packed f32x2 arithmetic
    bool grid_fast;    // PowerGrid-v0, uniform policy, default constraints, auto-reset: rollout_grid_kernel instead of the generic kernel
    MlpParams mlp;     // NIG_POLICY_MLP: the handle's network (block, pair and grid_fast do not apply)
};

cudaError_t launch_step(int kind, int vec, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool plain);
cudaError_t launch_step_pipelined(int kind, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used);
cudaError_t launch_rollout(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_reactor(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_grid(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_robot(const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const CUtensorMap& map, cudaStream_t st);
cudaError_t launch_rollout_mlp(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, cudaStream_t st);
cudaError_t launch_rollout_record(int kind, const RolloutLaunch& cfg, int64_t pitch, const RolloutArgs& a, const nig_trajectory_t& out,
                                  cudaStream_t st);
cudaError_t launch_selftest_mlp(int kind, const MlpParams& m, const float* obs, float* act, int64_t n, cudaStream_t st);
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
