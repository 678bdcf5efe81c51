// single-step kernels of the three envs (see nig_kernels.cuh)
#include <cstdlib>
#include "nig_launch.h"
namespace nig {
namespace {
template <class Env, int VEC>
cudaError_t go(int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool plain = false)
{
    const unsigned g = grid_for((pitch + VEC - 1) / VEC);
    if constexpr (VEC == 1) {
        // the plain SoA step with the env's default constraints: the flavour with every option branch compiled out
        if (plain && cons == CONS_DEFAULT) {
            // launched with programmatic stream serialisation: back-to-back steps (a captured graph of them above all) overlap
            // the launch latency and prologue of step t + 1 with the tail of step t (griddepcontrol.wait in the kernel)
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(g); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            return cudaLaunchKernelEx(&cfg, step_kernel<Env, 1, CONS_DEFAULT, true>, a);
        }
    }
    if (cons == CONS_DEFAULT) step_kernel<Env, VEC, CONS_DEFAULT><<<g, kThreads, 0, st>>>(a);
    else if (cons == CONS_PREFIX) step_kernel<Env, VEC, CONS_PREFIX><<<g, kThreads, 0, st>>>(a);
    else step_kernel<Env, VEC, CONS_GENERIC><<<g, kThreads, 0, st>>>(a);
    return cudaGetLastError();
}

// persistent launch geometry of one step_pipe_kernel instantiation: SMs x resident CTAs, cached per device
template <class Env, int VEC, int CONS>
cudaError_t pipe_capacity(int* ctas)
{
    static int cache[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (!cache[dev]) {
        auto kern = step_pipe_kernel<Env, VEC, CONS>;
        const size_t smem = step_pipe_smem<Env, VEC>();
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        int per_sm = 0, sms = 0;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
        cache[dev] = per_sm > 0 ? per_sm * sms : sms;
    }
    *ctas = cache[dev];
    return cudaSuccess;
}

template <class Env, int VEC, int CONS>
cudaError_t go_pipe_t(int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used)
{
    int cap = 0;
    const cudaError_t e = pipe_capacity<Env, VEC, CONS>(&cap);
    if (e != cudaSuccess) return e;
    const int64_t tiles = (pitch + kThreads * VEC - 1) / (kThreads * VEC);
    if (tiles <= cap) { *used = false; return cudaSuccess; }      // one tile per CTA: nothing to pipeline
    step_pipe_kernel<Env, VEC, CONS><<<(unsigned)cap, kThreads, step_pipe_smem<Env, VEC>(), st>>>(a);
    *used = true;
    return cudaGetLastError();
}

// PowerGrid-v0: the dedicated persistent single-step kernel (NIG_GRID_STEP = 0: off); gridDim = the CTAs resident on the
// device. CTA shapes <threads, registers, normal-table replication> measured at 1M / 4M envs, us per launch
// (profiles/r02_f_grid_step_ab.txt): <256, 128, 4> 82.9 / 280 (two CTAs per SM, 16 warps, 8 B of spills), <128, 168, 4>
// 87.0 / 308 (three CTAs per SM, 12 warps, table copies shared by lane pairs), <192, 168, 4> 89.1, <192, 168, 8>
// 89.1 / 304 (two CTAs per SM, 12 warps), <384, 168, 8> 93.2 / 313 (one CTA per SM, 12 warps). The first is the one built.
cudaError_t go_grid(int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used)
{
    const char* const v = getenv("NIG_GRID_STEP");         // (read per launch: the tests switch kernels inside one process)
    if (v && atoi(v) == 0) return cudaSuccess;
    constexpr int THREADS = 256, REGS = 128, REP = 4;
    static int cache[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    auto kern = step_grid_kernel<THREADS, REGS, REP>;
    constexpr size_t smem = grid_step_smem<THREADS, REP>();
    if (!cache[dev]) {
        int per_sm = 0, sms = 0;
        if ((e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
        if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem)) != cudaSuccess) return e;
        if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
        cache[dev] = (per_sm > 0 ? per_sm : 1) * sms;
    }
    const int64_t tiles = (pitch + THREADS - 1) / THREADS;
    if (tiles < 3 * (int64_t)cache[dev]) return cudaSuccess;     // fewer than three tiles per resident CTA (131,072 envs: 24.1 vs 23.5 us): step_kernel
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)cache[dev]); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    *used = true;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

template <class Env, int VEC>
cudaError_t go_pipe(int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used)
{
    return cons == CONS_DEFAULT ? go_pipe_t<Env, VEC, CONS_DEFAULT>(pitch, a, st, used)
         : cons == CONS_PREFIX  ? go_pipe_t<Env, VEC, CONS_PREFIX>(pitch, a, st, used)
                                : go_pipe_t<Env, VEC, CONS_GENERIC>(pitch, a, st, used);
}
} // namespace

cudaError_t launch_step(int kind, int vec, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool plain)
{
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR:
        return vec == 4 ? go<Reactor, 4>(cons, pitch, a, st) : vec == 2 ? go<Reactor, 2>(cons, pitch, a, st) : go<Reactor, 1>(cons, pitch, a, st, plain);
    case NIG_ENV_POWER_GRID: return vec >= 2 ? go<Grid, 2>(cons, pitch, a, st) : go<Grid, 1>(cons, pitch, a, st, plain);
    default: return vec >= 2 ? go<Robot, 2>(cons, pitch, a, st) : go<Robot, 1>(cons, pitch, a, st, plain);
    }
}

// the persistent TMA-pipelined flavour (plain SoA step: no teacher forcing, no obs copies); *used = false when the
// population is too small to give every resident CTA more than one tile (the caller then takes launch_step)
cudaError_t launch_step_pipelined(int kind, int cons, int64_t pitch, const StepArgs& a, cudaStream_t st, bool* used)
{
    switch (kind) {
    case NIG_ENV_CHEMICAL_REACTOR: return go_pipe<Reactor, 2>(cons, pitch, a, st, used);
    case NIG_ENV_ROBOT_ASSEMBLY:
        // measured on B200 (tools/step_pipe_all_ab.py, steady-state episode mix): 92 -> 80 us at 1M envs, 328 -> 293 us
        // at 4M (0.41 -> 0.47 and 0.46 -> 0.52 of the HBM peak). Two envs per thread spill at the 128-register cap (115 us).
        return go_pipe<Robot, 1>(cons, pitch, a, st, used);
    default:
        // PowerGrid (23 Gaussian draws per step, block-cooperative reset buffer) is latency-bound at the pipeline's two
        // resident CTAs per SM (115 -> 136 us at 1M envs): with the env's default constraints it takes its own persistent
        // kernel (lean in-place step, 4 x replicated normal table), otherwise step_kernel.
        *used = false;
        if (cons == CONS_DEFAULT) return go_grid(pitch, a, st, used);
        return cudaSuccess;
    }
}
} // namespace nig
