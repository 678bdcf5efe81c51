// nig_api.cu -- C-ABI of libnig_b200.so (see include/nig_b200.h). Host-side handle management,
// argument validation, kernel dispatch and the host<->device staging of the *_host entry points.
// There is no CPU implementation of the step path in this library: without an sm_100 device
// nig_create() fails with NIG_ERR_NO_DEVICE.
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <new>
#include <dlfcn.h>

#include "nig_launch.h"

using namespace nig;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define NIG_CUDA(expr)                                                                                \
    do {                                                                                              \
        cudaError_t e_ = (expr);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(NIG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

const int kS[3] = {Reactor::S, Grid::S, Robot::S};
const int kA[3] = {Reactor::A, Grid::A, Robot::A};
const int kNZ[3] = {Reactor::NZ, Grid::NZ, Robot::NZ};
const int kMaxSteps[3] = {Reactor::MAX_STEPS, Grid::MAX_STEPS, Robot::MAX_STEPS};

void builtin_constraints(int kind, nig_constraint_t* c)
{
    // penalties / critical flags in registration order: chemical_reactor.py:38-60, power_grid.py:53-72,
    // robot_assembly.py:56-75
    const float pen[3][3] = {{-100.f, -50.f, -25.f}, {-50.f, -30.f, -20.f}, {-100.f, -200.f, -50.f}};
    for (int k = 0; k < 3; ++k) {
        c[k] = nig_constraint_t{NIG_CON_BUILTIN, k, 0, -1, 0.f, 0.f, 0.f, pen[kind][k], k < 2 ? 1 : 0};
    }
}

// how the kernels evaluate a constraint set: CONS_DEFAULT = exactly the env's three built-ins in registration order with
// their default penalties (compile-time code); CONS_PREFIX = those three first, then extra descriptors (a SafetyWrapper
// that appends constraints: built-ins stay compile-time code, a loop walks descriptors 3..n-1), or CONS_BOUNDS1 / 2 when
// the extras are one / two pure state bounds (straight-line code in the fused rollout); CONS_GENERIC otherwise.
int cons_mode(int kind, const nig_constraint_t* c, int n)
{
    if (n < 3) return CONS_GENERIC;
    nig_constraint_t d[3];
    builtin_constraints(kind, d);
    for (int k = 0; k < 3; ++k)
        if (c[k].kind != NIG_CON_BUILTIN || c[k].id != k || c[k].penalty != d[k].penalty || (c[k].critical != 0) != (d[k].critical != 0))
            return CONS_GENERIC;
    if (n == 3) return CONS_DEFAULT;
    bool pure_bounds = n <= 5;              // one or two extras, each lo <= s[i] <= hi without an action term
    for (int k = 3; k < n && pure_bounds; ++k) pure_bounds = c[k].kind == NIG_CON_BOUND && c[k].ai < 0;
    return pure_bounds ? (n == 4 ? CONS_BOUNDS1 : CONS_BOUNDS2) : CONS_PREFIX;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

} // namespace

constexpr int kMaxHostSlices = 16;
struct nig_env {
    nig_config_t cfg;
    int kind, S, A, NZ;
    int64_t n, pitch;
    int max_steps;
    ConsParams cons;
    RngKey key;
    uint32_t tick, epoch;
    float* state;
    uint32_t* ep_word;
    double* ep_return;
    unsigned long long* stats;
    cudaStream_t stream;       // internal stream of the *_host calls
    cudaStream_t dev_streams[4];   // caller streams device-API work was submitted on since the last *_host call ...
    int n_dev_streams;             // ... (more than four distinct ones: dev_sync_all) ...
    bool dev_sync_all;
    bool dev_dirty;                // ... and whether a *_host call still has to wait for them
    // device staging of the *_host calls (lazily allocated)
    float *h_actions, *h_noise, *h_reset, *h_obs, *h_next_obs, *h_reward;
    uint8_t *h_hostmask, *h_flags, *h_viol, *h_mask, *h_terminated, *h_truncated;
    int32_t *h_i32a, *h_i32b;
    unsigned long long* stats_shards;   // kStatsShards x NIG_STATS_SLOTS: where the PLAIN single-step kernel adds (folded into stats on read)
    bool shards_dirty;
    unsigned long long* extrema; // [2] min / max finished-episode return keys (outside the summable stats block)
    bool track_extrema;          // nig_track_extrema: rollouts run the EXTREMA kernel flavour
    bool track_step_stats;       // nig_track_step_stats (default on): the single-step kernels add to the device counter block
    bool track_returns;          // nig_track_returns (default on, set in nig_create): the single-step kernels keep the episode-return accumulator too
    // nig_rollout_host over env slices: slice s runs H2D -> reset -> K-step launches -> D2H on its own stream, so the
    // copies of one slice overlap the stepping of the others (and the slices' launches fill each other's tails)
    cudaStream_t slice_stream[kMaxHostSlices];
    cudaEvent_t slice_done[kMaxHostSlices], slice_begin;
    // ... and that whole pipeline captured once in a CUDA graph and replayed (one driver call per nig_rollout_host instead
    // of ~25 per slice): the kernels of a captured pipeline take tick / epoch as offsets from d_tickbase, which the graph's
    // first node refreshes from the pinned word h_tickbase
    cudaGraphExec_t host_graph;
    struct HostGraphKey {
        const void* ptr[5]; int32_t T, K, policy, reset, slices; int64_t launches; uint64_t config; nig_policy_params_t pp;
    } host_graph_key;
    uint32_t *d_tickbase, *h_tickbase;
    // nig_rollout_steps (device-resident): its sliced launch sequence (fork, slices x ceil(T / K) launches, join) captured once
    // on the internal stream and replayed on the caller's stream -- 2 driver calls per call instead of ~150, so the host
    // thread no longer paces the first steps of a short run. Tick / epoch reach the replay through d_tickbase, written by a
    // one-thread kernel launched (arguments by value) right before the graph.
    cudaGraphExec_t steps_graph;
    struct StepsGraphKey {
        const void* ptr[3]; int32_t T, K, policy, flags, slices; int64_t launches; uint64_t config; nig_policy_params_t pp;
    } steps_graph_key, steps_graph_candidate;
    int steps_graph_enable;     // NIG_STEPS_GRAPH (default 1)
    unsigned long long* h_stats_pinned;   // nig_rollout_host: page-locked landing block of the statistics copy
    double host_direct_max_mb[2];  // NIG_HOST_DIRECT_MAX_MB: ingest, export
    int host_direct;            // NIG_HOST_DIRECT (default 1): nig_rollout_host's slices read / write mapped host arrays in-kernel
    bool graph_mode;            // set while a pipeline is being captured: rollout_range / reset_range emit base-relative counters
    uint32_t graph_tick0;       // tick at the start of the call being captured
    uint64_t config_version;    // bumped by every setter whose value is baked into kernel arguments (invalidates host_graph)
    int host_graph_enable;      // NIG_HOST_GRAPH (default 1)
    uint32_t* cons_masks;       // device copy of the NIG_CON_BOUND one-hot masks (ConsParams::masks)
    uint32_t* tick_dev;         // device-tick modes (CUDA-graph capture): [0] tick, [1] finished-CTA counter; null = host tick
    int tick_mode;              // 0 host tick; 1 device tick advanced by every launch; 2 device BASE + per-launch sequence offsets
    uint32_t tick_commit;       // mode 2: host tick at the last nig_commit_ticks (launch offset = tick - tick_commit)
    double* pid_state;          // [2][A][pitch] PID integral / previous error of NIG_POLICY_BASELINE (lazily allocated, zeroed)
    float *r_act[2], *r_nz[2];  // nig_rollout_host: double-buffered action / noise chunks
    int32_t r_cap;              // steps each chunk buffer holds
    cudaStream_t copy_stream;
    cudaEvent_t r_ev_copy[2], r_ev_done[2];
    int64_t launches;
    int step_vec;              // 0 = auto
    int rollout_block;         // 0 = 128
    int rollout_pair;          // two envs per thread + packed f32x2 (NIG_ROLLOUT_PAIR)
    bool grid_fast;            // PowerGrid-v0 dedicated rollout kernel (NIG_GRID_FAST = 0: off)
    int zero_copy;             // 1 (default): small-population *_host steps run in place on page-locked host buffers
    int step_pipe;             // 1 (default): large plain SoA steps take the persistent TMA-pipelined kernel
    PFN_encodeTiled encode_tiled;
    int64_t *d_len, *d_off, *d_total;   // dataset: per-episode lengths, offsets, total
    int64_t d_len_cap;
    uint32_t dataset_gen;      // datasets generated so far (each one draws from a fresh derived key)
    struct { int64_t n_episodes; int32_t n_steps, policy; nig_policy_params_t pp; ConsParams cons; RngKey key; int64_t total; bool valid; } probe;
    void* mlp_blob;            // NIG_POLICY_MLP: the packed network (nig_set_mlp_policy; MlpParams::blob)
    size_t mlp_cap;            // bytes allocated at mlp_blob
    MlpParams mlp;             // blob null until a network is set
};

namespace {

template <class T>
int dev_alloc(T** p, size_t count)
{
    if (*p) return NIG_OK;
    NIG_CUDA(cudaMalloc((void**)p, count * sizeof(T)));
    NIG_CUDA(cudaMemset(*p, 0, count * sizeof(T)));
    // cudaMemset runs on the legacy default stream and may return before it has executed; the buffers are used on
    // non-blocking streams (e->stream, the caller's) that do not synchronise with it -- without this barrier the zero
    // fill can land AFTER the first cudaMemcpyAsync into a freshly allocated staging buffer (found by tools/soak_parity.py)
    NIG_CUDA(cudaDeviceSynchronize());
    return NIG_OK;
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// device-API calls run on the caller's stream, *_host calls on e->stream: a *_host call first waits for the device
// work submitted since the last one (no cost for loops of device calls; the *_host calls are synchronous anyway)
inline void note_device_work(nig_env* e, cudaStream_t st)
{
    if (st == e->stream) return;
    e->dev_dirty = true;
    for (int k = 0; k < e->n_dev_streams; ++k)
        if (e->dev_streams[k] == st) return;
    if (e->n_dev_streams < 4) e->dev_streams[e->n_dev_streams++] = st;
    else e->dev_sync_all = true;
}
int host_entry(nig_env* e)
{
    if (e->dev_dirty) {
        if (e->dev_sync_all) NIG_CUDA(cudaDeviceSynchronize());
        else for (int k = 0; k < e->n_dev_streams; ++k) NIG_CUDA(cudaStreamSynchronize(e->dev_streams[k]));
        e->dev_dirty = false; e->dev_sync_all = false; e->n_dev_streams = 0;
    }
    return NIG_OK;
}

// how a launch at host tick `tick` gets its counters (see nig_use_device_tick): kernel argument, device tick, or base + offset
template <class Args>
void fill_tick(const nig_env* e, Args& a, uint32_t tick)
{
    if (e->graph_mode) { a.tick = tick - e->graph_tick0; a.tick_dev = nullptr; a.tick_base = e->d_tickbase; }
    else if (e->tick_mode == 2) { a.tick = tick - e->tick_commit; a.tick_dev = nullptr; a.tick_base = e->tick_dev; }
    else { a.tick = tick; a.tick_dev = e->tick_dev; a.tick_base = nullptr; }
}

// the PLAIN single-step kernel adds its counters to shard copies of the stats block: fold them in before the block is read
int fold_stats(nig_env* e, cudaStream_t st)
{
    if (!e->shards_dirty) return NIG_OK;
    e->launches++;
    NIG_CUDA(nig::launch_fold_stats(e->stats_shards, e->stats, st));
    e->shards_dirty = false;
    return NIG_OK;
}

// the VEC > 1 flavours move VEC envs per thread with one vector load / store per row: every caller array must be aligned
// to it (a torch view at an odd element offset is not)
bool vec_aligned(const StepArgs& a, int vec)
{
    const uintptr_t f = (uintptr_t)(4 * vec) - 1, b = (uintptr_t)vec - 1;
    return !((((uintptr_t)a.actions | (uintptr_t)a.noise | (uintptr_t)a.reset_states | (uintptr_t)a.obs | (uintptr_t)a.next_obs |
               (uintptr_t)a.reward) & f) | (((uintptr_t)a.flags | (uintptr_t)a.viol_mask) & b));
}

int pick_vec(const nig_env* e, const StepArgs& a)
{
    // AoS calls always take VEC = 1: the wider flavours store reward / flags / masks for every env up to the pitch, which
    // would write past the caller's exact-size [n] arrays (nig_step_host's zero-copy path hands those to the kernel)
    if (a.action_aos || a.aux_aos) return 1;
    int vec = 1;
    if (e->step_vec) vec = e->step_vec;
    // reactor: two envs per thread (64-bit LDG/STG, 96 registers) once there are enough threads to fill the GPU
    // twice over; measured on B200 (tools/perf_sweep.py): VEC=2 beats VEC=1 and VEC=4 from 1M envs up.
    // (32-/24-d states: two envs per thread would need > 190 registers)
    else if (e->kind == NIG_ENV_CHEMICAL_REACTOR && e->pitch >= 2 * 148LL * 2048) vec = 2;
    while (vec > 1 && !vec_aligned(a, vec)) vec /= 2;
    return vec;
}

int launch_step(nig_env* e, const StepArgs& a, cudaStream_t st)
{
    const int vec = pick_vec(e, a);
    e->launches++;
    note_device_work(e, st);
    // plain SoA step (no teacher forcing, no observation copies, no host-evaluated constraints): persistent TMA pipeline
    const bool plain_args = !a.action_aos && !a.aux_aos && !a.noise && !a.reset_states && !a.hostmask && !a.obs && !a.next_obs && !a.terminated && !a.truncated;
    const bool plain = plain_args && ((uintptr_t)a.actions & 15u) == 0 && e->step_pipe != 0 && e->step_vec == 0;
    if (plain) {
        bool used = false;
        NIG_CUDA(nig::launch_step_pipelined(e->kind, cons_for_step(e->cons.is_default), e->pitch, a, st, &used));
        if (used) return NIG_OK;
    }
    NIG_CUDA(nig::launch_step(e->kind, vec, cons_for_step(e->cons.is_default), e->pitch, a, st, plain_args));
    return NIG_OK;
}

int make_action_map(nig_env* e, const float* actions, int n_steps, CUtensorMap* map)
{
    if (!e->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        NIG_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) return fail(NIG_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
        e->encode_tiled = (PFN_encodeTiled)fn;
    }
    // actions[K][A][pitch] fp32 as a 3-D tensor (x = env, y = action component, z = step); one box = the
    // tma_chunk(A) x A x 128 tile a CTA consumes over tma_chunk(A) steps
    const cuuint64_t gdim[3] = {(cuuint64_t)e->pitch, (cuuint64_t)e->A, (cuuint64_t)n_steps};
    const cuuint64_t gstr[2] = {(cuuint64_t)e->pitch * sizeof(float), (cuuint64_t)e->pitch * e->A * sizeof(float)};
    const cuuint32_t box[3] = {(cuuint32_t)kThreads, (cuuint32_t)e->A, (cuuint32_t)tma_chunk(e->A)};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = e->encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)actions, gdim, gstr, box, estr,
                                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(NIG_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return NIG_OK;
}

int validate_constraints(int kind, const nig_constraint_t* c, int n)
{
    if (n < 0 || n > NIG_MAX_CONSTRAINTS) return fail(NIG_ERR_INVALID, "n_constraints %d outside [0, %d]", n, NIG_MAX_CONSTRAINTS);
    for (int k = 0; k < n; ++k) {
        switch (c[k].kind) {
        case NIG_CON_BUILTIN:
            if (c[k].id < 0 || c[k].id > 2) return fail(NIG_ERR_INVALID, "constraint %d: builtin id %d outside [0, 2]", k, c[k].id);
            break;
        case NIG_CON_BOUND:
            if (c[k].si < 0 || c[k].si >= kS[kind]) return fail(NIG_ERR_INVALID, "constraint %d: state index %d outside [0, %d)", k, c[k].si, kS[kind]);
            if (c[k].ai >= kA[kind]) return fail(NIG_ERR_INVALID, "constraint %d: action index %d outside [-1, %d)", k, c[k].ai, kA[kind]);
            break;
        case NIG_CON_HOSTMASK:
            if (c[k].id < 0 || c[k].id > 7) return fail(NIG_ERR_INVALID, "constraint %d: hostmask bit %d outside [0, 7]", k, c[k].id);
            break;
        default: return fail(NIG_ERR_INVALID, "constraint %d: unknown kind %d", k, c[k].kind);
        }
    }
    return NIG_OK;
}

int set_cons(nig_env* e, const nig_constraint_t* c, int n)
{
    memset(&e->cons, 0, sizeof e->cons);
    e->cons.n = n;
    uint32_t host_masks[NIG_MAX_CONSTRAINTS * kConsMaskRow];
    memset(host_masks, 0, sizeof host_masks);
    for (int k = 0; k < n; ++k) {
        e->cons.c[k] = c[k];
        if (c[k].kind == NIG_CON_BOUND) {
            host_masks[k * kConsMaskRow + c[k].si] = 0xffffffffu;
            if (c[k].ai >= 0) host_masks[k * kConsMaskRow + NIG_MAX_STATE_DIM + c[k].ai] = 0xffffffffu;
        }
    }
    e->cons.masks = e->cons_masks;
    if (e->cons_masks) {       // allocated in nig_create before the first set_cons
        NIG_CUDA(cudaDeviceSynchronize());
        NIG_CUDA(cudaMemcpy(e->cons_masks, host_masks, sizeof host_masks, cudaMemcpyHostToDevice));
        NIG_CUDA(cudaDeviceSynchronize());   // a pageable H2D cudaMemcpy may return before the DMA lands; kernels run on non-blocking streams
    }
    e->cons.is_default = cons_mode(e->kind, c, n);
    return NIG_OK;
}

#define NIG_CHECK_ENV(e)                                                        \
    if (!(e)) return fail(NIG_ERR_INVALID, "null env handle");                  \
    DeviceGuard guard_((e)->cfg.device);                                        \
    if (!guard_.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", (e)->cfg.device)

int state_io(nig_env* e, float* ext_state, int layout, int32_t* st, int32_t* vi, uint8_t* dn, bool to_ext, cudaStream_t s)
{
    StateIoArgs a{e->state, e->ep_word, e->n, e->pitch, ext_state, st, vi, dn, e->S, layout == NIG_LAYOUT_AOS ? 1 : 0, to_ext ? 1 : 0};
    // importing an episode step counter re-bases the episode: its return accumulator restarts from zero
    a.ep_return = (!to_ext && st) ? e->ep_return : nullptr;
    e->launches++;
    note_device_work(e, s);
    NIG_CUDA(nig::launch_state_io(a, s));
    return NIG_OK;
}

// envs [i0, i0 + ns) of the handle -> rows [i0, i0 + ns) of an AoS [n][S] device array
int state_to_aos_range(nig_env* e, float* ext_aos, int64_t i0, int64_t ns, cudaStream_t s)
{
    StateIoArgs a{e->state + i0, e->ep_word + i0, ns, e->pitch, ext_aos + i0 * e->S, nullptr, nullptr, nullptr, e->S, 1, 1};
    a.ep_return = nullptr;
    e->launches++;
    NIG_CUDA(nig::launch_state_io(a, s));
    return NIG_OK;
}

// IndustrialEnv.reset of envs [i0, i0 + ns) with an explicit epoch (the caller bumps e->epoch once for all slices)
int reset_range(nig_env* e, const float* init_aos, int64_t i0, int64_t ns, uint32_t epoch, cudaStream_t s)
{
    ResetArgs a{e->state + i0, e->ep_word + i0, e->ep_return + i0, ns, e->pitch, (uint32_t)e->cfg.env_id_offset + (uint32_t)i0, e->tick, epoch,
                e->tick_dev, e->key, nullptr, init_aos ? init_aos + i0 * e->S : nullptr, 1, nullptr};
    fill_tick(e, a, e->tick);
    if (e->graph_mode) a.epoch = 0u;
    e->launches++;
    NIG_CUDA(nig::launch_reset(e->kind, a, s));
    return NIG_OK;
}

// argument checks of a fused rollout (shared by nig_rollout and the sliced nig_rollout_host); allocates the PID state
int rollout_checks(nig_env* e, const nig_rollout_t* r)
{
    if (!r) return fail(NIG_ERR_INVALID, "nig_rollout: null descriptor");
    if (r->n_steps <= 0 || r->n_steps > NIG_MAX_LAUNCH_STEPS)
        return fail(NIG_ERR_INVALID, "nig_rollout: n_steps %d outside [1, NIG_MAX_LAUNCH_STEPS = %d]", r->n_steps, NIG_MAX_LAUNCH_STEPS);
    if (r->policy == NIG_POLICY_ACTIONS && !r->actions) return fail(NIG_ERR_INVALID, "nig_rollout: NIG_POLICY_ACTIONS needs an actions tensor");
    if (r->noise && e->NZ == 0) return fail(NIG_ERR_INVALID, "nig_rollout: env kind %d has no process noise", e->kind);
    if (r->noise && r->policy != NIG_POLICY_ACTIONS)
        return fail(NIG_ERR_UNSUPPORTED, "nig_rollout: teacher-forced noise is only available together with teacher-forced actions (NIG_POLICY_ACTIONS)");
    if (r->policy < NIG_POLICY_ACTIONS || r->policy > NIG_POLICY_MLP) return fail(NIG_ERR_INVALID, "unknown rollout policy %d", r->policy);
    if (r->policy == NIG_POLICY_MLP && !e->mlp.blob) return fail(NIG_ERR_INVALID, "nig_rollout: NIG_POLICY_MLP needs a network (nig_set_mlp_policy)");
    if (r->noise && e->track_extrema)
        return fail(NIG_ERR_UNSUPPORTED, "nig_rollout: teacher-forced noise has no return-extrema kernel flavour (nig_track_extrema(env, 0) first)");
    if (r->policy == NIG_POLICY_BASELINE) {
        const nig_baseline_t& b = r->pp.baseline;
        if (b.kind < NIG_BASELINE_RANDOM || b.kind > NIG_BASELINE_CONSTANT) return fail(NIG_ERR_INVALID, "unknown baseline controller %d", b.kind);
        if (b.kind == NIG_BASELINE_PID) {
            const int prc = dev_alloc(&e->pid_state, (size_t)2 * e->A * e->pitch);      // zero-initialised = a fresh agent
            if (prc != NIG_OK) return prc;
        }
    }
    for (int k = 0; k < e->cons.n; ++k)
        if (e->cons.c[k].kind == NIG_CON_HOSTMASK) return fail(NIG_ERR_UNSUPPORTED, "nig_rollout: host-evaluated constraints cannot run inside a fused rollout");
    return NIG_OK;
}

// how many env slices nig_rollout_host uses: 1 for teacher-forced inputs (their [T][D][n] chunks are already
// double-buffered on a copy stream), for device-tick handles (graph capture) and for small populations; else
// NIG_HOST_SLICES (default: 4 through the host-buffer call, 8 through the device call -- measured on B200 at 65,536 reactor
// envs, bench.py: device 6.76 / 7.51 / 7.70 / 7.81e10 env-steps/s and host 5.69 / 6.38 / 6.58 / 6.26e10 for 1 / 2 / 4 / 8
// slices), at least 8,192 envs per slice
int host_slices(const nig_env* e, bool forced, int want = 4)
{
    if (forced || e->tick_dev) return 1;
    if (const char* v = getenv("NIG_HOST_SLICES")) want = atoi(v);
    if (want > kMaxHostSlices) want = kMaxHostSlices;
    int64_t min_slice = 8192;
    if (const char* v = getenv("NIG_MIN_SLICE")) min_slice = atoll(v) > 0 ? atoll(v) : min_slice;
    const int64_t fit = e->n / min_slice;
    if (want > fit) want = (int)fit;
    return want < 1 ? 1 : want;
}

// one fused launch over envs [i0, i0 + ns) at an explicit tick (validation and e->tick bookkeeping are the callers')
int rollout_range(nig_env* e, const nig_rollout_t* r, cudaStream_t stream, int64_t i0, int64_t ns, uint32_t tick)
{
    RolloutArgs a;
    memset(&a, 0, sizeof a);
    a.state = e->state + i0; a.ep_word = e->ep_word + i0; a.ep_return = e->ep_return + i0; a.n = ns; a.pitch = e->pitch;
    a.env0 = (uint32_t)e->cfg.env_id_offset + (uint32_t)i0; a.tick = tick; a.epoch = e->epoch; a.key = e->key; a.tick_dev = e->tick_dev;
    a.max_steps = e->max_steps; a.auto_reset = e->cfg.auto_reset; a.n_steps = r->n_steps;
    a.actions = r->actions ? r->actions + i0 : nullptr; a.noise = r->noise ? r->noise + i0 : nullptr; a.pp = r->pp;
    a.reward_sum = r->reward_sum ? r->reward_sum + i0 : nullptr;
    a.viol_count = r->viol_count ? r->viol_count + i0 : nullptr;
    a.done_count = r->done_count ? r->done_count + i0 : nullptr;
    a.accumulate = (r->flags & NIG_ROLLOUT_ACCUMULATE) ? 1 : 0;
    a.pid_state = e->pid_state ? e->pid_state + i0 : nullptr;
    a.extrema = e->extrema;
    a.stats = e->stats; a.cons = e->cons;
    fill_tick(e, a, tick);
    if (e->graph_mode) a.epoch = 0u;
    CUtensorMap map;
    memset(&map, 0, sizeof map);
    const bool tma = r->policy == NIG_POLICY_ACTIONS && (r->flags & NIG_ROLLOUT_USE_TMA) && !e->track_extrema && i0 == 0 && ns == e->n;
    int rc;
    if (tma && (rc = make_action_map(e, r->actions, r->n_steps, &map)) != NIG_OK) return rc;
    RolloutLaunch cfg;
    cfg.policy = r->policy; cfg.cons = e->cons.is_default; cfg.tma = tma; cfg.tf_noise = r->noise != nullptr;
    // one-warp CTAs for small reactor launches (a slice, or a whole population of <= 16,384 envs): finer-grained placement
    // on the SMs, measured 7.82 / 7.93 / 7.98e10 env-steps/s for 128 / 64 / 32 threads per CTA at 8 slices of 8,192 envs
    cfg.block = e->rollout_block ? e->rollout_block : (e->kind == NIG_ENV_CHEMICAL_REACTOR && ns <= 16384 ? 32 : 128);
    cfg.extrema = e->track_extrema;
    // two envs per thread + packed f32x2 arithmetic: measured +7 .. 8 % from 262,144 envs per launch up, -11 % at 65,536
    // (half the warps: profiles/r02_e_pair_f32x2_ab.txt); NIG_ROLLOUT_PAIR = 0 / 1 forces it off / on
    cfg.pair = (e->rollout_pair == 1 || (e->rollout_pair < 0 && ns >= 131072)) && e->kind == NIG_ENV_CHEMICAL_REACTOR &&
               e->cfg.auto_reset != 0 && (i0 % 2) == 0;
    // PowerGrid-v0: the dedicated lean kernel (NIG_GRID_FAST = 0 falls back to the generic one)
    cfg.grid_fast = e->grid_fast && e->kind == NIG_ENV_POWER_GRID && e->cfg.auto_reset != 0;
    cfg.mlp = e->mlp;
    cfg.mlp.extrema = e->track_extrema ? 1 : 0;
    e->launches++;
    const int64_t extent = (ns + 127) / 128 * 128;          // launch extent; <= the rows' pitch because slices start at multiples of 128
    NIG_CUDA(nig::launch_rollout(e->kind, cfg, extent, a, map, stream));
    return NIG_OK;
}

// T steps of every env as ceil(T / K) fused launches per env slice, slice q on e->slice_stream[q] (already forked by
// the caller). Launches are issued chunk-major so that every stream always has work queued; per-env outputs accumulate
// from the second chunk on (or from the first, with NIG_ROLLOUT_ACCUMULATE in proto.flags).
int sliced_launches(nig_env* e, const nig_rollout_t& proto, int32_t T, int32_t K, int slices, int64_t per)
{
    const uint32_t tick0 = e->tick;
    int32_t done = 0;
    for (int c = 0; done < T; ++c) {
        nig_rollout_t d = proto;
        d.n_steps = T - done < K ? T - done : K;
        if (c > 0) d.flags |= NIG_ROLLOUT_ACCUMULATE;
        if (c == 0) if (int rc = rollout_checks(e, &d)) return rc;
        for (int q = 0; q < slices; ++q) {
            const int64_t i0 = q * per, ns = std::min<int64_t>(per, e->n - i0);
            if (ns <= 0) continue;
            if (int rc = rollout_range(e, &d, e->slice_stream[q], i0, ns, tick0 + (uint32_t)done)) return rc;
        }
        done += d.n_steps;
    }
    e->tick = tick0 + (uint32_t)T;
    return NIG_OK;
}

int prepare_slices(nig_env* e, int slices);
// create the slice streams / events on first use and make slices 0..slices-1 wait for the work queued on `st`
int fork_slices(nig_env* e, int slices, cudaStream_t st)
{
    if (int rc = prepare_slices(e, slices)) return rc;
    NIG_CUDA(cudaEventRecord(e->slice_begin, st));
    for (int k = 0; k < slices; ++k) NIG_CUDA(cudaStreamWaitEvent(e->slice_stream[k], e->slice_begin, 0));
    return NIG_OK;
}

// the caller's stream waits for everything queued on the slice streams (also on the error paths: whatever a failed call
// did launch must not be left running unordered with the caller's next work)
int join_slices(nig_env* e, int slices, cudaStream_t st)
{
    for (int k = 0; k < slices; ++k) {
        NIG_CUDA(cudaEventRecord(e->slice_done[k], e->slice_stream[k]));
        NIG_CUDA(cudaStreamWaitEvent(st, e->slice_done[k], 0));
    }
    return NIG_OK;
}

// create the slice streams / events (outside any capture)
int prepare_slices(nig_env* e, int slices)
{
    if (!e->slice_begin) NIG_CUDA(cudaEventCreateWithFlags(&e->slice_begin, cudaEventDisableTiming));
    for (int k = 0; k < slices; ++k) {
        if (!e->slice_stream[k]) NIG_CUDA(cudaStreamCreateWithFlags(&e->slice_stream[k], cudaStreamNonBlocking));
        if (!e->slice_done[k]) NIG_CUDA(cudaEventCreateWithFlags(&e->slice_done[k], cudaEventDisableTiming));
    }
    return NIG_OK;
}

static bool is_pinned_or_null(const void* p)
{
    if (!p) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost) return true;
    (void)cudaGetLastError();
    return false;
}
bool host_buffers_pinned(const nig_rollout_host_t* r)
{
    return is_pinned_or_null(r->init_states) && is_pinned_or_null(r->reward_sum) && is_pinned_or_null(r->viol_count) &&
           is_pinned_or_null(r->done_count) && is_pinned_or_null(r->final_obs);
}

// nig_rollout_host over env slices, enqueued on st and the slice streams (forked from / joined back to st): slice s copies its
// initial states in, resets, runs its ceil(T / K) fused launches and copies its results out independently of the others, so
// the PCIe copies overlap the stepping and a slice's next launch fills the SMs another slice's tail leaves idle. Trajectories
// do not depend on the slicing (random streams are keyed by global env id and tick). Capturable (no synchronisation inside).
// device-side alias of a page-locked host array a kernel may read / write directly (16-byte aligned), or null
template <class T>
T* mapped_alias(T* host)
{
    if (!host || ((uintptr_t)host & 15u) != 0) return nullptr;
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, (void*)host, 0) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }
    return ((uintptr_t)d & 15u) == 0 ? (T*)d : nullptr;
}

bool host_direct_ok(const nig_env* e, const nig_rollout_host_t* r)
{
    return e->host_direct != 0 && e->S % 4 == 0 && (!r->init_states || mapped_alias(r->init_states)) && (!r->final_obs || mapped_alias(r->final_obs)) &&
           (!r->reward_sum || mapped_alias(r->reward_sum)) && (!r->viol_count || mapped_alias(r->viol_count)) &&
           (!r->done_count || mapped_alias(r->done_count));
}

int enqueue_sliced_host(nig_env* e, const nig_rollout_host_t* r, int slices, int64_t per, int32_t T, int32_t K, bool reset, cudaStream_t st)
{
    const int64_t n = e->n;
    int rc;
    // direct mode (NIG_HOST_DIRECT, default on): no staging copies -- the ingest / export kernels of a slice touch the caller's
    // page-locked arrays themselves. Needs every supplied array mapped into the device's address space; else the copy path.
    const float* m_init = mapped_alias(r->init_states);
    float* m_obs = mapped_alias(r->final_obs);
    float* m_rew = mapped_alias(r->reward_sum);
    int32_t* m_vi = mapped_alias(r->viol_count);
    int32_t* m_dn = mapped_alias(r->done_count);
    const bool direct = host_direct_ok(e, r);
    // which side goes direct: bit 0 of NIG_HOST_DIRECT = ingest, bit 1 = export, each up to a size (megabytes per call) above
    // which the copy engines' DMA wins: SM-issued PCIe READS are 32..128-byte requests with a bounded number in flight
    // (measured: direct ingest wins at 3 MB, loses from 6 MB up), posted WRITES stay level with DMA up to ~32 MB
    // (tools/host_direct_check.py, profiles/r02_h_host_direct_ab.txt). NIG_HOST_DIRECT_MAX_MB="in,out" overrides.
    const double mb_in = r->init_states ? (double)n * e->S * 4 / 1e6 : 0.0;
    const double mb_out = ((r->final_obs ? (double)n * e->S * 4 : 0.0) + (r->reward_sum ? n * 4.0 : 0.0) + (r->viol_count ? n * 4.0 : 0.0) +
                           (r->done_count ? n * 4.0 : 0.0)) / 1e6;
    const bool direct_in = direct && (e->host_direct & 1) && mb_in <= e->host_direct_max_mb[0];
    const bool direct_out = direct && (e->host_direct & 2) && mb_out <= e->host_direct_max_mb[1];
    if ((rc = fork_slices(e, slices, st)) != NIG_OK) return rc;
    for (int k = 0; k < slices; ++k) {
        const int64_t i0 = k * per, ns = std::min<int64_t>(per, n - i0);
        if (ns <= 0) continue;
        cudaStream_t ss = e->slice_stream[k];
        if (direct_in && r->init_states) {
            HostIoArgs a;
            memset(&a, 0, sizeof a);
            a.state = e->state + i0; a.ep_word = e->ep_word + i0; a.ep_return = e->ep_return + i0; a.n = ns; a.pitch = e->pitch; a.S = e->S;
            a.in_aos = m_init + i0 * e->S;
            e->launches++;
            const cudaError_t ce = nig::launch_host_ingest(a, ss);
            if (ce != cudaSuccess) { join_slices(e, slices, st); return fail(NIG_ERR_CUDA, "host_ingest_kernel: %s", cudaGetErrorString(ce)); }
            continue;
        }
        if (r->init_states)
            NIG_CUDA(cudaMemcpyAsync(e->h_reset + i0 * e->S, r->init_states + i0 * e->S, (size_t)ns * e->S * sizeof(float), cudaMemcpyHostToDevice, ss));
        if (reset && (rc = reset_range(e, r->init_states ? e->h_reset : nullptr, i0, ns, e->epoch, ss)) != NIG_OK) { join_slices(e, slices, st); return rc; }
    }
    nig_rollout_t d;
    memset(&d, 0, sizeof d);
    d.policy = r->policy; d.pp = r->pp;
    d.reward_sum = r->reward_sum ? e->h_reward : nullptr;
    d.viol_count = r->viol_count ? e->h_i32a : nullptr;
    d.done_count = r->done_count ? e->h_i32b : nullptr;
    if ((rc = sliced_launches(e, d, T, K, slices, per)) != NIG_OK) { join_slices(e, slices, st); return rc; }
    for (int k = 0; k < slices; ++k) {
        const int64_t i0 = k * per, ns = std::min<int64_t>(per, n - i0);
        if (ns <= 0) continue;
        cudaStream_t ss = e->slice_stream[k];
        if (direct_out) {
            if (!r->final_obs && !r->reward_sum && !r->viol_count && !r->done_count) continue;
            HostIoArgs a;
            memset(&a, 0, sizeof a);
            a.state = e->state + i0; a.ep_word = e->ep_word + i0; a.ep_return = e->ep_return + i0; a.n = ns; a.pitch = e->pitch; a.S = e->S;
            a.out_aos = m_obs ? m_obs + i0 * e->S : nullptr;
            if (m_rew) { a.d_reward = e->h_reward + i0; a.h_reward = m_rew + i0; }
            if (m_vi) { a.d_viol = e->h_i32a + i0; a.h_viol = m_vi + i0; }
            if (m_dn) { a.d_done = e->h_i32b + i0; a.h_done = m_dn + i0; }
            e->launches++;
            const cudaError_t ce = nig::launch_host_export(a, ss);
            if (ce != cudaSuccess) { join_slices(e, slices, st); return fail(NIG_ERR_CUDA, "host_export_kernel: %s", cudaGetErrorString(ce)); }
            continue;
        }
        if (r->final_obs) {
            if ((rc = state_to_aos_range(e, e->h_obs, i0, ns, ss)) != NIG_OK) { join_slices(e, slices, st); return rc; }
            NIG_CUDA(cudaMemcpyAsync(r->final_obs + i0 * e->S, e->h_obs + i0 * e->S, (size_t)ns * e->S * sizeof(float), cudaMemcpyDeviceToHost, ss));
        }
        if (r->reward_sum) NIG_CUDA(cudaMemcpyAsync(r->reward_sum + i0, e->h_reward + i0, (size_t)ns * sizeof(float), cudaMemcpyDeviceToHost, ss));
        if (r->viol_count) NIG_CUDA(cudaMemcpyAsync(r->viol_count + i0, e->h_i32a + i0, (size_t)ns * sizeof(int32_t), cudaMemcpyDeviceToHost, ss));
        if (r->done_count) NIG_CUDA(cudaMemcpyAsync(r->done_count + i0, e->h_i32b + i0, (size_t)ns * sizeof(int32_t), cudaMemcpyDeviceToHost, ss));
    }
    return join_slices(e, slices, st);
}

inline int64_t slice_size(int64_t n, int slices) { return ((n + slices - 1) / slices + 127) / 128 * 128; }

} // namespace

// =====================================================================================================
extern "C" {

int nig_abi_version(void) { return NIG_ABI_VERSION; }
const char* nig_last_error(void) { return g_err; }

int nig_device_count(int* count)
{
    if (!count) return fail(NIG_ERR_INVALID, "null count");
    int n = 0;
    const cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { *count = 0; (void)cudaGetLastError(); return fail(NIG_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
    *count = n;
    return NIG_OK;
}

int nig_env_spec(int kind, nig_env_spec_t* out)
{
    if (!out) return fail(NIG_ERR_INVALID, "null spec");
    if (kind < 0 || kind > 2) return fail(NIG_ERR_INVALID, "unknown env kind %d", kind);
    memset(out, 0, sizeof *out);
    out->state_dim = kS[kind];
    out->action_dim = kA[kind];
    out->noise_dim = kNZ[kind];
    out->max_episode_steps = kMaxSteps[kind];
    out->n_constraints = 3;
    builtin_constraints(kind, out->constraints);
    return NIG_OK;
}

int nig_create(const nig_config_t* cfg, nig_env_t** out)
{
    if (!cfg || !out) return fail(NIG_ERR_INVALID, "null config or output pointer");
    *out = nullptr;
    if (cfg->env_kind < 0 || cfg->env_kind > 2) return fail(NIG_ERR_INVALID, "unknown env kind %d", cfg->env_kind);
    if (cfg->n_envs <= 0) return fail(NIG_ERR_INVALID, "n_envs must be positive (got %lld)", (long long)cfg->n_envs);
    if (cfg->n_envs > (1LL << 31)) return fail(NIG_ERR_INVALID, "n_envs %lld exceeds 2^31", (long long)cfg->n_envs);
    if (cfg->max_episode_steps < 0 || cfg->max_episode_steps > 65535) return fail(NIG_ERR_INVALID, "max_episode_steps %d outside [0, 65535]", cfg->max_episode_steps);
    if (cfg->env_id_offset < 0 || cfg->env_id_offset > (1LL << 32) - cfg->n_envs)      // global env ids are 32-bit
        return fail(NIG_ERR_INVALID, "env ids env_id_offset %lld + [0, %lld) outside [0, 2^32)", (long long)cfg->env_id_offset, (long long)cfg->n_envs);
    int ndev = 0;
    if (nig_device_count(&ndev) != NIG_OK || ndev == 0) {
        char why[256];
        snprintf(why, sizeof why, "%.255s", ndev == 0 && g_err[0] ? g_err : "device count is 0");
        return fail(NIG_ERR_NO_DEVICE, "no CUDA device visible (%s): libnig_b200 has no CPU fallback", why);
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(NIG_ERR_INVALID, "device %d outside [0, %d)", cfg->device, ndev);
    cudaDeviceProp prop;
    NIG_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10) return fail(NIG_ERR_NO_DEVICE, "device %d is sm_%d%d; this library carries sm_100a code only", cfg->device, prop.major, prop.minor);
    DeviceGuard guard(cfg->device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", cfg->device);

    nig_env* e = new (std::nothrow) nig_env();
    if (!e) return fail(NIG_ERR_INVALID, "out of host memory");
    memset(e, 0, sizeof *e);
    e->track_returns = true;
    e->track_step_stats = true;
    e->cfg = *cfg;
    e->kind = cfg->env_kind;
    e->S = kS[e->kind]; e->A = kA[e->kind]; e->NZ = kNZ[e->kind];
    e->n = cfg->n_envs;
    e->pitch = (e->n + 127) / 128 * 128;
    e->max_steps = cfg->max_episode_steps ? cfg->max_episode_steps : kMaxSteps[e->kind];
    e->key = RngKey{(uint32_t)cfg->seed, (uint32_t)(cfg->seed >> 32)};
    if (const char* v = getenv("NIG_STEP_VEC")) e->step_vec = atoi(v);
    if (const char* v = getenv("NIG_ROLLOUT_BLOCK")) e->rollout_block = atoi(v);
    e->rollout_pair = -1;            // auto
    if (const char* v = getenv("NIG_ROLLOUT_PAIR")) e->rollout_pair = atoi(v);
    e->grid_fast = true;
    if (const char* v = getenv("NIG_GRID_FAST")) e->grid_fast = atoi(v) != 0;
    e->host_graph_enable = 1;
    if (const char* v = getenv("NIG_HOST_GRAPH")) e->host_graph_enable = atoi(v);
    e->host_direct = 3;
    if (const char* v = getenv("NIG_HOST_DIRECT")) e->host_direct = atoi(v);
    e->host_direct_max_mb[0] = 4.0; e->host_direct_max_mb[1] = 48.0;
    if (const char* v = getenv("NIG_HOST_DIRECT_MAX_MB")) {
        double a = 0, b = 0;
        const int got = sscanf(v, "%lf,%lf", &a, &b);
        if (got >= 1) e->host_direct_max_mb[0] = e->host_direct_max_mb[1] = a;
        if (got == 2) e->host_direct_max_mb[1] = b;
    }
    e->steps_graph_enable = 1;
    if (const char* v = getenv("NIG_STEPS_GRAPH")) e->steps_graph_enable = atoi(v);
    e->step_pipe = 1;
    if (const char* v = getenv("NIG_STEP_PIPE")) e->step_pipe = atoi(v);
    e->zero_copy = 1;
    if (const char* v = getenv("NIG_ZERO_COPY")) e->zero_copy = atoi(v);
    if (e->rollout_block != 0 && e->rollout_block != 32 && e->rollout_block != 64 && e->rollout_block != 128) e->rollout_block = 0;
    nig_constraint_t def[3];
    const nig_constraint_t* c = cfg->constraints;
    int nc = cfg->n_constraints;
    if (nc < 0) { builtin_constraints(e->kind, def); c = def; nc = 3; }
    int rc = validate_constraints(e->kind, c, nc);
    if (rc == NIG_OK) rc = dev_alloc(&e->cons_masks, (size_t)NIG_MAX_CONSTRAINTS * kConsMaskRow);
    if (rc == NIG_OK) {
        rc = set_cons(e, c, nc);
    }
    if (rc == NIG_OK) {
        rc = dev_alloc(&e->state, (size_t)e->S * e->pitch);
    }
    if (rc == NIG_OK) rc = dev_alloc(&e->ep_word, (size_t)e->pitch);
    if (rc == NIG_OK) rc = dev_alloc(&e->ep_return, (size_t)e->pitch);
    if (rc == NIG_OK) rc = dev_alloc(&e->stats, (size_t)NIG_STATS_SLOTS);
    if (rc == NIG_OK) rc = dev_alloc(&e->stats_shards, (size_t)nig::kStatsShards * NIG_STATS_SLOTS);
    if (rc == NIG_OK) rc = dev_alloc(&e->extrema, (size_t)2);
    if (rc == NIG_OK && cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess)
        rc = fail(NIG_ERR_CUDA, "cudaStreamCreate failed");

    if (rc != NIG_OK) { nig_destroy(e); return rc; }
    *out = e;
    return NIG_OK;
}

int nig_destroy(nig_env_t* e)
{
    if (!e) return NIG_OK;
    DeviceGuard guard(e->cfg.device);
    if (e->host_graph) cudaGraphExecDestroy(e->host_graph);
    if (e->steps_graph) cudaGraphExecDestroy(e->steps_graph);
    if (e->h_tickbase) cudaFreeHost(e->h_tickbase);
    if (e->h_stats_pinned) cudaFreeHost(e->h_stats_pinned);
    cudaFree(e->d_tickbase);
    cudaFree(e->state); cudaFree(e->ep_word); cudaFree(e->ep_return); cudaFree(e->stats); cudaFree(e->stats_shards);
    cudaFree(e->h_actions); cudaFree(e->h_noise); cudaFree(e->h_reset); cudaFree(e->h_obs); cudaFree(e->h_next_obs);
    cudaFree(e->h_reward); cudaFree(e->h_hostmask); cudaFree(e->h_flags); cudaFree(e->h_viol); cudaFree(e->h_mask);
    cudaFree(e->h_terminated); cudaFree(e->h_truncated);
    cudaFree(e->h_i32a); cudaFree(e->h_i32b); cudaFree(e->pid_state); cudaFree(e->tick_dev); cudaFree(e->cons_masks); cudaFree(e->extrema); cudaFree(e->d_len); cudaFree(e->d_off); cudaFree(e->d_total);
    cudaFree(e->mlp_blob);
    for (int b = 0; b < 2; ++b) {
        cudaFree(e->r_act[b]); cudaFree(e->r_nz[b]);
        if (e->r_ev_copy[b]) cudaEventDestroy(e->r_ev_copy[b]);
        if (e->r_ev_done[b]) cudaEventDestroy(e->r_ev_done[b]);
    }
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    for (int k = 0; k < kMaxHostSlices; ++k) {
        if (e->slice_stream[k]) cudaStreamDestroy(e->slice_stream[k]);
        if (e->slice_done[k]) cudaEventDestroy(e->slice_done[k]);
    }
    if (e->slice_begin) cudaEventDestroy(e->slice_begin);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return NIG_OK;
}

int64_t nig_pitch(const nig_env_t* e) { return e ? e->pitch : 0; }
int64_t nig_num_envs(const nig_env_t* e) { return e ? e->n : 0; }
int64_t nig_launch_count(const nig_env_t* e) { return e ? e->launches : 0; }

int nig_set_constraints(nig_env_t* e, const nig_constraint_t* cons, int32_t n)
{
    if (e) e->config_version++;
    if (!e) return fail(NIG_ERR_INVALID, "null env handle");
    if (n > 0 && !cons) return fail(NIG_ERR_INVALID, "null constraint array");
    const int rc = validate_constraints(e->kind, cons, n);
    if (rc != NIG_OK) return rc;
    DeviceGuard guard(e->cfg.device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", e->cfg.device);
    return set_cons(e, cons, n);
}

int nig_reset(nig_env_t* e, const uint8_t* mask, const float* init_states, int32_t layout, void* stream)
{
    NIG_CHECK_ENV(e);
    e->epoch += 1;     // explicit resets draw with a fresh epoch; auto-resets reuse the current one
    ResetArgs a{e->state, e->ep_word, e->ep_return, e->n, e->pitch, (uint32_t)e->cfg.env_id_offset, e->tick, e->epoch, e->tick_dev,
                e->key, mask, init_states, layout == NIG_LAYOUT_AOS ? 1 : 0};
    fill_tick(e, a, e->tick);
    e->launches++;
    note_device_work(e, (cudaStream_t)stream);
    NIG_CUDA(nig::launch_reset(e->kind, a, (cudaStream_t)stream));
    return NIG_OK;
}

int nig_reset_host(nig_env_t* e, const uint8_t* mask, const float* init_states_aos, float* obs_aos_out)
{
    NIG_CHECK_ENV(e);
    if (int hrc = host_entry(e)) return hrc;
    int rc;
    const uint8_t* dmask = nullptr;
    const float* dinit = nullptr;
    if (mask) {
        if ((rc = dev_alloc(&e->h_mask, (size_t)e->pitch)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_mask, mask, (size_t)e->n, cudaMemcpyHostToDevice, e->stream));
        dmask = e->h_mask;
    }
    if (init_states_aos) {
        if ((rc = dev_alloc(&e->h_reset, (size_t)e->pitch * e->S)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_reset, init_states_aos, (size_t)e->n * e->S * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        dinit = e->h_reset;
    }
    if ((rc = nig_reset(e, dmask, dinit, NIG_LAYOUT_AOS, e->stream)) != NIG_OK) return rc;
    if (obs_aos_out) {
        if ((rc = dev_alloc(&e->h_obs, (size_t)e->pitch * e->S)) != NIG_OK) return rc;
        if ((rc = state_io(e, e->h_obs, NIG_LAYOUT_AOS, nullptr, nullptr, nullptr, true, e->stream)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(obs_aos_out, e->h_obs, (size_t)e->n * e->S * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    }
    NIG_CUDA(cudaStreamSynchronize(e->stream));
    return NIG_OK;
}

int nig_step(nig_env_t* e, const nig_step_io_t* io, void* stream)
{
    NIG_CHECK_ENV(e);
    if (!io || !io->actions) return fail(NIG_ERR_INVALID, "nig_step: null io or actions");
    if (io->noise && e->NZ == 0) return fail(NIG_ERR_INVALID, "nig_step: env kind %d has no process noise", e->kind);
    StepArgs a;
    memset(&a, 0, sizeof a);
    a.state = e->state; a.ep_word = e->ep_word; a.n = e->n; a.pitch = e->pitch;
    a.ep_return = e->track_returns ? e->ep_return : nullptr;
    a.env0 = (uint32_t)e->cfg.env_id_offset; a.tick = e->tick; a.epoch = e->epoch; a.key = e->key; a.tick_dev = e->tick_dev;
    a.max_steps = e->max_steps; a.auto_reset = e->cfg.auto_reset;
    a.actions = io->actions; a.noise = io->noise; a.reset_states = io->reset_states; a.hostmask = io->hostmask;
    a.obs = io->obs; a.next_obs = io->next_obs; a.reward = io->reward; a.flags = io->flags; a.viol_mask = io->viol_mask;
    a.terminated = io->terminated; a.truncated = io->truncated;
    a.action_aos = io->action_layout == NIG_LAYOUT_AOS; a.aux_aos = io->aux_layout == NIG_LAYOUT_AOS;
    a.stats = e->track_step_stats ? e->stats : nullptr; a.stats_shards = e->track_step_stats ? e->stats_shards : nullptr; a.cons = e->cons;
    e->shards_dirty = true;
    fill_tick(e, a, e->tick);
    const int rc = launch_step(e, a, (cudaStream_t)stream);
    if (rc == NIG_OK) e->tick += 1;
    return rc;
}

// Small populations (the single-env gym API above all) are pure latency: one H2D, one launch, four D2H copies and a
// synchronise cost ~35 us for 12 bytes in and ~110 bytes out. When every host array of the call is page-locked
// (nig_host_alloc) the kernel reads and writes them in place over PCIe through their device aliases (unified
// addressing): one launch + one synchronise. Returns true and sets *dev when `host` is such a buffer.
static bool device_alias(const void* host, void** dev)
{
    // queried on every call (about half a microsecond per pointer): a cached answer could outlive the allocation
    cudaPointerAttributes at;
    *dev = nullptr;
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost) *dev = at.devicePointer;
    else (void)cudaGetLastError();
    return *dev != nullptr;
}

// in place on the caller's page-locked arrays up to this population: measured 62 -> 43 us per call at 4,096 envs, 93 -> 70 us at
// 16,384, 203 -> 188 us at 65,536 (one launch, no copy nodes; the AoS rows leave through the warp-cooperative store)
constexpr int64_t kZeroCopyMaxEnvsDefault = 131072;
inline int64_t zero_copy_max_envs()
{
    static const int64_t v = [] { const char* s = getenv("NIG_ZERO_COPY_MAX_ENVS"); return s && atoll(s) > 0 ? atoll(s) : kZeroCopyMaxEnvsDefault; }();
    return v;
}

int nig_step_host(nig_env_t* e, const nig_step_io_t* io)
{
    NIG_CHECK_ENV(e);
    if (int hrc = host_entry(e)) return hrc;
    if (!io || !io->actions) return fail(NIG_ERR_INVALID, "nig_step_host: null io or actions");
    if (io->noise && e->NZ == 0) return fail(NIG_ERR_INVALID, "nig_step_host: env kind %d has no process noise", e->kind);
    int rc;
    if (e->n <= zero_copy_max_envs() && e->zero_copy) {
        const void* hp[11] = {io->actions, io->noise, io->reset_states, io->hostmask, io->obs, io->next_obs, io->reward,
                              io->flags, io->viol_mask, io->terminated, io->truncated};
        void* dp[11];
        bool all = true;
        for (int k = 0; k < 11 && all; ++k) {
            dp[k] = nullptr;
            if (hp[k]) all = device_alias(hp[k], &dp[k]);
        }
        if (all) {
            nig_step_io_t z;
            memset(&z, 0, sizeof z);
            z.actions = (const float*)dp[0]; z.noise = (const float*)dp[1]; z.reset_states = (const float*)dp[2];
            z.hostmask = (const uint8_t*)dp[3]; z.obs = (float*)dp[4]; z.next_obs = (float*)dp[5]; z.reward = (float*)dp[6];
            z.flags = (uint8_t*)dp[7]; z.viol_mask = (uint8_t*)dp[8]; z.terminated = (uint8_t*)dp[9]; z.truncated = (uint8_t*)dp[10];
            z.action_layout = NIG_LAYOUT_AOS; z.aux_layout = NIG_LAYOUT_AOS;
            if ((rc = nig_step(e, &z, e->stream)) != NIG_OK) return rc;
            NIG_CUDA(cudaStreamSynchronize(e->stream));
            return NIG_OK;
        }
    }
    const size_t n = (size_t)e->n, cap = (size_t)e->pitch;
    nig_step_io_t d;
    memset(&d, 0, sizeof d);
    d.action_layout = NIG_LAYOUT_AOS; d.aux_layout = NIG_LAYOUT_AOS;
    cudaStream_t st = e->stream;
    if ((rc = dev_alloc(&e->h_actions, cap * e->A)) != NIG_OK) return rc;
    NIG_CUDA(cudaMemcpyAsync(e->h_actions, io->actions, n * e->A * sizeof(float), cudaMemcpyHostToDevice, st));
    d.actions = e->h_actions;
    if (io->noise) {
        if ((rc = dev_alloc(&e->h_noise, cap * e->NZ)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_noise, io->noise, n * e->NZ * sizeof(float), cudaMemcpyHostToDevice, st));
        d.noise = e->h_noise;
    }
    if (io->reset_states) {
        if ((rc = dev_alloc(&e->h_reset, cap * e->S)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_reset, io->reset_states, n * e->S * sizeof(float), cudaMemcpyHostToDevice, st));
        d.reset_states = e->h_reset;
    }
    if (io->hostmask) {
        if ((rc = dev_alloc(&e->h_hostmask, cap)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_hostmask, io->hostmask, n, cudaMemcpyHostToDevice, st));
        d.hostmask = e->h_hostmask;
    }
    if (io->obs) { if ((rc = dev_alloc(&e->h_obs, cap * e->S)) != NIG_OK) return rc; d.obs = e->h_obs; }
    if (io->next_obs) { if ((rc = dev_alloc(&e->h_next_obs, cap * e->S)) != NIG_OK) return rc; d.next_obs = e->h_next_obs; }
    if (io->reward) { if ((rc = dev_alloc(&e->h_reward, cap)) != NIG_OK) return rc; d.reward = e->h_reward; }
    if (io->flags) { if ((rc = dev_alloc(&e->h_flags, cap)) != NIG_OK) return rc; d.flags = e->h_flags; }
    if (io->viol_mask) { if ((rc = dev_alloc(&e->h_viol, cap)) != NIG_OK) return rc; d.viol_mask = e->h_viol; }
    if (io->terminated) { if ((rc = dev_alloc(&e->h_terminated, cap)) != NIG_OK) return rc; d.terminated = e->h_terminated; }
    if (io->truncated) { if ((rc = dev_alloc(&e->h_truncated, cap)) != NIG_OK) return rc; d.truncated = e->h_truncated; }
    if ((rc = nig_step(e, &d, st)) != NIG_OK) return rc;
    if (io->obs) NIG_CUDA(cudaMemcpyAsync(io->obs, e->h_obs, n * e->S * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->next_obs) NIG_CUDA(cudaMemcpyAsync(io->next_obs, e->h_next_obs, n * e->S * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->reward) NIG_CUDA(cudaMemcpyAsync(io->reward, e->h_reward, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (io->flags) NIG_CUDA(cudaMemcpyAsync(io->flags, e->h_flags, n, cudaMemcpyDeviceToHost, st));
    if (io->viol_mask) NIG_CUDA(cudaMemcpyAsync(io->viol_mask, e->h_viol, n, cudaMemcpyDeviceToHost, st));
    if (io->terminated) NIG_CUDA(cudaMemcpyAsync(io->terminated, e->h_terminated, n, cudaMemcpyDeviceToHost, st));
    if (io->truncated) NIG_CUDA(cudaMemcpyAsync(io->truncated, e->h_truncated, n, cudaMemcpyDeviceToHost, st));
    NIG_CUDA(cudaStreamSynchronize(st));
    return NIG_OK;
}

int nig_rollout(nig_env_t* e, const nig_rollout_t* r, void* stream)
{
    NIG_CHECK_ENV(e);
    if (int crc = rollout_checks(e, r)) return crc;
    note_device_work(e, (cudaStream_t)stream);
    if (int rc = rollout_range(e, r, (cudaStream_t)stream, 0, e->n, e->tick)) return rc;
    e->tick += (uint32_t)r->n_steps;
    return NIG_OK;
}

int nig_rollout_steps(nig_env_t* e, const nig_rollout_t* r, int32_t total_steps, void* stream)
{
    NIG_CHECK_ENV(e);
    if (!r) return fail(NIG_ERR_INVALID, "nig_rollout_steps: null descriptor");
    if (total_steps <= 0 || r->n_steps <= 0) return fail(NIG_ERR_INVALID, "nig_rollout_steps: total_steps and n_steps must be positive");
    if (r->n_steps > NIG_MAX_LAUNCH_STEPS)
        return fail(NIG_ERR_INVALID, "nig_rollout_steps: n_steps %d exceeds NIG_MAX_LAUNCH_STEPS = %d", r->n_steps, NIG_MAX_LAUNCH_STEPS);
    if (r->policy == NIG_POLICY_ACTIONS) return fail(NIG_ERR_UNSUPPORTED, "nig_rollout_steps: in-kernel policies only (teacher-forced actions: nig_rollout per chunk)");
    cudaStream_t st = (cudaStream_t)stream;
    note_device_work(e, st);
    const int slices = host_slices(e, false, 8);
    if (slices <= 1) {                       // small population / device tick: plain launch sequence on the caller's stream
        int32_t done = 0;
        for (int c = 0; done < total_steps; ++c) {
            nig_rollout_t d = *r;
            d.n_steps = total_steps - done < r->n_steps ? total_steps - done : r->n_steps;
            if (c > 0) d.flags |= NIG_ROLLOUT_ACCUMULATE;
            if (c == 0) if (int rc = rollout_checks(e, &d)) return rc;
            if (int rc = rollout_range(e, &d, st, 0, e->n, e->tick)) return rc;
            e->tick += (uint32_t)d.n_steps;
            done += d.n_steps;
        }
        return NIG_OK;
    }
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { (void)cudaGetLastError(); cap = cudaStreamCaptureStatusActive; }
    if (e->steps_graph_enable != 0 && cap == cudaStreamCaptureStatusNone) {
        // ---- replay of the captured launch sequence (captured on first use and whenever an argument that is baked into the
        // kernel parameters changes: horizon, K, policy, output pointers, constraint set, seed, tracking switches)
        nig_env::StepsGraphKey key;
        memset(&key, 0, sizeof key);
        key.ptr[0] = r->reward_sum; key.ptr[1] = r->viol_count; key.ptr[2] = r->done_count;
        key.T = total_steps; key.K = r->n_steps; key.policy = r->policy; key.flags = (int32_t)r->flags; key.slices = slices;
        key.config = e->config_version; key.pp = r->pp;
        if (!e->d_tickbase) NIG_CUDA(cudaMalloc((void**)&e->d_tickbase, 2 * sizeof(uint32_t)));
        key.launches = e->steps_graph ? e->steps_graph_key.launches : 0;
        const bool hit = e->steps_graph && memcmp(&key, &e->steps_graph_key, sizeof key) == 0;
        if (!hit) {
            // capture only a call pattern that repeats: the first call with a new argument set is enqueued launch by launch and
            // remembered, the second one captures (a one-off horizon or a caller that rotates its output buffers never pays
            // ~1 ms of capture + instantiation per call)
            nig_env::StepsGraphKey cand = key;
            cand.launches = 0;
            const bool repeat = memcmp(&cand, &e->steps_graph_candidate, sizeof cand) == 0;
            e->steps_graph_candidate = cand;
            if (!repeat) goto plain_enqueue;
        }
        if (!hit) {
            if (e->steps_graph) { cudaGraphExecDestroy(e->steps_graph); e->steps_graph = nullptr; }
            if (int rc = prepare_slices(e, slices)) return rc;
            {   // argument checks and lazy allocations (PID controller state) happen before the capture starts
                nig_rollout_t probe = *r;
                probe.n_steps = total_steps < r->n_steps ? total_steps : r->n_steps;
                if (int rc = rollout_checks(e, &probe)) return rc;
            }
            const uint32_t tick0 = e->tick;
            const int64_t launches0 = e->launches;
            cudaGraph_t graph = nullptr;
            NIG_CUDA(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeRelaxed));
            e->graph_mode = true; e->graph_tick0 = tick0;
            int rc = fork_slices(e, slices, e->stream);
            if (rc == NIG_OK) rc = sliced_launches(e, *r, total_steps, r->n_steps, slices, slice_size(e->n, slices));
            const int jrc = join_slices(e, slices, e->stream);
            e->graph_mode = false;
            const cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
            key.launches = e->launches - launches0;
            e->tick = tick0; e->launches = launches0;
            if (rc != NIG_OK || jrc != NIG_OK) { if (graph) cudaGraphDestroy(graph); return rc ? rc : jrc; }
            if (ce != cudaSuccess) return fail(NIG_ERR_CUDA, "nig_rollout_steps: cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
            const cudaError_t ci = cudaGraphInstantiate(&e->steps_graph, graph, 0);
            cudaGraphDestroy(graph);
            if (ci != cudaSuccess) { e->steps_graph = nullptr; return fail(NIG_ERR_CUDA, "nig_rollout_steps: cudaGraphInstantiate failed: %s", cudaGetErrorString(ci)); }
            e->steps_graph_key = key;
        }
        NIG_CUDA(nig::launch_set_ticks(e->d_tickbase, e->tick, e->epoch, st));
        NIG_CUDA(cudaGraphLaunch(e->steps_graph, st));
        e->tick += (uint32_t)total_steps;
        e->launches += e->steps_graph_key.launches + 1;
        return NIG_OK;
    }
plain_enqueue:
    if (int rc = fork_slices(e, slices, st)) return rc;
    const int rc = sliced_launches(e, *r, total_steps, r->n_steps, slices, slice_size(e->n, slices));
    const int jrc = join_slices(e, slices, st);
    return rc ? rc : jrc;
}

} // extern "C"

// ---- NIG_POLICY_MLP ------------------------------------------------------------------------------------------------------
namespace {
uint16_t bf16_rne(float x)
{
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40u);      // NaN stays a (quiet) NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
// [n_out][n_in] fp32 (nn.Linear order) -> bf16 [n_rows][k_pad] in the canonical layout of MlpParams, zero-padded
void pack_weight(uint8_t* dst, const float* w, int n_out, int n_in, int n_rows, int k_pad)
{
    for (int n = 0; n < n_rows; ++n)
        for (int k = 0; k < k_pad; ++k) {
            const uint16_t v = (n < n_out && k < n_in) ? bf16_rne(w[(size_t)n * n_in + k]) : (uint16_t)0;
            memcpy(dst + (size_t)(k / 8) * n_rows * 16 + (size_t)n * 16 + (k % 8) * 2, &v, 2);
        }
}
} // namespace

extern "C" {

int nig_set_mlp_policy(nig_env_t* e, const nig_mlp_t* m)
{
    NIG_CHECK_ENV(e);
    if (!m) return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: null network");
    if (m->n_hidden != 1 && m->n_hidden != 2) return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: %d hidden layers (1 or 2 are supported)", m->n_hidden);
    for (int l = 0; l < m->n_hidden; ++l)
        if (m->hidden[l] != 64 && m->hidden[l] != 128 && m->hidden[l] != 256)
            return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: hidden width %d (64, 128 or 256 are supported)", m->hidden[l]);
    if (m->output_activation != NIG_MLP_OUT_IDENTITY && m->output_activation != NIG_MLP_OUT_TANH)
        return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: unknown output activation %d", m->output_activation);
    if (m->in_dim != e->S || m->out_dim != e->A)
        return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: network maps %d -> %d, the env needs %d -> %d", m->in_dim, m->out_dim, e->S, e->A);
    for (int l = 0; l <= m->n_hidden; ++l)
        if (!m->weight[l]) return fail(NIG_ERR_INVALID, "nig_set_mlp_policy: null weight of layer %d", l);
    MlpParams p;
    memset(&p, 0, sizeof p);
    p.layers = m->n_hidden; p.h1 = m->hidden[0]; p.h2 = m->n_hidden == 2 ? m->hidden[1] : m->hidden[0];
    p.out_tanh = m->output_activation == NIG_MLP_OUT_TANH ? 1 : 0;
    const MlpLayout L = mlp_layout(e->S, p);
    p.blob_bytes = L.blob;
    uint8_t* h = (uint8_t*)calloc(L.blob, 1);
    if (!h) return fail(NIG_ERR_INVALID, "out of host memory");
    const int widths[3] = {p.h1, p.layers == 2 ? p.h2 : kMlpOut, kMlpOut};
    const int rows[3] = {p.h1, p.layers == 2 ? p.h2 : kMlpOut, kMlpOut};
    const int ins[3] = {e->S, p.h1, p.h2};
    const uint32_t woff[3] = {L.w1, p.layers == 2 ? L.w2 : L.w3, L.w3};
    const uint32_t boff[3] = {L.b1, p.layers == 2 ? L.b2 : L.b3, L.b3};
    for (int l = 0; l <= p.layers; ++l) {
        const bool last = l == p.layers;
        const int n_out = last ? e->A : widths[l];
        pack_weight(h + woff[l], m->weight[l], n_out, ins[l], rows[l], l == 0 ? L.sp : ins[l]);
        if (m->bias[l]) memcpy(h + boff[l], m->bias[l], (size_t)n_out * sizeof(float));
    }
    float* mean = (float*)(h + L.mean);
    float* istd = (float*)(h + L.istd);
    for (int k = 0; k < L.sp; ++k) {
        mean[k] = (m->obs_mean && k < e->S) ? m->obs_mean[k] : 0.0f;
        istd[k] = (m->obs_inv_std && k < e->S) ? m->obs_inv_std[k] : 1.0f;
    }
    // a rollout still running on any stream keeps reading the old blob: finish it before the buffer is reused or freed
    cudaError_t ce = cudaDeviceSynchronize();
    // from here on the old network is gone, whether or not the upload below succeeds: no launch and no replay of a captured
    // nig_rollout_steps / nig_rollout_host graph (the network is baked into them) may read the buffer until the new one is
    // complete. A failed upload leaves the handle without a network (NIG_POLICY_MLP then fails with NIG_ERR_INVALID).
    e->mlp.blob = nullptr;
    e->config_version++;
    if (e->steps_graph) { cudaGraphExecDestroy(e->steps_graph); e->steps_graph = nullptr; }
    if (e->host_graph) { cudaGraphExecDestroy(e->host_graph); e->host_graph = nullptr; }
    if (ce == cudaSuccess && L.blob > e->mlp_cap) {
        cudaFree(e->mlp_blob);
        e->mlp_blob = nullptr; e->mlp_cap = 0;
        ce = cudaMalloc(&e->mlp_blob, L.blob);
        if (ce == cudaSuccess) e->mlp_cap = L.blob;
    }
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(e->mlp_blob, h, L.blob, cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    free(h);
    if (ce != cudaSuccess) return fail(NIG_ERR_CUDA, "nig_set_mlp_policy: %s", cudaGetErrorString(ce));
    p.blob = e->mlp_blob;
    e->mlp = p;
    return NIG_OK;
}

int nig_selftest_mlp(nig_env_t* e, const float* obs, int64_t n, float* actions)
{
    NIG_CHECK_ENV(e);
    if (!e->mlp.blob) return fail(NIG_ERR_INVALID, "nig_selftest_mlp: no network set (nig_set_mlp_policy)");
    if (n <= 0 || !obs || !actions) return fail(NIG_ERR_INVALID, "nig_selftest_mlp: bad arguments");
    if (int hrc = host_entry(e)) return hrc;
    float *d_obs = nullptr, *d_act = nullptr;
    cudaError_t ce = cudaMalloc((void**)&d_obs, (size_t)n * e->S * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMalloc((void**)&d_act, (size_t)n * e->A * sizeof(float));
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_obs, obs, (size_t)n * e->S * sizeof(float), cudaMemcpyHostToDevice, e->stream);
    if (ce == cudaSuccess) { e->launches++; ce = nig::launch_selftest_mlp(e->kind, e->mlp, d_obs, d_act, n, e->stream); }
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(actions, d_act, (size_t)n * e->A * sizeof(float), cudaMemcpyDeviceToHost, e->stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    cudaFree(d_obs); cudaFree(d_act);
    if (ce != cudaSuccess) return fail(NIG_ERR_CUDA, "nig_selftest_mlp: %s", cudaGetErrorString(ce));
    return NIG_OK;
}

int nig_reset_policy_state(nig_env_t* e, void* stream)
{
    NIG_CHECK_ENV(e);
    if (e->pid_state) NIG_CUDA(cudaMemsetAsync(e->pid_state, 0, (size_t)2 * e->A * e->pitch * sizeof(double), (cudaStream_t)stream));
    return NIG_OK;
}

int nig_rollout_host(nig_env_t* e, const nig_rollout_host_t* r)
{
    NIG_CHECK_ENV(e);
    if (int hrc = host_entry(e)) return hrc;
    if (!r) return fail(NIG_ERR_INVALID, "nig_rollout_host: null descriptor");
    if (r->n_steps <= 0) return fail(NIG_ERR_INVALID, "nig_rollout_host: n_steps must be positive (got %d)", r->n_steps);
    if (r->steps_per_launch < 0) return fail(NIG_ERR_INVALID, "nig_rollout_host: steps_per_launch must be >= 0");
    if (r->policy == NIG_POLICY_ACTIONS && !r->actions) return fail(NIG_ERR_INVALID, "nig_rollout_host: NIG_POLICY_ACTIONS needs actions");
    if (r->noise && r->policy != NIG_POLICY_ACTIONS) return fail(NIG_ERR_UNSUPPORTED, "nig_rollout_host: teacher-forced noise needs NIG_POLICY_ACTIONS");
    if (r->noise && e->NZ == 0) return fail(NIG_ERR_INVALID, "nig_rollout_host: env kind %d has no process noise", e->kind);
    int rc;
    const size_t n = (size_t)e->n, cap = (size_t)e->pitch;
    const int32_t T = r->n_steps;
    const int32_t K = std::min(std::min(r->steps_per_launch > 0 ? r->steps_per_launch : T, T), (int32_t)NIG_MAX_LAUNCH_STEPS);
    cudaStream_t st = e->stream;
    const bool forced = r->policy == NIG_POLICY_ACTIONS;
    if (forced) {
        if (!e->copy_stream) {
            NIG_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
            for (int b = 0; b < 2; ++b) {
                NIG_CUDA(cudaEventCreateWithFlags(&e->r_ev_copy[b], cudaEventDisableTiming));
                NIG_CUDA(cudaEventCreateWithFlags(&e->r_ev_done[b], cudaEventDisableTiming));
            }
        }
        if (K > e->r_cap) {
            NIG_CUDA(cudaDeviceSynchronize());
            for (int b = 0; b < 2; ++b) { cudaFree(e->r_act[b]); cudaFree(e->r_nz[b]); e->r_act[b] = e->r_nz[b] = nullptr; }
            e->r_cap = 0;
            for (int b = 0; b < 2; ++b) {
                NIG_CUDA(cudaMalloc((void**)&e->r_act[b], (size_t)K * e->A * cap * sizeof(float)));
                NIG_CUDA(cudaMemset(e->r_act[b], 0, (size_t)K * e->A * cap * sizeof(float)));
                if (e->NZ > 0) {
                    NIG_CUDA(cudaMalloc((void**)&e->r_nz[b], (size_t)K * e->NZ * cap * sizeof(float)));
                    NIG_CUDA(cudaMemset(e->r_nz[b], 0, (size_t)K * e->NZ * cap * sizeof(float)));
                }
            }
            NIG_CUDA(cudaDeviceSynchronize());      // the zero fills must land before the copies on copy_stream
            e->r_cap = K;
        }
    }
    if (r->reward_sum && (rc = dev_alloc(&e->h_reward, cap)) != NIG_OK) return rc;
    if (r->viol_count && (rc = dev_alloc(&e->h_i32a, cap)) != NIG_OK) return rc;
    if (r->done_count && (rc = dev_alloc(&e->h_i32b, cap)) != NIG_OK) return rc;
    if (r->init_states && (rc = dev_alloc(&e->h_reset, cap * e->S)) != NIG_OK) return rc;
    if (r->final_obs && (rc = dev_alloc(&e->h_obs, cap * e->S)) != NIG_OK) return rc;

    // ---- in-kernel policies on a large population: env slices on their own streams. Slice s copies its initial states in,
    // resets, runs its ceil(T / K) fused launches and copies its results out independently of the others, so the PCIe
    // copies overlap the stepping, and a slice's next launch fills the SMs another slice's tail leaves idle. Trajectories
    // do not depend on the slicing (random streams are keyed by global env id and tick).
    const bool use_graph = e->host_graph_enable != 0 && !forced && !e->tick_dev && host_buffers_pinned(r);
    // copy path: 4 slices (8 measured slower, with and without the graph); direct path (the slices' kernels read / write the
    // mapped host arrays, no copy nodes): 8 slices -- 0.730 ms per 65,536 x 1,000 call against 0.762 with 4 and 0.835 for the
    // copy path (tools/host_path_breakdown.py, profiles/r02_h_host_direct_ab.txt)
    const int slices = host_slices(e, forced, host_direct_ok(e, r) ? 8 : 4);
    if (slices > 1) {
        const int64_t per = slice_size((int64_t)n, slices);
        const bool reset = r->reset_first || r->init_states;
        if (reset) e->epoch += 1;
        if (use_graph) {
            // ---- the whole sliced pipeline as ONE graph launch: captured on first use (and again whenever a buffer address,
            // the horizon, the policy or a baked-in setting changes), replayed afterwards with fresh tick / epoch words
            nig_env::HostGraphKey key;
            memset(&key, 0, sizeof key);
            key.ptr[0] = r->init_states; key.ptr[1] = r->reward_sum; key.ptr[2] = r->viol_count; key.ptr[3] = r->done_count; key.ptr[4] = r->final_obs;
            key.T = T; key.K = K; key.policy = r->policy; key.reset = reset ? 1 : 0; key.slices = slices;
            key.config = e->config_version; key.pp = r->pp;
            if (!e->h_tickbase) NIG_CUDA(cudaHostAlloc((void**)&e->h_tickbase, 2 * sizeof(uint32_t), cudaHostAllocPortable));
            if (!e->d_tickbase) NIG_CUDA(cudaMalloc((void**)&e->d_tickbase, 2 * sizeof(uint32_t)));
            key.launches = e->host_graph ? e->host_graph_key.launches : 0;
            if (!e->host_graph || memcmp(&key, &e->host_graph_key, sizeof key) != 0) {
                if (e->host_graph) { cudaGraphExecDestroy(e->host_graph); e->host_graph = nullptr; }
                if ((rc = prepare_slices(e, slices)) != NIG_OK) return rc;
                {   // argument checks and lazy allocations (PID controller state) happen before the capture starts
                    nig_rollout_t probe;
                    memset(&probe, 0, sizeof probe);
                    probe.policy = r->policy; probe.pp = r->pp; probe.n_steps = K;
                    if ((rc = rollout_checks(e, &probe)) != NIG_OK) return rc;
                }
                const uint32_t tick0 = e->tick;
                const int64_t launches0 = e->launches;
                cudaGraph_t graph = nullptr;
                NIG_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
                e->graph_mode = true; e->graph_tick0 = tick0;
                cudaError_t ce = cudaMemcpyAsync(e->d_tickbase, e->h_tickbase, 2 * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
                rc = ce == cudaSuccess ? enqueue_sliced_host(e, r, slices, per, T, K, reset, st) : fail(NIG_ERR_CUDA, "capturing the tick copy failed: %s", cudaGetErrorString(ce));
                e->graph_mode = false;
                ce = cudaStreamEndCapture(st, &graph);
                key.launches = e->launches - launches0;
                e->tick = tick0; e->launches = launches0;
                if (rc != NIG_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
                if (ce != cudaSuccess) return fail(NIG_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
                ce = cudaGraphInstantiate(&e->host_graph, graph, 0);
                cudaGraphDestroy(graph);
                if (ce != cudaSuccess) { e->host_graph = nullptr; return fail(NIG_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
                e->host_graph_key = key;
            }
            e->h_tickbase[0] = e->tick; e->h_tickbase[1] = e->epoch;
            NIG_CUDA(cudaGraphLaunch(e->host_graph, st));
            e->tick += (uint32_t)T;
            e->launches += e->host_graph_key.launches;
        } else {
            if ((rc = enqueue_sliced_host(e, r, slices, per, T, K, reset, st)) != NIG_OK) return rc;
        }
        // the statistics block lands in a page-locked word block of the handle (a copy into pageable memory is staged by the driver)
        if (!e->h_stats_pinned) NIG_CUDA(cudaHostAlloc((void**)&e->h_stats_pinned, NIG_STATS_SLOTS * sizeof(unsigned long long), cudaHostAllocPortable));
        unsigned long long* hs = e->h_stats_pinned;
        if (r->counters24 || r->sums8) {
            if ((rc = fold_stats(e, st)) != NIG_OK) return rc;
            NIG_CUDA(cudaMemcpyAsync(hs, e->stats, NIG_STATS_SLOTS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        }
        NIG_CUDA(cudaStreamSynchronize(st));
        if (r->counters24) for (int k = 0; k < 24; ++k) r->counters24[k] = (int64_t)hs[k];
        if (r->sums8) memcpy(r->sums8, &hs[24], 8 * sizeof(double));
        return NIG_OK;
    }

    if (r->reset_first || r->init_states) {
        const float* dinit = nullptr;
        if (r->init_states) {
            NIG_CUDA(cudaMemcpyAsync(e->h_reset, r->init_states, n * e->S * sizeof(float), cudaMemcpyHostToDevice, st));
            dinit = e->h_reset;
        }
        if ((rc = nig_reset(e, nullptr, dinit, NIG_LAYOUT_AOS, st)) != NIG_OK) return rc;
    }
    // rows of a [T][D][n] host tensor -> [K][D][pitch] device chunk
    auto copy_chunk = [&](float* dst, const float* src, int D, int32_t t0, int32_t k) -> cudaError_t {
        return cudaMemcpy2DAsync(dst, cap * sizeof(float), src + (size_t)t0 * D * n, n * sizeof(float), n * sizeof(float),
                                 (size_t)k * D, cudaMemcpyHostToDevice, e->copy_stream);
    };
    int32_t done = 0;
    for (int c = 0; done < T; ++c) {
        const int32_t k = T - done < K ? T - done : K;
        const int b = c & 1;
        nig_rollout_t d;
        memset(&d, 0, sizeof d);
        d.n_steps = k; d.policy = r->policy; d.pp = r->pp;
        d.flags = c > 0 ? NIG_ROLLOUT_ACCUMULATE : 0;
        if (forced) {
            NIG_CUDA(cudaStreamWaitEvent(e->copy_stream, e->r_ev_done[b], 0));     // the launch that last read this buffer
            NIG_CUDA(copy_chunk(e->r_act[b], r->actions, e->A, done, k));
            if (r->noise) NIG_CUDA(copy_chunk(e->r_nz[b], r->noise, e->NZ, done, k));
            NIG_CUDA(cudaEventRecord(e->r_ev_copy[b], e->copy_stream));
            NIG_CUDA(cudaStreamWaitEvent(st, e->r_ev_copy[b], 0));
            d.actions = e->r_act[b];
            d.noise = r->noise ? e->r_nz[b] : nullptr;
            d.flags |= NIG_ROLLOUT_USE_TMA;
        }
        d.reward_sum = r->reward_sum ? e->h_reward : nullptr;
        d.viol_count = r->viol_count ? e->h_i32a : nullptr;
        d.done_count = r->done_count ? e->h_i32b : nullptr;
        if ((rc = nig_rollout(e, &d, st)) != NIG_OK) return rc;
        if (forced) NIG_CUDA(cudaEventRecord(e->r_ev_done[b], st));
        done += k;
    }
    if (r->final_obs) {
        if ((rc = state_io(e, e->h_obs, NIG_LAYOUT_AOS, nullptr, nullptr, nullptr, true, st)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(r->final_obs, e->h_obs, n * e->S * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    if (r->reward_sum) NIG_CUDA(cudaMemcpyAsync(r->reward_sum, e->h_reward, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (r->viol_count) NIG_CUDA(cudaMemcpyAsync(r->viol_count, e->h_i32a, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (r->done_count) NIG_CUDA(cudaMemcpyAsync(r->done_count, e->h_i32b, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    unsigned long long hs[NIG_STATS_SLOTS];
    if (r->counters24 || r->sums8) {
        if ((rc = fold_stats(e, st)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(hs, e->stats, sizeof hs, cudaMemcpyDeviceToHost, st));
    }
    NIG_CUDA(cudaStreamSynchronize(st));
    if (r->counters24) for (int k = 0; k < 24; ++k) r->counters24[k] = (int64_t)hs[k];
    if (r->sums8) memcpy(r->sums8, &hs[24], 8 * sizeof(double));
    return NIG_OK;
}

} // extern "C"

namespace {

template <bool WRITE>
int launch_dataset(nig_env* e, const DatasetArgs& a, cudaStream_t st)
{
    e->launches++;
    note_device_work(e, st);
    NIG_CUDA(nig::launch_dataset(e->kind, e->cons.is_default, WRITE, a, st));
    return NIG_OK;
}

int dataset_args(nig_env* e, int64_t n_episodes, int32_t n_steps, int32_t policy, const nig_policy_params_t* pp, DatasetArgs* a)
{
    if (n_episodes <= 0 || n_episodes > (1LL << 31)) return fail(NIG_ERR_INVALID, "n_episodes %lld outside [1, 2^31]", (long long)n_episodes);
    if (e->cfg.env_id_offset > (1LL << 32) - n_episodes)          // episode e is the env of global id env_id_offset + e
        return fail(NIG_ERR_INVALID, "episode ids env_id_offset %lld + [0, %lld) exceed 2^32", (long long)e->cfg.env_id_offset, (long long)n_episodes);
    if (n_steps <= 0) return fail(NIG_ERR_INVALID, "n_steps must be positive (got %d)", n_steps);
    if (policy == NIG_POLICY_MLP) return fail(NIG_ERR_UNSUPPORTED, "the dataset kernels have no NIG_POLICY_MLP flavour");
    if (policy != NIG_POLICY_UNIFORM && policy != NIG_POLICY_ZERO && policy != NIG_POLICY_PCTRL)
        return fail(NIG_ERR_INVALID, "dataset policy must be UNIFORM, ZERO or PCTRL (got %d)", policy);
    if (policy == NIG_POLICY_PCTRL && !pp) return fail(NIG_ERR_INVALID, "NIG_POLICY_PCTRL needs policy parameters");
    for (int k = 0; k < e->cons.n; ++k)
        if (e->cons.c[k].kind == NIG_CON_HOSTMASK) return fail(NIG_ERR_UNSUPPORTED, "host-evaluated constraints cannot run inside the dataset kernels");
    if (n_episodes > e->d_len_cap) {
        cudaFree(e->d_len); cudaFree(e->d_off); e->d_len = e->d_off = nullptr; e->d_len_cap = 0;
        int rc;
        if ((rc = dev_alloc(&e->d_len, (size_t)n_episodes)) != NIG_OK) return rc;
        if ((rc = dev_alloc(&e->d_off, (size_t)n_episodes)) != NIG_OK) return rc;
        e->d_len_cap = n_episodes;
    }
    int rc;
    if ((rc = dev_alloc(&e->d_total, 1)) != NIG_OK) return rc;
    memset(a, 0, sizeof *a);
    a->n_episodes = n_episodes; a->n_steps = n_steps; a->max_steps = e->max_steps; a->policy = policy;
    a->env0 = (uint32_t)e->cfg.env_id_offset; a->epoch = 0;
    // every dataset draws from its own key derived from (seed, number of datasets generated so far)
    a->key = RngKey{e->key.k0 ^ (0x9E3779B9u * (e->dataset_gen + 1u)), e->key.k1 ^ 0x85EBCA6Bu};
    if (pp) a->pp = *pp;
    a->cons = e->cons;
    a->lengths = e->d_len; a->offsets = e->d_off;
    return NIG_OK;
}

// pass 1 + scan; the result is cached so that nig_dataset() right after nig_dataset_size() does not repeat it. The cache is
// keyed on the derived key, not on the handle's seed or dataset count, so that whatever changes the random streams
// (nig_set_seed, a dataset written in between) also misses it.
int dataset_probe(nig_env* e, int64_t n_episodes, int32_t n_steps, int32_t policy, const nig_policy_params_t* pp, DatasetArgs* a,
                  int64_t* total, cudaStream_t st)
{
    int rc;
    if ((rc = dataset_args(e, n_episodes, n_steps, policy, pp, a)) != NIG_OK) return rc;
    auto& c = e->probe;
    const bool hit = c.valid && c.n_episodes == n_episodes && c.n_steps == n_steps && c.policy == policy && c.key.k0 == a->key.k0 &&
                     c.key.k1 == a->key.k1 && memcmp(&c.pp, &a->pp, sizeof c.pp) == 0 && memcmp(&c.cons, &e->cons, sizeof c.cons) == 0;
    if (!hit) {
        if ((rc = launch_dataset<false>(e, *a, st)) != NIG_OK) return rc;
        e->launches++;
        NIG_CUDA(nig::launch_scan_lengths(e->d_len, e->d_off, n_episodes, e->d_total, st));
        int64_t t = 0;
        NIG_CUDA(cudaMemcpyAsync(&t, e->d_total, sizeof t, cudaMemcpyDeviceToHost, st));
        NIG_CUDA(cudaStreamSynchronize(st));
        c.n_episodes = n_episodes; c.n_steps = n_steps; c.policy = policy; c.pp = a->pp; c.cons = e->cons; c.key = a->key;
        c.total = t; c.valid = true;
    }
    *total = c.total;
    return NIG_OK;
}

} // namespace

extern "C" {

int nig_dataset_size(nig_env_t* e, int64_t n_episodes, int32_t n_steps, int32_t policy, const nig_policy_params_t* pp,
                     int64_t* n_transitions, void* stream)
{
    NIG_CHECK_ENV(e);
    if (!n_transitions) return fail(NIG_ERR_INVALID, "null n_transitions");
    DatasetArgs a;
    return dataset_probe(e, n_episodes, n_steps, policy, pp, &a, n_transitions, (cudaStream_t)stream);
}

int nig_dataset(nig_env_t* e, int64_t n_episodes, int32_t n_steps, int32_t policy, const nig_policy_params_t* pp,
                const nig_dataset_out_t* out, int64_t* n_written, void* stream)
{
    NIG_CHECK_ENV(e);
    if (!out || !out->observations || !out->actions || !out->rewards || !out->terminals)
        return fail(NIG_ERR_INVALID, "nig_dataset: observations, actions, rewards and terminals are required");
    DatasetArgs a;
    int64_t total = 0;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = dataset_probe(e, n_episodes, n_steps, policy, pp, &a, &total, st);
    if (rc != NIG_OK) return rc;
    if (total > out->capacity) return fail(NIG_ERR_INVALID, "nig_dataset: %lld transitions exceed the capacity %lld", (long long)total, (long long)out->capacity);
    a.terminals_include_truncation = out->terminals_include_truncation;
    a.observations = out->observations; a.actions = out->actions; a.rewards = out->rewards; a.terminals = out->terminals;
    a.timeouts = out->timeouts; a.next_observations = out->next_observations; a.safety = out->safety;
    if ((rc = launch_dataset<true>(e, a, st)) != NIG_OK) return rc;
    e->dataset_gen += 1;
    e->probe.valid = false;
    if (n_written) *n_written = total;
    return NIG_OK;
}

int nig_get_state(nig_env_t* e, float* state_dev, int32_t layout, int32_t* st, int32_t* vi, uint8_t* dn, void* stream)
{
    NIG_CHECK_ENV(e);
    return state_io(e, state_dev, layout, st, vi, dn, true, (cudaStream_t)stream);
}
int nig_set_state(nig_env_t* e, const float* state_dev, int32_t layout, const int32_t* st, const int32_t* vi, const uint8_t* dn, void* stream)
{
    NIG_CHECK_ENV(e);
    return state_io(e, const_cast<float*>(state_dev), layout, const_cast<int32_t*>(st), const_cast<int32_t*>(vi), const_cast<uint8_t*>(dn), false, (cudaStream_t)stream);
}

int nig_get_state_host(nig_env_t* e, float* state_aos, int32_t* st, int32_t* vi, uint8_t* dn)
{
    NIG_CHECK_ENV(e);
    if (int hrc = host_entry(e)) return hrc;
    int rc;
    const size_t n = (size_t)e->n, cap = (size_t)e->pitch;
    if ((rc = dev_alloc(&e->h_obs, cap * e->S)) != NIG_OK) return rc;
    if ((rc = dev_alloc(&e->h_i32a, cap)) != NIG_OK) return rc;
    if ((rc = dev_alloc(&e->h_i32b, cap)) != NIG_OK) return rc;
    if ((rc = dev_alloc(&e->h_flags, cap)) != NIG_OK) return rc;
    if ((rc = state_io(e, e->h_obs, NIG_LAYOUT_AOS, e->h_i32a, e->h_i32b, e->h_flags, true, e->stream)) != NIG_OK) return rc;
    if (state_aos) NIG_CUDA(cudaMemcpyAsync(state_aos, e->h_obs, n * e->S * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    if (st) NIG_CUDA(cudaMemcpyAsync(st, e->h_i32a, n * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    if (vi) NIG_CUDA(cudaMemcpyAsync(vi, e->h_i32b, n * sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    if (dn) NIG_CUDA(cudaMemcpyAsync(dn, e->h_flags, n, cudaMemcpyDeviceToHost, e->stream));
    NIG_CUDA(cudaStreamSynchronize(e->stream));
    return NIG_OK;
}

int nig_set_state_host(nig_env_t* e, const float* state_aos, const int32_t* st, const int32_t* vi, const uint8_t* dn)
{
    NIG_CHECK_ENV(e);
    if (int hrc = host_entry(e)) return hrc;
    int rc;
    const size_t n = (size_t)e->n, cap = (size_t)e->pitch;
    for (size_t i = 0; st && i < n; ++i)           // the episode word holds 16 bits of episode step
        if (st[i] < 0 || st[i] > 65535) return fail(NIG_ERR_INVALID, "nig_set_state_host: ep_step[%zu] = %d outside [0, 65535]", i, st[i]);
    for (size_t i = 0; vi && i < n; ++i)           // (above 32,767 it saturates like the kernels' running count)
        if (vi[i] < 0) return fail(NIG_ERR_INVALID, "nig_set_state_host: ep_viol[%zu] = %d is negative", i, vi[i]);
    float* ds = nullptr; int32_t *dst = nullptr, *dvi = nullptr; uint8_t* ddn = nullptr;
    if (state_aos) {
        if ((rc = dev_alloc(&e->h_obs, cap * e->S)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_obs, state_aos, n * e->S * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        ds = e->h_obs;
    }
    if (st) {
        if ((rc = dev_alloc(&e->h_i32a, cap)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_i32a, st, n * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
        dst = e->h_i32a;
    }
    if (vi) {
        if ((rc = dev_alloc(&e->h_i32b, cap)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_i32b, vi, n * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
        dvi = e->h_i32b;
    }
    if (dn) {
        if ((rc = dev_alloc(&e->h_flags, cap)) != NIG_OK) return rc;
        NIG_CUDA(cudaMemcpyAsync(e->h_flags, dn, n, cudaMemcpyHostToDevice, e->stream));
        ddn = e->h_flags;
    }
    if ((rc = state_io(e, ds, NIG_LAYOUT_AOS, dst, dvi, ddn, false, e->stream)) != NIG_OK) return rc;
    NIG_CUDA(cudaStreamSynchronize(e->stream));
    return NIG_OK;
}

int nig_state_ptr(nig_env_t* e, float** state, uint32_t** ep_word)
{
    if (!e) return fail(NIG_ERR_INVALID, "null env handle");
    if (state) *state = e->state;
    if (ep_word) *ep_word = e->ep_word;
    return NIG_OK;
}

int nig_get_tick(const nig_env_t* e, uint32_t* tick, uint32_t* epoch)
{
    if (!e) return fail(NIG_ERR_INVALID, "null env handle");
    if (tick) {
        *tick = e->tick;
        if (e->tick_dev) {          // device-tick modes: the counter lives on the device (graph replays advance it)
            DeviceGuard guard(e->cfg.device);
            NIG_CUDA(cudaDeviceSynchronize());
            NIG_CUDA(cudaMemcpy(tick, e->tick_dev, sizeof(uint32_t), cudaMemcpyDeviceToHost));
            if (e->tick_mode == 2) *tick += e->tick - e->tick_commit;      // launches since the last commit
        }
    }
    if (epoch) *epoch = e->epoch;
    return NIG_OK;
}
int nig_set_tick(nig_env_t* e, uint32_t tick, uint32_t epoch)
{
    if (!e) return fail(NIG_ERR_INVALID, "null env handle");
    e->tick = tick; e->epoch = epoch; e->tick_commit = tick;
    if (e->tick_dev) {
        DeviceGuard guard(e->cfg.device);
        NIG_CUDA(cudaDeviceSynchronize());
        NIG_CUDA(cudaMemcpy(e->tick_dev, &tick, sizeof(uint32_t), cudaMemcpyHostToDevice));
        NIG_CUDA(cudaDeviceSynchronize());
    }
    return NIG_OK;
}

int nig_use_device_tick(nig_env_t* e, int32_t enable)
{
    if (e) e->config_version++;
    NIG_CHECK_ENV(e);
    if (enable < 0 || enable > 2) return fail(NIG_ERR_INVALID, "nig_use_device_tick: mode must be 0, 1 or 2");
    uint32_t now = 0;
    if (int rc = nig_get_tick(e, &now, nullptr)) return rc;      // (synchronises in the device modes)
    NIG_CUDA(cudaDeviceSynchronize());
    if (enable && !e->tick_dev) NIG_CUDA(cudaMalloc((void**)&e->tick_dev, 2 * sizeof(uint32_t)));
    if (!enable && e->tick_dev) { cudaFree(e->tick_dev); e->tick_dev = nullptr; }
    e->tick = now; e->tick_commit = now; e->tick_mode = enable;
    if (e->tick_dev) {
        const uint32_t init[2] = {now, 0u};
        NIG_CUDA(cudaMemcpy(e->tick_dev, init, sizeof init, cudaMemcpyHostToDevice));
        NIG_CUDA(cudaDeviceSynchronize());
    }
    return NIG_OK;
}

int nig_commit_ticks(nig_env_t* e, void* stream)
{
    NIG_CHECK_ENV(e);
    if (e->tick_mode != 2) return NIG_OK;                        // nothing to commit in the other modes
    const uint32_t by = e->tick - e->tick_commit;
    if (by) {
        e->launches++;
        note_device_work(e, (cudaStream_t)stream);
        NIG_CUDA(nig::launch_commit_ticks(e->tick_dev, by, (cudaStream_t)stream));
    }
    e->tick_commit = e->tick;
    return NIG_OK;
}

int nig_set_seed(nig_env_t* e, uint64_t seed)
{
    if (!e) return fail(NIG_ERR_INVALID, "null env handle");
    e->cfg.seed = seed;
    e->config_version++;
    e->key = RngKey{(uint32_t)seed, (uint32_t)(seed >> 32)};
    // a new key starts its streams at their origin: reset(seed = s) is reproducible whatever the handle did before
    return nig_set_tick(e, 0u, 0u);
}

int nig_stats_ptr(nig_env_t* e, void** p)
{
    if (!e || !p) return fail(NIG_ERR_INVALID, "null env handle or pointer");
    *p = e->stats;
    return NIG_OK;
}

int nig_fold_stats(nig_env_t* e, void* stream)
{
    NIG_CHECK_ENV(e);
    note_device_work(e, (cudaStream_t)stream);
    return fold_stats(e, (cudaStream_t)stream);
}

int nig_read_stats(nig_env_t* e, int64_t* counters24, double* sums8)
{
    NIG_CHECK_ENV(e);
    unsigned long long h[NIG_STATS_SLOTS];
    NIG_CUDA(cudaDeviceSynchronize());
    if (int rc = fold_stats(e, nullptr)) return rc;
    NIG_CUDA(cudaMemcpy(h, e->stats, sizeof h, cudaMemcpyDeviceToHost));
    if (counters24) for (int k = 0; k < 24; ++k) counters24[k] = (int64_t)h[k];
    if (sums8) memcpy(sums8, &h[24], 8 * sizeof(double));
    return NIG_OK;
}

// ---- the path's one collective, for callers that do not come through torch.distributed ------------------------------
// NCCL is bound lazily with dlopen (libnccl.so.2: the copy already loaded into the process -- e.g. torch's -- wins, else
// the system's), so the library has no link-time dependency on it and loads on machines without NCCL.
namespace {
struct nccl_id_t { char internal[128]; };            // == ncclUniqueId
struct NcclApi {
    void* lib = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    int (*GetUniqueId)(nccl_id_t*) = nullptr;
    int (*CommInitRank)(void**, int, nccl_id_t, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
};
enum { kNcclInt64 = 4, kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2 };   // ncclDataType_t / ncclRedOp_t values (nccl.h)

const NcclApi* nccl_api()
{
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (h) {
            api.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
            api.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
            api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
            api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
            api.GetUniqueId = (int (*)(nccl_id_t*))dlsym(h, "ncclGetUniqueId");
            api.CommInitRank = (int (*)(void**, int, nccl_id_t, int))dlsym(h, "ncclCommInitRank");
            api.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
            if (api.GroupStart && api.GroupEnd && api.AllReduce && api.GetUniqueId && api.CommInitRank && api.CommDestroy) api.lib = h;
        }
    }
    return api.lib ? &api : nullptr;
}
int nccl_fail(const NcclApi* a, int rc, const char* what)
{
    return fail(NIG_ERR_CUDA, "%s failed: %s", what, a->GetErrorString ? a->GetErrorString(rc) : "NCCL error");
}
#define NIG_NCCL(api, call, what) do { const int nrc_ = (call); if (nrc_ != 0) return nccl_fail(api, nrc_, what); } while (0)
} // namespace

int nig_nccl_unique_id(void* id128)
{
    const NcclApi* a = nccl_api();
    if (!a) return fail(NIG_ERR_UNSUPPORTED, "libnccl.so.2 not found (NCCL is only needed for nig_allreduce_stats)");
    if (!id128) return fail(NIG_ERR_INVALID, "nig_nccl_unique_id: null buffer");
    nccl_id_t id;
    NIG_NCCL(a, a->GetUniqueId(&id), "ncclGetUniqueId");
    memcpy(id128, &id, sizeof id);
    return NIG_OK;
}

int nig_nccl_comm_init(void** comm, int32_t n_ranks, const void* id128, int32_t rank, int32_t device)
{
    const NcclApi* a = nccl_api();
    if (!a) return fail(NIG_ERR_UNSUPPORTED, "libnccl.so.2 not found (NCCL is only needed for nig_allreduce_stats)");
    if (!comm || !id128 || n_ranks <= 0 || rank < 0 || rank >= n_ranks) return fail(NIG_ERR_INVALID, "nig_nccl_comm_init: bad arguments");
    DeviceGuard guard(device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    nccl_id_t id;
    memcpy(&id, id128, sizeof id);
    *comm = nullptr;
    NIG_NCCL(a, a->CommInitRank(comm, n_ranks, id, rank), "ncclCommInitRank");
    return NIG_OK;
}

int nig_nccl_comm_destroy(void* comm)
{
    const NcclApi* a = nccl_api();
    if (!a) return fail(NIG_ERR_UNSUPPORTED, "libnccl.so.2 not found");
    if (comm) NIG_NCCL(a, a->CommDestroy(comm), "ncclCommDestroy");
    return NIG_OK;
}

int nig_allreduce_stats(nig_env_t* e, void* nccl_comm, void* stream)
{
    NIG_CHECK_ENV(e);
    const NcclApi* a = nccl_api();
    if (!a) return fail(NIG_ERR_UNSUPPORTED, "libnccl.so.2 not found (NCCL is only needed for nig_allreduce_stats)");
    if (!nccl_comm) return fail(NIG_ERR_INVALID, "nig_allreduce_stats: null communicator");
    cudaStream_t st = (cudaStream_t)stream;
    note_device_work(e, st);
    // one group = one fused launch: 24 int64 counters (SUM: exact, order independent), 8 fp64 sums (SUM), and the two
    // order-preserving return-extremum keys (MAX; zeros when nothing was tracked)
    if (int frc = fold_stats(e, st)) return frc;
    NIG_NCCL(a, a->GroupStart(), "ncclGroupStart");
    int rc = a->AllReduce(e->stats, e->stats, 24, kNcclInt64, kNcclSum, nccl_comm, st);
    if (rc == 0) rc = a->AllReduce(e->stats + 24, e->stats + 24, NIG_STATS_SLOTS - 24, kNcclFloat64, kNcclSum, nccl_comm, st);
    if (rc == 0) rc = a->AllReduce(e->extrema, e->extrema, 2, kNcclInt64, kNcclMax, nccl_comm, st);
    const int rc_end = a->GroupEnd();
    if (rc != 0) return nccl_fail(a, rc, "ncclAllReduce");
    NIG_NCCL(a, rc_end, "ncclGroupEnd");
    return NIG_OK;
}

int nig_clear_stats(nig_env_t* e, void* stream)
{
    NIG_CHECK_ENV(e);
    NIG_CUDA(cudaMemsetAsync(e->stats, 0, NIG_STATS_SLOTS * sizeof(unsigned long long), (cudaStream_t)stream));
    NIG_CUDA(cudaMemsetAsync(e->stats_shards, 0, (size_t)nig::kStatsShards * NIG_STATS_SLOTS * sizeof(unsigned long long), (cudaStream_t)stream));
    e->shards_dirty = false;
    NIG_CUDA(cudaMemsetAsync(e->extrema, 0, 2 * sizeof(unsigned long long), (cudaStream_t)stream));
    return NIG_OK;
}

int nig_track_returns(nig_env_t* e, int32_t on)
{
    if (e) e->config_version++;
    NIG_CHECK_ENV(e);
    e->track_returns = on != 0;
    return NIG_OK;
}

int nig_track_step_stats(nig_env_t* e, int32_t on)
{
    if (e) e->config_version++;
    NIG_CHECK_ENV(e);
    e->track_step_stats = on != 0;
    return NIG_OK;
}

int nig_track_extrema(nig_env_t* e, int32_t on)
{
    if (e) e->config_version++;
    NIG_CHECK_ENV(e);
    e->track_extrema = on != 0;
    return NIG_OK;
}

int nig_extrema_ptr(nig_env_t* e, void** p)
{
    if (!e || !p) return fail(NIG_ERR_INVALID, "null env handle or pointer");
    *p = e->extrema;
    return NIG_OK;
}

int nig_decode_extrema(const int64_t* keys2, double* ret_min, double* ret_max, int32_t* have)
{
    if (!keys2) return fail(NIG_ERR_INVALID, "null keys");
    auto decode = [](unsigned long long k) {
        const unsigned long long key = k << 1;                    // the dropped mantissa bit comes back as 0
        const unsigned long long b = (key >> 63) ? (key & 0x7fffffffffffffffull) : ~key;
        double x;
        memcpy(&x, &b, sizeof x);
        return x;
    };
    const bool any = keys2[0] != 0 && keys2[1] != 0;
    if (have) *have = any ? 1 : 0;
    if (ret_min) *ret_min = any ? -decode((unsigned long long)keys2[0]) : 0.0;
    if (ret_max) *ret_max = any ? decode((unsigned long long)keys2[1]) : 0.0;
    return NIG_OK;
}

int nig_read_extrema(nig_env_t* e, double* ret_min, double* ret_max, int32_t* have)
{
    NIG_CHECK_ENV(e);
    int64_t h[2];
    NIG_CUDA(cudaDeviceSynchronize());
    NIG_CUDA(cudaMemcpy(h, e->extrema, sizeof h, cudaMemcpyDeviceToHost));
    return nig_decode_extrema(h, ret_min, ret_max, have);
}

int nig_sync(nig_env_t* e)
{
    NIG_CHECK_ENV(e);
    NIG_CUDA(cudaDeviceSynchronize());
    return NIG_OK;
}

int nig_host_alloc(size_t bytes, void** out)
{
    if (!out) return fail(NIG_ERR_INVALID, "null output pointer");
    *out = nullptr;
    NIG_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped));
    return NIG_OK;
}
int nig_host_free(void* p)
{
    if (p) NIG_CUDA(cudaFreeHost(p));
    return NIG_OK;
}

int nig_selftest_division(int device, int64_t n, uint64_t seed, int64_t* mismatches, int64_t* accepted)
{
    DeviceGuard guard(device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    if (n <= 0 || !mismatches) return fail(NIG_ERR_INVALID, "nig_selftest_division: n must be positive and mismatches non-null");
    unsigned long long* d = nullptr;
    NIG_CUDA(cudaMalloc((void**)&d, 2 * sizeof(unsigned long long)));
    NIG_CUDA(cudaMemset(d, 0, 2 * sizeof(unsigned long long)));
    const int blocks = 148 * 8, threads = blocks * 256;
    const int iters = (int)((n + threads - 1) / threads);
    cudaError_t ce = nig::launch_selftest_division(RngKey{(uint32_t)seed, (uint32_t)(seed >> 32)}, iters, blocks, d, nullptr);
    unsigned long long h[2] = {0, 0};
    if (ce == cudaSuccess) ce = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d);
    NIG_CUDA(ce);
    *mismatches = (int64_t)h[0];
    if (accepted) *accepted = (int64_t)h[1];
    return NIG_OK;
}

int nig_selftest_normal(int device, uint32_t first, uint32_t stride, int64_t count, uint64_t* sums2)
{
    DeviceGuard guard(device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    if (!sums2 || count < 0) return fail(NIG_ERR_INVALID, "nig_selftest_normal: null sums or negative count");
    unsigned long long* d = nullptr;
    NIG_CUDA(cudaMalloc((void**)&d, 2 * sizeof(unsigned long long)));
    NIG_CUDA(cudaMemset(d, 0, 2 * sizeof(unsigned long long)));
    cudaError_t ce = nig::launch_selftest_normal(first, stride, (unsigned long long)count, d, nullptr);
    unsigned long long h[2] = {0, 0};
    if (ce == cudaSuccess) ce = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d);
    NIG_CUDA(ce);
    sums2[0] = h[0]; sums2[1] = h[1];
    return NIG_OK;
}

int nig_selftest_policy(int device, int32_t env_kind, int32_t policy, const nig_policy_params_t* pp, int64_t n, int32_t n_steps,
                         const float* states, const float* coin, const float* z, const float* u, float* actions)
{
    DeviceGuard guard(device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    if (env_kind < 0 || env_kind > NIG_ENV_ROBOT_ASSEMBLY || !pp || !states || !actions || n <= 0 || n_steps <= 0)
        return fail(NIG_ERR_INVALID, "nig_selftest_policy: bad env kind, null pointer or empty shape");
    if (policy != NIG_POLICY_PCTRL && policy != NIG_POLICY_BASELINE)
        return fail(NIG_ERR_INVALID, "nig_selftest_policy: policy must be NIG_POLICY_PCTRL or NIG_POLICY_BASELINE");
    nig_env_spec_t spec;
    nig_env_spec(env_kind, &spec);
    const size_t rows = (size_t)n * (size_t)n_steps;
    const size_t b_s = rows * spec.state_dim * sizeof(float), b_c = rows * sizeof(float), b_r = rows * 8 * sizeof(float),
                 b_a = rows * spec.action_dim * sizeof(float);
    char* d = nullptr;
    NIG_CUDA(cudaMalloc((void**)&d, b_s + b_c + 2 * b_r + b_a));
    float* d_s = (float*)d; float* d_c = (float*)(d + b_s); float* d_z = (float*)(d + b_s + b_c);
    float* d_u = (float*)(d + b_s + b_c + b_r); float* d_a = (float*)(d + b_s + b_c + 2 * b_r);
    cudaError_t ce = cudaMemcpy(d_s, states, b_s, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && coin) ce = cudaMemcpy(d_c, coin, b_c, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && z) ce = cudaMemcpy(d_z, z, b_r, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && u) ce = cudaMemcpy(d_u, u, b_r, cudaMemcpyHostToDevice);
    nig::PolicyTestArgs a{};
    a.policy = policy; a.T = n_steps; a.n = n; a.pp = *pp;
    a.states = d_s; a.coin = coin ? d_c : nullptr; a.z = z ? d_z : nullptr; a.u = u ? d_u : nullptr; a.actions = d_a;
    if (ce == cudaSuccess) ce = nig::launch_selftest_policy(env_kind, a, nullptr);
    if (ce == cudaSuccess) ce = cudaMemcpy(actions, d_a, b_a, cudaMemcpyDeviceToHost);
    cudaFree(d);
    NIG_CUDA(ce);
    return NIG_OK;
}

int nig_fp32_probe(int device, int32_t iters, double* ops, void* stream)
{
    DeviceGuard guard(device);
    if (!guard.ok) return fail(NIG_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    static float* sinks[64] = {nullptr};          // one scratch word per device (a pointer is only valid on its own device)
    if (device < 0 || device >= 64) return fail(NIG_ERR_INVALID, "nig_fp32_probe: device ordinal %d out of range", device);
    if (!sinks[device]) NIG_CUDA(cudaMalloc((void**)&sinks[device], 256));
    float* sink = sinks[device];
    const int blocks = 148 * 8;
    NIG_CUDA(nig::launch_fp32_probe(sink, iters, blocks, (cudaStream_t)stream));
    if (ops) *ops = (double)blocks * 256.0 * (double)iters * 16.0;
    return NIG_OK;
}

} // extern "C"
