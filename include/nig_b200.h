/* nig_b200.h -- C ABI of the B200-native batched IndustrialEnv step path (libnig_b200.so).
 *
 * The reference (danieleschmidt/neoRL-industrial-gym) is pure Python and has no FFI layer; its
 * boundary for this path is the public env API. Each entry point below names the reference
 * interface it replaces (paths relative to the reference's src/neorl_industrial/). The Python
 * package neorl_industrial (neorl-industrial-gym_b200/neorl_industrial) binds these with ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *  - Every function returns a nig_status (0 = ok); nig_last_error() gives the thread-local message.
 *    No exceptions cross the ABI; nothing allocates after nig_create() except the lazily created
 *    host staging of the *_host calls.
 *  - "dev" pointers are CUDA device pointers on the env's device; `stream` is a cudaStream_t
 *    (NULL = legacy default stream). The *_host calls take ordinary host pointers, do the
 *    host<->device copies themselves (pinned staging, cudaMemcpyAsync) and return synchronised.
 *  - Device state is SoA fp32: component k of env i lives at state[k * pitch + i];
 *    pitch = nig_pitch(env) (n_envs rounded up to 128 elements). Every per-env DEVICE array handed to
 *    nig_step()/nig_rollout() must have capacity >= pitch elements (rows of SoA arrays are
 *    `pitch` apart); host arrays are exact-size.
 *  - Envs are identified by a global id = env_id_offset + local index; all random streams are
 *    keyed by (seed, global id, tick) so a sharded run reproduces the unsharded one bit-for-bit.
 *    Global ids are 32-bit: env_id_offset + n_envs (or + n_episodes of nig_dataset) must not exceed 2^32.
 *  - The tick (one per batched step) is a uint32 Philox counter word and wraps modulo 2^32: stepping across the wrap is
 *    the same as anywhere else. Explicit resets draw with the counter word (epoch << 8) | j, so the draws of epoch e and
 *    e + 2^24 at the same tick coincide: a period of 2^24 explicit resets (auto-resets reuse the current epoch).
 */
#ifndef NIG_B200_H
#define NIG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define NIG_API __attribute__((visibility("default")))
#else
#define NIG_API
#endif

#define NIG_ABI_VERSION 6
#define NIG_MAX_CONSTRAINTS 8
#define NIG_MAX_STATE_DIM 32
#define NIG_MAX_ACTION_DIM 8
#define NIG_MAX_NOISE_DIM 23
#define NIG_STATS_SLOTS 32
/* Most steps one fused launch may run (nig_rollout_t.n_steps; nig_rollout_host caps steps_per_launch at it). A CTA counts
 * its statistics in 32-bit registers and shared slots before it adds them to the int64 block: the largest is
 * 256 envs x NIG_MAX_CONSTRAINTS x K violations (the two-env reactor kernel's 128-thread CTAs), < 2^31 at K = 2^20, and so
 * are a one-warp CTA's 32 x 8 x K and every env's int32 viol_count of one launch. Above it the counters would wrap. */
#define NIG_MAX_LAUNCH_STEPS (1 << 20)

typedef struct nig_env nig_env_t; /* opaque */

typedef enum nig_status {
    NIG_OK = 0,
    NIG_ERR_INVALID = 1,     /* bad argument (shape, kind, null pointer, limit) -> Python ValueError   */
    NIG_ERR_CUDA = 2,        /* CUDA runtime/driver failure                      -> Python RuntimeError */
    NIG_ERR_NO_DEVICE = 3,   /* no usable sm_100 device: the library never falls back to the CPU        */
    NIG_ERR_UNSUPPORTED = 4
} nig_status;

/* utils.make registry (utils.py:26-32); the two "Advanced" ids are not instantiable upstream */
typedef enum nig_env_kind {
    NIG_ENV_CHEMICAL_REACTOR = 0, /* environments/chemical_reactor.py */
    NIG_ENV_POWER_GRID = 1,       /* environments/power_grid.py       */
    NIG_ENV_ROBOT_ASSEMBLY = 2    /* environments/robot_assembly.py   */
} nig_env_kind;

/* SafetyConstraint (core/types.py:56-64) as a declarative descriptor.
 *  BUILTIN : the env's own check_fn number `id` (registration order in the env's __init__)
 *  BOUND   : lo <= s[si] + coef * a[ai] <= hi on the pre-step state and clipped action (ai < 0: no
 *            action term) -- the SafetyWrapper temperature/pressure-bound form (README.md:126-139)
 *  HOSTMASK: bit `id` of the caller-supplied per-env mask says "violated" (lets the Python layer keep
 *            arbitrary check_fn callables: it evaluates them on the host, the kernel applies them) */
typedef enum nig_con_kind { NIG_CON_BUILTIN = 0, NIG_CON_BOUND = 1, NIG_CON_HOSTMASK = 2 } nig_con_kind;

typedef struct nig_constraint {
    int32_t kind;
    int32_t id;
    int32_t si;
    int32_t ai;
    float coef;
    float lo;
    float hi;
    float penalty;    /* added to the reward when violated (base.py:179-183) */
    int32_t critical; /* violated -> terminated = true, reward -= 1000 (base.py:195-198) */
} nig_constraint_t;

typedef struct nig_env_spec {
    int32_t state_dim;
    int32_t action_dim;
    int32_t noise_dim;          /* Gaussian draws per step, in the reference's draw order */
    int32_t max_episode_steps;  /* 500 reactor (chemical_reactor.py:66), 1000 others (base.py:27) */
    int32_t n_constraints;
    int32_t reserved;
    nig_constraint_t constraints[NIG_MAX_CONSTRAINTS]; /* the built-ins with their penalties */
} nig_env_spec_t;

typedef struct nig_config {
    int32_t env_kind;
    int32_t device;            /* CUDA device ordinal */
    int64_t n_envs;            /* envs owned by THIS handle (this GPU's shard) */
    int64_t env_id_offset;     /* global id of local env 0; >= 0 and env_id_offset + n_envs <= 2^32 */
    uint64_t seed;
    int32_t max_episode_steps; /* 0 = env default; <= 65535 */
    int32_t auto_reset;        /* 1: a finished env is re-initialised inside the same step call */
    int32_t n_constraints;     /* -1 = the env's built-ins */
    int32_t reserved;
    nig_constraint_t constraints[NIG_MAX_CONSTRAINTS];
} nig_config_t;

/* per-step output flag bits */
enum {
    NIG_F_TERMINATED = 1,  /* base.py:190 / :196 */
    NIG_F_TRUNCATED = 2,   /* base.py:191 */
    NIG_F_CRITICAL = 4,    /* info["critical_shutdown"], base.py:210 */
    NIG_F_RESET = 8,       /* the env was auto-reset after this transition */
    NIG_F_INACTIVE = 128   /* env already finished and auto_reset == 0: nothing was stepped */
};

enum { NIG_LAYOUT_SOA = 0, NIG_LAYOUT_AOS = 1 };

/* One IndustrialEnv.step (base.py:157-213) over all envs of the handle.
 * SoA arrays are [dim][pitch]; AoS arrays are [n][dim]. NULL = not supplied / not wanted. */
typedef struct nig_step_io {
    const float* actions;       /* in : [A][pitch] or [n][A]; clipped to [-1, 1] by the kernel (base.py:167) */
    const float* noise;         /* in : teacher-forced process noise [NZ][pitch] or [n][NZ]; NULL -> in-kernel Philox */
    const float* reset_states;  /* in : teacher-forced post-done states [S][pitch] or [n][S]; NULL -> in-kernel draw */
    const uint8_t* hostmask;    /* in : [n] bits for NIG_CON_HOSTMASK constraints; NULL -> 0 */
    float* obs;                 /* out: state AFTER the call (post auto-reset): [S][pitch] or [n][S] */
    float* next_obs;            /* out: s' of the transition (pre auto-reset); same layout as obs */
    float* reward;              /* out: [n] */
    uint8_t* flags;             /* out: [n] NIG_F_* bits */
    uint8_t* viol_mask;         /* out: [n] bit k = constraint k violated on the pre-step state */
    int32_t action_layout;      /* NIG_LAYOUT_* of actions */
    int32_t aux_layout;         /* NIG_LAYOUT_* of noise / reset_states / obs / next_obs */
    uint8_t* terminated;        /* out: [n] 0/1, the gym `terminated` of base.py:190/196 unpacked from flags; NULL ok */
    uint8_t* truncated;         /* out: [n] 0/1, the gym `truncated` of base.py:191; NULL ok */
} nig_step_io_t;

/* fused K-step rollout policies */
enum {
    NIG_POLICY_ACTIONS = 0,  /* actions[K][A][pitch] read from HBM (TMA-staged through shared memory) */
    NIG_POLICY_UNIFORM = 1,  /* a ~ U(-1,1)^A from the in-kernel Philox policy stream (= action_space.sample(),
                                the reference's timing harness performance_benchmark.py:106-133) */
    NIG_POLICY_ZERO = 2,
    NIG_POLICY_PCTRL = 3,    /* get_dataset's "PID-like" P-controller mixes (chemical_reactor.py:364-390) */
    NIG_POLICY_BASELINE = 4, /* the benchmark baseline controllers (benchmarks/baseline_agents.py:28-114), nig_baseline_t */
    NIG_POLICY_MLP = 5       /* a deterministic MLP actor (nig_set_mlp_policy) evaluated by the tensor cores in the kernel */
};

/* NIG_POLICY_MLP: the deterministic actor of an offline-RL agent (TD3+BC / IQL / CQL style), evaluated inside the fused
 * rollout by tcgen05 MMAs, 128 envs per tile, one env per accumulator row. Network family and numeric contract:
 *  - input: the observation the env hands the policy, i.e. the pre-step state s (base.py:201). Optional normalisation
 *    x = (s - obs_mean) * obs_inv_std in fp32 (round to nearest, no contraction); NULL mean / inv_std = 0 / 1.
 *  - n_hidden = 1 or 2 hidden layers, each of width 64, 128 or 256, ReLU (NaN-propagating, like torch.relu);
 *    then an output layer of width A followed by tanh or identity. The env clips the action to [-1, 1] as always.
 *  - weights and every layer's INPUT are rounded to bf16 (nearest even); products are accumulated in fp32 by the tensor
 *    core in the hardware's order; biases and activations are applied in fp32. Inputs are zero-padded to a multiple of 16
 *    (reactor 12 -> 16, robot 24 -> 32), the output to 16 columns; the padding is invisible.
 *  - actions are therefore specified to a tolerance against an fp64 forward pass of the bf16-rounded network, not bit for
 *    bit (where every layer's exact sum is fp32-representable the order does not matter and the action is exact: bit for
 *    bit with identity output, within tanhf's 2 ulp with tanh); everything downstream of the action keeps the bit-exact
 *    contract. Env i's action depends only on its own
 *    observation and the weights (row i mod 128 of its tile), not on the population, slicing or launch shape.
 * Not supported (NIG_ERR_INVALID): more layers, other widths, other activations; stochastic actors; fp16 / fp8 / tf32 weights
 * (the ABI takes fp32, the library rounds to bf16). */
enum { NIG_MLP_OUT_IDENTITY = 0, NIG_MLP_OUT_TANH = 1 };
typedef struct nig_mlp {
    int32_t n_hidden;           /* hidden layers: 1 or 2 */
    int32_t hidden[2];          /* hidden widths (64, 128 or 256); hidden[1] ignored when n_hidden == 1 */
    int32_t output_activation;  /* NIG_MLP_OUT_* */
    int32_t in_dim;             /* must equal the env's state_dim */
    int32_t out_dim;            /* must equal the env's action_dim */
    const float* weight[3];     /* host fp32 [out][in] (torch nn.Linear order): the hidden layers, then the output layer
                                   (weight[1] is the output layer when n_hidden == 1) */
    const float* bias[3];       /* host fp32 [out] per layer, same order; NULL = zeros */
    const float* obs_mean;      /* host fp32 [in_dim] or NULL */
    const float* obs_inv_std;   /* host fp32 [in_dim] or NULL */
} nig_mlp_t;

/* Baseline controllers evaluated inside the fused rollout kernel (benchmarks/baseline_agents.py). The reference
 * computes them in numpy float64 from the float32 observation; so does the kernel (fp64 registers), then the action
 * is rounded to fp32 and clipped by the env like any other action.
 *  RANDOM   : a ~ U(setpoint[0], setpoint[1])^A (RandomAgent :28-43; drawn from the Philox policy stream)
 *  PID      : e = setpoint - s[:A]; I += e; a = clip(kp*e + ki*I + kd*(e - e_prev), -1, 1) (PIDControllerAgent :46-81).
 *             I and e_prev persist across episodes like the agent object does; nig_reset_policy_state() zeroes them
 *             (= constructing a new agent).
 *  MPC      : a = clip(0.5 * (0 - s[:A]), -1, 1) (MPC_Agent :84-100, the "simplified MPC" heuristic)
 *  CONSTANT : a = setpoint (ConstantAgent :103-114) */
enum { NIG_BASELINE_RANDOM = 0, NIG_BASELINE_PID = 1, NIG_BASELINE_MPC = 2, NIG_BASELINE_CONSTANT = 3 };
typedef struct nig_baseline {
    int32_t kind;
    int32_t reserved;
    double kp, ki, kd;
    double setpoint[NIG_MAX_ACTION_DIM];
} nig_baseline_t;

/* get_dataset policy parameters (chemical_reactor.py:333-390, power_grid.py:216-232,
 * robot_assembly.py:266-291; SURVEY Appendix D). Per step, with probability p_ctrl the env's controller
 * branch is taken, else a ~ U(-uniform_scale, uniform_scale)^A:
 *   reactor: a_j = gain[j][0]*(T-320)/50 + gain[j][1]*(level-55)/50 + sigma[j]*N(0,1)
 *   grid   : a_j = gain[j][0]*freq_dev   + gain[j][1]*(sum load - sum gen)/8 + sigma[j]*N(0,1)
 *   robot  : mode 0: a[0:3] = gain[0][0]*(target-pos), a[3:7] = gain[3][0]*q[3:7]  (expert, :268-277)
 *            mode 1: a[0:3] = gain[0][0]*(target-pos), a[3:7] ~ U(-sigma[3], sigma[3])  (mixed, :284-287)
 * store_clip > 0: the dataset stores clip(a, +-store_clip) (reactor 1, robot 2); the env itself always
 * clips to +-1 (base.py:167). */
typedef struct nig_policy_params {
    float p_ctrl;
    float uniform_scale;
    float store_clip;
    int32_t mode;
    float gain[NIG_MAX_ACTION_DIM][2];
    float sigma[NIG_MAX_ACTION_DIM];
    nig_baseline_t baseline;    /* NIG_POLICY_BASELINE only */
} nig_policy_params_t;

enum {
    NIG_ROLLOUT_USE_TMA = 1,     /* stage NIG_POLICY_ACTIONS through cp.async.bulk.tensor */
    NIG_ROLLOUT_ACCUMULATE = 2   /* reward_sum / viol_count / done_count: add to the arrays instead of overwriting them */
};

typedef struct nig_rollout {
    int32_t n_steps;            /* K, 1 .. NIG_MAX_LAUNCH_STEPS (NIG_ERR_INVALID above) */
    int32_t policy;             /* NIG_POLICY_* */
    int32_t flags;              /* NIG_ROLLOUT_* */
    int32_t reserved;
    const float* actions;       /* dev [K][A][pitch] when policy == NIG_POLICY_ACTIONS */
    const float* noise;         /* dev teacher-forced noise [K][NZ][pitch]; NULL -> in-kernel Philox */
    nig_policy_params_t pp;
    float* reward_sum;          /* out dev [n]: sum over the K steps of this call (fp32, step order); NULL ok */
    int32_t* viol_count;        /* out dev [n]: violations over the K steps; NULL ok */
    int32_t* done_count;        /* out dev [n]: episodes finished over the K steps; NULL ok */
} nig_rollout_t;

/* D4RL-layout transition arrays written by the on-device get_dataset (chemical_reactor.py:414-420,
 * power_grid.py:244-249, robot_assembly.py:303-308). Row-major, episode-contiguous, device pointers
 * with capacity for `capacity` transitions. next_observations / safety are documented extensions. */
typedef struct nig_dataset_out {
    float* observations;        /* [M][S] */
    float* actions;             /* [M][A] (clipped, as stored by the reference) */
    float* rewards;             /* [M]    */
    uint8_t* terminals;         /* [M]    terminated | truncated (reactor); terminated (grid/robot) */
    uint8_t* timeouts;          /* [M]    all zero (chemical_reactor.py:419); NULL ok */
    float* next_observations;   /* [M][S] extension; NULL ok */
    uint8_t* safety;            /* [M]    extension: violation mask of the transition; NULL ok */
    int64_t capacity;
    int32_t terminals_include_truncation; /* 1: terminals = terminated | truncated (chemical_reactor.py:394-399);
                                             0: terminals = terminated (power_grid.py:239, robot_assembly.py:298) */
    int32_t reserved;
} nig_dataset_out_t;

/* stats block: NIG_STATS_SLOTS x 8 bytes on the device; slots < 24 are int64 counters, slots >= 24 are
 * fp64 sums. Summable across ranks (one NCCL all-reduce, SURVEY 8e). */
enum {
    NIG_ST_STEPS = 0, NIG_ST_EPISODES = 1, NIG_ST_TERMINATED = 2, NIG_ST_TRUNCATED = 3,
    NIG_ST_CRITICAL = 4, NIG_ST_VIOLATIONS = 5, NIG_ST_SUCCESSES = 6 /* episodes with return > 0 */,
    NIG_ST_EP_LEN_SUM = 7, NIG_ST_CON0 = 8 /* .. NIG_ST_CON0+7 per-constraint violation counts */,
    NIG_ST_EP_LEN_SQ = 16,
    NIG_ST_F_RETURN_SUM = 24, NIG_ST_F_RETURN_SQ = 25, NIG_ST_F_REWARD_SUM = 26
};

NIG_API int nig_abi_version(void);
NIG_API const char* nig_last_error(void);
NIG_API int nig_device_count(int* count);

/* env metadata: replaces reading state_dim/action_dim/safety_constraints/max_episode_steps off the
 * env object (environments/base.py:41-72, chemical_reactor.py:38-69, power_grid.py:53-79,
 * robot_assembly.py:56-82) */
NIG_API int nig_env_spec(int env_kind, nig_env_spec_t* out);

/* utils.make (utils.py:12-39) + IndustrialEnv.__init__ (base.py:22-72) for n_envs envs */
NIG_API int nig_create(const nig_config_t* cfg, nig_env_t** out);
NIG_API int nig_destroy(nig_env_t* env);
NIG_API int64_t nig_pitch(const nig_env_t* env);
NIG_API int64_t nig_num_envs(const nig_env_t* env);

/* add_safety_constraint / remove_safety_constraint (base.py:220-228) and SafetyWrapper (README.md:126-139) */
NIG_API int nig_set_constraints(nig_env_t* env, const nig_constraint_t* cons, int32_t n);

/* IndustrialEnv.reset (base.py:133-155) + _get_initial_state (chemical_reactor.py:89-107,
 * power_grid.py:90-110, robot_assembly.py:113-137). mask NULL = all envs; init_states NULL = draw. */
NIG_API int nig_reset(nig_env_t* env, const uint8_t* mask_dev, const float* init_states_dev, int32_t layout, void* stream);
NIG_API int nig_reset_host(nig_env_t* env, const uint8_t* mask, const float* init_states_aos, float* obs_aos_out);

/* IndustrialEnv.step (base.py:157-213) incl. _check_safety_constraints (:94-124), _dynamics,
 * _compute_reward, _is_done of the three envs */
NIG_API int nig_step(nig_env_t* env, const nig_step_io_t* io, void* stream);
/* same with HOST pointers (AoS, exact-size): H2D of the inputs, the kernel, D2H of the outputs */
NIG_API int nig_step_host(nig_env_t* env, const nig_step_io_t* io);

/* K fused steps with state in registers: the `for step: action = policy(obs); env.step(action)` loops of
 * performance_benchmark.py:106-133, utils.evaluate_with_safety (utils.py:82-125) and get_dataset */
NIG_API int nig_rollout(nig_env_t* env, const nig_rollout_t* r, void* stream);
/* nig_rollout that also records every step: the per-step tuple (obs, action, reward, terminated, truncated, info) of
 * `for t in range(K): env.step(policy(obs))` -- the caller's own gym vector-env loop that stores each step -- written by the one
 * fused launch into time-major device arrays. Everything nig_rollout does, the call does too, bit for bit, with the same
 * descriptor: state, episode words and returns, tick (+K), per-env reward_sum / viol_count / done_count (NIG_ROLLOUT_ACCUMULATE
 * included), the statistics block, the return extrema and the PID controller state; recording is a side output. Validation is
 * nig_rollout's (same statuses for the same descriptor); out == NULL is NIG_ERR_INVALID, a descriptor whose fields are all NULL
 * records nothing. NIG_ROLLOUT_USE_TMA is accepted and has no effect. One launch on `stream`; the device tick modes of
 * nig_use_device_tick apply as for nig_rollout (the call can be captured into a CUDA graph). Row (t, i) holds exactly what
 * nig_step writes for env i stepped with the recorded action at the same tick: obs[t] is nig_step's post-auto-reset obs of
 * step t - 1 (row 0: the state at the call); an inactive env (auto_reset == 0, already finished) keeps its state, reward 0,
 * flags NIG_F_INACTIVE, viol_mask 0. The kernel runs rollout_kernel's generic loop (or the MLP rollout's), not the
 * specialised throughput loops of nig_rollout. */
typedef struct nig_trajectory {
    /* device arrays, time-major, exact-size rows ([K][n][dim]: row t * n + i is env i at step t of this call, the layout of a
     * contiguous torch tensor [K, n, dim]); NULL = not recorded. Offsets are 64-bit: K * n * S may exceed 2^31. */
    float*   obs;         /* [K][n][S] s_t: the observation the policy acted on (row 0 = the state at the call) */
    float*   actions;     /* [K][n][A] the action handed to the env at step t, BEFORE the env's clip to [-1, 1] */
    float*   rewards;     /* [K][n]    */
    uint8_t* flags;       /* [K][n]    NIG_F_* bits */
    uint8_t* viol_mask;   /* [K][n]    bit k = constraint k violated on s_t */
    uint8_t* terminated;  /* [K][n]    0/1 */
    uint8_t* truncated;   /* [K][n]    0/1 */
    float*   next_obs;    /* [K][n][S] s' of the transition, before auto-reset (gym's final_observation) */
} nig_trajectory_t;
NIG_API int nig_rollout_record(nig_env_t* env, const nig_rollout_t* r, const nig_trajectory_t* out, void* stream);
/* total_steps steps of every env as ceil(total_steps / r->n_steps) fused launches (in-kernel policies only). On a large
 * population the envs are split into slices that advance on internal streams forked from and joined back to `stream`
 * (NIG_HOST_SLICES, default 8, >= 8,192 envs per slice): a slice's next launch fills the SMs another slice's tail leaves
 * idle, which a single sequence of whole-population launches cannot do. Results do not depend on the slicing. Per-env
 * outputs cover the whole call (or add to the arrays with NIG_ROLLOUT_ACCUMULATE). Asynchronous like nig_rollout.
 * A call pattern that repeats (same horizon, K, policy, output pointers, settings) is captured once as a CUDA graph on an
 * internal stream and replayed on `stream` from then on (2 driver calls per call instead of one per launch; NIG_STEPS_GRAPH=0
 * disables it; a caller that is itself capturing `stream` always gets the plain launch sequence). */
NIG_API int nig_rollout_steps(nig_env_t* env, const nig_rollout_t* r, int32_t total_steps, void* stream);

/* The same loops with HOST buffers: what performance_benchmark.py:106-133 / utils.evaluate_with_safety do per env in
 * Python, for every env of the handle in one call. Host arrays are exact-size ([n] or [n][dim]); the call runs
 * ceil(n_steps / steps_per_launch) fused launches and returns synchronised. With an in-kernel policy and at least
 * 16,384 envs the population is split into env slices (NIG_HOST_SLICES) that each take their states in, step and put their
 * results out on their own stream, so the PCIe traffic of one slice overlaps the stepping of the others; results do not
 * depend on it. Two data paths, chosen per call: DIRECT (every supplied array page-locked -- nig_host_alloc /
 * cudaHostAlloc / cudaHostRegister -- and 16-byte aligned; NIG_HOST_DIRECT=0 disables): the slices' own kernels read the
 * initial states from and write the results into the caller's arrays over PCIe, no staging, 8 slices; STAGED (anything else):
 * cudaMemcpyAsync through device buffers (true DMA when page-locked), 4 slices. With page-locked arrays the whole sliced
 * pipeline is one captured CUDA graph replayed per call (NIG_HOST_GRAPH=0 disables). Identical results either way.
 * Teacher-forced inputs (optional): init_states [n][S]; actions [T][A][n] with policy == NIG_POLICY_ACTIONS and
 * noise [T][NZ][n] (time-major, SoA per step -- the layout the kernel consumes; copied chunk by chunk,
 * double-buffered so the copy of chunk c+1 overlaps the launch of chunk c). */
typedef struct nig_rollout_host {
    int32_t n_steps;            /* T: total steps per env */
    int32_t steps_per_launch;   /* K fused steps per kernel launch; 0 = T; either way at most NIG_MAX_LAUNCH_STEPS (a longer
                                   horizon runs as several launches, whose fp32 reward sums are added launch by launch, as
                                   for any K < T) */
    int32_t policy;             /* NIG_POLICY_* */
    int32_t reset_first;        /* 1: IndustrialEnv.reset() of every env before stepping (drawn, or init_states) */
    const float* init_states;   /* in  [n][S] AoS or NULL */
    const float* actions;       /* in  [T][A][n] (NIG_POLICY_ACTIONS) or NULL */
    const float* noise;         /* in  [T][NZ][n] or NULL (in-kernel Philox) */
    nig_policy_params_t pp;
    float* reward_sum;          /* out [n] sum of rewards over the T steps (fp32; per launch in step order, launches added in order) */
    int32_t* viol_count;        /* out [n] constraint violations over the T steps */
    int32_t* done_count;        /* out [n] episodes finished over the T steps */
    float* final_obs;           /* out [n][S] AoS state after the last step (post auto-reset) */
    int64_t* counters24;        /* out [24] the stats block after the call (NULL ok) */
    double* sums8;              /* out [8] */
} nig_rollout_host_t;
NIG_API int nig_rollout_host(nig_env_t* env, const nig_rollout_host_t* r);

/* NIG_POLICY_MLP's network: validated against the env's S / A, converted and packed once into a handle-owned device buffer.
 * A network that fails validation leaves the previous one in place. Otherwise the call synchronises the device (a rollout
 * still running on any stream finishes with the old network), then drops the old network and the captured nig_rollout_steps /
 * nig_rollout_host graphs before it touches the device buffer; if the upload then fails (NIG_ERR_CUDA) the handle has no
 * network. The network is copied: changing the caller's arrays afterwards changes nothing. nig_rollout, nig_rollout_steps and nig_rollout_host then accept
 * NIG_POLICY_MLP (NIG_ERR_INVALID before a network is set; NIG_ERR_UNSUPPORTED with teacher-forced noise); nig_dataset and
 * nig_dataset_size do not (NIG_ERR_UNSUPPORTED). */
NIG_API int nig_set_mlp_policy(nig_env_t* env, const nig_mlp_t* mlp);

/* zero the persistent controller state of NIG_POLICY_BASELINE / NIG_BASELINE_PID (integral, previous error) */
NIG_API int nig_reset_policy_state(nig_env_t* env, void* stream);

/* get_dataset (chemical_reactor.py:324-420): n_episodes episodes of <= n_steps steps each with the given
 * policy, written episode-contiguously in D4RL layout on the device. Episodes are independent envs with
 * global ids env_id_offset + [0, n_episodes). *n_written receives the transition count. */
NIG_API int nig_dataset(nig_env_t* env, int64_t n_episodes, int32_t n_steps, int32_t policy,
                        const nig_policy_params_t* pp, const nig_dataset_out_t* out, int64_t* n_written, void* stream);
/* length probe only (pass 1 of nig_dataset): total transitions the same call would write */
NIG_API int nig_dataset_size(nig_env_t* env, int64_t n_episodes, int32_t n_steps, int32_t policy,
                             const nig_policy_params_t* pp, int64_t* n_transitions, void* stream);

/* checkpoint / teacher forcing: env.state, env.current_step, env.violation_count (base.py:50-57). The episode word keeps the
 * step in 16 bits and the violation count in 15, saturating at 32,767 (the kernels saturate a running count the same way; the
 * per-env viol_count of the rollouts and the statistics block count every violation). Ranges of an import: ep_step in
 * [0, 65535], ep_viol >= 0 (above 32,767 it saturates). nig_set_state_host rejects values outside them (NIG_ERR_INVALID,
 * nothing imported); nig_set_state, whose arrays are on the device, clamps them into range. */
NIG_API int nig_get_state(nig_env_t* env, float* state_dev, int32_t layout, int32_t* ep_step_dev, int32_t* ep_viol_dev, uint8_t* done_dev, void* stream);
NIG_API int nig_set_state(nig_env_t* env, const float* state_dev, int32_t layout, const int32_t* ep_step_dev, const int32_t* ep_viol_dev, const uint8_t* done_dev, void* stream);
NIG_API int nig_get_state_host(nig_env_t* env, float* state_aos, int32_t* ep_step, int32_t* ep_viol, uint8_t* done);
NIG_API int nig_set_state_host(nig_env_t* env, const float* state_aos, const int32_t* ep_step, const int32_t* ep_viol, const uint8_t* done);
/* raw device views (zero-copy wrapping by the host language) */
NIG_API int nig_state_ptr(nig_env_t* env, float** state_dev_soa, uint32_t** ep_word_dev);
NIG_API int nig_get_tick(const nig_env_t* env, uint32_t* tick, uint32_t* epoch);
NIG_API int nig_set_tick(nig_env_t* env, uint32_t tick, uint32_t epoch);
/* CUDA-graph capture: a captured graph replays the SAME kernel arguments, so the batched-step counter that keys the random
 * streams must not be one. Two device-resident modes (enable BEFORE capturing; nig_get_tick / nig_set_tick keep working,
 * they synchronise):
 *   1  every launch reads the counter from device memory and its last CTA advances it. Simple, any captured sequence
 *      replays correctly; costs a fence + an atomic round trip at the end of every launch.
 *   2  the device word is a BASE; every launch carries its offset from it (the launches since the last commit) as an
 *      argument, nothing is advanced per launch, and the tick is known before the previous launch has finished (the
 *      single-step kernel draws its noise while the previous step drains: programmatic dependent launch). The captured
 *      sequence must END with nig_commit_ticks(env, stream), which moves the base on by the sequence's length; without it
 *      every replay would repeat the same draws.
 *   0  back to the host-side counter. */
NIG_API int nig_use_device_tick(nig_env_t* env, int32_t mode);
NIG_API int nig_commit_ticks(nig_env_t* env, void* stream);
/* reset(seed=...) made effective (the reference ignores it, base.py:135; SURVEY Appendix E.3): re-keys the random streams
 * AND rewinds the handle's tick / epoch to 0, so that set_seed(s) + reset gives the same states and noise every time */
NIG_API int nig_set_seed(nig_env_t* env, uint64_t seed);

/* violation / return counters (info["violations"], info["total_violations"], evaluate_with_safety's
 * aggregates utils.py:128-152). The device block can be all-reduced in place (NCCL sum over int64/fp64). */
NIG_API int nig_stats_ptr(nig_env_t* env, void** stats_dev);
/* The plain single-step kernel adds its counters to 128 shard copies of the block (one hot block serialised ~1,600
 * reductions per launch in L2 at 65,536 envs); nig_read_stats, nig_allreduce_stats and the *_host calls fold the shards in
 * first. A caller that reads the raw device block of nig_stats_ptr itself queues nig_fold_stats on its stream before. */
NIG_API int nig_fold_stats(nig_env_t* env, void* stream);
NIG_API int nig_read_stats(nig_env_t* env, int64_t* counters24, double* sums8);
NIG_API int nig_clear_stats(nig_env_t* env, void* stream);

/* The path's only collective (SURVEY 8e; the aggregation utils.py:128-152 does over one env, over every shard): sums the
 * device stats block over the ranks of an NCCL communicator, in place, as ONE grouped launch on `stream` -- 24 int64
 * counters (SUM: exact and order independent), 8 fp64 sums (SUM) and the two order-preserving return-extremum keys (MAX).
 * `nccl_comm` is an ncclComm_t: any communicator whose ranks own the shards (torch.distributed's:
 * ProcessGroupNCCL._comm_ptr(); or one made with the three helpers below, which need nothing but a way to hand rank 0's
 * 128-byte id to the other ranks). NCCL is dlopen()ed on first use (libnccl.so.2); without it these four calls return
 * NIG_ERR_UNSUPPORTED and everything else works. */
NIG_API int nig_allreduce_stats(nig_env_t* env, void* nccl_comm, void* stream);
NIG_API int nig_nccl_unique_id(void* id128);                                  /* rank 0: ncclGetUniqueId -> 128 bytes */
NIG_API int nig_nccl_comm_init(void** nccl_comm, int32_t n_ranks, const void* id128, int32_t rank, int32_t device);
NIG_API int nig_nccl_comm_destroy(void* nccl_comm);

/* smallest / largest return among the episodes finished inside nig_rollout / nig_rollout_host since the last
 * nig_clear_stats (return_min / return_max of evaluate_with_safety, utils.py:131-132). Opt-in per handle with
 * nig_track_extrema(env, 1): the rollout then runs the kernel flavour that carries the two running extrema (measured
 * 2 % slower than the plain one, which is why it is not always on; teacher-forced noise has no such flavour ->
 * NIG_ERR_UNSUPPORTED). Two order-preserving int64 keys on the device (0 = none yet), kept outside the summable stats
 * block: ranks combine them with one MAX all-reduce, then decode. Accurate to the last mantissa bit of the fp64 return. */
NIG_API int nig_track_extrema(nig_env_t* env, int32_t on);
/* The running return of every env's current episode is kept in one fp64 accumulator per env, shared by nig_step and
 * nig_rollout, so that the two can be mixed freely on one handle: finished-episode statistics (return / length sums,
 * successes -- utils.py:128-152) count every episode whichever call ended it, and nig_set_state with an episode step
 * counter restarts the accumulator. On by default. nig_track_returns(env, 0) makes the SINGLE-STEP kernels skip the
 * accumulator (16 B less HBM traffic per env-step: the plain gym loop of performance_benchmark.py:106-133 keeps no
 * returns either); statistics then cover only episodes that ran entirely inside nig_rollout calls. */
NIG_API int nig_track_returns(nig_env_t* env, int32_t on);
/* The single-step kernels also add every step to the device counter block (steps, episodes, violations per constraint, ...:
 * nig_read_stats), which IndustrialEnv.step itself does not have -- its per-env outputs (reward, flags, violation mask, the
 * episode word behind current_step / violation_count) are complete without it. On by default. nig_track_step_stats(env, 0)
 * makes nig_step / nig_step_host skip the counters: at 65,536 envs the warp reductions and the atomics at the tail of the
 * kernel are 1.1 us of a 3.8 us launch. The fused rollouts always count. */
NIG_API int nig_track_step_stats(nig_env_t* env, int32_t on);
NIG_API int nig_extrema_ptr(nig_env_t* env, void** keys2_dev);
NIG_API int nig_read_extrema(nig_env_t* env, double* ret_min, double* ret_max, int32_t* have);
NIG_API int nig_decode_extrema(const int64_t* keys2, double* ret_min, double* ret_max, int32_t* have);

NIG_API int nig_sync(nig_env_t* env);
/* page-locked host buffers for the *_host calls (the copies are then true async DMA) */
NIG_API int nig_host_alloc(size_t bytes, void** out);
NIG_API int nig_host_free(void* p);
/* kernels launched by this handle since creation (bench.py's gpu_launches claim) */
NIG_API int64_t nig_launch_count(const nig_env_t* env);
/* measured-peak probe: issues a dependent-free stream of unfused fp32 add/mul and returns ops per launch */
NIG_API int nig_fp32_probe(int device, int32_t iters, double* ops, void* stream);

/* self-test of the guarded fast divisions of the step kernels against IEEE division, on the device: n Philox-drawn
 * operand sets (all-exponent pairs, physics-regime pairs, every constant divisor); *mismatches must come back 0 */
NIG_API int nig_selftest_division(int device, int64_t n, uint64_t seed, int64_t* mismatches, int64_t* accepted);

/* self-test of the inverse-CDF Gaussian of the math spec (csrc/nig_math.cuh spec_normal): two wrapping checksums over the
 * bit patterns of normal(first + k * stride), k < count -- sums2[0] = sum bits, sums2[1] = sum bits * (k + 1). The CPU
 * oracle computes the same sums; the whole 2^32-word domain is (first 0, stride 1, count 2^32). */
NIG_API int nig_selftest_normal(int device, uint32_t first, uint32_t stride, int64_t count, uint64_t* sums2);

/* teacher-forced replay of the in-kernel policies (test hook): the get_dataset controller / random branches
 * (chemical_reactor.py:364-390, power_grid.py:216-232, robot_assembly.py:266-291; policy = NIG_POLICY_PCTRL) and the
 * benchmark baseline controllers (benchmarks/baseline_agents.py:46-114; NIG_POLICY_BASELINE) evaluated by the device code on
 * HOST arrays of caller-supplied states and random inputs instead of the in-kernel draws: states [n_steps][n][S],
 * coin [n_steps][n] (the np.random.random() of the mix, NULL = 0.5), z [n_steps][n][8] standard normals,
 * u [n_steps][n][8] uniforms in [-1, 1] (NULL = zeros) -> actions [n_steps][n][A] as get_dataset stores them. Env i keeps
 * its PID integral / previous error across the n_steps rows like one agent object does. */
NIG_API int nig_selftest_policy(int device, int32_t env_kind, int32_t policy, const nig_policy_params_t* pp, int64_t n, int32_t n_steps,
                                const float* states, const float* coin, const float* z, const float* u, float* actions);

/* test hook of NIG_POLICY_MLP: the handle's network evaluated by the rollout's own device function and 128-row tiling on
 * HOST arrays: obs [n][S] -> actions [n][A] (before the env's clip). Synchronous. */
NIG_API int nig_selftest_mlp(nig_env_t* env, const float* obs, int64_t n, float* actions);

#ifdef __cplusplus
}
#endif
#endif /* NIG_B200_H */
