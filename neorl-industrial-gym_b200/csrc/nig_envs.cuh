// nig_envs.cuh -- per-env physics of the IndustrialEnv step path as register-resident device functions.
//
// One struct per reference env, each restating (NOT translating: the reference is scalar numpy
// with Python control flow, one env per object) the four hooks of environments/base.py:74-92:
//   _get_initial_state -> reset(), _dynamics -> dynamics(), _compute_reward -> reward(),
//   _is_done -> is_done(), plus the env's constraint check_fns -> builtin().
// Arithmetic contract (SURVEY.md Appendix A/B/C): IEEE binary32 round-to-nearest, NO contraction,
// evaluated in the reference's order; only the explicit intrinsics below are used so no compiler
// flag can change the rounding. Flags / masks / counters are therefore bit-exact w.r.t. numpy.
#pragma once
#include "../../include/nig_b200.h"
#include "nig_math.cuh"

namespace nig {

__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// numpy pairwise_sum for n == 8 (eight accumulators folded as a tree); SURVEY Appendix B
__device__ __forceinline__ float pairwise8(const float (&x)[8])
{
    return add(add(add(x[0], x[1]), add(x[2], x[3])), add(add(x[4], x[5]), add(x[6], x[7])));
}
__device__ __forceinline__ double pairwise8d(const double (&x)[8])
{
    return dadd(dadd(dadd(x[0], x[1]), dadd(x[2], x[3])), dadd(dadd(x[4], x[5]), dadd(x[6], x[7])));
}

// action_space.sample() of the envs without a fused noise / policy block: blocks 0.. of the POLICY stream, one word per action
template <int A>
__device__ __forceinline__ void uniform_actions_policy_stream(const Rng& key, uint32_t env, uint32_t tick, float (&a)[A])
{
#pragma unroll
    for (int j = 0; j < (A + 3) / 4; ++j) {
        const uint4 w = rng_words(key, env, tick, STREAM_POLICY, (uint32_t)j);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * j + q < A) a[4 * j + q] = u_sym(ww[q]);
    }
}

// ================================================================================================
// ChemicalReactor-v0  (environments/chemical_reactor.py)
// ================================================================================================
struct Reactor {
    static constexpr int KIND = 0, S = 12, A = 3, NZ = 2, NB = 3, MAX_STEPS = 500;
    static constexpr bool FAST_DIV = true;           // 5 divisions by constants per step (dynamics 3, reward 2)
    static constexpr uint32_t CRIT_MASK = 0x3;       // temperature_limit, pressure_limit (:38-52)
    using acc_t = float;                              // reward stays np.float32 upstream
    __device__ static constexpr float penalty(int k) { return k == 0 ? -100.0f : (k == 1 ? -50.0f : -25.0f); }

    // ONE Philox block per step, (env, tick, NOISE, 0): words x, y -> the two process-noise normals of the step; words z, w
    // are the action_space.sample() of the uniform-random policy (uniform_from_words). (The first builds used half a
    // noise block + a whole policy block per step: 1.5 blocks; IMAD.WIDE issues at a quarter of the FMA-pipe rate on
    // sm_100a -- tools/pipe_probe.cu -- so a Philox block is 56 pipe cycles, not 28 instructions.)
    struct NoiseGen {
        uint4 w;
        __device__ __forceinline__ void get(const Rng& key, uint32_t env, uint32_t tick, float (&nz)[NZ])
        {
            w = rng_words(key, env, tick, STREAM_NOISE, 0u);
            float za, zb;
            normal_pair(key.tab, w.x, w.y, za, zb);
            nz[0] = mul(0.1f, za);      // np.random.normal(0, temp_noise_std / 10)      (:149)
            nz[1] = mul(500.0f, zb);    // np.random.normal(0, pressure_noise_std / 10)  (:159)
        }
        __device__ static __forceinline__ void get_single(const Rng& key, uint32_t env, uint32_t tick, float (&nz)[NZ])
        {
            NoiseGen g;
            g.get(key, env, tick, nz);
        }
    };
    // action_space.sample() (performance_benchmark.py:118) from words z, w of the step's block: a0 / a1 from bits 21..0 of
    // z / w, a2 from the two 10-bit tops; the bits go straight into the mantissa of a float in [4, 6) / [16, 18) (one LOP3
    // each, no int -> float conversion) and one exact add maps it to [-1, 1): a0, a1 = v * 2^-21 - 1, a2 = v * 2^-19 - 1.
    // (The same values as fma(1 + v * 2^-23, 4 or 16, -5 or -17): the sums are multiples of 2^-21 / 2^-19 below 2 in
    // magnitude, exact in binary32, and an add needs no second constant in a register.)
    __device__ static __forceinline__ void uniform_from_words(uint32_t wz, uint32_t ww, float (&a)[A])
    {
        a[0] = __fadd_rn(__uint_as_float((wz & 0x3fffffu) | 0x40800000u), -5.0f);
        a[1] = __fadd_rn(__uint_as_float((ww & 0x3fffffu) | 0x40800000u), -5.0f);
        const uint32_t v2 = __funnelshift_l(ww, wz >> 22, 10);          // (wz[31:22] << 10) | ww[31:22]
        a[2] = __fadd_rn(__uint_as_float(v2 | 0x41800000u), -17.0f);
    }
    __device__ static __forceinline__ void uniform_actions(const Rng& key, uint32_t env, uint32_t tick, float (&a)[A])
    {
        const uint4 w = rng_words(key, env, tick, STREAM_NOISE, 0u);    // (the same block as NoiseGen::get: CSE'd when both are live)
        uniform_from_words(w.z, w.w, a);
    }

    // _get_initial_state (:89-107) drawn from the RESET stream: 8 standard normals = word pairs 0..3 of
    // Philox blocks (epoch << 8) | {0, 1}
    // measured on B200 (tools/steady_step.py, tools/rollout_sweep.py): the single-step kernels gain 6 % at 16M envs
    // (0.86 -> 0.92 of the HBM peak), the fused rollout loses 2 % (one extra ballot per step) and keeps Env::reset()
    static constexpr bool COOP_RESET = true;
    static constexpr int COOP_BLOCKS = 0;
    static constexpr bool COOP_FK = false;
    static constexpr int RESET_NORMALS = 8;
    // resident CTAs per SM the fused rollout is compiled for (register cap): measured, more resident warps LOSE for
    // the reactor (7.0 -> 6.8 -> 6.3e10 env-steps/s at 1M envs for 4 / 6 / 8 CTAs)
    static constexpr int ROLLOUT_MIN_CTAS = 1;
    static constexpr bool TAB_SMEM = false;          // 2 normals per step: the L1-cached global table is as fast, no staging prologue
    // the fused rollout reads a shared-memory copy of the table: LEA.HI + LDS.128 [R.X16] instead of LEA.HI + IMAD.WIDE (a
    // quarter-rate instruction) + LDG per normal; measured +5 % at 65,536 envs, +1.4 % at 1M (gpurun_out r2_ab1)
    static constexpr bool ROLLOUT_TAB_SMEM = true;
    static constexpr int STEP_MIN_CTAS = 1;
    __device__ static __forceinline__ void reset_from_normals(const float (&z)[8], float (&s)[S])
    {
        s[0] = add(320.0f, mul(2.0f, z[0]));
        s[1] = add(253312.5f, mul(10000.0f, z[1]));
        s[2] = add(50.0f, mul(5.0f, z[2]));
        s[3] = add(30.0f, mul(3.0f, z[3]));
        s[4] = add(0.5f, mul(0.1f, z[4]));
        s[5] = add(95.0f, mul(2.0f, z[5]));
        s[6] = add(295.0f, mul(1.0f, z[6]));
        s[7] = 0.0f; s[8] = 0.0f; s[9] = 0.0f;
        s[10] = add(60.0f, mul(5.0f, z[7]));
        s[11] = 0.0f;
    }
    // pair of normals `pair` (0..3) of the 8: the unit of work of the warp-cooperative reset (one pair per lane)
    __device__ static __forceinline__ void reset_pair(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, uint32_t pair,
                                                      float& z0, float& z1)
    {
        const uint4 w = rng_words(key, env, tick, STREAM_RESET, (epoch << 8) | (pair >> 1));
        normal_pair(key.tab, (pair & 1u) ? w.z : w.x, (pair & 1u) ? w.w : w.y, z0, z1);
    }
    __device__ static __forceinline__ void reset(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, float (&s)[S])
    {
        float z[8];
        rng_normals4(key, env, tick, STREAM_RESET, (epoch << 8) | 0u, reinterpret_cast<float (&)[4]>(z[0]));
        rng_normals4(key, env, tick, STREAM_RESET, (epoch << 8) | 1u, reinterpret_cast<float (&)[4]>(z[4]));
        reset_from_normals(z, s);
    }

    // constraint check_fns (:292-305): true = satisfied
    __device__ static __forceinline__ bool builtin(int id, const float (&s)[S], const float (&)[A])
    {
        return id == 0 ? (s[0] <= 350.0f) : id == 1 ? (s[1] <= 506625.0f) : (20.0f <= s[10] && s[10] <= 90.0f);
    }

    // _dynamics (:109-226). `div` performs the divisions by constants (DivExact / DivFast, nig_math.cuh)
    template <class Div>
    __device__ static __forceinline__ void dynamics(const float (&s)[S], const float (&a)[A], const float (&nz)[NZ], float (&o)[S], Div& div)
    {
        const float temp = s[0], pressure = s[1], cool = s[2], feed = s[3], conc = s[4], cat = s[5];
        const float hx = s[6], relief = s[7], estop = s[8], alarm = s[9], level = s[10], bt = s[11];
        const bool manual = estop < 0.5f;                                     // :126
        const float hp = manual ? mul(a[0], 50000.0f) : -10000.0f;            // :127 / :132
        const float cadj = manual ? mul(a[1], 0.1f) : 0.1f;                   // :128 / :133
        const float fadj = manual ? mul(a[2], 0.1f) : -0.1f;                  // :129 / :134
        const float kca = mul(mul(0.1f, conc), NIG_CDIV(div, cat, 100.0f));            // k * conc * (cat / 100)
        const float rh = mul(kca, 10000.0f);                                  // :137-140
        const float ch = mul(mul(mul(cool, 100.0f), sub(temp, hx)), 0.1f);    // :141
        float dT = NIG_CDIV(div, sub(add(hp, rh), ch), 418000.0f);                     // :143-146 (4.18e3*1000*0.1)
        dT = add(dT, nz[0]);                                                  // :149
        const float nT = add(temp, mul(dT, 0.1f));                            // :151
        const float pfr = mul(mul(conc, 0.1f), 1000.0f);                      // :156
        float nP = add(mul(pressure, div.vdiv(nT, temp)), mul(pfr, 0.1f));        // :155, :158
        nP = add(nP, nz[1]);                                                  // :159
        const float nrv = py_clamp(add(relief, mul(sub(nP, 506625.0f), 0.001f)), 0.0f, 100.0f);  // :162-163
        if (nrv > 0.0f) {                                                     // :166-168
            const float x = sub(nP, mul(mul(nrv, 0.01f), 10000.0f));
            nP = (x > 101325.0f) ? x : 101325.0f;
        }
        const float ncool = py_clamp(add(cool, cadj), 10.0f, 100.0f);         // :171
        const float feed_v = add(feed, fadj);                                 // :172
        const float nfeed = py_clamp(feed_v, 5.0f, 50.0f);
        const float ex = spec_expf(NIG_CDIV(div, -sub(nT, 320.0f), 20.0f));            // :177
        const float rr = mul(kca, ex);                                        // :175-178
        // :180 -- a clamped feed is the Python int 5 / 50 upstream, so 5*0.001 is a Python float (0.005)
        // rounded to binary32, which differs from float32(5)*float32(0.001) in the last bit.
        float fdil = mul(nfeed, 0.001f);
        fdil = (feed_v > 5.0f) ? fdil : 0x1.47ae14p-8f;
        fdil = (feed_v < 50.0f) ? fdil : 0x1.99999ap-5f;
        const float cv = add(conc, mul(sub(rr, fdil), 0.1f));                 // :181-182
        const float nconc = (cv > 0.0f) ? cv : 0.0f;
        const float catv = sub(cat, (nT > 340.0f) ? 0.001f : 0.0001f);        // :185-186
        const float ncat = (catv > 50.0f) ? catv : 50.0f;
        const float nhx = add(hx, mul(mul(0.1f, sub(add(290.0f, mul(cool, 0.1f)), hx)), 0.1f));  // :189-190
        float nestop = estop, nalarm = alarm;                                 // :193-201
        if (nT > 345.0f || nP > 480000.0f) nalarm = 1.0f;
        if (nT > 350.0f || nP > 506625.0f) { nestop = 1.0f; nalarm = 1.0f; }
        const float lchg = mul(sub(nfeed, 20.0f), 0.1f);                      // :204
        const float nlevel = py_clamp(add(level, mul(lchg, 0.1f)), 0.0f, 100.0f);   // :205
        o[0] = nT; o[1] = nP; o[2] = ncool; o[3] = nfeed; o[4] = nconc; o[5] = ncat;
        o[6] = nhx; o[7] = nrv; o[8] = nestop; o[9] = nalarm; o[10] = nlevel; o[11] = add(bt, 0.1f);  // :208
    }

    // _compute_reward (:228-270)
    template <class Div>
    __device__ static __forceinline__ acc_t reward(const float (&ns)[S], const float (&a)[A], Div& div)
    {
        float r = add(0.0f, mul(ns[4], 100.0f));                                   // :238-241
        r = sub(r, mul(fabsf(sub(ns[0], 320.0f)), 0.5f));                          // :244-245
        r = sub(r, mul(NIG_CDIV(div, fabsf(sub(ns[1], 253312.5f)), 1000.0f), 0.1f));        // :248-249
        r = add(r, mul(NIG_CDIV(div, ns[5], 100.0f), 10.0f));                               // :252
        const bool band = (30.0f <= ns[10]) && (ns[10] <= 80.0f);                  // :255-258
        r = band ? add(r, 5.0f) : sub(r, mul(fabsf(sub(ns[10], 55.0f)), 0.2f));
        if (ns[9] > 0.5f) r = sub(r, 50.0f);                                       // :261-262
        if (ns[8] > 0.5f) r = sub(r, 200.0f);                                      // :263-264
        const float asum = add(add(fabsf(a[0]), fabsf(a[1])), fabsf(a[2]));        // :267
        return sub(r, mul(asum, 0.1f));                                            // :268
    }

    // _is_done (:272-290)
    __device__ static __forceinline__ bool is_done(const float (&s)[S])
    {
        return (s[8] > 0.5f) || (s[10] < 5.0f) || (s[10] > 95.0f) || (s[11] > 50.0f);
    }

    // get_dataset controller branch (:366-385): a_j = g0_j*(T-320)/50 + g1_j*(level-55)/50 + sigma_j*N(0,1)
    // policy_ctrl_from: the arithmetic for given standard normals z (the draw is separated so that the reference's own
    // get_dataset transitions can be replayed teacher-forced, tests/golden/policy_forced.npz)
    __device__ static __forceinline__ void policy_ctrl_from(const nig_policy_params_t& pp, const float (&s)[S], const float (&z)[8],
                                                            const float (&)[4], float (&a)[A])
    {
        DivExact div;    // the controller branch is taken by a subset of the lanes: keep the IEEE division here
        const float te = NIG_CDIV(div, sub(s[0], 320.0f), 50.0f);
        const float le = NIG_CDIV(div, sub(s[10], 55.0f), 50.0f);
#pragma unroll
        for (int k = 0; k < A; ++k)
            a[k] = add(add(mul(pp.gain[k][0], te), mul(pp.gain[k][1], le)), mul(pp.sigma[k], z[k]));
    }
    __device__ static __forceinline__ void policy_ctrl(const Rng& key, const nig_policy_params_t& pp, uint32_t env, uint32_t tick,
                                                       const float (&s)[S], float (&a)[A])
    {
        float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const float u[4] = {0.f, 0.f, 0.f, 0.f};
        rng_normals4(key, env, tick, STREAM_POLICY, 1u, reinterpret_cast<float (&)[4]>(z[0]));
        policy_ctrl_from(pp, s, z, u, a);
    }
};

// ================================================================================================
// PowerGrid-v0  (environments/power_grid.py)
// ================================================================================================
struct Grid {
    static constexpr int KIND = 1, S = 32, A = 8, NZ = 23, NB = 3, MAX_STEPS = 1000;
    static constexpr bool FAST_DIV = true;           // one fp32 division by 5 per step
    static constexpr bool COOP_RESET = false;
    static constexpr uint32_t CRIT_MASK = 0x3;       // frequency_stability, voltage_limits (:53-65)
    using acc_t = double;                             // _compute_reward returns a Python float (:177)
    __device__ static constexpr float penalty(int k) { return k == 0 ? -50.0f : (k == 1 ? -30.0f : -20.0f); }
    __device__ static constexpr float base_load(int i)
    {   // :82
        return i == 0 ? 50.f : i == 1 ? 60.f : i == 2 ? 45.f : i == 3 ? 55.f : i == 4 ? 40.f : i == 5 ? 65.f : i == 6 ? 35.f : 50.f;
    }
    __device__ static constexpr double gen_cost(int i)
    {   // :88 (int64 array -> the cost term is fp64 upstream)
        return i == 0 ? 25. : i == 1 ? 30. : i == 2 ? 28. : i == 3 ? 35. : i == 4 ? 32. : i == 5 ? 27. : i == 6 ? 40. : 33.;
    }

    struct NoiseGen {
        // draw order V(8) sigma .005, load(8) sigma 1, flow(7) sigma 2  (:136, :140, :144)
        __device__ __forceinline__ void get(const Rng& key, uint32_t env, uint32_t tick, float (&nz)[NZ])
        {
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                float z[4];
                rng_normals4(key, env, tick, STREAM_NOISE, (uint32_t)j, z);
                const float sg = j < 2 ? 0.005f : (j < 4 ? 1.0f : 2.0f);
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (4 * j + q < NZ) nz[4 * j + q] = mul(sg, z[q]);
            }
        }
        __device__ static __forceinline__ void get_single(const Rng& key, uint32_t env, uint32_t tick, float (&nz)[NZ])
        {
            NoiseGen g;
            g.get(key, env, tick, nz);
        }
    };

    __device__ static __forceinline__ void uniform_actions(const Rng& key, uint32_t env, uint32_t tick, float (&a)[A])
    {
        uniform_actions_policy_stream<A>(key, env, tick, a);
    }

    // _get_initial_state (:90-110): 8 Philox blocks of the RESET stream -- blocks 0,1 voltages ~ N(1, .01), 2,3
    // generation ~ N(base_load, 2), 4,5 loads = base_load * U(.8, 1.2), 6,7 line flows ~ N(0, 10). One block (4 raw
    // values) is the unit of work of the warp-cooperative reset.
    // 206 registers uncapped = 2 resident CTAs per SM; capped at 168 (3 CTAs, 24 B of spills): +15 % at 1M envs, 4 CTAs (128
    // registers) no better
    static constexpr int ROLLOUT_MIN_CTAS = 3;
    static constexpr bool TAB_SMEM = true;           // 23 normals per step: shared-memory copy of the normal table (+7 %)
    static constexpr bool ROLLOUT_TAB_SMEM = true;
    static constexpr int STEP_MIN_CTAS = 4;          // single step: 146 -> 128 registers, 3 -> 4 CTAs per SM, +11 % (5, 6: worse)
    static constexpr int COOP_BLOCKS = 8;
    static constexpr bool COOP_FK = false;
    __device__ static __forceinline__ void reset_block(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, uint32_t j, float (&v)[4])
    {
        if (j == 4u || j == 5u) {
            const uint4 w = rng_words(key, env, tick, STREAM_RESET, (epoch << 8) | j);
            v[0] = u_sym(w.x); v[1] = u_sym(w.y); v[2] = u_sym(w.z); v[3] = u_sym(w.w);
        } else rng_normals4(key, env, tick, STREAM_RESET, (epoch << 8) | j, v);
    }
    __device__ static __forceinline__ void reset_from_values(const float (&v)[32], float (&s)[S])
    {
        s[0] = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            s[1 + i] = add(1.0f, mul(0.01f, v[i]));
            s[9 + i] = add(base_load(i), mul(2.0f, v[8 + i]));
            s[17 + i] = mul(base_load(i), add(1.0f, mul(0.2f, v[16 + i])));
            if (i < 7) s[25 + i] = mul(10.0f, v[24 + i]);
        }
    }
    __device__ static __forceinline__ void reset(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, float (&s)[S])
    {
        float v[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) reset_block(key, env, tick, epoch, (uint32_t)j, reinterpret_cast<float (&)[4]>(v[4 * j]));
        reset_from_values(v, s);
    }

    __device__ static __forceinline__ bool builtin(int id, const float (&s)[S], const float (&a)[A])
    {
        if (id == 0) return fabsf(s[0]) < 0.5f;                                  // :10-14
        bool ok = true;
        if (id == 1) {                                                           // :17-21
#pragma unroll
            for (int i = 0; i < 8; ++i) ok = ok && (s[1 + i] >= 0.95f) && (s[1 + i] <= 1.05f);
        } else {                                                                 // :24-30
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float g = add(s[9 + i], a[i]); ok = ok && (g >= 0.0f) && (g <= 100.0f); }
        }
        return ok;
    }

    template <class Div>
    __device__ static __forceinline__ void dynamics(const float (&s)[S], const float (&a)[A], const float (&nz)[NZ], float (&o)[S], Div& div)
    {   // _dynamics (:112-153)
        float gen[8], load[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float g = add(s[9 + i], a[i]);                                       // :124 np.clip(gen + a, 0, 100)
            g = g < 0.0f ? 0.0f : g;
            g = g > 100.0f ? 100.0f : g;
            gen[i] = g; load[i] = s[17 + i];
        }
        const float imb = sub(pairwise8(gen), pairwise8(load));                  // :127-129
        const float fd = NIG_CDIV(div, add(mul(-1.0f, s[0]), imb), 5.0f);                 // :132
        o[0] = add(s[0], mul(fd, 0.1f));                                         // :133
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            o[1 + i] = add(s[1 + i], nz[i]);                                     // :136-137
            o[9 + i] = gen[i];
            const float l = add(s[17 + i], nz[8 + i]);                           // :140-141
            o[17 + i] = (l > 0.0f) ? l : ((l != l) ? l : 0.0f);
        }
#pragma unroll
        for (int i = 0; i < 7; ++i) o[25 + i] = add(s[25 + i], nz[16 + i]);      // :144
    }

    template <class Div>
    __device__ static __forceinline__ acc_t reward(const float (&ns)[S], const float (&a)[A], Div&)
    {   // _compute_reward (:155-177): fp32 terms, fp64 cost term, summed left to right
        const float fr = mul(-100.0f, mul(ns[0], ns[0]));                        // :162
        float d2[8], a2[8]; double cg[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float d = fabsf(sub(ns[1 + i], 1.0f));
            d2[i] = mul(d, d);                                                   // :165-166
            a2[i] = mul(a[i], a[i]);                                             // :173
            cg[i] = dmul(gen_cost(i), (double)ns[9 + i]);                        // :169
        }
        const float vr = mul(-50.0f, pairwise8(d2));
        const double ec = ddiv_const(-pairwise8d(cg), 1000.0, 1.0 / 1000.0);     // :170
        const float ap = mul(-5.0f, pairwise8(a2));
        return dadd(dadd((double)add(fr, vr), ec), (double)ap);                  // :175
    }

    __device__ static __forceinline__ bool is_done(const float (&s)[S])
    {   // :179-192
        bool d = fabsf(s[0]) > 1.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) d = d || (s[1 + i] < 0.9f) || (s[1 + i] > 1.1f);
        return d;
    }

    // get_dataset heuristics (:216-232): a_j = g0_j*freq_dev + g1_j*(sum load - sum gen)/8 + sigma_j*N(0,1)
    __device__ static __forceinline__ void policy_ctrl_from(const nig_policy_params_t& pp, const float (&s)[S], const float (&z)[8],
                                                            const float (&)[4], float (&a)[A])
    {
        float gen[8], load[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { gen[i] = s[9 + i]; load[i] = s[17 + i]; }
        const float imb8 = fdiv(sub(pairwise8(load), pairwise8(gen)), 8.0f);
#pragma unroll
        for (int k = 0; k < A; ++k)
            a[k] = add(add(mul(pp.gain[k][0], s[0]), mul(pp.gain[k][1], imb8)), mul(pp.sigma[k], z[k]));
    }
    __device__ static __forceinline__ void policy_ctrl(const Rng& key, const nig_policy_params_t& pp, uint32_t env, uint32_t tick,
                                                       const float (&s)[S], float (&a)[A])
    {
        float z[8];
        const float u[4] = {0.f, 0.f, 0.f, 0.f};
        rng_normals4(key, env, tick, STREAM_POLICY, 1u, reinterpret_cast<float (&)[4]>(z[0]));
        rng_normals4(key, env, tick, STREAM_POLICY, 2u, reinterpret_cast<float (&)[4]>(z[4]));
        policy_ctrl_from(pp, s, z, u, a);
    }
};

// ================================================================================================
// RobotAssembly-v0  (environments/robot_assembly.py) -- FK and reward in fp64 like the reference
// ================================================================================================
struct Robot {
    static constexpr int KIND = 2, S = 24, A = 7, NZ = 0, NB = 3, MAX_STEPS = 1000;
    static constexpr bool FAST_DIV = false;          // fp64 divisions only
    static constexpr bool COOP_RESET = false;
    static constexpr int COOP_BLOCKS = 0;
    static constexpr bool COOP_FK = true;            // warp-cooperative forward kinematics of the reset (coop_reset_fk)
    static constexpr bool TAB_SMEM = false;          // normals only in reset / policy draws
    static constexpr bool ROLLOUT_TAB_SMEM = false;
    static constexpr int ROLLOUT_MIN_CTAS = 4;       // 177 -> 128 registers: 1.76 -> 2.05e10 env-steps/s at 1M envs
    static constexpr int STEP_MIN_CTAS = 6;          // 104 -> 80 registers: 0.39 -> 0.47 of the HBM peak at 4M envs
    static constexpr uint32_t CRIT_MASK = 0x3;       // force_limits, collision_avoidance (:56-68)
    using acc_t = double;
    __device__ static constexpr float penalty(int k) { return k == 0 ? -100.0f : (k == 1 ? -200.0f : -50.0f); }
    __device__ static constexpr double link(int i)
    {   // :85
        return i == 0 ? 0.3 : i == 1 ? 0.3 : i == 2 ? 0.25 : i == 3 ? 0.25 : i == 4 ? 0.15 : i == 5 ? 0.1 : 0.05;
    }
    static constexpr double PI = 3.141592653589793;

    struct NoiseGen {
        __device__ __forceinline__ void get(const Rng&, uint32_t, uint32_t, float (&)[1]) {}
        __device__ static __forceinline__ void get_single(const Rng&, uint32_t, uint32_t, float (&)[1]) {}
    };

    __device__ static __forceinline__ void uniform_actions(const Rng& key, uint32_t env, uint32_t tick, float (&a)[A])
    {
        uniform_actions_policy_stream<A>(key, env, tick, a);
    }

    __device__ static __forceinline__ void fk(const double (&q)[7], double (&pos)[3])
    {   // _forward_kinematics (:94-111)
        double x = 0.0, y = 0.0, z = 0.0;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            double sn, cs;
            spec_sincos_f64(q[i], sn, cs);
            if ((i & 1) == 0) { x = dadd(x, dmul(link(i), cs)); z = dadd(z, dmul(link(i), sn)); }
            else y = dadd(y, dmul(link(i), sn));
        }
        pos[0] = x; pos[1] = y; pos[2] = z;
    }

    __device__ static __forceinline__ void reset(const Rng& key, uint32_t env, uint32_t tick, uint32_t epoch, float (&s)[S])
    {   // _get_initial_state (:113-137): q ~ U(-pi/2, pi/2)
        double q[7], pos[3];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const uint4 w = rng_words(key, env, tick, STREAM_RESET, (epoch << 8) | (uint32_t)j);
            const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * j + k < 7) q[4 * j + k] = (double)mul(0x1.921fb6p+0f, u_sym(ww[k]));
        }
        fk(q, pos);
#pragma unroll
        for (int i = 0; i < S; ++i) s[i] = 0.0f;
        s[0] = (float)pos[0]; s[1] = (float)pos[1]; s[2] = (float)pos[2];
        s[6] = 1.0f;
#pragma unroll
        for (int i = 0; i < 7; ++i) s[7 + i] = (float)q[i];
    }

    __device__ static __forceinline__ bool builtin(int id, const float (&s)[S], const float (&)[A])
    {
        bool ok = true;
        if (id == 0) {                                                           // :10-15
#pragma unroll
            for (int i = 0; i < 3; ++i) ok = ok && (fabsf(s[18 + i]) < 50.0f);
        } else if (id == 1) {                                                    // :18-25 (fp64 bounds)
            ok = ((double)s[0] >= -0.5) && ((double)s[0] <= 0.5) && ((double)s[1] >= -0.5) && ((double)s[1] <= 0.5) &&
                 ((double)s[2] >= 0.0) && ((double)s[2] <= 0.8);
        } else {                                                                 // :28-32
#pragma unroll
            for (int i = 0; i < 7; ++i) ok = ok && (fabsf(s[7 + i]) < 2.0f);
        }
        return ok;
    }

    template <class Div>
    __device__ static __forceinline__ void dynamics(const float (&s)[S], const float (&a)[A], const float (&)[1], float (&o)[S], Div&)
    {   // _dynamics (:139-188)
        double q[7], pos[3];
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            double qd = (double)add(s[7 + i], mul(a[i], 0.1f));                  // :148 fp32, :149-153 fp64 clip
            qd = qd < -PI ? -PI : qd;
            qd = qd > PI ? PI : qd;
            q[i] = qd;
        }
        fk(q, pos);                                                              // :156
        const double dx = dsub(pos[0], 0.3), dy = dsub(pos[1], 0.0), dz = dsub(pos[2], 0.4);
        const double dxy2 = dadd(dmul(dx, dx), dmul(dy, dy));
        const double dist = __dsqrt_rn(dadd(dxy2, dmul(dz, dz)));               // :163
        double fz = 0.0;
        if (dist < 0.01) {                                                       // :164-169
            double nf = dsub(0.01, dist);
            nf = nf > 0.0 ? nf : 0.0;
            fz = -dmul(nf, 1000.0);
        }
        const double aerr = __dsqrt_rn(dxy2);                                    // :172
        double align = dsub(1.0, __ddiv_rn(aerr, 0.005));                        // :173
        align = align > 0.0 ? align : 0.0;
        double ins = dsub(0.4, pos[2]);                                          // :175
        ins = ins > 0.0 ? ins : 0.0;
        double depth = __ddiv_rn(ins, 0.05);                                     // :176
        depth = depth < 1.0 ? depth : 1.0;
        o[0] = (float)pos[0]; o[1] = (float)pos[1]; o[2] = (float)pos[2];
        o[3] = 0.0f; o[4] = 0.0f; o[5] = 0.0f; o[6] = 1.0f;
#pragma unroll
        for (int i = 0; i < 7; ++i) o[7 + i] = (float)q[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) o[14 + i] = (float)__ddiv_rn(dsub(pos[i], (double)s[i]), 0.1);   // :160
        o[17] = 0.0f;
        o[18] = 0.0f; o[19] = 0.0f; o[20] = (float)fz;
        o[21] = (float)align; o[22] = (float)depth; o[23] = (float)dmul(align, depth);               // :178
    }

    template <class Div>
    __device__ static __forceinline__ acc_t reward(const float (&ns)[S], const float (&a)[A], Div&)
    {   // _compute_reward (:190-222)
        const double completion = (double)mul(100.0f, ns[23]);                   // :197 (fp32)
        const double dx = dsub((double)ns[0], 0.3), dy = dsub((double)ns[1], 0.0), dz = dsub((double)ns[2], 0.4);
        const double dist = __dsqrt_rn(dadd(dadd(dmul(dx, dx), dmul(dy, dy)), dmul(dz, dz)));
        const double dr = dmul(-10.0, dist);                                     // :200-201
        const float fm = __fsqrt_rn(add(add(mul(ns[18], ns[18]), mul(ns[19], ns[19])), mul(ns[20], ns[20])));
        const double frw = (fm > 30.0f) ? (double)mul(-50.0f, sub(fm, 30.0f)) : 0.0;   // :204-208
        float sa = 0.0f;
#pragma unroll
        for (int i = 0; i < 7; ++i) sa = add(sa, mul(a[i], a[i]));               // :211 (n < 8: sequential)
        float sv = 0.0f;
#pragma unroll
        for (int i = 0; i < 4; ++i) sv = add(sv, mul(ns[14 + i], ns[14 + i]));   // :214-215
        return dadd(dadd(dadd(dadd(completion, dr), frw), (double)mul(-0.1f, sa)), (double)mul(-0.5f, sv));
    }

    __device__ static __forceinline__ bool is_done(const float (&s)[S])
    {   // :224-244
        bool d = s[23] > 0.95f;
#pragma unroll
        for (int i = 0; i < 3; ++i) d = d || (fabsf(s[18 + i]) > 80.0f);
        const bool inside = ((double)s[0] >= -0.6) && ((double)s[0] <= 0.6) && ((double)s[1] >= -0.6) && ((double)s[1] <= 0.6) &&
                            ((double)s[2] >= -0.1) && ((double)s[2] <= 0.9);
        return d || !inside;
    }

    // get_dataset controllers (:266-287): P-control of the end-effector error on the first three joints, in binary64
    // like the reference (target_position is a float64 array, :83) and rounded to fp32 where the dataset stores it;
    // mode 0 (expert) damps joints 3..6 (fp32: obs * Python float), mode 1 (mixed) drives them with U(-sigma[3], sigma[3])
    __device__ static __forceinline__ void policy_ctrl_from(const nig_policy_params_t& pp, const float (&s)[S], const float (&)[8],
                                                            const float (&u)[4], float (&a)[A])
    {
        const double kp = (double)pp.gain[0][0];
        a[0] = (float)dmul(kp, dsub(0.3, (double)s[0]));
        a[1] = (float)dmul(kp, dsub(0.0, (double)s[1]));
        a[2] = (float)dmul(kp, dsub(0.4, (double)s[2]));
#pragma unroll
        for (int k = 0; k < 4; ++k)
            a[3 + k] = pp.mode == 0 ? mul(pp.gain[3][0], s[10 + k]) : mul(pp.sigma[3], u[k]);
    }
    __device__ static __forceinline__ void policy_ctrl(const Rng& key, const nig_policy_params_t& pp, uint32_t env, uint32_t tick,
                                                       const float (&s)[S], float (&a)[A])
    {
        const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const uint4 w = rng_words(key, env, tick, STREAM_POLICY, 3u);
        const float u[4] = {u_sym(w.x), u_sym(w.y), u_sym(w.z), u_sym(w.w)};
        policy_ctrl_from(pp, s, z, u, a);
    }
};

} // namespace nig
