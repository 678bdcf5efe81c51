/* Exhaustive CPU checks of three shortcuts the reactor's fused rollout loop (reactor_fast_steps_v,
 * neorl-industrial-gym_b200/csrc/nig_kernels.cuh) takes, each against the oracle's own functions:
 *   1. spec_expf_small_v: for every binary32 x in [-6, 6], both zeros included, the shortened exp returns the bits of the
 *      math spec's spec_expf. |x| <= 6 is the range of the exp argument in every step the loop commits.
 *   2. the episode-end catd = cat / 100 by the constant division (cdiv_noguard_v: q = RN(x rc), r = fma(-q, c, x),
 *      q' = fma(r, rc, q)) equals the IEEE division for every cat Reactor::reset can draw: 95 + 2 z over the whole range of
 *      the spec's table normal z, found by evaluating spec_normal on all 2^31 unsigned words;
 *   3. the uniform-policy actions built by one add on the random mantissa bits equal the fma form, for every draw.
 * Compiled together with oracle/nig_oracle.c and the oracle's flags (tests/test_fast_exp_cpu.py):
 *   gcc -O2 -std=c11 -ffp-contract=off -fno-fast-math -mfma -fopenmp tests/fast_exp_check.c -lm
 * Exit status 0 when all three hold. */
#include "../oracle/nig_oracle.c"

#include <stdio.h>

/* the sequence of spec_expf_small_v, one lane */
static float expf_small(float x)
{
    const float t = x * 0x1.715476p+0f;
    const float m = t + 0x1.8p23f;
    const float n = m + -0x1.8p23f;
    float r = fmaf(n, -0x1.62e4p-1f, x);
    r = fmaf(n, -0x1.7f7d1cp-20f, r);
    float p = 0x1.a17e08p-13f;
    p = fmaf(p, r, 0x1.6d7548p-10f);
    p = fmaf(p, r, 0x1.1110a6p-7f);
    p = fmaf(p, r, 0x1.5554acp-5f);
    p = fmaf(p, r, 0x1.555556p-3f);
    p = fmaf(p, r, 0x1.0p-1f);
    p = fmaf(p, r, 1.0f);
    p = fmaf(p, r, 1.0f);
    return p * bits_f((f_bits(m) + 127u) << 23);
}

static float cdiv(float x, float c)
{
    const float rc = 1.0f / c;
    const float q = x * rc;
    const float r = fmaf(-q, c, x);
    return fmaf(r, rc, q);
}

static int check_exp(void)
{
    const uint32_t top = f_bits(6.0f);
    uint64_t n = 0, bad = 0;
#pragma omp parallel for reduction(+ : n, bad) schedule(static)
    for (int64_t i = 0; i <= (int64_t)top; ++i) {
        for (int neg = 0; neg < 2; ++neg) {
            const float x = bits_f((uint32_t)i | (neg ? 0x80000000u : 0u));
            const uint32_t want = f_bits(spec_expf(x)), got = f_bits(expf_small(x));
            n++;
            if (got != want) {
                bad++;
                if (bad <= 8) printf("exp mismatch: x = %a: spec_expf %08x, shortened %08x\n", x, want, got);
            }
        }
    }
    printf("exp: %llu values in [-6, 6], %llu mismatches\n", (unsigned long long)n, (unsigned long long)bad);
    return bad != 0 || n != 2ull * ((uint64_t)top + 1u);
}

static int check_reset_cat_division(void)
{
    /* bit 31 of the word only flips the sign of z, so the 2^31 words without it give every |z| */
    float zlo = INFINITY, zhi = -INFINITY;
#pragma omp parallel for reduction(min : zlo) reduction(max : zhi) schedule(static)
    for (int64_t w = 0; w < (1ll << 31); ++w) {
        const float z = spec_normal((uint32_t)w);
        zlo = z < zlo ? z : zlo;
        zhi = z > zhi ? z : zhi;
    }
    const float zmax = fabsf(zlo) > zhi ? fabsf(zlo) : zhi;
    /* Reactor::reset_from_normals: cat = RN(95 + RN(2 z)), monotone in z */
    const float lo = 95.0f + 2.0f * -zmax, hi = 95.0f + 2.0f * zmax;
    uint64_t n = 0, bad = 0;
    for (uint32_t u = f_bits(lo); u <= f_bits(hi); ++u) {
        const float x = bits_f(u);
        n++;
        if (f_bits(cdiv(x, 100.0f)) != f_bits(x / 100.0f)) {
            bad++;
            if (bad <= 8) printf("division mismatch: cat = %a\n", x);
        }
    }
    printf("reset cat: max |z| = %a, cat in [%a, %a] = [%.6f, %.6f]: %llu values, %llu mismatches of cat / 100\n", zmax, lo,
           hi, lo, hi, (unsigned long long)n, (unsigned long long)bad);
    return bad != 0 || !(lo > 0.0f) || n == 0;
}

/* Reactor::uniform_from_words: the mantissa bits placed under the exponent of 4 / 16 and one add give the values of the fma
 * form fma(1 + v 2^-23, 4 / 16, -5 / -17), for every 22-bit (a0, a1) and 20-bit (a2) v */
static int check_uniform_actions(void)
{
    uint64_t bad = 0;
    for (uint32_t v = 0; v < (1u << 22); ++v) {
        const float want = fmaf(bits_f(v | 0x3f800000u), 4.0f, -5.0f), got = bits_f(v | 0x40800000u) + -5.0f;
        bad += f_bits(want) != f_bits(got);
        if (v < (1u << 20)) {
            const float want2 = fmaf(bits_f(v | 0x3f800000u), 16.0f, -17.0f), got2 = bits_f(v | 0x41800000u) + -17.0f;
            bad += f_bits(want2) != f_bits(got2);
        }
    }
    printf("uniform actions: %llu mismatches\n", (unsigned long long)bad);
    return bad != 0;
}

int main(void)
{
    const int e = check_exp();
    const int d = check_reset_cat_division();
    const int a = check_uniform_actions();
    return e | d | a;
}
