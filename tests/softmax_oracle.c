/*
 * tests/softmax_oracle.c — CPU restatement of spmm_b200_edge_softmax and spmm_b200_edge_softmax_backward. TEST
 * INFRASTRUCTURE, NOT PRODUCT CODE: loaded by tests/softmax_oracle.py for the tests and tools/attention_bench.py;
 * nothing under hpc_b200/ links or calls it.
 *
 * Parity status: UNPINNED by construction (the reference has no softmax). This file restates the engine's own documented
 * order and exp routine (hpc_b200/csrc/edge_softmax.cu); tests/test_edge_softmax_oracle.py checks it against an
 * independent numpy restatement and against fp64.
 *
 * Order, per row of n nonzeros: tiles of T = 256 positions; in tile t lane l (of 32) chains from 0.0f over positions
 * t*T + l + 32*j (j = 0..7, < n), forward c = c + exp(s - m), backward c = fmaf(p, dp, c); then for o = 16..1 every
 * lane sets c_l = c_l + c_(l xor o); the row sum adds the tile sums (c_0) from 0.0f in tile order.
 * ftz != 0 models the engine's -ftz=true build: every add, subtract, multiply, FMA and division reads and writes
 * subnormals as signed zero.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define TILE 256
#define LANES 32

static inline float ftz1(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0) { u &= 0x80000000u; memcpy(&x, &u, 4); }
    return x;
}
static inline float fma_m(float a, float b, float c, int ftz) {
    return ftz ? ftz1(fmaf(ftz1(a), ftz1(b), ftz1(c))) : fmaf(a, b, c);
}
static inline float add_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) + ftz1(b)) : a + b; }
static inline float sub_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) - ftz1(b)) : a - b; }
static inline float mul_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) * ftz1(b)) : a * b; }
static inline float div_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) / ftz1(b)) : a / b; }
static inline float bits_f(uint32_t u) {
    float x;
    memcpy(&x, &u, 4);
    return x;
}

/* sm_exp of edge_softmax.cu, for x <= 0 */
float oracle_softmax_exp(float x, int ftz) {
    if (x < -88.0f) return 0.0f;
    const float kf = sub_m(fma_m(x, 1.44269504f, 12582912.0f, ftz), 12582912.0f, ftz);
    const int k = (int)kf;
    if (k < -126) return 0.0f;
    float r = fma_m(kf, -0.693145751953125f, x, ftz);
    r = fma_m(kf, -1.428606765330187e-6f, r, ftz);
    float p = 1.98412698e-4f;
    p = fma_m(p, r, 1.38888889e-3f, ftz);
    p = fma_m(p, r, 8.33333333e-3f, ftz);
    p = fma_m(p, r, 4.16666667e-2f, ftz);
    p = fma_m(p, r, 1.66666667e-1f, ftz);
    p = fma_m(p, r, 0.5f, ftz);
    p = fma_m(p, r, 1.0f, ftz);
    p = fma_m(p, r, 1.0f, ftz);
    const float y = mul_m(p, bits_f((uint32_t)(k + 127) << 23), ftz);
    return y < FLT_MIN ? 0.0f : y;
}

void oracle_softmax_exp_array(const float *x, float *y, long long n, int ftz) {
    for (long long i = 0; i < n; ++i) y[i] = oracle_softmax_exp(x[i], ftz);
}

/* The row sum of the documented order over terms term(i), i < n (bwd: fmaf(a[i], b[i], c); fwd: c + a[i]). */
static float row_sum(const float *a, const float *b, int n, int bwd, int ftz) {
    float total = 0.0f;
    for (int t0 = 0; t0 < n; t0 += TILE) {
        float c[LANES], nc[LANES];
        for (int l = 0; l < LANES; ++l) {
            float acc = 0.0f;
            for (int i = t0 + l; i < t0 + TILE && i < n; i += LANES)
                acc = bwd ? fma_m(a[i], b[i], acc, ftz) : add_m(acc, a[i], ftz);
            c[l] = acc;
        }
        for (int o = LANES / 2; o > 0; o >>= 1) {
            for (int l = 0; l < LANES; ++l) nc[l] = add_m(c[l], c[l ^ o], ftz);
            memcpy(c, nc, sizeof(c));
        }
        total = add_m(total, c[0], ftz);
    }
    return total;
}

void oracle_edge_softmax_f32(const int *ptr, const float *s, float *out, int num_v, int ftz, int nthreads) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int r = 0; r < num_v; ++r) {
        const int beg = ptr[r], n = ptr[r + 1] - beg;
        const float *x = s + beg;
        float *o = out + beg;
        float m = -INFINITY;
        int bad = 0;
        for (int i = 0; i < n; ++i) {
            m = fmaxf(m, x[i]);
            bad |= isnan(x[i]) || x[i] == INFINITY;
        }
        if (bad || m == -INFINITY) {
            const float fill = bad ? bits_f(0x7fffffffu) : 0.0f;
            for (int i = 0; i < n; ++i) o[i] = fill;
            continue;
        }
        for (int i = 0; i < n; ++i) o[i] = oracle_softmax_exp(sub_m(x[i], m, ftz), ftz);   // the exps, in place
        const float S = row_sum(o, NULL, n, 0, ftz);
        for (int i = 0; i < n; ++i) o[i] = div_m(o[i], S, ftz);
    }
}

void oracle_edge_softmax_backward_f32(const int *ptr, const float *p, const float *dp, float *ds, int num_v, int ftz,
                                      int nthreads) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int r = 0; r < num_v; ++r) {
        const int beg = ptr[r], n = ptr[r + 1] - beg;
        const float d = row_sum(p + beg, dp + beg, n, 1, ftz);
        for (int i = beg; i < beg + n; ++i) ds[i] = mul_m(p[i], sub_m(dp[i], d, ftz), ftz);
    }
}

/* The exp contract over every float32 in [-87.5, 0] (both zeros included): stats[0] = values checked, stats[1] =
 * violations (> 2 ulp from fp64 exp, a subnormal result, a nonzero result where exp < FLT_MIN beyond 2 ulp of
 * FLT_MIN, or exp(+-0) != 1), stats[2] = the largest error in ulp of the float32 at the fp64 value (normal range). */
void oracle_softmax_exp_check(int ftz, int nthreads, double *stats) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    const int64_t lo = 0x80000000ll, hi = 0xC2AF0000ll;   /* -0.0 .. -87.5 */
    long long checked = 0, bad = 0;
    double worst = 0.0;
#pragma omp parallel for schedule(static) num_threads(nthreads) reduction(+ : checked, bad) reduction(max : worst)
    for (int64_t u = lo - 1; u <= hi; ++u) {
        const float x = u < lo ? 0.0f : bits_f((uint32_t)u);
        const float y = oracle_softmax_exp(x, ftz);
        const double ref = exp((double)x);
        uint32_t yb;
        memcpy(&yb, &y, 4);
        int ok = (yb & 0x7F800000u) != 0 || yb == 0;   /* never subnormal, never -0 */
        if (x == 0.0f) ok &= y == 1.0f;
        if (ref < FLT_MIN) {
            ok &= y == 0.0f || (y == FLT_MIN && (double)y - ref <= 2.0 * ldexp(1.0, -149));
        } else {
            int e;
            frexp(ref, &e);                              /* ref in [2^(e-1), 2^e) */
            const double err = fabs((double)y - ref) / ldexp(1.0, e - 1 - 23);
            if (err > worst) worst = err;
            ok &= err <= 2.0;
        }
        checked += 1;
        bad += !ok;
    }
    stats[0] = (double)checked;
    stats[1] = (double)bad;
    stats[2] = worst;
}
