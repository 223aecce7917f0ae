/*
 * tests/sddmm_oracle.c — CPU restatement of spmm_b200_sddmm. TEST INFRASTRUCTURE, NOT PRODUCT CODE: loaded by
 * tests/sddmm_oracle.py for the tests and tools/sddmm_bench.py; nothing under hpc_b200/ links or calls it.
 *
 * Parity status: UNPINNED by construction. The reference (liblaf/hpc PA4) is forward only and has no SDDMM, so this
 * file restates the engine's own documented order (hpc_b200/csrc/sddmm.cu), like the transposed product's
 * oracle_spmm_t_f32; tests/test_sddmm_oracle.py checks it against an independent numpy restatement of the same order.
 *
 * Order, K = feat. K % 4 == 0: Q = K/4 groups of W = 4 columns; otherwise Q = K groups of W = 1. L = min(32,
 * pow2ceil(Q)) lanes. Lane l: s_l = 0.0f; for q = l, l+L, ... < Q, t = 0..W-1: s_l = fmaf(x_row[qW+t], x_col[qW+t], s_l).
 * Then for o = L/2, ..., 1: s_l = s_l + s_(l xor o) for every lane at once. out[e] = s_0.
 * ftz != 0 models the engine's -ftz=true build: every FMA and add reads and writes subnormals as signed zero.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static inline float ftz1(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0) { u &= 0x80000000u; memcpy(&x, &u, 4); }
    return x;
}
static inline float fma_m(float a, float b, float c, int ftz) {
    return ftz ? ftz1(fmaf(ftz1(a), ftz1(b), ftz1(c))) : fmaf(a, b, c);
}
static inline float add_m(float a, float b, int ftz) {
    return ftz ? ftz1(ftz1(a) + ftz1(b)) : a + b;
}

static int sddmm_lanes(int q) {
    int l = 1;
    while (l < q && l < 32) l <<= 1;
    return l;
}

void oracle_sddmm_f32(const int *ptr, const int *idx, const float *x_row, const float *x_col, float *out, int num_v,
                      int feat, int ftz, int nthreads) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
    const int w = feat % 4 == 0 ? 4 : 1, q_n = feat / w, lanes = sddmm_lanes(q_n);
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int r = 0; r < num_v; ++r) {
        const float *xr = x_row + (size_t)r * feat;
        for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
            const float *xc = x_col + (size_t)idx[e] * feat;
            float s[32], t[32];
            for (int l = 0; l < lanes; ++l) {
                float acc = 0.0f;
                for (int q = l; q < q_n; q += lanes)
                    for (int c = 0; c < w; ++c) acc = fma_m(xr[q * w + c], xc[q * w + c], acc, ftz);
                s[l] = acc;
            }
            for (int o = lanes / 2; o > 0; o >>= 1) {
                for (int l = 0; l < lanes; ++l) t[l] = add_m(s[l], s[l ^ o], ftz);
                memcpy(s, t, sizeof(float) * (size_t)lanes);
            }
            out[e] = s[0];
        }
    }
}

/* fp64 dot and fp64 sum of |terms| per nonzero (tolerance checks; no order to restate). */
void oracle_sddmm_f64(const int *ptr, const int *idx, const float *x_row, const float *x_col, double *out, double *abs_out,
                      int num_v, int feat, int nthreads) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
    (void)nthreads;
#endif
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int r = 0; r < num_v; ++r) {
        const float *xr = x_row + (size_t)r * feat;
        for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
            const float *xc = x_col + (size_t)idx[e] * feat;
            double acc = 0.0, ab = 0.0;
            for (int j = 0; j < feat; ++j) {
                const double p = (double)xr[j] * (double)xc[j];
                acc += p;
                ab += fabs(p);
            }
            out[e] = acc;
            if (abs_out) abs_out[e] = ab;
        }
    }
}
