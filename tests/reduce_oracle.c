/*
 * tests/reduce_oracle.c — CPU restatement of spmm_b200_reduce and spmm_b200_reduce_backward. TEST INFRASTRUCTURE, NOT
 * PRODUCT CODE: loaded by tests/reduce_oracle.py for the tests and tools/reduce_bench.py; nothing under hpc_b200/ links
 * or calls it.
 *
 * Restates the contract documented in hpc_b200/csrc/reduce.cu:
 *   forward   m(e, j) = val[e] * vin[idx[e]*K + j] (one rounded multiply); the winner is the maximum of the total order
 *             "NaN above every number; larger (amax) / smaller (amin) value; equal values (-0 == +0) to the smaller
 *             position". Walking a row in position order, a later message replaces the winner when it is a NaN over
 *             a number, or strictly larger (amax) / smaller (amin). Empty row: +0.0f, arg = -1.
 *   db        Aᵀ row c = the positions e with idx[e] == c in ascending order (the transposed operator's storage order);
 *             tiles of REDUCE_TILE entries; s = fmaf(val[e], dc[r*K + j], s) from 0.0f over the matching entries of a
 *             tile; db = 0.0f + tile sums in tile order.
 *   dval      sddmm's order (tests/sddmm_oracle.c) over x_row = dc[r], x_col = vin[c], non-matching terms skipped.
 * ftz != 0 models the engine's -ftz=true build: every multiply, FMA and add reads and writes subnormals as signed zero.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define REDUCE_TILE 1024   /* kTile of hpc_b200/csrc/reduce.cu */

int oracle_reduce_tile(void) { return REDUCE_TILE; }

static inline float ftz1(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0) { u &= 0x80000000u; memcpy(&x, &u, 4); }
    return x;
}
static inline float mul_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) * ftz1(b)) : a * b; }
static inline float fma_m(float a, float b, float c, int ftz) {
    return ftz ? ftz1(fmaf(ftz1(a), ftz1(b), ftz1(c))) : fmaf(a, b, c);
}
static inline float add_m(float a, float b, int ftz) { return ftz ? ftz1(ftz1(a) + ftz1(b)) : a + b; }

static int nthreads_or_max(int n) {
#ifdef _OPENMP
    return n > 0 ? n : omp_get_max_threads();
#else
    (void)n;
    return 1;
#endif
}

/* arg may be NULL */
void oracle_reduce_f32(const int *ptr, const int *idx, const float *val, const float *vin, float *vout, int *arg,
                       int num_v, int feat, int amax, int ftz, int nthreads) {
    nthreads = nthreads_or_max(nthreads);
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
    for (int r = 0; r < num_v; ++r) {
        for (int j = 0; j < feat; ++j) {
            float best = 0.0f;
            int pos = -1;
            for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
                const float m = mul_m(val[e], vin[(size_t)idx[e] * feat + j], ftz);
                const int wins = pos < 0 || (isnan(m) && !isnan(best)) || (amax ? m > best : m < best);
                if (wins) {
                    best = m;
                    pos = e;
                }
            }
            vout[(size_t)r * feat + j] = best;
            if (arg) arg[(size_t)r * feat + j] = pos;
        }
    }
}

/* the transposed storage order: tptr[b_rows + 1], tpos[num_e] = positions e by column, ascending */
static void transpose_positions(const int *ptr, const int *idx, int num_v, int b_rows, int *tptr, int *tpos, int *trow) {
    memset(tptr, 0, sizeof(int) * ((size_t)b_rows + 1));
    const int nnz = ptr[num_v];
    for (int e = 0; e < nnz; ++e) tptr[idx[e] + 1]++;
    for (int c = 0; c < b_rows; ++c) tptr[c + 1] += tptr[c];
    int *fill = (int *)malloc(sizeof(int) * ((size_t)b_rows + 1));
    memcpy(fill, tptr, sizeof(int) * ((size_t)b_rows + 1));
    for (int r = 0; r < num_v; ++r)
        for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
            const int k = fill[idx[e]]++;
            tpos[k] = e;
            trow[k] = r;
        }
    free(fill);
}

static int lanes_for(int q) {
    int l = 1;
    while (l < q && l < 32) l <<= 1;
    return l;
}

/* db (b_rows x feat) and dval (num_e); either may be NULL; vin is read only for dval */
void oracle_reduce_backward_f32(const int *ptr, const int *idx, const float *val, const float *dc, const int *arg,
                                const float *vin, float *db, float *dval, int num_v, int b_rows, int feat, int ftz,
                                int nthreads) {
    nthreads = nthreads_or_max(nthreads);
    const int nnz = ptr[num_v];
    int *tptr = (int *)malloc(sizeof(int) * ((size_t)b_rows + 1));
    int *tpos = (int *)malloc(sizeof(int) * ((size_t)nnz + 1));
    int *trow = (int *)malloc(sizeof(int) * ((size_t)nnz + 1));
    transpose_positions(ptr, idx, num_v, b_rows, tptr, tpos, trow);
    if (db) {
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
        for (int c = 0; c < b_rows; ++c) {
            for (int j = 0; j < feat; ++j) {
                float total = 0.0f;
                for (int tb = tptr[c]; tb < tptr[c + 1]; tb += REDUCE_TILE) {
                    const int te = tb + REDUCE_TILE < tptr[c + 1] ? tb + REDUCE_TILE : tptr[c + 1];
                    float s = 0.0f;
                    for (int k = tb; k < te; ++k) {
                        const int e = tpos[k], r = trow[k];
                        if (arg[(size_t)r * feat + j] == e) s = fma_m(val[e], dc[(size_t)r * feat + j], s, ftz);
                    }
                    total = add_m(total, s, ftz);
                }
                db[(size_t)c * feat + j] = total;
            }
        }
    }
    if (dval) {
        const int w = feat % 4 == 0 ? 4 : 1, q_n = feat / w, lanes = lanes_for(q_n);
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads)
        for (int r = 0; r < num_v; ++r) {
            const float *xr = dc + (size_t)r * feat;
            const int *ar = arg + (size_t)r * feat;
            for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
                const float *xc = vin + (size_t)idx[e] * feat;
                float s[32], t[32];
                for (int l = 0; l < lanes; ++l) {
                    float acc = 0.0f;
                    for (int q = l; q < q_n; q += lanes)
                        for (int i = 0; i < w; ++i)
                            if (ar[q * w + i] == e) acc = fma_m(xr[q * w + i], xc[q * w + i], acc, ftz);
                    s[l] = acc;
                }
                for (int o = lanes / 2; o > 0; o >>= 1) {
                    for (int l = 0; l < lanes; ++l) t[l] = add_m(s[l], s[l ^ o], ftz);
                    memcpy(s, t, sizeof(float) * (size_t)lanes);
                }
                dval[e] = s[0];
            }
        }
    }
    free(tptr);
    free(tpos);
    free(trow);
}

/* fp64 gradients for the same arg, and the fp64 sums of |terms| (distance bounds); NULL outputs are skipped */
void oracle_reduce_backward_f64(const int *ptr, const int *idx, const float *val, const float *dc, const int *arg,
                                const float *vin, double *db, double *db_abs, double *dval, double *dval_abs,
                                int *db_terms, int num_v, int b_rows, int feat) {
    if (db) memset(db, 0, sizeof(double) * (size_t)b_rows * feat);
    if (db_abs) memset(db_abs, 0, sizeof(double) * (size_t)b_rows * feat);
    if (db_terms) memset(db_terms, 0, sizeof(int) * (size_t)b_rows * feat);
    for (int r = 0; r < num_v; ++r)
        for (int e = ptr[r]; e < ptr[r + 1]; ++e) {
            const int c = idx[e];
            double acc = 0.0, ab = 0.0;
            for (int j = 0; j < feat; ++j) {
                if (arg[(size_t)r * feat + j] != e) continue;
                const double g = (double)dc[(size_t)r * feat + j];
                const size_t o = (size_t)c * feat + j;
                if (db) db[o] += (double)val[e] * g;
                if (db_abs) db_abs[o] += fabs((double)val[e] * g);
                if (db_terms) db_terms[o] += 1;
                const double p = g * (double)vin[o];
                acc += p;
                ab += fabs(p);
            }
            if (dval) dval[e] = acc;
            if (dval_abs) dval_abs[e] = ab;
        }
}
