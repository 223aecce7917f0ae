// spmm_b200.hpp — C++ host adapter over the C ABI (include/spmm_b200.h).
//
// Mirrors the reference's operator surface so its harness logic runs with SpMMOpt swapped out:
//   struct CSR    PA4/handout/include/util.h:120-129
//   class  SpMM   PA4/handout/include/spmm_base.h:8-46   (preprocess / run virtuals, set_feat)
//   SpMMOpt slot  PA4/handout/include/spmm_opt.h:5-26    -> class SpMMB200
//
// Inside the reference tree define SPMM_B200_WITH_HANDOUT before including this header: it then
// uses the handout's own "spmm_base.h" (and its CSR / SpMM) instead of the stand-alone mirror
// below, and SpMMB200 derives from the handout's class. See INTEGRATION.md.
#ifndef SPMM_B200_HPP_
#define SPMM_B200_HPP_

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "spmm_b200.h"

#ifdef SPMM_B200_WITH_HANDOUT
#include "spmm_base.h"
#else
struct CSR {
    CSR(int out_num_v, int out_num_e, int *outptr, int *outidx, float *outval)
        : num_v(out_num_v), num_e(out_num_e), ptr(outptr), idx(outidx), val(outval) {}
    int num_v = 0;
    int num_e = 0;
    int *ptr = nullptr;   // device
    int *idx = nullptr;   // device
    float *val = nullptr; // device
};

class SpMM {
   public:
    SpMM(int *dev_out_ptr, int *dev_out_idx, int out_num_v, int out_num_e, int out_feat_in)
        : d_ptr(dev_out_ptr), d_idx(dev_out_idx), feat_in(out_feat_in), num_v(out_num_v), num_e(out_num_e) {}
    SpMM(CSR *g, int out_feat_in)
        : d_ptr(g->ptr), d_idx(g->idx), d_val(g->val), feat_in(out_feat_in), num_v(g->num_v), num_e(g->num_e) {}
    virtual ~SpMM() {}
    virtual void set_feat(int given_feat) { feat_in = given_feat; }
    virtual void preprocess(float *vin, float *vout) = 0;
    virtual void run(float *vin, float *vout) = 0;

   protected:
    int *d_ptr = nullptr;
    int *d_idx = nullptr;
    float *d_val = nullptr;
    int feat_in = 0;
    int num_v = 0;
    int num_e = 0;
};
#endif

// The engine in the slot of SpMMOpt. Errors follow the handout's convention
// (checkCudaErrors -> FatalError, include/util.h:63-84): print, cudaDeviceReset, exit(1).
class SpMMB200 : public SpMM {
   public:
    SpMMB200(CSR *g, int out_feat_in) : SpMM(g, out_feat_in) { create(); }
    SpMMB200(int *dev_out_ptr, int *dev_out_idx, int out_num_v, int out_num_e, int out_feat_in)
        : SpMM(dev_out_ptr, dev_out_idx, out_num_v, out_num_e, out_feat_in) {
        // the handout's raw-pointer constructor leaves d_val NULL (spmm_base.h:11-13); SpMM needs values
        create();
    }
    ~SpMMB200() { spmm_b200_destroy(h_); }
    SpMMB200(const SpMMB200 &) = delete;
    SpMMB200 &operator=(const SpMMB200 &) = delete;

    void set_feat(int given_feat) {
        this->feat_in = given_feat;
        check(spmm_b200_set_feat(h_, given_feat), "set_feat");
    }
    void set_option(const char *name, long long value) { check(spmm_b200_set_option(h_, name, value), name); }
    void set_stream(cudaStream_t s) { stream_ = s; }

    virtual void preprocess(float *vin, float *vout) { check(spmm_b200_preprocess(h_, vin, vout, stream_), "preprocess"); }
    // asynchronous on the stream (default stream unless set_stream), like SpMMRef::run (spmm_ref.cu:27-30)
    virtual void run(float *vin, float *vout) { check(spmm_b200_run(h_, vin, vout, stream_), "run"); }
    // run with this call's edge values (val: the source operator's num_e floats); needs option live_values = 1
    void run_values(const float *val, const float *vin, float *vout) {
        check(spmm_b200_run_values(h_, val, vin, vout, stream_), "run_values");
    }

    // re-stage the plan's copy of idx / val after the caller changed the edge values in place (the reference's
    // SpMMOpt::run reads them live, PA4/workspace/src/spmm_opt.cu:22-25)
    void refresh_values() { check(spmm_b200_refresh_values(h_, stream_), "refresh_values"); }
    // host buffers in and out: upload B band by band under the passes, final rows stored straight into pinned vout
    void run_host(const float *h_vin, float *h_vout) { check(spmm_b200_run_host(h_, h_vin, h_vout, stream_), "run_host"); }
    // the operator over A^T (gradient dB = A^T dC): run(dC, dB). Owns its CSR; delete it before this operator.
    SpMMB200 *transposed(int feat = -1) const {
        spmm_b200_t t = nullptr;
        check(spmm_b200_create_transposed(h_, feat < 0 ? this->feat_in : feat, stream_, &t), "create_transposed");
        return new SpMMB200(t, feat < 0 ? this->feat_in : feat, stream_);
    }

    // SDDMM over this operator's pattern: out[e] = <x_row[row(e)], x_col[idx[e]]> for every nonzero e (out: num_e
    // floats in CSR position order). With x_row = dC and x_col = B, out is the gradient of C = A*B for the edge values.
    void sddmm(const float *x_row, const float *x_col, float *out) { check(spmm_b200_sddmm(h_, x_row, x_col, out, stream_), "sddmm"); }

    // softmax over each row's nonzeros (out: num_e floats in CSR position order, not overlapping scores), and its
    // gradient ds = p * (dp - rowsum(p * dp)) with p the softmax output. Need no preprocess.
    void edge_softmax(const float *scores, float *out) {
        check(spmm_b200_edge_softmax(h_, scores, out, stream_), "edge_softmax");
    }
    void edge_softmax_backward(const float *p, const float *dp, float *ds) {
        check(spmm_b200_edge_softmax_backward(h_, p, dp, ds, stream_), "edge_softmax_backward");
    }

    // amax / amin over each row's messages val[e] * vin[idx[e], j] (op: SPMM_B200_REDUCE_AMAX / _AMIN): vout and arg
    // (the winner's CSR position, may be NULL) are num_v x feat_in. Reads the current edge values; needs preprocess.
    void reduce(int op, const float *vin, float *vout, int *arg) { check(spmm_b200_reduce(h_, op, vin, vout, arg, stream_), "reduce"); }
    // on the operator transposed() returned: the gradients of the source's reduce for B (db) and for the edge values
    // (dval), each optional; vin (the forward's B) is needed only with dval
    void reduce_backward(const float *dc, const int *arg, const float *vin, float *db, float *dval) {
        check(spmm_b200_reduce_backward(h_, dc, arg, vin, db, dval, stream_), "reduce_backward");
    }

    // the same matrix with every row in ascending column order — for CSR inputs whose rows are not column-sorted (they
    // otherwise stay in one column block). Results associate in column order. Delete it before this operator.
    SpMMB200 *column_sorted(int feat = -1) const {
        spmm_b200_t t = nullptr;
        check(spmm_b200_create_column_sorted(h_, feat < 0 ? this->feat_in : feat, stream_, &t), "create_column_sorted");
        return new SpMMB200(t, feat < 0 ? this->feat_in : feat, stream_);
    }
    // destroyed operators leave their plan memory in the library's pool for the next one; this hands it back to the driver
    static void trim_memory() { check(spmm_b200_trim_memory(), "trim_memory"); }

    spmm_b200_t handle() const { return h_; }

   private:
    // adopts a handle made by the library (the transposed operator); d_ptr / d_idx stay NULL: the handle owns its CSR
    SpMMB200(spmm_b200_t adopted, int feat, cudaStream_t s) : SpMM(nullptr, nullptr, 0, 0, feat), h_(adopted), stream_(s) {}
    void create() { check(spmm_b200_create(d_ptr, d_idx, d_val, num_v, num_e, feat_in, &h_), "create"); }
    static void check(int rc, const char *what) {
        if (rc == 0) return;
        std::fprintf(stderr, "Cuda failure: SpMMB200::%s: status %d: %s\nAborting...\n", what, rc,
                     spmm_b200_last_error());
        cudaDeviceReset();
        std::exit(1);
    }
    spmm_b200_t h_ = nullptr;
    cudaStream_t stream_ = nullptr;
};

#endif  // SPMM_B200_HPP_
