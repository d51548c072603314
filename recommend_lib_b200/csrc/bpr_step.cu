// BPR-MF training step for sm_100a: daisy_bpr_step / daisy_bpr_step_host / daisy_bpr_adam_step.
//
// Replaces (reference, file:line): zero_grad + BPR.forward + loss + backward + optim.SGD.step,
// BPRMFRecommender.py:42-50,154,172-176 -- i.e. ATen embedding gathers, embedding_dense_backward and the
// dense _foreach SGD pass (SURVEY.md section 2c).
//
// Pipeline of one step (B triples, tables P [U,D], Q [I,D], all gradients at the PRE-step tables):
//
//   prep     validate ids; key = positive item, value = triple id
//   sort_i   radix sort (CUB) -> triples grouped by positive item ("sorted triple" k)
//   refs     gather triples into sorted order; emit user refs (u, k), negative-item refs (j, k) and one
//            positive-item ref per RUN HEAD (a run = consecutive sorted triples with the same positive item
//            inside one warp chunk of C triples); non-heads get a sentinel key that sorts last
//   sort_u / sort_q   radix sort refs by row -> every row's contributions are contiguous, in a fixed order
//   slots    a row referenced once in the whole batch is DIRECT (updated in place by the main kernel);
//            every other contribution gets a staging slot = its position in the sorted ref array
//   main     one warp per chunk of C sorted triples: 128-bit row gathers (next triple prefetched), warp
//            shuffle dot, sigmoid coefficient in registers, positive-item gradient accumulated in registers
//            over the run; DIRECT rows are written back in place (read once, written once), the others
//            write their contribution to the staging slot
//   seg_u / seg_q   one warp per window of 32 sorted refs: for every multi-contribution row, sum the staged
//            contributions in sorted order (contiguous, streaming reads) and update the row once
//   heavy    rows with more contributions than `heavy_len` are reduced in two levels: one warp per slice of 64
//            contributions, then one block per row over the slice partials
//   loss     fixed-order reduction of the per-warp loss partials into *loss_accum
//
// No float atomics anywhere: the result is bit-reproducible run to run.
// The L2 weight decay of optim.SGD (every row shrinks by 1 - lr*wd per step) is carried by the scalar c
// (ctx.cuh: scale): stored tables are W/c, scores use c^2, the row update is
//   W_hat += [lr / (1 - lr*wd)] * s * (...)          (derivation in DESIGN.md)
// so untouched rows cost no traffic.
#include "step_kernels.cuh"

namespace {


// ------------------------------------------------------------------------------------------------
// optimiser functors: apply(table id, row, f4 index in the row, old row slice, descent direction d = -gradient)
// ------------------------------------------------------------------------------------------------
struct SgdOpt {
    static constexpr bool kNeedOldItem = true;
    float *P, *Q;
    float alpha;  // lr / (1 - lr*wd)
    int D4;
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 old, float4 d) const {
        const size_t idx = row * D4 + e;
        float4 r = make_float4(fmaf(alpha, d.x, old.x), fmaf(alpha, d.y, old.y), fmaf(alpha, d.z, old.z),
                               fmaf(alpha, d.w, old.w));
        st_row(tbl ? Q : P, idx, r);
    }
};

// torch.optim.SparseAdam semantics on the rows present in the batch (lazy: other rows and their moments
// are untouched).  g = -d.
struct AdamOpt {
    static constexpr bool kNeedOldItem = true;
    float *P, *Q, *mP, *vP, *mQ, *vQ;
    float omb1, omb2, step_size, eps;   // 1 - beta1, 1 - beta2 (rounded from double: 1.f - 0.999f is off by 1.3e-5 of
                                        // its value); step_size = lr * sqrt(1 - b2^t) / (1 - b1^t)
    int D4;
    // torch/optim/_functional.py: sparse_adam -- old += (1 - b) * (new - old); denom = sqrt(v) + eps (eps is NOT
    // divided by the bias correction, unlike dense Adam); param -= step_size * m / denom
    __device__ __forceinline__ float one(float w, float g, float &m, float &v) const {
        m = fmaf(omb1, g - m, m);
        v = fmaf(omb2, g * g - v, v);
        return w - step_size * (m / (sqrtf(v) + eps));
    }
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 old, float4 d) const {
        const size_t idx = row * D4 + e;
        float *M = tbl ? mQ : mP, *Vv = tbl ? vQ : vP;
        float4 m = ld_row(M, idx), v = ld_row(Vv, idx), r;
        r.x = one(old.x, -d.x, m.x, v.x);
        r.y = one(old.y, -d.y, m.y, v.y);
        r.z = one(old.z, -d.z, m.z, v.z);
        r.w = one(old.w, -d.w, m.w, v.w);
        st_row(M, idx, m);
        st_row(Vv, idx, v);
        st_row(tbl ? Q : P, idx, r);
    }
};

// torch.optim.Adagrad (lr_decay 0) on the rows present in the batch: state_sum += g^2; w -= lr * g / (sqrt(state_sum) +
// eps).  An element with zero gradient does not move under Adagrad, so the reference's dense optimiser and this sparse
// one are the same function.  BPR-FM (daisy_bprfm_adagrad_step) runs on AUGMENTED rows [e_0 .. e_{F-1}, x, 0, 0, 0]:
// x = 1 for a user row (a constant, not a parameter: float4 `const_e` of table 0 is never written), x = b_i for an item
// row, so that <user row, item_i row - item_j row> = <e_u, e_i - e_j> + b_i - b_j and the bias gradient falls out of
// the same kernels.  g = -d.
struct AdagradOpt {
    static constexpr bool kNeedOldItem = true;
    float *P, *Q, *aP, *aQ;
    float lr, eps;
    int D4, const_e;
    __device__ __forceinline__ float one(float w, float g, float &acc) const {
        acc = fmaf(g, g, acc);
        return w - lr * g / (sqrtf(acc) + eps);
    }
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 old, float4 d) const {
        if (tbl == 0 && e == const_e) return;
        const size_t idx = row * D4 + e;
        float *A = tbl ? aQ : aP;
        float4 acc = ld_row(A, idx), r;
        r.x = one(old.x, -d.x, acc.x);
        r.y = one(old.y, -d.y, acc.y);
        r.z = one(old.z, -d.z, acc.z);
        r.w = one(old.w, -d.w, acc.w);
        st_row(A, idx, acc);
        st_row(tbl ? Q : P, idx, r);
    }
};

// shared body of daisy_bpr_step / daisy_bpr_step_host
static int sgd_step(daisy_ctx *h, float *P, float *Q, const int32_t *triples_dev, const int32_t *host_src, int64_t B,
                    float lr, float wd, double *loss_accum, daisy_stream_t stream, bool inputs_ready) {
    const double shrink = 1.0 - (double)lr * (double)wd;
    DAISY_REQUIRE(shrink > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1: the L2 shrink factor is not positive", (double)lr * wd);
    if (B == 0) {  // an empty batch still decays every row (optim.SGD.step with zero gradients)
        h->scale *= shrink;
        return DAISY_OK;
    }
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    SgdOpt opt;
    opt.P = P;
    opt.Q = Q;
    opt.alpha = (float)((double)lr / shrink);
    opt.D4 = h->D / 4;
    const float c2 = (float)(h->scale * h->scale);
    int rc = run_step<SgdOpt>(h, P, Q, triples_dev, B, opt, c2, loss_accum, (cudaStream_t)stream, host_src,
                              host_src != nullptr || inputs_ready);
    if (rc) return rc;
    h->scale *= shrink;
    if ((h->flags & DAISY_FLAG_EAGER_DECAY) || h->scale < 1e-4) return daisy_materialize(h, P, Q, stream);
    return DAISY_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int daisy_bpr_step(daisy_handle_t h, float *P, float *Q, const int32_t *triples, int64_t B, float lr,
                              float wd, double *loss_accum, daisy_stream_t stream) {
    int rc = check_step_args(h, P, Q, triples, B);
    if (rc) return rc;
    return sgd_step(h, P, Q, triples, nullptr, B, lr, wd, loss_accum, stream, h->inputs_ready != 0);
}

extern "C" int daisy_bpr_step_host(daisy_handle_t h, float *P, float *Q, const int32_t *triples_host, int64_t B,
                                   float lr, float wd, double *loss_accum, daisy_stream_t stream) {
    int rc = check_step_args(h, P, Q, triples_host, B);
    if (rc) return rc;
    // landing buffer of the bookkeeping set this step will use; the H2D copy is issued on the side stream as the
    // first node of the step's bookkeeping chain, so it overlaps the previous step's kernels
    int32_t *dst = h->triples + (size_t)h->book_idx * 3 * (size_t)h->maxB;
    return sgd_step(h, P, Q, dst, triples_host, B, lr, wd, loss_accum, stream, true);
}

extern "C" int daisy_bpr_epoch(daisy_handle_t h, float *P, float *Q, const int32_t *triples, int64_t n, int64_t batch,
                               int on_host, float lr, float wd, double *loss_accum, daisy_stream_t stream) {
    DAISY_REQUIRE(n >= 0 && batch > 0, DAISY_EINVAL, "epoch of %lld triples in batches of %lld", (long long)n, (long long)batch);
    int rc = check_step_args(h, P, Q, triples, batch < n ? batch : n);
    if (rc) return rc;
    if (!on_host && n > 0 && h->pipeline) {
        // the triples are complete once the work already queued on `stream` is: order the bookkeeping stream behind
        // it ONCE, then every step's bookkeeping may run ahead of the previous step's kernels.  Whatever the handle's
        // inputs-ready flag says: it describes the triples of daisy_bpr_step calls, not these.
        DeviceGuard g(h->device);
        DAISY_CUDA(cudaEventRecord(h->ev_call, (cudaStream_t)stream));
        DAISY_CUDA(cudaStreamWaitEvent(h->side_stream, h->ev_call, 0));
    }
    for (int64_t s = 0; s < n; s += batch) {
        const int64_t B = n - s < batch ? n - s : batch;
        const int32_t *src = triples + 3 * s;
        if (on_host) {
            int32_t *dst = h->triples + (size_t)h->book_idx * 3 * (size_t)h->maxB;
            rc = sgd_step(h, P, Q, dst, src, B, lr, wd, loss_accum, stream, true);
        } else {
            rc = sgd_step(h, P, Q, src, nullptr, B, lr, wd, loss_accum, stream, true);
        }
        if (rc) return rc;
    }
    return DAISY_OK;
}

extern "C" int daisy_bpr_adam_step(daisy_handle_t h, float *P, float *Q, float *mP, float *vP, float *mQ, float *vQ,
                                   const int32_t *triples, int64_t B, float lr, double beta1, double beta2, float eps,
                                   int64_t step_no, double *loss_accum, daisy_stream_t stream) {
    int rc = check_step_args(h, P, Q, triples, B);
    if (rc) return rc;
    DAISY_REQUIRE(mP && vP && mQ && vQ, DAISY_EINVAL, "null Adam moment pointer");
    DAISY_REQUIRE(step_no >= 1, DAISY_EINVAL, "step_no is 1-based");
    DAISY_REQUIRE(h->scale == 1.0, DAISY_EINVAL, "lazy L2 scale is %g: call daisy_materialize before an Adam step", h->scale);
    if (B == 0) return DAISY_OK;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    AdamOpt opt;
    opt.P = P; opt.Q = Q; opt.mP = mP; opt.vP = vP; opt.mQ = mQ; opt.vQ = vQ;
    opt.omb1 = (float)(1.0 - beta1);
    opt.omb2 = (float)(1.0 - beta2);
    const double bc1 = 1.0 - pow(beta1, (double)step_no);
    const double bc2 = 1.0 - pow(beta2, (double)step_no);
    opt.step_size = (float)((double)lr * sqrt(bc2) / bc1);
    opt.eps = eps;
    opt.D4 = h->D / 4;
    // the triples may have been produced by earlier work on `stream` (the inputs-ready flag is daisy_bpr_step's)
    return run_step<AdamOpt>(h, P, Q, triples, B, opt, 1.0f, loss_accum, (cudaStream_t)stream, nullptr, false);
}

extern "C" int daisy_bprfm_adagrad_step(daisy_handle_t h, float *E, float *acc, const int32_t *triples, int64_t B, float lr,
                                        float eps, double *loss_accum, daisy_stream_t stream) {
    DAISY_REQUIRE(h != nullptr && E && acc, DAISY_EINVAL, "null argument");
    float *P = E, *Q = E + (size_t)h->U * h->D;            // users first, then items, in ONE feature table
    int rc = check_step_args(h, P, Q, triples, B);
    if (rc) return rc;
    DAISY_REQUIRE(h->D >= 8, DAISY_EINVAL, "augmented row width %d: need num_factors + 4", h->D);
    DAISY_REQUIRE(h->scale == 1.0, DAISY_EINVAL, "lazy L2 scale is %g: call daisy_materialize first", h->scale);
    if (B == 0) return DAISY_OK;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    AdagradOpt opt;
    opt.P = P; opt.Q = Q;
    opt.aP = acc; opt.aQ = acc + (size_t)h->U * h->D;
    opt.lr = lr;
    opt.eps = eps;
    opt.D4 = h->D / 4;
    opt.const_e = h->D / 4 - 1;                             // the last float4 of a row: [x, 0, 0, 0]
    // the triples may have been produced by earlier work on `stream` (the inputs-ready flag is daisy_bpr_step's)
    return run_step<AdagradOpt>(h, P, Q, triples, B, opt, 1.0f, loss_accum, (cudaStream_t)stream, nullptr, false);
}
