// NCF in its GMF variant for sm_100a: daisy_gmf_step / daisy_gmf_forward  (SURVEY.md section 8f, row N3).
//
// Replaces (reference, file:line): NCF.forward with model == 'GMF' (NCFRecommender.py:105-125), nn.BCEWithLogitsLoss
// (:255), model.zero_grad / loss.backward / optim.Adam(lr).step (:260, :283-287) -- ATen embedding gathers, the dense
// embedding backward and the foreach Adam pass.
//
//   logit_t = w . (P[u_t] * Q[i_t]) + b          loss = mean_t BCE(logit_t, y_t)
//
// Same gather / score / scatter skeleton as the BPR step, one item ref per sample:
//   bookkeeping  k_small_book in pairs mode (step_kernels.cuh): user refs and item refs sorted by row, slots
//   main         k_gmf_main: one warp per sample; rows gathered with 128-bit loads, warp-shuffle dot, sigmoid and
//                BCE in registers; the descent direction of a row referenced once goes straight to the dense
//                gradient buffer, the others to their staging slot; the sample's contribution to the predict
//                layer's gradient goes to wpart
//   rows         k_seg_all<GradOpt>: deterministic segmented sums of the staged contributions -> gradient buffer
//   predict      k_gmf_wb: fixed-order sum of wpart per feature (and the bias) + Adam on w, b
//   Adam         k_dense_adam: torch.optim.Adam is DENSE -- a row without a gradient keeps moving while its first
//                moment decays -- so every element of both tables is stepped, and the gradient buffer is zeroed for
//                the next step in the same pass.  Bytes: 8 * 4 * D * (U + I) per step, whatever B is; at the
//                reference's sizes (ml-100k, D 32: 2.7 MB) that is L2 traffic.  An exact lazy variant (replay the
//                zero-gradient steps a row missed when it is next touched) is the design for large tables
//                (DESIGN.md section 9); it is not built.
// No float atomics: bit-reproducible.  Batches of up to DAISY_SMALL_MAX (8 192) samples; the reference's is 256.
#include "step_kernels.cuh"

namespace {

struct GradOpt {  // "apply" = file the finished descent sum of a row as its gradient
    static constexpr bool kNeedOldItem = false;
    float *gP, *gQ;
    int D4;
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 /*old*/, float4 d) const {
        st_row(tbl ? gQ : gP, row * D4 + e, make_float4(-d.x, -d.y, -d.z, -d.w));
    }
};

template <int V>
__global__ void __launch_bounds__(256) k_gmf_main(const float *__restrict__ P, const float *__restrict__ Q,
                                                   const float *__restrict__ w, const float *__restrict__ b,
                                                   const int32_t *__restrict__ st, const uint32_t *__restrict__ uslot,
                                                   const uint32_t *__restrict__ islot, float *__restrict__ stageU,
                                                   float *__restrict__ stageQ, float *__restrict__ loss_part,
                                                   float *__restrict__ wpart, int B, int D4, GradOpt opt) {
    const int lane = threadIdx.x & 31;
    const int t = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (t >= B) return;  // warp-uniform
    const int u = st[3 * (size_t)t], i = st[3 * (size_t)t + 1];
    const float y = (float)st[3 * (size_t)t + 2];
    const uint32_t us = uslot[t], is = islot[t];
    const float invB = 1.f / (float)B;
    float4 pu[V], qi[V], wv[V];
    float dotp = 0.f;
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int e = lane + 32 * v;
        pu[v] = qi[v] = wv[v] = f4_zero();
        if (e < D4) {
            pu[v] = ld_row(P, (size_t)u * D4 + e);
            qi[v] = ld_row(Q, (size_t)i * D4 + e);
            wv[v] = ld_row(w, e);
            dotp += wv[v].x * (pu[v].x * qi[v].x) + wv[v].y * (pu[v].y * qi[v].y) + wv[v].z * (pu[v].z * qi[v].z) +
                    wv[v].w * (pu[v].w * qi[v].w);
        }
    }
    const float x = warp_sum(dotp) + b[0];
    const float sig = 1.f / (1.f + expf(-x));
    const float dx = (sig - y) * invB;  // d loss / d logit (mean reduction)
    if (lane == 0) {
        loss_part[t] = (fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x)))) * invB;
        wpart[(size_t)B * (4 * D4) + t] = dx;  // bias gradient contribution
    }
#pragma unroll
    for (int v = 0; v < V; ++v) {
        const int e = lane + 32 * v;
        if (e < D4) {
            // gradients: dL/dP[u] = dx * (w * Q[i]), dL/dQ[i] = dx * (w * P[u]), dL/dw = dx * (P[u] * Q[i]);
            // the step kernels carry DESCENT directions (-gradient), GradOpt flips the sign back
            const float4 du = make_float4(-dx * (wv[v].x * qi[v].x), -dx * (wv[v].y * qi[v].y), -dx * (wv[v].z * qi[v].z),
                                          -dx * (wv[v].w * qi[v].w));
            const float4 di = make_float4(-dx * (wv[v].x * pu[v].x), -dx * (wv[v].y * pu[v].y), -dx * (wv[v].z * pu[v].z),
                                          -dx * (wv[v].w * pu[v].w));
            if (us == DAISY_DIRECT) opt.apply(0, (size_t)u, e, pu[v], du); else st_stream(stageU, (size_t)us * D4 + e, du);
            if (is == DAISY_DIRECT) opt.apply(1, (size_t)i, e, qi[v], di); else st_stream(stageQ, (size_t)is * D4 + e, di);
            st_row(wpart, (size_t)t * D4 + e, make_float4(dx * (pu[v].x * qi[v].x), dx * (pu[v].y * qi[v].y),
                                                            dx * (pu[v].z * qi[v].z), dx * (pu[v].w * qi[v].w)));
        }
    }
}

struct AdamScalars {
    float b1, b2, step_size, inv_sqrt_bc2, eps;
};
__device__ __forceinline__ float adam_one(float th, float g, float &m, float &v, const AdamScalars &a) {
    m = a.b1 * m + (1.f - a.b1) * g;
    v = a.b2 * v + (1.f - a.b2) * g * g;
    return th - a.step_size * m / (sqrtf(v) * a.inv_sqrt_bc2 + a.eps);
}

// Block f < D: feature f of the predict layer's weight; block D: its bias.  Fixed-order sum of the per-sample
// contributions (strided per thread, then a fixed tree), then the element's Adam step.
__global__ void __launch_bounds__(256) k_gmf_wb(const float *__restrict__ wpart, int B, int D, float *__restrict__ w,
                                                 float *__restrict__ b, float *__restrict__ mwb, AdamScalars a) {
    __shared__ double sh[8];
    const int f = blockIdx.x;
    double s = 0.0;
    if (f < D) {
        for (int t = threadIdx.x; t < B; t += 256) s += (double)wpart[(size_t)t * D + f];
    } else {
        for (int t = threadIdx.x; t < B; t += 256) s += (double)wpart[(size_t)B * D + t];
    }
    s = warp_sum_d(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double g = 0.0;
        for (int k = 0; k < 8; ++k) g += sh[k];
        float *theta = f < D ? w + f : b;
        float m = mwb[f], v = mwb[(D + 1) + f];  // moments: [m of w.., m of b, v of w.., v of b]
        *theta = adam_one(*theta, (float)g, m, v, a);
        mwb[f] = m;
        mwb[(D + 1) + f] = v;
    }
}

// torch.optim.Adam over every element of both tables; the gradient buffers are left zero for the next step.
__global__ void k_dense_adam(float4 *__restrict__ P, float4 *__restrict__ mP, float4 *__restrict__ vP, float4 *__restrict__ gP,
                             size_t nP4, float4 *__restrict__ Q, float4 *__restrict__ mQ, float4 *__restrict__ vQ,
                             float4 *__restrict__ gQ, size_t nQ4, AdamScalars a) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < nP4 + nQ4; k += stride) {
        const bool q = k >= nP4;
        const size_t e = q ? k - nP4 : k;
        float4 *T = q ? Q : P, *M = q ? mQ : mP, *Vv = q ? vQ : vP, *G = q ? gQ : gP;
        float4 th = T[e], m = M[e], v = Vv[e];
        const float4 g = G[e];
        th.x = adam_one(th.x, g.x, m.x, v.x, a);
        th.y = adam_one(th.y, g.y, m.y, v.y, a);
        th.z = adam_one(th.z, g.z, m.z, v.z, a);
        th.w = adam_one(th.w, g.w, m.w, v.w, a);
        T[e] = th;
        M[e] = m;
        Vv[e] = v;
        G[e] = f4_zero();
    }
}

__global__ void __launch_bounds__(256) k_gmf_forward(const float *__restrict__ P, const float *__restrict__ Q,
                                                      const float *__restrict__ w, const float *__restrict__ b,
                                                      const int32_t *__restrict__ samples, int B, uint32_t U, uint32_t I,
                                                      int D4, float *__restrict__ pred, int *err) {
    const int lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < B; t += nwarps) {
        uint32_t u = (uint32_t)samples[3 * (size_t)t], i = (uint32_t)samples[3 * (size_t)t + 1];
        if (u >= U || i >= I) {
            if (lane == 0) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], t);
            }
            u = u < U ? u : 0u;
            i = i < I ? i : 0u;
        }
        float d = 0.f;
        for (int e = lane; e < D4; e += 32) {
            const float4 pu = ld_row(P, (size_t)u * D4 + e), qi = ld_row(Q, (size_t)i * D4 + e), wv = ld_row(w, e);
            d += wv.x * (pu.x * qi.x) + wv.y * (pu.y * qi.y) + wv.z * (pu.z * qi.z) + wv.w * (pu.w * qi.w);
        }
        d = warp_sum(d);
        if (lane == 0) pred[t] = d + b[0];
    }
}

template <int V>
static int gmf_table_phase(daisy_ctx *h, const StepPlan &pl, float *P, float *Q, float *w, float *b, float *mP, float *vP,
                           float *mQ, float *vQ, float *mwb, const AdamScalars &a, double *loss_accum) {
    const int B = pl.B, D4 = h->D / 4;
    cudaStream_t s = pl.s;
    BookSet &k = *pl.k;
    GradOpt opt;
    opt.gP = h->gradP;
    opt.gQ = h->gradQ;
    opt.D4 = D4;
    k_gmf_main<V><<<daisy_ceil_div(B, 8), 256, 0, s>>>(P, Q, w, b, k.st, k.uslot, k.jslot, h->stageU, h->stageQ, h->loss_part,
                                                      h->wpart, B, D4, opt);
    DAISY_LAUNCH_CHECK(h);
    const int NS = 64, blocksU = daisy_ceil_div(B, 8 * DAISY_SMALL_WIN), blocksQ = blocksU;
    k_seg_all<V, GradOpt, DAISY_SMALL_WIN, DAISY_SMALL_SLICE><<<NS + blocksU + blocksQ + (loss_accum ? 1 : 0), 256, 0, s>>>(
        P, Q, k.ukey_s, k.qkey_s, B, B, 0xFFFFFFFFu, h->stageU, h->stageQ, h->stage2, D4, opt, NS, blocksU, blocksQ,
        DAISY_SMALL_SLICE, k.longs, h->longs_cap, h->ticket, h->loss_part, B, loss_accum, 0, nullptr);
    DAISY_LAUNCH_CHECK(h);
    k_gmf_wb<<<h->D + 1, 256, 0, s>>>(h->wpart, B, h->D, w, b, mwb, a);
    DAISY_LAUNCH_CHECK(h);
    const size_t nP4 = (size_t)h->U * D4, nQ4 = (size_t)h->I * D4;
    const size_t want = (nP4 + nQ4 + 255) / 256;
    const int grid = (int)(want < (size_t)h->num_sms * 16 ? want : (size_t)h->num_sms * 16);
    k_dense_adam<<<grid, 256, 0, s>>>((float4 *)P, (float4 *)mP, (float4 *)vP, (float4 *)h->gradP, nP4, (float4 *)Q,
                                      (float4 *)mQ, (float4 *)vQ, (float4 *)h->gradQ, nQ4, a);
    DAISY_LAUNCH_CHECK(h);
    if (pl.piped) DAISY_CUDA(cudaEventRecord(k.freed, s));
    return DAISY_OK;
}

}  // namespace

namespace {
struct GmfParams {
    float *P, *Q, *w, *b, *mP, *vP, *mQ, *vQ, *mwb;
    float lr, beta1, beta2, eps;
};

static int gmf_check(daisy_ctx *h, const GmfParams &p, const void *samples, int64_t B, int64_t step_no) {
    int rc = check_step_args(h, p.P, p.Q, samples, B);
    if (rc) return rc;
    DAISY_REQUIRE(p.w && p.b && p.mP && p.vP && p.mQ && p.vQ && p.mwb, DAISY_EINVAL, "null predict-layer or Adam moment pointer");
    DAISY_REQUIRE(((uintptr_t)p.w % 16 == 0), DAISY_EINVAL, "predict-layer weight must be 16-byte aligned");
    DAISY_REQUIRE(step_no >= 1, DAISY_EINVAL, "step_no is 1-based");
    DAISY_REQUIRE(h->scale == 1.0, DAISY_EINVAL, "lazy L2 scale is %g: call daisy_materialize before a GMF step", h->scale);
    return DAISY_OK;
}

// one step; samples_dev is what the kernels read (for host_src != null: the landing buffer the copy fills)
static int gmf_step_impl(daisy_ctx *h, const GmfParams &p, const int32_t *samples_dev, const int32_t *host_src, int64_t B,
                         int64_t step_no, double *loss_accum, cudaStream_t s, bool inputs_ready) {
    if (!h->gradP) {  // dense gradient buffers: zero once, k_dense_adam keeps them zero
        const size_t nP = (size_t)h->U * h->D, nQ = (size_t)h->I * h->D;
        DAISY_CUDA(cudaMalloc((void **)&h->gradP, nP * sizeof(float)));
        DAISY_CUDA(cudaMalloc((void **)&h->gradQ, nQ * sizeof(float)));
        DAISY_CUDA(cudaMalloc((void **)&h->wpart, (size_t)h->maxB * (h->D + 1) * sizeof(float)));
        DAISY_CUDA(cudaMemsetAsync(h->gradP, 0, nP * sizeof(float), s));
        DAISY_CUDA(cudaMemsetAsync(h->gradQ, 0, nQ * sizeof(float), s));
    }
    if (B == 0) return DAISY_OK;  // optimizer.step() without gradients: Adam skips parameters whose .grad is None
    AdamScalars a;
    a.b1 = p.beta1;
    a.b2 = p.beta2;
    a.eps = p.eps;
    a.step_size = (float)((double)p.lr / (1.0 - pow((double)p.beta1, (double)step_no)));
    a.inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)p.beta2, (double)step_no)));
    StepPlan pl;
    h->pairs_mode = 1;
    int rc = book_phase(h, pl, samples_dev, B, (uint32_t)h->U, (uint32_t)h->I, s, host_src, host_src != nullptr || inputs_ready,
                        nullptr);
    h->pairs_mode = 0;
    if (rc) return rc;
    const int D4 = h->D / 4;
    if (D4 <= 32) return gmf_table_phase<1>(h, pl, p.P, p.Q, p.w, p.b, p.mP, p.vP, p.mQ, p.vQ, p.mwb, a, loss_accum);
    if (D4 <= 64) return gmf_table_phase<2>(h, pl, p.P, p.Q, p.w, p.b, p.mP, p.vP, p.mQ, p.vQ, p.mwb, a, loss_accum);
    if (D4 <= 96) return gmf_table_phase<3>(h, pl, p.P, p.Q, p.w, p.b, p.mP, p.vP, p.mQ, p.vQ, p.mwb, a, loss_accum);
    return gmf_table_phase<4>(h, pl, p.P, p.Q, p.w, p.b, p.mP, p.vP, p.mQ, p.vQ, p.mwb, a, loss_accum);
}
}  // namespace

extern "C" int daisy_gmf_step(daisy_handle_t h, float *P, float *Q, float *w, float *b, float *mP, float *vP, float *mQ,
                              float *vQ, float *mwb, const int32_t *samples, int64_t B, float lr, float beta1, float beta2,
                              float eps, int64_t step_no, double *loss_accum, daisy_stream_t stream) {
    const GmfParams p = {P, Q, w, b, mP, vP, mQ, vQ, mwb, lr, beta1, beta2, eps};
    int rc = gmf_check(h, p, samples, B, step_no);
    if (rc) return rc;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    return gmf_step_impl(h, p, samples, nullptr, B, step_no, loss_accum, (cudaStream_t)stream, h->inputs_ready != 0);
}

extern "C" int daisy_gmf_epoch(daisy_handle_t h, float *P, float *Q, float *w, float *b, float *mP, float *vP, float *mQ,
                               float *vQ, float *mwb, const int32_t *samples, int64_t n, int64_t batch, int on_host, float lr,
                               float beta1, float beta2, float eps, int64_t first_step_no, double *loss_accum,
                               daisy_stream_t stream) {
    DAISY_REQUIRE(n >= 0 && batch > 0, DAISY_EINVAL, "epoch of %lld samples in batches of %lld", (long long)n, (long long)batch);
    const GmfParams p = {P, Q, w, b, mP, vP, mQ, vQ, mwb, lr, beta1, beta2, eps};
    int rc = gmf_check(h, p, samples, batch < n ? batch : n, first_step_no);
    if (rc) return rc;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (!on_host && n > 0 && h->pipeline) {  // cf. daisy_bpr_epoch: whatever the inputs-ready flag says
        DAISY_CUDA(cudaEventRecord(h->ev_call, s));
        DAISY_CUDA(cudaStreamWaitEvent(h->side_stream, h->ev_call, 0));
    }
    int64_t step_no = first_step_no;
    for (int64_t at = 0; at < n; at += batch, ++step_no) {
        const int64_t B = n - at < batch ? n - at : batch;
        const int32_t *src = samples + 3 * at;
        if (on_host) {
            int32_t *dst = h->triples + (size_t)h->book_idx * 3 * (size_t)h->maxB;
            rc = gmf_step_impl(h, p, dst, src, B, step_no, loss_accum, s, true);
        } else {
            rc = gmf_step_impl(h, p, src, nullptr, B, step_no, loss_accum, s, true);
        }
        if (rc) return rc;
    }
    return DAISY_OK;
}

extern "C" int daisy_gmf_forward(daisy_handle_t h, const float *P, const float *Q, const float *w, const float *b,
                                 const int32_t *samples, int64_t B, float *pred, daisy_stream_t stream) {
    DAISY_REQUIRE(h && P && Q && w && b, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(h->D % 4 == 0 && h->D <= 512, DAISY_EUNSUPPORTED, "dim %d unsupported (need dim %% 4 == 0, dim <= 512)", h->D);
    DAISY_REQUIRE(B >= 0 && B < (1LL << 31), DAISY_EINVAL, "bad batch size");
    if (B == 0) return DAISY_OK;
    DAISY_REQUIRE(samples && pred, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    int64_t blocks = (B + 7) / 8;
    const int64_t cap = (int64_t)h->num_sms * 16;
    if (blocks > cap) blocks = cap;
    k_gmf_forward<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(P, Q, w, b, samples, (int)B, (uint32_t)h->U, (uint32_t)h->I,
                                                               h->D / 4, pred, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}
