// Ranking with NCF's MLP tower ('MLP') and the script's default 'NeuMF-end' on sm_100a: daisy_neumf_topk_candidates,
// daisy_neumf_topk_full.
//
// Replaces (reference, file:line):
//   metric_eval(model, test_loader, top_k, algo='ncf') -> _ncf_topk    util/metrics.py:68-86,88-94
//     (one NCF.forward over the user's candidates + torch.topk + torch.take per user)
//   and the ranking of a user against the whole catalogue with the same model (forward over every item + topk).
//
// A tower score is not a dot product, so the dot-product ranking kernels do not apply.  Layer 0 splits into a user half
// and an item half, so with Dm = factor * 2^(L-1):
//   A[u] = W0[:, :Dm] . Pm[u]     once per user of the call      } k_score_tile (topk_exact.cuh), fp32 CUDA cores
//   C[i] = W0[:, Dm:] . Qm[i]     once per catalogue item         }
//   k_nr_pairs   a tile of one user x TI items: h0 = relu((A[u] + C[i]) + b0) in shared memory, layers 1..L-1 as
//                register-tiled GEMMs (8 or 4 items x 4 neurons per thread, weights staged through shared memory in
//                64-neuron x 32-input chunks), predict layer + GMF dot; scores go to the handle's score workspace
//   selection    candidate lists: topk_cand_rounds (topk_cand.cuh, as daisy_topk_candidates);
//                full catalogue: k_mask + k_select_topk (topk_exact.cuh, as daisy_topk_full's exact path).
// Every sum runs in one fixed order that does not depend on the tile a pair lands in: a user's scores are the same bits
// whether it is ranked alone or with others, and in both modes.  fp32 on CUDA cores on purpose (ranking parity with
// forward(); a tensor-core tower would move scores by ~1e-3 relative).
#include "ctx.cuh"
#include "topk_cand.cuh"
#include "topk_exact.cuh"

namespace {

constexpr int NR_T = 256;   // threads of the pair kernel
constexpr int NR_NO = 64;   // output neurons per weight chunk
constexpr int NR_KC = 32;   // inputs per weight chunk

struct NrTower {  // the forward fields k_nr_pairs reads, by value
    int L, F, Dm, neumf;
    const float *W[DAISY_NEUMF_MAX_LAYERS], *b[DAISY_NEUMF_MAX_LAYERS];
    const float *Pg, *Qg, *wp, *bp;
};

// Shared memory of k_nr_pairs in floats: the activations feature-major ([feature][TI + 4], layer l >= 1 reads one of
// two regions and writes the other), a weight chunk, the GMF dots, A[u], b0, wp and Pg[u].
static size_t nr_smem_floats(int Dm, int L, int F, int neumf, int TI) {
    const size_t tip = (size_t)TI + 4;
    return (size_t)(Dm + (L > 1 ? Dm / 2 : 0)) * tip + NR_KC * NR_NO + TI + 2 * (size_t)Dm + (neumf ? 3 : 1) * (size_t)F;
}

// grid (ceil(cols / TI), rows): block (x, y) scores user users[y] against items x*TI .. x*TI+TI-1 of its row, the item
// of column c being items[y * cols + c] (candidate lists) or c itself (items == NULL: the catalogue).
template <int TI>
__global__ void __launch_bounds__(NR_T) k_nr_pairs(NrTower t, const float *__restrict__ A, const float *__restrict__ Cc,
                                                    const int32_t *__restrict__ users,
                                                    const int32_t *__restrict__ items, int64_t cols, uint32_t U,
                                                    uint32_t I, int64_t row0, float *__restrict__ S, int *err) {
    extern __shared__ float4 nr_smem4[];
    constexpr int TIP = TI + 4, IPT = TI / 16;
    float *sm = reinterpret_cast<float *>(nr_smem4);
    const int Dm = t.Dm, F = t.F, L = t.L, P = t.neumf ? 2 * F : F;
    float *R0 = sm, *R1 = R0 + (size_t)Dm * TIP;
    float *Wc = R1 + (L > 1 ? (size_t)(Dm / 2) * TIP : 0);
    float *gs = Wc + NR_KC * NR_NO, *arow = gs + TI, *bz = arow + Dm, *wps = bz + Dm, *pg = wps + P;
    const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
    const int y = blockIdx.y;
    const int64_t c0 = (int64_t)blockIdx.x * TI;
    uint32_t u = (uint32_t)users[y];
    if (u >= U) {  // never fault: park on row 0, the error flag tells the caller
        if (tid == 0) {
            atomicOr(&err[0], 1);
            atomicMin(&err[1], (int)(row0 + y));
        }
        u = 0;
    }
    for (int k = tid; k < Dm; k += NR_T) {
        arow[k] = A[(size_t)y * Dm + k];
        bz[k] = t.b[0][k];
    }
    for (int f = tid; f < P; f += NR_T) wps[f] = t.wp[f];
    if (t.neumf)
        for (int f = tid; f < F; f += NR_T) pg[f] = t.Pg[(size_t)u * F + f];
    __syncthreads();
    // layer 0 from its two halves, and the GMF dot wp[:F] . (Pg[u] * Qg[i]): a warp per item, lanes over features
    for (int j = wv; j < TI; j += NR_T / 32) {
        const int64_t col = c0 + j;
        if (col >= cols) {
            for (int k = lane; k < Dm; k += 32) R0[(size_t)k * TIP + j] = 0.f;
            continue;
        }
        uint32_t it = items ? (uint32_t)items[(size_t)y * cols + col] : (uint32_t)col;
        if (it >= I) {
            if (lane == 0) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], (int)(row0 + y));
            }
            it = 0;
        }
        const float *crow = Cc + (size_t)it * Dm;
        for (int k = lane; k < Dm; k += 32) R0[(size_t)k * TIP + j] = fmaxf((arow[k] + crow[k]) + bz[k], 0.f);
        if (t.neumf) {
            float g = 0.f;
            for (int f = lane; f < F; f += 32) g = fmaf(wps[f], pg[f] * t.Qg[(size_t)it * F + f], g);
            g = warp_sum(g);
            if (lane == 0) gs[j] = g;
        }
    }
    // layers 1 .. L-1: thread (tx, ty) owns items {g*64 + tx*4 + 0..3 : g < IPT/4} x neurons n0 + ty*4 + 0..3; every
    // output is one fmaf chain over its inputs in order 0 .. in-1
    const int tx = tid & 15, ty = tid >> 4;
    const float *X = R0;
    for (int l = 1; l < L; ++l) {
        const int in = Dm >> (l - 1), out = in >> 1;
        float *Y = (l & 1) ? R1 : R0;
        const float *__restrict__ W = t.W[l];
        for (int n0 = 0; n0 < out; n0 += NR_NO) {
            float acc[IPT][4];
#pragma unroll
            for (int a = 0; a < IPT; ++a)
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[a][q] = 0.f;
            for (int k0 = 0; k0 < in; k0 += NR_KC) {
                __syncthreads();  // the previous chunk (or layer) is consumed
                {
                    const int nn = tid & (NR_NO - 1), kq = (tid / NR_NO) * 8, n = n0 + nn;
#pragma unroll
                    for (int e = 0; e < 8; ++e) {
                        const int k = k0 + kq + e;
                        Wc[(kq + e) * NR_NO + nn] = (n < out && k < in) ? W[(size_t)n * in + k] : 0.f;
                    }
                }
                __syncthreads();
                auto step = [&](int kk) {
                    const float *xr = X + (size_t)(k0 + kk) * TIP + tx * 4;
                    const float4 w = *reinterpret_cast<const float4 *>(&Wc[kk * NR_NO + ty * 4]);
#pragma unroll
                    for (int g = 0; g < IPT / 4; ++g) {
                        const float4 a = *reinterpret_cast<const float4 *>(xr + g * 64);
                        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            acc[g * 4 + e][0] = fmaf(av[e], w.x, acc[g * 4 + e][0]);
                            acc[g * 4 + e][1] = fmaf(av[e], w.y, acc[g * 4 + e][1]);
                            acc[g * 4 + e][2] = fmaf(av[e], w.z, acc[g * 4 + e][2]);
                            acc[g * 4 + e][3] = fmaf(av[e], w.w, acc[g * 4 + e][3]);
                        }
                    }
                };
                if (in - k0 >= NR_KC) {
#pragma unroll
                    for (int kk = 0; kk < NR_KC; ++kk) step(kk);
                } else {
                    for (int kk = 0; kk < in - k0; ++kk) step(kk);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int n = n0 + ty * 4 + q;
                if (n < out) {
                    const float bn = t.b[l][n];
#pragma unroll
                    for (int g = 0; g < IPT / 4; ++g)
                        *reinterpret_cast<float4 *>(&Y[(size_t)n * TIP + g * 64 + tx * 4]) =
                            make_float4(fmaxf(acc[g * 4 + 0][q] + bn, 0.f), fmaxf(acc[g * 4 + 1][q] + bn, 0.f),
                                        fmaxf(acc[g * 4 + 2][q] + bn, 0.f), fmaxf(acc[g * 4 + 3][q] + bn, 0.f));
                }
            }
        }
        X = Y;
    }
    __syncthreads();
    // predict layer: bp + [GMF dot] + wp[moff:] . h_(L-1), one thread per item
    const int moff = t.neumf ? F : 0;
    for (int j = tid; j < TI; j += NR_T) {
        const int64_t col = c0 + j;
        if (col >= cols) continue;
        float s = t.neumf ? gs[j] : 0.f;
        for (int f = 0; f < F; ++f) s = fmaf(wps[moff + f], X[(size_t)f * TIP + j], s);
        S[(size_t)y * cols + col] = s + t.bp[0];
    }
}

// dst [rows, dst_width] = src rows of `width` floats (row stride src_stride), zero-padded: the operands of k_score_tile
// need rows of a multiple of 4 floats
__global__ void k_nr_pad(const float *__restrict__ src, int64_t src_stride, int64_t rows, int width, int dst_width,
                         float *__restrict__ dst) {
    const int64_t n = rows * dst_width;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / dst_width;
        const int c = (int)(e - r * dst_width);
        dst[e] = c < width ? src[r * src_stride + c] : 0.f;
    }
}

__global__ void k_nr_iota(int32_t *__restrict__ out, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = (int32_t)e;
}

// one block per group: the group's C scores into shared memory, then the selection of daisy_topk_candidates
__global__ void __launch_bounds__(256) k_nr_cand_select(const float *__restrict__ S, const int32_t *__restrict__ cand,
                                                         int C, int K, int32_t *__restrict__ out_pos,
                                                         int32_t *__restrict__ out_item, float *__restrict__ out_score) {
    extern __shared__ float nr_sc[];
    const size_t n = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += 256) nr_sc[c] = S[n * C + c];
    __syncthreads();
    topk_cand_rounds(nr_sc, C, K, cand + n * C, out_pos + n * K, out_item + n * K, out_score + n * K);
}

static int nr_check(daisy_ctx *h, const daisy_neumf_params *p) {
    DAISY_REQUIRE(h != nullptr && p != nullptr, DAISY_EINVAL, "null handle or parameter block");
    DAISY_REQUIRE(p->num_layers >= 1 && p->num_layers <= DAISY_NEUMF_MAX_LAYERS && p->factor >= 1, DAISY_EINVAL,
                  "num_layers %d / factor_num %d out of range", p->num_layers, p->factor);
    DAISY_REQUIRE(((int64_t)p->factor << p->num_layers) <= 1024, DAISY_EUNSUPPORTED,
                  "MLP input of %lld values (factor_num * 2^num_layers) exceeds 1024", (long long)p->factor << p->num_layers);
    DAISY_REQUIRE(p->user_num > 0 && p->item_num > 0 && p->user_num < 0x7fffffffLL && p->item_num < 0x7fffffffLL, DAISY_EINVAL,
                  "bad table sizes");
    DAISY_REQUIRE(p->Pm && p->Qm && p->wp && p->bp && (!p->neumf || (p->Pg && p->Qg)), DAISY_EINVAL, "null table / predict pointer");
    for (int l = 0; l < p->num_layers; ++l) DAISY_REQUIRE(p->W[l] && p->b[l], DAISY_EINVAL, "null MLP layer %d", l);
    return DAISY_OK;
}

// Per-call state: the layer-0 halves of the catalogue, and scratch for the halves of a tile of users.
struct NrCall {
    NrTower t;
    int Dm, Dmp, TI;
    size_t smem;
    const float *Pm, *Qm;             // the MLP tables as k_score_tile reads them (padded copies when Dm % 4 != 0)
    float *w0l, *w0r, *pm_pad, *qm_pad, *cat, *a;
    int32_t *iota;
};

static void nr_free(NrCall &c, cudaStream_t s) {
    for (void *q : {(void *)c.w0l, (void *)c.w0r, (void *)c.pm_pad, (void *)c.qm_pad, (void *)c.cat, (void *)c.a,
                    (void *)c.iota})
        if (q) cudaFreeAsync(q, s);
}

// Validates, allocates, and computes C[i] = W0[:, Dm:] . Qm[i] for the whole catalogue.  max_rows: the most users one
// tile of nr_tile will hold.  On failure the caller still calls nr_free.
static int nr_begin(daisy_ctx *h, const daisy_neumf_params *p, int64_t max_rows, cudaStream_t s, NrCall &c) {
    memset(&c, 0, sizeof(c));
    const int L = p->num_layers, F = p->factor, Dm = F << (L - 1), Dmp = (Dm + 3) & ~3;
    const int64_t U = p->user_num, I = p->item_num;
    c.Dm = Dm;
    c.Dmp = Dmp;
    c.TI = Dm > 256 ? 64 : 128;
    c.smem = nr_smem_floats(Dm, L, F, p->neumf ? 1 : 0, c.TI) * sizeof(float);
    c.t.L = L;
    c.t.F = F;
    c.t.Dm = Dm;
    c.t.neumf = p->neumf ? 1 : 0;
    for (int l = 0; l < DAISY_NEUMF_MAX_LAYERS; ++l) {
        c.t.W[l] = l < L ? p->W[l] : nullptr;
        c.t.b[l] = l < L ? p->b[l] : nullptr;
    }
    c.t.Pg = p->Pg;
    c.t.Qg = p->Qg;
    c.t.wp = p->wp;
    c.t.bp = p->bp;
    bool ok = daisy_scratch_alloc(h, (void **)&c.w0l, (size_t)Dm * Dmp * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&c.w0r, (size_t)Dm * Dmp * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&c.iota, (size_t)I * sizeof(int32_t), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&c.cat, (size_t)I * Dm * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&c.a, (size_t)max_rows * Dm * sizeof(float), s) == cudaSuccess;
    if (Dm != Dmp) {
        ok = ok && daisy_scratch_alloc(h, (void **)&c.pm_pad, (size_t)U * Dmp * sizeof(float), s) == cudaSuccess;
        ok = ok && daisy_scratch_alloc(h, (void **)&c.qm_pad, (size_t)I * Dmp * sizeof(float), s) == cudaSuccess;
    }
    if (!ok) {
        cudaGetLastError();
        daisy_set_error("NeuMF ranking workspace allocation failed");
        return DAISY_ENOMEM;
    }
    const int g = h->num_sms * 4;
    k_nr_pad<<<g, 256, 0, s>>>(p->W[0], 2 * Dm, Dm, Dm, Dmp, c.w0l);
    DAISY_LAUNCH_CHECK(h);
    k_nr_pad<<<g, 256, 0, s>>>(p->W[0] + Dm, 2 * Dm, Dm, Dm, Dmp, c.w0r);
    DAISY_LAUNCH_CHECK(h);
    c.Pm = p->Pm;
    c.Qm = p->Qm;
    if (Dm != Dmp) {
        k_nr_pad<<<g, 256, 0, s>>>(p->Pm, Dm, U, Dm, Dmp, c.pm_pad);
        DAISY_LAUNCH_CHECK(h);
        k_nr_pad<<<g, 256, 0, s>>>(p->Qm, Dm, I, Dm, Dmp, c.qm_pad);
        DAISY_LAUNCH_CHECK(h);
        c.Pm = c.pm_pad;
        c.Qm = c.qm_pad;
    }
    k_nr_iota<<<g, 256, 0, s>>>(c.iota, I);
    DAISY_LAUNCH_CHECK(h);
    const int64_t chunk = (int64_t)65535 * BM;  // rows per k_score_tile launch (grid.y limit)
    for (int64_t first = 0; first < I; first += chunk) {
        const int n = (int)(I - first < chunk ? I - first : chunk);
        dim3 grid((unsigned)((Dm + BN - 1) / BN), (unsigned)((n + BM - 1) / BM));
        k_score_tile<false><<<grid, 256, 0, s>>>(c.Qm, c.w0r, c.iota + first, n, (uint32_t)I, Dm, Dmp, 1.0f,
                                                 c.cat + (size_t)first * Dm, h->err, nullptr, nullptr, nullptr, 0);
        DAISY_LAUNCH_CHECK(h);
    }
    if (c.TI == 128)
        cudaFuncSetAttribute(k_nr_pairs<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
    else
        cudaFuncSetAttribute(k_nr_pairs<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
    return DAISY_OK;
}

// Scores S[y, col] of users[y] (y < nu) against the items of columns 0 .. cols-1 (items[y * cols + col], or col).
static int nr_tile(daisy_ctx *h, const daisy_neumf_params *p, const NrCall &c, const int32_t *users, int nu,
                   const int32_t *items, int64_t cols, int64_t row0, float *S, cudaStream_t s) {
    dim3 ga((unsigned)((c.Dm + BN - 1) / BN), (unsigned)((nu + BM - 1) / BM));
    k_score_tile<false><<<ga, 256, 0, s>>>(c.Pm, c.w0l, users, nu, (uint32_t)p->user_num, c.Dm, c.Dmp, 1.0f, c.a, h->err,
                                           nullptr, nullptr, nullptr, 0);
    DAISY_LAUNCH_CHECK(h);
    dim3 gp((unsigned)((cols + c.TI - 1) / c.TI), (unsigned)nu);
    if (c.TI == 128)
        k_nr_pairs<128><<<gp, NR_T, c.smem, s>>>(c.t, c.a, c.cat, users, items, cols, (uint32_t)p->user_num,
                                                 (uint32_t)p->item_num, row0, S, h->err);
    else
        k_nr_pairs<64><<<gp, NR_T, c.smem, s>>>(c.t, c.a, c.cat, users, items, cols, (uint32_t)p->user_num,
                                                (uint32_t)p->item_num, row0, S, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

// users per tile: as many rows of `cols` scores as fit ~1 GiB, at most 4096 (the tiling of daisy_topk_full)
static int64_t nr_tile_rows(int64_t cols, int64_t N) {
    int64_t tile = (int64_t)((1ull << 30) / ((uint64_t)cols * sizeof(float)));
    if (tile < 1) tile = 1;
    if (tile > 4096) tile = 4096;
    return tile < N ? tile : N;
}

}  // namespace

extern "C" int daisy_neumf_topk_candidates(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *users,
                                           const int32_t *cand, int64_t N, int C, int K, int32_t *out_pos,
                                           int32_t *out_item, float *out_score, daisy_stream_t stream) {
    int rc = nr_check(h, p);
    if (rc) return rc;
    DAISY_REQUIRE(C >= 1 && C <= 8192, DAISY_EUNSUPPORTED, "candidate list length %d unsupported (1..8192)", C);
    DAISY_REQUIRE(K >= 1 && K <= 128 && K <= C, DAISY_EUNSUPPORTED, "top_k %d unsupported (1..min(128, C))", K);
    DAISY_REQUIRE(N >= 0 && N < (1LL << 31), DAISY_EINVAL, "bad group count");
    if (N == 0) return DAISY_OK;
    DAISY_REQUIRE(users && cand && out_pos && out_item && out_score, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t tile = nr_tile_rows(C, N);
    rc = exact_scores_reserve(h, (size_t)tile * C, s);
    if (rc) return rc;
    NrCall c;
    rc = nr_begin(h, p, tile, s, c);
    for (int64_t first = 0; first < N && !rc; first += tile) {
        const int ng = (int)((N - first < tile) ? (N - first) : tile);
        rc = nr_tile(h, p, c, users + first, ng, cand + (size_t)first * C, C, first, h->scores, s);
        if (rc) break;
        k_nr_cand_select<<<ng, 256, (size_t)C * sizeof(float), s>>>(h->scores, cand + (size_t)first * C, C, K,
                                                                   out_pos + (size_t)first * K, out_item + (size_t)first * K,
                                                                   out_score + (size_t)first * K);
        h->launches++;
        if (cudaGetLastError() != cudaSuccess) {
            daisy_set_error("NeuMF candidate selection launch failed");
            rc = DAISY_ECUDA;
        }
    }
    nr_free(c, s);
    return rc;
}

extern "C" int daisy_neumf_topk_full(daisy_handle_t h, const daisy_neumf_params *p, const int32_t *users, int64_t N, int K,
                                     const int64_t *excl_ptr, const int32_t *excl_idx, int32_t *out_item,
                                     float *out_score, daisy_stream_t stream) {
    int rc = nr_check(h, p);
    if (rc) return rc;
    DAISY_REQUIRE(K >= 1 && K <= 128 && (int64_t)K <= p->item_num, DAISY_EUNSUPPORTED,
                  "top_k %d unsupported (1..min(128, item_num))", K);
    DAISY_REQUIRE(N >= 0 && N < (1LL << 31), DAISY_EINVAL, "bad user count");
    if (N == 0) return DAISY_OK;
    DAISY_REQUIRE(users && out_item && out_score, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t I = p->item_num;
    const int64_t tile = nr_tile_rows(I, N);
    rc = exact_scores_reserve(h, (size_t)tile * I, s);
    if (rc) return rc;
    NrCall c;
    rc = nr_begin(h, p, tile, s, c);
    for (int64_t first = 0; first < N && !rc; first += tile) {
        const int nu = (int)((N - first < tile) ? (N - first) : tile);
        rc = nr_tile(h, p, c, users + first, nu, nullptr, I, first, h->scores, s);
        if (rc) break;
        if (excl_ptr && excl_idx) {
            k_mask<<<nu, 128, 0, s>>>(h->scores, I, excl_ptr, excl_idx, first, nu, h->err);
            h->launches++;
        }
        k_select_topk<<<nu, SEL_THREADS, 0, s>>>(h->scores, I, K, first, out_item, out_score);
        h->launches++;
        if (cudaGetLastError() != cudaSuccess) {
            daisy_set_error("NeuMF full-catalogue selection launch failed");
            rc = DAISY_ECUDA;
        }
    }
    nr_free(c, s);
    return rc;
}
