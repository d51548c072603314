// Scoring and top-K evaluation for sm_100a: daisy_bpr_forward, daisy_topk_candidates, daisy_topk_full.
//
// Replaces (reference, file:line):
//   BPR.forward                      BPRMFRecommender.py:42-50   (3 index_select gathers + 2 mul + 2 row sums)
//   _bpr_topk / _hit / _ndcg input   util/metrics.py:46-66       (forward + torch.topk + torch.take per user)
//   final ranking loop               BPRMFRecommender.py:196-207 (one scalar forward per candidate)
#include <float.h>

#include "ctx.cuh"
#include "topk_cand.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// forward: one warp per triple, 128-bit row loads, two warp-shuffle dots
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_forward(const float *__restrict__ P, const float *__restrict__ Q,
                                                  const int32_t *__restrict__ triples, int B, uint32_t U, uint32_t I,
                                                  int D4, float c2, float *__restrict__ pred_i,
                                                  float *__restrict__ pred_j, int *err) {
    const int lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < B; t += nwarps) {
        uint32_t u = (uint32_t)triples[3 * (size_t)t], i = (uint32_t)triples[3 * (size_t)t + 1],
                 j = (uint32_t)triples[3 * (size_t)t + 2];
        if (u >= U || i >= I || j >= I) {
            if (lane == 0) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], t);
            }
            u = u < U ? u : 0u; i = i < I ? i : 0u; j = j < I ? j : 0u;
        }
        float di = 0.f, dj = 0.f;
        for (int e = lane; e < D4; e += 32) {
            const float4 pu = ld_row(P, (size_t)u * D4 + e);
            di += f4_dot(pu, ld_row(Q, (size_t)i * D4 + e));
            dj += f4_dot(pu, ld_row(Q, (size_t)j * D4 + e));
        }
        di = warp_sum(di);
        dj = warp_sum(dj);
        if (lane == 0) {
            pred_i[t] = di * c2;
            pred_j[t] = dj * c2;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// candidate-list top-K: one block per (user, candidate list) group
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_topk_cand(const float *__restrict__ P, const float *__restrict__ Q,
                                                    const int32_t *__restrict__ users,
                                                    const int32_t *__restrict__ cand, int N, int C, int K, uint32_t U,
                                                    uint32_t I, int D4, float c2, int32_t *__restrict__ out_pos,
                                                    int32_t *__restrict__ out_item, float *__restrict__ out_score,
                                                    int *err) {
    extern __shared__ float sc[];  // [C] scores of the current group
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int n = blockIdx.x; n < N; n += gridDim.x) {
        uint32_t u = (uint32_t)users[n];
        if (u >= U) {
            if (threadIdx.x == 0) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], n);
            }
            u = 0;
        }
        float4 pu[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) pu[v] = (lane + 32 * v < D4) ? ld_row(P, (size_t)u * D4 + lane + 32 * v) : f4_zero();
        const int32_t *cn = cand + (size_t)n * C;
        // scores: each warp takes candidates wid, wid+8, ...; two rows in flight per warp
        for (int c = wid; c < C; c += 16) {
            const int c2nd = c + 8;
            uint32_t r0 = (uint32_t)cn[c], r1 = (c2nd < C) ? (uint32_t)cn[c2nd] : 0u;
            if (r0 >= I || r1 >= I) {
                if (lane == 0) {
                    atomicOr(&err[0], 1);
                    atomicMin(&err[1], n);
                }
                r0 = r0 < I ? r0 : 0u; r1 = r1 < I ? r1 : 0u;
            }
            float d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int v = 0; v < 4; ++v)
                if (lane + 32 * v < D4) {
                    const float4 a = ld_row(Q, (size_t)r0 * D4 + lane + 32 * v);
                    const float4 b = ld_row(Q, (size_t)r1 * D4 + lane + 32 * v);
                    d0 += f4_dot(pu[v], a);
                    d1 += f4_dot(pu[v], b);
                }
            d0 = warp_sum(d0);
            d1 = warp_sum(d1);
            if (lane == 0) {
                sc[c] = d0 * c2;
                if (c2nd < C) sc[c2nd] = d1 * c2;
            }
        }
        __syncthreads();
        topk_cand_rounds(sc, C, K, cn, out_pos + (size_t)n * K, out_item + (size_t)n * K, out_score + (size_t)n * K);
    }
}

}  // namespace

extern "C" int daisy_bpr_forward(daisy_handle_t h, const float *P, const float *Q, const int32_t *triples, int64_t B,
                                 float *pred_i, float *pred_j, daisy_stream_t stream) {
    DAISY_REQUIRE(h && P && Q, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(B >= 0 && B < (1LL << 31), DAISY_EINVAL, "bad batch size");
    if (B == 0) return DAISY_OK;
    DAISY_REQUIRE(triples && pred_i && pred_j, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    const int warps_per_block = 8;
    int64_t blocks = (B + warps_per_block - 1) / warps_per_block;
    const int64_t cap = (int64_t)h->num_sms * 32;
    if (blocks > cap) blocks = cap;
    k_forward<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(P, Q, triples, (int)B, (uint32_t)h->U, (uint32_t)h->I,
                                                           h->D / 4, (float)(h->scale * h->scale), pred_i, pred_j,
                                                           h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

extern "C" int daisy_topk_candidates(daisy_handle_t h, const float *P, const float *Q, const int32_t *users,
                                     const int32_t *cand, int64_t N, int C, int K, int32_t *out_pos, int32_t *out_item,
                                     float *out_score, daisy_stream_t stream) {
    DAISY_REQUIRE(h && P && Q, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(C >= 1 && C <= 8192, DAISY_EUNSUPPORTED, "candidate list length %d unsupported (1..8192)", C);
    DAISY_REQUIRE(K >= 1 && K <= 128 && K <= C, DAISY_EUNSUPPORTED, "top_k %d unsupported (1..min(128, C))", K);
    DAISY_REQUIRE(N >= 0 && N < (1LL << 31), DAISY_EINVAL, "bad group count");
    if (N == 0) return DAISY_OK;
    DAISY_REQUIRE(users && cand && out_pos && out_item && out_score, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    int64_t blocks = N;
    const int64_t cap = (int64_t)h->num_sms * 8;
    if (blocks > cap) blocks = cap;
    k_topk_cand<<<(int)blocks, 256, (size_t)C * sizeof(float), (cudaStream_t)stream>>>(
        P, Q, users, cand, (int)N, C, K, (uint32_t)h->U, (uint32_t)h->I, h->D / 4, (float)(h->scale * h->scale), out_pos,
        out_item, out_score, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}
