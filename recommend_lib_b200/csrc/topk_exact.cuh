// The exact full-catalogue path shared by daisy_topk_full (topk_full.cu) and daisy_neumf_topk_full (neumf_rank.cu):
//   k_score_tile   fp32 register-tiled S[m, i] = c^2 <P[users[m]], Q[i]> (also the layer-0 GEMM of the NeuMF ranking),
//   k_mask         -inf on each user's excluded items (CSR lists),
//   k_select_topk  exact radix select of the K best scores of a row, order (score desc, item asc).
// A header rather than a separate unit because tests/emu builds one translation unit at a time.
#pragma once
#include "ctx.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 16;

__device__ __forceinline__ uint32_t okey(float f) {  // order-preserving float -> uint32
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float okey_inv(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// FILTER = false: scores are written to S [n_users, I].
// FILTER = true : nothing is materialised -- a score at or above the user's threshold thr[m] is appended to the user's
//                 candidate list (cand_key [n_users, cap], count in cnt[m]); see daisy_topk_full.
// 128 x 128 x 16 block tile, 256 threads, 8 x 8 register tile per thread (two 4-wide groups 64 apart in each
// direction, so that the shared-memory operand loads are conflict-free 128-bit loads): 4 LDS.128 per 64 FMA.
template <bool FILTER>
__global__ void __launch_bounds__(256, 2) k_score_tile(const float *__restrict__ P, const float *__restrict__ Q,
                                                        const int32_t *__restrict__ users, int n_users, uint32_t U,
                                                        int64_t I, int D, float c2, float *__restrict__ S, int *err,
                                                        const float *__restrict__ thr, int *__restrict__ cnt,
                                                        unsigned long long *__restrict__ cand_key, int cap) {
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Bs[2][BK][BN + 4];
    const int tid = threadIdx.x;
    const int m0 = blockIdx.y * BM;
    const int64_t i0 = (int64_t)blockIdx.x * BN;
    const int lr = tid >> 2, lk = (tid & 3) * 4;  // loader coordinates: rows lr and lr + 64, k offset 0,4,8,12
    int64_t urow[2] = {-1, -1};
#pragma unroll
    for (int hh = 0; hh < 2; ++hh)
        if (m0 + lr + 64 * hh < n_users) {
            uint32_t u = (uint32_t)users[m0 + lr + 64 * hh];
            if (u >= U) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], m0 + lr + 64 * hh);
                u = 0;
            }
            urow[hh] = (int64_t)u;
        }
    const int64_t it[2] = {i0 + lr, i0 + lr + 64};
    const int ty = tid >> 4, tx = tid & 15;
    float acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

    float4 ra[2], rb[2];
    auto gload = [&](int k0) {
        const int k = k0 + lk;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            ra[hh] = (urow[hh] >= 0 && k < D) ? *reinterpret_cast<const float4 *>(P + urow[hh] * D + k) : f4_zero();
            rb[hh] = (it[hh] < I && k < D) ? *reinterpret_cast<const float4 *>(Q + it[hh] * D + k) : f4_zero();
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int r = lr + 64 * hh;
            As[buf][lk + 0][r] = ra[hh].x; As[buf][lk + 1][r] = ra[hh].y; As[buf][lk + 2][r] = ra[hh].z; As[buf][lk + 3][r] = ra[hh].w;
            Bs[buf][lk + 0][r] = rb[hh].x; Bs[buf][lk + 1][r] = rb[hh].y; Bs[buf][lk + 2][r] = rb[hh].z; Bs[buf][lk + 3][r] = rb[hh].w;
        }
    };
    gload(0);
    sstore(0);
    __syncthreads();
    const int nk = (D + BK - 1) / BK;
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][kk][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int x = 0; x < 8; ++x)
#pragma unroll
                for (int y = 0; y < 8; ++y) acc[x][y] = fmaf(av[x], bv[y], acc[x][y]);
        }
        if (kt + 1 < nk) {
            sstore(buf ^ 1);
            __syncthreads();
        }
    }
#pragma unroll
    for (int x = 0; x < 8; ++x) {
        const int m = m0 + (x >> 2) * 64 + ty * 4 + (x & 3);
        if (m >= n_users) continue;
        if (FILTER) {
            const float t = thr[m];
#pragma unroll
            for (int y = 0; y < 8; ++y) {
                const int64_t i = i0 + (y >> 2) * 64 + tx * 4 + (y & 3);
                const float v = acc[x][y] * c2;
                if (i < I && v >= t) {
                    const int pos = atomicAdd(&cnt[m], 1);
                    if (pos < cap)  // (score desc, item asc) as one descending 64-bit key
                        cand_key[(size_t)m * cap + pos] =
                            ((unsigned long long)okey(v) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
                }
            }
        } else {
            float *row = S + (size_t)m * (size_t)I;
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int64_t i = i0 + half * 64 + tx * 4;
                if (i + 3 < I && (((size_t)m * (size_t)I + (size_t)i) & 3) == 0) {
                    *reinterpret_cast<float4 *>(row + i) = make_float4(acc[x][half * 4 + 0] * c2, acc[x][half * 4 + 1] * c2,
                                                                       acc[x][half * 4 + 2] * c2, acc[x][half * 4 + 3] * c2);
                } else {
#pragma unroll
                    for (int y = 0; y < 4; ++y)
                        if (i + y < I) row[i + y] = acc[x][half * 4 + y] * c2;
                }
            }
        }
    }
}

__global__ void k_mask(float *__restrict__ S, int64_t I, const int64_t *__restrict__ excl_ptr,
                       const int32_t *__restrict__ excl_idx, int64_t first_user, int n_users, int *err) {
    const int m = blockIdx.x;
    if (m >= n_users) return;
    const int64_t a = excl_ptr[first_user + m], b = excl_ptr[first_user + m + 1];
    for (int64_t e = a + threadIdx.x; e < b; e += blockDim.x) {
        const uint32_t i = (uint32_t)excl_idx[e];
        if ((int64_t)i < I)
            S[(size_t)m * (size_t)I + i] = -INFINITY;
        else {
            atomicOr(&err[0], 1);
            atomicMin(&err[1], (int)(first_user + m));
        }
    }
}


// From a histogram (bins ascending), find the bin holding the `need`-th largest element; returns the bin and
// updates need to the rank inside that bin (1-based count still required from it).
__device__ int pick_bin(const unsigned *hist, int nbins, int &need, unsigned *scratch) {
    // single-thread scan from the top: nbins <= 2048, called by thread 0 only
    int b = nbins - 1;
    int acc = 0;
    for (; b > 0; --b) {
        if (acc + (int)hist[b] >= need) break;
        acc += (int)hist[b];
    }
    need -= acc;
    (void)scratch;
    return b;
}

constexpr int SEL_THREADS = 1024;

__global__ void __launch_bounds__(SEL_THREADS) k_select_topk(const float *__restrict__ S, int64_t I, int K,
                                                             int64_t first_user, int32_t *__restrict__ out_item,
                                                             float *__restrict__ out_score) {
    __shared__ unsigned hist[2048];
    __shared__ uint32_t sel_key[128];
    __shared__ int32_t sel_idx[128];
    __shared__ int s_bin, s_need, s_cnt, s_eqtaken;
    __shared__ int warp_cnt[SEL_THREADS / 32];
    const int tid = threadIdx.x;
    const float *row = S + (size_t)blockIdx.x * (size_t)I;
    const int64_t n = I;

    uint32_t prefix = 0;     // key bits decided so far
    uint32_t pmask = 0;      // which bits of the key are decided
    int need = K;
    const int shifts[3] = {21, 10, 0};
    const int widths[3] = {11, 11, 10};
    for (int pass = 0; pass < 3; ++pass) {
        const int nb = 1 << widths[pass];
        for (int b = tid; b < nb; b += SEL_THREADS) hist[b] = 0;
        __syncthreads();
        for (int64_t i = tid; i < n; i += SEL_THREADS) {
            const uint32_t k = okey(row[i]);
            if ((k & pmask) == prefix) atomicAdd(&hist[(k >> shifts[pass]) & (nb - 1)], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            int nd = need;
            s_bin = pick_bin(hist, nb, nd, nullptr);
            s_need = nd;
        }
        __syncthreads();
        prefix |= (uint32_t)s_bin << shifts[pass];
        pmask |= (uint32_t)(nb - 1) << shifts[pass];
        need = s_need;
        __syncthreads();
    }
    const uint32_t T = prefix;        // key of the K-th largest score
    const int take_eq = need;         // how many elements equal to T belong to the top K (lowest item ids first)
    const int eq_total = (int)hist[T & 1023u];
    if (tid == 0) {
        s_cnt = 0;
        s_eqtaken = 0;
    }
    __syncthreads();
    if (eq_total == take_eq) {  // common case: no tie straddles the K boundary -> one unordered collection pass
        for (int64_t i = tid; i < n; i += SEL_THREADS) {
            const uint32_t k = okey(row[i]);
            if (k >= T) {
                const int slot = atomicAdd(&s_cnt, 1);
                if (slot < 128) {
                    sel_key[slot] = k;
                    sel_idx[slot] = (int32_t)i;
                }
            }
        }
    } else {  // ties across the boundary: equal elements are taken in ascending item order
        for (int64_t base = 0; base < n; base += SEL_THREADS) {
            const int64_t i = base + tid;
            const uint32_t k = (i < n) ? okey(row[i]) : 0u;
            const bool gt = (i < n) && (k > T);
            const bool eq = (i < n) && (k == T);
            if (gt) {
                const int slot = atomicAdd(&s_cnt, 1);
                if (slot < 128) {
                    sel_key[slot] = k;
                    sel_idx[slot] = (int32_t)i;
                }
            }
            // ordered rank of the equal elements of this stripe
            const unsigned bal = __ballot_sync(0xffffffffu, eq);
            const int lane = tid & 31, w = tid >> 5;
            if (lane == 0) warp_cnt[w] = __popc(bal);
            __syncthreads();
            int before = s_eqtaken;
            for (int ww = 0; ww < w; ++ww) before += warp_cnt[ww];
            const int rank = before + __popc(bal & ((1u << lane) - 1u));
            if (eq && rank < take_eq) {
                const int slot = atomicAdd(&s_cnt, 1);
                if (slot < 128) {
                    sel_key[slot] = k;
                    sel_idx[slot] = (int32_t)i;
                }
            }
            __syncthreads();
            if (tid == 0) {
                int tot = 0;
                for (int ww = 0; ww < SEL_THREADS / 32; ++ww) tot += warp_cnt[ww];
                s_eqtaken += tot;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    // order the K winners: (score desc, item asc) by rank counting
    const int cnt = min(s_cnt, 128);
    if (tid < cnt) {
        const uint32_t k = sel_key[tid];
        const int32_t idx = sel_idx[tid];
        int rank = 0;
        for (int j = 0; j < cnt; ++j) {
            const uint32_t kj = sel_key[j];
            const int32_t ij = sel_idx[j];
            rank += (kj > k) || (kj == k && ij < idx);
        }
        if (rank < K) {
            out_item[(size_t)(first_user + blockIdx.x) * K + rank] = idx;
            out_score[(size_t)(first_user + blockIdx.x) * K + rank] = okey_inv(k);
        }
    }
}

// Grow-only [rows, I] score tile in the handle's workspace (h->scores, `need` floats).
static int exact_scores_reserve(daisy_ctx *h, size_t need, cudaStream_t s) {
    if (h->scores_cap < need) {
        DAISY_CUDA(cudaStreamSynchronize(s));
        if (h->scores) cudaFree(h->scores);
        h->scores = nullptr;
        h->scores_cap = 0;
        cudaError_t e = cudaMalloc((void **)&h->scores, need * sizeof(float));
        DAISY_REQUIRE(e == cudaSuccess, DAISY_ENOMEM, "cudaMalloc of the %zu-byte score tile failed: %s",
                      need * sizeof(float), cudaGetErrorString(e));
        h->scores_cap = need;
    }
    return DAISY_OK;
}

}  // namespace
