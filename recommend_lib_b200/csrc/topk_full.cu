// Full-catalogue scoring + exact top-K for sm_100a: daisy_topk_full.
//
// Replaces (reference, file:line): the final ranking loop BPRMFRecommender.py:196-207 -- one scalar
// model(tensor(u), tensor(i), tensor(i)) forward per (user, candidate) followed by np.argsort -- by
//   k_score_tile   fp32 register-tiled scores S[m, i] = c^2 <P[users[m]], Q[i]> for a tile of users x ALL items
//                  (CUDA cores on purpose: the scores must be fp32 sums of fp32 products for ranking parity),
//   k_mask         optional -inf on each user's training positives (CSR lists),
//   k_select_topk  one block per user: exact radix select (11 + 11 + 10 bits of the order-preserving key) of the
//                  K-th largest score, then collection and a (score desc, item asc) ordering of the K winners.
// The score tile lives in the handle's workspace (<= ~1 GiB), users are processed tile by tile.
#include <float.h>
#include <string.h>

#include "ctx.cuh"
#include "topk_tc.cuh"

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

// rows of a strided sample of the catalogue, gathered contiguously: Qs[j] = Q[j * stride]
__global__ void k_sample_rows(const float *__restrict__ Q, int64_t stride, int Ms, int D4, float *__restrict__ Qs) {
    const int lane = threadIdx.x & 31;
    const int w = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (w >= Ms) return;
    for (int e = lane; e < D4; e += 32) st_row(Qs, (size_t)w * D4 + e, ld_row(Q, (size_t)w * stride * D4 + e));
}

__global__ void k_thr_from_topk(const float *__restrict__ top_scores, int r, int n, float *__restrict__ thr,
                                int *__restrict__ cnt) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    thr[m] = top_scores[(size_t)m * r + (r - 1)];  // r-th largest score of the user's sample
    cnt[m] = 0;
}

// Exact top-K of one user's candidate list: bitonic sort of the 64-bit (score desc, item asc) keys in shared memory.
// Excluded items (the user's training positives, CSR) are dropped first; an exclusion id outside [0, I) raises the
// handle's error flag, as k_mask does on the exact path.  A user whose list overflowed, holds fewer than K admissible
// candidates, or whose K-th admissible candidate scores below the threshold thr[m] is handed to the exact fallback (flag
// in redo[m]).  The last case needs a candidate list that is a superset: the list holds every item at or above thr, but
// only some of those below (the tensor-core filter's margin), so once the exclusions reach below thr the best items
// left need not be in it.
__global__ void __launch_bounds__(1024) k_select_cand(const unsigned long long *__restrict__ cand_key,
                                                       const int *__restrict__ cnt, const float *__restrict__ thr, int cap,
                                                       int K, int64_t first_user,
                                                       const int64_t *__restrict__ excl_ptr,
                                                       const int32_t *__restrict__ excl_idx, int64_t I,
                                                       int32_t *__restrict__ out_item, float *__restrict__ out_score,
                                                       int *__restrict__ redo, int *err) {
    extern __shared__ unsigned long long keys[];
    const int m = blockIdx.x, tid = threadIdx.x;
    if (excl_ptr && excl_idx)
        for (int64_t e = excl_ptr[first_user + m] + tid; e < excl_ptr[first_user + m + 1]; e += blockDim.x)
            if ((int64_t)(uint32_t)excl_idx[e] >= I) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], (int)(first_user + m));
            }
    const int n = cnt[m];
    if (n > cap || n < K) {
        if (tid == 0) redo[m] = 1;
        return;
    }
    int P2 = 1;
    while (P2 < n) P2 <<= 1;
    const int64_t ea = excl_ptr ? excl_ptr[first_user + m] : 0, eb = excl_ptr ? excl_ptr[first_user + m + 1] : 0;
    for (int p = tid; p < P2; p += blockDim.x) {
        unsigned long long k = (p < n) ? cand_key[(size_t)m * cap + p] : 0ull;
        if (p < n && eb > ea) {
            const int32_t item = (int32_t)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull));
            for (int64_t e = ea; e < eb; ++e)
                if (excl_idx[e] == item) {
                    k = 0ull;
                    break;
                }
        }
        keys[p] = k;
    }
    __syncthreads();
    for (int size = 2; size <= P2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int p = tid; p < P2 / 2; p += blockDim.x) {
                const int lo = 2 * p - (p & (stride - 1)), hi = lo + stride;
                const bool desc = ((lo & size) == 0);
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a < b) == desc) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
            __syncthreads();
        }
    // fewer than K admissible candidates after the exclusions, or the K-th of them below the threshold
    if (keys[K - 1] == 0ull || okey_inv((uint32_t)(keys[K - 1] >> 32)) < thr[m]) {
        if (tid == 0) redo[m] = 1;
        return;
    }
    if (tid < K) {
        const unsigned long long k = keys[tid];
        out_item[(size_t)(first_user + m) * K + tid] = (int32_t)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull));
        out_score[(size_t)(first_user + m) * K + tid] = okey_inv((uint32_t)(k >> 32));
    }
}

}  // namespace

extern "C" int daisy_topk_full(daisy_handle_t h, const float *P, const float *Q, const int32_t *users, int64_t N, int K,
                               const int64_t *excl_ptr, const int32_t *excl_idx, int32_t *out_item, float *out_score,
                               daisy_stream_t stream) {
    DAISY_REQUIRE(h && P && Q, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(h->D % 4 == 0, DAISY_EUNSUPPORTED, "daisy_topk_full needs dim %% 4 == 0 (dim is %d)", h->D);
    DAISY_REQUIRE(K >= 1 && K <= 128 && (int64_t)K <= h->I, DAISY_EUNSUPPORTED, "top_k %d unsupported (1..min(128, item_num))", K);
    DAISY_REQUIRE(N >= 0 && N < (1LL << 31), DAISY_EINVAL, "bad user count");
    h->topk_path = DAISY_TOPK_PATH_EXACT;
    h->topk_filtered = h->topk_redone = 0;
    if (N == 0) return DAISY_OK;
    DAISY_REQUIRE(users && out_item && out_score, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE((excl_ptr == nullptr) == (excl_idx == nullptr) || excl_ptr != nullptr, DAISY_EINVAL,
                  "exclusion lists need both excl_ptr and excl_idx");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t I = h->I;
    // user tile: as many rows of scores as fit ~1 GiB, at least BM so the score kernel's tiles are full
    int64_t tile = (int64_t)((1ull << 30) / ((uint64_t)I * sizeof(float)));
    if (tile < 1) tile = 1;
    if (tile > 4096) tile = 4096;
    if (tile > N) tile = N;
    const float c2 = (float)(h->scale * h->scale);
    // ---- exact path over a user range (materialised score tile + radix select); used for small catalogues and as
    //      the fallback of the filtered path ----
    auto exact_range = [&](const int32_t *us, int64_t n_us, int64_t out_first) -> int {
        const int64_t rows = tile < n_us ? tile : n_us;
        const size_t need = (size_t)rows * (size_t)I;
        if (h->scores_cap < need) {  // grow-only score tile in the handle's workspace
            DAISY_CUDA(cudaStreamSynchronize(s));
            if (h->scores) cudaFree(h->scores);
            h->scores = nullptr;
            h->scores_cap = 0;
            cudaError_t e = cudaMalloc((void **)&h->scores, need * sizeof(float));
            DAISY_REQUIRE(e == cudaSuccess, DAISY_ENOMEM, "cudaMalloc of the %zu-byte score tile failed: %s",
                          need * sizeof(float), cudaGetErrorString(e));
            h->scores_cap = need;
        }
        for (int64_t first = 0; first < n_us; first += tile) {
            const int nu = (int)((n_us - first < tile) ? (n_us - first) : tile);
            dim3 grid((unsigned)((I + BN - 1) / BN), (unsigned)((nu + BM - 1) / BM));
            k_score_tile<false><<<grid, 256, 0, s>>>(P, Q, us + first, nu, (uint32_t)h->U, I, h->D, c2, h->scores, h->err,
                                                     nullptr, nullptr, nullptr, 0);
            DAISY_LAUNCH_CHECK(h);
            if (excl_ptr && excl_idx) {
                k_mask<<<nu, 128, 0, s>>>(h->scores, I, excl_ptr, excl_idx, out_first + first, nu, h->err);
                DAISY_LAUNCH_CHECK(h);
            }
            k_select_topk<<<nu, SEL_THREADS, 0, s>>>(h->scores, I, K, out_first + first, out_item, out_score);
            DAISY_LAUNCH_CHECK(h);
        }
        return DAISY_OK;
    };
    // ---- filtered path (large catalogues): no score matrix is materialised.
    //   1. scores of a strided SAMPLE of Ms items per user -> the r-th largest is the user's threshold; r is chosen so
    //      that about E >= 16 K items of the full catalogue exceed it (Beta(r, Ms - r + 1) fraction: E +- E / sqrt(r))
    //   2. the full score GEMM appends every item at or above the threshold to the user's candidate list
    //   3. exact (score desc, item asc) top-K of the list; a user whose list is short of K admissible items or
    //      overflowed (never seen in practice) is redone by the exact path.
    const int Ms = 8192;
    const char *force = getenv("DAISY_TOPK_PATH");
    const bool want_filter = force ? (strcmp(force, "filter") == 0) : (I >= 16 * (int64_t)Ms);
    if (!want_filter || I < 4 * (int64_t)Ms) {
        return exact_range(users, N, 0);
    }
    const int64_t stride = I / Ms;
    const int E = K * 16 > 2048 ? K * 16 : 2048;
    int r = (int)(((int64_t)E * Ms + I - 1) / I);
    if (r < 8) r = 8;
    if (r > 128) return exact_range(users, N, 0);
    const int cap = 4 * E;  // 8192 at K <= 128: 64 KB of keys in shared memory for the final sort
    // step 2 on the tensor cores (topk_tc.cu: BF16 tcgen05 filter with an error-bounded threshold, then the exact fp32
    // re-scoring of the candidates) unless DAISY_TOPK_TC=0 or the shape is outside its range (dim > 128)
    const char *tc_env = getenv("DAISY_TOPK_TC");
    const bool use_tc = !(tc_env && atoi(tc_env) == 0) && daisy_tc_supported(h);
    h->topk_path = use_tc ? DAISY_TOPK_PATH_TC : DAISY_TOPK_PATH_SIMT;
    const int64_t Tu_max = use_tc ? 16384 : 4096;
    const int64_t Tu = N < Tu_max ? N : Tu_max;
    TcItems tci = {nullptr, nullptr, 0};
    float *Qs = nullptr, *Ss = nullptr, *tscore = nullptr, *thr = nullptr;
    int32_t *titem = nullptr;
    int *cnt = nullptr, *redo = nullptr;
    unsigned long long *cand = nullptr;
    bool ok = daisy_scratch_alloc(h, (void **)&Qs, (size_t)Ms * h->D * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&Ss, (size_t)Tu * Ms * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&tscore, (size_t)Tu * r * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&titem, (size_t)Tu * r * sizeof(int32_t), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&thr, (size_t)Tu * sizeof(float), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&cnt, (size_t)Tu * sizeof(int), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&redo, (size_t)N * sizeof(int), s) == cudaSuccess;
    ok = ok && daisy_scratch_alloc(h, (void **)&cand, (size_t)Tu * cap * sizeof(unsigned long long), s) == cudaSuccess;
    int rc = DAISY_OK;
    int *redo_host = nullptr;
    if (!ok) {
        cudaGetLastError();
        daisy_set_error("top-K workspace allocation failed");
        rc = DAISY_ENOMEM;
    } else {
        cudaMemsetAsync(redo, 0, (size_t)N * sizeof(int), s);
        k_sample_rows<<<daisy_ceil_div(Ms, 8), 256, 0, s>>>(Q, stride, Ms, h->D / 4, Qs);
        h->launches++;
        cudaFuncSetAttribute(k_select_cand, cudaFuncAttributeMaxDynamicSharedMemorySize, cap * (int)sizeof(unsigned long long));
        if (use_tc) rc = daisy_tc_prepare_items(h, Q, &tci, s);
        for (int64_t first = 0; first < N && !rc; first += Tu) {
            const int nu = (int)((N - first < Tu) ? (N - first) : Tu);
            dim3 gs((unsigned)((Ms + BN - 1) / BN), (unsigned)((nu + BM - 1) / BM));
            k_score_tile<false><<<gs, 256, 0, s>>>(P, Qs, users + first, nu, (uint32_t)h->U, Ms, h->D, c2, Ss, h->err, nullptr,
                                                   nullptr, nullptr, 0);
            k_select_topk<<<nu, SEL_THREADS, 0, s>>>(Ss, Ms, r, 0, titem, tscore);
            k_thr_from_topk<<<daisy_ceil_div(nu, 256), 256, 0, s>>>(tscore, r, nu, thr, cnt);
            if (use_tc) {
                rc = daisy_tc_filter(h, P, Q, &tci, users + first, nu, c2, thr, cnt, cand, cap, (int)((int64_t)r * I / Ms), s);
                if (rc) break;
            } else {
                dim3 gf((unsigned)((I + BN - 1) / BN), (unsigned)((nu + BM - 1) / BM));
                k_score_tile<true><<<gf, 256, 0, s>>>(P, Q, users + first, nu, (uint32_t)h->U, I, h->D, c2, nullptr, h->err, thr,
                                                      cnt, cand, cap);
            }
            k_select_cand<<<nu, 1024, cap * sizeof(unsigned long long), s>>>(cand, cnt, thr, cap, K, first, excl_ptr, excl_idx, I,
                                                                             out_item, out_score, redo + first, h->err);
            h->launches += 5;
        }
        if (!rc && cudaGetLastError() != cudaSuccess) {
            daisy_set_error("top-K launch failed");
            rc = DAISY_ECUDA;
        }
        daisy_tc_free_items(&tci, s);
        redo_host = (int *)malloc((size_t)N * sizeof(int));
        if (!rc && (!redo_host || cudaMemcpyAsync(redo_host, redo, (size_t)N * sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                    cudaStreamSynchronize(s) != cudaSuccess)) {
            daisy_set_error("top-K fallback list read-back failed");
            rc = DAISY_ECUDA;
        }
    }
    for (void *p : {(void *)Qs, (void *)Ss, (void *)tscore, (void *)titem, (void *)thr, (void *)cnt, (void *)redo, (void *)cand})
        if (p) cudaFreeAsync(p, s);
    if (!rc)
        for (int64_t m = 0; m < N && !rc; ++m)
            if (redo_host[m]) {
                rc = exact_range(users + m, 1, m);
                h->topk_redone++;
            }
    if (!rc) h->topk_filtered = N - h->topk_redone;
    free(redo_host);
    return rc;
}

extern "C" int daisy_topk_full_path(daisy_handle_t h, int *path, int64_t *filtered, int64_t *redone) {
    DAISY_REQUIRE(h && path && filtered && redone, DAISY_EINVAL, "null argument");
    *path = h->topk_path;
    *filtered = h->topk_filtered;
    *redone = h->topk_redone;
    return DAISY_OK;
}

