// SVD++ (SURVEY.md section 8f, row N4): SVDpp.fit / SVDpp.predict of util/matrix_factorization.pyx:169-288.
//
// STATUS: GPU-verified in round 2 (tests/test_svdpp_gpu.py passes on a B200 and runs in the default -m gpu suite; bench line under
// profiles/r02a_bench_svdpp.json).  Before that it had run under the host emulation of tests/emu
// (tests/test_kernel_emulation.py: golden run + oracle green), which still covers it on CPU.
// The checker (the C restatement of the loop under oracle/) is bit-identical to the reference's own compiled class.
//
// The reference loop (:236-263) is strictly sequential, and unlike funk-SVD (csrc/mf.cu) it has no dataflow
// parallelism to speak of: rating t of user u rewrites the implicit-feedback row yj[j] of EVERY item j the user rated
// (:261-263), so two ratings conflict whenever their users share one item -- on ml-1m practically always.  What is
// left is the parallelism INSIDE one rating: |Iu| rows of D doubles gathered, then rewritten (165 rows x 128 factors
// on ml-1m at D = 128).  First version, deliberately without any inter-block synchronisation (nothing can spin):
//
//   k_svdpp_validate   grid-wide id check (users, items, the lists) -> the handle's sticky error flag
//   k_svdpp_seq<M>     ONE thread block walks the ratings in order; a warp per history row, a lane per 32-strided
//                      factor.  Per rating: (1) warps sum their rows of yj, fixed-order cross-warp sum in shared
//                      memory -> u_impl; (2) dot product <qi, pu + u_impl> by warp tree + fixed-order sum over warps
//                      -> err; (3) biases, pu, qi (old values, :254-258), then every yj row of the history with the
//                      OLD qi (:261-263).  The header (u, i, r, list range) of rating t + 2, the item list and the
//                      rating's own rows of rating t + 1 are fetched while rating t computes, so the dependent-load
//                      chain users[t] -> ur_ptr[u] -> ur_idx[k] -> yj row is off the critical path: no load issued
//                      between two barriers of a rating is consumed before the next one, except the history rows.
//                      A history that holds an item m times (a repeated (user, item) rating) applies that row's update
//                      m times in a row from the thread owning its first occurrence (`ur_mult`), which is what the
//                      reference's `for j in Iu` does.
//   k_svdpp_user_factors   z[u] = pu[u] + sum_{j in Iu} yj[j] / sqrt|Iu| (:281-286), a warp per user; predict is then
//                      daisy_mf_predict(z, qi, bu, bi) -- the history is summed once per user, not once per candidate.
//
// Arithmetic: float64 throughout; the result is the sequential result up to the rounding of the two re-associated sums
// (rows over warps, factors over lanes); the element-wise updates are the reference's expressions.  The tables of the
// reference script's sizes are L2-resident (ml-1m, D = 128: 3 x 3.8 MB + 6 MB), so the bound is one SM's L2 bandwidth:
// 2 x |Iu| x 8D bytes per rating.  Measured (ml-1m shape, n_factors 20): 5 us per rating = 0.19-0.20 M ratings/s, the barrier
// chain (3 block barriers + one L2 round trip per rating), barely ahead of one host core.  Second version (not built): the factors are independent
// given err, so a thread-block cluster can own D / 16 factors per block -- its slice of yj in shared memory --
// and exchange one partial dot product per rating through distributed shared memory.
#include "ctx.cuh"

namespace {

constexpr int SP_MAX_D = 512;   // 16 lane-strided factors per lane
constexpr int SP_CAP = 2048;    // history entries of the next rating prefetched into shared memory (longer ones: global reads)

struct SpHdr {
    long long p0;   // first entry of the user's list in ur_idx
    double r;
    int u, i, nI, pad;
};

struct SpArgs {
    double *pu, *qi, *yj, *bu, *bi;
    const int32_t *users, *items;
    const double *ratings;
    const int64_t *ur_ptr;
    const int32_t *ur_idx, *ur_mult;   // ur_mult may be null: no item repeats inside a list
    double *sse_out;                   // [epochs] or null
    const int *err;
    long long n;
    int epochs, D;
    daisy_svdpp_params prm;
};

__global__ void k_svdpp_validate(const int32_t *users, const int32_t *items, long long n, const int64_t *ur_ptr,
                                 const int32_t *ur_idx, long long U, long long I, int *err) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long t = g; t < n; t += stride) {
        const long long u = users[t], i = items[t];
        if (u < 0 || u >= U || i < 0 || i >= I) {
            atomicOr(err, (u < 0 || u >= U) ? 1 : 2);
            atomicMin(err + 1, (int)(t < 0x7fffffffLL ? t : 0x7fffffffLL));
        }
    }
    for (long long u = g; u < U; u += stride)
        if (ur_ptr[u + 1] < ur_ptr[u] || ur_ptr[u] < 0) atomicOr(err, 4);
    const long long total = ur_ptr[U];
    for (long long k = g; k < total; k += stride)
        if (ur_idx[k] < 0 || ur_idx[k] >= I) atomicOr(err, 2);
}

template <int M>
__global__ void __launch_bounds__(M >= 8 ? 512 : 1024, 1) k_svdpp_seq(SpArgs a) {   // D > 128: 512 threads, 128 registers
    extern __shared__ double sp_smem[];
    constexpr int KEEP = M == 1 ? 6 : (M == 2 ? 3 : 0);   // history rows per warp held in registers between phases (1) and (3)
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, W = blockDim.x >> 5, T = blockDim.x;
    const int D = a.D;
    double *red = sp_smem;                  // [W][D]  per-warp partial sums of the history rows
    double *qold = red + (size_t)W * D;     // [D]     qi[i] before this rating's update
    double *wsum = qold + D;                // [32]    per-warp partial dot products
    double *nb = wsum + 32;                 // [2]     bu[u], bi[i] of the current rating
    SpHdr *hdr = reinterpret_cast<SpHdr *>(nb + 2);              // [3]     ring: current, next, the one being fetched
    int *list = reinterpret_cast<int *>(hdr + 3);                // [2][SP_CAP] item ids of the current / next history
    int *mlist = list + 2 * SP_CAP;                              // [2][SP_CAP] their multiplicities
    if (a.err[0] != 0) return;              // an id failed validation: touch nothing (block-uniform)
    const long long total = a.n * (long long)a.epochs;
    if (total == 0) return;
    const daisy_svdpp_params prm = a.prm;
    const int Dw = (D + 31) >> 5;           // warps holding factors in the dot product

    auto load_hdr = [&](long long t, SpHdr *h) {   // prologue only: one thread, two dependent loads
        const int u = a.users[t], i = a.items[t];
        h->u = u;
        h->i = i;
        h->r = a.ratings[t];
        const long long p0 = a.ur_ptr[u];
        h->p0 = p0;
        h->nI = (int)(a.ur_ptr[u + 1] - p0);
    };
    auto copy_list = [&](const SpHdr *h, int buf) {   // all threads
        const int m = h->nI < SP_CAP ? h->nI : SP_CAP;
        for (int k = tid; k < m; k += T) {
            list[buf * SP_CAP + k] = a.ur_idx[h->p0 + k];
            mlist[buf * SP_CAP + k] = a.ur_mult ? a.ur_mult[h->p0 + k] : 1;
        }
    };

    // Everything a rating needs besides the history rows travels ahead of it, so that no dependent load sits between two
    // of its barriers: the header (u, i, r, list range) two ratings ahead -- ids fetched at the top of a rating, the list
    // range after its second barrier, written to the ring before its third; the item list and the rating's own rows
    // pu[u], qi[i], bu[u], bi[i] one rating ahead, the latter fetched by the very thread that wrote them last, so a
    // rating that repeats the user or the item reads its predecessor's values by program order.
    if (tid == 0) {
        load_hdr(0, &hdr[0]);
        if (total > 1) load_hdr(a.n > 1 ? 1 : 0, &hdr[1]);
    }
    __syncthreads();
    copy_list(&hdr[0], 0);
    double puf = 0.0, qif = 0.0, nbu = 0.0, nbi = 0.0;
    if (tid < D) {
        puf = a.pu[(size_t)hdr[0].u * D + tid];
        qif = a.qi[(size_t)hdr[0].i * D + tid];
    }
    if (tid == 0) {
        nbu = a.bu[hdr[0].u];
        nbi = a.bi[hdr[0].i];
    }
    __syncthreads();

    double sse = 0.0;                       // thread 0
    long long t = 0;                        // position of rating s inside its epoch
    long long t2 = 2 % a.n;                 // ... of rating s + 2
    int epoch = 0, c0 = 0;                  // c0 = s % 3
    for (long long s = 0; s < total; ++s) {
        const int c1 = c0 == 2 ? 0 : c0 + 1, c2 = c1 == 2 ? 0 : c1 + 1, lb = (int)(s & 1);
        const SpHdr *h = &hdr[c0];
        const int u = h->u, i = h->i, nI = h->nI;
        const long long p0 = h->p0;
        const double r = h->r;
        const double sqrt_Iu = sqrt((double)nI);                                  // :241
        const int *lst = list + lb * SP_CAP, *mls = mlist + lb * SP_CAP;
        if (tid == 0) {                     // fetched during the previous rating; read after the second barrier
            nb[0] = nbu;
            nb[1] = nbi;
        }
        const bool pf2 = tid == T - 1 && s + 2 < total;
        int h2u = 0, h2i = 0;
        double h2r = 0.0;
        if (pf2) {                          // issued here, consumed after the second barrier
            h2u = a.users[t2];
            h2i = a.items[t2];
            h2r = a.ratings[t2];
        }

        // (1) implicit feedback: sum of the history rows (:243-246)
        // The first KEEP rows of every warp (histories of up to KEEP * W rows: all of them at the script's sizes) are
        // loaded back to back into registers -- KEEP independent L2 round trips in flight instead of a load -> add chain
        // per row -- and stay there for phase (3), which used to read every row a second time.  Same additions in the
        // same order: bit-identical to the row-by-row walk.
        double acc[M], keep[KEEP > 0 ? KEEP : 1][M];
#pragma unroll
        for (int m = 0; m < M; ++m) acc[m] = 0.0;
#pragma unroll
        for (int j = 0; j < KEEP; ++j) {
            const int k = w + j * W;
            const bool on = k < nI;         // warp-uniform
            const double *row = on ? a.yj + (size_t)(k < SP_CAP ? lst[k] : a.ur_idx[p0 + k]) * D : nullptr;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const int f = lane + 32 * m;
                keep[j][m] = (on && f < D) ? row[f] : 0.0;
            }
        }
#pragma unroll
        for (int j = 0; j < KEEP; ++j)
#pragma unroll
            for (int m = 0; m < M; ++m)
                if (w + j * W < nI) acc[m] += keep[j][m];
        for (int k = w + KEEP * W; k < nI; k += W) {
            const double *row = a.yj + (size_t)(k < SP_CAP ? lst[k] : a.ur_idx[p0 + k]) * D;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const int f = lane + 32 * m;
                if (f < D) acc[m] += row[f];
            }
        }
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const int f = lane + 32 * m;
            if (f < D) red[(size_t)w * D + f] = acc[m];
        }
        __syncthreads();

        // (2) u_impl, dot product, err (:248-252)
        double ui = 0.0, prod = 0.0;
        if (tid < D) {
            double sum = 0.0;
            // every warp has written its partial (zeros where it had no row), so the loop runs over all W of them with a
            // fixed trip count the compiler can unroll: the shared-memory loads go out together instead of one per add
            // (adding the trailing zeros changes nothing)
#pragma unroll 8
            for (int w2 = 0; w2 < W; ++w2) sum += red[(size_t)w2 * D + tid];
            ui = nI > 0 ? sum / sqrt_Iu : 0.0;
            qold[tid] = qif;
            prod = qif * (puf + ui);
        }
        if (w < Dw) {
            const double ws = warp_sum_d(prod);
            if (lane == 0) wsum[w] = ws;
        }
        __syncthreads();
        long long h2p0 = 0, h2p1 = 0;
        if (pf2) {                          // second link of the header chain, consumed before the third barrier
            h2p0 = a.ur_ptr[h2u];
            h2p1 = a.ur_ptr[h2u + 1];
        }
        double dot = 0.0;
        for (int w2 = 0; w2 < Dw; ++w2) dot += wsum[w2];
        const double b_u = nb[0], b_i = nb[1];
        const double err = r - (prm.global_mean + b_u + b_i + dot);               // identical in every thread

        // (3) updates (:254-263)
        const bool more = s + 1 < total;
        const SpHdr *hn = &hdr[c1];         // the next rating (complete since the previous rating's third barrier)
        if (tid == 0) {
            sse += err * err;
            a.bu[u] = b_u + prm.lr_bu * (err - prm.reg_bu * b_u);
            a.bi[i] = b_i + prm.lr_bi * (err - prm.reg_bi * b_i);
            if (t == a.n - 1) {
                if (a.sse_out) a.sse_out[epoch] = sse;
                sse = 0.0;
            }
            if (more) {                     // after the two stores above, in program order
                nbu = a.bu[hn->u];
                nbi = a.bi[hn->i];
            }
        }
        if (tid < D) {
            a.pu[(size_t)u * D + tid] = puf + prm.lr_pu * (err * qif - prm.reg_pu * puf);
            a.qi[(size_t)i * D + tid] = qif + prm.lr_qi * (err * (puf + ui) - prm.reg_qi * qif);
            if (more) {                     // next rating's rows: issued now, consumed after the next two barriers
                puf = a.pu[(size_t)hn->u * D + tid];
                qif = a.qi[(size_t)hn->i * D + tid];
            }
        }
        double c[M];
#pragma unroll
        for (int m = 0; m < M; ++m) {
            const int f = lane + 32 * m;
            c[m] = f < D ? err * qold[f] / sqrt_Iu : 0.0;
        }
#pragma unroll
        for (int j = 0; j < KEEP; ++j) {    // the rows still in registers
            const int k = w + j * W;
            if (k >= nI) break;             // warp-uniform
            const int mult = k < SP_CAP ? mls[k] : (a.ur_mult ? a.ur_mult[p0 + k] : 1);
            if (mult == 0) continue;        // a later occurrence of an item: its first occurrence applies both
            double *row = a.yj + (size_t)(k < SP_CAP ? lst[k] : a.ur_idx[p0 + k]) * D;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const int f = lane + 32 * m;
                if (f < D) {
                    double y = keep[j][m];
                    for (int rep = 0; rep < mult; ++rep) y += prm.lr_yj * (c[m] - prm.reg_yj * y);
                    row[f] = y;
                }
            }
        }
        for (int k = w + KEEP * W; k < nI; k += W) {
            const int mult = k < SP_CAP ? mls[k] : (a.ur_mult ? a.ur_mult[p0 + k] : 1);
            if (mult == 0) continue;        // a later occurrence of an item: its first occurrence applies both
            double *row = a.yj + (size_t)(k < SP_CAP ? lst[k] : a.ur_idx[p0 + k]) * D;
#pragma unroll
            for (int m = 0; m < M; ++m) {
                const int f = lane + 32 * m;
                if (f < D) {
                    double y = row[f];
                    for (int rep = 0; rep < mult; ++rep) y += prm.lr_yj * (c[m] - prm.reg_yj * y);
                    row[f] = y;
                }
            }
        }
        if (more) copy_list(hn, lb ^ 1);
        if (pf2) {
            SpHdr *hw = &hdr[c2];           // last read as the current header one rating ago
            hw->u = h2u;
            hw->i = h2i;
            hw->r = h2r;
            hw->p0 = h2p0;
            hw->nI = (int)(h2p1 - h2p0);
        }
        __syncthreads();
        c0 = c1;
        if (++t == a.n) {
            t = 0;
            ++epoch;
        }
        if (++t2 == a.n) t2 = 0;
    }
}

// z[u] = pu[u] + sum_{j in Iu} yj[j] / sqrt|Iu|   (SVDpp.predict, :281-286; a user without history keeps pu[u])
__global__ void k_svdpp_user_factors(const double *pu, const double *yj, const int64_t *ur_ptr, const int32_t *ur_idx,
                                     long long U, int D, double *z) {
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long u = wid; u < U; u += nw) {
        const long long p0 = ur_ptr[u], p1 = ur_ptr[u + 1];
        const double sq = sqrt((double)(p1 - p0));
        for (int f = lane; f < D; f += 32) {
            double sum = 0.0;
            for (long long k = p0; k < p1; ++k) sum += yj[(size_t)ur_idx[k] * D + f];
            z[(size_t)u * D + f] = pu[(size_t)u * D + f] + (p1 > p0 ? sum / sq : 0.0);
        }
    }
}

static size_t sp_smem_bytes(int threads, int D) {
    return ((size_t)(threads / 32) * D + (size_t)D + 32 + 2) * sizeof(double) + 3 * sizeof(SpHdr) + 4 * (size_t)SP_CAP * sizeof(int);
}

template <int M>
static int sp_launch(daisy_ctx *h, const SpArgs &a, int threads, cudaStream_t s) {
    const size_t smem = sp_smem_bytes(threads, a.D);
    DAISY_CUDA(cudaFuncSetAttribute(k_svdpp_seq<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_svdpp_seq<M><<<1, threads, smem, s>>>(a);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

}  // namespace

extern "C" int daisy_svdpp_fit(daisy_handle_t h, double *pu, double *qi, double *yj, double *bu, double *bi,
                               const int32_t *users, const int32_t *items, const double *ratings, int64_t n, int n_epochs,
                               const int64_t *ur_ptr, const int32_t *ur_idx, const int32_t *ur_mult,
                               const daisy_svdpp_params *prm, double *sse_out, daisy_stream_t stream) {
    DAISY_REQUIRE(h != nullptr && prm != nullptr, DAISY_EINVAL, "null handle or parameter block");
    DAISY_REQUIRE(pu && qi && yj && bu && bi && ur_ptr, DAISY_EINVAL, "null table / list pointer");
    DAISY_REQUIRE(n >= 0 && n_epochs >= 0, DAISY_EINVAL, "negative rating / epoch count");
    DAISY_REQUIRE(n == 0 || (users && items && ratings && ur_idx), DAISY_EINVAL, "null rating arrays");
    DAISY_REQUIRE(h->D >= 1 && h->D <= SP_MAX_D, DAISY_EUNSUPPORTED, "n_factors %d out of range (1..%d)", h->D, SP_MAX_D);
    DAISY_REQUIRE(h->U >= 1 && h->I >= 1, DAISY_EINVAL, "the handle was created without table sizes");
    if (n == 0 || n_epochs == 0) return DAISY_OK;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int D = h->D;
    const int vgrid = h->num_sms * 4;
    k_svdpp_validate<<<vgrid > 0 ? vgrid : 1, 256, 0, s>>>(users, items, (long long)n, ur_ptr, ur_idx, (long long)h->U,
                                                           (long long)h->I, h->err);
    DAISY_LAUNCH_CHECK(h);
    int threads = 1024;     // a warp per history row: 32 rows in flight
    if (const char *e = getenv("DAISY_SVDPP_THREADS")) threads = atoi(e);
    if (D > 128 && threads > 512) threads = 512;    // the launch bound of the wide instantiations (128 registers)
    const int need = ((D + 31) / 32) * 32;      // the factor phase wants one thread per factor
    DAISY_REQUIRE(threads % 32 == 0 && threads >= need && threads >= 32 && threads <= 1024, DAISY_EINVAL,
                  "DAISY_SVDPP_THREADS=%d: need a multiple of 32 in [%d, 1024]", threads, need > 32 ? need : 32);
    DAISY_REQUIRE(sp_smem_bytes(threads, D) <= 227 * 1024, DAISY_EUNSUPPORTED, "n_factors %d with %d threads needs %zu bytes of "
                  "shared memory", D, threads, sp_smem_bytes(threads, D));
    SpArgs a;
    a.pu = pu; a.qi = qi; a.yj = yj; a.bu = bu; a.bi = bi;
    a.users = users; a.items = items; a.ratings = ratings;
    a.ur_ptr = ur_ptr; a.ur_idx = ur_idx; a.ur_mult = ur_mult;
    a.sse_out = sse_out;
    a.err = h->err;
    a.n = (long long)n;
    a.epochs = n_epochs;
    a.D = D;
    a.prm = *prm;
    // No yj rows are kept resident in shared memory: measured at n_factors 20, 203 k ratings/s without them and 189 k
    // with (a row comes from L2 as fast as the slot indirection costs), so that option was removed (it is in git history).
    if (D <= 32) return sp_launch<1>(h, a, threads, s);
    if (D <= 64) return sp_launch<2>(h, a, threads, s);
    if (D <= 128) return sp_launch<4>(h, a, threads, s);
    if (D <= 256) return sp_launch<8>(h, a, threads, s);
    return sp_launch<16>(h, a, threads, s);
}

extern "C" int daisy_svdpp_user_factors(daisy_handle_t h, const double *pu, const double *yj, const int64_t *ur_ptr,
                                        const int32_t *ur_idx, double *z_out, daisy_stream_t stream) {
    DAISY_REQUIRE(h != nullptr && pu && yj && ur_ptr && z_out, DAISY_EINVAL, "null handle / table / list pointer");
    DAISY_REQUIRE(h->D >= 1 && h->U >= 1, DAISY_EINVAL, "the handle was created without table sizes");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    const int want = daisy_ceil_div(h->U, 8);
    const int cap = h->num_sms * 8;
    const int grid = want < cap ? want : cap;
    k_svdpp_user_factors<<<grid > 0 ? grid : 1, 256, 0, (cudaStream_t)stream>>>(pu, yj, ur_ptr, ur_idx, (long long)h->U, h->D,
                                                                               z_out);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}
