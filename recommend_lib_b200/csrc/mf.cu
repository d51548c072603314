// funk-SVD / RSVD SGD for sm_100a: daisy_mf_fit, daisy_mf_predict.
//
// Replaces (reference, file:line): the per-rating loops of util/matrix_factorization.pyx
//   SVD.fit  :132-151   RSVD.fit  :41-61   SVD.predict :157-167   RSVD.predict :68-78
//
// The reference loop is STRICTLY SEQUENTIAL: the update for rating t+1 reads the rows rating t wrote.  Two
// ratings only interact when they share the user row or the item row, so the loop is a dataflow graph: rating t
// depends on the previous rating of the same user and the previous rating of the same item.  The kernel runs
// that graph directly:
//   * per row a version counter = number of updates applied so far;
//   * for rating t of epoch e the expected versions are   e * (#ratings of the row) + (rank of t among the
//     ratings of the row), computed once per fit with two radix sorts + a max-scan;
//   * persistent warps claim ratings in sequence order from a ticket counter, wait (acquire loads, L2-coherent)
//     until both rows reached the expected version, apply the update in float64, and publish version + 1
//     (release stores).  A claimed ticket only ever waits on lower tickets, which are held by warps that are
//     already running, so the schedule cannot deadlock; a spin cap aborts with an error instead of hanging.
// Independent ratings run in parallel, dependent ones in the reference's order: the result is the sequential
// result up to float64 rounding of the warp-tree dot product (the row updates themselves are element-wise and
// therefore identical).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "ctx.cuh"

namespace {

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned *p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

struct MfArgs {
    double *pu, *qi, *bu, *bi;
    const int32_t *users, *items;
    const double *ratings;
    const int *need_u, *need_i, *cnt_u, *cnt_i;
    unsigned *ver_u, *ver_i;
    unsigned long long *ticket;
    double *err2;  // [epochs * n] squared errors (may be null)
    int *abort_flag;
    long long n;
    int epochs, D;
    daisy_mf_params prm;
    unsigned long long stall_ns;   // a waiter gives up when the whole grid made no progress for this long
};

__device__ __forceinline__ unsigned long long mf_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Stall detector of the two schedules' spin loops, called by the polling lane every 2^12 polls.  A wait may be
// legitimately long (a light warp waiting for the hot item's warp to finish an epoch), so the test is not "how long
// have I waited" but "how long has NOBODY moved": *progress is bumped by every warp as it works (the ticket counter
// of the ticket schedule, a link counter of the item-owner schedule); if it stands still for stall_ns of wall time
// (globaltimer), or another warp has already given up, the waiter raises the abort flag and leaves.
struct StallWatch {
    unsigned long long t_last = 0, prog_last = 0;
    __device__ __forceinline__ bool stalled(const unsigned long long *progress, int *abort_flag, unsigned long long stall_ns) {
        if (*(volatile int *)abort_flag) return true;
        const unsigned long long now = mf_globaltimer();
        const unsigned long long pr = *(volatile const unsigned long long *)progress;
        if (t_last == 0 || pr != prog_last) {
            t_last = now;
            prog_last = pr;
            return false;
        }
        if (now - t_last > stall_ns) {
            atomicExch(abort_flag, 1);
            return true;
        }
        return false;
    }
};

__global__ void __launch_bounds__(128) k_mf_dataflow(MfArgs a) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned long long total = (unsigned long long)a.n * (unsigned long long)a.epochs;
    const int D = a.D;
    const daisy_mf_params prm = a.prm;
    while (true) {
        unsigned long long tk = 0;
        if (lane == 0) tk = atomicAdd(a.ticket, 1ULL);
        tk = __shfl_sync(FULL, tk, 0);
        if (tk >= total) break;
        const int e = (int)(tk / (unsigned long long)a.n);
        const long long t = (long long)(tk % (unsigned long long)a.n);
        const int u = a.users[t], i = a.items[t];
        const double r = a.ratings[t];
        const unsigned want_u = (unsigned)e * (unsigned)a.cnt_u[u] + (unsigned)a.need_u[t];
        const unsigned want_i = (unsigned)e * (unsigned)a.cnt_i[i] + (unsigned)a.need_i[t];
        int bail = 0;
        if (lane == 0) {
            unsigned spins = 0;
            StallWatch watch;
            while (ld_acquire_u32(&a.ver_u[u]) != want_u || ld_acquire_u32(&a.ver_i[i]) != want_i) {
                __nanosleep(32);
                if ((++spins & 0xfffu) == 0 && watch.stalled(a.ticket, a.abort_flag, a.stall_ns)) {
                    bail = 1;
                    break;
                }
            }
        }
        bail = __shfl_sync(FULL, bail, 0);
        if (bail) break;
        // Every lane acquires the two versions itself (satisfied at once: lane 0 has just seen them).  A shuffle is
        // not a memory barrier -- without this the compiler may hoist the bias / row loads above the wait.
        if (ld_acquire_u32(&a.ver_u[u]) != want_u || ld_acquire_u32(&a.ver_i[i]) != want_i) {
            atomicExch(a.abort_flag, 2);  // cannot happen: versions only advance through this warp
        }
        __syncwarp();
        double *p = a.pu + (size_t)u * D;
        double *q = a.qi + (size_t)i * D;
        // rows live in L2 (ld.cg): other SMs wrote them
        double dot = 0.0;
        for (int f = lane; f < D; f += 32) dot += __ldcg(q + f) * __ldcg(p + f);
        dot = warp_sum_d(dot);
        double err;
        // the two biases are read by lane 0 alone and broadcast: one load each, taken strictly before lane 0's
        // stores below whatever the intra-warp schedule is
        double b0 = 0.0, b1 = 0.0;
        if (lane == 0) {
            b0 = __ldcg(a.bu + u);
            b1 = __ldcg(a.bi + i);
        }
        b0 = __shfl_sync(FULL, b0, 0);
        b1 = __shfl_sync(FULL, b1, 0);
        if (prm.variant == 0) {  // SVD, util/matrix_factorization.pyx:140-151
            const double b_u = b0, b_i = b1;
            err = r - (prm.global_mean + b_u + b_i + dot);
            if (prm.biased && lane == 0) {
                __stcg(a.bu + u, b_u + prm.lr_bu * (err - prm.reg_bu * b_u));
                __stcg(a.bi + i, b_i + prm.lr_bi * (err - prm.reg_bi * b_i));
            }
        } else {  // RSVD, :49-61
            const double c_i = b0, d_j = b1;
            err = r - (c_i + d_j + dot);
            if (prm.variant == 2 && lane == 0) {
                const double inc = prm.lr_bu * (err - prm.reg2 * (c_i + d_j - prm.global_mean));
                __stcg(a.bu + u, c_i + inc);
                __stcg(a.bi + i, d_j + inc);
            }
        }
        for (int f = lane; f < D; f += 32) {
            const double puf = __ldcg(p + f), qif = __ldcg(q + f);
            __stcg(p + f, puf + prm.lr_pu * (err * qif - prm.reg_pu * puf));
            __stcg(q + f, qif + prm.lr_qi * (err * puf - prm.reg_qi * qif));
        }
        if (a.err2 && lane == 0) a.err2[(size_t)e * a.n + t] = err * err;
        __threadfence();
        __syncwarp();
        if (lane == 0) {
            st_release_u32(&a.ver_u[u], want_u + 1);
            st_release_u32(&a.ver_i[i], want_i + 1);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Item-owner schedule (default).  The ticket schedule above pays a full L2 hand-off (poll, acquire, row loads,
// stores, fence, release: ~10 us measured) for EVERY link of the longest dependency chain -- and with a Zipf
// catalogue the hottest item's chain is ~12 % of all ratings.  Here every item belongs to one warp for the whole
// fit: item of hotness rank r -> warp r mod W (W = resident warps), so the hottest W items have a warp of their
// own.  A warp walks the ratings of its items in sequence order, epoch after epoch, and keeps the current item's
// row and bias IN REGISTERS from one rating to the next: an item chain link costs a dot product and an update,
// no memory round trip.  Only user rows travel through memory, guarded by the per-user version counters exactly
// as above (expected version = e * #ratings(u) + rank of the rating among u's ratings); the next link's user row
// is loaded speculatively behind an acquire load of its version while the current link computes.
// Deadlock-free: the earliest unprocessed rating of the whole sequence has its user predecessor done (it is
// earlier) and its item predecessor done (same warp, earlier in that warp's list), so its owner can proceed;
// all W warps are resident (persistent launch sized by the occupancy query).
// Same arithmetic as the reference loop: the result is the sequential result up to the rounding of the warp-tree
// dot product, identical to the ticket schedule's.
// ------------------------------------------------------------------------------------------------
struct OwnArgs {
    double *pu, *qi, *bu, *bi;
    const int *lk_u, *lk_i;        // per link: links are grouped by owner warp, in sequence order inside a warp
    const double *lk_r;
    const unsigned *lk_need, *lk_cnt, *lk_t;  // rank among the user's ratings, #ratings of the user, position t
    const unsigned *wptr;          // [W + 1] first link of every warp
    unsigned *ver_u;
    double *err2;
    int *abort_flag;
    unsigned long long *stats;  // optional (DAISY_MF_STATS=1): [0] links, [1] links that took the blocking path, [2] item switches
    unsigned long long *progress;  // links done by all warps (bumped once per group): what the stall detector watches
    long long n;
    int epochs, D;
    daisy_mf_params prm;
    unsigned long long stall_ns;
    int batch;                     // DAISY_MF_BATCH (default 1): batched groups (k_mf_owner)
};

// back-off between two polls of a version in k_mf_owner (200 and 1 000 ns were measured no different, DESIGN.md section 6)
constexpr unsigned MF_OWNER_POLL_NS = 20;

__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(unsigned *p, unsigned v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// Links are processed in GROUPS of K.  A memory fence costs a warp ~0.4 us whatever it covers, so a group shares ONE:
// after the K links of group g are done (their user rows stored, K version updates pending), lanes j < K read the
// versions of group g+1's users (relaxed), every lane executes one fence.acq_rel -- it orders this warp's row stores
// before the K pending version stores (release pattern) and the version reads before the row reads that follow
// (acquire pattern) -- then the pending versions are published and the K user rows of group g+1 are loaded for the
// links whose version was already the expected one.  A link whose user row is not ready yet (its previous rating is
// held by another warp, or by an earlier link of the same group) takes the blocking path; pending versions are
// always published BEFORE blocking, so no warp ever waits on a version that its owner is holding back.
template <int DV>
__global__ void __launch_bounds__(128) k_mf_owner(OwnArgs a) {
    constexpr int K = DV <= 4 ? 8 : (DV == 8 ? 4 : 2);
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const unsigned w = (unsigned)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const unsigned beg = a.wptr[w], end = a.wptr[w + 1];
    if (beg == end) return;  // warp-uniform
    const unsigned len = end - beg;
    const unsigned long long L = (unsigned long long)len * (unsigned long long)a.epochs;  // links of this warp, all epochs
    const int D = a.D;
    const daisy_mf_params prm = a.prm;
    bool act[DV];
#pragma unroll
    for (int v = 0; v < DV; ++v) act[v] = (lane + 32 * v) < D;

    double q[DV];
#pragma unroll
    for (int v = 0; v < DV; ++v) q[v] = 0.0;
    double b_i = 0.0;
    int cur_item = -1;

    // metadata of the current group (M0) and the next one (M1): lane j < K holds link x0 + j
    int u0 = -1, i0 = 0, u1 = -1, i1 = 0;
    double r0 = 0.0, r1 = 0.0;
    unsigned want0 = 0, want1 = 0, t0 = 0, t1 = 0, e0 = 0, e1 = 0;
    // (epoch, offset) of the link x the next load_meta call starts at; advanced by K per call (no 64-bit divisions)
    unsigned meta_e = 0, meta_off = 0;
    // The expected version of a link is e * (#ratings of its user) + (rank among them).  The two factors are kept as
    // loaded (cnt1, need1) and only combined where want1 is first needed, a whole group later: an in-order warp stalls
    // at the first USE of a load, and combining them here exposed one global round trip per group (~1000 cycles
    // of the hottest warp's ~10 000 per group, DAISY_MF_STATS).
    unsigned cnt1 = 0, need1 = 0;
    auto load_meta = [&](unsigned long long x, int &mu, int &mi, double &mr, unsigned &mc, unsigned &mn, unsigned &mt, unsigned &me) {
        mu = -1;
        unsigned e = meta_e, off = meta_off + (unsigned)lane;
        while (off >= len) { off -= len; ++e; }
        meta_off += K;
        while (meta_off >= len) { meta_off -= len; ++meta_e; }
        if (lane < K && x + lane < L) {
            const unsigned k = beg + off;
            mu = a.lk_u[k];
            mi = a.lk_i[k];
            mr = a.lk_r[k];
            mc = a.lk_cnt[k];
            mn = a.lk_need[k];
            mt = a.lk_t[k];
            me = e;
        }
    };
    load_meta(0, u0, i0, r0, cnt1, need1, t0, e0);
    want0 = e0 * cnt1 + need1;
    load_meta(K, u1, i1, r1, cnt1, need1, t1, e1);

    double R[K][DV], Bu[K];  // prefetched user rows / biases of the current group (valid where `valid` has the bit)
#pragma unroll
    for (int j = 0; j < K; ++j) {
        Bu[j] = 0.0;
#pragma unroll
        for (int v = 0; v < DV; ++v) R[j][v] = 0.0;
    }
    unsigned valid = 0;
    unsigned long long n_slow = 0, n_switch = 0, n_batch = 0;
    long long tm[6] = {0, 0, 0, 0, 0, 0};  // DAISY_MF_STATS: cycles of the hottest warp by segment (see daisy_mf_fit)
    const bool timed = a.stats != nullptr && w == 0;
    long long tc = timed ? clock64() : 0;
#define DAISY_MF_TICK(slot)                       \
    if (timed) {                                  \
        const long long now_ = clock64();         \
        tm[slot] += now_ - tc;                    \
        tc = now_;                                \
    }
    int pend_u = -1;         // lane j: user whose version update from link j of the current group is not published yet
    unsigned pend_v = 0;

    for (unsigned long long x0 = 0; x0 < L; x0 += K) {
        // ---- batched group (K == 8): see mf_batched_group below the loop body ------------------------------------
        bool batched = false;
        if (K == 8 && a.batch) {
            const int i_first = __shfl_sync(FULL, i0, 0);
            const unsigned same = __match_any_sync(FULL, lane < K ? u0 : -2 - lane);
            batched = __all_sync(FULL, lane >= K || (u0 >= 0 && i0 == i_first && same == (1u << lane)));
        }
        if (batched) {
            // A full group on ONE item with pairwise distinct users -- decided from the link list alone, never from
            // timing, so a fit takes the same arithmetic path on every run (bit-reproducible).  The K dot products
            // q_k . p_k form a chain through the item row: q_{k+1} = al q_k + be_k p_k, al = 1 - lr_qi reg_qi,
            // be_k = lr_qi err_k, so  q_k . p_k = al^k (q_0 . p_k) + sum_{l<k} al^(k-1-l) be_l (p_l . p_k).
            // The K + K(K-1)/2 = 36 vector dot products on the right do not depend on each other: they are formed
            // first (independent FMAs, ONE transposing reduction for 32 of them), and the chain shrinks to a scalar
            // recurrence (~k FMAs per link) -- instead of a 5-round warp reduction per link.  The row updates then
            // follow the reference's formulas element by element with those errors.
            ++n_batch;
            const int i = __shfl_sync(FULL, i0, 0);
            if (i != cur_item) {
                ++n_switch;
                if (cur_item >= 0) {
#pragma unroll
                    for (int v = 0; v < DV; ++v)
                        if (act[v]) __stcg(a.qi + (size_t)cur_item * D + lane + 32 * v, q[v]);
                    if (lane == 0) __stcg(a.bi + cur_item, b_i);
                }
#pragma unroll
                for (int v = 0; v < DV; ++v) q[v] = act[v] ? __ldcg(a.qi + (size_t)i * D + lane + 32 * v) : 0.0;
                b_i = __ldcg(a.bi + i);
                cur_item = i;
            }
            const double al = 1.0 - prm.lr_qi * prm.reg_qi;
            double a0 = 1.0, cf[8], bi_run = b_i;
            // one link of the scalar recurrence: dot = a0 * dk + sum_l cf[l] * g(l, k) has been formed by the caller
#define DAISY_MF_SCALAR_STEP(k, dot, err_out, nbu_out)                                                       \
            {                                                                                                \
                const double r_ = __shfl_sync(FULL, r0, (k));                                                \
                const double bu_ = Bu[(k)];                                                                  \
                double err_, nbu_ = bu_, nbi_ = bi_run;                                                      \
                if (prm.variant == 0) {                                                                      \
                    err_ = r_ - (prm.global_mean + bu_ + bi_run + (dot));                                    \
                    if (prm.biased) {                                                                        \
                        nbu_ = bu_ + prm.lr_bu * (err_ - prm.reg_bu * bu_);                                  \
                        nbi_ = bi_run + prm.lr_bi * (err_ - prm.reg_bi * bi_run);                            \
                    }                                                                                        \
                } else {                                                                                     \
                    err_ = r_ - (bu_ + bi_run + (dot));                                                      \
                    if (prm.variant == 2) {                                                                  \
                        const double inc_ = prm.lr_bu * (err_ - prm.reg2 * (bu_ + bi_run - prm.global_mean)); \
                        nbu_ = bu_ + inc_;                                                                   \
                        nbi_ = bi_run + inc_;                                                                \
                    }                                                                                        \
                }                                                                                            \
                (err_out) = err_;                                                                            \
                (nbu_out) = nbu_;                                                                            \
                bi_run = nbi_;                                                                               \
                _Pragma("unroll") for (int l_ = 0; l_ < (k); ++l_) cf[l_] *= al;                             \
                cf[(k)] = prm.lr_qi * err_;                                                                  \
                a0 *= al;                                                                                    \
            }
            // the row update of link k with its error: the reference's formulas, element by element
#define DAISY_MF_ROW_UPDATE(k, err, nbu_k)                                                                   \
            {                                                                                                \
                const int u_ = __shfl_sync(FULL, u0, (k));                                                   \
                _Pragma("unroll") for (int v = 0; v < DV; ++v)                                               \
                    if (act[v]) {                                                                            \
                        const double puf = R[(k)][v], qif = q[v];                                            \
                        __stcg(a.pu + (size_t)u_ * D + lane + 32 * v, puf + prm.lr_pu * ((err) * qif - prm.reg_pu * puf)); \
                        q[v] = qif + prm.lr_qi * ((err) * puf - prm.reg_qi * qif);                           \
                    }                                                                                        \
                if (lane == 0 && (nbu_k) != Bu[(k)]) __stcg(a.bu + u_, (nbu_k));                             \
                if (a.err2) {                                                                                \
                    const unsigned t_ = __shfl_sync(FULL, t0, (k)), e_ = __shfl_sync(FULL, e0, (k));         \
                    if (lane == 0) a.err2[(size_t)e_ * a.n + t_] = (err) * (err);                            \
                }                                                                                            \
            }
            if (valid == (1u << K) - 1u) {
                // ---- every row of the group was ready when it was prefetched: all dot products at once ------------
                // (1) per-lane partial sums of the 36 dot products: s[0..7] = q . p_j, then p_l . p_j for l < j
                double sa[32], sb[4];
                {
                    int idx = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        double t = 0.0;
#pragma unroll
                        for (int v = 0; v < DV; ++v) t = fma(q[v], R[j][v], t);   // inactive slices hold zeros
                        sa[idx++] = t;
                    }
#pragma unroll
                    for (int l = 0; l < 8; ++l)
#pragma unroll
                        for (int j = l + 1; j < 8; ++j) {
                            double t = 0.0;
#pragma unroll
                            for (int v = 0; v < DV; ++v) t = fma(R[l][v], R[j][v], t);
                            if (idx < 32) sa[idx] = t; else sb[idx - 32] = t;
                            ++idx;
                        }
                }
                // (2) transposing reduction: after the five rounds lane L holds the warp total of value L in sa[0].  Every
                // total is formed by the same additions as warp_sum_d's butterfly (offsets 16, 8, 4, 2, 1), which is
                // what the one-link-at-a-time variant below uses: the two variants agree bit for bit.
#define DAISY_RS_ROUND(H)                                                            \
                {                                                                    \
                    const bool up = (lane & (H)) != 0;                               \
                    _Pragma("unroll") for (int ii = 0; ii < (H); ++ii) {             \
                        const double send = up ? sa[ii] : sa[ii + (H)];              \
                        const double keep = up ? sa[ii + (H)] : sa[ii];              \
                        sa[ii] = keep + __shfl_xor_sync(FULL, send, (H));            \
                    }                                                                \
                }
                DAISY_RS_ROUND(16) DAISY_RS_ROUND(8) DAISY_RS_ROUND(4) DAISY_RS_ROUND(2) DAISY_RS_ROUND(1)
#undef DAISY_RS_ROUND
                const double tot = sa[0];
#pragma unroll
                for (int x = 0; x < 4; ++x) sb[x] = warp_sum_d(sb[x]);
                DAISY_MF_TICK(0)
                // value index of p_l . p_j (l < j) in the order they were formed
#define DAISY_GIDX(l, j) (8 + (l) * 7 - ((l) * ((l) - 1)) / 2 + ((j) - (l) - 1))
                // (3) the scalar recurrence, computed redundantly by every lane
                double errs[8], nbu[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    double dot = a0 * __shfl_sync(FULL, tot, k);
#pragma unroll
                    for (int l = 0; l < k; ++l) {
                        const int gi = DAISY_GIDX(l, k);
                        const double g = gi < 32 ? __shfl_sync(FULL, tot, gi & 31) : sb[(gi - 32) & 3];
                        dot = fma(cf[l], g, dot);
                    }
                    DAISY_MF_SCALAR_STEP(k, dot, errs[k], nbu[k])
                }
#undef DAISY_GIDX
                DAISY_MF_TICK(1)
                // (4) the row updates in the reference's order
#pragma unroll
                for (int k = 0; k < 8; ++k) DAISY_MF_ROW_UPDATE(k, errs[k], nbu[k])
                DAISY_MF_TICK(2)
                if (lane < K) {  // version updates of the group: published with the group's fence below
                    pend_u = u0;
                    pend_v = want0 + 1;
                }
            } else {
                // ---- some rows were not ready: one link at a time, SAME arithmetic (dot products against the group's
                // initial item row q_0 and the earlier rows of the group, each reduced by warp_sum_d), so the result does
                // not depend on which variant ran.  Before blocking on a row, everything this warp holds back is
                // published -- an earlier link of the group may be what the row's producer is waiting for.
                double q_0[DV];
#pragma unroll
                for (int v = 0; v < DV; ++v) q_0[v] = q[v];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (!(valid & (1u << k))) {  // warp-uniform
                        ++n_slow;
                        const int u = __shfl_sync(FULL, u0, k);
                        const unsigned want = __shfl_sync(FULL, want0, k);
                        fence_acq_rel_gpu();
                        __syncwarp();
                        if (pend_u >= 0) st_relaxed_u32(&a.ver_u[pend_u], pend_v);
                        pend_u = -1;
                        int bail = 0;
                        if (lane == 0) {
                            unsigned spins = 0;
                            StallWatch watch;
                            while (ld_acquire_u32(&a.ver_u[u]) != want) {
                                __nanosleep(MF_OWNER_POLL_NS);
                                if ((++spins & 0xfffu) == 0 && watch.stalled(a.progress, a.abort_flag, a.stall_ns)) {
                                    bail = 1;
                                    break;
                                }
                            }
                        }
                        bail = __shfl_sync(FULL, bail, 0);
                        if (bail) return;
                        if (ld_acquire_u32(&a.ver_u[u]) != want) atomicExch(a.abort_flag, 2);
#pragma unroll
                        for (int v = 0; v < DV; ++v) R[k][v] = act[v] ? __ldcg(a.pu + (size_t)u * D + lane + 32 * v) : 0.0;
                        Bu[k] = __ldcg(a.bu + u);
                    }
                    double t = 0.0;
#pragma unroll
                    for (int v = 0; v < DV; ++v) t = fma(q_0[v], R[k][v], t);
                    double dot = a0 * warp_sum_d(t);
#pragma unroll
                    for (int l = 0; l < k; ++l) {
                        double g = 0.0;
#pragma unroll
                        for (int v = 0; v < DV; ++v) g = fma(R[l][v], R[k][v], g);
                        dot = fma(cf[l], warp_sum_d(g), dot);
                    }
                    double err_k, nbu_k;
                    DAISY_MF_SCALAR_STEP(k, dot, err_k, nbu_k)
                    DAISY_MF_ROW_UPDATE(k, err_k, nbu_k)
                    if (lane == k) {
                        pend_u = u0;
                        pend_v = want0 + 1;
                    }
                }
            }
#undef DAISY_MF_SCALAR_STEP
#undef DAISY_MF_ROW_UPDATE
            b_i = bi_run;
        } else
#pragma unroll
        for (int j = 0; j < K; ++j) {
            const int u = __shfl_sync(FULL, u0, j);
            if (u < 0) break;  // warp-uniform: past the end of the list
            const int i = __shfl_sync(FULL, i0, j);
            const double r = __shfl_sync(FULL, r0, j);
            const unsigned want = __shfl_sync(FULL, want0, j);
            if (i != cur_item) {  // another item of this warp: park the current row, fetch the other
                ++n_switch;
                if (cur_item >= 0) {
#pragma unroll
                    for (int v = 0; v < DV; ++v)
                        if (act[v]) __stcg(a.qi + (size_t)cur_item * D + lane + 32 * v, q[v]);
                    if (lane == 0) __stcg(a.bi + cur_item, b_i);
                }
#pragma unroll
                for (int v = 0; v < DV; ++v) q[v] = act[v] ? __ldcg(a.qi + (size_t)i * D + lane + 32 * v) : 0.0;
                b_i = __ldcg(a.bi + i);
                cur_item = i;
            }
            double p[DV], b_u;
            if (valid & (1u << j)) {
#pragma unroll
                for (int v = 0; v < DV; ++v) p[v] = R[j][v];
                b_u = Bu[j];
            } else {
                ++n_slow;
                // blocking path.  Publish what this warp holds back first (another warp may be waiting for it, and
                // the version we are about to wait for may even be one of ours).
                fence_acq_rel_gpu();
                __syncwarp();
                if (pend_u >= 0) st_relaxed_u32(&a.ver_u[pend_u], pend_v);
                pend_u = -1;
                int bail = 0;
                if (lane == 0) {
                    unsigned spins = 0;
                    StallWatch watch;
                    while (ld_acquire_u32(&a.ver_u[u]) != want) {
                        __nanosleep(MF_OWNER_POLL_NS);
                        if ((++spins & 0xfffu) == 0 && watch.stalled(a.progress, a.abort_flag, a.stall_ns)) {
                            bail = 1;
                            break;
                        }
                    }
                }
                bail = __shfl_sync(FULL, bail, 0);
                if (bail) return;
                if (ld_acquire_u32(&a.ver_u[u]) != want) atomicExch(a.abort_flag, 2);  // every lane acquires itself
#pragma unroll
                for (int v = 0; v < DV; ++v) p[v] = act[v] ? __ldcg(a.pu + (size_t)u * D + lane + 32 * v) : 0.0;
                b_u = __ldcg(a.bu + u);
            }
            double dot = 0.0;
#pragma unroll
            for (int v = 0; v < DV; ++v)
                if (act[v]) dot += q[v] * p[v];
            dot = warp_sum_d(dot);
            double err;
            double nb_u = b_u, nb_i = b_i;
            if (prm.variant == 0) {  // SVD, util/matrix_factorization.pyx:140-151
                err = r - (prm.global_mean + b_u + b_i + dot);
                if (prm.biased) {
                    nb_u = b_u + prm.lr_bu * (err - prm.reg_bu * b_u);
                    nb_i = b_i + prm.lr_bi * (err - prm.reg_bi * b_i);
                }
            } else {  // RSVD, :49-61
                err = r - (b_u + b_i + dot);
                if (prm.variant == 2) {
                    const double inc = prm.lr_bu * (err - prm.reg2 * (b_u + b_i - prm.global_mean));
                    nb_u = b_u + inc;
                    nb_i = b_i + inc;
                }
            }
            b_i = nb_i;
#pragma unroll
            for (int v = 0; v < DV; ++v)
                if (act[v]) {
                    const double puf = p[v], qif = q[v];
                    __stcg(a.pu + (size_t)u * D + lane + 32 * v, puf + prm.lr_pu * (err * qif - prm.reg_pu * puf));
                    q[v] = qif + prm.lr_qi * (err * puf - prm.reg_qi * qif);
                }
            if (lane == 0) {
                if (nb_u != b_u) __stcg(a.bu + u, nb_u);
            }
            if (a.err2) {
                const unsigned t = __shfl_sync(FULL, t0, j), e = __shfl_sync(FULL, e0, j);
                if (lane == 0) a.err2[(size_t)e * a.n + t] = err * err;
            }
            if (lane == j) {  // version update of this link: published with the group's fence
                pend_u = u;
                pend_v = want + 1;
            }
        }
        // ---- one fence for the group: publish its versions, pick up the next group's user rows ----------------
        DAISY_MF_TICK(5)   // (everything of the group that is not one of the batched segments)
        unsigned vnext = 0;
        if (u1 >= 0) vnext = ld_relaxed_u32(&a.ver_u[u1]);
        fence_acq_rel_gpu();
        __syncwarp();
        if (pend_u >= 0) st_relaxed_u32(&a.ver_u[pend_u], pend_v);
        pend_u = -1;
        if (lane == 0) atomicAdd(a.progress, (unsigned long long)K);  // fire and forget: the stall detector's clock
        want1 = e1 * cnt1 + need1;
        valid = __ballot_sync(FULL, u1 >= 0 && vnext == want1);
        DAISY_MF_TICK(3)
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (valid & (1u << j)) {  // warp-uniform
                const int un = __shfl_sync(FULL, u1, j);
#pragma unroll
                for (int v = 0; v < DV; ++v) R[j][v] = act[v] ? __ldcg(a.pu + (size_t)un * D + lane + 32 * v) : 0.0;
                Bu[j] = __ldcg(a.bu + un);
            }
        }
        u0 = u1; i0 = i1; r0 = r1; want0 = want1; t0 = t1; e0 = e1;
        load_meta(x0 + 2 * K, u1, i1, r1, cnt1, need1, t1, e1);
        DAISY_MF_TICK(4)
    }
    // (the loop's last iteration published every pending version)
    if (a.stats && lane == 0) {
        atomicAdd(&a.stats[0], L);
        atomicAdd(&a.stats[1], n_slow);
        atomicAdd(&a.stats[2], n_switch);
        atomicAdd(&a.stats[6], n_batch);
        if (w == 0) {
            a.stats[7] = n_batch;
            for (int x = 0; x < 6; ++x) a.stats[8 + x] = (unsigned long long)tm[x];  // the hottest item's warp
            a.stats[3] = L;
            a.stats[4] = n_slow;
            a.stats[5] = n_switch;
        }
    }
    if (cur_item >= 0) {
#pragma unroll
        for (int v = 0; v < DV; ++v)
            if (act[v]) __stcg(a.qi + (size_t)cur_item * D + lane + 32 * v, q[v]);
        if (lane == 0) __stcg(a.bi + cur_item, b_i);
    }
}

__global__ void k_mf_hot_keys(const int *__restrict__ cnt_i, unsigned I, uint32_t *key, uint32_t *val) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= I) return;
    key[i] = 0xFFFFFFFFu - (uint32_t)cnt_i[i];  // ascending sort = hottest first
    val[i] = i;
}
__global__ void k_mf_hot_rank(const uint32_t *__restrict__ val_s, unsigned I, uint32_t *rank) {
    unsigned p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < I) rank[val_s[p]] = p;
}
__global__ void k_mf_owner_keys(const int32_t *__restrict__ items, long long n, const uint32_t *__restrict__ rank,
                                unsigned W, uint32_t *key, uint32_t *val) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= n) return;
    key[t] = rank[items[t]] % W;
    val[t] = (uint32_t)t;
}
__global__ void k_mf_links(const uint32_t *__restrict__ order, long long n, const int32_t *__restrict__ users,
                           const int32_t *__restrict__ items, const double *__restrict__ ratings,
                           const int *__restrict__ need_u, const int *__restrict__ cnt_u, int *lk_u, int *lk_i,
                           double *lk_r, unsigned *lk_need, unsigned *lk_cnt, unsigned *lk_t) {
    long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t t = order[p];
    const int u = users[t];
    lk_u[p] = u;
    lk_i[p] = items[t];
    lk_r[p] = ratings[t];
    lk_need[p] = (unsigned)need_u[t];
    lk_cnt[p] = (unsigned)cnt_u[u];
    lk_t[p] = t;
}
__global__ void k_mf_wptr(const uint32_t *__restrict__ okey_s, long long n, unsigned W, unsigned *wptr) {
    unsigned w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w > W) return;
    long long lo = 0, hi = n;  // first position with key >= w
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (okey_s[mid] < w) lo = mid + 1; else hi = mid;
    }
    wptr[w] = (unsigned)lo;
}

// ---- rank of each rating among the ratings of its row, and per-row counts ------------------------
__global__ void k_mf_keys(const int32_t *__restrict__ ids, long long n, unsigned rows, uint32_t *key, uint32_t *val,
                          int *err) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= n) return;
    uint32_t r = (uint32_t)ids[t];
    if (r >= rows) {
        atomicOr(&err[0], 1);
        atomicMin(&err[1], (int)t);
        r = 0;
    }
    key[t] = r;
    val[t] = (uint32_t)t;
}
__global__ void k_mf_starts(const uint32_t *__restrict__ key_s, long long n, int *start) {
    long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (p >= n) return;
    start[p] = (p == 0 || key_s[p - 1] != key_s[p]) ? (int)p : 0;
}
__global__ void k_mf_need(const uint32_t *__restrict__ key_s, const uint32_t *__restrict__ val_s,
                          const int *__restrict__ seg_start, long long n, int *need, int *cnt) {
    long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int rank = (int)p - seg_start[p];
    need[val_s[p]] = rank;
    if (p == n - 1 || key_s[p + 1] != key_s[p]) cnt[key_s[p]] = rank + 1;
}
__global__ void k_mf_sse(const double *__restrict__ err2, long long n, int epochs, double *sse_out) {
    __shared__ double sh[32];
    const int e = blockIdx.x;
    double s = 0.0;
    for (long long t = threadIdx.x; t < n; t += blockDim.x) s += err2[(size_t)e * n + t];
    s = warp_sum_d(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
        v = warp_sum_d(v);
        if (threadIdx.x == 0) sse_out[e] = v;
    }
}
__global__ void k_mf_predict(const double *__restrict__ pu, const double *__restrict__ qi, const double *__restrict__ bu,
                             const double *__restrict__ bi, const int32_t *__restrict__ users,
                             const int32_t *__restrict__ items, long long n, unsigned U, unsigned I, int D, int with_bias,
                             double mu, double *__restrict__ est, int *err) {
    const int lane = threadIdx.x & 31;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long t = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; t < n; t += nw) {
        unsigned u = (unsigned)users[t], i = (unsigned)items[t];
        if (u >= U || i >= I) {
            if (lane == 0) {
                atomicOr(&err[0], u >= U ? 2 : 4);  // 2: invalid user code, 4: invalid item code
                atomicMin(&err[1], (int)t);
            }
            u = u < U ? u : 0;
            i = i < I ? i : 0;
        }
        double dot = 0.0;
        for (int f = lane; f < D; f += 32) dot += qi[(size_t)i * D + f] * pu[(size_t)u * D + f];
        dot = warp_sum_d(dot);
        if (lane == 0) est[t] = with_bias ? mu + bu[u] + bi[i] + dot : dot;
    }
}

// Stream-ordered scratch (the handle's private pool, kept cached between fits): ~45 buffers per fit cost
// microseconds instead of the ~100 ms of as many cudaMalloc / cudaFree pairs.  Freed on scope exit.
struct Scratch {
    void *p[64];
    int n = 0;
    cudaStream_t s;
    daisy_ctx *h;
    explicit Scratch(cudaStream_t stream, daisy_ctx *ctx) : s(stream), h(ctx) {}
    template <class T>
    int get(T **out, size_t count) {
        *out = nullptr;
        cudaError_t e = daisy_scratch_alloc(h, (void **)out, (count ? count : 1) * sizeof(T), s);
        if (e != cudaSuccess) {
            daisy_set_error("cudaMallocAsync of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
            return DAISY_ENOMEM;
        }
        p[n++] = *out;
        return DAISY_OK;
    }
    ~Scratch() {
        for (int i = 0; i < n; ++i) cudaFreeAsync(p[i], s);
    }
};

int rank_in_row(daisy_ctx *h, const int32_t *ids, long long n, unsigned rows, uint32_t *key, uint32_t *key_s, uint32_t *val,
                uint32_t *val_s, int *start, int *start_scan, void *tmp, size_t tmp_bytes, int *need, int *cnt,
                cudaStream_t s) {
    const int T = 256;
    const int G = daisy_ceil_div(n, T);
    k_mf_keys<<<G, T, 0, s>>>(ids, n, rows, key, val, h->err);
    DAISY_LAUNCH_CHECK(h);
    int bits = 1;
    while (bits < 32 && ((uint64_t)(rows - 1) >> bits)) ++bits;
    size_t tb = tmp_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, key, key_s, val, val_s, (int)n, 0, bits, s));
    k_mf_starts<<<G, T, 0, s>>>(key_s, n, start);
    DAISY_LAUNCH_CHECK(h);
    tb = tmp_bytes;
    DAISY_CUDA(cub::DeviceScan::InclusiveScan(tmp, tb, start, start_scan, cub::Max(), (int)n, s));
    k_mf_need<<<G, T, 0, s>>>(key_s, val_s, start_scan, n, need, cnt);
    DAISY_LAUNCH_CHECK(h);
    h->launches += 8;
    return DAISY_OK;
}

}  // namespace

extern "C" int daisy_mf_fit(daisy_handle_t h, double *pu, double *qi, double *bu, double *bi, const int32_t *users,
                            const int32_t *items, const double *ratings, int64_t n, int n_epochs,
                            const daisy_mf_params *prm, double *sse_out, daisy_stream_t stream) {
    DAISY_REQUIRE(h && pu && qi && bu && bi && prm, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(n >= 0 && n < (1LL << 30), DAISY_EINVAL, "bad rating count");
    DAISY_REQUIRE(n_epochs >= 0, DAISY_EINVAL, "bad epoch count");
    DAISY_REQUIRE(prm->variant >= 0 && prm->variant <= 2, DAISY_EINVAL, "variant must be 0 (SVD), 1 (RSVD1) or 2 (RSVD2)");
    DAISY_REQUIRE((double)n * (double)n_epochs < 4.0e9, DAISY_EUNSUPPORTED, "n * n_epochs must stay below 2^32 row versions");
    if (n == 0 || n_epochs == 0) return DAISY_OK;
    DAISY_REQUIRE(users && items && ratings, DAISY_EINVAL, "null rating arrays");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)n;
    Scratch ws(s, h);
    uint32_t *key, *key_s, *val, *val_s;
    int *start, *start_scan, *need_u, *need_i, *cnt_u, *cnt_i, *abort_flag;
    unsigned *ver_u, *ver_i;
    unsigned long long *ticket;
    double *err2 = nullptr;
    void *tmp;
    int rc = DAISY_OK;
#define G_(x, c) if (!rc) rc = ws.get(&x, (c))
    G_(key, N); G_(key_s, N); G_(val, N); G_(val_s, N); G_(start, N); G_(start_scan, N);
    G_(need_u, N); G_(need_i, N); G_(cnt_u, (size_t)h->U); G_(cnt_i, (size_t)h->I);
    G_(ver_u, (size_t)h->U); G_(ver_i, (size_t)h->I); G_(ticket, 1); G_(abort_flag, 1);
    if (sse_out) G_(err2, N * (size_t)n_epochs);
#undef G_
    if (rc) return rc;
    size_t tb_sort = 0, tb_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, key, key_s, val, val_s, (int)n, 0, 32, s);
    cub::DeviceScan::InclusiveScan(nullptr, tb_scan, start, start_scan, cub::Max(), (int)n, s);
    const size_t tmp_bytes = (tb_sort > tb_scan ? tb_sort : tb_scan) + 256;
    char *tmpc;
    rc = ws.get(&tmpc, tmp_bytes);
    if (rc) return rc;
    tmp = tmpc;
    DAISY_CUDA(cudaMemsetAsync(cnt_u, 0, (size_t)h->U * sizeof(int), s));
    DAISY_CUDA(cudaMemsetAsync(cnt_i, 0, (size_t)h->I * sizeof(int), s));
    DAISY_CUDA(cudaMemsetAsync(ver_u, 0, (size_t)h->U * sizeof(unsigned), s));
    DAISY_CUDA(cudaMemsetAsync(ver_i, 0, (size_t)h->I * sizeof(unsigned), s));
    DAISY_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), s));
    DAISY_CUDA(cudaMemsetAsync(abort_flag, 0, sizeof(int), s));
    rc = rank_in_row(h, users, n, (unsigned)h->U, key, key_s, val, val_s, start, start_scan, tmp, tmp_bytes, need_u, cnt_u, s);
    if (rc) return rc;
    rc = rank_in_row(h, items, n, (unsigned)h->I, key, key_s, val, val_s, start, start_scan, tmp, tmp_bytes, need_i, cnt_i, s);
    if (rc) return rc;
    // ids out of range were parked on row 0 by k_mf_keys but the dataflow kernel indexes with the raw ids:
    // stop here and let daisy_check report it
    DAISY_CUDA(cudaMemcpyAsync(h->err_host, h->err, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
    DAISY_CUDA(cudaStreamSynchronize(s));
    if (h->err_host[0]) {
        daisy_set_error("Invalid user or item code at rating %d", h->err_host[1]);
        return DAISY_EINDEX;
    }
    unsigned long long *dbg_stats = nullptr;
    const char *sched = getenv("DAISY_MF_SCHEDULE");
    bool owner = !(sched && strcmp(sched, "ticket") == 0) && h->D <= 512;
    // Copies of the four arrays as they came in: a fit that aborts (stall detector) hands the tables back untouched
    // instead of partially trained.  Funk-SVD tables are small (config 2: 10 MB).
    double *bk_pu, *bk_qi, *bk_bu, *bk_bi;
    const size_t n_pu = (size_t)h->U * h->D, n_qi = (size_t)h->I * h->D;
    rc = ws.get(&bk_pu, n_pu);
    if (!rc) rc = ws.get(&bk_qi, n_qi);
    if (!rc) rc = ws.get(&bk_bu, (size_t)h->U);
    if (!rc) rc = ws.get(&bk_bi, (size_t)h->I);
    if (rc) return rc;
    DAISY_CUDA(cudaMemcpyAsync(bk_pu, pu, n_pu * sizeof(double), cudaMemcpyDeviceToDevice, s));
    DAISY_CUDA(cudaMemcpyAsync(bk_qi, qi, n_qi * sizeof(double), cudaMemcpyDeviceToDevice, s));
    DAISY_CUDA(cudaMemcpyAsync(bk_bu, bu, (size_t)h->U * sizeof(double), cudaMemcpyDeviceToDevice, s));
    DAISY_CUDA(cudaMemcpyAsync(bk_bi, bi, (size_t)h->I * sizeof(double), cudaMemcpyDeviceToDevice, s));
    const char *stall_env = getenv("DAISY_MF_STALL_MS");
    const unsigned long long stall_ns = (unsigned long long)((stall_env && atof(stall_env) > 0 ? atof(stall_env) : 10000.0) * 1e6);
    if (owner) {
        int occ = 0;
        const int DVsel = h->D <= 32 ? 1 : h->D <= 64 ? 2 : h->D <= 128 ? 4 : h->D <= 256 ? 8 : 16;
#define OCC_(DVV) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_mf_owner<DVV>, 128, 0)
        DAISY_CUDA(DVsel == 1 ? OCC_(1) : DVsel == 2 ? OCC_(2) : DVsel == 4 ? OCC_(4) : DVsel == 8 ? OCC_(8) : OCC_(16));
#undef OCC_
        if (occ < 1) occ = 1;
        const int per_sm = occ < 8 ? occ : 8;
        const unsigned W = (unsigned)(h->num_sms * per_sm * 4);
        uint32_t *hkey, *hkey_s, *hval, *hval_s, *rank;
        int *lk_u, *lk_i;
        double *lk_r;
        unsigned *lk_need, *lk_cnt, *lk_t, *wptr;
        const size_t I = (size_t)h->I;
        rc = DAISY_OK;
#define G2_(x, c) if (!rc) rc = ws.get(&x, (c))
        G2_(hkey, I); G2_(hkey_s, I); G2_(hval, I); G2_(hval_s, I); G2_(rank, I);
        G2_(lk_u, N); G2_(lk_i, N); G2_(lk_r, N); G2_(lk_need, N); G2_(lk_cnt, N); G2_(lk_t, N); G2_(wptr, (size_t)W + 1);
#undef G2_
        if (rc) return rc;
        const int T = 256;
        k_mf_hot_keys<<<daisy_ceil_div((int64_t)I, T), T, 0, s>>>(cnt_i, (unsigned)I, hkey, hval);
        DAISY_LAUNCH_CHECK(h);
        size_t tb = tmp_bytes;
        if (I > (size_t)n) {  // the shared CUB scratch was sized for n pairs
            size_t need = 0;
            cub::DeviceRadixSort::SortPairs(nullptr, need, hkey, hkey_s, hval, hval_s, (int)I, 0, 32, s);
            DAISY_REQUIRE(need <= tmp_bytes, DAISY_EUNSUPPORTED, "item table much larger than the rating list");
        }
        DAISY_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, hkey, hkey_s, hval, hval_s, (int)I, 0, 32, s));
        k_mf_hot_rank<<<daisy_ceil_div((int64_t)I, T), T, 0, s>>>(hval_s, (unsigned)I, rank);
        DAISY_LAUNCH_CHECK(h);
        k_mf_owner_keys<<<daisy_ceil_div(n, T), T, 0, s>>>(items, n, rank, W, key, val);
        DAISY_LAUNCH_CHECK(h);
        int wbits = 1;
        while (wbits < 32 && ((uint64_t)(W - 1) >> wbits)) ++wbits;
        tb = tmp_bytes;
        DAISY_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, key, key_s, val, val_s, (int)n, 0, wbits, s));
        k_mf_links<<<daisy_ceil_div(n, T), T, 0, s>>>(val_s, n, users, items, ratings, need_u, cnt_u, lk_u, lk_i, lk_r,
                                                      lk_need, lk_cnt, lk_t);
        DAISY_LAUNCH_CHECK(h);
        k_mf_wptr<<<daisy_ceil_div((int64_t)W + 1, T), T, 0, s>>>(key_s, n, W, wptr);
        DAISY_LAUNCH_CHECK(h);
        h->launches += 8;
        OwnArgs o;
        o.pu = pu; o.qi = qi; o.bu = bu; o.bi = bi;
        o.lk_u = lk_u; o.lk_i = lk_i; o.lk_r = lk_r; o.lk_need = lk_need; o.lk_cnt = lk_cnt; o.lk_t = lk_t;
        o.wptr = wptr; o.ver_u = ver_u; o.err2 = err2; o.abort_flag = abort_flag;
        o.n = n; o.epochs = n_epochs; o.D = h->D; o.prm = *prm;
        o.stall_ns = stall_ns;
        const char *be = getenv("DAISY_MF_BATCH");
        o.batch = (be && *be) ? (atoi(be) != 0) : 1;
        o.progress = ticket;   // the ticket word is free under this schedule
        o.stats = nullptr;
        const char *st_env = getenv("DAISY_MF_STATS");
        if (st_env && atoi(st_env) > 0) {
            rc = ws.get(&o.stats, 16);
            if (rc) return rc;
            DAISY_CUDA(cudaMemsetAsync(o.stats, 0, 16 * sizeof(unsigned long long), s));
            dbg_stats = o.stats;
        }
        // The schedule is deadlock-free only if all W warps are resident at once (a resident warp may wait for a
        // version owned by any other warp): a COOPERATIVE launch either gets the whole grid co-resident -- whatever
        // else is running on the device -- or fails, in which case the fit falls back to the ticket schedule, whose
        // earliest unprocessed rating is always held by a resident warp.
        const int grid = h->num_sms * per_sm;
        void *kargs[] = {(void *)&o};
        const void *fn = DVsel == 1 ? (const void *)k_mf_owner<1> : DVsel == 2 ? (const void *)k_mf_owner<2>
                       : DVsel == 4 ? (const void *)k_mf_owner<4> : DVsel == 8 ? (const void *)k_mf_owner<8>
                                                                                  : (const void *)k_mf_owner<16>;
        cudaError_t le = cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(128), kargs, 0, s);
        if (le != cudaSuccess) {
            (void)cudaGetLastError();
            owner = false;
        } else {
            h->launches += 1;
        }
    }
    if (!owner) {
        MfArgs a;
        a.pu = pu; a.qi = qi; a.bu = bu; a.bi = bi;
        a.users = users; a.items = items; a.ratings = ratings;
        a.need_u = need_u; a.need_i = need_i; a.cnt_u = cnt_u; a.cnt_i = cnt_i;
        a.ver_u = ver_u; a.ver_i = ver_i; a.ticket = ticket; a.err2 = err2; a.abort_flag = abort_flag;
        a.n = n; a.epochs = n_epochs; a.D = h->D; a.prm = *prm;
        a.stall_ns = stall_ns;
        int occ = 0;
        DAISY_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_mf_dataflow, 128, 0));
        if (occ < 1) occ = 1;
        const int per_sm = occ < 8 ? occ : 8;
        k_mf_dataflow<<<h->num_sms * per_sm, 128, 0, s>>>(a);
        DAISY_LAUNCH_CHECK(h);
    }
    if (sse_out) {
        k_mf_sse<<<n_epochs, 256, 0, s>>>(err2, n, n_epochs, sse_out);
        DAISY_LAUNCH_CHECK(h);
    }
    int aborted = 0;
    DAISY_CUDA(cudaMemcpyAsync(&aborted, abort_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    DAISY_CUDA(cudaStreamSynchronize(s));
    if (dbg_stats) {
        unsigned long long hs[16];
        DAISY_CUDA(cudaMemcpy(hs, dbg_stats, sizeof(hs), cudaMemcpyDeviceToHost));
        fprintf(stderr, "[daisy_mf_fit] hottest warp, cycles: batched dots + reduction %llu, recurrence %llu, row updates %llu | "
                        "version reads + fence + publish %llu, row prefetch issue + next metadata %llu, rest of the groups %llu\n",
                hs[8], hs[9], hs[10], hs[11], hs[12], hs[13]);
        fprintf(stderr, "[daisy_mf_fit] links %llu blocking %llu item-switches %llu batched groups %llu | hottest warp: links %llu "
                        "blocking %llu switches %llu batched groups %llu\n",
                hs[0], hs[1], hs[2], hs[6], hs[3], hs[4], hs[5], hs[7]);
    }
    if (aborted) {  // hand the tables back as they came in
        DAISY_CUDA(cudaMemcpyAsync(pu, bk_pu, n_pu * sizeof(double), cudaMemcpyDeviceToDevice, s));
        DAISY_CUDA(cudaMemcpyAsync(qi, bk_qi, n_qi * sizeof(double), cudaMemcpyDeviceToDevice, s));
        DAISY_CUDA(cudaMemcpyAsync(bu, bk_bu, (size_t)h->U * sizeof(double), cudaMemcpyDeviceToDevice, s));
        DAISY_CUDA(cudaMemcpyAsync(bi, bk_bi, (size_t)h->I * sizeof(double), cudaMemcpyDeviceToDevice, s));
        DAISY_CUDA(cudaStreamSynchronize(s));
    }
    DAISY_REQUIRE(!aborted, DAISY_ECUDA, "daisy_mf_fit: schedule stalled (no rating processed for %.0f ms) -- the tables "
                  "were restored to their state before the call", (double)stall_ns * 1e-6);
    return DAISY_OK;
}

extern "C" int daisy_mf_predict(daisy_handle_t h, const double *pu, const double *qi, const double *bu, const double *bi,
                                const int32_t *users, const int32_t *items, int64_t n, int with_bias, double mu,
                                double *est, daisy_stream_t stream) {
    DAISY_REQUIRE(h && pu && qi, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(!with_bias || (bu && bi), DAISY_EINVAL, "bias arrays required when with_bias");
    DAISY_REQUIRE(n >= 0, DAISY_EINVAL, "bad count");
    if (n == 0) return DAISY_OK;
    DAISY_REQUIRE(users && items && est, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    long long blocks = (n + 7) / 8;
    const long long cap = (long long)h->num_sms * 16;
    if (blocks > cap) blocks = cap;
    k_mf_predict<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(pu, qi, bu, bi, users, items, n, (unsigned)h->U,
                                                              (unsigned)h->I, h->D, with_bias, mu, est, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}
