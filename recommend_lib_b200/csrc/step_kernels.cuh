// Shared pipeline of the fused BPR step (kernels + host orchestration), included by bpr_step.cu (single GPU:
// SGD / lazy sparse Adam) and shard.cu (row-sharded tables).  The optimiser / destination of a finished row sum is a
// functor `Opt` with
//     apply(int tbl, size_t row, int e, float4 old, float4 d)
// tbl 0 = user table, 1 = item table; e = float4 index inside the row; old = the row slice as read before the step;
// d = the complete descent direction (-gradient sum) of that slice.  `Opt::kNeedOldItem` tells the reduce kernels
// whether `old` of an item row has to be loaded at all.
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "ctx.cuh"
#include "ref_sort.cuh"

namespace {
// ------------------------------------------------------------------------------------------------
// prep: validate, emit sort keys
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_triple(const int32_t *__restrict__ triples, int t, uint32_t U, uint32_t I,
                                            uint32_t &u, uint32_t &i, uint32_t &j, bool &bad) {
    u = (uint32_t)triples[3 * (size_t)t];
    i = (uint32_t)triples[3 * (size_t)t + 1];
    j = (uint32_t)triples[3 * (size_t)t + 2];
    bad = (u >= U) | (i >= I) | (j >= I);
    if (bad) {  // never fault: park the triple on row 0, the error flag tells the caller
        u = u < U ? u : 0u;
        i = i < I ? i : 0u;
        j = j < I ? j : 0u;
    }
}

__global__ void k_prep(const int32_t *__restrict__ triples, int B, uint32_t U, uint32_t I, uint32_t *__restrict__ key,
                       uint32_t *__restrict__ val, int *err) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B) return;
    uint32_t u, i, j;
    bool bad;
    load_triple(triples, t, U, I, u, i, j, bad);
    if (bad) {
        atomicOr(&err[0], 1);
        atomicMin(&err[1], t);
    }
    key[t] = i;
    val[t] = (uint32_t)t;
}

// ------------------------------------------------------------------------------------------------
// refs: sorted triples + reference lists
// ------------------------------------------------------------------------------------------------
__global__ void k_refs(const int32_t *__restrict__ triples, const uint32_t *__restrict__ order,
                       const uint32_t *__restrict__ sorted_i, int B, uint32_t U, uint32_t I, int C,
                       int32_t *__restrict__ st, uint32_t *__restrict__ ukey, uint32_t *__restrict__ uval,
                       uint32_t *__restrict__ qkey, uint32_t *__restrict__ qval, uint32_t *__restrict__ islot,
                       uint32_t ukey_off, uint32_t *__restrict__ longs_hdr, uint32_t *seen, uint32_t *dup) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0 && longs_hdr) longs_hdr[0] = longs_hdr[1] = 0u;  // merged sort: the list is filled by k_slots_dup
    if (k >= B) return;
    uint32_t u, i, j;
    bool bad;
    load_triple(triples, (int)order[k], U, I, u, i, j, bad);
    st[3 * (size_t)k] = (int32_t)u;
    st[3 * (size_t)k + 1] = (int32_t)i;
    st[3 * (size_t)k + 2] = (int32_t)j;
    ukey[k] = u + ukey_off;  // merged sort (book_kernels): user keys follow the item keys and the sentinel
    qkey[k] = j;  // negative-item ref of sorted triple k
    const bool head = (k % C == 0) || (sorted_i[k - 1] != i);
    qkey[B + k] = head ? i : I;  // I = sentinel, sorts after every real row
    if (qval) {  // the merged sort's values are the ref positions themselves
        uval[k] = (uint32_t)k;
        qval[k] = (uint32_t)k;
        qval[B + k] = (uint32_t)(B + k);
    }
    if (!head) islot[k] = DAISY_NOT_HEAD;  // heads get their slot from k_slots_item
    if (seen) {  // merged sort: which rows are referenced more than once (item rows, then user rows from bit I)
        mark_row(seen, dup, I + u);
        mark_row(seen, dup, j);
        if (head) mark_row(seen, dup, i);
    }
}

// ------------------------------------------------------------------------------------------------
// slots: DIRECT (single contribution in the batch) or staging slot = sorted position
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void list_long_row(const uint32_t *__restrict__ keys, int n, int p, uint32_t row, int tbl,
                                              int long_len, int slice, uint32_t *longs, int longs_cap);

__global__ void k_slots_user(const uint32_t *__restrict__ key, const uint32_t *__restrict__ val, int n,
                             uint32_t *__restrict__ uslot, uint32_t *longs, int longs_cap, int long_len) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t r = key[p];
    const bool first = (p == 0) || (key[p - 1] != r);
    const bool last = (p == n - 1) || (key[p + 1] != r);
    uslot[val[p]] = (first && last) ? DAISY_DIRECT : (uint32_t)p;
    if (first && longs) list_long_row(key, n, p, r, 0, long_len, DAISY_SLICE, longs, longs_cap);
}

__global__ void k_slots_item(const uint32_t *__restrict__ key, const uint32_t *__restrict__ val, int n, int B,
                             uint32_t sentinel, uint32_t *__restrict__ jslot, uint32_t *__restrict__ islot,
                             uint32_t *longs, int longs_cap, int long_len) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t r = key[p];
    if (r == sentinel) return;
    const bool first = (p == 0) || (key[p - 1] != r);
    const bool last = (p == n - 1) || (key[p + 1] != r);
    const uint32_t slot = (first && last) ? DAISY_DIRECT : (uint32_t)p;
    const uint32_t v = val[p];
    if (v < (uint32_t)B)
        jslot[v] = slot;
    else
        islot[v - B] = slot;
    if (first && longs) list_long_row(key, n, p, r, 1, long_len, DAISY_SLICE, longs, longs_cap);
}

// Merged sort (book_kernels): ref x of the 3B refs k_refs wrote -- negatives [0, B), run heads [B, 2B) (key I: not a
// head), users [2B, 3B) (key I + 1 + u) -- goes into the sort only if its row has another ref in the same table.  A ref
// whose row has none is DIRECT, and is settled here.
struct BprRefSrc {
    const uint32_t *key, *dup;
    int B;
    uint32_t I;
    uint32_t *jslot, *islot, *uslot;
    __device__ __forceinline__ bool operator()(int x, uint32_t &k) const {
        const uint32_t r = key[x];
        if (r == I) return false;
        const uint32_t bit = r < I ? r : r - 1u;
        if (dup[bit >> 5] >> (bit & 31) & 1u) {
            k = r;
            return true;
        }
        if (x < B)
            jslot[x] = DAISY_DIRECT;
        else if (x < 2 * B)
            islot[x - B] = DAISY_DIRECT;
        else
            uslot[x - 2 * B] = DAISY_DIRECT;
        return false;
    }
};

// The sorted refs of repeated rows: ss->n of them, the ss->n_lo item refs first (keys < I), then the user refs (keys
// I + 1 + u), each row's refs in their order among the 3B.  Every one of them shares its row, so it is staged at its
// position in its table's part.  Splits the keys into the set's qkey_s / ukey_s (user keys back to row ids), which is
// what the table kernels read, lists the rows longer than long_len and records both counts for k_seg_all.
__global__ void k_slots_dup(const uint32_t *__restrict__ key, const uint32_t *__restrict__ val, const DsortState *ss, int B,
                            uint32_t I, uint32_t *__restrict__ qkey_s, uint32_t *__restrict__ ukey_s,
                            uint32_t *__restrict__ uslot, uint32_t *__restrict__ jslot, uint32_t *__restrict__ islot,
                            uint32_t *__restrict__ counts, uint32_t *longs, int longs_cap, int long_len) {
    const int n = (int)ss->n, nq = (int)ss->n_lo, nu = n - nq;
    const int p0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (p0 == 0) {
        counts[0] = (uint32_t)nu;
        counts[1] = (uint32_t)nq;
    }
    for (int p = p0; p < n; p += gridDim.x * blockDim.x) {
        const uint32_t r = key[p], v = val[p];
        if (p < nq) {
            qkey_s[p] = r;
            if (v < (uint32_t)B)
                jslot[v] = (uint32_t)p;
            else
                islot[v - B] = (uint32_t)p;
            if (p == 0 || key[p - 1] != r) list_long_row(key, nq, p, r, 1, long_len, DAISY_SLICE, longs, longs_cap);
        } else {
            const int q = p - nq;
            const uint32_t *ukey = key + nq;
            ukey_s[q] = r - (I + 1u);
            uslot[v - 2u * (uint32_t)B] = (uint32_t)q;
            if ((q == 0 || ukey[q - 1] != r) && q + long_len < nu && ukey[q + long_len] == r) {
                // a long user row: the list holds row ids, so search the run in the offset keys and record the row
                int lo = q + long_len, hi = nu - 1;
                while (lo < hi) {
                    const int mid = (int)(((long long)lo + hi + 1) >> 1);
                    if (ukey[mid] == r) lo = mid; else hi = mid - 1;
                }
                const uint32_t len = (uint32_t)(lo - q + 1);
                const uint32_t rr = atomicAdd(&longs[0], 1u);
                const uint32_t sl0 = atomicAdd(&longs[1], (len + DAISY_SLICE - 1) / DAISY_SLICE);
                if ((int)rr < longs_cap) {
                    uint32_t *rec = longs + 2 + 5 * (size_t)rr;
                    rec[0] = 0u;
                    rec[1] = r - (I + 1u);
                    rec[2] = (uint32_t)q;
                    rec[3] = len;
                    rec[4] = sl0;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// main fused kernel
// ------------------------------------------------------------------------------------------------
struct MainArgs {
    const float *P;
    const float *Q;
    const int32_t *st;
    const uint32_t *uslot, *jslot, *islot;
    float *stageU, *stageQ;
    float *loss_part;
    int B, D4, C;
    float c2;  // score scale = c^2
    // PTR mode (row-sharded step): where to read the item rows of sorted triple k from -- the owner's memory (peer
    // or local address) for rows referenced once, the fetched-row cache otherwise.  st then holds cache rows.
    const float *const *jsrc, *const *isrc;
    // PTR mode: the chunks (sorted by positive item = grouped by OWNER) are dealt to the warps round-robin over `ilv`
    // equal ranges of the sorted order, so that at any moment a rank's loads and stores are spread over all owners
    // instead of every rank walking the owners 0, 1, 2, ... at the same time (incast on one owner's links).
    // 0 / 1 = sorted order.  Scheduling only: which warp takes which chunk never changes a result.
    int ilv;
};

// warp -> chunk in PTR mode (see MainArgs::ilv); -1 = no chunk for this warp
__host__ __device__ __forceinline__ int interleaved_chunk(int raw, int nchunks, int ilv) {
    if (ilv <= 1) return raw < nchunks ? raw : -1;
    const int per = (nchunks + ilv - 1) / ilv;
    const int q = raw / ilv, r = raw - q * ilv;
    if (q >= per) return -1;
    const int c = r * per + q;
    return c < nchunks ? c : -1;
}

template <int V, class Opt, bool PTR>
__global__ void __launch_bounds__(256) k_bpr_main(MainArgs a, Opt opt) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    int warp = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int C = a.C;
    if (PTR) {
        warp = interleaved_chunk(warp, (a.B + C - 1) / C, a.ilv);
        if (warp < 0) return;
    }
    const long long k0 = (long long)warp * C;  // (k0 + lane fits size_t below: k0 < B)
    if (k0 >= a.B) return;  // warp-uniform
    const int n = (int)min((long long)C, (long long)a.B - k0);
    const int D4 = a.D4;

    // chunk metadata: lane l holds sorted triple k0 + l (C <= 32)
    int mu = 0, mi = 0, mj = 0;
    uint32_t mus = 0, mjs = 0, mis = 0;
    if (lane < n) {
        const size_t k = (size_t)(k0 + lane);
        mu = a.st[3 * k];
        mi = a.st[3 * k + 1];
        mj = a.st[3 * k + 2];
        mus = a.uslot[k];
        mjs = a.jslot[k];
        mis = a.islot[k];  // DAISY_NOT_HEAD unless this triple starts a positive-item run
    }
    const float *pj = nullptr, *pi = nullptr;
    if (PTR && lane < n) {
        pj = a.jsrc[k0 + lane];
        if (mis != DAISY_NOT_HEAD) pi = a.isrc[k0 + lane];
    }
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;

    float4 pu[V], qj[V], qi[V], acc[V], pu_n[V], qj_n[V], qi_n[V];
#pragma unroll
    for (int v = 0; v < V; ++v) pu[v] = qj[v] = qi[v] = acc[v] = pu_n[v] = qj_n[v] = qi_n[v] = f4_zero();
    {
        const int u = __shfl_sync(FULL, mu, 0), i = __shfl_sync(FULL, mi, 0), j = __shfl_sync(FULL, mj, 0);
        const float *rj = PTR ? shfl_ptr(pj, 0) : a.Q + (size_t)j * (4 * D4);
        const float *ri = PTR ? shfl_ptr(pi, 0) : a.Q + (size_t)i * (4 * D4);
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                pu_n[v] = ld_row(a.P, (size_t)u * D4 + lane + 32 * v);
                qj_n[v] = ld_row(rj, lane + 32 * v);
                qi_n[v] = ld_row(ri, lane + 32 * v);
            }
    }
    int cur_i = -1;
    uint32_t cur_is = 0;
    float loss = 0.f;

    for (int t = 0; t < n; ++t) {
        const int u = __shfl_sync(FULL, mu, t), i = __shfl_sync(FULL, mi, t), j = __shfl_sync(FULL, mj, t);
        const uint32_t us = __shfl_sync(FULL, mus, t), js = __shfl_sync(FULL, mjs, t);
        const uint32_t is_t = __shfl_sync(FULL, mis, t);
        if (is_t != DAISY_NOT_HEAD) {  // a new positive-item run starts here (warp-uniform; t == 0 is always a head)
            if (t > 0) {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v]) {
                        const int e = lane + 32 * v;
                        if (cur_is == DAISY_DIRECT)
                            opt.apply(1, (size_t)cur_i, e, qi[v], acc[v]);
                        else
                            st_stream(a.stageQ, (size_t)cur_is * D4 + e, acc[v]);
                    }
            }
            cur_i = i;
            cur_is = is_t;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                qi[v] = qi_n[v];
                acc[v] = f4_zero();
            }
        }
#pragma unroll
        for (int v = 0; v < V; ++v) {
            pu[v] = pu_n[v];
            qj[v] = qj_n[v];
        }
        // prefetch the rows of sorted triple t+1 before touching triple t.  Safe: a row that is written in
        // place below is referenced exactly once in the whole batch, so no later triple reads it.
        if (t + 1 < n) {
            const int un = __shfl_sync(FULL, mu, t + 1), in = __shfl_sync(FULL, mi, t + 1),
                      jn = __shfl_sync(FULL, mj, t + 1);
            const bool head_n = __shfl_sync(FULL, mis, t + 1) != DAISY_NOT_HEAD;
            const float *rj = PTR ? shfl_ptr(pj, t + 1) : a.Q + (size_t)jn * (4 * D4);
            const float *ri = PTR ? shfl_ptr(pi, t + 1) : a.Q + (size_t)in * (4 * D4);
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v]) {
                    pu_n[v] = ld_row(a.P, (size_t)un * D4 + lane + 32 * v);
                    qj_n[v] = ld_row(rj, lane + 32 * v);
                    if (head_n) qi_n[v] = ld_row(ri, lane + 32 * v);
                }
        }
        // x = c^2 <P[u], Q[i] - Q[j]>;  s = sigmoid(-x) = -d(loss)/dx
        float d = 0.f;
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) d += f4_dot(pu[v], f4_sub(qi[v], qj[v]));
        d = warp_sum(d);
        const float x = d * a.c2;
        const float s = 1.f / (1.f + expf(x));
        loss += fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));  // -log sigmoid(x), overflow-safe
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                const int e = lane + 32 * v;
                // user row: descent direction +s (Q[i] - Q[j])
                const float4 gu = f4_scale(f4_sub(qi[v], qj[v]), s);
                if (us == DAISY_DIRECT)
                    opt.apply(0, (size_t)u, e, pu[v], gu);
                else
                    st_stream(a.stageU, (size_t)us * D4 + e, gu);
                // negative item row: descent direction -s P[u]
                const float4 gj = f4_scale(pu[v], -s);
                if (js == DAISY_DIRECT)
                    opt.apply(1, (size_t)j, e, qj[v], gj);
                else
                    st_stream(a.stageQ, (size_t)js * D4 + e, gj);
                // positive item row: +s P[u], accumulated over the run in sorted order
                acc[v].x = fmaf(s, pu[v].x, acc[v].x);
                acc[v].y = fmaf(s, pu[v].y, acc[v].y);
                acc[v].z = fmaf(s, pu[v].z, acc[v].z);
                acc[v].w = fmaf(s, pu[v].w, acc[v].w);
            }
    }
#pragma unroll
    for (int v = 0; v < V; ++v)
        if (act[v]) {
            const int e = lane + 32 * v;
            if (cur_is == DAISY_DIRECT)
                opt.apply(1, (size_t)cur_i, e, qi[v], acc[v]);
            else
                st_stream(a.stageQ, (size_t)cur_is * D4 + e, acc[v]);
        }
    if (lane == 0) a.loss_part[warp] = loss;
}

// ------------------------------------------------------------------------------------------------
// main fused kernel, TMA-pipelined: the same arithmetic in the same order as k_bpr_main (bit-identical results), but
// the rows of the next S sorted triples of a warp are in flight at once.  Every warp owns a ring of S stages in
// shared memory (3 rows each); one elected lane issues one bulk async copy per row (cp.async.bulk global ->
// shared, completion on the stage's mbarrier), the warp waits on the stage's phase, reads its float4 slices
// (conflict-free 16-byte-per-lane shared loads) and immediately refills the stage with triple t + S.
// With register prefetching one triple ahead, a warp's next loads are only issued once the previous ones have
// landed, which makes the sharded step latency-bound on peer loads (~2-3 us over NVLink); here the depth is S
// triples per warp and the loads cost no registers.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

template <int V, class Opt, bool PTR>
__global__ void __launch_bounds__(256) k_bpr_main_tma(MainArgs a, Opt opt, int S) {
    extern __shared__ __align__(128) unsigned char dsm[];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int warp = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int C = a.C;
    if (PTR) {
        warp = interleaved_chunk(warp, (a.B + C - 1) / C, a.ilv);
        if (warp < 0) return;
    }
    const long long k0 = (long long)warp * C;
    if (k0 >= a.B) return;  // warp-uniform; no block-wide barrier is used below
    const int n = (int)min((long long)C, (long long)a.B - k0);
    const int D4 = a.D4;
    const uint32_t rowB = (uint32_t)D4 * 16u;
    // ring of this warp: S stages x 3 rows; the mbarriers of all warps sit behind the rings
    unsigned char *ring = dsm + (size_t)wid * S * 3 * rowB;
    const uint32_t ring_s = smem_u32(ring);
    const uint32_t bars = smem_u32(dsm + (size_t)8 * S * 3 * rowB) + (uint32_t)(wid * S) * 8u;
    if (lane == 0) {
        for (int st = 0; st < S; ++st) mbar_init(bars + 8u * st, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    int mu = 0, mi = 0, mj = 0;
    uint32_t mus = 0, mjs = 0, mis = 0;
    const float *pj = nullptr, *pi = nullptr;
    if (lane < n) {
        const size_t k = (size_t)(k0 + lane);
        mu = a.st[3 * k];
        mi = a.st[3 * k + 1];
        mj = a.st[3 * k + 2];
        mus = a.uslot[k];
        mjs = a.jslot[k];
        mis = a.islot[k];
        if (PTR) {
            pj = a.jsrc[k];
            if (mis != DAISY_NOT_HEAD) pi = a.isrc[k];
        }
    }
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;

    // issue the copies of sorted triple t into stage t % S (warp-uniform arguments; lane 0 elected)
    auto issue = [&](int t) {
        const int u = __shfl_sync(FULL, mu, t), i = __shfl_sync(FULL, mi, t), j = __shfl_sync(FULL, mj, t);
        const bool head = __shfl_sync(FULL, mis, t) != DAISY_NOT_HEAD;
        const float *rj = PTR ? shfl_ptr(pj, t) : a.Q + (size_t)j * (4 * D4);
        const float *ri = PTR ? shfl_ptr(pi, t) : a.Q + (size_t)i * (4 * D4);
        if (lane == 0) {
            const int stg = t % S;
            const uint32_t bar = bars + 8u * stg, dst = ring_s + (uint32_t)stg * 3u * rowB;
            mbar_expect_tx(bar, head ? 3u * rowB : 2u * rowB);
            bulk_g2s(dst, a.P + (size_t)u * (4 * D4), rowB, bar);
            bulk_g2s(dst + rowB, rj, rowB, bar);
            if (head) bulk_g2s(dst + 2u * rowB, ri, rowB, bar);
        }
    };
    for (int t = 0; t < S && t < n; ++t) issue(t);

    float4 pu[V], qj[V], qi[V], acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) pu[v] = qj[v] = qi[v] = acc[v] = f4_zero();
    int cur_i = -1;
    uint32_t cur_is = 0;
    float loss = 0.f;

    for (int t = 0; t < n; ++t) {
        const int u = __shfl_sync(FULL, mu, t), i = __shfl_sync(FULL, mi, t), j = __shfl_sync(FULL, mj, t);
        const uint32_t us = __shfl_sync(FULL, mus, t), js = __shfl_sync(FULL, mjs, t);
        const uint32_t is_t = __shfl_sync(FULL, mis, t);
        const bool head = is_t != DAISY_NOT_HEAD;
        if (head && t > 0) {  // flush the finished positive-item run
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v]) {
                    const int e = lane + 32 * v;
                    if (cur_is == DAISY_DIRECT)
                        opt.apply(1, (size_t)cur_i, e, qi[v], acc[v]);
                    else
                        st_stream(a.stageQ, (size_t)cur_is * D4 + e, acc[v]);
                }
        }
        const int stg = t % S;
        mbar_wait(bars + 8u * stg, (uint32_t)(t / S) & 1u);
        const float4 *sp = reinterpret_cast<const float4 *>(ring + (size_t)stg * 3 * rowB);
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                pu[v] = sp[lane + 32 * v];
                qj[v] = sp[D4 + lane + 32 * v];
                if (head) {
                    qi[v] = sp[2 * D4 + lane + 32 * v];
                    acc[v] = f4_zero();
                }
            }
        if (head) {
            cur_i = i;
            cur_is = is_t;
        }
        __syncwarp();                   // every lane has read the stage: it can be refilled
        if (t + S < n) issue(t + S);
        float d = 0.f;
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) d += f4_dot(pu[v], f4_sub(qi[v], qj[v]));
        d = warp_sum(d);
        const float x = d * a.c2;
        const float s = 1.f / (1.f + expf(x));
        loss += fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                const int e = lane + 32 * v;
                const float4 gu = f4_scale(f4_sub(qi[v], qj[v]), s);
                if (us == DAISY_DIRECT)
                    opt.apply(0, (size_t)u, e, pu[v], gu);
                else
                    st_stream(a.stageU, (size_t)us * D4 + e, gu);
                const float4 gj = f4_scale(pu[v], -s);
                if (js == DAISY_DIRECT)
                    opt.apply(1, (size_t)j, e, qj[v], gj);
                else
                    st_stream(a.stageQ, (size_t)js * D4 + e, gj);
                acc[v].x = fmaf(s, pu[v].x, acc[v].x);
                acc[v].y = fmaf(s, pu[v].y, acc[v].y);
                acc[v].z = fmaf(s, pu[v].z, acc[v].z);
                acc[v].w = fmaf(s, pu[v].w, acc[v].w);
            }
    }
#pragma unroll
    for (int v = 0; v < V; ++v)
        if (act[v]) {
            const int e = lane + 32 * v;
            if (cur_is == DAISY_DIRECT)
                opt.apply(1, (size_t)cur_i, e, qi[v], acc[v]);
            else
                st_stream(a.stageQ, (size_t)cur_is * D4 + e, acc[v]);
        }
    if (lane == 0) a.loss_part[warp] = loss;
}

// ------------------------------------------------------------------------------------------------
// segmented reduce + row update for rows with several contributions
// ------------------------------------------------------------------------------------------------
template <int V>
__device__ __forceinline__ void sum_staged(const float *__restrict__ stage, size_t q0, int len, int D4, int lane,
                                           const bool (&act)[V], float4 (&acc)[V]) {
    constexpr int UN = (V == 1) ? 8 : (V == 2 ? 4 : 2);
    for (int c = 0; c < len; c += UN) {
        float4 r[UN][V];
#pragma unroll
        for (int jj = 0; jj < UN; ++jj)
#pragma unroll
            for (int v = 0; v < V; ++v)
                r[jj][v] = (c + jj < len && act[v]) ? ld_stream(stage, (q0 + c + jj) * D4 + lane + 32 * v) : f4_zero();
#pragma unroll
        for (int jj = 0; jj < UN; ++jj)  // fixed order: sorted position ascending
            if (c + jj < len) {
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] = f4_add(acc[v], r[jj][v]);
            }
    }
}

// One warp, window w of WIN sorted refs: every multi-contribution row that STARTS in the window is summed and updated.
// The warp always looks at 32 refs from the window's first one; WIN < 32 only narrows which row starts it owns (the
// small-batch path has SMs to spare and uses 8: a warp walks its rows one after the other, each an L2 round trip).
template <int V, class Opt, int WIN = 32>
__device__ __forceinline__ void seg_window(long long w, int tbl, const float *__restrict__ table,
                                           const uint32_t *__restrict__ keys, int n, uint32_t sentinel,
                                           const float *__restrict__ stage, int D4, const Opt &opt, int heavy_len) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const long long base = w * WIN;
    if (base >= n) return;
    const long long p = base + lane;
    const uint32_t key = (p < n) ? keys[p] : sentinel;
    uint32_t prev = __shfl_up_sync(FULL, key, 1);
    if (lane == 0) prev = (p > 0) ? keys[p - 1] : ~key;
    uint32_t next = __shfl_down_sync(FULL, key, 1);
    if (lane == 31) next = (p + 1 < n) ? keys[p + 1] : sentinel;
    const bool valid = (p < n) && (key != sentinel);
    const bool start = valid && (prev != key);
    const bool multi = start && (next == key) && (p + 1 < n);
    const unsigned boundary = __ballot_sync(FULL, start || !valid);
    unsigned todo = __ballot_sync(FULL, multi && lane < WIN);
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;

    while (todo) {
        const int b = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t row = __shfl_sync(FULL, key, b);
        const unsigned after = (b == 31) ? 0u : (boundary & ~((2u << b) - 1u));
        int len;
        if (after) {
            len = (__ffs(after) - 1) - b;
        } else {  // the segment runs past this window: count matching keys in the following windows
            len = 32 - b;
            long long q = base + 32;
            while (true) {
                const bool ok = (q + lane < n) && (keys[q + lane] == row);
                const unsigned m = __ballot_sync(FULL, ok);
                const int c = (m == FULL) ? 32 : (__ffs(~m) - 1);
                len += c;
                if (c < 32 || len > heavy_len) break;
                q += 32;
            }
        }
        const size_t q0 = (size_t)(base + b);
        if (len > heavy_len) continue;  // a long row: the bookkeeping listed it, k_seg_all's slice blocks take it
        float4 old[V], acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) {
            old[v] = (act[v] && (tbl == 0 || Opt::kNeedOldItem)) ? ld_row(table, (size_t)row * D4 + lane + 32 * v) : f4_zero();
            acc[v] = f4_zero();
        }
        sum_staged<V>(stage, q0, len, D4, lane, act, acc);
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) opt.apply(tbl, (size_t)row, lane + 32 * v, old[v], acc[v]);
    }
}

// ------------------------------------------------------------------------------------------------
// Small-batch path (B <= DAISY_SMALL_CAP): the step is launch-bound, not bandwidth-bound (the 22 launches of the
// general pipeline cost ~80 us for 4 096 triples), so the whole bookkeeping is ONE kernel and the table phase two.
//
//   k_small_book   block 0 sorts the B user refs, block 1 the 2B item refs (negatives, then positives), each with a
//                  block-wide radix sort in shared memory.  A ref is one 32-bit word (row << vb | ref index), sorted
//                  on the row bits only; the ref index rides along, so there is no value array.  Rows referenced once
//                  are DIRECT, every other ref is staged at its sorted position -- the contract of the general path,
//                  without the positive-item runs (every triple heads its own run: C = 1).
//   k_bpr_main     the general main kernel with C = 1 (one warp per triple)
//   k_seg_all      segmented reduces of both tables + hot-row slices + loss in one launch (at most 16 384
//                  contributions exist) + the loss reduction
//
// The accumulation order of a row is its sorted-ref order, fixed by the sort => bit-reproducible.  It differs from
// the general path's order (which groups triples by positive item first), so the two paths agree to rounding only.
// ------------------------------------------------------------------------------------------------
// Block-wide stable LSD radix sort of up to 1024 * IPT 32-bit words on bits [lo, lo + nbits), digits of up to 9 bits
// ranked the way CUB's onesweep ranks them: a warp counts its digits by matching lanes (lanes holding the same digit
// find each other, the lowest one bumps the warp's histogram), one block scan over (digit, warp) turns the
// histograms into offsets.  Words live in registers in warp-striped order (word k < ipt of lane l of warp w is
// position w*32*ipt + k*32 + l; ipt <= IPT is block-uniform); the sorted words are left in `out` (shared memory).
// The whole block runs on ONE SM, 8 warps per scheduler, so the cost is the instruction count: ~70 per word and pass.
template <int IPT>
__device__ __forceinline__ void block_sort_words(uint32_t (&keys)[IPT], int ipt, int lo, int nbits,
                                                 uint32_t *hist /*[32 * 513]*/, uint32_t *out,
                                                 uint32_t *scan_tmp /*[33]*/) {
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    if (nbits < 1) nbits = 1;
    const int passes = (nbits + 8) / 9;
    int done = 0;
    for (int p = 0; p < passes; ++p) {
        int db = (nbits - done + (passes - p) - 1) / (passes - p);  // balanced digit widths, each <= 9
        if (db < 5) db = 5;                                          // >= 32 bins: one (digit, warp) cell per thread at least
        const int NB = 1 << db, shift = lo + done;
        const uint32_t dmask = (uint32_t)NB - 1u;
        const int HS = NB + 1;  // row stride: (digit, warp) cells of one scan step fall into 32 different banks
        uint32_t *wh = hist + (size_t)w * HS;
        for (int i = lane; i < NB; i += 32) wh[i] = 0;
        __syncwarp();
        uint32_t rank[IPT];
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            if (k < ipt) {
                const uint32_t d = (keys[k] >> shift) & dmask;
                // lanes holding the same digit, found with one ballot per digit bit (match.any serialises over the
                // distinct values of the warp: no faster here)
                unsigned m = FULL;
                for (int bb = 0; bb < db; ++bb) {
                    const bool bit = (d >> bb) & 1u;
                    const unsigned v = __ballot_sync(FULL, bit);
                    m &= bit ? v : ~v;
                }
                const int leader = __ffs(m) - 1;
                uint32_t base = 0;
                if (lane == leader) {
                    base = wh[d];
                    wh[d] = base + __popc(m);
                }
                base = __shfl_sync(FULL, base, leader);
                rank[k] = base + __popc(m & lt);
                __syncwarp();
            }
        }
        __syncthreads();
        // exclusive scan of the cells in (digit, warp) order: thread t owns E consecutive cells
        const int E = NB / 32;
        uint32_t sum = 0;
        for (int e = 0; e < E; ++e) {
            const int L = tid * E + e;
            sum += hist[(size_t)(L & 31) * HS + (L >> 5)];
        }
        uint32_t incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) scan_tmp[w] = incl;
        __syncthreads();
        if (w == 0) {
            const uint32_t tot = scan_tmp[lane];
            uint32_t inc2 = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(FULL, inc2, o);
                if (lane >= o) inc2 += v;
            }
            scan_tmp[lane] = inc2 - tot;
        }
        __syncthreads();
        uint32_t run = scan_tmp[w] + incl - sum;
        for (int e = 0; e < E; ++e) {
            const int L = tid * E + e;
            uint32_t *cell = hist + (size_t)(L & 31) * HS + (L >> 5);
            const uint32_t c = *cell;
            *cell = run;
            run += c;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < IPT; ++k)
            if (k < ipt) out[wh[(keys[k] >> shift) & dmask] + rank[k]] = keys[k];
        __syncthreads();
        if (p + 1 < passes) {
#pragma unroll
            for (int k = 0; k < IPT; ++k)
                if (k < ipt) keys[k] = out[w * 32 * ipt + k * 32 + lane];
        }
        done += db;
    }
}

#define DAISY_SMALL_HIST_WORDS (32 * 513)
#define DAISY_SEG_WIN_BLOCKS 8  // general path, merged sort: k_seg_all's window blocks per table and SM (they stride)
#define DAISY_SMALL_WIN 8       // sorted refs per warp of k_seg_all
#define DAISY_SMALL_SLICE 16   // contributions per slice of a long row (k_seg_all): short, so that a hot row's
                               // sum is spread over many warps on many SMs and is not a latency chain
#define DAISY_SMALL_CB 3        // k_small_book: rows are split over 2^CB blocks per table by their low CB bits
// Grid: 2 << CB blocks; block b < 2^CB handles the user refs whose row has low bits b, the others the item refs
// (negatives, then positives) likewise.  Only equal rows have to be adjacent in the "sorted" ref arrays, in a
// reproducible order -- not ascending rows -- so the arrays are ordered by (low row bits, high row bits, ref index)
// and every block can work alone: it reads ALL refs of its table (cheap), counts how many belong to lower classes
// (its base position) and compacts its own class into shared memory, then sorts that eighth on the high row bits.
// No block waits for another one, and the sort -- bound by the instruction throughput of one SM -- shrinks 8x.
template <int IPT>
__global__ void __launch_bounds__(1024) k_small_book(const int32_t *__restrict__ triples, int B, uint32_t U, uint32_t I,
                                                      int vbU, int kbU, int vbQ, int kbQ, int32_t *__restrict__ st,
                                                      uint32_t *__restrict__ ukey_s, uint32_t *__restrict__ qkey_s,
                                                      uint32_t *__restrict__ uslot, uint32_t *__restrict__ jslot,
                                                      uint32_t *__restrict__ islot, uint32_t *longs, int longs_cap,
                                                      int *err, int pairs) {
    // pairs != 0 (csrc/gmf.cu): the batch holds (user, item, label) samples -- ONE item ref per sample (column 1, filed
    // under jslot), column 2 is a label and is neither a row nor range-checked
    extern __shared__ __align__(16) unsigned char small_dsm[];
    uint32_t *hist = reinterpret_cast<uint32_t *>(small_dsm);
    uint32_t *sk = hist + DAISY_SMALL_HIST_WORDS;  // [1024 * IPT] compacted, then sorted words
    __shared__ uint32_t scan_tmp[33], wcnt[32], wlow[32];
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    constexpr uint32_t NC = 1u << DAISY_SMALL_CB;
    const bool items = blockIdx.x >= NC;
    const uint32_t cls = blockIdx.x & (NC - 1);
    const int n = items ? (pairs ? B : 2 * B) : B;
    const int vb = items ? vbQ : vbU, kb = items ? kbQ : kbU;
    const uint32_t bound = items ? I : U;
    uint32_t keys[IPT];
    // ---- every ref of the table: mine / lower class / neither ----
    const bool checker = !items && cls == 0;  // this block also validates the triples and writes the clamped copy
#pragma unroll
    for (int k = 0; k < IPT; ++k) {  // the loads first, all in flight together
        const int idx = w * 32 * IPT + k * 32 + lane;  // ref index; refs of a row keep this order
        uint32_t row = 0;
        if (idx < n) {
            const int t = idx < B ? idx : idx - B;
            if (checker) {
                uint32_t u, i, j;
                bool bad;
                load_triple(triples, t, U, pairs ? 0xFFFFFFFFu : I, u, i, j, bad);
                if (pairs && i >= I) {  // (the label column was let through by the unbounded check above)
                    bad = true;
                    i = 0;
                }
                st[3 * (size_t)t] = (int32_t)u;
                st[3 * (size_t)t + 1] = (int32_t)i;
                st[3 * (size_t)t + 2] = (int32_t)j;
                if (bad) {
                    atomicOr(&err[0], 1);
                    atomicMin(&err[1], t);
                }
                row = u;
            } else {
                row = (uint32_t)__ldg(triples + 3 * (size_t)t + (items ? ((idx < B && !pairs) ? 2 : 1) : 0));
            }
        }
        keys[k] = row;
    }
    uint32_t mine_cnt = 0, low_cnt = 0;
    unsigned mine_mask[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const int idx = w * 32 * IPT + k * 32 + lane;
        uint32_t row = keys[k];
        if (row >= bound) row = 0;  // parked on row 0 like load_triple does
        const uint32_t c = row & (NC - 1);
        const bool in = idx < n;
        keys[k] = in ? ((row << vb) | (uint32_t)idx) : 0xFFFFFFFFu;
        mine_mask[k] = __ballot_sync(FULL, in && c == cls);
        mine_cnt += __popc(mine_mask[k]);
        low_cnt += __popc(__ballot_sync(FULL, in && c < cls));
    }
    if (lane == 0) {
        wcnt[w] = mine_cnt;
        wlow[w] = low_cnt;
    }
    __syncthreads();
    uint32_t wbase, n_c, base_c;
    {
        const uint32_t c = wcnt[lane];
        uint32_t inc = c, lo = wlow[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lo += __shfl_xor_sync(FULL, lo, o);
        n_c = __shfl_sync(FULL, inc, 31);
        wbase = __shfl_sync(FULL, inc - c, w);
        base_c = lo;  // refs of lower classes come first in the table's sorted array
    }
    {
        uint32_t run = wbase;
#pragma unroll
        for (int k = 0; k < IPT; ++k) {
            if (mine_mask[k] >> lane & 1u) sk[run + __popc(mine_mask[k] & lt)] = keys[k];
            run += __popc(mine_mask[k]);
        }
    }
    __syncthreads();
    const int ipt = (int)((n_c + 1023u) / 1024u);
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t q = (uint32_t)(w * 32 * ipt + k * 32 + lane);
        keys[k] = (k < ipt && q < n_c) ? sk[q] : 0xFFFFFFFFu;  // padding behind the real refs; the sort is stable
    }
    __syncthreads();
    if (ipt > 0) block_sort_words<IPT>(keys, ipt, vb + DAISY_SMALL_CB, kb - DAISY_SMALL_CB, hist, sk, scan_tmp);
    const uint32_t vmask = (1u << vb) - 1u;
    uint32_t *key_out = (items ? qkey_s : ukey_s) + base_c;
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        const uint32_t p = (uint32_t)(k * 1024 + tid);
        if (p >= n_c) continue;
        const uint32_t wd = sk[p];
        const uint32_t row = wd >> vb, idx = wd & vmask;
        const bool first = (p == 0) || ((sk[p - 1] >> vb) != row);
        const bool last = (p == n_c - 1) || ((sk[p + 1] >> vb) != row);
        const uint32_t slot = (first && last) ? DAISY_DIRECT : base_c + p;
        key_out[p] = row;
        if (first && p + DAISY_SMALL_SLICE < n_c && (sk[p + DAISY_SMALL_SLICE] >> vb) == row) {
            // a row with more than DAISY_SMALL_SLICE contributions: too much for one warp (and for the L2 port of one SM).
            // List it -- (table, row, first sorted position, length, first slice) like the general path's
            // list -- for the slice blocks of k_seg_all.
            uint32_t lo = p + DAISY_SMALL_SLICE, hi = n_c - 1;
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if ((sk[mid] >> vb) == row) lo = mid; else hi = mid - 1;
            }
            const uint32_t len = lo - p + 1;
            const uint32_t r = atomicAdd(&longs[0], 1u);
            const uint32_t sl0 = atomicAdd(&longs[1], (len + DAISY_SMALL_SLICE - 1) / DAISY_SMALL_SLICE);
            if ((int)r < longs_cap) {
                uint32_t *rec = longs + 2 + 5 * (size_t)r;
                rec[0] = items ? 1u : 0u;
                rec[1] = row;
                rec[2] = base_c + p;
                rec[3] = len;
                rec[4] = sl0;
            }
        }
        if (!items)
            uslot[idx] = slot;
        else if (idx < (uint32_t)B)
            jslot[idx] = slot;
        else
            islot[idx - B] = slot;
    }
}

// ------------------------------------------------------------------------------------------------
// Mid-size batches (DAISY_SMALL_CAP < B <= DAISY_MID_CAP): the same class-split bookkeeping, generalised.
// At these sizes the CUB chain of the general path is a latency chain of ~15 kernels (~140 us whatever B is), while
// the table kernels need 20-80 us.  k_mid_book does the whole bookkeeping in ONE launch of 2 * 2^cb blocks: block c of
// a table sweeps ALL refs of its table twice (count, then compact its class -- rows with low bits c -- as (row >> cb,
// ref index) pairs into its slice [base_c, base_c + n_c) of a global scratch array; base_c = refs of lower classes),
// sorts its slice on the remaining row bits with the LSD passes of block_sort_words -- here between two global
// (L2-resident) buffers, so a class may have any size: a warp owns a contiguous range of the slice, counts its digits
// in one sweep and recomputes the lane matches in the scatter sweep instead of keeping ranks in registers -- and
// assigns the slots.  Refs are pairs, so there is no 32-bit packing limit.  No block waits for another one.
// ------------------------------------------------------------------------------------------------
static int bits_for(uint64_t max_value);
#define DAISY_MID_CAP 131072
#define DAISY_MID_TILE 8192  // refs per sweep tile: 1024 threads x 8
struct MidScratch {
    uint32_t *ak, *av, *bk, *bv;  // [3 * mid cap] each: user refs at [0, B), item refs at [B, 3B)
};

// Item sweep slots 2t and 2t + 1 are the negative and the positive item of triple t (adjacent words: a warp's loads
// cover contiguous bytes); mid_ref gives the ref index a slot is filed under (negatives [0, B), positives [B, 2B)).
__device__ __forceinline__ uint32_t mid_ref(int s, int B, bool items) {
    return items ? (uint32_t)((s & 1) ? B + (s >> 1) : (s >> 1)) : (uint32_t)s;
}

__global__ void __launch_bounds__(1024) k_mid_book(const int32_t *__restrict__ triples, int B, uint32_t U, uint32_t I, int cb,
                                                    int kbU, int kbQ, MidScratch ms, int32_t *__restrict__ st,
                                                    uint32_t *__restrict__ ukey_s, uint32_t *__restrict__ qkey_s,
                                                    uint32_t *__restrict__ uslot, uint32_t *__restrict__ jslot,
                                                    uint32_t *__restrict__ islot, uint32_t *longs, int longs_cap,
                                                    int *err) {
    extern __shared__ __align__(16) unsigned char mid_dsm[];
    uint32_t *hist = reinterpret_cast<uint32_t *>(mid_dsm);  // [32 * 513]
    __shared__ uint32_t scan_tmp[33], tw_off[32 * 32 + 1], s_low;
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t NC = 1u << cb;
    const bool items = blockIdx.x >= NC;
    const uint32_t cls = blockIdx.x & (NC - 1);
    const int n = items ? 2 * B : B;
    const int kb = items ? kbQ : kbU;
    const uint32_t bound = items ? I : U;
    const size_t tbl_off = items ? (size_t)B : 0;  // this table's part of the scratch arrays
    const int tiles = (n + DAISY_MID_TILE - 1) / DAISY_MID_TILE;  // <= 32
    if (tid == 0) s_low = 0;
    for (int i = tid; i < 32 * 32 + 1; i += 1024) tw_off[i] = 0;
    __syncthreads();
    // ---- sweep 1: how many refs of this class every (tile, warp) holds; how many refs belong to lower classes ----
    uint32_t low = 0;
    const bool checker = !items && cls == 0;  // this block also validates the triples and writes the clamped copy
    // slot s = tile base + w*256 + k*32 + lane.  Its word in the packed triples: users 3s; items 3(s>>1) + 2 - (s&1)
    // (slots 2t, 2t+1 = negative, positive item of triple t) -- both advance by a constant per k, so a full tile is 8
    // loads at immediate offsets from one base; the sweeps are bound by the instruction count of one SM.
    const int wstep = items ? 48 : 96;
    auto load_tile = [&](int tl, uint32_t (&rows)[8]) {
        const int s0 = tl * DAISY_MID_TILE + w * 256 + lane;
        const int32_t *p0 = triples + (items ? 3 * (s0 >> 1) + 2 - (s0 & 1) : 3 * s0);
        if (tl * DAISY_MID_TILE + DAISY_MID_TILE <= n) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t r = (uint32_t)__ldg(p0 + k * wstep);
                rows[k] = r < bound ? r : 0u;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                rows[k] = 0xFFFFFFFFu;
                if (s0 + k * 32 < n) {
                    const uint32_t r = (uint32_t)__ldg(p0 + k * wstep);
                    rows[k] = r < bound ? r : 0u;
                }
            }
        }
    };
    uint32_t nxt[8];
    load_tile(0, nxt);
    for (int tl = 0; tl < tiles; ++tl) {
        uint32_t rows[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) rows[k] = nxt[k];
        if (tl + 1 < tiles) load_tile(tl + 1, nxt);  // the next tile's loads fly while this one is counted
        if (checker) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int t = tl * DAISY_MID_TILE + w * 256 + k * 32 + lane;
                if (t < n) {
                    uint32_t u, i, j;
                    bool bad;
                    load_triple(triples, t, U, I, u, i, j, bad);
                    st[3 * (size_t)t] = (int32_t)u;
                    st[3 * (size_t)t + 1] = (int32_t)i;
                    st[3 * (size_t)t + 2] = (int32_t)j;
                    if (bad) {
                        atomicOr(&err[0], 1);
                        atomicMin(&err[1], t);
                    }
                }
            }
        }
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const bool in = rows[k] != 0xFFFFFFFFu;
            const uint32_t c = rows[k] & (NC - 1);
            mine += (in && c == cls) ? 1u : 0u;
            low += (in && c < cls) ? 1u : 0u;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(FULL, mine, o);
        if (lane == 0) tw_off[tl * 32 + w] = mine;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) low += __shfl_xor_sync(FULL, low, o);
    if (lane == 0 && low) atomicAdd(&s_low, low);
    __syncthreads();
    // exclusive scan of the 1024 (tile, warp) counts: thread t owns cell t
    uint32_t n_c;
    {
        const uint32_t c = tw_off[tid];
        uint32_t incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) scan_tmp[w] = incl;
        __syncthreads();
        if (w == 0) {
            const uint32_t tot = scan_tmp[lane];
            uint32_t inc2 = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(FULL, inc2, o);
                if (lane >= o) inc2 += v;
            }
            scan_tmp[lane] = inc2 - tot;
            if (lane == 31) scan_tmp[32] = inc2;
        }
        __syncthreads();
        tw_off[tid] = scan_tmp[w] + incl - c;
        n_c = scan_tmp[32];
    }
    const uint32_t base_c = s_low;
    __syncthreads();
    uint32_t *ak = ms.ak + tbl_off + base_c, *av = ms.av + tbl_off + base_c;
    uint32_t *bk = ms.bk + tbl_off + base_c, *bv = ms.bv + tbl_off + base_c;
    // ---- sweep 2: compact this class's refs, in ref order, as (row >> cb, ref index) ----
    load_tile(0, nxt);
    for (int tl = 0; tl < tiles; ++tl) {
        uint32_t rows[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) rows[k] = nxt[k];
        if (tl + 1 < tiles) load_tile(tl + 1, nxt);
        uint32_t run = tw_off[tl * 32 + w];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const bool mine = rows[k] != 0xFFFFFFFFu && (rows[k] & (NC - 1)) == cls;
            const unsigned m = __ballot_sync(FULL, mine);
            if (mine) {
                const uint32_t pos = run + __popc(m & lt);
                ak[pos] = rows[k] >> cb;
                av[pos] = mid_ref(tl * DAISY_MID_TILE + w * 256 + k * 32 + lane, B, items);
            }
            run += __popc(m);
        }
    }
    __syncthreads();  // (block-scope visibility of the global stores above)
    // ---- LSD passes between (ak, av) and (bk, bv): warp w owns [w * len_w, (w + 1) * len_w) of the slice ----
    const uint32_t len_w = (((n_c + 31u) / 32u) + 31u) & ~31u;
    const uint32_t r0 = (uint32_t)w * len_w, r1 = min(r0 + len_w, n_c);
    int nbits = kb - cb;
    if (nbits < 1) nbits = 1;
    const int passes = (nbits + 8) / 9;
    int done = 0;
    for (int p = 0; p < passes && n_c > 0; ++p) {
        int db = (nbits - done + (passes - p) - 1) / (passes - p);
        if (db < 5) db = 5;
        const int NB = 1 << db, HS = NB + 1;
        const uint32_t dmask = (uint32_t)NB - 1u;
        uint32_t *wh = hist + (size_t)w * HS;
        for (int i = lane; i < NB; i += 32) wh[i] = 0;
        __syncwarp();
        for (uint32_t q = r0 + lane; q - lane < r1; q += 32) {  // count
            const bool valid = q < r1;
            const uint32_t d = valid ? ((ak[q] >> done) & dmask) : 0u;
            const unsigned vm = __ballot_sync(FULL, valid);
            unsigned m = vm;
            for (int bb = 0; bb < db; ++bb) {
                const bool bit = (d >> bb) & 1u;
                const unsigned v = __ballot_sync(FULL, valid && bit);
                m &= bit ? v : (vm & ~v);
            }
            if (valid && lane == __ffs(m) - 1) wh[d] += __popc(m);
            __syncwarp();
        }
        __syncthreads();
        {   // exclusive scan of the cells in (digit, warp) order: thread t owns E consecutive cells
            const int E = NB / 32;
            uint32_t sum = 0;
            for (int e = 0; e < E; ++e) {
                const int L = tid * E + e;
                sum += hist[(size_t)(L & 31) * HS + (L >> 5)];
            }
            uint32_t incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += v;
            }
            if (lane == 31) scan_tmp[w] = incl;
            __syncthreads();
            if (w == 0) {
                const uint32_t tot = scan_tmp[lane];
                uint32_t inc2 = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t v = __shfl_up_sync(FULL, inc2, o);
                    if (lane >= o) inc2 += v;
                }
                scan_tmp[lane] = inc2 - tot;
            }
            __syncthreads();
            uint32_t run = scan_tmp[w] + incl - sum;
            for (int e = 0; e < E; ++e) {
                const int L = tid * E + e;
                uint32_t *cell = hist + (size_t)(L & 31) * HS + (L >> 5);
                const uint32_t c = *cell;
                *cell = run;
                run += c;
            }
        }
        __syncthreads();
        for (uint32_t q = r0 + lane; q - lane < r1; q += 32) {  // scatter: the matches again, offsets advance as we go
            const bool valid = q < r1;
            const uint32_t key = valid ? ak[q] : 0u, val = valid ? av[q] : 0u;
            const uint32_t d = (key >> done) & dmask;
            const unsigned vm = __ballot_sync(FULL, valid);
            unsigned m = vm;
            for (int bb = 0; bb < db; ++bb) {
                const bool bit = (d >> bb) & 1u;
                const unsigned v = __ballot_sync(FULL, valid && bit);
                m &= bit ? v : (vm & ~v);
            }
            const int leader = valid ? __ffs(m) - 1 : 0;
            uint32_t base = 0;
            if (valid && lane == leader) {
                base = wh[d];
                wh[d] = base + __popc(m);
            }
            base = __shfl_sync(FULL, base, leader);
            if (valid) {
                const uint32_t pos = base + __popc(m & lt);
                bk[pos] = key;
                bv[pos] = val;
            }
            __syncwarp();
        }
        __syncthreads();
        uint32_t *t;
        t = ak; ak = bk; bk = t;
        t = av; av = bv; bv = t;
        done += db;
    }
    // ---- slots: (ak, av) is the class's slice, sorted by row, refs of a row in ref order ----
    uint32_t *key_out = (items ? qkey_s : ukey_s) + base_c;
    for (uint32_t p = tid; p < n_c; p += 1024) {
        const uint32_t key = ak[p], idx = av[p];
        const bool first = (p == 0) || (ak[p - 1] != key);
        const bool last = (p == n_c - 1) || (ak[p + 1] != key);
        const uint32_t slot = (first && last) ? DAISY_DIRECT : base_c + p;
        const uint32_t row = (key << cb) | cls;
        key_out[p] = row;
        if (!items)
            uslot[idx] = slot;
        else if (idx < (uint32_t)B)
            jslot[idx] = slot;
        else
            islot[idx - B] = slot;
        if (first && p + DAISY_SMALL_SLICE < n_c && ak[p + DAISY_SMALL_SLICE] == key) {  // a long row (cf. k_small_book)
            uint32_t lo = p + DAISY_SMALL_SLICE, hi = n_c - 1;
            while (lo < hi) {
                const uint32_t mid = (lo + hi + 1) >> 1;
                if (ak[mid] == key) lo = mid; else hi = mid - 1;
            }
            const uint32_t len = lo - p + 1;
            const uint32_t r = atomicAdd(&longs[0], 1u);
            const uint32_t sl0 = atomicAdd(&longs[1], (len + DAISY_SMALL_SLICE - 1) / DAISY_SMALL_SLICE);
            if ((int)r < longs_cap) {
                uint32_t *rec = longs + 2 + 5 * (size_t)r;
                rec[0] = items ? 1u : 0u;
                rec[1] = row;
                rec[2] = base_c + p;
                rec[3] = len;
                rec[4] = sl0;
            }
        }
    }
}

static int launch_mid_book(daisy_ctx *h, cudaStream_t bs, const int32_t *triples, int B, uint32_t U, uint32_t I, BookSet &k) {
    const size_t smem = sizeof(uint32_t) * DAISY_SMALL_HIST_WORDS;
    static bool granted[64];
    if (!granted[h->device & 63]) {
        DAISY_CUDA(cudaFuncSetAttribute(k_mid_book, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        granted[h->device & 63] = true;
    }
    // classes: enough blocks to fill the GPU, few enough that a class still holds a few thousand refs
    const int cb = B <= 16384 ? 4 : (B <= 65536 ? 5 : 6);
    MidScratch ms;
    const size_t cap3 = 3 * (size_t)h->mid_cap;
    ms.ak = h->mid_buf; ms.av = ms.ak + cap3; ms.bk = ms.av + cap3; ms.bv = ms.bk + cap3;
    DAISY_CUDA(cudaMemsetAsync(k.longs, 0, 2 * sizeof(uint32_t), bs));
    k_mid_book<<<2 << cb, 1024, smem, bs>>>(triples, B, U, I, cb, bits_for(U), bits_for(I), ms, k.st, k.ukey_s, k.qkey_s,
                                            k.uslot, k.jslot, k.islot, k.longs, h->longs_cap, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

template <int IPT>
static int launch_small_book(daisy_ctx *h, cudaStream_t bs, const int32_t *triples, int B, uint32_t U, uint32_t I, int vbU,
                             int kbU, int vbQ, int kbQ, BookSet &k, int pairs = 0) {
    const size_t smem = sizeof(uint32_t) * (DAISY_SMALL_HIST_WORDS + 1024 * IPT);
    static bool granted[64];
    if (!granted[h->device & 63]) {
        DAISY_CUDA(cudaFuncSetAttribute(k_small_book<IPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        granted[h->device & 63] = true;
    }
    DAISY_CUDA(cudaMemsetAsync(k.longs, 0, 2 * sizeof(uint32_t), bs));
    k_small_book<IPT><<<2 << DAISY_SMALL_CB, 1024, smem, bs>>>(triples, B, U, I, vbU, kbU, vbQ, kbQ, k.st, k.ukey_s,
                                                             k.qkey_s, k.uslot, k.jslot, k.islot, k.longs,
                                                             h->longs_cap, h->err, pairs);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

// ------------------------------------------------------------------------------------------------
// Every row with several contributions, both tables, ONE launch (all paths; in the row-sharded step `opt` is PushOpt,
// which stores a finished item-row sum into its owner's memory over NVLink).
//   blocks [0, NS)                  slice blocks: the rows the bookkeeping listed as longer than `long_len`.  One SM
//        draws ~40 B/clk from L2 however many loads it has in flight (DESIGN.md §4b), so a hot row's
//        staged contributions are spread over the SMs slice by slice: a warp sums one slice of SLICE contributions
//        into stage2, takes a ticket of its row, and the warp that draws the row's last ticket adds the slice sums
//        IN SLICE ORDER and updates the row -- the order of the sum is fixed by the slice numbers, not by who
//        arrives when.  They come first in the grid so that they run under the window blocks, not after them.
//   blocks [NS, NS + blocksU + blocksQ)   8 windows of WIN sorted refs each; a warp reduces the rows of up to
//        `long_len` contributions that start in its window
//   the last block                  the loss reduction
// ------------------------------------------------------------------------------------------------
template <int V, class Opt, int WIN, int SLICE>
__global__ void __launch_bounds__(256) k_seg_all(const float *__restrict__ P, const float *__restrict__ Q,
                                                  const uint32_t *__restrict__ ukey_s,
                                                  const uint32_t *__restrict__ qkey_s, int B, int nQ, uint32_t q_sentinel,
                                                  const float *__restrict__ stageU, const float *__restrict__ stageQ,
                                                  float *__restrict__ stage2, int D4, Opt opt, int NS, int blocksU,
                                                  int blocksQ, int long_len, const uint32_t *__restrict__ longs,
                                                  int longs_cap, uint32_t *ticket, const float *__restrict__ loss_part,
                                                  int n_part, double *loss_accum, int ilvQ,
                                                  const uint32_t *__restrict__ counts) {
    const int b = blockIdx.x, wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    if (b >= NS + blocksU + blocksQ) {  // fixed-order reduction of the per-warp loss partials (double accumulation)
        if (!loss_accum) return;
        __shared__ double sh[8];
        double s = 0.0;
        for (int i = threadIdx.x; i < n_part; i += 256) s += (double)loss_part[i];
        s = warp_sum_d(s);
        if (lane == 0) sh[wid] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int i = 0; i < 8; ++i) t += sh[i];
            *loss_accum += t;
        }
        return;
    }
    if (b >= NS) {
        const int wb = b - NS;
        const int tbl = wb < blocksU ? 0 : 1;
        int w = tbl ? wb - blocksU : wb;
        if (tbl && ilvQ > 1) {
            // row-sharded step: the sorted item refs are grouped by owner, so blocks that start together would all
            // push to the same owner (incast); deal the item blocks round-robin over ilvQ ranges of the order instead
            // (blocksQ was rounded up to a multiple of ilvQ by the launcher; windows past the end find no refs)
            const int per = blocksQ / ilvQ;
            w = (w % ilvQ) * per + w / ilvQ;
        }
        // counts (merged sort of the refs of repeated rows): the ref counts of the two tables are known on the device
        // only, and the grid may hold fewer windows than there are -- a table's blocks stride over its windows
        const int n = counts ? (int)counts[tbl] : (tbl ? nQ : B);
        const long long stride = 8LL * (tbl ? blocksQ : blocksU);
        for (long long ww = (long long)w * 8 + wid; ww * WIN < n; ww += stride)
            seg_window<V, Opt, WIN>(ww, tbl, tbl ? Q : P, tbl ? qkey_s : ukey_s, n, tbl ? q_sentinel : 0xFFFFFFFFu,
                                    tbl ? stageQ : stageU, D4, opt, long_len);
        return;
    }
    const int count = min((int)longs[0], longs_cap);
    if (count == 0) return;
    const int total = (int)longs[1];
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;
    // consecutive slices go to different blocks (SMs): slice s is taken by warp (s / NS) % 8 of block s % NS
    for (int s = b + NS * wid; s < total; s += NS * 8) {
        int r = -1;
        for (int r0 = 0; r0 < count && r < 0; r0 += 32) {  // the row this slice belongs to
            bool hit = false;
            if (r0 + lane < count) {
                const uint32_t *rec = longs + 2 + 5 * (size_t)(r0 + lane);
                const int sl0 = (int)rec[4], nsl = (int)((rec[3] + SLICE - 1) / SLICE);
                hit = s >= sl0 && s < sl0 + nsl;
            }
            const unsigned m = __ballot_sync(FULL, hit);
            if (m) r = r0 + __ffs(m) - 1;
        }
        if (r < 0) continue;  // a record beyond longs_cap was dropped (cannot happen: the cap covers 3B / long_len rows)
        const uint32_t *rec = longs + 2 + 5 * (size_t)r;
        const int tbl = (int)rec[0];
        const uint32_t row = rec[1];
        const size_t q0 = rec[2];
        const int len = (int)rec[3], sl0 = (int)rec[4];
        const int nsl = (len + SLICE - 1) / SLICE, j = s - sl0;
        float4 acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = f4_zero();
        sum_staged<V>(tbl ? stageQ : stageU, q0 + (size_t)j * SLICE, min(SLICE, len - j * SLICE), D4, lane, act, acc);
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) __stcg(reinterpret_cast<float4 *>(stage2) + (size_t)s * D4 + lane + 32 * v, acc[v]);
        __threadfence();
        __syncwarp();
        uint32_t t = 0;
        if (lane == 0) t = atomicAdd(&ticket[r], 1u);
        t = __shfl_sync(FULL, t, 0);
        if ((int)t != nsl - 1) continue;
        // last slice of the row to finish: every slice sum is in L2
        __threadfence();
        if (lane == 0) ticket[r] = 0;  // ready for the next step
        const float *table = tbl ? Q : P;
        const float4 *s2 = reinterpret_cast<const float4 *>(stage2) + (size_t)sl0 * D4;
        float4 tot[V];
#pragma unroll
        for (int v = 0; v < V; ++v) tot[v] = f4_zero();
        // fixed order: groups of 64 slices (group sums added in group order), slices of a group in slice order, 8
        // loads in flight -- two levels so that the rounding error of a very long row does not grow with its length
        for (int g0 = 0; g0 < nsl; g0 += 64) {
            float4 grp[V];
#pragma unroll
            for (int v = 0; v < V; ++v) grp[v] = f4_zero();
            const int g1 = min(nsl, g0 + 64);
            constexpr int CT = 8;
            for (int j0 = g0; j0 < g1; j0 += CT) {
                float4 rr[CT][V];
#pragma unroll
                for (int jj = 0; jj < CT; ++jj)
#pragma unroll
                    for (int v = 0; v < V; ++v)
                        rr[jj][v] = (j0 + jj < g1 && act[v]) ? __ldcg(s2 + (size_t)(j0 + jj) * D4 + lane + 32 * v) : f4_zero();
#pragma unroll
                for (int jj = 0; jj < CT; ++jj)
                    if (j0 + jj < g1) {
#pragma unroll
                        for (int v = 0; v < V; ++v) grp[v] = f4_add(grp[v], rr[jj][v]);
                    }
            }
#pragma unroll
            for (int v = 0; v < V; ++v) tot[v] = f4_add(tot[v], grp[v]);
        }
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                const int e = lane + 32 * v;
                const float4 old = (tbl == 0 || Opt::kNeedOldItem) ? ld_row(table, (size_t)row * D4 + e) : f4_zero();
                opt.apply(tbl, (size_t)row, e, old, tot[v]);
            }
    }
}

// General path: list the rows with more than `long_len` contributions while the slots are assigned (bookkeeping
// stream), so that k_seg_all's slice blocks can start on them at once.  Called by the thread at a row's FIRST sorted
// position p; keys[p .. ] == row.
__device__ __forceinline__ void list_long_row(const uint32_t *__restrict__ keys, int n, int p, uint32_t row, int tbl,
                                              int long_len, int slice, uint32_t *longs, int longs_cap) {
    if (p + long_len >= n || keys[p + long_len] != row) return;
    int lo = p + long_len, hi = n - 1;
    while (lo < hi) {
        const int mid = (int)(((long long)lo + hi + 1) >> 1);
        if (keys[mid] == row) lo = mid; else hi = mid - 1;
    }
    const uint32_t len = (uint32_t)(lo - p + 1);
    const uint32_t r = atomicAdd(&longs[0], 1u);
    const uint32_t sl0 = atomicAdd(&longs[1], (len + slice - 1) / slice);
    if ((int)r < longs_cap) {
        uint32_t *rec = longs + 2 + 5 * (size_t)r;
        rec[0] = (uint32_t)tbl;
        rec[1] = row;
        rec[2] = (uint32_t)p;
        rec[3] = len;
        rec[4] = sl0;
    }
}

__global__ void k_list_long_items(const uint32_t *__restrict__ key, int n, uint32_t sentinel, uint32_t *longs,
                                  int longs_cap, int long_len) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t r = key[p];
    if (r == sentinel) return;
    if (p == 0 || key[p - 1] != r) list_long_row(key, n, p, r, 1, long_len, DAISY_SLICE, longs, longs_cap);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int bits_for(uint64_t max_value) {  // number of low bits needed to represent max_value
    int b = 1;
    while (b < 32 && (max_value >> b)) ++b;
    return b;
}

// merged sort of the 3B refs (book_kernels): worth it when it costs no more element-passes than the two separate sorts
// (it always saves the fixed cost of one sort: histogram + scan launches and one wave per pass)
static bool use_merged_sort(const daisy_ctx *h, uint32_t U, uint32_t I) {
    if (h->merged_sort == 0 || !h->ref_ws) return false;
    if ((uint64_t)U + I > 0xFFFFFFF0ull || (int64_t)U + I > h->ref_rows) return false;
    if (h->merged_sort == 1) return true;
    const int pu = (bits_for(U - 1) + 7) / 8, pq = (bits_for(I) + 7) / 8, pm = (bits_for((uint64_t)I + U) + 7) / 8;
    return 3 * pm <= pu + 2 * pq;
}

static int auto_chunk(const daisy_ctx *h, int64_t B) {
    if (h->chunk > 0) return h->chunk;
    // keep >= ~4 waves of 32 resident warps per SM before growing the chunk
    const int64_t want_warps = (int64_t)h->num_sms * 32 * 4;
    int c = 1;
    while (c < 32 && B / (2 * c) >= want_warps) c *= 2;  // 32 at 1 M triples: main kernel 0.43 ms vs 0.45 at 16
    return c;
}

static inline void phase_mark(daisy_ctx *h, int ph, cudaStream_t s) {
    if (h->timing == 2) cudaEventRecord(h->ev[ph + 1], s);
}

// ------------------------------------------------------------------------------------------------
// row-sharded bookkeeping (shard.cu): item refs carry GLOBAL ids; the sorted, de-duplicated ids of the batch are
// its CACHE rows (cache row c = c-th smallest id => grouped by owner block)
// ------------------------------------------------------------------------------------------------
struct StartFlag {  // 1 where a new row starts in the sorted item refs
    const uint32_t *key;
    uint32_t sentinel;
    __host__ __device__ __forceinline__ uint32_t operator()(int p) const {
        const uint32_t r = key[p];
        return (r != sentinel && (p == 0 || key[p - 1] != r)) ? 1u : 0u;
    }
};

// k_slots_item + cache-row assignment: cidx[p] = inclusive count of row starts up to p, so the cache row of sorted
// ref p is cidx[p] - 1.  Rewrites the item columns of the sorted triples from global ids to cache rows, lists the
// global id of every cache row and the first cache row of every owner.
__global__ void k_slots_item_shard(const uint32_t *__restrict__ key, const uint32_t *__restrict__ val,
                                   const uint32_t *__restrict__ cidx, int n, int B, uint32_t sentinel, uint32_t i_per,
                                   int G, uint32_t *__restrict__ jslot, uint32_t *__restrict__ islot,
                                   int32_t *__restrict__ st, uint32_t *__restrict__ uniq_gid,
                                   uint32_t *__restrict__ owner_off, ShardPeers peers, const float *__restrict__ cache,
                                   int D, const float **__restrict__ jsrc, const float **__restrict__ isrc,
                                   uint8_t *__restrict__ uniq_multi) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t r = key[p];
    if (r == sentinel) return;
    const bool first = (p == 0) || (key[p - 1] != r);
    const bool last = (p == n - 1) || (key[p + 1] != r);
    const uint32_t slot = (first && last) ? DAISY_DIRECT : (uint32_t)p;
    const uint32_t c = cidx[p] - 1u;
    const uint32_t v = val[p];
    // where the main kernel reads this ref's pre-step row: a row referenced once in the batch is read straight from
    // its owner (peer load over NVLink, or local); a repeated row from the cache the fetch kernel fills once
    const uint32_t o_r = r / i_per;
    const float *from = (first && last) ? peers.q[o_r] + (size_t)(r - o_r * i_per) * D : cache + (size_t)c * D;
    if (v < (uint32_t)B) {
        jslot[v] = slot;
        st[3 * (size_t)v + 2] = (int32_t)c;
        jsrc[v] = from;
    } else {
        islot[v - B] = slot;
        st[3 * (size_t)(v - B) + 1] = (int32_t)c;
        isrc[v - B] = from;
    }
    if (first) {
        uniq_gid[c] = r;
        uniq_multi[c] = last ? 0 : 1;
        const int o_cur = (int)(r / i_per);
        const int o_prev = (p == 0) ? -1 : (int)(key[p - 1] / i_per);
        for (int o = o_prev + 1; o <= o_cur; ++o) owner_off[o] = c;
    }
    if (last && (p == n - 1 || key[p + 1] == sentinel)) {  // the last real ref: close the offsets
        for (int o = (int)(r / i_per) + 1; o <= G; ++o) owner_off[o] = c + 1u;
    }
}

// Sorted item-ref keys become cache rows (same grouping and order: the map gid -> cache row is monotone), and every
// cache row gets the address it is fetched from (owner's q) and the address its descent sum is pushed to (region
// `me` of the owner's recv_g).
__global__ void k_shard_finish(uint32_t *__restrict__ key, const uint32_t *__restrict__ cidx, int n, uint32_t sentinel,
                               const uint32_t *__restrict__ uniq_gid, const uint32_t *__restrict__ owner_off, int G,
                               uint32_t i_per, int me, size_t cap, int D, ShardPeers peers,
                               const float **__restrict__ src, float **__restrict__ dst) {
    const uint32_t nuniq = owner_off[G];
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        if (key[p] != sentinel) key[p] = cidx[p] - 1u;
        if ((uint32_t)p < nuniq) {
            const uint32_t g = uniq_gid[p];
            const uint32_t o = g / i_per;
            src[p] = peers.q[o] + (size_t)(g - o * i_per) * D;
            dst[p] = peers.recv_g[o] + ((size_t)me * cap + ((uint32_t)p - owner_off[o])) * D;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// host orchestration: bookkeeping phase (depends on the triples only) + table phase
// ------------------------------------------------------------------------------------------------
struct StepPlan {
    int B, C;
    uint32_t U, I;        // id bounds: user rows, item ids (I is also the sentinel key of the item refs)
    bool piped;
    cudaStream_t bs, s;   // bookkeeping stream, caller's stream
    BookSet *k;
    int set;              // index of k in h->book
    const float *const *jsrc, *const *isrc;  // row-sharded step only (else null)
    bool small;           // small-batch path: k_small_book / C = 1 / k_seg_all
    int ilv;              // row-sharded step: chunk interleave of the main kernel (MainArgs::ilv), else 0
    const uint32_t *counts;  // merged sort: the set's device-side ref counts (BookSet::counts) for k_seg_all, else null
};

// Does a batch of B triples take the small-batch path?  Its refs must pack into 32 bits: row bits (of the VALUE U
// resp. I, so that the all-ones padding sorts behind every real row) + ref-index bits.
static bool small_path(const daisy_ctx *h, int64_t B, uint32_t U, uint32_t I, int *vbU, int *kbU, int *vbQ, int *kbQ) {
    if (B <= 0 || B > h->small_max) return false;
    *vbU = bits_for((uint64_t)(B - 1));
    *vbQ = bits_for((uint64_t)(2 * B - 1));
    *kbU = bits_for(U);
    *kbQ = bits_for(I);
    return *vbU + *kbU <= 32 && *vbQ + *kbQ <= 32;
}

// The kernels of the general bookkeeping chain (prep .. slots) on stream bs; phase marks go to the caller's stream.
static int book_kernels(daisy_ctx *h, BookSet &k, const StepPlan &pl, const int32_t *triples, int B, uint32_t U, uint32_t I,
                        int C, cudaStream_t bs, cudaStream_t s, const daisy_shard *sh) {
    const int T = 256;
    // prep
    k_prep<<<daisy_ceil_div(B, T), T, 0, bs>>>(triples, B, U, I, h->ikey_in, h->ival_in, h->err);
    DAISY_LAUNCH_CHECK(h);
    phase_mark(h, PH_PREP, s);
    // sort by positive item
    size_t tmp = h->cub_tmp_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_tmp, tmp, h->ikey_in, h->ikey_out, h->ival_in, h->ival_out, B, 0,
                                               bits_for(I - 1), bs));
    h->launches += 4;
    phase_mark(h, PH_SORT_I, s);
    // refs
    // One sort for the user and item refs when the table is not sharded and the combined key space costs no extra radix
    // passes (config 4: 10 M users + 2 M items = 24 bits = 3 passes).  Only the refs of rows referenced more than once
    // in their table go into it: k_refs marks every row in two bitmaps (seen / dup), the compaction settles every other
    // ref as DIRECT and keeps the rest in their order (negatives, run heads, users), and ref_sort.cuh sorts those --
    // about 0.7 M of the 3 M refs of a config-4 batch -- with a count that stays on the device.  The sort is stable and
    // the refs of a row keep their order, so every row is summed in the same order as by two full sorts.
    if (pl.counts) {
        uint32_t *ws = h->ref_ws;
        DsortState *ss = reinterpret_cast<DsortState *>(ws);
        const size_t bm_words = (size_t)((h->ref_rows + 31) / 32);
        uint32_t *seen = ws + sizeof(DsortState) / 4, *dup = seen + bm_words, *status = dup + bm_words;
        DAISY_CUDA(cudaMemsetAsync(ws, 0, (sizeof(DsortState) / 4 + 2 * bm_words + dsort_tiles(3 * (int64_t)B)) * sizeof(uint32_t), bs));
        k_refs<<<daisy_ceil_div(B, T), T, 0, bs>>>(triples, h->ival_out, h->ikey_out, B, U, I, C, k.st, h->key_in + 2 * (size_t)B,
                                                   nullptr, h->key_in, nullptr, k.islot, I + 1u, k.longs, seen, dup);
        DAISY_LAUNCH_CHECK(h);
        phase_mark(h, PH_REFS, s);
        uint32_t *skey, *sval;
        const BprRefSrc src{h->key_in, dup, B, I, k.jslot, k.islot, k.uslot};
        h->launches += dsort_launch(src, 3 * B, I, bits_for((uint64_t)I + U), h->key_out, h->val_out, h->key_in, h->val_in,
                                    ss, status, 2 * h->num_sms, bs, &skey, &sval) - 1;
        DAISY_LAUNCH_CHECK(h);
        phase_mark(h, PH_SORT_U, s);
        phase_mark(h, PH_SORT_Q, s);
        const int gs = daisy_ceil_div(3 * (int64_t)B, T);
        k_slots_dup<<<gs < 8 * h->num_sms ? gs : 8 * h->num_sms, T, 0, bs>>>(skey, sval, ss, B, I, k.qkey_s, k.ukey_s, k.uslot,
                                                                          k.jslot, k.islot, k.counts, k.longs, h->longs_cap,
                                                                          h->heavy_len);
        DAISY_LAUNCH_CHECK(h);
        return DAISY_OK;
    }
    k_refs<<<daisy_ceil_div(B, T), T, 0, bs>>>(triples, h->ival_out, h->ikey_out, B, U, I, C, k.st, h->ukey_in,
                                               h->uval_in, h->key_in, h->val_in, k.islot, 0u, nullptr, nullptr, nullptr);
    DAISY_LAUNCH_CHECK(h);
    phase_mark(h, PH_REFS, s);
    tmp = h->cub_tmp_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_tmp, tmp, h->ukey_in, k.ukey_s, h->uval_in, h->uval_out, B, 0,
                                               bits_for(U - 1), bs));
    h->launches += 4;
    phase_mark(h, PH_SORT_U, s);
    tmp = h->cub_tmp_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(h->cub_tmp, tmp, h->key_in, k.qkey_s, h->val_in, h->val_out, 2 * B, 0,
                                               bits_for(I), bs));
    h->launches += 4;
    phase_mark(h, PH_SORT_Q, s);
    // slots
    // the rows too long for one warp are listed here for k_seg_all's slice blocks
    uint32_t *longs = k.longs;
    DAISY_CUDA(cudaMemsetAsync(longs, 0, 2 * sizeof(uint32_t), bs));
    k_slots_user<<<daisy_ceil_div(B, T), T, 0, bs>>>(k.ukey_s, h->uval_out, B, k.uslot, longs, h->longs_cap, h->heavy_len);
    DAISY_LAUNCH_CHECK(h);
    if (!sh) {
        k_slots_item<<<daisy_ceil_div(2 * (int64_t)B, T), T, 0, bs>>>(k.qkey_s, h->val_out, 2 * B, B, I, k.jslot, k.islot,
                                                                      longs, h->longs_cap, h->heavy_len);
        DAISY_LAUNCH_CHECK(h);
    } else {
        const ShardSet &ss = sh->set[pl.set];
        auto flags = thrust::make_transform_iterator(thrust::counting_iterator<int>(0), StartFlag{k.qkey_s, I});
        tmp = h->cub_tmp_bytes;
        DAISY_CUDA(cub::DeviceScan::InclusiveSum(h->cub_tmp, tmp, flags, sh->cidx, 2 * B, bs));
        h->launches += 2;
        k_slots_item_shard<<<daisy_ceil_div(2 * (int64_t)B, T), T, 0, bs>>>(
            k.qkey_s, h->val_out, sh->cidx, 2 * B, B, I, (uint32_t)sh->i_per, sh->world, k.jslot, k.islot, k.st,
            ss.uniq_gid, ss.owner_off, sh->peers, sh->cache, h->D, ss.jsrc, ss.isrc, ss.multi);
        DAISY_LAUNCH_CHECK(h);
        k_shard_finish<<<daisy_ceil_div(2 * (int64_t)B, T), T, 0, bs>>>(k.qkey_s, sh->cidx, 2 * B, I, ss.uniq_gid,
                                                                         ss.owner_off, sh->world, (uint32_t)sh->i_per,
                                                                         sh->rank, (size_t)sh->cap, h->D, sh->peers,
                                                                         ss.src, ss.dst);
        DAISY_LAUNCH_CHECK(h);
        // the sorted item-ref keys now hold cache rows (same grouping): list the long ones
        k_list_long_items<<<daisy_ceil_div(2 * (int64_t)B, T), T, 0, bs>>>(k.qkey_s, 2 * B, I, longs, h->longs_cap,
                                                                           h->heavy_len);
        DAISY_LAUNCH_CHECK(h);
    }
    return DAISY_OK;
}

// The integer bookkeeping of a step (prep .. slots) depends on the triples only, never on the tables.  It runs on
// the handle's side stream into one of two bookkeeping sets, so that for step n+1 it overlaps the bandwidth-bound
// kernels of step n on the caller's stream.  Per-phase timing (mode 2) serialises everything on the caller's
// stream so that phase times do not overlap.
static int book_phase(daisy_ctx *h, StepPlan &pl, const int32_t *triples, int64_t B64, uint32_t U, uint32_t I,
                      cudaStream_t s, const int32_t *host_src, bool inputs_ready, const daisy_shard *sh) {
    const int B = (int)B64;
    int vbU = 0, kbU = 0, vbQ = 0, kbQ = 0;
    const int pairs = h->pairs_mode;  // csrc/gmf.cu: (user, item, label) samples, one item ref each
    bool tiny = !sh && small_path(h, B64, U, I, &vbU, &kbU, &vbQ, &kbQ);
    if (pairs) {
        vbQ = bits_for((uint64_t)(B64 > 1 ? B64 - 1 : 1));
        tiny = B64 > 0 && B64 <= DAISY_SMALL_CAP && vbU + kbU <= 32 && vbQ + kbQ <= 32 && h->small_max > 0 && B64 <= h->small_max;
        DAISY_REQUIRE(tiny, DAISY_EUNSUPPORTED, "the (user, item, label) step takes batches of 1..%d samples whose row and "
                      "sample indices pack into 32 bits (batch %lld, %u users, %u items)", h->small_max, (long long)B64, U, I);
    }
    const bool mid = !sh && !tiny && B64 > 0 && B64 <= h->mid_max;   // also small batches whose refs do not pack
    const bool small = tiny || mid;  // C = 1, one-launch bookkeeping, k_seg_all with short windows and slices
    const int C = small ? 1 : auto_chunk(h, B);
    const bool piped = h->pipeline && h->timing != 2;
    cudaStream_t bs = piped ? h->side_stream : s;
    pl.B = B; pl.C = C; pl.U = U; pl.I = I; pl.piped = piped; pl.bs = bs; pl.s = s;
    pl.set = h->book_idx;
    pl.small = small;
    pl.counts = nullptr;
    pl.jsrc = sh ? sh->set[pl.set].jsrc : nullptr;
    pl.isrc = sh ? sh->set[pl.set].isrc : nullptr;
    pl.ilv = sh ? sh->ilv : 0;
    BookSet &k = h->book[h->book_idx];
    pl.k = &k;
    if (!sh && !small && use_merged_sort(h, U, I)) pl.counts = k.counts;
    h->book_idx = (h->book_idx + 1) % DAISY_NSETS;
    if (h->timing == 2) {
        if (h->ev_pending) {  // fold the previous step's phase times in
            cudaEventSynchronize(h->ev[PH_COUNT]);
            for (int ph = 0; ph < PH_COUNT; ++ph) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, h->ev[ph], h->ev[ph + 1]);
                h->phase_ms_sum[ph] += ms;
            }
            h->timed_steps++;
            h->ev_pending = 0;
        }
        cudaEventRecord(h->ev[0], s);
    }
    if (piped) {
        if (!inputs_ready) {  // the triples may have been produced by earlier work on the caller's stream
            DAISY_CUDA(cudaEventRecord(h->ev_call, s));
            DAISY_CUDA(cudaStreamWaitEvent(bs, h->ev_call, 0));
        }
        DAISY_CUDA(cudaStreamWaitEvent(bs, k.freed, 0));  // the step that last used this set has finished
    }
    const bool tr = h->trace && h->tr_n < DAISY_TRACE_STEPS;
    if (tr) cudaEventRecord(h->tr_ev[4 * h->tr_n + 0], bs);
    if (host_src) {  // *_step_host: the H2D copy heads the bookkeeping chain
        // ... on a stream of its own: 12 MB of triples take ~0.22 ms over PCIe, and on the bookkeeping stream that time
        // adds to the chain's 0.56 ms -- more than the 0.65 ms the table kernels take, so the COPY set the pace of the
        // host-fed step (0.75 ms against 0.70 from device-resident triples, profiles/r02g).  The copy of step n+2 now
        // runs under the bookkeeping of step n+1; the landing zone is the set's own (free once the set is).
        if (piped) {
            DAISY_CUDA(cudaStreamWaitEvent(h->copy_stream, k.freed, 0));
            DAISY_CUDA(cudaMemcpyAsync((void *)triples, host_src, (size_t)B * 3 * sizeof(int32_t), cudaMemcpyHostToDevice,
                                       h->copy_stream));
            DAISY_CUDA(cudaEventRecord(k.copied, h->copy_stream));
            DAISY_CUDA(cudaStreamWaitEvent(bs, k.copied, 0));
        } else {
            DAISY_CUDA(cudaMemcpyAsync((void *)triples, host_src, (size_t)B * 3 * sizeof(int32_t), cudaMemcpyHostToDevice, bs));
        }
    }
    if (small) {
        for (int ph = PH_PREP; ph < PH_SLOTS; ++ph) phase_mark(h, ph, s);
        int rc;
        if (mid)
            rc = launch_mid_book(h, bs, triples, B, U, I, k);
        else if (2 * B <= 4096)
            rc = launch_small_book<4>(h, bs, triples, B, U, I, vbU, kbU, vbQ, kbQ, k, pairs);
        else if (2 * B <= 8192)
            rc = launch_small_book<8>(h, bs, triples, B, U, I, vbU, kbU, vbQ, kbQ, k, pairs);
        else
            rc = launch_small_book<16>(h, bs, triples, B, U, I, vbU, kbU, vbQ, kbQ, k, pairs);
        if (rc) return rc;
        phase_mark(h, PH_SLOTS, s);
        if (piped) {
            DAISY_CUDA(cudaEventRecord(k.ready, bs));
            DAISY_CUDA(cudaStreamWaitEvent(s, k.ready, 0));
        }
        if (tr) {
            cudaEventRecord(h->tr_ev[4 * h->tr_n + 1], bs);
            cudaEventRecord(h->tr_ev[4 * h->tr_n + 2], s);
        }
        return DAISY_OK;
    }
    // Mid-size batches are bound by what the HOST spends on these ~15 launches (three CUB dispatches among them:
    // 0.16 ms per step against 0.1 ms of device time at 65 536 triples), so the single-GPU bookkeeping chain of a
    // (set, batch size) is captured once into a CUDA graph and replayed: one launch.  Nothing in it varies from step
    // to step -- it reads the set's landing buffer and writes the set's arrays.
    const int32_t *landing = h->triples + (size_t)pl.set * 3 * (size_t)h->maxB;
    const bool graphed = piped && !sh && !tr && B64 <= h->graph_max_b;
    if (graphed && triples != landing) {  // device-resident triples: bring them to the fixed address the graph reads
        DAISY_CUDA(cudaMemcpyAsync((void *)landing, triples, (size_t)B * 3 * sizeof(int32_t), cudaMemcpyDeviceToDevice, bs));
        triples = landing;
    }
    if (graphed) {
        BookGraph *g = nullptr;
        for (int i = 0; i < h->n_bgraph; ++i)
            if (h->bgraph[i].set == pl.set && h->bgraph[i].B == B && h->bgraph[i].U == U && h->bgraph[i].I == I) g = &h->bgraph[i];
        if (!g) {
            const int64_t l0 = h->launches;
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            bool ok = cudaStreamBeginCapture(bs, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                const int rc = book_kernels(h, k, pl, triples, B, U, I, C, bs, s, sh);
                ok = (cudaStreamEndCapture(bs, &graph) == cudaSuccess) && rc == DAISY_OK && graph != nullptr;
                if (ok) ok = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
                if (graph) cudaGraphDestroy(graph);
            }
            if (ok) {
                int slot = h->n_bgraph < DAISY_MAX_BGRAPH ? h->n_bgraph++ : (h->bgraph_next++ % DAISY_MAX_BGRAPH);
                if (h->bgraph[slot].exec) cudaGraphExecDestroy(h->bgraph[slot].exec);
                g = &h->bgraph[slot];
                g->exec = exec; g->set = pl.set; g->B = B; g->U = U; g->I = I;
                g->launches = (int)(h->launches - l0);
            } else {  // capture is not available here: never try again, launch directly
                cudaGetLastError();
                h->graph_max_b = 0;
            }
            h->launches = l0;
        }
        if (g) {
            DAISY_CUDA(cudaGraphLaunch(g->exec, bs));
            h->launches += g->launches;
        } else {
            const int rc = book_kernels(h, k, pl, triples, B, U, I, C, bs, s, sh);
            if (rc) return rc;
        }
    } else {
        const int rc = book_kernels(h, k, pl, triples, B, U, I, C, bs, s, sh);
        if (rc) return rc;
    }
    phase_mark(h, PH_SLOTS, s);
    if (piped) {
        DAISY_CUDA(cudaEventRecord(k.ready, bs));
        DAISY_CUDA(cudaStreamWaitEvent(s, k.ready, 0));
    }
    if (tr) {
        cudaEventRecord(h->tr_ev[4 * h->tr_n + 1], bs);
        cudaEventRecord(h->tr_ev[4 * h->tr_n + 2], s);
    }
    return DAISY_OK;
}

// The table-touching kernels of a step, on the caller's stream: main, segmented reduces, hot rows, loss.
// Q is the item table (or, sharded, the cache of fetched rows; the sorted item-ref keys then hold cache rows).
template <int V, class Opt>
static int table_phase_v(daisy_ctx *h, const StepPlan &pl, const float *P, const float *Q, const Opt &opt, float c2,
                         double *loss_accum) {
    const int B = pl.B, C = pl.C;
    const int D4 = h->D / 4;
    cudaStream_t s = pl.s;
    BookSet &k = *pl.k;
    MainArgs a;
    a.P = P; a.Q = Q; a.st = k.st; a.uslot = k.uslot; a.jslot = k.jslot; a.islot = k.islot;
    a.stageU = h->stageU; a.stageQ = h->stageQ; a.loss_part = h->loss_part;
    a.B = B; a.D4 = D4; a.C = C; a.c2 = c2;
    a.jsrc = pl.jsrc; a.isrc = pl.isrc;
    a.ilv = pl.jsrc ? pl.ilv : 0;
    const int warps = daisy_ceil_div(B, C);
    const bool pool = (h->timing == 1 && h->pool_used < DAISY_EVPOOL);
    if (pool) cudaEventRecord(h->evpool[2 * h->pool_used], s);
    // interleaved (row-sharded step): ilv ranges of ceil(warps / ilv) chunks each, dealt round-robin
    const int warps_launched = a.ilv > 1 ? a.ilv * daisy_ceil_div(warps, a.ilv) : warps;
    const int blocks = daisy_ceil_div(warps_launched, 8);
    // TMA-pipelined variant: S stages of 3 rows per warp in shared memory, at most ~56 KB per block so that four
    // blocks stay resident per SM; rows too long for two stages fall back to the register-prefetch kernel
    const size_t stage_bytes = (size_t)8 * 3 * D4 * 16;
    int S = h->main_stages;
    if ((size_t)S * stage_bytes > (size_t)56 * 1024) S = (int)((size_t)56 * 1024 / stage_bytes);
    if (pl.small) S = 0;  // one triple per warp: nothing to pipeline
    if (S >= 2) {
        const size_t smem = S * stage_bytes + (size_t)8 * S * 8;
        static size_t granted_tab[2][64];  // per instantiation (V, Opt): shared memory already granted, by PTR and device
        size_t &granted = granted_tab[pl.jsrc ? 1 : 0][h->device & 63];
        if (pl.jsrc) {
            if (granted != smem)
                DAISY_CUDA(cudaFuncSetAttribute(k_bpr_main_tma<V, Opt, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_bpr_main_tma<V, Opt, true><<<blocks, 256, smem, s>>>(a, opt, S);
        } else {
            if (granted != smem)
                DAISY_CUDA(cudaFuncSetAttribute(k_bpr_main_tma<V, Opt, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_bpr_main_tma<V, Opt, false><<<blocks, 256, smem, s>>>(a, opt, S);
        }
        granted = smem;
    } else if (pl.jsrc) {
        k_bpr_main<V, Opt, true><<<blocks, 256, 0, s>>>(a, opt);
    } else {
        k_bpr_main<V, Opt, false><<<blocks, 256, 0, s>>>(a, opt);
    }
    DAISY_LAUNCH_CHECK(h);
    if (pool) {
        cudaEventRecord(h->evpool[2 * h->pool_used + 1], s);
        h->pool_used++;
    }
    phase_mark(h, PH_MAIN, s);
    {   // every multi-contribution row of both tables + the loss in one launch
        const int NS = (pl.small && B <= DAISY_SMALL_CAP) ? 64 : 2 * h->num_sms;
        int blocksU, blocksQ;
        const int ilvQ = (pl.jsrc && pl.ilv > 1) ? pl.ilv : 0;   // row-sharded step: owner-interleaved item blocks
        if (pl.small) {
            blocksU = daisy_ceil_div(B, 8 * DAISY_SMALL_WIN), blocksQ = daisy_ceil_div(2 * B, 8 * DAISY_SMALL_WIN);
            k_seg_all<V, Opt, DAISY_SMALL_WIN, DAISY_SMALL_SLICE><<<NS + blocksU + blocksQ + (loss_accum ? 1 : 0), 256, 0, s>>>(
                P, Q, k.ukey_s, k.qkey_s, B, 2 * B, 0xFFFFFFFFu, h->stageU, h->stageQ, h->stage2, D4, opt, NS, blocksU, blocksQ,
                DAISY_SMALL_SLICE, k.longs, h->longs_cap, h->ticket, h->loss_part, warps, loss_accum, 0, nullptr);
        } else {
            blocksU = daisy_ceil_div(B, 8 * 32), blocksQ = daisy_ceil_div(2 * (int64_t)B, 8 * 32);
            if (ilvQ) blocksQ = daisy_ceil_div(blocksQ, ilvQ) * ilvQ;
            if (pl.counts) {  // the merged sort holds only the refs of repeated rows, a count known on the device only
                const int cap = DAISY_SEG_WIN_BLOCKS * h->num_sms;
                if (blocksU > cap) blocksU = cap;
                if (blocksQ > cap) blocksQ = cap;
            }
            k_seg_all<V, Opt, 32, DAISY_SLICE><<<NS + blocksU + blocksQ + (loss_accum ? 1 : 0), 256, 0, s>>>(
                P, Q, k.ukey_s, k.qkey_s, B, 2 * B, pl.I, h->stageU, h->stageQ, h->stage2, D4, opt, NS, blocksU, blocksQ,
                h->heavy_len, k.longs, h->longs_cap, h->ticket, h->loss_part, warps, loss_accum, ilvQ, pl.counts);
        }
        DAISY_LAUNCH_CHECK(h);
        for (int ph = PH_SEG_U; ph <= PH_LOSS; ++ph) phase_mark(h, ph, s);
    }
    if (pl.piped) DAISY_CUDA(cudaEventRecord(k.freed, s));
    if (h->trace && h->tr_n < DAISY_TRACE_STEPS) {
        cudaEventRecord(h->tr_ev[4 * h->tr_n + 3], s);
        h->tr_n++;
    }
    if (h->timing == 2) {
        h->ev_pending = 1;
        h->ev_stream = s;
    }
    return DAISY_OK;
}

template <class Opt>
static int table_phase(daisy_ctx *h, const StepPlan &pl, const float *P, const float *Q, const Opt &opt, float c2,
                       double *loss_accum) {
    const int D4 = h->D / 4;
    if (D4 <= 32) return table_phase_v<1, Opt>(h, pl, P, Q, opt, c2, loss_accum);
    if (D4 <= 64) return table_phase_v<2, Opt>(h, pl, P, Q, opt, c2, loss_accum);
    if (D4 <= 96) return table_phase_v<3, Opt>(h, pl, P, Q, opt, c2, loss_accum);
    return table_phase_v<4, Opt>(h, pl, P, Q, opt, c2, loss_accum);
}

template <class Opt>
static int run_step(daisy_ctx *h, const float *P, const float *Q, const int32_t *triples, int64_t B, const Opt &opt,
                    float c2, double *loss_accum, cudaStream_t s, const int32_t *host_src, bool inputs_ready) {
    // the NCCL-exchange sharded step runs against a cache of fetched item rows whose row count differs from the
    // local item shard
    const uint32_t U = (uint32_t)h->U, I = (uint32_t)(h->item_rows_override ? h->item_rows_override : h->I);
    StepPlan pl;
    const int rc = book_phase(h, pl, triples, B, U, I, s, host_src, inputs_ready, nullptr);
    if (rc) return rc;
    return table_phase<Opt>(h, pl, P, Q, opt, c2, loss_accum);
}

static int check_step_args(daisy_ctx *h, const void *P, const void *Q, const void *triples, int64_t B) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DAISY_REQUIRE(P && Q && (triples || B == 0), DAISY_EINVAL, "null table or triples pointer");
    DAISY_REQUIRE(h->maxB > 0 && h->D % 4 == 0 && h->D <= 512, DAISY_EUNSUPPORTED,
                  "BPR step needs a handle created with max_batch > 0 and dim %% 4 == 0, dim <= 512 (dim is %d)", h->D);
    DAISY_REQUIRE(B >= 0 && B <= h->maxB, DAISY_EINVAL, "batch of %lld triples exceeds max_batch %lld", (long long)B,
                  (long long)h->maxB);
    DAISY_REQUIRE(((uintptr_t)P % 16 == 0) && ((uintptr_t)Q % 16 == 0), DAISY_EINVAL, "tables must be 16-byte aligned");
    return DAISY_OK;
}


}  // namespace
