// Row-sharded BPR step (SURVEY.md section 8e): see the header comment of each section.
#include "step_kernels.cuh"

namespace {

// Row-sharded step (SURVEY 8e): users are local (SGD + lazy L2 as above); the "item table" is a cache of rows fetched
// from their owners, and instead of updating it the step emits the complete descent sum of every cache row -- the
// owners apply them (k_owner_apply).  Every cache row is referenced by at least one triple, so every row of G is
// written exactly once.
struct ShardOpt {
    static constexpr bool kNeedOldItem = false;
    float *P, *G;
    float alpha;
    int D4;
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 old, float4 d) const {
        const size_t idx = row * D4 + e;
        if (tbl) {
            st_row(G, idx, d);
        } else {
            st_row(P, idx, make_float4(fmaf(alpha, d.x, old.x), fmaf(alpha, d.y, old.y), fmaf(alpha, d.z, old.z),
                                       fmaf(alpha, d.w, old.w)));
        }
    }
};

// ------------------------------------------------------------------------------------------------
// owner side of the sharded step: received (row, gradient-sum) pairs from all ranks, concatenated in rank order.
// A stable sort by row keeps the rank order inside each row; one warp per window of 32 sorted entries sums each
// row's contributions in that order and applies  Q[row] += alpha * sum  once.
// ------------------------------------------------------------------------------------------------
__global__ void k_owner_keys(const int32_t *__restrict__ rows, int n, uint32_t I, uint32_t *__restrict__ key,
                             uint32_t *__restrict__ val, int *err) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    uint32_t r = (uint32_t)rows[p];
    if (r >= I) {
        atomicOr(&err[0], 1);
        atomicMin(&err[1], p);
        r = 0;
    }
    key[p] = r;
    val[p] = (uint32_t)p;
}

template <int V>
__global__ void __launch_bounds__(256) k_owner_apply(float *__restrict__ Q, const uint32_t *__restrict__ keys,
                                                      const uint32_t *__restrict__ perm, int n,
                                                      const float *__restrict__ grads, int D4, float alpha) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const long long base = (long long)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5) * 32;
    if (base >= n) return;
    const long long p = base + lane;
    const uint32_t key = (p < n) ? keys[p] : 0xFFFFFFFFu;
    uint32_t prev = __shfl_up_sync(FULL, key, 1);
    if (lane == 0) prev = (p > 0) ? keys[p - 1] : ~key;
    const bool start = (p < n) && (prev != key);
    unsigned todo = __ballot_sync(FULL, start);
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;
    while (todo) {
        const int b = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t row = __shfl_sync(FULL, key, b);
        float4 acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = f4_zero();
        for (long long q = base + b; q < n; ++q) {  // contributions of this row: at most one per rank
            if (keys[q] != row) break;
            const size_t src = perm[q];
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v]) acc[v] = f4_add(acc[v], ld_stream(grads, src * D4 + lane + 32 * v));
        }
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) {
                const size_t e = (size_t)row * D4 + lane + 32 * v;
                const float4 old = ld_row(Q, e);
                st_row(Q, e, make_float4(fmaf(alpha, acc[v].x, old.x), fmaf(alpha, acc[v].y, old.y),
                                         fmaf(alpha, acc[v].z, old.z), fmaf(alpha, acc[v].w, old.w)));
            }
    }
}

}  // namespace

extern "C" int daisy_bpr_shard_step(daisy_handle_t h, float *P_local, const float *cache, int64_t cache_rows,
                                    const int32_t *triples, int64_t B, float lr, float wd, float *grad_out,
                                    double *loss_accum, daisy_stream_t stream) {
    if (h && B == 0) {  // a rank without triples this step still decays its rows
        const double sh = 1.0 - (double)lr * (double)wd;
        DAISY_REQUIRE(sh > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1", (double)lr * wd);
        h->scale *= sh;
        return DAISY_OK;
    }
    int rc = check_step_args(h, P_local, cache, triples, B);
    if (rc) return rc;
    DAISY_REQUIRE(grad_out != nullptr, DAISY_EINVAL, "null grad_out");
    DAISY_REQUIRE(cache_rows > 0 && cache_rows <= 2 * h->maxB, DAISY_EINVAL,
                  "cache_rows %lld must be in [1, 2 * max_batch]", (long long)cache_rows);
    DAISY_REQUIRE((uintptr_t)grad_out % 16 == 0, DAISY_EINVAL, "grad_out must be 16-byte aligned");
    const double shrink = 1.0 - (double)lr * (double)wd;
    DAISY_REQUIRE(shrink > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1", (double)lr * wd);
    if (B == 0) {
        h->scale *= shrink;
        return DAISY_OK;
    }
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    ShardOpt opt;
    opt.P = P_local;
    opt.G = grad_out;
    opt.alpha = (float)((double)lr / shrink);
    opt.D4 = h->D / 4;
    h->item_rows_override = cache_rows;
    rc = run_step<ShardOpt>(h, P_local, cache, triples, B, opt, (float)(h->scale * h->scale), loss_accum,
                            (cudaStream_t)stream, nullptr, h->inputs_ready != 0);
    h->item_rows_override = 0;
    if (rc) return rc;
    h->scale *= shrink;
    return DAISY_OK;
}

extern "C" int daisy_owner_apply(daisy_handle_t h, float *Q_local, const int32_t *rows, const float *grads, int64_t n,
                                 float lr, float wd, daisy_stream_t stream) {
    DAISY_REQUIRE(h && Q_local, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(h->D % 4 == 0 && h->D <= 512, DAISY_EUNSUPPORTED, "dim %d unsupported", h->D);
    DAISY_REQUIRE(n >= 0 && n < (1LL << 30), DAISY_EINVAL, "bad row count");
    const double shrink = 1.0 - (double)lr * (double)wd;
    DAISY_REQUIRE(shrink > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1", (double)lr * wd);
    if (n == 0) return DAISY_OK;
    DAISY_REQUIRE(rows && grads, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (h->own_cap < n) {  // grow-only scratch: (key, value) ping/pong + CUB temp
        DAISY_CUDA(cudaStreamSynchronize(s));
        for (void *p : {(void *)h->own_key, (void *)h->own_key_s, (void *)h->own_val, (void *)h->own_val_s, h->own_tmp})
            if (p) cudaFree(p);
        h->own_key = h->own_key_s = h->own_val = h->own_val_s = nullptr;
        h->own_tmp = nullptr;
        const size_t cap = (size_t)n + (size_t)n / 4 + 1024;
        size_t tb = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr,
                                        (uint32_t *)nullptr, (int)cap, 0, 32, s);
        bool ok = cudaMalloc((void **)&h->own_key, cap * 4) == cudaSuccess &&
                  cudaMalloc((void **)&h->own_key_s, cap * 4) == cudaSuccess &&
                  cudaMalloc((void **)&h->own_val, cap * 4) == cudaSuccess &&
                  cudaMalloc((void **)&h->own_val_s, cap * 4) == cudaSuccess &&
                  cudaMalloc(&h->own_tmp, tb + 256) == cudaSuccess;
        DAISY_REQUIRE(ok, DAISY_ENOMEM, "owner-side scratch allocation failed");
        h->own_cap = (int64_t)cap;
        h->own_tmp_bytes = tb + 256;
    }
    const int T = 256;
    k_owner_keys<<<daisy_ceil_div(n, T), T, 0, s>>>(rows, (int)n, (uint32_t)h->I, h->own_key, h->own_val, h->err);
    DAISY_LAUNCH_CHECK(h);
    size_t tb = h->own_tmp_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(h->own_tmp, tb, h->own_key, h->own_key_s, h->own_val, h->own_val_s, (int)n,
                                               0, bits_for((uint64_t)h->I - 1), s));
    h->launches += 4;
    const int D4 = h->D / 4;
    const float alpha = (float)((double)lr / shrink);
    const int grid = daisy_ceil_div(daisy_ceil_div(n, 32), 8);
    if (D4 <= 32) k_owner_apply<1><<<grid, 256, 0, s>>>(Q_local, h->own_key_s, h->own_val_s, (int)n, grads, D4, alpha);
    else if (D4 <= 64) k_owner_apply<2><<<grid, 256, 0, s>>>(Q_local, h->own_key_s, h->own_val_s, (int)n, grads, D4, alpha);
    else if (D4 <= 96) k_owner_apply<3><<<grid, 256, 0, s>>>(Q_local, h->own_key_s, h->own_val_s, (int)n, grads, D4, alpha);
    else k_owner_apply<4><<<grid, 256, 0, s>>>(Q_local, h->own_key_s, h->own_val_s, (int)n, grads, D4, alpha);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}


// =====================================================================================================================
// Row-sharded step over PEER MEMORY (NVLink / NVSwitch): no collective library on the data path.
//
// Every rank owns a block of user rows (local tensor) and a block of item rows that lives in its ARENA (ctx.cuh:
// daisy_shard), which all ranks of the node map through CUDA IPC.  Triples are routed to the owner of their user.
// One step of rank `me`, all asynchronous on the caller's stream, no host synchronisation:
//
//   bookkeeping  (side stream, overlaps the previous step)  the single-GPU bookkeeping on GLOBAL item ids + cache-row
//                assignment: the batch's distinct item ids, ascending = grouped by owner, each with the address it is
//                fetched from (owner's q) and the address its descent sum is pushed to (owner's recv_g, region `me`)
//   fetch        k_shard_fetch: pre-step rows of the batch's distinct items are READ from their owners' memory
//                (128-bit peer loads over NVLink, several rows in flight per warp) into the local cache; the ids and
//                counts of what this rank will push are WRITTEN into the owners' recv_ids / recv_cnt
//   compute      the fused step kernels against (P_local, cache); a finished item-row sum is stored straight into the
//                owner's memory by the kernel that completes it (PushOpt: k_bpr_main for rows referenced once,
//                k_seg_all for repeated rows) -- the transfer overlaps the arithmetic
//   barrier      k_shard_barrier: arrival flags written into every peer's arena, acquire-spin on the own flags
//   apply        k_owner_add, one pass per sender in sender-rank order (a sender's id list is duplicate-free, so a pass
//                is a plain streaming read-modify-write of distinct rows) -> deterministic
//   barrier      owners are done: peers may fetch the next step's rows and overwrite the receive regions
// =====================================================================================================================
namespace {

struct PushOpt {
    static constexpr bool kNeedOldItem = true;
    float *P;
    float *const *dst;  // per cache row: where its descent sum goes (peer or local address).  Bit 0 set (exclusive-row
                        // bypass): no other rank references the row this step, the address is the row itself in its
                        // owner's q and what is stored is the UPDATED ROW -- the same fmaf the owner's pass would do
    float alpha;
    int D4;
    __device__ __forceinline__ void apply(int tbl, size_t row, int e, float4 old, float4 d) const {
        if (tbl) {
            const uintptr_t a = reinterpret_cast<uintptr_t>(dst[row]);
            float4 *p = reinterpret_cast<float4 *>(a & ~(uintptr_t)1);
            if (a & 1)
                p[e] = make_float4(fmaf(alpha, d.x, old.x), fmaf(alpha, d.y, old.y), fmaf(alpha, d.z, old.z),
                                   fmaf(alpha, d.w, old.w));
            else
                p[e] = d;
        } else {
            st_row(P, row * D4 + e,
                   make_float4(fmaf(alpha, d.x, old.x), fmaf(alpha, d.y, old.y), fmaf(alpha, d.z, old.z),
                               fmaf(alpha, d.w, old.w)));
        }
    }
};

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// The id list every owner merges by: one thread per cache row => consecutive rows of one owner coalesce into full
// 128-byte peer stores.  Also tells every owner how many entries this rank pushes this step.
__global__ void k_shard_push_ids(const uint32_t *__restrict__ owner_off, int G, const uint32_t *__restrict__ uniq_gid,
                                 uint32_t i_per, int me, size_t cap, ShardPeers peers) {
    const uint32_t nuniq = owner_off[G];
    if (blockIdx.x == 0 && threadIdx.x < G)
        peers.recv_cnt[threadIdx.x][me] = owner_off[threadIdx.x + 1] - owner_off[threadIdx.x];
    for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < nuniq; c += gridDim.x * blockDim.x) {
        const uint32_t g = uniq_gid[c];
        const uint32_t o = g / i_per;
        peers.recv_ids[o][(size_t)me * cap + (c - owner_off[o])] = (int32_t)(g - o * i_per);
    }
}

// R rows in flight per warp: a peer load takes ~2000 cycles (NVLink + remote L2/DRAM), so bandwidth needs depth.
template <int V, int R>
__global__ void __launch_bounds__(256) k_shard_fetch(const float *const *__restrict__ src,
                                                      const uint8_t *__restrict__ multi,
                                                      const uint32_t *__restrict__ owner_off, int G,
                                                      float *__restrict__ cache, int D4, int ilv) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (uint32_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const uint32_t nwarps = (uint32_t)((gridDim.x * (size_t)blockDim.x) >> 5);
    const uint32_t nuniq = owner_off[G];
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;
    // groups of R cache rows (ascending = grouped by owner) are dealt round-robin over `ilv` ranges of the list, so the
    // loads in flight are spread over all owners (MainArgs::ilv has the reason)
    const int ngroups = (int)((nuniq + R - 1) / R);
    const uint32_t nraw = ilv > 1 ? (uint32_t)ilv * (uint32_t)((ngroups + ilv - 1) / ilv) : (uint32_t)ngroups;
    for (uint32_t raw = warp; raw < nraw; raw += nwarps) {
        const int grp = interleaved_chunk((int)raw, ngroups, ilv);
        if (grp < 0) continue;
        const uint32_t c0 = (uint32_t)grp * R;
        float4 r[R][V];
        bool take[R];  // rows referenced once are read by the main kernel straight from their owner
#pragma unroll
        for (int jj = 0; jj < R; ++jj) {
            const uint32_t c = c0 + jj;
            take[jj] = c < nuniq && multi[c];
            if (take[jj]) {
                const float *p = src[c];
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v]) r[jj][v] = ld_stream(p, lane + 32 * v);
            }
        }
#pragma unroll
        for (int jj = 0; jj < R; ++jj) {
            const uint32_t c = c0 + jj;
            if (take[jj]) {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v]) st_row(cache, (size_t)c * D4 + lane + 32 * v, r[jj][v]);
            }
        }
    }
}

// A rank without triples this step pushes nothing: tell every owner so.
__global__ void k_shard_push_none(int G, int me, ShardPeers peers) {
    if (threadIdx.x < G) peers.recv_cnt[threadIdx.x][me] = 0u;
}

// Exclusive-row bypass, owner side.  After every rank's id list has arrived (barrier), the owner marks which of its rows
// are referenced by ONE rank only this step: two bitmaps over the local rows (seen by >= 1 rank, by >= 2 ranks; a
// sender's list is duplicate-free, so a second hit is a second rank) ...
__global__ void k_owner_count(const int32_t *__restrict__ recv_ids, const uint32_t *__restrict__ recv_cnt, size_t cap,
                              uint32_t rows_local, uint32_t *__restrict__ seen, uint32_t *__restrict__ multi) {
    const int snd = blockIdx.y;
    uint32_t n = recv_cnt[snd];
    if (n > cap) n = (uint32_t)cap;
    const int32_t *ids = recv_ids + (size_t)snd * cap;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)ids[k];
        if (r >= rows_local) continue;
        mark_row(seen, multi, r);
    }
}

// ... and tells every sender, entry by entry, whether the row is its alone (1-byte peer stores into region `me` of the
// sender's excl array).  The sender then stores the updated row straight into the owner's q instead of pushing a sum
// the owner would have to read, add and write back.  What stays with the owner are the rows SHARED between ranks: every
// such row gets a SLOT (claimed once through a third bitmap) with one cell per sender, filled by k_owner_pairs, so that
// the owner's kernel can walk the shared rows directly; the shared entries are also listed per sender for the
// pass-per-sender variant (order inside a list is arbitrary and does not matter: a sender's entries name distinct rows).
__global__ void k_owner_classify(const int32_t *__restrict__ recv_ids, const uint32_t *__restrict__ recv_cnt, size_t cap,
                                 uint32_t rows_local, const uint32_t *__restrict__ multi, int me, ShardPeers peers,
                                 uint32_t *__restrict__ shared_idx, uint32_t *__restrict__ shared_cnt,
                                 uint32_t *__restrict__ claim, uint32_t *__restrict__ slot_of_row,
                                 uint32_t *__restrict__ slot_row, uint32_t *__restrict__ pairs, uint32_t *__restrict__ slot_n,
                                 uint32_t max_slots, int G, int *err) {
    const int snd = blockIdx.y;
    uint32_t n = recv_cnt[snd];
    if (n > cap) n = (uint32_t)cap;
    const int32_t *ids = recv_ids + (size_t)snd * cap;
    uint8_t *out = peers.excl[snd] + (size_t)me * cap;
    const int lane = threadIdx.x & 31;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t n_up = (n + 31u) & ~31u;  // whole warps iterate together (ballot below)
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_up; k += stride) {
        bool keep = false;
        if (k < n) {
            const uint32_t r = (uint32_t)ids[k];
            if (r >= rows_local) {  // cannot happen (senders park bad ids on row 0 and flag them); never index with it
                atomicOr(&err[0], 1);
                out[k] = 0;
            } else {
                const uint32_t bit = 1u << (r & 31);
                const bool excl = !(multi[r >> 5] & bit);
                out[k] = excl ? 1 : 0;
                keep = !excl;
                if (keep && !(atomicOr(&claim[r >> 5], bit) & bit)) {  // first entry of this row seen by the kernel
                    const uint32_t sl = atomicAdd(slot_n, 1u);
                    slot_of_row[r] = sl;
                    if (sl < max_slots) {
                        slot_row[sl] = r;
                        for (int sp = 0; sp < G; ++sp) pairs[(size_t)sl * G + sp] = 0xFFFFFFFFu;
                    }
                }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(&shared_cnt[snd], (uint32_t)__popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (keep) shared_idx[(size_t)snd * cap + base + __popc(m & ((1u << lane) - 1u))] = k;
        }
    }
}

// Every listed entry enters its row's slot: pairs[slot][sender] = entry index in the sender's region.
__global__ void k_owner_pairs(const int32_t *__restrict__ recv_ids, const uint32_t *__restrict__ shared_idx,
                              const uint32_t *__restrict__ shared_cnt, size_t cap, const uint32_t *__restrict__ slot_of_row,
                              uint32_t *__restrict__ pairs, uint32_t max_slots, int G) {
    const int snd = blockIdx.y;
    const uint32_t n = shared_cnt[snd];
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const uint32_t k = shared_idx[(size_t)snd * cap + t];
        const uint32_t sl = slot_of_row[(uint32_t)recv_ids[(size_t)snd * cap + k]];
        if (sl < max_slots) pairs[(size_t)sl * G + snd] = k;
    }
}

// Sender side, after the owners' verdicts have arrived (barrier): the destination of an exclusive cache row becomes
// the row itself in its owner's q, tagged in bit 0 (PushOpt::apply).
__global__ void k_shard_tag_dst(const uint32_t *__restrict__ owner_off, int G, const uint32_t *__restrict__ uniq_gid,
                                uint32_t i_per, size_t cap, int D, const uint8_t *__restrict__ excl, ShardPeers peers,
                                float **__restrict__ dst) {
    const uint32_t nuniq = owner_off[G];
    for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < nuniq; c += gridDim.x * blockDim.x) {
        const uint32_t g = uniq_gid[c];
        const uint32_t o = g / i_per;
        if (excl[(size_t)o * cap + (c - owner_off[o])])
            dst[c] = reinterpret_cast<float *>(reinterpret_cast<uintptr_t>(peers.q[o] + (size_t)(g - o * i_per) * D) | 1u);
    }
}

// Cross-GPU barrier on the stream: everything this rank wrote to peer memory in earlier kernels of the stream is
// complete (kernel boundary) and made visible system-wide before the arrival flag (release); the spin acquires the
// peers' arrivals.  Epochs only grow, so flags are never reset.  One rank per GPU: the waiting kernels run on different
// devices (never several of them on one GPU).
__global__ void k_shard_barrier(ShardPeers peers, int me, int G, uint32_t epoch, unsigned long long timeout_ns, int *err) {
    const int t = threadIdx.x;
    if (t >= G) return;
    __threadfence_system();
    st_release_sys(peers.flags[t] + me, epoch);
    const unsigned long long t0 = global_ns();
    while ((int32_t)(ld_acquire_sys(peers.flags[me] + t) - epoch) < 0) {
        if (global_ns() - t0 > timeout_ns) {
            atomicOr(&err[0], 16);
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

// Owner side.  Region s of recv_ids holds the ascending, duplicate-free local row ids sender s pushed sums for
// (recv_cnt[s] of them), recv_g the sums.  One lane per entry: it is the row's LEADER if no lower-ranked sender
// pushed the same row (binary searches); the warp then handles its leaders one at a time, adding the senders'
// sums in rank order and updating the row once.
template <int V>
__global__ void __launch_bounds__(256) k_owner_merge(float *__restrict__ Q, const float *__restrict__ recv_g,
                                                      const int32_t *__restrict__ recv_ids,
                                                      const uint32_t *__restrict__ recv_cnt, int G, size_t cap, int D4,
                                                      float alpha, uint32_t rows_local, int *err) {
    const unsigned FULL = 0xffffffffu;
    const uint32_t NONE = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (uint32_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const uint32_t nwarps = (uint32_t)((gridDim.x * (size_t)blockDim.x) >> 5);
    uint32_t cnt_l = (lane < G) ? recv_cnt[lane] : 0u;
    if (cnt_l > cap) {  // cannot happen (a sender has at most 2*maxB = cap distinct rows); never read out of bounds
        atomicOr(&err[0], 32);
        cnt_l = (uint32_t)cap;
    }
    uint32_t total = 0;
    for (int s = 0; s < G; ++s) total += (__shfl_sync(FULL, cnt_l, s) + 31u) >> 5;
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;

    for (uint32_t task = warp; task < total; task += nwarps) {
        int s = 0;
        uint32_t rem = task;
        while (true) {
            const uint32_t ch = (__shfl_sync(FULL, cnt_l, s) + 31u) >> 5;
            if (rem < ch) break;
            rem -= ch;
            ++s;
        }
        const uint32_t n_s = __shfl_sync(FULL, cnt_l, s);
        const uint32_t k = rem * 32u + lane;
        const bool valid = k < n_s;
        uint32_t r = valid ? (uint32_t)recv_ids[(size_t)s * cap + k] : NONE;
        bool leader = valid;
        if (valid && r >= rows_local) {
            atomicOr(&err[0], 1);
            leader = false;
        }
        uint32_t pos[DAISY_MAX_RANKS];
#pragma unroll
        for (int sp = 0; sp < DAISY_MAX_RANKS; ++sp) {
            pos[sp] = NONE;
            if (sp < G && sp != s) {  // warp-uniform
                const uint32_t n2 = __shfl_sync(FULL, cnt_l, sp);
                const int32_t *ids2 = recv_ids + (size_t)sp * cap;
                uint32_t lo = 0, hi = n2;
                while (__any_sync(FULL, lo < hi)) {
                    if (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if ((uint32_t)ids2[mid] < r) lo = mid + 1; else hi = mid;
                    }
                }
                const bool found = valid && lo < n2 && (uint32_t)ids2[lo] == r;
                if (found) {
                    if (sp < s) leader = false; else pos[sp] = lo;
                }
            }
        }
        unsigned todo = __ballot_sync(FULL, leader);
        while (todo) {
            const int b = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t row = __shfl_sync(FULL, r, b);
            float4 acc[V];
            const size_t own = ((size_t)s * cap + rem * 32u + b) * D4;
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] = act[v] ? ld_stream(recv_g, own + lane + 32 * v) : f4_zero();
#pragma unroll
            for (int sp = 0; sp < DAISY_MAX_RANKS; ++sp) {
                const uint32_t pp = __shfl_sync(FULL, pos[sp], b);
                if (pp != NONE) {  // warp-uniform; sp > s ascending = sender-rank order
                    const size_t at = ((size_t)sp * cap + pp) * D4;
#pragma unroll
                    for (int v = 0; v < V; ++v)
                        if (act[v]) acc[v] = f4_add(acc[v], ld_stream(recv_g, at + lane + 32 * v));
                }
            }
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v]) {
                    const size_t e = (size_t)row * D4 + lane + 32 * v;
                    const float4 old = ld_row(Q, e);
                    st_row(Q, e, make_float4(fmaf(alpha, acc[v].x, old.x), fmaf(alpha, acc[v].y, old.y),
                                             fmaf(alpha, acc[v].z, old.z), fmaf(alpha, acc[v].w, old.w)));
                }
        }
    }
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Arena layout (identical on every rank): a function of (dim, max_batch, world, item_num_global) only.
static void shard_layout(daisy_shard *sh, int dim, int64_t max_batch, int world, int64_t item_num_global) {
    sh->world = world;
    sh->I_global = item_num_global;
    sh->i_per = (item_num_global + world - 1) / world;
    sh->cap = 2 * max_batch;
    const size_t D = (size_t)dim, cap = (size_t)sh->cap, G = (size_t)world;
    size_t off = 0;
    sh->off_q = off;      off = align_up(off + (size_t)sh->i_per * D * sizeof(float), 256);
    sh->off_g = off;      off = align_up(off + G * cap * D * sizeof(float), 256);
    sh->off_ids = off;    off = align_up(off + G * cap * sizeof(int32_t), 256);
    sh->off_cnt = off;    off = align_up(off + DAISY_MAX_RANKS * sizeof(uint32_t), 256);
    sh->off_flags = off;  off = align_up(off + DAISY_MAX_RANKS * sizeof(uint32_t), 256);
    sh->off_excl = off;   off = align_up(off + G * cap, 256);
    sh->arena_bytes = off;
}

static void shard_set_peers(daisy_shard *sh, int r, char *base) {
    sh->peer_arena[r] = base;
    sh->peers.q[r] = (float *)(base + sh->off_q);
    sh->peers.recv_g[r] = (float *)(base + sh->off_g);
    sh->peers.recv_ids[r] = (int32_t *)(base + sh->off_ids);
    sh->peers.recv_cnt[r] = (uint32_t *)(base + sh->off_cnt);
    sh->peers.flags[r] = (uint32_t *)(base + sh->off_flags);
    sh->peers.excl[r] = (uint8_t *)(base + sh->off_excl);
}

static int shard_ready(daisy_ctx *h) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DAISY_REQUIRE(h->sh != nullptr, DAISY_EINVAL, "handle is not sharded: call daisy_shard_init first");
    DAISY_REQUIRE(h->sh->attached, DAISY_EINVAL, "peers are not attached: call daisy_shard_attach first");
    return DAISY_OK;
}

template <int V>
static void launch_fetch(daisy_ctx *h, const ShardSet &ss, cudaStream_t s) {
    daisy_shard *sh = h->sh;
    k_shard_fetch<V, 4><<<h->num_sms * 4, 256, 0, s>>>(ss.src, ss.multi, ss.owner_off, sh->world, sh->cache, h->D / 4, sh->ilv);
}

// Owner side, default: ONE PASS PER SENDER, in sender-rank order.  A sender's id list is duplicate-free, so the
// entries of one region touch distinct rows and a pass is a plain streaming read-modify-write (R entries in flight per
// warp); passes follow each other on the stream, which fixes the order in which a row shared by several senders
// receives their sums => deterministic, no membership searches at all.  (k_owner_merge, the single-pass variant that
// finds every row's senders by binary search, cost 0.57 ms at 8 ranks -- 7 x 17 dependent L2 loads per entry; it is
// kept behind DAISY_OWNER_MERGE=1.)
template <int V, int R>
__global__ void __launch_bounds__(256) k_owner_add(float *__restrict__ Q, const float *__restrict__ recv_g,
                                                    const int32_t *__restrict__ recv_ids,
                                                    const uint32_t *__restrict__ recv_cnt_s, size_t cap, int D4, float alpha,
                                                    uint32_t rows_local, int *err, const uint32_t *__restrict__ list,
                                                    const uint32_t *__restrict__ list_cnt) {
    // list != null (exclusive-row bypass live this step): an entry whose row no other rank referenced has already been
    // written, updated, by its sender -- only the listed entries (rows shared between ranks) are added here
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (uint32_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const uint32_t nwarps = (uint32_t)((gridDim.x * (size_t)blockDim.x) >> 5);
    uint32_t n = list ? *list_cnt : *recv_cnt_s;
    if (n > cap) {  // cannot happen (a sender has at most 2*maxB = cap distinct rows); never read out of bounds
        if (threadIdx.x == 0 && blockIdx.x == 0) atomicOr(&err[0], 32);
        n = (uint32_t)cap;
    }
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;
    for (uint32_t k0 = warp * R; k0 < n; k0 += nwarps * R) {
        float4 g[R][V], old[R][V];
        uint32_t row[R], ent[R];
#pragma unroll
        for (int jj = 0; jj < R; ++jj) {
            row[jj] = 0xFFFFFFFFu;
            ent[jj] = 0;
            if (k0 + jj < n) {
                ent[jj] = list ? list[k0 + jj] : k0 + jj;
                row[jj] = (uint32_t)recv_ids[ent[jj]];
                if (row[jj] >= rows_local) {
                    if (lane == 0) atomicOr(&err[0], 1);
                    row[jj] = 0xFFFFFFFFu;
                }
            }
        }
#pragma unroll
        for (int jj = 0; jj < R; ++jj)
            if (row[jj] != 0xFFFFFFFFu) {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v]) {
                        g[jj][v] = ld_stream(recv_g, (size_t)ent[jj] * D4 + lane + 32 * v);
                        old[jj][v] = ld_row(Q, (size_t)row[jj] * D4 + lane + 32 * v);
                    }
            }
#pragma unroll
        for (int jj = 0; jj < R; ++jj)
            if (row[jj] != 0xFFFFFFFFu) {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (act[v])
                        st_row(Q, (size_t)row[jj] * D4 + lane + 32 * v,
                               make_float4(fmaf(alpha, g[jj][v].x, old[jj][v].x), fmaf(alpha, g[jj][v].y, old[jj][v].y),
                                           fmaf(alpha, g[jj][v].z, old[jj][v].z), fmaf(alpha, g[jj][v].w, old[jj][v].w)));
            }
    }
}

// Owner side with the exclusive-row bypass live: what is left are the rows SHARED between ranks (a few per cent of the
// entries).  One launch instead of one pass per sender: a warp per shared row (its slot names the row and, per sender,
// the entry holding that sender's sum) adds the senders' sums IN RANK ORDER, one fmaf each -- exactly what the passes
// of k_owner_add do one after the other, so the result is bit-identical -- and updates the row once.  (A first version
// found a row's senders by binary searches in the id lists: 17 dependent loads per entry, slower than the passes at
// 2 GPUs -- profiles/r02p_bench_n2_*.)
template <int V>
__global__ void __launch_bounds__(256) k_owner_add_slots(float *__restrict__ Q, const float *__restrict__ recv_g,
                                                          const uint32_t *__restrict__ slot_row,
                                                          const uint32_t *__restrict__ pairs,
                                                          const uint32_t *__restrict__ slot_n, uint32_t max_slots, int G,
                                                          size_t cap, int D4, float alpha) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (uint32_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const uint32_t nwarps = (uint32_t)((gridDim.x * (size_t)blockDim.x) >> 5);
    uint32_t n = *slot_n;
    if (n > max_slots) n = max_slots;
    bool act[V];
#pragma unroll
    for (int v = 0; v < V; ++v) act[v] = (lane + 32 * v) < D4;
    for (uint32_t sl = warp; sl < n; sl += nwarps) {
        const uint32_t row = slot_row[sl];
        const uint32_t ent = lane < G ? pairs[(size_t)sl * G + lane] : 0xFFFFFFFFu;
        unsigned has = __ballot_sync(FULL, ent != 0xFFFFFFFFu);
        float4 q[V];
#pragma unroll
        for (int v = 0; v < V; ++v) q[v] = act[v] ? ld_row(Q, (size_t)row * D4 + lane + 32 * v) : f4_zero();
        while (has) {
            const int sp = __ffs(has) - 1;
            has &= has - 1;
            const size_t at = ((size_t)sp * cap + __shfl_sync(FULL, ent, sp)) * D4;
#pragma unroll
            for (int v = 0; v < V; ++v)
                if (act[v]) {
                    const float4 g = ld_stream(recv_g, at + lane + 32 * v);
                    q[v] = make_float4(fmaf(alpha, g.x, q[v].x), fmaf(alpha, g.y, q[v].y), fmaf(alpha, g.z, q[v].z),
                                       fmaf(alpha, g.w, q[v].w));
                }
        }
#pragma unroll
        for (int v = 0; v < V; ++v)
            if (act[v]) st_row(Q, (size_t)row * D4 + lane + 32 * v, q[v]);
    }
}

template <int V>
static void launch_merge(daisy_ctx *h, float alpha, cudaStream_t s) {
    daisy_shard *sh = h->sh;
    const int me = sh->rank;
    static const int single_pass = getenv("DAISY_OWNER_MERGE") && atoi(getenv("DAISY_OWNER_MERGE")) == 1;
    if (single_pass) {
        k_owner_merge<V><<<h->num_sms * 8, 256, 0, s>>>(sh->peers.q[me], sh->peers.recv_g[me], sh->peers.recv_ids[me],
                                                        sh->peers.recv_cnt[me], sh->world, (size_t)sh->cap, h->D / 4, alpha,
                                                        (uint32_t)h->I, h->err);
        return;
    }
    constexpr int R = V == 1 ? 4 : 2;
    const size_t cap = (size_t)sh->cap;
    static const int shared_passes = getenv("DAISY_OWNER_SHARED_PASSES") && atoi(getenv("DAISY_OWNER_SHARED_PASSES")) == 1;
    if (sh->classified && !shared_passes) {
        k_owner_add_slots<V><<<h->num_sms * 8, 256, 0, s>>>(sh->peers.q[me], sh->peers.recv_g[me], sh->slot_row, sh->pairs,
                                                            sh->slot_n, sh->max_slots, sh->world, cap, h->D / 4, alpha);
        return;
    }
    for (int snd = 0; snd < sh->world; ++snd) {
        k_owner_add<V, R><<<h->num_sms * 8, 256, 0, s>>>(sh->peers.q[me], sh->peers.recv_g[me] + (size_t)snd * cap * h->D,
                                                         sh->peers.recv_ids[me] + (size_t)snd * cap,
                                                         sh->peers.recv_cnt[me] + snd, cap, h->D / 4, alpha, (uint32_t)h->I,
                                                         h->err, sh->classified ? sh->shared_idx + (size_t)snd * cap : nullptr,
                                                         sh->shared_cnt + snd);
        if (snd + 1 < sh->world) h->launches++;
    }
}

// First part of a step: this rank's bookkeeping, and the id list / counts of what it will push stored into the owners.
// xs: the stream the id exchange runs on.  daisy_shard_step passes the handle's auxiliary stream so that the chain
// ids -> barrier -> verdicts -> barrier -> tagged destinations runs NEXT TO the fetch of the repeated rows (both only
// need the bookkeeping and the previous step); everything else passes xs = s.
static int shard_prepare(daisy_ctx *h, const int32_t *triples_dev, const int32_t *host_src, int64_t B, cudaStream_t s,
                         cudaStream_t xs) {
    daisy_shard *sh = h->sh;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    sh->prepared = 1;
    sh->prepared_B = B;
    sh->classified = 0;
    if (B == 0) {  // no triples here this step: the owners must see empty regions
        if (xs != s) {
            DAISY_CUDA(cudaEventRecord(sh->aux_ev[0], s));
            DAISY_CUDA(cudaStreamWaitEvent(xs, sh->aux_ev[0], 0));
        }
        k_shard_push_none<<<1, 32, 0, xs>>>(sh->world, sh->rank, sh->peers);
        DAISY_LAUNCH_CHECK(h);
        return DAISY_OK;
    }
    StepPlan &pl = *(StepPlan *)sh->plan;
    const bool prof = h->timing == 2;
    if (prof) {
        if (!sh->pev[0])
            for (int i = 0; i < 7; ++i) cudaEventCreate(&sh->pev[i]);
        cudaEventRecord(sh->pev[0], s);
    }
    int rc = book_phase(h, pl, triples_dev, B, (uint32_t)h->U, (uint32_t)sh->I_global, s, host_src,
                        host_src != nullptr || h->inputs_ready, sh);
    if (rc) return rc;
    if (prof) cudaEventRecord(sh->pev[1], s);
    sh->prepared_set = pl.set;
    const ShardSet &ss = sh->set[pl.set];
    if (xs != s) {  // s has just been ordered behind the bookkeeping (book_phase) and carries the previous step
        DAISY_CUDA(cudaEventRecord(sh->aux_ev[0], s));
        DAISY_CUDA(cudaStreamWaitEvent(xs, sh->aux_ev[0], 0));
    }
    k_shard_push_ids<<<h->num_sms * 2, 256, 0, xs>>>(ss.owner_off, sh->world, ss.uniq_gid, (uint32_t)sh->i_per, sh->rank,
                                                    (size_t)sh->cap, sh->peers);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

// Exclusive-row bypass, owner side (every rank's id list has arrived): which entries name a row no other rank references.
static int shard_classify(daisy_ctx *h, cudaStream_t s) {
    daisy_shard *sh = h->sh;
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    DAISY_CUDA(cudaMemsetAsync(sh->bm_seen, 0, sh->bm_words * sizeof(uint32_t), s));
    DAISY_CUDA(cudaMemsetAsync(sh->bm_multi, 0, sh->bm_words * sizeof(uint32_t), s));
    DAISY_CUDA(cudaMemsetAsync(sh->bm_claim, 0, sh->bm_words * sizeof(uint32_t), s));
    DAISY_CUDA(cudaMemsetAsync(sh->shared_cnt, 0, (DAISY_MAX_RANKS + 1) * sizeof(uint32_t), s));
    const dim3 grid((unsigned)(h->num_sms * 2), (unsigned)sh->world);
    const int me = sh->rank;
    k_owner_count<<<grid, 256, 0, s>>>(sh->peers.recv_ids[me], sh->peers.recv_cnt[me], (size_t)sh->cap, (uint32_t)h->I,
                                       sh->bm_seen, sh->bm_multi);
    DAISY_LAUNCH_CHECK(h);
    k_owner_classify<<<grid, 256, 0, s>>>(sh->peers.recv_ids[me], sh->peers.recv_cnt[me], (size_t)sh->cap, (uint32_t)h->I,
                                          sh->bm_multi, me, sh->peers, sh->shared_idx, sh->shared_cnt, sh->bm_claim,
                                          sh->slot_of_row, sh->slot_row, sh->pairs, sh->slot_n, sh->max_slots, sh->world, h->err);
    DAISY_LAUNCH_CHECK(h);
    k_owner_pairs<<<grid, 256, 0, s>>>(sh->peers.recv_ids[me], sh->shared_idx, sh->shared_cnt, (size_t)sh->cap,
                                       sh->slot_of_row, sh->pairs, sh->max_slots, sh->world);
    DAISY_LAUNCH_CHECK(h);
    h->launches += 4;
    sh->classified = 1;
    return DAISY_OK;
}

// Rest of the step on this rank: fetch of the repeated rows + the fused compute / push kernels.
static int shard_finish(daisy_ctx *h, float *P_local, float lr, float wd, double *loss_accum, cudaStream_t s,
                        cudaStream_t xs) {
    daisy_shard *sh = h->sh;
    const double shrink = 1.0 - (double)lr * (double)wd;
    DAISY_REQUIRE(shrink > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1: the L2 shrink factor is not positive", (double)lr * wd);
    DAISY_REQUIRE(sh->prepared, DAISY_EINVAL, "no prepared step");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    sh->prepared = 0;
    if (sh->prepared_B == 0) {  // the rank's rows still decay
        if (xs != s) {
            DAISY_CUDA(cudaEventRecord(sh->aux_ev[1], xs));
            DAISY_CUDA(cudaStreamWaitEvent(s, sh->aux_ev[1], 0));
        }
        h->scale *= shrink;
        return DAISY_OK;
    }
    const StepPlan &pl = *(const StepPlan *)sh->plan;
    const bool prof = h->timing == 2;
    const ShardSet &ss = sh->set[pl.set];
    const int D4 = h->D / 4;
    if (sh->classified) {
        k_shard_tag_dst<<<h->num_sms * 2, 256, 0, xs>>>(ss.owner_off, sh->world, ss.uniq_gid, (uint32_t)sh->i_per,
                                                        (size_t)sh->cap, h->D, sh->peers.excl[sh->rank], sh->peers, ss.dst);
        DAISY_LAUNCH_CHECK(h);
    }
    if (xs != s) DAISY_CUDA(cudaEventRecord(sh->aux_ev[1], xs));
    if (D4 <= 32) launch_fetch<1>(h, ss, s);
    else if (D4 <= 64) launch_fetch<2>(h, ss, s);
    else if (D4 <= 96) launch_fetch<3>(h, ss, s);
    else launch_fetch<4>(h, ss, s);
    DAISY_LAUNCH_CHECK(h);
    if (xs != s) DAISY_CUDA(cudaStreamWaitEvent(s, sh->aux_ev[1], 0));
    if (prof) cudaEventRecord(sh->pev[2], s);
    PushOpt opt;
    opt.P = P_local;
    opt.dst = ss.dst;
    opt.alpha = (float)((double)lr / shrink);
    opt.D4 = D4;
    int rc = table_phase<PushOpt>(h, pl, P_local, sh->cache, opt, (float)(h->scale * h->scale), loss_accum);
    if (rc) return rc;
    if (prof) cudaEventRecord(sh->pev[3], s);
    h->scale *= shrink;
    return DAISY_OK;
}

static int shard_apply(daisy_ctx *h, float lr, float wd, cudaStream_t s) {
    const double shrink = 1.0 - (double)lr * (double)wd;
    DAISY_REQUIRE(shrink > 0.0, DAISY_EINVAL, "lr*wd = %g >= 1", (double)lr * wd);
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    const float alpha = (float)((double)lr / shrink);
    const int D4 = h->D / 4;
    if (D4 <= 32) launch_merge<1>(h, alpha, s);
    else if (D4 <= 64) launch_merge<2>(h, alpha, s);
    else if (D4 <= 96) launch_merge<3>(h, alpha, s);
    else launch_merge<4>(h, alpha, s);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

static int shard_barrier(daisy_ctx *h, cudaStream_t s) {
    daisy_shard *sh = h->sh;
    if (sh->world == 1) return DAISY_OK;
    // ranks emulated in ONE process share a device and a stream: a barrier kernel of rank r would spin on flags that
    // only later launches of the same stream can set.  The caller orders the phases there (daisy_shard_compute /
    // daisy_shard_apply), so a barrier -- and with it daisy_shard_step -- is a usage error, reported at once.
    DAISY_REQUIRE(!sh->in_process, DAISY_EINVAL, "in-process sharding (daisy_shard_attach(.., in_process=1)) has no barrier: "
                  "drive daisy_shard_compute / daisy_shard_apply of all ranks in lockstep instead of daisy_shard_step");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    sh->epoch++;
    k_shard_barrier<<<1, 32, 0, s>>>(sh->peers, sh->rank, sh->world, sh->epoch, 20ull * 1000000000ull, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

}  // namespace

void daisy_shard_free(daisy_ctx *h) {
    daisy_shard *sh = h->sh;
    if (!sh) return;
    for (int i = 0; i < 7; ++i)
        if (sh->pev[i]) cudaEventDestroy(sh->pev[i]);
    for (int r = 0; r < sh->world; ++r)
        if (sh->ipc_opened[r] && sh->peer_arena[r]) cudaIpcCloseMemHandle(sh->peer_arena[r]);
    if (sh->bm_seen) cudaFree(sh->bm_seen);
    if (sh->bm_multi) cudaFree(sh->bm_multi);
    if (sh->shared_idx) cudaFree(sh->shared_idx);
    if (sh->shared_cnt) cudaFree(sh->shared_cnt);
    for (void *p : {(void *)sh->bm_claim, (void *)sh->slot_of_row, (void *)sh->slot_row, (void *)sh->pairs})
        if (p) cudaFree(p);
    if (sh->aux_stream) cudaStreamDestroy(sh->aux_stream);
    for (int i = 0; i < 2; ++i)
        if (sh->aux_ev[i]) cudaEventDestroy(sh->aux_ev[i]);
    if (sh->plan) delete (StepPlan *)sh->plan;
    for (int i = 0; i < DAISY_NSETS; ++i) {
        void *ptrs[] = {sh->set[i].uniq_gid, (void *)sh->set[i].src, (void *)sh->set[i].dst, sh->set[i].owner_off,
                        sh->set[i].multi, (void *)sh->set[i].jsrc, (void *)sh->set[i].isrc};
        for (void *p : ptrs)
            if (p) cudaFree(p);
    }
    if (sh->cidx) cudaFree(sh->cidx);
    if (sh->cache) cudaFree(sh->cache);
    if (sh->arena && sh->arena_owned) cudaFree(sh->arena);
    free(sh);
    h->sh = nullptr;
}

extern "C" int daisy_shard_schedule(int warp, int nchunks, int interleave, int *chunk) {
    DAISY_REQUIRE(chunk != nullptr && warp >= 0 && nchunks >= 0 && interleave >= 0, DAISY_EINVAL, "bad schedule query");
    *chunk = interleaved_chunk(warp, nchunks, interleave);
    return DAISY_OK;
}

extern "C" int daisy_shard_arena_size(int dim, int64_t max_batch, int world, int64_t item_num_global, int64_t *bytes) {
    DAISY_REQUIRE(bytes != nullptr, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(dim > 0 && dim % 4 == 0 && dim <= 512 && max_batch > 0 && world >= 1 && world <= DAISY_MAX_RANKS &&
                      item_num_global > 0, DAISY_EINVAL, "bad shape");
    daisy_shard tmp;
    memset(&tmp, 0, sizeof(tmp));
    shard_layout(&tmp, dim, max_batch, world, item_num_global);
    *bytes = (int64_t)tmp.arena_bytes;
    return DAISY_OK;
}

extern "C" int daisy_shard_init(daisy_handle_t h, int rank, int world, int64_t item_num_global, void *arena) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DAISY_REQUIRE(h->sh == nullptr, DAISY_EINVAL, "handle is already sharded");
    DAISY_REQUIRE(world >= 1 && world <= DAISY_MAX_RANKS && rank >= 0 && rank < world, DAISY_EINVAL,
                  "rank %d / world %d out of range (at most %d ranks)", rank, world, DAISY_MAX_RANKS);
    DAISY_REQUIRE(h->maxB > 0 && h->D % 4 == 0 && h->D <= 512, DAISY_EUNSUPPORTED,
                  "sharding needs a handle with max_batch > 0, dim %% 4 == 0, dim <= 512");
    DAISY_REQUIRE(item_num_global > 0 && item_num_global < 0x7ffffffeLL, DAISY_EINVAL, "bad global item count");
    DAISY_REQUIRE((uintptr_t)arena % 256 == 0, DAISY_EINVAL, "a caller-provided arena must be 256-byte aligned");
    const int64_t i_per = (item_num_global + world - 1) / world;
    int64_t lo = (int64_t)rank * i_per, hi = lo + i_per;
    if (lo > item_num_global) lo = item_num_global;
    if (hi > item_num_global) hi = item_num_global;
    DAISY_REQUIRE(h->I == (hi - lo > 0 ? hi - lo : 1), DAISY_EINVAL,
                  "handle was created with item_num %lld but rank %d of %d owns %lld of %lld items", (long long)h->I, rank,
                  world, (long long)(hi - lo), (long long)item_num_global);
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    daisy_shard *sh = (daisy_shard *)calloc(1, sizeof(daisy_shard));
    DAISY_REQUIRE(sh != nullptr, DAISY_ENOMEM, "host allocation failed");
    sh->rank = rank;
    shard_layout(sh, h->D, h->maxB, world, item_num_global);
    {   // schedule of the main kernel: chunks dealt round-robin over `world` ranges of the owner-grouped order
        const char *v = getenv("DAISY_SHARD_INTERLEAVE");
        sh->ilv = (v && *v) ? atoi(v) : world;
        if (sh->ilv < 0 || sh->ilv > 1024) sh->ilv = world;
    }
    const size_t D = (size_t)h->D, cap = (size_t)sh->cap;
    h->sh = sh;
    bool ok = true;
    if (arena) {  // caller-owned (e.g. a torch symmetric-memory buffer the peers have mapped)
        sh->arena = (char *)arena;
    } else {
        ok = cudaMalloc((void **)&sh->arena, sh->arena_bytes) == cudaSuccess;
        sh->arena_owned = ok ? 1 : 0;
    }
    ok = ok && cudaMalloc((void **)&sh->cidx, cap * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->cache, cap * D * sizeof(float)) == cudaSuccess;
    sh->bm_words = ((size_t)sh->i_per + 31) / 32 + 1;
    ok = ok && cudaMalloc((void **)&sh->bm_seen, sh->bm_words * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->bm_multi, sh->bm_words * sizeof(uint32_t)) == cudaSuccess;
    {
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        ok = ok && cudaStreamCreateWithPriority(&sh->aux_stream, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
        for (int i = 0; i < 2 && ok; ++i) ok = cudaEventCreateWithFlags(&sh->aux_ev[i], cudaEventDisableTiming) == cudaSuccess;
    }
    ok = ok && cudaMalloc((void **)&sh->shared_idx, (size_t)world * cap * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->shared_cnt, (DAISY_MAX_RANKS + 1) * sizeof(uint32_t)) == cudaSuccess;
    sh->slot_n = sh->shared_cnt ? sh->shared_cnt + DAISY_MAX_RANKS : nullptr;
    {   // a shared row is named by >= 2 senders: at most half of all entries, and at most every local row
        const size_t half = (size_t)world * cap / 2 + 1, rows = (size_t)sh->i_per + 1;
        sh->max_slots = (uint32_t)(half < rows ? half : rows);
    }
    ok = ok && cudaMalloc((void **)&sh->bm_claim, sh->bm_words * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->slot_of_row, ((size_t)sh->i_per + 1) * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->slot_row, (size_t)sh->max_slots * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&sh->pairs, (size_t)sh->max_slots * world * sizeof(uint32_t)) == cudaSuccess;
    sh->plan = new StepPlan();
    {   // exclusive-row bypass (on by default; the single-pass owner merge does not know about it)
        const char *v = getenv("DAISY_SHARD_BYPASS");
        const char *m = getenv("DAISY_OWNER_MERGE");
        sh->bypass = ((v && *v) ? atoi(v) != 0 : 1) && !(m && atoi(m) == 1);
    }
    for (int i = 0; i < DAISY_NSETS && ok; ++i) {
        ok = ok && cudaMalloc((void **)&sh->set[i].uniq_gid, cap * sizeof(uint32_t)) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].src, cap * sizeof(float *)) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].dst, cap * sizeof(float *)) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].owner_off, (DAISY_MAX_RANKS + 1) * sizeof(uint32_t)) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].multi, cap) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].jsrc, (size_t)h->maxB * sizeof(float *)) == cudaSuccess;
        ok = ok && cudaMalloc((void **)&sh->set[i].isrc, (size_t)h->maxB * sizeof(float *)) == cudaSuccess;
    }
    if (!ok) {
        cudaGetLastError();
        daisy_set_error("sharding workspace allocation failed (arena of %zu bytes)", sh->arena_bytes);
        daisy_shard_free(h);
        return DAISY_ENOMEM;
    }
    // counts, flags and the tail of the arena start at zero; q is filled by the caller
    DAISY_CUDA(cudaMemset(sh->arena + sh->off_cnt, 0, sh->arena_bytes - sh->off_cnt));
    DAISY_CUDA(cudaDeviceSynchronize());
    shard_set_peers(sh, rank, sh->arena);
    if (world == 1) sh->attached = 1;
    return DAISY_OK;
}

extern "C" int daisy_shard_arena(daisy_handle_t h, void **arena, float **q_local, int64_t *arena_bytes) {
    DAISY_REQUIRE(h && h->sh, DAISY_EINVAL, "handle is not sharded");
    if (arena) *arena = h->sh->arena;
    if (q_local) *q_local = (float *)(h->sh->arena + h->sh->off_q);
    if (arena_bytes) *arena_bytes = (int64_t)h->sh->arena_bytes;
    return DAISY_OK;
}

extern "C" int daisy_shard_ipc_handle(daisy_handle_t h, void *out64) {
    DAISY_REQUIRE(h && h->sh && out64, DAISY_EINVAL, "null argument or handle not sharded");
    DAISY_REQUIRE(h->sh->arena_owned, DAISY_EINVAL, "the arena is caller-owned: the caller maps it into the peers");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    DeviceGuard g(h->device);
    cudaIpcMemHandle_t m;
    DAISY_CUDA(cudaIpcGetMemHandle(&m, h->sh->arena));
    memcpy(out64, &m, 64);
    return DAISY_OK;
}

extern "C" int daisy_shard_attach(daisy_handle_t h, const void *ipc_handles, void *const *arena_ptrs, int in_process) {
    DAISY_REQUIRE(h && h->sh, DAISY_EINVAL, "handle is not sharded");
    DAISY_REQUIRE((ipc_handles != nullptr) != (arena_ptrs != nullptr) || h->sh->world == 1, DAISY_EINVAL,
                  "pass either the ranks' IPC handles or (same process) their arena pointers");
    daisy_shard *sh = h->sh;
    DAISY_REQUIRE(!sh->attached || sh->world == 1, DAISY_EINVAL, "peers are already attached");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    for (int r = 0; r < sh->world; ++r) {
        if (r == sh->rank) continue;
        if (arena_ptrs) {
            DAISY_REQUIRE(arena_ptrs[r] != nullptr, DAISY_EINVAL, "null arena pointer for rank %d", r);
            shard_set_peers(sh, r, (char *)arena_ptrs[r]);
        } else {
            cudaIpcMemHandle_t m;
            memcpy(&m, (const char *)ipc_handles + 64 * (size_t)r, 64);
            void *p = nullptr;
            DAISY_CUDA(cudaIpcOpenMemHandle(&p, m, cudaIpcMemLazyEnablePeerAccess));
            sh->ipc_opened[r] = 1;
            shard_set_peers(sh, r, (char *)p);
        }
    }
    sh->in_process = (arena_ptrs && in_process) ? 1 : 0;
    sh->attached = 1;
    return DAISY_OK;
}

extern "C" int daisy_shard_compute(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B, float lr,
                                   float wd, double *loss_accum, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    rc = check_step_args(h, P_local, h->sh->cache, triples, B);
    if (rc) return rc;
    if (!h->sh->prepared) {  // one-call form: no classification => every sum goes through the owner's pass
        rc = shard_prepare(h, triples, nullptr, B, (cudaStream_t)stream, (cudaStream_t)stream);
        if (rc) return rc;
    } else {
        DAISY_REQUIRE(B == h->sh->prepared_B, DAISY_EINVAL, "daisy_shard_compute: %lld triples, but %lld were prepared",
                      (long long)B, (long long)h->sh->prepared_B);
    }
    return shard_finish(h, P_local, lr, wd, loss_accum, (cudaStream_t)stream, (cudaStream_t)stream);
}

extern "C" int daisy_shard_prepare(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B,
                                   daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    rc = check_step_args(h, P_local, h->sh->cache, triples, B);
    if (rc) return rc;
    DAISY_REQUIRE(!h->sh->prepared, DAISY_EINVAL, "a prepared step is pending: call daisy_shard_compute first");
    return shard_prepare(h, triples, nullptr, B, (cudaStream_t)stream, (cudaStream_t)stream);
}

extern "C" int daisy_shard_classify(daisy_handle_t h, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    DAISY_REQUIRE(h->sh->prepared, DAISY_EINVAL, "daisy_shard_classify follows daisy_shard_prepare of every rank");
    if (!h->sh->bypass) return DAISY_OK;
    return shard_classify(h, (cudaStream_t)stream);
}

extern "C" int daisy_shard_apply(daisy_handle_t h, float lr, float wd, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    return shard_apply(h, lr, wd, (cudaStream_t)stream);
}

extern "C" int daisy_shard_barrier(daisy_handle_t h, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    return shard_barrier(h, (cudaStream_t)stream);
}

static int shard_step_impl(daisy_handle_t h, float *P_local, const int32_t *triples_dev, const int32_t *host_src,
                           int64_t B, float lr, float wd, double *loss_accum, daisy_stream_t stream) {
    cudaStream_t s = (cudaStream_t)stream;
    daisy_shard *sh = h->sh;
    const bool prof = h->timing == 2 && B > 0;
    const bool live = sh->bypass && sh->world > 1;
    cudaStream_t xs = (live && sh->aux_stream && h->timing != 2) ? sh->aux_stream : s;
    int rc = shard_prepare(h, triples_dev, host_src, B, s, xs);
    if (!rc && live) {  // ids are in the owners' memory -> verdicts are in the senders' memory
        rc = shard_barrier(h, xs);
        if (!rc) rc = shard_classify(h, xs);
        if (!rc) rc = shard_barrier(h, xs);
    }
    if (!rc) rc = shard_finish(h, P_local, lr, wd, loss_accum, s, xs);
    if (!rc) rc = shard_barrier(h, s);
    if (!rc && prof) cudaEventRecord(sh->pev[4], s);
    if (!rc) rc = shard_apply(h, lr, wd, s);
    if (!rc && prof) cudaEventRecord(sh->pev[5], s);
    if (!rc) rc = shard_barrier(h, s);
    if (!rc && prof) {
        cudaEventRecord(sh->pev[6], s);
        cudaEventSynchronize(sh->pev[6]);
        for (int i = 0; i < 6; ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, sh->pev[i], sh->pev[i + 1]);
            sh->pms[i] += ms;
        }
        sh->psteps++;
    }
    if (!rc && h->scale < 1e-4) rc = daisy_shard_materialize(h, P_local, stream);  // same step on every rank
    return rc;
}

extern "C" int daisy_shard_step(daisy_handle_t h, float *P_local, const int32_t *triples, int64_t B, float lr, float wd,
                                double *loss_accum, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    rc = check_step_args(h, P_local, h->sh->cache, triples, B);
    if (rc) return rc;
    return shard_step_impl(h, P_local, triples, nullptr, B, lr, wd, loss_accum, stream);
}

extern "C" int daisy_shard_step_host(daisy_handle_t h, float *P_local, const int32_t *triples_host, int64_t B, float lr,
                                     float wd, double *loss_accum, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    rc = check_step_args(h, P_local, h->sh->cache, triples_host, B);
    if (rc) return rc;
    int32_t *dst = h->triples + (size_t)h->book_idx * 3 * (size_t)h->maxB;
    return shard_step_impl(h, P_local, dst, triples_host, B, lr, wd, loss_accum, stream);
}

extern "C" int daisy_shard_materialize(daisy_handle_t h, float *P_local, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    DAISY_REQUIRE(P_local != nullptr, DAISY_EINVAL, "null argument");
    // peers fetch rows of this rank's q: the in-place rescale must not overlap their next fetch
    rc = daisy_materialize(h, P_local, h->sh->peers.q[h->sh->rank], stream);
    if (!rc && !h->sh->in_process)
        rc = shard_barrier(h, (cudaStream_t)stream);
    return rc;
}

extern "C" int daisy_shard_last_counts(daisy_handle_t h, uint32_t *owner_off_out, daisy_stream_t stream) {
    int rc = shard_ready(h);
    if (rc) return rc;
    DAISY_REQUIRE(owner_off_out != nullptr, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    DAISY_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    DAISY_CUDA(cudaStreamSynchronize(h->side_stream));
    const ShardSet &ss = h->sh->set[(h->book_idx + DAISY_NSETS - 1) % DAISY_NSETS];  // the set the most recent step used
    DAISY_CUDA(cudaMemcpy(owner_off_out, ss.owner_off, (h->sh->world + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return DAISY_OK;
}

extern "C" int daisy_shard_phase_ms(daisy_handle_t h, double *avg_ms6, int64_t *steps) {
    DAISY_REQUIRE(h && h->sh && avg_ms6 && steps, DAISY_EINVAL, "null argument or handle not sharded");
    for (int i = 0; i < 6; ++i) avg_ms6[i] = h->sh->psteps ? h->sh->pms[i] / (double)h->sh->psteps : 0.0;
    *steps = h->sh->psteps;
    for (int i = 0; i < 6; ++i) h->sh->pms[i] = 0.0;
    h->sh->psteps = 0;
    return DAISY_OK;
}

// Diagnostic / building block: dst[c] = src[idx[c]] for rows of h->D floats; src may be a peer address.
namespace {
template <int V, int R>
__global__ void __launch_bounds__(256) k_gather_rows(const float *__restrict__ src, const int32_t *__restrict__ idx,
                                                      int n, float *__restrict__ dst, int D4) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (uint32_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const uint32_t nwarps = (uint32_t)((gridDim.x * (size_t)blockDim.x) >> 5);
    for (uint32_t c0 = warp * R; c0 < (uint32_t)n; c0 += nwarps * R) {
        float4 r[R][V];
#pragma unroll
        for (int jj = 0; jj < R; ++jj)
            if (c0 + jj < (uint32_t)n) {
                const size_t row = (size_t)idx[c0 + jj];
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (lane + 32 * v < D4) r[jj][v] = ld_stream(src, row * D4 + lane + 32 * v);
            }
#pragma unroll
        for (int jj = 0; jj < R; ++jj)
            if (c0 + jj < (uint32_t)n) {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (lane + 32 * v < D4) st_row(dst, (size_t)(c0 + jj) * D4 + lane + 32 * v, r[jj][v]);
            }
    }
}
}  // namespace

extern "C" int daisy_gather_rows(daisy_handle_t h, const float *src, const int32_t *idx, int64_t n, float *dst,
                                 daisy_stream_t stream) {
    DAISY_REQUIRE(h && src && idx && dst, DAISY_EINVAL, "null argument");
    DAISY_REQUIRE(h->D % 4 == 0 && h->D <= 512 && n >= 0 && n < (1LL << 31), DAISY_EUNSUPPORTED, "unsupported shape");
    if (n == 0) return DAISY_OK;
    DeviceGuard g(h->device);
    const int D4 = h->D / 4;
    cudaStream_t s = (cudaStream_t)stream;
    if (D4 <= 32) k_gather_rows<1, 4><<<h->num_sms * 4, 256, 0, s>>>(src, idx, (int)n, dst, D4);
    else if (D4 <= 64) k_gather_rows<2, 4><<<h->num_sms * 4, 256, 0, s>>>(src, idx, (int)n, dst, D4);
    else if (D4 <= 96) k_gather_rows<3, 2><<<h->num_sms * 4, 256, 0, s>>>(src, idx, (int)n, dst, D4);
    else k_gather_rows<4, 2><<<h->num_sms * 4, 256, 0, s>>>(src, idx, (int)n, dst, D4);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

extern "C" int daisy_shard_peer_q(daisy_handle_t h, int rank, float **q) {
    int rc = shard_ready(h);
    if (rc) return rc;
    DAISY_REQUIRE(q && rank >= 0 && rank < h->sh->world, DAISY_EINVAL, "bad rank");
    *q = h->sh->peers.q[rank];
    return DAISY_OK;
}
