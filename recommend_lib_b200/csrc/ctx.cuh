// Shared context, error plumbing and device helpers for libdaisy_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/daisy_b200.h"

#define DAISY_DIRECT 0xFFFFFFFFu    // slot value: "this row has a single contribution -> update it in place"
#define DAISY_NOT_HEAD 0xFFFFFFFEu  // positive-item slot of a sorted triple that continues the run of its predecessor
#define DAISY_MAX_RANKS 16          // ranks of a row-sharded model (one node)
#define DAISY_SLICE 64     // contributions per level-1 slice of a very hot row
#define DAISY_TRACE_STEPS 48
#define DAISY_SMALL_CAP 8192  // largest batch of the small-batch path: 2B item refs are sorted by ONE thread block
// Bookkeeping sets (sorted triples, sorted ref keys, slots) in flight.  With 2, the bookkeeping of step n+1 can only start
// once the table kernels of step n-1 are done -- i.e. together with the kernels of step n -- and, sharing the device with
// them, its 0.33 ms stretch to the whole 0.66 ms period: every step's kernels then wait for their own bookkeeping
// (profiles/r02e_bench_trace.json).  A third set lets the side stream run a full step ahead.
#define DAISY_NSETS 3
#define DAISY_EVPOOL 2048  // main-kernel event pairs kept between two daisy_main_kernel_ms() calls

// Phases of one BPR step, in launch order (daisy_last_step_phases).
enum {
    PH_PREP = 0,   // validate ids, emit (pos-item key, triple id)
    PH_SORT_I,     // radix sort triples by positive item
    PH_REFS,       // gather triples into sorted order, emit user refs and item refs (negatives + run heads)
    PH_SORT_U,     // radix sort user refs by row
    PH_SORT_Q,     // radix sort item refs by row
    PH_SLOTS,      // singleton / staged classification, slot scatter
    PH_MAIN,       // fused gather + score + sigmoid coefficient + in-place update / staging   (dominant)
    PH_SEG_U,      // segmented reduce + update of repeated user rows
    PH_SEG_Q,      // segmented reduce + update of repeated item rows
    PH_HEAVY,      // block-per-row reduce of very hot rows
    PH_LOSS,       // deterministic loss reduction
    PH_COUNT
};

struct BookSet {
    int32_t *st;                    // [maxB,3]  triples in positive-item order
    uint32_t *ukey_s, *qkey_s;      // [maxB], [2*maxB]  sorted user / item ref keys (rows)
    uint32_t *uslot, *jslot, *islot;  // [maxB]  per sorted triple: DAISY_DIRECT or staging slot
    uint32_t *longs;                // rows too long for one warp (k_seg_all): [0] = #rows, [1] = #slices, then 5 words per
                                    // row (table, row, first sorted position, length, first slice), like `heavy`
    uint32_t *counts;               // [2] staged user refs, staged item refs: the lengths of ukey_s / qkey_s when the
                                    // bookkeeping sorted only the refs of repeated rows (step_kernels.cuh: book_kernels)
    cudaEvent_t ready, freed, copied;  // bookkeeping done / table kernels done / host triples landed (copy stream)
};

// ---- row-sharded tables over peer memory (shard.cu) ----------------------------------------------------------------
// Every rank allocates one ARENA (a single cudaMalloc, exported through CUDA IPC) laid out identically on all ranks:
//   q        [i_per, D]      fp32   this rank's block of item rows
//   recv_g   [G][cap][D]     fp32   descent sums pushed by rank s for rows this rank owns (region s)
//   recv_ids [G][cap]        int32  the LOCAL row ids those sums belong to (ascending, duplicate-free per sender)
//   recv_cnt [G]             uint32 how many entries sender s pushed this step
//   flags    [G]             uint32 barrier arrivals (epoch numbers), written by the peers
//   excl     [G][cap]        uint8  written by owner o into region o: 1 = the row of this rank's k-th entry for owner o is
//                                   referenced by no other rank this step (exclusive-row bypass, shard.cu)
struct ShardPeers {  // the same regions of every rank's arena, as mapped into THIS process; passed to kernels by value
    float *q[DAISY_MAX_RANKS];
    float *recv_g[DAISY_MAX_RANKS];
    int32_t *recv_ids[DAISY_MAX_RANKS];
    uint32_t *recv_cnt[DAISY_MAX_RANKS];
    uint32_t *flags[DAISY_MAX_RANKS];
    uint8_t *excl[DAISY_MAX_RANKS];
};

struct ShardSet {         // per bookkeeping set (double-buffered like BookSet)
    uint32_t *uniq_gid;   // [2*maxB]  global id of cache row c (ascending => grouped by owner block)
    const float **src;    // [2*maxB]  where cache row c lives in its owner's q (a peer or local address)
    float **dst;          // [2*maxB]  where this rank's descent sum of cache row c goes in its owner's recv_g
    uint32_t *owner_off;  // [G+1]     first cache row owned by rank o; [G] = number of cache rows
    uint8_t *multi;       // [2*maxB]  1: cache row c is referenced more than once in the batch => fetched into the cache
    const float **jsrc;   // [maxB]    per sorted triple: where its negative-item row is read from
    const float **isrc;   // [maxB]    per sorted triple that heads a positive-item run: where that row is read from
};

struct daisy_shard {
    int rank, world;
    int64_t I_global, i_per, cap;  // cap = entries per sender region = 2 * maxB (a batch references at most 2B item rows)
    char *arena;
    int arena_owned;  // 1: cudaMalloc'ed by daisy_shard_init (legacy CUDA IPC export), 0: provided by the caller
    size_t arena_bytes, off_q, off_g, off_ids, off_cnt, off_flags, off_excl;
    char *peer_arena[DAISY_MAX_RANKS];
    int ipc_opened[DAISY_MAX_RANKS];
    int attached;
    int in_process;  // peers live in this process (lockstep emulation): the caller orders the phases, no barrier kernels
    ShardPeers peers;
    ShardSet set[DAISY_NSETS];
    uint32_t *cidx;   // [2*maxB] scan scratch (bookkeeping stream only)
    float *cache;     // [2*maxB, D] fetched pre-step item rows of the current batch
    uint32_t epoch;   // barrier epoch (same sequence on every rank)
    // exclusive-row bypass: owner-side bitmaps over the local item rows (referenced by >= 1 / >= 2 ranks this step)
    uint32_t *bm_seen, *bm_multi;
    cudaStream_t aux_stream;  // daisy_shard_step: the id exchange runs here, next to the fetch on the caller's stream
    cudaEvent_t aux_ev[2];
    uint32_t *shared_idx, *shared_cnt;  // [G][cap], [G]: per sender, the entries whose row is shared between ranks
    // one SLOT per shared row: slot_of_row [i_per], slot_row [max_slots], pairs [max_slots][G] = the entry of every sender
    // naming the row (or 0xFFFFFFFF), slot_n = slots claimed this step (lives behind shared_cnt), bm_claim = claim bitmap
    uint32_t *bm_claim, *slot_of_row, *slot_row, *pairs, *slot_n;
    uint32_t max_slots;
    size_t bm_words;
    int bypass;       // DAISY_SHARD_BYPASS (default 1)
    int classified;   // this step's entries have been classified (daisy_shard_classify ran): bypass is live
    int prepared;     // daisy_shard_prepare ran for the step daisy_shard_compute is about to finish
    int prepared_set; // ... into this bookkeeping set
    int64_t prepared_B;
    void *plan;       // StepPlan of the prepared step (step_kernels.cuh), owned by shard.cu
    int ilv;          // chunk interleave of the main kernel = world (MainArgs::ilv)
    // phase profile (daisy_set_timing(h, 2)): bookkeeping, fetch, compute+push, barrier, apply, barrier
    cudaEvent_t pev[7];
    double pms[6];
    int64_t psteps;
};

// A captured bookkeeping chain (step_kernels.cuh: book_phase) of one bookkeeping set at one batch size.
struct BookGraph {
    cudaGraphExec_t exec;
    int set, B, launches;
    uint32_t U, I;
};
#define DAISY_MAX_BGRAPH 9

struct daisy_ctx {
    int device;
    int num_sms;
    int64_t U, I, maxB;
    int D;
    unsigned flags;
    double scale;  // lazy L2 decay factor c: true tables = c * stored tables

    // --- workspace (device) ---
    int32_t *triples;       // [DAISY_NSETS][maxB,3]  H2D landing zones of daisy_bpr_step_host (one per bookkeeping set)
    // Bookkeeping products the table-touching kernels read; double-buffered so that the bookkeeping of step n+1
    // (side stream) overlaps the kernels of step n (caller's stream).
    BookSet book[DAISY_NSETS];
    int book_idx;
    cudaStream_t side_stream;
    cudaStream_t copy_stream;  // H2D of *_step_host triples when pipelined (created when max_batch > 0)
    cudaEvent_t ev_call;
    int pipeline;           // 1: bookkeeping on the side stream (default), 0: everything on the caller's stream
    int inputs_ready;       // 1: device triples passed to daisy_bpr_step are complete at call time (no stream dependency)
    // bookkeeping scratch, used on the bookkeeping stream only
    uint32_t *key_in, *val_in, *val_out;    // [3*maxB] item refs (negatives + run heads) [2*maxB]: unsorted keys/values, sorted
                                            // values; the merged sort (step_kernels.cuh) appends the user refs [maxB]
    uint32_t *key_out;                      // [3*maxB] merged sort: sorted keys before k_slots_dup splits them
    // merged sort of the refs of repeated rows (book_kernels): DsortState (ref_sort.cuh), the seen / dup bitmaps over
    // ref_rows rows (user row u is bit I + u), the sort's look-back words for 3*maxB refs
    uint32_t *ref_ws;
    int64_t ref_rows;
    uint32_t *ukey_in, *uval_in, *uval_out; // [maxB]   user refs
    uint32_t *ikey_in, *ikey_out, *ival_in, *ival_out;  // [maxB]   (positive item, triple id), unsorted / sorted
    void *cub_tmp;
    size_t cub_tmp_bytes;
    // staging, used on the caller's stream only
    float *stageU;          // [maxB, D]   staged user-row gradient contributions (by sorted user-ref position)
    float *stageQ;          // [2*maxB, D] staged item-row contributions (by sorted item-ref position)
    float *stage2;          // [slice_cap, D] level-1 partial sums of very hot rows
    float *loss_part;       // [maxB] per-warp loss partials
    int heavy_cap, slice_cap, longs_cap;
    uint32_t *ticket;       // [longs_cap] finished-slice counters of k_seg_all's long rows (zero between steps)
    int *err;               // [2]: flag, first bad position
    int *err_host;          // pinned mirror
    // sharded step: row count of the fetched-row cache standing in for the item table (0 = use I)
    int64_t item_rows_override;
    daisy_shard *sh;        // peer-memory sharding state (daisy_shard_init), else null
    // owner-side apply scratch (grown on demand by daisy_owner_apply)
    uint32_t *own_key, *own_key_s, *own_val, *own_val_s;
    void *own_tmp;
    size_t own_tmp_bytes;
    int64_t own_cap;
    // full-catalogue top-K workspace (grown on demand by daisy_topk_full)
    float *scores;          // [tile_users, item_num] score tile
    size_t scores_cap;      // floats
    // what the last daisy_topk_full call did (daisy_topk_full_path): DAISY_TOPK_PATH_*, users whose top K the filter
    // produced, users the exact fallback redid
    int topk_path;
    int64_t topk_filtered, topk_redone;

    // tuning (env overridable, see api.cu)
    int chunk;       // max positive-item run length handled by one warp in the main kernel (0 = auto)
    int heavy_len;   // segments longer than this go to the block-per-row kernel
    int main_stages; // > 0: TMA-pipelined main kernel with this many stages (triples in flight) per warp; 0: register prefetch
    int pairs_mode;  // set by csrc/gmf.cu around book_phase: the batch holds (user, item, label) samples
    float *gradP, *gradQ;  // [U, D], [I, D] dense gradient buffers of the GMF step (allocated on first use, kept zero between steps)
    float *wpart;    // [maxB, D + 1] per-sample contributions to the predict layer's gradient (GMF step)
    int merged_sort; // general path: ONE radix sort for user + item refs: 1 always, 0 never, -1 (default) when it costs no extra passes
    int small_max;   // batches up to this many triples take the 3-launch small-batch path (0 = never; <= DAISY_SMALL_CAP)
    int64_t mid_max; // ... and up to this many the same path with k_mid_book (0 = never; <= mid_cap)
    int64_t mid_cap; // min(maxB, 131072): what mid_buf is sized for
    uint32_t *mid_buf;  // [4][3 * mid_cap] k_mid_book's two (key, value) scratch buffers

    // --- CUDA-graph replay of the general bookkeeping chain for mid-size batches ---
    int64_t graph_max_b;     // batches up to this size replay a captured graph (0 = never; DAISY_GRAPH_MAX_B)
    BookGraph bgraph[DAISY_MAX_BGRAPH];
    int n_bgraph, bgraph_next;

    // stream-ordered scratch of the calls that size their workspace per call (sampler, full-catalogue top-K, funk-SVD,
    // SVD++): a PRIVATE memory pool of this handle, created on first use, that keeps freed blocks cached between calls
    // (release threshold = max) -- the device's default pool, which the rest of the process shares, is left alone
    cudaMemPool_t pool;
    int pool_state;  // 0 not created, 1 ready, -1 creation failed (cudaMallocAsync from the default pool, untuned)

    // --- instrumentation ---
    cudaEvent_t tc_ev[3];             // timing != 0: around k_filter_tc and k_rescore of the last daisy_tc_filter call
    int tc_ev_pending;
    double tc_filter_ms, tc_rescore_ms;
    int64_t tc_count;
    int64_t launches;
    int timing;                       // 0 off, 1 main kernel only (asynchronous event pool), 2 every phase (syncs per step)
    cudaEvent_t ev[PH_COUNT + 1];     // timing == 2
    double phase_ms_sum[PH_COUNT];
    int64_t timed_steps;
    int ev_pending;
    cudaStream_t ev_stream;
    cudaEvent_t evpool[2 * DAISY_EVPOOL];  // timing == 1
    int pool_used;
    double main_ms_sum;
    int64_t main_count;
    // optional timeline of the first DAISY_TRACE_STEPS steps (DAISY_TRACE=1): bookkeeping begin/end on the
    // bookkeeping stream, table kernels begin/end on the caller's stream
    int trace, tr_n;
    cudaEvent_t tr_ev[4 * DAISY_TRACE_STEPS];
};

void daisy_set_error(const char *fmt, ...);
void daisy_shard_free(daisy_ctx *h);  // shard.cu

#define DAISY_CUDA(call)                                                                     \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            daisy_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DAISY_ECUDA;                                                              \
        }                                                                                    \
    } while (0)

#define DAISY_REQUIRE(cond, code, ...)      \
    do {                                    \
        if (!(cond)) {                      \
            daisy_set_error(__VA_ARGS__);   \
            return (code);                  \
        }                                   \
    } while (0)

#define DAISY_LAUNCH_CHECK(h)                                                                \
    do {                                                                                     \
        (h)->launches++;                                                                     \
        cudaError_t e__ = cudaGetLastError();                                                \
        if (e__ != cudaSuccess) {                                                            \
            daisy_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
            return DAISY_ECUDA;                                                              \
        }                                                                                    \
    } while (0)

static inline int daisy_ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Stream-ordered allocation from the handle's private pool (see daisy_ctx::pool); freed with cudaFreeAsync.
static inline cudaError_t daisy_scratch_alloc(daisy_ctx *h, void **p, size_t bytes, cudaStream_t s) {
    if (h->pool_state == 0) {
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = h->device;
        if (cudaMemPoolCreate(&h->pool, &props) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(h->pool, cudaMemPoolAttrReleaseThreshold, &keep);
            h->pool_state = 1;
        } else {
            (void)cudaGetLastError();
            h->pool_state = -1;
        }
    }
    if (h->pool_state == 1) return cudaMallocFromPoolAsync(p, bytes ? bytes : 1, h->pool, s);
    return cudaMallocAsync(p, bytes ? bytes : 1, s);
}

// RAII-less device guard: the handle is bound to one device.
struct DeviceGuard {
    int prev;
    bool ok;
    explicit DeviceGuard(int dev) : prev(-1), ok(true) {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && prev >= 0 && cur != prev) cudaSetDevice(prev);
    }
};

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// 128-bit row-slice accessors.  Table rows are re-used across triples (hot items) so they take the normal
// cached path; staging rows are written once and read once much later, so they stream past L1.
__device__ __forceinline__ float4 ld_row(const float *base, size_t f4_index) {
    return reinterpret_cast<const float4 *>(base)[f4_index];
}
__device__ __forceinline__ void st_row(float *base, size_t f4_index, float4 v) {
    reinterpret_cast<float4 *>(base)[f4_index] = v;
}
__device__ __forceinline__ float4 ld_stream(const float *base, size_t f4_index) {
    float4 r;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(reinterpret_cast<const float4 *>(base) + f4_index));
    return r;
}
__device__ __forceinline__ void st_stream(float *base, size_t f4_index, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(
                     reinterpret_cast<float4 *>(base) + f4_index),
                 "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

__device__ __forceinline__ const float *shfl_ptr(const float *p, int src_lane) {
    return reinterpret_cast<const float *>(__shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)p, src_lane));
}

__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4_sub(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4_scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
// a + s * b with separately rounded multiply and add (no FMA contraction): keeps "row + alpha*grad"
// the same number whether grad was applied directly or staged and re-read.
__device__ __forceinline__ float4 f4_axpy(float4 a, float s, float4 b) {
    return make_float4(__fadd_rn(a.x, __fmul_rn(s, b.x)), __fadd_rn(a.y, __fmul_rn(s, b.y)),
                       __fadd_rn(a.z, __fmul_rn(s, b.z)), __fadd_rn(a.w, __fmul_rn(s, b.w)));
}
__device__ __forceinline__ float f4_dot(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }

// One more reference to row r: sets its `seen` bit, and its `multi` bit if `seen` was already set.
__device__ __forceinline__ void mark_row(uint32_t *seen, uint32_t *multi, uint32_t r) {
    const uint32_t bit = 1u << (r & 31);
    if (atomicOr(&seen[r >> 5], bit) & bit) atomicOr(&multi[r >> 5], bit);
}
#endif
