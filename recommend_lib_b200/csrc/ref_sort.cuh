// Stable compaction + LSD radix sort of (32-bit key, 32-bit index) pairs whose COUNT lives in device memory.
//
// The general BPR bookkeeping (step_kernels.cuh: book_kernels) sorts only the refs whose row is referenced more than
// once in the batch.  How many that is, is known on the device only, and reading it back would cost a host sync inside
// a chain that runs one step ahead on a side stream and is captured into a CUDA graph -- so cub::DeviceRadixSort, which
// takes its item count from the host, cannot sort them.  This header can:
//
//   k_dsort_compact   input element x < n_in is kept when the functor `src(x, key)` says so; the kept pairs (key, x)
//                     are written densely in x order (stable), the device-side count and the digit counts of every
//                     radix pass are accumulated in DsortState
//   k_dsort_pass      one stable 8-bit counting pass per launch over the n kept pairs; tile offsets by decoupled
//                     look-back (each tile publishes its digit counts, a tile sums its predecessors' back to the
//                     first complete prefix)
//
// Tiles are taken from an atomic counter, not from blockIdx: a block only ever waits for tiles that blocks which are
// already running took before it, so the look-back makes progress however the blocks are placed (on the bookkeeping
// stream they are placed as the main kernel's blocks retire, in no particular order).  Plain CUDA only -- no inline PTX,
// no CUB device calls -- so that tests/emu can run the kernels on the host.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define DSORT_THREADS 256
#define DSORT_IPT 8                                 // pairs per thread and tile
#define DSORT_TILE (DSORT_THREADS * DSORT_IPT)      // 2048
#define DSORT_RADIX 256
#define DSORT_MAX_PASSES 4
// look-back word: flag in the top two bits, count below (counts < 2^30: the caller keeps n_in below that)
#define DSORT_AGG 0x40000000u    // the tile's own count is available
#define DSORT_INCL 0x80000000u   // the count of every tile up to and including this one is available
#define DSORT_FLAGS 0xC0000000u
#define DSORT_COUNT 0x3FFFFFFFu

static_assert(DSORT_THREADS == DSORT_RADIX, "one thread per digit");

namespace {  // every unit that includes this header gets its own copy of the kernels

// Zero before k_dsort_compact.  Written by the sort kernels, read by the caller's later kernels (n, n_lo).
struct DsortState {
    uint32_t tile[1 + DSORT_MAX_PASSES];            // tile counters: compaction, then one per pass
    uint32_t n;                                     // kept pairs
    uint32_t n_lo;                                  // kept pairs whose key is below `split`
    uint32_t pad;
    uint32_t hist[DSORT_MAX_PASSES][DSORT_RADIX];   // digit counts of the kept keys, per pass
};

// Look-back words: [tiles] of the compaction (zero before it, like DsortState), then [passes][tiles][RADIX] of the
// passes (zeroed by the compaction kernel).
static inline int dsort_tiles(int64_t n_in) { return (int)((n_in + DSORT_TILE - 1) / DSORT_TILE); }
static inline size_t dsort_status_words(int64_t n_in) {
    return (size_t)dsort_tiles(n_in) * (1 + (size_t)DSORT_MAX_PASSES * DSORT_RADIX);
}

__device__ __forceinline__ uint32_t dsort_ld(const uint32_t *p) { return *(const volatile uint32_t *)p; }
__device__ __forceinline__ void dsort_st(uint32_t *p, uint32_t v) { *(volatile uint32_t *)p = v; }

// Decoupled look-back over one count: word `tile` of `status` (stride `stride`) gets this tile's aggregate, then its
// inclusive prefix.  Returns the exclusive prefix.  Tile t only waits for tiles < t, which were taken earlier by blocks
// that are running, and tile 0 never waits.
__device__ __forceinline__ uint32_t dsort_lookback(uint32_t *status, int stride, int tile, uint32_t agg) {
    uint32_t *me = status + (size_t)tile * stride;
    if (tile == 0) {
        dsort_st(me, DSORT_INCL | agg);
        return 0;
    }
    dsort_st(me, DSORT_AGG | agg);
    uint32_t excl = 0;
    for (int t = tile - 1;; --t) {
        uint32_t v;
        do {
            v = dsort_ld(status + (size_t)t * stride);
        } while (!(v & DSORT_FLAGS));
        excl += v & DSORT_COUNT;
        if (v & DSORT_INCL) break;
    }
    dsort_st(me, DSORT_INCL | (excl + agg));
    return excl;
}

// Exclusive scan of one value per thread over the block (256 threads); `tmp` holds 8 words.
__device__ __forceinline__ uint32_t dsort_block_excl(uint32_t v, uint32_t *tmp) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_sync(FULL, incl, lane >= o ? lane - o : lane);
        if (lane >= o) incl += t;
    }
    if (lane == 31) tmp[w] = incl;
    __syncthreads();
    uint32_t wbase = 0;
    for (int i = 0; i < w; ++i) wbase += tmp[i];
    __syncthreads();  // tmp may be reused by the caller's next scan
    return wbase + incl - v;
}

// Element x in [0, n_in) is kept when src(x, key) returns true (the functor may also act on the elements it drops).
template <class Src>
__global__ void __launch_bounds__(DSORT_THREADS)
    k_dsort_compact(Src src, int n_in, uint32_t split, int passes, uint32_t *__restrict__ okey,
                    uint32_t *__restrict__ oval, DsortState *ss, uint32_t *status_c, uint32_t *status_p) {
    __shared__ uint32_t s_hist[DSORT_MAX_PASSES][DSORT_RADIX];
    __shared__ uint32_t s_warp[DSORT_THREADS / 32];
    __shared__ uint32_t s_tile, s_base, s_agg, s_lo;
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    if (tid == 0) {
        s_tile = atomicAdd(&ss->tile[0], 1u);
        s_lo = 0;
    }
    for (int p = 0; p < passes; ++p) s_hist[p][tid] = 0;
    __syncthreads();
    const int tile = (int)s_tile;  // < gridDim.x: the grid has one block per tile
    // the passes' look-back words of this tile start at zero (no pass has more tiles than the compaction)
    for (int p = 0; p < passes; ++p) status_p[((size_t)p * gridDim.x + tile) * DSORT_RADIX + tid] = 0;

    uint32_t key[DSORT_IPT];
    unsigned m[DSORT_IPT];
    const int x0 = tile * DSORT_TILE + w * 32 * DSORT_IPT + lane;  // warp-striped: x = x0 + 32 k
    uint32_t cnt = 0, lo = 0;
#pragma unroll
    for (int k = 0; k < DSORT_IPT; ++k) {
        const int x = x0 + 32 * k;
        key[k] = 0;
        const bool keep = x < n_in && src(x, key[k]);
        m[k] = __ballot_sync(FULL, keep);
        cnt += __popc(m[k]);
        lo += __popc(__ballot_sync(FULL, keep && key[k] < split));
        if (keep)
            for (int p = 0; p < passes; ++p) atomicAdd(&s_hist[p][(key[k] >> (8 * p)) & 0xFFu], 1u);
    }
    if (lane == 0) {
        s_warp[w] = cnt;
        atomicAdd(&s_lo, lo);
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0;
        for (int i = 0; i < DSORT_THREADS / 32; ++i) {
            const uint32_t c = s_warp[i];
            s_warp[i] = run;
            run += c;
        }
        s_agg = run;
        s_base = dsort_lookback(status_c, 1, tile, run);
        atomicAdd(&ss->n, run);
        atomicAdd(&ss->n_lo, s_lo);
    }
    for (int p = 0; p < passes; ++p)
        if (s_hist[p][tid]) atomicAdd(&ss->hist[p][tid], s_hist[p][tid]);
    __syncthreads();
    uint32_t pos = s_base + s_warp[w];
#pragma unroll
    for (int k = 0; k < DSORT_IPT; ++k) {
        if (m[k] >> lane & 1u) {
            const uint32_t q = pos + __popc(m[k] & lt);
            okey[q] = key[k];
            oval[q] = (uint32_t)(x0 + 32 * k);
        }
        pos += __popc(m[k]);
    }
}

// One stable pass on bits [8 pass, 8 pass + 8) over the ss->n pairs.  `tiles` = the compaction's grid (the stride of
// the look-back words).  Blocks loop over tiles, so the grid can be smaller than the worst case.
__global__ void __launch_bounds__(DSORT_THREADS)
    k_dsort_pass(const uint32_t *__restrict__ ikey, const uint32_t *__restrict__ ival, uint32_t *__restrict__ okey,
                 uint32_t *__restrict__ oval, int pass, int tiles, DsortState *ss, uint32_t *status_p) {
    __shared__ uint32_t s_wh[DSORT_THREADS / 32][DSORT_RADIX];  // per warp: digit counts, then offsets
    __shared__ uint32_t s_start[DSORT_RADIX];                   // first tile-local index of each digit
    __shared__ uint32_t s_gofs[DSORT_RADIX];                    // output position of the tile's first key of each digit
    __shared__ uint32_t s_key[DSORT_TILE], s_val[DSORT_TILE];
    __shared__ uint32_t s_tmp[DSORT_THREADS / 32];
    __shared__ uint32_t s_tile;
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t n = ss->n;
    const int shift = 8 * pass;
    uint32_t *status = status_p + (size_t)pass * tiles * DSORT_RADIX + tid;
    // where digit `tid` starts in the output: exclusive scan of the pass's digit counts
    const uint32_t gdig = dsort_block_excl(ss->hist[pass][tid], s_tmp);
    while (true) {
        if (tid == 0) s_tile = atomicAdd(&ss->tile[1 + pass], 1u);
        for (int i = 0; i < DSORT_THREADS / 32; ++i) s_wh[i][tid] = 0;
        __syncthreads();
        const int tile = (int)s_tile;
        const int64_t base = (int64_t)tile * DSORT_TILE;
        if (base >= (int64_t)n) return;  // block-uniform
        const int cnt_tile = (int64_t)n - base < DSORT_TILE ? (int)((int64_t)n - base) : DSORT_TILE;
        uint32_t key[DSORT_IPT], val[DSORT_IPT], rank[DSORT_IPT];
#pragma unroll
        for (int k = 0; k < DSORT_IPT; ++k) {
            const int e = w * 32 * DSORT_IPT + 32 * k + lane;
            const bool ok = e < cnt_tile;
            key[k] = ok ? ikey[base + e] : 0u;
            val[k] = ok ? ival[base + e] : 0u;
        }
        // rank inside the warp, in tile order: the lanes holding the same digit find each other with one ballot per
        // digit bit, the lowest of them bumps the warp's count
#pragma unroll
        for (int k = 0; k < DSORT_IPT; ++k) {
            const int e = w * 32 * DSORT_IPT + 32 * k + lane;
            const bool ok = e < cnt_tile;
            const uint32_t d = (key[k] >> shift) & 0xFFu;
            unsigned mm = __ballot_sync(FULL, ok);
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const bool bit = (d >> b) & 1u;
                const unsigned v = __ballot_sync(FULL, bit);
                mm &= bit ? v : ~v;
            }
            const int leader = ok ? __ffs((int)mm) - 1 : lane;
            uint32_t c = 0;
            if (ok && lane == leader) {
                c = s_wh[w][d];
                s_wh[w][d] = c + __popc(mm);
            }
            c = __shfl_sync(FULL, c, leader);
            rank[k] = c + __popc(mm & lt);
            __syncwarp();
        }
        __syncthreads();
        // digit tid: the tile's count and every warp's offset inside it
        uint32_t tot = 0;
        for (int i = 0; i < DSORT_THREADS / 32; ++i) {
            const uint32_t c = s_wh[i][tid];
            s_wh[i][tid] = tot;
            tot += c;
        }
        const uint32_t start = dsort_block_excl(tot, s_tmp);
        s_start[tid] = start;
        s_gofs[tid] = gdig + dsort_lookback(status, DSORT_RADIX, tile, tot);
        __syncthreads();
#pragma unroll
        for (int k = 0; k < DSORT_IPT; ++k) {
            const int e = w * 32 * DSORT_IPT + 32 * k + lane;
            if (e < cnt_tile) {
                const uint32_t d = (key[k] >> shift) & 0xFFu;
                const uint32_t li = s_start[d] + s_wh[w][d] + rank[k];
                s_key[li] = key[k];
                s_val[li] = val[k];
            }
        }
        __syncthreads();
        for (int i = tid; i < cnt_tile; i += DSORT_THREADS) {  // runs of one digit land on consecutive positions
            const uint32_t kk = s_key[i];
            const uint32_t d = (kk >> shift) & 0xFFu;
            const uint32_t pos = s_gofs[d] + (uint32_t)i - s_start[d];
            okey[pos] = kk;
            oval[pos] = s_val[i];
        }
        __syncthreads();  // shared memory is refilled by the next tile
    }
}

static inline int dsort_passes(int key_bits) { return key_bits <= 8 ? 1 : (key_bits + 7) / 8; }

// Compaction + passes on one stream.  DsortState and the compaction's look-back words (status[0, tiles)) must be zero.
// (k0, v0) receive the compacted pairs, the passes alternate between (k0, v0) and (k1, v1); *out_k / *out_v = where the
// sorted pairs are.  `pass_blocks` bounds the grid of each pass.  Returns the number of launches.
template <class Src>
static int dsort_launch(const Src &src, int n_in, uint32_t split, int key_bits, uint32_t *k0, uint32_t *v0,
                        uint32_t *k1, uint32_t *v1, DsortState *ss, uint32_t *status, int pass_blocks,
                        cudaStream_t st, uint32_t **out_k, uint32_t **out_v) {
    const int passes = dsort_passes(key_bits);
    *out_k = k0;
    *out_v = v0;
    if (n_in <= 0) return 0;
    const int tiles = dsort_tiles(n_in);
    uint32_t *status_p = status + tiles;
    k_dsort_compact<Src><<<tiles, DSORT_THREADS, 0, st>>>(src, n_in, split, passes, k0, v0, ss, status, status_p);
    const int grid = pass_blocks > 0 && pass_blocks < tiles ? pass_blocks : tiles;
    uint32_t *ik = k0, *iv = v0, *ok = k1, *ov = v1;
    for (int p = 0; p < passes; ++p) {
        k_dsort_pass<<<grid, DSORT_THREADS, 0, st>>>(ik, iv, ok, ov, p, tiles, ss, status_p);
        uint32_t *tk = ik, *tv = iv;
        ik = ok; iv = ov; ok = tk; ov = tv;
    }
    *out_k = ik;
    *out_v = iv;
    return 1 + passes;
}

}  // namespace
