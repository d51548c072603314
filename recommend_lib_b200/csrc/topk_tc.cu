// Tensor-core candidate filter of the full-catalogue top-K (daisy_topk_full, filtered path) for sm_100a:
// tcgen05.mma (BF16 operands, FP32 accumulators in TMEM) fed by TMA (cp.async.bulk.tensor, 128-byte swizzle), TMEM
// read back with tcgen05.ld by the epilogue warps.
//
// Replaces (reference, file:line): the per-candidate scalar forward of the final ranking loop BPRMFRecommender.py:196-207
// -- together with topk_full.cu, which keeps the exact fp32 arithmetic that decides the ranking.
//
// What the tensor cores compute is NOT the ranking score.  The exact path ranks by fp32 scores (fp32 products summed in
// ascending k by fused multiply-adds); that arithmetic stays.  The tensor cores only answer "which items CAN be at or
// above user u's threshold thr_u".  BF16 keeps 8 significant bits, so round-to-nearest gives p~, q~ with
// |x~ - x| <= 2^-8 |x| (1 + 2^-8 rounds to 1), and per product |p~q~ - pq| <= (2 * 2^-8 + 2^-16) |pq|:
//     | sum_k p~_k q~_k  -  sum_k p_k q_k |  <=  (2^-7 + 2^-16) sum_k |p_k q_k|  <=  2^-7 (1 + 2^-9) |p_u| |q_i|
// (Cauchy-Schwarz for the last step).  BF16 x BF16 products are exact in fp32.  Two fp32 sums remain: the tensor
// core's accumulation of D <= 128 terms and the exact path's fma chain over the same terms, each off by at most
// gamma_D (1 + 2^-6) |p_u| |q_i| with gamma_D = D 2^-24 / (1 - D 2^-24) <= 2^-17 = 2^-7 * 2^-10 (twice that if the
// tensor core truncates instead of rounding).  Together with the product term that is at most 2^-7 * 3 * 2^-9
// |p_u| |q_i|, and kappa = 2^-7 * 17/16 leaves 2^-7 * 2^-4, more than ten times as much (the norms' own fp32 error is
// covered by the 1.0001 by which k_rows_bf16 rounds them up).  So every item
// whose EXACT score reaches thr_u satisfies
//     s~(u, i)  >=  thr_u / c^2  -  kappa |p_u| max_{j in tile(i)} |q_j|  =:  tau_u,t ,
// where tile(i) is the 128-item tile of i (the bound holds with |q_i| itself; the largest norm of the tile keeps it to
// one fma per row and tile in the epilogue, and is far tighter than the catalogue-wide largest norm when row norms
// spread: with log-normal norms of sigma 1 that one lets through ten times the candidates and overflows the list).
// The epilogue appends exactly the items with s~ >= tau_u,t to the user's candidate list: a guaranteed superset.  k_rescore then recomputes the candidates'
// scores with the exact path's arithmetic and k_select_cand (topk_full.cu) orders them, so the result is bit-identical
// to the exact path -- tests/test_bpr_gpu.py::test_topk_full_*.
//
// Kernel k_filter_tc (persistent, one CTA per SM, 640 threads):
//   warp 0      TMA producer: the unit's user tile A [256 users x Dp] once, then item tiles B [128 items x Dp] through a
//               3-stage ring (mbarrier full / empty pairs)
//   warp 1      MMA issuer (one elected lane): per item tile 2 x (Dp / 16) tcgen05.mma 128x128x16 into one of two
//               256-column accumulator buffers; tcgen05.commit frees the smem stage and publishes the accumulator
//   warp 2      TMEM allocation (all 512 columns) / deallocation
//   warps 4..19 epilogue (four per TMEM lane quarter, each a quarter of the columns: with 8 warps the kernel took 19.8 ms
//               for 16 384 x 2 M x 128, with 16 it takes 16.8 -- the scan is latency-bound, issue slots 23 % busy; issuing
//               the next TMEM load before scanning the current one was tried and is SLOWER, profiles/r02o_*):
//               tcgen05.ld 32 lanes x 32 columns, max tree
//               of the 32 scores against the row's tau, rare append into slots reserved in blocks
// Work unit = (group of 256 users, chunk of item tiles); units are dealt round-robin so that the CTAs running at the
// same time stream the same few chunks of Q~ (they stay in L2: every item tile is read from HBM about once and from L2
// once per user group).  Rooflines: tensor pipe 128 x 128 x 16 per 64 cycles per SM (2 N I D flops); L2 -> SM
// 32 KB per 1024 cycles per SM at Dp = 128.
#include <cuda.h>
#include <cuda_bf16.h>

#include "ctx.cuh"
#include "topk_tc.cuh"

namespace {

constexpr int TM = 128;      // users per MMA tile (UMMA M, one TMEM lane per user)
constexpr int MT = 2;        // MMA tiles of users per CTA (A stays in shared memory for a whole unit)
constexpr int TN = 128;      // items per tile (UMMA N)
constexpr int KATOM = 64;    // bf16 elements per 128-byte swizzle row
constexpr int STAGES = 3;
constexpr int ATOM_BYTES = 128 * 128;  // 128 rows x 128 bytes: one TMA box, 16 KB
constexpr int EPI_WARPS = 16;  // epilogue warps: EPI_WARPS / 4 per TMEM lane quarter, each takes an equal share of a
                               // tile's columns
constexpr int TC_THREADS = 32 * (4 + EPI_WARPS);

// ---- PTX wrappers ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void bar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol error (bad descriptor, lost arrive) must end the kernel with an error flag, not hang the
// device.  ~2 s of polling at 1.9 GHz; returns false on timeout.
__device__ __forceinline__ bool bar_wait(uint32_t bar, uint32_t parity, int *err) {
    const long long t0 = clock64();
    while (true) {
        uint32_t done;
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return true;
        if (clock64() - t0 > 4000000000ll || (*(volatile int *)err & 256)) {
            atomicOr(err, 256);
            return false;
        }
    }
}
__device__ __forceinline__ bool bar_wait_t(uint32_t bar, uint32_t parity, int *err, long long &acc) {
    const long long t0 = clock64();
    const bool ok = bar_wait(bar, parity, err);
    acc += clock64() - t0;
    return ok;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(map), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, BF16 x BF16 -> FP32, both operands K-major
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accum)
        : "memory");
}
// 32 lanes (this warp's TMEM quarter) x 32 consecutive columns -> 32 registers per thread
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}

// Shared-memory matrix descriptor of a K-major operand tile stored as [rows][64 bf16] with the 128-byte swizzle
// (what a TMA box of 64 x rows with CU_TENSOR_MAP_SWIZZLE_128B writes): 8-row groups are 1024 bytes apart (SBO), the
// leading-dimension offset is unused for swizzled K-major layouts (1), descriptor version 1 (sm_100), layout type 2 =
// SWIZZLE_128B.  Advancing by 16 bf16 along K inside the swizzle row = +32 bytes on the start address.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
           ((uint64_t)2 << 61);
}
// Instruction descriptor of kind::f16: D = F32 (bits 4-5 = 1), A = B = BF16 (bits 7-9, 10-12 = 1), both K-major (bits
// 15, 16 = 0), N >> 3 at bits 17-22, M >> 4 at bits 24-28.
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

struct FilterArgs {
    const float *tau;           // [rows padded to 256] per-user threshold in accumulator units (+inf on padding rows)
    const float *kp;            // [rows padded to 256] kappa |p_u|: the tile's threshold is tau - kp * tile_norm[t]
    const float *tile_norm;     // [n_tiles] largest |q_i| of each item tile (rounded up)
    int *cnt;                   // [rows] candidates appended so far
    unsigned long long *cand;   // [rows, cap] candidate slots (low word = item id; k_rescore completes the key)
    int cap;
    int reserve0, reserve1;     // candidate slots a thread reserves per (user, unit) up front / when its stock runs out
    int n_groups;               // groups of 256 users
    int n_tiles;                // item tiles of 128
    int tiles_per_chunk;
    int n_units;                // n_groups * n_chunks
    long long I;
    int *err;                   // handle error word: bit 256 = tensor-core pipeline timeout
    unsigned long long *stats;  // optional (DAISY_TC_STATS=1): cycles the roles spent waiting, summed over CTAs -- [0] producer on
                                // empty stages, [1] producer on A, [2] MMA on full stages, [3] MMA on drained accumulators,
                                // [4] epilogue on complete accumulators, [5] epilogue busy, [6] kernel cycles (CTA 0)
};

template <int KATOMS>
__global__ void __launch_bounds__(TC_THREADS, 1) k_filter_tc(const __grid_constant__ CUtensorMap mapA,
                                                              const __grid_constant__ CUtensorMap mapB, FilterArgs a) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment: the swizzle pattern is a function of the shared-memory address bits
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    constexpr uint32_t A_BYTES = MT * KATOMS * ATOM_BYTES;
    constexpr uint32_t B_STAGE = KATOMS * ATOM_BYTES;
    const uint32_t sA = base, sB = base + A_BYTES, sBar = sB + STAGES * B_STAGE;
    const uint32_t bar_full = sBar, bar_empty = sBar + 8u * STAGES, bar_afull = sBar + 16u * STAGES,
                   bar_aempty = bar_afull + 8u, bar_tfull = bar_afull + 16u, bar_tempty = bar_afull + 32u,
                   tmem_slot = bar_afull + 48u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            bar_init(bar_full + 8u * s, 1);
            bar_init(bar_empty + 8u * s, 1);
        }
        bar_init(bar_afull, 1);
        bar_init(bar_aempty, 1);
        for (int b = 0; b < 2; ++b) {
            bar_init(bar_tfull + 8u * b, 1);
            bar_init(bar_tempty + 8u * b, EPI_WARPS);  // one arrive per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t it = 0;  // item tiles issued so far (all units): stage = it % STAGES, phase = (it / STAGES) & 1
            uint32_t n_done = 0;
            bool ok = true;
            long long w_empty = 0, w_a = 0;
            for (int u = blockIdx.x; u < a.n_units && ok; u += gridDim.x, ++n_done) {
                const int g = u % a.n_groups, chunk = u / a.n_groups;
                const int t0 = chunk * a.tiles_per_chunk;
                const int t1 = min(t0 + a.tiles_per_chunk, a.n_tiles);
                if (n_done > 0) ok = bar_wait_t(bar_aempty, (n_done - 1) & 1u, a.err, w_a);  // the MMAs of the last unit are done with A
                if (!ok) break;
                bar_expect_tx(bar_afull, A_BYTES);
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int ka = 0; ka < KATOMS; ++ka)
                        tma_load_2d(sA + (uint32_t)(mt * KATOMS + ka) * ATOM_BYTES, &mapA, bar_afull, ka * KATOM,
                                    g * (MT * TM) + mt * TM);
                for (int t = t0; t < t1 && ok; ++t, ++it) {
                    const uint32_t st = it % STAGES, ph = (it / STAGES) & 1u;
                    if (it >= (uint32_t)STAGES) ok = bar_wait_t(bar_empty + 8u * st, ph ^ 1u, a.err, w_empty);
                    if (!ok) break;
                    bar_expect_tx(bar_full + 8u * st, B_STAGE);
#pragma unroll
                    for (int ka = 0; ka < KATOMS; ++ka)
                        tma_load_2d(sB + st * B_STAGE + (uint32_t)ka * ATOM_BYTES, &mapB, bar_full + 8u * st, ka * KATOM, t * TN);
                }
            }
            if (a.stats) {
                atomicAdd(a.stats + 0, (unsigned long long)w_empty);
                atomicAdd(a.stats + 1, (unsigned long long)w_a);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            uint32_t it = 0, n_done = 0;
            bool ok = true;
            long long w_full = 0, w_te = 0;
            const long long k0 = clock64();
            for (int u = blockIdx.x; u < a.n_units && ok; u += gridDim.x, ++n_done) {
                const int chunk = u / a.n_groups;
                const int t0 = chunk * a.tiles_per_chunk;
                const int t1 = min(t0 + a.tiles_per_chunk, a.n_tiles);
                ok = bar_wait(bar_afull, n_done & 1u, a.err);
                for (int t = t0; t < t1 && ok; ++t, ++it) {
                    const uint32_t st = it % STAGES, ph = (it / STAGES) & 1u;
                    const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
                    ok = bar_wait_t(bar_full + 8u * st, ph, a.err, w_full);
                    if (ok && it >= 2u) ok = bar_wait_t(bar_tempty + 8u * ab, aph ^ 1u, a.err, w_te);  // the epilogue drained this buffer
                    if (!ok) break;
                    tc_fence_after();
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        const uint32_t d = tmem_base + ab * (uint32_t)(MT * TN) + (uint32_t)(mt * TN);
#pragma unroll
                        for (int ka = 0; ka < KATOMS; ++ka) {
                            const uint64_t da = umma_desc(sA + (uint32_t)(mt * KATOMS + ka) * ATOM_BYTES);
                            const uint64_t db = umma_desc(sB + st * B_STAGE + (uint32_t)ka * ATOM_BYTES);
#pragma unroll
                            for (int k = 0; k < KATOM / 16; ++k)  // +32 bytes per K step of 16 bf16 = +2 in descriptor units
                                tc_mma_bf16(d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), kIdesc, (ka | k) ? 1u : 0u);
                        }
                    }
                    tc_commit(bar_empty + 8u * st);   // smem stage free once these MMAs have read it
                    tc_commit(bar_tfull + 8u * ab);   // accumulators complete
                }
                if (ok) tc_commit(bar_aempty);        // A may be overwritten once every MMA of the unit is done
            }
            if (a.stats) {
                atomicAdd(a.stats + 2, (unsigned long long)w_full);
                atomicAdd(a.stats + 3, (unsigned long long)w_te);
                if (blockIdx.x == 0) a.stats[6] = (unsigned long long)(clock64() - k0);
                a.stats[8 + blockIdx.x] = (unsigned long long)(clock64() - k0);
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int q = warp & 3;            // TMEM lane quarter this warp may read (hardware: lanes 32 (warp % 4) .. + 31)
        const int half = (warp - 4) >> 2;  // which share of a tile's columns this warp scans
        constexpr int CHUNKS = TN / 32 / (EPI_WARPS / 4);
        uint32_t it = 0;
        bool ok = true;
        long long w_tf = 0;
        const long long e0 = clock64();
        for (int u = blockIdx.x; u < a.n_units && ok; u += gridDim.x) {
            const int g = u % a.n_groups, chunk = u / a.n_groups;
            const int t0 = chunk * a.tiles_per_chunk;
            const int t1 = min(t0 + a.tiles_per_chunk, a.n_tiles);
            int row[MT];
            float tau[MT], kp[MT];
            // Candidate slots are RESERVED in blocks: an atomicAdd that returns a position costs a global round trip
            // (~1 us) and the append cannot proceed without it.  A thread owns its (row, column half) for the whole
            // unit, so it takes reserve0 slots per row up front (the round trips of all rows overlap, nothing waits
            // for them until the first candidate), refills by reserve1, and fills what it did not use with HOLE
            // entries (k_rescore gives them the lowest key).
            uint32_t nxt[MT], end[MT];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                row[mt] = g * (MT * TM) + mt * TM + q * 32 + lane;
                tau[mt] = a.tau[row[mt]];
                kp[mt] = a.kp[row[mt]];
                nxt[mt] = end[mt] = 0;
                if (tau[mt] < INFINITY) {
                    nxt[mt] = (uint32_t)atomicAdd(&a.cnt[row[mt]], a.reserve0);
                    end[mt] = nxt[mt] + (uint32_t)a.reserve0;
                }
            }
            for (int t = t0; t < t1 && ok; ++t, ++it) {
                const uint32_t ab = it & 1u, aph = (it >> 1) & 1u;
                ok = bar_wait_t(bar_tfull + 8u * ab, aph, a.err, w_tf);
                if (!ok) break;
                tc_fence_after();
                const long long i0 = (long long)t * TN;
                const float qmax = __ldg(a.tile_norm + t);
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + ab * (uint32_t)(MT * TN) + (uint32_t)(mt * TN);
                    unsigned long long *slots = a.cand + (size_t)row[mt] * a.cap;
                    const float th = fmaf(-kp[mt], qmax, tau[mt]);
#pragma unroll 1
                    for (int cc = 0; cc < CHUNKS; ++cc) {
                        const int c = half * CHUNKS + cc;
                        float v[32];
                        tc_ld32(tbase + (uint32_t)(c * 32), v);
                        // One warp per scheduler hides no latency, so the scan is written as independent operations: a
                        // max tree (4 sub-maxima of 8 scores, then their maximum) instead of 32 compares chained through
                        // one predicate; only a sub-group whose maximum reaches the threshold is looked at score by score.
                        float m8[4];
#pragma unroll
                        for (int gq = 0; gq < 4; ++gq) {
                            const float a0 = fmaxf(v[8 * gq + 0], v[8 * gq + 1]), a1 = fmaxf(v[8 * gq + 2], v[8 * gq + 3]);
                            const float a2 = fmaxf(v[8 * gq + 4], v[8 * gq + 5]), a3 = fmaxf(v[8 * gq + 6], v[8 * gq + 7]);
                            m8[gq] = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
                        }
                        if (fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3])) >= th) {
#pragma unroll
                            for (int gq = 0; gq < 4; ++gq)
                                if (m8[gq] >= th) {
#pragma unroll
                                    for (int j = 8 * gq; j < 8 * gq + 8; ++j)
                                        if (v[j] >= th) {
                                            const long long item = i0 + c * 32 + j;
                                            if (item < a.I) {
                                                if (nxt[mt] == end[mt]) {
                                                    nxt[mt] = (uint32_t)atomicAdd(&a.cnt[row[mt]], a.reserve1);
                                                    end[mt] = nxt[mt] + (uint32_t)a.reserve1;
                                                }
                                                if (nxt[mt] < (uint32_t)a.cap) slots[nxt[mt]] = (unsigned long long)item;
                                                ++nxt[mt];
                                            }
                                        }
                                }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) bar_arrive(bar_tempty + 8u * ab);
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)  // unused reservations become holes
                for (; nxt[mt] < end[mt]; ++nxt[mt])
                    if (nxt[mt] < (uint32_t)a.cap) a.cand[(size_t)row[mt] * a.cap + nxt[mt]] = 0xFFFFFFFFull;
        }
        if (a.stats && lane == 0 && warp == 4) {
            atomicAdd(a.stats + 4, (unsigned long long)w_tf);
            atomicAdd(a.stats + 5, (unsigned long long)(clock64() - e0 - w_tf));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}

// ---- operand preparation --------------------------------------------------------------------------------------------
// One warp per row: BF16 copy padded to Dp columns, Euclidean norm of the fp32 row (into norm[w] and / or as the
// maximum over the row's item tile, tile_norm_bits[w / TN]).  users != nullptr gathers rows
// users[m] (validated: a bad id raises the handle's error flag and reads row 0); rows >= n_rows are zero padding.
__global__ void __launch_bounds__(256) k_rows_bf16(const float *__restrict__ W, const int32_t *__restrict__ users,
                                                    long long n_rows, long long n_rows_padded, uint32_t limit, int D, int Dp,
                                                    __nv_bfloat16 *__restrict__ out, float *__restrict__ norm,
                                                    unsigned *__restrict__ tile_norm_bits, int *err) {
    const int lane = threadIdx.x & 31;
    const long long w = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (w >= n_rows_padded) return;
    __nv_bfloat16 *o = out + (size_t)w * Dp;
    if (w >= n_rows) {
        for (int k = lane; k < Dp; k += 32) o[k] = __float2bfloat16_rn(0.f);
        if (norm && lane == 0) norm[w] = 0.f;
        return;
    }
    long long r = w;
    if (users) {
        uint32_t u = (uint32_t)users[w];
        if (u >= limit) {
            if (lane == 0) {
                atomicOr(&err[0], 1);
                atomicMin(&err[1], (int)w);
            }
            u = 0;
        }
        r = (long long)u;
    }
    const float *src = W + (size_t)r * D;
    float ss = 0.f;
    for (int k = lane; k < Dp; k += 32) {
        const float x = k < D ? src[k] : 0.f;
        ss = fmaf(x, x, ss);
        o[k] = __float2bfloat16_rn(x);
    }
    ss = warp_sum(ss);
    const float nrm = sqrtf(ss) * 1.0001f;  // rounded up a little: the norm is used as an upper bound
    if (lane == 0) {
        if (norm) norm[w] = nrm;
        if (tile_norm_bits) atomicMax(tile_norm_bits + w / TN, __float_as_uint(nrm));  // non-negative floats order like their bits
    }
}

// tau_u = thr_u / c^2 (moved down by 2^-20 of its magnitude: the exact path's final multiply by c^2 rounds) and
// kp_u = kappa |p_u|: the epilogue's threshold for item tile t is tau_u - kp_u tile_norm[t].  +inf / 0 on padding rows;
// candidate counters cleared
__global__ void k_tau(const float *__restrict__ thr, const float *__restrict__ pnorm, float inv_c2, int n, int n_padded,
                      float *__restrict__ tau, float *__restrict__ kp, int *__restrict__ cnt) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_padded) return;
    if (m >= n) {
        tau[m] = INFINITY;
        kp[m] = 0.f;
        return;
    }
    const float kappa = 0.0078125f * 1.0625f;  // 2^-7 * 17/16: see the bound at the top of this file
    const float t = thr[m] * inv_c2;
    tau[m] = t - fabsf(t) * 9.5367431640625e-7f;
    kp[m] = kappa * pnorm[m];
    cnt[m] = 0;
}

__device__ __forceinline__ uint32_t okey_tc(float f) {  // order-preserving float -> uint32 (as in topk_full.cu)
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// Exact scores of the candidates, with the arithmetic of the exact path (k_score_tile: acc = fma(p_k, q_k, acc) for
// ascending k from 0, then acc * c^2): one thread per candidate, the user's row broadcast from shared memory.
// grid (ceil(cap / 256), n_users); completes the 64-bit (score desc, item asc) key in place.
__global__ void __launch_bounds__(256) k_rescore(const float *__restrict__ P, const float *__restrict__ Q,
                                                  const int32_t *__restrict__ users, uint32_t U, int D, float c2,
                                                  const int *__restrict__ cnt, int cap, unsigned long long *__restrict__ cand) {
    extern __shared__ float prow[];
    const int m = blockIdx.y;
    const int n = min(cnt[m], cap);
    if ((int)(blockIdx.x * blockDim.x) >= n) return;
    uint32_t u = (uint32_t)users[m];
    if (u >= U) u = 0;  // already flagged by k_rows_bf16
    for (int k = threadIdx.x; k < D; k += blockDim.x) prow[k] = P[(size_t)u * D + k];
    __syncthreads();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t item = (uint32_t)(cand[(size_t)m * cap + p] & 0xFFFFFFFFull);
    if (item == 0xFFFFFFFFu) {  // a reserved slot the filter did not use: lowest possible key, sorts behind everything
        cand[(size_t)m * cap + p] = 0ull;
        return;
    }
    const float4 *q4 = reinterpret_cast<const float4 *>(Q + (size_t)item * D);
    float acc = 0.f;
    for (int k4 = 0; k4 < D / 4; ++k4) {
        const float4 b = q4[k4];
        acc = fmaf(prow[4 * k4 + 0], b.x, acc);
        acc = fmaf(prow[4 * k4 + 1], b.y, acc);
        acc = fmaf(prow[4 * k4 + 2], b.z, acc);
        acc = fmaf(prow[4 * k4 + 3], b.w, acc);
    }
    const float v = acc * c2;
    cand[(size_t)m * cap + p] = ((unsigned long long)okey_tc(v) << 32) | (unsigned long long)(0xFFFFFFFFu - item);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
        else
            (void)cudaGetLastError();
    }
    return fn;
}

// [rows, Dp] bf16 row-major, box = 64 columns x 128 rows, 128-byte swizzle, rows beyond the end read as zero
static bool make_map(CUtensorMap *map, void *base, uint64_t rows, int Dp) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)Dp, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)Dp * 2};
    const cuuint32_t box[2] = {(cuuint32_t)KATOM, 128u};
    const cuuint32_t estr[2] = {1u, 1u};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

// fold the event pair of the last timed daisy_tc_filter call into the running sums (synchronises on the events)
void daisy_tc_collect(daisy_ctx *h) {
    if (!h->tc_ev_pending) return;
    float a = 0.f, b = 0.f;
    if (cudaEventSynchronize(h->tc_ev[2]) == cudaSuccess && cudaEventElapsedTime(&a, h->tc_ev[0], h->tc_ev[1]) == cudaSuccess &&
        cudaEventElapsedTime(&b, h->tc_ev[1], h->tc_ev[2]) == cudaSuccess) {
        h->tc_filter_ms += a;
        h->tc_rescore_ms += b;
        h->tc_count++;
    } else {
        (void)cudaGetLastError();
    }
    h->tc_ev_pending = 0;
}

extern "C" int daisy_topk_tc_ms(daisy_handle_t h, double *filter_ms, double *rescore_ms, int64_t *count) {
    DAISY_REQUIRE(h && filter_ms && rescore_ms && count, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    daisy_tc_collect(h);
    *count = h->tc_count;
    *filter_ms = h->tc_count ? h->tc_filter_ms / (double)h->tc_count : 0.0;
    *rescore_ms = h->tc_count ? h->tc_rescore_ms / (double)h->tc_count : 0.0;
    h->tc_filter_ms = h->tc_rescore_ms = 0.0;
    h->tc_count = 0;
    return DAISY_OK;
}

bool daisy_tc_supported(const daisy_ctx *h) { return h->D % 4 == 0 && h->D <= 128 && encode_fn() != nullptr; }

int daisy_tc_prepare_items(daisy_ctx *h, const float *Q, TcItems *ti, cudaStream_t s) {
    const int Dp = h->D <= 64 ? 64 : 128;
    ti->Dp = Dp;
    ti->Qb = nullptr;
    ti->tile_norm = nullptr;
    const size_t norm_bytes = (size_t)((h->I + TN - 1) / TN) * sizeof(unsigned);
    cudaError_t e = daisy_scratch_alloc(h, (void **)&ti->Qb, (size_t)h->I * Dp * 2, s);
    if (e == cudaSuccess) e = daisy_scratch_alloc(h, (void **)&ti->tile_norm, norm_bytes, s);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        daisy_tc_free_items(ti, s);
        daisy_set_error("top-K tensor-core workspace allocation failed (%zu bytes of bf16 item rows)", (size_t)h->I * Dp * 2);
        return DAISY_ENOMEM;
    }
    cudaMemsetAsync(ti->tile_norm, 0, norm_bytes, s);
    const long long rows = h->I;
    k_rows_bf16<<<daisy_ceil_div(rows, 8), 256, 0, s>>>(Q, nullptr, rows, rows, 0u, h->D, Dp, (__nv_bfloat16 *)ti->Qb, nullptr,
                                                       (unsigned *)ti->tile_norm, h->err);
    h->launches++;
    return DAISY_OK;
}

void daisy_tc_free_items(TcItems *ti, cudaStream_t s) {
    if (ti->Qb) cudaFreeAsync(ti->Qb, s);
    if (ti->tile_norm) cudaFreeAsync(ti->tile_norm, s);
    ti->Qb = nullptr;
    ti->tile_norm = nullptr;
}

// Candidate lists of users[0 .. nu) against the whole catalogue; thr [nu] are the users' thresholds in SCORE units
// (c^2 folded in), cnt [>= nu rounded up to 256], cand [rows, cap].  On return (stream order) cand holds complete keys.
int daisy_tc_filter(daisy_ctx *h, const float *P, const float *Q, const TcItems *ti, const int32_t *users, int nu, float c2,
                    const float *thr, int *cnt, unsigned long long *cand, int cap, int expected, cudaStream_t s) {
    const int Dp = ti->Dp;
    const int rows_p = (nu + MT * TM - 1) / (MT * TM) * (MT * TM);
    void *Pb = nullptr;
    float *pnorm = nullptr, *tau = nullptr;
    cudaError_t e = daisy_scratch_alloc(h, &Pb, (size_t)rows_p * Dp * 2, s);
    if (e == cudaSuccess) e = daisy_scratch_alloc(h, (void **)&pnorm, (size_t)rows_p * 4, s);
    if (e == cudaSuccess) e = daisy_scratch_alloc(h, (void **)&tau, (size_t)rows_p * 2 * 4, s);  // tau, then kp
    int rc = DAISY_OK;
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        daisy_set_error("top-K tensor-core workspace allocation failed");
        rc = DAISY_ENOMEM;
    }
    CUtensorMap mapA, mapB;
    if (!rc && (!make_map(&mapA, Pb, (uint64_t)rows_p, Dp) || !make_map(&mapB, ti->Qb, (uint64_t)h->I, Dp))) {
        daisy_set_error("cuTensorMapEncodeTiled failed");
        rc = DAISY_ECUDA;
    }
    if (!rc) {
        k_rows_bf16<<<daisy_ceil_div(rows_p, 8), 256, 0, s>>>(P, users, nu, rows_p, (uint32_t)h->U, h->D, Dp, (__nv_bfloat16 *)Pb,
                                                             pnorm, nullptr, h->err);
        k_tau<<<daisy_ceil_div(rows_p, 256), 256, 0, s>>>(thr, pnorm, 1.0f / c2, nu, rows_p, tau, tau + rows_p, cnt);
        FilterArgs a;
        a.tau = tau;
        a.kp = tau + rows_p;
        a.tile_norm = ti->tile_norm;
        a.cnt = cnt;
        a.cand = cand;
        a.cap = cap;
        a.n_groups = rows_p / (MT * TM);
        a.n_tiles = (int)((h->I + TN - 1) / TN);
        a.I = h->I;
        a.err = h->err;
        a.stats = nullptr;
        const char *st_env = getenv("DAISY_TC_STATS");
        unsigned long long *stats_dev = nullptr;
        if (st_env && atoi(st_env) > 0 && daisy_scratch_alloc(h, (void **)&stats_dev, (8 + 1024) * sizeof(unsigned long long), s) == cudaSuccess) {
            cudaMemsetAsync(stats_dev, 0, (8 + 1024) * sizeof(unsigned long long), s);
            a.stats = stats_dev;
        }
        // Chunks of item tiles: enough units to balance the SMs (>= 4 per CTA), and chunks small enough that the ones
        // being streamed at the same time (ceil(SMs / groups) of them) stay in L2 together (<= 48 MB)
        const int grid = h->num_sms;
        const double q_bytes = (double)h->I * Dp * 2.0;
        const int live = (grid + a.n_groups - 1) / a.n_groups;
        int n_chunks = (int)(q_bytes * live / (48.0 * 1024 * 1024)) + 1;
        const int for_balance = (4 * grid + a.n_groups - 1) / a.n_groups;
        if (n_chunks < for_balance) n_chunks = for_balance;
        // ... but few enough that the slots a row reserves up front (n_chunks * (EPI_WARPS / 4) * reserve0, at most
        // 1.5 expected + 4 (EPI_WARPS / 4) n_chunks) leave half of cap to the candidates: k_select_cand counts
        // reservations, used or not, and sends a row past cap to the exact fallback
        const int max_chunks = (int)((cap / 2 - 1.5 * expected) / (4 * (EPI_WARPS / 4)));
        if (n_chunks > max_chunks) n_chunks = max_chunks > 1 ? max_chunks : 1;
        if (n_chunks > a.n_tiles) n_chunks = a.n_tiles;
        a.tiles_per_chunk = (a.n_tiles + n_chunks - 1) / n_chunks;
        n_chunks = (a.n_tiles + a.tiles_per_chunk - 1) / a.tiles_per_chunk;
        a.n_units = a.n_groups * n_chunks;
        // slots reserved per (user, unit): the expected share of the user's candidates (+ 15 % for the widened
        // threshold, + 30 % headroom) up front, refills by a quarter of that
        a.reserve0 = (int)(1.5 * expected / n_chunks / (EPI_WARPS / 4)) + 4;   // per thread: a row has EPI_WARPS / 4 scanners
        a.reserve1 = a.reserve0 / 4 > 8 ? a.reserve0 / 4 : 8;
        const bool timed = h->timing != 0;
        if (timed) {
            daisy_tc_collect(h);
            for (int i = 0; i < 3; ++i)
                if (!h->tc_ev[i]) cudaEventCreate(&h->tc_ev[i]);
            cudaEventRecord(h->tc_ev[0], s);
        }
        const int katoms = Dp / KATOM;
        const size_t smem = (size_t)(MT + STAGES) * katoms * ATOM_BYTES + 1024 + 256;
        if (katoms == 1) {
            cudaFuncSetAttribute(k_filter_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k_filter_tc<1><<<grid, TC_THREADS, smem, s>>>(mapA, mapB, a);
        } else {
            cudaFuncSetAttribute(k_filter_tc<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k_filter_tc<2><<<grid, TC_THREADS, smem, s>>>(mapA, mapB, a);
        }
        if (timed) cudaEventRecord(h->tc_ev[1], s);
        if (stats_dev) {  // diagnostic: synchronises
            static unsigned long long hs[8 + 1024];
            if (cudaMemcpyAsync(hs, stats_dev, sizeof(hs), cudaMemcpyDeviceToHost, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess) {
                const double n = (double)grid, k = (double)hs[6];
                unsigned long long mn = ~0ull, mx = 0;
                double sum = 0;
                for (int b = 0; b < grid && b < 1024; ++b) {
                    mn = hs[8 + b] < mn ? hs[8 + b] : mn;
                    mx = hs[8 + b] > mx ? hs[8 + b] : mx;
                    sum += (double)hs[8 + b];
                }
                fprintf(stderr, "[k_filter_tc] CTA cycles min %llu mean %.0f max %llu\n", mn, sum / n, mx);
                fprintf(stderr, "[k_filter_tc] kernel %.0f cycles; per CTA, fraction of it: producer waits for a free stage %.3f, for A %.3f | "
                                "MMA waits for a full stage %.3f, for a drained accumulator %.3f | epilogue (warp 4) waits for an accumulator "
                                "%.3f, busy %.3f | units %d, tiles per chunk %d, reserve %d/%d\n",
                        k, hs[0] / n / k, hs[1] / n / k, hs[2] / n / k, hs[3] / n / k, hs[4] / n / k, hs[5] / n / k, a.n_units,
                        a.tiles_per_chunk, a.reserve0, a.reserve1);
            }
            cudaFreeAsync(stats_dev, s);
        }
        dim3 gr((unsigned)((cap + 255) / 256), (unsigned)nu);
        k_rescore<<<gr, 256, h->D * sizeof(float), s>>>(P, Q, users, (uint32_t)h->U, h->D, c2, cnt, cap, cand);
        if (timed) {
            cudaEventRecord(h->tc_ev[2], s);
            h->tc_ev_pending = 1;
        }
        h->launches += 4;
        if (cudaGetLastError() != cudaSuccess) {
            daisy_set_error("top-K tensor-core launch failed");
            rc = DAISY_ECUDA;
        }
    }
    for (void *p : {Pb, (void *)pnorm, (void *)tau})
        if (p) cudaFreeAsync(p, s);
    return rc;
}
