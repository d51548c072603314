// Candidate-list top-K selection shared by daisy_topk_candidates (bpr_eval.cu) and daisy_neumf_topk_candidates
// (neumf_rank.cu): K rounds of block arg-best over one group's scores in shared memory, order (score desc, position asc).
// A header rather than a separate unit because tests/emu builds one translation unit at a time.
#pragma once
#include "ctx.cuh"

namespace {

struct Best {
    float v;
    int idx;
};
__device__ __forceinline__ bool better(float v, int idx, float bv, int bidx) {
    return (v > bv) || (v == bv && idx < bidx);  // score desc, position asc
}
__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, b.v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, b.idx, o);
        if (better(ov, oi, b.v, b.idx)) {
            b.v = ov;
            b.idx = oi;
        }
    }
    return b;
}

// Called by all 256 threads of a block once sc[0, C) holds the group's scores.  cn = the group's candidate ids;
// op / oi / os = the group's K output slots (position, item, score).  A taken entry is marked with -inf, so sc is
// consumed.  Positions holding only -inf / NaN scores are never taken: their slots get (-1, -1, -inf).
__device__ __forceinline__ void topk_cand_rounds(float *sc, int C, int K, const int32_t *__restrict__ cn,
                                                 int32_t *__restrict__ op, int32_t *__restrict__ oi,
                                                 float *__restrict__ os) {
    __shared__ Best wbest[8];
    __shared__ int s_win;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int k = 0; k < K; ++k) {
        Best b;
        b.v = -INFINITY;
        b.idx = 0x7fffffff;
        for (int c = threadIdx.x; c < C; c += 256) {
            const float v = sc[c];
            if (!(v != v) && better(v, c, b.v, b.idx) && v != -INFINITY) {
                b.v = v;
                b.idx = c;
            }
        }
        b = warp_best(b);
        if (lane == 0) wbest[wid] = b;
        __syncthreads();
        if (wid == 0) {
            Best t = (lane < 8) ? wbest[lane] : Best{-INFINITY, 0x7fffffff};
            t = warp_best(t);
            if (lane == 0) {
                int w = t.idx;
                if (w == 0x7fffffff) {  // only -inf / NaN scores left: take the lowest untaken position
                    w = -1;
                }
                s_win = w;
                if (w >= 0) {
                    op[k] = w;
                    oi[k] = cn[w];
                    os[k] = t.v;
                } else {
                    op[k] = -1;
                    oi[k] = -1;
                    os[k] = -INFINITY;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0 && s_win >= 0) sc[s_win] = -INFINITY;
        __syncthreads();
    }
}

}  // namespace
