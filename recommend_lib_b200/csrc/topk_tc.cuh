// Interface between topk_full.cu (daisy_topk_full) and topk_tc.cu (the tcgen05 candidate filter).
#pragma once
#include "ctx.cuh"

struct TcItems {      // per daisy_topk_full call: BF16 copy of the item table and the largest item-row norm per tile
    void *Qb;         // [item_num, Dp] bf16, Dp = 64 or 128
    float *tile_norm;    // [ceil(item_num / 128)] max |q_i| over each 128-item tile (rounded up)
    int Dp;
};

bool daisy_tc_supported(const daisy_ctx *h);
void daisy_tc_collect(daisy_ctx *h);
int daisy_tc_prepare_items(daisy_ctx *h, const float *Q, TcItems *ti, cudaStream_t s);
void daisy_tc_free_items(TcItems *ti, cudaStream_t s);
int daisy_tc_filter(daisy_ctx *h, const float *P, const float *Q, const TcItems *ti, const int32_t *users, int nu, float c2,
                    const float *thr, int *cnt, unsigned long long *cand, int cap, int expected, cudaStream_t s);
