// TEST INFRASTRUCTURE ONLY: csrc/ref_sort.cuh (the device-counted compaction + radix sort of the BPR bookkeeping) built
// for the host against tests/emu/emu.h by tests/test_ref_sort_emulation.py.  Blocks run one after the other there, so
// every look-back finds its predecessor's prefix at once; the test checks the ranking, the scatter and the counts.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "ref_sort.cuh"

struct FlagSrc {  // element x is kept when keep[x] != 0
    const uint32_t *key;
    const uint8_t *keep;
    bool operator()(int x, uint32_t &k) const {
        if (!keep[x]) return false;
        k = key[x];
        return true;
    }
};

// Sorts the kept elements of key[0, n_in) stably by key; out_key / out_val get the sorted keys and their input
// positions, counts = {kept, kept with key < split}.  Returns the number of launches.
extern "C" int rs_sort(const uint32_t *key, const uint8_t *keep, int n_in, uint32_t split, int key_bits, int pass_blocks,
                       uint32_t *out_key, uint32_t *out_val, uint32_t *counts) {
    const size_t n = n_in > 0 ? (size_t)n_in : 1;
    const size_t ws_words = sizeof(DsortState) / 4 + dsort_status_words(n_in);
    uint32_t *ws = (uint32_t *)calloc(ws_words, 4);
    uint32_t *buf = (uint32_t *)malloc(4 * n * sizeof(uint32_t));
    DsortState *ss = reinterpret_cast<DsortState *>(ws);
    uint32_t *status = ws + sizeof(DsortState) / 4;
    memset(status, 0xAB, dsort_status_words(n_in) * 4);  // the passes' words must be cleared by the compaction
    memset(status, 0, (size_t)dsort_tiles(n_in) * 4);
    uint32_t *sk = nullptr, *sv = nullptr;
    const int launches = dsort_launch(FlagSrc{key, keep}, n_in, split, key_bits, buf, buf + n, buf + 2 * n, buf + 3 * n,
                                      ss, status, pass_blocks, nullptr, &sk, &sv);
    counts[0] = ss->n;
    counts[1] = ss->n_lo;
    memcpy(out_key, sk, ss->n * sizeof(uint32_t));
    memcpy(out_val, sv, ss->n * sizeof(uint32_t));
    free(buf);
    free(ws);
    return launches;
}
