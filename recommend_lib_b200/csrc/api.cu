// Handle lifecycle, error reporting, lazy-decay materialisation, timing and L2 window for libdaisy_b200.
#include <stdarg.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "ctx.cuh"
#include "ref_sort.cuh"

static thread_local char g_err[512] = "";

void daisy_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *daisy_last_error(void) { return g_err; }
extern "C" int daisy_abi_version(void) { return DAISY_ABI_VERSION; }

namespace {

template <class T>
int dalloc(T **p, size_t count) {
    *p = nullptr;
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void **)p, count * sizeof(T));
    if (e != cudaSuccess) {
        daisy_set_error("cudaMalloc of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
        return DAISY_ENOMEM;
    }
    return DAISY_OK;
}

int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

__global__ void k_scale2(float4 *__restrict__ a, size_t na4, float4 *__restrict__ b, size_t nb4, float c) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < na4 + nb4; i += stride) {
        float4 *p = (i < na4) ? a + i : b + (i - na4);
        float4 v = *p;
        v.x *= c; v.y *= c; v.z *= c; v.w *= c;
        *p = v;
    }
}

__global__ void k_err_reset(int *err) {
    err[0] = 0;
    err[1] = 0x7fffffff;
}

}  // namespace

extern "C" int daisy_create(daisy_handle_t *out, int device, int64_t user_num, int64_t item_num, int dim,
                            int64_t max_batch, unsigned flags) {
    DAISY_REQUIRE(out != nullptr, DAISY_EINVAL, "null out pointer");
    *out = nullptr;
    DAISY_REQUIRE(user_num > 0 && item_num > 0, DAISY_EINVAL, "user_num and item_num must be positive");
    DAISY_REQUIRE(user_num < 0x7fffffffLL && item_num < 0x7ffffffeLL, DAISY_EUNSUPPORTED, "row ids must fit int32");
    DAISY_REQUIRE(dim > 0 && dim <= 4096, DAISY_EUNSUPPORTED, "dim %d unsupported", dim);
    DAISY_REQUIRE(max_batch >= 0 && max_batch <= (1LL << 28), DAISY_EUNSUPPORTED, "max_batch must be in [0, 2^28]");
    // BPR kernels move rows as 128-bit vectors: they need dim % 4 == 0 and dim <= 512 (checked per call); a handle
    // created with max_batch == 0 carries no BPR workspace and serves the funk-SVD / eval entry points only.
    if (max_batch > 0)
        DAISY_REQUIRE(dim % 4 == 0 && dim <= 512, DAISY_EUNSUPPORTED,
                      "dim %d unsupported by the BPR step: need dim %% 4 == 0 and dim <= 512", dim);
    int ndev = 0;
    DAISY_CUDA(cudaGetDeviceCount(&ndev));
    DAISY_REQUIRE(device >= 0 && device < ndev, DAISY_EINVAL, "device %d not present (%d visible)", device, ndev);
    DeviceGuard g(device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", device);
    cudaDeviceProp prop;
    DAISY_CUDA(cudaGetDeviceProperties(&prop, device));
    DAISY_REQUIRE(prop.major == 10, DAISY_EUNSUPPORTED, "libdaisy_b200 is built for sm_100a only; device %d is sm_%d%d",
                  device, prop.major, prop.minor);

    daisy_ctx *h = (daisy_ctx *)calloc(1, sizeof(daisy_ctx));
    DAISY_REQUIRE(h != nullptr, DAISY_ENOMEM, "host allocation failed");
    h->device = device;
    h->num_sms = prop.multiProcessorCount;
    h->U = user_num;
    h->I = item_num;
    h->D = dim;
    h->maxB = max_batch;
    h->flags = flags;
    h->scale = 1.0;
    h->chunk = env_int("DAISY_CHUNK", 0);
    if (h->chunk > 32) h->chunk = 32;
    if (h->chunk < 0) h->chunk = 0;
    h->heavy_len = env_int("DAISY_HEAVY_LEN", 128);
    if (h->heavy_len < 8) h->heavy_len = 8;
    // a row is "very hot" above heavy_len contributions; at most 3B contributions exist per step
    h->heavy_cap = (int)(3 * max_batch / h->heavy_len) + 4;
    h->mid_cap = max_batch < 131072 ? max_batch : 131072;
    {   // small-batch path: rows with more than 16 (DAISY_SMALL_SLICE, step_kernels.cuh) contributions, slices of 16
        const int64_t sb = h->mid_cap;
        h->longs_cap = (int)(3 * sb / 16) + 4;
        if (h->longs_cap < h->heavy_cap) h->longs_cap = h->heavy_cap;  // the general path lists rows longer than heavy_len
        h->slice_cap = (int)(3 * max_batch / DAISY_SLICE) + h->heavy_cap + 4;
        if (h->slice_cap < 2 * h->longs_cap) h->slice_cap = 2 * h->longs_cap;
    }
    h->pipeline = env_int("DAISY_PIPELINE", 1) ? 1 : 0;
    h->main_stages = env_int("DAISY_MAIN_STAGES", 3);
    if (h->main_stages < 0) h->main_stages = 0;
    if (h->main_stages > 16) h->main_stages = 16;
    h->inputs_ready = 0;
    h->seg_win = env_int("DAISY_SEG_WIN", 32) == 16 ? 16 : 32;
    h->mid_max = env_int("DAISY_MID_MAX", 65536);  // measured: above ~100 k triples the general pipeline (graph-replayed) is faster
    if (h->mid_max < 0) h->mid_max = 0;
    if (h->mid_max > h->mid_cap) h->mid_max = h->mid_cap;
    h->graph_max_b = env_int("DAISY_GRAPH_MAX_B", 262144);
    if (h->graph_max_b < 0) h->graph_max_b = 0;
    h->merged_sort = env_int("DAISY_MERGED_SORT", -1);
    h->main_max_blocks = env_int("DAISY_MAIN_MAX_BLOCKS", 0);
    h->small_max = env_int("DAISY_SMALL_MAX", DAISY_SMALL_CAP);
    if (h->small_max < 0) h->small_max = 0;
    if (h->small_max > DAISY_SMALL_CAP) h->small_max = DAISY_SMALL_CAP;

    const size_t B = (size_t)max_batch;
    int rc = DAISY_OK;
#define A(ptr, n) if (!rc) rc = dalloc(&h->ptr, (n))
    A(err, 2);
    if (B > 0) {
        A(triples, DAISY_NSETS * 3 * B);
        for (int i = 0; i < DAISY_NSETS; ++i) {
            A(book[i].st, 3 * B);
            A(book[i].ukey_s, B); A(book[i].qkey_s, 2 * B);
            A(book[i].uslot, B); A(book[i].jslot, B); A(book[i].islot, B);
            A(book[i].longs, 2 + 5 * (size_t)h->longs_cap);
            A(book[i].counts, 2);
        }
        A(key_in, 3 * B); A(val_in, 3 * B); A(val_out, 3 * B); A(key_out, 3 * B);
        A(ukey_in, B); A(uval_in, B); A(uval_out, B);
        A(ikey_in, B); A(ikey_out, B); A(ival_in, B); A(ival_out, B);
        A(stageU, B * dim);
        A(stageQ, 2 * B * dim);
        A(stage2, (size_t)h->slice_cap * dim);
        A(loss_part, B);
        A(ticket, (size_t)h->longs_cap);
        A(mid_buf, 4 * 3 * (size_t)h->mid_cap);
        if (h->merged_sort != 0) {  // item refs name at most max(I, 2B) rows: the sharded step's cache rows stand in for I
            h->ref_rows = user_num + (item_num > 2 * max_batch ? item_num : 2 * max_batch);
            A(ref_ws, sizeof(DsortState) / 4 + 2 * (size_t)((h->ref_rows + 31) / 32) + dsort_status_words(3 * max_batch));
        }
    }
#undef A
    if (!rc && B > 0) {
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, (uint32_t *)nullptr, (uint32_t *)nullptr, (uint32_t *)nullptr,
                                        (uint32_t *)nullptr, (int)(3 * B), 0, 32, (cudaStream_t)0);
        size_t need_scan = 0;  // the sharded bookkeeping also scans 2B flags (step_kernels.cuh)
        cub::DeviceScan::InclusiveSum(nullptr, need_scan, (uint32_t *)nullptr, (uint32_t *)nullptr, (int)(2 * B),
                                      (cudaStream_t)0);
        if (need_scan > need) need = need_scan;
        h->cub_tmp_bytes = need + 4096;
        rc = dalloc((char **)&h->cub_tmp, h->cub_tmp_bytes);
    }
    if (!rc && cudaMallocHost((void **)&h->err_host, 2 * sizeof(int)) != cudaSuccess) {
        daisy_set_error("cudaMallocHost failed");
        rc = DAISY_ENOMEM;
    }
    if (!rc) {
        if (B > 0) {
            for (int i = 0; i < DAISY_NSETS; ++i) cudaMemset(h->book[i].islot, 0xFF, B * sizeof(uint32_t));
            cudaMemset(h->ticket, 0, (size_t)h->longs_cap * sizeof(uint32_t));
        }
        k_err_reset<<<1, 1>>>(h->err);
        for (int i = 0; i <= PH_COUNT; ++i) cudaEventCreate(&h->ev[i]);
        // highest priority: the short bookkeeping kernels of step n+1 must get SM slots while the long
        // bandwidth-bound kernels of step n are still dispatching blocks
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        cudaStreamCreateWithPriority(&h->side_stream, cudaStreamNonBlocking,
                                     env_int("DAISY_BOOK_LOW_PRIORITY", 0) ? prio_lo : prio_hi);
        // DAISY_BOOK_SMS = n > 0: the bookkeeping stream gets n SMs of its own and the table kernels the rest
        // (partition.cu); a driver that cannot partition leaves the shared-SM pipeline in place
        if (B > 0 && h->pipeline && env_int("DAISY_BOOK_SMS", 0) > 0) {
            if (daisy_partition_create(h, env_int("DAISY_BOOK_SMS", 0)) == DAISY_OK && h->part_ok) {
                cudaStreamDestroy(h->side_stream);
                h->side_stream = h->part_book_stream;
            } else if (env_int("DAISY_BOOK_SMS_REQUIRED", 0)) {
                rc = DAISY_EUNSUPPORTED;
            }
        }
        cudaEventCreateWithFlags(&h->ev_call, cudaEventDisableTiming);
        for (int i = 0; i < DAISY_NSETS; ++i) {
            cudaEventCreateWithFlags(&h->book[i].ready, cudaEventDisableTiming);
            cudaEventCreateWithFlags(&h->book[i].freed, cudaEventDisableTiming);
            cudaEventCreateWithFlags(&h->book[i].copied, cudaEventDisableTiming);
        }
        if (B > 0 && env_int("DAISY_COPY_STREAM", 1)) cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
        if (cudaDeviceSynchronize() != cudaSuccess) {
            daisy_set_error("workspace initialisation failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = DAISY_ECUDA;
        }
    }
    if (rc) {
        daisy_destroy(h);
        return rc;
    }
    *out = h;
    return DAISY_OK;
}

extern "C" int daisy_destroy(daisy_handle_t h) {
    if (!h) return DAISY_OK;
    DeviceGuard g(h->device);
    cudaDeviceSynchronize();
    daisy_shard_free(h);
    void *ptrs[] = {h->triples, h->key_in, h->val_in, h->val_out, h->ukey_in, h->uval_in, h->uval_out, h->ikey_in,
                    h->ikey_out, h->ival_in, h->ival_out, h->stageU, h->stageQ, h->stage2, h->loss_part, h->key_out,
                    h->err, h->cub_tmp, h->ticket, h->mid_buf, h->gradP, h->gradQ, h->wpart, h->scores, h->sel_hist, h->own_key, h->own_key_s, h->own_val, h->own_val_s,
                    h->own_tmp, h->ref_ws};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (int i = 0; i < DAISY_NSETS; ++i) {
        void *bp[] = {h->book[i].st, h->book[i].ukey_s, h->book[i].qkey_s, h->book[i].uslot, h->book[i].jslot,
                      h->book[i].islot, h->book[i].longs, h->book[i].counts};
        for (void *p : bp)
            if (p) cudaFree(p);
        if (h->book[i].ready) cudaEventDestroy(h->book[i].ready);
        if (h->book[i].freed) cudaEventDestroy(h->book[i].freed);
        if (h->book[i].copied) cudaEventDestroy(h->book[i].copied);
    }
    for (int i = 0; i < DAISY_MAX_BGRAPH; ++i)
        if (h->bgraph[i].exec) cudaGraphExecDestroy(h->bgraph[i].exec);
    for (int i = 0; i < 3; ++i)
        if (h->tc_ev[i]) cudaEventDestroy(h->tc_ev[i]);
    if (h->pool_state == 1) cudaMemPoolDestroy(h->pool);
    if (h->err_host) cudaFreeHost(h->err_host);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->part_ok) {
        h->side_stream = nullptr;  // it is the partition's bookkeeping stream
        daisy_partition_destroy(h);
    }
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->ev_call) cudaEventDestroy(h->ev_call);
    for (int i = 0; i <= PH_COUNT; ++i)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    for (int i = 0; i < 2 * DAISY_EVPOOL; ++i)
        if (h->evpool[i]) cudaEventDestroy(h->evpool[i]);
    for (int i = 0; i < 4 * DAISY_TRACE_STEPS; ++i)
        if (h->tr_ev[i]) cudaEventDestroy(h->tr_ev[i]);
    free(h);
    return DAISY_OK;
}

extern "C" int daisy_check(daisy_handle_t h, daisy_stream_t stream) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DeviceGuard g(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    DAISY_CUDA(cudaMemcpyAsync(h->err_host, h->err, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
    DAISY_CUDA(cudaStreamSynchronize(s));
    if (h->err_host[0]) {
        const int pos = h->err_host[1];
        const int bits = h->err_host[0];
        k_err_reset<<<1, 1, 0, s>>>(h->err);
        cudaStreamSynchronize(s);
        if (bits & 16) {
            daisy_set_error("sharded step: a peer rank did not reach the barrier within 20 s (ranks out of step or a peer died)");
            return DAISY_ECUDA;
        }
        if (bits & 64) {
            daisy_set_error("negative sampler: a user has no item left to draw as a negative (4096 rejected draws)");
            return DAISY_EINDEX;
        }
        if (bits & 32) {
            daisy_set_error("sharded step: a receive region overflowed");
            return DAISY_ECUDA;
        }
        if (bits & 256) {
            daisy_set_error("daisy_topk_full: the tensor-core filter pipeline timed out (an mbarrier never completed)");
            return DAISY_ECUDA;
        }
        daisy_set_error("index out of range in self (first offending position %d; user ids must be < %lld, item ids < %lld)",
                        pos, (long long)h->U, (long long)h->I);
        return DAISY_EINDEX;
    }
    return DAISY_OK;
}

extern "C" int daisy_get_scale(daisy_handle_t h, double *c) {
    DAISY_REQUIRE(h && c, DAISY_EINVAL, "null argument");
    *c = h->scale;
    return DAISY_OK;
}

extern "C" int daisy_set_scale(daisy_handle_t h, double c) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DAISY_REQUIRE(c > 0.0, DAISY_EINVAL, "scale must be positive");
    h->scale = c;
    return DAISY_OK;
}

extern "C" int daisy_materialize(daisy_handle_t h, float *P, float *Q, daisy_stream_t stream) {
    DAISY_REQUIRE(h && P && Q, DAISY_EINVAL, "null argument");
    if (h->scale == 1.0) return DAISY_OK;
    DeviceGuard g(h->device);
    const size_t na4 = (size_t)h->U * h->D / 4, nb4 = (size_t)h->I * h->D / 4;
    const size_t want = (na4 + nb4 + 255) / 256;
    const int grid = (int)(want < (size_t)h->num_sms * 16 ? want : (size_t)h->num_sms * 16);
    k_scale2<<<grid, 256, 0, (cudaStream_t)stream>>>((float4 *)P, na4, (float4 *)Q, nb4, (float)h->scale);
    DAISY_LAUNCH_CHECK(h);
    h->scale = 1.0;
    return DAISY_OK;
}

extern "C" int daisy_trace(daisy_handle_t h, int on, double *ms, int cap, int *n_steps) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DeviceGuard g(h->device);
    if (ms && n_steps) {  // dump what was recorded: 4 offsets (ms from the first event) per step
        DAISY_CUDA(cudaDeviceSynchronize());
        int n = h->tr_n < cap / 4 ? h->tr_n : cap / 4;
        for (int i = 0; i < 4 * n; ++i) {
            float v = 0.f;
            DAISY_CUDA(cudaEventElapsedTime(&v, h->tr_ev[0], h->tr_ev[i]));
            ms[i] = v;
        }
        *n_steps = n;
    }
    if (on && !h->tr_ev[0])
        for (int i = 0; i < 4 * DAISY_TRACE_STEPS; ++i) DAISY_CUDA(cudaEventCreate(&h->tr_ev[i]));
    h->trace = on ? 1 : 0;
    h->tr_n = 0;
    return DAISY_OK;
}

extern "C" int daisy_set_inputs_ready(daisy_handle_t h, int on) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    h->inputs_ready = on ? 1 : 0;
    return DAISY_OK;
}

extern "C" int daisy_launch_count(daisy_handle_t h, int64_t *n) {
    DAISY_REQUIRE(h && n, DAISY_EINVAL, "null argument");
    *n = h->launches;
    return DAISY_OK;
}

extern "C" int daisy_set_timing(daisy_handle_t h, int mode) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DAISY_REQUIRE(mode >= 0 && mode <= 2, DAISY_EINVAL, "timing mode must be 0, 1 or 2");
    DeviceGuard g(h->device);
    DAISY_CUDA(cudaDeviceSynchronize());  // mode 2 moves the bookkeeping onto the caller's stream: drain first
    if (mode == 1 && !h->evpool[0])
        for (int i = 0; i < 2 * DAISY_EVPOOL; ++i) DAISY_CUDA(cudaEventCreate(&h->evpool[i]));
    h->timing = mode;
    h->ev_pending = 0;
    h->pool_used = 0;
    h->timed_steps = 0;
    h->main_ms_sum = 0.0;
    h->main_count = 0;
    for (int i = 0; i < PH_COUNT; ++i) h->phase_ms_sum[i] = 0.0;
    return DAISY_OK;
}

// timing == 1: average duration of the main fused kernel over the steps since daisy_set_timing(h, 1).
extern "C" int daisy_main_kernel_ms(daisy_handle_t h, double *avg_ms, int64_t *count) {
    DAISY_REQUIRE(h && avg_ms && count, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    for (int i = 0; i < h->pool_used; ++i) {
        DAISY_CUDA(cudaEventSynchronize(h->evpool[2 * i + 1]));
        float ms = 0.f;
        DAISY_CUDA(cudaEventElapsedTime(&ms, h->evpool[2 * i], h->evpool[2 * i + 1]));
        h->main_ms_sum += ms;
        h->main_count++;
    }
    h->pool_used = 0;
    *count = h->main_count;
    *avg_ms = h->main_count ? h->main_ms_sum / (double)h->main_count : 0.0;
    return DAISY_OK;
}

// timing == 2: average duration (ms) of every phase of the step (enum in ctx.cuh), n <= PH_COUNT.
extern "C" int daisy_phase_ms(daisy_handle_t h, double *avg_ms, int n, int64_t *steps) {
    DAISY_REQUIRE(h && avg_ms && steps, DAISY_EINVAL, "null argument");
    DeviceGuard g(h->device);
    if (h->ev_pending) {
        DAISY_CUDA(cudaEventSynchronize(h->ev[PH_COUNT]));
        for (int ph = 0; ph < PH_COUNT; ++ph) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, h->ev[ph], h->ev[ph + 1]);
            h->phase_ms_sum[ph] += ms;
        }
        h->timed_steps++;
        h->ev_pending = 0;
    }
    for (int i = 0; i < n && i < PH_COUNT; ++i)
        avg_ms[i] = h->timed_steps ? h->phase_ms_sum[i] / (double)h->timed_steps : 0.0;
    *steps = h->timed_steps;
    return DAISY_OK;
}

extern "C" int daisy_last_step_timing(daisy_handle_t h, float *ms_main_kernel, float *ms_total) {
    DAISY_REQUIRE(h && ms_main_kernel && ms_total, DAISY_EINVAL, "null argument");
    double ph[PH_COUNT];
    int64_t steps = 0;
    int rc = daisy_phase_ms(h, ph, PH_COUNT, &steps);
    if (rc) return rc;
    double tot = 0.0;
    for (int i = 0; i < PH_COUNT; ++i) tot += ph[i];
    *ms_main_kernel = (float)ph[PH_MAIN];
    *ms_total = (float)tot;
    return DAISY_OK;
}

extern "C" int daisy_set_l2_window(daisy_handle_t h, const float *Q, int64_t n_rows, float hit_ratio,
                                   daisy_stream_t stream) {
    DAISY_REQUIRE(h != nullptr, DAISY_EINVAL, "null handle");
    DeviceGuard g(h->device);
    cudaDeviceProp prop;
    DAISY_CUDA(cudaGetDeviceProperties(&prop, h->device));
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (n_rows > 0 && Q) {
        size_t bytes = (size_t)n_rows * h->D * sizeof(float);
        if (bytes > (size_t)prop.accessPolicyMaxWindowSize) bytes = (size_t)prop.accessPolicyMaxWindowSize;
        size_t carve = bytes < (size_t)prop.persistingL2CacheMaxSize ? bytes : (size_t)prop.persistingL2CacheMaxSize;
        DAISY_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
        attr.accessPolicyWindow.base_ptr = (void *)Q;
        attr.accessPolicyWindow.num_bytes = bytes;
        attr.accessPolicyWindow.hitRatio = hit_ratio;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    } else {
        attr.accessPolicyWindow.num_bytes = 0;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    }
    DAISY_CUDA(cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    if (n_rows <= 0) cudaCtxResetPersistingL2Cache();
    return DAISY_OK;
}
