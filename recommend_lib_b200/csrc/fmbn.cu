// BPR-FM with two one-hot features at the reference script's DEFAULTS: batch norm + dropout on the FM vector
// (BPRFMRecommender.py:45-80 model, :116-125 defaults, :214-219 step; SURVEY.md section 8f row N3).
//
// Parity: tests/test_bprfm_bn_gpu.py (golden run of the unmodified reference class + oracle/bprfm_oracle.py: BPRFMFull
// on seeded shapes); the same translation unit also runs under the host emulation of tests/emu.
//
// With features = [user, user_num + item] and values 1 the bi-interaction vector is x = e_u (.) e_i.  BatchNorm1d in
// training mode couples the samples of a batch through per-factor column statistics, so one step is a short chain of
// passes over the gathered rows (the tables are L2-resident at the script's sizes; this first version is written for
// clarity: every pass is a plain kernel, every reduction has a fixed order => bit-reproducible):
//   k_fm_x        x_i = e_u (.) e_i, x_j = e_u (.) e_j                                   -> X [2][B][F]
//   k_fm_stats_sum / _var / _finish   per (call, factor): mean and biased variance over the batch (double; the batch
//                 is cut into FM_Z slices, one block each, partials added in slice order)   -> mu, var, inv
//   k_fm_score    xhat, z = gamma xhat + beta, dropout mask, pred_i - pred_j, s_b, loss    -> s [B], loss partials
//   k_fm_colsums_part / _finish   per (call, factor): sum_b dz, sum_b dz xhat (double, same slicing)  -> c1, c2, d gamma, d beta
//   k_fm_grad     dx = inv (gamma dz - c1 - xhat c2); row-gradient contributions           -> contrib [3B][F+1], keys
//   cub sort      contributions grouped by feature row (stable: ascending triple order inside a row)
//   k_fm_apply_slices / k_fm_apply   a row's contributions summed in slices of FM_SLICE (one warp each), then one warp
//                 per row adds its slices in order + Adagrad on the row and its bias
//   k_fm_bn_step  Adagrad on gamma / beta, running statistics (positive call first, then negative), loss
// The user bias and bias_ cancel in pred_i - pred_j: their gradient is exactly zero here (the reference's is -s + s,
// zero up to rounding).
#include <cub/cub.cuh>

#include "ctx.cuh"

namespace {

constexpr int FM_MAX_F = 255;  // k_fm_apply keeps (F + 1) / 32 accumulators per lane in registers
constexpr int FM_Z = 64;       // batch slices of the column reductions (one block per slice and 32 factors)
constexpr int FM_SLICE = 32;   // sorted contributions per slice of k_fm_apply_slices

struct FmScratch {
    float *X, *s, *lossp, *mu, *var, *inv, *c1, *c2, *contrib;
    double *part;    // [FM_Z][2 calls][F][2] partial column sums of the batch slices (k_fm_stats_*, k_fm_colsums_*)
    float *spart;    // [3B][F + 1] slice sums of k_fm_apply_slices (indexed by the slice's first sorted position)
    double *A, *Bs;  // per (call, factor) sums of dz and dz * xhat: the two calls' sums nearly cancel in d beta, so they
                     // stay double until they have been added (a float here costs 1e-4 of d beta at batch 333)
    uint32_t *kin, *kout, *vin, *vout;
    void *cub;
    size_t cub_bytes, total;
};

// Temporary storage of cub::DeviceRadixSort::SortPairs on n (uint32, uint32) pairs: the alternate key and value buffers
// plus histograms and alignment.  A bound, not a query, so that sizing needs no device; CUB refuses a buffer that is
// too small (reported as an error by the step), it never overruns one.
static size_t fm_sort_bytes(int64_t n) { return (size_t)n * 16 + ((size_t)1 << 20); }

static void fm_carve(char *base, int64_t B, int F, FmScratch &w) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char *p = base ? base + off : nullptr;
        off += (bytes + 255) / 256 * 256;
        return p;
    };
    const size_t b = (size_t)B, f = (size_t)F;
    w.X = (float *)take(2 * b * f * 4);
    w.s = (float *)take(b * 4);
    w.lossp = (float *)take(b * 4);
    w.mu = (float *)take(2 * f * 4);
    w.var = (float *)take(2 * f * 4);
    w.inv = (float *)take(2 * f * 4);
    w.A = (double *)take(2 * f * 8);
    w.Bs = (double *)take(2 * f * 8);
    w.c1 = (float *)take(2 * f * 4);
    w.c2 = (float *)take(2 * f * 4);
    w.contrib = (float *)take(3 * b * (f + 1) * 4);
    w.part = (double *)take((size_t)FM_Z * 2 * f * 2 * 8);
    w.spart = (float *)take(3 * b * (f + 1) * 4);
    w.kin = (uint32_t *)take(3 * b * 4);
    w.kout = (uint32_t *)take(3 * b * 4);
    w.vin = (uint32_t *)take(3 * b * 4);
    w.vout = (uint32_t *)take(3 * b * 4);
    w.cub_bytes = fm_sort_bytes(3 * B);
    w.cub = take(w.cub_bytes);
    w.total = off;
}

__device__ __forceinline__ void fm_ids(const int32_t *__restrict__ tri, int b, uint32_t U, uint32_t I, uint32_t &u,
                                       uint32_t &i, uint32_t &j, bool &bad) {
    u = (uint32_t)tri[3 * (size_t)b];
    i = (uint32_t)tri[3 * (size_t)b + 1];
    j = (uint32_t)tri[3 * (size_t)b + 2];
    bad = (u >= U) | (i >= I) | (j >= I);
    if (bad) {  // never fault: park the triple on row 0, the error flag tells the caller
        u = u < U ? u : 0u;
        i = i < I ? i : 0u;
        j = j < I ? j : 0u;
    }
}

// one warp per triple
__global__ void __launch_bounds__(256) k_fm_x(const float *__restrict__ E, const int32_t *__restrict__ tri, int B, int F,
                                               uint32_t U, uint32_t I, float *__restrict__ X, int *err) {
    const int lane = threadIdx.x & 31;
    const int b = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (b >= B) return;
    uint32_t u, i, j;
    bool bad;
    fm_ids(tri, b, U, I, u, i, j, bad);
    if (bad && lane == 0) {
        atomicOr(&err[0], 1);
        atomicMin(&err[1], b);
    }
    const float *eu = E + (size_t)u * F, *ei = E + (size_t)(U + i) * F, *ej = E + (size_t)(U + j) * F;
    float *xi = X + (size_t)b * F, *xj = X + ((size_t)B + b) * F;
    for (int f = lane; f < F; f += 32) {
        const float a = eu[f];
        xi[f] = a * ei[f];
        xj[f] = a * ej[f];
    }
}

// Column statistics of the batch (two-pass mean / variance in double, every sum in a fixed order).  The first version
// walked the whole batch in ONE block per 32 factors -- 4 blocks on the GPU, 65 us at batch 4 096, and the same shape
// cost k_fm_colsums 283 us (profiles/r02u_launches_bprfm_bn_summary.md).  Now: grid (ceil(F / 32), 2 calls, FM_Z batch
// slices), block (32 factors, 8 row groups); a slice block leaves its partial sum in `part`, and whoever needs the
// total adds the FM_Z partials in slice order (identical in every block).
__device__ __forceinline__ void fm_slice(int B, int z, int &b0, int &b1) {
    const int per = (B + FM_Z - 1) / FM_Z;
    b0 = z * per;
    b1 = min(B, b0 + per);
}
__device__ __forceinline__ double fm_total(const double *__restrict__ part, int c, int f, int F, int which) {
    double t = 0.0;
    for (int z = 0; z < FM_Z; ++z) t += part[(((size_t)z * 2 + c) * F + f) * 2 + which];
    return t;
}

__global__ void __launch_bounds__(256) k_fm_stats_sum(const float *__restrict__ X, int B, int F, double *__restrict__ part) {
    __shared__ double sh[8][33];
    const int tx = threadIdx.x, ty = threadIdx.y, f = blockIdx.x * 32 + tx, c = blockIdx.y, z = blockIdx.z;
    const float *x = X + (size_t)c * B * F;
    int b0, b1;
    fm_slice(B, z, b0, b1);
    double a = 0.0;
    if (f < F)
        for (int b = b0 + ty; b < b1; b += 8) a += (double)x[(size_t)b * F + f];
    sh[ty][tx] = a;
    __syncthreads();
    if (ty == 0 && f < F) {
        double m = 0.0;
        for (int k = 0; k < 8; ++k) m += sh[k][tx];
        part[(((size_t)z * 2 + c) * F + f) * 2 + 0] = m;
    }
}

__global__ void __launch_bounds__(256) k_fm_stats_var(const float *__restrict__ X, int B, int F, double *__restrict__ part) {
    __shared__ double sh[8][33];
    const int tx = threadIdx.x, ty = threadIdx.y, f = blockIdx.x * 32 + tx, c = blockIdx.y, z = blockIdx.z;
    const float *x = X + (size_t)c * B * F;
    int b0, b1;
    fm_slice(B, z, b0, b1);
    double v = 0.0;
    if (f < F) {
        const double m = fm_total(part, c, f, F, 0) / (double)B;
        for (int b = b0 + ty; b < b1; b += 8) {
            const double d = (double)x[(size_t)b * F + f] - m;
            v += d * d;
        }
    }
    sh[ty][tx] = v;
    __syncthreads();
    if (ty == 0 && f < F) {
        double t = 0.0;
        for (int k = 0; k < 8; ++k) t += sh[k][tx];
        part[(((size_t)z * 2 + c) * F + f) * 2 + 1] = t;
    }
}

__global__ void k_fm_stats_finish(const double *__restrict__ part, int B, int F, float bn_eps, float *__restrict__ mu,
                                  float *__restrict__ var, float *__restrict__ inv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * F) return;
    const int c = i / F, f = i - c * F;
    const double m = fm_total(part, c, f, F, 0) / (double)B;
    const double sv = fm_total(part, c, f, F, 1) / (double)B;  // biased variance normalises (nn.BatchNorm1d, training mode)
    mu[i] = (float)m;
    var[i] = (float)sv;
    inv[i] = (float)(1.0 / sqrt(sv + (double)bn_eps));
}

// one warp per triple: prediction difference, s_b = sigmoid(-(pred_i - pred_j)), loss
__global__ void __launch_bounds__(256) k_fm_score(const float *__restrict__ X, const float *__restrict__ bias,
                                                   const int32_t *__restrict__ tri, int B, int F, uint32_t U, uint32_t I,
                                                   const float *__restrict__ mu, const float *__restrict__ inv,
                                                   const float *__restrict__ gamma, const float *__restrict__ beta,
                                                   const float *__restrict__ mask_i, const float *__restrict__ mask_j,
                                                   float *__restrict__ s_out, float *__restrict__ lossp) {
    const int lane = threadIdx.x & 31;
    const int b = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (b >= B) return;
    uint32_t u, i, j;
    bool bad;
    fm_ids(tri, b, U, I, u, i, j, bad);
    const float *xi = X + (size_t)b * F, *xj = X + ((size_t)B + b) * F;
    float d = 0.f;
    for (int f = lane; f < F; f += 32) {
        float zi = gamma[f] * ((xi[f] - mu[f]) * inv[f]) + beta[f];
        float zj = gamma[f] * ((xj[f] - mu[F + f]) * inv[F + f]) + beta[f];
        if (mask_i) zi *= mask_i[(size_t)b * F + f];
        if (mask_j) zj *= mask_j[(size_t)b * F + f];
        d += zi - zj;
    }
    d = warp_sum(d);
    if (lane == 0) {
        const float x = d + bias[U + i] - bias[U + j];
        s_out[b] = 1.f / (1.f + expf(x));
        lossp[b] = fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
    }
}

// grid (ceil(F / 32), 2 calls), block (32, 8): column sums of dz and dz * xhat in double, fixed order
__global__ void __launch_bounds__(256) k_fm_colsums_part(const float *__restrict__ X, const float *__restrict__ s, int B, int F,
                                                          const float *__restrict__ mu, const float *__restrict__ inv,
                                                          const float *__restrict__ mask_i, const float *__restrict__ mask_j,
                                                          double *__restrict__ part) {
    __shared__ double shA[8][33], shB[8][33];
    const int tx = threadIdx.x, ty = threadIdx.y, f = blockIdx.x * 32 + tx, c = blockIdx.y, z = blockIdx.z;
    const float *x = X + (size_t)c * B * F;
    const float *mask = c ? mask_j : mask_i;
    const float sign = c ? 1.f : -1.f;  // d loss / d pred_i = -s, d loss / d pred_j = +s
    int b0, b1;
    fm_slice(B, z, b0, b1);
    double a = 0.0, bs = 0.0;
    if (f < F) {
        const float m = mu[c * F + f], iv = inv[c * F + f];
        for (int b = b0 + ty; b < b1; b += 8) {
            float dz = sign * s[b];
            if (mask) dz *= mask[(size_t)b * F + f];
            const float xh = (x[(size_t)b * F + f] - m) * iv;
            a += (double)dz;
            bs += (double)dz * (double)xh;
        }
    }
    shA[ty][tx] = a;
    shB[ty][tx] = bs;
    __syncthreads();
    if (ty == 0 && f < F) {
        double ta = 0.0, tb = 0.0;
        for (int k = 0; k < 8; ++k) {
            ta += shA[k][tx];
            tb += shB[k][tx];
        }
        part[(((size_t)z * 2 + c) * F + f) * 2 + 0] = ta;
        part[(((size_t)z * 2 + c) * F + f) * 2 + 1] = tb;
    }
}

__global__ void k_fm_colsums_finish(const double *__restrict__ part, int B, int F, const float *__restrict__ gamma,
                                    double *__restrict__ A, double *__restrict__ Bs, float *__restrict__ c1,
                                    float *__restrict__ c2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * F) return;
    const int c = i / F, f = i - c * F;
    const double ta = fm_total(part, c, f, F, 0), tb = fm_total(part, c, f, F, 1);
    A[i] = ta;
    Bs[i] = tb;
    c1[i] = (float)((double)gamma[f] * ta / (double)B);   // mean_b(d xhat)
    c2[i] = (float)((double)gamma[f] * tb / (double)B);   // mean_b(d xhat * xhat)
}

// one warp per triple: BN backward per element, contributions of the triple to its three feature rows
__global__ void __launch_bounds__(256) k_fm_grad(const float *__restrict__ E, const float *__restrict__ X,
                                                  const float *__restrict__ s, const int32_t *__restrict__ tri, int B, int F,
                                                  uint32_t U, uint32_t I, const float *__restrict__ mu,
                                                  const float *__restrict__ inv, const float *__restrict__ gamma,
                                                  const float *__restrict__ c1, const float *__restrict__ c2,
                                                  const float *__restrict__ mask_i, const float *__restrict__ mask_j,
                                                  float *__restrict__ contrib, uint32_t *__restrict__ kin,
                                                  uint32_t *__restrict__ vin) {
    const int lane = threadIdx.x & 31;
    const int b = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (b >= B) return;
    uint32_t u, i, j;
    bool bad;
    fm_ids(tri, b, U, I, u, i, j, bad);
    const float *eu = E + (size_t)u * F, *ei = E + (size_t)(U + i) * F, *ej = E + (size_t)(U + j) * F;
    const float *xi = X + (size_t)b * F, *xj = X + ((size_t)B + b) * F;
    const float sb = s[b];
    const size_t W = (size_t)F + 1;
    float *gu = contrib + (3 * (size_t)b) * W, *gi = gu + W, *gj = gi + W;
    for (int f = lane; f < F; f += 32) {
        float dzi = -sb, dzj = sb;
        if (mask_i) dzi *= mask_i[(size_t)b * F + f];
        if (mask_j) dzj *= mask_j[(size_t)b * F + f];
        const float g = gamma[f];
        const float xhi = (xi[f] - mu[f]) * inv[f], xhj = (xj[f] - mu[F + f]) * inv[F + f];
        const float dxi = inv[f] * (g * dzi - c1[f] - xhi * c2[f]);
        const float dxj = inv[F + f] * (g * dzj - c1[F + f] - xhj * c2[F + f]);
        const float a = eu[f];
        gu[f] = dxi * ei[f] + dxj * ej[f];
        gi[f] = dxi * a;
        gj[f] = dxj * a;
    }
    if (lane == 0) {
        gu[F] = 0.f;   // user bias: -s + s
        gi[F] = -sb;
        gj[F] = sb;
        kin[3 * (size_t)b] = u;
        kin[3 * (size_t)b + 1] = U + i;
        kin[3 * (size_t)b + 2] = U + j;
        vin[3 * (size_t)b] = 3u * (uint32_t)b;
        vin[3 * (size_t)b + 1] = 3u * (uint32_t)b + 1u;
        vin[3 * (size_t)b + 2] = 3u * (uint32_t)b + 2u;
    }
}

// A row's contributions are consecutive in the sorted list; they are summed in slices so that a hot row (a Zipf item takes
// hundreds of a batch's 3B contributions) is not one warp's serial walk (292 us at batch 4 096, first version).  A slice
// starts at every row head and at every sorted position that is a multiple of FM_SLICE, and ends where the next one starts.
// k_fm_apply_slices: one warp per sorted position; the warp at a slice start sums the slice in sorted (= triple) order.
__global__ void __launch_bounds__(256) k_fm_apply_slices(const uint32_t *__restrict__ kout, const uint32_t *__restrict__ vout,
                                                          int n, const float *__restrict__ contrib, int F,
                                                          float *__restrict__ spart) {
    const int lane = threadIdx.x & 31;
    const int p = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (p >= n) return;
    const uint32_t row = kout[p];
    if (p % FM_SLICE != 0 && kout[p - 1] == row) return;  // warp-uniform: inside a slice
    const size_t W = (size_t)F + 1;
    const int stop = min(n, (p / FM_SLICE + 1) * FM_SLICE);
    float acc[(FM_MAX_F + 1 + 31) / 32];
#pragma unroll
    for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) acc[k] = 0.f;
#pragma unroll 4  // independent index -> row chains: let the scheduler put several rows in flight
    for (int q = p; q < stop && kout[q] == row; ++q) {
        const float *g = contrib + (size_t)vout[q] * W;
#pragma unroll
        for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) {
            const int f = lane + 32 * k;
            if (f <= F) acc[k] += g[f];
        }
    }
    float *dst = spart + (size_t)p * W;
#pragma unroll
    for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) {
        const int f = lane + 32 * k;
        if (f <= F) dst[f] = acc[k];
    }
}

// k_fm_apply: the warp at the FIRST contribution of a row adds the row's slice sums in slice order and applies Adagrad:
// state_sum += g^2, w -= lr g / (sqrt(state_sum) + eps)  (torch.optim.Adagrad, lr_decay 0)
__global__ void __launch_bounds__(256) k_fm_apply(const uint32_t *__restrict__ kout, int n, const float *__restrict__ spart, int F,
                                                   float *__restrict__ E, float *__restrict__ bias, float *__restrict__ accE,
                                                   float *__restrict__ accb, float lr, float eps) {
    const int lane = threadIdx.x & 31;
    const int p = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (p >= n) return;
    const uint32_t row = kout[p];
    if (p > 0 && kout[p - 1] == row) return;  // warp-uniform: not the head of its row
    const size_t W = (size_t)F + 1;
    float acc[(FM_MAX_F + 1 + 31) / 32];
#pragma unroll
    for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) acc[k] = 0.f;
    for (int q = p; q < n && kout[q] == row; q = (q / FM_SLICE + 1) * FM_SLICE) {  // the row's slice starts
        const float *g = spart + (size_t)q * W;
#pragma unroll
        for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) {
            const int f = lane + 32 * k;
            if (f <= F) acc[k] += g[f];
        }
    }
#pragma unroll
    for (int k = 0; k < (FM_MAX_F + 1 + 31) / 32; ++k) {
        const int f = lane + 32 * k;
        if (f > F) continue;
        const float g = acc[k];
        if (f < F) {
            const size_t e = (size_t)row * F + f;
            const float a = accE[e] + g * g;
            accE[e] = a;
            E[e] -= lr * g / (sqrtf(a) + eps);
        } else {
            const float a = accb[row] + g * g;
            accb[row] = a;
            bias[row] -= lr * g / (sqrtf(a) + eps);
        }
    }
}

// one block: Adagrad on gamma / beta, running statistics (two _out calls per step: positive, then negative), loss
__global__ void __launch_bounds__(256) k_fm_bn_step(int B, int F, const float *__restrict__ mu, const float *__restrict__ var,
                                                     const double *__restrict__ A, const double *__restrict__ Bs,
                                                     float *__restrict__ gamma, float *__restrict__ beta,
                                                     float *__restrict__ acc_gamma, float *__restrict__ acc_beta,
                                                     float *__restrict__ rmean, float *__restrict__ rvar, float lr, float eps,
                                                     float momentum, const float *__restrict__ lossp, double *loss_accum) {
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        const float dg = (float)(Bs[f] + Bs[F + f]), db = (float)(A[f] + A[F + f]);
        float a = acc_gamma[f] + dg * dg;
        acc_gamma[f] = a;
        gamma[f] -= lr * dg / (sqrtf(a) + eps);
        a = acc_beta[f] + db * db;
        acc_beta[f] = a;
        beta[f] -= lr * db / (sqrtf(a) + eps);
        const float unbias = (float)B / (float)(B - 1);
        float rm = rmean[f], rv = rvar[f];
        for (int c = 0; c < 2; ++c) {
            rm += momentum * (mu[c * F + f] - rm);
            rv += momentum * (var[c * F + f] * unbias - rv);
        }
        rmean[f] = rm;
        rvar[f] = rv;
    }
    if (!loss_accum) return;
    __shared__ double sh[8];
    double t = 0.0;
    for (int b = threadIdx.x; b < B; b += 256) t += (double)lossp[b];
    t = warp_sum_d(t);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int k = 0; k < 8; ++k) tot += sh[k];
        *loss_accum += tot;
    }
}

// evaluation mode: running statistics, no dropout; pred = sum_f BN(e_u (.) e_item) + b_item  (the caller adds the user
// bias and bias_, which are the same for every item of a user)
__global__ void __launch_bounds__(256) k_fm_forward(const float *__restrict__ E, const float *__restrict__ bias,
                                                     const int32_t *__restrict__ tri, int B, int F, uint32_t U, uint32_t I,
                                                     const float *__restrict__ gamma, const float *__restrict__ beta,
                                                     const float *__restrict__ rmean, const float *__restrict__ rvar,
                                                     float bn_eps, float *__restrict__ pred_i, float *__restrict__ pred_j,
                                                     int *err) {
    const int lane = threadIdx.x & 31;
    const int b = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (b >= B) return;
    uint32_t u, i, j;
    bool bad;
    fm_ids(tri, b, U, I, u, i, j, bad);
    if (bad && lane == 0) {
        atomicOr(&err[0], 1);
        atomicMin(&err[1], b);
    }
    const float *eu = E + (size_t)u * F, *ei = E + (size_t)(U + i) * F, *ej = E + (size_t)(U + j) * F;
    float di = 0.f, dj = 0.f;
    for (int f = lane; f < F; f += 32) {
        const float iv = 1.f / sqrtf(rvar[f] + bn_eps), a = eu[f];
        di += gamma[f] * ((a * ei[f] - rmean[f]) * iv) + beta[f];
        dj += gamma[f] * ((a * ej[f] - rmean[f]) * iv) + beta[f];
    }
    di = warp_sum(di);
    dj = warp_sum(dj);
    if (lane == 0) {
        pred_i[b] = di + bias[U + i];
        pred_j[b] = dj + bias[U + j];
    }
}

// Ranking tables of the evaluation-mode model, one warp per row.  With a_f = gamma_f / sqrt(rvar_f + bn_eps) the score
// of k_fm_forward is sum_f a_f e_u,f e_i,f + b_i + (b_u + bias_ + C0), C0 = sum_f (beta_f - a_f mu_f); the rows
// P[u] = [a (.) e_u, 1, 0...] and Q[i] = [e_i, b_i, 0...] make the first two terms a dot product, so the ranking kernels
// of bpr_eval.cu / topk_full.cu rank them unchanged.  a_f is formed as k_fm_forward forms its factors.  C0 is summed by
// one thread in ascending f: the same bits on every call.
__global__ void __launch_bounds__(256) k_fm_rank_rows(const float *__restrict__ E, const float *__restrict__ bias,
                                                       int64_t rows, int64_t U, int F, int W,
                                                       const float *__restrict__ gamma, const float *__restrict__ beta,
                                                       const float *__restrict__ rmean, const float *__restrict__ rvar,
                                                       float bn_eps, float *__restrict__ P, float *__restrict__ Q,
                                                       float *__restrict__ c0) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (r == 0 && lane == 0) {
        double c = 0.0;
        for (int f = 0; f < F; ++f) {
            const float a = gamma[f] * (1.f / sqrtf(rvar[f] + bn_eps));
            c += (double)beta[f] - (double)a * (double)rmean[f];
        }
        *c0 = (float)c;
    }
    if (r >= rows) return;
    const float *e = E + (size_t)r * F;
    if (r < U) {
        float *p = P + (size_t)r * W;
        for (int f = lane; f < W; f += 32)
            p[f] = f < F ? gamma[f] * (1.f / sqrtf(rvar[f] + bn_eps)) * e[f] : (f == F ? 1.f : 0.f);
    } else {
        float *q = Q + (size_t)(r - U) * W;
        for (int f = lane; f < W; f += 32) q[f] = f < F ? e[f] : (f == F ? bias[r] : 0.f);
    }
}

static int fm_check(daisy_ctx *h, const daisy_fmbn_params *p, const void *triples, int64_t B) {
    DAISY_REQUIRE(h != nullptr && p != nullptr, DAISY_EINVAL, "null handle or parameter block");
    DAISY_REQUIRE(p->E && p->bias && p->gamma && p->beta && p->running_mean && p->running_var, DAISY_EINVAL,
                  "null table / batch-norm pointer");
    DAISY_REQUIRE(p->F >= 1 && p->F <= FM_MAX_F, DAISY_EUNSUPPORTED, "num_factors %d out of range (1..%d)", p->F, FM_MAX_F);
    DAISY_REQUIRE(p->user_num > 0 && p->num_features > p->user_num && p->num_features < 0x7fffffffLL, DAISY_EINVAL,
                  "bad feature counts (user_num %lld, num_features %lld)", (long long)p->user_num, (long long)p->num_features);
    DAISY_REQUIRE(B >= 0 && B <= 0x7fffffffLL / 3 / (p->F + 1), DAISY_EINVAL, "batch %lld out of range", (long long)B);
    DAISY_REQUIRE(B == 0 || triples != nullptr, DAISY_EINVAL, "null triples");
    return DAISY_OK;
}

}  // namespace

extern "C" int daisy_fmbn_scratch_bytes(int64_t B, int F, int64_t *bytes) {
    DAISY_REQUIRE(bytes != nullptr && B >= 0 && F >= 1 && F <= FM_MAX_F, DAISY_EINVAL, "bad scratch query");
    FmScratch w;
    fm_carve(nullptr, B > 0 ? B : 1, F, w);
    *bytes = (int64_t)w.total;
    return DAISY_OK;
}

extern "C" int daisy_fmbn_step(daisy_handle_t h, const daisy_fmbn_params *p, const int32_t *triples, int64_t B,
                               const float *mask_i, const float *mask_j, void *scratch, int64_t scratch_bytes,
                               double *loss_accum, daisy_stream_t stream) {
    int rc = fm_check(h, p, triples, B);
    if (rc) return rc;
    DAISY_REQUIRE(p->accE && p->accb && p->acc_gamma && p->acc_beta, DAISY_EINVAL, "null Adagrad accumulator");
    if (B == 0) return DAISY_OK;
    DAISY_REQUIRE(B >= 2, DAISY_EINVAL, "batch norm in training mode needs at least 2 samples per batch (got %lld)", (long long)B);
    DAISY_REQUIRE((uintptr_t)scratch % 256 == 0 && scratch != nullptr, DAISY_EINVAL, "scratch must be 256-byte aligned");
    FmScratch w;
    fm_carve((char *)scratch, B, p->F, w);
    DAISY_REQUIRE((int64_t)w.total <= scratch_bytes, DAISY_EINVAL, "scratch of %lld bytes, %zu needed (daisy_fmbn_scratch_bytes)",
                  (long long)scratch_bytes, w.total);
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int Bi = (int)B, F = p->F, n = 3 * Bi;
    const uint32_t U = (uint32_t)p->user_num, I = (uint32_t)(p->num_features - p->user_num);
    const int wblocks = daisy_ceil_div(B, 8);
    const dim3 cgrid(daisy_ceil_div(F, 32), 2, FM_Z), cblock(32, 8);
    const int fgrid = daisy_ceil_div(2 * F, 256);
    k_fm_x<<<wblocks, 256, 0, s>>>(p->E, triples, Bi, F, U, I, w.X, h->err);
    DAISY_LAUNCH_CHECK(h);
    k_fm_stats_sum<<<cgrid, cblock, 0, s>>>(w.X, Bi, F, w.part);
    DAISY_LAUNCH_CHECK(h);
    k_fm_stats_var<<<cgrid, cblock, 0, s>>>(w.X, Bi, F, w.part);
    DAISY_LAUNCH_CHECK(h);
    k_fm_stats_finish<<<fgrid, 256, 0, s>>>(w.part, Bi, F, p->bn_eps, w.mu, w.var, w.inv);
    DAISY_LAUNCH_CHECK(h);
    h->launches += 2;
    k_fm_score<<<wblocks, 256, 0, s>>>(w.X, p->bias, triples, Bi, F, U, I, w.mu, w.inv, p->gamma, p->beta, mask_i, mask_j, w.s,
                                       w.lossp);
    DAISY_LAUNCH_CHECK(h);
    k_fm_colsums_part<<<cgrid, cblock, 0, s>>>(w.X, w.s, Bi, F, w.mu, w.inv, mask_i, mask_j, w.part);
    DAISY_LAUNCH_CHECK(h);
    k_fm_colsums_finish<<<fgrid, 256, 0, s>>>(w.part, Bi, F, p->gamma, w.A, w.Bs, w.c1, w.c2);
    DAISY_LAUNCH_CHECK(h);
    h->launches += 1;
    k_fm_grad<<<wblocks, 256, 0, s>>>(p->E, w.X, w.s, triples, Bi, F, U, I, w.mu, w.inv, p->gamma, w.c1, w.c2, mask_i, mask_j,
                                      w.contrib, w.kin, w.vin);
    DAISY_LAUNCH_CHECK(h);
    int bits = 1;
    while (bits < 32 && (1ll << bits) < p->num_features) ++bits;
    size_t cub_bytes = w.cub_bytes;
    DAISY_CUDA(cub::DeviceRadixSort::SortPairs(w.cub, cub_bytes, w.kin, w.kout, w.vin, w.vout, n, 0, bits, s));
    h->launches += 3;
    k_fm_apply_slices<<<daisy_ceil_div(n, 8), 256, 0, s>>>(w.kout, w.vout, n, w.contrib, F, w.spart);
    DAISY_LAUNCH_CHECK(h);
    k_fm_apply<<<daisy_ceil_div(n, 8), 256, 0, s>>>(w.kout, n, w.spart, F, p->E, p->bias, p->accE, p->accb, p->lr, p->eps);
    DAISY_LAUNCH_CHECK(h);
    h->launches += 1;
    k_fm_bn_step<<<1, 256, 0, s>>>(Bi, F, w.mu, w.var, w.A, w.Bs, p->gamma, p->beta, p->acc_gamma, p->acc_beta, p->running_mean,
                                   p->running_var, p->lr, p->eps, p->momentum, w.lossp, loss_accum);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

extern "C" int daisy_fmbn_forward(daisy_handle_t h, const daisy_fmbn_params *p, const int32_t *triples, int64_t B,
                                  float *pred_i, float *pred_j, daisy_stream_t stream) {
    int rc = fm_check(h, p, triples, B);
    if (rc) return rc;
    if (B == 0) return DAISY_OK;
    DAISY_REQUIRE(pred_i && pred_j, DAISY_EINVAL, "null output");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    cudaStream_t s = (cudaStream_t)stream;
    k_fm_forward<<<daisy_ceil_div(B, 8), 256, 0, s>>>(p->E, p->bias, triples, (int)B, p->F, (uint32_t)p->user_num,
                                                      (uint32_t)(p->num_features - p->user_num), p->gamma, p->beta,
                                                      p->running_mean, p->running_var, p->bn_eps, pred_i, pred_j, h->err);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}

extern "C" int daisy_fmbn_rank_tables(daisy_handle_t h, const daisy_fmbn_params *p, int W, float *P_out, float *Q_out,
                                      float *c0_out, daisy_stream_t stream) {
    int rc = fm_check(h, p, nullptr, 0);
    if (rc) return rc;
    DAISY_REQUIRE(W >= p->F + 1 && W % 4 == 0, DAISY_EINVAL, "row width %d: need W >= F + 1 = %d and W %% 4 == 0", W, p->F + 1);
    DAISY_REQUIRE(P_out && Q_out && c0_out, DAISY_EINVAL, "null output");
    DeviceGuard g(h->device);
    DAISY_REQUIRE(g.ok, DAISY_ECUDA, "cannot select device %d", h->device);
    const int64_t rows = p->num_features;
    k_fm_rank_rows<<<daisy_ceil_div(rows, 8), 256, 0, (cudaStream_t)stream>>>(
        p->E, p->bias, rows, p->user_num, p->F, W, p->gamma, p->beta, p->running_mean, p->running_var, p->bn_eps, P_out,
        Q_out, c0_out);
    DAISY_LAUNCH_CHECK(h);
    return DAISY_OK;
}
