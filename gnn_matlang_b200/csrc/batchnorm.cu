// Training-mode BatchNorm over the first `cnt` rows of a node matrix (mutag.py:283-285: a BatchNorm1d after every layer), with
// `cnt` read on the device: the real node count graph_ptr[real_graphs] of a padded batch.  The rows beyond it (the dummy graph
// of a captured step) get the same affine map but never reach a statistic, a real row's output or a parameter gradient.
//
// Two launches per direction.  Pass 1: every (row chunk, 32-column tile) block sums its real rows in FP64 (lane = column,
// eight warps striding over the chunk's rows, combined in warp order) into a partial [chunk][F].  Pass 2: every block of the
// same tile reduces the partials of its 32 columns in chunk order -- all blocks get bit-identical statistics -- and maps its
// chunk's rows; the blocks of chunk 0 also write the per-column outputs (statistics, running buffers, parameter gradients).
// The chunking depends on N only, so a replay with another `cnt` keeps the summation order of an eager call.  No atomics.
//
// The forward sums x - x[0] (row 0 is real whenever cnt > 0): the shifted sums keep the biased variance Σd²/n - (Σd/n)² free of
// cancellation when the column mean dwarfs its spread.
#include "common.cuh"

namespace gnnml3 {
namespace {

constexpr int kBnWarps = 8;
constexpr int kBnThreads = kBnWarps * 32;
constexpr int kBnChunkRows = 256;    // rows per chunk at least ...
constexpr int kBnMaxChunks = 128;    // ... and at most this many chunks (the partials every pass-2 block reduces)

struct BnPlan {
    int chunks, tiles;
    int64_t rows;                    // rows per chunk
};

BnPlan bn_plan(int64_t N, int F) {
    BnPlan p;
    p.chunks = (int)(N < (int64_t)kBnChunkRows * kBnMaxChunks ? cdiv(N, kBnChunkRows) : kBnMaxChunks);
    p.rows = (N + p.chunks - 1) / p.chunks;
    p.tiles = cdiv(F, 32);
    return p;
}

__device__ __forceinline__ int64_t bn_count(const int32_t* cnt, int64_t N) {
    const int64_t c = __ldg(cnt);
    return c < 0 ? 0 : (c > N ? N : c);
}

// Sums of the block's eight warps (sh[warp][lane]) in warp order, into warp 0.
__device__ __forceinline__ double2 bn_block_sum(double2 (&sh)[kBnWarps][32], double2 v, int warp, int lane) {
    sh[warp][lane] = v;
    __syncthreads();
    double2 t = sh[0][lane];
    for (int w = 1; w < kBnWarps; ++w) {
        t.x += sh[w][lane].x;
        t.y += sh[w][lane].y;
    }
    return t;
}

// partials of the forward: part[c * F + f] = (Σ d, Σ d²), d = x[r, f] - x[0, f], over the real rows r of chunk c;
// part[chunks * F + f].x = x[0, f] (the shift)
__global__ void __launch_bounds__(kBnThreads) k_bn_fwd_stats(const float* __restrict__ x, int64_t ldx, int64_t N, int F,
                                                             const int32_t* __restrict__ cnt, int64_t rows, double2* __restrict__ part) {
    __shared__ double2 sh[kBnWarps][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y * 32 + lane;
    const int64_t n = bn_count(cnt, N);
    const int64_t r0 = blockIdx.x * rows, r1 = min(r0 + rows, n);
    double s = 0.0, q = 0.0, pivot = 0.0;
    if (f < F && n > 0) {
        pivot = (double)__ldg(x + f);
        int64_t r = r0 + warp;
        for (; r + 3 * kBnWarps < r1; r += 4 * kBnWarps) {
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = __ldg(x + (r + u * kBnWarps) * ldx + f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double d = (double)v[u] - pivot;
                s += d;
                q = fma(d, d, q);
            }
        }
        for (; r < r1; r += kBnWarps) {
            const double d = (double)__ldg(x + r * ldx + f) - pivot;
            s += d;
            q = fma(d, d, q);
        }
    }
    const double2 t = bn_block_sum(sh, make_double2(s, q), warp, lane);
    if (warp == 0 && f < F) {
        part[(int64_t)blockIdx.x * F + f] = t;
        if (blockIdx.x == 0) part[(int64_t)gridDim.x * F + f] = make_double2(pivot, 0.0);
    }
}

// Σ over the chunks' partials of column f, in chunk order, into warp 0 (every block of a tile gets the same bits)
__device__ __forceinline__ double2 bn_reduce_partials(double2 (&sh)[kBnWarps][32], const double2* __restrict__ part, int chunks,
                                                      int F, int f, int warp, int lane) {
    double2 v = make_double2(0.0, 0.0);
    if (f < F)
        for (int c = warp; c < chunks; c += kBnWarps) {
            const double2 p = part[(int64_t)c * F + f];
            v.x += p.x;
            v.y += p.y;
        }
    return bn_block_sum(sh, v, warp, lane);
}

__global__ void __launch_bounds__(kBnThreads) k_bn_fwd_apply(const float* __restrict__ x, int64_t ldx, int64_t N, int F,
                                                             const int32_t* __restrict__ cnt, int64_t rows,
                                                             const double2* __restrict__ part, const float* __restrict__ weight,
                                                             const float* __restrict__ bias, double eps, double momentum,
                                                             float* __restrict__ running_mean, float* __restrict__ running_var,
                                                             int64_t* __restrict__ nbt, float* __restrict__ y, int64_t ldy,
                                                             float* __restrict__ save_mean, float* __restrict__ save_invstd) {
    __shared__ double2 sh[kBnWarps][32];
    __shared__ float s_mean[32], s_scale[32], s_bias[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y * 32 + lane;
    const int64_t n = bn_count(cnt, N);
    const double2 t = bn_reduce_partials(sh, part, gridDim.x, F, f, warp, lane);
    if (warp == 0 && f < F) {
        const double m = n > 0 ? t.x / (double)n : 0.0;
        const double var = n > 0 ? fmax(t.y / (double)n - m * m, 0.0) : 0.0;        // biased: what normalises
        const double mean = n > 0 ? part[(int64_t)gridDim.x * F + f].x + m : 0.0;
        const float invstd = (float)(1.0 / sqrt(var + eps));
        s_mean[lane] = (float)mean;
        s_scale[lane] = invstd * __ldg(weight + f);
        s_bias[lane] = __ldg(bias + f);
        if (blockIdx.x == 0) {
            save_mean[f] = (float)mean;
            save_invstd[f] = invstd;
            if (n > 0) running_mean[f] = (float)((1.0 - momentum) * (double)running_mean[f] + momentum * mean);
            if (n > 1)                                                              // unbiased; one row has no variance
                running_var[f] = (float)((1.0 - momentum) * (double)running_var[f] + momentum * var * (double)n / (double)(n - 1));
        }
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *nbt += 1;
    __syncthreads();
    if (f >= F) return;
    const float mu = s_mean[lane], sc = s_scale[lane], b = s_bias[lane];
    const int64_t r0 = blockIdx.x * rows, r1 = min(r0 + rows, N);
    for (int64_t r = r0 + warp; r < r1; r += kBnWarps) y[r * ldy + f] = (__ldg(x + r * ldx + f) - mu) * sc + b;
}

// partials of the backward: (Σ gy, Σ gy (x - mean)) over the real rows of chunk c
__global__ void __launch_bounds__(kBnThreads) k_bn_bwd_stats(const float* __restrict__ x, int64_t ldx, const float* __restrict__ gy,
                                                             int64_t ldg, int64_t N, int F, const int32_t* __restrict__ cnt,
                                                             int64_t rows, const float* __restrict__ save_mean,
                                                             double2* __restrict__ part) {
    __shared__ double2 sh[kBnWarps][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y * 32 + lane;
    const int64_t n = bn_count(cnt, N);
    const int64_t r0 = blockIdx.x * rows, r1 = min(r0 + rows, n);
    double s = 0.0, q = 0.0;
    if (f < F) {
        const float mu = __ldg(save_mean + f);
        int64_t r = r0 + warp;
        for (; r + 3 * kBnWarps < r1; r += 4 * kBnWarps) {
            float v[4], g[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                v[u] = __ldg(x + (r + u * kBnWarps) * ldx + f);
                g[u] = __ldg(gy + (r + u * kBnWarps) * ldg + f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                s += (double)g[u];
                q = fma((double)g[u], (double)(v[u] - mu), q);
            }
        }
        for (; r < r1; r += kBnWarps) {
            const float g = __ldg(gy + r * ldg + f);
            s += (double)g;
            q = fma((double)g, (double)(__ldg(x + r * ldx + f) - mu), q);
        }
    }
    const double2 t = bn_block_sum(sh, make_double2(s, q), warp, lane);
    if (warp == 0 && f < F) part[(int64_t)blockIdx.x * F + f] = t;
}

// dx = w invstd (gy - Σgy / n - (x - mean) invstd² Σgy(x - mean) / n) on real rows, 0 on the others;
// dbias = Σ gy, dweight = invstd Σ gy (x - mean)
__global__ void __launch_bounds__(kBnThreads) k_bn_bwd_apply(const float* __restrict__ x, int64_t ldx, const float* __restrict__ gy,
                                                             int64_t ldg, int64_t N, int F, const int32_t* __restrict__ cnt,
                                                             int64_t rows, const double2* __restrict__ part,
                                                             const float* __restrict__ weight, const float* __restrict__ save_mean,
                                                             const float* __restrict__ save_invstd, float* __restrict__ dx,
                                                             int64_t lddx, float* __restrict__ dweight, float* __restrict__ dbias) {
    __shared__ double2 sh[kBnWarps][32];
    __shared__ float s_c0[32], s_c1[32], s_c2[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.y * 32 + lane;
    const int64_t n = bn_count(cnt, N);
    const double2 t = bn_reduce_partials(sh, part, gridDim.x, F, f, warp, lane);
    if (warp == 0 && f < F) {
        const double is = (double)__ldg(save_invstd + f);
        s_c0[lane] = (float)(is * (double)__ldg(weight + f));
        s_c1[lane] = n > 0 ? (float)(t.x / (double)n) : 0.f;
        s_c2[lane] = n > 0 ? (float)(is * is * t.y / (double)n) : 0.f;
        if (blockIdx.x == 0) {
            dbias[f] = (float)t.x;
            dweight[f] = (float)(t.y * is);
        }
    }
    __syncthreads();
    if (f >= F) return;
    const float mu = __ldg(save_mean + f), c0 = s_c0[lane], c1 = s_c1[lane], c2 = s_c2[lane];
    const int64_t r0 = blockIdx.x * rows, r1 = min(r0 + rows, N);
    for (int64_t r = r0 + warp; r < r1; r += kBnWarps)
        dx[r * lddx + f] = r < n ? c0 * (__ldg(gy + r * ldg + f) - c1 - (__ldg(x + r * ldx + f) - mu) * c2) : 0.f;
}

}  // namespace
}  // namespace gnnml3

using namespace gnnml3;

extern "C" size_t gnnml3_bn_rows_workspace_bytes(int64_t N, int F) {
    if (N < 1 || F < 1) return 0;
    const BnPlan p = bn_plan(N, F);
    return (size_t)(p.chunks + 1) * (size_t)F * sizeof(double2);
}

extern "C" int gnnml3_bn_rows_fwd(const float* x, int64_t ldx, int64_t N, int F, const int32_t* cnt, const float* weight,
                                  const float* bias, double eps, double momentum, float* running_mean, float* running_var,
                                  int64_t* num_batches_tracked, float* y, int64_t ldy, float* save_mean, float* save_invstd,
                                  void* workspace, size_t workspace_bytes, void* stream_) {
    GNNML3_REQUIRE(N >= 1 && F >= 1, "bn_rows_fwd: need N >= 1 and F >= 1 (got %lld, %d)", (long long)N, F);
    GNNML3_REQUIRE(x && cnt && weight && bias && running_mean && running_var && num_batches_tracked && y && save_mean && save_invstd,
                   "bn_rows_fwd: NULL argument");
    GNNML3_REQUIRE(ldx >= F && ldy >= F, "bn_rows_fwd: row strides below F");
    GNNML3_REQUIRE(eps > 0.0 && momentum >= 0.0 && momentum <= 1.0, "bn_rows_fwd: need eps > 0 and momentum in [0, 1]");
    GNNML3_REQUIRE(workspace, "bn_rows_fwd: workspace required");
    if (workspace_bytes < gnnml3_bn_rows_workspace_bytes(N, F)) return set_err(GNNML3_ERR_WORKSPACE, "bn_rows_fwd: workspace too small");
    const BnPlan p = bn_plan(N, F);
    cudaStream_t st = (cudaStream_t)stream_;
    double2* part = (double2*)workspace;
    const dim3 grid(p.chunks, p.tiles);
    k_bn_fwd_stats<<<grid, kBnThreads, 0, st>>>(x, ldx, N, F, cnt, p.rows, part);
    GNNML3_LAUNCH_CHECK();
    k_bn_fwd_apply<<<grid, kBnThreads, 0, st>>>(x, ldx, N, F, cnt, p.rows, part, weight, bias, eps, momentum, running_mean,
                                                running_var, num_batches_tracked, y, ldy, save_mean, save_invstd);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

extern "C" int gnnml3_bn_rows_bwd(const float* x, int64_t ldx, const float* gy, int64_t ldgy, int64_t N, int F, const int32_t* cnt,
                                  const float* weight, const float* save_mean, const float* save_invstd, float* dx, int64_t lddx,
                                  float* dweight, float* dbias, void* workspace, size_t workspace_bytes, void* stream_) {
    GNNML3_REQUIRE(N >= 1 && F >= 1, "bn_rows_bwd: need N >= 1 and F >= 1 (got %lld, %d)", (long long)N, F);
    GNNML3_REQUIRE(x && gy && cnt && weight && save_mean && save_invstd && dx && dweight && dbias, "bn_rows_bwd: NULL argument");
    GNNML3_REQUIRE(ldx >= F && ldgy >= F && lddx >= F, "bn_rows_bwd: row strides below F");
    GNNML3_REQUIRE(workspace, "bn_rows_bwd: workspace required");
    if (workspace_bytes < gnnml3_bn_rows_workspace_bytes(N, F)) return set_err(GNNML3_ERR_WORKSPACE, "bn_rows_bwd: workspace too small");
    const BnPlan p = bn_plan(N, F);
    cudaStream_t st = (cudaStream_t)stream_;
    double2* part = (double2*)workspace;
    const dim3 grid(p.chunks, p.tiles);
    k_bn_bwd_stats<<<grid, kBnThreads, 0, st>>>(x, ldx, gy, ldgy, N, F, cnt, p.rows, save_mean, part);
    GNNML3_LAUNCH_CHECK();
    k_bn_bwd_apply<<<grid, kBnThreads, 0, st>>>(x, ldx, gy, ldgy, N, F, cnt, p.rows, part, weight, save_mean, save_invstd, dx, lddx,
                                                dweight, dbias);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}
