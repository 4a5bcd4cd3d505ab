// Pair-distinguishing kernels of the isomorphism test (graph8c.py:281-302, sr25.py, exp_iso.py): a pair of graphs counts as
// distinguished once the L1 distance of its embeddings exceeds the threshold under any seed.  The cross-seed state is a bitmap
// (one bit per pair) that each seed's embeddings are OR-ed into; nothing materialises the [n, n] distance matrix.
//
//   k_pairs_mark_all : upper triangle (i < j < n) in 128 x 128 pair tiles, row blocks staged in shared memory in chunks of
//                      the embedding dimension, an 8 x 8 register micro-tile per thread.  A tile whose pairs are all marked
//                      already does no arithmetic (after the first seed of a model that separates almost everything, a later
//                      seed reads the bitmap once).
//   k_pairs_mark_list: listed pairs [P, 2] (exp_iso.py's E[0::2] against E[1::2]), one thread per pair, one warp per word.
//   k_pairs_count    : pairs whose bit is still 0, reduced in a fixed order inside one thread-block cluster.
//
// dist = sum_{k = 0..d-1} |a_k - b_k| in FP32, in dimension order, in both marking kernels: the same pair gets the same bits
// in either mode and in every run.  The test is dist > threshold; NaN compares false (not distinguished), as cdist > thr.
#include <cooperative_groups.h>
#include <math.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace gnnml3 {
namespace {

constexpr int kTile = 128;            // pair tile: 128 rows x 128 columns = 4 bitmap words per row
constexpr int kMarkThreads = 256;     // 16 x 16 threads, 8 x 8 pairs each
constexpr int kChunk = 32;            // embedding dimensions staged per pass
constexpr int kCountThreads = 1024;
constexpr int kCountCluster = 16;     // non-portable cluster size (sm_100 allows 16)

// bits j of word w of row i that are valid pairs: i < j < limit (row i = -1 for the listed-pairs bitmap)
__device__ __forceinline__ uint32_t valid_mask(int64_t i, int64_t w, int64_t limit) {
    const int64_t lo = max(i + 1, w * 32), hi = min(limit, w * 32 + 32);
    if (lo >= hi) return 0u;
    const int a = (int)(lo - w * 32), b = (int)(hi - w * 32);            // bits [a, b)
    const uint32_t upto_b = b == 32 ? 0xffffffffu : ((1u << b) - 1u);
    return upto_b & ~((1u << a) - 1u);
}

// upper-triangle tile t -> (bi, bj), bi <= bj < T, row-major over the triangle
__device__ __forceinline__ void tri_tile(int64_t t, int64_t T, int64_t& bi, int64_t& bj) {
    // start(b) = b T - b (b - 1) / 2 is the first tile of tile-row b
    const double tt = (double)T + 0.5;
    int64_t b = (int64_t)floor(tt - sqrt(tt * tt - 2.0 * (double)t));
    b = max((int64_t)0, min(b, T - 1));
    while (b > 0 && b * T - b * (b - 1) / 2 > t) --b;
    while (b + 1 < T && (b + 1) * T - (b + 1) * b / 2 <= t) ++b;
    bi = b;
    bj = b + (t - (b * T - b * (b - 1) / 2));
}

__global__ void __launch_bounds__(kMarkThreads, 2)
k_pairs_mark_all(const float* __restrict__ emb, int64_t ld, int64_t n, int d, float threshold, uint32_t* __restrict__ bits,
                 int64_t wpr, int64_t T) {
    __shared__ float As[kChunk][kTile + 1];                              // +1: the transposing stores do not collide on banks
    __shared__ float Bs[kChunk][kTile + 1];
    __shared__ uint32_t old[kTile][4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31;
    int64_t bi, bj;
    tri_tile(blockIdx.x, T, bi, bj);
    const int64_t row0 = bi * kTile, col0 = bj * kTile, words = (n + 31) / 32;

    // skip rule: read the tile's words; a tile whose valid pairs are all marked is done
    bool full = true;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int q = tid + s * kMarkThreads, r = q >> 2, w = q & 3;
        const int64_t i = row0 + r, gw = bj * 4 + w;
        uint32_t o = 0, vm = 0;
        if (i < n && gw < words) {
            o = bits[i * wpr + gw];
            vm = valid_mask(i, gw, n);
        }
        old[r][w] = o;
        full &= (o & vm) == vm;
    }
    if (__syncthreads_and(full)) return;

    float acc[8][8];
#pragma unroll
    for (int m = 0; m < 8; ++m)
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[m][k] = 0.f;

    for (int d0 = 0; d0 < d; d0 += kChunk) {
        const int dk = min(kChunk, d - d0);
        for (int q = tid; q < kTile * dk; q += kMarkThreads) {
            const int r = q / dk, kk = q - r * dk;
            const int64_t i = row0 + r, j = col0 + r;
            As[kk][r] = i < n ? emb[i * ld + d0 + kk] : 0.f;
            Bs[kk][r] = j < n ? emb[j * ld + d0 + kk] : 0.f;
        }
        __syncthreads();
        for (int kk = 0; kk < dk; ++kk) {
            float a[8], b[8];
#pragma unroll
            for (int m = 0; m < 8; ++m) a[m] = As[kk][ty + 16 * m];
#pragma unroll
            for (int k = 0; k < 8; ++k) b[k] = Bs[kk][tx + 16 * k];
#pragma unroll
            for (int m = 0; m < 8; ++m)
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[m][k] += fabsf(a[m] - b[k]);
        }
        __syncthreads();
    }

    // Thread (ty, tx) holds rows ty + 16 m and columns tx + 16 k; a warp is two rows (ty even / odd) by 16 columns, so the
    // ballots of k = 2w and 2w + 1 give word w of each of its two rows.  Lanes tx = w of each half keep that word.
    const int half = lane >> 4;
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int r = ty + 16 * m;
        const int64_t i = row0 + r;
        uint32_t mine = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const int64_t j0 = col0 + 32 * w + tx, j1 = j0 + 16;
            const bool p0 = i < n && j0 < n && j0 > i && acc[m][2 * w] > threshold;
            const bool p1 = i < n && j1 < n && j1 > i && acc[m][2 * w + 1] > threshold;
            const uint32_t b0 = __ballot_sync(0xffffffffu, p0), b1 = __ballot_sync(0xffffffffu, p1);
            const uint32_t word = ((b0 >> (16 * half)) & 0xffffu) | (((b1 >> (16 * half)) & 0xffffu) << 16);
            if (tx == w) mine = word;
        }
        const int64_t gw = bj * 4 + tx;
        if (tx < 4 && i < n && gw < words) {
            const uint32_t o = old[r][tx];
            if (mine & ~o) bits[i * wpr + gw] = o | mine;
        }
    }
}

__global__ void __launch_bounds__(256)
k_pairs_mark_list(const float* __restrict__ emb, int64_t ld, int64_t n, int d, const int64_t* __restrict__ pairs, int64_t P,
                  float threshold, uint32_t* __restrict__ bits) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w * 32 >= P) return;
    const uint32_t o = bits[w], vm = valid_mask(-1, w, P);
    if ((o & vm) == vm) return;                                           // warp-uniform
    const int64_t p = w * 32 + lane;
    bool mark = false;
    if (p < P) {
        const int64_t i = pairs[2 * p], j = pairs[2 * p + 1];
        if (i >= 0 && i < n && j >= 0 && j < n) {
            const float* a = emb + i * ld;
            const float* b = emb + j * ld;
            float dist = 0.f;
            for (int k = 0; k < d; ++k) dist += fabsf(__ldg(a + k) - __ldg(b + k));
            mark = dist > threshold;
        }
    }
    const uint32_t word = __ballot_sync(0xffffffffu, mark);
    if (lane == 0 && (word & ~o)) bits[w] = o | word;
}

// Marked valid pairs of rows [0, R): row r covers words [(i + 1) / 32, ceil(limit / 32)) with i = r (all pairs) or i = -1
// (listed pairs, R = 1).  One warp per row (rows strided over the cluster's warps), per-thread integer sums, then a fixed
// order: warp butterfly, warps in index order, CTAs in cluster-rank order through distributed shared memory.
__global__ void __launch_bounds__(kCountThreads)
k_pairs_count(const uint32_t* __restrict__ bits, int64_t R, int64_t wpr, int64_t limit, int listed, int64_t total,
              int64_t* __restrict__ out) {
    __shared__ unsigned long long warp_sum[kCountThreads / 32];
    __shared__ unsigned long long cta_sum;
    cg::cluster_group cluster = cg::this_cluster();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t nwarps = (int64_t)kCountCluster * (kCountThreads / 32);
    const int64_t gwarp = (int64_t)cluster.block_rank() * (kCountThreads / 32) + warp;
    const int64_t wend = (limit + 31) / 32;
    unsigned long long s = 0;
    for (int64_t r = gwarp; r < R; r += nwarps) {
        const int64_t i = listed ? -1 : r;
        const uint32_t* row = bits + r * wpr;
        const int64_t w0 = (i + 1) / 32;
        // head words up to a 16-byte boundary, then 128-bit loads, then the tail
        int64_t wa = w0;
        while (wa < wend && (reinterpret_cast<uintptr_t>(row + wa) & 15)) ++wa;
        wa = min(wa, wend);
        const int64_t nv = (wend - wa) / 4, wb = wa + nv * 4;
        for (int64_t w = w0 + lane; w < wa; w += 32) s += __popc(__ldg(row + w) & valid_mask(i, w, limit));
        const uint4* v = reinterpret_cast<const uint4*>(row + wa);
#pragma unroll 4
        for (int64_t q = lane; q < nv; q += 32) {
            const uint4 x = __ldg(v + q);
            const int64_t w = wa + 4 * q;
            s += __popc(x.x & valid_mask(i, w, limit)) + __popc(x.y & valid_mask(i, w + 1, limit)) +
                 __popc(x.z & valid_mask(i, w + 2, limit)) + __popc(x.w & valid_mask(i, w + 3, limit));
        }
        for (int64_t w = wb + lane; w < wend; w += 32) s += __popc(__ldg(row + w) & valid_mask(i, w, limit));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) warp_sum[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long c = 0;
        for (int k = 0; k < kCountThreads / 32; ++k) c += warp_sum[k];
        cta_sum = c;
    }
    cluster.sync();
    if (cluster.block_rank() == 0 && threadIdx.x == 0) {
        unsigned long long marked = 0;
        for (unsigned k = 0; k < (unsigned)kCountCluster; ++k) marked += *cluster.map_shared_rank(&cta_sum, k);
        *out = total - (int64_t)marked;
    }
    cluster.sync();                                                       // keep every CTA's shared memory alive until read
}

}  // namespace
}  // namespace gnnml3

using namespace gnnml3;

extern "C" int gnnml3_pairs_mark(const float* emb, int64_t ld, int64_t n, int d, const int64_t* pairs, int64_t P,
                                 float threshold, uint32_t* bits, int64_t wpr, void* stream_) {
    GNNML3_REQUIRE(d >= 1 && ld >= d, "pairs_mark: need d >= 1 and ld >= d (d = %d, ld = %lld)", d, (long long)ld);
    GNNML3_REQUIRE(n >= 0 && P >= 0, "pairs_mark: negative n or P");
    GNNML3_REQUIRE(isfinite(threshold) && threshold >= 0.f, "pairs_mark: the threshold must be finite and >= 0");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (pairs == nullptr) {
        GNNML3_REQUIRE(P == 0, "pairs_mark: P must be 0 in all-pairs mode (pairs == NULL)");
        GNNML3_REQUIRE(wpr >= (n + 31) / 32, "pairs_mark: wpr = %lld < ceil(n / 32) = %lld", (long long)wpr, (long long)((n + 31) / 32));
        const int64_t T = (n + kTile - 1) / kTile, tiles = T * (T + 1) / 2;
        GNNML3_REQUIRE(tiles <= 0x7fffffffLL, "pairs_mark: n = %lld is too large for one launch", (long long)n);
        if (n < 2) return GNNML3_OK;
        GNNML3_REQUIRE(emb && bits, "pairs_mark: NULL emb or bits");
        k_pairs_mark_all<<<(unsigned)tiles, kMarkThreads, 0, stream>>>(emb, ld, n, d, threshold, bits, wpr, T);
        GNNML3_LAUNCH_CHECK();
        return GNNML3_OK;
    }
    if (P == 0) return GNNML3_OK;
    GNNML3_REQUIRE(bits && (n == 0 || emb), "pairs_mark: NULL emb or bits");
    const int64_t threads = (P + 31) / 32 * 32;
    k_pairs_mark_list<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(emb, ld, n, d, pairs, P, threshold, bits);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

extern "C" int gnnml3_pairs_count(const uint32_t* bits, int64_t n, int64_t wpr, int64_t P, int64_t* out, void* stream_) {
    GNNML3_REQUIRE(n >= 0 && P >= 0, "pairs_count: negative n or P");
    GNNML3_REQUIRE(out, "pairs_count: NULL out");
    const int listed = P > 0;
    if (!listed) GNNML3_REQUIRE(wpr >= (n + 31) / 32, "pairs_count: wpr = %lld < ceil(n / 32)", (long long)wpr);
    const int64_t limit = listed ? P : n, total = listed ? P : n * (n - 1) / 2, R = total == 0 ? 0 : listed ? 1 : n;
    GNNML3_REQUIRE(bits || R == 0, "pairs_count: NULL bits");
    static bool configured[64];
    if (auto once = first_use_on_device(configured))
        GNNML3_CUDA(cudaFuncSetAttribute(k_pairs_count, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kCountCluster);
    cfg.blockDim = dim3(kCountThreads);
    cfg.stream = (cudaStream_t)stream_;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kCountCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    GNNML3_CUDA(cudaLaunchKernelEx(&cfg, k_pairs_count, bits, R, wpr, limit, listed, total, out));
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}
