// GNNML1 layer (the paper's 1-WL model) on Blackwell tensor cores: unweighted CSR aggregate + projection.
//
// Layer (reference GNNML1 classes: relu(fc11(x) + conv11(x, edge_index, ones) + fc12(x) * fc13(x)) and its torch.cat form):
//     p0 = x fcA^T + bA + (A x) Wc + bc,   p1 = x fcB^T + bB,   p2 = x fcC^T + bC
//     sum mode   : y = relu(p0 + p1 * p2)                                                  [N, Fo]
//     concat mode: y = [relu(x fcA^T + bA) | relu((A x) Wc + bc) | relu(p1 * p2)]          [N, 3 Fo]
// with (A x)[t] = sum of x[s] over the edges s -> t (dst-sorted CSR, edge order kept), all edge weights one and never read.
//
// One kernel (k_ml1_agg_proj) serves both directions.  A persistent CTA of 512 threads owns tiles of 128 rows.  Per tile it
// walks a list of 32-wide k-blocks: first the "self" blocks (row t of a dense matrix S), then the "gathered" blocks (the sum
// of X[s] over the CSR row t).  Every k-block is written by all threads into a shared-memory A operand in the UMMA K-major
// SWIZZLE_128B layout (raw FP32 plane + residual plane lo = a - trunc(a)), and one thread issues tcgen05.mma kind::tf32
// with the tile's rows as M = 128 and the output columns as N, against weight planes (hi = RN-TF32(w), lo = w - hi) that
// stay resident in shared memory for the whole launch.  Three MMAs per 8-wide k-step (a*w_hi + a*w_lo + a_lo*w_hi) give
// FP32-grade (3xTF32) products.  Two A buffers alternate, so the gather of one k-block overlaps the MMAs of the previous.
// The accumulator D[row, column] lives in tensor memory (lane = tile row); the epilogue reads it back and applies the layer.
//
// Precision (template PREC = GNNML3_PREC_*; the aggregation, the epilogues and their FP32 outputs are the same in every mode):
//   0 3xTF32 : as above (default, FP32-grade).
//   1 TF32   : one kind::tf32 MMA per 8-wide k-step, raw A (truncated by the tensor core) x RN-TF32(w); no residual planes,
//              so each A buffer and the resident weights are half the size.
//   2 BF16   : A and w RN-converted to BF16 and stored in the first 64 bytes of each 128-byte swizzled row (32 values; the
//              16-byte chunk c >> 1 of a row holds features 8 (c >> 1) .. + 7, XOR-swizzled with row & 7 as in FP32); two
//              kind::f16 MMAs (K = 16) per k-block, FP32 accumulate.  No residual planes either.
//
//   forward : self = x, weights [fcA^T | fcB^T | fcC^T] -> columns [p0 | p1 | p2] (pitch Fop = ceil16(Fo));
//             gathered = x over the CSR, weights Wc -> columns [0, Fop) (sum: adds into p0) or [3 Fop, 4 Fop) (concat).
//   dx pass : self = [gA | gP*p2 | gP*p1] (d p0, d p1, d p2), weights [fcA ; fcB ; fcC]; gathered = gc over the transposed
//             CSR, weights Wc^T; both accumulate into columns [0, Fi).
// Deterministic: every sum has a fixed order (edges in CSR order, k-blocks in list order), no atomics.  No host sync.
#include "tc_common.cuh"

#include <cuda_bf16.h>

namespace gnnml3 {

constexpr int ML1_THREADS = 512;
constexpr int ML1_ROWS = 128;                      // tile rows = MMA M = tensor-memory lanes
constexpr int ML1_APLANE = ML1_ROWS * 128;         // bytes of one 128-row x 32-float swizzled plane
constexpr int ML1_ABUF = 2 * ML1_APLANE;           // raw plane + residual plane (3xTF32; the flagged modes use the first)

// planes per k-block of an A buffer and of the weights: raw/hi + residual/lo in 3xTF32, one plane in TF32 and BF16
__host__ __device__ constexpr int ml1_planes(int prec) { return prec == GNNML3_PREC_3XTF32 ? 2 : 1; }
__host__ __device__ constexpr int ml1_abuf(int prec) { return ml1_planes(prec) * ML1_APLANE; }    // bytes of one A buffer

struct ML1Params {
    const int* rowptr;      // [N+1] CSR of the gathered blocks (dst-sorted forward, src-sorted for dx)
    const int* col;         // [E]
    int64_t N;
    int n_tiles;
    const float* X;         // gathered matrix [*, Fg], row stride ldx
    int64_t ldx;
    int Fg, ngb;            // width, 32-wide k-blocks
    const float* S;         // self matrix [N, Fs], row stride lds
    int64_t lds;
    int Fs, nsb;
    const float* planes;    // weight planes in the shared-memory byte layout: self blocks, then gathered blocks
    int wbytes;
    int NsP, NgP, colG;     // MMA N of the self / gathered blocks, tensor-memory column of the gathered accumulator
    int tmem_cols;
    int project;            // 0: aggregate only (hout), no MMA
    int epi;                // 0: out[:, :Nout] = D | 1: GNNML1 sum mode | 2: GNNML1 concat mode
    int Fo, Fop;
    const float *bA, *bB, *bC, *bc;
    float* out;
    int64_t ldo;
    int Nout;
    float* aux;             // [N, 2 Fo] = [p1 | p2] (bias included), for the backward
    int64_t ldaux;
    float* hout;            // optional copy of the gathered aggregate [N, Fg] (row stride ldh)
    int64_t ldh;
};

// four consecutive columns f.. f+3 of a row (zero beyond F); 128-bit load when the whole chunk is inside
__device__ __forceinline__ float4 ml1_load4(const float* __restrict__ row, int f, int F) {
    if (f + 3 < F) return ldg4(row + f);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (f < F) v.x = __ldg(row + f);
    if (f + 1 < F) v.y = __ldg(row + f + 1);
    if (f + 2 < F) v.z = __ldg(row + f + 2);
    return v;
}

__device__ __forceinline__ float ml1_lo(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// AUX = false: the forward-only instantiation of the GNNML1 epilogues (aux == NULL), which stores y and not [p1 | p2].
// PREC: the arithmetic of the projection (GNNML3_PREC_*, see the top of this file).
template <bool AUX = true, int PREC = GNNML3_PREC_3XTF32>
__global__ void __launch_bounds__(ML1_THREADS, 1) k_ml1_agg_proj(const __grid_constant__ ML1Params P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* wsm = smem;                                     // resident weight planes
    uint8_t* abuf = smem + P.wbytes;                         // [2][raw plane | lo plane (3xTF32 only)]
    uint64_t* bars = reinterpret_cast<uint64_t*>(abuf + 2 * ml1_abuf(PREC));   // [2] MMAs reading A buffer b retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (P.project) {
        const uint4* src = reinterpret_cast<const uint4*>(P.planes);
        uint4* dst = reinterpret_cast<uint4*>(wsm);
        for (int i = tid; i < P.wbytes / 16; i += ML1_THREADS) dst[i] = __ldg(src + i);
        if (tid == 0) {
            mbar_init(bars, 1);
            mbar_init(bars + 1, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        if (warp == 0) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
        fence_proxy_async_smem();                            // weight planes (generic stores) -> tensor core (async proxy)
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = P.project ? *tmem_slot : 0u;

    const int c = tid & 7;                                   // 16-byte chunk of a 32-float k-block row
    const int rsub = tid >> 3;                               // rows rsub and rsub + 64 of the tile
    const int nph = P.nsb + P.ngb;
    uint32_t ph0 = 0, ph1 = 0;
    bool pend0 = false, pend1 = false;
    uint32_t it = 0;
    const uint32_t wsm0 = smem_u32(wsm), abuf0 = smem_u32(abuf);
    const uint32_t self_bytes = (uint32_t)P.nsb * (uint32_t)ml1_planes(PREC) * (uint32_t)P.NsP * 128u;

    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
        const int64_t row0 = (int64_t)tile * ML1_ROWS;
        for (int i = 0; i < nph; ++i, ++it) {
            const int b = it & 1;
            if (b == 0 && pend0) { mbar_wait(bars, ph0); ph0 ^= 1; pend0 = false; }
            if (b == 1 && pend1) { mbar_wait(bars + 1, ph1); ph1 ^= 1; pend1 = false; }
            const bool self = i < P.nsb;
            const int kb = self ? i : i - P.nsb;
            const int f = kb * 32 + 4 * c;
            uint8_t* A = abuf + b * ml1_abuf(PREC);
            float4 v[2];
            int64_t r[2];
            int rs[2] = {0, 0}, re[2] = {0, 0};
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                r[h] = row0 + rsub + 64 * h;
                v[h] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r[h] < P.N) {
                    if (self) {
                        v[h] = ml1_load4(P.S + r[h] * P.lds, f, P.Fs);
                    } else {
                        rs[h] = __ldg(P.rowptr + r[h]);
                        re[h] = __ldg(P.rowptr + r[h] + 1);
                    }
                }
            }
            if (!self) {
                // both rows' edge lists in lock-step (two independent gather chains in flight), each summed in CSR order
                const int n0 = re[0] - rs[0], n1 = re[1] - rs[1];
                const int n = n0 > n1 ? n0 : n1;
                for (int e = 0; e < n; ++e) {
                    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
                    if (e < n0) a0 = ml1_load4(P.X + (int64_t)__ldg(P.col + rs[0] + e) * P.ldx, f, P.Fg);
                    if (e < n1) a1 = ml1_load4(P.X + (int64_t)__ldg(P.col + rs[1] + e) * P.ldx, f, P.Fg);
                    if (e < n0) { v[0].x += a0.x; v[0].y += a0.y; v[0].z += a0.z; v[0].w += a0.w; }
                    if (e < n1) { v[1].x += a1.x; v[1].y += a1.y; v[1].z += a1.z; v[1].w += a1.w; }
                }
                if (P.hout) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (r[h] >= P.N || f >= P.Fg) continue;
                        float* hr = P.hout + r[h] * P.ldh + f;
                        if (f + 3 < P.Fg) {
                            *reinterpret_cast<float4*>(hr) = v[h];
                        } else {
                            hr[0] = v[h].x;
                            if (f + 1 < P.Fg) hr[1] = v[h].y;
                            if (f + 2 < P.Fg) hr[2] = v[h].z;
                        }
                    }
                }
            }
            if (!P.project) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int m = rsub + 64 * h;
                if constexpr (PREC == GNNML3_PREC_3XTF32) {
                    const uint32_t off = (uint32_t)(m >> 3) * 1024u + (uint32_t)(m & 7) * 128u + (uint32_t)((c ^ (m & 7)) << 4);
                    *reinterpret_cast<float4*>(A + off) = v[h];
                    *reinterpret_cast<float4*>(A + ML1_APLANE + off) =
                        make_float4(ml1_lo(v[h].x), ml1_lo(v[h].y), ml1_lo(v[h].z), ml1_lo(v[h].w));
                } else if constexpr (PREC == GNNML3_PREC_TF32) {     // raw plane alone
                    const uint32_t off = (uint32_t)(m >> 3) * 1024u + (uint32_t)(m & 7) * 128u + (uint32_t)((c ^ (m & 7)) << 4);
                    *reinterpret_cast<float4*>(A + off) = v[h];
                } else {                                             // 4 BF16 = half of the 16-byte chunk c >> 1
                    const uint32_t off = (uint32_t)(m >> 3) * 1024u + (uint32_t)(m & 7) * 128u +
                                         (uint32_t)(((c >> 1) ^ (m & 7)) << 4) + (uint32_t)(c & 1) * 8u;
                    const __nv_bfloat162 lo = __floats2bfloat162_rn(v[h].x, v[h].y), hi = __floats2bfloat162_rn(v[h].z, v[h].w);
                    *reinterpret_cast<uint2*>(A + off) =
                        make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
                }
            }
            fence_proxy_async_smem();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                const int N = self ? P.NsP : P.NgP;
                if constexpr (PREC == GNNML3_PREC_3XTF32) {
                    const uint32_t idesc = make_idesc_tf32_mn(ML1_ROWS, N);
                    const uint32_t d = tmem_base + (uint32_t)(self ? 0 : P.colG);
                    const bool fresh = self ? kb == 0 : (kb == 0 && P.colG >= P.NsP);   // first k-block into these columns
                    const uint32_t wb = wsm0 + (self ? (uint32_t)kb * 2u * (uint32_t)P.NsP * 128u
                                                     : self_bytes + (uint32_t)kb * 2u * (uint32_t)P.NgP * 128u);
                    const uint64_t a_hi = make_kmajor_sw128_desc(abuf0 + (uint32_t)b * ML1_ABUF);
                    const uint64_t a_lo = make_kmajor_sw128_desc(abuf0 + (uint32_t)b * ML1_ABUF + ML1_APLANE);
                    const uint64_t w_hi = make_kmajor_sw128_desc(wb);
                    const uint64_t w_lo = make_kmajor_sw128_desc(wb + (uint32_t)N * 128u);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t adv = (uint64_t)((k * 32) >> 4);     // 8 TF32 = 32 bytes along K inside the swizzled row
                        umma_tf32(d, a_hi + adv, w_hi + adv, idesc, (fresh && k == 0) ? 0u : 1u);
                        umma_tf32(d, a_hi + adv, w_lo + adv, idesc, 1u);
                        umma_tf32(d, a_lo + adv, w_hi + adv, idesc, 1u);
                    }
                } else {                                             // one plane each of A and w: a single product per k-step
                    const uint32_t d = tmem_base + (uint32_t)(self ? 0 : P.colG);
                    const bool fresh = self ? kb == 0 : (kb == 0 && P.colG >= P.NsP);
                    const uint32_t wb = wsm0 + (self ? (uint32_t)kb * (uint32_t)P.NsP * 128u : self_bytes + (uint32_t)kb * (uint32_t)P.NgP * 128u);
                    const uint64_t a = make_kmajor_sw128_desc(abuf0 + (uint32_t)b * ml1_abuf(PREC));
                    const uint64_t w = make_kmajor_sw128_desc(wb);
                    if constexpr (PREC == GNNML3_PREC_TF32) {
                        const uint32_t idesc = make_idesc_tf32_mn(ML1_ROWS, N);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint64_t adv = (uint64_t)((k * 32) >> 4);
                            umma_tf32(d, a + adv, w + adv, idesc, (fresh && k == 0) ? 0u : 1u);
                        }
                    } else {
                        const uint32_t idesc = make_idesc_bf16(ML1_ROWS, N);
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            const uint64_t adv = (uint64_t)((k * 32) >> 4); // 16 BF16 = 32 bytes along K
                            umma_bf16(d, a + adv, w + adv, idesc, (fresh && k == 0) ? 0u : 1u);
                        }
                    }
                }
                umma_commit(bars + b);                                   // A buffer b reusable once these retire
            }
            if (b == 0) pend0 = true; else pend1 = true;
        }
        if (!P.project) continue;
        // the last commit retires after every MMA of the tile: wait for both buffers, then drain the accumulator
        if (pend0) { mbar_wait(bars, ph0); ph0 ^= 1; pend0 = false; }
        if (pend1) { mbar_wait(bars + 1, ph1); ph1 ^= 1; pend1 = false; }
        tc_fence_after();
        const int q = warp & 3, part = warp >> 2;            // tensor-memory lane quarter of this warp, column share
        const int64_t rr = row0 + 32 * q + lane;
        const bool ok = rr < P.N;
        const uint32_t trow = tmem_base + ((uint32_t)(32 * q) << 16);
        if (P.epi == 0) {
            for (int j = part; j * 16 < P.Nout; j += 4) {
                float a[16];
                tmem_ld16(trow + j * 16, a);
                if (ok) {
                    float* o = P.out + rr * P.ldo;
#pragma unroll
                    for (int u = 0; u < 16; ++u)
                        if (j * 16 + u < P.Nout) o[j * 16 + u] = a[u];
                }
            }
        } else {
            const int Fo = P.Fo, Fop = P.Fop;
            for (int j = part; j * 16 < Fo; j += 4) {
                float p0[16], p1[16], p2[16], pc[16];
                tmem_ld16(trow + j * 16, p0);
                tmem_ld16(trow + Fop + j * 16, p1);
                tmem_ld16(trow + 2 * Fop + j * 16, p2);
                if (P.epi == 2) tmem_ld16(trow + P.colG + j * 16, pc);
                if (ok) {
                    float* yr = P.out + rr * P.ldo;
                    float* ar = P.aux + rr * P.ldaux;
#pragma unroll
                    for (int u = 0; u < 16; ++u) {
                        const int o = j * 16 + u;
                        if (o >= Fo) break;
                        const float q1 = p1[u] + (P.bB ? __ldg(P.bB + o) : 0.f);
                        const float q2 = p2[u] + (P.bC ? __ldg(P.bC + o) : 0.f);
                        const float ba = P.bA ? __ldg(P.bA + o) : 0.f, bc = P.bc ? __ldg(P.bc + o) : 0.f;
                        if constexpr (AUX) {
                            ar[o] = q1;
                            ar[Fo + o] = q2;
                        }
                        if (P.epi == 1) {
                            yr[o] = fmaxf(p0[u] + ba + bc + q1 * q2, 0.f);
                        } else {
                            yr[o] = fmaxf(p0[u] + ba, 0.f);
                            yr[Fo + o] = fmaxf(pc[u] + bc, 0.f);
                            yr[2 * Fo + o] = fmaxf(q1 * q2, 0.f);
                        }
                    }
                }
            }
        }
        tc_fence_before();
        __syncthreads();                                     // accumulator drained before the next tile's MMAs
    }
    tc_fence_before();
    __syncthreads();
    if (P.project && warp == 0) tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
}

__device__ __forceinline__ int ml1_swz(int n, int k) {      // float index of element (row n, column k) of a swizzled plane
    return (n >> 3) * 256 + (n & 7) * 32 + ((((k >> 2) ^ (n & 7))) << 2) + (k & 3);
}

// Weight planes of one launch in the kernel's shared-memory byte layout.  dir 0 (forward): self block rows n = output
// column (group b = n / Fop of [fcA | fcB | fcC], feature o = n % Fop), k = input feature; gathered rows n = output column of
// Wc [Fi, Fo].  dir 1 (dx): self rows n = input feature i, k over [gA | gP p2 | gP p1] (block pitch Fo4); gathered rows
// n = i, k = o of Wc^T.  PREC 0: a hi plane (RN-TF32) then a lo plane (w - hi) per k-block; PREC 1: the hi plane alone;
// PREC 2: one plane of RN-BF16 values in the first 64 bytes of each row (the kernel's BF16 A layout), the rest zero.
template <int PREC = GNNML3_PREC_3XTF32>
__global__ void k_ml1_prep(const float* __restrict__ wc, const float* __restrict__ wA, const float* __restrict__ wB,
                           const float* __restrict__ wC, int Fi, int Fo, int dir, int nsb, int NsP, int ngb, int NgP, int Fop,
                           int Fo4, float* __restrict__ planes) {
    const int ts = nsb * NsP * 32, total = ts + ngb * NgP * 32;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const bool self = idx < ts;
        const int NP = self ? NsP : NgP;
        const int j = self ? idx : idx - ts;
        const int kb = j / (NP * 32), n = (j / 32) % NP, k = j % 32, kk = kb * 32 + k;
        float v = 0.f;
        if (dir == 0) {
            if (self) {
                const int g = n / Fop, o = n % Fop;
                const float* w = g == 0 ? wA : (g == 1 ? wB : wC);
                if (g < 3 && o < Fo && kk < Fi) v = __ldg(w + (int64_t)o * Fi + kk);
            } else if (kk < Fi && n < Fo) {
                v = __ldg(wc + (int64_t)kk * Fo + n);
            }
        } else {
            if (self) {
                const int g = kk / Fo4, o = kk % Fo4;
                const float* w = g == 0 ? wA : (g == 1 ? wB : wC);
                if (g < 3 && o < Fo && n < Fi) v = __ldg(w + (int64_t)o * Fi + n);
            } else if (kk < Fo && n < Fi) {
                v = __ldg(wc + (int64_t)n * Fo + kk);
            }
        }
        if constexpr (PREC == GNNML3_PREC_3XTF32) {
            const float h = tf32_rn(v);
            float* base = planes + (self ? (size_t)kb * 2 * NsP * 32 : (size_t)nsb * 2 * NsP * 32 + (size_t)kb * 2 * NgP * 32);
            base[ml1_swz(n, k)] = h;
            base[NP * 32 + ml1_swz(n, k)] = v - h;
        } else {
            float* base = planes + (self ? (size_t)kb * NsP * 32 : (size_t)nsb * NsP * 32 + (size_t)kb * NgP * 32);
            if constexpr (PREC == GNNML3_PREC_TF32) {
                base[ml1_swz(n, k)] = tf32_rn(v);
            } else {
                __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(base) + (n >> 3) * 512 + (n & 7) * 64 + (k & 7);
                row[((k >> 3) ^ (n & 7)) << 3] = __float2bfloat16_rn(v);
                row[(((k >> 3) + 4) ^ (n & 7)) << 3] = __float2bfloat16_rn(0.f);
            }
        }
    }
}

// d pre of the layer from its outputs.  GG [N, 5 Fo4] (block pitch Fo4, padding columns zero):
//   block 0 = d p0 (gA), 1 = d p1 = gP * p2, 2 = d p2 = gP * p1, 3 = A^T gc (written by the dx pass), 4 = gc (concat mode)
// sum mode: gA = gP = gc = gy * (y > 0);  concat mode: the three branch masks.
__global__ void k_ml1_act_bwd(const float* __restrict__ y, int64_t ldy, const float* __restrict__ aux, int64_t ldaux,
                              const float* __restrict__ gy, int64_t ldgy, int64_t N, int Fo, int Fo4, int concat,
                              float* __restrict__ GG, int64_t ldgg) {
    const int64_t total = N * Fo4;
    for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = idx / Fo4;
        const int o = (int)(idx - r * Fo4);
        float* g = GG + r * ldgg + o;
        if (o >= Fo) {
            g[0] = 0.f;
            g[Fo4] = 0.f;
            g[2 * Fo4] = 0.f;
            g[4 * Fo4] = 0.f;
            continue;
        }
        const float* yr = y + r * ldy;
        const float* gr = gy + r * ldgy;
        const float p1 = __ldg(aux + r * ldaux + o), p2 = __ldg(aux + r * ldaux + Fo + o);
        if (!concat) {
            const float gz = __ldg(yr + o) > 0.f ? __ldg(gr + o) : 0.f;
            g[0] = gz;
            g[Fo4] = gz * p2;
            g[2 * Fo4] = gz * p1;
            g[4 * Fo4] = gz;
        } else {
            const float ga = __ldg(yr + o) > 0.f ? __ldg(gr + o) : 0.f;
            const float gc = __ldg(yr + Fo + o) > 0.f ? __ldg(gr + Fo + o) : 0.f;
            const float gp = __ldg(yr + 2 * Fo + o) > 0.f ? __ldg(gr + 2 * Fo + o) : 0.f;
            g[0] = ga;
            g[Fo4] = gp * p2;
            g[2 * Fo4] = gp * p1;
            g[4 * Fo4] = gc;
        }
    }
}

// dcat [Fi, 4 Fo4] = x^T GG[:, 0:4 Fo4], csum [5 Fo4] = column sums of GG  ->  the eight parameter gradients
__global__ void k_ml1_unpack(const float* __restrict__ dcat, const float* __restrict__ csum, int Fi, int Fo, int Fo4,
                             float* __restrict__ dwc, float* __restrict__ dbc, float* __restrict__ dwA, float* __restrict__ dbA,
                             float* __restrict__ dwB, float* __restrict__ dbB, float* __restrict__ dwC, float* __restrict__ dbC) {
    const int t = Fi * Fo, ld = 4 * Fo4;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 4 * t + 4 * Fo; idx += gridDim.x * blockDim.x) {
        if (idx < t) {                                            // Wc [1, Fi, Fo]
            const int i = idx / Fo, o = idx % Fo;
            dwc[idx] = __ldg(dcat + (int64_t)i * ld + 3 * Fo4 + o);
        } else if (idx < 4 * t) {                                 // fcA / fcB / fcC weight [Fo, Fi]
            const int g = idx / t - 1, j = idx % t, o = j / Fi, i = j % Fi;
            float* dw = g == 0 ? dwA : (g == 1 ? dwB : dwC);
            dw[j] = __ldg(dcat + (int64_t)i * ld + g * Fo4 + o);
        } else {
            const int j = idx - 4 * t, g = j / Fo, o = j % Fo;
            if (g == 0 && dbA) dbA[o] = __ldg(csum + o);
            if (g == 1 && dbB) dbB[o] = __ldg(csum + Fo4 + o);
            if (g == 2 && dbC) dbC[o] = __ldg(csum + 2 * Fo4 + o);
            if (g == 3 && dbc) dbc[o] = __ldg(csum + 4 * Fo4 + o);
        }
    }
}

static inline size_t ml1_a256(size_t x) { return align_up(x, 256); }
static inline int ml1_c16(int v) { return (v + 15) / 16 * 16; }
static inline int ml1_c4(int v) { return (v + 3) / 4 * 4; }

// launch geometry of one direction
struct ML1Shape {
    int nsb, NsP, ngb, NgP, colG, tmem_cols, Fop, Fo4;
    size_t wbytes, smem;
};

static ML1Shape ml1_shape(int Fi, int Fo, int concat, int dir, int prec = GNNML3_PREC_3XTF32) {
    ML1Shape s;
    s.Fop = ml1_c16(Fo);
    s.Fo4 = ml1_c4(Fo);
    if (dir == 0) {
        s.nsb = (Fi + 31) / 32;
        s.NsP = 3 * s.Fop;
        s.ngb = (Fi + 31) / 32;
        s.NgP = s.Fop;
        s.colG = concat ? 3 * s.Fop : 0;
    } else {
        s.nsb = (3 * s.Fo4 + 31) / 32;
        s.NsP = ml1_c16(Fi);
        s.ngb = (Fo + 31) / 32;
        s.NgP = ml1_c16(Fi);
        s.colG = 0;
    }
    const int cols = s.colG + s.NgP > s.NsP ? s.colG + s.NgP : s.NsP;
    s.tmem_cols = 32;
    while (s.tmem_cols < cols) s.tmem_cols *= 2;
    s.wbytes = (size_t)ml1_planes(prec) * 128 * ((size_t)s.nsb * s.NsP + (size_t)s.ngb * s.NgP);
    s.smem = 1024 + s.wbytes + (size_t)2 * ml1_planes(prec) * ML1_APLANE + 64;
    return s;
}

// workspace layout: [planes | GG | dcat | csum | colsum scratch | gemm_tn scratch]; sized by the 3xTF32 shapes, the largest
struct ML1Ws {
    size_t planes, gg, dcat, csum, cs, tn, total_fwd, total;
    int64_t ldgg;
};

static ML1Ws ml1_ws(int64_t N, int Fi, int Fo, int concat) {
    ML1Ws w;
    const ML1Shape f = ml1_shape(Fi, Fo, concat, 0), b = ml1_shape(Fi, Fo, concat, 1);
    const int Fo4 = f.Fo4;
    size_t off = 0;
    w.planes = off; off += ml1_a256(f.wbytes > b.wbytes ? f.wbytes : b.wbytes);
    w.total_fwd = off;
    w.ldgg = 5 * Fo4;
    w.gg = off; off += ml1_a256((size_t)N * w.ldgg * 4);
    w.dcat = off; off += ml1_a256((size_t)Fi * 4 * Fo4 * 4);
    w.csum = off; off += ml1_a256((size_t)5 * Fo4 * 4);
    w.cs = off; off += ml1_a256(gnnml3_colsum_workspace_bytes(N > 0 ? N : 1, 5 * Fo4));
    w.tn = off; off += ml1_a256(gnnml3_gemm_tn_workspace_bytes(N > 0 ? N : 1, Fi, 4 * Fo4));
    w.total = off;
    return w;
}

template <bool AUX, int PREC>
static int ml1_launch(const ML1Params& P, size_t smem, cudaStream_t st) {
    static bool configured[64] = {};
    if (auto once = first_use_on_device(configured))
        GNNML3_CUDA(cudaFuncSetAttribute(k_ml1_agg_proj<AUX, PREC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    const int grid = P.n_tiles < kNumSMs ? P.n_tiles : kNumSMs;
    k_ml1_agg_proj<AUX, PREC><<<grid, ML1_THREADS, smem, st>>>(P);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

// the instantiation of (aux written, precision)
static int ml1_launch(const ML1Params& P, size_t smem, bool aux, int prec, cudaStream_t st) {
    if (prec == GNNML3_PREC_TF32) return aux ? ml1_launch<true, GNNML3_PREC_TF32>(P, smem, st) : ml1_launch<false, GNNML3_PREC_TF32>(P, smem, st);
    if (prec == GNNML3_PREC_BF16) return aux ? ml1_launch<true, GNNML3_PREC_BF16>(P, smem, st) : ml1_launch<false, GNNML3_PREC_BF16>(P, smem, st);
    return aux ? ml1_launch<true, GNNML3_PREC_3XTF32>(P, smem, st) : ml1_launch<false, GNNML3_PREC_3XTF32>(P, smem, st);
}

static int ml1_prep(const float* wc, const float* wA, const float* wB, const float* wC, int Fi, int Fo, int dir, const ML1Shape& s,
                    int prec, float* planes, cudaStream_t st) {
    const int grid = cdiv((int64_t)s.wbytes / (4 * ml1_planes(prec)), 256);     // one thread per weight
    if (prec == GNNML3_PREC_TF32)
        k_ml1_prep<GNNML3_PREC_TF32><<<grid, 256, 0, st>>>(wc, wA, wB, wC, Fi, Fo, dir, s.nsb, s.NsP, s.ngb, s.NgP, s.Fop, s.Fo4, planes);
    else if (prec == GNNML3_PREC_BF16)
        k_ml1_prep<GNNML3_PREC_BF16><<<grid, 256, 0, st>>>(wc, wA, wB, wC, Fi, Fo, dir, s.nsb, s.NsP, s.ngb, s.NgP, s.Fop, s.Fo4, planes);
    else
        k_ml1_prep<GNNML3_PREC_3XTF32><<<grid, 256, 0, st>>>(wc, wA, wB, wC, Fi, Fo, dir, s.nsb, s.NsP, s.ngb, s.NgP, s.Fop, s.Fo4, planes);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

}  // namespace gnnml3

using namespace gnnml3;

extern "C" int gnnml3_ml1layer_supported(int Fi, int Fo, int concat) {
    (void)concat;
    return Fi >= 1 && Fi <= 64 && Fo >= 1 && Fo <= 64 ? 1 : 0;
}

extern "C" size_t gnnml3_ml1layer_workspace_bytes(int64_t N, int Fi, int Fo, int concat) {
    return ml1_ws(N, Fi, Fo, concat).total;
}

extern "C" int gnnml3_ml1layer_forward(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E, const float* x, int64_t ldx,
                                       int Fi, const float* wconv, const float* bconv, const float* wA, const float* bA,
                                       const float* wB, const float* bB, const float* wC, const float* bC, int Fo, int concat,
                                       float* y, int64_t ldy, float* aux, int64_t ldaux, float* hside, int64_t ldh,
                                       void* workspace, size_t workspace_bytes, void* stream, int precision) {
    GNNML3_REQUIRE(prec_valid(precision), "ml1layer_forward: unknown precision %d (GNNML3_PREC_3XTF32, _TF32 or _BF16)", precision);
    GNNML3_REQUIRE(gnnml3_ml1layer_supported(Fi, Fo, concat), "ml1layer_forward: unsupported shape Fi=%d Fo=%d", Fi, Fo);
    GNNML3_REQUIRE(N >= 0 && E >= 0 && rowptr && x && wconv && wA && wB && wC && y, "ml1layer_forward: NULL pointer");
    GNNML3_REQUIRE(E == 0 || col, "ml1layer_forward: NULL col");
    GNNML3_REQUIRE(ldx >= Fi && ldx % 4 == 0 && ((uintptr_t)x & 15) == 0, "ml1layer_forward: x rows must be 16-byte aligned");
    GNNML3_REQUIRE(ldy >= (concat ? 3 : 1) * Fo && (!aux || ldaux >= 2 * Fo), "ml1layer_forward: output leading dimensions too small");
    GNNML3_REQUIRE(hside == nullptr || (ldh >= Fi && ldh % 4 == 0 && ((uintptr_t)hside & 15) == 0),
                   "ml1layer_forward: hside rows must be 16-byte aligned and hold Fi floats");
    const ML1Ws w = ml1_ws(N, Fi, Fo, concat);
    if (workspace_bytes < w.total_fwd) return set_err(GNNML3_ERR_WORKSPACE, "ml1layer_forward: workspace too small");
    if (N == 0) return GNNML3_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const ML1Shape s = ml1_shape(Fi, Fo, concat, 0, precision);
    float* planes = (float*)((uint8_t*)workspace + w.planes);
    int rc;
    if ((rc = ml1_prep(wconv, wA, wB, wC, Fi, Fo, 0, s, precision, planes, st))) return rc;
    ML1Params P = {};
    P.rowptr = rowptr; P.col = col; P.N = N; P.n_tiles = cdiv(N, ML1_ROWS);
    P.X = x; P.ldx = ldx; P.Fg = Fi; P.ngb = s.ngb;
    P.S = x; P.lds = ldx; P.Fs = Fi; P.nsb = s.nsb;
    P.planes = planes; P.wbytes = (int)s.wbytes; P.NsP = s.NsP; P.NgP = s.NgP; P.colG = s.colG; P.tmem_cols = s.tmem_cols;
    P.project = 1; P.epi = concat ? 2 : 1; P.Fo = Fo; P.Fop = s.Fop;
    P.bA = bA; P.bB = bB; P.bC = bC; P.bc = bconv;
    P.out = y; P.ldo = ldy; P.aux = aux; P.ldaux = ldaux; P.hout = hside; P.ldh = ldh;
    return ml1_launch(P, s.smem, aux != nullptr, precision, st);     // no aux: the forward-only instantiation
}

extern "C" int gnnml3_ml1layer_backward(const int32_t* rowptrT, const int32_t* colT, int64_t N, int64_t E, const float* x, int64_t ldx,
                                        int Fi, const float* wconv, const float* wA, const float* wB, const float* wC, int Fo, int concat,
                                        const float* y, int64_t ldy, const float* aux, int64_t ldaux, const float* gy, int64_t ldgy,
                                        int need_dx, float* dx, int64_t lddx, float* dwconv, float* dbconv, float* dwA, float* dbA,
                                        float* dwB, float* dbB, float* dwC, float* dbC, void* workspace, size_t workspace_bytes,
                                        void* stream, int precision) {
    GNNML3_REQUIRE(prec_valid(precision), "ml1layer_backward: unknown precision %d (GNNML3_PREC_3XTF32, _TF32 or _BF16)", precision);
    GNNML3_REQUIRE(gnnml3_ml1layer_supported(Fi, Fo, concat), "ml1layer_backward: unsupported shape Fi=%d Fo=%d", Fi, Fo);
    GNNML3_REQUIRE(N > 0, "ml1layer_backward: empty batch");
    GNNML3_REQUIRE(E >= 0 && rowptrT && (E == 0 || colT) && x && wconv && wA && wB && wC && y && aux && gy && dwconv && dwA && dwB && dwC,
                   "ml1layer_backward: NULL pointer");
    GNNML3_REQUIRE(!need_dx || (dx && lddx >= Fi), "ml1layer_backward: dx missing");
    GNNML3_REQUIRE(ldx >= Fi && ldx % 4 == 0 && ((uintptr_t)x & 15) == 0, "ml1layer_backward: x rows must be 16-byte aligned");
    const ML1Ws w = ml1_ws(N, Fi, Fo, concat);
    if (workspace_bytes < w.total) return set_err(GNNML3_ERR_WORKSPACE, "ml1layer_backward: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)workspace;
    const ML1Shape s = ml1_shape(Fi, Fo, concat, 1, precision);
    const int Fo4 = s.Fo4;
    float* GG = (float*)(ws + w.gg);
    k_ml1_act_bwd<<<cdiv(N * Fo4, 256) > 4 * kNumSMs * 8 ? 4 * kNumSMs * 8 : cdiv(N * Fo4, 256), 256, 0, st>>>(
        y, ldy, aux, ldaux, gy, ldgy, N, Fo, Fo4, concat, GG, w.ldgg);
    GNNML3_LAUNCH_CHECK();
    // dx = (A^T gc) Wc^T + [gA | gP p2 | gP p1] [fcA ; fcB ; fcC]; the aggregate A^T gc lands in block 3 of GG either way
    float* planes = (float*)(ws + w.planes);
    int rc;
    if (need_dx && (rc = ml1_prep(wconv, wA, wB, wC, Fi, Fo, 1, s, precision, planes, st))) return rc;
    ML1Params P = {};
    P.rowptr = rowptrT; P.col = colT; P.N = N; P.n_tiles = cdiv(N, ML1_ROWS);
    P.X = GG + 4 * Fo4; P.ldx = w.ldgg; P.Fg = Fo; P.ngb = s.ngb;
    P.S = GG; P.lds = w.ldgg; P.Fs = 3 * Fo4; P.nsb = need_dx ? s.nsb : 0;
    P.planes = planes; P.wbytes = need_dx ? (int)s.wbytes : 0; P.NsP = s.NsP; P.NgP = s.NgP; P.colG = 0; P.tmem_cols = s.tmem_cols;
    P.project = need_dx ? 1 : 0; P.epi = 0; P.out = dx; P.ldo = lddx; P.Nout = Fi;
    P.hout = GG + 3 * Fo4; P.ldh = w.ldgg;
    if ((rc = ml1_launch(P, need_dx ? s.smem : 1024 + 2 * ML1_ABUF + 64, true, precision, st))) return rc;
    // [dfcA^T | dfcB^T | dfcC^T | dWc] = x^T GG[:, 0:4 Fo4] in one contraction (the GEMM runs BF16 as single-pass TF32);
    // bias gradients = column sums (fixed order)
    float* dcat = (float*)(ws + w.dcat);
    float* csum = (float*)(ws + w.csum);
    if ((rc = gnnml3_gemm_tn(x, ldx, GG, w.ldgg, dcat, 4 * Fo4, N, Fi, 4 * Fo4, precision, ws + w.tn, w.total - w.tn, stream)))
        return rc;
    if ((rc = gnnml3_colsum(GG, w.ldgg, N, 5 * Fo4, csum, ws + w.cs, w.tn - w.cs, stream))) return rc;
    k_ml1_unpack<<<cdiv(4 * Fi * Fo + 4 * Fo, 256), 256, 0, st>>>(dcat, csum, Fi, Fo, Fo4, dwconv, dbconv, dwA, dbA, dwB, dbB, dwC, dbC);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}
