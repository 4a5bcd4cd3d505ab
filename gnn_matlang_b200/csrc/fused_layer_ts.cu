// Fused aggregate + project kernel, second generation: the aggregate lives in TENSOR MEMORY.
//
// Same contract as fused_layer.cu (reference libs/spect_conv.py:70-80,93-94 and :208-212):
//     conv[t, :] = sum_k ( sum_{e: dst_e = t} ea[e, k] * x[src_e, :] ) W_k  + bias            (SpectConv)
//     y[t, :]    = [ relu(conv[t, :]) || tanh(x[t] W11^T + b11) * tanh(x[t] W12^T + b12) ]    (ML3Layer)
// What changed, and why (measured on B200, profiles/r02_tmem_probe.txt and the round-1 ncu captures):
//   * the round-1 kernel wrote every 32-column block of the aggregate H twice into shared memory (raw + residual plane,
//     8 bytes per element) and the tensor core read both back: ~0.9 MB of shared-memory traffic per 128-row tile, more than
//     anything else the SM did.  Here the aggregator warps hand H to the tensor core through TENSOR MEMORY: tcgen05.st
//     (16x64b.x16: two threads per row, each thread owns one row's odd or even columns) writes the raw FP32 block (the
//     tensor core truncates it to TF32 itself = the hi part) and the residual block lo = a - trunc(a) into a ring of four
//     64-column slots, and tcgen05.mma reads its A operand from there (A in TMEM, M = 128 tile rows on the 128 lanes).
//     Shared memory now only holds the weights (B operand, N side) and the staged source rows.
//   * tcgen05.mma costs max(45, N/2) cycles (not "143 whatever the shape": that was the round-1 probe's own loop).  With
//     the rows on M and the weights on N, a k-step is  D[:, 0:2B] += H_raw [W_hi | W_lo]^T  (N = 2B)  followed by
//     D[:, B:2B] += H_lo W_hi^T  (N = B):  ~90 cycles per 128 rows instead of 128, and no wasted lo x lo product.
//     The hi x hi sum keeps its own accumulator columns (chain of 4 * K additions per tile, as before).
//   * the gathered source rows come from SHARED MEMORY: a batched disjoint graph only has edges inside a graph, so the
//     sources of a 128-row tile lie in a window of at most 128 + 2 * (largest graph - 1) consecutive rows of X.  The
//     per-tile window [first, last] is part of the graph plan (gnnml3_tile_windows); a producer thread brings the window
//     in with ONE TMA box load (256 rows x 128 B, 128B-swizzled, zero-filled outside X), one tile ahead, double buffered.
//     Each source row is then read from L2 once per tile instead of once per edge and pass (5.6x less L2 traffic on the
//     ZINC batches), and the dependent chain col -> x row ends in a 29-cycle LDS instead of a ~300-cycle L2 round trip.
//     Tiles whose window does not fit (general graphs) gather from global memory as before -- same arithmetic.
// Summation order per row = edge order of the CSR row (the reference's CPU scatter order); no atomics.
#include "tc_common.cuh"

#include <cuda_bf16.h>
#include <atomic>
#include <vector>

namespace gnnml3 {

constexpr int TS_ROWS = 128;                     // dst rows per tile = TMEM lanes = MMA M
constexpr int TS_WIN_ROWS = 256;                 // rows of the staged source window (one TMA box)
constexpr int TS_NSLOT = 6;                      // ring of H slots in tensor memory (64 columns each: raw | lo)
constexpr int TS_SLOT0 = 128;                    // first tensor-memory column of the ring (columns 0-127: the accumulator)
constexpr int TS_THREADS = 512;
// Warp roles.  The scheduler arbitrates highest warp id first, so the roles that issue few but latency-critical instructions
// sit at the top: warp 15 MMA issuer, 12-14 stagers, 8-11 epilogue, 0-7 aggregators (the bulk of the instruction stream).
constexpr int TS_AGG0 = 0;
constexpr int TS_EPI0 = 8;
constexpr int TS_STG0 = 12;
constexpr int TS_MMAW = 15;

struct TSParams {
    const int* rowptr;
    const int* col;
    const int* eperm;
    const float* ea;
    int Kstride, K;
    const float* X;
    int64_t ldx;
    int F;
    const float* S;
    int64_t lds;
    int Fs;
    int self_mode;          // 0 none | 1 own output columns (ML3 gates) | 2 accumulates into the main columns
    int64_t N;
    int n_tiles;
    int nkb_main;           // = K (one 32-wide feature block per support)
    const int2* tilewin;    // [n_tiles] {first, last + 1} source row of the tile's CSR slots; NULL: gather from global memory
    int win_rows;           // rows of the TMA box (<= TS_WIN_ROWS)
    int edge_cap;           // CSR slots per tile the staging buffer holds (0: never stage)
    const float* bias;
    const float* bias_s;
    float* out;
    int64_t ldo;
    int Nc;
    float* aux;
    int64_t ldaux;
    int G;
    int epi;                // 0 plain (+bias) | 1 ml3: relu on the main columns, tanh*tanh gating on the self columns
    int prec;               // 0 FP32-grade 3xTF32 | 1 single-pass TF32 | 2 BF16 inputs (both: FP32 accumulate, no residual blocks)
    float* hout;            // optional copy of the aggregate [N, ldh]: support k at column 32 k, self block behind
    int64_t ldh;
    unsigned long long* dbg;
};

__device__ __forceinline__ void ts_mbar_wait_idle(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(32);
    }
}

// mbarrier wait for the stagers (a tile ahead of everybody, never latency-critical): long sleeps between polls, so that the
// waiting warps do not spend issue slots (the try_wait suspend-time hint did not reduce the polling: measured)
__device__ __forceinline__ void ts_mbar_wait_sleepy(uint64_t* bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(200);
    }
}

__device__ __forceinline__ bool ts_elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// contiguous global -> shared bulk copy (16-byte aligned, size % 16 == 0), completion counted in bytes on an mbarrier
__device__ __forceinline__ void ts_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float ts_lo(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

__device__ __forceinline__ float4 ts_lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}

// 16 TMEM lanes x 32 columns: thread T owns lane 8 * (T & 1) + (T >> 2) and the 16 columns ((T >> 1) & 1) + 2 j
// (layout pinned on the B200 by scratch/tmem_probe.cu)
__device__ __forceinline__ void ts_st_16x64b_x16(uint32_t taddr, const float* v) {
    asm volatile("tcgen05.st.sync.aligned.16x64b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
                 "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]), "f"(v[10]),
                 "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
                 : "memory");
}
// 16 TMEM lanes x 16 columns (same thread <-> lane / column-parity map, 8 registers)
__device__ __forceinline__ void ts_st_16x64b_x8(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.16x64b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
                 "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void ts_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// tensor-memory loads without the trailing wait (several loads, then one ts_ld_wait)
__device__ __forceinline__ void ts_tmem_ld32_nw(uint32_t taddr, float (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]), "=f"(v[10]),
          "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15]), "=f"(v[16]), "=f"(v[17]), "=f"(v[18]), "=f"(v[19]), "=f"(v[20]),
          "=f"(v[21]), "=f"(v[22]), "=f"(v[23]), "=f"(v[24]), "=f"(v[25]), "=f"(v[26]), "=f"(v[27]), "=f"(v[28]), "=f"(v[29]), "=f"(v[30]),
          "=f"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void ts_tmem_ld16_nw(uint32_t taddr, float (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]), "=f"(v[8]), "=f"(v[9]), "=f"(v[10]),
          "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void ts_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem desc]^T, TF32 inputs (truncated by the tensor core), FP32 accumulate
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// same with BF16 inputs (kind::f16, K = 16 per instruction: two BF16 per 32-bit tensor-memory column), FP32 accumulate
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// this thread's 16 features of a block -> 8 packed BF16 pairs (features 2j, 2j+1 of the thread's 16 in register j)
__device__ __forceinline__ void ts_pack_bf16(const float* v, uint32_t (&r)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        r[j] = *reinterpret_cast<const uint32_t*>(&h);
    }
}

template <int KT>
__device__ __forceinline__ void ts_load_w(const float* __restrict__ p, float (&w)[KT]) {
    if constexpr (KT == 4) {
        const float4 v = ldg4(p);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    } else if constexpr (KT == 2) {
        const float2 v = ldg2(p);
        w[0] = v.x; w[1] = v.y;
    } else {
#pragma unroll
        for (int k = 0; k < KT; ++k) w[k] = __ldg(p + k);
    }
}

template <int KT>
__device__ __forceinline__ void ts_fma(float (&acc)[KT][16], const float (&w)[KT], const float4& x0, const float4& x1, const float4& x2,
                                       const float4& x3) {
#pragma unroll
    for (int k = 0; k < KT; ++k) {
        acc[k][0] = fmaf(w[k], x0.x, acc[k][0]);
        acc[k][1] = fmaf(w[k], x0.y, acc[k][1]);
        acc[k][2] = fmaf(w[k], x0.z, acc[k][2]);
        acc[k][3] = fmaf(w[k], x0.w, acc[k][3]);
        acc[k][4] = fmaf(w[k], x1.x, acc[k][4]);
        acc[k][5] = fmaf(w[k], x1.y, acc[k][5]);
        acc[k][6] = fmaf(w[k], x1.z, acc[k][6]);
        acc[k][7] = fmaf(w[k], x1.w, acc[k][7]);
        acc[k][8] = fmaf(w[k], x2.x, acc[k][8]);
        acc[k][9] = fmaf(w[k], x2.y, acc[k][9]);
        acc[k][10] = fmaf(w[k], x2.z, acc[k][10]);
        acc[k][11] = fmaf(w[k], x2.w, acc[k][11]);
        acc[k][12] = fmaf(w[k], x3.x, acc[k][12]);
        acc[k][13] = fmaf(w[k], x3.y, acc[k][13]);
        acc[k][14] = fmaf(w[k], x3.z, acc[k][14]);
        acc[k][15] = fmaf(w[k], x3.w, acc[k][15]);
    }
}

// eight of a thread's sixteen features (two 16-byte chunks of the source row) into the KT accumulator sets
template <int KT, int H>
__device__ __forceinline__ void ts_fma_half(float (&acc)[KT][16], const float (&w)[KT], const float4& a, const float4& b) {
#pragma unroll
    for (int k = 0; k < KT; ++k) {
        acc[k][8 * H + 0] = fmaf(w[k], a.x, acc[k][8 * H + 0]);
        acc[k][8 * H + 1] = fmaf(w[k], a.y, acc[k][8 * H + 1]);
        acc[k][8 * H + 2] = fmaf(w[k], a.z, acc[k][8 * H + 2]);
        acc[k][8 * H + 3] = fmaf(w[k], a.w, acc[k][8 * H + 3]);
        acc[k][8 * H + 4] = fmaf(w[k], b.x, acc[k][8 * H + 4]);
        acc[k][8 * H + 5] = fmaf(w[k], b.y, acc[k][8 * H + 5]);
        acc[k][8 * H + 6] = fmaf(w[k], b.z, acc[k][8 * H + 6]);
        acc[k][8 * H + 7] = fmaf(w[k], b.w, acc[k][8 * H + 7]);
    }
}

// shared-memory loads the compiler may schedule (no volatile, no memory clobber): only for data that does not change between
// the barrier wait their address depends on and the barrier arrive that releases the buffer
__device__ __forceinline__ float4 ts_lds128_nv(uint32_t a) {
    float4 v;
    asm("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ int ts_lds32_nv(uint32_t a) {
    int v;
    asm("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
template <int KT>
__device__ __forceinline__ void ts_lds_w_nv(uint32_t a, float (&w)[KT]) {
    if constexpr (KT == 4) {
        const float4 t = ts_lds128_nv(a);
        w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
    } else {
#pragma unroll
        for (int k = 0; k < KT; ++k) asm("ld.shared.f32 %0, [%1];" : "=f"(w[k]) : "r"(a + 4 * k));
    }
}

template <int KT>
__device__ __forceinline__ void ts_lds_w(uint32_t a, float (&w)[KT]) {
    if constexpr (KT == 4) {
        const float4 t = ts_lds128(a);
        w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w;
    } else {
#pragma unroll
        for (int k = 0; k < KT; ++k) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(w[k]) : "r"(a + 4 * k));
    }
}

#ifdef FL_PROFILE
#define TS_CNT(...) __VA_ARGS__
#else
#define TS_CNT(...)
#endif

// Per-tile staging buffer (two of them): the source-row window, then the tile's CSR slots.
//   [0, TS_WIN_ROWS * 128)                      x window (TMA box, 128B swizzle)
//   + cap * Kstride floats                      edge weights of the tile's slots, slot-major (already through eperm)
//   + cap ints                                  source row of every slot
//   + 132 ints                                  rowptr of the tile's 129 row bounds
//   + 4 ints                                    {first slot, last slot + 1, first window row, staged}
__host__ __device__ constexpr size_t ts_stage_bytes(int cap, int Kstride) {
    return (size_t)TS_WIN_ROWS * 128 + (size_t)cap * Kstride * 4 + (size_t)cap * 4 + 132 * 4 + 16;
}

// KT = supports per register pass (K % KT == 0).  BNH = 32: Nc <= 32 (+ optional gate block), 64: Nc <= 64.
// Tensor-memory map (512 columns): ONE accumulator at columns 0-127 (main [0, 2 BNH): hi-weight | lo-weight partial sums,
// gates [64, 128) when BNH = 32) and a ring of six H slots at 128 + 64 s (raw columns 0-31, residual columns 32-63).  A tile
// hands over K + 1 blocks in bursts of KT: six slots give the aggregator warps a whole register pass of slack against each
// other (the MMA on a block needs all eight warps' parts), which a second accumulator buffer + four slots did not (measured:
// 17 % of the aggregators' time was spent waiting for slots).  The epilogue drains the accumulator while the aggregators
// gather the next tile's first pass.
// Column c of a slot holds feature 16 * (c & 1) + (c >> 1) of the 32-wide block (the store layout gives a thread the even
// or the odd columns; it gathers features 0-15 or 16-31): the weight planes are permuted the same way (k_ts_prep_weights).
// AUX = false: the forward-only instantiation of the gated epilogue (aux == NULL), which stores y and not the tanh factors.
template <int KT, int BNH, bool AUX = true>
__global__ void __launch_bounds__(TS_THREADS, 1)
k_fused_ts(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapX, const __grid_constant__ TSParams P) {
    constexpr int WPLANE = 2 * BNH * 128;               // bytes of one weight plane: rows [W_hi^T ; W_lo^T] x 32 k-columns
    constexpr uint32_t ID_FULL = make_idesc_tf32_mn(128, 2 * BNH), ID_HALF = make_idesc_tf32_mn(128, BNH);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // offset arithmetic keeps the shared address space (LDS/STS, not generic LD/ST)
    const int nkb_total = P.nkb_main + (P.self_mode != 0 ? 1 : 0);
    const int cap = P.edge_cap;
    const int Kstride = P.Kstride;
    const uint32_t stage_bytes = (uint32_t)((ts_stage_bytes(cap, Kstride) + 1023) & ~(size_t)1023);
    uint8_t* stage0 = smem;                                                 // [2][stage_bytes]
    uint8_t* wres = smem + 2 * (size_t)stage_bytes;                         // [nkb_total][WPLANE]
    uint64_t* bars = reinterpret_cast<uint64_t*>(wres + (size_t)nkb_total * WPLANE);
    uint64_t* full = bars;                       // [6]  slot written by the 8 aggregator warps      -> MMA
    uint64_t* empty = bars + 6;                  // [6]  MMAs that read the slot have retired         -> aggregators
    uint64_t* tfull = bars + 12;                 // [1]  tile accumulator complete                    -> epilogue
    uint64_t* tempty = bars + 13;                // [1]  accumulator drained                          -> MMA
    uint64_t* wfull = bars + 14;                 // [1]  weight planes landed                         -> MMA
    uint64_t* sfull = bars + 15;                 // [2]  tile staging buffer complete                 -> aggregators
    uint64_t* sempty = bars + 17;                // [2]  staging buffer no longer read                -> stagers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 19);
    float* sbias = reinterpret_cast<float*>(bars + 32);          // [64] main bias (zeros if none) | [32] gate biases

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TS_NSLOT; ++s) {
            mbar_init(full + s, 8);
            mbar_init(empty + s, 1);
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 4);
        for (int b = 0; b < 2; ++b) {
            mbar_init(sfull + b, 4);             // stager thread 0: expect_tx arrive (TMA / bulk-copy bytes); three stager warps: arrive
            mbar_init(sempty + b, 8);
        }
        mbar_init(wfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapW) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapX) : "memory");
    }
    if (threadIdx.x < 96) {
        float bv = 0.f;
        if (threadIdx.x < 64) {
            if (P.bias && (int)threadIdx.x < P.Nc) bv = __ldg(P.bias + threadIdx.x);
        } else if (P.bias_s && (int)threadIdx.x - 64 < 2 * P.G) {
            bv = __ldg(P.bias_s + threadIdx.x - 64);
        }
        sbias[threadIdx.x] = bv;
    }
    if (warp == TS_MMAW) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= TS_STG0 && warp < TS_STG0 + 3) {
        // =================================================================== stagers (3 warps), one tile ahead of the aggregators:
        // row bounds, source window (TMA box), CSR slots and edge weights of the tile -> shared memory
        const int tid = (warp - TS_STG0) * 32 + lane;
        constexpr int NSTG = 96;
        if (tid == 0) {                              // weight planes, once
            mbar_arrive_expect_tx(wfull, (uint32_t)nkb_total * WPLANE);
            for (int kb = 0; kb < nkb_total; ++kb) tma_load_2d(wres + (size_t)kb * WPLANE, &mapW, wfull, 0, kb * 2 * BNH);
        }
        const int KC = Kstride >> 2;                 // 16-byte chunks per edge-weight row (staging needs Kstride % 4 == 0)
        const int* __restrict__ col = P.col;
        const int* __restrict__ eperm = P.eperm;
        const float* __restrict__ ea = P.ea;
        uint32_t ts = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++ts) {
            const uint32_t b = ts & 1;
            uint8_t* sb = stage0 + (size_t)b * stage_bytes;
            float* sea = reinterpret_cast<float*>(sb + TS_WIN_ROWS * 128);
            int* scol = reinterpret_cast<int*>(sea + (size_t)cap * Kstride);
            int* srp = scol + cap;
            int* smeta = srp + 132;
            ts_mbar_wait_sleepy(sempty + b, ((ts >> 1) & 1) ^ 1);
            const int64_t r0 = (int64_t)tile * TS_ROWS;
            for (int i = tid; i <= TS_ROWS; i += NSTG) {
                const int64_t r = r0 + i < P.N ? r0 + i : P.N;
                srp[i] = __ldg(P.rowptr + r);
            }
            const int e0 = __ldg(P.rowptr + r0);
            const int e1 = __ldg(P.rowptr + (r0 + TS_ROWS < P.N ? r0 + TS_ROWS : P.N));
            int2 w = make_int2(0, 0);
            if (P.tilewin) w = __ldg(P.tilewin + tile);
            const bool staged = cap > 0 && w.y > w.x && w.y - w.x <= P.win_rows && e1 - e0 <= cap;
            const bool bulk_ea = staged && eperm == nullptr;          // contiguous edge weights: one bulk copy
            if (tid == 0) {
                smeta[0] = e0; smeta[1] = e1; smeta[2] = w.x; smeta[3] = staged ? 1 : 0;
                const uint32_t ea_bytes = bulk_ea ? (uint32_t)(e1 - e0) * (uint32_t)Kstride * 4u : 0u;
                mbar_arrive_expect_tx(sfull + b, staged ? (uint32_t)P.win_rows * 128u + ea_bytes : 0u);
                if (staged) tma_load_2d(sb, &mapX, sfull + b, 0, w.x);
                if (bulk_ea) ts_bulk_g2s(sea, ea + (int64_t)e0 * Kstride, ea_bytes, sfull + b);
            }
            if (staged) {
                if (bulk_ea) {
                    for (int e = e0 + tid; e < e1; e += NSTG) scol[e - e0] = __ldg(col + e);
                } else {
                    for (int e = e0 + tid; e < e1; e += 8 * NSTG) {            // eight slots per lane in flight
                        int c[8], ix[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int eu = e + NSTG * u;
                            c[u] = eu < e1 ? __ldg(col + eu) : 0;
                            ix[u] = eu < e1 ? __ldg(eperm + eu) : 0;
                        }
                        for (int h = 0; h < KC; ++h) {
                            float4 v[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (e + NSTG * u < e1) v[u] = ldg4(ea + (int64_t)ix[u] * Kstride + 4 * h);
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (e + NSTG * u < e1) *reinterpret_cast<float4*>(sea + (size_t)(e + NSTG * u - e0) * Kstride + 4 * h) = v[u];
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u)
                            if (e + NSTG * u < e1) scol[e + NSTG * u - e0] = c[u];
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(sfull + b);
        }
    } else if (warp == TS_MMAW) {
        // =================================================================== MMA issuer: the whole warp runs the loop (addresses
        // stay in uniform registers), one elected lane issues -- ~10 dependent instructions less per tcgen05.mma than a
        // single-lane branch
        mbar_wait(wfull, 0);
        uint32_t tt = 0, s = 0, sph = 0;
        const uint32_t wres0 = smem_u32(wres);
        TS_CNT(long long c_full = 0, c_tempty = 0; const long long c_begin = clock64();)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tt) {
            TS_CNT(long long c0 = clock64();)
            mbar_wait(tempty, (tt & 1) ^ 1);                    // the epilogue has drained the previous tile
            TS_CNT(c_tempty += clock64() - c0;)
            tc_fence_after();
            const uint32_t d_main = tmem_base;
            for (int kb = 0; kb < nkb_total; ++kb) {
                TS_CNT(c0 = clock64();)
                mbar_wait(full + s, sph);
                TS_CNT(c_full += clock64() - c0;)
                tc_fence_after();
                const uint32_t a_raw = tmem_base + TS_SLOT0 + s * 64, a_lo = a_raw + 32;
                const uint64_t dw = make_kmajor_sw128_desc(wres0 + (uint32_t)kb * WPLANE);
                const bool gate = P.self_mode == 1 && kb == P.nkb_main;
                const uint32_t d = gate ? d_main + 64 : d_main;
                if (ts_elect_one()) {
                    if (P.prec == 0) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint64_t adv = (uint64_t)((k * 32) >> 4);     // 8 TF32 = 32 bytes along K inside the swizzled row
                            umma_tf32_ts(d, a_raw + 8 * k, dw + adv, ID_FULL, ((gate || kb == 0) && k == 0) ? 0u : 1u);
                            umma_tf32_ts(d + BNH, a_lo + 8 * k, dw + adv, ID_HALF, 1u);
                        }
                    } else if (P.prec == 1) {                                   // single-pass TF32: hi weights only (first BNH plane rows)
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            umma_tf32_ts(d, a_raw + 8 * k, dw + (uint64_t)((k * 32) >> 4), ID_HALF, ((gate || kb == 0) && k == 0) ? 0u : 1u);
                    } else {                                                    // BF16: 16 k-elements (8 packed columns, 32 bytes) per MMA
#pragma unroll
                        for (int k = 0; k < 2; ++k)
                            umma_bf16_ts(d, a_raw + 8 * k, dw + (uint64_t)((k * 32) >> 4), make_idesc_bf16(128, BNH),
                                         ((gate || kb == 0) && k == 0) ? 0u : 1u);
                    }
                    umma_commit(empty + s);
                    if (kb == nkb_total - 1) umma_commit(tfull);
                }
                __syncwarp();
                if (++s == TS_NSLOT) {
                    s = 0;
                    sph ^= 1;
                }
            }
        }
        TS_CNT(if (P.dbg && lane == 0) {
            atomicAdd(P.dbg + 3, (unsigned long long)c_full);
            atomicAdd(P.dbg + 4, (unsigned long long)c_tempty);
            atomicAdd(P.dbg + 5, (unsigned long long)(clock64() - c_begin));
        })
    } else if (warp >= TS_EPI0 && warp < TS_EPI0 + 4) {
        const int ew = warp - TS_EPI0;                                  // TMEM lane quarter (= warp % 4)
        // =================================================================== epilogue: thread = tile row = TMEM lane
        const int Fo = P.Nc, G = P.G;
        const bool has_gates = BNH == 32 && P.self_mode == 1;
        const bool vec_out = (P.ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(P.out) & 15) == 0);
        uint32_t tt = 0;
        TS_CNT(long long c_tfull = 0; const long long c_begin = clock64();)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tt) {
            TS_CNT(const long long cw = clock64();)
            mbar_wait(tfull, tt & 1);
            TS_CNT(c_tfull += clock64() - cw;)
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16);
            const int64_t r = (int64_t)tile * TS_ROWS + ew * 32 + lane;
            const bool live = r < P.N;
            float* orow = P.out + (live ? r : 0) * P.ldo;
#pragma unroll
            for (int c0 = 0; c0 < BNH; c0 += 32) {
                float vh[32], vl[32];
                ts_tmem_ld32_nw(taddr + c0, vh);
                if (P.prec == 0) {
                    ts_tmem_ld32_nw(taddr + BNH + c0, vl);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) vl[i] = 0.f;
                }
                ts_ld_wait();
                if (live) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const float4 b4 = *reinterpret_cast<const float4*>(sbias + c0 + i);
                        float4 o = make_float4(vh[i] + vl[i] + b4.x, vh[i + 1] + vl[i + 1] + b4.y, vh[i + 2] + vl[i + 2] + b4.z,
                                               vh[i + 3] + vl[i + 3] + b4.w);
                        if (P.epi == 1) {
                            o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                        }
                        if (vec_out && c0 + i + 3 < Fo) {
                            *reinterpret_cast<float4*>(orow + c0 + i) = o;
                        } else {
                            if (c0 + i + 0 < Fo) orow[c0 + i + 0] = o.x;
                            if (c0 + i + 1 < Fo) orow[c0 + i + 1] = o.y;
                            if (c0 + i + 2 < Fo) orow[c0 + i + 2] = o.z;
                            if (c0 + i + 3 < Fo) orow[c0 + i + 3] = o.w;
                        }
                    }
                }
            }
            if (has_gates) {
                // gate accumulator: p1_j in columns 64 + j (hi weights) / 96 + j (lo weights), p2_j in 80 + j / 112 + j
                float g1h[16], g2h[16], g1l[16], g2l[16];
                ts_tmem_ld16_nw(taddr + 64, g1h);
                ts_tmem_ld16_nw(taddr + 80, g2h);
                if (P.prec == 0) {
                    ts_tmem_ld16_nw(taddr + 96, g1l);
                    ts_tmem_ld16_nw(taddr + 112, g2l);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) g1l[i] = g2l[i] = 0.f;
                }
                ts_ld_wait();
                if (live) {
                    float* ax = P.aux + r * P.ldaux;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        if (j < G) {
                            const float p1 = g1h[j] + g1l[j] + sbias[64 + j], p2 = g2h[j] + g2l[j] + sbias[64 + G + j];
                            const float t1 = tanh_fast(p1), t2 = tanh_fast(p2);
                            orow[Fo + j] = t1 * t2;
                            if constexpr (AUX) {
                                ax[j] = t1;
                                ax[G + j] = t2;
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
        }
        TS_CNT(if (P.dbg && lane == 0) {
            atomicAdd(P.dbg + 6, (unsigned long long)c_tfull);
            atomicAdd(P.dbg + 7, (unsigned long long)(clock64() - c_begin));
        })
    } else if (warp < TS_AGG0 + 8) {
        // =================================================================== aggregators (8 warps x 16 rows, 2 threads per row)
        const int aw = warp - TS_AGG0;
        const int lrow = 32 * (aw & 3) + 16 * (aw >> 2) + 8 * (lane & 1) + (lane >> 2);     // tile row = TMEM lane of this thread
        const int p = (lane >> 1) & 1;                                                      // features 16 p .. 16 p + 15
        const uint32_t lane_addr = (uint32_t)(32 * (aw & 3) + 16 * (aw >> 2)) << 16;
        const int* __restrict__ col = P.col;
        const int* __restrict__ eperm = P.eperm;
        const float* __restrict__ ea = P.ea;
        const float* __restrict__ X = P.X;
        const int64_t ldx = P.ldx;
        const int F = P.F;
        const uint32_t stage32 = smem_u32(stage0);
        uint32_t st_i = 0, st_ph = 1, ts = 0;
        TS_CNT(long long c_gather = 0, c_wait = 0, c_xwait = 0, c_dump = 0, c_loop = 0, n_steps = 0; const long long c_begin = clock64();)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++ts) {
            const int64_t row = (int64_t)tile * TS_ROWS + lrow;
            const uint32_t sb = ts & 1;
            const uint32_t x32 = stage32 + sb * stage_bytes;                 // window rows
            const uint32_t sea32 = x32 + TS_WIN_ROWS * 128;                  // staged edge weights
            const uint32_t scol32 = sea32 + (uint32_t)cap * Kstride * 4;     // staged source rows
            const uint32_t srp32 = scol32 + (uint32_t)cap * 4;
            TS_CNT(const long long cx = clock64();)
            mbar_wait(sfull + sb, (ts >> 1) & 1);
            TS_CNT(c_xwait += clock64() - cx;)
            int e0, win0, staged;
            {
                const uint32_t m32 = srp32 + 132 * 4;
                asm volatile("ld.shared.s32 %0, [%1];" : "=r"(e0) : "r"(m32));
                asm volatile("ld.shared.s32 %0, [%1];" : "=r"(win0) : "r"(m32 + 8));
                asm volatile("ld.shared.s32 %0, [%1];" : "=r"(staged) : "r"(m32 + 12));
            }
            int rs, re;
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(rs) : "r"(srp32 + (uint32_t)lrow * 4));
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(re) : "r"(srp32 + (uint32_t)lrow * 4 + 4));
            TS_CNT(long long cg0 = clock64();)
            for (int k0 = 0; k0 < P.K; k0 += KT) {
                float acc[KT][16];
#pragma unroll
                for (int k = 0; k < KT; ++k)
#pragma unroll
                    for (int i = 0; i < 16; ++i) acc[k][i] = 0.f;
                if (staged) {
                    // every operand from shared memory: slot -> source row -> window row, edge weights slot-major.  Software
                    // pipeline without extra registers: the first half of the NEXT slot's source row is loaded right after the
                    // FMAs that consumed the current first half, the second half after the second batch of FMAs, so every LDS
                    // has 8 * KT FMAs of the same thread (and the other warp of the scheduler) to land behind.
                    const int n = re - rs;
                    const uint32_t ca0 = scol32 + (uint32_t)(rs - e0) * 4;
                    const uint32_t wa0 = sea32 + (uint32_t)((rs - e0) * Kstride + k0) * 4;
                    const uint32_t wstep = (uint32_t)Kstride * 4;
                    const uint32_t c0 = (uint32_t)p << 6;
                    // (schedulable shared-memory loads, branch-free: the slot after the row's last one is clamped to the last one,
                    // so the compiler is free to hoist every load as far ahead of its FMAs as registers allow)
                    auto xrow = [&](int sidx, uint32_t chunk) -> float4 {
                        const int s = sidx - win0;
                        return ts_lds128_nv(x32 + (uint32_t)s * 128u + ((c0 + 16u * chunk) ^ ((uint32_t)(s & 7) << 4)));
                    };
                    float4 xa0, xa1, xb0, xb1;
                    xa0 = xa1 = xb0 = xb1 = make_float4(0.f, 0.f, 0.f, 0.f);
                    float w[KT];
#pragma unroll
                    for (int k = 0; k < KT; ++k) w[k] = 0.f;
                    int sidx_n = 0;
                    if (n > 0) {
                        const int s0 = ts_lds32_nv(ca0);
                        xa0 = xrow(s0, 0); xa1 = xrow(s0, 1); xb0 = xrow(s0, 2); xb1 = xrow(s0, 3);
                        ts_lds_w_nv<KT>(wa0, w);
                        sidx_n = ts_lds32_nv(ca0 + (n > 1 ? 4u : 0u));
                    }
                    TS_CNT(__syncwarp(); const long long cl0 = clock64(); n_steps += __reduce_max_sync(0xffffffffu, n);)
                    for (int i = 0; i < n; ++i) {
                        const uint32_t inext = i + 1 < n ? i + 1 : i, inn = i + 2 < n ? i + 2 : n - 1;
                        const int sn = sidx_n;
                        float wn[KT];
                        ts_lds_w_nv<KT>(wa0 + inext * wstep, wn);
                        sidx_n = ts_lds32_nv(ca0 + inn * 4u);
                        ts_fma_half<KT, 0>(acc, w, xa0, xa1);
                        xa0 = xrow(sn, 0);
                        xa1 = xrow(sn, 1);
                        ts_fma_half<KT, 1>(acc, w, xb0, xb1);
                        xb0 = xrow(sn, 2);
                        xb1 = xrow(sn, 3);
#pragma unroll
                        for (int k = 0; k < KT; ++k) w[k] = wn[k];
                    }
                    TS_CNT(__syncwarp(); c_loop += clock64() - cl0;)
                } else {
                    // general graphs: slots, edge weights and source rows from global memory (indices two slots ahead, edge
                    // weights one slot ahead)
                    int sidx_n = 0, sidx_nn = 0, eidx_nn = 0;
                    float w_n[KT];
#pragma unroll
                    for (int k = 0; k < KT; ++k) w_n[k] = 0.f;
                    if (rs < re) {
                        sidx_n = __ldg(col + rs);
                        const int ee = eperm ? __ldg(eperm + rs) : rs;
                        ts_load_w<KT>(ea + (int64_t)ee * Kstride + k0, w_n);
                        if (rs + 1 < re) {
                            sidx_nn = __ldg(col + rs + 1);
                            eidx_nn = eperm ? __ldg(eperm + rs + 1) : rs + 1;
                        }
                    }
                    for (int p0 = rs; p0 < re; ++p0) {
                        const int sidx = sidx_n;
                        float w[KT];
#pragma unroll
                        for (int k = 0; k < KT; ++k) w[k] = w_n[k];
                        sidx_n = sidx_nn;
                        if (p0 + 1 < re) ts_load_w<KT>(ea + (int64_t)eidx_nn * Kstride + k0, w_n);
                        if (p0 + 2 < re) {
                            sidx_nn = __ldg(col + p0 + 2);
                            eidx_nn = eperm ? __ldg(eperm + p0 + 2) : p0 + 2;
                        }
                        const float* xr = X + (int64_t)sidx * ldx + 16 * p;
                        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                        const float4 x0 = 16 * p + 0 < F ? ldg4(xr + 0) : z;
                        const float4 x1 = 16 * p + 4 < F ? ldg4(xr + 4) : z;
                        const float4 x2 = 16 * p + 8 < F ? ldg4(xr + 8) : z;
                        const float4 x3 = 16 * p + 12 < F ? ldg4(xr + 12) : z;
                        ts_fma<KT>(acc, w, x0, x1, x2, x3);
                    }
                }
                if (P.hout && row < P.N) {           // side output for the weight-gradient contraction of the backward
                    float* hr = P.hout + row * P.ldh + (int64_t)k0 * 32 + 16 * p;
#pragma unroll
                    for (int k = 0; k < KT; ++k)
#pragma unroll
                        for (int i = 0; i < 16; i += 4) st_na4(hr + k * 32 + i, make_float4(acc[k][i], acc[k][i + 1], acc[k][i + 2], acc[k][i + 3]));
                }
                __syncwarp();
                TS_CNT(c_gather += clock64() - cg0;)
                const bool last_pass = k0 + KT >= P.K;
                if (last_pass && lane == 0) mbar_arrive(sempty + sb);      // staging buffer no longer read by this warp
                // the self block's row (consumed after this pass's hand-off): its latency hides behind the tensor-memory stores
                float sv[16];
                if (last_pass && P.self_mode != 0) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) sv[i] = 0.f;
                    if (row < P.N) {
                        const float* sr = P.S + row * P.lds + 16 * p;
#pragma unroll
                        for (int i = 0; i < 16; i += 4) {
                            if (16 * p + i < P.Fs) {
                                const float4 t = ldg4(sr + i);
                                sv[i] = t.x; sv[i + 1] = t.y; sv[i + 2] = t.z; sv[i + 3] = t.w;
                            }
                        }
                    }
                }
                // hand the KT finished k-blocks to the tensor core: all stores first, one wait, then the arrivals
                TS_CNT(const long long cd0 = clock64();)
                {
                    uint32_t si = st_i, sp = st_ph;
#pragma unroll
                    for (int k = 0; k < KT; ++k) {          // the MMAs that read these slots last have retired
                        TS_CNT(const long long cw = clock64();)
                        mbar_wait(empty + si, sp);
                        TS_CNT(c_wait += clock64() - cw;)
                        if (++si == TS_NSLOT) {
                            si = 0;
                            sp ^= 1;
                        }
                    }
                    tc_fence_after();
                    si = st_i;
#pragma unroll
                    for (int k = 0; k < KT; ++k) {
                        const uint32_t ta = tmem_base + lane_addr + TS_SLOT0 + si * 64;
                        if (P.prec == 2) {
                            uint32_t pk[8];
                            ts_pack_bf16(acc[k], pk);
                            ts_st_16x64b_x8(ta, pk);
                        } else {
                            ts_st_16x64b_x16(ta, acc[k]);
                            if (P.prec == 0) {
                                float lo[16];
#pragma unroll
                                for (int i = 0; i < 16; ++i) lo[i] = ts_lo(acc[k][i]);
                                ts_st_16x64b_x16(ta + 32, lo);
                            }
                        }
                        if (++si == TS_NSLOT) si = 0;
                    }
                    ts_st_wait();
                    tc_fence_before();
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < KT; ++k) {
                        if (lane == 0) mbar_arrive(full + st_i);
                        if (++st_i == TS_NSLOT) {
                            st_i = 0;
                            st_ph ^= 1;
                        }
                    }
                }
                if (last_pass && P.self_mode != 0) {
                    if (P.hout && row < P.N) {
                        float* hr = P.hout + row * P.ldh + (int64_t)P.K * 32 + 16 * p;
#pragma unroll
                        for (int i = 0; i < 16; i += 4) st_na4(hr + i, make_float4(sv[i], sv[i + 1], sv[i + 2], sv[i + 3]));
                    }
                    TS_CNT(const long long cw = clock64();)
                    mbar_wait(empty + st_i, st_ph);
                    TS_CNT(c_wait += clock64() - cw;)
                    tc_fence_after();
                    const uint32_t ta = tmem_base + lane_addr + TS_SLOT0 + st_i * 64;
                    if (P.prec == 2) {
                        uint32_t pk[8];
                        ts_pack_bf16(sv, pk);
                        ts_st_16x64b_x8(ta, pk);
                    } else {
                        ts_st_16x64b_x16(ta, sv);
                        if (P.prec == 0) {
                            float lo[16];
#pragma unroll
                            for (int i = 0; i < 16; ++i) lo[i] = ts_lo(sv[i]);
                            ts_st_16x64b_x16(ta + 32, lo);
                        }
                    }
                    ts_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full + st_i);
                    if (++st_i == TS_NSLOT) {
                        st_i = 0;
                        st_ph ^= 1;
                    }
                }
                TS_CNT(c_dump += clock64() - cd0; cg0 = clock64();)
            }
        }
        TS_CNT(if (P.dbg && lane == 0) {
            atomicAdd(P.dbg + 0, (unsigned long long)c_gather);
            atomicAdd(P.dbg + 1, (unsigned long long)c_wait);
            atomicAdd(P.dbg + 2, (unsigned long long)(clock64() - c_begin));
            atomicAdd(P.dbg + 8, (unsigned long long)c_xwait);
            atomicAdd(P.dbg + 9, (unsigned long long)c_dump);
            atomicAdd(P.dbg + 10, (unsigned long long)c_loop);
            atomicAdd(P.dbg + 13, (unsigned long long)n_steps);
        })
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TS_MMAW) tmem_dealloc(tmem_base, 512);
}

// Weight planes of the TS kernel: one [2 BNH rows x 32 k-columns] K-major plane per k-block (kb = k for the K supports,
// kb = K for the self block).  Plane row n < BNH: hi = RN-TF32(w) of output column n; row BNH + n: lo = w - hi.  Plane
// column c holds feature f(c) = 16 * (c & 1) + (c >> 1) of the block (the tensor-memory column order of the aggregators).
// Self plane: mode 2 -> Bself [Fs, Nc]; mode 1 -> the gate weights Bself [Fs, Ns = 2G] = [W11^T | W12^T]: p1_j in plane row j,
// p2_j in plane row 16 + j (so the epilogue pairs accumulator columns j and 16 + j whatever G is).
// prec 2 (BF16): plane row n = 64 BF16 slots (the same 128 bytes), slot kappa < 32 holds feature 16 * ((kappa >> 1) & 1) +
// 2 * (kappa >> 2) + (kappa & 1) -- the order in which the aggregators pack their accumulators into tensor memory; rows
// >= BNH unused.
__global__ void k_ts_prep_weights(const float* __restrict__ Bmain, int64_t ldb, int K, int F, int Nc, int BNH,
                                  const float* __restrict__ Bself, int64_t ldbs, int Fs, int Ns, int self_mode, int prec,
                                  float* __restrict__ planes) {
    const int nkb_total = K + (self_mode != 0 ? 1 : 0);
    const int MR = 2 * BNH;
    const int total = nkb_total * MR * 32;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int kb = i / (MR * 32), m = (i / 32) % MR, c = i % 32;
        const int n = m % BNH;
        const bool is_lo = m >= BNH;
        const int f = prec == 2 ? 16 * ((c >> 1) & 1) + 2 * (c >> 2) + (c & 1) : 16 * (c & 1) + (c >> 1);
        float v = 0.f;
        if (kb < K) {
            if (f < F && n < Nc) v = __ldg(Bmain + ((int64_t)kb * F + f) * ldb + n);
        } else if (self_mode == 2) {
            if (f < Fs && n < Nc) v = __ldg(Bself + (int64_t)f * ldbs + n);
        } else {
            const int j = n & 15, which = n >> 4, G = Ns >> 1;      // plane row j: p1_j, row 16 + j: p2_j
            if (f < Fs && j < G) v = __ldg(Bself + (int64_t)f * ldbs + which * G + j);
        }
        if (prec == 2) {
            __nv_bfloat16* row = reinterpret_cast<__nv_bfloat16*>(planes + (size_t)(kb * MR + m) * 32);
            row[c] = __float2bfloat16_rn(is_lo ? 0.f : v);
            row[32 + c] = __float2bfloat16_rn(0.f);
        } else {
            const float h = tf32_rn(v);
            planes[i] = is_lo ? v - h : h;
        }
    }
}

// Source window of every tile of `rows_per_tile` CSR rows: win[t] = {min col, max col + 1} over the tile's slots
// ({0, 0} for a tile without slots).  Integer work, exact.
__global__ void k_tile_windows(const int* __restrict__ rowptr, const int* __restrict__ col, int64_t N, int rows_per_tile, int n_tiles,
                               int2* __restrict__ win) {
    const int tile = blockIdx.x;
    if (tile >= n_tiles) return;
    const int64_t r0 = (int64_t)tile * rows_per_tile;
    const int64_t r1 = r0 + rows_per_tile < N ? r0 + rows_per_tile : N;
    const int e0 = __ldg(rowptr + r0), e1 = __ldg(rowptr + r1);
    int lo = 0x7fffffff, hi = -1;
    for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
        const int c = __ldg(col + e);
        lo = c < lo ? c : lo;
        hi = c > hi ? c : hi;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const int l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = l2 < lo ? l2 : lo;
        hi = h2 > hi ? h2 : hi;
    }
    __shared__ int slo[8], shi[8];
    if ((threadIdx.x & 31) == 0) {
        slo[threadIdx.x >> 5] = lo;
        shi[threadIdx.x >> 5] = hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            lo = slo[w] < lo ? slo[w] : lo;
            hi = shi[w] > hi ? shi[w] : hi;
        }
        win[tile] = hi >= 0 ? make_int2(lo, hi + 1) : make_int2(0, 0);
    }
}

}  // namespace gnnml3

using namespace gnnml3;

extern "C" int gnnml3_tile_rows(void) { return TS_ROWS; }

extern "C" int gnnml3_tile_windows(const int32_t* rowptr, const int32_t* col, int64_t N, int32_t* win, void* stream) {
    GNNML3_REQUIRE(N > 0 && rowptr && win, "tile_windows: bad arguments");
    const int n_tiles = cdiv(N, TS_ROWS);
    k_tile_windows<<<n_tiles, 128, 0, (cudaStream_t)stream>>>(rowptr, col, N, TS_ROWS, n_tiles, reinterpret_cast<int2*>(win));
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

static const bool g_ts_enabled = [] {
    const char* e = getenv("GNNML3_FUSED_TS");
    return !(e && e[0] == '0');
}();
static int g_ts_runtime_enabled = 1;

// which kernel gnnml3_fused_agg_proj dispatched to since the last reset: [0] tensor-memory kernel, [1] round-1 shared-memory
// plane kernel; the Python side adds the counts of the two-kernel fallback (bench.py prints them as `path_taken`)
static std::atomic<long long> g_fused_paths[2];
extern "C" int gnnml3_fused_path_counts(long long* out2_host, int reset) {
    out2_host[0] = reset ? g_fused_paths[0].exchange(0) : g_fused_paths[0].load();
    out2_host[1] = reset ? g_fused_paths[1].exchange(0) : g_fused_paths[1].load();
    return GNNML3_OK;
}
namespace gnnml3 {
void fused_path_count(int which) { ++g_fused_paths[which]; }
}

// 1 = use the tensor-memory kernel where the shape allows (default), 0 = always the round-1 kernel; returns the old value
extern "C" int gnnml3_fused_set_ts(int enable) {
    const int old = g_ts_runtime_enabled;
    if (enable == 0 || enable == 1) g_ts_runtime_enabled = enable;
    return old;
}

static inline int ts_kt_for(int K, int Kstride) {
    if (K % 4 == 0 && Kstride % 4 == 0) return 4;
    if (K % 2 == 0 && Kstride % 2 == 0) return 2;
    return 0;
}

constexpr size_t TS_SMEM_MAX = 227 * 1024;

static inline size_t ts_stage_aligned(int cap, int Kstride) { return (ts_stage_bytes(cap, Kstride) + 1023) & ~(size_t)1023; }
static inline size_t ts_smem_bytes(int K, int Kstride, int Nc, int self_mode, int cap) {
    const size_t wplane = 2 * (size_t)(Nc <= 32 ? 32 : 64) * 128;
    return 1024 + 2 * ts_stage_aligned(cap, Kstride) + (size_t)(K + (self_mode != 0 ? 1 : 0)) * wplane + 768;
}
// largest slot capacity (multiple of 32, at most 2048) whose two staging buffers fit beside the weight planes; 0 if not even
// 256 slots fit or the edge weights cannot be staged with 128-bit copies
static inline int ts_edge_cap(int K, int Kstride, int Nc, int self_mode) {
    if (Kstride % 4 != 0) return 0;
    for (int cap = 2048; cap >= 256; cap -= 32)
        if (ts_smem_bytes(K, Kstride, Nc, self_mode, cap) <= TS_SMEM_MAX) return cap;
    return 0;
}

extern "C" int gnnml3_fused_ts_supported(int K, int Kstride, int F, int Nc, int Fs, int self_mode, int Ns) {
    if (!g_ts_enabled || !g_ts_runtime_enabled) return 0;
    if (ts_kt_for(K, Kstride) == 0 || K < 1 || K > 24) return 0;     // accumulation chain per tile kept short (TMEM adds truncate)
    if (F < 1 || F > 32 || Nc < 1 || Nc > 64) return 0;
    if (self_mode != 0 && (Fs < 1 || Fs > 32)) return 0;
    if (self_mode == 1 && (Ns < 2 || Ns > 32 || Ns % 2 != 0 || Nc > 32)) return 0;
    if (ts_smem_bytes(K, Kstride, Nc, self_mode, 0) > TS_SMEM_MAX) return 0;
    return 1;
}

extern "C" size_t gnnml3_fused_ts_workspace_bytes(int K, int Nc, int self_mode) {
    return align_up((size_t)(K + (self_mode != 0 ? 1 : 0)) * 2 * (Nc <= 32 ? 32 : 64) * 128, 256);
}

namespace gnnml3 {

struct TSProfHook {
    void (*begin)(cudaStream_t, const double*);
    void (*end)(cudaStream_t);
};
TSProfHook g_ts_prof = {nullptr, nullptr};

template <int KT, int BNH, bool AUX = true>
static int ts_launch(const CUtensorMap& mW, const CUtensorMap& mX, TSParams& P, size_t smem, cudaStream_t st) {
    static bool configured[64] = {};
    if (auto once_ = first_use_on_device(configured))
        GNNML3_CUDA(cudaFuncSetAttribute(k_fused_ts<KT, BNH, AUX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TS_SMEM_MAX));
    const int grid = P.n_tiles < kNumSMs ? P.n_tiles : kNumSMs;
    k_fused_ts<KT, BNH, AUX><<<grid, TS_THREADS, smem, st>>>(mW, mX, P);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

// X [N, F] (row stride ldx) -> 2-D tensor map with a [box_rows x 32 columns] box, 128B swizzle; columns >= F and rows >= N
// are zero-filled by the TMA unit
int ts_make_xmap(CUtensorMap* map, const float* base, int64_t rows, int F, int64_t ld, int box_rows) {
    PFN_encodeTiled enc = get_encoder();
    if (!enc) return set_err(GNNML3_ERR_CUDA, "fused_agg_proj: cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t gdim[2] = {(cuuint64_t)F, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_err(GNNML3_ERR_CUDA, "fused_agg_proj: cuTensorMapEncodeTiled(X) failed (%d)", (int)r);
    return GNNML3_OK;
}

// called by gnnml3_fused_agg_proj (fused_layer.cu) after argument validation, when gnnml3_fused_ts_supported() holds
int fused_ts_run(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea, int Kstride, int K, const float* X,
                 int64_t ldx, int F, const float* S, int64_t lds, int Fs, int self_mode, const float* Bmain, int64_t ldb,
                 const float* Bself, int64_t ldbs, int Ns, const float* bias, const float* bias_s, int64_t N, int Nc, float* out,
                 int64_t ldo, float* aux, int64_t ldaux, int G, int epilogue, int precision, float* hout, int64_t ldh,
                 const int32_t* tilewin, void* workspace, size_t workspace_bytes, unsigned long long* dbg, cudaStream_t st) {
    if (workspace_bytes < gnnml3_fused_ts_workspace_bytes(K, Nc, self_mode))
        return set_err(GNNML3_ERR_WORKSPACE, "fused_agg_proj: workspace too small");
    const int BNH = Nc <= 32 ? 32 : 64;
    const int KT = ts_kt_for(K, Kstride);
    const int nkb_total = K + (self_mode != 0 ? 1 : 0);
    float* planes = (float*)workspace;
    {
        const int total = nkb_total * 2 * BNH * 32;
        const int blocks = cdiv(total, 256) > 592 ? 592 : cdiv(total, 256);
        k_ts_prep_weights<<<blocks, 256, 0, st>>>(Bmain, ldb, K, F, Nc, BNH, Bself, ldbs, Fs, Ns, self_mode, precision, planes);
        GNNML3_LAUNCH_CHECK();
    }
    CUtensorMap mW, mX;
    int rc;
    if ((rc = make_map(&mW, planes, (int64_t)nkb_total * 2 * BNH, 32, 32, 2 * BNH))) return rc;
    const int win_rows = N < TS_WIN_ROWS ? (int)N : TS_WIN_ROWS;
    if ((rc = ts_make_xmap(&mX, X, N, F, ldx, win_rows))) return rc;
    TSParams P;
    P.rowptr = rowptr; P.col = col; P.eperm = eperm; P.ea = ea; P.Kstride = Kstride; P.K = K;
    P.X = X; P.ldx = ldx; P.F = F; P.S = S; P.lds = lds; P.Fs = Fs; P.self_mode = self_mode;
    P.N = N; P.n_tiles = cdiv(N, TS_ROWS); P.nkb_main = K; P.tilewin = reinterpret_cast<const int2*>(tilewin); P.win_rows = win_rows;
    P.bias = bias; P.bias_s = bias_s; P.out = out; P.ldo = ldo; P.Nc = Nc; P.aux = aux; P.ldaux = ldaux; P.G = G; P.epi = epilogue; P.prec = precision;
    P.hout = hout; P.ldh = ldh; P.dbg = dbg;
    P.edge_cap = tilewin ? ts_edge_cap(K, Kstride, Nc, self_mode) : 0;
    const size_t smem = ts_smem_bytes(K, Kstride, Nc, self_mode, P.edge_cap);
    if (BNH == 32 && self_mode == 1 && !aux)      // gated epilogue without aux: the forward-only instantiation
        return KT == 4 ? ts_launch<4, 32, false>(mW, mX, P, smem, st) : ts_launch<2, 32, false>(mW, mX, P, smem, st);
    if (BNH == 32) return KT == 4 ? ts_launch<4, 32>(mW, mX, P, smem, st) : ts_launch<2, 32>(mW, mX, P, smem, st);
    return KT == 4 ? ts_launch<4, 64>(mW, mX, P, smem, st) : ts_launch<2, 64>(mW, mX, P, smem, st);
}

}  // namespace gnnml3
