// Fused aggregate + project kernel of the GNNML3 layer on Blackwell tensor cores.
//
// Reference semantics (libs/spect_conv.py:70-80,93-94 and :208-212):
//     conv[t, :] = sum_k ( sum_{e: dst_e = t} ea[e, k] * x[src_e, :] ) W_k  + bias            (SpectConv)
//     y[t, :]    = [ relu(conv[t, :]) || tanh(x[t] W11^T + b11) * tanh(x[t] W12^T + b12) ]    (ML3Layer)
// The reference materialises K message tensors [E, Fi], K scatter results [N, Fi] and K matmul results; the
// two-kernel design of spmm.cu + gemm*.cu still round-trips H = [P_0(x) .. P_{K-1}(x)]  ([N, K*Fi]) through HBM.
// Here H never leaves the SM: a persistent CTA owns a tile of ROWS dst rows,
//   * aggregator warps walk the tile's CSR rows (4 lanes per row, 8 features per lane, KT supports in registers,
//     128-bit gathers of the source rows, summation in edge order, no atomics) and write each 32-column block
//     of H straight into shared memory in the UMMA K-major SWIZZLE_128B layout, as the raw FP32 plane (= the hi
//     part: the tensor core truncates to TF32 itself) and, right behind it, the residual plane lo = a - trunc(a);
//   * one thread issues tcgen05.mma kind::tf32.  A tcgen05.mma costs ~143 cycles on B200 whatever its shape
//     (measured, scratch/umma_bench.cu), so the operands are arranged to make every instruction as large as
//     possible: the weights are the M side -- rows [W_hi^T ; W_lo^T ; gate weights hi ; lo] of one 128-row plane per
//     k-block, streamed from L2 by a TMA warp -- and the tile's rows are the N side, hi and lo planes side by side
//     (N = 2 * ROWS).  ONE instruction per 8-wide k-step therefore produces all four products
//     {W_hi, W_lo} x {H_hi, H_lo} of the error-compensated 3xTF32 split (FP32-grade) for the whole tile;
//   * epilogue warps drain the transposed accumulator D[feature, row] from tensor memory, add the hi/lo partial
//     sums (pairs of warps exchange through shared memory), add the bias, apply ReLU / tanh*tanh gating and write
//     y (and the two tanh factors the backward needs) with fully coalesced 128-byte row stores.
// The same kernel computes dx in the backward: rows = source nodes over the transposed CSR, gathered matrix =
// d pre (conv columns), weights = W_k^T, and the gate gradients enter as one more k-block ("self" block) that
// accumulates into the same output columns.  SpectConv(selfconn=True) uses that mode in the forward, too.
#include "tc_common.cuh"

#include <vector>

// cycle counters of the warp roles (gnnml3_fused_debug_counters): compiled in only with -DFL_PROFILE, they cost issue
// slots and registers in the single-thread control loops that pace the whole kernel
#ifndef FL_UD
#define FL_UD 2          // edges in flight per lane in the global-gather aggregator
#endif
#ifdef FL_PROFILE
#define FL_CNT(...) __VA_ARGS__
#else
#define FL_CNT(...)
#endif

namespace gnnml3 {

constexpr int FL_MAX_STAGES = 4;
constexpr int FL_CTRL_WARPS = 6;      // warps 0-3: epilogue | warp 4: TMA (weights) | warp 5: MMA issuer | then aggregators
constexpr int FL_XCH = 32 * 68 + 8;    // half the floats of the epilogue's transpose tile T (>= 32 x 132 in total)

struct FLParams {
    const int* rowptr;      // [N+1] CSR over the rows of this launch
    const int* col;         // [E]   gathered row of X per CSR slot
    const int* eperm;       // [E]   row of `ea` per CSR slot (NULL: identity)
    const float* ea;        // [E, Kstride]
    int Kstride, K;
    const float* X;         // gathered matrix [*, F], row stride ldx (16-byte aligned rows)
    int64_t ldx;
    int F;
    const float* S;         // self block [N, Fs] (row t of the tile itself), NULL if self_mode == 0
    int64_t lds;
    int Fs;
    int self_mode;          // 0 none | 1 own output columns (the ML3 gates, M rows 64..127) | 2 accumulates into the main columns
    int64_t N;
    int n_tiles;
    int nfh;                // 32-wide feature blocks per support = ceil(F / 32)
    int nkb_main;           // nfh * K
    int pf_rows;            // rows of X prefetched into L1 on either side of a tile (0: off)
    int slot_cap;           // edges per aggregator-warp prefetch slot (0: the aggregators gather straight from global memory)
    int nstages;            // depth of the H-plane ring (2..4, whatever shared memory is left beside resident weights)
    const float* bias;      // [Nc] or NULL
    const float* bias_s;    // [2G] or NULL (mode 1)
    float* out;             // plain: [N, Nc]; ml3: y [N, Fo + G]
    int64_t ldo;
    int Nc;                 // main output columns (= Fo)
    float* aux;             // ml3 with G > 0: [N, 2G] tanh factors (t1 | t2)
    int64_t ldaux;
    int G;
    int epi;                // 0 plain (+bias) | 1 ml3: relu on the main columns, gating on the self columns
    float* hout;            // optional copy of the aggregate: [N, ldh], support k at column k * 32 * nfh (zero padded), self block behind
    int64_t ldh;
    unsigned long long* dbg; // optional cycle counters (GNNML3_FUSED_DEBUG=1): see gnnml3_fused_debug_counters
};

template <int KT>
__device__ __forceinline__ void fl_load_ea(const float* __restrict__ p, float (&w)[KT]) {
    if constexpr (KT % 4 == 0) {
#pragma unroll
        for (int k = 0; k < KT; k += 4) {
            const float4 v = ldg4(p + k);
            w[k] = v.x; w[k + 1] = v.y; w[k + 2] = v.z; w[k + 3] = v.w;
        }
    } else if constexpr (KT % 2 == 0) {
#pragma unroll
        for (int k = 0; k < KT; k += 2) {
            const float2 v = ldg2(p + k);
            w[k] = v.x; w[k + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int k = 0; k < KT; ++k) w[k] = __ldg(p + k);
    }
}

// mbarrier wait with back-off for the control warps (TMA / MMA / epilogue): they spend most of their time waiting and the
// kernel is instruction-issue bound, so their polling must not take issue slots from the aggregators
__device__ __forceinline__ void mbar_wait_idle(uint64_t* bar, uint32_t parity) {
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

__device__ __forceinline__ float fl_lo(float v) { return v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }

// raw plane + residual plane (LO_OFF bytes behind it) of one 16-byte chunk
template <int LO_OFF>
__device__ __forceinline__ void fl_store_chunk(uint8_t* a_raw, uint32_t off, const float* v) {
    *reinterpret_cast<float4*>(a_raw + off) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(a_raw + LO_OFF + off) = make_float4(fl_lo(v[0]), fl_lo(v[1]), fl_lo(v[2]), fl_lo(v[3]));
}

// BNH = output columns per hi/lo half of the weight plane's M side: 32 (Nc <= 32: M = 64, rows [W_hi^T ; W_lo^T]; the ML3
// gate weights form a second M = 64 operand whose accumulator interleaves with the main one in tensor memory at a lane
// offset of 16) or 64 (Nc <= 64: M = 128, no gates).  RES: all weight planes stay resident in shared memory (loaded once);
// otherwise the plane of every k-block is streamed from L2 into the stage.
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_16s(uint32_t smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// AUX = false: the forward-only instantiation of the gated epilogue (aux == NULL), which stores y and not the tanh factors.
template <int KT, int BNH, int NAGG, bool RES, bool AUX = true>
__global__ void __launch_bounds__(32 * (FL_CTRL_WARPS + NAGG), 1)
k_fused_agg_proj(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ FLParams P) {
    constexpr int ROWS = 8 * NAGG;                      // dst rows per tile
    constexpr int NMMA = 2 * ROWS;                      // MMA N: hi plane rows then lo plane rows
    constexpr int MROWS = 2 * BNH;                      // MMA M: weight-plane rows
    constexpr int WPLANE = MROWS * 128;                 // bytes of one weight plane
    constexpr int HP_BYTES = 2 * ROWS * 128;            // both H planes of a k-block
    constexpr int STAGE_BYTES = HP_BYTES + (RES ? 0 : WPLANE);
    static_assert(NMMA <= 256 && NMMA % 16 == 0, "bad tile size");
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // offset arithmetic keeps the shared address space (LDS/STS, not generic LD/ST)
    const int nkb_total = P.nkb_main + (P.self_mode != 0 ? 1 : 0);
    const int nstages = P.nstages;
    uint8_t* wres = smem;                                                               // [nkb_total][WPLANE] if RES
    uint8_t* stages = smem + (RES ? (size_t)nkb_total * WPLANE : 0);
    float* xch = reinterpret_cast<float*>(stages + (size_t)nstages * STAGE_BYTES);      // [2 pairs][2][32][33]
    uint64_t* bars = reinterpret_cast<uint64_t*>(xch + 2 * FL_XCH);
    uint64_t* full = bars;                             // [STAGES]  H planes written (+ weight bytes landed) -> MMA
    uint64_t* empty = bars + FL_MAX_STAGES;            // [STAGES]  MMAs retired                             -> writers
    uint64_t* tfull = bars + 2 * FL_MAX_STAGES;        // [2]       tile accumulator complete                -> epilogue
    uint64_t* tempty = bars + 2 * FL_MAX_STAGES + 2;   // [2]       accumulator drained                      -> MMA
    uint64_t* wfull = bars + 2 * FL_MAX_STAGES + 4;    // [1]       resident weights landed                  -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * FL_MAX_STAGES + 5);
    int* agg_seq = reinterpret_cast<int*>(tmem_slot + 1);
    uint8_t* slots = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(bars) + 256 + 127) & ~(uintptr_t)127);   // 128-byte aligned    // [NAGG][slot_cap x (128 B source row | Kstride floats)] if slot_cap > 0      // tiles started by the aggregators (paces the prefetch warp)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < FL_MAX_STAGES; ++s) {
            mbar_init(full + s, NAGG + (RES ? 0 : 1));
            mbar_init(empty + s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(tfull + b, 1);
            mbar_init(tempty + b, 4);
        }
        mbar_init(wfull, 1);
        *agg_seq = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&mapW) : "memory");
    }
    if (warp == 5) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4) {
        // =================================================================== TMA: weight planes (+ L2 prefetch of the edge data)
        if (lane == 0) {
            if constexpr (RES) {
                mbar_arrive_expect_tx(wfull, (uint32_t)nkb_total * WPLANE);
                for (int kb = 0; kb < nkb_total; ++kb)
                    tma_load_2d(wres + (size_t)kb * WPLANE, &mapW, wfull, 0, kb * MROWS);
            } else {
                uint32_t it = 0;
                for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
                    for (int kb = 0; kb < nkb_total; ++kb, ++it) {
                        const uint32_t s = it % nstages;
                        mbar_wait_idle(empty + s, ((it / nstages) & 1) ^ 1);
                        mbar_arrive_expect_tx(full + s, WPLANE);
                        tma_load_2d(stages + (size_t)s * STAGE_BYTES + HP_BYTES, &mapW, full + s, 0, kb * MROWS);
                    }
                }
            }
        }
        if constexpr (RES) {
            // The warp is idle from here on: it stays one tile ahead of the aggregators and pulls the next tile's CSR slots,
            // edge weights (contiguous per tile when eperm == NULL) and the block of X rows around the tile (the sources of a
            // batched disjoint graph lie within a graph's size of their targets) into L1, so that the aggregators' dependent
            // gathers hit L1 instead of paying an L2 / HBM round trip per edge pair.  Purely a hint: wrong guesses cost nothing.
            __syncwarp();
            int j = 0;
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++j) {
                while (*reinterpret_cast<volatile int*>(agg_seq) < j - 1) __nanosleep(64);
                const int64_t r0 = (int64_t)tile * ROWS;
                const int64_t r1 = r0 + ROWS < P.N ? r0 + ROWS : P.N;
                const int e0 = __ldg(P.rowptr + r0), e1 = __ldg(P.rowptr + r1);
                const char* pc = reinterpret_cast<const char*>(P.col + e0);
                const int64_t nbc = (int64_t)(e1 - e0) * 4;
                for (int64_t o = (int64_t)lane * 128; o < nbc; o += 32 * 128)
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(pc + o));
                if (P.eperm) {
                    const char* pp = reinterpret_cast<const char*>(P.eperm + e0);
                    for (int64_t o = (int64_t)lane * 128; o < nbc; o += 32 * 128)
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(pp + o));
                } else {
                    const char* pe = reinterpret_cast<const char*>(P.ea + (int64_t)e0 * P.Kstride);
                    const int64_t nbe = (int64_t)(e1 - e0) * P.Kstride * 4;
                    for (int64_t o = (int64_t)lane * 128; o < nbe; o += 32 * 128)
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(pe + o));
                }
                if (P.pf_rows > 0) {
                    const int64_t x0 = r0 - P.pf_rows > 0 ? r0 - P.pf_rows : 0;
                    const int64_t x1 = r1 + P.pf_rows < P.N ? r1 + P.pf_rows : P.N;
                    const char* px = reinterpret_cast<const char*>(P.X + x0 * P.ldx);
                    const int64_t nbx = (x1 - x0) * P.ldx * 4;
                    for (int64_t o = (int64_t)lane * 128; o < nbx; o += 32 * 128)
                        asm volatile("prefetch.global.L1 [%0];" ::"l"(px + o));
                }
            }
        }
    } else if (warp == 5) {
        // =================================================================== MMA issuer (one lane)
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_tf32_mn(MROWS, NMMA);
            if constexpr (RES) mbar_wait_idle(wfull, 0);
            uint32_t tt = 0, s = 0, sph = 0;                       // stage index / phase kept incrementally (no divisions)
            const uint32_t stage0 = smem_u32(stages), wres0 = smem_u32(wres);
            FL_CNT(long long c_full = 0, c_tempty = 0, c_issue = 0; const long long c_begin = clock64();)
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tt) {
                const uint32_t buf = tt & 1;
                FL_CNT(long long c0 = clock64();)
                mbar_wait_idle(tempty + buf, ((tt >> 1) & 1) ^ 1);          // epilogue has drained this accumulator
                FL_CNT(c_tempty += clock64() - c0;)
                tc_fence_after();
                const uint32_t d_main = tmem_base + buf * 256;
                const uint32_t d_gate = d_main + (16u << 16);          // second M = 64 accumulator, interleaved at lane 16
                for (int kb = 0; kb < nkb_total; ++kb) {
                    FL_CNT(c0 = clock64();)
                    mbar_wait(full + s, sph);
                    FL_CNT(c_full += clock64() - c0;)
                    tc_fence_after();
                    const uint32_t sa = stage0 + s * (uint32_t)STAGE_BYTES;
                    const uint64_t dh = make_kmajor_sw128_desc(sa);                 // N side: [H raw ; H lo]  (2 * ROWS rows)
                    const uint64_t dw = make_kmajor_sw128_desc(RES ? wres0 + (uint32_t)kb * WPLANE : sa + HP_BYTES);
                    const bool gate = P.self_mode == 1 && kb == P.nkb_main;
                    const uint32_t d = gate ? d_gate : d_main;
                    FL_CNT(const long long ci0 = clock64();)
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t adv = (uint64_t)((k * 32) >> 4);      // 8 TF32 = 32 bytes along K inside the swizzled row
                        umma_tf32(d, dw + adv, dh + adv, idesc, ((gate || kb == 0) && k == 0) ? 0u : 1u);
                    }
                    umma_commit(empty + s);                                    // stage reusable once these MMAs retire
                    FL_CNT(c_issue += clock64() - ci0;)
                    if (++s == (uint32_t)nstages) {
                        s = 0;
                        sph ^= 1;
                    }
                }
                umma_commit(tfull + buf);                                      // tile complete -> epilogue
            }
            FL_CNT(if (P.dbg) {
                atomicAdd(P.dbg + 3, (unsigned long long)c_full);
                atomicAdd(P.dbg + 4, (unsigned long long)c_tempty);
                atomicAdd(P.dbg + 5, (unsigned long long)(clock64() - c_begin));
                atomicAdd(P.dbg + 10, (unsigned long long)c_issue);
                atomicMax(P.dbg + 11, (unsigned long long)(clock64() - c_begin));
                atomicMin(P.dbg + 12, (unsigned long long)(clock64() - c_begin));
            })
        }
    } else if (warp < 4) {
        // =================================================================== epilogue (128 threads)
        // Accumulator D[m, n]: column n = tile row (n < ROWS: x H_hi, n >= ROWS: x H_lo); weight-plane row m sits in TMEM lane
        //   BNH = 64 (M = 128): lane m;  rows 0-63 W_hi (output column m), 64-127 W_lo
        //   BNH = 32 (M = 64) : lane (m % 16) + 32 * (m / 16);  rows 0-31 W_hi, 32-63 W_lo; the gate accumulator uses the
        //                       same mapping 16 lanes higher.  So warp q sees in lanes 0-15 main rows 16q.., in 16-31 gate rows.
        // Per chunk of 32 tile rows: every warp adds its H_hi and H_lo columns and transposes its lanes through shared memory
        // (T[row][m], conflict-free); then thread (row r, group g) finishes 8 output columns of one row: hi-weight + lo-weight
        // partial sums + bias, ReLU, two 128-bit stores; the gates of a row are spread over its 4 threads.
        const int q = warp;
        constexpr int TS = BNH == 32 ? 68 : 132;                       // row stride of T in floats
        float* Tm = xch;
        float* Tg = xch + 32 * 68 + 16;                                // gate rows (BNH = 32), shifted by 16 banks
        const int Fo = P.Nc, G = P.G;
        const bool has_gates = BNH == 32 && P.self_mode == 1;
        const int et = threadIdx.x;                                    // 0..127
        const int fr = et >> 2, fg = et & 3;                           // finishing role: row of the chunk, column group
        const bool vec_out = (P.ldo % 4 == 0) && ((reinterpret_cast<uintptr_t>(P.out) & 15) == 0);
        uint32_t tt = 0;
        FL_CNT(long long c_tfull = 0; const long long c_begin = clock64();)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tt) {
            const uint32_t buf = tt & 1;
            FL_CNT(const long long cw = clock64();)
            mbar_wait_idle(tfull + buf, (tt >> 1) & 1);
            FL_CNT(c_tfull += clock64() - cw;)
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * 256;
            const int64_t row0 = (int64_t)tile * ROWS;
#pragma unroll 1
            for (int c0 = 0; c0 < ROWS; c0 += 32) {
                {
                    float vh[32], vl[32];
                    tmem_ld32(taddr + c0, vh);
                    tmem_ld32(taddr + ROWS + c0, vl);
                    float* dst;
                    if constexpr (BNH == 32) dst = lane < 16 ? Tm + 16 * q + lane : Tg + 16 * q + (lane - 16);
                    else dst = Tm + 32 * q + lane;
#pragma unroll
                    for (int i = 0; i < 32; ++i) dst[i * TS] = vh[i] + vl[i];
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
                const int64_t r = row0 + c0 + fr;
                if (c0 + fr < ROWS && r < P.N) {
                    const float* trow = Tm + fr * TS;
                    float* orow = P.out + r * P.ldo;
#pragma unroll
                    for (int gg = 0; gg < BNH / 32; ++gg) {
                        const int f0 = 8 * (fg + 4 * gg);
                        if (f0 < Fo) {
                            float o[8];
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const float4 a = *reinterpret_cast<const float4*>(trow + f0 + 4 * h);
                                const float4 b = *reinterpret_cast<const float4*>(trow + BNH + f0 + 4 * h);
                                o[4 * h + 0] = a.x + b.x; o[4 * h + 1] = a.y + b.y; o[4 * h + 2] = a.z + b.z; o[4 * h + 3] = a.w + b.w;
                            }
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                if (P.bias && f0 + k < Fo) o[k] += __ldg(P.bias + f0 + k);
                                if (P.epi == 1) o[k] = fmaxf(o[k], 0.f);
                            }
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                if (vec_out && f0 + 4 * h + 3 < Fo) {
                                    *reinterpret_cast<float4*>(orow + f0 + 4 * h) = make_float4(o[4 * h], o[4 * h + 1], o[4 * h + 2], o[4 * h + 3]);
                                } else {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        if (f0 + 4 * h + k < Fo) orow[f0 + 4 * h + k] = o[4 * h + k];
                                }
                            }
                        }
                    }
                    if (has_gates) {
                        const float* grow = Tg + fr * TS;          // gate rows interleave p1_j (2j) and p2_j (2j+1); lo rows 32 further
                        float* ax = P.aux + r * P.ldaux;
                        for (int j = fg; j < G; j += 4) {
                            float p1 = grow[2 * j] + grow[32 + 2 * j], p2 = grow[2 * j + 1] + grow[32 + 2 * j + 1];
                            if (P.bias_s) {
                                p1 += __ldg(P.bias_s + j);
                                p2 += __ldg(P.bias_s + G + j);
                            }
                            const float t1 = tanh_fast(p1), t2 = tanh_fast(p2);
                            orow[Fo + j] = t1 * t2;
                            if constexpr (AUX) {
                                ax[j] = t1;
                                ax[G + j] = t2;
                            }
                        }
                    }
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + buf);
        }
        FL_CNT(if (P.dbg && lane == 0) {
            atomicAdd(P.dbg + 6, (unsigned long long)c_tfull);
            atomicAdd(P.dbg + 7, (unsigned long long)(clock64() - c_begin));
        })
    } else if (warp >= FL_CTRL_WARPS) {
        // =================================================================== aggregators
        const int aw = warp - FL_CTRL_WARPS;
        const int q = lane >> 2, g = lane & 3;
        const int rq = (q >> 1) | ((q & 1) << 2);          // row of the 8-row group owned by this quad: 0,4,1,5,2,6,3,7
        const int rloc = aw * 8 + rq;                      // (bank-conflict-free 128-bit stores into the swizzled plane)
        const uint32_t row_off = (uint32_t)aw * 1024u + (uint32_t)rq * 128u;
        const uint32_t off0 = row_off + (uint32_t)((g ^ rq) << 4);            // chunk g     (features 4g .. 4g+3)
        const uint32_t off1 = row_off + (uint32_t)(((g + 4) ^ rq) << 4);      // chunk g + 4 (features 16+4g .. 16+4g+3)
        const int* __restrict__ rowptr = P.rowptr;
        const int* __restrict__ col = P.col;
        const int* __restrict__ eperm = P.eperm;
        const float* __restrict__ ea = P.ea;
        const float* __restrict__ X = P.X;
        const int64_t ldx = P.ldx;
        const int Kstride = P.Kstride;
        uint32_t it = 0;
        FL_CNT(long long c_gather = 0, c_wait = 0; const long long c_begin = clock64();)
        uint32_t st_i = 0, st_ph = 1;                    // H-plane stage index / producer parity, kept incrementally
        int tseq = 0;
        if (P.slot_cap > 0) {
            // ------------------------------------------------------------------------------------------------------------
            // Self-prefetching mode (one 32-wide feature block per support).  The rows of a warp are consecutive, so their
            // CSR slots [eb, ee) are contiguous: while the tile's finished k-blocks are handed to the tensor core, the warp
            // already streams the NEXT tile's source rows and edge weights into its private shared-memory slot with 16-byte
            // cp.async copies (no registers held, every edge of the 8 rows in flight at once); the CSR slots of the tile after
            // that and the row bounds of the one after are fetched in the same step, so every dependent global latency
            // (rowptr -> col -> source row) is hidden behind a whole tile period.  The FMAs then read shared memory only.
            // ------------------------------------------------------------------------------------------------------------
            const int CAP = P.slot_cap;
            if (aw == 0 && lane == 0) *reinterpret_cast<volatile int*>(agg_seq) = 1 << 30;      // never hold the L1 prefetch warp back
            const int KC = Kstride >> 2;                                   // 16-byte chunks per edge-weight row
            uint8_t* xs = slots + (size_t)aw * CAP * (128 + 4 * Kstride);  // [CAP][128 B], chunk c of edge pos at (c ^ (pos & 7))
            float* es = reinterpret_cast<float*>(xs + (size_t)CAP * 128);  // [CAP][Kstride]
            const uint32_t xs32 = smem_u32(xs), es32 = smem_u32(es);
            const int kc_shift = KC == 1 ? 0 : (KC == 2 ? 1 : (KC == 4 ? 2 : -1));   // KC = 3 takes the division
            const int nchunk = (P.F + 3) >> 2;                             // valid 16-byte chunks of a source row
            auto bounds = [&](int tile) -> int {                           // lane l <- rowptr[first row of the warp + l], l <= 8
                int v = 0;
                if (tile < P.n_tiles) {
                    const int64_t r = (int64_t)tile * ROWS + aw * 8 + (lane < 8 ? lane : 8);
                    v = __ldg(rowptr + (r < P.N ? r : P.N));
                }
                return v;
            };
            auto loadcols = [&](int ebv, int (&cv)[2], int (&pv)[2]) {
                const int eb = __shfl_sync(0xffffffffu, ebv, 0), n = __shfl_sync(0xffffffffu, ebv, 8) - eb;
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int e = eb + 32 * b + lane;
                    const bool ok = 32 * b + lane < n && n <= CAP;
                    cv[b] = ok ? __ldg(col + e) : 0;
                    pv[b] = ok ? (eperm ? __ldg(eperm + e) : e) : 0;
                }
            };
            auto issue = [&](int ebv, const int (&cv)[2], const int (&pv)[2]) {
                const int eb = __shfl_sync(0xffffffffu, ebv, 0), n = __shfl_sync(0xffffffffu, ebv, 8) - eb;
                if (n <= CAP) {
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        if (32 * b < n) {
                            const int c = lane & 7;
                            const float* xcol = X + 4 * c;
#pragma unroll
                            for (int i = 0; i < 8; ++i) {                  // 4 edges x 8 chunks per instruction: whole 128-byte lines
                                const int j = 4 * i + (lane >> 3), pos = 32 * b + j;
                                const int sidx = __shfl_sync(0xffffffffu, cv[b], j);
                                if (pos < n && c < nchunk)
                                    cp_async_16s(xs32 + (uint32_t)pos * 128u + (uint32_t)((c ^ (pos & 7)) << 4), xcol + (int64_t)sidx * ldx);
                            }
                            for (int i0 = 0; i0 < KC; ++i0) {
                                const int idx = i0 * 32 + lane;
                                const int j = kc_shift >= 0 ? (idx >> kc_shift) : idx / KC;
                                const int h = idx - j * KC, pos = 32 * b + j;
                                const int pe = __shfl_sync(0xffffffffu, pv[b], j);
                                if (pos < n)
                                    cp_async_16s(es32 + (uint32_t)(pos * Kstride + 4 * h) * 4u, ea + (int64_t)pe * Kstride + 4 * h);
                            }
                        }
                    }
                }
            };
            const int t0 = blockIdx.x, gs = gridDim.x;
            int ebvA = bounds(t0), ebvB = bounds(t0 + gs), ebvC = bounds(t0 + 2 * gs);
            int cvB[2], pvB[2];
            {
                int cvA[2], pvA[2];
                loadcols(ebvA, cvA, pvA);
                issue(ebvA, cvA, pvA);
            }
            loadcols(ebvB, cvB, pvB);
            for (int tile = t0; tile < P.n_tiles; tile += gs) {
                FL_CNT(long long cg0 = clock64();)
                const int eb = __shfl_sync(0xffffffffu, ebvA, 0), ntile = __shfl_sync(0xffffffffu, ebvA, 8) - eb;
                const int rs = __shfl_sync(0xffffffffu, ebvA, rq), re = __shfl_sync(0xffffffffu, ebvA, rq + 1);
                const bool staged = ntile <= CAP;
                cp_async_wait_all();
                __syncwarp();
                const int f0 = g * 4, f1 = f0 + 16;
                const bool v0 = f0 < P.F, v1 = f1 < P.F;
                for (int k0 = 0; k0 < P.K; k0 += KT) {
                    float acc[KT][8];
#pragma unroll
                    for (int k = 0; k < KT; ++k)
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc[k][i] = 0.f;
                    if (staged) {
                        // edges of a row in their original order (the reference's CPU order); operands from the warp's slot
                        uint32_t xa_addr = xs32 + (uint32_t)(rs - eb) * 128u;
                        uint32_t w_addr = es32 + (uint32_t)((rs - eb) * Kstride + k0) * 4u;
                        int sw = ((rs - eb) & 7) << 4;
                        const uint32_t wstep = (uint32_t)Kstride * 4u;
                        for (int p = rs; p < re; ++p) {
                            float w[KT];
                            if constexpr (KT % 4 == 0) {
#pragma unroll
                                for (int k = 0; k < KT; k += 4) {
                                    const float4 t = lds128(w_addr + 4 * k);
                                    w[k] = t.x; w[k + 1] = t.y; w[k + 2] = t.z; w[k + 3] = t.w;
                                }
                            } else {
#pragma unroll
                                for (int k = 0; k < KT; ++k) w[k] = lds32(w_addr + 4 * k);
                            }
                            const uint32_t a0 = xa_addr + (uint32_t)((g << 4) ^ sw);
                            float4 xa = make_float4(0.f, 0.f, 0.f, 0.f), xb = xa;
                            if (v0) xa = lds128(a0);
                            if (v1) xb = lds128(a0 ^ 64u);
                            xa_addr += 128u;
                            w_addr += wstep;
                            sw = (sw + 16) & 112;
#pragma unroll
                            for (int k = 0; k < KT; ++k) {
                                acc[k][0] = fmaf(w[k], xa.x, acc[k][0]);
                                acc[k][1] = fmaf(w[k], xa.y, acc[k][1]);
                                acc[k][2] = fmaf(w[k], xa.z, acc[k][2]);
                                acc[k][3] = fmaf(w[k], xa.w, acc[k][3]);
                                acc[k][4] = fmaf(w[k], xb.x, acc[k][4]);
                                acc[k][5] = fmaf(w[k], xb.y, acc[k][5]);
                                acc[k][6] = fmaf(w[k], xb.z, acc[k][6]);
                                acc[k][7] = fmaf(w[k], xb.w, acc[k][7]);
                            }
                        }
                    } else {
                        for (int p = rs; p < re; ++p) {        // more edges than the slot holds: straight from global memory
                            float w[KT];
                            float4 xa = make_float4(0.f, 0.f, 0.f, 0.f), xb = xa;
                            const int sidx = __ldg(col + p);
                            const int eidx = eperm ? __ldg(eperm + p) : p;
#pragma unroll
                            for (int k = 0; k < KT; ++k) w[k] = __ldg(ea + (int64_t)eidx * Kstride + k0 + k);
                            const float* xr = X + (int64_t)sidx * ldx;
                            if (v0) xa = ldg4(xr + f0);
                            if (v1) xb = ldg4(xr + f1);
#pragma unroll
                            for (int k = 0; k < KT; ++k) {
                                acc[k][0] = fmaf(w[k], xa.x, acc[k][0]);
                                acc[k][1] = fmaf(w[k], xa.y, acc[k][1]);
                                acc[k][2] = fmaf(w[k], xa.z, acc[k][2]);
                                acc[k][3] = fmaf(w[k], xa.w, acc[k][3]);
                                acc[k][4] = fmaf(w[k], xb.x, acc[k][4]);
                                acc[k][5] = fmaf(w[k], xb.y, acc[k][5]);
                                acc[k][6] = fmaf(w[k], xb.z, acc[k][6]);
                                acc[k][7] = fmaf(w[k], xb.w, acc[k][7]);
                            }
                        }
                    }
                    __syncwarp();
                    FL_CNT(c_gather += clock64() - cg0;)
                    if (k0 + KT >= P.K) {
                        // the slot is free: stream the next tile in, fetch the CSR slots / bounds of the two after it
                        issue(ebvB, cvB, pvB);
                        ebvA = ebvB;
                        ebvB = ebvC;
                        loadcols(ebvB, cvB, pvB);
                        ebvC = bounds(tile + 3 * gs);
                    }
#pragma unroll
                    for (int k = 0; k < KT; ++k, ++it) {
                        const uint32_t s = st_i;
                        FL_CNT(const long long cw = clock64();)
                        mbar_wait(empty + s, st_ph);
                        FL_CNT(c_wait += clock64() - cw;)
                        uint8_t* a_raw = stages + (size_t)s * STAGE_BYTES;
                        if (++st_i == (uint32_t)nstages) {
                            st_i = 0;
                            st_ph ^= 1;
                        }
                        fl_store_chunk<ROWS * 128>(a_raw, off0, &acc[k][0]);
                        fl_store_chunk<ROWS * 128>(a_raw, off1, &acc[k][4]);
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(full + s);
                    }
                    FL_CNT(cg0 = clock64();)
                }
                if (P.self_mode != 0) {
                    const int64_t row = (int64_t)tile * ROWS + rloc;
                    float sv[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) sv[i] = 0.f;
                    if (row < P.N) {
                        const float* sr = P.S + row * P.lds;
                        if (g * 4 < P.Fs) {
                            const float4 t = ldg4(sr + g * 4);
                            sv[0] = t.x; sv[1] = t.y; sv[2] = t.z; sv[3] = t.w;
                        }
                        if (16 + g * 4 < P.Fs) {
                            const float4 t = ldg4(sr + 16 + g * 4);
                            sv[4] = t.x; sv[5] = t.y; sv[6] = t.z; sv[7] = t.w;
                        }
                    }
                    const uint32_t s = st_i;
                    mbar_wait(empty + s, st_ph);
                    uint8_t* a_raw = stages + (size_t)s * STAGE_BYTES;
                    if (++st_i == (uint32_t)nstages) {
                        st_i = 0;
                        st_ph ^= 1;
                    }
                    fl_store_chunk<ROWS * 128>(a_raw, off0, &sv[0]);
                    fl_store_chunk<ROWS * 128>(a_raw, off1, &sv[4]);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full + s);
                    ++it;
                }
            }
            cp_async_wait_all();
        } else
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
            if (aw == 0 && lane == 0) *reinterpret_cast<volatile int*>(agg_seq) = ++tseq;
            const int64_t row = (int64_t)tile * ROWS + rloc;
            int rs = 0, re = 0;
            FL_CNT(long long cg0 = clock64();)
            if (row < P.N) {
                rs = __ldg(rowptr + row);
                re = __ldg(rowptr + row + 1);
            }
            for (int fh = 0; fh < P.nfh; ++fh) {
                const int f0 = fh * 32 + g * 4, f1 = f0 + 16;
                const bool v0 = f0 < P.F, v1 = f1 < P.F;
                for (int k0 = 0; k0 < P.K; k0 += KT) {
                    float acc[KT][8];
#pragma unroll
                    for (int k = 0; k < KT; ++k)
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc[k][i] = 0.f;
                    constexpr int U = FL_UD;   // edges in flight per lane
                    // the CSR slots of the NEXT iteration are fetched one iteration ahead, so that the index -> gather chain
                    // costs one memory latency per iteration instead of two
                    int sidx_n[U], eidx_n[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int p = max(min(rs + u, re - 1), 0);
                        sidx_n[u] = rs < re ? __ldg(col + p) : 0;
                        eidx_n[u] = (rs < re && eperm) ? __ldg(eperm + p) : p;
                    }
                    for (int p0 = rs; p0 < re; p0 += U) {
                        int sidx[U], eidx[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            sidx[u] = sidx_n[u];
                            eidx[u] = eidx_n[u];
                        }
                        if (p0 + U < re) {
#pragma unroll
                            for (int u = 0; u < U; ++u) {
                                const int p = min(p0 + U + u, re - 1);
                                sidx_n[u] = __ldg(col + p);
                                eidx_n[u] = eperm ? __ldg(eperm + p) : p;
                            }
                        }
                        float w[U][KT];
                        float4 xa[U], xb[U];
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            fl_load_ea<KT>(ea + (int64_t)eidx[u] * Kstride + k0, w[u]);
                            const float* xr = X + (int64_t)sidx[u] * ldx;
                            xa[u] = v0 ? ldg4(xr + f0) : make_float4(0.f, 0.f, 0.f, 0.f);
                            xb[u] = v1 ? ldg4(xr + f1) : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int u = 0; u < U; ++u) {
                            if (p0 + u < re) {       // edges of a row in their original order (the reference's CPU order)
#pragma unroll
                                for (int k = 0; k < KT; ++k) {
                                    acc[k][0] = fmaf(w[u][k], xa[u].x, acc[k][0]);
                                    acc[k][1] = fmaf(w[u][k], xa[u].y, acc[k][1]);
                                    acc[k][2] = fmaf(w[u][k], xa[u].z, acc[k][2]);
                                    acc[k][3] = fmaf(w[u][k], xa[u].w, acc[k][3]);
                                    acc[k][4] = fmaf(w[u][k], xb[u].x, acc[k][4]);
                                    acc[k][5] = fmaf(w[u][k], xb[u].y, acc[k][5]);
                                    acc[k][6] = fmaf(w[u][k], xb[u].z, acc[k][6]);
                                    acc[k][7] = fmaf(w[u][k], xb[u].w, acc[k][7]);
                                }
                            }
                        }
                    }
                    if (P.hout && row < P.N) {           // side output for the weight-gradient contraction of the backward
                        float* hr = P.hout + row * P.ldh + (int64_t)k0 * 32 * P.nfh + fh * 32 + g * 4;
#pragma unroll
                        for (int k = 0; k < KT; ++k) {
                            st_na4(hr + k * 32 * P.nfh, make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]));
                            st_na4(hr + k * 32 * P.nfh + 16, make_float4(acc[k][4], acc[k][5], acc[k][6], acc[k][7]));
                        }
                    }
                    // hand the KT finished k-blocks to the tensor core
                    __syncwarp();
                    FL_CNT(c_gather += clock64() - cg0;)
#pragma unroll
                    for (int k = 0; k < KT; ++k, ++it) {
                        const uint32_t s = st_i;
                        FL_CNT(const long long cw = clock64();)
                        mbar_wait(empty + s, st_ph);
                        FL_CNT(c_wait += clock64() - cw;)
                        uint8_t* a_raw = stages + (size_t)s * STAGE_BYTES;
                        if (++st_i == (uint32_t)nstages) {
                            st_i = 0;
                            st_ph ^= 1;
                        }
                        fl_store_chunk<ROWS * 128>(a_raw, off0, &acc[k][0]);
                        fl_store_chunk<ROWS * 128>(a_raw, off1, &acc[k][4]);
                        fence_proxy_async_smem();      // generic-proxy stores -> visible to the tensor core (async proxy)
                        __syncwarp();
                        if (lane == 0) mbar_arrive(full + s);
                    }
                    FL_CNT(cg0 = clock64();)
                }
            }
            if (P.self_mode != 0) {
                float sv[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) sv[i] = 0.f;
                if (row < P.N) {
                    const float* sr = P.S + row * P.lds;
                    if (g * 4 < P.Fs) {
                        const float4 t = ldg4(sr + g * 4);
                        sv[0] = t.x; sv[1] = t.y; sv[2] = t.z; sv[3] = t.w;
                    }
                    if (16 + g * 4 < P.Fs) {
                        const float4 t = ldg4(sr + 16 + g * 4);
                        sv[4] = t.x; sv[5] = t.y; sv[6] = t.z; sv[7] = t.w;
                    }
                }
                if (P.hout && row < P.N) {
                    float* hr = P.hout + row * P.ldh + (int64_t)P.K * 32 * P.nfh + g * 4;
                    st_na4(hr, make_float4(sv[0], sv[1], sv[2], sv[3]));
                    st_na4(hr + 16, make_float4(sv[4], sv[5], sv[6], sv[7]));
                }
                const uint32_t s = st_i;
                mbar_wait(empty + s, st_ph);
                uint8_t* a_raw = stages + (size_t)s * STAGE_BYTES;
                if (++st_i == (uint32_t)nstages) {
                    st_i = 0;
                    st_ph ^= 1;
                }
                fl_store_chunk<ROWS * 128>(a_raw, off0, &sv[0]);
                fl_store_chunk<ROWS * 128>(a_raw, off1, &sv[4]);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full + s);
                ++it;
            }
        }
        FL_CNT(if (P.dbg && lane == 0) {
            atomicAdd(P.dbg + 0, (unsigned long long)c_gather);
            atomicAdd(P.dbg + 1, (unsigned long long)c_wait);
            atomicAdd(P.dbg + 2, (unsigned long long)(clock64() - c_begin));
        })
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, 512);
}

// Pre-split, transposed (K-major) weight planes: one [2*BNH rows x 32] plane per k-block, in the order the aggregators
// produce the k-blocks: kb = fh * K + k covers rows (k * F + fh * 32 + c), c < 32, of Bmain [K*F, Nc]; kb = nfh * K is
// the self block.  Plane rows (the MMA's M side): [0, BNH) hi = RN-TF32(w) of output column n, [BNH, 2 BNH) lo = w - hi.
// Self plane: mode 2 -> Bself [Fs, Nc] in the same layout; mode 1 -> the gate weights Bself [Fs, 2G] with the gate
// columns interleaved (p1_0 p2_0 p1_1 p2_1 ..).
__global__ void k_fl_prep_weights(const float* __restrict__ Bmain, int64_t ldb, int K, int F, int Nc, int nfh, int BNH,
                                  const float* __restrict__ Bself, int64_t ldbs, int Fs, int Ns, int self_mode,
                                  float* __restrict__ planes) {
    const int nkb_main = nfh * K;
    const int nkb_total = nkb_main + (self_mode != 0 ? 1 : 0);
    const int MR = 2 * BNH;
    const int total = nkb_total * MR * 32;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int kb = i / (MR * 32), m = (i / 32) % MR, c = i % 32;
        const int n = m % BNH;
        const bool is_lo = m >= BNH;
        float v = 0.f;
        if (kb < nkb_main) {
            const int fh = kb / K, k = kb % K, f = fh * 32 + c;
            if (f < F && n < Nc) v = __ldg(Bmain + ((int64_t)k * F + f) * ldb + n);
        } else if (self_mode == 2) {
            if (c < Fs && n < Nc) v = __ldg(Bself + (int64_t)c * ldbs + n);
        } else {
            const int src_n = (n & 1) ? (Ns / 2 + (n >> 1)) : (n >> 1);
            if (c < Fs && n < Ns) v = __ldg(Bself + (int64_t)c * ldbs + src_n);
        }
        const float h = tf32_rn(v);
        planes[i] = is_lo ? v - h : h;
    }
}

}  // namespace gnnml3

using namespace gnnml3;

static inline int fl_bnh_for(int Nc) { return Nc <= 32 ? 32 : 64; }
static inline int fl_kt_for(int K) {
    if (K >= 4 && K <= 8) return K;
    if (K > 8 && K <= 16 && K % 2 == 0) return K / 2;
    return 0;
}

// optional cycle counters (GNNML3_FUSED_DEBUG=1): [0] aggregator gather, [1] aggregator waiting for a free stage,
// [2] aggregator total, [3] MMA thread waiting for stages, [4] MMA thread waiting for a drained accumulator, [5] MMA
// thread total, [6] epilogue waiting for a tile, [7] epilogue total (sums over warps / CTAs)
static unsigned long long* g_fl_dbg = nullptr;
static const bool g_fl_debug = [] {
    const char* e = getenv("GNNML3_FUSED_DEBUG");
    return e && e[0] == '1';
}();

extern "C" int gnnml3_fused_debug_counters(unsigned long long* out8_host, int reset) {
    if (!g_fl_dbg) {
        for (int i = 0; i < 16; ++i) out8_host[i] = 0;
        return GNNML3_OK;
    }
    GNNML3_CUDA(cudaDeviceSynchronize());
    GNNML3_CUDA(cudaMemcpy(out8_host, g_fl_dbg, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (reset) {
        GNNML3_CUDA(cudaMemset(g_fl_dbg, 0, 16 * sizeof(unsigned long long)));
        GNNML3_CUDA(cudaMemset(g_fl_dbg + 12, 0xff, sizeof(unsigned long long)));      // slot 12 is a minimum
    }
    return GNNML3_OK;
}

static const int g_fl_pf_rows = [] {
    const char* e = getenv("GNNML3_FUSED_PF_ROWS");
    return e ? atoi(e) : 40;
}();

// K = 8 (the ZINC configuration) runs as two register passes of 4 supports with 16 aggregator warps and 128-row tiles
// (N = 256: the largest tcgen05.mma, a third fewer instructions per row than the 80-row tiles): measured 7-10 % faster than
// the single pass with 10 warps.  GNNML3_FUSED_NAGG16=0 restores the single pass.
static int g_fl_nagg16 = [] {
    const char* e = getenv("GNNML3_FUSED_NAGG16");
    return (e && e[0] == '0') ? 0 : 1;
}();

extern "C" int gnnml3_fused_supported(int K, int Kstride, int F, int Nc, int Fs, int self_mode, int Ns) {
    if (gnnml3_fused_ts_supported(K, Kstride, F, Nc, Fs, self_mode, Ns)) return 1;
    const int kt = fl_kt_for(K);
    if (kt == 0 || F < 1 || Nc < 1 || Nc > 64) return 0;
    if (((F + 31) / 32) * K > 24) return 0;               // accumulation chain per tile kept short (TMEM adds truncate)
    if (kt % 4 == 0 && Kstride % 4 != 0) return 0;        // 128-bit edge-weight loads
    if (kt % 4 != 0 && kt % 2 == 0 && Kstride % 2 != 0) return 0;
    if (self_mode != 0 && (Fs < 1 || Fs > 32)) return 0;
    if (self_mode == 1 && (Ns < 2 || Ns > 32 || Ns % 2 != 0 || Nc > 32)) return 0;
    return 1;
}

extern "C" size_t gnnml3_fused_workspace_bytes(int K, int F, int Nc, int self_mode) {
    const int nfh = cdiv(F, 32);
    const size_t a = align_up((size_t)(nfh * K + (self_mode != 0 ? 1 : 0)) * 2 * fl_bnh_for(Nc) * 128, 256);
    const size_t b = gnnml3_fused_ts_workspace_bytes(K, Nc, self_mode);
    return a > b ? a : b;
}

constexpr size_t FL_SMEM_MAX = 227 * 1024;                                              // opt-in limit per CTA on sm_100
constexpr size_t FL_SMEM_FIXED = 2 * FL_XCH * sizeof(float) + 1024 /*alignment slack*/ + 256 /*barriers*/ + 128 /*slot alignment*/;

// Per-launch device timing for bench.py's roofline: CUDA events recorded on the launching stream around the kernel
// (gnnml3_fused_profile / gnnml3_fused_profile_fetch).  Off by default; not thread-safe (a measurement aid).
struct FLProfRec {
    cudaEvent_t a, b;
    double meta[9];      // N, K, F, Nc, Fs, self_mode, Ns, G, has_perm
};
static bool g_fl_prof_on = false;
static std::vector<FLProfRec> g_fl_prof;

extern "C" int gnnml3_fused_profile(int enable) {
    for (auto& r : g_fl_prof) {
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    g_fl_prof.clear();
    g_fl_prof_on = enable != 0;
    return GNNML3_OK;
}

// out [max][10]: milliseconds, N, K, F, Nc, Fs, self_mode, Ns, G, has_perm of every fused launch since profiling was
// enabled; synchronises the device.  Returns the number of records written.
extern "C" int gnnml3_fused_profile_fetch(double* out, int max) {
    cudaDeviceSynchronize();
    int n = 0;
    for (auto& r : g_fl_prof) {
        if (n >= max) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        out[n * 10] = ms;
        for (int i = 0; i < 9; ++i) out[n * 10 + 1 + i] = r.meta[i];
        ++n;
    }
    return n;
}

template <int KT, int BNH, int NAGG, bool RES, bool AUX>
static int fl_launch2(const CUtensorMap& mW, FLParams& P, size_t smem, cudaStream_t st) {
    static bool configured[64] = {};
    if (auto once_ = first_use_on_device(configured))
        GNNML3_CUDA(cudaFuncSetAttribute(k_fused_agg_proj<KT, BNH, NAGG, RES, AUX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)FL_SMEM_MAX));
    const int grid = P.n_tiles < kNumSMs ? P.n_tiles : kNumSMs;
    FLProfRec rec;
    if (g_fl_prof_on) {
        cudaEventCreate(&rec.a);
        cudaEventCreate(&rec.b);
        const double m[9] = {(double)P.N, (double)P.K, (double)P.F, (double)P.Nc, (double)P.Fs, (double)P.self_mode,
                             (double)(P.self_mode == 1 ? 2 * P.G : 0), (double)P.G, P.eperm ? 1.0 : 0.0};
        for (int i = 0; i < 9; ++i) rec.meta[i] = m[i];
        cudaEventRecord(rec.a, st);
    }
    k_fused_agg_proj<KT, BNH, NAGG, RES, AUX><<<grid, 32 * (FL_CTRL_WARPS + NAGG), smem, st>>>(mW, P);
    if (g_fl_prof_on) {
        cudaEventRecord(rec.b, st);
        g_fl_prof.push_back(rec);
    }
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

namespace gnnml3 {
// tensor-memory generation of the kernel (fused_layer_ts.cu)
int fused_ts_run(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea, int Kstride, int K, const float* X,
                 int64_t ldx, int F, const float* S, int64_t lds, int Fs, int self_mode, const float* Bmain, int64_t ldb,
                 const float* Bself, int64_t ldbs, int Ns, const float* bias, const float* bias_s, int64_t N, int Nc, float* out,
                 int64_t ldo, float* aux, int64_t ldaux, int G, int epilogue, float* hout, int64_t ldh, const int32_t* tilewin,
                 void* workspace, size_t workspace_bytes, unsigned long long* dbg, cudaStream_t st);
void fused_path_count(int which);
}
extern "C" int gnnml3_fused_ts_supported(int K, int Kstride, int F, int Nc, int Fs, int self_mode, int Ns);
extern "C" size_t gnnml3_fused_ts_workspace_bytes(int K, int Nc, int self_mode);

// Weight planes stay resident in shared memory when at least 3 H-plane stages fit beside them; otherwise every k-block's
// plane is streamed from L2 into its stage (large K * F: L2-bandwidth bound, see DESIGN.md).
// Aggregator mode (gnnml3_fused_set_mode): 0 = gather straight from global memory, weight planes resident (default: the
// two modes measure the same on B200 -- the kernel is paced by the plane hand-off / MMA chain, see DESIGN.md -- and this is
// the simpler one); 1 = per-warp cp.async prefetch slots.  GNNML3_FUSED_SLOT=1 selects mode 1 at load time.
static int g_fl_slot_mode = [] {
    const char* e = getenv("GNNML3_FUSED_SLOT");
    return (e && e[0] == '1') ? 1 : 0;
}();
#define g_fl_no_slot (g_fl_slot_mode == 0)

extern "C" int gnnml3_fused_set_mode(int slot_mode) {
    const int old = g_fl_slot_mode;
    if (slot_mode == 0 || slot_mode == 1) g_fl_slot_mode = slot_mode;
    return old;
}

static const size_t g_fl_max_stages = [] {
    const char* e = getenv("GNNML3_FUSED_MAXSTAGES");       // experiments: cap the depth of the H-plane ring
    return (size_t)(e ? atoi(e) : FL_MAX_STAGES);
}();

// Shared-memory plan.  Preferred: per-warp prefetch slots (64 edges each) + as many H-plane stages as fit, weight planes
// resident if there is still room for 3 stages, otherwise streamed from L2 into the stages.  Without slots (wide feature
// blocks, odd edge-weight strides): resident weights when 3 stages fit beside them, else streamed.
template <int KT, int BNH, int NAGG, bool AUX = true>
static int fl_launch(const CUtensorMap& mW, FLParams& P, cudaStream_t st) {
    constexpr int ROWS = 8 * NAGG;
    constexpr size_t HP = 2 * ROWS * 128, WPLANE = 2 * BNH * 128;
    P.n_tiles = cdiv(P.N, ROWS);
    const size_t nkb_total = P.nkb_main + (P.self_mode != 0 ? 1 : 0);
    const size_t resident = nkb_total * WPLANE;
    const size_t slot_cap = 64;
    const size_t slots = (P.nfh == 1 && P.Kstride % 4 == 0 && P.Kstride <= 16 && !g_fl_no_slot)
                             ? (size_t)NAGG * slot_cap * (128 + 4 * (size_t)P.Kstride) : 0;
    P.slot_cap = 0;
    if (slots) {
        if (resident + slots + 3 * HP + FL_SMEM_FIXED <= FL_SMEM_MAX) {
            size_t ns = (FL_SMEM_MAX - FL_SMEM_FIXED - resident - slots) / HP;
            if (ns > FL_MAX_STAGES) ns = FL_MAX_STAGES;
        if (ns > g_fl_max_stages) ns = g_fl_max_stages;
            P.nstages = (int)ns;
            P.slot_cap = (int)slot_cap;
            return fl_launch2<KT, BNH, NAGG, true, AUX>(mW, P, resident + ns * HP + FL_SMEM_FIXED + slots, st);
        }
        if (slots + 2 * (HP + WPLANE) + FL_SMEM_FIXED <= FL_SMEM_MAX) {
            size_t ns = (FL_SMEM_MAX - FL_SMEM_FIXED - slots) / (HP + WPLANE);
            if (ns > FL_MAX_STAGES) ns = FL_MAX_STAGES;
        if (ns > g_fl_max_stages) ns = g_fl_max_stages;
            P.nstages = (int)ns;
            P.slot_cap = (int)slot_cap;
            return fl_launch2<KT, BNH, NAGG, false, AUX>(mW, P, ns * (HP + WPLANE) + FL_SMEM_FIXED + slots, st);
        }
    }
    if (resident + 3 * HP + FL_SMEM_FIXED <= FL_SMEM_MAX) {
        size_t ns = (FL_SMEM_MAX - FL_SMEM_FIXED - resident) / HP;
        if (ns > FL_MAX_STAGES) ns = FL_MAX_STAGES;
        if (ns > g_fl_max_stages) ns = g_fl_max_stages;
        P.nstages = (int)ns;
        return fl_launch2<KT, BNH, NAGG, true, AUX>(mW, P, resident + ns * HP + FL_SMEM_FIXED, st);
    }
    size_t ns = (FL_SMEM_MAX - FL_SMEM_FIXED) / (HP + WPLANE);
    if (ns > FL_MAX_STAGES) ns = FL_MAX_STAGES;
        if (ns > g_fl_max_stages) ns = g_fl_max_stages;
    P.nstages = (int)ns;
    return fl_launch2<KT, BNH, NAGG, false, AUX>(mW, P, ns * (HP + WPLANE) + FL_SMEM_FIXED, st);
}

// aggregator warps per CTA by register need: KT x 8 accumulators per lane.  512 threads leave 128 registers per thread
// (KT >= 7), 640 threads 96 (KT <= 6); the 16-warp / 4-supports-per-pass variant runs at 80.
// K supports are processed in register tiles of KT; with the prefetch slots (operands re-read from shared memory at no
// global cost) K = 8 runs as two passes of 4 so that the tensor core works on the first four k-blocks while the second
// pass accumulates (GNNML3_FUSED_SPLIT=0 restores the single pass).
static const bool g_fl_split = [] {
    const char* e = getenv("GNNML3_FUSED_SPLIT");
    return !(e && e[0] == '0');
}();

static const bool g_fl_wide = [] {
    const char* e = getenv("GNNML3_FUSED_WIDE");      // experiment: K = 8 as two passes of 4 with 14 aggregator warps (112-row tiles)
    return e && e[0] == '1';
}();

#define FL_DISPATCH_KT(KTV, BNV, AUXV)                                                                \
    switch (KTV) {                                                                                    \
        case 4: return (K == 8 && !g_fl_wide) ? fl_launch<4, BNV, 10, AUXV>(mW, P, st) : fl_launch<4, BNV, 14, AUXV>(mW, P, st); \
        case 5: return fl_launch<5, BNV, 14, AUXV>(mW, P, st);                                        \
        case 6: return fl_launch<6, BNV, 14, AUXV>(mW, P, st);                                        \
        case 7: return fl_launch<7, BNV, 10, AUXV>(mW, P, st);                                        \
        case 8: return fl_launch<8, BNV, 10, AUXV>(mW, P, st);                                        \
        default: return set_err(GNNML3_ERR_INVALID, "fused_agg_proj: no kernel for K tile %d", KTV);  \
    }

extern "C" int gnnml3_fused_agg_proj(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea,
                                     int Kstride, int K, const float* X, int64_t ldx, int F, const float* S, int64_t lds,
                                     int Fs, int self_mode, const float* Bmain, int64_t ldb, const float* Bself,
                                     int64_t ldbs, int Ns, const float* bias, const float* bias_s, int64_t N, int Nc,
                                     float* out, int64_t ldo, float* aux, int64_t ldaux, int G, int epilogue,
                                     float* hout, int64_t ldh, const int32_t* tilewin, void* workspace, size_t workspace_bytes,
                                     void* stream_) {
    GNNML3_REQUIRE(N > 0 && N < (1ll << 31) - 256, "fused_agg_proj: bad N");
    GNNML3_REQUIRE(rowptr && col && ea && X && Bmain && out && workspace, "fused_agg_proj: NULL pointer");
    GNNML3_REQUIRE(gnnml3_fused_supported(K, Kstride, F, Nc, Fs, self_mode, Ns), "fused_agg_proj: unsupported shape "
                   "K=%d Kstride=%d F=%d Nc=%d Fs=%d self_mode=%d Ns=%d", K, Kstride, F, Nc, Fs, self_mode, Ns);
    GNNML3_REQUIRE(ldx % 4 == 0 && (uintptr_t)X % 16 == 0, "fused_agg_proj: X rows must be 16-byte aligned (ldx %% 4 == 0)");
    GNNML3_REQUIRE((uintptr_t)ea % 16 == 0, "fused_agg_proj: ea must be 16-byte aligned");
    GNNML3_REQUIRE(self_mode == 0 || (S && Bself && lds % 4 == 0 && (uintptr_t)S % 16 == 0),
                   "fused_agg_proj: self block needs S, Bself and 16-byte aligned rows");
    const int prec_bits = epilogue & 0x300;                  // GNNML3_FUSED_TF32 / GNNML3_FUSED_BF16 (tensor-memory kernel only)
    epilogue &= 0xff;
    GNNML3_REQUIRE(epilogue == 0 || epilogue == 1, "fused_agg_proj: unknown epilogue");
    GNNML3_REQUIRE(prec_bits == 0 || prec_bits == 0x100 || prec_bits == 0x200, "fused_agg_proj: unknown precision flag");
    GNNML3_REQUIRE(prec_bits == 0 || (gnnml3_fused_ts_supported(K, Kstride, F, Nc, Fs, self_mode, Ns) && g_fl_slot_mode == 0),
                   "fused_agg_proj: the single-pass TF32 / BF16 modes exist in the tensor-memory kernel only (F <= 32, even K)");
    GNNML3_REQUIRE(self_mode != 1 || (epilogue == 1 && G >= 1 && G <= 16 && Ns == 2 * G),
                   "fused_agg_proj: gate columns need the ML3 epilogue and Ns == 2G <= 32");
    GNNML3_REQUIRE(ldo >= Nc + (self_mode == 1 ? G : 0), "fused_agg_proj: ldo too small");
    GNNML3_REQUIRE(hout == nullptr || (ldh % 4 == 0 && (uintptr_t)hout % 16 == 0 && g_fl_slot_mode == 0 &&
                                       ldh >= (int64_t)(K + (self_mode != 0 ? 1 : 0)) * 32 * cdiv(F, 32)),
                   "fused_agg_proj: hout needs the default aggregator mode and 16-byte aligned rows of (K [+1]) * 32 * ceil(F/32) floats");
    if (workspace_bytes < gnnml3_fused_workspace_bytes(K, F, Nc, self_mode))
        return set_err(GNNML3_ERR_WORKSPACE, "fused_agg_proj: workspace too small");
    cudaStream_t st = (cudaStream_t)stream_;
    if (g_fl_debug && !g_fl_dbg) {
        GNNML3_CUDA(cudaMalloc(&g_fl_dbg, 16 * sizeof(unsigned long long)));
        GNNML3_CUDA(cudaMemset(g_fl_dbg, 0, 16 * sizeof(unsigned long long)));
    }
    if (gnnml3_fused_ts_supported(K, Kstride, F, Nc, Fs, self_mode, Ns) && g_fl_slot_mode == 0) {
        // tensor-memory generation (fused_layer_ts.cu): one 32-wide feature block per support, K % 2 == 0
        FLProfRec rec;
        if (g_fl_prof_on) {
            cudaEventCreate(&rec.a);
            cudaEventCreate(&rec.b);
            const double m[9] = {(double)N, (double)K, (double)F, (double)Nc, (double)Fs, (double)self_mode,
                                 (double)(self_mode == 1 ? 2 * G : 0), (double)G, eperm ? 1.0 : 0.0};
            for (int i = 0; i < 9; ++i) rec.meta[i] = m[i];
            cudaEventRecord(rec.a, st);
        }
        const int rc = fused_ts_run(rowptr, col, eperm, ea, Kstride, K, X, ldx, F, S, lds, Fs, self_mode, Bmain, ldb, Bself, ldbs, Ns, bias,
                                    bias_s, N, Nc, out, ldo, aux, ldaux, G, epilogue | prec_bits, hout, ldh, tilewin, workspace, workspace_bytes,
                                    g_fl_dbg, st);
        if (g_fl_prof_on) {
            cudaEventRecord(rec.b, st);
            g_fl_prof.push_back(rec);
        }
        if (rc == GNNML3_OK) fused_path_count(0);
        return rc;
    }
    fused_path_count(1);
    const int BNH = fl_bnh_for(Nc);
    int KT = fl_kt_for(K);
    GNNML3_REQUIRE(KT != 0, "fused_agg_proj: no shared-memory-plane kernel for K=%d", K);
    const int nfh = cdiv(F, 32);
    if (K == 8 && g_fl_split && nfh == 1 && Kstride % 4 == 0 && !g_fl_no_slot) KT = 4;
    if (K == 8 && g_fl_wide) KT = 4;
    const int nkb_main = nfh * K;
    const int nkb_total = nkb_main + (self_mode != 0 ? 1 : 0);
    float* planes = (float*)workspace;
    {
        const int total = nkb_total * 2 * BNH * 32;
        const int blocks = cdiv(total, 256) > 592 ? 592 : cdiv(total, 256);
        k_fl_prep_weights<<<blocks, 256, 0, st>>>(Bmain, ldb, K, F, Nc, nfh, BNH, Bself, ldbs, Fs, Ns, self_mode, planes);
        GNNML3_LAUNCH_CHECK();
    }
    CUtensorMap mW;
    int rc;
    if ((rc = make_map(&mW, planes, (int64_t)nkb_total * 2 * BNH, 32, 32, 2 * BNH))) return rc;
    FLParams P;
    P.rowptr = rowptr; P.col = col; P.eperm = eperm; P.ea = ea; P.Kstride = Kstride; P.K = K;
    P.X = X; P.ldx = ldx; P.F = F; P.S = S; P.lds = lds; P.Fs = Fs; P.self_mode = self_mode;
    P.N = N; P.n_tiles = 0; P.nfh = nfh; P.nkb_main = nkb_main; P.nstages = 0; P.pf_rows = g_fl_pf_rows; P.slot_cap = 0;
    P.bias = bias; P.bias_s = bias_s; P.out = out; P.ldo = ldo; P.Nc = Nc; P.aux = aux; P.ldaux = ldaux; P.G = G;
    P.epi = epilogue;
    P.hout = hout; P.ldh = ldh;
    P.dbg = g_fl_dbg;
    // gated epilogue without aux (inference): the forward-only instantiations; gates exist with BNH == 32 only
    const bool fwd_only = self_mode == 1 && !aux;
    if (g_fl_nagg16 && K == 8 && Kstride % 4 == 0 && g_fl_no_slot) {     // 16 aggregator warps, 4 supports per pass, 128-row tiles
        if (BNH == 32) return fwd_only ? fl_launch<4, 32, 16, false>(mW, P, st) : fl_launch<4, 32, 16>(mW, P, st);
        return fl_launch<4, 64, 16>(mW, P, st);
    }
    if (BNH == 32 && fwd_only) { FL_DISPATCH_KT(KT, 32, false) }
    if (BNH == 32) { FL_DISPATCH_KT(KT, 32, true) }
    FL_DISPATCH_KT(KT, 64, true)
}
