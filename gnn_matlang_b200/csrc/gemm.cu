// Tall-skinny tensor-core contractions of the SpectConv projection and its gradients.
//
//   gemm_nn : C[M, Nc] = A[M, Kc] * B[Kc, Nc] (+ bias) (+ ReLU)   -- sum_k P_k(x) W_k as ONE contraction over K*Fi
//             (reference libs/spect_conv.py:80 issues K separate matmuls + K adds; bias :93-94)
//   gemm_tn : C[Ka, Nb] = A[M, Ka]^T * B[M, Nb]                   -- weight gradients (contraction over the nodes),
//             split over M with a fixed-order second pass => deterministic, no atomics
//   colsum  : out[c] = sum_r A[r, c]                              -- bias gradient
//
// M (nodes) is 1e3..1e6+, Nc/Ka/Nb/Kc are 2..2560, so the kernels are bound by streaming the tall operand from
// HBM once; the math runs on the tensor cores as TF32 m16n8k8 with FP32 accumulation.  Default arithmetic is
// the error-compensated 3xTF32 split (a = hi + lo, a*b ~= lo*hi + hi*lo + hi*hi), which restores FP32-grade
// accuracy (needed for the rtol 1e-5 parity bar); GNNML3_PREC_TF32 and GNNML3_PREC_BF16 run the single-pass variant.
#include "common.cuh"

namespace gnnml3 {

__device__ __forceinline__ uint32_t f2tf32(float f) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(f));
    return r;
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int N>
__device__ __forceinline__ void split_tf32(const float (&v)[N], uint32_t (&hi)[N], uint32_t (&lo)[N]) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        hi[i] = f2tf32(v[i]);
        lo[i] = f2tf32(v[i] - __uint_as_float(hi[i]));
    }
}

// 16-byte cp.async that reads only the first `bytes` (0..16) from global memory and zero-fills the rest
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int bytes) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem, const void* gmem, bool valid) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
    int sz = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(s), "l"(gmem), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// rows x cols tile of a row-major matrix -> padded smem tile (row stride LDS floats); out-of-range -> 0
template <int ROWS, int COLS, int LDS, int THREADS, bool VEC16>
__device__ __forceinline__ void load_tile(float* __restrict__ s, const float* __restrict__ g, int64_t ld, int64_t r0,
                                          int c0, int64_t rmax, int cmax) {
    if constexpr (VEC16) {
        constexpr int CV = COLS / 4;
        constexpr int TOTAL = ROWS * CV;
#pragma unroll
        for (int i = threadIdx.x; i < TOTAL; i += THREADS) {
            const int r = i / CV, c = (i % CV) * 4;
            int nb = (r0 + r < rmax) ? (cmax - (c0 + c)) * 4 : 0;     // rows need 16-byte alignment only; the row
            nb = nb < 0 ? 0 : (nb > 16 ? 16 : nb);                    // tail is a partial vector (zero-filled)
            const float* src = nb > 0 ? g + (r0 + r) * ld + c0 + c : g;
            cp_async16(s + r * LDS + c, src, nb);
        }
    } else {
        constexpr int TOTAL = ROWS * COLS;
#pragma unroll 4
        for (int i = threadIdx.x; i < TOTAL; i += THREADS) {
            const int r = i / COLS, c = i % COLS;
            const bool ok = (r0 + r < rmax) && (c0 + c < cmax);
            const float* src = ok ? g + (r0 + r) * ld + c0 + c : g;
            cp_async4(s + r * LDS + c, src, ok);
        }
    }
}

// ------------------------------------------------------------------------------------------------ gemm_nn
constexpr int NN_BM = 128, NN_BK = 32, NN_STAGES = 3, NN_THREADS = 256, NN_LDA = NN_BK + 4;

template <int BN>
constexpr size_t nn_smem_bytes() {
    return sizeof(float) * NN_STAGES * (NN_BM * NN_LDA + NN_BK * (BN + 8));
}

template <int BN, bool VA, bool VB, bool X3>
__global__ void __launch_bounds__(NN_THREADS)
k_gemm_nn(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb,
          const float* __restrict__ bias, float* __restrict__ C, int64_t ldc, int64_t M, int Nc, int Kc, int epi) {
    constexpr int LDB = BN + 8;
    constexpr int NT = BN / 16;  // n-tiles (8 wide) per warp: the block's BN columns are split over 2 warp columns
    extern __shared__ __align__(16) float smem[];
    float* As = smem;
    float* Bs = smem + NN_STAGES * NN_BM * NN_LDA;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    const int64_t m0 = (int64_t)blockIdx.x * NN_BM;
    const int n0 = blockIdx.y * BN;
    const int nk = (Kc + NN_BK - 1) / NN_BK;

    float acc[2][NT][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[i][j][r] = 0.f;

    auto issue = [&](int kt) {
        const int st = kt % NN_STAGES;
        load_tile<NN_BM, NN_BK, NN_LDA, NN_THREADS, VA>(As + st * NN_BM * NN_LDA, A, lda, m0, kt * NN_BK, M, Kc);
        load_tile<NN_BK, BN, LDB, NN_THREADS, VB>(Bs + st * NN_BK * LDB, B, ldb, (int64_t)kt * NN_BK, n0, Kc, Nc);
    };
#pragma unroll
    for (int s = 0; s < NN_STAGES - 1; ++s) {
        if (s < nk) issue(s);
        cp_async_commit();
    }
    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<NN_STAGES - 2>();
        __syncthreads();
        if (kt + NN_STAGES - 1 < nk) issue(kt + NN_STAGES - 1);
        cp_async_commit();
        const float* as = As + (kt % NN_STAGES) * NN_BM * NN_LDA + (wm * 32) * NN_LDA;
        const float* bs = Bs + (kt % NN_STAGES) * NN_BK * LDB + wn * (BN / 2);
        // The tensor core adds into its accumulator with truncation; over thousands of k-steps that bias would
        // exceed the FP32 parity bar.  Each k-tile therefore accumulates from zero and is folded into the running
        // sum with a round-to-nearest FADD.
        float tacc[2][NT][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int r = 0; r < 4; ++r) tacc[i][j][r] = 0.f;
#pragma unroll
        for (int kk = 0; kk < NN_BK / 8; ++kk) {
            float af[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float* p = as + (i * 16 + g) * NN_LDA + kk * 8 + t;
                af[i][0] = p[0];
                af[i][1] = p[8 * NN_LDA];
                af[i][2] = p[4];
                af[i][3] = p[8 * NN_LDA + 4];
            }
            uint32_t ah[2][4], al[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if constexpr (X3) {
                    split_tf32<4>(af[i], ah[i], al[i]);
                } else {
#pragma unroll
                    for (int r = 0; r < 4; ++r) ah[i][r] = f2tf32(af[i][r]);
                }
            }
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const float* p = bs + (kk * 8 + t) * LDB + j * 8 + g;
                const float bf[2] = {p[0], p[4 * LDB]};
                uint32_t bh[2], bl[2];
                if constexpr (X3) {
                    split_tf32<2>(bf, bh, bl);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        mma_tf32(tacc[i][j], al[i], bh);
                        mma_tf32(tacc[i][j], ah[i], bl);
                        mma_tf32(tacc[i][j], ah[i], bh);
                    }
                } else {
                    bh[0] = f2tf32(bf[0]);
                    bh[1] = f2tf32(bf[1]);
#pragma unroll
                    for (int i = 0; i < 2; ++i) mma_tf32(tacc[i][j], ah[i], bh);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < NT; ++j)
#pragma unroll
                for (int r = 0; r < 4; ++r) acc[i][j][r] += tacc[i][j][r];
    }
    cp_async_wait<0>();

    // epilogue: bias (+ ReLU); c0,c1 -> (row g, cols 2t,2t+1), c2,c3 -> row g+8
    const bool vec2 = (ldc % 2 == 0) && ((uintptr_t)C % 8 == 0);
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            const int cn = n0 + wn * (BN / 2) + j * 8 + 2 * t;
            float b0 = 0.f, b1 = 0.f;
            if (bias) {
                if (cn < Nc) b0 = __ldg(bias + cn);
                if (cn + 1 < Nc) b1 = __ldg(bias + cn + 1);
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int64_t r = m0 + wm * 32 + i * 16 + g + h * 8;
                if (r >= M) continue;
                float v0 = acc[i][j][2 * h] + b0, v1 = acc[i][j][2 * h + 1] + b1;
                if (epi == GNNML3_EPI_RELU) {
                    v0 = fmaxf(v0, 0.f);
                    v1 = fmaxf(v1, 0.f);
                }
                float* dst = C + r * ldc + cn;
                if (vec2 && cn + 1 < Nc) {
                    *reinterpret_cast<float2*>(dst) = make_float2(v0, v1);
                } else {
                    if (cn < Nc) dst[0] = v0;
                    if (cn + 1 < Nc) dst[1] = v1;
                }
            }
        }
}

// ------------------------------------------------------------------------------------------------ gemm_tn
constexpr int TN_BK = 32, TN_STAGES = 3, TN_THREADS = 128;
template <int BA, int BB>
constexpr size_t tn_smem_bytes() { return sizeof(float) * TN_STAGES * TN_BK * (BA + 8 + BB + 8); }

// BA = 64: 2 x 2 warps of 32 x 32;  BA = 32 (Ka <= 32, e.g. x^T G' with 32 input features): 1 x 4 warps of 32 x 16, so
// no MMA is spent on padding rows of the A^T tile.  BB = 128 with BA = 32 gives every warp a 32 x 32 tile (the A^T fragments
// and their hi/lo split are shared by twice as many MMAs); used when B has at least 128 columns.
template <int BA, int BB, bool VA, bool VB, bool X3>
__global__ void __launch_bounds__(TN_THREADS)
k_gemm_tn(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, float* __restrict__ P,
          int64_t M, int Ka, int Nb, int64_t rows_per_split) {
    constexpr int LDA = BA + 8, TN_BB = BB, TN_LD = BB + 8;
    constexpr int WA = BA / 32, WB = 4 / WA;       // warp grid
    constexpr int NTB = TN_BB / WB / 8;            // n-tiles per warp
    extern __shared__ __align__(16) float smem[];
    float* As = smem;
    float* Bs = smem + TN_STAGES * TN_BK * LDA;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wa = warp % WA, wb = warp / WA;
    const int a0 = blockIdx.x * BA, b0 = blockIdx.y * TN_BB;
    const int64_t mbeg = (int64_t)blockIdx.z * rows_per_split;
    const int64_t mend = min(M, mbeg + rows_per_split);
    const int nk = (int)((mend - mbeg + TN_BK - 1) / TN_BK);

    float acc[2][NTB][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NTB; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[i][j][r] = 0.f;

    auto issue = [&](int kt) {
        const int st = kt % TN_STAGES;
        load_tile<TN_BK, BA, LDA, TN_THREADS, VA>(As + st * TN_BK * LDA, A, lda, mbeg + (int64_t)kt * TN_BK, a0, mend, Ka);
        load_tile<TN_BK, TN_BB, TN_LD, TN_THREADS, VB>(Bs + st * TN_BK * TN_LD, B, ldb, mbeg + (int64_t)kt * TN_BK, b0, mend, Nb);
    };
#pragma unroll
    for (int s = 0; s < TN_STAGES - 1; ++s) {
        if (s < nk) issue(s);
        cp_async_commit();
    }
    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<TN_STAGES - 2>();
        __syncthreads();
        if (kt + TN_STAGES - 1 < nk) issue(kt + TN_STAGES - 1);
        cp_async_commit();
        const float* as = As + (kt % TN_STAGES) * TN_BK * LDA + wa * 32;
        const float* bs = Bs + (kt % TN_STAGES) * TN_BK * TN_LD + wb * (TN_BB / WB);
        // per-k-tile accumulators (see k_gemm_nn); the hi*hi products and the two correction products go to separate
        // accumulators so a tile's three MMAs do not form one dependent chain (4 -> 8 independent chains per warp)
        float tacc[2][NTB][4], tlo[X3 ? 2 : 1][X3 ? NTB : 1][4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < NTB; ++j)
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    tacc[i][j][r] = 0.f;
                    if constexpr (X3) tlo[i][j][r] = 0.f;
                }
#pragma unroll
        for (int kk = 0; kk < TN_BK / 8; ++kk) {
            float af[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {  // A^T fragment: (row = A column, col = node)
                const float* p = as + (kk * 8 + t) * LDA + i * 16 + g;
                af[i][0] = p[0];
                af[i][1] = p[8];
                af[i][2] = p[4 * LDA];
                af[i][3] = p[4 * LDA + 8];
            }
            uint32_t ah[2][4], al[2][4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if constexpr (X3) {
                    split_tf32<4>(af[i], ah[i], al[i]);
                } else {
#pragma unroll
                    for (int r = 0; r < 4; ++r) ah[i][r] = f2tf32(af[i][r]);
                }
            }
#pragma unroll
            for (int j = 0; j < NTB; ++j) {
                const float* p = bs + (kk * 8 + t) * TN_LD + j * 8 + g;
                const float bf[2] = {p[0], p[4 * TN_LD]};
                uint32_t bh[2], bl[2];
                if constexpr (X3) {
                    split_tf32<2>(bf, bh, bl);
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        mma_tf32(tlo[i][j], al[i], bh);
                        mma_tf32(tacc[i][j], ah[i], bh);
                        mma_tf32(tlo[i][j], ah[i], bl);
                    }
                } else {
                    bh[0] = f2tf32(bf[0]);
                    bh[1] = f2tf32(bf[1]);
#pragma unroll
                    for (int i = 0; i < 2; ++i) mma_tf32(tacc[i][j], ah[i], bh);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < NTB; ++j)
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if constexpr (X3) acc[i][j][r] += tacc[i][j][r] + tlo[i][j][r];
                    else acc[i][j][r] += tacc[i][j][r];
                }
    }
    cp_async_wait<0>();
    float* Pz = P + (int64_t)blockIdx.z * Ka * Nb;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < NTB; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int ra = a0 + wa * 32 + i * 16 + g + (r >> 1) * 8;
                const int cb = b0 + wb * (TN_BB / WB) + j * 8 + 2 * t + (r & 1);
                if (ra < Ka && cb < Nb) Pz[(int64_t)ra * Nb + cb] = acc[i][j][r];
            }
}

// Narrow weight gradient (Nb <= 8 columns, Ka <= 64: the tanh-gate columns of ML3Layer, x^T [g11 | g12]).  A 64-column
// tensor-core tile would spend 16x the MMAs on padding; this is a plain FP32 FMA kernel that streams A once: a warp owns
// TNN_ROWS_PER_WARP consecutive rows, lane = A column, the Nb values of the B row are warp-uniform loads.  Partials per CTA
// (8 warps combined in a fixed order) go to the workspace and k_reduce_partials finishes -- deterministic, no atomics.
constexpr int TNN_MAXNB = 8, TNN_ROWS_PER_WARP = 32, TNN_WARPS = 8, TNN_ROWS = TNN_ROWS_PER_WARP * TNN_WARPS;
__global__ void __launch_bounds__(TNN_WARPS * 32)
k_gemm_tn_narrow(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, float* __restrict__ P,
                 int64_t M, int Ka, int Nb) {
    __shared__ float red[TNN_WARPS][2 * 32 * TNN_MAXNB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t r0 = (int64_t)blockIdx.x * TNN_ROWS + warp * TNN_ROWS_PER_WARP;
    const int64_t r1 = min(M, r0 + TNN_ROWS_PER_WARP);
    float acc[2][TNN_MAXNB];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int b = 0; b < TNN_MAXNB; ++b) acc[h][b] = 0.f;
    const bool two = Ka > 32;
    const bool ok0 = lane < Ka, ok1 = lane + 32 < Ka;
    // TNN_UNR rows per iteration, every load issued before the first FMA (in-order issue: a load placed after a dependent
    // FMA would wait a full memory latency per row)
    constexpr int TNN_UNR = 8;
    for (int64_t rr = r0; rr < r1; rr += TNN_UNR) {
        float a0[TNN_UNR], a1[TNN_UNR], bv[TNN_UNR][TNN_MAXNB];
#pragma unroll
        for (int u = 0; u < TNN_UNR; ++u) {
            const int64_t r = rr + u;
            const bool in = r < r1;
            a0[u] = (in && ok0) ? __ldg(A + r * lda + lane) : 0.f;
            a1[u] = (in && two && ok1) ? __ldg(A + r * lda + 32 + lane) : 0.f;
#pragma unroll
            for (int b = 0; b < TNN_MAXNB; ++b) bv[u][b] = (in && b < Nb) ? __ldg(B + r * ldb + b) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < TNN_UNR; ++u)
#pragma unroll
            for (int b = 0; b < TNN_MAXNB; ++b) {
                acc[0][b] = fmaf(a0[u], bv[u][b], acc[0][b]);
                acc[1][b] = fmaf(a1[u], bv[u][b], acc[1][b]);
            }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int b = 0; b < TNN_MAXNB; ++b) red[warp][(h * 32 + lane) * TNN_MAXNB + b] = acc[h][b];
    __syncthreads();
    float* Pz = P + (int64_t)blockIdx.x * Ka * Nb;
    for (int i = threadIdx.x; i < Ka * Nb; i += blockDim.x) {
        const int a = i / Nb, b = i % Nb;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < TNN_WARPS; ++w) v += red[w][a * TNN_MAXNB + b];
        Pz[i] = v;
    }
}
static inline bool tn_narrow(int Ka, int Nb) { return Nb <= TNN_MAXNB && Ka <= 64; }

// tcgen05 path for the big weight gradients (gemm_tn_tc.cu)
bool gemm_tn_tc_shape_ok(int64_t M, int Ka, int Nb);
bool gemm_tn_tc_ok(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int Ka, int Nb);
int gemm_tn_tc_parts(int64_t M);
int gemm_tn_tc_launch(const float* A, int64_t lda, const float* B, int64_t ldb, float* P, int64_t M, int Ka, int Nb, cudaStream_t st);

// C[i] = sum_z P[z][i] in a fixed order: TY split-lanes per output accumulate strided partial sums, then a fixed tree.
// TY = 8 for wide outputs (many blocks); TY = 32 when a few outputs are summed over hundreds of partials (the bias sums and
// the narrow weight gradients: 128 outputs x 740 partials ran as 4 blocks of 92 dependent loads per thread, 16 us)
template <int TY>
__global__ void __launch_bounds__(32 * TY) k_reduce_partials(const float* __restrict__ P, int splits, int64_t n, int cols,
                                                            float* __restrict__ C, int64_t ldc) {
    __shared__ float red[TY][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 32 + tx;
    float s = 0.f;
    if (i < n)
        for (int z = ty; z < splits; z += TY) s += __ldg(P + (int64_t)z * n + i);
    red[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && i < n) {
        float v = 0.f;
#pragma unroll
        for (int y = 0; y < TY; ++y) v += red[y][tx];
        C[(i / cols) * ldc + (i % cols)] = v;
    }
}
static inline void launch_reduce_partials(const float* P, int splits, int64_t n, int cols, float* C, int64_t ldc, cudaStream_t st) {
    const int blocks = cdiv(n, 32);
    if (splits >= 128 && blocks <= 2 * kNumSMs) k_reduce_partials<32><<<blocks, 1024, 0, st>>>(P, splits, n, cols, C, ldc);
    else k_reduce_partials<8><<<blocks, 256, 0, st>>>(P, splits, n, cols, C, ldc);
}

static inline int tn_ba_for(int Ka) { return Ka <= 32 ? 32 : 64; }

static inline int tn_bb_for(int Ka, int Nb) { return (Ka <= 32 && Nb >= 128) ? 128 : 64; }

static void tn_plan(int64_t M, int Ka, int Nb, int* splits, int64_t* rows_per_split) {
    const int tiles = cdiv(Ka, tn_ba_for(Ka)) * cdiv(Nb, tn_bb_for(Ka, Nb));
    int s = (4 * kNumSMs + tiles - 1) / tiles;
    int64_t maxs = (M + 4 * TN_BK - 1) / (4 * TN_BK);
    if (s > maxs) s = (int)maxs;
    if (s < 1) s = 1;
    if (s > 1024) s = 1024;
    int64_t rps = (M + s - 1) / s;
    rps = (rps + TN_BK - 1) / TN_BK * TN_BK;
    *splits = (int)((M + rps - 1) / rps);
    *rows_per_split = rps;
}

// ------------------------------------------------------------------------------------------------ colsum
constexpr int CS_ROWS = 256;
__global__ void __launch_bounds__(256) k_colsum_partial(const float* __restrict__ A, int64_t lda, int64_t M, int Nc,
                                                        float* __restrict__ P) {
    __shared__ float red[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.x * CS_ROWS;
    const int64_t r1 = min(M, r0 + CS_ROWS);
    for (int c0 = 0; c0 < Nc; c0 += 32) {
        const int c = c0 + tx;
        float s = 0.f;
        if (c < Nc)
            for (int64_t r = r0 + ty; r < r1; r += 8) s += __ldg(A + r * lda + c);
        red[ty][tx] = s;
        __syncthreads();
        if (ty == 0 && c < Nc) {
            float v = 0.f;
#pragma unroll
            for (int y = 0; y < 8; ++y) v += red[y][tx];
            P[(int64_t)blockIdx.x * Nc + c] = v;
        }
        __syncthreads();
    }
}

}  // namespace gnnml3

using namespace gnnml3;

template <int BN, bool VA, bool VB, bool X3>
static int launch_nn(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C, int64_t ldc,
                     int64_t M, int Nc, int Kc, int epi, cudaStream_t st) {
    static bool configured[64] = {};
    if (auto once_ = first_use_on_device(configured)) {
        GNNML3_CUDA(cudaFuncSetAttribute(k_gemm_nn<BN, VA, VB, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)nn_smem_bytes<BN>()));
    }
    dim3 grid(cdiv(M, NN_BM), cdiv(Nc, BN));
    k_gemm_nn<BN, VA, VB, X3><<<grid, NN_THREADS, nn_smem_bytes<BN>(), st>>>(A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epi);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

template <int BN, bool X3>
static int launch_nn_v(bool va, bool vb, const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                       int64_t ldc, int64_t M, int Nc, int Kc, int epi, cudaStream_t st) {
    if (va && vb) return launch_nn<BN, true, true, X3>(A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epi, st);
    if (va) return launch_nn<BN, true, false, X3>(A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epi, st);
    if (vb) return launch_nn<BN, false, true, X3>(A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epi, st);
    return launch_nn<BN, false, false, X3>(A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epi, st);
}

extern "C" int gnnml3_gemm_nn(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                              int64_t ldc, int64_t M, int Nc, int Kc, int precision, int epilogue, void* stream_) {
    GNNML3_REQUIRE(M > 0 && Nc > 0 && Kc > 0, "gemm_nn: bad shape M=%lld Nc=%d Kc=%d", (long long)M, Nc, Kc);
    GNNML3_REQUIRE(A && B && C, "gemm_nn: NULL pointer");
    GNNML3_REQUIRE(lda >= Kc && ldb >= Nc && ldc >= Nc, "gemm_nn: leading dimensions too small");
    GNNML3_REQUIRE(prec_valid(precision), "gemm_nn: unknown precision %d", precision);
    GNNML3_REQUIRE(epilogue == GNNML3_EPI_NONE || epilogue == GNNML3_EPI_RELU, "gemm_nn: unknown epilogue %d", epilogue);
    GNNML3_REQUIRE(cdiv(M, NN_BM) > 0 && cdiv(Nc, 32) < 65536, "gemm_nn: grid too large");
    cudaStream_t st = (cudaStream_t)stream_;
    // 128-bit loads need 16-byte aligned rows only (partial vectors at the row tail are zero-filled)
    const bool va = (lda % 4 == 0 || M == 1) && (uintptr_t)A % 16 == 0;
    const bool vb = (ldb % 4 == 0 || Kc == 1) && (uintptr_t)B % 16 == 0;
    const bool x3 = precision == GNNML3_PREC_3XTF32;
    if (Nc > 32) {
        return x3 ? launch_nn_v<64, true>(va, vb, A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epilogue, st)
                  : launch_nn_v<64, false>(va, vb, A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epilogue, st);
    }
    return x3 ? launch_nn_v<32, true>(va, vb, A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epilogue, st)
              : launch_nn_v<32, false>(va, vb, A, lda, B, ldb, bias, C, ldc, M, Nc, Kc, epilogue, st);
}

extern "C" size_t gnnml3_gemm_tn_workspace_bytes(int64_t M, int Ka, int Nb) {
    int splits;
    int64_t rps;
    tn_plan(M > 0 ? M : 1, Ka, Nb, &splits, &rps);
    if (tn_narrow(Ka, Nb)) splits = (int)cdiv(M > 0 ? M : 1, (int64_t)TNN_ROWS);
    if (gemm_tn_tc_shape_ok(M, Ka < 32 ? Ka : 32, Nb) && gemm_tn_tc_parts(M) > splits) splits = gemm_tn_tc_parts(M);
    return align_up((size_t)splits * Ka * Nb * sizeof(float), 256);
}

template <int BA, int BB, bool VA, bool VB, bool X3>
static int launch_tn(const float* A, int64_t lda, const float* B, int64_t ldb, float* P, int64_t M, int Ka, int Nb,
                     int splits, int64_t rps, cudaStream_t st) {
    static bool configured[64] = {};
    if (auto once_ = first_use_on_device(configured)) {
        GNNML3_CUDA(cudaFuncSetAttribute(k_gemm_tn<BA, BB, VA, VB, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tn_smem_bytes<BA, BB>()));
    }
    dim3 grid(cdiv(Ka, BA), cdiv(Nb, BB), splits);
    k_gemm_tn<BA, BB, VA, VB, X3><<<grid, TN_THREADS, tn_smem_bytes<BA, BB>(), st>>>(A, lda, B, ldb, P, M, Ka, Nb, rps);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

template <int BA, int BB, bool X3>
static int launch_tn_v(bool va, bool vb, const float* A, int64_t lda, const float* B, int64_t ldb, float* P, int64_t M, int Ka,
                       int Nb, int splits, int64_t rps, cudaStream_t st) {
    if (va && vb) return launch_tn<BA, BB, true, true, X3>(A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    if (va) return launch_tn<BA, BB, true, false, X3>(A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    if (vb) return launch_tn<BA, BB, false, true, X3>(A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    return launch_tn<BA, BB, false, false, X3>(A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
}

extern "C" int gnnml3_gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int64_t M,
                              int Ka, int Nb, int precision, void* workspace, size_t workspace_bytes, void* stream_) {
    GNNML3_REQUIRE(M > 0 && Ka > 0 && Nb > 0, "gemm_tn: bad shape");
    GNNML3_REQUIRE(A && B && C && workspace, "gemm_tn: NULL pointer");
    GNNML3_REQUIRE(lda >= Ka && ldb >= Nb && ldc >= Nb, "gemm_tn: leading dimensions too small");
    GNNML3_REQUIRE(prec_valid(precision), "gemm_tn: unknown precision %d", precision);
    GNNML3_REQUIRE(cdiv(Nb, 64) < 65536, "gemm_tn: grid too large");
    if (workspace_bytes < gnnml3_gemm_tn_workspace_bytes(M, Ka, Nb))
        return set_err(GNNML3_ERR_WORKSPACE, "gemm_tn: workspace %zu < %zu bytes", workspace_bytes,
                       gnnml3_gemm_tn_workspace_bytes(M, Ka, Nb));
    int splits;
    int64_t rps;
    tn_plan(M, Ka, Nb, &splits, &rps);
    cudaStream_t st = (cudaStream_t)stream_;
    const bool va = (lda % 4 == 0 || M == 1) && (uintptr_t)A % 16 == 0;
    const bool vb = (ldb % 4 == 0 || M == 1) && (uintptr_t)B % 16 == 0;
    float* P = (float*)workspace;
    int rc;
    if (tn_narrow(Ka, Nb)) {   // exact FP32 FMAs: at least as accurate as any requested precision
        const int64_t nblk = cdiv(M, (int64_t)TNN_ROWS);
        GNNML3_REQUIRE(nblk < (int64_t)1 << 31, "gemm_tn: too many rows");
        k_gemm_tn_narrow<<<(unsigned)nblk, TNN_WARPS * 32, 0, st>>>(A, lda, B, ldb, P, M, Ka, Nb);
        GNNML3_LAUNCH_CHECK();
        const int64_t n = (int64_t)Ka * Nb;
        launch_reduce_partials(P, (int)nblk, n, Nb, C, ldc, st);
        GNNML3_LAUNCH_CHECK();
        return GNNML3_OK;
    }
    const bool x3 = precision == GNNML3_PREC_3XTF32;
    static const bool no_tc = getenv("GNNML3_NO_TN_TC") != nullptr;
    if (x3 && !no_tc && gemm_tn_tc_ok(A, lda, B, ldb, M, Ka < 32 ? Ka : 32, Nb)) {
        // 32 columns of A (the M side of the instruction: [x_hi; x_lo] = 64 lanes) x 256 columns of B (one TMEM accumulator set)
        // per launch; the partial buffer is reused, launches are stream-ordered.  Wide A (the F = 64..256 sweep) re-reads B once
        // per 32-column block of A -- still less time than the mma.sync kernel (F = 64: 1.3 vs 2.1 ms per 1 M rows x 640 columns).
        for (int a0 = 0; a0 < Ka; a0 += 32) {
            const int kac = Ka - a0 < 32 ? Ka - a0 : 32;
            for (int c0 = 0; c0 < Nb; c0 += 256) {
                const int nbc = Nb - c0 < 256 ? Nb - c0 : 256;
                if ((rc = gemm_tn_tc_launch(A + a0, lda, B + c0, ldb, P, M, kac, nbc, st))) return rc;
                const int64_t n = (int64_t)kac * nbc;
                launch_reduce_partials(P, gemm_tn_tc_parts(M), n, nbc, C + (int64_t)a0 * ldc + c0, ldc, st);
                GNNML3_LAUNCH_CHECK();
            }
        }
        return GNNML3_OK;
    }
    if (tn_ba_for(Ka) == 32 && tn_bb_for(Ka, Nb) == 128)
        rc = x3 ? launch_tn_v<32, 128, true>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st)
                : launch_tn_v<32, 128, false>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    else if (tn_ba_for(Ka) == 32)
        rc = x3 ? launch_tn_v<32, 64, true>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st)
                : launch_tn_v<32, 64, false>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    else
        rc = x3 ? launch_tn_v<64, 64, true>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st)
                : launch_tn_v<64, 64, false>(va, vb, A, lda, B, ldb, P, M, Ka, Nb, splits, rps, st);
    if (rc) return rc;
    const int64_t n = (int64_t)Ka * Nb;
    launch_reduce_partials(P, splits, n, Nb, C, ldc, st);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

extern "C" size_t gnnml3_colsum_workspace_bytes(int64_t M, int Nc) {
    return align_up((size_t)cdiv(M > 0 ? M : 1, CS_ROWS) * Nc * sizeof(float), 256);
}

extern "C" int gnnml3_colsum(const float* A, int64_t lda, int64_t M, int Nc, float* out, void* workspace,
                             size_t workspace_bytes, void* stream_) {
    GNNML3_REQUIRE(M > 0 && Nc > 0 && A && out && workspace && lda >= Nc, "colsum: bad arguments");
    if (workspace_bytes < gnnml3_colsum_workspace_bytes(M, Nc))
        return set_err(GNNML3_ERR_WORKSPACE, "colsum: workspace too small");
    cudaStream_t st = (cudaStream_t)stream_;
    const int nb = cdiv(M, CS_ROWS);
    k_colsum_partial<<<nb, 256, 0, st>>>(A, lda, M, Nc, (float*)workspace);
    GNNML3_LAUNCH_CHECK();
    launch_reduce_partials((const float*)workspace, nb, Nc, Nc, out, Nc, st);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}
