/*
 * gnnml3_b200.h -- C ABI of the B200-native GNNML3 hot path (libgnnml3_b200.so, sm_100a only).
 *
 * Drop-in boundary for the hot path of balcilar/gnn-matlang (citations relative to the reference root):
 *   libs/spect_conv.py:64-99   SpectConv.forward / message   (+ PyG MessagePassing.propagate, aggr='add')
 *   libs/spect_conv.py:204-212 ML3Layer.forward              (edge MLP, tanh*tanh gating, concat)
 *   libs/utils.py:546-610      SpectralDesign.__call__       (supports M .* U f_k(L) U^T as edge features)
 *   PyG global_add_pool / global_mean_pool (graph8c.py:277, Zinc12k.py:343, exp_classify.py:293, counting.py:370)
 *   PyG Batch.from_data_list collation of edge_index2 (Zinc12k.py:20-22 etc.)
 * The reference is pure Python and has no FFI; the binding a maintainer would add is the ctypes stub shown
 * in INTEGRATION.md (and implemented in gnn_matlang_b200/_lib.py).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  Unless a parameter name ends in `_host`, every
 *     pointer is a DEVICE pointer valid on the current CUDA device.
 *   - all matrices are row-major FP32, indices are int32 inside the library; the reference's int64
 *     edge_index [2,E] (row 0 = source j, row 1 = target i) is accepted by gnnml3_csr_build.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Nothing synchronises the
 *     device except the *_host entry points and functions documented to do so; everything else is
 *     CUDA-graph capturable.
 *   - return value: 0 = success, otherwise one of GNNML3_ERR_*; gnnml3_last_error() returns a
 *     thread-local human-readable message.  There is no CPU fallback anywhere in this library.
 *   - determinism: no floating-point atomics; every reduction has a fixed order.
 */
#ifndef GNNML3_B200_H_
#define GNNML3_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GNNML3_API __attribute__((visibility("default")))
#else
#define GNNML3_API
#endif

#define GNNML3_OK 0
#define GNNML3_ERR_INVALID 1     /* bad argument (shape, alignment, NULL, unsupported size) */
#define GNNML3_ERR_CUDA 2        /* a CUDA runtime call or kernel launch failed */
#define GNNML3_ERR_WORKSPACE 3   /* workspace too small */

/* GEMM arithmetic: FP32-grade error-compensated 3xTF32 (default, meets rtol 1e-5), single-pass TF32.  BF16 inputs with FP32
 * accumulation: the GNNML1 layer (gnnml3_ml1layer_*_precision); the stand-alone GEMMs take it as single-pass TF32. */
#define GNNML3_PREC_3XTF32 0
#define GNNML3_PREC_TF32 1
#define GNNML3_PREC_BF16 2

/* precision flags OR-ed into the `epilogue` argument of gnnml3_fused_agg_proj (tensor-memory kernel only): one tensor-core
 * product per k-step on TF32-truncated / BF16-rounded inputs instead of the FP32-grade 3xTF32 triple; FP32 accumulation.
 * Stated tolerances (tests/test_gpu_fused.py): TF32 2e-3, BF16 2e-2 of the result's scale. */
#define GNNML3_FUSED_TF32 0x100
#define GNNML3_FUSED_BF16 0x200

/* epilogues of gnnml3_gemm_nn */
#define GNNML3_EPI_NONE 0
#define GNNML3_EPI_RELU 1

GNNML3_API const char* gnnml3_last_error(void);
GNNML3_API int gnnml3_version(void);
/* number of kernels launched by this library in the calling process so far (for bench.py's gpu_launches) */
GNNML3_API int64_t gnnml3_launch_count(void);

/* ---------------------------------------------------------------------------------------------------
 * Graph structure: dst-sorted CSR + src-sorted (transposed) CSR of the batched disjoint graph.
 * Replaces the index_select / scatter_add indexing of PyG propagate (libs/spect_conv.py:77) and is
 * bit-exact integer work: within a row, entries keep the original edge order (stable).
 *   rowptr [N+1], col [E] (= source of the p-th dst-sorted edge), perm [E] (= original edge id of p)
 *   rowptrT [N+1], colT [E] (= target of the q-th src-sorted edge), permT [E] (= dst-sorted position p of q)
 * err_flag (device int32, may be NULL) is set to 1 if any index is outside [0, N).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API size_t gnnml3_csr_workspace_bytes(int64_t E, int64_t N);
GNNML3_API int gnnml3_csr_build(const int64_t* edge_index, int64_t E, int64_t N,
                     int32_t* rowptr, int32_t* col, int32_t* perm,
                     int32_t* rowptrT, int32_t* colT, int32_t* permT,
                     int32_t* err_flag, void* workspace, size_t workspace_bytes, void* stream);

/* out[p, :] = in[perm[p], :]  (gather) and out[perm[p], :] = in[p, :] (scatter); rows of `width` floats */
GNNML3_API int gnnml3_gather_rows(const float* in, const int32_t* perm, int64_t rows, int width, float* out, void* stream);
GNNML3_API int gnnml3_scatter_rows(const float* in, const int32_t* perm, int64_t rows, int width, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * K-channel segmented reduction (the aggregate of SpectConv, libs/spect_conv.py:76-77,98-99):
 *   out[t, k*F + f] = sum_{p in [rowptr[t], rowptr[t+1])} ea[e(p), k] * x[col[p], f],  e(p) = eperm ? eperm[p] : p
 * x [N, F] (ldx floats per row), ea [E, K] row-major, out [N, ldo] with ldo >= K*F.  Atomic-free, summation
 * in row order.  Used forward with the dst-sorted CSR and backward (on grad_out) with the transposed CSR.
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_spmm_k(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea,
                  const float* x, int64_t ldx, int64_t N, int K, int F, float* out, int64_t ldo, void* stream);

/* Project-first order of SpectConv (the sum over supports moved inside the edge sum; libs/spect_conv.py:70-80):
 *   out[t, f] = sum_{p in row t} sum_k ea[e(p), k] * Y[col[p], k*Fo + f]  (+ bias[f]),   Y = x [W_0 .. W_{K-1}]  ([N, K*Fo])
 * Gathers K*Fo floats per support entry instead of F_in: chosen when the layer narrows (DESIGN.md section 4.5). */
GNNML3_API int gnnml3_spmm_projected(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea, int K,
                          const float* Y, int64_t ldy, int64_t N, int Fo, const float* bias, float* out, int64_t ldo, void* stream);

/* d ea[e(p), k] = < x[col[p], :], g[t, k*F : (k+1)*F] >  for every edge p of every row t (SDDMM). */
GNNML3_API int gnnml3_sddmm_k(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* x, int64_t ldx,
                   const float* g, int64_t ldg, int64_t N, int K, int F, float* dea, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Tensor-core contractions (mma TF32 with FP32 accumulate; 3xTF32 split for FP32-grade results).
 *   gemm_nn: C[M, Nc] = A[M, Kc] * B[Kc, Nc] (+ bias[Nc]) (+ epilogue)     -- projection  H * W
 *   gemm_tn: C[Ka, Nb] = A[M, Ka]^T * B[M, Nb]                              -- weight gradient, fixed-order split-M
 *            (Ka <= 32, 8 < Nb <= 256, M >= 8192, 16-byte aligned rows: tcgen05 with MN-major operands fed by TMA;
 *             Nb <= 8: FP32 FMA kernel; otherwise mma.sync.  Same result contract on every path: deterministic,
 *             FP32-grade with GNNML3_PREC_3XTF32.  GNNML3_NO_TN_TC=1 in the environment disables the tcgen05 path.)
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_gemm_nn(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias,
                   float* C, int64_t ldc, int64_t M, int Nc, int Kc, int precision, int epilogue, void* stream);
GNNML3_API size_t gnnml3_gemm_tn_workspace_bytes(int64_t M, int Ka, int Nb);
GNNML3_API int gnnml3_gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                   int64_t M, int Ka, int Nb, int precision, void* workspace, size_t workspace_bytes, void* stream);
/* out[c] = sum_r A[r, c]  (bias gradient), fixed order */
GNNML3_API size_t gnnml3_colsum_workspace_bytes(int64_t M, int Nc);
GNNML3_API int gnnml3_colsum(const float* A, int64_t lda, int64_t M, int Nc, float* out, void* workspace,
                  size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused per-edge MLP of ML3Layer (libs/spect_conv.py:191-194,206-207):
 *   out[p, :] = relu(W4 [relu(W1 a) || tanh(W2 a) * tanh(W3 a)]),  a = ea[e(p), :],  e(p) = eperm ? eperm[p] : p
 * W1,W2,W3 [2K, K], W4 [Kout, 4K] are the nn.Linear.weight tensors (bias-free).  Instantiated for even
 * K <= 16 with Kout == K (gnnml3_edge_mlp_supported); other shapes are composed from gnnml3_gemm_*.
 * bwd recomputes the activations; dea (nullable) receives d ea at e(p); dw1..dw4 are overwritten.
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_edge_mlp_supported(int K, int Kout);
/* Two generations of the same contract: tcgen05 (default: edges on the tensor-memory lanes, weights as shared-memory planes,
 * 3xTF32 FP32-grade) and the FP32-FMA kernels of round 1.  set_tc(0/1) selects (returns the old value; GNNML3_EDGE_TC=0 in the
 * environment does the same at load time); path_counts reports {tensor-core, CUDA-core} calls since the last reset. */
GNNML3_API int gnnml3_edge_mlp_set_tc(int enable);
GNNML3_API int gnnml3_edge_mlp_path_counts(long long* out2_host, int reset);
GNNML3_API int gnnml3_edge_mlp_fwd(const float* ea, const int32_t* eperm, const float* w1, const float* w2, const float* w3,
                        const float* w4, int64_t E, int K, int Kout, float* out, void* stream);
GNNML3_API size_t gnnml3_edge_mlp_bwd_workspace_bytes(int64_t E, int K);
GNNML3_API int gnnml3_edge_mlp_bwd(const float* ea, const int32_t* eperm, const float* gout, const float* w1, const float* w2,
                        const float* w3, const float* w4, int64_t E, int K, int Kout, float* dea, float* dw1,
                        float* dw2, float* dw3, float* dw4, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Node-side epilogue of ML3Layer (libs/spect_conv.py:209-212) on pre = [c | p1 | p2]  ([N, Fo + 2G]):
 *   y = [relu(c) || tanh(p1) * tanh(p2)]  ([N, Fo + G]);  bwd gives d pre (and optionally a second copy of its
 *   2G gate columns into gate_out, row stride ldgate).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_ml3_act_fwd(const float* pre, int64_t ldp, int64_t N, int Fo, int G, float* y, int64_t ldy, void* stream);
GNNML3_API size_t gnnml3_ml3_act_bwd_workspace_bytes(int64_t N, int Fo, int G);
/* colsum (nullable, [Fo + 2G]) receives the column sums of d pre = the bias gradients (needs workspace) */
GNNML3_API int gnnml3_ml3_act_bwd(const float* pre, int64_t ldp, const float* gy, int64_t ldy, int64_t N, int Fo, int G,
                       float* gpre, int64_t ldg, float* gate_out, int64_t ldgate, float* colsum,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Same gradient from the outputs of gnnml3_fused_agg_proj (ReLU mask = y > 0, aux = [tanh(p1) | tanh(p2)]).  gpre layout:
 * conv gradient in columns [0, Fo), zeros to Fo4 = ceil4(Fo), gate gradients [g1 | g2] in [Fo4, Fo4 + 2G), zeros up to ldg --
 * the 16-byte aligned blocks the fused dx kernel gathers.  colsum in the logical order [conv | g1 | g2]. */
GNNML3_API int gnnml3_ml3_act_bwd_y(const float* y, int64_t ldy, const float* aux, int64_t ldaux, const float* gy, int64_t ldgy,
                         int64_t N, int Fo, int G, float* gpre, int64_t ldg, float* colsum,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused aggregate + project on tcgen05 / TMEM (fused_layer.cu): for every row t of the CSR
 *   main[t, :] = sum_k ( sum_{p in row t} ea[e(p), k] * X[col[p], :] ) Bmain[k*F:(k+1)*F, :]   (+ bias)
 * without materialising the [N, K*F] aggregate (libs/spect_conv.py:70-80,93-94).  Optional self block S [N, Fs]:
 *   self_mode 1: own output columns  s[t, :] = S[t, :] Bself [Fs, Ns = 2G] (+ bias_s)  -- with epilogue 1 this is the whole
 *                ML3Layer node branch (:208-212): out[t] = [relu(main) || tanh(s[:G]) * tanh(s[G:])], aux[t] = tanh(s);
 *                aux may be NULL (inference: nothing is saved for a backward): a forward-only kernel then stores out alone;
 *   self_mode 2: main[t, :] += S[t, :] Bself [Fs, Nc]  (SpectConv selfconn; gate gradients in the dx pass).
 * epilogue 0: out [N, Nc] = main.  X and S rows must be 16-byte aligned (ld % 4 == 0) and every column below
 * ceil4(F) / ceil4(Fs) must hold finite values.  3xTF32 arithmetic (FP32-grade).  Backward dx = the same call over the
 * transposed CSR with X = d pre, Bmain = W_k^T.  hout (nullable, [N, ldh]) receives a copy of the aggregate: support k in
 * columns [k * Fp, k * Fp + F) with Fp = 32 * ceil(F / 32) (zero padded), the self block S behind them at K * Fp (32 columns) --
 * the operand of the weight-gradient contraction x^T [S_0^T g .. S_{K-1}^T g | g1 g2], so the backward needs no separate SpMM.
 * --------------------------------------------------------------------------------------------------- */
/* debugging aid: cycle counters of the fused kernel's warp roles (all zero unless GNNML3_FUSED_DEBUG=1); synchronises */
GNNML3_API int gnnml3_fused_debug_counters(unsigned long long* out8_host, int reset);
/* aggregator mode of gnnml3_fused_agg_proj: 0 (default) gathers from global memory with the weight planes resident in shared
 * memory, 1 prefetches every warp's next tile into shared-memory slots with cp.async; returns the previous mode */
GNNML3_API int gnnml3_fused_set_mode(int slot_mode);
/* measurement aid (bench.py roofline): CUDA events on the launching stream around every fused launch while enabled;
 * fetch synchronises and writes [n][10] doubles: ms, N, K, F, Nc, Fs, self_mode, Ns, G, has_perm */
GNNML3_API int gnnml3_fused_profile(int enable);
GNNML3_API int gnnml3_fused_profile_fetch(double* out, int max_records);
GNNML3_API int gnnml3_fused_supported(int K, int Kstride, int F, int Nc, int Fs, int self_mode, int Ns);
GNNML3_API size_t gnnml3_fused_workspace_bytes(int K, int F, int Nc, int self_mode);
GNNML3_API int gnnml3_fused_agg_proj(const int32_t* rowptr, const int32_t* col, const int32_t* eperm, const float* ea,
                          int Kstride, int K, const float* X, int64_t ldx, int F, const float* S, int64_t lds,
                          int Fs, int self_mode, const float* Bmain, int64_t ldb, const float* Bself,
                          int64_t ldbs, int Ns, const float* bias, const float* bias_s, int64_t N, int Nc,
                          float* out, int64_t ldo, float* aux, int64_t ldaux, int G, int epilogue,
                          float* hout, int64_t ldh, const int32_t* tilewin, void* workspace, size_t workspace_bytes,
                          void* stream);
/* Second generation of the same kernel (fused_layer_ts.cu), taken automatically when the shape allows (F <= 32, even K):
 * the aggregate is handed to the tensor core through TENSOR MEMORY (tcgen05.st + A-in-TMEM tcgen05.mma) and the gathered
 * rows are staged in shared memory by one TMA box load per tile.  `tilewin` (nullable) = gnnml3_tile_windows() of the SAME
 * CSR: [ceil(N / gnnml3_tile_rows())][2] int32 {first, last + 1} source row of each tile's slots; tiles whose window has
 * at most 256 rows read their sources from shared memory, the others (and tilewin == NULL) gather from global memory.
 * gnnml3_fused_set_ts(0) forces the first-generation kernel; gnnml3_fused_path_counts reports which kernel ran
 * ([0] tensor-memory, [1] shared-memory planes) since the last reset. */
GNNML3_API int gnnml3_tile_rows(void);
GNNML3_API int gnnml3_tile_windows(const int32_t* rowptr, const int32_t* col, int64_t N, int32_t* win, void* stream);
GNNML3_API int gnnml3_fused_ts_supported(int K, int Kstride, int F, int Nc, int Fs, int self_mode, int Ns);
GNNML3_API size_t gnnml3_fused_ts_workspace_bytes(int K, int Nc, int self_mode);
GNNML3_API int gnnml3_fused_set_ts(int enable);
GNNML3_API int gnnml3_fused_path_counts(long long* out2_host, int reset);

/* ---------------------------------------------------------------------------------------------------
 * Fused edge-feature gradient (fused_sddmm.cu):  dea[p, k] = < X[col[p], :], GC[t, :] W[k]^T >  for every CSR slot p of
 * every row t -- the gradient of SpectConv w.r.t. edge_attr (autograd through libs/spect_conv.py:76-80) without
 * materialising dH = GC [W_0^T .. W_{K-1}^T] in HBM: per tile of 64 rows the dH tile is produced by tcgen05 MMAs
 * (3xTF32) into tensor memory, transposed into shared memory and consumed by the SDDMM warps.  W [K, Fi, Fo] contiguous;
 * X / GC rows 16-byte aligned; dea [E, K] in CSR slot order.  Supported: even K <= 8, Fi <= 32, Fo <= 32.
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_fused_sddmm_supported(int K, int Fi, int Fo);
GNNML3_API size_t gnnml3_fused_sddmm_workspace_bytes(int K);
/* win (nullable): per-128-row-tile source windows of (rowptr, col) from gnnml3_tile_windows -- with them the source rows of a
 * tile are staged in shared memory by one TMA box load (batched disjoint graphs); without, every edge gathers from global memory. */
GNNML3_API int gnnml3_fused_sddmm(const int32_t* rowptr, const int32_t* col, const int32_t* win, const float* X, int64_t ldx, int Fi,
                       const float* GC, int64_t ldg, int Fo, const float* W, int K, int64_t N, float* dea, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Whole-layer entry points (layer_api.cu): ONE call enqueues every kernel of an ML3Layer forward
 * (libs/spect_conv.py:204-212: edge MLP -> SpectConv -> ReLU || tanh*tanh gates) or of its backward, on a caller-provided
 * workspace (gnnml3_ml3layer_workspace_bytes).  Same kernels and arithmetic as composing the single-kernel entry points;
 * the point is the host cost (one call instead of ~30 small operations per layer and direction).
 *   forward : ea_s [E,K] dst-sorted edge features; w1..w4 = fc1_1..fc1_4.weight (NULL: learnedge = False, ea2 unused);
 *             wconv [K,Fi,Fo], bconv [Fo] (nullable); w11,b11,w12,b12 = fc11/fc12 (NULL iff G == 0);
 *             outputs ea2 [E,K], y [N, ldy >= Fo+G], aux [N, 2G] (tanh factors, saved for the backward).  aux == NULL
 *             (with hside == NULL: an inference forward) stores y alone, through the forward-only instantiation of the fused
 *             kernel; the backward still requires aux.
 *   backward: gy [N, ldgy]; outputs dx [N, lddx] (if need_dx), dea [E,K] (if need_dea), dw1..dw4, dwconv [K,Fi,Fo],
 *             dbias [Fo + 2G] = (d bconv | d b11 | d b12), dw11/dw12 [G,Fi].
 *   hside   : optional [N, ldh >= (K [+1 if G > 0]) * 32] (nullable, Fi <= 32).  The forward leaves the aggregate
 *             H = [S_0 x .. S_{K-1} x] there (support k at column 32 k); a backward that gets it and does not need dx (the first
 *             layer of a model) takes the weight gradient as dW_k = H_k^T gc in one contraction instead of aggregating
 *             S_k^T gc over the transposed CSR first.  Pass NULL to both for the plain behaviour.
 * x rows must be 16-byte aligned (ldx % 4 == 0).  gnnml3_ml3layer_supported tells whether a shape is covered.
 * win / winT (nullable) = gnnml3_tile_windows of the dst-sorted / transposed CSR (see gnnml3_fused_agg_proj).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_ml3layer_supported(int K, int Fi, int Fo, int G, int learnedge);
GNNML3_API size_t gnnml3_ml3layer_workspace_bytes(int64_t N, int64_t E, int K, int Fi, int Fo, int G);
GNNML3_API int gnnml3_ml3layer_forward(const int32_t* rowptr, const int32_t* col, const int32_t* win, int64_t N, int64_t E, const float* x, int64_t ldx,
                            int Fi, const float* ea_s, int K, const float* w1, const float* w2, const float* w3,
                            const float* w4, const float* wconv, const float* bconv, int Fo, const float* w11,
                            const float* b11, const float* w12, const float* b12, int G, float* ea2, float* y,
                            int64_t ldy, float* aux, float* hside, int64_t ldh, void* workspace, size_t workspace_bytes, void* stream);
GNNML3_API int gnnml3_ml3layer_backward(const int32_t* rowptr, const int32_t* col, const int32_t* win, const int32_t* rowptrT,
                             const int32_t* colT, const int32_t* permT, const int32_t* winT, int64_t N, int64_t E, const float* x, int64_t ldx, int Fi,
                             const float* ea_s, const float* ea2, int K, const float* w1, const float* w2, const float* w3,
                             const float* w4, const float* wconv, int Fo, const float* w11, const float* w12, int G,
                             const float* y, int64_t ldy, const float* aux, const float* gy, int64_t ldgy, int need_dx,
                             int need_dea, float* dx, int64_t lddx, float* dea, float* dw1, float* dw2, float* dw3,
                             float* dw4, float* dwconv, float* dbias, float* dw11, float* dw12, const float* hside, int64_t ldh,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Whole-layer entry points of GNNML1, the paper's 1-WL model (ml1_layer.cu).  With A the adjacency of the plain edge_index
 * ((A x)[t] = sum of x[s] over the edges s -> t; every edge weight is one and none is read), wconv [1, Fi, Fo] / bconv [Fo]
 * (SpectConv(Fi, Fo, K=1, selfconn=False)) and the nn.Linear(Fi, Fo) weights wA, wB, wC [Fo, Fi] with biases bA, bB, bC:
 *   p0 = x wA^T + bA + (A x) wconv[0] + bconv,   p1 = x wB^T + bB,   p2 = x wC^T + bC
 *   concat = 0: y = relu(p0 + p1 * p2)                                                        [N, Fo]
 *   concat = 1: y = [relu(x wA^T + bA) | relu((A x) wconv[0] + bconv) | relu(p1 * p2)]         [N, 3 Fo]
 * One fused kernel per direction: the aggregate and the four projections meet in tensor memory (tcgen05, 3xTF32, FP32-grade).
 * The *_precision entry points take the same arguments plus the projection's arithmetic: GNNML3_PREC_3XTF32 (what the plain
 * entry points run), GNNML3_PREC_TF32 (one MMA per k-step on the raw FP32 operand, truncated by the tensor core, and RN-TF32
 * weights) or GNNML3_PREC_BF16 (RN-BF16 operands and weights); anything else is GNNML3_ERR_INVALID.  In every mode the
 * aggregation (FP32 sums in CSR order), the epilogues, y / aux / dx (float32) and determinism are unchanged; the weight
 * gradient contraction runs at GNNML3_PREC_TF32 in both flagged modes.  Stated tolerances (tests/test_gpu_gnnml1_precision.py):
 * TF32 2e-3, BF16 2e-2 of the result's scale.
 *   forward : rowptr / col = the dst-sorted CSR of edge_index (gnnml3_csr_build); outputs y [N, ldy] and aux [N, ldaux >= 2 Fo]
 *             = [p1 | p2] (saved for the backward); hside (nullable, [N, ldh >= Fi]) receives A x.  Biases are nullable.
 *             aux may be NULL (inference): a forward-only instantiation of the kernel then stores y alone (a third of the
 *             sum-mode stores).  The backward requires the aux of a forward that wrote it.
 *   backward: rowptrT / colT = the transposed CSR; gy [N, ldgy]; dx [N, lddx] if need_dx (else dx may be NULL: the aggregate
 *             A^T gc is still formed for d wconv); outputs the eight parameter gradients (dw* overwritten; db* nullable).
 * Supported: 1 <= Fi <= 64, 1 <= Fo <= 64 (gnnml3_ml1layer_supported) in every precision, E = 0 allowed; x rows 16-byte
 * aligned (ldx % 4 == 0).  Deterministic (fixed summation order, no atomics), no host sync; caller-provided workspace
 * (gnnml3_ml1layer_workspace_bytes covers every precision).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_ml1layer_supported(int Fi, int Fo, int concat);
GNNML3_API size_t gnnml3_ml1layer_workspace_bytes(int64_t N, int Fi, int Fo, int concat);
GNNML3_API int gnnml3_ml1layer_forward(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E, const float* x, int64_t ldx,
                            int Fi, const float* wconv, const float* bconv, const float* wA, const float* bA, const float* wB,
                            const float* bB, const float* wC, const float* bC, int Fo, int concat, float* y, int64_t ldy,
                            float* aux, int64_t ldaux, float* hside, int64_t ldh, void* workspace, size_t workspace_bytes,
                            void* stream);
GNNML3_API int gnnml3_ml1layer_backward(const int32_t* rowptrT, const int32_t* colT, int64_t N, int64_t E, const float* x, int64_t ldx,
                             int Fi, const float* wconv, const float* wA, const float* wB, const float* wC, int Fo, int concat,
                             const float* y, int64_t ldy, const float* aux, int64_t ldaux, const float* gy, int64_t ldgy,
                             int need_dx, float* dx, int64_t lddx, float* dwconv, float* dbconv, float* dwA, float* dbA,
                             float* dwB, float* dbB, float* dwC, float* dbC, void* workspace, size_t workspace_bytes,
                             void* stream);
GNNML3_API int gnnml3_ml1layer_forward_precision(const int32_t* rowptr, const int32_t* col, int64_t N, int64_t E, const float* x,
                            int64_t ldx, int Fi, const float* wconv, const float* bconv, const float* wA, const float* bA,
                            const float* wB, const float* bB, const float* wC, const float* bC, int Fo, int concat, float* y,
                            int64_t ldy, float* aux, int64_t ldaux, float* hside, int64_t ldh, void* workspace,
                            size_t workspace_bytes, void* stream, int precision);
GNNML3_API int gnnml3_ml1layer_backward_precision(const int32_t* rowptrT, const int32_t* colT, int64_t N, int64_t E, const float* x,
                             int64_t ldx, int Fi, const float* wconv, const float* wA, const float* wB, const float* wC, int Fo,
                             int concat, const float* y, int64_t ldy, const float* aux, int64_t ldaux, const float* gy,
                             int64_t ldgy, int need_dx, float* dx, int64_t lddx, float* dwconv, float* dbconv, float* dwA,
                             float* dbA, float* dwB, float* dbB, float* dwC, float* dbC, void* workspace, size_t workspace_bytes,
                             void* stream, int precision);

/* ---------------------------------------------------------------------------------------------------
 * Readout: PyG global_add_pool (mean = 0) / global_mean_pool (mean = 1) over contiguous node ranges
 * graph_ptr [B+1] (graph b owns nodes graph_ptr[b] .. graph_ptr[b+1]-1, as produced by batching).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_segment_pool_fwd(const float* x, int64_t ldx, const int32_t* graph_ptr, int B, int F, int mean,
                            float* out, void* stream);
GNNML3_API int gnnml3_segment_pool_bwd(const float* gout, const int32_t* graph_ptr, int B, int F, int mean, float* gx,
                            int64_t ldx, void* stream);
/* PyG global_max_pool (read-out of the GNNML3 variants, enzymes.py:340,384): out [B,F] = per-graph maximum, arg [B,F] = the
 * node attaining it (first on ties; -1 and 0 for an empty graph); bwd routes gout to that node and writes zeros elsewhere. */
GNNML3_API int gnnml3_segment_max_fwd(const float* x, int64_t ldx, const int32_t* graph_ptr, int B, int F, float* out, int32_t* arg,
                           void* stream);
GNNML3_API int gnnml3_segment_max_bwd(const float* gout, const int32_t* arg, const int32_t* graph_ptr, int B, int F, float* gx,
                           int64_t ldx, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * SpectralDesign (libs/utils.py:525-610), batched: one thread block per graph, FP64 Jacobi eigensolver.
 * Input graphs are given as concatenated LOCAL edge lists: edge_index [2, Etot] int64 (row 0 = src, row 1 = dst,
 * node ids local to their graph), edge_ptr [B+1], node_ptr [B+1] (int32).  nmax = largest node count.
 *   gnnml3_spectral_count : counts[b] = number of mask entries of graph b (to size the output)
 *   gnnml3_spectral_design: writes, in the reference's row-major np.where order and at offset out_ptr[b]
 *       (int64 exclusive scan of counts), edge_index2 [2, E2] int64 (+ node_ptr[b] if global_ids) and
 *       edge_attr2 [E2, nfreq + 1 (+1 if addadj)] FP32; lmax [B] (max Laplacian eigenvalue, :586) and
 *       degree [Ntot] (column sums of A, the adddegree feature, :562-563) are optional (NULL to skip).
 *   recfield 0 -> mask A; r >= 1 -> (A + I)^(2^(r-1)) > 0.  has_vmax = 0 -> vmax = largest eigenvalue.
 *   gnnml3_spectral_max_nodes(nfreq): largest graph the shared-memory eigensolver holds (~118).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_spectral_max_nodes(int nfreq);
GNNML3_API int gnnml3_spectral_count(const int64_t* edge_index, int64_t Etot, const int32_t* edge_ptr, const int32_t* node_ptr,
                          int B, int recfield, int nmax, int32_t* counts, void* stream);
GNNML3_API int gnnml3_spectral_design(const int64_t* edge_index, int64_t Etot, const int32_t* edge_ptr, const int32_t* node_ptr,
                           int B, int recfield, double dv, int nfreq, int laplacien, int addadj, int has_vmax,
                           double vmax, int nmax, const int64_t* out_ptr, int global_ids, int64_t* edge_index2,
                           int64_t E2, float* edge_attr2, float* lmax, float* degree, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Blackwell tensor-core path of gemm_nn: tcgen05.mma kind::tf32 with TMEM accumulators, 3xTF32 split,
 * persistent warp-specialised CTAs (csrc/gemm_tc.cu).  Same contract as gnnml3_gemm_nn (FP32-grade result);
 * requires 16-byte aligned rows of A (lda % 4 == 0).  chunk_kblocks = number of 32-wide k-blocks accumulated
 * inside the tensor core before the partial sum is folded into FP32 registers (0 = default 4).
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_gemm_nn_tc_supported(int64_t lda, int Nc, int Kc);
GNNML3_API size_t gnnml3_gemm_nn_tc_workspace_bytes(int Nc, int Kc);
GNNML3_API int gnnml3_gemm_nn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                      int64_t ldc, int64_t M, int Nc, int Kc, int epilogue, int chunk_kblocks, void* workspace,
                      size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Batching on the device (collate.cu): per-graph records -> one disjoint-union batch with the reference's attributes -- the
 * semantics of PyG's Batch.from_data_list for the fields GNNML3 reads (DataLoader at graph8c.py:18, Zinc12k.py:20-22,
 * exp_classify.py:19-21, counting.py:29-31).  The records are rows of tables in device memory: n / e (nodes / support entries
 * per record), node_off / edge_off (first row of a record in x|xc and el|ea; NULL = the records are laid out in batch order),
 * idx (the B records to batch, NULL = records 0..B-1).  Features are x [*, F] or, for concatenated one-hot blocks, uint8 class
 * codes xc [*, C] with block widths (host array, sum = F).  el [2, el_stride] holds graph-local (src, dst) ids in el_bytes-wide
 * integers.  Outputs: x [Np, F], edge_index2 [2, Ep] (int64, global ids), edge_attr2 [Ep, K], batch [Np] (int64),
 * graph_ptr [B + 1] (int32; one more entry = Np when Np exceeds the batch's node count).  Rows beyond the batch's nodes /
 * entries receive the neutral padding of a captured step: isolated zero-feature nodes forming one dummy graph B, all-zero
 * self-loop entries spread over them.  Integer work, bit-exact with the host collation.  Two launches, no host sync.
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API size_t gnnml3_collate_workspace_bytes(int B);
GNNML3_API int gnnml3_collate(const int64_t* idx, const int32_t* n, const int32_t* e, const int64_t* node_off, const int64_t* edge_off,
                   const uint8_t* xc, int C, const int32_t* widths_host, const float* x, int F, const void* el, int el_bytes,
                   int64_t el_stride, const float* ea, int K, int B, int64_t Np, int64_t Ep, float* out_x,
                   int64_t* out_edge_index, float* out_edge_attr, int64_t* out_batch, int32_t* out_graph_ptr,
                   void* workspace, size_t workspace_bytes, void* stream);

/* The general form: records may carry the support list (e / edge_off / el / ea, K >= 1), the graph's plain edge list (what
 * GNNML1 reads: m = edges per record, adj_off = first edge of a record in al, al [2, al_stride] graph-local ids in al_bytes-wide
 * integers), or both.  K = 0 with NULL el / ea / out_edge_index2 / out_edge_attr2 (and Ep = 0): no supports.  m = NULL with NULL
 * al / out_edge_index (and Mp = 0): no plain list.  out_edge_index [2, Mp] receives int64 global ids in record order; columns
 * beyond the batch's edges get the same padding self-loops as the supports.  Padding a list (Ep > E or Mp > M) needs dummy
 * nodes (Np > N): the caller checks this, the kernel writes no padding edges without them.  gnnml3_collate is this call without
 * the plain list.  Workspace: 3 * (B + 1) int64. */
GNNML3_API size_t gnnml3_collate_graphs_workspace_bytes(int B);
GNNML3_API int gnnml3_collate_graphs(const int64_t* idx, const int32_t* n, const int64_t* node_off, const uint8_t* xc, int C,
                   const int32_t* widths_host, const float* x, int F, const int32_t* e, const int64_t* edge_off, const void* el,
                   int el_bytes, int64_t el_stride, const float* ea, int K, const int32_t* m, const int64_t* adj_off, const void* al,
                   int al_bytes, int64_t al_stride, int B, int64_t Np, int64_t Ep, int64_t Mp, float* out_x,
                   int64_t* out_edge_index2, float* out_edge_attr2, int64_t* out_edge_index, int64_t* out_batch,
                   int32_t* out_graph_ptr, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Isomorphism test (pairs.cu; graph8c.py:281-302, sr25.py, exp_iso.py): a pair of graphs is distinguished once the L1 distance
 * of its embeddings, dist = sum_{k=0..d-1} |a_k - b_k| (FP32, summed in dimension order: deterministic), exceeds `threshold`
 * under any seed.  NaN compares false: a pair whose distance is NaN stays undistinguished, as with the reference's cdist > thr.
 * Each call ORs one seed's embeddings emb [n, d] (row stride ld >= d) into a bitmap of uint32 words.
 *   gnnml3_pairs_mark, pairs == NULL (P = 0): every pair i < j < n; bit j of row i is bit (j % 32) of bits[i * wpr + j / 32],
 *       wpr >= ceil(n / 32).  128 x 128 pair tiles; a tile whose pairs are all marked already does no arithmetic.
 *   gnnml3_pairs_mark, pairs != NULL: the P listed pairs pairs [P, 2] int64 (row ids in [0, n); a pair with an id outside is
 *       never marked); bit p is bit (p % 32) of bits[p / 32], bits of ceil(P / 32) words (wpr unused).
 *   gnnml3_pairs_count: *out (device int64) = the number of pairs whose bit is still 0 -- the undistinguished pairs.  P == 0: the
 *       all-pairs bitmap of n rows; P > 0: the listed-pairs bitmap of P bits (n and wpr unused).  Fixed-order integer reduction
 *       in one thread-block cluster.
 * Returns GNNML3_ERR_INVALID for d < 1, ld < d, a negative n or P, a non-finite or negative threshold, or wpr < ceil(n / 32) in
 * all-pairs mode.  Bits that stand for no valid pair are ignored and never set.  No host sync; both calls are CUDA-graph
 * capturable.
 * --------------------------------------------------------------------------------------------------- */
GNNML3_API int gnnml3_pairs_mark(const float* emb, int64_t ld, int64_t n, int d, const int64_t* pairs, int64_t P,
                                 float threshold, uint32_t* bits, int64_t wpr, void* stream);
GNNML3_API int gnnml3_pairs_count(const uint32_t* bits, int64_t n, int64_t wpr, int64_t P, int64_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GNNML3_B200_H_ */
