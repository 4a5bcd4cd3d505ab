// Whole-layer entry points: ONE C call enqueues every kernel of an ML3Layer forward (reference libs/spect_conv.py:204-212)
// or backward.  The arithmetic is exactly the sequence gnn_matlang_b200/libs/spect_conv.py::_ML3LayerFn composes from the
// single-kernel entry points (edge MLP -> fused aggregate+project+gates; backward: d pre, fused dx, SpMM + contraction for
// the weight gradients, fused dH+SDDMM, edge-MLP backward); what changes is the host cost: ~4 ctypes calls, ~25 small
// torch ops and as many allocations per layer and direction collapse into one call on a caller-provided workspace.  On
// B200 the host enqueue time of a training step (3.6 ms) had caught up with its GPU time (3.9 ms) -- see DESIGN.md.
#include "common.cuh"

namespace gnnml3 {

// wg [Fi, 2G] = [W11^T | W12^T], bg [2G] = [b11 | b12]   (operands of the fused forward's gate block)
__global__ void k_pack_gates_fwd(const float* __restrict__ w11, const float* __restrict__ w12, const float* __restrict__ b11,
                                 const float* __restrict__ b12, int Fi, int G, float* __restrict__ wg, float* __restrict__ bg) {
    const int total = Fi * 2 * G;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total + 2 * G; i += gridDim.x * blockDim.x) {
        if (i < total) {
            const int r = i / (2 * G), c = i % (2 * G);
            wg[i] = c < G ? __ldg(w11 + c * Fi + r) : __ldg(w12 + (c - G) * Fi + r);
        } else {
            const int c = i - total;
            bg[c] = c < G ? (b11 ? __ldg(b11 + c) : 0.f) : (b12 ? __ldg(b12 + c - G) : 0.f);
        }
    }
}

// wT [K*Fo, Fi]: wT[k*Fo + o][i] = W[k][i][o];  ws2 [2G, Fi] = [W11 ; W12]   (operands of the fused dx pass)
__global__ void k_pack_bwd(const float* __restrict__ W, const float* __restrict__ w11, const float* __restrict__ w12, int K, int Fi,
                           int Fo, int G, float* __restrict__ wT, float* __restrict__ ws2) {
    const int t1 = K * Fo * Fi, t2 = 2 * G * Fi;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < t1 + t2; idx += gridDim.x * blockDim.x) {
        if (idx < t1) {
            const int i = idx % Fi, o = (idx / Fi) % Fo, k = idx / (Fi * Fo);
            wT[idx] = __ldg(W + ((int64_t)k * Fi + i) * Fo + o);
        } else {
            const int j = idx - t1, r = j / Fi, i = j % Fi;
            ws2[j] = r < G ? __ldg(w11 + r * Fi + i) : __ldg(w12 + (r - G) * Fi + i);
        }
    }
}

// dst[r, c] = src[r, c] for a [rows x cols] block (row strides lds / ldd)
__global__ void k_copy_block(const float* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd, int64_t rows, int cols) {
    const int64_t total = rows * cols;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols;
        const int c = (int)(i - r * cols);
        dst[r * ldd + c] = __ldg(src + r * lds + c);
    }
}

// dcat [Fi, K*Fo + 2G] = x^T [G_0 .. G_{K-1} | g1 | g2]  ->  dW [K, Fi, Fo], dW11 [G, Fi], dW12 [G, Fi]
__global__ void k_unpack_dw(const float* __restrict__ dcat, int K, int Fi, int Fo, int G, int pitch, float* __restrict__ dw,
                            float* __restrict__ dw11, float* __restrict__ dw12) {
    const int ld = K * pitch + 2 * G;          // support k occupies columns [k * pitch, k * pitch + Fo)
    const int t1 = K * Fi * Fo, t2 = G * Fi;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < t1 + 2 * t2; idx += gridDim.x * blockDim.x) {
        if (idx < t1) {
            const int o = idx % Fo, i = (idx / Fo) % Fi, k = idx / (Fo * Fi);
            dw[idx] = __ldg(dcat + (int64_t)i * ld + k * pitch + o);
        } else if (dw11 == nullptr) {
            // gate weight gradients already written (ml3_act_bwd_y_gw)
        } else if (idx < t1 + t2) {
            const int j = idx - t1, g = j / Fi, i = j % Fi;
            dw11[j] = __ldg(dcat + (int64_t)i * ld + K * pitch + g);
        } else {
            const int j = idx - t1 - t2, g = j / Fi, i = j % Fi;
            dw12[j] = __ldg(dcat + (int64_t)i * ld + K * pitch + G + g);
        }
    }
}

// Layout of the forward-aggregate form of the weight gradient (first layer, no dx pass):
// ct [Fo, K*32] = gc^T [H_0 .. H_{K-1}] (H_k = S_k x, support k at columns [32 k, 32 k + Fi)), cg [Fi, 2G] = x^T [g1 | g2]
//   ->  dW [K, Fi, Fo], dW11 [G, Fi], dW12 [G, Fi]
__global__ void k_unpack_dw_t(const float* __restrict__ ct, const float* __restrict__ cg, int K, int Fi, int Fo, int G,
                              float* __restrict__ dw, float* __restrict__ dw11, float* __restrict__ dw12) {
    const int t1 = K * Fi * Fo, t2 = G * Fi;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < t1 + 2 * t2; idx += gridDim.x * blockDim.x) {
        if (idx < t1) {
            const int o = idx % Fo, i = (idx / Fo) % Fi, k = idx / (Fo * Fi);
            dw[idx] = __ldg(ct + (int64_t)o * (K * 32) + k * 32 + i);
        } else if (idx < t1 + t2) {
            const int j = idx - t1, g = j / Fi, i = j % Fi;
            dw11[j] = __ldg(cg + (int64_t)i * 2 * G + g);
        } else {
            const int j = idx - t1 - t2, g = j / Fi, i = j % Fi;
            dw12[j] = __ldg(cg + (int64_t)i * 2 * G + G + g);
        }
    }
}

// layer_ops.cu
int ml3_act_bwd_y_gw(const float* y, int64_t ldy, const float* aux, int64_t ldaux, const float* gy, int64_t ldgy, int64_t N, int Fo, int G,
                     float* gpre, int64_t ldg, float* colsum, const float* x, int64_t ldx, int Fi, float* dw11, float* dw12,
                     int* gate_dw_done, void* workspace, size_t workspace_bytes, void* stream);

static inline size_t a256(size_t x) { return align_up(x, 256); }

}  // namespace gnnml3

using namespace gnnml3;

extern "C" int gnnml3_ml3layer_supported(int K, int Fi, int Fo, int G, int learnedge) {
    if (learnedge && !gnnml3_edge_mlp_supported(K, K)) return 0;
    if (G > 0 && Fi > 32) return 0;
    if (!gnnml3_fused_supported(K, K, Fi, Fo, G > 0 ? Fi : 0, G > 0 ? 1 : 0, 2 * G)) return 0;
    if (!gnnml3_fused_supported(K, K, Fo, Fi, 2 * G, G > 0 ? 2 : 0, 0)) return 0;
    if (!gnnml3_fused_sddmm_supported(K, Fi, Fo)) return 0;
    return 1;
}

// workspace layout helpers -------------------------------------------------------------------------------------------
struct LayerWs {
    size_t fused, wg, bg, total_fwd;
    size_t gpre, act, wT, ws2, Gp, tn, dcat, dea2, sd, emlp, total_bwd;
    int64_t ldg;
};

static LayerWs layer_ws(int64_t N, int64_t E, int K, int Fi, int Fo, int G) {
    LayerWs w;
    const size_t f1 = gnnml3_fused_workspace_bytes(K, Fi, Fo, G > 0 ? 1 : 0), f2 = gnnml3_fused_workspace_bytes(K, Fo, Fi, G > 0 ? 2 : 0);
    size_t off = 0;
    w.fused = off; off += a256(f1 > f2 ? f1 : f2);
    w.wg = off; off += a256((size_t)Fi * 2 * G * 4 + 4);
    w.bg = off; off += a256((size_t)2 * G * 4 + 4);
    w.total_fwd = off;
    const int Fo4 = (Fo + 3) / 4 * 4;
    w.ldg = (Fo4 + 2 * G + 3) / 4 * 4;
    w.gpre = off; off += a256((size_t)N * w.ldg * 4);
    w.act = off; off += a256(gnnml3_ml3_act_bwd_workspace_bytes(N, Fo, G));
    w.wT = off; off += a256((size_t)K * Fo * Fi * 4);
    w.ws2 = off; off += a256((size_t)2 * G * Fi * 4 + 4);
    w.Gp = off; off += a256((size_t)N * ((K + 1) * 32) * 4);
    {   // the split count of gemm_tn depends on the column count: size for both layouts of G' (pitch 32 / pitch Fo)
        size_t t = gnnml3_gemm_tn_workspace_bytes(N, Fi, K * 32 + 2 * G);
        const size_t t2 = gnnml3_gemm_tn_workspace_bytes(N, Fi, K * Fo + 2 * G), t3 = gnnml3_gemm_tn_workspace_bytes(N, Fi, K * 32),
                     t4 = gnnml3_gemm_tn_workspace_bytes(N, Fi, 2 * G > 0 ? 2 * G : 1);
        t = t > t2 ? t : t2;
        t = t > t3 ? t : t3;
        t = t > t4 ? t : t4;
        const size_t t5 = gnnml3_gemm_tn_workspace_bytes(N, Fo, K * 32);       // gc^T H (forward-aggregate form)
        t = t > t5 ? t : t5;
        w.tn = off; off += a256(t);
    }
    w.dcat = off; off += a256((size_t)(Fi > Fo ? Fi : Fo) * (K * 32 + 2 * G) * 4);
    w.dea2 = off; off += a256((size_t)E * K * 4 + 4);
    w.sd = off; off += a256(gnnml3_fused_sddmm_workspace_bytes(K));
    w.emlp = off; off += a256(gnnml3_edge_mlp_bwd_workspace_bytes(E, K));
    w.total_bwd = off;
    return w;
}

extern "C" size_t gnnml3_ml3layer_workspace_bytes(int64_t N, int64_t E, int K, int Fi, int Fo, int G) {
    return layer_ws(N, E, K, Fi, Fo, G).total_bwd;
}

extern "C" int gnnml3_ml3layer_forward(const int32_t* rowptr, const int32_t* col, const int32_t* win, int64_t N, int64_t E, const float* x, int64_t ldx,
                                       int Fi, const float* ea_s, int K, const float* w1, const float* w2, const float* w3,
                                       const float* w4, const float* wconv, const float* bconv, int Fo, const float* w11,
                                       const float* b11, const float* w12, const float* b12, int G, float* ea2, float* y,
                                       int64_t ldy, float* aux, float* hside, int64_t ldh, void* workspace, size_t workspace_bytes,
                                       void* stream) {
    GNNML3_REQUIRE(N > 0 && E > 0, "ml3layer_forward: empty batch (the host takes the unfused path)");
    GNNML3_REQUIRE(hside == nullptr || (Fi <= 32 && ldh >= (int64_t)(K + (G > 0 ? 1 : 0)) * 32 && ldh % 4 == 0),
                   "ml3layer_forward: hside needs Fi <= 32 and rows of (K [+1]) * 32 floats");
    GNNML3_REQUIRE(gnnml3_ml3layer_supported(K, Fi, Fo, G, w1 != nullptr), "ml3layer_forward: unsupported shape K=%d Fi=%d Fo=%d G=%d", K,
                   Fi, Fo, G);
    const LayerWs w = layer_ws(N, E, K, Fi, Fo, G);
    if (workspace_bytes < w.total_fwd) return set_err(GNNML3_ERR_WORKSPACE, "ml3layer_forward: workspace too small");
    uint8_t* ws = (uint8_t*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    const float* eaw = ea_s;
    if (w1) {
        if ((rc = gnnml3_edge_mlp_fwd(ea_s, nullptr, w1, w2, w3, w4, E, K, K, ea2, stream))) return rc;
        eaw = ea2;
    }
    float *wg = nullptr, *bg = nullptr;
    if (G > 0) {
        wg = (float*)(ws + w.wg);
        bg = (float*)(ws + w.bg);
        k_pack_gates_fwd<<<cdiv((int64_t)Fi * 2 * G + 2 * G, 256), 256, 0, st>>>(w11, w12, b11, b12, Fi, G, wg, bg);
        GNNML3_LAUNCH_CHECK();
    }
    return gnnml3_fused_agg_proj(rowptr, col, nullptr, eaw, K, K, x, ldx, Fi, G > 0 ? x : nullptr, ldx, G > 0 ? Fi : 0, G > 0 ? 1 : 0, wconv,
                                 Fo, wg, 2 * G, 2 * G, bconv, bg, N, Fo, y, ldy, aux, 2 * G, G, 1, GNNML3_PREC_3XTF32, hside, hside ? ldh : 0, win, ws + w.fused,
                                 w.wg - w.fused, stream);
}

extern "C" int gnnml3_ml3layer_backward(const int32_t* rowptr, const int32_t* col, const int32_t* win, const int32_t* rowptrT,
                                        const int32_t* colT, const int32_t* permT, const int32_t* winT, int64_t N, int64_t E, const float* x, int64_t ldx, int Fi,
                                        const float* ea_s, const float* ea2, int K, const float* w1, const float* w2, const float* w3,
                                        const float* w4, const float* wconv, int Fo, const float* w11, const float* w12, int G,
                                        const float* y, int64_t ldy, const float* aux, const float* gy, int64_t ldgy, int need_dx,
                                        int need_dea, float* dx, int64_t lddx, float* dea, float* dw1, float* dw2, float* dw3,
                                        float* dw4, float* dwconv, float* dbias /* [Fo + 2G]: conv | fc11 | fc12 */, float* dw11,
                                        float* dw12, const float* hside, int64_t ldh, void* workspace, size_t workspace_bytes,
                                        void* stream) {
    GNNML3_REQUIRE(N > 0 && E > 0, "ml3layer_backward: empty batch (the host takes the unfused path)");
    GNNML3_REQUIRE(gnnml3_ml3layer_supported(K, Fi, Fo, G, w1 != nullptr), "ml3layer_backward: unsupported shape");
    const LayerWs w = layer_ws(N, E, K, Fi, Fo, G);
    if (workspace_bytes < w.total_bwd) return set_err(GNNML3_ERR_WORKSPACE, "ml3layer_backward: workspace too small");
    uint8_t* ws = (uint8_t*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    const float* eaw = w1 ? ea2 : ea_s;
    const int Fo4 = (Fo + 3) / 4 * 4;
    float* gpre = (float*)(ws + w.gpre);
    // d pre = [gc | 0 | g1 g2 | 0] and the three bias gradients (column sums)
    // (gate width 2: the same two launches also contract the gate gradients with x -> dW11 / dW12; the narrow GEMM below is skipped)
    int gate_dw_done = 0;
    const bool hside_form = !need_dx && hside;
    const bool side_form = need_dx && gnnml3_fused_set_mode(-1) == 0;
    if ((rc = ml3_act_bwd_y_gw(y, ldy, aux, 2 * G, gy, ldgy, N, Fo, G, gpre, w.ldg, dbias, (hside_form || side_form) ? x : nullptr, ldx, Fi, dw11,
                               dw12, &gate_dw_done, ws + w.act, w.wT - w.act, stream)))
        return rc;
    float* wT = (float*)(ws + w.wT);
    float* ws2 = (float*)(ws + w.ws2);
    k_pack_bwd<<<cdiv((int64_t)K * Fo * Fi + 2 * G * Fi, 256), 256, 0, st>>>(wconv, w11, w12, K, Fi, Fo, G, wT, ws2);
    GNNML3_LAUNCH_CHECK();
    // weight gradients: x^T [S_0^T gc .. S_{K-1}^T gc | g1 | g2].  When dx is needed the fused dx kernel leaves the aggregate
    // behind (pitch 32 per support, gate block at K * 32), so no separate SpMM runs; otherwise (first layer) SpMM builds it.
    float* Gp = (float*)(ws + w.Gp);
    float* dcat = (float*)(ws + w.dcat);
    int64_t ldG;
    int pitch;
    if (!need_dx && hside) {
        // first layer: no dx pass runs, and the forward left H = [S_0 x .. S_{K-1} x] behind (pitch 32): dW_k = H_k^T gc is one
        // contraction over the rows of (gc, H) -- no SpMM over the transposed CSR, no second aggregate (86 us on the ZINC step)
        float* ct = dcat;                                   // [Fo, K * 32]
        float* cg = dcat + (size_t)Fo * K * 32;             // [Fi, 2G]
        if ((rc = gnnml3_gemm_tn(gpre, w.ldg, hside, ldh, ct, K * 32, N, Fo, K * 32, GNNML3_PREC_3XTF32, ws + w.tn, w.dcat - w.tn, stream)))
            return rc;
        if (G > 0 && !gate_dw_done &&
            (rc = gnnml3_gemm_tn(x, ldx, gpre + Fo4, w.ldg, cg, 2 * G, N, Fi, 2 * G, GNNML3_PREC_3XTF32, ws + w.tn, w.dcat - w.tn, stream)))
            return rc;
        k_unpack_dw_t<<<cdiv((int64_t)K * Fi * Fo + 2 * G * Fi, 256), 256, 0, st>>>(ct, cg, K, Fi, Fo, gate_dw_done ? 0 : G, dwconv, dw11, dw12);
        GNNML3_LAUNCH_CHECK();
    } else {
    if (need_dx && gnnml3_fused_set_mode(-1) == 0) {          // (the side output exists in the default aggregator mode only)
        pitch = 32;
        ldG = (int64_t)(K + (G > 0 ? 1 : 0)) * 32;
        if ((rc = gnnml3_fused_agg_proj(rowptrT, colT, permT, eaw, K, K, gpre, w.ldg, Fo, G > 0 ? gpre + Fo4 : nullptr, w.ldg, 2 * G,
                                        G > 0 ? 2 : 0, wT, Fi, G > 0 ? ws2 : nullptr, Fi, 0, nullptr, nullptr, N, Fi, dx, lddx, nullptr, 0, 0,
                                        0, GNNML3_PREC_3XTF32, Gp, ldG, winT, ws + w.fused, w.wg - w.fused, stream)))
            return rc;
    } else {
        if (need_dx) {
            if ((rc = gnnml3_fused_agg_proj(rowptrT, colT, permT, eaw, K, K, gpre, w.ldg, Fo, G > 0 ? gpre + Fo4 : nullptr, w.ldg, 2 * G,
                                            G > 0 ? 2 : 0, wT, Fi, G > 0 ? ws2 : nullptr, Fi, 0, nullptr, nullptr, N, Fi, dx, lddx, nullptr, 0,
                                            0, 0, GNNML3_PREC_3XTF32, nullptr, 0, winT, ws + w.fused, w.wg - w.fused, stream)))
                return rc;
        }
        pitch = Fo;
        ldG = (int64_t)K * Fo + 2 * G;
        if ((rc = gnnml3_spmm_k(rowptrT, colT, permT, eaw, gpre, w.ldg, N, K, Fo, Gp, ldG, stream))) return rc;
        if (G > 0) {
            k_copy_block<<<cdiv(N * 2 * G, 256) > 1184 ? 1184 : cdiv(N * 2 * G, 256), 256, 0, st>>>(gpre + Fo4, w.ldg, Gp + (int64_t)K * Fo, ldG,
                                                                                                 N, 2 * G);
            GNNML3_LAUNCH_CHECK();
        }
    }
    const int ncols = K * pitch + 2 * G;
    if (pitch == 32 && G > 0) {
        // K * 32 columns are exactly four 64-wide column tiles of the contraction kernel; the 2G gate columns would open a
        // fifth, almost empty one (+30 % time), so they get their own small contraction straight from d pre
        if ((rc = gnnml3_gemm_tn(x, ldx, Gp, ldG, dcat, ncols, N, Fi, K * 32, GNNML3_PREC_3XTF32, ws + w.tn, w.dcat - w.tn, stream))) return rc;
        if (!gate_dw_done && (rc = gnnml3_gemm_tn(x, ldx, gpre + Fo4, w.ldg, dcat + K * 32, ncols, N, Fi, 2 * G, GNNML3_PREC_3XTF32, ws + w.tn,
                                                  w.dcat - w.tn, stream)))
            return rc;
    } else if ((rc = gnnml3_gemm_tn(x, ldx, Gp, ldG, dcat, ncols, N, Fi, ncols, GNNML3_PREC_3XTF32, ws + w.tn, w.dcat - w.tn, stream))) {
        return rc;
    }
    k_unpack_dw<<<cdiv((int64_t)K * Fi * Fo + 2 * G * Fi, 256), 256, 0, st>>>(dcat, K, Fi, Fo, G, pitch, dwconv, gate_dw_done ? nullptr : dw11,
                                                                              gate_dw_done ? nullptr : dw12);
    GNNML3_LAUNCH_CHECK();
    }
    // edge-feature gradient: fused dH + SDDMM, then back through the edge MLP
    if (w1 || need_dea) {
        float* dea2 = w1 ? (float*)(ws + w.dea2) : dea;
        if ((rc = gnnml3_fused_sddmm(rowptr, col, win, x, ldx, Fi, gpre, w.ldg, Fo, wconv, K, N, dea2, ws + w.sd, w.emlp - w.sd, stream))) return rc;
        if (w1) {
            if ((rc = gnnml3_edge_mlp_bwd(ea_s, nullptr, dea2, w1, w2, w3, w4, E, K, K, need_dea ? dea : nullptr, dw1, dw2, dw3, dw4,
                                          ws + w.emlp, w.total_bwd - w.emlp, stream)))
                return rc;
        }
    }
    return GNNML3_OK;
}
