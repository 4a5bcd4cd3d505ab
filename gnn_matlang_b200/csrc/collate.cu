// Batching on the device: per-graph records -> one disjoint-union batch with the reference's attributes (the semantics of PyG's
// Batch.from_data_list for the fields GNNML3 and GNNML1 read -- DataLoader at graph8c.py:18, Zinc12k.py:20-22, exp_classify.py:19-21,
// counting.py:29-31; host restatement: gnn_matlang_b200/batch.py::collate).  Two launches replace ~30 index kernels:
//   k_collate_scan   one block: node / support-entry / plain-edge offsets of the batch's graphs (exclusive scans of their sizes),
//                    graph_ptr
//   k_collate_fill   one warp per graph: batch vector, node features (copied, or expanded from uint8 class codes of one-hot
//                    blocks), edge_index2 = graph-local ids + node offset (int64, global), edge_attr2 rows, and the plain
//                    edge_index the same way; then the neutral padding up to the static shapes of a captured step (isolated
//                    zero-feature nodes forming one dummy graph, self-loops spread over them in both lists, all-zero supports --
//                    train.py::pad_batch)
// Either list is optional (GNNML1 reads only the plain one, GNNML3 only the supports).  The records come either from a pool
// resident in HBM (idx = graph ids, node_off / edge_off / adj_off = the pool's offsets: the step's only host -> device traffic is
// the id list) or from a batch in the compact wire format (idx = NULL, offsets = the scans).
// Integer work: bit-exact with the host collation (tests/test_gpu_data_path.py, tests/test_gpu_gnnml1_training.py).
#include "common.cuh"

namespace gnnml3 {

struct CollateParams {
    const int64_t* idx;          // [B] graph ids into the record tables, or NULL (identity)
    const int32_t* n;            // nodes per record
    const int32_t* e;            // support entries per record, or NULL (no supports: K = 0)
    const int32_t* m;            // plain edges per record, or NULL (no plain edge list)
    const int64_t* node_off;     // first node of a record in x / xc, or NULL (= offset inside the batch)
    const int64_t* edge_off;     // first entry of a record in el / ea, or NULL
    const int64_t* adj_off;      // first edge of a record in al, or NULL
    const uint8_t* xc;           // [*, C] class codes of C one-hot blocks, or NULL
    int C;
    int widths[4];
    const float* x;              // [*, F] features (when xc is NULL)
    int F;
    const void* el;              // [2, el_stride] graph-local (src, dst) of every support entry
    int el_bytes;                // 1 (uint8), 2 (int16), 4 (int32) or 8 (int64)
    int64_t el_stride;
    const float* ea;             // [*, K]
    int K;
    const void* al;              // [2, al_stride] graph-local (src, dst) of every plain edge
    int al_bytes;                // as el_bytes
    int64_t al_stride;
    int B;
    int64_t Np, Ep, Mp;          // rows of the output buffers (>= the batch's nodes / entries / edges; the rest is padding)
    float* out_x;                // [Np, F]
    int64_t* out_ei;             // [2, Ep]  edge_index2
    float* out_ea;               // [Ep, K]  edge_attr2
    int64_t* out_adj;            // [2, Mp]  edge_index
    int64_t* out_batch;          // [Np]
    int32_t* out_gp;             // [B + 1] (+ 1 more entry = Np when the batch is padded)
    int64_t* gp;                 // workspace [B + 1]
    int64_t* ep;                 // workspace [B + 1]
    int64_t* mp;                 // workspace [B + 1] (only read or written when m is given)
};

// Three exclusive scans (nodes, support entries, plain edges per graph) in one block, 1024 graphs per chunk.
__global__ void __launch_bounds__(1024) k_collate_scan(const CollateParams P) {
    __shared__ int64_t wsum[3][32];
    __shared__ int64_t carry[3];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        carry[0] = carry[1] = carry[2] = 0;
        P.gp[0] = 0;
        P.ep[0] = 0;
        if (P.m) P.mp[0] = 0;
        P.out_gp[0] = 0;
    }
    __syncthreads();
    for (int base = 0; base < P.B; base += 1024) {
        const int g = base + tid;
        int64_t vn = 0, ve = 0, vm = 0;
        if (g < P.B) {
            const int64_t id = P.idx ? P.idx[g] : g;
            vn = P.n[id];
            if (P.e) ve = P.e[id];
            if (P.m) vm = P.m[id];
        }
        int64_t sn = vn, se = ve, sm = vm;              // inclusive warp scans
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t tn = __shfl_up_sync(0xffffffffu, sn, o), te = __shfl_up_sync(0xffffffffu, se, o),
                          tm = __shfl_up_sync(0xffffffffu, sm, o);
            if (lane >= o) { sn += tn; se += te; sm += tm; }
        }
        if (lane == 31) { wsum[0][warp] = sn; wsum[1][warp] = se; wsum[2][warp] = sm; }
        __syncthreads();
        if (warp == 0) {
            int64_t a = wsum[0][lane], b = wsum[1][lane], c = wsum[2][lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t ta = __shfl_up_sync(0xffffffffu, a, o), tb = __shfl_up_sync(0xffffffffu, b, o),
                              tc = __shfl_up_sync(0xffffffffu, c, o);
                if (lane >= o) { a += ta; b += tb; c += tc; }
            }
            wsum[0][lane] = a;
            wsum[1][lane] = b;
            wsum[2][lane] = c;
        }
        __syncthreads();
        const int64_t on = carry[0] + (warp ? wsum[0][warp - 1] : 0) + sn, oe = carry[1] + (warp ? wsum[1][warp - 1] : 0) + se,
                      om = carry[2] + (warp ? wsum[2][warp - 1] : 0) + sm;
        if (g < P.B) {
            P.gp[g + 1] = on;
            P.ep[g + 1] = oe;
            if (P.m) P.mp[g + 1] = om;
            P.out_gp[g + 1] = (int32_t)on;
        }
        __syncthreads();
        if (tid == 1023) { carry[0] = on; carry[1] = oe; carry[2] = om; }
        __syncthreads();
    }
    if (tid == 0 && P.Np > P.gp[P.B]) P.out_gp[P.B + 1] = (int32_t)P.Np;      // the dummy graph of the padding
}

__device__ __forceinline__ int64_t load_local_id(const void* el, int bytes, int64_t i) {
    switch (bytes) {
        case 1: return (int64_t) reinterpret_cast<const uint8_t*>(el)[i];
        case 2: return (int64_t) reinterpret_cast<const int16_t*>(el)[i];
        case 4: return (int64_t) reinterpret_cast<const int32_t*>(el)[i];
        default: return reinterpret_cast<const int64_t*>(el)[i];
    }
}

// [2, cnt] graph-local ids (row stride `stride`) from `src` -> global ids (+ nb) at column `dst` of a [2, ld] int64 list
__device__ __forceinline__ void copy_edges(const void* ids, int bytes, int64_t stride, int64_t src, int cnt, int64_t nb, int64_t* out,
                                           int64_t ld, int64_t dst, int lane) {
    for (int p = lane; p < cnt; p += 32) {
        out[dst + p] = load_local_id(ids, bytes, src + p) + nb;
        out[ld + dst + p] = load_local_id(ids, bytes, stride + src + p) + nb;
    }
}

// self-loops on the dummy nodes N .. Np-1, round-robin, for the padding columns [from, ld) of a [2, ld] list
__device__ __forceinline__ void pad_edges(int64_t* out, int64_t from, int64_t ld, int64_t N, int64_t nd, int64_t tid, int64_t nthr) {
    for (int64_t p = from + tid; p < ld; p += nthr) {
        const int64_t v = N + (p - from) % nd;
        out[p] = v;
        out[ld + p] = v;
    }
}

__global__ void __launch_bounds__(256) k_collate_fill(const CollateParams P) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    const int64_t w0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int F = P.F, K = P.K;
    for (int64_t g = w0; g < P.B; g += nwarps) {
        const int64_t id = P.idx ? P.idx[g] : g;
        const int64_t nb = P.gp[g], ne = P.ep[g];
        const int cn = P.n[id], ce = P.e ? P.e[id] : 0;
        const int64_t sn = P.node_off ? P.node_off[id] : nb, se = P.edge_off ? P.edge_off[id] : ne;
        for (int i = lane; i < cn; i += 32) P.out_batch[nb + i] = g;
        if (P.xc) {
            for (int t = lane; t < cn * F; t += 32) {
                const int i = t / F, f = t - i * F;
                float v = 0.f;
                int off = 0;
                for (int c = 0; c < P.C; ++c) {
                    if ((int)P.xc[(sn + i) * P.C + c] + off == f) v = 1.f;
                    off += P.widths[c];
                }
                P.out_x[(nb + i) * F + f] = v;
            }
        } else {
            for (int t = lane; t < cn * F; t += 32) P.out_x[nb * F + t] = __ldg(P.x + sn * F + t);
        }
        copy_edges(P.el, P.el_bytes, P.el_stride, se, ce, nb, P.out_ei, P.Ep, ne, lane);
        if ((K & 3) == 0 && ((uintptr_t)P.ea & 15) == 0 && ((uintptr_t)P.out_ea & 15) == 0) {
            const float4* s4 = reinterpret_cast<const float4*>(P.ea + se * K);
            float4* d4 = reinterpret_cast<float4*>(P.out_ea + ne * K);
            for (int t = lane; t < ce * (K >> 2); t += 32) d4[t] = __ldg(s4 + t);
        } else {
            for (int t = lane; t < ce * K; t += 32) P.out_ea[ne * K + t] = __ldg(P.ea + se * K + t);
        }
        if (P.m) {
            const int64_t nm = P.mp[g];
            copy_edges(P.al, P.al_bytes, P.al_stride, P.adj_off ? P.adj_off[id] : nm, P.m[id], nb, P.out_adj, P.Mp, nm, lane);
        }
    }
    // neutral padding up to the static shapes
    const int64_t N = P.gp[P.B], E = P.ep[P.B];
    const int64_t nd = P.Np - N;                     // dummy nodes (the host checked Np > N whenever Ep > E or Mp > M)
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthr = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = N + tid; i < P.Np; i += nthr) P.out_batch[i] = P.B;
    for (int64_t t = N * F + tid; t < P.Np * F; t += nthr) P.out_x[t] = 0.f;
    if (P.Ep > E && nd > 0) {
        pad_edges(P.out_ei, E, P.Ep, N, nd, tid, nthr);
        for (int64_t t = E * K + tid; t < P.Ep * K; t += nthr) P.out_ea[t] = 0.f;
    }
    if (P.m && P.Mp > P.mp[P.B] && nd > 0) pad_edges(P.out_adj, P.mp[P.B], P.Mp, N, nd, tid, nthr);
}

static int collate_launch(const CollateParams& P, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    k_collate_scan<<<1, 1024, 0, st>>>(P);
    GNNML3_LAUNCH_CHECK();
    int64_t blocks = ((int64_t)P.B + 7) / 8;
    if (blocks < 1) blocks = 1;
    if (blocks > (int64_t)kNumSMs * 8) blocks = (int64_t)kNumSMs * 8;
    k_collate_fill<<<(int)blocks, 256, 0, st>>>(P);
    GNNML3_LAUNCH_CHECK();
    return GNNML3_OK;
}

}  // namespace gnnml3

using namespace gnnml3;

extern "C" size_t gnnml3_collate_workspace_bytes(int B) { return align_up((size_t)2 * (B + 1) * sizeof(int64_t), 256); }

extern "C" size_t gnnml3_collate_graphs_workspace_bytes(int B) { return align_up((size_t)3 * (B + 1) * sizeof(int64_t), 256); }

extern "C" int gnnml3_collate_graphs(const int64_t* idx, const int32_t* n, const int64_t* node_off, const uint8_t* xc, int C,
                                     const int32_t* widths_host, const float* x, int F, const int32_t* e, const int64_t* edge_off,
                                     const void* el, int el_bytes, int64_t el_stride, const float* ea, int K, const int32_t* m,
                                     const int64_t* adj_off, const void* al, int al_bytes, int64_t al_stride, int B, int64_t Np,
                                     int64_t Ep, int64_t Mp, float* out_x, int64_t* out_edge_index2, float* out_edge_attr2,
                                     int64_t* out_edge_index, int64_t* out_batch, int32_t* out_graph_ptr, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    GNNML3_REQUIRE(B >= 0 && Np >= 0 && Ep >= 0 && Mp >= 0 && F >= 1 && K >= 0, "collate_graphs: bad shape");
    if (B == 0 && Np == 0) return GNNML3_OK;
    GNNML3_REQUIRE(n && out_x && out_batch && out_graph_ptr && workspace, "collate_graphs: NULL pointer");
    GNNML3_REQUIRE(K == 0 ? (Ep == 0 && !el && !ea && !out_edge_index2 && !out_edge_attr2)
                          : (e && el && ea && out_edge_index2 && out_edge_attr2),
                   "collate_graphs: supports need K >= 1 and e, el, ea and both outputs; K = 0 needs Ep = 0 and NULL el / ea / outputs");
    GNNML3_REQUIRE(m ? (al && out_edge_index) : (Mp == 0 && !al && !out_edge_index),
                   "collate_graphs: the plain edge list needs m, al and out_edge_index; without m, Mp must be 0 and al / out_edge_index NULL");
    GNNML3_REQUIRE((xc != nullptr) != (x != nullptr), "collate_graphs: exactly one of xc (class codes) and x (features) must be given");
    GNNML3_REQUIRE(!el || el_bytes == 1 || el_bytes == 2 || el_bytes == 4 || el_bytes == 8, "collate_graphs: el_bytes must be 1, 2, 4 or 8");
    GNNML3_REQUIRE(!al || al_bytes == 1 || al_bytes == 2 || al_bytes == 4 || al_bytes == 8, "collate_graphs: al_bytes must be 1, 2, 4 or 8");
    GNNML3_REQUIRE(!xc || (C >= 1 && C <= 4 && widths_host), "collate_graphs: 1..4 one-hot blocks are supported");
    if (workspace_bytes < gnnml3_collate_graphs_workspace_bytes(B))
        return set_err(GNNML3_ERR_WORKSPACE, "collate_graphs: workspace too small");
    CollateParams P;
    P.idx = idx; P.n = n; P.e = K ? e : nullptr; P.m = m; P.node_off = node_off; P.edge_off = K ? edge_off : nullptr;
    P.adj_off = m ? adj_off : nullptr;
    P.xc = xc; P.C = xc ? C : 0;
    int wsum = 0;
    for (int c = 0; c < 4; ++c) {
        P.widths[c] = (xc && c < C) ? widths_host[c] : 0;
        wsum += P.widths[c];
    }
    GNNML3_REQUIRE(!xc || wsum == F, "collate_graphs: the one-hot block widths must add up to F");
    P.x = x; P.F = F; P.el = el; P.el_bytes = el_bytes; P.el_stride = el_stride; P.ea = ea; P.K = K;
    P.al = al; P.al_bytes = al_bytes; P.al_stride = al_stride; P.B = B; P.Np = Np; P.Ep = Ep; P.Mp = Mp;
    P.out_x = out_x; P.out_ei = out_edge_index2; P.out_ea = out_edge_attr2; P.out_adj = out_edge_index; P.out_batch = out_batch;
    P.out_gp = out_graph_ptr;
    P.gp = (int64_t*)workspace;
    P.ep = P.gp + (B + 1);
    P.mp = P.ep + (B + 1);
    return collate_launch(P, stream);
}

extern "C" int gnnml3_collate(const int64_t* idx, const int32_t* n, const int32_t* e, const int64_t* node_off, const int64_t* edge_off,
                              const uint8_t* xc, int C, const int32_t* widths_host, const float* x, int F, const void* el, int el_bytes,
                              int64_t el_stride, const float* ea, int K, int B, int64_t Np, int64_t Ep, float* out_x,
                              int64_t* out_edge_index, float* out_edge_attr, int64_t* out_batch, int32_t* out_graph_ptr,
                              void* workspace, size_t workspace_bytes, void* stream) {
    GNNML3_REQUIRE(B >= 0 && Np >= 0 && Ep >= 0 && F >= 1 && K >= 1, "collate: bad shape");
    if (B == 0 && Np == 0) return GNNML3_OK;
    GNNML3_REQUIRE(n && e && el && ea && out_x && out_edge_index && out_edge_attr && out_batch && out_graph_ptr && workspace,
                   "collate: NULL pointer");
    GNNML3_REQUIRE((xc != nullptr) != (x != nullptr), "collate: exactly one of xc (class codes) and x (features) must be given");
    GNNML3_REQUIRE(el_bytes == 1 || el_bytes == 2 || el_bytes == 4 || el_bytes == 8, "collate: el_bytes must be 1, 2, 4 or 8");
    GNNML3_REQUIRE(!xc || (C >= 1 && C <= 4 && widths_host), "collate: 1..4 one-hot blocks are supported");
    if (workspace_bytes < gnnml3_collate_workspace_bytes(B)) return set_err(GNNML3_ERR_WORKSPACE, "collate: workspace too small");
    int wsum = 0;
    for (int c = 0; xc && c < C; ++c) wsum += widths_host[c];
    GNNML3_REQUIRE(!xc || wsum == F, "collate: the one-hot block widths must add up to F");
    // the support list only: the workspace holds the node and entry scans, the plain-edge scan is never touched (m = NULL)
    CollateParams P = {};
    P.idx = idx; P.n = n; P.e = e; P.node_off = node_off; P.edge_off = edge_off; P.xc = xc; P.C = xc ? C : 0;
    for (int c = 0; c < 4; ++c) P.widths[c] = (xc && c < C) ? widths_host[c] : 0;
    P.x = x; P.F = F; P.el = el; P.el_bytes = el_bytes; P.el_stride = el_stride; P.ea = ea; P.K = K; P.B = B; P.Np = Np; P.Ep = Ep;
    P.out_x = out_x; P.out_ei = out_edge_index; P.out_ea = out_edge_attr; P.out_batch = out_batch; P.out_gp = out_graph_ptr;
    P.gp = (int64_t*)workspace;
    P.ep = P.gp + (B + 1);
    return collate_launch(P, stream);
}
