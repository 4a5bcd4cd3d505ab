"""Tensor-level wrappers over the C ABI (one function per entry point of include/gnnml3_b200.h).

PyTorch is used here only for device memory (torch.empty on the input's device) and for the current
stream; all arithmetic happens inside libgnnml3_b200.so.  Every wrapper refuses CPU tensors.
"""
import os

import torch

from . import _lib

_workspaces = {}


class _NullCtx(object):
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NULL = _NullCtx()


def _on(device):
    """Context that makes ``device`` current -- a no-op object when it already is (torch.cuda.device() costs ~10 us of
    host time per call, and every training step makes ~90 library calls)."""
    idx = device.index
    if idx is None or idx == torch.cuda.current_device():
        return _NULL
    return torch.cuda.device(device)


def _ws(device, nbytes, tag="main"):
    """Grow-only scratch buffer per (device, current stream of that device, tag).  Reuse is ordered by the stream the buffer
    is keyed on: two streams driving the library on one device (evaluation overlapped with training, a side-stream prefetch
    that runs a layer) get separate buffers instead of overwriting each other's weight planes / partial sums."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (idx, torch._C._cuda_getCurrentRawStream(idx), tag)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def _f32c(t, name):
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32 (got %s)" % (name, t.dtype))
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: gnn_matlang_b200 has no CPU fallback" % name)
    return t if t.is_contiguous() else t.contiguous()


def _rows(t, name):
    """float32 CUDA matrix whose rows are unit-stride (row stride may exceed the width: column-block views)."""
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32 (got %s)" % (name, t.dtype))
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: gnn_matlang_b200 has no CPU fallback" % name)
    if t.dim() == 2 and (t.size(1) == 1 or t.stride(1) == 1) and (t.size(0) <= 1 or t.stride(0) >= t.size(1)):
        return t
    return t if t.is_contiguous() else t.contiguous()


def _ld(t):
    """Row stride in floats (size-1 leading dims can carry arbitrary strides, so fall back to the width)."""
    return t.stride(0) if t.size(0) > 1 else max(t.size(1), 1)


def csr_build(edge_index, num_nodes, check_range=True):
    """edge_index [2,E] int64 (row 0 = source, row 1 = target) -> dict of int32 CSR / transposed-CSR arrays."""
    lib = _lib.load()
    if edge_index.dtype != torch.int64 or edge_index.dim() != 2 or edge_index.size(0) != 2:
        raise RuntimeError("edge_index must be an int64 tensor of shape [2, E]")
    if not edge_index.is_cuda:
        raise RuntimeError("edge_index must be a CUDA tensor: gnn_matlang_b200 has no CPU fallback")
    ei = edge_index.contiguous()
    E, N = ei.size(1), int(num_nodes)
    dev = ei.device
    i32 = dict(dtype=torch.int32, device=dev)
    out = dict(rowptr=torch.empty(N + 1, **i32), col=torch.empty(E, **i32), perm=torch.empty(E, **i32),
               rowptrT=torch.empty(N + 1, **i32), colT=torch.empty(E, **i32), permT=torch.empty(E, **i32))
    flag = torch.zeros(1, **i32)
    nbytes = lib.gnnml3_csr_workspace_bytes(E, N)
    ws = _ws(dev, nbytes)
    with _on(dev):
        rc = lib.gnnml3_csr_build(_lib.ptr(ei), E, N, _lib.ptr(out["rowptr"]), _lib.ptr(out["col"]), _lib.ptr(out["perm"]),
                                  _lib.ptr(out["rowptrT"]), _lib.ptr(out["colT"]), _lib.ptr(out["permT"]),
                                  _lib.ptr(flag), _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
    _lib.check(rc, "gnnml3_csr_build")
    if check_range and int(flag.item()) != 0:
        raise RuntimeError("edge_index contains node ids outside [0, %d)" % N)
    if E > 0:
        # per-tile source windows of both CSRs (the fused layer kernel stages a tile's source rows in shared memory)
        nt = (N + lib.gnnml3_tile_rows() - 1) // lib.gnnml3_tile_rows()
        out["win"] = torch.empty(nt, 2, **i32)
        out["winT"] = torch.empty(nt, 2, **i32)
        with _on(dev):
            _lib.check(lib.gnnml3_tile_windows(_lib.ptr(out["rowptr"]), _lib.ptr(out["col"]), N, _lib.ptr(out["win"]),
                                               _lib.stream_ptr()), "gnnml3_tile_windows")
            _lib.check(lib.gnnml3_tile_windows(_lib.ptr(out["rowptrT"]), _lib.ptr(out["colT"]), N, _lib.ptr(out["winT"]),
                                               _lib.stream_ptr()), "gnnml3_tile_windows")
    else:
        out["win"] = out["winT"] = None
    return out


def tile_windows(rowptr, col):
    """[n_tiles, 2] int32 {first, last + 1} source row of each tile of the CSR (gnnml3_tile_windows)."""
    lib = _lib.load()
    N = rowptr.numel() - 1
    nt = (N + lib.gnnml3_tile_rows() - 1) // lib.gnnml3_tile_rows()
    win = torch.empty(nt, 2, dtype=torch.int32, device=rowptr.device)
    with _on(rowptr.device):
        _lib.check(lib.gnnml3_tile_windows(_lib.ptr(rowptr), _lib.ptr(col), N, _lib.ptr(win), _lib.stream_ptr()),
                   "gnnml3_tile_windows")
    return win


def gather_rows(src, perm):
    lib = _lib.load()
    src = _f32c(src, "src")
    rows, width = perm.numel(), src.size(1)
    out = torch.empty(rows, width, dtype=torch.float32, device=src.device)
    with _on(src.device):
        _lib.check(lib.gnnml3_gather_rows(_lib.ptr(src), _lib.ptr(perm), rows, width, _lib.ptr(out), _lib.stream_ptr()),
                   "gnnml3_gather_rows")
    return out


def scatter_rows(src, perm):
    lib = _lib.load()
    src = _f32c(src, "src")
    rows, width = perm.numel(), src.size(1)
    out = torch.empty(rows, width, dtype=torch.float32, device=src.device)
    with _on(src.device):
        _lib.check(lib.gnnml3_scatter_rows(_lib.ptr(src), _lib.ptr(perm), rows, width, _lib.ptr(out), _lib.stream_ptr()),
                   "gnnml3_scatter_rows")
    return out


def spmm_k(rowptr, col, eperm, ea, x, out=None):
    """out[t, k*F + f] = sum_{p in row t} ea[e(p), k] * x[col[p], f]  -> [N, K*F]"""
    lib = _lib.load()
    x = _rows(x, "x")
    ea = _f32c(ea, "edge_attr")
    N, F = x.shape
    K = ea.size(1)
    if out is None:
        out = torch.empty(N, K * F, dtype=torch.float32, device=x.device)
    if N == 0:
        return out
    with _on(x.device):
        _lib.check(lib.gnnml3_spmm_k(_lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(eperm), _lib.ptr(ea), _lib.ptr(x), _ld(x),
                                     N, K, F, _lib.ptr(out), _ld(out), _lib.stream_ptr()), "gnnml3_spmm_k")
    return out


def spmm_projected(rowptr, col, eperm, ea, Y, Fo, bias=None):
    """out[t, f] = sum_{p in row t} sum_k ea[e(p), k] * Y[col[p], k*Fo + f] (+ bias)  -> [N, Fo]  (project-first SpectConv)"""
    lib = _lib.load()
    Y = _rows(Y, "Y")
    ea = _f32c(ea, "edge_attr")
    N, K = Y.size(0), ea.size(1)
    out = torch.empty(N, Fo, dtype=torch.float32, device=Y.device)
    if N == 0:
        return out
    if bias is not None:
        bias = _f32c(bias, "bias")
    with _on(Y.device):
        _lib.check(lib.gnnml3_spmm_projected(_lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(eperm), _lib.ptr(ea), K, _lib.ptr(Y), _ld(Y), N, Fo,
                                             _lib.ptr(bias), _lib.ptr(out), _ld(out), _lib.stream_ptr()), "gnnml3_spmm_projected")
    return out


def sddmm_k(rowptr, col, eperm, x, g, K, E):
    """dea[e(p), k] = <x[col[p]], g[t, k*F:(k+1)*F]>  -> [E, K]"""
    lib = _lib.load()
    x = _rows(x, "x")
    g = _rows(g, "g")
    N, F = x.shape
    dea = torch.empty(E, K, dtype=torch.float32, device=x.device)
    if N == 0 or E == 0:
        return dea
    with _on(x.device):
        _lib.check(lib.gnnml3_sddmm_k(_lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(eperm), _lib.ptr(x), _ld(x), _lib.ptr(g),
                                      _ld(g), N, K, F, _lib.ptr(dea), _lib.stream_ptr()), "gnnml3_sddmm_k")
    return dea


USE_TCGEN05 = os.environ.get("GNNML3_NO_TCGEN05", "0") != "1"
TC_MIN_ROWS = 1024          # below this the persistent tcgen05 kernel cannot fill the machine; use the mma.sync path


def gemm_nn_tc(A, B, bias=None, epilogue=_lib.EPI_NONE, out=None, chunk_kblocks=0):
    """C = A @ B (+ bias) (+ relu) on tcgen05 / TMEM (3xTF32, FP32-grade).  A rows must be 16-byte aligned."""
    lib = _lib.load()
    A = _rows(A, "A")
    B = _f32c(B, "B")
    M, Kc = A.shape
    Nc = B.size(1)
    if B.size(0) != Kc:
        raise RuntimeError("gemm_nn_tc: inner dimensions differ (%d vs %d)" % (Kc, B.size(0)))
    if out is None:
        out = torch.empty(M, Nc, dtype=torch.float32, device=A.device)
    if M == 0:
        return out
    if bias is not None:
        bias = _f32c(bias, "bias")
    ws = _ws(A.device, lib.gnnml3_gemm_nn_tc_workspace_bytes(Nc, Kc), tag="tc")
    with _on(A.device):
        _lib.check(lib.gnnml3_gemm_nn_tc(_lib.ptr(A), _ld(A), _lib.ptr(B), _ld(B), _lib.ptr(bias), _lib.ptr(out), _ld(out),
                                         M, Nc, Kc, epilogue, chunk_kblocks, _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                   "gnnml3_gemm_nn_tc")
    return out


def gemm_nn(A, B, bias=None, precision=_lib.PREC_3XTF32, epilogue=_lib.EPI_NONE, out=None):
    """C = A @ B (+ bias) (+ relu) on the tensor cores; A [M,Kc], B [Kc,Nc].  FP32-grade (3xTF32) requests with
    16-byte aligned rows run on tcgen05/TMEM; everything else on the mma.sync kernel."""
    lib = _lib.load()
    A = _rows(A, "A")
    B = _f32c(B, "B")
    M, Kc = A.shape
    Nc = B.size(1)
    if B.size(0) != Kc:
        raise RuntimeError("gemm_nn: inner dimensions differ (%d vs %d)" % (Kc, B.size(0)))
    if (USE_TCGEN05 and precision == _lib.PREC_3XTF32 and M >= TC_MIN_ROWS and _ld(A) % 4 == 0 and A.data_ptr() % 16 == 0
            and lib.gnnml3_gemm_nn_tc_supported(_ld(A), Nc, Kc)):
        return gemm_nn_tc(A, B, bias, epilogue, out)
    if out is None:
        out = torch.empty(M, Nc, dtype=torch.float32, device=A.device)
    if M == 0:
        return out
    if bias is not None:
        bias = _f32c(bias, "bias")
    with _on(A.device):
        _lib.check(lib.gnnml3_gemm_nn(_lib.ptr(A), _ld(A), _lib.ptr(B), _ld(B), _lib.ptr(bias), _lib.ptr(out),
                                      _ld(out), M, Nc, Kc, precision, epilogue, _lib.stream_ptr()), "gnnml3_gemm_nn")
    return out


def gemm_tn(A, B, precision=_lib.PREC_3XTF32):
    """C = A^T @ B; A [M,Ka], B [M,Nb] -> [Ka,Nb]; deterministic split over M."""
    lib = _lib.load()
    A = _rows(A, "A")
    B = _rows(B, "B")
    M, Ka = A.shape
    Nb = B.size(1)
    out = torch.empty(Ka, Nb, dtype=torch.float32, device=A.device)
    if M == 0:
        return out.zero_()
    nbytes = lib.gnnml3_gemm_tn_workspace_bytes(M, Ka, Nb)
    ws = _ws(A.device, nbytes)
    with _on(A.device):
        _lib.check(lib.gnnml3_gemm_tn(_lib.ptr(A), _ld(A), _lib.ptr(B), _ld(B), _lib.ptr(out), _ld(out), M, Ka,
                                      Nb, precision, _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "gnnml3_gemm_tn")
    return out


def colsum(A):
    lib = _lib.load()
    A = _rows(A, "A")
    M, Nc = A.shape
    out = torch.empty(Nc, dtype=torch.float32, device=A.device)
    if M == 0:
        return out.zero_()
    nbytes = lib.gnnml3_colsum_workspace_bytes(M, Nc)
    ws = _ws(A.device, nbytes)
    with _on(A.device):
        _lib.check(lib.gnnml3_colsum(_lib.ptr(A), _ld(A), M, Nc, _lib.ptr(out), _lib.ptr(ws), ws.numel(),
                                     _lib.stream_ptr()), "gnnml3_colsum")
    return out


def edge_mlp_supported(K, Kout):
    return bool(_lib.load().gnnml3_edge_mlp_supported(int(K), int(Kout)))


def edge_mlp_fwd(ea, eperm, w1, w2, w3, w4):
    """relu(W4 [relu(W1 a) || tanh(W2 a) tanh(W3 a)]) per edge; output in the order of eperm (or ea's)."""
    lib = _lib.load()
    ea = _f32c(ea, "edge_attr")
    w1, w2, w3, w4 = (_f32c(w, "w") for w in (w1, w2, w3, w4))
    E, K = ea.shape
    Kout = w4.size(0)
    out = torch.empty(E, Kout, dtype=torch.float32, device=ea.device)
    with _on(ea.device):
        _lib.check(lib.gnnml3_edge_mlp_fwd(_lib.ptr(ea), _lib.ptr(eperm), _lib.ptr(w1), _lib.ptr(w2), _lib.ptr(w3), _lib.ptr(w4),
                                           E, K, Kout, _lib.ptr(out), _lib.stream_ptr()), "gnnml3_edge_mlp_fwd")
    return out


def edge_mlp_bwd(ea, eperm, gout, w1, w2, w3, w4, need_dea):
    lib = _lib.load()
    ea = _f32c(ea, "edge_attr")
    gout = _f32c(gout, "gout")
    w1, w2, w3, w4 = (_f32c(w, "w") for w in (w1, w2, w3, w4))
    E, K = ea.shape
    Kout = w4.size(0)
    dev = ea.device
    dea = torch.empty_like(ea) if need_dea else None
    dw = [torch.empty_like(w) for w in (w1, w2, w3, w4)]
    nbytes = lib.gnnml3_edge_mlp_bwd_workspace_bytes(E, K)
    ws = _ws(dev, nbytes)
    with _on(dev):
        _lib.check(lib.gnnml3_edge_mlp_bwd(_lib.ptr(ea), _lib.ptr(eperm), _lib.ptr(gout), _lib.ptr(w1), _lib.ptr(w2), _lib.ptr(w3),
                                           _lib.ptr(w4), E, K, Kout, _lib.ptr(dea), _lib.ptr(dw[0]), _lib.ptr(dw[1]),
                                           _lib.ptr(dw[2]), _lib.ptr(dw[3]), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                   "gnnml3_edge_mlp_bwd")
    return dea, dw


def ml3_act_fwd(pre, Fo, G):
    lib = _lib.load()
    N = pre.size(0)
    y = torch.empty(N, Fo + G, dtype=torch.float32, device=pre.device)
    with _on(pre.device):
        _lib.check(lib.gnnml3_ml3_act_fwd(_lib.ptr(pre), _ld(pre), N, Fo, G, _lib.ptr(y), _ld(y), _lib.stream_ptr()),
                   "gnnml3_ml3_act_fwd")
    return y


def ml3_act_bwd(pre, gy, Fo, G, gate_out=None):
    """-> (d pre [N, Fo+2G], column sums of d pre [Fo+2G] = bias gradients); ``gate_out`` (a [N, >=2G] strided
    view) receives a copy of the gate columns."""
    lib = _lib.load()
    gy = _f32c(gy, "gy")
    N = pre.size(0)
    # rows padded to a multiple of 4 floats: the column-block views of gpre then have 16-byte aligned rows and
    # qualify for 128-bit loads / the tcgen05 GEMM
    ld4 = (Fo + 2 * G + 3) // 4 * 4
    gpre = torch.empty(N, ld4, dtype=torch.float32, device=pre.device)[:, :Fo + 2 * G]
    csum = torch.empty(Fo + 2 * G, dtype=torch.float32, device=pre.device)
    ws = _ws(pre.device, lib.gnnml3_ml3_act_bwd_workspace_bytes(N, Fo, G))
    with _on(pre.device):
        _lib.check(lib.gnnml3_ml3_act_bwd(_lib.ptr(pre), _ld(pre), _lib.ptr(gy), _ld(gy), N, Fo, G, _lib.ptr(gpre),
                                          _ld(gpre), _lib.ptr(gate_out) if gate_out is not None else None,
                                          _ld(gate_out) if gate_out is not None else 0, _lib.ptr(csum), _lib.ptr(ws),
                                          ws.numel(), _lib.stream_ptr()),
                   "gnnml3_ml3_act_bwd")
    return gpre, csum


def _padded_rows(N, W, device):
    """[N, W] float32 view of a buffer whose rows are padded to a multiple of 4 floats, padding columns zeroed (they are read,
    and multiplied by zero weights, by the next fused gather); the base carries the mark ``aligned_rows`` looks for."""
    ld = (W + 3) // 4 * 4
    buf = torch.empty(N, ld, dtype=torch.float32, device=device)
    if ld != W:
        buf[:, W:].zero_()
        buf._gnnml3_zero_pad = True
        return buf[:, :W]
    return buf


def aligned_rows(t):
    """float32 CUDA matrix with unit column stride, row stride % 4 == 0 and a 16-byte aligned base (what the 128-bit
    gathers of the fused kernels need); otherwise a zero-padded copy [N, ceil4(F)] (data movement only)."""
    if t.dtype != torch.float32 or not t.is_cuda:
        raise RuntimeError("expected a float32 CUDA tensor: gnn_matlang_b200 has no CPU fallback")
    if t.dim() == 2 and t.stride(1) == 1 and t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0 and t.stride(0) >= t.size(1):
        # F % 4 != 0: the kernels gather ceil4(F) columns and rely on zero weights for the padding -- 0 * NaN is NaN, so a view
        # passes through only when its padding columns are known to be zero (tensors allocated by _padded_rows below); a
        # caller's column block of a wider matrix is copied
        if t.size(1) % 4 == 0 or getattr(t._base, "_gnnml3_zero_pad", False):
            return t
    N, F = t.shape
    buf = torch.zeros(N, (F + 3) // 4 * 4, dtype=torch.float32, device=t.device)
    buf[:, :F] = t
    return buf[:, :F]


def fused_supported(K, Kstride, F, Nc, Fs=0, self_mode=0, Ns=0):
    return bool(_lib.load().gnnml3_fused_supported(int(K), int(Kstride), int(F), int(Nc), int(Fs), int(self_mode), int(Ns)))


def fused_ts_supported(K, Kstride, F, Nc, Fs=0, self_mode=0, Ns=0):
    """gnnml3_fused_agg_proj runs the tensor-memory generation of the fused kernel (the only one with the TF32 / BF16 modes)
    for this shape: the shape is covered (gnnml3_fused_ts_supported) and the aggregator mode is the default one -- the slot
    mode (gnnml3_fused_set_mode(1)) always runs the shared-memory-plane kernel."""
    lib = _lib.load()
    return bool(lib.gnnml3_fused_ts_supported(int(K), int(Kstride), int(F), int(Nc), int(Fs), int(self_mode), int(Ns))
                and lib.gnnml3_fused_set_mode(-1) == 0)


def fused_agg_proj(rowptr, col, eperm, ea, x, Bmain, bias=None, S=None, self_mode=0, Bself=None, bias_s=None, G=0,
                   epilogue=0, hout=None, win=None, precision=_lib.PREC_3XTF32, aux=True):
    """Fused aggregate + project (gnnml3_fused_agg_proj).  x [*, F] and S [N, Fs] must satisfy ``aligned_rows``.
    epilogue 0 -> out [N, Nc];  epilogue 1 -> (y [N, Nc + G], aux [N, 2G]) = the ML3Layer node branch.
    ``aux=False`` (a forward nobody differentiates): the kernel stores y alone and the returned aux is None."""
    lib = _lib.load()
    ea = _f32c(ea, "edge_attr")
    Bmain = _f32c(Bmain, "Bmain")
    N = rowptr.numel() - 1
    F, K = x.size(1), ea.size(1)
    Nc = Bmain.size(1)
    if Bmain.size(0) != K * F:
        raise RuntimeError("fused_agg_proj: Bmain must be [K*F, Nc] = [%d, %d], got %s" % (K * F, Nc, tuple(Bmain.shape)))
    Fs = Ns = 0
    if self_mode:
        Bself = _f32c(Bself, "Bself")
        Fs, Ns = S.size(1), Bself.size(1)
        if Bself.size(0) != Fs:
            raise RuntimeError("fused_agg_proj: Bself must have %d rows" % Fs)
    dev = x.device
    W = Nc + (G if self_mode == 1 else 0)
    out = _padded_rows(N, W, dev)
    save_aux = self_mode == 1 and aux
    aux = torch.empty(N, 2 * G, dtype=torch.float32, device=dev) if save_aux else None
    if bias is not None:
        bias = _f32c(bias, "bias")
    if bias_s is not None:
        bias_s = _f32c(bias_s, "bias_s")
    # algorithmic HBM bytes of this launch (SURVEY.md 8d: every operand once, the [N, K*F] aggregate never counted)
    E = ea.size(0)
    _prof["last_bytes"] = 4.0 * (N * F + (N * Fs if (self_mode and S.data_ptr() != x.data_ptr()) else 0) + E * K + E * (2 if eperm is not None else 1)
                                 + (N + 1) + K * F * Nc + Fs * Ns + Nc + N * W + (N * 2 * G if save_aux else 0))
    ws = _ws(dev, lib.gnnml3_fused_workspace_bytes(K, F, Nc, self_mode), tag="fused")
    with _on(dev):
        _lib.check(lib.gnnml3_fused_agg_proj(
            _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(eperm), _lib.ptr(ea), K, K, _lib.ptr(x), _ld(x), F,
            _lib.ptr(S) if self_mode else None, _ld(S) if self_mode else 0, Fs, self_mode, _lib.ptr(Bmain), _ld(Bmain),
            _lib.ptr(Bself) if self_mode else None, _ld(Bself) if self_mode else 0, Ns, _lib.ptr(bias), _lib.ptr(bias_s),
            N, Nc, _lib.ptr(out), (W + 3) // 4 * 4, _lib.ptr(aux), 2 * G, G, epilogue, precision, _lib.ptr(hout), _ld(hout) if hout is not None else 0,
            _lib.ptr(win), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
            "gnnml3_fused_agg_proj")
    return out, aux


def ml3_act_bwd_y(y, aux, gy, Fo, G):
    """d pre from the fused layer's outputs -> (gpre [N, ldg] in the layout [conv | 0.. | g1 g2 | 0..] with the gate block
    at column ceil4(Fo), column sums [Fo + 2G] = bias gradients)."""
    lib = _lib.load()
    gy = _rows(gy, "gy")
    N = y.size(0)
    Fo4 = (Fo + 3) // 4 * 4
    ldg = (Fo4 + 2 * G + 3) // 4 * 4
    gpre = torch.empty(N, ldg, dtype=torch.float32, device=y.device)
    csum = torch.empty(Fo + 2 * G, dtype=torch.float32, device=y.device)
    ws = _ws(y.device, lib.gnnml3_ml3_act_bwd_workspace_bytes(N, Fo, G))
    with _on(y.device):
        _lib.check(lib.gnnml3_ml3_act_bwd_y(_lib.ptr(y), _ld(y), _lib.ptr(aux), 2 * G, _lib.ptr(gy), _ld(gy), N, Fo, G,
                                            _lib.ptr(gpre), ldg, _lib.ptr(csum), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                   "gnnml3_ml3_act_bwd_y")
    return gpre, csum


def fused_path_counts(reset=False):
    """(launches of the tensor-memory fused kernel, launches of the shared-memory-plane kernel) since the last reset."""
    import ctypes
    buf = (ctypes.c_longlong * 2)()
    _lib.load().gnnml3_fused_path_counts(buf, int(bool(reset)))
    return int(buf[0]), int(buf[1])


def edge_mlp_path_counts(reset=False):
    """(calls served by the tcgen05 edge-MLP kernels, calls served by the FP32-FMA kernels) since the last reset."""
    import ctypes
    buf = (ctypes.c_longlong * 2)()
    _lib.load().gnnml3_edge_mlp_path_counts(buf, int(bool(reset)))
    return int(buf[0]), int(buf[1])


def edge_mlp_set_tc(enable):
    """Select the tcgen05 (True, default) or the FP32-FMA (False) generation of the edge-MLP kernels; returns the old setting."""
    return bool(_lib.load().gnnml3_edge_mlp_set_tc(int(bool(enable))))


def fused_side_output_ok():
    """The aggregate side output (``hout``) of fused_agg_proj exists in the default aggregator mode only."""
    return _lib.load().gnnml3_fused_set_mode(-1) == 0


def fused_sddmm_supported(K, Fi, Fo):
    return bool(_lib.load().gnnml3_fused_sddmm_supported(int(K), int(Fi), int(Fo)))


def fused_sddmm(rowptr, col, x, gc, W, E, win=None):
    """dea[p, k] = <x[col[p]], gc[t] W[k]^T> for every CSR slot p of row t (gnnml3_fused_sddmm) -> [E, K].
    x [N, Fi] and gc [N, Fo] must satisfy ``aligned_rows``; W [K, Fi, Fo]; ``win`` = the plan's per-tile source windows of
    (rowptr, col) (``plan.win``): with them the source rows are staged in shared memory."""
    lib = _lib.load()
    W = _f32c(W, "W")
    K, Fi, Fo = W.shape
    N = rowptr.numel() - 1
    dea = torch.empty(E, K, dtype=torch.float32, device=x.device)
    ws = _ws(x.device, lib.gnnml3_fused_sddmm_workspace_bytes(K), tag="fused_sddmm")
    with _on(x.device):
        _lib.check(lib.gnnml3_fused_sddmm(_lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(win), _lib.ptr(x), _ld(x), Fi, _lib.ptr(gc), _ld(gc), Fo,
                                          _lib.ptr(W), K, N, _lib.ptr(dea), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
                   "gnnml3_fused_sddmm")
    return dea


def ml3layer_supported(K, Fi, Fo, G, learnedge):
    return bool(_lib.load().gnnml3_ml3layer_supported(int(K), int(Fi), int(Fo), int(G), int(bool(learnedge))))


def ml3layer_forward(plan, x, ea_s, ws4, wconv, bconv, gates, keep_aggregate=False, aux=True):
    """Whole ML3Layer forward in one library call (gnnml3_ml3layer_forward).  ``ws4`` = (w1, w2, w3, w4) or None,
    ``gates`` = (w11, b11, w12, b12) or None.  -> (y [N, Fo+G], aux [N, 2G] | None, ea2 [E, K] | None, hside | None)
    ``keep_aggregate``: also leave H = [S_0 x .. S_{K-1} x] behind ([N, (K [+1]) * 32]) for a backward that needs the weight
    gradient but no dx (first layer): dW_k = H_k^T gc then needs no aggregation over the transposed CSR.
    ``aux=False`` (a forward nobody differentiates): the tanh factors are not stored and the returned aux is None."""
    lib = _lib.load()
    N, Fi = x.shape
    E, K = ea_s.shape
    Fo = wconv.size(2)
    G = gates[0].size(0) if gates is not None else 0
    dev = x.device
    W = Fo + G
    y = _padded_rows(N, W, dev)
    ldy = (W + 3) // 4 * 4
    aux = torch.empty(N, 2 * G, dtype=torch.float32, device=dev) if (G > 0 and aux) else None
    ea2 = torch.empty(E, K, dtype=torch.float32, device=dev) if ws4 is not None else None
    ldh = (K + (1 if G > 0 else 0)) * 32
    hside = torch.empty(N, ldh, dtype=torch.float32, device=dev) if (keep_aggregate and Fi <= 32) else None
    ws = _ws(dev, lib.gnnml3_ml3layer_workspace_bytes(N, E, K, Fi, Fo, G), tag="layer")
    p = _lib.ptr
    w = ws4 if ws4 is not None else (None,) * 4
    g = gates if gates is not None else (None,) * 4
    with _on(dev):
        _lib.check(lib.gnnml3_ml3layer_forward(p(plan.rowptr), p(plan.col), p(plan.win), N, E, p(x), _ld(x), Fi, p(ea_s), K, p(w[0]), p(w[1]), p(w[2]),
                                               p(w[3]), p(wconv), p(bconv), Fo, p(g[0]), p(g[1]), p(g[2]), p(g[3]), G, p(ea2), p(y), ldy,
                                               p(aux), p(hside), ldh, p(ws), ws.numel(), _lib.stream_ptr()), "gnnml3_ml3layer_forward")
    return y, aux, ea2, hside


def ml3layer_backward(plan, x, ea_s, ea2, ws4, wconv, gates_w, y, aux, gy, need_dx, need_dea, has_bias, hside=None):
    """Whole ML3Layer backward in one library call (gnnml3_ml3layer_backward).
    -> dx, dea, (dw1..dw4), dwconv, dbconv, dw11, db11, dw12, db12 (None where not applicable)"""
    lib = _lib.load()
    N, Fi = x.shape
    E, K = ea_s.shape
    Fo = wconv.size(2)
    G = gates_w[0].size(0) if gates_w is not None else 0
    dev = x.device
    f32 = dict(dtype=torch.float32, device=dev)
    lddx = (Fi + 3) // 4 * 4
    dx = torch.empty(N, lddx, **f32) if need_dx else None
    dea = torch.empty(E, K, **f32) if need_dea else None
    dws = [torch.empty_like(t) for t in ws4] if ws4 is not None else [None] * 4
    dwc = torch.empty_like(wconv)
    dbias = torch.empty(Fo + 2 * G, **f32)
    dw11 = torch.empty(G, Fi, **f32) if G > 0 else None
    dw12 = torch.empty(G, Fi, **f32) if G > 0 else None
    ws = _ws(dev, lib.gnnml3_ml3layer_workspace_bytes(N, E, K, Fi, Fo, G), tag="layer")
    p = _lib.ptr
    w = ws4 if ws4 is not None else (None,) * 4
    gw = gates_w if gates_w is not None else (None, None)
    with _on(dev):
        _lib.check(lib.gnnml3_ml3layer_backward(
            p(plan.rowptr), p(plan.col), p(plan.win), p(plan.rowptrT), p(plan.colT), p(plan.permT), p(plan.winT), N, E, p(x), _ld(x), Fi, p(ea_s), p(ea2), K,
            p(w[0]), p(w[1]), p(w[2]), p(w[3]), p(wconv), Fo, p(gw[0]), p(gw[1]), G, p(y), _ld(y), p(aux), p(gy), _ld(gy),
            int(need_dx), int(need_dea), p(dx), lddx, p(dea), p(dws[0]), p(dws[1]), p(dws[2]), p(dws[3]), p(dwc), p(dbias), p(dw11),
            p(dw12), p(hside), _ld(hside) if hside is not None else 0, p(ws), ws.numel(), _lib.stream_ptr()), "gnnml3_ml3layer_backward")
    dbc = dbias[:Fo] if has_bias else None
    db11 = dbias[Fo:Fo + G] if G > 0 else None
    db12 = dbias[Fo + G:] if G > 0 else None
    return (dx[:, :Fi] if need_dx else None), dea, dws, dwc, dbc, dw11, db11, dw12, db12


def ml1layer_supported(Fi, Fo, concat=False):
    return bool(_lib.load().gnnml3_ml1layer_supported(int(Fi), int(Fo), int(bool(concat))))


def ml1layer_forward(plan, x, wconv, bconv, wA, bA, wB, bB, wC, bC, concat=False, keep_aggregate=False, aux=True,
                     precision=_lib.PREC_3XTF32):
    """Whole GNNML1 layer forward in one library call (gnnml3_ml1layer_forward) over the plan of the plain ``edge_index``.
    x [N, Fi] must satisfy ``aligned_rows``; wconv [1, Fi, Fo]; wA/wB/wC [Fo, Fi].  -> (y [N, Fo] or [N, 3 Fo],
    aux [N, 2 Fo] = [p1 | p2] (None with ``aux=False``: a forward nobody differentiates stores y alone),
    A x [N, Fi] if ``keep_aggregate`` else None).  ``precision`` (PREC_3XTF32 | PREC_TF32 | PREC_BF16): the arithmetic of the
    projection."""
    lib = _lib.load()
    N, Fi = x.shape
    Fo = wconv.size(2)
    dev = x.device
    W = 3 * Fo if concat else Fo
    y = _padded_rows(N, W, dev)
    aux = torch.empty(N, 2 * Fo, dtype=torch.float32, device=dev) if aux else None
    hside = _padded_rows(N, Fi, dev) if keep_aggregate else None
    ws = _ws(dev, lib.gnnml3_ml1layer_workspace_bytes(N, Fi, Fo, int(bool(concat))), tag="ml1")
    p = _lib.ptr
    args = (p(plan.rowptr), p(plan.col), N, plan.E, p(x), _ld(x), Fi, p(wconv), p(bconv), p(wA), p(bA), p(wB), p(bB), p(wC), p(bC), Fo,
            int(bool(concat)), p(y), _ld(y) if N > 1 else (W + 3) // 4 * 4, p(aux), 2 * Fo, p(hside), (Fi + 3) // 4 * 4, p(ws), ws.numel(),
            _lib.stream_ptr(), precision)
    with _on(dev):
        _lib.check(lib.gnnml3_ml1layer_forward(*args), "gnnml3_ml1layer_forward")
    return y, aux, hside


def ml1layer_backward(plan, x, wconv, wA, wB, wC, y, aux, gy, need_dx, concat=False, precision=_lib.PREC_3XTF32):
    """Whole GNNML1 layer backward in one library call (gnnml3_ml1layer_backward) in ``precision``.
    -> dx (None unless need_dx), dwconv, dbconv, dwA, dbA, dwB, dbB, dwC, dbC"""
    lib = _lib.load()
    N, Fi = x.shape
    Fo = wconv.size(2)
    dev = x.device
    f32 = dict(dtype=torch.float32, device=dev)
    lddx = (Fi + 3) // 4 * 4
    dx = torch.empty(N, lddx, **f32) if need_dx else None
    dwc = torch.empty_like(wconv)
    dwA, dwB, dwC = torch.empty_like(wA), torch.empty_like(wB), torch.empty_like(wC)
    dbs = torch.empty(4, Fo, **f32)                      # conv | fcA | fcB | fcC
    ws = _ws(dev, lib.gnnml3_ml1layer_workspace_bytes(N, Fi, Fo, int(bool(concat))), tag="ml1")
    p = _lib.ptr
    args = (p(plan.rowptrT), p(plan.colT), N, plan.E, p(x), _ld(x), Fi, p(wconv), p(wA), p(wB), p(wC), Fo, int(bool(concat)),
            p(y), _ld(y) if N > 1 else y.size(1), p(aux), 2 * Fo, p(gy), _ld(gy), int(bool(need_dx)), p(dx), lddx, p(dwc), p(dbs[0]),
            p(dwA), p(dbs[1]), p(dwB), p(dbs[2]), p(dwC), p(dbs[3]), p(ws), ws.numel(), _lib.stream_ptr(), precision)
    with _on(dev):
        _lib.check(lib.gnnml3_ml1layer_backward(*args), "gnnml3_ml1layer_backward")
    return (dx[:, :Fi] if need_dx else None), dwc, dbs[0], dwA, dbs[1], dwB, dbs[2], dwC, dbs[3]


def collate_device(n, e, el, ea, B, out, idx=None, node_off=None, edge_off=None, xc=None, widths=None, x=None, m=None, al=None,
                   adj_off=None):
    """Batch B per-graph records on the device (gnnml3_collate / gnnml3_collate_graphs) into the tensors of ``out`` (a ``Batch``
    whose ``x [Np, F]``, ``edge_index2 [2, Ep]`` int64, ``edge_attr2 [Ep, K]``, ``batch [Np]`` int64 and ``graph_ptr`` int32 are
    preallocated; rows beyond the batch's nodes / entries get the neutral padding of a captured step).  Records: ``n`` / ``e``
    int32 sizes, ``el [2, *]`` graph-local ids (uint8 / int16 / int32 / int64), ``ea [*, K]``, features ``x [*, F]`` or uint8
    class codes ``xc [*, C]`` + ``widths``; ``idx`` (int64 graph ids) with ``node_off`` / ``edge_off`` (int64) select records of a
    resident pool, None = the records are the batch itself in order.

    The plain edge list (what GNNML1 reads): ``m`` int32 edges per record, ``al [2, *]`` graph-local ids (same dtypes as ``el``),
    ``adj_off`` int64 pool offsets (with ``idx``); ``out.edge_index [2, Mp]`` int64 receives it, padded like the supports.
    ``ea=None``: the records have no supports (``e`` / ``el`` are ignored and ``out`` needs no ``edge_index2`` / ``edge_attr2``)."""
    import ctypes
    lib = _lib.load()
    sup, adj = ea is not None, m is not None
    if not sup and not adj:
        raise RuntimeError("collate_device: the records carry neither supports (ea) nor a plain edge list (m, al)")
    dev = n.device
    if sup and el.is_cuda and not el.is_contiguous():
        el = el.contiguous()
    if adj and al is not None and al.is_cuda and not al.is_contiguous():
        al = al.contiguous()
    checks = [("n", n), ("out.x", out.x), ("out.batch", out.batch), ("out.graph_ptr", out.graph_ptr)]
    if sup:
        checks += [("e", e), ("el", el), ("ea", ea), ("out.edge_index2", out.edge_index2), ("out.edge_attr2", out.edge_attr2)]
    if adj:
        if al is None or getattr(out, "edge_index", None) is None:
            raise RuntimeError("collate_device: the plain edge list needs m, al and out.edge_index")
        checks += [("m", m), ("al", al), ("out.edge_index", out.edge_index)]
    for name, t in checks:
        if not t.is_cuda or not t.is_contiguous():
            raise RuntimeError("collate_device: %s must be a contiguous CUDA tensor (no CPU fallback)" % name)
    if n.dtype != torch.int32 or out.batch.dtype != torch.int64 or out.graph_ptr.dtype != torch.int32 or out.x.dtype != torch.float32 \
            or (sup and (e.dtype != torch.int32 or out.edge_index2.dtype != torch.int64 or ea.dtype != torch.float32)) \
            or (adj and (m.dtype != torch.int32 or out.edge_index.dtype != torch.int64)):
        raise RuntimeError("collate_device: unexpected dtype")
    for t in ((el,) if sup else ()) + ((al,) if adj else ()):
        if t.dtype not in (torch.uint8, torch.int16, torch.int32, torch.int64) or t.dim() != 2 or t.size(0) != 2:
            raise RuntimeError("collate_device: el / al must be [2, *] uint8 / int16 / int32 / int64")
    Np, F = out.x.shape
    Ep, K = out.edge_attr2.shape if sup else (0, 0)
    Mp = out.edge_index.size(1) if adj else 0
    if (sup and (out.edge_index2.size(1) != Ep or ea.size(1) != K)) or (adj and out.edge_index.size(0) != 2) \
            or out.batch.numel() != Np or out.graph_ptr.numel() < B + 1:
        raise RuntimeError("collate_device: output shapes do not match")
    wh = None
    C = 0
    if xc is not None:
        C = xc.size(1)
        wh = (ctypes.c_int32 * C)(*[int(w) for w in widths])
        if xc.dtype != torch.uint8 or not xc.is_contiguous():
            raise RuntimeError("collate_device: xc must be a contiguous uint8 tensor")
    elif x is None or x.dtype != torch.float32 or not x.is_contiguous() or x.size(1) != F:
        raise RuntimeError("collate_device: x [*, F] float32 or xc + widths must be given")
    for t in (idx, node_off, edge_off, adj_off):
        if t is not None and (t.dtype != torch.int64 or not t.is_cuda or not t.is_contiguous()):
            raise RuntimeError("collate_device: idx / node_off / edge_off / adj_off must be contiguous int64 CUDA tensors")
    P = _lib.ptr
    if sup and not adj:
        ws = _ws(dev, lib.gnnml3_collate_workspace_bytes(int(B)), tag="collate")
        with _on(dev):
            _lib.check(lib.gnnml3_collate(P(idx), P(n), P(e), P(node_off), P(edge_off), P(xc), C, wh, P(x), F, P(el),
                                          el.element_size(), el.size(1), P(ea), K, int(B), Np, Ep, P(out.x), P(out.edge_index2),
                                          P(out.edge_attr2), P(out.batch), P(out.graph_ptr), P(ws), ws.numel(), _lib.stream_ptr()),
                       "gnnml3_collate")
        return out
    ws = _ws(dev, lib.gnnml3_collate_graphs_workspace_bytes(int(B)), tag="collate")
    with _on(dev):
        _lib.check(lib.gnnml3_collate_graphs(
            P(idx), P(n), P(node_off), P(xc), C, wh, P(x), F, P(e) if sup else None, P(edge_off) if sup else None,
            P(el) if sup else None, el.element_size() if sup else 0, el.size(1) if sup else 0, P(ea), K, P(m),
            P(adj_off) if adj else None, P(al) if adj else None, al.element_size() if adj else 0, al.size(1) if adj else 0, int(B),
            Np, Ep, Mp, P(out.x), P(out.edge_index2) if sup else None, P(out.edge_attr2) if sup else None,
            P(out.edge_index) if adj else None, P(out.batch), P(out.graph_ptr), P(ws), ws.numel(), _lib.stream_ptr()),
            "gnnml3_collate_graphs")
    return out


def segment_pool_fwd(x, graph_ptr, mean):
    lib = _lib.load()
    x = _f32c(x, "x")
    B, F = graph_ptr.numel() - 1, x.size(1)
    out = torch.empty(B, F, dtype=torch.float32, device=x.device)
    with _on(x.device):
        _lib.check(lib.gnnml3_segment_pool_fwd(_lib.ptr(x), _ld(x), _lib.ptr(graph_ptr), B, F, int(mean), _lib.ptr(out),
                                               _lib.stream_ptr()), "gnnml3_segment_pool_fwd")
    return out


def segment_pool_bwd(gout, graph_ptr, mean, N):
    lib = _lib.load()
    gout = _f32c(gout, "gout")
    B, F = gout.shape
    gx = torch.empty(N, F, dtype=torch.float32, device=gout.device)
    with _on(gout.device):
        _lib.check(lib.gnnml3_segment_pool_bwd(_lib.ptr(gout), _lib.ptr(graph_ptr), B, F, int(mean), _lib.ptr(gx), _ld(gx),
                                               _lib.stream_ptr()), "gnnml3_segment_pool_bwd")
    return gx


def segment_max_fwd(x, graph_ptr):
    lib = _lib.load()
    x = _f32c(x, "x")
    B, F = graph_ptr.numel() - 1, x.size(1)
    out = torch.empty(B, F, dtype=torch.float32, device=x.device)
    arg = torch.empty(B, F, dtype=torch.int32, device=x.device)
    with _on(x.device):
        _lib.check(lib.gnnml3_segment_max_fwd(_lib.ptr(x), _ld(x), _lib.ptr(graph_ptr), B, F, _lib.ptr(out), _lib.ptr(arg),
                                              _lib.stream_ptr()), "gnnml3_segment_max_fwd")
    return out, arg


def segment_max_bwd(gout, arg, graph_ptr, N):
    lib = _lib.load()
    gout = _f32c(gout, "gout")
    B, F = gout.shape
    gx = torch.empty(N, F, dtype=torch.float32, device=gout.device)
    with _on(gout.device):
        _lib.check(lib.gnnml3_segment_max_bwd(_lib.ptr(gout), _lib.ptr(arg), _lib.ptr(graph_ptr), B, F, _lib.ptr(gx), _ld(gx),
                                              _lib.stream_ptr()), "gnnml3_segment_max_bwd")
    return gx


def _bn_cnt(cnt, device):
    if cnt.dtype != torch.int32 or cnt.numel() != 1 or cnt.device != device:
        raise RuntimeError("cnt must be a one-element int32 tensor on %s" % device)
    return cnt


def bn_rows_fwd(x, cnt, weight, bias, running_mean, running_var, num_batches_tracked, eps, momentum):
    """Training-mode BatchNorm over the first ``cnt`` rows of x [N, F] (``cnt``: one-element int32 CUDA tensor, read on the
    device); running buffers updated in place.  -> (y [N, F], save_mean [F], save_invstd [F])."""
    lib = _lib.load()
    x = _rows(x, "x")
    N, F = x.shape
    cnt = _bn_cnt(cnt, x.device)
    for t, name in ((weight, "weight"), (bias, "bias"), (running_mean, "running_mean"), (running_var, "running_var")):
        if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != F or t.device != x.device:
            raise RuntimeError("%s must be a contiguous float32 [%d] tensor on %s" % (name, F, x.device))
    if num_batches_tracked.dtype != torch.int64 or num_batches_tracked.numel() != 1 or num_batches_tracked.device != x.device:
        raise RuntimeError("num_batches_tracked must be a one-element int64 tensor on %s" % x.device)
    y = torch.empty(N, F, dtype=torch.float32, device=x.device)
    mean = torch.empty(F, dtype=torch.float32, device=x.device)
    invstd = torch.empty(F, dtype=torch.float32, device=x.device)
    with _on(x.device):
        nb = lib.gnnml3_bn_rows_workspace_bytes(N, F)
        ws = _ws(x.device, nb, "bn")
        _lib.check(lib.gnnml3_bn_rows_fwd(_lib.ptr(x), _ld(x), N, F, _lib.ptr(cnt), _lib.ptr(weight), _lib.ptr(bias), float(eps),
                                          float(momentum), _lib.ptr(running_mean), _lib.ptr(running_var),
                                          _lib.ptr(num_batches_tracked), _lib.ptr(y), F, _lib.ptr(mean), _lib.ptr(invstd),
                                          _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "gnnml3_bn_rows_fwd")
    return y, mean, invstd


def bn_rows_bwd(x, gy, cnt, weight, save_mean, save_invstd):
    """Backward of ``bn_rows_fwd``: -> (dx [N, F] with zero rows from ``cnt`` on, dweight [F], dbias [F])."""
    lib = _lib.load()
    x, gy = _rows(x, "x"), _rows(gy, "gy")
    N, F = x.shape
    cnt = _bn_cnt(cnt, x.device)
    dx = torch.empty(N, F, dtype=torch.float32, device=x.device)
    dw = torch.empty(F, dtype=torch.float32, device=x.device)
    db = torch.empty(F, dtype=torch.float32, device=x.device)
    with _on(x.device):
        nb = lib.gnnml3_bn_rows_workspace_bytes(N, F)
        ws = _ws(x.device, nb, "bn")
        _lib.check(lib.gnnml3_bn_rows_bwd(_lib.ptr(x), _ld(x), _lib.ptr(gy), _ld(gy), N, F, _lib.ptr(cnt), _lib.ptr(weight),
                                          _lib.ptr(save_mean), _lib.ptr(save_invstd), _lib.ptr(dx), F, _lib.ptr(dw), _lib.ptr(db),
                                          _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "gnnml3_bn_rows_bwd")
    return dx, dw, db


def pairs_mark(emb, bits, wpr, threshold, pairs=None):
    """OR one seed's embeddings emb [n, d] (float32 CUDA, unit-stride rows) into the pair bitmap ``bits`` (int32 words read as
    uint32): all pairs i < j (``pairs`` None, ``wpr`` words per row) or the listed pairs ``pairs`` [P, 2] int64."""
    lib = _lib.load()
    emb = _rows(emb, "emb")
    n, d = emb.shape
    P = 0 if pairs is None else pairs.size(0)
    with _on(emb.device):
        _lib.check(lib.gnnml3_pairs_mark(_lib.ptr(emb), _ld(emb), n, d, _lib.ptr(pairs), P, float(threshold), _lib.ptr(bits), wpr,
                                         _lib.stream_ptr()), "gnnml3_pairs_mark")


def pairs_count(bits, n, wpr, P, out):
    """out (int64 CUDA scalar) = the pairs of the bitmap whose bit is still 0 (P == 0: all pairs of n rows; P > 0: P listed pairs)."""
    lib = _lib.load()
    with _on(bits.device):
        _lib.check(lib.gnnml3_pairs_count(_lib.ptr(bits), n, wpr, P, _lib.ptr(out), _lib.stream_ptr()), "gnnml3_pairs_count")
    return out


# --------------------------------------------------------------------------------------------------
# optional per-call device timing (CUDA events on the launching stream) used by bench.py
# --------------------------------------------------------------------------------------------------
_prof = {"enabled": False, "names": None, "records": [], "last_bytes": None}


def profile_start(names=None):
    _prof["enabled"], _prof["names"], _prof["records"] = True, (set(names) if names else None), []


def profile_stop():
    """-> list of (name, milliseconds, shapes); synchronises the device."""
    _prof["enabled"] = False
    torch.cuda.synchronize()
    out = [(n, s.elapsed_time(e), shp) for n, s, e, shp in _prof["records"]]
    _prof["records"] = []
    return out


def _instrument(name, fn):
    def wrapped(*a, **k):
        if not _prof["enabled"] or (_prof["names"] is not None and name not in _prof["names"]):
            return fn(*a, **k)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = fn(*a, **k)
        e.record()
        shapes = tuple(tuple(t.shape) for t in a if isinstance(t, torch.Tensor))
        if name == "fused_agg_proj":
            shapes = ("algorithmic_bytes", _prof["last_bytes"])
        _prof["records"].append((name, s, e, shapes))
        return out
    wrapped.__name__ = fn.__name__
    wrapped.__doc__ = fn.__doc__
    return wrapped


for _n in ("csr_build", "gather_rows", "scatter_rows", "spmm_k", "spmm_projected", "sddmm_k", "gemm_nn_tc", "gemm_nn", "gemm_tn", "colsum", "edge_mlp_fwd",
           "edge_mlp_bwd", "ml3_act_fwd", "ml3_act_bwd", "ml3_act_bwd_y", "fused_agg_proj", "fused_sddmm", "ml3layer_forward", "ml3layer_backward", "segment_pool_fwd",
           "segment_pool_bwd", "bn_rows_fwd", "bn_rows_bwd"):
    globals()[_n] = _instrument(_n, globals()[_n])
