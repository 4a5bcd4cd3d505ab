"""ctypes binding of libgnnml3_b200.so (the C ABI declared in include/gnnml3_b200.h).

This is the binding a maintainer of the reference would add (see INTEGRATION.md): the reference is pure
Python, so its "FFI" for the hot path is a ctypes stub that hands raw device pointers, sizes and the current
CUDA stream to the library.  There is NO fallback: if the shared library is missing or a call fails, a
RuntimeError is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GNNML3_LIB", os.path.join(_HERE, "libgnnml3_b200.so"))   # override: experiments only

_p = ctypes.c_void_p
_i64 = ctypes.c_int64
_i = ctypes.c_int
_sz = ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol include/gnnml3_b200.h declares (tests check this)
SIGNATURES = {
    "gnnml3_last_error": (ctypes.c_char_p, []),
    "gnnml3_version": (_i, []),
    "gnnml3_launch_count": (_i64, []),
    "gnnml3_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "gnnml3_csr_build": (_i, [_p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gnnml3_gather_rows": (_i, [_p, _p, _i64, _i, _p, _p]),
    "gnnml3_scatter_rows": (_i, [_p, _p, _i64, _i, _p, _p]),
    "gnnml3_spmm_k": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i, _i, _p, _i64, _p]),
    "gnnml3_spmm_projected": (_i, [_p, _p, _p, _p, _i, _p, _i64, _i64, _i, _p, _p, _i64, _p]),
    "gnnml3_sddmm_k": (_i, [_p, _p, _p, _p, _i64, _p, _i64, _i64, _i, _i, _p, _p]),
    "gnnml3_gemm_nn": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i64, _i, _i, _i, _i, _p]),
    "gnnml3_gemm_tn_workspace_bytes": (_sz, [_i64, _i, _i]),
    "gnnml3_gemm_tn": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i, _i, _i, _p, _sz, _p]),
    "gnnml3_gemm_nn_tc_supported": (_i, [_i64, _i, _i]),
    "gnnml3_gemm_nn_tc_workspace_bytes": (_sz, [_i, _i]),
    "gnnml3_gemm_nn_tc": (_i, [_p, _i64, _p, _i64, _p, _p, _i64, _i64, _i, _i, _i, _i, _p, _sz, _p]),
    "gnnml3_colsum_workspace_bytes": (_sz, [_i64, _i]),
    "gnnml3_colsum": (_i, [_p, _i64, _i64, _i, _p, _p, _sz, _p]),
    "gnnml3_edge_mlp_supported": (_i, [_i, _i]),
    "gnnml3_collate_workspace_bytes": (_sz, [_i]),
    "gnnml3_collate": (_i, [_p, _p, _p, _p, _p, _p, _i, _p, _p, _i, _p, _i, _i64, _p, _i, _i, _i64, _i64, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gnnml3_collate_graphs_workspace_bytes": (_sz, [_i]),
    "gnnml3_collate_graphs": (_i, [_p, _p, _p, _p, _i, _p, _p, _i, _p, _p, _p, _i, _i64, _p, _i, _p, _p, _p, _i, _i64, _i, _i64, _i64, _i64,
                                   _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gnnml3_edge_mlp_set_tc": (_i, [_i]),
    "gnnml3_edge_mlp_path_counts": (_i, [_p, _i]),
    "gnnml3_edge_mlp_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, _i, _p, _p]),
    "gnnml3_edge_mlp_bwd_workspace_bytes": (_sz, [_i64, _i]),
    "gnnml3_edge_mlp_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gnnml3_ml3_act_fwd": (_i, [_p, _i64, _i64, _i, _i, _p, _i64, _p]),
    "gnnml3_ml3_act_bwd_workspace_bytes": (_sz, [_i64, _i, _i]),
    "gnnml3_ml3_act_bwd": (_i, [_p, _i64, _p, _i64, _i64, _i, _i, _p, _i64, _p, _i64, _p, _p, _sz, _p]),
    "gnnml3_ml3_act_bwd_y": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i, _i, _p, _i64, _p, _p, _sz, _p]),
    "gnnml3_fused_debug_counters": (_i, [_p, _i]),
    "gnnml3_fused_set_mode": (_i, [_i]),
    "gnnml3_fused_profile": (_i, [_i]),
    "gnnml3_fused_profile_fetch": (_i, [_p, _i]),
    "gnnml3_fused_supported": (_i, [_i, _i, _i, _i, _i, _i, _i]),
    "gnnml3_fused_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "gnnml3_fused_agg_proj": (_i, [_p, _p, _p, _p, _i, _i, _p, _i64, _i, _p, _i64, _i, _i, _p, _i64, _p, _i64, _i, _p, _p,
                                   _i64, _i, _p, _i64, _p, _i64, _i, _i, _p, _i64, _p, _p, _sz, _p]),
    "gnnml3_tile_rows": (_i, []),
    "gnnml3_tile_windows": (_i, [_p, _p, _i64, _p, _p]),
    "gnnml3_fused_ts_supported": (_i, [_i, _i, _i, _i, _i, _i, _i]),
    "gnnml3_fused_ts_workspace_bytes": (_sz, [_i, _i, _i]),
    "gnnml3_fused_set_ts": (_i, [_i]),
    "gnnml3_fused_path_counts": (_i, [_p, _i]),
    "gnnml3_fused_sddmm_supported": (_i, [_i, _i, _i]),
    "gnnml3_fused_sddmm_workspace_bytes": (_sz, [_i]),
    "gnnml3_fused_sddmm": (_i, [_p, _p, _p, _p, _i64, _i, _p, _i64, _i, _p, _i, _i64, _p, _p, _sz, _p]),
    "gnnml3_ml3layer_supported": (_i, [_i, _i, _i, _i, _i]),
    "gnnml3_ml3layer_workspace_bytes": (_sz, [_i64, _i64, _i, _i, _i, _i]),
    "gnnml3_ml3layer_forward": (_i, [_p, _p, _p, _i64, _i64, _p, _i64, _i, _p, _i, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _p, _p,
                                     _i64, _p, _p, _i64, _p, _sz, _p]),
    "gnnml3_ml3layer_backward": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _p, _i64, _i, _p, _p, _i, _p, _p, _p, _p, _p, _i, _p, _p, _i,
                                      _p, _i64, _p, _p, _i64, _i, _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _sz, _p]),
    "gnnml3_ml1layer_supported": (_i, [_i, _i, _i]),
    "gnnml3_ml1layer_workspace_bytes": (_sz, [_i64, _i, _i, _i]),
    "gnnml3_ml1layer_forward": (_i, [_p, _p, _i64, _i64, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _p, _i64, _p, _i64,
                                     _p, _i64, _p, _sz, _p]),
    "gnnml3_ml1layer_backward": (_i, [_p, _p, _i64, _i64, _p, _i64, _i, _p, _p, _p, _p, _i, _i, _p, _i64, _p, _i64, _p, _i64, _i,
                                      _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gnnml3_ml1layer_forward_precision": (_i, [_p, _p, _i64, _i64, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _p, _i64, _p,
                                               _i64, _p, _i64, _p, _sz, _p, _i]),
    "gnnml3_ml1layer_backward_precision": (_i, [_p, _p, _i64, _i64, _p, _i64, _i, _p, _p, _p, _p, _i, _i, _p, _i64, _p, _i64, _p, _i64,
                                                _i, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _i]),
    "gnnml3_segment_pool_fwd":(_i, [_p, _i64, _p, _i, _i, _i, _p, _p]),
    "gnnml3_segment_pool_bwd": (_i, [_p, _p, _i, _i, _i, _p, _i64, _p]),
    "gnnml3_segment_max_fwd": (_i, [_p, _i64, _p, _i, _i, _p, _p, _p]),
    "gnnml3_segment_max_bwd": (_i, [_p, _p, _p, _i, _i, _p, _i64, _p]),
    "gnnml3_spectral_max_nodes": (_i, [_i]),
    "gnnml3_spectral_count": (_i, [_p, _i64, _p, _p, _i, _i, _i, _p, _p]),
    "gnnml3_spectral_design": (_i, [_p, _i64, _p, _p, _i, _i, ctypes.c_double, _i, _i, _i, _i, ctypes.c_double, _i, _p, _i, _p,
                                    _i64, _p, _p, _p, _p]),
    "gnnml3_pairs_mark": (_i, [_p, _i64, _i64, _i, _p, _i64, ctypes.c_float, _p, _i64, _p]),
    "gnnml3_pairs_count": (_i, [_p, _i64, _i64, _i64, _p, _p]),
}

PREC_3XTF32 = 0
PREC_TF32 = 1
PREC_BF16 = 2          # fused layer kernels only (GNNML3_FUSED_BF16, the GNNML1 layer); the stand-alone GEMMs run it as single-pass TF32
FUSED_FLAGS = {0: 0, 1: 0x100, 2: 0x200}
EPI_NONE = 0
EPI_RELU = 1

_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "gnn_matlang_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C gnn_matlang_b200/csrc`).  There is no CPU / PyTorch fallback for the hot path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().gnnml3_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def stream_ptr():
    """cudaStream_t of the current stream of the current device (raw fast path: torch.cuda.current_stream() builds a Python
    Stream object per call, ~15 us)."""
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


def ptr(t):
    """Device pointer of a tensor (None -> NULL); refuses non-CUDA tensors: there is no CPU path."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("gnn_matlang_b200: expected a CUDA tensor (the hot path has no CPU fallback)")
    return t.data_ptr()


def launch_count():
    return int(load().gnnml3_launch_count())
