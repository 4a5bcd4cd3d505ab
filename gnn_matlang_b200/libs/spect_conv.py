"""Drop-in replacements for the reference's ``libs/spect_conv.py`` modules (same import path suffix, same
constructor / forward signatures, parameter names, shapes, initialisation and ``state_dict`` keys):

    from gnn_matlang_b200.libs.spect_conv import SpectConv, ML3Layer

* ``SpectConv(in_channels, out_channels, K=1, selfconn=True, depthwise=False, bias=True)``
  -- reference libs/spect_conv.py:23-103 (a PyG ``MessagePassing`` module there).
* ``ML3Layer(learnedge, nedgeinput, nedgeoutput, ninp, nout1, nout2)`` -- reference libs/spect_conv.py:182-212.
* ``ML1Layer(ninp, nout, concat=False)`` -- the GNNML1 layer the reference's experiment scripts define next to GNNML3
  (``SpectConv`` K=1 on all-ones edge weights + three ``nn.Linear``), as one fused library call per direction.

What runs underneath is different: instead of K x (index_select, mul, scatter_add, matmul, add) the batch's
edge list is turned once into a dst-sorted CSR (``graph.GraphPlan``), one segmented-reduction kernel applies
all K edge-weight channels, and the per-support projections are ONE tensor-core contraction over K*F_in.
The backward is atomic-free and deterministic:  with G_k = S_k^T grad_out (the same kernel over the
transposed CSR)  dx = [G_0..G_{K-1}] W'^T,  dW_k = x^T G_k,  d edge_attr = SDDMM(x, grad_out W^T).
All arithmetic happens in libgnnml3_b200.so; there is no CPU fallback (CPU tensors raise RuntimeError).
"""
import math
import os

import torch
import torch.nn as nn
from torch.nn import Parameter

from .. import _lib, ops
from ..graph import get_plan, sorted_edge_attr

_PRECISIONS = {"fp32": _lib.PREC_3XTF32, "3xtf32": _lib.PREC_3XTF32, "tf32": _lib.PREC_TF32, "bf16": _lib.PREC_BF16}
USE_FUSED = os.environ.get("GNNML3_NO_FUSED", "0") != "1"
USE_LAYER_API = os.environ.get("GNNML3_NO_LAYER_API", "0") != "1"
# first layer (no gradient w.r.t. x): keep the forward aggregate for the weight gradient (GNNML3_KEEP_AGGREGATE=0 restores the
# SpMM over the transposed CSR in the backward)
KEEP_FIRST_LAYER_AGGREGATE = os.environ.get("GNNML3_KEEP_AGGREGATE", "1") != "0"


def _precision_code(precision):
    """The library's PREC_* code of a precision name ("fp32" = "3xtf32", "tf32", "bf16"); ValueError for any other value."""
    if precision not in _PRECISIONS:
        raise ValueError("precision must be one of %s" % sorted(_PRECISIONS))
    return _PRECISIONS[precision]


def _fused_ok(precision, K, Kstride, F, Nc, Fs=0, self_mode=0, Ns=0):
    """The fused layer kernels cover this shape in ``precision``: 3xTF32 in both generations, the flagged single-pass TF32 and
    BF16 modes in the tensor-memory generation only."""
    if precision == _lib.PREC_3XTF32:
        return ops.fused_supported(K, Kstride, F, Nc, Fs, self_mode, Ns)
    return ops.fused_ts_supported(K, Kstride, F, Nc, Fs, self_mode, Ns)


def glorot(tensor):
    """reference libs/spect_conv.py:13-16"""
    if tensor is not None:
        stdv = math.sqrt(6.0 / (tensor.size(-2) + tensor.size(-1)))
        tensor.data.uniform_(-stdv, stdv)


def zeros(tensor):
    """reference libs/spect_conv.py:18-20"""
    if tensor is not None:
        tensor.data.fill_(0)


def _aggregate(plan, ea_s, x, width_blocks, transposed=False):
    """[N, width_blocks*F] buffer whose first K blocks are the K-channel aggregates of ``x``."""
    N, F = x.shape
    K = ea_s.size(1)
    out = torch.empty(N, width_blocks * F, dtype=torch.float32, device=x.device)
    if plan.E == 0:
        out[:, :K * F].zero_()
    elif transposed:
        ops.spmm_k(plan.rowptrT, plan.colT, plan.permT, ea_s, x, out=out)
    else:
        ops.spmm_k(plan.rowptr, plan.col, None, ea_s, x, out=out)
    return out


class _SpectConvFn(torch.autograd.Function):
    """out = sum_k P_k(x) W_k (+ x W_K if selfconn) (+ bias)   -- reference libs/spect_conv.py:70-80,93-94.

    Forward and d x run as ONE fused tcgen05 kernel each (aggregate + projection, the [N, K*Fi] aggregate never exists;
    selfconn rides along as one more k-block); d edge_attr through the fused dH + SDDMM kernel; shapes outside the fused
    kernels' envelope take the two-kernel path (SpMM + GEMM)."""

    @staticmethod
    def forward(ctx, x, ea_s, weight, bias, plan, selfconn, precision):
        if x.stride(1) != 1:
            x = x.contiguous()
        ea_s = ea_s.contiguous()
        weight = weight.contiguous()
        N, Fi = x.shape
        Kw, _, Fo = weight.shape
        K = ea_s.size(1)
        fused = (USE_FUSED and N > 0 and plan.E > 0 and (not selfconn or Fi <= 32)
                 and _fused_ok(precision, K, K, Fi, Fo, Fi if selfconn else 0, 2 if selfconn else 0, 0))
        ctx.plan, ctx.selfconn, ctx.precision, ctx.has_bias = plan, selfconn, precision, bias is not None
        ctx.fused = fused
        if fused:
            x = ops.aligned_rows(x)
            out, _ = ops.fused_agg_proj(plan.rowptr, plan.col, None, ea_s, x, weight[:K].reshape(K * Fi, Fo), bias=bias,
                                        S=x if selfconn else None, self_mode=2 if selfconn else 0,
                                        Bself=weight[K] if selfconn else None, epilogue=0, win=plan.win, precision=precision)
        else:
            H = _aggregate(plan, ea_s, x, Kw)
            if selfconn:
                H[:, K * Fi:] = x
            out = ops.gemm_nn(H, weight.view(Kw * Fi, Fo), bias, precision=precision)
        ctx.save_for_backward(x, ea_s, weight)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, ea_s, weight = ctx.saved_tensors
        plan, prec = ctx.plan, ctx.precision
        N, Fi = x.shape
        Kw, _, Fo = weight.shape
        K = ea_s.size(1)
        need_x, need_ea, need_w, need_b = ctx.needs_input_grad[:4]
        dx = dea = dw = db = None
        if N == 0:
            return (torch.zeros_like(x) if need_x else None, torch.zeros_like(ea_s) if need_ea else None,
                    torch.zeros_like(weight) if need_w else None,
                    torch.zeros(Fo, device=x.device) if (need_b and ctx.has_bias) else None, None, None, None)
        gout = ops.aligned_rows(gout) if ctx.fused else gout.contiguous()
        fused_dx = (ctx.fused and need_x and (not ctx.selfconn or Fo <= 32)
                    and _fused_ok(prec, K, K, Fo, Fi, Fo if ctx.selfconn else 0, 2 if ctx.selfconn else 0, 0))
        G = None
        if fused_dx:
            # dx = sum_k S_k^T gout W_k^T (+ gout W_K^T): the same fused kernel over the transposed CSR; when the weight
            # gradient is wanted too it leaves the aggregate G' = [S_0^T gout .. | gout] behind (no separate SpMM)
            Fp = (Fo + 31) // 32 * 32
            side = need_w and ops.fused_side_output_ok()
            if side:
                G = torch.empty(N, (K + (1 if ctx.selfconn else 0)) * Fp, dtype=torch.float32, device=x.device)
            dx, _ = ops.fused_agg_proj(plan.rowptrT, plan.colT, plan.permT, ea_s, gout,
                                       weight[:K].transpose(1, 2).reshape(K * Fo, Fi).contiguous(),
                                       S=gout if ctx.selfconn else None, self_mode=2 if ctx.selfconn else 0,
                                       Bself=weight[K].t().contiguous() if ctx.selfconn else None, epilogue=0, hout=G,
                                       win=plan.winT, precision=prec)
            if side:
                dcat = ops.gemm_tn(x, G, precision=prec)                                          # [Fi, Kw * Fp]
                dw = dcat.view(Fi, Kw, Fp)[:, :, :Fo].permute(1, 0, 2).contiguous()
                need_w = False
        if need_w or (need_x and not fused_dx):
            G = _aggregate(plan, ea_s, gout, Kw, transposed=True)           # G_k = S_k^T gout  [N, Kw*Fo]
            if ctx.selfconn:
                G[:, K * Fo:] = gout
            if need_x and not fused_dx:
                dx = ops.gemm_nn(G, weight.transpose(1, 2).contiguous().view(Kw * Fo, Fi), precision=prec)
            if need_w:
                dw = ops.gemm_tn(x, G, precision=prec).view(Fi, Kw, Fo).permute(1, 0, 2).contiguous()
        if need_b and ctx.has_bias:
            db = ops.colsum(gout)
        if need_ea:
            if plan.E == 0:
                dea = torch.zeros_like(ea_s)
            elif ctx.fused and ops.fused_sddmm_supported(K, Fi, Fo):      # (FP32-grade in every mode)
                dea = ops.fused_sddmm(plan.rowptr, plan.col, x, gout, weight[:K].contiguous(), plan.E, win=plan.win)
            else:
                wp = weight[:K].permute(2, 0, 1).reshape(Fo, K * Fi).contiguous()
                dH = ops.gemm_nn(gout, wp, precision=prec)                   # [N, K*Fi]
                dea = ops.sddmm_k(plan.rowptr, plan.col, None, x, dH, K, plan.E)
        return dx, dea, dw, db, None, None, None


class _SpectConvProjectFirstFn(torch.autograd.Function):
    """Project-first order of the same layer (north_star: "or alternatively pre-projects and then aggregates"):

        Y = x [W_0 .. W_{K-1}]  ([N, K*Fo], one tensor-core GEMM);   out[t] = sum_{e: dst_e = t} sum_k ea[e, k] Y[src_e, k, :]  (+ bias)

    -- reference libs/spect_conv.py:70-80 with the sum over k moved inside the edge sum.  Backward, atomic-free:
    dY = [S_0^T gout .. S_{K-1}^T gout] (the K-channel aggregation over the transposed CSR), dx = dY Wcat^T, dWcat = x^T dY,
    d ea[e, k] = <Y[src_e, k, :], gout[dst_e]> (SDDMM over the transposed CSR)."""

    @staticmethod
    def forward(ctx, x, ea_s, weight, bias, plan, precision):
        x, ea_s = x.contiguous(), ea_s.contiguous()
        K, Fi, Fo = weight.shape
        wcat = weight.permute(1, 0, 2).reshape(Fi, K * Fo).contiguous()
        Y = ops.gemm_nn(x, wcat, precision=precision)
        if plan.E == 0:
            out = torch.zeros(x.size(0), Fo, device=x.device) + (bias if bias is not None else 0)
        else:
            out = ops.spmm_projected(plan.rowptr, plan.col, None, ea_s, Y, Fo, bias)
        ctx.save_for_backward(x, ea_s, wcat, Y)
        ctx.plan, ctx.precision, ctx.has_bias, ctx.shape = plan, precision, bias is not None, (K, Fi, Fo)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, ea_s, wcat, Y = ctx.saved_tensors
        plan, prec = ctx.plan, ctx.precision
        K, Fi, Fo = ctx.shape
        gout = gout.contiguous()
        dY = _aggregate(plan, ea_s, gout, K, transposed=True)                       # [N, K*Fo]
        dx = ops.gemm_nn(dY, wcat.t().contiguous(), precision=prec) if ctx.needs_input_grad[0] else None
        dw = None
        if ctx.needs_input_grad[2]:
            dw = ops.gemm_tn(x, dY, precision=prec).view(Fi, K, Fo).permute(1, 0, 2).contiguous()
        dea = None
        if ctx.needs_input_grad[1]:
            dea = (torch.zeros_like(ea_s) if plan.E == 0 else
                   ops.sddmm_k(plan.rowptrT, plan.colT, plan.permT, gout, Y, K, plan.E))
        db = ops.colsum(gout) if (ctx.has_bias and ctx.needs_input_grad[3]) else None
        return dx, dea, dw, db, None, None


def project_first_pays(N, E, K, Fi, Fo):
    """HBM words moved by the aggregation side of the two orders when H = [P_0(x) .. P_{K-1}(x)] / Y = x [W_0 ..] round-trips
    through HBM (the two-kernel designs): aggregate-first gathers Fi words per support entry and writes + reads H [N, K*Fi];
    project-first gathers K*Fo words per entry and writes + reads Y [N, K*Fo].  The GEMM flops are the same."""
    return K * Fo * (E + 2 * N) < Fi * (E + 2 * N * K)


class _AggregateFn(torch.autograd.Function):
    """H = [P_0(x) .. P_{K-1}(x)]  ([N, K*F]) with gradients: dx[s] = sum_{e: src_e = s} sum_k ea[e, k] dH[dst_e, k, :] (the
    project-first aggregation kernel over the transposed CSR), d ea[e, k] = <x[src_e], dH[dst_e, k, :]> (SDDMM)."""

    @staticmethod
    def forward(ctx, x, ea_s, plan):
        x, ea_s = x.contiguous(), ea_s.contiguous()
        ctx.save_for_backward(x, ea_s)
        ctx.plan = plan
        return _aggregate(plan, ea_s, x, ea_s.size(1))

    @staticmethod
    def backward(ctx, dH):
        x, ea_s = ctx.saved_tensors
        plan = ctx.plan
        dH = dH.contiguous()
        K, F = ea_s.size(1), x.size(1)
        if plan.E == 0:
            return torch.zeros_like(x), torch.zeros_like(ea_s), None
        dx = ops.spmm_projected(plan.rowptrT, plan.colT, plan.permT, ea_s, dH, F) if ctx.needs_input_grad[0] else None
        dea = ops.sddmm_k(plan.rowptr, plan.col, None, x, dH, K, plan.E) if ctx.needs_input_grad[1] else None
        return dx, dea, None


class _DepthwiseAggFn(torch.autograd.Function):
    """Z = sum_k scale[k] * P_k(x)   -- the aggregation of the depthwise branch (reference :81-89)."""

    @staticmethod
    def forward(ctx, x, ea_s, scale, plan):
        x, ea_s, scale = x.contiguous(), ea_s.contiguous(), scale.contiguous()
        N, F = x.shape
        K = ea_s.size(1)
        H = _aggregate(plan, ea_s, x, K)
        ctx.save_for_backward(x, ea_s, scale, H)
        ctx.plan = plan
        return (H.view(N, K, F) * scale.unsqueeze(0)).sum(1)

    @staticmethod
    def backward(ctx, dZ):
        x, ea_s, scale, H = ctx.saved_tensors
        plan = ctx.plan
        dZ = dZ.contiguous()
        N, F = x.shape
        K = ea_s.size(1)
        G = _aggregate(plan, ea_s, dZ, K, transposed=True)
        dx = (G.view(N, K, F) * scale.unsqueeze(0)).sum(1)
        dscale = (H.view(N, K, F) * dZ.unsqueeze(1)).sum(0)
        if plan.E == 0:
            dea = torch.zeros_like(ea_s)
        else:
            g = (dZ.unsqueeze(1) * scale.unsqueeze(0)).reshape(N, K * F).contiguous()
            dea = ops.sddmm_k(plan.rowptr, plan.col, None, x, g, K, plan.E)
        return dx, dea, dscale, None


class _LinearFn(torch.autograd.Function):
    """y = x @ Wt (+ b) with Wt [in, out]; tensor-core GEMMs of this library in both directions."""

    @staticmethod
    def forward(ctx, x, wt, bias, precision):
        x, wt = x.contiguous(), wt.contiguous()
        ctx.save_for_backward(x, wt)
        ctx.precision, ctx.has_bias = precision, bias is not None
        return ops.gemm_nn(x, wt, bias, precision=precision)

    @staticmethod
    def backward(ctx, g):
        x, wt = ctx.saved_tensors
        g = g.contiguous()
        dx = dw = db = None
        if x.size(0) == 0:
            return torch.zeros_like(x), torch.zeros_like(wt), (torch.zeros(wt.size(1), device=x.device) if ctx.has_bias else None), None
        if ctx.needs_input_grad[0]:
            dx = ops.gemm_nn(g, wt.t().contiguous(), precision=ctx.precision)
        if ctx.needs_input_grad[1]:
            dw = ops.gemm_tn(x, g, precision=ctx.precision)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = ops.colsum(g)
        return dx, dw, db, None


class _ML3LayerFn(torch.autograd.Function):
    """Whole ML3Layer (reference libs/spect_conv.py:204-212) as one autograd node:

        ea' = edge_mlp(ea)                       (fused per-edge kernel; skipped if ``fused_edge`` is False)
        pre = [ [P_0(x)..P_{K-1}(x)] Wc + b | x W11^T + b11 | x W12^T + b12 ]
        y   = [ relu(pre_c) || tanh(pre_1) * tanh(pre_2) ]

    Backward (atomic-free): d pre from the activation kernel; G' = [S_0^T gc .. S_{K-1}^T gc | gp1 | gp2];
    dx = G' [Wc'^T ; W11 ; W12];  [dWc | dW11^T | dW12^T] = x^T G';  biases = column sums of d pre;
    d ea' = SDDMM(x, gc Wc^T) and then through the edge MLP (activations recomputed).

    ``save`` (decided by the caller: inside ``forward`` grad mode is always off): False for a forward nobody differentiates
    (``no_grad``, ``inference_mode``, frozen parameters) -- the fused kernels then store y alone (no tanh factors, no aggregate
    side output) and nothing is saved for a backward."""

    @staticmethod
    def forward(ctx, x, ea_s, w1, w2, w3, w4, wconv, bconv, w11, b11, w12, b12, plan, fused_edge, precision, save=True):
        if x.stride(1) != 1:        # row-strided views (padded layer outputs) are consumed as they are
            x = x.contiguous()
        ea_s = ea_s.contiguous()
        wconv = wconv.contiguous()
        N, Fi = x.shape
        K, _, Fo = wconv.shape
        G = 0 if w11 is None else w11.size(0)
        ctx.composite = False
        if (USE_FUSED and precision == _lib.PREC_3XTF32 and USE_LAYER_API and N > 0 and plan.E > 0
                and (fused_edge or w1 is None) and ops.ml3layer_supported(K, Fi, Fo, G, fused_edge)):
            # the whole layer in ONE library call (layer_api.cu): same kernels as below, a fraction of the host time
            xa = ops.aligned_rows(x)
            ws4 = tuple(w.contiguous() for w in (w1, w2, w3, w4)) if fused_edge else None
            gates = (w11.contiguous(), b11.contiguous(), w12.contiguous(), b12.contiguous()) if G > 0 else None
            # first layer of a model (x carries no gradient, the weights do): the forward also leaves the aggregate behind and the
            # backward takes dW_k = H_k^T gc from it instead of aggregating S_k^T gc over the transposed CSR
            keep = (not ctx.needs_input_grad[0]) and ctx.needs_input_grad[6] and Fi <= 32 and KEEP_FIRST_LAYER_AGGREGATE
            if save:
                y, aux, ea2, hside = ops.ml3layer_forward(plan, xa, ea_s, ws4, wconv, bconv.contiguous() if bconv is not None else None,
                                                          gates, keep_aggregate=keep)
            else:
                y, aux, ea2, hside = ops.ml3layer_forward(plan, xa, ea_s, ws4, wconv, bconv.contiguous() if bconv is not None else None,
                                                          gates, keep_aggregate=False, aux=False)
            ctx.plan, ctx.fused_edge, ctx.precision, ctx.G = plan, fused_edge, precision, G
            ctx.has_bias, ctx.fused, ctx.composite = bconv is not None, True, True
            if save:
                ctx.save_for_backward(xa, ea_s, ea2, y, aux, w1, w2, w3, w4, wconv, w11, w12, hside)
            return y
        if fused_edge:
            w1, w2, w3, w4 = w1.contiguous(), w2.contiguous(), w3.contiguous(), w4.contiguous()
            ea2 = ops.edge_mlp_fwd(ea_s, None, w1, w2, w3, w4)
        else:
            ea2 = ea_s
        fused = (USE_FUSED and N > 0 and plan.E > 0 and (G == 0 or Fi <= 32)
                 and _fused_ok(precision, K, K, Fi, Fo, Fi if G else 0, 1 if G else 0, 2 * G)
                 and _fused_ok(precision, K, K, Fo, Fi, 2 * G, 2 if G else 0, 0))
        ctx.plan, ctx.fused_edge, ctx.precision, ctx.G = plan, fused_edge, precision, G
        ctx.has_bias = bconv is not None
        ctx.fused = fused
        if fused:
            # aggregate + project + gate linears + activations in ONE kernel (fused_layer.cu); H and pre never exist
            xa = ops.aligned_rows(x)
            wg = torch.cat([w11.t(), w12.t()], 1).contiguous() if G > 0 else None
            bg = torch.cat([b11, b12]) if G > 0 else None
            if save:
                y, aux = ops.fused_agg_proj(plan.rowptr, plan.col, None, ea2, xa, wconv.view(K * Fi, Fo), bias=bconv,
                                            S=xa if G > 0 else None, self_mode=1 if G > 0 else 0, Bself=wg, bias_s=bg, G=G,
                                            epilogue=1, win=plan.win, precision=precision)
                ctx.save_for_backward(xa, ea_s, ea2 if fused_edge else None, y, aux, w1, w2, w3, w4, wconv, w11, w12, None)
            else:
                y, _ = ops.fused_agg_proj(plan.rowptr, plan.col, None, ea2, xa, wconv.view(K * Fi, Fo), bias=bconv,
                                          S=xa if G > 0 else None, self_mode=1 if G > 0 else 0, Bself=wg, bias_s=bg, G=G,
                                          epilogue=1, win=plan.win, precision=precision, aux=False)
            return y
        H = _aggregate(plan, ea2, x, K)
        # rows padded to a multiple of 4 floats so that the GEMM epilogues can store 128-bit vectors
        pre = torch.empty(N, (Fo + 2 * G + 3) // 4 * 4, dtype=torch.float32, device=x.device)[:, :Fo + 2 * G]
        if N > 0:
            ops.gemm_nn(H, wconv.view(K * Fi, Fo), bconv, precision=precision, out=pre[:, :Fo])
            if G > 0:
                wg = torch.cat([w11.t(), w12.t()], 1).contiguous()
                ops.gemm_nn(x, wg, torch.cat([b11, b12]), precision=precision, out=pre[:, Fo:])
        y = ops.ml3_act_fwd(pre, Fo, G)
        if save:
            ctx.save_for_backward(x, ea_s, ea2 if fused_edge else None, pre, None, w1, w2, w3, w4, wconv, w11, w12, None)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, ea_s, ea2, pre, aux, w1, w2, w3, w4, wconv, w11, w12, hside = ctx.saved_tensors
        plan, prec, G = ctx.plan, ctx.precision, ctx.G
        if ea2 is None:
            ea2 = ea_s
        N, Fi = x.shape
        K, _, Fo = wconv.shape
        need = ctx.needs_input_grad
        if ctx.composite and N > 0:
            gy = gy if gy.stride(1) == 1 else gy.contiguous()
            ws4 = (w1, w2, w3, w4) if ctx.fused_edge else None
            dx, dea, dws, dwc, dbc, dw11, db11, dw12, db12 = ops.ml3layer_backward(
                plan, x, ea_s, ea2, ws4, wconv, (w11, w12) if G > 0 else None, pre, aux, gy, need[0], need[1], ctx.has_bias, hside=hside)
            return (dx, dea, dws[0], dws[1], dws[2], dws[3], dwc, dbc, dw11, db11, dw12, db12, None, None, None, None)
        gy = gy.contiguous()
        Gp = torch.empty(N, K * Fo + 2 * G, dtype=torch.float32, device=x.device)
        if ctx.fused:
            # `pre` holds the layer OUTPUT y here; gpre = [gc | 0 | g1 g2 | 0] with the gate block at column ceil4(Fo)
            Fo4 = (Fo + 3) // 4 * 4
            gpre, dball = ops.ml3_act_bwd_y(pre, aux, gy, Fo, G)
            if G > 0:
                Gp[:, K * Fo:] = gpre[:, Fo4:Fo4 + 2 * G]
        else:
            gpre, dball = ops.ml3_act_bwd(pre, gy, Fo, G, gate_out=Gp[:, K * Fo:] if G > 0 else None)
        gc = gpre[:, :Fo]
        dx = dea = None
        dws = [None, None, None, None]
        dwc = dbc = dw11 = db11 = dw12 = db12 = None
        if N == 0:
            z = torch.zeros_like
            return (z(x), z(ea_s), *(z(w) if w is not None else None for w in (w1, w2, w3, w4)), z(wconv),
                    torch.zeros(Fo, device=x.device) if ctx.has_bias else None,
                    z(w11) if G else None, torch.zeros(G, device=x.device) if G else None,
                    z(w12) if G else None, torch.zeros(G, device=x.device) if G else None, None, None, None, None)
        if plan.E == 0:
            Gp[:, :K * Fo].zero_()
        else:
            ops.spmm_k(plan.rowptrT, plan.colT, plan.permT, ea2, gc, out=Gp)
        if need[0] and ctx.fused:
            # dx = sum_k S_k^T gc W_k^T + g1 W11 + g2 W12: the fused kernel over the transposed CSR, gate gradients as
            # one more k-block accumulating into the same columns
            dx, _ = ops.fused_agg_proj(plan.rowptrT, plan.colT, plan.permT, ea2, gpre[:, :Fo],
                                       wconv.transpose(1, 2).reshape(K * Fo, Fi).contiguous(),
                                       S=gpre[:, Fo4:Fo4 + 2 * G] if G > 0 else None, self_mode=2 if G > 0 else 0,
                                       Bself=torch.cat([w11, w12], 0).contiguous() if G > 0 else None, epilogue=0,
                                       win=plan.winT, precision=prec)
        elif need[0]:
            blocks = [wconv.transpose(1, 2).reshape(K * Fo, Fi)]
            if G > 0:
                blocks += [w11, w12]
            dx = ops.gemm_nn(Gp, torch.cat(blocks, 0).contiguous(), precision=prec)
        dcat = ops.gemm_tn(x, Gp, precision=prec)                                   # [Fi, K*Fo + 2G]
        dwc = dcat[:, :K * Fo].reshape(Fi, K, Fo).permute(1, 0, 2).contiguous()
        if ctx.has_bias:
            dbc = dball[:Fo].contiguous()
        if G > 0:
            dw11 = dcat[:, K * Fo:K * Fo + G].t().contiguous()
            dw12 = dcat[:, K * Fo + G:].t().contiguous()
            db11 = dball[Fo:Fo + G].contiguous()
            db12 = dball[Fo + G:].contiguous()
        if ctx.fused_edge or need[1]:
            if plan.E == 0:
                dea2 = torch.zeros_like(ea2)
            elif ctx.fused and ops.fused_sddmm_supported(K, Fi, Fo):
                # dH = gc [W_0^T ..] tile by tile in tensor memory / shared memory, consumed in place by the SDDMM
                dea2 = ops.fused_sddmm(plan.rowptr, plan.col, x, gc, wconv, plan.E, win=plan.win)
            else:
                wp = wconv.permute(2, 0, 1).reshape(Fo, K * Fi).contiguous()
                dH = ops.gemm_nn(gc, wp, precision=prec)
                dea2 = ops.sddmm_k(plan.rowptr, plan.col, None, x, dH, K, plan.E)
            if ctx.fused_edge:
                dea, dws = ops.edge_mlp_bwd(ea_s, None, dea2, w1, w2, w3, w4, need_dea=need[1])
            else:
                dea = dea2
        return (dx, dea, dws[0], dws[1], dws[2], dws[3], dwc, dbc, dw11, db11, dw12, db12, None, None, None, None)


def _needs_save(*tensors):
    """Whether a layer's forward must keep what its backward reads: grad mode is on and some input or parameter requires a
    gradient.  Decided before the autograd Function runs -- inside its ``forward`` grad mode is always off, and
    ``ctx.needs_input_grad`` reports ``requires_grad`` whatever the grad mode."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _check_inputs(x, edge_index, edge_attr):
    if not (x.is_cuda and edge_index.is_cuda and edge_attr.is_cuda):
        raise RuntimeError("gnn_matlang_b200: x, edge_index and edge_attr must be CUDA tensors "
                           "(the B200 hot path has no CPU fallback)")
    if x.dim() != 2 or x.dtype != torch.float32 or edge_attr.dtype != torch.float32:
        raise RuntimeError("gnn_matlang_b200: x [N,F] and edge_attr [E,K] must be float32")


class SpectConv(nn.Module):
    r"""Spectral convolution with K supports given as edge features (reference libs/spect_conv.py:23-103).

    ``forward(x, edge_index, edge_attr)``: ``x [N, in]``, ``edge_index [2, E]`` int64 (row 0 source, row 1
    target), ``edge_attr [E, K]``; returns ``[N, out]``.  ``edge_weight``, ``batch`` and ``lambda_max`` are
    accepted and ignored exactly as in the reference (:64-65).
    """

    def __init__(self, in_channels, out_channels, K=1, selfconn=True, depthwise=False, bias=True, **kwargs):
        kwargs.setdefault('aggr', 'add')
        if kwargs.pop('aggr') != 'add':
            raise ValueError("SpectConv only implements aggr='add' (the reference's default, :27)")
        self.precision = kwargs.pop('precision', 'fp32')
        _precision_code(self.precision)
        # 'auto' (default): the fused aggregate-first kernels where they apply, else whichever order moves fewer HBM words
        # (project_first_pays); 'aggregate_first' / 'project_first' force one order (measurements, DESIGN.md section 4.5)
        self.order = kwargs.pop('order', 'auto')
        if self.order not in ('auto', 'aggregate_first', 'project_first'):
            raise ValueError("order must be 'auto', 'aggregate_first' or 'project_first'")
        super(SpectConv, self).__init__()
        assert K > 0
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.depthwise = depthwise
        self.selfconn = selfconn
        if self.selfconn:
            K = K + 1
        if self.depthwise:
            self.DSweight = Parameter(torch.Tensor(K, in_channels))
            self.nsup = K
            K = 1
        self.weight = Parameter(torch.Tensor(K, in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.Tensor(out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot(self.weight)
        zeros(self.bias)
        if self.depthwise:
            zeros(self.DSweight)

    def forward(self, x, edge_index, edge_attr, edge_weight=None, batch=None, lambda_max=None):
        _check_inputs(x, edge_index, edge_attr)
        plan = get_plan(edge_index, x.size(0))
        return self.forward_sorted(x, plan, sorted_edge_attr(edge_attr, plan))

    def forward_sorted(self, x, plan, ea_s):
        """Same as ``forward`` with the graph plan and the dst-sorted edge features already at hand."""
        prec = _precision_code(self.precision)
        if not self.depthwise:
            nk = self.weight.size(0) - (1 if self.selfconn else 0)
            if ea_s.size(1) < nk:
                raise RuntimeError("SpectConv: edge_attr has %d channels but the layer was built with K=%d"
                                   % (ea_s.size(1), nk))
            if ea_s.size(1) > nk:          # the reference only reads edge_attr[:, i] for i < K (:76-77)
                ea_s = ea_s[:, :nk]
            order = self.order
            if order == 'auto':
                Fi, Fo = self.in_channels, self.out_channels
                fused = USE_FUSED and _fused_ok(prec, nk, nk, Fi, Fo, Fi if self.selfconn else 0, 2 if self.selfconn else 0, 0)
                order = 'project_first' if (not fused and Fo <= 256 and project_first_pays(plan.N, plan.E, nk, Fi, Fo)) else 'aggregate_first'
            if order == 'project_first' and self.out_channels <= 256:
                out = _SpectConvProjectFirstFn.apply(x, ea_s, self.weight[:nk], None if self.selfconn else self.bias, plan, prec)
                if self.selfconn:
                    out = out + _LinearFn.apply(x, self.weight[nk], self.bias, prec)
                return out
            return _SpectConvFn.apply(x, ea_s, self.weight, self.bias, plan, self.selfconn, prec)
        nk = self.nsup - (1 if self.selfconn else 0)
        if ea_s.size(1) < nk:
            raise RuntimeError("SpectConv(depthwise): edge_attr has %d channels, need %d" % (ea_s.size(1), nk))
        scale = self.DSweight[:nk] + torch.cat([torch.ones(1, self.in_channels, device=x.device),
                                                torch.zeros(nk - 1, self.in_channels, device=x.device)], 0)
        z = _DepthwiseAggFn.apply(x, ea_s[:, :nk], scale, plan)
        if self.selfconn:
            z = z + x * self.DSweight[-1]
        return _LinearFn.apply(z, self.weight[0], self.bias, prec)

    def __repr__(self):
        return '{}({}, {}, K={})'.format(self.__class__.__name__, self.in_channels, self.out_channels,
                                         self.weight.size(0))


class SpectConCatConv(nn.Module):
    r"""Concatenating variant (reference libs/spect_conv.py:105-165): ``out = [x W_K (if selfconn) || P_0(x) W_0 || .. ||
    P_{K-1}(x) W_{K-1}] + bias`` with ``bias [K' * out]``; same constructor, parameter names / shapes and ``forward`` signature.
    One K-channel aggregation kernel builds every ``P_k(x)``, each block is projected by its own tensor-core GEMM."""

    def __init__(self, in_channels, out_channels, K, selfconn=True, bias=True, **kwargs):
        kwargs.setdefault('aggr', 'add')
        if kwargs.pop('aggr') != 'add':
            raise ValueError("SpectConCatConv only implements aggr='add' (the reference's default, :109)")
        self.precision = kwargs.pop('precision', 'fp32')
        _precision_code(self.precision)
        super(SpectConCatConv, self).__init__()
        assert K > 0
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.selfconn = selfconn
        if self.selfconn:
            K = K + 1
        self.weight = Parameter(torch.Tensor(K, in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.Tensor(K * out_channels))
        else:
            self.register_parameter('bias', None)
        self.reset_parameters()

    def reset_parameters(self):
        glorot(self.weight)
        zeros(self.bias)

    def forward(self, x, edge_index, edge_attr, edge_weight=None, batch=None, lambda_max=None):
        _check_inputs(x, edge_index, edge_attr)
        plan = get_plan(edge_index, x.size(0))
        ea_s = sorted_edge_attr(edge_attr, plan)
        prec = _precision_code(self.precision)
        nk = self.weight.size(0) - (1 if self.selfconn else 0)
        if ea_s.size(1) < nk:
            raise RuntimeError("SpectConCatConv: edge_attr has %d channels but the layer was built with K=%d" % (ea_s.size(1), nk))
        Fi = self.in_channels
        out = []
        if self.selfconn:
            out.append(_LinearFn.apply(x, self.weight[-1], None, prec))
        H = _AggregateFn.apply(x, ea_s[:, :nk], plan)
        for i in range(nk):
            out.append(_LinearFn.apply(H[:, i * Fi:(i + 1) * Fi], self.weight[i], None, prec))
        out = torch.cat(out, 1)
        if self.bias is not None:
            out = out + self.bias
        return out

    def __repr__(self):
        return '{}({}, {}, K={})'.format(self.__class__.__name__, self.in_channels, self.out_channels, self.weight.size(0))


class EdgeEncoder(torch.nn.Module):
    """reference libs/spect_conv.py:168-179 (two ReLU linears on the edge features; unused by the reference's scripts)."""

    def __init__(self, emb_dim):
        super(EdgeEncoder, self).__init__()
        self.fc1 = torch.nn.Linear(emb_dim[0], emb_dim[1])
        self.fc2 = torch.nn.Linear(emb_dim[1], emb_dim[2])

    def forward(self, edge_attr):
        h = torch.relu(_LinearFn.apply(edge_attr, self.fc1.weight.t(), self.fc1.bias, _lib.PREC_3XTF32))
        return torch.relu(_LinearFn.apply(h, self.fc2.weight.t(), self.fc2.bias, _lib.PREC_3XTF32))


class ML3Layer(torch.nn.Module):
    """GNNML3 layer (reference libs/spect_conv.py:182-212): learned edge features, SpectConv, tanh*tanh
    gating branch, concatenation."""

    def __init__(self, learnedge, nedgeinput, nedgeoutput, ninp, nout1, nout2, precision='fp32'):
        super(ML3Layer, self).__init__()
        _precision_code(precision)
        self.learnedge = learnedge
        self.nout2 = nout2
        self.precision = precision
        if self.learnedge:
            self.fc1_1 = torch.nn.Linear(nedgeinput, 2 * nedgeinput, bias=False)
            self.fc1_2 = torch.nn.Linear(nedgeinput, 2 * nedgeinput, bias=False)
            self.fc1_3 = torch.nn.Linear(nedgeinput, 2 * nedgeinput, bias=False)
            self.fc1_4 = torch.nn.Linear(4 * nedgeinput, nedgeoutput, bias=False)
        else:
            nedgeoutput = nedgeinput
        self.conv1 = SpectConv(ninp, nout1, nedgeoutput, selfconn=False, precision=precision)
        if nout2 > 0:
            self.fc11 = torch.nn.Linear(ninp, nout2)
            self.fc12 = torch.nn.Linear(ninp, nout2)

    def forward(self, x, edge_index, edge_attr):
        _check_inputs(x, edge_index, edge_attr)
        plan = get_plan(edge_index, x.size(0))
        ea = sorted_edge_attr(edge_attr, plan)
        prec = _precision_code(self.precision)
        c = self.conv1
        if not self.learnedge and ea.size(1) > c.weight.size(0):
            # the reference's SpectConv reads edge_attr[:, i] for i < K only (libs/spect_conv.py:76-80): extra channels are ignored
            ea = ea[:, :c.weight.size(0)].contiguous()
        if ea.size(1) != (self.fc1_1.in_features if self.learnedge else c.weight.size(0)):
            raise RuntimeError("ML3Layer: edge_attr has %d channels, expected %d"
                               % (ea.size(1), self.fc1_1.in_features if self.learnedge else c.weight.size(0)))
        fused_edge = self.learnedge and ops.edge_mlp_supported(self.fc1_1.in_features, self.fc1_4.out_features)
        if self.learnedge and not fused_edge:
            # shapes outside the fused per-edge kernel (odd K, K > 16, nedgeoutput != nedgeinput): the same MLP
            # composed from this library's tensor-core GEMMs
            tmp = torch.cat([torch.relu(_LinearFn.apply(ea, self.fc1_1.weight.t(), None, prec)),
                             torch.tanh(_LinearFn.apply(ea, self.fc1_2.weight.t(), None, prec)) *
                             torch.tanh(_LinearFn.apply(ea, self.fc1_3.weight.t(), None, prec))], 1)
            ea = torch.relu(_LinearFn.apply(tmp, self.fc1_4.weight.t(), None, prec))
        w = (self.fc1_1.weight, self.fc1_2.weight, self.fc1_3.weight, self.fc1_4.weight) if fused_edge else (None,) * 4
        g = (self.fc11.weight, self.fc11.bias, self.fc12.weight, self.fc12.bias) if self.nout2 > 0 else (None,) * 4
        return _ML3LayerFn.apply(x, ea, *w, c.weight, c.bias, *g, plan, fused_edge, prec, _needs_save(x, ea, *w, c.weight, c.bias, *g))


# paths taken by ML1Layer since import (tests and benchmarks read it): "fused" = one library call per direction, "composed" =
# the layer composed from the aggregation kernel and the tensor-core GEMMs (shapes outside gnnml3_ml1layer_supported)
ML1_PATH_COUNTS = {"fused": 0, "composed": 0}


class _ML1LayerFn(torch.autograd.Function):
    """Whole GNNML1 layer as one autograd node (gnnml3_ml1layer_forward / _backward):

        p0 = x WA^T + bA + (A x) Wc + bc,   p1 = x WB^T + bB,   p2 = x WC^T + bC
        y  = relu(p0 + p1 * p2)   or, concatenated,   [relu(x WA^T + bA) | relu((A x) Wc + bc) | relu(p1 * p2)]

    Backward: G = [gA | gP p2 | gP p1] from the masks of y; dx = (A^T gc) Wc^T + G [WA ; WB ; WC] (one fused kernel over the
    transposed CSR); [dWA^T | dWB^T | dWC^T | dWc] = x^T [G | A^T gc] (one contraction); biases = column sums of G and gc.

    ``save`` False (a forward nobody differentiates): the kernel stores y alone, without [p1 | p2], and nothing is saved.
    ``precision`` (PREC_*) is the arithmetic of the layer's projections in both directions."""

    @staticmethod
    def forward(ctx, x, wconv, bconv, wA, bA, wB, bB, wC, bC, plan, concat, precision=_lib.PREC_3XTF32, save=True):
        xa = ops.aligned_rows(x)
        ws = [w.contiguous() for w in (wconv, wA, wB, wC)]
        bs = [b.contiguous() if b is not None else None for b in (bconv, bA, bB, bC)]
        if save:
            y, aux, _ = ops.ml1layer_forward(plan, xa, ws[0], bs[0], ws[1], bs[1], ws[2], bs[2], ws[3], bs[3], concat=concat,
                                             precision=precision)
        else:
            y, aux, _ = ops.ml1layer_forward(plan, xa, ws[0], bs[0], ws[1], bs[1], ws[2], bs[2], ws[3], bs[3], concat=concat, aux=False,
                                             precision=precision)
        ctx.plan, ctx.concat, ctx.precision = plan, concat, precision
        ctx.has_bias = tuple(b is not None for b in (bconv, bA, bB, bC))
        if save:
            ctx.save_for_backward(xa, *ws, y, aux)
        return y

    @staticmethod
    def backward(ctx, gy):
        xa, wconv, wA, wB, wC, y, aux = ctx.saved_tensors
        need = ctx.needs_input_grad
        N, Fi = xa.shape
        if N == 0:
            z = torch.zeros_like
            bz = [torch.zeros(wconv.size(2), device=xa.device) if h else None for h in ctx.has_bias]
            return z(xa), z(wconv), bz[0], z(wA), bz[1], z(wB), bz[2], z(wC), bz[3], None, None, None, None
        gy = gy if gy.stride(1) == 1 else gy.contiguous()
        dx, dwc, dbc, dwA, dbA, dwB, dbB, dwC, dbC = ops.ml1layer_backward(ctx.plan, xa, wconv, wA, wB, wC, y, aux, gy, need[0],
                                                                          concat=ctx.concat, precision=ctx.precision)
        hb = ctx.has_bias
        return (dx, dwc, dbc if hb[0] else None, dwA, dbA if hb[1] else None, dwB, dbB if hb[2] else None, dwC,
                dbC if hb[3] else None, None, None, None, None)


class ML1Layer(torch.nn.Module):
    """GNNML1 layer, the paper's 1-WL model (the GNNML1 classes of the reference's experiment scripts):
    ``relu(fc11(x) + conv1(x, edge_index, ones) + fc12(x) * fc13(x))`` or, with ``concat=True``,
    ``[relu(fc11(x)) | relu(conv1(x, edge_index, ones)) | relu(fc12(x) * fc13(x))]``.

    ``conv1`` is a ``SpectConv(ninp, nout, K=1, selfconn=False)`` on the graph's plain ``edge_index`` with every edge weight
    one; ``fc11``, ``fc12``, ``fc13`` are ``nn.Linear(ninp, nout)``.  ``forward(x, edge_index)`` -> [N, nout] (or [N, 3 nout]).
    Shapes with ninp, nout <= 64 run as one fused library call per direction; larger ones are composed from the aggregation
    kernel and the tensor-core GEMMs of this library, with the same result.  ``precision`` ("fp32" = 3xTF32, "tf32", "bf16"):
    the arithmetic of the projections, as for ML3Layer; aggregation, epilogues and outputs stay float32."""

    def __init__(self, ninp, nout, concat=False, precision="fp32"):
        super(ML1Layer, self).__init__()
        _precision_code(precision)
        self.concat = bool(concat)
        self.precision = precision
        self.conv1 = SpectConv(ninp, nout, 1, selfconn=False)
        self.fc11 = torch.nn.Linear(ninp, nout)
        self.fc12 = torch.nn.Linear(ninp, nout)
        self.fc13 = torch.nn.Linear(ninp, nout)

    @property
    def out_features(self):
        return self.conv1.out_channels * (3 if self.concat else 1)

    def forward(self, x, edge_index):
        return ml1_layer(x, edge_index, self.conv1, self.fc11, self.fc12, self.fc13, self.concat, self.precision)


def ml1_layer(x, edge_index, conv, fcA, fcB, fcC, concat=False, precision="fp32"):
    """The GNNML1 layer on given modules (``conv`` a SpectConv(K=1, selfconn=False), ``fcA``/``fcB``/``fcC`` nn.Linear):
    what ``ML1Layer.forward`` and ``models.GNNML1`` run, in ``precision`` ("fp32", "tf32" or "bf16")."""
    prec = _precision_code(precision)
    if not (x.is_cuda and edge_index.is_cuda):
        raise RuntimeError("gnn_matlang_b200: x and edge_index must be CUDA tensors (the B200 hot path has no CPU fallback)")
    if x.dim() != 2 or x.dtype != torch.float32:
        raise RuntimeError("gnn_matlang_b200: x [N, F] must be float32")
    plan = get_plan(edge_index, x.size(0))
    Fi, Fo = conv.in_channels, conv.out_channels
    if ops.ml1layer_supported(Fi, Fo, concat):
        ML1_PATH_COUNTS["fused"] += 1
        ps = (conv.weight, conv.bias, fcA.weight, fcA.bias, fcB.weight, fcB.bias, fcC.weight, fcC.bias)
        return _ML1LayerFn.apply(x, *ps, plan, bool(concat), prec, _needs_save(x, *ps))
    ML1_PATH_COUNTS["composed"] += 1
    ones = torch.ones(plan.E, 1, dtype=torch.float32, device=x.device)
    ax = _AggregateFn.apply(x, ones, plan)
    pa = _LinearFn.apply(x, fcA.weight.t(), fcA.bias, prec)
    pc = _LinearFn.apply(ax, conv.weight[0], conv.bias, prec)
    pp = _LinearFn.apply(x, fcB.weight.t(), fcB.bias, prec) * _LinearFn.apply(x, fcC.weight.t(), fcC.bias, prec)
    if concat:
        return torch.cat([torch.relu(pa), torch.relu(pc), torch.relu(pp)], 1)
    return torch.relu(pa + pc + pp)
