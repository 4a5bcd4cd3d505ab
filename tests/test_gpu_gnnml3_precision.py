"""GNNML3 in its reduced-precision modes on the B200, against float64: ``precision="tf32"`` (one tensor-core product per k-step on
TF32 operands) and ``precision="bf16"`` (RN-BF16 operands and weights, FP32 accumulation) of the tensor-memory fused kernel
(fused_layer_ts.cu) in both of its forms, the composed routes (gemm_nn / gemm_tn single-pass, where BF16 runs as TF32), the
modules (ML3Layer, SpectConv, SpectConCatConv), the whole models, the captured training step and evaluation pass, and the C
ABI's precision argument.

Bars, relative to the result's scale (test_gpu_kernels.assert_close), as in test_gpu_gnnml1_precision: kernel level 2e-3 (TF32)
and 2e-2 (BF16), module and model level 5e-3 and 5e-2.  Gradients are held to the module bar in the Frobenius norm and
entry-wise for at least 99 % of the entries of large tensors; the layer tests zero gy where the conv pre-activation lies within
twice the kernel bar of the ReLU kink, so that no mask flip can happen there.  Every flagged result must also be measurably
reduced (a silent fall-through to 3xTF32 sits at ~1e-7 of the scale).

The tensor-memory kernel takes K <= 18 (K <= 8 when Nc > 32): its weight planes and two staging buffers must fit in 227 KB of
shared memory, so K = 18 is the largest K of the forward grid below."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import gnnml3_oracle as O  # noqa: E402
from test_gpu_fused import _graph, _ref_main  # noqa: E402
from test_gpu_gnnml1_precision import FLAGGED, KERNEL_BAR, MODULE_BAR, _close_in_norm, _rel_err  # noqa: E402
from test_gpu_kernels import assert_close, dev  # noqa: E402
from test_gpu_model import _random_graphs  # noqa: E402


def _prec(name):
    from gnn_matlang_b200.libs.spect_conv import _PRECISIONS
    return _PRECISIONS[name]


def _aggregates(x, ei, ea):
    """[N, K, F] float64: the K-channel aggregates sum_{e: dst_e = t} ea[e, k] x[src_e] (the side output hout holds them)."""
    N, K = x.size(0), ea.size(1)
    H = torch.zeros(N, K, x.size(1), dtype=torch.float64)
    for k in range(K):
        H[:, k] = torch.zeros(N, x.size(1), dtype=torch.float64).index_add_(0, ei[1], ea[:, k:k + 1].double() * x.double()[ei[0]])
    return H


def _check_hout(hout, H, S, name):
    """hout [N, (K [+1]) * 32]: block k holds the aggregate H[:, k] at the FP32 bar (the aggregate is FP32 in every mode); the
    self block (S given) a copy of S."""
    K, F = H.size(1), H.size(2)
    h = hout.detach().cpu().view(hout.size(0), -1, 32)
    assert_close(h[:, :K, :F], H, rtol=1e-5, name=name + " aggregate side output")
    if S is not None:
        assert torch.equal(h[:, K, :S.size(1)], S.cpu()), name + ": self block of the side output is not a copy of S"


# ----------------------------------------------------------------------------------------------------------------------------
# A. ops.fused_agg_proj in TF32 and BF16
# ----------------------------------------------------------------------------------------------------------------------------

FWD_CASES = [  # N, K, F, Nc, G
    (2000, 2, 1, 1, 0),
    (1800, 2, 17, 64, 0),
    (1700, 2, 31, 30, 1),
    (1000, 6, 2, 32, 16),        # graph8c / EXP layer 1
    (1600, 6, 31, 9, 1),
    (1500, 6, 25, 64, 0),        # the 64-wide half
    (3001, 8, 25, 30, 2),        # ZINC layer 1
    (2000, 8, 32, 33, 0),
    (1900, 8, 17, 48, 0),
    (95, 8, 32, 30, 2),          # less than one tile
    (1300, 12, 31, 30, 4),
    (1200, 12, 17, 1, 4),
    (2000, 12, 32, 16, 16),      # counting layers 2-5
    (1100, 16, 2, 30, 2),
    (1400, 18, 25, 32, 16),      # largest K of the kernel, with the gate block
    (1000, 18, 1, 9, 2),
    (900, 18, 32, 32, 0),
]


@pytest.mark.parametrize("N,K,F,Nc,G", FWD_CASES)
def test_fused_forward_form(N, K, F, Nc, G):
    """Forward form (self_mode 0, or 1 with the gate block and the ML3 epilogue) in both flagged modes: y / aux against float64
    at the kernel bar, the side output at the FP32 bar, the tensor-memory kernel ran once per launch, staged (tile windows) and
    unstaged (global gathers) results bit-identical, repeated launches bit-identical, the error above 1e-5 of the scale, and TF32
    and BF16 different."""
    from gnn_matlang_b200 import ops
    Fs, mode, Ns = (F, 1, 2 * G) if G else (0, 0, 0)
    assert ops.fused_ts_supported(K, K, F, Nc, Fs, mode, Ns), "case outside the tensor-memory kernel"
    ei, g = _graph(N, 5, 31 * N + K)
    E = ei.size(1)
    x = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    bias = torch.randn(Nc, generator=g) * 0.3
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    ea_s = ea.to(d)[plan["perm"].long()].contiguous()
    xa = ops.aligned_rows(x.to(d))
    conv = _ref_main(x, ei, ea, W, bias)
    kw = dict(bias=bias.to(d), epilogue=0)
    refs = [("conv", lambda y, aux: y, conv)]
    if G:
        w11 = torch.randn(G, F, generator=g) / np.sqrt(F)
        w12 = torch.randn(G, F, generator=g) / np.sqrt(F)
        b11, b12 = torch.randn(G, generator=g) * 0.2, torch.randn(G, generator=g) * 0.2
        kw.update(S=xa, self_mode=1, Bself=torch.cat([w11.t(), w12.t()], 1).contiguous().to(d), bias_s=torch.cat([b11, b12]).to(d),
                  G=G, epilogue=1)
        t1 = torch.tanh(x.double() @ w11.double().t() + b11.double())
        t2 = torch.tanh(x.double() @ w12.double().t() + b12.double())
        refs = [("relu(conv)", lambda y, aux: y[:, :Nc], torch.relu(conv)), ("gate", lambda y, aux: y[:, Nc:], t1 * t2),
                ("aux", lambda y, aux: aux, torch.cat([t1, t2], 1))]
    H = _aggregates(x, ei, ea)
    Wm = W.view(K * F, Nc).to(d)
    outs = {}
    for name in FLAGGED:
        def launch(win, hout=None):
            return ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, Wm, win=win, hout=hout, precision=_prec(name), **kw)
        hout = torch.full((N, (K + (1 if G else 0)) * 32), float("nan"), device=d)
        before = ops.fused_path_counts()
        y, aux = launch(plan["win"], hout)
        assert ops.fused_path_counts() == (before[0] + 1, before[1]), "the tensor-memory kernel did not run"
        for other in (launch(None), launch(plan["win"])):
            assert torch.equal(other[0], y) and (aux is None or torch.equal(other[1], aux)), \
                "%s: staged / unstaged / repeated launches differ" % name
        errs = []
        for what, get, ref in refs:
            assert_close(get(y, aux), ref, rtol=KERNEL_BAR[name], name="%s %s" % (name, what))
            errs.append(_rel_err(get(y, aux), ref))
        _check_hout(hout, H, x if G else None, name)
        print("forward K=%d F=%d Nc=%d G=%d %s: error %s of the scale (tensor-memory kernel)"
              % (K, F, Nc, G, name, " / ".join("%.2e" % e for e in errs)))
        assert errs[0] > 1e-5, "suspiciously exact for %s: %.2e" % (name, errs[0])
        outs[name] = y
    assert not torch.equal(outs["tf32"], outs["bf16"]), "TF32 and BF16 give the same bits"


DX_CASES = [  # N, K, F (width of the transposed operand), Nc, Fs
    (3000, 8, 30, 32, 4),        # ZINC dx: gate gradients as the self block
    (2000, 6, 32, 2, 32),        # graph8c / EXP layer 1 dx
    (1000, 12, 16, 32, 32),      # counting dx
    (1500, 8, 25, 48, 2),
    (1200, 18, 17, 9, 16),
    (900, 6, 1, 64, 0),
    (800, 2, 31, 30, 0),
]


@pytest.mark.parametrize("N,K,F,Nc,Fs", DX_CASES)
def test_fused_dx_form(N, K, F, Nc, Fs):
    """The dx form every flagged backward runs: transposed CSR, edge weights read through permT, a self block accumulating
    into the main columns (self_mode 2, packed by its own BF16 path); same checks as the forward form."""
    from gnn_matlang_b200 import ops
    assert ops.fused_ts_supported(K, K, F, Nc, Fs, 2 if Fs else 0, 0), "case outside the tensor-memory kernel"
    ei, g = _graph(N, 5, 7 * N + K)
    E = ei.size(1)
    gout = torch.randn(N, F, generator=g)
    ea = torch.randn(E, K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    ea_s = ea.to(d)[plan["perm"].long()].contiguous()
    eiT = torch.stack([ei[1], ei[0]])
    ref = _ref_main(gout, eiT, ea, W, None)
    F4 = (F + 3) // 4 * 4
    buf = torch.zeros(N, F4 + (Fs + 3) // 4 * 4)
    buf[:, :F] = gout
    sv = Bs = None
    if Fs:
        sv = torch.randn(N, Fs, generator=g)
        Bs = torch.randn(Fs, Nc, generator=g) / np.sqrt(Fs)
        buf[:, F4:F4 + Fs] = sv
        ref = ref + sv.double() @ Bs.double()
    bufd = buf.to(d)
    H = _aggregates(gout, eiT, ea)
    Wm = W.view(K * F, Nc).to(d)
    outs = {}
    for name in FLAGGED:
        def launch(win, hout=None):
            return ops.fused_agg_proj(plan["rowptrT"], plan["colT"], plan["permT"], ea_s, bufd[:, :F], Wm,
                                      S=bufd[:, F4:F4 + Fs] if Fs else None, self_mode=2 if Fs else 0,
                                      Bself=Bs.to(d) if Fs else None, epilogue=0, hout=hout, win=win, precision=_prec(name))[0]
        hout = torch.full((N, (K + (1 if Fs else 0)) * 32), float("nan"), device=d)
        before = ops.fused_path_counts()
        out = launch(plan["winT"], hout)
        assert ops.fused_path_counts() == (before[0] + 1, before[1]), "the tensor-memory kernel did not run"
        assert torch.equal(launch(None), out) and torch.equal(launch(plan["winT"]), out), \
            "%s: staged / unstaged / repeated launches differ" % name
        assert_close(out, ref, rtol=KERNEL_BAR[name], name=name + " dx form")
        _check_hout(hout, H, sv, name + " dx form")
        err = _rel_err(out, ref)
        print("dx form K=%d F=%d Nc=%d Fs=%d %s: error %.2e of the scale (tensor-memory kernel)" % (K, F, Nc, Fs, name, err))
        assert err > 1e-5, "suspiciously exact for %s: %.2e" % (name, err)
        outs[name] = out
    assert not torch.equal(outs["tf32"], outs["bf16"]), "TF32 and BF16 give the same bits"


def test_fused_mixed_and_crowded_tiles():
    """One launch per form with all three kinds of tiles: local edges (staged), long-range edges (window wider than the TMA
    box) and a tile with more CSR slots than any staging buffer holds (both gather from global memory); staged and unstaged
    results bit-identical, and against float64 at the kernel bar."""
    from gnn_matlang_b200 import _lib, ops
    N, deg, K, F, Nc, G = 6000, 5, 8, 25, 30, 2
    rows = _lib.load().gnnml3_tile_rows()
    g = torch.Generator().manual_seed(23)
    E = N * deg
    src = torch.randint(0, N, (E,), generator=g)
    near = ((src // 40) * 40 + torch.randint(0, 40, (E,), generator=g)).clamp(max=N - 1)
    far = torch.randint(N // 2, N, (E,), generator=g)
    dst = torch.where(src < N // 2, near, far)
    xs = torch.randint(0, rows, (rows * 40,), generator=g)          # the first tile: 40 extra local slots per row
    xd = torch.arange(rows).repeat_interleave(40)
    ei = torch.stack([torch.cat([src, xs]), torch.cat([dst, xd])])
    d = dev()
    plan = ops.csr_build(ei.to(d), N)
    for w, rp in ((plan["win"], plan["rowptr"]), (plan["winT"], plan["rowptrT"])):
        width = (w[:, 1] - w[:, 0]).cpu()
        assert (width <= 256).any() and (width > 256).any(), "the case must contain staged and unstaged tiles"
        assert int(rp[rows] - rp[0]) > 2048, "the first tile must hold more slots than a staging buffer"
    x = torch.randn(N, F, generator=g)
    ea = torch.randn(ei.size(1), K, generator=g)
    W = torch.randn(K, F, Nc, generator=g) / np.sqrt(K * F)
    w11 = torch.randn(G, F, generator=g) / np.sqrt(F)
    w12 = torch.randn(G, F, generator=g) / np.sqrt(F)
    Wt = torch.randn(K, Nc, F, generator=g) / np.sqrt(K * Nc)        # dx form: gout [N, Nc] -> [N, F]
    gg = torch.randn(N, 2 * G, generator=g)
    ea_s = ea.to(d)[plan["perm"].long()].contiguous()
    xa = ops.aligned_rows(x.to(d))
    gc = ops.aligned_rows(torch.randn(N, Nc, generator=g).to(d))
    gga = ops.aligned_rows(gg.to(d))
    wg = torch.cat([w11.t(), w12.t()], 1).contiguous().to(d)
    conv = torch.relu(_ref_main(x, ei, ea, W, None))
    dx_ref = _ref_main(gc.cpu(), torch.stack([ei[1], ei[0]]), ea, Wt, None) + gg.double() @ torch.cat([w11, w12], 0).double()
    for name in FLAGGED:
        p = _prec(name)
        fwd = [ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, xa, W.view(K * F, Nc).to(d), S=xa, self_mode=1, Bself=wg,
                                  bias_s=torch.zeros(2 * G, device=d), G=G, epilogue=1, win=win, precision=p)[0] for win in (plan["win"], None)]
        dx = [ops.fused_agg_proj(plan["rowptrT"], plan["colT"], plan["permT"], ea_s, gc, Wt.reshape(K * Nc, F).to(d), S=gga, self_mode=2,
                                 Bself=torch.cat([w11, w12], 0).contiguous().to(d), epilogue=0, win=win, precision=p)[0]
              for win in (plan["winT"], None)]
        assert torch.equal(fwd[0], fwd[1]) and torch.equal(dx[0], dx[1]), name + ": staged and unstaged results differ"
        assert_close(fwd[0][:, :Nc], conv, rtol=KERNEL_BAR[name], name=name + " relu(conv) (mixed tiles)")
        assert_close(dx[0], dx_ref, rtol=KERNEL_BAR[name], name=name + " dx form (mixed tiles)")
        print("mixed and crowded tiles %s: forward error %.2e, dx error %.2e of the scale"
              % (name, _rel_err(fwd[0][:, :Nc], conv), _rel_err(dx[0], dx_ref)))


def test_flagged_precision_is_rejected_outside_the_tensor_memory_kernel():
    """A flagged precision on a shape only the shared-memory-plane kernel serves (F = 40, odd K), or with that kernel forced
    (slot aggregator mode, tensor-memory kernel off), is GNNML3_ERR_INVALID; the same shapes run in 3xTF32."""
    from gnn_matlang_b200 import _lib, ops
    lib = _lib.load()
    N, Nc = 700, 30
    ei, g = _graph(N, 4, 5)
    d = dev()
    plan = ops.csr_build(ei.to(d), N)

    def call(K, F, prec):
        ea_s = torch.randn(ei.size(1), K, generator=g).to(d)
        x = ops.aligned_rows(torch.randn(N, F, generator=g).to(d))
        return ops.fused_agg_proj(plan["rowptr"], plan["col"], None, ea_s, x, torch.randn(K * F, Nc, generator=g).to(d), epilogue=0,
                                  win=plan["win"], precision=prec)

    msg = r"code 1\).*tensor-memory kernel only"
    for name in FLAGGED:
        for K, F in ((8, 40), (5, 16)):
            assert ops.fused_supported(K, K, F, Nc) and not ops.fused_ts_supported(K, K, F, Nc)
            with pytest.raises(RuntimeError, match=msg):
                call(K, F, _prec(name))
            call(K, F, _lib.PREC_3XTF32)
        for setter in (lambda: lib.gnnml3_fused_set_mode(1), lambda: lib.gnnml3_fused_set_ts(0)):
            old_mode, old_ts = lib.gnnml3_fused_set_mode(-1), lib.gnnml3_fused_set_ts(-1)
            try:
                setter()
                assert not ops.fused_ts_supported(8, 8, 32, Nc)
                with pytest.raises(RuntimeError, match=msg):
                    call(8, 32, _prec(name))
                call(8, 32, _lib.PREC_3XTF32)
            finally:
                lib.gnnml3_fused_set_mode(old_mode)
                lib.gnnml3_fused_set_ts(old_ts)
        call(8, 32, _prec(name))


# ----------------------------------------------------------------------------------------------------------------------------
# B. ML3Layer(precision=...) on both routes
# ----------------------------------------------------------------------------------------------------------------------------

@pytest.fixture
def precision_log(monkeypatch):
    """Records (entry point, precision) of every fused_agg_proj / gemm_nn / gemm_tn call the modules make (no precision given =
    the wrappers' default, 3xTF32)."""
    from gnn_matlang_b200 import _lib, ops
    log = []
    for fn in ("fused_agg_proj", "gemm_nn", "gemm_tn"):
        def spy(*a, _real=getattr(ops, fn), _fn=fn, **k):
            log.append((_fn, k.get("precision", _lib.PREC_3XTF32), k.get("hout") is not None, len(a) > 2 and a[2] is not None))
            return _real(*a, **k)
        monkeypatch.setattr(ops, fn, spy)
    return log


def _expected_route(precision, K, Fi, Fo, G):
    """The route _ML3LayerFn takes in ``precision``: fused when both directions fit the fused kernels."""
    from gnn_matlang_b200.libs.spect_conv import _fused_ok
    p = _prec(precision)
    fused = ((G == 0 or Fi <= 32) and _fused_ok(p, K, K, Fi, Fo, Fi if G else 0, 1 if G else 0, 2 * G)
             and _fused_ok(p, K, K, Fo, Fi, 2 * G, 2 if G else 0, 0))
    return "fused" if fused else "composed"


def _layer_setup(learnedge, K, Fi, Fo, G, N, seed):
    """Graph, inputs and a float32 oracle layer with non-zero conv bias (the reference initialises it to zero).  Where the edge
    MLP is composed from the single-pass GEMMs (TF32 in both flagged modes), edges with a ReLU input of the MLP within twice
    the TF32 kernel bar of 0 are dropped: a mask flipped there moves d edge_attr and the MLP's weight gradients by O(1) per
    edge -- the discontinuity of the function, not an error of the arithmetic."""
    from gnn_matlang_b200 import ops
    ei, g = _graph(N, 5, seed)
    x = torch.randn(N, Fi, generator=g)
    ea = torch.randn(ei.size(1), K, generator=g)
    torch.manual_seed(seed)
    ref = O.OracleML3Layer(learnedge, K, K, Fi, Fo, G)
    with torch.no_grad():
        ref.conv1.bias.normal_(0, 0.3)
        if learnedge and not ops.edge_mlp_supported(K, K):
            w = [getattr(ref, "fc1_%d" % i).weight.double() for i in range(1, 5)]
            e = ea.double()
            pre1 = e @ w[0].t()
            pre4 = torch.cat([torch.relu(pre1), torch.tanh(e @ w[1].t()) * torch.tanh(e @ w[2].t())], 1) @ w[3].t()
            margin = 2 * KERNEL_BAR["tf32"]
            keep = ((pre1.abs() > margin * pre1.abs().max()).all(1) & (pre4.abs() > margin * pre4.abs().max()).all(1))
            ei, ea = ei[:, keep], ea[keep]
    return ei, x, ea, ref


def _layer_ref(ref, x, ei, ea, margin, seed):
    """float64 oracle forward + backward with gy zeroed on the conv block where |pre-activation| <= margin * max|pre-activation|.
    -> (y, gy used, dx, d edge_attr, {parameter: gradient})"""
    ref = ref.double()
    p = dict(ref.named_parameters())
    xd = x.double().requires_grad_(True)
    ead = ea.double().requires_grad_(True)
    y = ref(xd, ei, ead)
    with torch.no_grad():
        e2 = O.edge_mlp_forward(ead, p["fc1_1.weight"], p["fc1_2.weight"], p["fc1_3.weight"], p["fc1_4.weight"]) if ref.learnedge else ead
        pre = O.spectconv_forward(xd, ei, e2, p["conv1.weight"], p["conv1.bias"])
    gy = torch.randn(*y.shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    gy[:, :pre.size(1)] *= (pre.abs() > margin * pre.abs().max()).double()
    y.backward(gy)
    return y.detach(), gy.float(), xd.grad, ead.grad, {k: v.grad for k, v in p.items()}


def _run_layer(learnedge, K, Fi, Fo, G, precision, N=2000, seed=0, strided=False, log=None, margin=None):
    """ML3Layer(precision=...) forward + backward against the float64 oracle: y at the kernel bar, dx, d edge_attr and every
    parameter gradient at the module bar in norm (gy zeroed where the conv pre-activation lies within ``margin`` -- default twice
    the kernel bar -- of the kink).  Returns (route taken, {result: tensor})."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.libs.spect_conv import ML3Layer
    kb, mb = KERNEL_BAR[precision], MODULE_BAR[precision]
    ei, x, ea, ref = _layer_setup(learnedge, K, Fi, Fo, G, N, seed)
    lay = ML3Layer(learnedge, K, K, Fi, Fo, G, precision=precision)
    lay.load_state_dict(ref.state_dict())
    yr, gy, dxr, dear, gr = _layer_ref(ref, x, ei, ea, 2 * kb if margin is None else margin, seed + 1)
    d = dev()
    lay = lay.to(d)
    if strided:      # x = a column block of a wider activation (row stride Fi + 12, offset 8 floats)
        leaf = torch.zeros(N, Fi + 12)
        leaf[:, 8:8 + Fi] = x
        leaf = leaf.to(d).requires_grad_(True)
        xin = leaf[:, 8:8 + Fi]
    else:
        leaf = x.to(d).requires_grad_(True)
        xin = leaf
    eag = ea.to(d).requires_grad_(True)
    if log is not None:
        del log[:]
    before = ops.fused_path_counts()
    y = lay(xin, ei.to(d), eag)
    y.backward(gy.to(d))
    ts, planes = ops.fused_path_counts()
    route = "fused" if (ts, planes) == (before[0] + 2, before[1]) else "composed" if (ts, planes) == before else "mixed"
    name = "%s learnedge=%d K=%d Fi=%d Fo=%d G=%d" % (precision, learnedge, K, Fi, Fo, G)
    assert_close(y, yr, rtol=kb, name=name + " y")
    err = _rel_err(y, yr)
    print("ML3Layer %s: y error %.2e of the scale, %s route" % (name, err, route))
    assert err > 1e-5, "suspiciously exact: %.2e" % err
    dx = leaf.grad[:, 8:8 + Fi] if strided else leaf.grad
    if strided:
        assert float(leaf.grad[:, :8].abs().max()) == 0.0 and float(leaf.grad[:, 8 + Fi:].abs().max()) == 0.0
    _close_in_norm(dx, dxr, mb, name + " dx")
    _close_in_norm(eag.grad, dear, mb, name + " d edge_attr")
    res = {"y": y.detach(), "dx": dx, "dea": eag.grad}
    for k, v in lay.named_parameters():
        _close_in_norm(v.grad, gr[k], mb, name + " d" + k)
        res[k] = v.grad
    return route, res


def _reduced_backward_passes(learnedge, K, Fi, Fo, G, precision, route, N=2000, seed=0):
    """The backward's own arithmetic, isolated: the dx pass (fused dx form, or gemm_nn on the composed route) and the weight-
    gradient contraction gemm_tn(x, Gp) on identical gpre / Gp, flagged against 3xTF32.  Reduced, and within the kernel bar."""
    from gnn_matlang_b200 import _lib, ops
    from gnn_matlang_b200.graph import get_plan
    ei, x, ea, ref = _layer_setup(learnedge, K, Fi, Fo, G, N, seed)
    d = dev()
    g = torch.Generator().manual_seed(seed + 2)
    plan = get_plan(ei.to(d), N)
    ea_s = ea.to(d)[plan.perm.long()].contiguous()
    xa = ops.aligned_rows(x.to(d))
    wconv = ref.conv1.weight.detach().to(d)
    Fo4 = (Fo + 3) // 4 * 4
    gpre = torch.zeros(N, (Fo4 + 2 * G + 3) // 4 * 4, device=d)
    gpre[:, :Fo] = torch.randn(N, Fo, generator=g).to(d)
    gpre[:, Fo4:Fo4 + 2 * G] = torch.randn(N, 2 * G, generator=g).to(d)
    Gp = torch.empty(N, K * Fo + 2 * G, device=d)
    ops.spmm_k(plan.rowptrT, plan.colT, plan.permT, ea_s, gpre[:, :Fo], out=Gp)
    Gp[:, K * Fo:] = gpre[:, Fo4:Fo4 + 2 * G]
    wgate = torch.cat([ref.fc11.weight, ref.fc12.weight], 0).detach().contiguous().to(d) if G else None

    def passes(p):
        if route == "fused":
            dx, _ = ops.fused_agg_proj(plan.rowptrT, plan.colT, plan.permT, ea_s, gpre[:, :Fo],
                                       wconv.transpose(1, 2).reshape(K * Fo, Fi).contiguous(), S=gpre[:, Fo4:Fo4 + 2 * G] if G else None,
                                       self_mode=2 if G else 0, Bself=wgate, epilogue=0, win=plan.winT, precision=p)
        else:
            blocks = [wconv.transpose(1, 2).reshape(K * Fo, Fi)] + ([wgate] if G else [])
            dx = ops.gemm_nn(Gp, torch.cat(blocks, 0).contiguous(), precision=p)
        return dx[:, :Fi], ops.gemm_tn(xa, Gp, precision=p)

    got, full = passes(_prec(precision)), passes(_lib.PREC_3XTF32)
    for what, a, r in zip(("dx pass", "weight-gradient contraction"), got, full):
        rel = float((a.double() - r.double()).norm() / r.double().norm())
        print("ML3Layer %s K=%d Fi=%d Fo=%d G=%d %s: %s differs from 3xTF32 by %.2e (Frobenius, relative)"
              % (precision, K, Fi, Fo, G, route, what, rel))
        assert rel > 1e-6, "%s suspiciously exact for %s: %.2e" % (what, precision, rel)
        assert rel <= KERNEL_BAR[precision], "%s off by %.2e" % (what, rel)


LAYER_CASES = [  # learnedge, K, Fi, Fo, G, route, strided x
    (True, 8, 25, 30, 2, "fused", False),        # ZINC layer 1
    (True, 8, 32, 30, 2, "fused", True),         # ZINC layers 2-4
    (True, 6, 2, 32, 16, "fused", False),        # graph8c / EXP layer 1
    (True, 12, 32, 16, 16, "fused", False),      # counting layers 2-5
    (True, 8, 32, 30, 0, "fused", False),        # nout2 = 0
    (True, 18, 16, 16, 4, "fused", False),       # K > 16: the composed edge MLP in front of the fused layer
    (True, 6, 48, 32, 16, "composed", True),     # graph8c / EXP layers 2-3
    (False, 8, 64, 64, 0, "composed", False),    # enzymes layers 2-4
    (False, 5, 16, 32, 16, "composed", False),   # odd K
    (True, 5, 16, 16, 8, "composed", False),     # odd K: composed edge MLP and layer
]


@pytest.mark.parametrize("learnedge,K,Fi,Fo,G,route,strided", LAYER_CASES)
def test_ml3layer_matches_oracle_on_its_route(learnedge, K, Fi, Fo, G, route, strided, precision_log):
    """Both flagged modes: the route _fused_ok predicts is the one that ran; output and gradients against float64; every
    library call of the forward and backward carries the layer's precision and the isolated backward passes are reduced;
    BF16 is bit-equal to TF32 on the composed route (BF16 runs as TF32 in gemm_nn / gemm_tn) and differs on the fused one."""
    res = {}
    for name in FLAGGED:
        assert _expected_route(name, K, Fi, Fo, G) == route
        # one gy for both modes (BF16's margin), so that the composed route's results can be compared bit for bit
        taken, res[name] = _run_layer(learnedge, K, Fi, Fo, G, name, seed=K + Fi, strided=strided, log=precision_log,
                                      margin=2 * KERNEL_BAR["bf16"])
        assert taken == route, "%s: %s route expected, %s taken" % (name, route, taken)
        assert precision_log and all(e[1] == _prec(name) for e in precision_log), \
            "%s: library calls in another precision: %s" % (name, sorted(set(precision_log)))
        if route == "fused":
            assert any(e[0] == "fused_agg_proj" and e[3] for e in precision_log), "no fused dx pass"
        _reduced_backward_passes(learnedge, K, Fi, Fo, G, name, route, seed=K + Fi)
    if route == "composed":
        for k in res["tf32"]:
            assert torch.equal(res["tf32"][k], res["bf16"][k]), "composed route: BF16 and TF32 differ in " + k
    else:
        assert not torch.equal(res["tf32"]["y"], res["bf16"]["y"]) and not torch.equal(res["tf32"]["dx"], res["bf16"]["dx"])


@pytest.mark.parametrize("switch", ["slot_mode", "tensor_memory_off"])
def test_flagged_layer_takes_the_composed_route_when_the_tensor_memory_kernel_cannot_run(switch):
    """With the slot aggregator mode on, or the tensor-memory kernel switched off, a TF32 layer of a fused shape routes to the
    composed path (which has the single-pass modes) instead of calling the fused kernel, which would refuse the precision."""
    from gnn_matlang_b200 import _lib
    lib = _lib.load()
    old_mode, old_ts = lib.gnnml3_fused_set_mode(-1), lib.gnnml3_fused_set_ts(-1)
    try:
        if switch == "slot_mode":
            lib.gnnml3_fused_set_mode(1)
        else:
            lib.gnnml3_fused_set_ts(0)
        assert _expected_route("tf32", 8, 32, 30, 2) == "composed"
        route, _ = _run_layer(True, 8, 32, 30, 2, "tf32", seed=3)
        assert route == "composed"
    finally:
        lib.gnnml3_fused_set_mode(old_mode)
        lib.gnnml3_fused_set_ts(old_ts)


@pytest.mark.parametrize("precision,K", [("tf32", 8), ("bf16", 8), ("tf32", 18), ("bf16", 18)])
def test_edge_mlp_precision(precision, K, monkeypatch):
    """The fused edge MLP (K <= 16, even) is FP32 in every mode: its output equals float64 at the FP32 bar.  The composed one
    (K = 18) runs its four linears in the layer's precision."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.libs import spect_conv
    from gnn_matlang_b200.libs.spect_conv import ML3Layer
    ei, x, ea, ref = _layer_setup(True, K, 16, 16, 4, 1500, K)
    lay = ML3Layer(True, K, K, 16, 16, 4, precision=precision)
    lay.load_state_dict(ref.state_dict())
    d = dev()
    lay = lay.to(d)
    outs, precs = [], []
    real_mlp, real_lin = ops.edge_mlp_fwd, spect_conv._LinearFn.apply

    def mlp_spy(ea_, *a, **k):
        outs.append((ea_, real_mlp(ea_, *a, **k)))
        return outs[-1][1]

    def lin_spy(*a):
        precs.append(a[3])
        return real_lin(*a)

    monkeypatch.setattr(ops, "edge_mlp_fwd", mlp_spy)
    monkeypatch.setattr(spect_conv._LinearFn, "apply", lin_spy)
    with torch.no_grad():
        lay(x.to(d), ei.to(d), ea.to(d))
    if ops.edge_mlp_supported(K, K):
        assert len(outs) == 1 and precs == []
        w = [getattr(ref, "fc1_%d" % i).weight.detach().double() for i in range(1, 5)]
        assert_close(outs[0][1], O.edge_mlp_forward(outs[0][0].cpu().double(), *w), rtol=1e-5, name="fused edge MLP " + precision)
    else:
        assert outs == [] and precs == [_prec(precision)] * 4


@pytest.mark.parametrize("learnedge,K,Fi,Fo,G,precision", [(True, 8, 32, 30, 2, "bf16"), (True, 6, 48, 32, 16, "tf32")])
def test_ml3layer_is_deterministic(learnedge, K, Fi, Fo, G, precision):
    """Forward + backward twice at a ZINC-batch size give identical bits (one fused and one composed shape)."""
    from gnn_matlang_b200.libs.spect_conv import ML3Layer
    N = 30000
    ei, x, ea, ref = _layer_setup(learnedge, K, Fi, Fo, G, N, 9)
    d = dev()
    lay = ML3Layer(learnedge, K, K, Fi, Fo, G, precision=precision)
    lay.load_state_dict(ref.state_dict())
    lay = lay.to(d)
    eid, gy = ei.to(d), torch.randn(N, Fo + G, generator=torch.Generator().manual_seed(4)).to(d)
    runs = []
    for _ in range(2):
        xg, eag = x.to(d).requires_grad_(True), ea.to(d).requires_grad_(True)
        lay.zero_grad()
        y = lay(xg, eid, eag)
        y.backward(gy)
        runs.append([y.detach(), xg.grad, eag.grad] + [p.grad.clone() for p in lay.parameters()])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ----------------------------------------------------------------------------------------------------------------------------
# C. SpectConv and SpectConCatConv with precision=
# ----------------------------------------------------------------------------------------------------------------------------

SPECT_CASES = [  # Fi, Fo, K, selfconn, order, tensor-memory launches (forward + dx)
    (25, 30, 8, False, "auto", 2),
    (32, 32, 6, True, "auto", 2),
    (17, 9, 8, True, "aggregate_first", 2),
    (30, 64, 8, False, "aggregate_first", 1),     # dx (F = 64) outside the fused kernel: the two-kernel dx
    (48, 32, 6, True, "auto", 0),
    (48, 40, 6, False, "aggregate_first", 0),
    (16, 24, 4, True, "project_first", 0),
    (16, 24, 4, False, "project_first", 0),
]


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("Fi,Fo,K,selfconn,order,ts_launches", SPECT_CASES)
def test_spectconv_matches_oracle(Fi, Fo, K, selfconn, order, ts_launches, precision, precision_log):
    """SpectConv(precision=...) forward at the kernel bar, d x, d edge_attr, d weight and d bias at the module bar in norm,
    against float64; the fused backward leaves the aggregate side output behind for the weight gradient."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.libs.spect_conv import SpectConv
    N = 1800
    ei, g = _graph(N, 5, Fi * Fo + K)
    x = torch.randn(N, Fi, generator=g)
    ea = torch.randn(ei.size(1), K, generator=g)
    torch.manual_seed(Fi + Fo + K)
    conv = SpectConv(Fi, Fo, K, selfconn=selfconn, precision=precision, order=order)
    with torch.no_grad():
        conv.bias.normal_(0, 0.3, generator=g)
    W, b = conv.weight.detach().double(), conv.bias.detach().double()
    xr, ear = x.double().requires_grad_(True), ea.double().requires_grad_(True)
    Wr, br = W.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = O.spectconv_forward(xr, ei, ear, Wr, br, selfconn=selfconn)
    gout = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    ref.backward(gout)
    d = dev()
    conv = conv.to(d)
    xg, eag = x.to(d).requires_grad_(True), ea.to(d).requires_grad_(True)
    before = ops.fused_path_counts()
    out = conv(xg, ei.to(d), eag)
    out.backward(gout.float().to(d))
    assert ops.fused_path_counts() == (before[0] + ts_launches, before[1])
    assert all(e[1] == _prec(precision) for e in precision_log), sorted(set(precision_log))
    if ts_launches == 2:
        assert any(e[0] == "fused_agg_proj" and e[2] for e in precision_log), "the fused dx pass left no side output"
    name = "SpectConv %s Fi=%d Fo=%d K=%d selfconn=%d %s" % (precision, Fi, Fo, K, selfconn, order)
    assert_close(out, ref, rtol=KERNEL_BAR[precision], name=name)
    err = _rel_err(out, ref)
    print("%s: error %.2e of the scale, %d tensor-memory launches" % (name, err, ts_launches))
    assert err > 1e-6, "suspiciously exact: %.2e" % err
    mb = MODULE_BAR[precision]
    for what, a, r in (("dx", xg.grad, xr.grad), ("d edge_attr", eag.grad, ear.grad), ("d weight", conv.weight.grad, Wr.grad),
                       ("d bias", conv.bias.grad, br.grad)):
        _close_in_norm(a, r, mb, name + " " + what)


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("Fi,Fo,K,selfconn", [(16, 8, 4, True), (40, 16, 6, False)])
def test_spectconcatconv_matches_oracle(Fi, Fo, K, selfconn, precision, precision_log):
    from gnn_matlang_b200.libs.spect_conv import SpectConCatConv
    N = 1500
    ei, g = _graph(N, 5, Fi + K)
    x = torch.randn(N, Fi, generator=g)
    ea = torch.randn(ei.size(1), K, generator=g)
    torch.manual_seed(Fi + Fo + K)
    conv = SpectConCatConv(Fi, Fo, K, selfconn=selfconn, precision=precision)
    with torch.no_grad():
        conv.bias.normal_(0, 0.3, generator=g)
    xr, ear = x.double().requires_grad_(True), ea.double().requires_grad_(True)
    Wr, br = conv.weight.detach().double().requires_grad_(True), conv.bias.detach().double().requires_grad_(True)
    ref = O.spectconcatconv_forward(xr, ei, ear, Wr, br, selfconn=selfconn)
    gout = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    ref.backward(gout)
    d = dev()
    conv = conv.to(d)
    xg, eag = x.to(d).requires_grad_(True), ea.to(d).requires_grad_(True)
    out = conv(xg, ei.to(d), eag)
    out.backward(gout.float().to(d))
    assert all(e[1] == _prec(precision) for e in precision_log), sorted(set(precision_log))
    name = "SpectConCatConv %s Fi=%d Fo=%d K=%d selfconn=%d" % (precision, Fi, Fo, K, selfconn)
    assert_close(out, ref, rtol=KERNEL_BAR[precision], name=name)
    err = _rel_err(out, ref)
    print("%s: error %.2e of the scale" % (name, err))
    assert err > 1e-6, "suspiciously exact: %.2e" % err
    mb = MODULE_BAR[precision]
    for what, a, r in (("dx", xg.grad, xr.grad), ("d edge_attr", eag.grad, ear.grad), ("d weight", conv.weight.grad, Wr.grad),
                       ("d bias", conv.bias.grad, br.grad)):
        _close_in_norm(a, r, mb, name + " " + what)


# ----------------------------------------------------------------------------------------------------------------------------
# D. Whole models
# ----------------------------------------------------------------------------------------------------------------------------

class _ReplayedRelu(object):
    """Stands in for torch.nn.functional inside the oracle: ``relu`` of a tensor shaped like the next recorded mask applies that
    mask (the device's), every other call is torch's own."""

    def __init__(self, masks):
        self.masks = list(masks)

    def relu(self, v):
        if self.masks and self.masks[0].shape == v.shape:
            return v * self.masks.pop(0)
        return torch.relu(v)

    def __getattr__(self, name):
        return getattr(torch.nn.functional, name)


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("cfg", ["zinc", "graph8c", "exp", "counting", "mutag", "enzymes"])
def test_model_matches_oracle_model(cfg, precision, monkeypatch):
    """GNNML3(cfg, ne, ninp, precision=...) on records with real supports against the float64 oracle model with the same
    weights: output at the module bar, every gradient at the module bar in norm, the output measurably reduced.  mutag in
    training mode (BatchNorm batch statistics), enzymes in eval mode (add + max read-out, BatchNorm running statistics).

    Reduced precision moves some of the model's many ReLU inputs (every layer's conv block, the head) across the kink, and each
    flip moves whole-graph gradient contributions by O(1) (a relative error of about the square root of the flipped share,
    whatever the mantissa).  The oracle's backward therefore runs with the ReLU masks of the device's forward (taken from each
    layer's output and the head's first linear), so that the gradients measure the arithmetic; the output is held to the
    unmodified oracle as well."""
    from gnn_matlang_b200 import models
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.models import GNNML3
    g = torch.Generator().manual_seed(41)
    variant = cfg in ("mutag", "enzymes")
    graphs = _random_graphs("exp" if variant else cfg, 24, g)
    ne, ninp = graphs[0]["edge_attr2"].shape[1], graphs[0]["x"].shape[1]
    torch.manual_seed(5)
    ref = O.OracleGNNML3Variant(cfg, ne, ninp) if variant else O.OracleGNNML3(cfg, ne, ninp)
    if cfg == "enzymes":
        with torch.no_grad():
            ref.bn4.running_mean.normal_(0, 1.0)
            ref.bn4.running_var.uniform_(0.5, 2.0)
    model = GNNML3(cfg, ne, ninp, precision=precision)
    model.load_state_dict(ref.state_dict())
    train = cfg != "enzymes"
    ref = ref.double().train(train)
    model = model.to(dev()).train(train)
    c = model.cfg
    masks, lin_outs = [], []
    for l in range(c["nlayer"]):
        getattr(model, "conv%d" % (l + 1)).register_forward_hook(
            lambda mod, inp, y: masks.append((y[:, :c["nout1"]] > 0).detach().cpu().double()))
    real_lin = models._LinearFn

    class LinSpy(object):
        @staticmethod
        def apply(*a):
            out = real_lin.apply(*a)
            lin_outs.append(out.detach())
            return out

    monkeypatch.setattr(models, "_LinearFn", LinSpy)
    out = model(collate(graphs).to(dev()))
    if len(c["head"]) > 1:
        masks.append((lin_outs[0] > 0).cpu().double())
    ob = O.collate(graphs)
    ob["x"], ob["edge_attr2"] = ob["x"].double(), ob["edge_attr2"].double()
    mb = MODULE_BAR[precision]
    with torch.no_grad():
        plain = ref(ob)
    assert_close(out, plain, rtol=mb, name="%s %s out" % (cfg, precision))
    err = _rel_err(out, plain)
    replay = _ReplayedRelu(masks)
    monkeypatch.setattr(O, "F", replay)
    out_r = ref(ob)
    assert replay.masks == [], "not every recorded ReLU mask was used"
    print("GNNML3 %s %s: output error %.2e of the scale" % (cfg, precision, err))
    assert err > 1e-6, "suspiciously exact: %.2e" % err
    assert_close(out, out_r, rtol=mb, name="%s %s out (replayed masks)" % (cfg, precision))
    gout = torch.randn(out_r.shape, generator=g, dtype=torch.float64)
    out_r.backward(gout)
    out.backward(gout.float().to(dev()))
    refp = dict(ref.named_parameters())
    for k, v in model.named_parameters():
        _close_in_norm(v.grad, refp[k].grad, mb, "%s %s d%s" % (cfg, precision, k))


# ----------------------------------------------------------------------------------------------------------------------------
# E. Captured paths
# ----------------------------------------------------------------------------------------------------------------------------

def test_captured_bf16_step_equals_eager_step():
    """GraphedTrainer on a BF16 GNNML3 zinc model equals the eager Trainer step after step (loss 2e-5 relative, parameters 2e-6
    absolute after each Adam step), through both input routes: a padded device batch, and an unpadded batch written into the
    captured buffers on the device."""
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch
    pool = GraphPool("zinc", 64, seed=6)
    rng = np.random.default_rng(3)
    host = [pool.draw(rng, 48) for _ in range(4)]
    Np, Ep = max(h.x.shape[0] for h in host) + 5, max(h.edge_index2.shape[1] for h in host) + 17
    d = dev()
    torch.manual_seed(0)
    m1 = GNNML3("zinc", pool.K, pool.F, precision="bf16").to(d)
    torch.manual_seed(0)
    m2 = GNNML3("zinc", pool.K, pool.F, precision="bf16").to(d)
    eager = Trainer(m1, loss="l1", lr=1e-3)
    gt = GraphedTrainer(m2, pad_batch(host[0], Np, Ep), loss="l1", lr=1e-3, warmup=1)
    with torch.no_grad():                          # rewind the warm-up step in place (the graph holds these addresses)
        for a, b in zip(m2.parameters(), m1.parameters()):
            a.copy_(b)
        for st in gt.opt.state.values():
            for v in st.values():
                if isinstance(v, torch.Tensor):
                    v.zero_()
    for i, hb in enumerate(host):
        l1 = float(eager.step(hb.to(d)))
        if i % 2 == 0:
            l2 = float(gt.step(pad_batch(hb, Np, Ep).to(d)))
        else:
            gt.load_unpadded(hb.to(d))
            l2 = float(gt.step())
        assert abs(l1 - l2) <= 2e-5 * abs(l1), (i, l1, l2)
        for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
            assert torch.allclose(a, b, rtol=0, atol=2e-6), (i, k)


def test_evaluator_on_a_tf32_gnnml3_equals_eager_loop():
    from gnn_matlang_b200.models import GNNML3
    from test_gpu_eval import _check, _pool_dataset
    pool, dds = _pool_dataset("zinc", 1200, 11)
    ids = np.random.default_rng(2).permutation(1200)[:1000]
    torch.manual_seed(0)
    model = GNNML3("zinc", pool.K, pool.F, precision="tf32").to(dev())
    _check(model, dds, ids, 128, "l1", "GNNML3 zinc tf32")


# ----------------------------------------------------------------------------------------------------------------------------
# F. C ABI
# ----------------------------------------------------------------------------------------------------------------------------

def test_gemm_abi_rejects_unknown_precision():
    """gnnml3_gemm_nn / gnnml3_gemm_tn: an unknown precision is GNNML3_ERR_INVALID (1) with a message naming it, and the
    output is left untouched."""
    from gnn_matlang_b200 import _lib
    lib = _lib.load()
    P = _lib.ptr
    d = dev()
    g = torch.Generator().manual_seed(2)
    M, Kc, Nc = 3000, 40, 24
    A = torch.randn(M, Kc, generator=g).to(d)
    B = torch.randn(Kc, Nc, generator=g).to(d)
    Bt = torch.randn(M, Nc, generator=g).to(d)
    ws = torch.empty(lib.gnnml3_gemm_tn_workspace_bytes(M, Kc, Nc), dtype=torch.uint8, device=d)
    for bad in (3, -1, 0x100):
        C = torch.full((M, Nc), 7.0, device=d)
        assert lib.gnnml3_gemm_nn(P(A), Kc, P(B), Nc, None, P(C), Nc, M, Nc, Kc, bad, _lib.EPI_NONE, _lib.stream_ptr()) == 1
        assert b"precision" in lib.gnnml3_last_error()
        Ct = torch.full((Kc, Nc), 7.0, device=d)
        assert lib.gnnml3_gemm_tn(P(A), Kc, P(Bt), Nc, P(Ct), Nc, M, Kc, Nc, bad, P(ws), ws.numel(), _lib.stream_ptr()) == 1
        assert b"precision" in lib.gnnml3_last_error()
        torch.cuda.synchronize()
        assert bool((C == 7.0).all()) and bool((Ct == 7.0).all())
