"""GNNML1 in its reduced-precision modes on the B200: ``precision="tf32"`` (one tensor-core product per k-step on the raw FP32
operand, truncated by the tensor core, against RN-TF32 weights) and ``precision="bf16"`` (RN-BF16 operands and weights, FP32
accumulation) of the fused layer kernel (ml1_layer.cu), the C ABI's *_precision entry points, the composed path, the whole
model, forward-only inference and the captured training step and evaluation pass.

Bars, relative to the result's scale (test_gpu_kernels.assert_close: |a - ref| <= rtol |ref| + rtol max|ref|), the ones
GNNML3's flagged modes state: at the kernel level 2e-3 (TF32: 10-bit mantissa, A truncated) and 2e-2 (BF16: 8-bit mantissa);
module and model level 5e-3 and 5e-2.  Reduced precision moves pre-activations within about the bar of zero across the ReLU
kink, which changes single gradient entries by O(1): gradients are held to the module bar in the Frobenius norm and entry-wise
for at least 99 % of the entries of large tensors (as test_gpu_fused.test_ml3layer_module_in_flagged_precision does), and the
layer tests zero gy where a pre-activation lies within twice the kernel bar of the kink, so that no flip can happen there."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from gnnml1_oracle import OracleGNNML1, ml1layer_forward  # noqa: E402
from test_gpu_kernels import assert_close, dev  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
PNAMES = ["conv1.weight", "conv1.bias", "fc11.weight", "fc11.bias", "fc12.weight", "fc12.bias", "fc13.weight", "fc13.bias"]
ONAMES = ["conv.weight", "conv.bias", "fcA.weight", "fcA.bias", "fcB.weight", "fcB.bias", "fcC.weight", "fcC.bias"]
KERNEL_BAR = {"tf32": 2e-3, "bf16": 2e-2}
MODULE_BAR = {"tf32": 5e-3, "bf16": 5e-2}
FLAGGED = ["tf32", "bf16"]


def _random_graph(N, E, seed, isolated=0.1):
    rng = np.random.default_rng(seed)
    live = np.flatnonzero(rng.random(N) >= isolated) if N > 1 else np.arange(N)
    if len(live) == 0 or E == 0:
        return torch.zeros(2, 0, dtype=torch.int64)
    return torch.from_numpy(live[rng.integers(0, len(live), (2, E))].astype(np.int64))


def _layer(Fi, Fo, concat, precision, seed=0):
    from gnn_matlang_b200.libs.spect_conv import ML1Layer
    torch.manual_seed(seed)
    layer = ML1Layer(Fi, Fo, concat=concat, precision=precision)
    with torch.no_grad():                          # non-zero biases (the reference initialises conv.bias to zero)
        layer.conv1.bias.normal_(0, 0.3)
    return layer.to(dev())


def _oracle_params(layer):
    return {o: getattr(layer, n.split(".")[0]).__getattr__(n.split(".")[1]).detach().cpu().double().requires_grad_(True)
            for n, o in zip(PNAMES, ONAMES)}


def _layer_ref(layer, x, ei, seed, margin):
    """float64 oracle forward + autograd with gy zeroed where |pre-activation| <= margin * max|pre-activation| (per layer block).
    -> (y, [p1 | p2], gy used, dx, {param: grad})"""
    p = _oracle_params(layer)
    xd = x.detach().cpu().double().requires_grad_(True)
    eic = ei.cpu()
    y = ml1layer_forward(xd, eic, p, layer.concat)
    with torch.no_grad():
        pre = ml1layer_forward(xd, eic, p, layer.concat, act=lambda v: v)
        p1 = xd @ p["fcB.weight"].t() + p["fcB.bias"]
        p2 = xd @ p["fcC.weight"].t() + p["fcC.bias"]
        keep = pre.abs() > margin * pre.abs().max().clamp_min(1e-30)
        if layer.concat:                           # the product block flips where a factor does: its factors carry the margin
            Fo = p1.size(1)
            for q in (p1, p2):
                keep[:, 2 * Fo:] &= q.abs() > margin * q.abs().max().clamp_min(1e-30)
    g = torch.Generator().manual_seed(seed)
    gy = torch.randn(*y.shape, generator=g, dtype=torch.float64) * keep.double()
    y.backward(gy)
    return y.detach(), torch.cat([p1, p2], 1), gy.float(), xd.grad, {n: p[o].grad for n, o in zip(PNAMES, ONAMES)}


def _rel_err(a, ref):
    a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _close_in_norm(a, ref, rtol, name):
    """Frobenius-norm bound at 4 rtol; entry-wise (rtol |ref| + rtol max|ref|) for at least 99 % of a large tensor's entries."""
    a, ref = a.detach().cpu().double(), ref.detach().cpu().double()
    assert a.shape == ref.shape, (name, a.shape, ref.shape)
    if ref.numel() == 0 or float(ref.norm()) == 0.0:
        assert float(a.abs().max()) == 0.0 if a.numel() else True, name
        return
    rel = float((a - ref).norm() / ref.norm())
    frac_bad = float(((a - ref).abs() > rtol * ref.abs() + rtol * ref.abs().max()).double().mean())
    assert rel <= 4 * rtol, "%s: relative Frobenius error %.3e" % (name, rel)
    if ref.numel() >= 10000:
        assert frac_bad <= 0.01, "%s: %.2f %% entries off" % (name, 100 * frac_bad)


def _check_layer(layer, x, ei, precision, seed, name, x_leaf=None):
    """Forward (y and aux through the library call, y through the module) at the kernel bar, the mode really reduced, the
    backward (dx and the eight parameter gradients) at the module bar, and the backward passes really reduced."""
    from gnn_matlang_b200 import _lib, ops
    from gnn_matlang_b200.graph import get_plan
    from gnn_matlang_b200.libs.spect_conv import _PRECISIONS
    kb, mb = KERNEL_BAR[precision], MODULE_BAR[precision]
    yr, auxr, gy, dxr, gr = _layer_ref(layer, x, ei, seed, margin=2 * kb)
    plan = get_plan(ei, x.size(0))
    w = [getattr(layer, n.split(".")[0]).__getattr__(n.split(".")[1]).detach() for n in PNAMES]
    y0, aux0, _ = ops.ml1layer_forward(plan, ops.aligned_rows(x.detach()), w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7],
                                       concat=layer.concat, precision=_PRECISIONS[precision])
    assert_close(y0, yr, rtol=kb, name=name + " y")
    assert_close(aux0, auxr, rtol=kb, name=name + " aux")
    ey, ea = _rel_err(y0, yr), _rel_err(aux0, auxr)
    print("%s: y error %.2e, aux error %.2e of the scale" % (name, ey, ea))
    if yr.numel() and float(yr.abs().max()) > 0:
        # a silent fall-through to 3xTF32 would sit at ~1e-7
        assert ey > 1e-5 or ea > 1e-5, "suspiciously exact for %s: %.2e / %.2e" % (precision, ey, ea)
    xg = x_leaf if x_leaf is not None else x.detach().clone().requires_grad_(True)
    layer.zero_grad()
    y = layer(xg[:, 8:8 + x.size(1)] if x_leaf is not None else xg, ei)
    assert torch.equal(y.detach(), y0), name + ": the module and the library call differ"
    y.backward(gy.to(y.device))
    dx = xg.grad[:, 8:8 + x.size(1)] if x_leaf is not None else xg.grad
    _close_in_norm(dx, dxr, mb, name + " dx")
    for n in PNAMES:
        mod, attr = n.split(".")
        _close_in_norm(getattr(getattr(layer, mod), attr).grad, gr[n], mb, name + " d" + n)
    # the backward's own arithmetic, isolated: the flagged dx pass and weight-gradient contraction against the 3xTF32 ones on
    # identical inputs (the same y, aux and gy; d fc11.weight = x^T gA depends on nothing else).  A silent fall-through to
    # 3xTF32 gives the same bits; the reduced passes stay within the kernel bar in the Frobenius norm.
    args = (plan, ops.aligned_rows(x.detach()), w[0], w[2], w[4], w[6], y0, aux0, gy.to(dev()), True)
    got = ops.ml1layer_backward(*args, concat=layer.concat, precision=_PRECISIONS[precision])
    full = ops.ml1layer_backward(*args, concat=layer.concat, precision=_lib.PREC_3XTF32)
    for i, what in ((0, "dx pass"), (3, "weight-gradient contraction (d fc11.weight)")):
        a, r = got[i].detach().cpu().double(), full[i].detach().cpu().double()
        if float(r.norm()) == 0.0:
            continue
        rel = float((a - r).norm() / r.norm())
        print("%s: %s differs from 3xTF32 by %.2e (Frobenius, relative)" % (name, what, rel))
        assert rel > 1e-6, "%s: %s suspiciously exact for %s: %.2e" % (name, what, precision, rel)
        assert rel <= kb, "%s: %s off by %.2e" % (name, what, rel)
    return xg


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
@pytest.mark.parametrize("Fo", [8, 30, 64])
@pytest.mark.parametrize("Fi", [1, 3, 25, 32, 64])
def test_layer_matches_oracle(Fi, Fo, concat, precision):
    from gnn_matlang_b200.libs.spect_conv import ML1_PATH_COUNTS
    N, E = 1000 + 37 * Fi + Fo, 4000 + 11 * Fo
    ei = _random_graph(N, E, seed=Fi * 100 + Fo).to(dev())
    x = torch.randn(N, Fi, generator=torch.Generator().manual_seed(Fi + Fo)).to(dev())
    layer = _layer(Fi, Fo, concat, precision, seed=Fi + 3 * Fo)
    before = dict(ML1_PATH_COUNTS)
    _check_layer(layer, x, ei, precision, seed=Fo, name="%s Fi=%d Fo=%d concat=%d" % (precision, Fi, Fo, concat))
    assert ML1_PATH_COUNTS["fused"] == before["fused"] + 1 and ML1_PATH_COUNTS["composed"] == before["composed"]


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("case", ["no_edges", "isolated_heavy", "column_block_view"])
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_layer_edge_cases(case, concat, precision):
    Fi, Fo = 16, 24
    g = torch.Generator().manual_seed(11)
    if case == "no_edges":
        N, ei = 333, torch.zeros(2, 0, dtype=torch.int64)
    elif case == "isolated_heavy":
        N, ei = 517, _random_graph(517, 300, seed=5, isolated=0.7)
    else:
        N, ei = 700, _random_graph(700, 2500, seed=6)
    ei = ei.to(dev())
    layer = _layer(Fi, Fo, concat, precision, seed=4)
    name = "%s %s concat=%d" % (precision, case, concat)
    if case == "column_block_view":
        # x = a column block of a wider activation (row stride 40, offset 8 floats): consumed in place
        wide = torch.randn(N, 40, generator=g).to(dev()).requires_grad_(True)
        _check_layer(layer, wide.detach()[:, 8:8 + Fi], ei, precision, seed=2, name=name, x_leaf=wide)
        assert float(wide.grad[:, :8].abs().max()) == 0.0 and float(wide.grad[:, 8 + Fi:].abs().max()) == 0.0
        return
    _check_layer(layer, torch.randn(N, Fi, generator=g).to(dev()), ei, precision, seed=3, name=name)


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_out_of_envelope_shape_takes_the_composed_path_in_tf32(concat):
    """Fo = 96 is outside the fused kernel: the layer composes the aggregation kernel and the tensor-core GEMMs at the given
    precision.  Bit-equal to that composition written out at PREC_TF32, at the TF32 bar against the oracle, and not 3xTF32."""
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.graph import get_plan
    from gnn_matlang_b200.libs.spect_conv import ML1_PATH_COUNTS, _AggregateFn, _LinearFn
    N, Fi, Fo = 900, 32, 96
    ei = _random_graph(N, 3000, seed=9).to(dev())
    x = torch.randn(N, Fi, generator=torch.Generator().manual_seed(4)).to(dev())
    layer = _layer(Fi, Fo, concat, "tf32", seed=8)
    before = dict(ML1_PATH_COUNTS)
    with torch.no_grad():
        y = layer(x, ei)
        plan = get_plan(ei, N)
        prec = _lib.PREC_TF32
        ax = _AggregateFn.apply(x, torch.ones(plan.E, 1, device=dev()), plan)
        pa = _LinearFn.apply(x, layer.fc11.weight.t(), layer.fc11.bias, prec)
        pc = _LinearFn.apply(ax, layer.conv1.weight[0], layer.conv1.bias, prec)
        pp = _LinearFn.apply(x, layer.fc12.weight.t(), layer.fc12.bias, prec) * _LinearFn.apply(x, layer.fc13.weight.t(), layer.fc13.bias, prec)
        comp = torch.cat([torch.relu(pa), torch.relu(pc), torch.relu(pp)], 1) if concat else torch.relu(pa + pc + pp)
    assert ML1_PATH_COUNTS["composed"] == before["composed"] + 1 and ML1_PATH_COUNTS["fused"] == before["fused"]
    assert torch.equal(y, comp)
    yr = ml1layer_forward(x.cpu().double(), ei.cpu(), {k: v.detach() for k, v in _oracle_params(layer).items()}, concat)
    assert_close(y, yr, rtol=KERNEL_BAR["tf32"], name="composed tf32 y")
    err = _rel_err(y, yr)
    print("composed Fo=96 tf32 concat=%d: y error %.2e of the scale" % (concat, err))
    assert err > 1e-5, "suspiciously exact: %.2e" % err


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_forward_only_equals_grad_mode(concat, precision, monkeypatch):
    """no_grad, inference_mode and frozen parameters take the forward-only instantiation: y bit-equal to the grad-mode forward,
    and no aux requested from the library."""
    from gnn_matlang_b200.libs import spect_conv
    layer = _layer(40, 64, concat, precision, seed=3)
    ei = _random_graph(5000, 30000, seed=4).to(dev())
    x = torch.randn(5000, 40, generator=torch.Generator().manual_seed(5)).to(dev())
    calls = []
    real = spect_conv.ops.ml1layer_forward

    def spy(*a, **k):
        calls.append((k.get("aux", True), k.get("precision")))
        return real(*a, **k)

    monkeypatch.setattr(spect_conv.ops, "ml1layer_forward", spy)
    ref = layer(x, ei)
    assert ref.requires_grad and calls[-1] == (True, spect_conv._PRECISIONS[precision])
    outs = {}
    with torch.no_grad():
        outs["no_grad"] = layer(x, ei)
    with torch.inference_mode():
        outs["inference_mode"] = layer(x, ei)
    for p in layer.parameters():
        p.requires_grad_(False)
    outs["frozen"] = layer(x, ei)
    assert [c[0] for c in calls[1:]] == [False] * 3
    assert all(c[1] == spect_conv._PRECISIONS[precision] for c in calls)
    for k, v in outs.items():
        assert torch.equal(v, ref.detach()), "%s: %s forward differs from the grad-mode forward" % (precision, k)


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_layer_is_deterministic(concat, precision):
    N = 20000
    ei = _random_graph(N, 150000, seed=12).to(dev())
    x = torch.randn(N, 64, generator=torch.Generator().manual_seed(1)).to(dev())
    gy = torch.randn(N, 64 * (3 if concat else 1), generator=torch.Generator().manual_seed(2)).to(dev())
    layer = _layer(64, 64, concat, precision, seed=3)
    outs = []
    for _ in range(2):
        xg = x.clone().requires_grad_(True)
        layer.zero_grad()
        y = layer(xg, ei)
        y.backward(gy)
        outs.append([y.detach().clone(), xg.grad.clone()] + [p.grad.clone() for p in layer.parameters()])
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _abi_args(plan, x, layer, concat):
    """Arguments of gnnml3_ml1layer_forward / _backward (fresh outputs each call) for the layer's parameters."""
    from gnn_matlang_b200 import _lib
    lib = _lib.load()
    N, Fi = x.shape
    Fo = layer.conv1.out_channels
    W = 3 * Fo if concat else Fo
    P = _lib.ptr
    w = [getattr(layer, n.split(".")[0]).__getattr__(n.split(".")[1]).detach().contiguous() for n in PNAMES]
    out = dict(y=torch.zeros(N, W, device=dev()), aux=torch.zeros(N, 2 * Fo, device=dev()), w=w,
               ws=torch.empty(lib.gnnml3_ml1layer_workspace_bytes(N, Fi, Fo, int(concat)), dtype=torch.uint8, device=dev()))
    fwd = (P(plan.rowptr), P(plan.col), N, plan.E, P(x), x.stride(0), Fi, P(w[0]), P(w[1]), P(w[2]), P(w[3]), P(w[4]), P(w[5]), P(w[6]),
           P(w[7]), Fo, int(concat), P(out["y"]), W, P(out["aux"]), 2 * Fo, None, 0, P(out["ws"]), out["ws"].numel(), _lib.stream_ptr())
    return out, fwd


def _abi_bwd(plan, x, out, gy, concat, Fo):
    from gnn_matlang_b200 import _lib
    N, Fi = x.shape
    P = _lib.ptr
    w = out["w"]
    g = dict(dx=torch.zeros(N, Fi, device=dev()), dwc=torch.zeros_like(w[0]), dwA=torch.zeros_like(w[2]), dwB=torch.zeros_like(w[4]),
             dwC=torch.zeros_like(w[6]), dbs=torch.zeros(4, Fo, device=dev()))
    args = (P(plan.rowptrT), P(plan.colT), N, plan.E, P(x), x.stride(0), Fi, P(w[0]), P(w[2]), P(w[4]), P(w[6]), Fo, int(concat),
            P(out["y"]), out["y"].stride(0), P(out["aux"]), 2 * Fo, P(gy), gy.stride(0), 1, P(g["dx"]), Fi, P(g["dwc"]), P(g["dbs"][0]),
            P(g["dwA"]), P(g["dbs"][1]), P(g["dwB"]), P(g["dbs"][2]), P(g["dwC"]), P(g["dbs"][3]), P(out["ws"]), out["ws"].numel(),
            _lib.stream_ptr())
    return g, args


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_abi_precision_entry_points(concat):
    """*_precision(..., GNNML3_PREC_3XTF32) is bit-identical to the plain entry points; an unknown precision is
    GNNML3_ERR_INVALID (1) with a message, and writes nothing."""
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.graph import get_plan
    lib = _lib.load()
    N, Fi, Fo = 3000, 32, 30
    ei = _random_graph(N, 12000, seed=31).to(dev())
    x = torch.randn(N, Fi, generator=torch.Generator().manual_seed(7)).to(dev())
    layer = _layer(Fi, Fo, concat, "fp32", seed=6)
    plan = get_plan(ei, N)
    gy = torch.randn(N, 3 * Fo if concat else Fo, generator=torch.Generator().manual_seed(8)).to(dev())
    res = {}
    for name in ("plain", "precision"):
        out, fwd = _abi_args(plan, x, layer, concat)
        rc = lib.gnnml3_ml1layer_forward(*fwd) if name == "plain" else lib.gnnml3_ml1layer_forward_precision(*fwd, _lib.PREC_3XTF32)
        assert rc == 0
        g, bwd = _abi_bwd(plan, x, out, gy, concat, Fo)
        rc = lib.gnnml3_ml1layer_backward(*bwd) if name == "plain" else lib.gnnml3_ml1layer_backward_precision(*bwd, _lib.PREC_3XTF32)
        assert rc == 0
        torch.cuda.synchronize()
        res[name] = [out["y"], out["aux"]] + [g[k] for k in ("dx", "dwc", "dwA", "dwB", "dwC", "dbs")]
    for a, b in zip(res["plain"], res["precision"]):
        assert torch.equal(a, b)
    for bad in (3, -1, 0x100):
        out, fwd = _abi_args(plan, x, layer, concat)
        assert lib.gnnml3_ml1layer_forward_precision(*fwd, bad) == 1
        assert b"precision" in lib.gnnml3_last_error()
        g, bwd = _abi_bwd(plan, x, out, gy, concat, Fo)
        assert lib.gnnml3_ml1layer_backward_precision(*bwd, bad) == 1
        assert b"precision" in lib.gnnml3_last_error()
        torch.cuda.synchronize()
        assert float(out["y"].abs().max()) == 0.0 and float(g["dx"].abs().max()) == 0.0


def _zinc_batch(B, seed):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.synthetic import zinc_graph
    rng = np.random.default_rng(seed)
    gs = []
    for _ in range(B):
        n, ei, x = zinc_graph(rng)
        gs.append(dict(x=x, edge_index=ei, y=np.float32(rng.standard_normal())))
    return collate(gs, adjacency=True)


def _graph8c_batch(first, count):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.datasets import read_graph6
    return collate(read_graph6(os.path.join(GOLDEN, "graph8c.g6"))[first:first + count], adjacency=True)


@pytest.mark.parametrize("precision", FLAGGED)
@pytest.mark.parametrize("cfg,ninp,concat", [("zinc", 25, False), ("graph8c", 1, True)])
def test_model_matches_oracle_model(cfg, ninp, concat, precision):
    """GNNML1(cfg, ninp, precision=...) forward at the module bar and every gradient at the module bar in norm, against the
    float64 oracle model with the same parameters."""
    from gnn_matlang_b200.models import GNNML1
    nlayer = 4 if cfg == "zinc" else 3
    b = _zinc_batch(64, 2) if cfg == "zinc" else _graph8c_batch(100, 200)
    torch.manual_seed(1)
    model = GNNML1(cfg, ninp, nlayer, 64, concat, precision=precision)
    o = OracleGNNML1(cfg, ninp, nlayer, 64, concat).double()
    o.load_state_dict({k: v.detach().cpu().double() for k, v in model.state_dict().items()})
    ref = o(dict(x=b.x.double(), edge_index=b.edge_index, batch=b.batch, num_graphs=b.num_graphs))
    ref.sum().backward() if cfg == "graph8c" else (ref ** 2).sum().backward()
    m = model.to(dev())
    out = m(b.to(dev()))
    out.sum().backward() if cfg == "graph8c" else (out ** 2).sum().backward()
    rtol = MODULE_BAR[precision]
    assert_close(out, ref, rtol=rtol, name="%s %s out" % (cfg, precision))
    err = _rel_err(out, ref)
    print("GNNML1 %s %s: output error %.2e of the scale" % (cfg, precision, err))
    assert err > 1e-6, "suspiciously exact: %.2e" % err
    refp = dict(o.named_parameters())
    for k, v in m.named_parameters():
        _close_in_norm(v.grad, refp[k].grad, rtol, "%s %s d%s" % (cfg, precision, k))


def _strip(hb):
    return hb.__class__(**{k: v for k, v in hb.__dict__.items() if k not in ("edge_index2", "edge_attr2")})


def test_captured_bf16_step_equals_eager_step():
    """GraphedTrainer runs whatever the model runs: a BF16 GNNML1 step, captured, equals the eager Trainer step to the bar of
    the fp32 GNNML1 training test (loss 2e-5 relative, parameters 2e-6 absolute after each Adam step)."""
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch, padded_shapes
    pool = GraphPool("zinc", 64, seed=6)
    rng = np.random.default_rng(3)
    ids = [rng.integers(0, 64, 48) for _ in range(3)]
    host = [_strip(pool.collate(i, adjacency=True)) for i in ids]
    Np, Ep, Mp = padded_shapes(host, adjacency=True)
    d = dev()
    torch.manual_seed(0)
    m1 = GNNML1("zinc", ninp=pool.F, precision="bf16").to(d)
    torch.manual_seed(0)
    m2 = GNNML1("zinc", ninp=pool.F, precision="bf16").to(d)
    eager = Trainer(m1, loss="l1", lr=1e-3)
    gt = GraphedTrainer(m2, pad_batch(host[0], Np, None, Mp), loss="l1", lr=1e-3, warmup=1)
    with torch.no_grad():                          # rewind the warm-up step in place (the graph holds these addresses)
        for a, b in zip(m2.parameters(), m1.parameters()):
            a.copy_(b)
        for st in gt.opt.state.values():
            for v in st.values():
                if isinstance(v, torch.Tensor):
                    v.zero_()
    dds = DeviceDataset(pool, d, adjacency=True, supports=False)
    for i, hb in enumerate(host):
        l1 = float(eager.step(hb.to(d)))
        if i == 0:
            l2 = float(gt.step(pad_batch(hb, Np, None, Mp).to(d)))
        else:
            if i == 1:
                gt.load_unpadded(hb.to(d))
            else:
                gt.load_from_dataset(dds, ids[i])
            l2 = float(gt.step())
        assert abs(l1 - l2) <= 2e-5 * abs(l1), (i, l1, l2)
    for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.allclose(a, b, rtol=0, atol=2e-6), k


def test_evaluator_on_a_bf16_model_equals_eager_loop():
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedEvaluator
    pool = GraphPool("zinc", 600, seed=12)
    dds = DeviceDataset(pool, dev(), adjacency=True, supports=False)
    ids = np.random.default_rng(3).permutation(600)[:450]
    torch.manual_seed(0)
    model = GNNML1("zinc", pool.F, precision="bf16").to(dev())
    res = GraphedEvaluator(model, dds, ids, 100, metric="l1").run(outputs=True)
    outs, s = [], 0.0
    model.eval()
    with torch.no_grad():
        for i in range(0, len(ids), 100):
            b = dds.collate(np.asarray(ids[i:i + 100], np.int64))
            o = model(b)
            o = o.unsqueeze(1) if o.dim() == 1 else o
            outs.append(o)
            s += float(np.abs(o.double().cpu().numpy() - b.y.double().cpu().numpy().reshape(o.shape)).sum())
    ref = torch.cat(outs)
    print("bf16 GNNML1 through the evaluator: sum %.9g (eager %.9g), largest output difference %.3e"
          % (res["sum"], s, float((res["outputs"] - ref).abs().max())))
    assert res["graphs"] == len(ids)
    assert_close(res["outputs"], ref, name="bf16 evaluator outputs")
    assert abs(res["sum"] - s) <= 1e-6 * abs(s), (res["sum"], s)
