"""GNNML1 on the B200: the fused layer kernels (ml1_layer.cu) against oracle autograd, determinism, full-size properties,
the model against the oracle model, the 1-WL known answers of the paper (EXP, SR25, graph8c) and CUDA-graph capture.

Layer bar: |a - ref| <= 1e-5 |ref| + 1e-5 max|ref| (test_gpu_kernels.assert_close) against a float64 evaluation of the oracle.
Gradients are compared with gy zeroed where a pre-activation lies within 1e-4 of the ReLU kink (two evaluations may put it on
different sides); everything else is compared as is."""
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


def _random_graph(N, E, seed, isolated=0.1):
    rng = np.random.default_rng(seed)
    live = np.flatnonzero(rng.random(N) >= isolated) if N > 1 else np.arange(N)
    if len(live) == 0 or E == 0:
        return torch.zeros(2, 0, dtype=torch.int64)
    return torch.from_numpy(live[rng.integers(0, len(live), (2, E))].astype(np.int64))


def _layer_ref(layer, x, ei, gy_fn):
    """float64 oracle forward + autograd; returns (y, gy used, dx, {param: grad})."""
    p = {o: getattr(layer, n.split(".")[0]).__getattr__(n.split(".")[1]).detach().cpu().double().requires_grad_(True)
         for n, o in zip(PNAMES, ONAMES)}
    xd = x.detach().cpu().double().requires_grad_(True)
    eic = ei.cpu()
    y = ml1layer_forward(xd, eic, p, layer.concat)
    with torch.no_grad():
        pre = ml1layer_forward(xd, eic, p, layer.concat, act=lambda v: v)
    gy = gy_fn(y.shape) * (pre.abs() > 1e-4).double()
    y.backward(gy)
    return y.detach(), gy.float(), xd.grad, {n: p[o].grad for n, o in zip(PNAMES, ONAMES)}


def _check_layer(layer, x, ei, seed=0, name=""):
    g = torch.Generator().manual_seed(seed)
    yr, gy, dxr, gr = _layer_ref(layer, x, ei, lambda s: torch.randn(*s, generator=g, dtype=torch.float64))
    xg = x.detach().clone().requires_grad_(True) if x.is_leaf else x
    layer.zero_grad()
    y = layer(xg, ei)
    y.backward(gy.to(y.device))
    assert_close(y, yr, name=name + " y")
    assert_close(xg.grad if x.is_leaf else x.grad, dxr, name=name + " dx")
    for n in PNAMES:
        mod, attr = n.split(".")
        assert_close(getattr(getattr(layer, mod), attr).grad, gr[n], name=name + " d" + n)


def _layer(Fi, Fo, concat, seed=0):
    from gnn_matlang_b200.libs.spect_conv import ML1Layer
    torch.manual_seed(seed)
    layer = ML1Layer(Fi, Fo, concat=concat)
    with torch.no_grad():                          # non-zero biases (the reference initialises conv.bias to zero)
        layer.conv1.bias.normal_(0, 0.3)
    return layer.to(dev())


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
@pytest.mark.parametrize("Fo", [8, 30, 64])
@pytest.mark.parametrize("Fi", [1, 3, 25, 32, 64])
def test_layer_matches_oracle(Fi, Fo, concat):
    from gnn_matlang_b200.libs.spect_conv import ML1_PATH_COUNTS
    N, E = 1000 + 37 * Fi + Fo, 4000 + 11 * Fo
    ei = _random_graph(N, E, seed=Fi * 100 + Fo).to(dev())
    x = torch.randn(N, Fi, generator=torch.Generator().manual_seed(Fi + Fo)).to(dev())
    layer = _layer(Fi, Fo, concat, seed=Fi + 3 * Fo)
    before = dict(ML1_PATH_COUNTS)
    _check_layer(layer, x, ei, seed=Fo, name="Fi=%d Fo=%d concat=%d" % (Fi, Fo, concat))
    assert ML1_PATH_COUNTS["fused"] == before["fused"] + 1 and ML1_PATH_COUNTS["composed"] == before["composed"]


@pytest.mark.parametrize("case", ["graph8c_batch", "no_edges", "tiny", "column_block_view", "isolated_heavy"])
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_layer_edge_cases(case, concat):
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.batch import collate
    Fi, Fo = 16, 24
    if case == "graph8c_batch":
        gs = read_graph6(os.path.join(GOLDEN, "graph8c.g6"), feature_dim=Fi)[:301]
        b = collate(gs, adjacency=True)
        ei, N = b.edge_index, b.x.shape[0]
    elif case == "no_edges":
        N, ei = 333, torch.zeros(2, 0, dtype=torch.int64)
    elif case == "tiny":
        N, ei = 1, torch.zeros(2, 0, dtype=torch.int64)
    elif case == "isolated_heavy":
        N, ei = 517, _random_graph(517, 300, seed=5, isolated=0.7)
    else:
        N, ei = 700, _random_graph(700, 2500, seed=6)
    g = torch.Generator().manual_seed(11)
    ei = ei.to(dev())
    layer = _layer(Fi, Fo, concat, seed=4)
    if case == "column_block_view":
        # x = a column block of a wider activation (row stride 40, offset 8 floats): consumed in place, no copy
        wide = torch.randn(N, 40, generator=g).to(dev()).requires_grad_(True)
        x = wide[:, 8:8 + Fi]
        gref = torch.Generator().manual_seed(2)
        yr, gy, dxr, gr = _layer_ref(layer, x, ei, lambda s: torch.randn(*s, generator=gref, dtype=torch.float64))
        n0 = _lib.launch_count()
        y = layer(x, ei)
        y.backward(gy.to(dev()))
        assert _lib.launch_count() > n0
        assert_close(y, yr, name="view y")
        assert_close(wide.grad[:, 8:8 + Fi], dxr, name="view dx")
        assert float(wide.grad[:, :8].abs().max()) == 0.0 and float(wide.grad[:, 8 + Fi:].abs().max()) == 0.0
        for n in PNAMES:
            mod, attr = n.split(".")
            assert_close(getattr(getattr(layer, mod), attr).grad, gr[n], name="view d" + n)
        return
    x = torch.randn(N, Fi, generator=g).to(dev())
    _check_layer(layer, x, ei, seed=3, name=case)


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_out_of_envelope_shape_takes_the_composed_path(concat):
    """Fo = 96 is outside the fused kernel (gnnml3_ml1layer_supported): the layer composes the aggregation kernel and the
    tensor-core GEMMs, with the same result contract."""
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.libs.spect_conv import ML1_PATH_COUNTS
    assert not ops.ml1layer_supported(32, 96, concat) and not ops.ml1layer_supported(80, 32, concat)
    N = 900
    ei = _random_graph(N, 3000, seed=9).to(dev())
    x = torch.randn(N, 32, generator=torch.Generator().manual_seed(4)).to(dev())
    layer = _layer(32, 96, concat, seed=8)
    before = dict(ML1_PATH_COUNTS)
    _check_layer(layer, x, ei, seed=5, name="Fo=96")
    assert ML1_PATH_COUNTS["composed"] == before["composed"] + 1 and ML1_PATH_COUNTS["fused"] == before["fused"]


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_layer_is_deterministic(concat):
    N = 20000
    ei = _random_graph(N, 150000, seed=12).to(dev())
    x = torch.randn(N, 64, generator=torch.Generator().manual_seed(1)).to(dev())
    gy = torch.randn(N, 64 * (3 if concat else 1), generator=torch.Generator().manual_seed(2)).to(dev())
    layer = _layer(64, 64, concat, seed=3)
    outs = []
    for _ in range(2):
        xg = x.clone().requires_grad_(True)
        layer.zero_grad()
        y = layer(xg, ei)
        y.backward(gy)
        outs.append([y.detach().clone(), xg.grad.clone()] + [p.grad.clone() for p in layer.parameters()])
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _dot(a, b):
    return float((a.double() * b.double()).sum())


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_full_size_adjoint_and_linearity_properties(concat):
    """1 M nodes (batched ZINC-shaped graphs), Fi = Fo = 64.  With the fc12 / fc13 branch switched off (zero weights and biases)
    and no biases, the layer's pre-activation z is linear in x; y = relu(z) with the mask fixed by a forward pass, so
    <y, g> = <x, dx> (adjointness of the fused forward and the fused dx kernel) and sum over parameters <W, dW> = <y, g>
    (weight-gradient contraction).  Linearity: z(a x1 + b x2) = a z(x1) + b z(x2) on the pre-activation (no ReLU: checked
    through the concat mode's conv and fc11 blocks, which are exactly relu of linear maps, on inputs where the mask agrees)."""
    from gnn_matlang_b200.synthetic import zinc_graph
    rng = np.random.default_rng(0)
    eis, off = [], 0
    while off < 1000000:
        n, ei, _ = zinc_graph(rng)
        eis.append(ei + off)
        off += n
    N = off
    ei = torch.from_numpy(np.concatenate(eis, 1)).to(dev())
    layer = _layer(64, 64, concat, seed=1)
    with torch.no_grad():
        for fc in (layer.fc12, layer.fc13):
            fc.weight.zero_()
            fc.bias.zero_()
        layer.fc11.bias.zero_()
        layer.conv1.bias.zero_()
    g = torch.Generator().manual_seed(3)
    x1 = torch.randn(N, 64, generator=g).to(dev()).requires_grad_(True)
    x2 = torch.randn(N, 64, generator=g).to(dev())
    y1 = layer(x1, ei)
    gout = torch.randn(*y1.shape, generator=g).to(dev())
    y1.backward(gout)
    L = _dot(y1.detach(), gout)
    scale = float((y1.detach().double().abs() * gout.double().abs()).sum())
    assert abs(_dot(x1.detach(), x1.grad) - L) <= 2e-6 * scale, ("dx", _dot(x1.detach(), x1.grad), L, scale)
    wsum = sum(_dot(p.detach(), p.grad) for p in (layer.conv1.weight, layer.fc11.weight))
    assert abs(wsum - L) <= 2e-6 * scale, ("dW", wsum, L)
    with torch.no_grad():
        a, b = 0.75, -1.5
        y2 = layer(x2, ei)
        y3 = layer(a * x1.detach() + b * x2, ei)
        # relu(z) for the three inputs; where z(x1), z(x2) and z(a x1 + b x2) = a z1 + b z2 are all positive the outputs are linear
        both = (y1 > 1e-3) & (y2 > 1e-3) & (y3 > 1e-3)
        ref = a * y1.double() + b * y2.double()
        err = ((y3.double() - ref).abs() * both).max().item()
    assert int(both.sum()) > N // 20
    assert err <= 2e-5 * ref.abs().max().item(), (err, ref.abs().max().item())


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


def _oracle_copy(model, cfg, ninp, nlayer, nout, concat):
    o = OracleGNNML1(cfg, ninp, nlayer, nout, concat).double()
    o.load_state_dict({k: v.detach().cpu().double() for k, v in model.state_dict().items()})
    return o


def _ob(b):
    return dict(x=b.x.double(), edge_index=b.edge_index, batch=b.batch, num_graphs=b.num_graphs)


@pytest.mark.parametrize("cfg", ["graph8c", "zinc"])
@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_model_matches_oracle_model(cfg, concat):
    """Forward and every gradient at 1e-4 (the model bar of test_gpu_model.py) on batches whose pre-activations all keep a margin
    of 2e-6 of their layer's scale from the ReLU kink (seeds are drawn until one does; a real defect fails every seed).  The
    batches are small (40 graph8c graphs, 8 ZINC-shaped graphs) so that such a batch exists."""
    from gnn_matlang_b200.models import GNNML1
    ninp, nlayer, nout = (1, 3, 64) if cfg == "graph8c" else (25, 4, 64)
    for seed in range(32):
        b = _graph8c_batch(500 * seed, 40) if cfg == "graph8c" else _zinc_batch(8, seed)
        torch.manual_seed(seed)
        model = GNNML1(cfg, ninp, nlayer, nout, concat)
        o = _oracle_copy(model, cfg, ninp, nlayer, nout, concat)
        margin_ok = True
        xo = _ob(b)
        with torch.no_grad():
            h = xo["x"]
            for l in range(1, nlayer + 1):
                p = {}
                p["conv.weight"], p["conv.bias"] = getattr(o, "conv%d1" % l).weight, getattr(o, "conv%d1" % l).bias
                for j, n in ((1, "fcA"), (2, "fcB"), (3, "fcC")):
                    p[n + ".weight"], p[n + ".bias"] = getattr(o, "fc%d%d" % (l, j)).weight, getattr(o, "fc%d%d" % (l, j)).bias
                pre = ml1layer_forward(h, xo["edge_index"], p, concat, act=lambda v: v)
                # (concat: the product block changes sign only where a factor does, so its factors carry the margin)
                blocks = [pre[:, :2 * nout], h @ p["fcB.weight"].t() + p["fcB.bias"], h @ p["fcC.weight"].t() + p["fcC.bias"]] if concat else [pre]
                margin_ok &= all(bool((t.abs() > 2e-6 * t.abs().max()).all()) for t in blocks)
                h = torch.relu(pre)
        if not margin_ok:
            continue
        ref = o(xo)
        ref.sum().backward() if cfg == "graph8c" else (ref ** 2).sum().backward()
        m = model.to(dev())
        bd = b.to(dev())
        out = m(bd)
        out.sum().backward() if cfg == "graph8c" else (out ** 2).sum().backward()
        assert_close(out, ref, rtol=1e-4, name=cfg + " out")
        refp = dict(o.named_parameters())
        for k, v in m.named_parameters():
            assert_close(v.grad, refp[k].grad, rtol=1e-4, name=cfg + " d" + k)
        return
    pytest.fail("no seed gave a batch with a kink margin")


def _embed(model, b):
    with torch.no_grad():
        return model(b.to(dev())).double()


def _undistinguished(emb, thr=1e-3):
    """Pairs (i < j) whose embeddings are within thr in L1 (the reference's criterion); also the smallest |d - thr|."""
    n = emb.size(0)
    count, margin = 0, float("inf")
    for i0 in range(0, n, 2048):
        d = torch.cdist(emb[i0:i0 + 2048], emb, p=1)
        rows = torch.arange(i0, min(i0 + 2048, n), device=emb.device)
        upper = torch.arange(n, device=emb.device)[None, :] > rows[:, None]
        count += int(((d < thr) & upper).sum())
        margin = min(margin, float(((d - thr).abs() + (~upper) * 1e9).min()))
    return count, margin


def test_exp_pairs_are_not_distinguished():
    """EXP pairs are 1-WL-equivalent by construction: GNNML1 gives both graphs of each of the 100 committed pairs the same output
    (L1 < 1e-3), whereas GNNML3 separates them (test_gpu_config3_exp.py)."""
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import ExpPool
    pool = ExpPool()
    gs = []
    for i in range(len(pool.n)):
        gs.append(dict(x=pool.x[pool.node_off[i]:pool.node_off[i + 1]],
                       edge_index=pool.ei1[:, pool.edge_off1[i]:pool.edge_off1[i + 1]]))
    torch.manual_seed(0)
    model = GNNML1("exp", ninp=1).to(dev()).eval()
    emb = _embed(model, collate(gs, adjacency=True))
    d = (emb[0::2] - emb[1::2]).abs().sum(1)
    print("EXP: largest pair distance %.3e over %d pairs" % (float(d.max()), d.numel()))
    assert d.numel() == 100 and bool((d < 1e-3).all())


def test_sr25_pairs_are_not_distinguished():
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.models import GNNML1
    gs = read_graph6(os.path.join(GOLDEN, "sr251256.g6"))
    torch.manual_seed(0)
    model = GNNML1("graph8c", ninp=1).to(dev()).eval()
    emb = _embed(model, collate(gs, adjacency=True))
    count, margin = _undistinguished(emb)
    print("SR25: %d of %d pairs undistinguished" % (count, len(gs) * (len(gs) - 1) // 2))
    assert len(gs) == 15 and count == 105


def test_graph8c_undistinguished_pairs_match_the_oracle():
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.models import GNNML1
    gs = read_graph6(os.path.join(GOLDEN, "graph8c.g6"))
    b = collate(gs, adjacency=True)
    torch.manual_seed(0)
    model = GNNML1("graph8c", ninp=1).eval()
    o = _oracle_copy(model, "graph8c", 1, 3, 64, False).eval()
    with torch.no_grad():
        ref = o(_ob(b)).to(dev())
    emb = _embed(model.to(dev()), b)
    count, margin = _undistinguished(emb)
    rcount, rmargin = _undistinguished(ref)
    print("graph8c: %d graphs, %d undistinguished pairs (oracle %d); nearest pair |L1 - 1e-3| = %.3e (oracle %.3e)"
          % (len(gs), count, rcount, margin, rmargin))
    assert len(gs) == 11117 and count == rcount
    assert_close(emb, ref, rtol=1e-4, name="graph8c embeddings")


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_captured_layer_replays_to_the_eager_result(concat):
    N = 5000
    ei = _random_graph(N, 20000, seed=21).to(dev())
    layer = _layer(32, 30, concat, seed=2)
    x = torch.randn(N, 32, generator=torch.Generator().manual_seed(1)).to(dev()).requires_grad_(True)
    gy = torch.randn(N, 30 * (3 if concat else 1), generator=torch.Generator().manual_seed(2)).to(dev())
    y = layer(x, ei)                                  # eager (also builds the graph plan outside the capture)
    y.backward(gy)
    eager = [y.detach().clone(), x.grad.clone()] + [p.grad.clone() for p in layer.parameters()]
    del y                                             # (frees the eager autograd graph: no node of it may outlive into the capture)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                        # warm-up on the capture stream (workspaces are per stream)
        for _ in range(2):
            x.grad = None
            layer.zero_grad(set_to_none=True)
            layer(x, ei).backward(gy)
    torch.cuda.current_stream().wait_stream(s)
    x.grad = None
    layer.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        yc = layer(x, ei)
        yc.backward(gy)
    graph.replay()
    torch.cuda.synchronize()
    got = [yc.detach(), x.grad] + [p.grad for p in layer.parameters()]
    for a, b in zip(got, eager):
        assert torch.equal(a, b)
