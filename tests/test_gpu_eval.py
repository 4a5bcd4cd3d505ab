"""Forward-only inference and the captured evaluation pass on the B200.

* A forward nobody differentiates (``no_grad``, ``inference_mode``, every parameter frozen) takes the forward-only kernels: its
  output equals the grad-mode forward's bit for bit, and the library is asked for no aux / aggregate side output.
* ``train.GraphedEvaluator`` equals an eager reference loop (``DeviceDataset.collate`` + a ``no_grad`` forward, the metric in
  float64 on the host), including eval-mode modules, training steps in between, the graph8c known answers and two ranks."""
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_kernels import assert_close, dev  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _graph(N, E, K, seed):
    g = torch.Generator().manual_seed(seed)
    ei = torch.randint(0, N, (2, E), generator=g)
    return ei.to(dev()), torch.randn(E, K, generator=g).to(dev())


def _modes(layer, fn):
    """Outputs of fn() in grad mode, under no_grad, under inference_mode and with every parameter frozen."""
    outs = {"grad": fn()}
    with torch.no_grad():
        outs["no_grad"] = fn()
    with torch.inference_mode():
        outs["inference_mode"] = fn()
    flags = [p.requires_grad for p in layer.parameters()]
    for p in layer.parameters():
        p.requires_grad_(False)
    try:
        outs["frozen"] = fn()
    finally:
        for p, f in zip(layer.parameters(), flags):
            p.requires_grad_(f)
    assert outs["grad"].requires_grad
    return outs


def _all_equal(outs, name):
    ref = outs["grad"].detach()
    for k, v in outs.items():
        assert torch.equal(v.detach(), ref), "%s: %s forward differs from the grad-mode forward" % (name, k)


ML3_CASES = {
    # tensor-memory kernel (fp32: the whole-layer call; tf32 / bf16: the fused call), 30||2 and 32||16
    **{"ts_30_2_%s" % p: dict(args=(True, 8, 8, 25, 30, 2), precision=p) for p in ("fp32", "tf32", "bf16")},
    **{"ts_32_16_%s" % p: dict(args=(True, 8, 8, 32, 32, 16), precision=p) for p in ("fp32", "tf32", "bf16")},
    "round1_fi64": dict(args=(False, 8, 8, 64, 32, 0)),              # shared-memory-plane kernel, no gates
    "round1_gated_k5": dict(args=(False, 5, 5, 16, 32, 16)),         # shared-memory-plane kernel, gated epilogue (odd K)
    "two_kernel": dict(args=(True, 8, 8, 25, 30, 2), fused=False),
    "no_learnedge": dict(args=(False, 8, 8, 25, 32, 16)),
    "nout2_0": dict(args=(True, 8, 8, 25, 32, 0)),
}


@pytest.mark.parametrize("case", sorted(ML3_CASES))
@pytest.mark.parametrize("x_grad", [False, True])
def test_ml3layer_forward_only_equals_grad_mode(case, x_grad, monkeypatch):
    from gnn_matlang_b200.libs import spect_conv
    from gnn_matlang_b200.libs.spect_conv import ML3Layer
    c = ML3_CASES[case]
    if not c.get("fused", True):
        monkeypatch.setattr(spect_conv, "USE_FUSED", False)
    torch.manual_seed(1)
    layer = ML3Layer(*c["args"], precision=c.get("precision", "fp32")).to(dev())
    K, Fi = c["args"][1], c["args"][3]
    ei, ea = _graph(3000, 24000, K, 2)
    x = torch.randn(3000, Fi, device=dev()).requires_grad_(x_grad)     # x_grad False: a model's first layer
    spect_conv.ops.fused_path_counts(reset=True)
    _all_equal(_modes(layer, lambda: layer(x, ei, ea)), case)
    if case == "round1_gated_k5":
        assert spect_conv.ops.fused_path_counts()[1] > 0


@pytest.mark.parametrize("Fo", [64, 96])
@pytest.mark.parametrize("concat", [False, True])
def test_ml1layer_forward_only_equals_grad_mode(Fo, concat):
    from gnn_matlang_b200.libs.spect_conv import ML1_PATH_COUNTS, ML1Layer
    torch.manual_seed(3)
    layer = ML1Layer(40, Fo, concat).to(dev())
    ei, _ = _graph(5000, 30000, 1, 4)
    x = torch.randn(5000, 40, device=dev())
    before = dict(ML1_PATH_COUNTS)
    _all_equal(_modes(layer, lambda: layer(x, ei)), "ML1Layer Fo=%d concat=%s" % (Fo, concat))
    assert ML1_PATH_COUNTS["fused" if Fo <= 64 else "composed"] > before["fused" if Fo <= 64 else "composed"]


def _zinc_batch(B, seed, adjacency=False):
    from gnn_matlang_b200.synthetic import GraphPool
    pool = GraphPool("zinc", 256, seed=seed)
    return pool, pool.collate(np.random.default_rng(seed).integers(0, 256, B), adjacency=adjacency).to(dev())


@pytest.mark.parametrize("family", ["GNNML3", "GNNML1"])
def test_whole_models_forward_only_equals_grad_mode(family):
    from gnn_matlang_b200.models import GNNML1, GNNML3
    pool, b = _zinc_batch(512, 5, adjacency=True)
    torch.manual_seed(0)
    model = (GNNML3("zinc", pool.K, pool.F) if family == "GNNML3" else GNNML1("zinc", pool.F)).to(dev())
    _all_equal(_modes(model, lambda: model(b.fresh())), family)


class _Recorder(object):
    def __init__(self, monkeypatch, ops):
        self.calls = []
        for name in ("ml3layer_forward", "fused_agg_proj", "ml1layer_forward"):
            fn = getattr(ops, name)
            monkeypatch.setattr(ops, name, self._wrap(name, fn))

    def _wrap(self, name, fn):
        def wrapped(*a, **k):
            self.calls.append((name, dict(k)))
            return fn(*a, **k)
        return wrapped

    def take(self):
        out, self.calls = self.calls, []
        return out


def test_forward_only_asks_for_no_aux_and_no_aggregate(monkeypatch):
    """Under no_grad and with every parameter frozen the library gets keep_aggregate=False and aux=False; in grad mode the calls
    are exactly those of a training forward (no aux argument; the aggregate kept for a first layer)."""
    from gnn_matlang_b200.libs import spect_conv
    from gnn_matlang_b200.libs.spect_conv import ML1Layer, ML3Layer
    rec = _Recorder(monkeypatch, spect_conv.ops)
    torch.manual_seed(0)
    layers = {"layer_api": ML3Layer(True, 8, 8, 25, 30, 2).to(dev()), "fused": ML3Layer(True, 8, 8, 25, 30, 2, precision="tf32").to(dev()),
              "ml1": ML1Layer(25, 64).to(dev())}
    ei, ea = _graph(2000, 16000, 8, 1)
    x = torch.randn(2000, 25, device=dev())
    run = {"layer_api": lambda l: l(x, ei, ea), "fused": lambda l: l(x, ei, ea), "ml1": lambda l: l(x, ei)}
    op = {"layer_api": "ml3layer_forward", "fused": "fused_agg_proj", "ml1": "ml1layer_forward"}
    for name, layer in layers.items():
        run[name](layer)                                        # grad mode, x without gradient: a first layer
        calls = [k for n, k in rec.take() if n == op[name]]
        assert len(calls) == 1 and "aux" not in calls[0], (name, calls)
        if name == "layer_api":
            assert calls[0]["keep_aggregate"] is True
        with torch.no_grad():
            run[name](layer)
        for p in layer.parameters():
            p.requires_grad_(False)
        run[name](layer)
        calls = [k for n, k in rec.take() if n == op[name]]
        assert len(calls) == 2, (name, calls)
        for k in calls:
            assert k.get("aux") is False and not k.get("keep_aggregate", False), (name, k)


def test_c_abi_without_aux_returns_the_same_y():
    from gnn_matlang_b200 import ops
    from gnn_matlang_b200.graph import get_plan, sorted_edge_attr
    torch.manual_seed(0)
    N, E, K = 4000, 30000, 8
    ei, ea = _graph(N, E, K, 7)
    plan = get_plan(ei, N)
    ea_s = sorted_edge_attr(ea, plan)
    r = lambda *s: torch.randn(*s, device=dev()) * 0.2
    x = ops.aligned_rows(r(N, 25))
    ws4 = (r(16, 8), r(16, 8), r(16, 8), r(8, 32))
    gates = (r(2, 25), r(2), r(2, 25), r(2))
    wc, bc = r(K, 25, 30), r(30)
    a = ops.ml3layer_forward(plan, x, ea_s, ws4, wc, bc, gates)
    b = ops.ml3layer_forward(plan, x, ea_s, ws4, wc, bc, gates, aux=False)
    assert a[1] is not None and b[1] is None and torch.equal(a[0], b[0])
    # the fused call with a gated epilogue on both kernel generations (K = 8: tensor memory; K = 5: shared-memory planes)
    for k in (8, 5):
        eak = ea_s[:, :k].contiguous()
        wg, bg = r(25, 32), r(32)
        args = (plan.rowptr, plan.col, None, eak, x, r(k * 25, 32))
        kw = dict(bias=r(32), S=x, self_mode=1, Bself=wg, bias_s=bg, G=16, epilogue=1, win=plan.win)
        ya, aux = ops.fused_agg_proj(*args, **kw)
        yb, none = ops.fused_agg_proj(*args, aux=False, **kw)
        assert aux is not None and none is None and torch.equal(ya, yb), k
    for concat in (False, True):
        w = [r(1, 25, 64), r(64), r(64, 25), r(64), r(64, 25), r(64), r(64, 25), r(64)]
        ya, aux, _ = ops.ml1layer_forward(plan, x, *w, concat=concat)
        yb, none, _ = ops.ml1layer_forward(plan, x, *w, concat=concat, aux=False)
        assert aux is not None and none is None and torch.equal(ya, yb), concat


# ------------------------------------------------------------------------------------------------------ the evaluator
def _host_terms(metric, o, y):
    o, y = o.detach().cpu().double().numpy(), y.detach().cpu().double().numpy().reshape(o.shape)
    if metric == "l1":
        return np.abs(o - y).sum(1), None
    if metric == "mse":
        return ((o - y) ** 2).sum(1), None
    p = 1.0 / (1.0 + np.exp(-o))
    t = -(y * np.maximum(np.log(p), -100) + (1 - y) * np.maximum(np.log(1 - p), -100)).sum(1)
    return t, (((o[:, 0] > 0) == (y[:, 0] > 0.5)).sum() if o.shape[1] == 1 else None)


def _eager(model, dds, ids, B, metric):
    """The reference's test() loop: device collation of consecutive chunks, a no_grad forward, the metric in float64 on the host."""
    was = model.training
    model.eval()
    outs, s, correct = [], 0.0, 0
    with torch.no_grad():
        for i in range(0, len(ids), B):
            b = dds.collate(np.asarray(ids[i:i + B], np.int64))
            o = model(b)
            o = o.unsqueeze(1) if o.dim() == 1 else o
            outs.append(o)
            if metric is not None:
                t, c = _host_terms(metric, o, b.y)
                s += float(t.sum())
                correct += int(c) if c is not None else 0
    model.train(was)
    return torch.cat(outs), s, correct


def _check(model, dds, ids, B, metric, name):
    from gnn_matlang_b200.train import GraphedEvaluator
    ev = GraphedEvaluator(model, dds, ids, B, metric=metric)
    res = ev.run(outputs=True)
    ref_out, ref_sum, ref_correct = _eager(model, dds, ids, min(B, len(ids)), metric)
    diff = float((res["outputs"] - ref_out).abs().max())
    print("%s: %d graphs, sum %.9g (eager %.9g), largest output difference %.3e" % (name, res["graphs"], res.get("sum", 0.0), ref_sum, diff))
    assert res["graphs"] == len(ids) and res["outputs"].shape == ref_out.shape
    assert_close(res["outputs"], ref_out, name=name + " outputs")
    if metric is not None:
        assert abs(res["sum"] - ref_sum) <= 1e-6 * abs(ref_sum), (res["sum"], ref_sum)
        assert abs(res["mean"] - res["sum"] / len(ids)) <= 1e-12 * abs(res["mean"])
    if metric == "bce":
        assert res["correct"] == ref_correct and res["accuracy"] == ref_correct / len(ids)
    return ev, res


def _pool_dataset(kind, count, seed, adjacency=False, supports=True):
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    pool = GraphPool(kind, count, seed=seed)
    return pool, DeviceDataset(pool, dev(), adjacency=adjacency, supports=supports)


@pytest.mark.parametrize("preset,metric,n_ids,B", [("zinc", "l1", 1000, 128), ("zinc", "l1", 300, 64), ("counting", "mse", 250, 100)])
def test_evaluator_equals_eager_loop_gnnml3(preset, metric, n_ids, B):
    from gnn_matlang_b200.models import GNNML3
    pool, dds = _pool_dataset(preset, 1200, 11)
    ids = np.random.default_rng(2).permutation(1200)[:n_ids]
    torch.manual_seed(0)
    model = GNNML3(preset, pool.K, pool.F).to(dev())
    _check(model, dds, ids, B, metric, "GNNML3 %s" % preset)


def test_evaluator_equals_eager_loop_gnnml1_and_outputs_only():
    from gnn_matlang_b200.models import GNNML1
    pool, dds = _pool_dataset("zinc", 600, 12, adjacency=True, supports=False)
    ids = np.random.default_rng(3).permutation(600)[:450]
    torch.manual_seed(0)
    model = GNNML1("zinc", pool.F).to(dev())
    _check(model, dds, ids, 100, "l1", "GNNML1 zinc")
    ev, res = _check(model, dds, ids, 100, None, "GNNML1 zinc outputs")
    assert set(res) == {"graphs", "outputs"}


def _exp_dataset():
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset, ExpPool
    ep = ExpPool()
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    design = sd.design_batch(torch.from_numpy(ep.ei1).to(dev()), torch.from_numpy(ep.edge_off1).to(dev()), torch.from_numpy(ep.node_off),
                             device=dev())
    x = torch.cat([torch.from_numpy(ep.x).to(dev()), design["degree"].unsqueeze(-1)], 1)
    return DeviceDataset.from_design(design, ep.node_off, x, ep.y)


def test_evaluator_equals_eager_loop_exp_bce():
    from gnn_matlang_b200.models import GNNML3
    dds = _exp_dataset()
    torch.manual_seed(0)
    model = GNNML3("exp", 6, 2).to(dev())
    ids = np.arange(200)[::-1].copy()
    ev, res = _check(model, dds, ids, 64, "bce", "GNNML3 exp")
    print("EXP: accuracy %.3f over %d graphs" % (res["accuracy"], res["graphs"]))


@pytest.mark.parametrize("preset", ["mutag", "enzymes"])
def test_evaluator_uses_eval_mode_and_restores_the_training_flag(preset):
    from gnn_matlang_b200.models import GNNML3
    pool, dds = _pool_dataset("zinc", 500, 13)
    torch.manual_seed(0)
    model = GNNML3(preset, pool.K, pool.F).to(dev())
    with torch.no_grad():                                      # non-trivial BatchNorm running statistics
        for i in range(3):
            model(dds.collate(np.arange(100 * i, 100 * i + 100)))
    for training in (True, False):
        model.train(training)
        ids = np.arange(37, 437)
        _check(model, dds, ids, 96, "l1" if preset == "mutag" else None, "GNNML3 %s" % preset)
        assert model.training is training


def test_evaluator_sees_training_steps_in_between():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.train import GraphedEvaluator, GraphedTrainer, pad_batch, padded_shapes
    pool, dds = _pool_dataset("zinc", 800, 14)
    rng = np.random.default_rng(4)
    train_ids = [rng.integers(0, 600, 128) for _ in range(4)]
    host = [pool.collate(i) for i in train_ids]
    Np, Ep = padded_shapes(host)
    torch.manual_seed(0)
    model = GNNML3("zinc", pool.K, pool.F).to(dev())
    gt = GraphedTrainer(model, pad_batch(host[0], Np, Ep), loss="l1", lr=1e-3, warmup=1)
    val = np.arange(600, 800)
    ev = GraphedEvaluator(model, dds, val, 64, metric="l1")
    prev = None
    for rnd in range(2):
        for i in train_ids:
            gt.load_from_dataset(dds, i)
            gt.step()
        res = ev.run(outputs=True)
        ref_out, ref_sum, _ = _eager(model, dds, val, 64, "l1")
        print("after round %d: evaluator %.9g, eager %.9g" % (rnd, res["sum"], ref_sum))
        assert abs(res["sum"] - ref_sum) <= 1e-6 * abs(ref_sum)
        assert_close(res["outputs"], ref_out, name="outputs after training")
        if prev is not None:
            assert res["sum"] != prev
        prev = res["sum"]


def _graph8c_pairs_bench(emb):
    """bench.py's count: pairs whose embeddings are within 1e-3 in L1."""
    G = emb.size(0)
    similar = 0
    for r in range(0, G, 2048):
        similar += int((torch.cdist(emb[r:r + 2048], emb, p=1) <= 0.001).sum())
    return (similar - G) // 2


def _graph8c_pairs_strict(emb, thr=1e-3):
    n = emb.size(0)
    count = 0
    for i0 in range(0, n, 2048):
        d = torch.cdist(emb[i0:i0 + 2048], emb, p=1)
        rows = torch.arange(i0, min(i0 + 2048, n), device=emb.device)
        count += int(((d < thr) & (torch.arange(n, device=emb.device)[None, :] > rows[:, None])).sum())
    return count


def test_graph8c_known_answers_through_the_evaluator():
    """graph8c at 100 graphs per batch (111 full chunks and one of 17): GNNML3 seed 0 on the GPU design leaves 1 pair
    undistinguished (bench.py's known answer), GNNML1 the oracle's 14,579."""
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.models import GNNML1, GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset
    from gnn_matlang_b200.train import GraphedEvaluator
    recs = read_graph6(os.path.join(GOLDEN, "graph8c.g6"))
    G = len(recs)
    ns = np.array([r["x"].shape[0] for r in recs], np.int64)
    es = np.array([r["edge_index"].shape[1] for r in recs], np.int64)
    node_ptr, edge_ptr = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(es)])
    ei = torch.from_numpy(np.concatenate([r["edge_index"] for r in recs], 1)).to(dev())
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    design = sd.design_batch(ei, torch.from_numpy(edge_ptr).to(dev()), torch.from_numpy(node_ptr), device=dev())
    x = torch.cat([torch.ones(int(node_ptr[-1]), 1, device=dev()), design["degree"].unsqueeze(-1)], 1)
    dds = DeviceDataset.from_design(design, node_ptr, x)
    torch.manual_seed(0)
    m3 = GNNML3("graph8c", ne=6, ninp=2).to(dev()).eval()
    ev = GraphedEvaluator(m3, dds, np.arange(G), 100, metric=None)
    assert ev.chunks.shape == (112, 100) and float(ev._w_all[:-1].sum()) == 11100 and float(ev._w_all[-1].sum()) == 17
    emb3 = ev.run(outputs=True)["outputs"]
    pairs3 = _graph8c_pairs_bench(emb3)
    torch.manual_seed(0)
    m1 = GNNML1("graph8c", ninp=1).to(dev()).eval()
    dds1 = DeviceDataset.from_graphs(recs, dev())
    emb1 = GraphedEvaluator(m1, dds1, np.arange(G), 100, metric=None).run(outputs=True)["outputs"].double()
    pairs1 = _graph8c_pairs_strict(emb1)
    print("graph8c through the evaluator: GNNML3 %d undistinguished pair(s), GNNML1 %d" % (pairs3, pairs1))
    assert emb3.shape == (G, 10) and pairs3 == 1
    assert emb1.shape[0] == G and pairs1 == 14579


# ------------------------------------------------------------------------------------------------------ two ranks
def _worker(rank, world, port, out_path):
    import torch.distributed as dist
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedEvaluator, shard_graphs
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    pool = GraphPool("zinc", 700, seed=15)
    dds = DeviceDataset(pool, d)
    ids = np.arange(50, 650)
    lo, hi = shard_graphs(pool.n[ids], world, rank)
    torch.manual_seed(0)
    model = GNNML3("zinc", pool.K, pool.F).to(d)
    res = GraphedEvaluator(model, dds, ids[lo:hi], 64, metric="l1", distributed=True).run()
    if rank == 0:
        torch.save(res, out_path)
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_sum_to_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedEvaluator
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "eval.pt")
        port = 29500 + (os.getpid() + 7) % 2000
        mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
        two = torch.load(out)
    pool = GraphPool("zinc", 700, seed=15)
    torch.manual_seed(0)
    model = GNNML3("zinc", pool.K, pool.F).to(dev())
    one = GraphedEvaluator(model, DeviceDataset(pool, dev()), np.arange(50, 650), 64, metric="l1").run()
    print("two ranks %.9g over %d graphs, one rank %.9g over %d" % (two["sum"], two["graphs"], one["sum"], one["graphs"]))
    assert two["graphs"] == one["graphs"] == 600
    assert abs(two["sum"] - one["sum"]) <= 1e-6 * abs(one["sum"])
