"""GNNML1 through the device data path: collation of the plain edge list on the GPU (wire format, HBM-resident pool, resident
reader records) bit-exact against host collation + pad_batch, and the captured GNNML1 training step against the eager one."""
import ctypes
import os
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev():
    return torch.device("cuda:0")


def _strip(hb):
    """The same batch without the support list (what GNNML1 records carry)."""
    return hb.__class__(**{k: v for k, v in hb.__dict__.items() if k not in ("edge_index2", "edge_attr2")})


def _static(ref, d):
    """Sentinel-filled device buffers with ref's shapes: the kernel must write every element."""
    out = ref.__class__(num_graphs=ref.num_graphs)
    for k, v in ref.__dict__.items():
        if isinstance(v, torch.Tensor):
            fill = 0 if k == "y" else 7 if v.is_floating_point() else -1
            out.__dict__[k] = torch.full(tuple(v.shape), fill, dtype=v.dtype, device=d)      # contiguous, as the library requires
    return out


def _same(out, ref):
    for k, v in ref.__dict__.items():
        if isinstance(v, torch.Tensor) and k != "real_graphs":
            w = getattr(out, k)
            assert w.dtype == v.dtype and torch.equal(w.cpu(), v), k


@pytest.mark.parametrize("supports", [True, False], ids=["both_lists", "plain_only"])
@pytest.mark.parametrize("padded", [True, False], ids=["padded", "exact"])
@pytest.mark.parametrize("kind,widths", [("zinc", (21, 4)), ("counting", None)])
def test_device_collation_of_the_plain_list_is_bit_exact(kind, widths, supports, padded):
    from gnn_matlang_b200.batch import CompactBatch
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import pad_batch
    pool = GraphPool(kind, 64, seed=9)
    idx = np.random.default_rng(5).integers(0, 64, 1500)          # more than 1024 graphs: two chunks of the offset scan
    hb = pool.collate(idx, adjacency=True)
    if not supports:
        hb = _strip(hb)
    N, M = hb.x.size(0), hb.edge_index.size(1)
    E = hb.edge_index2.size(1) if supports else None
    ref = pad_batch(hb, N + 37, E + 211 if supports else None, M + 101) if padded else hb
    d = dev()
    cb = CompactBatch.from_batch(hb, widths).pin_memory().to(d)
    dds = DeviceDataset(pool, d, adjacency=True, supports=supports)
    ids = torch.from_numpy(idx).pin_memory()
    _same(cb.expand_into(_static(ref, d)), ref)
    _same(dds.collate_into(ids, _static(ref, d)), ref)
    if not padded:
        _same(cb.expand(), ref)
        _same(dds.collate(ids), ref)


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int16, torch.int32, torch.int64])
def test_every_local_id_dtype_and_graphs_without_edges(dtype):
    from gnn_matlang_b200.batch import CompactBatch, collate
    from gnn_matlang_b200.train import pad_batch
    rng = np.random.default_rng(7)
    gs = []
    for i in range(1100):
        n = int(rng.integers(1, 30))
        m = 0 if i % 7 == 0 else int(rng.integers(0, 60))           # every seventh graph (and some others) has no edges
        e2 = int(rng.integers(1, 20))
        gs.append(dict(x=rng.standard_normal((n, 5)).astype(np.float32), edge_index=rng.integers(0, n, (2, m)),
                       edge_index2=rng.integers(0, n, (2, e2)), edge_attr2=rng.standard_normal((e2, 3)).astype(np.float32),
                       y=np.float32(i)))
    hb = collate(gs, adjacency=True)
    cb = CompactBatch.from_batch(hb)
    cb.al, cb.el = cb.al.to(dtype), cb.el.to(dtype)
    d = dev()
    _same(cb.pin_memory().to(d).expand(), hb)
    N, E, M = hb.x.size(0), hb.edge_index2.size(1), hb.edge_index.size(1)
    ref = pad_batch(hb, N + 3, E + 10, M + 29)
    _same(cb.to(d).expand_into(_static(ref, d)), ref)
    bare = _strip(hb)
    cbb = CompactBatch.from_batch(bare)
    cbb.al = cbb.al.to(dtype)
    _same(cbb.to(d).expand(), bare)


def test_resident_reader_records_graph8c():
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.synthetic import DeviceDataset
    from gnn_matlang_b200.train import pad_batch
    recs = read_graph6(os.path.join(ROOT, "tests", "golden", "graph8c.g6"))
    d = dev()
    dds = DeviceDataset.from_graphs(recs, d)
    idx = np.random.default_rng(3).integers(0, len(recs), 3000)
    hb = collate([recs[i] for i in idx], adjacency=True)
    _same(dds.collate(idx), hb)
    ref = pad_batch(hb, hb.x.size(0) + 5, None, hb.edge_index.size(1) + 50)
    _same(dds.collate_into(idx, _static(ref, d)), ref)


def test_error_paths():
    from gnn_matlang_b200 import _lib, ops
    from gnn_matlang_b200.batch import CompactBatch
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import pad_batch
    pool = GraphPool("zinc", 16, seed=1)
    idx = np.arange(16)
    hb = _strip(pool.collate(idx, adjacency=True))
    d = dev()
    N, M = hb.x.size(0), hb.edge_index.size(1)
    cb = CompactBatch.from_batch(hb, (21, 4)).to(d)
    dds = DeviceDataset(pool, d, adjacency=True, supports=False)
    # padding the plain list needs a dummy node
    no_dummy = _static(hb, d)
    no_dummy.edge_index = torch.full((2, M + 4), -1, dtype=torch.int64, device=d)
    with pytest.raises(ValueError):
        cb.expand_into(no_dummy)
    with pytest.raises(ValueError):
        dds.collate_into(idx, no_dummy)
    # mismatched shapes
    ok = pad_batch(hb, N + 4, None, M + 8)
    bad = _static(ok, d)
    bad.edge_index = torch.full((3, M + 8), -1, dtype=torch.int64, device=d)
    with pytest.raises(RuntimeError):
        ops.collate_device(cb.n, None, None, None, cb.num_graphs, bad, xc=cb.xc, widths=cb.widths, m=cb.m, al=cb.al)
    bad = _static(ok, d)
    bad.batch = torch.full((N + 3,), -1, dtype=torch.int64, device=d)
    with pytest.raises(RuntimeError):
        ops.collate_device(cb.n, None, None, None, cb.num_graphs, bad, xc=cb.xc, widths=cb.widths, m=cb.m, al=cb.al)
    with pytest.raises(RuntimeError):                          # the plain list without its ids
        ops.collate_device(cb.n, None, None, None, cb.num_graphs, _static(ok, d), xc=cb.xc, widths=cb.widths, m=cb.m)
    short = _static(pad_batch(hb, N + 4, None, M), d)
    short.edge_index = torch.full((2, M - 1), -1, dtype=torch.int64, device=d)
    with pytest.raises(ValueError):                            # more edges than the output holds
        dds.collate_into(idx, short)
    # the C entry point: a plain-list output without m, and K = 0 with a support output, are refused
    lib = _lib.load()
    out = _static(ok, d)
    ws = torch.empty(lib.gnnml3_collate_graphs_workspace_bytes(16), dtype=torch.uint8, device=d)
    P = _lib.ptr
    wh = (ctypes.c_int32 * 2)(21, 4)
    args = lambda m, Mp, ei2: (None, P(cb.n), None, P(cb.xc), 2, wh, None, 25, None, None, None, 0, 0, None, 0, m,  # noqa: E731
                               None, P(cb.al), 1, cb.al.size(1), 16, N + 4, 0, Mp, P(out.x), ei2, None, P(out.edge_index),
                               P(out.batch), P(out.graph_ptr), P(ws), ws.numel(), _lib.stream_ptr())
    assert lib.gnnml3_collate_graphs(*args(None, M + 8, None)) != 0
    assert lib.gnnml3_collate_graphs(*args(P(cb.m), M + 8, P(out.edge_index))) != 0
    assert lib.gnnml3_collate_graphs(*args(P(cb.m), M + 8, None)) == 0
    torch.cuda.synchronize()
    _same(out, ok.__class__(**{k: v for k, v in ok.__dict__.items() if k != "y"}))      # (the labels are not the kernel's)


def _rewind(gt, ref_model, model):
    """The warm-up steps trained ``model`` and initialised Adam: rewind both IN PLACE (the captured graph holds these tensors'
    addresses)."""
    with torch.no_grad():
        for a, b in zip(model.parameters(), ref_model.parameters()):
            a.copy_(b)
        for st in gt.opt.state.values():
            for v in st.values():
                if isinstance(v, torch.Tensor):
                    v.zero_()


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_captured_gnnml1_step_equals_eager_step_on_every_route(concat):
    from gnn_matlang_b200.batch import CompactBatch
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch, padded_shapes
    pool = GraphPool("zinc", 64, seed=6)
    rng = np.random.default_rng(3)
    ids = [rng.integers(0, 64, 48) for _ in range(4)]
    host = [_strip(pool.collate(i, adjacency=True)) for i in ids]
    Np, Ep, Mp = padded_shapes(host, adjacency=True)
    assert Ep is None
    d = dev()
    torch.manual_seed(0)
    m1 = GNNML1("zinc", ninp=pool.F, concat=concat).to(d)
    torch.manual_seed(0)
    m2 = GNNML1("zinc", ninp=pool.F, concat=concat).to(d)
    eager = Trainer(m1, loss="l1", lr=1e-3)
    gt = GraphedTrainer(m2, pad_batch(host[0], Np, None, Mp), loss="l1", lr=1e-3, warmup=1)
    assert gt.fields == ("x", "edge_index", "batch", "graph_ptr", "y")
    _rewind(gt, m1, m2)
    dds = DeviceDataset(pool, d, adjacency=True, supports=False)
    for i, hb in enumerate(host):
        l1 = float(eager.step(hb.to(d)))
        if i == 0:
            l2 = float(gt.step(pad_batch(hb, Np, None, Mp).to(d)))
        else:
            if i == 1:
                gt.load_unpadded(hb.to(d))
            elif i == 2:
                gt.load_compact(CompactBatch.from_batch(hb, (21, 4)).pin_memory().to(d))
            else:
                gt.load_from_dataset(dds, ids[i])
            l2 = float(gt.step())
        assert abs(l1 - l2) <= 2e-5 * abs(l1), (i, l1, l2)
    for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.allclose(a, b, rtol=0, atol=2e-6), k


def test_gnnml3_graphed_trainer_keeps_its_captured_fields():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, pad_batch, padded_shapes
    pool = GraphPool("zinc", 16, seed=2)
    hb = pool.collate(np.arange(16))
    Np, Ep = padded_shapes([hb])
    gt = GraphedTrainer(GNNML3("zinc", pool.K, pool.F).to(dev()), pad_batch(hb, Np, Ep), loss="l1", warmup=1)
    assert gt.fields == ("x", "edge_index2", "edge_attr2", "batch", "graph_ptr", "y")


def test_gnnml1_exp_step_from_resident_reader_records():
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import DeviceDataset, ExpPool
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch, padded_shapes
    ep = ExpPool()
    recs = [dict(x=ep.x[ep.node_off[i]:ep.node_off[i + 1]], edge_index=ep.ei1[:, ep.edge_off1[i]:ep.edge_off1[i + 1]], y=ep.y[i])
            for i in range(len(ep.n))]
    d = dev()
    dds = DeviceDataset.from_graphs(recs, d)
    rng = np.random.default_rng(1)
    ids = [rng.integers(0, len(recs), 50) for _ in range(3)]
    host = [collate([recs[i] for i in ix], adjacency=True) for ix in ids]
    Np, _, Mp = padded_shapes(host, adjacency=True)
    torch.manual_seed(0)
    m1 = GNNML1("exp", ninp=1).to(d)
    torch.manual_seed(0)
    m2 = GNNML1("exp", ninp=1).to(d)
    eager = Trainer(m1, loss="bce", lr=1e-3)
    gt = GraphedTrainer(m2, pad_batch(host[0], Np, None, Mp), loss="bce", lr=1e-3, warmup=1)
    _rewind(gt, m1, m2)
    for ix, hb in zip(ids, host):
        _same(dds.collate(ix), hb)
        l1 = float(eager.step(dds.collate(ix)))
        gt.load_from_dataset(dds, ix)
        l2 = float(gt.step())
        assert np.isfinite(l1) and abs(l1 - l2) <= 2e-5 * abs(l1), (l1, l2)
    for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        assert torch.allclose(a, b, rtol=0, atol=2e-6), k


B_DP, STEPS_DP = 64, 2


def _dp_batches(pool):
    rng = np.random.default_rng(5)
    return [rng.integers(0, len(pool.n), B_DP) for _ in range(STEPS_DP)]


def _dp_worker(rank, world, port, out_path):
    import torch.distributed as dist
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import GraphedTrainer, pad_batch, padded_shapes
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    d = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    pool = GraphPool("zinc", 96, seed=9)
    per = B_DP // world
    host = [_strip(pool.collate(idx[rank * per:(rank + 1) * per], adjacency=True)) for idx in _dp_batches(pool)]
    Np, _, Mp = padded_shapes(host, adjacency=True)
    torch.manual_seed(0)
    model = GNNML1("zinc", ninp=pool.F).to(d)
    torch.manual_seed(0)
    init = GNNML1("zinc", ninp=pool.F).to(d)
    gt = GraphedTrainer(model, pad_batch(host[0], Np, None, Mp), loss="l1", lr=1e-3, distributed=True, warmup=1)
    _rewind(gt, init, model)
    grads = None
    for hb in host:
        gt.load_unpadded(hb.to(d))
        gt.step()
        if grads is None:                  # all-reduced gradient of the first step (a view of the reduced bucket)
            grads = {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters()}
    torch.cuda.synchronize()
    if rank == 0:
        torch.save(({k: v.detach().cpu() for k, v in model.state_dict().items()}, grads), out_path)
    dist.barrier()
    dist.destroy_process_group()


def test_gnnml1_two_ranks_on_half_batches_equal_one_rank_on_full_batches():
    """The bars of tests/test_gpu_dp.py: first-step gradients to 1e-5 of their scale, parameters to 10 % of the update."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.synthetic import GraphPool
    from gnn_matlang_b200.train import Trainer
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "dp.pt")
        port = 29500 + (os.getpid() + 1000) % 2000
        mp.spawn(_dp_worker, args=(2, port, out), nprocs=2, join=True)
        dp, dp_grads = torch.load(out)
    d = torch.device("cuda", 0)
    pool = GraphPool("zinc", 96, seed=9)
    torch.manual_seed(0)
    model = GNNML1("zinc", ninp=pool.F).to(d)
    init = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    tr = Trainer(model, loss="l1", lr=1e-3)
    for s, idx in enumerate(_dp_batches(pool)):
        tr.step(_strip(pool.collate(idx, adjacency=True)).to(d))
        if s == 0:
            for k, p in model.named_parameters():
                a, b = dp_grads[k].double(), p.grad.detach().cpu().double()
                err, scale = (a - b).abs().max().item(), b.abs().max().item()
                assert err <= 1e-5 * scale + 1e-12, "grad %s: 2-rank vs 1-rank differ by %.3e (max|grad| %.3e)" % (k, err, scale)
    for k, v in model.state_dict().items():
        a, b = dp[k].double(), v.detach().cpu().double()
        moved = (b - init[k].double()).abs().max().item()
        assert moved > 0, "parameter %s did not train" % k
        err = (a - b).abs().max().item()
        assert err <= 0.1 * moved, "%s: 2-rank vs 1-rank differ by %.3e (update size %.3e)" % (k, err, moved)
