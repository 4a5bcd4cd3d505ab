"""The TU-dataset GNNML3 variants end to end on the GPU: the padding-neutral node BatchNorm kernels against float64
``nn.BatchNorm1d``, the captured training step of the ``mutag`` / ``enzymes`` presets against the eager step, the ``nll`` loss and
metric, and resident datasets built from reader records (``DeviceDataset.from_records``)."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def _sd():
    from gnn_matlang_b200.libs.utils import SpectralDesign
    return SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)


def _designed(records, sd):
    """The per-record path: ``sd(data)`` on every record, as the reference's dataset transform does."""
    out = []
    for r in records:
        d = sd(types.SimpleNamespace(x=torch.as_tensor(np.asarray(r["x"], np.float32)),
                                     edge_index=torch.as_tensor(np.asarray(r["edge_index"], np.int64)).reshape(2, -1)))
        out.append(dict(x=d.x, edge_index2=d.edge_index2, edge_attr2=d.edge_attr2, y=r["y"]))
    return out


# ------------------------------------------------------------------------------------------------ node BatchNorm kernels

def _bn_inputs(N, F, cnt, seed, pad_fill=None):
    g = torch.Generator(device="cpu").manual_seed(seed)
    big = torch.randn(N, F + 3, generator=g) * 2.0 + 0.5                      # strided rows: x is a column block of big
    gyb = torch.randn(N, F + 5, generator=g)
    if pad_fill is not None and cnt < N:
        big[cnt:, :F] = pad_fill
        big[cnt::2, :F] = float("inf")
        gyb[cnt:, :F] = float("nan")
    w, b = torch.randn(F, generator=g), torch.randn(F, generator=g)
    rm, rv = torch.randn(F, generator=g), torch.rand(F, generator=g) + 0.5
    return big.to(dev()), gyb.to(dev()), w.to(dev()), b.to(dev()), rm.to(dev()), rv.to(dev())


def _bn_run(big, gyb, w, b, rm, rv, F, cnt, momentum=0.1):
    from gnn_matlang_b200 import ops
    x, gy = big[:, :F], gyb[:, :F]
    rm, rv = rm.clone(), rv.clone()
    nbt = torch.zeros((), dtype=torch.int64, device=dev())
    c = torch.tensor([cnt], dtype=torch.int32, device=dev())
    y, mean, invstd = ops.bn_rows_fwd(x, c, w, b, rm, rv, nbt, 1e-5, momentum)
    dx, dw, db = ops.bn_rows_bwd(x, gy, c, w, mean, invstd)
    return dict(y=y, rm=rm, rv=rv, nbt=nbt, dx=dx, dw=dw, db=db)


def _close(a, ref, what, rel=1e-5, scale=None):
    a, ref = a.double().cpu(), ref.double().cpu()
    err = (a - ref).abs().max().item()
    scale = max(ref.abs().max().item(), scale or 0.0)
    assert err <= rel * scale + 1e-12, "%s: max |diff| %.3e, scale %.3e" % (what, err, scale)


@pytest.mark.parametrize("F_", [1, 24, 48, 128])
@pytest.mark.parametrize("N", [2, 127, 4097, 200000])
def test_bn_rows_matches_float64_batchnorm_on_the_real_rows(N, F_):
    cnts = sorted({2, (N + 1) // 2 + 1 if N > 4 else 2, N})
    for cnt in cnts:
        big, gyb, w, b, rm, rv = _bn_inputs(N, F_, cnt, seed=N + F_ + cnt, pad_fill=float("nan"))
        got = _bn_run(big, gyb, w, b, rm, rv, F_, cnt)
        # float64 reference on x[:cnt]: nn.BatchNorm1d's training-mode forward and its autograd
        xr = big[:cnt, :F_].double().clone().requires_grad_(True)
        wr, br = w.double().clone().requires_grad_(True), b.double().clone().requires_grad_(True)
        rmr, rvr = rm.double().clone(), rv.double().clone()
        yr = F.batch_norm(xr, rmr, rvr, wr, br, training=True, momentum=0.1, eps=1e-5)
        yr.backward(gyb[:cnt, :F_].double())
        tag = "N=%d F=%d cnt=%d" % (N, F_, cnt)
        _close(got["y"][:cnt], yr.detach(), tag + " y")
        _close(got["rm"], rmr, tag + " running_mean")
        _close(got["rv"], rvr, tag + " running_var")
        assert int(got["nbt"]) == 1
        # dx = w invstd (gy - ...) cancels to ~0 (exactly 0 for two rows): its scale is that of the terms, |w| invstd |gy|
        invstd = 1.0 / torch.sqrt(xr.detach().var(0, unbiased=False) + 1e-5)
        _close(got["dx"][:cnt], xr.grad, tag + " dx",
               scale=(wr.detach().abs() * invstd).max().item() * gyb[:cnt, :F_].abs().max().item())
        assert torch.equal(got["dx"][cnt:], torch.zeros_like(got["dx"][cnt:])), tag + " dx of padding rows"
        _close(got["dw"], wr.grad, tag + " dweight")
        _close(got["db"], br.grad, tag + " dbias")
        # the padding rows' NaN / inf reach nothing real: the same real rows with finite padding give the same bits
        big2, gyb2 = big.clone(), gyb.clone()
        big2[cnt:], gyb2[cnt:] = 0.25, -1.0
        fin = _bn_run(big2, gyb2, w, b, rm, rv, F_, cnt)
        for k in ("rm", "rv", "dw", "db"):
            assert torch.equal(fin[k], got[k]), tag + " " + k + " depends on the padding rows"
        for k in ("y", "dx"):
            assert torch.equal(fin[k][:cnt], got[k][:cnt]), tag + " " + k + " depends on the padding rows"
        # deterministic: a second run gives the same bits
        again = _bn_run(big, gyb, w, b, rm, rv, F_, cnt)
        for k in got:
            assert torch.equal(again[k].nan_to_num(7.0), got[k].nan_to_num(7.0)), tag + " rerun differs in " + k


def test_bn_rows_single_real_row():
    """nn.BatchNorm1d refuses one row; here the output is the bias, the running mean moves to the row, the running variance
    stays, and the only gradient is dbias = gy."""
    N, F_ = 9, 24
    big, gyb, w, b, rm, rv = _bn_inputs(N, F_, 1, seed=3, pad_fill=float("nan"))
    got = _bn_run(big, gyb, w, b, rm, rv, F_, 1)
    assert torch.equal(got["y"][0], b)
    _close(got["rm"], 0.9 * rm.double() + 0.1 * big[0, :F_].double(), "running_mean")
    assert torch.equal(got["rv"], rv)
    assert int(got["nbt"]) == 1
    assert torch.equal(got["dx"], torch.zeros_like(got["dx"]))
    assert torch.equal(got["dw"], torch.zeros_like(got["dw"]))
    assert torch.equal(got["db"], gyb[0, :F_])


def test_bn_rows_captured_replays_follow_the_device_count():
    from gnn_matlang_b200 import ops
    N, F_ = 4097, 48
    big, gyb, w, b, rm0, rv0 = _bn_inputs(N, F_, N, seed=5)
    x, gy = big[:, :F_], gyb[:, :F_]
    c = torch.tensor([N], dtype=torch.int32, device=dev())
    rm, rv, nbt = rm0.clone(), rv0.clone(), torch.zeros((), dtype=torch.int64, device=dev())

    def step():
        y, mean, invstd = ops.bn_rows_fwd(x, c, w, b, rm, rv, nbt, 1e-5, 0.1)
        return (y,) + ops.bn_rows_bwd(x, gy, c, w, mean, invstd)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = step()
    for cnt in (N, 2, 1000, 4001):
        c.fill_(cnt)
        rm.copy_(rm0)
        rv.copy_(rv0)
        g.replay()
        ref = _bn_run(big, gyb, w, b, rm0, rv0, F_, cnt)
        for k, v in zip(("y", "dx", "dw", "db"), outs):
            assert torch.equal(v, ref[k]), "cnt=%d: replay differs from the eager call in %s" % (cnt, k)
        assert torch.equal(rm, ref["rm"]) and torch.equal(rv, ref["rv"]), cnt


# ------------------------------------------------------------------------------------------------ model, trainer, evaluator

def _cfg(preset, **kw):
    from gnn_matlang_b200.models import MODEL_CONFIGS
    c = dict(MODEL_CONFIGS[preset])
    c.update(kw)
    return c


def _host_batches(kind, n_records, n_batches, B, seed):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.synthetic import tu_records
    recs = _designed(tu_records(kind, n_records, seed), _sd())
    rng = np.random.default_rng(seed)
    return [collate([recs[i] for i in rng.choice(n_records, B, replace=False)]) for _ in range(n_batches)]


def _rewind(gt, ref_model, model):
    """Undo the warm-up step IN PLACE (the captured graph holds these tensors' addresses): parameters and BatchNorm buffers from
    the reference model, Adam state zeroed."""
    with torch.no_grad():
        for a, b in zip(model.state_dict().values(), ref_model.state_dict().values()):
            a.copy_(b)
        for st in gt.opt.state.values():
            for v in st.values():
                if isinstance(v, torch.Tensor):
                    v.zero_()


@pytest.mark.parametrize("preset,cfg,loss", [("mutag", {}, "bce"), ("enzymes", dict(dropout=0.0), "nll")], ids=["mutag", "enzymes"])
def test_captured_bn_step_equals_eager_step(preset, cfg, loss):
    """The padded captured step trains the model the eager step trains on the unpadded graphs: BatchNorm statistics leave the
    dummy graph out (node BatchNorm of mutag, read-out BatchNorm of enzymes)."""
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, pad_batch, padded_shapes
    host = _host_batches(preset, 160, 3, 64, seed=11)
    Np, Ep = padded_shapes(host)
    d = dev()
    ninp = host[0].x.size(1)
    torch.manual_seed(0)
    m1 = GNNML3(_cfg(preset, **cfg), 6, ninp).to(d)
    torch.manual_seed(0)
    m2 = GNNML3(_cfg(preset, **cfg), 6, ninp).to(d)
    init = {k: v.detach().clone() for k, v in m1.state_dict().items()}
    eager = Trainer(m1, loss=loss, lr=1e-3)
    gt = GraphedTrainer(m2, pad_batch(host[0], Np, Ep), loss=loss, lr=1e-3, warmup=1)
    _rewind(gt, m1, m2)
    # A BatchNorm's dx sums to zero over its rows, so the gradient of a bias in front of one nearly cancels; Adam turns the FP32
    # noise left in such an element into a full lr-sized step of either sign.  The update-relative rule of the parameters holds
    # for the elements whose gradient stays above 1e-3 of its tensor's largest at every step; the first-step gradients of all
    # elements are held to the FP32 bar.
    resolved = {k: torch.ones_like(p, dtype=torch.bool) for k, p in m1.named_parameters()}
    for i, hb in enumerate(host):
        l1 = float(eager.step(hb.to(d)))
        l2 = float(gt.step(pad_batch(hb, Np, Ep).to(d)))
        assert abs(l1 - l2) <= 2e-5 * abs(l1), (i, l1, l2)
        for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
            if i == 0:
                _close(b.grad, a.grad, "first-step gradient " + k)
            resolved[k] &= a.grad.abs() > 1e-3 * a.grad.abs().max()
        if i == 0:
            # the running buffers of the first step come from the same parameters; later ones inherit the noise above
            s2 = m2.state_dict()
            for k, v in m1.state_dict().items():
                if "running" in k:
                    _close(s2[k], v, "first-step " + k)
    p2 = dict(m2.named_parameters())
    for k, a in m1.named_parameters():
        moved = (a.detach() - init[k]).abs().max().item()
        assert moved > 0, k
        diff = (a.detach() - p2[k].detach()).abs()
        assert diff.max().item() <= 3 * 1e-3 * 1.01, k                          # Adam moves no element more than lr per step
        err = diff[resolved[k]].max().item() if resolved[k].any() else 0.0
        assert err <= 0.1 * moved, "%s: captured vs eager differ by %.3e (update size %.3e)" % (k, err, moved)
    s2 = m2.state_dict()
    for k, v in m1.state_dict().items():
        if "num_batches_tracked" in k:
            assert int(s2[k]) == int(v) == len(host), k


def test_captured_dropout_differs_per_replay_and_evaluation_is_deterministic():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, tu_records
    from gnn_matlang_b200.train import GraphedEvaluator, GraphedTrainer, pad_batch, padded_shapes
    host = _host_batches("enzymes", 120, 1, 32, seed=4)
    Np, Ep = padded_shapes(host)
    d = dev()
    pb = pad_batch(host[0], Np, Ep).to(d)
    losses, models = {}, {}
    for p in (0.1, 0.0):
        torch.manual_seed(0)
        models[p] = GNNML3(_cfg("enzymes", dropout=p), 6, host[0].x.size(1)).to(d)
        gt = GraphedTrainer(models[p], pb, loss="nll", lr=0.0, warmup=1)        # lr 0: only dropout can change the loss
        losses[p] = [float(gt.step(pb)) for _ in range(2)]
    assert all(np.isfinite(losses[0.1])) and losses[0.1][0] != losses[0.1][1], losses
    assert losses[0.0][0] == losses[0.0][1], losses
    dds = DeviceDataset.from_records(tu_records("enzymes", 120, 4), _sd(), d)
    ev = GraphedEvaluator(models[0.1], dds, np.arange(100), 32, metric="nll")
    assert ev.run() == ev.run()


def test_nll_trainer_and_evaluator_against_eager():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, tu_records
    from gnn_matlang_b200.train import GraphedEvaluator, GraphedTrainer, eval_shapes, pad_batch
    d = dev()
    recs = tu_records("enzymes", 150, 8)
    dds = DeviceDataset.from_records(recs, _sd(), d)
    chunks = np.stack([np.random.default_rng(s).choice(150, 48, replace=False) for s in range(2)])
    Np, Ep, _ = eval_shapes(dds, chunks)
    torch.manual_seed(0)
    model = GNNML3(_cfg("enzymes", dropout=0.0), 6, dds.x.size(1)).to(d)
    gt = GraphedTrainer(model, pad_batch(dds.collate(chunks[0]).to("cpu"), Np, Ep).to(d), loss="nll", warmup=1)
    for c in chunks:
        b = dds.collate(c)
        ref = F.nll_loss(model(b), b.y.reshape(-1), reduction="sum").item()       # the parameters the step starts from
        gt.load_from_dataset(dds, c)
        got = float(gt.step())
        assert abs(got - ref) <= 1e-5 * abs(ref), (got, ref)
    ids = np.arange(3, 150, 2)                                                      # 74 graphs: a short last chunk of 10
    ev = GraphedEvaluator(model, dds, ids, 32, metric="nll")
    res = ev.run()
    model.eval()
    s, correct = 0.0, 0
    with torch.no_grad():
        for k in range(0, len(ids), 32):
            b = dds.collate(ids[k:k + 32])
            out = model(b)
            s += F.nll_loss(out, b.y.reshape(-1), reduction="sum").item()
            correct += int((out.argmax(1) == b.y.reshape(-1)).sum())
    assert res["graphs"] == len(ids)
    assert abs(res["sum"] - s) <= 1e-5 * abs(s), (res["sum"], s)
    assert res["correct"] == correct and res["accuracy"] == correct / len(ids)


# ------------------------------------------------------------------------------------------------ resident reader records

@pytest.mark.parametrize("adddegree", [True, False], ids=["degree", "no_degree"])
def test_from_records_equals_per_record_design_and_collate(adddegree):
    from gnn_matlang_b200.batch import collate
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset, _local_graph, tu_records
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=adddegree)
    lim = sd.max_kernel_nodes()
    rng = np.random.default_rng(0)
    recs = tu_records("enzymes", 40, 2)
    for n in (lim - 1, lim, lim + 1, 126, 1, 5):
        ei = _local_graph(rng, n, n, 6) if n != 5 else np.zeros((2, 0), np.int64)      # n = 5: an edgeless graph
        recs.insert(int(rng.integers(0, len(recs) + 1)), dict(x=np.eye(3, dtype=np.float32)[rng.integers(0, 3, n)], edge_index=ei,
                                                              y=np.array([int(rng.integers(0, 6))], np.int64)))
    d = dev()
    dds = DeviceDataset.from_records(recs, sd, d)
    ids = np.concatenate([np.arange(len(recs)), rng.integers(0, len(recs), 30)])
    got = dds.collate(ids)
    des = _designed(recs, sd)
    ref = collate([des[i] for i in ids])
    for k in ("x", "edge_index2", "y", "batch"):
        assert torch.equal(getattr(got, k).cpu(), getattr(ref, k)), k
    assert torch.equal(got.graph_ptr.cpu(), ref.graph_ptr)
    ea, ear = got.edge_attr2.cpu().double(), ref.edge_attr2.double()
    assert ((ea - ear).abs() <= 1e-5 * ear.abs().max(0).values).all()


def test_smoke_enzymes_training_loss_falls():
    """50 seeded captured steps on ENZYMES-shaped records from a resident dataset lower the training loss."""
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, tu_records
    from gnn_matlang_b200.train import GraphedTrainer, eval_shapes, pad_batch
    d = dev()
    dds = DeviceDataset.from_records(tu_records("enzymes", 600, 1), _sd(), d)
    rng = np.random.default_rng(1)
    chunks = np.stack([rng.choice(600, 128, replace=False) for _ in range(10)])
    Np, Ep, _ = eval_shapes(dds, chunks)
    torch.manual_seed(0)
    model = GNNML3("enzymes", 6, dds.x.size(1)).to(d)
    gt = GraphedTrainer(model, pad_batch(dds.collate(chunks[0]).to("cpu"), Np, Ep).to(d), loss="nll", warmup=1)
    losses = []
    for s in range(50):
        gt.load_from_dataset(dds, chunks[s % 10])
        losses.append(float(gt.step()))
    assert np.all(np.isfinite(losses))
    assert np.mean(losses[-10:]) < 0.9 * np.mean(losses[:10]), losses
