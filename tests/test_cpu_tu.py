"""CPU checks of the TU-dataset additions: the ``nll`` loss and metric against numpy, the argument checks of the new names, of
``DeviceDataset.from_records`` and of the node BatchNorm path, the new C ABI symbols, and the shape of the synthetic TU records."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _logp(B, C, seed):
    out = torch.log_softmax(torch.from_numpy(np.random.default_rng(seed).standard_normal((B, C))), 1)
    y = torch.from_numpy(np.random.default_rng(seed + 1).integers(0, C, (B, 1)).astype(np.int64))
    return out, y


def test_nll_loss_and_terms_against_numpy():
    from gnn_matlang_b200.train import eval_terms, loss_fn
    out, y = _logp(37, 6, 0)
    o, yy = out.numpy(), y.numpy()[:, 0]
    ref_terms = -o[np.arange(37), yy]
    np.testing.assert_allclose(loss_fn("nll", out, y).item(), ref_terms.sum(), rtol=1e-12)
    term, correct = eval_terms("nll", out, y)
    np.testing.assert_allclose(term.numpy(), ref_terms, rtol=1e-12)
    assert np.array_equal(correct.numpy(), (o.argmax(1) == yy).astype(np.float64))
    # labels as read_mat gives them (int64 [B, 1]) and flat int32 labels are the same labels
    assert loss_fn("nll", out, y.reshape(-1).int()).item() == loss_fn("nll", out, y).item()


def test_nll_rejects_labels_that_are_not_class_ids():
    from gnn_matlang_b200.train import eval_terms, loss_fn
    out, y = _logp(8, 6, 1)
    with pytest.raises(ValueError, match="class ids"):
        loss_fn("nll", out, y.double())
    with pytest.raises(ValueError, match="class ids"):
        loss_fn("nll", out, y[:7])
    with pytest.raises(ValueError, match="class ids"):
        eval_terms("nll", out, torch.zeros(8, 2, dtype=torch.int64))


def test_loss_and_metric_names():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.train import EVAL_METRICS, LOSSES, GraphedTrainer, Trainer
    assert "nll" in LOSSES and "nll" in EVAL_METRICS
    model = GNNML3("enzymes", 6, 4)
    with pytest.raises(ValueError, match="loss must be one of"):
        Trainer(model, loss="cross_entropy")
    with pytest.raises(ValueError, match="loss must be one of"):
        GraphedTrainer(model, None, loss="cross_entropy")
    Trainer(model, loss="nll")                                         # a known name builds (CPU Adam)


def test_from_records_argument_checks():
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    good = dict(x=np.ones((3, 2), np.float32), edge_index=np.array([[0, 1], [1, 0]]), y=np.array([1]))
    with pytest.raises(ValueError, match="no records"):
        DeviceDataset.from_records([], sd, "cpu")
    with pytest.raises(ValueError, match="outside its graph"):
        DeviceDataset.from_records([good, dict(good, edge_index=np.array([[0, 3], [3, 0]]))], sd, "cpu")
    with pytest.raises(ValueError, match="outside its graph"):
        DeviceDataset.from_records([dict(good, edge_index=np.array([[-1], [0]]))], sd, "cpu")
    with pytest.raises(ValueError, match="width"):
        DeviceDataset.from_records([good, dict(good, x=np.ones((3, 3), np.float32))], sd, "cpu")
    with pytest.raises(ValueError, match="label"):
        DeviceDataset.from_records([good, dict(good, y=None)], sd, "cpu")


def test_node_batchnorm_path_accepts_only_the_presets_configuration():
    from gnn_matlang_b200.norm import batch_norm_rows
    x, cnt = torch.zeros(4, 3), torch.tensor([2], dtype=torch.int32)
    for bn in (torch.nn.BatchNorm1d(3, affine=False), torch.nn.BatchNorm1d(3, track_running_stats=False),
               torch.nn.BatchNorm1d(3, momentum=None), torch.nn.LayerNorm(3)):
        with pytest.raises(ValueError):
            batch_norm_rows(x, cnt, bn)


def test_bn_rows_abi_symbols_in_header_and_binding():
    from gnn_matlang_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gnnml3_b200.h")).read()
    names = set(re.findall(r"GNNML3_API\s+[\w\s\*]+?\b(gnnml3_bn_rows_\w+)\s*\(", hdr))
    assert names == {"gnnml3_bn_rows_workspace_bytes", "gnnml3_bn_rows_fwd", "gnnml3_bn_rows_bwd"}
    for n in names:
        assert n in _lib.SIGNATURES
    assert len(_lib.SIGNATURES["gnnml3_bn_rows_fwd"][1]) == 19 and len(_lib.SIGNATURES["gnnml3_bn_rows_bwd"][1]) == 17


def test_tu_records_shapes():
    from gnn_matlang_b200.synthetic import tu_records
    enz = tu_records("enzymes", 200, 0)
    n = np.array([r["x"].shape[0] for r in enz])
    assert n.min() >= 2 and n.max() <= 126 and (n >= 120).sum() == 4
    assert all(r["x"].shape[1] == 3 and r["y"].dtype == np.int64 and r["y"].shape == (1,) for r in enz)
    assert set(int(r["y"][0]) for r in enz) == set(range(6))
    for r in enz:
        ei = r["edge_index"]
        assert ei.min() >= 0 and ei.max() < r["x"].shape[0]
    mut = tu_records("mutag", 50, 0)
    assert all(10 <= r["x"].shape[0] <= 28 and r["x"].shape[1] == 7 and r["y"].dtype == np.float32 for r in mut)
    with pytest.raises(ValueError):
        tu_records("proteins", 1)


def test_evaluator_nll_needs_a_log_softmax_head():
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.train import GraphedEvaluator

    class _Sizes(object):
        n_h, e_h, m_h = np.full(4, 5, np.int64), np.full(4, 20, np.int64), None

    with pytest.raises(ValueError, match="log_softmax"):
        GraphedEvaluator(GNNML3("mutag", 6, 8), _Sizes(), [0, 1], 2, metric="nll")
