"""Host side of the isomorphism test: every argument of ``PairTracker`` and ``isomorphism_test`` is rejected before any device
is touched (these tests run without a GPU), and the pair kernels are declared, bound and exported."""
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n", [-1, 2.5, True, "10", None])
def test_tracker_rejects_bad_n(n):
    from gnn_matlang_b200.isomorphism import PairTracker
    with pytest.raises(ValueError, match="n must be"):
        PairTracker(n, "cuda:0")


@pytest.mark.parametrize("thr", [-1e-3, float("nan"), float("inf"), "0.001", None, True])
def test_tracker_rejects_bad_threshold(thr):
    from gnn_matlang_b200.isomorphism import PairTracker
    with pytest.raises(ValueError, match="threshold"):
        PairTracker(10, "cuda:0", threshold=thr)


def test_tracker_rejects_a_cpu_device():
    from gnn_matlang_b200.isomorphism import PairTracker
    with pytest.raises(ValueError, match="CUDA device"):
        PairTracker(10, "cpu")


@pytest.mark.parametrize("pairs,match", [
    (np.array([[0, 10]]), "outside"),
    (np.array([[-1, 3]]), "outside"),
    (np.zeros((0, 2), np.int64), "shape"),
    (np.zeros((4, 3), np.int64), "shape"),
    (np.zeros(4, np.int64), "shape"),
    (np.array([[0.0, 1.0]]), "integer"),
    (torch.tensor([[0, 1], [2, 12]]), "outside"),
])
def test_tracker_rejects_bad_host_pairs(pairs, match):
    from gnn_matlang_b200.isomorphism import PairTracker
    with pytest.raises(ValueError, match=match):
        PairTracker(10, "cuda:0", pairs=pairs)


class _FakeDataset(object):
    """Enough of a DeviceDataset for the argument checks: host size arrays and a device-typed ``x``."""

    def __init__(self, G, device="cuda:0"):
        self.n_h = np.full(G, 8, np.int64)
        self.x = _Dev(device)


class _Dev(object):
    def __init__(self, device):
        self.device = torch.device(device)


def _make():
    raise AssertionError("no model may be built when an argument is rejected")


@pytest.mark.parametrize("kw,match", [
    (dict(seeds=[]), "seeds is empty"),
    (dict(seeds=range(0)), "seeds is empty"),
    (dict(batch_size=0), "batch_size"),
    (dict(batch_size=2.5), "batch_size"),
    (dict(threshold=-1.0), "threshold"),
    (dict(threshold=float("nan")), "threshold"),
    (dict(ids=[]), "ids is empty"),
    (dict(ids=[0, 20]), "ids must be"),
    (dict(ids=[-1]), "ids must be"),
    (dict(ids=[0.5, 1.5]), "ids must be"),
])
def test_isomorphism_test_rejects_bad_arguments(kw, match):
    from gnn_matlang_b200.isomorphism import isomorphism_test
    with pytest.raises(ValueError, match=match):
        isomorphism_test(_make, _FakeDataset(20), **kw)


def test_isomorphism_test_rejects_a_cpu_dataset_and_a_non_callable():
    from gnn_matlang_b200.isomorphism import isomorphism_test
    with pytest.raises(ValueError, match="CUDA device"):
        isomorphism_test(_make, _FakeDataset(20, "cpu"))
    with pytest.raises(TypeError, match="callable"):
        isomorphism_test(None, _FakeDataset(20))


def test_isomorphism_test_rejects_pairs_outside_the_ids():
    """Listed pairs index positions in ``ids``: with 5 ids, 5 is out of range although the dataset has 20 graphs."""
    from gnn_matlang_b200.isomorphism import isomorphism_test
    with pytest.raises(ValueError, match="outside"):
        isomorphism_test(_make, _FakeDataset(20), ids=np.arange(5), pairs=np.array([[0, 5]]))


def test_update_rejects_cpu_and_misshaped_embeddings():
    """``update`` checks the embeddings before the library is called: a tracker whose fields are set by hand (no bitmap, no
    device) must refuse misshaped, float64 and CPU inputs."""
    from gnn_matlang_b200.isomorphism import PairTracker
    tr = PairTracker.__new__(PairTracker)
    tr.n, tr.device, tr.threshold, tr.pairs, tr.P, tr.wpr = 10, torch.device("cuda", 0), 1e-3, None, 0, 4
    with pytest.raises(ValueError, match="d >= 1"):
        tr.update(torch.zeros(10, 0))
    with pytest.raises(ValueError, match="shape"):
        tr.update(torch.zeros(9, 3))
    with pytest.raises(ValueError, match="float32"):
        tr.update(torch.zeros(10, 3, dtype=torch.float64))
    with pytest.raises(ValueError, match="no CPU path"):
        tr.update(torch.zeros(10, 3))
    with pytest.raises(TypeError):
        tr.update(np.zeros((10, 3), np.float32))


def test_pair_symbols_are_declared_and_bound():
    from gnn_matlang_b200 import _lib
    with open(os.path.join(ROOT, "include", "gnnml3_b200.h")) as f:
        header = f.read()
    for name, nargs in (("gnnml3_pairs_mark", 10), ("gnnml3_pairs_count", 6)):
        assert "GNNML3_API int %s(" % name in header
        assert name in _lib.SIGNATURES and len(_lib.SIGNATURES[name][1]) == nargs
    lib = _lib.load()
    assert hasattr(lib, "gnnml3_pairs_mark") and hasattr(lib, "gnnml3_pairs_count")
