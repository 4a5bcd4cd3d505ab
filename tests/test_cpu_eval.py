"""Host side of the captured evaluation pass (train.GraphedEvaluator): the padded-shape rule computed from size arrays, the
chunking and filling of a split, the metric terms against a numpy restatement, and the constructor's argument checks (which
run before anything touches a device)."""
import numpy as np
import pytest
import torch

from gnn_matlang_b200.synthetic import GraphPool
from gnn_matlang_b200.train import (GraphedEvaluator, eval_chunks, eval_shapes, eval_terms, padded_shapes,
                                    padded_shapes_from_sizes)


class _Sizes(object):
    """The host size arrays of a DeviceDataset (what the shape rule reads), built from a GraphPool without a device."""

    def __init__(self, pool, supports=True, adjacency=False):
        self.n_h = pool.n
        self.e_h = pool.e if supports else None
        self.m_h = pool.e1 if adjacency else None


@pytest.fixture(scope="module")
def pool():
    return GraphPool("zinc", 120, seed=3)


@pytest.mark.parametrize("supports,adjacency", [(True, False), (True, True), (False, True)])
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_shapes_from_sizes_equal_padded_shapes_of_the_collated_chunks(pool, supports, adjacency, seed):
    rng = np.random.default_rng(seed)
    B = int(rng.integers(7, 30))
    ids = rng.permutation(len(pool.n))[:B * int(rng.integers(2, 4)) + int(rng.integers(1, B))]     # a short last chunk
    chunks, w = eval_chunks(ids, B, pool.n)
    assert w[-1, -1] == 0
    batches = [pool.collate(c, adjacency=adjacency) for c in chunks]
    if not supports:
        for b in batches:
            del b.edge_index2, b.edge_attr2
    for deg in (8, 3):
        Np, Ep, Mp = eval_shapes(_Sizes(pool, supports, adjacency), chunks, max_pad_degree=deg)
        if adjacency:
            assert (Np, Ep, Mp) == padded_shapes(batches, max_pad_degree=deg, adjacency=True)
        else:
            assert Mp is None and (Np, Ep) == padded_shapes(batches, max_pad_degree=deg)


def test_padded_shapes_from_sizes_keeps_the_rule():
    """Both forms of the rule on hand-made totals (the formula padded_shapes had before it was shared)."""
    n, e, m = [30, 41, 35], [200, 260, 190], [60, 75, 70]
    assert padded_shapes_from_sizes(n, e) == (41 + 1 + (260 - 190 + 7) // 8, 260)
    Np, Ep, Mp = padded_shapes_from_sizes(n, e, m, max_pad_degree=8)
    nd = Np - 41
    assert Ep == 260 and Mp == 75 and -(-70 // nd) + -(-15 // nd) <= 8 and -(-70 // (nd - 1)) + -(-15 // (nd - 1)) > 8
    assert padded_shapes_from_sizes(n, None, m)[1] is None


def test_chunks_follow_ids_and_fill_with_the_smallest_graph(pool):
    ids = np.array([17, 3, 99, 42, 5, 64, 8, 77, 23, 11, 50], np.int64)
    chunks, w = eval_chunks(ids, 4, pool.n)
    assert chunks.shape == (3, 4) and w.shape == (3, 4)
    assert np.array_equal(chunks.reshape(-1)[:len(ids)], ids)
    smallest = ids[np.argmin(pool.n[ids])]
    assert pool.n[smallest] == pool.n[ids].min()
    assert np.array_equal(chunks[2, 3:], [smallest])
    assert np.array_equal(w.reshape(-1), [1.0] * len(ids) + [0.0])
    assert w.dtype == np.float32 and chunks.dtype == np.int64


def test_full_chunks_have_no_fillers_and_batch_size_is_clipped(pool):
    ids = np.arange(12)
    chunks, w = eval_chunks(ids, 4, pool.n)
    assert chunks.shape == (3, 4) and bool((w == 1).all())
    chunks, w = eval_chunks(ids[:5], 64, pool.n)                # batch_size larger than the split
    assert chunks.shape == (1, 5) and np.array_equal(chunks[0], ids[:5]) and bool((w == 1).all())


def _np_terms(metric, o, y):
    o, y = o.astype(np.float64), y.astype(np.float64).reshape(o.shape)
    if metric == "l1":
        return np.abs(o - y).sum(1), None
    if metric == "mse":
        return ((o - y) ** 2).sum(1), None
    p = 1.0 / (1.0 + np.exp(-o))
    t = -(y * np.maximum(np.log(p), -100) + (1 - y) * np.maximum(np.log(1 - p), -100)).sum(1)
    return t, (((o[:, 0] > 0) == (y[:, 0] > 0.5)).astype(np.float64) if o.shape[1] == 1 else None)


@pytest.mark.parametrize("metric", ["l1", "mse", "bce"])
@pytest.mark.parametrize("width", [1, 3])
def test_metric_terms_match_numpy(metric, width):
    g = torch.Generator().manual_seed(width)
    o = torch.randn(37, width, generator=g) * 3
    y = (torch.rand(37, width, generator=g) > 0.5).float() if metric == "bce" else torch.randn(37 * width, generator=g)
    term, correct = eval_terms(metric, o, y)
    rt, rc = _np_terms(metric, o.numpy(), y.numpy())
    np.testing.assert_allclose(term.numpy(), rt, rtol=1e-5, atol=1e-6)
    if rc is None:
        assert correct is None
    else:
        assert np.array_equal(correct.numpy(), rc)
    from gnn_matlang_b200.train import loss_fn
    assert abs(float(term.double().sum()) - float(loss_fn(metric, o, y))) <= 1e-5 * max(1.0, abs(float(rt.sum())))
    with pytest.raises(ValueError):
        eval_terms("nll", o, y)


class _NoDevice(object):
    """A dataset whose device tensors raise when touched: the constructor's checks must come first."""

    def __init__(self, n):
        self.n_h = np.full(n, 5, np.int64)
        self.e_h = np.full(n, 20, np.int64)
        self.m_h = None

    def __getattr__(self, k):
        raise AssertionError("the constructor touched dataset.%s before rejecting its arguments" % k)


class _NoModel(torch.nn.Module):
    def forward(self, data):
        raise AssertionError("the constructor ran the model before rejecting its arguments")


@pytest.mark.parametrize("kw,msg", [(dict(metric="nll"), "metric"), (dict(ids=[]), "empty"), (dict(ids=[0, 10]), "outside"),
                                    (dict(ids=[-1, 2]), "outside"), (dict(batch_size=0), "batch_size")])
def test_constructor_rejects_bad_arguments_before_touching_a_device(kw, msg):
    args = dict(ids=[0, 1, 2], batch_size=2, metric="l1")
    args.update(kw)
    with pytest.raises(ValueError, match=msg):
        GraphedEvaluator(_NoModel(), _NoDevice(10), args["ids"], args["batch_size"], metric=args["metric"])
