"""GNNML1 on the CPU: the oracle layer against an independent float64 dense-matrix statement, its 1-WL blindness on a known
pair, the adjacency collation and the model's parameter names and shapes.  No GPU needed."""
import numpy as np
import pytest
import torch

from gnnml1_oracle import OracleGNNML1, ml1layer_forward


def _params(Fi, Fo, seed):
    g = torch.Generator().manual_seed(seed)
    p = {"conv.weight": torch.randn(1, Fi, Fo, generator=g), "conv.bias": torch.randn(Fo, generator=g)}
    for n in ("fcA", "fcB", "fcC"):
        p[n + ".weight"] = torch.randn(Fo, Fi, generator=g)
        p[n + ".bias"] = torch.randn(Fo, generator=g)
    return p


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_oracle_layer_matches_dense_float64_statement(concat):
    rng = np.random.default_rng(0)
    N, E, Fi, Fo = 40, 150, 7, 5
    ei = torch.from_numpy(rng.integers(0, N, (2, E)).astype(np.int64))
    x = torch.randn(N, Fi, generator=torch.Generator().manual_seed(1))
    p = _params(Fi, Fo, 2)
    A = np.zeros((N, N))
    np.add.at(A, (ei[1].numpy(), ei[0].numpy()), 1.0)                 # A[t, s] = number of edges s -> t
    xd = x.double().numpy()
    W = {k: v.double().numpy() for k, v in p.items()}
    fa = xd @ W["fcA.weight"].T + W["fcA.bias"]
    fc = (A @ xd) @ W["conv.weight"][0] + W["conv.bias"]
    fbc = (xd @ W["fcB.weight"].T + W["fcB.bias"]) * (xd @ W["fcC.weight"].T + W["fcC.bias"])
    relu = lambda v: np.maximum(v, 0)                                   # noqa: E731
    ref = np.concatenate([relu(fa), relu(fc), relu(fbc)], 1) if concat else relu(fa + fc + fbc)
    out = ml1layer_forward(x, ei, p, concat).double().numpy()
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() <= 1e-5 * np.abs(ref).max()


def _cycle(n, off=0):
    u = np.arange(n)
    v = (u + 1) % n
    return np.concatenate([np.vstack((u, v)), np.vstack((v, u))], 1) + off


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_oracle_model_is_blind_to_two_triangles_versus_a_hexagon(concat):
    """1-WL cannot tell two disjoint triangles from a 6-cycle (both 2-regular on 6 nodes): nor can GNNML1."""
    torch.manual_seed(0)
    model = OracleGNNML1("graph8c", ninp=1, nlayer=3, nout=16, concat=concat).double()
    two_tri = np.concatenate([_cycle(3), _cycle(3, 3)], 1)
    hexagon = _cycle(6)
    x = torch.ones(12, 1, dtype=torch.float64)
    b = dict(x=x, edge_index=torch.from_numpy(np.concatenate([two_tri, hexagon + 6], 1)),
             batch=torch.tensor([0] * 6 + [1] * 6), num_graphs=2)
    with torch.no_grad():
        out = model(b)
    assert torch.allclose(out[0], out[1], rtol=0, atol=1e-12)
    with torch.no_grad():                  # (and it is not constant: a 4-cycle plus an isolated edge pair differs)
        b2 = dict(b, edge_index=torch.from_numpy(np.concatenate([_cycle(4), np.array([[4, 5], [5, 4]]), hexagon + 6], 1)))
        out2 = model(b2)
    assert not torch.allclose(out2[0], out2[1], rtol=0, atol=1e-9)


def test_collate_adjacency_is_bit_exact_and_optional():
    from gnn_matlang_b200.batch import collate
    rng = np.random.default_rng(3)
    graphs, off = [], 0
    ref_ei = []
    for i in range(7):
        n = int(rng.integers(1, 12))
        m = int(rng.integers(0, 20))
        ei = rng.integers(0, n, (2, m)).astype(np.int64)
        e2 = int(rng.integers(1, 30))
        graphs.append(dict(x=rng.standard_normal((n, 3)).astype(np.float32), edge_index=ei,
                           edge_index2=rng.integers(0, n, (2, e2)).astype(np.int64),
                           edge_attr2=rng.standard_normal((e2, 4)).astype(np.float32), y=np.float32(i)))
        ref_ei.append(ei + off)
        off += n
    plain = collate(graphs)
    adj = collate(graphs, adjacency=True)
    assert not hasattr(plain, "edge_index")
    assert list(plain.__dict__) == ["x", "edge_index2", "edge_attr2", "batch", "num_graphs", "graph_ptr", "y"]
    assert adj.edge_index.dtype == torch.int64 and np.array_equal(adj.edge_index.numpy(), np.concatenate(ref_ei, 1))
    for k, v in plain.__dict__.items():
        w = getattr(adj, k)
        assert (torch.equal(v, w) if isinstance(v, torch.Tensor) else v == w), k
    # records without SpectralDesign supports (all GNNML1 needs)
    bare = collate([dict(x=g["x"], edge_index=g["edge_index"]) for g in graphs], adjacency=True)
    assert torch.equal(bare.edge_index, adj.edge_index) and not hasattr(bare, "edge_index2")
    assert torch.equal(bare.batch, adj.batch) and torch.equal(bare.graph_ptr, adj.graph_ptr)


@pytest.mark.parametrize("concat", [False, True], ids=["sum", "concat"])
def test_gnnml1_parameter_names_and_shapes(concat):
    from gnn_matlang_b200.models import GNNML1
    from gnn_matlang_b200.libs.spect_conv import ML1Layer
    m = GNNML1("zinc", ninp=25, nlayer=4, nout=64, concat=concat)
    w = 64 * (3 if concat else 1)
    exp = []
    for l in range(1, 5):
        nin = 25 if l == 1 else w
        exp += [("conv%d1.weight" % l, (1, nin, 64)), ("conv%d1.bias" % l, (64,))]
        for j in (1, 2, 3):
            exp += [("fc%d%d.weight" % (l, j), (64, nin)), ("fc%d%d.bias" % (l, j), (64,))]
    exp += [("fc1.weight", (32, w)), ("fc1.bias", (32,)), ("fc2.weight", (1, 32)), ("fc2.bias", (1,))]
    assert [(k, tuple(v.shape)) for k, v in m.named_parameters()] == exp
    o = OracleGNNML1("zinc", 25, 4, 64, concat)
    assert [(k, tuple(v.shape)) for k, v in o.named_parameters()] == exp
    layer = ML1Layer(25, 64, concat=concat)
    assert [k for k, _ in layer.named_parameters()] == ["conv1.weight", "conv1.bias", "fc11.weight", "fc11.bias", "fc12.weight",
                                                         "fc12.bias", "fc13.weight", "fc13.bias"]
    assert layer.out_features == w
    with pytest.raises(ValueError):
        GNNML1("enzymes", ninp=3)
