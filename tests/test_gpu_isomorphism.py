"""The isomorphism test on the B200: the pair-distinguishing kernels (``gnnml3_pairs_mark`` / ``gnnml3_pairs_count``) against a
float64 torch reference, the cross-seed bitmap of ``isomorphism.PairTracker``, and the paper's known answers through
``isomorphism.isomorphism_test`` (graph8c, SR25, the committed EXP pairs)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_kernels import assert_close, dev  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
EPS32 = 2.0 ** -24


# ------------------------------------------------------------------------------------------------------ references
def _unpack(tr):
    """The tracker's bitmap as bools: [n, n] (bit j of row i at [i, j]) or [P] for listed pairs."""
    b = tr.bits.long() & 0xffffffff
    if tr.pairs is None:
        j = torch.arange(tr.n, device=b.device)
        return ((b[:, j // 32] >> (j % 32)) & 1).bool()
    p = torch.arange(tr.P, device=b.device)
    return ((b[p // 32] >> (p % 32)) & 1).bool()


def _dist64(emb, a_rows=None, b_rows=None):
    """Exact-ish L1 distances in float64 from the float32 values, and the FP32 rounding bound of each: the kernel's sum of
    d terms |a_k - b_k| carries at most (d + 1) EPS32 * sum_k (|a_k| + |b_k|)."""
    e = emb.double()
    a = e if a_rows is None else e[a_rows]
    b = e if b_rows is None else e[b_rows]
    if a_rows is None:
        dist = torch.cdist(a, b, p=1) if bool(torch.isfinite(e).all()) else (a[:, None] - b[None]).abs().sum(-1)
        mag = a.abs().sum(1)[:, None] + b.abs().sum(1)[None, :]
    else:
        dist = (a - b).abs().sum(1)
        mag = a.abs().sum(1) + b.abs().sum(1)
    return dist, (emb.size(1) + 2) * EPS32 * mag


def _expected(emb, thr):
    """float64 reference of the all-pairs bitmap (upper triangle) and the mask of pairs within FP32 rounding of thr."""
    n = emb.size(0)
    thr32 = float(np.float32(thr))
    dist, bound = _dist64(emb)
    upper = torch.ones(n, n, dtype=torch.bool, device=emb.device).triu_(1)
    ref = (dist > thr32) & upper
    near = ((dist - thr32).abs() <= bound) & upper
    return ref, upper, near


# ------------------------------------------------------------------------------------------------------ the kernels
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 1000, 4097])
@pytest.mark.parametrize("d", [1, 3, 10, 32, 100])
def test_all_pairs_bitmap_against_float64(n, d):
    """Random embeddings in a strided buffer (ld = d + 3, the extra columns hold NaN that must not be read), threshold at the
    median distance so that both outcomes are common; bit for bit against float64, except pairs within FP32 rounding."""
    from gnn_matlang_b200.isomorphism import PairTracker
    g = torch.Generator(device=dev()).manual_seed(1000 * n + d)
    buf = torch.full((n, d + 3), float("nan"), device=dev())
    buf[:, :d] = torch.randn(n, d, generator=g, device=dev())
    emb = buf[:, :d]
    assert emb.stride(0) == d + 3
    if n > 1:
        dist, _ = _dist64(emb)
        thr = float(dist[torch.ones(n, n, dtype=torch.bool, device=dev()).triu(1)].median())
    else:
        thr = 1e-3
    tr = PairTracker(n, dev(), threshold=thr)
    tr.update(emb)
    got = _unpack(tr)
    ref, upper, near = _expected(emb, thr)
    assert not bool((got & ~upper).any()), "bits set outside the upper triangle"
    bad = (got != ref) & ~near
    print("n=%d d=%d: %d pairs, %d distinguished, %d within FP32 rounding of the threshold (excluded)"
          % (n, d, int(upper.sum()), int(ref.sum()), int(near.sum())))
    assert int(bad.sum()) == 0, "%d pairs differ from the float64 reference" % int(bad.sum())
    cnt = int(tr.count())
    assert cnt == int((~got & upper).sum())


def test_constructed_ties_nan_inf_duplicates():
    """dist == thr is not distinguished (strict >), NaN distances are not distinguished, inf against a finite row is, inf
    against inf (inf - inf = NaN) is not, duplicates are not; n = 161 is a multiple of neither 32 nor 128."""
    from gnn_matlang_b200.isomorphism import PairTracker
    n, d = 161, 4
    g = torch.Generator().manual_seed(3)
    e = torch.randn(n, d, generator=g) * 10.0
    e[0] = torch.tensor([1.0, 2.0, 4.0, 8.0])
    e[1] = torch.tensor([1.0, 2.0, 4.5, 8.0])                  # |row 1 - row 0| = 0.5 exactly in FP32: a tie
    e[2] = torch.tensor([1.0, 2.0, 4.5, 8.0000010])            # just over 0.5 from row 0
    e[3] = e[40]                                               # duplicates
    e[100] = e[160]
    e[5, 1] = float("nan")                                     # NaN row: never distinguished from anything
    e[6, 0] = float("inf")                                     # inf rows: distinguished from finite rows ...
    e[7, 0] = float("inf")                                     # ... not from each other (inf - inf = NaN)
    emb = e.to(dev())
    tr = PairTracker(n, dev(), threshold=0.5)
    tr.update(emb)
    got = _unpack(tr)
    ref = ((e.double()[:, None] - e.double()[None]).abs().sum(-1) > 0.5).to(dev()) & torch.ones(n, n, dtype=torch.bool,
                                                                                                   device=dev()).triu(1)
    assert not bool(got[0, 1]), "a tie (dist == threshold) must not count as distinguished"
    assert bool(got[0, 2])
    assert not bool(got[3, 40]) and not bool(got[100, 160])
    assert not bool(got[5].any()) and not bool(got[:5, 5].any())
    assert bool(got[6, 8]) and not bool(got[6, 7])
    assert torch.equal(got, ref)
    assert int(tr.count()) == int((~got).triu(1).sum())


def test_updates_accumulate_and_the_skip_rule_keeps_marked_bits():
    """Two clusterings OR into one bitmap; a tile pre-filled by hand (full: skipped) and a tile partly marked by hand keep
    every bit they had, and the partly marked tile gains the new ones; count() equals the unpacked bitmap after every step."""
    from gnn_matlang_b200.isomorphism import PairTracker
    n, d = 600, 10
    g = torch.Generator().manual_seed(5)
    centers = torch.randn(8, d, generator=g)
    lab1 = torch.randint(0, 8, (n,), generator=g)
    lab2 = torch.randint(0, 8, (n,), generator=g)
    e1, e2 = centers[lab1].to(dev()), centers[lab2].to(dev())      # rows of one cluster are identical
    tr = PairTracker(n, dev())
    upper = torch.ones(n, n, dtype=torch.bool, device=dev()).triu(1)
    # tile (row block 1, column block 3): every valid bit set by hand; tile (0, 2): one word of each row set by hand
    tr.bits[128:256, 12:16] = -1
    tr.bits[0:128, 8] = 0x0f0f0f0f
    manual = _unpack(tr) & upper
    steps = [manual]
    for e, lab in ((e1, lab1), (e2, lab2)):
        tr.update(e)
        steps.append(steps[-1] | ((lab[:, None] != lab[None, :]).to(dev()) & upper))
        got = _unpack(tr) & upper
        assert torch.equal(got, steps[-1])
        assert int(tr.count()) == int((~got & upper).sum())
    tr.update(torch.zeros(n, d, device=dev()))                 # distinguishes nothing: the bitmap must not change
    assert torch.equal(_unpack(tr) & upper, steps[-1])
    assert bool(tr.bits[128:256, 12:16].eq(-1).all())
    tr.reset()
    assert int(tr.count()) == n * (n - 1) // 2


def test_listed_pairs_mode():
    """exp_iso.py's mode: P listed pairs, including self pairs (distance 0) and repeats, against float64; the same pair gets
    the same bit as in all-pairs mode (same arithmetic)."""
    from gnn_matlang_b200.isomorphism import PairTracker
    n, d, P = 300, 10, 1001
    g = torch.Generator().manual_seed(8)
    e = torch.randn(n, d, generator=g)
    e[10] = e[11]
    pairs = torch.randint(0, n, (P, 2), generator=g)
    pairs[0] = torch.tensor([10, 11])
    pairs[1] = torch.tensor([7, 7])
    pairs[2] = pairs[3]
    emb = e.to(dev())
    dist, _ = _dist64(emb)
    thr = float(dist.median())
    for src in ("host", "device"):
        tr = PairTracker(n, dev(), threshold=thr, pairs=pairs.numpy() if src == "host" else pairs.to(dev()))
        tr.update(emb)
        got = _unpack(tr)
        allp = PairTracker(n, dev(), threshold=thr)
        allp.update(emb)
        full = _unpack(allp)
        i, j = pairs[:, 0].to(dev()), pairs[:, 1].to(dev())
        ref = full[torch.minimum(i, j), torch.maximum(i, j)]
        assert torch.equal(got, ref), src
        assert not bool(got[0]) and not bool(got[1])
        d64, bound = _dist64(emb, i, j)
        thr32 = float(np.float32(thr))
        far = (d64 - thr32).abs() > bound
        assert torch.equal(got[far], (d64 > thr32)[far])
        assert int(tr.count()) == int((~got).sum())
        tr.update(emb)                                         # idempotent
        assert torch.equal(_unpack(tr), got)


@pytest.mark.parametrize("mode", ["all", "listed"])
def test_update_and_count_replay_in_a_cuda_graph(mode):
    from gnn_matlang_b200.isomorphism import PairTracker
    n, d = 1000, 10
    g = torch.Generator().manual_seed(11)
    pairs = torch.randint(0, n, (333, 2), generator=g) if mode == "listed" else None
    static = torch.zeros(n, d, device=dev())
    cnt = torch.zeros((), dtype=torch.int64, device=dev())
    tr = PairTracker(n, dev(), threshold=6.0, pairs=pairs)
    ref = PairTracker(n, dev(), threshold=6.0, pairs=pairs)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        tr.update(static)
        tr.count(out=cnt)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        tr.update(static)
        tr.count(out=cnt)
    tr.reset()
    for k in range(3):
        e = torch.randn(n, d, generator=g).to(dev())
        static.copy_(e)
        graph.replay()
        ref.update(e)
        torch.cuda.synchronize()
        assert torch.equal(tr.bits, ref.bits)
        assert int(cnt) == int(ref.count()), k


# ------------------------------------------------------------------------------------------------------ known answers
@pytest.fixture(scope="module")
def graph8c_recs():
    from gnn_matlang_b200.datasets import read_graph6
    return read_graph6(os.path.join(GOLDEN, "graph8c.g6"))


def _designed(edge_lists, xs):
    """Resident dataset with the graph8c design (recfield=1, dv=2, nfreq=5, adddegree=True) designed on the GPU."""
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset
    ns = np.array([x.shape[0] for x in xs], np.int64)
    es = np.array([e.shape[1] for e in edge_lists], np.int64)
    node_ptr, edge_ptr = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(es)])
    ei = torch.from_numpy(np.concatenate(edge_lists, 1).astype(np.int64)).to(dev())
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    design = sd.design_batch(ei, torch.from_numpy(edge_ptr).to(dev()), torch.from_numpy(node_ptr), device=dev())
    x = torch.cat([torch.from_numpy(np.concatenate(xs, 0).astype(np.float32)).reshape(-1, 1).to(dev()),
                   design["degree"].unsqueeze(-1)], 1)
    return DeviceDataset.from_design(design, node_ptr, x)


def _ml3():
    from gnn_matlang_b200.models import GNNML3
    return GNNML3("graph8c", ne=6, ninp=2)                    # graph8c.py, sr25.py and exp_iso.py share the architecture


def _ml1(preset="graph8c"):
    from gnn_matlang_b200.models import GNNML1
    return lambda: GNNML1(preset, ninp=1)


@pytest.fixture(scope="module")
def graph8c_ml3(graph8c_recs):
    return _designed([r["edge_index"] for r in graph8c_recs], [np.ones((r["x"].shape[0], 1)) for r in graph8c_recs])


def test_graph8c_gnnml3_two_seeds(graph8c_ml3):
    from gnn_matlang_b200.isomorphism import isomorphism_test
    res = isomorphism_test(_ml3, graph8c_ml3, seeds=range(2))
    print("graph8c GNNML3, seeds 0-1:", res)
    assert res["graphs"] == 11117 and res["pairs"] == 11117 * 11116 // 2
    assert res["counts"] == [1, 0]


def test_graph8c_gnnml1_seed0_matches_the_oracle_count(graph8c_recs):
    from gnn_matlang_b200.isomorphism import isomorphism_test
    from gnn_matlang_b200.synthetic import DeviceDataset
    dds = DeviceDataset.from_graphs(graph8c_recs, dev())
    res = isomorphism_test(_ml1(), dds, seeds=[0], return_embeddings=True)
    emb = res["embeddings"][0].double()
    margin = float("inf")
    n = emb.size(0)
    for i0 in range(0, n, 2048):
        dd = torch.cdist(emb[i0:i0 + 2048], emb, p=1)
        rows = torch.arange(i0, min(i0 + 2048, n), device=dev())
        upper = torch.arange(n, device=dev())[None, :] > rows[:, None]
        margin = min(margin, float(((dd - 1e-3).abs() + (~upper) * 1e9).min()))
    print("graph8c GNNML1 seed 0: %d undistinguished; nearest pair |L1 - 1e-3| = %.3e" % (res["counts"][0], margin))
    assert res["counts"] == [14579]


def test_sr25_no_pair_distinguished():
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.isomorphism import isomorphism_test
    from gnn_matlang_b200.synthetic import DeviceDataset
    recs = read_graph6(os.path.join(GOLDEN, "sr251256.g6"))
    assert len(recs) == 15
    dds3 = _designed([r["edge_index"] for r in recs], [np.ones((r["x"].shape[0], 1)) for r in recs])
    r3 = isomorphism_test(_ml3, dds3, seeds=range(2))
    r1 = isomorphism_test(_ml1(), DeviceDataset.from_graphs(recs, dev()), seeds=range(2))
    print("SR25: GNNML3 %s, GNNML1 %s" % (r3["counts"], r1["counts"]))
    assert r3["pairs"] == 105 and r3["counts"] == [105, 105]
    assert r1["counts"] == [105, 105]


def test_exp_listed_pairs():
    """exp_iso.py on the 100 committed pairs (E[0::2] against E[1::2]), seed 0: GNNML3 separates every pair, GNNML1 none."""
    from gnn_matlang_b200.isomorphism import isomorphism_test
    from gnn_matlang_b200.synthetic import DeviceDataset, ExpPool
    ep = ExpPool()
    G = len(ep.n)
    edge_lists = [ep.ei1[:, ep.edge_off1[i]:ep.edge_off1[i + 1]] for i in range(G)]
    xs = [ep.x[ep.node_off[i]:ep.node_off[i + 1]] for i in range(G)]
    pairs = np.stack([np.arange(0, G, 2), np.arange(1, G, 2)], 1)
    r3 = isomorphism_test(_ml3, _designed(edge_lists, xs), seeds=[0], pairs=pairs)
    recs = [dict(x=x, edge_index=e, y=np.zeros(1, np.float32)) for x, e in zip(xs, edge_lists)]
    r1 = isomorphism_test(_ml1("exp"), DeviceDataset.from_graphs(recs, dev()), seeds=[0], pairs=pairs)
    print("EXP: GNNML3 %s, GNNML1 %s of %d pairs" % (r3["counts"], r1["counts"], r3["pairs"]))
    assert r3["pairs"] == 100 and r3["counts"] == [0]
    assert r1["counts"] == [100]


def test_in_place_reseeding_equals_fresh_models(graph8c_ml3):
    """The embeddings isomorphism_test used for seeds 0, 1 and 5 (one captured evaluator, later models loaded in place) equal
    an eager no_grad forward of a model freshly built under that seed."""
    from gnn_matlang_b200.isomorphism import isomorphism_test
    seeds = [0, 1, 5]
    ids = np.arange(0, 11117, 7)
    res = isomorphism_test(_ml3, graph8c_ml3, seeds=seeds, ids=ids, return_embeddings=True)
    for seed, emb in zip(seeds, res["embeddings"]):
        torch.manual_seed(seed)
        model = _ml3().to(dev()).eval()
        with torch.no_grad():
            ref = torch.cat([model(graph8c_ml3.collate(ids[i:i + 100])) for i in range(0, len(ids), 100)])
        print("seed %d: largest embedding difference %.3e" % (seed, float((emb - ref).abs().max())))
        assert_close(emb, ref, name="seed %d embeddings" % seed)
    assert not torch.equal(res["embeddings"][0], res["embeddings"][1])
