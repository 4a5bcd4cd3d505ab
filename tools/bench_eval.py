#!/usr/bin/env python
"""bench_eval.py -- forward-only inference and the captured evaluation pass on one B200.  Prints ONE JSON line with

* ``forward_only``: one batch of 8192 ZINC-shaped graphs (``synthetic.zinc_graph``, real SpectralDesign supports as in bench.py)
  through the GNNML3 ``zinc`` preset and the GNNML1 ``zinc`` preset: device time of the model forward with grad enabled (what a
  training step's forward writes) and under ``no_grad`` (the forward-only kernels), alternating; the peak allocation of each;
  whether the outputs are bit-identical; the bytes the forward no longer writes, computed from the shapes;
* ``evaluator``: a resident dataset of 65,536 ZINC-shaped graphs (``DeviceDataset``), evaluated at 8192 graphs per batch (all
  graphs) and at 64 (a split of 8192 graphs), for both models: the eager loop (``dds.collate``, a ``no_grad`` forward, the L1 metric
  accumulated on the device) against ``train.GraphedEvaluator.run()``, in graphs/s, each pass ending in one read of the metric;
* ``graph8c``: all 11,117 graph8c graphs at 100 per batch with a seed-0 GNNML3 (bench.py's protocol): the eager loop against the
  evaluator, and the undistinguished-pair count of each;
* the card's name and power limit, read in the same run.

    python tools/bench_eval.py [--rounds 3] [--out FILE]

Nothing is written unless --out is given.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # pragma: no cover
        q = "unavailable (%s)" % e
    return dict(name=name, power_limit_and_max_sm_clock=q)


def _ms(fn, reps):
    """Median device time of fn() over reps calls, each bracketed by CUDA events (outputs dropped after the synchronise)."""
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        del out
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def _peak(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out
    return int(peak)


def forward_only(dev, rounds):
    from gnn_matlang_b200.models import GNNML1, GNNML3
    from gnn_matlang_b200.synthetic import GraphPool
    B = 8192
    pool = GraphPool("zinc", B, seed=0).attach_spectral_supports(dev)
    batch = pool.collate(np.arange(B), adjacency=True).to(dev)
    N = int(batch.x.size(0))
    out = {"graphs": B, "nodes": N, "support_entries": int(batch.edge_index2.size(1)), "edges": int(batch.edge_index.size(1))}
    torch.manual_seed(0)
    models = {"gnnml3_zinc": GNNML3("zinc", pool.K, pool.F).to(dev), "gnnml1_zinc": GNNML1("zinc", pool.F).to(dev)}
    K, G3 = pool.K, 2                    # zinc preset: 4 x ML3Layer(30||2), the first with Fi = 25 <= 32 (aggregate kept)
    saved = {"gnnml3_zinc": {"first_layer_aggregate_bytes": N * (K + 1) * 32 * 4, "tanh_factor_bytes": 4 * N * 2 * G3 * 4},
             "gnnml1_zinc": {"p1_p2_bytes": 3 * N * 2 * 64 * 4, "y_bytes": 3 * N * 64 * 4}}
    for name, m in models.items():
        grad = lambda: m(batch.fresh())

        def nograd():
            with torch.no_grad():
                return m(batch.fresh())
        for _ in range(3):
            grad(), nograd()
        same = bool(torch.equal(grad().detach(), nograd()))
        tg, tn = [], []
        for _ in range(rounds):                             # alternating
            tg.append(_ms(grad, 10))
            tn.append(_ms(nograd, 10))
        s = dict(saved[name])
        s["total_bytes"] = sum(v for k, v in s.items() if k != "y_bytes")
        if name == "gnnml1_zinc":
            s["share_of_layer_stores"] = s["p1_p2_bytes"] / (s["p1_p2_bytes"] + s["y_bytes"])
        out[name] = {"ms_forward_grad_enabled": float(np.median(tg)), "ms_forward_no_grad": float(np.median(tn)),
                     "ms_rounds_grad": tg, "ms_rounds_no_grad": tn, "peak_alloc_bytes_grad_enabled": _peak(grad),
                     "peak_alloc_bytes_no_grad": _peak(nograd), "outputs_bit_identical": same, "bytes_not_written": s}
    return out


def _eager_pass(model, dds, chunks):
    from gnn_matlang_b200.train import eval_terms
    acc = torch.zeros((), dtype=torch.float64, device=dds.x.device)
    with torch.no_grad():
        for ix in chunks:
            b = dds.collate(ix)
            o = model(b)
            acc += eval_terms("l1", o, b.y)[0].double().sum()
    return float(acc)


def _wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    v = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, v


def evaluator(dev, rounds, pool_size):
    from gnn_matlang_b200.models import GNNML1, GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset, GraphPool
    from gnn_matlang_b200.train import GraphedEvaluator
    pool = GraphPool("zinc", pool_size, seed=1).attach_spectral_supports(dev)
    data = {"gnnml3_zinc": DeviceDataset(pool, dev), "gnnml1_zinc": DeviceDataset(pool, dev, adjacency=True, supports=False)}
    torch.manual_seed(0)
    models = {"gnnml3_zinc": GNNML3("zinc", pool.K, pool.F).to(dev).eval(), "gnnml1_zinc": GNNML1("zinc", pool.F).to(dev).eval()}
    out = {"pool_graphs": pool_size}
    for B, n_ids in ((8192, pool_size), (64, 8192)):
        ids = np.arange(n_ids)
        chunks = [torch.from_numpy(ids[i:i + B]).pin_memory() for i in range(0, n_ids, B)]
        for name, m in models.items():
            dds = data[name]
            ev = GraphedEvaluator(m, dds, ids, B, metric="l1")
            _eager_pass(m, dds, chunks)
            ev.run()
            te, tc = [], []
            for _ in range(rounds):
                ms, se = _wall(lambda: _eager_pass(m, dds, chunks))
                te.append(ms)
                ms, r = _wall(ev.run)
                tc.append(ms)
            e, c = float(np.median(te)), float(np.median(tc))
            out["%s_b%d" % (name, B)] = {"graphs": n_ids, "batches": len(chunks), "eager_ms": e, "evaluator_ms": c,
                                          "eager_graphs_per_s": n_ids / (e * 1e-3), "evaluator_graphs_per_s": n_ids / (c * 1e-3),
                                          "l1_sum_eager": se, "l1_sum_evaluator": r["sum"]}
            del ev
    return out


def graph8c(dev, rounds):
    from gnn_matlang_b200.datasets import read_graph6
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.synthetic import DeviceDataset
    from gnn_matlang_b200.train import GraphedEvaluator
    recs = read_graph6(os.path.join(ROOT, "tests", "golden", "graph8c.g6"))
    ns = np.array([r["x"].shape[0] for r in recs], np.int64)
    es = np.array([r["edge_index"].shape[1] for r in recs], np.int64)
    node_ptr, edge_ptr = np.concatenate([[0], np.cumsum(ns)]), np.concatenate([[0], np.cumsum(es)])
    ei = torch.from_numpy(np.concatenate([r["edge_index"] for r in recs], 1)).to(dev)
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    design = sd.design_batch(ei, torch.from_numpy(edge_ptr).to(dev), torch.from_numpy(node_ptr), device=dev)
    x = torch.cat([torch.ones(int(node_ptr[-1]), 1, device=dev), design["degree"].unsqueeze(-1)], 1)
    dds = DeviceDataset.from_design(design, node_ptr, x)
    torch.manual_seed(0)
    model = GNNML3("graph8c", ne=6, ninp=2).to(dev).eval()
    G = len(recs)
    idx = [torch.arange(s, min(s + 100, G)).pin_memory() for s in range(0, G, 100)]

    def embed_all():
        with torch.no_grad():
            return torch.cat([model(dds.collate(ix)) for ix in idx])

    def pairs(emb):
        similar = 0
        for r in range(0, G, 2048):
            similar += int((torch.cdist(emb[r:r + 2048], emb, p=1) <= 0.001).sum())
        return (similar - G) // 2

    ev = GraphedEvaluator(model, dds, np.arange(G), 100, metric=None)
    embed_all()
    ev.run(outputs=True)
    te, tc = [], []
    for _ in range(rounds):
        ms, emb_e = _wall(embed_all)
        te.append(ms)
        ms, r = _wall(lambda: ev.run(outputs=True))
        tc.append(ms)
    e, c = float(np.median(te)), float(np.median(tc))
    return {"graphs": G, "batches": len(idx), "eager_ms": e, "evaluator_ms": c, "eager_graphs_per_s": G / (e * 1e-3),
            "evaluator_graphs_per_s": G / (c * 1e-3), "undistinguished_pairs_eager": pairs(emb_e),
            "undistinguished_pairs_evaluator": pairs(r["outputs"]), "known_answer": 1,
            "largest_embedding_difference": float((r["outputs"] - emb_e).abs().max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pool", type=int, default=65536)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py measures on a CUDA device; none is visible")
    from gnn_matlang_b200 import _lib
    from gnn_matlang_b200.graph import set_range_check
    _lib.load()
    set_range_check(False)
    dev = torch.device("cuda:0")
    res = {"bench": "bench_eval", "card": card()}
    res["forward_only"] = forward_only(dev, args.rounds)
    res["evaluator"] = evaluator(dev, args.rounds, args.pool)
    res["graph8c"] = graph8c(dev, args.rounds)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
