#!/usr/bin/env python
"""bench_tu.py -- the TU-dataset GNNML3 variants on one B200.  Prints ONE JSON line with

* ``training``: the ``enzymes`` (loss ``nll``) and ``mutag`` (loss ``bce``) presets on resident datasets of synthetic records shaped
  like ENZYMES / MUTAG (``synthetic.tu_records``; SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True), the ENZYMES-shaped
  graphs above the one-block eigensolver's envelope designed on the dense path), at the reference-like batch of 128 graphs and at
  8192: the eager ``Trainer`` (``dds.collate`` + step) against the captured ``GraphedTrainer`` (``load_from_dataset`` + replay),
  ms per step and graphs/s, each timed window ending in a device synchronise;
* ``node_batchnorm``: the node BatchNorm of a padded batch (``gnnml3_bn_rows_fwd`` / ``_bwd``) against the same masked statistics
  composed from torch ops (the composition lives only here), forward and forward + backward, CUDA events around each call;
* the card's name and power limit, read in the same run.

    python tools/bench_tu.py [--steps 20] [--out FILE]

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
    """Median device time of fn() over reps calls, each bracketed by CUDA events."""
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def training(kind, loss, dds, B, steps, dev):
    from gnn_matlang_b200.models import GNNML3
    from gnn_matlang_b200.train import GraphedTrainer, Trainer, eval_shapes, pad_batch
    rng = np.random.default_rng(B)
    G = len(dds.n_h)
    chunks = np.stack([rng.choice(G, B, replace=B > G) for _ in range(steps)])
    Np, Ep, _ = eval_shapes(dds, chunks)
    res = dict(batch=B, steps=steps, nodes_per_batch=int(dds.n_h[chunks].sum(1).mean()),
               support_entries_per_batch=int(dds.e_h[chunks].sum(1).mean()))
    torch.manual_seed(0)
    eager = Trainer(GNNML3(kind, 6, dds.x.size(1)).to(dev), loss=loss)
    torch.manual_seed(0)
    gt = GraphedTrainer(GNNML3(kind, 6, dds.x.size(1)).to(dev), pad_batch(dds.collate(chunks[0]).to("cpu"), Np, Ep).to(dev),
                        loss=loss)
    for c in chunks[:3]:                                     # warm-up of both at every shape the window uses
        eager.step(dds.collate(c))
        gt.load_from_dataset(dds, c)
        gt.step()
    torch.cuda.synchronize()
    for name, run in (("eager", lambda c: eager.step(dds.collate(c))),
                      ("captured", lambda c: (gt.load_from_dataset(dds, c), gt.step()))):
        t0 = time.perf_counter()
        for c in chunks:
            run(c)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        res[name] = dict(ms_per_step=round(ms, 4), graphs_per_s=round(B * 1e3 / ms, 1))
    res["captured_speedup"] = round(res["eager"]["ms_per_step"] / res["captured"]["ms_per_step"], 3)
    return res


def torch_masked_bn(x, cnt, w, b, rm, rv, eps=1e-5, momentum=0.1):
    """The node BatchNorm of a padded batch from torch ops: statistics over rows < cnt (device count), the affine map on all rows."""
    real = (torch.arange(x.size(0), device=x.device) < cnt).unsqueeze(1)
    n = cnt.to(x.dtype)
    mean = torch.where(real, x, 0.0).sum(0) / n
    d = torch.where(real, x - mean, 0.0)
    var = (d * d).sum(0) / n
    with torch.no_grad():
        rm.mul_(1 - momentum).add_(momentum * mean.detach())
        rv.mul_(1 - momentum).add_(momentum * var.detach() * n / (n - 1))
    return (x - mean) * torch.rsqrt(var + eps) * w + b


def node_batchnorm(N, F, dev, reps):
    from gnn_matlang_b200.norm import batch_norm_rows
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(N, F, device=dev, generator=g).requires_grad_(True)
    gy = torch.randn(N, F, device=dev, generator=g)
    cnt = torch.tensor([N - N // 50], dtype=torch.int32, device=dev)      # 2 % of the rows: the padding graph
    bn = torch.nn.BatchNorm1d(F).to(dev)
    w, b = bn.weight, bn.bias
    rm, rv = bn.running_mean.clone(), bn.running_var.clone()
    kern = lambda: batch_norm_rows(x, cnt, bn)
    comp = lambda: torch_masked_bn(x, cnt, w, b, rm, rv)
    res = dict(N=N, F=F, real_rows=int(cnt))
    for name, fn in (("kernel", kern), ("torch_ops", comp)):
        for _ in range(3):
            fn().backward(gy)
        with torch.no_grad():
            fwd = _ms(fn, reps)
        fb = _ms(lambda: fn().backward(gy), reps)
        res[name] = dict(fwd_ms=round(fwd, 4), fwd_bwd_ms=round(fb, 4))
    with torch.no_grad():
        y1, y2 = kern(), comp()
    res["max_abs_diff_fwd"] = float((y1 - y2).abs()[:int(cnt)].max())
    # bytes the kernel pair must move: x read twice + y written (forward), x and gy read twice + dx written (backward)
    res["kernel_min_bytes_fwd_bwd"] = 4 * N * F * 8
    res["kernel_fwd_bwd_GBps"] = round(res["kernel_min_bytes_fwd_bwd"] / (res["kernel"]["fwd_bwd_ms"] * 1e6), 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tu.py measures on a CUDA device; none found")
    from gnn_matlang_b200.libs.utils import SpectralDesign
    from gnn_matlang_b200.synthetic import DeviceDataset, tu_records
    dev = torch.device("cuda:0")
    sd = SpectralDesign(recfield=1, dv=2, nfreq=5, adddegree=True)
    out = dict(tool="bench_tu", card=card(), envelope_nodes=sd.max_kernel_nodes(), training={}, node_batchnorm=[])
    for kind, loss, G in (("enzymes", "nll", 10000), ("mutag", "bce", 10000)):
        t0 = time.perf_counter()
        recs = tu_records(kind, G, seed=0)
        dds = DeviceDataset.from_records(recs, sd, dev)
        torch.cuda.synchronize()
        n = dds.n_h
        out["training"][kind] = dict(graphs=G, above_envelope=int((n > out["envelope_nodes"]).sum()),
                                     from_records_s=round(time.perf_counter() - t0, 3),
                                     runs=[training(kind, loss, dds, B, a.steps, dev) for B in (128, 8192)])
    for N, F in ((147000, 48), (200000, 128)):
        out["node_batchnorm"].append(node_batchnorm(N, F, dev, 50))
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
