"""The GNNML3 model wrappers of the reference's four configured scripts, as one parameterised module with
the reference's sub-module names (``conv1..convL``, ``fc1``, ``fc2``), creation order and forward:

* ``graph8c``  -- graph8c.py:249-279      3 x ML3Layer(32||16), add-pool, tanh(fc1 -> 10)
* ``zinc``     -- Zinc12k.py:310-345      4 x ML3Layer(30||2),  add-pool, fc2(relu(fc1 -> 32)) -> 1
* ``exp``      -- exp_classify.py:264-295 3 x ML3Layer(32||16), mean-pool, fc2(relu(fc1 -> 10)) -> 1
* ``counting`` -- counting.py:335-372     5 x ML3Layer(16||16), add-pool, fc2(relu(fc1 -> 32)) -> 1

plus the GNNML3 variants of the TU-dataset scripts (SURVEY.md 8f rank 4) -- unlearned edge features, dropout, BatchNorm,
concatenated read-outs, log-softmax heads:

* ``enzymes``  -- enzymes.py:345-386       4 x ML3Layer(64||0, learnedge=False), dropout 0.1 before every layer, add||max pool,
                                          BatchNorm1d(128), log_softmax(fc2 -> 6)
* ``mutag``    -- mutag.py:268-307         3 x ML3Layer(24||24, learnedge=False) each followed by BatchNorm1d, mean-pool,
                                          fc2(relu(fc1 -> 32)) -> 1
* ``filtering`` -- filtering.py:252-281    3 x ML3Layer(32||16, learnedge=False) on ONE 900-node grid (supports from the dense
                                          path of SpectralDesign), no read-out: a per-node regression, fc2 -> 1

The same (unlearned) ``edge_attr2`` feeds every layer; the graph plan (CSR) is built once per batch.  BatchNorm, dropout and
log-softmax are torch modules (statistics / elementwise work on [N, F] and [B, F], outside the hot path of SURVEY.md 8a).
On a padded batch in training mode (``train.pad_batch``, ``real_graphs < num_graphs``) the BatchNorm statistics leave the dummy
graph out: ``bn="layers"`` runs the node BatchNorm kernels of ``norm.batch_norm_rows`` over the first ``graph_ptr[real_graphs]``
rows, ``bn="readout"`` applies the module to the first ``real_graphs`` pooled rows and passes the dummy row through.

``GNNML1`` is the paper's 1-WL model, defined next to GNNML3 in every experiment script of the reference: ``nlayer`` GNNML1
layers (``libs.spect_conv.ML1Layer``) on the graph's plain ``edge_index``, then the pool and head of the same-named GNNML3
preset (``graph8c``, ``zinc``, ``exp``, ``counting``).
"""
import torch
import torch.nn as nn

from .libs.spect_conv import ML3Layer, SpectConv, _LinearFn, _precision_code, ml1_layer
import torch.nn.functional as F

from .norm import batch_norm_rows
from .pool import global_add_pool, global_max_pool, global_mean_pool

MODEL_CONFIGS = {
    "graph8c": dict(nlayer=3, nout1=32, nout2=16, head=(10,), pool="add", final="tanh"),
    "zinc": dict(nlayer=4, nout1=30, nout2=2, head=(32, 1), pool="add", final=None),
    "exp": dict(nlayer=3, nout1=32, nout2=16, head=(10, 1), pool="mean", final=None),
    "counting": dict(nlayer=5, nout1=16, nout2=16, head=(32, 1), pool="add", final=None),
    "enzymes": dict(nlayer=4, nout1=64, nout2=0, head=(6,), pool="add_max", final="log_softmax", learnedge=False, dropout=0.1,
                    bn="readout", fc_name="fc2"),
    "mutag": dict(nlayer=3, nout1=24, nout2=24, head=(32, 1), pool="mean", final=None, learnedge=False, bn="layers"),
    "filtering": dict(nlayer=3, nout1=32, nout2=16, head=(1,), pool="none", final=None, learnedge=False, fc_name="fc2"),
}


class GNNML3(nn.Module):
    def __init__(self, config, ne, ninp, precision="fp32"):
        super().__init__()
        _precision_code(precision)
        c = dict(MODEL_CONFIGS[config]) if isinstance(config, str) else dict(config)
        self.cfg = c
        self.precision = precision
        nin = c["nout1"] + c["nout2"]
        for l in range(c["nlayer"]):
            setattr(self, "conv%d" % (l + 1),
                    ML3Layer(learnedge=c.get("learnedge", True), nedgeinput=ne, nedgeoutput=ne, ninp=ninp if l == 0 else nin,
                             nout1=c["nout1"], nout2=c["nout2"], precision=precision))
        if c.get("bn") == "layers":                      # mutag.py:283-285 (creation order: convs, then bn1.., then the head)
            for l in range(c["nlayer"]):
                setattr(self, "bn%d" % (l + 1), nn.BatchNorm1d(nin))
        npool = nin * (2 if "_" in c["pool"] else 1)
        if c.get("bn") == "readout":                     # enzymes.py:362
            setattr(self, "bn%d" % c["nlayer"], nn.BatchNorm1d(npool))
        if len(c["head"]) == 1 and c.get("fc_name") == "fc2":      # enzymes.py:364: the single head layer is called fc2
            self.fc2 = nn.Linear(npool, c["head"][0])
        else:
            self.fc1 = nn.Linear(npool, c["head"][0])
            if len(c["head"]) > 1:
                self.fc2 = nn.Linear(c["head"][0], c["head"][1])

    def forward(self, data):
        x = data.x
        edge_index = data.edge_index2
        edge_attr = data.edge_attr2
        c = self.cfg
        B = getattr(data, "num_graphs", None)
        # a padded batch (train.pad_batch: one dummy graph behind the real ones) in training mode: BatchNorm statistics over the
        # real rows only, so that the captured step trains the model the eager step trains on the same graphs
        real = getattr(data, "real_graphs", None)
        padded = self.training and c.get("bn") is not None and real is not None and B is not None and real < B
        for l in range(c["nlayer"]):
            if c.get("dropout"):
                x = F.dropout(x, p=c["dropout"], training=self.training)
            x = getattr(self, "conv%d" % (l + 1))(x, edge_index, edge_attr)
            if c.get("bn") == "layers":
                bn = getattr(self, "bn%d" % (l + 1))
                x = batch_norm_rows(x, data.graph_ptr[real:real + 1], bn) if padded else bn(x)
        pools = {"add": global_add_pool, "mean": global_mean_pool, "max": global_max_pool}
        if c["pool"] != "none":                          # "none": node-level output (filtering.py:281)
            x = torch.cat([pools[k](x, data.batch, B) for k in c["pool"].split("_")], 1)
        if c.get("bn") == "readout":
            bn = getattr(self, "bn%d" % c["nlayer"])
            x = torch.cat([bn(x[:real]), x[real:]], 0) if padded else bn(x)
        prec = _precision_code(self.precision)
        if len(c["head"]) == 1:
            fc = self.fc2 if c.get("fc_name") == "fc2" else self.fc1
            x = _LinearFn.apply(x, fc.weight.t(), fc.bias, prec)
            if c["final"] == "tanh":
                return torch.tanh(x)
            return F.log_softmax(x, dim=1) if c["final"] == "log_softmax" else x
        x = _LinearFn.apply(x, self.fc1.weight.t(), self.fc1.bias, prec)
        return _LinearFn.apply(torch.relu(x), self.fc2.weight.t(), self.fc2.bias, prec)


GNNML1_PRESETS = ("graph8c", "zinc", "exp", "counting")


class GNNML1(nn.Module):
    """GNNML1: ``nlayer`` x [relu(fc{l}1(x) + conv{l}1(x, edge_index, ones) + fc{l}2(x) * fc{l}3(x))] (or the concatenated
    form with ``concat=True``: layer width 3 * nout), then the read-out and head of ``MODEL_CONFIGS[config]``.  Parameters keep
    the reference's names: ``conv{l}1`` (SpectConv(K=1, selfconn=False)), ``fc{l}1``, ``fc{l}2``, ``fc{l}3`` (nn.Linear) for
    l = 1..nlayer, then the head (``fc1``, ``fc2``).  ``forward(data)`` reads ``data.x``, ``data.edge_index``, ``data.batch``
    (``batch.collate(graphs, adjacency=True)`` provides ``edge_index``).  ``precision`` ("fp32" = 3xTF32, "tf32", "bf16") is
    the arithmetic of every layer's projections and of the head, as for GNNML3; parameters are the same in every mode."""

    def __init__(self, config, ninp, nlayer=3, nout=64, concat=False, precision="fp32"):
        super().__init__()
        if isinstance(config, str) and config not in GNNML1_PRESETS:
            raise ValueError("GNNML1 presets: %s" % (GNNML1_PRESETS,))
        _precision_code(precision)
        c = dict(MODEL_CONFIGS[config]) if isinstance(config, str) else dict(config)
        self.cfg = c
        self.precision = precision
        self.nlayer, self.concat = int(nlayer), bool(concat)
        width = nout * (3 if concat else 1)
        for l in range(1, self.nlayer + 1):
            nin = ninp if l == 1 else width
            setattr(self, "conv%d1" % l, SpectConv(nin, nout, 1, selfconn=False))
            setattr(self, "fc%d1" % l, nn.Linear(nin, nout))
            setattr(self, "fc%d2" % l, nn.Linear(nin, nout))
            setattr(self, "fc%d3" % l, nn.Linear(nin, nout))
        self.fc1 = nn.Linear(width, c["head"][0])
        if len(c["head"]) > 1:
            self.fc2 = nn.Linear(c["head"][0], c["head"][1])

    def forward(self, data):
        x = data.x
        edge_index = data.edge_index
        for l in range(1, self.nlayer + 1):
            x = ml1_layer(x, edge_index, getattr(self, "conv%d1" % l), getattr(self, "fc%d1" % l), getattr(self, "fc%d2" % l),
                          getattr(self, "fc%d3" % l), self.concat, self.precision)
        c = self.cfg
        B = getattr(data, "num_graphs", None)
        pool = {"add": global_add_pool, "mean": global_mean_pool}[c["pool"]]
        x = pool(x, data.batch, B)
        prec = _precision_code(self.precision)
        x = _LinearFn.apply(x, self.fc1.weight.t(), self.fc1.bias, prec)
        if len(c["head"]) == 1:
            return torch.tanh(x) if c["final"] == "tanh" else x
        return _LinearFn.apply(torch.relu(x), self.fc2.weight.t(), self.fc2.bias, prec)
