"""CPU restatement of GNNML1 (the paper's 1-WL model, defined next to GNNML3 in every experiment script of the reference) for the
GNNML1 tests: the layer formula in the op order of the reference's GNNML1 classes,
``F.relu(fc11(x) + conv11(x, edge_index, ones) + fc12(x) * fc13(x))`` and its ``torch.cat`` form, on the oracle's
``propagate_add`` with a ones weight.  No fixture made by the reference pins it; ``test_cpu_gnnml1.py`` checks it against an
independent float64 dense-matrix statement."""
import torch
import torch.nn.functional as F

from oracle.gnnml3_oracle import MODEL_CONFIGS, global_add_pool, global_mean_pool, glorot_, propagate_add


def ml1layer_forward(x, edge_index, p, concat=False, prefix="", act=F.relu):
    """GNNML1 layer.  ``p`` maps ``{prefix}conv.weight`` [1, Fi, Fo], ``{prefix}conv.bias``, ``{prefix}fcA/fcB/fcC.weight`` [Fo, Fi]
    and ``.bias`` to tensors; the aggregate is ``propagate_add`` over the plain ``edge_index`` with a ones weight.  ``act``
    replaces the ReLU (the identity gives the pre-activations, which the tests use to keep gradients off the kinks)."""
    ones = torch.ones(edge_index.size(1), dtype=x.dtype)
    fa = x @ p[prefix + "fcA.weight"].t() + p[prefix + "fcA.bias"]
    fc = propagate_add(x, edge_index, ones) @ p[prefix + "conv.weight"][0] + p[prefix + "conv.bias"]
    fbc = (x @ p[prefix + "fcB.weight"].t() + p[prefix + "fcB.bias"]) * (x @ p[prefix + "fcC.weight"].t() + p[prefix + "fcC.bias"])
    if concat:
        return torch.cat([act(fa), act(fc), act(fbc)], 1)
    return act(fa + fc + fbc)


class OracleGNNML1(torch.nn.Module):
    """GNNML1 model: ``nlayer`` GNNML1 layers (parameters ``conv{l}1``, ``fc{l}1``, ``fc{l}2``, ``fc{l}3``), then the read-out and
    head of the same-named GNNML3 preset.  ``forward(b)`` reads ``x``, ``edge_index``, ``batch``, ``num_graphs``."""

    def __init__(self, config, ninp, nlayer=3, nout=64, concat=False):
        super().__init__()
        c = MODEL_CONFIGS[config] if isinstance(config, str) else config
        self.c, self.nlayer, self.concat = c, nlayer, concat
        width = nout * (3 if concat else 1)
        for l in range(1, nlayer + 1):
            nin = ninp if l == 1 else width
            conv = torch.nn.Module()
            conv.weight = torch.nn.Parameter(glorot_(torch.empty(1, nin, nout)))
            conv.bias = torch.nn.Parameter(torch.zeros(nout))
            setattr(self, "conv%d1" % l, conv)
            for j in (1, 2, 3):
                setattr(self, "fc%d%d" % (l, j), torch.nn.Linear(nin, nout))
        self.fc1 = torch.nn.Linear(width, c["head"][0])
        if len(c["head"]) > 1:
            self.fc2 = torch.nn.Linear(c["head"][0], c["head"][1])

    def forward(self, b):
        x = b["x"]
        for l in range(1, self.nlayer + 1):
            p = {"conv.weight": getattr(self, "conv%d1" % l).weight, "conv.bias": getattr(self, "conv%d1" % l).bias}
            for j, n in ((1, "fcA"), (2, "fcB"), (3, "fcC")):
                fc = getattr(self, "fc%d%d" % (l, j))
                p[n + ".weight"], p[n + ".bias"] = fc.weight, fc.bias
            x = ml1layer_forward(x, b["edge_index"], p, self.concat)
        pool = global_add_pool if self.c["pool"] == "add" else global_mean_pool
        x = pool(x, b["batch"], b["num_graphs"])
        if len(self.c["head"]) == 1:
            x = self.fc1(x)
            return torch.tanh(x) if self.c["final"] == "tanh" else x
        return self.fc2(F.relu(self.fc1(x)))
