"""GNNML1 precision modes on the CPU: an unknown precision is rejected before any device work (by the GNNML3 modules too),
and the precision changes no parameter.  No GPU needed."""
import pytest
import torch


@pytest.mark.parametrize("bad", ["fp16", "FP32", "", None, 1])
def test_bad_precision_is_rejected(bad):
    from gnn_matlang_b200.libs.spect_conv import ML1Layer, ML3Layer, ml1_layer
    from gnn_matlang_b200.models import GNNML1, GNNML3
    with pytest.raises(ValueError, match="precision must be one of"):
        ML1Layer(8, 16, precision=bad)
    with pytest.raises(ValueError, match="precision must be one of"):
        GNNML1("zinc", 25, precision=bad)
    with pytest.raises(ValueError, match="precision must be one of"):
        ML3Layer(True, 4, 4, 8, 16, 2, precision=bad)
    with pytest.raises(ValueError, match="precision must be one of"):
        GNNML3("zinc", 4, 25, precision=bad)
    lay = ML1Layer(8, 16)
    # CPU tensors: the precision is checked before the device check (and before any library call)
    with pytest.raises(ValueError, match="precision must be one of"):
        ml1_layer(torch.zeros(4, 8), torch.zeros(2, 0, dtype=torch.int64), lay.conv1, lay.fc11, lay.fc12, lay.fc13, precision=bad)


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_layer_and_model_accept_every_precision(precision):
    from gnn_matlang_b200.libs.spect_conv import ML1Layer
    from gnn_matlang_b200.models import GNNML1
    assert ML1Layer(8, 16, concat=True, precision=precision).precision == precision
    assert GNNML1("graph8c", 1, concat=True, precision=precision).precision == precision


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("cfg,ninp,concat", [("zinc", 25, False), ("graph8c", 1, True)])
def test_model_parameters_do_not_depend_on_the_precision(precision, cfg, ninp, concat):
    from gnn_matlang_b200.models import GNNML1
    torch.manual_seed(0)
    ref = GNNML1(cfg, ninp, concat=concat)
    torch.manual_seed(0)
    m = GNNML1(cfg, ninp, concat=concat, precision=precision)
    a, b = ref.state_dict(), m.state_dict()
    assert list(a) == list(b)
    for k in a:
        assert a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k
    assert [n for n, _ in ref.named_parameters()] == [n for n, _ in m.named_parameters()]
