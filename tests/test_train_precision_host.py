"""CPU: the training-precision switch (``DGNBase.set_train_precision``) and the input checks of the CUDA training Functions,
which must refuse what they cannot read before the library is loaded or any kernel launched."""
import pytest
import torch

DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})


def _net(kind="l_dgn", **kw):
    from melissa_b200.networks import NETWORKS
    return NETWORKS[kind](5, 128, 2, 4, 12, dueling_param=DUELING(), device="cpu", **kw)


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"})])
def test_set_train_precision_values_clone_and_state_dict(kind, kw):
    net = _net(kind, **kw)
    keys = sorted(net.state_dict())
    assert net.train_precision == "fp32"
    assert net.set_train_precision("bf16") is net and net.train_precision == "bf16"
    assert net.precision == "fp32"                          # the rollout precision is a separate switch
    assert sorted(net.state_dict()) == keys
    assert net.clone_for_target().train_precision == "bf16"
    net.set_precision("bf16")
    net.set_train_precision("fp32")
    assert (net.precision, net.train_precision) == ("bf16", "fp32")
    assert net.clone_for_target().train_precision == "fp32"
    for bad in ("bf16 ", "BF16", "fp16", "tf32", None):
        with pytest.raises(ValueError):
            net.set_train_precision(bad)
    assert net.train_precision == "fp32"


def test_bf16_training_precision_on_cpu_parameters_raises():
    from melissa_b200._lib import MelissaLibraryError
    from melissa_b200.networks.autograd import q_values
    from test_training_host import _rows
    net = _net().set_train_precision("bf16")
    with pytest.raises(MelissaLibraryError, match="set_train_precision"):
        q_values(net, _rows(12, 4, 1))


@pytest.fixture
def no_library(monkeypatch):
    """Loading the library (or launching through it) fails the test: the checks must come first."""
    from melissa_b200 import _lib

    def refuse():
        raise AssertionError("the library was loaded before the input check")
    monkeypatch.setattr(_lib, "lib", refuse)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
def test_training_functions_reject_inputs_they_cannot_read(no_library, dtype):
    """Half-precision tensors (what the dense layers return under torch.autocast) and CPU tensors of any dtype."""
    from melissa_b200._lib import MelissaLibraryError
    from melissa_b200.networks.autograd import _GATv2Edge, _LinearBF16, _TransformerEdge
    t, hc = 6, 128
    lists = (torch.zeros(t, dtype=torch.int32), torch.zeros(t, 40, dtype=torch.int32), torch.ones(t, dtype=torch.int32))
    x = torch.zeros(t, hc, dtype=dtype)
    att = torch.zeros(hc)
    with pytest.raises(MelissaLibraryError, match=r'set_train_precision\("bf16"\)'):
        _GATv2Edge.apply(x, x, att, *lists)
    with pytest.raises(MelissaLibraryError, match=r'set_train_precision\("bf16"\)'):
        _TransformerEdge.apply(x, x, x, *lists)
    lin = torch.nn.Linear(hc, 64)
    with pytest.raises(MelissaLibraryError, match=r'set_train_precision\("bf16"\)'):
        _LinearBF16.apply(x, lin.weight, lin.bias)
    with pytest.raises(MelissaLibraryError, match=r'set_train_precision\("bf16"\)'):
        _LinearBF16.apply(x, lin.weight.to(dtype), None)
