"""QMixMixer at qmix_hidden_dim != 32: the reference's modules at any E in 1..128 and the flat layout the kernels read."""
import pytest
import torch

from marl_b200.network.mixer import QMixMixer, hy_cols
from tests import parity_util as PU


def _args(E, N=5, S=7, **kw):
    return PU.make_args("qmix", N, 4, 6, S, 10, qmix_hidden_dim=E, **kw)


@pytest.mark.parametrize("E", [1, 16, 64, 128])
@pytest.mark.parametrize("two_hyper_layers", [False, True])
def test_module_names_and_shapes(E, two_hyper_layers):
    N, S, hh = 5, 7, 16
    m = QMixMixer(_args(E, N, S, two_hyper_layers=two_hyper_layers, hyper_hidden_dim=hh))
    got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    want = {"hyper_b1.weight": (E, S), "hyper_b1.bias": (E,), "hyper_b2.0.weight": (E, S), "hyper_b2.0.bias": (E,),
            "hyper_b2.2.weight": (1, E), "hyper_b2.2.bias": (1,)}
    if two_hyper_layers:
        want.update({"hyper_w1.0.weight": (hh, S), "hyper_w1.0.bias": (hh,), "hyper_w1.2.weight": (N * E, hh),
                     "hyper_w1.2.bias": (N * E,), "hyper_w2.0.weight": (hh, S), "hyper_w2.0.bias": (hh,),
                     "hyper_w2.2.weight": (E, hh), "hyper_w2.2.bias": (E,)})
    else:
        want.update({"hyper_w1.weight": (N * E, S), "hyper_w1.bias": (N * E,), "hyper_w2.weight": (E, S),
                     "hyper_w2.bias": (E,)})
    assert got == want


@pytest.mark.parametrize("E,N,S", [(1, 2, 3), (7, 2, 5), (16, 5, 7), (33, 3, 1), (64, 27, 9), (128, 5, 120)])
def test_flat_layout_is_one_wcat_matrix(E, N, S):
    """The four state-conditioned heads are one [N*E + 3E, S] matrix and their biases one [N*E + 3E] vector in the flat
    buffer, whatever E (odd widths included): the hyper-network GEMM reads them that way."""
    m = QMixMixer(_args(E, N, S))
    fl, C = m._flat, hy_cols(N, E)
    w0, b0 = fl.offsets["hyper_w1.weight"], fl.offsets["hyper_w1.bias"]
    assert w0 % 4 == 0 and b0 % 4 == 0
    wcat = fl.data[w0:w0 + C * S].view(C, S)
    bcat = fl.data[b0:b0 + C]
    heads = ("hyper_w1", "hyper_b1", "hyper_w2", "hyper_b2.0")
    sd = m.state_dict()
    assert torch.equal(wcat, torch.cat([sd[h + ".weight"] for h in heads]))
    assert torch.equal(bcat, torch.cat([sd[h + ".bias"] for h in heads]))
    for name, p in m.named_parameters():                      # the module's parameters are views of that storage
        assert p.data_ptr() == fl.data.data_ptr() + 4 * fl.offsets[name], name


@pytest.mark.parametrize("E", [0, 129, -3])
def test_out_of_range_width_is_rejected(E):
    with pytest.raises(ValueError, match="1..128"):
        QMixMixer(_args(E))
