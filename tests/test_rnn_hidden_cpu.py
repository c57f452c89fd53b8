"""rnn_hidden_dim on the host: module names and shapes at every supported width, the range errors, the flat layout at the
default width, and the separated stride at every width."""
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.flat import FlatBuffer
from oracle import marl_oracle as MO
from tests import parity_util as PU

WIDTHS = (32, 64, 128)


def _args(H, alg="qmix", **kw):
    return PU.make_args(alg, 3, 4, 5, 6, 8, rnn_hidden_dim=H, **kw)


@pytest.mark.parametrize("H", WIDTHS)
def test_agent_modules_have_the_reference_names_and_shapes(H):
    from marl_b200.network.q_network import RNNQNet
    args = _args(H)
    I = 5 + 4 + 3
    net = RNNQNet(I, args)
    got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    want = {k: tuple(v.shape) for k, v in MO.init_agent(MO.make_cfg(n_agents=3, n_actions=4, obs_shape=5,
                                                                     rnn_hidden_dim=H)).items()}
    assert got == want
    assert got["rnn.weight_hh"] == (3 * H, H) and got["fc1.weight"] == (H, I) and got["fc2.weight"] == (4, H)
    assert net.param_struct().hidden == H


@pytest.mark.parametrize("H", WIDTHS)
def test_qtran_modules_follow_the_width(H):
    from marl_b200.network.qtran import QtranQBase, QtranV
    args = _args(H, "qtran_base")
    q, v = QtranQBase(args), QtranV(args)
    assert tuple(q.state_dict()["hidden_action_encoding.0.weight"].shape) == (H + 4, H + 4)
    assert tuple(q.state_dict()["q.0.weight"].shape) == (args.qtran_hidden_dim, 6 + 4 + H)
    assert tuple(v.state_dict()["hidden_encoding.0.weight"].shape) == (H, H)
    assert tuple(v.state_dict()["v.0.weight"].shape) == (args.qtran_hidden_dim, 6 + H)


@pytest.mark.parametrize("H", [0, 16, 48, 96, 256])
def test_unsupported_widths_raise(H):
    from marl_b200.network.q_network import RNNQNet
    from marl_b200.network.qtran import QtranQBase, QtranV
    from marl_b200.controller.share_params import SharedMAC, SeparatedMAC
    args = _args(H, "qtran_base")
    for build in (lambda: RNNQNet(12, args), lambda: QtranQBase(args), lambda: QtranV(args), lambda: SharedMAC(args),
                  lambda: SeparatedMAC(_args(H, reuse_network=False))):
        with pytest.raises(ValueError, match="rnn_hidden_dim"):
            build()


def test_flat_layout_at_64_is_unchanged():
    """Offsets of the agent's parameters in its flat buffer at the default width: the layout every earlier release used."""
    from marl_b200.network.q_network import RNNQNet
    net = RNNQNet(12, _args(64))
    flat = FlatBuffer(net.flat_named_parameters(), device="cpu", with_grad=False)
    sizes = [64 * 12, 64, 192 * 64, 192 * 64, 192, 192, 4 * 64, 4]
    off, want = 0, {}
    for (name, _), n in zip(net.flat_named_parameters(), sizes):
        want[name] = flat.offsets[name]
        assert flat.view(name).numel() == n
    assert list(want.values()) == sorted(want.values())
    assert [n for n, _ in net.flat_named_parameters()] == ["fc1.weight", "fc1.bias", "rnn.weight_ih", "rnn.weight_hh",
                                                           "rnn.bias_ih", "rnn.bias_hh", "fc2.weight", "fc2.bias"]


@pytest.mark.parametrize("H", WIDTHS)
def test_separated_stride_is_a_multiple_of_4(H):
    from marl_b200.algorithm.q_learner import separated_stride
    from marl_b200.network.q_network import RNNQNet
    args = _args(H)
    nets = [RNNQNet(9, args) for _ in range(3)]
    named = [(f"agent.{n}.{k}", p) for n, net in enumerate(nets) for k, p in net.flat_named_parameters()]
    flat = FlatBuffer(named, device="cpu", with_grad=False)
    stride = separated_stride(flat, 3)
    assert stride > 0 and stride % 4 == 0
    assert stride >= sum(p.numel() for _, p in nets[0].flat_named_parameters())


def test_struct_builders_carry_the_width():
    from marl_b200.network.q_network import agent_param_struct, AGENT_FLAT_ORDER
    from marl_b200.network.qtran import net_struct
    named = {n: 0 for n in AGENT_FLAT_ORDER}
    assert agent_param_struct(named, hidden=128).hidden == 128
    assert net_struct([0] * 10, hidden=32).hidden == 32
    assert L.AgentParams().hidden == 0 and L.QtranNetParams().hidden == 0      # zero-initialised: the default width
