"""The agent stride the fused step hands the library for one network per agent (q_learner.separated_stride): host logic."""
import pytest
import torch

from marl_b200.algorithm.q_learner import separated_stride
from marl_b200.flat import FlatBuffer, prefixed
from marl_b200.network.q_network import RNNQNet
from tests import parity_util as PU


def _agents(N, I=13):
    args = PU.make_args("vdn", N, 5, 7, 9, 10)
    return [RNNQNet(I, args) for _ in range(N)]


def _flat(named):
    return FlatBuffer(named, device=torch.device("cpu"), with_grad=False)


@pytest.mark.parametrize("N", [1, 2, 7])
def test_stride_is_one_agent_set(N):
    nets = _agents(N)
    named = []
    for i, net in enumerate(nets):
        named += prefixed(f"agent.{i}.", net.flat_named_parameters())
    flat = _flat(named + [("mixer.w", torch.zeros(3))])
    stride = separated_stride(flat, N)
    assert stride > 0 and stride % 4 == 0
    assert stride >= sum(p.numel() for _, p in nets[0].flat_named_parameters())
    for i in range(N):
        for name, _ in nets[i].flat_named_parameters():
            assert flat.offsets[f"agent.{i}.{name}"] == flat.offsets[f"agent.0.{name}"] + i * stride


def test_uneven_agent_sets_are_rejected():
    nets = _agents(3)
    named = prefixed("agent.0.", nets[0].flat_named_parameters()) + [("gap", torch.zeros(8))]     # agent 1 sits 8 floats further
    named += prefixed("agent.1.", nets[1].flat_named_parameters()) + prefixed("agent.2.", nets[2].flat_named_parameters())
    with pytest.raises(ValueError):
        separated_stride(_flat(named), 3)
