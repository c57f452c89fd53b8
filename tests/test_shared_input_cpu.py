"""The shared controller's input blocks without a GPU: SharedMAC's input width for the four (last_action, reuse_network)
compositions (share_params.py:114-123), and the oracle's shared unroll without the last-action block pinned against the
UNMODIFIED reference's SharedMAC.get_current_q_values / get_next_q_values when it is staged in oracle/_ref
(oracle/fetch_ref.py)."""
import numpy as np
import pytest
import torch

from marl_b200.common.arguments import default_args
from marl_b200.synthetic import synthetic_batch
from oracle import fetch_ref as FR
from oracle import marl_oracle as MO


@pytest.mark.parametrize("last_action,reuse_network", [(True, True), (True, False), (False, True), (False, False)])
def test_shared_mac_input_shape(last_action, reuse_network):
    from marl_b200.controller.share_params import SharedMAC
    N, A, O = 5, 11, 80
    args = default_args(n_agents=N, n_actions=A, obs_shape=O, state_shape=120, episode_limit=30,
                        last_action=last_action, reuse_network=reuse_network)
    mac = SharedMAC(args)
    want = O + (A if last_action else 0) + (N if reuse_network else 0)
    assert mac._get_input_shape() == want
    assert tuple(mac.agent.state_dict()["fc1.weight"].shape) == (64, want)


@pytest.mark.skipif(not FR.available(), reason="reference not staged in oracle/_ref")
@pytest.mark.parametrize("reuse_network", [True, False])
def test_oracle_shared_unroll_without_last_action_matches_reference(reuse_network):
    """get_current_q_values, then get_next_q_values continuing from the carried hidden state (q_learner.py:96,110), of the
    reference's SharedMAC with last_action=False against MO.unroll on the same weights."""
    ref = FR.load()
    N, A, O, S, T, B = 3, 5, 7, 4, 8, 6
    args = FR.make_args(ref, "qmix", N, A, O, S, T, last_action=False, reuse_network=reuse_network)
    torch.manual_seed(0)
    mac = ref.SharedMAC(args)
    p = {k: v.detach().clone() for k, v in mac.agent.state_dict().items()}
    assert tuple(p["fc1.weight"].shape) == (64, O + (N if reuse_network else 0))
    batch = synthetic_batch(3, B, T, N, A, O, S)
    b = {k: torch.tensor(v, dtype=torch.long if k == "u" else torch.float32) for k, v in batch.items()}
    with torch.no_grad():
        mac.init_hidden(B)
        q_cur = mac.get_current_q_values(b, T)[0]
        q_next = mac.get_next_q_values(b, T)[0]
        cfg = MO.make_cfg(n_agents=N, n_actions=A, obs_shape=O, last_action=False, reuse_network=reuse_network)
        oq, _, hl = MO.unroll(p, b["o"], MO.shift_onehot(b["u_onehot"]), torch.zeros(B * N, 64), cfg)
        oq2, _, _ = MO.unroll(p, b["o_next"], b["u_onehot"], hl, cfg)
    assert np.allclose(q_cur.numpy(), oq.numpy(), rtol=0, atol=1e-5 * float(oq.abs().max()))
    assert np.allclose(q_next.numpy(), oq2.numpy(), rtol=0, atol=1e-5 * float(oq2.abs().max()))
