"""Host-side checks of BigVGANFlowVAE's flow (the VITS ResidualCouplingBlock), without a GPU:

  * a seeded BigVGANFlowVAE(BIGVGAN_H) builds flow.* in the reference's order (WN layers interleaved, ``post``
    zeroed), so all 112 flow tensors equal the reference's own module recorded in tests/golden/bigvgan.npz, and every
    tensor outside the flow keeps the value the parameter-container layout gave it;
  * the state-dict keys of the whole model are the golden's;
  * the float64 restatement (flow_oracle.py) inverts itself: reverse(forward(x)) = x mask to 1e-12 with an all-ones
    mask and per-clip prefix masks, with ``post`` randomised (a zero ``post`` makes the flow an identity);
  * the flow kernels' argument checks refuse bad calls before any device access."""
import os
import sys

import numpy as np
import pytest
import torch

import helpers  # noqa: F401  (sys.path)
import flow_oracle as FO
from kalle_audio_b200 import _lib
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.layers import WNConv1d

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bigvgan.npz")


class AttrDict(dict):
    __getattr__ = dict.__getitem__


def _golden_sd():
    z = np.load(GOLDEN)
    return {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}


def _model(h=BIGVGAN_H, seed=0):
    torch.manual_seed(seed)
    return BV.BigVGANFlowVAE(AttrDict(h, causal=True))


def test_seeded_flow_equals_golden():
    g = _golden_sd()
    sd = _model().state_dict()
    keys = [k for k in g if k.startswith("flow.")]
    assert len(keys) == 112
    for k in keys:
        assert torch.equal(sd[k], g[k].to(sd[k].dtype)), k
    assert all(not sd[k].any() for k in keys if ".post." in k)        # mean_only: post zeroed


def test_state_dict_keys_unchanged():
    g = _golden_sd()
    sd = _model().state_dict()
    assert list(k for k in sd if k.startswith("flow.")) == [k for k in g if k.startswith("flow.")]
    assert set(sd) == set(g)


class _ParamContainerLayout(torch.nn.Module):
    """The flow's parameter container before the flow ran: all in_layers first, then all res_skip_layers (no
    padding), plain nn.Conv1d pre / post, post left random.  Same number of RNG draws per tensor."""

    def __init__(self, channels, hidden, k, n_layers, n_flows=4):
        super().__init__()
        self.flows = torch.nn.ModuleList()
        for _ in range(n_flows):
            lay = torch.nn.Module()
            lay.pre = torch.nn.Conv1d(channels // 2, hidden, 1)
            lay.enc = torch.nn.Module()
            lay.enc.in_layers = torch.nn.ModuleList([WNConv1d(hidden, 2 * hidden, k) for _ in range(n_layers)])
            lay.enc.res_skip_layers = torch.nn.ModuleList(
                [WNConv1d(hidden, 2 * hidden if i < n_layers - 1 else hidden, 1) for i in range(n_layers)])
            lay.post = torch.nn.Conv1d(hidden, channels // 2, 1)
            self.flows.append(lay)
            self.flows.append(torch.nn.Module())


def test_non_flow_parameters_keep_their_seeded_values(monkeypatch):
    new = _model().state_dict()
    monkeypatch.setattr(BV, "ResidualCouplingBlock",
                        lambda c, hid, k, d, n: _ParamContainerLayout(c, hid, k, n))
    old = _model().state_dict()
    assert set(old) == set(new)
    other = [k for k in new if not k.startswith("flow.")]
    assert other and all(torch.equal(old[k], new[k]) for k in other)


def _randomised_sd(seed=3):
    sd = {k: v.double() for k, v in _golden_sd().items()}
    gen = torch.Generator().manual_seed(seed)
    for k in sd:
        if k.startswith("flow.") and ".post." in k:
            sd[k] = 0.3 * torch.randn(sd[k].shape, dtype=torch.float64, generator=gen)
    return sd


@pytest.mark.parametrize("masks", ["ones", "prefix"])
def test_oracle_inverts_itself(masks):
    sd = _randomised_sd()
    B, C, T = 3, BIGVGAN_H["latent_dim"], 37
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(B, C, T, dtype=torch.float64, generator=gen)
    lens = [T] * B if masks == "ones" else [T, 20, 1]
    mask = torch.zeros(B, 1, T, dtype=torch.float64)
    for b, n in enumerate(lens):
        mask[b, :, :n] = 1
    z = FO.flow(sd, BIGVGAN_H, x, mask)
    assert float((z - x * mask).abs().max()) > 1e-2                  # not an identity: post is random
    assert not z[mask.expand_as(z) == 0].any()                       # masked frames come out 0
    back = FO.flow(sd, BIGVGAN_H, z, mask, reverse=True)
    assert float((back - x * mask).abs().max()) <= 1e-12


def test_flow_kernel_argument_checks():
    L = _lib.lib()
    p = 16                # placeholder pointer, never dereferenced: every call below fails its checks first
    assert L.kvae_flow_split(p, p, p, 1, 7, 10, 0, 0, None) != 0
    assert b"odd" in L.kvae_last_error()
    assert L.kvae_flow_mask(p, p, p, 1, 4, 10, 5, None) != 0
    assert b"dtype" in L.kvae_last_error()
    assert L.kvae_wn_gate_fwd(p, p, 0, 4, 10, 0, None) != 0
    assert b"empty" in L.kvae_last_error()
    assert L.kvae_wn_update_fwd(p, p, None, p, None, p, 1, 4, 0, 10, 0, None) != 0      # x_out missing
    assert b"null" in L.kvae_last_error()
    assert L.kvae_flow_coupling_fwd(p, p, p, p, None, 1024, 128, 10, 1, 0, 0, None) != 0
    assert b"too large" in L.kvae_last_error()
    assert L.kvae_flow_coupling_bwd(None, None, p, None, p, 1, 4, 10, 1, 0, 0, None) != 0
    assert b"null" in L.kvae_last_error()


def test_constructor_refusals():
    with pytest.raises(NotImplementedError):
        BV.ResidualCouplingBlock(16, 8, 5, 1, 4, gin_channels=4)
    with pytest.raises(NotImplementedError):
        BV.ResidualCouplingLayer(16, 8, 5, 1, 4, mean_only=False)
    blk = BV.ResidualCouplingBlock(16, 8, 5, 2, 3)
    assert [m.dilation[0] for m in blk.flows[0].enc.in_layers] == [1, 2, 4]
    assert [m.padding[0] for m in blk.flows[0].enc.in_layers] == [2, 4, 8]
    assert [type(f).__name__ for f in blk.flows] == ["ResidualCouplingLayer", "Flip"] * 4
