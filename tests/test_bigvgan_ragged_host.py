"""Host-side checks of BigVGANFlowVAE's ragged batches: the per-clip output lengths (``latent_length`` / ``wav_length``,
pure host arithmetic over the layer descriptions) against the float64 oracle, and the longest-first ordering and
tensor-core split that the ragged path applies."""
import os
import sys

import pytest
import torch

import helpers  # noqa: F401  (sys.path)
from kalle_audio_b200 import bigvgan as BV
from oracle import bigvgan_oracle as BO

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


BENCH_GEOMETRY = dict(BIGVGAN_H, causal=True, latent_dim=8, resblock_kernel_sizes=[3, 7, 11],
                      resblock_dilation_sizes=[[1, 3, 5]] * 3, upsample_rates=[8, 5, 4, 2, 2, 2],
                      upsample_kernel_sizes=[16, 10, 8, 4, 4, 4], upsample_initial_channel=64, resblock="1",
                      activation="snakebeta", snake_logscale=True)
CONFIGS = {"golden_causal": dict(BIGVGAN_H, causal=True), "golden_noncausal": dict(BIGVGAN_H, causal=False),
           "bench_geometry": BENCH_GEOMETRY}


def _model(h):
    torch.manual_seed(0)
    m = BV.BigVGANFlowVAE(AttrDict(h))
    return m, {n: p.detach().double() for n, p in m.state_dict().items()}


@pytest.mark.parametrize("tag", ["golden_causal", "golden_noncausal"])
def test_latent_length_matches_oracle(tag):
    h = CONFIGS[tag]
    m, sd = _model(h)
    shortest = min(n for n in range(1, 64) if m.latent_length(n) > 0)
    for n in sorted({shortest, shortest + 1, 9, 15, 16, 17, 31, 8 * 12 + 5, 8 * 37}):
        x = torch.randn(1, 1, n, dtype=torch.float64, generator=torch.Generator().manual_seed(n))
        assert m.latent_length(n) == BO.extract_latents(sd, h, x).shape[2], n
    for n in range(1, shortest):                      # too short: the reference's own convs refuse the clip
        with pytest.raises(RuntimeError):
            BO.extract_latents(sd, h, torch.zeros(1, 1, n, dtype=torch.float64))
        assert m.latent_length(n) == 0
    assert m.latent_length(8 * 37) == 37 and m.latent_length(8 * 37 + 7) == 38     # floors, not n // ratio


@pytest.mark.parametrize("tag", list(CONFIGS))
def test_wav_length_matches_oracle(tag):
    h = CONFIGS[tag]
    m, sd = _model(h)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)            # the oracle's anti-aliasing filters follow the default dtype
    try:
        for n in (1, 2, 3, 7) if tag == "bench_geometry" else (1, 2, 3, 7, 30):
            z = torch.randn(1, h["latent_dim"], n, generator=torch.Generator().manual_seed(n))
            assert m.wav_length(n) == BO.inference_from_latents(sd, h, z).shape[2], n
    finally:
        torch.set_default_dtype(prev)


def test_ragged_order_and_inverse():
    lens = [5, 9, 1, 9, 7, 5]
    order, inverse = BV.ragged_order(lens)
    assert order == [1, 3, 4, 0, 5, 2]                # longest first, ties in index order
    assert [lens[b] for b in order] == sorted(lens, reverse=True)
    assert [order[i] for i in inverse] == list(range(len(lens)))
    sorted_batch = torch.tensor(lens)[order]
    assert torch.equal(sorted_batch[inverse], torch.tensor(lens))
    assert BV.ragged_order([3]) == ([0], [0])


def test_tc_split_is_a_prefix_at_the_row_threshold():
    assert BV.TC_MIN_ROWS == 64
    assert BV.tc_split([500, 64, 63, 1]) == 2
    assert BV.tc_split([64, 64]) == 2
    assert BV.tc_split([63, 2]) == 0
    with pytest.raises(ValueError):
        BV.tc_split([63, 64])


def test_valid_len_checks():
    m, _ = _model(CONFIGS["golden_causal"])
    ok = BV._check_valid_len(torch.tensor([296, 7]), 2, 296, m.latent_length, "t")
    assert ok == [296, 7]
    for bad in ([296], [0, 10], [297, 10], [296, 3]):  # wrong count, 0, past the padded length, no latent frame
        with pytest.raises(ValueError):
            BV._check_valid_len(bad, 2, 296, m.latent_length, "t")
    with pytest.raises(ValueError):
        BV._check_valid_len([1] * 65, 65, 4, m.wav_length, "t")
