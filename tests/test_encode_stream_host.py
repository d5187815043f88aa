"""Host-side checks of the streaming encoder: the receptive field ``encoder_context_samples`` derives from the
constructor arguments against the float64 CPU oracle, and the argument checks that need no GPU."""
import pytest
import torch

import helpers as H
import kalle_audio_b200 as k
from oracle import oobleck_oracle as O


def _encoder_sd(case):
    if case == "even_strides":
        torch.manual_seed(3)
        enc = k.OobleckEncoder(in_channels=2, channels=8, latent_dim=8, c_mults=[1, 2], strides=[2, 4], use_snake=True)
        return enc.state_dict(), [2, 4]
    m = H.build(case, 0, snake_seed=7)
    return m.encoder.state_dict(), list(H.strides_of(case))


@pytest.mark.parametrize("case", ["tiny", "tiny_sym", "even_strides"])
def test_context_is_the_exact_dependency(case):
    """A NaN at input sample x reaches every frame that reads x, however small the path's weights.  Over 2 * ratio
    consecutive positions (every phase of every stride), the farthest frame reached on each side is exactly
    ``encoder_context_samples`` away: the bound is tight, not just safe."""
    sd, strides = _encoder_sd(case)
    sd = {n: v.detach().double() for n, v in sd.items()}
    ratio = 1
    for s in strides:
        ratio *= s
    left, right = k.encoder_context_samples(strides)
    T = ratio * max(64, 4 * ((left + right) // ratio + 4))
    x = torch.randn(1, 2, T, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    base = T // 2 - ratio
    got_right = got_left = -10 ** 9
    for pos in range(base, base + 2 * ratio):
        xp = x.clone()
        xp[..., pos] = float("nan")
        frames = torch.isnan(O.oobleck_encoder(sd, xp, strides)).any(dim=1).flatten().nonzero().flatten()
        f_first, f_last = int(frames.min()), int(frames.max())
        assert f_first > 0 and f_last < T // ratio - 1, "the NaN reached the clip edge: make T longer"
        got_right = max(got_right, pos - ((f_first + 1) * ratio - 1))   # past the first reached frame's last sample
        got_left = max(got_left, f_last * ratio - pos)                  # before the last reached frame's first sample
    assert (got_left, got_right) == (left, right)


def test_context_of_the_shipped_strides():
    assert k.encoder_context_samples([2, 4, 4, 8, 8]) == (14885, 14885)   # SAO: 7.27 frames, 0.34 s at 44.1 kHz
    assert k.encoder_context_samples([2, 4, 4, 5, 8])[1] == 9925          # 12.5 Hz models: 7.75 frames, 0.62 s at 16 kHz
    assert k.encoder_context_samples([2, 4, 5])[1] == 493


def test_streaming_encoder_wraps_encoders_only():
    dec = k.OobleckDecoder(out_channels=2, channels=8, latent_dim=8, c_mults=[1, 2], strides=[2, 4], use_snake=True)
    with pytest.raises(TypeError):
        k.StreamingEncoder(dec)
    enc = k.OobleckEncoder(in_channels=2, channels=8, latent_dim=8, c_mults=[1, 2], strides=[2, 4], use_snake=True)
    se = k.StreamingEncoder(enc)
    assert se.ratio == 8 and se.lookahead is None
    with pytest.raises(ValueError):
        se.flush()
