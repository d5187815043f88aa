"""Host-side check of BigVGANFlowVAE's op lists (``bigvgan._program`` / ``_encoder_program``): every conv and transposed
conv op carries the geometry of the module it names, and the two lists name every conv of the model's inference path.
The streams, the ragged calls and the length helpers all read that geometry, so a list that drifts from the module tree
fails here instead of as a stream that no longer equals the whole call."""
import os
import sys

import pytest
import torch

import helpers  # noqa: F401  (sys.path)
from kalle_audio_b200 import bigvgan as BV
from kalle_audio_b200.layers import WNConv1d, WNConvTranspose1d

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden import BIGVGAN_H  # noqa: E402


class AttrDict(dict):
    __getattr__ = dict.__getitem__


# bench.py's BigVGAN geometry (decoder rates 8/5/4/2/2/2, AMPBlock1 k 3/7/11; encoder rates 2/2/4/4/4/5) with few
# channels: the geometry does not depend on the widths
BENCH_GEOMETRY = dict(BIGVGAN_H, latent_dim=8, resblock_kernel_sizes=[3, 7, 11], resblock_dilation_sizes=[[1, 3, 5]] * 3,
                      upsample_rates=[8, 5, 4, 2, 2, 2], upsample_kernel_sizes=[16, 10, 8, 4, 4, 4],
                      upsample_initial_channel=64, resblock="1", activation="snakebeta", snake_logscale=True,
                      downsample_channels=[12] + [4] * 6, downsample_rates=[2, 2, 4, 4, 4, 5])
CONFIGS = {"golden": BIGVGAN_H, "bench_geometry": BENCH_GEOMETRY}


@pytest.mark.parametrize("causal", [True, False], ids=["causal", "noncausal"])
@pytest.mark.parametrize("tag", list(CONFIGS))
def test_conv_ops_carry_their_modules_geometry(tag, causal):
    h = dict(CONFIGS[tag], causal=causal)
    m = BV.BigVGANFlowVAE(AttrDict(h))
    named = set()
    for encoder, program in ((False, BV._program), (True, BV._encoder_program)):
        ops, _ = program(h)
        for op in ops:
            if op.kind not in ("conv", "convT"):
                continue
            mod, g = BV._module(m, op.module), op.geom
            assert mod.transposed == (op.kind == "convT"), op.module
            assert (mod.kernel_size[0], mod.dilation[0], mod.stride[0]) == (g.K, g.d, g.s), op.module
            assert mod.padding[0] == (g.pl if op.kind == "conv" else g.p), op.module
            assert getattr(mod, "causal", False) == g.causal, op.module     # the encoder's convs have no attribute
            assert hasattr(mod, "causal") != encoder, op.module
            named.add(op.module)
    convs = {n for n, x in m.named_modules() if isinstance(x, (WNConv1d, WNConvTranspose1d))}
    assert named == {n for n in convs if not n.startswith("flow.")}
