"""kalle_audio_b200 -- B200-native (sm_100a) implementation of kalle-audio's sigmaVAE / Oobleck
autoencoder hot path, as a drop-in for the reference's module surface.

    from kalle_audio_b200 import create_autoencoder_from_config, sample
    ae = create_autoencoder_from_config(model_config).cuda().eval()
    wav = ae.decode(latents)

Every compute call goes through libkvae.so (C ABI in include/kvae.h); there is no CPU or eager fallback.
"""
from . import _lib
from ._lib import KvaeError, LIB_PATH
from .autoencoders import (AudioAutoencoder, DecoderBlock, EncoderBlock, OobleckDecoder, OobleckEncoder,
                           ResidualUnit, create_autoencoder_from_config, create_decoder_from_config,
                           create_encoder_from_config, get_activation)
from .bottleneck import Bottleneck, VAEBottleneck, create_bottleneck_from_config, vae_sample
from .factory import create_model_from_config, create_model_from_config_path, create_pretransform_from_config
from .layers import SnakeBeta, WNConv1d, WNConvTranspose1d, snake_beta
from .pretransforms import AutoencoderPretransform, Pretransform
from .sampling import SigmaVAESampler, sample
from .streaming import StreamingDecoder, decoder_context_frames
from .hostio import HostPipeline
from .glue import LatentGlue
from .dataset import LatentExtractor
from .bigvgan import BigVGANFlowVAE
from .bigvgan_stream import BigVGANStreamingDecoder, bigvgan_stream_geometry
from .losses import MultiResolutionSTFTLoss, SumAndDifferenceSTFTLoss, aw_fir_taps
from .discriminators import OobleckDiscriminator, get_hinge_losses
from .utils import load_ckpt_state_dict, prepare_audio, remove_weight_norm_from_model, to_pcm16
from .training import AutoencoderTrainer, FlatAdamW, GradSync, flatten_parameters, gaussian_nll, vae_sample_with_grad

__all__ = [
    "MultiResolutionSTFTLoss", "SumAndDifferenceSTFTLoss", "aw_fir_taps", "OobleckDiscriminator", "get_hinge_losses",
    "AudioAutoencoder", "AutoencoderPretransform", "Bottleneck", "DecoderBlock", "EncoderBlock", "KvaeError",
    "OobleckDecoder", "OobleckEncoder", "Pretransform", "ResidualUnit", "SigmaVAESampler", "SnakeBeta",
    "VAEBottleneck", "WNConv1d", "WNConvTranspose1d", "create_autoencoder_from_config",
    "create_bottleneck_from_config", "create_decoder_from_config", "create_encoder_from_config",
    "create_model_from_config", "create_model_from_config_path", "create_pretransform_from_config",
    "get_activation", "load_ckpt_state_dict", "prepare_audio", "remove_weight_norm_from_model", "sample",
    "snake_beta", "vae_sample", "to_pcm16", "AutoencoderTrainer", "FlatAdamW", "GradSync", "flatten_parameters",
    "gaussian_nll", "vae_sample_with_grad", "StreamingDecoder", "decoder_context_frames", "HostPipeline", "LatentGlue", "LatentExtractor", "BigVGANFlowVAE",
    "BigVGANStreamingDecoder", "bigvgan_stream_geometry",
]
