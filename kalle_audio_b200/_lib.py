"""ctypes binding of libkvae.so (C ABI declared in include/kvae.h).

There is deliberately no fallback: if the shared library is missing, or no sm_100 device is
visible, every compute call raises.  PyTorch is used above this layer only for device memory,
streams and torch.distributed plumbing.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# KVAE_LIB: development override (A/B builds of the same sources); there is still no non-CUDA fallback
LIB_PATH = os.environ.get("KVAE_LIB") or os.path.join(_HERE, "libkvae.so")

KVAE_F32, KVAE_BF16 = 0, 1
KVAE_ENCODER, KVAE_DECODER = 0, 1
KVAE_PREC_BF16, KVAE_PREC_F32 = 0, 1
KVAE_MAX_STAGES = 8


class KvaeArch(C.Structure):
    _fields_ = [
        ("io_channels", C.c_int),
        ("channels", C.c_int),
        ("latent_dim", C.c_int),
        ("n_stages", C.c_int),
        ("c_mults", C.c_int * KVAE_MAX_STAGES),
        ("strides", C.c_int * KVAE_MAX_STAGES),
        ("final_tanh", C.c_int),
        ("use_nearest_upsample", C.c_int),
    ]


class KvaeError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None

# name -> (restype, argtypes); also the list tests/test_abi.py checks against include/kvae.h
SIGNATURES = {
    "kvae_version": (C.c_int, []),
    "kvae_last_error": (C.c_char_p, []),
    "kvae_device_count": (C.c_int, []),
    "kvae_launch_count": (C.c_longlong, [C.c_int]),
    "kvae_plan_create": (C.c_int, [C.POINTER(KvaeArch), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "kvae_plan_destroy": (None, [C.c_void_p]),
    "kvae_plan_num_convs": (C.c_int, [C.c_void_p]),
    "kvae_plan_num_snakes": (C.c_int, [C.c_void_p]),
    "kvae_plan_conv_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int * 8)]),
    "kvae_plan_snake_channels": (C.c_int, [C.c_void_p, C.c_int]),
    "kvae_plan_set_conv": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "kvae_plan_set_snake": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "kvae_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_longlong]),
    "kvae_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_decode_ragged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                     C.POINTER(C.c_int), C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_encode_ragged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                     C.POINTER(C.c_int), C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_decode_stream_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "kvae_decode_stream_samples": (C.c_longlong, [C.c_void_p, C.c_int, C.c_int]),
    "kvae_decode_stream_lookahead": (C.c_longlong, [C.c_void_p]),
    "kvae_decode_stream_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_longlong,
                                          C.POINTER(C.c_longlong), C.c_void_p]),
    "kvae_decode_stream_end": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.POINTER(C.c_longlong),
                                         C.c_void_p]),
    "kvae_decode_stream_destroy": (None, [C.c_void_p]),
    "kvae_encode_stream_begin": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.POINTER(C.c_void_p)]),
    "kvae_encode_stream_frames": (C.c_longlong, [C.c_void_p, C.c_longlong, C.c_int]),
    "kvae_encode_stream_lookahead": (C.c_longlong, [C.c_void_p]),
    "kvae_encode_stream_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_int, C.c_longlong,
                                          C.POINTER(C.c_longlong), C.c_void_p]),
    "kvae_encode_stream_end": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.POINTER(C.c_longlong),
                                         C.c_void_p]),
    "kvae_encode_stream_destroy": (None, [C.c_void_p]),
    "kvae_encode_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                     C.c_float, C.c_int, C.c_longlong, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_plan_fused_sample_supported": (C.c_int, [C.c_void_p]),
    "kvae_decode_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_longlong,
                                    C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "kvae_plan_fused_pcm_supported": (C.c_int, [C.c_void_p]),
    "kvae_aa_act_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                  C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_aa_act_win_fwd": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_longlong,
                                      C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "kvae_aa_act_ragged_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_int), C.c_int, C.c_void_p]),
    "kvae_zero_tail_cf": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.POINTER(C.c_int),
                                    C.c_int, C.c_void_p]),
    "kvae_conv1d_packed_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "kvae_conv1d_pack": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                   C.c_void_p]),
    "kvae_conv1d_win_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_longlong, C.c_int]),
    "kvae_conv1d_win_fwd": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                      C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
    "kvae_conv1d_stream_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int]),
    "kvae_conv1d_stream_fwd": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_longlong,
                                         C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_unary_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "kvae_axpby": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float, C.c_int, C.c_void_p]),
    "kvae_gauss_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "kvae_aa_act_bwd_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_longlong]),
    "kvae_aa_act_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p,
                                  C.c_size_t, C.c_void_p]),
    "kvae_unary_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "kvae_gauss_sample_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                        C.c_int, C.c_void_p]),
    "kvae_conv1d_win_bwd_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                                                       C.c_int, C.c_int, C.c_int]),
    "kvae_conv1d_win_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    "kvae_conv1d_dgrad_geom": (C.c_int, [C.c_int] * 7 + [C.POINTER(C.c_int * 6)]),
    "kvae_conv1d_dgrad_form": (C.c_int, [C.c_int] * 7 + [C.POINTER(C.c_int * 7)]),
    "kvae_flow_split": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "kvae_flow_split_bwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "kvae_flow_mask": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_wn_gate_fwd": (C.c_int, [C.c_void_p] * 2 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_wn_gate_bwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_wn_update_fwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_wn_update_bwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_flow_coupling_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                                            C.c_void_p]),
    "kvae_flow_coupling_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                                            C.c_void_p]),
    "kvae_plan_out_length": (C.c_longlong, [C.c_void_p, C.c_longlong]),
    "kvae_mrstft_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int]),
    "kvae_mrstft_loss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                   C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_prep_mono_clips": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "kvae_lm_glue_step": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.c_void_p] * 5 +
                          [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "kvae_plan_flops": (C.c_double, [C.c_void_p, C.c_int, C.c_longlong]),
    "kvae_plan_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "kvae_plan_step_profile": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double),
                                         C.POINTER(C.c_int), C.c_int]),
    "kvae_snake_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_weight_norm_fold": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "kvae_conv1d_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_conv1d_tc_supported": (C.c_int, [C.c_int] * 6),
    "kvae_conv1d_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "kvae_plan_param_count": (C.c_longlong, [C.c_void_p]),
    "kvae_plan_param_sizes": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong), C.c_int]),
    "kvae_plan_load_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "kvae_train_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_longlong]),
    "kvae_forward_train": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_longlong,
                                     C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                C.c_longlong, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "kvae_weight_norm_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_void_p]),
    "kvae_snake_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                 C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "kvae_vae_sample_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_gaussian_nll": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_float,
                                    C.c_int, C.c_void_p, C.c_void_p]),
    "kvae_adamw_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float,
                                  C.c_float, C.c_float, C.c_float, C.c_int, C.c_float, C.c_void_p]),
    "kvae_pcm16": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "kvae_sigma_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_float,
                                    C.c_void_p, C.c_float, C.c_size_t, C.c_void_p]),
    "kvae_vae_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                  C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "kvae_disc_period_fold": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "kvae_disc_avg_pool2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_disc_folded_width": (C.c_int, [C.c_int] * 4),
    "kvae_disc_fold_weight2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "kvae_disc_silu_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_disc_silu_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_disc_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.c_void_p]),
    "kvae_disc_score_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_void_p]),
    "kvae_disc_hinge": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "kvae_disc_feature_match_scratch_bytes": (C.c_size_t, [C.POINTER(C.c_longlong), C.c_int]),
    "kvae_disc_feature_match": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_longlong), C.c_int, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_disc_conv15_supported": (C.c_int, [C.c_int] * 3),
    "kvae_disc_conv15_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong,
                                       C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_disc_conv15_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_int, C.c_longlong, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kvae_disc_conv1x1_supported": (C.c_int, [C.c_int] * 4),
    "kvae_disc_conv1x1_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong,
                                        C.c_void_p]),
    "kvae_disc_conv1x1_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                        C.c_int, C.c_longlong, C.c_void_p]),
}


def lib() -> C.CDLL:
    """Loads libkvae.so once.  Raises if it has not been built (``make`` / ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KvaeError(f"{LIB_PATH} not found: build it with `make` (there is no fallback path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise KvaeError(lib().kvae_last_error().decode("utf-8", "replace"))


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise KvaeError(f"{what}: tensor is on {t.device}; kalle_audio_b200 runs on B200 GPUs only "
                        "(no CPU path; the reference's DataLoader-worker CPU encode must keep using the reference)")


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return KVAE_F32
    if dt == torch.bfloat16:
        return KVAE_BF16
    raise KvaeError(f"unsupported dtype {dt} at the C ABI (fp32 and bf16 only)")


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()
