"""ctypes binding of include/st2_b200.h.

There is no CPU fallback: if the library has not been built (python -m
styletts2_lite_b200.build, or __graft_entry__.build()) importing the symbols
raises, and every call checks the returned st2_status.
"""
from __future__ import annotations

import ctypes as C
import os

from .config import DecoderConfig

_HERE = os.path.dirname(os.path.abspath(__file__))
# ST2_B200_LIB selects another build of the same library (A/B timing of kernel variants on one GPU box)
LIB_PATH = os.environ.get("ST2_B200_LIB") or os.path.join(_HERE, "lib", "libst2_b200.so")

PREC = {"fp32": 0, "bf16": 1, "fp16": 2}
DTYPE = {"fp32": 0, "bf16": 1, "fp16": 2}
ACT = {"none": 0, "lrelu": 1, "snake": 2}


class St2Error(RuntimeError):
    pass


class St2Config(C.Structure):
    _fields_ = [("variant", C.c_int32), ("dim_in", C.c_int32), ("style_dim", C.c_int32),
                ("upsample_initial_channel", C.c_int32), ("n_stages", C.c_int32),
                ("upsample_rates", C.c_int32 * 4), ("upsample_kernel_sizes", C.c_int32 * 4),
                ("n_kernels", C.c_int32), ("resblock_kernel_sizes", C.c_int32 * 3),
                ("resblock_dilations", (C.c_int32 * 3) * 3),
                ("gen_istft_n_fft", C.c_int32), ("gen_istft_hop_size", C.c_int32),
                ("intermediate_dim", C.c_int32), ("num_layers", C.c_int32)]

    @staticmethod
    def from_config(cfg: DecoderConfig) -> "St2Config":
        c = St2Config()
        c.variant = 4 if cfg.is_vocos else (1 if cfg.is_istft else 0)
        c.intermediate_dim = cfg.intermediate_dim
        c.num_layers = cfg.num_layers
        c.dim_in = cfg.dim_in
        c.style_dim = cfg.style_dim
        c.upsample_initial_channel = cfg.upsample_initial_channel
        c.n_stages = cfg.num_stages
        for i, (u, k) in enumerate(zip(cfg.upsample_rates, cfg.upsample_kernel_sizes)):
            c.upsample_rates[i] = u
            c.upsample_kernel_sizes[i] = k
        c.n_kernels = len(cfg.resblock_kernel_sizes)
        for j, k in enumerate(cfg.resblock_kernel_sizes):
            c.resblock_kernel_sizes[j] = k
            for m, d in enumerate(cfg.resblock_dilation_sizes[j]):
                c.resblock_dilations[j][m] = d
        c.gen_istft_n_fft = cfg.gen_istft_n_fft
        c.gen_istft_hop_size = cfg.gen_istft_hop_size
        return c


_P = C.c_void_p
_I = C.c_int32
_L = C.c_int64

# name -> (restype, argtypes); exactly the declarations of include/st2_b200.h
SIGNATURES = {
    "st2_abi_version": (C.c_int, []),
    "st2_last_error": (C.c_char_p, []),
    "st2_decoder_create": (C.c_int, [C.POINTER(St2Config), C.POINTER(_P)]),
    "st2_decoder_destroy": (None, [_P]),
    "st2_decoder_set_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(_L), _I]),
    "st2_decoder_finalize": (C.c_int, [_P, _P]),
    "st2_decoder_num_params": (_L, [_P]),
    "st2_decoder_workspace_bytes": (_L, [_P, _I, _I, _I]),
    "st2_decoder_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_uint64, _P, _I, _I, _I, _P, _L, _P]),
    "st2_decoder_set_tap": (C.c_int, [_P, C.c_char_p, _P, _L]),
    "st2_decoder_set_option": (C.c_int, [_P, C.c_char_p, _I]),
    "st2_set_tuning": (C.c_int, [C.c_char_p, _I]),
    "st2_decoder_set_seed_buffer": (C.c_int, [_P, _P]),
    "st2_decoder_last_launch_count": (_L, [_P]),
    "st2_decoder_set_profiling": (C.c_int, [_P, _I]),
    "st2_profile_num_categories": (C.c_int, []),
    "st2_profile_category_name": (C.c_char_p, [_I]),
    "st2_decoder_get_profile": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(_L), C.POINTER(C.c_double),
                                          C.POINTER(C.c_double)]),
    "st2_decoder_get_profile_launches": (_L, [_P, _L, C.POINTER(_I), C.POINTER(C.c_float), C.POINTER(C.c_double),
                                              C.POINTER(C.c_double)]),
    "st2_f0n_create": (C.c_int, [_I, _I, C.POINTER(_P)]),
    "st2_f0n_workspace_bytes": (_L, [_P, _I, _I, _I]),
    "st2_f0n_forward": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _L, _P]),
    "st2_dur_workspace_bytes": (_L, [_P, _I, _I, _I]),
    "st2_dur_forward": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _L, _P]),
    "st2_dur_forward_ragged": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _L, _P]),
    "st2_text_create": (C.c_int, [_I, _I, _I, _I, C.POINTER(_P)]),
    "st2_text_workspace_bytes": (_L, [_P, _I, _I, _I]),
    "st2_text_forward": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _L, _P]),
    "st2_text_forward_ragged": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P, _L, _P]),
    "st2_round_durations": (C.c_int, [_P, _P, _P, _P, _I, _I, _P]),
    "st2_smooth_durations": (C.c_int, [_P, _P, _P, _P, C.c_float, C.c_float, _P, _P, _I, _I, _P]),
    "st2_smooth_durations_chained": (C.c_int, [_P, _P, _P, _P, C.c_float, C.c_float, _P, _P, _I, _I, _P]),
    "st2_length_regulate": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "st2_sinegen_phase": (C.c_int, [_P, _P, _P, _I, _I, _I, _P]),
    "st2_har_source": (C.c_int, [_P, _P, C.c_uint64, _P, _P, _P, _P, _I, _I, _I, _P]),
    "st2_noise_conv_scratch_bytes": (_L, [_I, _I, _I, _I, _I]),
    "st2_noise_conv": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "st2_post_hifigan": (C.c_int, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "st2_style_fc": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "st2_adain_scratch_bytes": (_L, [_I, _I, _I]),
    "st2_adain_act": (C.c_int, [_P, _I, _P, _I, _P, _I, C.c_float, _P, _I, _I, _I, _I, _I, _P, _P]),
    "st2_conv1d_scratch_bytes": (_L, [_I, _I, _I, _I, _I, _I]),
    "st2_adain_conv1d_fused_scratch_bytes": (_L, [_I, _I, _I, _I, _I]),
    "st2_adain_conv1d_fused": (C.c_int, [_P, _P, _P, _I, C.c_float, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I,
                                         C.c_float, _I, _I, _P]),
    "st2_postprocess_scratch_bytes": (_L, [_I]),
    "st2_postprocess_max_samples": (_L, [_I, _I, _I, _I]),
    "st2_postprocess": (C.c_int, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "st2_adain_conv1d_fused_ex_scratch_bytes": (_L, [_I, _I, _I, _I, _I]),
    "st2_adain_conv1d_fused_ex": (C.c_int, [_P, _P, _P, _I, C.c_float, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I,
                                            _I, C.c_float, _I, _I, _I, _I, _I, _I, _I, _P]),
    "st2_adain_conv1d_row_scratch_bytes": (_L, [_I, _I, _I, _I]),
    "st2_adain_conv1d_row": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, C.c_float, _I, _I, _I,
                                       _P]),
    "st2_adain_conv1d_row_pair_scratch_bytes": (_L, [_I, _I, _I, _I, _I]),
    "st2_adain_conv1d_row_pair": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(_I), _P, _I, _I, _I, _I,
                                            _I, _I, _I, _I, _P]),
    "st2_act_conv_transpose1d_fused_scratch_bytes": (_L, [_I, _I, _I, _I, _I, _I]),
    "st2_act_conv_transpose1d_fused": (C.c_int, [_P, _P, _I, C.c_float, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I,
                                                 _I, _P]),
    "st2_act_conv_transpose1d_fused_ex_scratch_bytes": (_L, [_I, _I, _I, _I, _I, _I]),
    "st2_act_conv_transpose1d_fused_ex": (C.c_int, [_P, _P, _I, C.c_float, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I,
                                                    _I, _I, _I, _P]),
    "st2_conv1d": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the C-ABI library; raises St2Error (never falls back) if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise St2Error("%s not found: build it with `python -m styletts2_lite_b200.build` "
                       "(there is no CPU fallback for this path)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.st2_abi_version() != 1:
        raise St2Error("ABI version mismatch: library %d, binding 1" % lib.st2_abi_version())
    _lib = lib
    return lib


def check(status: int, what: str = "") -> int:
    if status < 0:
        msg = load().st2_last_error()
        raise St2Error("%s failed (%d): %s" % (what or "st2 call", status, msg.decode() if msg else ""))
    return status


_tuning_generation = 0


def set_tuning(name: str, value: int) -> None:
    """st2_set_tuning (a process-wide kernel-selection / planner switch), noted in tuning_generation() so that decoder modules
    plan their workspace and capture their CUDA graphs again instead of reusing what the old switches produced."""
    global _tuning_generation
    check(load().st2_set_tuning(name.encode(), int(value)), "st2_set_tuning(%s)" % name)
    _tuning_generation += 1


def tuning_generation() -> int:
    """How many times set_tuning() has changed a switch in this process."""
    return _tuning_generation


def ptr(t) -> C.c_void_p:
    """Raw device pointer of a torch tensor (None -> NULL)."""
    return C.c_void_p(None if t is None else t.data_ptr())
