"""ctypes binding of libptts_b200.so (the C ABI declared in include/ptts_b200.h).

The product path has NO CPU fallback: if the shared library is missing this module raises at first
use.  Errors cross the ABI as integer codes; they are re-raised here as ValueError (contract
violations, like the reference's ValueError guards) or RuntimeError.
"""
from __future__ import annotations
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# PTTS_LIB selects an alternative in-tree build of the same ABI (csrc/build.py --tag <t> -> libptts_b200_<t>.so), so that several
# kernel variants can be compared inside one GPU session; the default is the product library.
LIB_PATH = os.environ.get("PTTS_LIB") or os.path.join(_HERE, "csrc", "libptts_b200.so")

BF16, F32, I64, I32 = 0, 1, 2, 3
OK, EINVAL, ECUDA, ESTATE = 0, 1, 2, 3


class DecoderConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "hidden_size", "num_layers", "num_heads", "num_kv_heads", "num_cross_kv_heads", "ffn_dim", "vocab_size",
        "num_codebooks", "max_positions", "rope", "activation", "dtype", "bos_token_id", "pad_token_id",
        "eos_token_id")] + [("rope_theta", C.c_float), ("layer_norm_eps", C.c_float)]


class GenParamsC(C.Structure):
    _fields_ = [("max_length", C.c_int32), ("min_new_tokens", C.c_int32), ("do_sample", C.c_int32),
                ("top_k", C.c_int32), ("top_p", C.c_float), ("temperature", C.c_float), ("seed", C.c_uint64),
                ("suppress_special", C.c_int32), ("codebook_size", C.c_int32),
                ("row_base", C.c_int32), ("reserved_", C.c_int32)]


class DacConfigC(C.Structure):
    _fields_ = [("n_codebooks", C.c_int32), ("codebook_size", C.c_int32), ("codebook_dim", C.c_int32),
                ("latent_dim", C.c_int32), ("decoder_dim", C.c_int32), ("n_blocks", C.c_int32),
                ("strides", C.c_int32 * 8), ("dtype", C.c_int32)]


class DacEncoderConfigC(C.Structure):
    _fields_ = [("encoder_dim", C.c_int32), ("n_blocks", C.c_int32), ("strides", C.c_int32 * 8), ("latent_dim", C.c_int32),
                ("n_codebooks", C.c_int32), ("codebook_size", C.c_int32), ("codebook_dim", C.c_int32), ("dtype", C.c_int32)]


# tensor ids (include/ptts_b200.h)
T_EMBED_TOKENS, T_POS_TABLE, T_LN1_W, T_LN1_B, T_SELF_Q, T_SELF_K, T_SELF_V, T_SELF_O = range(8)
T_LN2_W, T_LN2_B, T_CROSS_Q, T_CROSS_K, T_CROSS_V, T_CROSS_O, T_LN3_W, T_LN3_B = range(8, 16)
T_FC1, T_FC2, T_FINAL_LN_W, T_FINAL_LN_B, T_LM_HEAD, T_ROPE_COS, T_ROPE_SIN = range(16, 23)

_VP, _I32, _I64 = C.c_void_p, C.c_int32, C.c_int64
_SIGS = {
    "ptts_last_error": (C.c_char_p, []),
    "ptts_version": (C.c_int, []),
    "ptts_decoder_blob_bytes": (C.c_int, [C.POINTER(DecoderConfigC), C.POINTER(_I64)]),
    "ptts_decoder_pack": (C.c_int, [C.POINTER(DecoderConfigC), _VP, _I32, _I32, _VP, _I32, _I64, _I64, _VP]),
    "ptts_decoder_finalize": (C.c_int, [C.POINTER(DecoderConfigC), _VP, _VP]),
    "ptts_workspace_bytes": (C.c_int, [C.POINTER(DecoderConfigC), _I32, _I32, _I32, _I32, C.POINTER(_I64)]),
    "ptts_session_create": (C.c_int, [C.POINTER(DecoderConfigC), _VP, _VP, _I64, _I32, _I32, _I32, _I32, C.POINTER(_VP)]),
    "ptts_workspace_bytes_ex": (C.c_int, [C.POINTER(DecoderConfigC), _I32, _I32, _I32, _I32, _I32, C.POINTER(_I64)]),
    "ptts_session_create_ex": (C.c_int, [C.POINTER(DecoderConfigC), _VP, _VP, _I64, _I32, _I32, _I32, _I32, _I32, C.POINTER(_VP)]),
    "ptts_prefill_ids": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _I32, _VP]),
    "ptts_session_destroy": (C.c_int, [_VP]),
    "ptts_generate_begin": (C.c_int, [_VP, C.POINTER(GenParamsC), _VP]),
    "ptts_prefill": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    "ptts_decode_forward": (C.c_int, [_VP, _VP]),
    "ptts_sample": (C.c_int, [_VP, _VP, _VP]),
    "ptts_decode_steps": (C.c_int, [_VP, _I32, _VP]),
    "ptts_session_logits": (C.c_int, [_VP, C.POINTER(_VP)]),
    "ptts_session_scores": (C.c_int, [_VP, C.POINTER(_VP)]),
    "ptts_session_raw_ids": (C.c_int, [_VP, C.POINTER(_VP), C.POINTER(_I32)]),
    "ptts_session_state": (C.c_int, [_VP, C.POINTER(_VP)]),
    "ptts_session_launches": (C.c_int, [_VP, C.POINTER(_I64)]),
    "ptts_session_fused": (C.c_int, [_VP, C.POINTER(_I32)]),
    "ptts_session_set_profile": (C.c_int, [_VP, _VP]),
    "ptts_delay_build": (C.c_int, [_VP, _I32, _I32, _I32, _I64, _I64, _I32, _VP, _VP]),
    "ptts_delay_apply": (C.c_int, [_VP, _I32, _I32, _I64, _VP, _I64, _VP, _VP]),
    "ptts_logits_processor": (C.c_int, [_VP, _I32, _I32, _I64, _VP, _I32, _I64, _I32, _VP, _VP]),
    "ptts_op_linear": (C.c_int, [C.POINTER(DecoderConfigC), _VP, _I32, _I32, _VP, _I32, _I32, _I32, _VP, _VP, _VP]),
    "ptts_dac_blob_bytes": (C.c_int, [C.POINTER(DacConfigC), C.POINTER(_I64)]),
    "ptts_dac_num_tensors": (C.c_int, [C.POINTER(DacConfigC), C.POINTER(_I32)]),
    "ptts_dac_pack": (C.c_int, [C.POINTER(DacConfigC), _VP, _I32, _VP, _I32, _I64, _VP]),
    "ptts_dac_workspace_bytes": (C.c_int, [C.POINTER(DacConfigC), _I32, _I32, C.POINTER(_I64)]),
    "ptts_dac_decode": (C.c_int, [C.POINTER(DacConfigC), _VP, _VP, _I64, _VP, _I32, _I32, _VP, _VP]),
    "ptts_dac_encoder_blob_bytes": (C.c_int, [C.POINTER(DacEncoderConfigC), C.POINTER(_I64)]),
    "ptts_dac_encoder_num_tensors": (C.c_int, [C.POINTER(DacEncoderConfigC), C.POINTER(_I32)]),
    "ptts_dac_encoder_pack": (C.c_int, [C.POINTER(DacEncoderConfigC), _VP, _I32, _VP, _I32, _I64, _VP]),
    "ptts_dac_encoder_workspace_bytes": (C.c_int, [C.POINTER(DacEncoderConfigC), _I32, _I64, C.POINTER(_I64)]),
    "ptts_dac_encode": (C.c_int, [C.POINTER(DacEncoderConfigC), _VP, _VP, _I64, _VP, _I32, _I64, _I32, _VP, _VP, _VP]),
}
EXPORTED_SYMBOLS = tuple(_SIGS)

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python parler_tts_b200/csrc/build.py` "
                "(or __graft_entry__.build()).  parler_tts_b200 has no CPU / PyTorch fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(code: int):
    if code == OK:
        return
    msg = lib().ptts_last_error().decode("utf-8", "replace")
    if code == EINVAL:
        raise ValueError(msg)
    raise RuntimeError(msg)


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.bfloat16:
        return BF16
    if dt == torch.float32:
        return F32
    raise ValueError(f"unsupported dtype {dt}: the B200 path computes in bfloat16 or float32")


def torch_dtype(code: int) -> torch.dtype:
    return torch.bfloat16 if code == BF16 else torch.float32


def ptr(t: torch.Tensor | None):
    if t is None:
        return None
    if not t.is_cuda:
        raise ValueError("parler_tts_b200 operates on CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
