"""DACModel: the reference's codec wrapper surface, backed by the sm_100a DAC decode kernels.

Mirrors parler_tts/dac_wrapper/modeling_dac.py:14-164:
  DACModel.encode(input_values, padding_mask=None, bandwidth=None, return_dict=None, n_quantizers=None,
                  sample_rate=None)                                                 (:33-104, voice prompts)
  DACModel.decode(audio_codes, audio_scales, padding_mask=None, return_dict=None)   (:106-142)
Weights: either folded tensors under transformers-DacModel style keys (decoder.conv1.weight, ...) or
descript-audio-codec checkpoint keys with weight-norm parameters (weight_g / weight_v, or
parametrizations.weight.original0/1), folded here as w = g * v / ||v|| (reference :148-157).
The encoder (encoder.*, quantizer.quantizers.N.in_proj.*) is packed into its own blob when the state dict has it;
a decoder-only state dict loads as before and `encode` then raises.
"""
from __future__ import annotations
import ctypes as C
import math
import re
from dataclasses import dataclass

import torch

from . import _lib
from .configuration import DACConfig


@dataclass
class DACDecoderOutput:
    """Stands in for transformers' EncodecDecoderOutput (audio_values [B, 1, samples])."""
    audio_values: torch.Tensor = None

    def __getitem__(self, i):
        return (self.audio_values,)[i]


def _dac_tensor_list(cfg: DACConfig) -> list[str]:
    """(id -> key) table in the order csrc/dac.h::make_dac_layout enumerates tensors."""
    names = []
    for i in range(cfg.num_codebooks):
        q = f"quantizer.quantizers.{i}."
        names += [q + "codebook.weight", q + "out_proj.weight", q + "out_proj.bias"]
    names += ["decoder.conv1.weight", "decoder.conv1.bias"]
    for bi in range(len(cfg.decoder_rates)):
        p = f"decoder.block.{bi}."
        names += [p + "snake1.alpha", p + "conv_t1.weight", p + "conv_t1.bias"]
        for r in (1, 2, 3):
            u = p + f"res_unit{r}."
            names += [u + "snake1.alpha", u + "conv1.weight", u + "conv1.bias", u + "snake2.alpha", u + "conv2.weight", u + "conv2.bias"]
    names += ["decoder.snake1.alpha", "decoder.conv2.weight", "decoder.conv2.bias"]
    return names


@dataclass
class DACEncoderOutput:
    """Stands in for transformers' EncodecEncoderOutput (audio_codes [1, B, n_q, T], audio_scales [None])."""
    audio_codes: torch.Tensor = None
    audio_scales: list = None

    def __getitem__(self, i):
        return (self.audio_codes, self.audio_scales)[i]


def _dac_encoder_tensor_list(cfg: DACConfig) -> list[str]:
    """(id -> key) table in the order csrc/dac.h::make_dac_encoder_layout enumerates tensors."""
    names = ["encoder.conv1.weight", "encoder.conv1.bias"]
    for bi in range(len(cfg.encoder_rates)):
        p = f"encoder.block.{bi}."
        for r in (1, 2, 3):
            u = p + f"res_unit{r}."
            names += [u + "snake1.alpha", u + "conv1.weight", u + "conv1.bias", u + "snake2.alpha", u + "conv2.weight", u + "conv2.bias"]
        names += [p + "snake1.alpha", p + "conv1.weight", p + "conv1.bias"]
    names += ["encoder.snake1.alpha", "encoder.conv2.weight", "encoder.conv2.bias"]
    for i in range(cfg.num_codebooks):
        q = f"quantizer.quantizers.{i}."
        names += [q + "in_proj.weight", q + "in_proj.bias", q + "codebook.weight", q + "out_proj.weight", q + "out_proj.bias"]
    return names


def _fold_weight_norm(sd: dict[str, torch.Tensor]) -> dict[str, torch.Tensor]:
    """g * v / ||v|| over all dims but 0 (torch weight_norm default dim=0), in fp32."""
    out = {}
    pairs = {}
    for k, v in sd.items():
        m = re.match(r"(.*)\.(weight_g|weight_v|parametrizations\.weight\.original0|parametrizations\.weight\.original1)$", k)
        if m:
            kind = "g" if (m.group(2).endswith("_g") or m.group(2).endswith("original0")) else "v"
            pairs.setdefault(m.group(1), {})[kind] = v
        else:
            out[k] = v
    for base, gv in pairs.items():
        g, v = gv["g"].float(), gv["v"].float()
        norm = v.flatten(1).norm(dim=1).view(-1, *([1] * (v.dim() - 1)))
        out[base + ".weight"] = g * v / norm
    return out


def _from_descript_keys(sd: dict[str, torch.Tensor], n_blocks: int) -> dict[str, torch.Tensor]:
    """descript-audio-codec module paths -> the transformers-DacModel style keys used internally.

    descript layout: decoder.model = [WNConv1d, DecoderBlock x n, Snake1d, WNConv1d, Tanh];
    DecoderBlock.block = [Snake1d, WNConvTranspose1d, ResidualUnit x 3]; ResidualUnit.block =
    [Snake1d, WNConv1d(k7), Snake1d, WNConv1d(k1)]."""
    out = {}
    for k, v in sd.items():
        if k.startswith("quantizer."):
            out[k] = v
            continue
        m = re.match(r"decoder\.model\.(\d+)\.(.*)$", k)
        if not m:
            continue
        i, rest = int(m.group(1)), m.group(2)
        if i == 0:
            out["decoder.conv1." + rest] = v
        elif 1 <= i <= n_blocks:
            bi = i - 1
            mm = re.match(r"block\.(\d+)\.(.*)$", rest)
            j, r2 = int(mm.group(1)), mm.group(2)
            p = f"decoder.block.{bi}."
            if j == 0:
                out[p + "snake1." + r2] = v
            elif j == 1:
                out[p + "conv_t1." + r2] = v
            else:
                m3 = re.match(r"block\.(\d+)\.(.*)$", r2)
                u, r3 = int(m3.group(1)), m3.group(2)
                name = {0: "snake1.", 1: "conv1.", 2: "snake2.", 3: "conv2."}[u]
                out[p + f"res_unit{j - 1}." + name + r3] = v
        elif i == n_blocks + 1:
            out["decoder.snake1." + rest] = v
        elif i == n_blocks + 2:
            out["decoder.conv2." + rest] = v
    return out


def _encoder_from_descript_keys(sd: dict[str, torch.Tensor], n_blocks: int) -> dict[str, torch.Tensor]:
    """descript-audio-codec encoder module paths -> the transformers-DacModel style keys used internally.

    descript layout: encoder.block = [WNConv1d, EncoderBlock x n, Snake1d, WNConv1d]; EncoderBlock.block =
    [ResidualUnit x 3, Snake1d, WNConv1d(k 2s, stride s)]; ResidualUnit.block = [Snake1d, WNConv1d(k7), Snake1d, WNConv1d(k1)].
    Other keys are dropped."""
    out = {}
    for k, v in sd.items():
        m = re.match(r"encoder\.block\.(\d+)\.(.*)$", k)
        if not m:
            continue
        i, rest = int(m.group(1)), m.group(2)
        if i == 0:
            out["encoder.conv1." + rest] = v
        elif 1 <= i <= n_blocks:
            p = f"encoder.block.{i - 1}."
            mm = re.match(r"block\.(\d+)\.(.*)$", rest)
            j, r2 = int(mm.group(1)), mm.group(2)
            if j <= 2:
                m3 = re.match(r"block\.(\d+)\.(.*)$", r2)
                u, r3 = int(m3.group(1)), m3.group(2)
                name = {0: "snake1.", 1: "conv1.", 2: "snake2.", 3: "conv2."}[u]
                out[p + f"res_unit{j + 1}." + name + r3] = v
            elif j == 3:
                out[p + "snake1." + r2] = v
            elif j == 4:
                out[p + "conv1." + r2] = v
        elif i == n_blocks + 1:
            out["encoder.snake1." + rest] = v
        elif i == n_blocks + 2:
            out["encoder.conv2." + rest] = v
    return out


class DACModel:
    config_class = DACConfig
    main_input_name = "input_values"

    def __init__(self, config: DACConfig, device="cuda", dtype=torch.float32):
        self.config = config
        self.device = torch.device(device)
        self.dtype = dtype
        self._c = _lib.DacConfigC()
        self._c.n_codebooks = config.num_codebooks
        self._c.codebook_size = config.codebook_size
        self._c.codebook_dim = config.codebook_dim
        self._c.latent_dim = config.latent_dim
        self._c.decoder_dim = config.decoder_dim
        self._c.n_blocks = len(config.decoder_rates)
        for i, s in enumerate(config.decoder_rates):
            self._c.strides[i] = int(s)
        self._c.dtype = _lib.dtype_code(dtype)
        self.hop_length = math.prod(config.decoder_rates)
        # the packed weight blob exists from construction on (zeros until load_state_dict / a broadcast fills it), so that
        # every rank of a sharded run owns a buffer of the right size for the init broadcast (dist.broadcast_model_weights)
        nbytes = C.c_int64()
        _lib.check(_lib.lib().ptts_dac_blob_bytes(C.byref(self._c), C.byref(nbytes)))
        self.blob = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)
        self.loaded = False
        self._ws = None
        self._ec = _lib.DacEncoderConfigC()
        self._ec.encoder_dim = config.encoder_dim
        self._ec.n_blocks = len(config.encoder_rates)
        for i, s in enumerate(config.encoder_rates):
            self._ec.strides[i] = int(s)
        self._ec.latent_dim = config.latent_dim
        self._ec.n_codebooks = config.num_codebooks
        self._ec.codebook_size = config.codebook_size
        self._ec.codebook_dim = config.codebook_dim
        self._ec.dtype = _lib.dtype_code(dtype)
        self.encoder_hop_length = math.prod(config.encoder_rates)
        # allocated by load_state_dict when the state dict carries the encoder: decoder-only models do not pay for it
        self.encoder_blob = None
        self.encoder_loaded = False
        self._enc_ws = None

    # -- weights -----------------------------------------------------------------------------------
    def load_state_dict(self, sd: dict[str, torch.Tensor], strict: bool = True):
        sd = {(k[len("model."):] if k.startswith("model.") else k): v for k, v in sd.items()}
        sd = _fold_weight_norm(sd)
        if any(re.match(r"encoder\.block\.\d+\.block\.", k) for k in sd):
            sd = {**{k: v for k, v in sd.items() if not k.startswith("encoder.")},
                  **_encoder_from_descript_keys(sd, len(self.config.encoder_rates))}
        if any(k.startswith("encoder.") for k in sd):
            self._load_encoder(sd, strict)
        if any(k.startswith("decoder.model.") for k in sd):
            sd = _from_descript_keys(sd, len(self.config.decoder_rates))
        names = _dac_tensor_list(self.config)
        missing = [n for n in names if n not in sd]
        if missing and strict:
            raise ValueError(f"DACModel.load_state_dict: missing keys {missing[:5]}{'...' if len(missing) > 5 else ''}")
        lib = _lib.lib()
        n = C.c_int32()
        _lib.check(lib.ptts_dac_num_tensors(C.byref(self._c), C.byref(n)))
        assert n.value == len(names), (n.value, len(names))
        self.blob.zero_()
        for i, name in enumerate(names):
            if name not in sd:
                continue
            t = sd[name].to(device=self.device)
            if t.dtype not in (torch.float32, torch.bfloat16):
                t = t.float()
            t = t.contiguous()
            _lib.check(lib.ptts_dac_pack(C.byref(self._c), _lib.ptr(self.blob), i, _lib.ptr(t), _lib.dtype_code(t.dtype),
                                         t.numel(), _lib.stream_ptr()))
        torch.cuda.current_stream().synchronize()  # staging tensors above go out of scope
        self.loaded = True
        return self

    def _load_encoder(self, sd: dict[str, torch.Tensor], strict: bool):
        names = _dac_encoder_tensor_list(self.config)
        missing = [n for n in names if n not in sd]
        if missing and strict:
            raise ValueError(f"DACModel.load_state_dict: missing encoder keys {missing[:5]}{'...' if len(missing) > 5 else ''}")
        lib = _lib.lib()
        nbytes, n = C.c_int64(), C.c_int32()
        _lib.check(lib.ptts_dac_encoder_blob_bytes(C.byref(self._ec), C.byref(nbytes)))
        _lib.check(lib.ptts_dac_encoder_num_tensors(C.byref(self._ec), C.byref(n)))
        assert n.value == len(names), (n.value, len(names))
        self.encoder_blob = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)
        for i, name in enumerate(names):
            if name not in sd:
                continue
            t = sd[name].to(device=self.device)
            if t.dtype not in (torch.float32, torch.bfloat16):
                t = t.float()
            t = t.contiguous()
            _lib.check(lib.ptts_dac_encoder_pack(C.byref(self._ec), _lib.ptr(self.encoder_blob), i, _lib.ptr(t), _lib.dtype_code(t.dtype),
                                                 t.numel(), _lib.stream_ptr()))
        torch.cuda.current_stream().synchronize()  # staging tensors above go out of scope
        self.encoder_loaded = True

    def to(self, *args, **kwargs):
        return self

    def eval(self):
        return self

    # -- reference surface -------------------------------------------------------------------------
    @torch.no_grad()
    def encode(self, input_values, padding_mask=None, bandwidth=None, return_dict=None, n_quantizers=None, sample_rate=None):
        """input_values [B, 1, samples] -> DACEncoderOutput(audio_codes [1, B, n_q, ceil(samples / hop)], audio_scales [None]).

        As the reference: the audio is right-padded with zeros to a multiple of the hop and encoded as one chunk;
        n_quantizers=None uses every codebook.  padding_mask and bandwidth are accepted and unused, as there."""
        codes, _ = self._encode(input_values, n_quantizers, sample_rate, want_z=False)
        if return_dict is False:
            return (codes[None], [None])
        return DACEncoderOutput(codes[None], [None])

    def _encode(self, input_values, n_quantizers=None, sample_rate=None, want_z=False):
        """encode() plus, with want_z, the quantized latent z [B, latent_dim, frames] (DAC.encode's first output)."""
        if input_values.dim() != 3:
            raise ValueError(f"input_values must be [batch, channels, samples], got {tuple(input_values.shape)}")
        B, channels, length = input_values.shape
        if channels < 1 or channels > 2:
            raise ValueError(f"Number of audio channels must be 1 or 2, but got {channels}")
        if channels != 1:
            raise ValueError("the DAC encoder takes mono audio (its first convolution has one input channel); got 2 channels")
        if sample_rate is not None and sample_rate != self.config.sampling_rate:
            raise ValueError(f"sample_rate {sample_rate} does not match the model's {self.config.sampling_rate}")
        if not self.encoder_loaded:
            raise RuntimeError("DACModel has no encoder weights loaded (the state dict had no encoder.* tensors)")
        if B == 0 or length == 0:
            raise ValueError("input_values is empty")
        K = self.config.num_codebooks
        n_q = K if n_quantizers is None else min(int(n_quantizers), K)
        if n_q < 1:
            raise ValueError(f"n_quantizers must be >= 1, got {n_quantizers}")
        hop = self.encoder_hop_length
        n = -(-length // hop) * hop
        audio = torch.nn.functional.pad(input_values[:, 0].to(device=self.device, dtype=self.dtype), (0, n - length)).contiguous()
        lib = _lib.lib()
        need = C.c_int64()
        _lib.check(lib.ptts_dac_encoder_workspace_bytes(C.byref(self._ec), B, n, C.byref(need)))
        if self._enc_ws is None or self._enc_ws.numel() < need.value:
            self._enc_ws = None
            self._enc_ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        codes = torch.empty(B, n_q, n // hop, dtype=torch.int64, device=self.device)
        z = torch.empty(B, n // hop, self.config.latent_dim, dtype=self.dtype, device=self.device) if want_z else None
        _lib.check(lib.ptts_dac_encode(C.byref(self._ec), _lib.ptr(self.encoder_blob), _lib.ptr(self._enc_ws), self._enc_ws.numel(),
                                       _lib.ptr(audio), B, n, n_q, _lib.ptr(codes), _lib.ptr(z), _lib.stream_ptr()))
        return codes, (z.transpose(1, 2) if want_z else None)

    @torch.no_grad()
    def decode(self, audio_codes, audio_scales=None, padding_mask=None, return_dict=None):
        """audio_codes [1, B, K, T] int64 (CUDA) -> DACDecoderOutput(audio_values [B, 1, hop*T])."""
        if not self.loaded:
            raise RuntimeError("DACModel has no weights loaded")
        if len(audio_codes) != 1:
            raise ValueError(f"Expected one frame, got {len(audio_codes)}")
        codes = audio_codes.squeeze(0)
        if codes.dim() != 3 or codes.shape[1] != self.config.num_codebooks:
            raise ValueError(f"audio_codes must be [1, B, {self.config.num_codebooks}, T], got {tuple(audio_codes.shape)}")
        codes = codes.to(device=self.device, dtype=torch.int64).contiguous()
        B, K, T = codes.shape
        if T == 0 or B == 0:
            raise ValueError("audio_codes is empty")
        if bool(((codes < 0) | (codes >= self.config.codebook_size)).any()):
            raise IndexError("audio code out of range for the codebook (the reference's embedding lookup raises too)")
        lib = _lib.lib()
        need = C.c_int64()
        _lib.check(lib.ptts_dac_workspace_bytes(C.byref(self._c), B, T, C.byref(need)))
        if self._ws is None or self._ws.numel() < need.value:
            self._ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        audio = torch.empty(B, 1, T * self.hop_length, dtype=self.dtype, device=self.device)
        _lib.check(lib.ptts_dac_decode(C.byref(self._c), _lib.ptr(self.blob), _lib.ptr(self._ws), self._ws.numel(),
                                       _lib.ptr(codes), B, T, _lib.ptr(audio), _lib.stream_ptr()))
        if return_dict is False:
            return (audio,)
        return DACDecoderOutput(audio)

    def forward(self, tensor):
        raise ValueError("`DACModel.forward` not implemented yet")
