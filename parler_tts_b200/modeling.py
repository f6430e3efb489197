"""Host-side mirror of the reference's generation surface, calling the sm_100a kernels through the C ABI.

Mirrors (same names, argument meaning and error behaviour; nothing here computes on the CPU):
  build_delay_pattern_mask / apply_delay_pattern_mask   parler_tts/modeling_parler_tts.py:205-276
  ParlerTTSLogitsProcessor                              parler_tts/logits_processors.py:6-53
  ParlerTTSForCausalLM (step operator)                  parler_tts/modeling_parler_tts.py:1824-1974
  ParlerTTSForConditionalGeneration.generate            parler_tts/modeling_parler_tts.py:3322-3653
PyTorch is used for device memory, streams and the one-off side inputs the path does not replace
(text encoder, prompt embedding lookup: SURVEY.md section 1).
"""
from __future__ import annotations
import ctypes as C
import json
import math
import os
from typing import Any, Optional

import torch

from . import _lib
from .configuration import DACConfig, GenerationConfig, ParlerTTSConfig, ParlerTTSDecoderConfig
from .dac_wrapper import DACModel

_ACT = {"gelu": 0, "relu": 1, "silu": 2, "swish": 2, "gelu_new": 3, "gelu_pytorch_tanh": 3}


# ---- delay pattern (stand-alone operators) -------------------------------------------------------
def build_delay_pattern_mask(input_ids: torch.LongTensor, bos_token_id: int, pad_token_id: int, max_length: int,
                             num_codebooks: int):
    """Same contract as the reference function: returns (input_ids[:, :first_start], pattern_mask)."""
    ids = input_ids.reshape(-1, num_codebooks, input_ids.shape[-1])
    bsz, K, seq_len = ids.shape
    ids2 = ids.reshape(bsz * K, seq_len).to(torch.int64).contiguous()
    mask = torch.empty(bsz * K, max_length, dtype=torch.int64, device=ids2.device)
    _lib.check(_lib.lib().ptts_delay_build(_lib.ptr(ids2), bsz * K, seq_len, K, int(bos_token_id), int(pad_token_id),
                                           int(max_length), _lib.ptr(mask), _lib.stream_ptr()))
    if max_length < 2 * K - 1:
        return ids2, mask
    first = mask.view(bsz, K, max_length)[:, 0, :]
    starts = (first == -1).nonzero()[:, 1]
    first_start = int(starts.min()) if len(starts) > 0 else seq_len
    out_ids = mask.view(bsz, K, max_length)[..., :first_start].reshape(bsz * K, -1)
    return out_ids, mask


def apply_delay_pattern_mask(input_ids: torch.LongTensor, decoder_pad_token_mask: torch.LongTensor):
    seq_len = input_ids.shape[-1]
    ids = input_ids.reshape(-1, seq_len).to(torch.int64).contiguous()
    mask = decoder_pad_token_mask.reshape(-1, decoder_pad_token_mask.shape[-1]).to(torch.int64).contiguous()
    if mask.shape[-1] < seq_len:
        raise ValueError(f"delay pattern mask is shorter ({mask.shape[-1]}) than the ids ({seq_len})")
    out = torch.empty_like(ids)
    _lib.check(_lib.lib().ptts_delay_apply(_lib.ptr(ids), ids.shape[0], seq_len, seq_len, _lib.ptr(mask), mask.shape[-1],
                                           _lib.ptr(out), _lib.stream_ptr()))
    return out.reshape(input_ids.shape)


class ParlerTTSLogitsProcessor:
    """Stateful EOS gating across codebooks; HF LogitsProcessor protocol (__call__(input_ids, scores))."""

    def __init__(self, eos_token_id, num_codebooks: int, batch_size: int, device: str = "cuda"):
        if isinstance(eos_token_id, torch.Tensor):
            if torch.is_floating_point(eos_token_id) or (eos_token_id < 0).any():
                raise ValueError(f"`eos_token_id` has to be a list of positive integers, but is {eos_token_id}")
            eos_token_id = eos_token_id.reshape(-1).tolist()
        if isinstance(eos_token_id, int):
            eos_token_id = [eos_token_id]
        if len(eos_token_id) != 1 or eos_token_id[0] < 0:
            raise ValueError(f"`eos_token_id` has to be a list of positive integers, but is {eos_token_id}")
        self.eos_token_id = int(eos_token_id[0])
        self.batch_size, self.num_codebooks, self.device = batch_size, num_codebooks, device
        self.first_codebooks_unfinished = torch.arange(batch_size, device=device, dtype=torch.int64) * num_codebooks

    def __call__(self, input_ids: torch.LongTensor, scores: torch.FloatTensor) -> torch.FloatTensor:
        ids = input_ids.to(torch.int64).contiguous()
        if scores.dtype != torch.float32 or not scores.is_contiguous():
            raise ValueError("scores must be a contiguous float32 tensor (as `_sample` passes it)")
        _lib.check(_lib.lib().ptts_logits_processor(_lib.ptr(ids), ids.shape[0], ids.shape[1], ids.shape[1], _lib.ptr(scores),
                                                    scores.shape[1], self.eos_token_id, self.num_codebooks,
                                                    _lib.ptr(self.first_codebooks_unfinished), _lib.stream_ptr()))
        return scores  # mutated in place like the reference (:52)


# ---- decoder engine ------------------------------------------------------------------------------
def _decoder_config_c(cfg: ParlerTTSDecoderConfig, dtype: torch.dtype) -> _lib.DecoderConfigC:
    c = _lib.DecoderConfigC()
    c.hidden_size = cfg.hidden_size
    c.num_layers = cfg.num_hidden_layers
    c.num_heads = cfg.num_attention_heads
    c.num_kv_heads = cfg.num_key_value_heads
    c.num_cross_kv_heads = cfg.num_cross_attention_key_value_heads
    c.ffn_dim = cfg.ffn_dim
    c.vocab_size = cfg.vocab_size
    c.num_codebooks = cfg.num_codebooks
    c.max_positions = cfg.max_position_embeddings
    c.rope = 1 if cfg.rope_embeddings else 0
    if cfg.activation_function not in _ACT:
        raise ValueError(f"activation_function {cfg.activation_function!r} is not supported by the B200 decoder kernels")
    c.activation = _ACT[cfg.activation_function]
    c.dtype = _lib.dtype_code(dtype)
    c.bos_token_id, c.pad_token_id, c.eos_token_id = cfg.bos_token_id, cfg.pad_token_id, cfg.eos_token_id
    c.rope_theta = float(cfg.rope_theta)
    c.layer_norm_eps = float(getattr(cfg, "layer_norm_eps", 1e-5))
    if cfg.hidden_size // cfg.num_attention_heads != 64:
        raise ValueError("the B200 decoder kernels are specialised for head_dim == 64 (Parler-TTS Mini and Large)")
    return c


def _sinusoidal_table(n: int, dim: int) -> torch.Tensor:
    # ParlerTTSSinusoidalPositionalEmbedding.get_embedding semantics (:346-359): [cos | sin] halves
    half = dim // 2
    e = math.log(10000) / (half - 1)
    e = torch.exp(torch.arange(half, dtype=torch.int64).float() * -e)
    e = torch.arange(n, dtype=torch.int64).float().unsqueeze(1) * e.unsqueeze(0)
    return torch.cat([torch.cos(e), torch.sin(e)], dim=1)


def _rope_tables(cfg: ParlerTTSDecoderConfig):
    # ParlerTTSRotaryEmbedding (:380, :394-406): fp32 cos/sin of position x inv_freq, duplicated halves
    hd = cfg.hidden_size // cfg.num_attention_heads
    inv = 1.0 / (cfg.rope_theta ** (torch.arange(0, hd, 2, dtype=torch.int64).float() / hd))
    fr = torch.arange(cfg.max_position_embeddings, dtype=torch.int64).float()[:, None] * inv[None, :]
    emb = torch.cat((fr, fr), dim=-1)
    return emb.cos(), emb.sin()


class DecoderEngine:
    """Packed decoder weights on one GPU + generation sessions.  One instance per model per device."""

    def __init__(self, cfg: ParlerTTSDecoderConfig, device, dtype: torch.dtype):
        self.cfg, self.device, self.dtype = cfg, torch.device(device), dtype
        self.c = _decoder_config_c(cfg, dtype)
        n = C.c_int64()
        _lib.check(_lib.lib().ptts_decoder_blob_bytes(C.byref(self.c), C.byref(n)))
        self.blob = torch.zeros(n.value, dtype=torch.uint8, device=self.device)
        self._sessions: dict[tuple, "GenSession"] = {}

    def _pack(self, tid: int, index: int, t: torch.Tensor):
        t = t.to(device=self.device)
        if t.dtype not in (torch.float32, torch.bfloat16):
            t = t.float()
        t = t.contiguous()
        rows, cols = (t.shape[0], t.numel() // t.shape[0]) if t.dim() >= 2 else (1, t.numel())
        _lib.check(_lib.lib().ptts_decoder_pack(C.byref(self.c), _lib.ptr(self.blob), tid, index, _lib.ptr(t),
                                                _lib.dtype_code(t.dtype), rows, cols, _lib.stream_ptr()))

    def load_state_dict(self, sd: dict[str, torch.Tensor], prefix: str = "decoder."):
        """sd uses the reference's parameter names (ParlerTTSForConditionalGeneration.state_dict())."""
        cfg, L = self.cfg, _lib
        p = prefix + "model.decoder."
        need = lambda k: sd[k] if k in sd else (_ for _ in ()).throw(ValueError(f"missing weight {k}"))
        for k in range(cfg.num_codebooks):
            self._pack(L.T_EMBED_TOKENS, k, need(f"{p}embed_tokens.{k}.weight"))
            self._pack(L.T_LM_HEAD, k, self._head(sd, prefix, k))
        if cfg.rope_embeddings:
            cos, sin = _rope_tables(cfg)
            self._pack(L.T_ROPE_COS, 0, cos)
            self._pack(L.T_ROPE_SIN, 0, sin)
        else:
            key = f"{p}embed_positions.weights"
            self._pack(L.T_POS_TABLE, 0, sd[key] if key in sd else _sinusoidal_table(cfg.max_position_embeddings, cfg.hidden_size))
        names = [("self_attn_layer_norm.weight", L.T_LN1_W), ("self_attn_layer_norm.bias", L.T_LN1_B),
                 ("self_attn.q_proj.weight", L.T_SELF_Q), ("self_attn.k_proj.weight", L.T_SELF_K),
                 ("self_attn.v_proj.weight", L.T_SELF_V), ("self_attn.out_proj.weight", L.T_SELF_O),
                 ("encoder_attn_layer_norm.weight", L.T_LN2_W), ("encoder_attn_layer_norm.bias", L.T_LN2_B),
                 ("encoder_attn.q_proj.weight", L.T_CROSS_Q), ("encoder_attn.k_proj.weight", L.T_CROSS_K),
                 ("encoder_attn.v_proj.weight", L.T_CROSS_V), ("encoder_attn.out_proj.weight", L.T_CROSS_O),
                 ("final_layer_norm.weight", L.T_LN3_W), ("final_layer_norm.bias", L.T_LN3_B),
                 ("fc1.weight", L.T_FC1), ("fc2.weight", L.T_FC2)]
        for i in range(cfg.num_hidden_layers):
            for nm, tid in names:
                self._pack(tid, i, need(f"{p}layers.{i}.{nm}"))
        self._pack(L.T_FINAL_LN_W, 0, need(p + "layer_norm.weight"))
        self._pack(L.T_FINAL_LN_B, 0, need(p + "layer_norm.bias"))
        _lib.check(_lib.lib().ptts_decoder_finalize(C.byref(self.c), _lib.ptr(self.blob), _lib.stream_ptr()))
        torch.cuda.current_stream().synchronize()
        return self

    def _head(self, sd, prefix, k):
        if f"{prefix}lm_heads.{k}.weight" in sd:
            return sd[f"{prefix}lm_heads.{k}.weight"]
        if f"{prefix}lm_heads.weight" in sd:  # use_fused_lm_heads (:1836): [K*V, H]
            V = self.cfg.vocab_size
            return sd[f"{prefix}lm_heads.weight"][k * V:(k + 1) * V]
        raise ValueError(f"missing weight {prefix}lm_heads.{k}.weight")

    def session(self, B: int, P: int, S: int, max_cache_len: int, max_prefix: int = 1) -> "GenSession":
        key = (B, P, S)
        s = self._sessions.get(key)
        if s is None or s.max_cache_len < max_cache_len or s.max_prefix < max_prefix:
            if s is not None:
                s.close()
            s = GenSession(self, B, P, S, max_cache_len, max_prefix)
            self._sessions = {key: s}  # keep one live session (the reference keeps one `_cache`, :3254-3309)
        return s


class GenSession:
    """Device-resident generation state for (B, P, S): KV caches, token history, processor state."""

    def __init__(self, eng: DecoderEngine, B: int, P: int, S: int, max_cache_len: int, max_prefix: int = 1):
        self.eng, self.B, self.P, self.S, self.max_cache_len, self.max_prefix = eng, B, P, S, max_cache_len, max_prefix
        lib = _lib.lib()
        n = C.c_int64()
        _lib.check(lib.ptts_workspace_bytes_ex(C.byref(eng.c), B, P, S, max_cache_len, max_prefix, C.byref(n)))
        self.ws = torch.zeros(n.value, dtype=torch.uint8, device=eng.device)
        h = C.c_void_p()
        _lib.check(lib.ptts_session_create_ex(C.byref(eng.c), _lib.ptr(eng.blob), _lib.ptr(self.ws), n.value, B, P, S,
                                              max_cache_len, max_prefix, C.byref(h)))
        self.h = h
        self.K, self.V = eng.cfg.num_codebooks, eng.cfg.vocab_size
        self._keep: list[Any] = []
        self._forced = None

    def close(self):
        if self.h is not None:
            _lib.lib().ptts_session_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _view(self, fn, shape, dtype):
        p = C.c_void_p()
        _lib.check(fn(self.h, C.byref(p)))
        off = p.value - self.ws.data_ptr()
        n = int(torch.tensor(shape).prod()) * torch.empty((), dtype=dtype).element_size()
        return self.ws[off:off + n].view(dtype).view(*shape)

    @property
    def logits(self) -> torch.Tensor:
        return self._view(_lib.lib().ptts_session_logits, (self.B * self.K, self.V), torch.float32)

    @property
    def scores(self) -> torch.Tensor:
        return self._view(_lib.lib().ptts_session_scores, (self.B * self.K, self.V), torch.float32)

    @property
    def raw_ids(self) -> torch.Tensor:
        p, ld = C.c_void_p(), C.c_int32()
        _lib.check(_lib.lib().ptts_session_raw_ids(self.h, C.byref(p), C.byref(ld)))
        off = p.value - self.ws.data_ptr()
        return self.ws[off:off + self.B * self.K * ld.value * 8].view(torch.int64).view(self.B * self.K, ld.value)

    @property
    def state(self) -> torch.Tensor:
        """int32 [8]: cur_len, active, n_unfinished, done_blocks, steps_run, ..."""
        return self._view(_lib.lib().ptts_session_state, (8,), torch.int32)

    @property
    def launches(self) -> int:
        n = C.c_int64()
        _lib.check(_lib.lib().ptts_session_launches(self.h, C.byref(n)))
        return n.value

    @property
    def fused(self) -> int:
        """0: decode steps use the multi-kernel path; 1: the fused persistent step kernel (one launch per token, step.cu);
        2: its cluster variant (step2.cu: one cluster per head, 6 device-wide phases per layer)."""
        n = C.c_int32()
        _lib.check(_lib.lib().ptts_session_fused(self.h, C.byref(n)))
        return n.value

    def begin(self, max_length: int, do_sample=False, temperature=1.0, top_k=0, top_p=1.0, min_new_tokens=0, seed=0,
              suppress_special=False, codebook_size=1024, row_base=0):
        g = _lib.GenParamsC()
        g.max_length, g.min_new_tokens, g.do_sample = int(max_length), int(min_new_tokens or 0), int(bool(do_sample))
        g.top_k, g.top_p, g.temperature = int(top_k or 0), float(1.0 if top_p is None else top_p), float(temperature or 1.0)
        g.seed, g.suppress_special, g.codebook_size = int(seed) & (2 ** 64 - 1), int(bool(suppress_special)), int(codebook_size)
        g.row_base = int(row_base)  # global row of this shard's first (utterance, codebook) stream: Philox substream key
        _lib.check(_lib.lib().ptts_generate_begin(self.h, C.byref(g), _lib.stream_ptr()))
        self.max_length = int(max_length)

    def prefill(self, prompt_hidden, prompt_mask, enc_hidden, enc_mask, prefix_ids=None):
        """prefix_ids: None (the BOS column begin() staged) or [B*K, n] delay-patterned decoder ids (ptts_prefill_ids)."""
        dt, dev = self.eng.dtype, self.eng.device
        H = self.eng.cfg.hidden_size
        enc_hidden = enc_hidden.to(device=dev, dtype=dt).contiguous()
        if tuple(enc_hidden.shape) != (self.B, self.S, H):
            raise ValueError(f"encoder states must be [{self.B}, {self.S}, {H}], got {tuple(enc_hidden.shape)}")
        if self.P > 0:
            if prompt_hidden is None:
                raise ValueError("prompt_hidden_states are required for a session created with P > 0")
            prompt_hidden = prompt_hidden.to(device=dev, dtype=dt).contiguous()
            if tuple(prompt_hidden.shape) != (self.B, self.P, H):
                raise ValueError(f"prompt states must be [{self.B}, {self.P}, {H}], got {tuple(prompt_hidden.shape)}")
        pm = None if prompt_mask is None else prompt_mask.to(device=dev, dtype=torch.int64).contiguous()
        em = None if enc_mask is None else enc_mask.to(device=dev, dtype=torch.int64).contiguous()
        if prefix_ids is None:
            self._keep = [prompt_hidden, enc_hidden, pm, em]
            _lib.check(_lib.lib().ptts_prefill(self.h, _lib.ptr(prompt_hidden) if self.P > 0 else None, _lib.ptr(pm),
                                               _lib.ptr(enc_hidden), _lib.ptr(em), _lib.stream_ptr()))
            return
        ids = prefix_ids.to(device=dev, dtype=torch.int64).contiguous()
        if ids.dim() != 2 or ids.shape[0] != self.B * self.K:
            raise ValueError(f"prefix ids must be [{self.B * self.K}, n], got {tuple(ids.shape)}")
        if bool(((ids < 0) | (ids > self.V)).any()):
            raise ValueError(f"prefix ids must lie in [0, {self.V}] (the embedding tables have vocab_size + 1 rows)")
        self._keep = [prompt_hidden, enc_hidden, pm, em, ids]
        _lib.check(_lib.lib().ptts_prefill_ids(self.h, _lib.ptr(prompt_hidden) if self.P > 0 else None, _lib.ptr(pm),
                                               _lib.ptr(enc_hidden), _lib.ptr(em), _lib.ptr(ids), ids.shape[1], _lib.stream_ptr()))

    def decode_forward(self):
        _lib.check(_lib.lib().ptts_decode_forward(self.h, _lib.stream_ptr()))

    def sample(self, forced: Optional[torch.Tensor] = None):
        f = None if forced is None else forced.to(device=self.eng.device, dtype=torch.int64).contiguous()
        self._forced = f   # keep the staging tensor alive until the next call (the launch is asynchronous); never accumulates
        _lib.check(_lib.lib().ptts_sample(self.h, _lib.ptr(f), _lib.stream_ptr()))

    def decode_steps(self, n: int):
        _lib.check(_lib.lib().ptts_decode_steps(self.h, int(n), _lib.stream_ptr()))


# ---- model classes -------------------------------------------------------------------------------
class GenerateOutput(dict):
    """Stands in for HF's GenerateEncoderDecoderOutput: .sequences plus ["audios_length"] (:3648-3651)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


class ParlerTTSCache:
    """`past_key_values` of ParlerTTSForCausalLM.forward: the device session that owns the pre-allocated self-attention K/V
    cache (append in place at cache_position) and the cross-attention K/V projected once at the first call -- the roles of
    EncoderDecoderCache(StaticCache, StaticCache) in the reference (:3254-3309)."""

    def __init__(self, session: "GenSession"):
        self.session = session
        self.steps = 0
        self.n_first = 1   # decoder columns of the first call (> 1: a voice-prompt prefix)

    def get_seq_length(self) -> int:
        return self.session.P + self.n_first + self.steps

    def get_max_cache_shape(self) -> int:
        return self.session.max_cache_len


class ParlerTTSForCausalLM:
    """Decoder + K LM heads as a step operator over a KV-cached session (reference :1824-1974)."""

    def __init__(self, config: ParlerTTSDecoderConfig, device="cuda", dtype=torch.bfloat16):
        self.config = config
        self.num_codebooks = config.num_codebooks
        self.vocab_size = config.vocab_size
        self.device, self.dtype = torch.device(device), dtype
        self.engine = DecoderEngine(config, device, dtype)

    def load_state_dict(self, sd, prefix=""):
        self.engine.load_state_dict(sd, prefix=prefix)
        return self

    def build_delay_pattern_mask(self, input_ids, bos_token_id, pad_token_id, max_length):
        return build_delay_pattern_mask(input_ids, bos_token_id, pad_token_id, max_length, self.num_codebooks)

    @torch.no_grad()
    def forward(self, input_ids: torch.LongTensor = None, attention_mask=None, encoder_hidden_states=None,
                encoder_attention_mask=None, prompt_hidden_states=None, prompt_attention_mask=None, past_key_values=None,
                use_cache: bool = True, cache_position=None, return_dict: bool = True, max_cache_len: Optional[int] = None, **kwargs):
        """The step operator an HF-style loop calls (reference :1865-1974): input_ids [B*K, 1] (delay mask already applied, as
        prepare_inputs_for_generation does at :2909) -> logits [B*K, 1, V], over a KV cache kept in `past_key_values`.

        * first call (past_key_values None): `encoder_hidden_states` [B, S, H] (already multiplied by their mask) and optionally
          `prompt_hidden_states` [B, P, H] are required; the prompt prefix + the given ids go through ptts_prefill and a
          ParlerTTSCache (the session: pre-allocated self- and cross-attention K/V) is returned as `past_key_values`.
          Only the LAST position's logits are materialised (what `_sample` reads): shape [B*K, 1, V], not [B*K, P+1, V].
        * later calls: the ids are appended (ptts_sample with forced tokens) and one cached step runs on the fused kernel
          (ptts_decode_forward).
        * the first call may also take input_ids [B*K, n] (a delay-patterned voice-prompt prefix, column 0 = BOS): the n columns go
          through ptts_prefill_ids in one forward and get_seq_length() counts them.
        Later calls with more than one column, `inputs_embeds`, `labels` and `use_cache=False` belong to training / the no-cache
        path and are outside this operator (ValueError)."""
        if kwargs.get("inputs_embeds") is not None or kwargs.get("labels") is not None or not use_cache:
            raise ValueError("ParlerTTSForCausalLM.forward on the B200 path is the cached decode-step operator: input_ids [B*K, 1], use_cache=True")
        n_cols = 1 if past_key_values is not None else (input_ids.shape[-1] if input_ids is not None and input_ids.dim() == 2 else 0)
        if input_ids is None or input_ids.dim() != 2 or input_ids.shape[1] != n_cols or n_cols < 1 or input_ids.shape[0] % self.num_codebooks != 0:
            raise ValueError(f"input_ids must be [batch * num_codebooks, 1] (or [batch * num_codebooks, n] on the first call), got "
                             f"{None if input_ids is None else tuple(input_ids.shape)}")
        B = input_ids.shape[0] // self.num_codebooks
        ids = input_ids[:, 0].to(self.device, torch.int64).contiguous()
        if past_key_values is None:
            if encoder_hidden_states is None:
                raise ValueError("the first call needs `encoder_hidden_states`")
            S = encoder_hidden_states.shape[1]
            P = 0 if prompt_hidden_states is None else prompt_hidden_states.shape[1]
            cap = int(max_cache_len or self.config.max_position_embeddings)
            sess = GenSession(self.engine, B, P, S, cap, max_prefix=n_cols)   # an independent cache, not generate()'s shared session
            sess.begin(cap - P, do_sample=False)
            if not bool((ids == self.config.bos_token_id).all()):
                raise ValueError("the first call must feed the decoder start (BOS) column")
            sess.prefill(prompt_hidden_states, prompt_attention_mask if P > 0 else None, encoder_hidden_states, encoder_attention_mask,
                         prefix_ids=input_ids if n_cols > 1 else None)
            past_key_values = ParlerTTSCache(sess)
            past_key_values.n_first = n_cols
        else:
            if not isinstance(past_key_values, ParlerTTSCache) or past_key_values.session.B != B:
                raise ValueError("past_key_values must be the ParlerTTSCache returned by the first call (same batch)")
            sess = past_key_values.session
            sess.sample(forced=ids)
            sess.decode_forward()
            past_key_values.steps += 1
        logits = sess.logits.clone().unsqueeze(1)   # [B*K, 1, V] fp32
        if not return_dict:
            return (logits, past_key_values)
        return GenerateOutput(logits=logits, past_key_values=past_key_values)

    __call__ = forward

    @staticmethod
    def apply_delay_pattern_mask(input_ids, decoder_pad_token_mask):
        return apply_delay_pattern_mask(input_ids, decoder_pad_token_mask)


class ParlerTTSForConditionalGeneration:
    """generate(): description/prompt conditioning -> audio tokens -> waveform, hot path on sm_100a kernels."""

    config_class = ParlerTTSConfig
    main_input_name = "input_ids"
    # model kwargs generate() understands (reference: _validate_model_kwargs over forward()'s signature)
    _MODEL_KWARGS = frozenset({"input_ids", "attention_mask", "prompt_input_ids", "prompt_attention_mask", "prompt_hidden_states",
                               "encoder_outputs", "input_values", "decoder_input_ids", "padding_mask", "use_cache",
                               "cache_implementation", "output_attentions", "output_hidden_states", "output_scores"})
    # GenerationConfig fields the device loop does not implement, with the value that means "off"
    _NEUTRAL_GENERATION_KNOBS = {"num_return_sequences": 1, "num_beam_groups": 1, "repetition_penalty": 1.0, "no_repeat_ngram_size": 0,
                                 "length_penalty": 1.0, "typical_p": 1.0, "epsilon_cutoff": 0.0, "eta_cutoff": 0.0, "min_length": 0,
                                 "penalty_alpha": None, "bad_words_ids": None, "force_words_ids": None, "guidance_scale": None}

    def __init__(self, config: ParlerTTSConfig, device="cuda", dtype=torch.bfloat16, text_encoder=None):
        if not isinstance(config, ParlerTTSConfig):
            raise ValueError(f"Config: {config} has to be of type {self.config_class}")
        self.config = config
        self.device, self.dtype = torch.device(device), dtype
        self.decoder = ParlerTTSForCausalLM(config.decoder, device, dtype)
        self.audio_encoder = DACModel(config.audio_encoder, device, dtype)
        self.text_encoder = text_encoder  # a torch module (T5 encoder) or None; not part of the replaced path
        self.prompt_cross_attention = config.prompt_cross_attention
        if self.prompt_cross_attention:
            raise ValueError("prompt_cross_attention=True checkpoints are not supported by the B200 path yet")
        # Side-input parameters exist (zero-filled) from construction on, with shapes that depend on the config only, so every
        # rank of a sharded run issues the SAME list of broadcasts at init (dist.broadcast_model_weights); `_side_loaded`
        # says whether they hold real weights.  enc_to_dec_proj exists iff the text encoder's width differs (:2388-2392).
        dd = config.decoder
        self.embed_prompts_weight: torch.Tensor = torch.zeros(config.vocab_size, dd.hidden_size, device=self.device, dtype=dtype)
        te_hidden = (config.text_encoder or {}).get("d_model", (config.text_encoder or {}).get("hidden_size"))
        self.enc_to_dec_proj: Optional[tuple] = None
        if te_hidden is not None and int(te_hidden) != dd.hidden_size:
            self.enc_to_dec_proj = (torch.zeros(dd.hidden_size, int(te_hidden), device=self.device, dtype=dtype),
                                    torch.zeros(dd.hidden_size, device=self.device, dtype=dtype))
        self._side_loaded = False
        self.use_audio_scales = True   # DACModel.decode has an `audio_scales` parameter (:2416-2417)
        self.use_4dim_audio_codes = True  # dac_on_the_hub (:2419-2422, quirk Q14)
        d = config.decoder
        self.generation_config = GenerationConfig(
            max_length=int(30 * config.audio_encoder.frame_rate), do_sample=True, bos_token_id=d.bos_token_id,
            pad_token_id=d.pad_token_id, eos_token_id=d.eos_token_id, decoder_start_token_id=d.bos_token_id)

    # -- weights -----------------------------------------------------------------------------------
    def load_state_dict(self, sd: dict[str, torch.Tensor], dac_state_dict: Optional[dict] = None):
        self.decoder.engine.load_state_dict(sd, prefix="decoder.")
        if "embed_prompts.weight" in sd:
            w = sd["embed_prompts.weight"].to(self.device, self.dtype)
            if w.shape == self.embed_prompts_weight.shape:
                self.embed_prompts_weight.copy_(w)
            else:  # a checkpoint whose text vocabulary differs from config.vocab_size: follow the checkpoint
                self.embed_prompts_weight = w.contiguous()
            self._side_loaded = True
        if "enc_to_dec_proj.weight" in sd:
            w, b = sd["enc_to_dec_proj.weight"].to(self.device, self.dtype), sd["enc_to_dec_proj.bias"].to(self.device, self.dtype)
            if self.enc_to_dec_proj is not None and self.enc_to_dec_proj[0].shape == w.shape:
                self.enc_to_dec_proj[0].copy_(w); self.enc_to_dec_proj[1].copy_(b)
            else:
                self.enc_to_dec_proj = (w.contiguous(), b.contiguous())
        ae = {k[len("audio_encoder."):]: v for k, v in sd.items() if k.startswith("audio_encoder.")}
        if dac_state_dict is not None:
            ae = dac_state_dict
        if ae:
            self.audio_encoder.load_state_dict(ae)
        return self

    @classmethod
    def from_pretrained(cls, path: str, device="cuda", torch_dtype=torch.bfloat16, **kwargs):
        """Load a local reference checkpoint directory (config.json + *.safetensors)."""
        config = ParlerTTSConfig.from_pretrained(path)
        from safetensors.torch import load_file
        sd = {}
        for f in sorted(os.listdir(path)):
            if f.endswith(".safetensors"):
                sd.update(load_file(os.path.join(path, f)))
        if not sd:
            raise ValueError(f"no .safetensors weights found under {path}")
        text_encoder = None
        te = {k[len("text_encoder."):]: v for k, v in sd.items() if k.startswith("text_encoder.")}
        if te and config.text_encoder:
            from transformers import AutoConfig, AutoModelForTextEncoding
            tcfg = dict(config.text_encoder)
            tc = AutoConfig.for_model(tcfg.pop("model_type"), **tcfg)
            text_encoder = AutoModelForTextEncoding.from_config(tc)
            text_encoder.load_state_dict(te, strict=False)
            text_encoder = text_encoder.to(device=device, dtype=torch_dtype).eval()
        m = cls(config, device=device, dtype=torch_dtype, text_encoder=text_encoder)
        m.load_state_dict(sd)
        gpath = os.path.join(path, "generation_config.json")
        if os.path.exists(gpath):
            with open(gpath) as f:
                m.generation_config.update(**json.load(f))
        return m

    def to(self, *a, **k):
        return self

    def eval(self):
        return self

    # -- side inputs (not replaced; PyTorch) -------------------------------------------------------
    def _encode_text_eager(self, input_ids, attention_mask):
        enc_mask = attention_mask
        if attention_mask is not None and attention_mask.dim() == 2:
            # the 4-D additive form HF derives from a 2-D padding mask (0 keep / finfo.min drop), built here with device ops only:
            # the library's own conversion creates CPU scalars on the way, which a CUDA-graph capture cannot contain
            edt = next(self.text_encoder.parameters()).dtype
            enc_mask = (1 - attention_mask)[:, None, None, :].to(edt) * torch.finfo(edt).min
        h = self.text_encoder(input_ids=input_ids, attention_mask=enc_mask, return_dict=True).last_hidden_state
        if self.enc_to_dec_proj is not None:
            h = torch.nn.functional.linear(h, *self.enc_to_dec_proj)        # :2388-2392 / :3087-3090
        if attention_mask is not None:
            h = h * attention_mask[..., None]                               # :3092-3093
        return h.to(self.dtype)

    def _encode_text(self, input_ids, attention_mask):
        """Description ids -> encoder_hidden_states (reference :3048-3097): T5 encoder + enc_to_dec_proj + mask multiply.
        These PyTorch modules are not replaced (SURVEY section 8 f3); what this path adds is ONE CUDA graph per (batch, length) shape
        over the whole chain -- a T5 encoder is ~150 small launches whose launch latency, not their math, is the time-to-first-audio
        once the decode loop is fast.  Inputs are copied into static buffers and the graph is replayed; if capture is impossible
        (a module that synchronises), the eager path is used and said so once."""
        if self.text_encoder is None:
            raise ValueError("this model was built without a text encoder: pass `encoder_outputs`")
        input_ids = input_ids.to(self.device)
        attention_mask = None if attention_mask is None else attention_mask.to(self.device)
        if not hasattr(self, "_enc_graphs"):
            self._enc_graphs, self._enc_graph_ok = {}, True
        if not self._enc_graph_ok or self.device.type != "cuda":
            return self._encode_text_eager(input_ids, attention_mask)
        key = (tuple(input_ids.shape), attention_mask is not None)
        entry = self._enc_graphs.get(key)
        if entry is None:
            try:
                s_ids = input_ids.clone()
                s_mask = None if attention_mask is None else attention_mask.clone()
                side = torch.cuda.Stream(device=self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    for _ in range(2):                                   # warm-up: lazy initialisations happen outside the capture
                        self._encode_text_eager(s_ids, s_mask)
                torch.cuda.current_stream(self.device).wait_stream(side)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    s_out = self._encode_text_eager(s_ids, s_mask)
                entry = (graph, s_ids, s_mask, s_out)
                if len(self._enc_graphs) >= 16:
                    self._enc_graphs.clear()
                self._enc_graphs[key] = entry
            except Exception as ex:  # pragma: no cover - depends on the encoder implementation
                import warnings
                warnings.warn(f"text-encoder CUDA graph capture failed ({ex!r}); running the encoder eagerly")
                self._enc_graph_ok = False
                torch.cuda.synchronize(self.device)
                return self._encode_text_eager(input_ids, attention_mask)
        graph, s_ids, s_mask, s_out = entry
        s_ids.copy_(input_ids)
        if s_mask is not None:
            s_mask.copy_(attention_mask)
        graph.replay()
        return s_out.clone()

    # -- generate with user-supplied processors / stopping criteria --------------------------------
    def _host_driven_loop(self, sess: "GenSession", gc, max_length, user_processors, user_criteria, streamer, seed):
        """One host iteration per token, like GenerationMixin._sample: the decoder step still runs on the fused kernel
        (ptts_decode_forward), the built-in processors run as their device operators (MinNewTokens as a mask,
        ParlerTTSLogitsProcessor = ptts_logits_processor), then the caller's `logits_processor` list, the HF warpers and the draw
        as torch ops on the device scores, and the token is appended with ptts_sample(forced).  Used only when the caller passes
        processors or criteria the device loop does not know (the reference merges such lists at :3540-3552)."""
        d = self.config.decoder
        K, BK = d.num_codebooks, sess.B * d.num_codebooks
        parler = ParlerTTSLogitsProcessor(d.eos_token_id, K, sess.B, self.device)
        gen = torch.Generator(device=self.device).manual_seed(int(seed))
        unfinished = torch.ones(BK, dtype=torch.long, device=self.device)
        cur = 1
        while True:
            ids = sess.raw_ids[:, :cur]
            scores = sess.logits.clone()
            if (gc.min_new_tokens or 0) > 0 and cur - 1 < gc.min_new_tokens:
                scores[:, d.eos_token_id] = -float("inf")
            scores = parler(ids, scores)
            for proc in user_processors:
                scores = proc(ids, scores)
            if gc.do_sample:
                if gc.temperature and gc.temperature != 1.0:
                    scores = scores / gc.temperature
                if gc.top_k:
                    kth = torch.topk(scores, min(int(gc.top_k), scores.shape[-1]))[0][..., -1, None]
                    scores = scores.masked_fill(scores < kth, -float("inf"))
                if gc.top_p is not None and gc.top_p < 1.0:
                    ss, si = torch.sort(scores, descending=False)
                    rem = ss.softmax(-1).cumsum(-1) <= (1 - gc.top_p)
                    rem[..., -1:] = False
                    scores = scores.masked_fill(rem.scatter(1, si, rem), -float("inf"))
                nxt = torch.multinomial(scores.softmax(-1), 1, generator=gen).squeeze(1)
            else:
                nxt = scores.argmax(-1)
            nxt = nxt * unfinished + d.pad_token_id * (1 - unfinished)
            sess.sample(forced=nxt)           # append (+ delay-pattern override of the next input), device-side stopping state
            cur += 1
            if streamer is not None:
                streamer.put(nxt.cpu())
            unfinished = unfinished & ~((nxt == d.eos_token_id) | (cur >= max_length)).long()
            stop = unfinished.max().item() == 0
            for crit in user_criteria:
                r = crit(sess.raw_ids[:, :cur], scores)
                r = r if isinstance(r, torch.Tensor) else torch.full((BK,), bool(r), device=self.device)
                unfinished = unfinished & ~r.long()
                stop = stop or unfinished.max().item() == 0
            if stop:
                break
            sess.decode_forward()
        if streamer is not None:
            streamer.end()

    def _fused_batch_limit(self):
        """Rows one fused decode-step launch covers (None: the fused kernels are not in play, the batch runs as one session)."""
        if self.dtype != torch.bfloat16 or os.environ.get("PTTS_FUSED", "1") == "0":
            return None
        return 32

    def _run_token_loop(self, enc_hidden, attention_mask, prompt_hidden, prompt_mask, *, gc, max_length, seed, suppress_special, row_base,
                        streamer=None, custom=None, prefix=None, forced=None):
        """begin + prefill + the token loop of one session; returns the raw token matrix [B * K, generated length].

        prefix [B*K, n]: the model's first n input columns of a voice-prompt continuation (delay-patterned, column 0 = BOS);
        forced [B*K, max_length]: the prompt codes the delay pattern puts after the prefix (codebook k: columns n .. n+k-1), -1
        elsewhere."""
        d = self.config.decoder
        K = d.num_codebooks
        B, S, _ = enc_hidden.shape
        P = 0 if prompt_hidden is None else prompt_hidden.shape[1]
        n = 1 if prefix is None else prefix.shape[1]
        sess = self.decoder.engine.session(B, P, S, P + max_length, max_prefix=n)
        # MinNewTokensLengthLogitsProcessor skips the n prompt columns (:3540-3547); the kernel tests cur_len - 1 < min_new_tokens
        min_new = gc.min_new_tokens or 0
        if min_new > 0:
            min_new += n - 1
        sess.begin(max_length, do_sample=gc.do_sample, temperature=gc.temperature, top_k=gc.top_k if gc.do_sample else 0,
                   top_p=gc.top_p, min_new_tokens=min_new, seed=seed, suppress_special=suppress_special,
                   codebook_size=self.config.audio_encoder.codebook_size, row_base=row_base)
        if streamer is not None:
            delayed = torch.full((B * K, 1), d.bos_token_id, dtype=torch.int64)
            streamer.put(delayed)
        sess.prefill(prompt_hidden, prompt_mask, enc_hidden, attention_mask, prefix_ids=prefix)
        if custom is not None:
            self._host_driven_loop(sess, gc, max_length, custom[0], custom[1], streamer, seed)
        elif streamer is not None:
            sess.sample()
            steps_left = max_length - 2
            # the streamer contract is one host-visible token column per step (_sample -> streamer.put(next.cpu()))
            col = 1
            streamer.put(sess.raw_ids[:, col].cpu())
            while steps_left > 0 and int(sess.state[1].item()) == 1:
                sess.decode_steps(1)
                col += 1
                steps_left -= 1
                streamer.put(sess.raw_ids[:, col].cpu())
            streamer.end()
        else:
            # After a prefix, the first K-1 columns run one step at a time with the pattern's prompt codes forced (a negative entry
            # draws).  That matches the reference in output and in stopping: the Parler processor lets codebook k draw EOS at
            # column n + k at the earliest and first_codebooks_unfinished moves by at most one per step, so a forced cell never
            # holds a drawn EOS there; the reference's history differs only in cells its final mask overwrites.
            sess.sample(None if prefix is None else forced[:, n])
            col = n + 1
            while prefix is not None and col < min(n + K - 1, max_length):
                sess.decode_forward()
                sess.sample(forced[:, col])
                col += 1
            steps_left = max_length - col
            # no per-step host sync: enqueue graph replays in chunks and poll the device `active` flag between chunks
            chunk = 64
            while steps_left > 0:
                n = min(chunk, steps_left)
                sess.decode_steps(n)
                steps_left -= n
                if steps_left > 0 and int(sess.state[1].item()) == 0:
                    break
        cur_len = int(sess.state[0].item())
        return sess.raw_ids[:, :cur_len].clone()

    # -- generate ----------------------------------------------------------------------------------
    @torch.no_grad()
    def generate(self, inputs: Optional[torch.Tensor] = None, generation_config: Optional[GenerationConfig] = None,
                 logits_processor=None, stopping_criteria=None, synced_gpus=None, streamer=None, **kwargs):
        """Same call contract as the reference generate() (:3322-3653) for greedy / sampling modes.

        Extra kwargs: `seed` (Philox key for sampling, default 0), `return_codes` (also return audio codes).
        """
        import copy
        gc = copy.deepcopy(generation_config if generation_config is not None else self.generation_config)
        seed = kwargs.pop("seed", 0)
        row_base = kwargs.pop("row_base", 0)   # batch shards: global (utterance x codebook) row of this shard's first row (dist.py)
        return_codes = kwargs.pop("return_codes", False)
        suppress_special = kwargs.pop("_suppress_special", False)
        user_max_length = kwargs.get("max_length")
        mk = gc.update(**kwargs)
        # The reference would honour (or reject) every generation knob; silently dropping one changes the output without an error.
        unknown = sorted(k for k in mk if k not in self._MODEL_KWARGS)
        if unknown:
            raise ValueError(f"The following `model_kwargs` are not used by the model: {unknown} (note: typos in the generate "
                             "arguments will also show up in this list)")
        for k in ("use_cache", "cache_implementation", "output_attentions", "output_hidden_states", "output_scores"):
            mk.pop(k, None)   # accepted for call compatibility: the device loop always uses its static cache
        unsupported = {k: getattr(gc, k) for k, neutral in self._NEUTRAL_GENERATION_KNOBS.items() if getattr(gc, k, neutral) != neutral}
        if unsupported:
            raise ValueError(f"generation options {unsupported} are not supported by the B200 device loop "
                             "(greedy / temperature / top-k / top-p sampling with min_new_tokens only)")
        if gc.num_beams != 1:
            raise ValueError("Got incompatible mode for generation, should be one of greedy or sampling. "
                             "Ensure that beam search is de-activated by setting `num_beams=1` and `num_beam_groups=1`.")
        custom_loop = bool(logits_processor) or bool(stopping_criteria)   # merged with the built-in ones like :3540-3552
        prefix = mk.get("decoder_input_ids")
        if (prefix is not None or mk.get("input_values") is not None) and (streamer is not None or custom_loop):
            raise ValueError("an audio prompt (decoder_input_ids / input_values) together with streamer= or user logits_processor / "
                             "stopping_criteria is not supported")
        if prefix is None and mk.get("input_values") is not None:
            # :3442-3446: the codec's codes of the reference audio, [B, K, T_a] -> [B*K, T_a]
            codes = self.audio_encoder.encode(mk["input_values"], n_quantizers=self.config.decoder.num_codebooks).audio_codes[0]
            prefix = codes.reshape(-1, codes.shape[-1])
        input_ids = mk.get("input_ids", inputs)
        attention_mask = mk.get("attention_mask")
        enc = mk.get("encoder_outputs")
        if enc is not None:
            enc_hidden = enc[0] if isinstance(enc, (tuple, list)) else getattr(enc, "last_hidden_state", enc)
        else:
            if input_ids is None:
                raise ValueError("generate() needs `input_ids` (description) or `encoder_outputs`")
            enc_hidden = self._encode_text(input_ids, attention_mask)   # encoder + enc_to_dec_proj + mask multiply, one CUDA graph
        enc_hidden = enc_hidden.to(self.device, self.dtype)
        B, S, _ = enc_hidden.shape
        prompt_hidden = mk.get("prompt_hidden_states")
        if prompt_hidden is None and mk.get("prompt_input_ids") is not None:
            if not self._side_loaded:
                raise ValueError("no embed_prompts weights loaded")
            prompt_hidden = torch.nn.functional.embedding(mk["prompt_input_ids"].to(self.device), self.embed_prompts_weight)
        prompt_mask = mk.get("prompt_attention_mask") if prompt_hidden is not None else None
        P = 0 if prompt_hidden is None else prompt_hidden.shape[1]

        d = self.config.decoder
        K = d.num_codebooks
        if prefix is not None:
            prefix = prefix.to(self.device, torch.int64)
            if prefix.dim() != 2 or prefix.shape[0] != B * K or prefix.shape[1] < 1:
                raise ValueError(f"decoder_input_ids must be [{B * K}, n], got {tuple(prefix.shape)}")
            if bool((prefix[:, 0] != d.bos_token_id).all()):   # :3017-3031: BOS column unless every row already starts with it
                prefix = torch.cat([torch.full((B * K, 1), d.bos_token_id, dtype=torch.int64, device=self.device), prefix], dim=1)
        n = 1 if prefix is None else prefix.shape[1]
        # generated length (:3458-3469): max_new_tokens wins over max_length; input_ids_length == n
        if gc.max_new_tokens is not None:
            max_length = int(gc.max_new_tokens) + n
        else:
            max_length = int(user_max_length if user_max_length is not None else gc.max_length)
        if max_length < n + 1:
            raise ValueError(f"max_length must allow at least one new token, got {max_length} for {n} decoder input columns")
        run = dict(gc=gc, max_length=max_length, seed=seed, suppress_special=suppress_special)
        pattern = forced = None
        if prefix is not None:
            # :3523-3528: the model's first input is the first n columns of the pattern built from the whole prefix; the prompt codes
            # it shifts past column n are forced where the BOS-only pattern the device applies has a free cell
            prefix, pattern = build_delay_pattern_mask(prefix, d.bos_token_id, d.pad_token_id, max_length, K)
            _, device_pattern = build_delay_pattern_mask(prefix[:, :1], d.bos_token_id, d.pad_token_id, max_length, K)
            forced = torch.where((device_pattern == -1) & (pattern != -1), pattern, torch.full_like(pattern, -1))
        limit = self._fused_batch_limit()
        if limit is not None and B > limit and not custom_loop and streamer is None:
            # The fused decode-step kernels hold one 32-row tile: a larger batch runs as consecutive shards of <= 32 utterances through
            # the same session.  The result is the one the whole batch would give: the Philox draw is keyed by the global row
            # (row_base), the processors' state is per utterance, and a finished utterance emits pad ids until the longest one ends.
            parts = []
            for b0 in range(0, B, limit):
                sl = slice(b0, min(B, b0 + limit))
                rows = slice(sl.start * K, sl.stop * K)
                parts.append(self._run_token_loop(enc_hidden[sl], None if attention_mask is None else attention_mask[sl],
                                                  None if prompt_hidden is None else prompt_hidden[sl],
                                                  None if prompt_mask is None else prompt_mask[sl], row_base=row_base + b0 * K,
                                                  prefix=None if prefix is None else prefix[rows].contiguous(),
                                                  forced=None if forced is None else forced[rows].contiguous(), **run))
            n = max(t.shape[1] for t in parts)
            output_ids = torch.cat([torch.nn.functional.pad(t, (0, n - t.shape[1]), value=d.pad_token_id) for t in parts], dim=0)
        else:
            output_ids = self._run_token_loop(enc_hidden, attention_mask, prompt_hidden, prompt_mask, row_base=row_base, streamer=streamer,
                                              custom=(logits_processor or [], stopping_criteria or []) if custom_loop else None,
                                              prefix=prefix, forced=forced, **run)

        # apply the stashed delay mask (built from the whole prefix: the output starts with the prompt's own frames), then keep only
        # the free cells (:3586-3597)
        if pattern is not None:
            full_mask = pattern
        else:
            _, full_mask = build_delay_pattern_mask(output_ids[:, :1], d.bos_token_id, d.pad_token_id, max_length, K)
        output_ids = apply_delay_pattern_mask(output_ids, full_mask)
        _, mask = build_delay_pattern_mask(output_ids[:, :1], d.bos_token_id, d.pad_token_id, output_ids.shape[1], K)
        keep = (mask != d.bos_token_id) & (mask != d.pad_token_id)
        codes = output_ids[keep].reshape(B, K, -1)
        audio_codes = codes[None, ...]  # frame dim (:3600)

        # The reference decodes sample by sample when any bos/pad/eos id survived (:3615-3619).  Ids in
        # (codebook_size, vocab) other than those (reachable on untrained weights, quirk Q5) would make its
        # embedding lookup fail; here any id >= codebook_size takes the per-sample filtering path.
        cs = self.config.audio_encoder.codebook_size
        decode_sequentially = bool((audio_codes >= cs).any())
        if not decode_sequentially and codes.shape[-1] > 0:
            vals = self.audio_encoder.decode(audio_codes=audio_codes, audio_scales=[None] * B).audio_values.squeeze(1)
            lengths = [vals.shape[1]] * B
            output_values = vals
        else:
            outs = []
            for b in range(B):
                sample = audio_codes[:, b]
                ok = (sample >= cs).sum(dim=(0, 1)) == 0
                if int(ok.sum()) > 0:
                    sample = sample[:, :, ok]
                    a = self.audio_encoder.decode(audio_codes=sample[None, ...], audio_scales=[None]).audio_values
                    outs.append(a.reshape(-1))
                else:
                    outs.append(torch.zeros(1, device=self.device, dtype=self.dtype))  # :3641
            lengths = [o.shape[0] for o in outs]
            output_values = torch.nn.utils.rnn.pad_sequence(outs, batch_first=True, padding_value=0)
        if gc.return_dict_in_generate or return_codes:
            out = GenerateOutput(sequences=output_values, audios_length=lengths, audio_codes=codes, raw_ids=output_ids)
            if gc.return_dict_in_generate:
                return out
            return output_values, out
        return output_values
