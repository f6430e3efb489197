"""Configuration records with the reference's field names and defaults.

Mirrors (fields and defaults only, re-written -- these are plain Python records, not PretrainedConfig):
  ParlerTTSDecoderConfig   parler_tts/configuration_parler_tts.py:107-172
  ParlerTTSConfig          parler_tts/configuration_parler_tts.py:240-291
  DACConfig                parler_tts/dac_wrapper/configuration_dac.py:7-27
"""
from __future__ import annotations
import copy
import json
import os
from typing import Any


class _Record:
    model_type = "record"

    def to_dict(self) -> dict[str, Any]:
        out = {}
        for k, v in self.__dict__.items():
            out[k] = v.to_dict() if isinstance(v, _Record) else copy.deepcopy(v)
        out["model_type"] = self.model_type
        return out

    def __repr__(self):
        return f"{type(self).__name__} {json.dumps(self.to_dict(), indent=2, default=str)}"


class ParlerTTSDecoderConfig(_Record):
    model_type = "parler_tts_decoder"

    def __init__(self, vocab_size=2049, max_position_embeddings=2048, num_hidden_layers=24, ffn_dim=4096,
                 num_attention_heads=16, num_key_value_heads=None, num_cross_attention_key_value_heads=None,
                 layerdrop=0.0, use_cache=True, activation_function="gelu", hidden_size=1024, dropout=0.1,
                 attention_dropout=0.0, activation_dropout=0.0, initializer_factor=0.02, scale_embedding=False,
                 num_codebooks=4, pad_token_id=2048, bos_token_id=2049, eos_token_id=2048,
                 tie_word_embeddings=False, rope_embeddings=False, rope_theta=10_000.0,
                 cross_attention_implementation_strategy=None, use_fused_lm_heads=False, codebook_weights=None,
                 layer_norm_eps=1e-5, **kwargs):
        self.vocab_size = vocab_size
        self.max_position_embeddings = max_position_embeddings
        self.hidden_size = hidden_size
        self.ffn_dim = ffn_dim
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.num_key_value_heads = num_attention_heads if num_key_value_heads is None else num_key_value_heads
        self.num_cross_attention_key_value_heads = (
            self.num_key_value_heads if num_cross_attention_key_value_heads is None else num_cross_attention_key_value_heads)
        self.dropout = dropout
        self.attention_dropout = attention_dropout
        self.activation_dropout = activation_dropout
        self.activation_function = activation_function
        self.initializer_factor = initializer_factor
        self.layerdrop = layerdrop
        self.use_cache = use_cache
        self.scale_embedding = scale_embedding
        self.num_codebooks = num_codebooks
        self.rope_embeddings = rope_embeddings
        self.rope_theta = rope_theta
        self.cross_attention_implementation_strategy = cross_attention_implementation_strategy
        self.use_fused_lm_heads = use_fused_lm_heads
        self.codebook_weights = codebook_weights
        if codebook_weights is not None and len(codebook_weights) != num_codebooks:
            raise ValueError(f"`codebook_weights` has length {len(codebook_weights)} when it should be of length {num_codebooks}.")
        self.pad_token_id = pad_token_id
        self.bos_token_id = bos_token_id
        self.eos_token_id = eos_token_id
        self.tie_word_embeddings = tie_word_embeddings
        self.layer_norm_eps = layer_norm_eps  # nn.LayerNorm default; not a reference config field


class DACConfig(_Record):
    model_type = "dac_on_the_hub"

    def __init__(self, num_codebooks=9, model_bitrate=8, codebook_size=1024, latent_dim=1024, frame_rate=86,
                 sampling_rate=44100, codebook_dim=8, decoder_dim=1536, decoder_rates=(8, 8, 4, 2), encoder_dim=64,
                 encoder_rates=(2, 4, 8, 8), **kwargs):
        self.codebook_size = codebook_size
        self.model_bitrate = model_bitrate
        self.latent_dim = latent_dim
        self.num_codebooks = num_codebooks
        self.frame_rate = frame_rate
        self.sampling_rate = sampling_rate
        # descript-audio-codec DAC() constructor defaults for the 44.1 kHz model (the reference passes only
        # n_codebooks / latent_dim / codebook_size, dac_wrapper/modeling_dac.py:24-28)
        self.codebook_dim = codebook_dim
        self.decoder_dim = decoder_dim
        self.decoder_rates = list(decoder_rates)
        self.encoder_dim = encoder_dim
        self.encoder_rates = list(encoder_rates)


class GenerationConfig(_Record):
    """The HF GenerationConfig fields generate() reads (init_model_600M.py:57-63 sets the Parler defaults)."""
    model_type = "generation_config"

    def __init__(self, max_length=2580, max_new_tokens=None, min_new_tokens=None, do_sample=True, temperature=1.0,
                 top_k=50, top_p=1.0, bos_token_id=None, pad_token_id=None, eos_token_id=None,
                 decoder_start_token_id=None, return_dict_in_generate=False, num_beams=1, num_beam_groups=1,
                 num_return_sequences=1, repetition_penalty=1.0, no_repeat_ngram_size=0, length_penalty=1.0, typical_p=1.0,
                 epsilon_cutoff=0.0, eta_cutoff=0.0, min_length=0, penalty_alpha=None, bad_words_ids=None, force_words_ids=None,
                 guidance_scale=None, **kwargs):
        self.max_length = max_length
        self.max_new_tokens = max_new_tokens
        self.min_new_tokens = min_new_tokens
        self.do_sample = do_sample
        self.temperature = temperature
        self.top_k = top_k
        self.top_p = top_p
        self.bos_token_id = bos_token_id
        self.pad_token_id = pad_token_id
        self.eos_token_id = eos_token_id
        self.decoder_start_token_id = decoder_start_token_id
        self.return_dict_in_generate = return_dict_in_generate
        self.num_beams = num_beams
        # knobs the device loop does not implement: kept so that generate() can REJECT a non-neutral value instead of
        # silently ignoring it (modeling.py::_NEUTRAL_GENERATION_KNOBS)
        self.num_beam_groups, self.num_return_sequences = num_beam_groups, num_return_sequences
        self.repetition_penalty, self.no_repeat_ngram_size, self.length_penalty = repetition_penalty, no_repeat_ngram_size, length_penalty
        self.typical_p, self.epsilon_cutoff, self.eta_cutoff, self.min_length = typical_p, epsilon_cutoff, eta_cutoff, min_length
        self.penalty_alpha, self.bad_words_ids, self.force_words_ids, self.guidance_scale = penalty_alpha, bad_words_ids, force_words_ids, guidance_scale

    def update(self, **kwargs) -> dict[str, Any]:
        """Like HF GenerationConfig.update: consume known attributes, return the rest (model kwargs)."""
        rest = {}
        for k, v in kwargs.items():
            if k in self.__dict__:
                setattr(self, k, v)
            else:
                rest[k] = v
        return rest


class ParlerTTSConfig(_Record):
    model_type = "parler_tts"
    is_composition = True

    def __init__(self, vocab_size=1024, prompt_cross_attention=False, **kwargs):
        if "audio_encoder" not in kwargs or "decoder" not in kwargs:
            raise ValueError("Config has to be initialized with text_encoder, audio_encoder and decoder config")
        self.vocab_size = vocab_size
        self.prompt_cross_attention = prompt_cross_attention
        te = kwargs.get("text_encoder") or {}
        self.text_encoder = dict(te.to_dict() if hasattr(te, "to_dict") else te)
        ae = kwargs["audio_encoder"]
        self.audio_encoder = ae if isinstance(ae, DACConfig) else DACConfig(**{k: v for k, v in dict(ae).items() if k != "model_type"})
        de = kwargs["decoder"]
        self.decoder = de if isinstance(de, ParlerTTSDecoderConfig) else ParlerTTSDecoderConfig(**{k: v for k, v in dict(de).items() if k != "model_type"})
        self.is_encoder_decoder = True
        self.pad_token_id = kwargs.get("pad_token_id", self.decoder.pad_token_id)
        self.decoder_start_token_id = kwargs.get("decoder_start_token_id", self.decoder.bos_token_id)

    @classmethod
    def from_sub_models_config(cls, text_encoder_config, audio_encoder_config, decoder_config, **kwargs):
        return cls(text_encoder=text_encoder_config, audio_encoder=audio_encoder_config, decoder=decoder_config, **kwargs)

    @classmethod
    def from_pretrained(cls, path: str):
        with open(os.path.join(path, "config.json")) as f:
            d = json.load(f)
        return cls(**d)

    @property
    def sampling_rate(self):
        return self.audio_encoder.sampling_rate
