"""Voice-prompt continuation: decoder prefill over a multi-column prefix (ptts_prefill_ids), generate() from decoder_input_ids /
input_values, and the multi-column first forward() call."""
import numpy as np
import pytest
import torch

from oracle import delay_pattern as odp
from oracle.config import tiny_cfg, tiny_dac_cfg
from oracle.decoder import OracleDecoder
from oracle.sampling import ParlerLogitsProcessorOracle, frames_from_raw, process_scores
from oracle.weights import make_dac_weights, make_decoder_weights
from tests.dac_encode_oracle import make_dac_encoder_weights, tiny_encoder_cfg
from tests.helpers import build_product_model, synth_inputs

DEV = "cuda"
VARIANTS = {"abs": dict(rope_embeddings=False), "rope": dict(rope_embeddings=True),
            "gqa": dict(rope_embeddings=True, num_attention_heads=4, num_key_value_heads=2, num_cross_attention_key_value_heads=1,
                        hidden_size=256)}


def oracle_prefix_greedy(dec, cfg, enc, enc_mask, prompt, prompt_mask, prefix, L):
    """generate() from decoder_input_ids (modeling_parler_tts.py:3017-3044, :3458-3469, :3523-3597), greedy, restated on the
    oracle: pattern from the whole prefix, the model's first input = its first n columns, the rest as the reference's loop."""
    B, K = enc.shape[0], cfg.num_codebooks
    bos, pad, eos = cfg.bos_token_id, cfg.pad_token_id, cfg.eos_token_id
    ids, mask = odp.build_delay_pattern_mask(prefix, bos, pad, L, K)
    parler = ParlerLogitsProcessorOracle(eos, K, B)
    unfinished = np.ones(B * K, dtype=np.int64)
    step = 0
    while True:
        model_in = odp.apply_delay_pattern_mask(ids, mask)
        if step == 0:
            logits = dec.prefill(torch.from_numpy(model_in), enc, enc_mask, prompt, prompt_mask)
        else:
            logits = dec.step(torch.from_numpy(model_in[:, -1:]))
        nxt = process_scores(logits[:, -1, :].float().numpy(), ids, parler, dict(max_length=L)).argmax(-1)
        nxt = nxt * unfinished + pad * (1 - unfinished)
        ids = np.concatenate([ids, nxt[:, None]], axis=1)
        unfinished = unfinished & ~((ids[:, -1] == eos) | (ids.shape[1] >= L))
        step += 1
        if unfinished.max() == 0:
            break
    return frames_from_raw(ids, mask, cfg, B)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_prefill_ids_matches_reference_teacher_forced_logits(golden_dir, variant):
    """decoder_forward.npz holds the reference's own ParlerTTSForCausalLM.forward logits over [prompt | 6 decoder columns]:
    a prefill over the first n columns must give the logits of position P + n - 1."""
    import os
    from parler_tts_b200.modeling import GenSession
    f = np.load(os.path.join(golden_dir, "decoder_forward.npz"))
    cfg = tiny_cfg(**VARIANTS[variant])
    model = build_product_model(cfg, tiny_dac_cfg(), make_decoder_weights(cfg, seed=3), make_dac_weights(tiny_dac_cfg(), seed=1),
                                dtype=torch.float32)
    ids, enc = torch.from_numpy(f[f"{variant}_ids"]), torch.from_numpy(f[f"{variant}_enc"])
    prompt, pmask, emask = torch.from_numpy(f[f"{variant}_prompt"]), torch.from_numpy(f[f"{variant}_pmask"]), torch.from_numpy(f[f"{variant}_enc_mask"])
    ref = f[f"{variant}_logits"]
    B, P, S = enc.shape[0], prompt.shape[1], enc.shape[1]
    sess = GenSession(model.decoder.engine, B, P, S, P + 8, max_prefix=6)
    for n in range(1, 7):
        sess.begin(8)
        sess.prefill(prompt, pmask, enc, emask, prefix_ids=ids[:, :n])
        got = sess.logits.cpu().numpy()
        err = np.abs(got - ref[:, P + n - 1]).max()
        assert err < 2e-4, (n, err)
        assert np.array_equal(sess.raw_ids[:, :n].cpu().numpy(), ids[:, :n].numpy())
        assert int(sess.state[0].item()) == n
    sess.close()


def _tiny_model(dtype=torch.float32, with_encoder=False):
    cfg, dcfg = tiny_cfg(), tiny_dac_cfg()
    w = make_decoder_weights(cfg, seed=51, head_std=0.5)
    dw = make_dac_weights(dcfg, seed=2)
    if with_encoder:
        ecfg = tiny_encoder_cfg()
        dw = {**dw, **make_dac_encoder_weights(ecfg, seed=6)}
        from parler_tts_b200 import ParlerTTSConfig, ParlerTTSForConditionalGeneration
        from tests.helpers import product_decoder_config
        from tests.test_dac_encode import _product_config
        pc = ParlerTTSConfig(vocab_size=cfg.text_vocab_size, text_encoder={}, audio_encoder=_product_config(ecfg), decoder=product_decoder_config(cfg))
        m = ParlerTTSForConditionalGeneration(pc, device=DEV, dtype=dtype)
        m.load_state_dict(w, dac_state_dict=dw)
        return cfg, w, m
    return cfg, w, build_product_model(cfg, dcfg, w, dw, dtype=dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("T_a,L_new", [(7, 12), (3, 2), (1, 9)])
def test_generate_from_decoder_input_ids_greedy_fp32(T_a, L_new):
    """Tokens bit-exact with the oracle's greedy prefix loop; the returned codes start with the prompt's own frames.
    (3, 2): max_length = n + 2 < 2K - 1, where the reference's pattern forces nothing."""
    cfg, w, model = _tiny_model()
    B, S, P, K = 2, 8, 4, cfg.num_codebooks
    enc, enc_mask, prompt, prompt_mask = synth_inputs(cfg, B, S, P, seed=8)
    g = torch.Generator().manual_seed(T_a)
    codes_in = torch.randint(0, cfg.codebook_size, (B * K, T_a), generator=g)
    _, out = model.generate(encoder_outputs=(enc.to(DEV),), attention_mask=enc_mask.to(DEV), prompt_hidden_states=prompt.to(DEV),
                            prompt_attention_mask=prompt_mask.to(DEV), decoder_input_ids=codes_in.to(DEV), do_sample=False,
                            max_new_tokens=L_new, return_codes=True)
    prefix = np.concatenate([np.full((B * K, 1), cfg.bos_token_id), codes_in.numpy()], axis=1)
    ref = oracle_prefix_greedy(OracleDecoder(cfg, w, torch.float32), cfg, enc, enc_mask, prompt, prompt_mask, prefix, L_new + 1 + T_a)
    got = out.audio_codes.cpu().numpy()
    assert np.array_equal(got, ref)
    if L_new + 1 + T_a >= 2 * K - 1:
        assert np.array_equal(got[:, :, :T_a], codes_in.numpy().reshape(B, K, T_a))


@pytest.mark.gpu
def test_generate_input_values_equals_encoded_ids_and_shards():
    cfg, w, model = _tiny_model(torch.bfloat16, with_encoder=True)
    K, S, P = cfg.num_codebooks, 8, 4
    B = 40   # bf16: the fused step kernels take 32 rows, so this runs as shards of 32 + 8
    enc, enc_mask, prompt, prompt_mask = synth_inputs(cfg, B, S, P, seed=3)
    audio = torch.randn(B, 1, 4 * 512 + 100, generator=torch.Generator().manual_seed(5)) * 0.3
    kw = dict(encoder_outputs=(enc.to(DEV),), attention_mask=enc_mask.to(DEV), prompt_hidden_states=prompt.to(DEV),
              prompt_attention_mask=prompt_mask.to(DEV), do_sample=False, max_new_tokens=12, return_codes=True, _suppress_special=True)
    _, a = model.generate(input_values=audio.to(DEV), **kw)
    ids = model.audio_encoder.encode(audio.to(DEV)).audio_codes[0].reshape(B * K, -1)
    _, b = model.generate(decoder_input_ids=ids, **kw)
    assert torch.equal(a.audio_codes, b.audio_codes)
    assert torch.equal(a.audio_codes[:, :, :ids.shape[1]], ids.reshape(B, K, -1))
    for lo, hi in ((0, 32), (32, 40)):
        kws = dict(kw, encoder_outputs=(enc[lo:hi].to(DEV),), attention_mask=enc_mask[lo:hi].to(DEV),
                   prompt_hidden_states=prompt[lo:hi].to(DEV), prompt_attention_mask=prompt_mask[lo:hi].to(DEV))
        _, part = model.generate(decoder_input_ids=ids[lo * K:hi * K], **kws)
        n = part.audio_codes.shape[-1]
        assert torch.equal(a.audio_codes[lo:hi, :, :n], part.audio_codes)


@pytest.mark.gpu
def test_forward_multi_column_first_call_equals_prefill_ids():
    from parler_tts_b200.modeling import GenSession
    cfg, w, model = _tiny_model()
    B, S, P, K, n = 2, 8, 4, cfg.num_codebooks, 5
    enc, enc_mask, prompt, prompt_mask = synth_inputs(cfg, B, S, P, seed=2)
    ids = torch.randint(0, cfg.codebook_size, (B * K, n), generator=torch.Generator().manual_seed(1))
    ids[:, 0] = cfg.bos_token_id
    out = model.decoder.forward(input_ids=ids.to(DEV), encoder_hidden_states=enc.to(DEV), encoder_attention_mask=enc_mask.to(DEV),
                                prompt_hidden_states=prompt.to(DEV), prompt_attention_mask=prompt_mask.to(DEV), max_cache_len=P + 16)
    assert out["past_key_values"].get_seq_length() == P + n
    sess = GenSession(model.decoder.engine, B, P, S, P + 16, max_prefix=n)
    sess.begin(16)
    sess.prefill(prompt, prompt_mask, enc, enc_mask, prefix_ids=ids)
    assert torch.equal(out["logits"][:, 0], sess.logits)
    nxt = torch.full((B * K, 1), 3, dtype=torch.int64)
    out2 = model.decoder.forward(input_ids=nxt.to(DEV), past_key_values=out["past_key_values"])
    assert out2["past_key_values"].get_seq_length() == P + n + 1
    sess.close()


@pytest.mark.gpu
def test_audio_prompt_value_errors():
    cfg, w, model = _tiny_model()
    B, S, P, K = 1, 8, 4, cfg.num_codebooks
    enc, enc_mask, prompt, prompt_mask = synth_inputs(cfg, B, S, P, seed=1)
    kw = dict(encoder_outputs=(enc.to(DEV),), prompt_hidden_states=prompt.to(DEV), do_sample=False, max_new_tokens=4)
    ids = torch.zeros(B * K, 3, dtype=torch.int64, device=DEV)
    from parler_tts_b200 import ParlerTTSStreamer
    with pytest.raises(ValueError, match="audio prompt"):
        model.generate(decoder_input_ids=ids, streamer=ParlerTTSStreamer(model, device=DEV, play_steps=4), **kw)
    with pytest.raises(ValueError, match="audio prompt"):
        model.generate(decoder_input_ids=ids, logits_processor=[lambda i, s: s], **kw)
    with pytest.raises(ValueError, match="decoder_input_ids must be"):
        model.generate(decoder_input_ids=ids[:1], **kw)
    with pytest.raises(RuntimeError, match="encoder"):   # this model was loaded without DAC encoder weights
        model.generate(input_values=torch.zeros(B, 1, 1024, device=DEV), **kw)
