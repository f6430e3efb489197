"""DAC encode (voice-prompt audio -> codes): the oracle against transformers' DacModel.encode, the encoder key mapping, the
C-ABI bookkeeping, and on the GPU the sm_100a encoder + residual vector quantizer against the fixture and the oracle."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from oracle.weights import make_dac_weights
from tests.dac_encode_oracle import OracleDACEncoder, encoder_cfg, make_dac_encoder_weights, tiny_encoder_cfg

DEV = "cuda"


def _product_config(cfg):
    from parler_tts_b200 import DACConfig
    return DACConfig(num_codebooks=cfg.n_codebooks, codebook_size=cfg.codebook_size, latent_dim=cfg.hidden_size,
                     codebook_dim=cfg.codebook_dim, decoder_dim=cfg.decoder_hidden_size, decoder_rates=tuple(cfg.upsampling_ratios),
                     encoder_dim=cfg.encoder_hidden_size, encoder_rates=tuple(cfg.downsampling_ratios))


def _tiny_weights():
    cfg = tiny_encoder_cfg()
    return cfg, {**make_dac_weights(cfg, seed=2), **make_dac_encoder_weights(cfg, seed=6)}


# ---- host ---------------------------------------------------------------------------------------------------------------
def test_oracle_encode_matches_transformers_fixture(golden_dir):
    f = np.load(os.path.join(golden_dir, "dac_encode.npz"))
    cfg, w = _tiny_weights()
    codes, z = OracleDACEncoder(cfg, w).encode(torch.from_numpy(f["audio"]))
    assert np.array_equal(codes[0].numpy(), f["codes"])
    np.testing.assert_allclose(z.numpy(), f["z"], rtol=0, atol=1e-5)


def test_encoder_descript_keys_and_weight_norm_fold():
    from parler_tts_b200.dac_wrapper import _dac_encoder_tensor_list, _encoder_from_descript_keys, _fold_weight_norm
    cfg = tiny_encoder_cfg()
    w = make_dac_encoder_weights(cfg, seed=1)
    n = len(cfg.downsampling_ratios)
    # transformers key -> descript key (encoder.block = [conv, EncoderBlock x n, snake, conv])
    inv = {"encoder.conv1.": "encoder.block.0.", "encoder.snake1.": f"encoder.block.{n + 1}.", "encoder.conv2.": f"encoder.block.{n + 2}."}
    for bi in range(n):
        p, q = f"encoder.block.{bi}.", f"encoder.block.{bi + 1}.block."
        for r in (1, 2, 3):
            for u, nm in ((0, "snake1."), (1, "conv1."), (2, "snake2."), (3, "conv2.")):
                inv[p + f"res_unit{r}." + nm] = q + f"{r - 1}.block.{u}."
        inv[p + "snake1."] = q + "3."
        inv[p + "conv1."] = q + "4."
    desc = {}
    for k, v in w.items():
        pre = max((a for a in inv if k.startswith(a)), key=len, default=None)
        desc[(inv[pre] + k[len(pre):]) if pre else k] = v
    # one convolution in weight-norm form: g * v / ||v|| must give the original weight back
    key = inv["encoder.block.1.conv1."] + "weight"
    wv = desc.pop(key)
    gnorm = wv.flatten(1).norm(dim=1).view(-1, 1, 1)
    desc[key[:-len("weight")] + "weight_g"] = gnorm
    desc[key[:-len("weight")] + "weight_v"] = wv * 3.0
    mapped = {**{k: v for k, v in desc.items() if k.startswith("quantizer.")}, **_encoder_from_descript_keys(_fold_weight_norm(desc), n)}
    names = [k for k in _dac_encoder_tensor_list(_product_config(cfg)) if not k.endswith(("codebook.weight", "out_proj.weight", "out_proj.bias"))]
    assert set(mapped) == set(names)
    for k in names:
        assert torch.allclose(mapped[k], w[k], atol=1e-6), k


def test_encoder_abi_table_and_validation():
    from parler_tts_b200 import _lib
    from parler_tts_b200.dac_wrapper import _dac_encoder_tensor_list
    pc = _product_config(encoder_cfg())
    c = _lib.DacEncoderConfigC(encoder_dim=64, n_blocks=4, latent_dim=1024, n_codebooks=9, codebook_size=1024, codebook_dim=8, dtype=_lib.BF16)
    for i, s in enumerate((2, 4, 8, 8)):
        c.strides[i] = s
    lib = _lib.lib()
    n, nb, ws = C.c_int32(), C.c_int64(), C.c_int64()
    _lib.check(lib.ptts_dac_encoder_num_tensors(C.byref(c), C.byref(n)))
    assert n.value == len(_dac_encoder_tensor_list(pc))
    _lib.check(lib.ptts_dac_encoder_blob_bytes(C.byref(c), C.byref(nb)))
    assert nb.value > 2 * 2 * 21_000_000   # ~21 M parameters in bf16, plus the tensor-core copies of the convolutions
    _lib.check(lib.ptts_dac_encoder_workspace_bytes(C.byref(c), 2, 512 * 10, C.byref(ws)))
    assert ws.value >= 3 * 2 * 512 * 10 * 64 * 2
    with pytest.raises(ValueError, match="hop"):
        _lib.check(lib.ptts_dac_encoder_workspace_bytes(C.byref(c), 2, 512 * 10 + 1, C.byref(ws)))
    c.strides[1] = 3
    with pytest.raises(ValueError, match="stride"):
        _lib.check(lib.ptts_dac_encoder_num_tensors(C.byref(c), C.byref(n)))


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _product(cfg, w, dtype):
    from parler_tts_b200 import DACModel
    return DACModel(_product_config(cfg), DEV, dtype).load_state_dict(w)


@pytest.mark.gpu
def test_encode_tiny_fp32_matches_fixture(golden_dir):
    f = np.load(os.path.join(golden_dir, "dac_encode.npz"))
    cfg, w = _tiny_weights()
    m = _product(cfg, w, torch.float32)
    audio = torch.from_numpy(f["audio"]).to(DEV)
    codes, z = m._encode(audio, want_z=True)
    assert np.array_equal(codes.cpu().numpy(), f["codes"])
    np.testing.assert_allclose(z.cpu().numpy(), f["z"], rtol=0, atol=1e-4)
    out = m.encode(audio)
    assert out.audio_codes.shape == (1,) + f["codes"].shape and out.audio_scales == [None]
    assert torch.equal(out.audio_codes[0], codes)
    two = m.encode(audio, n_quantizers=2, return_dict=False)[0]
    assert torch.equal(two[0], codes[:, :2])
    # the decode blob is untouched by loading the encoder: decode still works on the encoded codes
    assert m.decode(out.audio_codes, [None]).audio_values.shape == (2, 1, codes.shape[-1] * m.hop_length)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


def _check_bf16(cfg, w, audio):
    """The kernel's bf16 run is judged against torch's own bf16 run of the oracle, both measured from the fp32 oracle:
    z's distance from fp32 may be at most 1.5x torch's, and each chosen code's distance gap to the best (re-scored in fp32
    from the fp32 latent, given the kernel's own earlier codes) may be at most 1.5x the largest gap torch's bf16 choices
    show under the same judge, or four bf16 ulps of the distance near its maximum (2^-5; dist = 2 cos lies in [-2, 2]) when
    torch's choices happen to show none."""
    o32 = OracleDACEncoder(cfg, w, torch.float32, DEV)
    o16 = OracleDACEncoder(cfg, w, torch.bfloat16, DEV)
    x = audio.to(DEV)
    with torch.no_grad():
        ze32 = o32.encoder(o32.preprocess(x))
        z32, _ = o32.quantize(ze32)
        codes16, z16 = o16.encode(x)
        gap_torch = o32.choice_gaps(ze32, codes16[0]).max().item()
    m = _product(cfg, w, torch.bfloat16)
    codes, z = m._encode(x, want_z=True)
    with torch.no_grad():
        gap_kernel = o32.choice_gaps(ze32, codes).max().item()
    rel_k, rel_t = _rel(z, z32), _rel(z16, z32)
    agree = float((codes == codes16[0]).float().mean())
    print(f"z rel err vs fp32: kernel {rel_k:.4g} torch-bf16 {rel_t:.4g}; max gap kernel {gap_kernel:.4g} torch {gap_torch:.4g}; "
          f"codes equal to torch-bf16 {agree:.3f}")
    assert rel_k <= 1.5 * rel_t + 1e-3
    assert gap_kernel <= max(1.5 * gap_torch, 2.0 ** -5)


@pytest.mark.gpu
def test_encode_tiny_bf16_generic_path(golden_dir):
    f = np.load(os.path.join(golden_dir, "dac_encode.npz"))
    cfg, w = _tiny_weights()
    _check_bf16(cfg, w, torch.from_numpy(f["audio"]))


@pytest.mark.gpu
def test_encode_real_shape_bf16_tensor_cores():
    cfg = encoder_cfg()
    w = {**make_dac_weights(cfg, seed=3), **make_dac_encoder_weights(cfg, seed=4)}
    g = torch.Generator().manual_seed(12)
    audio = torch.randn(2, 1, 3 * 44100, generator=g) * 0.3
    _check_bf16(cfg, w, audio)


@pytest.mark.gpu
def test_encode_argument_errors():
    from parler_tts_b200 import DACModel
    cfg, w = _tiny_weights()
    m = _product(cfg, w, torch.float32)
    a = torch.randn(1, 1, 1000, device=DEV)
    with pytest.raises(ValueError, match="channels"):
        m.encode(torch.randn(1, 3, 1000, device=DEV))
    with pytest.raises(ValueError, match="mono"):
        m.encode(torch.randn(1, 2, 1000, device=DEV))
    with pytest.raises(ValueError, match="sample_rate"):
        m.encode(a, sample_rate=24000)
    with pytest.raises(ValueError, match="n_quantizers"):
        m.encode(a, n_quantizers=0)
    assert m.encode(a, sample_rate=44100, n_quantizers=99).audio_codes.shape == (1, 1, cfg.n_codebooks, math.ceil(1000 / 512))
    dec_only = DACModel(_product_config(cfg), DEV, torch.float32).load_state_dict(make_dac_weights(cfg, seed=2))
    with pytest.raises(RuntimeError, match="encoder"):
        dec_only.encode(a)
