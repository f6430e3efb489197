"""Generate tests/golden/dac_encode.npz by EXECUTING transformers' DacModel.encode (stand-in for descript-audio-codec,
which is not installed), at a tiny shape with the seeded weights of tests/dac_encode_oracle.py.

The reference wrapper's own part of DACModel.encode -- right zero-padding to the hop (DAC.preprocess) -- is applied here
before the call; the fixture keeps the unpadded audio, so a test exercises that padding too.
Stored: audio [B, 1, samples] f32, z [B, latent, T] (the quantized latent), codes [B, K, T].

Usage:  python tests/golden/make_golden_dac_encode.py
"""
from __future__ import annotations
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def gen_dac_encode():
    from transformers.models.dac import DacConfig, DacModel
    from oracle.weights import make_dac_weights
    from tests.dac_encode_oracle import tiny_encoder_cfg, make_dac_encoder_weights
    cfg = tiny_encoder_cfg()
    hc = DacConfig(encoder_hidden_size=cfg.encoder_hidden_size, downsampling_ratios=cfg.downsampling_ratios,
                   decoder_hidden_size=cfg.decoder_hidden_size, n_codebooks=cfg.n_codebooks, codebook_size=cfg.codebook_size,
                   codebook_dim=cfg.codebook_dim, hidden_size=cfg.hidden_size, upsampling_ratios=cfg.upsampling_ratios,
                   sampling_rate=44100)
    m = DacModel(hc).eval()
    w = {**make_dac_weights(cfg, seed=2), **make_dac_encoder_weights(cfg, seed=6)}
    sd = m.state_dict()
    for k, v in w.items():
        assert k in sd and sd[k].shape == v.shape, k
        sd[k] = v
    m.load_state_dict(sd)
    assert set(sd) == set(w), set(sd) ^ set(w)   # every tensor of the model is a seeded one
    g = torch.Generator().manual_seed(9)
    hop = int(np.prod(cfg.downsampling_ratios))
    n = 5 * hop + 77                              # not a multiple of the hop: the wrapper pads to 6 frames
    audio = torch.randn(2, 1, n, generator=g) * 0.3
    padded = torch.nn.functional.pad(audio, (0, 6 * hop - n))
    with torch.no_grad():
        out = m.encode(padded)
    np.savez_compressed(os.path.join(HERE, "dac_encode.npz"), audio=audio.numpy(), z=out.quantized_representation.numpy(),
                        codes=out.audio_codes.numpy())


if __name__ == "__main__":
    gen_dac_encode()
    print("dac_encode.npz", os.path.getsize(os.path.join(HERE, "dac_encode.npz")))
