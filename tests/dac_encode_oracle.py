"""Torch restatement of the DAC encode path and its seeded synthetic weights (test infrastructure only).

Reference call site: DACModel.encode -> model.preprocess (right zero-pad to the hop) then model.encode(x, n_quantizers)
(parler_tts/dac_wrapper/modeling_dac.py:33-104).  descript-audio-codec is not installed; the network is pinned against
transformers 5.5.0's DacModel, which restates it:
  encoder          transformers/models/dac/modeling_dac.py:442-473   block :210-232   residual unit :173-207
  quantizer        :281-343 (DacResidualVectorQuantizer.forward)    vector quantize :122-170
It lives beside the tests rather than in oracle/ so that the decode oracle and the fixtures made from it stay as they are;
it reuses oracle.dac.snake and the decode config records.
"""
from __future__ import annotations
import math

import torch
import torch.nn.functional as F

from oracle.config import Cfg, dac_cfg, tiny_dac_cfg
from oracle.dac import snake


def encoder_cfg(**kw) -> Cfg:
    """DAC 44.1 kHz with the descript encoder defaults (encoder_dim 64, strides 2, 4, 8, 8)."""
    d = dict(encoder_hidden_size=64, downsampling_ratios=[2, 4, 8, 8])
    d.update(kw)
    return dac_cfg(**d)


def tiny_encoder_cfg() -> Cfg:
    return tiny_dac_cfg().clone(encoder_hidden_size=8, downsampling_ratios=[2, 4, 8, 8])


def make_dac_encoder_weights(cfg: Cfg, seed: int = 0) -> dict[str, torch.Tensor]:
    """Folded DAC encoder + quantizer in_proj weights, fp32, keyed like transformers.models.dac.DacModel.

    A separate generator from oracle.weights.make_dac_weights (whose stream the decode fixtures depend on); the codebooks and
    out_proj come from there.  Fan-in scales keep the activations O(1) through the ~30-layer stack."""
    g = torch.Generator().manual_seed(seed)

    def conv(co, ci, k, gain=1.0):
        return torch.randn(co, ci, k, generator=g) * (gain / math.sqrt(ci * k)), torch.randn(co, generator=g) * 0.02

    def alpha(c):
        return (1.0 + 0.3 * torch.randn(1, c, 1, generator=g)).abs() + 0.1

    w: dict[str, torch.Tensor] = {}
    D = cfg.encoder_hidden_size
    w["encoder.conv1.weight"], w["encoder.conv1.bias"] = conv(D, 1, 7, gain=2.0)
    for bi, s in enumerate(cfg.downsampling_ratios):
        c = D * 2 ** bi
        p = f"encoder.block.{bi}."
        for ri in (1, 2, 3):
            r = p + f"res_unit{ri}."
            w[r + "snake1.alpha"] = alpha(c)
            w[r + "conv1.weight"], w[r + "conv1.bias"] = conv(c, c, 7, gain=0.5)
            w[r + "snake2.alpha"] = alpha(c)
            w[r + "conv2.weight"], w[r + "conv2.bias"] = conv(c, c, 1, gain=0.5)
        w[p + "snake1.alpha"] = alpha(c)
        w[p + "conv1.weight"], w[p + "conv1.bias"] = conv(2 * c, c, 2 * s)
    dm = D * 2 ** len(cfg.downsampling_ratios)
    w["encoder.snake1.alpha"] = alpha(dm)
    w["encoder.conv2.weight"], w["encoder.conv2.bias"] = conv(cfg.hidden_size, dm, 3)
    for i in range(cfg.n_codebooks):
        w[f"quantizer.quantizers.{i}.in_proj.weight"], w[f"quantizer.quantizers.{i}.in_proj.bias"] = conv(cfg.codebook_dim, cfg.hidden_size, 1)
    return w


class OracleDACEncoder:
    """weights: encoder.* plus the full quantizer (in_proj, codebook, out_proj)."""

    def __init__(self, cfg: Cfg, weights: dict[str, torch.Tensor], dtype=torch.float32, device="cpu"):
        self.cfg, self.dtype = cfg, dtype
        self.w = {k: v.to(device=device, dtype=dtype) for k, v in weights.items()}
        self.hop = math.prod(cfg.downsampling_ratios)

    def preprocess(self, audio: torch.Tensor) -> torch.Tensor:
        n = audio.shape[-1]
        return F.pad(audio, (0, math.ceil(n / self.hop) * self.hop - n))

    def _res(self, x, p, dil):
        y = F.conv1d(snake(x, self.w[p + "snake1.alpha"]), self.w[p + "conv1.weight"], self.w[p + "conv1.bias"], dilation=dil, padding=3 * dil)
        y = F.conv1d(snake(y, self.w[p + "snake2.alpha"]), self.w[p + "conv2.weight"], self.w[p + "conv2.bias"])
        return x + y

    def encoder(self, x: torch.Tensor) -> torch.Tensor:
        """[B, 1, n] -> z_e [B, latent, n / hop]"""
        w = self.w
        x = F.conv1d(x, w["encoder.conv1.weight"], w["encoder.conv1.bias"], padding=3)
        for bi, s in enumerate(self.cfg.downsampling_ratios):
            p = f"encoder.block.{bi}."
            for ri, dil in ((1, 1), (2, 3), (3, 9)):
                x = self._res(x, p + f"res_unit{ri}.", dil)
            x = F.conv1d(snake(x, w[p + "snake1.alpha"]), w[p + "conv1.weight"], w[p + "conv1.bias"], stride=s, padding=math.ceil(s / 2))
        x = snake(x, w["encoder.snake1.alpha"])
        return F.conv1d(x, w["encoder.conv2.weight"], w["encoder.conv2.bias"], padding=1)

    def _vq(self, i, residual, indices=None):
        """DacVectorQuantize.forward on residual [B, latent, T]; with `indices` given, that choice replaces the argmax.
        Returns (out_proj output, indices, dist [B*T, codebook_size])."""
        q = f"quantizer.quantizers.{i}."
        proj = F.conv1d(residual, self.w[q + "in_proj.weight"], self.w[q + "in_proj.bias"])
        B, Dc, T = proj.shape
        enc = F.normalize(proj.permute(0, 2, 1).reshape(B * T, Dc))
        cb = F.normalize(self.w[q + "codebook.weight"])
        l2 = enc.pow(2).sum(1, keepdim=True)
        dist = -(l2 - 2 * enc @ cb.t()) + cb.pow(2).sum(1, keepdim=True).t()
        if indices is None:
            indices = dist.max(1)[1].reshape(B, T)
        zq = F.embedding(indices, self.w[q + "codebook.weight"]).transpose(1, 2)
        st = proj + (zq - proj)
        return F.conv1d(st, self.w[q + "out_proj.weight"], self.w[q + "out_proj.bias"]), indices, dist

    def quantize(self, ze: torch.Tensor, n_q: int | None = None):
        """DacResidualVectorQuantizer.forward (eval): -> (z [B, latent, T], codes [B, n_q, T])"""
        n_q = self.cfg.n_codebooks if n_q is None else n_q
        z, residual, codes = 0, ze, []
        for i in range(n_q):
            qi, idx, _ = self._vq(i, residual)
            z = z + qi
            residual = residual - qi
            codes.append(idx)
        return z, torch.stack(codes, dim=1)

    def encode(self, audio: torch.Tensor, n_q: int | None = None):
        """DACModel.encode: audio [B, 1, samples] -> (audio_codes [1, B, n_q, T], z [B, latent, T])"""
        z, codes = self.quantize(self.encoder(self.preprocess(audio.to(self.dtype))), n_q)
        return codes[None], z

    def choice_gaps(self, ze: torch.Tensor, codes: torch.Tensor) -> torch.Tensor:
        """Judge a code sequence [B, n_q, T]: codebook k's residual is recomputed from the GIVEN earlier codes, and the
        gap best_dist - dist[chosen] (>= 0; 0 = an argmax) is returned as [B, n_q, T] in fp32."""
        residual, gaps = ze, []
        for i in range(codes.shape[1]):
            qi, _, dist = self._vq(i, residual, codes[:, i])
            d = dist.float()
            chosen = d.gather(1, codes[:, i].reshape(-1, 1)).squeeze(1)
            gaps.append((d.max(1)[0] - chosen).reshape(codes.shape[0], -1))
            residual = residual - qi
        return torch.stack(gaps, dim=1)
