"""DACModel.encode timing (waveform -> codes, the voice-prompt path) for the 44.1 kHz DAC shape in bf16.

Reports, with the card name and power limit read in the same run: time per call and achieved TFLOP/s (operations counted from
the shapes by encode_flops below) for B = 1 and 32 utterances of 3 s and 10 s, and the per-kernel share of one B = 32 x 3 s call
from a torch.profiler run of its own.  Inputs are seeded noise; the working set (activations of >= 25 MB per utterance-second)
is larger than L2 for the B = 32 rows.

Usage: python tools/bench_dac_encode.py [--out DIR]   (writes DIR/dac_encode_bench.json when --out is given)
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from parler_tts_b200 import DACConfig, DACModel  # noqa: E402
from oracle.weights import make_dac_weights  # noqa: E402
from tests.dac_encode_oracle import encoder_cfg, make_dac_encoder_weights  # noqa: E402

SR = 44100


def encode_flops(cfg: DACConfig, n: int) -> float:
    """Multiply-adds x 2 of one utterance of n samples (n a multiple of the hop): convolutions and the quantizer."""
    D, f, rate = cfg.encoder_dim, 2 * 7 * cfg.encoder_dim * n, n
    for bi, s in enumerate(cfg.encoder_rates):
        c = D << bi
        f += rate * 3 * 2 * (7 * c * c + c * c)      # three residual units (k7 + k1)
        rate //= s
        f += rate * 2 * (2 * s) * c * (2 * c)         # strided conv
    dm = D << len(cfg.encoder_rates)
    f += rate * 2 * 3 * dm * cfg.latent_dim            # conv2
    f += rate * cfg.num_codebooks * 2 * (2 * cfg.latent_dim * cfg.codebook_dim + cfg.codebook_size * cfg.codebook_dim)
    return float(f)


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dac_encode: needs a CUDA device")
    dev = torch.device("cuda", 0)
    ocfg = encoder_cfg()
    cfg = DACConfig()
    w = {**make_dac_weights(ocfg, seed=3), **make_dac_encoder_weights(ocfg, seed=4)}
    m = DACModel(cfg, dev, torch.bfloat16).load_state_dict(w)
    g = torch.Generator().manual_seed(0)
    out = {**gpu_info(), "dtype": "bf16", "runs": []}
    for B, sec in ((1, 3), (1, 10), (32, 3), (32, 10)):
        x = (torch.randn(B, 1, sec * SR, generator=g) * 0.3).to(dev, torch.bfloat16)
        for _ in range(2):
            m.encode(x)
        torch.cuda.synchronize()
        reps = 20 if B == 1 else 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            codes = m.encode(x).audio_codes
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        n = math.ceil(sec * SR / m.encoder_hop_length) * m.encoder_hop_length
        fl = B * encode_flops(cfg, n)
        out["runs"].append({"B": B, "seconds": sec, "frames": codes.shape[-1], "ms": round(ms, 3), "gflop": round(fl / 1e9, 1),
                            "tflops": round(fl / ms / 1e9, 1)})
        print(json.dumps(out["runs"][-1]), flush=True)
    # kernel shares of one B = 32 x 3 s call, profiled in a run of its own
    x = (torch.randn(32, 1, 3 * SR, generator=g) * 0.3).to(dev, torch.bfloat16)
    m.encode(x)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        m.encode(x)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            name = ev.key.split("(")[0].split("<")[0].replace("void ", "").replace("ptts::", "")
            if "conv_tc_kernel" in ev.key:
                name = "conv_tc_kernel<down>" if "<true>" in ev.key else "conv_tc_kernel"
            per[name] = per.get(name, 0.0) + ev.self_device_time_total / 1e3
    total = sum(per.values())
    out["profile_B32_3s"] = {"kernel_ms_total": round(total, 3),
                             "share": {k: round(v / total, 3) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}}
    print(json.dumps(out["profile_B32_3s"]))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "dac_encode_bench.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
