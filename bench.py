#!/usr/bin/env python
"""bench.py -- audio codec tokens/s (all codebooks) of the generate() hot path on N x B200.

Workload (BASELINE.json configs[1], `--config 1`, the default): Parler-TTS-Mini shape, bf16, batch 32 per GPU, 256 decode
steps, top-k 50 sampling, synthetic inputs (S=64 description states, P=32 prompt prefix, left-padded masks), random-init
weights (no network -> no checkpoints).  One bench "step" = one full pass of the hot path over one batch:
begin + prefill + 255 fused decode steps + sampling = 32 x 9 x 256 tokens.
`--config 2` = configs[2] per GPU (Mini, 1024 steps + DAC decode), `--config 3` = configs[3] (Large, B=64, long cache).

  value      : tokens/s with inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        : the same through the PUBLIC API -- model.generate() -- with HOST (pinned) inputs, the DAC decode included and the
               waveform read back to the host; `e2e.tokens_only` is the token loop alone (GenSession calls, token matrix back)
  roofline   : decode step vs the HBM roofline: algorithmic bytes per step (SURVEY.md 8d formula, T taken
               per step) / measured step time, against MEASURED_PEAKS.json hbm_gbs; `traffic` from the committed ncu capture
  cpu_baseline: the oracle port (CPU restatement of the reference loop) timed on this box's host cores on a
               bounded sample of the same workload (prefill + 32 decode steps, median of 3)
  vs_reference_gpu: the reference's fast GPU recipe (SDPA + static cache + CUDA-graph replay, INFERENCE.md:57-72) as a
               labelled PyTorch RESTATEMENT (oracle/decoder_static.py) timed on the same GPU in the same process
`--impl reference` times the CPU port alone (the reference itself cannot be imported on the GPU box).
`--dump-outputs DIR` writes what the last timed step computed (tokens, last logits, waveform) as .npy files; inputs, weights and
sampling seeds depend only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MINI = dict(vocab_size=1088, max_position_embeddings=4096, num_hidden_layers=24, ffn_dim=4096, num_attention_heads=16,
            hidden_size=1024, num_codebooks=9, pad_token_id=1024, eos_token_id=1024, bos_token_id=1025)
LARGE = dict(MINI, num_hidden_layers=30, ffn_dim=6144, num_attention_heads=24, hidden_size=1536)  # init_large_model.py:25-43
B_PER_GPU, DECODE_STEPS, S_LEN, P_LEN = 32, 256, 64, 32
# BASELINE.json configs[1..3]: (model, batch per GPU, decode steps, what it is)
CONFIGS = {1: (MINI, "Parler-TTS-Mini", 32, 256), 2: (MINI, "Parler-TTS-Mini", 32, 1024), 3: (LARGE, "Parler-TTS-Large", 64, 4096 - P_LEN - 1)}


def step_weight_params(m):
    """SURVEY.md 8(d): parameters streamed per decode step = L x (4H^2 self + 2H^2 cross q/o + 2HF + 6H LN) + K V H heads + 2H."""
    H, F, L = m["hidden_size"], m["ffn_dim"], m["num_hidden_layers"]
    return L * (6 * H * H + 2 * H * F + 6 * H) + m["num_codebooks"] * m["vocab_size"] * H + 2 * H


def kv_tok_bytes(m):
    return m["num_hidden_layers"] * 2 * m["hidden_size"] * 2   # bytes per cached token per sequence (bf16)


assert step_weight_params(MINI) == 362_498_048 and kv_tok_bytes(MINI) == 98_304 and step_weight_params(LARGE) == 1_006_224_384


def algorithmic_bytes_per_step(B, K, V, T, S, m=MINI):
    """SURVEY.md 8(d): 2*W_step + B*kv_tok*(T + S) + B*kv_tok + 4*B*K*V."""
    return 2 * step_weight_params(m) + B * kv_tok_bytes(m) * (T + S) + B * kv_tok_bytes(m) + 4 * B * K * V


def ncu_step_traffic():
    """DRAM bytes of ONE decode_step_kernel launch, read from the committed raw ncu capture (profiles/r02_step_raw.csv:
    `ncu --set full` raw page, dram__bytes_read.sum + dram__bytes_write.sum).  None when the capture is not in the tree."""
    import csv
    p = os.path.join(ROOT, "profiles", "r02_step_raw.csv")
    if not os.path.exists(p):
        return None, "profiles/r02_step_raw.csv missing"
    try:
        rows = list(csv.reader(open(p)))
        hdr = next(r for r in rows if "Kernel Name" in r)
        units = rows[rows.index(hdr) + 1]
        data = next(r for r in rows[rows.index(hdr) + 2:] if len(r) == len(hdr) and "decode_step" in r[hdr.index("Kernel Name")])
        tot = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(name)
            mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[units[i]]
            tot += float(data[i].replace(",", "")) * mult
        return tot, "dram__bytes_read.sum + dram__bytes_write.sum of one decode step kernel launch, profiles/r02_step_raw.csv"
    except Exception as ex:  # pragma: no cover
        return None, f"could not parse profiles/r02_step_raw.csv: {ex!r}"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, idx=0):
        self.idx, self.rows, self.p = idx, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.p.wait()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def synthetic_state_dict(cfg, device, seed=0):
    """Reference init (normal(0, 0.02), modeling_parler_tts.py:1093-1102) generated on the GPU, bf16."""
    g = torch.Generator(device=device).manual_seed(seed)
    H, F, V, K = cfg["hidden_size"], cfg["ffn_dim"], cfg["vocab_size"], cfg["num_codebooks"]

    def n(*s):
        return (torch.randn(*s, generator=g, device=device) * 0.02).to(torch.bfloat16)

    sd = {}
    p = "decoder.model.decoder."
    for k in range(K):
        sd[f"{p}embed_tokens.{k}.weight"] = n(V + 1, H)
        sd[f"decoder.lm_heads.{k}.weight"] = n(V, H)
    for i in range(cfg["num_hidden_layers"]):
        q = f"{p}layers.{i}."
        for a in ("self_attn", "encoder_attn"):
            for m in ("q", "k", "v", "out"):
                sd[f"{q}{a}.{m}_proj.weight"] = n(H, H)
        sd[q + "fc1.weight"], sd[q + "fc2.weight"] = n(F, H), n(H, F)
        for ln in ("self_attn_layer_norm", "encoder_attn_layer_norm", "final_layer_norm"):
            sd[q + ln + ".weight"] = torch.ones(H, device=device)
            sd[q + ln + ".bias"] = torch.zeros(H, device=device)
    sd[p + "layer_norm.weight"], sd[p + "layer_norm.bias"] = torch.ones(H, device=device), torch.zeros(H, device=device)
    sd["embed_prompts.weight"] = n(32128, H)
    return sd


def synth_dac_weights(cfg, device):
    import math
    g = torch.Generator(device=device).manual_seed(0)
    sd = {}
    C = cfg.decoder_dim
    def rn(*s, scale=1.0): return torch.randn(*s, generator=g, device=device) * scale
    for i in range(cfg.num_codebooks):
        sd[f"quantizer.quantizers.{i}.codebook.weight"] = rn(cfg.codebook_size, cfg.codebook_dim)
        sd[f"quantizer.quantizers.{i}.out_proj.weight"] = rn(cfg.latent_dim, cfg.codebook_dim, 1, scale=1 / math.sqrt(8 * 9))
        sd[f"quantizer.quantizers.{i}.out_proj.bias"] = rn(cfg.latent_dim, scale=0.02)
    sd["decoder.conv1.weight"] = rn(C, cfg.latent_dim, 7, scale=1 / math.sqrt(7 * cfg.latent_dim)); sd["decoder.conv1.bias"] = rn(C, scale=0.02)
    for bi, s in enumerate(cfg.decoder_rates):
        cin, cout = C >> bi, C >> (bi + 1)
        p = f"decoder.block.{bi}."
        sd[p + "snake1.alpha"] = torch.ones(1, cin, 1, device=device)
        sd[p + "conv_t1.weight"] = rn(cin, cout, 2 * s, scale=1 / math.sqrt(2 * cin)); sd[p + "conv_t1.bias"] = rn(cout, scale=0.02)
        for r in (1, 2, 3):
            u = p + f"res_unit{r}."
            sd[u + "snake1.alpha"] = torch.ones(1, cout, 1, device=device)
            sd[u + "conv1.weight"] = rn(cout, cout, 7, scale=0.5 / math.sqrt(7 * cout)); sd[u + "conv1.bias"] = rn(cout, scale=0.02)
            sd[u + "snake2.alpha"] = torch.ones(1, cout, 1, device=device)
            sd[u + "conv2.weight"] = rn(cout, cout, 1, scale=0.5 / math.sqrt(cout)); sd[u + "conv2.bias"] = rn(cout, scale=0.02)
    cl = C >> len(cfg.decoder_rates)
    sd["decoder.snake1.alpha"] = torch.ones(1, cl, 1, device=device)
    sd["decoder.conv2.weight"] = rn(1, cl, 7, scale=1 / math.sqrt(7 * cl)); sd["decoder.conv2.bias"] = rn(1, scale=0.02)
    return sd


def synthetic_inputs(B, H, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    enc_mask = torch.ones(B, S_LEN, dtype=torch.long)
    for b, ln in enumerate(torch.randint(32, S_LEN + 1, (B,), generator=g).tolist()):
        enc_mask[b, : S_LEN - ln] = 0
    enc = (torch.randn(B, S_LEN, H, generator=g) * enc_mask[..., None]).to(torch.bfloat16)
    pmask = torch.ones(B, P_LEN, dtype=torch.long)
    for b, ln in enumerate(torch.randint(16, P_LEN + 1, (B,), generator=g).tolist()):
        pmask[b, : P_LEN - ln] = 0
    prompt = (torch.randn(B, P_LEN, H, generator=g) * 0.02).to(torch.bfloat16)
    ts = [enc, enc_mask, prompt, pmask]
    if pin:
        ts = [t.pin_memory() for t in ts]
    return [t.to(device) for t in ts] if device != "cpu" else ts


def cpu_port_measure(n_dec=32, repeats=3):
    """The oracle port of the reference generate() loop (fp32, the reference's CPU code path) on the host cores: Mini, B=32,
    prefill (33 positions) + n_dec decode steps, top-k 50.  Prefill and decode are timed separately (median of `repeats`) so the
    figure can be stated for the SAME workload as the GPU arm (256 decode steps, prefill amortised over them) instead of a
    prefill-dominated short sample."""
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))   # torchrun exports OMP_NUM_THREADS=1: use the physical cores
    from oracle.config import mini_cfg
    from oracle.weights import make_decoder_weights
    from oracle.decoder import OracleDecoder
    from oracle.sampling import generate_tokens
    torch.manual_seed(0)
    cfg = mini_cfg()
    Bc = 32
    dec = OracleDecoder(cfg, make_decoder_weights(cfg, seed=0), torch.float32)
    enc, enc_mask, prompt, pmask = synthetic_inputs(Bc, cfg.hidden_size, 1)
    enc, prompt = enc.float(), prompt.float()
    K = cfg.num_codebooks

    def run(n):
        t0 = time.perf_counter()
        generate_tokens(dec, cfg, enc, enc_mask, prompt, pmask, dict(max_length=n + 1, do_sample=True, top_k=50, min_new_tokens=n))
        return time.perf_counter() - t0

    run(2)  # warm-up
    t_short = sorted(run(1) for _ in range(repeats))[repeats // 2]            # prefill + 1 sampled token
    t_long = sorted(run(n_dec) for _ in range(repeats))[repeats // 2]         # prefill + n_dec tokens
    t_step = (t_long - t_short) / (n_dec - 1)
    sample_tps = Bc * K * n_dec / t_long
    full_tps = Bc * K * DECODE_STEPS / (t_short + (DECODE_STEPS - 1) * t_step)
    sample = (f"oracle port, Mini fp32 B={Bc}: prefill + {n_dec} decode steps, top-k 50, median of {repeats} "
              f"(prefill+1st token {t_short:.2f} s, {1e3 * t_step:.0f} ms per cached step); value = the {DECODE_STEPS}-step workload "
              f"at these rates, sample itself = {sample_tps:.0f} tok/s")
    return {"value": full_tps, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample,
            "os_cpu_count": os.cpu_count(), "sample_tokens_per_s": sample_tps, "prefill_s": t_short, "ms_per_decode_step": 1e3 * t_step,
            "decode_steps_timed": n_dec, "seconds": t_long}


def run_reference(args, rank):
    """CPU arm: the oracle port of the reference generate() loop on the host cores (fp32, like configs[0]).  Each bench step
    is one bounded sample (prefill + 32 decode steps, median of 3)."""
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        m = cpu_port_measure(32, 1 if i < args.warmup else 3)
        if i >= args.warmup:
            vals.append(m)
    m = sorted(vals, key=lambda d: d["value"])[len(vals) // 2]
    v = m["value"]
    line = {"impl": "reference", "metric": "audio codec tokens/sec (all codebooks)", "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * m["seconds"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"Parler-TTS-Mini bf16 batch={B_PER_GPU}/GPU {DECODE_STEPS} decode steps top-k=50 (BASELINE configs[1])",
                       "global_batch": args.gpus * B_PER_GPU, "prompt_len": P_LEN, "desc_len": S_LEN, "parallelism": f"batch-shard x{args.gpus}",
                       "sample": m["sample"] + " -- the reference's CPU code path computes in fp32; same shapes, prompt and description lengths",
                       "same_config": False, "kind": "port (CPU restatement of the reference loop, not the reference package)"},
            "cpu_baseline": m,
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gpu_reference_restatement(dev, B, n_steps=96):
    """The reference's fast GPU recipe (SDPA + static KV cache + CUDA-graph replay = torch.compile "reduce-overhead",
    INFERENCE.md:57-72) restated with stock torch ops (oracle/decoder_static.py), Mini bf16, same batch / prompt / description
    shapes and top-k 50 sampling, on the same GPU.  Returns decode tokens/s over graph-replayed steps (prefill excluded: it is
    amortised to ~nothing over 256 steps on the GPU arm too)."""
    from oracle.config import mini_cfg
    from oracle.decoder_static import StaticCacheDecoder
    cfg = mini_cfg()
    K = cfg.num_codebooks
    g = torch.Generator(device=dev).manual_seed(0)
    sdict = synthetic_state_dict(MINI, dev)
    from parler_tts_b200.modeling import _sinusoidal_table
    sdict["decoder.model.decoder.embed_positions.weights"] = _sinusoidal_table(cfg.max_position_embeddings, cfg.hidden_size).to(dev)
    Tmax = P_LEN + 1 + DECODE_STEPS   # the cache the reference would allocate for this generate() call
    dec = StaticCacheDecoder(cfg, sdict, torch.bfloat16, dev, B, S_LEN, P_LEN, Tmax)
    enc, emask, prompt, pmask = synthetic_inputs(B, cfg.hidden_size, 1, device=dev)
    ids = torch.full((B * K, 1), cfg.bos_token_id, dtype=torch.long, device=dev)
    dec.prefill(ids, enc, emask, prompt, pmask)
    dec.ids.random_(0, 1024, generator=g)
    out = {"kind": "restatement", "what": "oracle/decoder_static.py: SDPA + static KV cache (max_len %d) + HF top-k/multinomial, bf16, B=%d" % (Tmax, B)}
    # eager (the reference's default path runs eager SDPA with a growing cache; this is its static-cache equivalent without graphs)
    for _ in range(3):
        dec.step_and_sample(50)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(16):
        dec.step_and_sample(50)
    e1.record()
    torch.cuda.synchronize()
    out["eager_ms_per_step"] = e0.elapsed_time(e1) / 16
    out["eager_tokens_per_s"] = B * K / (out["eager_ms_per_step"] * 1e-3)
    # CUDA-graph replay of the whole step (what mode="reduce-overhead" produces)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            dec.step_and_sample(50)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    dec.pos.fill_(P_LEN + 1)
    with torch.cuda.graph(graph):
        dec.step_and_sample(50)
    for _ in range(3):
        graph.replay()
    dec.pos.fill_(P_LEN + 1)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_steps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n_steps
    out.update({"value": B * K / (ms * 1e-3), "unit": "tokens/s", "ms_per_step": ms, "mode": "cuda_graph", "steps_timed": n_steps})
    del graph, dec
    torch.cuda.empty_cache()
    return out


def streaming_measure(model, dev, batch, steps, play_steps=20):
    """SURVEY 8f rank 1 / BASELINE configs[4] style: generate() with a ParlerTTSStreamer(incremental=True) consumer thread -- one host-visible
    token column per step (the streamer contract), codec windows of new frames + receptive-field context.  Time to the first audio chunk and
    real-time factor, second run (the first one creates the session and the tensor maps)."""
    import threading
    from parler_tts_b200 import ParlerTTSStreamer
    enc, em, pr, pm = [t[:batch] for t in synthetic_inputs(32, MINI["hidden_size"], 1, device=dev)]

    def run():
        st = ParlerTTSStreamer(model, device=dev, play_steps=play_steps, incremental=True)
        kw = dict(encoder_outputs=(enc,), attention_mask=em, prompt_hidden_states=pr, prompt_attention_mask=pm, do_sample=True, top_k=50,
                  min_new_tokens=steps, max_new_tokens=steps, seed=3, _suppress_special=True, streamer=st)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        th = threading.Thread(target=lambda: model.generate(**kw))
        th.start()
        first, n = None, 0
        for chunk in st:
            m = chunk.shape[-1]
            if m > 0 and first is None:
                first = time.perf_counter() - t0
            n += m
        th.join()
        return first, time.perf_counter() - t0, n

    run()
    first, total, n = run()
    return {"batch": batch, "decode_steps": steps, "play_steps": play_steps, "time_to_first_audio_ms": 1e3 * first, "wall_s": total,
            "samples_per_utterance": n, "rtf_all_utterances": batch * n / 44100 / total, "rtf_per_utterance": (n / 44100) / total,
            "tokens_per_s": batch * MINI["num_codebooks"] * steps / total,
            "api": "model.generate(..., streamer=ParlerTTSStreamer(model, play_steps=20, incremental=True)) consumed on a thread"}


DUMP_AUDIO_MAX = 8 << 20   # waveform samples written in full; above that a fixed sample, so a dump stays under 64 MB for every --config


def dump_outputs(out_dir, shards, wav, suffix=""):
    """What the last timed step computed, as float32 DIR/<name>.npy, so that two builds can be compared output for output:
      tokens [B*K, L]: the token history of every (utterance, codebook) row, BOS column first (token ids are exact in float32)
      logits [B*K, V]: the logits of the last decode step
      audio  [B, samples]: the waveform of the generate() leg; when it holds more than DUMP_AUDIO_MAX samples, the samples at
             DUMP_AUDIO_MAX sorted flat indices drawn with a fixed seed (the same indices for the same arguments)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"tokens": torch.cat([t for t, _ in shards]), "logits": torch.cat([lg for _, lg in shards])}
    if wav is not None:
        wav = wav.float()
        if wav.numel() > DUMP_AUDIO_MAX:
            idx = np.sort(np.random.default_rng(0).choice(wav.numel(), DUMP_AUDIO_MAX, replace=False))
            wav = wav.flatten()[torch.from_numpy(idx)]
        arrays["audio"] = wav
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), t.float().cpu().numpy())



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="BASELINE.json configs[i]; 1 = the headline metric")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-dac", action="store_true")
    ap.add_argument("--decode-steps", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from parler_tts_b200 import DACConfig, ParlerTTSConfig, ParlerTTSDecoderConfig, ParlerTTSForConditionalGeneration
    from parler_tts_b200.dist import broadcast_model_weights, shard_row_base

    MODEL, model_name, B, cfg_steps = CONFIGS[args.config]
    headline = args.config == 1
    dcfg = ParlerTTSDecoderConfig(**MODEL)
    cfg = ParlerTTSConfig(vocab_size=32128, text_encoder={}, audio_encoder=DACConfig(), decoder=dcfg)
    model = ParlerTTSForConditionalGeneration(cfg, device=dev, dtype=torch.bfloat16)
    if rank == 0:
        model.load_state_dict(synthetic_state_dict(MODEL, dev))
        if not args.no_dac:
            model.audio_encoder.load_state_dict(synth_dac_weights(cfg.audio_encoder, dev))
    if world > 1:
        broadcast_model_weights(model)   # the one collective on this path: packed weights from rank 0 (NVLink)
        torch.cuda.synchronize()
    K, V, H = MODEL["num_codebooks"], MODEL["vocab_size"], MODEL["hidden_size"]
    n_dec = args.decode_steps or cfg_steps
    L = n_dec + 1
    eng = model.decoder.engine
    # the fused step kernels hold one 32-row tile: a larger per-GPU batch (configs[3]) runs as consecutive 32-row shards through the
    # same session, exactly as generate() does (modeling.py _fused_batch_limit)
    TILE = 32
    shards = [(b0, min(B, b0 + TILE)) for b0 in range(0, B, TILE)]
    assert len({b1 - b0 for b0, b1 in shards}) == 1, "per-GPU batch must be <= 32 or a multiple of 32"
    Bs = shards[0][1] - shards[0][0]
    sess = eng.session(Bs, P_LEN, S_LEN, P_LEN + L)
    host = synthetic_inputs(B, H, seed=1 + rank, pin=True)
    enc_d, emask_d, prompt_d, pmask_d = [t.to(dev) for t in host]
    row_base = shard_row_base(world * B, rank, world, K)   # global (utterance, codebook) row of this shard: Philox substreams
    gen = dict(do_sample=True, top_k=50, temperature=1.0, top_p=1.0, min_new_tokens=n_dec, suppress_special=True, codebook_size=1024,
               row_base=row_base)

    def one_pass(seed, from_host):
        if from_host:
            e, em, p, pm = [t.to(dev, non_blocking=True) for t in host]
        else:
            e, em, p, pm = enc_d, emask_d, prompt_d, pmask_d
        outs = []
        for b0, b1 in shards:
            sess.begin(L, seed=seed, **dict(gen, row_base=row_base + b0 * K))
            sess.prefill(p[b0:b1], pm[b0:b1], e[b0:b1], em[b0:b1])
            sess.sample()
            sess.decode_steps(n_dec - 1)
            if from_host:
                outs.append(sess.raw_ids[:, :L].to("cpu", non_blocking=False))
            elif args.dump_outputs:
                outs.append((sess.raw_ids[:, :L].clone(), sess.logits.clone()))   # the next shard reuses the session's buffers
        return outs

    def generate_pass(seed):
        """The public call: host tensors in, waveform on the host out (DAC decode inside generate())."""
        e, em, p, pm = [t.to(dev, non_blocking=True) for t in host]
        wav = model.generate(encoder_outputs=(e,), attention_mask=em, prompt_hidden_states=p, prompt_attention_mask=pm,
                             do_sample=True, top_k=50, temperature=1.0, min_new_tokens=n_dec, max_new_tokens=n_dec, seed=seed,
                             row_base=row_base, _suppress_special=True)
        return wav.to("cpu", non_blocking=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for i in range(args.warmup):
            fn(100 + i)
        barrier()
        l0 = sess.launches
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(args.steps):
            out = fn(200 + i)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, sess.launches - l0, out

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    try:
        ms, launches, last_pass = timed(lambda s: one_pass(s, False))
    finally:
        clk = clocks.stop() if rank == 0 else None
    st = sess.state.cpu().tolist()
    assert st[0] == L, f"generation stopped early at length {st[0]} (expected {L})"
    fused = sess.fused
    ms_tok, _, _ = timed(lambda s: one_pass(s, True))
    e2e_full, wav = None, None
    if not args.no_dac:
        if world > 1 and rank != 0:
            pass  # DAC weights arrived with the broadcast
        ms_e2e, _, wav = timed(generate_pass)
        assert wav.shape == (B, (L - K) * 512), wav.shape
        e2e_full = (ms_e2e, wav.numel() * wav.element_size())
        sess = eng.session(Bs, P_LEN, S_LEN, P_LEN + L)  # (generate() may have re-created the session)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_pass, wav, f"_rank{rank}" if world > 1 else "")

    # decode-only timing for the roofline: the fused decode steps of one pass, T taken per step
    barrier()
    sess.begin(L, seed=7, **gen)
    sess.prefill(prompt_d[:Bs], pmask_d[:Bs], enc_d[:Bs], emask_d[:Bs])
    sess.sample()
    sess.decode_steps(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    sess.decode_steps(n_dec - 3)
    e1.record()
    torch.cuda.synchronize()
    dec_ms = e0.elapsed_time(e1)
    n_timed = n_dec - 3
    # step s (1-based count of tokens already appended) attends over T = P + s + 1 keys
    byts = sum(algorithmic_bytes_per_step(Bs, K, V, P_LEN + s + 1, S_LEN, MODEL) for s in range(3, 3 + n_timed))
    hbm_peak, peak_src = peaks()
    achieved = byts / (dec_ms * 1e-3) / 1e9

    # DAC decode of the generated frames alone (the metric is the token loop, SURVEY 8d; configs[2] adds the codec)
    dac_info = None
    if rank == 0 and not args.no_dac:
        frames = L - K
        codes = torch.randint(0, 1024, (1, B, K, frames), device=dev)
        for _ in range(2):
            model.audio_encoder.decode(codes, [None] * B)
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(3):
            model.audio_encoder.decode(codes, [None] * B).audio_values
        d1.record()
        torch.cuda.synchronize()
        dms = d0.elapsed_time(d1) / 3
        flops = 1.608e9 * B * frames
        dac_info = {"ms": dms, "frames": frames, "batch": B, "tflops": flops / dms / 1e9, "audio_seconds": B * frames * 512 / 44100,
                    "rtf": (B * frames * 512 / 44100) / (dms / 1e3), "kernel": "conv_tc_kernel (tcgen05 implicit GEMM, bf16 in / f32 TMEM accumulate)",
                    "flop_per_frame": 1.608e9}
        tp = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(tp):
            pk = json.load(open(tp))
            dac_info["frac_of_bf16_peak_sustained"] = dac_info["tflops"] / float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"]))
    if rank == 0:
        tokens = world * B * K * n_dec * args.steps
        value = tokens / (ms * 1e-3)
        h2d = sum(t.numel() * t.element_size() for t in host)
        tok_only = {"value": tokens / (ms_tok * 1e-3), "unit": "tokens/s", "d2h_bytes_per_step": B * K * L * 8,
                    "api": "GenSession begin/prefill/sample/decode_steps (the calls generate() makes), token matrix read back to host"}
        if e2e_full is not None:
            e2e = {"value": tokens / (e2e_full[0] * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": e2e_full[1],
                   "api": "model.generate(encoder_outputs=..., prompt_hidden_states=..., masks) with pinned host inputs; includes the DAC "
                          "decode; the waveform [B, samples] is read back to the host", "ms_per_step": e2e_full[0] / args.steps,
                   "audio_seconds_per_step": world * B * (L - K) * 512 / 44100,
                   "rtf": (world * B * (L - K) * 512 / 44100) / (e2e_full[0] / args.steps * 1e-3),   # seconds of audio per second of wall time, all utterances
                   "tokens_only": tok_only}
        else:
            e2e = dict(tok_only, h2d_bytes_per_step=h2d)
        traffic, traffic_src = ncu_step_traffic() if (headline and int(fused) == 2) else (None, "no ncu capture committed for this configuration")
        line = {
            "metric": "audio codec tokens/sec (all codebooks)", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{model_name} bf16 batch={B}/GPU {n_dec} decode steps top-k=50 (BASELINE configs[{args.config}])",
                       "global_batch": world * B, "prompt_len": P_LEN, "desc_len": S_LEN, "parallelism": f"batch-shard x{world}", "row_tiles_per_gpu": len(shards),
                       "l2": f"inputs larger than L2 ({2 * step_weight_params(MODEL) / 1e9:.3f} GB weights + KV streamed per step)",
                       "timed_region": "generate_begin + prefill + sampling + fused decode steps",
                       "decode_path": {2: "cluster step kernel (step2.cu)", 1: "fused step kernel (step.cu)", 0: "multi-kernel path (shape outside the fused kernels' range)"}[int(fused)]},
            "clocks": clk,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "kernel": {2: "decode_step_cluster_kernel (one persistent kernel per token: 32 clusters x 4 CTAs, embed + L x 6 phases + heads + sample)",
                                    1: "decode_step_kernel (one persistent kernel per token: 148 CTAs, embed + L x 8 phases + heads + sample)",
                                    0: "multi-kernel decode path"}[int(fused)],
                         "ms_per_decode_step": dec_ms / n_timed, "algorithmic_bytes_per_step_avg": byts / n_timed},
        }
        if dac_info is not None:
            line["dac_decode"] = dac_info
        if world == 1 and headline and not args.no_dac:
            try:
                line["streaming"] = streaming_measure(model, dev, 8, n_dec)
            except Exception as ex:  # pragma: no cover
                line["streaming"] = {"value": None, "error": repr(ex)}
        if world == 1 and headline and not args.no_gpu_reference:
            try:
                r = gpu_reference_restatement(dev, B)
                r["decode_only_ratio"] = (Bs * K / (dec_ms / n_timed * 1e-3)) / r["value"]
                line["vs_reference_gpu"] = r
            except Exception as ex:  # pragma: no cover
                line["vs_reference_gpu"] = {"value": None, "error": repr(ex)}
        if world == 1 and headline and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_port_measure(32, 3)
            except Exception as ex:  # pragma: no cover
                line["cpu_baseline"] = {"value": None, "error": repr(ex)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
