"""Per-phase timing of the CLUSTER decode-step kernel (step2.cu; CTA 0 clock64 stamps) for the bench workload.
Usage: python tools/profile_step2.py [decode steps before the stamped launch]"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from parler_tts_b200 import DACConfig, ParlerTTSConfig, ParlerTTSDecoderConfig, ParlerTTSForConditionalGeneration, _lib

steps_before = int(sys.argv[1]) if len(sys.argv) > 1 else 100
dev = torch.device("cuda", 0)
cfg = ParlerTTSConfig(vocab_size=32128, text_encoder={}, audio_encoder=DACConfig(), decoder=ParlerTTSDecoderConfig(**bench.MINI))
model = ParlerTTSForConditionalGeneration(cfg, device=dev, dtype=torch.bfloat16)
model.load_state_dict(bench.synthetic_state_dict(bench.MINI, dev))
B, L, NL = 32, 257, 24
sess = model.decoder.engine.session(B, bench.P_LEN, bench.S_LEN, bench.P_LEN + L)
enc, em, pr, pm = bench.synthetic_inputs(B, 1024, 1, device=dev)
gen = dict(do_sample=True, top_k=50, min_new_tokens=256, suppress_special=True, codebook_size=1024)
sess.begin(L, seed=1, **gen)
sess.prefill(pr, pm, enc, em)
assert sess.fused == 2, f"cluster step kernel not in use (fused kind {sess.fused})"
sess.sample()
sess.decode_steps(steps_before)
nph = 6 * NL
STRIDE = 16
buf = torch.zeros((6 * NL + 4) * STRIDE + 6 * 128, dtype=torch.int64, device=dev)   # + per-CTA arrival times of the middle layer's barriers
_lib.check(_lib.lib().ptts_session_set_profile(sess.h, _lib.ptr(buf)))
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
sess.decode_steps(1)
e1.record()
torch.cuda.synchronize()
arrive = buf[(6 * NL + 4) * STRIDE:].cpu().view(6, 128).numpy().astype(np.float64)
t = buf[:(6 * NL + 4) * STRIDE].cpu().view(-1, STRIDE).numpy()
_lib.check(_lib.lib().ptts_session_set_profile(sess.h, None))
us = lambda c: c / 1.965 / 1e3
names = ["qkv+self-attn", "o-proj", "q_cross+cross-attn", "o_cross", "fc1", "fc2"]
print(f"step (event) {e0.elapsed_time(e1) * 1e3:.1f} us ; T = {bench.P_LEN + steps_before + 2} cached keys")
print("per phase (us, mean over 24 layers, CTA 0): wait = phase start -> slice + weights landed | mma | exch = partials sent and received |"
      " epi | attn | barrier = done -> released")
out = {}
tot_l = 0.0
for sub in range(6):
    rows = np.array([t[1 + 6 * l + sub] for l in range(NL)], dtype=np.float64)
    wait, mma, exch, epi = us(rows[:, 1] - rows[:, 0]), us(rows[:, 2] - rows[:, 1]), us(rows[:, 3] - rows[:, 2]), us(rows[:, 4] - rows[:, 3])
    attn = us(rows[:, 6] - rows[:, 4])
    barr = us(rows[:, 7] - rows[:, 6])
    work = us(rows[:, 6] - rows[:, 0])
    out[names[sub]] = dict(work=work.mean(), barrier=barr.mean(), wait=wait.mean(), mma=mma.mean(), exch=exch.mean(), epi=epi.mean(), attn=attn.mean())
    tot_l += work.mean() + barr.mean()
    extra = (f"  [exch: pre {us(rows[:, 12] - rows[:, 2]).mean():.2f} clwait {us(rows[:, 13] - rows[:, 12]).mean():.2f} stage {us(rows[:, 14] - rows[:, 13]).mean():.2f}"
             f" issue {us(rows[:, 15] - rows[:, 14]).mean():.2f} wait {us(rows[:, 3] - rows[:, 15]).mean():.2f}]")
    if sub in (0, 2):   # attention internals (warp 0): cluster sync + set-up | ring sweep | own key + merge | store
        extra += (f"  [attn: setup {us(rows[:, 8] - rows[:, 4]).mean():.2f} sweep {us(rows[:, 9] - rows[:, 8]).mean():.2f} ({rows[:, 11].mean():.1f} chunks)"
                 f" merge {us(rows[:, 10] - rows[:, 9]).mean():.2f} store {us(rows[:, 5] - rows[:, 10]).mean():.2f}]")
    print(f"{names[sub]:20s} work {work.mean():6.2f}  barrier {barr.mean():5.2f} | wait {wait.mean():5.2f}  mma {mma.mean():5.2f}  exch {exch.mean():5.2f}"
          f"  epi {epi.mean():5.2f}  attn {attn.mean():5.2f}{extra}")
print(f"per layer {tot_l:.1f} us -> {tot_l * NL:.0f} us for {NL} layers")
span = [us(float(t[1 + 6 * l + 5][7] - t[1 + 6 * l][0])) for l in range(NL)]
print(f"layer spans (us): first {span[0]:.1f}, second {span[1]:.1f}, mean of the rest {np.mean(span[2:]):.1f}, max {max(span[2:]):.1f}")
if arrive.max() > 0:   # barrier arrival skew of the middle layer (globaltimer, ns): who is late?
    for sub in range(6):
        a = (arrive[sub] - arrive[sub].min()) / 1e3
        order = np.argsort(a)
        by_rank = [a[r::4].mean() for r in range(4)]
        print(f"arrival skew {names[sub]:20s}: CTA0 {a[0]:.2f}  median {np.median(a):.2f}  p90 {np.percentile(a, 90):.2f}  max {a.max():.2f} us (CTA {order[-1]}, {order[-2]}, {order[-3]}); "
              f"mean by cluster rank {' '.join(f'{x:.2f}' for x in by_rank)}; clusters 0-15 {a[:64].mean():.2f} / 16-31 {a[64:].mean():.2f}")
r0, rh, rt = t[0], t[nph + 1], t[nph + 2]
print(f"prologue {us(r0[0] - rt[3]):.2f} | embed {us(r0[6] - r0[0]):.2f} + barrier {us(r0[7] - r0[6]):.2f} | lm heads {us(rh[6] - rh[0]):.2f} "
      f"(tile + stats {us(rh[1] - rh[0]):.2f}) | barrier {us(rt[0] - rh[6]):.2f} | sampling {us(rt[1] - rt[0]):.2f} | last barrier {us(rt[2] - rt[1]):.2f} "
      f"| kernel span {us(rt[2] - rt[3]):.1f} us")
os.makedirs("gpurun_out", exist_ok=True)
json.dump({"step_us": e0.elapsed_time(e1) * 1e3, "phases_us": out}, open("gpurun_out/step2_phases.json", "w"), indent=1)
