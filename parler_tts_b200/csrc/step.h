// step.h -- parameters of the fused decode-step kernel (step.cu).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace ptts {

struct StepParams {
  // shapes
  int B, H, F, V, K, L, nh, nkv, nckv, S, P, Tmax, rope, act, qkv_rows;
  float eps, scale;
  // packed weights
  const char* blob;
  int64_t embed, pos, layer0, layer_stride, wqkv, wo, wqc, woc, fc1, fc2;
  int64_t c_qkv, c_qc, c_fc1, c_heads;   // folded-LayerNorm vectors
  int64_t heads, rope_cos, rope_sin;
  // workspace
  bf16 *x, *qkv, *attn, *qc, *hbuf;  // x / attn / hbuf are tile images (row pitch H + 8; hbuf: F/H images), qkv / qc plain rows
  float* logits;
  char* cross_kv; int64_t cross_layer_stride;
  char* self_kv; int64_t self_layer_stride;
  const int* prompt_mask;  // nullable
  const int* enc_mask;     // nullable
  SampleArgs sa;
  unsigned* bar;           // [2] device-wide barrier counters (Ctrl::bar)
  // schedule
  int nt_qkv, nt_h, nt_fc1, nt_heads;
  int nbuf;                // activation-tile buffers (2 = double-buffered K chunks)
  int64_t tile_region_bytes;   // scratch after the header: [activation tiles | weight buffer], aliased by attention
  int64_t wbuf_offset;         // weight buffer offset inside the scratch region
  int do_sample_phase;     // 1: logits -> token inside the kernel (ptts_decode_steps); 0: stop at the logits
  int sample_items;        // ceil(V / 256): logits per thread of the one-CTA-per-row sampler
  int* progress;           // debug: last phase each CTA arrived at (printed on a barrier timeout)
  int n_steps;             // cluster kernel: tokens one launch may run (stops early when every row is finished); 0 / 1 = one
  long long* prof;         // optional [(8L+3)][8] clock64 timestamps written by CTA 0 (debug / profiles)
  // ---- cluster step kernel (step2.cu) ----
  int64_t cp[6], cp_slice[6];   // per-layer offsets / slice bytes of the (phase, cluster, rank) weight slices (layout.h)
  bf16 *cl_x, *cl_attn, *cl_h;  // K-sliced activation images [4][32][K/4 + 8]
};

int step_smem_bytes(const StepParams& p);
int launch_decode_step(const StepParams& p, int grid, cudaStream_t st);
// cluster step kernel (step2.cu)
bool cluster_step_available(const StepParams& p);
int launch_decode_step_cluster(const StepParams& p, cudaStream_t st);
int cluster_pack_layer(const char* layer_src, char* layer_dst, const int64_t* mat_off, const int64_t* cp_off, int nh, int H, int F, cudaStream_t st);

}  // namespace ptts
