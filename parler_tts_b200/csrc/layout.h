// layout.h -- byte layout of the packed decoder weight blob and of the generation workspace.
//
// HBM layout (DESIGN.md "Data layout"):
//   blob      : [embed tables K x (V+1) x H][pos table][L x layer][final LN][lm heads (K*V) x H]
//               GEMM matrices are stored in mma.m16n8k16 B-fragment order (bf16) so a warp's 512 B
//               load is one fully coalesced request and needs no shared-memory staging.
//   workspace : control block, token history, activations, cross K/V [L][B*S][2*nckv*64],
//               self K/V cache [L][2][B][nkv][Tmax][64].
#pragma once
#include "common.cuh"

namespace ptts {

struct MatSlot {
  int64_t off;  // byte offset in blob
  int N, K;     // fused matrix shape (rows = output features)
  int row_off;  // row offset of this tensor inside the fused matrix
};

struct DecoderLayout {
  int es;  // element size of model dtype
  int H, F, V, K, L, nh, nkv, nckv, qkv_rows, ckv_rows;
  int64_t embed, pos, layer0, layer_stride;
  // offsets inside one layer
  int64_t ln1_w, ln1_b, wqkv, wo, ln2_w, ln2_b, wqc, wkvc, woc, ln3_w, ln3_b, fc1, fc2;
  int64_t c_qkv, c_qc, c_fc1;   // folded-LayerNorm vectors (c1 | c2), f32, per layer (ln_stats.cuh)
  int64_t final_ln_w, final_ln_b, heads, rope_cos, rope_sin, c_heads;
  // cluster step kernel (step2.cu): a second copy of the six per-layer matrices, cut into one contiguous slice per
  // (phase, cluster, rank): the n-tiles the cluster owns x the K range the rank reduces.  cl_NC == 0: shape not covered.
  int cl_C, cl_NC;          // CTAs per cluster (8), clusters (= heads)
  int64_t rm[7];            // per layer (bf16 only): ROW-MAJOR copies of wqkv, wo, wqc, wkvc, woc, fc1, fc2 for the tcgen05 prefill
                            // GEMM (gemm_tc.cu: TMA-tiled K-major operands); same order as rm_src()
  int64_t cp[6];            // per layer: offset of phase p's slices (A qkv | B o | C q_cross | D o_cross | E fc1 | F fc2)
  int64_t cp_slice[6];      // bytes of one (cluster, rank) slice of phase p
  int64_t total;
};

// Shapes the cluster step kernel covers: bf16, MHA for self- and cross-attention, two clusters of 4 CTAs per head (<= 18 heads on
// 148 SMs), K halves that are whole k32 tiles, H / (2 heads) = 32 out-proj features per cluster, at most 4 fc1 n-tiles per rank, and
// the shared-memory plan of step2.cu (sized for H <= 1024, F <= 4096).
static inline bool cluster_shape_ok(const ptts_decoder_config& c) {
  const int H = c.hidden_size, nh = c.num_heads, F = c.ffn_dim;
  return c.dtype == PTTS_BF16 && c.num_kv_heads == nh && c.num_cross_kv_heads == nh && nh * 8 <= 144 && H == nh * PTTS_HEAD_DIM &&
         H % 256 == 0 && F % 256 == 0 && F % (nh * 64) == 0 && (F / (nh * 64) == 1 || F / (nh * 64) == 2 || F / (nh * 64) == 4) && H <= 1024 && F <= 4096 && c.num_codebooks <= 16 &&
         (c.vocab_size * c.num_codebooks) % 32 == 0;
}

static inline int dtype_size(int dt) { return dt == PTTS_BF16 ? 2 : 4; }

static inline DecoderLayout make_layout(const ptts_decoder_config& c) {
  DecoderLayout l{};
  l.es = dtype_size(c.dtype);
  l.H = c.hidden_size; l.F = c.ffn_dim; l.V = c.vocab_size; l.K = c.num_codebooks; l.L = c.num_layers;
  l.nh = c.num_heads; l.nkv = c.num_kv_heads; l.nckv = c.num_cross_kv_heads;
  l.qkv_rows = (l.nh + 2 * l.nkv) * PTTS_HEAD_DIM;
  l.ckv_rows = 2 * l.nckv * PTTS_HEAD_DIM;
  int64_t o = 0;
  auto take = [&](int64_t bytes) { int64_t r = o; o = align_up(o + bytes, 256); return r; };
  l.embed = take((int64_t)l.K * (l.V + 1) * l.H * l.es);
  l.pos = take(c.rope ? 0 : (int64_t)c.max_positions * l.H * l.es);
  l.layer0 = o;
  int64_t base = o;
  l.ln1_w = take(l.H * 4) - base; l.ln1_b = take(l.H * 4) - base;
  l.wqkv = take((int64_t)l.qkv_rows * l.H * l.es) - base;
  l.wo = take((int64_t)l.H * l.H * l.es) - base;
  l.ln2_w = take(l.H * 4) - base; l.ln2_b = take(l.H * 4) - base;
  l.wqc = take((int64_t)l.H * l.H * l.es) - base;
  l.wkvc = take((int64_t)l.ckv_rows * l.H * l.es) - base;
  l.woc = take((int64_t)l.H * l.H * l.es) - base;
  l.ln3_w = take(l.H * 4) - base; l.ln3_b = take(l.H * 4) - base;
  l.fc1 = take((int64_t)l.F * l.H * l.es) - base;
  l.fc2 = take((int64_t)l.H * l.F * l.es) - base;
  l.c_qkv = take((int64_t)2 * l.qkv_rows * 4) - base;
  l.c_qc = take((int64_t)2 * l.H * 4) - base;
  l.c_fc1 = take((int64_t)2 * l.F * 4) - base;
  for (int i = 0; i < 7; i++) l.rm[i] = 0;
  if (c.dtype == PTTS_BF16) {
    const int64_t sz[7] = {(int64_t)l.qkv_rows * l.H, (int64_t)l.H * l.H, (int64_t)l.H * l.H, (int64_t)l.ckv_rows * l.H, (int64_t)l.H * l.H,
                           (int64_t)l.F * l.H, (int64_t)l.H * l.F};
    for (int i = 0; i < 7; i++) l.rm[i] = take(sz[i] * 2) - base;
  }
  l.cl_C = l.cl_NC = 0;
  for (int i = 0; i < 6; i++) l.cp[i] = l.cp_slice[i] = 0;
  if (cluster_shape_ok(c)) {
    l.cl_C = 4; l.cl_NC = 2 * l.nh;
    const int64_t ks = l.H / 4 / 32, ksf = l.F / 4 / 32;                 // k32 tiles per rank: K = H phases, K = F phase
    // n-tiles per slice: a head's q|k|v (192 features), a cluster's 32 out-proj features, a head's q_cross, ..., F / 32 fc1 features
    const int64_t nt[6] = {24, 4, 8, 4, l.F / (2 * l.nh) / 8, 4};
    const int64_t owners[6] = {l.nh, 2 * l.nh, l.nh, 2 * l.nh, 2 * l.nh, 2 * l.nh};   // head phases: one slice set per head
    for (int i = 0; i < 6; i++) {
      l.cp_slice[i] = nt[i] * (i == 5 ? ksf : ks) * 512;
      l.cp[i] = take(l.cp_slice[i] * owners[i] * l.cl_C) - base;
    }
  }
  l.layer_stride = o - base;
  o = base + l.layer_stride * l.L;
  l.final_ln_w = take(l.H * 4); l.final_ln_b = take(l.H * 4);
  l.heads = take((int64_t)l.K * l.V * l.H * l.es);
  l.rope_cos = take(c.rope ? (int64_t)c.max_positions * PTTS_HEAD_DIM * l.es : 0);
  l.rope_sin = take(c.rope ? (int64_t)c.max_positions * PTTS_HEAD_DIM * l.es : 0);
  l.c_heads = take((int64_t)2 * l.K * l.V * 4);
  l.total = o;
  return l;
}

static inline int validate_config(const ptts_decoder_config& c) {
  PTTS_REQUIRE(c.dtype == PTTS_BF16 || c.dtype == PTTS_F32, "dtype must be bf16(0) or f32(1), got %d", c.dtype);
  PTTS_REQUIRE(c.hidden_size > 0 && c.num_heads > 0 && c.hidden_size == c.num_heads * PTTS_HEAD_DIM,
               "hidden_size (%d) must equal num_heads (%d) * %d", c.hidden_size, c.num_heads, PTTS_HEAD_DIM);
  PTTS_REQUIRE(c.num_kv_heads > 0 && c.num_heads % c.num_kv_heads == 0, "num_heads %% num_kv_heads != 0");
  PTTS_REQUIRE(c.num_cross_kv_heads > 0 && c.num_heads % c.num_cross_kv_heads == 0, "num_heads %% num_cross_kv_heads != 0");
  PTTS_REQUIRE(c.hidden_size % 32 == 0 && c.ffn_dim % 32 == 0, "hidden_size and ffn_dim must be multiples of 32");
  PTTS_REQUIRE(c.ffn_dim % c.hidden_size == 0, "ffn_dim must be a multiple of hidden_size");
  PTTS_REQUIRE(c.vocab_size % 8 == 0, "vocab_size must be a multiple of 8, got %d", c.vocab_size);
  PTTS_REQUIRE(c.hidden_size <= 2048, "hidden_size > 2048 not supported by the activation tile");
  PTTS_REQUIRE(c.num_codebooks >= 1 && c.num_codebooks <= 32, "num_codebooks out of range");
  PTTS_REQUIRE(c.num_layers >= 1 && c.activation >= 0 && c.activation <= 3, "bad num_layers/activation");
  return PTTS_OK;
}

// Resolve (tensor_id, index) -> fused matrix slot.  Returns false for non-matrix tensors.
static inline bool matrix_slot(const DecoderLayout& l, int tensor_id, int index, MatSlot* s) {
  int64_t lb = l.layer0 + l.layer_stride * index;
  const int D = PTTS_HEAD_DIM;
  switch (tensor_id) {
    case PTTS_T_SELF_Q: *s = {lb + l.wqkv, l.qkv_rows, l.H, 0}; return true;
    case PTTS_T_SELF_K: *s = {lb + l.wqkv, l.qkv_rows, l.H, l.nh * D}; return true;
    case PTTS_T_SELF_V: *s = {lb + l.wqkv, l.qkv_rows, l.H, (l.nh + l.nkv) * D}; return true;
    case PTTS_T_SELF_O: *s = {lb + l.wo, l.H, l.H, 0}; return true;
    case PTTS_T_CROSS_Q: *s = {lb + l.wqc, l.H, l.H, 0}; return true;
    case PTTS_T_CROSS_K: *s = {lb + l.wkvc, l.ckv_rows, l.H, 0}; return true;
    case PTTS_T_CROSS_V: *s = {lb + l.wkvc, l.ckv_rows, l.H, l.nckv * D}; return true;
    case PTTS_T_CROSS_O: *s = {lb + l.woc, l.H, l.H, 0}; return true;
    case PTTS_T_FC1: *s = {lb + l.fc1, l.F, l.H, 0}; return true;
    case PTTS_T_FC2: *s = {lb + l.fc2, l.H, l.F, 0}; return true;
    case PTTS_T_LM_HEAD: *s = {l.heads, l.K * l.V, l.H, index * l.V}; return true;
    default: return false;
  }
}

// ---- workspace ----------------------------------------------------------------------------------
struct WorkspaceLayout {
  int B, P, S, Tmax, Mmax, BK;    // Mmax = B * (P + max_prefix) rows of the first forward
  int64_t ctrl, progress, gen, raw_ids, cur_ids, eos_seen, unfinished, first_unf, prompt_mask, enc_mask;
  int64_t x, qkv, attn, qc, hbuf, hidden, logits, scores, cross_tmp, cross_kv, self_kv;
  int64_t img_x, img_attn, img_h;  // fused step kernel: activations as tile images [chunk][32][H + 8] (step.cu stage_tile)
  int64_t cl_x, cl_attn, cl_h;     // cluster step kernel: K-sliced images [4][32][K/4 + 8] (step2.cu)
  int64_t row_stats;               // [max(B*(P+1), B*S)][2] f32: LayerNorm row statistics of the tcgen05 prefill GEMMs
  int64_t cross_layer_stride, self_layer_stride;  // bytes
  int64_t raw_ld;                                  // raw_ids leading dimension (elements)
  int64_t total;
};

// max_prefix: decoder columns the first forward may take (1 = the BOS column; more for a voice-prompt prefix, ptts_prefill_ids)
static inline WorkspaceLayout make_workspace(const ptts_decoder_config& c, int B, int P, int S, int Tmax, int max_prefix = 1) {
  DecoderLayout l = make_layout(c);
  WorkspaceLayout w{};
  w.B = B; w.P = P; w.S = S; w.Tmax = Tmax; w.BK = B * c.num_codebooks;
  w.Mmax = B * (P + max_prefix);
  int64_t o = 0;
  auto take = [&](int64_t bytes) { int64_t r = o; o = align_up(o + bytes, 256); return r; };
  w.ctrl = take(sizeof(Ctrl));
  w.progress = take(1024 * 4);
  w.gen = take(sizeof(ptts_gen_params));
  w.raw_ld = Tmax - P + 1;  // >= max_length
  w.raw_ids = take((int64_t)w.BK * w.raw_ld * 8);
  w.cur_ids = take((int64_t)w.BK * 4);
  w.eos_seen = take((int64_t)w.BK * 4);
  w.unfinished = take((int64_t)w.BK * 4);
  w.first_unf = take((int64_t)2 * B * 4);
  w.prompt_mask = take((int64_t)B * (P > 0 ? P : 1) * 4);
  w.enc_mask = take((int64_t)B * S * 4);
  int64_t rows_enc = (int64_t)B * S;
  w.x = take((int64_t)w.Mmax * l.H * l.es);
  w.qkv = take((int64_t)w.Mmax * l.qkv_rows * l.es);
  w.attn = take((int64_t)w.Mmax * l.H * l.es);
  w.qc = take((int64_t)w.Mmax * l.H * l.es);
  w.hbuf = take((int64_t)w.Mmax * l.F * l.es);
  w.hidden = take((int64_t)B * l.H * l.es);
  w.img_x = take((int64_t)32 * (l.H + 8) * 2);
  w.img_attn = take((int64_t)32 * (l.H + 8) * 2);
  w.img_h = take((int64_t)((l.F + l.H - 1) / l.H) * 32 * (l.H + 8) * 2);
  w.row_stats = take((int64_t)(w.Mmax > rows_enc ? w.Mmax : rows_enc) * 2 * 4);
  w.cl_x = take((int64_t)4 * 32 * (l.H / 4 + 8) * 2);
  w.cl_attn = take((int64_t)4 * 32 * (l.H / 4 + 8) * 2);
  w.cl_h = take((int64_t)4 * 32 * (l.F / 4 + 8) * 2);
  w.logits = take((int64_t)w.BK * l.V * 4);
  w.scores = take((int64_t)w.BK * l.V * 4);
  w.cross_layer_stride = align_up(rows_enc * l.ckv_rows * l.es, 256);
  w.cross_tmp = take(w.cross_layer_stride);   // GEMM output of one layer before the item-major re-layout
  w.cross_kv = take(w.cross_layer_stride * l.L);
  w.self_layer_stride = align_up((int64_t)2 * B * l.nkv * Tmax * PTTS_HEAD_DIM * l.es, 256);
  w.self_kv = take(w.self_layer_stride * l.L);
  w.total = o;
  return w;
}

}  // namespace ptts
