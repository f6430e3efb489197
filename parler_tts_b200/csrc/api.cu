// api.cu -- the C ABI (include/ptts_b200.h): argument validation, weight packing, the generation
// session (prefill / decode step / sample / CUDA-graph replay) and DAC decode orchestration.
#include <cstdarg>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <new>

#include "common.cuh"
#include "dac.h"
#include "kernels.h"
#include "layout.h"
#include "step.h"

namespace ptts {
static thread_local std::string g_err;
void set_error(const std::string& m) { g_err = m; }
int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
static bool env_flag(const char* name, bool dflt) {
  const char* v = getenv(name);
  if (!v || !*v) return dflt;
  return !(v[0] == '0' || v[0] == 'n' || v[0] == 'N' || v[0] == 'f' || v[0] == 'F');
}
}  // namespace ptts

using namespace ptts;

struct ptts_session {
  ptts_decoder_config cfg;
  DecoderLayout L;
  WorkspaceLayout W;
  const char* blob;
  char* ws;
  int sm_count;
  bool use_graph;
  bool has_prompt_mask, has_enc_mask, begun, prefilled;
  ptts_gen_params gen;
  cudaStream_t cap_stream;
  cudaGraphExec_t exec;
  bool graph_ready;
  int64_t launches;  // kernels launched through this session (bench.py reports it)
  long long* prof;
  bool fused;        // decode steps run as the single persistent kernel (step.cu) instead of 8L+3 kernels
  bool cluster;      // ... and that kernel is the cluster variant (step2.cu: 6 device-wide phases per layer)
  StepParams sp;
  // prefill linear layers as tcgen05 GEMMs (gemm_tc.cu) over the row-major weight copies ptts_decoder_finalize leaves in the
  // blob (layout.h rm[]); PTTS_PREFILL_TC=0 keeps the mma.sync kernel (A/B runs)
  bool prefill_tc;
  int max_prefix;    // decoder columns ptts_prefill_ids may take (workspace rows B * (P + max_prefix))
};

extern "C" {

const char* ptts_last_error(void) { return g_err.c_str(); }
int ptts_version(void) { return 100; }

// ---- weights ------------------------------------------------------------------------------------
int ptts_decoder_blob_bytes(const ptts_decoder_config* cfg, int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes, "null argument");
  if (int e = validate_config(*cfg)) return e;
  *out_bytes = make_layout(*cfg).total;
  return PTTS_OK;
}

int ptts_decoder_pack(const ptts_decoder_config* cfg, void* blob, int32_t tensor_id, int32_t index, const void* src,
                      int32_t src_dtype, int64_t rows, int64_t cols, void* stream) {
  PTTS_REQUIRE(cfg && blob && src, "null argument");
  if (int e = validate_config(*cfg)) return e;
  PTTS_REQUIRE(src_dtype == PTTS_BF16 || src_dtype == PTTS_F32, "pack: src dtype must be bf16 or f32");
  const DecoderLayout L = make_layout(*cfg);
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)blob;
  MatSlot ms;
  const bool per_layer = (tensor_id >= PTTS_T_LN1_W && tensor_id <= PTTS_T_FC2);
  if (per_layer) PTTS_REQUIRE(index >= 0 && index < L.L, "pack: layer %d out of range", index);
  if (matrix_slot(L, tensor_id, index, &ms)) {
    if (tensor_id == PTTS_T_LM_HEAD) PTTS_REQUIRE(index >= 0 && index < L.K, "pack: codebook %d out of range", index);
    PTTS_REQUIRE(cols == ms.K, "pack: tensor %d expects %d columns, got %lld", tensor_id, ms.K, (long long)cols);
    PTTS_REQUIRE(rows > 0 && ms.row_off + rows <= ms.N, "pack: tensor %d rows %lld do not fit fused matrix of %d rows", tensor_id, (long long)rows, ms.N);
    return pack_matrix(src, src_dtype, rows, cols, ms.row_off, ms.K, base + ms.off, cfg->dtype, st);
  }
  const int64_t lb = L.layer0 + L.layer_stride * index;
  const int H = L.H;
  switch (tensor_id) {
    case PTTS_T_EMBED_TOKENS:
      PTTS_REQUIRE(index >= 0 && index < L.K && rows == L.V + 1 && cols == H, "pack: embed_tokens shape");
      return pack_plain(src, src_dtype, rows * cols, base + L.embed + (int64_t)index * (L.V + 1) * H * L.es, cfg->dtype, st);
    case PTTS_T_POS_TABLE:
      PTTS_REQUIRE(!cfg->rope && rows == cfg->max_positions && cols == H, "pack: pos table shape");
      return pack_plain(src, src_dtype, rows * cols, base + L.pos, cfg->dtype, st);
    case PTTS_T_ROPE_COS:
    case PTTS_T_ROPE_SIN:
      PTTS_REQUIRE(cfg->rope && rows == cfg->max_positions && cols == PTTS_HEAD_DIM, "pack: rope table shape");
      return pack_plain(src, src_dtype, rows * cols, base + (tensor_id == PTTS_T_ROPE_COS ? L.rope_cos : L.rope_sin), cfg->dtype, st);
    case PTTS_T_LN1_W: case PTTS_T_LN1_B: case PTTS_T_LN2_W: case PTTS_T_LN2_B: case PTTS_T_LN3_W: case PTTS_T_LN3_B: {
      PTTS_REQUIRE(rows * cols == H, "pack: LayerNorm parameter must have %d elements", H);
      const int64_t off[6] = {L.ln1_w, L.ln1_b, 0, 0, 0, 0};
      (void)off;
      int64_t o = 0;
      switch (tensor_id) {
        case PTTS_T_LN1_W: o = L.ln1_w; break; case PTTS_T_LN1_B: o = L.ln1_b; break;
        case PTTS_T_LN2_W: o = L.ln2_w; break; case PTTS_T_LN2_B: o = L.ln2_b; break;
        case PTTS_T_LN3_W: o = L.ln3_w; break; default: o = L.ln3_b; break;
      }
      return pack_plain(src, src_dtype, H, base + lb + o, PTTS_F32, st);
    }
    case PTTS_T_FINAL_LN_W:
    case PTTS_T_FINAL_LN_B:
      PTTS_REQUIRE(rows * cols == H, "pack: LayerNorm parameter must have %d elements", H);
      return pack_plain(src, src_dtype, H, base + (tensor_id == PTTS_T_FINAL_LN_W ? L.final_ln_w : L.final_ln_b), PTTS_F32, st);
    default:
      return fail(PTTS_EINVAL, "pack: unknown tensor id %d", tensor_id);
  }
}

int ptts_decoder_finalize(const ptts_decoder_config* cfg, void* blob, void* stream) {
  PTTS_REQUIRE(cfg && blob, "null argument");
  if (int e = validate_config(*cfg)) return e;
  if (cfg->dtype != PTTS_BF16) return PTTS_OK;  // the f32 path applies LayerNorm explicitly
  const DecoderLayout L = make_layout(*cfg);
  cudaStream_t st = (cudaStream_t)stream;
  char* b = (char*)blob;
  for (int i = 0; i < L.L; i++) {
    char* lb = b + L.layer0 + L.layer_stride * i;
    float* cq = (float*)(lb + L.c_qkv);
    if (int e = fold_layernorm(lb + L.wqkv, L.qkv_rows, L.H, (const float*)(lb + L.ln1_w), (const float*)(lb + L.ln1_b), cq, cq + L.qkv_rows, st)) return e;
    float* cc = (float*)(lb + L.c_qc);
    if (int e = fold_layernorm(lb + L.wqc, L.H, L.H, (const float*)(lb + L.ln2_w), (const float*)(lb + L.ln2_b), cc, cc + L.H, st)) return e;
    float* cf = (float*)(lb + L.c_fc1);
    if (int e = fold_layernorm(lb + L.fc1, L.F, L.H, (const float*)(lb + L.ln3_w), (const float*)(lb + L.ln3_b), cf, cf + L.F, st)) return e;
  }
  float* ch = (float*)(b + L.c_heads);
  if (int e = fold_layernorm(b + L.heads, L.K * L.V, L.H, (const float*)(b + L.final_ln_w), (const float*)(b + L.final_ln_b), ch, ch + L.K * L.V, st)) return e;
  {  // row-major copies for the tcgen05 prefill GEMM (gemm_tc.cu), unpacked AFTER the LayerNorm fold
    const struct { int64_t off; int64_t N; int K; } mats[7] = {{L.wqkv, L.qkv_rows, L.H}, {L.wo, L.H, L.H}, {L.wqc, L.H, L.H}, {L.wkvc, L.ckv_rows, L.H},
                                                               {L.woc, L.H, L.H}, {L.fc1, L.F, L.H}, {L.fc2, L.H, L.F}};
    for (int i = 0; i < L.L; i++) {
      char* lb = b + L.layer0 + L.layer_stride * i;
      for (int m = 0; m < 7; m++)
        if (int e = unpack_fragments(lb + mats[m].off, lb + L.rm[m], mats[m].N, mats[m].K, st)) return e;
    }
  }
  if (L.cl_NC > 0) {  // second copy of the layer matrices, sliced per (phase, cluster, rank) for the cluster step kernel (step2.cu)
    const int64_t mat_off[6] = {L.wqkv, L.wo, L.wqc, L.woc, L.fc1, L.fc2};
    for (int i = 0; i < L.L; i++) {
      char* lb = b + L.layer0 + L.layer_stride * i;
      if (int e = cluster_pack_layer(lb, lb, mat_off, L.cp, L.nh, L.H, L.F, st)) return e;
    }
  }
  return PTTS_OK;
}

int ptts_workspace_bytes_ex(const ptts_decoder_config* cfg, int32_t B, int32_t P, int32_t S, int32_t max_cache_len, int32_t max_prefix,
                            int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes, "null argument");
  if (int e = validate_config(*cfg)) return e;
  PTTS_REQUIRE(B > 0 && P >= 0 && S > 0 && max_cache_len > P, "workspace: need B>0, P>=0, S>0, max_cache_len>P (got %d %d %d %d)", B, P, S, max_cache_len);
  PTTS_REQUIRE(max_prefix >= 1 && P + max_prefix <= max_cache_len, "workspace: max_prefix %d out of [1, max_cache_len - P]", max_prefix);
  *out_bytes = make_workspace(*cfg, B, P, S, max_cache_len, max_prefix).total;
  return PTTS_OK;
}
int ptts_workspace_bytes(const ptts_decoder_config* cfg, int32_t B, int32_t P, int32_t S, int32_t max_cache_len, int64_t* out_bytes) {
  return ptts_workspace_bytes_ex(cfg, B, P, S, max_cache_len, 1, out_bytes);
}

// ---- session ------------------------------------------------------------------------------------
int ptts_session_create_ex(const ptts_decoder_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes,
                           int32_t B, int32_t P, int32_t S, int32_t max_cache_len, int32_t max_prefix, ptts_session** out) {
  PTTS_REQUIRE(cfg && blob && workspace && out, "null argument");
  if (int e = validate_config(*cfg)) return e;
  PTTS_REQUIRE(B > 0 && P >= 0 && S > 0 && max_cache_len > P, "session: bad shape B=%d P=%d S=%d Tmax=%d", B, P, S, max_cache_len);
  PTTS_REQUIRE(max_prefix >= 1 && P + max_prefix <= max_cache_len, "session: max_prefix %d out of [1, max_cache_len - P]", max_prefix);
  PTTS_REQUIRE(max_cache_len <= cfg->max_positions, "session: cache length %d exceeds max_position_embeddings %d", max_cache_len, cfg->max_positions);
  ptts_session* s = new (std::nothrow) ptts_session();
  PTTS_REQUIRE(s, "out of host memory");
  s->cfg = *cfg;
  s->L = make_layout(*cfg);
  s->W = make_workspace(*cfg, B, P, S, max_cache_len, max_prefix);
  s->max_prefix = max_prefix;
  if (workspace_bytes < s->W.total) {
    int64_t need = s->W.total;
    delete s;
    return fail(PTTS_EINVAL, "session: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)need);
  }
  s->blob = (const char*)blob;
  s->ws = (char*)workspace;
  int dev = 0;
  cudaGetDevice(&dev);
  s->sm_count = 148;
  cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, dev);
  s->use_graph = env_flag("PTTS_GRAPH", true);
  s->graph_ready = false;
  s->exec = nullptr;
  s->cap_stream = nullptr;
  s->begun = s->prefilled = false;
  s->fused = false;
  s->cluster = false;
  s->prof = nullptr;
  s->launches = 0;
  s->prefill_tc = (cfg->dtype == PTTS_BF16) && env_flag("PTTS_PREFILL_TC", true);
  *out = s;
  return PTTS_OK;
}
int ptts_session_create(const ptts_decoder_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes,
                        int32_t B, int32_t P, int32_t S, int32_t max_cache_len, ptts_session** out) {
  return ptts_session_create_ex(cfg, blob, workspace, workspace_bytes, B, P, S, max_cache_len, 1, out);
}

int ptts_session_destroy(ptts_session* s) {
  if (!s) return PTTS_OK;
  if (s->exec) cudaGraphExecDestroy(s->exec);
  if (s->cap_stream) cudaStreamDestroy(s->cap_stream);
  delete s;
  return PTTS_OK;
}

static SampleArgs sample_args(ptts_session* s) {
  SampleArgs a{};
  const WorkspaceLayout& W = s->W;
  a.logits = (const float*)(s->ws + W.logits);
  a.scores = (float*)(s->ws + W.scores);
  a.raw_ids = (int64_t*)(s->ws + W.raw_ids);
  a.raw_ld = W.raw_ld;
  a.cur_ids = (int*)(s->ws + W.cur_ids);
  a.eos_seen = (int*)(s->ws + W.eos_seen);
  a.unfinished = (int*)(s->ws + W.unfinished);
  a.first_unf = (int*)(s->ws + W.first_unf);
  a.ctrl = (Ctrl*)(s->ws + W.ctrl);
  a.gen = (const ptts_gen_params*)(s->ws + W.gen);
  a.B = W.B; a.K = s->cfg.num_codebooks; a.V = s->cfg.vocab_size;
  a.bos = s->cfg.bos_token_id; a.pad = s->cfg.pad_token_id; a.eos = s->cfg.eos_token_id;
  return a;
}


// Fused-step schedule: largest n-tile count that keeps ~one task per CTA.
static int pick_nt(int ntiles, int grid) {
  const int cand[4] = {4, 3, 2, 1};  // the variants instantiated in step.cu::run_gemm
  for (int i = 0; i < 4; i++)
    if (ntiles % cand[i] == 0 && ntiles / cand[i] >= (grid * 8) / 10) return cand[i];
  for (int i = 0; i < 4; i++)
    if (ntiles % cand[i] == 0 && ntiles / cand[i] >= grid / 2) return cand[i];
  return 1;
}

// The fused kernel covers bf16, B <= 32, K <= 16: anything else runs the 8L+3-kernel path -- a 2x slower step.  Say so once per
// process instead of degrading silently, and count it (ptts_session_fused reports which path a session uses).
static bool fused_declined(ptts_session* s, const char* why) {
  static bool warned = false;
  if (!warned) {
    fprintf(stderr, "ptts_b200: fused decode step not used for this session (B=%d, H=%d, K=%d: %s); decode steps run the multi-kernel path\n",
            s->W.B, s->L.H, s->L.K, why);
    warned = true;
  }
  return false;
}

static bool setup_fused(ptts_session* s) {
  const ptts_decoder_config& c = s->cfg;
  const DecoderLayout& L = s->L;
  const WorkspaceLayout& W = s->W;
  if (c.dtype != PTTS_BF16 || !env_flag("PTTS_FUSED", true)) return false;
  if (W.B > 32 || L.K > 16 || L.H % 64 != 0 || L.F % L.H != 0) return fused_declined(s, "batch > 32 rows, > 16 codebooks or an unsupported width");
  StepParams& p = s->sp;
  memset(&p, 0, sizeof(p));
  p.B = W.B; p.H = L.H; p.F = L.F; p.V = L.V; p.K = L.K; p.L = L.L; p.nh = L.nh; p.nkv = L.nkv; p.nckv = L.nckv;
  p.S = W.S; p.P = W.P; p.Tmax = W.Tmax; p.rope = c.rope; p.act = c.activation; p.qkv_rows = L.qkv_rows;
  p.eps = c.layer_norm_eps; p.scale = 0.125f;
  p.blob = s->blob;
  p.embed = L.embed; p.pos = L.pos; p.layer0 = L.layer0; p.layer_stride = L.layer_stride;
  p.wqkv = L.wqkv; p.wo = L.wo; p.wqc = L.wqc; p.woc = L.woc; p.fc1 = L.fc1; p.fc2 = L.fc2;
  p.c_qkv = L.c_qkv; p.c_qc = L.c_qc; p.c_fc1 = L.c_fc1; p.c_heads = L.c_heads;
  p.heads = L.heads; p.rope_cos = L.rope_cos; p.rope_sin = L.rope_sin;
  char* ws = s->ws;
  p.x = (bf16*)(ws + W.img_x); p.qkv = (bf16*)(ws + W.qkv); p.attn = (bf16*)(ws + W.img_attn); p.qc = (bf16*)(ws + W.qc); p.hbuf = (bf16*)(ws + W.img_h);
  p.logits = (float*)(ws + W.logits);
  p.cross_kv = ws + W.cross_kv; p.cross_layer_stride = W.cross_layer_stride;
  p.self_kv = ws + W.self_kv; p.self_layer_stride = W.self_layer_stride;
  p.prompt_mask = s->has_prompt_mask ? (const int*)(ws + W.prompt_mask) : nullptr;
  p.enc_mask = s->has_enc_mask ? (const int*)(ws + W.enc_mask) : nullptr;
  p.sa = sample_args(s);
  p.bar = ((Ctrl*)(ws + W.ctrl))->bar;
  p.progress = (int*)(ws + W.progress);
  const int G = s->sm_count;
  p.nt_qkv = pick_nt(L.qkv_rows / 8, G);
  p.nt_h = pick_nt(L.H / 8, G);
  p.nt_fc1 = pick_nt(L.F / 8, G);
  p.nt_heads = pick_nt(L.K * L.V / 8, G);
  int ntmax = p.nt_qkv;
  if (p.nt_h > ntmax) ntmax = p.nt_h;
  if (p.nt_fc1 > ntmax) ntmax = p.nt_fc1;
  if (p.nt_heads > ntmax) ntmax = p.nt_heads;
  const int64_t tile = (int64_t)32 * (L.H + 8) * 2;
  const int64_t red = (int64_t)8 * 32 * (8 * ntmax + 8) * 4;  // K-reduction scratch [8 warps][32][RS], step.cu
  // weight buffer: the largest per-task slice (nt n-tiles x K, 16 bytes per (n-tile, k-pair) fragment row)
  int64_t wbytes = (int64_t)p.nt_qkv * L.H * 16;
  if ((int64_t)p.nt_h * L.F * 16 > wbytes) wbytes = (int64_t)p.nt_h * L.F * 16;
  if ((int64_t)p.nt_fc1 * L.H * 16 > wbytes) wbytes = (int64_t)p.nt_fc1 * L.H * 16;
  if ((int64_t)p.nt_heads * L.H * 16 > wbytes) wbytes = (int64_t)p.nt_heads * L.H * 16;
  const int64_t att = (int64_t)8 * (2 * 2 * 32 * 64 * 2 + 3 * 64 * 4) + 4 * 128 * 4;  // 8 x attn_decode_smem_per_warp<bf16>() + pair exchange
  const int64_t budget = 215 * 1024 - 2816;  // step.cu ST_HEADER
  p.nbuf = (2 * tile + wbytes <= budget) ? 2 : 1;
  if (p.nbuf * tile < red) return fused_declined(s, "the K-reduction scratch does not fit the activation tile");
  p.wbuf_offset = align_up(p.nbuf * tile, 128);
  int64_t region = p.wbuf_offset + wbytes;
  if (att > region) region = att;
  region = align_up(region, 16);
  if (region > budget) return fused_declined(s, "tile + weight slice exceed the shared memory of an SM");
  p.tile_region_bytes = region;
  p.sample_items = (L.V + 255) / 256;
  if (p.sample_items > 9) return fused_declined(s, "vocab_size > 2304");
  p.do_sample_phase = 1;
  p.prof = s->prof;
  // cluster variant (step2.cu) when the shape and the device allow it; PTTS_STEP=legacy keeps step.cu (A/B runs, cross-checks)
  for (int i = 0; i < 6; i++) { p.cp[i] = L.cp[i]; p.cp_slice[i] = L.cp_slice[i]; }
  p.cl_x = (bf16*)(ws + W.cl_x); p.cl_attn = (bf16*)(ws + W.cl_attn); p.cl_h = (bf16*)(ws + W.cl_h);
  const char* mode = getenv("PTTS_STEP");
  s->cluster = L.cl_NC > 0 && !(mode && strcmp(mode, "legacy") == 0) && cluster_step_available(p);
  return true;
}

int ptts_generate_begin(ptts_session* s, const ptts_gen_params* gen, void* stream) {
  PTTS_REQUIRE(s && gen, "null argument");
  PTTS_REQUIRE(gen->max_length >= 2, "generate: max_length must be >= 2, got %d", gen->max_length);
  PTTS_REQUIRE(gen->max_length <= s->W.raw_ld, "generate: max_length %d exceeds the session's capacity %lld", gen->max_length, (long long)s->W.raw_ld);
  PTTS_REQUIRE(!gen->do_sample || gen->temperature > 0.f, "`temperature` has to be a strictly positive float, got %f", gen->temperature);
  PTTS_REQUIRE(gen->top_k >= 0, "`top_k` has to be a non-negative integer");
  PTTS_REQUIRE(s->cfg.eos_token_id >= 0 && s->cfg.eos_token_id < s->cfg.vocab_size, "eos_token_id out of vocabulary");
  cudaStream_t st = (cudaStream_t)stream;
  s->gen = *gen;
  PTTS_CHECK_CUDA(cudaMemcpyAsync(s->ws + s->W.gen, &s->gen, sizeof(ptts_gen_params), cudaMemcpyHostToDevice, st));
  if (int e = launch_generate_begin(sample_args(s), st)) return e;
  s->begun = true;
  s->prefilled = false;
  return PTTS_OK;
}

// one decoder pass over q_len new positions per batch row (q_len = P + n_cols at prefill, 1 at decode); col_ids: the prefill's
// [B*K][n_cols] decoder ids, or nullptr for the single staged column
static int run_forward(ptts_session* s, cudaStream_t st, bool prefill, const void* prompt_hidden, const void* enc_hidden,
                       int n_cols = 1, const int64_t* col_ids = nullptr) {
  const ptts_decoder_config& c = s->cfg;
  const DecoderLayout& L = s->L;
  const WorkspaceLayout& W = s->W;
  const int B = W.B, P = W.P, S = W.S, H = L.H, D = PTTS_HEAD_DIM;
  const int q_len = prefill ? P + n_cols : 1;
  const int M = B * q_len;
  const bool pdl = !prefill;  // the one-off prefill stays on plain stream order
  const Ctrl* ctrl = prefill ? nullptr : (const Ctrl*)(s->ws + W.ctrl);
  const int es = L.es;
  char* ws = s->ws;
  const char* blob = s->blob;

  EmbedArgs ea{};
  ea.tables = blob + L.embed;
  ea.pos = c.rope ? nullptr : blob + L.pos;
  ea.prefix = prefill ? prompt_hidden : nullptr;
  ea.ids = (const int*)(ws + W.cur_ids);
  ea.x = ws + W.x;
  ea.ctrl = ctrl;
  ea.B = B; ea.K = L.K; ea.V1 = L.V + 1; ea.H = H; ea.P = prefill ? P : 0;
  ea.pos_from_ctrl = prefill ? 0 : 1; ea.pos0 = 0; ea.prefix_len = P;
  ea.n_cols = prefill ? n_cols : 1; ea.col_ids = prefill ? col_ids : nullptr;
  if (int e = launch_embed(ea, c.dtype, st, pdl)) return e;
  s->launches++;

  auto lin = [&](const void* X, int64_t ldx, int64_t woff, int N, int K, const float* lw, const float* lb, int epi,
                 const void* R, void* Y, int64_t ldy, int Mrows, int64_t coff = -1) -> int {
    LinearArgs a{};
    a.X = X; a.ldx = ldx; a.W = blob + woff; a.Y = Y; a.ldy = ldy; a.R = R; a.ldr = ldy;
    a.ln_w = lw; a.ln_b = lb; a.eps = c.layer_norm_eps;
    if (lw != nullptr && c.dtype == PTTS_BF16) {  // bf16: LayerNorm folded into the weights at load (ptts_decoder_finalize)
      a.c1 = (const float*)(blob + coff); a.c2 = a.c1 + N;
    }
    a.M = Mrows; a.N = N; a.K = K; a.Kc = (K > H && K % H == 0) ? H : K;
    a.epi = epi; a.act = c.activation; a.ctrl = ctrl;
    s->launches++;
    if (prefill && s->prefill_tc && woff >= L.layer0 && woff < L.layer0 + L.layer_stride * L.L && linear_tc_supported(a)) {
      // the same matrix, row-major (layout.h rm[]): M = B*(P+1) or B*S rows are tensor-core work (tcgen05, gemm_tc.cu)
      const int64_t in_layer = (woff - L.layer0) % L.layer_stride, lbase = woff - in_layer;
      const int64_t frag[7] = {L.wqkv, L.wo, L.wqc, L.wkvc, L.woc, L.fc1, L.fc2};
      for (int m = 0; m < 7; m++)
        if (in_layer == frag[m]) {
          if (a.c1 != nullptr) s->launches++;  // row statistics kernel
          return launch_linear_tc(a, blob + lbase + L.rm[m], (float*)(ws + W.row_stats), st);
        }
    }
    return launch_linear(a, c.dtype, st, pdl, s->sm_count);
  };

  for (int i = 0; i < L.L; i++) {
    const int64_t lb = L.layer0 + L.layer_stride * i;
    char* x = ws + W.x;
    if (prefill) {  // cross-attention K/V of the encoder states, once per generate() (:872-878)
      if (int e = lin(enc_hidden, H, lb + L.wkvc, L.ckv_rows, H, nullptr, nullptr, EPI_STORE, nullptr,
                      ws + W.cross_tmp, L.ckv_rows, B * S)) return e;
      if (int e = launch_cross_kv_relayout(ws + W.cross_tmp, ws + W.cross_kv + W.cross_layer_stride * i, B, S, L.nckv, c.dtype, st)) return e;
      s->launches++;
    }
    if (int e = lin(x, H, lb + L.wqkv, L.qkv_rows, H, (const float*)(blob + lb + L.ln1_w), (const float*)(blob + lb + L.ln1_b),
                    EPI_STORE, nullptr, ws + W.qkv, L.qkv_rows, M, lb + L.c_qkv)) return e;
    AttnArgs at{};
    at.q = ws + W.qkv; at.ldq = L.qkv_rows; at.q_col0 = 0;
    at.knew = ws + W.qkv; at.vnew = ws + W.qkv; at.ldkv = L.qkv_rows; at.k_col0 = L.nh * D; at.v_col0 = (L.nh + L.nkv) * D;
    char* kc = ws + W.self_kv + W.self_layer_stride * i;
    at.kcache = kc; at.vcache = kc + (int64_t)B * L.nkv * W.Tmax * D * es;
    at.kv_b_stride = (int64_t)L.nkv * W.Tmax * D; at.kv_h_stride = (int64_t)W.Tmax * D; at.kv_t_stride = D;
    at.out = ws + W.attn; at.ldo = H;
    at.key_mask = s->has_prompt_mask ? (const int*)(ws + W.prompt_mask) : nullptr; at.mask_len = P; at.mask_ld = P;
    at.ctrl = ctrl; at.B = B; at.nh = L.nh; at.nkv = L.nkv; at.q_len = q_len;
    at.past_from_ctrl = prefill ? 0 : 1; at.past_len = 0; at.prefix = P;
    at.cross = 0; at.kv_len = 0;
    at.rope = c.rope; at.rope_cos = blob + L.rope_cos; at.rope_sin = blob + L.rope_sin;
    at.kv_capacity = prefill ? q_len : W.Tmax;
    at.scale = 0.125f;  // head_dim ** -0.5, applied inside SDPA (quirk Q1)
    if (int e = launch_attention(at, c.dtype, st, pdl)) return e;
    s->launches++;
    if (int e = lin(ws + W.attn, H, lb + L.wo, H, H, nullptr, nullptr, EPI_RESIDUAL, x, x, H, M)) return e;
    if (int e = lin(x, H, lb + L.wqc, H, H, (const float*)(blob + lb + L.ln2_w), (const float*)(blob + lb + L.ln2_b),
                    EPI_STORE, nullptr, ws + W.qc, H, M, lb + L.c_qc)) return e;
    AttnArgs ct = at;
    ct.q = ws + W.qc; ct.ldq = H; ct.q_col0 = 0;
    ct.knew = ct.vnew = nullptr;
    char* ck = ws + W.cross_kv + W.cross_layer_stride * i;
    ct.kcache = ck; ct.vcache = ck + (int64_t)B * L.nckv * S * D * es;   // item-major: K [B][nckv][S][64] | V [...]
    ct.kv_b_stride = (int64_t)L.nckv * S * D; ct.kv_h_stride = (int64_t)S * D; ct.kv_t_stride = D;
    ct.key_mask = s->has_enc_mask ? (const int*)(ws + W.enc_mask) : nullptr; ct.mask_len = S; ct.mask_ld = S;
    ct.nkv = L.nckv; ct.cross = 1; ct.kv_len = S; ct.kv_capacity = S;
    if (int e = launch_attention(ct, c.dtype, st, pdl)) return e;
    s->launches++;
    if (int e = lin(ws + W.attn, H, lb + L.woc, H, H, nullptr, nullptr, EPI_RESIDUAL, x, x, H, M)) return e;
    if (int e = lin(x, H, lb + L.fc1, L.F, H, (const float*)(blob + lb + L.ln3_w), (const float*)(blob + lb + L.ln3_b),
                    EPI_ACT, nullptr, ws + W.hbuf, L.F, M, lb + L.c_fc1)) return e;
    if (int e = lin(ws + W.hbuf, L.F, lb + L.fc2, H, L.F, nullptr, nullptr, EPI_RESIDUAL, x, x, H, M)) return e;
  }
  // final LayerNorm + K lm heads on the last position of every batch row -> f32 logits [B, K*V] == [B*K, V]
  const char* xlast = ws + W.x + (int64_t)(q_len - 1) * H * es;
  return lin(xlast, (int64_t)q_len * H, L.heads, L.K * L.V, H, (const float*)(blob + L.final_ln_w), (const float*)(blob + L.final_ln_b),
             EPI_F32, nullptr, ws + W.logits, (int64_t)L.K * L.V, B, L.c_heads);
}

static int prefill_common(ptts_session* s, const void* prompt_hidden, const int64_t* prompt_mask, const void* enc_hidden,
                          const int64_t* enc_mask, const int64_t* prefix_ids, int n, cudaStream_t st) {
  PTTS_REQUIRE(s && enc_hidden, "null argument");
  if (!s->begun) return fail(PTTS_ESTATE, "ptts_prefill called before ptts_generate_begin");
  PTTS_REQUIRE(s->W.P == 0 || prompt_hidden, "prefill: prompt_hidden is required when P > 0");
  if (prefix_ids != nullptr) {
    // raw_ids[:, :n] = the given columns, cur_len = n: ptts_sample then appends column n
    PTTS_CHECK_CUDA(cudaMemcpy2DAsync(s->ws + s->W.raw_ids, (size_t)s->W.raw_ld * 8, prefix_ids, (size_t)n * 8, (size_t)n * 8, s->W.BK,
                                      cudaMemcpyDeviceToDevice, st));
    const int cur_len = n;
    PTTS_CHECK_CUDA(cudaMemcpyAsync(s->ws + s->W.ctrl + offsetof(Ctrl, cur_len), &cur_len, sizeof(int), cudaMemcpyHostToDevice, st));
  }
  s->has_prompt_mask = (prompt_mask != nullptr && s->W.P > 0);
  s->has_enc_mask = (enc_mask != nullptr);
  if (s->has_prompt_mask) { if (int e = launch_mask_convert(prompt_mask, s->W.B * s->W.P, (int*)(s->ws + s->W.prompt_mask), st)) return e; }
  if (s->has_enc_mask) { if (int e = launch_mask_convert(enc_mask, s->W.B * s->W.S, (int*)(s->ws + s->W.enc_mask), st)) return e; }
  if (int e = run_forward(s, st, true, prompt_hidden, enc_hidden, n, prefix_ids)) return e;
  s->prefilled = true;
  s->fused = setup_fused(s);
  // mask presence is baked into the captured graph: re-capture if it changed
  if (s->exec) { cudaGraphExecDestroy(s->exec); s->exec = nullptr; s->graph_ready = false; }
  return PTTS_OK;
}
int ptts_prefill(ptts_session* s, const void* prompt_hidden, const int64_t* prompt_mask, const void* enc_hidden,
                 const int64_t* enc_mask, void* stream) {
  return prefill_common(s, prompt_hidden, prompt_mask, enc_hidden, enc_mask, nullptr, 1, (cudaStream_t)stream);
}
int ptts_prefill_ids(ptts_session* s, const void* prompt_hidden, const int64_t* prompt_mask, const void* enc_hidden,
                     const int64_t* enc_mask, const int64_t* prefix_ids, int32_t n, void* stream) {
  PTTS_REQUIRE(s && prefix_ids, "null argument");
  PTTS_REQUIRE(n >= 1 && n <= s->max_prefix, "prefill_ids: n = %d out of [1, max_prefix = %d]", n, s->max_prefix);
  PTTS_REQUIRE(!s->begun || n < s->gen.max_length, "prefill_ids: n = %d leaves no new token below max_length %d", n, s->gen.max_length);
  return prefill_common(s, prompt_hidden, prompt_mask, enc_hidden, enc_mask, prefix_ids, n, (cudaStream_t)stream);
}

int ptts_decode_forward(ptts_session* s, void* stream) {
  PTTS_REQUIRE(s, "null argument");
  if (!s->prefilled) return fail(PTTS_ESTATE, "ptts_decode_forward called before ptts_prefill");
  if (s->fused) {
    StepParams p = s->sp;
    p.do_sample_phase = 0;
    s->launches++;
    if (s->cluster) return launch_decode_step_cluster(p, (cudaStream_t)stream);
    return launch_decode_step(p, s->sm_count, (cudaStream_t)stream);
  }
  return run_forward(s, (cudaStream_t)stream, false, nullptr, nullptr);
}

int ptts_sample(ptts_session* s, const int64_t* forced_tokens, void* stream) {
  PTTS_REQUIRE(s, "null argument");
  if (!s->prefilled) return fail(PTTS_ESTATE, "ptts_sample called before ptts_prefill");
  s->launches++;
  return launch_sample(sample_args(s), forced_tokens, (cudaStream_t)stream, false);
}

int ptts_decode_steps(ptts_session* s, int32_t n_steps, void* stream) {
  PTTS_REQUIRE(s && n_steps >= 0, "bad argument");
  if (!s->prefilled) return fail(PTTS_ESTATE, "ptts_decode_steps called before ptts_prefill");
  cudaStream_t st = (cudaStream_t)stream;
  if (s->fused && s->cluster) {  // the cluster kernel loops over tokens itself: up to PTTS_STEPS_PER_LAUNCH (default 64) per launch
    const char* env = getenv("PTTS_STEPS_PER_LAUNCH");   // (read per call: tests compare 1 against the default)
    const int per_launch = env ? (atoi(env) < 1 ? 1 : atoi(env)) : 64;
    for (int done = 0; done < n_steps;) {
      const int m = (n_steps - done < per_launch) ? n_steps - done : per_launch;
      s->sp.n_steps = m;
      const int e = launch_decode_step_cluster(s->sp, st);
      s->sp.n_steps = 1;
      if (e) return e;
      done += m;
      s->launches += 1;
    }
    return PTTS_OK;
  }
  if (s->fused) {  // one persistent kernel per token: nothing to gain from a graph
    for (int i = 0; i < n_steps; i++)
      if (int e = launch_decode_step(s->sp, s->sm_count, st)) return e;
    s->launches += n_steps;
    return PTTS_OK;
  }
  if (!s->use_graph) {
    for (int i = 0; i < n_steps; i++) {
      if (int e = run_forward(s, st, false, nullptr, nullptr)) return e;
      s->launches++;
      if (int e = launch_sample(sample_args(s), nullptr, st, true)) return e;
    }
    return PTTS_OK;
  }
  if (!s->graph_ready) {
    if (!s->cap_stream) PTTS_CHECK_CUDA(cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking));
    const int64_t before = s->launches;
    PTTS_CHECK_CUDA(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
    int e = run_forward(s, s->cap_stream, false, nullptr, nullptr);
    if (!e) { s->launches++; e = launch_sample(sample_args(s), nullptr, s->cap_stream, true); }
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(s->cap_stream, &graph);
    s->launches = before;
    if (e) { if (graph) cudaGraphDestroy(graph); return e; }
    if (ce != cudaSuccess) return fail(PTTS_ECUDA, "graph capture failed: %s", cudaGetErrorString(ce));
    ce = cudaGraphInstantiate(&s->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return fail(PTTS_ECUDA, "graph instantiate failed: %s", cudaGetErrorString(ce));
    s->graph_ready = true;
  }
  const int per_step = 2 + 8 * s->L.L + 1;  // embed + 8 kernels/layer + heads + sample
  for (int i = 0; i < n_steps; i++) PTTS_CHECK_CUDA(cudaGraphLaunch(s->exec, st));
  s->launches += (int64_t)per_step * n_steps;
  return PTTS_OK;
}

int ptts_session_logits(ptts_session* s, float** out) { PTTS_REQUIRE(s && out, "null"); *out = (float*)(s->ws + s->W.logits); return PTTS_OK; }
int ptts_session_scores(ptts_session* s, float** out) { PTTS_REQUIRE(s && out, "null"); *out = (float*)(s->ws + s->W.scores); return PTTS_OK; }
int ptts_session_raw_ids(ptts_session* s, int64_t** out, int32_t* ld) {
  PTTS_REQUIRE(s && out && ld, "null");
  *out = (int64_t*)(s->ws + s->W.raw_ids);
  *ld = (int32_t)s->W.raw_ld;
  return PTTS_OK;
}
int ptts_session_state(ptts_session* s, int32_t** out) { PTTS_REQUIRE(s && out, "null"); *out = (int32_t*)(s->ws + s->W.ctrl); return PTTS_OK; }
// Debug / profiling aid: CTA 0 of the fused step kernel writes clock64() stamps per phase into `buf`
// (device int64 [(8L+2)*8]); pass NULL to switch it off.  Only the next launches are affected.
int ptts_session_set_profile(ptts_session* s, void* buf) {
  PTTS_REQUIRE(s, "null");
  s->prof = (long long*)buf;
  s->sp.prof = s->prof;
  return PTTS_OK;
}
int ptts_session_fused(ptts_session* s, int32_t* out) { PTTS_REQUIRE(s && out, "null"); *out = s->fused ? (s->cluster ? 2 : 1) : 0; return PTTS_OK; }
int ptts_session_launches(ptts_session* s, int64_t* out) { PTTS_REQUIRE(s && out, "null"); *out = s->launches; return PTTS_OK; }

// ---- stand-alone operators ----------------------------------------------------------------------
int ptts_delay_build(const int64_t* input_ids, int32_t BK, int32_t seq_len, int32_t num_codebooks, int64_t bos, int64_t pad,
                     int32_t max_length, int64_t* pattern_mask, void* stream) {
  PTTS_REQUIRE(input_ids && pattern_mask, "null argument");
  PTTS_REQUIRE(num_codebooks > 0 && BK > 0 && BK % num_codebooks == 0 && seq_len > 0 && max_length > 0, "delay_build: bad shape");
  return launch_delay_build(input_ids, BK, seq_len, num_codebooks, bos, pad, max_length, pattern_mask, (cudaStream_t)stream);
}
int ptts_delay_apply(const int64_t* input_ids, int32_t BK, int32_t seq_len, int64_t ld_ids, const int64_t* pattern_mask,
                     int64_t ld_mask, int64_t* out, void* stream) {
  PTTS_REQUIRE(input_ids && pattern_mask && out, "null argument");
  PTTS_REQUIRE(BK > 0 && seq_len > 0 && ld_mask >= seq_len && ld_ids >= seq_len, "delay_apply: mask shorter than ids");
  return launch_delay_apply(input_ids, BK, seq_len, ld_ids, pattern_mask, ld_mask, out, (cudaStream_t)stream);
}
int ptts_logits_processor(const int64_t* input_ids, int32_t BK, int32_t seq_len, int64_t ld_ids, float* scores, int32_t V,
                          int64_t eos, int32_t num_codebooks, int64_t* first_unfinished, void* stream) {
  PTTS_REQUIRE(input_ids && scores && first_unfinished, "null argument");
  return launch_logits_processor(input_ids, BK, seq_len, ld_ids, scores, V, eos, num_codebooks, first_unfinished, (cudaStream_t)stream);
}

int ptts_op_linear(const ptts_decoder_config* cfg, const void* blob, int32_t tensor_id, int32_t index, const void* x, int32_t M,
                   int32_t use_ln, int32_t epilogue, const void* residual, void* y, void* stream) {
  PTTS_REQUIRE(cfg && blob && x && y, "null argument");
  if (int e = validate_config(*cfg)) return e;
  const DecoderLayout L = make_layout(*cfg);
  MatSlot ms;
  PTTS_REQUIRE(matrix_slot(L, tensor_id, index, &ms), "op_linear: tensor %d is not a matrix", tensor_id);
  const int64_t lb = L.layer0 + L.layer_stride * index;
  LinearArgs a{};
  a.X = x; a.ldx = ms.K; a.W = (const char*)blob + ms.off; a.Y = y; a.ldy = ms.N; a.R = residual; a.ldr = ms.N;
  if (use_ln) {
    PTTS_REQUIRE(ms.K == L.H, "op_linear: LayerNorm needs K == hidden_size");
    int64_t w = 0, b = 0;
    switch (tensor_id) {
      case PTTS_T_SELF_Q: case PTTS_T_SELF_K: case PTTS_T_SELF_V: w = lb + L.ln1_w; b = lb + L.ln1_b; break;
      case PTTS_T_CROSS_Q: w = lb + L.ln2_w; b = lb + L.ln2_b; break;
      case PTTS_T_FC1: w = lb + L.ln3_w; b = lb + L.ln3_b; break;
      case PTTS_T_LM_HEAD: w = L.final_ln_w; b = L.final_ln_b; break;
      default: return fail(PTTS_EINVAL, "op_linear: tensor %d has no LayerNorm in front", tensor_id);
    }
    a.ln_w = (const float*)((const char*)blob + w);
    a.ln_b = (const float*)((const char*)blob + b);
    if (cfg->dtype == PTTS_BF16) {
      int64_t co = 0;
      switch (tensor_id) {
        case PTTS_T_SELF_Q: case PTTS_T_SELF_K: case PTTS_T_SELF_V: co = lb + L.c_qkv; break;
        case PTTS_T_CROSS_Q: co = lb + L.c_qc; break;
        case PTTS_T_FC1: co = lb + L.c_fc1; break;
        default: co = L.c_heads; break;
      }
      a.c1 = (const float*)((const char*)blob + co);
      a.c2 = a.c1 + ms.N;
    }
  }
  a.eps = cfg->layer_norm_eps;
  a.M = M; a.N = ms.N; a.K = ms.K; a.Kc = (ms.K > L.H && ms.K % L.H == 0) ? L.H : ms.K;
  a.epi = epilogue; a.act = cfg->activation; a.ctrl = nullptr;
  PTTS_REQUIRE(epilogue >= 0 && epilogue <= 3, "op_linear: bad epilogue");
  PTTS_REQUIRE(epilogue != EPI_RESIDUAL || residual, "op_linear: residual required");
  int sm = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
  return launch_linear(a, cfg->dtype, (cudaStream_t)stream, false, sm);
}

// ---- DAC ----------------------------------------------------------------------------------------
int ptts_dac_blob_bytes(const ptts_dac_config* cfg, int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes, "null argument");
  if (int e = validate_dac(*cfg)) return e;
  *out_bytes = make_dac_layout(*cfg).total;
  return PTTS_OK;
}
int ptts_dac_num_tensors(const ptts_dac_config* cfg, int32_t* out) {
  PTTS_REQUIRE(cfg && out, "null argument");
  if (int e = validate_dac(*cfg)) return e;
  *out = (int32_t)make_dac_layout(*cfg).t.size();
  return PTTS_OK;
}
int ptts_dac_pack(const ptts_dac_config* cfg, void* blob, int32_t name_id, const void* src, int32_t src_dtype, int64_t numel, void* stream) {
  PTTS_REQUIRE(cfg && blob && src, "null argument");
  if (int e = validate_dac(*cfg)) return e;
  PTTS_REQUIRE(src_dtype == PTTS_BF16 || src_dtype == PTTS_F32, "dac pack: src dtype must be bf16 or f32");
  const DacLayout L = make_dac_layout(*cfg);
  PTTS_REQUIRE(name_id >= 0 && name_id < (int)L.t.size(), "dac pack: tensor id %d out of range", name_id);
  const DacTensor& t = L.t[name_id];
  PTTS_REQUIRE(numel == t.numel, "dac pack: tensor %d expects %lld elements, got %lld", name_id, (long long)t.numel, (long long)numel);
  char* dst = (char*)blob + t.off;
  if (t.kind == DK_PLAIN) return pack_plain(src, src_dtype, numel, dst, cfg->dtype, (cudaStream_t)stream);
  if (t.off_k >= 0) {
    if (int e = pack_conv_kmajor(src, src_dtype, (char*)blob + t.off_k, t.d0, t.d1, t.k, t.kind == DK_CONVT, (cudaStream_t)stream)) return e;
  }
  return pack_conv(src, src_dtype, dst, cfg->dtype, t.d0, t.d1, t.k, t.kind == DK_CONVT, (cudaStream_t)stream);
}
int ptts_dac_workspace_bytes(const ptts_dac_config* cfg, int32_t B, int32_t T, int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes && B > 0 && T > 0, "bad argument");
  if (int e = validate_dac(*cfg)) return e;
  *out_bytes = 3 * align_up(dac_max_act_per_frame(*cfg) * B * T * dtype_size(cfg->dtype), 1024) + align_up((int64_t)cfg->latent_dim * B * T * dtype_size(cfg->dtype), 1024);
  return PTTS_OK;
}

int ptts_dac_decode(const ptts_dac_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes, const int64_t* codes,
                    int32_t B, int32_t T, void* audio_out, void* stream) {
  PTTS_REQUIRE(cfg && blob && workspace && codes && audio_out, "null argument");
  if (int e = validate_dac(*cfg)) return e;
  PTTS_REQUIRE(B > 0 && T > 0, "dac decode: empty input B=%d T=%d", B, T);
  const DacLayout L = make_dac_layout(*cfg);
  const int es = L.es;
  const int64_t half = align_up(dac_max_act_per_frame(*cfg) * B * T * es, 1024);
  const int64_t zbytes = align_up((int64_t)cfg->latent_dim * B * T * es, 1024);
  PTTS_REQUIRE(workspace_bytes >= 3 * half + zbytes, "dac decode: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const char* bl = (const char*)blob;
  char* cur = (char*)workspace;
  char* oth = cur + half;
  const int K = cfg->n_codebooks;
  // ---- tensor-core path: bf16 storage, every conv but the last (Cout = 1) as a tcgen05 implicit GEMM ----
  bool use_tc = (cfg->dtype == PTTS_BF16) && env_flag("PTTS_DAC_TC", true) && conv_tc_supported(cfg->latent_dim, cfg->decoder_dim);
  for (int bi = 0; bi < cfg->n_blocks && use_tc; bi++) use_tc = conv_tc_supported(cfg->decoder_dim >> bi, cfg->decoder_dim >> (bi + 1)) && conv_tc_supported(cfg->decoder_dim >> (bi + 1), cfg->decoder_dim >> (bi + 1));
  if (use_tc) {
    char* bufA = (char*)workspace;
    char* bufB = bufA + half;
    char* bufX = bufB + half;
    char* bufZ = bufX + half;
    FromCodesArgs fz{codes, bl + L.codebooks, bl + L.proj_w, bl + L.proj_b, bufZ, K, cfg->codebook_dim, cfg->latent_dim, T, cfg->codebook_size};
    if (int e = launch_from_codes(fz, cfg->dtype, B, st)) return e;
    int ti = 3 * K;
    auto tpk = [&](int i) { return bl + L.t[i].off_k; };
    auto tpp = [&](int i) { return bl + L.t[i].off; };
    auto convk = [&](const void* x, int w_i, int b_i, const void* res, void* out_raw, void* out_act, const void* alpha_next, int Cin, int Cout, int Tlen, int ks, int dil) {
      ConvArgs a{};
      a.x = x; a.bias = tpp(b_i); a.res = res;
      a.Cin = Cin; a.Cout = Cout; a.Tin = Tlen; a.Tout = Tlen; a.q_count = Tlen;
      a.n_taps = ks; a.off_base = -((ks - 1) / 2) * dil; a.off_step = dil; a.wt_base = 0; a.wt_step = 1;
      a.n_phase = 1; a.wt_phase_step = 0; a.o_mul = 1; a.o_add = 0; a.o_phase_step = 0;
      return launch_conv_tc(a, tpk(w_i), ks, alpha_next, out_raw, out_act, B, st);
    };
    const int C = cfg->decoder_dim;
    char* act = bufA;   // snake'd input of the next conv
    char* oth2 = bufB;
    // conv1: latent -> C, output only as snake_{block0.snake1}(y)
    if (int e = convk(bufZ, ti, ti + 1, nullptr, nullptr, act, tpp(ti + 2), cfg->latent_dim, C, T, 7, 1)) return e;
    ti += 2;
    int Tlen = T;
    for (int bi = 0; bi < cfg->n_blocks; bi++) {
      const int cin = C >> bi, cout = C >> (bi + 1), sd = cfg->strides[bi];
      const int pad = (sd + 1) / 2;
      ConvArgs a{};
      a.x = act; a.bias = tpp(ti + 2); a.res = nullptr;
      a.Cin = cin; a.Cout = cout; a.Tin = Tlen; a.Tout = Tlen * sd; a.q_count = Tlen + 1;
      a.n_taps = 2; a.off_base = 0; a.off_step = -1; a.wt_base = 0; a.wt_step = sd;
      a.n_phase = sd; a.wt_phase_step = 1; a.o_mul = sd; a.o_add = -pad; a.o_phase_step = 1;
      // raw -> X (residual stream of the block), snake_{res1.snake1}(x) -> the other activation buffer
      if (int e = launch_conv_tc(a, tpk(ti + 1), 2 * sd, tpp(ti + 3), bufX, oth2, B, st)) return e;
      ti += 3;
      std::swap(act, oth2);
      Tlen *= sd;
      const int dil[3] = {1, 3, 9};
      for (int r = 0; r < 3; r++) {
        // y = conv7(snake1(x)) -> only snake2(y) is stored; x += conv1(snake2(y)), plus snake_next(x) for the next unit
        if (int e = convk(act, ti + 1, ti + 2, nullptr, nullptr, oth2, tpp(ti + 3), cout, cout, Tlen, 7, dil[r])) return e;
        const int next_alpha = ti + 6;  // next unit's snake1, next block's snake1, or the decoder's final snake1
        if (int e = convk(oth2, ti + 4, ti + 5, bufX, bufX, act, tpp(next_alpha), cout, cout, Tlen, 1, 1)) return e;
        ti += 6;
      }
    }
    const int cl = C >> cfg->n_blocks;
    if (final_conv_supported(cl))   // one thread per output sample (dac.cu)
      return launch_final_conv_tanh(act, tpp(ti + 1), tpp(ti + 2), audio_out, cl, Tlen, B, st);
    ConvArgs f{};  // final conv (Cout = 1) + tanh on the already snake'd tensor: generic kernel
    f.x = act; f.w = tpp(ti + 1); f.bias = tpp(ti + 2); f.alpha = nullptr; f.res = nullptr; f.out = audio_out;
    f.Cin = cl; f.Cout = 1; f.Tin = Tlen; f.Tout = Tlen; f.q_count = Tlen;
    f.n_taps = 7; f.off_base = -3; f.off_step = 1; f.wt_base = 0; f.wt_step = 1;
    f.n_phase = 1; f.wt_phase_step = 0; f.o_mul = 1; f.o_add = 0; f.o_phase_step = 0; f.tanh_out = 1;
    return launch_conv(f, cfg->dtype, B, st);
  }
  FromCodesArgs fc{codes, bl + L.codebooks, bl + L.proj_w, bl + L.proj_b, cur, K, cfg->codebook_dim, cfg->latent_dim, T, cfg->codebook_size};
  if (int e = launch_from_codes(fc, cfg->dtype, B, st)) return e;
  int ti = 3 * K;  // tensor cursor (see make_dac_layout order)
  auto tp = [&](int i) { return bl + L.t[i].off; };
  auto conv = [&](const void* x, int w_i, int b_i, const void* alpha, const void* res, void* out, int Cin, int Cout, int Tlen, int ks, int dil, int tanh_out) {
    ConvArgs a{};
    a.x = x; a.w = tp(w_i); a.bias = tp(b_i); a.alpha = alpha; a.res = res; a.out = out;
    a.Cin = Cin; a.Cout = Cout; a.Tin = Tlen; a.Tout = Tlen; a.q_count = Tlen;
    a.n_taps = ks; a.off_base = -((ks - 1) / 2) * dil; a.off_step = dil; a.wt_base = 0; a.wt_step = 1;
    a.n_phase = 1; a.wt_phase_step = 0; a.o_mul = 1; a.o_add = 0; a.o_phase_step = 0; a.tanh_out = tanh_out;
    return launch_conv(a, cfg->dtype, B, st);
  };
  const int C = cfg->decoder_dim;
  if (int e = conv(cur, ti, ti + 1, nullptr, nullptr, oth, cfg->latent_dim, C, T, 7, 1, 0)) return e;
  ti += 2;
  std::swap(cur, oth);
  int Tlen = T;
  for (int bi = 0; bi < cfg->n_blocks; bi++) {
    const int cin = C >> bi, cout = C >> (bi + 1), sd = cfg->strides[bi];
    const int pad = (sd + 1) / 2;
    ConvArgs a{};
    a.x = cur; a.alpha = tp(ti); a.w = tp(ti + 1); a.bias = tp(ti + 2); a.res = nullptr; a.out = oth;
    a.Cin = cin; a.Cout = cout; a.Tin = Tlen; a.Tout = Tlen * sd; a.q_count = Tlen + 1;
    a.n_taps = 2; a.off_base = 0; a.off_step = -1; a.wt_base = 0; a.wt_step = sd;
    a.n_phase = sd; a.wt_phase_step = 1; a.o_mul = sd; a.o_add = -pad; a.o_phase_step = 1; a.tanh_out = 0;
    if (int e = launch_conv(a, cfg->dtype, B, st)) return e;
    ti += 3;
    std::swap(cur, oth);
    Tlen *= sd;
    const int dil[3] = {1, 3, 9};
    for (int r = 0; r < 3; r++) {
      // y = conv7(snake1(x)) -> oth ; x = x + conv1(snake2(y)) in place
      if (int e = conv(cur, ti + 1, ti + 2, tp(ti), nullptr, oth, cout, cout, Tlen, 7, dil[r], 0)) return e;
      if (int e = conv(oth, ti + 4, ti + 5, tp(ti + 3), cur, cur, cout, cout, Tlen, 1, 1, 0)) return e;
      ti += 6;
    }
  }
  const int cl = C >> cfg->n_blocks;
  return conv(cur, ti + 1, ti + 2, tp(ti), nullptr, audio_out, cl, 1, Tlen, 7, 1, 1);
}

// ---- DAC encode --------------------------------------------------------------------------------
int ptts_dac_encoder_blob_bytes(const ptts_dac_encoder_config* cfg, int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes, "null argument");
  if (int e = validate_dac_encoder(*cfg)) return e;
  *out_bytes = make_dac_encoder_layout(*cfg).total;
  return PTTS_OK;
}
int ptts_dac_encoder_num_tensors(const ptts_dac_encoder_config* cfg, int32_t* out) {
  PTTS_REQUIRE(cfg && out, "null argument");
  if (int e = validate_dac_encoder(*cfg)) return e;
  *out = (int32_t)make_dac_encoder_layout(*cfg).t.size();
  return PTTS_OK;
}
int ptts_dac_encoder_pack(const ptts_dac_encoder_config* cfg, void* blob, int32_t name_id, const void* src, int32_t src_dtype, int64_t numel,
                          void* stream) {
  PTTS_REQUIRE(cfg && blob && src, "null argument");
  if (int e = validate_dac_encoder(*cfg)) return e;
  PTTS_REQUIRE(src_dtype == PTTS_BF16 || src_dtype == PTTS_F32, "dac encoder pack: src dtype must be bf16 or f32");
  const DacEncLayout L = make_dac_encoder_layout(*cfg);
  PTTS_REQUIRE(name_id >= 0 && name_id < (int)L.t.size(), "dac encoder pack: tensor id %d out of range", name_id);
  const DacTensor& t = L.t[name_id];
  PTTS_REQUIRE(numel == t.numel, "dac encoder pack: tensor %d expects %lld elements, got %lld", name_id, (long long)t.numel, (long long)numel);
  cudaStream_t st = (cudaStream_t)stream;
  char* dst = (char*)blob + t.off;
  if (t.kind == DK_PLAIN) {
    if (int e = pack_plain(src, src_dtype, numel, dst, cfg->dtype, st)) return e;
    const bool is_codebook = name_id >= L.first_q && (name_id - L.first_q) % 5 == 2;
    if (!is_codebook) return PTTS_OK;
    const int64_t k = (name_id - L.first_q) / 5, cb_bytes = (int64_t)cfg->codebook_size * cfg->codebook_dim * L.es;
    return normalize_codebook(dst, (char*)blob + L.cb_norm + k * cb_bytes, cfg->codebook_size, cfg->codebook_dim, cfg->dtype, st);
  }
  if (t.off_k >= 0) {
    if (int e = pack_conv_kmajor(src, src_dtype, (char*)blob + t.off_k, t.d0, t.d1, t.k, 0, st)) return e;
  }
  return pack_conv(src, src_dtype, dst, cfg->dtype, t.d0, t.d1, t.k, 0, st);
}
int ptts_dac_encoder_workspace_bytes(const ptts_dac_encoder_config* cfg, int32_t B, int64_t n_samples, int64_t* out_bytes) {
  PTTS_REQUIRE(cfg && out_bytes && B > 0 && n_samples > 0, "bad argument");
  if (int e = validate_dac_encoder(*cfg)) return e;
  PTTS_REQUIRE(n_samples % dac_encoder_hop(*cfg) == 0, "dac encoder: n_samples %lld is not a multiple of the hop %lld", (long long)n_samples,
               (long long)dac_encoder_hop(*cfg));
  *out_bytes = dac_encoder_workspace(*cfg, B, n_samples);
  return PTTS_OK;
}
int ptts_dac_encode(const ptts_dac_encoder_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes, const void* audio, int32_t B,
                    int64_t n_samples, int32_t n_q, int64_t* codes_out, void* z_out, void* stream) {
  PTTS_REQUIRE(cfg && blob && workspace && audio && codes_out, "null argument");
  if (int e = validate_dac_encoder(*cfg)) return e;
  return dac_encode(*cfg, (const char*)blob, (char*)workspace, workspace_bytes, audio, B, n_samples, n_q, codes_out, z_out, (cudaStream_t)stream);
}

}  // extern "C"
