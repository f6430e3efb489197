// kernels.h -- host-side launch interface of the kernel translation units.
#pragma once
#include "common.cuh"

namespace ptts {

enum { EPI_STORE = 0, EPI_ACT = 1, EPI_RESIDUAL = 2, EPI_F32 = 3 };

struct LinearArgs {
  const void* X; int64_t ldx;  // activations [M, K], row stride ldx (elements)
  const void* W;               // packed weight slot (fragment order for bf16, row-major for f32)
  void* Y; int64_t ldy;
  const void* R; int64_t ldr;  // residual (EPI_RESIDUAL)
  const float* ln_w; const float* ln_b; float eps;  // fused LayerNorm on x (needs Kc == K); f32 path uses gamma/beta directly
  const float* c1; const float* c2;                 // bf16 path: folded LayerNorm vectors (ln_stats.cuh); LN on iff c1 != nullptr
  int M, N, K, Kc;             // Kc = activation tile width (0 = choose)
  int epi, act;
  const Ctrl* ctrl;            // device control block: kernels no-op once generation has finished
};
int launch_linear(const LinearArgs& a, int dtype, cudaStream_t st, bool pdl, int sm_count);
// EXPERIMENTAL tcgen05 prefill GEMM (gemm_tc.cu; only reached with PTTS_PREFILL_TC=1)
bool linear_tc_supported(const LinearArgs& a);
int launch_linear_tc(const LinearArgs& a, const void* w_rowmajor, float* stats_scratch, cudaStream_t st);
int unpack_fragments(const void* frag, void* dst_rowmajor, int64_t N, int K, cudaStream_t st);
int pack_matrix(const void* src, int src_dtype, int64_t rows, int64_t cols, int row_off, int K, void* dst, int dst_dtype, cudaStream_t st);
int fold_layernorm(void* w_packed, int N, int K, const float* gamma, const float* beta, float* c1, float* c2, cudaStream_t st);
int pack_plain(const void* src, int src_dtype, int64_t n, void* dst, int dst_dtype, cudaStream_t st);

// ---- attention (attention.cu) -------------------------------------------------------------------
struct AttnArgs {
  // query / new-token projections: row r = b*q_len + j of a [B*q_len, ld] matrix
  const void* q; int64_t ldq; int q_col0;       // q head h at columns q_col0 + h*64
  const void* knew; const void* vnew; int64_t ldkv; int k_col0, v_col0;  // self: new K/V rows (same matrix as q)
  void* kcache; void* vcache;                   // self: [B][nkv][Tmax][64]; cross: strided view
  int64_t kv_b_stride, kv_h_stride, kv_t_stride; // element strides of (batch, kv head, token)
  void* out; int64_t ldo;                       // [B*q_len, H]
  const int* key_mask; int mask_len, mask_ld;   // keys t < mask_len with key_mask[b*mask_ld+t]==0 are excluded
  const Ctrl* ctrl;
  int B, nh, nkv, q_len;
  int past_from_ctrl;   // 1: past = prefix + ctrl->cur_len - 1 (decode); 0: past = past_len (prefill)
  int past_len, prefix; // cache position of the first new row
  int cross;            // 1: keys = kv_len encoder positions, no append, no causal structure
  int kv_len;
  int rope; const void* rope_cos; const void* rope_sin;  // [max_pos][64] tables in the model dtype (Q3)
  int kv_capacity;      // upper bound on keys per query (sizes the score buffer)
  float scale;
};
int launch_attention(const AttnArgs& a, int dtype, cudaStream_t st, bool pdl);

// ---- embedding (embed.cu) -----------------------------------------------------------------------
struct EmbedArgs {
  const void* tables;  // [K][V+1][H]
  const void* pos;     // [max_pos][H] or nullptr (rope)
  const void* prefix;  // [B][P][H] prompt hidden states or nullptr
  const int* ids;      // [B*K] current (delay-masked) input ids
  void* x;             // [B*(P+1) or B][H]
  const Ctrl* ctrl;
  int B, K, V1, H, P;  // P = prefix rows per batch in THIS call (0 at decode)
  int pos_from_ctrl, pos0, prefix_len;  // decode: position = prefix_len + cur_len - 1
  int n_cols;              // decoder columns per batch row in THIS call (1 at decode; n for a voice-prompt prefill)
  const int64_t* col_ids;  // [B*K][n_cols] ids of those columns, or nullptr: one column from `ids`
};
int launch_embed(const EmbedArgs& a, int dtype, cudaStream_t st, bool pdl);

// ---- sampling / generation state (sample.cu) ----------------------------------------------------
struct SampleArgs {
  const float* logits; float* scores;  // [BK][V]
  int64_t* raw_ids; int64_t raw_ld;
  int* cur_ids; int* eos_seen; int* unfinished; int* first_unf;  // first_unf [2][B]
  Ctrl* ctrl;
  const ptts_gen_params* gen;  // device copy
  int B, K, V;
  int bos, pad, eos;
};
int launch_sample(const SampleArgs& a, const int64_t* forced, cudaStream_t st, bool pdl);
int launch_generate_begin(const SampleArgs& a, cudaStream_t st);
int launch_delay_build(const int64_t* ids, int BK, int seq, int K, int64_t bos, int64_t pad, int L, int64_t* mask, cudaStream_t st);
int launch_delay_apply(const int64_t* ids, int BK, int seq, int64_t ld_ids, const int64_t* mask, int64_t ld_mask, int64_t* out, cudaStream_t st);
int launch_logits_processor(const int64_t* ids, int BK, int seq, int64_t ld_ids, float* scores, int V, int64_t eos, int K, int64_t* first_unf, cudaStream_t st);
int launch_mask_convert(const int64_t* src, int n, int* dst, cudaStream_t st);  // int64 0/1 -> int32; src==nullptr -> ones
int launch_cross_kv_relayout(const void* src, void* dst, int B, int S, int nckv, int dtype, cudaStream_t st);
int launch_gather_rows(const void* src, int64_t ld_src, int64_t row0, int64_t row_step, void* dst, int rows, int cols, int dtype, cudaStream_t st);

}  // namespace ptts
