/*
 * ptts_b200.h -- C ABI of the B200-native Parler-TTS generation path.
 *
 * Drop-in boundary: the reference (huggingface/parler-tts) has NO native layer; its hot path is
 * Python calling stock PyTorch ops.  Each entry point below names the reference interface it
 * replaces (file:line under the reference repo).  The Python shim in parler_tts_b200/ mirrors the
 * reference's public classes and calls these functions through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every function returns 0 on success, non-zero on error; ptts_last_error() gives the message
 *     (thread-local).  The Python shim raises ValueError (PTTS_EINVAL) or RuntimeError (others),
 *     matching the reference's ValueError-on-contract-violation behaviour
 *     (e.g. dac_wrapper/modeling_dac.py:135-136, modeling_parler_tts.py:3471-3475).
 *   - the library never allocates caller-visible device memory: weights blob and workspace are
 *     caller-allocated (torch tensors), sized by the *_bytes() queries.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *     `device` pointers are raw CUDA device pointers on the current device of the calling thread.
 *   - dtype codes: 0 = bf16, 1 = f32, 2 = int64, 3 = int32.
 */
#ifndef PTTS_B200_H
#define PTTS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTTS_OK 0
#define PTTS_EINVAL 1   /* contract violation -> ValueError */
#define PTTS_ECUDA 2    /* CUDA runtime error -> RuntimeError */
#define PTTS_ESTATE 3   /* wrong call order   -> RuntimeError */

#define PTTS_BF16 0
#define PTTS_F32 1
#define PTTS_I64 2
#define PTTS_I32 3

#define PTTS_HEAD_DIM 64

/* ParlerTTSDecoderConfig fields the path needs (configuration_parler_tts.py:107-172). */
typedef struct ptts_decoder_config {
  int32_t hidden_size;
  int32_t num_layers;
  int32_t num_heads;
  int32_t num_kv_heads;        /* self-attention KV heads (GQA, :948) */
  int32_t num_cross_kv_heads;  /* cross-attention KV heads (:970) */
  int32_t ffn_dim;
  int32_t vocab_size;          /* lm-head rows; embedding tables have vocab_size+1 rows (:1353) */
  int32_t num_codebooks;
  int32_t max_positions;
  int32_t rope;                /* rope_embeddings (:130); 0 -> sinusoidal table added to embeds */
  int32_t activation;          /* 0 gelu(erf), 1 relu, 2 silu, 3 gelu(tanh) */
  int32_t dtype;               /* PTTS_BF16 or PTTS_F32: model dtype (weights, activations, KV) */
  int32_t bos_token_id, pad_token_id, eos_token_id;
  float rope_theta;
  float layer_norm_eps;
} ptts_decoder_config;

/* Generation knobs (HF GenerationConfig subset used by generate(), modeling_parler_tts.py:3395-3552). */
typedef struct ptts_gen_params {
  int32_t max_length;      /* total decoder length incl. BOS column */
  int32_t min_new_tokens;
  int32_t do_sample;       /* 0 = greedy argmax */
  int32_t top_k;           /* 0 = off */
  float top_p;             /* >= 1 = off */
  float temperature;       /* 1 = off */
  uint64_t seed;           /* Philox key; substream = (row_base + row, step) */
  int32_t suppress_special; /* bench aid: mask ids >= codebook_size (never set by generate()) */
  int32_t codebook_size;
  int32_t row_base;        /* global index of this session's first row (= first utterance * num_codebooks): with a batch
                            * sharded over GPUs every shard passes its own offset, so the draws of an utterance do not
                            * depend on the number of shards (SURVEY 8e) */
  int32_t reserved_;
} ptts_gen_params;

/* Tensor ids for ptts_decoder_pack(). `index` = layer (per-layer tensors) or codebook (EMBED/LM_HEAD). */
enum {
  PTTS_T_EMBED_TOKENS = 0, /* [vocab+1, H]  decoder.model.decoder.embed_tokens.N.weight (:1354) */
  PTTS_T_POS_TABLE = 1,    /* [max_pos, H]  embed_positions.weights (:1360), absent when rope */
  PTTS_T_LN1_W = 2, PTTS_T_LN1_B = 3,      /* self_attn_layer_norm (:961) */
  PTTS_T_SELF_Q = 4, PTTS_T_SELF_K = 5, PTTS_T_SELF_V = 6, PTTS_T_SELF_O = 7,    /* :481-484 */
  PTTS_T_LN2_W = 8, PTTS_T_LN2_B = 9,      /* encoder_attn_layer_norm (:978) */
  PTTS_T_CROSS_Q = 10, PTTS_T_CROSS_K = 11, PTTS_T_CROSS_V = 12, PTTS_T_CROSS_O = 13,
  PTTS_T_LN3_W = 14, PTTS_T_LN3_B = 15,    /* final_layer_norm (:981) */
  PTTS_T_FC1 = 16, PTTS_T_FC2 = 17,        /* :979-980 */
  PTTS_T_FINAL_LN_W = 18, PTTS_T_FINAL_LN_B = 19, /* decoder.layer_norm (:1373) */
  PTTS_T_LM_HEAD = 20,     /* [vocab, H] decoder.lm_heads.N.weight (:1838) */
  PTTS_T_ROPE_COS = 21,    /* [max_pos, 64] cos table, fp32 -> model dtype as the reference does (:394-406, :1534) */
  PTTS_T_ROPE_SIN = 22,    /* [max_pos, 64] sin table (only when rope != 0) */
  PTTS_T_COUNT = 23
};

const char* ptts_last_error(void);
int ptts_version(void);

/* ---- decoder: weights --------------------------------------------------------------------- */
/* Size of the packed weight blob (device bytes) for this config. */
int ptts_decoder_blob_bytes(const ptts_decoder_config* cfg, int64_t* out_bytes);
/* Repack one reference-layout tensor (row-major [rows, cols], dtype src_dtype, device memory) into
 * the blob: GEMM matrices go to MMA-fragment order (bf16) / row-major (f32); q,k,v are fused into one
 * matrix; LayerNorm parameters are kept in f32.  Replaces nothing in the reference (load-time only). */
int ptts_decoder_pack(const ptts_decoder_config* cfg, void* blob, int32_t tensor_id, int32_t index,
                      const void* src, int32_t src_dtype, int64_t rows, int64_t cols, void* stream);

/* Call once after every tensor has been packed (bf16 model dtype): folds each LayerNorm's affine part into the
 * linear layer that follows it (W' = gamma*W, c1 = rowsum(W'), c2 = W*beta), so that the run-time GEMM consumes the
 * raw residual stream and only needs per-row (mean, rstd).  No-op for f32. */
int ptts_decoder_finalize(const ptts_decoder_config* cfg, void* blob, void* stream);

/* ---- decoder: generation session ----------------------------------------------------------- */
/* Workspace bytes for a batch of B utterances, prompt prefix length P, encoder length S and a
 * self-attention cache of max_cache_len positions (>= P + max_length - 1). */
int ptts_workspace_bytes(const ptts_decoder_config* cfg, int32_t B, int32_t P, int32_t S,
                         int32_t max_cache_len, int64_t* out_bytes);
/* Same, for a session whose first forward may take up to max_prefix (>= 1) decoder columns (ptts_prefill_ids: a
 * voice-prompt prefix, modeling_parler_tts.py:3136-3194).  ptts_workspace_bytes is the max_prefix = 1 case. */
int ptts_workspace_bytes_ex(const ptts_decoder_config* cfg, int32_t B, int32_t P, int32_t S,
                            int32_t max_cache_len, int32_t max_prefix, int64_t* out_bytes);

typedef struct ptts_session ptts_session; /* host-side object: pointers into blob/workspace + CUDA graphs */

int ptts_session_create(const ptts_decoder_config* cfg, const void* blob, void* workspace,
                        int64_t workspace_bytes, int32_t B, int32_t P, int32_t S, int32_t max_cache_len,
                        ptts_session** out);
int ptts_session_create_ex(const ptts_decoder_config* cfg, const void* blob, void* workspace,
                           int64_t workspace_bytes, int32_t B, int32_t P, int32_t S, int32_t max_cache_len,
                           int32_t max_prefix, ptts_session** out);
int ptts_session_destroy(ptts_session* s);

/* Start a generate() call: reset per-call state (ids history = BOS column, processor state,
 * unfinished flags, delay-pattern parameters).  Replaces generate() steps 5-9
 * (modeling_parler_tts.py:3449-3552), build_delay_pattern_mask (:3523) and the
 * ParlerTTSLogitsProcessor constructor (logits_processors.py:23-42). */
int ptts_generate_begin(ptts_session* s, const ptts_gen_params* gen, void* stream);

/* Step 0 (prefill): prompt prefix + BOS through the decoder, cross-attention K/V projected once,
 * self-attention cache filled at positions [0, P].  Leaves f32 logits [B*K, V] in the workspace.
 * Replaces ParlerTTSForCausalLM.forward at step 0 (:1865-1974, :1392-1655, :872-889).
 *   prompt_hidden [B, P, H] model dtype (may be NULL when P == 0)   (:3099-3134 output)
 *   prompt_mask   [B, P] int64 or NULL                              (prompt_attention_mask)
 *   enc_hidden    [B, S, H] model dtype, already multiplied by the mask (:3092-3093)
 *   enc_mask      [B, S] int64 or NULL                              (attention_mask)            */
int ptts_prefill(ptts_session* s, const void* prompt_hidden, const int64_t* prompt_mask,
                 const void* enc_hidden, const int64_t* enc_mask, void* stream);
/* Prefill over n decoder columns (voice-prompt continuation, :3017-3044, :3523-3528): prompt prefix + prefix_ids
 * [B*K, n] int64 (already delay-patterned, column 0 = BOS) in one forward of q_len = P + n; writes raw_ids[:, :n], sets the
 * device cur_len = n and leaves the logits of the last position.  1 <= n <= the session's max_prefix, n < max_length.
 * ptts_prefill is the n = 1 case with the BOS column ptts_generate_begin staged. */
int ptts_prefill_ids(ptts_session* s, const void* prompt_hidden, const int64_t* prompt_mask,
                     const void* enc_hidden, const int64_t* enc_mask, const int64_t* prefix_ids, int32_t n,
                     void* stream);

/* One cached decode step for the ids currently staged in the workspace (the delay-masked last
 * column).  Leaves f32 logits [B*K, V] in the workspace.  Replaces prepare_inputs_for_generation
 * (:2882-2986) + ParlerTTSForCausalLM.forward with q_len == 1. */
int ptts_decode_forward(ptts_session* s, void* stream);

/* logits -> next token for every row, on device: MinNewTokens, ParlerTTSLogitsProcessor
 * (logits_processors.py:44-53), temperature/top-k/top-p, softmax + sampling or argmax, finished-row
 * padding, history append, EOS/max-length stopping, delay-mask override of the next input.
 * Replaces one iteration of GenerationMixin._sample (transformers 4.46.1) + :2909.
 * forced_tokens: NULL, or [B*K] int64 device tokens that replace the drawn ones (teacher forcing); a negative entry
 * means "draw this row" (the prompt codes the delay pattern puts after a voice-prompt prefix are forced per row). */
int ptts_sample(ptts_session* s, const int64_t* forced_tokens, void* stream);

/* n_steps x (ptts_decode_forward + ptts_sample), replayed from a CUDA graph, no host sync.
 * Steps after every row finished are device-side no-ops. */
int ptts_decode_steps(ptts_session* s, int32_t n_steps, void* stream);

/* Device pointers into the workspace (valid for the session lifetime). */
int ptts_session_logits(ptts_session* s, float** out);          /* [B*K, V] f32, last step's raw logits */
int ptts_session_scores(ptts_session* s, float** out);          /* [B*K, V] f32, processed scores      */
int ptts_session_raw_ids(ptts_session* s, int64_t** out, int32_t* ld); /* [B*K, ld] raw (un-masked) history */
int ptts_session_state(ptts_session* s, int32_t** out);         /* int32[8]: {cur_len, n_unfinished, ...} */
int ptts_session_launches(ptts_session* s, int64_t* out);       /* kernels launched through this session  */
/* After ptts_prefill: 0 = decode steps run the multi-kernel path (shape outside the fused kernel's range; a warning is printed
 * once), 1 = the fused persistent step kernel (one launch per token, step.cu), 2 = its cluster variant (step2.cu). */
int ptts_session_fused(ptts_session* s, int32_t* out);
/* Profiling aid: per-phase clock64() stamps of the fused step kernel into buf (device int64 [(8L+3)*8]); NULL = off. */
int ptts_session_set_profile(ptts_session* s, void* buf);

/* ---- stand-alone operators (same kernels, used by the Python mirrors and the tests) -------- */
/* build_delay_pattern_mask (:214-276): input_ids [B*K, seq] int64 -> pattern_mask [B*K, max_length]
 * int64 (the truncated input_ids the reference also returns is a slice the shim takes). */
int ptts_delay_build(const int64_t* input_ids, int32_t BK, int32_t seq_len, int32_t num_codebooks,
                     int64_t bos, int64_t pad, int32_t max_length, int64_t* pattern_mask, void* stream);
/* apply_delay_pattern_mask (:205-211): out = where(mask[:, :seq]==-1, ids, mask). */
int ptts_delay_apply(const int64_t* input_ids, int32_t BK, int32_t seq_len, int64_t ld_ids,
                     const int64_t* pattern_mask, int64_t ld_mask, int64_t* out, void* stream);
/* ParlerTTSLogitsProcessor.__call__ (logits_processors.py:44-53): scores [B*K, V] f32 in place;
 * first_unfinished [B] int64 is the processor's persistent state. */
int ptts_logits_processor(const int64_t* input_ids, int32_t BK, int32_t seq_len, int64_t ld_ids,
                          float* scores, int32_t V, int64_t eos, int32_t num_codebooks,
                          int64_t* first_unfinished, void* stream);
/* y[M,N] = epi(LN?(x[M,K]) @ W^T): W taken from a packed blob slot. Test hook for the GEMM kernels. */
int ptts_op_linear(const ptts_decoder_config* cfg, const void* blob, int32_t tensor_id, int32_t index,
                   const void* x, int32_t M, int32_t use_ln, int32_t epilogue /*0 store,1 act,2 +res,3 f32*/,
                   const void* residual, void* y, void* stream);

/* ---- DAC decode ------------------------------------------------------------------------------ */
typedef struct ptts_dac_config {
  int32_t n_codebooks, codebook_size, codebook_dim;
  int32_t latent_dim;          /* DACConfig.latent_dim = 1024 (configuration_dac.py:14) */
  int32_t decoder_dim;         /* 1536 */
  int32_t n_blocks;            /* 4 */
  int32_t strides[8];          /* 8,8,4,2 */
  int32_t dtype;               /* storage dtype of activations/weights: PTTS_BF16 or PTTS_F32 */
} ptts_dac_config;

int ptts_dac_blob_bytes(const ptts_dac_config* cfg, int64_t* out_bytes);
int ptts_dac_num_tensors(const ptts_dac_config* cfg, int32_t* out);
/* Pack one weight-norm-folded tensor.  `name_id` enumerates tensors in network order; see
 * parler_tts_b200/dac_wrapper.py::_dac_tensor_list for the (id -> state-dict key) table. */
int ptts_dac_pack(const ptts_dac_config* cfg, void* blob, int32_t name_id, const void* src,
                  int32_t src_dtype, int64_t numel, void* stream);
int ptts_dac_workspace_bytes(const ptts_dac_config* cfg, int32_t B, int32_t T, int64_t* out_bytes);
/* DACModel.decode (dac_wrapper/modeling_dac.py:106-142): codes [B, K, T] int64 ->
 * audio [B, 1, hop*T] in cfg->dtype.  = quantizer.from_codes (:138) + model.decode (:139). */
int ptts_dac_decode(const ptts_dac_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes,
                    const int64_t* codes, int32_t B, int32_t T, void* audio_out, void* stream);

/* ---- DAC encode (voice prompt) ------------------------------------------------------------- */
/* Separate from ptts_dac_config so that the decode ABI and the decode blob keep their layout.  Shapes per
 * transformers' DacEncoder / DacResidualVectorQuantizer (models/dac/modeling_dac.py:442-473, :281-343). */
typedef struct ptts_dac_encoder_config {
  int32_t encoder_dim;         /* 64: conv1 width; block i runs at encoder_dim << i channels, outputs encoder_dim << (i+1) */
  int32_t n_blocks;            /* 4 */
  int32_t strides[8];          /* 2,4,8,8 (even) */
  int32_t latent_dim;          /* 1024 */
  int32_t n_codebooks, codebook_size, codebook_dim;
  int32_t dtype;               /* PTTS_BF16 or PTTS_F32 */
} ptts_dac_encoder_config;

int ptts_dac_encoder_blob_bytes(const ptts_dac_encoder_config* cfg, int64_t* out_bytes);
int ptts_dac_encoder_num_tensors(const ptts_dac_encoder_config* cfg, int32_t* out);
/* Pack one weight-norm-folded tensor; see parler_tts_b200/dac_wrapper.py::_dac_encoder_tensor_list for the
 * (id -> state-dict key) table.  Packing a codebook also stores its L2-normalised copy for the code search. */
int ptts_dac_encoder_pack(const ptts_dac_encoder_config* cfg, void* blob, int32_t name_id, const void* src,
                          int32_t src_dtype, int64_t numel, void* stream);
int ptts_dac_encoder_workspace_bytes(const ptts_dac_encoder_config* cfg, int32_t B, int64_t n_samples, int64_t* out_bytes);
/* DACModel.encode (dac_wrapper/modeling_dac.py:33-104) = DAC.encode: encoder network + residual vector quantizer.
 *   audio     [B][n_samples] cfg->dtype, already right-padded to a multiple of the hop (prod(strides))
 *   codes_out [B][n_q][n_samples / hop] int64 (n_q in 1..n_codebooks)
 *   z_out     [B][n_samples / hop][latent_dim] cfg->dtype, the quantized latent (sum of the n_q codebooks'
 *             out_proj outputs); NULL = not written */
int ptts_dac_encode(const ptts_dac_encoder_config* cfg, const void* blob, void* workspace, int64_t workspace_bytes,
                    const void* audio, int32_t B, int64_t n_samples, int32_t n_q, int64_t* codes_out, void* z_out,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PTTS_B200_H */
