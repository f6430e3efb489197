// embed.cu -- decoder input embeddings: sum of K codebook embeddings (+ prompt prefix) + positions.
//
// Replaces ParlerTTSDecoder.forward's input stage (modeling_parler_tts.py:1433 embedding sum with
// Python-sum rounding order, :1437-1439 prompt prefix concat at step 0, :1506-1511 sinusoidal add)
// and the step-0 inputs_embeds of _prepare_decoder_input_ids_for_generation (:3033-3044).
// Bytes: B*K gathered rows of H elements -- negligible next to the weight stream.
#include "common.cuh"
#include "kernels.h"

namespace ptts {

template <typename T>
__global__ void __launch_bounds__(128) embed_kernel(EmbedArgs p) {
  pdl_launch_dependents();
  pdl_wait();
  if (p.ctrl != nullptr && p.ctrl->active == 0) return;
  const int rows_per_b = p.P + p.n_cols;
  const int b = blockIdx.x / rows_per_b, j = blockIdx.x - b * rows_per_b;
  const int position = p.pos_from_ctrl ? (p.prefix_len + p.ctrl->cur_len - 1) : (p.pos0 + j);
  const T* tables = reinterpret_cast<const T*>(p.tables);
  const T* pos = reinterpret_cast<const T*>(p.pos);
  T* x = reinterpret_cast<T*>(p.x) + (size_t)blockIdx.x * p.H;
  for (int c = threadIdx.x; c < p.H; c += blockDim.x) {
    float v;
    if (j < p.P) {
      v = DT<T>::to_f(reinterpret_cast<const T*>(p.prefix)[((size_t)b * p.P + j) * p.H + c]);
    } else {
      v = 0.f;
      for (int k = 0; k < p.K; k++) {
        const int id = p.col_ids != nullptr ? (int)p.col_ids[(size_t)(b * p.K + k) * p.n_cols + (j - p.P)] : p.ids[b * p.K + k];
        const float e = DT<T>::to_f(tables[((size_t)k * p.V1 + id) * p.H + c]);
        v = (k == 0) ? e : DT<T>::rnd(v + e);  // sum([...]) accumulates left to right in the model dtype
      }
    }
    if (pos != nullptr) v = DT<T>::rnd(v + DT<T>::to_f(pos[(size_t)position * p.H + c]));
    x[c] = DT<T>::from_f(v);
  }
}

int launch_embed(const EmbedArgs& a, int dtype, cudaStream_t st, bool pdl) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(a.B * (a.P + a.n_cols));
  cfg.blockDim = dim3(128);
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  if (dtype == PTTS_BF16) PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, embed_kernel<bf16>, a));
  else PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, embed_kernel<float>, a));
  return PTTS_OK;
}

// ---- small plumbing kernels ---------------------------------------------------------------------
__global__ void mask_convert_kernel(const int64_t* src, int n, int* dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src ? (src[i] != 0 ? 1 : 0) : 1;
}
int launch_mask_convert(const int64_t* src, int n, int* dst, cudaStream_t st) {
  if (n <= 0) return PTTS_OK;
  mask_convert_kernel<<<(n + 255) / 256, 256, 0, st>>>(src, n, dst);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

template <typename T>
__global__ void gather_rows_kernel(const T* src, int64_t ld_src, int64_t row0, int64_t row_step, T* dst, int rows, int cols) {
  int r = blockIdx.x;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) dst[(size_t)r * cols + c] = src[(size_t)(row0 + r * row_step) * ld_src + c];
}
int launch_gather_rows(const void* src, int64_t ld_src, int64_t row0, int64_t row_step, void* dst, int rows, int cols, int dtype, cudaStream_t st) {
  if (dtype == PTTS_BF16) gather_rows_kernel<bf16><<<rows, 128, 0, st>>>((const bf16*)src, ld_src, row0, row_step, (bf16*)dst, rows, cols);
  else gather_rows_kernel<float><<<rows, 128, 0, st>>>((const float*)src, ld_src, row0, row_step, (float*)dst, rows, cols);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// cross-attention K/V: GEMM output rows [B*S][K(nckv*64) | V(nckv*64)] -> item-major K [B][nckv][S][64] then
// V [B][nckv][S][64], so a (batch row, kv head) item is ONE contiguous run the TMA engine fetches with a
// single bulk copy per stage (done once per generate() at prefill; reference keeps [B, heads, S, 64] too, :877-878).
template <typename T>
__global__ void cross_kv_relayout_kernel(const T* __restrict__ src, T* __restrict__ dst, int B, int S, int nckv) {
  const int row = blockIdx.x;  // b*S + s
  const int b = row / S, sidx = row - b * S;
  const int width = 2 * nckv * 64;
  for (int c = threadIdx.x; c < width; c += blockDim.x) {
    const int is_v = c >= nckv * 64;
    const int cc = c - is_v * nckv * 64;
    const int h = cc >> 6, d = cc & 63;
    dst[(size_t)is_v * B * nckv * S * 64 + (((size_t)b * nckv + h) * S + sidx) * 64 + kv_swz(sidx, d)] = src[(size_t)row * width + c];  // swizzled rows (common.cuh)
  }
}
int launch_cross_kv_relayout(const void* src, void* dst, int B, int S, int nckv, int dtype, cudaStream_t st) {
  if (dtype == PTTS_BF16) cross_kv_relayout_kernel<bf16><<<B * S, 128, 0, st>>>((const bf16*)src, (bf16*)dst, B, S, nckv);
  else cross_kv_relayout_kernel<float><<<B * S, 128, 0, st>>>((const float*)src, (float*)dst, B, S, nckv);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

}  // namespace ptts
