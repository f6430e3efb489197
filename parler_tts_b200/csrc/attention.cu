// attention.cu -- self- and cross-attention over the KV cache for q_len new positions.
//
// Replaces ParlerTTSSdpaAttention.forward after the projections (modeling_parler_tts.py:858-914):
// rotary embedding of q/k (:858-859, :880-882, quirks Q2/Q3/Q7), KV-cache append (:887-889, a
// pre-allocated [B][nkv][Tmax][64] cache instead of DynamicCache's torch.cat), repeat_kv (:896-897,
// done by indexing), the 4-D additive masks (:1546-1562, :1658-1736 -> here a per-key exclude flag)
// and F.scaled_dot_product_attention (:906-914).
//
// Roofline: HBM.  Algorithmic bytes per (batch row, kv head) = 2 * T * 64 * sizeof(T) (K and V read
// once) -- SURVEY 8(d)'s kv_tok term.  One CTA per (kv head, batch row); 8 lanes cover one 128 B key
// row with 16 B loads (fully coalesced), 16 keys in flight per CTA iteration, fp32 softmax,
// probabilities rounded to the model dtype before P.V exactly like the flash kernels torch calls.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"
#include "attn_core.cuh"

namespace ptts {

template <typename T>
__global__ void __launch_bounds__(ATT_THREADS) attention_kernel(AttnArgs p) {
  extern __shared__ __align__(16) float sm[];
  pdl_launch_dependents();
  pdl_wait();
  if (p.ctrl != nullptr && p.ctrl->active == 0) return;
  const int per = (p.q_len + (int)gridDim.z - 1) / (int)gridDim.z;   // query positions per CTA (launch_attention: ~8)
  attention_item<T>(p, blockIdx.y, blockIdx.x, sm, threadIdx.x, [] { __syncthreads(); }, (int)blockIdx.z * per, (int)(blockIdx.z + 1) * per);
}

// decode (q_len == 1): 8 items per CTA, one warp each (TMA-staged K/V ring per warp)
template <typename T>
__global__ void __launch_bounds__(256) attention_decode_kernel(AttnArgs p) {
  extern __shared__ __align__(128) unsigned char smd[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smd) + 2 * warp;  // 128 B header: 8 warps x 2 mbarriers
  unsigned char* sm_warp = smd + 128 + (size_t)warp * attn_decode_smem_per_warp<T>();
  attention_decode_init_warp(bars, lane);
  pdl_launch_dependents();
  pdl_wait();
  if (p.ctrl != nullptr && p.ctrl->active == 0) return;
  const int pair = warp >> 1, part = warp & 1;   // two warps per item (they split the cached keys)
  const int it = blockIdx.x * 4 + pair;
  if (it >= p.B * p.nkv) return;
  int past = p.past_len;
  if (p.past_from_ctrl) past = p.prefix + p.ctrl->cur_len - 1;
  uint32_t parity = 0;
  float* xch = reinterpret_cast<float*>(smd + 128 + (size_t)8 * attn_decode_smem_per_warp<T>()) + pair * 128;
  attention_decode_item_warp<T>(p, it / p.nkv, it % p.nkv, past, sm_warp, bars, lane, parity, part, 2, xch, pair + 1);
}

// prefill (q_len > 1) on the tensor-core decode sweep, bf16 MHA: one CTA per (row, head) appends the q_len new K/V rows, then its 8
// warps take the query positions round-robin, each one a TcItem whose cached keys are the rows 0 .. past + j (or the encoder
// positions).  The scalar kernel above spends 92 us per launch on 33 positions x 512 (row, head) pairs (4.4 ms of a 9 ms prefill).
constexpr int PRE_TC_WARPS = 8;
constexpr int PRE_TC_WARP_BYTES = 2 * ATT_TC_STAGE_BYTES + 768;
__global__ void __launch_bounds__(PRE_TC_WARPS * 32) attention_prefill_tc_kernel(AttnArgs p) {
  extern __shared__ __align__(128) unsigned char smp[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smp) + 2 * warp;
  unsigned char* ring0 = smp + 128 + (size_t)warp * PRE_TC_WARP_BYTES;
  unsigned char* ring1 = ring0 + ATT_TC_STAGE_BYTES;
  float* fbuf = reinterpret_cast<float*>(ring1 + ATT_TC_STAGE_BYTES);
  attention_decode_init_warp(bars, lane);
  pdl_launch_dependents();
  pdl_wait();
  if (p.ctrl != nullptr && p.ctrl->active == 0) return;
  const int b = blockIdx.y, h = blockIdx.x;
  const int past = p.past_len;
  bf16* kc = reinterpret_cast<bf16*>(p.kcache) + (size_t)b * p.kv_b_stride + (size_t)h * p.kv_h_stride;
  bf16* vc = reinterpret_cast<bf16*>(p.vcache) + (size_t)b * p.kv_b_stride + (size_t)h * p.kv_h_stride;
  if (!p.cross) {   // append the new rows (same arithmetic as attention_item's phase A)
    const bf16* rope_cos = reinterpret_cast<const bf16*>(p.rope_cos);
    const bf16* rope_sin = reinterpret_cast<const bf16*>(p.rope_sin);
    for (int idx = threadIdx.x; idx < p.q_len * 2 * HD; idx += PRE_TC_WARPS * 32) {
      const int j = idx / (2 * HD), e = idx - j * 2 * HD, d = e & (HD - 1);
      const size_t r = (size_t)b * p.q_len + j;
      const int pos = past + j;
      if (e < HD) {
        const bf16* src = reinterpret_cast<const bf16*>(p.knew) + r * p.ldkv + p.k_col0 + h * HD;
        float x = __bfloat162float(src[d]);
        if (p.rope) {
          const float xp = __bfloat162float(src[d < HD / 2 ? d + HD / 2 : d - HD / 2]);
          x = rope_elem<bf16>(x, xp, d, rope_cos + (size_t)pos * HD, rope_sin + (size_t)pos * HD);
        }
        kc[(size_t)pos * HD + kv_swz(pos, d)] = __float2bfloat16_rn(x);
      } else {
        const bf16* src = reinterpret_cast<const bf16*>(p.vnew) + r * p.ldkv + p.v_col0 + h * HD;
        vc[(size_t)pos * HD + kv_swz(pos, d)] = src[d];
      }
    }
    __threadfence();
    asm volatile("fence.proxy.async.global;" ::: "memory");   // generic writes -> this CTA's bulk-copy reads
    __syncthreads();
  }
  uint32_t parity = 0;
  for (int j = warp; j < p.q_len; j += PRE_TC_WARPS) {
    const size_t r = (size_t)b * p.q_len + j;
    TcItem it{};
    it.q = reinterpret_cast<const bf16*>(p.q) + r * p.ldq + p.q_col0 + (size_t)h * HD;
    it.knew = nullptr; it.vnew = nullptr;
    it.kc = kc; it.vc = vc;
    it.km = p.key_mask ? p.key_mask + (size_t)b * p.mask_ld : nullptr; it.mask_len = p.mask_len;
    it.n_cached = p.cross ? p.kv_len : past + j + 1;   // causal: the rows up to and including this position (already in the cache)
    it.pos = past + j; it.cross = 1;                    // (no separate "own key" step)
    it.rope = p.rope; it.rope_cos = reinterpret_cast<const bf16*>(p.rope_cos); it.rope_sin = reinterpret_cast<const bf16*>(p.rope_sin);
    it.scale = p.scale;
    it.out = reinterpret_cast<bf16*>(p.out) + r * p.ldo + (size_t)h * HD;
    attention_decode_item_warp_tc(it, ring0, ring1, fbuf, bars, lane, parity, 0, 1, nullptr, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the zero-filled tail of a partial V stage (generic writes) before the next item's refill
    __syncwarp();
  }
}

int launch_attention(const AttnArgs& a, int dtype, cudaStream_t st, bool pdl) {
  if (a.q_len > 1 && dtype == PTTS_BF16 && a.nh == a.nkv && a.kv_t_stride == HD && !a.past_from_ctrl) {
    const size_t smem = 128 + (size_t)PRE_TC_WARPS * PRE_TC_WARP_BYTES;
    static bool attr_p = false;
    if (!attr_p) {
      PTTS_CHECK_CUDA(cudaFuncSetAttribute(attention_prefill_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr_p = true;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(a.nkv, a.B);
    cfg.blockDim = dim3(PRE_TC_WARPS * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attention_prefill_tc_kernel, a));
    return PTTS_OK;
  }
  if (a.q_len == 1) {
    const size_t smem_d = 128 + (size_t)8 * (dtype == PTTS_BF16 ? attn_decode_smem_per_warp<bf16>() : attn_decode_smem_per_warp<float>()) + 4 * 128 * sizeof(float);
    static bool attr_d = false;
    if (!attr_d) {
      PTTS_CHECK_CUDA(cudaFuncSetAttribute(attention_decode_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      PTTS_CHECK_CUDA(cudaFuncSetAttribute(attention_decode_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr_d = true;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((a.B * a.nkv + 3) / 4);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem_d;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    if (dtype == PTTS_BF16) PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attention_decode_kernel<bf16>, a));
    else PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attention_decode_kernel<float>, a));
    return PTTS_OK;
  }
  const int kv_capacity = a.kv_capacity;
  PTTS_REQUIRE(a.B > 0 && a.nkv > 0 && a.q_len > 0, "attention: empty problem");
  const size_t smem = (size_t)(HD + ATT_WARPS * HD + 8 + kv_capacity) * sizeof(float);
  PTTS_REQUIRE(smem <= 200 * 1024, "attention: kv length %d needs %zu B of shared memory (> 200 KB)", kv_capacity, smem);
  static bool attr_done = false;
  if (!attr_done) {
    PTTS_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    PTTS_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_done = true;
  }
  cudaLaunchConfig_t cfg{};
  // one CTA per (K/V head, row, slice of ~8 query positions): a 33-position prefill was 87 us per launch with one CTA sweeping all of them
  cfg.gridDim = dim3(a.nkv, a.B, (a.q_len + 7) / 8);
  cfg.blockDim = dim3(ATT_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  if (dtype == PTTS_BF16)
    PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attention_kernel<bf16>, a));
  else
    PTTS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, attention_kernel<float>, a));
  return PTTS_OK;
}

}  // namespace ptts
