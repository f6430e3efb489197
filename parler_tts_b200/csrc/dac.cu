// dac.cu -- DAC codec decode: codebook ids -> latent -> waveform.
//
// Replaces DACModel.decode (parler_tts/dac_wrapper/modeling_dac.py:106-142), i.e. the two calls into
// descript-audio-codec: quantizer.from_codes (:138) and model.decode (:139).  Arithmetic restated from
// transformers' DacModel (models/dac/modeling_dac.py:345-369 from_codes, :405-440 decoder, :234-262
// block, :173-207 residual unit, :85-99 snake); weight-norm is folded at load (reference :148-157).
//
// Layout: activations are channels-last [B][T][C] so one time step's channels are contiguous (the
// implicit-GEMM K dimension) -- the reference's cuDNN path is channels-first.
// This file is the generic fp32-accumulate implicit-GEMM path (any channel count, any dtype):
// one kernel covers Conv1d(k=7, dilated), Conv1d(k=1) and ConvTranspose1d(k=2s, stride s) by
// describing each as "n_taps shifted input rows x per-tap weight slice"; snake on the input, bias,
// residual add and tanh are fused.  Roofline: tensor/FMA-bound (1.608 GFLOP per code frame, SURVEY 8d).
#include "common.cuh"
#include "dac.h"

namespace ptts {

constexpr int CT_M = 64, CT_N = 64, CT_K = 16, CT_AROWS = 128, CT_MAXTAPS = 7;

template <typename T>
__global__ void __launch_bounds__(256) conv_kernel(ConvArgs p) {
  __shared__ float As[CT_K][CT_AROWS];
  __shared__ __align__(16) float Bs[CT_MAXTAPS][CT_K][CT_N];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int phase = blockIdx.z % p.n_phase, b = blockIdx.z / p.n_phase;
  const int q0 = blockIdx.x * CT_M, co0 = blockIdx.y * CT_N;
  const int wt_base = p.wt_base + phase * p.wt_phase_step;
  // input row window of this tile: q0 + off_lo .. q0 + CT_M - 1 + off_hi
  const int off_last = p.off_base + (p.n_taps - 1) * p.off_step;
  const int off_lo = min(p.off_base, off_last);
  const T* __restrict__ x = reinterpret_cast<const T*>(p.x) + (size_t)b * p.Tin * p.Cin;
  const T* __restrict__ w = reinterpret_cast<const T*>(p.w);
  const T* __restrict__ alpha = reinterpret_cast<const T*>(p.alpha);
  const int arows = CT_M + abs(off_last - p.off_base);

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; i++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[i][j] = 0.f;

  for (int ci0 = 0; ci0 < p.Cin; ci0 += CT_K) {
    __syncthreads();
    // A tile: (snake of) x[q0+off_lo+r][ci0+c], zero outside [0,Tin) -- conv zero padding
    for (int e = tid; e < arows * CT_K; e += 256) {
      const int r = e / CT_K, c = e - r * CT_K;
      const int t = q0 + off_lo + r, ci = ci0 + c;
      float v = 0.f;
      if (t >= 0 && t < p.Tin && ci < p.Cin) {
        v = DT<T>::to_f(x[(size_t)t * p.Cin + ci]);
        if (alpha != nullptr) {
          const float a = DT<T>::to_f(alpha[ci]);
          v = snake_fn<T>(v, a, DT<T>::rnd(1.0f / DT<T>::rnd(a + 1e-9f)));
        }
      }
      As[c][r] = v;
    }
    // B tile: w[tap][ci0+c][co0+n]
    for (int e = tid; e < p.n_taps * CT_K * CT_N; e += 256) {
      const int n = e % CT_N, c = (e / CT_N) % CT_K, j = e / (CT_N * CT_K);
      const int ci = ci0 + c, co = co0 + n;
      float v = 0.f;
      if (ci < p.Cin && co < p.Cout) v = DT<T>::to_f(w[((size_t)(wt_base + j * p.wt_step) * p.Cin + ci) * p.Cout + co]);
      Bs[j][c][n] = v;
    }
    __syncthreads();
    for (int j = 0; j < p.n_taps; j++) {
      const int roff = p.off_base + j * p.off_step - off_lo;
#pragma unroll
      for (int c = 0; c < CT_K; c++) {
        const float4 bv = *reinterpret_cast<const float4*>(&Bs[j][c][tx * 4]);
        float av[4];
#pragma unroll
        for (int i = 0; i < 4; i++) av[i] = As[c][ty * 4 + i + roff];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          acc[i][0] = fmaf(av[i], bv.x, acc[i][0]);
          acc[i][1] = fmaf(av[i], bv.y, acc[i][1]);
          acc[i][2] = fmaf(av[i], bv.z, acc[i][2]);
          acc[i][3] = fmaf(av[i], bv.w, acc[i][3]);
        }
      }
    }
  }
  const T* __restrict__ bias = reinterpret_cast<const T*>(p.bias);
  const T* __restrict__ res = reinterpret_cast<const T*>(p.res);
  T* __restrict__ out = reinterpret_cast<T*>(p.out);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int q = q0 + ty * 4 + i;
    if (q >= p.q_count) continue;
    const int to = q * p.o_mul + p.o_add + phase * p.o_phase_step;
    if (to < 0 || to >= p.Tout) continue;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int co = co0 + tx * 4 + j;
      if (co >= p.Cout) continue;
      float v = DT<T>::rnd(acc[i][j] + DT<T>::to_f(bias[co]));
      const size_t o = ((size_t)b * p.Tout + to) * p.Cout + co;
      if (res != nullptr) v = DT<T>::rnd(DT<T>::to_f(res[o]) + v);
      if (p.tanh_out) v = tanhf(v);
      out[o] = DT<T>::from_f(v);
    }
  }
}

int launch_conv(const ConvArgs& a, int dtype, int B, cudaStream_t st) {
  PTTS_REQUIRE(a.n_taps >= 1 && a.n_taps <= CT_MAXTAPS, "conv: n_taps %d out of range", a.n_taps);
  PTTS_REQUIRE(CT_M + abs((a.n_taps - 1) * a.off_step) <= CT_AROWS, "conv: receptive field too wide");
  dim3 grid((a.q_count + CT_M - 1) / CT_M, (a.Cout + CT_N - 1) / CT_N, B * a.n_phase);
  if (dtype == PTTS_BF16) conv_kernel<bf16><<<grid, 256, 0, st>>>(a);
  else conv_kernel<float><<<grid, 256, 0, st>>>(a);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// quantizer.from_codes: z[b][t][c] = sum_k ( out_proj_k.bias[c] + sum_d out_proj_k.w[c][d] * codebook_k[code][d] )
// accumulated codebook by codebook in the storage dtype (quantized_representation += ..., :367).
template <typename T>
__global__ void __launch_bounds__(256) from_codes_kernel(FromCodesArgs p) {
  __shared__ float e[32][16];  // [k][d] for this (b, t)
  const int t = blockIdx.x, b = blockIdx.y;
  const int K = p.K, D = p.D;
  if (threadIdx.x < K * D) {
    const int k = threadIdx.x / D, d = threadIdx.x - k * D;
    const int64_t code = p.codes[((size_t)b * K + k) * p.T + t];
    e[k][d] = DT<T>::to_f(reinterpret_cast<const T*>(p.codebooks)[((size_t)k * p.codebook_size + code) * D + d]);
  }
  __syncthreads();
  const T* __restrict__ W = reinterpret_cast<const T*>(p.proj_w);
  const T* __restrict__ Bv = reinterpret_cast<const T*>(p.proj_b);
  T* __restrict__ z = reinterpret_cast<T*>(p.z) + ((size_t)b * p.T + t) * p.C;
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < K; k++) {
      float s = 0.f;
      for (int d = 0; d < D; d++) s = fmaf(DT<T>::to_f(W[((size_t)k * p.C + c) * D + d]), e[k][d], s);
      s = DT<T>::rnd(s + DT<T>::to_f(Bv[(size_t)k * p.C + c]));
      acc = (k == 0) ? s : DT<T>::rnd(acc + s);
    }
    z[c] = DT<T>::from_f(acc);
  }
}
int launch_from_codes(const FromCodesArgs& a, int dtype, int B, cudaStream_t st) {
  PTTS_REQUIRE(a.K <= 32 && a.D <= 16 && a.K * a.D <= 256, "from_codes: K=%d D=%d unsupported", a.K, a.D);
  dim3 grid(a.T, B);
  if (dtype == PTTS_BF16) from_codes_kernel<bf16><<<grid, 256, 0, st>>>(a);
  else from_codes_kernel<float><<<grid, 256, 0, st>>>(a);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// ---- weight repack: Conv1d [co][ci][k] / ConvTranspose1d [ci][co][k] -> [k][ci][co] ---------------
template <typename S, typename D>
__global__ void pack_conv_kernel(const S* src, D* dst, int d0, int d1, int k, int transposed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = (int64_t)d0 * d1 * k;
  if (i >= n) return;
  const int kk = (int)(i % k);
  const int b1 = (int)((i / k) % d1), b0 = (int)(i / ((int64_t)k * d1));
  // conv: (b0,b1)=(co,ci); convT: (b0,b1)=(ci,co)
  const int ci = transposed ? b0 : b1, co = transposed ? b1 : b0;
  const int Cin = transposed ? d0 : d1, Cout = transposed ? d1 : d0;
  float v;
  if constexpr (sizeof(S) == 2) v = __bfloat162float(src[i]); else v = src[i];
  const size_t o = ((size_t)kk * Cin + ci) * Cout + co;
  if constexpr (sizeof(D) == 2) dst[o] = __float2bfloat16_rn(v); else dst[o] = v;
}
int pack_conv(const void* src, int src_dtype, void* dst, int dst_dtype, int d0, int d1, int k, int transposed, cudaStream_t st) {
  const int64_t n = (int64_t)d0 * d1 * k;
  const int blocks = (int)((n + 255) / 256);
  if (src_dtype == PTTS_BF16 && dst_dtype == PTTS_BF16) pack_conv_kernel<bf16, bf16><<<blocks, 256, 0, st>>>((const bf16*)src, (bf16*)dst, d0, d1, k, transposed);
  else if (src_dtype == PTTS_BF16) pack_conv_kernel<bf16, float><<<blocks, 256, 0, st>>>((const bf16*)src, (float*)dst, d0, d1, k, transposed);
  else if (dst_dtype == PTTS_BF16) pack_conv_kernel<float, bf16><<<blocks, 256, 0, st>>>((const float*)src, (bf16*)dst, d0, d1, k, transposed);
  else pack_conv_kernel<float, float><<<blocks, 256, 0, st>>>((const float*)src, (float*)dst, d0, d1, k, transposed);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// audio [B][T][1] is already [B, 1, T] contiguous: nothing to transpose for the final layer.


// ---- output convolution: Conv1d(C -> 1, k = 7) + tanh on the channels-last, already snake'd tensor ----------------------------
// The generic tile kernel above computes a 64 x 64 output tile: with ONE output channel 63/64 of its FMAs are wasted and it took
// 2.5 ms for 32 x 57 frames (11 ms at the bench's 248 frames: a third of the whole decode; profiles/r02_launches.md).
// Here one thread owns one output sample: the 128 + 6 input rows of a block are staged in shared memory (row pitch padded to
// C + 8 elements so that 8 consecutive threads' 16-byte reads hit 8 different bank groups), weights [7][C] as fp32.
// bf16 inputs, fp32 accumulation in tap-major / channel order, one rounding of acc + bias, tanh, one rounding (torch's ops).
constexpr int FC_T = 128;   // outputs per block
__global__ void __launch_bounds__(FC_T) final_conv_tanh_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w, const bf16* __restrict__ bias,
                                                               bf16* __restrict__ out, int C, int T) {
  extern __shared__ __align__(16) unsigned char fsm[];
  const int pitch = C + 8;                                   // elements
  bf16* xs = reinterpret_cast<bf16*>(fsm);                   // [FC_T + 6][pitch]
  float* ws = reinterpret_cast<float*>(fsm + (size_t)(FC_T + 6) * pitch * 2);   // [7][C]
  const int b = blockIdx.y, t0 = blockIdx.x * FC_T, tid = threadIdx.x;
  const bf16* xb = x + (size_t)b * T * C;
  const int vec_per_row = C / 8;
  for (int e = tid; e < (FC_T + 6) * vec_per_row; e += FC_T) {
    const int r = e / vec_per_row, c = e - r * vec_per_row;
    const int t = t0 - 3 + r;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);                    // zero padding outside [0, T)
    if (t >= 0 && t < T) v = *reinterpret_cast<const uint4*>(xb + (size_t)t * C + c * 8);
    *reinterpret_cast<uint4*>(xs + (size_t)r * pitch + c * 8) = v;
  }
  for (int e = tid; e < 7 * C; e += FC_T) ws[e] = __bfloat162float(w[e]);   // packed [tap][Cin][Cout = 1]
  __syncthreads();
  const int t = t0 + tid;
  if (t >= T) return;
  float acc = 0.f;
  for (int j = 0; j < 7; j++) {
    const bf16* row = xs + (size_t)(tid + j) * pitch;
    const float* wj = ws + j * C;
    for (int c = 0; c < C; c += 8) {
      float v[8];
      load8(row + c, v);
#pragma unroll
      for (int e = 0; e < 8; e++) acc = fmaf(v[e], wj[c + e], acc);
    }
  }
  const float y = DT<bf16>::rnd(acc + __bfloat162float(bias[0]));
  out[(size_t)b * T + t] = __float2bfloat16_rn(tanhf(y));
}

bool final_conv_supported(int C) { return C % 8 == 0 && C <= 512; }
int launch_final_conv_tanh(const void* x, const void* w, const void* bias, void* out, int C, int T, int B, cudaStream_t st) {
  const size_t smem = (size_t)(FC_T + 6) * (C + 8) * 2 + (size_t)7 * C * 4;
  static bool attr = false;
  if (!attr) { PTTS_CHECK_CUDA(cudaFuncSetAttribute(final_conv_tanh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024)); attr = true; }
  final_conv_tanh_kernel<<<dim3((T + FC_T - 1) / FC_T, B), FC_T, smem, st>>>((const bf16*)x, (const bf16*)w, (const bf16*)bias, (bf16*)out, C, T);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

}  // namespace ptts
