// dac_enc.cu -- DAC codec encode: waveform -> latent -> residual-vector-quantized codes (the voice-prompt path).
//
// Replaces DACModel.encode (parler_tts/dac_wrapper/modeling_dac.py:33-104), i.e. DAC.encode = encoder + quantizer.  Arithmetic
// restated from transformers' DacModel (models/dac/modeling_dac.py:442-473 encoder, :210-232 block, :173-207 residual unit,
// :281-343 residual vector quantizer, :122-170 vector quantize); weight-norm is folded at load.
//
// Activations are channels-last [B][T][C] like the decoder's (dac.cu).  bf16 with tcgen05-sized channel counts:
//   conv1 (1 -> D, k7)        enc_conv1_kernel below, also writes snake(x) for the first residual unit
//   residual units, conv2     launch_conv_tc (dac_tc.cu), the next layer's snake fused into the epilogue
//   strided conv (k 2s, /s)   launch_conv_tc_down (dac_tc.cu)
// f32 (and channel counts the tensor-core path does not take): conv1 below, residual units and conv2 on the generic conv_kernel
// (dac.cu), the strided conv on conv_down_kernel below.  The quantizer is rvq_kernel below for both.
// Roofline: ~1.39 MFLOP per input sample in the convolutions (tensor pipe); the quantizer is ~0.4 MFLOP per code frame.
#include <algorithm>

#include "common.cuh"
#include "dac.h"
#include "kernels.h"

namespace ptts {

// ---- conv1: Conv1d(1 -> D, k = 7, padding 3) on the [B][n] waveform ----------------------------------------------------
// out_raw = bf16(acc + bias) (taps in order, fp32), out_act = snake_{alpha}(out_raw) for the first residual unit (nullptr: skip).
constexpr int C1_T = 64;   // samples per block
template <typename T>
__global__ void __launch_bounds__(256) enc_conv1_kernel(const T* __restrict__ audio, const T* __restrict__ w /*[7][D]*/, const T* __restrict__ bias,
                                                        const T* __restrict__ alpha, T* __restrict__ out_raw, T* __restrict__ out_act, int D, int64_t n) {
  __shared__ float xs[C1_T + 6];
  const int b = blockIdx.y;
  const int64_t t0 = (int64_t)blockIdx.x * C1_T;
  const T* xb = audio + (size_t)b * n;
  for (int i = threadIdx.x; i < C1_T + 6; i += blockDim.x) {
    const int64_t t = t0 - 3 + i;
    xs[i] = (t >= 0 && t < n) ? DT<T>::to_f(xb[t]) : 0.f;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < C1_T * D; e += blockDim.x) {
    const int f = e / D, co = e - f * D;
    const int64_t t = t0 + f;
    if (t >= n) break;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 7; k++) acc = fmaf(xs[f + k], DT<T>::to_f(w[k * D + co]), acc);
    const float v = DT<T>::rnd(acc + DT<T>::to_f(bias[co]));
    const size_t o = ((size_t)b * n + t) * D + co;
    out_raw[o] = DT<T>::from_f(v);
    if (out_act != nullptr) {
      const float a = DT<T>::to_f(alpha[co]);
      out_act[o] = DT<T>::from_f(snake_fn<T>(v, a, DT<T>::rnd(1.0f / DT<T>::rnd(a + 1e-9f))));
    }
  }
}

// ---- strided conv, SIMT: Conv1d(k = 2s, stride s, padding s/2) of snake_{alpha}(x), one output row per block --------------
// x [B][Tin][Cin], w [2s][Cin][Cout] (pack_conv order) -> out [B][Tin/s][Cout].
template <typename T>
__global__ void __launch_bounds__(256) conv_down_kernel(const T* __restrict__ x, const T* __restrict__ w, const T* __restrict__ bias,
                                                        const T* __restrict__ alpha, T* __restrict__ out, int Cin, int Cout, int Tin, int s) {
  extern __shared__ float win[];   // [2s][Cin] snake'd input window of this output row
  const int q = blockIdx.x, b = blockIdx.y;
  const T* xb = x + (size_t)b * Tin * Cin;
  for (int e = threadIdx.x; e < 2 * s * Cin; e += blockDim.x) {
    const int k = e / Cin, ci = e - k * Cin;
    const int t = q * s + k - s / 2;
    float v = 0.f;
    if (t >= 0 && t < Tin) {
      const float a = DT<T>::to_f(alpha[ci]);
      v = snake_fn<T>(DT<T>::to_f(xb[(size_t)t * Cin + ci]), a, DT<T>::rnd(1.0f / DT<T>::rnd(a + 1e-9f)));
    }
    win[e] = v;
  }
  __syncthreads();
  for (int co = threadIdx.x; co < Cout; co += blockDim.x) {
    float acc = 0.f;
    for (int e = 0; e < 2 * s * Cin; e++) acc = fmaf(win[e], DT<T>::to_f(w[(size_t)e * Cout + co]), acc);
    out[((size_t)b * (Tin / s) + q) * Cout + co] = DT<T>::from_f(DT<T>::rnd(acc + DT<T>::to_f(bias[co])));
  }
}

// ---- codebook normalisation at pack time: F.normalize(codebook) = x / max(||x||, 1e-12), norm and quotient rounded ----------
template <typename T>
__global__ void normalize_codebook_kernel(const T* __restrict__ cb, T* __restrict__ out, int cs, int D) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= cs) return;
  float s = 0.f;
  for (int d = 0; d < D; d++) { const float v = DT<T>::to_f(cb[(size_t)j * D + d]); s = fmaf(v, v, s); }
  const float den = fmaxf(DT<T>::rnd(sqrtf(s)), 1e-12f);
  for (int d = 0; d < D; d++) out[(size_t)j * D + d] = DT<T>::from_f(DT<T>::to_f(cb[(size_t)j * D + d]) / den);
}
int normalize_codebook(const void* codebook, void* out, int cs, int D, int dtype, cudaStream_t st) {
  const int blocks = (cs + 255) / 256;
  if (dtype == PTTS_BF16) normalize_codebook_kernel<bf16><<<blocks, 256, 0, st>>>((const bf16*)codebook, (bf16*)out, cs, D);
  else normalize_codebook_kernel<float><<<blocks, 256, 0, st>>>((const float*)codebook, (float*)out, cs, D);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// ---- residual vector quantizer ----------------------------------------------------------------------------------------
// One CTA per RVQ_TF frames; the residual stays in shared memory (fp32 holding model-dtype values) and the CTA walks the n_q
// codebooks in order.  Per codebook, with every torch op's output rounded to the model dtype:
//   proj = in_proj(residual)                    enc = proj / max(||proj||, 1e-12)
//   code = argmax_j  -(|enc|^2 - 2 enc.cbn_j) + |cbn_j|^2   (cbn = normalised codebook; fp32 from the rounded operands,
//                                                            ties to the lowest index -- DESIGN.md section 5)
//   st   = proj + (codebook[code] - proj)       q = out_proj(st)       residual -= q       z += q
constexpr int RVQ_TF = 8, RVQ_THREADS = 256, RVQ_WARPS = RVQ_THREADS / 32, RVQ_DMAX = 16;
struct RvqArgs {
  const void* ze;                  // [B][T][Z]
  const void* in_w; const void* in_b; const void* codebooks; const void* cb_norm; const void* out_w; const void* out_b;
  int64_t* codes;                  // [B][n_q][T]
  void* z;                         // [B][T][Z] or nullptr
  int T, Z, D, cs, n_q;
};

template <typename T>
__global__ void __launch_bounds__(RVQ_THREADS) rvq_kernel(RvqArgs p) {
  extern __shared__ float rsm[];
  const int Z = p.Z, D = p.D, cs = p.cs;
  float* res = rsm;                                  // [TF][Z]
  float* zacc = res + RVQ_TF * Z;                    // [TF][Z]
  float* proj = zacc + RVQ_TF * Z;                   // [TF][DMAX]
  float* enc = proj + RVQ_TF * RVQ_DMAX;             // [TF][DMAX]
  float* stq = enc + RVQ_TF * RVQ_DMAX;              // [TF][DMAX]
  float* l2 = stq + RVQ_TF * RVQ_DMAX;               // [TF]
  float* wbest = l2 + RVQ_TF;                        // [WARPS][TF]
  int* widx = reinterpret_cast<int*>(wbest + RVQ_WARPS * RVQ_TF);   // [WARPS][TF]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.y, t0 = blockIdx.x * RVQ_TF;
  const int nf = min(RVQ_TF, p.T - t0);
  const T* ze = reinterpret_cast<const T*>(p.ze) + ((size_t)b * p.T + t0) * Z;
  for (int e = tid; e < RVQ_TF * Z; e += RVQ_THREADS) {
    const int f = e / Z;
    res[e] = f < nf ? DT<T>::to_f(ze[e]) : 0.f;
    zacc[e] = 0.f;
  }
  __syncthreads();
  for (int k = 0; k < p.n_q; k++) {
    const T* in_w = reinterpret_cast<const T*>(p.in_w) + (size_t)k * D * Z;
    const T* in_b = reinterpret_cast<const T*>(p.in_b) + (size_t)k * D;
    // in_proj: one warp per (frame, d) dot product over Z
    for (int o = warp; o < RVQ_TF * D; o += RVQ_WARPS) {
      const int f = o / D, d = o - f * D;
      float acc = 0.f;
      for (int c = lane; c < Z; c += 32) acc = fmaf(res[f * Z + c], DT<T>::to_f(in_w[(size_t)d * Z + c]), acc);
      acc = warp_sum(acc);
      if (lane == 0) proj[f * RVQ_DMAX + d] = DT<T>::rnd(acc + DT<T>::to_f(in_b[d]));
    }
    __syncthreads();
    if (tid < RVQ_TF) {   // F.normalize and |enc|^2 (pow(2) rounded, then summed)
      const int f = tid;
      float s = 0.f;
      for (int d = 0; d < D; d++) s = fmaf(proj[f * RVQ_DMAX + d], proj[f * RVQ_DMAX + d], s);
      const float den = fmaxf(DT<T>::rnd(sqrtf(s)), 1e-12f);
      float n2 = 0.f;
      for (int d = 0; d < D; d++) {
        const float e = DT<T>::rnd(proj[f * RVQ_DMAX + d] / den);
        enc[f * RVQ_DMAX + d] = e;
        n2 += DT<T>::rnd(e * e);
      }
      for (int d = D; d < RVQ_DMAX; d++) enc[f * RVQ_DMAX + d] = 0.f;
      l2[f] = DT<T>::rnd(n2);
    }
    __syncthreads();
    // code search: each thread scans codes tid, tid + 256, ... (ascending, so a strict > keeps the lowest index of a tie)
    float best[RVQ_TF];
    int bidx[RVQ_TF];
#pragma unroll
    for (int f = 0; f < RVQ_TF; f++) { best[f] = -INFINITY; bidx[f] = 0x7fffffff; }
    const T* cbn = reinterpret_cast<const T*>(p.cb_norm) + (size_t)k * cs * D;
    for (int j = tid; j < cs; j += RVQ_THREADS) {
      float cv[RVQ_DMAX];
      float csq = 0.f;
#pragma unroll
      for (int d = 0; d < RVQ_DMAX; d++) {
        cv[d] = d < D ? DT<T>::to_f(cbn[(size_t)j * D + d]) : 0.f;
        csq += cv[d] * cv[d];
      }
#pragma unroll
      for (int f = 0; f < RVQ_TF; f++) {
        float dot = 0.f;
#pragma unroll
        for (int d = 0; d < RVQ_DMAX; d++) dot = fmaf(enc[f * RVQ_DMAX + d], cv[d], dot);
        const float dist = -(l2[f] - 2.f * dot) + csq;
        if (dist > best[f]) { best[f] = dist; bidx[f] = j; }
      }
    }
#pragma unroll
    for (int f = 0; f < RVQ_TF; f++) {
      float v = best[f];
      int i = bidx[f];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float v2 = __shfl_xor_sync(0xffffffffu, v, o);
        const int i2 = __shfl_xor_sync(0xffffffffu, i, o);
        if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
      }
      if (lane == 0) { wbest[warp * RVQ_TF + f] = v; widx[warp * RVQ_TF + f] = i; }
    }
    __syncthreads();
    if (tid < RVQ_TF) {
      const int f = tid;
      float v = wbest[f];
      int i = widx[f];
      for (int w = 1; w < RVQ_WARPS; w++) {
        const float v2 = wbest[w * RVQ_TF + f];
        const int i2 = widx[w * RVQ_TF + f];
        if (v2 > v || (v2 == v && i2 < i)) { v = v2; i = i2; }
      }
      if (i < 0 || i >= cs) i = 0;   // all distances NaN: torch's max would return some index too; stay in range
      if (f < nf) p.codes[((size_t)b * p.n_q + k) * p.T + t0 + f] = i;
      // straight-through value on the un-normalised codebook: proj + (z_q - proj)
      const T* cb = reinterpret_cast<const T*>(p.codebooks) + ((size_t)k * cs + i) * D;
      for (int d = 0; d < D; d++) {
        const float pr = proj[f * RVQ_DMAX + d];
        stq[f * RVQ_DMAX + d] = DT<T>::rnd(pr + DT<T>::rnd(DT<T>::to_f(cb[d]) - pr));
      }
    }
    __syncthreads();
    const T* out_w = reinterpret_cast<const T*>(p.out_w) + (size_t)k * Z * D;
    const T* out_b = reinterpret_cast<const T*>(p.out_b) + (size_t)k * Z;
    for (int e = tid; e < RVQ_TF * Z; e += RVQ_THREADS) {
      const int f = e / Z, c = e - f * Z;
      float acc = 0.f;
      for (int d = 0; d < D; d++) acc = fmaf(DT<T>::to_f(out_w[(size_t)c * D + d]), stq[f * RVQ_DMAX + d], acc);
      const float q = DT<T>::rnd(acc + DT<T>::to_f(out_b[c]));
      res[e] = DT<T>::rnd(res[e] - q);
      zacc[e] = k == 0 ? q : DT<T>::rnd(zacc[e] + q);
    }
    __syncthreads();
  }
  if (p.z != nullptr) {
    T* z = reinterpret_cast<T*>(p.z) + ((size_t)b * p.T + t0) * Z;
    for (int e = tid; e < nf * Z; e += RVQ_THREADS) z[e] = DT<T>::from_f(zacc[e]);
  }
}

static size_t rvq_smem(int Z) {
  return (size_t)(2 * RVQ_TF * Z + 3 * RVQ_TF * RVQ_DMAX + RVQ_TF + 2 * RVQ_WARPS * RVQ_TF) * 4;
}

template <typename T>
static int launch_rvq(const RvqArgs& a, int B, cudaStream_t st) {
  const size_t smem = rvq_smem(a.Z);
  static bool attr = false;
  if (!attr) { PTTS_CHECK_CUDA(cudaFuncSetAttribute(rvq_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rvq_smem(2048))); attr = true; }
  rvq_kernel<T><<<dim3((a.T + RVQ_TF - 1) / RVQ_TF, B), RVQ_THREADS, smem, st>>>(a);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

template <typename T>
static int launch_conv_down(const void* x, const void* w, const void* bias, const void* alpha, void* out, int Cin, int Cout, int Tin, int s, int B,
                            cudaStream_t st) {
  const size_t smem = (size_t)2 * s * Cin * 4;
  PTTS_REQUIRE(smem <= 200 * 1024, "conv_down: window of %d x %d too large", 2 * s, Cin);
  static bool attr = false;
  if (!attr) { PTTS_CHECK_CUDA(cudaFuncSetAttribute(conv_down_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); attr = true; }
  conv_down_kernel<T><<<dim3(Tin / s, B), 256, smem, st>>>((const T*)x, (const T*)w, (const T*)bias, (const T*)alpha, (T*)out, Cin, Cout, Tin, s);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

// largest activation of one utterance, in elements
static int64_t max_act(const ptts_dac_encoder_config& c, int64_t n) {
  int64_t m = n * c.encoder_dim, len = n;
  for (int i = 0; i < c.n_blocks; i++) {
    len /= c.strides[i];
    m = std::max(m, len * (int64_t)(c.encoder_dim << (i + 1)));
  }
  return std::max(m, len * (int64_t)c.latent_dim);
}

int64_t dac_encoder_workspace(const ptts_dac_encoder_config& c, int B, int64_t n) {
  return 3 * align_up(max_act(c, n) * B * dtype_size(c.dtype), 1024);
}

int dac_encode(const ptts_dac_encoder_config& c, const char* bl, char* ws, int64_t ws_bytes, const void* audio, int B, int64_t n, int n_q,
               int64_t* codes, void* z, cudaStream_t st) {
  const int64_t hop = dac_encoder_hop(c);
  PTTS_REQUIRE(B > 0 && n > 0 && n % hop == 0, "dac encode: n_samples %lld must be a positive multiple of the hop %lld", (long long)n, (long long)hop);
  PTTS_REQUIRE(n <= (int64_t)1 << 30, "dac encode: n_samples %lld too large", (long long)n);
  PTTS_REQUIRE(n_q >= 1 && n_q <= c.n_codebooks, "dac encode: n_q %d out of [1, %d]", n_q, c.n_codebooks);
  PTTS_REQUIRE(ws_bytes >= dac_encoder_workspace(c, B, n), "dac encode: workspace too small");
  const DacEncLayout L = make_dac_encoder_layout(c);
  const int64_t buf = align_up(max_act(c, n) * B * L.es, 1024);
  char* bufX = ws;
  char* bufA = ws + buf;
  char* bufB = ws + 2 * buf;
  const int D = c.encoder_dim, dm = D << c.n_blocks, Z = c.latent_dim;
  const bool bf = c.dtype == PTTS_BF16;
  auto tp = [&](int i) { return bl + L.t[i].off; };
  auto tpk = [&](int i) { return bl + L.t[i].off_k; };

  bool use_tc = bf && conv_tc_supported(dm, Z);
  for (int bi = 0; bi < c.n_blocks && use_tc; bi++) use_tc = conv_tc_supported(D << bi, D << bi) && conv_tc_down_supported(D << bi, D << (bi + 1));

  const int c1_blocks = (int)((n + C1_T - 1) / C1_T);
  if (bf) enc_conv1_kernel<bf16><<<dim3(c1_blocks, B), 256, 0, st>>>((const bf16*)audio, (const bf16*)tp(0), (const bf16*)tp(1), (const bf16*)tp(2),
                                                                     (bf16*)bufX, use_tc ? (bf16*)bufA : nullptr, D, n);
  else enc_conv1_kernel<float><<<dim3(c1_blocks, B), 256, 0, st>>>((const float*)audio, (const float*)tp(0), (const float*)tp(1), (const float*)tp(2),
                                                                   (float*)bufX, nullptr, D, n);
  PTTS_LAUNCH_CHECK();
  int ti = 2;
  int Tlen = (int)n;
  const int dil[3] = {1, 3, 9};
  char* ze;
  if (use_tc) {
    // bufX: raw residual stream; act: snake'd input of the next conv; oth: scratch
    char* act = bufA;
    char* oth = bufB;
    auto convk = [&](const void* x, int w_i, int b_i, const void* res, void* out_raw, void* out_act, const void* alpha_next, int Cin, int Cout, int ks, int dl) {
      ConvArgs a{};
      a.x = x; a.bias = tp(b_i); a.res = res;
      a.Cin = Cin; a.Cout = Cout; a.Tin = Tlen; a.Tout = Tlen; a.q_count = Tlen;
      a.n_taps = ks; a.off_base = -((ks - 1) / 2) * dl; a.off_step = dl; a.wt_base = 0; a.wt_step = 1;
      a.n_phase = 1; a.wt_phase_step = 0; a.o_mul = 1; a.o_add = 0; a.o_phase_step = 0;
      return launch_conv_tc(a, tpk(w_i), ks, alpha_next, out_raw, out_act, B, st);
    };
    for (int bi = 0; bi < c.n_blocks; bi++) {
      const int ch = D << bi, s = c.strides[bi];
      for (int r = 0; r < 3; r++) {
        // y = conv7(snake1(x)) -> only snake2(y) is stored; x += conv1(snake2(y)), plus snake_next(x) for what follows
        if (int e = convk(act, ti + 1, ti + 2, nullptr, nullptr, oth, tp(ti + 3), ch, ch, 7, dil[r])) return e;
        if (int e = convk(oth, ti + 4, ti + 5, bufX, bufX, act, tp(ti + 6), ch, ch, 1, 1)) return e;   // ti + 6: next unit's or the block's snake
        ti += 6;
      }
      // act = snake_block(x): strided conv -> raw (the next block's residual stream) + snake for the next block / final snake
      if (int e = launch_conv_tc_down(act, tpk(ti + 1), tp(ti + 2), tp(ti + 3), bufX, oth, ch, 2 * ch, Tlen, s, B, st)) return e;
      std::swap(act, oth);
      ti += 3;
      Tlen /= s;
    }
    if (int e = convk(act, ti + 1, ti + 2, nullptr, oth, nullptr, nullptr, dm, Z, 3, 1)) return e;
    ze = oth;
  } else {
    char* cur = bufX;
    char* oth = bufA;
    auto conv = [&](const void* x, int w_i, int b_i, const void* alpha, const void* res, void* out, int Cin, int Cout, int ks, int dl) {
      ConvArgs a{};
      a.x = x; a.w = tp(w_i); a.bias = tp(b_i); a.alpha = alpha; a.res = res; a.out = out;
      a.Cin = Cin; a.Cout = Cout; a.Tin = Tlen; a.Tout = Tlen; a.q_count = Tlen;
      a.n_taps = ks; a.off_base = -((ks - 1) / 2) * dl; a.off_step = dl; a.wt_base = 0; a.wt_step = 1;
      a.n_phase = 1; a.wt_phase_step = 0; a.o_mul = 1; a.o_add = 0; a.o_phase_step = 0; a.tanh_out = 0;
      return launch_conv(a, c.dtype, B, st);
    };
    for (int bi = 0; bi < c.n_blocks; bi++) {
      const int ch = D << bi, s = c.strides[bi];
      for (int r = 0; r < 3; r++) {
        if (int e = conv(cur, ti + 1, ti + 2, tp(ti), nullptr, oth, ch, ch, 7, dil[r])) return e;
        if (int e = conv(oth, ti + 4, ti + 5, tp(ti + 3), cur, cur, ch, ch, 1, 1)) return e;
        ti += 6;
      }
      int e = bf ? launch_conv_down<bf16>(cur, tp(ti + 1), tp(ti + 2), tp(ti), oth, ch, 2 * ch, Tlen, s, B, st)
                 : launch_conv_down<float>(cur, tp(ti + 1), tp(ti + 2), tp(ti), oth, ch, 2 * ch, Tlen, s, B, st);
      if (e) return e;
      std::swap(cur, oth);
      ti += 3;
      Tlen /= s;
    }
    if (int e = conv(cur, ti + 1, ti + 2, tp(ti), nullptr, oth, dm, Z, 3, 1)) return e;
    ze = oth;
  }
  RvqArgs q{ze, bl + L.in_w, bl + L.in_b, bl + L.codebooks, bl + L.cb_norm, bl + L.out_w, bl + L.out_b, codes, z, Tlen, Z, c.codebook_dim,
            c.codebook_size, n_q};
  return bf ? launch_rvq<bf16>(q, B, st) : launch_rvq<float>(q, B, st);
}

}  // namespace ptts
