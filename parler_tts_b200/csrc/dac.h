// dac.h -- DAC decode: kernel argument structs, blob layout and tensor table.
#pragma once
#include <vector>
#include "common.cuh"
#include "layout.h"

namespace ptts {

// snake(x) = x + (alpha + 1e-9)^-1 * sin(alpha x)^2, every op rounded to the storage dtype like torch.
template <typename T>
__device__ __forceinline__ float snake_fn(float x, float alpha, float inv) {
  const float s = DT<T>::rnd(sinf(DT<T>::rnd(alpha * x)));
  return DT<T>::rnd(x + DT<T>::rnd(inv * DT<T>::rnd(s * s)));
}

// One launch of the generic implicit-GEMM kernel.  Output row of tile row q (per phase):
//   to = q*o_mul + o_add + phase*o_phase_step;   input row for tap j: q + off_base + j*off_step;
//   weight slice for tap j: wt_base + phase*wt_phase_step + j*wt_step   (weights are [tap][Cin][Cout]).
struct ConvArgs {
  const void* x; const void* w; const void* bias; const void* alpha; const void* res; void* out;
  int Cin, Cout, Tin, Tout, q_count;
  int n_taps, off_base, off_step, wt_base, wt_step;
  int n_phase, wt_phase_step, o_mul, o_add, o_phase_step;
  int tanh_out;
};
int launch_conv(const ConvArgs& a, int dtype, int B, cudaStream_t st);

struct FromCodesArgs {
  const int64_t* codes;  // [B][K][T]
  const void* codebooks; const void* proj_w; const void* proj_b;  // [K][cs][D], [K][C][D], [K][C]
  void* z;               // [B][T][C]
  int K, D, C, T, codebook_size;
};
int launch_from_codes(const FromCodesArgs& a, int dtype, int B, cudaStream_t st);
int pack_conv(const void* src, int src_dtype, void* dst, int dst_dtype, int d0, int d1, int k, int transposed, cudaStream_t st);
// tcgen05 path (dac_tc.cu)
bool conv_tc_supported(int Cin, int Cout);
int launch_conv_tc(const ConvArgs& a, const void* w_kmajor, int taps_total, const void* alpha_next, void* out_raw, void* out_act, int B, cudaStream_t st);
// Conv1d(k = 2s, stride s, padding s/2) on tcgen05, s even, Cin % 64 == 0: x [B][Tin][Cin] -> [B][Tin/s][Cout] (encoder downsampling)
bool conv_tc_down_supported(int Cin, int Cout);
int launch_conv_tc_down(const void* x, const void* w_kmajor, const void* bias, const void* alpha_next, void* out_raw, void* out_act,
                        int Cin, int Cout, int Tin, int s, int B, cudaStream_t st);
int pack_conv_kmajor(const void* src, int src_dtype, void* dst, int d0, int d1, int k, int transposed, cudaStream_t st);
// output convolution (C -> 1, k = 7) + tanh on the already snake'd channels-last tensor, bf16 (dac.cu)
bool final_conv_supported(int C);
int launch_final_conv_tanh(const void* x, const void* w, const void* bias, void* out, int C, int T, int B, cudaStream_t st);

enum { DK_PLAIN = 0, DK_CONV = 1, DK_CONVT = 2 };
struct DacTensor {
  int kind;
  int d0, d1, k;   // source dims (conv: co,ci,k; convT: ci,co,k; plain: numel,1,1)
  int64_t off;     // byte offset in blob
  int64_t numel;
  int64_t off_k;   // conv weights: second copy [tap][Cout][Cin] bf16 for the tcgen05 path (-1: none)
};

struct DacLayout {
  std::vector<DacTensor> t;
  int64_t codebooks, proj_w, proj_b;
  int64_t total;
  int es;
};

static inline int validate_dac(const ptts_dac_config& c) {
  PTTS_REQUIRE(c.dtype == PTTS_BF16 || c.dtype == PTTS_F32, "dac dtype must be bf16 or f32");
  PTTS_REQUIRE(c.n_blocks >= 1 && c.n_blocks <= 8, "dac n_blocks out of range");
  PTTS_REQUIRE(c.n_codebooks >= 1 && c.n_codebooks <= 32 && c.codebook_dim >= 1 && c.codebook_dim <= 16 &&
               c.n_codebooks * c.codebook_dim <= 256, "dac codebook shape unsupported");
  PTTS_REQUIRE((c.decoder_dim >> c.n_blocks) >= 1, "dac decoder_dim too small for n_blocks");
  for (int i = 0; i < c.n_blocks; i++) PTTS_REQUIRE(c.strides[i] >= 1 && c.strides[i] % 2 == 0 && c.strides[i] <= 32, "dac stride %d must be even and <= 32", c.strides[i]);
  return PTTS_OK;
}

static inline DacLayout make_dac_layout(const ptts_dac_config& c) {
  DacLayout L;
  L.es = dtype_size(c.dtype);
  int64_t o = 0;
  auto add = [&](int kind, int d0, int d1, int k) {
    DacTensor t{kind, d0, d1, k, o, (int64_t)d0 * d1 * k, -1};
    o = align_up(o + t.numel * L.es, 256);
    if (kind != DK_PLAIN && c.dtype == PTTS_BF16) { t.off_k = o; o = align_up(o + t.numel * 2, 1024); }
    L.t.push_back(t);
  };
  const int K = c.n_codebooks, D = c.codebook_dim, Z = c.latent_dim;
  // from_codes tensors are laid out as three contiguous arrays; ids interleave per codebook
  L.codebooks = 0;
  L.proj_w = align_up((int64_t)K * c.codebook_size * D * L.es, 256);
  L.proj_b = L.proj_w + align_up((int64_t)K * Z * D * L.es, 256);
  o = L.proj_b + align_up((int64_t)K * Z * L.es, 256);
  for (int k = 0; k < K; k++) {
    L.t.push_back({DK_PLAIN, c.codebook_size * D, 1, 1, L.codebooks + (int64_t)k * c.codebook_size * D * L.es, (int64_t)c.codebook_size * D, -1});
    L.t.push_back({DK_PLAIN, Z * D, 1, 1, L.proj_w + (int64_t)k * Z * D * L.es, (int64_t)Z * D, -1});
    L.t.push_back({DK_PLAIN, Z, 1, 1, L.proj_b + (int64_t)k * Z * L.es, (int64_t)Z, -1});
  }
  const int C = c.decoder_dim;
  add(DK_CONV, C, Z, 7); add(DK_PLAIN, C, 1, 1);
  for (int bi = 0; bi < c.n_blocks; bi++) {
    const int cin = C >> bi, cout = C >> (bi + 1), s = c.strides[bi];
    add(DK_PLAIN, cin, 1, 1);
    add(DK_CONVT, cin, cout, 2 * s); add(DK_PLAIN, cout, 1, 1);
    for (int r = 0; r < 3; r++) {
      add(DK_PLAIN, cout, 1, 1);
      add(DK_CONV, cout, cout, 7); add(DK_PLAIN, cout, 1, 1);
      add(DK_PLAIN, cout, 1, 1);
      add(DK_CONV, cout, cout, 1); add(DK_PLAIN, cout, 1, 1);
    }
  }
  const int cl = C >> c.n_blocks;
  add(DK_PLAIN, cl, 1, 1);
  add(DK_CONV, 1, cl, 7); add(DK_PLAIN, 1, 1, 1);
  L.total = o;
  return L;
}

static inline int dac_hop(const ptts_dac_config& c) {
  int h = 1;
  for (int i = 0; i < c.n_blocks; i++) h *= c.strides[i];
  return h;
}
// elements per (batch, code frame) of the largest activation
static inline int64_t dac_max_act_per_frame(const ptts_dac_config& c) {
  int64_t m = c.latent_dim > c.decoder_dim ? c.latent_dim : c.decoder_dim;
  int64_t up = 1;
  for (int i = 0; i < c.n_blocks; i++) {
    up *= c.strides[i];
    int64_t e = up * (c.decoder_dim >> (i + 1));
    if (e > m) m = e;
  }
  return m;
}

// ---- encoder (voice prompt): blob layout and tensor table -------------------------------------------------------------
// Tensor ids, in network order (dac_wrapper.py::_dac_encoder_tensor_list is the same table with state-dict keys):
//   conv1.{weight,bias}
//   per block: res_unit{1,2,3}.{snake1.alpha, conv1.weight, conv1.bias, snake2.alpha, conv2.weight, conv2.bias},
//              snake1.alpha, conv1.{weight,bias}                                   (21 tensors)
//   snake1.alpha, conv2.{weight,bias}
//   per codebook: in_proj.{weight,bias}, codebook.weight, out_proj.{weight,bias}   (5 tensors)
// The quantizer tensors live in five contiguous [K][...] arrays (plus the normalised codebooks) so that the RVQ kernel
// indexes them by codebook.
struct DacEncLayout {
  std::vector<DacTensor> t;
  int64_t in_w, in_b, codebooks, cb_norm, out_w, out_b;   // [K][D][Z], [K][D], [K][cs][D], [K][cs][D], [K][Z][D], [K][Z]
  int first_q;                                            // id of quantizer 0's in_proj.weight
  int64_t total;
  int es;
};

static inline int validate_dac_encoder(const ptts_dac_encoder_config& c) {
  PTTS_REQUIRE(c.dtype == PTTS_BF16 || c.dtype == PTTS_F32, "dac encoder dtype must be bf16 or f32");
  PTTS_REQUIRE(c.n_blocks >= 1 && c.n_blocks <= 8, "dac encoder n_blocks out of range");
  PTTS_REQUIRE(c.encoder_dim >= 1 && ((int64_t)c.encoder_dim << c.n_blocks) <= 4096, "dac encoder_dim out of range");
  for (int i = 0; i < c.n_blocks; i++) PTTS_REQUIRE(c.strides[i] >= 2 && c.strides[i] % 2 == 0 && c.strides[i] <= 32, "dac encoder stride %d must be even and in [2, 32]", c.strides[i]);
  PTTS_REQUIRE(c.latent_dim >= 1 && c.latent_dim <= 2048, "dac encoder latent_dim out of range");
  PTTS_REQUIRE(c.n_codebooks >= 1 && c.n_codebooks <= 32 && c.codebook_dim >= 1 && c.codebook_dim <= 16 && c.codebook_size >= 1,
               "dac encoder codebook shape unsupported");
  return PTTS_OK;
}

static inline DacEncLayout make_dac_encoder_layout(const ptts_dac_encoder_config& c) {
  DacEncLayout L;
  L.es = dtype_size(c.dtype);
  int64_t o = 0;
  // tc: also a [tap][Cout][Cin] bf16 copy for the tcgen05 convolutions (not for conv1, Cin = 1)
  auto add = [&](int kind, int d0, int d1, int k, bool tc) {
    DacTensor t{kind, d0, d1, k, o, (int64_t)d0 * d1 * k, -1};
    o = align_up(o + t.numel * L.es, 256);
    if (tc && c.dtype == PTTS_BF16) { t.off_k = o; o = align_up(o + t.numel * 2, 1024); }
    L.t.push_back(t);
  };
  const int D = c.encoder_dim;
  add(DK_CONV, D, 1, 7, false); add(DK_PLAIN, D, 1, 1, false);
  for (int bi = 0; bi < c.n_blocks; bi++) {
    const int ch = D << bi, s = c.strides[bi];
    for (int r = 0; r < 3; r++) {
      add(DK_PLAIN, ch, 1, 1, false);
      add(DK_CONV, ch, ch, 7, true); add(DK_PLAIN, ch, 1, 1, false);
      add(DK_PLAIN, ch, 1, 1, false);
      add(DK_CONV, ch, ch, 1, true); add(DK_PLAIN, ch, 1, 1, false);
    }
    add(DK_PLAIN, ch, 1, 1, false);
    add(DK_CONV, 2 * ch, ch, 2 * s, true); add(DK_PLAIN, 2 * ch, 1, 1, false);
  }
  const int dm = D << c.n_blocks, Z = c.latent_dim, K = c.n_codebooks, Dc = c.codebook_dim, cs = c.codebook_size;
  add(DK_PLAIN, dm, 1, 1, false);
  add(DK_CONV, Z, dm, 3, true); add(DK_PLAIN, Z, 1, 1, false);
  L.in_w = o;                 o = align_up(o + (int64_t)K * Dc * Z * L.es, 256);
  L.in_b = o;                 o = align_up(o + (int64_t)K * Dc * L.es, 256);
  L.codebooks = o;            o = align_up(o + (int64_t)K * cs * Dc * L.es, 256);
  L.cb_norm = o;              o = align_up(o + (int64_t)K * cs * Dc * L.es, 256);
  L.out_w = o;                o = align_up(o + (int64_t)K * Z * Dc * L.es, 256);
  L.out_b = o;                o = align_up(o + (int64_t)K * Z * L.es, 256);
  L.first_q = (int)L.t.size();
  for (int k = 0; k < K; k++) {
    L.t.push_back({DK_PLAIN, Dc * Z, 1, 1, L.in_w + (int64_t)k * Dc * Z * L.es, (int64_t)Dc * Z, -1});
    L.t.push_back({DK_PLAIN, Dc, 1, 1, L.in_b + (int64_t)k * Dc * L.es, (int64_t)Dc, -1});
    L.t.push_back({DK_PLAIN, cs * Dc, 1, 1, L.codebooks + (int64_t)k * cs * Dc * L.es, (int64_t)cs * Dc, -1});
    L.t.push_back({DK_PLAIN, Z * Dc, 1, 1, L.out_w + (int64_t)k * Z * Dc * L.es, (int64_t)Z * Dc, -1});
    L.t.push_back({DK_PLAIN, Z, 1, 1, L.out_b + (int64_t)k * Z * L.es, (int64_t)Z, -1});
  }
  L.total = o;
  return L;
}

static inline int64_t dac_encoder_hop(const ptts_dac_encoder_config& c) {
  int64_t h = 1;
  for (int i = 0; i < c.n_blocks; i++) h *= c.strides[i];
  return h;
}
// encoder (dac_enc.cu)
int normalize_codebook(const void* codebook, void* out, int cs, int D, int dtype, cudaStream_t st);
int64_t dac_encoder_workspace(const ptts_dac_encoder_config& c, int B, int64_t n);   // n: samples per utterance, multiple of the hop
int dac_encode(const ptts_dac_encoder_config& c, const char* blob, char* ws, int64_t ws_bytes, const void* audio, int B, int64_t n,
               int n_q, int64_t* codes, void* z, cudaStream_t st);

}  // namespace ptts
