// sample_core.cuh -- one row of logits -> next token (shared by sample_kernel and the fused step kernel).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace ptts {

__device__ __forceinline__ uint32_t fkey(float f) {  // order-preserving float -> uint
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  c[0] = hi1 ^ c[1] ^ k0; c[1] = lo1; c[2] = hi0 ^ c[3] ^ k1; c[3] = lo0;
}
__device__ __forceinline__ float philox_uniform(uint64_t seed, uint32_t row, uint32_t col) {
  uint32_t c[4] = {row, col, 0x5054u, 0x5453u};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int i = 0; i < 10; i++) { philox_round(c, k0, k1); k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
  return (float)(c[0] >> 8) * (1.0f / 16777216.0f);  // [0, 1)
}


// Processes up to R rows (row0, row0 + stride, ...; those >= n_rows are skipped) with ONE CTA of SMP_THREADS threads (element i of a
// row lives on thread i % 256, slot i / 256): the bitwise top-k / top-p searches, the softmax sums and the inverse-CDF draw are
// CTA-wide reductions / scans with a fixed order (lanes by butterfly, then warps 0..7), so results are bit-reproducible and identical
// between sample_kernel (R = 1) and the fused step kernels (both run exactly this code; per row the arithmetic does not depend on R).
// The R rows share every CTA barrier: a row costs ~9 us of mostly latency (two dependent L2 loads up front, 32 barrier-separated
// search iterations, 10 more for the draw, three dependent global accesses at the end), and the step kernel's 288 rows over 128 CTAs
// took three such rounds back to back (27 us per token); three rows per pass take little longer than one.
// One warp per row left 75 % of the fused kernel's warps idle for 33 us per token and held 72 live values per lane.
// Every thread of the CTA must call it (it contains __syncthreads()).
constexpr int SMP_WARPS = 8;
constexpr int SMP_THREADS = SMP_WARPS * 32;

constexpr int SMP_MAX_ROWS = 3;
struct SmpScratch {
  float f[2][SMP_MAX_ROWS][SMP_WARPS];
  int i[2][SMP_MAX_ROWS][SMP_WARPS];
  int z[2][SMP_MAX_ROWS][SMP_WARPS];
};
__device__ __forceinline__ SmpScratch& smp_scratch() {
  __shared__ SmpScratch sc;
  return sc;
}

template <int ITEMS, int R>
__device__ __forceinline__ void sample_rows_cta(const SampleArgs& p, const ptts_gen_params& g, const int64_t* __restrict__ forced,
                                                int row0, int stride, int n_rows, int cur_len) {
  static_assert(R >= 1 && R <= SMP_MAX_ROWS, "rows per pass");
  SmpScratch& sc = smp_scratch();   // one static buffer for every instantiation inlined into a kernel
  float (&s_f)[2][SMP_MAX_ROWS][SMP_WARPS] = sc.f;
  int (&s_i)[2][SMP_MAX_ROWS][SMP_WARPS] = sc.i;
  int (&s_z)[2][SMP_MAX_ROWS][SMP_WARPS] = sc.z;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int buf = 0;  // reductions alternate between two scratch rows: a warp may enter the next reduction while others still read this one
  auto cta_sum_i = [&](int (&v)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) {
      const int w = __reduce_add_sync(0xffffffffu, v[r]);
      if (lane == 0) s_i[buf][r][warp] = w;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; r++) {
      int a = 0;
#pragma unroll
      for (int w = 0; w < SMP_WARPS; w++) a += s_i[buf][r][w];
      v[r] = a;
    }
    buf ^= 1;
  };
  auto cta_sum_f = [&](float (&v)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) {
      const float w = warp_sum(v[r]);
      if (lane == 0) s_f[buf][r][warp] = w;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; r++) {
      float a = 0.f;
#pragma unroll
      for (int w = 0; w < SMP_WARPS; w++) a += s_f[buf][r][w];
      v[r] = a;
    }
    buf ^= 1;
  };
  auto cta_max_f = [&](float (&v)[R]) {
#pragma unroll
    for (int r = 0; r < R; r++) {
      const float w = warp_max(v[r]);
      if (lane == 0) s_f[buf][r][warp] = w;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; r++) {
      float a = s_f[buf][r][0];
#pragma unroll
      for (int w = 1; w < SMP_WARPS; w++) a = fmaxf(a, s_f[buf][r][w]);
      v[r] = a;
    }
    buf ^= 1;
  };

  int row[R];
  bool valid[R];
  float v[R][ITEMS];
#pragma unroll
  for (int r = 0; r < R; r++) {
    row[r] = row0 + r * stride;
    valid[r] = row[r] < n_rows;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      const int i = tid + SMP_THREADS * j;
      v[r][j] = (valid[r] && i < p.V) ? __ldcg(p.logits + (size_t)row[r] * p.V + i) : -INFINITY;  // written by other CTAs of this launch: L2, not L1
    }
  }
  // the tail's inputs (thread r finishes row r): requested now, consumed after the draw
  int t_unf = 0, t_es = 0;
  if (tid < R && row0 + tid * stride < n_rows) { t_unf = p.unfinished[row0 + tid * stride]; t_es = p.eos_seen[row0 + tid * stride]; }
#pragma unroll
  for (int r = 0; r < R; r++) {
    const int b = row[r] / p.K, k = row[r] - b * p.K;
    bool mask_eos = false;
    // MinNewTokensLength: prompt_length_to_skip = 1 (the BOS column)
    if (cur_len - 1 < g.min_new_tokens) mask_eos = true;
    // ParlerTTSLogitsProcessor (stateful; state double-buffered on the column parity)
    if (valid[r]) {
      const int par = cur_len & 1;
      int fu = p.first_unf[par * p.B + b];
      // eos_seen[r] = 1 + column of row r's first EOS (0 = none).  The reference counts EOS over input_ids, i.e. columns
      // < cur_len (logits_processors.py:46): an EOS written by another CTA during THIS step (column cur_len) must not count,
      // so the test is on the column, not on a flag (rows of one batch item are sampled by different CTAs).
      const int es = __ldcg(p.eos_seen + fu);
      if (es > 0 && es <= cur_len && fu < b * p.K + p.K - 1) fu++;
      if (k == 0 && tid == 0) p.first_unf[(par ^ 1) * p.B + b] = fu;
      if (row[r] > fu) mask_eos = true;
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      const int i = tid + SMP_THREADS * j;
      if (mask_eos && i == p.eos) v[r][j] = -INFINITY;
      if (g.suppress_special && i >= g.codebook_size) v[r][j] = -INFINITY;
    }
  }
  int tok[R];
#pragma unroll
  for (int r = 0; r < R; r++) tok[r] = 0;
  if (g.do_sample) {
    if (g.temperature != 1.0f) {
#pragma unroll
      for (int r = 0; r < R; r++)
#pragma unroll
        for (int j = 0; j < ITEMS; j++) v[r][j] = v[r][j] / g.temperature;
    }
    if (g.top_k > 0) {
      const int kk = g.top_k < p.V ? g.top_k : p.V;
      uint32_t key[R][ITEMS];
      uint32_t th[R];
#pragma unroll
      for (int r = 0; r < R; r++) {
        th[r] = 0;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) key[r][j] = (tid + SMP_THREADS * j < p.V) ? fkey(v[r][j]) : 0u;   // 0 < every candidate
      }
      for (int bit = 31; bit >= 0; bit--) {  // bitwise binary search of the k-th largest key
        int cnt[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
          const uint32_t cand = th[r] | (1u << bit);
          cnt[r] = 0;
#pragma unroll
          for (int j = 0; j < ITEMS; j++) cnt[r] += (key[r][j] >= cand) ? 1 : 0;
        }
        cta_sum_i(cnt);
#pragma unroll
        for (int r = 0; r < R; r++)
          if (cnt[r] >= kk) th[r] |= (1u << bit);
      }
#pragma unroll
      for (int r = 0; r < R; r++)
#pragma unroll
        for (int j = 0; j < ITEMS; j++)
          if (fkey(v[r][j]) < th[r]) v[r][j] = -INFINITY;  // scores < kth largest
    }
    float m[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
      m[r] = -INFINITY;
#pragma unroll
      for (int j = 0; j < ITEMS; j++) m[r] = fmaxf(m[r], v[r][j]);
    }
    cta_max_f(m);
    float e[R][ITEMS];
    float s[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
      s[r] = 0.f;
#pragma unroll
      for (int j = 0; j < ITEMS; j++) { e[r][j] = expf(v[r][j] - m[r]); s[r] += e[r][j]; }
    }
    cta_sum_f(s);
    if (g.top_p < 1.0f) {
      // remove tokens whose ascending cumulative probability is <= 1 - top_p (the max is always kept)
      uint32_t th[R];
#pragma unroll
      for (int r = 0; r < R; r++) th[r] = 0;
      for (int bit = 31; bit >= 0; bit--) {
        float c[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
          const uint32_t cand = th[r] | (1u << bit);
          c[r] = 0.f;
#pragma unroll
          for (int j = 0; j < ITEMS; j++) c[r] += (fkey(v[r][j]) <= cand) ? e[r][j] : 0.f;
        }
        cta_sum_f(c);
#pragma unroll
        for (int r = 0; r < R; r++)
          if (c[r] <= (1.0f - g.top_p) * s[r]) th[r] |= (1u << bit);
      }
#pragma unroll
      for (int r = 0; r < R; r++) {
        const uint32_t kmax = fkey(m[r]);
        s[r] = 0.f;
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
          const uint32_t key = fkey(v[r][j]);
          if (key <= th[r] && key != kmax) { v[r][j] = -INFINITY; e[r][j] = 0.f; }
          s[r] += e[r][j];
        }
      }
      cta_sum_f(s);
    }
    // inverse-CDF draw in index order: CTA-wide inclusive scan per slot j (elements 256 j .. 256 j + 255)
    float target[R], carry[R];
    int found[R], last_nz[R];
#pragma unroll
    for (int r = 0; r < R; r++) {
      target[r] = philox_uniform(g.seed, (uint32_t)(row[r] + g.row_base), (uint32_t)cur_len) * s[r];
      carry[r] = 0.f; found[r] = -1; last_nz[r] = -1;
    }
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      float x[R];
#pragma unroll
      for (int r = 0; r < R; r++) {
        x[r] = e[r][j];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float y = __shfl_up_sync(0xffffffffu, x[r], o);
          if (lane >= o) x[r] += y;
        }
        if (lane == 31) s_f[buf][r][warp] = x[r];  // this warp's total
      }
      __syncthreads();
      float tot[R];
#pragma unroll
      for (int r = 0; r < R; r++) {
        float base = carry[r];
        tot[r] = carry[r];
#pragma unroll
        for (int w = 0; w < SMP_WARPS; w++) {
          const float tw = s_f[buf][r][w];
          if (w < warp) base += tw;
          tot[r] += tw;
        }
        const float cum = base + x[r];
        const unsigned hit = __ballot_sync(0xffffffffu, cum > target[r] && e[r][j] > 0.f);
        const unsigned nz = __ballot_sync(0xffffffffu, e[r][j] > 0.f);
        if (lane == 0) {
          s_i[buf][r][warp] = hit ? SMP_THREADS * j + 32 * warp + (__ffs(hit) - 1) : 0x7fffffff;
          s_z[buf][r][warp] = nz ? SMP_THREADS * j + 32 * warp + (31 - __clz(nz)) : -1;
        }
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < R; r++) {
        int first = 0x7fffffff, lastz = -1;
#pragma unroll
        for (int w = 0; w < SMP_WARPS; w++) { first = min(first, s_i[buf][r][w]); lastz = max(lastz, s_z[buf][r][w]); }
        if (found[r] < 0 && first != 0x7fffffff) found[r] = first;
        if (lastz >= 0) last_nz[r] = lastz;
        carry[r] = tot[r];
      }
      buf ^= 1;
    }
#pragma unroll
    for (int r = 0; r < R; r++) tok[r] = found[r] >= 0 ? found[r] : last_nz[r];
  } else {
    // argmax, smallest index on ties
#pragma unroll
    for (int r = 0; r < R; r++) {
      float m = -INFINITY;
      int mi = 0x7fffffff;
#pragma unroll
      for (int j = 0; j < ITEMS; j++) {
        const int i = tid + SMP_THREADS * j;
        if (i < p.V && (v[r][j] > m || (v[r][j] == m && i < mi))) { m = v[r][j]; mi = i; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, m, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
      }
      if (lane == 0) { s_f[buf][r][warp] = m; s_i[buf][r][warp] = mi; }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < R; r++) {
      float m = s_f[buf][r][0];
      int mi = s_i[buf][r][0];
#pragma unroll
      for (int w = 1; w < SMP_WARPS; w++) {
        const float om = s_f[buf][r][w];
        const int oi = s_i[buf][r][w];
        if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
      }
      tok[r] = mi;
    }
    buf ^= 1;
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    if (!valid[r]) continue;
#pragma unroll
    for (int j = 0; j < ITEMS; j++) {
      const int i = tid + SMP_THREADS * j;
      if (i < p.V) p.scores[(size_t)row[r] * p.V + i] = v[r][j];
    }
  }
  // thread r finishes row r (the rows are independent: each owns its entries of every array below)
  int my_tok = 0, my_row = 0;
  bool my_valid = false;
#pragma unroll
  for (int r = 0; r < R; r++)
    if (tid == r) { my_tok = tok[r]; my_row = row[r]; my_valid = valid[r]; }
  if (tid < R && my_valid) {
    const int b = my_row / p.K, k = my_row - b * p.K;
    int t = my_tok;
    if (forced != nullptr && forced[my_row] >= 0) t = (int)forced[my_row];   // negative: draw this row (ptts_sample)
    if (!t_unf) t = p.pad;  // next_tokens * unfinished + pad * (1 - unfinished)
    p.raw_ids[(size_t)my_row * p.raw_ld + cur_len] = t;
    if (t == p.eos && t_es == 0) p.eos_seen[my_row] = cur_len + 1;
    const int new_len = cur_len + 1;
    const int done = (t == p.eos) || (new_len >= g.max_length);
    const int still_unfinished = t_unf && !done;
    p.unfinished[my_row] = still_unfinished;
    // delay-pattern override of the NEXT model input (column `cur_len`), build_delay_pattern_mask :252-261
    int nxt = t;
    if (g.max_length >= 2 * p.K - 1) {
      const bool is_bos = cur_len <= k;
      const bool is_pad = (cur_len - k) >= (g.max_length - p.K + 1);
      if (is_bos || is_pad) nxt = (is_bos ? p.bos : 0) + (is_pad ? p.pad : 0);
    }
    p.cur_ids[my_row] = nxt;
    if (still_unfinished) atomicAdd(&p.ctrl->n_unfinished, 1);
  }
  __syncthreads();  // the scratch rows may be reused by the next pass of this CTA
}

template <int ITEMS>
__device__ __forceinline__ void sample_row_cta(const SampleArgs& p, const ptts_gen_params& g, const int64_t* __restrict__ forced,
                                               int row, int cur_len) {
  sample_rows_cta<ITEMS, 1>(p, g, forced, row, 0, row + 1, cur_len);
}

// all rows of the token over the CTAs of a fused step kernel: passes of up to three rows per CTA
template <int ITEMS>
__device__ __forceinline__ void sample_all_rows_cta(const SampleArgs& p, const ptts_gen_params& g, int cta, int n_ctas, int n_rows, int cur_len) {
  if (n_rows <= n_ctas) {
    if (cta < n_rows) sample_rows_cta<ITEMS, 1>(p, g, nullptr, cta, n_ctas, n_rows, cur_len);
  } else {
    for (int row0 = cta; row0 < n_rows; row0 += 3 * n_ctas) sample_rows_cta<ITEMS, 3>(p, g, nullptr, row0, n_ctas, n_rows, cur_len);
  }
}

}  // namespace ptts
