// attn_core.cuh -- one (batch row, kv head) attention item processed by a 128-thread group.
// Shared by attention_kernel (one CTA per item) and the fused step kernel (two items per CTA, named barriers).
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace ptts {

constexpr int ATT_THREADS = 128;
constexpr int ATT_WARPS = 4;
constexpr int HD = PTTS_HEAD_DIM;

template <typename Sync>
__device__ __forceinline__ float block_reduce(float v, float* sh, bool is_max, int tid, Sync sync) {
  const int warp = tid >> 5, lane = tid & 31;
  v = is_max ? warp_max(v) : warp_sum(v);
  sync();
  if (lane == 0) sh[warp] = v;
  sync();
  float r = sh[0];
#pragma unroll
  for (int w = 1; w < ATT_WARPS; w++) r = is_max ? fmaxf(r, sh[w]) : r + sh[w];
  return r;
}

// RoPE on one 64-vector held as "element d per thread": out = x*cos + rotate_half(x)*sin with every
// intermediate rounded to the model dtype (apply_rotary_pos_emb, :416-436).
template <typename T>
__device__ __forceinline__ float rope_elem(float x, float x_pair, int d, const T* cos_row, const T* sin_row) {
  const float c = DT<T>::to_f(cos_row[d]), s = DT<T>::to_f(sin_row[d]);
  const float rot = (d < HD / 2) ? -x_pair : x_pair;
  return DT<T>::rnd(DT<T>::rnd(x * c) + DT<T>::rnd(rot * s));
}


// sm: [64] q | [4][64] partials | [8] scratch | [kv capacity] scores.  `tid` in [0,128); sync() = barrier of the group.
template <typename T, typename Sync>
__device__ __forceinline__ void attention_item(const AttnArgs& p, int b, int kvh, float* sm, int tid, Sync sync, int q_lo = 0, int q_hi = 1 << 30) {
  const T* __restrict__ rope_cos = reinterpret_cast<const T*>(p.rope_cos);
  const T* __restrict__ rope_sin = reinterpret_cast<const T*>(p.rope_sin);
  float* qs = sm;
  float* red = sm + HD;
  float* sh = red + ATT_WARPS * HD;
  float* sc = sh + 8;
  const int warp = tid >> 5, lane = tid & 31;
  const int rep = p.nh / p.nkv;
  int past = p.past_len;
  if (p.past_from_ctrl) past = p.prefix + p.ctrl->cur_len - 1;

  T* kc = reinterpret_cast<T*>(p.kcache) + (size_t)b * p.kv_b_stride + (size_t)kvh * p.kv_h_stride;
  T* vc = reinterpret_cast<T*>(p.vcache) + (size_t)b * p.kv_b_stride + (size_t)kvh * p.kv_h_stride;

  // ---- phase A: append the new K/V rows (self-attention only) ----
  if (!p.cross) {
    const int d = tid & 63;
    const bool is_v = tid >= 64;
    for (int j = 0; j < p.q_len && j < q_hi; j++) {   // (causal: positions >= q_hi are not read by this group)
      const size_t r = (size_t)b * p.q_len + j;
      const int pos = past + j;
      if (!is_v) {
        const T* src = reinterpret_cast<const T*>(p.knew) + r * p.ldkv + p.k_col0 + kvh * HD;
        float x = DT<T>::to_f(src[d]);
        if (p.rope) {
          const float xp = DT<T>::to_f(src[d < HD / 2 ? d + HD / 2 : d - HD / 2]);
          x = rope_elem<T>(x, xp, d, rope_cos + (size_t)pos * HD, rope_sin + (size_t)pos * HD);
        }
        kc[(size_t)pos * p.kv_t_stride + kv_swz(pos, d)] = DT<T>::from_f(x);
      } else {
        const T* src = reinterpret_cast<const T*>(p.vnew) + r * p.ldkv + p.v_col0 + kvh * HD;
        vc[(size_t)pos * p.kv_t_stride + kv_swz(pos, d)] = src[d];
      }
    }
    sync();  // this CTA is the only reader of the rows it just wrote
  }

  const int grp = lane >> 3;           // key group inside the warp (4 keys per warp per iteration)
  const int d0 = (lane & 7) * 8;       // this lane's 8 dims
  const int kslot = warp * 4 + grp;    // 0..15
  const int* km = p.key_mask ? p.key_mask + (size_t)b * p.mask_ld : nullptr;

  // [q_lo, q_hi): the query positions this group sweeps (the prefill kernel cuts the positions over blockIdx.z; every group appends
  // ALL new K/V rows itself above -- identical values, so the duplicate global writes are benign -- and reads only what it wrote)
  for (int j = q_lo; j < p.q_len && j < q_hi; j++) {
    const size_t r = (size_t)b * p.q_len + j;
    const int pos = past + j;
    const int T_keys = p.cross ? p.kv_len : pos + 1;
    for (int rr = 0; rr < rep; rr++) {
      const int h = kvh * rep + rr;
      sync();
      if (tid < HD) {
        const T* src = reinterpret_cast<const T*>(p.q) + r * p.ldq + p.q_col0 + h * HD;
        float x = DT<T>::to_f(src[tid]);
        if (p.rope) {
          const float xp = DT<T>::to_f(src[tid < HD / 2 ? tid + HD / 2 : tid - HD / 2]);
          x = rope_elem<T>(x, xp, tid, rope_cos + (size_t)pos * HD, rope_sin + (size_t)pos * HD);
        }
        qs[tid] = x;
      }
      sync();
      float qv[8];
#pragma unroll
      for (int e = 0; e < 8; e++) qv[e] = qs[d0 + e];

      // ---- scores ----
      float lmax = -INFINITY;
      for (int t0 = 0; t0 < T_keys; t0 += 64) {
        float kv[4][8];
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int t = t0 + u * 16 + kslot;
          ok[u] = t < T_keys;
          if (ok[u]) load8(kc + (size_t)t * p.kv_t_stride + kv_swz(t, d0), kv[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int t = t0 + u * 16 + kslot;
          float s = 0.f;
          if (ok[u]) {
#pragma unroll
            for (int e = 0; e < 8; e++) s = fmaf(qv[e], kv[u][e], s);
          }
          s += __shfl_xor_sync(0xffffffffu, s, 1);
          s += __shfl_xor_sync(0xffffffffu, s, 2);
          s += __shfl_xor_sync(0xffffffffu, s, 4);
          if (ok[u] && (lane & 7) == 0) {
            s *= p.scale;
            if (km != nullptr && t < p.mask_len && km[t] == 0) s = -INFINITY;
            sc[t] = s;
            lmax = fmaxf(lmax, s);
          }
        }
      }
      const float m = block_reduce(lmax, sh, true, tid, sync);  // (contains the barrier that publishes sc[])
      // ---- softmax numerators; fully-masked rows degrade to uniform attention (never consumed) ----
      float lsum = 0.f;
      for (int t = tid; t < T_keys; t += ATT_THREADS) {
        const float e = (m == -INFINITY) ? 1.0f : expf(sc[t] - m);
        sc[t] = e;
        lsum += e;
      }
      const float l = block_reduce(lsum, sh, false, tid, sync);
      // ---- P.V ----
      float acc[8];
#pragma unroll
      for (int e = 0; e < 8; e++) acc[e] = 0.f;
      for (int t0 = 0; t0 < T_keys; t0 += 64) {
        float vv[4][8];
        float pw[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int t = t0 + u * 16 + kslot;
          pw[u] = 0.f;
          if (t < T_keys) {
            load8(vc + (size_t)t * p.kv_t_stride + kv_swz(t, d0), vv[u]);
            pw[u] = DT<T>::rnd(sc[t]);
          } else {
#pragma unroll
            for (int e = 0; e < 8; e++) vv[u][e] = 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
          for (int e = 0; e < 8; e++) acc[e] = fmaf(pw[u], vv[u][e], acc[e]);
      }
#pragma unroll
      for (int e = 0; e < 8; e++) {
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
      }
      if (lane < 8) {
#pragma unroll
        for (int e = 0; e < 8; e++) red[warp * HD + d0 + e] = acc[e];
      }
      sync();
      if (tid < HD) {
        float o = red[tid] + red[HD + tid] + red[2 * HD + tid] + red[3 * HD + tid];
        o = o / l;
        reinterpret_cast<T*>(p.out)[r * p.ldo + h * HD + tid] = DT<T>::from_f(o);
      }
    }
  }
}

}  // namespace ptts

namespace ptts {

// ---- decode fast path (q_len == 1): ONE WARP per (batch row, kv head) item, TMA-staged K/V tiles ---------
// The cached K/V rows of the item stream through a per-warp 2-stage shared-memory ring filled by the TMA
// engine (cp.async.bulk + mbarrier; CH keys = CH*128 B of K and of V per stage), so HBM/L2 latency is hidden
// without holding loads in registers.  Scores, online softmax (running max / sum, fp32) and P.V are fused in
// one sweep: 8 lanes x 16 B cover one key row (conflict-free LDS.128), 4 keys per warp instruction; the
// probabilities are rounded to the model dtype before P.V like torch's flash kernels.  The step's own K/V row
// is taken from shared memory (it is also written to the cache for later steps), so no global read-after-write.
// No block-level barrier anywhere: used by attention_decode_kernel (8 items per CTA) and by the fused step
// kernel -- both run exactly this code, hence bit-identical results.
__device__ __forceinline__ uint32_t att_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// keys per ring stage
template <typename T> struct AttChunk { static constexpr int CH = 32; };
template <> struct AttChunk<float> { static constexpr int CH = 16; };

// bytes of shared memory one warp needs
template <typename T>
__host__ __device__ constexpr int attn_decode_smem_per_warp() {
  return 2 * 2 * AttChunk<T>::CH * HD * (int)sizeof(T) + (3 * HD) * (int)sizeof(float);
}

template <typename T>
__device__ __forceinline__ void attention_decode_item_warp(const AttnArgs& p, int b, int kvh, int pos, unsigned char* sm_warp, uint64_t* bars,
                                                           int lane, uint32_t& parity, int part = 0, int nparts = 1, float* xch = nullptr,
                                                           int pair_bar = 0) {
  // part / nparts: the item's cached keys are split between `nparts` warps (chunk c belongs to warp c % nparts);
  // partial (max, sum, accumulator) triples are merged through `xch` with a 64-thread named barrier `pair_bar`.
  constexpr int CH = AttChunk<T>::CH;
  constexpr int STAGE_ELEMS = CH * HD;  // per K (or V) stage
  T* kst = reinterpret_cast<T*>(sm_warp);                   // [2][CH][64]
  T* vst = kst + 2 * STAGE_ELEMS;                            // [2][CH][64]
  float* qs = reinterpret_cast<float*>(vst + 2 * STAGE_ELEMS);  // [64] query
  float* kn = qs + HD;                                       // [64] this step's key   (self only)
  float* vn = kn + HD;                                       // [64] this step's value (self only)
  // bars[2]: this warp's mbarriers, initialised ONCE per kernel in memory that is never aliased (re-initialising
  // a live mbarrier is undefined behaviour); `parity` carries their phase across items and phases.
  const T* __restrict__ rope_cos = reinterpret_cast<const T*>(p.rope_cos) + (size_t)pos * HD;
  const T* __restrict__ rope_sin = reinterpret_cast<const T*>(p.rope_sin) + (size_t)pos * HD;
  const int rep = p.nh / p.nkv;
  T* kc = reinterpret_cast<T*>(p.kcache) + (size_t)b * p.kv_b_stride + (size_t)kvh * p.kv_h_stride;
  T* vc = reinterpret_cast<T*>(p.vcache) + (size_t)b * p.kv_b_stride + (size_t)kvh * p.kv_h_stride;
  const int lo = lane, hi = lane + HD / 2;
  const int n_cached = p.cross ? p.kv_len : pos;  // keys that come from the cache
  const int n_chunks_all = (n_cached + CH - 1) / CH;
  const int n_chunks = (n_chunks_all > part) ? (n_chunks_all - part + nparts - 1) / nparts : 0;  // chunks of THIS warp

  auto issue = [&](int i) {  // TMA: this warp's i-th chunk -> stage i&1
    const int st = i & 1;
    const int t0 = (part + nparts * i) * CH;
    const int n = (n_cached - t0 < CH) ? (n_cached - t0) : CH;
    const uint32_t bar = att_smem_u32(&bars[st]);
    if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(2 * n * HD * sizeof(T))) : "memory");
    __syncwarp();
    if (lane < 2) {  // one bulk copy for the K rows, one for the V rows (rows of an item are contiguous)
      const T* src = (lane == 0 ? kc : vc) + (size_t)t0 * HD;
      T* dst = (lane == 0 ? kst : vst) + st * STAGE_ELEMS;
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(att_smem_u32(dst)), "l"(src), "r"((uint32_t)(n * HD * sizeof(T))), "r"(bar) : "memory");
    }
  };
  auto wait_stage = [&](int st) {
    const uint32_t bar = att_smem_u32(&bars[st]);
    const uint32_t par = (parity >> st) & 1u;
    uint32_t ok, spins = 0;
    do {
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(par) : "memory");
      if (!ok && ++spins > (1u << 16)) { if (lane == 0) printf("ptts: attention KV mbarrier timeout (cta %d b %d kvh %d stage %d cross %d n_cached %d chunks %d par %u)\n", (int)blockIdx.x, b, kvh, st, p.cross, n_cached, n_chunks, parity); __trap(); }
    } while (!ok);
    parity ^= (1u << st);
  };

  // all lanes are past their shared-memory reads of the previous item: the ring may be refilled
  __syncwarp();
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (n_chunks > 0) issue(0);
  if (n_chunks > 1) issue(1);

  // the first query head's elements are requested before the K/V append below (its stores would otherwise order the loads
  // behind a second L2 round trip)
  const T* q_first = reinterpret_cast<const T*>(p.q) + (size_t)b * p.ldq + p.q_col0 + (size_t)(kvh * rep) * HD;
  const float qf0 = DT<T>::to_f(q_first[lo]), qf1 = DT<T>::to_f(q_first[hi]);
  if (!p.cross && part == 0) {  // this step's K (rotary applied) and V: to the cache (for later steps) and to shared memory (for now)
    const T* ksrc = reinterpret_cast<const T*>(p.knew) + (size_t)b * p.ldkv + p.k_col0 + kvh * HD;
    const T* vsrc = reinterpret_cast<const T*>(p.vnew) + (size_t)b * p.ldkv + p.v_col0 + kvh * HD;
    float x0 = DT<T>::to_f(ksrc[lo]), x1 = DT<T>::to_f(ksrc[hi]);
    if (p.rope) {
      const float y0 = rope_elem<T>(x0, x1, lo, rope_cos, rope_sin);
      const float y1 = rope_elem<T>(x1, x0, hi, rope_cos, rope_sin);
      x0 = y0; x1 = y1;
    }
    const T v0 = vsrc[lo], v1 = vsrc[hi];
    kc[(size_t)pos * p.kv_t_stride + kv_swz(pos, lo)] = DT<T>::from_f(x0);
    kc[(size_t)pos * p.kv_t_stride + kv_swz(pos, hi)] = DT<T>::from_f(x1);
    vc[(size_t)pos * p.kv_t_stride + kv_swz(pos, lo)] = v0;
    vc[(size_t)pos * p.kv_t_stride + kv_swz(pos, hi)] = v1;
    kn[lo] = DT<T>::rnd(x0); kn[hi] = DT<T>::rnd(x1);
    vn[lo] = DT<T>::to_f(v0); vn[hi] = DT<T>::to_f(v1);
  }
  const int grp = lane >> 3, d0 = (lane & 7) * 8;
  const int* km = p.key_mask ? p.key_mask + (size_t)b * p.mask_ld : nullptr;

  for (int rr = 0; rr < rep; rr++) {
    const int h = kvh * rep + rr;
    {
      const T* qsrc = reinterpret_cast<const T*>(p.q) + (size_t)b * p.ldq + p.q_col0 + h * HD;
      float x0 = (rr == 0) ? qf0 : DT<T>::to_f(qsrc[lo]), x1 = (rr == 0) ? qf1 : DT<T>::to_f(qsrc[hi]);
      if (p.rope) {
        const float y0 = rope_elem<T>(x0, x1, lo, rope_cos, rope_sin);
        const float y1 = rope_elem<T>(x1, x0, hi, rope_cos, rope_sin);
        x0 = y0; x1 = y1;
      }
      __syncwarp();
      qs[lo] = x0; qs[hi] = x1;
      __syncwarp();
    }
    float qv[8];
#pragma unroll
    for (int e = 0; e < 8; e++) qv[e] = qs[d0 + e];
    float m_run = -INFINITY, l_run = 0.f;
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; e++) acc[e] = 0.f;

    // One block of n <= CH keys whose K/V rows sit in shared memory at kb/vb (row stride 64); bit r of `mword` = key r is
    // attendable.  Branch-free: rows >= n are clamped to row n-1 (valid data) and get probability 0 through a -inf score,
    // so the 8 per-key chains of a lane group are independent and interleave (a divergent `if` per key serialised them).
    auto process = [&](const T* kb, const T* vb, uint32_t mword, int n) {
      constexpr int PER = CH / 4;  // keys per 8-lane group
      float sloc[PER];
#pragma unroll
      for (int u = 0; u < PER; u++) {
        const int r = u * 4 + grp, rc = r < n ? r : n - 1;
        float kf[8];
        load8(kb + rc * HD + kv_swz(rc, d0), kf);   // (stages start at multiples of 8 keys: t & 7 == rc & 7)
        float s = 0.f;
#pragma unroll
        for (int e = 0; e < 8; e++) s = fmaf(qv[e], kf[e], s);
        sloc[u] = s;
      }
#pragma unroll
      for (int u = 0; u < PER; u++) sloc[u] += __shfl_xor_sync(0xffffffffu, sloc[u], 1);
#pragma unroll
      for (int u = 0; u < PER; u++) sloc[u] += __shfl_xor_sync(0xffffffffu, sloc[u], 2);
#pragma unroll
      for (int u = 0; u < PER; u++) sloc[u] += __shfl_xor_sync(0xffffffffu, sloc[u], 4);
      float cmax = -INFINITY;
#pragma unroll
      for (int u = 0; u < PER; u++) {
        const int r = u * 4 + grp;
        sloc[u] = (r < n && ((mword >> r) & 1u)) ? sloc[u] * p.scale : -INFINITY;
        cmax = fmaxf(cmax, sloc[u]);
      }
      cmax = warp_max(cmax);
      const float m_new = fmaxf(m_run, cmax);
      if (m_new == -INFINITY) return;  // every key so far is masked: nothing to accumulate (warp-uniform)
      const float corr = (m_run == -INFINITY) ? 0.f : expf(m_run - m_new);
      l_run *= corr;
#pragma unroll
      for (int e = 0; e < 8; e++) acc[e] *= corr;
      float lsum = 0.f;
#pragma unroll
      for (int u = 0; u < PER; u++) {
        const int r = u * 4 + grp, rc = r < n ? r : n - 1;
        const float pe = expf(sloc[u] - m_new);  // exactly 0 for a masked / out-of-range key
        lsum += pe;  // identical on the 8 lanes of the group; counted once below
        const float pw = DT<T>::rnd(pe);
        float vf[8];
        load8(vb + rc * HD + kv_swz(rc, d0), vf);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[e] = fmaf(pw, vf[e], acc[e]);
      }
      // sum of probabilities over the 4 groups (each group's 8 lanes hold the same value)
      lsum += __shfl_xor_sync(0xffffffffu, lsum, 8);
      lsum += __shfl_xor_sync(0xffffffffu, lsum, 16);
      l_run += lsum;
      m_run = m_new;
    };
    // attendable-key bits of the chunk starting at key t0 (the loads are issued before the wait on the chunk's TMA stage)
    auto mask_bits = [&](int t0) -> int {
      const int t = t0 + lane;
      return (km != nullptr && lane < CH && t < p.mask_len && t < n_cached) ? km[t] : 1;
    };

    if (rr > 0) {  // GQA: further query heads re-stream the same cache rows
      __syncwarp();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      if (n_chunks > 0) issue(0);
      if (n_chunks > 1) issue(1);
    }
    for (int c = 0; c < n_chunks; c++) {
      const int st = c & 1;
      const int t0 = (part + nparts * c) * CH;
      const int n = (n_cached - t0 < CH) ? (n_cached - t0) : CH;
      const int mk = mask_bits(t0);
      wait_stage(st);
      process(kst + st * STAGE_ELEMS, vst + st * STAGE_ELEMS, __ballot_sync(0xffffffffu, mk != 0), n);
      if (c + 2 < n_chunks) {
        __syncwarp();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        issue(c + 2);
      }
    }
    if (!p.cross && part == 0) {  // the step's own key (position `pos`), held in shared memory as fp32
      __syncwarp();
      float s = 0.f;
      if (grp == 0) {
#pragma unroll
        for (int e = 0; e < 8; e++) s = fmaf(qv[e], kn[d0 + e], s);
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      s = __shfl_sync(0xffffffffu, s, 0) * p.scale;
      if (km != nullptr && pos < p.mask_len && km[pos] == 0) s = -INFINITY;
      const float m_new = fmaxf(m_run, s);
      if (m_new != -INFINITY) {
        const float corr = (m_run == -INFINITY) ? 0.f : expf(m_run - m_new);
        const float pe = (s == -INFINITY) ? 0.f : expf(s - m_new);
        const float pw = DT<T>::rnd(pe);
        l_run = l_run * corr + pe;
#pragma unroll
        for (int e = 0; e < 8; e++) acc[e] = acc[e] * corr + ((grp == 0) ? pw * vn[d0 + e] : 0.f);
        m_run = m_new;
      }
    }
#pragma unroll
    for (int e = 0; e < 8; e++) {
      acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
      acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
    }
    if (nparts == 2) {  // merge the two warps' partial softmax states (fixed order: part 0 then part 1)
      if (part == 1) {
        if (lane < 8) {
#pragma unroll
          for (int e = 0; e < 8; e++) xch[d0 + e] = acc[e];
        }
        if (lane == 0) { xch[HD] = m_run; xch[HD + 1] = l_run; }
      }
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
      if (part == 0) {
        const float m1 = xch[HD], l1 = xch[HD + 1];
        const float mm = fmaxf(m_run, m1);
        const float c0 = (m_run == -INFINITY) ? 0.f : expf(m_run - mm);
        const float c1 = (m1 == -INFINITY) ? 0.f : expf(m1 - mm);
        l_run = l_run * c0 + l1 * c1;
        if (lane < 8) {
#pragma unroll
          for (int e = 0; e < 8; e++) acc[e] = acc[e] * c0 + xch[d0 + e] * c1;
        }
      }
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
    }
    if (lane < 8 && part == 0) {
      float o[8];
      const float inv = (l_run > 0.f) ? 1.0f / l_run : 0.f;  // fully masked row -> zeros (never consumed)
#pragma unroll
      for (int e = 0; e < 8; e++) o[e] = acc[e] * inv;
      store8(reinterpret_cast<T*>(p.out) + (size_t)b * p.ldo + h * HD + d0, o);
    }
  }
}

// ---- decode attention on the tensor cores (bf16, MHA: one query head per K/V head) -----------------------------------------
// Same contract, ring and merge protocol as attention_decode_item_warp, but 16 keys cost 16 mma.m16n8k16 instead of
// ~250 scalar instructions (the SIMT sweep measured 37 ns per key per warp, latency-bound: profiles/r02_step2_phases.md):
//   S = q K^T : A = the query in row 0 of an m16 x k16 fragment (4 k-steps over the 64 dims; rows 1..15 are zero),
//               B = K rows straight from the staged tile with ldmatrix (keys are the n dimension) -> 2 n-tiles x 4 k-steps = 8 MMAs;
//   O += P V  : A = the probabilities, which already sit in the A-fragment registers after the S MMAs (row 0 of the C fragment
//               of n-tile 0 / 1 = columns 0-7 / 8-15 of the A fragment), B = V rows with ldmatrix.trans -> 8 n-tiles = 8 MMAs.
// The K/V rows are stored swizzled (kv_swz, common.cuh), so the contiguous bulk copy of a stage is a conflict-free ldmatrix tile.
// Only lanes 0..3 (fragment row 0) carry softmax state; fp32 scores / running max / sum, probabilities rounded to bf16 before
// P V like the SIMT path and torch's flash kernels.
__device__ __forceinline__ void att_ldsm4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void att_ldsm4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void att_mma(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t att_pack(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

__device__ __forceinline__ float att_ex2(float x) {   // 2^x, 2 ulp; ex2(-inf) = +0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// one K or V stage: global -> shared memory; `stream`: evict-first in L2 (the rows are read once per token; step2.cu bulk_g2s_stream)
__device__ __forceinline__ void att_bulk_kv(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, bool stream) {
  if (stream) {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
  } else {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
  }
}

constexpr int ATT_TC_CH = 32;   // keys per ring stage: one softmax / rescale chain per 32 keys (the chain, not the MMAs, bounds a stage)
constexpr int ATT_TC_STAGE_BYTES = 2 * ATT_TC_CH * HD * 2;   // one stage: K rows then V rows (8 KB)

// What the tensor-core decode attention needs to know about ONE (row, head) item -- resolved pointers instead of the generic AttnArgs,
// so that the step kernel can build it from a handful of per-warp constants (the AttnArgs route cost ~500 instructions per phase
// between the exchange send and its wait: profiles/r02_step2_phases.md).  K/V cache rows are HD wide (kv_t_stride = HD).
struct TcItem {
  const bf16* q;        // [HD] this step's query (shared or global memory)
  const bf16* knew;     // [HD] this step's key / value (self-attention; nullptr for cross-attention)
  const bf16* vnew;
  bf16* kc;             // the item's K rows [capacity][HD] (swizzled, common.cuh kv_swz) and V rows
  bf16* vc;
  const int* km;        // key mask of the row (nullptr: none), valid for keys < mask_len
  int mask_len;
  int n_cached;         // cached keys to sweep (self: pos; cross: the description length)
  int pos;              // position of this step's token (self: its K/V row index; rotary angle)
  int cross;
  int rope;
  const bf16* rope_cos; // [positions][HD] tables (rope only)
  const bf16* rope_sin;
  float scale;
  bf16* out;            // [HD] destination of the attention output
};

// Requests the FIRST K/V stage of an item into `ring0`.  The cached rows do not depend on the projection the same phase computes,
// so the cluster step kernel calls this right after its MMA loop -- a microsecond or two before the attention itself starts --
// and passes pre_issued = true below.
__device__ __forceinline__ void attention_tc_issue_first(const TcItem& p, unsigned char* ring0, uint64_t* bars, int lane,
                                                         int part, int nparts, bool stream = false) {
  constexpr int CH = ATT_TC_CH;
  const int n_cached = p.n_cached;
  const int t0 = part * CH;
  if (t0 >= n_cached) return;
  const int n = (n_cached - t0 < CH) ? (n_cached - t0) : CH;
  const bf16* kc = p.kc;
  const bf16* vc = p.vc;
  // (no proxy fence: the stage was last written by the async proxy and read with generic loads; see step2.cu issue_weight_job)
  __syncwarp();
  const uint32_t bar = att_smem_u32(&bars[0]);
  if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(2 * n * HD * 2)) : "memory");
  __syncwarp();
  if (lane < 2) {
    const bf16* src = (lane == 0 ? kc : vc) + (size_t)t0 * HD;
    bf16* dst = reinterpret_cast<bf16*>(ring0) + (lane == 0 ? 0 : CH * HD);
    att_bulk_kv(att_smem_u32(dst), src, (uint32_t)(n * HD * 2), bar, stream);
  }
}

// ring0 / ring1: this warp's two K/V stages ([32][64] K | [32][64] V each, 16-byte aligned, anywhere in shared memory);
// fbuf: 192 floats (query, this step's key / value); bars: this warp's two mbarriers.
__device__ __forceinline__ void attention_decode_item_warp_tc(const TcItem& p, unsigned char* ring0, unsigned char* ring1, float* fbuf,
                                                              uint64_t* bars, int lane, uint32_t& parity, int part, int nparts, float* xch, int pair_bar,
                                                              long long* prof = nullptr, bool pre_issued = false, bool stream = false) {
  constexpr int CH = ATT_TC_CH;
  constexpr int NTS = CH / 8;     // score n-tiles per stage
  constexpr int KPV = CH / 16;    // k16 steps of P V per stage
  float* qs = fbuf;               // [64] query (fp32 of the bf16 values)
  float* kn = qs + HD;            // [64] this step's key   (self only)
  float* vn = kn + HD;            // [64] this step's value (self only)
  const int pos = p.pos;
  const bf16* __restrict__ rope_cos = p.rope ? p.rope_cos + (size_t)pos * HD : nullptr;
  const bf16* __restrict__ rope_sin = p.rope ? p.rope_sin + (size_t)pos * HD : nullptr;
  bf16* kc = p.kc;
  bf16* vc = p.vc;
  const int lo = lane, hi = lane + HD / 2;
  const int n_cached = p.n_cached;
  const int n_chunks_all = (n_cached + CH - 1) / CH;
  const int n_chunks = (n_chunks_all > part) ? (n_chunks_all - part + nparts - 1) / nparts : 0;

  auto issue = [&](int i) {
    const int st = i & 1;
    const int t0 = (part + nparts * i) * CH;
    const int n = (n_cached - t0 < CH) ? (n_cached - t0) : CH;
    const uint32_t bar = att_smem_u32(&bars[st]);
    if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(2 * n * HD * 2)) : "memory");
    __syncwarp();
    if (lane < 2) {
      const bf16* src = (lane == 0 ? kc : vc) + (size_t)t0 * HD;
      bf16* dst = reinterpret_cast<bf16*>(st ? ring1 : ring0) + (lane == 0 ? 0 : CH * HD);
      att_bulk_kv(att_smem_u32(dst), src, (uint32_t)(n * HD * 2), bar, stream);
    }
  };
  auto wait_stage = [&](int st) {
    const uint32_t bar = att_smem_u32(&bars[st]);
    const uint32_t par = (parity >> st) & 1u;
    uint32_t ok, spins = 0;
    do {
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(bar), "r"(par) : "memory");
      if (!ok && ++spins > (1u << 16)) { if (lane == 0) printf("ptts: tc attention KV mbarrier timeout (cta %d warp %d stage %d cross %d n_cached %d)\n", (int)blockIdx.x, (int)(threadIdx.x >> 5), st, p.cross, n_cached); __trap(); }
    } while (!ok);
    parity ^= (1u << st);
  };

  const int* km = p.km;
  auto load_mask = [&](int c) -> int {   // one key per lane (CH == 32); requested one stage ahead of its use
    const int t0 = (part + nparts * c) * CH;
    return (km != nullptr && c < n_chunks && t0 + lane < p.mask_len && t0 + lane < n_cached) ? km[t0 + lane] : 1;
  };
  int mk_next = load_mask(0);   // (first use: the ballot after the first stage has landed)

  // The stages are written by bulk copies (async proxy) and read with ldmatrix / generic loads: refilling one is a write-after-read
  // across proxies, which needs no proxy fence -- and fence.proxy.async would wait for every bulk copy the CTA has in flight
  // (the 64 KB weight jobs of the step kernel: ~0.5 us each time).  The only generic WRITE into a stage (zero-filling the tail of
  // an item's last, partial stage) is followed by the device-wide barrier's fence before the stage is refilled.
  __syncwarp();
  if (!pre_issued && n_chunks > 0) issue(0);
  if (n_chunks > 1) issue(1);   // (ring1 may alias buffers that were live when the first stage was requested early)

  // query (+ rotary), this step's K/V row (self): to the cache and to shared memory
  {
    const bf16* qsrc = p.q;
    float x0 = __bfloat162float(qsrc[lo]), x1 = __bfloat162float(qsrc[hi]);
    if (p.rope) {
      const float y0 = rope_elem<bf16>(x0, x1, lo, rope_cos, rope_sin), y1 = rope_elem<bf16>(x1, x0, hi, rope_cos, rope_sin);
      x0 = y0; x1 = y1;
    }
    qs[lo] = x0; qs[hi] = x1;
  }
  if (!p.cross && part == 0) {
    const bf16* ksrc = p.knew;
    const bf16* vsrc = p.vnew;
    float x0 = __bfloat162float(ksrc[lo]), x1 = __bfloat162float(ksrc[hi]);
    if (p.rope) {
      const float y0 = rope_elem<bf16>(x0, x1, lo, rope_cos, rope_sin), y1 = rope_elem<bf16>(x1, x0, hi, rope_cos, rope_sin);
      x0 = y0; x1 = y1;
    }
    const bf16 v0 = vsrc[lo], v1 = vsrc[hi];
    kc[(size_t)pos * HD + kv_swz(pos, lo)] = __float2bfloat16_rn(x0);
    kc[(size_t)pos * HD + kv_swz(pos, hi)] = __float2bfloat16_rn(x1);
    vc[(size_t)pos * HD + kv_swz(pos, lo)] = v0;
    vc[(size_t)pos * HD + kv_swz(pos, hi)] = v1;
    kn[lo] = DT<bf16>::rnd(x0); kn[hi] = DT<bf16>::rnd(x1);
    vn[lo] = __bfloat162float(v0); vn[hi] = __bfloat162float(v1);
  }
  __syncwarp();
  const int g = lane >> 2, t = lane & 3;
  // A fragments of the query: the SAME row in fragment rows 0..3 (lanes g < 4); k-step ks covers dims 16 ks .. 16 ks + 15.
  // Every row g < 4 then receives the scores of all 32 keys of a stage, and lane (g, t) takes the two of n-tile g: the softmax
  // arithmetic (mask, exp2, sums) is spread over 16 lanes instead of repeated 8 times on 4, and row g of the P V product
  // accumulates the keys of n-tile g only -- the four partial rows are added once per item, after the sweep.
  uint32_t qa0[4], qa2[4];
#pragma unroll
  for (int ks = 0; ks < 4; ks++) {
    qa0[ks] = (g < 4) ? att_pack(qs[16 * ks + 2 * t], qs[16 * ks + 2 * t + 1]) : 0u;
    qa2[ks] = (g < 4) ? att_pack(qs[16 * ks + 8 + 2 * t], qs[16 * ks + 8 + 2 * t + 1]) : 0u;
  }
  if (prof != nullptr && lane == 0) prof[8] = clock64();   // set-up done (query, K/V append, stages requested)
  const float scale_l2 = p.scale * 1.4426950408889634f;   // scores and running maximum live in the log2 domain (ex2.approx)
  float m_run = -INFINITY, l_run = 0.f;                    // l_run: THIS lane's share of the denominator until the final reduction
  float o[8][4];
#pragma unroll
  for (int j = 0; j < 8; j++)
#pragma unroll
    for (int e = 0; e < 4; e++) o[j][e] = 0.f;
  // ldmatrix lane addressing inside a stage: matrix mi = lane >> 3, row r = lane & 7 (16-byte chunk c of key row k at (c ^ (k & 7)) * 16)
  const int mi = lane >> 3, r8 = lane & 7;
  const int my_key = (8 * g + 2 * t) & 31;   // (g < 4) this lane's two keys inside a stage

  for (int c = 0; c < n_chunks; c++) {
    const int st = c & 1;
    const int t0 = (part + nparts * c) * CH;
    const int n = (n_cached - t0 < CH) ? (n_cached - t0) : CH;
    const int mk = mk_next;
    mk_next = load_mask(c + 1);
    wait_stage(st);
    uint32_t vword = __ballot_sync(0xffffffffu, mk != 0);
    if (n < CH) vword &= (1u << n) - 1u;
    bf16* stage = reinterpret_cast<bf16*>(st ? ring1 : ring0);
    const uint32_t kbase = att_smem_u32(stage), vbase = att_smem_u32(stage + CH * HD);
    if (n < CH) {  // last, partial stage: the copy filled n rows; whatever the rest of the V stage holds must not meet the MMA
      // (probability 0 x a stale NaN bit pattern is NaN); stale K rows only produce scores that are replaced by -inf below
      for (int i = lane; i < (CH - n) * 8; i += 32)
        *reinterpret_cast<uint4*>(stage + CH * HD + (size_t)(n + (i >> 3)) * HD + (i & 7) * 8) = make_uint4(0u, 0u, 0u, 0u);
      __syncwarp();
    }
    // ---- scores of the 32 keys: 4 n-tiles x 4 k-steps ----
    float s[NTS][4];
#pragma unroll
    for (int nt = 0; nt < NTS; nt++) {
#pragma unroll
      for (int e = 0; e < 4; e++) s[nt][e] = 0.f;
#pragma unroll
      for (int half = 0; half < 2; half++) {   // chunks 4 half .. 4 half + 3 of the key rows = k-steps 2 half, 2 half + 1
        uint32_t kb[4];
        att_ldsm4(kb, kbase + (uint32_t)((8 * nt + r8) * 128 + (((4 * half + mi) ^ r8) << 4)));
        att_mma(s[nt], qa0[2 * half], 0u, qa2[2 * half], 0u, kb[0], kb[1]);
        att_mma(s[nt], qa0[2 * half + 1], 0u, qa2[2 * half + 1], 0u, kb[2], kb[3]);
      }
    }
    // rows g < 4 all hold s[nt][0], s[nt][1] = keys 8 nt + 2 t, 8 nt + 2 t + 1; lane (g, t) keeps n-tile g
    static_assert(NTS == 4, "one score n-tile per fragment row 0..3");
    const float r0 = (g & 2) ? ((g & 1) ? s[3][0] : s[2][0]) : ((g & 1) ? s[1][0] : s[0][0]);
    const float r1 = (g & 2) ? ((g & 1) ? s[3][1] : s[2][1]) : ((g & 1) ? s[1][1] : s[0][1]);
    const float sv0 = (g < 4 && ((vword >> my_key) & 1u)) ? r0 * scale_l2 : -INFINITY;
    const float sv1 = (g < 4 && ((vword >> my_key) & 2u)) ? r1 * scale_l2 : -INFINITY;
    float cmax = fmaxf(sv0, sv1);
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, off));   // warp-uniform
    const float m_new = fmaxf(m_run, cmax);
    if (m_new != -INFINITY) {                          // (warp-uniform) otherwise every key so far is masked
      const float corr = att_ex2(m_run - m_new);       // ex2(-inf) = 0: nothing accumulated yet
      const float pe0 = att_ex2(sv0 - m_new), pe1 = att_ex2(sv1 - m_new);   // exactly 0 for masked / out-of-range keys and rows >= 4
      l_run = l_run * corr + (pe0 + pe1);
      m_run = m_new;
#pragma unroll
      for (int j = 0; j < 8; j++) { o[j][0] *= corr; o[j][1] *= corr; }
      const uint32_t pk = att_pack(pe0, pe1);          // probabilities rounded to bf16, like the SIMT path and torch's flash kernels
#pragma unroll
      for (int kp = 0; kp < KPV; kp++) {               // keys 16 kp .. 16 kp + 15 = n-tiles 2 kp (fragment columns 0-7), 2 kp + 1 (8-15)
        const uint32_t pa0 = (g == 2 * kp) ? pk : 0u, pa2 = (g == 2 * kp + 1) ? pk : 0u;
#pragma unroll
        for (int jp = 0; jp < 4; jp++) {               // dims 16 jp .. 16 jp + 15: n-tiles 2 jp, 2 jp + 1
          uint32_t vb[4];
          // matrices: (n-tile 2jp, keys 0-7), (2jp, keys 8-15), (2jp+1, keys 0-7), (2jp+1, keys 8-15) of this k-step; rows = keys, transposed on load
          const int key = 16 * kp + (mi & 1) * 8 + r8, chunk = 2 * jp + (mi >> 1);
          att_ldsm4_t(vb, vbase + (uint32_t)(key * 128 + ((chunk ^ r8) << 4)));
          att_mma(o[2 * jp], pa0, 0u, pa2, 0u, vb[0], vb[1]);
          att_mma(o[2 * jp + 1], pa0, 0u, pa2, 0u, vb[2], vb[3]);
        }
      }
    }
    if (c + 2 < n_chunks) {
      __syncwarp();
      issue(c + 2);
    }
  }
  if (prof != nullptr && lane == 0) { prof[9] = clock64(); prof[11] = n_chunks; }   // cached keys swept
  // rows 0..3 (lanes g < 4) hold partial output rows: o[j][0], o[j][1] = dims 8 j + 2 t, 8 j + 2 t + 1 over the keys of n-tile g
  if (!p.cross && part == 0) {  // the step's own key (position `pos`), from shared memory: accounted to row 0
    float sdot = 0.f;
#pragma unroll
    for (int e = 0; e < 2; e++) sdot = fmaf(qs[lane * 2 + e], kn[lane * 2 + e], sdot);
    sdot = warp_sum(sdot) * scale_l2;
    if (km != nullptr && pos < p.mask_len && km[pos] == 0) sdot = -INFINITY;
    const float m_new = fmaxf(m_run, sdot);
    if (m_new != -INFINITY) {
      const float corr = att_ex2(m_run - m_new);
      const float pe = att_ex2(sdot - m_new);
      const float pw = (g == 0) ? DT<bf16>::rnd(pe) : 0.f;
      l_run = l_run * corr + ((lane == 0) ? pe : 0.f);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        o[j][0] = o[j][0] * corr + pw * vn[8 * j + 2 * t];
        o[j][1] = o[j][1] * corr + pw * vn[8 * j + 2 * t + 1];
      }
      m_run = m_new;
    }
  }
  // add the four partial rows (lanes g = 0..3 of each t) and the 16 shares of the denominator: fixed order, once per item
#pragma unroll
  for (int j = 0; j < 8; j++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      float v = o[j][e];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      o[j][e] = v;
    }
#pragma unroll
  for (int off = 1; off < 16; off <<= 1) l_run += __shfl_xor_sync(0xffffffffu, l_run, off);
  l_run = __shfl_sync(0xffffffffu, l_run, 0);
  if (nparts == 2) {  // merge the two warps' partial softmax states (fixed order: part 0 then part 1)
    if (part == 1) {
      if (lane < 4) {
#pragma unroll
        for (int j = 0; j < 8; j++) { xch[8 * j + 2 * t] = o[j][0]; xch[8 * j + 2 * t + 1] = o[j][1]; }
      }
      if (lane == 0) { xch[HD] = m_run; xch[HD + 1] = l_run; }
    }
    asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
    if (part == 0) {
      const float m1 = xch[HD], l1 = xch[HD + 1];
      const float mm = fmaxf(m_run, m1);
      const float c0 = (m_run == -INFINITY) ? 0.f : att_ex2(m_run - mm);   // (-inf) - (-inf) would be NaN
      const float c1 = (m1 == -INFINITY) ? 0.f : att_ex2(m1 - mm);
      l_run = l_run * c0 + l1 * c1;
      if (lane < 4) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          o[j][0] = o[j][0] * c0 + xch[8 * j + 2 * t] * c1;
          o[j][1] = o[j][1] * c0 + xch[8 * j + 2 * t + 1] * c1;
        }
      }
    }
    asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
  }
  if (prof != nullptr && lane == 0) prof[10] = clock64();    // merged with the partner warp
  if (lane < 4 && part == 0) {
    const float inv = (l_run > 0.f) ? 1.0f / l_run : 0.f;  // fully masked row -> zeros (never consumed)
    bf16* out = p.out;
#pragma unroll
    for (int j = 0; j < 8; j++)
      *reinterpret_cast<__nv_bfloat162*>(out + 8 * j + 2 * t) = __floats2bfloat162_rn(o[j][0] * inv, o[j][1] * inv);
  }
}

// per-warp mbarrier setup (once per kernel); bars = this warp's two mbarriers
__device__ __forceinline__ void attention_decode_init_warp(uint64_t* bars, int lane) {
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(att_smem_u32(&bars[0])));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(att_smem_u32(&bars[1])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
}

}  // namespace ptts
