// step2.cu -- the CLUSTER decode step: one persistent kernel per generated token, 6 device-wide phases per layer (bf16).
//
// Replaces the same reference code as step.cu (ParlerTTSForCausalLM.forward with q_len == 1, modeling_parler_tts.py:1865-1974 /
// :983-1074, plus one iteration of GenerationMixin._sample) for the shapes layout.h::cluster_shape_ok() accepts (Parler-TTS-Mini:
// MHA, 16 heads).  step.cu's design -- 148 CTAs that each need the WHOLE 32 x H activation tile in every one of the 8 dependent
// phases of a layer -- measured 6.5 us per phase: ~2 us device-wide barrier, 1.3 us to pull the 66 KB tile, 0.6 us of LayerNorm
// statistics over it, an 8-warp split-K reduction through shared memory; 4.5 x the HBM time of the bytes it moves
// (profiles/r01_step_phases.md).  This kernel cuts the dependent chain and the per-CTA fixed work:
//
//   * grid = 32 clusters x 4 CTAs (cudaLaunchAttributeClusterDimension; this B200 co-schedules only 15 clusters of 8 -- seven
//     GPCs of 20 SMs and one of 8 -- but 37 clusters of 4).  Every GEMM is split 8 ways along K: rank r of a cluster stages K-slice
//     r (K/4 columns: 8-17 KB of activations instead of 66 KB) and its two warp groups reduce one half of it each ("virtual
//     ranks" v = 2 r + half).  Every warp owns whole n-tiles (no split-K through shared memory inside a CTA); the eight partial
//     sums meet through DISTRIBUTED SHARED MEMORY: one cp.async.bulk (shared::cta -> shared::cluster, mbarrier complete_tx) per peer.
//   * out-proj / cross out-proj / fc1 / fc2: cluster c owns N/32 output features, rank d finalises a quarter of them
//     (feature-partitioned exchange).  The residual-stream slice a CTA owns (32 rows x 8 features) never leaves its shared memory.
//   * QKV and q_cross: clusters 2h and 2h+1 own HEAD h for batch rows 0-15 / 16-31; the exchange is ROW-partitioned (rank d
//     receives rows 4d..4d+3 of q|k|v), so RoPE, the KV-cache append and the attention of those 4 (row, head) items run inside
//     the same phase: QKV -> self-attention and q_cross -> cross-attention need no device-wide barrier between them.
//     6 barriers per layer instead of 8.
//   * weights: one contiguous slice per (phase, cluster, rank) (layout.h cpack, built once by ptts_decoder_finalize), streamed by
//     ONE bulk copy per job into a 2 x 64 KB ring two jobs ahead, with an L2 evict-first policy like the K/V rows (1.2 GB per token
//     must not evict the kernel's own instructions and the small reused tensors).  No HBM -> L2 prefetches a layer ahead: they
//     measured slower (profiles/r02_step2_phases.md).
//   * fc2 (one n-tile per destination, K slice F/4): every warp takes all four n-tiles over an eighth of the K slice, the partial
//     tiles are added inside the CTA and one block per destination crosses the cluster (A fragments read once per CTA).
//   * the activation slice of the next phase is requested by the barrier's polling thread the moment the barrier opens; the
//     per-phase cluster barrier that guards buffer reuse arrives .relaxed (its default .release is a gpu-scope MEMBAR per warp).
//   * one launch runs up to StepParams.n_steps tokens: cur_len, the unfinished count and the stop decision advance on the device.
// Reduction orders are fixed (k-tiles ascending inside a warp, virtual ranks 0..7 across the cluster): bit-reproducible run to
// run.  They differ from step.cu / gemm.cu, so the two paths agree to bf16 accumulation-order noise, not bitwise.
#include "attn_core.cuh"
#include "common.cuh"
#include "kernels.h"
#include "ln_stats.cuh"
#include "sample_core.cuh"
#include "step.h"
#include <type_traits>

#include <cstdlib>

namespace ptts {
namespace cl {

constexpr int C = 4;            // CTAs per cluster
constexpr int V = 8;            // virtual ranks = warps per CTA: warp w reduces K-half (w >> 2) for destination rank (w & 3)
constexpr int THREADS = 256;
constexpr int ROWS = 32;        // batch rows (two m16 tiles; the head phases work on one half = one m16 tile)
constexpr int PROF_STRIDE = 16;  // clock64 stamps per phase row of the optional profile buffer (tools/profile_step2.py)
constexpr int QMAX = 6;         // n-tiles per warp (QKV: 24 n-tiles of a head over 4 destination groups)
constexpr int OFF_STATS = 256, OFF_PART = 512, OFF_RES = 2560, OFF_CVEC = 3584;
constexpr int HDR = 5632;       // mbarriers | row stats | stat partials | residual slice | folded-LN vectors c1[256] c2[256]
constexpr int WB_BYTES = 65536; // one weight ring buffer
constexpr int R_OFF = HDR + 2 * WB_BYTES;
// R region: [activation slice | 8 send blocks | 8 receive slots], split per phase; attention scratch and the lm-head tile alias it.
// Sized for Mini (H = 1024, F = 4096): fc1 = 16.5 KB slice + 2 x 8 blocks of (256 B stats + 32 x 34 floats).
constexpr int R_BYTES = 92160;
constexpr int QKV_OFF = R_BYTES - 2048;   // [4 rows][192] bf16 q|k|v (or [4][64] q_cross) of this rank's attention items
constexpr int SMEM_BYTES = R_OFF + R_BYTES;
static_assert(SMEM_BYTES + 1024 <= 227 * 1024, "cluster step kernel shared memory");

// ---- PTX helpers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int what) {
  uint32_t ok, spins = 0;
  do {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(s32(bar)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 22)) { printf("ptts: cluster step mbarrier timeout (cta %d, barrier kind %d)\n", (int)blockIdx.x, what); __trap(); }
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(s32(dst_smem)), "l"(src), "r"(bytes), "r"(s32(bar)) : "memory");
}
// Streamed-once data (the weights, the K/V rows: ~1.2 GB per token, ten times the L2) is requested with an evict-first policy so that
// it does not push out what IS reused between and inside launches: this kernel's instructions (the once-per-token phases ran at
// ~10 cycles per instruction on cold fetches), the folded-LayerNorm vectors, the activation images, the logits.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_stream(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(s32(dst_smem)), "l"(src), "r"(bytes), "r"(s32(bar)), "l"(l2_evict_first_policy()) : "memory");
}
// this CTA's shared memory -> a peer's shared memory (DSMEM), completion counted on the PEER's mbarrier
__device__ __forceinline__ void bulk_s2peer(uint32_t dst_cluster_addr, const void* src_smem, uint32_t bytes, uint32_t bar_cluster_addr) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_cluster_addr), "r"(s32(src_smem)), "r"(bytes), "r"(bar_cluster_addr) : "memory");
}
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) { uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r; }
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// The per-phase cluster barrier only guards buffer REUSE (a peer may overwrite my receive slots / I may overwrite a send block once
// everyone has consumed the previous phase's); the data itself is ordered by the exchange mbarrier.  A write-after-read needs no
// release: the default .release arrive is a gpu-scope MEMBAR per warp (it waits for the epilogue's global stores to be acknowledged,
// ~0.5 us, a second time before the layer barrier does).
__device__ __forceinline__ void cluster_arrive_reuse() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ unsigned ld_relaxed(const unsigned* p) { unsigned v; asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) { asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], const void* smem_ptr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(s32(smem_ptr)));
}
__device__ __forceinline__ void prof_mark(long long* prof, int slot) { if (prof != nullptr && threadIdx.x == 0) prof[slot] = clock64(); }

// ---- device-wide barrier (same protocol as step.cu) -----------------------------------------------
// `post` runs on thread 0 the moment the barrier opens (before the CTA is released): the next phase's activation copy.
template <typename Post>
__device__ __forceinline__ unsigned grid_sync(unsigned* ctr, unsigned target, int ph, Post post, bool acq_fence = true) {
  target += gridDim.x;
  asm volatile("fence.proxy.async.global;" ::: "memory");  // this thread's global writes -> other CTAs' TMA reads (writer side)
  __syncthreads();
  if (threadIdx.x == 0) {
    red_release_add(ctr, 1u);
    unsigned spins = 0;
    while (ld_relaxed(ctr) < target) {
      if (++spins > (1u << 24)) { printf("ptts: cluster step grid barrier timeout (cta %d target %u seen %u phase %d)\n", (int)blockIdx.x, target, ld_relaxed(ctr), ph); __trap(); }
    }
    // Everything this kernel reads that another CTA wrote during the same launch goes through L2 (TMA bulk copies of the images
    // and the K/V rows, __ldcg of the logits / EOS columns), so the L1 invalidation of an acquire fence protects nothing here and
    // costs 0.4 us per barrier (profiles/r02_step2_phases.md): the per-layer barriers skip it.
    if (acq_fence) asm volatile("fence.acq_rel.gpu;" ::: "memory");
    post();
  }
  __syncthreads();
  return target;
}

// One warp's MMA loop: QN n-tiles x MT m-tiles over k-tiles [kt_lo, kt_hi) of the staged slice.  SETS independent accumulator
// sets (k-tile parity x k16 half) break the dependent HMMA chain of the narrow phases (q = 1: out-proj, fc2 -- 32 dependent
// MMAs at 16 k-tiles otherwise); they are summed in a fixed order at the end.  STATS: the warp also accumulates the LayerNorm
// row sums of its k-tiles from the A fragments it has loaded anyway (the four destination groups of a K half repeat this work:
// 6 extra MMAs per k-tile and m-tile buy an exchange without any CTA-wide synchronisation).
template <int QN, int MT, int SETS, bool STATS>
__device__ __forceinline__ void mma_slice(float (&out)[2][6][4], RowStatFrag& rst, const bf16* xs, int apitch, const uint4* wb, int KT, int kt_lo,
                                          int kt_hi, int lrow, int lcol) {
  float acc[SETS][MT][QN][4];
#pragma unroll
  for (int s = 0; s < SETS; s++)
#pragma unroll
    for (int a = 0; a < MT; a++)
#pragma unroll
      for (int j = 0; j < QN; j++)
#pragma unroll
        for (int e = 0; e < 4; e++) acc[s][a][j][e] = 0.f;
  constexpr int KU = (SETS == 4) ? 2 : 1;   // k-tiles per iteration: the accumulator set index must be a compile-time constant
  for (int kt0 = kt_lo; kt0 < kt_hi; kt0 += KU) {   // (kt_hi - kt_lo is even: half of a slice of 8 or 32 k-tiles)
#pragma unroll
    for (int u = 0; u < KU; u++) {
      const int kt = kt0 + u;
      uint32_t a[MT][2][4];
#pragma unroll
      for (int mt = 0; mt < MT; mt++)
#pragma unroll
        for (int j = 0; j < 2; j++) ldsm4(a[mt][j], xs + (size_t)(mt * 16 + lrow) * apitch + kt * 32 + j * 16 + lcol);
      if (STATS) {   // every k-tile of this warp's K half: the (dest, K half) block then carries complete statistics for its K range
#pragma unroll
        for (int mt = 0; mt < MT; mt++) { row_stat_mma(rst, mt, a[mt][0]); row_stat_mma(rst, mt, a[mt][1]); }
      }
      constexpr int SB = (SETS >= 2) ? 1 : 0;
      const int s0 = (SETS == 4) ? 2 * u : 0;   // u is an unrolled constant
#pragma unroll
      for (int j = 0; j < QN; j++) {
        const uint4 w = wb[((size_t)j * KT + kt) * 32];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
          mma_bf16_16816(acc[s0][mt][j], a[mt][0], w.x, w.y);
          mma_bf16_16816(acc[s0 + SB][mt][j], a[mt][1], w.z, w.w);
        }
      }
    }
  }
#pragma unroll
  for (int mt = 0; mt < MT; mt++)
#pragma unroll
    for (int j = 0; j < QN; j++)
#pragma unroll
      for (int e = 0; e < 4; e++) {
        float v = acc[0][mt][j][e];
#pragma unroll
        for (int s2 = 1; s2 < SETS; s2++) v += acc[s2][mt][j][e];
        out[mt][j][e] = v;
      }
}

// phase kinds of a layer
enum { PH_QKV = 0, PH_O = 1, PH_QC = 2, PH_OC = 3, PH_FC1 = 4, PH_FC2 = 5 };
constexpr int JOBS_PER_LAYER = 7;   // weight jobs: QKV (two halves of 12 n-tiles), O, QC, OC, FC1, FC2

// source of weight job j for this CTA (7 per layer, then this CTA's lm-head tasks)
__device__ __forceinline__ bool weight_job(const StepParams& p, int j, int cta, int rank, const char*& src, uint32_t& bytes) {
  const int nl = JOBS_PER_LAYER * p.L;
  if (j < nl) {
    const int l = j / JOBS_PER_LAYER, jl = j - JOBS_PER_LAYER * l;
    const int ph = jl < 2 ? 0 : jl - 1;
    // the head phases' slices are shared by the two row-half clusters of a head: indexed (head, rank)
    const int64_t idx = (ph == PH_QKV || ph == PH_QC) ? (int64_t)(cta >> 3) * C + rank : (int64_t)cta;
    const int64_t sz = p.cp_slice[ph];
    bytes = (uint32_t)(ph == PH_QKV ? sz / 2 : sz);
    src = p.blob + p.layer0 + p.layer_stride * l + p.cp[ph] + idx * sz + (jl == 1 ? sz / 2 : 0);
    return true;
  }
  const int task = cta + (int)gridDim.x * (j - nl);
  const int ntasks = p.K * p.V / 32;
  if (task >= ntasks) return false;
  bytes = (uint32_t)(4 * p.H * 16);  // 4 n-tiles x K (fragment order: 16 B per (n-tile, k-pair) lane row)
  src = p.blob + p.heads + (int64_t)task * bytes;
  return true;
}

template <int ITEMS>
__global__ void __launch_bounds__(THREADS, 1) decode_step_cluster_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(128) unsigned char smem[];
  Ctrl* ctrl = p.sa.ctrl;
  if (p.prof != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.prof[(size_t)(6 * p.L + 2) * PROF_STRIDE + 3] = clock64();
  if (ctrl->active == 0) return;  // generation finished: the rest of the enqueued steps are no-ops (uniform over the grid)
  int cur_len = ctrl->cur_len;     // advanced locally when one launch runs several steps
  const unsigned gen = (unsigned)ctrl->launch_gen;
  int pos = p.P + cur_len - 1;  // cache position of the token being fed
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = p.H, F = p.F, B = p.B;
  const int rank = (int)cluster_rank();
  const int cta = (int)blockIdx.x;         // = cluster * 4 + rank
  const int cluster = cta >> 2;
  const int head = cluster >> 1, half = cluster & 1;   // head phases: this cluster's head and its batch-row half (rows 16 half ..)
  const int Ks = H / C, KsF = F / C;       // K-slice widths of a CTA
  const int pitch = Ks + 8, pitchF = KsF + 8;
  const int qe = F / p.nh / 64;            // fc1 n-tiles per destination rank (Mini: 4)
  const int dgrp = warp & 3, kh = warp >> 2;  // this warp: destination group, K half of the CTA's slice

  uint64_t* abar = reinterpret_cast<uint64_t*>(smem);        // activation slice
  uint64_t* wbar = abar + 1;                                  // [2] weight ring
  uint64_t* xbar = abar + 3;                                  // cluster exchange
  uint64_t* attbars = reinterpret_cast<uint64_t*>(smem + 128);  // [8 warps][2] K/V rings
  float* stats = reinterpret_cast<float*>(smem + OFF_STATS);   // [32][2] mean, rstd
  float* part = reinterpret_cast<float*>(smem + OFF_PART);     // [8][32][2]
  float* res_s = reinterpret_cast<float*>(smem + OFF_RES);     // [32][8] residual stream slice owned by this CTA
  float* cvec = reinterpret_cast<float*>(smem + OFF_CVEC);     // c1[256] | c2[256] of the current phase's features
  unsigned char* Rg = smem + R_OFF;
  uint32_t par_a = 0, par_w = 0, par_x = 0, att_parity = 0;

  if (tid == 0) {
    mbar_init(abar, 1); mbar_init(&wbar[0], 1); mbar_init(&wbar[1], 1); mbar_init(xbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  attention_decode_init_warp(attbars + 2 * warp, lane);
  cluster_arrive(); cluster_wait();   // every peer's mbarriers exist before any remote complete_tx
  // No HBM -> L2 prefetches a layer ahead: they cost more than they bring here (1097 -> 1070 us per step without them: the
  // shared-memory ring already runs two jobs = ~8 us ahead of its consumer, and every cp.async.bulk.prefetch.L2 is ~100 cycles of
  // issue time inside a phase; profiles/r02_step2_phases.md)
  unsigned* const bar_ctr = p.bar + (gen & 1u);
  unsigned bar_target = 0u;
  if (cta == 0 && tid == 0) p.bar[(gen + 1u) & 1u] = 0u;  // the counter the NEXT launch will use

  const char* blob = p.blob;
  long long* const prof0 = (p.prof != nullptr && cta == 0) ? p.prof : nullptr;
  long long* prof = prof0;
  prof_mark(prof, 0);

  // weight ring: job j lives in buffer j & 1; jobs 0 and 1 are requested now, job j + 2 when job j's MMA loop has retired
  auto issue_weight_job = [&](int j) {  // ONE thread
    const char* src; uint32_t bytes;
    if (!weight_job(p, j, cta, rank, src, bytes)) return;
    // No proxy fence here: the ring buffers are only ever WRITTEN through the async proxy (weights, K/V stages) and read with
    // generic loads -- a write-after-read across proxies needs none -- and fence.proxy.async waits for every bulk copy the CTA has
    // in flight (it cost ~0.5 us wherever one sat behind a 64 KB weight copy).  The one generic-written corner (the attention
    // merge scratch of the q_cross phase) is covered by the fence thread 0 executes at every device-wide barrier (request_slice).
    mbar_expect_tx(&wbar[j & 1], bytes);
    bulk_g2s_stream(smem + HDR + (j & 1) * WB_BYTES, src, bytes, &wbar[j & 1]);
  };
  // ---- one launch runs up to p.n_steps tokens (ptts_decode_steps): the ~10 us between dependent cooperative launches, the launch
  // skew in front of the first barrier and the cold instruction fetches of the once-per-token phases are paid once per launch.
  // Nothing below depends on the launch except the barrier counter, which simply keeps counting.
  __shared__ int s_next_active;
  const int n_steps = (p.do_sample_phase && p.n_steps > 1 && prof0 == nullptr) ? p.n_steps : 1;
  int unfinished_prev = 0;   // ctrl->n_unfinished is 0 at launch and only grows inside it (one add per unfinished row and step)
#pragma unroll 1
  for (int it = 0; it < n_steps; it++) {
  pos = p.P + cur_len - 1;
  prof = prof0;
  cluster_arrive_reuse();        // pre-arm: pairs with the first phase's "exchange buffers free" wait
  if (tid == 0) { issue_weight_job(0); issue_weight_job(1); }

  // global activation images, K-sliced for their consumer: [4 slices][32 rows][slice width + 8] bf16
  bf16* const x_img = p.cl_x;       // slices of H/4 columns (consumers: QKV, q_cross, fc1, lm heads)
  bf16* const a_img = p.cl_attn;    // slices of H/4 columns = 4 heads (consumers: out_proj, cross out_proj)
  bf16* const h_img = p.cl_h;       // slices of F/4 columns (consumer: fc2)
  const int x_slice_elems = ROWS * pitch, h_slice_elems = ROWS * pitchF;
  // where this CTA's 8 residual / out-proj features live in the x image: feature n = cta * 8 + f
  const int xo_slice = (cta * 8) / Ks, xo_col = (cta * 8) % Ks;

  // ---- embeddings: this CTA's 32 x 8 slice of sum_k embed_k[id] (+ position) -> residual slice + x image -----------------
  {
    const bf16* tables = reinterpret_cast<const bf16*>(blob + p.embed);
    const bf16* postab = p.rope ? nullptr : reinterpret_cast<const bf16*>(blob + p.pos);
    const int row = tid >> 3, f = tid & 7, n = cta * 8 + f;
    float v = 0.f;
    if (row < B) {
      float ev[16];
#pragma unroll
      for (int k = 0; k < 16; k++)
        if (k < p.K) ev[k] = __bfloat162float(tables[((size_t)k * (p.V + 1) + p.sa.cur_ids[row * p.K + k]) * H + n]);
#pragma unroll
      for (int k = 0; k < 16; k++)
        if (k < p.K) v = (k == 0) ? ev[k] : DT<bf16>::rnd(v + ev[k]);
      if (postab != nullptr) v = DT<bf16>::rnd(v + __bfloat162float(postab[(size_t)pos * H + n]));
    }
    res_s[row * 8 + f] = v;
    x_img[(size_t)xo_slice * x_slice_elems + row * pitch + xo_col + f] = __float2bfloat16_rn(v);
  }
  prof_mark(prof, 6);
  auto request_slice = [&](const bf16* img_slice, uint32_t bytes) {  // thread 0, the moment a device-wide barrier opens
    fence_proxy_async_smem();
    mbar_expect_tx(abar, bytes);
    bulk_g2s(Rg, img_slice, bytes, abar);
  };
  // activation slice of phase kind `sub`: rows of this cluster's half for the head phases, all 32 rows otherwise
  auto slice_of = [&](int sub, const bf16*& img, uint32_t& bytes) {
    if (sub == PH_QKV || sub == PH_QC) { img = x_img + (size_t)rank * x_slice_elems + (size_t)(16 * half) * pitch; bytes = (uint32_t)(16 * pitch * 2); }
    else if (sub == PH_O || sub == PH_OC) { img = a_img + (size_t)rank * x_slice_elems; bytes = (uint32_t)(x_slice_elems * 2); }
    else if (sub == PH_FC1) { img = x_img + (size_t)rank * x_slice_elems; bytes = (uint32_t)(x_slice_elems * 2); }
    else { img = h_img + (size_t)rank * h_slice_elems; bytes = (uint32_t)(h_slice_elems * 2); }
  };
  {
    const bf16* nimg; uint32_t nbytes;
    slice_of(PH_QKV, nimg, nbytes);
    bar_target = grid_sync(bar_ctr, bar_target, -1, [&]() { request_slice(nimg, nbytes); }, false);
  }
  prof_mark(prof, 7);

  const int lrow = (lane & 7) + ((lane >> 3) & 1) * 8, lcol = (lane >> 4) * 8;
  const int g = lane >> 2, t4 = lane & 3;
  const int n_phases = 6 * p.L;

  // per-warp constants of the attention items (row 16 half + 4 rank + (warp >> 1), this cluster's head): element offsets of the item's
  // K rows inside a layer's self / cross cache, the V planes' distance, and where its output goes in the attn image
  const int att_row = 16 * half + 4 * rank + (warp >> 1);
  const size_t self_item = ((size_t)att_row * p.nh + head) * p.Tmax * HD, self_vofs = (size_t)B * p.nh * p.Tmax * HD;
  const size_t cross_item = ((size_t)att_row * p.nh + head) * p.S * HD, cross_vofs = (size_t)B * p.nh * p.S * HD;
  bf16* const att_out = a_img + (size_t)(head >> 2) * x_slice_elems + (size_t)att_row * pitch + (head & 3) * HD;

#pragma unroll 1
  for (int ph = 0; ph < n_phases; ph++) {
    const int l = ph / 6, sub = ph - 6 * l;
    prof = prof0 ? prof0 + (size_t)(ph + 1) * PROF_STRIDE : nullptr;
    prof_mark(prof, 0);
    const char* lb = blob + p.layer0 + p.layer_stride * l;
    const bool rowpart = (sub == PH_QKV || sub == PH_QC);
    const bool has_ln = (sub == PH_QKV || sub == PH_QC || sub == PH_FC1);
    const int q = (sub == PH_QKV) ? 6 : (sub == PH_QC ? 2 : (sub == PH_FC1 ? qe : 1));   // n-tiles per warp
    const int Nc = 4 * q * 8;                                        // features of this cluster in this phase
    const int KT = (sub == PH_FC2 ? KsF : Ks) >> 5;                  // k32 tiles of this CTA's slice; a warp reduces half of them
    const int apitch = (sub == PH_FC2) ? pitchF : pitch;
    const int act_bytes = (rowpart ? 16 : ROWS) * apitch * 2;
    // exchange geometry: block (destination rank d, K half) at index 2 d + kh
    const int RS = (q == 1) ? 8 : 8 * q + 2;                         // floats per row of a feature-partitioned block
    const int blk = rowpart ? 32 + 4 * 8 * q * 4 : 256 + ROWS * RS * 4;   // one exchanged block: [statistics][rows][columns]
    const int wsend = rowpart ? C * blk : blk;                       // bytes a warp stages (one block per destination rank)
    const int j0 = JOBS_PER_LAYER * l + (sub == 0 ? 0 : sub + 1);    // first weight job of this phase
    const int njobs = sub == 0 ? 2 : 1;
    // fc2 (K slice of F/4, one n-tile per destination): with the (destination, K half) warp mapping four warps read the same A
    // fragments -- 512 B of shared memory per HMMA, 262 KB per phase, and the shared-memory port (128 B/clk), not the tensor pipe,
    // sets the 1.5 us.  Instead every warp takes ALL four n-tiles over an eighth of the K slice (A read once per CTA); the eight
    // partial tiles are added inside the CTA (shared memory, fixed order) and ONE block per destination crosses the cluster.
    const bool fc2_wide = (sub == PH_FC2) && q == 1 && (KT & 7) == 0;

    // folded-LayerNorm vectors of this phase's features: requested now, parked in shared memory after the MMA loop (a global
    // load followed at once by its shared-memory store would park the warp for an L2 round trip in front of the MMAs)
    float cv1 = 0.f, cv2 = 0.f;
    if (has_ln) {
      const float* c1; int ntot;
      if (sub == PH_QKV) { c1 = reinterpret_cast<const float*>(lb + p.c_qkv); ntot = p.qkv_rows; }
      else if (sub == PH_QC) { c1 = reinterpret_cast<const float*>(lb + p.c_qc); ntot = H; }
      else { c1 = reinterpret_cast<const float*>(lb + p.c_fc1); ntot = F; }
      const int nown = rowpart ? Nc : 8 * q;
      if (tid < nown) {
        int n;
        if (sub == PH_QKV) n = (tid >> 6) * (p.nh * HD) + head * HD + (tid & 63);
        else if (sub == PH_QC) n = head * HD + tid;
        else n = cta * 8 * q + tid;
        cv1 = c1[n];
        cv2 = c1[ntot + n];
      }
    }

    // ---- MMA: this warp's q n-tiles (destination group dgrp) over its half of the CTA's K slice ----
    for (int i = 0; i < njobs; i++) {
      mbar_wait(&wbar[(j0 + i) & 1], (par_w >> ((j0 + i) & 1)) & 1u, 1);
      par_w ^= 1u << ((j0 + i) & 1);
    }
    mbar_wait(abar, par_a, 0);
    par_a ^= 1u;
    prof_mark(prof, 1);
    float acc[2][QMAX][4];
    RowStatFrag rst;
    row_stat_zero(rst);
    {
      const bf16* xs = reinterpret_cast<const bf16*>(Rg);
      // QKV: destination groups 0,1 read the first weight job (n-tiles 0..11), groups 2,3 the second (12..23)
      const int wjob = (sub == PH_QKV) ? j0 + (dgrp >> 1) : j0;
      const int nt0 = (sub == PH_QKV) ? (dgrp & 1) * q : dgrp * q;   // first n-tile of this warp inside that job's slice
      const uint4* wb = reinterpret_cast<const uint4*>(smem + HDR + (wjob & 1) * WB_BYTES) + (size_t)nt0 * KT * 32 + lane;
      const int kt_lo = kh * (KT >> 1), kt_hi = kt_lo + (KT >> 1);
      if (sub == PH_QKV) mma_slice<6, 1, 1, true>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
      else if (sub == PH_QC) mma_slice<2, 1, 4, true>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
      else if (sub == PH_FC1) {
        if (q == 4) mma_slice<4, 2, 1, true>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
        else if (q == 2) mma_slice<2, 2, 2, true>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
        else mma_slice<1, 2, 4, true>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
      } else if (fc2_wide) {
        const uint4* wall = reinterpret_cast<const uint4*>(smem + HDR + (j0 & 1) * WB_BYTES) + lane;   // all four n-tiles
        mma_slice<4, 2, 1, false>(acc, rst, xs, apitch, wall, KT, warp * (KT >> 3), (warp + 1) * (KT >> 3), lrow, lcol);
      } else mma_slice<1, 2, 4, false>(acc, rst, xs, apitch, wb, KT, kt_lo, kt_hi, lrow, lcol);
    }
    prof_mark(prof, 2);
    if (has_ln && tid < (rowpart ? Nc : 8 * q)) { cvec[tid] = cv1; cvec[256 + tid] = cv2; }   // read in the epilogue, several barriers later
    __syncthreads();  // activation slice and weight buffer(s) are dead
    prof_mark(prof, 12);
    cluster_wait();  // every peer is past its previous epilogue: my send blocks have been read, its receive slots are free
    prof_mark(prof, 13);

    // ---- exchange: each warp stages its partial block in shared memory and ships it with ONE cp.async.bulk per destination
    // (shared::cta -> shared::cluster, complete_tx on the destination's mbarrier); no CTA-wide synchronisation on the way ----
    //   feature-partitioned: warp (dgrp, kh) -> rank dgrp, slot 2 rank + kh: [stats 32 x 2][32 rows][RS]
    //   row-partitioned    : warp w -> every rank d, slot 8 rank + w:        [stats 4 x 2][4 rows][8 q]  (rows 4d..4d+3, the warp's columns)
    const int nslots = rowpart ? V * C : (fc2_wide ? C : V);
    unsigned char* send = Rg + ((act_bytes + 127) & ~127);
    unsigned char* recv = send + ((V * wsend + 127) & ~127);
    if (tid == 0) mbar_expect_tx(xbar, (uint32_t)(nslots * blk));
    if (fc2_wide) {
      // stage the warp's four partial tiles in the (dead) activation slice: [warp][destination][32 rows][8] fp32
      float* stg = reinterpret_cast<float*>(Rg) + (size_t)warp * (C * ROWS * 8);
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          float* base = stg + (size_t)j * (ROWS * 8) + (mt * 16 + g) * 8 + 2 * t4;
          *reinterpret_cast<float2*>(base) = make_float2(acc[mt][j][0], acc[mt][j][1]);
          *reinterpret_cast<float2*>(base + 64) = make_float2(acc[mt][j][2], acc[mt][j][3]);
        }
      __syncthreads();
      prof_mark(prof, 14);
      // warp w adds the eight tiles of destination w >> 1, rows 16 (w & 1) .. + 15 (lane: row l & 15, features 4 (l >> 4) .. + 3)
      {
        const int d = warp >> 1, row = 16 * (warp & 1) + (lane & 15), f0 = 4 * (lane >> 4);
        const float* src = reinterpret_cast<const float*>(Rg) + (size_t)d * (ROWS * 8) + row * 8 + f0;
        float4 v = *reinterpret_cast<const float4*>(src);
#pragma unroll
        for (int sw = 1; sw < 8; sw++) {
          const float4 x = *reinterpret_cast<const float4*>(src + (size_t)sw * (C * ROWS * 8));
          v.x += x.x; v.y += x.y; v.z += x.z; v.w += x.w;
        }
        unsigned char* blk_d = send + (size_t)d * blk;
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(blk_d + 256) + row * RS + f0) = v;
        asm volatile("bar.sync %0, 64;" ::"r"((warp >> 1) + 1) : "memory");   // the two warps of this destination
        if ((warp & 1) == 0 && lane == 0) {
          fence_proxy_async_smem();
          bulk_s2peer(mapa(s32(recv + (size_t)rank * blk), (uint32_t)d), blk_d, (uint32_t)blk, mapa(s32(xbar), (uint32_t)d));
        }
      }
    } else {
      unsigned char* mine = send + (size_t)warp * wsend;
      if (!rowpart) {
        float* bp = reinterpret_cast<float*>(mine + 256);
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int j = 0; j < QMAX; j++) {
            if (j < q) {
              float* base = bp + (size_t)(mt * 16 + g) * RS + j * 8 + 2 * t4;
              *reinterpret_cast<float2*>(base) = make_float2(acc[mt][j][0], acc[mt][j][1]);
              *reinterpret_cast<float2*>(base + 8 * RS) = make_float2(acc[mt][j][2], acc[mt][j][3]);
            }
          }
        if (has_ln) {   // (S1, S2) of rows g / g+8 of each m-tile over this warp's K half (lane layout: ln_stats.cuh)
          float* st = reinterpret_cast<float*>(mine);
#pragma unroll
          for (int mt = 0; mt < 2; mt++) {
            const int r0 = mt * 16 + g;
            if (t4 == 0) { st[2 * r0] = rst.s1[mt][0]; st[2 * (r0 + 8)] = rst.s1[mt][2]; }
            if (t4 == (g >> 1)) {
              st[2 * r0 + 1] = (g & 1) ? rst.sq[mt][0][1] : rst.sq[mt][0][0];
              st[2 * (r0 + 8) + 1] = (g & 1) ? rst.sq[mt][1][3] : rst.sq[mt][1][2];
            }
          }
        }
      } else {
        const int qc = 8 * q;   // this warp's columns
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
          const int row = g + 8 * hh;
          // block of destination rank d = row >> 2: [destination][warp] order, so that ONE copy per destination ships all eight warps'
          // blocks (a bulk copy costs ~0.1 us of issue time through the uniform datapath: 4 per warp were 0.4 us of every warp's
          // critical path)
          unsigned char* blk_d = send + ((size_t)(row >> 2) * V + warp) * blk;
          float* bp = reinterpret_cast<float*>(blk_d + 32) + (row & 3) * qc + 2 * t4;
#pragma unroll
          for (int j = 0; j < QMAX; j++)
            if (j < q) *reinterpret_cast<float2*>(bp + j * 8) = make_float2(acc[0][j][2 * hh], acc[0][j][2 * hh + 1]);
          float* st = reinterpret_cast<float*>(blk_d) + (row & 3) * 2;
          if (t4 == 0) st[0] = hh ? rst.s1[0][2] : rst.s1[0][0];
          if (t4 == (g >> 1)) st[1] = hh ? ((g & 1) ? rst.sq[0][1][3] : rst.sq[0][1][2]) : ((g & 1) ? rst.sq[0][0][1] : rst.sq[0][0][0]);
        }
      }
      __syncwarp();
      prof_mark(prof, 14);
      if (!rowpart) {
        if (lane == 0) {
          fence_proxy_async_smem();
          bulk_s2peer(mapa(s32(recv + (size_t)(2 * rank + kh) * blk), (uint32_t)dgrp), mine, (uint32_t)blk, mapa(s32(xbar), (uint32_t)dgrp));
        }
      } else {
        __syncthreads();   // all eight warps' blocks are staged
        if (warp < C && lane == 0) {   // warp d ships [d][0..7] to rank d: it lands as slots 8 rank .. 8 rank + 7 there
          fence_proxy_async_smem();
          bulk_s2peer(mapa(s32(recv + (size_t)(8 * rank) * blk), (uint32_t)warp), send + (size_t)warp * V * blk, (uint32_t)(V * blk), mapa(s32(xbar), (uint32_t)warp));
        }
      }
    }
    // Requests that are not on the critical path go out now, while the partial sums travel: the weight ring's refill (two jobs
    // ahead; q_cross holds fc1's weights back until its attention is done, the K/V rings live in that buffer meanwhile) and, for
    // the head phases, the first K/V stage of this warp's attention item.  The rings live in the weight ring's idle space (the
    // phase's own weights are dead, the next jobs fill only the heads of the buffers), so they alias nothing the exchange uses.
    if (warp == 1 && lane == 0 && sub != PH_QC) for (int i = 0; i < njobs; i++) issue_weight_job(j0 + i + 2);
    TcItem item{};
    int att_b = B;
    unsigned char* att_ring = nullptr; unsigned char* att_ring1 = nullptr; float* att_f = nullptr; float* att_xch = nullptr;
    if (rowpart) {
      // row b = 16 half + 4 rank + (warp >> 1), this cluster's head: q at qkv_s[warp >> 1][0..63] (k at +64, v at +128 in the self phase)
      const bf16* qrow = reinterpret_cast<const bf16*>(Rg + QKV_OFF) + (size_t)(warp >> 1) * Nc;
      att_b = att_row;
      item.q = qrow;
      item.pos = pos; item.rope = p.rope; item.scale = p.scale;
      item.rope_cos = reinterpret_cast<const bf16*>(blob + p.rope_cos); item.rope_sin = reinterpret_cast<const bf16*>(blob + p.rope_sin);
      // attn image: row b, head h -> slice h / 4, column (h % 4) * 64
      item.out = att_out;
      unsigned char* wb0 = smem + HDR;   // the two weight ring buffers
      if (sub == PH_QKV) {
        item.knew = qrow + HD; item.vnew = qrow + 2 * HD;
        bf16* kc = reinterpret_cast<bf16*>(p.self_kv + p.self_layer_stride * l) + self_item;
        item.kc = kc; item.vc = kc + self_vofs;
        item.km = p.prompt_mask ? p.prompt_mask + (size_t)att_b * p.P : nullptr; item.mask_len = p.P;
        item.cross = 0; item.n_cached = pos;
        // out-proj's 16 KB go to the head of buffer (j0+2)&1, q_cross's 32 KB to the head of the other one.  Stage 0 of every warp
        // (requested now) sits in those buffers' tails; stage 1 (requested when the attention starts) in what the exchange has
        // released by then: the receive slots [34 KB, 58 KB) and the activation slice [0, 8 KB) of R, the gap behind the query
        // scratch [71 KB, 87 KB), and the rest of the q_cross buffer's tail.
        unsigned char* bB = wb0 + ((j0 + 2) & 1) * WB_BYTES; unsigned char* bC = wb0 + ((j0 + 3) & 1) * WB_BYTES;
        att_ring = warp < 6 ? bB + 16384 + warp * ATT_TC_STAGE_BYTES : bC + 32768 + (warp - 6) * ATT_TC_STAGE_BYTES;
        att_ring1 = warp < 3 ? Rg + 34048 + warp * ATT_TC_STAGE_BYTES : (warp < 5 ? Rg + 72704 + (warp - 3) * ATT_TC_STAGE_BYTES
                  : (warp == 5 ? Rg : bC + 49152 + (warp - 6) * ATT_TC_STAGE_BYTES));
        att_xch = reinterpret_cast<float*>(Rg + 59648) + (warp >> 1) * 128;
      } else {
        item.knew = nullptr; item.vnew = nullptr;
        bf16* ck = reinterpret_cast<bf16*>(p.cross_kv + p.cross_layer_stride * l) + cross_item;
        item.kc = ck; item.vc = ck + cross_vofs;
        item.km = p.enc_mask ? p.enc_mask + (size_t)att_b * p.S : nullptr; item.mask_len = p.S;
        item.cross = 1; item.n_cached = p.S;
        // this phase's own (dead) weight buffer holds stage 0 of every warp; cross out-proj's 16 KB sit at the head of the other one.
        // Stage 1 (descriptions longer than 64 positions): R behind the exchange buffers, the gap behind the query scratch, and
        // the cross out-proj buffer's tail.
        unsigned char* bD = wb0 + ((j0 + 1) & 1) * WB_BYTES;
        att_ring = wb0 + (j0 & 1) * WB_BYTES + warp * ATT_TC_STAGE_BYTES;
        att_ring1 = warp < 4 ? Rg + 28672 + warp * ATT_TC_STAGE_BYTES : (warp < 6 ? Rg + 72704 + (warp - 4) * ATT_TC_STAGE_BYTES
                  : bD + 16384 + (warp - 6) * ATT_TC_STAGE_BYTES);
        att_xch = reinterpret_cast<float*>(bD + 32768) + (warp >> 1) * 128;
      }
      att_f = reinterpret_cast<float*>(Rg + 65536) + warp * 192;   // query / new key / new value: a corner of R the exchange never uses
      if (att_b < B) attention_tc_issue_first(item, att_ring, attbars + 2 * warp, lane, warp & 1, 2, true);
    }
    prof_mark(prof, 15);
    mbar_wait(xbar, par_x, 2);
    par_x ^= 1u;
    prof_mark(prof, 3);

    // ---- epilogue: sum the partial blocks in a fixed order, LayerNorm fix-up, activation / residual ----
    if (!rowpart) {
      const int row = tid >> 3, f0 = tid & 7;
      float ln_mean = 0.f, ln_rstd = 0.f;
      if (has_ln) {   // (fc1) every thread adds its row's eight partial statistics itself, in block order: broadcast loads instead of a
        float S1 = 0.f, S2 = 0.f;   // 32-thread pass + CTA barrier
#pragma unroll
        for (int v = 0; v < V; v++) { const float2 x = *reinterpret_cast<const float2*>(recv + (size_t)v * blk + row * 8); S1 += x.x; S2 += x.y; }
        ln_mean = S1 / (float)H;
        ln_rstd = rsqrtf(fmaxf(S2 / (float)H - ln_mean * ln_mean, 0.f) + p.eps);
      }
      if (row < B && sub == PH_FC1 && q == 4) {   // 4 consecutive features per thread: 8-byte loads, one 8-byte store
        const int f = 4 * f0;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int sv = 0; sv < V; sv++) {
          const float* bp = reinterpret_cast<const float*>(recv + (size_t)sv * blk + 256) + row * RS + f;
          const float2 a = *reinterpret_cast<const float2*>(bp), b2 = *reinterpret_cast<const float2*>(bp + 2);
          v[0] += a.x; v[1] += a.y; v[2] += b2.x; v[3] += b2.y;
        }
#pragma unroll
        for (int e = 0; e < 4; e++) v[e] = apply_act(DT<bf16>::rnd(ln_rstd * (v[e] - ln_mean * cvec[f + e]) + cvec[256 + f + e]), p.act);
        const int n = cta * 32 + f;
        uint2 pk;
        pk.x = att_pack(v[0], v[1]); pk.y = att_pack(v[2], v[3]);
        *reinterpret_cast<uint2*>(h_img + (size_t)(n / KsF) * h_slice_elems + row * pitchF + (n % KsF)) = pk;
      } else if (row < B) {
        for (int i = 0; i < q; i++) {
          const int f = f0 + 8 * i;
          float v = 0.f;
          if (fc2_wide) {
#pragma unroll
            for (int sv = 0; sv < C; sv++) v += reinterpret_cast<const float*>(recv + (size_t)sv * blk + 256)[row * RS + f];
          } else {
#pragma unroll
            for (int sv = 0; sv < V; sv++) v += reinterpret_cast<const float*>(recv + (size_t)sv * blk + 256)[row * RS + f];
          }
          if (sub == PH_FC1) {
            v = ln_rstd * (v - ln_mean * cvec[f]) + cvec[256 + f];
            v = apply_act(DT<bf16>::rnd(v), p.act);
            const int n = cta * 8 * q + f;   // h feature -> slice n / KsF of the fc2 image
            h_img[(size_t)(n / KsF) * h_slice_elems + row * pitchF + (n % KsF)] = __float2bfloat16_rn(v);
          } else {  // out-proj / cross out-proj / fc2: residual add on the slice this CTA owns
            v = DT<bf16>::rnd(res_s[row * 8 + f] + DT<bf16>::rnd(v));
            res_s[row * 8 + f] = v;
            x_img[(size_t)xo_slice * x_slice_elems + row * pitch + xo_col + f] = __float2bfloat16_rn(v);
          }
        }
      }
    } else {
      bf16* qkv_s = reinterpret_cast<bf16*>(Rg + QKV_OFF);  // [4][Nc]
      auto gather = [&](auto qc_tag) {   // (the column count per warp is a constant of the phase: no run-time divisions)
        constexpr int QC = decltype(qc_tag)::value, NC = 4 * QC;
        for (int idx = tid; idx < 4 * NC; idx += THREADS) {
          const int r4 = idx / NC, col = idx - r4 * NC;
          const int dg = col / QC, cw = col - dg * QC;           // the warps with dgrp == dg hold this column
          // row 16 half + 4 rank + r4: statistics from the dgrp == 0 warp of every (source rank, K half), added by every thread itself
          // (broadcast loads: a warp's 32 elements share the row) instead of a 4-thread pass + CTA barrier
          float S1 = 0.f, S2 = 0.f;
#pragma unroll
          for (int sr = 0; sr < C; sr++)
#pragma unroll
            for (int k2 = 0; k2 < 2; k2++) {
              const float2 x = *reinterpret_cast<const float2*>(recv + (size_t)(8 * sr + 4 * k2) * blk + r4 * 8);
              S1 += x.x; S2 += x.y;
            }
          const float ln_mean = S1 / (float)H;
          const float ln_rstd = rsqrtf(fmaxf(S2 / (float)H - ln_mean * ln_mean, 0.f) + p.eps);
          float v = 0.f;
#pragma unroll
          for (int sv = 0; sv < V; sv++)   // (source rank, K half) in order: warp index = 4 (sv & 1) + dg of rank sv >> 1
            v += reinterpret_cast<const float*>(recv + (size_t)(8 * (sv >> 1) + 4 * (sv & 1) + dg) * blk + 32)[r4 * QC + cw];
          v = ln_rstd * (v - ln_mean * cvec[col]) + cvec[256 + col];
          qkv_s[idx] = __float2bfloat16_rn(v);
        }
      };
      if (sub == PH_QKV) gather(std::integral_constant<int, 48>{}); else gather(std::integral_constant<int, 16>{});
      static_assert(HD == 64, "q = 6 (q|k|v of a head over 4 warps) and q = 2 n-tiles per warp");
    }
    prof_mark(prof, 4);
    __syncthreads();   // this CTA's receive slots are consumed (and q|k|v complete): peers may send the next phase's partials
    cluster_arrive_reuse();

    // ---- attention of this rank's 4 (row, head) items: two warps per item (first two K/V stages were requested after the MMA) ----
    if (rowpart) {
      if (att_b < B)
        attention_decode_item_warp_tc(item, att_ring, att_ring1, att_f, attbars + 2 * warp, lane, att_parity, warp & 1, 2, att_xch,
                                      (warp >> 1) + 1, warp == 0 ? prof : nullptr, true, true);
      prof_mark(prof, 5);
      if (sub == PH_QC) {   // fc1's weights were held back: the K/V rings used their buffer
        __syncthreads();
        if (tid == 32) issue_weight_job(j0 + 2);
      }
    }
    prof_mark(prof, 6);
    if (p.prof != nullptr && l == p.L / 2 && tid == 0) {   // profiling runs: when does EACH CTA reach the barrier of the middle layer's phases
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      p.prof[(size_t)(n_phases + 4) * PROF_STRIDE + sub * (int)gridDim.x + cta] = (long long)ns;
    }

    // ---- device-wide barrier; the next phase's activation slice is requested the moment it opens ----
    const bool last = (ph + 1 == n_phases);
    const bf16* nimg; uint32_t nbytes;
    if (last) { nimg = x_img; nbytes = (uint32_t)(C * x_slice_elems * 2); }   // lm heads: the whole x image
    else slice_of((sub + 1) % 6, nimg, nbytes);
    bar_target = grid_sync(bar_ctr, bar_target, ph, [&]() { request_slice(nimg, nbytes); }, false);
    prof_mark(prof, 7);
  }
  cluster_wait();  // balance the last phase's arrive

  // ---- final LayerNorm + K lm heads: N-split over all CTAs (4 n-tiles per task, full K), no exchange ----
  prof = prof0 ? prof0 + (size_t)(n_phases + 1) * PROF_STRIDE : nullptr;
  prof_mark(prof, 0);
  {
    const int ntasks = p.K * p.V / 32;
    const float* c1 = reinterpret_cast<const float*>(blob + p.c_heads);
    const float* c2 = c1 + p.K * p.V;
    mbar_wait(abar, par_a, 3);
    par_a ^= 1u;
    const bf16* xs = reinterpret_cast<const bf16*>(Rg);   // [4 slices][32][pitch]
    const int KTH = H >> 5, KTS = Ks >> 5;                 // k32 tiles of the full row / of one slice
    {  // row statistics over the full rows: k-tile kt by warp kt % 8
      RowStatFrag rst;
      row_stat_zero(rst);
      for (int kt = warp; kt < KTH; kt += 8) {
        const bf16* sl = xs + (size_t)(kt / KTS) * x_slice_elems + (kt % KTS) * 32;
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int j = 0; j < 2; j++) {
            uint32_t a[4];
            ldsm4(a, sl + (size_t)(mt * 16 + lrow) * pitch + j * 16 + lcol);
            row_stat_mma(rst, mt, a);
          }
      }
      row_stat_store(rst, part, warp, lane);
      __syncthreads();
      row_stat_finalize(part, H, ROWS, p.eps, stats);
      __syncthreads();
    }
    prof_mark(prof, 1);
    float* red = reinterpret_cast<float*>(Rg + (size_t)C * x_slice_elems * 2);  // [4 n-tiles][32][8] partials of the upper K half
    const int jn = warp >> 1, khh = warp & 1;   // this warp: n-tile jn of the task, K half khh
    int job = JOBS_PER_LAYER * p.L;
    for (int task = cta; task < ntasks; task += (int)gridDim.x, job++) {
      mbar_wait(&wbar[job & 1], (par_w >> (job & 1)) & 1u, 4);
      par_w ^= 1u << (job & 1);
      float acc[2][4];
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int e = 0; e < 4; e++) acc[a][e] = 0.f;
      const uint4* wb = reinterpret_cast<const uint4*>(smem + HDR + (job & 1) * WB_BYTES) + (size_t)jn * KTH * 32 + lane;
      for (int kt = khh * (KTH / 2); kt < (khh + 1) * (KTH / 2); kt++) {
        const bf16* sl = xs + (size_t)(kt / KTS) * x_slice_elems + (kt % KTS) * 32;
        const uint4 w = wb[(size_t)kt * 32];
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
          uint32_t a0[4], a1[4];
          ldsm4(a0, sl + (size_t)(mt * 16 + lrow) * pitch + lcol);
          ldsm4(a1, sl + (size_t)(mt * 16 + lrow) * pitch + 16 + lcol);
          mma_bf16_16816(acc[mt], a0, w.x, w.y);
          mma_bf16_16816(acc[mt], a1, w.z, w.w);
        }
      }
      if (khh == 1) {
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
          float* base = red + ((size_t)jn * 32 + mt * 16 + g) * 8 + 2 * t4;
          *reinterpret_cast<float2*>(base) = make_float2(acc[mt][0], acc[mt][1]);
          *reinterpret_cast<float2*>(base + 64) = make_float2(acc[mt][2], acc[mt][3]);
        }
      }
      __syncthreads();  // weight buffer dead, upper-half partials visible
      if (tid == 32) issue_weight_job(job + 2);
      if (khh == 0) {
        const int n0 = task * 32 + jn * 8 + 2 * t4;
        const float2 c1v = *reinterpret_cast<const float2*>(c1 + n0), c2v = *reinterpret_cast<const float2*>(c2 + n0);
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const int row = mt * 16 + g + 8 * hh;
            if (row < B) {
              const float2 up = *reinterpret_cast<const float2*>(red + ((size_t)jn * 32 + row) * 8 + 2 * t4);
              const float mean = stats[2 * row], rstd = stats[2 * row + 1];
              const float v0 = DT<bf16>::rnd(rstd * (acc[mt][2 * hh] + up.x - mean * c1v.x) + c2v.x);
              const float v1 = DT<bf16>::rnd(rstd * (acc[mt][2 * hh + 1] + up.y - mean * c1v.y) + c2v.y);
              *reinterpret_cast<float2*>(p.logits + (size_t)row * p.K * p.V + n0) = make_float2(v0, v1);
            }
          }
      }
      __syncthreads();  // `red` is reused by the next task
    }
  }
  prof_mark(prof, 6);
  bar_target = grid_sync(bar_ctr, bar_target, n_phases, []() {});
  prof = prof0 ? prof0 + (size_t)(n_phases + 2) * PROF_STRIDE : nullptr;  // tail row: sampling / barrier
  prof_mark(prof, 0);
  if (p.do_sample_phase) {
    const ptts_gen_params gp = *p.sa.gen;
    const int BK = B * p.K;
    sample_all_rows_cta<ITEMS>(p.sa, gp, cta, (int)gridDim.x, BK, cur_len);
    prof_mark(prof, 1);
    // every CTA learns whether any row is still unfinished: thread 0 reads the counter the moment the barrier opens (after its
    // acquire fence); the counter is reset only when the launch ends, so a step's count is the growth since the previous step
    bar_target = grid_sync(bar_ctr, bar_target, n_phases + 1, [&]() {
      const int tot = *reinterpret_cast<volatile int*>(&ctrl->n_unfinished);
      s_next_active = (tot - unfinished_prev > 0) ? 1 : 0;
      unfinished_prev = tot;
    });
    prof_mark(prof, 2);
  }
  bool go_on = false;
  if (p.do_sample_phase) {
    const int act = s_next_active;   // (written before the barrier's closing __syncthreads)
    if (cta == 0 && tid == 0) {
      ctrl->cur_len = cur_len + 1;
      ctrl->active = act;
      ctrl->steps_run += 1;
    }
    go_on = act != 0;
    cur_len += 1;
  }
  if (!go_on) break;
  }  // steps of this launch
  if (cta == 0 && tid == 0) {
    // (a CTA that is slower out of the last barrier may still read the counter: it then sees a count <= the one it expects and
    // concludes "finished", which is what leaving the loop means anyway)
    if (p.do_sample_phase) ctrl->n_unfinished = 0;
    ctrl->launch_gen = (int)(gen + 1u);
  }
}

// ---- weight repack: fragment-order matrices -> one contiguous slice per (phase, cluster or head, rank) -------------------
// Both layouts are made of the same 512-byte (n8 x k32) tiles, so the repack is a tile gather.
//   head phases (QKV, q_cross): slice (head, rank) = the head's n-tiles x k-tiles [rank kts, (rank + 1) kts)
//   the others: slice cta = cluster * 4 + rank = the cluster's ntc n-tiles x the rank's k-tiles
__global__ void cluster_pack_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int ph, int nh, int ntc, int kts, int KT_src) {
  const int64_t tile = blockIdx.x;   // dst tile index = (slice * ntc + j) * kts + ktl
  const int ktl = (int)(tile % kts);
  const int j = (int)((tile / kts) % ntc);
  const int slice = (int)(tile / ((int64_t)kts * ntc));
  const int rank = slice & 3, owner = slice >> 2;   // owner = head (head phases) or cluster
  int n_tile;
  if (ph == PH_QKV) n_tile = (j >> 3) * (nh * 8) + owner * 8 + (j & 7);   // q | k | v rows of head `owner` in the fused matrix
  else n_tile = owner * ntc + j;
  const int kt = rank * kts + ktl;
  dst[tile * 32 + threadIdx.x] = src[((int64_t)n_tile * KT_src + kt) * 32 + threadIdx.x];
}

}  // namespace cl

// ---- host side ----------------------------------------------------------------------------------
int cluster_pack_layer(const char* layer_src, char* layer_dst, const int64_t* mat_off, const int64_t* cp_off, int nh, int H, int F, cudaStream_t st) {
  // mat_off: byte offsets (inside the layer) of wqkv, wo, wqc, woc, fc1, fc2; cp_off: of the six packed regions
  const int ks = H / 4 / 32, ksf = F / 4 / 32;
  const int ntc[6] = {24, 4, 8, 4, F / (2 * nh) / 8, 4};
  const int owners[6] = {nh, 2 * nh, nh, 2 * nh, 2 * nh, 2 * nh};
  for (int ph = 0; ph < 6; ph++) {
    const int kts = (ph == 5) ? ksf : ks;
    const int KT_src = (ph == 5) ? F / 32 : H / 32;
    const int64_t tiles = (int64_t)owners[ph] * 4 * ntc[ph] * kts;
    cl::cluster_pack_kernel<<<(unsigned)tiles, 32, 0, st>>>(reinterpret_cast<const uint4*>(layer_src + mat_off[ph]),
                                                            reinterpret_cast<uint4*>(layer_dst + cp_off[ph]), ph, nh, ntc[ph], kts, KT_src);
  }
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

static const void* cluster_kernel_fn(const StepParams& p) {
  if (p.sample_items <= 1) return (const void*)cl::decode_step_cluster_kernel<1>;
  if (p.sample_items <= 5) return (const void*)cl::decode_step_cluster_kernel<5>;
  return (const void*)cl::decode_step_cluster_kernel<9>;
}

static void cluster_launch_config(const StepParams& p, cudaLaunchConfig_t& cfg, cudaLaunchAttribute* at, cudaStream_t st) {
  cfg = cudaLaunchConfig_t{};
  cfg.gridDim = dim3((unsigned)(2 * p.nh * cl::C));   // 2 clusters per head
  cfg.blockDim = dim3(cl::THREADS);
  cfg.dynamicSmemBytes = cl::SMEM_BYTES;
  cfg.stream = st;
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cl::C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeCooperative;   // every CTA spins on the others: co-residency must be guaranteed
  at[1].val.cooperative = 1;
  cfg.attrs = at;
  // PTTS_STEP_COOP=0: cluster attribute only (Nsight Compute cannot launch a cooperative cluster grid; the 128 CTAs of an
  // otherwise idle GPU are co-resident anyway -- profiling runs only)
  static const bool coop = [] { const char* v = getenv("PTTS_STEP_COOP"); return !(v && v[0] == '0'); }();
  cfg.numAttrs = coop ? 2 : 1;
}

// true when the 32 x 4 cluster grid can be co-resident on this device
bool cluster_step_available(const StepParams& p) {
  const void* fn = cluster_kernel_fn(p);
  static bool told = false;
  auto why = [&](const char* what, cudaError_t e, int n) {
    if (!told) fprintf(stderr, "ptts_b200: cluster step kernel not used (%s: %s, %d co-resident clusters of %d, need %d); the 148-CTA step kernel runs instead\n",
                       what, cudaGetErrorString(e), n, cl::C, 2 * p.nh);
    told = true;
    cudaGetLastError();
    return false;
  };
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, cl::SMEM_BYTES);
  if (e != cudaSuccess) return why("shared memory attribute", e, 0);
  cudaLaunchConfig_t cfg; cudaLaunchAttribute at[2];
  cluster_launch_config(p, cfg, at, nullptr);
  cfg.numAttrs = 1;  // the occupancy query takes the cluster shape
  int n = 0;
  e = cudaOccupancyMaxActiveClusters(&n, fn, &cfg);
  if (e != cudaSuccess) return why("cluster occupancy query", e, n);
  if (n < 2 * p.nh) return why("too few co-resident clusters", cudaSuccess, n);
  return true;
}

int launch_decode_step_cluster(const StepParams& p, cudaStream_t st) {
  const void* fn = cluster_kernel_fn(p);
  cudaLaunchConfig_t cfg; cudaLaunchAttribute at[2];
  cluster_launch_config(p, cfg, at, st);
  void* args[] = {(void*)&p};
  PTTS_CHECK_CUDA(cudaLaunchKernelExC(&cfg, fn, args));
  return PTTS_OK;
}

}  // namespace ptts
