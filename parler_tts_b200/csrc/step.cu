// step.cu -- the fused decode step: ONE persistent kernel per generated token (bf16 model dtype).
//
// Replaces, per step, everything ptts_decode_forward + ptts_sample launch as 195 separate kernels:
// embedding sum, L x {LN+QKV, self-attention with KV append, out_proj+residual, LN+q, cross-attention,
// out_proj+residual, LN+fc1+GELU, fc2+residual}, final LN + K lm heads, logits processors + sampling
// (reference: ParlerTTSForCausalLM.forward with q_len==1, modeling_parler_tts.py:1865-1974 / :983-1074, and one
// iteration of GenerationMixin._sample).
//
// Why one kernel: the step is a chain of ~195 dependent phases, each moving only 0.3-8 MB.  At the HBM
// roofline the whole step lasts ~220 us (Mini, B=32), i.e. ~1.1 us per phase, so launch latency and per-kernel
// ramp dominate a multi-kernel design.  Here one CTA per SM stays resident for the whole step:
//   * phases are separated by a device-wide barrier (monotonic counter in global memory, release/acquire);
//   * the next layer's weight slices are pulled into L2 one layer ahead with cp.async.bulk.prefetch.L2
//     (the stream is static, so HBM keeps flowing while the chain waits on barriers);
//   * the 32-row activation tile is staged by the TMA engine (cp.async.bulk -> shared memory, mbarrier
//     completion), double-buffered over K for fc2;
//   * weights stream from L2 in mma B-fragment order straight into registers (gemm.cu's layout);
//   * attention processes two (row, kv head) items per CTA concurrently (128 threads each, named barriers).
// All reductions keep a fixed order: results are bit-reproducible and identical to the multi-kernel path.
#include "attn_core.cuh"
#include "common.cuh"
#include "kernels.h"
#include "ln_stats.cuh"
#include "sample_core.cuh"
#include "step.h"

namespace ptts {

constexpr int ST_THREADS = 256;
constexpr int ST_WARPS = 8;
constexpr int ST_HEADER = 512 + 8 * 32 * 2 * 4 + 256;  // mbarriers [0,256) | row stats [256,512) | stat partials [512,2560) | c1,c2 of the task [2560,2816)

// ---- PTX helpers --------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  uint32_t spins = 0;
  do {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 22)) { printf("ptts: tile mbarrier timeout (cta %d)\n", (int)blockIdx.x); __trap(); }
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// orders this thread's prior generic-proxy accesses (shared AND the acquired global data) before later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void l2_prefetch(const void* p, uint32_t bytes) {
  const char* c = reinterpret_cast<const char*>(p);
  while (bytes > 0) {
    const uint32_t n = bytes > 32768u ? 32768u : bytes;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(c), "r"(n) : "memory");
    c += n;
    bytes -= n;
  }
}
__device__ __forceinline__ unsigned ld_relaxed(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void ldmatrix_x4s(uint32_t (&r)[4], const void* smem_ptr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(smem_ptr)));
}
__device__ __forceinline__ void mma_bf16s(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint4 ldg_stream_s(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// ---- device-wide barrier ------------------------------------------------------------------------
// Arrive = red.release (cumulative over the CTA's writes ordered by the preceding bar.sync); the spin is a
// RELAXED load (an acquire load would invalidate L1 on every poll); one acquire fence after the exit.
// `side` runs on thread 32 between the two CTA barriers, i.e. while thread 0 polls: work that needs the whole CTA to be
// past its shared-memory accesses but not the other CTAs (the next phase's weight copy) costs nothing there.
struct NoSideJob { __device__ __forceinline__ void operator()() const {} };
template <typename Side = NoSideJob>
__device__ __forceinline__ unsigned grid_sync(unsigned* ctr, unsigned target, int* progress = nullptr, int ph = 0, Side side = Side()) {
  target += gridDim.x;
  // this thread's global writes (generic proxy) -> later TMA reads by other CTAs (async proxy): the proxy fence sits on the
  // writer side of the release/acquire chain, where it overlaps the store drain instead of delaying the next tile copy
  asm volatile("fence.proxy.async.global;" ::: "memory");
  __syncthreads();
  if (threadIdx.x == 0) {
    if (progress) progress[blockIdx.x] = ph;
    red_release_add(ctr, 1u);
    unsigned spins = 0;
    while (ld_relaxed(ctr) < target) {
      if (++spins > (1u << 24)) {
        printf("ptts: grid barrier timeout (cta %d target %u seen %u ph %d)\n", (int)blockIdx.x, target, ld_relaxed(ctr), ph);
        if (progress) for (int i = 0; i < (int)gridDim.x; i++) if (((volatile int*)progress)[i] != ph) printf("ptts:   cta %d is at phase %d\n", i, ((volatile int*)progress)[i]);
        __trap();
      }
    }
    fence_acq_rel_gpu();
  } else if (threadIdx.x == 32) {
    side();
  }
  __syncthreads();
  return target;
}

__device__ __forceinline__ void prof_mark(long long* prof, int slot) {
  if (prof != nullptr && threadIdx.x == 0) prof[slot] = clock64();
}

// ---- shared-memory context ----------------------------------------------------------------------
struct Smem {
  uint64_t* bars;   // [2] tile buffers
  float* stats;     // [64] (mean, rstd) per row of the staged tile
  float* part;      // [8][32][2] per-warp partial row sums (ln_stats.cuh)
  float* cvec;      // [2][32] folded-LN vectors c1, c2 of the current task's features
  const uint4* wbuf; // this CTA's weight slice of the current (or next) GEMM task, staged by TMA (B-fragment order)
  bf16* tile0;      // activation tile buffers (tile_of(sm, buf)), row pitch = H + 8
  unsigned char* scratch;  // start of the tile region (aliased by the K-reduction buffer and by attention)
  uint32_t parity;  // bit i: parity to wait for on bars[i] (bit 2: the weight barrier)
  long long* prof;  // CTA 0 / thread 0 timestamps of the current phase (nullptr = off)
  int pitch;
  int nbuf;
};

__device__ __forceinline__ bf16* tile_of(const Smem& sm, int buf) { return sm.tile0 + (size_t)buf * 32 * sm.pitch; }

// TMA-stage one K-chunk of the activations into tile buffer `buf` (called by all threads).  The fused kernel keeps its
// transient activations in global memory as TILE IMAGES: [chunk][32 rows][H + 8] with the shared-memory row pitch, so a
// chunk is ONE contiguous bulk copy.  (The TMA front end takes ~29 ns per cp.async.bulk: 32 per-row copies cost 0.95 us
// of issue time on the critical path of every GEMM phase; tools/ubench.cu, profiles/r01_step_phases.md.)
__device__ __forceinline__ void stage_tile(Smem& sm, int buf, const bf16* img, int M, bool mark) {
  __syncthreads();  // every generic-proxy access to the buffer (ldmatrix, reduction scratch) is done
  if (threadIdx.x == 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // tile buffer: generic accesses (above barrier) before the async write
    const uint32_t bytes = (uint32_t)(M * sm.pitch * 2);
    mbar_expect_tx(&sm.bars[buf], bytes);
    bulk_g2s(tile_of(sm, buf), img, bytes, &sm.bars[buf]);
    if (mark) prof_mark(sm.prof, 5);  // copy issued
  }
}
__device__ __forceinline__ void wait_tile(Smem& sm, int buf) {  // buf 0/1: activation tiles; 2: the weight buffer (bars[18])
  mbar_wait(&sm.bars[buf == 2 ? 18 : buf], (sm.parity >> buf) & 1u);
  sm.parity ^= (1u << buf);
}

// L2 prefetch job issued by one thread right after the CTA's first tile copy (never before: fence.proxy.async waits
// for outstanding bulk operations of the CTA, prefetches included)
struct PrefetchJob {
  const char* w; int N, K, nt;       // this CTA's weight slices of a [N][K] matrix packed with nt n-tiles per task (nullptr = none)
  const char* v; uint32_t v_bytes;   // folded-LayerNorm vectors riding along (nullptr = none)
  int kv_layer, pos;                 // kv_layer >= 0: also prefetch this layer's K/V rows up to cache position pos (warps 4-7)
};

struct GemmDesc {
  const bf16* X; int64_t x_chunk_stride;  // activation tile images: chunk c (H columns) at X + c * x_chunk_stride
  const uint4* W;
  int N, K;
  const float* c1; const float* c2;  // folded LayerNorm vectors (ln_stats.cuh) or nullptr
  int epi;
  const bf16* R;
  void* Y; int64_t ldy;
  int y_chunk; int64_t y_chunk_stride;  // feature n of row r lives at (n / y_chunk) * y_chunk_stride + r * ldy + n % y_chunk
  PrefetchJob pf;
  int ph;  // phase index (weight staging of the next job)
};

// bytes of this CTA's weight slice for a GEMM (first task only) -> L2, one layer ahead
__device__ __forceinline__ void prefetch_slice(const char* w, int N, int K, int nt) {
  const int ntasks = N / (8 * nt);
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x)
    l2_prefetch(w + (size_t)task * nt * K * 16, (uint32_t)(nt * K * 16));
}

// L2 prefetch of the K/V rows this CTA's warps will read in the coming attention phases of layer l.
__device__ __forceinline__ void prefetch_kv(const StepParams& p, int l, int pos) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp < 4) return;  // warps 0-3 go straight to the GEMM (warp 0 issues its TMA tile copies)
  const int pw = warp - 4;  // 4 prefetching warps cover the CTA's items
  if (pos > 0 && lane == 0) {
    const char* kc = p.self_kv + p.self_layer_stride * l;
    const size_t vofs = (size_t)p.B * p.nkv * p.Tmax * HD * 2;
    for (int it = blockIdx.x + gridDim.x * pw; it < p.B * p.nkv; it += gridDim.x * 4) {  // (any warp may prefetch any item)
      const char* k = kc + (size_t)it * p.Tmax * HD * 2;  // [B][nkv][Tmax][64]: item-major
      l2_prefetch(k, (uint32_t)(pos * HD * 2));
      l2_prefetch(k + vofs, (uint32_t)(pos * HD * 2));
    }
  }
  if (lane == 0) {  // cross K/V of this CTA's items (item-major, contiguous)
    const char* ck = p.cross_kv + p.cross_layer_stride * l;
    const size_t vofs = (size_t)p.B * p.nckv * p.S * HD * 2;
    for (int it = blockIdx.x + gridDim.x * pw; it < p.B * p.nckv; it += gridDim.x * 4) {
      const char* k = ck + (size_t)it * p.S * HD * 2;
      l2_prefetch(k, (uint32_t)(p.S * HD * 2));
      l2_prefetch(k + vofs, (uint32_t)(p.S * HD * 2));
    }
  }
}

__device__ __forceinline__ void issue_prefetch(const StepParams& p, const PrefetchJob& j) {
  if (j.kv_layer >= 0) prefetch_kv(p, j.kv_layer, j.pos);
  if (threadIdx.x == ST_THREADS - 32) {
    if (j.w != nullptr) prefetch_slice(j.w, j.N, j.K, j.nt);
    if (j.v != nullptr) l2_prefetch(j.v, j.v_bytes);
  }
}

// ---- weight staging -------------------------------------------------------------------------------
// The weight slice of a GEMM task (NT n-tiles x K, contiguous in the packed layout) is ONE bulk copy into shared
// memory, issued as soon as the buffer is free -- i.e. right after the previous task's MMA loop, a full phase before
// it is needed -- so the weights cross HBM/L2 -> SM during the previous epilogue and the device-wide barrier instead of
// on the critical path (registers could keep only ~32 KB of loads in flight per SM: 2-3 us for a 64 KB slice).
constexpr int WBAR = 18;  // sm.bars index of the weight mbarrier (0,1: tiles; 2..17: attention rings)

struct WeightJob { const char* src; uint32_t bytes; };

// matrix of GEMM phase `ph` (not an attention phase): packed weights, N, K and n-tiles per task
__device__ __forceinline__ void gemm_matrix(const StepParams& p, int ph, const char*& W, int& N, int& K, int& nt) {
  const int l = ph >> 3, sub = (ph >= 8 * p.L) ? 8 : (ph & 7);
  const char* lb = p.blob + p.layer0 + p.layer_stride * (l < p.L ? l : p.L - 1);
  const int H = p.H;
  switch (sub) {
    case 0: W = lb + p.wqkv; N = p.qkv_rows; K = H; nt = p.nt_qkv; break;
    case 2: W = lb + p.wo; N = H; K = H; nt = p.nt_h; break;
    case 3: W = lb + p.wqc; N = H; K = H; nt = p.nt_h; break;
    case 5: W = lb + p.woc; N = H; K = H; nt = p.nt_h; break;
    case 6: W = lb + p.fc1; N = p.F; K = H; nt = p.nt_fc1; break;
    case 7: W = lb + p.fc2; N = H; K = p.F; nt = p.nt_h; break;
    default: W = p.blob + p.heads; N = p.K * p.V; K = H; nt = p.nt_heads; break;
  }
}

// Called by all threads AFTER a __syncthreads() that retired every reader of the weight buffer.
__device__ __forceinline__ void issue_weights_thread(const StepParams& p, Smem& sm, int ph, int task) {  // ONE thread
  const char* W; int N, K, nt;
  gemm_matrix(p, ph, W, N, K, nt);
  if (task >= N / (8 * nt)) return;
  const uint32_t bytes = (uint32_t)nt * (uint32_t)K * 16u;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  mbar_expect_tx(&sm.bars[WBAR], bytes);
  bulk_g2s(const_cast<uint4*>(sm.wbuf), W + (size_t)task * bytes, bytes, &sm.bars[WBAR]);
}
__device__ __forceinline__ void issue_weights(const StepParams& p, Smem& sm, int ph, int task) {
  if (threadIdx.x == 0) issue_weights_thread(p, sm, ph, task);
}
__device__ __forceinline__ bool is_attn_phase(const StepParams& p, int ph) { return ph < 8 * p.L && ((ph & 7) == 1 || (ph & 7) == 4); }

// All tasks (n-blocks of 8*NT features) of one linear layer assigned to this CTA.  M = B <= 32 rows.
// (A single run-time-nt body was tried to shrink the instruction footprint: the predicated inner loop cost more than
// the smaller code saved -- 1.39 vs 1.32 ms/step.)
template <int NT>
__device__ __forceinline__ void gemm_tasks(const StepParams& p, Smem& sm, const GemmDesc& d) {
  constexpr int NT_MAX = NT, nt = NT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int M = p.B, H = p.H;
  const int Kc = d.K < H ? d.K : H;
  const int n_chunks = d.K / Kc;
  const int kt_per_chunk = Kc >> 5, KT = d.K >> 5;
  constexpr int FB = 8 * NT;
  constexpr int RS = (FB & 15) ? FB : FB + 8;  // row stride of the reduction scratch (floats): conflict-free for the epilogue reads
  const int ntasks = d.N / FB;
  // single-chunk GEMMs with two tile buffers keep the staged tile (and its row statistics) resident across this CTA's
  // tasks: the K-reduction scratch then lives in the second buffer (lm heads: 2-3 tasks per CTA)
  const bool resident = (n_chunks == 1 && sm.nbuf > 1);
  const int er = threadIdx.x >> 3, ec = threadIdx.x & 7;  // epilogue: this thread owns row er, feature ec of every n-tile
  for (int task = blockIdx.x; task < ntasks; task += gridDim.x) {
    const bool fresh = !resident || task == (int)blockIdx.x;
    const int n0 = task * FB;
    // activations: chunk 0 and, when double-buffered, chunk 1 (the weights were requested a phase ago)
    if (fresh) stage_tile(sm, 0, d.X, M, true);
    if (sm.nbuf > 1 && n_chunks > 1) stage_tile(sm, 1, d.X + d.x_chunk_stride, M, false);
    auto y_offset = [&](int n) -> size_t {
      const int yc = n / d.y_chunk;
      return (size_t)yc * d.y_chunk_stride + (size_t)er * d.ldy + (n - yc * d.y_chunk);
    };
    unsigned short rraw = 0;  // residual of this thread's first output (raw bf16 bits: no dependent instruction until the epilogue)
    if (d.epi == EPI_RESIDUAL && er < M) rraw = *reinterpret_cast<const unsigned short*>(d.R + y_offset(n0 + ec));
    float cv = 0.f;  // this task's c1 | c2 (one element per thread): requested now, parked in shared memory after the MMA loop
    if (d.c1 != nullptr && (int)threadIdx.x < 2 * FB) cv = (threadIdx.x < FB ? d.c1 : d.c2)[n0 + threadIdx.x % FB];
    if (task == (int)blockIdx.x) issue_prefetch(p, d.pf);  // next layer's weights / this layer's K/V -> L2, off the critical path
    float acc[2][NT_MAX][4];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int j = 0; j < NT_MAX; j++)
#pragma unroll
        for (int e = 0; e < 4; e++) acc[a][j][e] = 0.f;

    const int lrow = (lane & 7) + ((lane >> 3) & 1) * 8;
    const int lcol = (lane >> 4) * 8;
    for (int c = 0; c < n_chunks; c++) {
      const int buf = (sm.nbuf > 1) ? (c & 1) : 0;
      if (c > 0 && sm.nbuf == 1) stage_tile(sm, 0, d.X + c * d.x_chunk_stride, M, false);
      if (fresh) wait_tile(sm, buf);
      if (c == 0) prof_mark(sm.prof, 1);
      if (fresh && d.c1 != nullptr) {  // row sums on the tensor cores (LN-fused GEMMs are single-chunk: K == H)
        RowStatFrag rst;
        row_stat_zero(rst);
        row_stat_pass(rst, tile_of(sm, buf), sm.pitch, kt_per_chunk, warp, lane);
        row_stat_store(rst, sm.part, warp, lane);
      }
      if (c == 0) {
        prof_mark(sm.prof, 2);
        wait_tile(sm, 2);  // this task's weights (bars[WBAR]: parity bit 2)
      }
      const bf16* xs = tile_of(sm, buf);
      for (int kt = warp; kt < kt_per_chunk; kt += ST_WARPS) {  // K split over the 8 warps
        const uint4* wk = sm.wbuf + ((size_t)(c * kt_per_chunk + kt)) * 32 + lane;
        uint4 w[NT_MAX];
#pragma unroll
        for (int j = 0; j < NT_MAX; j++)
          if (j < nt) w[j] = wk[(size_t)j * KT * 32];
        uint32_t a[2][2][4];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
          for (int j = 0; j < 2; j++) ldmatrix_x4s(a[mt][j], xs + (size_t)(mt * 16 + lrow) * sm.pitch + kt * 32 + j * 16 + lcol);
#pragma unroll
        for (int j = 0; j < NT_MAX; j++) {
          if (j < nt) {
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
              mma_bf16s(acc[mt][j], a[mt][0], w[j].x, w[j].y);
              mma_bf16s(acc[mt][j], a[mt][1], w[j].z, w[j].w);
            }
          }
        }
      }
      if (sm.nbuf > 1 && c + 2 < n_chunks) stage_tile(sm, buf, d.X + (c + 2) * d.x_chunk_stride, M, false);
    }
    prof_mark(sm.prof, 3);
    if (d.c1 != nullptr && (int)threadIdx.x < 2 * FB) sm.cvec[(threadIdx.x < FB ? 0 : 32) + (threadIdx.x % FB)] = cv;  // read two barriers later
    __syncthreads();
    // the weight buffer is free: request the next task's slice of this matrix (the NEXT phase's first slice is requested
    // from inside the device-wide barrier, see the phase loop)
    if (task + (int)gridDim.x < ntasks) issue_weights(p, sm, d.ph, task + gridDim.x);
    if (fresh && d.c1 != nullptr) row_stat_finalize(sm.part, d.K, M, p.eps, sm.stats);  // (mean, rstd) per row; read in the epilogue
    float* red = reinterpret_cast<float*>(resident ? tile_of(sm, 1) : tile_of(sm, 0));  // [8][32][RS], in an idle tile buffer
    {
      const int g = lane >> 2, t = lane & 3;
#pragma unroll
      for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int j = 0; j < NT_MAX; j++) {
          if (j < nt) {
            float* base = red + ((size_t)warp * 32 + mt * 16 + g) * RS + j * 8 + 2 * t;
            *reinterpret_cast<float2*>(base) = make_float2(acc[mt][j][0], acc[mt][j][1]);
            *reinterpret_cast<float2*>(base + 8 * RS) = make_float2(acc[mt][j][2], acc[mt][j][3]);
          }
        }
    }
    __syncthreads();
    if (er < M) {
      const float mean = sm.stats[2 * er], rstd = sm.stats[2 * er + 1];
#pragma unroll
      for (int j = 0; j < NT_MAX; j++) {
        if (j < nt) {
          const int cidx = j * 8 + ec;
          float v = 0.f;
#pragma unroll
          for (int w = 0; w < ST_WARPS; w++) v += red[((size_t)w * 32 + er) * RS + cidx];
          if (d.c1 != nullptr) v = rstd * (v - mean * sm.cvec[cidx]) + sm.cvec[32 + cidx];
          v = DT<bf16>::rnd(v);
          if (d.epi == EPI_ACT) v = apply_act(v, p.act);
          const size_t yo = y_offset(n0 + cidx);
          if (d.epi == EPI_RESIDUAL) v = (j == 0 ? __bfloat162float(__ushort_as_bfloat16(rraw)) : DT<bf16>::to_f(d.R[yo])) + v;
          if (d.epi == EPI_F32) reinterpret_cast<float*>(d.Y)[yo] = v;
          else reinterpret_cast<bf16*>(d.Y)[yo] = __float2bfloat16_rn(v);
        }
      }
    }
    prof_mark(sm.prof, 4);
  }
}

__device__ __forceinline__ void run_gemm(const StepParams& p, Smem& sm, const GemmDesc& d, int nt) {
  switch (nt) {
    case 1: gemm_tasks<1>(p, sm, d); break;
    case 2: gemm_tasks<2>(p, sm, d); break;
    case 3: gemm_tasks<3>(p, sm, d); break;
    default: gemm_tasks<4>(p, sm, d); break;
  }
}

// Attention phase: one warp per (batch row, kv head) item, TMA-staged K/V.  Items are dealt round-robin over
// CTAs first (item i -> CTA i % grid, warp i / grid) so all 148 SMs pull K/V, 3-4 warps each at Mini/B=32.
__device__ __forceinline__ void attn_phase(const StepParams& p, Smem& sm, const AttnArgs& a, int nkv, int pos, uint32_t& att_parity, int ph) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* region = sm.scratch + (size_t)warp * attn_decode_smem_per_warp<bf16>();
  uint64_t* bars = sm.bars + 2 + 2 * warp;
  const int items = p.B * nkv;
  const int pair = warp >> 1, part = warp & 1;  // two warps per item split its cached keys
  float* xch = reinterpret_cast<float*>(sm.scratch + (size_t)ST_WARPS * attn_decode_smem_per_warp<bf16>()) + pair * 128;
  __syncthreads();  // the tile / reduction scratch of the previous GEMM phase is dead
  for (int it = blockIdx.x + gridDim.x * pair; it < items; it += gridDim.x * (ST_WARPS / 2))
    attention_decode_item_warp<bf16>(a, it / nkv, it % nkv, pos, region, bars, lane, att_parity, part, 2, xch, pair + 1);
}

// one CTA per (utterance, codebook) row (sample_core.cuh): 288 rows over 148 CTAs at Mini / batch 32
template <int ITEMS>
__device__ __noinline__ void sample_phase(const SampleArgs& sa, const ptts_gen_params& gp, int BK, int cur_len) {
  sample_all_rows_cta<ITEMS>(sa, gp, (int)blockIdx.x, (int)gridDim.x, BK, cur_len);
}

template <int ITEMS>
__global__ void __launch_bounds__(ST_THREADS, 1) decode_step_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Ctrl* ctrl = p.sa.ctrl;
  if (p.prof != nullptr && blockIdx.x == 0 && threadIdx.x == 0) p.prof[(size_t)(8 * p.L + 2) * 8 + 3] = clock64();  // kernel entry
  if (ctrl->active == 0) return;  // generation finished: the rest of the enqueued steps are no-ops
  const int cur_len = ctrl->cur_len;
  const unsigned gen = (unsigned)ctrl->launch_gen;
  const int pos = p.P + cur_len - 1;  // cache position of the token being fed
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = p.H;

  Smem sm;
  sm.bars = reinterpret_cast<uint64_t*>(smem_raw);
  sm.stats = reinterpret_cast<float*>(smem_raw + 256);
  sm.part = reinterpret_cast<float*>(smem_raw + 512);
  sm.cvec = reinterpret_cast<float*>(smem_raw + 2560);
  sm.scratch = smem_raw + ST_HEADER;
  sm.wbuf = reinterpret_cast<const uint4*>(smem_raw + ST_HEADER + p.wbuf_offset);
  sm.pitch = H + 8;
  sm.nbuf = p.nbuf;
  sm.tile0 = reinterpret_cast<bf16*>(sm.scratch);
  sm.parity = 0;
  sm.prof = nullptr;
  if (tid == 0) {
    mbar_init(&sm.bars[0], 1);
    mbar_init(&sm.bars[1], 1);
    mbar_init(&sm.bars[WBAR], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  attention_decode_init_warp(sm.bars + 2 + 2 * warp, lane);  // per-warp K/V ring barriers: header bytes [16, 144)
  uint32_t att_parity = 0;
  // rows >= B of the tile buffers are never written by the TMA copies: clear them once
  for (int i = tid; i < (int)(p.tile_region_bytes / 16); i += ST_THREADS) reinterpret_cast<uint4*>(sm.scratch)[i] = make_uint4(0, 0, 0, 0);
  unsigned* const bar_ctr = p.bar + (gen & 1u);
  unsigned bar_target = 0u;
  if (blockIdx.x == 0 && tid == 0) p.bar[(gen + 1u) & 1u] = 0u;  // the counter the NEXT launch will use
  __syncthreads();
  issue_weights(p, sm, 0, blockIdx.x);  // layer 0's qkv slice lands during the embedding phase

  const char* blob = p.blob;
  // (Several tokens per launch were tried -- loop here, one extra barrier per token: no gain, back-to-back cooperative
  // launches leave no measurable gap on the device.)
  long long* const prof0 = (p.prof != nullptr && blockIdx.x == 0) ? p.prof : nullptr;
  sm.prof = prof0;
  prof_mark(sm.prof, 0);
  // ---- phase 0: embeddings + L2 prefetch of layer 0 ----
  if (tid == 0) {
    const char* lb = blob + p.layer0;
    prefetch_slice(lb + p.wqkv, p.qkv_rows, H, p.nt_qkv);
    l2_prefetch(lb + p.c_qkv, (uint32_t)p.qkv_rows * 8); l2_prefetch(lb + p.c_qc, (uint32_t)H * 8); l2_prefetch(lb + p.c_fc1, (uint32_t)p.F * 8);
    prefetch_slice(lb + p.wo, H, H, p.nt_h);
    prefetch_slice(lb + p.wqc, H, H, p.nt_h);
    prefetch_slice(lb + p.woc, H, H, p.nt_h);
    prefetch_slice(lb + p.fc1, p.F, H, p.nt_fc1);
    prefetch_slice(lb + p.fc2, H, p.F, p.nt_h);
  }
  {
    const bf16* tables = reinterpret_cast<const bf16*>(blob + p.embed);
    const bf16* postab = p.rope ? nullptr : reinterpret_cast<const bf16*>(blob + p.pos);
    const int cpr = (H + ST_THREADS - 1) / ST_THREADS;  // column chunks per row: (row, chunk) items spread over all CTAs
    for (int it = blockIdx.x; it < p.B * cpr; it += gridDim.x) {
      const int b = it / cpr, c = (it - b * cpr) * ST_THREADS + tid;
      if (c >= H) continue;
      float ev[16];
#pragma unroll
      for (int k = 0; k < 16; k++)  // all K gathers in flight, then the left-to-right rounded sum
        if (k < p.K) ev[k] = __bfloat162float(tables[((size_t)k * (p.V + 1) + p.sa.cur_ids[b * p.K + k]) * H + c]);
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < 16; k++)
        if (k < p.K) v = (k == 0) ? ev[k] : DT<bf16>::rnd(v + ev[k]);
      if (postab != nullptr) v = DT<bf16>::rnd(v + __bfloat162float(postab[(size_t)pos * H + c]));
      p.x[(size_t)b * sm.pitch + c] = __float2bfloat16_rn(v);
    }
  }
  prof_mark(sm.prof, 6);
  bar_target = grid_sync(bar_ctr, bar_target);
  prof_mark(sm.prof, 7);

  // One loop over all 8L+1 dependent phases (single call site per phase type keeps code size and registers sane).
#pragma unroll 1
  for (int ph = 0; ph <= 8 * p.L; ph++) {
    const int l = ph >> 3, sub = (ph == 8 * p.L) ? 8 : (ph & 7);
    sm.prof = prof0 ? prof0 + (size_t)(ph + 1) * 8 : nullptr;
    prof_mark(sm.prof, 0);
    const char* lb = blob + p.layer0 + p.layer_stride * (l < p.L ? l : p.L - 1);
    if (sub == 1 || sub == 4) {
      AttnArgs a{};
      a.ldo = sm.pitch; a.out = p.attn; a.ctrl = nullptr; a.B = p.B; a.nh = p.nh; a.q_len = 1;
      a.past_from_ctrl = 0; a.past_len = pos; a.prefix = p.P;
      a.rope = p.rope; a.rope_cos = blob + p.rope_cos; a.rope_sin = blob + p.rope_sin; a.scale = p.scale;
      if (sub == 1) {  // self-attention over the cache (+ append of the new K/V row)
        a.q = p.qkv; a.ldq = p.qkv_rows; a.q_col0 = 0;
        a.knew = p.qkv; a.vnew = p.qkv; a.ldkv = p.qkv_rows; a.k_col0 = p.nh * HD; a.v_col0 = (p.nh + p.nkv) * HD;
        char* kc = p.self_kv + p.self_layer_stride * l;
        a.kcache = kc; a.vcache = kc + (size_t)p.B * p.nkv * p.Tmax * HD * 2;
        a.kv_b_stride = (int64_t)p.nkv * p.Tmax * HD; a.kv_h_stride = (int64_t)p.Tmax * HD; a.kv_t_stride = HD;
        a.key_mask = p.prompt_mask; a.mask_len = p.P; a.mask_ld = p.P;
        a.nkv = p.nkv; a.cross = 0; a.kv_len = 0; a.kv_capacity = p.Tmax;
      } else {         // cross-attention over the cached encoder K/V
        a.q = p.qc; a.ldq = H; a.q_col0 = 0; a.knew = nullptr; a.vnew = nullptr;
        char* ck = p.cross_kv + p.cross_layer_stride * l;
        a.kcache = ck; a.vcache = ck + (size_t)p.B * p.nckv * p.S * HD * 2;
        a.kv_b_stride = (int64_t)p.nckv * p.S * HD; a.kv_h_stride = (int64_t)p.S * HD; a.kv_t_stride = HD;
        a.key_mask = p.enc_mask; a.mask_len = p.S; a.mask_ld = p.S;
        a.nkv = p.nckv; a.cross = 1; a.kv_len = p.S; a.kv_capacity = p.S;
      }
      attn_phase(p, sm, a, a.nkv, pos, att_parity, ph);
    } else {
      // Activations live in tile images (row pitch H + 8, see stage_tile).  Each GEMM phase also pulls the matrix the
      // SAME phase of the next layer will use into L2 (PrefetchJob), so the HBM stream is spread over the layer;
      // folded-LayerNorm vectors ride along, and the qkv phase prefetches this layer's K/V rows.
      const bool last = (l + 1 >= p.L);
      const char* nb = lb + p.layer_stride;
      const int64_t img = (int64_t)32 * sm.pitch;  // elements per tile image
      const int ld = sm.pitch;
      GemmDesc g{};
      g.y_chunk = 1 << 30; g.y_chunk_stride = 0; g.x_chunk_stride = img;
      g.pf.w = nullptr; g.pf.v = nullptr; g.pf.kv_layer = -1; g.pf.pos = pos; g.ph = ph;
      int nt = p.nt_h;
      auto set_pf = [&](int64_t w, int N, int K, int pnt, int64_t v, int vn) {
        if (last) return;
        g.pf.w = nb + w; g.pf.N = N; g.pf.K = K; g.pf.nt = pnt;
        if (vn > 0) { g.pf.v = nb + v; g.pf.v_bytes = (uint32_t)vn * 8; }
      };
      switch (sub) {
        case 0:  // qkv = LN1(x) Wqkv^T
          g.X = p.x; g.W = reinterpret_cast<const uint4*>(lb + p.wqkv); g.N = p.qkv_rows; g.K = H;
          g.c1 = reinterpret_cast<const float*>(lb + p.c_qkv); g.c2 = g.c1 + p.qkv_rows;
          g.epi = EPI_STORE; g.R = nullptr; g.Y = p.qkv; g.ldy = p.qkv_rows;
          nt = p.nt_qkv;
          set_pf(p.wqkv, p.qkv_rows, H, p.nt_qkv, p.c_qkv, p.qkv_rows);
          if (last) { g.pf.w = blob + p.heads; g.pf.N = p.K * p.V; g.pf.K = H; g.pf.nt = p.nt_heads; g.pf.v = blob + p.c_heads; g.pf.v_bytes = (uint32_t)(p.K * p.V) * 8; }
          g.pf.kv_layer = l;
          break;
        case 2:  // x += attn Wo^T
          g.X = p.attn; g.W = reinterpret_cast<const uint4*>(lb + p.wo); g.N = H; g.K = H; g.c1 = nullptr; g.c2 = nullptr;
          g.epi = EPI_RESIDUAL; g.R = p.x; g.Y = p.x; g.ldy = ld;
          set_pf(p.wo, H, H, p.nt_h, 0, 0);
          break;
        case 3:  // q_cross = LN2(x) Wq^T
          g.X = p.x; g.W = reinterpret_cast<const uint4*>(lb + p.wqc); g.N = H; g.K = H;
          g.c1 = reinterpret_cast<const float*>(lb + p.c_qc); g.c2 = g.c1 + H;
          g.epi = EPI_STORE; g.R = nullptr; g.Y = p.qc; g.ldy = H;
          set_pf(p.wqc, H, H, p.nt_h, p.c_qc, H);
          break;
        case 5:  // x += attn Wo_cross^T
          g.X = p.attn; g.W = reinterpret_cast<const uint4*>(lb + p.woc); g.N = H; g.K = H; g.c1 = nullptr; g.c2 = nullptr;
          g.epi = EPI_RESIDUAL; g.R = p.x; g.Y = p.x; g.ldy = ld;
          set_pf(p.woc, H, H, p.nt_h, 0, 0);
          break;
        case 6:  // h = act(LN3(x) W1^T), written as F/H tile images
          g.X = p.x; g.W = reinterpret_cast<const uint4*>(lb + p.fc1); g.N = p.F; g.K = H;
          g.c1 = reinterpret_cast<const float*>(lb + p.c_fc1); g.c2 = g.c1 + p.F;
          g.epi = EPI_ACT; g.R = nullptr; g.Y = p.hbuf; g.ldy = ld; g.y_chunk = H; g.y_chunk_stride = img;
          nt = p.nt_fc1;
          set_pf(p.fc1, p.F, H, p.nt_fc1, p.c_fc1, p.F);
          break;
        case 7:  // x += h W2^T
          g.X = p.hbuf; g.W = reinterpret_cast<const uint4*>(lb + p.fc2); g.N = H; g.K = p.F; g.c1 = nullptr; g.c2 = nullptr;
          g.epi = EPI_RESIDUAL; g.R = p.x; g.Y = p.x; g.ldy = ld;
          set_pf(p.fc2, H, p.F, p.nt_h, 0, 0);
          break;
        default:  // final LayerNorm + K lm heads -> f32 logits [B, K*V]
          g.X = p.x; g.W = reinterpret_cast<const uint4*>(blob + p.heads); g.N = p.K * p.V; g.K = H;
          g.c1 = reinterpret_cast<const float*>(blob + p.c_heads); g.c2 = g.c1 + p.K * p.V;
          g.epi = EPI_F32; g.R = nullptr; g.Y = p.logits; g.ldy = (int64_t)p.K * p.V;
          nt = p.nt_heads;
          break;
      }
      run_gemm(p, sm, g, nt);
    }
    prof_mark(sm.prof, 6);
    if (ph < 8 * p.L) {
      // while thread 0 polls the barrier, thread 32 requests this CTA's weight slice of the next phase when that is a GEMM
      // (every reader of the weight buffer -- and of the attention scratch it may alias -- is past the CTA barrier by then)
      const int wph = is_attn_phase(p, ph + 1) ? -1 : ph + 1;
      bar_target = grid_sync(bar_ctr, bar_target, p.progress, ph + 1, [&]() { if (wph >= 0) issue_weights_thread(p, sm, wph, blockIdx.x); });
    }
    prof_mark(sm.prof, 7);
  }
  bar_target = grid_sync(bar_ctr, bar_target);
  sm.prof = prof0 ? prof0 + (size_t)(8 * p.L + 2) * 8 : nullptr;  // tail row: barrier / sampling / barrier
  prof_mark(sm.prof, 0);
  if (p.do_sample_phase) {
    const ptts_gen_params gp = *p.sa.gen;
    const int BK = p.B * p.K;
    sample_phase<ITEMS>(p.sa, gp, BK, cur_len);
    prof_mark(sm.prof, 1);
    bar_target = grid_sync(bar_ctr, bar_target);
    prof_mark(sm.prof, 2);
  }
  if (blockIdx.x == 0 && tid == 0) {
    if (p.do_sample_phase) {
      const int n = atomicAdd(&ctrl->n_unfinished, 0);
      ctrl->cur_len = cur_len + 1;
      ctrl->active = (n > 0) ? 1 : 0;
      ctrl->steps_run += 1;
      ctrl->n_unfinished = 0;
    }
    ctrl->launch_gen = (int)(gen + 1u);
  }
}

// ---- host side ----------------------------------------------------------------------------------
int step_smem_bytes(const StepParams& p) {
  return (int)(ST_HEADER + p.tile_region_bytes);
}

int launch_decode_step(const StepParams& p, int grid, cudaStream_t st) {
  const int smem = step_smem_bytes(p);
  void* args[] = {(void*)&p};
  const void* fn;
  if (p.sample_items <= 1) fn = (const void*)decode_step_kernel<1>;
  else if (p.sample_items <= 5) fn = (const void*)decode_step_kernel<5>;
  else fn = (const void*)decode_step_kernel<9>;
  static int attr_done[3] = {0, 0, 0};
  const int fi = p.sample_items <= 1 ? 0 : (p.sample_items <= 5 ? 1 : 2);
  if (!attr_done[fi]) {
    PTTS_CHECK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));  // (+ 256 B of static shared memory: the sampler scratch)
    attr_done[fi] = 1;
  }
  PTTS_CHECK_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(ST_THREADS), args, (size_t)smem, st));
  return PTTS_OK;
}

}  // namespace ptts
