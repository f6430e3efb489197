// dac_tc.cu -- DAC decoder convolutions as tcgen05 implicit GEMMs (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces the cuDNN Conv1d / ConvTranspose1d calls inside dac.model.DAC.decode (reached from
// parler_tts/dac_wrapper/modeling_dac.py:139; arithmetic per transformers/models/dac/modeling_dac.py:173-262).
// Roofline: tensor pipe -- 1.608 GFLOP per code frame (SURVEY 8d); the SIMT path in dac.cu is FMA-bound.
//
// One CTA computes a 128 (time) x N_TILE (output channel) tile:
//   D[t, co] = sum_{tap j} sum_{ci} X[t + off_j, ci] * W[j][co][ci]
//   * activations are channels-last bf16 [B][T][C]: the K dimension (ci) is contiguous, so the A tile of tap j is
//     a plain 3-D TMA box {64 ci, 128 t, 1 b} at row offset off_j; rows outside [0, T) are ZERO-FILLED by the TMA
//     unit, which is exactly the convolution's zero padding (and the channel tail when Cin % 64 != 0);
//   * weights are pre-packed [tap][Cout][Cin] (K-major), B tile = box {64 ci, N_TILE co, 1 tap};
//   * both land in shared memory with the 128-byte swizzle the UMMA smem descriptors expect;
//   * warp 0 (one thread) is the TMA producer, warp 1 (one thread) issues tcgen05.mma (M=128, N=N_TILE, K=16) with
//     the accumulator in tensor memory, tcgen05.commit releases smem stages / signals the epilogue;
//   * warps 2-5 read the accumulator with tcgen05.ld (32 lanes x 32 columns per instruction), add the bias and the
//     residual, and write the raw tensor and/or snake(x) for the NEXT layer, so every layer's A operand is a
//     ready-to-MMA bf16 tensor (snake is x + sin^2(alpha x)/(alpha + 1e-9), rounded like torch's bf16 ops).
// ConvTranspose1d(k = 2s, stride s) = s output phases x 2 taps (dac.cu explains the mapping).
#include <cuda.h>

#include <mutex>
#include <vector>

#include "common.cuh"
#include "dac.h"

namespace ptts {

constexpr int TC_M = 128;      // time rows per tile (UMMA M)
constexpr int TC_K = 64;       // ci per pipeline stage (one 128-byte swizzle row of bf16)
constexpr int TC_STAGES = 2;   // 2 stages x <= 48 KB: two CTAs per SM, so one tile's epilogue overlaps the other's MMA mainloop
constexpr int TC_THREADS = 192;

__device__ __forceinline__ uint32_t tc_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_mbar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem(b)), "r"(n)); }
__device__ __forceinline__ void tc_mbar_expect(uint64_t* b, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem(b)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void tc_mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok, spins = 0;
  do {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(tc_smem(b)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 24)) { printf("ptts: dac_tc mbarrier timeout (cta %d,%d,%d thread %d)\n", (int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x); __trap(); }
  } while (!ok);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
               ::"r"(tc_smem(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(tc_smem(bar)) : "memory");
}
// UMMA shared-memory descriptor, K-major, 128-byte swizzle: 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
               ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                 "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
                 "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct ConvTcArgs {
  int Cin, Cout, Tin, Tout, q_count;
  int n_taps, off_base, off_step, wt_base, wt_step;
  int n_phase, wt_phase_step, o_mul, o_add, o_phase_step;
  int n_tile, tmem_cols;
  const bf16* bias;        // [Cout]
  const bf16* res;         // residual (raw tensor, [B][Tout][Cout]) or nullptr
  bf16* out_raw;           // raw result or nullptr
  bf16* out_act;           // snake_{alpha_next}(result) for the next layer or nullptr
  const bf16* alpha_next;  // [Cout]
};

// kDown: Conv1d(k = 2s, stride s = off_step, padding s/2), the encoder's downsampling.  map_x then views the input as rows of s
// samples ([B][Tin/s][s*Cin]); tap j of output q reads sample s*q + j - s/2 = row q + (j + s/2)/s - 1 at column ((j + s/2) % s)*Cin,
// so every (tap, 64-channel chunk) is still one TMA box and the box's zero fill outside [0, Tin/s) is the convolution's padding.
template <bool kDown>
__global__ void __launch_bounds__(TC_THREADS, 2)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const ConvTcArgs p) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int a_bytes = TC_M * TC_K * 2, b_bytes = p.n_tile * TC_K * 2;
  const int stage_bytes = (a_bytes + b_bytes + 1023) & ~1023;
  unsigned char* stages = smem;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + TC_STAGES * stage_bytes);
  uint64_t* empty = full + TC_STAGES;
  uint64_t* acc_full = empty + TC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  bf16* chan = reinterpret_cast<bf16*>(smem + TC_STAGES * stage_bytes + 128);  // [3][n_tile]: bias | alpha | 1/(alpha+1e-9)

  const int phase = blockIdx.z % p.n_phase, b = blockIdx.z / p.n_phase;
  const int q0 = blockIdx.x * TC_M, n0 = blockIdx.y * p.n_tile;
  const int k_chunks = (p.Cin + TC_K - 1) / TC_K;
  const int n_iter = p.n_taps * k_chunks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_STAGES; s++) { tc_mbar_init(&full[s], 1); tc_mbar_init(&empty[s], 1); }
    tc_mbar_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
  }
  if (warp == 2) {  // TMEM allocation (and later deallocation) by one warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      for (int it = 0; it < n_iter; it++) {
        const int s = it % TC_STAGES, use = it / TC_STAGES;
        if (use > 0) tc_mbar_wait(&empty[s], (use - 1) & 1);
        const int j = it / k_chunks, kc = it - j * k_chunks;
        unsigned char* a_dst = stages + (size_t)s * stage_bytes;
        unsigned char* b_dst = a_dst + a_bytes;
        tc_mbar_expect(&full[s], (uint32_t)(a_bytes + b_bytes));
        if constexpr (kDown) {
          const int sh = j + (p.off_step >> 1);
          tma_load_3d(a_dst, &map_x, (sh % p.off_step) * p.Cin + kc * TC_K, q0 + sh / p.off_step - 1, b, &full[s]);
        } else {
          tma_load_3d(a_dst, &map_x, kc * TC_K, q0 + p.off_base + j * p.off_step, b, &full[s]);
        }
        tma_load_3d(b_dst, &map_w, kc * TC_K, n0, p.wt_base + phase * p.wt_phase_step + j * p.wt_step, &full[s]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ===== MMA issuer =====
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
      for (int it = 0; it < n_iter; it++) {
        const int s = it % TC_STAGES, use = it / TC_STAGES;
        tc_mbar_wait(&full[s], use & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_addr = tc_smem(stages + (size_t)s * stage_bytes);
        const uint32_t b_addr = a_addr + a_bytes;
        const uint64_t da = umma_desc_sw128(a_addr), db = umma_desc_sw128(b_addr);
#pragma unroll
        for (int k = 0; k < TC_K / 16; k++)  // 32 bytes (16 bf16) further along K inside the swizzled row: +2 in the address field
          umma_bf16(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (it > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty[s]);  // smem stage reusable once these MMAs have read it
      }
      umma_commit(acc_full);     // accumulator complete
    }
  } else {
    // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
    // per-channel constants of this N tile -> shared memory while the mainloop runs: bias, alpha, 1/(alpha+1e-9)
    {
      const int et = threadIdx.x - 64;  // 0..127
      for (int c = et; c < p.n_tile; c += 128) {
        chan[c] = p.bias[n0 + c];
        if (p.out_act != nullptr) {
          const bf16 a = p.alpha_next[n0 + c];
          chan[p.n_tile + c] = a;
          chan[2 * p.n_tile + c] = __float2bfloat16_rn(1.0f / __bfloat162float(__float2bfloat16_rn(__bfloat162float(a) + 1e-9f)));
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // epilogue warps only
    }
    tc_mbar_wait(acc_full, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int q = q0 + row;
    const int to = q * p.o_mul + p.o_add + phase * p.o_phase_step;
    const bool row_ok = (q < p.q_count) && (to >= 0) && (to < p.Tout);
    const size_t orow = ((size_t)b * p.Tout + (row_ok ? to : 0)) * p.Cout + n0;
    const __nv_bfloat162* bias2 = reinterpret_cast<const __nv_bfloat162*>(chan);
    const __nv_bfloat162* alpha2 = reinterpret_cast<const __nv_bfloat162*>(chan + p.n_tile);
    const __nv_bfloat162* inv2 = reinterpret_cast<const __nv_bfloat162*>(chan + 2 * p.n_tile);
    for (int c0 = 0; c0 < p.n_tile; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, v);  // warp-collective: all lanes take part
      if (row_ok) {
        // native bf16x2 arithmetic: every op rounds to bf16 exactly like the torch ops it replaces
        __nv_bfloat162 r2[16];
#pragma unroll
        for (int i = 0; i < 16; i++) {
          // conv output = bf16(acc + bias) (one rounding of the fp32 sum)
          const float2 bb = __bfloat1622float2(bias2[(c0 >> 1) + i]);
          r2[i] = __floats2bfloat162_rn(__uint_as_float(v[2 * i]) + bb.x, __uint_as_float(v[2 * i + 1]) + bb.y);
        }
        if (p.res != nullptr) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const uint4 u = *reinterpret_cast<const uint4*>(p.res + orow + c0 + 2 * i);
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
            for (int e = 0; e < 4; e++) r2[i + e] = __hadd2(h[e], r2[i + e]);
          }
        }
        if (p.out_raw != nullptr) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<uint4*>(p.out_raw + orow + c0 + 2 * i) = *reinterpret_cast<const uint4*>(&r2[i]);
        }
        if (p.out_act != nullptr) {
          __nv_bfloat162 s2[16];
#pragma unroll
          for (int i = 0; i < 16; i++) {
            const __nv_bfloat162 ax = __hmul2(alpha2[(c0 >> 1) + i], r2[i]);          // alpha * x
            const float2 axf = __bfloat1622float2(ax);
            const __nv_bfloat162 sn = __floats2bfloat162_rn(__sinf(axf.x), __sinf(axf.y));  // sin(.)  (MUFU; bf16 result)
            const __nv_bfloat162 sq = __hmul2(sn, sn);                                  // ^2
            s2[i] = __hadd2(r2[i], __hmul2(inv2[(c0 >> 1) + i], sq));                   // x + inv * sin^2
          }
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<uint4*>(p.out_act + orow + c0 + 2 * i) = *reinterpret_cast<const uint4*>(&s2[i]);
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
  }
  return fn;
}
// 3-D bf16 tensor [d2][d1][d0] (d0 contiguous), box {64, box1, 1}, 128-byte swizzle, zero OOB fill
static int encode_map(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t box1);

// A decode issues ~60 convolution launches over the SAME buffers and shapes every time (the workspace and the weight blob are
// caller-owned and stable): encode each tensor map once and reuse it (cuTensorMapEncodeTiled is a few microseconds of host time
// per call, 60 of them sat between the launches of every decode -- profiles/r01_dac_ncu_full.md).
struct MapKey { const void* base; uint64_t d0, d1, d2; uint32_t box1; };
struct MapEntry { MapKey k; CUtensorMap m; };
static int make_map(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t box1) {
  static std::mutex mu;
  static std::vector<MapEntry> cache;
  std::lock_guard<std::mutex> lock(mu);
  for (const MapEntry& e : cache)
    if (e.k.base == base && e.k.d0 == d0 && e.k.d1 == d1 && e.k.d2 == d2 && e.k.box1 == box1) { *m = e.m; return PTTS_OK; }
  if (int e = encode_map(m, base, d0, d1, d2, box1)) return e;
  if (cache.size() >= 4096) cache.clear();   // many distinct (B, T) shapes over a long-lived process: start over
  cache.push_back(MapEntry{MapKey{base, d0, d1, d2, box1}, *m});
  return PTTS_OK;
}
static int encode_map(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t box1) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(PTTS_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {d0 * 2, d0 * d1 * 2};
  cuuint32_t box[3] = {(cuuint32_t)TC_K, box1, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(PTTS_ECUDA, "cuTensorMapEncodeTiled failed (%d) dims %llu %llu %llu box1 %u", (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, box1);
  return PTTS_OK;
}

template <bool kDown>
static int launch_tc(const CUtensorMap& mx, const CUtensorMap& mw, const ConvTcArgs& p, dim3 grid, cudaStream_t st) {
  const int stage_bytes = (TC_M * TC_K * 2 + p.n_tile * TC_K * 2 + 1023) & ~1023;
  const size_t smem = (size_t)TC_STAGES * stage_bytes + 128 + 3 * 256 * 2;
  static bool attr = false;
  if (!attr) {
    PTTS_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel<kDown>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
    attr = true;
  }
  conv_tc_kernel<kDown><<<grid, TC_THREADS, smem, st>>>(mx, mw, p);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

bool conv_tc_supported(int Cin, int Cout) {
  return Cin % 8 == 0 && Cin >= 64 && Cout % 32 == 0 && Cout >= 32;  // row pitch multiple of 16 B; epilogue works in 32-column chunks
}
int conv_tc_ntile(int Cout) {
  if (Cout % 256 == 0) return 256;
  if (Cout % 192 == 0) return 192;
  if (Cout % 128 == 0) return 128;
  if (Cout % 96 == 0) return 96;
  if (Cout % 64 == 0) return 64;
  return 32;
}

// x: [B][Tin][Cin] bf16, w: [taps_total][Cout][Cin] bf16
int launch_conv_tc(const ConvArgs& a, const void* w_kmajor, int taps_total, const void* alpha_next, void* out_raw, void* out_act, int B, cudaStream_t st) {
  ConvTcArgs p{};
  p.Cin = a.Cin; p.Cout = a.Cout; p.Tin = a.Tin; p.Tout = a.Tout; p.q_count = a.q_count;
  p.n_taps = a.n_taps; p.off_base = a.off_base; p.off_step = a.off_step; p.wt_base = a.wt_base; p.wt_step = a.wt_step;
  p.n_phase = a.n_phase; p.wt_phase_step = a.wt_phase_step; p.o_mul = a.o_mul; p.o_add = a.o_add; p.o_phase_step = a.o_phase_step;
  p.n_tile = conv_tc_ntile(a.Cout);
  p.tmem_cols = p.n_tile <= 32 ? 32 : (p.n_tile <= 64 ? 64 : (p.n_tile <= 128 ? 128 : 256));
  p.bias = (const bf16*)a.bias; p.res = (const bf16*)a.res; p.out_raw = (bf16*)out_raw; p.out_act = (bf16*)out_act; p.alpha_next = (const bf16*)alpha_next;
  CUtensorMap mx, mw;
  if (int e = make_map(&mx, a.x, (uint64_t)a.Cin, (uint64_t)a.Tin, (uint64_t)B, TC_M)) return e;
  if (int e = make_map(&mw, w_kmajor, (uint64_t)a.Cin, (uint64_t)a.Cout, (uint64_t)taps_total, (uint32_t)p.n_tile)) return e;
  dim3 grid((a.q_count + TC_M - 1) / TC_M, a.Cout / p.n_tile, B * a.n_phase);
  return launch_tc<false>(mx, mw, p, grid, st);
}

bool conv_tc_down_supported(int Cin, int Cout) { return Cin % TC_K == 0 && conv_tc_supported(Cin, Cout); }

// x: [B][Tin][Cin] bf16 (Tin % s == 0), w: [2s][Cout][Cin] bf16 -> [B][Tin/s][Cout]
int launch_conv_tc_down(const void* x, const void* w_kmajor, const void* bias, const void* alpha_next, void* out_raw, void* out_act,
                        int Cin, int Cout, int Tin, int s, int B, cudaStream_t st) {
  PTTS_REQUIRE(conv_tc_down_supported(Cin, Cout) && s >= 2 && s % 2 == 0 && Tin % s == 0, "conv_tc_down: Cin=%d Cout=%d s=%d Tin=%d unsupported", Cin, Cout, s, Tin);
  ConvTcArgs p{};
  p.Cin = Cin; p.Cout = Cout; p.Tin = Tin; p.Tout = Tin / s; p.q_count = Tin / s;
  p.n_taps = 2 * s; p.off_base = 0; p.off_step = s; p.wt_base = 0; p.wt_step = 1;
  p.n_phase = 1; p.wt_phase_step = 0; p.o_mul = 1; p.o_add = 0; p.o_phase_step = 0;
  p.n_tile = conv_tc_ntile(Cout);
  p.tmem_cols = p.n_tile <= 32 ? 32 : (p.n_tile <= 64 ? 64 : (p.n_tile <= 128 ? 128 : 256));
  p.bias = (const bf16*)bias; p.res = nullptr; p.out_raw = (bf16*)out_raw; p.out_act = (bf16*)out_act; p.alpha_next = (const bf16*)alpha_next;
  CUtensorMap mx, mw;
  if (int e = make_map(&mx, x, (uint64_t)s * Cin, (uint64_t)(Tin / s), (uint64_t)B, TC_M)) return e;
  if (int e = make_map(&mw, w_kmajor, (uint64_t)Cin, (uint64_t)Cout, (uint64_t)(2 * s), (uint32_t)p.n_tile)) return e;
  dim3 grid((p.q_count + TC_M - 1) / TC_M, Cout / p.n_tile, B);
  return launch_tc<true>(mx, mw, p, grid, st);
}

// weight repack for the tensor-core path: Conv1d [co][ci][k] / ConvTranspose1d [ci][co][k] -> [k][co][ci] bf16
template <typename S>
__global__ void pack_conv_kmajor_kernel(const S* src, bf16* dst, int d0, int d1, int k, int transposed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = (int64_t)d0 * d1 * k;
  if (i >= n) return;
  const int kk = (int)(i % k);
  const int b1 = (int)((i / k) % d1), b0 = (int)(i / ((int64_t)k * d1));
  const int ci = transposed ? b0 : b1, co = transposed ? b1 : b0;
  const int Cin = transposed ? d0 : d1, Cout = transposed ? d1 : d0;
  float v;
  if constexpr (sizeof(S) == 2) v = __bfloat162float(src[i]); else v = src[i];
  dst[((size_t)kk * Cout + co) * Cin + ci] = __float2bfloat16_rn(v);
}
int pack_conv_kmajor(const void* src, int src_dtype, void* dst, int d0, int d1, int k, int transposed, cudaStream_t st) {
  const int64_t n = (int64_t)d0 * d1 * k;
  const int blocks = (int)((n + 255) / 256);
  if (src_dtype == PTTS_BF16) pack_conv_kmajor_kernel<bf16><<<blocks, 256, 0, st>>>((const bf16*)src, (bf16*)dst, d0, d1, k, transposed);
  else pack_conv_kmajor_kernel<float><<<blocks, 256, 0, st>>>((const float*)src, (bf16*)dst, d0, d1, k, transposed);
  PTTS_LAUNCH_CHECK();
  return PTTS_OK;
}

}  // namespace ptts
