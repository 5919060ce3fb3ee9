// Implicit-GEMM conv1d / linear kernel for sm_100a.
//
// Replaces, on time-major bf16 activations, every dense contraction of the hot path:
//   CausalConv1d k=3          speech/cosyvoice/flow/decoder.py:36-62
//   res_conv / final_proj 1x1 speech/matcha/models/components/decoder.py:54,60 ; flow/decoder.py:403
//   to_q/k/v, to_out, FF      speech/matcha/models/components/transformer.py:196-204,109-126
//   WNConv1d k=7 dilated, k=1 dac-vae/model.py:128-130,343,364
//   WNConvTranspose1d         dac-vae/model.py:255-262 (two-tap polyphase form, N = stride*Cout)
// with the surrounding row-local work fused into the epilogue (bias, LeakyReLU / exact GELU / LayerNorm+Mish /
// tanh, time-embedding add, residual add, length masking, and a second bf16 output holding LayerNorm / Snake /
// copy of the result for the next GEMM).
//
// Structure: persistent CTAs (one per SM), warp-specialised:
//   warp 0  TMEM allocator, then TMA producer  (A: 128 rows x 64 ch box per tap via a 3-D map, OOB rows -> 0 = conv zero padding;
//                          B: block_n x 64 weight box), multi-stage mbarrier ring
//   warp 1  tcgen05.mma issuer (one lane), fp32 accumulators in TMEM, double buffered
//   warps 2-17 epilogue (512 threads): warp w owns TMEM lanes 32*(w%4).. (= 32 output rows) and every 4th
//              16-column chunk; accumulators are pulled into registers in one burst and the TMEM stage is
//              released immediately, LayerNorm statistics are combined across the 4 column groups through smem
#include <cstdio>
#include <string>
#include <unordered_map>

#include "kernels.h"
#include "profiler.h"
#include "ptx.cuh"

namespace ls {
namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;
constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
#ifndef CONV_PRODUCER_WARPS
#define CONV_PRODUCER_WARPS 3
#endif
constexpr int kProducerWarps = CONV_PRODUCER_WARPS;  // warp 0: activation boxes; warps 1..: weight boxes (one thread each)
constexpr int kWeightProducers = kProducerWarps - 1;
static_assert(kProducerWarps >= 2, "need one activation and at least one weight producer");
constexpr int kMmaWarp = kProducerWarps;
constexpr int kFirstEpiWarp = kProducerWarps + 1;
constexpr int kThreads = kFirstEpiWarp * 32 + kEpiThreads;
constexpr int kMaxStages = 16;
#ifndef CONV_DETAIL_TL
#define CONV_DETAIL_TL 0  // development aid: 1 = per-tap stamps of the MMA warp, 2 = per-load stamps of weight producer 1
#endif
#ifndef CONV_DUAL_RESIDENT
#define CONV_DUAL_RESIDENT 0
#endif
#ifndef CONV_HALO_A_STAGES
#define CONV_HALO_A_STAGES 3  // activation stages of a streamed-weight halo launch with more than one K block
#endif

constexpr int kRedBytes = 2 * 2 * 4 * kBlockM * 8;  // [tile parity][phase][column group][row] float2
constexpr int kSmemBudget = 157 * 1024;             // for the operand rings

struct TileCoord {
  int b, mt, nt;
};

__device__ __forceinline__ TileCoord decode_tile(int tile, int m_tiles, int n_tiles) {
  TileCoord c;
  c.nt = tile % n_tiles;
  const int rest = tile / n_tiles;
  c.mt = rest % m_tiles;
  c.b = rest / m_tiles;
  return c;
}

__device__ __forceinline__ bool tile_skipped(const ConvGemmParams& p, const TileCoord& c) {
  if (p.lengths == nullptr) return false;
  const long long need = (long long)p.lengths[c.b] * p.m_len_mul + p.m_len_add + p.skip_halo;
  return (long long)c.mt * kBlockM >= need;
}

// 16 consecutive output columns of one row.  state: 2 store values, 1 store zeros, 0 drop.
struct ChunkStore {
  long long valid, alloc;
  int n_store;
  bool row_in;
  __device__ __forceinline__ int state(long long flat, int width = 16) const {
    if (!row_in || flat < 0) return 0;
    if (flat + width <= valid) return 2;
    if (flat + width <= alloc) return 1;
    return 0;
  }
  __device__ __forceinline__ void f32(float* base, long long flat, int n, const float (&u)[16]) const {
    const int st = state(flat, min(16, n_store - n));
    if (st == 0 || n >= n_store) return;
    if (n + 16 <= n_store) {
      float4* d = reinterpret_cast<float4*>(base + flat);
#pragma unroll
      for (int g = 0; g < 4; ++g)
        d[g] = st == 2 ? make_float4(u[4 * g], u[4 * g + 1], u[4 * g + 2], u[4 * g + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (n + i < n_store) base[flat + i] = st == 2 ? u[i] : 0.f;
    }
  }
  __device__ __forceinline__ void bf16(__nv_bfloat16* base, long long flat, int n, const float (&u)[16]) const {
    const int st = state(flat, min(16, n_store - n));
    if (st == 0 || n >= n_store) return;
    if (n + 16 <= n_store) {
      uint4* d = reinterpret_cast<uint4*>(base + flat);
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (st == 2) {
          v.x = LS_PACK_H2(u[8 * g + 0], u[8 * g + 1]);
          v.y = LS_PACK_H2(u[8 * g + 2], u[8 * g + 3]);
          v.z = LS_PACK_H2(u[8 * g + 4], u[8 * g + 5]);
          v.w = LS_PACK_H2(u[8 * g + 6], u[8 * g + 7]);
        }
        d[g] = v;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (n + i < n_store) reinterpret_cast<uint16_t*>(base)[flat + i] = LS_CVT_H_BITS(st == 2 ? u[i] : 0.f);
    }
  }
};

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }


// ---- coalesced global access for the epilogue --------------------------------------------------------------------
// TMEM hands every thread one output ROW (32x32b loads), so a direct store makes each warp instruction touch 32
// different rows with 16 B each: partial sectors and 32 lines per instruction (measured: 7 B/clk per SM).  Each warp
// therefore transposes one 16-column chunk at a time through a private 2 KB staging buffer: rows are written/read by
// their owner threads, global memory is accessed with consecutive lanes on consecutive 16 B pieces of a row
// (fp32: 8 rows x 64 B per instruction, bf16: 16 rows x 32 B), i.e. whole 32 B sectors only.
// 16 B units are XOR-swizzled so that both access patterns are bank-conflict free.
constexpr int kStageBytesPerWarp = 3072;  // [0,2048): fp32 chunk / residual transposes, [2048,3072): 16-bit out1 chunk
constexpr int kStageB16Off = 2048;
constexpr int kStageOut0H = 1024;  // 16-bit out0 chunk (the 16-bit residual transposes use [0,1024))
__device__ __forceinline__ int stg_f32(int row, int unit) { return row * 64 + ((unit ^ ((row >> 1) & 3)) << 4); }
__device__ __forceinline__ int stg_b16(int row, int unit) { return row * 32 + ((unit ^ ((row >> 2) & 1)) << 4); }

// geometry of one warp's 32 rows for the coalesced side
struct WarpRows {
  long long t_base;        // time index of the warp's first row inside the batch item
  long long out_ld, out_shift, valid, alloc;
  int M;
  __device__ __forceinline__ int state(int rr, int n, long long* flat) const {  // same rule as ChunkStore::state
    const long long t = t_base + rr;
    const long long f = t * out_ld + out_shift + n;
    *flat = f;
    if (t >= M || f < 0) return 0;
    if (f + 16 <= valid) return 2;
    if (f + 16 <= alloc) return 1;
    return 0;
  }
};

// Residual (addend) chunk, fetched coalesced into registers: fp32 = 4 x 16 B per lane (8 rows x 64 B per instruction),
// bf16 = 2 x 16 B per lane (16 rows x 32 B).  Issued before the accumulator is waited for, so the global latency
// overlaps the MMA wait and the other chunks instead of sitting in the middle of the chunk's dependent chain.
struct AddRegs {
  uint4 v[4];
};
// 16-bit element kinds of out0 / addend: OUT_BF16 = this build's operand type (bf16, or fp16 in the fp16-operand build),
// OUT_F16 = IEEE half whatever the operand type (the DAC decoder's residual stream: 11 significand bits, so 15 chained
// residual additions cost nothing measurable, where bf16 would)
template <int kKind>
__device__ __forceinline__ uint32_t pack_kind(float lo, float hi) {
  return kKind == OUT_F16 ? pack_f16x2(lo, hi) : LS_PACK_H2(lo, hi);
}
template <int kKind>
__device__ __forceinline__ void unpack_kind(uint32_t w, float& lo, float& hi) {
  if (kKind == OUT_F16) unpack_f16x2(w, lo, hi);
  else LS_UNPACK_H2(w, lo, hi);
}
template <bool kF32>
__device__ __forceinline__ void fetch_chunk(int lane, const WarpRows& wr, int n, const void* base, AddRegs& a) {
  if (kF32) {
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
      const int rr = ps * 8 + (lane >> 2), seg = lane & 3;
      long long flat;
      a.v[ps] = make_uint4(0u, 0u, 0u, 0u);
      if (wr.state(rr, n, &flat) == 2) a.v[ps] = *reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(base) + flat + seg * 4);
    }
  } else {
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {
      const int rr = ps * 16 + (lane >> 1), seg = lane & 1;
      long long flat;
      a.v[ps] = make_uint4(0u, 0u, 0u, 0u);
      if (wr.state(rr, n, &flat) == 2) a.v[ps] = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + flat + seg * 8);
    }
  }
}
// v (this thread's row, 16 fp32) += the fetched chunk, transposed through the warp's staging buffer
template <int kKind>
__device__ __forceinline__ void apply_chunk(uint8_t* stg, int lane, const AddRegs& a, float (&v)[16]) {
  if (kKind == OUT_F32) {
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
      const int rr = ps * 8 + (lane >> 2), seg = lane & 3;
      *reinterpret_cast<uint4*>(stg + stg_f32(rr, seg)) = a.v[ps];
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float4 t = *reinterpret_cast<const float4*>(stg + stg_f32(lane, u));
      v[4 * u] += t.x, v[4 * u + 1] += t.y, v[4 * u + 2] += t.z, v[4 * u + 3] += t.w;
    }
  } else {
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {
      const int rr = ps * 16 + (lane >> 1), seg = lane & 1;
      *reinterpret_cast<uint4*>(stg + stg_b16(rr, seg)) = a.v[ps];
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const uint4 t = *reinterpret_cast<const uint4*>(stg + stg_b16(lane, u));
      const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float lo, hi;
        unpack_kind<kKind>(w[k], lo, hi);
        v[8 * u + 2 * k] += lo;
        v[8 * u + 2 * k + 1] += hi;
      }
    }
  }
  __syncwarp();
}

// store this thread's row chunk (16 fp32 values) coalesced, as fp32 or bf16; rows in the zero-fill range get zeros
template <int kKind>
__device__ __forceinline__ void store_chunk(uint8_t* stg, int lane, const WarpRows& wr, int n, void* base,
                                            const float (&v)[16]) {
  if (kKind == OUT_F32) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<float4*>(stg + stg_f32(lane, u)) = make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]);
    __syncwarp();
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) {
      const int rr = ps * 8 + (lane >> 2), seg = lane & 3;
      long long flat;
      const int st = wr.state(rr, n, &flat);
      if (st != 0) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        if (st == 2) a = *reinterpret_cast<const float4*>(stg + stg_f32(rr, seg));
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + flat + seg * 4) = a;
      }
    }
  } else {
#pragma unroll
    for (int u = 0; u < 2; ++u)
      *reinterpret_cast<uint4*>(stg + stg_b16(lane, u)) =
          make_uint4(pack_kind<kKind>(v[8 * u], v[8 * u + 1]), pack_kind<kKind>(v[8 * u + 2], v[8 * u + 3]),
                     pack_kind<kKind>(v[8 * u + 4], v[8 * u + 5]), pack_kind<kKind>(v[8 * u + 6], v[8 * u + 7]));
    __syncwarp();
#pragma unroll
    for (int ps = 0; ps < 2; ++ps) {
      const int rr = ps * 16 + (lane >> 1), seg = lane & 1;
      long long flat;
      const int st = wr.state(rr, n, &flat);
      if (st != 0) {
        uint4 a = make_uint4(0u, 0u, 0u, 0u);
        if (st == 2) a = *reinterpret_cast<const uint4*>(stg + stg_b16(rr, seg));
        *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(base) + flat + seg * 8) = a;
      }
    }
  }
  __syncwarp();
}

// Dense outputs ([B][M][N], whole rows stored) leave through TMA instead: the staging layouts above ARE TMA's 64 B
// (fp32) / 32 B (bf16) swizzle patterns, so the warp writes its 32 rows x 16 columns once and one lane hands the
// buffer to cp.async.bulk.tensor (box 16 x 32; rows past M are clipped by the tensor map).  Rows past the valid
// length are written as zeros.  Before a staging region is rewritten, the bulk group that last read it must be done:
// kPending = how many younger groups of this lane may still be in flight at that point.  kOff = the staging region of a
// 16-bit chunk: kStageB16Off for out1, kStageOut0H for a 16-bit out0 (so that out0 and out1 alternate between two
// regions like an fp32 out0 and out1 do, and neither is the region the 16-bit residual transposes use).
template <int kKind, int kPending, int kOff = kStageB16Off>
__device__ __forceinline__ void store_chunk_tma(uint8_t* stg, int lane, const CUtensorMap* map, int n, int t_base, int b,
                                                bool row_valid, const float (&v)[16]) {
  constexpr bool kF32 = kKind == OUT_F32;
  if (lane == 0) bulk_wait_read<kPending>();
  __syncwarp();
  if (kF32) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
      *reinterpret_cast<float4*>(stg + stg_f32(lane, u)) =
          row_valid ? make_float4(v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    uint8_t* sb = stg + kOff;
#pragma unroll
    for (int u = 0; u < 2; ++u)
      *reinterpret_cast<uint4*>(sb + stg_b16(lane, u)) =
          row_valid ? make_uint4(pack_kind<kKind>(v[8 * u], v[8 * u + 1]), pack_kind<kKind>(v[8 * u + 2], v[8 * u + 3]),
                                 pack_kind<kKind>(v[8 * u + 4], v[8 * u + 5]), pack_kind<kKind>(v[8 * u + 6], v[8 * u + 7]))
                    : make_uint4(0u, 0u, 0u, 0u);
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    tma_store_3d(map, kF32 ? stg : stg + kOff, n, t_base, b);
    bulk_commit();
  }
}

template <int kKind, int kOff = kStageB16Off>
__device__ __forceinline__ void store_chunk_tma_p(bool one_pending, uint8_t* stg, int lane, const CUtensorMap* map, int n,
                                                  int t_base, int b, bool row_valid, const float (&v)[16]) {
  if (one_pending) store_chunk_tma<kKind, 1, kOff>(stg, lane, map, n, t_base, b, row_valid, v);
  else store_chunk_tma<kKind, 0, kOff>(stg, lane, map, n, t_base, b, row_valid, v);
}

// The epilogue mode (activation, outputs, residual, time embedding) is a template parameter for the combinations the
// engines launch (-1 = decided at run time: the generic instance, used by everything else).  A specialised instance
// carries a fraction of the generic epilogue's code: the unrolled epilogue is executed once per tile, so its
// footprint in the instruction cache -- not its instruction count -- is what the generic instance pays for.
template <int kAct, int kOut0, int kOut1, int kAdd, int kTemb>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                 const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapOut0,
                 const __grid_constant__ CUtensorMap mapOut1, const __grid_constant__ ConvGemmParams p,
                 const int tmem_cols, const int acc_stride) {
  const int act = kAct >= 0 ? kAct : p.act;
  const int out0_dtype = kOut0 >= 0 ? kOut0 : p.out0_dtype;
  const int out1_mode = kOut1 >= 0 ? kOut1 : p.out1_mode;
  const int add_dtype = kAdd >= 0 ? kAdd : (p.addend_dtype == ADD_GEMM ? (int)ADD_GEMM : p.addend ? p.addend_dtype : (int)OUT_NONE);  // OUT_NONE: no residual
  const bool has_temb = kTemb >= 0 ? kTemb != 0 : p.temb != nullptr;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // Two operand rings.  A stage: one (128 + halo)-row x 64-channel activation box (halo = (taps-1)*dil rows when
  // p.halo_mode, so the box is fetched ONCE per K block and every tap reads it through a row-shifted descriptor;
  // without halo_mode the box is 128 rows and is fetched per tap).  B stage: one block_n x 64 weight box per (K block, tap).
  const int a_bytes = ls_conv_a_stage_bytes(p.a_box_rows);
  const int b_bytes = p.block_n * kBlockK * 2;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)p.a_stages * a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)p.b_stages * b_bytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + kMaxStages;
  uint64_t* b_full = bars + 2 * kMaxStages;
  uint64_t* b_empty = bars + 3 * kMaxStages;
  uint64_t* tfull = bars + 4 * kMaxStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float2* red_base = reinterpret_cast<float2*>(bars + 128);  // 1 KB for the barriers + TMEM slot (keeps the staging
                                                             // buffers below aligned for TMA)
  uint8_t* stg_base = reinterpret_cast<uint8_t*>(red_base) + p.red_bytes;  // per-epilogue-warp transpose buffers
  float* svec = reinterpret_cast<float*>(stg_base + kEpiWarps * kStageBytesPerWarp);  // per-channel epilogue vectors

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = (p.M + kBlockM - 1) / kBlockM;
  const int n_tiles = p.N / p.block_n;
  const int total_tiles = p.B * m_tiles * n_tiles;
  const bool halo = p.halo_mode != 0;
  long long* tl = p.timeline ? p.timeline + (size_t)blockIdx.x * 64 : nullptr;
#define TL(i)                    \
  do {                           \
    if (tl) tl[(i)] = clock64(); \
  } while (0)
  if (threadIdx.x == 0) TL(0);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapA0);
    prefetch_tmap(&mapA1);
    prefetch_tmap(&mapW);
    if (p.res_kb > 0) {
      prefetch_tmap(&p.res_a0);
      prefetch_tmap(&p.res_a1);
      prefetch_tmap(&p.res_w);
    }
    if (p.tma_out) {
      prefetch_tmap(&mapOut0);
      prefetch_tmap(&mapOut1);
    }
  }
#ifndef CONV_L2_PREFETCH
#define CONV_L2_PREFETCH 1
#endif
  if (CONV_L2_PREFETCH && p.tag == 0 && warp == 1 && lane == 0) {
    // Flow-estimator launches: ask for the launch's weight boxes, spread over the CTAs of the grid, to be brought into L2
    // before the PDL wait (weights do not depend on the previous kernel).  Inside a solve they are cold (the estimator's
    // 212 MB of weights and > 1 GB of activations pass through the 126 MB L2 between two uses) and every CTA streams them
    // in the same order at about the same time: without this each box is a DRAM miss the whole grid waits for.
    const int per_tile = p.taps * p.kb_per_tap;
    const int n_boxes = per_tile * n_tiles;
    for (int j = blockIdx.x; j < n_boxes; j += gridDim.x) {
      const int nt = j / per_tile, r = j - nt * per_tile;
      const int tap = r / p.kb_per_tap, kb = r - tap * p.kb_per_tap;
      tma_prefetch_l2_2d(&mapW, kb * kBlockK, tap * p.N + nt * p.block_n);
    }
    for (int j = blockIdx.x; j < p.res_kb; j += gridDim.x) tma_prefetch_l2_2d(&p.res_w, j * kBlockK, 0);
  }
  if (warp == kMmaWarp && lane == 0) {
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], (p.dual && !p.b_resident) ? 2 : 1);  // dual mode: both MMA warps release a weight slot
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiThreads);
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    __syncwarp();
    tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
    tmem_relinquish();
  }
  // Per-channel vectors (bias, LayerNorm affine, Snake alpha) are weights: they are copied into shared memory here,
  // before the PDL wait.  Read from global in the epilogue, each of them is a dependent L2 round trip per chunk.
  {
    auto stage_vec = [&](int off, const float* src, int n) {
      if (off >= 0)
        for (int i = threadIdx.x; i < n; i += kThreads) svec[off + i] = __ldg(src + i);
    };
    stage_vec(p.sv_bias, p.bias, p.chan_mod);
    stage_vec(p.sv_p1a, p.p1_a, p.chan_mod);
    stage_vec(p.sv_p1b, p.p1_b, p.chan_mod);
    stage_vec(p.sv_lng, p.ln_g, p.N);
    stage_vec(p.sv_lnb, p.ln_b, p.N);
  }
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TL(1);
  pdl_wait();
  if (threadIdx.x == 0) TL(2);  // everything above overlapped the previous kernel's tail; activations are read only from here on

  // next tile of this CTA that is not all padding (every role walks the same sequence)
  auto next_tile = [&](int& cur) -> int {
    while (cur < total_tiles) {
      const int t = cur;
      cur += (int)gridDim.x;
      if (!tile_skipped(p, decode_tile(t, m_tiles, n_tiles))) return t;
    }
    return -1;
  };
  if (p.dual && warp < 2) {
    // ------------------------------------------------------------ dual mode: TMA producers
    // Thin layers are bound by the MMA-issuing THREAD (profiles/r02_timeline_conv_issue.log: ~600 clk of waits, descriptor
    // arithmetic and issue per tap for 4 MMAs that execute in ~350), so two warps issue, one per accumulator, on
    // alternating tiles (pairs).  Every weight box is fetched once per PAIR and released by both; each MMA warp has its
    // own activation stages [m*depth, (m+1)*depth).  Warp 0: activation boxes (and, streamed weights, those of both
    // tiles); warp 1: the weight boxes (and, once they are resident, the second tile's activation boxes).
    if (lane == 0) {
      const int depth = p.a_stages >> 1;
      const uint32_t a_tx = (uint32_t)p.a_box_rows * 128u;
      int cur = blockIdx.x, pair = 0, bs = 0;
      uint32_t bph = 0;
      int cnt[2] = {0, 0};
      for (;; ++pair) {
        int t[2];
        t[0] = next_tile(cur);
        if (t[0] < 0) break;
        t[1] = next_tile(cur);
        if (warp == 1 && (!p.b_resident || pair == 0)) {
          for (int kb = 0; kb < p.kb_per_tap; ++kb)
            for (int tap = 0; tap < p.taps; ++tap) {
              if (!p.b_resident) mbar_wait(&b_empty[bs], bph ^ 1);
              mbar_arrive_expect_tx(&b_full[bs], (uint32_t)b_bytes);
              tma_load_2d(smem_b + (size_t)bs * b_bytes, &mapW, &b_full[bs], kb * kBlockK, tap * p.N);
              if (++bs == p.b_stages) bs = 0, bph ^= 1;
            }
        }
        for (int kb = 0; kb < p.kb_per_tap; ++kb)
          for (int m = 0; m < 2; ++m) {
            if (t[m] < 0 || warp != (p.b_resident ? m : 0)) continue;
            const TileCoord tc = decode_tile(t[m], m_tiles, n_tiles);
            const int st = m * depth + cnt[m] % depth;
            mbar_wait(&a_empty[st], (uint32_t)(((cnt[m] / depth) & 1) ^ 1));
            uint8_t* sa = smem_a + (size_t)st * a_bytes;
            mbar_arrive_expect_tx(&a_full[st], a_tx);
            if (kb < p.kb_split)
              tma_load_3d(sa, &mapA0, &a_full[st], kb * kBlockK, tc.mt * kBlockM - p.pad, tc.b);
            else
              tma_load_3d(sa, &mapA1, &a_full[st], (kb - p.kb_split) * kBlockK, tc.mt * kBlockM - p.pad, tc.b);
            ++cnt[m];
          }
      }
    }
  } else if (p.dual && (warp == 2 || warp == kMmaWarp)) {
    // ------------------------------------------------------------ dual mode: MMA issuers (m = 0: kMmaWarp, m = 1: warp 2)
    const int m = warp == kMmaWarp ? 0 : 1;
    const int depth = p.a_stages >> 1;
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t idesc = make_idesc_bf16(kBlockM, p.block_n, false, false);
    const uint32_t d_tmem = tmem_u + (uint32_t)(m * acc_stride);
    int cur = blockIdx.x, bs = 0, cnt = 0;
    uint32_t bph = 0, acc_phase = 0;
    for (int pair = 0;; ++pair) {
      int te = next_tile(cur);
      te = __shfl_sync(0xffffffffu, te, 0);
      if (te < 0) break;
      int to = next_tile(cur);
      to = __shfl_sync(0xffffffffu, to, 0);
      cur = __shfl_sync(0xffffffffu, cur, 0);
      const bool lone = to < 0;  // the other warp has no tile in this pair: release the weight slots for it too
      if ((m == 0 ? te : to) < 0) break;
      const bool wait_b = !p.b_resident || pair == 0;
      mbar_wait(&tempty[m], acc_phase ^ 1);
      tc_fence_after();
      for (int kb = 0; kb < p.kb_per_tap; ++kb) {
        const int st = m * depth + cnt % depth;
        mbar_wait(&a_full[st], (uint32_t)((cnt / depth) & 1));
        tc_fence_after();
        int nk = kBlockK / 16;
        if (p.k_true > 0 && p.kb_split == p.kb_per_tap) nk = min(nk, (p.k_true - kb * kBlockK + 15) >> 4);
        const uint32_t a_addr = smem_u32(smem_a + (size_t)st * a_bytes);
        const uint32_t b_addr = smem_u32(smem_b);
        if (elect_one()) {
          int bl = p.b_resident ? kb * p.taps : bs;
          uint32_t bphl = bph;
          for (int tap = 0; tap < p.taps; ++tap) {
            if (wait_b) {
              mbar_wait(&b_full[bl], bphl);
              tc_fence_after();
            }
            const int shift = tap * p.dil;
            const uint64_t adesc = make_smem_desc_sw128(a_addr + (uint32_t)shift * 128u, p.halo_mode == 1 ? ((uint32_t)shift & 7u) : 0u);
            const uint64_t bdesc = make_smem_desc_sw128(b_addr + (uint32_t)bl * (uint32_t)b_bytes);
#pragma unroll
            for (int k = 0; k < kBlockK / 16; ++k)
              if (k < nk) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | tap | k) != 0 ? 1u : 0u);
            if (!p.b_resident) {
              umma_commit(&b_empty[bl]);
              if (lone) umma_commit(&b_empty[bl]);
            }
            if (++bl == p.b_stages) bl = 0, bphl ^= 1;
          }
          umma_commit(&a_empty[st]);
        }
        __syncwarp();
        for (int tap = 0; tap < p.taps; ++tap)
          if (++bs == p.b_stages) bs = 0, bph ^= 1;
        ++cnt;
      }
      if (elect_one()) umma_commit(&tfull[m]);
      __syncwarp();
      acc_phase ^= 1;
    }
  } else if (warp < kProducerWarps) {
    // ------------------------------------------------------------ TMA producers
    // A thread can start a TMA load only every ~500 clk (issue latency; profiles/micro/tma_bw3.cu) but different warps
    // overlap.  Warp 0 issues every activation box; warps 1.. share the weight boxes, warp w taking those whose sequence
    // number is (w-1) mod kWeightProducers.  Interleaving P producers over a ring of D stages keeps the parity waits
    // unambiguous only while P <= D (a producer is then never two uses ahead of the consumer): launch_conv_gemm
    // guarantees b_stages >= kWeightProducers, and the activation ring (1-3 stages) has a single producer.
    // (Separate warps, not lanes: a lane blocked in mbarrier.try_wait suspends its whole warp.)
    // (Issuing the weight boxes from 4 or 8 lanes of one warp instead was measured: no change.)
    if (lane == 0) {
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      int b_seq = 0, p_tile = 0;
      int a_seq = 0;
#if CONV_DETAIL_TL == 2
      int dn = 0;
#endif
      // Resident weights leave the weight producers idle after the first tile: the activation boxes are then shared
      // round-robin by ALL producer warps (one load per ~2 k clk and warp was what bounded the thin DAC layers once the MMA
      // issue loop had been fixed).  Safe while producers <= ring stages (see above); every producer tracks the ring.
      const bool a_share = p.b_resident && p.a_stages >= kProducerWarps;
      const uint32_t a_tx = (uint32_t)p.a_box_rows * 128u;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(tile, m_tiles, n_tiles);
        if (tile_skipped(p, tc)) continue;
        const int t0 = tc.mt * kBlockM;
        const int n0 = tc.nt * p.block_n;
        if (tl && warp == 0 && p_tile < 8) tl[56 + p_tile] = clock64();
        ++p_tile;
        for (int kb = 0; kb < p.kb_per_tap; ++kb) {
          for (int tap = 0; tap < p.taps; ++tap) {
            if (!halo || tap == 0) {
              if (warp == (a_share ? a_seq : 0)) {
                const int trow = t0 - p.pad + (halo ? 0 : tap * p.dil);
                mbar_wait(&a_empty[as], aph ^ 1);
                uint8_t* sa = smem_a + (size_t)as * a_bytes;
                mbar_arrive_expect_tx(&a_full[as], a_tx);
                if (kb < p.kb_split)
                  tma_load_3d(sa, &mapA0, &a_full[as], kb * kBlockK, trow, tc.b);
                else
                  tma_load_3d(sa, &mapA1, &a_full[as], (kb - p.kb_split) * kBlockK, trow, tc.b);
              }
              if (++a_seq == kProducerWarps) a_seq = 0;
              if (++as == p.a_stages) as = 0, aph ^= 1;
            }
            if (warp != 0 && (!p.b_resident || p_tile == 1)) {  // resident weights: fetched with the CTA's first tile only
              if (b_seq == warp - 1) {
#if CONV_DETAIL_TL == 2
                const bool dt = tl && warp == 1 && p_tile == 4 && dn < 7;
                if (dt) tl[8 + 3 * dn] = clock64();
#endif
                if (!p.b_resident) mbar_wait(&b_empty[bs], bph ^ 1);
#if CONV_DETAIL_TL == 2
                if (dt) tl[9 + 3 * dn] = clock64();
#endif
                mbar_arrive_expect_tx(&b_full[bs], (uint32_t)b_bytes);
                tma_load_2d(smem_b + (size_t)bs * b_bytes, &mapW, &b_full[bs], kb * kBlockK, tap * p.N + n0);
#if CONV_DETAIL_TL == 2
                if (dt) tl[10 + 3 * dn] = clock64(), ++dn;
#endif
              }
              if (++b_seq == kWeightProducers) b_seq = 0;
              if (++bs == p.b_stages) bs = 0, bph ^= 1;
            }
          }
        }
        // fused residual GEMM: its 128-row activation boxes and weight boxes follow in the same rings
        for (int kb2 = 0; kb2 < p.res_kb; ++kb2) {
          if (warp == 0) {
            mbar_wait(&a_empty[as], aph ^ 1);
            mbar_arrive_expect_tx(&a_full[as], (uint32_t)(kBlockM * 128));
            if (kb2 < p.res_split) tma_load_3d(smem_a + (size_t)as * a_bytes, &p.res_a0, &a_full[as], kb2 * kBlockK, t0, tc.b);
            else tma_load_3d(smem_a + (size_t)as * a_bytes, &p.res_a1, &a_full[as], (kb2 - p.res_split) * kBlockK, t0, tc.b);
          }
          if (++as == p.a_stages) as = 0, aph ^= 1;
          if (warp != 0) {
            if (b_seq == warp - 1) {
              mbar_wait(&b_empty[bs], bph ^ 1);
              mbar_arrive_expect_tx(&b_full[bs], (uint32_t)b_bytes);
              tma_load_2d(smem_b + (size_t)bs * b_bytes, &p.res_w, &b_full[bs], kb2 * kBlockK, n0);
            }
            if (++b_seq == kWeightProducers) b_seq = 0;
            if (++bs == p.b_stages) bs = 0, bph ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------ MMA issuer
    // The whole warp walks the tile / k loops in uniform control flow (every value below is warp-uniform); one elected
    // lane issues the MMAs and commits (see elect_one()).
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = make_idesc_bf16(kBlockM, p.block_n, false, false);
      int as = 0, bs = 0;
      uint32_t aph = 0, bph = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int n_it = 0, n_tile = 0;  // timeline aid
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(tile, m_tiles, n_tiles);
        if (__shfl_sync(0xffffffffu, (int)tile_skipped(p, tc), 0)) continue;
        mbar_wait(&tempty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + (uint32_t)(acc * acc_stride);
        if (halo && p.b_resident && n_tile > 0) {
          // Resident weights + halo box (the thin DAC layers): nothing to wait for inside a K block.  The lean form of the
          // loop below -- the issuing lane is bound by its own instruction latencies, every per-tap instruction counts
          // (DAC conv7 at C = 48: 362 us with this loop, 512 us through the general one).
          for (int kb = 0; kb < p.kb_per_tap; ++kb) {
            mbar_wait(&a_full[as], aph);
            tc_fence_after();
            int nk = kBlockK / 16;
            if (p.k_true > 0 && p.kb_split == p.kb_per_tap) nk = min(nk, (p.k_true - kb * kBlockK + 15) >> 4);
            const uint32_t a_addr = smem_u32(smem_a + (size_t)as * a_bytes);
            const uint32_t b_addr = smem_u32(smem_b) + (uint32_t)(kb * p.taps) * (uint32_t)b_bytes;
            if (tl && n_it < 24 && lane == 0) tl[8 + n_it] = clock64();
            n_it += p.taps;
            if (elect_one()) {
              for (int tap = 0; tap < p.taps; ++tap) {
                const int shift = tap * p.dil;
                const uint64_t adesc = make_smem_desc_sw128(a_addr + (uint32_t)shift * 128u, p.halo_mode == 1 ? ((uint32_t)shift & 7u) : 0u);
                const uint64_t bdesc = make_smem_desc_sw128(b_addr + (uint32_t)tap * (uint32_t)b_bytes);
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k)
                  if (k < nk) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | tap | k) != 0 ? 1u : 0u);
              }
              umma_commit(&a_empty[as]);
            }
            __syncwarp();
            if (++as == p.a_stages) as = 0, aph ^= 1;
          }
        } else if (halo) {
          // Halo box: the taps of a K block read ONE activation box, so the only waits inside a K block are for weight
          // boxes (none once the weights are resident).  All its taps are issued under ONE election -- the per-tap loop
          // overhead (barrier bookkeeping, election, warp sync) was several times the cost of the small-N MMAs it wrapped
          // (DAC conv7 at C = 96, streamed weights: 595 -> 524 us).
          for (int kb = 0; kb < p.kb_per_tap; ++kb) {
            mbar_wait(&a_full[as], aph);
            tc_fence_after();
            int nk = kBlockK / 16;
            if (p.k_true > 0 && p.kb_split == p.kb_per_tap) nk = min(nk, (p.k_true - kb * kBlockK + 15) >> 4);
            const uint32_t a_addr = smem_u32(smem_a + (size_t)as * a_bytes);
            const bool wait_b = !p.b_resident || n_tile == 0;
#if CONV_DETAIL_TL == 0
            if (tl && n_it < 24 && lane == 0) tl[8 + n_it] = clock64();
#endif
            n_it += p.taps;
            if (elect_one()) {
              int bl = bs;
              uint32_t bphl = bph;
              for (int tap = 0; tap < p.taps; ++tap) {
#if CONV_DETAIL_TL == 1
                const bool dt = tl && n_tile == 3 && kb == 0;
                if (dt) tl[8 + 3 * tap] = clock64();
#endif
                if (wait_b) {
                  mbar_wait(&b_full[bl], bphl);
                  tc_fence_after();
                }
#if CONV_DETAIL_TL == 1
                if (dt) tl[9 + 3 * tap] = clock64();
#endif
                const int shift = tap * p.dil;
                const uint64_t adesc = make_smem_desc_sw128(a_addr + (uint32_t)shift * 128u, p.halo_mode == 1 ? ((uint32_t)shift & 7u) : 0u);
                const uint64_t bdesc = make_smem_desc_sw128(smem_u32(smem_b + (size_t)bl * b_bytes));
#pragma unroll
                for (int k = 0; k < kBlockK / 16; ++k)
                  if (k < nk) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | tap | k) != 0 ? 1u : 0u);
                if (!p.b_resident) umma_commit(&b_empty[bl]);
#if CONV_DETAIL_TL == 1
                if (dt) tl[10 + 3 * tap] = clock64();
#endif
                if (++bl == p.b_stages) bl = 0, bphl ^= 1;
              }
              umma_commit(&a_empty[as]);
            }
            __syncwarp();
            for (int tap = 0; tap < p.taps; ++tap)
              if (++bs == p.b_stages) bs = 0, bph ^= 1;
            if (++as == p.a_stages) as = 0, aph ^= 1;
          }
        } else
        for (int kb = 0; kb < p.kb_per_tap; ++kb) {
          for (int tap = 0; tap < p.taps; ++tap) {
            if (!halo || tap == 0) {
              mbar_wait(&a_full[as], aph);
              tc_fence_after();
            }
            if (!p.b_resident || n_tile == 0) {
              mbar_wait(&b_full[bs], bph);
              tc_fence_after();
            }
            if (tl && n_it < 24 && lane == 0) tl[8 + n_it] = clock64();
            ++n_it;
            // tap t of the halo box = the same rows shifted down by t*dil: start address + t*dil*128 B, with the
            // swizzle phase of the first row in the descriptor's base-offset field
            const int shift = halo ? tap * p.dil : 0;
            const uint64_t adesc = make_smem_desc_sw128(smem_u32(smem_a + (size_t)as * a_bytes) + (uint32_t)shift * 128u,
                                                        p.halo_mode == 1 ? ((uint32_t)shift & 7u) : 0u);
            const uint64_t bdesc = make_smem_desc_sw128(smem_u32(smem_b + (size_t)bs * b_bytes));
            const bool a_done = !halo || tap == p.taps - 1;
            // the last K block of a single-source launch may be partly padding (C = 48, 80, 96 ...): whole 16-wide
            // K steps of zeros are not issued (an SS-mode MMA costs the same ~130 clk whatever it multiplies)
            int nk = kBlockK / 16;
            if (p.k_true > 0 && p.kb_split == p.kb_per_tap) nk = min(nk, (p.k_true - kb * kBlockK + 15) >> 4);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k)
                if (k < nk) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | tap | k) != 0 ? 1u : 0u);
              if (!p.b_resident) umma_commit(&b_empty[bs]);
              if (a_done) umma_commit(&a_empty[as]);
            }
            __syncwarp();
            if (++bs == p.b_stages) bs = 0, bph ^= 1;
            if (a_done) {
              if (++as == p.a_stages) as = 0, aph ^= 1;
            }
          }
        }
        if (elect_one()) umma_commit(&tfull[acc]);
        __syncwarp();
        if (p.res_kb > 0) {
          // fused residual GEMM into the other accumulator (single-tile launches: it is free); the epilogue's LayerNorm
          // statistics pass over the main accumulator runs under these MMAs
          const uint32_t d2 = tmem_u + (uint32_t)((acc ^ 1) * acc_stride);
          for (int kb2 = 0; kb2 < p.res_kb; ++kb2) {
            mbar_wait(&a_full[as], aph);
            mbar_wait(&b_full[bs], bph);
            tc_fence_after();
            const int nk2 = min(kBlockK / 16, (p.res_k_true - kb2 * kBlockK + 15) >> 4);
            const uint64_t adesc = make_smem_desc_sw128(smem_u32(smem_a + (size_t)as * a_bytes));
            const uint64_t bdesc = make_smem_desc_sw128(smem_u32(smem_b + (size_t)bs * b_bytes));
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < kBlockK / 16; ++k)
                if (k < nk2) umma_bf16(d2, adesc + 2 * k, bdesc + 2 * k, idesc, (kb2 | k) != 0 ? 1u : 0u);
              umma_commit(&b_empty[bs]);
              umma_commit(&a_empty[as]);
            }
            __syncwarp();
            if (++as == p.a_stages) as = 0, aph ^= 1;
            if (++bs == p.b_stages) bs = 0, bph ^= 1;
          }
          if (elect_one()) umma_commit(&tfull[acc ^ 1]);
          __syncwarp();
        }
        if (tl && lane == 0 && n_it <= p.taps * p.kb_per_tap) tl[32] = clock64();
        if (tl && lane == 0 && n_tile < 8) tl[24 + n_tile] = clock64();  // (overlaps the late k-iteration stamps: fine for multi-tile runs)
        ++n_tile;
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue
    const int q = warp & 3;                     // TMEM lane quarter this warp may read (warp id % 4)
    const int g = (warp - kFirstEpiWarp) >> 2;  // column group: owns 16-column chunks g, g+4, g+8, g+12
    const int row = q * 32 + lane;
    const int n_chunks = p.block_n >> 4;
    uint8_t* stg = stg_base + (warp - kFirstEpiWarp) * kStageBytesPerWarp;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t parity = 0;
    int e_tile = 0;  // timeline aid
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(tile, m_tiles, n_tiles);
      const int t = tc.mt * kBlockM + row;
      const int n0 = tc.nt * p.block_n;
      ChunkStore st;
      st.alloc = p.out_alloc;
      st.n_store = p.n_store;
      st.row_in = t < p.M;
      const long long row_flat = (long long)t * p.out_ld + p.out_shift;
      const long long boff = (long long)tc.b * p.out_bstride;
      float* out0f = reinterpret_cast<float*>(p.out0) + boff;
      __nv_bfloat16* out0h = reinterpret_cast<__nv_bfloat16*>(p.out0) + boff;
      __nv_bfloat16* out1 = reinterpret_cast<__nv_bfloat16*>(p.out1) + boff;

      if (tile_skipped(p, tc)) {
        if (p.zero_skipped) {  // keep "everything past the valid length is zero" true for final outputs
          st.valid = 0;
          float zero[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) zero[i] = 0.f;
          for (int c = g; c < n_chunks; c += 4) {
            const int n = n0 + c * 16;
            if (out0_dtype == OUT_F32) st.f32(out0f, row_flat + n, n, zero);
            else if (out0_dtype != OUT_NONE) st.bf16(out0h, row_flat + n, n, zero);
            if (out1_mode != OUT1_NONE) st.bf16(out1, row_flat + n, n, zero);
          }
        }
        continue;
      }
      st.valid = p.lengths ? min((long long)p.lengths[tc.b] * p.out_valid_mul, p.out_alloc) : p.out_alloc;
      const float* addf = reinterpret_cast<const float*>(p.addend) + boff;
      const __nv_bfloat16* addh = reinterpret_cast<const __nv_bfloat16*>(p.addend) + boff;
      const float* temb = has_temb ? p.temb + (long long)tc.b * p.temb_bstride : nullptr;
      float2* red = red_base + parity * (2 * 4 * kBlockM);
      parity ^= 1;

      // ---- streaming epilogue: one 16-column chunk at a time, re-read from TMEM in every pass (TMEM reads are cheap,
      // registers are not: with ~220 KB of shared memory there is hardly any L1 left to absorb a spill).  LayerNorm
      // needs whole-row statistics first, so those modes make an extra pass; the second LayerNorm (OUT1_LN) parks the
      // finished values back in the accumulator columns (tcgen05.st) and re-reads them once its statistics are known.
      WarpRows wr;
      wr.t_base = (long long)tc.mt * kBlockM + q * 32;
      wr.out_ld = p.out_ld, wr.out_shift = p.out_shift, wr.valid = st.valid, wr.alloc = st.alloc, wr.M = p.M;
      // TMA-store mode: this thread's row is stored with values iff it lies inside the valid length (else zeros)
      const bool tma_out = p.tma_out != 0;
      const bool row_valid = st.row_in && row_flat + p.N <= st.valid;
      const int tma_t = tc.mt * kBlockM + q * 32;  // first row of this warp
      // fp32 out0 and a bf16 out1 alternate between two staging regions: one younger bulk group may be in flight
      const bool one_pending = out0_dtype != OUT_NONE && (out1_mode == OUT1_COPY || out1_mode == OUT1_SNAKE);
      // residual chunks of this tile: the first of this warp's chunks is fetched now (see fetch_chunk); the
      // next tile's residual rows are pulled into L2 so that its fetches do not wait for HBM
      constexpr int kPre = 1;  // (2 spills in the 96-register epilogue; later chunks hit L2 thanks to the prefetch below)
#ifndef CONV_PRE
#define CONV_PRE 0  // measured: the 16 extra live registers spill, and the spills cost more than the L2 hit they hide
#endif
      const bool pre_ok = CONV_PRE && add_dtype != OUT_NONE && add_dtype != ADD_GEMM && act != ACT_LN_MISH;  // (LayerNorm epilogues: registers are scarce)
      AddRegs pre0;
      if (pre_ok) {
        auto fetch = [&](int k, AddRegs& a) {
          const int c = g + 4 * k;
          const int n = n0 + c * 16;
          if (c < n_chunks && n + 16 <= p.n_store) {
            if (add_dtype == OUT_F32) fetch_chunk<true>(lane, wr, n, addf, a);
            else fetch_chunk<false>(lane, wr, n, addh, a);
          }
        };
        fetch(0, pre0);
      }
      if (add_dtype != OUT_NONE && add_dtype != ADD_GEMM) {
        const int nxt = tile + (int)gridDim.x;
        if (nxt < total_tiles) {
          const TileCoord nc = decode_tile(nxt, m_tiles, n_tiles);
          const int esz = add_dtype == OUT_F32 ? 4 : 2;
          const int lines = (p.block_n * esz + 127) >> 7;  // 128-byte lines per row (the first may start mid-line)
          const uint8_t* nb = reinterpret_cast<const uint8_t*>(p.addend) + (long long)nc.b * p.out_bstride * esz;
          for (int i = threadIdx.x - kFirstEpiWarp * 32; i < kBlockM * lines; i += kEpiThreads) {
            const int rr = i / lines, ln = i - rr * lines;
            const long long tt = (long long)nc.mt * kBlockM + rr;
            const long long f = tt * p.out_ld + p.out_shift + nc.nt * p.block_n;
            if (tt < p.M && f >= 0 && f + p.block_n <= p.out_alloc)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(nb + f * esz + ln * 128));
          }
        }
      }
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      long long* tle = (threadIdx.x == kFirstEpiWarp * 32 && tile == (int)blockIdx.x) ? tl : nullptr;
      if (tle) tle[40] = clock64();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * acc_stride);
      // accumulator chunk c + bias, then the pointwise activations
      auto load_x = [&](int c, float (&x)[16]) {
        tmem_ld16(taddr + (uint32_t)(c * 16), reinterpret_cast<uint32_t(&)[16]>(x));
        tmem_ld_wait();
        if (p.bias) {
          const int ch0 = (n0 + c * 16) % p.chan_mod;
          const float4* bp = reinterpret_cast<const float4*>(p.sv_bias >= 0 ? svec + p.sv_bias + ch0 : p.bias + ch0);
#pragma unroll
          for (int g4 = 0; g4 < 4; ++g4) {
            const float4 bv = bp[g4];
            x[4 * g4] += bv.x, x[4 * g4 + 1] += bv.y, x[4 * g4 + 2] += bv.z, x[4 * g4 + 3] += bv.w;
          }
        }
        if (act == ACT_LRELU || act == ACT_LRELU_TANH) {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = x[i] > 0.f ? x[i] : 0.1f * x[i];
          if (act == ACT_LRELU_TANH) {
#pragma unroll
            for (int i = 0; i < 16; ++i) x[i] = tanhf(x[i]);
          }
        } else if (act == ACT_GELU) {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = gelu_erf(x[i]);
        } else if (act == ACT_SILU) {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = x[i] / (1.0f + __expf(-x[i]));
        } else if (act == ACT_LRELU001) {
#pragma unroll
          for (int i = 0; i < 16; ++i) x[i] = x[i] > 0.f ? x[i] : 0.01f * x[i];
        }
      };
      // statistics of this thread's 64 columns (4 chunks), merged chunk by chunk (Chan), then across the 4 column
      // groups through shared memory
      struct Stats {
        float n = 0.f, mean = 0.f, m2 = 0.f;
        __device__ __forceinline__ void add16(const float (&x)[16]) {
          float sm = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) sm += x[i];
          const float cm = sm * (1.0f / 16.0f);
          float cm2 = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float d = x[i] - cm;
            cm2 = fmaf(d, d, cm2);
          }
          const float nn = n + 16.0f;
          const float delta = cm - mean;
          mean += delta * (16.0f / nn);
          m2 += cm2 + delta * delta * (n * 16.0f / nn);
          n = nn;
        }
      };
      auto combine = [&](const Stats& stt, float2* r, float& mean, float& rstd) {
        r[g * kBlockM + row] = make_float2(stt.mean, stt.m2);
        epi_barrier();
        const float2 a = r[row], b = r[kBlockM + row], c = r[2 * kBlockM + row], d = r[3 * kBlockM + row];
        mean = 0.25f * (a.x + b.x + c.x + d.x);
        const float da = a.x - mean, db = b.x - mean, dc = c.x - mean, dd = d.x - mean;
        const float M2 = a.y + b.y + c.y + d.y + 64.0f * (da * da + db * db + dc * dc + dd * dd);
        rstd = rsqrtf(M2 * (1.0f / 256.0f) + 1e-5f);
      };

      float mean1 = 0.f, rstd1 = 1.f;
      if (act == ACT_LN_MISH) {  // pass A: LayerNorm statistics of the 256-wide row (block_n == N == 256)
        Stats s1;
#pragma unroll 1
        for (int c = g; c < n_chunks; c += 4) {
          float x[16];
          load_x(c, x);
          s1.add16(x);
        }
        combine(s1, red, mean1, rstd1);
      }
      if (tle) tle[45] = clock64();

      Stats s2;
      if (add_dtype == ADD_GEMM) {  // the fused residual GEMM (second accumulator) has retired
        mbar_wait(&tfull[acc ^ 1], acc_phase);
        tc_fence_after();
      }
      const uint32_t taddr_res = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((acc ^ 1) * acc_stride);
      // pass B: finish the values, store the primary / copy / snake outputs
#pragma unroll 1
      for (int c = g; c < n_chunks; c += 4) {
        float x[16];
#if CONV_DETAIL_TL == 3
        const int dk = (c - g) >> 2;
        long long* dt = (tle && dk < 4) ? tle + 8 + 6 * dk : nullptr;
        if (dt) dt[0] = clock64();
#endif
        load_x(c, x);
#if CONV_DETAIL_TL == 3
        if (dt) dt[1] = clock64();
#endif
        const int n = n0 + c * 16;
        if (act == ACT_LN_MISH) {
#pragma unroll
          for (int g4 = 0; g4 < 4; ++g4) {
            const float4 gm = reinterpret_cast<const float4*>(p.sv_lng >= 0 ? svec + p.sv_lng + c * 16 : p.ln_g + c * 16)[g4];
            const float4 bt = reinterpret_cast<const float4*>(p.sv_lnb >= 0 ? svec + p.sv_lnb + c * 16 : p.ln_b + c * 16)[g4];
            x[4 * g4 + 0] = mish_f(fmaf((x[4 * g4 + 0] - mean1) * rstd1, gm.x, bt.x));
            x[4 * g4 + 1] = mish_f(fmaf((x[4 * g4 + 1] - mean1) * rstd1, gm.y, bt.y));
            x[4 * g4 + 2] = mish_f(fmaf((x[4 * g4 + 2] - mean1) * rstd1, gm.z, bt.z));
            x[4 * g4 + 3] = mish_f(fmaf((x[4 * g4 + 3] - mean1) * rstd1, gm.w, bt.w));
          }
        }
        if (has_temb) {
#pragma unroll
          for (int g4 = 0; g4 < 4; ++g4) {
            const float4 tv = __ldg(reinterpret_cast<const float4*>(temb + n) + g4);
            x[4 * g4] += tv.x, x[4 * g4 + 1] += tv.y, x[4 * g4 + 2] += tv.z, x[4 * g4 + 3] += tv.w;
          }
        }
#if CONV_DETAIL_TL == 3
        if (dt) dt[2] = clock64();
#endif
        const long long flat = row_flat + n;
        // only the padded final conv (n_store = 1): the scalar tail indexes x dynamically, which would put x in local
        // memory for every instance that contains it
        const bool partial = (kAct == ACT_LRELU_TANH || kAct < 0) && n + 16 > p.n_store;
        if (add_dtype == ADD_GEMM) {  // residual = the second accumulator's chunk + its bias
          float r[16];
          tmem_ld16(taddr_res + (uint32_t)(c * 16), reinterpret_cast<uint32_t(&)[16]>(r));
          tmem_ld_wait();
          const float4* rb = reinterpret_cast<const float4*>(p.res_bias + n);
#pragma unroll
          for (int g4 = 0; g4 < 4; ++g4) {
            const float4 bv = __ldg(rb + g4);
            x[4 * g4] += r[4 * g4] + bv.x, x[4 * g4 + 1] += r[4 * g4 + 1] + bv.y;
            x[4 * g4 + 2] += r[4 * g4 + 2] + bv.z, x[4 * g4 + 3] += r[4 * g4 + 3] + bv.w;
          }
        } else if (add_dtype != OUT_NONE && !partial) {
          // the transposes below reuse the fp32 staging region (an fp32 residual also covers a 16-bit out0's region)
          if (tma_out && (out0_dtype == OUT_F32 || (out0_dtype != OUT_NONE && add_dtype == OUT_F32))) {
            if (lane == 0) {
              if (one_pending) bulk_wait_read<1>();
              else bulk_wait_read<0>();
            }
            __syncwarp();
          }
          const int k = (c - g) >> 2;
          if (pre_ok && k < kPre) {
            if (add_dtype == OUT_F32) apply_chunk<OUT_F32>(stg, lane, pre0, x);
            else if (add_dtype == OUT_F16) apply_chunk<OUT_F16>(stg, lane, pre0, x);
            else apply_chunk<OUT_BF16>(stg, lane, pre0, x);
          } else {
            AddRegs a;
            if (add_dtype == OUT_F32) fetch_chunk<true>(lane, wr, n, addf, a), apply_chunk<OUT_F32>(stg, lane, a, x);
            else if (add_dtype == OUT_F16) fetch_chunk<false>(lane, wr, n, addh, a), apply_chunk<OUT_F16>(stg, lane, a, x);
            else fetch_chunk<false>(lane, wr, n, addh, a), apply_chunk<OUT_BF16>(stg, lane, a, x);
          }
        }
#if CONV_DETAIL_TL == 3
        if (dt) dt[3] = clock64();
#endif
        if (partial) {  // scalar tail: column 0 of consecutive rows is contiguous when out_ld == n_store == 1
          const int stt = st.state(flat, max(p.n_store - n, 1));
          if (stt != 0 && n < p.n_store) {
            for (int i = 0; i < 16 && n + i < p.n_store; ++i) {
              const float xv = stt == 2 ? x[i] : 0.f;
              if (out0_dtype == OUT_F32) out0f[flat + i] = xv;
              else if (out0_dtype == OUT_BF16) reinterpret_cast<uint16_t*>(out0h)[flat + i] = LS_CVT_H_BITS(xv);
              else if (out0_dtype == OUT_F16) reinterpret_cast<uint16_t*>(out0h)[flat + i] = cvt_f16_bits(xv);
              if (out1_mode == OUT1_COPY) reinterpret_cast<uint16_t*>(out1)[flat + i] = LS_CVT_H_BITS(xv);
            }
          }
        } else {
          if (tma_out) {
            if (out0_dtype == OUT_F32) store_chunk_tma_p<OUT_F32>(one_pending, stg, lane, &mapOut0, n, tma_t, tc.b, row_valid, x);
            else if (out0_dtype == OUT_BF16)
              store_chunk_tma_p<OUT_BF16, kStageOut0H>(one_pending, stg, lane, &mapOut0, n, tma_t, tc.b, row_valid, x);
            else if (out0_dtype == OUT_F16)
              store_chunk_tma_p<OUT_F16, kStageOut0H>(one_pending, stg, lane, &mapOut0, n, tma_t, tc.b, row_valid, x);
          } else {
            if (out0_dtype == OUT_F32) store_chunk<OUT_F32>(stg, lane, wr, n, out0f, x);
            else if (out0_dtype == OUT_BF16) store_chunk<OUT_BF16>(stg, lane, wr, n, out0h, x);
            else if (out0_dtype == OUT_F16) store_chunk<OUT_F16>(stg, lane, wr, n, out0h, x);
          }
#if CONV_DETAIL_TL == 3
          if (dt) dt[4] = clock64();
#endif
          if (out1_mode == OUT1_COPY) {
            if (tma_out) store_chunk_tma_p<OUT_BF16>(one_pending, stg, lane, &mapOut1, n, tma_t, tc.b, row_valid, x);
            else store_chunk<OUT_BF16>(stg, lane, wr, n, out1, x);
          } else if (out1_mode == OUT1_SNAKE) {
            const int ch0 = n % p.chan_mod;
#pragma unroll
            for (int g4 = 0; g4 < 4; ++g4) {
              const float4 al = reinterpret_cast<const float4*>(p.sv_p1a >= 0 ? svec + p.sv_p1a + ch0 : p.p1_a + ch0)[g4];
              const float4 ia = reinterpret_cast<const float4*>(p.sv_p1b >= 0 ? svec + p.sv_p1b + ch0 : p.p1_b + ch0)[g4];
              x[4 * g4 + 0] = snake_f(x[4 * g4 + 0], al.x, ia.x);
              x[4 * g4 + 1] = snake_f(x[4 * g4 + 1], al.y, ia.y);
              x[4 * g4 + 2] = snake_f(x[4 * g4 + 2], al.z, ia.z);
              x[4 * g4 + 3] = snake_f(x[4 * g4 + 3], al.w, ia.w);
            }
            if (tma_out) store_chunk_tma_p<OUT_BF16>(one_pending, stg, lane, &mapOut1, n, tma_t, tc.b, row_valid, x);
            else store_chunk<OUT_BF16>(stg, lane, wr, n, out1, x);
          } else if (out1_mode == OUT1_LN) {
            s2.add16(x);
            tmem_st16(taddr + (uint32_t)(c * 16), reinterpret_cast<const uint32_t(&)[16]>(x));
          }
        }
      }
      if (tle) tle[42] = clock64();
      if (out1_mode == OUT1_LN) {  // pass C: second output = LayerNorm(u), the bf16 operand of the next GEMM
        tmem_st_wait();
        float mean2, rstd2;
        combine(s2, red + 4 * kBlockM, mean2, rstd2);
#pragma unroll 1
        for (int c = g; c < n_chunks; c += 4) {
          float x[16];
          tmem_ld16(taddr + (uint32_t)(c * 16), reinterpret_cast<uint32_t(&)[16]>(x));
          tmem_ld_wait();
#pragma unroll
          for (int g4 = 0; g4 < 4; ++g4) {
            const float4 ga = reinterpret_cast<const float4*>(p.sv_p1a >= 0 ? svec + p.sv_p1a + c * 16 : p.p1_a + c * 16)[g4];
            const float4 be = reinterpret_cast<const float4*>(p.sv_p1b >= 0 ? svec + p.sv_p1b + c * 16 : p.p1_b + c * 16)[g4];
            x[4 * g4 + 0] = fmaf((x[4 * g4 + 0] - mean2) * rstd2, ga.x, be.x);
            x[4 * g4 + 1] = fmaf((x[4 * g4 + 1] - mean2) * rstd2, ga.y, be.y);
            x[4 * g4 + 2] = fmaf((x[4 * g4 + 2] - mean2) * rstd2, ga.z, be.z);
            x[4 * g4 + 3] = fmaf((x[4 * g4 + 3] - mean2) * rstd2, ga.w, be.w);
          }
          if (tma_out) store_chunk_tma<OUT_BF16, 0>(stg, lane, &mapOut1, n0 + c * 16, tma_t, tc.b, row_valid, x);
          else store_chunk<OUT_BF16>(stg, lane, wr, n0 + c * 16, out1, x);
        }
      }
      // every TMEM access of this tile is done: hand the accumulator stage back to the MMA warp
      if (tl && threadIdx.x == kFirstEpiWarp * 32 && e_tile < 8) tl[48 + e_tile] = clock64();
      ++e_tile;
      tc_fence_before();
      mbar_arrive(&tempty[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (p.tma_out && lane == 0) bulk_wait<0>();  // every bulk store of this lane has been written
  }

  if (threadIdx.x == kFirstEpiWarp * 32) TL(43);
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) TL(44);
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  }
#undef TL
}

int pow2_at_least(int x, int lo) {
  int v = lo;
  while (v < x) v <<= 1;
  return v;
}

template <int kAct, int kOut0, int kOut1, int kAdd, int kTemb>
cudaError_t launch_instance(int grid, size_t smem, cudaStream_t stream, const CUtensorMap& mapA0, const CUtensorMap& mapA1,
                            const CUtensorMap& mapW, const CUtensorMap& mapO0, const CUtensorMap& mapO1,
                            const ConvGemmParams& pp, int tmem_cols, int acc_stride) {
  auto* kernel = conv_gemm_kernel<kAct, kOut0, kOut1, kAdd, kTemb>;
  static std::atomic<unsigned long long> optin{0};  // per instance, one bit per device
  if (cudaError_t e = smem_optin_once(optin, reinterpret_cast<const void*>(kernel), 227 * 1024); e != cudaSuccess) return e;
  return launch_pdl(kernel, dim3(grid), dim3(kThreads), smem, stream, 1, mapA0, mapA1, mapW, mapO0, mapO1, pp, tmem_cols,
                    acc_stride);
}

}  // namespace

cudaError_t LS_FN(launch_conv_gemm)(const CUtensorMap& mapA0, const CUtensorMap& mapA1, const CUtensorMap& mapW,
                                    const ConvGemmParams& p, int num_sms, cudaStream_t stream, int* plan_out) {
#if !LS_HALF_FP16
  if (p.fp16) return launch_conv_gemm_fp16(mapA0, mapA1, mapW, p, num_sms, stream, plan_out);  // fp16-operand build of this file
#endif
  if (plan_out)
    for (int i = 0; i < kConvPlanInts; ++i) plan_out[i] = 0;
  if (num_sms <= 0) return cudaErrorInvalidValue;
  if (p.block_n % 16 || p.block_n < 16 || p.block_n > 256 || p.N % p.block_n || p.chan_mod % 16) return cudaErrorInvalidValue;
  if ((p.act == ACT_LN_MISH || p.out1_mode == OUT1_LN) && p.block_n != p.N) return cudaErrorInvalidValue;
  if (p.out1_mode == OUT1_LN && p.out0_dtype != OUT_F32) return cudaErrorInvalidValue;
  if (p.out1_mode != OUT1_NONE && p.out1 == nullptr) return cudaErrorInvalidValue;
  if (p.addend_dtype == ADD_GEMM) {  // fused residual GEMM: one tile per CTA, one N tile, a bias and at least one K block
    const long long tiles = (long long)p.B * ((p.M + kBlockM - 1) / kBlockM);
    if (p.res_kb <= 0 || p.res_bias == nullptr || p.N != p.block_n || tiles > num_sms) return cudaErrorInvalidValue;
  } else if (p.res_kb != 0) {
    return cudaErrorInvalidValue;
  }
  ConvGemmParams pp = p;
  pp.timeline = (g_debug_buffer && g_debug_bytes >= 148 * 64 * 8) ? g_debug_buffer : nullptr;
  pp.a_box_rows = p.halo_mode ? conv_halo_box_rows(p.taps, p.dil) : kBlockM;
  if (pp.a_box_rows > 256) return cudaErrorInvalidValue;  // TMA box limit
  const int a_bytes = ls_conv_a_stage_bytes(pp.a_box_rows);
  const int b_bytes = p.block_n * kBlockK * 2;
  // per-channel epilogue vectors staged in shared memory (up to 16 KB; larger ones stay in global memory)
  pp.sv_bias = pp.sv_p1a = pp.sv_p1b = pp.sv_lng = pp.sv_lnb = -1;
  pp.sv_floats = 0;
  {
    auto place = [&](int& off, const void* ptr, int n) {
      if (ptr && (pp.sv_floats + n) * 4 <= 16 * 1024) off = pp.sv_floats, pp.sv_floats += (n + 3) & ~3;
    };
    place(pp.sv_bias, p.bias, p.chan_mod);
    if (p.out1_mode == OUT1_SNAKE || p.out1_mode == OUT1_LN) place(pp.sv_p1a, p.p1_a, p.chan_mod), place(pp.sv_p1b, p.p1_b, p.chan_mod);
    if (p.act == ACT_LN_MISH) place(pp.sv_lng, p.ln_g, p.N), place(pp.sv_lnb, p.ln_b, p.N);
  }
  // the LayerNorm statistics area is only there for launches that normalise: the thin DAC layers' weight rings are
  // latency-bound (bytes in flight), so they get those 16 KB
  pp.red_bytes = (p.act == ACT_LN_MISH || p.out1_mode == OUT1_LN || p.act < 0) ? kRedBytes : 0;
  const int budget = kSmemBudget + (kRedBytes - pp.red_bytes) - pp.sv_floats * 4;
  const int m_tiles_ = (p.M + kBlockM - 1) / kBlockM;
  const long long tiles_per_cta = ((long long)p.B * m_tiles_ * (p.N / p.block_n) + num_sms - 1) / num_sms;
  const int w_boxes = p.taps * p.kb_per_tap;
  pp.b_resident = 0;
  if (p.N == p.block_n && tiles_per_cta >= 3 && w_boxes <= kMaxStages && w_boxes >= kWeightProducers &&
      w_boxes * b_bytes + 3 * a_bytes <= budget && conv_resident_enabled()) {
    // small weight tensors (DAC stages with C <= 96, 1x1 layers): resident weights, the whole budget left to activations
    pp.b_resident = 1;
    pp.b_stages = w_boxes;
    pp.a_stages = (budget - w_boxes * b_bytes) / a_bytes;
    if (pp.a_stages > 6) pp.a_stages = 6;
  } else if (p.halo_mode && p.taps > 1) {
    // one A box feeds `taps` B boxes: two A stages are enough, the rest of the budget goes to the weight ring
    pp.a_stages = p.kb_per_tap > 1 ? 2 : 1;
    if (p.kb_per_tap > 1 && 3 * a_bytes + 4 * b_bytes <= budget) pp.a_stages = CONV_HALO_A_STAGES;
    pp.b_stages = (budget - pp.a_stages * a_bytes) / b_bytes;
  } else {
    pp.a_stages = pp.b_stages = budget / (a_bytes + b_bytes);
  }
  // dual-issue mode (see the kernel): halo launches with ONE N tile and enough tiles per CTA to pair
  pp.dual = 0;
  if (kProducerWarps == 3 && p.halo_mode && p.taps > 1 && p.N == p.block_n && tiles_per_cta >= 4 && w_boxes <= kMaxStages * 4 &&
      conv_dual_enabled()) {
    if (w_boxes <= kMaxStages && w_boxes * b_bytes + 4 * a_bytes <= budget && conv_resident_enabled()) {
      // resident weights: the single-issuer lean loop with all three producer warps sharing the activation loads is
      // faster (C = 48 conv7: 335-358 us vs 406-421 us dual) -- dual only under -DCONV_DUAL_RESIDENT=1
      if (CONV_DUAL_RESIDENT) {
        pp.dual = 1, pp.b_resident = 1, pp.b_stages = w_boxes;
        pp.a_stages = (budget - w_boxes * b_bytes) / a_bytes;
        if (pp.a_stages > 6) pp.a_stages = 6;
        pp.a_stages &= ~1;
      }
    } else if (4 * a_bytes + 3 * b_bytes <= budget) {
      pp.dual = 1, pp.b_resident = 0, pp.a_stages = 4;
      pp.b_stages = (budget - 4 * a_bytes) / b_bytes;
    }
  }
  if (pp.a_stages > kMaxStages) pp.a_stages = kMaxStages;
  if (pp.b_stages > kMaxStages) pp.b_stages = kMaxStages;
  if (pp.a_stages < 1 || pp.b_stages < 2 || pp.b_stages < kWeightProducers) return cudaErrorInvalidValue;
  const int acc_stride = pow2_at_least(p.block_n, 32);
  const int tmem_cols = 2 * acc_stride;
  size_t smem = (size_t)pp.a_stages * a_bytes + (size_t)pp.b_stages * b_bytes + 1024 + 1024 + pp.red_bytes +
                kEpiWarps * kStageBytesPerWarp + (size_t)pp.sv_floats * 4;
  // tmem_cols == 512 must never share an SM with a second CTA of this kernel (alloc would spin):
  if (tmem_cols > 256 && smem < 120 * 1024) smem = 120 * 1024;
  const int m_tiles = (p.M + kBlockM - 1) / kBlockM;
  const long long total = (long long)p.B * m_tiles * (p.N / p.block_n);
  if (total <= 0) return cudaSuccess;
  const int grid = (int)(total < num_sms ? total : num_sms);
  const double kt = p.k_true > 0 ? p.k_true : p.kb_per_tap * kBlockK;
  const double rows = (double)p.B * p.M;
  const double out_b = (p.out0_dtype == OUT_F32 ? 4.0 : p.out0_dtype != OUT_NONE ? 2.0 : 0.0) +
                       (p.out1_mode != OUT1_NONE ? 2.0 : 0.0) +
                       (p.addend ? (p.addend_dtype == OUT_F32 ? 4.0 : 2.0) : 0.0);
  ProfScope prof(stream, p.tag == 1 ? PK_CONV_DAC : PK_CONV_FLOW, 2.0 * rows * p.N * (kt * p.taps + (p.res_kb > 0 ? p.res_k_true : 0)),
                 rows * kt * 2.0 + (double)p.taps * p.N * kt * 2.0 + rows * (p.n_store < p.N ? p.n_store : p.N) * out_b);
  count_launch();
  // dense outputs go out through TMA stores (see store_chunk_tma); tensor maps cached per (buffer, shape).  The cache
  // hands maps out BY VALUE: an insertion may evict (clear) the table, so no pointer into it survives a second lookup.
  static thread_local std::unordered_map<std::string, CUtensorMap> out_maps;
  auto out_map = [&](const void* base, int elem_bytes, CUtensorMap* dst) -> bool {
    char key[96];
    snprintf(key, sizeof key, "%p/%d/%d/%d/%d", base, elem_bytes, p.N, p.M, p.B);
    auto it = out_maps.find(key);
    if (it == out_maps.end()) {
      CUtensorMap m;
      if (!make_out_map(&m, base, elem_bytes, p.N, p.M, p.B)) return false;
      if (out_maps.size() > 4096) out_maps.clear();
      it = out_maps.emplace(key, m).first;
    }
    *dst = it->second;
    return true;
  };
  const bool dense = p.out_ld == p.N && p.out_shift == 0 && p.n_store == p.N && p.out_bstride == (long long)p.M * p.N &&
                     p.out_alloc == (long long)p.M * p.N && (p.out_valid_mul % p.N) == 0 && p.N % 16 == 0 &&
                     (p.out0_dtype != OUT_NONE || p.out1_mode != OUT1_NONE) && conv_tma_out_enabled();
  CUtensorMap mo0v = mapW, mo1v = mapW;  // placeholders when unused
  pp.tma_out = 0;
  if (dense) {
    const bool a = p.out0_dtype == OUT_NONE || out_map(p.out0, p.out0_dtype == OUT_F32 ? 4 : 2, &mo0v);
    const bool b = p.out1_mode == OUT1_NONE || out_map(p.out1, 2, &mo1v);
    if (a && b) pp.tma_out = 1;
    else mo0v = mapW, mo1v = mapW;
  }
  const CUtensorMap* mo0 = &mo0v;
  const CUtensorMap* mo1 = &mo1v;
  if (plan_out) {
    const int plan[kConvPlanInts] = {grid, (int)((total + grid - 1) / grid), pp.dual, pp.b_resident, pp.a_stages,
                                     pp.b_stages, pp.tma_out, pp.halo_mode};
    for (int i = 0; i < kConvPlanInts; ++i) plan_out[i] = plan[i];
  }
  const int add = p.addend_dtype == ADD_GEMM ? (int)ADD_GEMM : p.addend ? p.addend_dtype : (int)OUT_NONE;
  const int temb = p.temb ? 1 : 0;
#define LS_CONV_CASE(A, O0, O1, AD, TE)                                                                          \
  if (p.act == (A) && p.out0_dtype == (O0) && p.out1_mode == (O1) && add == (AD) && temb == (TE))               \
    return launch_instance<A, O0, O1, AD, TE>(grid, smem, stream, mapA0, mapA1, mapW, *mo0, *mo1, pp, tmem_cols, acc_stride);
  // flow estimator: resnet conv1 | res_conv, final_proj | resnet conv2 | QKV, down / up conv | final block
  LS_CONV_CASE(ACT_LN_MISH, OUT_NONE, OUT1_COPY, OUT_NONE, 1)
  LS_CONV_CASE(ACT_NONE, OUT_F32, OUT1_NONE, OUT_NONE, 0)
  LS_CONV_CASE(ACT_LN_MISH, OUT_F32, OUT1_LN, OUT_F32, 0)
  LS_CONV_CASE(ACT_LN_MISH, OUT_F32, OUT1_NONE, OUT_F32, 0)
  LS_CONV_CASE(ACT_LN_MISH, OUT_F32, OUT1_NONE, ADD_GEMM, 0)  // resnet conv2 with res_conv fused in (single-tile launches)
  LS_CONV_CASE(ACT_LN_MISH, OUT_F32, OUT1_LN, ADD_GEMM, 0)
  LS_CONV_CASE(ACT_NONE, OUT_NONE, OUT1_COPY, OUT_NONE, 0)
  LS_CONV_CASE(ACT_LN_MISH, OUT_NONE, OUT1_COPY, OUT_NONE, 0)
  // DAC decoder: de_conv_pre | input conv, conv7 | transposed conv | conv1 + residual (x kept / last unit) | final conv
  // (both builds: the fp16-operand build serves the flow estimator and the fp16 DAC decoder / encoder handles)
  LS_CONV_CASE(ACT_LRELU, OUT_NONE, OUT1_COPY, OUT_NONE, 0)
  LS_CONV_CASE(ACT_LRELU, OUT_NONE, OUT1_SNAKE, OUT_NONE, 0)
  LS_CONV_CASE(ACT_NONE, OUT_F32, OUT1_SNAKE, OUT_NONE, 0)
  LS_CONV_CASE(ACT_LRELU, OUT_F32, OUT1_SNAKE, OUT_F32, 0)
  LS_CONV_CASE(ACT_LRELU, OUT_NONE, OUT1_SNAKE, OUT_F32, 0)
  LS_CONV_CASE(ACT_NONE, OUT_F16, OUT1_SNAKE, OUT_NONE, 0)  // the same three with the residual stream kept as fp16
  LS_CONV_CASE(ACT_LRELU, OUT_F16, OUT1_SNAKE, OUT_F16, 0)
  LS_CONV_CASE(ACT_LRELU, OUT_NONE, OUT1_SNAKE, OUT_F16, 0)
  LS_CONV_CASE(ACT_LRELU_TANH, OUT_F32, OUT1_NONE, OUT_NONE, 0)
#undef LS_CONV_CASE
  return launch_instance<-1, -1, -1, -1, -1>(grid, smem, stream, mapA0, mapA1, mapW, *mo0, *mo1, pp, tmem_cols, acc_stride);
}

}  // namespace ls
