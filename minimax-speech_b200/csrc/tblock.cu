// Fused transformer-block tail for the estimator, sm_100a: everything of a BasicTransformerBlock that is
// row-local, in ONE kernel per 128-row tile, chained through TMEM / shared memory instead of HBM:
//
//   u'   = att . Wo^T + bo + u                 attn1.to_out.0 + residual    matcha transformer.py:266-277
//   n3   = LayerNorm(u'; norm3)                                              transformer.py:303
//   h    = GELU_erf(n3 . W1^T + b1)            ff.net.0 (diffusers GELU)     transformer.py:109-110,131-134
//   u''  = u' + h . W2^T + b2                  ff.net.2 + residual           transformer.py:313-314
//   tail 0:  n1 = LayerNorm(u''; next block's norm1);  qkv = n1 . Wqkv^T     transformer.py:243-271 (next block)
//   tail 1:  masked bf16 copy of u'' (input of the conv that follows the block group, decoder.py:452-455)
//
// `att` is the flash kernel's output (bf16 [R][512]); `u` the fp32 residual stream (read once, written once).
// The 1024-wide FF intermediate and both LayerNorm outputs never leave the SM.
//
// Structure (one CTA per SM, persistent over tiles, 20 warps):
//   warps 0-2   TMA producers: stream every weight tile (128 rows x 64 K, 16 KB, 128B swizzle) through a 5-slot mbarrier
//               ring in exactly the order the MMA warp consumes them (load i is issued by warp i % 3)
//   warp 3      TMEM allocator + tcgen05.mma issuer (one elected lane); M=128 x N=128 x K=16 MMAs, fp32 accumulate
//   warps 4-19  epilogue: warp w owns TMEM lanes 32*(w%4).. (= 32 rows) and column group (w-4)/4; its first warp also
//               issues the tile's att boxes, the u boxes that follow them, and every TMA store
// TMEM (512 columns): D = [0,256) holds u' then u''; H0/H1 = [256,384) / [384,512) double-buffer the 128-wide
// FF1 chunks (and later the 128-wide QKV chunks).  FF2 accumulates straight onto u' in D (the epilogue writes
// u' back with tcgen05.st), so the residual add costs nothing; its A operand, the GELU output, is written back over
// its own H columns as packed 16-bit pairs and read from there (tcgen05.mma TS form).
// Shared memory: A3 (64 KB) = LayerNorm output as the K-major A operand of FF1 / QKV; AH (64 KB) = staging boxes of the
// TMA stores (u'', qkv, tail); A3 + AH together hold the att tile, then the fp32 u tile, while the out-proj runs;
// ring (80 KB); per-block vectors (10 KB).
#include "kernels.h"
#include "profiler.h"
#include "ptx.cuh"

namespace ls {
namespace {

constexpr int kC = 256, kInner = 512, kFF = 1024, kQKV = 1536;
constexpr int kTileM = 128;
constexpr int kSlotBytes = 128 * 64 * 2;  // 16 KB: 128 rows x 128 B
// Pair mode (TBLOCK_PAIR): the two CTAs of a cluster form one 256-row tcgen05 cta_group::2 MMA.  Each CTA keeps its
// own 128 rows of A and D and provides HALF of every weight box (64 rows, 8 KB), so the ring holds twice as many
// boxes and each SM pulls half the weight bytes per tile -- the weight stream is what bounds this kernel.
constexpr bool kPair = TBLOCK_PAIR != 0;
// One TMA instruction per issuing warp is in flight at a time (measured), so pair mode spends its halved weight bytes on
// HALF AS MANY instructions of the same 16 KB: 128 own rows of Wo / W2 (the pair's N = 256 operand), or two K blocks of a
// 64-row half of a W1 / Wqkv chunk (3-D box), per instruction.
constexpr int kRingSlotBytes = kSlotBytes;
#ifndef TBLOCK_SLOTS
#define TBLOCK_SLOTS 5
#endif
constexpr int kSlots = TBLOCK_SLOTS;
#ifndef TBLOCK_PRODUCER_WARPS
#define TBLOCK_PRODUCER_WARPS 3
#endif
constexpr int kProducerWarps = TBLOCK_PRODUCER_WARPS;  // warps 0..: one TMA-issuing thread each (issue latencies overlap)
constexpr int kMmaWarp = kProducerWarps;
#ifndef TBLOCK_PRODUCER_LANES
#define TBLOCK_PRODUCER_LANES 1
#endif
constexpr int kProducerLanes = TBLOCK_PRODUCER_LANES;  // issuing lanes per producer warp
constexpr int kIssuers = kProducerWarps * kProducerLanes;
static_assert(kIssuers <= kSlots, "interleaved producers must not outnumber the ring slots (parity waits)");
static_assert(!kPair || TBLOCK_CLUSTER == 2, "pair mode is a cluster of two");
constexpr int kCS = TBLOCK_CLUSTER;          // CTAs per cluster: each loads 1/kCS of every weight box and multicasts it
constexpr int kPartRows = 128 / kCS;         // weight rows per CTA per box
constexpr int kPartBytes = kPartRows * 128;
constexpr uint16_t kCtaMask = (uint16_t)((1u << kCS) - 1);
// Second weight ring (single-CTA form only): the four 16 KB boxes of W2[:, chunk] get slots of their own in the AH region,
// which is idle in the FF phase now that the GELU output lives in tensor memory.  With one 5-slot ring the boxes of W2(c)
// sat in it while the MMA warp waited for GELU(c), W1(c+2) could not be prefetched behind them, and every FF chunk paid a
// TMA round trip (measured: 3.8 k clk per chunk against 2.8 k of MMA work).  The region doubles as the staging tile of the
// residual-stream loads / stores outside the FF phase: its first use per tile waits for the epilogue's stage_free.
#ifndef TBLOCK_RING_B
#define TBLOCK_RING_B 0  // measured: 3.4 k instead of 3.8 k clk per FF chunk on the first tile of a CTA, but not yet correct for a CTA's later tiles
#endif
constexpr bool kRingB = TBLOCK_RING_B != 0 && !kPair && kCS == 1;
// FF2 with its A operand (the GELU output) in tensor memory -- the tcgen05 "TS" form: 73 instead of 102 clk per N = 128
// MMA (profiles/micro/mma_bw.cu), no AH staging, no ah_free barrier.  With the att tile still in the weight ring it
// measured 38.5 against 37.8 ms of fused-block time per bench step; with TBLOCK_ATT_DIRECT it is the faster form (52.9
// against 54.5 us per launch, 34.7 against 36.1 ms per step: profiles/r02_ab_tblock_att_direct.log) and the default.
// TBLOCK_WIDE_FF: in the FF phase the weight ring is NINE slots -- the four boxes of the AH region, idle there once the
// GELU output lives in tensor memory (TS form of FF2), join the five ring slots.  A slot takes ~1.9 k clk from "MMAs
// issued" through "retired -> producer woken -> TMA issued -> landed" (profiles/r02_timeline_tblock_*.log), so five 16 KB
// slots feed ~35-43 B/clk where the MMAs of a box want 64.  Ring slots 4..8 and AH slots 0..3 are two cyclic sub-rings with
// running counters: out-proj, FF1 chunks 0 / 1, the QKV phase and head mode use the ring alone, the 56 loads of the FF chunk
// loop follow the pattern 4 x AH, 5 x ring.  Slot and use number are closed forms of (tile, load) for the producers and
// incremental uniform-register state for the MMA warp (a first version looked them up in a shared-memory table: the look-ups
// sat on the slot-turnaround path and cost 500 clk per K block, 73 instead of 53 us).  Each slot has TWO release barriers,
// for its even and odd uses, so that a producer warp that runs ahead of the consumer across a phase boundary cannot mistake
// an older phase for its own (profiles/ring_protocol_sim.py checks the invariant and simulates the protocol); the first
// four AH loads of a tile wait for the epilogue to be done with the u tile (stage_free).
// Measured (profiles/r02_ab_tblock_wide_ff.log): 56.1 us against 52.7 us for the five-slot ring with the same TS form -- the
// FF chunk period goes UP (4.3 k from 3.9 k clk) and the ring-only phases pay ~150 clk per K block for the extra slot
// bookkeeping: ring depth is not what bounds the weight stream, the per-box handling chain is.  Off.
#ifndef TBLOCK_WIDE_FF
#define TBLOCK_WIDE_FF 0
#endif
#ifndef TBLOCK_FF2_TS
#define TBLOCK_FF2_TS 1
#endif
constexpr bool kFf2Ts = TBLOCK_FF2_TS != 0 && !kPair;
// TBLOCK_DETAIL_TL=1 adds per-sub-step clock64 stamps of FF chunk 4 / QKV chunk 6 (profiles/timeline_tblock.py); they cost
// registers in the 96-register epilogue (spills), so product builds leave them out.
#ifndef TBLOCK_DETAIL_TL
#define TBLOCK_DETAIL_TL 0
#endif
constexpr bool kDetailTl = TBLOCK_DETAIL_TL != 0;
// TBLOCK_MERGE_ELECT: the slot-release commits are issued inside the election that issued the box's MMAs
#ifndef TBLOCK_MERGE_ELECT
#define TBLOCK_MERGE_ELECT 0  // measured: 58.3 vs 57.3 us per launch (profiles/r02_ab_tblock_merge_elect.log)
#endif
constexpr bool kMergeElect = TBLOCK_MERGE_ELECT != 0;
// TBLOCK_L2_PREFETCH: in the prologue (before the PDL wait: weights do not depend on the previous kernel) the CTAs of the
// grid ask for the launch's weight boxes, one or two each, to be brought into L2.  Inside a bench step the 2.2 MB of a
// block's weights are cold (112 MB of block weights and > 1 GB of activations pass through the 126 MB L2 per step), every
// CTA streams them in the same order at about the same time, so without this each box is a DRAM miss that all 125 CTAs
// wait for, on the ring's critical path (ncu launch list with flushed caches: 56.9 / 37.8 / 27.8 us per tail-0 / tail-1 /
// head launch against 52.7 / 32.6 / 23.5 us with L2-warm operands).
#ifndef TBLOCK_L2_PREFETCH
#define TBLOCK_L2_PREFETCH 1
#endif
constexpr bool kL2Prefetch = TBLOCK_L2_PREFETCH != 0 && !kPair && kCS == 1;
// TBLOCK_ATT_DIRECT: the out-proj's A operand (the 128 x 512 attention-output tile, 8 boxes) does not travel through the
// weight ring.  It is loaded at the start of the tile straight into the 8 boxes of A3 + AH that used to hold the fp32 u
// tile from the start (all 8 loads in flight at once, on top of the ring's), and u box j follows into the same place as
// soon as the MMAs of K block j have retired (the u tile is only read by the out-proj EPILOGUE).  The ring then carries
// the 16 Wo boxes alone, in groups of two -- with three boxes per K block in five slots the third box of every K block
// could only be requested after the previous block had retired, one TMA round trip per K block
// (profiles/r02_timeline_tblock_detail.log).
#ifndef TBLOCK_ATT_DIRECT
#define TBLOCK_ATT_DIRECT 1
#endif
constexpr bool kAttDirect = TBLOCK_ATT_DIRECT != 0 && !kPair && kCS == 1 && !kRingB;
constexpr int kOutLoads = kAttDirect ? 16 : 24;  // ring loads of the out-proj phase (single-CTA form)
constexpr bool kWide = TBLOCK_WIDE_FF != 0 && kAttDirect && kFf2Ts && kSlots == 5 && !kMergeElect;
constexpr int kWideSlots = 9;       // AH boxes 0..3 + ring slots 4..8 (contiguous in shared memory)
constexpr int kWideAhPerTile = 26;  // AH-slot loads of one tile's FF chunk loop: 6 patterns of (4 AH + 5 ring) + 2
static_assert(!kRingB || kFf2Ts, "the second ring lives in the AH region: it needs the TS form of FF2");
constexpr int kSlotsB = 4;
constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kFirstEpiWarp = kProducerWarps + 1;
constexpr int kThreads = kFirstEpiWarp * 32 + kEpiThreads;

constexpr int kOffA3 = 0;
constexpr int kOffAH = 4 * kSlotBytes;
constexpr int kOffRing = kOffAH + 4 * kSlotBytes;
constexpr int kOffVec = kOffRing + kSlots * kRingSlotBytes;
constexpr int kOffRed = kOffVec + TBLOCK_VEC_FLOATS * 4;
constexpr int kOffBars = kOffRed + 4 * kTileM * 8;  // [column group][row] float2
constexpr int kBarBytes = 1024;  // ~60 mbarriers, the TMEM slot
constexpr int kSmemBytes = kOffBars + kBarBytes + 1024;
static_assert(kSmemBytes <= 227 * 1024, "tblock shared memory budget");

// offsets (floats) inside the per-block vector pack
constexpr int V_BO = 0, V_G3 = 256, V_BE3 = 512, V_B1 = 768, V_B2 = 1792, V_G1N = 2048, V_BE1N = 2304;
static_assert(V_BE1N + 256 == TBLOCK_VEC_FLOATS, "vector pack layout");

constexpr uint32_t kTmemD = 0, kTmemH = 256;

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

// true if every row of the tile is padding (t >= lengths[b])
__device__ __forceinline__ bool tile_all_padding(const TBlockParams& p, int row0) {
  if (p.lengths == nullptr || p.no_skip) return false;
  const int last = min(row0 + kTileM, p.R) - 1;
  for (int b = row0 / p.T; b <= last / p.T; ++b) {
    const int t_start = max(row0, b * p.T) - b * p.T;
    if (t_start < p.lengths[b]) return false;
  }
  return true;
}

struct RowStats {
  float n = 0.f, mean = 0.f, m2 = 0.f;
  // merge a 32-value chunk (Chan's parallel update); exact two-pass statistics inside the chunk
  __device__ __forceinline__ void add32(const float (&x)[32]) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) s += x[i];
    const float cm = s * (1.0f / 32.0f);
    float cm2 = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float d = x[i] - cm;
      cm2 = fmaf(d, d, cm2);
    }
    const float nn = n + 32.0f;
    const float delta = cm - mean;
    mean += delta * (32.0f / nn);
    m2 += cm2 + delta * delta * (n * 32.0f / nn);
    n = nn;
  }
};

// combine the four 64-column groups of a row through shared memory -> (mean, rstd) of the 256-wide row
__device__ __forceinline__ void combine_groups(const RowStats& st, float2* red, int cg, int row, float& mean,
                                               float& rstd) {
  red[cg * kTileM + row] = make_float2(st.mean, st.m2);
  epi_barrier();
  const float2 a = red[row], b = red[kTileM + row], c = red[2 * kTileM + row], d = red[3 * kTileM + row];
  mean = 0.25f * (a.x + b.x + c.x + d.x);
  const float da = a.x - mean, db = b.x - mean, dc = c.x - mean, dd = d.x - mean;
  const float m2 = a.y + b.y + c.y + d.y + 64.0f * (da * da + db * db + dc * dc + dd * dd);
  rstd = rsqrtf(m2 * (1.0f / 256.0f) + 1e-5f);
}

// 32 values -> bf16 -> 4 x 16 B chunks (chunk0 .. chunk0+3) of one 128-byte swizzled smem row
__device__ __forceinline__ void store_row_chunks(uint8_t* row_base, int sw, int chunk0, const float (&y)[32]) {
#pragma unroll
  for (int q4 = 0; q4 < 4; ++q4) {
    uint4 v;
    v.x = LS_PACK_H2(y[8 * q4 + 0], y[8 * q4 + 1]);
    v.y = LS_PACK_H2(y[8 * q4 + 2], y[8 * q4 + 3]);
    v.z = LS_PACK_H2(y[8 * q4 + 4], y[8 * q4 + 5]);
    v.w = LS_PACK_H2(y[8 * q4 + 6], y[8 * q4 + 7]);
    *reinterpret_cast<uint4*>(row_base + (((chunk0 + q4) ^ sw) << 4)) = v;
  }
}

// y[i] = (x[i] * rstd + nmr) * g[i] + b[i]  (nmr = -mean * rstd), g / b read from shared memory (warp-uniform)
__device__ __forceinline__ void normalize32(const float (&x)[32], float rstd, float nmr, const float* g,
                                            const float* b, float (&y)[32]) {
#pragma unroll
  for (int g4 = 0; g4 < 8; ++g4) {
    const float4 gv = reinterpret_cast<const float4*>(g)[g4];
    const float4 bv = reinterpret_cast<const float4*>(b)[g4];
    y[4 * g4 + 0] = fmaf(fmaf(x[4 * g4 + 0], rstd, nmr), gv.x, bv.x);
    y[4 * g4 + 1] = fmaf(fmaf(x[4 * g4 + 1], rstd, nmr), gv.y, bv.y);
    y[4 * g4 + 2] = fmaf(fmaf(x[4 * g4 + 2], rstd, nmr), gv.z, bv.z);
    y[4 * g4 + 3] = fmaf(fmaf(x[4 * g4 + 3], rstd, nmr), gv.w, bv.w);
  }
}

__global__ void __launch_bounds__(kThreads, 1)
tblock_kernel(const __grid_constant__ CUtensorMap mapAtt, const __grid_constant__ CUtensorMap mapWo,
              const __grid_constant__ CUtensorMap mapW1, const __grid_constant__ CUtensorMap mapW2,
              const __grid_constant__ CUtensorMap mapWqkv, const __grid_constant__ CUtensorMap mapU,
              const __grid_constant__ CUtensorMap mapQkvOut, const __grid_constant__ CUtensorMap mapTail,
              const __grid_constant__ TBlockParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA3 = smem + kOffA3;
  uint8_t* sAH = smem + kOffAH;
  uint8_t* sRing = smem + kOffRing;
  // place j of the 8 boxes of A3 + AH that hold the tile's fp32 u (u box j = columns 32 j .. 32 j + 31: even j in the AH
  // region, odd j in A3, which is how the out-proj epilogue reads them) and, before that, att box j (kAttDirect)
  auto att_place = [&](int j) -> uint8_t* { return ((j & 1) ? sA3 : sAH) + (j >> 1) * kSlotBytes; };
  float* sVec = reinterpret_cast<float*>(smem + kOffVec);
  float2* sRed = reinterpret_cast<float2*>(smem + kOffRed);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBars);
  uint64_t* full = bars;                  // [kWideSlots]  TMA -> MMA (the first kSlots of them without the wide ring)
  uint64_t* empty = bars + kWideSlots;    // [2][kWideSlots]  MMA -> TMA (wide ring: [use & 1][slot]; else the first kSlots)
  uint64_t* d_full = bars + 3 * kWideSlots;  // MMA -> epilogue: D holds out-proj / FF2 result
  uint64_t* a3_ready = d_full + 1;   // epilogue -> MMA: A3 written (and D read / rewritten)
  uint64_t* h_full = a3_ready + 1;   // [2] MMA -> epilogue: H[i] holds an FF1 / QKV chunk
  uint64_t* ah_ready = h_full + 2;   // [2] epilogue -> MMA: H[i] drained (and AH[i] written in the FF phase)
  uint64_t* ah_free = ah_ready + 2;  // [2] MMA -> epilogue: FF2 MMAs that read AH[i] have retired
  uint64_t* u_full = ah_free + 2;    // TMA -> epilogue: the u tile sits in the staging boxes (AH region + A3)
  uint64_t* full_b = u_full + 1;       // [kSlotsB] TMA -> MMA: W2 box r of the current FF chunk
  uint64_t* empty_b = full_b + kSlotsB;  // [kSlotsB] MMA -> TMA
  uint64_t* stage_free = empty_b + kSlotsB;  // epilogue -> TMA: the staging region may take this tile's W2 boxes
  uint64_t* full_c = stage_free + 1;         // [8] TMA -> MMA: att box kb of this tile has landed in its A3 / AH place
  uint64_t* empty_c = full_c + 8;            // [8] MMA -> epilogue leader: K block kb retired, u box kb may take the place
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(empty_c + 8);
  static_assert((3 * kWideSlots + 10 + 2 * kSlotsB + 1 + 16) * 8 + 8 <= kBarBytes, "barrier area");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_tiles = (p.R + kTileM - 1) / kTileM;
  const bool head = p.tail_mode == 2;    // LayerNorm(u) + QKV only: the first block of a group
  const bool do_qkv = p.tail_mode != 1;
  // Clusters of kCS CTAs walk the tiles together (tile = group*kCS + rank): all of them stream the same weight
  // sequence, so each CTA fetches 1/kCS of every weight box from L2 and multicasts it to the whole cluster.  A group
  // past the end of the tensor (rows >= R) is a phantom tile: TMA reads zeros and drops the stores.
  const int rank = kCS > 1 ? (int)cluster_ctarank() : 0;
  const int n_groups = (n_tiles + kCS - 1) / kCS;
  const int group0 = blockIdx.x / kCS, group_step = gridDim.x / kCS;
  auto group_skipped = [&](int g) {
    for (int r = 0; r < kCS; ++r)
      if (!tile_all_padding(p, (g * kCS + r) * kTileM)) return false;
    return true;
  };
  long long* tl = p.timeline ? p.timeline + (size_t)blockIdx.x * 256 : nullptr;
#define TL(i)                         \
  do {                                \
    if (tl) tl[(i)] = clock64();      \
  } while (0)

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&mapAtt);
    prefetch_tmap(&mapWo);
    prefetch_tmap(&mapW1);
    prefetch_tmap(&mapW2);
    prefetch_tmap(&mapWqkv);
    prefetch_tmap(&mapU);
    prefetch_tmap(&mapQkvOut);
    prefetch_tmap(&mapTail);
    for (int i = 0; i < kWideSlots; ++i) {
      mbar_init(&full[i], kPair ? 2 : 1);        // pair: one arrive.expect_tx per CTA, on the leader's barrier
      mbar_init(&empty[i], kPair ? 1 : kCS);     // multicast: released by the MMA warp of every CTA of the cluster
      mbar_init(&empty[kWideSlots + i], 1);
    }
    mbar_init(d_full, 1);
    mbar_init(a3_ready, kPair ? 2 * kEpiWarps : kEpiWarps);  // pair: both CTAs' epilogue warps arrive at the leader
    for (int i = 0; i < 2; ++i) {
      mbar_init(&h_full[i], 1);
      mbar_init(&ah_ready[i], kPair ? 2 * kEpiWarps : kEpiWarps);
      mbar_init(&ah_free[i], 1);
    }
    mbar_init(u_full, 1);
    for (int i = 0; i < kSlotsB; ++i) {
      mbar_init(&full_b[i], 1);
      mbar_init(&empty_b[i], 1);
    }
    mbar_init(stage_free, 1);
    for (int i = 0; i < 8; ++i) {
      mbar_init(&full_c[i], 1);
      mbar_init(&empty_c[i], 1);
    }
    fence_barrier_init();
  }
  if (kL2Prefetch && warp == 1 && lane == 0) {
    const int n_boxes = head ? 48 : (do_qkv ? 128 : 80);  // 16 Wo + 32 W1 + 32 W2 (+ 48 Wqkv), 16 KB each
    for (int j = blockIdx.x; j < n_boxes; j += gridDim.x) {
      int q = j;
      if (head || q >= 80) {
        if (!head) q -= 80;
        tma_prefetch_l2_2d(&mapWqkv, (q & 3) * 64, (q >> 2) * 128);
      } else if (q < 16) {
        tma_prefetch_l2_2d(&mapWo, (q >> 1) * 64, (q & 1) * 128);
      } else if (q < 48) {
        q -= 16;
        tma_prefetch_l2_2d(&mapW1, (q & 3) * 64, (q >> 2) * 128);
      } else {
        q -= 48;
        tma_prefetch_l2_2d(&mapW2, (q >> 1) * 64, (q & 1) * 128);
      }
    }
  }
  if (warp == kMmaWarp) {
    __syncwarp();
    if (kPair) {
      tmem_alloc_pair(tmem_slot, 512);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, 512);
      tmem_relinquish();
    }
  }
  if (warp >= kFirstEpiWarp) {
    for (int i = threadIdx.x - kFirstEpiWarp * 32; i < TBLOCK_VEC_FLOATS; i += kEpiThreads) sVec[i] = __ldg(p.vec + i);
  }
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  if (kCS > 1) cluster_sync_all();  // peers' barriers are initialised before anything is multicast at them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();  // the prologue above (and the weight-vector preload) overlapped the attention kernel's tail

  if (warp < kProducerWarps) {
    // ======================================================================== TMA producers
    // One thread can only start a TMA load every ~500 clk (issue latency, measured: profiles/micro/tma_bw3.cu), far
    // less than the MMA warp consumes, but different warps overlap.  kProducerWarps threads walk the same fixed load
    // sequence of a tile; warp w issues the loads whose sequence number is w mod kProducerWarps.  (Separate warps, not
    // lanes of one warp: a lane blocked in mbarrier.try_wait suspends its whole warp.)
    // kProducerLanes == 1 (default): the whole warp walks the load sequence in uniform control flow and one elected lane
    // issues, so the tensor-map pointer, coordinates and barrier addresses stay in uniform registers (inside a
    // single-lane region every UTMALDG is wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop, on the critical path
    // between "slot free" and "load issued").
    constexpr bool kWarpIssue = kProducerLanes == 1;
    if (kWarpIssue || lane < kProducerLanes) {
      const int issuer = warp * kProducerLanes + (kWarpIssue ? 0 : lane);
      const int per_tile = kPair ? (head ? 24 : (do_qkv ? 72 : 48)) : (head ? 48 : (do_qkv ? kOutLoads + 112 : kOutLoads + 64));
      long long seq0 = 0;  // sequence number of the tile's first ring-A load (slot = seq % kSlots, use = seq / kSlots)
      uint32_t tile_n = 0;  // tiles processed by this CTA (ring B: eight uses of every slot per tile)
      for (int g = group0; g < n_groups; g += group_step) {
        const int row0 = (g * kCS + rank) * kTileM;
        if (kWarpIssue ? __shfl_sync(0xffffffffu, (int)group_skipped(g), 0) != 0 : group_skipped(g)) continue;
        // With the second ring, its loads all go through the LAST producer warp, in order: successive uses of one of its
        // slots are then waited for by one thread, which can never be two uses ahead of the consumer (interleaved over
        // several warps they could, and a parity wait cannot tell "two phases ahead" from "done"); the other warps
        // share the ring-A loads.  It also keeps a W2 box from queueing behind a W1 box that waits for a ring-A slot.
        const bool two_rings = kRingB && !head;
        const bool b_warp = two_rings && warp == kProducerWarps - 1;
        const int n_a = two_rings ? kIssuers - kProducerLanes : kIssuers;  // issuers of ring-A loads
        for (int i = two_rings ? 0 : issuer; i < per_tile; i += two_rings ? 1 : kIssuers) {
          // decode load i of the tile: (tensor map, column, row), in exactly the order the MMA warp consumes them
          const CUtensorMap* m;
          int c0, c1;
          bool own_rows = false;
          int c2 = -1;  // >= 0: 3-D weight box (pair mode: 64 rows x 2 K blocks), third coordinate
          int ring_b = -1, chunk_b = 0;  // >= 0: a W2 box of FF chunk chunk_b -> slot ring_b of the second ring
          int a_idx = i;                 // index of this load among the tile's ring-A loads
          if (kPair) {
            auto chunk_half = [&](const CUtensorMap* wm, int chunk, int half) {  // W1 / Wqkv chunk: this CTA's 64 rows
              m = wm, c0 = 0, c1 = chunk * 128 + rank * kPartRows, c2 = half * 2;
            };
            if (head) {
              chunk_half(&mapWqkv, i >> 1, i & 1);
            } else if (i < 16) {  // out-proj: per K block the att box (own rows), then this CTA's 128 rows of Wo
              const int kb = i >> 1;
              if ((i & 1) == 0) m = &mapAtt, c0 = kb * 64, c1 = row0, own_rows = true;
              else m = &mapWo, c0 = kb * 64, c1 = rank * 128, own_rows = true;
            } else if (i < 20) {  // FF1 chunks 0 and 1
              chunk_half(&mapW1, (i - 16) >> 1, i & 1);
            } else if (i < 48) {  // per FF chunk c: W2 (2 K blocks, this CTA's 128 rows), then FF1 chunk c+2
              const int j = i - 20;
              int c, r;
              if (j < 24) c = j >> 2, r = j & 3;
              else c = 6 + ((j - 24) >> 1), r = (j - 24) & 1;
              if (r < 2) m = &mapW2, c0 = c * 128 + r * 64, c1 = rank * 128, own_rows = true;
              else chunk_half(&mapW1, c + 2, r - 2);
            } else {  // next block's QKV weight, 12 chunks
              chunk_half(&mapWqkv, (i - 48) >> 1, i & 1);
            }
          } else if (head) {  // QKV weight only
            m = &mapWqkv, c0 = (i & 3) * 64, c1 = (i >> 2) * 128;
          } else if (kAttDirect && i < kOutLoads) {  // out-proj: per 64-wide K block Wo rows 0-127 and 128-255
            m = &mapWo, c0 = (i >> 1) * 64, c1 = (i & 1) * 128;
          } else if (i < kOutLoads) {  // out-proj: per 64-wide K block the att box, then Wo rows 0-127 and 128-255
            const int kb = i / 3, r = i - kb * 3;
            if (r == 0) m = &mapAtt, c0 = kb * 64, c1 = row0, own_rows = true;
            else m = &mapWo, c0 = kb * 64, c1 = (r - 1) * 128;
          } else if (i < kOutLoads + 8) {  // FF1 chunks 0 and 1
            const int j = i - kOutLoads;
            m = &mapW1, c0 = (j & 3) * 64, c1 = (j >> 2) * 128;
          } else if (i < kOutLoads + 64) {  // per FF chunk c: W2 (2 K blocks x 2 row halves), then FF1 chunk c+2
            const int j = i - (kOutLoads + 8);
            int c, r;
            if (j < 48) c = j >> 3, r = j & 7;
            else c = 6 + ((j - 48) >> 2), r = (j - 48) & 3;
            if (r < 4) {
              m = &mapW2, c0 = c * 128 + (r >> 1) * 64, c1 = (r & 1) * 128;
              if (kRingB) ring_b = r, chunk_b = c;
            } else {
              m = &mapW1, c0 = (r - 4) * 64, c1 = (c + 2) * 128;
            }
            if (kRingB) a_idx = i - (4 * c + (r < 4 ? r : 4));  // W2 boxes before this load travel in ring B
          } else {  // next block's QKV weight, 12 chunks of 128 rows
            const int j = i - (kOutLoads + 64);
            m = &mapWqkv, c0 = (j & 3) * 64, c1 = (j >> 2) * 128;
            if (kRingB) a_idx = i - 32;
          }
          if (two_rings && (ring_b >= 0 ? !b_warp : (b_warp || a_idx % n_a != issuer))) continue;  // another warp's load
          uint64_t* full_bar;
          uint8_t* dst;
          if (kWide) {
            int sl, rc = i, hc = -1;
            uint32_t use;
            if (!head && i >= kOutLoads + 8) {
              if (i < kOutLoads + 64) {  // FF chunk loop: 4 x AH, 5 x ring
                const int f = i - (kOutLoads + 8), q9 = f / 9, m9 = f - q9 * 9;
                if (m9 < 4) hc = q9 * 4 + m9;
                else rc = 24 + q9 * 5 + (m9 - 4);
              } else {
                rc = i - kWideAhPerTile;
              }
            }
            if (hc >= 0) {
              const uint32_t cnt = tile_n * (uint32_t)kWideAhPerTile + (uint32_t)hc;
              sl = (int)(cnt & 3u), use = cnt >> 2;
              if (hc < 4) mbar_wait(stage_free, tile_n & 1);  // the u tile has been read out of the AH boxes
            } else {
              const uint32_t cnt = tile_n * (uint32_t)(per_tile - (head ? 0 : kWideAhPerTile)) + (uint32_t)rc;
              sl = 4 + (int)(cnt % 5u), use = cnt / 5u;
            }
            if (use > 0) mbar_wait(&empty[((use - 1) & 1) * kWideSlots + sl], ((use - 1) >> 1) & 1);
            if (tl && i < 48 && tile_n == 0 && (!kWarpIssue || lane == 0)) tl[64 + i] = clock64();
            full_bar = &full[sl];
            dst = sAH + sl * kSlotBytes;
          } else if (ring_b >= 0) {
            // second ring: slot r holds W2 box r of one chunk at a time; the first box of a tile waits for the epilogue to
            // hand the staging region over, the others for the MMAs that read the slot's previous box
            if (chunk_b == 0) mbar_wait(stage_free, tile_n & 1);
            else mbar_wait(&empty_b[ring_b], (tile_n * 7 + (uint32_t)chunk_b - 1) & 1);
            full_bar = &full_b[ring_b];
            dst = sAH + ring_b * kSlotBytes;
          } else {
            const long long seq = seq0 + a_idx;
            const int slot = (int)(seq % kSlots);
            const uint32_t use = (uint32_t)(seq / kSlots);
            mbar_wait(&empty[slot], (use & 1) ^ 1);
            if (tl && seq < 48 && (!kWarpIssue || lane == 0)) tl[64 + seq] = clock64();  // load `seq` may start (its slot is free)
            full_bar = &full[slot];
            dst = sRing + slot * kRingSlotBytes;
          }
          const int qk6 = kOutLoads + 64 + 24;  // first load of QKV chunk 6 (detailed timeline)
          const bool stamp_q6 = kDetailTl && tl && !kWide && do_qkv && !head && i >= qk6 && i < qk6 + 4 && seq0 == 0;
          if (stamp_q6 && (!kWarpIssue || lane == 0)) tl[216 + 2 * (i - qk6)] = clock64();  // slot free seen by the producer
          if (kWarpIssue && !elect_one()) {
            // (the other lanes only keep the warp's control flow uniform)
          } else if (kPair) {
            // this CTA's half of the box (own rows for att), completion signalled on the LEADER's barrier
            const uint32_t fb = cluster_addr(full_bar, 0);
            mbar_arrive_expect_tx_cluster(fb, kRingSlotBytes);
            if (c2 >= 0) tma_load_3d_pair(dst, m, fb, c0, c1, c2);
            else tma_load_2d_pair(dst, m, fb, c0, c1);
          } else {
            mbar_arrive_expect_tx(full_bar, kSlotBytes);
            if (kCS > 1 && !own_rows) tma_load_2d_mc(dst + rank * kPartBytes, m, full_bar, c0, c1 + rank * kPartRows, kCtaMask);
            else tma_load_2d(dst, m, full_bar, c0, c1);
          }
          if (kWarpIssue) __syncwarp();
          if (stamp_q6 && (!kWarpIssue || lane == 0)) tl[217 + 2 * (i - qk6)] = clock64();  // load issued
        }
        seq0 += (kRingB && !head) ? per_tile - 32 : per_tile;
        tile_n += 1;
      }
    }
  } else if (warp == kMmaWarp) {
    // ======================================================================== MMA issuer
    // The whole warp walks the phases in uniform control flow (every descriptor and TMEM address stays in uniform
    // registers); one elected lane issues the MMAs and commits (see elect_one() in ptx.cuh).
    if (!kPair || rank == 0) {  // pair: the leader CTA issues every MMA of both CTAs
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
#define TLM(i)                                 \
  do {                                         \
    if (tl && lane == 0) tl[(i)] = clock64();  \
  } while (0)
      const uint32_t idesc = make_idesc_bf16(kPair ? 2 * kTileM : kTileM, 128, false, false);
      const uint32_t idesc256 = make_idesc_bf16(2 * kTileM, 256, false, false);  // pair: one N = 256 MMA fills D
      auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t acc) {
        if (kPair) umma_bf16_pair(d, ad, bd, idesc, acc);
        else umma_bf16(d, ad, bd, idesc, acc);
      };
      auto commit = [&](uint64_t* bar) {  // MMA -> epilogue barriers exist in both CTAs
        if (elect_one()) {
          if (kPair) umma_commit_pair(bar);
          else umma_commit(bar);
        }
        __syncwarp();
      };
      auto wait_epi = [&](uint64_t* bar, uint32_t parity) {  // epilogue -> MMA (pair: arrivals come from both CTAs)
        if (kPair) mbar_wait_cluster(bar, parity);
        else mbar_wait(bar, parity);
      };
      int slot = 0;
      uint32_t phase = 0;
      uint32_t a3_cnt = 0;
      uint32_t fills0 = 0, fills1 = 0;      // fills issued into H[i]
      uint32_t drained0 = 0, drained1 = 0;  // fills of H[i] known to be consumed by the epilogue
      // wait for the ring slot `ahead` positions after the current one; returns its descriptor
      int n_full = 0;  // timeline aid: arrival of the first slots as seen by this thread
      uint32_t tile_n = 0;  // tiles processed (second ring / wide ring parities)
      // wide ring: the two sub-rings' next slot and its use number, and the position in the FF loop's 4 x AH, 5 x ring pattern
      int r_slot = 0, h_slot = 0, f_pos = 0;
      uint32_t r_use = 0, h_use = 0;
      bool in_f = false;
      auto wide_peek = [&](int ahead, uint32_t& use) -> int {  // slot (and use number) of the box `ahead` after the next one
        int rs = r_slot, hs = h_slot, fp = f_pos;
        uint32_t ru = r_use, hu = h_use;
        for (int a = 0;; ++a) {
          const bool ah = in_f && fp < 4;
          if (a == ahead) {
            use = ah ? hu : ru;
            return ah ? hs : 4 + rs;
          }
          if (ah) {
            if (++hs == 4) hs = 0, ++hu;
          } else {
            if (++rs == 5) rs = 0, ++ru;
          }
          if (in_f && ++fp == 9) fp = 0;
        }
      };
      auto wide_advance = [&](int n) {
        for (int a = 0; a < n; ++a) {
          if (in_f && f_pos < 4) {
            if (++h_slot == 4) h_slot = 0, ++h_use;
          } else {
            if (++r_slot == 5) r_slot = 0, ++r_use;
          }
          if (in_f && ++f_pos == 9) f_pos = 0;
        }
      };
      auto slot_desc = [&](int ahead) -> uint64_t {
        if (kWide) {
          uint32_t use;
          const int sl = wide_peek(ahead, use);
          mbar_wait(&full[sl], use & 1);
          tc_fence_after();
          if (tl && lane == 0 && n_full < 16) tl[112 + n_full] = clock64();
          n_full += (ahead == 0);
          return make_smem_desc_sw128(smem_u32(sAH + sl * kSlotBytes));
        }
        int s = slot + ahead;
        uint32_t ph = phase;
        if (s >= kSlots) s -= kSlots, ph ^= 1;
        if (kPair) mbar_wait_cluster(&full[s], ph);
        else mbar_wait(&full[s], ph);
        tc_fence_after();
        if (tl && lane == 0 && n_full < 16) tl[112 + n_full] = clock64();
        n_full += (ahead == 0);
        return make_smem_desc_sw128(smem_u32(sRing + s * kRingSlotBytes));
      };
      auto release = [&](int n) {  // hand the next n slots back once the MMAs issued so far retire
        if (kWide) {
          if (elect_one()) {
            for (int j = 0; j < n; ++j) {
              uint32_t use;
              const int sl = wide_peek(j, use);
              umma_commit(&empty[(use & 1) * kWideSlots + sl]);
            }
          }
          __syncwarp();
          wide_advance(n);
          return;
        }
        if (elect_one()) {
          int sl = slot;
          for (int j = 0; j < n; ++j) {
            if (kPair) umma_commit_pair(&empty[sl]);
            else if (kCS > 1) umma_commit_mc(&empty[sl], kCtaMask);
            else umma_commit(&empty[sl]);
            if (++sl == kSlots) sl = 0;
          }
        }
        __syncwarp();
        for (int j = 0; j < n; ++j)
          if (++slot == kSlots) slot = 0, phase ^= 1;
      };
      // the same in two halves, so that the commits ride in the election that issued the MMAs (one ELECT / BRA.DIV
      // sequence per weight box instead of two): release_elected inside the elected region, advance by every lane
      auto release_elected = [&](int n) {
        int sl = slot;
        for (int j = 0; j < n; ++j) {
          if (kPair) umma_commit_pair(&empty[sl]);
          else if (kCS > 1) umma_commit_mc(&empty[sl], kCtaMask);
          else umma_commit(&empty[sl]);
          if (++sl == kSlots) sl = 0;
        }
      };
      auto advance = [&](int n) {
        __syncwarp();
        for (int j = 0; j < n; ++j)
          if (++slot == kSlots) slot = 0, phase ^= 1;
      };
      auto wait_drained = [&](int i) {  // the epilogue has finished with the latest fill of H[i]
        const uint32_t f = i ? fills1 : fills0;
        if ((i ? drained1 : drained0) < f) {
          wait_epi(&ah_ready[i], (f - 1) & 1);
          tc_fence_after();
          if (i) drained1 = f;
          else drained0 = f;
        }
      };
      // H[i] = A3 (128 x 256, K-major in smem) . Wchunk^T, weights from 4 ring slots
      auto gemm_from_a3 = [&](int i, int tlb = -1) {  // tlb >= 0: detailed timeline stamps of this call (development aid)
        if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb] = clock64();
        wait_drained(i);
        if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb + 1] = clock64();
        const uint32_t d = tmem_u + kTmemH + (uint32_t)i * 128;
        for (int kb = 0; kb < kC / 64; ++kb) {
          // pair: a slot holds two K blocks of this CTA's 64 weight rows (8 KB each)
          const uint64_t bdesc = slot_desc(0) + (kPair ? (uint64_t)((kb & 1) * (8192 >> 4)) : 0);
          if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb + 2 + kb] = clock64();
          const uint64_t adesc = make_smem_desc_sw128(smem_u32(sA3 + kb * kSlotBytes));
          if (kMergeElect && !kPair) {
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k) mma(d, adesc + 2 * k, bdesc + 2 * k, (kb | k) != 0 ? 1u : 0u);
              release_elected(1);
            }
            advance(1);
            continue;
          }
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) mma(d, adesc + 2 * k, bdesc + 2 * k, (kb | k) != 0 ? 1u : 0u);
          }
          if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb + 56 + 2 * kb] = clock64();  // MMAs issued
          if (!kPair || (kb & 1)) release(1);
          if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb + 57 + 2 * kb] = clock64();  // slot handed back (commit issued)
        }
        commit(&h_full[i]);
        if (kDetailTl && tl && tlb >= 0 && lane == 0) tl[tlb + 6] = clock64();
        if (i) fills1 += 1;
        else fills0 += 1;
      };
      const uint32_t dD = tmem_u + kTmemD;
      TLM(0);
      for (int g = group0; g < n_groups; g += group_step, ++tile_n) {
        if (__shfl_sync(0xffffffffu, (int)group_skipped(g), 0)) {
          --tile_n;
          continue;
        }
        if (g != group0) tl = nullptr;
        if (!head) {
        // ---- out-proj: D = att . Wo^T.  D is free: the previous tile's second a3_ready was waited below.
        for (int kb = 0; kb < kInner / 64; ++kb) {
          if (kAttDirect) {
            // A = att box kb in its own place (A3 / AH, see att_place); the ring holds the two Wo boxes of the K block
            mbar_wait(&full_c[kb], tile_n & 1);
            tc_fence_after();
            const uint64_t adesc = make_smem_desc_sw128(smem_u32(att_place(kb)));
            const uint64_t b0 = slot_desc(0);
            const uint64_t b1 = slot_desc(1);
            if (kb == 0) TLM(1);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t acc = (kb | k) != 0 ? 1u : 0u;
                mma(dD, adesc + 2 * k, b0 + 2 * k, acc);
                mma(dD + 128, adesc + 2 * k, b1 + 2 * k, acc);
              }
              if (!kWide) release_elected(2);
              umma_commit(&empty_c[kb]);  // K block kb has retired: u box kb may take the att box's place
            }
            if (kWide) release(2);
            else advance(2);
            continue;
          }
          const uint64_t adesc = slot_desc(0);
          const uint64_t b0 = slot_desc(1);
          if (kPair) {  // b0 = this CTA's 128 rows of Wo: the pair's operand is all 256
            if (kb == 0) TLM(1);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_bf16_pair(dD, adesc + 2 * k, b0 + 2 * k, idesc256, (kb | k) != 0 ? 1u : 0u);
            }
            release(2);
            continue;
          }
          const uint64_t b1 = slot_desc(2);
          if (kb == 0) TLM(1);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t acc = (kb | k) != 0 ? 1u : 0u;
              mma(dD, adesc + 2 * k, b0 + 2 * k, acc);
              mma(dD + 128, adesc + 2 * k, b1 + 2 * k, acc);
            }
            if (kMergeElect) release_elected(3);
          }
          if (kMergeElect) advance(3);
          else release(3);
        }
        commit(d_full);
        TLM(2);
        // ---- FF: H[c&1] = n3 . W1[c]^T ; D += gelu(H[c&1]) . W2[:, c]^T
        wait_epi(a3_ready, a3_cnt & 1);  // n3 in A3, u' written back to D
        a3_cnt += 1;
        tc_fence_after();
        TLM(3);
        gemm_from_a3(0);
        gemm_from_a3(1);
        in_f = true, f_pos = 0;  // (wide ring) the loads of the chunk loop alternate between the AH boxes and the ring
        for (int c = 0; c < kFF / 128; ++c) {
          const int i = c & 1;
          if (kDetailTl && c == 4) TLM(128);
          wait_drained(i);  // AH[i] holds gelu(FF1 chunk c)
          TLM(4 + c);
          for (int kb2 = 0; kb2 < 2; ++kb2) {
            // A = gelu(FF1 chunk c), packed 16-bit pairs in TENSOR MEMORY: the GELU epilogue wrote the pairs of column
            // group cg over the first 16 of that group's 32 columns of H[i] (tcgen05.mma TS form: no shared-memory read
            // for A, 73 instead of 102 clk per N = 128 MMA; profiles/micro/mma_bw.cu).  K step k of this 64-wide K block
            // covers chunk columns [64 kb2 + 16 k, +16) = column group 2 kb2 + k / 2, packed columns 8 (k & 1) .. +8.
            const uint32_t a_tm = tmem_u + kTmemH + (uint32_t)i * 128 + (uint32_t)kb2 * 64;
            const uint64_t adesc = make_smem_desc_sw128(smem_u32(sAH + i * 2 * kSlotBytes + kb2 * kSlotBytes));
            if (kPair) {  // this CTA's 128 rows of W2[:, chunk]: one N = 256 MMA per K step
              const uint64_t b0 = slot_desc(0);
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_bf16_pair(dD, adesc + 2 * k, b0 + 2 * k, idesc256, 1u);
              }
              release(1);
              continue;
            }
            uint64_t b0, b1;
            if (kRingB) {  // W2 boxes 2 kb2 and 2 kb2 + 1 of this chunk sit in their own slots of the second ring
              const uint32_t par = (tile_n * 8 + (uint32_t)c) & 1;
              mbar_wait(&full_b[2 * kb2], par);
              if (kDetailTl && c == 4) TLM(129 + 2 * kb2);
              mbar_wait(&full_b[2 * kb2 + 1], par);
              tc_fence_after();
              b0 = make_smem_desc_sw128(smem_u32(sAH + (2 * kb2) * kSlotBytes));
              b1 = make_smem_desc_sw128(smem_u32(sAH + (2 * kb2 + 1) * kSlotBytes));
            } else {
              b0 = slot_desc(0);
              if (kDetailTl && c == 4) TLM(129 + 2 * kb2);
              b1 = slot_desc(1);
            }
            if (kDetailTl && c == 4) TLM(130 + 2 * kb2);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                if (kFf2Ts) {
                  const uint32_t a_k = a_tm + (uint32_t)(k >> 1) * 32 + (uint32_t)(k & 1) * 8;
                  umma_bf16_ts(dD, a_k, b0 + 2 * k, idesc, 1u);
                  umma_bf16_ts(dD + 128, a_k, b1 + 2 * k, idesc, 1u);
                } else {
                  mma(dD, adesc + 2 * k, b0 + 2 * k, 1u);
                  mma(dD + 128, adesc + 2 * k, b1 + 2 * k, 1u);
                }
              }
              // (the last chunk's boxes are not handed back: the next tile's first boxes wait for stage_free instead)
              if (kRingB && c + 1 < kFF / 128) umma_commit(&empty_b[2 * kb2]), umma_commit(&empty_b[2 * kb2 + 1]);
              if (!kRingB && kMergeElect) release_elected(2);
            }
            if (kRingB) __syncwarp();
            else if (kMergeElect) advance(2);
            else release(2);
          }
          if (!kFf2Ts) commit(&ah_free[i]);  // (TS form: H[i] is reused in tensor-pipe order, nothing to signal)
          if (kDetailTl && c == 4) TLM(133);
          if (c + 2 < kFF / 128) gemm_from_a3(i, kDetailTl && c == 4 ? 134 : -1);
        }
        in_f = false;
        commit(d_full);
        TLM(12);
        }  // !head
        // ---- tail: D drained by the epilogue (and, tail 0 / 2, the LayerNorm output written to A3)
        wait_epi(a3_ready, a3_cnt & 1);
        a3_cnt += 1;
        tc_fence_after();
        TLM(13);
        if (do_qkv)
          for (int c = 0; c < kQKV / 128; ++c) {
            gemm_from_a3(c & 1, kDetailTl && c == 6 ? 144 : -1);
            TLM(14 + c);
          }
        TLM(26);
      }
    }
  } else {
#undef TLM
    // ======================================================================== epilogue warps
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int cg = (warp - kFirstEpiWarp) >> 2;  // column group: 64 of D's 256 columns, 32 of an H chunk's 128
    const int row = q * 32 + lane;
    const int sw = row & 7;
    const bool leader = threadIdx.x == kFirstEpiWarp * 32;  // issues the TMA loads / stores of the staging boxes
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    // Staging boxes (16 KB = 128 rows x 128 B, 128B swizzle) for TMA loads of u and TMA stores of u'' / qkv / tail:
    // outside the FF phase the AH region holds 4 of them; while the out-proj MMAs run, A3 is free as well and
    // takes the other half of the u tile.  Thread (row, cg) only ever touches row `row` of box `cg`, in both regions.
    uint8_t* stage = sAH;
    uint32_t d_cnt = 0, u_cnt = 0;
    uint32_t h_cnt0 = 0, h_cnt1 = 0;    // H[i] fills consumed
    uint32_t ah_cnt0 = 0, ah_cnt1 = 0;  // AH[i] writes done
    // one arrival per warp: every lane's smem / TMEM accesses are ordered before lane 0's arrive by __syncwarp
    auto warp_arrive = [&](uint64_t* bar) {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kPair) mbar_arrive_cluster(cluster_addr(bar, 0));  // epilogue -> MMA barriers live in the leader CTA
        else mbar_arrive(bar);
      }
    };
    for (int g = group0; g < n_groups; g += group_step) {
      const int row0 = (g * kCS + rank) * kTileM;
      if (group_skipped(g)) continue;
      const int grow = row0 + row;
      bool valid = grow < p.R;
      if (valid && p.lengths) {
        const int b = grow / p.T;
        valid = grow - b * p.T < p.lengths[b];
      }
      long long* tle = (leader && g == group0) ? tl : nullptr;
#define TLE(i)                        \
  do {                                \
    if (tle) tle[(i)] = clock64();    \
  } while (0)
      if (warp == kFirstEpiWarp) {
        if (leader) {
          // the previous tile's stores have left the staging boxes; its QKV MMAs (A3 readers) retired before the
          // last h_full this thread waited on
          bulk_wait_read<0>();
          mbar_arrive_expect_tx(u_full, 8 * kSlotBytes);
        }
        __syncwarp();
        if (kAttDirect && !head) {
          // att boxes first (all eight in flight at once), each followed into the same place by its u box once the
          // MMAs of that K block have retired; the last u box lands one TMA round trip after the out-proj
          if (lane < 8) {
            mbar_arrive_expect_tx(&full_c[lane], kSlotBytes);
            tma_load_2d(att_place(lane), &mapAtt, &full_c[lane], lane * 64, row0);
          }
          __syncwarp();
          if (lane == 0) {
            for (int j = 0; j < 8; ++j) {
              mbar_wait(&empty_c[j], u_cnt & 1);
              tma_load_2d(att_place(j), &mapU, u_full, j * 32, row0);
            }
          }
          __syncwarp();
        } else if (lane < 8) {  // one box per lane: the issue latencies overlap
          tma_load_2d(att_place(lane), &mapU, u_full, lane * 32, row0);
        }
      }

      // ------------------------------------------------ out-proj epilogue: u' = D + bo + u ; n3 = LN(u')
      {
        mbar_wait(u_full, u_cnt & 1);
        u_cnt += 1;
        if (!head) {
          mbar_wait(d_full, d_cnt & 1);
          d_cnt += 1;
        }
        tc_fence_after();
        TLE(32);
        // Only 32 values are live at a time: u' goes back to TMEM (FF2 accumulates onto it anyway) and is re-read
        // for the LayerNorm pass.  Registers are scarce here -- a spill costs an L2 round trip, the L1 is all smem.
        // (Measured, profiles/r02_timeline_tblock_ln_detail.log: pass 1 costs 1.5-2.0 k clk per 32-column chunk, pass 2
        // 1.4 k; keeping columns 32..63 in registers across the barrier instead of re-reading them takes pass 2 from
        // 2.85 k to 2.8 k -- the chunk time is the per-column constants (48 LDS.128 per thread and LayerNorm), the
        // FMAs / conversions and the swizzled stores of 16 warps, not the tcgen05.ld -- and four accumulator chains in
        // the statistics change nothing; neither is kept.)
        RowStats st;
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          const int col = cg * 64 + ch * 32;
          const uint8_t* urow = (ch ? sA3 : stage) + cg * kSlotBytes + row * 128;
          float x[32];
          if (head) {  // x = u
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 uv = *reinterpret_cast<const float4*>(urow + ((k ^ sw) << 4));
              x[4 * k + 0] = uv.x, x[4 * k + 1] = uv.y, x[4 * k + 2] = uv.z, x[4 * k + 3] = uv.w;
            }
          } else {
            tmem_ld32(trow + kTmemD + col, reinterpret_cast<uint32_t(&)[32]>(x));
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 uv = *reinterpret_cast<const float4*>(urow + ((k ^ sw) << 4));
              const float4 bo = reinterpret_cast<const float4*>(sVec + V_BO + col)[k];
              x[4 * k + 0] += bo.x + uv.x;
              x[4 * k + 1] += bo.y + uv.y;
              x[4 * k + 2] += bo.z + uv.z;
              x[4 * k + 3] += bo.w + uv.w;
            }
          }
          st.add32(x);
          tmem_st32(trow + kTmemD + col, reinterpret_cast<const uint32_t(&)[32]>(x));
          if (kDetailTl) TLE(56 + ch);
        }
        tmem_st_wait();
        if (kDetailTl) TLE(58);
        float mean, rstd;
        combine_groups(st, sRed, cg, row, mean, rstd);  // the barrier inside also orders every thread's u reads
        const float nmr = -mean * rstd;                 // before the A3 writes below (A3 held half of the u tile)
        if (kDetailTl) TLE(59);
        // every thread is done with the u tile and the previous tile's stores have left the staging region (the leader
        // waited for them before loading u): it may take this tile's W2 boxes
        if ((kRingB || kWide) && leader && !head) mbar_arrive(stage_free);
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          const int col = cg * 64 + ch * 32;
          float x[32];
          tmem_ld32(trow + kTmemD + col, reinterpret_cast<uint32_t(&)[32]>(x));
          tmem_ld_wait();
          normalize32(x, rstd, nmr, sVec + (head ? V_G1N : V_G3) + col, sVec + (head ? V_BE1N : V_BE3) + col, x);
          store_row_chunks(sA3 + cg * kSlotBytes + row * 128, sw, ch * 4, x);
          if (kDetailTl) TLE(60 + ch);
        }
        tmem_st_wait();
        warp_arrive(a3_ready);
        TLE(33);
      }

      // ------------------------------------------------ FF1 chunks: AH[i] = gelu(H[i] + b1)
      for (int c = 0; c < (head ? 0 : kFF / 128); ++c) {
        const int i = c & 1;
        if (kDetailTl && c == 4) TLE(160);
        mbar_wait(&h_full[i], (i ? h_cnt1 : h_cnt0) & 1);
        if (i) h_cnt1 += 1;
        else h_cnt0 += 1;
        tc_fence_after();
        if (kDetailTl && c == 4) TLE(161);
        float y[32];
        tmem_ld32(trow + kTmemH + i * 128 + cg * 32, reinterpret_cast<uint32_t(&)[32]>(y));
        tmem_ld_wait();
        if (kDetailTl && c == 4) TLE(162);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 b1 = reinterpret_cast<const float4*>(sVec + V_B1 + c * 128 + cg * 32)[k];
          y[4 * k + 0] = gelu_fast(y[4 * k + 0] + b1.x);
          y[4 * k + 1] = gelu_fast(y[4 * k + 1] + b1.y);
          y[4 * k + 2] = gelu_fast(y[4 * k + 2] + b1.z);
          y[4 * k + 3] = gelu_fast(y[4 * k + 3] + b1.w);
        }
        if (kDetailTl && c == 4) TLE(163);
        if (!kFf2Ts) {
          const uint32_t ahc = i ? ah_cnt1 : ah_cnt0;
          if (ahc >= 1) mbar_wait(&ah_free[i], (ahc - 1) & 1);  // FF2 of chunk c-2 has read AH[i]
          if (i) ah_cnt1 += 1;
          else ah_cnt0 += 1;
          store_row_chunks(sAH + (i * 2 + (cg >> 1)) * kSlotBytes + row * 128, sw, (cg & 1) * 4, y);
        } else {
          // 32 values -> 16 packed pairs, written over the first 16 of this thread's own 32 columns of H[i]: the A
          // operand of FF2 chunk c lives in tensor memory.  FF1 chunk c + 2 overwrites H[i] only after FF2 chunk c
          // (tcgen05.mma instructions execute in issue order), so no "A consumed" barrier is needed.
          uint32_t pk[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) pk[k] = LS_PACK_H2(y[2 * k], y[2 * k + 1]);
          tmem_st16(trow + kTmemH + i * 128 + cg * 32, pk);
          tmem_st_wait();
        }
        if (kDetailTl && c == 4) TLE(164);
        warp_arrive(&ah_ready[i]);
        if (kDetailTl && c == 4) TLE(165);
        TLE(34 + c);
      }

      // ------------------------------------------------ FF2 epilogue: u'' = D + b2
      if (!head) {
        mbar_wait(d_full, d_cnt & 1);
        d_cnt += 1;
        tc_fence_after();
      }
      TLE(42);
      // u'' = D + b2, 32 columns at a time (see the register note above)
      auto load_u2 = [&](int ch, float (&x)[32]) {
        const int col = cg * 64 + ch * 32;
        tmem_ld32(trow + kTmemD + col, reinterpret_cast<uint32_t(&)[32]>(x));
        tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 b2 = reinterpret_cast<const float4*>(sVec + V_B2 + col)[k];
          x[4 * k + 0] += b2.x;
          x[4 * k + 1] += b2.y;
          x[4 * k + 2] += b2.z;
          x[4 * k + 3] += b2.w;
        }
      };
      if (head) {
        epi_barrier();  // every warp is done with the u staging boxes: the QKV chunks below reuse them
      } else if (!do_qkv) {
        // masked bf16 copy of u'': this thread's 64 columns are one full row of staging box cg -> TMA store
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          float x[32];
          load_u2(ch, x);
          if (!valid) {
#pragma unroll
            for (int k = 0; k < 32; ++k) x[k] = 0.f;
          }
          store_row_chunks(stage + cg * kSlotBytes + row * 128, sw, ch * 4, x);
        }
        warp_arrive(a3_ready);  // D is drained
        epi_barrier();
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k) tma_store_2d(&mapTail, stage + k * kSlotBytes, k * 64, row0);
          bulk_commit();
        }
      } else {
        // u'' (fp32) leaves through the 4 staging boxes in two rounds of 32 columns per column group
        auto stage_u = [&](const float (&v)[32]) {
          uint8_t* dst = stage + cg * kSlotBytes + row * 128;
#pragma unroll
          for (int k = 0; k < 8; ++k)
            *reinterpret_cast<float4*>(dst + ((k ^ sw) << 4)) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
          fence_proxy_async_smem();
        };
        auto store_u = [&](int ch) {
#pragma unroll
          for (int k = 0; k < 4; ++k) tma_store_2d(&mapU, stage + k * kSlotBytes, k * 64 + ch * 32, row0);
          bulk_commit();
        };
        // pass 1: finish u'' (bias), statistics, park it in D again; round 0 of the fp32 store is staged on the way
        RowStats st;
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          float x[32];
          load_u2(ch, x);
          st.add32(x);
          tmem_st32(trow + kTmemD + cg * 64 + ch * 32, reinterpret_cast<const uint32_t(&)[32]>(x));
          if (ch == 0) stage_u(x);
        }
        tmem_st_wait();
        float mean, rstd;
        combine_groups(st, sRed, cg, row, mean, rstd);  // contains the barrier that also publishes round 0
        if (leader) store_u(0);
        const float nmr = -mean * rstd;
        // pass 2: next block's LayerNorm -> A3
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          const int col = cg * 64 + ch * 32;
          float x[32];
          tmem_ld32(trow + kTmemD + col, reinterpret_cast<uint32_t(&)[32]>(x));
          tmem_ld_wait();
          normalize32(x, rstd, nmr, sVec + V_G1N + col, sVec + V_BE1N + col, x);
          store_row_chunks(sA3 + cg * kSlotBytes + row * 128, sw, ch * 4, x);
        }
        // round 1 of the fp32 store re-reads its 32 columns from D.  D is rewritten only by the next tile's
        // out-proj MMAs, which are issued after all 12 QKV chunks -- and those need every epilogue warp to have
        // drained chunks 0..9, i.e. to be past this point.
        {
          float x[32];
          tmem_ld32(trow + kTmemD + cg * 64 + 32, reinterpret_cast<uint32_t(&)[32]>(x));
          tmem_ld_wait();
          warp_arrive(a3_ready);  // n1 in A3: the QKV MMAs may start
          TLE(43);
          if (leader) bulk_wait_read<0>();
          epi_barrier();
          stage_u(x);
        }
        epi_barrier();
        if (leader) {
          store_u(1);
          bulk_wait_read<0>();  // the QKV chunks below reuse the staging boxes
        }
        epi_barrier();
      }
      if (do_qkv) {
        // -------------------------------------------- QKV chunks of the next block -> staging pair -> TMA store
        for (int c = 0; c < kQKV / 128; ++c) {
          const int i = c & 1;
          if (kDetailTl && c == 6) TLE(170);
          mbar_wait(&h_full[i], (i ? h_cnt1 : h_cnt0) & 1);
          if (i) h_cnt1 += 1;
          else h_cnt0 += 1;
          tc_fence_after();
          if (kDetailTl && c == 6) TLE(171);
          float y[32];
          tmem_ld32(trow + kTmemH + i * 128 + cg * 32, reinterpret_cast<uint32_t(&)[32]>(y));
          tmem_ld_wait();
          warp_arrive(&ah_ready[i]);  // H[i] is drained: the MMA warp may refill it
          if (kDetailTl && c == 6) TLE(172);
          // staging pair i is free: the leader waited for the store of chunk c-2 before the barrier of chunk c-1
          store_row_chunks(stage + (i * 2 + (cg >> 1)) * kSlotBytes + row * 128, sw, (cg & 1) * 4, y);
          fence_proxy_async_smem();
          if (kDetailTl && c == 6) TLE(173);
          if (leader) bulk_wait_read<0>();  // store of chunk c-1 (issued a whole chunk ago) has left pair i^1
          if (kDetailTl && c == 6) TLE(174);
          epi_barrier();
          if (kDetailTl && c == 6) TLE(175);
          if (leader) {
            tma_store_2d(&mapQkvOut, stage + (i * 2 + 0) * kSlotBytes, c * 128, row0);
            tma_store_2d(&mapQkvOut, stage + (i * 2 + 1) * kSlotBytes, c * 128 + 64, row0);
            bulk_commit();
          }
          if (kDetailTl && c == 6) TLE(176);
          TLE(44 + c);
        }
      }
    }
    if (leader) bulk_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (kCS > 1) cluster_sync_all();  // no CTA leaves while a peer may still multicast into it
  if (warp == kMmaWarp) {
    tc_fence_after();
    if (kPair) tmem_dealloc_pair(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

cudaError_t LS_FN(launch_tblock)(const TBlockMaps& m, const TBlockParams& p, int num_sms, cudaStream_t stream,
                                 int* plan_out) {
#if !LS_HALF_FP16
  if (p.fp16) return launch_tblock_fp16(m, p, num_sms, stream, plan_out);  // fp16-operand build of this file
#endif
  if (p.R <= 0 || p.T <= 0 || p.vec == nullptr || num_sms < kCS) return cudaErrorInvalidValue;
  static std::atomic<unsigned long long> optin{0};  // one bit per device
  if (cudaError_t e = smem_optin_once(optin, reinterpret_cast<const void*>(tblock_kernel), kSmemBytes); e != cudaSuccess) return e;
  const int n_tiles = (p.R + kTileM - 1) / kTileM;
  const int n_groups = (n_tiles + kCS - 1) / kCS;
  int max_clusters = num_sms / kCS;
  if (kCS > 1) {
    // clusters are placed inside one GPC: ask how many fit at once.  The answer depends on the device only, so it is
    // asked once per device (racing first calls may both ask; they get the same answer).
    static std::atomic<int> fit[64];  // clusters of this kernel that fit at once, per device (0: not asked yet)
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return e;
    int n = fit[dev & 63].load(std::memory_order_acquire);
    if (n == 0) {
      cudaLaunchConfig_t qc = {};
      qc.gridDim = dim3(num_sms / kCS * kCS), qc.blockDim = dim3(kThreads), qc.dynamicSmemBytes = kSmemBytes;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = kCS, qa[0].val.clusterDim.y = 1, qa[0].val.clusterDim.z = 1;
      qc.attrs = qa, qc.numAttrs = 1;
      if (cudaOccupancyMaxActiveClusters(&n, tblock_kernel, &qc) != cudaSuccess || n < 0) n = 0;
      if (n > 0) fit[dev & 63].store(n, std::memory_order_release);
    }
    if (n > 0 && n < max_clusters) max_clusters = n;
  }
  const int grid = (n_groups < max_clusters ? n_groups : max_clusters) * kCS;
  if (plan_out) {
    const int ctas_groups = grid / kCS;
    plan_out[0] = grid;
    plan_out[1] = (n_groups + ctas_groups - 1) / ctas_groups;
  }
  const double rows = (double)p.R;
  const double macs = (p.tail_mode == 2 ? 0.0 : (double)kInner * kC + 2.0 * kC * kFF) + (p.tail_mode != 1 ? (double)kC * kQKV : 0.0);
  const double bytes = (p.tail_mode == 2 ? rows * (kC * 4.0 + kQKV * 2.0)
                                          : rows * (kInner * 2.0 + kC * 4.0 + (p.tail_mode == 0 ? kC * 4.0 + kQKV * 2.0 : kC * 2.0))) +
                       macs * 2.0;
  TBlockParams pp = p;
  pp.timeline = (g_debug_buffer && g_debug_bytes >= (long long)grid * 256 * 8) ? g_debug_buffer : nullptr;
  ProfScope prof(stream, PK_TBLOCK, 2.0 * rows * macs, bytes);
  count_launch();
  return launch_pdl(tblock_kernel, dim3(grid), dim3(kThreads), (size_t)kSmemBytes, stream, kCS, m.att, m.wo, m.w1,
                    m.w2, m.wqkv, m.u, m.qkv_out, m.tail_out, pp);
}

}  // namespace ls
