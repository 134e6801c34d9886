// K5-TC: the gather-GEMM convolution on 5th-gen tensor cores (tcgen05 + TMEM), fp32-faithful via 3xTF32.
//
// Same contract as conv_rows_kernel (conv.cu), different engine.  One CTA per SM owns a 256 x N output tile
// (two UMMA M=128 halves sharing one B tile, N = 128 / 64 / 32) and walks K = (c0 + c1) x taps in 32-channel chunks,
// the taps of a channel chunk innermost (their source rows overlap: L2 hits).
// Warp-specialised, mbarrier-pipelined (no CTA-wide barrier inside the K loop):
//
//   gather warps (8-12)
//     * implicit im2col by the TMA: `cp.async.bulk.tensor.2d...tile::gather4` fetches the 128-byte channel slice of
//       four arbitrary source rows (indices from the per-tile tap table; row -1 = inactive / padded tap and the
//       channel tail are zero-filled by the TMA) into a raw fp32, 128B-swizzled shared tile, completion by mbarrier
//       transaction bytes.  3x3 layers: one fill per (chunk, dy) serves the three dx taps (shared-tap form, below);
//       1x1 stages over consecutive rows: one tiled load of the whole 256-row box;
//   weight loader (warp 13)
//     * B (weights) is pre-split, pre-swizzled by wmd_pack_conv_weight_tc_f32 into one [hi | lo] image per (n-tile,
//       chunk): a single cp.async.bulk per chunk into a 3- or 4-deep ring, B_STAGES - 1 chunks ahead of the MMAs;
//   split warps (0-7), thread = tile row = TMEM lane
//     * read the row's 128 bytes back (the swizzle makes this transposed read conflict-free), split x = hi + lo
//       (hi = x with the 13 low mantissa bits cleared, lo = x - hi: exact) and write hi / lo into TENSOR MEMORY with
//       tcgen05.st - the MMAs take A from TMEM (".ts" form), because an SS-mode M=128 x N=128 MMA would need the
//       full 128 B/clk of shared-memory bandwidth three times per k-step;
//   issuers (warps 14-15, one per M half = one per accumulator)
//     * whole warp in the loop, one elected lane issues: 4 k-steps x 3 terms (lo*hi + hi*lo + hi*hi) per chunk, then
//       commits to the mbarriers that recycle the TMEM A stage / shared B stage;
//   all 16 warps
//     * the tensor core's fp32 accumulation rounds toward zero, a bias that grows linearly with K (measured
//       ~6.5e-9 * K relative).  So accumulation runs in EPOCHS of kFlushChunks chunks: a finished epoch is drained
//       (tcgen05.ld) into per-thread fp32 registers with round-to-nearest adds and the TMEM accumulators are
//       re-zeroed.  Each thread ends up owning one output row x N/2 channels: bias + activation (picked once per tile,
//       vector bias loads: the epilogue is instruction bound) + one contiguous store;
//     * balanced scheduling (long reductions): whole tiles for the full rounds, the (tile, chunk) units of the remainder
//       dealt out evenly on the device (stream-K); the last segment of a cut tile to arrive sums all segments in slab
//       order, cooperatively and coalesced.
// What bounds it (scripts/tc_layer_trace.py, scripts/tc_ablate.py, DESIGN.md 4): the tensor pipe.  24 UTCHMMAs per chunk
// cost 64 clk each at N = 128 (1536 clk) and ~52 clk at any N <= 64 (an instruction-rate floor); the feed - A 16 KB
// (shared-tap) + B 32 KB per chunk through an L2 that delivers ~45 B/clk per SM when all SMs stream - fits under it.
// Optional fp16-pair operand form (F16 = true, wmd_conv_desc.precision): x 2^e = h1 + h2 as fp16, kind::f16 MMAs with K = 16
// (half the instructions), scale from the sources' max |x| (device scalars), weights' scale in the packed image's header.
// Shared-tap gather (SH = true, every 3x3 layer): the three dx taps of a (channel chunk, dy) read almost the same source
// rows - tap dx of tile row r is tap 0 of row r + dx whenever the two output pixels are neighbours in the active list.
// One raw stage fill per (chunk, dy) therefore serves THREE chunks: slots 0..255 hold the dx = 0 sources of the tile's
// rows, slots 256.. the few "extra" rows that no centre tap fetches (run ends, list gaps); a per-tile slot table
// (uint16 per (source, dy, side, row)) tells the split warps which slot feeds each row of the dx = +-1 chunks.  The
// L2->SM traffic of the A operand and the TMA gather4 count drop ~3x (measured intake limit: ~45 B/clk/SM, at which
// re-gathering every tap bounds all layers with N <= 64).  A tile whose extras overflow (isolated pixels: > 128 per
// (source, dy)) falls back to one fill per chunk with identity slots - same code, group size 1.
// TMEM map (512 columns): [0,2N) accumulators (half h at h*N), [A_COL0,512) A operand: tf32 form stage s, half h at
// A_COL0 + s*128 + h*64, hi in the first 32 columns, lo in the next 32 (2 stages at N = 128, 3 below); f16 form stage s,
// half h at A_COL0 + s*64 + h*32, h1 in the first 16 columns, h2 in the next 16 (4 stages).
#include <cuda_fp16.h>
#include <cuda.h>   // CUtensorMap + enums only; the encoder is fetched through cudaGetDriverEntryPoint (no -lcuda)

#include "common.cuh"

namespace wmd {

constexpr int TC_BM = 256;                      // rows per CTA tile = 2 UMMA halves of 128
constexpr int TC_BK = 32;                       // floats per chunk = one 128-byte swizzle-atom row
constexpr int TC_THREADS = 512;                 // 16 warps: 8 split + 5 gather + 1 weight loader + 2 issuers; all drain (lane quarter w&3, half (w>>2)&1, cols w>>3)
constexpr int TC_SPLIT_WARPS = 8;               // warps 0-7: warp w owns tile rows (w>>2)*128 + (w&3)*32 + lane (its TMEM lane quarter)
constexpr int TC_GATHER_WARPS = 5;              // warps 8-12
constexpr int TC_WLOAD_WARP = 13;               // warp 13: weight (B) loader - keeps the issuers' loop free of the stage-reuse wait
constexpr int TC_ISSUERS = 2;                   // warps 14-15: one per M half, each the only writer of its accumulator
constexpr int TC_A_STAGES = 3;                  // raw A tiles in shared memory (two gathers in flight + one being split)
constexpr int TC_T_STAGES_MAX = 4;              // split A stages in tensor memory: 2 (N = 128) or 3 (N <= 64), 4 in the f16 form, see TcCfg
constexpr int TC_B_STAGES_MAX = 4;              // [Bhi | Blo] images in shared memory: 3 (N = 128) or 4 (N <= 64)
constexpr int TC_A_TILE = TC_BM * TC_BK * 4;    // 32 KB raw fp32
constexpr int TC_TABLES = 2 * 9 * TC_BM * 4;
constexpr int TC_TMEM_COLS = 512;
// shared-tap gather (SH): 2 raw stages of 256 tile rows + 128 extra rows
constexpr int TC_SH_STAGES = 2;
constexpr int TC_SH_EXTRA = 128;
constexpr int TC_SH_ROWS = TC_BM + TC_SH_EXTRA;
constexpr int TC_SH_TILE = TC_SH_ROWS * 128;     // 48 KB
constexpr int TC_SH_TABLES = 2 * 3 * TC_SH_EXTRA * 4 /* extra source rows */ + 2 * 3 * 2 * TC_BM * 2 /* slots */ + 64 /* counters */;
constexpr uint16_t kZeroSlot = 0xFFFFu;          // slot-table entry of a tap that reads nothing (inactive / padded source)

// Per N-tile configuration.  Accumulators: M half h at TMEM column h*BN; each is written by exactly one issuer, so the
// order of the round-toward-zero accumulations - and with it every output bit - is fixed.
template <int BN, bool SH = false, bool F16 = false>
struct TcCfg {
  static constexpr int B_TILE = BN * TC_BK * 4;            // bytes of one of hi / lo (tf32 form)
  // weight image of one chunk: tf32 form [hi: BN x 128 B | lo: BN x 128 B]; f16 form ONE BN x 128 B tile whose rows hold
  // [h1: 32 channels | h2: 32 channels] as fp16
  static constexpr int B_IMG = F16 ? B_TILE : 2 * B_TILE;
  static constexpr int ACC = BN / 2;                       // accumulator registers per thread: its row x BN/2 columns
  static constexpr int A_BYTES = SH ? TC_SH_STAGES * TC_SH_TILE : TC_A_STAGES * TC_A_TILE;   // 96 KB either way
  // Pipeline depth.  The loop split(c) -> MMA(c) -> [TMEM stage free] -> split(c + T) and the weight prefetch
  // MMA(c-1) done -> load B(c + B - 1) -> MMA(c + B - 1) make the chunk period max(issue, split, (issue + split) / (T-1)...,
  // (issue + L2 latency) / (B - 1)).  At N = 128 the MMA issue (12 x 64 clk) hides both with T = 2 / B = 3 and TMEM / shared
  // memory are full; at N <= 64 the issue is short (12 x ~35 clk per half) and the measured period was twice it
  // (scripts/tc_layer_trace.py: 1715 clk vs 960 of issue), so those tiles take a third A stage (TMEM columns 128..511 are
  // free next to <= 128 accumulator columns) and a fourth weight stage.
  // f16 form: a stage is half as wide (per M half 16 columns of h1 + 16 of h2), so four fit at every N and the split
  // warps never wait for the MMAs of an earlier chunk; its weight images are half as large: four stages as well.
  static constexpr int A_STAGE = F16 ? 64 : 128;                    // TMEM columns of one split A stage (both M halves)
  static constexpr int T_STAGES = F16 ? 4 : (BN <= 64 ? 3 : 2);
  static constexpr int B_STAGES = (F16 || BN <= 64) ? 4 : 3;
  static constexpr uint32_t A_COL0 = 512u - T_STAGES * A_STAGE;     // first TMEM column of the split A operand
  static constexpr size_t SMEM = static_cast<size_t>(A_BYTES) + static_cast<size_t>(B_STAGES) * B_IMG + TC_TABLES +
                                 (SH ? TC_SH_TABLES : 0) + 1024;
  static_assert(2 * BN <= static_cast<int>(A_COL0), "accumulators must leave the A operand's TMEM columns free");
};
#ifndef WMD_TC_EXP
#define WMD_TC_EXP 0                              // timing ablations of scripts/tc_ablate.py (non-zero: results are WRONG)
#endif
constexpr int kFlushChunks = 32;                // epoch length: K = 1024 per TMEM accumulation run
constexpr int32_t kNoRow = -1;                  // tap-table entry of an inactive / padded source: an out-of-bounds TMA row reads zeros


__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
#ifdef WMD_TC_DEBUG
__device__ unsigned int g_dbg[4];
#define MBAR_FAIL(id) do { if (atomicCAS(&g_dbg[0], 0u, (id)) == 0u) { g_dbg[1] = blockIdx.x; g_dbg[2] = threadIdx.x; } return; } while (0)
#define MBAR_SPINS (1u << 21)
#else
#define MBAR_FAIL(id) __trap()
#define MBAR_SPINS (1u << 28)
#endif
// -DWMD_TC_TRACE (scripts/tc_trace.py builds a separate library): CTA 0 records clock64() at fixed points of the
// first kTraceChunks chunks for split warp 0, gather warp 8 and issuer 0.
#ifdef WMD_TC_TRACE
constexpr int kTraceChunks = 256, kTraceSlots = 8;
__device__ long long g_trace[3 * kTraceSlots * kTraceChunks];
#define TC_TRACE(role, slot, c) do { if (blockIdx.x == 0 && lane == 0 && (c) < kTraceChunks) \
    g_trace[((role) * kTraceSlots + (slot)) * kTraceChunks + (c)] = clock64(); } while (0)
// per-tile timeline of CTA 0 (thread 0 = split warp 0): tile top, tables built, first raw A landed, chunk loop done,
// last epoch complete, drained, stored, end-of-tile barrier passed
constexpr int kTraceTiles = 64, kTileSlots = 12;   // slots 8..10: inside the table build (init, tap tables, slot tables)
__device__ long long g_tile_trace[kTraceTiles * kTileSlots];
#define TC_TILE_TRACE(slot) do { if (blockIdx.x == 0 && tid == 0 && tile_iter < kTraceTiles) \
    g_tile_trace[tile_iter * kTileSlots + (slot)] = clock64(); } while (0)
#else
#define TC_TRACE(role, slot, c) do {} while (0)
#define TC_TILE_TRACE(slot) do {} while (0)
#endif
// bounded spin: a protocol bug traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t id = 0) {
  uint32_t done = 0;
  for (uint32_t spin = 0; spin < MBAR_SPINS; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
  }
  MBAR_FAIL(id);
}
// one non-blocking look (per-lane result; the user votes when it consumes it).  Issued a few hundred clocks before the
// answer is needed - the ~200 clk round trip of a barrier query then overlaps other work; a `false` just means the
// blocking wait still has to run
__device__ __forceinline__ uint32_t mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done;
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "version 1"); rows are 128 bytes, 8-row groups
// are 1024 bytes apart (SBO), LBO is the canonical 1 for swizzled K-major operands.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

// D[tmem] (+)= A[tmem] * B[smem]^T : A is 128 lanes x 8 tf32 columns in tensor memory, B a K-major smem tile
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// same with fp16 operands (kind::f16): A is 128 lanes x 16 halves = 8 columns in tensor memory
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// two floats -> packed fp16 pair, round to nearest even, saturating at +-65504 (a stray out-of-range value must not turn
// into inf - inf = NaN in the remainder piece); `lo` lands in bits 0..15 (the lower K index)
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;\n" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float f16_lo_to_f32(uint32_t pair) {
  float f;
  asm("{\n\t.reg .f16 l, h;\n\tmov.b32 {l, h}, %1;\n\tcvt.f32.f16 %0, l;\n\t}\n" : "=f"(f) : "r"(pair));
  return f;
}
__device__ __forceinline__ float f16_hi_to_f32(uint32_t pair) {
  float f;
  asm("{\n\t.reg .f16 l, h;\n\tmov.b32 {l, h}, %1;\n\tcvt.f32.f16 %0, h;\n\t}\n" : "=f"(f) : "r"(pair));
  return f;
}
// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}

__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// this thread's TMEM lane (warp quarter base + lane), 8 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_zero16(uint32_t taddr) {
  const uint32_t z = 0u;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};\n" ::"r"(taddr),
      "r"(z)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  // the load and its wait are ONE asm statement: with two, the compiler may schedule uses of v[] between them (the wait
  // has no register dependence on the load's outputs) and read registers the asynchronous load has not written yet -
  // seen as a timing-dependent wrong accumulator slice on a cold first launch
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}

// Balanced mode plan, shared by the conv kernel and the reduce pass (both derive it from the device-side row count).
// All but the last full round of tiles run data-parallel (whole tiles); the last full round and the partial round
// after it - between 1 and 2 x CTAs - 1 tiles - are cut stream-K style into equal ranges of U units per CTA.  Merging
// the last full round in keeps the ranges long (>= one tile's reduction), so a tile has <= 2 segments; only when
// there is no full round at all (fewer tiles than CTAs) the ranges are shorter: U >= nchunks/6, <= 7 segments.
constexpr int kBalSlabs = 8;                    // workspace slabs: CTAs x kBalSlabs tiles of 256 x N floats
constexpr int kBalCounterBytes = 4096;          // balanced mode: per stream-K tile arrival counters at the head of the workspace
struct BalPlan {
  long long rem_tile0;                          // first stream-K tile
  long long U;                                  // units (chunks) per CTA
  int slabs;                                    // workspace slabs per stream-K tile
};
__host__ __device__ __forceinline__ BalPlan bal_plan(long long tiles, long long grid, int nchunks) {
  BalPlan p;
  const long long rounds = tiles / grid;
  const long long dp_rounds = (tiles % grid == 0) ? rounds : (rounds > 0 ? rounds - 1 : 0);
  p.rem_tile0 = dp_rounds * grid;
  const long long rem_tiles = tiles - p.rem_tile0;
  const long long even = (rem_tiles * nchunks + grid - 1) / grid;
  const long long floor_u = (nchunks + 5) / 6;
  p.U = even > floor_u ? even : floor_u;
  p.slabs = rem_tiles >= grid ? 3 : kBalSlabs;  // rem_tiles * slabs <= grid * kBalSlabs either way (rem_tiles < 2 * grid)
  return p;
}

template <int BN, bool SH, bool F16>
__global__ void __launch_bounds__(TC_THREADS, 1) conv_rows_tc_kernel(const wmd_conv_desc d, const float* __restrict__ wtc,
                                                                     const int splits, float* __restrict__ partial,
                                                                     const __grid_constant__ CUtensorMap tm0,
                                                                     const __grid_constant__ CUtensorMap tm1) {
  using Cfg = TcCfg<BN, SH, F16>;
  constexpr int TC_B_TILE = Cfg::B_TILE;
  constexpr int B_IMG = Cfg::B_IMG;                         // bytes of one chunk's weight image
  constexpr int ACC = Cfg::ACC;
  constexpr int TC_T_STAGES = Cfg::T_STAGES;
  constexpr int TC_B_STAGES = Cfg::B_STAGES;
  extern __shared__ unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t bar_raw_full[TC_A_STAGES];   // raw A tile of the stage has landed (TMA transaction bytes)
  __shared__ __align__(8) uint64_t bar_raw_empty[TC_A_STAGES];  // ... has been read by the 8 split warps
  __shared__ __align__(8) uint64_t bar_asplit[TC_T_STAGES_MAX]; // split A of the TMEM stage is stored (8 split warps)
  __shared__ __align__(8) uint64_t bar_mma[TC_T_STAGES_MAX];    // chunk's MMAs done (2 issuers): TMEM A stage + B stage reusable
  __shared__ __align__(8) uint64_t bar_b[TC_B_STAGES_MAX]; // weight image of the stage has landed (bulk copy)
  __shared__ __align__(8) uint64_t bar_bfree[TC_B_STAGES_MAX];  // chunk's MMAs done (2 issuers): weight stage reusable
  __shared__ __align__(8) uint64_t bar_epoch;              // accumulation epoch complete (4 issuers)
  __shared__ uint32_t tmem_base_slot;
  __shared__ int s_fixup;                                  // balanced mode: segments of the tile to reduce here (0 = not the last)

  // warp index through a shuffle: provably warp-uniform, so the role branches and everything the issuer warps
  // compute from it stay on the uniform datapath (see the issuer section)
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~static_cast<uintptr_t>(1023));
  unsigned char* sA_base = base;
  unsigned char* sB_base = base + Cfg::A_BYTES;
  int32_t* tab0 = reinterpret_cast<int32_t*>(sB_base + TC_B_STAGES * B_IMG);   // [tap][row]: source row in x0, -1 = none
  int32_t* tab1 = tab0 + 9 * TC_BM;                                                    // ... in x1
  // shared-tap gather tables (SH): extra source rows [src][dy][128], slots [src][dy][side][row], counters [src*3+dy], [6] = overflow
  int32_t* xtra = tab1 + 9 * TC_BM;
  uint16_t* slots = reinterpret_cast<uint16_t*>(xtra + 2 * 3 * TC_SH_EXTRA);
  int* nx = reinterpret_cast<int*>(slots + 2 * 3 * 2 * TC_BM);

  if (tid == 0) {
    for (int s = 0; s < TC_A_STAGES; ++s) {
      mbar_init(smem_u32(&bar_raw_full[s]), 1);               // one expect_tx arrival; the gathers complete the bytes
      mbar_init(smem_u32(&bar_raw_empty[s]), TC_SPLIT_WARPS);
    }
    for (int s = 0; s < TC_T_STAGES; ++s) {
      mbar_init(smem_u32(&bar_asplit[s]), TC_SPLIT_WARPS);
      mbar_init(smem_u32(&bar_mma[s]), TC_ISSUERS);
    }
    for (int s = 0; s < TC_B_STAGES; ++s) {
      mbar_init(smem_u32(&bar_b[s]), 1);
      mbar_init(smem_u32(&bar_bfree[s]), TC_ISSUERS);
    }
    mbar_init(smem_u32(&bar_epoch), TC_ISSUERS);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"(static_cast<uint32_t>(TC_TMEM_COLS))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = tmem_base_slot;

  // F16: operands are fed as fp16 pairs.  Activations are scaled by a power of two chosen from the sources' max |x| (device
  // scalars written by their producers: layout moves, earlier convolutions) so that max |x| s lies in (2^13, 2^14] - no
  // overflow, the low piece stays normal for everything within 2^-11 .. 1 of the maximum; weights carry their own
  // power-of-two scale in the packed image's header.  Both scales are undone exactly in the epilogue.
  float ascale = 1.f, out_scale = 1.f;
  if (F16) {
    float amax = d.amax0 ? __ldg(d.amax0) : 0.f;
    if (d.c1 > 0 && d.amax1) amax = fmaxf(amax, __ldg(d.amax1));
    int e = 0;
    if (amax > 0.f && amax < INFINITY) {
      int ex;
      frexpf(amax, &ex);                         // amax = m * 2^ex, m in [0.5, 1)
      e = 14 - ex;                               // amax * 2^e in [2^13, 2^14)
    }
    e = max(-100, min(100, e));
    ascale = ldexpf(1.f, e);
    out_scale = ldexpf(1.f, -e) * __ldg(wtc);    // header word 0: 1 / weight scale
  }
  const long long HW = static_cast<long long>(d.H) * d.W;
  const int total_px = static_cast<int>(static_cast<long long>(d.N) * HW);
  int rows = d.pixels ? *d.count : total_px;
  rows = min(rows, d.max_rows);
  const int nch0 = (d.c0 + TC_BK - 1) / TC_BK, nch1 = (d.c1 + TC_BK - 1) / TC_BK;
  const int per_tap = nch0 + nch1;
  const int nchunks = d.taps * per_tap;
  const int n_tiles = (d.cout + BN - 1) / BN;
  const long long tiles = static_cast<long long>((rows + TC_BM - 1) / TC_BM) * n_tiles;
  const int Hs = d.H >> d.shift0, Ws = d.W >> d.shift0;
  const bool aligned_rows = (d.taps == 1 && d.map0 == nullptr);
  // tm0 then has a 256-row box (launch_tc).  A box load cannot zero gated-off rows, so a gate takes the per-row gathers;
  // source-1 chunks always go through the tap table
  const bool tiled_rows = aligned_rows && d.rows0 > 0 && d.gate == nullptr;
  // instruction descriptor: D=f32, A=B=tf32, both K-major, N = BN, M = 128
  // (F16: A = B = f16, format code 0, K = 16 per instruction)
  constexpr uint32_t kFmt = F16 ? 0u : 2u;
  constexpr uint32_t kIdesc = (1u << 4) | (kFmt << 7) | (kFmt << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                              (static_cast<uint32_t>(128 >> 4) << 24);

  // drain / store ownership (all 16 warps): TMEM lane quarter, M half, column half (ACC = BN/2 columns of every copy)
  const int my_q = warp & 3, my_half = (warp >> 2) & 1, my_ch = warp >> 3;
  const int my_row = my_half * 128 + my_q * 32 + lane;          // row within the CTA tile
  const uint32_t lane_field = static_cast<uint32_t>(my_q * 32) << 16;
  const uint32_t my_acc_addr = tmem_acc + lane_field + static_cast<uint32_t>(my_half * BN + my_ch * ACC);
  uint32_t mma_rounds = 0;                                       // chunks issued so far by this CTA (all tiles)
  uint32_t epochs = 0;                                           // epoch commits so far
  uint32_t fill_rounds = 0;                                      // SH: raw-stage fills so far by this CTA (all tiles)

  // accumulators start (and are left by every drain) at zero: every MMA accumulates
#pragma unroll
  for (int cc = 0; cc < ACC; cc += 16) tmem_zero16(my_acc_addr + static_cast<uint32_t>(cc));
  asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // Work decomposition.  A "unit" is one 32-channel chunk of one output tile.
  //   splits >= 1 : every tile's reduction is cut into `splits` equal ranges (split-K); splits == 1 = whole tiles.
  //   splits == 0 : BALANCED (data-parallel + stream-K, see bal_plan): all but the last full round run whole tiles;
  //                 the units of the remaining tiles are dealt out to all CTAs in equal contiguous ranges of U
  //                 units, so the SMs finish together however many tiles the (device-side) row count yields, and
  //                 only tiles cut by a range boundary pay for partial sums.
  // Segments that do not cover a whole tile write raw partial sums to the workspace; tc_reduce_kernel sums a tile's
  // segments in a fixed order and applies bias + activation, so results stay deterministic.
  const bool balanced = (splits == 0);
  const BalPlan plan = bal_plan(tiles, gridDim.x, nchunks);
  const long long rem_tile0 = balanced ? plan.rem_tile0 : 0;            // first stream-K tile
  const long long rem_units = balanced ? (tiles - rem_tile0) * nchunks : 0;
  const long long U = plan.U;
  long long u = balanced ? static_cast<long long>(blockIdx.x) * U : 0;
  const long long u_end = balanced ? min(rem_units, u + U) : 0;
  long long item = blockIdx.x;
  const long long items = balanced ? rem_tile0 : tiles * splits;
  int tile_iter = -1;
  while (true) {
    ++tile_iter;
    long long tile;
    int cb, ce, slab;
    bool whole;
    long long rem_t = 0;                                                // remainder-tile index (balanced partials)
    if (balanced && item < items) {                                     // data-parallel rounds
      tile = item;
      cb = 0; ce = nchunks; slab = 0; whole = true;
      item += gridDim.x;
    } else if (balanced) {                                              // stream-K over the remainder tiles
      if (u >= u_end) break;
      rem_t = u / nchunks;
      tile = rem_tile0 + rem_t;
      cb = static_cast<int>(u - rem_t * nchunks);
      ce = static_cast<int>(min(static_cast<long long>(nchunks), cb + (u_end - u)));
      slab = static_cast<int>(blockIdx.x - (rem_t * nchunks) / U);
      whole = (cb == 0 && ce == nchunks);
      u += ce - cb;
    } else {
      if (item >= items) break;
      tile = item / splits;
      slab = static_cast<int>(item - tile * splits);
      cb = static_cast<int>(static_cast<long long>(slab) * nchunks / splits);
      ce = static_cast<int>(static_cast<long long>(slab + 1) * nchunks / splits);
      whole = (splits == 1);
      item += gridDim.x;
    }
    const int len = ce - cb;
    const int m0 = static_cast<int>(tile / n_tiles) * TC_BM;
    const int nt = static_cast<int>(tile % n_tiles);
    const int n0 = nt * BN;
    // rows / bias 16-byte aligned: the epilogue's vector form for the quads inside cout
    const bool al_ok = (d.ldy % 4 == 0) && ((reinterpret_cast<uintptr_t>(d.y) & 15) == 0) &&
                       ((reinterpret_cast<uintptr_t>(d.bias) & 15) == 0);
    TC_TILE_TRACE(0);

    if (SH) {                                      // extras default to "no row" (the tail of a 4-row load group), counters to 0
      for (int e = tid; e < 2 * 3 * TC_SH_EXTRA; e += TC_THREADS) xtra[e] = kNoRow;
      if (tid < 8) nx[tid] = 0;
    }
    TC_TILE_TRACE(8);
    // thread t: tile row t % 256, taps [t / 256 * 5, ...): the output pixel is read and decoded once per row, the taps'
    // gate / map lookups are independent loads
    {
      const int r = tid & (TC_BM - 1);
      const int t_lo = (tid >> 8) * 5, t_hi = min(d.taps, t_lo + 5);
      const int m = m0 + r;
      int n = 0, y = 0, x = 0;
      const bool live = m < rows;
      if (live && t_lo < t_hi) {
        const unsigned p = static_cast<unsigned>(d.pixels ? d.pixels[m] : m);     // < 2^31 (checked by the host): 32-bit divisions
        const unsigned hw = static_cast<unsigned>(HW);
        n = static_cast<int>(p / hw);
        const unsigned rem = p - static_cast<unsigned>(n) * hw;
        y = static_cast<int>(rem / static_cast<unsigned>(d.W));
        x = static_cast<int>(rem - static_cast<unsigned>(y) * static_cast<unsigned>(d.W));
      }
      // Two rounds of loads for the thread's (up to) five taps instead of one dependent chain per tap: first every tap's
      // coordinates and its three look-ups (gate byte, source-0 index map, source-1 index map) are issued together - the maps
      // are read whether or not the gate turns out to be set, their indices are valid for every in-range coordinate - then
      // the results are combined.  (One tap at a time cost ~800 clk per tap: 3.3-5.0k clk of a 5-10k clk table build.)
      constexpr int kTapsPerThread = 5;
      int qv[kTapsPerThread];                        // source-1 pixel of the tap, -1 = out of range / dead row
      uint8_t gv[kTapsPerThread];
      int32_t m0v[kTapsPerThread], m1v[kTapsPerThread];
#pragma unroll
      for (int k = 0; k < kTapsPerThread; ++k) {
        const int tap = t_lo + k;
        qv[k] = -1;
        gv[k] = 1;
        m0v[k] = kNoRow;
        m1v[k] = kNoRow;
        if (live && tap < t_hi) {
          int qy = y, qx = x;
          if (d.taps == 9) { qy += tap / 3 - 1; qx += tap % 3 - 1; }
          bool ok = pad_coord(qy, d.H, d.pad_mode);
          ok = pad_coord(qx, d.W, d.pad_mode) && ok;
          if (ok) {
            const int q = (n * d.H + qy) * d.W + qx;
            qv[k] = q;
            if (d.gate) gv[k] = d.gate[q];
            m1v[k] = d.map1 ? d.map1[q] : q;        // -1 (not in the compact skip list) = kNoRow
            if (aligned_rows) {
              m0v[k] = m;
            } else {
              const int qs = (n * Hs + (qy >> d.shift0)) * Ws + (qx >> d.shift0);
              m0v[k] = d.map0 ? d.map0[qs] : qs;
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < kTapsPerThread; ++k) {
        const int tap = t_lo + k;
        if (tap < t_hi) {
          const bool ok = qv[k] >= 0 && gv[k] != 0;
          tab0[tap * TC_BM + r] = (ok && m0v[k] >= 0) ? m0v[k] : kNoRow;
          tab1[tap * TC_BM + r] = ok ? m1v[k] : kNoRow;
        }
      }
    }
    TC_TILE_TRACE(9);
    __syncthreads();
    TC_TILE_TRACE(10);
    // SH: slot tables of the dx = -1 / +1 taps.  Tap (dy, dx) of tile row r reads source row s; if the centre tap of row
    // r + dx reads the same s (the two output pixels are neighbours in the list) the row is already in slot r + dx of the
    // (chunk, dy) stage, otherwise it becomes an extra (slot 256 + k).  Extras past the capacity switch the whole tile to
    // one fill per chunk (group size 1).
    int gsz = 1;
    if (SH) {
      const int nsrc = d.c1 > 0 ? 2 : 1;
      for (int e = tid; e < nsrc * 3 * 2 * TC_BM; e += TC_THREADS) {
        const int r = e % TC_BM;
        int t = e / TC_BM;
        const int side = t & 1; t >>= 1;
        const int dy = t % 3, src = t / 3;
        const int dx = side ? 1 : -1;
        const int32_t* tb = src ? tab1 : tab0;
        const int32_t sidx = tb[(dy * 3 + 1 + dx) * TC_BM + r];
        uint16_t slot = kZeroSlot;
        bool extra = false;
        if (sidx >= 0) {
          const int rn = r + dx;
          if (rn >= 0 && rn < TC_BM && tb[(dy * 3 + 1) * TC_BM + rn] == sidx) {
            slot = static_cast<uint16_t>(rn);
          } else {
            extra = true;
          }
        }
        // a warp's 32 entries share (source, dy, side): ONE shared-memory atomic per warp reserves its extras' slots
        // (run ends are common in sparse tiles; one atomic per entry serialised on six counters)
        const unsigned xm = __ballot_sync(0xffffffffu, extra);
        if (xm) {
          int base_k = 0;
          if (lane == __ffs(xm) - 1) base_k = atomicAdd(&nx[src * 3 + dy], __popc(xm));
          base_k = __shfl_sync(0xffffffffu, base_k, __ffs(xm) - 1);
          if (extra) {
            const int k = base_k + __popc(xm & ((1u << lane) - 1u));
            if (k < TC_SH_EXTRA) {
              xtra[(src * 3 + dy) * TC_SH_EXTRA + k] = sidx;
              slot = static_cast<uint16_t>(TC_BM + k);
            } else {
              nx[6] = 1;
            }
          }
        }
        slots[((src * 3 + dy) * 2 + side) * TC_BM + r] = slot;
      }
      __syncthreads();
      gsz = nx[6] ? 1 : 3;
    }
    // raw-stage fills of this segment: fill index (tile-relative) of chunk c is c / gsz
    const int f0 = cb / gsz;
    const int nfills = (ce - 1) / gsz - f0 + 1;
    const uint32_t fround0 = fill_rounds;
    TC_TILE_TRACE(1);

    const unsigned char* wtile = reinterpret_cast<const unsigned char*>(wtc) +
                                 (F16 ? 128 : 0) + static_cast<long long>(nt) * nchunks * B_IMG;   // f16 images follow a 128-byte header
    const uint32_t round0 = mma_rounds;

    float acc[ACC];
#pragma unroll
    for (int j = 0; j < ACC; ++j) acc[j] = 0.f;
    float out_max = 0.f;                          // max |y| this thread stores in this tile (-> d.amax_out)

    // drains this thread's slice (its row, ACC columns of every issuer's copy) with round-to-nearest adds, re-zeroes it
    auto drain = [&]() {
#pragma unroll
      for (int cc = 0; cc < ACC; cc += 16) {
        uint32_t v[16];
        tmem_ld16(my_acc_addr + static_cast<uint32_t>(cc), v);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[cc + j] += __uint_as_float(v[j]);
        tmem_zero16(my_acc_addr + static_cast<uint32_t>(cc));
      }
      asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
    };

    // epoch boundary (every role, top of chunk c): the accumulation run that ended with chunk c-1 is drained by all
    // 16 warps before any MMA of chunk c is issued
    auto epoch_boundary = [&](int c) {
      if ((c % kFlushChunks) == 0 && c > 0) {
        mbar_wait(smem_u32(&bar_epoch), (epochs - 1) & 1, 0x10000u + round0 + c);
        tc_fence_after();
        drain();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
      }
    };

    // Implicit im2col through the TMA: every `tile::gather4` load fetches the 128-byte channel slice of FOUR arbitrary
    // source rows (row indices from the tap table; -1 and channels past C are zero-filled by the TMA) into 512
    // contiguous, 128B-swizzled bytes of the raw stage and completes on the stage's mbarrier.  A chunk is 64 loads:
    // gather warp g issues groups g, g+5, ...  One load costs the issuing warp ~140 clk here - that is the TMA unit's
    // queue, not the warp.  Everything a load needs except the four row indices is made provably warp-uniform
    // (shuffles), so ptxas keeps it in uniform registers across the unrolled loop; per load that leaves one LDS.128 +
    // four R2URs.
    const uint32_t sA_u = __shfl_sync(0xffffffffu, smem_u32(sA_base), 0);
    const int gw = warp - TC_SPLIT_WARPS;                               // gather warp index (valid for warps 8-12)
    // ---- one-fill-per-chunk form (SH = false): chunk c -> raw stage round % 3, rows = the tap's table
    constexpr int kMaxLoadsPerWarp = (TC_BM / 4 + TC_GATHER_WARPS - 1) / TC_GATHER_WARPS;
    auto gather_chunk = [&](int c, uint32_t round) {
      const uint32_t st = round % TC_A_STAGES;
      if (tiled_rows && c < nch0) {
        // 1x1 stages read tile rows m0 .. m0+255 of x0 as they are: ONE tiled TMA load (box = 256 rows x 32 channels, tm0 is
        // encoded with that box by the host) instead of 64 four-row gathers - 690 vs 974 clk per chunk measured
        // (scripts/bench_cu/tma_tile_rate.cu) and no issue pressure.  Rows past the tensor / channels past C read zeros.
        if (gw == 0 && elect_one()) {
          const uint32_t bar = smem_u32(&bar_raw_full[st]);
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(static_cast<uint32_t>(TC_A_TILE)) : "memory");
          asm volatile(
              "cp.async.bulk.tensor.2d.shared::cta.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
                  sA_u + st * TC_A_TILE),
              "l"(reinterpret_cast<uint64_t>(&tm0)), "r"(c * TC_BK), "r"(m0), "r"(bar)
              : "memory");
        }
        return;
      }
      const int rr = c / d.taps;                  // channel chunk outermost, taps innermost: the nine taps of a
      const int tap = c - rr * d.taps;            // chunk re-read (almost) the same rows while they are hot in L2
      const bool src1 = rr >= nch0;
      const int col = __shfl_sync(0xffffffffu, (src1 ? rr - nch0 : rr) * TC_BK, 0);
      const uint32_t tab_u = __shfl_sync(0xffffffffu, smem_u32((src1 ? tab1 : tab0) + tap * TC_BM + 4 * gw), 0);
      const uint64_t tmp = reinterpret_cast<uint64_t>(src1 ? &tm1 : &tm0);
      const uint64_t tm_u = (static_cast<uint64_t>(__shfl_sync(0xffffffffu, static_cast<uint32_t>(tmp >> 32), 0)) << 32) |
                            __shfl_sync(0xffffffffu, static_cast<uint32_t>(tmp), 0);
      const uint32_t bar = __shfl_sync(0xffffffffu, smem_u32(&bar_raw_full[st]), 0);
      const uint32_t dst_u = __shfl_sync(0xffffffffu, sA_u + st * TC_A_TILE + gw * 512, 0);
      if (gw == 0 && elect_one())
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(static_cast<uint32_t>(TC_A_TILE)) : "memory");
#pragma unroll
      for (int i = 0; i < kMaxLoadsPerWarp; ++i) {
        if (gw + i * TC_GATHER_WARPS < TC_BM / 4) {
          int4 r4;
          asm("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];\n"
              : "=r"(r4.x), "=r"(r4.y), "=r"(r4.z), "=r"(r4.w)
              : "r"(tab_u + static_cast<uint32_t>(i * TC_GATHER_WARPS * 16)));
          if (elect_one())
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];\n" ::"r"(
                    dst_u + static_cast<uint32_t>(i * TC_GATHER_WARPS * 512)),
                "l"(tm_u), "r"(col), "r"(r4.x), "r"(r4.y), "r"(r4.z), "r"(r4.w), "r"(bar)
                : "memory");
        }
      }
    };
    // ---- shared-tap form (SH = true): fill `fr` (tile-relative) = chunks fr*gsz .. of one (channel chunk, dy); slots
    // 0..255 <- the centre tap's table, slots 256.. <- the (source, dy)'s extras; stage = global fill round % 2
    constexpr int kMaxFillLoads = (TC_SH_ROWS / 4 + TC_GATHER_WARPS - 1) / TC_GATHER_WARPS;
    auto issue_fill = [&](int fr, uint32_t fround) {
      const uint32_t st = fround % TC_SH_STAGES;
      const int c = fr * gsz;
      const int rr = c / 9;
      const int tap = c - rr * 9;                 // gsz == 3: the (dy, dx = -1) tap, centre = tap + 1; gsz == 1: the tap itself
      const bool src1 = rr >= nch0;
      const int sd = (src1 ? 3 : 0) + tap / 3;
      const int col = __shfl_sync(0xffffffffu, (src1 ? rr - nch0 : rr) * TC_BK, 0);
      const int ctap = gsz == 3 ? tap + 1 : tap;
      const int ne = gsz == 3 ? min(nx[sd], TC_SH_EXTRA) : 0;
      const int ngroups = __shfl_sync(0xffffffffu, TC_BM / 4 + ((ne + 3) >> 2), 0);
      const uint32_t tab_u = __shfl_sync(0xffffffffu, smem_u32((src1 ? tab1 : tab0) + ctap * TC_BM), 0);
      const uint32_t xtr_u = __shfl_sync(0xffffffffu, smem_u32(xtra + sd * TC_SH_EXTRA) - static_cast<uint32_t>(TC_BM * 4), 0);
      const uint64_t tmp = reinterpret_cast<uint64_t>(src1 ? &tm1 : &tm0);
      const uint64_t tm_u = (static_cast<uint64_t>(__shfl_sync(0xffffffffu, static_cast<uint32_t>(tmp >> 32), 0)) << 32) |
                            __shfl_sync(0xffffffffu, static_cast<uint32_t>(tmp), 0);
      const uint32_t bar = __shfl_sync(0xffffffffu, smem_u32(&bar_raw_full[st]), 0);
      const uint32_t dst_u = __shfl_sync(0xffffffffu, sA_u + st * TC_SH_TILE, 0);
      if (gw == 0 && elect_one())
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(static_cast<uint32_t>(ngroups * 512)) : "memory");
#pragma unroll
      for (int i = 0; i < kMaxFillLoads; ++i) {
        const int g = gw + i * TC_GATHER_WARPS;   // warp-uniform
        if (g < ngroups) {
          int4 r4;
          asm("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];\n"
              : "=r"(r4.x), "=r"(r4.y), "=r"(r4.z), "=r"(r4.w)
              : "r"((g < TC_BM / 4 ? tab_u : xtr_u) + static_cast<uint32_t>(g * 16)));
          if (elect_one())
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];\n" ::"r"(
                    dst_u + static_cast<uint32_t>(g * 512)),
                "l"(tm_u), "r"(col), "r"(r4.x), "r"(r4.y), "r"(r4.z), "r"(r4.w), "r"(bar)
                : "memory");
        }
      }
    };

    if (warp < TC_SPLIT_WARPS) {
      // =================================================================================== split warps
      // raw fp32 row (128 B of the smem stage) -> hi / lo in tensor memory.  Thread = tile row `my_row` = TMEM lane.
      // running position of chunk cb + c: tap, source, place in its fill group, fill round (no divisions in the loop)
      int tapi = cb % 9, rri = cb / 9;
      int gpos = cb % gsz;
      uint32_t fround = fround0;
      uint32_t pre_raw = 0, pre_mma = 0;              // early looks at THIS chunk's barriers, taken during the previous chunk
      for (int c = 0; c < len; ++c) {
        const uint32_t round = round0 + c;
        const uint32_t ts = round % TC_T_STAGES;
        epoch_boundary(c);
        if (warp == 0) TC_TRACE(0, 0, c);
        const unsigned char* rowp;
        uint32_t swz;                                   // row's swizzle key (slot & 7)
        uint32_t release_bar = 0;                       // raw stage to hand back after this chunk (0 = keep)
        bool zero_row = false;
        if (SH) {
          const uint32_t st = fround % TC_SH_STAGES;
          if ((c == 0 || gpos == 0) && !__all_sync(0xffffffffu, pre_raw != 0u)) mbar_wait(smem_u32(&bar_raw_full[st]), (fround / TC_SH_STAGES) & 1, 0x20000u + round);
          int slot = my_row;
          if (gsz == 3 && gpos != 1) slot = slots[(((rri >= nch0 ? 3 : 0) + tapi / 3) * 2 + (gpos >> 1)) * TC_BM + my_row];
          zero_row = slot == kZeroSlot;
          if (zero_row) slot = my_row;
          rowp = sA_base + st * TC_SH_TILE + slot * 128;
          swz = static_cast<uint32_t>(slot & 7);
          if (gpos == gsz - 1 || c == len - 1) release_bar = smem_u32(&bar_raw_empty[st]);
          if (++gpos == gsz) { gpos = 0; ++fround; }
          if (++tapi == 9) { tapi = 0; ++rri; }
        } else {
          const uint32_t rs = round % TC_A_STAGES;
          if (!__all_sync(0xffffffffu, pre_raw != 0u)) mbar_wait(smem_u32(&bar_raw_full[rs]), (round / TC_A_STAGES) & 1, 0x20000u + round);
          rowp = sA_base + rs * TC_A_TILE + my_row * 128;
          swz = static_cast<uint32_t>(my_row & 7);
          release_bar = smem_u32(&bar_raw_empty[rs]);
        }
        if (warp == 0) TC_TRACE(0, 1, c);
        if (c == 0) TC_TILE_TRACE(2);
        // N <= 64: the row's 128 bytes first (the raw stage is ready), then the wait for the TMEM A stage - the
        // shared-memory latency overlaps the barrier's.  N = 128 keeps 64 accumulator registers per thread and has no
        // room for the whole row: it reads 64 bytes at a time after the wait.
        constexpr bool kEarly = BN <= 64;
        uint4 rawv[kEarly ? 8 : 1];
        if (kEarly) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            rawv[kEarly ? q : 0] = *reinterpret_cast<const uint4*>(rowp + ((static_cast<uint32_t>(q) ^ swz) << 4));   // swizzle: conflict-free
            if (SH && zero_row) rawv[kEarly ? q : 0] = make_uint4(0u, 0u, 0u, 0u);
          }
        }
        // TMEM A stage free?  It was read by the MMAs of round - T_STAGES.
        if (round >= TC_T_STAGES && !__all_sync(0xffffffffu, pre_mma != 0u)) mbar_wait(smem_u32(&bar_mma[ts]), ((round - TC_T_STAGES) / TC_T_STAGES) & 1, 0x28000u + round);
        tc_fence_after();
        if (kEarly) {
          // hand the raw stage back only once the row has provably arrived in registers: one dependent use of every
          // loaded word precedes the arrive (a release does not wait for outstanding shared-memory loads by itself)
          uint32_t touch = 0;
#pragma unroll
          for (int q = 0; q < 8; ++q) touch |= rawv[kEarly ? q : 0].x ^ rawv[kEarly ? q : 0].y ^ rawv[kEarly ? q : 0].z ^ rawv[kEarly ? q : 0].w;
          asm volatile("" ::"r"(touch) : "memory");
          __syncwarp();
          if (lane == 0 && release_bar) mbar_arrive(release_bar);       // raw stage may be overwritten
        }
        if (warp == 0) TC_TRACE(0, 2, c);
        const uint32_t ta = tmem_acc + lane_field + Cfg::A_COL0 + ts * Cfg::A_STAGE + static_cast<uint32_t>(my_half * (Cfg::A_STAGE / 2));
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {              // 16 channels at a time
          uint4 v4[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (kEarly) {
              v4[q] = rawv[kEarly ? 4 * hf + q : 0];
            } else if (WMD_TC_EXP == 2 || WMD_TC_EXP == 3) {
              v4[q] = make_uint4(round, swz, ts, 4u * hf + q);   // ablation: no shared-memory row reads
            } else {
              v4[q] = *reinterpret_cast<const uint4*>(rowp + ((static_cast<uint32_t>(4 * hf + q) ^ swz) << 4));
              if (SH && zero_row) v4[q] = make_uint4(0u, 0u, 0u, 0u);
            }
          }
          if (F16) {
            // x * s (s a power of two: exact) = h1 + h2 with h1 = fp16(x s) and h2 = fp16(x s - h1): 22 mantissa bits, the
            // precision of the tf32 hi / lo pair; two halves per 32-bit TMEM column, lower channel in the lower half
            uint32_t h1[8], h2[8];
#if WMD_TC_EXP >= 1 && WMD_TC_EXP <= 3
#pragma unroll
            for (int q = 0; q < 4; ++q) {              // ablation: no conversion arithmetic
              h1[2 * q] = v4[q].x; h1[2 * q + 1] = v4[q].y; h2[2 * q] = v4[q].z; h2[2 * q + 1] = v4[q].w;
            }
#else
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float b0 = __uint_as_float(v4[q].x) * ascale, b1 = __uint_as_float(v4[q].y) * ascale;
              const float b2 = __uint_as_float(v4[q].z) * ascale, b3 = __uint_as_float(v4[q].w) * ascale;
              const uint32_t p0 = pack_f16x2(b0, b1), p1 = pack_f16x2(b2, b3);
              h1[2 * q] = p0;
              h1[2 * q + 1] = p1;
              h2[2 * q] = pack_f16x2(b0 - f16_lo_to_f32(p0), b1 - f16_hi_to_f32(p0));
              h2[2 * q + 1] = pack_f16x2(b2 - f16_lo_to_f32(p1), b3 - f16_hi_to_f32(p1));
            }
#endif
            tmem_st8(ta + static_cast<uint32_t>(8 * hf), h1);
            tmem_st8(ta + 16u + static_cast<uint32_t>(8 * hf), h2);
          } else {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const uint32_t raw[4] = {v4[q].x, v4[q].y, v4[q].z, v4[q].w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                hi[4 * q + e] = raw[e] & 0xFFFFE000u;                                                    // tf32 by truncation
                lo[4 * q + e] = __float_as_uint(__uint_as_float(raw[e]) - __uint_as_float(hi[4 * q + e]));   // exact remainder
              }
            }
            tmem_st16(ta + static_cast<uint32_t>(16 * hf), hi);
            tmem_st16(ta + 32u + static_cast<uint32_t>(16 * hf), lo);
          }
        }
        if (!kEarly) {
          __syncwarp();
          if (lane == 0 && release_bar) mbar_arrive(release_bar);       // raw stage may be overwritten
        }
        if (warp == 0) TC_TRACE(0, 3, c);
        // early look at the next chunk's barriers: the queries' latency overlaps the tcgen05.st drain below
        pre_raw = pre_mma = 0;
        if (c + 1 < len) {
          const uint32_t nr = round + 1;
          if (nr >= TC_T_STAGES) pre_mma = mbar_test(smem_u32(&bar_mma[nr % TC_T_STAGES]), ((nr - TC_T_STAGES) / TC_T_STAGES) & 1);
          if (SH) {                                   // gpos / fround already describe chunk c + 1
            if (gpos == 0) pre_raw = mbar_test(smem_u32(&bar_raw_full[fround % TC_SH_STAGES]), (fround / TC_SH_STAGES) & 1);
          } else {
            pre_raw = mbar_test(smem_u32(&bar_raw_full[nr % TC_A_STAGES]), (nr / TC_A_STAGES) & 1);
          }
        }
        if (WMD_TC_EXP != 3) asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bar_asplit[ts]));
        if (warp == 0) TC_TRACE(0, 4, c);
        if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) epochs += 1;
      }
    } else if (warp < TC_SPLIT_WARPS + TC_GATHER_WARPS) {
      // =================================================================================== gather warps
      // the raw stages are free at the start of a tile (every split of the previous tile has completed)
      if (SH) {
        issue_fill(f0, fround0);
        if (nfills > 1) issue_fill(f0 + 1, fround0 + 1);
        int gpos = cb % gsz, j = 0;                      // chunk's place in its fill group, fill index within the segment
        for (int c = 0; c < len; ++c) {
          epoch_boundary(c);
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 0, c);
          // at the first chunk of fill j >= 1 the stage of fill j - 1 is about to be released: refill it with fill j + 1
          if (gpos == 0 && j >= 1 && j + 1 < nfills) {
            const uint32_t fr2 = fround0 + static_cast<uint32_t>(j + 1);
            mbar_wait(smem_u32(&bar_raw_empty[fr2 % TC_SH_STAGES]), ((fr2 / TC_SH_STAGES) - 1) & 1, 0x30000u + fr2);
            if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 1, c);
            issue_fill(f0 + j + 1, fr2);
          }
          if (++gpos == gsz) { gpos = 0; ++j; }
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 2, c);
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 3, c);
          if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) epochs += 1;
        }
      } else {
        gather_chunk(cb, round0);
        if (len > 1) gather_chunk(cb + 1, round0 + 1);
        for (int c = 0; c < len; ++c) {
          const uint32_t round = round0 + c;
          epoch_boundary(c);
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 0, c);
          if (c + 2 < len) {
            const uint32_t r2 = round + 2, st2 = r2 % TC_A_STAGES;
            // stage st2 was last filled for round r2-3: wait until the split warps have read it
            if (c + 2 >= TC_A_STAGES) mbar_wait(smem_u32(&bar_raw_empty[st2]), ((r2 - TC_A_STAGES) / TC_A_STAGES) & 1, 0x30000u + round);
            if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 1, c);
            gather_chunk(cb + c + 2, r2);
          }
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 2, c);
          if (warp == TC_SPLIT_WARPS) TC_TRACE(1, 3, c);
          if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) epochs += 1;
        }
      }
    } else if (warp == TC_WLOAD_WARP) {
      // =================================================================================== weight loader
      // One [hi | lo] image per chunk, B_STAGES - 1 chunks ahead of the MMAs, a single cp.async.bulk each.  The stage
      // of chunk c + B - 1 is the one chunk c - 1 used: it is free when both issuers' MMAs of chunk c - 1 have
      // completed (bar_bfree, committed by the issuers: its next completion after chunk c - 1 is chunk c - 1 + B, which
      // needs the very load issued here - no phase can be skipped).  A warp of its own, so that this wait is not in
      // the issuers' loop.
      const uint32_t sB_u = __shfl_sync(0xffffffffu, smem_u32(sB_base), 0);
      if (elect_one()) {
        const unsigned char* w0 = wtile + static_cast<long long>(cb) * B_IMG;
        // the first B_STAGES - 1 weight images (their stages are free: every MMA of the previous tile has completed)
        for (int k = 0; k < TC_B_STAGES - 1 && k < len; ++k)
          bulk_g2s(sB_u + ((round0 + k) % TC_B_STAGES) * B_IMG, w0 + static_cast<long long>(k) * B_IMG, B_IMG,
                   smem_u32(&bar_b[(round0 + k) % TC_B_STAGES]));
      }
      __syncwarp();
      for (int c = 0; c < len; ++c) {
        const uint32_t round = round0 + c;
        epoch_boundary(c);
        if (c + TC_B_STAGES - 1 < len) {
          // c == 0: the stage belonged to the previous tile's last chunk - free since the tile's closing barrier
          if (c >= 1) mbar_wait(smem_u32(&bar_bfree[(round - 1) % TC_B_STAGES]), ((round - 1) / TC_B_STAGES) & 1, 0x50000u + round);
          if (elect_one()) {
            const uint32_t ns = (round + TC_B_STAGES - 1) % TC_B_STAGES;
            bulk_g2s(sB_u + ns * B_IMG, wtile + static_cast<long long>(cb + c + TC_B_STAGES - 1) * B_IMG, B_IMG,
                     smem_u32(&bar_b[ns]));
          }
          __syncwarp();
        }
        if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) epochs += 1;
      }
    } else {
      // =================================================================================== issuers
      // The whole warp runs the loop and one elected lane issues.  Written this way (warp-uniform control flow,
      // operands derived from warp-uniform values) ptxas keeps the MMA operands in uniform registers and emits the
      // UTCHMMAs back to back: ~78 clk per instruction.  A `lane == 0` branch instead makes it wrap every MMA in an
      // ELECT / R2UR.BROADCAST / BRA.U.ANY loop: ~210 clk (scripts/bench_cu/mma_rate*.cu).
      const int ih = warp - (TC_WLOAD_WARP + 1);                    // this issuer's M half = its accumulator
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_acc, 0);
      const uint32_t sB_u = __shfl_sync(0xffffffffu, smem_u32(sB_base), 0);
      const uint32_t dh = tmem_u + static_cast<uint32_t>(ih * BN);
      for (int c = 0; c < len; ++c) {
        const uint32_t round = round0 + c;
        const uint32_t ts = round % TC_T_STAGES;
        const uint32_t bs = round % TC_B_STAGES;
        epoch_boundary(c);
        if (ih == 0) TC_TRACE(2, 0, c);
        mbar_wait(smem_u32(&bar_b[bs]), (round / TC_B_STAGES) & 1, 0x48000u + round);        // weight image has landed (long ago)
        if (ih == 0) TC_TRACE(2, 1, c);
        mbar_wait(smem_u32(&bar_asplit[ts]), (round / TC_T_STAGES) & 1, 0x40000u + round);   // split A of this chunk is in TMEM
        if (ih == 0) TC_TRACE(2, 2, c);
        tc_fence_after();
        const uint64_t b0 = umma_desc_sw128(sB_u + bs * B_IMG);
        const uint32_t ah = tmem_u + Cfg::A_COL0 + ts * Cfg::A_STAGE + static_cast<uint32_t>(ih * (Cfg::A_STAGE / 2));
        if (elect_one()) {
          if (F16) {
            // rows of the weight tile: [h1: 64 B | h2: 64 B]; a k-step is 16 channels = 32 B; A: h1 columns 0..15, h2 16..31
#pragma unroll
            for (int ks = 0; ks < TC_BK / 16; ++ks) {
              const uint64_t bh = b0 + static_cast<uint64_t>(2 * ks);
              const uint64_t bl = bh + 4u;
              const uint32_t a = ah + static_cast<uint32_t>(8 * ks);
              umma_f16_ts(dh, a + 16u, bh, kIdesc, 1u);    // lo*hi
              umma_f16_ts(dh, a, bl, kIdesc, 1u);          // hi*lo
              umma_f16_ts(dh, a, bh, kIdesc, 1u);          // hi*hi
            }
          } else {
#pragma unroll
            for (int ks = 0; ks < TC_BK / 8; ++ks) {
              const uint64_t bh = b0 + static_cast<uint64_t>(2 * ks);
              const uint64_t bl = bh + static_cast<uint64_t>(TC_B_TILE >> 4);
              const uint32_t a = ah + static_cast<uint32_t>(8 * ks);
              umma_tf32_ts(dh, a + 32u, bh, kIdesc, 1u);     // lo*hi
              umma_tf32_ts(dh, a, bl, kIdesc, 1u);           // hi*lo
              umma_tf32_ts(dh, a, bh, kIdesc, 1u);           // hi*hi
            }
          }
          umma_commit(smem_u32(&bar_mma[ts]));             // TMEM A stage reusable
          umma_commit(smem_u32(&bar_bfree[bs]));           // weight stage reusable
          if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) umma_commit(smem_u32(&bar_epoch));
        }
        __syncwarp();
        if (ih == 0) TC_TRACE(2, 3, c);
        if (((c + 1) % kFlushChunks == 0) || (c == len - 1)) epochs += 1;
      }
    }
    mma_rounds = round0 + static_cast<uint32_t>(len);
    fill_rounds = fround0 + static_cast<uint32_t>(nfills);
    TC_TILE_TRACE(3);

    // ---- last epoch + epilogue (all 16 warps): bias, activation, one contiguous 256-byte store per thread
    {
      mbar_wait(smem_u32(&bar_epoch), (epochs - 1) & 1, 0x60000u + mma_rounds);
      tc_fence_after();
      TC_TILE_TRACE(4);
      drain();
      TC_TILE_TRACE(5);
      const int m = m0 + my_row;
      if (m < rows && !whole) {
        // raw partial sums of this segment (bias / activation are applied by the reduce pass)
        if (balanced) {                                // compact workspace: [remainder tile][slab][256 rows][BN]
          float* pr = partial + kBalCounterBytes / 4 + ((rem_t * plan.slabs + slab) * TC_BM + my_row) * BN + my_ch * ACC;
#pragma unroll
          for (int j = 0; j < ACC; j += 4) __stcg(reinterpret_cast<float4*>(pr + j), make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]));
        } else {                                       // split-K: [slab][max_rows][ldy]
          float* pr = partial + kBalCounterBytes / 4 + (static_cast<long long>(slab) * d.max_rows + m) * d.ldy;
#pragma unroll
          for (int j = 0; j < ACC; j += 4) {
            const int co = n0 + my_ch * ACC + j;     // ldy % 4 == 0: a quad that starts below cout stays inside the row
            if (co < d.cout) *reinterpret_cast<float4*>(pr + co) = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
          }
        }
      } else if (m < rows) {
        float* yr = d.y + static_cast<long long>(m) * d.ldy;
        // The epilogue is instruction bound (64 outputs per thread at N = 128): the activation is picked once per tile, not
        // per element (act is a kernel argument), quads that lie inside cout take vector bias loads and no per-element
        // bounds; only a quad that straddles cout goes element by element.
        const float ap = d.act_param;
        auto store_all = [&](auto actf) {
#pragma unroll
          for (int j = 0; j < ACC; j += 4) {
            const int co = n0 + my_ch * ACC + j;
            if (al_ok && co + 3 < d.cout) {
              const float4 bq = d.bias ? __ldg(reinterpret_cast<const float4*>(d.bias + co)) : make_float4(0.f, 0.f, 0.f, 0.f);
              float4 o;
              if (F16) {                               // out_scale is a power of two: the product is exact
                o.x = fmaf(acc[j], out_scale, bq.x); o.y = fmaf(acc[j + 1], out_scale, bq.y);
                o.z = fmaf(acc[j + 2], out_scale, bq.z); o.w = fmaf(acc[j + 3], out_scale, bq.w);
              } else {
                o.x = acc[j] + bq.x; o.y = acc[j + 1] + bq.y; o.z = acc[j + 2] + bq.z; o.w = acc[j + 3] + bq.w;
              }
              o.x = actf(o.x); o.y = actf(o.y); o.z = actf(o.z); o.w = actf(o.w);
              out_max = fmaxf(fmaxf(out_max, fabsf(o.x)), fmaxf(fabsf(o.y), fmaxf(fabsf(o.z), fabsf(o.w))));
#if WMD_TC_EXP == 5                               // ablation: same stores, but into a 2 MB window that stays in L2
              *reinterpret_cast<float4*>(d.y + ((static_cast<long long>(m) * d.ldy + co) & 0x7FFFCll)) = o;
#elif WMD_TC_EXP == 6                             // ablation: no store at all (the arithmetic survives through out_max)
              if (o.x == 123456.f) *reinterpret_cast<float4*>(yr + co) = o;
#else
              *reinterpret_cast<float4*>(yr + co) = o;
#endif
            } else if (co < d.cout) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (co + e < d.cout) {
                  const float a = F16 ? __fmul_rn(acc[j + e], out_scale) : acc[j + e];
                  const float o = actf(a + (d.bias ? __ldg(d.bias + co + e) : 0.f));
                  out_max = fmaxf(out_max, fabsf(o));
                  yr[co + e] = o;
                }
              }
            }
          }
        };
        if (d.act == WMD_ACT_ELU) store_all([](float v) { return v > 0.f ? v : expm1_nonpos(v); });
        else if (d.act == WMD_ACT_LRELU) store_all([ap](float v) { return v > 0.f ? v : v * ap; });
        else if (d.act == WMD_ACT_NONE) store_all([](float v) { return v; });
        else store_all([&](float v) { return activate(v, d.act, ap); });
      }
    }
    // ---- balanced mode, stream-K fix-up: the LAST segment of a cut tile to arrive (arrival counter per tile, left at zero
    // for the next launch) sums all segments in slab order - bias first, the order of every earlier version - applies the
    // activation and writes the rows.  No CTA waits for another one and the result does not depend on who is last.
    if (balanced && !whole) {
      __threadfence();
      __syncthreads();
      if (tid == 0) {
        const long long first = (rem_t * nchunks) / U, last = ((rem_t + 1) * nchunks - 1) / U;
        const int nseg = static_cast<int>(last - first + 1);
        unsigned* cnt = reinterpret_cast<unsigned*>(partial) + rem_t;
        const unsigned t = atomicAdd(cnt, 1u);
        s_fixup = (t == static_cast<unsigned>(nseg - 1)) ? nseg : 0;
        if (s_fixup) *cnt = 0u;
      }
      __syncthreads();
      const int nseg = s_fixup;
      if (nseg > 0) {
        __threadfence();
        // Cooperative and coalesced: the slabs are row-major [256][BN], so consecutive threads take consecutive float4s
        // (a warp reads 512 contiguous bytes per slab and writes 512 contiguous bytes of one output row); four quads per
        // thread are in flight, i.e. 4 x nseg independent L2 loads instead of one dependent load per quad.
        // tf32 form: bias first, then the slabs in slab order (the order of every earlier version); f16: slabs, scale, bias.
        const float* pb = partial + kBalCounterBytes / 4 + rem_t * plan.slabs * TC_BM * BN;
        constexpr int kQuadsPerRow = BN / 4;
        constexpr int kQuads = TC_BM * kQuadsPerRow;
        constexpr int kUnroll = 4;
        static_assert(kQuads % (TC_THREADS * kUnroll) == 0, "quads of a tile divide evenly");
        const int tile_rows = min(TC_BM, rows - m0);
        const float ap = d.act_param;
        for (int base = tid; base < kQuads; base += TC_THREADS * kUnroll) {
          float4 v[kUnroll], bq[kUnroll];
          int r[kUnroll], co[kUnroll];
          bool live[kUnroll];
#pragma unroll
          for (int q = 0; q < kUnroll; ++q) {
            const int idx = base + q * TC_THREADS;
            r[q] = idx / kQuadsPerRow;
            co[q] = n0 + 4 * (idx % kQuadsPerRow);
            live[q] = r[q] < tile_rows && co[q] < d.cout;
            bq[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (live[q] && d.bias) {
              if (al_ok && co[q] + 3 < d.cout) {
                bq[q] = __ldg(reinterpret_cast<const float4*>(d.bias + co[q]));
              } else {
                bq[q].x = __ldg(d.bias + co[q]);
                if (co[q] + 1 < d.cout) bq[q].y = __ldg(d.bias + co[q] + 1);
                if (co[q] + 2 < d.cout) bq[q].z = __ldg(d.bias + co[q] + 2);
                if (co[q] + 3 < d.cout) bq[q].w = __ldg(d.bias + co[q] + 3);
              }
            }
            v[q] = F16 ? make_float4(0.f, 0.f, 0.f, 0.f) : bq[q];
          }
          for (int sidx = 0; sidx < nseg; ++sidx) {
            const float4* ps = reinterpret_cast<const float4*>(pb + static_cast<long long>(sidx) * TC_BM * BN) + base;
#pragma unroll
            for (int q = 0; q < kUnroll; ++q) {
              if (live[q]) {
                const float4 pq = __ldcg(ps + q * TC_THREADS);
                v[q].x += pq.x; v[q].y += pq.y; v[q].z += pq.z; v[q].w += pq.w;
              }
            }
          }
#pragma unroll
          for (int q = 0; q < kUnroll; ++q) {
            if (live[q]) {
              float4 o = v[q];
              if (F16) {
                o.x = __fadd_rn(__fmul_rn(o.x, out_scale), bq[q].x); o.y = __fadd_rn(__fmul_rn(o.y, out_scale), bq[q].y);
                o.z = __fadd_rn(__fmul_rn(o.z, out_scale), bq[q].z); o.w = __fadd_rn(__fmul_rn(o.w, out_scale), bq[q].w);
              }
              o.x = activate(o.x, d.act, ap); o.y = activate(o.y, d.act, ap);
              o.z = activate(o.z, d.act, ap); o.w = activate(o.w, d.act, ap);
              float* yq = d.y + static_cast<long long>(m0 + r[q]) * d.ldy + co[q];
              out_max = fmaxf(out_max, fabsf(o.x));
              if (co[q] + 3 < d.cout) {                // balanced mode requires ldy % 4 == 0 and a 16-byte aligned y
                out_max = fmaxf(fmaxf(out_max, fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w)));
                *reinterpret_cast<float4*>(yq) = o;
              } else {
                yq[0] = o.x;
                if (co[q] + 1 < d.cout) { yq[1] = o.y; out_max = fmaxf(out_max, fabsf(o.y)); }
                if (co[q] + 2 < d.cout) { yq[2] = o.z; out_max = fmaxf(out_max, fabsf(o.z)); }
              }
            }
          }
        }
      }
    }
    if (d.amax_out) {                              // max |y| of the layer for its consumers' operand scaling (order independent)
      for (int o = 16; o > 0; o >>= 1) out_max = fmaxf(out_max, __shfl_xor_sync(0xffffffffu, out_max, o));
      if (lane == 0 && out_max > __ldcg(d.amax_out)) atomicMax(reinterpret_cast<unsigned*>(d.amax_out), __float_as_uint(out_max));   // most warps skip the atomic
    }
    TC_TILE_TRACE(6);
    tc_fence_before();
    __syncthreads();   // accumulators drained + re-zeroed by every warp, tap tables free
    tc_fence_after();
    TC_TILE_TRACE(7);
  }

  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_acc),
                 "r"(static_cast<uint32_t>(TC_TMEM_COLS))
                 : "memory");
  }
}

// w (Cout, Cin, taps) fp32 -> per (n-tile, chunk) smem image [tf32 hi: BN x 32 | tf32 lo: BN x 32], K-major,
// 128B-swizzled.  Chunk order = the kernel's: source-0 channel chunks then source-1 chunks, the taps of a chunk innermost.
__global__ void pack_weight_tc_kernel(const float* __restrict__ w, float* __restrict__ out, int Cout, int c0, int c1,
                                      int taps, int BN, long long total) {
  const int nch0 = (c0 + TC_BK - 1) / TC_BK, nch1 = (c1 + TC_BK - 1) / TC_BK;
  const int per_tap = nch0 + nch1;
  const int nchunks = taps * per_tap;
  const int Cin = c0 + c1;
  const long long tile_floats = static_cast<long long>(BN) * TC_BK;
  const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += step) {
    // i indexes LOGICAL (nt, chunk, hilo, n, kk); the store address applies the swizzle
    long long t = i;
    const int kk = static_cast<int>(t % TC_BK); t /= TC_BK;
    const int n = static_cast<int>(t % BN); t /= BN;
    const int hilo = static_cast<int>(t % 2); t /= 2;
    const int c = static_cast<int>(t % nchunks);
    const int nt = static_cast<int>(t / nchunks);
    const int rr = c / taps;
    const int tap = c - rr * taps;
    const bool src1 = rr >= nch0;
    const int ci_local = (src1 ? rr - nch0 : rr) * TC_BK + kk;
    const int csrc = src1 ? c1 : c0;
    const int co = nt * BN + n;
    float v = 0.f;
    if (ci_local < csrc && co < Cout) {
      const int ci = (src1 ? c0 : 0) + ci_local;
      v = __ldg(w + (static_cast<long long>(co) * Cin + ci) * taps + tap);
    }
    const float hi = tf32_rna(v);
    const float val = hilo == 0 ? hi : tf32_rna(v - hi);
    const long long tile_base = ((static_cast<long long>(nt) * nchunks + c) * 2 + hilo) * tile_floats;
    const int piece = kk >> 2, within = kk & 3;
    out[tile_base + static_cast<long long>(n) * TC_BK + ((piece ^ (n & 7)) << 2) + within] = val;
  }
}

// y[m, co] = act(bias[co] + sum_s partial_s[m][co]) in a fixed order (deterministic).  splits >= 2: every tile has
// `splits` slabs laid out [slab][max_rows][ldy].  splits == 0 (balanced): only the remainder tiles have partial sums,
// laid out [remainder tile][slab][256][BN]; the number of segments of a tile follows from the same unit arithmetic the
// conv kernel used (grid = its CTA count); a remainder tile that one CTA covered entirely was finished there.
__global__ void tc_reduce_kernel(const float* __restrict__ partial, int splits, int grid, int BN, int nchunks,
                                 const float* __restrict__ bias, float* __restrict__ y, int ldy, int cout,
                                 const int32_t* __restrict__ count, int max_rows, int act, float act_param) {
  partial += kBalCounterBytes / 4;                   // the workspace starts with the balanced mode's arrival counters (kept zero)
  const int rows = count ? min(*count, max_rows) : max_rows;
  const long long slab_sz = static_cast<long long>(max_rows) * ldy;
  const int n_tiles = (cout + BN - 1) / BN;
  const long long tiles = static_cast<long long>((rows + TC_BM - 1) / TC_BM) * n_tiles;
  const BalPlan plan = bal_plan(tiles, grid, nchunks);
  const long long rem_tile0 = splits == 0 ? plan.rem_tile0 : 0;
  const long long U = plan.U;
  const int quads = BN >> 2;                         // float4 columns of a tile (ldy is a multiple of 4)
  // one CTA per tile per round: the slab arithmetic is per tile, the element loop has no divisions by run-time values
  for (long long tile = rem_tile0 + blockIdx.x; tile < tiles; tile += gridDim.x) {
    int nslabs = splits;
    const long long rem_t = tile - rem_tile0;
    if (splits == 0) {
      const long long first = (rem_t * nchunks) / U, last = ((rem_t + 1) * nchunks - 1) / U;
      if (first == last) continue;                   // whole tile: already written with bias + activation
      nslabs = static_cast<int>(last - first + 1);
    }
    const int m0 = static_cast<int>(tile / n_tiles) * TC_BM;
    const int co0 = static_cast<int>(tile % n_tiles) * BN;
    const int mrows = min(TC_BM, rows - m0);
    const float* pbal = partial + rem_t * plan.slabs * TC_BM * BN;
    for (int e = threadIdx.x; e < mrows * quads; e += blockDim.x) {
      const int r = e / quads, q = e - r * quads;
      const int co = co0 + (q << 2);
      if (co >= cout) continue;
      const long long o = static_cast<long long>(m0 + r) * ldy + co;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bias) {
        v.x = __ldg(bias + co);
        if (co + 1 < cout) v.y = __ldg(bias + co + 1);
        if (co + 2 < cout) v.z = __ldg(bias + co + 2);
        if (co + 3 < cout) v.w = __ldg(bias + co + 3);
      }
      for (int sidx = 0; sidx < nslabs; ++sidx) {
        const float4 p = splits == 0 ? __ldg(reinterpret_cast<const float4*>(pbal + (static_cast<long long>(sidx) * TC_BM + r) * BN + (q << 2)))
                                     : __ldg(reinterpret_cast<const float4*>(partial + sidx * slab_sz + o));
        v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
      }
      v.x = activate(v.x, act, act_param); v.y = activate(v.y, act, act_param);
      v.z = activate(v.z, act, act_param); v.w = activate(v.w, act, act_param);
      if (co + 3 < cout) {
        *reinterpret_cast<float4*>(y + o) = v;
      } else {
        y[o] = v.x;
        if (co + 1 < cout) y[o + 1] = v.y;
        if (co + 2 < cout) y[o + 2] = v.z;
      }
    }
  }
}

// ---- fp16 weight images (precision = WMD_PREC_F16X3) -----------------------------------------------------------------
__global__ void absmax_kernel(const float* __restrict__ x, long long count, float* __restrict__ out) {
  float m = 0.f;
  const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < count; i += step) m = fmaxf(m, fabsf(__ldg(x + i)));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > __ldcg(out)) atomicMax(reinterpret_cast<unsigned*>(out), __float_as_uint(m));
}

// header word 0 holds max |w| when this runs; it is replaced by 1 / s_w by the last block... no: by a second tiny kernel
// (finish_header) so that every pack thread reads the same maximum.
__global__ void pack_weight_tc16_kernel(const float* __restrict__ w, unsigned char* __restrict__ out, int Cout, int c0, int c1,
                                        int taps, int BN, long long total) {
  const float wmax = *reinterpret_cast<const float*>(out);        // header word 0: max |w| (absmax_kernel)
  int e = 0;
  if (wmax > 0.f && wmax < INFINITY) {
    int ex;
    frexpf(wmax, &ex);
    e = 14 - ex;
  }
  e = max(-100, min(100, e));
  const float sw = ldexpf(1.f, e);
  const int nch0 = (c0 + TC_BK - 1) / TC_BK, nch1 = (c1 + TC_BK - 1) / TC_BK;
  const int per_tap = nch0 + nch1;
  const int nchunks = taps * per_tap;
  const int Cin = c0 + c1;
  __half* img = reinterpret_cast<__half*>(out + 128);
  const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += step) {
    // i indexes LOGICAL (nt, chunk, n, kk); the row of a tile is 64 halves: [h1: kk 0..31 | h2: kk 0..31], 128B-swizzled
    long long t = i;
    const int kk = static_cast<int>(t % TC_BK); t /= TC_BK;
    const int n = static_cast<int>(t % BN); t /= BN;
    const int c = static_cast<int>(t % nchunks);
    const int nt = static_cast<int>(t / nchunks);
    const int rr = c / taps;
    const int tap = c - rr * taps;
    const bool src1 = rr >= nch0;
    const int ci_local = (src1 ? rr - nch0 : rr) * TC_BK + kk;
    const int csrc = src1 ? c1 : c0;
    const int co = nt * BN + n;
    float v = 0.f;
    if (ci_local < csrc && co < Cout) {
      const int ci = (src1 ? c0 : 0) + ci_local;
      v = __ldg(w + (static_cast<long long>(co) * Cin + ci) * taps + tap) * sw;
    }
    const __half h1 = __float2half_rn(v);
    const __half h2 = __float2half_rn(v - __half2float(h1));
    const long long tile_base = (static_cast<long long>(nt) * nchunks + c) * (static_cast<long long>(BN) * 64);
    // halves kk (h1) and 32 + kk (h2) of row n; 16-byte pieces (8 halves) are XOR-swizzled with the row index
    const int p1 = kk >> 3, p2 = (32 + kk) >> 3, within = kk & 7;
    img[tile_base + static_cast<long long>(n) * 64 + ((p1 ^ (n & 7)) << 3) + within] = h1;
    img[tile_base + static_cast<long long>(n) * 64 + ((p2 ^ (n & 7)) << 3) + within] = h2;
  }
}
__global__ void finish_header_tc16_kernel(unsigned char* out) {
  float* h = reinterpret_cast<float*>(out);
  const float wmax = h[0];
  int e = 0;
  if (wmax > 0.f && wmax < INFINITY) {
    int ex;
    frexpf(wmax, &ex);
    e = 14 - ex;
  }
  e = max(-100, min(100, e));
  h[1] = wmax;
  h[0] = ldexpf(1.f, -e);                          // 1 / s_w: what the conv kernel reads
}

static int tc_tile_n(int cout) { return cout >= 96 ? 128 : (cout >= 48 ? 64 : 32); }

// TMA descriptor of a source: 2-D fp32 tensor [rows][C] with row pitch ld floats, box = one row x 32 channels,
// 128-byte swizzle, zero fill outside (inactive taps are row -1; a channel tail reads zeros)
typedef CUresult (*TmEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int make_rows_map(CUtensorMap* tm, const float* x, int C, long long rows, int ld, int box_rows = 1) {
  static TmEncodeFn encode = nullptr;
  if (!encode) {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) return WMD_ERR_UNSUPPORTED;
    encode = reinterpret_cast<TmEncodeFn>(fn);
  }
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(rows < 1 ? 1 : rows)};
  const cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * 4};
  const cuuint32_t box[2] = {TC_BK, static_cast<cuuint32_t>(box_rows)}, estr[2] = {1, 1};
  const CUresult rc = encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x), gdim, gstr, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS ? WMD_OK : WMD_ERR_UNSUPPORTED;
}

static int g_reserved_sms = 0;     // SMs the persistent grid leaves free (for a collective's kernel on multi-GPU runs)
static int g_shared_taps = 1;      // 3x3 layers: one raw-stage fill per (chunk, dy) shared by the three dx taps (tuning / A-B knob)

template <int BN, bool SH, bool F16>
static int launch_tc(const wmd_conv_desc& d, int splits, float* partial, cudaStream_t stream) {
  using Cfg = TcCfg<BN, SH, F16>;
  CUtensorMap tm0, tm1;
  {
    const long long px = static_cast<long long>(d.N) * d.H * d.W;
    const long long rows0 = static_cast<long long>(d.N) * (d.H >> d.shift0) * (d.W >> d.shift0);
    // 1x1 stage over its own rows (taps == 1, no index map, no gate): the kernel loads whole 256-row tiles of source 0
    const bool tiled = (d.taps == 1 && d.map0 == nullptr && d.rows0 > 0 && d.gate == nullptr);
    int rc = make_rows_map(&tm0, d.x0, d.c0, tiled ? d.rows0 : rows0, d.ld0, tiled ? TC_BM : 1);
    if (rc != WMD_OK) return rc;
    if (d.c1 > 0) {
      rc = make_rows_map(&tm1, d.x1, d.c1, px, d.ld1);
      if (rc != WMD_OK) return rc;
    } else {
      tm1 = tm0;
    }
  }
  static bool attr_done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_done[dev]) {   // outside the cache: set it on every launch
    int rc = record(cudaFuncSetAttribute(conv_rows_tc_kernel<BN, SH, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(Cfg::SMEM)));
    if (rc != WMD_OK) return rc;
    if (dev >= 0 && dev < 64) attr_done[dev] = true;
  }
  const long long tiles = static_cast<long long>(ceil_div(d.max_rows, TC_BM)) * ceil_div(d.cout, BN) * (splits > 0 ? splits : 1);
  const long long cap = sm_count() - g_reserved_sms > 1 ? sm_count() - g_reserved_sms : 1;
  const int grid = splits == 0 ? static_cast<int>(cap) : static_cast<int>(tiles < cap ? (tiles < 1 ? 1 : tiles) : cap);
  conv_rows_tc_kernel<BN, SH, F16><<<grid, TC_THREADS, Cfg::SMEM, stream>>>(d, d.w, splits, partial, tm0, tm1);
  int rc = launched();
  if (rc != WMD_OK || splits <= 1) return rc;      // whole tiles, or balanced: the kernel's own fix-up finishes cut tiles
  const int nchunks = d.taps * ((d.c0 + TC_BK - 1) / TC_BK + (d.c1 + TC_BK - 1) / TC_BK);
  const long long all_tiles = static_cast<long long>(ceil_div(d.max_rows, TC_BM)) * ceil_div(d.cout, BN);
  const long long red_grid = all_tiles < 8 * cap ? all_tiles : 8 * cap;
  tc_reduce_kernel<<<static_cast<int>(red_grid < 1 ? 1 : red_grid), 256, 0, stream>>>(partial, splits, grid, BN, nchunks, d.bias, d.y, d.ldy, d.cout,
                                                              d.count, d.max_rows, d.act, d.act_param);
  return launched();
}

}  // namespace wmd

#ifdef WMD_TC_TRACE
extern "C" int wmd_debug_tc_trace(long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, wmd::g_trace, sizeof(wmd::g_trace)) == cudaSuccess ? 0 : 1;
}
extern "C" int wmd_debug_tc_tile_trace(long long* host_out) {
  return cudaMemcpyFromSymbol(host_out, wmd::g_tile_trace, sizeof(wmd::g_tile_trace)) == cudaSuccess ? 0 : 1;
}
#endif

extern "C" int wmd_conv_tc_tile_n(int cout) { return wmd::tc_tile_n(cout); }

extern "C" int wmd_conv_tc_set_reserved_sms(int n) {
  const int was = wmd::g_reserved_sms;
  if (n >= 0) wmd::g_reserved_sms = n;
  return was;
}

extern "C" int wmd_conv_tc_set_shared_taps(int on) {
  const int was = wmd::g_shared_taps;
  if (on >= 0) wmd::g_shared_taps = on ? 1 : 0;
  return was;
}

extern "C" size_t wmd_conv_tc_weight_floats(int cout, int c0, int c1, int taps) {
  using namespace wmd;
  const int bn = tc_tile_n(cout);
  const int nchunks = taps * ((c0 + TC_BK - 1) / TC_BK + (c1 + TC_BK - 1) / TC_BK);
  return static_cast<size_t>(ceil_div(cout, bn)) * nchunks * 2 * bn * TC_BK;
}

extern "C" int wmd_pack_conv_weight_tc_f32(const float* w, float* packed, int Cout, int c0, int c1, int taps,
                                           wmd_stream_t stream) {
  using namespace wmd;
  WMD_REQUIRE(w && packed, WMD_ERR_ARG);
  WMD_REQUIRE(Cout > 0 && c0 > 0 && c1 >= 0 && (taps == 1 || taps == 9), WMD_ERR_SHAPE);
  const long long total = static_cast<long long>(wmd_conv_tc_weight_floats(Cout, c0, c1, taps));
  pack_weight_tc_kernel<<<stride_grid(total, 256), 256, 0, as_stream(stream)>>>(w, packed, Cout, c0, c1, taps,
                                                                               tc_tile_n(Cout), total);
  return launched();
}

extern "C" size_t wmd_conv_tc16_weight_bytes(int cout, int c0, int c1, int taps) {
  using namespace wmd;
  const int bn = tc_tile_n(cout);
  const int nchunks = taps * ((c0 + TC_BK - 1) / TC_BK + (c1 + TC_BK - 1) / TC_BK);
  return 128 + static_cast<size_t>(ceil_div(cout, bn)) * nchunks * bn * 128;
}

extern "C" int wmd_pack_conv_weight_tc16_f32(const float* w, void* packed, int Cout, int c0, int c1, int taps,
                                             wmd_stream_t stream) {
  using namespace wmd;
  WMD_REQUIRE(w && packed, WMD_ERR_ARG);
  WMD_REQUIRE(Cout > 0 && c0 > 0 && c1 >= 0 && (taps == 1 || taps == 9), WMD_ERR_SHAPE);
  WMD_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 127) == 0, WMD_ERR_SHAPE);
  cudaStream_t st = as_stream(stream);
  unsigned char* out = static_cast<unsigned char*>(packed);
  int rc = record(cudaMemsetAsync(out, 0, 128, st));
  if (rc != WMD_OK) return rc;
  const long long nw = static_cast<long long>(Cout) * (c0 + c1) * taps;
  absmax_kernel<<<stride_grid(nw, 256), 256, 0, st>>>(w, nw, reinterpret_cast<float*>(out));
  rc = launched();
  if (rc != WMD_OK) return rc;
  const int bn = tc_tile_n(Cout);
  const int nchunks = taps * ((c0 + TC_BK - 1) / TC_BK + (c1 + TC_BK - 1) / TC_BK);
  const long long total = static_cast<long long>(ceil_div(Cout, bn)) * nchunks * bn * TC_BK;
  pack_weight_tc16_kernel<<<stride_grid(total, 256), 256, 0, st>>>(w, out, Cout, c0, c1, taps, bn, total);
  rc = launched();
  if (rc != WMD_OK) return rc;
  finish_header_tc16_kernel<<<1, 1, 0, st>>>(out);
  return launched();
}

extern "C" int wmd_amax_f32(const float* x, long long count, float* amax, wmd_stream_t stream) {
  using namespace wmd;
  WMD_REQUIRE(x && amax, WMD_ERR_ARG);
  if (count <= 0) return WMD_OK;
  absmax_kernel<<<stride_grid(count, 256, 16), 256, 0, as_stream(stream)>>>(x, count, amax);
  return launched();
}

extern "C" size_t wmd_conv_tc_splitk_ws_bytes(int max_rows, int ldy, int splits) {
  if (splits == 1) return 0;
  if (splits == 0)   // balanced: [stream-K tile][slab][256 rows][N <= 128] floats, tiles x slabs <= CTAs x kBalSlabs whatever the layer size
    return wmd::kBalCounterBytes + static_cast<size_t>(wmd::sm_count()) * wmd::kBalSlabs * wmd::TC_BM * 128 * sizeof(float);
  return wmd::kBalCounterBytes + static_cast<size_t>(splits) * static_cast<size_t>(max_rows) * static_cast<size_t>(ldy) * sizeof(float);
}

extern "C" int wmd_conv_rows_tc_f32(const wmd_conv_desc* dp, wmd_stream_t stream) {
  return wmd_conv_rows_tc_splitk_f32(dp, 1, nullptr, 0, stream);
}

extern "C" int wmd_conv_rows_tc_splitk_f32(const wmd_conv_desc* dp, int splits, void* ws, size_t ws_bytes,
                                           wmd_stream_t stream) {
  using namespace wmd;
  WMD_REQUIRE(dp, WMD_ERR_ARG);
  WMD_REQUIRE(splits >= 0 && splits <= 16, WMD_ERR_ARG);
  WMD_REQUIRE(splits == 1 || (ws != nullptr && ws_bytes >= wmd_conv_tc_splitk_ws_bytes(dp->max_rows, dp->ldy, splits)),
              WMD_ERR_WORKSPACE);
  wmd_conv_desc d = *dp;
  WMD_REQUIRE(d.x0 && d.w && d.y, WMD_ERR_ARG);
  WMD_REQUIRE(d.taps == 1 || d.taps == 9, WMD_ERR_ARG);
  WMD_REQUIRE(d.pad_mode >= WMD_PAD_ZERO && d.pad_mode <= WMD_PAD_REPLICATE, WMD_ERR_ARG);
  WMD_REQUIRE(d.act >= WMD_ACT_NONE && d.act <= WMD_ACT_SIGMOID, WMD_ERR_ARG);
  WMD_REQUIRE(d.precision == WMD_PREC_TF32X3 || d.precision == WMD_PREC_F16X3, WMD_ERR_ARG);
  WMD_REQUIRE(d.shift0 == 0 || d.shift0 == 1, WMD_ERR_ARG);
  WMD_REQUIRE((d.pixels == nullptr) == (d.count == nullptr), WMD_ERR_ARG);
  WMD_REQUIRE(d.N > 0 && d.H > 0 && d.W > 0 && d.c0 > 0 && d.cout > 0 && d.max_rows >= 0, WMD_ERR_SHAPE);
  WMD_REQUIRE(static_cast<long long>(d.N) * d.H * d.W < (1ll << 31), WMD_ERR_SHAPE);
  if (d.x1 == nullptr) { d.c1 = 0; d.ld1 = 0; }
  WMD_REQUIRE(d.c1 >= 0 && (d.c1 == 0 || d.x1), WMD_ERR_ARG);
  WMD_REQUIRE(d.ld0 >= d.c0 && d.ld0 % 4 == 0 && (reinterpret_cast<uintptr_t>(d.x0) & 15) == 0, WMD_ERR_SHAPE);
  WMD_REQUIRE(d.c1 == 0 || (d.ld1 >= d.c1 && d.ld1 % 4 == 0 && (reinterpret_cast<uintptr_t>(d.x1) & 15) == 0),
              WMD_ERR_SHAPE);
  WMD_REQUIRE((reinterpret_cast<uintptr_t>(d.w) & 15) == 0, WMD_ERR_SHAPE);
  WMD_REQUIRE(d.ldy >= d.cout, WMD_ERR_SHAPE);
  // the partial-sum passes move float4s
  WMD_REQUIRE(splits == 1 || (d.ldy % 4 == 0 && (reinterpret_cast<uintptr_t>(d.y) & 15) == 0 &&
                              (reinterpret_cast<uintptr_t>(ws) & 15) == 0), WMD_ERR_SHAPE);
  if (d.shift0 == 1) WMD_REQUIRE(d.H % 2 == 0 && d.W % 2 == 0, WMD_ERR_SHAPE);
  if (d.pad_mode == WMD_PAD_REFLECT && d.taps == 9) WMD_REQUIRE(d.H >= 2 && d.W >= 2, WMD_ERR_SHAPE);
  // tap tables hold 32-bit offsets in 16-byte units
  WMD_REQUIRE(static_cast<long long>(d.N) * d.H * d.W * (d.ld0 / 4) < (1ll << 32) &&
                  static_cast<long long>(d.N) * d.H * d.W * (d.ld1 / 4) < (1ll << 32),
              WMD_ERR_UNSUPPORTED);
  if (d.max_rows == 0) return WMD_OK;
  {
    const int nchunks = d.taps * ((d.c0 + TC_BK - 1) / TC_BK + (d.c1 + TC_BK - 1) / TC_BK);
    if (splits > nchunks) splits = nchunks;      // every split needs at least one chunk
    if (splits == 0 && nchunks < 2) splits = 1;   // nothing to balance inside a one-chunk reduction
  }
  float* partial = static_cast<float*>(ws);
  const bool sh = d.taps == 9 && g_shared_taps != 0;
  const bool f16 = d.precision == WMD_PREC_F16X3;
  if (f16) WMD_REQUIRE(d.amax0 != nullptr && (d.c1 == 0 || d.amax1 != nullptr), WMD_ERR_ARG);
  if (f16) WMD_REQUIRE(splits <= 1, WMD_ERR_UNSUPPORTED);   // tc_reduce_kernel sums unscaled slabs: tf32 operands only
  cudaStream_t st = as_stream(stream);
#define WMD_TC_LAUNCH(BN_)                                                                                              \
  return f16 ? (sh ? launch_tc<BN_, true, true>(d, splits, partial, st) : launch_tc<BN_, false, true>(d, splits, partial, st)) \
             : (sh ? launch_tc<BN_, true, false>(d, splits, partial, st) : launch_tc<BN_, false, false>(d, splits, partial, st))
  switch (tc_tile_n(d.cout)) {
    case 128: WMD_TC_LAUNCH(128);
    case 64: WMD_TC_LAUNCH(64);
    default: WMD_TC_LAUNCH(32);
  }
#undef WMD_TC_LAUNCH
}
