// Dense stages of the Faster R-CNN TEST graph as ONE implicit-GEMM kernel for sm_100a:
//   slim.conv2d 3x3 / 1x1 (any stride), slim.fully_connected  (lib/nets/vgg16.py:26-60,
//   resnet_v1 bottlenecks, mobilenet pointwise, lib/nets/network.py:323-378)
//
// This file holds two generations of that kernel.  The one in production is conv_gemm_f16x3_kernel (r02, second half of the
// file: its own header comment describes it); the r01 kernel below, conv_gemm_tf32x3_kernel, is kept behind
// FRCNN_CONV_TF32X3 for A/B measurements.  What follows is the r01 design, which the r02 kernel inherits (implicit GEMM over
// TMA boxes, A operand in tensor memory, two-level accumulation, persistent units, split-K).
//
// Math: D[M=pixels, N=cout] = sum over (filter tap, cin chunk) A_tap[M, 32] * W[N, 32]^T, fp32-grade via the
// 3xTF32 split  a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi  (hi = RN_tf32(x), lo = RN_tf32(x - hi)),
// accumulated in fp32 in TMEM by tcgen05.mma.kind::tf32.
//
// Data movement: activations stay plain NHWC fp32 in HBM.  For filter tap (r,s) the A operand of a tile of
// tn x th x tw output pixels is ONE 4-D TMA box {32 ch, tw, th, tn} of the input at offset
// (w0*stride+s-pad_l, h0*stride+r-pad_t): out-of-bounds rows/cols are zero-filled by TMA, which IS the
// convolution's zero padding -- no im2col buffer ever exists.  Weights are pre-split (hi/lo planes), K-major,
// SWIZZLE_128B in shared memory (the UMMA B operand).
//
// r01 finding 1 (profiles/r01_*): with both operands in shared memory the kernel was bound by the shared-memory
// data pipe (3 MMAs re-read A and B, the splitter rewrote A twice: ~190 KB of smem traffic per 32-wide k-block,
// l1tex data pipe ~90% busy, tensor pipe 23-56%).  So the A operand now lives in TENSOR MEMORY: the splitter
// warps read the raw fp32 tile from smem once (un-swizzling their own 128-byte row), and tcgen05.st the hi and
// lo planes into a 4-deep TMEM ring; tcgen05.mma runs in TS mode (A from TMEM, B from smem).
// r01 finding 2: the tensor core adds into its fp32 accumulator with truncation (error grows linearly with the
// number of MMA steps, ~2.4e-5 relative at K=3136), so accumulation is two-level: TMEM holds only the partial
// sum of a short chunk of k-blocks, which the epilogue warps add into fp32 REGISTER
// accumulators with round-to-nearest adds.  r01 finding 3: every such promotion stalls the tensor pipe for ~950
// cycles (tcgen05.ld of a 128x128 fp32 tile vs the MMAs' own TMEM traffic; independent of warp placement and of
// code shape), so the chunk length trades accuracy for speed (with all 12 MMAs of a k-block in one accumulator:
// 1/2/4/8 k-blocks -> 6e-7/7e-7/1.0e-6/1.9e-6 error vs fp64, the fp32 CPU reference sitting at 0.6e-6..2e-6).  Hence
// the D_main / D_small separation described at the TMEM map below, and a default chunk of 8 k-blocks.
//
// PERSISTENT: grid = #SMs; every role walks the same sequence of work units (output tile x split-K range); ring slots and
// barrier phases run on across units, so the next unit's loads / splits / MMAs overlap this unit's epilogue stores.
// Warp roles (448 threads, 1 CTA/SM), rings are 4 deep (index kb & 3):
//   warp 12     TMA producer      A: wait a_empty[s] -> a_full[s];  B: wait mma_done[s] -> full[s] (tx)
//   warps 0..3  operand splitter  wait a_full[s], mma_done[s]; smem row -> hi/lo -> tcgen05.st; arrive a_empty[s], full[s]
//   warp 13     MMA issuer        wait full[s] (B landed + A stored); 4 k-slices x 3 tcgen05.mma (TS); commit -> mma_done[s];
//                                 per chunk: wait acc_empty first, commit -> acc_full last
//   warps 4..11 accumulate+epilogue (two per TMEM lane quarter, half the columns each)  per chunk: wait acc_full; tcgen05.ld D_main; acc += partial; arrive acc_empty;
//                                 finally y = act(acc*scale + shift (+res)); st.global
// TMEM map (512 columns): [0, BN) D_main = chunk partial of the a_hi*b_hi products; [128, 128+BN) D_small = the two
// cross terms a_lo*b_hi + a_hi*b_lo over the WHOLE k loop (2^-11 of the result, so its truncation is harmless and it is
// read once per tile); [256, 512) A ring: slot s = 32 cols hi + 32 cols lo.  Only D_main is promoted per chunk, and it
// takes 4 instead of 12 truncating adds per k-block, so the chunk can be 3x longer for the same error.
#include <cuda_fp16.h>
#include "common.cuh"
#include "../../include/frcnn_b200.h"
#include <stdlib.h>
#include <string.h>

namespace frcnn {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 32;                          // fp32 elements: 128 B = one swizzle row
constexpr int A_TILE_BYTES = BLOCK_M * BLOCK_K * 4;  // 16 KiB
constexpr int NUM_THREADS = 448;
constexpr int SPLIT_THREADS = 128;
constexpr int EPI_THREADS = 256;                     // 8 warps: two per TMEM lane quarter, each owning half the columns
constexpr int RING = 4;                              // depth of the A-raw, B and TMEM-A rings
constexpr int TMEM_COLS = 512;
constexpr int TMEM_A_COL0 = 256;

struct ConvKernelParams {
  float* out;
  const float* residual;
  const float* scale;   // [n_tiles*BN] plan-owned: (scale or 1) * out_mult (out_mult = 2^-wexp undoes the f16x3 weight scaling, exact)
  const float* shift;   // [n_tiles*BN] plan-owned: shift or 0
  int cout, ho, wo, nimg;
  int tn, th, tw;
  int tiles_h, tiles_w;
  int kh, kw, cin, stride, pad_t, pad_l;
  int act;
  int a_box_bytes;
  int kb_per_chunk;   // k-blocks accumulated in TMEM before promotion to registers
  // Work units.  Tiles t = mt + m_tiles*nblk.  Units [0, n_full) are whole tiles (direct epilogue).  The remaining
  // `n_tail` tiles -- the ragged last round of the persistent loop, or every tile of a layer too small to fill the GPU --
  // are each split over `splits` units along K: unit n_full + v -> tile n_full + v / splits, split v % splits, which writes
  // its raw partial tile to ws[(v / splits)][v % splits][128][BN]; tail_reduce_kernel sums them in index order and
  // runs the epilogue (r02 measured an in-kernel 'last CTA to arrive reduces' fix-up: 21 us instead of 13 us for a 38x50 1x1 layer).
  int kb_per_split;
  int m_tiles, n_tiles, total_units, n_full, splits;
  int raster_n;       // 1: consecutive tile indices walk the N-blocks of one M-tile (activations streamed once), 0: M-tiles first
  float* ws;
  long long* trace;   // debug: clock64() stamps of CTA (0,0)'s pipeline hand-offs; normally NULL
  int num_kb_total;   // f16x3: 64-wide k-blocks of the whole K loop
  int dbg;            // development ablations (FRCNN_CONV_DBG, read at plan creation): 1 splitter skips load+convert, 2 MMA issues only
                      // the hi*hi product, 4 / 8 producer A / B skip their TMA, 16 epilogue skips the chunk promotion loads.  0 in production.
};

// clock64 stamps of CTA 0's pipeline hand-offs: compiled in only in the development build (libfrcnn_b200_wd.so, -DFRCNN_WATCHDOG);
// in the production library the macros vanish (r02: the stamp sites cost ~5 instructions each -- 20 per k-block on a splitter
// warp, 15 on the MMA-issuing warp, both of which bound the k-block period).
#ifdef FRCNN_WATCHDOG
#define FRCNN_TRACE2(base, idx)                                                             \
  do {                                                                                      \
    if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && (idx) < 64) p.trace[(base) + (idx)] = clock64(); \
  } while (0)
#define FRCNN_TRACE(slot, kbv)                                                              \
  do {                                                                                      \
    if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && (kbv) < 64) p.trace[(kbv) * 8 + (slot)] = clock64(); \
  } while (0)
#else
#define FRCNN_TRACE2(base, idx) do { } while (0)
#define FRCNN_TRACE(slot, kbv) do { } while (0)
#endif

constexpr int STAGE_BYTES = 8 * 32 * 32 * 4;          // epilogue transposition buffer: 8 warps x 32 rows x 32 columns fp32
template <int BN> constexpr int b_stage_bytes() { return 2 * BN * BLOCK_K * 4; }
template <int BN> constexpr int smem_bytes() {
  return RING * (A_TILE_BYTES + b_stage_bytes<BN>()) + STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (8-row x 128 B atoms, 1024 B apart)
__device__ __forceinline__ uint64_t sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;                  // LBO: unused for swizzled K-major
  d |= (uint64_t)(1024u >> 4) << 32;       // SBO
  d |= (uint64_t)1 << 46;                  // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
  return d;
}

// Work unit u (persistent loop: u = blockIdx.x, += gridDim.x) -> output tile + split-K range.
struct Unit {
  int w0, h0, n0, nblk, z, kb0, num_kb, slot;   // slot >= 0: tail tile index (raw partial output), -1: whole tile
};
__device__ __forceinline__ Unit decode_unit(const ConvKernelParams& p, int u, int num_kb_total) {
  Unit t;
  int tile;
  if (u < p.n_full) { tile = u; t.z = 0; t.slot = -1; }
  else { const int v = u - p.n_full; t.slot = v / p.splits; t.z = v - t.slot * p.splits; tile = p.n_full + t.slot; }
  // raster order of the tile index (r02 finding 4, ncu on the batch-4 head: with all M-tiles of one N-block first, the 241 MB
  // activation of block4's shortcut was streamed from DRAM once per N-block -- 16 x, 3.9 GB, DRAM 67 % busy): the operand
  // with the larger footprint is walked ONCE, the other one stays L2 resident (decide_geometry sets raster_n).
  int mt;
  if (p.raster_n) { t.nblk = tile % p.n_tiles; mt = tile / p.n_tiles; }
  else { mt = tile % p.m_tiles; t.nblk = tile / p.m_tiles; }
  const int tile_w = mt % p.tiles_w;
  const int tile_h = (mt / p.tiles_w) % p.tiles_h;
  const int tile_n = mt / (p.tiles_w * p.tiles_h);
  t.w0 = tile_w * p.tw; t.h0 = tile_h * p.th; t.n0 = tile_n * p.tn;
  if (t.slot < 0) { t.kb0 = 0; t.num_kb = num_kb_total; }
  else { t.kb0 = t.z * p.kb_per_split; t.num_kb = min(p.kb_per_split, num_kb_total - t.kb0); }
  return t;
}

// ---------------- tile epilogue shared by both kernels (overlaps the next unit's main loop) ----------------
// `acc` = this thread's W = BN/2 fp32 sums of output row (q*32 + lane), columns [col0, col0 + W) of the tile; ew = index of the
// epilogue warp (0..7) = its 4 KB slice of the transposition buffer.
//
// r01 finding 4: writing each thread's own output row straight from registers (32 lanes = 32 rows, 8 KB apart) made every
// global access 32 separate sectors.  The tile is transposed through shared memory 32 columns at a time: thread = row writes
// XOR-swizzled 16-byte chunks (conflict free), then each lane owns 4 fixed channels and walks the warp's rows with coalesced
// 128-bit accesses (one full 128-byte line per row).  r01 finding 5: epilogue inputs are loaded with pinned (asm volatile)
// loads -- with __ldg the compiler sank the loads into the row loop.
// r02 finding 3 (ncu source page, head 1x1 512->2048): the generic epilogue -- every flag a run-time test per element, scalar
// tails, `continue`s that stop the scheduler from overlapping rows -- executed ~2500 instructions per warp per tile and took
// ~20 000 cycles, 3x the tile's MMA time: short-K layers were EPILOGUE bound.  Hence: p.scale / p.shift are always present
// (plan-owned vectors padded to the tile grid, scale pre-multiplied by the exact power-of-two out_mult), residual and
// activation are template parameters, and rows are computed unconditionally with only the store predicated.
constexpr int EPI_CH = 8;                                  // 16-byte chunks per staged 32-column row
constexpr int EPI_ROWS_PER_IT = 4;
constexpr int EPI_ITERS = 8;

template <int ACT>
__device__ __forceinline__ float apply_act(float a) {
  if (ACT == FRCNN_ACT_RELU) return fmaxf(a, 0.f);
  if (ACT == FRCNN_ACT_RELU6) return fminf(fmaxf(a, 0.f), 6.f);
  return a;
}

// y = act(v*scale + shift (+ res)) with one rounding per operation (the oracle's order: tf.nn.batch_normalization /
// bias_add, then the shortcut add, then the activation)
template <bool RES, int ACT>
__device__ __forceinline__ float4 finish4(const float4 v, const float4 sc, const float4 sh, const float4 r) {
  float4 y;
  y.x = __fadd_rn(__fmul_rn(v.x, sc.x), sh.x); y.y = __fadd_rn(__fmul_rn(v.y, sc.y), sh.y);
  y.z = __fadd_rn(__fmul_rn(v.z, sc.z), sh.z); y.w = __fadd_rn(__fmul_rn(v.w, sc.w), sh.w);
  if (RES) { y.x = __fadd_rn(y.x, r.x); y.y = __fadd_rn(y.y, r.y); y.z = __fadd_rn(y.z, r.z); y.w = __fadd_rn(y.w, r.w); }
  y.x = apply_act<ACT>(y.x); y.y = apply_act<ACT>(y.y); y.z = apply_act<ACT>(y.z); y.w = apply_act<ACT>(y.w);
  return y;
}

// whole tile, cout % 4 == 0: stage -> coalesced float4 stores
template <int BN, bool RES, int ACT>
__device__ __forceinline__ void epilogue_vec(const ConvKernelParams& p, const int cbase, const float (&acc)[BN / 2], float4* stage,
                                             const int lane, const int my_pix) {
  constexpr int W = BN / 2;
  const int cg = lane & (EPI_CH - 1), rsub = lane >> 3;
  const int cout = p.cout;
  int pixr[EPI_ITERS];
#pragma unroll
  for (int it = 0; it < EPI_ITERS; ++it) pixr[it] = __shfl_sync(0xffffffffu, my_pix, it * EPI_ROWS_PER_IT + rsub);
#pragma unroll
  for (int pass = 0; pass < W / 32; ++pass) {
    const int c = cbase + pass * 32 + cg * 4;              // first of this lane's 4 output channels in this pass
    const bool col_ok = c < cout;
    const float4 sc = ld_nc_f4_pinned(p.scale + c);        // padded to the tile grid: always in bounds
    const float4 sh = ld_nc_f4_pinned(p.shift + c);
    __syncwarp();                                           // previous pass's reads are done
#pragma unroll
    for (int j = 0; j < EPI_CH; ++j) {
      const int a0 = pass * 32 + 4 * j;
      stage[lane * EPI_CH + ((j ^ lane) & (EPI_CH - 1))] = make_float4(acc[a0], acc[a0 + 1], acc[a0 + 2], acc[a0 + 3]);
    }
    // residual rows of this pass: issued after the pass's accumulators are staged (their registers are free again)
    float4 rv[EPI_ITERS];
    if (RES) {
#pragma unroll
      for (int it = 0; it < EPI_ITERS; ++it)
        rv[it] = (pixr[it] >= 0 && col_ok) ? ld_nc_f4_pinned(p.residual + (size_t)pixr[it] * cout + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();
#pragma unroll
    for (int it = 0; it < EPI_ITERS; ++it) {
      const int r = it * EPI_ROWS_PER_IT + rsub;
      const float4 v = stage[r * EPI_CH + ((cg ^ r) & (EPI_CH - 1))];
      const float4 y = finish4<RES, ACT>(v, sc, sh, RES ? rv[it] : v);
      if (pixr[it] >= 0 && col_ok) *reinterpret_cast<float4*>(p.out + (size_t)pixr[it] * cout + c) = y;
    }
  }
}

// any cout (scalar tails): same arithmetic, run-time flags
template <int BN>
__device__ __forceinline__ void epilogue_generic(const ConvKernelParams& p, const int cbase, const float (&acc)[BN / 2], float4* stage,
                                                 const int lane, const int my_pix) {
  constexpr int W = BN / 2;
  const int cg = lane & (EPI_CH - 1), rsub = lane >> 3;
#pragma unroll
  for (int pass = 0; pass < W / 32; ++pass) {
    const int c = cbase + pass * 32 + cg * 4;
    const float4 sc4 = ld_nc_f4_pinned(p.scale + c), sh4 = ld_nc_f4_pinned(p.shift + c);
    const float sc[4] = {sc4.x, sc4.y, sc4.z, sc4.w}, sh[4] = {sh4.x, sh4.y, sh4.z, sh4.w};
    __syncwarp();
#pragma unroll
    for (int j = 0; j < EPI_CH; ++j) {
      const int a0 = pass * 32 + 4 * j;
      stage[lane * EPI_CH + ((j ^ lane) & (EPI_CH - 1))] = make_float4(acc[a0], acc[a0 + 1], acc[a0 + 2], acc[a0 + 3]);
    }
    __syncwarp();
#pragma unroll 1
    for (int it = 0; it < EPI_ITERS; ++it) {
      const int r = it * EPI_ROWS_PER_IT + rsub;
      const int pix = __shfl_sync(0xffffffffu, my_pix, r);
      if (pix < 0) continue;
      const float4 v = stage[r * EPI_CH + ((cg ^ r) & (EPI_CH - 1))];
      const float y[4] = {v.x, v.y, v.z, v.w};
      float* optr = p.out + (size_t)pix * p.cout + c;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (c + e >= p.cout) break;
        float a = __fadd_rn(__fmul_rn(y[e], sc[e]), sh[e]);
        if (p.residual) a = __fadd_rn(a, __ldg(p.residual + (size_t)pix * p.cout + c + e));
        if (p.act == FRCNN_ACT_RELU) a = fmaxf(a, 0.f);
        else if (p.act == FRCNN_ACT_RELU6) a = fminf(fmaxf(a, 0.f), 6.f);
        optr[e] = a;
      }
    }
  }
}

template <int BN, bool RES>
__device__ __forceinline__ void epilogue_dispatch(const ConvKernelParams& p, const int cbase, const float (&acc)[BN / 2], float4* stage,
                                                  const int lane, const int my_pix) {
  if (p.act == FRCNN_ACT_RELU) epilogue_vec<BN, RES, FRCNN_ACT_RELU>(p, cbase, acc, stage, lane, my_pix);
  else if (p.act == FRCNN_ACT_RELU6) epilogue_vec<BN, RES, FRCNN_ACT_RELU6>(p, cbase, acc, stage, lane, my_pix);
  else epilogue_vec<BN, RES, FRCNN_ACT_NONE>(p, cbase, acc, stage, lane, my_pix);
}

template <int BN>
__device__ __forceinline__ void epilogue_tile(const ConvKernelParams& p, const Unit& t, const float (&acc)[BN / 2],
                                              uint8_t* smem_stage, int ew, int q, int lane) {
  constexpr int W = BN / 2;
  const int col0 = (ew >> 2) * W;
  float4* stage = reinterpret_cast<float4*>(smem_stage + ew * (32 * 32 * 4));
  const int row = q * 32 + lane;
  const int rows_img = p.th * p.tw;
  const int dn = row / rows_img, rem = row % rows_img;
  const int dh = rem / p.tw, dw = rem % p.tw;
  const int n = t.n0 + dn, h = t.h0 + dh, w = t.w0 + dw;
  const bool valid = (row < p.tn * rows_img) && n < p.nimg && h < p.ho && w < p.wo;
  const int cg = lane & (EPI_CH - 1);
  const int rsub = lane >> 3;
  const int my_pix = valid ? (int)(((long long)n * p.ho + h) * p.wo + w) : -1;
  const int cbase = t.nblk * BN + col0;
  if (t.slot >= 0) {
    // split tile: raw partial sums into the tile-local [128][BN] workspace (row-major, coalesced through the transposition buffer)
    float* const wbase = p.ws + ((size_t)t.slot * p.splits + t.z) * (size_t)(BLOCK_M * BN) + (size_t)(q * 32) * BN + col0;
#pragma unroll
    for (int pass = 0; pass < W / 32; ++pass) {
      __syncwarp();
#pragma unroll
      for (int j = 0; j < EPI_CH; ++j) {
        const int a0 = pass * 32 + 4 * j;
        stage[lane * EPI_CH + ((j ^ lane) & (EPI_CH - 1))] = make_float4(acc[a0], acc[a0 + 1], acc[a0 + 2], acc[a0 + 3]);
      }
      __syncwarp();
#pragma unroll
      for (int it = 0; it < EPI_ITERS; ++it) {
        const int r = it * EPI_ROWS_PER_IT + rsub;
        __stcg(reinterpret_cast<float4*>(wbase + (size_t)r * BN + pass * 32 + cg * 4), stage[r * EPI_CH + ((cg ^ r) & (EPI_CH - 1))]);
      }
    }
    return;                                                // the epilogue of split tiles runs in tail_reduce_kernel
  }
  if ((p.cout & 3) != 0) {
    // scalar-tail layers are never split (decide_geometry) -- generic path
    epilogue_generic<BN>(p, cbase, acc, stage, lane, my_pix);
    return;
  }
  if (p.residual) epilogue_dispatch<BN, true>(p, cbase, acc, stage, lane, my_pix);
  else epilogue_dispatch<BN, false>(p, cbase, acc, stage, lane, my_pix);
}

template <int BN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                        const __grid_constant__ CUtensorMap tmBlo, const ConvKernelParams p) {
  constexpr int kBTile = BN * BLOCK_K * 4;
  constexpr int kBStage = b_stage_bytes<BN>();
  constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
  static_assert(BN <= 128, "D_main/D_small are 128 columns apart");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;                               // RING x 16 KiB raw fp32 A tiles (TMA, swizzled)
  uint8_t* smem_b = smem + RING * A_TILE_BYTES;         // RING x (B_hi | B_lo)
  uint8_t* smem_stage = smem_b + RING * kBStage;        // epilogue transposition buffer (own region: overlaps next tile's loads)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem_stage + STAGE_BYTES);
  uint64_t* a_empty = a_full + RING;
  uint64_t* full = a_empty + RING;            // B bytes landed (tx) AND the 128 splitter threads stored A hi/lo
  uint64_t* mma_done = full + RING;
  uint64_t* acc_full = mma_done + RING;       // D_main holds a finished chunk partial (tcgen05.commit)
  uint64_t* acc_empty = acc_full + 1;         // the epilogue warps have read it (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) FRCNN_TRACE2(700, 0);
  const int num_kb_total = p.kh * p.kw * (p.cin / BLOCK_K);

  if (warp == 12 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmBhi); tma_prefetch_desc(&tmBlo);
    for (int s = 0; s < RING; ++s) {
      mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], SPLIT_THREADS);
      mbar_init(&full[s], SPLIT_THREADS + 1); mbar_init(&mma_done[s], 1);
    }
    mbar_init(acc_full, 1); mbar_init(acc_empty, EPI_THREADS);
    mbar_fence_init();
  }
  if (warp == 12) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) FRCNN_TRACE2(701, 0);
  // Programmatic dependent launch: the next kernel of the stream may begin (its prologue and weight prefetch overlap our
  // tail); we ourselves touch the previous kernel's outputs only behind pdl_wait() (A loads, residual loads, stores).
  pdl_launch_dependents();

  // Every role walks the same unit sequence; ring slots / barrier phases run on across units (kbt, ct are running totals).
  if (warp == 12) {
    if (lane == 0) {
      const int cchunks = p.cin / BLOCK_K;
      // weights do not depend on the previous kernel: prefetch the first unit's leading B tiles before the dependency wait
      int b_issued = 0;
      if ((int)blockIdx.x < p.total_units) {
        const Unit t0 = decode_unit(p, blockIdx.x, num_kb_total);
        for (int kb = 0; kb < t0.num_kb && kb < RING; ++kb, ++b_issued) {
          const int g = t0.kb0 + kb;
          const int tap = g / cchunks, kc = g - tap * cchunks;
          mbar_expect_tx(&full[kb], (uint32_t)(2 * kBTile));
          const int kcoord = tap * p.cin + kc * BLOCK_K;
          tma_load_2d(smem_b + kb * kBStage, &tmBhi, &full[kb], kcoord, t0.nblk * BN);
          tma_load_2d(smem_b + kb * kBStage + kBTile, &tmBlo, &full[kb], kcoord, t0.nblk * BN);
        }
      }
      pdl_wait();
      int kbt = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const Unit t = decode_unit(p, u, num_kb_total);
#pragma unroll 1
        for (int kb = 0; kb < t.num_kb; ++kb, ++kbt) {
          const int g = t.kb0 + kb;                               // global k-block -> (filter tap, channel chunk)
          const int tap = g / cchunks, kc = g - tap * cchunks;
          const int r = tap / p.kw, s = tap - r * p.kw;
          const int slot = kbt & (RING - 1);
          const uint32_t par = (uint32_t)(kbt / RING) & 1u;
          mbar_wait(&a_empty[slot], par ^ 1u);                 // splitter has consumed the raw tile
          mbar_expect_tx(&a_full[slot], (uint32_t)p.a_box_bytes);
          tma_load_4d(smem_a + slot * A_TILE_BYTES, &tmA, &a_full[slot], kc * BLOCK_K, t.w0 * p.stride + s - p.pad_l,
                      t.h0 * p.stride + r - p.pad_t, t.n0);
          if (kbt >= b_issued) {
            mbar_wait(&mma_done[slot], par ^ 1u);              // MMAs that read this B slot have completed
            FRCNN_TRACE(0, kbt);
            mbar_expect_tx(&full[slot], (uint32_t)(2 * kBTile));
            const int kcoord = tap * p.cin + kc * BLOCK_K;
            tma_load_2d(smem_b + slot * kBStage, &tmBhi, &full[slot], kcoord, t.nblk * BN);
            tma_load_2d(smem_b + slot * kBStage + kBTile, &tmBlo, &full[slot], kcoord, t.nblk * BN);
          }
          FRCNN_TRACE(1, kbt);
        }
      }
    }
    __syncwarp();
  } else if (warp == 13) {
    if (lane == 0) {
      int kbt = 0, ct = 0;
      const uint32_t d_main = tmem_base, d_small = tmem_base + 128u;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const Unit t = decode_unit(p, u, num_kb_total);
        int in_chunk = 0;
#pragma unroll 1
        for (int kb = 0; kb < t.num_kb; ++kb, ++kbt) {
          const int slot = kbt & (RING - 1);
          const uint32_t par = (uint32_t)(kbt / RING) & 1u;
          if (in_chunk == 0) {
            mbar_wait(acc_empty, ((uint32_t)ct & 1u) ^ 1u);          // previous chunk partial (and, across units, D_small) has been read
            FRCNN_TRACE2(576, ct);
          }
          mbar_wait(&full[slot], par);
          tc_fence_after();
          FRCNN_TRACE(4, kbt);
          const uint32_t sb = smem_u32(smem_b + slot * kBStage);
          const uint64_t b_hi = sw128_desc(sb);
          const uint64_t b_lo = sw128_desc(sb + kBTile);
          const uint32_t a_hi = tmem_base + (uint32_t)(TMEM_A_COL0 + slot * 64);
          const uint32_t a_lo = a_hi + 32u;
#pragma unroll
          for (int k = 0; k < BLOCK_K / 8; ++k) {
            const uint64_t off = (uint64_t)(k * 8 * 4) >> 4;   // B: advance 8 tf32 = 32 B inside the swizzle row
            const uint32_t ak = (uint32_t)(k * 8);             // A: 8 tf32 = 8 TMEM columns
            umma_tf32_ts(d_small, a_lo + ak, b_hi + off, kIdesc, (k > 0 || kb > 0) ? 1u : 0u);
            umma_tf32_ts(d_small, a_hi + ak, b_lo + off, kIdesc, 1u);
            umma_tf32_ts(d_main, a_hi + ak, b_hi + off, kIdesc, (k > 0 || in_chunk > 0) ? 1u : 0u);
          }
          umma_commit(&mma_done[slot]);
          FRCNN_TRACE(5, kbt);
          if (++in_chunk == p.kb_per_chunk || kb + 1 == t.num_kb) {
            umma_commit(acc_full);
            in_chunk = 0; ++ct;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp < 4) {
    // ---------------- operand splitter: smem raw tile row -> (hi, lo) planes in the TMEM A ring ----------------
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    int kbt = 0;
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit t = decode_unit(p, u, num_kb_total);
#pragma unroll 1
      for (int kb = 0; kb < t.num_kb; ++kb, ++kbt) {
        const int slot = kbt & (RING - 1);
        const uint32_t par = (uint32_t)(kbt / RING) & 1u;
        mbar_wait(&a_full[slot], par);
        // SWIZZLE_128B: 16-byte chunk c of row r sits at chunk (c ^ (r & 7)); quarter-warp phases are conflict-free
        const uint8_t* arow = smem_a + slot * A_TILE_BYTES + row * 128;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 v = *reinterpret_cast<const float4*>(arow + ((c ^ (row & 7)) << 4));
          const float h0 = to_tf32_fast(v.x), h1 = to_tf32_fast(v.y), h2 = to_tf32_fast(v.z), h3 = to_tf32_fast(v.w);
          hi[4 * c + 0] = __float_as_uint(h0); hi[4 * c + 1] = __float_as_uint(h1);
          hi[4 * c + 2] = __float_as_uint(h2); hi[4 * c + 3] = __float_as_uint(h3);
          lo[4 * c + 0] = __float_as_uint(to_tf32_fast(__fsub_rn(v.x, h0))); lo[4 * c + 1] = __float_as_uint(to_tf32_fast(__fsub_rn(v.y, h1)));
          lo[4 * c + 2] = __float_as_uint(to_tf32_fast(__fsub_rn(v.z, h2))); lo[4 * c + 3] = __float_as_uint(to_tf32_fast(__fsub_rn(v.w, h3)));
        }
        mbar_arrive(&a_empty[slot]);                          // raw tile consumed (values are in registers)
        mbar_wait(&mma_done[slot], par ^ 1u);                  // TMEM A slot no longer read by the tensor core
        tc_fence_after();
        const uint32_t ta = tmem_base + lane_field + (uint32_t)(TMEM_A_COL0 + slot * 64);
        tmem_st_32x32(ta, hi);
        tmem_st_32x32(ta + 32u, lo);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&full[slot]);
        if (threadIdx.x == 0) FRCNN_TRACE(3, kbt);
      }
    }
  } else {
    // ---------------- accumulate (TMEM chunk partials -> fp32 registers, RN adds) + epilogue ----------------
    constexpr int W = BN / 2;                 // columns owned by this warp (two warps share a TMEM lane quarter)
    const int q = warp & 3;                   // TMEM lane quarter this warp may access
    const int col0 = ((warp - 4) >> 2) * W;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col0;
    pdl_wait();                               // residual / output buffers belong to earlier kernels until they completed
    int ct = 0;
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit t = decode_unit(p, u, num_kb_total);
      const int num_chunks = (t.num_kb + p.kb_per_chunk - 1) / p.kb_per_chunk;
      float acc[W];
#pragma unroll
      for (int j = 0; j < W; ++j) acc[j] = 0.f;
      for (int c = 0; c < num_chunks; ++c, ++ct) {
        mbar_wait(acc_full, (uint32_t)ct & 1u);
        tc_fence_after();
        if (threadIdx.x == 128) FRCNN_TRACE(7, ct);
#pragma unroll
        for (int c0 = 0; c0 < W; c0 += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tq + (uint32_t)c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[c0 + j] = __fadd_rn(acc[c0 + j], __uint_as_float(v[j]));
        }
        if (c + 1 == num_chunks) {
          // the cross terms of the unit's whole k range (complete: this acc_full commit covered every MMA)
#pragma unroll
          for (int c0 = 0; c0 < W; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32(tq + (uint32_t)(128 + c0), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[c0 + j] = __fadd_rn(acc[c0 + j], __uint_as_float(v[j]));
          }
        }
        tc_fence_before();
        mbar_arrive(acc_empty);               // the MMA warp may overwrite D_main (and, for the next unit, D_small)
        if (threadIdx.x == 128) FRCNN_TRACE2(512, ct);
      }
      if (threadIdx.x == 128) FRCNN_TRACE2(702, 0);
      epilogue_tile<BN>(p, t, acc, smem_stage, warp - 4, q, lane);
      if (threadIdx.x == 128) FRCNN_TRACE2(703, 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 12) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
  if (threadIdx.x == 384) FRCNN_TRACE2(704, 0);
}

// =====================================================================================================================
// r02: FP16x3 kernel.  Same math contract as the TF32x3 kernel above (fp32-grade products from a two-term split of both
// operands, three MMAs per product, chunked fp32 accumulation), re-cut around what the ncu source pages showed:
//   (1) a TF32 MMA moves 8 k per instruction, an FP16 MMA 16 k at the same 64 cycles (128x128 tile) -- and fp16 has the
//       SAME 11-bit significand as tf32.  With x_hi = RN_f16(x), x_lo = RN_f16((x - x_hi) * 2^11) every operand is carried
//       to 2^-22 relative exactly like the tf32 hi/lo pair, at half the tensor time and half the B bytes (shared memory,
//       L2).  Range: the lo planes are pre-scaled by 2^11 (D_small is folded back with one fma by 2^-11), weights are
//       pre-scaled per layer by a power of two so that max|w| sits in [2^13, 2^14) (undone exactly by `out_mult` in the
//       epilogue).  Activations are converted with round-to-nearest and IEEE overflow: fp32-grade for |x| < 65520 (then
//       |x - x_hi| <= 16, so the lo plane stays in range), while a larger |x|, Inf or NaN turns every output it feeds into
//       Inf / NaN, as fp32 arithmetic would -- never into a finite wrong value.  Tiny values lose little: an activation
//       below fp16's normal range (|x| < 2^-14) keeps 2^-36 absolute through the subnormal lo plane.
//   (2) r01's operand splitter was issue bound: ONE warp per TMEM lane quarter, 334 instructions per k-block at the 0.5 IPC a
//       single warp gets from the fma/alu pipes.  Now 8 splitter warps (group g converts the g-th 32-channel half of every
//       64-wide k-block), 4 instructions per element on packed pairs, and A / B have their own producer warps and rings.
//   (3) r02 finding 1+2: the single MMA-issuing thread is a serial instruction stream at ~5 cycles per instruction (no other
//       warp hides its latencies).  Inside `if (lane == 0)` ptxas wrapped every UTCHMMA in an ELECT / R2UR.BROADCAST /
//       BRA.U.ANY loop (~150 instructions per 32-wide k-block = 1050 cycles); with the whole warp converged and elect.sync
//       only around the tcgen05 instructions it was still 114 instructions = 600 cycles per 32 k (tensor floor: 384).  Hence
//       k-blocks of 64: 12 MMAs, 2 waits and 2-3 commits per loop trip halve the per-k issue cost.
//   (4) the chunk accumulator D_main is double buffered: the MMA warp fills D_main[c & 1] while the epilogue warps drain
//       D_main[(c - 1) & 1] (tcgen05.ld reads ~64 B/clk: ~1000 cycles per 128x128 fp32 tile, formerly a stall per chunk).
//   (5) setmaxnreg moves registers from the producer / MMA / splitter warps to the 8 accumulate+epilogue warps (no spills).
// Warp roles (640 threads = 5 warpgroups, 1 CTA/SM):
//   warps 0-3   splitter group 0 (channels  0..31 of the k-block)  wait a_full[sa]; smem row -> fp16 hi/lo pairs; arrive a_empty[sa];
//   warps 4-7   splitter group 1 (channels 32..63)                 wait ta_empty[st]; tcgen05.st 32 columns; arrive ta_full[st]
//   warps 8-15  accumulate + epilogue (two per TMEM lane quarter, half the columns each)
//   warp 16     TMA producer A: wait a_empty[sa] -> two 4-D boxes (one per 32-channel half: each its own filter tap) -> a_full[sa] (tx)
//   warp 17     TMA producer B: wait b_empty[sb] -> hi + lo weight tiles -> b_full[sb] (tx); never waits for the previous kernel
//   warp 18     MMA issuer: wait ta_full[st], b_full[sb]; 4 k-slices x 3 tcgen05.mma.kind::f16 (TS); commit -> ta_empty, b_empty;
//               per chunk: wait acc_empty[b] first, commit -> acc_full[b] last; per unit: wait small_empty first
//   warp 19     idle (completes the warpgroup for setmaxnreg)
// TMEM map (512 columns): [0,128) D_main[0] | [128,256) D_main[1] | [256,384) D_small | [384,512) A ring: slot s = 64 columns =
// (hi pairs | lo pairs) of channels 0..31, then of channels 32..63.
constexpr int F_THREADS = 640;
constexpr int F_BK = 64;                                // channels per k-block (two 32-channel TMA boxes)
constexpr int F_SA = 3;                                 // smem ring of raw fp32 A stages (2 x 16 KiB each)
constexpr int F_SB = 3;                                 // smem ring of B (hi | lo) fp16 stages
constexpr int F_ST = 2;                                 // TMEM ring of split A tiles
constexpr int F_RDY = 6;                                // 'operands ready' barriers: lcm(F_ST, F_SB)
constexpr int F_A_STAGE = 2 * A_TILE_BYTES;
constexpr int F_TMEM_DSMALL = 256, F_TMEM_A0 = 384;
constexpr int F_REGS_SPLIT = 80, F_REGS_EPI = 136, F_REGS_CTRL = 40;
constexpr int F_SPLIT_THREADS = 256;
template <int BN> constexpr int f_b_tile_bytes() { return BN * F_BK * 2; }          // one fp16 plane [BN][64]: 128-byte rows
template <int BN> constexpr int f_smem_bytes() {
  return F_SA * F_A_STAGE + F_SB * 2 * f_b_tile_bytes<BN>() + STAGE_BYTES + 1024 /*align slack*/ + 512 /*barriers*/;
}

// X1 = throughput mode (FRCNN_CONV_F16X1, NOT fp32-grade): plain fp16 operands -- only the hi planes of A and B, ONE MMA per
// k-slice, fp32 accumulate with the same chunked promotion; D_small, the lo planes and their loads / conversions are skipped.
template <int BN, bool X1>
__global__ void __launch_bounds__(F_THREADS, 1)
conv_gemm_f16x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                       const __grid_constant__ CUtensorMap tmBlo, const ConvKernelParams p) {
  constexpr int kBTile = f_b_tile_bytes<BN>();
  constexpr int kBStage = 2 * kBTile;
  // instruction descriptor: D = f32 (bits 4-5 = 1), A = B = f16 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
  constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
  static_assert(BN <= 128, "accumulators are 128 columns apart");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;                               // F_SA x 2 x 16 KiB raw fp32 A tiles (TMA, SWIZZLE_128B)
  uint8_t* smem_b = smem + F_SA * F_A_STAGE;            // F_SB x (B_hi | B_lo) fp16 tiles (TMA, SWIZZLE_128B)
  uint8_t* smem_stage = smem_b + F_SB * kBStage;        // epilogue transposition buffer
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem_stage + STAGE_BYTES);
  uint64_t* a_empty = a_full + F_SA;
  // ready[kbt % 6]: k-block kbt's operands are complete -- the 256 splitter threads stored its A planes into the TMEM slot AND
  // its B tiles landed (the B producer's arrive.expect_tx + the TMA bytes).  One barrier (6 = lcm of the 2-deep TMEM ring and
  // the 3-deep B ring), so the MMA issuer pays ONE try_wait per k-block (r02 trace: a try_wait costs ~90-170 cycles of the
  // single issuing warp even when the phase is already complete, and the tensor queue is too shallow to cover it).
  uint64_t* ready = a_empty + F_SA;
  uint64_t* b_empty = ready + F_RDY;
  uint64_t* ta_empty = b_empty + F_SB;        // the MMAs reading the TMEM slot completed (tcgen05.commit)
  uint64_t* acc_full = ta_empty + F_ST;       // [2] D_main[b] holds a finished chunk partial (tcgen05.commit)
  uint64_t* acc_empty = acc_full + 2;         // [2] the epilogue warps have read D_main[b] (256 arrivals)
  uint64_t* small_empty = acc_empty + 2;      // the epilogue warps have read D_small of the finished unit (256 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(small_empty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_kb_total = p.num_kb_total;    // 64-wide k-blocks of the whole K loop (the last may be half empty)

  if (warp == 16 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmBhi); tma_prefetch_desc(&tmBlo);
    for (int s = 0; s < F_SA; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], F_SPLIT_THREADS); }
    for (int s = 0; s < F_RDY; ++s) mbar_init(&ready[s], F_SPLIT_THREADS + 1);
    for (int s = 0; s < F_SB; ++s) mbar_init(&b_empty[s], 1);
    for (int s = 0; s < F_ST; ++s) mbar_init(&ta_empty[s], 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], EPI_THREADS); }
    mbar_init(small_empty, EPI_THREADS);
    mbar_fence_init();
  }
  if (warp == 18) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();

  if (warp < 8) {
    // ---------------- operand splitter: raw fp32 row in smem -> fp16 (hi, lo * 2^11) pairs in the TMEM A ring ----------------
    reg_dec<F_REGS_SPLIT>();
    const int g = warp >> 2;                  // group = 32-channel half of the k-block
    const int q = warp & 3;                   // TMEM lane quarter
    const int row = q * 32 + lane;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    int total_kb = 0;                         // k-blocks of all units of this CTA (the splitter needs nothing else about them)
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) total_kb += decode_unit(p, u, num_kb_total).num_kb;
    int sa = 0; uint32_t pa = 0;
    int r6 = 0;
    // SWIZZLE_128B: 16-byte chunk c of row r sits at chunk (c ^ (r & 7)); quarter-warp phases are conflict-free.  The eight
    // chunk addresses of this thread's row are loop invariants up to the stage offset (32-bit shared-space addresses: the
    // generic-pointer form cost ~40 address instructions per k-block).
    const uint32_t arow0 = smem_u32(smem_a) + (uint32_t)(g * A_TILE_BYTES + row * 128);
    uint32_t coff[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) coff[c] = arow0 + (uint32_t)((c ^ (row & 7)) << 4);
#pragma unroll 1
    for (int kbt = 0; kbt < total_kb; ++kbt) {
      MBAR_WAIT(&a_full[sa], pa, 1, kbt);
      if (threadIdx.x == 0) FRCNN_TRACE(0, kbt);
      const uint32_t stage_off = (uint32_t)(sa * F_A_STAGE);
      uint32_t pk[32];                        // [0,16): hi pairs (k, k+1), [16,32): lo pairs
      if (p.dbg & 1) {
#pragma unroll
        for (int j = 0; j < 32; ++j) pk[j] = 0u;
      } else {
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 v = lds_f4(coff[c] + stage_off);
          const uint32_t h01 = pack_f16x2_rn(v.x, v.y), h23 = pack_f16x2_rn(v.z, v.w);
          const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&h01));
          const float2 f23 = __half22float2(*reinterpret_cast<const __half2*>(&h23));
          pk[2 * c] = h01; pk[2 * c + 1] = h23;
          if (!X1) {
            pk[16 + 2 * c] = pack_f16x2_rn(__fmul_rn(__fsub_rn(v.x, f01.x), 2048.f), __fmul_rn(__fsub_rn(v.y, f01.y), 2048.f));
            pk[16 + 2 * c + 1] = pack_f16x2_rn(__fmul_rn(__fsub_rn(v.z, f23.x), 2048.f), __fmul_rn(__fsub_rn(v.w, f23.y), 2048.f));
          } else {
            pk[16 + 2 * c] = 0u; pk[16 + 2 * c + 1] = 0u;
          }
        }
      }
      // raw tile consumed: the arrive carries a data dependency on every one of the 8 row loads, so it cannot be issued
      // while a load is still outstanding (the A producer re-fills the stage as soon as all 256 threads arrived)
      mbar_arrive_after(&a_empty[sa], (pk[0] | pk[2] | pk[4]) | (pk[6] | pk[8] | pk[10]) | (pk[12] | pk[14]));
      const int st = kbt & (F_ST - 1);
      if (threadIdx.x == 0) FRCNN_TRACE(1, kbt);
      MBAR_WAIT(&ta_empty[st], (((uint32_t)kbt >> 1) & 1u) ^ 1u, 2, kbt);   // TMEM slot no longer read by the tensor core
      if (threadIdx.x == 0) FRCNN_TRACE(2, kbt);
      tc_fence_after();
      if (X1) tmem_st_32x16(tmem_base + lane_field + (uint32_t)(F_TMEM_A0 + st * 64 + g * 32), pk);   // hi pairs only
      else tmem_st_32x32(tmem_base + lane_field + (uint32_t)(F_TMEM_A0 + st * 64 + g * 32), pk);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&ready[r6]);              // k-block kbt: this thread's part of the A planes is in tensor memory
      if (threadIdx.x == 0) FRCNN_TRACE(3, kbt);
      if (++r6 == F_RDY) r6 = 0;
      if (++sa == F_SA) { sa = 0; pa ^= 1u; }
    }
  } else if (warp < 16) {
    // ---------------- accumulate (TMEM chunk partials -> fp32 registers, RN adds) + epilogue ----------------
    reg_inc<F_REGS_EPI>();
    constexpr int W = BN / 2;                 // columns owned by this warp (two warps share a TMEM lane quarter)
    const int q = warp & 3;                   // TMEM lane quarter this warp may access
    const int ew = warp - 8;
    const int col0 = (ew >> 2) * W;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col0;
    pdl_wait();                               // residual / output buffers belong to earlier kernels until they completed
    uint32_t ct = 0;
    for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
      const Unit t = decode_unit(p, u, num_kb_total);
      const int num_chunks = (t.num_kb + p.kb_per_chunk - 1) / p.kb_per_chunk;
      float acc[W];
#pragma unroll
      for (int j = 0; j < W; ++j) acc[j] = 0.f;
      for (int c = 0; c < num_chunks; ++c, ++ct) {
        const uint32_t b = ct & 1u;
        MBAR_WAIT(&acc_full[b], (ct >> 1) & 1u, 3, ct);
        tc_fence_after();
        if (threadIdx.x == 256) FRCNN_TRACE(7, ct);
        if (!X1 && c + 1 == num_chunks) {
          // the cross terms of the unit's whole k range (complete: this acc_full commit covered every MMA), scaled by 2^11.
          // Drained BEFORE the last chunk partial: D_small is single buffered, the next unit's first MMA waits for it.
#pragma unroll
          for (int c0 = 0; c0 < W; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32(tq + (uint32_t)(F_TMEM_DSMALL + c0), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) acc[c0 + j] = __fmaf_rn(__uint_as_float(v[j]), 0.00048828125f, acc[c0 + j]);
          }
          tc_fence_before();
          mbar_arrive(small_empty);           // the next unit's first MMA may overwrite D_small
        }
        if (!(p.dbg & 16))
#pragma unroll
        for (int c0 = 0; c0 < W; c0 += 32) {
          uint32_t v[32];
          tmem_ld_32x32(tq + b * 128u + (uint32_t)c0, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[c0 + j] = __fadd_rn(acc[c0 + j], __uint_as_float(v[j]));
        }
        tc_fence_before();
        mbar_arrive(&acc_empty[b]);           // the MMA warp may overwrite D_main[b]
      }
      epilogue_tile<BN>(p, t, acc, smem_stage, ew, q, lane);
    }
  } else {
    reg_dec<F_REGS_CTRL>();
    if (warp == 16 && lane == 0) {
      // ---------------- TMA producer, activations ----------------
      const int cchunks = p.cin / BLOCK_K;                        // 32-channel chunks per filter tap
      const int total32 = p.kh * p.kw * cchunks;
      pdl_wait();                             // the input belongs to the previous kernel until it completed
      int sa = 0; uint32_t pa = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const Unit t = decode_unit(p, u, num_kb_total);
#pragma unroll 1
        for (int kb = 0; kb < t.num_kb; ++kb) {
          MBAR_WAIT(&a_empty[sa], pa ^ 1u, 4, kb);                // both splitter groups have consumed the stage
          if (p.dbg & 4) mbar_arrive(&a_full[sa]);
          else {
            mbar_expect_tx(&a_full[sa], (uint32_t)(2 * p.a_box_bytes));
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int g32 = (t.kb0 + kb) * 2 + i;               // global 32-channel block -> (filter tap, channel chunk)
              int tap = g32 / cchunks, kc = g32 - tap * cchunks;
              if (g32 >= total32) { tap = 0; kc = cchunks; }      // odd tail: a box past the last channel is zero-filled by TMA
              const int r = tap / p.kw, s = tap - r * p.kw;
              tma_load_4d(smem_a + sa * F_A_STAGE + i * A_TILE_BYTES, &tmA, &a_full[sa], kc * BLOCK_K, t.w0 * p.stride + s - p.pad_l,
                          t.h0 * p.stride + r - p.pad_t, t.n0);
            }
          }
          if (++sa == F_SA) { sa = 0; pa ^= 1u; }
        }
      }
    } else if (warp == 17 && lane == 0) {
      // ---------------- TMA producer, weights (static data: runs ahead of the previous kernel's tail) ----------------
      int sb = 0; uint32_t pb = 0;
      int r6 = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x) {
        const Unit t = decode_unit(p, u, num_kb_total);
#pragma unroll 1
        for (int kb = 0; kb < t.num_kb; ++kb) {
          const int kcoord = (t.kb0 + kb) * F_BK;                 // K axis of the packed weights = (tap, cin) flattened; past the end: zeros
          MBAR_WAIT(&b_empty[sb], pb ^ 1u, 5, kb);                // the MMAs that read this slot completed
          if (p.dbg & 8) mbar_arrive(&ready[r6]);
          else {
            mbar_expect_tx(&ready[r6], (uint32_t)(X1 ? kBTile : kBStage));
            tma_load_2d(smem_b + sb * kBStage, &tmBhi, &ready[r6], kcoord, t.nblk * BN);
            if (!X1) tma_load_2d(smem_b + sb * kBStage + kBTile, &tmBlo, &ready[r6], kcoord, t.nblk * BN);
          }
          if (++r6 == F_RDY) r6 = 0;
          if (++sb == F_SB) { sb = 0; pb ^= 1u; }
        }
      }
    } else if (warp == 18) {
      // ---------------- MMA issuer: the whole warp walks the loop converged (operands in uniform registers) ----------------
      // r02 finding 5 (ablations, tools/r02_conv_check.py ablate + SASS): this loop was ~140 instructions per k-block -- four
      // dependent try_waits (~90 cycles each even when the phase has completed), 64-bit descriptor arithmetic and R2UR moves
      // per MMA -- i.e. ~1000 cycles on a warp that issues one instruction every ~5 cycles, against 768 cycles of tensor work:
      // the head layers were ISSUE bound.  Now: the two per-k-block waits are one try_wait pair, every operand is base +
      // immediate (descriptor high word constant, low word = 14-bit address field), the chunk / unit waits sit outside the
      // common path (one try_wait on the joint `ready` barrier).  (Measured: neutral -- 170 vs 167 us on the head 3x3 -- so the issue stream is not the limiter either;
      // one elected arrive per splitter warp + releasing the TMEM slot's first channel half early measured 5 % SLOWER.  With every
      // load, convert and 2/3 of the MMAs ablated the k-block period is still ~600 cycles: the 2-deep TMEM operand ring's
      // round trip (commit -> splitter wake -> tcgen05.st -> wait::st -> arrive -> issuer wake) bounds the loop; a deeper ring
      // needs TMEM columns that D_main[2] + D_small + A[2] already use up at BN = 128.  Two issuing warps alternating k-blocks
      // behind an mbarrier order token (tcgen05 fences on both sides) also measured neutral -- 175.7 vs 174.5 us -- and is not kept.)
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
      uint32_t kbt = 0, ct = 0, ut = 0;
      uint32_t sb = 0;
      const uint32_t d_small = tb + (uint32_t)F_TMEM_DSMALL;
      const uint32_t blo0 = ((smem_u32(smem_b) & 0x3FFFFu) >> 4) | (1u << 16);   // low descriptor word of stage 0's hi plane (LBO field = 1)
      constexpr uint32_t kDescHi = (uint32_t)(1024u >> 4) | (1u << 14) | (2u << 29);   // SBO = 1024 B, version 1, SWIZZLE_128B
      constexpr uint32_t kStageStep = (uint32_t)kBStage >> 4, kPlaneStep = (uint32_t)kBTile >> 4;
      const int kpc = p.kb_per_chunk;
      uint32_t r6 = 0, pr = 0;
      for (int u = blockIdx.x; u < p.total_units; u += gridDim.x, ++ut) {
        const Unit t = decode_unit(p, u, num_kb_total);
        const int nkb = __shfl_sync(0xffffffffu, t.num_kb, 0);
        int in_chunk = 0;
        if (!X1) MBAR_WAIT(small_empty, (ut & 1u) ^ 1u, 7, kbt);                        // D_small of the previous unit has been read
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb, ++kbt) {
          const uint32_t b = ct & 1u;
          if (in_chunk == 0) MBAR_WAIT(&acc_empty[b], ((ct >> 1) & 1u) ^ 1u, 6, kbt);   // D_main[b]'s previous chunk has been drained
          const uint32_t st = kbt & (uint32_t)(F_ST - 1);
          if (lane == 0) FRCNN_TRACE(4, kbt);
          MBAR_WAIT(&ready[r6], pr, 8, kbt);                                             // A planes stored AND B tiles landed
          tc_fence_after();
          if (lane == 0) FRCNN_TRACE(5, kbt);
          const uint32_t bl = blo0 + sb * kStageStep;
          const uint32_t a0 = tb + (uint32_t)F_TMEM_A0 + st * 64u;
          const uint32_t d_main = tb + b * 128u;
          const bool last = (in_chunk + 1 == kpc) || (kb + 1 == nkb);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < F_BK / 16; ++j) {
              // B: 16 fp16 = 32 B inside the 128-byte swizzle row = +2 in the address field; A: 32-channel half, then 8 TMEM columns
              const uint32_t bh_j = bl + 2u * j, bl_j = bl + kPlaneStep + 2u * j;
              const uint32_t a_hi = a0 + (uint32_t)((j >> 1) * 32 + (j & 1) * 8), a_lo = a_hi + 16u;
              if (j == 0) {
                if (!X1) {
                  umma_f16_ts_lo(d_small, a_lo, bh_j, kDescHi, kIdesc, kb > 0 ? 1u : 0u);
                  umma_f16_ts_acc(d_small, a_hi, bl_j, kDescHi, kIdesc);
                }
                umma_f16_ts_lo(d_main, a_hi, bh_j, kDescHi, kIdesc, in_chunk > 0 ? 1u : 0u);
              } else {
                if (!X1) {
                  umma_f16_ts_acc(d_small, a_lo, bh_j, kDescHi, kIdesc);
                  umma_f16_ts_acc(d_small, a_hi, bl_j, kDescHi, kIdesc);
                }
                umma_f16_ts_acc(d_main, a_hi, bh_j, kDescHi, kIdesc);
              }
            }
            umma_commit(&ta_empty[st]);
            umma_commit(&b_empty[sb]);
            if (last) umma_commit(&acc_full[b]);
          }
          __syncwarp();
          if (lane == 0) FRCNN_TRACE(6, kbt);
          if (last) { in_chunk = 0; ++ct; } else ++in_chunk;
          if (++sb == F_SB) sb = 0;
          if (++r6 == F_RDY) { r6 = 0; pr ^= 1u; }
        }
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 18) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// Second pass for split tiles: out = act((sum_z ws[slot][z]) * scale + shift (+ residual)), z summed in index order
// (deterministic).  One block per (tail tile, group of 256/(BN/4) rows); thread = (row, 4 channels).
template <int BN>
__global__ void __launch_bounds__(256)
tail_reduce_kernel(const ConvKernelParams p) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int RPB = 256 / (BN / 4);                 // rows per block: one (row, 4-channel group) per thread
  constexpr int GROUPS = BLOCK_M / RPB;
  const int slot = blockIdx.x / GROUPS, rgroup = blockIdx.x % GROUPS;
  const int tile = p.n_full + slot;
  const int mt = p.raster_n ? tile / p.n_tiles : tile % p.m_tiles, nblk = p.raster_n ? tile % p.n_tiles : tile / p.m_tiles;
  const int tile_w = mt % p.tiles_w, tile_h = (mt / p.tiles_w) % p.tiles_h, tile_n = mt / (p.tiles_w * p.tiles_h);
  const int rows_img = p.th * p.tw;
  constexpr int C4 = BN / 4;
  static_assert(256 % C4 == 0, "each thread keeps one fixed channel group");
  const float* base = p.ws + (size_t)slot * p.splits * (size_t)(BLOCK_M * BN);
  const bool vec_ok = (p.cout & 3) == 0;
  const int cg = threadIdx.x % C4;
  const int c = nblk * BN + cg * 4;
  if (c >= p.cout) return;
  const float4 sc4 = __ldg(reinterpret_cast<const float4*>(p.scale + c)), sh4 = __ldg(reinterpret_cast<const float4*>(p.shift + c));   // padded vectors
  const float sc[4] = {sc4.x, sc4.y, sc4.z, sc4.w}, sh[4] = {sh4.x, sh4.y, sh4.z, sh4.w};
  {
    const int row = rgroup * RPB + threadIdx.x / C4;
    const int dn = row / rows_img, rem = row % rows_img;
    const int n = tile_n * p.tn + dn, h = tile_h * p.th + rem / p.tw, w = tile_w * p.tw + rem % p.tw;
    if (row >= p.tn * rows_img || n >= p.nimg || h >= p.ho || w >= p.wo) return;
    const size_t o = ((((size_t)n * p.ho + h) * p.wo + w)) * p.cout + c;
    float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.residual) {
      if (vec_ok) rv = __ldg(reinterpret_cast<const float4*>(p.residual + o));
      else { float t[4] = {0.f, 0.f, 0.f, 0.f}; for (int e = 0; e < 4; ++e) if (c + e < p.cout) t[e] = __ldg(p.residual + o + e); rv = make_float4(t[0], t[1], t[2], t[3]); }
    }
    float4 a = __ldg(reinterpret_cast<const float4*>(base + (size_t)row * BN) + cg);
    for (int z = 1; z < p.splits; ++z) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(base + ((size_t)z * BLOCK_M + row) * BN) + cg);
      a.x = __fadd_rn(a.x, b.x); a.y = __fadd_rn(a.y, b.y); a.z = __fadd_rn(a.z, b.z); a.w = __fadd_rn(a.w, b.w);
    }
    float y[4] = {a.x, a.y, a.z, a.w};
    const float res[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v = y[e];
      v = __fadd_rn(__fmul_rn(v, sc[e]), sh[e]);
      if (p.residual) v = __fadd_rn(v, res[e]);
      if (p.act == FRCNN_ACT_RELU) v = fmaxf(v, 0.f);
      else if (p.act == FRCNN_ACT_RELU6) v = fminf(fmaxf(v, 0.f), 6.f);
      y[e] = v;
    }
    if (vec_ok) *reinterpret_cast<float4*>(p.out + o) = make_float4(y[0], y[1], y[2], y[3]);
    else for (int e = 0; e < 4; ++e) if (c + e < p.cout) p.out[o + e] = y[e];
  }
}

// plan creation: the epilogue's per-channel vectors, padded to the tile grid (no bounds tests in the kernel)
__global__ void prep_epilogue_vectors_kernel(const float* scale, const float* shift, float out_mult, int cout, int padded,
                                             float* eff_scale, float* eff_shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= padded) return;
  const float sc = (c < cout && scale) ? scale[c] : 1.f;
  eff_scale[c] = __fmul_rn(sc, out_mult);                  // exact: out_mult is a power of two
  eff_shift[c] = (c < cout && shift) ? shift[c] : 0.f;
}

// ---------------------------------------------------------------------------------------------------
// host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

static int encode_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box, const uint32_t* estr, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                      CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return ERR_DRIVER_ENTRY; }
  cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = estr[i]; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = fn(m, dtype, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu,%llu,%llu] box=[%u,%u,%u,%u]", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], rank > 2 ? (unsigned long long)dims[2] : 0ull,
              rank > 3 ? (unsigned long long)dims[3] : 0ull, box[0], box[1], rank > 2 ? box[2] : 0u, rank > 3 ? box[3] : 0u);
    return ERR_CUDA;
  }
  return OK;
}

}  // namespace frcnn

using namespace frcnn;

struct frcnn_conv_plan {
  CUtensorMap tmA, tmBhi, tmBlo;
  ConvKernelParams kp;
  int block_n, stages, smem;
  int impl;                // FRCNN_CONV_F16X3 | FRCNN_CONV_TF32X3 | FRCNN_CONV_F16X1
  dim3 grid;
  int n_tail;
  float* ws;               // owned workspace of the split tiles 
  float* eff;              // owned epilogue vectors: scale * out_mult | shift, each padded to n_tiles * block_n
};

// choose the tile of output pixels (tn x th x tw <= 128) that needs the fewest tiles
static void choose_tile(int n, int ho, int wo, int stride, int* tn, int* th, int* tw) {
  long best_tiles = -1; int bn = 1, bh = 1, bw = 1; int best_rows = 0;
  const int lim = 256 / stride;
  for (int a = 1; a <= n && a <= BLOCK_M; ++a)
    for (int b = 1; b <= ho && a * b <= BLOCK_M && b <= lim; ++b) {
      int c = BLOCK_M / (a * b);
      if (c > wo) c = wo;
      if (c > lim) c = lim;
      if (c < 1) continue;
      // shrink c to the smallest width giving the same tile count (less garbage rows)
      int tiles_w = cdiv(wo, c);
      c = cdiv(wo, tiles_w);
      long tiles = (long)cdiv(n, a) * cdiv(ho, b) * tiles_w;
      int rows = a * b * c;
      if (best_tiles < 0 || tiles < best_tiles || (tiles == best_tiles && rows < best_rows)) {
        best_tiles = tiles; bn = a; bh = b; bw = c; best_rows = rows;
      }
    }
  *tn = bn; *th = bh; *tw = bw;
}

// FRCNN_NO_PDL=1 disables programmatic dependent launch (debug / A-B measurements)
static bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("FRCNN_NO_PDL"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

template <int BN>
static int launch(const frcnn_conv_plan* p, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    FRCNN_CUDA(cudaFuncSetAttribute(conv_gemm_tf32x3_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes<BN>()));
    attr_done = true;
  }
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  const bool pdl = pdl_enabled();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = p->grid; cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = smem_bytes<BN>(); cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  FRCNN_CUDA(cudaLaunchKernelEx(&cfg, conv_gemm_tf32x3_kernel<BN>, p->tmA, p->tmBhi, p->tmBlo, p->kp));
  if (p->n_tail > 0) {
    cudaLaunchConfig_t rc{};
    rc.gridDim = dim3((unsigned)(p->n_tail * (BLOCK_M / (256 / (BN / 4))))); rc.blockDim = dim3(256); rc.dynamicSmemBytes = 0; rc.stream = st;
    rc.attrs = attr; rc.numAttrs = pdl ? 1 : 0;
    FRCNN_CUDA(cudaLaunchKernelEx(&rc, tail_reduce_kernel<BN>, p->kp));
  }
  return OK;
}

template <int BN, bool X1>
static int launch_f16(const frcnn_conv_plan* p, cudaStream_t st) {
  static bool attr_done = false;
  if (!attr_done) {
    FRCNN_CUDA(cudaFuncSetAttribute(conv_gemm_f16x3_kernel<BN, X1>, cudaFuncAttributeMaxDynamicSharedMemorySize, f_smem_bytes<BN>()));
    attr_done = true;
  }
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  const bool pdl = pdl_enabled();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = p->grid; cfg.blockDim = dim3(F_THREADS); cfg.dynamicSmemBytes = f_smem_bytes<BN>(); cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  FRCNN_CUDA(cudaLaunchKernelEx(&cfg, conv_gemm_f16x3_kernel<BN, X1>, p->tmA, p->tmBhi, p->tmBlo, p->kp));
  if (p->n_tail > 0) {
    cudaLaunchConfig_t rc{};
    rc.gridDim = dim3((unsigned)(p->n_tail * (BLOCK_M / (256 / (BN / 4))))); rc.blockDim = dim3(256); rc.dynamicSmemBytes = 0; rc.stream = st;
    rc.attrs = attr; rc.numAttrs = pdl ? 1 : 0;
    FRCNN_CUDA(cudaLaunchKernelEx(&rc, tail_reduce_kernel<BN>, p->kp));
  }
  return OK;
}

// Host-side work decomposition of one layer (no CUDA calls: unit-testable on a CPU box through frcnn_conv_plan_geometry).
struct Geometry {
  int n, h, w, ho, wo;           // after flattening 1x1/stride-1 layers to one row of n*h*w pixels
  int tn, th, tw, tiles_w, tiles_h, tiles_n;
  long m_tiles;
  int num_kb, bn, n_tiles, kpc;
  long tiles, n_tail;
  int splits, kbs;
  long total_units;
  int grid;
  int raster_n;
};

static int decide_geometry(const frcnn_conv_desc* d, int sms, Geometry* g) {
  FRCNN_REQUIRE(d->cin > 0 && d->cin % BLOCK_K == 0, "cin=%d must be a positive multiple of 32", d->cin);
  FRCNN_REQUIRE(d->kh >= 1 && d->kw >= 1 && d->stride >= 1 && d->stride <= 8, "bad filter geometry");
  FRCNN_REQUIRE(d->n > 0 && d->h > 0 && d->w > 0 && d->ho > 0 && d->wo > 0 && d->cout > 0, "bad shape");
  FRCNN_REQUIRE(sms > 0, "bad SM count");
  g->n = d->n; g->h = d->h; g->w = d->w; g->ho = d->ho; g->wo = d->wo;
  const bool pointwise = d->kh == 1 && d->kw == 1 && d->stride == 1 && d->pad_t == 0 && d->pad_l == 0 && g->ho == g->h && g->wo == g->w;
  if (pointwise) {  // flatten all pixels into one row of "width" n*h*w: perfect 128-row tiles
    g->w = g->wo = g->n * g->h * g->w; g->n = 1; g->h = g->ho = 1;
  }
  choose_tile(g->n, g->ho, g->wo, d->stride, &g->tn, &g->th, &g->tw);
  g->tiles_w = cdiv(g->wo, g->tw); g->tiles_h = cdiv(g->ho, g->th); g->tiles_n = cdiv(g->n, g->tn);
  g->m_tiles = (long)g->tiles_w * g->tiles_h * g->tiles_n;
  const bool f16 = d->impl != FRCNN_CONV_TF32X3;
  const int ks = f16 ? 2 : 1;                                   // 32-channel blocks per k-block (f16x3: 64-wide k-blocks)
  g->num_kb = cdiv(d->kh * d->kw * d->cin / BLOCK_K, ks);
  g->kpc = d->kb_per_chunk > 0 ? d->kb_per_chunk : 8 / ks;
  int bn = d->block_n;
  if (bn == 0) {
    long best = -1;
    const int cands[2] = {128, 64};
    for (int i = 0; i < 2; ++i) {
      const int c = cands[i];
      if (c > 64 && c / 2 >= d->cout) continue;        // tile mostly empty
      const long ctas = g->m_tiles * cdiv(d->cout, c);
      const long waves = (ctas + sms - 1) / sms;
      // measured (profiles/r01): a k-block costs about the same whatever block_n is (the 128-row A operand dominates for
      // N <= 128), plus a fixed per-unit cost => fewest rounds wins, widest tile on ties
      const long cost = f16 ? waves * (g->num_kb * 900L + 4000L) : waves * (g->num_kb * 1400L + 6000L);
      if (best < 0 || cost < best) { best = cost; bn = c; }
    }
  }
  FRCNN_REQUIRE(bn == 64 || bn == 128, "block_n must be 64 or 128");
  g->bn = bn;
  g->n_tiles = cdiv(d->cout, bn);
  g->tiles = g->m_tiles * g->n_tiles;
  FRCNN_REQUIRE(g->tiles <= 0x3fffffffL, "too many tiles");
  // ---- whole tiles + K-split tail (see ConvKernelParams) ---------------------------------------------------------------
  long n_tail = 0; int splits = 1;
  const int num_kb = g->num_kb;
  const int max_split = num_kb * ks / 8 < 8 ? num_kb * ks / 8 : 8;   // >= 8 32-wide k-blocks (one chunk) per split, at most 8 splits
  if (d->split_k > 1) {                                         // forced: every tile is split
    n_tail = g->tiles; splits = d->split_k;
  } else if (d->split_k == 0 && max_split >= 2) {
    const long rem = g->tiles % sms;
    // measured (r01): a split unit still pays ~7 us of per-unit overhead and the reduce pass ~10 us, so the ragged round is
    // only worth splitting when the K loop is long (>= 48 k-blocks); small layers gain from 16 k-blocks on.
    if (g->tiles <= sms / 2) { if (num_kb * ks >= 16) { n_tail = g->tiles; splits = (int)(sms / g->tiles); } }   // layer too small to fill the GPU
    else if (g->tiles > sms && rem > 0 && rem <= sms / 2 && num_kb * ks >= 48) { n_tail = rem; splits = (int)(sms / rem); }   // ragged last round
    if (splits > max_split) splits = max_split;
    if (splits < 2) { n_tail = 0; splits = 1; }
  }
  int kbs = cdiv(num_kb, splits);                              // (a unit's last chunk may be shorter than kb_per_chunk)
  splits = cdiv(num_kb, kbs);
  if (splits < 2 || (d->cout & 3) != 0) { n_tail = 0; splits = 1; kbs = num_kb; }   // tail_reduce_kernel reads the padded epilogue vectors as float4
  FRCNN_REQUIRE(splits <= 64, "bad split_k");
  g->n_tail = n_tail; g->splits = splits; g->kbs = kbs;
  g->total_units = (g->tiles - n_tail) + n_tail * splits;
  FRCNN_REQUIRE(g->total_units <= 0x7fffffffL, "too many work units");
  g->grid = (int)(g->total_units < sms ? g->total_units : sms);   // persistent: one CTA per SM walks the units
  {
    const char* e = getenv("FRCNN_CONV_RASTER");          // development override: m | n
    const double a_bytes = (double)d->n * d->h * d->w * d->cin * 4.0, b_bytes = (double)d->cout * d->kh * d->kw * d->cin * 4.0;
    g->raster_n = (e && (e[0] == 'm' || e[0] == 'n')) ? (e[0] == 'n') : (a_bytes > b_bytes && g->n_tiles > 1);
  }
  return OK;
}

extern "C" int frcnn_conv_plan_geometry(const frcnn_conv_desc* d, int sm_count, int* out16) {
  FRCNN_REQUIRE(d && out16, "null argument");
  Geometry g;
  int rc = decide_geometry(d, sm_count, &g);
  if (rc) return rc;
  const int v[16] = {g.bn, g.tn, g.th, g.tw, (int)g.m_tiles, g.n_tiles, (int)g.tiles, (int)g.n_tail, g.splits, g.kbs,
                     (int)g.total_units, g.grid, g.num_kb, g.kpc, g.tiles_h, g.tiles_w};
  for (int i = 0; i < 16; ++i) out16[i] = v[i];
  return OK;
}

extern "C" int frcnn_conv_plan_create(frcnn_conv_plan** out, const frcnn_conv_desc* d) {
  FRCNN_REQUIRE(out && d, "null argument");
  FRCNN_REQUIRE(d->in_dev && d->w_hi_dev && d->w_lo_dev && d->out_dev, "null device pointer");
  int sms = 148;
  { int dev = 0; cudaDeviceProp pr; if (cudaGetDevice(&dev) == cudaSuccess && cudaGetDeviceProperties(&pr, dev) == cudaSuccess && pr.multiProcessorCount > 0) sms = pr.multiProcessorCount; }
  Geometry g;
  int grc = decide_geometry(d, sms, &g);
  if (grc) return grc;
  frcnn_conv_plan* p = (frcnn_conv_plan*)aligned_alloc(64, (sizeof(frcnn_conv_plan) + 63) / 64 * 64);
  if (!p) { set_error("out of host memory"); return ERR_ARG; }
  memset(p, 0, sizeof(*p));
  const int bn = g.bn;
  // A: NHWC activations as a rank-4 tensor {C, W, H, N}; traversal stride = conv stride on W and H
  {
    uint64_t dims[4] = {(uint64_t)d->cin, (uint64_t)g.w, (uint64_t)g.h, (uint64_t)g.n};
    uint64_t strides[3] = {(uint64_t)d->cin * 4, (uint64_t)g.w * d->cin * 4, (uint64_t)g.h * g.w * d->cin * 4};
    uint32_t box[4] = {(uint32_t)BLOCK_K, (uint32_t)(g.tw * d->stride), (uint32_t)(g.th * d->stride), (uint32_t)g.tn};
    uint32_t es[4] = {1, (uint32_t)d->stride, (uint32_t)d->stride, 1};
    int rc = encode_map(&p->tmA, d->in_dev, 4, dims, strides, box, es);
    if (rc) { free(p); return rc; }
  }
  const bool f16 = d->impl != FRCNN_CONV_TF32X3;
  {
    const uint64_t ktot = (uint64_t)d->kh * d->kw * d->cin;
    uint64_t dims[2] = {ktot, (uint64_t)d->cout};
    uint64_t strides[1] = {ktot * (f16 ? 2 : 4)};
    uint32_t box[2] = {(uint32_t)(f16 ? F_BK : BLOCK_K), (uint32_t)bn};   // 128-byte rows either way
    uint32_t es[2] = {1, 1};
    const CUtensorMapDataType dt = f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B;
    int rc = encode_map(&p->tmBhi, d->w_hi_dev, 2, dims, strides, box, es, dt, sw);
    if (!rc) rc = encode_map(&p->tmBlo, d->w_lo_dev, 2, dims, strides, box, es, dt, sw);
    if (rc) { free(p); return rc; }
  }
  ConvKernelParams& k = p->kp;
  k.out = d->out_dev; k.residual = d->residual_dev;
  k.cout = d->cout; k.ho = g.ho; k.wo = g.wo; k.nimg = g.n;
  k.tn = g.tn; k.th = g.th; k.tw = g.tw; k.tiles_h = g.tiles_h; k.tiles_w = g.tiles_w;
  k.kh = d->kh; k.kw = d->kw; k.cin = d->cin; k.stride = d->stride; k.pad_t = d->pad_t; k.pad_l = d->pad_l;
  k.act = d->act;
  k.a_box_bytes = g.tn * g.th * g.tw * BLOCK_K * 4;
  k.kb_per_chunk = g.kpc;
  k.trace = nullptr;
  { const char* e = getenv("FRCNN_CONV_DBG"); k.dbg = e ? atoi(e) : 0; }
  k.num_kb_total = g.num_kb;
  k.m_tiles = (int)g.m_tiles; k.n_tiles = g.n_tiles;
  k.kb_per_split = g.kbs; k.splits = g.splits; k.n_full = (int)(g.tiles - g.n_tail);
  k.total_units = (int)g.total_units;
  k.raster_n = g.raster_n;
  k.ws = nullptr; p->ws = nullptr; p->eff = nullptr; p->n_tail = (int)g.n_tail;
  {
    // NOTE: the vectors are snapshots of scale_dev / shift_dev taken now (they are weights: constant after load)
    const int padded = g.n_tiles * bn;
    const float om = f16 ? (d->out_mult != 0.f ? d->out_mult : 1.f) : 1.f;
    cudaError_t e = cudaMalloc(&p->eff, (size_t)2 * padded * sizeof(float));
    if (e != cudaSuccess) { free(p); return cuda_fail(e, "epilogue vectors", __FILE__, __LINE__); }
    prep_epilogue_vectors_kernel<<<cdiv(padded, 256), 256>>>(d->scale_dev, d->shift_dev, om, d->cout, padded, p->eff, p->eff + padded);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cudaFree(p->eff); free(p); return cuda_fail(e, "prep_epilogue_vectors", __FILE__, __LINE__); }
    k.scale = p->eff; k.shift = p->eff + padded;
  }
  if (g.n_tail > 0) {
    cudaError_t e = cudaMalloc(&p->ws, (size_t)g.n_tail * g.splits * BLOCK_M * bn * sizeof(float));
    if (e != cudaSuccess) { cudaFree(p->eff); free(p); return cuda_fail(e, "split-tile workspace", __FILE__, __LINE__); }
    k.ws = p->ws;
  }
  p->grid = dim3((unsigned)g.grid, 1, 1);
  p->block_n = bn;
  p->impl = f16 ? (d->impl == FRCNN_CONV_F16X1 ? FRCNN_CONV_F16X1 : FRCNN_CONV_F16X3) : FRCNN_CONV_TF32X3;
  p->stages = f16 ? F_SA : RING;
  p->smem = f16 ? (bn == 128 ? f_smem_bytes<128>() : f_smem_bytes<64>()) : (bn == 128 ? smem_bytes<128>() : smem_bytes<64>());
  *out = p;
  return OK;
}

extern "C" int frcnn_conv_plan_run(const frcnn_conv_plan* p, void* stream) {
  FRCNN_REQUIRE(p, "null plan");
  cudaStream_t st = (cudaStream_t)stream;
  if (p->impl == FRCNN_CONV_F16X3) return p->block_n == 128 ? launch_f16<128, false>(p, st) : launch_f16<64, false>(p, st);
  if (p->impl == FRCNN_CONV_F16X1) return p->block_n == 128 ? launch_f16<128, true>(p, st) : launch_f16<64, true>(p, st);
  return p->block_n == 128 ? launch<128>(p, st) : launch<64>(p, st);
}

extern "C" int frcnn_conv_plan_info(const frcnn_conv_plan* p, int* block_n, int* tile_n, int* tile_h, int* tile_w,
                                    int* grid_m, int* grid_n, int* stages, int* smem) {
  FRCNN_REQUIRE(p, "null plan");
  if (block_n) *block_n = p->block_n;
  if (tile_n) *tile_n = p->kp.tn;
  if (tile_h) *tile_h = p->kp.th;
  if (tile_w) *tile_w = p->kp.tw;
  if (grid_m) *grid_m = p->kp.m_tiles;
  if (grid_n) *grid_n = p->kp.n_tiles;
  if (stages) *stages = p->n_tail > 0 ? p->kp.splits : 1;   /* "splits" of the tail tiles */
  if (smem) *smem = p->smem;
  return OK;
}

extern "C" int frcnn_debug_watchdog(unsigned int* out16, int reset) {
  FRCNN_REQUIRE(out16, "null argument");
#ifdef FRCNN_WATCHDOG
  FRCNN_CUDA(cudaMemcpyFromSymbol(out16, g_watchdog, 16 * sizeof(unsigned int)));
  if (reset) { unsigned int z[16] = {0}; FRCNN_CUDA(cudaMemcpyToSymbol(g_watchdog, z, sizeof(z))); }
  return OK;
#else
  (void)reset;
  for (int i = 0; i < 16; ++i) out16[i] = 0;
  out16[15] = 0xffffffffu;   // "not a watchdog build"
  return OK;
#endif
}

extern "C" int frcnn_conv_plan_set_trace(frcnn_conv_plan* p, long long* trace_dev) {
  FRCNN_REQUIRE(p, "null plan");
  p->kp.trace = trace_dev;
  return OK;
}

extern "C" void frcnn_conv_plan_destroy(frcnn_conv_plan* p) {
  if (p && p->ws) cudaFree(p->ws);
  if (p && p->eff) cudaFree(p->eff);
  free(p);
}
