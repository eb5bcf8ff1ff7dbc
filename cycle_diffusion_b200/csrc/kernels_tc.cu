// kernels_tc.cu -- tcgen05 / TMEM / TMA back end for the dense contractions (conv3x3, conv1x1 / Linear, batched attention products):
// fp32-faithful products from three tensor-core terms.
//
// Why three terms: the path's acceptance bar is parity with the reference's fp32 CPU path (|d pixel| <= 1e-3 through 50-250 sequential
// U-Net calls with a 1/sigma_t amplification), which plain TF32/BF16/FP16 tensor-core math cannot hold (SURVEY.md section 7; the
// single-term fast path ends at 6e-3).  Every fp32 operand is split into hi + lo and the product is accumulated as
// lo*hi + hi*lo + hi*hi in the fp32 TMEM accumulator (the dropped lo*lo term is < 2^-22 relative):
//   MODE_H16 / MODE_H16X2 (default)  x' = x * 2^e (e from the tensor's tracked range), hi = fp16(x'), lo = fp16(x' - hi): three
//                         tcgen05.mma.kind::f16 per 16-wide K step, exact power-of-two rescale in the epilogue;
//   MODE_TS / MODE_SS     hi = rn_tf32(x), lo = rn_tf32(x - hi): three kind::tf32 per 8-wide K step (round-1 scheme: --mma 3, and the
//                         activation x activation products, where neither operand has pre-split planes).
//
// Tensor-core accumulation truncates (measured: the error of one long accumulation grows linearly with K, 5.8e-5 relative at
// K = 11520), so the K loop is cut into chunks of 256 elements (one chunk if K <= 512): each chunk accumulates in one of two TMEM
// buffers and is drained by the epilogue warps into fp32 registers with round-to-nearest adds while the next chunk already runs in the
// other buffer.  Measured error after both fixes: ~1.3e-6 relative, independent of K.
//
// Persistent kernel, one CTA (MODE_H16X2: one 2-CTA cluster = 256 rows, cta_group::2) per SM walks work items (tile, K split) of
// 128 (256) rows x w <= 128 columns, K in 128-byte blocks.  640 threads = 5 warpgroups with setmaxnreg budgets:
//   warp 0      TMA producer (cp.async.bulk.tensor, 128B-swizzled smem).  A is a 2D [M,K] row matrix (dense / 1x1 conv / Linear,
//               optionally two channel-concatenated sources), or for conv3x3 a 4D box of the NHWC activation -- per tap {32 ch, bw, bh,
//               bn} shifted by (dy-1, dx-1), or on the HALO schedule the (bw+2) x (bh+2) pixel halo of a 64-channel block fetched
//               once: TMA's out-of-bounds zero fill *is* the conv's zero padding, im2col is never materialised; or (batched mode) 4D
//               maps over (k, head, row, batch) for the attention contractions.  B: pre-split weight planes (fp16 or TF32) by TMA.
//   warp 1      MMA issuer: one lane issues the three-term MMAs of a K block (A operand from TMEM), tcgen05.commit hands the stage
//               back (pair: multicast to both CTAs' barriers).  Warps 2-3 idle (they only return their registers).
//   warps 4-11  split warps: raw fp32 A rows (or, halo schedule, the halo converted once in place into fp16 hi / lo planes and then
//               copied per tap) -> hi / lo -> tcgen05.st into the TMEM A ring.
//   warps 12-19 drain + epilogue (two warps per TMEM lane quadrant, 32 rows x 64 columns each): tcgen05.ld per chunk -> RN add into
//               64 fp32 registers per thread; then alpha / rescale, +bias, +per-sample row vector (timestep embedding), GEGLU,
//               +residual, range / GroupNorm side outputs, and the store: TMA boxes staged in the map's swizzle for the dense layers
//               (template parameter EPI), a swizzled smem transpose with 128-bit global stores otherwise.
// DESIGN.md 5.1 has the measured history of each of these choices (profiles/r01_*, r02_*).
#include <algorithm>

#include <mutex>
#include <array>
#include <map>
#include <unordered_map>
#include <vector>
#include <cstdlib>
#include <cmath>
#include <type_traits>

#include <cuda_fp16.h>

#include "tc_common.cuh"

namespace cdx {
namespace {

using namespace tc;

constexpr int TBM = 128, TBN = 128, TBK = 32;
constexpr double CDX_H16_KC0 = 640.0, CDX_H16_KC1 = 4.2;   // planner cost of one 64-k stage of the fp16-split kernel (cycles)
constexpr int TILE_BYTES = TBM * TBK * 4;          // 16 KB
constexpr int HALO_PLANE_1CTA = 24 * 1024;        // one 32-channel plane of a conv3x3 halo box (<= 192 pixels x 128 B)
constexpr int HALO_PLANE_PAIR = 25 * 1024;        // pair kernel (its B ring is half the size): 200 pixels = the two 10 x 10 halos of an 8 x 8 tile
constexpr int NUM_SPLIT_WARPS = 8;               // two per TMEM lane quadrant (MODE_H16: one per 32-k sub-block of a stage)
constexpr int NUM_EPI_WARPS = 8;
constexpr int FIRST_SPLIT_WARP = 4, FIRST_EPI_WARP = FIRST_SPLIT_WARP + NUM_SPLIT_WARPS;
constexpr int TC_THREADS = (FIRST_EPI_WARP + NUM_EPI_WARPS) * 32;      // 20 warps = 5 warpgroups (setmaxnreg is per warpgroup)

// Operand path of the kernel (template parameter MODE):
//   MODE_SS   both operands raw fp32 in smem, split in smem into TF32 hi / lo (generic: B may be an activation)
//   MODE_TS   B = pre-split TF32 planes by TMA, A split by the split warps into TMEM (3 x kind::tf32 per 8-wide K chunk)
//   MODE_H16  fp16 split at the kind::f16 rate (3 x kind::f16 per 16-wide K chunk = half the tensor time and half the
//             B bytes of MODE_TS): x' = x * 2^e (e from the tensor's tracked max: |x'| < 2^15), hi = fp16(x'), lo = fp16(x' - hi).
//             hi + lo carries >= 22 significant bits of x' down to |x'| = 2^-3 and an absolute error <= 2^-25 below that
//             (2^-40 of the tensor's max), products of 11-bit significands are exact in the fp32 accumulator, and the result is
//             rescaled by the exact power of two 2^-(ea + eb) in the epilogue.  B planes are pre-scaled fp16 in HBM.
//   MODE_H16X2  MODE_H16 on CTA pairs (cta_group::2): a 2-CTA cluster owns a 256-row tile, each CTA splits its own 128 rows into its
//             own TMEM and holds HALF of the B rows in its smem; the leader issues M = 256 MMAs over both.  B bytes per CTA and stage
//             halve (ingress, smem fill, tensor-core operand fetch), which buys a 4th pipeline stage in the same shared memory
enum { MODE_SS = 0, MODE_TS = 1, MODE_H16 = 2, MODE_H16X2 = 3 };

template <int MODE>
struct Cfg {
  static constexpr bool TS = MODE != MODE_SS;
  static constexpr bool CG2 = MODE == MODE_H16X2;
  static constexpr bool H16 = MODE == MODE_H16 || CG2;
  static constexpr int BK = H16 ? 64 : 32;         // K elements per pipeline stage
  static constexpr int KCHUNK = 256 / BK;          // stages per TMEM accumulation chunk (256 K elements)
  static constexpr int STAGES = (MODE == MODE_TS || CG2) ? 4 : 3;
  static constexpr int B_PLANE = CG2 ? TILE_BYTES / 2 : TILE_BYTES;      // smem bytes of one B plane of a stage (CG2: half the rows)
  static constexpr int HALO_PLANE = CG2 ? HALO_PLANE_PAIR : HALO_PLANE_1CTA;
  // SS: A_hi, A_lo, B_hi, B_lo ; TS: A_raw, B_hi, B_lo ; H16: A_raw(k 0..31), A_raw(k 32..63), B_hi, B_lo (fp16, 128 B rows)
  static constexpr int STAGE_BYTES = MODE == MODE_TS ? 3 * TILE_BYTES : 2 * TILE_BYTES + 2 * B_PLANE;
  static constexpr int TMEM_COLS = TS ? 512 : 256;
  static constexpr int A_COL0 = 256;               // TS / H16: A stage s lives at columns A_COL0 + 64 s (hi) / + 32 (lo)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 2048 /*barriers + bias staging*/ + 32768 /*epilogue transpose: 8 warps x 4 KB*/ + 1024 /*alignment slack*/;
};

struct TcParams {
  int M, N, K;
  int mode;                 // 0 dense, 1 conv3x3 (stride 1, pad 1), 2 batched dense
  int C1, C2;               // dense: channels of source 1 / 2 (k-blocks never straddle: C1 % 32 == 0 when C2 > 0)
  int Cin;                  // conv: input channels (multiple of 32)
  int H, W, B;              // conv: spatial size (in == out) and batch
  int bw, bh, bn;           // conv: pixel box of one M tile (bw*bh*bn == 128)
  int tiles_x, tiles_y;     // conv: tiles per row / column
  int cstride, cpad;        // conv: stride (1 or 2: TMA element traversal stride) and low-side padding
  // MODE_H16 conv3x3 "halo" schedule (stride 1, pad 1, Cin % 64 == 0): the K loop runs (64-channel block, tap) instead of
  // (tap, channel block); the (bw+2) x (bh+2) x bn pixel halo of a 64-channel block is fetched ONCE (two 32-channel TMA boxes,
  // OOB zero fill = padding) and the split warps read all nine shifted taps from it, so the activation crosses L2 -> SM once
  // per tile and channel block instead of nine times (A ingress per stage 32 KB -> ~5 KB; the kernel was L2->SM bound)
  int halo;
  // halo schedule, optional: the A operand is silu?(x * a + o), (a, o) = gn_ab[b * Cin + c] (GroupNorm of the input applied during the
  // halo conversion; out-of-image pixels stay 0).  Needs bn == 1.  C1 < Cin: channels >= C1 come from the second source (mapA2)
  const float2* gn_ab; int gn_silu;
  float* C; int ldc;
  // dense mode, final epilogue: tiles leave through TMA (mapC / mapClo: 32 x 32 float boxes of C / C_lo, mapR: of the residual;
  // map*16: 16-column boxes for the tail of a ragged tile); the epilogue warps stage column blocks in the map's swizzle and one lane issues the bulk store (no per-row address arithmetic,
  // predicates or 16-byte global stores on the warps that also drain TMEM)
  int epi_tma;
  float* C_lo;              // optional: C <- rn_tf32(result), C_lo <- rn_tf32(result - hi)
  float* Ct_hi; float* Ct_lo; int t_col0; long long ldt;   // optional transposed plane output for columns >= t_col0
  const float* bias;
  const float* rowvec; int ld_rowvec; int rows_per_batch;
  const float* residual; int ldr;
  float alpha;
  int geglu;                    // N tiles hold [32 value | 32 gate] column blocks: store value * gelu(gate) to [M, N/2]
  int out_nchw, rows_per_img;   // store C as [B, N, rows_per_img] (final conv of a network, reference NCHW layout)
  // mode 2 (blockIdx.z = zb*heads + zh): 4D maps, coordinate recipe per operand
  int heads;
  int a_code[4], b_code[4];   // per map dim: 0 -> k0, 1 -> row0, 2 -> zh, 3 -> zb, 4 -> 0
  int a_rowoff_h, b_rowoff_h; // row0 += zh * rowoff (heads packed along the row dimension)
  long long sC_b, sC_h;       // output offsets per zb / zh
  // persistent tile scheduler: tile t -> (tm = t % tiles_m, tn = (t / tiles_m) % tiles_n, z = t / (tiles_m * tiles_n))
  int tiles_m, tiles_n, total_tiles;
  int tn_w;                 // tile width along N (multiple of 16, <= TBN): chosen per problem against wave quantisation;
                            // the MMA of a tile is issued with N = its valid columns rounded up to 16
  // split-K (small-M layers that cannot fill 148 SMs): work item = (tile, split); split s covers k-blocks
  // [s*kb_per_split, min(num_kb, (s+1)*kb_per_split)) and writes its raw partial tile to ws[s][M][N]; splitk_reduce_kernel
  // then sums the partials in fixed order and applies alpha / bias / row vector / residual
  int splits, kb_per_split;
  float* ws;
  // MODE_H16: tracked max |A| (device scalars written by the producers of A / A2), exponent of the pre-scaled fp16 weight
  // planes, `fast` = hi*hi term only (the separately reported reduced-precision path)
  const float* a_amax; const float* a2_amax;
  int b_exp;
  int fast;
  float* c_amax;            // optional: atomic max of |C| over everything this launch stores (operand range for the consumer GEMM)
  double* c_stats;          // optional: per-(image, channel) fp64 {sum, sum sq} of C, for the GroupNorm that consumes it; requires
                            // every 32-row quadrant of a tile to lie inside one image (checked on the host)
};

__device__ __forceinline__ int h16_a_exp(const TcParams& p) {
  if (p.gn_ab) return 0;         // normalised (+SiLU) activations are O(1..100): inside the no-rescale range by construction
  float m = p.a_amax ? *p.a_amax : 0.f;
  if (p.a2_amax) m = fmaxf(m, *p.a2_amax);
  return h16_exp_of(m);
}

struct TileCoord { int n0, nend, nw, m0, x0, y0, b0, zb, zh, kb0, kb1, split; };

// EPI: the TMA-store epilogue of the dense layers is compiled in (TcParams::epi_tma selects it per launch).  A separate instantiation,
// because the extra live state of that path costs the conv launches' epilogue registers (ptxas: 92 -> 304 bytes of spill stores in
// the shared body; the short-K convs of the pixel U-Net slowed by 8 %)
template <int MODE, bool EPI>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapA2,
               const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo,
               const __grid_constant__ CUtensorMap mapC, const __grid_constant__ CUtensorMap mapClo, const __grid_constant__ CUtensorMap mapR,
               const __grid_constant__ CUtensorMap mapC16, const __grid_constant__ CUtensorMap mapClo16, const __grid_constant__ CUtensorMap mapR16,
               const TcParams p) {
  constexpr bool TS = Cfg<MODE>::TS;
  constexpr bool H16 = Cfg<MODE>::H16;
  constexpr bool CG2 = Cfg<MODE>::CG2;
  constexpr int B_PLANE = Cfg<MODE>::B_PLANE;
  constexpr int HALO_PLANE = Cfg<MODE>::HALO_PLANE;
  constexpr int BK = Cfg<MODE>::BK;
  // stages per TMEM accumulation chunk: 256 K elements; a work item of at most 512 K elements is ONE chunk (its truncation error stays
  // ~2e-6 relative, and the short-K projections -- epilogue-bound -- save a drain round trip per tile)
  const int KCHUNK = p.kb_per_split <= 2 * Cfg<MODE>::KCHUNK ? 2 * Cfg<MODE>::KCHUNK : Cfg<MODE>::KCHUNK;
  constexpr int STAGES = Cfg<MODE>::STAGES;
  constexpr int STAGE_BYTES = Cfg<MODE>::STAGE_BYTES;
  constexpr int TMEM_COLS = Cfg<MODE>::TMEM_COLS;
  constexpr int SPLIT_ARRIVALS = MODE == MODE_TS ? 4 : NUM_SPLIT_WARPS;   // MODE_TS: only the first four split warps work
  // smem offsets inside a stage
  constexpr int OFF_A = 0;                                   // SS: A_hi (raw in place) ; TS: A_raw ; H16: A_raw k 0..31, then k 32..63
  constexpr int OFF_ALO = TILE_BYTES;                        // SS only
  constexpr int OFF_BHI = MODE == MODE_TS ? TILE_BYTES : 2 * TILE_BYTES;
  constexpr int OFF_BLO = MODE == MODE_TS ? 2 * TILE_BYTES : 2 * TILE_BYTES + B_PLANE;
  // CTA pair: rank in the 2-CTA cluster (0 = leader: issues the MMAs); work items are walked per cluster
  const uint32_t rank = CG2 ? cluster_ctarank() : 0u;
  const int t_first = CG2 ? (int)cluster_id_x() : (int)blockIdx.x, t_step = CG2 ? (int)nclusters_x() : (int)gridDim.x;

  pdl_trigger();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // 1024-byte aligned (swizzle atoms)
  const uint32_t bars = base + STAGES * STAGE_BYTES;
  // barrier layout (8 B each): full_raw[S], full_split[S], empty[S], acc_full[2], acc_empty[2], then the TMEM base word
  auto bar_full_raw = [&](int s) { return bars + 8u * s; };
  auto bar_full_split = [&](int s) { return bars + 8u * (STAGES + s); };
  auto bar_empty = [&](int s) { return bars + 8u * (2 * STAGES + s); };
  auto bar_acc_full = [&](int b) { return bars + 8u * (3 * STAGES + b); };
  auto bar_acc_empty = [&](int b) { return bars + 8u * (3 * STAGES + 2 + b); };
  auto bar_halo_full = [&](int h) { return bars + 8u * (3 * STAGES + 4 + h); };
  auto bar_halo_empty = [&](int h) { return bars + 8u * (3 * STAGES + 6 + h); };
  const uint32_t tmem_slot = bars + 8u * (3 * STAGES + 8);
  auto bar_res = [&](int w) { return bars + 256u + 8u * w; };       // per epilogue warp: its residual box has landed
  // halo schedule smem map: B ring of STAGES x (hi 16 KB | lo 16 KB) at the base, then 2 halo buffers x 2 planes of HALO_PLANE bytes
  const bool halo = H16 && p.halo;
  const uint32_t b_ring = halo ? base : base + OFF_BHI;
  const uint32_t b_stride = halo ? 2u * B_PLANE : (uint32_t)STAGE_BYTES;
  const uint32_t halo_base = base + STAGES * 2 * B_PLANE;
  float* const s_bias = reinterpret_cast<float*>(smem_raw + (bars - smem_u32(smem_raw)) + 512);   // [2][TBN], epilogue warps only
  float4* const s_stage = reinterpret_cast<float4*>(smem_raw + (bars - smem_u32(smem_raw)) + 2048);   // 8 warps x 4 KB
  float2* const s_gn = reinterpret_cast<float2*>(smem_raw + (bars - smem_u32(smem_raw)) + 1536);      // 64 (a, o) pairs of the fused GroupNorm

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_full_raw(s), 1);
      mbar_init(bar_full_split(s), CG2 ? 2 * SPLIT_ARRIVALS : SPLIT_ARRIVALS);     // pair: both CTAs' split warps arrive at the leader
      mbar_init(bar_empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_acc_full(b), 1);
      mbar_init(bar_acc_empty(b), CG2 ? 2 * NUM_EPI_WARPS : NUM_EPI_WARPS);
      mbar_init(bar_halo_full(b), 1);
      mbar_init(bar_halo_empty(b), SPLIT_ARRIVALS);
    }
    for (int w = 0; w < NUM_EPI_WARPS; ++w) mbar_init(bar_res(w), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CG2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CG2) cluster_sync_all();          // the peer's barriers must be initialised before any remote arrive / multicast commit
  else __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  pdl_wait();                     // everything above touched shared memory / TMEM only
  // register budget per warpgroup (640 threads launch with 96 each): the TMA / MMA warpgroup gives most of its share back,
  // the epilogue warpgroups (64 fp32 accumulators + a 32-register residual prefetch per thread) take it
  // (each setmaxnreg sits at the top of its role's branch: ptxas budgets the code it dominates)

  // ---- persistent tile loop: every role walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... with GLOBAL k-block and
  // chunk counters, so the smem ring and the two TMEM accumulator buffers keep rolling across tiles and the MMAs of tile
  // i+1 overlap the global stores of tile i
  auto tile_coord = [&](int t) {
    TileCoord c;
    const int split = t % p.splits;
    t /= p.splits;
    c.split = split;
    c.kb0 = split * p.kb_per_split;
    c.kb1 = min(num_kb, c.kb0 + p.kb_per_split);
    const int tm = CG2 ? 2 * (t % p.tiles_m) + (int)rank : t % p.tiles_m;      // pair: p.tiles_m counts 256-row pair tiles
    const int r = t / p.tiles_m;
    const int tn = r % p.tiles_n, z = r / p.tiles_n;
    c.n0 = tn * p.tn_w;
    c.nend = min(p.N, c.n0 + p.tn_w);
    c.nw = ((c.nend - c.n0 + 15) >> 4) << 4;
    c.m0 = 0; c.x0 = 0; c.y0 = 0; c.b0 = 0; c.zb = 0; c.zh = 0;
    if (p.mode == 1) {
      int u = tm;
      const int tx = u % p.tiles_x; u /= p.tiles_x;
      const int ty = u % p.tiles_y; u /= p.tiles_y;
      c.x0 = tx * p.bw; c.y0 = ty * p.bh; c.b0 = u * p.bn;
    } else {
      c.m0 = tm * TBM;
      c.zb = z / p.heads;
      c.zh = z - c.zb * p.heads;
    }
    return c;
  };

  if (warp < FIRST_SPLIT_WARP) {
  // warpgroup 0 (TMA producer, MMA issuer, two warps without a role): all four warps release registers at this one instruction
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  if (warp == 0) {
    // =========================================================================== TMA producer (whole warp, elected issue)
    {
      const int cblocks = p.mode == 1 ? p.Cin / TBK : 0;
      int gkb = 0, ghalo = 0, hl = 0;
      for (int t = t_first; t < p.total_tiles; t += t_step) {
      const TileCoord tc_ = tile_coord(t);
      const int n0 = tc_.n0, m0 = tc_.m0, x0 = tc_.x0, y0 = tc_.y0, b0 = tc_.b0, zb = tc_.zb, zh = tc_.zh;
      // pair: this CTA holds rows [rank * nw/2, +nw/2) of the B tile (the TMA box is tn_w/2 rows; surplus rows of a ragged tile are unused)
      const int b_rows = CG2 ? p.tn_w / 2 : p.tn_w, b_row0 = CG2 ? (int)rank * (tc_.nw / 2) : 0;
      for (int kb = tc_.kb0; kb < tc_.kb1; ++kb, ++gkb) {
        const int s = gkb % STAGES, it = gkb / STAGES;
        if (halo) {
          // stage = (64-channel block cb, tap).  Halo boxes are fetched in channel-block order: the item's first one before its
          // first stage, the next block's from tap 3 on (by then the split warps are done with the buffer it lands in: this
          // warp runs at most STAGES stages ahead of the MMAs), so a box is in flight for ~5 stages before its first use
          const int cb = kb / 9, tap = kb - cb * 9;
          if (kb == tc_.kb0) hl = cb;
          const bool need = hl * 9 < tc_.kb1 && (hl == cb || (hl == cb + 1 && tap >= 3));
          const int hs = ghalo & 1, hcb = hl;
          if (need) {
            mbar_wait(bar_halo_empty(hs), ((ghalo >> 1) & 1) ^ 1);
            ++ghalo;
            ++hl;
          }
          mbar_wait(bar_empty(s), (it & 1) ^ 1);
          if (!elect_one()) continue;
          if (need) {
            const uint32_t hb = halo_base + (uint32_t)hs * 2u * HALO_PLANE;
            const uint32_t box_bytes = (uint32_t)((p.bw + 2) * (p.bh + 2) * p.bn) * 128u;
            mbar_expect_tx(bar_halo_full(hs), 2u * box_bytes);
            const int hc = hcb * 64;                                   // channel concat: blocks >= C1 come from the second source
            const CUtensorMap* hm = hc < p.C1 ? &mapA : &mapA2;
            const int hcc = hc < p.C1 ? hc : hc - p.C1;
            tma_load_4d(hb, hm, hcc, x0 - 1, y0 - 1, b0, bar_halo_full(hs));                  // OOB -> zeros = padding
            tma_load_4d(hb + HALO_PLANE, hm, hcc + 32, x0 - 1, y0 - 1, b0, bar_halo_full(hs));
          }
          const uint32_t sbh = b_ring + (uint32_t)s * b_stride;
          const int kB = tap * p.Cin + cb * 64;                      // weight planes stay in (tap, channel) order
          mbar_expect_tx(bar_full_raw(s), 2 * b_rows * BK * 2);
          tma_load_2d(sbh, &mapB, kB, n0 + b_row0, bar_full_raw(s));
          tma_load_2d(sbh + B_PLANE, &mapBlo, kB, n0 + b_row0, bar_full_raw(s));
          continue;
        }
        mbar_wait(bar_empty(s), (it & 1) ^ 1);
        const uint32_t st = base + s * STAGE_BYTES;
        const uint32_t sa = st + OFF_A, sb = st + OFF_BHI;
        const int k0 = kb * BK;
        if (!elect_one()) continue;
        if (H16) {
          // two 32-float A sub-blocks (each its own tap / source: a stage may straddle) + fp16 B planes of 64 k (128 B rows)
          const int nsub = (k0 + TBK < p.K) ? 2 : 1;               // K % 32 == 0; an odd tail stage carries one sub-block
          mbar_expect_tx(bar_full_raw(s), nsub * TILE_BYTES + 2 * b_rows * BK * 2);
          for (int sub = 0; sub < nsub; ++sub) {
            const int ks = k0 + sub * TBK;
            const uint32_t dst = sa + sub * TILE_BYTES;
            if (p.mode == 0) {
              if (ks < p.C1) tma_load_2d(dst, &mapA, ks, m0, bar_full_raw(s));
              else tma_load_2d(dst, &mapA2, ks - p.C1, m0, bar_full_raw(s));
            } else {
              const int kq = ks / TBK;
              const int tap = kq / cblocks, cb = kq - tap * cblocks;
              const int dy = tap / 3, dx = tap - dy * 3;
              tma_load_4d(dst, &mapA, cb * TBK, x0 * p.cstride + dx - p.cpad, y0 * p.cstride + dy - p.cpad, b0, bar_full_raw(s));
            }
          }
          tma_load_2d(sb, &mapB, k0, n0 + b_row0, bar_full_raw(s));
          tma_load_2d(st + OFF_BLO, &mapBlo, k0, n0 + b_row0, bar_full_raw(s));
          continue;
        }
        mbar_expect_tx(bar_full_raw(s), TILE_BYTES + (TS ? 2 : 1) * p.tn_w * TBK * 4);
        if (p.mode == 0) {
          if (k0 < p.C1) tma_load_2d(sa, &mapA, k0, m0, bar_full_raw(s));
          else tma_load_2d(sa, &mapA2, k0 - p.C1, m0, bar_full_raw(s));
        } else if (p.mode == 2) {
          int ca[4], cb4[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int ac = p.a_code[i], bc = p.b_code[i];
            ca[i] = ac == 0 ? k0 : ac == 1 ? m0 + zh * p.a_rowoff_h : ac == 2 ? zh : ac == 3 ? zb : 0;
            cb4[i] = bc == 0 ? k0 : bc == 1 ? n0 + zh * p.b_rowoff_h : bc == 2 ? zh : bc == 3 ? zb : 0;
          }
          tma_load_4d(sa, &mapA, ca[0], ca[1], ca[2], ca[3], bar_full_raw(s));
          tma_load_4d(sb, &mapB, cb4[0], cb4[1], cb4[2], cb4[3], bar_full_raw(s));
          continue;                                               // (batched mode is SS only)
        } else {
          const int tap = kb / cblocks, cb = kb - tap * cblocks;
          const int dy = tap / 3, dx = tap - dy * 3;
          tma_load_4d(sa, &mapA, cb * TBK, x0 * p.cstride + dx - p.cpad, y0 * p.cstride + dy - p.cpad, b0, bar_full_raw(s));   // OOB -> zeros = padding
        }
        tma_load_2d(sb, &mapB, k0, n0, bar_full_raw(s));
        if (TS) tma_load_2d(st + OFF_BLO, &mapBlo, k0, n0, bar_full_raw(s));
      }
      }
    }
  } else if (warp == 1) {
    // =========================================================================== MMA issuer (whole warp, elected issue)
    // The profile of the previous version showed this warp busy ~75 % of the time with ~150 SASS instructions per stage (div / mod
    // of the stage counters, descriptor construction, per-MMA branches) around 12 tcgen05.mma: the issue loop, not the tensor pipe,
    // set the pace.  Counters are now carried incrementally, the smem descriptors are one add per stage, and the reduced-precision
    // variant has its own copy of the loop.
    {
      int slot = 0;
      uint32_t ph = 0;                              // stage slot of the ring and its phase parity
      int chunk = 0;                                // global chunk counter (TMEM accumulator buffer = chunk & 1)
      const bool fast = H16 && p.fast == 1;
      const int kb_half = (H16 && (p.K % BK) != 0) ? num_kb - 1 : -1;   // H16: K % 64 == 32 -> the last stage carries one sub-block
      const uint64_t desc0 = make_desc(0);
      for (int t = (CG2 && rank != 0) ? p.total_tiles : t_first; t < p.total_tiles; t += t_step) {      // pair: only the leader issues
        const TileCoord tc_ = tile_coord(t);
        // instruction descriptor: D fp32; A / B format tf32 (2) or f16 (0), both K-major; N >> 3; M >> 4 (pair: M = 256)
        const uint32_t idesc = (1u << 4) | (H16 ? 0u : ((2u << 7) | (2u << 10))) | ((uint32_t)(tc_.nw >> 3) << 17) | ((uint32_t)((CG2 ? 2 * TBM : TBM) >> 4) << 24);
        int kin = 0;
        for (int kb = tc_.kb0; kb < tc_.kb1; ++kb) {
          const int buf = chunk & 1;
          if (kin == 0 && chunk >= 2) {       // the buffer's previous chunk must have been drained (pair: by both CTAs)
            if (CG2) mbar_wait_cluster(bar_acc_empty(buf), ((chunk >> 1) - 1) & 1);
            else mbar_wait(bar_acc_empty(buf), ((chunk >> 1) - 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          }
          if (CG2) mbar_wait_cluster(bar_full_split(slot), ph);
          else mbar_wait(bar_full_split(slot), ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const bool chunk_end = kin == KCHUNK - 1 || kb == tc_.kb1 - 1;
          const uint32_t acc = tmem_base + (uint32_t)(buf * TBN);
          const uint32_t st = base + slot * STAGE_BYTES;
          const uint32_t sbh = H16 ? b_ring + (uint32_t)slot * b_stride : st + OFF_BHI;
          const uint64_t b_hi = desc0 | (uint64_t)((sbh >> 4) & 0x3FFF);
          const uint64_t b_lo = H16 ? b_hi + (B_PLANE >> 4) : desc0 | (uint64_t)(((st + OFF_BLO) >> 4) & 0x3FFF);
          const uint32_t first = kin > 0 ? 1u : 0u;
          if (elect_one()) {
            if (H16) {
              // A: packed fp16 pairs in TMEM (hi: 32 columns = 64 k, lo: the next 32); a K = 16 MMA consumes 8 columns of A and
              // 32 bytes (2 descriptor units) of each B row
              const uint32_t a_hi = tmem_base + (uint32_t)(Cfg<MODE>::A_COL0 + slot * 64), a_lo = a_hi + 32;
              auto umma_ts_f16 = [](uint32_t d, uint32_t a, uint64_t b, uint32_t id, uint32_t accu) {
                if (CG2) tc::umma2_ts_f16(d, a, b, id, accu);
                else tc::umma_ts_f16(d, a, b, id, accu);
              };
              if (!fast) {
                umma_ts_f16(acc, a_lo, b_hi, idesc, first);      // small terms first
                umma_ts_f16(acc, a_hi, b_lo, idesc, 1u);
                umma_ts_f16(acc, a_hi, b_hi, idesc, 1u);
                umma_ts_f16(acc, a_lo + 8, b_hi + 2, idesc, 1u);
                umma_ts_f16(acc, a_hi + 8, b_lo + 2, idesc, 1u);
                umma_ts_f16(acc, a_hi + 8, b_hi + 2, idesc, 1u);
                if (kb != kb_half) {
                  umma_ts_f16(acc, a_lo + 16, b_hi + 4, idesc, 1u);
                  umma_ts_f16(acc, a_hi + 16, b_lo + 4, idesc, 1u);
                  umma_ts_f16(acc, a_hi + 16, b_hi + 4, idesc, 1u);
                  umma_ts_f16(acc, a_lo + 24, b_hi + 6, idesc, 1u);
                  umma_ts_f16(acc, a_hi + 24, b_lo + 6, idesc, 1u);
                  umma_ts_f16(acc, a_hi + 24, b_hi + 6, idesc, 1u);
                }
              } else {
                umma_ts_f16(acc, a_hi, b_hi, idesc, first);
                umma_ts_f16(acc, a_hi + 8, b_hi + 2, idesc, 1u);
                if (kb != kb_half) {
                  umma_ts_f16(acc, a_hi + 16, b_hi + 4, idesc, 1u);
                  umma_ts_f16(acc, a_hi + 24, b_hi + 6, idesc, 1u);
                }
              }
            } else if (TS) {
              const uint32_t a_hi = tmem_base + (uint32_t)(Cfg<MODE>::A_COL0 + slot * 64), a_lo = a_hi + 32;
#pragma unroll
              for (int j = 0; j < TBK / 8; ++j) {
                const uint64_t adv = (uint64_t)((j * 8 * 4) >> 4);    // 32 bytes per K chunk of 8 tf32 in smem; 8 columns in TMEM
                umma_ts(acc, a_lo + j * 8, b_hi + adv, idesc, j > 0 ? 1u : first);      // small terms first
                umma_ts(acc, a_hi + j * 8, b_lo + adv, idesc, 1u);
                umma_ts(acc, a_hi + j * 8, b_hi + adv, idesc, 1u);
              }
            } else {
              const uint64_t a_hi = desc0 | (uint64_t)(((st + OFF_A) >> 4) & 0x3FFF), a_lo = desc0 | (uint64_t)(((st + OFF_ALO) >> 4) & 0x3FFF);
#pragma unroll
              for (int j = 0; j < TBK / 8; ++j) {
                const uint64_t adv = (uint64_t)((j * 8 * 4) >> 4);
                umma_ss(acc, a_lo + adv, b_hi + adv, idesc, j > 0 ? 1u : first);
                umma_ss(acc, a_hi + adv, b_lo + adv, idesc, 1u);
                umma_ss(acc, a_hi + adv, b_hi + adv, idesc, 1u);
              }
            }
            if (CG2) {
              umma2_commit_mc(bar_empty(slot));     // both CTAs' stage slots
              if (chunk_end) umma2_commit_mc(bar_acc_full(buf));
            } else {
              umma_commit(bar_empty(slot));       // stage (smem and, for TS, its TMEM A columns) reusable once these MMAs are done
              if (chunk_end) umma_commit(bar_acc_full(buf));   // chunk complete
            }
          }
          __syncwarp();
          if (chunk_end) { kin = 0; ++chunk; } else ++kin;
          if (++slot == STAGES) { slot = 0; ph ^= 1u; }
        }
      }
    }
  }
  }   // warpgroup 0
  else if (warp < FIRST_EPI_WARP) {
    // register pool of the CTA = 640 x 96: warpgroup 0 gives back 40 per thread and the split warpgroups 16, which is exactly
    // what lets the two epilogue warpgroups grow to 128 (a setmaxnreg.inc that the pool cannot serve spins forever)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    // =========================================================================== split warps
    if (H16) {
      // x' = x * 2^ea, hi = fp16(x'), lo = fp16(x' - hi), packed two per 32-bit TMEM column (even k in the low half).  Eight warps,
      // two per TMEM lane quadrant (the profile of the 4-warp version showed the split warps issue-bound with nothing else resident on
      // their schedulers).
      const int q = warp & 3;
      const int sub = (warp - FIRST_SPLIT_WARP) >> 2;
      const int row = q * 32 + lane;
      const int ea = h16_a_exp(p);
      const float asc = exp2i(ea);
      auto split2 = [&](uint32_t a0, uint32_t a1, uint32_t& h_out, uint32_t& l_out) {
        float x0 = __uint_as_float(a0), x1 = __uint_as_float(a1);
        if (ea != 0) { x0 *= asc; x1 *= asc; }
        const __half2 h = __floats2half2_rn(x0, x1);          // .x (low half) = even k
        const float2 hf = __half22float2(h);
        const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
        h_out = *reinterpret_cast<const uint32_t*>(&h);
        l_out = *reinterpret_cast<const uint32_t*>(&l);
      };
      if (halo) {
        // ---- halo schedule.  Every activation element used to be converted once per tap and N tile it takes part in (9 x per tile);
        // now the halo box of a 64-channel block is converted ONCE, in place, into an fp16 hi plane (plane 0: 64 channels = 128 B per
        // pixel) and a lo plane (plane 1) -- one pixel per thread -- and the per-tap work of a stage is a copy: 8 x LDS.128 of this
        // thread's shifted pixel -> one tcgen05.st of 32 columns (warps of sub 0 copy the hi plane, sub 1 the lo plane).
        const int tid = (int)threadIdx.x - FIRST_SPLIT_WARP * 32;      // 0..255
        const int npx = (p.bw + 2) * (p.bh + 2) * p.bn;                 // <= 200 <= 256 threads (host-checked against the plane size)
        const int hrow0 = ((row / (p.bw * p.bh)) * (p.bh + 2) + (row / p.bw) % p.bh) * (p.bw + 2) + row % p.bw;   // pixel at tap (0, 0)
        int gkb = 0, ghalo = 0, cur_h = 0;
        for (int t = t_first; t < p.total_tiles; t += t_step) {
        const TileCoord tc_ = tile_coord(t);
        for (int kb = tc_.kb0; kb < tc_.kb1; ++kb, ++gkb) {
          const int s = gkb % STAGES, it = gkb / STAGES;
          const int cb = kb / 9, tap = kb - cb * 9;
          if (tap == 0 || kb == tc_.kb0) {
            cur_h = ghalo & 1;
            mbar_wait(bar_halo_full(cur_h), (ghalo >> 1) & 1);
            ++ghalo;
            bool inside = true;
            if (p.gn_ab) {
              // fused GroupNorm (+SiLU): this block's 64 (a, o) pairs of the tile's image -> shared memory (bn == 1), and whether
              // this thread's halo pixel lies inside the image (padding pixels must stay 0 AFTER the activation)
              if (tid < 64) s_gn[tid] = p.gn_ab[(long long)tc_.b0 * p.Cin + cb * 64 + tid];
              asm volatile("bar.sync 3, %0;" ::"n"(NUM_SPLIT_WARPS * 32) : "memory");
              const int hx = tc_.x0 - 1 + tid % (p.bw + 2), hy = tc_.y0 - 1 + (tid / (p.bw + 2)) % (p.bh + 2);
              inside = hx >= 0 && hx < p.W && hy >= 0 && hy < p.H && tc_.b0 < p.B;
            }
            auto gn_act = [&](uint32_t& bits, int c) {
              const float2 ao = s_gn[c];
              float t = fmaf(__uint_as_float(bits), ao.x, ao.y);
              if (p.gn_silu) t = __fdividef(t, 1.f + __expf(-t));
              bits = inside ? __float_as_uint(t) : 0u;
            };
            if (tid < npx) {
              const uint32_t r0 = halo_base + (uint32_t)(cur_h * 2) * HALO_PLANE + (uint32_t)tid * 128u, r1 = r0 + HALO_PLANE;
              const uint32_t px = (uint32_t)(tid & 7);
              uint32_t v[32], lo0[16];
              // channels 0..31 (raw plane 0) -> hi chunks 0..3 of plane 0 (written now: the whole raw row is in registers), lo kept
#pragma unroll
              for (int c = 0; c < 8; ++c)
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[4 * c]), "=r"(v[4 * c + 1]), "=r"(v[4 * c + 2]), "=r"(v[4 * c + 3]) : "r"(r0 + (((uint32_t)c ^ px) << 4)));
              if (p.gn_ab) {
#pragma unroll
                for (int c = 0; c < 32; ++c) gn_act(v[c], c);
              }
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                uint32_t h[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) split2(v[8 * c + 2 * e], v[8 * c + 2 * e + 1], h[e], lo0[4 * c + e]);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + (((uint32_t)c ^ px) << 4)), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
              }
              // channels 32..63 (raw plane 1) -> hi chunks 4..7 of plane 0, then the whole lo row into plane 1
#pragma unroll
              for (int c = 0; c < 8; ++c)
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[4 * c]), "=r"(v[4 * c + 1]), "=r"(v[4 * c + 2]), "=r"(v[4 * c + 3]) : "r"(r1 + (((uint32_t)c ^ px) << 4)));
              if (p.gn_ab) {
#pragma unroll
                for (int c = 0; c < 32; ++c) gn_act(v[c], 32 + c);
              }
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                uint32_t h[4], l[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) split2(v[8 * c + 2 * e], v[8 * c + 2 * e + 1], h[e], l[e]);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(r0 + (((uint32_t)(c + 4) ^ px) << 4)), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(r1 + (((uint32_t)(c + 4) ^ px) << 4)), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
              }
#pragma unroll
              for (int c = 0; c < 4; ++c)
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(r1 + (((uint32_t)c ^ px) << 4)), "r"(lo0[4 * c]), "r"(lo0[4 * c + 1]), "r"(lo0[4 * c + 2]), "r"(lo0[4 * c + 3]) : "memory");
            }
            asm volatile("bar.sync 2, %0;" ::"n"(NUM_SPLIT_WARPS * 32) : "memory");      // every pixel converted before any tap reads it
          }
          const int dy = tap / 3, dx = tap - dy * 3;
          const int hp = hrow0 + dy * (p.bw + 2) + dx;
          const uint32_t sa = halo_base + (uint32_t)(cur_h * 2 + sub) * HALO_PLANE + (uint32_t)hp * 128u, hx = (uint32_t)(hp & 7);
          uint32_t w[32];
#pragma unroll
          for (int c = 0; c < 8; ++c)
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[4 * c]), "=r"(w[4 * c + 1]), "=r"(w[4 * c + 2]), "=r"(w[4 * c + 3]) : "r"(sa + (((uint32_t)c ^ hx) << 4)));
          // the stage slot's barrier says "TMEM A columns free, B landed": waited for only now, after the loads were issued
          mbar_wait(bar_full_raw(s), it & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          tmem_st32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg<MODE>::A_COL0 + s * 64 + sub * 32), w);
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            if (CG2) mbar_arrive_cluster(mapa_rank(bar_full_split(s), 0));      // the leader's barrier counts both CTAs' split warps
            else mbar_arrive(bar_full_split(s));
            if (tap == 8 || kb == tc_.kb1 - 1) {                                 // all taps of this block read: the buffer may be refilled
              asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic-proxy accesses before the next TMA write
              mbar_arrive(bar_halo_empty(cur_h));
            }
          }
        }
        }
      } else {
        // ---- raw A tiles by TMA: thread = one tile row of ONE 32-float sub-block of the stage (warps of sub 0 / sub 1)
        const uint32_t rbase = (uint32_t)row * 128u;
        const uint32_t rx = (uint32_t)(row & 7);
        int gkb = 0;
        for (int t = t_first; t < p.total_tiles; t += t_step) {
        const TileCoord tc_ = tile_coord(t);
        for (int kb = tc_.kb0; kb < tc_.kb1; ++kb, ++gkb) {
          const int s = gkb % STAGES, it = gkb / STAGES;
          const uint32_t sa = base + s * STAGE_BYTES + OFF_A + sub * TILE_BYTES + rbase;
          mbar_wait(bar_full_raw(s), it & 1);
          const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg<MODE>::A_COL0 + s * 64 + sub * 16);
          if (sub == 0 || kb * BK + TBK < p.K) {          // an odd tail stage carries only sub-block 0
            uint32_t v[32], hi[16], lo[16];
#pragma unroll
            for (int c = 0; c < 8; ++c)
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[4 * c]), "=r"(v[4 * c + 1]), "=r"(v[4 * c + 2]), "=r"(v[4 * c + 3]) : "r"(sa + (((uint32_t)c ^ rx) << 4)));
#pragma unroll
            for (int e2 = 0; e2 < 16; ++e2) split2(v[2 * e2], v[2 * e2 + 1], hi[e2], lo[e2]);
            tmem_st16(ta, hi);
            tmem_st16(ta + 32, lo);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            if (CG2) mbar_arrive_cluster(mapa_rank(bar_full_split(s), 0));
            else mbar_arrive(bar_full_split(s));
          }
        }
        }
      }
    } else if (TS) {
      // thread = one tile row: read its 128 raw bytes (8 swizzled 16-byte chunks), store hi / lo into TMEM lane `row`
      // (the TF32-plane path keeps the one-warp-per-quadrant split: warps 6..9 have nothing to do)
      const int q = warp & 3;                    // TMEM lane quadrant (warps 2..5 -> 2,3,0,1)
      const int row = q * 32 + lane;
      const uint32_t rbase = (uint32_t)row * 128u;
      const uint32_t rx = (uint32_t)(row & 7);
      int gkb = 0;
      for (int t = warp < FIRST_SPLIT_WARP + 4 ? t_first : p.total_tiles; t < p.total_tiles; t += t_step) {
      const TileCoord tc_ = tile_coord(t);
      for (int kb = tc_.kb0; kb < tc_.kb1; ++kb, ++gkb) {
        const int s = gkb % STAGES, it = gkb / STAGES;
        mbar_wait(bar_full_raw(s), it & 1);
        const uint32_t sa = base + s * STAGE_BYTES + OFF_A + rbase;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          uint32_t v[4];
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(sa + (((uint32_t)c ^ rx) << 4)));
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const uint32_t h = rn_tf32(v[e]);
            hi[c * 4 + e] = h;
            lo[c * 4 + e] = rn_tf32(__float_as_uint(__uint_as_float(v[e]) - __uint_as_float(h)));
          }
        }
        const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(Cfg<MODE>::A_COL0 + s * 64);
        tmem_st32(ta, hi);
        tmem_st32(ta + 32, lo);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full_split(s));
      }
      }
    } else {
      const int st_ = threadIdx.x - FIRST_SPLIT_WARP * 32;        // 0..255
      int gkb = 0;
      for (int t = t_first; t < p.total_tiles; t += t_step) {
      const TileCoord tc_ = tile_coord(t);
      for (int kb = tc_.kb0; kb < tc_.kb1; ++kb, ++gkb) {
        const int s = gkb % STAGES, it = gkb / STAGES;
        mbar_wait(bar_full_raw(s), it & 1);
        const uint32_t sa = base + s * STAGE_BYTES;
#pragma unroll 4
        for (int i = 0; i < (2 * TILE_BYTES / 16) / (NUM_SPLIT_WARPS * 32); ++i) {
          const int idx = st_ + i * NUM_SPLIT_WARPS * 32;            // float4 index over [A | B]
          const uint32_t off = (uint32_t)idx * 16u;
          const uint32_t src = off < (uint32_t)TILE_BYTES ? sa + off : sa + 2 * TILE_BYTES + (off - TILE_BYTES);
          uint32_t v[4], h[4], l[4];
          asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(src));
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            h[c] = rn_tf32(v[c]);                                                           // hi = rn_tf32(x)
            l[c] = rn_tf32(__float_as_uint(__uint_as_float(v[c]) - __uint_as_float(h[c])));   // lo = rn_tf32(x - hi)
          }
          asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(src), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
          asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(src + TILE_BYTES), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_full_split(s));
      }
      }
    }
  } else if (warp >= FIRST_EPI_WARP) {
    // =========================================================================== drain + epilogue warps
    asm volatile("setmaxnreg.inc.sync.aligned.u32 128;");
    // eight warps: two per TMEM lane quadrant, each owning 32 rows x 64 columns (hf = column half) of the tile
    const int q = warp & 3;                        // TMEM lane quadrant this warp may access (warps 6..13 -> 2,3,0,1,2,3,0,1)
    const int ew = warp - FIRST_EPI_WARP;          // 0..7
    const int hf = ew >> 2;                        // column half
    const int r = q * 32 + lane;                   // tile row owned by this thread
    const int et = hf * 128 + q * 32 + lane;       // 0..255: threads 0..127 stage the tile's bias vector
    constexpr int HN = TBN / 2;                    // 64 columns per thread
    // MODE_H16: the accumulator holds 2^(ea + eb) times the product -> exact power-of-two rescale folded into alpha
    const float alpha = H16 ? p.alpha * exp2i(-h16_a_exp(p)) * exp2i(-p.b_exp) : p.alpha;
    float omax = 0.f;                              // max |C| stored by this thread (p.c_amax)
    float4* const stg = s_stage + ew * 256;        // this warp's 4 KB staging block: [32 rows][8 float4], chunk index XOR (row & 7)
    const uint32_t stg_addr = smem_u32(stg);
    uint32_t res_ph = 0;
    int gchunk0 = 0, tile_it = 0;
#pragma unroll 1
    for (int t = t_first; t < p.total_tiles; t += t_step, ++tile_it) {
    const TileCoord tc_ = tile_coord(t);
    const int num_chunks = (tc_.kb1 - tc_.kb0 + KCHUNK - 1) / KCHUNK;
    const int n0 = tc_.n0, m0 = tc_.m0, x0 = tc_.x0, y0 = tc_.y0, b0 = tc_.b0, zb = tc_.zb, zh = tc_.zh;
    // the tile's 128 bias values: one coalesced load issued before the drain (latency hidden behind it), handed to
    // all rows through shared memory; double-buffered by tile parity so a fast warp cannot overwrite a slow warp's tile
    float bias_v = 0.f;
    if (et < TBN && p.bias && p.splits == 1 && n0 + et < p.N) bias_v = __ldg(p.bias + n0 + et);
    // TMA epilogue (p.epi_tma): this warp's 32 rows x 64 columns leave as one or two boxes of 32 (the last one possibly 16) columns;
    // it needs whole rows and whole 16-column blocks (anything else takes the per-row path below).  The residual box of the first
    // slot is requested before the drain, so it is in shared memory by the time the accumulator is
    const int wcols = p.geglu ? HN / 2 : min(max(tc_.nend - (n0 + hf * HN), 0), HN);       // columns this warp stores
    const bool tma_tile = EPI && p.epi_tma && m0 + TBM <= p.M && (wcols & 15) == 0 && !(p.Ct_hi && n0 >= p.t_col0);
    const int tparts = (wcols + 31) >> 5;
    const int tcol0 = p.geglu ? (n0 >> 1) + hf * 32 : n0 + hf * HN, trow0 = m0 + q * 32;
    if (EPI && p.epi_tma) {
      if (lane == 0) {
        bulk_wait_read0();                         // the previous tile's stores have left the staging block
        if (tma_tile && p.residual && wcols > 0) {
          mbar_expect_tx(bar_res(ew), wcols >= 32 ? 4096 : 2048);
          tma_load_2d(stg_addr, wcols >= 32 ? &mapR : &mapR16, tcol0, trow0, bar_res(ew));
        }
      }
      __syncwarp();
    }
    float acc[HN];
#pragma unroll
    for (int j = 0; j < HN; ++j) acc[j] = 0.f;
#pragma unroll 1
    for (int lchunk = 0; lchunk < num_chunks; ++lchunk) {
      const int chunk = gchunk0 + lchunk;
      const int buf = chunk & 1;
      mbar_wait(bar_acc_full(buf), (chunk >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * TBN + hf * HN);
#pragma unroll
      for (int part = 0; part < HN / 32; ++part) {
        uint32_t v[32];
        tmem_ld32(taddr + part * 32, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[part * 32 + j] += __uint_as_float(v[j]);     // round-to-nearest fp32 add
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        if (CG2) mbar_arrive_cluster(mapa_rank(bar_acc_empty(buf), 0));
        else mbar_arrive(bar_acc_empty(buf));
      }
    }
    float* const sb = s_bias + (tile_it & 1) * TBN;
    if (et < TBN) sb[et] = bias_v;
    asm volatile("bar.sync 1, %0;" ::"n"(NUM_EPI_WARPS * 32) : "memory");

    long long m;
    bool row_ok;
    if (p.mode != 1) {
      m = (long long)m0 + r;
      row_ok = m < p.M;
    } else {
      const int xl = r % p.bw, yl = (r / p.bw) % p.bh, nl = r / (p.bw * p.bh);
      const int b = b0 + nl;
      row_ok = b < p.B;
      m = ((long long)b * p.H + (y0 + yl)) * p.W + (x0 + xl);
    }
    gchunk0 += num_chunks;
    if (p.out_nchw) {
      if (row_ok) {
        const long long bimg = m / p.rows_per_img, rimg = m - bimg * p.rows_per_img;
#pragma unroll
        for (int j = 0; j < HN; ++j) {
          const int n = n0 + hf * HN + j;
          if (n < tc_.nend) p.C[(bimg * p.N + n) * p.rows_per_img + rimg] = alpha * acc[j] + sb[hf * HN + j];   // lanes = pixels: coalesced
        }
      }
    } else if (p.Ct_hi && n0 >= p.t_col0) {
      // transposed TF32-plane output (V^T): thread = row m, so for a fixed column the 32 lanes write 32 consecutive floats
      if (row_ok) {
#pragma unroll
        for (int j = 0; j < HN; ++j) {
          const int n = n0 + hf * HN + j;
          if (n < tc_.nend) {
            const float o = alpha * acc[j] + sb[hf * HN + j];
            const float hi = __uint_as_float(rn_tf32(__float_as_uint(o)));
            const long long at = (long long)(n - p.t_col0) * p.ldt + m;
            p.Ct_hi[at] = hi;
            p.Ct_lo[at] = __uint_as_float(rn_tf32(__float_as_uint(o - hi)));
            omax = fmaxf(omax, fabsf(hi));                        // the range of the stored hi plane, as for the row-major planes
          }
        }
      }
    } else if (tma_tile) {
      if (tparts > 0) {
#pragma unroll
        for (int j = 0; j < HN; j += 4) {
          const float4 bv = *reinterpret_cast<const float4*>(sb + hf * HN + j);
          acc[j + 0] = alpha * acc[j + 0] + bv.x;
          acc[j + 1] = alpha * acc[j + 1] + bv.y;
          acc[j + 2] = alpha * acc[j + 2] + bv.z;
          acc[j + 3] = alpha * acc[j + 3] + bv.w;
        }
        if (p.rowvec) {
          const float* rv = p.rowvec + (m / p.rows_per_batch) * p.ld_rowvec + n0 + hf * HN;
#pragma unroll
          for (int j = 0; j < HN; j += 4) {
            if (j < wcols) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(rv + j));
              acc[j + 0] += bv.x; acc[j + 1] += bv.y; acc[j + 2] += bv.z; acc[j + 3] += bv.w;
            }
          }
        }
        if (p.geglu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float gt = acc[32 + j];
            acc[j] *= 0.5f * gt * (1.f + erff(gt * 0.70710678118654752440f));     // exact-erf GELU as F.gelu
          }
        }
        // The warp's 64 columns leave as two slots of 32 (4 KB box, 128 B swizzle: [32 rows][8 chunks], chunk ^ (row & 7)); a ragged
        // tile's last slot may be 16 wide (2 KB box of the 64 B-swizzle maps: [32 rows][4 chunks], index ^ ((row >> 1) & 3)).
        // Measured: 16-column boxes everywhere cost 10-15 % on the 128-wide tiles (twice the bulk operations, half-line writes)
        auto epi_block = [&](auto partc, auto ncc) {
          constexpr int part = decltype(partc)::value;
          constexpr int NC = decltype(ncc)::value;          // 16-byte chunks per row: 8 or 4
          auto sidx = [&](int row, int c) { return NC == 8 ? row * 8 + (c ^ (row & 7)) : (row * 4 + c) ^ ((row >> 1) & 3); };
          if (p.residual) {
            mbar_wait(bar_res(ew), res_ph);
            res_ph ^= 1u;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
              const float4 v = stg[sidx(lane, c)];
              acc[part * 32 + 4 * c + 0] += v.x; acc[part * 32 + 4 * c + 1] += v.y;
              acc[part * 32 + 4 * c + 2] += v.z; acc[part * 32 + 4 * c + 3] += v.w;
            }
          }
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            float4 o = make_float4(acc[part * 32 + 4 * c], acc[part * 32 + 4 * c + 1], acc[part * 32 + 4 * c + 2], acc[part * 32 + 4 * c + 3]);
            if (p.C_lo) {
              o.x = __uint_as_float(rn_tf32(__float_as_uint(o.x))); o.y = __uint_as_float(rn_tf32(__float_as_uint(o.y)));
              o.z = __uint_as_float(rn_tf32(__float_as_uint(o.z))); o.w = __uint_as_float(rn_tf32(__float_as_uint(o.w)));
            }
            omax = fmaxf(omax, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
            stg[sidx(lane, c)] = o;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy writes -> visible to the bulk store
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(stg_addr, NC == 8 ? &mapC : &mapC16, tcol0 + part * 32, trow0);
            bulk_commit();
          }
          if (p.c_stats) {
            // GroupNorm statistics of the tensor being written, from the staged block (the warp's 32 rows lie inside one image).
            // The fp32 partial sums are taken about the column's row-0 value v0 and re-centred in fp64: plain fp32 sums of x and
            // x^2 lose the variance when |mean| >> std (E[x^2] - mean^2 cancels; |mean| / std = 100 costs 4e-5 of the normalised output)
            const float* const sf = reinterpret_cast<const float*>(stg);
            const int col = NC == 8 ? lane : (lane & 15);
            const float v0 = sf[(sidx(0, col >> 2) << 2) | (lane & 3)];
            float cs = 0.f, cq = 0.f;
            if (NC == 8) {                       // lane -> column, all 32 rows (the swizzle permutes chunks: no bank conflict)
#pragma unroll
              for (int rr = 0; rr < 32; ++rr) {
                const float v = sf[(sidx(rr, lane >> 2) << 2) | (lane & 3)] - v0;
                cs += v; cq += v * v;
              }
            } else {                             // lane & 15 -> column, half-warp -> 16 rows (opposite row parity: different banks)
              const int hh = lane >> 4;
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int rr = hh * 16 + (i ^ hh);
                const float v = sf[(sidx(rr, (lane & 15) >> 2) << 2) | (lane & 3)] - v0;
                cs += v; cq += v * v;
              }
              cs += __shfl_xor_sync(0xffffffffu, cs, 16);
              cq += __shfl_xor_sync(0xffffffffu, cq, 16);
            }
            if (NC == 8 || lane < 16) {
              double* st = p.c_stats + ((long long)(trow0 / p.rows_per_batch) * p.N + (tcol0 + part * 32 + col)) * 2;
              const double s0 = v0, ds = cs;
              atomicAdd(st, ds + 32.0 * s0);
              atomicAdd(st + 1, (double)cq + s0 * (2.0 * ds + 32.0 * s0));
            }
          }
          if (p.C_lo) {
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
#pragma unroll
            for (int c = 0; c < NC; ++c) {
              float4 o = make_float4(acc[part * 32 + 4 * c], acc[part * 32 + 4 * c + 1], acc[part * 32 + 4 * c + 2], acc[part * 32 + 4 * c + 3]);
              o.x = __uint_as_float(rn_tf32(__float_as_uint(o.x - __uint_as_float(rn_tf32(__float_as_uint(o.x))))));
              o.y = __uint_as_float(rn_tf32(__float_as_uint(o.y - __uint_as_float(rn_tf32(__float_as_uint(o.y))))));
              o.z = __uint_as_float(rn_tf32(__float_as_uint(o.z - __uint_as_float(rn_tf32(__float_as_uint(o.z))))));
              o.w = __uint_as_float(rn_tf32(__float_as_uint(o.w - __uint_as_float(rn_tf32(__float_as_uint(o.w))))));
              stg[sidx(lane, c)] = o;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(stg_addr, NC == 8 ? &mapClo : &mapClo16, tcol0 + part * 32, trow0);
              bulk_commit();
            }
          }
        };
        using std::integral_constant;
        if (wcols >= 32) epi_block(integral_constant<int, 0>{}, integral_constant<int, 8>{});
        else epi_block(integral_constant<int, 0>{}, integral_constant<int, 4>{});
        if (wcols > 32) {
          if (lane == 0) {
            bulk_wait_read0();                     // slot 0 has left the staging block
            if (p.residual) {
              mbar_expect_tx(bar_res(ew), wcols == 64 ? 4096 : 2048);
              tma_load_2d(stg_addr, wcols == 64 ? &mapR : &mapR16, tcol0 + 32, trow0, bar_res(ew));
            }
          }
          __syncwarp();
          if (wcols == 64) epi_block(integral_constant<int, 1>{}, integral_constant<int, 8>{});
          else epi_block(integral_constant<int, 1>{}, integral_constant<int, 4>{});
        }
      }
    } else {
      const bool fin = p.splits == 1;                // otherwise: raw partial sums to ws[split][M][N]
      // the thread-per-row accumulator layout would store 16 B to 32 different rows per instruction (32 L1 wavefronts
      // each, which also starves the split warps' LDS behind them); instead each warp transposes 32x32 blocks through a
      // swizzled 4 KB staging buffer so that one instruction covers 4 rows x 128 contiguous bytes -- for the residual
      // loads as well, which are issued a whole 32-column block ahead of their use (L2 latency off the critical path)
      float* const dst = fin ? p.C + zb * p.sC_b + zh * p.sC_h : p.ws + (long long)tc_.split * p.M * p.N;
      const long long dld = fin ? p.ldc : p.N;
      const float* const rsd = fin ? p.residual : nullptr;
      float* const dst_lo = (fin && p.C_lo) ? p.C_lo + zb * p.sC_b + zh * p.sC_h : nullptr;
      const int m32 = row_ok ? (int)m : -1;
      const int g = lane & 7, rsub = lane >> 3;
      // GEGLU tiles are [32 value | 32 gate | 32 value | 32 gate]: this thread's 64 columns are 32 values + their gates
      const int nparts = p.geglu ? 1 : HN / 32;
      const int ncol0 = p.geglu ? (n0 >> 1) + hf * 32 : n0 + hf * HN, nlim = p.geglu ? (p.N >> 1) : tc_.nend;
      int mm[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) mm[i] = __shfl_sync(0xffffffffu, m32, 4 * i + rsub);
      float4 t[8];
      auto load_residual = [&](int part) {
        const int n = ncol0 + part * 32 + 4 * g;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          t[i] = (rsd && mm[i] >= 0 && n < nlim) ? *reinterpret_cast<const float4*>(rsd + (long long)mm[i] * p.ldr + n)
                                                 : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      load_residual(0);
      if (fin && row_ok) {
        // pass 1 (registers only): alpha, bias from smem, per-image row vector
#pragma unroll
        for (int j = 0; j < HN; j += 4) {
          const float4 bv = *reinterpret_cast<const float4*>(sb + hf * HN + j);
          acc[j + 0] = alpha * acc[j + 0] + bv.x;
          acc[j + 1] = alpha * acc[j + 1] + bv.y;
          acc[j + 2] = alpha * acc[j + 2] + bv.z;
          acc[j + 3] = alpha * acc[j + 3] + bv.w;
        }
        if (p.rowvec) {
          const float* rv = p.rowvec + (m / p.rows_per_batch) * p.ld_rowvec + n0 + hf * HN;
#pragma unroll
          for (int j = 0; j < HN; j += 4) {
            if (n0 + hf * HN + j < p.N) {                // N % 4 == 0 is an eligibility condition
              const float4 bv = __ldg(reinterpret_cast<const float4*>(rv + j));
              acc[j + 0] += bv.x; acc[j + 1] += bv.y; acc[j + 2] += bv.z; acc[j + 3] += bv.w;
            }
          }
        }
        if (p.geglu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float gt = acc[32 + j];
            acc[j] *= 0.5f * gt * (1.f + erff(gt * 0.70710678118654752440f));     // exact-erf GELU as F.gelu
          }
        }
      }
#pragma unroll
      for (int part = 0; part < HN / 32; ++part) {
        if (part >= nparts) break;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          stg[lane * 8 + (c ^ (lane & 7))] =
              make_float4(acc[part * 32 + 4 * c], acc[part * 32 + 4 * c + 1], acc[part * 32 + 4 * c + 2], acc[part * 32 + 4 * c + 3]);
        __syncwarp();
        const int n = ncol0 + part * 32 + 4 * g;
        float gs[4] = {0.f, 0.f, 0.f, 0.f}, gq[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          float4 o[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int rl = 4 * (half * 4 + i) + rsub;
            const float4 v = stg[rl * 8 + (g ^ (rl & 7))];
            const float4 tt = t[half * 4 + i];
            o[i] = make_float4(v.x + tt.x, v.y + tt.y, v.z + tt.z, v.w + tt.w);
          }
          if (half == 1) {
            __syncwarp();                                         // staging buffer free for the next block
            if (part + 1 < nparts) load_residual(part + 1);      // in flight while this block is stored
          }
          if (p.c_stats) {
            // GroupNorm statistics of the tensor being written: this thread holds 4 columns x 4 rows here (8 rows over both
            // halves); rows of one quadrant belong to one image.  Partial sums about the quadrant's row-0 values, re-centred in fp64
            // below (see the TMA epilogue).  Lane g (rsub 0) is the only reader of row 0's staged chunk g: it puts the final row-0
            // value there, where every lane finds it until the next block is staged (after the fold's shuffles below)
            if (half == 0) {
              if (rsub == 0) stg[g] = o[0];
              __syncwarp();
            }
            const float4 v0 = stg[g];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (mm[half * 4 + i] >= 0) {
                const float dx = o[i].x - v0.x, dy = o[i].y - v0.y, dz = o[i].z - v0.z, dw = o[i].w - v0.w;
                gs[0] += dx; gq[0] += dx * dx;
                gs[1] += dy; gq[1] += dy * dy;
                gs[2] += dz; gq[2] += dz * dz;
                gs[3] += dw; gq[3] += dw * dw;
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int mi = mm[half * 4 + i];
            if (mi >= 0 && n < nlim) {
              if (dst_lo) {                          // operand planes for a following tcgen05 consumer
                float4 hi, lo;
                hi.x = __uint_as_float(rn_tf32(__float_as_uint(o[i].x))); lo.x = __uint_as_float(rn_tf32(__float_as_uint(o[i].x - hi.x)));
                hi.y = __uint_as_float(rn_tf32(__float_as_uint(o[i].y))); lo.y = __uint_as_float(rn_tf32(__float_as_uint(o[i].y - hi.y)));
                hi.z = __uint_as_float(rn_tf32(__float_as_uint(o[i].z))); lo.z = __uint_as_float(rn_tf32(__float_as_uint(o[i].z - hi.z)));
                hi.w = __uint_as_float(rn_tf32(__float_as_uint(o[i].w))); lo.w = __uint_as_float(rn_tf32(__float_as_uint(o[i].w - hi.w)));
                *reinterpret_cast<float4*>(dst_lo + (long long)mi * dld + n) = lo;
                o[i] = hi;
              }
              *reinterpret_cast<float4*>(dst + (long long)mi * dld + n) = o[i];
              omax = fmaxf(omax, fmaxf(fmaxf(fabsf(o[i].x), fabsf(o[i].y)), fmaxf(fabsf(o[i].z), fabsf(o[i].w))));
            }
          }
        }
        if (p.c_stats) {
          const float4 v0 = stg[g];                            // (read before the shuffles: the next block may be staged after them)
          // fold the 4 row-subgroups (lanes g, g+8, g+16, g+24), then one fp64 atomic per (column, statistic)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            gs[j] += __shfl_xor_sync(0xffffffffu, gs[j], 8);  gq[j] += __shfl_xor_sync(0xffffffffu, gq[j], 8);
            gs[j] += __shfl_xor_sync(0xffffffffu, gs[j], 16); gq[j] += __shfl_xor_sync(0xffffffffu, gq[j], 16);
          }
          const int mq = __shfl_sync(0xffffffffu, m32, 0) >= 0 ? __shfl_sync(0xffffffffu, m32, 0) : -1;   // first row of the quadrant
          const double nv = (double)__popc(__ballot_sync(0xffffffffu, m32 >= 0));      // rows of the quadrant inside the tensor
          if (rsub == 0 && mq >= 0 && n < nlim && fin) {
            double* st = p.c_stats + ((long long)(mq / p.rows_per_batch) * p.N + n) * 2;
            const float v0a[4] = {v0.x, v0.y, v0.z, v0.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const double s0 = v0a[j], ds = gs[j];
              atomicAdd(st + 2 * j, ds + nv * s0);
              atomicAdd(st + 2 * j + 1, (double)gq[j] + s0 * (2.0 * ds + nv * s0));
            }
          }
        }
      }
    }
    }   // tile loop
    if (EPI && p.epi_tma && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // bulk stores done before the CTA retires
    if (p.c_amax && p.splits == 1) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) omax = fmaxf(omax, __shfl_xor_sync(0xffffffffu, omax, o));
      if (lane == 0) atomicMax(reinterpret_cast<unsigned int*>(p.c_amax), __float_as_uint(omax));     // non-negative floats order like their bit patterns
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  if (CG2) cluster_sync_all();          // the leader's MMAs read the peer's smem / TMEM: both CTAs stay until both are done
  else __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (CG2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// C = alpha * sum_s ws[s] (+bias) (+row vector) (+residual): fixed summation order, so split-K stays deterministic
__global__ void splitk_reduce_kernel(const float* __restrict__ ws, int splits, TcParams p, int h16) {
  pdl_trigger();
  pdl_wait();
  const long long total4 = (long long)p.M * p.N / 4;
  const float alpha = h16 ? p.alpha * exp2i(-h16_a_exp(p)) * exp2i(-p.b_exp) : p.alpha;
  float omax = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i * 4;
    const long long m = e / p.N;
    const int n = (int)(e - m * p.N);
    float4 a = *reinterpret_cast<const float4*>(ws + e);
    for (int s = 1; s < splits; ++s) {
      const float4 b = *reinterpret_cast<const float4*>(ws + (long long)s * p.M * p.N + e);
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    a.x *= alpha; a.y *= alpha; a.z *= alpha; a.w *= alpha;
    if (p.bias) { const float4 t = *reinterpret_cast<const float4*>(p.bias + n); a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w; }
    if (p.rowvec) { const float4 t = *reinterpret_cast<const float4*>(p.rowvec + (m / p.rows_per_batch) * p.ld_rowvec + n); a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w; }
    if (p.residual) { const float4 t = *reinterpret_cast<const float4*>(p.residual + m * p.ldr + n); a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w; }
    if (p.C_lo) {
      float4 hi, lo;
      hi.x = __uint_as_float(rn_tf32(__float_as_uint(a.x))); lo.x = __uint_as_float(rn_tf32(__float_as_uint(a.x - hi.x)));
      hi.y = __uint_as_float(rn_tf32(__float_as_uint(a.y))); lo.y = __uint_as_float(rn_tf32(__float_as_uint(a.y - hi.y)));
      hi.z = __uint_as_float(rn_tf32(__float_as_uint(a.z))); lo.z = __uint_as_float(rn_tf32(__float_as_uint(a.z - hi.z)));
      hi.w = __uint_as_float(rn_tf32(__float_as_uint(a.w))); lo.w = __uint_as_float(rn_tf32(__float_as_uint(a.w - hi.w)));
      *reinterpret_cast<float4*>(p.C_lo + m * p.ldc + n) = lo;
      a = hi;
    }
    *reinterpret_cast<float4*>(p.C + m * p.ldc + n) = a;
    omax = fmaxf(omax, fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))));
  }
  if (p.c_amax) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) omax = fmaxf(omax, __shfl_xor_sync(0xffffffffu, omax, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(p.c_amax), __float_as_uint(omax));
  }
}

// x -> (rn_tf32(x), rn_tf32(x - rn_tf32(x)))  : one-time preparation of the weight planes for the TS variant
__global__ void split_planes_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t b = __float_as_uint(w[i]);
    const uint32_t h = rn_tf32(b);
    hi[i] = __uint_as_float(h);
    lo[i] = __uint_as_float(rn_tf32(__float_as_uint(w[i] - __uint_as_float(h))));
  }
}

// w' = w * 2^exp ; hi = fp16(w'), lo = fp16(w' - hi): one-time preparation of the weight planes for MODE_H16
__global__ void split_planes_h16_kernel(const float* __restrict__ w, __half* __restrict__ hi, __half* __restrict__ lo, size_t n, float scale) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float x = w[i] * scale;
    const __half h = __float2half_rn(x);
    hi[i] = h;
    lo[i] = __float2half_rn(x - __half2float(h));
  }
}

__global__ void amax_rows_kernel(const float* __restrict__ x, long long rows, int C, long long ld, float* __restrict__ slot) {
  float m = 0.f;
  const long long total = rows * (long long)(C >> 2);
  const int c4n = C >> 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / c4n;
    const int c4 = (int)(i - r * c4n);
    const float4 v = *reinterpret_cast<const float4*>(x + r * ld + 4 * c4);
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(slot), __float_as_uint(m));
}

// any C / stride (few-channel tensors: a 3-channel VQ latent)
__global__ void amax_rows_scalar_kernel(const float* __restrict__ x, long long rows, int C, long long ld, float* __restrict__ slot) {
  float m = 0.f;
  const long long total = rows * (long long)C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C;
    m = fmaxf(m, fabsf(x[r * ld + (i - r * C)]));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned int*>(slot), __float_as_uint(m));
}

// cudaFuncSetAttribute is per DEVICE: remember which devices of this process have it (engines on several devices share the library)
void ensure_attr(int device) {
  static bool attr_set[64] = {};
  static std::mutex mtx;
  std::lock_guard<std::mutex> lock(mtx);
  const int d = device & 63;
  if (!attr_set[d]) {
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_SS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_SS>::SMEM_BYTES));
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_TS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_TS>::SMEM_BYTES));
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_H16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_H16>::SMEM_BYTES));
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_H16X2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_H16X2>::SMEM_BYTES));
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_H16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_H16>::SMEM_BYTES));
    CDX_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<MODE_H16X2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<MODE_H16X2>::SMEM_BYTES));
    attr_set[d] = true;
  }
}

}  // namespace

void split_planes(Engine& e, const float* w, float* hi, float* lo, size_t n, cudaStream_t s) {
  if (e.dry()) return;
  size_t blocks = (n + 255) / 256;
  if (blocks > (size_t)e.num_sms * 16) blocks = (size_t)e.num_sms * 16;
  split_planes_kernel<<<(unsigned)(blocks ? blocks : 1), 256, 0, s>>>(w, hi, lo, n);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}

void split_planes_h16(Engine& e, const float* w, void* hi, void* lo, size_t n, int exp, cudaStream_t s) {
  if (e.dry()) return;
  size_t blocks = (n + 255) / 256;
  if (blocks > (size_t)e.num_sms * 16) blocks = (size_t)e.num_sms * 16;
  split_planes_h16_kernel<<<(unsigned)(blocks ? blocks : 1), 256, 0, s>>>(w, (__half*)hi, (__half*)lo, n, ldexpf(1.f, exp));
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}

void amax_rows(Engine& e, const float* x, long long rows, int C, long long ld, float* slot, cudaStream_t s) {
  if (e.dry()) return;
  if ((C & 3) || (ld & 3) || !a16(x)) {
    const long long total = rows * (long long)C;
    const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)e.num_sms * 8);
    amax_rows_scalar_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(x, rows, C, ld, slot);
    CDX_CUDA(cudaGetLastError());
    e.launches++;
    return;
  }
  const long long total = rows * (long long)(C >> 2);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)e.num_sms * 8);
  amax_rows_kernel<<<blocks > 0 ? blocks : 1, 256, 0, s>>>(x, rows, C, ld, slot);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
}

int h16_exp_host(float amax) {
  if (!(amax > 0.f) || !std::isfinite(amax)) return 0;
  int ex;
  frexpf(amax, &ex);                    // amax = f * 2^ex, f in [0.5, 1)  ->  floor(log2 amax) = ex - 1
  return std::min(std::max(14 - (ex - 1), -100), 100);
}

// softmax(q k^T * scale) v on the tensor cores: two batched 3xTF32 contractions around the row-softmax kernel.
//   q, k : [B, N*, ...] token matrices (row strides ldq / ldk, head h at column h*head_stride)
//   vt   : V transposed, [heads*d, B*Nk] (row c = channel, column b*Nk + j), produced by a swapped-role GEMM
//   out  : [B, Nq, ldo], head h at column h*d
// Requires Nk % 32 == 0 (a K block must not run into the next sample's columns of vt), d % 4 == 0.
bool attention_tc(Engine& e, const float* q, int ldq, const float* k, int ldk, int head_stride, const float* vt, float* out, int ldo, int B,
                  int Nq, int Nk, int heads, int d, float scale, cudaStream_t s) {
  if ((Nk % TBK) || (d & 3) || (ldq & 3) || (ldk & 3) || (head_stride & 3) || (ldo & 3) || Nq < 64) return false;
  if (!a16(q) || !a16(k) || !a16(vt) || !a16(out)) return false;
  Scope sc(e.arena);
  const int ldS = Nk;
  float* S = (float*)e.arena.alloc((size_t)B * heads * Nq * ldS * sizeof(float));
  if (e.dry()) return true;
  ensure_attr(e.device);
  TcParams p;
  // ---- S = scale * Q K^T
  {
    memset(&p, 0, sizeof(p));
    p.mode = 2; p.M = Nq; p.N = Nk; p.K = d; p.heads = heads; p.alpha = scale;
    p.C = S; p.ldc = ldS; p.sC_b = (long long)heads * Nq * ldS; p.sC_h = (long long)Nq * ldS;
    p.rows_per_batch = 1;
    const int code[4] = {0, 2, 1, 3};      // dims {d, heads, rows, B}
    for (int i = 0; i < 4; ++i) { p.a_code[i] = code[i]; p.b_code[i] = code[i]; }
    uint64_t da[4] = {(uint64_t)d, (uint64_t)heads, (uint64_t)Nq, (uint64_t)B};
    uint64_t sa[3] = {(uint64_t)head_stride * 4, (uint64_t)ldq * 4, (uint64_t)Nq * ldq * 4};
    uint64_t db[4] = {(uint64_t)d, (uint64_t)heads, (uint64_t)Nk, (uint64_t)B};
    uint64_t sb[3] = {(uint64_t)head_stride * 4, (uint64_t)ldk * 4, (uint64_t)Nk * ldk * 4};
    uint32_t bx[4] = {TBK, 1, TBM, 1};
    const CUtensorMap& mA = get_map(q, 4, da, sa, bx);
    const CUtensorMap& mB = get_map(k, 4, db, sb, bx);
    ProfScope ps(e, s, PROF_BATCHED_TC, 2.0 * Nq * Nk * d * B * heads, 4.0 * B * heads * ((double)Nq * d + (double)Nk * d + (double)Nq * Nk), 1);
    p.splits = 1; p.kb_per_split = cdiv(d, TBK);
    p.tn_w = TBN;
    p.tiles_m = cdiv(Nq, TBM); p.tiles_n = cdiv(Nk, TBN); p.total_tiles = p.tiles_m * p.tiles_n * B * heads;
    launch_ex(tc_gemm_kernel<MODE_SS, false>, dim3((unsigned)std::min(p.total_tiles, e.num_sms)), dim3(TC_THREADS), Cfg<MODE_SS>::SMEM_BYTES, s, 1, mA, mA, mB, mB, mA, mA, mA, mA, mA, mA, p);
    CDX_CUDA(cudaGetLastError());
    e.launches++;
  }
  softmax_rows(e, S, (long long)B * heads * Nq, Nk, ldS, s);
  // ---- O = P V   (B operand = V^T rows h*d .. h*d+d-1, K along the sample's Nk columns)
  {
    memset(&p, 0, sizeof(p));
    p.mode = 2; p.M = Nq; p.N = d; p.K = Nk; p.heads = heads; p.alpha = 1.f;
    p.C = out; p.ldc = ldo; p.sC_b = (long long)Nq * ldo; p.sC_h = d;
    p.rows_per_batch = 1;
    const int ac[4] = {0, 1, 2, 3};        // P dims {Nk, Nq, heads, B}
    const int bc[4] = {0, 3, 1, 4};        // V^T dims {Nk, B, heads*d, 1}
    for (int i = 0; i < 4; ++i) { p.a_code[i] = ac[i]; p.b_code[i] = bc[i]; }
    p.b_rowoff_h = d;
    uint64_t da[4] = {(uint64_t)Nk, (uint64_t)Nq, (uint64_t)heads, (uint64_t)B};
    uint64_t sa[3] = {(uint64_t)ldS * 4, (uint64_t)Nq * ldS * 4, (uint64_t)heads * Nq * ldS * 4};
    uint32_t bxa[4] = {TBK, TBM, 1, 1};
    uint64_t db[4] = {(uint64_t)Nk, (uint64_t)B, (uint64_t)heads * d, 1};
    uint64_t sb[3] = {(uint64_t)Nk * 4, (uint64_t)B * Nk * 4, (uint64_t)B * Nk * 4 * heads * d};
    uint32_t bxb[4] = {TBK, 1, TBN, 1};
    const CUtensorMap& mA = get_map(S, 4, da, sa, bxa);
    const CUtensorMap& mB = get_map(vt, 4, db, sb, bxb);
    ProfScope ps(e, s, PROF_BATCHED_TC, 2.0 * Nq * Nk * d * B * heads, 4.0 * B * heads * ((double)Nq * Nk + (double)Nk * d + (double)Nq * d), 1);
    p.splits = 1; p.kb_per_split = cdiv(Nk, TBK);
    p.tn_w = TBN;
    p.tiles_m = cdiv(Nq, TBM); p.tiles_n = cdiv(d, TBN); p.total_tiles = p.tiles_m * p.tiles_n * B * heads;
    launch_ex(tc_gemm_kernel<MODE_SS, false>, dim3((unsigned)std::min(p.total_tiles, e.num_sms)), dim3(TC_THREADS), Cfg<MODE_SS>::SMEM_BYTES, s, 1, mA, mA, mB, mB, mA, mA, mA, mA, mA, mA, p);
    CDX_CUDA(cudaGetLastError());
    e.launches++;
  }
  return true;
}

bool conv_halo_eligible(const Engine& e, int B, int H, int W, int C1, int C2, int Cout, bool out_nchw) {
  // Measured on B200 (profiles/r02_gn_fusion_negative.txt): parity holds (89 GPU tests), GroupNorm time 1.73 -> 1.01 ms per SD
  // U-Net call, but conv3x3 8.6 -> 13.8 ms: every N tile of a conv re-applies the norm and the SiLU (two MUFU ops per element) while
  // converting its halo, which puts the split warps back on the critical path.  Opt-in (CDX_GN_FUSION=1) until the conversion is
  // shared between the N tiles of a row block.
  static const bool no_fuse = getenv("CDX_GN_FUSION") == nullptr;
  const long long M = (long long)B * H * W;
  if (no_fuse || e.mma_mode != 1 || e.tc_kind < 1 || !pow2(H) || !pow2(W) || (C1 % 64) || (C2 % 64) || M < 64) return false;
  if ((Cout < 32 && M < 2048) || (!out_nchw && (Cout & 3))) return false;       // (the shapes gemm_tc leaves to the FFMA tiles)
  const int bw = W < 16 ? W : 16;
  const int bh = H < TBM / bw ? H : TBM / bw;
  const int bn = TBM / (bw * bh);
  return bn == 1 && (bw + 2) * (bh + 2) * 128 <= HALO_PLANE_1CTA;
}

bool gemm_tc(Engine& e, const GemmArgs& a, cudaStream_t s, int* side_done) {
  // ---- eligibility (everything else takes the FFMA tiles)
  if (a.batch * a.heads != 1 || a.b_kn) return false;
  if (a.geglu && ((a.N % TBN) || a.out_nchw || a.Cout_lo || a.residual || a.rowvec || a.mode != 0)) return false;
  if (a.Cout_lo && a.out_nchw) return false;
  if (a.Ct_hi && (a.mode != 0 || !a.Ct_lo || a.out_nchw || a.geglu || a.residual || a.rowvec || (a.t_col0 % TBN) || a.t_col0 >= a.N)) return false;
  if (a.out_nchw && (a.rowvec || a.residual)) return false;
  if (!a.out_nchw && ((a.N & 3) || (a.ldc & 3) || !a16(a.Cout))) return false;   // (the NCHW epilogue stores scalars: any N)
  if (!a16(a.Bw) || (a.ldb & 3)) return false;
  if (a.rowvec && (!a16(a.rowvec) || (a.ld_rowvec & 3))) return false;
  if (a.residual && (!a16(a.residual) || (a.ldr & 3))) return false;
  if (!a16(a.A) || (a.lda & 3)) return false;
  if (a.M < 64) return false;
  if (a.N < 32 && a.M < 2048) return false;         // tiny problems: tile quantisation loses to the FFMA 64x64 tiles; thin-N with a
                                                    // large M (e.g. the 320 -> 4 output conv) still wins by a wide margin

  TcParams p;
  memset(&p, 0, sizeof(p));
  p.M = a.M; p.N = a.N; p.K = a.K;
  p.C = a.Cout; p.ldc = a.ldc;
  p.C_lo = a.out_nchw ? nullptr : a.Cout_lo;
  p.Ct_hi = a.Ct_hi; p.Ct_lo = a.Ct_lo; p.t_col0 = a.t_col0; p.ldt = a.ldt;
  p.bias = a.bias;
  p.rowvec = a.rowvec; p.ld_rowvec = a.ld_rowvec; p.rows_per_batch = a.rows_per_batch > 0 ? a.rows_per_batch : 1;
  p.residual = a.residual; p.ldr = a.ldr;
  p.alpha = a.alpha;
  p.geglu = a.geglu;
  p.out_nchw = a.out_nchw; p.rows_per_img = a.rows_per_img > 0 ? a.rows_per_img : 1;
  p.heads = 1;
  const CUtensorMap *mA, *mA2, *mB, *mBlo;
  if (a.mode == 0) {
    if (a.K & 3) return false;
    if (a.A2) {
      if ((a.C1 % TBK) || !a16(a.A2) || (a.lda2 & 3) || (a.C2 & 3)) return false;
    }
    p.mode = 0; p.C1 = a.C1; p.C2 = a.C2;
    {
      uint64_t d[2] = {(uint64_t)a.C1, (uint64_t)a.M}, st[1] = {(uint64_t)a.lda * 4};
      uint32_t bx[2] = {TBK, TBM};
      mA = &get_map(a.A, 2, d, st, bx);
    }
    if (a.A2) {
      uint64_t d[2] = {(uint64_t)a.C2, (uint64_t)a.M}, st[1] = {(uint64_t)a.lda2 * 4};
      uint32_t bx[2] = {TBK, TBM};
      mA2 = &get_map(a.A2, 2, d, st, bx);
    } else {
      mA2 = mA;
    }
    p.tiles_m = cdiv(a.M, TBM);
  } else {
    const int Cin = a.C1 + (a.A2 ? a.C2 : 0);
    if ((a.stride != 1 && a.stride != 2) || a.up != 1) return false;
    if (Cin % TBK) return false;
    // a channel-concat input or a fused GroupNorm exists only on the halo schedule; the caller asks conv_halo_eligible() first
    const bool needs_halo = a.A2 != nullptr || a.gn_ab != nullptr;
    CDX_CHECK(!a.A2 || a.gn_ab, "conv3x3: a channel-concat input is only supported together with the fused GroupNorm");
    if (a.Hin != a.Hout * a.stride || a.Win != a.Wout * a.stride || !pow2(a.Hout) || !pow2(a.Wout)) return false;
    const int B = a.M / (a.Hout * a.Wout);
    int bw = a.Wout < 16 ? a.Wout : 16;
    int bh = a.Hout < TBM / bw ? a.Hout : TBM / bw;
    int bn = TBM / (bw * bh);
    if (bn > 256 || bw * a.stride > 256 || bh * a.stride > 256) return false;
    p.mode = 1; p.Cin = Cin; p.H = a.Hout; p.W = a.Wout; p.B = B;      // H, W: OUTPUT grid (tile -> row mapping)
    p.bw = bw; p.bh = bh; p.bn = bn;
    p.cstride = a.stride; p.cpad = a.pad;
    p.tiles_x = a.Wout / bw; p.tiles_y = a.Hout / bh;
    uint64_t d[4] = {(uint64_t)a.C1, (uint64_t)a.Win, (uint64_t)a.Hin, (uint64_t)B};
    uint64_t st[3] = {(uint64_t)a.lda * 4, (uint64_t)a.lda * 4 * a.Win, (uint64_t)a.lda * 4 * a.Win * a.Hin};
    // stride 2 (Downsample convs): TMA traverses every 2nd pixel; box = 2x the number of pixels wanted
    uint32_t bx[4] = {TBK, (uint32_t)(bw * a.stride), (uint32_t)(bh * a.stride), (uint32_t)bn};
    uint32_t es[4] = {1, (uint32_t)a.stride, (uint32_t)a.stride, 1};
    // halo schedule (see TcParams::halo): needs the fp16-split path (decided below), 64-channel blocks and a halo box that fits a plane
    static const bool no_halo = getenv("CDX_TC_NO_HALO") != nullptr;
    // (the pair kernel has room for a 25 KB plane: the 8 x 8 level, two images per tile, joins the halo schedule when the launch pairs)
    static const bool no_pair = getenv("CDX_TC_NO_PAIR") != nullptr;
    const bool will_pair = !no_pair && ((p.tiles_x * p.tiles_y * cdiv(B, bn)) % 2) == 0 && e.num_sms >= 2;
    const int plane_cap = will_pair ? HALO_PLANE_PAIR : HALO_PLANE_1CTA;
    if ((!no_halo || needs_halo) && e.tc_kind >= 1 && a.stride == 1 && a.pad == 1 && (a.C1 % 64) == 0 && (!a.A2 || (a.C2 % 64) == 0) &&
        (bw + 2) * (bh + 2) * bn * 128 <= plane_cap && a.Bw_h_hi && a.Bw_h_lo && a16(a.Bw_h_hi) && a16(a.Bw_h_lo) && (a.ldb % 8) == 0 &&
        (!a.gn_ab || bn == 1)) {
      p.halo = 1;
      bx[1] = (uint32_t)(bw + 2); bx[2] = (uint32_t)(bh + 2);
    }
    CDX_CHECK(p.halo || !needs_halo, "conv3x3: a concat input / fused GroupNorm needs the halo schedule (C1=%d C2=%d %dx%d): check conv_halo_eligible() first",
              a.C1, a.C2, a.Hout, a.Wout);
    p.C1 = a.C1;
    p.gn_ab = reinterpret_cast<const float2*>(a.gn_ab); p.gn_silu = a.gn_silu;
    mA = &get_map(a.A, 4, d, st, bx, es);
    mA2 = mA;
    if (a.A2) {
      CDX_CHECK(a16(a.A2) && (a.lda2 & 3) == 0, "conv3x3: misaligned second source");
      uint64_t d2[4] = {(uint64_t)a.C2, (uint64_t)a.Win, (uint64_t)a.Hin, (uint64_t)B};
      uint64_t st2[3] = {(uint64_t)a.lda2 * 4, (uint64_t)a.lda2 * 4 * a.Win, (uint64_t)a.lda2 * 4 * a.Win * a.Hin};
      mA2 = &get_map(a.A2, 4, d2, st2, bx, es);
    }
    p.tiles_m = p.tiles_x * p.tiles_y * cdiv(B, bn);
  }
  // ---- operand path: fp16-split (MODE_H16) when the engine selects it, the weights have fp16 planes and the geometry allows it
  // (K a multiple of 32: the stage's two 32-float A sub-blocks; fp16 B rows 16-byte aligned); else TF32 planes (MODE_TS); else SS
  const bool ts = a.Bw_hi != nullptr && a.Bw_lo != nullptr && a16(a.Bw_hi) && a16(a.Bw_lo);
  const bool h16 = e.tc_kind >= 1 && a.Bw_h_hi && a.Bw_h_lo && a16(a.Bw_h_hi) && a16(a.Bw_h_lo) && (a.K % TBK) == 0 && (a.ldb % 8) == 0 &&
                   (a.mode == 1 || !a.A2 || (a.C2 % TBK) == 0);
  CDX_CHECK(!(a.mode == 1 && (a.A2 || a.gn_ab)) || h16, "conv3x3: concat / fused GroupNorm input without the fp16-split path");
  if (p.halo && !h16) return false;        // (cannot happen: the halo conditions imply the fp16-split conditions)
  const int bk = h16 ? Cfg<MODE_H16>::BK : TBK;
  const int num_kb = cdiv(a.K, bk);
  // CTA pairs (MODE_H16X2): two adjacent 128-row tiles share one B tile, half of it in each CTA's shared memory
  // Measured on B200: the single-CTA kernel saturates the SM's shared-memory pipe (TMA fill of B + tensor-core fetch of B + the
  // split warps' LDS = ~93 % of its cycles in the ncu capture); the pair halves the first two.  conv3x3 330 -> 420-480 TFLOP/s
  // (profiles/r02_ops_h16_pair.txt).  The first pair version used cluster-scope acquire / release on the per-stage barriers and
  // ran at 0.6x: ptxas puts an L1 invalidation (CCTL.IVALL) behind each of them (profiles/r02_ops_h16_pair_negative.txt).
  static const bool no_cg2 = getenv("CDX_TC_NO_PAIR") != nullptr;
  const bool cg2 = h16 && !no_cg2 && (p.tiles_m % 2) == 0 && e.num_sms >= 2;
  CDX_CHECK(!p.halo || cg2 || (p.bw + 2) * (p.bh + 2) * p.bn * 128 <= HALO_PLANE_1CTA, "conv3x3: halo plane sized for the pair kernel on a single-CTA launch");
  if (cg2) p.tiles_m /= 2;                 // from here on: 256-row pair tiles
  // Work partition: tile width w along N (MMA N = valid columns rounded up to 16, so a ragged last tile costs only its
  // share) and split-K factor S, chosen together against wave quantisation on num_sms persistent CTAs by replaying the
  // kernel's static schedule (CTA c runs items c, c + grid, ...) with a cost model in cycles: one k-block of a w-wide
  // tile ~ 540 + 4.2 w (fitted on B200: ~1080 at w = 128, 0.80x at w = 80 -- the A-side work of a k-block does not shrink
  // with w), ~5000 per work item for drain + epilogue, plus the split-K
  // partial-sum traffic (S writes + S reads + 1 write of M*N floats at ~4 TB/s); a split must buy >= 10 %.
  int best_w = TBN, best_s = 1;
  {
    static const bool fixed_w = getenv("CDX_TC_FIXED_W") != nullptr;      // tuning aid: always 128-wide tiles
    static std::map<std::array<int64_t, 5>, int> plan_cache;      // exact key (no hashing of packed fields: nothing can collide)
    static std::mutex plan_mutex;                                          // engines on different devices may plan concurrently
    std::lock_guard<std::mutex> plan_lock(plan_mutex);
    const std::array<int64_t, 5> key = {p.tiles_m, a.N, num_kb, ((a.geglu || a.Ct_hi) ? 1 : 0) | (a.out_nchw ? 2 : 0) | (h16 ? 4 : 0) | (p.halo ? 8 : 0) | (cg2 ? 16 : 0), e.num_sms};
    // cycles per pipeline stage of a w-wide tile (fitted on B200): TF32 planes 540 + 4.2 w per 32 k; fp16 split per 64 k
    const double kc0 = h16 ? CDX_H16_KC0 : 540.0, kc1 = h16 ? CDX_H16_KC1 : 4.2;
    const int min_kbs = h16 ? 4 : 8;
    auto it = plan_cache.find(key);
    if (it != plan_cache.end()) {
      best_w = it->second >> 8;
      best_s = it->second & 255;
    } else {
      const int wmin = (a.geglu || a.Ct_hi || a.N <= 64 || fixed_w) ? TBN : 64;
      const int G = cg2 ? e.num_sms / 2 : e.num_sms;      // persistent CTAs (pair mode: clusters)
      double best = 1e30;
      std::vector<double> load((size_t)G);
      for (int w = TBN; w >= wmin; w -= 16) {
        const int tn = cdiv(a.N, w);
        const int wl = ((a.N - (tn - 1) * w + 15) >> 4) << 4;               // MMA width of the last column tile
        double base = 0.0;
        for (int S = 1; S <= 8; ++S) {
          const int kbs = cdiv(num_kb, S);
          const int Sx = cdiv(num_kb, kbs);                                  // no empty splits
          if (S > 1 && (Sx != S || kbs < min_kbs || a.out_nchw || a.geglu || a.Ct_hi || (long long)p.tiles_m * tn >= 4LL * G)) continue;
          const long long items = (long long)p.tiles_m * tn * S;
          const int kb_last = num_kb - (S - 1) * kbs;
          double cost;
          if (items <= 200000) {
            const int g = (int)std::min<long long>(items, G);
            std::fill(load.begin(), load.end(), 0.0);
            for (long long t = 0; t < items; ++t) {                          // t -> (split fastest, then tm, then tn)
              const int sp = (int)(t % S);
              const int col = (int)((t / S / p.tiles_m) % tn);
              load[(size_t)(t % g)] += (sp == S - 1 ? kb_last : kbs) * (kc0 + kc1 * (col == tn - 1 ? wl : w)) + 5000.0;
            }
            cost = *std::max_element(load.begin(), load.begin() + g);
          } else {
            cost = (double)cdiv(items, (long long)G) * (kbs * (kc0 + kc1 * w) + 5000.0);
          }
          if (S == 1) base = cost;
          else cost += 4000.0 + (2.0 * S + 1.0) * (double)a.M * a.N * 4.0 / 4e12 * 1.9e9;
          if (cost < best - 1e-9 && (S == 1 || cost < 0.9 * base)) { best = cost; best_w = w; best_s = S; }
        }
      }
      plan_cache[key] = (best_w << 8) | best_s;
    }
  }
  p.tn_w = best_w;
  p.tiles_n = cdiv(a.N, best_w);
  const int tiles = p.tiles_m * p.tiles_n;
  p.splits = best_s;
  p.kb_per_split = cdiv(num_kb, best_s);
  p.splits = cdiv(num_kb, p.kb_per_split);            // no empty splits
  p.total_tiles = tiles * p.splits;
  Scope ws_scope(e.arena);
  if (best_s > 1) p.ws = (float*)e.arena.alloc((size_t)p.splits * a.M * a.N * sizeof(float));
  // fp16-split path: the A operand's range.  Tracked by its producer (a.a_amax), else measured here (one small extra launch).
  if (h16) {
    p.a_amax = a.a_amax;
    p.a2_amax = a.A2 ? a.a2_amax : nullptr;
    if (!p.a_amax && !p.gn_ab) {
      float* slot = e.amax_slot();
      if (a.mode == 1) amax_rows(e, a.A, (long long)(a.M / (a.Hout * a.Wout)) * a.Hin * a.Win, a.C1, a.lda, slot, s);
      else amax_rows(e, a.A, a.M, a.C1, a.lda, slot, s);
      p.a_amax = slot;
    }
    if (a.A2 && !p.a2_amax && !p.gn_ab && a.mode == 0) {
      float* slot = e.amax_slot();
      amax_rows(e, a.A2, a.M, a.C2, a.lda2, slot, s);
      p.a2_amax = slot;
    }
    p.b_exp = a.b_exp;
    p.fast = e.tc_kind == 2 ? 1 : 0;
  }
  // side outputs fused into the epilogue: range of C always (the split-K reduce kernel covers the split case); GroupNorm
  // statistics when every 32-row quadrant of a tile lies inside one image and the epilogue is the final one
  p.c_amax = a.out_nchw ? nullptr : a.c_amax;
  const bool quad_ok = a.mode == 1 ? ((p.bw * p.bh) % 32 == 0) : (a.rows_per_batch % 32 == 0);
  p.c_stats = (a.c_stats && quad_ok && p.splits == 1 && !a.out_nchw && !a.geglu && !a.Ct_hi && !a.Cout_lo && a.ldc == a.N) ? a.c_stats : nullptr;
  if (side_done) *side_done = (p.c_amax ? 1 : 0) | (p.c_stats ? 2 : 0);
  if (e.dry()) return true;
  static const int grid_cap = getenv("CDX_TC_GRID") ? atoi(getenv("CDX_TC_GRID")) : 0;      // experiment aid: run on fewer SMs
  const int grid = cg2 ? 2 * std::min(p.total_tiles, (grid_cap > 0 ? std::min(grid_cap, e.num_sms) : e.num_sms) / 2)
                       : std::min(p.total_tiles, grid_cap > 0 ? std::min(grid_cap, e.num_sms) : e.num_sms);
  if (h16) {
    uint64_t d[2] = {(uint64_t)a.K, (uint64_t)a.N}, st[1] = {(uint64_t)a.ldb * 2};
    uint32_t bx[2] = {(uint32_t)Cfg<MODE_H16>::BK, (uint32_t)(cg2 ? p.tn_w / 2 : p.tn_w)};
    mB = &get_map(a.Bw_h_hi, 2, d, st, bx, nullptr, 2);
    mBlo = &get_map(a.Bw_h_lo, 2, d, st, bx, nullptr, 2);
  } else {
    uint64_t d[2] = {(uint64_t)a.K, (uint64_t)a.N}, st[1] = {(uint64_t)a.ldb * 4};
    uint32_t bx[2] = {TBK, (uint32_t)p.tn_w};
    mB = &get_map(ts ? a.Bw_hi : a.Bw, 2, d, st, bx);
    mBlo = ts ? &get_map(a.Bw_lo, 2, d, st, bx) : mB;
  }
  // TMA epilogue (TcParams::epi_tma): dense layers whose epilogue is the final one and needs no per-column statistics
  const CUtensorMap *mC = mA, *mClo = mA, *mR = mA, *mC16 = mA, *mClo16 = mA, *mR16 = mA;
  static const bool no_epi_tma = getenv("CDX_TC_NO_EPI_TMA") != nullptr;
  bool tail16 = false;
  if (!no_epi_tma && h16 && a.mode == 0 && !a.out_nchw && p.splits == 1 && a.M >= TBM) {       // (compiled into the fp16-split kernels only)
    const uint64_t nc = (uint64_t)(a.geglu ? a.N / 2 : a.N);
    uint64_t d[2] = {nc, (uint64_t)a.M}, st[1] = {(uint64_t)a.ldc * 4};
    uint32_t bx[2] = {32, 32}, bx16[2] = {16, 32};
    tail16 = (p.tn_w & 31) != 0 || ((a.N % p.tn_w) & 31) != 0;      // some warp stores a 16-column tail slot
    mC = &get_map(a.Cout, 2, d, st, bx);
    if (tail16) mC16 = &get_map(a.Cout, 2, d, st, bx16, nullptr, 4, 64);
    if (p.C_lo) {
      mClo = &get_map(p.C_lo, 2, d, st, bx);
      if (tail16) mClo16 = &get_map(p.C_lo, 2, d, st, bx16, nullptr, 4, 64);
    }
    if (a.residual) {
      uint64_t sr[1] = {(uint64_t)a.ldr * 4};
      mR = &get_map(a.residual, 2, d, sr, bx);
      if (tail16) mR16 = &get_map(a.residual, 2, d, sr, bx16, nullptr, 4, 64);
    }
    p.epi_tma = 1;
  }
  e.last_gemm = cdx_gemm_plan{h16 ? (cg2 ? CDX_GEMM_H16_PAIR : CDX_GEMM_H16) : ts ? CDX_GEMM_TS : CDX_GEMM_SS, p.halo, p.epi_tma, p.tn_w, p.splits,
                              tail16 ? 1 : 0, (p.c_amax ? 1 : 0) | (p.c_stats ? 2 : 0)};
  ensure_attr(e.device);
  ProfScope ps(e, s, a.mode == 1 ? PROF_CONV_TC : PROF_DENSE_TC, 2.0 * a.M * a.N * a.K,
               4.0 * ((double)a.M * a.K / (a.mode == 1 ? 9 : 1) + (double)a.N * a.K + (double)a.M * a.N), 1);
  ps.note("M%d N%d K%d w%d tiles%d S%d %s%s%s%s", a.M, a.N, a.K, p.tn_w, tiles, p.splits, h16 ? (p.fast ? "H16x1" : p.halo ? (cg2 ? "H16halo-pair" : "H16halo") : (cg2 ? "H16-pair" : "H16")) : ts ? "TS" : "SS",
          a.Cout_lo ? " planes" : "", a.geglu ? " geglu" : "", a.residual ? " res" : "");
  if (cg2 && p.epi_tma) launch_ex(tc_gemm_kernel<MODE_H16X2, true>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_H16X2>::SMEM_BYTES, s, 2, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  else if (cg2) launch_ex(tc_gemm_kernel<MODE_H16X2, false>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_H16X2>::SMEM_BYTES, s, 2, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  else if (h16 && p.epi_tma) launch_ex(tc_gemm_kernel<MODE_H16, true>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_H16>::SMEM_BYTES, s, 1, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  else if (h16) launch_ex(tc_gemm_kernel<MODE_H16, false>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_H16>::SMEM_BYTES, s, 1, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  else if (ts) launch_ex(tc_gemm_kernel<MODE_TS, false>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_TS>::SMEM_BYTES, s, 1, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  else launch_ex(tc_gemm_kernel<MODE_SS, false>, dim3((unsigned)grid), dim3(TC_THREADS), Cfg<MODE_SS>::SMEM_BYTES, s, 1, *mA, *mA2, *mB, *mBlo, *mC, *mClo, *mR, *mC16, *mClo16, *mR16, p);
  CDX_CUDA(cudaGetLastError());
  e.launches++;
  if (p.splits > 1) {
    const long long total4 = (long long)a.M * a.N / 4;
    const int blocks = (int)std::min<long long>((total4 + 255) / 256, (long long)e.num_sms * 8);
    launch_ex(splitk_reduce_kernel, dim3((unsigned)blocks), dim3(256), 0, s, 1, p.ws, p.splits, p, h16 ? 1 : 0);
    CDX_CUDA(cudaGetLastError());
    e.launches++;
  }
  return true;
}

}  // namespace cdx
