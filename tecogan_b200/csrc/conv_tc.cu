// bf16 3x3 convolution / 3x3-stride-2 transposed convolution on the 5th-gen tensor cores (sm_100a):
// TMA halo tiles -> shared memory -> tcgen05.mma (kind::f16, fp32 accumulators in TMEM) -> tcgen05.ld
// epilogue (bias, activation, residual, bf16 store; or fp32 "+bicubic, *2-1" output stage).
//
// Replaces, layer by layer, the cuDNN convolutions behind conv2()/conv2_tran() of the reference
// (lib/ops.py:35-56) as used by generator_F (lib/frvsr.py:44-88) and fnet (lib/frvsr.py:4-41).
//
// Implicit GEMM, no im2col buffer:
//   CTA tile  = 16 image rows x (8*J) pixels; every 16x8 sub-tile is one UMMA accumulator with M = 128.
//   A operand = NHWC bf16 activations, 64 channels = one 128-byte row per pixel.  Per 64-channel block the halo is
//               staged by ONE 4-D TMA box (64 ch, 8J+2 px, 18 rows, 1 image) with SWIZZLE_128B, which is the UMMA
//               canonical K-major SW128 layout as it lands (SBO = one box row).  All nine taps are descriptor start
//               offsets into it: vertical taps ky whole box rows, horizontal taps kx 128-byte pixel rows (not
//               swizzle-atom aligned: the SW128 XOR is a function of the absolute shared-memory address bits, which is
//               also how TMA wrote the box; the descriptor's base-offset field stays 0 -- setting it to (addr >> 7) & 7
//               was tested on the B200 and gives wrong results).  TMA out-of-bounds zero fill implements TF 'SAME' padding.
//   B operand = weights pre-packed on the device as [cin/64][tap][cout][64 cin] bf16 in the same SW128 image,
//               streamed by 1-D bulk copies.  When a whole layer fits (64->64: 72 KB) the slabs are fetched once,
//               BEFORE the programmatic-dependent-launch wait (the one-tile kernel also multicasts them over a 4-CTA cluster).
//   D         = fp32 in TMEM, column block (sub-tile, phase) * Cout.
// Transposed conv (stride 2, TF 'SAME', y[i] = sum_j x[j] w[i-2j]) is the same loop with the nine taps routed to
// four sub-pixel phase accumulators (SURVEY.md A.3) and a 2x interleaving epilogue.
//
// Why SW128 and not the no-swizzle layout (round-1 measurement, profiles/conv_tc_r01_notes.md): with 16-byte core
// matrix rows every tcgen05.mma took ~250 cycles instead of ~32-48, and the 16-byte TMA rows ran at ~10 B/clk/SM.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..9 = epilogue
// (one epilogue warp per scheduler is latency-bound: ~1000 clk per 32 channels; two per scheduler halve it).
#include <type_traits>
#include "conv_tc_common.cuh"

namespace {

constexpr int NUM_EPI_WARPS = 8;      // two warps per TMEM lane quarter, each taking half of the output channels
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS + 32;   // + the output-store warp (staged epilogue)
constexpr int STORE_WARP = 2 + NUM_EPI_WARPS;

struct TcParams {
  int N, H, W, Cin, Cout;             // Cout = channel pitch of y / res / bias (all output channels)
  int Ncta, nsplit, G, AS;            // output channels per CTA (UMMA N), Cout splits, CTAs per split (persistent: each
                                      // walks tiles c, c+G, ...), TMEM accumulator stages (1 or 2)
  int tiles_x, tiles_y, J;
  int mode, act, out_f32_c;
  float post_scale, post_shift;
  int nblk, WST, TPS, KS;              // Cin/64, weight ring stages, taps per weight slab (1 or 3), K-split chains
  int HST, mcast, num_tiles;           // halo stages, resident weights, real tile count
  uint32_t halo_stage_bytes, w_slab_bytes, tmem_cols;
  int tma_out, tma_res;                // staged epilogue: bf16 output / residual tiles through swizzled smem + TMA (see conv_tc_sw.cu)
  const uint8_t* wpk;
  const float* bias;
  const __nv_bfloat16* res;
  __nv_bfloat16* y;
  const float* res_f32;
  float* out_f32;
  long long* dbg;                      // optional [gridDim][32] clock64 stamps (teco_debug_timing)
};

using namespace tcptx;   // mbarrier / TMA / tcgen05 wrappers and the UMMA descriptors: tc_ptx.cuh

// ------------------------------------------------------------------ the kernel
// MODE 0 conv / 1 transposed conv; TPS taps per weight slab; J sub-tiles per CTA; KS K-split accumulator chains.
// They are compile-time so that the MMA issue loop is a fully unrolled stream of UTCHMMA whose descriptors differ
// from per-stage bases by immediates (uniform-datapath adds, no per-instruction R2UR).
//
// Persistent and pipelined: a CTA walks tiles c, c+G, c+2G, ... of its Cout split.  The halo ring (HST stages), the
// weight ring (or the resident layer, loaded once) and AS TMEM accumulator stages let the TMA producer, the MMA
// issuer and the epilogue warps work on three different tiles at the same time.
template <int MODE, int TPS, int J, int KS>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_y,
                  const __grid_constant__ CUtensorMap tmap_r, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  uint8_t* halo_base = smem;                                             // HST halo stages
  uint8_t* w_base = smem + (size_t)p.HST * p.halo_stage_bytes;           // WST weight slabs
  uint64_t* bars = reinterpret_cast<uint64_t*>(w_base + (size_t)p.WST * p.w_slab_bytes);
  uint64_t* halo_full = bars;                    // [MAX_HST]
  uint64_t* halo_empty = bars + MAX_HST;         // [MAX_HST]
  uint64_t* w_full = bars + 2 * MAX_HST;         // [MAX_WST]
  uint64_t* w_empty = w_full + MAX_WST;          // [MAX_WST]
  uint64_t* acc_full = w_empty + MAX_WST;        // [2]
  uint64_t* acc_empty = acc_full + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* s_bias = reinterpret_cast<float*>(acc_empty + 3);   // [Ncta]
  uint64_t* res_full = acc_empty + 3 + 128;      // [2] after 256 floats of bias
  uint64_t* stage_free = res_full + 2;           // [4] the TMA store of this staging tile has finished reading it
  uint64_t* out_full = res_full + 6;             // [4] all epilogue warps have written their part of the staging tile
  // Staged epilogue: two staging tiles (tile it uses it & 1), each J x [128 pixels][128 B] in the SWIZZLE_128B image of the
  // TMA box (64 ch, 8 px, 16 rows).  A residual tile is TMA-loaded INTO the staging tile and the epilogue adds in place
  // (same thread, same address), so residual and output share one buffer and both are double-buffered.
  // Transposed conv (MODE 1, J == 1): four staging tiles, one per output phase (each the 16x8 pixels of that phase).
  uint8_t* stage_base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(res_full + 10) + 1023) & ~(uintptr_t)1023);

  // work assignment: grid = nsplit x G CTAs; CTA c of a split owns tiles c, c+G, ...
  const int c_in_split = blockIdx.x % p.G;
  const int n0 = (blockIdx.x / p.G) * p.Ncta;   // first output channel of this CTA
  const int my_tiles = c_in_split < p.num_tiles ? (p.num_tiles - c_in_split + p.G - 1) / p.G : 0;
  long long* dbg = p.dbg ? p.dbg + (size_t)blockIdx.x * 64 : nullptr;   // [0,32) phase stamps, [32,64) per-tile stamps
#define STAMP(i) do { if (dbg) dbg[i] = clock64(); } while (0)
#define TSTAMP(it, i) do { if (dbg && (it) < 8) dbg[32 + (it) * 4 + (i)] = clock64(); } while (0)
  if (threadIdx.x == 0) STAMP(0);

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.HST; ++i) {
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_empty[i]), 1);
    }
    for (int i = 0; i < p.WST; ++i) {
      mbar_init(smem_u32(&w_full[i]), 1);
      mbar_init(smem_u32(&w_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&acc_full[i]), 1);
      mbar_init(smem_u32(&acc_empty[i]), NUM_EPI_WARPS);
    }
    for (int i = 0; i < 4; ++i) {
      if (i < 2) mbar_init(smem_u32(&res_full[i]), 1);
      mbar_init(smem_u32(&stage_free[i]), 1);
      mbar_init(smem_u32(&out_full[i]), NUM_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    if (p.tma_out) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_y) : "memory");
    if (p.tma_res) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_r) : "memory");
  }
  if (warp == 1) {  // TMEM allocation (one full warp), result lands in smem
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  pdl_launch_dependents();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) STAMP(1);

  // MODE 2 ("kx-fused" conv for a narrow output: Cout padded to 16): ONE tcgen05.mma covers the three horizontal taps of a
  // kernel row -- B = [3 taps x Ncta] rows (the packed slab of row ky as it is), N = 3*Ncta, A = the halo pixels of the
  // sub-tile WITHOUT a horizontal shift.  D block kx at halo column c then holds tap kx's contribution to output column
  // c - kx, and the epilogue forms out(x) = D0(x) + D1(x+1) + D2(x+2) with warp shuffles.  A tile is 8J halo columns wide and
  // yields 8J-2 output columns.  Why: an MMA costs ~60 clk whatever N is (the 4 KB A tile read bounds it), so the 64->3
  // output stage at HR resolution used to cost as much per pixel as a 64->64 layer; this needs 12 MMAs per sub-tile, not 36.
  constexpr int nacc = MODE == 1 ? 4 : (MODE == 2 ? 3 : 1);
  constexpr int slabs_per_blk = 9 / TPS;
  constexpr int row_bytes = (MODE != 2 ? 8 * J + 2 : 8 * J) * 128;           // one box row (pixels x 128 B)
  constexpr int tile_w = MODE == 2 ? 8 * J - 2 : 8 * J;                      // output columns per tile
  constexpr uint32_t copy_bytes = (uint32_t)(HALO_ROWS * row_bytes);
  const int slabs_per_tile = slabs_per_blk * p.nblk;
  const uint32_t acc_stage_cols = (uint32_t)(J * nacc * KS * p.Ncta);   // TMEM columns of one accumulator stage

  auto tile_coords = [&](int it, int& n, int& y0, int& x0) {
    int tile = c_in_split + it * p.G;
    const int tx = tile % p.tiles_x;
    tile /= p.tiles_x;
    const int ty = tile % p.tiles_y;
    n = tile / p.tiles_y;
    x0 = tx * tile_w;
    y0 = ty * TILE_ROWS;
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Issue cost of one bulk/tensor copy is a few hundred cycles, so independent copies are issued by different lanes.
    // Resident weights (whole layer fits): they do not depend on the previous layer -> fetch them once, before the
    // dependency wait.
    if (p.mcast) fetch_resident_weights<TPS>(lane, slabs_per_tile, p.wpk, p.Cout, n0, p.w_slab_bytes, w_base, w_full, 1);
    // Ring mode: slab sequence q = 0 .. my_tiles*slabs_per_tile-1 through WST stages; the first WST do not depend on
    // the previous layer either -> issue them before the wait.
    const int total_slabs = my_tiles * slabs_per_tile;
    int next_slab = 0;
    auto issue_slab = [&](int q) {
      const int st = q % p.WST, use = q / p.WST, sl = q % slabs_per_tile;
      const int b = sl / slabs_per_blk, g = sl - slabs_per_blk * b;
      if (use > 0) mbar_wait(smem_u32(&w_empty[st]), (uint32_t)((use - 1) & 1));   // MMAs of the previous use have retired
      mbar_expect_tx(smem_u32(&w_full[st]), p.w_slab_bytes);
      const uint8_t* src = p.wpk + ((size_t)(b * 9 + g * TPS) * p.Cout + n0) * 128;
      bulk_load_1d(smem_u32(w_base + (size_t)st * p.w_slab_bytes), src, p.w_slab_bytes, smem_u32(&w_full[st]));
    };
    if (!p.mcast && lane == 0)
      for (; next_slab < total_slabs && next_slab < p.WST; ++next_slab) issue_slab(next_slab);
    if (lane == 0) STAMP(9);
    pdl_wait();   // the previous kernel's output (our input x) is complete and visible from here on
    if (lane == 0) STAMP(10);
    int hs = 0;
    uint32_t hph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      int n, y0, x0;
      tile_coords(it, n, y0, x0);
      for (int b = 0; b < p.nblk; ++b) {
        if (lane == 0) {
          mbar_wait(smem_u32(&halo_empty[hs]), hph ^ 1);
          mbar_expect_tx(smem_u32(&halo_full[hs]), copy_bytes);
        }
        __syncwarp();
        if (lane == 0)
          tma_load_4d(smem_u32(halo_base + (size_t)hs * p.halo_stage_bytes), &tmap, smem_u32(&halo_full[hs]), b * CB, x0 - 1, y0 - 1, n);
        if (!p.mcast && lane == 0)   // slabs up to the end of this block that are not in flight yet
          for (; next_slab < it * slabs_per_tile + (b + 1) * slabs_per_blk; ++next_slab) issue_slab(next_slab);
        __syncwarp();
        if (++hs == p.HST) { hs = 0; hph ^= 1; }
      }
      if (p.tma_res) {   // residual tile(s) of this output tile straight into staging tile it & 1: free once the store of tile it - 2 has read it
        const int sg = it & 1;
        if (lane == 0) {
          mbar_wait(smem_u32(&stage_free[sg]), (uint32_t)(((it >> 1) & 1) ^ 1));
          mbar_expect_tx(smem_u32(&res_full[sg]), (uint32_t)(J * 16384));
        }
        __syncwarp();
        if (lane < J)
          tma_load_4d(smem_u32(stage_base + (size_t)(sg * J + lane) * 16384), &tmap_r, smem_u32(&res_full[sg]), n0, x0 + 8 * lane, y0, n);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = umma_idesc(p.Ncta);
    constexpr uint32_t a_sbo = (uint32_t)row_bytes;   // next 8-pixel group of the M=128 sub-tile = next image row
    constexpr uint32_t b_sbo = 1024u;                 // next 8 output channels
    int hs = 0, ws = 0;
    uint32_t hph = 0, wph = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const int as = (p.AS == 2) ? (it & 1) : 0;
      const uint32_t ause = (uint32_t)((p.AS == 2) ? (it >> 1) : it);
      mbar_wait_warp(smem_u32(&acc_empty[as]), (ause & 1u) ^ 1u);   // the epilogue has drained this accumulator stage
      tcgen05_fence_after();
      const uint32_t tmem_acc = tmem_base + (uint32_t)as * acc_stage_cols;
      uint32_t started = 0;  // bit (j*nacc+phase): accumulator already written once (for this tile)
      for (int b = 0; b < p.nblk; ++b) {
        mbar_wait_warp(smem_u32(&halo_full[hs]), hph);
        tcgen05_fence_after();
        if (lane == 0 && b == 0 && it == 0) STAMP(2);
        if (lane == 0 && b == 0) TSTAMP(it, 0);
        const uint32_t halo_addr = smem_u32(halo_base + (size_t)hs * p.halo_stage_bytes);
        for (int g = 0; g < slabs_per_blk; ++g) {
          if (p.mcast) {   // resident: slab index is fixed, the barrier completes exactly once
            ws = b * slabs_per_blk + g;
            if (it == 0) mbar_wait_warp(smem_u32(&w_full[ws]), 0);
          } else {
            mbar_wait_warp(smem_u32(&w_full[ws]), wph);
          }
          tcgen05_fence_after();
          if (lane == 0 && b == 0 && it == 0) STAMP(16 + g);
          if (MODE == 2) {
            const uint32_t slab_addr = smem_u32(w_base + (size_t)ws * p.w_slab_bytes);
            const uint64_t a_row = umma_desc_sw128(halo_addr, a_sbo) + (uint64_t)((uint32_t)(g * row_bytes) >> 4);
            const uint64_t b3 = umma_desc_sw128(slab_addr, b_sbo);
            const uint32_t idesc3 = umma_idesc(3 * p.Ncta);
            const uint32_t first = (b == 0 && g == 0) ? 1u : 0u;
            if (elect_one()) {
#pragma unroll
              for (int s = 0; s < CB / 16; ++s)
#pragma unroll
                for (int j = 0; j < J; ++j)
                  umma_bf16(tmem_acc + (uint32_t)(j * 3) * (uint32_t)p.Ncta, a_row + (uint32_t)((j * 1024 + s * 32) >> 4),
                            b3 + (uint32_t)((s * 32) >> 4), idesc3, (first && s == 0) ? 0u : 1u);
            }
            __syncwarp();
          } else {
            // Whole (converged) warp computes the warp-uniform bases; one elected lane issues the unrolled MMA stream.
            const uint32_t slab_addr = smem_u32(w_base + (size_t)ws * p.w_slab_bytes);
            const uint64_t a_base = umma_desc_sw128(halo_addr, a_sbo);
            const uint64_t b_base = umma_desc_sw128(slab_addr, b_sbo);
            const uint32_t tap_stride16 = (uint32_t)(p.Ncta * 128) >> 4;   // weight bytes per tap, in descriptor units
            // per-tap row/copy/phase (TPS == 3: ky = g, kx = tt; TPS == 1: tap = g)
            uint32_t a_off16[TPS], acc_idx[TPS];
#pragma unroll
            for (int tt = 0; tt < TPS; ++tt) {
              const int t = g * TPS + tt;
              const int ky = (TPS == 3) ? g : t / 3, kx = (TPS == 3) ? tt : t - 3 * (t / 3);
              int ry, rx, phase;
              tap_route<MODE>(ky, kx, ry, rx, phase);
              a_off16[tt] = ((uint32_t)(rx * 128 + ry * row_bytes)) >> 4;
              acc_idx[tt] = (uint32_t)(phase * KS);   // first chain of this tap's accumulator
            }
            // K-split chain of an MMA: KS == 3 -> the tap within the slab (kx), KS == 2 -> parity of the k-step.
            // Order k-step, tap, sub-tile: consecutive MMAs hit J x KS different accumulators (dependent MMAs on one
            // accumulator cost ~125 cycles each; 3 chains ~72, 6 chains ~59: profiles/conv_tc_r01_notes.md).
            const uint32_t started_now = started;
            uint32_t touched = 0;
#pragma unroll
            for (int s = 0; s < CB / 16; ++s)
#pragma unroll
              for (int tt = 0; tt < TPS; ++tt)
#pragma unroll
                for (int j = 0; j < J; ++j)
                  touched |= 1u << ((uint32_t)(j * nacc * KS) + acc_idx[tt] + (uint32_t)(KS == 3 ? tt : (KS == 2 ? (s & 1) : 0)));
            if (elect_one()) {
              uint32_t seen = started_now;   // accumulators written so far (this tile); folds to constants when unrolled
#pragma unroll
              for (int s = 0; s < CB / 16; ++s) {
#pragma unroll
                for (int tt = 0; tt < TPS; ++tt) {
#pragma unroll
                  for (int j = 0; j < J; ++j) {
                    const uint32_t acc = (uint32_t)(j * nacc * KS) + acc_idx[tt] + (uint32_t)(KS == 3 ? tt : (KS == 2 ? (s & 1) : 0));
                    const uint32_t accum = (seen >> acc) & 1u;
                    seen |= 1u << acc;
                    umma_bf16(tmem_acc + acc * (uint32_t)p.Ncta, a_base + a_off16[tt] + (uint32_t)((j * 1024 + s * 32) >> 4),
                              b_base + tt * tap_stride16 + (uint32_t)((s * 32) >> 4), idesc, accum);
                  }
                }
              }
            }
            __syncwarp();
            started |= touched;
            if (!p.mcast && elect_one()) tcgen05_commit(smem_u32(&w_empty[ws]));  // frees the slab when these MMAs retire
          }
          __syncwarp();
          if (!p.mcast && ++ws == p.WST) { ws = 0; wph ^= 1; }
        }
        if (elect_one()) tcgen05_commit(smem_u32(&halo_empty[hs]));
        __syncwarp();
        if (++hs == p.HST) { hs = 0; hph ^= 1; }
      }
      if (elect_one()) tcgen05_commit(smem_u32(&acc_full[as]));
      if (lane == 0 && it == 0) STAMP(5);
      if (lane == 0) TSTAMP(it, 1);
      __syncwarp();
    }
  } else if (warp == STORE_WARP) {
    // ===================== output store (staged epilogue only) =====================
    if (MODE == 0 && p.tma_out && lane == 0) {
      for (int it = 0; it < my_tiles; ++it) {
        int n, y0, x0;
        tile_coords(it, n, y0, x0);
        const int sg = it & 1;
        mbar_wait(smem_u32(&out_full[sg]), (uint32_t)((it >> 1) & 1));   // every epilogue warp has fenced and arrived
        for (int j = 0; j < J; ++j) tma_store_4d(&tmap_y, smem_u32(stage_base + (size_t)(sg * J + j) * 16384), n0, x0 + 8 * j, y0, n);
        bulk_commit();
        bulk_wait_read();                                                 // the staging tile may be overwritten again
        mbar_arrive(smem_u32(&stage_free[sg]));
      }
    }
    if (MODE == 1 && p.tma_out && lane == 0) {
      for (int it = 0; it < my_tiles; ++it) {
        int n, y0, x0;
        tile_coords(it, n, y0, x0);
        for (int ph = 0; ph < 4; ++ph) {   // one 16x8-pixel box per sub-pixel phase through the 5-D map {C, px, x, py, n*H + y}
          mbar_wait(smem_u32(&out_full[ph]), (uint32_t)(it & 1));
          tma_store_5d(&tmap_y, smem_u32(stage_base + (size_t)ph * 16384), n0, ph & 1, x0, ph >> 1, n * p.H + y0);
          bulk_commit();
          bulk_wait_read();
          mbar_arrive(smem_u32(&stage_free[ph]));
        }
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..9) =====================
    for (int c = (int)threadIdx.x - 64; c < p.Ncta; c += 32 * NUM_EPI_WARPS) s_bias[c] = p.bias ? p.bias[n0 + c] : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(32 * NUM_EPI_WARPS) : "memory");   // the epilogue warps only
    pdl_wait();                                        // res / y belong to the dependency chain
    if (threadIdx.x == 64) STAMP(25);
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int chalf = (warp - 2) >> 2; // which half of the channel steps this warp takes (0 or 1)
    const int m = 32 * q + lane;       // accumulator row = pixel within the 16x8 sub-tile
    const int ry = m >> 3, rx = m & 7;
    const float act_slope = p.act == TECO_ACT_RELU ? 0.f : (p.act == TECO_ACT_LRELU02 ? 0.2f : 1.f);
    // EW output channels per step: 32 (two steps for 64 channels) or 16 (the 16-channel fp32 output stage)
    auto run = [&](auto ew_tag) {
      constexpr int EW = decltype(ew_tag)::value;
      for (int it = 0; it < my_tiles; ++it) {
        int n, y0, x0;
        tile_coords(it, n, y0, x0);
        const int as = (p.AS == 2) ? (it & 1) : 0;
        const uint32_t ause = (uint32_t)((p.AS == 2) ? (it >> 1) : it);
        mbar_wait_warp(smem_u32(&acc_full[as]), ause & 1u);
        tcgen05_fence_after();
        if (threadIdx.x == 64 && it == 0) STAMP(6);
        if (threadIdx.x == 64) TSTAMP(it, 2);
        const uint32_t tmem_acc = tmem_base + (uint32_t)as * acc_stage_cols;
        const int oy_in = y0 + ry;
        for (int j = 0; j < J; ++j) {
          const int ox_in = x0 + 8 * j + rx;
          const bool in_img = (oy_in < p.H) && (ox_in < p.W);
          for (int ph = 0; ph < nacc; ++ph) {
            int oy, ox, OH, OW;
            if (MODE == 1) {
              oy = 2 * oy_in + (ph >> 1); ox = 2 * ox_in + (ph & 1); OH = 2 * p.H; OW = 2 * p.W;
            } else {
              oy = oy_in; ox = ox_in; OH = p.H; OW = p.W;
            }
            const size_t pix = ((size_t)n * OH + oy) * OW + ox;
            const uint32_t tcol = tmem_acc + ((uint32_t)(32 * q) << 16) + (uint32_t)((j * nacc + ph) * KS * p.Ncta);
            for (int c0 = chalf * EW; c0 < p.Ncta; c0 += 2 * EW) {
              uint32_t r[EW];
              __syncwarp();
              if (EW == 32) tmem_ld32(tcol + (uint32_t)c0, r); else tmem_ld16(tcol + (uint32_t)c0, r);
              if (KS == 3) {   // K-split chains: issue all the TMEM loads, wait once, add
                uint32_t r2[EW], r3[EW];
                if (EW == 32) { tmem_ld32(tcol + (uint32_t)(p.Ncta + c0), r2); tmem_ld32(tcol + (uint32_t)(2 * p.Ncta + c0), r3); }
                else { tmem_ld16(tcol + (uint32_t)(p.Ncta + c0), r2); tmem_ld16(tcol + (uint32_t)(2 * p.Ncta + c0), r3); }
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < EW; ++i)
                  r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r2[i]) + __uint_as_float(r3[i]));
              } else if (KS == 2) {
                uint32_t r2[EW];
                if (EW == 32) tmem_ld32(tcol + (uint32_t)(p.Ncta + c0), r2); else tmem_ld16(tcol + (uint32_t)(p.Ncta + c0), r2);
                tmem_wait_ld();
#pragma unroll
                for (int i = 0; i < EW; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r2[i]));
              } else {
                tmem_wait_ld();
              }
              if (threadIdx.x == 64 && it == 0 && j == 0 && ph == 0 && c0 == 0) STAMP(11);
              // last TMEM read of this tile by this warp -> hand the accumulator stage back to the MMA issuer
              if (j == J - 1 && ph == nacc - 1 && c0 + 2 * EW >= p.Ncta) {
                tcgen05_fence_before();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[as])) : "memory");
              }
              float v[EW];
#pragma unroll
              for (int i = 0; i < EW; ++i) {
                const float a = __uint_as_float(r[i]) + s_bias[c0 + i];
                v[i] = fmaxf(a, a * act_slope);      // none: slope 1, relu: 0, lrelu: 0.2 -- no per-element branch
              }
              if (p.act >= TECO_ACT_TANH24) {        // uniform, outside the element loop; rare (FNet head).  Unrolled: a rolled
#pragma unroll                                       // loop indexes v[] dynamically and drags it into local memory for every layer
                for (int i = 0; i < EW; ++i) v[i] = teco_act(v[i], p.act);
              }
              if (!in_img) continue;
              if (p.out_f32) {
#pragma unroll
                for (int i = 0; i < EW; ++i) {
                  const int c = n0 + c0 + i;
                  if (c < p.out_f32_c) {
                    const float a = v[i] + (p.res_f32 ? p.res_f32[pix * p.out_f32_c + c] : 0.f);
                    p.out_f32[pix * p.out_f32_c + c] = a * p.post_scale + p.post_shift;
                  }
                }
              }
              if (p.y) {
                if (p.res) {
                  const uint4* rp = reinterpret_cast<const uint4*>(p.res + pix * p.Cout + n0 + c0);
#pragma unroll
                  for (int k = 0; k < EW / 8; ++k) add_bf16x8(v + 8 * k, rp[k]);
                }
                uint4* yp = reinterpret_cast<uint4*>(p.y + pix * p.Cout + n0 + c0);
#pragma unroll
                for (int k = 0; k < EW / 8; ++k) yp[k] = pack_bf16x8(v + 8 * k);
              }
              if (threadIdx.x == 64 && it == 0 && j == 0 && ph == 0) STAMP(12 + ((c0 / EW) & 3));
            }
          }
        }
        if (threadIdx.x == 64) TSTAMP(it, 3);
        // warps with no channel step of their own (16-channel output stage: chalf == 1) still release the stage
        if (chalf * EW >= p.Ncta) {
          if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[as])) : "memory");
        }
      }
    };
    if (MODE == 0 && p.tma_out) {
      // ---- staged epilogue (Ncta == 64): this warp owns channels [32*chalf, +32) of pixel row m of every sub-tile.
      // TMEM -> registers -> (+ bias, activation, + residual read from the staging tile) -> bf16 into the staging tile in
      // place; the store warp sends the tile out.  The TMEM loads of sub-tile 1 are in flight while sub-tile 0 is
      // processed (the epilogue was latency-bound: load -> wait -> math -> store per step, ~2300 clk per step).
      constexpr bool PREF = (J == 2 && KS <= 2);
      const uint32_t rowoff = (uint32_t)m * 128u, sw = (uint32_t)m & 7u;
      float bias_r[32];      // this thread's 32 output channels: registers, not a shared-memory read per tile (the L1/smem
#pragma unroll             // data pipe is what bounds this kernel: 48 operand wavefronts per N=64 MMA)
      for (int i = 0; i < 32; ++i) bias_r[i] = s_bias[32 * chalf + i];
      auto process = [&](uint32_t (&r)[KS][32], uint8_t* tile) {
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          float a = __uint_as_float(r[0][i]);
#pragma unroll
          for (int k = 1; k < KS; ++k) a += __uint_as_float(r[k][i]);
          a += bias_r[i];
          v[i] = fmaxf(a, a * act_slope);      // none: slope 1, relu: 0, lrelu: 0.2 -- no per-element branch
        }
        uint8_t* row = tile + rowoff;   // (tanh/sigmoid layers never take the staged path: a rolled loop would put v[] in local memory)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint4* cell = reinterpret_cast<uint4*>(row + ((((uint32_t)(4 * chalf + k)) ^ sw) << 4));   // XOR swizzle of the TMA box
          if (p.tma_res) add_bf16x8(v + 8 * k, *cell);
          *cell = pack_bf16x8(v + 8 * k);
        }
      };
      for (int it = 0; it < my_tiles; ++it) {
        const int as = (p.AS == 2) ? (it & 1) : 0;
        const uint32_t ause = (uint32_t)((p.AS == 2) ? (it >> 1) : it);
        const int sg = it & 1;
        const uint32_t suse = (uint32_t)(it >> 1);
        mbar_wait_warp(smem_u32(&acc_full[as]), ause & 1u);
        tcgen05_fence_after();
        if (threadIdx.x == 64 && it == 0) STAMP(6);
        if (threadIdx.x == 64) TSTAMP(it, 2);
        const uint32_t tb = tmem_base + (uint32_t)as * acc_stage_cols + ((uint32_t)(32 * q) << 16) + (uint32_t)(32 * chalf);
        auto release_acc = [&]() {     // last TMEM read of this tile by this warp -> hand the stage back to the MMA issuer
          tcgen05_fence_before();
          if (lane == 0) mbar_arrive(smem_u32(&acc_empty[as]));
        };
        uint8_t* tile0 = stage_base + (size_t)(sg * J) * 16384;
        uint32_t ra[KS][32];
#pragma unroll
        for (int k = 0; k < KS; ++k) tmem_ld32(tb + (uint32_t)(k * 64), ra[k]);
        tmem_wait_ld();
        if (PREF) {
          uint32_t rb[KS][32];
#pragma unroll
          for (int k = 0; k < KS; ++k) tmem_ld32(tb + (uint32_t)((KS + k) * 64), rb[k]);
          // the staging tile: residual landed (which implies it was free), or free of the store of tile it - 2
          if (p.tma_res) mbar_wait_warp(smem_u32(&res_full[sg]), suse & 1u);
          else mbar_wait_warp(smem_u32(&stage_free[sg]), (suse & 1u) ^ 1u);
          process(ra, tile0);
          tmem_wait_ld();
          release_acc();
          process(rb, tile0 + 16384);
        } else {
          if (J == 1) release_acc();
          if (p.tma_res) mbar_wait_warp(smem_u32(&res_full[sg]), suse & 1u);
          else mbar_wait_warp(smem_u32(&stage_free[sg]), (suse & 1u) ^ 1u);
          process(ra, tile0);
          if (J == 2) {
#pragma unroll
            for (int k = 0; k < KS; ++k) tmem_ld32(tb + (uint32_t)((KS + k) * 64), ra[k]);
            tmem_wait_ld();
            release_acc();
            process(ra, tile0 + 16384);
          }
        }
        fence_async_smem();            // generic-proxy writes -> visible to the TMA store
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&out_full[sg]));
        if (threadIdx.x == 64) TSTAMP(it, 3);
      }
    } else if (MODE == 2) {
      // ---- kx-fused narrow output stage (fp32 output, <= 4 channels): out(x) = D0(x) + D1(x+1) + D2(x+2)
      const int C = p.out_f32_c;
      for (int it = 0; it < my_tiles; ++it) {
        int n, y0, x0;
        tile_coords(it, n, y0, x0);
        const int as = (p.AS == 2) ? (it & 1) : 0;
        const uint32_t ause = (uint32_t)((p.AS == 2) ? (it >> 1) : it);
        mbar_wait_warp(smem_u32(&acc_full[as]), ause & 1u);
        tcgen05_fence_after();
        if (threadIdx.x == 64) TSTAMP(it, 2);
        const uint32_t tb = tmem_base + (uint32_t)as * acc_stage_cols + ((uint32_t)(32 * q) << 16);
        uint32_t d[J][3][4];
#pragma unroll
        for (int j = 0; j < J; ++j)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) tmem_ld4(tb + (uint32_t)((j * 3 + kx) * p.Ncta), d[j][kx]);
        tmem_wait_ld();
        tcgen05_fence_before();
        if (lane == 0) mbar_arrive(smem_u32(&acc_empty[as]));
        const int oy = y0 + ry;
#pragma unroll
        for (int j = 0; j < J; ++j) {
          float v[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            // neighbours one and two halo columns to the right: the same sub-tile (lane + 1, + 2) or the next one (lane - 7, - 6)
            const float s1 = __shfl_sync(0xffffffffu, __uint_as_float(d[j][1][c]), (lane + 1) & 31);
            const float s2 = __shfl_sync(0xffffffffu, __uint_as_float(d[j][2][c]), (lane + 2) & 31);
            float n1 = 0.f, n2 = 0.f;
            if (j + 1 < J) {
              n1 = __shfl_sync(0xffffffffu, __uint_as_float(d[j + 1 < J ? j + 1 : j][1][c]), (lane - 7) & 31);
              n2 = __shfl_sync(0xffffffffu, __uint_as_float(d[j + 1 < J ? j + 1 : j][2][c]), (lane - 6) & 31);
            }
            const float a = __uint_as_float(d[j][0][c]) + (rx < 7 ? s1 : n1) + (rx < 6 ? s2 : n2) + s_bias[c];
            v[c] = fmaxf(a, a * act_slope);
          }
          if (p.act >= TECO_ACT_TANH24) {
#pragma unroll
            for (int c = 0; c < 4; ++c) v[c] = teco_act(v[c], p.act);
          }
          const int tc = 8 * j + rx, ox = x0 + tc;
          // the two warps of a lane quarter take alternate sub-tiles (no early exit: the shuffles above are warp-collective)
          const bool mine = ((warp - 2) >> 2) == (j & 1) && tc < tile_w && ox < p.W && oy < p.H;
          const size_t pix = ((size_t)n * p.H + oy) * p.W + ox;
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (mine && c < C) {
              const float a = v[c] + (p.res_f32 ? p.res_f32[pix * C + c] : 0.f);
              p.out_f32[pix * C + c] = a * p.post_scale + p.post_shift;
            }
        }
        if (threadIdx.x == 64) TSTAMP(it, 3);
      }
    } else if (MODE == 1 && p.tma_out) {
      // ---- staged epilogue of the transposed conv (J == 1, KS == 1, Ncta == 64): the four phase accumulators of the tile
      // one after the other, the next phase's TMEM load in flight while this one is converted and written to its staging tile
      const uint32_t rowoff = (uint32_t)m * 128u, sw = (uint32_t)m & 7u;
      float bias_r[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) bias_r[i] = s_bias[32 * chalf + i];
      for (int it = 0; it < my_tiles; ++it) {
        const int as = (p.AS == 2) ? (it & 1) : 0;
        const uint32_t ause = (uint32_t)((p.AS == 2) ? (it >> 1) : it);
        mbar_wait_warp(smem_u32(&acc_full[as]), ause & 1u);
        tcgen05_fence_after();
        if (threadIdx.x == 64) TSTAMP(it, 2);
        const uint32_t tb = tmem_base + (uint32_t)as * acc_stage_cols + ((uint32_t)(32 * q) << 16) + (uint32_t)(32 * chalf);
        uint32_t r[2][32];
        tmem_ld32(tb, r[0]);
#pragma unroll
        for (int ph = 0; ph < 4; ++ph) {
          tmem_wait_ld();
          if (ph < 3) {
            tmem_ld32(tb + (uint32_t)((ph + 1) * 64), r[(ph + 1) & 1]);
          } else {
            tcgen05_fence_before();
            if (lane == 0) mbar_arrive(smem_u32(&acc_empty[as]));
          }
          mbar_wait_warp(smem_u32(&stage_free[ph]), (uint32_t)((it & 1) ^ 1));
          uint8_t* row = stage_base + (size_t)ph * 16384 + rowoff;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float a0 = __uint_as_float(r[ph & 1][8 * k + 2 * i]) + bias_r[8 * k + 2 * i];
              const float a1 = __uint_as_float(r[ph & 1][8 * k + 2 * i + 1]) + bias_r[8 * k + 2 * i + 1];
              __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(a0, a0 * act_slope), fmaxf(a1, a1 * act_slope));
              o[i] = *reinterpret_cast<uint32_t*>(&h);
            }
            *reinterpret_cast<uint4*>(row + ((((uint32_t)(4 * chalf + k)) ^ sw) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&out_full[ph]));
        }
        if (threadIdx.x == 64) TSTAMP(it, 3);
      }
    } else if (p.Ncta % 32 == 0) run(std::integral_constant<int, 32>{});   // (a single EW = 16 instantiation halves the SASS but
    else run(std::integral_constant<int, 16>{});                           //  measured 7.4 us vs 6.9 us on the 64->64 layer)
  }

  if (threadIdx.x == 64) STAMP(7);
  tcgen05_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) STAMP(8);
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

// ------------------------------------------------------------------ weight packing
// out[blk][tap][cout_pad][64] bf16 in the SWIZZLE_128B image (16-byte chunk j of row r stored at chunk j ^ (r & 7))
//   <- w[3,3,cin,cout] (or [3,3,cout,cin] when transpose_layout); packed input channel k reads cin_perm[k] (-1 = zero).
__global__ void pack_conv3x3_kernel(const float* __restrict__ w, int cin, int cout, int cin_pad, int cout_pad,
                                    int transpose_layout, const int* __restrict__ cin_perm, __nv_bfloat16* __restrict__ out) {
  long long total = 9LL * cin_pad * cout_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int e = (int)(i & 7);
    int jpos = (int)((i >> 3) & 7);
    long long t = i >> 6;
    int co = (int)(t % cout_pad);
    t /= cout_pad;
    int tap = (int)(t % 9);
    int blk = (int)(t / 9);
    int j = jpos ^ (co & 7);
    int ci = blk * 64 + j * 8 + e;
    int src_ci = cin_perm ? cin_perm[ci] : (ci < cin ? ci : -1);
    float v = 0.f;
    const int stap = (transpose_layout & 2) ? 8 - tap : tap;   // bit 1: spatially flipped taps (input-gradient convolution)
    if (src_ci >= 0 && src_ci < cin && co < cout)
      v = (transpose_layout & 1) ? w[((long long)stap * cout + co) * cin + src_ci] : w[((long long)stap * cin + src_ci) * cout + co];
    out[i] = __float2bfloat16_rn(v);
  }
}

}  // namespace

long long* teco_g_dbg_timing = nullptr;   // shared with conv_tc_sw.cu

extern "C" int teco_debug_timing(void* buf) {
  teco_g_dbg_timing = (long long*)buf;
  return TECO_OK;
}

extern "C" int64_t teco_packed_weight_bytes(int32_t cin_pad, int32_t cout_pad) {
  return 9LL * cin_pad * cout_pad * 2;
}

extern "C" int teco_pack_conv3x3_bf16(const float* w, int32_t cin, int32_t cout, int32_t cin_pad, int32_t cout_pad,
                                      int32_t transpose_layout, const int32_t* cin_perm, void* wpk, void* stream) {
  TECO_CHECK_ARG(w && wpk, "teco_pack_conv3x3_bf16: NULL tensor");
  TECO_CHECK_ARG(cin > 0 && cout > 0 && cin_pad >= cin && cout_pad >= cout && (cin_pad % 64) == 0 && (cout_pad % 16) == 0,
                 "teco_pack_conv3x3_bf16: cin_pad must be a multiple of 64 and cout_pad a multiple of 16, both >= the real channels");
  long long total = 9LL * cin_pad * cout_pad;
  int blocks = teco_ceil_div(total, 256);
  if (blocks > 4096) blocks = 4096;
  pack_conv3x3_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(w, cin, cout, cin_pad, cout_pad, transpose_layout, cin_perm,
                                                                (__nv_bfloat16*)wpk);
  TECO_CUDA_LAUNCH_CHECK("teco_pack_conv3x3_bf16");
  return TECO_OK;
}

extern "C" int teco_conv3x3_tc(const teco_tc_desc* d, const void* x, const void* wpk, const float* bias, const void* res,
                               void* y, const float* res_f32, float* out_f32, void* stream) {
  TECO_CHECK_ARG(d && x && wpk, "teco_conv3x3_tc: NULL argument");
  TECO_CHECK_ARG(y || out_f32, "teco_conv3x3_tc: no output buffer");
  TECO_CHECK_ARG(d->N > 0 && d->H > 0 && d->W > 0, "teco_conv3x3_tc: bad shape N=%d H=%d W=%d", d->N, d->H, d->W);
  TECO_CHECK_ARG(d->Cin >= 64 && d->Cin % 64 == 0 && d->Cin <= 512, "teco_conv3x3_tc: Cin must be a multiple of 64 in [64,512] (got %d)", d->Cin);
  TECO_CHECK_ARG(d->Cout >= 16 && d->Cout % 16 == 0 && d->Cout <= 512, "teco_conv3x3_tc: Cout must be a multiple of 16 in [16,512] (got %d)", d->Cout);
  TECO_CHECK_ARG(d->mode == 0 || d->mode == 1, "teco_conv3x3_tc: unknown mode %d", d->mode);
  TECO_CHECK_ARG(d->act >= 0 && d->act <= TECO_ACT_SIGMOID, "teco_conv3x3_tc: unknown activation %d", d->act);
  TECO_CHECK_ARG(!out_f32 || (d->out_f32_c > 0 && d->out_f32_c <= d->Cout), "teco_conv3x3_tc: bad out_f32_c");
  TECO_CHECK_ARG((((uintptr_t)x) & 15) == 0 && (((uintptr_t)wpk) & 15) == 0 && (((uintptr_t)y) & 15) == 0 &&
                     (((uintptr_t)res) & 15) == 0,
                 "teco_conv3x3_tc: tensors must be 16-byte aligned");
  TcPlan pl;
  if (int e = tc_plan(d, y != nullptr, res != nullptr, out_f32 != nullptr, teco_sm_count(), pl)) return e;
  if (pl.onetile) return teco_conv3x3_tc_onetile(pl, d, x, wpk, bias, res, y, res_f32, out_f32, stream);

  TcParams p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
  p.Ncta = pl.Ncta; p.nsplit = pl.nsplit; p.G = pl.G; p.AS = pl.AS;
  p.tiles_x = pl.tiles_x; p.tiles_y = pl.tiles_y; p.J = pl.J;
  p.mode = d->mode; p.act = d->act; p.out_f32_c = d->out_f32_c;
  p.post_scale = d->post_scale; p.post_shift = d->post_shift;
  p.nblk = pl.nblk; p.WST = pl.WST; p.TPS = pl.TPS; p.KS = pl.KS;
  p.HST = pl.HST; p.mcast = pl.mcast; p.num_tiles = pl.num_tiles;
  p.halo_stage_bytes = pl.halo_stage_bytes; p.w_slab_bytes = pl.w_slab_bytes; p.tmem_cols = pl.tmem_cols;
  p.tma_out = pl.tma_out; p.tma_res = pl.tma_res;
  p.wpk = (const uint8_t*)wpk; p.bias = bias; p.res = (const __nv_bfloat16*)res; p.y = (__nv_bfloat16*)y;
  p.res_f32 = res_f32; p.out_f32 = out_f32; p.dbg = teco_g_dbg_timing;
  CUtensorMap maps[3];
  if (int e = tc_encode_maps(pl, d, x, y, res, maps)) return e;
  void (*kern)(CUtensorMap, CUtensorMap, CUtensorMap, TcParams) = nullptr;
#define TECO_PICK(M, T, JJ, K) \
  if (pl.kmode == M && pl.TPS == T && pl.J == JJ && pl.KS == K) kern = conv3x3_tc_kernel<M, T, JJ, K>;
  TECO_PICK(0, 3, 2, 2) TECO_PICK(0, 3, 1, 3) TECO_PICK(0, 3, 1, 1) TECO_PICK(0, 1, 1, 1)
  TECO_PICK(1, 3, 1, 1)
  TECO_PICK(2, 3, 2, 1) TECO_PICK(2, 3, 3, 1) TECO_PICK(2, 3, 4, 1)
#undef TECO_PICK
  if (!kern) {
    teco_set_error("teco_conv3x3_tc: no kernel instantiation for mode=%d TPS=%d J=%d KS=%d", pl.kmode, pl.TPS, pl.J, pl.KS);
    return TECO_E_UNSUPPORTED;
  }
  return tc_launch(kern, (int)TC_SMEM_MAX, NUM_THREADS, pl, maps, p, stream);
}
