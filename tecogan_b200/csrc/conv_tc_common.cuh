// Shared by the two tcgen05 3x3 convolution kernels behind teco_conv3x3_tc: conv3x3_tc_kernel (conv_tc.cu, persistent,
// many tiles per CTA) and conv3x3_tc_onetile_kernel (conv_tc_sw.cu, one tile per CTA).  Holds the tile constants, the
// launch plan (which kernel, its template arguments, staging, grid and shared memory: tc_plan), the tensor maps, the
// launch, and the small device pieces both kernels use.
#pragma once
#include <cuda.h>
#include "teco_common.cuh"
#include "tc_ptx.cuh"

constexpr int TILE_ROWS = 16;
constexpr int HALO_ROWS = TILE_ROWS + 2;
constexpr int CB = 64;                 // channels per K block = one 128-byte swizzled row
constexpr int MAX_WST = 12;
constexpr int MAX_HST = 4;             // persistent halo ring depth: 2 when the input is L2-resident, up to 4 when it streams from HBM

// ------------------------------------------------------------------ device pieces
namespace {

// v[0..7] += the eight bf16 of rr
__device__ __forceinline__ void add_bf16x8(float* v, const uint4 rr) {
  const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rw[i]));
    v[2 * i] += f.x;
    v[2 * i + 1] += f.y;
  }
}

// v[0..7] -> eight bf16 (round to nearest even) in one 16-byte word
__device__ __forceinline__ uint4 pack_bf16x8(const float* v) {
  uint32_t o[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    o[i] = *reinterpret_cast<uint32_t*>(&h);
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// Tap (ky, kx) -> halo row / column offset and accumulator phase.  Transposed conv (stride 2, TF 'SAME',
// y[i] = sum_j x[j] w[i-2j]): the nine taps go to four sub-pixel phases and read only input offsets 0 and 1.
template <int MODE>
__device__ __forceinline__ void tap_route(int ky, int kx, int& ry, int& rx, int& phase) {
  if (MODE == 1) {
    ry = (ky == 2) ? 0 : 1;
    rx = (kx == 2) ? 0 : 1;
    phase = ((ky == 1) ? 2 : 0) + ((kx == 1) ? 1 : 0);
  } else {
    ry = ky; rx = kx; phase = 0;
  }
}

// Resident weights (the whole layer fits): lane s fetches slab s of output channels [n0, n0 + Ncta).  Global layout
// [blk][tap][cout][64]: a slab = TPS consecutive taps of one block.  With a cluster (CS > 1) each CTA fetches 1/CS of
// every slab and multicasts it to all CS CTAs (one L2 read per cluster).
template <int TPS>
__device__ __forceinline__ void fetch_resident_weights(int lane, int nslabs, const uint8_t* wpk, int Cout, int n0,
                                                       uint32_t w_slab_bytes, uint8_t* w_base, uint64_t* w_full, int CS) {
  using namespace tcptx;
  constexpr int slabs_per_blk = 9 / TPS;
  const int sidx = lane;
  if (sidx < nslabs) {
    const uint32_t crank = CS > 1 ? cluster_ctarank() : 0;
    const uint32_t part = w_slab_bytes / (uint32_t)CS;
    const uint16_t mask = (uint16_t)((1u << CS) - 1u);
    const int b = sidx / slabs_per_blk, g = sidx - slabs_per_blk * b;
    mbar_expect_tx(smem_u32(&w_full[sidx]), w_slab_bytes);
    const uint8_t* src = wpk + ((size_t)(b * 9 + g * TPS) * Cout + n0) * 128 + (size_t)crank * part;
    const uint32_t dst = smem_u32(w_base + (size_t)sidx * w_slab_bytes) + crank * part;
    if (CS > 1) bulk_load_1d_mcast(dst, src, part, smem_u32(&w_full[sidx]), mask);
    else bulk_load_1d(dst, src, part, smem_u32(&w_full[sidx]));
  }
  __syncwarp();
}

}  // namespace

// ------------------------------------------------------------------ launch plan (host, no CUDA calls)
struct TcPlan {
  bool onetile;                       // conv3x3_tc_onetile_kernel (else the persistent conv3x3_tc_kernel)
  int kmode, J, TPS, KS;              // template arguments; kmode 2 = kx-fused narrow output stage (persistent only)
  int nsplit, Ncta, nblk;             // Cout splits, output channels per CTA (UMMA N), Cin / 64
  int HST, WST, mcast, CS, AS;        // halo stages, weight stages, resident weights, cluster size, accumulator stages
  int tiles_x, tiles_y, num_tiles, G; // G: CTAs per Cout split
  int box_w;                          // halo box width in pixels
  int tma_out, tma_res, late_trigger;
  uint32_t halo_stage_bytes, w_slab_bytes, stage2_bytes, tmem_cols;
  size_t smem_bytes;
};

constexpr size_t TC_SMEM_BUDGET = 208 * 1024;   // halo stages + weights
constexpr size_t TC_SMEM_MAX = 232448;          // 227 KB: the opt-in maximum of dynamic shared memory per block on sm_100

inline uint32_t tc_halo_stage_bytes(int box_w) { return ((uint32_t)(HALO_ROWS * box_w * 128) + 1023u) & ~1023u; }

// Weight staging next to a_total bytes of halo stages: the whole layer resident (3-tap slabs, fetched once), a 2-deep
// ring of 3-tap slabs when that keeps the CTA within half an SM (two CTAs per SM), a deeper ring of 3-tap slabs, or a
// ring of single taps.
inline int tc_weight_staging(TcPlan& pl, const teco_tc_desc* d, size_t a_total, bool resident, bool half_sm_ring, bool three_tap) {
  const size_t tap_bytes = (size_t)pl.Ncta * 128;
  if (resident && a_total + 9 * tap_bytes * pl.nblk <= TC_SMEM_BUDGET && 3 * pl.nblk <= MAX_WST) {
    pl.mcast = 1; pl.TPS = 3; pl.WST = 3 * pl.nblk;
  } else if (half_sm_ring && 1024 + a_total + 2 * 3 * tap_bytes + 1024 <= 112 * 1024) {
    pl.TPS = 3; pl.WST = 2;
  } else if (three_tap && a_total + 2 * 3 * tap_bytes <= TC_SMEM_BUDGET) {
    pl.TPS = 3; pl.WST = (int)((TC_SMEM_BUDGET - a_total) / (3 * tap_bytes));
    if (pl.WST > 3 * pl.nblk) pl.WST = 3 * pl.nblk;
    if (pl.WST > MAX_WST) pl.WST = MAX_WST;
  } else {
    pl.TPS = 1;
    int wst = (int)((TC_SMEM_BUDGET - a_total) / tap_bytes);
    if (wst > 9 * pl.nblk) wst = 9 * pl.nblk;
    if (wst > MAX_WST) wst = MAX_WST;
    TECO_CHECK_ARG(wst >= 2, "teco_conv3x3_tc: shared memory budget too small (Cin=%d Cout=%d)", d->Cin, d->Cout);
    pl.WST = wst;
  }
  pl.w_slab_bytes = (uint32_t)(pl.TPS * tap_bytes);
  return TECO_OK;
}

inline uint32_t tc_tmem_cols(uint32_t cols) {
  uint32_t tc = 32;
  while (tc < cols) tc <<= 1;
  return tc;
}

// One tile per CTA.  Sub-tiles per CTA: the wider tile when it still yields >= 2 waves of CTAs and fits TMEM / smem.
inline int tc_plan_onetile(TcPlan& pl, const teco_tc_desc* d, bool y, bool res, bool out_f32, int sms) {
  const int nacc = d->mode == 1 ? 4 : 1;
  const size_t tap_bytes = (size_t)pl.Ncta * 128;
  pl.kmode = d->mode;
  pl.HST = pl.nblk > 1 ? 2 : 1;
  pl.J = (2 * nacc * pl.Ncta <= 512 && pl.HST * (size_t)tc_halo_stage_bytes(18) + 2 * tap_bytes <= TC_SMEM_BUDGET &&
          (long long)d->N * teco_ceil_div(d->H, TILE_ROWS) * teco_ceil_div(d->W, 16) >= 2LL * sms) ? 2 : 1;
  pl.box_w = 8 * pl.J + 2;
  pl.tiles_x = teco_ceil_div(d->W, 8 * pl.J);
  pl.tiles_y = teco_ceil_div(d->H, TILE_ROWS);
  pl.num_tiles = (int)((long long)d->N * pl.tiles_x * pl.tiles_y);
  pl.halo_stage_bytes = tc_halo_stage_bytes(pl.box_w);
  const size_t a_total = (size_t)pl.HST * pl.halo_stage_bytes;
  // Weight staging.  Preferred: a 2-deep ring of 3-tap slabs -- with the halo copies that is ~105 KB, so TWO CTAs fit per
  // SM and programmatic dependent launch really overlaps the next layer's prologue + weight prefetch with this layer's
  // MMA/epilogue (256x256: 14.7 us vs 24.0 us).  When there is one CTA per SM anyway (e.g. the 128x128 trunk: 128
  // tiles): the whole layer resident, fetched before the dependency wait and multicast over a 4-CTA cluster -- measured
  // 6.2 us vs 6.9 us for the ring on the 64->64 layer.  3-tap slabs only without a Cout split.
  const bool single_wave = (long long)pl.num_tiles * pl.nsplit <= (long long)sms;
  if (int e = tc_weight_staging(pl, d, a_total, single_wave && pl.nsplit == 1, pl.nsplit == 1, pl.nsplit == 1)) return e;
  pl.KS = (pl.TPS == 3 && d->mode == 0 && pl.J * 3 * pl.Ncta <= 512) ? 3 : 1;
  pl.CS = (pl.mcast && pl.num_tiles >= 8) ? 4 : 1;
  pl.AS = 1;
  pl.tmem_cols = tc_tmem_cols((uint32_t)(pl.J * nacc * pl.KS * pl.Ncta));
  // staged epilogue; tconv: rows of (n, y) are one map dimension
  pl.tma_out = (y && !out_f32 && pl.Ncta == 64 && (d->mode == 0 || (!res && pl.nsplit == 1 && d->H % TILE_ROWS == 0))) ? 1 : 0;
  pl.tma_res = (pl.tma_out && res) ? 1 : 0;
  pl.stage2_bytes = pl.tma_res ? (uint32_t)(pl.J * 16384) : ((pl.tma_out && d->mode == 1) ? 16384u : 0u);
  TECO_CHECK_ARG(!pl.tma_out || (size_t)pl.J * 16384 <= a_total, "teco_conv3x3_tc: output staging does not fit the halo stages");
  pl.smem_bytes = a_total + (size_t)pl.WST * pl.w_slab_bytes + pl.stage2_bytes + (4 + 2 * MAX_WST + 2) * 8 + 256 * sizeof(float) + 16;
  pl.late_trigger = (2 * (pl.smem_bytes + 1024) <= 228 * 1024) ? 1 : 0;   // only useful when two CTAs fit an SM
  pl.G = (pl.num_tiles + pl.CS - 1) / pl.CS * pl.CS;                         // padded to the cluster size
  return TECO_OK;
}

// Persistent CTAs (one per SM) walking tiles: double-buffered halo stages and -- when TMEM allows -- two accumulator
// stages, so TMA, MMA and epilogue overlap across tiles; the layer's weights stay resident in shared memory for the whole
// launch when they fit next to two halo stages.
inline int tc_plan_persistent(TcPlan& pl, const teco_tc_desc* d, bool y, bool res, bool out_f32, int sms, long long tiles1,
                              bool tconv) {
  const size_t tap_bytes = (size_t)pl.Ncta * 128;
  pl.HST = 2;
  if (int e = tc_weight_staging(pl, d, 2 * (size_t)tc_halo_stage_bytes(10), true, false, true)) return e;
  pl.J = 1;
  pl.KS = (pl.TPS == 3 && d->mode == 0 && 3 * pl.Ncta <= 512) ? 3 : 1;
  // Many tiles with <= 64 output channels per CTA: two 16x8 sub-tiles per tile and two K-split chains each (4 independent
  // accumulators) instead of one sub-tile with three -- a third less TMEM read traffic in the epilogue (the 64 B/clk
  // tcgen05.ld path bounds it) and a 16+2 pixel wide halo row instead of two 8+2 ones.
  if (d->mode == 0 && pl.TPS == 3 && pl.mcast && pl.Ncta <= 64 && tiles1 >= 4LL * sms &&
      2 * (size_t)tc_halo_stage_bytes(18) + 9 * tap_bytes * pl.nblk <= TC_SMEM_BUDGET) {
    pl.J = 2; pl.KS = 2;
  }
  // Narrow fp32 output stage (generator 64->3, fnet 32->2) on many tiles: the kx-fused kernel (MODE 2)
  const bool kx = d->mode == 0 && out_f32 && !y && !res && d->Cout == 16 && pl.nsplit == 1 && pl.nblk == 1 && d->out_f32_c <= 4 &&
                  pl.mcast && pl.TPS == 3;
  if (kx) {
    double best = 0.0;
    for (int jj = 2; jj <= 4; ++jj) {   // widest use of the 8*jj halo columns: W / (tiles * 8 jj)
      const double eff = (double)d->W / ((double)teco_ceil_div(d->W, 8 * jj - 2) * 8 * jj);
      if (eff > best + 1e-9) { best = eff; pl.J = jj; }
    }
    pl.KS = 1;
  }
  pl.kmode = kx ? 2 : d->mode;
  const int nacc = pl.kmode == 1 ? 4 : (pl.kmode == 2 ? 3 : 1);
  pl.box_w = kx ? 8 * pl.J : 8 * pl.J + 2;
  pl.tiles_x = kx ? teco_ceil_div(d->W, 8 * pl.J - 2) : teco_ceil_div(d->W, 8 * pl.J);
  pl.tiles_y = teco_ceil_div(d->H, TILE_ROWS);
  pl.num_tiles = (int)((long long)d->N * pl.tiles_x * pl.tiles_y);
  pl.halo_stage_bytes = tc_halo_stage_bytes(pl.box_w);
  // Input larger than ~half of L2 streams from HBM: one tile of look-ahead (HST = 2) leaves the CTA waiting on DRAM
  // latency (the 64->16 output stage at 296 x 128x128 ran 6300 clk per tile against ~2900 of work); use the shared memory
  // the configuration leaves free for a deeper ring.
  const bool tma_possible = tconv || (d->mode == 0 && y && !out_f32 && pl.Ncta == 64 && d->act < TECO_ACT_TANH24);
  const size_t staging_bytes = tconv ? 1024 + (size_t)4 * 16384 : 1024 + (size_t)2 * pl.J * 16384;
  if (pl.nblk == 1 && (double)d->N * d->H * d->W * d->Cin * 2.0 > 48e6) {
    const size_t fixed = (size_t)pl.WST * pl.w_slab_bytes + (tma_possible ? staging_bytes : 0) + 8192;
    while (pl.HST < MAX_HST && fixed + (size_t)(pl.HST + 1) * pl.halo_stage_bytes <= TC_SMEM_MAX - 2048) ++pl.HST;
  }
  const uint32_t stage_cols = (uint32_t)(pl.J * nacc * pl.KS * pl.Ncta);
  pl.CS = 1;
  pl.AS = 2 * stage_cols <= 512 ? 2 : 1;
  pl.tmem_cols = tc_tmem_cols(stage_cols * (uint32_t)pl.AS);
  pl.G = pl.num_tiles < sms ? pl.num_tiles : sms;
  pl.tma_out = tma_possible ? 1 : 0;
  pl.tma_res = (pl.tma_out && res) ? 1 : 0;
  pl.smem_bytes = 1024 + (size_t)pl.HST * pl.halo_stage_bytes + (size_t)pl.WST * pl.w_slab_bytes + (2 * MAX_HST + 2 * MAX_WST + 4 + 1) * 8 +
                  256 * sizeof(float) + 128 + (pl.tma_out ? staging_bytes : 0);
  if (pl.smem_bytes > TC_SMEM_MAX && pl.tma_out) {
    TECO_CHECK_ARG(!tconv, "teco_conv3x3_tc: persistent transposed conv does not fit in shared memory");
    pl.smem_bytes -= staging_bytes;
    pl.tma_out = pl.tma_res = 0;
  }
  return TECO_OK;
}

// The whole decision for one teco_conv3x3_tc call.  y / res / out_f32: whether the call passes those buffers.
inline int tc_plan(const teco_tc_desc* d, bool y, bool res, bool out_f32, int sms, TcPlan& pl) {
  pl = TcPlan{};
  pl.nblk = d->Cin / CB;
  // few spatial tiles but many output channels (FNet's 16x16 / 32x32 layers): split Cout over CTAs, 64 channels each
  const long long tiles1 = (long long)d->N * teco_ceil_div(d->H, TILE_ROWS) * teco_ceil_div(d->W, 8);
  pl.nsplit = (d->Cout >= 128 && d->Cout % 64 == 0 && tiles1 * (d->Cout / 64) <= 2LL * sms) ? d->Cout / 64 : 1;
  if (d->Cout / pl.nsplit > 256) pl.nsplit = d->Cout / 256;   // VGG's 512-channel layers: N <= 256 per UMMA / TMEM stage
  pl.Ncta = d->Cout / pl.nsplit;
  TECO_CHECK_ARG((d->mode == 1 ? 4 : 1) * pl.Ncta <= 512, "teco_conv3x3_tc: Cout=%d too large for mode %d (TMEM has 512 columns)",
                 d->Cout, d->mode);
  // Dispatch (same-box A/B, profiles/conv_tc_r01_notes.md): the one-tile-per-CTA kernel is faster for single-wave
  // launches and for the epilogue-heavy transposed conv (two CTAs per SM); the persistent kernel wins multi-wave convs
  // ... and large transposed convs (many waves), with one staging tile per output phase.
  const bool tconv_persist = d->mode == 1 && tiles1 >= 4LL * sms && pl.nsplit == 1 && pl.Ncta == 64 && y && !out_f32 && !res &&
                             d->H % TILE_ROWS == 0 && d->W % 8 == 0 && d->act < TECO_ACT_TANH24 && pl.nblk == 1;
  pl.onetile = tiles1 * pl.nsplit <= (long long)sms || (d->mode == 1 && !tconv_persist);
  return pl.onetile ? tc_plan_onetile(pl, d, y, res, out_f32, sms)
                    : tc_plan_persistent(pl, d, y, res, out_f32, sms, tiles1, tconv_persist);
}

// ------------------------------------------------------------------ tensor maps and launch
// m[0]: the input halo box; with the staged epilogue m[1] / m[2]: the output / residual tiles (16 rows x 8 pixels x 64
// channels; transposed conv: one sub-pixel phase of them through the 5-D map {C, px, x, py, n*H + y} of the 2x interleaved
// output -- H % 16 == 0, so a box never runs from one image into the next).  Unused maps are copies of m[0].
inline int tc_encode_maps(const TcPlan& pl, const teco_tc_desc* d, const void* x, void* y, const void* res, CUtensorMap (&m)[3]) {
  if (int e = teco_tmap_nhwc(&m[0], "teco_conv3x3_tc", x, d->N, d->H, d->W, d->Cin, CB, pl.box_w, HALO_ROWS)) return e;
  m[1] = m[2] = m[0];
  if (pl.tma_out && d->mode == 1) {
    const cuuint64_t odim[5] = {(cuuint64_t)d->Cout, 2, (cuuint64_t)d->W, 2, (cuuint64_t)d->N * d->H};
    const cuuint64_t ostr[4] = {(cuuint64_t)d->Cout * 2, (cuuint64_t)d->Cout * 4, (cuuint64_t)d->W * d->Cout * 4,
                                (cuuint64_t)d->W * d->Cout * 8};
    const cuuint32_t obox[5] = {64, 1, 8, 1, (cuuint32_t)TILE_ROWS};
    return teco_tmap_bf16(&m[1], "teco_conv3x3_tc (transposed-conv output)", y, 5, odim, ostr, obox);
  }
  if (pl.tma_out) {
    if (int e = teco_tmap_nhwc(&m[1], "teco_conv3x3_tc (output tile)", y, d->N, d->H, d->W, d->Cout, 64, 8, TILE_ROWS)) return e;
    if (pl.tma_res)
      return teco_tmap_nhwc(&m[2], "teco_conv3x3_tc (residual tile)", res, d->N, d->H, d->W, d->Cout, 64, 8, TILE_ROWS);
  }
  return TECO_OK;
}

// Programmatic dependent launch (the prologue overlaps the previous kernel's tail), in clusters of pl.CS CTAs.
template <typename Params>
inline int tc_launch(void (*kern)(CUtensorMap, CUtensorMap, CUtensorMap, Params), int smem_limit, int threads, const TcPlan& pl,
                     const CUtensorMap (&m)[3], const Params& p, void* stream) {
  TECO_CUDA_CALL(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_limit));
  const unsigned ctas = (unsigned)(pl.G * pl.nsplit);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ctas);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = pl.smem_bytes;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attrs[0].val.programmaticStreamSerializationAllowed = 1;
  attrs[1].id = cudaLaunchAttributeClusterDimension;
  attrs[1].val.clusterDim.x = (unsigned)pl.CS;
  attrs[1].val.clusterDim.y = 1;
  attrs[1].val.clusterDim.z = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = pl.CS > 1 ? 2 : 1;
  cudaError_t le = cudaLaunchKernelEx(&cfg, kern, m[0], m[1], m[2], p);
  if (le != cudaSuccess) {
    teco_set_error("teco_conv3x3_tc: launch failed: %s (grid %u, cluster %d, smem %zu)", cudaGetErrorString(le), ctas, pl.CS,
                   pl.smem_bytes);
    return TECO_E_CUDA;
  }
  return TECO_OK;
}

extern long long* teco_g_dbg_timing;   // set by teco_debug_timing (conv_tc.cu)
int teco_conv3x3_tc_onetile(const TcPlan& pl, const teco_tc_desc* d, const void* x, const void* wpk, const float* bias, const void* res,
                            void* y, const float* res_f32, float* out_f32, void* stream);   // conv_tc_sw.cu
