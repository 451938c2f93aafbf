// ONE-TILE-PER-CTA variant of the tcgen05 convolution (see conv_tc.cu for the design notes and the persistent variant;
// tc_plan in conv_tc_common.cuh picks between them).
// Used for single-wave launches (tiles <= SMs, e.g. the 128x128 generator trunk) and for most transposed convolutions:
// same-box A/B (profiles/conv_tc_r01_notes.md) showed this variant 1.3 us faster per single-wave layer and its
// two-CTAs-per-SM ring faster on the epilogue-heavy transposed conv, while the persistent kernel wins every multi-wave conv.
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..9 = epilogue
// (one epilogue warp per scheduler is latency-bound: ~1000 clk per 32 channels; two per scheduler halve it).
#include <type_traits>
#include "conv_tc_common.cuh"

namespace {

constexpr int NUM_EPI_WARPS = 8;       // two warps per TMEM lane quarter, each taking half of the output channels
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;

struct TcParams {
  int N, H, W, Cin, Cout;             // Cout = channel pitch of y / res / bias (all output channels)
  int Ncta, nsplit, tiles_pad;        // output channels per CTA (UMMA N), Cout splits, tile count padded to the cluster size
  int tiles_x, tiles_y, J;
  int mode, act, out_f32_c;
  float post_scale, post_shift;
  int nblk, WST, TPS, KS;              // Cin/64, weight ring stages, taps per weight slab (1 or 3), K-split chains
  int HST, CS, mcast, num_tiles;       // halo stages, cluster size, resident+multicast weights, real tile count
  int late_trigger;                    // trigger the dependent launch after the MMAs instead of after the prologue
  uint32_t stage2_bytes;               // second staging region after the weights: residual tiles (conv) / ping-pong tile (tconv)
  int tma_out, tma_res;                // bf16 output / residual tiles travel through swizzled smem staging + TMA (Ncta == 64, conv)
  uint32_t halo_stage_bytes, w_slab_bytes, tmem_cols;
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
// One halo box (8J+2 pixels wide) per block: 2.4x less L2->smem traffic than one box per horizontal tap, 23 KB per stage.
template <int MODE, int TPS, int J, int KS>
__global__ void __launch_bounds__(NUM_THREADS, 2)
conv3x3_tc_onetile_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_y,
                  const __grid_constant__ CUtensorMap tmap_r, const TcParams p) {
  // SWIZZLE_128B needs 1024-byte aligned tiles; the dynamic window starts on such a boundary (no static shared memory in
  // this kernel) -- relied upon instead of a 1 KB slack so that two trunk-layer CTAs (112.3 KB each) share an SM.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw;
  if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  uint8_t* halo_base = smem;                                             // HST halo stages
  uint8_t* w_base = smem + (size_t)p.HST * p.halo_stage_bytes;           // WST weight slabs
  // residual staging tiles (J x 16 KB, TMA box image) follow the weights; the OUTPUT staging tiles reuse the halo
  // stages, which are dead once the accumulators are complete
  uint8_t* stage_res = w_base + (size_t)p.WST * p.w_slab_bytes;
  uint8_t* stage_out = halo_base;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_res + p.stage2_bytes);
  uint64_t* halo_full = bars;
  uint64_t* halo_empty = bars + 2;
  uint64_t* w_full = bars + 4;
  uint64_t* w_empty = bars + 4 + MAX_WST;
  uint64_t* acc_full = bars + 4 + 2 * MAX_WST;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 + 2 * MAX_WST + 1);
  float* s_bias = reinterpret_cast<float*>(bars + 4 + 2 * MAX_WST + 2);   // [Cout]
  uint64_t* res_full = bars + 4 + 2 * MAX_WST + 2 + 128;                  // after 256 floats of bias

  // tile coordinates
  int tile = blockIdx.x % p.tiles_pad;      // grid = nsplit x (tiles padded to a multiple of the cluster size)
  const int n0 = (blockIdx.x / p.tiles_pad) * p.Ncta;   // first output channel of this CTA (all CTAs of a cluster share it)
  const bool active = tile < p.num_tiles;
  if (!active) tile = 0;
  const int tx = tile % p.tiles_x;
  tile /= p.tiles_x;
  const int ty = tile % p.tiles_y;
  const int n = tile / p.tiles_y;
  const int x0 = tx * 8 * J, y0 = ty * TILE_ROWS;
  long long* dbg = p.dbg ? p.dbg + (size_t)blockIdx.x * 32 : nullptr;
#define STAMP(i) do { if (dbg) dbg[i] = clock64(); } while (0)
#define GSTAMP(i) do { if (dbg) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); dbg[i] = (long long)t_; } } while (0)
  if (threadIdx.x == 0) { STAMP(0); GSTAMP(26); }

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.HST; ++i) {
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_empty[i]), 1);
    }
    for (int i = 0; i < p.WST; ++i) {
      mbar_init(smem_u32(&w_full[i]), 1);
      mbar_init(smem_u32(&w_empty[i]), 1);
    }
    mbar_init(smem_u32(acc_full), 1);
    mbar_init(smem_u32(res_full), 1);
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
  if (p.CS > 1) cluster_sync_all();   // every CTA's mbarriers are initialised before any multicast may signal them
  else __syncthreads();
  tcgen05_fence_after();
  // Programmatic dependent launch is triggered only once this CTA's own dependency wait has returned (producer warp):
  // the previous layer has retired by then, so the next layer's CTAs share an SM with exactly one CTA of this layer, run
  // their prologue + weight fetch under our halo load / MMAs / epilogue, and never pile up three layers deep (triggering
  // in the prologue let 2 CTAs of later layers land on the 20 idle SMs: 7.45 vs 6.5 us/layer).
  if (!active || !p.late_trigger) pdl_launch_dependents();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) STAMP(1);

  constexpr int nacc = MODE == 1 ? 4 : 1;
  constexpr int slabs_per_blk = 9 / TPS;
  constexpr int row_bytes = (8 * J + 2) * 128;   // one box row (pixels x 128 B)
  constexpr uint32_t copy_bytes = (uint32_t)(HALO_ROWS * row_bytes);

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Issue cost of one bulk/tensor copy is a few hundred cycles, so independent copies are issued by different lanes.
    // Weights do not depend on the previous layer: fetch them before the dependency wait.
    if (p.mcast) fetch_resident_weights<TPS>(lane, slabs_per_blk * p.nblk, p.wpk, p.Cout, n0, p.w_slab_bytes, w_base, w_full, p.CS);
    // Ring mode: the first WST weight slabs do not depend on the previous layer either -> issue them before the wait.
    const int total_slabs = slabs_per_blk * p.nblk;
    int next_slab = 0;
    if (!p.mcast && lane == 0) {
      for (; next_slab < total_slabs && next_slab < p.WST; ++next_slab) {
        const int b = next_slab / slabs_per_blk, g = next_slab - slabs_per_blk * b;
        mbar_expect_tx(smem_u32(&w_full[next_slab]), p.w_slab_bytes);
        const uint8_t* src = p.wpk + ((size_t)(b * 9 + g * TPS) * p.Cout + n0) * 128;
        bulk_load_1d(smem_u32(w_base + (size_t)next_slab * p.w_slab_bytes), src, p.w_slab_bytes, smem_u32(&w_full[next_slab]));
      }
    }
    if (lane == 0) STAMP(9);
    pdl_wait();   // the previous kernel's output (our input x) is complete and visible from here on
    if (p.late_trigger) pdl_launch_dependents();   // the layer before us has retired: at most two layers share an SM
    if (lane == 0) { STAMP(10); GSTAMP(27); }
    if (active) {
      int hs = 0;
      uint32_t hph = 0;
      for (int b = 0; b < p.nblk; ++b) {
        if (lane == 0) {
          mbar_wait(smem_u32(&halo_empty[hs]), hph ^ 1);
          mbar_expect_tx(smem_u32(&halo_full[hs]), copy_bytes);
        }
        __syncwarp();
        if (lane == 0)
          tma_load_4d(smem_u32(halo_base + (size_t)hs * p.halo_stage_bytes), &tmap, smem_u32(&halo_full[hs]), b * CB, x0 - 1, y0 - 1, n);
        if (!p.mcast && lane == 0) {
          for (; next_slab < (b + 1) * slabs_per_blk; ++next_slab) {   // slabs of this block not yet in flight
            const int st = next_slab % p.WST, use = next_slab / p.WST;
            const int g = next_slab - slabs_per_blk * b;
            mbar_wait(smem_u32(&w_empty[st]), (uint32_t)((use - 1) & 1));   // the MMAs of the previous use have retired
            mbar_expect_tx(smem_u32(&w_full[st]), p.w_slab_bytes);
            const uint8_t* src = p.wpk + ((size_t)(b * 9 + g * TPS) * p.Cout + n0) * 128;
            bulk_load_1d(smem_u32(w_base + (size_t)st * p.w_slab_bytes), src, p.w_slab_bytes, smem_u32(&w_full[st]));
          }
        }
        __syncwarp();
        if (++hs == p.HST) { hs = 0; hph ^= 1; }
      }
      if (p.tma_res) {   // the residual tile (same box as the output tile), after the halo: the MMAs are waiting for that one
        if (lane == 0) mbar_expect_tx(smem_u32(res_full), (uint32_t)(J * 16384));
        __syncwarp();
        if (lane < J) tma_load_4d(smem_u32(stage_res + (size_t)lane * 16384), &tmap_r, smem_u32(res_full), n0, x0 + 8 * lane, y0, n);
      }
    } else if (p.mcast && lane == 0) {
      // padding CTA of a cluster: it only relays its share of the weights; stay until they have landed here too
      for (int sidx = 0; sidx < slabs_per_blk * p.nblk; ++sidx) mbar_wait(smem_u32(&w_full[sidx]), 0);
    }
    __syncwarp();
  } else if (warp == 1 && active) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = umma_idesc(p.Ncta);
    constexpr uint32_t a_sbo = (uint32_t)row_bytes;   // next 8-pixel group of the M=128 sub-tile = next image row
    constexpr uint32_t b_sbo = 1024u;                 // next 8 output channels
    int hs = 0, ws = 0;
    uint32_t hph = 0, wph = 0;
    uint32_t started = 0;  // bit (j*nacc+phase): accumulator already written once
    for (int b = 0; b < p.nblk; ++b) {
      mbar_wait_warp(smem_u32(&halo_full[hs]), hph);
      tcgen05_fence_after();
      if (lane == 0 && b == 0) { STAMP(2); GSTAMP(28); }
      const uint32_t halo_addr = smem_u32(halo_base + (size_t)hs * p.halo_stage_bytes);
      for (int g = 0; g < slabs_per_blk; ++g) {
        mbar_wait_warp(smem_u32(&w_full[ws]), wph);
        tcgen05_fence_after();
        if (lane == 0 && b == 0) STAMP(16 + g);
        {
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
            acc_idx[tt] = (uint32_t)(phase * KS + (KS > 1 ? tt : 0));
          }
          const uint32_t started_now = started;
          if (elect_one()) {
            // order: k-step, tap, sub-tile -> consecutive MMAs hit different accumulators (J sub-tiles x KS chains)
#pragma unroll
            for (int s = 0; s < CB / 16; ++s) {
#pragma unroll
              for (int tt = 0; tt < TPS; ++tt) {
#pragma unroll
                for (int j = 0; j < J; ++j) {
                  const uint32_t acc = (uint32_t)(j * nacc * KS) + acc_idx[tt];
                  uint32_t accum = 1u;
                  if (s == 0) {   // first k-step of this slab: overwrite only if nobody has written this accumulator yet
                    accum = (started_now >> acc) & 1u;
#pragma unroll
                    for (int t2 = 0; t2 < tt; ++t2) accum |= (acc_idx[t2] == acc_idx[tt]) ? 1u : 0u;
                  }
                  umma_bf16(tmem_base + acc * (uint32_t)p.Ncta,
                            a_base + a_off16[tt] + (uint32_t)((j * 1024 + s * 32) >> 4),
                            b_base + tt * tap_stride16 + (uint32_t)((s * 32) >> 4), idesc, accum);
                }
              }
            }
          }
          __syncwarp();
#pragma unroll
          for (int j = 0; j < J; ++j)
#pragma unroll
            for (int tt = 0; tt < TPS; ++tt) started |= 1u << ((uint32_t)(j * nacc * KS) + acc_idx[tt]);
          if (elect_one()) tcgen05_commit(smem_u32(&w_empty[ws]));  // frees the weight slab when these MMAs retire
        }
        __syncwarp();
        if (++ws == p.WST) { ws = 0; wph ^= 1; }
      }
      if (elect_one()) tcgen05_commit(smem_u32(&halo_empty[hs]));
      __syncwarp();
      if (++hs == p.HST) { hs = 0; hph ^= 1; }
    }
    if (elect_one()) tcgen05_commit(smem_u32(acc_full));
    if (lane == 0) { STAMP(5); GSTAMP(29); }
    __syncwarp();
  } else if (warp >= 2 && active) {
    // ===================== epilogue (warps 2..5) =====================
    for (int c = (int)threadIdx.x - 64; c < p.Ncta; c += 32 * NUM_EPI_WARPS) s_bias[c] = p.bias ? p.bias[n0 + c] : 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(32 * NUM_EPI_WARPS) : "memory");   // the epilogue warps only
    pdl_wait();                                        // res / y belong to the dependency chain
    if (threadIdx.x == 64) STAMP(25);
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int chalf = (warp - 2) >> 2; // which half of the channel steps this warp takes (0 or 1)
    const int m = 32 * q + lane;       // accumulator row = pixel within the 16x8 sub-tile
    const int ry = m >> 3, rx = m & 7;
    const float act_slope = p.act == TECO_ACT_RELU ? 0.f : (p.act == TECO_ACT_LRELU02 ? 0.2f : 1.f);
    mbar_wait_warp(smem_u32(acc_full), 0);
    tcgen05_fence_after();
    if (threadIdx.x == 64) STAMP(6);
    const int oy_in = y0 + ry;
    // EW output channels per step: 32 (two steps for 64 channels) or 16 (the 16-channel fp32 output stage)
    auto run = [&](auto ew_tag) {
      constexpr int EW = decltype(ew_tag)::value;
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
          const uint32_t tcol = tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)((j * nacc + ph) * KS * p.Ncta);
          for (int c0 = chalf * EW; c0 < p.Ncta; c0 += 2 * EW) {
            uint32_t r[EW];
            __syncwarp();
            if (EW == 32) tmem_ld32(tcol + (uint32_t)c0, r); else tmem_ld16(tcol + (uint32_t)c0, r);
            if (KS == 3) {   // K-split chains: issue all three TMEM loads, wait once, add
              uint32_t r2[EW], r3[EW];
              if (EW == 32) { tmem_ld32(tcol + (uint32_t)(p.Ncta + c0), r2); tmem_ld32(tcol + (uint32_t)(2 * p.Ncta + c0), r3); }
              else { tmem_ld16(tcol + (uint32_t)(p.Ncta + c0), r2); tmem_ld16(tcol + (uint32_t)(2 * p.Ncta + c0), r3); }
              tmem_wait_ld();
#pragma unroll
              for (int i = 0; i < EW; ++i)
                r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r2[i]) + __uint_as_float(r3[i]));
            } else {
              tmem_wait_ld();
            }
            if (threadIdx.x == 64 && j == 0 && ph == 0 && c0 == 0) STAMP(11);
            float v[EW];
#pragma unroll
            for (int i = 0; i < EW; ++i) {
              const float a = __uint_as_float(r[i]) + s_bias[c0 + i];
              v[i] = fmaxf(a, a * act_slope);      // none: slope 1, relu: 0, lrelu: 0.2 -- no per-element branch
            }
            if (p.act >= TECO_ACT_TANH24) {        // uniform, outside the element loop
#pragma unroll
              for (int i = 0; i < EW; ++i) v[i] = teco_act(v[i], p.act);
            }
            if (MODE == 0 && EW == 32 && p.tma_out) {
              // c0 == 32 * chalf here (Ncta == 64).  Pixel m owns row m of the staging tile; its 64 B are chunks 4*chalf..+3,
              // XOR-swizzled with (m & 7) exactly like the TMA box -> conflict-free 16-byte accesses.
              const uint32_t rowoff = (uint32_t)m * 128u;
              if (p.tma_res) {
                mbar_wait_warp(smem_u32(res_full), 0);
                const uint8_t* rs = stage_res + (size_t)j * 16384 + rowoff;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  add_bf16x8(v + 8 * k, *reinterpret_cast<const uint4*>(rs + ((((uint32_t)(4 * chalf + k)) ^ ((uint32_t)m & 7u)) << 4)));
              }
              uint8_t* os = stage_out + (size_t)j * 16384 + rowoff;
#pragma unroll
              for (int k = 0; k < 4; ++k)
                *reinterpret_cast<uint4*>(os + ((((uint32_t)(4 * chalf + k)) ^ ((uint32_t)m & 7u)) << 4)) = pack_bf16x8(v + 8 * k);
              continue;
            }
            if (MODE == 1 && EW == 32 && p.tma_out) {
              // transposed conv: one staging tile per (sub-tile, output phase), two tiles in ping-pong (the dead halo stage and
              // the region after the weights); the phase's 16x8 pixels go out through a 5-D map over the 2x interleaved output
              const int t = j * 4 + ph;
              uint8_t* stg = (t & 1) ? stage_res : stage_out;
              if (t >= 2) {   // the store issued two steps ago has finished reading this tile
                if (threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                asm volatile("bar.sync 1, %0;" ::"n"(32 * NUM_EPI_WARPS) : "memory");
              }
              uint8_t* os = stg + (uint32_t)m * 128u;
#pragma unroll
              for (int k = 0; k < 4; ++k)
                *reinterpret_cast<uint4*>(os + ((((uint32_t)(4 * chalf + k)) ^ ((uint32_t)m & 7u)) << 4)) = pack_bf16x8(v + 8 * k);
              fence_async_smem();
              asm volatile("bar.sync 1, %0;" ::"n"(32 * NUM_EPI_WARPS) : "memory");
              if (threadIdx.x == 64) {
                tma_store_5d(&tmap_y, smem_u32(stg), n0, ph & 1, x0 + 8 * j, ph >> 1, n * p.H + y0);
                bulk_commit();
              }
              continue;
            }
            if (!in_img) continue;
            if (p.out_f32) {
              for (int i = 0; i < EW; ++i) {
                int c = n0 + c0 + i;
                if (c < p.out_f32_c) {
                  float a = v[i] + (p.res_f32 ? p.res_f32[pix * p.out_f32_c + c] : 0.f);
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
            if (threadIdx.x == 64 && j == 0 && ph == 0) STAMP(12 + ((c0 / EW) & 3));
          }
        }
      }
    };
    if (p.Ncta % 32 == 0) run(std::integral_constant<int, 32>{});
    else run(std::integral_constant<int, 16>{});
    if (MODE == 1 && p.tma_out && threadIdx.x == 64) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    if (MODE == 0 && p.tma_out) {
      // generic-proxy smem writes -> visible to the async proxy, all epilogue warps done, then one thread stores the tiles
      fence_async_smem();
      asm volatile("bar.sync 1, %0;" ::"n"(32 * NUM_EPI_WARPS) : "memory");
      if (threadIdx.x == 64) {
        for (int j = 0; j < J; ++j) tma_store_4d(&tmap_y, smem_u32(stage_out + (size_t)j * 16384), n0, x0 + 8 * j, y0, n);
        bulk_commit();
        // shared memory must outlive the store's reads; global visibility to the next layer comes with grid completion
        // (griddepcontrol.wait / stream order), as in any epilogue that ends with a TMA store
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      }
    }
  }

  if (threadIdx.x == 64) { STAMP(7); GSTAMP(30); }
  tcgen05_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) STAMP(8);
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
}

}  // namespace

// Launches conv3x3_tc_onetile_kernel as planned by tc_plan; teco_conv3x3_tc (conv_tc.cu) has validated the arguments.
int teco_conv3x3_tc_onetile(const TcPlan& pl, const teco_tc_desc* d, const void* x, const void* wpk, const float* bias, const void* res,
                            void* y, const float* res_f32, float* out_f32, void* stream) {
  TcParams p;
  p.N = d->N; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
  p.Ncta = pl.Ncta; p.nsplit = pl.nsplit; p.tiles_pad = pl.G;
  p.tiles_x = pl.tiles_x; p.tiles_y = pl.tiles_y; p.J = pl.J;
  p.mode = d->mode; p.act = d->act; p.out_f32_c = d->out_f32_c;
  p.post_scale = d->post_scale; p.post_shift = d->post_shift;
  p.nblk = pl.nblk; p.WST = pl.WST; p.TPS = pl.TPS; p.KS = pl.KS;
  p.HST = pl.HST; p.CS = pl.CS; p.mcast = pl.mcast; p.num_tiles = pl.num_tiles;
  p.late_trigger = pl.late_trigger; p.stage2_bytes = pl.stage2_bytes;
  p.tma_out = pl.tma_out; p.tma_res = pl.tma_res;
  p.halo_stage_bytes = pl.halo_stage_bytes; p.w_slab_bytes = pl.w_slab_bytes; p.tmem_cols = pl.tmem_cols;
  p.wpk = (const uint8_t*)wpk; p.bias = bias; p.res = (const __nv_bfloat16*)res; p.y = (__nv_bfloat16*)y;
  p.res_f32 = res_f32; p.out_f32 = out_f32; p.dbg = teco_g_dbg_timing;
  if (p.dbg) {   // consecutive launches stamp consecutive [256][32] slices (tools/bench_conv.py chain)
    static long long* last_base = nullptr;
    static int launch_idx = 0;
    if (last_base != teco_g_dbg_timing) { last_base = teco_g_dbg_timing; launch_idx = 0; }
    p.dbg = teco_g_dbg_timing + (size_t)(launch_idx % 8) * 256 * 32;
    ++launch_idx;
  }
  CUtensorMap maps[3];
  if (int e = tc_encode_maps(pl, d, x, y, res, maps)) return e;
  void (*kern)(CUtensorMap, CUtensorMap, CUtensorMap, TcParams) = nullptr;
#define TECO_PICK(M, T, JJ, K) \
  if (pl.kmode == M && pl.TPS == T && pl.J == JJ && pl.KS == K) kern = conv3x3_tc_onetile_kernel<M, T, JJ, K>;
  // J = 2 needs >= 2 waves of 16-pixel-wide tiles: a conv that large is multi-wave and runs persistent, and a transposed
  // conv that large always fits 3-tap slabs
  TECO_PICK(0, 3, 1, 3) TECO_PICK(0, 3, 1, 1) TECO_PICK(0, 1, 1, 1)
  TECO_PICK(1, 3, 1, 1) TECO_PICK(1, 3, 2, 1) TECO_PICK(1, 1, 1, 1)
#undef TECO_PICK
  if (!kern) {
    teco_set_error("teco_conv3x3_tc(one-tile): no kernel instantiation for mode=%d TPS=%d J=%d KS=%d", pl.kmode, pl.TPS, pl.J, pl.KS);
    return TECO_E_UNSUPPORTED;
  }
  return tc_launch(kern, 224 * 1024, NUM_THREADS, pl, maps, p, stream);
}
