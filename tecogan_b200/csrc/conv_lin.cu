// Row-linearised 3x3 conv chain for 32-pixel-wide images (the metric configuration: clips of 32x32 LR frames) on tcgen05:
// L consecutive 64 -> 64 layers (bias, ReLU / none, optional residual) in ONE launch.
//
// Replaces the input conv + residual blocks of generator_F (reference lib/frvsr.py:59-70: conv2 -> relu, then
// num_resblock x [conv2 -> relu -> conv2 -> + input]) when the frame is 32 pixels wide.
//
// Why a second formulation (measured with tools/micro/mma_rate.cu on B200, profiles/r02_mma_rate.txt):
//   a tcgen05.mma M=128 N=64 K=16 costs ~51 cycles whatever the number of accumulator chains (62 % of the 32-cycle tensor
//   floor: the 4 KB A tile + 2 KB B tile are fetched from shared memory at 128 B/clk), while N >= 128 runs AT the floor
//   (N=128: 64.1, N=192: 96.1, N=256: 128.1 cycles).  The per-tap implicit GEMM of conv_tc.cu is stuck at N = Cout = 64.
// Here ONE MMA covers the three horizontal taps of a kernel row: B = [kx][cout] = 192 rows (the packed slab of kernel row ky
// exactly as teco_pack_conv3x3_bf16 lays it out), A = 128 pixels WITHOUT a horizontal shift.  Accumulator block kx at pixel x
// then holds tap kx's contribution to output pixel x + 1 - kx, and the epilogue forms
//     out(x) = D1(x) + D0(x-1) + D2(x+1)
// An image row is 32 pixels = 32 x 128 B = four 1024-byte swizzle atoms, so with a halo box WITHOUT side columns the 128 rows
// of an A tile are four whole image rows back to back (row pitch 4096 B, SBO 1024): TMEM lane = 32 * row + x, i.e. every
// epilogue warp (one TMEM lane quarter) owns one image row, x - 1 / x + 1 are warp shuffles, and the left / right zero
// padding of TF 'SAME' is "lane 0 / lane 31 receives 0".  Vertical taps are descriptor start offsets of whole rows (4096 B,
// atom aligned); top / bottom padding is the TMA out-of-bounds zero fill.  12 MMAs of 96 cycles per 128 pixels instead of
// 36 of ~51-60.
//
// Multi-layer: CTA c owns images c, c+G, ... for EVERY layer, so a layer's input strips were written by this very CTA:
// no grid-wide dependency, no kernel boundary, the MMA stream runs through all L layers.  The store thread publishes a
// count of completed TMA stores; the producer checks it (it is far ahead in practice) before loading a strip of the next layer.
// Weights of layer l+1 are fetched into the second weight buffer while layer l computes.
//
// Warp roles (352 threads): warp 0 = TMA producer (one lane, three non-blocking cursors: weight slabs, halo strips, residual
// strips), warp 1 = TMEM owner + MMA issuer, warps 2..9 = epilogue (lane quarter = image row, two warps per row each taking 32
// output channels), warp 10 = TMA store.
// What the microbenchmarks say about feeding the tensor pipe (tools/micro/mma_rate.cu, profiles/r02_mma_rate.txt): the MMA queue
// is shallow, so everything the issuing thread does between strips drains it -- an mbarrier test costs ~120 cycles even when it
// succeeds, a commit ~50, an integer division ~100.  Hence: no divisions in the issue loop, the two barrier tests of a strip in
// one round trip (two lanes), waiting warps sleep on their barriers instead of polling shared memory.  (Two issuer warps
// alternating strips were tried: their MMAs interleave and run at ~137 cycles each instead of 96 -- slower than one issuer.)
#include <cuda.h>
#include <cstdlib>
#include "teco_common.cuh"
#include "tc_ptx.cuh"

using namespace tcptx;

namespace {

constexpr int LW = 32;                                // image width in pixels
constexpr int STRIP_ROWS = 4;                         // M = 128 = 4 rows x 32 pixels
constexpr int HALO_ROWS = STRIP_ROWS + 2;
constexpr uint32_t ROW_BYTES = LW * 128;              // 4096
constexpr uint32_t HALO_BYTES = HALO_ROWS * ROW_BYTES;    // 24576
constexpr uint32_t STRIP_BYTES = STRIP_ROWS * ROW_BYTES;  // 16384
constexpr uint32_t W_SLAB_BYTES = 3 * 64 * 128;       // one kernel row: [kx][cout][64 cin] = 24576
constexpr uint32_t W_LAYER_BYTES = 3 * W_SLAB_BYTES;  // 73728
static_assert(W_LAYER_BYTES == 9 * 64 * 128, "one packed 64x64 layer (teco_pack_conv3x3_bf16)");
constexpr int MAX_LAYERS = 40;
constexpr int EPI_WARP0 = 2;                          // warps 2..9: epilogue (warp & 3 = TMEM lane quarter, (warp - 2) >> 2 = channel half)
constexpr int NUM_EPI_WARPS = 8;
constexpr int STORE_WARP = EPI_WARP0 + NUM_EPI_WARPS;
constexpr int NUM_THREADS = 32 * (STORE_WARP + 1);
constexpr uint32_t ACC_COLS = 192;                    // TMEM columns of one accumulator slot (3 taps x 64 channels)
constexpr int HST = 4;                                // halo ring: a strip's TMA takes ~1900 cycles to land, an MMA strip 1152
constexpr int WRING = 4;                              // weight ring of kernel-row slabs: three of the current layer + one ahead
constexpr size_t SMEM_BYTES = 2048 + HST * HALO_BYTES + 2 * STRIP_BYTES + WRING * W_SLAB_BYTES;   // + alignment slack: 231424

struct LinMaps {
  CUtensorMap ld[3];   // halo loads  {64 ch, 32 px, 6 rows, 1 image} of x_in / buf_a / buf_b
  CUtensorMap st[3];   // strip boxes {64 ch, 32 px, 4 rows, 1 image}: output store and residual load
};

struct LinParams {
  int N, H, L, G, spi;           // images, rows, layers, CTAs, strips per image
  const uint8_t* wpk;            // [L][73728] packed layers
  const float* bias;             // [L][64]
  int8_t in_buf[MAX_LAYERS], out_buf[MAX_LAYERS], res_buf[MAX_LAYERS], act[MAX_LAYERS];
  long long* dbg;                // optional [G][64] clock64 stamps (teco_debug_timing)
  int dbg_flags;                 // TECO_LIN_DBG (developer bisection): 1 no TMA store, 2 no epilogue math/staging writes, 4 halo TMA only for the first ring, 8 no TMEM loads
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
conv3x3_lin_kernel(const __grid_constant__ LinMaps maps, const LinParams p) {
  extern __shared__ uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // small region first, then the 1024-byte aligned operand buffers
  uint64_t* bars = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 15) & ~(uintptr_t)15);
  uint64_t* halo_full = bars;            // [HST]
  uint64_t* halo_empty = bars + 4;       // [HST]
  uint64_t* acc_full = bars + 8;         // [2]
  uint64_t* acc_empty = bars + 10;       // [2]  count NUM_EPI_WARPS
  uint64_t* res_full = bars + 12;        // [2]
  uint64_t* stage_free = bars + 14;      // [2]
  uint64_t* out_full = bars + 16;        // [2]  count NUM_EPI_WARPS
  uint64_t* w_full = bars + 18;          // [WRING]
  uint64_t* w_empty = bars + 22;         // [WRING]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 26);
  uint32_t* store_cnt = tmem_slot + 1;   // strips whose TMA store has completed (monotone)
  uint8_t* big = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(bars + 28) + 1023) & ~(uintptr_t)1023);
  uint8_t* halo = big;                                   // HST stages
  uint8_t* stage = halo + HST * HALO_BYTES;              // 2 staging strips (residual in, output out)
  uint8_t* wbuf = stage + 2 * STRIP_BYTES;               // WRING kernel-row slabs

  const int bid = blockIdx.x;
  const int imgs = bid < p.N ? (p.N - bid + p.G - 1) / p.G : 0;
  const int S = imgs * p.spi;            // strips per layer of this CTA
  const int total = S * p.L;
  long long* dbg = p.dbg ? p.dbg + (size_t)bid * 64 : nullptr;
#define LSTAMP(i) do { if (dbg) dbg[i] = clock64(); } while (0)
#define ESTAMP(g, i) do { if (dbg && (g) < 15) dbg[4 + (g) * 4 + (i)] = clock64(); } while (0)
  if (threadIdx.x == 0) { LSTAMP(0); if (dbg) { unsigned long long ns; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns)); dbg[1] = (long long)ns; } }

  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) {
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_empty[i]), 1);
      mbar_init(smem_u32(&w_full[i]), 1);
      mbar_init(smem_u32(&w_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&acc_full[i]), 1);
      mbar_init(smem_u32(&acc_empty[i]), NUM_EPI_WARPS);
      mbar_init(smem_u32(&res_full[i]), 1);
      mbar_init(smem_u32(&stage_free[i]), 1);
      mbar_init(smem_u32(&out_full[i]), NUM_EPI_WARPS);
    }
    *store_cnt = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int i = 0; i < 3; ++i) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.ld[i]) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.st[i]) : "memory");
    }
  }
  if (warp == 1) {   // TMEM owner
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  pdl_launch_dependents();
  const uint32_t tmem_base = *tmem_slot;

  // element g of this CTA's sequence -> (layer, image, first row)
  auto decode = [&](int g, int& l, int& r, int& img, int& y0) {
    l = g / S;
    r = g - l * S;
    const int ii = r / p.spi;
    img = bid + ii * p.G;
    y0 = (r - ii * p.spi) * STRIP_ROWS;
  };

  if (warp == 0) {
    // ===================== TMA producer: ONE lane, three cursors (weight slabs, halo strips, residual strips) =====================
    // Each cursor advances only when its barrier test succeeds (mbarrier.test_wait: no blocking), so a stalled cursor never
    // holds the others back.  (Three lanes spinning in divergent loops of one warp starved each other: the multi-layer chain
    // crawled.)
    if (lane == 0 && total > 0) {
      const int nslab = 3 * p.L;
      int qw = 0, gh = 0, gr = 0;
      auto issue_slab = [&](int q) {
        const int st = q & (WRING - 1);
        mbar_expect_tx(smem_u32(&w_full[st]), W_SLAB_BYTES);
        bulk_load_1d(smem_u32(wbuf + (size_t)st * W_SLAB_BYTES), p.wpk + (size_t)q * W_SLAB_BYTES, W_SLAB_BYTES, smem_u32(&w_full[st]));
      };
      // Weight slab q = 3 * layer + ky through a ring of WRING slabs: three of the current layer + one ahead; slab (l, ky) is
      // released by the layer's LAST strip as soon as its ky group of MMAs has retired.  The first WRING slabs depend on nothing.
      for (; qw < nslab && qw < WRING; ++qw) issue_slab(qw);
      pdl_wait();                         // the previous kernel's output (x_in) is complete and visible from here on
      int hl = 0, hr = 0, himg = bid, hy0 = 0;          // decoded halo cursor
      int rl = 0, rr = 0, rimg = bid, ry0 = 0;          // decoded residual cursor
      while (qw < nslab || gh < total || gr < total) {
        const int before = qw + gh + gr;
        if (qw < nslab && mbar_test(smem_u32(&w_empty[qw & (WRING - 1)]), (uint32_t)(((qw >> 2) - 1) & 1))) {
          issue_slab(qw);
          ++qw;
        }
        if (gh < total) {
          // rows y0-1 .. y0+4 of the previous layer's output: strips r-1, r, r+1 of that layer (same image) must be stored.
          // Stores complete in sequence order, so "strip min(r+1, ..) of layer l-1 done" is a count.
          bool ok = true;
          if (hl > 0) {
            const uint32_t need = (uint32_t)((hl - 1) * S + hr + (hy0 / STRIP_ROWS + 1 < p.spi ? 1 : 0) + 1);
            ok = ld_acquire_cta_smem(smem_u32(store_cnt)) >= need;
          }
          const int hs = gh & (HST - 1);
          if (ok && mbar_test(smem_u32(&halo_empty[hs]), (uint32_t)(((gh >> 2) & 1) ^ 1))) {
            if ((p.dbg_flags & 4) && gh >= HST) {
              mbar_arrive(smem_u32(&halo_full[hs]));
            } else {
              if (hl > 0) fence_proxy_async_global();   // this CTA's async-proxy stores are ordered before this async-proxy load
              mbar_expect_tx(smem_u32(&halo_full[hs]), HALO_BYTES);
              tma_load_4d(smem_u32(halo + (size_t)hs * HALO_BYTES), &maps.ld[p.in_buf[hl]], smem_u32(&halo_full[hs]), 0, 0, hy0 - 1, himg);
            }
            ++gh;
            if (gh < total) decode(gh, hl, hr, himg, hy0);
          }
        }
        if (gr < total) {
          // residual strips go straight into the staging strip the epilogue will overwrite in place; the cursor waits for the
          // staging ring on EVERY strip (also in layers without a residual) so that it never runs more than one barrier phase
          // ahead -- a parity test two uses ahead would read a stale phase as "done"
          bool ok = true;
          const bool has_res = p.res_buf[rl] >= 0;
          if (has_res && rl >= 2)         // written by an earlier layer of this launch (the same strip, at least S strips ago)
            ok = ld_acquire_cta_smem(smem_u32(store_cnt)) >= (uint32_t)((rl - 2) * S + rr + 1);
          if (ok && mbar_test(smem_u32(&stage_free[gr & 1]), (uint32_t)(((gr >> 1) & 1) ^ 1))) {   // the store of strip g - 2 has read it
            if (has_res) {
              if (rl >= 2) fence_proxy_async_global();
              mbar_expect_tx(smem_u32(&res_full[gr & 1]), STRIP_BYTES);
              tma_load_4d(smem_u32(stage + (size_t)(gr & 1) * STRIP_BYTES), &maps.st[p.res_buf[rl]], smem_u32(&res_full[gr & 1]), 0, 0, ry0, rimg);
            }
            ++gr;
            if (gr < total) decode(gr, rl, rr, rimg, ry0);
          }
        }
        // nothing moved: the rings are full (the producer runs several strips ahead) -- stay off the shared-memory pipe for a while
        if (qw + gh + gr == before) __nanosleep(200);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = umma_idesc_mn(128, (int)ACC_COLS);
    int l = 0, r = 0;                     // layer and strip-in-layer of element g (no divisions in the loop)
    // the two barriers of a strip in ONE round trip: lane 0 polls the accumulator slot (drained by the epilogue), lane 1 the halo
    auto wait_strip = [&](int g) {
      const uint32_t bar = lane == 0 ? smem_u32(&acc_empty[g & 1]) : smem_u32(&halo_full[g & (HST - 1)]);
      const uint32_t par = lane == 0 ? (uint32_t)(((g >> 1) & 1) ^ 1) : (uint32_t)((g >> 2) & 1);
      if (lane < 2) mbar_wait(bar, par);
      __syncwarp();
    };
    for (int g = 0; g < total; ++g) {
      const int slot = g & 1, hs = g & (HST - 1);
      wait_strip(g);
      tcgen05_fence_after();
      if (lane == 0 && !(p.dbg_flags & 16)) ESTAMP(g, 0);
      const uint32_t d = tmem_base + (uint32_t)slot * ACC_COLS;
      const uint64_t a_base = umma_desc_sw128(smem_u32(halo + (size_t)hs * HALO_BYTES), 1024);
      const int q0 = 3 * l;
      if (r == 0) {                       // first strip of a layer: its weights may still be landing (three slabs, three lanes)
        if (lane < 3) mbar_wait(smem_u32(&w_full[(q0 + lane) & (WRING - 1)]), (uint32_t)(((q0 + lane) >> 2) & 1));
        __syncwarp();
        tcgen05_fence_after();
      }
      const bool last = r == S - 1;       // last strip of the layer: release the slabs as their MMAs retire
      auto issue_rows = [&](int ky0, int ky1) {
        if (elect_one()) {
#pragma unroll
          for (int ky = ky0; ky < ky1; ++ky) {
            const int ws = (q0 + ky) & (WRING - 1);
            const uint64_t b_base = umma_desc_sw128(smem_u32(wbuf + (size_t)ws * W_SLAB_BYTES), 1024);
#pragma unroll
            for (int s = 0; s < 4; ++s)
              umma_bf16(d, a_base + (uint32_t)((ky * ROW_BYTES + s * 32) >> 4), b_base + (uint32_t)((s * 32) >> 4), idesc,
                        (ky == 0 && s == 0) ? 0u : 1u);
            if (last) tcgen05_commit(smem_u32(&w_empty[ws]));
          }
          if (ky1 == 3) {
            tcgen05_commit(smem_u32(&halo_empty[hs]));
            tcgen05_commit(smem_u32(&acc_full[slot]));
          }
        }
        __syncwarp();
      };
      // (Polling the NEXT strip's barriers here, between the second and third kernel row, was tried: the accumulator slot of
      //  strip g + 1 is released by the epilogue of g - 1, which is only just starting -- the poll blocked and P rose to 2360.)
      issue_rows(0, 3);
      if (lane == 0 && !(p.dbg_flags & 16)) ESTAMP(g, 1);
      if (++r == S) { r = 0; ++l; }
    }
  } else if (warp == STORE_WARP) {
    // ===================== output store =====================
    if (lane == 0) {
      for (int g = 0; g < total; ++g) {
        int l, r, img, y0;
        decode(g, l, r, img, y0);
        const int sg = g & 1;
        mbar_wait_sleepy(smem_u32(&out_full[sg]), (uint32_t)((g >> 1) & 1));   // every epilogue warp has fenced and arrived
        if (!(p.dbg_flags & 1)) tma_store_4d(&maps.st[p.out_buf[l]], smem_u32(stage + (size_t)sg * STRIP_BYTES), 0, 0, y0, img);
        bulk_commit();
        bulk_wait_read();                 // the staging strip may be overwritten again
        mbar_arrive(smem_u32(&stage_free[sg]));
        // Publish completed stores (strips in global memory: later layers of this CTA may load them).  Waiting for the newest
        // store here would serialise the stores at their full latency, so the count lags two strips behind -- the consumers
        // are S - 1 strips away.  With fewer than four strips per layer the lag could stall the chain: wait for everything.
        if (S >= 4 && g + 1 < total) {
          asm volatile("cp.async.bulk.wait_group 2;" ::: "memory");
          if (g >= 2) {
            fence_proxy_async_global();
            st_release_cta_smem(smem_u32(store_cnt), (uint32_t)(g - 1));
          }
        } else {
          bulk_wait_all();
          fence_proxy_async_global();
          st_release_cta_smem(smem_u32(store_cnt), (uint32_t)(g + 1));
        }
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..9) =====================
    const int q = warp & 3;               // TMEM lane quarter = image row of the strip
    const int chalf = (warp - EPI_WARP0) >> 2;   // which 32 of the 64 output channels
    const uint32_t m = (uint32_t)(32 * q + lane);
    const uint32_t rowoff = m * 128u, sw = m & 7u;
    uint32_t res_uses0 = 0u, res_uses1 = 0u;   // residual strips seen per staging slot (res_full phase)
    float bias_r[32];
    int l = 0, r = 0, act = 0;
    bool has_res = false;
    for (int g = 0; g < total; ++g) {
      const int slot = g & 1;
      if (r == 0) {
        const float* bp = p.bias + (size_t)l * 64 + 32 * chalf;
#pragma unroll
        for (int i = 0; i < 32; ++i) bias_r[i] = __ldg(bp + i);
        act = p.act[l];
        has_res = p.res_buf[l] >= 0;
      }
      if (lane == 0 && !mbar_test(smem_u32(&acc_full[slot]), (uint32_t)((g >> 1) & 1)))   // usually complete already: the MMAs run ahead
        mbar_wait_sleepy(smem_u32(&acc_full[slot]), (uint32_t)((g >> 1) & 1));
      __syncwarp();
      tcgen05_fence_after();
      if (threadIdx.x == 64) ESTAMP(g, 2);
      const uint32_t tb = tmem_base + (uint32_t)slot * ACC_COLS + ((uint32_t)(32 * q) << 16) + (uint32_t)(32 * chalf);
      uint32_t d0[32], d1[32], d2[32];
      if (!(p.dbg_flags & 8)) {
        tmem_ld32(tb, d0);
        tmem_ld32(tb + 64, d1);
        tmem_ld32(tb + 128, d2);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) d0[i] = d1[i] = d2[i] = 0u;
      }
      // while the TMEM loads are in flight: the staging strip -- residual landed (which implies it was free), or free of the
      // store of strip g - 2
      if (has_res) {
        mbar_wait_warp_sleepy(smem_u32(&res_full[slot]), (slot ? res_uses1 : res_uses0) & 1u);
        if (slot) ++res_uses1; else ++res_uses0;
      } else {
        mbar_wait_warp_sleepy(smem_u32(&stage_free[slot]), (uint32_t)(((g >> 1) & 1) ^ 1));
      }
      if (!(p.dbg_flags & 8)) tmem_wait_ld();
      if (threadIdx.x == 64 && (p.dbg_flags & 16)) ESTAMP(g, 0);   // epilogue phase stamps: TMEM data in registers
      tcgen05_fence_before();
      if (lane == 0) mbar_arrive(smem_u32(&acc_empty[slot]));   // accumulator slot back to the MMA issuer
      if (!(p.dbg_flags & 2)) {
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float lo = __shfl_up_sync(0xffffffffu, __uint_as_float(d0[i]), 1);     // tap kx = 0 computed at pixel x - 1
          const float hi = __shfl_down_sync(0xffffffffu, __uint_as_float(d2[i]), 1);   // tap kx = 2 computed at pixel x + 1
          float a = __uint_as_float(d1[i]) + bias_r[i];
          if (lane != 0) a += lo;         // TF 'SAME' zero padding left / right of the 32-pixel row: lane 0 / 31 add nothing
          if (lane != 31) a += hi;
          v[i] = a;
        }
        if (act == TECO_ACT_RELU) {       // warp-uniform per layer
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.f);
        } else if (act == TECO_ACT_LRELU02) {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.2f * v[i]);
        }
        if (threadIdx.x == 64 && (p.dbg_flags & 16)) ESTAMP(g, 1);   // ... shuffles + bias + activation done
        uint8_t* row = stage + (size_t)slot * STRIP_BYTES + rowoff;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint4* cell = reinterpret_cast<uint4*>(row + ((((uint32_t)(4 * chalf + k)) ^ sw) << 4));   // XOR swizzle of the TMA box
          if (has_res) {
            const uint4 rr = *cell;
            const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rw[i]));
              v[8 * k + 2 * i] += f.x;
              v[8 * k + 2 * i + 1] += f.y;
            }
          }
          uint32_t o[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(v[8 * k + 2 * i], v[8 * k + 2 * i + 1]);
            o[i] = *reinterpret_cast<uint32_t*>(&h);
          }
          *cell = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
      fence_async_smem();                 // generic-proxy writes -> visible to the TMA store
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&out_full[slot]));
      if (threadIdx.x == 64) ESTAMP(g, 3);
      if (++r == S) { r = 0; ++l; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) { LSTAMP(3); if (dbg) { unsigned long long ns; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns)); dbg[2] = (long long)ns; } }
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

}  // namespace

extern long long* teco_g_dbg_timing;   // conv_tc.cu

extern "C" int teco_conv3x3_lin_supported(int32_t N, int32_t H, int32_t W, int32_t num_layers) {
  return (N > 0 && W == LW && H >= STRIP_ROWS && H % STRIP_ROWS == 0 && H <= 4096 && num_layers >= 1 && num_layers <= MAX_LAYERS) ? 1 : 0;
}

extern "C" int teco_conv3x3_lin_tc(int32_t N, int32_t H, int32_t W, int32_t num_layers, const void* x_in, void* buf_a, void* buf_b,
                                   const void* wpk_all, const float* bias_all, const int32_t* plan_host, void* stream) {
  TECO_CHECK_ARG(teco_conv3x3_lin_supported(N, H, W, num_layers),
                 "teco_conv3x3_lin_tc: needs W == 32, H a multiple of 4, 1..%d layers (got N=%d H=%d W=%d L=%d)", MAX_LAYERS, N, H, W, num_layers);
  TECO_CHECK_ARG(wpk_all && bias_all && plan_host, "teco_conv3x3_lin_tc: NULL weights / bias / plan");
  void* bufs[3] = {const_cast<void*>(x_in), buf_a, buf_b};
  LinParams p;
  p.N = N; p.H = H; p.L = num_layers; p.spi = H / STRIP_ROWS;
  p.wpk = (const uint8_t*)wpk_all; p.bias = bias_all; p.dbg = teco_g_dbg_timing;
  { const char* e = getenv("TECO_LIN_DBG"); p.dbg_flags = e ? atoi(e) : 0; }
  for (int l = 0; l < num_layers; ++l) {
    const int in = plan_host[4 * l], out = plan_host[4 * l + 1], res = plan_host[4 * l + 2], act = plan_host[4 * l + 3];
    TECO_CHECK_ARG(in >= 0 && in < 3 && out >= 1 && out < 3 && res >= -1 && res < 3 && in != out,
                   "teco_conv3x3_lin_tc: layer %d: bad buffer plan (in=%d out=%d res=%d; 0 = x_in, 1 = buf_a, 2 = buf_b, x_in is read-only)", l, in, out, res);
    TECO_CHECK_ARG(act == TECO_ACT_NONE || act == TECO_ACT_RELU || act == TECO_ACT_LRELU02, "teco_conv3x3_lin_tc: layer %d: activation %d", l, act);
    TECO_CHECK_ARG(bufs[in] && bufs[out] && (res < 0 || bufs[res]), "teco_conv3x3_lin_tc: layer %d uses a NULL buffer", l);
    // a layer may add its residual in place (res == out) but must never read its input from where it writes; the residual of
    // layer l is read by the strip that overwrites it, and only layers >= 2 back may have produced it inside this launch
    TECO_CHECK_ARG(res < 0 || l == 0 || res != plan_host[4 * (l - 1) + 1] || res == 0,
                   "teco_conv3x3_lin_tc: layer %d: the residual may not be the previous layer's output (its stores are not tracked)", l);
    p.in_buf[l] = (int8_t)in; p.out_buf[l] = (int8_t)out; p.res_buf[l] = (int8_t)res; p.act[l] = (int8_t)act;
  }
  for (int i = 0; i < 3; ++i)
    TECO_CHECK_ARG((((uintptr_t)bufs[i]) & 15) == 0, "teco_conv3x3_lin_tc: tensors must be 16-byte aligned");
  TECO_CHECK_ARG((((uintptr_t)wpk_all) & 15) == 0, "teco_conv3x3_lin_tc: packed weights must be 16-byte aligned");
  const int sms = teco_sm_count();
  p.G = N < sms ? N : sms;

  LinMaps maps;
  for (int i = 0; i < 3; ++i) {
    void* base = bufs[i] ? bufs[i] : bufs[1] ? bufs[1] : bufs[0];   // an unused slot still needs a valid map
    if (int e = teco_tmap_nhwc(&maps.ld[i], "teco_conv3x3_lin_tc", base, N, H, LW, 64, 64, LW, HALO_ROWS)) return e;
    if (int e = teco_tmap_nhwc(&maps.st[i], "teco_conv3x3_lin_tc", base, N, H, LW, 64, 64, LW, STRIP_ROWS)) return e;
  }
  TECO_CUDA_CALL(cudaFuncSetAttribute(conv3x3_lin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)p.G);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attrs[1];
  attrs[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // PDL: prologue + first weights overlap the previous kernel's tail
  attrs[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = 1;
  cudaError_t le = cudaLaunchKernelEx(&cfg, conv3x3_lin_kernel, maps, p);
  if (le != cudaSuccess) {
    teco_set_error("teco_conv3x3_lin_tc: launch failed: %s (grid %d, smem %zu)", cudaGetErrorString(le), p.G, SMEM_BYTES);
    return TECO_E_CUDA;
  }
  return TECO_OK;
}
