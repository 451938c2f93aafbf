// Weight gradient of the 3x3 stride-1 SAME convolution on the 5th-gen tensor cores (sm_100a).
//
// Replaces the gradient TensorFlow computes for slim.conv2d (reference lib/ops.py:47-56) inside
// tf.train.AdamOptimizer.compute_gradients (reference lib/Teco.py:426,446-447):
//     dW[ky][kx][ci][co] += sum over pixels p of  X[p + (ky-1, kx-1)][ci] * dZ[p][co]
// i.e. one GEMM per tap with the PIXELS as the contraction dimension.  Both operands are NHWC bf16 with 64 channels per
// 128-byte row, so as UMMA operands they are "MN-major" (the M / N index -- the channel -- is the contiguous one, K = the
// pixel steps from row to row): exactly the SWIZZLE_128B image a TMA box leaves in shared memory, no transposition.
//   * CTA = one 8x16-pixel tile of one image and one (64 input channel, 64 output channel) block pair.
//   * A K-step is one image row of the tile = 16 consecutive pixels = two 8-row swizzle atoms (SBO = 1024 B).
//   * Two taps share one MMA: M = 128 = [64 ci of tap t | 64 ci of tap t+1]; the second 64-row atom of the A operand is
//     simply the same halo box LBO bytes further on (one pixel = 128 B for the next kx, or a box row minus two pixels for
//     the wrap to the next ky).  9 taps = 4 pairs (M=128) + 1 single (M=64): five accumulators of 64 fp32 columns in TMEM,
//     written round-robin so consecutive MMAs never depend on each other.
//   * Epilogue: thread = (tap of the pair, ci), 64 co in registers -> 16-byte fp32 atomics into dW[3,3,Cin,Cout] (TF layout).
#include <cuda.h>
#include "teco_common.cuh"
#include "tc_ptx.cuh"

namespace {
using namespace tcptx;

constexpr int WG_ROWS = 8, WG_COLS = 16;
constexpr int WG_HALO_BYTES = (WG_ROWS + 2) * (WG_COLS + 2) * 128;   // 23040
constexpr int WG_DZ_BYTES = WG_ROWS * WG_COLS * 128;                 // 16384

struct WgParams {
  int N, H, W, Cin, Cout;      // real channel counts of dW
  int cob, tiles_x, tiles_y;   // 64-channel output blocks, tiles per image
  float* dw;
};

// MN-major SWIZZLE_128B shared-memory descriptor (cute::UMMA canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte
// units): 64 contiguous MN elements per 128-byte row, K advances row by row, LBO = next 64 MN elements, SBO = next 8 K rows.
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) |
         (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D fp32, A/B bf16, BOTH operands MN-major (bits 15, 16), N >> 3 @17, M >> 4 @24
__device__ __forceinline__ uint32_t idesc_mn(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__global__ void __launch_bounds__(128)
conv3x3_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dz, const WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* halo = smem;                                   // [10 rows][18 px][128 B]
  uint8_t* dzt = smem + ((WG_HALO_BYTES + 1023) & ~1023); // [8 rows][16 px][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(dzt + WG_DZ_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  int tile = blockIdx.x;
  const int tx = tile % p.tiles_x; tile /= p.tiles_x;
  const int ty = tile % p.tiles_y;
  const int n = tile / p.tiles_y;
  const int cb = blockIdx.y / p.cob, ob = blockIdx.y - cb * p.cob;
  const int x0 = tx * WG_COLS, y0 = ty * WG_ROWS;

  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&bars[0]), 1);
    mbar_init(smem_u32(&bars[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(smem_u32(&bars[0]), (uint32_t)(WG_HALO_BYTES + WG_DZ_BYTES));
      tma_load_4d(smem_u32(halo), &tmap_x, smem_u32(&bars[0]), cb * 64, x0 - 1, y0 - 1, n);   // zero fill = SAME padding
      tma_load_4d(smem_u32(dzt), &tmap_dz, smem_u32(&bars[0]), ob * 64, x0, y0, n);
    }
    mbar_wait_warp(smem_u32(&bars[0]), 0);
    tcgen05_fence_after();
    const uint32_t halo_a = smem_u32(halo), dz_a = smem_u32(dzt);
    const uint32_t id128 = idesc_mn(128, 64);
    if (elect_one()) {
#pragma unroll 1
      for (int r = 0; r < WG_ROWS; ++r) {
        const uint64_t b_desc = desc_mn_sw128(dz_a + (uint32_t)(r * WG_COLS * 128), 0u, 1024u);
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          const int t0 = 2 * q, t1 = 2 * q + 1;
          const int o0 = ((r + t0 / 3) * (WG_COLS + 2) + t0 % 3) * 128;
          const int o1 = ((r + t1 / 3) * (WG_COLS + 2) + t1 % 3) * 128;
          // (the ninth tap runs as M = 128 too, its second half re-reading the same rows: an M = 64 accumulator is laid out
          //  over 16 lanes of each TMEM sub-partition, not over lanes 0..63; the duplicate half is dropped in the epilogue)
          const uint64_t a_desc = desc_mn_sw128(halo_a + (uint32_t)o0, q < 4 ? (uint32_t)(o1 - o0) : 0u, 1024u);
          umma_bf16(tmem + (uint32_t)(q * 64), a_desc, b_desc, id128, r > 0 ? 1u : 0u);
        }
      }
      tcgen05_commit(smem_u32(&bars[1]));
    }
    __syncwarp();
  }
  mbar_wait_warp(smem_u32(&bars[1]), 0);
  tcgen05_fence_after();

  // ---- epilogue: accumulator q, lane m -> tap 2q + (m >= 64), input channel cb*64 + (m & 63); columns = output channels
  const int m = 32 * warp + lane;
  const int ci = cb * 64 + (m & 63);
  const int co0 = ob * 64;
#pragma unroll 1
  for (int q = 0; q < 5; ++q) {
    const int tap = 2 * q + (m >> 6);
    uint32_t r0[32], r1[32];
    __syncwarp();
    tmem_ld32(tmem + ((uint32_t)(32 * warp) << 16) + (uint32_t)(q * 64), r0);
    tmem_ld32(tmem + ((uint32_t)(32 * warp) << 16) + (uint32_t)(q * 64 + 32), r1);
    tmem_wait_ld();
    if (tap < 9 && ci < p.Cin) {
      float* dst = p.dw + ((size_t)tap * p.Cin + ci) * p.Cout + co0;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (co0 + 4 * k < p.Cout)
          atomicAdd(reinterpret_cast<float4*>(dst + 4 * k), make_float4(__uint_as_float(r0[4 * k]), __uint_as_float(r0[4 * k + 1]),
                                                                       __uint_as_float(r0[4 * k + 2]), __uint_as_float(r0[4 * k + 3])));
        if (co0 + 32 + 4 * k < p.Cout)
          atomicAdd(reinterpret_cast<float4*>(dst + 32 + 4 * k), make_float4(__uint_as_float(r1[4 * k]), __uint_as_float(r1[4 * k + 1]),
                                                                            __uint_as_float(r1[4 * k + 2]), __uint_as_float(r1[4 * k + 3])));
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

}  // namespace

extern "C" int teco_conv3x3_wgrad_tc(int32_t N, int32_t H, int32_t W, int32_t cin_pad, int32_t cout_pad, int32_t cin, int32_t cout,
                                     const void* x, const void* dz, float* dw, int32_t accumulate, void* stream) {
  TECO_CHECK_ARG(x && dz && dw, "teco_conv3x3_wgrad_tc: NULL tensor");
  TECO_CHECK_ARG(N > 0 && H > 0 && W > 0, "teco_conv3x3_wgrad_tc: bad shape N=%d H=%d W=%d", N, H, W);
  TECO_CHECK_ARG(cin_pad % 64 == 0 && cout_pad % 64 == 0 && cin > 0 && cout > 0 && cin <= cin_pad && cout <= cout_pad,
                 "teco_conv3x3_wgrad_tc: x / dz must carry multiples of 64 channels (got %d, %d for %d -> %d)", cin_pad, cout_pad, cin, cout);
  TECO_CHECK_ARG(cout % 4 == 0, "teco_conv3x3_wgrad_tc: Cout must be a multiple of 4 (16-byte atomics into dW), got %d", cout);
  TECO_CHECK_ARG((((uintptr_t)x) & 15) == 0 && (((uintptr_t)dz) & 15) == 0 && (((uintptr_t)dw) & 15) == 0,
                 "teco_conv3x3_wgrad_tc: tensors must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  if (!accumulate) TECO_CUDA_CALL(cudaMemsetAsync(dw, 0, sizeof(float) * (size_t)9 * cin * cout, s));
  CUtensorMap tx, tz;
  if (int e = teco_tmap_nhwc(&tx, "teco_conv3x3_wgrad_tc (x)", x, N, H, W, cin_pad, 64, WG_COLS + 2, WG_ROWS + 2)) return e;
  if (int e = teco_tmap_nhwc(&tz, "teco_conv3x3_wgrad_tc (dz)", dz, N, H, W, cout_pad, 64, WG_COLS, WG_ROWS)) return e;
  WgParams p;
  p.N = N; p.H = H; p.W = W; p.Cin = cin; p.Cout = cout;
  p.cob = teco_ceil_div(cout, 64);
  p.tiles_x = teco_ceil_div(W, WG_COLS);
  p.tiles_y = teco_ceil_div(H, WG_ROWS);
  p.dw = dw;
  const long long tiles = (long long)N * p.tiles_x * p.tiles_y;
  TECO_CHECK_ARG(tiles < (1LL << 31), "teco_conv3x3_wgrad_tc: too many tiles");
  const int cib = teco_ceil_div(cin, 64);
  const size_t smem = 1024 + ((WG_HALO_BYTES + 1023) & ~1023) + WG_DZ_BYTES + 64;
  TECO_CUDA_CALL(cudaFuncSetAttribute(conv3x3_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  conv3x3_wgrad_tc_kernel<<<dim3((unsigned)tiles, (unsigned)(cib * p.cob)), 128, smem, s>>>(tx, tz, p);
  TECO_CUDA_LAUNCH_CHECK("teco_conv3x3_wgrad_tc");
  return TECO_OK;
}
