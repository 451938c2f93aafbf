// warp_s2d_v2.cu -- second version of the fused feedback kernel for the inference layout (bf16 destination inside the packed
// 64-channel generator input, no fp32 copy of the warped frame):
//   flow_lr -> symmetric pad, x4, upscale_four -> dense_image_warp(previous HR output) -> space_to_depth
// (reference main.py:201,212-215; lib/ops.py:126-163 upscale_four; tf.contrib.image.dense_image_warp).  Same arithmetic,
// formula for formula, as warp_s2d_fused_kernel in resample.cu (which keeps every other layout: fp32 destinations,
// warped_out, unaligned channel offsets); what changes is the instruction count per HR pixel.  ncu of the first version
// (profiles/r02_warp_s2d_32x1024_summary.txt): 195 thread instructions per HR pixel, issue slots 76 % busy, DRAM at 37 % --
// issue-bound, not memory-bound.  Here:
//   * CTA tile 4 x 32 LR pixels (16 x 128 HR): the per-tile work (flow bound, window set-up, barriers) is paid once per 2048
//     HR pixels instead of 1024, and the staged source window carries 2 halo rows per 16 instead of per 8;
//   * the 5 x 33 flow samples of the tile are parked in shared memory once (no thread repeats the symmetric-pad index
//     arithmetic or goes back to global memory); warp 0 bounds them with four redux.sync on order-preserving integer keys
//     (was 40 shuffle / min / max instructions in four warps plus a serial stage), derives the source window and stages it
//     with ONE BULK COPY PER WINDOW ROW on an mbarrier (TMA engine: no register, LSU or issue-slot cost for the window;
//     the cp.async loop it replaced was 22 % of all instructions) while the other warps interpolate their flows;
//   * floor() is ONE add with round-toward-minus-infinity against 1.5 * 2^23 (the sum's mantissa is the integer), the index
//     arithmetic works directly on that bit pattern (two IMADs per pixel), clamps only on the axes whose tile can touch one;
//   * results go through a bf16 staging tile in shared memory in destination order and leave as 16-byte stores, six per LR
//     pixel (was: three shuffles, eight selects and an 8-byte store per HR pixel with a quarter of the lanes idle);
//   * rough motion (window larger than the 40 KB stage): the tile in two halves with their own windows, then an L1 gather.
// Measured (profiles/r02_warp_versions_ab.txt, r02_warp_s2d_v2_32x1024_summary.txt): 239 -> 160 us on 32 x 1024x1024 HR frames
// (0.39 -> 0.59 of the measured copy bandwidth), bit-identical output; 113 M instead of 204 M warp instructions.
#include "teco_common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int V2_TPB = 256;
constexpr int V2_TLH = 4, V2_TLW = 32;                       // LR tile; thread = one HR column x two LR rows (8 HR pixels)
constexpr int V2_WIN_FLOATS = 10 * 1024;                     // 40 KB source window: 24 rows x 140 px of fp32 RGB fit
constexpr int V2_STAGE_BYTES = V2_TLH * V2_TLW * 96;         // 12 KB: 48 bf16 per LR pixel
constexpr int V2_NSAMP = (V2_TLH + 1) * (V2_TLW + 1);        // 165 flow samples bound every HR flow vector of the tile
constexpr float V2_MAGIC = 12582912.f;                       // 1.5 * 2^23
constexpr int V2_MAGIC_BITS = 0x4B400000;

__device__ __forceinline__ int f2key(float v) {              // order-preserving float -> int
  const int i = __float_as_int(v);
  return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float key2f(int k) { return __int_as_float(k ^ ((k >> 31) & 0x7fffffff)); }

struct V2Smem {
  float2 flow[V2_NSAMP + 3];      // 4 * flow_lr at (ly0 + r, lx0 + j), clamped like upscale_four, symmetric pad applied
  unsigned long long bar;         // mbarrier of the window's bulk copies
  float mm[4];                    // min fy, max fy, min fx, max fx over the tile's flow samples
  int win[5];                     // y_lo, x_lo, rows, floats per window row, flags (1 staged, 2 interior in y, 4 interior in x)
};

struct V2Thread {                 // per-thread constants of the pixel loop
  float Xf, hy, hx, in_scale, in_shift;
  int pitch;
  unsigned cbase;
};

struct V2Window { int y_lo, x_lo, rows, rowf, flags; };

// Window of the previous HR frame that holds every query of HR rows [Yt, Yt + nrows) x columns [X0, X0 + 128) given the bounds
// of the flow over the tile (same construction as the first version): queries Y - fy lie in [Yt - mxy, Yt + nrows - 1 - mny],
// the floor is clamped to [0, H-2], plus the +1 neighbour row; columns alike.
__device__ __forceinline__ V2Window v2_window(float mny, float mxy, float mnx, float mxx, int Yt, int nrows, int X0, int H, int W,
                                              int win_floats = V2_WIN_FLOATS) {
  const float hy = (float)(H - 2), hx = (float)(W - 2);
  const float qy_lo = (float)Yt - mxy, qy_hi = (float)(Yt + nrows - 1) - mny;
  const float qx_lo = (float)X0 - mxx, qx_hi = (float)(X0 + 4 * V2_TLW - 1) - mnx;
  V2Window v;
  v.y_lo = (int)fminf(fmaxf(floorf(qy_lo) - 1.f, 0.f), hy);
  const int y_hi = (int)fminf(fmaxf(floorf(qy_hi) + 1.f, 0.f), hy) + 1;
  v.x_lo = (int)fminf(fmaxf(floorf(qx_lo) - 1.f, 0.f), hx) & ~3;               // whole groups of four pixels (48 bytes):
  const int x_hi = min(((int)fminf(fmaxf(floorf(qx_hi) + 1.f, 0.f), hx) + 1) | 3, W - 1);   // 16-byte aligned window rows
  v.rows = y_hi - v.y_lo + 1;
  v.rowf = (x_hi - v.x_lo + 1) * 3;
  v.flags = v.rows * v.rowf <= win_floats ? 1 : 0;
  // no query can touch a clamp on this axis: the floor needs no clamp and the fraction is already in [0,1)
  v.flags |= (qy_lo >= 1.f && qy_hi <= (float)(H - 3)) ? 2 : 0;
  v.flags |= (qx_lo >= 1.f && qx_hi <= (float)(W - 3)) ? 4 : 0;
  return v;
}

// One warp stages a window: one bulk copy (TMA engine, no register or LSU traffic) per window row, all signalling `bar`.
__device__ __forceinline__ void v2_stage(const float* img, int W, const V2Window& v, float* win, uint32_t bar, int lane) {
  const uint32_t row_bytes = (uint32_t)v.rowf * 4u;
  if (lane == 0) tcptx::mbar_expect_tx(bar, (uint32_t)v.rows * row_bytes);
  __syncwarp();
  const float* src0 = img + ((size_t)v.y_lo * W + v.x_lo) * 3;
  const uint32_t sbase = tcptx::smem_u32(win);
  for (int r = lane; r < v.rows; r += 32)
    tcptx::bulk_load_1d(sbase + (uint32_t)r * row_bytes, src0 + (size_t)r * (W * 3), row_bytes, bar);
}

// NK LR rows (4 NK HR pixels) of one thread's HR column.  Fy / Fx: x-interpolated flow of the NK + 1 LR sample rows around
// them; Yf: HR row of the first pixel; srow: this thread's slot of the first LR row in the staging tile.
// IY / IX: no query of the tile can touch a clamp on that axis (CTA-uniform) -- template parameters because ptxas otherwise
// predicates both variants into every pixel.
template <bool IY, bool IX, int NK>
__device__ __forceinline__ void v2_pixels(const float* __restrict__ base, const V2Thread& t, const float* Fy, const float* Fx,
                                          float Yf, unsigned char* srow) {
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    const float Ty = Fy[k], Dy = Fy[k + 1] - Ty, Tx = Fx[k], Dx = Fx[k + 1] - Tx;
    const float Yk = Yf + (float)(4 * k);
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      // flow = T + (B - T) * (dy / 4);  query = grid - flow
      const float fly = dy == 0 ? Ty : Ty + Dy * (0.25f * dy), flx = dy == 0 ? Tx : Tx + Dx * (0.25f * dy);
      const float qy = (Yk + (float)dy) - fly, qx = t.Xf - flx;
      float ty = __fadd_rd(qy, V2_MAGIC), tx = __fadd_rd(qx, V2_MAGIC);        // MAGIC + floor(q), exact for |q| < 2^22
      float ay, ax;
      if (IY) {
        ay = qy - (ty - V2_MAGIC);
      } else {                     // dense_image_warp: floor clamped to [0, size-2], fraction to [0,1]
        const float fy = fminf(fmaxf(ty - V2_MAGIC, 0.f), t.hy);
        ay = __saturatef(qy - fy);
        ty = fy + V2_MAGIC;
      }
      if (IX) {
        ax = qx - (tx - V2_MAGIC);
      } else {
        const float fx = fminf(fmaxf(tx - V2_MAGIC, 0.f), t.hx);
        ax = __saturatef(qx - fx);
        tx = fx + V2_MAGIC;
      }
      // offset = (iy - yo) * pitch + (ix - xo) * 3 with iy, ix still carrying the 1.5 * 2^23 exponent bits (mod 2^32)
      const float* p00 = base + (int)((unsigned)__float_as_int(ty) * (unsigned)t.pitch + (unsigned)__float_as_int(tx) * 3u + t.cbase);
      const float* p10 = p00 + t.pitch;
      unsigned short o[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float tl = p00[c], tr = p00[3 + c], bl = p10[c], br = p10[3 + c];
        const float top = ax * (tr - tl) + tl;
        const float bot = ax * (br - bl) + bl;
        const float v = (ay * (bot - top) + top) * t.in_scale + t.in_shift;
        o[c] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
      }
      // space-to-depth: element (dy*4 + dx)*3 + c of the 48 channels of LR pixel (ly, lx)
      unsigned short* d = reinterpret_cast<unsigned short*>(srow + k * (V2_TLW * 96) + dy * 24);
      d[0] = o[0];
      d[1] = o[1];
      d[2] = o[2];
    }
  }
}

__device__ __forceinline__ void v2_set_base(V2Thread& t, bool staged, const V2Window& v, int W) {
  t.pitch = staged ? v.rowf : W * 3;
  t.cbase = 0u - ((unsigned)(V2_MAGIC_BITS + (staged ? v.y_lo : 0)) * (unsigned)t.pitch +
                  (unsigned)(V2_MAGIC_BITS + (staged ? v.x_lo : 0)) * 3u);
}

__global__ void __launch_bounds__(V2_TPB, 4)
warp_s2d_v2_kernel(const float* __restrict__ pre_gen, const float* __restrict__ flow_lr, __nv_bfloat16* __restrict__ dst,
                   int h, int w, int fh, int fw, int dst_cpitch, int ch_off, float in_scale, float in_shift) {
  extern __shared__ __align__(16) unsigned char v2_smem[];
  float* win = reinterpret_cast<float*>(v2_smem);
  unsigned char* stage = v2_smem + V2_WIN_FLOATS * sizeof(float);
  V2Smem& S = *reinterpret_cast<V2Smem*>(stage + V2_STAGE_BYTES);
  const int H = 4 * h, W = 4 * w;
  const int n = blockIdx.z, ly0 = blockIdx.y * V2_TLH, lx0 = blockIdx.x * V2_TLW;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float* img = pre_gen + (size_t)n * H * W * 3;
  const int Y0 = 4 * ly0, X0 = 4 * lx0;
  const uint32_t bar = tcptx::smem_u32(&S.bar);

  // ---- (1) the 5 x 33 flow samples of the tile -> shared memory
  if (tid == 0) {
    tcptx::mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < V2_NSAMP) {
    const float* fb = flow_lr + (size_t)n * fh * fw * 2;
    const int r = tid / (V2_TLW + 1), j = tid - r * (V2_TLW + 1);
    const int i = min(ly0 + r, h - 1), jj = min(lx0 + j, w - 1);              // upscale_four replicates the last row / column
    const int si = i < fh ? i : 2 * fh - 1 - i, sj = jj < fw ? jj : 2 * fw - 1 - jj;   // tf.pad SYMMETRIC, main.py:212
    float2 f = *reinterpret_cast<const float2*>(fb + (si * fw + sj) * 2);
    f.x *= 4.f;
    f.y *= 4.f;
    S.flow[tid] = f;
  }
  __syncthreads();

  // ---- (2) warp 0: bounds of the flow over the tile -> window -> bulk copies in flight.  The other warps go on to (3).
  if (wid == 0) {
    int kmin_y = 0x7fffffff, kmax_y = (int)0x80000000, kmin_x = 0x7fffffff, kmax_x = (int)0x80000000;
#pragma unroll
    for (int s = 0; s < (V2_NSAMP + 31) / 32; ++s) {
      const float2 f = S.flow[min(lane + 32 * s, V2_NSAMP - 1)];
      const int ky = f2key(f.x), kx = f2key(f.y);
      kmin_y = min(kmin_y, ky);
      kmax_y = max(kmax_y, ky);
      kmin_x = min(kmin_x, kx);
      kmax_x = max(kmax_x, kx);
    }
    const float mny = key2f(__reduce_min_sync(0xffffffffu, kmin_y)), mxy = key2f(__reduce_max_sync(0xffffffffu, kmax_y));
    const float mnx = key2f(__reduce_min_sync(0xffffffffu, kmin_x)), mxx = key2f(__reduce_max_sync(0xffffffffu, kmax_x));
    const V2Window v = v2_window(mny, mxy, mnx, mxx, Y0, 4 * V2_TLH, X0, H, W);
    if (lane == 0) {
      S.mm[0] = mny; S.mm[1] = mxy; S.mm[2] = mnx; S.mm[3] = mxx;
      S.win[0] = v.y_lo; S.win[1] = v.x_lo; S.win[2] = v.rows; S.win[3] = v.rowf; S.win[4] = v.flags;
    }
    if (v.flags & 1) v2_stage(img, W, v, win, bar, lane);
  }

  // ---- (3) this thread: HR column X = X0 + xl of LR rows ly0 + 2 rh, + 1.  flow = upscale_four(4 flow_lr) written as
  // T + (B - T) * (dy / 4) per component with T / B the x-interpolated samples of the LR rows above / below.
  const int xl = tid & (4 * V2_TLW - 1), rh = tid >> 7;
  const int lxl = xl >> 2, dx = xl & 3;
  const float wx1 = 0.25f * (float)dx, wx0 = 1.f - wx1;
  V2Thread t;
  t.hy = (float)(H - 2);
  t.hx = (float)(W - 2);
  t.Xf = (float)(X0 + xl);
  t.in_scale = in_scale;
  t.in_shift = in_shift;
  float Fy[3], Fx[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float2 a = S.flow[(2 * rh + r) * (V2_TLW + 1) + lxl], b = S.flow[(2 * rh + r) * (V2_TLW + 1) + lxl + 1];
    Fy[r] = a.x * wx0 + b.x * wx1;
    Fx[r] = a.y * wx0 + b.y * wx1;
  }
  unsigned char* scol = stage + lxl * 96 + dx * 6;          // this thread's column slot in LR row 0 of the staging tile
  __syncthreads();
  V2Window v;
  v.y_lo = S.win[0]; v.x_lo = S.win[1]; v.rows = S.win[2]; v.rowf = S.win[3]; v.flags = S.win[4];

  if (v.flags & 1) {
    // the window fits: 8 pixels per thread straight from shared memory
    v2_set_base(t, true, v, W);
    const float Yf = (float)(Y0 + 8 * rh);
    unsigned char* srow = scol + (2 * rh) * (V2_TLW * 96);
    tcptx::mbar_wait_warp(bar, 0);
    if ((v.flags & 6) == 6) v2_pixels<true, true, 2>(win, t, Fy, Fx, Yf, srow);
    else if (v.flags & 2) v2_pixels<true, false, 2>(win, t, Fy, Fx, Yf, srow);
    else if (v.flags & 4) v2_pixels<false, true, 2>(win, t, Fy, Fx, Yf, srow);
    else v2_pixels<false, false, 2>(win, t, Fy, Fx, Yf, srow);
  } else {
    // rough flow: the tile in two halves of 2 LR rows (thread = HR column x ONE LR row per half), each with its own smaller
    // window; a half whose window still does not fit gathers from global memory through L1
    const float mny = S.mm[0], mxy = S.mm[1], mnx = S.mm[2], mxx = S.mm[3];
    uint32_t phase = 0;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const V2Window hv = v2_window(mny, mxy, mnx, mxx, Y0 + 8 * half, 8, X0, H, W);
      const bool staged = hv.flags & 1;
      if (staged) {
        __syncthreads();                                   // every reader of the previous half's window is done
        if (wid == 0) {
          tcptx::fence_async_smem();
          v2_stage(img, W, hv, win, bar, lane);
        }
      }
      const int lr = 2 * half + rh;                        // this thread's LR row of the tile
      float Gy[2], Gx[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float2 a = S.flow[(lr + r) * (V2_TLW + 1) + lxl], b = S.flow[(lr + r) * (V2_TLW + 1) + lxl + 1];
        Gy[r] = a.x * wx0 + b.x * wx1;
        Gx[r] = a.y * wx0 + b.y * wx1;
      }
      v2_set_base(t, staged, hv, W);
      if (staged) {
        tcptx::mbar_wait_warp(bar, phase);
        phase ^= 1;
      }
      v2_pixels<false, false, 1>(staged ? win : img, t, Gy, Gx, (float)(Y0 + 4 * lr), scol + lr * (V2_TLW * 96));
    }
  }
  __syncthreads();

  // ---- (4) staged tile -> destination: 96 contiguous bytes per LR pixel as six 16-byte stores
  unsigned char* dtile = reinterpret_cast<unsigned char*>(dst) + 2 * ((((size_t)n * h + ly0) * w + lx0) * dst_cpitch + ch_off);
  const int rpitch = w * dst_cpitch * 2, ppitch = dst_cpitch * 2;
#pragma unroll
  for (int it = 0; it < (V2_TLH * V2_TLW * 6) / V2_TPB; ++it) {
    const int q = tid + it * V2_TPB;
    const int p = q / 6, part = q - p * 6;
    const int r = p >> 5, c = p & 31;
    if (ly0 + r < h && lx0 + c < w) {
      const uint4 v4 = *reinterpret_cast<const uint4*>(stage + q * 16);
      *reinterpret_cast<uint4*>(dtile + r * rpitch + c * ppitch + part * 16) = v4;
    }
  }
}


}  // namespace

// Called by teco_warp_s2d_fused (resample.cu) for the layouts this version covers.  Returns false when it does not apply.
bool teco_warp_s2d_v2_applicable(const void* dst, int dst_cpitch, int ch_off, int dst_bf16, const float* warped_out) {
  return dst_bf16 && !warped_out && (ch_off & 7) == 0 && (dst_cpitch & 7) == 0 && ((uintptr_t)dst & 15) == 0;
}

int teco_warp_s2d_v2_launch(const float* pre_gen, const float* flow_lr, void* dst, int N, int h, int w, int fh, int fw,
                            int dst_cpitch, int ch_off, float in_scale, float in_shift, cudaStream_t stream) {
  const size_t smem = V2_WIN_FLOATS * sizeof(float) + V2_STAGE_BYTES + sizeof(V2Smem);
  TECO_CUDA_CALL(cudaFuncSetAttribute(warp_s2d_v2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles_x = teco_ceil_div(w, V2_TLW), tiles_y = teco_ceil_div(h, V2_TLH);
  TECO_CHECK_ARG(tiles_y <= 65535 && N <= 65535, "teco_warp_s2d_fused: more than 65535 row bands or images");
  warp_s2d_v2_kernel<<<dim3((unsigned)tiles_x, (unsigned)tiles_y, (unsigned)N), V2_TPB, smem, stream>>>(
      pre_gen, flow_lr, (__nv_bfloat16*)dst, h, w, fh, fw, dst_cpitch, ch_off, in_scale, in_shift);
  TECO_CUDA_LAUNCH_CHECK("teco_warp_s2d_fused (v2)");
  return TECO_OK;
}
