// HBM-bound resampling family: dense_image_warp (+gradients), the fused
// upscale_four -> warp -> space-to-depth feedback kernel, upscale_four, bicubic_four, legacy bilinear
// resize, max-pool, space-to-depth, Gaussian down-sampling.  Reference call sites are cited in
// include/teco.h next to each entry point.
#include "teco_common.cuh"
#include <stdlib.h>

namespace {

constexpr int TPB = 256;

inline unsigned grid_for(long long n, int per_block = TPB) {
  long long b = (n + per_block - 1) / per_block;
  long long cap = (long long)teco_sm_count() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

// ---- bilinear sample set-up shared by warp kernels (TF _interpolate_bilinear semantics)
struct Bil {
  int y0, x0;
  float ay, ax;
  bool gy, gx;  // gradient flows to the query coordinate (0 < alpha_raw <= 1)
};

__device__ __forceinline__ Bil bil_setup(float qy, float qx, int H, int W) {
  Bil b;
  float fy = fminf(fmaxf(floorf(qy), 0.f), (float)(H - 2));
  float fx = fminf(fmaxf(floorf(qx), 0.f), (float)(W - 2));
  float ary = qy - fy, arx = qx - fx;
  b.gy = ary > 0.f && ary <= 1.f;
  b.gx = arx > 0.f && arx <= 1.f;
  b.ay = fminf(fmaxf(ary, 0.f), 1.f);
  b.ax = fminf(fmaxf(arx, 0.f), 1.f);
  b.y0 = (int)fy;
  b.x0 = (int)fx;
  return b;
}

__global__ void warp_f32_kernel(const float* __restrict__ img, const float* __restrict__ flow, float* __restrict__ out,
                                int N, int H, int W, int C) {
  long long total = (long long)N * H * W;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int x = (int)(i % W);
    long long t = i / W;
    int y = (int)(t % H);
    int n = (int)(t / H);
    float2 f = *reinterpret_cast<const float2*>(flow + i * 2);
    Bil b = bil_setup((float)y - f.x, (float)x - f.y, H, W);
    const float* p00 = img + (((long long)n * H + b.y0) * W + b.x0) * C;
    const float* p10 = p00 + (long long)W * C;
    for (int c = 0; c < C; ++c) {
      float tl = p00[c], tr = p00[C + c], bl = p10[c], br = p10[C + c];
      float top = b.ax * (tr - tl) + tl;
      float bot = b.ax * (br - bl) + bl;
      out[i * C + c] = b.ay * (bot - top) + top;
    }
  }
}

__global__ void warp_bwd_f32_kernel(const float* __restrict__ img, const float* __restrict__ flow,
                                    const float* __restrict__ dout, float* __restrict__ dimg, float* __restrict__ dflow,
                                    int N, int H, int W, int C) {
  long long total = (long long)N * H * W;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int x = (int)(i % W);
    long long t = i / W;
    int y = (int)(t % H);
    int n = (int)(t / H);
    float2 f = *reinterpret_cast<const float2*>(flow + i * 2);
    Bil b = bil_setup((float)y - f.x, (float)x - f.y, H, W);
    long long o00 = (((long long)n * H + b.y0) * W + b.x0) * C;
    long long o10 = o00 + (long long)W * C;
    float gqy = 0.f, gqx = 0.f;
    for (int c = 0; c < C; ++c) {
      float g = dout[i * C + c];
      float tl = img[o00 + c], tr = img[o00 + C + c], bl = img[o10 + c], br = img[o10 + C + c];
      float top = b.ax * (tr - tl) + tl;
      float bot = b.ax * (br - bl) + bl;
      gqy += g * (bot - top);
      gqx += g * ((1.f - b.ay) * (tr - tl) + b.ay * (br - bl));
      if (dimg) {
        atomicAdd(&dimg[o00 + c], g * (1.f - b.ay) * (1.f - b.ax));
        atomicAdd(&dimg[o00 + C + c], g * (1.f - b.ay) * b.ax);
        atomicAdd(&dimg[o10 + c], g * b.ay * (1.f - b.ax));
        atomicAdd(&dimg[o10 + C + c], g * b.ay * b.ax);
      }
    }
    if (dflow) {
      // query = grid - flow  =>  d/dflow = -d/dquery
      dflow[i * 2 + 0] = b.gy ? -gqy : 0.f;
      dflow[i * 2 + 1] = b.gx ? -gqx : 0.f;
    }
  }
}

// ---- fused feedback: flow_lr -> (symmetric pad, x4, upscale_four) -> warp(pre_gen) -> s2d into dst.
// CTA tile = 2 LR rows x 32 LR columns (8 x 128 HR pixels); one thread per (LR pixel, dy): 4 HR pixels x 3 channels
// = 12 contiguous destination values.  The HR flow inside the tile is a convex combination of the 3 x 33 LR flow
// samples around it, so their min/max bound every query of the tile: the CTA stages that source window of the
// previous HR frame in shared memory with fully coalesced loads and gathers from there (round-1 ncu: the direct
// per-thread gather moved 30 sectors per request through L1, 31x the unique bytes).  Windows that do not fit
// (|flow| spread > ~40 px inside one tile) take the direct global gather path.
constexpr int WS_TLH = 2, WS_TLW = 32;                 // LR tile
constexpr int WS_SMEM_FLOATS = 8 * 1024;               // 32 KB window budget: up to ~16 x 168 source pixels, 7 CTAs / SM

struct FlowQ { float2 f00, f01, f10, f11; };

__device__ __forceinline__ FlowQ load_flow_quad(const float* __restrict__ fb, int ly, int lx, int h, int w, int fh, int fw) {
  // flow_lr neighbours (upscale_four pads bottom/right by replication AFTER the symmetric pad of main.py:212)
  int i0 = ly, i1 = min(ly + 1, h - 1), j0 = lx, j1 = min(lx + 1, w - 1);
  int si0 = i0 < fh ? i0 : 2 * fh - 1 - i0, si1 = i1 < fh ? i1 : 2 * fh - 1 - i1;
  int sj0 = j0 < fw ? j0 : 2 * fw - 1 - j0, sj1 = j1 < fw ? j1 : 2 * fw - 1 - j1;
  FlowQ q;
  q.f00 = *reinterpret_cast<const float2*>(fb + ((long long)si0 * fw + sj0) * 2);
  q.f01 = *reinterpret_cast<const float2*>(fb + ((long long)si0 * fw + sj1) * 2);
  q.f10 = *reinterpret_cast<const float2*>(fb + ((long long)si1 * fw + sj0) * 2);
  q.f11 = *reinterpret_cast<const float2*>(fb + ((long long)si1 * fw + sj1) * 2);
  q.f00.x *= 4.f; q.f00.y *= 4.f; q.f01.x *= 4.f; q.f01.y *= 4.f;
  q.f10.x *= 4.f; q.f10.y *= 4.f; q.f11.x *= 4.f; q.f11.y *= 4.f;
  return q;
}

// One tile per CTA (grid = tiles_x x tiles_y x N: no index divisions), five CTAs per SM.  Phases: (1) the first four warps
// bound the flow over the tile, (2) all threads issue 16-byte cp.async copies of the source window, (3) WHILE those are in
// flight every thread interpolates its own flow and sets up its four bilinear queries, (4) gather + blend from the window.
// Round-2 ncu of the first versions: 227 thread instructions per HR pixel at IPC 2.2 -- the kernel was instruction- and
// latency-bound, not memory-bound: generic loads through a run-time selected pointer, 64-bit index arithmetic and integer
// divisions.  This version keeps each address space in its own code path and all per-pixel index arithmetic in 32 bits.
template <bool kBf16>
__global__ void __launch_bounds__(TPB, 5)
warp_s2d_fused_kernel(const float* __restrict__ pre_gen, const float* __restrict__ flow_lr, void* __restrict__ dst,
                      float* __restrict__ warped_out, int N, int h, int w, int fh, int fw, int dst_cpitch, int ch_off,
                      float in_scale, float in_shift) {
  extern __shared__ __align__(16) float win[];
  __shared__ float red[4][4];
  __shared__ int s_win[6];   // y_lo, x_lo, rows, cols, use_smem, interior (no query of the tile can touch a clamp)
  const int H = 4 * h, W = 4 * w;
  const int n = blockIdx.z, ly0 = blockIdx.y * WS_TLH, lx0 = blockIdx.x * WS_TLW;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float* fb = flow_lr + (size_t)n * fh * fw * 2;
  const float* img = pre_gen + (size_t)n * H * W * 3;

  // ---- (1) bound the flow over the tile: samples (ly0..ly0+2) x (lx0..lx0+32), clamped like upscale_four
  if (wid < 4) {
    float mny = 1e30f, mxy = -1e30f, mnx = 1e30f, mxx = -1e30f;
    if (tid < (WS_TLH + 1) * (WS_TLW + 1)) {
      const int r = tid >= 2 * (WS_TLW + 1) ? 2 : (tid >= (WS_TLW + 1) ? 1 : 0);
      const int i = min(ly0 + r, h - 1), j = min(lx0 + tid - r * (WS_TLW + 1), w - 1);
      const int si = i < fh ? i : 2 * fh - 1 - i, sj = j < fw ? j : 2 * fw - 1 - j;
      const float2 f = *reinterpret_cast<const float2*>(fb + (si * fw + sj) * 2);
      mny = mxy = f.x * 4.f;
      mnx = mxx = f.y * 4.f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
      mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
      mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
      mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    }
    if (lane == 0) { red[0][wid] = mny; red[1][wid] = mxy; red[2][wid] = mnx; red[3][wid] = mxx; }
  }
  __syncthreads();
  if (tid == 0) {
    float mny = red[0][0], mxy = red[1][0], mnx = red[2][0], mxx = red[3][0];
    for (int k = 1; k < 4; ++k) {
      mny = fminf(mny, red[0][k]); mxy = fmaxf(mxy, red[1][k]);
      mnx = fminf(mnx, red[2][k]); mxx = fmaxf(mxx, red[3][k]);
    }
    const int Y0 = 4 * ly0, X0 = 4 * lx0;
    // queries: Y - fy in [Y0 - mxy, Y0 + 7 - mny]; floor clamped to [0, H-2], plus the +1 neighbour row
    int y_lo = (int)fminf(fmaxf(floorf((float)Y0 - mxy) - 1.f, 0.f), (float)(H - 2));
    int y_hi = (int)fminf(fmaxf(floorf((float)(Y0 + 4 * WS_TLH - 1) - mny) + 1.f, 0.f), (float)(H - 2)) + 1;
    int x_lo = (int)fminf(fmaxf(floorf((float)X0 - mxx) - 1.f, 0.f), (float)(W - 2));
    int x_hi = (int)fminf(fmaxf(floorf((float)(X0 + 4 * WS_TLW - 1) - mnx) + 1.f, 0.f), (float)(W - 2)) + 1;
    // columns in whole groups of four pixels (48 bytes): every window row then starts and ends on a 16-byte boundary of
    // the fp32 RGB image (W = 4w is a multiple of 4), so the window can be fetched with 16-byte asynchronous copies
    x_lo &= ~3;
    x_hi = min(x_hi | 3, W - 1);
    const int rows = y_hi - y_lo + 1, cols = x_hi - x_lo + 1;
    s_win[0] = y_lo; s_win[1] = x_lo; s_win[2] = rows; s_win[3] = cols;
    // stage only when the window is compact (<= 2.5x the tile's own 8x128 pixels): rough flow fields would re-read more
    // through the window than the direct L1 gather does
    s_win[4] = (rows * cols * 3 <= WS_SMEM_FLOATS && rows * cols * 2 <= 5 * (4 * WS_TLH) * (4 * WS_TLW)) ? 1 : 0;
    // every query of the tile lies at least one pixel inside [0, size-2]: floor needs no clamp and the fraction is in [0,1)
    s_win[5] = ((float)Y0 - mxy >= 1.f && (float)(Y0 + 4 * WS_TLH - 1) - mny <= (float)(H - 3) &&
                (float)X0 - mxx >= 1.f && (float)(X0 + 4 * WS_TLW - 1) - mnx <= (float)(W - 3)) ? 1 : 0;
  }
  __syncthreads();
  const int y_lo = s_win[0], x_lo = s_win[1], rowf = s_win[3] * 3;
  const bool use_smem = s_win[4] != 0, interior = s_win[5] != 0;

  // ---- (2) the whole window in flight at once: 16-byte cp.async copies (no register staging); a warp per window row
  if (use_smem) {
    const int rows = s_win[2], cpr = rowf >> 2;       // 16-byte chunks per window row (rowf is a multiple of 12 floats)
    const float* src0 = img + ((size_t)y_lo * W + x_lo) * 3;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(win);
    for (int r = wid; r < rows; r += TPB / 32) {
      const float* src = src0 + (size_t)r * (W * 3);
      const uint32_t drow = sbase + (uint32_t)(r * rowf) * 4u;
      for (int k = lane; k < cpr; k += 32)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(drow + 16u * k), "l"(src + 4 * k) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }

  // ---- (3) this thread's four queries: HR column X = 4 lx + dx of the four HR sub-rows dy of one LR row.  A warp covers 32
  // consecutive HR columns, so its window reads step by 3 floats from lane to lane (conflict-free; the (LR pixel, dy) mapping
  // of round 1 hit 8 of 32 banks).  flow = upscale_four(4 * flow_lr) written as T + (B - T) * (dy/4) per component.
  // floor / float->int by the 1.5*2^23 trick on the FMA pipe: ncu showed the XU pipe (FRND, F2I, I2F) 95 % busy.
  const int xl = tid & (4 * WS_TLW - 1), lyl = tid >> 7;
  const int dx = xl & 3, lx = lx0 + (xl >> 2), ly = ly0 + lyl;
  const bool valid = ly < h && lx < w;
  int off[4];
  float ax[4], ay[4];
  {
    const int lyc = min(ly, h - 1), lxc = min(lx, w - 1);
    const FlowQ q = load_flow_quad(fb, lyc, lxc, h, w, fh, fw);
    const float wx1 = 0.25f * dx, wx0 = 1.f - wx1;
    const float Ty = q.f00.x * wx0 + q.f01.x * wx1, Dy = (q.f10.x * wx0 + q.f11.x * wx1) - Ty;
    const float Tx = q.f00.y * wx0 + q.f01.y * wx1, Dx = (q.f10.y * wx0 + q.f11.y * wx1) - Tx;
    const float Yf = (float)(4 * lyc), Xf = (float)(4 * lxc + dx);
    const int pitch = use_smem ? rowf : W * 3;
    const int yo = use_smem ? y_lo : 0, xo = use_smem ? x_lo : 0;
    const float hy = (float)(H - 2), hx = (float)(W - 2);
    auto floor_fi = [](float v, float& f, int& i) {   // floor for |v| < 2^22 without FRND / F2I
      const float t = v + 12582912.f;                 // 1.5 * 2^23: round to nearest integer
      f = t - 12582912.f;
      i = __float_as_int(t) - 0x4B400000;
      if (f > v) { f -= 1.f; i -= 1; }
    };
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      const float qy = (Yf + (float)dy) - (Ty + Dy * (0.25f * dy)), qx = Xf - (Tx + Dx * (0.25f * dy));
      float fy, fx;
      int iy, ix;
      floor_fi(qy, fy, iy);
      floor_fi(qx, fx, ix);
      if (interior) {                                 // CTA-uniform: 14 instructions per pixel less on all but border tiles
        ay[dy] = qy - fy;
        ax[dy] = qx - fx;
      } else {
        fy = fminf(fmaxf(fy, 0.f), hy);               // dense_image_warp: floor clamped to [0, size-2], fraction to [0,1]
        fx = fminf(fmaxf(fx, 0.f), hx);
        iy = min(max(iy, 0), H - 2);
        ix = min(max(ix, 0), W - 2);
        ay[dy] = fminf(fmaxf(qy - fy, 0.f), 1.f);
        ax[dy] = fminf(fmaxf(qx - fx, 0.f), 1.f);
      }
      off[dy] = (iy - yo) * pitch + (ix - xo) * 3;
    }
  }
  if (use_smem) asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  // ---- (4) gather + blend; each address space in its own code path
  float vals[4][3];
  auto gather = [&](const float* __restrict__ base, int pitch) {
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      const float* p00 = base + off[dy];
      const float* p10 = p00 + pitch;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float tl = p00[c], tr = p00[3 + c], bl = p10[c], br = p10[3 + c];
        const float top = ax[dy] * (tr - tl) + tl;
        const float bot = ax[dy] * (br - bl) + bl;
        vals[dy][c] = ay[dy] * (bot - top) + top;
      }
    }
  };
  if (use_smem) gather(win, rowf);
  else gather(img, W * 3);

  if (warped_out && valid) {
    float* wo = warped_out + (((size_t)n * H + 4 * ly) * W + 4 * lx + dx) * 3;
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      wo[(size_t)dy * W * 3 + 0] = vals[dy][0];
      wo[(size_t)dy * W * 3 + 1] = vals[dy][1];
      wo[(size_t)dy * W * 3 + 2] = vals[dy][2];
    }
  }
  // space-to-depth: element (dy*4 + dx)*3 + c of the 48 channels of LR pixel (ly, lx)
  const size_t o = (((size_t)n * h + min(ly, h - 1)) * w + min(lx, w - 1)) * dst_cpitch + ch_off;
  if (kBf16) {
    __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(dst) + o;
    const bool vec = ((o & 3) == 0);                 // warp-uniform per LR row except through lx; all lanes shuffle anyway
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      const float v0 = vals[dy][0] * in_scale + in_shift, v1 = vals[dy][1] * in_scale + in_shift, v2 = vals[dy][2] * in_scale + in_shift;
      // the 12 values of (LR pixel, dy) sit in four neighbouring lanes (dx = 0..3): lanes dx = 0,1,2 each write 8 bytes
      const float n0 = __shfl_down_sync(0xffffffffu, v0, 1), n1 = __shfl_down_sync(0xffffffffu, v1, 1),
                  n2 = __shfl_down_sync(0xffffffffu, v2, 1);
      if (!valid) continue;
      if (vec) {
        if (dx < 3) {
          const float e0 = dx == 0 ? v0 : (dx == 1 ? v1 : v2), e1 = dx == 0 ? v1 : (dx == 1 ? v2 : n0),
                      e2 = dx == 0 ? v2 : (dx == 1 ? n0 : n1), e3 = dx == 0 ? n0 : (dx == 1 ? n1 : n2);
          __nv_bfloat162 a = __floats2bfloat162_rn(e0, e1), c = __floats2bfloat162_rn(e2, e3);
          uint2 u;
          u.x = *reinterpret_cast<uint32_t*>(&a);
          u.y = *reinterpret_cast<uint32_t*>(&c);
          *reinterpret_cast<uint2*>(d + dy * 12 + dx * 4) = u;
        }
      } else {
        d[dy * 12 + dx * 3 + 0] = __float2bfloat16_rn(v0);
        d[dy * 12 + dx * 3 + 1] = __float2bfloat16_rn(v1);
        d[dy * 12 + dx * 3 + 2] = __float2bfloat16_rn(v2);
      }
    }
  } else if (valid) {
    float* d = reinterpret_cast<float*>(dst) + o;
#pragma unroll
    for (int dy = 0; dy < 4; ++dy) {
      d[dy * 12 + dx * 3 + 0] = vals[dy][0] * in_scale + in_shift;
      d[dy * 12 + dx * 3 + 1] = vals[dy][1] * in_scale + in_shift;
      d[dy * 12 + dx * 3 + 2] = vals[dy][2] * in_scale + in_shift;
    }
  }
}

__global__ void upscale4_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int h, int w, int C,
                                    float scale) {
  long long total = (long long)N * h * 4 * w * 4 * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % (4 * w));
    t /= (4 * w);
    int Y = (int)(t % (4 * h));
    int n = (int)(t / (4 * h));
    int ly = Y >> 2, dy = Y & 3, lx = X >> 2, dx = X & 3;
    int i1 = min(ly + 1, h - 1), j1 = min(lx + 1, w - 1);
    const float* b = x + (long long)n * h * w * C;
    float tl = b[((long long)ly * w + lx) * C + c] * scale, tr = b[((long long)ly * w + j1) * C + c] * scale;
    float bl = b[((long long)i1 * w + lx) * C + c] * scale, br = b[((long long)i1 * w + j1) * C + c] * scale;
    float wy1 = 0.25f * dy, wy0 = 1.f - wy1, wx1 = 0.25f * dx, wx0 = 1.f - wx1;
    y[i] = tl * wy0 * wx0 + tr * wy0 * wx1 + bl * wy1 * wx0 + br * wy1 * wx1;
  }
}

// Keys bicubic weights, A = -0.75, t in {0,.25,.5,.75}: [1,t,t2,t3] . M  (reference lib/ops.py:186-188)
__device__ __forceinline__ void bicubic_w(int k, float* wt) {
  const float r = 0.75f;
  float t = 0.25f * k, t2 = t * t, t3 = t2 * t;
  wt[0] = -r * t + 2.f * r * t2 - r * t3;
  wt[1] = 1.f + (r - 3.f) * t2 + (2.f - r) * t3;
  wt[2] = r * t + (3.f - 2.f * r) * t2 + (r - 2.f) * t3;
  wt[3] = -r * t2 + r * t3;
}

__global__ void bicubic4_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int h, int w, int C,
                                    int in_cpitch) {
  long long total = (long long)N * h * 4 * w * 4 * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % (4 * w));
    t /= (4 * w);
    int Y = (int)(t % (4 * h));
    int n = (int)(t / (4 * h));
    int ly = Y >> 2, lx = X >> 2;
    float wy[4], wx[4];
    bicubic_w(Y & 3, wy);
    bicubic_w(X & 3, wx);
    const float* b = x + (long long)n * h * w * in_cpitch + c;
    float acc = 0.f;
    // rows first (vertical), then columns -- same association order as the reference
#pragma unroll
    for (int bj = 0; bj < 4; ++bj) {
      int xx = min(max(lx - 1 + bj, 0), w - 1);
      float col = 0.f;
#pragma unroll
      for (int bi = 0; bi < 4; ++bi) {
        int yy = min(max(ly - 1 + bi, 0), h - 1);
        col += wy[bi] * b[((long long)yy * w + xx) * in_cpitch];
      }
      acc += wx[bj] * col;
    }
    y[i] = acc;
  }
}

// C == 3 fast path: one thread per (LR pixel, output sub-row): 16 LR pixels in, 4 HR pixels x RGB = 48 contiguous bytes
// out (three float4 stores; a warp writes 1.5 KB contiguous).  Same association order as the generic kernel above
// (vertical taps first, then horizontal), so the results are identical.
__global__ void bicubic4_rgb_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int h, int w, int in_cpitch) {
  const long long total = (long long)N * h * 4 * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int lx = (int)(i % w);
    long long t = i / w;
    const int Y = (int)(t % (4 * h));
    const int n = (int)(t / (4 * h));
    const int ly = Y >> 2;
    float wy[4];
    bicubic_w(Y & 3, wy);
    const float* b = x + (long long)n * h * w * in_cpitch;
    float col[4][3];
#pragma unroll
    for (int bj = 0; bj < 4; ++bj) {
      const int xx = min(max(lx - 1 + bj, 0), w - 1);
      col[bj][0] = col[bj][1] = col[bj][2] = 0.f;
#pragma unroll
      for (int bi = 0; bi < 4; ++bi) {
        const int yy = min(max(ly - 1 + bi, 0), h - 1);
        const float* px = b + ((long long)yy * w + xx) * in_cpitch;
        col[bj][0] += wy[bi] * px[0];
        col[bj][1] += wy[bi] * px[1];
        col[bj][2] += wy[bi] * px[2];
      }
    }
    float o[12];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) {
      float wx[4];
      bicubic_w(dx, wx);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float acc = 0.f;
#pragma unroll
        for (int bj = 0; bj < 4; ++bj) acc += wx[bj] * col[bj][c];
        o[dx * 3 + c] = acc;
      }
    }
    float4* dst = reinterpret_cast<float4*>(y + (((long long)n * 4 * h + Y) * (4 * w) + 4 * lx) * 3);
    dst[0] = make_float4(o[0], o[1], o[2], o[3]);
    dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    dst[2] = make_float4(o[8], o[9], o[10], o[11]);
  }
}

__global__ void resize_bilinear_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int h, int w, int C,
                                           int oh, int ow) {
  long long total = (long long)N * oh * ow * C;
  float sy = (float)h / (float)oh, sx = (float)w / (float)ow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    float fy = Y * sy, fx = X * sx;
    int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
    int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
    float wy = fy - y0, wx = fx - x0;
    const float* b = x + (long long)n * h * w * C + c;
    float tl = b[((long long)y0 * w + x0) * C], tr = b[((long long)y0 * w + x1) * C];
    float bl = b[((long long)y1 * w + x0) * C], br = b[((long long)y1 * w + x1) * C];
    float top = tl + (tr - tl) * wx, bot = bl + (br - bl) * wx;
    y[i] = top + (bot - top) * wy;
  }
}

__global__ void resize_bilinear_bwd_f32_kernel(const float* __restrict__ dy, float* __restrict__ dx, int N, int h, int w,
                                               int C, int oh, int ow) {
  long long total = (long long)N * oh * ow * C;
  float sy = (float)h / (float)oh, sx = (float)w / (float)ow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    float fy = Y * sy, fx = X * sx;
    int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
    int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
    float wy = fy - y0, wx = fx - x0;
    float g = dy[i];
    float* b = dx + (long long)n * h * w * C + c;
    atomicAdd(&b[((long long)y0 * w + x0) * C], g * (1.f - wy) * (1.f - wx));
    atomicAdd(&b[((long long)y0 * w + x1) * C], g * (1.f - wy) * wx);
    atomicAdd(&b[((long long)y1 * w + x0) * C], g * wy * (1.f - wx));
    atomicAdd(&b[((long long)y1 * w + x1) * C], g * wy * wx);
  }
}

__global__ void maxpool2_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C) {
  int oh = H / 2, ow = W / 2;
  long long total = (long long)N * oh * ow * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    const float* b = x + (((long long)n * H + 2 * Y) * W + 2 * X) * C + c;
    y[i] = fmaxf(fmaxf(b[0], b[C]), fmaxf(b[(long long)W * C], b[(long long)W * C + C]));
  }
}

__global__ void maxpool2_bwd_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx,
                                        int N, int H, int W, int C) {
  int oh = H / 2, ow = W / 2;
  long long total = (long long)N * oh * ow * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    long long o = (((long long)n * H + 2 * Y) * W + 2 * X) * C + c;
    long long offs[4] = {0, C, (long long)W * C, (long long)W * C + C};
    int best = 0;
    float bv = x[o];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      float v = x[o + offs[k]];
      if (v > bv) { bv = v; best = k; }
    }
    float g = dy[i];
#pragma unroll
    for (int k = 0; k < 4; ++k) dx[o + offs[k]] = (k == best) ? g : 0.f;
  }
}

// bf16 NHWC, 8 channels (16 B) per thread
__device__ __forceinline__ uint32_t bf2_max(uint32_t a, uint32_t b) {
  __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
__global__ void maxpool2_bf16_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int N, int H, int W, int C8) {
  int oh = H / 2, ow = W / 2;
  long long total = (long long)N * oh * ow * C8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C8);
    long long t = i / C8;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    const uint4* b = x + (((long long)n * H + 2 * Y) * W + 2 * X) * C8 + c;
    uint4 a0 = b[0], a1 = b[C8], a2 = b[(long long)W * C8], a3 = b[(long long)W * C8 + C8], r;
    r.x = bf2_max(bf2_max(a0.x, a1.x), bf2_max(a2.x, a3.x));
    r.y = bf2_max(bf2_max(a0.y, a1.y), bf2_max(a2.y, a3.y));
    r.z = bf2_max(bf2_max(a0.z, a1.z), bf2_max(a2.z, a3.z));
    r.w = bf2_max(bf2_max(a0.w, a1.w), bf2_max(a2.w, a3.w));
    y[i] = r;
  }
}
__device__ __forceinline__ uint32_t bf2_avg(uint32_t a, uint32_t b) {
  float2 fa = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&a));
  float2 fb = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&b));
  __nv_bfloat162 r = __floats2bfloat162_rn(0.5f * (fa.x + fb.x), 0.5f * (fa.y + fb.y));
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ uint4 bf8_avg(uint4 a, uint4 b) {
  return make_uint4(bf2_avg(a.x, b.x), bf2_avg(a.y, b.y), bf2_avg(a.z, b.z), bf2_avg(a.w, b.w));
}
// legacy bilinear x2: out[2i]=x[i], out[2i+1]=(x[i]+x[min(i+1,n-1)])/2, separable
__global__ void resize2x_bf16_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int N, int h, int w, int C8) {
  int oh = 2 * h, ow = 2 * w;
  long long total = (long long)N * oh * ow * C8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C8);
    long long t = i / C8;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    int y0 = Y >> 1, x0 = X >> 1;
    int y1 = (Y & 1) ? min(y0 + 1, h - 1) : y0, x1 = (X & 1) ? min(x0 + 1, w - 1) : x0;
    const uint4* b = x + (long long)n * h * w * C8 + c;
    // fp32 math per pair, identical association to the fp32 kernel: top/bot lerp in x, then y
    uint4 tl = b[((long long)y0 * w + x0) * C8], tr = b[((long long)y0 * w + x1) * C8];
    uint4 bl = b[((long long)y1 * w + x0) * C8], br = b[((long long)y1 * w + x1) * C8];
    auto lerp4 = [&](uint32_t a00, uint32_t a01, uint32_t a10, uint32_t a11) {
      float2 f00 = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&a00));
      float2 f01 = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&a01));
      float2 f10 = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&a10));
      float2 f11 = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&a11));
      float wx = (X & 1) ? 0.5f : 0.f, wy = (Y & 1) ? 0.5f : 0.f;
      float tx = f00.x + (f01.x - f00.x) * wx, bx = f10.x + (f11.x - f10.x) * wx;
      float ty = f00.y + (f01.y - f00.y) * wx, by = f10.y + (f11.y - f10.y) * wx;
      __nv_bfloat162 r = __floats2bfloat162_rn(tx + (bx - tx) * wy, ty + (by - ty) * wy);
      return *reinterpret_cast<uint32_t*>(&r);
    };
    uint4 r;
    r.x = lerp4(tl.x, tr.x, bl.x, br.x);
    r.y = lerp4(tl.y, tr.y, bl.y, br.y);
    r.z = lerp4(tl.z, tr.z, bl.z, br.z);
    r.w = lerp4(tl.w, tr.w, bl.w, br.w);
    y[i] = r;
  }
}

__global__ void s2d4_f32_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int h, int w, int C,
                                int out_cpitch, int ch_off, bool inverse) {
  long long total = (long long)N * h * 4 * w * 4 * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % (4 * w));
    t /= (4 * w);
    int Y = (int)(t % (4 * h));
    int n = (int)(t / (4 * h));
    long long o = (((long long)n * h + (Y >> 2)) * w + (X >> 2)) * out_cpitch + ch_off + ((Y & 3) * 4 + (X & 3)) * C + c;
    if (!inverse) y[o] = x[i];
    else const_cast<float*>(x)[i] = y[o];
  }
}

__constant__ float c_gauss9[9];  // normalised 1-D factor; the 2-D kernel of the reference is its outer product

__global__ void gauss_down4_f32_kernel(const float* __restrict__ hr, float* __restrict__ lr, int N, int H, int W, int C) {
  int oh = (H - 9) / 4 + 1, ow = (W - 9) / 4 + 1;
  long long total = (long long)N * oh * ow * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % C);
    long long t = i / C;
    int X = (int)(t % ow);
    t /= ow;
    int Y = (int)(t % oh);
    int n = (int)(t / oh);
    const float* b = hr + (((long long)n * H + 4 * Y) * W + 4 * X) * C + c;
    float acc = 0.f;
#pragma unroll
    for (int ky = 0; ky < 9; ++ky) {
      float row = 0.f;
#pragma unroll
      for (int kx = 0; kx < 9; ++kx) row += c_gauss9[kx] * b[((long long)ky * W + kx) * C];
      acc += c_gauss9[ky] * row;
    }
    lr[i] = acc;
  }
}

}  // namespace

#define LAUNCH1D(kernel, total, ...)                                                          \
  kernel<<<grid_for(total), TPB, 0, (cudaStream_t)stream>>>(__VA_ARGS__);                     \
  TECO_CUDA_LAUNCH_CHECK(#kernel)

extern "C" {

int teco_warp_f32(const float* img, const float* flow, float* out, int32_t N, int32_t H, int32_t W, int32_t C,
                  void* stream) {
  TECO_CHECK_ARG(img && flow && out, "teco_warp_f32: NULL tensor");
  TECO_CHECK_ARG(N > 0 && H >= 2 && W >= 2 && C > 0, "teco_warp_f32: need H,W >= 2 (got N=%d H=%d W=%d C=%d)", N, H, W, C);
  LAUNCH1D(warp_f32_kernel, (long long)N * H * W, img, flow, out, N, H, W, C);
  return TECO_OK;
}

int teco_warp_bwd_f32(const float* img, const float* flow, const float* dout, float* dimg, float* dflow, int32_t N,
                      int32_t H, int32_t W, int32_t C, void* stream) {
  TECO_CHECK_ARG(img && flow && dout, "teco_warp_bwd_f32: NULL tensor");
  TECO_CHECK_ARG(N > 0 && H >= 2 && W >= 2 && C > 0, "teco_warp_bwd_f32: bad shape");
  LAUNCH1D(warp_bwd_f32_kernel, (long long)N * H * W, img, flow, dout, dimg, dflow, N, H, W, C);
  return TECO_OK;
}

}  // extern "C"
// warp_s2d_v2.cu: the low-instruction-count version for the inference layout (bf16 destination, aligned channel offset)
bool teco_warp_s2d_v2_applicable(const void* dst, int dst_cpitch, int ch_off, int dst_bf16, const float* warped_out);
int teco_warp_s2d_v2_launch(const float* pre_gen, const float* flow_lr, void* dst, int N, int h, int w, int fh, int fw,
                            int dst_cpitch, int ch_off, float in_scale, float in_shift, cudaStream_t stream);
extern "C" {

int teco_warp_s2d_fused(const float* pre_gen, const float* flow_lr, void* dst, float* warped_out, int32_t N, int32_t h,
                        int32_t w, int32_t fh, int32_t fw, int32_t dst_cpitch, int32_t ch_off, int32_t dst_bf16,
                        float in_scale, float in_shift, void* stream) {
  TECO_CHECK_ARG(pre_gen && flow_lr && dst, "teco_warp_s2d_fused: NULL tensor");
  TECO_CHECK_ARG(N > 0 && h > 0 && w > 0 && fh > 0 && fw > 0 && fh <= h && fw <= w && h - fh <= fh && w - fw <= fw,
                 "teco_warp_s2d_fused: bad shape h=%d w=%d fh=%d fw=%d", h, w, fh, fw);
  TECO_CHECK_ARG(ch_off >= 0 && ch_off + 48 <= dst_cpitch, "teco_warp_s2d_fused: 48 channels do not fit at ch_off=%d in pitch %d",
                 ch_off, dst_cpitch);
  TECO_CHECK_ARG((((uintptr_t)pre_gen) & 15) == 0, "teco_warp_s2d_fused: pre_gen must be 16-byte aligned");
  const char* v2_env = getenv("TECO_WARP_V2");                 // A/B switch, read per call: "0" selects the first version
  if ((!v2_env || v2_env[0] != '0') && teco_warp_s2d_v2_applicable(dst, dst_cpitch, ch_off, dst_bf16, warped_out))
    return teco_warp_s2d_v2_launch(pre_gen, flow_lr, dst, N, h, w, fh, fw, dst_cpitch, ch_off, in_scale, in_shift,
                                   (cudaStream_t)stream);
  const int tiles_x = teco_ceil_div(w, WS_TLW), tiles_y = teco_ceil_div(h, WS_TLH);
  TECO_CHECK_ARG(tiles_y <= 65535 && N <= 65535, "teco_warp_s2d_fused: more than 65535 row bands or images");
  const size_t smem = WS_SMEM_FLOATS * sizeof(float);
  if (dst_bf16) TECO_CUDA_CALL(cudaFuncSetAttribute(warp_s2d_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  else TECO_CUDA_CALL(cudaFuncSetAttribute(warp_s2d_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // the 4-float stores of warped_out need 16-byte alignment of every (row, 4*lx) start: W*3 floats per row, 4*lx*3 = 12 lx
  TECO_CHECK_ARG(!warped_out || ((((uintptr_t)warped_out) & 15) == 0), "teco_warp_s2d_fused: warped_out must be 16-byte aligned");
  TECO_CHECK_ARG((((uintptr_t)pre_gen) & 15) == 0, "teco_warp_s2d_fused: pre_gen must be 16-byte aligned");
  const dim3 grid((unsigned)tiles_x, (unsigned)tiles_y, (unsigned)N);
  if (dst_bf16)
    warp_s2d_fused_kernel<true><<<grid, TPB, smem, (cudaStream_t)stream>>>(pre_gen, flow_lr, dst, warped_out, N, h, w, fh, fw, dst_cpitch,
                                                                          ch_off, in_scale, in_shift);
  else
    warp_s2d_fused_kernel<false><<<grid, TPB, smem, (cudaStream_t)stream>>>(pre_gen, flow_lr, dst, warped_out, N, h, w, fh, fw, dst_cpitch,
                                                                           ch_off, in_scale, in_shift);
  TECO_CUDA_LAUNCH_CHECK("teco_warp_s2d_fused");
  return TECO_OK;
}

int teco_upscale4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, float scale, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0, "teco_upscale4_f32: bad argument");
  LAUNCH1D(upscale4_f32_kernel, (long long)N * h * w * 16 * C, x, y, N, h, w, C, scale);
  return TECO_OK;
}

int teco_bicubic4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t in_cpitch,
                      void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && in_cpitch >= C, "teco_bicubic4_f32: bad argument");
  if (C == 3 && (((uintptr_t)y) & 15) == 0) {
    LAUNCH1D(bicubic4_rgb_f32_kernel, (long long)N * h * w * 4, x, y, N, h, w, in_cpitch);
    return TECO_OK;
  }
  LAUNCH1D(bicubic4_f32_kernel, (long long)N * h * w * 16 * C, x, y, N, h, w, C, in_cpitch);
  return TECO_OK;
}

int teco_resize_bilinear_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t oh,
                             int32_t ow, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && oh > 0 && ow > 0, "teco_resize_bilinear_f32: bad argument");
  LAUNCH1D(resize_bilinear_f32_kernel, (long long)N * oh * ow * C, x, y, N, h, w, C, oh, ow);
  return TECO_OK;
}

int teco_resize_bilinear_bwd_f32(const float* dy, float* dx, int32_t N, int32_t h, int32_t w, int32_t C, int32_t oh,
                                 int32_t ow, void* stream) {
  TECO_CHECK_ARG(dy && dx && N > 0 && h > 0 && w > 0 && C > 0 && oh > 0 && ow > 0, "teco_resize_bilinear_bwd_f32: bad argument");
  TECO_CUDA_CALL(cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)N * h * w * C, (cudaStream_t)stream));
  LAUNCH1D(resize_bilinear_bwd_f32_kernel, (long long)N * oh * ow * C, dy, dx, N, h, w, C, oh, ow);
  return TECO_OK;
}

int teco_maxpool2_f32(const float* x, float* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && H >= 2 && W >= 2 && C > 0, "teco_maxpool2_f32: bad argument");
  LAUNCH1D(maxpool2_f32_kernel, (long long)N * (H / 2) * (W / 2) * C, x, y, N, H, W, C);
  return TECO_OK;
}

int teco_maxpool2_bwd_f32(const float* x, const float* dy, float* dx, int32_t N, int32_t H, int32_t W, int32_t C,
                          void* stream) {
  TECO_CHECK_ARG(x && dy && dx && N > 0 && H >= 2 && W >= 2 && C > 0, "teco_maxpool2_bwd_f32: bad argument");
  if ((H & 1) || (W & 1)) TECO_CUDA_CALL(cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)N * H * W * C, (cudaStream_t)stream));
  LAUNCH1D(maxpool2_bwd_f32_kernel, (long long)N * (H / 2) * (W / 2) * C, x, dy, dx, N, H, W, C);
  return TECO_OK;
}

int teco_maxpool2_bf16(const void* x, void* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && H >= 2 && W >= 2 && C > 0 && (C % 8) == 0, "teco_maxpool2_bf16: C must be a multiple of 8");
  LAUNCH1D(maxpool2_bf16_kernel, (long long)N * (H / 2) * (W / 2) * (C / 8), (const uint4*)x, (uint4*)y, N, H, W, C / 8);
  return TECO_OK;
}

int teco_resize2x_bf16(const void* x, void* y, int32_t N, int32_t h, int32_t w, int32_t C, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && (C % 8) == 0, "teco_resize2x_bf16: C must be a multiple of 8");
  LAUNCH1D(resize2x_bf16_kernel, (long long)N * h * w * 4 * (C / 8), (const uint4*)x, (uint4*)y, N, h, w, C / 8);
  return TECO_OK;
}

int teco_space_to_depth4_f32(const float* x, float* y, int32_t N, int32_t h, int32_t w, int32_t C, int32_t out_cpitch,
                             int32_t ch_off, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && ch_off >= 0 && ch_off + 16 * C <= out_cpitch,
                 "teco_space_to_depth4_f32: bad argument");
  LAUNCH1D(s2d4_f32_kernel, (long long)N * h * w * 16 * C, x, y, N, h, w, C, out_cpitch, ch_off, false);
  return TECO_OK;
}

int teco_depth_to_space4_f32(const float* y, float* x, int32_t N, int32_t h, int32_t w, int32_t C, int32_t in_cpitch,
                             int32_t ch_off, void* stream) {
  TECO_CHECK_ARG(x && y && N > 0 && h > 0 && w > 0 && C > 0 && ch_off >= 0 && ch_off + 16 * C <= in_cpitch,
                 "teco_depth_to_space4_f32: bad argument");
  LAUNCH1D(s2d4_f32_kernel, (long long)N * h * w * 16 * C, x, const_cast<float*>(y), N, h, w, C, in_cpitch, ch_off, true);
  return TECO_OK;
}

int teco_gauss_down4_f32(const float* hr, float* lr, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  TECO_CHECK_ARG(hr && lr && N > 0 && H >= 9 && W >= 9 && C > 0, "teco_gauss_down4_f32: need H,W >= 9");
  static bool init = false;
  if (!init) {
    double g[9], s = 0;
    for (int i = 0; i < 9; ++i) { double a = (i - 4) / 1.5; g[i] = exp(-0.5 * a * a); s += g[i]; }
    float gf[9];
    for (int i = 0; i < 9; ++i) gf[i] = (float)(g[i] / s);
    TECO_CUDA_CALL(cudaMemcpyToSymbol(c_gauss9, gf, sizeof(gf)));
    init = true;
  }
  int oh = (H - 9) / 4 + 1, ow = (W - 9) / 4 + 1;
  LAUNCH1D(gauss_down4_f32_kernel, (long long)N * oh * ow * C, hr, lr, N, H, W, C);
  return TECO_OK;
}

}  // extern "C"
