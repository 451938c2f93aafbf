// optflow.cu -- the tOF metric of the reference's metrics.py:135-169 on the device: cv2's COLOR_RGB2GRAY and
// cv2.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags = 0),
// batched over every frame pair of a scene, and the per-pair mean L2 norm of the flow difference inside crop_8x8.
// The algorithm, stage by stage, is pinned against cv2 in tests/golden/tof_ref.py; the comments here only name the
// stage.  Launches per pyramid level (coarsest first):
//   level_rows_kernel   per frame: horizontal Gaussian pre-blur of the grey frame fused with the horizontal resize;
//   level_poly_kernel   per frame: vertical pre-blur + vertical resize into a shared-memory tile, then the polynomial
//                       expansion R (5 floats per pixel).  Frame i is `next` of pair (i-1, i) and `prev` of pair
//                       (i, i+1): its expansion is computed once and read by both pairs;
//   flow_init_kernel    per pair: resize of the coarser flow (x 1/pyr_scale, or zero) and the matrices M;
//   flow_iter_kernel    per pair, once per iteration: box mean of M (double sums), the 2x2 solve, the flow write and,
//                       before the last iteration, the new M into the other M buffer (neighbouring tiles still read
//                       the old one).  Each iteration is a Jacobi step, as cv2's in-place sweep is.
// No atomics anywhere: a pair's flow does not depend on which other pairs share the batch.
#include <math.h>
#include "teco_common.cuh"

namespace {
constexpr int MAX_TAPS = 255;        // Gaussian pre-blur taps (level 3 at pyr_scale 0.5 needs 19)
constexpr int MAX_POLY_N = 7;        // expansion radius (cv2 recommends 5 or 7)
constexpr int MAX_BOX_R = 7;         // winsize <= 15
constexpr int TW = 32, TH = 8;       // output tile of the per-pixel kernels: 32 x 8 pixels, 256 threads
constexpr int PTH = 16;              // rows per tile of the expansion kernel (256 threads, 2 rows each)
constexpr int BORDER = 5;
__constant__ float kBorderW[BORDER] = {0.14f, 0.14f, 0.4472f, 0.4472f, 0.4472f};

struct Blur {
  int ksize;
  float k[MAX_TAPS];
};
struct Poly {
  int n;
  float g[MAX_POLY_N + 1], xg[MAX_POLY_N + 1], xxg[MAX_POLY_N + 1];
  double ig11, ig03, ig33, ig55;
};

__host__ __device__ inline int reflect101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
  return i;
}

// cv2's INTER_LINEAR source taps along one axis: half-pixel centres, clamped at both ends.
struct Tap { int i0, i1; float a; };
__device__ __forceinline__ Tap linear_tap(int d, int src, double scale) {
  float f = (float)((d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (s < 0) { s = 0; f = 0.f; }
  if (s >= src - 1) { s = src - 1; f = 0.f; }
  return {s, min(s + 1, src - 1), f};
}

// ---- pyramid level image -------------------------------------------------------------------------------------------
// T[f][y][dx] = (1-a) Hblur(y, sx0) + a Hblur(y, sx1): the full-height, level-width intermediate.
__global__ void __launch_bounds__(256) level_rows_kernel(const uint8_t* __restrict__ grey, int H, int W, int lw, double sx,
                                                         Blur b, float* __restrict__ T) {
  const int dx = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
  if (dx >= lw) return;
  const uint8_t* row = grey + ((size_t)f * H + y) * W;
  const Tap t = linear_tap(dx, W, sx);
  const int r = b.ksize >> 1;
  float v0 = 0.f, v1 = 0.f;
  for (int j = 0; j < b.ksize; ++j) v0 += b.k[j] * (float)row[reflect101(t.i0 + j - r, W)];
  if (t.a != 0.f)
    for (int j = 0; j < b.ksize; ++j) v1 += b.k[j] * (float)row[reflect101(t.i1 + j - r, W)];
  T[((size_t)f * H + y) * lw + dx] = t.a != 0.f ? v0 * (1.f - t.a) + v1 * t.a : v0;
}

// Level image tile (vertical blur + resize of T) with a poly.n halo in shared memory, then the expansion.
// R layout: frame stride rstride floats, pixel-major, 5 floats per pixel (r_y, r_x, r_yy, r_xx, r_xy).
__global__ void __launch_bounds__(256) level_poly_kernel(const float* __restrict__ T, int H, int lh, int lw, double sy,
                                                         Blur b, Poly p, float* __restrict__ R, size_t rstride) {
  constexpr int SW = TW + 2 * MAX_POLY_N, SH = PTH + 2 * MAX_POLY_N;
  __shared__ float img[SH][SW];
  __shared__ float vp[3][PTH][SW];
  const int f = blockIdx.z, n = p.n, x0 = blockIdx.x * TW, y0 = blockIdx.y * PTH;
  const int sw = TW + 2 * n, sh = PTH + 2 * n;
  const float* Tf = T + (size_t)f * H * lw;
  const int r = b.ksize >> 1;
  for (int i = threadIdx.x; i < sw * sh; i += 256) {
    const int ry = i / sw, rx = i - ry * sw;
    const int y = min(max(y0 + ry - n, 0), lh - 1), x = min(max(x0 + rx - n, 0), lw - 1);   // replicated borders
    const Tap t = linear_tap(y, H, sy);
    float v0 = 0.f, v1 = 0.f;
    for (int j = 0; j < b.ksize; ++j) v0 += b.k[j] * Tf[(size_t)reflect101(t.i0 + j - r, H) * lw + x];
    if (t.a != 0.f)
      for (int j = 0; j < b.ksize; ++j) v1 += b.k[j] * Tf[(size_t)reflect101(t.i1 + j - r, H) * lw + x];
    img[ry][rx] = t.a != 0.f ? v0 * (1.f - t.a) + v1 * t.a : v0;
  }
  __syncthreads();
  // vertical part, in float as cv2 keeps it
  for (int i = threadIdx.x; i < PTH * sw; i += 256) {
    const int ry = i / sw, rx = i - ry * sw;
    float c0 = img[ry + n][rx] * p.g[0], c1 = 0.f, c2 = 0.f;
    for (int k = 1; k <= n; ++k) {
      const float up = img[ry + n - k][rx], dn = img[ry + n + k][rx], s = up + dn;
      c0 += p.g[k] * s;
      c1 += p.xg[k] * (dn - up);
      c2 += p.xxg[k] * s;
    }
    vp[0][ry][rx] = c0; vp[1][ry][rx] = c1; vp[2][ry][rx] = c2;
  }
  __syncthreads();
  // horizontal part, in double
  const int tx = threadIdx.x & (TW - 1);
  for (int ty = threadIdx.x / TW; ty < PTH; ty += 256 / TW) {
    const int x = x0 + tx, y = y0 + ty;
    if (x >= lw || y >= lh) continue;
    const int c = tx + n;
    double b1 = (double)vp[0][ty][c] * p.g[0], b2 = 0.0, b3 = (double)vp[1][ty][c] * p.g[0];
    double b4 = 0.0, b5 = (double)vp[2][ty][c] * p.g[0], b6 = 0.0;
    for (int k = 1; k <= n; ++k) {
      const double a0 = vp[0][ty][c + k], m0 = vp[0][ty][c - k], a1 = vp[1][ty][c + k], m1 = vp[1][ty][c - k];
      const double tg = a0 + m0;
      b1 += tg * p.g[k];
      b4 += tg * p.xxg[k];
      b2 += (a0 - m0) * p.xg[k];
      b3 += (a1 + m1) * p.g[k];
      b6 += (a1 - m1) * p.xg[k];
      b5 += ((double)vp[2][ty][c + k] + (double)vp[2][ty][c - k]) * p.g[k];
    }
    float* o = R + f * rstride + ((size_t)y * lw + x) * 5;
    o[0] = (float)(b3 * p.ig11);
    o[1] = (float)(b2 * p.ig11);
    o[2] = (float)(b1 * p.ig03 + b5 * p.ig33);
    o[3] = (float)(b1 * p.ig03 + b4 * p.ig33);
    o[4] = (float)(b6 * p.ig55);
  }
}

// ---- matrices and flow ---------------------------------------------------------------------------------------------
struct PairLevel {
  const float* R;           // expansions of all frames at this level
  size_t rstride;           // floats per frame in R
  const int2* pairs;        // (prev, next) frame indices
  int lh, lw;
  float* flow;              // this level's flows, fstride floats per pair
  size_t fstride;
  size_t mstride;           // floats per pair in each M buffer
};

__device__ __forceinline__ float border_w(int x, int w) {
  return (x < BORDER ? kBorderW[x] : 1.f) * (x >= w - BORDER ? kBorderW[w - x - 1] : 1.f);
}

// cv2's matrix update at pixel (x, y) with flow (dx, dy): M = (G11, G12, G22, h1, h2).
__device__ __forceinline__ void update_m(const float* __restrict__ R0, const float* __restrict__ R1, int lh, int lw, int x,
                                         int y, float dx, float dy, float* __restrict__ M) {
  const float* r0 = R0 + ((size_t)y * lw + x) * 5;
  float fx = (float)x + dx, fy = (float)y + dy;
  const int x1 = (int)floorf(fx), y1 = (int)floorf(fy);
  fx -= (float)x1;
  fy -= (float)y1;
  float r2, r3, r4, r5, r6;
  if ((unsigned)x1 < (unsigned)(lw - 1) && (unsigned)y1 < (unsigned)(lh - 1)) {
    const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
    const float* q = R1 + ((size_t)y1 * lw + x1) * 5;
    const float* qd = q + (size_t)lw * 5;
    float s[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) s[c] = a00 * q[c] + a01 * q[5 + c] + a10 * qd[c] + a11 * qd[5 + c];
    r2 = s[0]; r3 = s[1];
    r4 = (r0[2] + s[2]) * 0.5f;
    r5 = (r0[3] + s[3]) * 0.5f;
    r6 = (r0[4] + s[4]) * 0.25f;
  } else {
    r2 = r3 = 0.f;
    r4 = r0[2];
    r5 = r0[3];
    r6 = r0[4] * 0.5f;
  }
  r2 = (r0[0] - r2) * 0.5f;
  r3 = (r0[1] - r3) * 0.5f;
  r2 += r4 * dy + r6 * dx;
  r3 += r6 * dy + r5 * dx;
  if ((unsigned)(x - BORDER) >= (unsigned)(lw - 2 * BORDER) || (unsigned)(y - BORDER) >= (unsigned)(lh - 2 * BORDER)) {
    const float s = border_w(x, lw) * border_w(y, lh);
    r2 *= s; r3 *= s; r4 *= s; r5 *= s; r6 *= s;
  }
  M[0] = r4 * r4 + r6 * r6;
  M[1] = (r4 + r5) * r6;
  M[2] = r5 * r5 + r6 * r6;
  M[3] = r4 * r2 + r6 * r3;
  M[4] = r6 * r2 + r5 * r3;
}

// Flow of this level from the coarser one (bilinear resize times 1/pyr_scale; zero at the coarsest level), then M.
__global__ void __launch_bounds__(256) flow_init_kernel(PairLevel L, const float* __restrict__ coarse, size_t cstride, int ch,
                                                        int cw, float inv_scale, float* __restrict__ M) {
  const int pr = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= L.lh * L.lw) return;
  const int y = i / L.lw, x = i - y * L.lw;
  float dx = 0.f, dy = 0.f;
  if (coarse != nullptr) {
    const float* c = coarse + pr * cstride;
    const Tap tx = linear_tap(x, cw, 1.0 / ((double)L.lw / cw)), ty = linear_tap(y, ch, 1.0 / ((double)L.lh / ch));
    const float* a0 = c + (size_t)ty.i0 * cw * 2;
    const float* a1 = c + (size_t)ty.i1 * cw * 2;
    const float u0 = a0[tx.i0 * 2] * (1.f - tx.a) + a0[tx.i1 * 2] * tx.a, v0 = a0[tx.i0 * 2 + 1] * (1.f - tx.a) + a0[tx.i1 * 2 + 1] * tx.a;
    const float u1 = a1[tx.i0 * 2] * (1.f - tx.a) + a1[tx.i1 * 2] * tx.a, v1 = a1[tx.i0 * 2 + 1] * (1.f - tx.a) + a1[tx.i1 * 2 + 1] * tx.a;
    dx = (u0 * (1.f - ty.a) + u1 * ty.a) * inv_scale;
    dy = (v0 * (1.f - ty.a) + v1 * ty.a) * inv_scale;
  }
  float* fl = L.flow + pr * L.fstride + (size_t)i * 2;
  fl[0] = dx;
  fl[1] = dy;
  const int2 pp = L.pairs[pr];
  update_m(L.R + pp.x * L.rstride, L.R + pp.y * L.rstride, L.lh, L.lw, x, y, dx, dy, M + pr * L.mstride + (size_t)i * 5);
}

// One iteration: box mean of M over (2m+1)^2 (replicated borders, double sums), the solve, and the next M if wanted.
__global__ void __launch_bounds__(256) flow_iter_kernel(PairLevel L, int m, const float* __restrict__ Min, float* __restrict__ Mout) {
  constexpr int SW = TW + 2 * MAX_BOX_R, SH = TH + 2 * MAX_BOX_R;
  __shared__ float sm[SH][SW][5];
  __shared__ double vs[TH][SW][5];
  const int pr = blockIdx.z, x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
  const int sw = TW + 2 * m, sh = TH + 2 * m;
  const float* Mi = Min + pr * L.mstride;
  for (int i = threadIdx.x; i < sw * sh; i += 256) {
    const int ry = i / sw, rx = i - ry * sw;
    const int y = min(max(y0 + ry - m, 0), L.lh - 1), x = min(max(x0 + rx - m, 0), L.lw - 1);
    const float* s = Mi + ((size_t)y * L.lw + x) * 5;
#pragma unroll
    for (int c = 0; c < 5; ++c) sm[ry][rx][c] = s[c];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < TH * sw; i += 256) {
    const int ry = i / sw, rx = i - ry * sw;
    double a[5] = {0, 0, 0, 0, 0};
    for (int k = 0; k <= 2 * m; ++k)
#pragma unroll
      for (int c = 0; c < 5; ++c) a[c] += (double)sm[ry + k][rx][c];
#pragma unroll
    for (int c = 0; c < 5; ++c) vs[ry][rx][c] = a[c];
  }
  __syncthreads();
  const int tx = threadIdx.x & (TW - 1), ty = threadIdx.x / TW;
  const int x = x0 + tx, y = y0 + ty;
  if (x >= L.lw || y >= L.lh) return;
  double a[5] = {0, 0, 0, 0, 0};
  for (int k = 0; k <= 2 * m; ++k)
#pragma unroll
    for (int c = 0; c < 5; ++c) a[c] += vs[ty][tx + k][c];
  const double scale = 1.0 / (double)((2 * m + 1) * (2 * m + 1));
  const double g11 = a[0] * scale, g12 = a[1] * scale, g22 = a[2] * scale, h1 = a[3] * scale, h2 = a[4] * scale;
  const double idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3);
  const float dx = (float)((g11 * h2 - g12 * h1) * idet), dy = (float)((g22 * h1 - g12 * h2) * idet);
  float* fl = L.flow + pr * L.fstride + ((size_t)y * L.lw + x) * 2;
  fl[0] = dx;
  fl[1] = dy;
  if (Mout != nullptr) {
    const int2 pp = L.pairs[pr];
    update_m(L.R + pp.x * L.rstride, L.R + pp.y * L.rstride, L.lh, L.lw, x, y, dx, dy,
             Mout + pr * L.mstride + ((size_t)y * L.lw + x) * 5);
  }
}

// ---- grey conversion and tOF sums ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grey_kernel(const uint8_t* __restrict__ rgb, int H, int W, int h, int w,
                                                   uint8_t* __restrict__ grey) {
  const int n = blockIdx.y;
  const long long total = (long long)h * w;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int y = (int)(i / w), x = (int)(i - (long long)y * w);
    const uint8_t* p = rgb + (((size_t)n * H + y) * W + x) * 3;
    grey[(size_t)n * total + i] = (uint8_t)((9798u * p[0] + 19235u * p[1] + 3735u * p[2] + (1u << 14)) >> 15);
  }
}

constexpr int SUM_TPB = 512;
__global__ void __launch_bounds__(SUM_TPB) tof_sums_kernel(const float* __restrict__ ft, const float* __restrict__ fo, int H,
                                                          int W, int y0, int x0, int h, int w, double* __restrict__ sums) {
  const int pr = blockIdx.x;
  const float* a = ft + (size_t)pr * H * W * 2;
  const float* b = fo + (size_t)pr * H * W * 2;
  double s = 0.0;
  for (long long i = threadIdx.x; i < (long long)h * w; i += SUM_TPB) {
    const int r = (int)(i / w), c = (int)(i - (long long)r * w);
    const size_t o = ((size_t)(y0 + r) * W + x0 + c) * 2;
    const double du = (double)(a[o] - b[o]), dv = (double)(a[o + 1] - b[o + 1]);
    s += sqrt(du * du + dv * dv);
  }
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
  __shared__ double red[SUM_TPB / 32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < SUM_TPB / 32; ++k) s += red[k];
    sums[pr] = s;
  }
}

// ---- host-side plan ------------------------------------------------------------------------------------------------
constexpr int MIN_SIZE = 32;

int top_level(int H, int W, double s, int levels) {
  double scale = 1.0;
  for (int k = 0; k < levels; ++k) {
    scale *= s;
    if (W * scale < MIN_SIZE || H * scale < MIN_SIZE) return k;
  }
  return levels;
}

double level_scale(double s, int k) {
  double scale = 1.0;
  for (int i = 0; i < k; ++i) scale *= s;
  return scale;
}

struct Layout {
  size_t T, R, F0, F1, M0, M1, pairs, total;
  size_t area1;
};

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

Layout plan(int F, int P, int H, int W, double s, int levels) {
  Layout L{};
  const int top = top_level(H, W, s, levels);
  L.area1 = top >= 1 ? (size_t)llrint(H * s) * (size_t)llrint(W * s) : 0;
  const size_t hw = (size_t)H * W;
  size_t off = 0;
  L.T = off; off += align256(sizeof(float) * F * hw);
  L.R = off; off += align256(sizeof(float) * F * hw * 5);
  L.F0 = off; off += align256(sizeof(float) * P * L.area1 * 2);
  L.F1 = off; off += align256(sizeof(float) * P * L.area1 * 2);
  L.M0 = off; off += align256(sizeof(float) * P * hw * 5);
  L.M1 = off; off += align256(sizeof(float) * P * hw * 5);
  L.pairs = off; off += align256(sizeof(int32_t) * P * 2);
  L.total = off;
  return L;
}

bool sizes_ok(int F, int P, int H, int W, double s, int levels) {
  return F > 0 && P > 0 && P <= 65535 && F <= 65535 && H >= 2 && W >= 2 && H <= 65535 && (long long)H * W < (1LL << 31) &&
         s > 0.0 && s < 1.0 && levels >= 0;
}

Blur make_blur(double scale) {
  Blur b{};
  const double sigma = (1.0 / scale - 1.0) * 0.5;
  b.ksize = max((int)lrint(sigma * 5) | 1, 3);
  if (b.ksize > MAX_TAPS) { b.ksize = 0; return b; }
  if (sigma <= 0.0 && b.ksize == 3) {
    b.k[0] = 0.25f; b.k[1] = 0.5f; b.k[2] = 0.25f;
    return b;
  }
  double sum = 0.0, tmp[MAX_TAPS];
  for (int i = 0; i < b.ksize; ++i) {
    const double x = i - (b.ksize - 1) * 0.5;
    tmp[i] = exp(-x * x / (2.0 * sigma * sigma));
    sum += tmp[i];
  }
  for (int i = 0; i < b.ksize; ++i) b.k[i] = (float)(tmp[i] / sum);
  return b;
}

// 6x6 Gram matrix of the weighted fit of 1, x, y, x^2, y^2, xy; its inverse is needed through four entries only.
Poly make_poly(int n, double sigma) {
  Poly p{};
  p.n = n;
  if (sigma < 1.1920928955078125e-7) sigma = n * 0.3;
  float g[2 * MAX_POLY_N + 1];
  double s = 0.0;
  for (int x = -n; x <= n; ++x) { g[x + n] = (float)exp(-x * x / (2 * sigma * sigma)); s += g[x + n]; }
  s = 1.0 / s;
  for (int x = -n; x <= n; ++x) g[x + n] = (float)(g[x + n] * s);
  for (int k = 0; k <= n; ++k) { p.g[k] = g[k + n]; p.xg[k] = (float)(k * g[k + n]); p.xxg[k] = (float)(k * k * g[k + n]); }
  double G00 = 0, G11 = 0, G33 = 0, G55 = 0;
  for (int y = -n; y <= n; ++y)
    for (int x = -n; x <= n; ++x) {
      const double w = (double)g[y + n] * g[x + n];
      G00 += w; G11 += w * x * x; G33 += w * x * x * x * x; G55 += w * x * x * y * y;
    }
  // The Gram matrix splits into the block {1, x^2, y^2} = [[G00, G11, G11], [G11, G33, G55], [G11, G55, G33]] and the
  // diagonal entries G11 (x, y) and G55 (xy).  Inverting the 3x3 block in closed form:
  const double a = G00, b = G11, c = G33, d = G55;
  const double det = a * (c * c - d * d) - b * (b * c - b * d) + b * (b * d - c * b);
  p.ig11 = 1.0 / b;
  p.ig55 = 1.0 / d;
  p.ig03 = (b * d - b * c) / det;              // cofactor (1,0) of the symmetric block over det
  p.ig33 = (a * c - b * b) / det;              // cofactor (1,1)
  return p;
}
}  // namespace

extern "C" {

int teco_grey_u8(const uint8_t* rgb, int32_t N, int32_t H, int32_t W, int32_t h, int32_t w, uint8_t* grey, void* stream) {
  TECO_CHECK_ARG(rgb && grey, "teco_grey_u8: NULL frame pointer");
  TECO_CHECK_ARG(N > 0 && N <= 65535 && h > 0 && w > 0 && h <= H && w <= W,
                 "teco_grey_u8: bad sizes N=%d, frames %dx%d, cut %dx%d", N, H, W, h, w);
  const long long total = (long long)h * w;
  const int bx = (int)max(1LL, min((total + 1023) / 1024, (long long)(4 * teco_sm_count())));
  grey_kernel<<<dim3(bx, N), 256, 0, (cudaStream_t)stream>>>(rgb, H, W, h, w, grey);
  TECO_CUDA_LAUNCH_CHECK("teco_grey_u8");
  return TECO_OK;
}

int64_t teco_farneback_workspace_bytes(int32_t F, int32_t P, int32_t H, int32_t W, double pyr_scale, int32_t levels) {
  if (!sizes_ok(F, P, H, W, pyr_scale, levels)) {
    teco_set_error("teco_farneback_workspace_bytes: bad sizes F=%d P=%d %dx%d pyr_scale=%g levels=%d", F, P, H, W, pyr_scale,
                   levels);
    return TECO_E_INVALID;
  }
  return (int64_t)plan(F, P, H, W, pyr_scale, levels).total;
}

int teco_farneback_flow(const uint8_t* grey, int32_t F, int32_t H, int32_t W, const int32_t* pairs_host, int32_t P,
                        double pyr_scale, int32_t levels, int32_t winsize, int32_t iterations, int32_t poly_n,
                        double poly_sigma, int32_t flags, void* workspace, int64_t workspace_bytes, float* flow, void* stream) {
  TECO_CHECK_ARG(grey && pairs_host && workspace && flow, "teco_farneback_flow: NULL pointer");
  TECO_CHECK_ARG(sizes_ok(F, P, H, W, pyr_scale, levels), "teco_farneback_flow: bad sizes F=%d P=%d %dx%d pyr_scale=%g levels=%d",
                 F, P, H, W, pyr_scale, levels);
  TECO_CHECK_ARG(flags == 0, "teco_farneback_flow: only flags = 0 is implemented (got %d)", flags);
  TECO_CHECK_ARG(winsize >= 1 && winsize <= 2 * MAX_BOX_R + 1 && (winsize & 1), "teco_farneback_flow: winsize must be odd, 1..%d",
                 2 * MAX_BOX_R + 1);
  TECO_CHECK_ARG(iterations >= 1, "teco_farneback_flow: iterations must be >= 1");
  TECO_CHECK_ARG(poly_n >= 1 && poly_n <= MAX_POLY_N, "teco_farneback_flow: poly_n must be 1..%d", MAX_POLY_N);
  TECO_CHECK_ARG(poly_sigma >= 0.0 && poly_sigma < 1e6, "teco_farneback_flow: bad poly_sigma %g", poly_sigma);
  for (int i = 0; i < 2 * P; ++i)
    TECO_CHECK_ARG(pairs_host[i] >= 0 && pairs_host[i] < F, "teco_farneback_flow: pair %d names frame %d of %d", i / 2,
                   pairs_host[i], F);
  const Layout Lo = plan(F, P, H, W, pyr_scale, levels);
  TECO_CHECK_ARG(workspace_bytes >= (int64_t)Lo.total, "teco_farneback_flow: workspace of %lld bytes, %zu needed",
                 (long long)workspace_bytes, Lo.total);
  const int top = top_level(H, W, pyr_scale, levels);
  Blur blurs[64];
  TECO_CHECK_ARG(top < 64, "teco_farneback_flow: too many pyramid levels");
  for (int k = 0; k <= top; ++k) {
    blurs[k] = make_blur(level_scale(pyr_scale, k));
    TECO_CHECK_ARG(blurs[k].ksize > 0, "teco_farneback_flow: level %d needs a pre-blur wider than %d taps", k, MAX_TAPS);
  }
  const Poly poly = make_poly(poly_n, poly_sigma);

  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  float* T = (float*)(ws + Lo.T);
  float* R = (float*)(ws + Lo.R);
  float* Fw[2] = {(float*)(ws + Lo.F0), (float*)(ws + Lo.F1)};
  float* Mb[2] = {(float*)(ws + Lo.M0), (float*)(ws + Lo.M1)};
  int2* pairs = (int2*)(ws + Lo.pairs);
  TECO_CUDA_CALL(cudaMemcpyAsync(pairs, pairs_host, sizeof(int32_t) * 2 * P, cudaMemcpyHostToDevice, st));

  const size_t rstride = (size_t)H * W * 5;
  const float* coarse = nullptr;
  size_t cstride = 0;
  int ch = 0, cw = 0;
  for (int k = top; k >= 0; --k) {
    const double scale = level_scale(pyr_scale, k);
    const int lw = (int)lrint(W * scale), lh = (int)lrint(H * scale);
    level_rows_kernel<<<dim3(teco_ceil_div(lw, 256), H, F), 256, 0, st>>>(grey, H, W, lw, 1.0 / ((double)lw / W), blurs[k], T);
    TECO_CUDA_LAUNCH_CHECK("teco_farneback_flow (level_rows_kernel)");
    level_poly_kernel<<<dim3(teco_ceil_div(lw, TW), teco_ceil_div(lh, PTH), F), 256, 0, st>>>(
        T, H, lh, lw, 1.0 / ((double)lh / H), blurs[k], poly, R, rstride);
    TECO_CUDA_LAUNCH_CHECK("teco_farneback_flow (level_poly_kernel)");

    PairLevel L{R, rstride, pairs, lh, lw, k == 0 ? flow : Fw[k & 1], k == 0 ? (size_t)H * W * 2 : Lo.area1 * 2, (size_t)H * W * 5};
    flow_init_kernel<<<dim3(teco_ceil_div((long long)lh * lw, 256), P), 256, 0, st>>>(L, coarse, cstride, ch, cw,
                                                                                      (float)(1.0 / pyr_scale), Mb[0]);
    TECO_CUDA_LAUNCH_CHECK("teco_farneback_flow (flow_init_kernel)");
    const dim3 grid(teco_ceil_div(lw, TW), teco_ceil_div(lh, TH), P);
    for (int it = 0; it < iterations; ++it) {
      flow_iter_kernel<<<grid, 256, 0, st>>>(L, winsize / 2, Mb[it & 1], it + 1 < iterations ? Mb[(it + 1) & 1] : nullptr);
      TECO_CUDA_LAUNCH_CHECK("teco_farneback_flow (flow_iter_kernel)");
    }
    coarse = L.flow;
    cstride = L.fstride;
    ch = lh;
    cw = lw;
  }
  return TECO_OK;
}

int teco_tof_sums(const float* flow_t, const float* flow_o, int32_t P, int32_t H, int32_t W, int32_t y0, int32_t x0, int32_t h,
                  int32_t w, double* sums, void* stream) {
  TECO_CHECK_ARG(flow_t && flow_o && sums, "teco_tof_sums: NULL pointer");
  TECO_CHECK_ARG(P > 0 && H > 0 && W > 0, "teco_tof_sums: bad sizes P=%d %dx%d", P, H, W);
  TECO_CHECK_ARG(y0 >= 0 && x0 >= 0 && h > 0 && w > 0 && y0 + h <= H && x0 + w <= W,
                 "teco_tof_sums: window %d+%d x %d+%d does not fit %dx%d", y0, h, x0, w, H, W);
  tof_sums_kernel<<<P, SUM_TPB, 0, (cudaStream_t)stream>>>(flow_t, flow_o, H, W, y0, x0, h, w, sums);
  TECO_CUDA_LAUNCH_CHECK("teco_tof_sums");
  return TECO_OK;
}

}  // extern "C"
