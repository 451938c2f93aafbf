"""numpy restatement of the tOF metric of the reference's metrics.py:135-169: cv2.cvtColor(RGB2GRAY), then
cv2.calcOpticalFlowFarneback(prev, next, None, 0.5, 3, 15, 3, 5, 1.2, 0) on consecutive target and result frames, then the
mean L2 norm of the flow difference inside crop_8x8.  It is the CPU yardstick of the CUDA kernels in
tecogan_b200/csrc/optflow.cu, and every rule below was confirmed against cv2 4.13 (tests/golden/make_golden_tof.py
builds the fixtures, tests/test_tof_host.py re-checks them):

Grey conversion (COLOR_RGB2GRAY on uint8)
  grey = (9798 R + 19235 G + 3735 B + 2^14) >> 15.  Equal to cv2 on all 2^24 triplets.  The textbook 14-bit rule
  (4899, 9617, 1868) and the 16-bit rule (19595, 38470, 7471) each miss tens of thousands of triplets.

Pyramid (flags = 0)
  * Depth: level k exists while W s^k >= 32 and H s^k >= 32 (s = pyr_scale).  At 144x180, levels=3 equals levels=2;
    at 63x100, levels=3 equals levels=0.
  * Level k is round-half-even(W s^k) x round-half-even(H s^k).  Its image is the float grey frame blurred by a Gaussian of
    sigma = (1/s^k - 1)/2, size max(round(5 sigma)|1, 3), reflect-101 borders, then resized bilinearly with half-pixel
    centres (source coordinates clamped at the edges).  At k = 0 sigma is 0 and cv2 uses its fixed size-3 kernel
    [1, 2, 1]/4: dropping that blur moves a single-level flow by up to 0.2 px, so it is not a rounding effect.
Polynomial expansion
  * poly_n is the window RADIUS: 2 poly_n + 1 taps (11 for poly_n = 5).  A 5-tap window (radius 2) misses cv2 by 0.14 px.
  * Weights g = normalised exp(-x^2 / 2 sigma^2), x g and x^2 g; the 6x6 Gram matrix enters through four constants of its
    inverse (ig11, ig03, ig33, ig55).  Vertical pass first, then horizontal; replicated borders.
  * Five coefficients per pixel, in cv2's order: r_y, r_x, r_yy, r_xx, r_xy (the constant term is not stored).
Flow initialisation
  Zero at the coarsest level; otherwise the coarser flow resized bilinearly (as above) and multiplied by 1/s.
Matrix update (per pixel x with flow d)
  * R1 is sampled bilinearly at x + d when the 2x2 neighbourhood is inside the level; the quadratic terms are averaged
    with R0 (xy term: sum times 1/4).  When the neighbourhood is outside, cv2 does NOT use zero matrices for the quadratic
    part: it uses R0's own (r_yy, r_xx unchanged, r_xy halved) and zero linear terms.  Zero matrices miss cv2 by 0.12 px.
    With zero flow the last row and column already take this branch.
  * Linear terms: (R0 - R1)/2, plus A d.  Within 5 pixels of an edge everything is scaled by the product of the border
    weights of the row and the column, {0.14, 0.14, 0.4472, 0.4472, 0.4472} at distance 0..4.  The often-quoted table
    {0.14, 0.14, 0.4472, 0.8943, 1} misses cv2 by 0.27 px; the one here was fitted to cv2 (residual 3e-6 px).
  * M = (G11, G12, G22, h1, h2) = (r4^2 + r6^2, (r4 + r5) r6, r5^2 + r6^2, r4 r2 + r6 r3, r6 r2 + r5 r3).
Flow update
  * winsize x winsize box mean of M with replicated borders (sums in double), then
    flow = ((G11 h2 - G12 h1), (G22 h1 - G12 h2)) / (G11 G22 - G12^2 + 1e-3).
  * Every iteration but the last updates M again from the new flow.  cv2 does that in place, for rows the box filter no
    longer reads, so each iteration is a pure Jacobi step: a single-level, two-iteration run matches this restatement,
    which updates all of M at once, to 3e-6 px.
tOF
  Frames cutfr .. n-cutfr-1; the result is cut to the target size; flows on the full grey frames; crop_8x8 on the flow
  fields; per-pixel L2 norm of the difference; mean over the window.  The first selected frame has no tOF.

Values are stored in cv2's types (float32 images, coefficients, matrices and flows; double box sums and solve) and
computed in double in between, so the restatement and cv2 differ only by rounding: on the calendar frames the flows
agree to 3e-6 px with the reference's parameters and to 6e-5 px with levels=1, winsize=9, iterations=2, pyr_scale=0.6,
poly_sigma=1.5.
"""
import numpy as np

f32 = np.float32
BORDER_W = np.array([0.14, 0.14, 0.4472, 0.4472, 0.4472], dtype=f32)
MIN_SIZE = 32


def rgb_to_grey_u8(rgb):
    """cv2.cvtColor(rgb, COLOR_RGB2GRAY) on uint8 [..., 3], bit for bit."""
    a = np.asarray(rgb)
    assert a.dtype == np.uint8 and a.shape[-1] == 3
    r, g, b = (a[..., i].astype(np.int32) for i in range(3))
    return ((9798 * r + 19235 * g + 3735 * b + (1 << 14)) >> 15).astype(np.uint8)


def pyramid_levels(h, w, pyr_scale, levels):
    """Number of coarser levels cv2 actually builds (0 = one level)."""
    scale = 1.0
    for k in range(levels):
        scale *= pyr_scale
        if w * scale < MIN_SIZE or h * scale < MIN_SIZE:
            return k
    return levels


def level_geometry(h, w, pyr_scale, k):
    """(scale, sigma, ksize, lh, lw) of level k, as cv2 computes them."""
    scale = 1.0
    for _ in range(k):
        scale *= pyr_scale
    sigma = (1.0 / scale - 1.0) * 0.5
    ksize = max(int(np.round(sigma * 5)) | 1, 3)
    return scale, sigma, ksize, int(np.round(h * scale)), int(np.round(w * scale))


def gaussian_kernel(ksize, sigma):
    """cv2.getGaussianKernel(ksize, sigma, CV_32F); sigma <= 0 with ksize 3 is the fixed [1,2,1]/4."""
    if sigma <= 0 and ksize == 3:
        return np.array([0.25, 0.5, 0.25], dtype=f32)
    if sigma <= 0:
        sigma = ((ksize - 1) * 0.5 - 1) * 0.3 + 0.8
    x = np.arange(ksize) - (ksize - 1) * 0.5
    k = np.exp(-x * x / (2.0 * sigma * sigma))
    return (k / k.sum()).astype(f32)


def _reflect101(n, r):
    i = np.arange(-r, n + r)
    if n == 1:
        return np.zeros_like(i)
    period = 2 * (n - 1)
    i = np.abs(i) % period
    return np.where(i >= n, period - i, i)


def gaussian_blur(img, ksize, sigma):
    k = gaussian_kernel(ksize, sigma).astype(np.float64)
    r = ksize // 2
    h, w = img.shape
    a = img.astype(np.float64)
    iy, ix = _reflect101(h, r), _reflect101(w, r)
    a = a[:, ix]
    t = sum(k[j] * a[:, j:j + w] for j in range(ksize))
    t = t[iy, :]
    return sum(k[j] * t[j:j + h, :] for j in range(ksize)).astype(f32)


def _linear_taps(src, dst):
    """Source index and weight of cv2's INTER_LINEAR along one axis (half-pixel centres, clamped)."""
    scale = 1.0 / (dst / src)
    fx = ((np.arange(dst) + 0.5) * scale - 0.5).astype(f32)
    sx = np.floor(fx).astype(np.int64)
    fx = (fx - sx).astype(f32)
    lo = sx < 0
    fx[lo], sx[lo] = 0, 0
    hi = sx >= src - 1
    fx[hi], sx[hi] = 0, src - 1
    return sx, np.minimum(sx + 1, src - 1), fx


def resize_linear(img, dh, dw):
    """cv2.resize(img, (dw, dh), interpolation=INTER_LINEAR) of a float32 [H,W] or [H,W,C] image."""
    h, w = img.shape[:2]
    if (h, w) == (dh, dw):
        return img.astype(f32)
    x0, x1, ax = _linear_taps(w, dw)
    y0, y1, ay = _linear_taps(h, dh)
    a = img.astype(np.float64)
    ex = (slice(None),) + (None,) * (a.ndim - 2)
    ax, ay = ax.astype(np.float64)[ex], ay.astype(np.float64)[:, None][(slice(None), slice(None)) + ex[1:]]
    t = a[:, x0] * (1 - ax) + a[:, x1] * ax
    return (t[y0] * (1 - ay) + t[y1] * ay).astype(f32)


def poly_constants(n, sigma):
    """g, xg, xxg (float32, index -n..n) and the constants ig11, ig03, ig33, ig55 of cv2's expansion."""
    if sigma < np.finfo(np.float32).eps:
        sigma = n * 0.3
    x = np.arange(-n, n + 1)
    g = np.exp(-x * x / (2.0 * sigma * sigma)).astype(f32).astype(np.float64)
    g = (g * (1.0 / g.sum())).astype(f32)
    xg, xxg = (x * g).astype(f32), (x * x * g).astype(f32)
    gd, xd = g.astype(np.float64), x.astype(np.float64)
    gg = gd[:, None] * gd[None, :]                   # [y, x]
    X, Y = xd[None, :], xd[:, None]
    G = np.zeros((6, 6))
    G[0, 0] = gg.sum()
    G[1, 1] = (gg * X * X).sum()
    G[3, 3] = (gg * X ** 4).sum()
    G[5, 5] = (gg * X * X * Y * Y).sum()
    G[2, 2] = G[0, 3] = G[0, 4] = G[3, 0] = G[4, 0] = G[1, 1]
    G[4, 4] = G[3, 3]
    G[3, 4] = G[4, 3] = G[5, 5]
    iG = np.linalg.inv(G)
    return g, xg, xxg, (iG[1, 1], iG[0, 3], iG[3, 3], iG[5, 5])


def poly_expansion(img, n, sigma):
    """[H,W] float32 -> [H,W,5] float32 (r_y, r_x, r_yy, r_xx, r_xy); 2n+1 taps, replicated borders."""
    g, xg, xxg, (ig11, ig03, ig33, ig55) = poly_constants(n, sigma)
    h, w = img.shape
    src = img.astype(np.float64)
    rows = lambda d: src[np.clip(np.arange(h) + d, 0, h - 1)]
    c0 = src * g[n]
    c1 = np.zeros_like(src)
    c2 = np.zeros_like(src)
    for k in range(1, n + 1):
        up, dn = rows(-k), rows(k)
        c0 = c0 + g[n + k] * (up + dn)
        c1 = c1 + xg[n + k] * (dn - up)
        c2 = c2 + xxg[n + k] * (up + dn)
    c0, c1, c2 = (c.astype(f32).astype(np.float64) for c in (c0, c1, c2))
    cols = lambda c, d: c[:, np.clip(np.arange(w) + d, 0, w - 1)]
    b1, b3, b5 = c0 * g[n], c1 * g[n], c2 * g[n]
    b2 = np.zeros_like(src)
    b4 = np.zeros_like(src)
    b6 = np.zeros_like(src)
    for k in range(1, n + 1):
        p0, m0 = cols(c0, k), cols(c0, -k)
        b1 = b1 + (p0 + m0) * g[n + k]
        b4 = b4 + (p0 + m0) * xxg[n + k]
        b2 = b2 + (p0 - m0) * xg[n + k]
        b3 = b3 + (cols(c1, k) + cols(c1, -k)) * g[n + k]
        b6 = b6 + (cols(c1, k) - cols(c1, -k)) * xg[n + k]
        b5 = b5 + (cols(c2, k) + cols(c2, -k)) * g[n + k]
    return np.stack([b3 * ig11, b2 * ig11, b1 * ig03 + b5 * ig33, b1 * ig03 + b4 * ig33, b6 * ig55], -1).astype(f32)


def border_scale(h, w):
    """Product of the row's and the column's border weight (1 beyond 5 pixels from every edge)."""
    sy = np.array([(BORDER_W[y] if y < 5 else f32(1)) * (BORDER_W[h - y - 1] if y >= h - 5 else f32(1))
                   for y in range(h)], dtype=f32)
    sx = np.array([(BORDER_W[x] if x < 5 else f32(1)) * (BORDER_W[w - x - 1] if x >= w - 5 else f32(1))
                   for x in range(w)], dtype=f32)
    return (sx[None, :] * sy[:, None]).astype(f32)


def update_matrices(R0, R1, flow):
    """cv2's FarnebackUpdateMatrices over a whole level: [H,W,5] x2, flow [H,W,2] -> M [H,W,5] (float32)."""
    h, w = flow.shape[:2]
    dx, dy = flow[..., 0].astype(f32), flow[..., 1].astype(f32)
    fx = np.arange(w, dtype=f32)[None, :] + dx
    fy = np.arange(h, dtype=f32)[:, None] + dy
    x1, y1 = np.floor(fx).astype(np.int64), np.floor(fy).astype(np.int64)
    fx, fy = (fx - x1).astype(np.float64), (fy - y1).astype(np.float64)
    inside = (x1 >= 0) & (x1 < w - 1) & (y1 >= 0) & (y1 < h - 1)
    xa, ya = np.clip(x1, 0, w - 2), np.clip(y1, 0, h - 2)
    R1d, R0d = R1.astype(np.float64), R0.astype(np.float64)
    a00, a01, a10, a11 = ((1 - fx) * (1 - fy))[..., None], (fx * (1 - fy))[..., None], ((1 - fx) * fy)[..., None], (fx * fy)[..., None]
    r = a00 * R1d[ya, xa] + a01 * R1d[ya, xa + 1] + a10 * R1d[ya + 1, xa] + a11 * R1d[ya + 1, xa + 1]
    ins = inside[..., None]
    r = np.where(ins, r, 0.0)
    r4 = np.where(inside, (R0d[..., 2] + r[..., 2]) * 0.5, R0d[..., 2])
    r5 = np.where(inside, (R0d[..., 3] + r[..., 3]) * 0.5, R0d[..., 3])
    r6 = np.where(inside, (R0d[..., 4] + r[..., 4]) * 0.25, R0d[..., 4] * 0.5)
    r2 = (R0d[..., 0] - r[..., 0]) * 0.5 + r4 * dy + r6 * dx
    r3 = (R0d[..., 1] - r[..., 1]) * 0.5 + r6 * dy + r5 * dx
    s = border_scale(h, w).astype(np.float64)
    r2, r3, r4, r5, r6 = (v * s for v in (r2, r3, r4, r5, r6))
    return np.stack([r4 * r4 + r6 * r6, (r4 + r5) * r6, r5 * r5 + r6 * r6, r4 * r2 + r6 * r3, r6 * r2 + r5 * r3],
                    -1).astype(f32)


def box_mean(M, winsize):
    """winsize x winsize mean with replicated borders, in double."""
    h, w = M.shape[:2]
    m = winsize // 2
    a = M.astype(np.float64)
    a = a[np.clip(np.arange(-m, h + m), 0, h - 1)]
    c = np.concatenate([np.zeros((1,) + a.shape[1:]), np.cumsum(a, 0)], 0)
    a = c[winsize:] - c[:-winsize]
    a = a[:, np.clip(np.arange(-m, w + m), 0, w - 1)]
    c = np.concatenate([np.zeros((a.shape[0], 1) + a.shape[2:]), np.cumsum(a, 1)], 1)
    return (c[:, winsize:] - c[:, :-winsize]) / float(winsize * winsize)


def solve_flow(Mb):
    g11, g12, g22, h1, h2 = (Mb[..., i] for i in range(5))
    idet = 1.0 / (g11 * g22 - g12 * g12 + 1e-3)
    return np.stack([(g11 * h2 - g12 * h1) * idet, (g22 * h1 - g12 * h2) * idet], -1).astype(f32)


def farneback_flow_np(prev, next, pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2):
    """cv2.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, 0)
    on uint8 [H,W] frames -> float32 [H,W,2]."""
    prev, next = np.asarray(prev), np.asarray(next)
    assert prev.shape == next.shape and prev.ndim == 2
    h, w = prev.shape
    top = pyramid_levels(h, w, pyr_scale, levels)
    flow = None
    for k in range(top, -1, -1):
        _, sigma, ksize, lh, lw = level_geometry(h, w, pyr_scale, k)
        if flow is None:
            flow = np.zeros((lh, lw, 2), dtype=f32)
        else:
            flow = (resize_linear(flow, lh, lw) * f32(1.0 / pyr_scale)).astype(f32)
        R = [poly_expansion(resize_linear(gaussian_blur(im.astype(f32), ksize, sigma), lh, lw), poly_n, poly_sigma)
             for im in (prev, next)]
        M = update_matrices(R[0], R[1], flow)
        for it in range(iterations):
            flow = solve_flow(box_mean(M, winsize))
            if it < iterations - 1:
                M = update_matrices(R[0], R[1], flow)
    return flow


def crop_window(ori_h, ori_w):
    """(y, x, h, w) of metrics.py:77-92 crop_8x8."""
    h, w = (ori_h // 32) * 32, (ori_w // 32) * 32
    while h > ori_h - 16:
        h -= 32
    while w > ori_w - 16:
        w -= 32
    return (ori_h - h) // 2, (ori_w - w) // 2, h, w


def tof_pair(flow_t, flow_o):
    y, x, h, w = crop_window(flow_t.shape[0], flow_t.shape[1])
    d = flow_t[y:y + h, x:x + w].astype(np.float64) - flow_o[y:y + h, x:x + w].astype(np.float64)
    return float(np.sqrt((d * d).sum(-1)).mean())


def tof_sequence(targets, results, cutfr=2, flow=farneback_flow_np):
    """Per-frame tOF of metrics.py:131-169 for uint8 RGB frame sequences [N,H,W,3]: one value for each of the frames
    cutfr+1 .. N-cutfr-1 (the first selected frame has none)."""
    n = len(targets)
    th, tw = targets[0].shape[:2]
    gt = [rgb_to_grey_u8(targets[i]) for i in range(cutfr, n - cutfr)]
    go = [rgb_to_grey_u8(np.asarray(results[i])[:th, :tw]) for i in range(cutfr, n - cutfr)]
    return [tof_pair(flow(gt[i - 1], gt[i]), flow(go[i - 1], go[i])) for i in range(1, len(gt))]
