"""Evaluation metrics of the reference's `metrics.py` that are plain image arithmetic -- PSNR and SSIM on the Y channel of the
uint8 result / target frames -- computed on the device (SURVEY.md 8f-3).  Same function names and argument order as the
reference (`psnr(img_true, img_pred)`, `ssim(img_true, img_pred)`, `crop_8x8(img)`, metrics.py:63-92); frames are uint8 RGB
CUDA tensors `[H,W,3]` (or `[N,H,W,3]` for the batched calls), i.e. exactly what `main.py` inference writes through `save_img`.

tOF (metrics.py:135-169) is here too: cv2's grey conversion and Farneback optical flow (flags = 0) run as the CUDA
kernels of optflow.cu, batched over all frame pairs of a scene (`farneback_flow`, `tof`).
Not here, on purpose: LPIPS / tLP (the AlexNet backbone weights of the vendored LPIPSmodels are not available) --
DESIGN.md section 6.
"""
import ctypes as C
import math

import torch

from ._ffi import call, check, lib, ptr, stream_ptr

u8, f32, f64 = torch.uint8, torch.float32, torch.float64


def crop_window(ori_h, ori_w):
    """(y, x, h, w) of the reference's crop_8x8 (metrics.py:77-92): multiples of 32, at least 16 pixels smaller, centred."""
    h, w = (ori_h // 32) * 32, (ori_w // 32) * 32
    while h > ori_h - 16:
        h -= 32
    while w > ori_w - 16:
        w -= 32
    return (ori_h - h) // 2, (ori_w - w) // 2, h, w


def crop_8x8(img):
    """Reference signature: returns (crop_img, y, x).  `img` is any [H,W,...] tensor or array; the crop is a view."""
    y, x, h, w = crop_window(img.shape[0], img.shape[1])
    if h <= 0 or w <= 0:
        raise ValueError("crop_8x8: a %dx%d frame leaves nothing after the crop" % (img.shape[0], img.shape[1]))
    return img[y:y + h, x:x + w], y, x


def _as_batch(t, name):
    if not torch.is_tensor(t) or t.dtype != u8:
        raise ValueError("%s must be a uint8 tensor (decoded RGB frames)" % name)
    if t.dim() == 3:
        t = t[None]
    if t.dim() != 4 or t.shape[-1] != 3:
        raise ValueError("%s must be [H,W,3] or [N,H,W,3], got %s" % (name, tuple(t.shape)))
    return t


def psnr_ssim_sums(img_true, img_pred, window=None, with_ssim=True):
    """Launches the two kernels and returns the raw accumulator [N,4] (float64, on device, no host sync) together with the
    window (y, x, h, w).  `window=None` means the whole common area of the two frames (the reference crops first with
    crop_8x8 and then calls psnr/ssim on the crops: pass `crop_window(...)` for that)."""
    t, p = _as_batch(img_true, "img_true"), _as_batch(img_pred, "img_pred")
    if t.shape[0] != p.shape[0]:
        raise ValueError("psnr/ssim: %d target frames but %d result frames" % (t.shape[0], p.shape[0]))
    N, tH, tW, _ = t.shape
    _, oH, oW, _ = p.shape
    if window is None:
        window = (0, 0, min(tH, oH), min(tW, oW))          # metrics.py:134-135: the result is cut to the target
    y0, x0, h, w = window
    acc = torch.empty((N, 4), device=t.device, dtype=f64)
    args = (ptr(t, u8), tH, tW, ptr(p, u8), oH, oW, N, y0, x0, h, w, ptr(acc, f64), stream_ptr())
    call("teco_metrics_psnr_y_u8", *args)
    if with_ssim:
        call("teco_metrics_ssim_y_u8", *args)
    return acc, window


def _finish(acc, window, with_ssim):
    _, _, h, w = window
    a = acc.cpu()
    ps, ss = [], []
    for n in range(a.shape[0]):
        mse = float(a[n, 0]) / (h * w)
        ps.append(20.0 * math.log10(255.0 / math.sqrt(mse)) if mse > 0.0 else float("inf"))   # numpy: 255/0 -> inf
        if with_ssim:
            ss.append(float(a[n, 3]) / ((h - 6) * (w - 6)))
    return ps, ss


def psnr(img_true, img_pred):
    """metrics.py:63-70 on one pair of uint8 RGB frames (already cropped, like the reference's call site :172)."""
    acc, win = psnr_ssim_sums(img_true, img_pred, with_ssim=False)
    return _finish(acc, win, False)[0][0]


def ssim(img_true, img_pred):
    """metrics.py:72-75 (skimage compare_ssim on Y, data_range = Y_pred.max() - Y_pred.min())."""
    acc, win = psnr_ssim_sums(img_true, img_pred)
    return _finish(acc, win, True)[1][0]


def frame_metrics(targets, results, crop=True):
    """PSNR and SSIM of N frame pairs in two launches: ([psnr_n], [ssim_n]).  crop=True applies crop_8x8 (as a window,
    without copying) exactly as the evaluation loop metrics.py:171-180 does before calling psnr/ssim."""
    t, p = _as_batch(targets, "targets"), _as_batch(results, "results")
    win = crop_window(min(t.shape[1], p.shape[1]), min(t.shape[2], p.shape[2])) if crop else None
    if crop and (win[2] <= 0 or win[3] <= 0):
        raise ValueError("crop_8x8 leaves nothing of %dx%d frames" % (t.shape[1], t.shape[2]))
    acc, win = psnr_ssim_sums(t, p, win)
    return _finish(acc, win, True)


KEYS = ("PSNR", "SSIM", "tOF")


def evaluate_sequence(targets, results, cutfr=2, keys=("PSNR", "SSIM")):
    """The reference's per-folder loop (metrics.py:124-181) for `keys` out of PSNR, SSIM and tOF: frames cutfr .. N-cutfr-1,
    crop_8x8, per-frame lists and their means (the 'FolderAvg' numbers).  tOF has one value fewer: the first selected
    frame has no predecessor."""
    bad = [k for k in keys if k not in KEYS]
    if bad:
        raise ValueError("evaluate_sequence: unknown keys %s (known: %s)" % (bad, ", ".join(KEYS)))
    t, p = _as_batch(targets, "targets"), _as_batch(results, "results")
    n = t.shape[0]
    if n - 2 * cutfr <= 0:
        raise ValueError("evaluate_sequence: %d frames with cutfr=%d leave nothing to evaluate" % (n, cutfr))
    out = {}
    if "PSNR" in keys or "SSIM" in keys:
        ps, ss = frame_metrics(t[cutfr:n - cutfr], p[cutfr:n - cutfr])
        for k, v in (("PSNR", ps), ("SSIM", ss)):
            if k in keys:
                out[k], out["FolderAvg_" + k] = v, sum(v) / len(v)
    if "tOF" in keys:
        v = tof(t, p, cutfr)
        out["tOF"], out["FolderAvg_tOF"] = v, (sum(v) / len(v) if v else float("nan"))
    return out


# ---- tOF -----------------------------------------------------------------------------------------------------------
def rgb_to_grey(frames, h=None, w=None):
    """cv2.cvtColor(frame, COLOR_RGB2GRAY) of uint8 RGB CUDA frames [H,W,3] or [N,H,W,3], bit for bit.  h, w cut each
    frame to its top-left h x w first (the reference's cut of the result to the target size, metrics.py:139-140)."""
    f = _as_batch(frames, "frames")
    N, H, W, _ = f.shape
    h, w = H if h is None else h, W if w is None else w
    g = torch.empty((N, h, w), device=f.device, dtype=u8)
    call("teco_grey_u8", ptr(f, u8), N, H, W, h, w, ptr(g, u8), stream_ptr())
    return g[0] if frames.dim() == 3 else g


def _farneback_pairs(grey, pairs, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags):
    """Flows [P,H,W,2] of the frame pairs `pairs` (list of (prev, next) indices) of grey frames [F,H,W], one batched call."""
    F, H, W = grey.shape
    P = len(pairs)
    idx = (C.c_int32 * (2 * P))(*[int(i) for pr in pairs for i in pr])
    nbytes = lib().teco_farneback_workspace_bytes(F, P, H, W, float(pyr_scale), int(levels))
    check(int(nbytes) if nbytes < 0 else 0)
    ws = torch.empty(int(nbytes), device=grey.device, dtype=u8)
    flow = torch.empty((P, H, W, 2), device=grey.device, dtype=f32)
    call("teco_farneback_flow", ptr(grey, u8), F, H, W, idx, P, float(pyr_scale), int(levels), int(winsize),
         int(iterations), int(poly_n), float(poly_sigma), int(flags), ptr(ws, u8), int(nbytes), ptr(flow, f32), stream_ptr())
    return flow


def farneback_flow(prev, next, pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2, flags=0):
    """cv2.calcOpticalFlowFarneback(prev, next, None, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma, flags)
    on the device; the defaults are the reference's call (metrics.py:147-148).  prev / next: uint8 grey CUDA frames [H,W]
    or [N,H,W] (N pairs in one batched call).  Returns float32 flows [H,W,2] or [N,H,W,2] (dx, dy).  Supported: flags = 0,
    odd winsize up to 15, poly_n 1..7; anything else raises ValueError."""
    for name, t in (("prev", prev), ("next", next)):
        if not torch.is_tensor(t) or t.dtype != u8 or not t.is_cuda:
            raise ValueError("farneback_flow: %s must be a uint8 CUDA tensor (grey frames)" % name)
    if prev.shape != next.shape or prev.dim() not in (2, 3):
        raise ValueError("farneback_flow: prev and next must both be [H,W] or [N,H,W], got %s and %s"
                         % (tuple(prev.shape), tuple(next.shape)))
    if flags != 0:
        raise ValueError("farneback_flow: only flags = 0 is implemented (OPTFLOW_FARNEBACK_GAUSSIAN and "
                         "OPTFLOW_USE_INITIAL_FLOW are not)")
    if not 1 <= poly_n <= 7:
        raise ValueError("farneback_flow: poly_n must be 1..7, got %r" % (poly_n,))
    single = prev.dim() == 2
    a, b = (prev[None], next[None]) if single else (prev, next)
    n = a.shape[0]
    grey = torch.cat([a, b]).contiguous()
    flow = _farneback_pairs(grey, [(i, n + i) for i in range(n)], pyr_scale, levels, winsize, iterations, poly_n,
                            poly_sigma, flags)
    return flow[0] if single else flow


def tof(targets, results, cutfr=2):
    """Per-frame tOF of metrics.py:131-169 for uint8 RGB CUDA sequences [N,H,W,3]: one value for each of the frames
    cutfr+1 .. N-cutfr-1.  The result is cut to the target size; the Farneback flows of all consecutive target pairs and
    all consecutive result pairs are computed in one batched call on the full grey frames; then the mean L2 norm of their
    difference inside crop_8x8."""
    t, p = _as_batch(targets, "targets"), _as_batch(results, "results")
    n, H, W, _ = t.shape
    if p.shape[0] != n:
        raise ValueError("tof: %d target frames but %d result frames" % (n, p.shape[0]))
    if p.shape[1] < H or p.shape[2] < W:
        raise ValueError("tof: result frames %dx%d are smaller than the targets %dx%d" % (p.shape[1], p.shape[2], H, W))
    y0, x0, h, w = crop_window(H, W)
    if h <= 0 or w <= 0:
        raise ValueError("tof: crop_8x8 leaves nothing of %dx%d frames" % (H, W))
    sel = n - 2 * cutfr
    if sel < 1:
        raise ValueError("tof: %d frames with cutfr=%d leave nothing to evaluate" % (n, cutfr))
    if sel < 2:
        return []
    grey = torch.cat([rgb_to_grey(t[cutfr:n - cutfr].contiguous()),
                      rgb_to_grey(p[cutfr:n - cutfr].contiguous(), H, W)])
    pairs = [(i, i + 1) for i in range(sel - 1)] + [(sel + i, sel + i + 1) for i in range(sel - 1)]
    flow = _farneback_pairs(grey, pairs, 0.5, 3, 15, 3, 5, 1.2, 0)
    P = sel - 1
    sums = torch.empty(P, device=t.device, dtype=f64)
    call("teco_tof_sums", ptr(flow[:P], f32), ptr(flow[P:], f32), P, H, W, y0, x0, h, w, ptr(sums, f64), stream_ptr())
    return [v / (h * w) for v in sums.cpu().tolist()]
