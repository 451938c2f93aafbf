"""Generate tests/golden/tof.npz: cv2's grey conversion, Farneback flows and tOF values (the reference's metrics.py:135-169)
on deterministic inputs, for the CUDA kernels of tecogan_b200/csrc/optflow.cu and the numpy restatement tof_ref.py.

Inputs are the calendar LR frames of tests/golden/calendar_lr.npz (144x180, three pyramid scales) and a 576x720 (Vid4
size, four scales) sequence derived from them with numpy only (`vid4_sequence`), so any host re-derives the same bytes;
the file stores their SHA-256.  Needs cv2 (the version is recorded in the file):
    python tests/golden/make_golden_tof.py
"""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ARGS = (0.5, 3, 15, 3, 5, 1.2)                   # pyr_scale, levels, winsize, iterations, poly_n, poly_sigma
CUSTOM_ARGS = (0.6, 1, 9, 2, 5, 1.5)
VID4_FRAMES = 6


def calendar():
    return np.load(os.path.join(HERE, "calendar_lr.npz"))["full_u8"]


def _upscale4(img, dy=0.0, dx=0.0):
    """float64 bilinear 4x upscale with half-pixel centres and clamped edges, sampled at a shift of (dy, dx) output pixels."""
    h, w = img.shape[:2]

    def taps(n_src, n_dst, shift):
        s = np.clip((np.arange(n_dst) + 0.5 + shift) / 4.0 - 0.5, 0, n_src - 1)
        i0 = np.floor(s).astype(np.int64)
        return i0, np.minimum(i0 + 1, n_src - 1), s - i0

    y0, y1, ay = taps(h, 4 * h, dy)
    x0, x1, ax = taps(w, 4 * w, dx)
    a = img.astype(np.float64)
    t = a[:, x0] * (1 - ax)[None, :, None] + a[:, x1] * ax[None, :, None]
    return t[y0] * (1 - ay)[:, None, None] + t[y1] * ay[:, None, None]


def vid4_sequence():
    """(targets, results) uint8 [6,576,720,3]: targets are the calendar frames upscaled 4x; results are the same frames
    sampled 0.35 px right and 0.2 px down, plus seeded integer noise in [-3, 3]."""
    cal = calendar()[:VID4_FRAMES]
    rng = np.random.RandomState(2024)
    tg = np.stack([np.clip(np.rint(_upscale4(f)), 0, 255) for f in cal]).astype(np.uint8)
    rs = np.stack([_upscale4(f, 0.2, 0.35) for f in cal]) + rng.randint(-3, 4, size=tg.shape)
    return tg, np.clip(np.rint(rs), 0, 255).astype(np.uint8)


def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def small_cases(grey):
    """name -> (prev, next, args) of the 144x180 cases."""
    g = grey
    return {
        "pair01": (g[0], g[1], REF_ARGS),
        "pair23": (g[2], g[3], REF_ARGS),
        "ragged141x178": (g[4][:141, :178], g[5][:141, :178], REF_ARGS),
        "single63x100": (g[5][40:103, 30:130], g[6][40:103, 30:130], REF_ARGS),
        "custom12": (g[1], g[2], CUSTOM_ARGS),
    }


def main():
    import cv2

    def grey(a):
        return cv2.cvtColor(np.ascontiguousarray(a), cv2.COLOR_RGB2GRAY)

    def flow(a, b, args):
        return cv2.calcOpticalFlowFarneback(np.ascontiguousarray(a), np.ascontiguousarray(b), None, *args, 0)

    out = {"cv2_version": np.array(cv2.__version__)}
    rng = np.random.RandomState(7)
    rgb = rng.randint(0, 256, size=(1, 8192, 3)).astype(np.uint8)
    out["grey_rgb"], out["grey_cv2"] = rgb[0], grey(rgb)[0]

    cal_grey = np.stack([grey(f) for f in calendar()])
    for name, (a, b, args) in small_cases(cal_grey).items():
        out["flow_" + name] = flow(a, b, args)

    tg, rs = vid4_sequence()
    out["vid4_sha256"] = np.array(sha256(tg, rs))
    gt, go = [grey(f) for f in tg], [grey(f) for f in rs]
    tofs = []
    for i in range(1, VID4_FRAMES):                 # metrics.py:143-169 with cutfr = 0
        ft, fo = flow(gt[i - 1], gt[i], REF_ARGS), flow(go[i - 1], go[i], REF_ARGS)
        y, x, h, w = 16, 8, 544, 704                 # crop_8x8 of 576x720
        d = np.absolute(ft[y:y + h, x:x + w] - fo[y:y + h, x:x + w])
        tofs.append(np.sqrt(np.sum(d * d, axis=-1)).mean())
        if i == 1:
            out["vid4_flow01_sub8"] = ft[::8, ::8]
    out["vid4_tof"] = np.array(tofs, dtype=np.float64)
    path = os.path.join(HERE, "tof.npz")
    np.savez_compressed(path, **out)
    print("wrote %s (%d bytes), cv2 %s, tOF %s" % (path, os.path.getsize(path), cv2.__version__, out["vid4_tof"]))


if __name__ == "__main__":
    main()
