#!/usr/bin/env python
"""Mirror of the reference's metrics.py command line (flags --output / --results / --targets, metrics.py:9-12) for the two
metrics that are image arithmetic: PSNR and SSIM on the Y channel, computed on the GPU by tecogan_b200/metrics.py
(teco_metrics_psnr_y_u8 / teco_metrics_ssim_y_u8).  Same frame selection (cutfr = 2, metrics.py:117,131), same cut of the
result to the target size (:134-135), same crop_8x8 (:171-172), same per-frame / per-folder / total printout and
metrics.csv layout (:205-242) for the keys named by --keys (the reference's `keys` list, :120): PSNR and SSIM by default,
tOF on request (cv2's Farneback flow, metrics.py:135-169, as the CUDA kernels of tecogan_b200/csrc/optflow.cu).
LPIPS / tLP (AlexNet weights not available) are not part of this path: DESIGN.md section 6.

  python metrics.py --output results/metric_log/ --results results/calendar --targets HR/calendar [--keys PSNR,SSIM,tOF]
"""
import argparse
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

KEYS = ["PSNR", "SSIM"]
KNOWN_KEYS = ("PSNR", "SSIM", "tOF")
CUTFR = 2


def parse_keys(text):
    """--keys: comma-separated subset of PSNR, SSIM, tOF; kept in the reference's order (metrics.py:120)."""
    keys = [k.strip() for k in text.split(",") if k.strip()]
    bad = [k for k in keys if k not in KNOWN_KEYS]
    if bad or not keys:
        raise ValueError("--keys: unknown or empty %s (known: %s)" % (bad or text, ",".join(KNOWN_KEYS)))
    return [k for k in KNOWN_KEYS if k in keys]


def listPNGinDir(dirpath):
    """metrics.py:28-35: *.png, not starting with IB, ordered by the digits in the name."""
    names = sorted(n for n in os.listdir(dirpath) if n.endswith(".png") and not n.startswith("IB"))
    names.sort(key=lambda f: int(''.join(filter(str.isdigit, f)) or -1))
    return [os.path.join(dirpath, n) for n in names]


def read_rgb(path):
    try:
        import cv2
        return np.ascontiguousarray(cv2.imread(path)[:, :, ::-1])
    except ImportError:
        from PIL import Image
        return np.ascontiguousarray(np.asarray(Image.open(path).convert("RGB")))


def evaluate_folder(result_dir, target_dir, log=print, keys=KEYS):
    """Per-frame lists of one scene (frames cutfr .. n-cutfr-1) for `keys`."""
    if "tOF" in keys:
        return _evaluate_folder_batched(result_dir, target_dir, log, keys)
    import torch
    from tecogan_b200 import metrics as M
    result, target = listPNGinDir(result_dir), listPNGinDir(target_dir)
    lists = {k: [] for k in KEYS}
    for i in range(CUTFR, len(target) - CUTFR):
        out, tar = read_rgb(result[i]), read_rgb(target[i])
        msg = "frame %d, tar %s, out %s, " % (i, str(tar.shape), str(out.shape))
        t, o = torch.from_numpy(tar).cuda(), torch.from_numpy(out).cuda()
        ps, ss = M.frame_metrics(t, o)            # window = crop_8x8 of the common area; no cropped copies
        y, x, _, _ = M.crop_window(min(tar.shape[0], out.shape[0]), min(tar.shape[1], out.shape[1]))
        lists["PSNR"].append(ps[0])
        lists["SSIM"].append(ss[0])
        log(result[i])
        log(msg + "psnr %02.2f, ssim %02.2f, crop (%d, %d)" % (ps[0], ss[0], y, x))
    return lists


def _evaluate_folder_batched(result_dir, target_dir, log, keys):
    """The folder loaded once, tOF of all frame pairs in one batched call, PSNR / SSIM of all frames in one batch; the
    per-frame lines follow metrics.py:169-185 (tOF before psnr, none on the first frame)."""
    import torch
    from tecogan_b200 import metrics as M
    result, target = listPNGinDir(result_dir), listPNGinDir(target_dir)
    idx = list(range(CUTFR, len(target) - CUTFR))
    tars = [read_rgb(target[i]) for i in idx]
    outs = [read_rgb(result[i]) for i in idx]
    th, tw = tars[0].shape[:2]
    if any(t.shape != tars[0].shape for t in tars) or any(o.shape[0] < th or o.shape[1] < tw for o in outs):
        raise ValueError("%s: tOF needs target frames of one size and result frames at least that large" % target_dir)
    t = torch.from_numpy(np.stack(tars)).cuda()
    o = torch.from_numpy(np.stack([x[:th, :tw] for x in outs])).cuda()      # metrics.py:139-140
    tof = M.tof(t, o, cutfr=0)
    ps, ss = M.frame_metrics(t, o) if ("PSNR" in keys or "SSIM" in keys) else ([], [])
    y, x, _, _ = M.crop_window(th, tw)
    lists = {"PSNR": ps, "SSIM": ss, "tOF": tof}
    for j, i in enumerate(idx):
        msg = "frame %d, tar %s, out %s, " % (i, str(tars[j].shape), str(outs[j].shape))
        if j > 0:
            msg += "tOF %02.2f, " % tof[j - 1]
        parts = []
        if "PSNR" in keys:
            parts.append("psnr %02.2f" % ps[j])
        if "SSIM" in keys:
            parts.append("ssim %02.2f" % ss[j])
        log(result[i])
        log(msg + ", ".join(parts + ["crop (%d, %d)" % (y, x)]))
    return {k: lists[k] for k in keys}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--output", required=True, help="the path of output directory")
    ap.add_argument("--results", required=True, help="the list of paths of result directory")
    ap.add_argument("--targets", required=True, help="the list of paths of target directory")
    ap.add_argument("--keys", default="PSNR,SSIM", help="comma-separated metrics out of PSNR, SSIM, tOF")
    F = ap.parse_args(argv)
    try:
        keys = parse_keys(F.keys)
    except ValueError as e:
        ap.error(str(e))
    import pandas as pd
    os.makedirs(F.output, exist_ok=True)
    logf = open(os.path.join(F.output, "metricsfile.txt"), "a")

    def log(m):
        print(m)
        logf.write(m + "\n")
    result_list, target_list = F.results.split(','), F.targets.split(',')
    folder_n = len(result_list)
    sum_d = {"FrameAvg_" + k: 0.0 for k in keys}
    len_d = {k: 0 for k in keys}
    avg_d = {"Avg_" + k: [] for k in keys}
    folder_d = {"FolderAvg_" + k: 0.0 for k in keys}
    csv = os.path.join(F.output, "metrics.csv")
    for fi in range(folder_n):
        lists = evaluate_folder(result_list[fi], target_list[fi], log, keys)
        pd_dict = {}
        for k in keys:
            cur = np.float32(lists[k])
            pd_dict["%s_%02d" % (k, fi)] = pd.Series(cur)
            mean = cur.sum() / cur.shape[0]
            log("%s_%02d, max %02.4f, min %02.4f, avg %02.4f" % (k, fi, cur.max(), cur.min(), mean))
            avg_d["Avg_" + k].append(mean)
            sum_d["FrameAvg_" + k] += cur.sum()
            len_d[k] += cur.shape[0]
            folder_d["FolderAvg_" + k] += mean
        pd.DataFrame(pd_dict).to_csv(csv, mode='w' if fi == 0 else 'a')
    for k in keys:
        sum_d["FrameAvg_" + k] = pd.Series([sum_d["FrameAvg_" + k] / len_d[k]])
        folder_d["FolderAvg_" + k] = pd.Series([folder_d["FolderAvg_" + k] / folder_n])
        avg_d["Avg_" + k] = pd.Series(np.float32(avg_d["Avg_" + k]))
        log("%s, total frame %d, total avg %02.4f, folder avg %02.4f" % (k, len_d[k], sum_d["FrameAvg_" + k][0], folder_d["FolderAvg_" + k][0]))
    for d in (avg_d, folder_d, sum_d):
        pd.DataFrame(d).to_csv(csv, mode='a')
    log("Finished.")
    logf.close()
    return {k: float(sum_d["FrameAvg_" + k][0]) for k in keys}


if __name__ == "__main__":
    main()
