#!/usr/bin/env python
"""Time tecogan_b200.metrics.tof on one 41-frame 576x720 scene (Vid4 calendar size; frames derived as in
tests/golden/make_golden_tof.py, the 6 calendar frames repeated) with CUDA events: warm-up, then the median of --reps.
Reports ms per scene, flows/s, the bytes this script's model of each kernel moves, the GB/s that implies, its fraction of
the copy bandwidth in MEASURED_PEAKS.json (when present), whether the working set exceeds the 126 MB L2, the card's name
and power limit, and cv2's CPU time for the same flows when cv2 is importable.  Prints one JSON line.

  python tools/bench_tof.py [--reps 20] [--cv2-flows 4]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
L2_BYTES = 126 * 2 ** 20


def traffic_model(F, P, H, W, levels=3, s=0.5, iters=3, winsize=15, poly_n=5):
    """Bytes each kernel reads + writes from DRAM/L2, counting each tensor element once per launch (halos ignored)."""
    from tests.golden import tof_ref as T
    top = T.pyramid_levels(H, W, s, levels)
    b = {"grey_u8": 2 * F * H * W * 3 + 2 * F * H * W}            # 2F RGB frames in, 2F grey frames out
    tot = {"level_rows": 0, "level_poly": 0, "flow_init": 0, "flow_iter": 0}
    for k in range(top, -1, -1):
        _, _, _, lh, lw = T.level_geometry(H, W, s, k)
        a = lh * lw
        tot["level_rows"] += 2 * F * (H * W + 4 * H * lw)
        tot["level_poly"] += 2 * F * (4 * H * lw + 20 * a)
        tot["flow_init"] += P * (8 * a + 40 * a + 20 * a)          # coarse flow (upper bound), R0 + R1, M out
        tot["flow_iter"] += P * (iters * (20 * a + 8 * a) + (iters - 1) * (40 * a + 20 * a))
    b.update(tot)
    b["tof_sums"] = P // 2 * 2 * 8 * H * W
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=41)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cv2-flows", type=int, default=4, help="flows to time with cv2 on the CPU (0: skip)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    A = ap.parse_args()
    import torch
    from tecogan_b200 import metrics as M
    from tests.golden import make_golden_tof as G
    if not torch.cuda.is_available():
        raise SystemExit("bench_tof: needs a CUDA device")
    tg, rs = G.vid4_sequence()
    idx = [i % len(tg) if (i // len(tg)) % 2 == 0 else len(tg) - 1 - i % len(tg) for i in range(A.frames)]
    t, r = torch.from_numpy(tg[idx]).cuda(), torch.from_numpy(rs[idx]).cuda()
    n, H, W, _ = t.shape
    sel = n - 4                                       # cutfr = 2
    P = 2 * (sel - 1)
    for _ in range(A.warmup):
        M.tof(t, r)
    torch.cuda.synchronize()
    times = []
    for _ in range(A.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        M.tof(t, r)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    model = traffic_model(sel, P, H, W)
    total = sum(model.values())
    ws = int(M.lib().teco_farneback_workspace_bytes(2 * sel, P, H, W, 0.5, 3))
    res = {"what": "tof() per 41-frame scene", "frames": n, "size": [H, W], "flows": P, "ms_per_scene": round(ms, 3),
           "ms_min": round(min(times), 3), "ms_max": round(max(times), 3), "flows_per_s": round(P / ms * 1e3, 1),
           "model_bytes": model, "model_GB_per_s": round(total / ms / 1e6, 1), "workspace_bytes": ws,
           "working_set_exceeds_L2": ws > L2_BYTES}
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks):
        pk = json.load(open(peaks))
        bw = next((pk[k] for k in ("copy_GBps", "copy_bw_GBps", "dram_copy_GBps", "hbm_copy_GBps") if k in pk), None)
        res["copy_GBps"] = bw
        res["fraction_of_copy_bw"] = round(total / ms / 1e6 / bw, 3) if bw else None
    else:
        res["fraction_of_copy_bw"] = "MEASURED_PEAKS.json not present"
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        res["gpu"] = q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        res["gpu"] = torch.cuda.get_device_name()
    if A.cv2_flows > 0:
        try:
            import cv2
            from tests.golden import tof_ref as T
            g = [T.rgb_to_grey_u8(f) for f in tg]
            t0 = time.perf_counter()
            for i in range(A.cv2_flows):
                cv2.calcOpticalFlowFarneback(g[i % 5], g[i % 5 + 1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
            per = (time.perf_counter() - t0) / A.cv2_flows
            res["cv2_cpu_ms_per_flow"] = round(per * 1e3, 1)
            res["cv2_cpu_s_per_scene"] = round(per * P, 2)
        except ImportError:
            res["cv2_cpu_ms_per_flow"] = "cv2 not importable"
    line = json.dumps(res)
    print(line)
    if A.out:
        os.makedirs(os.path.dirname(os.path.abspath(A.out)), exist_ok=True)
        open(A.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
