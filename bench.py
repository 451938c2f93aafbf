#!/usr/bin/env python
"""bench.py -- benchmark of the TecoGAN recurrent video-SR hot path on B200.

Headline (BASELINE.json `metric`: "HR frames/sec (4x SR, 10-frame clips)", north_star: "synthetic 32x32 -> 128x128
x10-frame clips at 1/2/4/8 GPUs"): every rank owns CLIPS independent synthetic clips of 10 LR frames 32x32 and runs them
in lock-step through the full recurrence (fnet on every consecutive pair -> upscale_four/warp/space-to-depth feedback ->
generator_F, 16 res-blocks, seeded random weights), bf16 tcgen05 convolutions, one CUDA-graph replay per clip batch.
A "step" = one batch of CLIPS clips x 10 frames per rank.
  value = HR frames of all ranks / max-over-ranks device time, LR clips resident in HBM;
  e2e   = the same through the public ClipEngine API from pinned HOST clips: H2D of every LR clip and D2H of every uint8
          HR frame inside the timed region (copies overlap the next batch's compute on copy streams).
Extra objects in the same JSON line (each timed the same way: CUDA events, max over ranks):
  configs1_single_clip  BASELINE configs[1]: one 120-frame 128x128 -> 512x512 clip per rank (latency-bound streaming case)
  config5_sweep         BASELINE configs[4]: 256x256 -> 1024x1024, 30-frame clips, b = 1/2/4 clips per rank
  train                 BASELINE configs[2]/[3]: FRVSR (case 4) and TecoGAN (case 3) training steps, B=4 clips per rank,
                        bf16 tensor-core convolutions, ONE NCCL all-reduce of the flat gradient bucket per step when N > 1

  python bench.py --gpus 1 --steps 10 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference        # CPU restatement of the reference (oracle/) on the host cores, same workload
  python bench.py --dump-outputs DIR      # also save what the last timed step returned (seeded clip sample) as DIR/*.npy
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark writes nothing into the source tree, which may be read-only
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

LR = 32                      # metric config: 32x32 LR -> 128x128 HR
CLIP_T = 10                  # frames per clip
NUM_RESBLOCK = 16
DEFAULT_CLIPS = 296          # clips per GPU = 2 x 148 SMs (each clip is 4 tiles of 16x16 LR pixels per layer)
# algorithmic MACs per LR pixel (SURVEY.md Appendix B): generator N=16, fnet
GEN_MACS, FNET_MACS = 1420992, 126720
WORKLOAD = ("metric config: 4x SR inference of synthetic 10-frame clips 32x32->128x128, %d clips per GPU in lock-step "
            "(generator N=16 + fnet, full recurrence)")
DUMP_CLIPS = 16              # --dump-outputs: 16 of the clips, 10 x 16 HR frames as float32 = 31 MB (all 296 would be 582 MB)


def clip_flop(T=CLIP_T, px=LR * LR):
    """Algorithmic FLOPs of one T-frame clip: generator on every frame, fnet on every consecutive pair."""
    return 2.0 * px * (GEN_MACS * T + FNET_MACS * (T - 1))


def synthetic_clips(T, B, h, w, seed):
    """[T,B,h,w,3] smooth-noise videos in [0,1], each translated by (1.5,-0.75) px/frame (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed)
    m = 8 + int(1.5 * T) + 2
    base = torch.rand(B, 3, (h + 2 * m) // 4 + 2, (w + 2 * m) // 4 + 2, generator=g)
    big = torch.nn.functional.interpolate(base, scale_factor=4, mode="bicubic", align_corners=False).clamp(0, 1)
    out = torch.empty(T, B, h, w, 3)
    for t in range(T):
        oy, ox = m + 1.5 * t, m + 0.75 * (T - t)
        y0, x0 = int(oy), int(ox)
        fy, fx = oy - y0, ox - x0
        p = big[:, :, y0:y0 + h + 1, x0:x0 + w + 1]
        fr = ((1 - fy) * (1 - fx) * p[:, :, :h, :w] + (1 - fy) * fx * p[:, :, :h, 1:w + 1]
              + fy * (1 - fx) * p[:, :, 1:h + 1, :w] + fy * fx * p[:, :, 1:h + 1, 1:w + 1])
        out[t] = fr.permute(0, 2, 3, 1)
    return out.contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        load = [s for s, p in zip(sm, pw) if p > 300.0] or sm     # samples taken while the GPU was actually busy
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


def host_threads():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota and by 64."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        pass
    return max(1, min(n, 64))


class CpuReference:
    """The CPU restatement of the reference path (oracle/, kind 'port'; the TensorFlow-1.x reference cannot be installed):
    the same recurrence (main.py:253-268 order per frame; frame 0 from pre_warp = 0) on `clips` of the same synthetic
    10-frame 32x32 clips, all clips as one batch, fp32."""

    def __init__(self, threads):
        from oracle import teco_oracle as O
        from tecogan_b200.init_params import xavier_params
        self.O = O
        torch.set_num_threads(threads)
        pw = xavier_params(1234, NUM_RESBLOCK)          # the same seeded weights the CUDA arm runs (TF variable names)
        self.pg = {k: v for k, v in pw.items() if k.startswith("generator/")}
        self.pf = {k: v for k, v in pw.items() if k.startswith("fnet/")}

    def run(self, clip):                                # clip [T,B,h,w,3]
        O = self.O
        T, B, h, w, _ = clip.shape
        with torch.no_grad():
            pre_gen = torch.zeros(B, 4 * h, 4 * w, 3)
            pre_warp = torch.zeros(B, 4 * h, 4 * w, 3)
            pre_inputs = None
            for t in range(T):
                cur = clip[t]
                if t != 0:
                    flow = O.upscale_four(O.fnet(self.pf, torch.cat((pre_inputs, cur), dim=-1)) * 4.0)
                    pre_warp = O.dense_image_warp(pre_gen, flow)
                out = O.generator_F(self.pg, torch.cat((cur, O.space_to_depth4(pre_warp)), dim=-1), NUM_RESBLOCK)
                pre_inputs, pre_gen = cur, O.deprocess(out)
        return pre_gen

    def timed(self, clips, samples, warm=1):
        clip = synthetic_clips(CLIP_T, clips, LR, LR, seed=0)
        for _ in range(warm):
            self.run(clip[:, :max(1, clips // 4)])
        ts = []
        for _ in range(samples):
            t0 = time.perf_counter()
            self.run(clip)
            ts.append(time.perf_counter() - t0)
        return ts


def cpu_sample_size(ref, budget_s):
    """Clips per CPU sample so that one sample costs about `budget_s` seconds (calibrated on 4 clips)."""
    t = ref.timed(4, 1)[0]
    return int(max(4, min(64, 4 * budget_s / max(t, 1e-3))))


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = host_threads()
    ref = CpuReference(cores)
    steps = max(1, args.steps)
    # bounded: the whole --steps K --warmup W run stays within ~2 minutes
    clips = cpu_sample_size(ref, min(8.0, 100.0 / (steps + max(1, args.warmup))))
    ref.timed(clips, max(1, min(args.warmup, 2)))
    ts = ref.timed(clips, steps, warm=0)
    total = float(sum(ts))
    v = clips * CLIP_T * steps / total
    line = {
        "impl": "reference", "metric": "HR frames/sec (4x SR, 10-frame clips)", "value": v, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1000.0 * total / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % args.clips, "num_resblock": NUM_RESBLOCK, "clips_per_gpu": args.clips,
                   "frames_per_clip": CLIP_T},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "each step = %d of the %d clips (x %d frames, 32x32->128x128), full recurrence, torch-CPU fp32 "
                                   "restatement of the reference (TensorFlow 1.x is not installable here)" % (clips, args.clips, CLIP_T)},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips", type=int, default=int(os.environ.get("TECO_BENCH_CLIPS", DEFAULT_CLIPS)), help="clips per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip configs[1], the config-5 sweep and the training steps")
    ap.add_argument("--train-steps", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save what the headline path returned in its last step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from tecogan_b200 import _ffi, config, variables as V
    from tecogan_b200 import kernels as K
    from tecogan_b200.engine import ClipEngine, InferenceEngine
    from tecogan_b200.init_params import xavier_params   # product-side seeded init; oracle/ is only the cpu_baseline leg

    # count our C-ABI kernel launches (every call launches exactly one kernel of libteco.so)
    counter = {"n": 0}
    orig_call = _ffi.call

    def counting_call(name, *a):
        counter["n"] += 1
        return orig_call(name, *a)
    _ffi.call = counting_call
    import tecogan_b200.kernels, tecogan_b200.engine, tecogan_b200.tc_nets
    for m in (tecogan_b200.kernels, tecogan_b200.engine, tecogan_b200.tc_nets):
        m.call = counting_call

    def note(msg):
        if rank == 0:
            print("[bench] " + msg, file=sys.stderr, flush=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def ev_time(fn):
        """Device time of fn() in ms on the current stream, synchronised on both sides."""
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def max_over_ranks(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_tf_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 1.59 PFLOP/s / 6.65 TB/s"

    config.set_precision("bf16")
    st = V.set_default_store(V.VariableStore())
    st.load(xavier_params(1234, NUM_RESBLOCK))

    # ================================================================== headline: metric config
    B = args.clips
    eng = ClipEngine(LR, LR, CLIP_T, NUM_RESBLOCK, batch=B)
    host_in = synthetic_clips(CLIP_T, B, LR, LR, seed=rank).pin_memory()
    eng.clip_in.copy_(host_in)
    c0 = counter["n"]
    eng.replay()                                     # eager warm-up + graph capture
    torch.cuda.synchronize()
    launches_per_step = (counter["n"] - c0) // 2     # the body ran twice (eager, then capture)
    note("clip engine ready: %d clips x %d frames per step, %d kernel launches per step" % (B, CLIP_T, launches_per_step))

    # e2e plumbing: copy streams + double buffers so that H2D of batch k+1 and D2H of batch k-1 overlap batch k
    cin, cout = torch.cuda.Stream(), torch.cuda.Stream()
    lr_dev = [torch.empty_like(eng.clip_in) for _ in range(2)]
    u8_dev = [torch.empty_like(eng.clip_u8) for _ in range(2)]
    host_out = [torch.empty(eng.clip_u8.shape, dtype=torch.uint8).pin_memory() for _ in range(2)]

    def run_resident(steps):
        for _ in range(steps):
            eng.replay()

    def run_e2e(steps):
        main_s = torch.cuda.current_stream()
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_cons = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        cin.wait_stream(main_s)
        cout.wait_stream(main_s)
        with torch.cuda.stream(cin):
            lr_dev[0].copy_(host_in, non_blocking=True)
            ev_in[0].record(cin)
        for k in range(steps):
            b = k & 1
            if k + 1 < steps:
                with torch.cuda.stream(cin):
                    if k >= 1:
                        cin.wait_event(ev_cons[b ^ 1])            # batch k-1 has left this staging buffer
                    lr_dev[b ^ 1].copy_(host_in, non_blocking=True)   # every batch is uploaded from pinned host memory
                    ev_in[b ^ 1].record(cin)
            main_s.wait_event(ev_in[b])
            eng.clip_in.copy_(lr_dev[b])
            ev_cons[b].record(main_s)
            eng.replay()
            if k >= 2:
                main_s.wait_event(ev_out[b])                      # the D2H of batch k-2 has drained this buffer
            u8_dev[b].copy_(eng.clip_u8)
            ev_done[b].record(main_s)
            with torch.cuda.stream(cout):
                cout.wait_event(ev_done[b])
                host_out[b].copy_(u8_dev[b], non_blocking=True)   # every uint8 HR frame goes back to pinned host memory
                ev_out[b].record(cout)
        main_s.wait_stream(cout)

    for _ in range(args.warmup):
        eng.replay()
    run_e2e(2)
    torch.cuda.synchronize()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    ms_res = ev_time(lambda: run_resident(args.steps))
    barrier()
    wall_res = time.perf_counter() - wall0
    ms_e2e = ev_time(lambda: run_e2e(args.steps))
    barrier()
    clocks = sampler.stop()
    note("headline: resident %.2f ms/step, e2e %.2f ms/step" % (ms_res / args.steps, ms_e2e / args.steps))
    # the e2e leg really moved the bytes: spot-check the host copy against the device result of the last batch
    assert torch.equal(host_out[(args.steps - 1) & 1][-1, 0], eng.clip_u8[-1, 0].cpu()), "e2e: host frames differ from device frames"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, host_out[(args.steps - 1) & 1], eng.out01)
        note("outputs of the last timed step written to %s" % args.dump_outputs)

    # --- dominant kernel: the generator trunk (input conv + 16 residual blocks = 33 layers of 3x3 64->64) on the whole clip
    # batch [B,32,32,64] -- ONE launch of conv3x3_lin_kernel (kx-fused N=192 MMAs, CTA-local clips) -- timed alone (graph replay).
    g = eng.gen
    reps = 16

    def trunk_pairs(gp, n):
        a1, a2 = gp.l_res[0]
        for _ in range(n // 2):
            K.conv3x3_tc(gp.a, a1.wpk, a1.bias, gp.b, cout=64, act=1)
            K.conv3x3_tc(gp.b, a2.wpk, a2.bias, gp.a, cout=64, act=0, res=gp.a)

    def graph_us(fn, n_inside, replays=5):
        fn()
        torch.cuda.synchronize()
        kg = torch.cuda.CUDAGraph()          # graph replay: device time of the launches, not ctypes/Python overhead
        with torch.cuda.graph(kg):
            fn()
        kg.replay()
        return ev_time(lambda: [kg.replay() for _ in range(replays)]) * 1000.0 / (replays * n_inside)

    def kernel_us(gp, n):
        return graph_us(lambda: trunk_pairs(gp, n), n)
    layer_flop = 2.0 * B * LR * LR * 576 * 64
    per_layer_us = kernel_us(g, reps)                     # the per-layer persistent kernel (N = 64 MMAs), for comparison
    if getattr(g, "lin", False):
        n_layers = len(g.trunk_plan)
        k_us = graph_us(lambda: [K.conv3x3_lin_chain(g.x_in, g.a, g.b, g.trunk_w, g.trunk_b, g.trunk_plan) for _ in range(2)], 2)
        k_flop = layer_flop * n_layers
        k_name = ("conv3x3_lin_kernel (generator trunk: %d layers of 3x3 64->64 on the clip batch [%d,32,32,64] in one launch; "
                  "kx-fused N=192 tcgen05.mma, x-shift by warp shuffles)" % (n_layers, B))
    else:
        k_us, k_flop = per_layer_us, layer_flop
        k_name = "conv3x3_tc_kernel (3x3 64->64 res-block layer on the clip batch [%d,32,32,64])" % B

    # --- HBM-bound kernel of the path: fused upscale_four + warp + space-to-depth feedback on a batch larger than L2
    # (32 clips of 256x256 LR -> 1024x1024 HR: 403 MB read + 201 MB written), algorithmic 18.5 B per HR pixel
    wn, wh = 32, 256
    w_pre = torch.rand(wn, 4 * wh, 4 * wh, 3, device=dev)
    yy, xx = torch.meshgrid(torch.linspace(0, 6.28, wh, device=dev), torch.linspace(0, 6.28, wh, device=dev), indexing="ij")
    w_flow = torch.stack((1.5 + 0.5 * torch.sin(yy + xx), -0.75 + 0.5 * torch.cos(yy - xx)), dim=-1).expand(wn, wh, wh, 2).contiguous()
    w_dst = torch.zeros(wn, wh, wh, 64, device=dev, dtype=torch.bfloat16)
    def warp_time(flow):
        for _ in range(3):
            K.warp_s2d_fused(w_pre, flow, w_dst, 0)
        return ev_time(lambda: [K.warp_s2d_fused(w_pre, flow, w_dst, 0) for _ in range(5)]) * 1000.0 / 5
    warp_us = warp_time(w_flow)
    # the same with a rough motion field: +-1.5 LR pixels of independent noise per flow sample (source windows 12 HR pixels
    # wider and taller than the tile, staged per half tile)
    w_rough = (w_flow + 3.0 * (torch.rand(wh, wh, 2, device=dev) - 0.5)).contiguous()
    warp_rough_us = warp_time(w_rough)
    warp_bytes = wn * (4 * wh) * (4 * wh) * 18.5
    del w_pre, w_flow, w_rough, w_dst

    ms_res, ms_e2e = max_over_ranks([ms_res, ms_e2e])
    frames_total = B * CLIP_T * args.steps * world
    value = frames_total / (ms_res / 1000.0)
    e2e = frames_total / (ms_e2e / 1000.0)
    ach_tf = k_flop / (k_us * 1e-6) / 1e12
    whole_tf = clip_flop() * B * args.steps / (ms_res / 1000.0) / 1e12      # per GPU (ms_res is the max over ranks)

    line = {
        "metric": "HR frames/sec (4x SR, 10-frame clips)", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD % B, "num_resblock": NUM_RESBLOCK, "clips_per_gpu": B, "frames_per_clip": CLIP_T,
                   "frames_per_step": B * CLIP_T,
                   "l2": "no flush needed: one step streams %.0f MB of activations (64-channel HR buffer alone %.0f MB), larger "
                         "than the 126 MB L2" % (B * 128 * 128 * (128 + 128 + 24) / 1e6, B * 128 * 128 * 128 / 1e6),
                   "weights": "seeded random init (xavier, res-block/output weights x0.5)", "cuda_graph": True,
                   "fnet": "all consecutive pairs of a clip first (lib/Teco.py:102-117 order), then the generator recurrence"},
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(host_in.numel() * 4),
                "d2h_bytes_per_step": int(eng.clip_u8.numel()), "result": "uint8 HR frames (save_img quantisation)",
                "api": "tecogan_b200.engine.ClipEngine, pinned host clips in, pinned host uint8 frames out, copies on "
                       "separate streams overlapping the next batch"},
        "gpu_launches": int(launches_per_step * args.steps),
        "roofline": {"bound": "tensor", "kernel": k_name,
                     "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf,
                     "peak_source": peak_src + ", burst bf16 (kernel timed alone)", "us_per_launch": k_us,
                     "flop_per_launch": k_flop, "traffic": _traffic("r02_conv_lin_traffic.json"),
                     "per_layer_kernel": {"kernel": "conv3x3_tc_kernel (same layers, one launch each, N=64 MMAs)", "us_per_layer": per_layer_us,
                                          "achieved": layer_flop / (per_layer_us * 1e-6) / 1e12, "frac": layer_flop / (per_layer_us * 1e-6) / 1e12 / peak_tf},
                     "whole_step": {"algorithmic_gflop_per_clip": clip_flop() / 1e9, "achieved_tflops": whole_tf,
                                    "frac_of_sustained": whole_tf / peak_tf_sus}},
        "roofline_hbm": {"bound": "hbm", "kernel": "warp_s2d_v2_kernel behind teco_warp_s2d_fused (upscale_four + dense_image_warp + "
                                                     "space_to_depth), 32 x 1024x1024 HR frames, smooth motion field, working set 604 MB > L2",
                         "achieved": warp_bytes / (warp_us * 1e-6) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                         "frac": warp_bytes / (warp_us * 1e-6) / 1e9 / peak_gbs, "us_per_launch": warp_us,
                         "algorithmic_bytes_per_launch": warp_bytes, "traffic": _traffic("r02_warp_v2_traffic.json"),
                         "rough_motion": {"us_per_launch": warp_rough_us, "achieved": warp_bytes / (warp_rough_us * 1e-6) / 1e9,
                                          "frac": warp_bytes / (warp_rough_us * 1e-6) / 1e9 / peak_gbs},
                         "peak_source": peak_src + ", copy bandwidth"},
        "wall_s_resident_leg": wall_res,
    }
    del eng, lr_dev, u8_dev, host_out
    torch.cuda.empty_cache()

    if not args.headline_only:
        # ============================================================== configs[1]: one 120-frame 128x128 clip per rank
        F1, H1 = 120, 128
        e1 = InferenceEngine(H1, H1, NUM_RESBLOCK, batch=1, use_graph=True)
        clip_host = synthetic_clips(F1, 1, H1, H1, seed=rank)[:, 0].contiguous().pin_memory()
        clip_dev = clip_host.to(dev)
        out_host = torch.empty((F1, 4 * H1, 4 * H1, 3), dtype=torch.uint8).pin_memory()

        def clip_resident():
            e1.reset()
            for t in range(F1):                                      # look-ahead: fnet(t, t+1) overlaps generator(t)
                e1.step(clip_dev[t], next_lr=clip_dev[t + 1] if t + 1 < F1 else None)

        def clip_e2e():
            e1.reset()
            for t in range(F1):
                e1.step(clip_host[t], next_lr=clip_host[t + 1] if t + 1 < F1 else None)
                out_host[t].copy_(e1.out_u8[0], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for _ in range(3):
            clip_resident()
        clip_e2e()
        n1 = 3
        barrier()
        t_res = sum(ev_time(clip_resident) for _ in range(n1))
        t_e2e = sum(ev_time(clip_e2e) for _ in range(n1))
        k1_us = kernel_us(e1.gen, 64)
        t_res, t_e2e = max_over_ranks([t_res, t_e2e])
        k1_flop = 2.0 * H1 * H1 * 576 * 64
        line["configs1_single_clip"] = {
            "workload": "configs[1]: 4x SR inference 128x128->512x512, one 120-frame synthetic clip per GPU (streaming, batch 1)",
            "value": F1 * n1 * world / (t_res / 1000.0), "e2e": F1 * n1 * world / (t_e2e / 1000.0), "unit": "frames/s",
            "ms_per_clip": t_res / n1, "fnet_lookahead": True,
            "roofline": {"bound": "tensor", "kernel": "conv3x3_tc_kernel (3x3 64->64 @128x128, one tile per CTA)",
                         "achieved": k1_flop / (k1_us * 1e-6) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": k1_flop / (k1_us * 1e-6) / 1e12 / peak_tf, "us_per_launch": k1_us}}
        note("configs[1]: %.1f ms/clip resident" % (t_res / n1))
        del e1, clip_dev
        torch.cuda.empty_cache()

        # ============================================================== configs[4]: 256x256 -> 1024x1024, 30 frames, b = 1/2/4
        sweep = {}
        for b in (1, 2, 4):
            e5 = ClipEngine(256, 256, 30, NUM_RESBLOCK, batch=b)
            e5.clip_in.copy_(synthetic_clips(30, b, 256, 256, seed=rank + 7))
            for _ in range(3):
                e5.replay()
            barrier()
            t5 = max_over_ranks([sum(ev_time(e5.replay) for _ in range(2))])[0]
            fps = 30 * b * 2 * world / (t5 / 1000.0)
            gflop = 2e-9 * 256 * 256 * (GEN_MACS + FNET_MACS)
            sweep["b%d" % b] = {"value": fps, "unit": "frames/s", "ms_per_clip_batch": t5 / 2,
                                "frac_of_sustained_bf16": gflop * fps / world / 1e3 / peak_tf_sus}
            note("config 5 b=%d: %.1f frames/s" % (b, fps))
            del e5
            torch.cuda.empty_cache()
        line["config5_sweep"] = {"workload": "configs[4]: 4x SR 256x256->1024x1024, 30-frame clips, b clips per GPU in lock-step",
                                 "algorithmic_gflop_per_frame": 2e-9 * 256 * 256 * (GEN_MACS + FNET_MACS), **sweep}

        # ============================================================== training: configs[2] (FRVSR) and configs[3] (TecoGAN)
        line["train"] = bench_train(args, rank, world, dev, dist, ev_time, max_over_ranks, note, peak_tf_sus)

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            cores = host_threads()
            ref = CpuReference(cores)
            clips = cpu_sample_size(ref, 6.0)
            ts = ref.timed(clips, 2, warm=0)
            line["cpu_baseline"] = {"value": clips * CLIP_T * 2 / sum(ts), "unit": "frames/s", "cores": cores, "kind": "port",
                                    "sample": "%d of the %d clips (x %d frames), full recurrence, torch-CPU fp32 oracle, 2 passes "
                                              "(%.1f s)" % (clips, B, CLIP_T, sum(ts))}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, frames_u8, last_f32):
    """Save what a ClipEngine caller received from one clip batch, for a fixed seeded sample of the clips, so that two builds
    can be compared output for output: hr_frames_u8 [T,S,128,128,3] (the uint8 HR frames as float32), hr_last_frame_f32
    [S,128,128,3] (fp32 output of the last frame) and sample_clips [S] (the clip indices, float64)."""
    B = frames_u8.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_CLIPS), replace=False))
    sel = torch.from_numpy(idx)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "hr_frames_u8.npy"), frames_u8[:, sel].float().numpy())
    np.save(os.path.join(out_dir, "hr_last_frame_f32.npy"), last_f32[sel.to(last_f32.device)].float().cpu().numpy())
    np.save(os.path.join(out_dir, "sample_clips.npy"), idx.astype(np.float64))


def _traffic(name):
    """DRAM bytes per launch of the kernel from the committed `ncu --set full` capture (profiles/), or None."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))["traffic_bytes_per_launch"]
    except Exception:
        return None


def bench_train(args, rank, world, dev, dist, ev_time, max_over_ranks, note, peak_tf_sus):
    """FRVSR (runGan.py case 4 flags) and TecoGAN (case 3 flags) training steps at B=4 clips per rank, RNN_N=10, 32x32 LR
    crops, bf16 tensor-core convolutions.  Under torchrun every step carries the single NCCL all-reduce of the flat
    gradient bucket (tecogan_b200/parallel.py).  Frames/s counts unique HR frames (B x RNN_N per rank and step)."""
    import main as M
    from tecogan_b200 import config, variables as V
    from tecogan_b200.init_params import xavier_params
    from tecogan_b200.lib.dataloader import frvsr_gpu_data_loader
    from tecogan_b200.lib.Teco import FRVSR, TecoGAN
    common = ["--mode", "train", "--output_dir", "/tmp/teco_bench", "--batch_size", "4", "--RNN_N", "10", "--crop_size", "32",
              "--learning_rate", "0.00005", "--decay_rate", "1.0", "--stair", "--beta", "0.9"]
    cases = {
        "config3_frvsr": (common + ["--num_resblock", "10", "--ratio", "-0.01", "--nopingpang"], 268.5),
        "config4_tecogan": (common + ["--num_resblock", "16", "--ratio", "0.01", "--pingpang", "--pp_scaling", "0.5",
                                      "--vgg_scaling", "0.2", "--Dt_mergeDs", "--D_LAYERLOSS"], 3.0 * 2239.0),
    }
    out = {"precision": os.environ.get("TECO_TRAIN_PRECISION", "bf16"), "clips_per_gpu": 4, "rnn_n": 10, "crop": 32,
           "allreduce": "one NCCL all-reduce (sum) of the flat fp32 bucket [G | FNet | D grads | t_balance | loss scalars] per step"
                        if world > 1 else "single rank: no collective"}
    config.set_train_precision(out["precision"])
    for name, (flags, gflop_step) in cases.items():
        F = M.parse_flags(flags)
        gan = F.ratio > 0
        st = V.set_default_store(V.VariableStore())
        st.load(xavier_params(1, F.num_resblock, gan, F.vgg_scaling > 0))
        lr, tg = frvsr_gpu_data_loader(M.synthetic_hr_batch(F, 0, rank, dev), F)
        Net = TecoGAN(lr, tg, F) if gan else FRVSR(lr, tg, F)
        for _ in range(3):
            r = Net.train()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        n = args.train_steps
        ms = ev_time(lambda: [Net.train() for _ in range(n)])
        ms = max_over_ranks([ms])[0] / n
        fps = F.batch_size * F.RNN_N * world / (ms / 1000.0)
        frame_len = (2 * F.RNN_N - 1) if F.pingpang else F.RNN_N
        out[name] = {"ms_per_step": ms, "value": fps, "unit": "unique HR frames/s",
                     "reference_style_rate": "image/sec %.1fx%02d" % (F.batch_size * world / (ms / 1000.0), frame_len),
                     "bucket_bytes": int(Net.train.bucket.numel() * 4),
                     "algorithmic_gflop_per_step_per_gpu": gflop_step,
                     "frac_of_sustained_bf16": gflop_step / ms / peak_tf_sus,
                     "finite_losses": bool(all(np.isfinite(v) for v in r["update_list"]))}
        note("%s: %.1f ms/step" % (name, ms))
        del Net
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
