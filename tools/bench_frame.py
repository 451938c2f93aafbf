"""Frame rate of the streaming recurrence at LR 128x128 (configs[1]) with and without the fnet look-ahead.
Usage: python tools/bench_frame.py [h w frames]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tecogan_b200.init_params import xavier_params  # noqa: E402
from tecogan_b200 import config, variables as V
from tecogan_b200.engine import InferenceEngine

h = int(sys.argv[1]) if len(sys.argv) > 1 else 128
w = int(sys.argv[2]) if len(sys.argv) > 2 else 128
T = int(sys.argv[3]) if len(sys.argv) > 3 else 60
config.set_precision("bf16")
st = V.set_default_store(V.VariableStore())
st.load(xavier_params(1234, 16))
clip = torch.rand(T, h, w, 3, device="cuda")
outs = {}
for la in (False, True):
    eng = InferenceEngine(h, w, 16)
    def run():
        eng.reset()
        res = None
        for t in range(T):
            eng.step(clip[t], next_lr=clip[t + 1] if (la and t + 1 < T) else None)
        return eng.out_u8.clone()
    for _ in range(2):
        outs[la] = run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    print("lookahead=%d: %.1f us/frame  %.0f frames/s" % (la, ms * 1e3 / T, T / ms * 1e3), flush=True)
print("last frame identical:", bool(torch.equal(outs[False], outs[True])))
