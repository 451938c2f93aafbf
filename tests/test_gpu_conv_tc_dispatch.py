"""Which tcgen05 conv kernel teco_conv3x3_tc launches for a shape: conv3x3_tc_onetile_kernel (one tile per CTA) or the
persistent conv3x3_tc_kernel, and with which template arguments <MODE, TPS, J, KS>.  A shape routed to the other kernel
still computes the right result, only slower, so the numerical tests cannot see it.  The tile-count thresholds depend on
the SM count; every case states the condition under which its expectation holds and is skipped on a device where it
does not."""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

KERNEL = re.compile(r"(conv3x3_tc(?:_onetile)?_kernel)<\s*(\d+),\s*(\d+),\s*(\d+),\s*(\d+)\s*>")


def _tiles(n, h, w):
    """16 x 8-pixel tiles of an n x h x w layer."""
    return n * -(-h // 16) * -(-w // 8)


# id: (n, h, w, cout, mode, fp32 output channels or 0), expected kernel, <MODE, TPS, J, KS>, holds for SM count s
CASES = {
    "single_wave_64": ((1, 128, 128, 64, 0, 0), "conv3x3_tc_onetile_kernel", (0, 3, 1, 3), lambda s: _tiles(1, 128, 128) <= s),
    "multi_wave_64": ((2, 256, 256, 64, 0, 0), "conv3x3_tc_kernel", (0, 3, 2, 2), lambda s: _tiles(2, 256, 256) >= 4 * s),
    "tconv_many_waves": ((5, 128, 128, 64, 1, 0), "conv3x3_tc_kernel", (1, 3, 1, 1), lambda s: _tiles(5, 128, 128) >= 4 * s),
    "tconv_small": ((1, 32, 32, 64, 1, 0), "conv3x3_tc_onetile_kernel", (1, 3, 1, 1), lambda s: _tiles(1, 32, 32) <= s),
    "narrow_fp32_output": ((3, 128, 128, 16, 0, 3), "conv3x3_tc_kernel", (2, 3, 3, 1), lambda s: _tiles(3, 128, 128) > s),
}


@pytest.mark.parametrize("case", list(CASES))
def test_conv3x3_tc_launches_the_planned_kernel(case):
    from tecogan_b200 import kernels as K
    (n, h, w, cout, mode, out_c), kernel, targs, holds = CASES[case]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if not holds(sms):
        pytest.skip("%s: expectation is for a different SM count than %d" % (case, sms))
    x = torch.zeros(n, h, w, 64, device="cuda", dtype=torch.bfloat16)
    wpk = K.packed_weight(torch.zeros(3, 3, 64, cout, device="cuda"), 64, cout, transpose_layout=(mode == 1))
    bias = torch.zeros(cout, device="cuda")
    out = torch.zeros(n, h, w, out_c, device="cuda") if out_c else None
    y = None if out_c else torch.empty(n, h * (2 if mode == 1 else 1), w * (2 if mode == 1 else 1), cout, device="cuda",
                                       dtype=torch.bfloat16)

    def run():
        K.conv3x3_tc(x, wpk, bias, y, cout=cout, act=K.ACT_RELU, mode=mode, out_f32=out)

    run()                                   # module load and first launch outside the trace
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    launched = [(m.group(1), tuple(int(g) for g in m.groups()[1:])) for m in (KERNEL.search(e.name) for e in prof.events()) if m]
    assert launched == [(kernel, targs)], launched
