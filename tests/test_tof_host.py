"""CPU: the numpy restatement of cv2's grey conversion, Farneback flow and tOF (tests/golden/tof_ref.py) against the cv2
fixtures of tests/golden/tof.npz, the workspace-size function of the C ABI, and the --keys flag of metrics.py."""
import ctypes
import os

import numpy as np
import pytest

from tests.conftest import GOLDEN, ROOT
from tests.golden import make_golden_tof as G
from tests.golden import tof_ref as T

# Flow tolerances against cv2 (px).  cv2 and the restatement differ only by float summation order; the measured errors
# are far below these (see each test).  The max allows rare flips of the in-image test of the bilinear gather.
FLOW_MEAN, FLOW_P999, FLOW_MAX = 1e-4, 5e-3, 0.1


def _g():
    return np.load(os.path.join(GOLDEN, "tof.npz"), allow_pickle=False)


def _flow_close(got, want):
    d = np.abs(got.astype(np.float64) - want)
    assert d.mean() <= FLOW_MEAN and np.quantile(d, 0.999) <= FLOW_P999 and d.max() <= FLOW_MAX, \
        (d.mean(), np.quantile(d, 0.999), d.max())
    return d.max()


def test_grey_rule_matches_cv2_on_every_rgb_triplet():
    cv2 = pytest.importorskip("cv2")
    a = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([(a >> 16) & 255, (a >> 8) & 255, a & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(T.rgb_to_grey_u8(rgb), cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY))


def test_grey_rule_matches_golden_sample():
    g = _g()
    assert np.array_equal(T.rgb_to_grey_u8(g["grey_rgb"]), g["grey_cv2"])


def test_vid4_sequence_derivation_is_pinned_by_hash():
    tg, rs = G.vid4_sequence()
    assert tg.shape == rs.shape == (G.VID4_FRAMES, 576, 720, 3)
    assert G.sha256(tg, rs) == str(_g()["vid4_sha256"])


def test_pyramid_depth_rule():
    assert T.pyramid_levels(144, 180, 0.5, 3) == 2
    assert T.pyramid_levels(63, 100, 0.5, 3) == 0
    assert T.pyramid_levels(576, 720, 0.5, 3) == 3
    assert [T.level_geometry(141, 178, 0.5, k)[3:] for k in range(3)] == [(141, 178), (70, 89), (35, 44)]


@pytest.mark.parametrize("name", ["pair01", "pair23", "ragged141x178", "single63x100", "custom12"])
def test_restated_flow_matches_cv2_small_frames(name):
    # measured max |diff|: 3e-6 px (reference parameters), 6e-5 px (custom12)
    g = _g()
    cal = np.stack([T.rgb_to_grey_u8(f) for f in G.calendar()])
    prev, nxt, args = G.small_cases(cal)[name]
    assert _flow_close(T.farneback_flow_np(prev, nxt, *args), g["flow_" + name]) < 2.5e-4


def test_restated_flow_and_tof_match_cv2_at_vid4_size():
    # measured: flow mean 5e-6 px, max 0.012 px (one gather flip); tOF max |diff| 3.3e-6
    g = _g()
    tg, rs = G.vid4_sequence()
    f = T.farneback_flow_np(T.rgb_to_grey_u8(tg[0]), T.rgb_to_grey_u8(tg[1]))
    _flow_close(f[::8, ::8], g["vid4_flow01_sub8"])
    tofs = T.tof_sequence(tg, rs, cutfr=0)
    assert np.abs(np.array(tofs) - g["vid4_tof"]).max() <= 2e-5     # 6x the measured value


def _workspace_formula(F, P, H, W, s, levels):
    a = lambda b: (b + 255) // 256 * 256
    top = T.pyramid_levels(H, W, s, levels)
    area1 = int(np.round(H * s)) * int(np.round(W * s)) if top >= 1 else 0
    hw = H * W
    return (a(4 * F * hw) + a(20 * F * hw) + 2 * a(8 * P * area1) + 2 * a(20 * P * hw) + a(8 * P))


def test_workspace_bytes_formula_and_rejections():
    lib = ctypes.CDLL(os.path.join(ROOT, "tecogan_b200", "libteco.so"))
    fn = lib.teco_farneback_workspace_bytes
    fn.argtypes = [ctypes.c_int32] * 4 + [ctypes.c_double, ctypes.c_int32]
    fn.restype = ctypes.c_int64
    for F, P, H, W, s, lv in ((74, 72, 576, 720, 0.5, 3), (2, 1, 144, 180, 0.5, 3), (2, 1, 63, 100, 0.5, 3),
                              (7, 6, 141, 178, 0.6, 1), (3, 2, 33, 40, 0.9, 5)):
        assert fn(F, P, H, W, s, lv) == _workspace_formula(F, P, H, W, s, lv), (F, P, H, W, s, lv)
    for bad in ((0, 1, 64, 64, 0.5, 3), (2, 0, 64, 64, 0.5, 3), (2, 1, 1, 64, 0.5, 3), (2, 1, 64, 64, 1.0, 3),
                (2, 1, 64, 64, 0.0, 3), (2, 1, 64, 64, 0.5, -1), (2, 70000, 64, 64, 0.5, 3)):
        assert fn(*bad) == -1, bad


def test_metrics_cli_keys_parsing():
    import metrics
    assert metrics.parse_keys("PSNR,SSIM") == ["PSNR", "SSIM"]
    assert metrics.parse_keys("tOF,PSNR") == ["PSNR", "tOF"]
    assert metrics.parse_keys("PSNR, SSIM, tOF") == ["PSNR", "SSIM", "tOF"]
    for bad in ("LPIPS", "PSNR,tof", "", ","):
        with pytest.raises(ValueError):
            metrics.parse_keys(bad)
    with pytest.raises(SystemExit):
        metrics.main(["--output", "/nonexistent", "--results", "a", "--targets", "b", "--keys", "PSNR,tLP100"])
