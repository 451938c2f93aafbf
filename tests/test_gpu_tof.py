"""GPU: grey conversion, Farneback flow and tOF kernels (tecogan_b200/csrc/optflow.cu via tecogan_b200/metrics.py) against
cv2's values in tests/golden/tof.npz and the numpy restatement tests/golden/tof_ref.py; batching invariance; the
metrics.py --keys CLI; and the tOF parity of the bf16 engine against the fp32 oracle."""
import os

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN
from tests.golden import make_golden_tof as G
from tests.golden import tof_ref as T

pytestmark = pytest.mark.gpu

# Flow tolerances (px).  The GPU and cv2 differ only by float summation order; the max allows rare flips of the in-image
# test of the bilinear gather (measured on a B200 at 576x720: mean 5.1e-6, p99.9 1.3e-3, max 1.3e-2).
FLOW_MEAN, FLOW_P999, FLOW_MAX = 1e-4, 5e-3, 0.1
# Per-frame tOF vs cv2 / the restatement: measured max |diff| 1.3e-6.
TOF_TOL = 1e-5


def _g():
    return np.load(os.path.join(GOLDEN, "tof.npz"), allow_pickle=False)


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _flow_close(got, want):
    d = np.abs(got.astype(np.float64) - want)
    stats = (d.mean(), np.quantile(d, 0.999), d.max())
    print("flow |diff| mean %.2e p99.9 %.2e max %.2e" % stats)
    assert stats[0] <= FLOW_MEAN and stats[1] <= FLOW_P999 and stats[2] <= FLOW_MAX, stats
    return stats[2]


def test_grey_kernel_is_cv2_rule_on_every_triplet_and_cuts_larger_results():
    from tecogan_b200 import metrics as M
    a = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([(a >> 16) & 255, (a >> 8) & 255, a & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(M.rgb_to_grey(_cu(rgb)).cpu().numpy(), T.rgb_to_grey_u8(rgb))
    big = np.random.RandomState(3).randint(0, 256, size=(3, 70, 90, 3)).astype(np.uint8)
    got = M.rgb_to_grey(_cu(big), 63, 81).cpu().numpy()
    assert got.shape == (3, 63, 81) and np.array_equal(got, T.rgb_to_grey_u8(big[:, :63, :81]))


@pytest.mark.parametrize("name", ["pair01", "pair23", "ragged141x178", "single63x100", "custom12"])
def test_flow_matches_cv2_golden(name):
    from tecogan_b200 import metrics as M
    g = _g()
    cal = np.stack([T.rgb_to_grey_u8(f) for f in G.calendar()])
    prev, nxt, args = G.small_cases(cal)[name]
    # measured max |diff| over the five cases: 5.8e-5 px
    assert _flow_close(M.farneback_flow(_cu(prev), _cu(nxt), *args).cpu().numpy(), g["flow_" + name]) <= 2.5e-4


def test_flow_matches_cv2_at_vid4_size():
    from tecogan_b200 import metrics as M
    tg, _ = G.vid4_sequence()
    f = M.farneback_flow(_cu(T.rgb_to_grey_u8(tg[0])), _cu(T.rgb_to_grey_u8(tg[1]))).cpu().numpy()
    _flow_close(f[::8, ::8], _g()["vid4_flow01_sub8"])


@pytest.mark.parametrize("hw,args", [((97, 131), G.REF_ARGS), ((40, 257), G.REF_ARGS), ((150, 66), (0.7, 4, 7, 4, 7, 1.5)),
                                     ((64, 64), (0.5, 2, 5, 2, 3, 0.9))])
def test_flow_matches_restatement_on_ragged_sizes(hw, args):
    from tecogan_b200 import metrics as M
    tg, rs = G.vid4_sequence()
    h, w = hw
    a, b = T.rgb_to_grey_u8(tg[2][100:100 + h, 50:50 + w]), T.rgb_to_grey_u8(rs[3][100:100 + h, 50:50 + w])
    # measured max |diff|: 2.7e-5 px.  (winsize 1 is left out: a one-pixel 2x2 solve is so ill-conditioned that cv2 and
    # the restatement already differ by 100 px there.)
    assert _flow_close(M.farneback_flow(_cu(a), _cu(b), *args).cpu().numpy(), T.farneback_flow_np(a, b, *args)) <= 1e-4


def test_pair_in_batch_is_bit_identical_to_pair_alone():
    from tecogan_b200 import metrics as M
    tg, rs = G.vid4_sequence()
    grey = np.stack([T.rgb_to_grey_u8(f[:288, :360]) for f in np.concatenate([tg, rs])])       # 12 frames
    g = _cu(grey)
    prev = torch.stack([g[i] for i in (0, 1, 2, 3, 4, 6, 7, 8)] * 2)
    nxt = torch.stack([g[i] for i in (1, 2, 3, 4, 5, 7, 8, 9)] * 2)           # a 2x8-pair batch
    batch = M.farneback_flow(prev, nxt)
    for k in (0, 5, 11):
        alone = M.farneback_flow(prev[k].contiguous(), nxt[k].contiguous())
        assert torch.equal(batch[k], alone), k
    assert torch.equal(batch[:8], batch[8:])


def test_tof_of_vid4_sequence_matches_cv2_golden():
    from tecogan_b200 import metrics as M
    tg, rs = G.vid4_sequence()
    got = M.tof(_cu(tg), _cu(rs), cutfr=0)
    want = _g()["vid4_tof"]
    print("tOF gpu", got, "cv2", want)
    assert len(got) == len(want) and np.abs(np.array(got) - want).max() <= TOF_TOL
    ref = T.tof_sequence(tg, rs, cutfr=0)
    assert np.abs(np.array(got) - np.array(ref)).max() <= TOF_TOL


def test_tof_is_zero_for_identical_sequences_and_cuts_larger_results():
    from tecogan_b200 import metrics as M
    tg, rs = G.vid4_sequence()
    t = _cu(tg[:, :200, :240])
    assert M.tof(t, t, cutfr=1) == [0.0] * 3
    bigger = _cu(np.pad(tg[:, :200, :240], ((0, 0), (0, 4), (0, 4), (0, 0)), constant_values=255))
    assert M.tof(t, bigger, cutfr=1) == [0.0] * 3                 # the result is cut to the target size first
    r = M.evaluate_sequence(t, t, cutfr=1, keys=("PSNR", "SSIM", "tOF"))
    assert r["tOF"] == [0.0] * 3 and r["FolderAvg_tOF"] == 0.0
    assert set(M.evaluate_sequence(t, t, cutfr=1)) == {"PSNR", "SSIM", "FolderAvg_PSNR", "FolderAvg_SSIM"}


def test_misuse_raises_value_error():
    from tecogan_b200 import metrics as M
    a = torch.zeros(64, 64, dtype=torch.uint8, device="cuda")
    for kw in ({"flags": 256}, {"poly_n": 9}, {"poly_n": 0}, {"winsize": 16}, {"winsize": 17}, {"pyr_scale": 1.0},
               {"iterations": 0}):
        with pytest.raises(ValueError):
            M.farneback_flow(a, a, **kw)
    with pytest.raises(ValueError):
        M.farneback_flow(a.cpu(), a.cpu())
    with pytest.raises(ValueError):
        M.farneback_flow(a.float(), a.float())
    with pytest.raises(ValueError):
        M.farneback_flow(a, a[:32])
    rgb = torch.zeros(5, 64, 64, 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):
        M.tof(rgb, rgb[:, :32])
    with pytest.raises(ValueError):
        M.evaluate_sequence(rgb, rgb, cutfr=1, keys=("tLP100",))


def _write_pngs(d, frames):
    cv2 = pytest.importorskip("cv2")
    os.makedirs(d)
    for i, f in enumerate(frames):
        cv2.imwrite(os.path.join(d, "frame_%03d.png" % i), np.ascontiguousarray(f[:, :, ::-1]))


def test_cli_keys_tof_columns_and_default_run_without_them(tmp_path):
    pd = pytest.importorskip("pandas")
    import metrics
    tg, rs = G.vid4_sequence()
    tg, rs = tg[:, :144, :176], rs[:, :148, :180]                  # results larger: cut to the target size
    _write_pngs(str(tmp_path / "tgt"), tg)
    _write_pngs(str(tmp_path / "res"), rs)
    out = str(tmp_path / "log")
    metrics.main(["--output", out, "--results", str(tmp_path / "res"), "--targets", str(tmp_path / "tgt"),
                  "--keys", "PSNR,SSIM,tOF"])
    text = open(os.path.join(out, "metrics.csv")).read()
    head = pd.read_csv(os.path.join(out, "metrics.csv"), nrows=2, index_col=0)
    assert list(head.columns) == ["PSNR_00", "SSIM_00", "tOF_00"]
    want = T.tof_sequence(tg, rs[:, :144, :176], cutfr=2)          # frames 2, 3 -> one tOF value (frame 3)
    assert abs(float(head["tOF_00"].iloc[0]) - want[0]) <= TOF_TOL and np.isnan(head["tOF_00"].iloc[1])
    assert "Avg_tOF" in text and "FolderAvg_tOF" in text and "FrameAvg_tOF" in text
    log = open(os.path.join(out, "metricsfile.txt")).read()
    assert "tOF %02.2f, psnr" % want[0] in log
    out2 = str(tmp_path / "log2")
    metrics.main(["--output", out2, "--results", str(tmp_path / "res"), "--targets", str(tmp_path / "tgt")])
    assert "tOF" not in open(os.path.join(out2, "metrics.csv")).read()


def test_tof_parity_of_bf16_engine_with_fp32_oracle_on_config1_calendar():
    """tOF(stand-in target, bf16 engine) vs tOF(stand-in target, fp32 oracle) on the config-1 setup of
    test_gpu_models.py (calendar 32x32 LR, 10 frames + 5 warm-up, N=16, damped weights)."""
    from oracle import teco_oracle as O
    from tecogan_b200 import config, metrics as M, variables as V
    from tecogan_b200.engine import InferenceEngine
    g = np.load(os.path.join(GOLDEN, "calendar_lr.npz"))
    fr = g["crop32_u8"][:10].astype(np.float32) / 255.0
    frames = [torch.from_numpy(fr[i]) for i in O.warmup_order(len(fr))]
    pg, pf = O.damp_generator(O.init_generator(seed=1234, num_resblock=16)), O.init_fnet(seed=4321)
    ref = O.inference_sequence(pg, pf, frames, 16)
    V.set_default_store(V.VariableStore()).load({**pg, **pf})
    config.set_precision("bf16")
    outs = InferenceEngine(32, 32, 16).run_sequence([f.cuda() for f in frames])
    tgt = np.stack([O.save_img_u8(O.bicubic_four(f.unsqueeze(0))[0]) for f in frames[5:]])
    eng = np.stack([O.save_img_u8(o[0].cpu()) for o in outs[5:]])
    orc = np.stack([O.save_img_u8(r) for r in ref[5:]])
    te, to = M.tof(_cu(tgt), _cu(eng)), M.tof(_cu(tgt), _cu(orc))
    d = max(abs(a - b) for a, b in zip(te, to))
    print("config-1 tOF engine %s oracle %s max |diff| %.4g" % (np.round(te, 4), np.round(to, 4), d))
    assert d <= 0.01, (te, to)
