"""CPU: host-side logic of the mirror -- variable scopes / TF variable names, flag parsing, sub-pixel phase
decomposition of the stride-2 transposed conv, clip sharding and the 2-rank gloo all-reduce of the gradient bucket."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import teco_oracle as O


def test_variable_scopes_produce_tf_variable_names():
    from tecogan_b200 import variables as V
    st = V.set_default_store(V.VariableStore(device="cpu"))
    with V.variable_scope('generator'), V.variable_scope('generator_unit'), V.variable_scope('resblock_3'):
        with V.variable_scope('conv_1'), V.variable_scope('Conv'):
            w = V.get_variable('weights', (3, 3, 64, 64), fans=(576, 576))
            b = V.get_variable('biases', (64,), init='zeros')
            assert V.get_variable('weights', (3, 3, 64, 64), fans=(576, 576)) is w       # reuse
            with pytest.raises(ValueError):
                V.get_variable('weights', (3, 3, 64, 32), fans=(576, 288))
    assert list(st) == ['generator/generator_unit/resblock_3/conv_1/Conv/weights',
                        'generator/generator_unit/resblock_3/conv_1/Conv/biases']
    assert float(w.abs().max()) <= (6.0 / 1152) ** 0.5 + 1e-7 and float(b.abs().max()) == 0.0


def test_init_params_cover_the_same_names_as_the_oracle():
    from tecogan_b200.init_params import xavier_params
    p = xavier_params(3, num_resblock=16, need_d=True, need_vgg=True)
    ref = {}
    for d in (O.init_generator(), O.init_fnet(), O.init_discriminator(), O.init_vgg19()):
        ref.update(d)
    assert set(p) == set(ref)
    for k in p:
        assert tuple(p[k].shape) == tuple(ref[k].shape), k


def test_flag_parsing_follows_tf_app_flags_conventions():
    import main
    F_ = main.parse_flags(['--mode', 'train', '--nopingpang', '--stair', '--ratio', '-0.01', '--output_dir', '/tmp/x',
                           '--Dt_mergeDs', '--learning_rate=0.00005', '--num_resblock', '10'])
    assert (F_.pingpang, F_.stair, F_.ratio, F_.Dt_mergeDs, F_.learning_rate, F_.num_resblock) == (False, True, -0.01, True, 5e-5, 10)
    assert F_.crop_dt == 0.75 and F_.Dbalance == 0.4 and F_.RNN_N == 10 and F_.EPS == 1e-12   # reference defaults


@pytest.mark.parametrize("K,pad", [(3, 0), (4, 1)])
def test_transposed_conv_phase_decomposition(K, pad):
    """kernels._phase_taps + the phase-weight slicing of conv_transpose2x_raw, emulated with torch-CPU convs, equals
    the oracle's conv2d_transpose (K=3, pad 0) / the input gradient of a stride-2 SAME conv (K=4, pad 1)."""
    from tecogan_b200.kernels import _phase_taps
    torch.manual_seed(0)
    n, h, w, cin, cout = 2, 5, 6, 3, 4
    x = torch.randn(n, h, w, cin)
    w_oi = torch.randn(K, K, cout, cin)
    y = torch.zeros(n, 2 * h, 2 * w, cout)
    for a in (0, 1):
        kys, pt = _phase_taps(K, pad, a)
        for b in (0, 1):
            kxs, pl = _phase_taps(K, pad, b)
            wp = torch.stack([torch.stack([w_oi[ky, kx] for kx in kxs], dim=0) for ky in kys], dim=0).permute(0, 1, 3, 2)
            xp = F.pad(x.permute(0, 3, 1, 2), (pl, len(kxs) - 1 - pl, pt, len(kys) - 1 - pt))
            y[:, a::2, b::2] = F.conv2d(xp, wp.permute(3, 2, 0, 1)).permute(0, 2, 3, 1)
    if K == 3:
        ref = O.conv2d_transpose(x, w_oi)
    else:
        inp = torch.zeros(n, 2 * h, 2 * w, cout, requires_grad=True)
        (ref,) = torch.autograd.grad(O.conv2d(inp, w_oi, None, stride=2), inp, x)   # w_oi as HWIO with I=cout
    assert (y - ref).abs().max().item() < 1e-5


def test_clip_sharding_is_balanced_and_complete():
    from tecogan_b200.parallel import shard_clips
    for n, w in ((8, 8), (10, 4), (3, 8), (32, 8)):
        spans = [shard_clips(n, r, w) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1


def _dp_worker(rank, world, port, ret):
    import torch.distributed as dist
    from tecogan_b200.parallel import allreduce_bucket, decide_with_d
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(rank)
    bucket = torch.cat((torch.randn(1000), torch.tensor([0.3 + 0.4 * rank, 1.0 + rank])))   # grads | t_balance | loss
    mine = bucket.clone()
    inv = allreduce_bucket(bucket)
    tb_ema = 0.0
    decisions = []
    for _ in range(3):
        with_d, tb_ema = decide_with_d(tb_ema, float(bucket[1000]) * inv, 0.004)
        decisions.append(with_d)
    ret[rank] = (mine.numpy(), bucket.numpy(), inv, decisions, tb_ema)
    dist.destroy_process_group()


def test_two_rank_gloo_allreduce_bucket_and_identical_control_flow():
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    port = 29500 + os.getpid() % 2000
    mp.spawn(_dp_worker, args=(2, port, ret), nprocs=2, join=True)
    (m0, b0, inv0, d0, e0), (m1, b1, inv1, d1, e1) = ret[0], ret[1]
    assert inv0 == inv1 == 0.5
    np.testing.assert_allclose(b0, m0 + m1, rtol=1e-6)
    np.testing.assert_array_equal(b0, b1)                    # every rank holds the same reduced bucket
    assert d0 == d1 and e0 == e1                             # hence the same with-D / without-D branch every step
    assert d0 == [True, False, False]                        # EMA(0.01 * 0.5) crosses Dbalance=0.004 after one update


def test_pt_checkpoint_is_validated_like_saver_restore(tmp_path):
    """A .pt checkpoint must hold every variable of the graph with the right shape (Saver.restore semantics,
    reference main.py:221-224,245,346-349); --pre_trained_model zero-fills missing generator/fnet variables
    (lib/ops.py:370-391) and leaves discriminator variables to their initialiser."""
    import main
    from tecogan_b200 import variables as V
    from tecogan_b200.init_params import xavier_params
    p10 = xavier_params(3, num_resblock=10)
    path = str(tmp_path / "m10.pt")
    torch.save(p10, path)
    st = V.VariableStore(device="cpu")
    main.load_checkpoint(st, path, 10)
    assert set(st) == set(p10)
    with pytest.raises(ValueError, match="lacks"):
        main.load_checkpoint(V.VariableStore(device="cpu"), path, 16)                 # a 10-block file for a 16-block graph
    with pytest.raises(ValueError, match="lacks"):
        main.load_checkpoint(V.VariableStore(device="cpu"), path, 10, need_d=True)    # FRVSR file where D weights are expected
    st2 = V.VariableStore(device="cpu")
    main.load_checkpoint(st2, path, 16, need_d=True, pre_trained_model=True)
    assert float(st2['generator/generator_unit/resblock_16/conv_2/Conv/weights'].abs().max()) == 0.0
    assert not any(k.startswith('tdiscriminator/') for k in st2)
    bad = dict(p10)
    bad['fnet/autoencode_unit/encoder_1/conv_1/Conv/weights'] = torch.zeros(3, 3, 6, 16)
    torch.save(bad, path)
    with pytest.raises(ValueError, match="Wrong shape"):
        main.load_checkpoint(V.VariableStore(device="cpu"), path, 10)


def test_train_mode_refuses_to_run_without_data_or_vgg_unless_opted_in():
    import main
    F = main.parse_flags(["--mode", "train", "--output_dir", "/tmp/x"])
    assert F.train_precision == "fp32" and F.synthetic_data is False
    with pytest.raises(ValueError, match="input_video_dir is not provided"):
        main.train(F)


def test_metrics_crop_window_matches_reference_crop_8x8_golden():
    """tecogan_b200.metrics.crop_window (host arithmetic) against the offsets/sizes the reference's crop_8x8 produced."""
    import os
    import numpy as np
    from tests.conftest import GOLDEN
    from tecogan_b200.metrics import crop_8x8, crop_window
    g = np.load(os.path.join(GOLDEN, "metrics.npz"), allow_pickle=False)
    for i in range(int(g["n_cases"])):
        t = g["tgt%d" % i]
        assert crop_window(t.shape[0], t.shape[1]) == tuple(int(v) for v in g["crop%d" % i])
        c, y, x = crop_8x8(t)
        assert c.shape[:2] == tuple(int(v) for v in g["crop%d" % i][2:])
    assert crop_window(144, 180) == (8, 10, 128, 160) and crop_window(32, 32)[2:] == (0, 0)


def test_adam_step_counts_from_a_reference_checkpoint():
    """Resuming from a checkpoint written by the reference: TensorFlow stores beta1^(t+1) per optimiser under
    generator_train/beta1_power{,_1,_2} (discriminator, generator, fnet); the discriminator stepped only withD_counter times."""
    from types import SimpleNamespace
    from tecogan_b200.lib.Teco import _TrainState
    ck = {"generator_train/beta1_power": 0.9 ** (37 + 1), "generator_train/beta1_power_1": 0.9 ** (100 + 1),
          "generator_train/beta1_power_2": 0.9 ** (100 + 1), "generator_train/gen_train_with_D_counter": 37}
    me = SimpleNamespace(GAN=True, global_step=100)
    opt = SimpleNamespace(b1=0.9)
    steps = {tag: _TrainState._tf_adam_steps(me, ck.get, tag, opt) for tag in "gfd"}
    assert steps == {"g": 100, "f": 100, "d": 37}
    only_counter = {"generator_train/gen_train_with_D_counter": 12}
    assert _TrainState._tf_adam_steps(me, only_counter.get, "d", opt) == 12
    assert _TrainState._tf_adam_steps(me, {}.get, "d", opt) == 100          # nothing known: every optimiser at global_step
    frvsr = SimpleNamespace(GAN=False, global_step=5)
    assert _TrainState._tf_adam_steps(frvsr, {"generator_train/beta1_power_1": 0.9 ** 6}.get, "f", opt) == 5


def test_metrics_cli_lists_png_like_the_reference(tmp_path):
    """metrics.py::listPNGinDir (reference metrics.py:28-35): only *.png, not the IB* inputs, ordered by the digits in the name."""
    import metrics as CLI
    for n in ("output_0010.png", "output_0002.png", "IB_0001.png", "output_0001.jpg", "col_high_0003.png", "notes.txt"):
        (tmp_path / n).write_bytes(b"")
    got = [p.split("/")[-1] for p in CLI.listPNGinDir(str(tmp_path))]
    assert got == ["output_0002.png", "col_high_0003.png", "output_0010.png"]


def test_warp_v2_source_window_holds_every_query_of_its_tile():
    """Host restatement of the window construction of warp_s2d_v2_kernel (csrc/warp_s2d_v2.cu::v2_window): from the min / max of
    the 4 x flow_lr samples around a 4 x 32 LR tile it derives the rows / columns of the previous HR frame that the tile's
    bilinear queries can touch.  Property: for random flows (smooth, rough, far out of range) and ragged frame sizes, every
    query of every HR pixel of the tile -- floor clamped to [0, size-2] plus its +1 neighbour, as dense_image_warp does --
    lies inside the window, and the 'interior' flags are only set when no clamp can trigger."""
    import numpy as np
    rng = np.random.RandomState(0)
    TLH, TLW = 4, 32

    def upscale4(f):                                   # upscale_four: legacy bilinear x4, edge-replicated (lib/ops.py:126-163)
        h, w, _ = f.shape
        fy = np.concatenate([f, f[-1:]], 0)
        rows = np.stack([(1 - k / 4) * fy[:-1] + (k / 4) * fy[1:] for k in range(4)], 1).reshape(4 * h, w, 2)
        fx = np.concatenate([rows, rows[:, -1:]], 1)
        return np.stack([(1 - k / 4) * fx[:, :-1] + (k / 4) * fx[:, 1:] for k in range(4)], 2).reshape(4 * h, 4 * w, 2)

    for case, (h, w, amp, off) in enumerate([(8, 32, 1.0, 0.0), (18, 45, 6.0, 0.0), (36, 40, 0.3, 2.5), (16, 64, 30.0, -40.0), (5, 9, 3.0, 1.0)]):
        H, W = 4 * h, 4 * w
        flow4 = (4.0 * (off + amp * (rng.rand(h, w, 2) - 0.5))).astype(np.float32)
        fl = upscale4(flow4.astype(np.float64))
        for ly0 in range(0, h, TLH):
            for lx0 in range(0, w, TLW):
                ii = np.minimum(np.arange(ly0, ly0 + TLH + 1), h - 1)
                jj = np.minimum(np.arange(lx0, lx0 + TLW + 1), w - 1)
                s = flow4[np.ix_(ii, jj)]
                mny, mxy, mnx, mxx = s[..., 0].min(), s[..., 0].max(), s[..., 1].min(), s[..., 1].max()
                Y0, X0 = 4 * ly0, 4 * lx0
                qy_lo, qy_hi = Y0 - mxy, Y0 + 4 * TLH - 1 - mny
                qx_lo, qx_hi = X0 - mxx, X0 + 4 * TLW - 1 - mnx
                clampf = lambda v, hi: min(max(v, 0.0), hi)
                y_lo = int(clampf(np.floor(qy_lo) - 1, H - 2))
                y_hi = int(clampf(np.floor(qy_hi) + 1, H - 2)) + 1
                x_lo = int(clampf(np.floor(qx_lo) - 1, W - 2)) & ~3
                x_hi = min((int(clampf(np.floor(qx_hi) + 1, W - 2)) + 1) | 3, W - 1)
                int_y = qy_lo >= 1 and qy_hi <= H - 3
                int_x = qx_lo >= 1 and qx_hi <= W - 3
                assert (x_hi - x_lo + 1) % 4 == 0 and x_lo % 4 == 0          # 16-byte aligned bulk copies of fp32 RGB rows
                ys = np.arange(Y0, min(Y0 + 4 * TLH, H))
                xs = np.arange(X0, min(X0 + 4 * TLW, W))
                qy = ys[:, None] - fl[np.ix_(ys, xs)][..., 0]
                qx = xs[None, :] - fl[np.ix_(ys, xs)][..., 1]
                fy, fx = np.floor(qy), np.floor(qx)
                if int_y:
                    assert fy.min() >= 0 and fy.max() <= H - 2, (case, ly0, lx0)
                if int_x:
                    assert fx.min() >= 0 and fx.max() <= W - 2, (case, ly0, lx0)
                iy, ix = np.clip(fy, 0, H - 2), np.clip(fx, 0, W - 2)
                assert y_lo <= iy.min() and iy.max() + 1 <= y_hi, (case, ly0, lx0, y_lo, y_hi, iy.min(), iy.max())
                assert x_lo <= ix.min() and ix.max() + 1 <= x_hi, (case, ly0, lx0, x_lo, x_hi, ix.min(), ix.max())


def test_conv_transpose_gradients_through_the_space_to_depth_identity():
    """kernels._ConvTranspose2xTC computes both gradients of conv2_tran as ordinary 3x3 stride-1 problems on the space-to-depth
    form of dz (W' = zero-scattered weights, rows kernels._tconv_rows()).  The identity itself, in fp32 on the CPU with the
    oracle's convolutions, against the oracle's autograd of conv2d_transpose (reference lib/ops.py:35-44, SURVEY A.3)."""
    import torch
    from oracle import teco_oracle as O
    from tecogan_b200 import kernels as K
    torch.manual_seed(0)
    N, H, W, C = 2, 5, 6, 4
    x = torch.randn(N, H, W, C, requires_grad=True)
    w = torch.randn(3, 3, C, C, requires_grad=True)             # [kh, kw, Cout, Cin]
    y = O.conv2d_transpose(x, w, torch.randn(C))
    dz = torch.randn_like(y)
    y.backward(dz)
    dzs = dz.view(N, H, 2, W, 2, C).permute(0, 1, 3, 2, 4, 5).reshape(N, H, W, 4 * C)          # channel (py, px, co)
    idx = torch.tensor(K._tconv_rows())
    assert sorted(K._tconv_rows()) == sorted(set(K._tconv_rows())) and len(idx) == 9
    wp = torch.zeros(36, C, C).index_copy_(0, idx, w.detach().reshape(9, C, C)).view(3, 3, 4 * C, C).requires_grad_(True)
    dx = O.conv2d(dzs, wp, None)                                                                  # input gradient
    assert (dx - x.grad).abs().max().item() < 1e-4
    (dx * x.detach()).sum().backward()            # d/dW' of sum_p conv(dzs, W')[p] . x[p]  =  the wgrad kernel's sum
    dw = wp.grad.view(36, C, C).index_select(0, idx).view(3, 3, C, C)
    assert (dw - w.grad).abs().max().item() < 1e-4 * max(1.0, w.grad.abs().max().item())


def test_bench_dump_outputs_is_a_small_seeded_float_sample(tmp_path):
    """bench.py --dump-outputs: for the metric configuration's clip batch (296 clips x 10 frames of 128x128 uint8) the
    files are float32 / float64, hold the same seeded clips on every run, and stay below 64 MB in all."""
    import bench
    T, B = bench.CLIP_T, bench.DEFAULT_CLIPS
    u8 = (torch.arange(B) % 256).to(torch.uint8).view(1, B, 1, 1, 1).expand(T, B, 4 * bench.LR, 4 * bench.LR, 3).contiguous()
    last = torch.arange(B, dtype=torch.float32).view(B, 1, 1, 1).expand(B, 4 * bench.LR, 4 * bench.LR, 3).contiguous()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), u8, last)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["hr_frames_u8.npy", "hr_last_frame_f32.npy", "sample_clips.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 * 2 ** 20
    a = {n: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert a[n].dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(a[n], np.load(tmp_path / "b" / n))
    idx = a["sample_clips.npy"].astype(np.int64)
    assert len(set(idx.tolist())) == len(idx) == bench.DUMP_CLIPS and idx.max() < B
    assert a["hr_frames_u8.npy"].shape == (T, len(idx), 128, 128, 3)
    np.testing.assert_array_equal(a["hr_frames_u8.npy"][:, :, 0, 0, 0], np.broadcast_to(idx % 256, (T, len(idx))))
    np.testing.assert_array_equal(a["hr_last_frame_f32.npy"][:, 5, 7, 1], idx)
