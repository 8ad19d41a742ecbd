"""GPU parity of the whole hot path (WCT.predict, wct.py:70-106) against the CPU oracle.

Two statements (DESIGN.md "Parity"):
  * teacher-forced: every level of the engine's own run is re-computed by the fp64 oracle
    FROM THE ENGINE'S INPUT TO THAT LEVEL; each level output must agree to <= 1e-3;
  * free-running: the final image vs the oracle's own 5-level run, reported next to the
    oracle's fp32-vs-fp64 distance (the chained levels amplify rounding noise ~1e3x with
    random weights, so this bound is stated relative to that noise floor).
"""
import os

import numpy as np
import pytest
import torch

from oracle import nets, ref_ops
from tests.test_oracle import PIPE_GOLDEN, load_pipeline_fixture
from wct_tf_b200.engine import Engine
from wct_tf_b200.weights import make_synthetic_weights
from wct_tf_b200.wct import WCT

pytestmark = pytest.mark.gpu
ALL = ["relu5_1", "relu4_1", "relu3_1", "relu2_1", "relu1_1"]
# The chained levels of a RANDOM-weight pipeline amplify rounding noise ~1e3x (DESIGN.md "Parity"):
# the reference's own fp32 run sits ~4e-3 from its fp64 run.  The free-running bound is therefore
# stated as a multiple of that measured noise floor; the <=1e-3 claim is the teacher-forced one.
# Round 1 measured 4.1x: the weights' lo plane fell into the fp16 subnormals (tests/noise_split_cpu.py,
# profiles/r02_noise_split.txt).  With the per-layer power-of-two weight scale the engine measures 2.5x (9.9e-3 vs 3.9e-3;
# fixture wct5: 4.1e-3 vs 1.6e-3).  What is left is the activation format itself: hi+lo keeps 22-23 bits, i.e. up to 4x the
# rounding error of fp32 per stored activation -- the fp32 CUDA-core validation conv on the same storage lands at the same
# level as the tensor-core path (profiles/r02_noise_split.txt, GPU part), so it is not the MMAs.
FREE_RUN_NOISE_FACTOR = 3


@pytest.fixture(scope="module")
def weights():
    return make_synthetic_weights(42)


def _imgs(n, s, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (n, s, s, 3), dtype=np.uint8)


def _teacher_forced(weights, sem, adain, targets, csize, ssize, alpha=0.8, seeds=(100, 7)):
    """Every level of the engine's own run is recomputed by the fp64 oracle FROM THE ENGINE'S INPUT TO THAT LEVEL.
    Returns the worst max-abs error over encoder output / transformed feature / level output (all levels)."""
    eng = Engine(weights, targets, semantics=sem)
    rng_c, rng_s = np.random.default_rng(seeds[0]), np.random.default_rng(seeds[1])
    content = rng_c.integers(0, 256, (1, csize[0], csize[1], 3), dtype=np.uint8)
    style = rng_s.integers(0, 256, (1, ssize[0], ssize[1], 3), dtype=np.uint8)
    cap = {}
    out = eng.stylize(torch.from_numpy(content).cuda(), torch.from_numpy(style).cuda(), alpha=alpha, adain=adain,
                      want_info=True, capture=cap)
    eng.check_device()
    sfe = nets.encode(nets.preprocess(style).astype(np.float64), weights, targets, np.float64)
    worst = 0.0
    for i, relu in enumerate(targets):
        x = cap["level_input"][i].cpu().numpy().astype(np.float64)
        if i == 0:
            assert np.abs(x - content / 255.0).max() < 1e-7
        else:
            assert x.min() >= 0 and x.max() <= 1                     # model.py:86 clip between levels
        cf = nets.encode(x, weights, [relu], np.float64)[relu]
        got_cf = eng.act_to_f32(cap["content_feat"][i]).cpu().numpy()
        e_enc = np.abs(got_cf - cf).max()
        if adain:
            f = ref_ops.adain(cf, sfe[relu], alpha)
        else:
            fn = ref_ops.wct_tf if sem == "tf" else ref_ops.wct_np
            f, info = fn(cf, sfe[relu], alpha, return_info=True)
            k = eng.last_info[i].cpu().numpy()
            assert ref_ops.spectral_gap_ok(info["wc"]) and ref_ops.spectral_gap_ok(info["ws"]), "ill-posed vector"
            assert (k[0], k[1]) == (info["k_c"], info["k_s"])         # relu-target / rank bookkeeping: bit-exact
        got_f = eng.act_to_f32(cap["transformed"][i]).cpu().numpy()
        e_wct = np.abs(got_f - f).max()
        y = nets.decode(np.asarray(f, dtype=np.float64), weights, relu, np.float64)
        if i < len(targets) - 1:
            y = np.clip(y, 0, 1)
        e_out = np.abs(cap["level_output"][i].cpu().numpy() - y).max()
        print("%s %dx%d: encoder %.2e  transform %.2e  level output %.2e" % (relu, csize[0], csize[1], e_enc, e_wct, e_out))
        worst = max(worst, e_enc, e_wct, e_out)
    assert out.shape[0] == 1 and out.shape[3] == 3
    return worst


@pytest.mark.parametrize("sem,adain,targets,size", [
    ("np", False, ALL, 128),
    ("tf", False, ALL, 128),
    ("tf", True, ALL, 96),
    ("np", False, ["relu3_1", "relu1_1", "relu2_1"], 72),     # any order / subset (README.md:46)
    ("tf", False, ["relu1_1"], 64),
])
def test_teacher_forced_levels(weights, sem, adain, targets, size):
    assert _teacher_forced(weights, sem, adain, targets, (size, size), (size + 16, size + 16)) <= 1e-3


# ---- the configurations BASELINE.json names, at their full sizes (SURVEY 8d) -------------------------------------------
@pytest.mark.parametrize("sem", ["tf", "np"])
def test_config2_512x512_five_levels_teacher_forced(weights, sem):
    """configs[1]: 5-level relu5_1->relu1_1, 512x512 content, 512x512 style, alpha 0.8 (HW up to 262 144 in the
    split-K covariance): every level <= 1e-3 from the fp64 oracle, k_c/k_s equal, spectral gap asserted."""
    assert _teacher_forced(weights, sem, False, ALL, (512, 512), (512, 512), seeds=(1000, 7)) <= 1e-3


def test_config4_1024_content_512_style_teacher_forced(weights):
    """configs[3]: 1024x1024 content / 512x512 style (HW = 1 048 576 at relu1_1, 262 144 at relu2_1)."""
    assert _teacher_forced(weights, "tf", False, ALL, (1024, 1024), (512, 512), seeds=(1000, 7)) <= 1e-3


def test_config5_adain_512_teacher_forced(weights):
    """configs[4]: --adain, 512x512, 5 levels."""
    assert _teacher_forced(weights, "tf", True, ALL, (512, 512), (512, 512), seeds=(1000, 7)) <= 1e-3


def test_config3_two_gpu_shards_equal_one_gpu_bit_for_bit(weights, tmp_path):
    """configs[2] / SURVEY 4: a batch sharded over 2 GPUs (torchrun, parallel.stylize_sharded, NCCL gather) gives the SAME
    uint8 frames as one GPU running the whole batch: per-frame arithmetic does not depend on the batch a frame is in
    (deterministic split-K partials, no atomics) nor on the GPU."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import subprocess
    import sys
    out = tmp_path / "sharded.npy"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tests", "sharded_worker.py"), str(out), "6", "256"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout.decode()[-3000:]
    sharded = np.load(str(out))
    from tests.sharded_worker import make_batch
    c, s = make_batch(6, 256)
    wct = WCT(checkpoints=None, relu_targets=ALL, vgg_path=None, weights=weights)
    single = wct.predict_batch(c, s, alpha=0.8)
    assert sharded.shape == single.shape and np.array_equal(sharded, single)
    one_by_one = np.concatenate([wct.predict_batch(c[i:i + 1], s, alpha=0.8) for i in range(c.shape[0])])
    assert np.array_equal(one_by_one, single)


def test_free_running_five_levels_vs_oracle(weights):
    size = 128
    content, style = _imgs(1, size, 1000), _imgs(1, size, 7)
    o64, info = nets.pipeline(content[0], style[0], weights, ALL, alpha=0.8, semantics="np", dtype=np.float64, return_info=True)
    o32 = nets.pipeline(content[0], style[0], weights, ALL, alpha=0.8, semantics="np", dtype=np.float32)
    for inf in info:
        assert ref_ops.spectral_gap_ok(inf["wc"]) and ref_ops.spectral_gap_ok(inf["ws"])
    eng = Engine(weights, ALL, semantics="np")
    out = eng.stylize(torch.from_numpy(content).cuda(), torch.from_numpy(style).cuda(), alpha=0.8, want_info=True)
    eng.check_device()
    got = out.cpu().numpy()
    noise = np.abs(o32 - o64).max()
    err = np.abs(got - o64).max()
    print("free-running 5-level: engine-vs-fp64 oracle %.3e ; oracle fp32-vs-fp64 %.3e" % (err, noise))
    for lvl, inf in zip(eng.last_info, info):
        k = lvl.cpu().numpy()
        assert (k[0], k[1]) == (inf["k_c"], inf["k_s"])
    assert err <= max(1e-3, FREE_RUN_NOISE_FACTOR * noise)


@pytest.mark.parametrize("path", PIPE_GOLDEN, ids=[os.path.basename(p)[9:-4] for p in PIPE_GOLDEN])
def test_engine_vs_reference_code_golden(path):
    """Engine vs fixtures computed by the reference's own model.py/ops.py/vgg_normalised.py (tests/golden/make_pipeline_golden.py)."""
    g, targets, w = load_pipeline_fixture(path)
    alpha, adain = float(g["alpha"]), bool(g["adain"])
    eng = Engine(w, targets, semantics="tf")
    cap = {}
    from tests.test_oracle import swap_kwargs
    out = eng.stylize(torch.from_numpy(g["content"][None]).cuda(), torch.from_numpy(g["style"][None]).cuda(), alpha=alpha,
                      adain=adain, want_info=True, capture=cap, **swap_kwargs(g))
    eng.check_device()
    got = out.cpu().numpy()
    assert got.shape == g["out_ref_fp64"].shape
    # level 0 has no chained amplification: the transformed feature (decoder input, model.py:150-158) must meet 1e-3
    t0 = eng.act_to_f32(cap["transformed"][0]).cpu().numpy()
    e0 = np.abs(t0 - g["lvl0_decoder_input"]).max()
    d0 = np.abs(cap["level_output"][0].cpu().numpy() - (np.clip(g["lvl0_decoded"], 0, 1) if len(targets) > 1 else g["lvl0_decoded"])).max()
    if not adain:
        ks = [tuple(int(v) for v in lvl.cpu().numpy()[:2]) for lvl in eng.last_info]
        assert ks == [tuple(r) for r in g["k"].tolist()]
    noise = np.abs(g["out_ref_fp32"] - g["out_ref_fp64"]).max()
    err = np.abs(got - g["out_ref_fp64"]).max()
    print("level-0 transform %.2e  level-0 decoded %.2e  final %.2e (reference fp32-vs-fp64 %.2e)" % (e0, d0, err, noise))
    assert e0 <= 1e-3 and d0 <= 1e-3
    assert err <= max(1e-3, FREE_RUN_NOISE_FACTOR * noise)


def test_batch_equals_single_frames_and_u8_postprocess(weights):
    eng = Engine(weights, ALL, semantics="tf")
    contents = _imgs(3, 64, 5)
    styles = _imgs(3, 64, 9)
    outs = eng.stylize(torch.from_numpy(contents).cuda(), torch.from_numpy(styles).cuda(), alpha=0.7).cpu().numpy()
    for i in range(3):
        o = eng.stylize(torch.from_numpy(contents[i:i + 1]).cuda(), torch.from_numpy(styles[i:i + 1]).cuda(), alpha=0.7)
        # same kernels per frame; the only batch dependence is the order of the fp64 atomics in the covariance
        # sums (a last-bit effect that the 5 chained random-weight levels amplify)
        assert np.abs(o.cpu().numpy()[0] - outs[i]).max() <= 1e-3
    shared = eng.stylize(torch.from_numpy(contents).cuda(), torch.from_numpy(styles[:1]).cuda(), alpha=0.7).cpu().numpy()
    assert np.abs(shared[0] - outs[0]).max() <= 1e-3
    u8 = eng.to_u8(torch.from_numpy(outs).cuda()).cpu().numpy()
    assert np.array_equal(u8, nets.postprocess(outs))                 # wct.py:66-68
    eng.check_device()


def test_wct_predict_surface(weights):
    wct = WCT(checkpoints=None, relu_targets=["relu2_1", "relu1_1"], vgg_path=None, device="/gpu:0", weights=weights)
    c, s = _imgs(1, 48, 1)[0], _imgs(1, 40, 2)[0]
    out = wct.predict(c, s, alpha=0.6)
    assert out.dtype == np.uint8 and out.shape == (48, 48, 3)
    ref = nets.pipeline(c, s, weights, ["relu2_1", "relu1_1"], alpha=0.6, semantics="tf", dtype=np.float64)
    diff = np.abs(out.astype(int) - nets.postprocess(ref[0]).astype(int))
    assert diff.max() <= 1                                            # 1e-3 float error may flip a u8 LSB (SURVEY a2)
    # --swap5 only acts at relu5_1 (model.py:144-158): without that target it changes nothing ...
    assert np.array_equal(wct.predict(c, s, alpha=0.6, swap5=True, ss_alpha=0.5), out)
    # ... while with relu5_1 and a stride the content is centre-cropped to a size the patches tile (wct.py:84-90,
    # utils.swap_filter_fit): 80x112 -> relu5_1 encoding 5x7; patch 3 / stride 2 tiles 5x7; 96x112 (6x7) is cropped to 80x112
    from wct_tf_b200.imageio import swap_filter_fit
    assert swap_filter_fit(96, 112, 3, 2) == (True, 80, 112) and swap_filter_fit(80, 112, 3, 2) == (False, 80, 112)
    t5 = ["relu5_1", "relu1_1"]
    w5 = make_synthetic_weights(15, relu_targets=t5)
    wct2 = WCT(checkpoints=None, relu_targets=t5, vgg_path=None, device="/gpu:0", weights=w5, ss_patch_size=3, ss_stride=2)
    c2, s2 = _imgs(1, 112, 3)[0][:96], _imgs(1, 112, 4)[0]
    o2 = wct2.predict(c2, s2, alpha=0.7, swap5=True, ss_alpha=0.6)
    assert o2.shape == (80, 112, 3)
    crop = c2[8:88]                                                    # centre crop of the 96 rows to 80
    r2 = nets.pipeline(crop, s2, w5, t5, alpha=0.7, semantics="tf", dtype=np.float64, swap5=True, ss_alpha=0.6, ss_patch_size=3, ss_stride=2)
    assert r2.shape[1:3] == (80, 112)
    out2 = wct.predict(c, s, alpha=0.6, adain=True)
    ref2 = nets.pipeline(c, s, weights, ["relu2_1", "relu1_1"], alpha=0.6, adain=True, dtype=np.float64)
    assert np.abs(out2.astype(int) - nets.postprocess(ref2[0]).astype(int)).max() <= 1


def test_grouped_streams_equal_single_stream(weights):
    """Engine.groups > 1 only changes the schedule (sub-batches on independent stream pairs)."""
    eng = Engine(weights, ALL, semantics="tf")
    contents = torch.from_numpy(_imgs(5, 64, 21)).cuda()
    styles = torch.from_numpy(_imgs(5, 64, 22)).cuda()
    ref = eng.stylize(contents, styles, alpha=0.8).cpu().numpy()
    eng.groups = 2
    got2 = eng.stylize(contents, styles, alpha=0.8).cpu().numpy()
    eng.groups = 4
    got4 = eng.stylize(contents, styles[:1], alpha=0.8).cpu().numpy()
    eng.groups = 1
    ref4 = eng.stylize(contents, styles[:1], alpha=0.8).cpu().numpy()
    eng.check_device()
    assert got2.shape == ref.shape and np.abs(got2 - ref).max() <= 1e-3
    assert np.abs(got4 - ref4).max() <= 1e-3


@pytest.mark.parametrize("hw,shw", [((70, 130), (50, 66)), ((33, 47), (128, 40)), ((16, 16), (16, 20))])
def test_odd_sizes_full_pipeline_vs_oracle(weights, hw, shw):
    """Sizes that are not multiples of 16: MaxPooling2D(padding='same') rounds up and UpSampling2D doubles,
    so the output grows like the reference graph's (vgg_normalised.py:42, model.py:293)."""
    targets = ["relu4_1", "relu2_1", "relu1_1"]
    rng = np.random.default_rng(hw[0])
    content = rng.integers(0, 256, (1, hw[0], hw[1], 3), dtype=np.uint8)
    style = rng.integers(0, 256, (1, shw[0], shw[1], 3), dtype=np.uint8)
    eng = Engine(weights, targets, semantics="tf")
    cap = {}
    out = eng.stylize(torch.from_numpy(content).cuda(), torch.from_numpy(style).cuda(), alpha=0.6, want_info=True, capture=cap)
    eng.check_device()
    sfe = nets.encode(nets.preprocess(style).astype(np.float64), weights, targets, np.float64)
    for i, relu in enumerate(targets):
        x = cap["level_input"][i].cpu().numpy().astype(np.float64)
        cf = nets.encode(x, weights, [relu], np.float64)[relu]
        f, info = ref_ops.wct_tf(cf, sfe[relu], 0.6, return_info=True)
        _, info32 = ref_ops.wct_tf(cf.astype(np.float32), sfe[relu].astype(np.float32), 0.6, return_info=True)
        if not (ref_ops.spectral_gap_ok(info["wc"]) and ref_ops.spectral_gap_ok(info["ws"])) or \
                (info32["k_c"], info32["k_s"]) != (info["k_c"], info["k_s"]):
            # rank-deficient map (HW < C): the null eigenvalues sit at the fp32 noise floor eps*lambda_max*sqrt(C)
            # ~ 1e-5, so the reference's OWN fp32 arithmetic does not agree with its fp64 run on k
            pytest.skip("ill-posed vector for any fp32 implementation (reference fp32 k != fp64 k)")
        k = eng.last_info[i].cpu().numpy()
        assert (k[0], k[1]) == (info["k_c"], info["k_s"])
        y = nets.decode(f, weights, relu, np.float64)
        if i < len(targets) - 1:
            y = np.clip(y, 0, 1)
        got = cap["level_output"][i].cpu().numpy()
        assert got.shape == y.shape
        assert np.abs(got - y).max() <= 1e-3
    ref_shape = nets.pipeline(content[0], style[0], weights, targets, alpha=0.6, semantics="tf", dtype=np.float32).shape
    assert tuple(out.shape) == tuple(ref_shape)


def test_cli_end_to_end(tmp_path):
    """stylize.py with the reference's flags on real image files (synthetic weights)."""
    from PIL import Image
    import stylize
    rng = np.random.default_rng(0)
    cdir, sdir, odir = tmp_path / "c", tmp_path / "s", tmp_path / "o"
    cdir.mkdir(); sdir.mkdir()
    Image.fromarray(rng.integers(0, 256, (40, 56, 3), dtype=np.uint8)).save(cdir / "a.png")
    Image.fromarray(rng.integers(0, 256, (64, 48, 3), dtype=np.uint8)).save(sdir / "st.png")
    stylize.main(["--synthetic-weights", "42", "--relu-targets", "relu2_1", "relu1_1", "--content-path", str(cdir),
                  "--style-path", str(sdir / "st.png"), "--out-path", str(odir), "--alpha", "0.7", "--style-size", "32",
                  "--passes", "2", "--concat"])
    out = np.asarray(Image.open(odir / "a_st.png"))      # {content}_{style}{ext}, stylize.py:114
    assert out.shape == (40, 40 + 56, 3) and out.dtype == np.uint8


def test_wct_from_reference_weight_files(tmp_path):
    """WCT(checkpoints=<TF checkpoint dirs>, vgg_path=<.t7>) -- the reference's own constructor arguments (wct.py:17-18)
    -- gives bit-identical output to the same weights passed as a dict."""
    from tests.t7_writer import write_vgg_t7
    from tests.tf_bundle_writer import write_bundle
    targets = ["relu3_1", "relu1_1"]
    w = make_synthetic_weights(21, relu_targets=targets)
    write_vgg_t7(str(tmp_path / "vgg_normalised.t7"), w["vgg"])
    dirs = []
    for t in targets:
        tensors = {}
        for l in w["decoders"][t]:
            scope = "encoder_decoder_%s/decoder_%s/decoder_model_%s/%s/%s" % (t, t, t, l["name"], l["name"])
            tensors[scope + "/kernel"], tensors[scope + "/bias"] = l["kernel"], l["bias"]
        write_bundle(str(tmp_path / t / "model.ckpt-1"), tensors)
        dirs.append(str(tmp_path / t))
    c, s = _imgs(1, 40, 3)[0], _imgs(1, 56, 4)[0]
    a = WCT(checkpoints=dirs, relu_targets=targets, vgg_path=str(tmp_path / "vgg_normalised.t7")).predict(c, s, alpha=0.7)
    b = WCT(checkpoints=None, relu_targets=targets, vgg_path=None, weights=w).predict(c, s, alpha=0.7)
    assert a.dtype == np.uint8 and np.array_equal(a, b)


def test_video_driver_matches_per_frame_predict(tmp_path, weights):
    """stylize_video.py on a directory of frames == WCT.predict frame by frame (the reference's loop, stylize_video.py:112-135),
    up to the 1-LSB uint8 effect of batch-vs-single fp64-atomic ordering."""
    from PIL import Image
    import stylize_video as V
    frames = tmp_path / "clip"
    frames.mkdir()
    imgs = _imgs(5, 64, 77)
    for i in range(5):
        Image.fromarray(imgs[i]).save(str(frames / ("frame_%d.png" % (i + 1))))
    style = _imgs(1, 48, 78)[0]
    Image.fromarray(style).save(str(tmp_path / "style.png"))
    targets = ["relu3_1", "relu2_1", "relu1_1"]
    n = V.main(["--relu-targets"] + targets + ["--in-path", str(frames), "--style-path", str(tmp_path / "style.png"),
                "--out-path", str(tmp_path / "out"), "--batch", "3", "--alpha", "0.7"],
               wct_factory=lambda a: WCT(checkpoints=None, relu_targets=targets, vgg_path=None, weights=weights))
    assert n == 5
    ref = WCT(checkpoints=None, relu_targets=targets, vgg_path=None, weights=weights)
    for i in range(5):
        got = np.array(Image.open(str(tmp_path / "out" / "clip_style_frames" / ("frame_%d.png" % (i + 1)))))
        want = ref.predict(imgs[i], style, alpha=0.7)
        assert got.shape == want.shape and np.abs(got.astype(int) - want.astype(int)).max() <= 1


def test_passes_on_device_equal_host_round_trips(weights):
    """predict_batch(passes=2) (frames stay on the GPU between passes) == predict(predict(x)) (stylize.py:102-104)."""
    targets = ["relu2_1", "relu1_1"]
    wct = WCT(checkpoints=None, relu_targets=targets, vgg_path=None, weights=weights)
    c, s = _imgs(2, 48, 31), _imgs(1, 40, 32)
    once = wct.predict_batch(c, s, alpha=0.6)
    twice = wct.predict_batch(once, s, alpha=0.6)
    fused = wct.predict_batch(c, s, alpha=0.6, passes=2)
    assert np.array_equal(fused, twice)
    dev = wct.predict_batch(c, s, alpha=0.6, passes=2, return_device=True)
    assert dev.is_cuda and dev.dtype == torch.uint8 and np.array_equal(dev.cpu().numpy(), twice)


def test_pool_fused_encoder_matches_separate_pool(weights):
    """Engine(fuse_pool=True) (MaxPooling2D in the conv epilogue, WCTB200_POOL2) vs Engine(fuse_pool=False).  The pooled maps
    are equal BY VALUE (tests/test_gpu_layers.py::test_conv3x3_pool2_equals_conv_then_maxpool), but a value that sits exactly
    between two fp16 numbers can be stored as (hi, +half ulp) or (hi + ulp, -half ulp): the separate pool re-splits the merged
    value (ties to even), the fused epilogue splits the fp32 accumulator, so the NEXT conv sees different operand bits and its
    dropped lo*lo term differs at the 2^-22 level.  Encoder outputs must therefore agree to ~1e-6 relative, not bit for bit."""
    targets = ["relu5_1", "relu4_1", "relu3_1", "relu2_1", "relu1_1"]
    a = Engine(weights, targets, fuse_pool=True)
    b = Engine(weights, targets, fuse_pool=False)
    for (hw, seed) in [((64, 96), 5), ((51, 70), 6), ((130, 67), 7)]:
        rng = np.random.default_rng(seed)
        img = torch.from_numpy(rng.random((2,) + hw + (3,)).astype(np.float32)).cuda()
        for t in targets:
            fa, _ = a.encode(img, t)
            fb, _ = b.encode(img, t)
            xa, xb = a.act_to_f32(fa), b.act_to_f32(fb)
            assert xa.shape == xb.shape
            assert (xa - xb).abs().max().item() <= 2e-6 * (1.0 + xb.abs().max().item()), (hw, t)
    a.check_device()
