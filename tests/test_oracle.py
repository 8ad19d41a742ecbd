"""CPU tests: pin the oracle restatement against the reference's own outputs
(committed golden vectors made by tests/golden/make_golden.py from
/root/reference/ops.py:92-140) and check its internal consistency."""
import glob
import os

import numpy as np
import pytest

from oracle import nets, ref_ops

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "wct_np_*.npz")))


def test_golden_present():
    assert len(GOLDEN) >= 5


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[7:-4] for p in GOLDEN])
def test_wct_np_restatement_matches_reference_golden(path):
    g = np.load(path)
    out, info = ref_ops.wct_np(g["content"], g["style"], float(g["alpha"]), return_info=True)
    assert out.dtype == np.float32  # ops.py:140
    assert info["k_c"] == int(g["k_c"]) and info["k_s"] == int(g["k_s"])
    # same arithmetic, same LAPACK: the fp32 restatement reproduces the reference run to fp32 noise
    assert np.abs(out - g["out_ref_fp32"]).max() <= 2e-4
    out64 = ref_ops.wct_np(g["content"].astype(np.float64), g["style"].astype(np.float64), float(g["alpha"]))
    assert np.abs(out64 - g["out_ref_fp64"]).max() <= 1e-6
    assert ref_ops.spectral_gap_ok(g["wc"]) and ref_ops.spectral_gap_ok(g["ws"])


REF_READS = os.path.join(os.path.dirname(__file__), "golden", "reference_reads.npz")


def test_reference_wct_np_reproduces_fixture():
    """The reference's own ops.wct_np, re-run on a fixture's inputs (tests/golden/make_reference_reads.py), returns the
    fixture's out_ref_fp32 bit for bit."""
    from tests.golden.make_reference_reads import array_digest
    ref = np.load(REF_READS)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", str(ref["wct_np_fixture"])))
    assert array_digest(g["out_ref_fp32"]) == str(ref["wct_np_out_sha256"])


def test_np_vs_tf_semantics_differ_only_as_documented():
    # SURVEY 8a "np-vs-tf deltas": at alpha=1 the blend term vanishes; the remaining
    # difference is eps placement (1e-8 on cov vs 1e-5 on eigenvalues)
    g = np.load(GOLDEN[0])
    c, s = g["content"].astype(np.float64), g["style"].astype(np.float64)
    a = ref_ops.wct_generic(c, s, 1.0, eps_cov=0.0, eps_eig=0.0, readd_content_mean=False)
    b = ref_ops.wct_generic(c, s, 1.0, eps_cov=0.0, eps_eig=0.0, readd_content_mean=True)
    assert np.abs(a - b).max() < 1e-12
    t = ref_ops.wct_tf(c, s, 0.5)
    n = ref_ops.wct_generic(c, s, 0.5, eps_cov=1e-8, eps_eig=0.0, readd_content_mean=False)
    mc = c.reshape(-1, c.shape[-1]).mean(0)
    assert np.allclose(t - n, 0.5 * mc, atol=1e-9)


def test_adain_matches_definition():
    rng = np.random.default_rng(0)
    c = rng.random((1, 6, 5, 8)); s = rng.random((1, 4, 7, 8)) * 3 + 1
    y = ref_ops.adain(c, s, 1.0, epsilon=0.0)
    assert np.allclose(y.mean((1, 2)), s.mean((1, 2)))
    assert np.allclose(y.var((1, 2)), s.var((1, 2)))
    y2 = ref_ops.adain(c, s, 0.25)
    y1 = ref_ops.adain(c, s, 1.0)
    assert np.allclose(y2, 0.25 * y1 + 0.75 * c)


def test_decoder_layer_names_match_reference_table():
    # model.py:283-298: relu5_1 -> layers 0..15 + output 16 (convs and upsamples both counted)
    l5 = nets.decoder_layers("relu5_1")
    assert [n for _, n, _, _ in l5] == ["relu5_1_%d" % i for i in range(17)]
    assert [t for t, _, _, _ in l5].count("up") == 4
    assert l5[-1][2] == 3 and l5[-1][3] is False
    assert [n for _, n, _, _ in nets.decoder_layers("relu1_1")] == ["relu1_1_0", "relu1_1_1"]


def test_encoder_shapes_and_pool_same():
    from wct_tf_b200.weights import make_synthetic_weights
    w = make_synthetic_weights(0)
    x = np.random.default_rng(0).random((1, 22, 18, 3)).astype(np.float32)
    f = nets.encode(x, w, ["relu1_1", "relu2_1", "relu3_1", "relu4_1", "relu5_1"])
    assert f["relu1_1"].shape == (1, 22, 18, 64)
    assert f["relu2_1"].shape == (1, 11, 9, 128)
    assert f["relu3_1"].shape == (1, 6, 5, 256)   # ceil: MaxPooling2D(padding='same')
    assert f["relu4_1"].shape == (1, 3, 3, 512)
    assert f["relu5_1"].shape == (1, 2, 2, 512)
    y = nets.decode(f["relu3_1"], w, "relu3_1")
    assert y.shape == (1, 24, 20, 3)


# ---- whole-path fixtures produced by the reference's OWN model.py / ops.py / vgg_normalised.py / torchfile.py
# (imported unmodified, evaluated over tests/golden/np_tf1.py; see tests/golden/make_pipeline_golden.py)
PIPE_GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "pipeline_*.npz")))


def load_pipeline_fixture(path):
    from tests.golden.make_pipeline_golden import weight_checksum
    from wct_tf_b200.weights import make_synthetic_weights
    g = np.load(path)
    targets = [str(t) for t in g["relu_targets"]]
    w = make_synthetic_weights(int(g["seed"]), relu_targets=targets)
    assert abs(weight_checksum(w) - float(g["wsum"])) <= 1e-9 * float(g["wsum"]), "synthetic weight generator drifted"
    return g, targets, w


def swap_kwargs(g):
    """--swap5 arguments of a fixture (older fixtures carry no patch / stride: the reference's defaults 3 / 1)."""
    kw = dict(swap5=bool(g["swap5"]), ss_alpha=float(g["ss_alpha"]))
    if "ss_patch_size" in g.files:
        kw.update(ss_patch_size=int(g["ss_patch_size"]), ss_stride=int(g["ss_stride"]))
    return kw


def test_pipeline_golden_present():
    assert len(PIPE_GOLDEN) >= 5


@pytest.mark.parametrize("path", PIPE_GOLDEN, ids=[os.path.basename(p)[9:-4] for p in PIPE_GOLDEN])
def test_oracle_pipeline_matches_reference_code_fixture(path):
    """oracle.nets.pipeline (encoder + wct_tf | adain + decoder + level wiring) == the reference's WCTModel code."""
    g, targets, w = load_pipeline_fixture(path)
    alpha, adain = float(g["alpha"]), bool(g["adain"])
    swap = swap_kwargs(g)
    o64, info = nets.pipeline(g["content"], g["style"], w, targets, alpha=alpha, adain=adain, semantics="tf",
                              dtype=np.float64, return_info=True, **swap)
    assert o64.shape == g["out_ref_fp64"].shape
    assert np.abs(o64 - g["out_ref_fp64"]).max() <= 1e-9          # same algorithm in exact arithmetic
    if not adain:
        assert [(i["k_c"], i["k_s"]) for i in info] == [tuple(r) for r in g["k"].tolist()]
    o32 = nets.pipeline(g["content"], g["style"], w, targets, alpha=alpha, adain=adain, semantics="tf", dtype=np.float32, **swap)
    noise = np.abs(g["out_ref_fp32"] - g["out_ref_fp64"]).max()     # the reference code's own fp32 rounding (chained levels amplify it)
    assert np.abs(o32 - g["out_ref_fp32"]).max() <= max(1e-4, 4 * noise)


def test_reference_code_reproduces_pipeline_fixture():
    """The reference's WCTModel code (over tests/golden/np_tf1.py), re-run in float64 on a fixture's inputs and weights
    (tests/golden/make_reference_reads.py), returns the fixture's out_ref_fp64."""
    ref = np.load(REF_READS)
    g, _, _ = load_pipeline_fixture(os.path.join(os.path.dirname(__file__), "golden", str(ref["pipeline_fixture"])))
    out = ref["pipeline_out_fp64"]
    assert out.shape == g["out_ref_fp64"].shape
    assert np.abs(out - g["out_ref_fp64"]).max() <= 1e-12


# ---------------------------------------------------------------------------
# scope row 8f-3: the image steps of the CLI
# ---------------------------------------------------------------------------
RESIZE_CASES = [(37, 53, 20, 29), (37, 53, 74, 91), (64, 64, 64, 64), (100, 40, 512, 205), (513, 301, 256, 150), (5, 7, 1, 1),
                (1, 1, 9, 4), (360, 640, 256, 455), (33, 70, 33, 35), (33, 70, 66, 70), (300, 400, 299, 401), (2, 3, 64, 64)]


@pytest.mark.parametrize("h,w,oh,ow", RESIZE_CASES)
def test_resample_oracle_is_pillow_bit_for_bit(h, w, oh, ow):
    """The restatement of Pillow's 8-bit bilinear ImagingResample (what scipy.misc.imresize(interp='bilinear') ran,
    utils.py:48,67) against the Pillow installed in this image: identical bytes for down-, up-scaling, identity and
    degenerate sizes."""
    from PIL import Image
    from oracle import image_ops
    img = np.random.default_rng(h * 1000 + w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    want = np.asarray(Image.fromarray(img).resize((ow, oh), Image.BILINEAR))
    assert np.array_equal(image_ops.resample_bilinear_u8(img, oh, ow), want)


def test_image_oracle_helpers_follow_the_reference_rules():
    from oracle import image_ops
    img = np.random.default_rng(3).integers(0, 256, (40, 64, 3), dtype=np.uint8)
    assert image_ops.resize_to(img, 20).shape == (20, 32, 3)                     # short side, aspect kept (utils.py:55-67)
    assert image_ops.resize_to(img.transpose(1, 0, 2), 20).shape == (32, 20, 3)
    assert np.array_equal(image_ops.center_crop(img, 32), img[4:36, 16:48])       # utils.py:29-38
    assert image_ops.center_crop(img[:10, :10], 16).shape == (16, 16, 3)          # too small -> upscale first
    assert image_ops.center_crop_to(img, 48, 64).shape == (48, 64, 3)             # utils.py:40-53 (upscale by the larger ratio)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "coral_keep_colors.npz"))
    assert np.abs(image_ops.coral(g["style"] / 255., g["content"] / 255.) - g["coraled"]).max() < 1e-9   # reference's coral.py output
    assert np.array_equal(image_ops.preserve_colors(g["style"], g["content"]), g["out"])


def test_resample_oracle_random_sizes_against_pillow():
    """40 random (size, target) pairs incl. extreme aspect ratios and 1-4 channels: the oracle stays bit-identical to Pillow."""
    from PIL import Image
    from oracle import image_ops
    rng = np.random.default_rng(2024)
    for _ in range(40):
        h, w = int(rng.integers(1, 90)), int(rng.integers(1, 90))
        oh, ow = int(rng.integers(1, 120)), int(rng.integers(1, 120))
        c = int(rng.choice([1, 3, 4]))
        img = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
        mode = {1: "L", 3: "RGB", 4: "RGBX"}[c]
        pil = Image.fromarray(img[:, :, 0] if c == 1 else img, mode)
        want = np.asarray(pil.resize((ow, oh), Image.BILINEAR)).reshape(oh, ow, c)
        assert np.array_equal(image_ops.resample_bilinear_u8(img, oh, ow), want), (h, w, c, oh, ow)
