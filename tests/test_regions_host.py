"""Spatial control, host side: the label resize rule, the per-region oracle, the mask reader and the CLI flags."""
import os

import numpy as np
import pytest
from PIL import Image

import stylize
from oracle import ref_ops, regions
from wct_tf_b200 import _capi
from wct_tf_b200 import imageio as io

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SIZES = [((37, 53), (9, 14)), ((9, 14), (37, 53)), ((20, 30), (20, 30)), ((1, 1), (5, 7)), ((7, 5), (1, 1)), ((13, 17), (7, 9))]


@pytest.mark.parametrize("src,dst", SIZES)
def test_nearest_labels_integer_rule(src, dst):
    rng = np.random.default_rng(src[0] * 100 + dst[1])
    lab = rng.integers(0, 256, src, dtype=np.uint8)
    got = regions.nearest_labels(lab, *dst)
    want = np.empty(dst, dtype=np.uint8)
    for y in range(dst[0]):
        for x in range(dst[1]):
            want[y, x] = lab[(y * src[0]) // dst[0], (x * src[1]) // dst[1]]
    assert np.array_equal(got, want)


def _feats(seed, h=8, w=9, c=16):
    rng = np.random.default_rng(seed)
    return np.maximum(rng.standard_normal((1, h, w, c)) @ rng.standard_normal((c, c)) / 4 + 0.3, 0)


@pytest.mark.parametrize("sem", ["tf", "np"])
def test_one_label_mask_is_the_plain_transform(sem):
    cf, sf = _feats(0), _feats(1, 11, 7)
    got, info = regions.wct_regions(cf, np.zeros(cf.shape[1:3], np.uint8), [sf], 0.7, sem)
    fn = ref_ops.wct_tf if sem == "tf" else ref_ops.wct_np
    want = fn(cf, sf, 0.7)
    assert np.array_equal(got, np.asarray(want, dtype=got.dtype)) or np.abs(got - want).max() <= 1e-6
    assert info[0]["n"] == cf.shape[1] * cf.shape[2]


def test_keep_pixels_and_tiny_regions_untouched():
    cf, s0, s1 = _feats(2), _feats(3), _feats(4)
    lab = np.full(cf.shape[1:3], 7, np.uint8)       # keep everywhere ...
    lab[:4] = 0                                      # ... but region 0 on the top half
    lab[6, 3] = 1                                    # region 1: one pixel (n < 2)
    got, info = regions.wct_regions(cf, lab, [s0, s1], 1.0)
    keep = lab != 0
    assert np.array_equal(got[0][keep], cf[0][keep])
    assert not np.allclose(got[0][~keep], cf[0][~keep])
    assert info[1]["n"] == 1 and info[1]["k_c"] == 0
    ad, _ = regions.adain_regions(cf, lab, [s0, s1], 0.5)
    assert np.array_equal(ad[0][keep], cf[0][keep])


def test_mask_reader_modes(tmp_path):
    lab = (np.arange(12 * 10) % 3).astype(np.uint8).reshape(12, 10)
    Image.fromarray(lab, mode="L").save(tmp_path / "m_l.png")
    p = Image.fromarray(lab, mode="P")
    p.putpalette([0, 0, 0, 255, 0, 0, 0, 255, 0] + [0] * (253 * 3))
    p.save(tmp_path / "m_p.png")
    Image.fromarray(np.stack([lab] * 3, -1), mode="RGB").save(tmp_path / "m_rgb.png")
    assert np.array_equal(io.get_mask(str(tmp_path / "m_l.png")), lab)
    assert np.array_equal(io.get_mask(str(tmp_path / "m_p.png")), lab)
    with pytest.raises(ValueError, match="mode"):
        io.get_mask(str(tmp_path / "m_rgb.png"))


def test_mask_flags():
    base = ["--relu-targets", "relu1_1", "--content-path", "c.png", "--out-path", "o"]
    a = stylize.parse_args(base + ["--mask-path", "m.png", "--mask-styles", "a.png", "b.png", "--passes", "2", "--keep-colors"])
    assert a.mask_path == "m.png" and a.mask_styles == ["a.png", "b.png"] and a.passes == 2 and a.keep_colors
    assert stylize.parse_args(base).mask_path is None
    for extra in (["--swap5"], ["--concat"], ["-r", "2"]):
        with pytest.raises(SystemExit):
            stylize.parse_args(base + ["--mask-path", "m.png", "--mask-styles", "a.png"] + extra)
    with pytest.raises(SystemExit):
        stylize.parse_args(base + ["--mask-path", "m.png"])
    with pytest.raises(SystemExit):
        stylize.parse_args(base + ["--mask-path", "m.png", "--mask-styles"] + ["s.png"] * 9)


def test_region_entry_points_declared():
    with open(os.path.join(ROOT, "include", "wctb200.h")) as f:
        header = f.read()
    for name in ("wctb200_labels_resize_nearest", "wctb200_wct_regions_workspace_bytes", "wctb200_wct_apply_regions",
                 "wctb200_adain_regions"):
        assert name in _capi.SIGNATURES and (name + "(") in header
