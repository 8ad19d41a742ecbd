"""Spatial control on the GPU: label resize kernel, per-region WCT / AdaIN levels against the fp64 oracle
(oracle/regions.py), keep pixels equal by value, the reduction to the unmasked path, batch invariance, the CLI."""
import ctypes
import os

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import nets, ref_ops, regions
from tests import gpu_util as U
from wct_tf_b200 import _capi
from wct_tf_b200.engine import Engine
from wct_tf_b200.weights import make_synthetic_weights
from wct_tf_b200.wct import WCT

pytestmark = pytest.mark.gpu
ALL = ["relu5_1", "relu4_1", "relu3_1", "relu2_1", "relu1_1"]
SEM = dict(tf=(1e-8, 0.0, 1), np=(0.0, 1e-5, 0))


@pytest.fixture(scope="module")
def weights():
    return make_synthetic_weights(42)


def _resize_dev(lab, h, w):
    src = U.dev(lab)
    n = lab.shape[0]
    dst = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    _capi.check(U.lib().wctb200_labels_resize_nearest(src.data_ptr(), n, lab.shape[1], lab.shape[2], h, w, dst.data_ptr(),
                                                        U.stream()))
    torch.cuda.synchronize()
    return dst.cpu().numpy()


@pytest.mark.parametrize("src,dst", [((37, 53), (9, 14)), ((9, 14), (37, 53)), ((20, 30), (20, 30)), ((1, 1), (5, 7)),
                                     ((7, 5), (1, 1)), ((13, 17), (7, 9)), ((512, 512), (32, 32))])
def test_labels_resize_kernel_equals_integer_rule(src, dst):
    rng = np.random.default_rng(src[0] + 7 * dst[1])
    lab = rng.integers(0, 256, (3,) + src, dtype=np.uint8)          # a batch of 3 maps
    assert np.array_equal(_resize_dev(lab, *dst), regions.nearest_labels(lab, *dst))


# ---- one level -------------------------------------------------------------------------------------------------------
def _mask(kind, h, w, R, rng):
    y, x = np.mgrid[0:h, 0:w]
    if kind == "blobs":
        lab = np.full((h, w), R, np.uint8)                             # keep label R outside the blobs
        for r in range(R):
            cy, cx = rng.integers(0, h), rng.integers(0, w)
            lab[(y - cy) ** 2 + (x - cx) ** 2 <= (0.35 * max(h, w)) ** 2] = r
        lab[0, 0] = R                                                  # at least one keep pixel
        return lab
    if kind == "checker":                                              # every 128-position tile is a boundary tile
        return ((x + y) % R).astype(np.uint8)
    if kind == "halves":
        return (x * R // w).astype(np.uint8)
    if kind == "tiny":                                                 # region 0 everywhere but 2 pixels of region 1
        lab = np.zeros((h, w), np.uint8)
        lab[3, 4] = lab[h - 2, w - 1] = 1
        if R > 2:
            lab[h // 2, w // 2] = 2                                    # one pixel: n_r = 1, copied
        return lab
    if kind == "empty":                                                # region R-1 has no pixel; a keep stripe
        lab = (x * max(R - 1, 1) // w).astype(np.uint8)
        lab[:, :2] = 200
        return lab
    raise ValueError(kind)


def _feats(n, h, w, c, seed):
    rng = np.random.default_rng(seed)
    f = rng.standard_normal((n, h, w, c)) @ (rng.standard_normal((c, c)) / np.sqrt(c)) + 0.3
    return np.maximum(f, 0).astype(np.float32)


def _run_regions(content, labels, styles, alpha, mode):
    """wctb200_wct_apply_regions (mode 'tf' / 'np') or wctb200_adain_regions ('adain') on SPF16 copies of the inputs."""
    n, h, w, c = content.shape
    R = len(styles)
    cin = U.act_from_numpy(content)
    out = U.act_alloc(n, h, w, c)
    lab = U.dev(labels)
    ws = torch.empty(U.lib().wctb200_wct_regions_workspace_bytes(c, n, R), dtype=torch.uint8, device="cuda")
    kbuf = torch.full((2 * n * R,), -1, dtype=torch.int32, device="cuda")
    sbufs = [U.act_from_numpy(s) for s in styles]
    if mode == "adain":
        ptrs = (ctypes.c_void_p * R)(*[b.data_ptr() for b in sbufs])
        hw = (ctypes.c_int * (2 * R))(*[v for s in styles for v in s.shape[1:3]])
        _capi.check(U.lib().wctb200_adain_regions(cin.data_ptr(), n, h, w, c, lab.data_ptr(), R, ptrs, hw, float(alpha), 1e-5,
                                                  out.data_ptr(), ws.data_ptr(), ws.numel(), U.stream()))
        kbuf = None
    else:
        eps_cov, eps_eig, readd = SEM[mode]
        states = []
        for s, b in zip(styles, sbufs):
            st = torch.empty(U.lib().wctb200_wct_style_state_bytes(c, 1), dtype=torch.uint8, device="cuda")
            sws = torch.empty(U.lib().wctb200_wct_workspace_bytes(c, 0, 1), dtype=torch.uint8, device="cuda")
            _capi.check(U.lib().wctb200_wct_style_prepare(b.data_ptr(), 1, s.shape[1], s.shape[2], c, eps_cov, eps_eig, 1e-5,
                                                          st.data_ptr(), sws.data_ptr(), sws.numel(), U.stream()))
            states.append((st, sws))
        ptrs = (ctypes.c_void_p * R)(*[st.data_ptr() for st, _ in states])
        _capi.check(U.lib().wctb200_wct_apply_regions(cin.data_ptr(), n, h, w, c, lab.data_ptr(), R, ptrs, float(alpha), eps_cov,
                                                      eps_eig, 1e-5, readd, out.data_ptr(), kbuf.data_ptr(), ws.data_ptr(),
                                                      ws.numel(), U.stream()))
    U.check_device()
    got = U.act_to_numpy(out, n, h, w, c)
    padded = U.act_raw_padded(out, n, h, w, c)
    assert np.isfinite(padded).all()
    assert np.array_equal(padded, np.pad(padded[:, 1:-1, 1:-1], ((0, 0), (1, 1), (1, 1), (0, 0)), mode="reflect"))
    return got, padded, U.act_raw_padded(cin, n, h, w, c), (kbuf.cpu().numpy() if kbuf is not None else None)


LEVEL_CASES = [
    # (C, h, w, R, mask, mode): the C = 512 / 256 cases have regions of n_r <= C pixels (rank-deficient: eigensolver fallback)
    (64, 40, 44, 1, "blobs", "tf"),
    (64, 40, 44, 3, "checker", "np"),
    (128, 30, 34, 2, "blobs", "tf"),
    (128, 30, 34, 3, "tiny", "tf"),
    (256, 24, 26, 2, "halves", "np"),
    (256, 10, 26, 3, "empty", "tf"),
    (512, 24, 24, 2, "halves", "tf"),
    (512, 20, 22, 3, "blobs", "np"),
    (512, 20, 22, 2, "checker", "tf"),
    (64, 40, 44, 3, "blobs", "adain"),
    (256, 24, 26, 2, "checker", "adain"),
    (512, 20, 22, 3, "tiny", "adain"),
]


@pytest.mark.parametrize("c,h,w,R,kind,mode", LEVEL_CASES)
def test_region_level_vs_fp64_oracle(c, h, w, R, kind, mode):
    rng = np.random.default_rng(c + R)
    content = _feats(2, h, w, c, c)
    labels = np.stack([_mask(kind, h, w, R, rng), _mask(kind, h, w, R, rng)[::-1].copy()])
    styles = [_feats(1, h + 3 * r, w + 5 - r, c, 100 + r) for r in range(R)]
    alpha = 0.8
    got, padded, pin, k = _run_regions(content, labels, styles, alpha, mode)
    worst = 0.0
    for i in range(2):
        cf = content[i:i + 1].astype(np.float64)
        sf = [s.astype(np.float64) for s in styles]
        if mode == "adain":
            ref, info = regions.adain_regions(cf, labels[i], sf, alpha)
        else:
            ref, info = regions.wct_regions(cf, labels[i], sf, alpha, mode)
        for r in range(R):
            if mode != "adain":
                assert k[i * R + r] == info[r]["k_c"], (i, r, k[i * R + r], info[r]["k_c"])
                assert k[2 * R + i * R + r] == int((labels[i] == r).sum())
                if info[r]["n"] >= 2:
                    assert ref_ops.spectral_gap_ok(info[r]["wc"]) and ref_ops.spectral_gap_ok(info[r]["ws"]), "ill-posed vector"
        worst = max(worst, float(np.abs(got[i:i + 1] - ref).max()))
        # keep pixels and regions of < 2 pixels: equal BY VALUE to the input
        counts = np.bincount(labels[i].ravel(), minlength=256)
        copied = (labels[i] >= R) | (counts[labels[i]] < 2)
        assert np.array_equal(padded[i, 1:-1, 1:-1][copied], pin[i, 1:-1, 1:-1][copied])
    print("C=%d R=%d %s %s: max-abs vs fp64 oracle %.2e" % (c, R, kind, mode, worst))
    assert worst <= 1e-3


# ---- the whole pipeline ----------------------------------------------------------------------------------------------
def _two_regions_and_keep(h, w):
    y, x = np.mgrid[0:h, 0:w]
    lab = np.where(x < w // 2, 0, 1).astype(np.uint8)
    lab[(y - h // 2) ** 2 + (x - w // 2) ** 2 < (h // 5) ** 2] = 9        # keep disc in the middle
    return lab


@pytest.mark.parametrize("sem,adain", [("tf", False), ("np", False), ("tf", True)])
def test_teacher_forced_five_levels_512(weights, sem, adain):
    eng = Engine(weights, ALL, semantics=sem)
    rng = np.random.default_rng(1000)
    content = rng.integers(0, 256, (1, 512, 512, 3), dtype=np.uint8)
    styles = [rng.integers(0, 256, (1, 512 - 64 * r, 512, 3), dtype=np.uint8) for r in range(2)]
    labels = _two_regions_and_keep(512, 512)
    cap = {}
    eng.stylize(torch.from_numpy(content).cuda(), [torch.from_numpy(s).cuda() for s in styles], alpha=0.8, adain=adain,
                want_info=True, capture=cap, labels=torch.from_numpy(labels[None]).cuda())
    eng.check_device()
    sfe = [nets.encode(nets.preprocess(s).astype(np.float64), weights, ALL, np.float64) for s in styles]
    worst = 0.0
    for i, relu in enumerate(ALL):
        x = cap["level_input"][i].cpu().numpy().astype(np.float64)
        cf = nets.encode(x, weights, [relu], np.float64)[relu]
        lab = regions.nearest_labels(labels, cf.shape[1], cf.shape[2])
        if adain:
            f, info = regions.adain_regions(cf, lab, [s[relu] for s in sfe], 0.8)
        else:
            f, info = regions.wct_regions(cf, lab, [s[relu] for s in sfe], 0.8, sem)
            k = eng.last_info[i].cpu().numpy()
            for r in range(2):
                assert ref_ops.spectral_gap_ok(info[r]["wc"]) and ref_ops.spectral_gap_ok(info[r]["ws"]), "ill-posed vector"
                assert k[r] == info[r]["k_c"] and k[2 + r] == info[r]["n"]
        got_cf = eng.act_to_f32(cap["content_feat"][i]).cpu().numpy()
        got_f = eng.act_to_f32(cap["transformed"][i]).cpu().numpy()
        keep = lab == 9
        assert np.array_equal(got_f[0][keep], got_cf[0][keep])
        y = nets.decode(np.asarray(f, dtype=np.float64), weights, relu, np.float64)
        if i < len(ALL) - 1:
            y = np.clip(y, 0, 1)
        e = (np.abs(got_cf - cf).max(), np.abs(got_f - f).max(), np.abs(cap["level_output"][i].cpu().numpy() - y).max())
        print("%s: encoder %.2e  transform %.2e  level output %.2e" % ((relu,) + e))
        worst = max(worst, *e)
    assert worst <= 1e-3


@pytest.mark.parametrize("size", [(64, 96), (70, 130)])
def test_all_zero_mask_reduces_to_unmasked_path(size):
    targets = ["relu3_1", "relu2_1", "relu1_1"]
    w = make_synthetic_weights(21, relu_targets=targets)
    eng = Engine(w, targets, semantics="tf")
    rng = np.random.default_rng(5)
    c = torch.from_numpy(rng.integers(0, 256, (2,) + size + (3,), dtype=np.uint8)).cuda()
    s = torch.from_numpy(rng.integers(0, 256, (1, 80, 72, 3), dtype=np.uint8)).cuda()
    other = torch.from_numpy(rng.integers(0, 256, (1, 64, 64, 3), dtype=np.uint8)).cuda()
    zeros = torch.zeros((1,) + size, dtype=torch.uint8, device="cuda")
    plain = eng.to_u8(eng.stylize(c, s, alpha=0.8)).cpu().numpy()
    one = eng.to_u8(eng.stylize(c, [s], alpha=0.8, labels=zeros)).cpu().numpy()
    two = eng.to_u8(eng.stylize(c, [s, other], alpha=0.8, labels=zeros)).cpu().numpy()   # region 1 empty everywhere
    eng.check_device()
    assert np.array_equal(one, plain)
    assert np.array_equal(two, plain)


def test_batch_with_different_masks_equals_frame_by_frame():
    targets = ["relu3_1", "relu2_1", "relu1_1"]
    w = make_synthetic_weights(21, relu_targets=targets)
    eng = Engine(w, targets, semantics="tf")
    eng.groups = 2
    rng = np.random.default_rng(9)
    n, h, wd = 4, 96, 80
    c = torch.from_numpy(rng.integers(0, 256, (n, h, wd, 3), dtype=np.uint8)).cuda()
    styles = [torch.from_numpy(rng.integers(0, 256, (1, 72, 64 + 8 * r, 3), dtype=np.uint8)).cuda() for r in range(3)]
    labs = np.stack([_mask(k, h, wd, 3, rng) for k in ("blobs", "checker", "halves", "tiny")])
    labels = torch.from_numpy(labs).cuda()
    batch = eng.to_u8(eng.stylize(c, styles, alpha=0.7, labels=labels)).cpu().numpy()
    for i in range(n):
        one = eng.to_u8(eng.stylize(c[i:i + 1], styles, alpha=0.7, labels=labels[i:i + 1])).cpu().numpy()
        assert np.array_equal(batch[i:i + 1], one), i
    eng.check_device()


def test_cli_mask_equals_predict_batch(tmp_path):
    import stylize
    from wct_tf_b200 import device_image as dimg
    targets = ["relu2_1", "relu1_1"]
    rng = np.random.default_rng(3)
    content = rng.integers(0, 256, (60, 76, 3), dtype=np.uint8)
    s0 = rng.integers(0, 256, (50, 64, 3), dtype=np.uint8)
    s1 = rng.integers(0, 256, (64, 48, 3), dtype=np.uint8)
    mask = np.zeros((30, 40), np.uint8)
    mask[:, 20:] = 1
    mask[10:20, 5:15] = 4                                              # keep
    Image.fromarray(content).save(tmp_path / "c.png")
    Image.fromarray(s0).save(tmp_path / "a.png")
    Image.fromarray(s1).save(tmp_path / "b.png")
    Image.fromarray(mask, mode="L").save(tmp_path / "m.png")
    out_dir = tmp_path / "out"
    stylize.main(["--synthetic-weights", "42", "--relu-targets"] + targets + ["--content-path", str(tmp_path / "c.png"),
                  "--out-path", str(out_dir), "--mask-path", str(tmp_path / "m.png"), "--mask-styles", str(tmp_path / "a.png"),
                  str(tmp_path / "b.png"), "--passes", "2", "--keep-colors", "--alpha", "0.7"])
    got = np.array(Image.open(out_dir / "c_m.png"))
    model = WCT(relu_targets=targets, weights=make_synthetic_weights(42, relu_targets=targets))
    cdev = dimg.to_device(content)
    styles = [dimg.preserve_colors_np(dimg.to_device(s), cdev) for s in (s0, s1)]
    lab = dimg.labels_resize(torch.from_numpy(mask[None]).cuda(), 60, 76)
    want = model.predict_batch(cdev, styles, alpha=0.7, passes=2, labels=lab)[0]
    assert np.array_equal(got, want)


def test_errors():
    targets = ["relu2_1", "relu1_1"]
    model = WCT(relu_targets=targets, weights=make_synthetic_weights(42, relu_targets=targets))
    c = np.zeros((1, 32, 32, 3), np.uint8)
    s = np.zeros((1, 32, 32, 3), np.uint8)
    with pytest.raises(ValueError):
        model.predict_batch(c, [s], labels=np.zeros((1, 31, 32), np.uint8))
    with pytest.raises(ValueError):
        model.predict_batch(c, [s] * 9, labels=np.zeros((1, 32, 32), np.uint8))
    with pytest.raises(ValueError):
        model.predict_batch(c, [s], labels=np.zeros((1, 32, 32), np.uint8), swap5=True)
    lib = U.lib()
    cin = U.act_from_numpy(np.zeros((1, 8, 8, 64), np.float32))
    out = U.act_alloc(1, 8, 8, 64)
    lab = torch.zeros((1, 8, 8), dtype=torch.uint8, device="cuda")
    ws = torch.empty(lib.wctb200_wct_regions_workspace_bytes(64, 1, 8), dtype=torch.uint8, device="cuda")
    st = torch.empty(lib.wctb200_wct_style_state_bytes(64, 1), dtype=torch.uint8, device="cuda")
    ptrs = (ctypes.c_void_p * 9)(*([st.data_ptr()] * 9))
    args = (0.5, 1e-8, 0.0, 1e-5, 1, out.data_ptr(), None, ws.data_ptr(), ws.numel(), U.stream())
    assert lib.wctb200_wct_apply_regions(cin.data_ptr(), 1, 8, 8, 64, lab.data_ptr(), 9, ptrs, *args) == _capi.EINVAL
    assert lib.wctb200_wct_apply_regions(cin.data_ptr(), 1, 8, 8, 64, lab.data_ptr(), 0, ptrs, *args) == _capi.EINVAL
    assert lib.wctb200_wct_apply_regions(cin.data_ptr(), 1, 8, 8, 64, None, 2, ptrs, *args) == _capi.EINVAL
    assert lib.wctb200_wct_apply_regions(cin.data_ptr(), 1, 8, 8, 96, lab.data_ptr(), 2, ptrs, *args) == _capi.EINVAL
    hw = (ctypes.c_int * 18)(*([8] * 18))
    assert lib.wctb200_adain_regions(cin.data_ptr(), 1, 8, 8, 64, lab.data_ptr(), 9, ptrs, hw, 0.5, 1e-5, out.data_ptr(),
                                     ws.data_ptr(), ws.numel(), U.stream()) == _capi.EINVAL
    assert lib.wctb200_adain_regions(cin.data_ptr(), 1, 8, 8, 64, None, 1, ptrs, hw, 0.5, 1e-5, out.data_ptr(),
                                     ws.data_ptr(), ws.numel(), U.stream()) == _capi.EINVAL
    assert lib.wctb200_labels_resize_nearest(None, 1, 8, 8, 4, 4, lab.data_ptr(), U.stream()) == _capi.EINVAL
    U.check_device()
