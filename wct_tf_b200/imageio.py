"""Host-side image helpers of the CLI (restating utils.py:11-67, coral.py:8-39 with
PIL/NumPy: ``scipy.misc.imread/imresize/imsave`` no longer exist).  Off the hot path."""
from __future__ import annotations

import os

import numpy as np
from PIL import Image


def get_files(img_dir):
    """utils.py:11-17"""
    return [os.path.join(img_dir, x) for x in os.listdir(img_dir)]


def get_img(src):
    """utils.py:23-27: RGB uint8 HxWx3"""
    return np.asarray(Image.open(src).convert("RGB"))


def save_img(out_path, img):
    """utils.py:19-21"""
    Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)).save(out_path)


def _imresize(img, hw):
    # scipy.misc.imresize(interp='bilinear') was PIL's bilinear resize on the uint8 image
    return np.asarray(Image.fromarray(np.asarray(img, dtype=np.uint8)).resize((int(hw[1]), int(hw[0])), Image.BILINEAR))


def resize_to(img, resize=512):
    """utils.py:55-67: resize the SHORT side to ``resize`` keeping the aspect ratio."""
    height, width = img.shape[0], img.shape[1]
    if height < width:
        shape = (resize, int(round(width / (height / resize))))
    else:
        shape = (int(round(height / (width / resize))), resize)
    return _imresize(img, shape)


def center_crop(img, size=256):
    """utils.py:29-38"""
    height, width = img.shape[0], img.shape[1]
    if height < size or width < size:
        img = resize_to(img, resize=size)
        height, width = img.shape[0], img.shape[1]
    h_off, w_off = (height - size) // 2, (width - size) // 2
    return img[h_off:h_off + size, w_off:w_off + size]


def _mat_sqrt(x):
    """coral.py:8-11 verbatim in effect: ``U, D, V = np.linalg.svd(x); U diag(sqrt D) V.T``.  numpy returns V^H as the third
    value, so for the symmetric input this is U sqrt(D) U -- NOT the symmetric square root U sqrt(D) U^T.  The reference's
    --keep-colors output depends on it, so it is reproduced (pinned by tests/golden/coral_keep_colors.npz)."""
    u, d, vh = np.linalg.svd(x)
    return (u * np.sqrt(d)) @ vh.T


def coral(source, target):
    """CORAL colour alignment of ``source`` to ``target`` statistics (coral.py:13-39):
    per-channel standardise, match the (cov + I) of the 3x3 channel covariance."""
    c = source.shape[-1]
    s = source.reshape(-1, c).T
    t = target.reshape(-1, c).T
    sm, ss = s.mean(1, keepdims=True), s.std(1, keepdims=True)
    tm, ts = t.mean(1, keepdims=True), t.std(1, keepdims=True)
    sn, tn = (s - sm) / ss, (t - tm) / ts
    cs = sn @ sn.T + np.eye(c)
    ct = tn @ tn.T + np.eye(c)
    out = _mat_sqrt(ct) @ np.linalg.inv(_mat_sqrt(cs)) @ sn
    out = out * ts + tm
    return out.T.reshape(source.shape)


def preserve_colors_np(style_rgb, content_rgb):
    """utils.py:87-90 (--keep-colors)"""
    return np.uint8(np.clip(coral(style_rgb / 255., content_rgb / 255.), 0, 1) * 255.)


def center_crop_to(img, H_target, W_target):
    """utils.py:40-53: centre crop a rectangle, upscaling first (bilinear, by the larger of the two ratios) if the image
    is too small."""
    height, width = img.shape[0], img.shape[1]
    if height < H_target or width < W_target:
        rat = max(H_target / height, W_target / width)
        # scipy.misc.imresize(img, <float>) scaled both sides by the fraction (PIL bilinear on the uint8 image)
        img = _imresize(img, (int(height * rat), int(width * rat)))
        height, width = img.shape[0], img.shape[1]
    h_off, w_off = (height - H_target) // 2, (width - W_target) // 2
    return img[h_off:h_off + H_target, w_off:w_off + W_target]


def swap_filter_fit(H, W, patch_size, stride, n_pools=4):
    """utils.py:115-138: style swap with a stride may not tile the relu5_1 encoding; returns (should_refit, H_out, W_out),
    the image size whose encoding the patch / stride combination tiles exactly."""
    def pool_out(x):
        return (x + 2 - 1) // 2
    hp, wp = H, W
    for _ in range(n_pools):
        hp, wp = pool_out(hp), pool_out(wp)
    hc, wc = (hp - patch_size) // stride + 1, (wp - patch_size) // stride + 1
    hd, wd = (hc - 1) * stride + patch_size, (wc - 1) * stride + patch_size
    return (hp != hd) or (wp != wd), hd * 2 ** n_pools, wd * 2 ** n_pools


def get_mask(path):
    """Label mask for spatial control: an 8-bit image in mode 'L' (grey value = label) or 'P' (palette index = label).
    Returns uint8 [H, W]; any other mode is refused."""
    img = Image.open(path)
    if img.mode not in ("L", "P"):
        raise ValueError("mask %s has mode %r: a label mask must be an 8-bit 'L' (grey) or 'P' (palette) image" % (path, img.mode))
    return np.array(img, dtype=np.uint8)
