"""The CLI's image steps on the device (scope row 8f-3): same names, arguments and results as the reference's helpers
(``utils.resize_to`` / ``center_crop`` / ``center_crop_to`` utils.py:29-67, ``utils.preserve_colors_np`` utils.py:87-90,
the ``--concat`` thumbnail stylize.py:107-111), operating on ``torch.uint8`` CUDA tensors HxWx3 (or NxHxWx3) through the C ABI
(``wctb200_resize_bilinear_u8``, ``wctb200_rgb_moments_u8``, ``wctb200_coral_apply_u8``).  A decoded image goes to the GPU once
and stays there through resize, crop, CORAL, every ``--passes`` round and the concat; only the finished frame comes back.

There is no CPU fallback: the functions raise ``WctB200Error`` when the library or a CUDA device is missing.  The only host
arithmetic is the 3x3 algebra of CORAL (the reference's ``matSqrt`` goes through ``np.linalg.svd`` and, as written, depends on
its sign conventions -- coral.py:8-11 -- so the same call is made here on the 3x3 matrices built from the device's exact
integer moments).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _capi


def _stream():
    return torch.cuda.current_stream().cuda_stream


def to_device(img, device="cuda:0"):
    """numpy / torch uint8 HxWxC -> contiguous CUDA tensor (one H2D copy)."""
    if not torch.cuda.is_available():
        raise _capi.WctB200Error("no CUDA device: the image steps have no CPU fallback")
    t = img if isinstance(img, torch.Tensor) else torch.from_numpy(np.array(img, dtype=np.uint8, order="C"))   # own, writable copy (PIL arrays are read-only)
    if t.dtype != torch.uint8:
        raise TypeError("expected a uint8 image, got %s" % t.dtype)
    return t.to(device, non_blocking=True).contiguous()


def to_host(img):
    """uint8 CUDA tensor -> numpy (synchronous D2H)."""
    return img.cpu().numpy()


def _as_batch(img):
    if img.dim() == 3:
        return img.unsqueeze(0), True
    if img.dim() == 4:
        return img, False
    raise ValueError("expected HxWxC or NxHxWxC, got shape %s" % (tuple(img.shape),))


def imresize(img, hw, window=None):
    """``scipy.misc.imresize(img, (H, W), interp='bilinear')`` (utils.py:48,67; bit-exact with Pillow's resample); ``window`` =
    (y0, x0, Hout, Wout) returns that crop of the result without computing the rest."""
    lib = _capi.load()
    x, single = _as_batch(img)
    if not x.is_cuda:
        raise _capi.WctB200Error("device_image works on CUDA tensors (use to_device)")
    x = x.contiguous()
    N, Hs, Ws, Cc = x.shape
    Hd, Wd = int(hw[0]), int(hw[1])
    y0, x0, Ho, Wo = (0, 0, Hd, Wd) if window is None else [int(v) for v in window]
    with torch.cuda.device(x.device):
        nbytes = lib.wctb200_resize_workspace_bytes(N, Hs, Ws, Cc, Hd, Wd, Wo)
        if nbytes == 0:
            raise _capi.WctB200Error("resize: bad geometry %s -> %s" % ((N, Hs, Ws, Cc), (Hd, Wd)))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        out = torch.empty((N, Ho, Wo, Cc), dtype=torch.uint8, device=x.device)
        _capi.check(lib.wctb200_resize_bilinear_u8(x.data_ptr(), N, Hs, Ws, Cc, Hd, Wd, y0, x0, Ho, Wo, out.data_ptr(),
                                                   ws.data_ptr(), nbytes, _stream()))
    return out[0] if single else out


def _short_side_shape(height, width, resize):
    # utils.py:57-65 (Python 3 round: banker's rounding, as in the reference)
    if height < width:
        return resize, int(round(width / (height / resize)))
    return int(round(height / (width / resize))), resize


def resize_to(img, resize=512):
    """utils.py:55-67: SHORT side to ``resize``, aspect ratio kept."""
    h, w = (img.shape[0], img.shape[1]) if img.dim() == 3 else (img.shape[1], img.shape[2])
    return imresize(img, _short_side_shape(h, w, resize))


def center_crop(img, size=256):
    """utils.py:29-38; the resize (when a side is too small) and the crop are one launch sequence: only the window is computed."""
    h, w = (img.shape[0], img.shape[1]) if img.dim() == 3 else (img.shape[1], img.shape[2])
    hd, wd = (h, w) if (h >= size and w >= size) else _short_side_shape(h, w, size)
    return imresize(img, (hd, wd), window=((hd - size) // 2, (wd - size) // 2, size, size))


def center_crop_to(img, H_target, W_target):
    """utils.py:40-53"""
    h, w = (img.shape[0], img.shape[1]) if img.dim() == 3 else (img.shape[1], img.shape[2])
    hd, wd = h, w
    if h < H_target or w < W_target:
        rat = max(H_target / h, W_target / w)
        hd, wd = int(h * rat), int(w * rat)          # imresize(img, <float>): both sides scaled by the fraction, truncated
    return imresize(img, (hd, wd), window=((hd - H_target) // 2, (wd - W_target) // 2, H_target, W_target))


def rgb_moments(img):
    """(npix, sum x_c [3], sum x_c x_d [3][3]) of an RGB uint8 image -- exact integers from the device."""
    lib = _capi.load()
    x = img.contiguous()
    if x.shape[-1] != 3:
        raise ValueError("expected an RGB image")
    npix = x.numel() // 3
    with torch.cuda.device(x.device):
        sums = torch.empty(9, dtype=torch.int64, device=x.device)
        _capi.check(lib.wctb200_rgb_moments_u8(x.data_ptr(), npix, sums.data_ptr(), _stream()))
        s = [int(v) for v in sums.cpu().tolist()]
    s1 = np.array(s[:3], dtype=object)
    s2 = np.empty((3, 3), dtype=object)
    s2[0, 0], s2[0, 1], s2[0, 2], s2[1, 1], s2[1, 2], s2[2, 2] = s[3:]
    s2[1, 0], s2[2, 0], s2[2, 1] = s2[0, 1], s2[0, 2], s2[1, 2]
    return npix, s1, s2


def _mat_sqrt(x):
    # coral.py:8-11 as written: U diag(sqrt D) (V^T)^T with numpy's (u, s, vh) -- for the symmetric input U sqrt(D) U
    u, d, vh = np.linalg.svd(x)
    return (u * np.sqrt(d)) @ vh.T


def _standardised_stats(img):
    """mean, std (population, np.std) and norm . norm^T + I of the [0,1]-scaled channels (coral.py:23-32), from the moments."""
    npix, s1, s2 = rgb_moments(img)
    mean = np.array([float(v) / npix for v in s1]) / 255.0
    # population covariance of x/255 from exact integers: (n*S2 - s s^T) / n^2 / 255^2 (the integer numerator is exact)
    cov = np.array([[float(npix * s2[i, j] - s1[i] * s1[j]) for j in range(3)] for i in range(3)]) / (float(npix) ** 2) / 255.0 ** 2
    std = np.sqrt(np.diag(cov))
    gram = npix * cov / np.outer(std, std) + np.eye(3)
    return mean, std, gram


def preserve_colors_np(style_rgb, content_rgb):
    """utils.py:87-90 (--keep-colors): CORAL of the style to the content's colour statistics; uint8 CUDA tensors in and out."""
    lib = _capi.load()
    src = style_rgb.contiguous()
    sm, ss, cs = _standardised_stats(src)
    tm, ts, ct = _standardised_stats(content_rgb)
    A = np.ascontiguousarray(_mat_sqrt(ct) @ np.linalg.inv(_mat_sqrt(cs)), dtype=np.float64)
    out = torch.empty_like(src)

    def dp(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        return a, a.ctypes.data_as(C.c_void_p)
    keep = [dp(A), dp(sm), dp(ss), dp(tm), dp(ts)]
    with torch.cuda.device(src.device):
        _capi.check(lib.wctb200_coral_apply_u8(src.data_ptr(), src.numel() // 3, keep[0][1], keep[1][1], keep[2][1], keep[3][1],
                                               keep[4][1], out.data_ptr(), _stream()))
    return out


def labels_resize(labels, H, W):
    """Nearest-neighbour resize of cuda uint8 label maps [N,Hs,Ws] -> [N,H,W]: L[(y*Hs) div H][(x*Ws) div W]."""
    labels = labels.contiguous()
    N, Hs, Ws = labels.shape
    out = torch.empty((N, H, W), dtype=torch.uint8, device=labels.device)
    _capi.check(_capi.load().wctb200_labels_resize_nearest(labels.data_ptr(), N, Hs, Ws, H, W, out.data_ptr(), _stream()))
    return out


def concat_with_style(style_img, result):
    """--concat (stylize.py:107-111): [style resized to the result's height, square | result]"""
    edge = result.shape[0]
    return torch.cat([imresize(style_img, (edge, edge)), result], dim=1)
