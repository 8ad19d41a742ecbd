"""Spatial control on the CPU (TEST INFRASTRUCTURE): the per-region form of the reference transforms.

A uint8 label map splits a frame into regions.  Region r < R is transformed by the reference's own op (ref_ops.wct_generic /
ref_ops.adain) applied to the content features RESTRICTED to its pixels (a 1 x n_r x 1 x C array) with the full features of
style r; the result is scattered back.  Labels >= R, and regions of fewer than 2 pixels (the reference's 1/(n-1) is undefined
there), keep the input.  Label maps follow a level's feature size by ``nearest_labels``, always from the original map.
"""
from __future__ import annotations

import numpy as np

from . import nets, ref_ops

SEMANTICS = {
    "tf": dict(eps_cov=1e-8, eps_eig=0.0, readd_content_mean=True),
    "np": dict(eps_cov=0.0, eps_eig=1e-5, readd_content_mean=False),
}


def nearest_labels(labels, h, w):
    """[..., H, W] -> [..., h, w]: L_l[y][x] = L[(y*H) div h][(x*W) div w] (exact integer arithmetic)."""
    labels = np.asarray(labels)
    H, W = labels.shape[-2:]
    ys = (np.arange(h, dtype=np.int64) * H) // h
    xs = (np.arange(w, dtype=np.int64) * W) // w
    return labels[..., ys[:, None], xs[None, :]]


def _per_region(cf, lab, R, fn):
    """Apply fn(features 1 x n_r x 1 x C, r) -> same shape to every region of one frame (1 x h x w x C); info per region."""
    cf = np.asarray(cf)
    out = cf.copy()
    infos = []
    for r in range(R):
        m = lab == r
        n_r = int(m.sum())
        info = dict(n=n_r, k_c=0)
        if n_r >= 2:
            sub = cf[0][m][None, :, None, :]
            res, inf = fn(sub, r)
            out[0][m] = np.asarray(res)[0, :, 0, :]
            info.update(inf)
        infos.append(info)
    return out, infos


def wct_regions(cf, lab, styles, alpha, semantics="tf"):
    """One frame's level: cf 1 x h x w x C, lab h x w (already at the feature size), styles: R style features."""
    sem = SEMANTICS[semantics]

    def fn(sub, r):
        res, inf = ref_ops.wct_generic(sub, styles[r], alpha, return_info=True, **sem)
        return res, dict(k_c=inf["k_c"], k_s=inf["k_s"], wc=inf["wc"], ws=inf["ws"])
    return _per_region(cf, lab, len(styles), fn)


def adain_regions(cf, lab, styles, alpha):
    return _per_region(cf, lab, len(styles), lambda sub, r: (ref_ops.adain(sub, styles[r], alpha), {}))


def pipeline_regions(content_u8, styles_u8, labels, weights, relu_targets, alpha=1.0, adain=False, semantics="tf",
                     dtype=np.float64, return_info=False):
    """nets.pipeline with a label map (H x W, the content's size) and R styles: a free-running masked run."""
    relu_targets = list(relu_targets)
    x = nets.preprocess(content_u8).astype(dtype)
    style_feats = [nets.encode(nets.preprocess(s).astype(dtype), weights, relu_targets, dtype) for s in styles_u8]
    info = []
    for i, relu in enumerate(relu_targets):
        if i > 0:
            x = np.clip(x, 0, 1)
        cf = nets.encode(x, weights, [relu], dtype)[relu]
        lab = nearest_labels(labels, cf.shape[1], cf.shape[2])
        sfs = [sf[relu] for sf in style_feats]
        if adain:
            f, inf = adain_regions(cf, lab, sfs, alpha)
        else:
            f, inf = wct_regions(cf, lab, sfs, alpha, semantics)
        info.append(dict(relu=relu, regions=inf))
        x = nets.decode(np.asarray(f, dtype=dtype), weights, relu, dtype)
    if return_info:
        return x, info
    return x
