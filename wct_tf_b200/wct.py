"""``WCT`` -- drop-in for the reference inference wrapper (wct.py:14-106).

Same constructor and ``predict`` signature; the TF session is replaced by the
sm_100a engine (engine.py -> libwctb200.so).  Differences, all explicit:
  * ``checkpoints`` / ``vgg_path`` may be file paths (``.npz`` bundles, see
    weights.py) OR ``weights=`` may pass an in-memory weights dict (the offline
    build has no .t7 / TF checkpoints, so benchmarks use synthetic weights);
  * ``device`` accepts the reference's TF strings ('/gpu:0') and torch strings;
  * ``swap5=True`` (style-swap at relu5_1, ops.py:145-278) honours ``ss_patch_size`` / ``ss_stride``; with a stride the
    content is centre-cropped so that the patches tile its relu5_1 encoding, as wct.py:84-90 does;
  * ``predict_batch`` is new: a batch of frames per call (frames are independent);
  * ``labels=`` (both calls) is new: spatial control, one style per region of a uint8 label mask (Li et al. 2017, sec. 4).
"""
from __future__ import annotations

import re
import time

import numpy as np
import torch

from .engine import Engine


def _torch_device(device):
    """'/gpu:0' (stylize.py:23) -> 'cuda:0'."""
    if isinstance(device, int):
        return "cuda:%d" % device
    if isinstance(device, str):
        m = re.match(r"^/?(?:device:)?gpu:(\d+)$", device.strip().lower())
        if m:
            return "cuda:%s" % m.group(1)
        if re.match(r"^\d+$", device.strip()):          # a bare ordinal, as the CLI help advertises
            return "cuda:%s" % device.strip()
        if device.strip().lower() in ("/cpu:0", "cpu"):
            raise ValueError("the B200 engine has no CPU path (device=%r)" % (device,))
    return device


class WCT(object):
    '''Stylize images with the multi-level WCT pipeline (mirror of wct.py:14)'''

    def __init__(self, checkpoints=None, relu_targets=None, vgg_path=None, device='/gpu:0',
                 ss_patch_size=3, ss_stride=1, weights=None, semantics="tf", verbose=False):
        if relu_targets is None:
            raise ValueError("relu_targets is required")
        self.ss_patch_size = ss_patch_size
        self.ss_stride = ss_stride
        self.verbose = verbose
        if weights is None:
            from .weights import load_weights
            weights = load_weights(vgg_path, checkpoints, relu_targets)   # pairs checkpoints[i] <-> relu_targets[i] (wct.py:47)
        self.engine = Engine(weights, relu_targets, device=_torch_device(device), semantics=semantics)
        self.engine.groups = 2                  # batches >= 2 frames run as two interleaved stream pairs
        self.engine.group_priorities = True
        self.model = self.engine.model

    @staticmethod
    def preprocess(image):
        """wct.py:60-64"""
        if len(image.shape) == 3:
            image = np.expand_dims(image, 0)
        return image / 255.

    @staticmethod
    def postprocess(image):
        """wct.py:66-68"""
        return np.uint8(np.clip(image, 0, 1) * 255)

    def predict_batch(self, contents, styles, alpha=1, adain=False, return_float=False, out=None, swap5=False, ss_alpha=1,
                      passes=1, return_device=False, labels=None):
        """contents: uint8 [N,H,W,3]; styles: uint8 [1|N,Hs,Ws,3] (numpy or torch; host buffers --
        ideally pinned -- or device tensors).  Returns uint8 [N,H',W',3] on the host: a numpy array,
        or ``out`` (a pinned uint8 torch tensor of the right shape) filled in place.  The call is
        synchronous like the reference's ``sess.run`` (wct.py:97).

        ``passes`` > 1 repeats the stylisation on the previous OUTPUT like stylize.py:102-104 (``--passes``), but keeps the
        intermediate frames on the device: each pass still ends in the uint8 quantisation of wct.py:66-68 and restarts from
        /255 (wct.py:60-64), so the result is bit-identical to calling predict once per pass; style swap only acts in the
        first pass, as in stylize_video.py:117-121.  ``return_device=True`` returns the uint8 cuda tensor instead of a host copy.

        ``labels`` (uint8 [N|1,H,W] or [H,W], the contents' size; numpy or torch): spatial control.  ``styles`` is then a
        list of R <= 8 style images; pixels labelled r < R take style r, labels >= R keep the content.  Every pass uses the
        same labels."""
        eng = self.engine
        dev = eng.device
        if labels is not None:
            if swap5:
                raise ValueError("swap5 cannot be combined with labels: style swap is not a per-region statistic")
            if not isinstance(styles, (list, tuple)):
                raise ValueError("with labels, styles must be a list of R style images (one per region)")

        def to_dev(a):
            if isinstance(a, np.ndarray):
                a = torch.from_numpy(np.array(a, copy=True, order="C"))    # own, writable, contiguous
            if a.dim() == 3:
                a = a.unsqueeze(0)
            if a.dtype != torch.uint8:
                a = a.clamp(0, 255).to(torch.uint8)   # the reference feeds arrays "in [0,255]" (wct.py:74)
            return a.to(dev, non_blocking=True).contiguous()

        if swap5 and self.ss_stride != 1:
            # wct.py:84-90: with a stride the filter may not fit; centre-crop the content (on the device) to a size it tiles
            from .device_image import center_crop_to
            from .imageio import swap_filter_fit
            with torch.cuda.device(dev):
                contents = to_dev(contents)
                refit, H, W = swap_filter_fit(contents.shape[1], contents.shape[2], self.ss_patch_size, self.ss_stride)
                if refit:
                    contents = center_crop_to(contents, H, W)
        with torch.cuda.device(dev):
            c = to_dev(contents)
            if labels is not None:
                lab = labels if isinstance(labels, torch.Tensor) else torch.from_numpy(np.array(labels, copy=True, order="C"))
                if lab.dim() == 2:
                    lab = lab.unsqueeze(0)
                if lab.dtype != torch.uint8 or lab.dim() != 3 or tuple(lab.shape[1:]) != tuple(c.shape[1:3]):
                    raise ValueError("labels must be uint8 [N|1,H,W] with the contents' H x W = %s, got %s %s"
                                     % (tuple(c.shape[1:3]), tuple(lab.shape), lab.dtype))
                lab = lab.to(dev, non_blocking=True).contiguous()
                s = [to_dev(x) for x in styles]
                out_f = eng.stylize(c, s, alpha=alpha, adain=adain, labels=lab)
            else:
                lab = None
                s = to_dev(styles)
                if swap5:
                    # one pair per call like the reference graph (ops.py:146); frames of a batch are swapped one by one
                    outs = [eng.stylize(c[i:i + 1], s[i:i + 1] if s.shape[0] > 1 else s, alpha=alpha, adain=adain, swap5=True,
                                        ss_alpha=ss_alpha, ss_patch_size=self.ss_patch_size, ss_stride=self.ss_stride)
                            for i in range(c.shape[0])]
                    out_f = outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)
                else:
                    out_f = eng.stylize(c, s, alpha=alpha, adain=adain)
            out_dev = eng.to_u8(out_f)
            for _ in range(int(passes) - 1):
                # an odd size grows through the decoder: the labels follow (nearest, always from the caller's map)
                lab_p = None if lab is None else eng.labels_resize(lab, out_dev.shape[1], out_dev.shape[2])
                out_f = eng.stylize(out_dev, s, alpha=alpha, adain=adain, labels=lab_p)
                out_dev = eng.to_u8(out_f)
            if return_device:
                eng.check_device()            # synchronises; raises WctB200Error if a kernel recorded a pipeline time-out
                return (out_dev, out_f) if return_float else out_dev
            if out is not None:
                out.copy_(out_dev, non_blocking=True)
                out_u8 = out
            else:
                out_u8 = torch.empty(out_dev.shape, dtype=torch.uint8, pin_memory=True)
                out_u8.copy_(out_dev, non_blocking=True)
            # the call is synchronous like sess.run (wct.py:97); a device-side time-out would otherwise leave every
            # later frame silently wrong (kernels skip their stores once the error word is set)
            eng.check_device()
            if out is None:
                out_u8 = out_u8.numpy().copy()
        if return_float:
            return out_u8, out_f.cpu().numpy()
        return out_u8

    def predict(self, content, style, alpha=1, swap5=False, ss_alpha=1, adain=False, labels=None):
        '''Stylize a single content/style pair (wct.py:70-106); with ``labels`` ([H,W] uint8), ``style`` is a list of R
        styles, one per region.'''
        s = time.time()
        styles = [np.asarray(x) for x in style] if labels is not None else np.asarray(style)
        out = self.predict_batch(np.asarray(content), styles, alpha=alpha, adain=adain, swap5=swap5, ss_alpha=ss_alpha,
                                 labels=None if labels is None else np.asarray(labels))
        if self.verbose:
            print("Stylized in:", time.time() - s)   # wct.py:104
        return out[0]
