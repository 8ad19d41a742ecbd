#!/usr/bin/env python
"""Command line front end with the flag surface of the reference's stylize.py (flags at stylize.py:14-37, the
content x style loop at stylize.py:70-119, output naming ``<content>_<style><ext>``): the TF session behind
``WCT.predict`` is replaced by the B200 engine.

  python stylize.py --checkpoints DIR5 DIR4 ... --relu-targets relu5_1 relu4_1 ... --vgg-path vgg_normalised.t7 \
      --content-path IN --style-path STYLE --out-path OUT --alpha 0.8

Spatial control: ``--mask-path MASK --mask-styles S0 S1 ...`` stylises the pixels labelled r in the 8-bit mask (mode L or P)
with style Sr and leaves labels >= the number of styles unstyled; the output is ``<content>_<mask stem><ext>``.

``--checkpoints`` are TF1 checkpoint directories or ``.npz`` bundles, ``--vgg-path`` a Torch7 ``.t7`` or ``.npz`` file
(wct_tf_b200.weights.load_weights); ``--synthetic-weights SEED`` runs with seeded random weights when the published
models are not on disk (offline build).
"""
from __future__ import division, print_function

import argparse
import os
import time

import numpy as np

# (flags, kwargs) -- names and defaults follow the reference one to one (tests/test_cli.py pins them)
_FLAGS = [
    (("--checkpoints",), dict(nargs="+", type=str, help="one decoder checkpoint (TF dir or .npz) per entry of --relu-targets")),
    (("--relu-targets",), dict(nargs="+", type=str, required=True, help="reluX_1 levels in pipeline order, paired with --checkpoints")),
    (("--vgg-path",), dict(type=str, default="models/vgg_normalised.t7", help="normalised VGG19 encoder (.t7 or .npz)")),
    (("--content-path",), dict(type=str, dest="content_path", help="content image, or a folder of them")),
    (("--style-path",), dict(type=str, dest="style_path", help="style image, or a folder of them")),
    (("--out-path",), dict(type=str, dest="out_path", help="folder that receives <content>_<style>.<ext>")),
    (("--keep-colors",), dict(action="store_true", default=False, help="CORAL: give the style the content's colours first")),
    (("--device",), dict(type=str, default="/gpu:0", help="/gpu:N (TF spelling), cuda:N or N")),
    (("--style-size",), dict(type=int, default=0, help="short side of the style before cropping (0: keep)")),
    (("--crop-size",), dict(type=int, default=0, help="centre-crop the style to a square of this size (0: off)")),
    (("--content-size",), dict(type=int, default=0, help="short side of the content (0: keep)")),
    (("--passes",), dict(type=int, default=1, help="feed the result back as content this many times")),
    (("-r", "--random"), dict(type=int, default=0, help="use a random subset of this many styles from the style folder")),
    (("--alpha",), dict(type=float, default=1, help="stylised / content feature blend")),
    (("--concat",), dict(action="store_true", default=False, help="write [style | result] side by side")),
    (("--adain",), dict(action="store_true", default=False, help="AdaIN statistics matching instead of WCT")),
    (("--swap5",), dict(action="store_true", default=False, help="style swap at relu5_1 (patch 3, stride 1)")),
    (("--ss-alpha",), dict(type=float, default=0.6, help="blend of the style-swapped feature")),
    (("--ss-patch-size",), dict(type=int, default=3)),
    (("--ss-stride",), dict(type=int, default=1)),
    # not in the reference
    (("--synthetic-weights",), dict(type=int, default=None, help="seeded random weights (no model files needed)")),
    (("--semantics",), dict(type=str, default="tf", choices=["tf", "np"], help="wct_tf (the reference graph) or wct_np eps/blend rules")),
    (("--mask-path",), dict(type=str, default=None, help="8-bit label mask (mode L or P): label r takes --mask-styles[r], others keep the content")),
    (("--mask-styles",), dict(nargs="+", type=str, default=None, help="one style image per mask label 0, 1, ... (at most 8)")),
]


def build_parser():
    parser = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    for names, kw in _FLAGS:
        parser.add_argument(*names, **kw)
    return parser


def parse_args(argv=None):
    """Parse and check the flag combinations the mask mode does not support."""
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.mask_path is not None or args.mask_styles is not None:
        if args.mask_path is None or not args.mask_styles:
            parser.error("--mask-path and --mask-styles go together")
        if len(args.mask_styles) > 8:
            parser.error("--mask-styles takes at most 8 styles")
        for flag, on in (("--swap5", args.swap5), ("--concat", args.concat), ("-r/--random", args.random > 0)):
            if on:
                parser.error("%s cannot be combined with --mask-path" % flag)
    return args


def _listing(path, io):
    return io.get_files(path) if os.path.isdir(path) else [path]


def _prepare_style(path, args, io, dimg, content_dev, device):
    """stylize.py:86-95 on the device: decode on the host, then resize / crop / CORAL without leaving the GPU."""
    img = dimg.to_device(io.get_img(path), device)
    if args.style_size > 0:
        img = dimg.resize_to(img, args.style_size)
    if args.crop_size > 0:
        img = dimg.center_crop(img, args.crop_size)
    if args.keep_colors:
        img = dimg.preserve_colors_np(img, content_dev)
    return img


def _stylize_masked(model, content_dev, styles_dev, labels_dev, args):
    """The --mask-path form of _stylize_pair: the labels ride along every pass."""
    kw = dict(alpha=args.alpha, adain=args.adain, return_device=True, passes=args.passes, labels=labels_dev)
    return model.predict_batch(content_dev, list(styles_dev), **kw)[0]


def _load_mask(path, content_dev, device):
    """The mask as cuda uint8 [1, H, W] at the content's size (nearest-neighbour resize on the device when it differs)."""
    import torch
    from wct_tf_b200 import imageio as io
    mask = torch.from_numpy(io.get_mask(path)).to(device).unsqueeze(0)
    H, W = content_dev.shape[-3], content_dev.shape[-2]
    if tuple(mask.shape[1:]) != (H, W):
        from wct_tf_b200 import device_image as dimg
        mask = dimg.labels_resize(mask, H, W)
    return mask


def _stylize_pair(model, content_dev, style_dev, args):
    """stylize.py:100-104; every pass takes and returns uint8 frames on the device (no host round trip between passes)."""
    kw = dict(alpha=args.alpha, swap5=args.swap5, ss_alpha=args.ss_alpha, adain=args.adain, return_device=True)
    result = model.predict_batch(content_dev, style_dev, **kw)
    for _ in range(args.passes - 1):
        result = model.predict_batch(result, style_dev, **kw)
    return result[0]


def make_model(args):
    from wct_tf_b200.wct import WCT
    weights = None
    if args.synthetic_weights is not None:
        from wct_tf_b200.weights import make_synthetic_weights
        weights = make_synthetic_weights(args.synthetic_weights, relu_targets=args.relu_targets)
    elif not args.checkpoints:
        raise SystemExit("--checkpoints is required (or --synthetic-weights SEED)")
    return WCT(checkpoints=args.checkpoints, relu_targets=args.relu_targets, vgg_path=args.vgg_path, device=args.device,
               ss_patch_size=args.ss_patch_size, ss_stride=args.ss_stride, weights=weights, semantics=args.semantics, verbose=True)


def main(argv=None):
    args = parse_args(argv)
    from wct_tf_b200 import device_image as dimg
    from wct_tf_b200 import imageio as io
    t_start = time.time()
    model = make_model(args)
    styles = _listing(args.style_path, io) if args.mask_path is None else []
    if args.mask_path is None and os.path.isdir(args.style_path) and args.random > 0:
        styles = list(np.random.choice(styles, args.random))
    os.makedirs(args.out_path, exist_ok=True)

    device = model.engine.device
    written = 0
    for content_path in _listing(args.content_path, io):
        stem, ext = os.path.splitext(os.path.basename(content_path))
        content_dev = dimg.to_device(io.get_img(content_path), device)
        if args.content_size > 0:
            content_dev = dimg.resize_to(content_dev, args.content_size)
        if args.mask_path is not None:
            labels = _load_mask(args.mask_path, content_dev, device)
            region_styles = [_prepare_style(p, args, io, dimg, content_dev, device) for p in args.mask_styles]
            result = _stylize_masked(model, content_dev, region_styles, labels, args)
            target = os.path.join(args.out_path, "{}_{}{}".format(stem, os.path.splitext(os.path.basename(args.mask_path))[0], ext))
            io.save_img(target, result.cpu().numpy())
            written += 1
            print("{}: Wrote stylized output image to {}".format(written, target))
            continue
        for style_path in styles:
            style_dev = _prepare_style(style_path, args, io, dimg, content_dev, device)
            result = _stylize_pair(model, content_dev, style_dev, args)
            if args.concat:
                result = dimg.concat_with_style(style_dev, result)
            target = os.path.join(args.out_path, "{}_{}{}".format(stem, os.path.splitext(os.path.basename(style_path))[0], ext))
            io.save_img(target, result.cpu().numpy())
            written += 1
            print("{}: Wrote stylized output image to {}".format(written, target))
    print("Finished stylizing {} outputs in {}s".format(written, time.time() - t_start))


if __name__ == "__main__":
    main()
