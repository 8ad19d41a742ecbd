"""Executes the multi-level WCT plan (model.py) on one GPU through libwctb200.

Host side of the hot path ``WCT.predict`` (wct.py:70-106): PyTorch is used only
for device memory, streams and H2D/D2H copies; every arithmetic step is a
hand-written sm_100a kernel behind the C-ABI (include/wctb200.h).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _capi
from .model import WCTModel, RELU_CHANNELS

# wct_tf (ops.py:24-90, what the graph executes) vs wct_np (ops.py:92-140, the named oracle)
SEMANTICS = {
    "tf": dict(eps_cov=1e-8, eps_eig=0.0, thresh=1e-5, readd=1),
    "np": dict(eps_cov=0.0, eps_eig=1e-5, thresh=1e-5, readd=0),
}


class Act(object):
    """SPF16 activation: device buffer + logical NHWC shape."""
    __slots__ = ("buf", "N", "H", "W", "C")

    def __init__(self, buf, N, H, W, C):
        self.buf, self.N, self.H, self.W, self.C = buf, N, H, W, C

    @property
    def ptr(self):
        return self.buf.data_ptr()


class Engine(object):
    def __init__(self, weights, relu_targets, device="cuda:0", semantics="tf", fuse_upsample=True, fuse_pool=True):
        if not torch.cuda.is_available():
            raise _capi.WctB200Error("no CUDA device: the WCT engine has no CPU fallback")
        self.lib = _capi.load()
        self.device = torch.device(device)
        self.model = WCTModel(mode="test", relu_targets=relu_targets)
        if semantics not in SEMANTICS:
            raise ValueError("semantics must be 'tf' or 'np'")
        self.semantics = semantics
        self.last_info = None
        self._ws = {}
        self.overlap_style = True  # run the style side (encode + per-level eigendecompositions) on a second stream
        self.groups = 1            # >1: split a batch into sub-batches that run as independent stream-pairs
        self.group_priorities = False
        self._group = 0
        self._style_streams = {}
        self._group_streams = {}
        self.fuse_pool = bool(fuse_pool)          # MaxPooling2D folded into the epilogue of the conv before it (WCTB200_POOL2)
        self.fuse_upsample = bool(fuse_upsample)  # UpSampling2D folded into the next conv (4 parity kernels, 4/9 of the MACs); fixed at construction
        self.launches = 0          # kernels launched through the C-ABI (bench.py "gpu_launches")
        self.profile = None        # optional dict: key -> [torch.cuda.Event pairs, flops, bytes]
        self._tag = None           # profiling only: "style" / relu target of the level being enqueued
        with torch.cuda.device(self.device):
            self._upload(weights)

    # ------------------------------------------------------------------ weights
    def _dev(self, a, dtype=torch.float32):
        return torch.from_numpy(np.ascontiguousarray(a)).to(device=self.device, dtype=dtype)

    def _prep_split(self, w_hwio, up2=False):
        """fp32 (kH,kW,Cin,Cout) -> device split-fp16 GEMM operand (``up2``: the four 2x2-tap parity kernels of
        UpSampling2D -> Conv2DReflect, see csrc/conv_tc.cu)."""
        kh, kw, cin, cout = w_hwio.shape
        src = self._dev(w_hwio.astype(np.float32))
        if up2:
            dst = torch.empty(self.lib.wctb200_conv_weight_bytes(16, cin, cout), dtype=torch.uint8, device=self.device)
            _capi.check(self.lib.wctb200_prep_conv_weights_up2(src.data_ptr(), cin, cout, dst.data_ptr(), self._stream()))
            return dst
        dst = torch.empty(self.lib.wctb200_conv_weight_bytes(kh * kw, cin, cout), dtype=torch.uint8, device=self.device)
        _capi.check(self.lib.wctb200_prep_conv_weights(src.data_ptr(), kh * kw, cin, cout, dst.data_ptr(), self._stream()))
        return dst

    @staticmethod
    def _fused_up(ops, i):
        """True when ops[i] is an 'up' that the engine folds into the conv that follows it (model.py:291-293)."""
        return ops[i].kind == "up" and i + 1 < len(ops) and ops[i + 1].kind == "conv" and ops[i + 1].act

    def _upload(self, weights):
        vgg = {l["name"]: l for l in weights["vgg"]}
        # fold the 1x1 'preprocess' conv (vgg_normalised.py:25-26) into conv1_1 (exact: a per-pixel affine
        # map commutes with reflect padding); done in float64 on the host, once.
        w0 = np.asarray(vgg["preprocess"]["weight"], dtype=np.float64)[:, :, 0, 0]  # (O=j, I=i)
        b0 = np.asarray(vgg["preprocess"]["bias"], dtype=np.float64)
        w1 = np.asarray(vgg["conv1_1"]["weight"], dtype=np.float64)                 # (O, j, kH, kW)
        b1 = np.asarray(vgg["conv1_1"]["bias"], dtype=np.float64)
        wf = np.einsum("ojyx,ji->yxio", w1, w0)                                      # (kH,kW,i,O)
        bf = b1 + np.einsum("ojyx,j->o", w1, b0)
        self.head_w = self._dev(wf.reshape(27, 64).astype(np.float32))
        self.head_b = self._dev(bf.astype(np.float32))
        self.enc_w, self.enc_b = {}, {}
        deepest_ops = [op for op in self.model.style_plan if op.kind == "conv" and op.name != "conv1_1"]
        for op in deepest_ops:
            l = vgg[op.name]
            hwio = np.transpose(np.asarray(l["weight"], dtype=np.float32), (2, 3, 1, 0))  # vgg_normalised.py:33
            self.enc_w[op.name] = self._prep_split(hwio)
            self.enc_b[op.name] = self._dev(np.asarray(l["bias"], dtype=np.float32))
        self.dec_w, self.dec_b, self.tail_w, self.tail_b = {}, {}, {}, {}
        for lvl in self.model.levels:
            relu = lvl.relu_target
            if relu in self.tail_w:
                continue
            if relu not in weights["decoders"]:
                raise Exception("No checkpoint found for target {}".format(relu))  # wct.py:57-58
            layers = {l["name"]: l for l in weights["decoders"][relu]}
            ops = self.model.decoder_plan(lvl.index)
            for i, op in enumerate(ops):
                if op.kind != "conv":
                    continue
                l = layers[op.name]
                k = np.asarray(l["kernel"], dtype=np.float32)
                assert k.shape == (3, 3, op.cin, op.cout), (op.name, k.shape)
                if op.act:
                    self.dec_w[op.name] = self._prep_split(k, up2=(self.fuse_upsample and i > 0 and self._fused_up(ops, i - 1)))
                    self.dec_b[op.name] = self._dev(np.asarray(l["bias"], dtype=np.float32))
                else:
                    self.tail_w[relu] = self._dev(k.reshape(9 * op.cin, 3))
                    self.tail_b[relu] = self._dev(np.asarray(l["bias"], dtype=np.float32))
        torch.cuda.synchronize(self.device)

    # ------------------------------------------------------------------ helpers
    def _call(self, key, nkernels, fn, *args, flops=0.0, bytes_=0.0):
        """Run one C-ABI call; count its kernels; optionally bracket it with CUDA events on
        the launching stream (bench.py roofline section)."""
        self.launches += nkernels
        if self.profile is None:
            _capi.check(fn(*args))
            return
        if self._tag:
            key = "%s:%s" % (self._tag, key)      # level the call belongs to (bench.py: per-level conv rates)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _capi.check(fn(*args))
        e1.record()
        rec = self.profile.setdefault(key, dict(events=[], flops=0.0, bytes=0.0, launches=0))
        rec["events"].append((e0, e1))
        rec["flops"] += flops
        rec["bytes"] += bytes_
        rec["launches"] += nkernels

    @staticmethod
    def _matfun_launches(C):
        """kernels the matrix-function fast path adds to a WCT call (matfun_tc.cu: norm + init + 3 products x 16 iterations + guard;
        launches of converged matrices return at once but are launches all the same)"""
        return 3 + 3 * 16 if C >= 128 else 0

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _act(self, N, H, W, C):
        nbytes = self.lib.wctb200_act_bytes(N, H, W, C)
        return Act(torch.empty(nbytes, dtype=torch.uint8, device=self.device), N, H, W, C)

    def _workspace(self, C, Nc, Ns):
        key = (self._group, C, Nc, Ns)    # concurrent groups (streams) must not share scratch
        ws = self._ws.get(key)
        if ws is None:
            ws = torch.empty(self.lib.wctb200_wct_workspace_bytes(C, Nc, Ns), dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    # ------------------------------------------------------------------ layers
    def encode(self, img, target, taps=()):
        """img: float32 cuda tensor [N,H,W,3] in [0,1].  Runs the shared encoder up to
        ``target`` (vgg_normalised.py:22-50); returns (act_at_target, {tap: act})."""
        N, H, W, _ = img.shape
        st = self._stream()
        lib = self.lib
        x = self._act(N, H, W, 64)
        self._call("conv_head", 1, lib.wctb200_conv_head, img.data_ptr(), N, H, W, self.head_w.data_ptr(),
                   self.head_b.data_ptr(), x.ptr, st, flops=2.0 * 27 * 64 * N * H * W,
                   bytes_=N * H * W * (12.0 + 64 * 4))
        kept = {}
        if "relu1_1" in taps:
            kept["relu1_1"] = x
        from .model import encoder_plan
        plan = encoder_plan(target)[1:]
        skip_pool = False
        for i, op in enumerate(plan):
            if op.kind == "conv":
                relu_name = op.name.replace("conv", "relu")
                # MaxPooling2D folded into the conv that feeds it (conv1_2 / 2_2 / 3_4 / 4_4: the pool is their only consumer)
                pooled = (self.fuse_pool and i + 1 < len(plan) and plan[i + 1].kind != "conv" and relu_name not in taps
                          and (x.H + 1) // 2 >= 2 and (x.W + 1) // 2 >= 2)
                y = self._act(N, (x.H + 1) // 2, (x.W + 1) // 2, op.cout) if pooled else self._act(N, x.H, x.W, op.cout)
                self._call("conv3x3_%s[%dx%d@%d]" % ("pool" if pooled else "tc", op.cin, op.cout, x.H), 1, lib.wctb200_conv3x3, x.ptr,
                           N, x.H, x.W, op.cin, self.enc_w[op.name].data_ptr(), self.enc_b[op.name].data_ptr(), op.cout,
                           _capi.RELU | (_capi.POOL2 if pooled else 0), y.ptr, st, flops=2.0 * 9 * op.cin * op.cout * N * x.H * x.W,
                           bytes_=4.0 * N * (x.H * x.W * op.cin + y.H * y.W * op.cout))
                x = y
                skip_pool = pooled
                if relu_name in taps:
                    kept[relu_name] = x
            elif skip_pool:
                skip_pool = False
            else:
                y = self._act(N, (x.H + 1) // 2, (x.W + 1) // 2, x.C)
                self._call("maxpool2", 1, lib.wctb200_maxpool2, x.ptr, N, x.H, x.W, x.C, y.ptr, st,
                           bytes_=4.0 * N * x.C * (x.H * x.W + y.H * y.W))
                x = y
        return x, kept

    def decode(self, feat, level_index, clip):
        """Run decoder ``level_index`` (model.py:279-300) -> float32 image [N,H',W',3];
        ``clip`` applies model.py:86's clip_by_value(0,1)."""
        st = self._stream()
        lib = self.lib
        relu = self.model.levels[level_index].relu_target
        x = feat
        N = x.N
        ops = self.model.decoder_plan(level_index)
        pending_up = False                     # an UpSampling2D waiting to be folded into the next conv
        for i, op in enumerate(ops):
            if op.kind == "up":
                if self.fuse_upsample and self._fused_up(ops, i):
                    pending_up = True          # x stays low-resolution (its producer wrote an edge halo)
                    continue
                y = self._act(N, x.H * 2, x.W * 2, x.C)
                self._call("upsample2", 1, lib.wctb200_upsample2, x.ptr, N, x.H, x.W, x.C, y.ptr, st,
                           bytes_=4.0 * N * x.C * x.H * x.W * 5)
                x = y
            elif op.act:
                # a conv whose output feeds a folded upsample writes an EDGE-replicated halo (conv_tc.cu, mode UP2)
                edge = self.fuse_upsample and i + 1 < len(ops) and self._fused_up(ops, i + 1)
                flags = _capi.RELU | (_capi.HALO_EDGE if edge else 0)
                if pending_up:
                    y = self._act(N, 2 * x.H, 2 * x.W, op.cout)
                    self._call("conv3x3_up2[%dx%d@%d]" % (op.cin, op.cout, y.H), 1, lib.wctb200_conv3x3_up2, x.ptr, N, x.H, x.W,
                               op.cin, self.dec_w[op.name].data_ptr(), self.dec_b[op.name].data_ptr(), op.cout,
                               flags, y.ptr, st, flops=2.0 * 4 * op.cin * op.cout * N * y.H * y.W,
                               bytes_=4.0 * N * (x.H * x.W * op.cin + y.H * y.W * op.cout))
                    pending_up = False
                else:
                    y = self._act(N, x.H, x.W, op.cout)
                    self._call("conv3x3_tc[%dx%d@%d]" % (op.cin, op.cout, x.H), 1, lib.wctb200_conv3x3, x.ptr, N, x.H, x.W,
                               op.cin, self.dec_w[op.name].data_ptr(), self.dec_b[op.name].data_ptr(), op.cout,
                               flags, y.ptr, st, flops=2.0 * 9 * op.cin * op.cout * N * x.H * x.W,
                               bytes_=4.0 * N * x.H * x.W * (op.cin + op.cout))
                x = y
            else:
                assert not pending_up
                img = torch.empty((N, x.H, x.W, 3), dtype=torch.float32, device=self.device)
                self._call("conv_tail", 1, lib.wctb200_conv_tail, x.ptr, N, x.H, x.W, op.cin, self.tail_w[relu].data_ptr(),
                           self.tail_b[relu].data_ptr(), _capi.CLIP01 if clip else 0, img.data_ptr(), st,
                           flops=2.0 * 9 * op.cin * 3 * N * x.H * x.W, bytes_=N * x.H * x.W * (4.0 * op.cin + 12))
                return img
        raise AssertionError("decoder plan without a tail conv")

    def transform(self, content, style, alpha, adain, want_info=False):
        """wct_tf / wct_np / adain on one level (model.py:144-158)."""
        st = self._stream()
        out = self._act(content.N, content.H, content.W, content.C)
        ws = self._workspace(content.C, content.N, style.N)
        if adain:
            self._call("adain_level[C%d]" % content.C, 6, self.lib.wctb200_adain_level, content.ptr, content.N, content.H,
                       content.W, style.ptr, style.N, style.H, style.W, content.C, float(alpha), 1e-5, out.ptr,
                       ws.data_ptr(), ws.numel(), st,
                       bytes_=4.0 * content.C * (2 * content.N * content.H * content.W + style.N * style.H * style.W))
            return out, None
        sem = SEMANTICS[self.semantics]
        kbuf = torch.empty(2 * (content.N + style.N), dtype=torch.int32, device=self.device) if want_info else None
        C = content.C
        hwc, hws = content.H * content.W, style.H * style.W
        self._call("wct_level[C%d]" % C, 14 + self._matfun_launches(C), self.lib.wctb200_wct_level, content.ptr, content.N, content.H, content.W,
                   style.ptr, style.N, style.H, style.W, C, float(alpha), sem["eps_cov"], sem["eps_eig"],
                   sem["thresh"], sem["readd"], out.ptr, kbuf.data_ptr() if want_info else None, ws.data_ptr(),
                   ws.numel(), st, flops=2.0 * C * C * (2 * content.N * hwc + style.N * hws),
                   bytes_=4.0 * C * (2 * content.N * hwc + style.N * hws))
        return out, kbuf

    def style_swap(self, content, style, ss_alpha, want_info=False, patch=3, stride=1):
        """wct_style_swap (ops.py:145-217) on one content/style pair with ``patch`` x ``patch`` windows every ``stride``."""
        assert content.N == 1 and style.N == 1, "style swap works on one content/style pair (ops.py:146)"
        st = self._stream()
        C = content.C
        out = self._act(1, content.H, content.W, C)
        nbytes = self.lib.wctb200_style_swap_workspace_bytes(C, content.H, content.W, style.H, style.W, int(patch), int(stride))
        if nbytes == 0:
            raise ValueError("style swap needs encodings of at least %dx%d (content %dx%d, style %dx%d)"
                             % (patch, patch, content.H, content.W, style.H, style.W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        kbuf = torch.empty(4, dtype=torch.int32, device=self.device) if want_info else None
        sem = SEMANTICS["tf"]                  # the reference only has the TF graph version of this op
        self._call("style_swap[C%d]" % C, 22, self.lib.wctb200_style_swap_level, content.ptr, content.H, content.W, style.ptr,
                   style.H, style.W, C, int(patch), int(stride), float(ss_alpha), sem["eps_cov"], sem["thresh"], out.ptr,
                   kbuf.data_ptr() if want_info else None, ws.data_ptr(), ws.numel(), st)
        ws.record_stream(torch.cuda.current_stream(self.device))   # freed by the caching allocator only after this stream is done
        return out, kbuf

    def style_prepare(self, style):
        """Style side of one level (ops.py:48-55,76): means, covariance, eigendecomposition, C_s.
        Returns the device state buffer consumed by ``wct_apply``."""
        st = self._stream()
        sem = SEMANTICS[self.semantics]
        C = style.C
        state = torch.empty(self.lib.wctb200_wct_style_state_bytes(C, style.N), dtype=torch.uint8, device=self.device)
        ws = self._workspace(C, 0, style.N)
        hws = style.H * style.W
        self._call("wct_style[C%d]" % C, 7 + self._matfun_launches(C), self.lib.wctb200_wct_style_prepare, style.ptr, style.N, style.H, style.W, C,
                   sem["eps_cov"], sem["eps_eig"], sem["thresh"], state.data_ptr(), ws.data_ptr(), ws.numel(), st,
                   flops=2.0 * C * C * style.N * hws, bytes_=4.0 * C * style.N * hws)
        return state

    def wct_apply(self, content, state, n_style, alpha, want_info=False):
        st = self._stream()
        sem = SEMANTICS[self.semantics]
        C = content.C
        out = self._act(content.N, content.H, content.W, C)
        ws = self._workspace(C, content.N, 0)
        kbuf = torch.empty(2 * (content.N + n_style), dtype=torch.int32, device=self.device) if want_info else None
        hwc = content.H * content.W
        self._call("wct_level[C%d]" % C, 9 + self._matfun_launches(C), self.lib.wctb200_wct_apply, content.ptr, content.N, content.H, content.W, C,
                   state.data_ptr(), n_style, float(alpha), sem["eps_cov"], sem["eps_eig"], sem["thresh"], sem["readd"],
                   out.ptr, kbuf.data_ptr() if want_info else None, ws.data_ptr(), ws.numel(), st,
                   flops=2.0 * C * C * 2 * content.N * hwc, bytes_=4.0 * C * 2 * content.N * hwc)
        return out, kbuf

    # ------------------------------------------------------------------ spatial control
    MAX_REGIONS = 8

    def labels_resize(self, labels, H, W):
        """Nearest-neighbour resize of cuda uint8 label maps [N,Hs,Ws] -> [N,H,W] (exact integer rule, include/wctb200.h)."""
        labels = labels.contiguous()
        N, Hs, Ws = labels.shape
        if (Hs, Ws) == (H, W):
            return labels
        out = torch.empty((N, H, W), dtype=torch.uint8, device=self.device)
        self._call("labels_nearest", 1, self.lib.wctb200_labels_resize_nearest, labels.data_ptr(), N, Hs, Ws, H, W, out.data_ptr(),
                   self._stream())
        return out

    def _regions_workspace(self, C, Nc, R):
        key = ("regions", self._group, C, Nc, R)
        ws = self._ws.get(key)
        if ws is None:
            ws = torch.empty(self.lib.wctb200_wct_regions_workspace_bytes(C, Nc, R), dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    def wct_apply_regions(self, content, labels, states, alpha, want_info=False):
        """One level with one style state per region; ``labels`` cuda uint8 [N, content.H, content.W]."""
        st = self._stream()
        sem = SEMANTICS[self.semantics]
        C, R, N = content.C, len(states), content.N
        out = self._act(N, content.H, content.W, C)
        ws = self._regions_workspace(C, N, R)
        kbuf = torch.empty(2 * N * R, dtype=torch.int32, device=self.device) if want_info else None
        ptrs = (ctypes.c_void_p * R)(*[s.data_ptr() for s in states])
        hwc = content.H * content.W
        self._call("wct_regions[C%d]" % C, 13 + R + self._matfun_launches(C), self.lib.wctb200_wct_apply_regions, content.ptr, N,
                   content.H, content.W, C, labels.data_ptr(), R, ctypes.cast(ptrs, ctypes.c_void_p), float(alpha), sem["eps_cov"],
                   sem["eps_eig"], sem["thresh"], sem["readd"], out.ptr, kbuf.data_ptr() if want_info else None, ws.data_ptr(),
                   ws.numel(), st, flops=2.0 * C * C * (R + 1) * N * hwc, bytes_=4.0 * C * (R + 1) * N * hwc)
        return out, kbuf

    def adain_regions(self, content, labels, styles, alpha):
        st = self._stream()
        C, R, N = content.C, len(styles), content.N
        out = self._act(N, content.H, content.W, C)
        ws = self._regions_workspace(C, N, R)
        ptrs = (ctypes.c_void_p * R)(*[s.ptr for s in styles])
        hw = (ctypes.c_int * (2 * R))(*[v for s in styles for v in (s.H, s.W)])
        self._call("adain_regions[C%d]" % C, 6 + 2 * R, self.lib.wctb200_adain_regions, content.ptr, N, content.H, content.W, C,
                   labels.data_ptr(), R, ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(hw, ctypes.c_void_p), float(alpha), 1e-5,
                   out.ptr, ws.data_ptr(), ws.numel(), st)
        return out, None

    def _check_labels(self, content_u8, styles, labels, swap5):
        if swap5:
            raise ValueError("style swap (swap5) cannot be combined with a label mask: it is not a per-region statistic")
        R = len(styles)
        if not 1 <= R <= self.MAX_REGIONS:
            raise ValueError("a label mask takes 1..%d styles, got %d" % (self.MAX_REGIONS, R))
        for s in styles:
            if s.dim() != 4 or s.shape[0] != 1 or s.dtype != torch.uint8:
                raise ValueError("each region style must be a uint8 [1,Hs,Ws,3] tensor")
        N, H, W = content_u8.shape[:3]
        if labels.dtype != torch.uint8 or labels.dim() != 3 or labels.shape[0] not in (1, N) or tuple(labels.shape[1:]) != (H, W):
            raise ValueError("labels must be uint8 [N|1, %d, %d] (the content's size), got %s %s"
                             % (H, W, tuple(labels.shape), labels.dtype))
        if labels.device != self.device:
            labels = labels.to(self.device)
        if labels.shape[0] != N:
            labels = labels.expand(N, H, W)
        return labels.contiguous()

    # ------------------------------------------------------------------ pipeline
    def stylize(self, content_u8, style_u8, alpha=1.0, adain=False, want_info=False, capture=None, swap5=False, ss_alpha=0.6,
                ss_patch_size=3, ss_stride=1, labels=None):
        """content_u8: cuda uint8 [N,H,W,3]; style_u8: cuda uint8 [Ns,Hs,Ws,3], Ns in {1, N}.
        Returns the float32 ``decoded_output`` [N,H',W',3] (unclipped, model.py:94).
        ``capture`` (dict) receives every level's input image / features for parity tests.

        With ``self.groups`` = G > 1 the batch is cut into G sub-batches whose level chains are
        enqueued on G independent stream pairs: frames are independent (wct.py:97-103), and the
        eigendecompositions are latency bound on a few SMs, so one group's Jacobi clusters overlap the
        other groups' convolutions (same arithmetic per frame; only the schedule changes).

        ``labels`` (cuda uint8 [N|1,H,W], the content's size): spatial control.  ``style_u8`` is then a sequence of R <= 8
        uint8 [1,Hs_r,Ws_r,3] styles; label r < R takes style r, labels >= R keep the content (include/wctb200.h)."""
        if labels is not None:
            styles = list(style_u8)
            labels = self._check_labels(content_u8, styles, labels, swap5)
            return self._stylize_regions(content_u8, styles, labels, alpha, adain, want_info, capture)
        N = content_u8.shape[0]
        swap5 = bool(swap5) and "relu5_1" in [l.relu_target for l in self.model.levels]    # model.py:148: only relu5_1 swaps
        if swap5:
            if N != 1 or style_u8.shape[0] != 1:
                raise ValueError("swap5 works on one content/style pair per call (ops.py:146)")
            return self._stylize_one(content_u8, style_u8, alpha, adain, want_info, capture, True, ss_alpha,
                                     ss_patch=ss_patch_size, ss_stride=ss_stride)
        G = min(self.groups, N) if (capture is None and not want_info) else 1
        if G > 1:
            main = torch.cuda.current_stream(self.device)
            bounds = [(g * N) // G for g in range(G + 1)]
            outs = []
            shared = None
            if style_u8.shape[0] == 1 and not adain:
                # ONE style for the whole batch (video, configs[2]): its encoder pass and eigendecompositions run once,
                # every sub-batch group waits for the per-level events
                self._group = 1
                try:
                    shared = self._style_side(style_u8, True, main)
                finally:
                    self._group = 0
            for g in range(G):
                lo, hi = bounds[g], bounds[g + 1]
                if g not in self._group_streams:
                    # descending priority: group 0 runs "in the foreground", later groups fill the SMs it
                    # leaves idle while its eigendecompositions are latency bound (self.group_priorities)
                    prio = -1 if (self.group_priorities and g == 0) else 0
                    self._group_streams[g] = torch.cuda.Stream(device=self.device, priority=prio)
                gs = self._group_streams[g]
                gs.wait_stream(main)
                self._group = g + 1
                try:
                    with torch.cuda.stream(gs):
                        sg = style_u8 if style_u8.shape[0] == 1 else style_u8[lo:hi]
                        outs.append(self._stylize_one(content_u8[lo:hi], sg, alpha, adain, False, None, shared_style=shared))
                finally:
                    self._group = 0
            for g in range(G):
                main.wait_stream(self._group_streams[g])
            out = torch.cat(outs, dim=0)
            for g in range(G):                      # sub-batch buffers die here: their streams wait for the cat
                self._group_streams[g].wait_stream(main)
            if shared is not None and shared["side"] is not main:
                shared["side"].wait_stream(main)    # the shared style states are recycled only after every group used them
            return out
        return self._stylize_one(content_u8, style_u8, alpha, adain, want_info, capture)

    def _stylize_regions(self, content_u8, styles, labels, alpha, adain, want_info, capture):
        """The masked form of ``stylize``: every style's encoder pass (and, for the WCT, its per-level preparation) runs
        once on the style stream; with groups > 1 every sub-batch waits on those events."""
        N = content_u8.shape[0]
        main = torch.cuda.current_stream(self.device)
        G = min(self.groups, N) if (capture is None and not want_info) else 1
        if G <= 1:
            shared = [self._style_side(s, not adain, main) for s in styles]
            out = self._stylize_one(content_u8, None, alpha, adain, want_info, capture, labels=labels, region_styles=shared)
            for sh in shared:
                if sh["side"] is not main:
                    sh["side"].wait_stream(main)
            return out
        self._group = 1
        try:
            shared = [self._style_side(s, not adain, main) for s in styles]
        finally:
            self._group = 0
        bounds = [(g * N) // G for g in range(G + 1)]
        outs = []
        for g in range(G):
            lo, hi = bounds[g], bounds[g + 1]
            if g not in self._group_streams:
                prio = -1 if (self.group_priorities and g == 0) else 0
                self._group_streams[g] = torch.cuda.Stream(device=self.device, priority=prio)
            gs = self._group_streams[g]
            gs.wait_stream(main)
            self._group = g + 1
            try:
                with torch.cuda.stream(gs):
                    outs.append(self._stylize_one(content_u8[lo:hi], None, alpha, adain, False, None, labels=labels[lo:hi],
                                                  region_styles=shared))
            finally:
                self._group = 0
        for g in range(G):
            main.wait_stream(self._group_streams[g])
        out = torch.cat(outs, dim=0)
        for g in range(G):
            self._group_streams[g].wait_stream(main)
        for sh in shared:
            if sh["side"] is not main:
                sh["side"].wait_stream(main)
        return out

    def _style_side(self, style_u8, split, main):
        """Style side of one call (model.py:70-72: ONE encoder pass emitting every target; ops.py:48-55,76 per level when
        ``split``): enqueued on this group's style stream when overlap is on.  Returns the states / events / features."""
        lib = self.lib
        side = main
        if split and self.overlap_style:
            if self._group not in self._style_streams:
                prio = -1 if (self.group_priorities and self._group <= 1) else 0
                self._style_streams[self._group] = torch.cuda.Stream(device=self.device, priority=prio)
            side = self._style_streams[self._group]
            side.wait_stream(main)             # style_u8 (and last step's buffers) are ready
        states, events, feats = {}, {}, None
        with torch.cuda.stream(side):
            tag, self._tag = self._tag, "style"
            style = torch.empty(style_u8.shape, dtype=torch.float32, device=self.device)
            self._call("u8_to_f32", 1, lib.wctb200_image_u8_to_f32, style_u8.data_ptr(), style_u8.numel(), style.data_ptr(),
                       self._stream())
            _, feats = self.encode(style, self.model.deepest_target, taps=self.model.style_taps)
            if split:
                for relu in self.model.style_taps:
                    if relu not in states:
                        states[relu] = self.style_prepare(feats[relu])
                        ev = torch.cuda.Event()
                        ev.record(side)
                        events[relu] = ev
            self._tag = tag
        return dict(states=states, events=events, feats=feats, side=side)

    def _stylize_one(self, content_u8, style_u8, alpha, adain, want_info, capture, swap5=False, ss_alpha=0.6, shared_style=None,
                     ss_patch=3, ss_stride=1, labels=None, region_styles=None):
        lib, st = self.lib, self._stream()
        N = content_u8.shape[0]
        assert content_u8.dtype == torch.uint8
        assert labels is not None or (style_u8.dtype == torch.uint8 and style_u8.shape[0] in (1, N))
        content = torch.empty(content_u8.shape, dtype=torch.float32, device=self.device)
        self._call("u8_to_f32", 1, lib.wctb200_image_u8_to_f32, content_u8.data_ptr(), content_u8.numel(), content.data_ptr(), st)
        main = torch.cuda.current_stream(self.device)
        split = not adain and not swap5        # WCT: style side on its own stream; AdaIN / style swap: keep it inline
        if labels is None:
            ss = shared_style if (shared_style is not None and split) else self._style_side(style_u8, split, main)
            side, style_states, style_events, style_feats = ss["side"], ss["states"], ss["events"], ss["feats"]
            n_style = style_u8.shape[0]
        else:
            side = main                        # the region styles' streams are joined by _stylize_regions
        infos = []
        x = content
        nlev = len(self.model.levels)
        for lvl in self.model.levels:
            self._tag = lvl.relu_target
            cf, _ = self.encode(x, lvl.relu_target)
            if labels is not None:
                relu = lvl.relu_target
                lab = self.labels_resize(labels, cf.H, cf.W)     # always from the call's label map (the decoder may grow odd sizes)
                if adain:
                    f, kbuf = self.adain_regions(cf, lab, [rs["feats"][relu] for rs in region_styles], alpha)
                else:
                    for rs in region_styles:
                        if rs["side"] is not main:
                            main.wait_event(rs["events"][relu])
                    f, kbuf = self.wct_apply_regions(cf, lab, [rs["states"][relu] for rs in region_styles], alpha, want_info)
            elif swap5 and lvl.relu_target == "relu5_1":     # model.py:148-152: style swap wins over AdaIN / WCT at relu5_1
                f, kbuf = self.style_swap(cf, style_feats[lvl.relu_target], ss_alpha, want_info, ss_patch, ss_stride)
            elif split:
                if side is not main:
                    main.wait_event(style_events[lvl.relu_target])
                f, kbuf = self.wct_apply(cf, style_states[lvl.relu_target], n_style, alpha, want_info)
            else:
                f, kbuf = self.transform(cf, style_feats[lvl.relu_target], alpha, adain, want_info)
            infos.append(kbuf)
            if capture is not None:
                capture.setdefault("level_input", []).append(x)
                capture.setdefault("content_feat", []).append(cf)
                capture.setdefault("transformed", []).append(f)
            # model.py:86: clip between levels; model.py:94: last output unclipped
            x = self.decode(f, lvl.index, clip=(lvl.index < nlev - 1))
            if capture is not None:
                capture.setdefault("level_output", []).append(x)
        self._tag = None
        if side is not main and shared_style is None:
            side.wait_stream(main)             # buffers handed across streams may be recycled only after both are done
            main.wait_stream(side)
        if want_info:
            self.last_info = infos
        return x

    def to_u8(self, img_f32):
        """WCT.postprocess (wct.py:66-68)."""
        out = torch.empty(img_f32.shape, dtype=torch.uint8, device=self.device)
        self._call("f32_to_u8", 1, self.lib.wctb200_image_f32_to_u8, img_f32.data_ptr(), img_f32.numel(), out.data_ptr(),
                   self._stream())
        return out

    def act_to_f32(self, act):
        out = torch.empty((act.N, act.H, act.W, act.C), dtype=torch.float32, device=self.device)
        _capi.check(self.lib.wctb200_act_to_f32(act.ptr, act.N, act.H, act.W, act.C, out.data_ptr(), self._stream()))
        return out

    def act_from_f32(self, t):
        N, H, W, C = t.shape
        a = self._act(N, H, W, C)
        t = t.contiguous()
        _capi.check(self.lib.wctb200_act_from_f32(t.data_ptr(), N, H, W, C, a.ptr, self._stream()))
        return a

    def check_device(self):
        _capi.check(self.lib.wctb200_check_device(self._stream()))
