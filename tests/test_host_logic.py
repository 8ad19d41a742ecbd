"""CPU tests of the host-side logic: level-wiring bookkeeping (bit-exact against the
reference's tables), weight IO, the C-ABI surface, frame sharding (gloo, world_size 2)."""
import ctypes
import itertools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import nets
from wct_tf_b200 import model as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_decoder_plan_matches_reference_naming():
    for relu in M.RELU_TARGETS_ALL:
        ours = [(op.kind, op.name, op.cout if op.kind == "conv" else None) for op in M.decoder_plan(relu)]
        ref = [(t, n, f) for t, n, f, _ in nets.decoder_layers(relu)]
        assert ours == ref
    p5 = M.decoder_plan("relu5_1")
    assert [op.name for op in p5] == ["relu5_1_%d" % i for i in range(17)]          # model.py:283-298
    assert [(op.cin, op.cout) for op in p5 if op.kind == "conv"][-1] == (64, 3)
    assert sum(op.kind == "up" for op in p5) == 4


def test_encoder_plan_matches_reference_module_walk():
    for relu in M.RELU_TARGETS_ALL:
        ours = [op.name for op in M.encoder_plan(relu)]
        ref = []
        for typ, name in nets.VGG_MODULES[1:]:
            if typ in ("conv", "pool"):
                ref.append(name)
            if name == relu:
                break
        assert ours == ref
    assert [op.name for op in M.encoder_plan("relu1_1")] == ["conv1_1"]
    assert sum(op.kind == "pool" for op in M.encoder_plan("relu5_1")) == 4


@pytest.mark.parametrize("r", [1, 2, 3, 5])
def test_level_wiring_for_every_ordered_subset(r):
    for targets in itertools.permutations(M.RELU_TARGETS_ALL, r):
        m = M.WCTModel(mode="test", relu_targets=list(targets))
        assert m.deepest_target == sorted(targets)[-1]                               # model.py:60
        assert [l.relu_target for l in m.levels] == list(targets)                   # zip order, model.py:78
        assert [l.clip_input for l in m.levels] == [False] + [True] * (r - 1)        # model.py:86, not the first
        assert m.style_taps == list(targets)                                         # model.py:70
        assert [l.channels for l in m.levels] == [M.RELU_CHANNELS[t] for t in targets]
        # the style plan reaches every tap
        names = [op.name.replace("conv", "relu") for op in m.style_plan if op.kind == "conv"]
        assert all(t in names for t in targets)


def test_transform_rule_matches_tf_case():
    # model.py:144-158
    assert M.WCTModel.transform_for("relu5_1", True, True) == "style_swap"
    assert M.WCTModel.transform_for("relu5_1", False, True) == "adain"
    assert M.WCTModel.transform_for("relu5_1", False, False) == "wct"
    assert M.WCTModel.transform_for("relu4_1", True, False) == "wct"     # swap5 only applies at relu5_1
    assert M.WCTModel.transform_for("relu4_1", True, True) == "adain"
    with pytest.raises(NotImplementedError):
        M.WCTModel(mode="train")
    with pytest.raises(ValueError):
        M.WCTModel(mode="test", relu_targets=["relu6_1"])


def test_weights_roundtrip_and_checkpoint_pairing(tmp_path):
    from wct_tf_b200 import weights as W
    w = W.make_synthetic_weights(1, relu_targets=["relu2_1", "relu1_1"])
    assert [l["name"] for l in w["vgg"]][:3] == ["preprocess", "conv1_1", "conv1_2"]
    assert w["vgg"][1]["weight"].shape == (64, 3, 3, 3)                              # (O,I,kH,kW), vgg_normalised.py:33
    assert w["decoders"]["relu2_1"][0]["kernel"].shape == (3, 3, 128, 64)
    p = str(tmp_path / "bundle.npz")
    W.save_weights(p, w)
    w2 = W.load_weights(p, [p, p], ["relu2_1", "relu1_1"])
    for a, b in zip(w["decoders"]["relu2_1"], w2["decoders"]["relu2_1"]):
        assert a["name"] == b["name"] and np.array_equal(a["kernel"], b["kernel"])
    assert np.array_equal(w["vgg"][5]["weight"], w2["vgg"][5]["weight"])
    with pytest.raises(Exception, match="No checkpoint found"):                        # wct.py:57-58
        W.load_weights(p, [p, p], ["relu2_1", "relu3_1"])
    w3 = W.make_synthetic_weights(1, relu_targets=["relu2_1", "relu1_1"])
    assert np.array_equal(w["vgg"][7]["weight"], w3["vgg"][7]["weight"])             # deterministic in the seed


def test_capi_exports_every_declared_symbol():
    """The shared library loads on a CPU-only box and exports exactly what include/wctb200.h declares."""
    from wct_tf_b200 import _capi
    header = open(os.path.join(ROOT, "include", "wctb200.h")).read()
    declared = set(re.findall(r"WCTB200_API[^;]*?\b(wctb200_\w+)\s*\(", header))
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    lib = _capi.load()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.wctb200_abi_version() == 1
    # argument validation runs before any CUDA call
    assert lib.wctb200_act_bytes(2, 4, 6, 64) == 2 * 2 * 6 * 8 * 64 * 2
    assert lib.wctb200_act_bytes(1, 1, 4, 64) == 0
    assert lib.wctb200_conv3x3(None, 1, 4, 4, 64, None, None, 64, 0, None, None) == -1
    assert b"null" in lib.wctb200_last_error()
    assert lib.wctb200_wct_workspace_bytes(512, 1, 1) > 6 * 512 * 512 * 4


def test_device_string_mapping_and_no_cpu_fallback():
    from wct_tf_b200.wct import _torch_device
    assert _torch_device("/gpu:0") == "cuda:0" and _torch_device("/GPU:3") == "cuda:3"
    assert _torch_device("cuda:1") == "cuda:1"
    with pytest.raises(ValueError):
        _torch_device("/cpu:0")
    import torch
    if not torch.cuda.is_available():
        from wct_tf_b200 import _capi
        from wct_tf_b200.engine import Engine
        from wct_tf_b200.weights import make_synthetic_weights
        with pytest.raises(_capi.WctB200Error):     # the product path fails loudly without a GPU
            Engine(make_synthetic_weights(0, relu_targets=["relu1_1"]), ["relu1_1"])


def test_shard_range_partition():
    from wct_tf_b200.parallel import owner_of, shard_range
    for B in [1, 3, 8, 64, 65]:
        for G in [1, 2, 4, 8]:
            cover = []
            for r in range(G):
                lo, hi = shard_range(B, G, r)
                cover += list(range(lo, hi))
                for i in range(lo, hi):
                    assert owner_of(i, B, G) == r
            assert cover == list(range(B))
    assert [shard_range(64, 8, r) for r in (0, 7)] == [(0, 8), (56, 64)]


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from wct_tf_b200.parallel import stylize_sharded
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%%s" %% sys.argv[1], rank=int(sys.argv[2]), world_size=2)
B = int(sys.argv[3])
contents = (torch.arange(B, dtype=torch.uint8).view(B, 1, 1, 1) * torch.ones(B, 4, 6, 3, dtype=torch.uint8))
styles = torch.full((B, 2, 2, 3), 7, dtype=torch.uint8)
seen = []
def fake_engine(c, s):           # stands in for WCT.predict_batch: marks which rank processed the frame
    seen.append(c.shape[0])
    return c + 100 + 10 * dist.get_rank() + s[:, :1, :1, :1] * 0
out = stylize_sharded(fake_engine, contents, styles)
exp = torch.stack([torch.full((4, 6, 3), i + 100 + 10 * ((i * 2) // B), dtype=torch.uint8) for i in range(B)])
assert out.shape == (B, 4, 6, 3) and torch.equal(out, exp), (out[:, 0, 0, 0], exp[:, 0, 0, 0])
assert sum(seen) == (B + 1 - dist.get_rank()) // 2 if B %% 2 else sum(seen) == B // 2
dist.destroy_process_group()
print("ok")
""" % ROOT


@pytest.mark.parametrize("B", [4, 5])
def test_frame_sharding_world2_gloo(B, tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + (os.getpid() % 400) + B)
    procs = [subprocess.Popen([sys.executable, str(script), port, str(r), str(B)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)


def test_t7_reader_against_reference_torchfile(tmp_path):
    """A VGG .t7 written by tests/t7_writer.py is read identically by the reference's own
    torchfile.py (vgg_normalised.py:16, force_8bytes_long=True) and by wct_tf_b200.t7.  What the
    reference read from this very file is stored in tests/golden/reference_reads.npz
    (tests/golden/make_reference_reads.py)."""
    from tests.golden import make_reference_reads as R
    from tests.t7_writer import write_vgg_t7
    from wct_tf_b200 import t7, weights as W
    w = W.make_synthetic_weights(R.T7_SEED, relu_targets=R.T7_TARGETS)
    path = str(tmp_path / "vgg_normalised.t7")
    write_vgg_t7(path, w["vgg"])
    ours = t7.load_vgg_t7(path, deepest="relu5_1")
    assert [l["name"] for l in ours] == [l["name"] for l in w["vgg"]]
    for a, b in zip(ours, w["vgg"]):
        assert np.array_equal(a["weight"], b["weight"]) and np.array_equal(a["bias"], b["bias"])
    assert [l["name"] for l in t7.load_vgg_t7(path, deepest="relu2_1")][-1] == "conv2_1"    # stops at the target (vgg_normalised.py:48)
    ref = np.load(os.path.join(ROOT, "tests", "golden", "reference_reads.npz"))
    assert R.file_digest(path) == str(ref["torchfile_t7_sha256"]), "not the file the reference read (writer or weights drifted)"
    convs = [str(d) for d in ref["torchfile_conv_digests"]]
    assert len(convs) == len(ours)
    for d, o in zip(convs, ours):
        assert R.array_digest(o["weight"], o["bias"]) == d, o["name"]
    assert [str(n) for n in ref["torchfile_conv_names"]] == [l["name"] for l in ours[1:]]
    # and through the public loader: checkpoints stay .npz
    ck = str(tmp_path / "dec.npz")
    W.save_weights(ck, w)
    w2 = W.load_weights(path, [ck], ["relu3_1"])
    assert np.array_equal(w2["vgg"][3]["weight"], w["vgg"][3]["weight"])
    assert [l["name"] for l in w2["vgg"]][-1] == "conv3_1"


def test_tf_checkpoint_reader_and_reference_loading_protocol(tmp_path):
    """Decoders come from TF1 Saver checkpoint DIRECTORIES like the reference (wct.py:45-58), the encoder from a .t7:
    the TF-free bundle reader returns exactly what tests/tf_bundle_writer.py stored, ignores optimizer slots and
    raises the reference's exception for an empty directory."""
    from tests.t7_writer import write_vgg_t7
    from tests.tf_bundle_writer import write_bundle
    from wct_tf_b200 import tf_checkpoint as T, weights as W
    targets = ["relu2_1", "relu3_1"]
    w = W.make_synthetic_weights(9, relu_targets=targets)
    write_vgg_t7(str(tmp_path / "vgg_normalised.t7"), w["vgg"])
    dirs = []
    for t in targets:
        tensors = {}
        for l in w["decoders"][t]:
            scope = "encoder_decoder_%s/decoder_%s/decoder_model_%s/%s/%s" % (t, t, t, l["name"], l["name"])
            tensors[scope + "/kernel"] = l["kernel"]
            tensors[scope + "/bias"] = l["bias"]
            tensors[scope + "/kernel/Adam"] = np.ones_like(l["kernel"])          # optimizer slots must be ignored
            tensors[scope + "/kernel/Adam_1"] = np.ones_like(l["kernel"])
        tensors["encoder_decoder_%s/train_%s/global_step_train" % (t, t)] = np.array(15000, dtype=np.int64)
        d = tmp_path / ("ckpt_" + t)
        write_bundle(str(d / "model.ckpt-15000"), tensors)
        dirs.append(str(d))
    assert T.crc32c(b"123456789") == 0xE3069283                                  # CRC-32C check value
    raw = T.read_bundle(T.latest_checkpoint(dirs[0]))
    assert int(raw["encoder_decoder_relu2_1/train_relu2_1/global_step_train"]) == 15000
    w2 = W.load_weights(str(tmp_path / "vgg_normalised.t7"), dirs, targets)
    for t in targets:
        assert [l["name"] for l in w2["decoders"][t]] == [l["name"] for l in w["decoders"][t]]
        for a, b in zip(w2["decoders"][t], w["decoders"][t]):
            assert np.array_equal(a["kernel"], b["kernel"]) and np.array_equal(a["bias"], b["bias"])
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(Exception, match="No checkpoint found for target relu3_1"):
        W.load_weights(str(tmp_path / "vgg_normalised.t7"), [dirs[0], str(empty)], targets)
    # a flipped byte in the shard is caught by the per-tensor checksum
    prefix = T.latest_checkpoint(dirs[1])
    blob = bytearray(open(prefix + ".data-00000-of-00001", "rb").read())
    blob[100] ^= 0xFF
    open(prefix + ".data-00000-of-00001", "wb").write(bytes(blob))
    with pytest.raises(T.TFCheckpointError, match="checksum"):
        T.read_bundle(prefix, verify=True)
    with pytest.raises(T.TFCheckpointError, match="checksum"):                   # default too: a corrupt TENSOR is always fatal
        T.read_bundle(prefix)                                                    # (only index-block CRCs merely warn)
    assert len(T.read_bundle(prefix, verify=False)) > 0
    # a decoder checkpoint that lacks a layer is reported as such, not as a KeyError later in the engine
    short = {k: v for k, v in tensors.items() if "/%s_0/" % targets[-1] not in k}
    write_bundle(str(tmp_path / "short" / "model.ckpt-1"), short)
    with pytest.raises(T.TFCheckpointError, match="lacks layer"):
        T.load_decoder_checkpoint(str(tmp_path / "short"), targets[-1])


def test_tf_checkpoint_snappy_block_decoder():
    """Index blocks may be snappy-compressed (LevelDB block type 1): literals, 1/2-byte-offset copies, overlapping copies."""
    from wct_tf_b200.tf_checkpoint import _snappy_decompress
    # "abcdabcdabcdabcdXYZ": literal "abcd", copy(len 12, offset 4) with a 2-byte offset, literal "XYZ"
    comp = bytes([19, (4 - 1) << 2]) + b"abcd" + bytes([((12 - 1) << 2) | 2, 4, 0]) + bytes([(3 - 1) << 2]) + b"XYZ"
    assert _snappy_decompress(comp) == b"abcdabcdabcdabcdXYZ"
    # copy with a 1-byte offset (tag type 1: len 4..11, offset < 2048): "xyxyxyxyxy"
    comp = bytes([10, (2 - 1) << 2]) + b"xy" + bytes([((8 - 4) << 2) | 1, 2])
    assert _snappy_decompress(comp) == b"xy" * 5


def test_device_image_geometry_matches_the_oracle_helpers(monkeypatch):
    """wct_tf_b200.device_image computes sizes and crop windows on the host and hands them to ONE device resample call; the
    arithmetic (utils.py:29-67: short-side rule with Python-3 rounding, upscale-when-too-small, centred windows) is checked here
    against the oracle's shapes without a GPU by intercepting the resample call."""
    import torch
    from oracle import image_ops as O
    from wct_tf_b200 import device_image as D

    calls = []

    def fake_imresize(img, hw, window=None):
        h, w = (img.shape[0], img.shape[1])
        calls.append((h, w, tuple(int(v) for v in hw), None if window is None else tuple(int(v) for v in window)))
        oh, ow = (hw if window is None else window[2:])
        return torch.zeros((int(oh), int(ow), 3), dtype=torch.uint8)

    monkeypatch.setattr(D, "imresize", fake_imresize)
    rng = np.random.default_rng(0)
    for (h, w) in [(40, 64), (64, 40), (37, 37), (300, 451), (5, 9), (501, 333)]:
        img_np = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        img = torch.from_numpy(img_np)
        for size in (16, 25, 96, 512):
            assert tuple(D.resize_to(img, size).shape) == O.resize_to(img_np, size).shape
            assert tuple(D.center_crop(img, size).shape) == O.center_crop(img_np, size).shape
            hh, ww, hw, win = calls[-1]
            assert win[2:] == (size, size) and win[0] == (hw[0] - size) // 2 and win[1] == (hw[1] - size) // 2
            assert win[0] >= 0 and win[1] >= 0 and win[0] + size <= hw[0] and win[1] + size <= hw[1]
        for (ht, wt) in [(32, 32), (h, w), (h + 9, w), (h, 2 * w), (96, 112)]:
            assert tuple(D.center_crop_to(img, ht, wt).shape) == O.center_crop_to(img_np, ht, wt).shape
            hh, ww, hw, win = calls[-1]
            assert win[0] + ht <= hw[0] and win[1] + wt <= hw[1]
