"""Generate tests/golden/reference_reads.npz by running the REFERENCE's own code (needs its source tree at np_tf1.REF_DIR).

  python tests/golden/make_reference_reads.py

Three tests compare with what the reference code itself returns.  The reference is not part of this
repository, so its answers are stored here once:

* torchfile_*  what the reference's torchfile.py (vgg_normalised.py:16, force_8bytes_long=True) reads from the
  VGG .t7 that tests/t7_writer.py writes for make_synthetic_weights(5, relu_targets=["relu3_1"]): the digest
  of the file it read, and per nn.SpatialConvolution its name and a digest of its weight and bias
  (tests/test_host_logic.py::test_t7_reader_against_reference_torchfile).
* wct_np_*     a digest of the reference's ops.wct_np on the inputs of wct_np_c128_a08_dead.npz, in float32
  (tests/test_oracle.py::test_reference_wct_np_reproduces_fixture).
* pipeline_*   the reference's WCTModel graph (model.py / ops.py / vgg_normalised.py over tests/golden/np_tf1.py)
  re-run in float64 on the inputs of pipeline_wct_31_11_odd_a08.npz
  (tests/test_oracle.py::test_reference_code_reproduces_pipeline_fixture).
"""
import hashlib
import importlib.util
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

T7_SEED, T7_TARGETS = 5, ["relu3_1"]
WCT_NP_FIXTURE = "wct_np_c128_a08_dead.npz"
PIPELINE_FIXTURE = "pipeline_wct_31_11_odd_a08.npz"


def array_digest(*arrays):
    """sha256 over shape and float64 value of each array: equal digests <=> np.array_equal on every array."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.asarray(a)
        h.update(repr(a.shape).encode())
        h.update(np.ascontiguousarray(a, dtype=np.float64).tobytes())
    return h.hexdigest()


def file_digest(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def main():
    from oracle import ref_ops
    from tests.golden import np_tf1
    from tests.t7_writer import write_vgg_t7
    from tests.test_oracle import load_pipeline_fixture
    from wct_tf_b200.weights import make_synthetic_weights
    arrays = {}

    tmp = tempfile.mkdtemp()
    t7 = os.path.join(tmp, "vgg_normalised.t7")
    write_vgg_t7(t7, make_synthetic_weights(T7_SEED, relu_targets=T7_TARGETS)["vgg"])
    spec = importlib.util.spec_from_file_location("_ref_torchfile", os.path.join(np_tf1.REF_DIR, "torchfile.py"))
    torchfile = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(torchfile)
    net = torchfile.load(t7, force_8bytes_long=True)
    convs = [m for m in net.modules if m._typename == b"nn.SpatialConvolution"]
    arrays["torchfile_t7_sha256"] = np.array(file_digest(t7))
    arrays["torchfile_conv_digests"] = np.array([array_digest(m.weight, m.bias) for m in convs])
    arrays["torchfile_conv_names"] = np.array([m.name.decode() for m in net.modules[1:]
                                               if m._typename == b"nn.SpatialConvolution"])
    os.remove(t7)

    ref = ref_ops.load_reference_ops(np_tf1.REF_DIR)
    g = np.load(os.path.join(HERE, WCT_NP_FIXTURE))
    out = ref.wct_np(g["content"], g["style"], float(g["alpha"]))
    arrays["wct_np_fixture"] = np.array(WCT_NP_FIXTURE)
    arrays["wct_np_out_sha256"] = np.array(array_digest(out))
    assert out.dtype == np.float32 and np.array_equal(out, g["out_ref_fp32"])

    g, targets, w = load_pipeline_fixture(os.path.join(HERE, PIPELINE_FIXTURE))
    t7 = os.path.join(tmp, "vgg.t7")
    write_vgg_t7(t7, w["vgg"])
    dec = {l["name"]: (l["kernel"], l["bias"]) for t in targets for l in w["decoders"][t]}
    with np_tf1.reference_modules() as r:
        out, _ = np_tf1.run_reference(r, g["content"][None] / 255.0, g["style"][None] / 255.0, t7, dec, targets,
                                      float(g["alpha"]), bool(g["adain"]), np.float64, swap5=bool(g["swap5"]),
                                      ss_alpha=float(g["ss_alpha"]))
    os.remove(t7)
    os.rmdir(tmp)
    arrays["pipeline_fixture"] = np.array(PIPELINE_FIXTURE)
    arrays["pipeline_out_fp64"] = np.asarray(out, dtype=np.float64)
    print("pipeline rerun vs fixture %.2e" % np.abs(out - g["out_ref_fp64"]).max())

    np.savez_compressed(os.path.join(HERE, "reference_reads.npz"), **arrays)
    print("torchfile: %d convs; wct_np digest %s" % (len(convs), arrays["wct_np_out_sha256"]))


if __name__ == "__main__":
    main()
