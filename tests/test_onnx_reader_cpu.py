"""CPU-only checks of the ONNX reader (csrc/onnx_reader.cu through rten_b200_onnx_summary; no GPU, no context): the
assertions of the reference's own decoder test (rten-onnx/src/onnx.rs:798-849) on the MNIST test model -- re-encoded from
tests/golden/mnist.npz by tests/onnx_writer.py, and on the reference's file itself (rten-onnx/test-data/mnist.onnx, stored
as tests/golden/mnist.onnx) -- plus the encodings a file may use for the same tensor."""
import os

import numpy as np
import pytest

import onnx_writer as W

HERE = os.path.dirname(os.path.abspath(__file__))
REF_MNIST = os.path.join(HERE, "golden", "mnist.onnx")  # rten-onnx/test-data/mnist.onnx, unchanged


@pytest.fixture(scope="module")
def summary():
    from rten_b200 import _build
    _build.build()
    from rten_b200.model import onnx_summary
    return onnx_summary


def _assert_mnist_structure(s):
    # = test_decode_mnist (rten-onnx/src/onnx.rs:812-849)
    assert s["opset"][""] == 18
    assert len(s["nodes"]) == 13 and len(s["initializers"]) == 8
    ops = [n["op"] for n in s["nodes"] if n["op"] != "Constant"]
    assert ops == ["Conv", "Relu", "MaxPool", "Conv", "Relu", "MaxPool", "Conv", "Relu", "ReduceMean", "Reshape", "Gemm"]
    assert len(s["inputs"]) == 1 and s["inputs"][0]["name"] == "input"
    assert len(s["outputs"]) == 1 and s["outputs"][0]["name"] == "logits"
    shapes = {i["name"]: i["dims"] for i in s["initializers"]}
    assert shapes["conv1.weight"] == [32, 1, 3, 3] and shapes["conv2.weight"] == [72, 32, 3, 3] and shapes["fc.weight"] == [10, 64]
    assert all(i["data_type"] == 1 and i["bytes"] == 4 * int(np.prod(i["dims"])) for i in s["initializers"])


def test_decode_empty_model(summary):
    # = test_decode_empty_model (rten-onnx/src/onnx.rs:798-804): succeeds, default model without a graph
    s = summary(b"")
    assert s["has_graph"] is False and s["nodes"] == []


def test_decode_mnist_reencoded(summary):
    s = summary(W.mnist_from_fixture(os.path.join(HERE, "golden", "mnist.npz")))
    _assert_mnist_structure(s)
    assert s["inputs"][0]["dims"] == [-1, 1, 28, 28]  # symbolic batch dimension -> -1


def test_decode_reference_mnist_file(summary):
    s = summary(open(REF_MNIST, "rb").read())
    _assert_mnist_structure(s)
    assert s["ir_version"] == 10 and s["inputs"][0]["dims"] == [1, 1, 28, 28]


def test_tensor_encodings_and_attributes(summary):
    """raw_data, packed float_data / int64_data / int32_data and every attribute kind decode to the same structure."""
    w = np.arange(12, dtype=np.float32).reshape(3, 4)
    idx = np.array([[2, 0], [1, 1]], np.int64)
    q = np.array([-3, 7, 127, -128], np.int8)
    for raw in (True, False):
        data = W.model([W.node("Gather", ["w", "idx"], ["y"], axis=0), W.node("Gelu", ["y"], ["z"], approximate="tanh"),
                        W.node("LayerNormalization", ["z", "g"], ["out"], axis=-1, epsilon=1e-12),
                        W.node("Transpose", ["out"], ["t"], perm=[1, 0, 2]), W.node("Foo", ["t", "", "q"], ["u"], domain="custom", alphas=[0.5, 1.5])],
                       [W.tensor("w", w, raw), W.tensor("idx", idx, raw), W.tensor("q", q, raw), W.tensor("g", np.ones(4, np.float32), raw)],
                       [], [W.value_info("u", W.FLOAT, [2, 2, 4])], opset=20, extra_opsets=[("custom", 3)])
        s = summary(data)
        assert s["opset"] == {"": 20, "custom": 3}
        assert [n["op"] for n in s["nodes"]] == ["Gather", "Gelu", "LayerNormalization", "Transpose", "Foo"]
        assert s["nodes"][4]["inputs"] == ["t", "", "q"] and s["nodes"][4]["attrs"] == ["alphas"]
        assert s["nodes"][2]["attrs"] == ["axis", "epsilon"]
        by = {i["name"]: i for i in s["initializers"]}
        assert by["w"]["dims"] == [3, 4] and by["w"]["bytes"] == 48 and by["idx"]["data_type"] == 7 and by["idx"]["bytes"] == 32
        assert by["q"]["data_type"] == 3 and by["q"]["bytes"] == 4


def test_malformed_input_is_an_error_not_a_crash(summary):
    import rten_b200 as rt
    good = W.mnist_from_fixture(os.path.join(HERE, "golden", "mnist.npz"))
    for bad in (good[:1000], b"\xff\xff\xff\xff\xff\xff\xff\xff\xff\xff\xff\x01", good[:50] + b"\x7f" * 40):
        try:
            summary(bad)
        except rt.OpError as e:
            assert e.kind == "InvalidValue"
