"""Builds tests/golden/mnist.npz from the reference's own test model (rten-onnx/test-data/mnist.onnx, the export of
tools/train-mnist.py; BASELINE configs[0]), stored unchanged beside this script as tests/golden/mnist.onnx:

    python tests/golden/make_mnist_fixture.py

The ONNX file is read with a minimal protobuf wire-format walker (no `onnx` package here).  The fixture holds the
initialisers (weights), the operator list with the attributes the hot path needs, and logits computed by PyTorch (CPU,
float64) for the input the reference's own test uses (`full([1,1,28,28], 0.5)`, src/model.rs:1284-1287) -- the reference
asserts only the output SHAPE, so the values are pinned by an independent implementation instead."""
import json
import os
import struct
import sys

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mnist.onnx")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "mnist.npz")


def varint(b, i):
    v, s = 0, 0
    while True:
        c = b[i]
        i += 1
        v |= (c & 0x7F) << s
        if not c & 0x80:
            return v, i
        s += 7


def fields(b):
    i = 0
    while i < len(b):
        key, i = varint(b, i)
        f, wt = key >> 3, key & 7
        if wt == 0:
            v, i = varint(b, i)
        elif wt == 2:
            n, i = varint(b, i)
            v = b[i:i + n]
            i += n
        elif wt == 5:
            v = b[i:i + 4]
            i += 4
        elif wt == 1:
            v = b[i:i + 8]
            i += 8
        else:
            raise ValueError(wt)
        yield f, wt, v


def tensor(b):
    dims, name, raw, floats, dtype, i64 = [], "", None, [], 0, []
    for f, wt, v in fields(b):
        if f == 1:
            if wt == 2:
                j = 0
                while j < len(v):
                    d, j = varint(v, j)
                    dims.append(d)
            else:
                dims.append(v)
        elif f == 2:
            dtype = v
        elif f == 4:
            floats += list(struct.unpack(f"<{len(v) // 4}f", v)) if wt == 2 else [struct.unpack("<f", v)[0]]
        elif f == 7:
            if wt == 2:
                j = 0
                while j < len(v):
                    d, j = varint(v, j)
                    i64.append(d)
            else:
                i64.append(v)
        elif f == 8:
            name = v.decode()
        elif f == 9:
            raw = bytes(v)
    if dtype == 1:
        a = np.frombuffer(raw, "<f4") if raw is not None else np.array(floats, np.float32)
    elif dtype == 7:
        a = np.frombuffer(raw, "<i8") if raw is not None else np.array(i64, np.int64)
    else:
        raise ValueError(f"dtype {dtype}")
    return name, a.reshape(dims).copy()


def attribute(b):
    name, ints, i, f = "", [], None, None
    for fld, wt, v in fields(b):
        if fld == 5:  # AttributeProto.t: a constant tensor
            return_name = name
            return return_name or "value", tensor(v)[1].tolist()
        if fld == 1:
            name = v.decode()
        elif fld == 3:
            i = v if v < (1 << 63) else v - (1 << 64)
        elif fld == 2:
            f = struct.unpack("<f", v)[0]
        elif fld == 8:
            if wt == 2:
                j = 0
                while j < len(v):
                    d, j = varint(v, j)
                    ints.append(d)
            else:
                ints.append(v)
    return name, (ints if ints else (i if i is not None else f))


def main():
    model = open(SRC, "rb").read()
    graph = next(v for f, _, v in fields(model) if f == 7)
    weights, nodes = {}, []
    for f, _, v in fields(graph):
        if f == 5:
            n, a = tensor(v)
            weights[n] = a
        elif f == 1:
            node = {"inputs": [], "outputs": [], "op": "", "attrs": {}}
            for g, _, w in fields(v):
                if g == 1:
                    node["inputs"].append(w.decode())
                elif g == 2:
                    node["outputs"].append(w.decode())
                elif g == 4:
                    node["op"] = w.decode()
                elif g == 5:
                    k, val = attribute(w)
                    node["attrs"][k] = val
            nodes.append(node)
    print([(n["op"], n["inputs"], n["attrs"]) for n in nodes])
    print({k: v.shape for k, v in weights.items()})

    # independent logits: PyTorch CPU, float64
    import torch
    import torch.nn.functional as F
    t = {k: torch.from_numpy(v.astype(np.float64)) if v.dtype == np.float32 else v for k, v in weights.items()}
    x = torch.full((1, 1, 28, 28), 0.5, dtype=torch.float64)
    vals = {"input": x}
    graph_in = None
    for n in nodes:
        ins = [vals[i] if i in vals else t[i] for i in n["inputs"] if i]
        a = n["attrs"]
        if n["op"] == "Constant":
            vals[n["outputs"][0]] = np.asarray(a["value"])
            continue
        if n["op"] == "Conv":
            pads = a.get("pads", [0, 0, 0, 0])
            y = F.conv2d(ins[0], ins[1], ins[2] if len(ins) > 2 else None, stride=tuple(a.get("strides", [1, 1])),
                         padding=(pads[0], pads[1]), dilation=tuple(a.get("dilations", [1, 1])), groups=a.get("group", 1))
        elif n["op"] == "Relu":
            y = F.relu(ins[0])
        elif n["op"] == "MaxPool":
            y = F.max_pool2d(ins[0], tuple(a["kernel_shape"]), tuple(a.get("strides", a["kernel_shape"])))
        elif n["op"] == "ReduceMean":
            axes = a.get("axes") or [int(v) for v in np.asarray(ins[1]).reshape(-1)]
            y = ins[0].mean(dim=tuple(int(v) for v in axes), keepdim=bool(a.get("keepdims", 1)))
        elif n["op"] == "Reshape":
            y = ins[0].reshape([int(v) for v in np.asarray(ins[1]).reshape(-1)])
        elif n["op"] == "Flatten":
            y = ins[0].flatten(a.get("axis", 1))
        elif n["op"] == "Gemm":
            A_, B_ = (ins[0].T if a.get("transA") else ins[0]), (ins[1].T if a.get("transB") else ins[1])
            y = a.get("alpha", 1.0) * (A_ @ B_) + (a.get("beta", 1.0) * ins[2] if len(ins) > 2 else 0)
        else:
            raise SystemExit(f"unexpected op {n['op']}")
        vals[n["outputs"][0]] = y
        last = y
        if graph_in is None:
            graph_in = n["inputs"][0]
    if graph_in != "input":
        raise SystemExit(f"first node reads {graph_in}; rename the graph input in this script")
    logits = last.numpy()
    print("logits", logits)
    np.savez_compressed(OUT, nodes=json.dumps(nodes), logits_f64=logits, **{"w:" + k: v for k, v in weights.items()})
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
