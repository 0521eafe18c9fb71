"""BSON checkpoint reader + Q-net layout conversion (host logic; CPU)."""
import json
import os
import struct

import numpy as np
import pytest
import torch

from oracle import qnet_oracle as QO
from tests.util import pkg

G = os.path.join(os.path.dirname(__file__), "golden")


# ---- a tiny BSON.jl-style writer (test scaffolding) -------------------------------------------------------
def _el(t, k, payload):
    return bytes([t]) + k.encode() + b"\0" + payload


def _doc(items):
    body = b"".join(items) + b"\0"
    return struct.pack("<i", len(body) + 4) + body


def _enc(v, k):
    if isinstance(v, dict):
        return _el(3, k, _doc([_enc(x, kk) for kk, x in v.items()]))
    if isinstance(v, list):
        return _el(4, k, _doc([_enc(x, str(i)) for i, x in enumerate(v)]))
    if isinstance(v, bytes):
        return _el(5, k, struct.pack("<i", len(v)) + b"\0" + v)
    if isinstance(v, bool):
        return _el(8, k, bytes([int(v)]))
    if isinstance(v, int):
        return _el(0x12, k, struct.pack("<q", v))
    if isinstance(v, float):
        return _el(1, k, struct.pack("<d", v))
    if isinstance(v, str):
        b = v.encode() + b"\0"
        return _el(2, k, struct.pack("<i", len(b)) + b)
    raise TypeError(type(v))


def _dtype(name):
    return {"tag": "datatype", "params": [], "name": name}


def _arr(a):
    return {"tag": "array", "type": _dtype(["Core", "Float32"]), "size": [int(d) for d in a.shape],
            "data": np.asfortranarray(a).astype("<f4").tobytes(order="F")}


def _tup(*xs):
    return {"tag": "tuple", "data": list(xs)}


def _chain(layers):
    out = []
    for kind, p in layers:
        if kind == "conv":
            out.append({"tag": "struct", "type": _dtype(["Main", "Flux", "Conv"]),
                        "data": [{"tag": "struct", "type": _dtype(["Main", "NNlib", "#relu"]), "data": []},
                                 _arr(p["W"]), _arr(p["b"]), _tup(1, 1), _tup(*p["pad"]), _tup(1, 1), 1]})
        elif kind == "flatten":
            out.append({"tag": "struct", "type": _dtype(["Main", "Flux", "#flatten"]), "data": []})
        else:
            out.append({"tag": "struct", "type": _dtype(["Main", "Flux", "Dense"]),
                        "data": [_arr(p["W"]), _arr(p["b"]),
                                 {"tag": "struct", "type": _dtype(["Main", "NNlib", "#relu"]), "data": []}]})
    return {"tag": "struct", "type": {"tag": "backref", "ref": 1}, "data": [_tup(*out)]}


def _trainer_bson(q_layers, t_layers):
    model = {"tag": "struct", "type": _dtype(["Main", "DQNModel"]), "data": [_chain(q_layers), _chain(t_layers), 0]}
    tr = {"tag": "struct", "type": _dtype(["Main", "Trainer"]), "data": [0, model, 0]}
    top = {"tr": tr, "_backrefs": [_dtype(["Main", "Flux", "Chain"])]}
    return _doc([_enc(v, k) for k, v in top.items()])


def test_bson_round_trip_and_destructure_order():
    S = pkg()
    from snake_b200 import bson_io, qnet
    q = qnet.glorot_layers(seed=1)
    t = qnet.glorot_layers(seed=2)
    raw = _trainer_bson(q, t)
    ql, tl = bson_io.load_trainer_nets(raw)
    assert [k for k, _ in ql] == ["conv", "conv", "conv", "flatten", "dense", "dense"]
    for (ka, pa), (kb, pb) in zip(q, ql):
        if ka in ("conv", "dense"):
            assert np.array_equal(pa["W"], pb["W"]) and np.array_equal(pa["b"], pb["b"])
    assert not np.array_equal(ql[0][1]["W"], tl[0][1]["W"])
    theta = bson_io.destructure(ql)
    assert theta.size == 181395                                   # SURVEY §8a: 304+4640+73792+102464+195
    assert np.array_equal(theta[:288], q[0][1]["W"].reshape(-1, order="F"))
    assert np.array_equal(theta[288:304], q[0][1]["b"])
    assert np.array_equal(theta[-3:], q[-1][1]["b"])


def test_truncated_or_damaged_files_raise_value_error():
    pkg()
    from snake_b200 import bson_io
    good = _trainer_bson(*[[("dense", {"W": np.ones((3, 4), np.float32), "b": np.zeros(3, np.float32)})]] * 2)
    bson_io.BsonFile(good)
    for cut in (0, 3, 17, len(good) // 2, len(good) - 1):
        with pytest.raises(ValueError):
            bson_io.BsonFile(good[:cut])
    with pytest.raises(ValueError):
        bson_io.BsonFile(struct.pack("<i", 2 ** 30) + good[4:])          # declared length beyond the buffer


def test_reads_a_deviation_matrix_file(tmp_path):
    """./D_matrices/<name>.bson as compute_D.jl:84 writes it and plot_traj.jl:7 loads it (none is committed in the reference,
    so the file is produced by the BSON.jl-style writer above): Float64 (P, K), Julia column-major."""
    pkg()
    from snake_b200 import bson_io
    rng = np.random.default_rng(5)
    D = rng.normal(size=(37, 6))
    arr = {"tag": "array", "type": _dtype(["Core", "Float64"]), "size": [37, 6], "data": np.asfortranarray(D).astype("<f8").tobytes(order="F")}
    path = tmp_path / "D_test.bson"
    path.write_bytes(_doc([_enc(arr, "deviation_matrix")]))
    got = bson_io.load_deviation_matrix(str(path))
    assert got.dtype == np.float64 and got.shape == (37, 6) and np.array_equal(got, D)
    bad = tmp_path / "other.bson"
    bad.write_bytes(_doc([_enc(arr, "buffer")]))
    with pytest.raises(ValueError):
        bson_io.load_deviation_matrix(str(bad))


def test_reads_a_one_frame_trainer_checkpoint():
    """The reference's trainer checkpoints hold the older one-frame network; golden/g6_bson_qnet.json records the layer
    layout of trainers/very_long_training1.bson (the checkpoint itself is not part of this project).  A trainer file of
    that layout with seeded weights reads back layer by layer and destructures to the same parameter count."""
    pkg()
    from snake_b200 import bson_io
    gold = json.load(open(os.path.join(G, "g6_bson_qnet.json")))
    rng = np.random.default_rng(11)
    q = []
    for layer in gold["layers"]:
        p = {}
        if layer["kind"] != "flatten":
            p = {"W": rng.normal(size=layer["shape"]).astype(np.float32), "b": rng.normal(size=layer["bias"]).astype(np.float32)}
        if layer["kind"] == "conv":
            p["pad"] = layer["pad"]
        q.append((layer["kind"], p))
    t = [(k, {n: 2 * v if n in ("W", "b") else v for n, v in p.items()}) for k, p in q]
    ql, tl = bson_io.load_trainer_nets(_trainer_bson(q, t))
    assert [k for k, _ in ql] == [layer["kind"] for layer in gold["layers"]]
    for (k, p), (_, want) in zip(ql, q):
        if k != "flatten":
            assert np.array_equal(p["W"], want["W"]) and np.array_equal(p["b"], want["b"])
        if k == "conv":
            assert p["pad"] == want["pad"]
    theta = bson_io.destructure(ql)
    assert theta.size == gold["n_params"] == 181251               # older one-frame net: conv1 is 3x3x1x16
    assert np.array_equal(theta, np.concatenate([x for k, p in q if k != "flatten" for x in (p["W"].reshape(-1, order="F"), p["b"])]))
    assert np.array_equal(bson_io.destructure(tl), 2 * theta)
    shapes = [list(p["W"].shape) for k, p in ql if k in ("conv", "dense")]
    assert shapes == [[3, 3, 1, 16], [3, 3, 16, 32], [6, 6, 32, 64], [64, 1600], [3, 64]]


def test_flux_to_torch_layout_matches_the_true_convolution_oracle():
    """torch (cuDNN-style cross-correlation, NCHW over Julia's bytes) with converted weights == the Flux/NNlib
    semantics restated in numpy Float64 (true convolution over WHCN, column-major flatten)."""
    pkg()
    from snake_b200 import qnet
    layers = qnet.glorot_layers(seed=3)
    for _, p in layers:
        if "b" in p:
            p["b"] = np.random.default_rng(len(p["b"])).normal(0, 0.1, p["b"].shape).astype(np.float32)
    rng = np.random.default_rng(0)
    N = 7
    state_julia = rng.integers(-1, 3, (10, 10, 2, N)).astype(np.float64)        # (10,10,2,N) WHCN
    want = QO.forward(layers, state_julia)                                       # (3, N)
    obs_torch = torch.from_numpy(np.ascontiguousarray(state_julia.transpose(3, 2, 1, 0)))   # same bytes as col-major
    from tools.torch_qnet import TorchQNet
    net = TorchQNet(layers, "cpu", dtype=torch.float64)
    got = net(obs_torch).numpy().T
    assert np.allclose(got, want, rtol=1e-5, atol=1e-6)
