"""fluidnet_b200/torch7.py: the Torch7 binary reader that brings a model trained with the reference into
this library (SURVEY.md section 8f-2).  A writer for the same format lives here (test-only) so the reader
is exercised without Torch7; the trained 2-D model the reference ships (tests/golden/myModel2D_slim: the file
with its large buffers emptied, tests/golden/make_model_fixture.py) must match the committed weights
(tests/golden/myModel2D_layers.npz)."""
import os
import struct

import numpy as np

from fluidnet_b200 import torch7

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "myModel2D_layers.npz")
REF_MODEL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "myModel2D_slim")


class W:
    """Minimal Torch7 binary writer (torch7/File.lua conventions)."""

    def __init__(self):
        self.b = bytearray()
        self.next = 1

    def i32(self, v): self.b += struct.pack("<i", v)
    def i64(self, v): self.b += struct.pack("<q", v)
    def s(self, v): self.i32(len(v)); self.b += v.encode()

    def number(self, v): self.i32(1); self.b += struct.pack("<d", v)
    def string(self, v): self.i32(2); self.s(v)
    def boolean(self, v): self.i32(5); self.i32(1 if v else 0)

    def table(self, items):
        self.i32(3); self.i32(self.next); self.next += 1
        self.i32(len(items))
        for k, wv in items:
            (self.number if not isinstance(k, str) else self.string)(k)
            wv()

    def backref_table(self, idx): self.i32(3); self.i32(idx)

    def tensor(self, a, cls="torch.FloatTensor", storage_cls="torch.FloatStorage"):
        a = np.ascontiguousarray(a, np.float32)
        self.i32(4); self.i32(self.next); self.next += 1
        self.s("V 1"); self.s(cls)
        self.i32(a.ndim)
        for d in a.shape: self.i64(d)
        stride = [int(np.prod(a.shape[i + 1:])) for i in range(a.ndim)]
        for d in stride: self.i64(d)
        self.i64(1)
        self.i32(4); self.i32(self.next); self.next += 1
        self.s("V 1"); self.s(storage_cls)
        self.i64(a.size); self.b += a.tobytes()

    def obj(self, cls, items):
        self.i32(4); self.i32(self.next); self.next += 1
        self.s("V 1"); self.s(cls)
        self.table(items)


def test_reader_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    w1, b1 = rng.standard_normal((4, 3, 3, 3)).astype(np.float32), rng.standard_normal(4).astype(np.float32)
    w2, b2 = rng.standard_normal((1, 4, 1, 1, 1)).astype(np.float32), rng.standard_normal(1).astype(np.float32)
    wr = W()

    def conv2d():
        wr.obj("cudnn.SpatialConvolution", [("weight", lambda: wr.tensor(w1, "torch.CudaTensor", "torch.CudaStorage")),
                                            ("bias", lambda: wr.tensor(b1)), ("nInputPlane", lambda: wr.number(3)),
                                            ("nOutputPlane", lambda: wr.number(4)), ("kH", lambda: wr.number(3)),
                                            ("kW", lambda: wr.number(3)), ("train", lambda: wr.boolean(False))])

    def conv3d():
        wr.obj("cudnn.VolumetricConvolution", [("weight", lambda: wr.tensor(w2)), ("bias", lambda: wr.tensor(b2)),
                                               ("nInputPlane", lambda: wr.number(4)), ("nOutputPlane", lambda: wr.number(1)),
                                               ("kT", lambda: wr.number(1)), ("kH", lambda: wr.number(1)),
                                               ("kW", lambda: wr.number(1))])

    wr.obj("nn.Sequential", [("modules", lambda: wr.table([(1, conv2d), (2, lambda: wr.obj("nn.ReLU", [("inf", lambda: wr.number(float("inf")))])),
                                                            (3, conv3d)])),
                             ("name", lambda: wr.string("net"))])
    path = tmp_path / "net.t7"
    path.write_bytes(bytes(wr.b))
    model = torch7.load(str(path))
    assert model.cls == "nn.Sequential" and model["name"] == "net"
    assert model["modules"][2]["inf"] == float("inf")
    layers = torch7.conv_layers(model)
    assert [w.shape for w, _ in layers] == [(4, 3, 1, 3, 3), (1, 4, 1, 1, 1)]
    assert np.array_equal(layers[0][0].reshape(w1.shape), w1) and np.array_equal(layers[0][1], b1)
    assert np.array_equal(layers[1][0], w2) and np.array_equal(layers[1][1], b2)


def test_back_references(tmp_path):
    wr = W()
    wr.table([("a", lambda: wr.table([(1, lambda: wr.number(7))])), ("b", lambda: wr.backref_table(2))])
    path = tmp_path / "t.t7"
    path.write_bytes(bytes(wr.b))
    t = torch7.load(str(path))
    assert t["a"] is t["b"] and t["a"][1] == 7


def test_shipped_2d_model_matches_fixture():
    """The reference's trained model (nngraph gModule of cudnn.SpatialConvolution layers): 'default' 2-D
    architecture of torch/lib/model.lua:179-186, and the same numbers as the committed fixture."""
    ref = torch7.load_reference_model(REF_MODEL)
    assert ref["is3D"] is False and ref["mconf"]["modelType"] == "default"
    assert [(w.shape[1], w.shape[0], w.shape[4]) for w, _ in ref["layers"]] == \
        [(3, 16, 3), (16, 16, 3), (16, 16, 3), (16, 16, 3), (16, 1, 1)]
    z = np.load(GOLD)
    assert int(z["n_layers"]) == len(ref["layers"])
    for i, (w, b) in enumerate(ref["layers"]):
        assert np.array_equal(z["w%d" % i], w) and np.array_equal(z["b%d" % i], b)
