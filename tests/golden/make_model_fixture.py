"""Writes the fixtures of the trained 2-D model the reference ships (data/models/myModel2D, Torch7 binary):

  myModel2D_layers.npz          its convolution weights, extracted with fluidnet_b200/torch7.py, plus the few
                                mconf keys the projection reads (the parity tests use real trained weights)
  myModel2D_slim, myModel2D_slim_mconf.bin
                                the model file and its `_mconf.bin` byte for byte, except that every storage
                                larger than 4 KB that holds no convolution weight or bias (buffers, gradients,
                                optimizer state) is written empty, with the tensors that view it as 0-d: the
                                reader's test parses the real nngraph file in well under 1 MB

    python tests/golden/make_model_fixture.py <reference checkout>/data/models/myModel2D
"""
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from fluidnet_b200 import torch7  # noqa: E402

KEEP_BYTES = 4096


class _Spans(torch7._Reader):
    """The reader, noting where each storage's payload and each tensor's ndim / sizes / strides lie."""

    def __init__(self, data):
        super().__init__(data)
        self.storages = {}          # idx -> (start, end)
        self.tensors = {}           # idx -> (start, end, storage idx or None)

    def _torch_object(self, idx, cls):
        start = self.o
        if cls in torch7._STORAGE_DTYPES:
            a = super()._torch_object(idx, cls)
            self.storages[idx] = (start, self.o)
            return a
        if cls.endswith("Tensor") and cls.startswith("torch."):
            end = start + 4 + 16 * struct.unpack_from("<i", self.d, start)[0]
            tag, sidx = struct.unpack_from("<ii", self.d, end + 8)      # after the storage offset
            a = super()._torch_object(idx, cls)
            self.tensors[idx] = (start, end, sidx if tag == 4 else None)
            return a
        return super()._torch_object(idx, cls)


def slim(src, dst):
    data = open(src, "rb").read()
    sys.setrecursionlimit(max(sys.getrecursionlimit(), 20000))
    r = _Spans(data)
    convs = []
    torch7._walk(r.value(), set(), convs)
    by_id = {id(v): k for k, v in r.memo.items()}
    keep = {r.tensors[by_id[id(c[f])]][2] for c in convs for f in ("weight", "bias")}
    drop = {i for i, (s, e) in r.storages.items() if e - s > KEEP_BYTES and i not in keep}
    edits = [(s, e, struct.pack("<q", 0)) for i, (s, e) in r.storages.items() if i in drop]
    edits += [(s, e, struct.pack("<i", 0)) for s, e, si in r.tensors.values() if si in drop]
    out = bytearray(data)
    for s, e, b in sorted(edits, reverse=True):
        out[s:e] = b
    with open(dst, "wb") as f:
        f.write(out)
    print(dst, len(data), "->", len(out), "bytes")


def main(src):
    ref = torch7.load_reference_model(src)
    out = {"is3D": np.array(ref["is3D"]), "n_layers": np.array(len(ref["layers"])),
           "normalizeInputThreshold": np.array(float(ref["mconf"]["normalizeInputThreshold"]))}
    for i, (w, b) in enumerate(ref["layers"]):
        out["w%d" % i] = w
        out["b%d" % i] = b
    np.savez_compressed(os.path.join(HERE, "myModel2D_layers.npz"), **out)
    print("layers:", [w.shape for w, _ in ref["layers"]])

    dst = os.path.join(HERE, "myModel2D_slim")
    slim(src, dst)
    slim(src + "_mconf.bin", dst + "_mconf.bin")


if __name__ == "__main__":
    main(sys.argv[1])
