#!/usr/bin/env python
"""Write the caffemodel fixtures of tests/test_caffemodel.py with the reference's own generated protobuf schema.

    python tests/golden/make_caffemodel_golden.py <reference checkout>/caffe_3d/python/caffe/proto

Writes, next to this script:
  caffemodel_reference_schema.bin             a NetParameter written by the reference's caffe_pb2: new-style blob
                                              shape, a BN layer with legacy 4-D dims (1, 1, 1, 64), an unknown layer
  caffemodel_reference_schema_bad_legacy.bin  the same with legacy dims (1, 64, 1, 1), which do not match a [64] blob
  caffe_pb2_fields.json                       the fields of NetParameter, LayerParameter, BlobProto and BlobShape
                                              (number, type, label, packed) that are scalars or one of these four
                                              messages: enough for the protobuf runtime to read a caffemodel's layer
                                              names, types and blobs the way the reference's schema does
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MESSAGES = ("NetParameter", "LayerParameter", "BlobProto", "BlobShape")


def write(pb2, legacy_dims):
    net = pb2.NetParameter()
    net.name = "from_reference_schema"
    lay = net.layer.add()
    lay.name, lay.type = "conv1_7x7_s2", "Convolution"
    b = lay.blobs.add()
    b.shape.dim.extend([64, 3, 7, 7])
    b.data.extend(np.arange(64 * 3 * 7 * 7, dtype=np.float32) * 1e-4)
    b = lay.blobs.add()
    b.shape.dim.extend([64])
    b.data.extend(np.ones(64, np.float32) * 0.5)
    lay = net.layer.add()
    lay.name, lay.type = "conv1_7x7_s2_bn", "BN"
    for v in (1.0, 2.0, 3.0, 4.0):
        b = lay.blobs.add()
        b.num, b.channels, b.height, b.width = legacy_dims
        b.data.extend(np.full(64, v, np.float32))
    lay = net.layer.add()
    lay.name, lay.type = "not_in_target_net", "Convolution"
    b = lay.blobs.add()
    b.shape.dim.extend([2])
    b.data.extend([1.0, 2.0])
    return net.SerializeToString()


def fields(pb2):
    out = {}
    for name in MESSAGES:
        out[name] = []
        for f in getattr(pb2, name).DESCRIPTOR.fields:
            if f.enum_type is not None or (f.message_type is not None and f.message_type.name not in MESSAGES):
                continue
            e = {"name": f.name, "number": f.number, "type": f.type, "label": f.label}
            if f.message_type is not None:
                e["message"] = f.message_type.name
            if f.GetOptions().packed:
                e["packed"] = True
            out[name].append(e)
    return out


def main():
    os.environ["PROTOCOL_BUFFERS_PYTHON_IMPLEMENTATION"] = "python"
    sys.path.insert(0, sys.argv[1])
    import caffe_pb2
    with open(os.path.join(HERE, "caffemodel_reference_schema.bin"), "wb") as f:
        f.write(write(caffe_pb2, (1, 1, 1, 64)))   # legacy blobs index from the END (blob.cpp:416-428)
    with open(os.path.join(HERE, "caffemodel_reference_schema_bad_legacy.bin"), "wb") as f:
        f.write(write(caffe_pb2, (1, 64, 1, 1)))
    with open(os.path.join(HERE, "caffe_pb2_fields.json"), "w") as f:
        json.dump(fields(caffe_pb2), f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
