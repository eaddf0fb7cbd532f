"""caffemodel I/O (csrc/caffemodel.cpp, no libprotobuf) -- round trip through the C ABI on the CPU, and
against the reference's own generated schema (caffe_3d/python/caffe/proto/caffe_pb2.py) in both directions:
what Net::ToProto / CopyTrainedLayersFrom (caffe_3d/src/caffe/net.cpp:852-904) would write and read.  The
schema's fields and two files it wrote are stored under tests/golden/."""
import json
import os

import numpy as np
import pytest

import caffe
import gen_eco_prototxt as gen
from oracle import refnet


def small_net():
    return gen.eco_lite_deploy(segments=4, classes=7, batch=1)


def test_save_and_copy_from_round_trip(tmp_path):
    txt = small_net()
    ref = refnet.RefNet(txt).init_params(11)
    a = caffe.Net.from_string(txt, caffe.TEST)
    for name, arrs in ref.params_dict().items():
        for blob, arr in zip(a.params[name], arrs):
            blob.data[...] = arr
    path = str(tmp_path / "w.caffemodel")
    a.save(path)
    b = caffe.Net.from_string(txt, caffe.TEST)
    assert not np.array_equal(b.params["res3a_2n"][0].data, a.params["res3a_2n"][0].data)
    b.copy_from(path)
    for name, blobs in a.params.items():
        for x, y in zip(blobs, b.params[name]):
            assert np.array_equal(x.data, y.data), name
    # constructor form Net(prototxt, caffemodel, phase) and the RuntimeError on missing files (_caffe.cpp:57-64)
    proto = tmp_path / "deploy.prototxt"
    proto.write_text(txt)
    c = caffe.Net(str(proto), path, caffe.TEST)
    assert np.array_equal(c.params["fc8u"][1].data, a.params["fc8u"][1].data)
    with pytest.raises(RuntimeError):
        caffe.Net(str(proto), str(tmp_path / "missing.caffemodel"), caffe.TEST)
    with pytest.raises(RuntimeError):
        caffe.Net(str(tmp_path / "missing.prototxt"), caffe.TEST)


def test_copy_from_rejects_shape_mismatch_and_ignores_unknown_layers(tmp_path):
    a = caffe.Net.from_string(gen.eco_lite_deploy(segments=4, classes=7, batch=1), caffe.TEST)
    path = str(tmp_path / "w.caffemodel")
    a.save(path)
    # a net with another class count: fc layer shape differs -> error like caffe's "shape mismatch" CHECK
    b = caffe.Net.from_string(gen.eco_lite_deploy(segments=4, classes=9, batch=1), caffe.TEST)
    with pytest.raises(RuntimeError, match="shape mismatch"):
        b.copy_from(path)
    # a net whose fc layer has a different NAME simply ignores the source layer (net.cpp:860-863)
    c = caffe.Net.from_string(gen.eco_lite_deploy(segments=4, classes=9, fc_name="fc8_other", batch=1), caffe.TEST)
    c.copy_from(path)
    assert np.array_equal(c.params["conv1_7x7_s2"][0].data, a.params["conv1_7x7_s2"][0].data)


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def reference_schema():
    """NetParameter of the reference's schema (caffe_3d/python/caffe/proto/caffe_pb2.py), built by the protobuf runtime
    from the fields stored in tests/golden/caffe_pb2_fields.json (tests/golden/make_caffemodel_golden.py)"""
    from google.protobuf import descriptor_pb2, descriptor_pool, message_factory
    with open(os.path.join(GOLDEN, "caffe_pb2_fields.json")) as f:
        spec = json.load(f)
    fdp = descriptor_pb2.FileDescriptorProto(name="caffe_fields.proto", package="caffe", syntax="proto2")
    for name, fields in spec.items():
        msg = fdp.message_type.add(name=name)
        for e in fields:
            fd = msg.field.add(name=e["name"], number=e["number"], type=e["type"], label=e["label"])
            if "message" in e:
                fd.type_name = ".caffe." + e["message"]
            if e.get("packed"):
                fd.options.packed = True
    pool = descriptor_pool.DescriptorPool()
    pool.Add(fdp)
    return message_factory.GetMessageClass(pool.FindMessageTypeByName("caffe.NetParameter"))


def test_wire_format_against_reference_schema(tmp_path):
    txt = small_net()
    ref = refnet.RefNet(txt).init_params(5)
    a = caffe.Net.from_string(txt, caffe.TEST)
    for name, arrs in ref.params_dict().items():
        for blob, arr in zip(a.params[name], arrs):
            blob.data[...] = arr
    ours = str(tmp_path / "ours.caffemodel")
    a.save(ours)
    # (1) the reference's protobuf schema parses what we wrote
    net = reference_schema()()
    with open(ours, "rb") as f:
        net.ParseFromString(f.read())
    assert len(net.layer) == 109
    lay = [l for l in net.layer if l.name == "res3a_2n"][0]
    assert lay.type == "Convolution" and len(lay.blobs) == 2
    assert list(lay.blobs[0].shape.dim) == [128, 96, 3, 3, 3]
    w = ref.params_dict()["res3a_2n"][0]
    assert abs(float(np.array(lay.blobs[0].data, np.float32).sum()) - float(w.sum())) < 1e-2
    # (2) we parse what the reference's schema writes (new-style shape, legacy 4-D dims, unknown layer)
    b = caffe.Net.from_string(txt, caffe.TEST)
    b.copy_from(os.path.join(GOLDEN, "caffemodel_reference_schema.bin"))
    assert np.allclose(b.params["conv1_7x7_s2"][0].data.ravel(), np.arange(64 * 3 * 7 * 7, dtype=np.float32) * 1e-4)
    assert np.all(b.params["conv1_7x7_s2"][1].data == 0.5)
    for k, v in enumerate((1.0, 2.0, 3.0, 4.0)):
        assert np.all(b.params["conv1_7x7_s2_bn"][k].data == v)
    # legacy dims are matched from the end, exactly as Blob::ShapeEquals does: (1,64,1,1) != a [1,64] blob
    with pytest.raises(RuntimeError, match="shape mismatch"):
        caffe.Net.from_string(txt, caffe.TEST).copy_from(os.path.join(GOLDEN, "caffemodel_reference_schema_bad_legacy.bin"))
