"""tools/gen_eco_prototxt.py must emit nets structurally identical to the reference's
hand-written prototxts (pinned by the SHA-256 of each file's parsed tree in
tests/golden/reference_nets.json), and the oracle's InsertSplits naming must follow
caffe_3d/src/caffe/util/insert_splits.cpp."""
import pytest

from oracle import prototxt, refnet
import gen_eco_prototxt as gen
from eco_testlib import norm_tree as norm, reference_net_text, reference_nets, tree_sha256

REF_NETS = {e["path"]: e for e in reference_nets()}


CASES = [
    ("models_ECO_Lite/ucf101/deploy.prototxt", lambda: gen.eco_lite_deploy(16, 101, "fc8u", 5, 0.6, "o3d")),
    ("models_ECO_Lite/hmdb51/deploy.prototxt", lambda: gen.eco_lite_deploy(16, 51, "fc8h", 5, 0.6, "o3d")),
    ("models_ECO_Lite/kinetics/deploy.prototxt", lambda: gen.eco_lite_deploy(16, 400, "fc8", 5, 0.3, "ECOLite")),
    ("models_ECO_Full/kinetics/deploy.prototxt", lambda: gen.eco_full_deploy(16, 400, "fc8N", 5, 0.5, 0.6)),
    ("models_ECO_Full/ucf101/deploy.prototxt", lambda: gen.eco_full_deploy(16, 101, "fc8N", 5, 0.5, 0.6)),
]


@pytest.mark.parametrize("path,make", CASES, ids=[c[0] for c in CASES])
def test_generated_equals_reference(path, make):
    ref = REF_NETS[path]
    mine = prototxt.parse(make())
    mine["name"] = [ref["kwargs"]["net_name"]]  # net name differs per dataset; not part of the graph
    assert len(mine["layer"]) == ref["layers"]
    assert tree_sha256(mine) == ref["sha256"]


def test_split_names_lite():
    net = refnet.RefNet(gen.eco_lite_deploy(16, 101))
    layers, blobs = net.split_names()
    # SURVEY F8: multi-consumer blobs get `<blob>_<producer layer>_<top idx>_split`
    for n in ("pool2_3x3_s2_pool2_3x3_s2_0_split", "inception_3a_output_inception_3a_output_0_split",
              "res3a_res3a_2n_0_split", "res3b_bn_res3b_relu_0_split", "res4a_res4a_0_split",
              "res4b_bn_res4b_relu_0_split", "res5a_res5a_0_split"):
        assert n in layers
    assert len(layers) == 109 + 7
    assert "res3a_res3a_2n_0_split_1" in blobs and "res2b_bn_pre" in blobs and "fc8" in blobs
    assert layers.index("res3a_res3a_2n_0_split") == layers.index("res3a_2n") + 1


def test_shapes_lite_n16():
    net = refnet.RefNet(gen.eco_lite_deploy(16, 101, batch=2))
    net.param_shapes()
    s = net.shapes
    assert s["conv1_7x7_s2"] == [32, 64, 112, 112] and s["pool1_3x3_s2"] == [32, 64, 56, 56]
    assert s["inception_3a_output"] == [32, 256, 28, 28] and s["inception_3b_output"] == [32, 320, 28, 28]
    assert s["res2b_bn_pre"] == [2, 16, 96, 28, 28] and s["res2b_bn"] == [2, 96, 16, 28, 28]
    assert s["res4a_1"] == [2, 256, 8, 14, 14] and s["res5b_bn"] == [2, 512, 4, 7, 7]
    assert s["global_pool"] == [2, 512, 1, 1, 1] and s["fc8"] == [2, 101]


TRAIN_CASES = [
    ("models_ECO_Lite/kinetics/ECO_Lite.prototxt", lambda: gen.eco_lite_train(16, 400, "fc8", 17, 0.3)),
    ("models_ECO_Full/kinetics/ECO_full.prototxt", lambda: gen.eco_full_train(16, 400, "fc8N", 8, 0.5, 0.5)),
]


@pytest.mark.parametrize("path,make", TRAIN_CASES, ids=[c[0] for c in TRAIN_CASES])
def test_generated_train_net_equals_reference_after_the_data_layers(path, make):
    """the train/test definition: everything behind the VideoData layers (which the generator replaces by the two net
    inputs they produce) must be the reference's graph: names, types, bottoms/tops, phase rules, every numeric parameter"""
    entry = REF_NETS[path]
    text = make()
    ref_tree = prototxt.parse(reference_net_text(entry, text))
    assert tree_sha256(ref_tree) == entry["sha256"], "the generator no longer rebuilds " + path
    ref = norm(ref_tree)
    mine = norm(prototxt.parse(text))
    ref_layers = [l for l in ref["layer"] if l["type"] != ["VideoData"]]
    assert len(ref_layers) == len(mine["layer"])
    for a, b in zip(ref_layers, mine["layer"]):
        assert a["name"] == b["name"] and a["type"] == b["type"], (a["name"], b["name"])
        assert a.get("bottom") == b.get("bottom") and a.get("top") == b.get("top"), a["name"]
        assert a.get("include") == b.get("include"), a["name"]
        for key in ("convolution_param", "pooling_param", "inner_product_param", "reshape_param", "permute_param",
                    "dropout_param", "accuracy_param", "eltwise_param", "concat_param"):
            if key in a or key in b:
                ra, rb = dict(a.get(key, [{}])[0]), dict(b.get(key, [{}])[0])
                for filler in ("weight_filler", "bias_filler"):
                    ra.pop(filler, None), rb.pop(filler, None)
                assert ra == rb, (a["name"], key, ra, rb)
        if a["type"] == ["BN"]:
            fa = a.get("bn_param", [{}])[0].get("frozen", [False])
            fb = b.get("bn_param", [{}])[0].get("frozen", [False])
            assert fa == fb, a["name"]
        assert a.get("param") == b.get("param"), (a["name"], a.get("param"), b.get("param"))
    vd = [l for l in ref["layer"] if l["type"] == ["VideoData"]][0]
    assert vd["top"] == ["data", "label"]
