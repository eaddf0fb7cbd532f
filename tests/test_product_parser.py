"""Every net definition the reference ships loads through the PRODUCT's own prototxt parser and graph
builder (csrc/prototxt.hpp, Net::build_graph -- no GPU needed for construction), and the caffe-visible
layer / blob names -- including the automatically inserted Split layers (insert_splits.cpp:13-142) --
agree with the oracle's independent restatement of InsertSplits.  The nets are rebuilt from
tests/golden/reference_nets.json; each rebuild must parse to the reference file's tree (SHA-256)."""
import pytest

from oracle import prototxt, refnet
from eco_testlib import reference_net_text, reference_nets, tree_sha256

NETS = reference_nets()


def test_reference_tree_has_the_expected_nets():
    names = {e["path"] for e in NETS}
    assert "models_ECO_Lite/ucf101/deploy.prototxt" in names
    assert "models_ECO_Full/kinetics/ECO_full.prototxt" in names or any("ECO_full" in n or "ECO_Full" in n for n in names)
    assert len(NETS) >= 9
    for e in NETS:
        assert tree_sha256(prototxt.parse(reference_net_text(e))) == e["sha256"], e["path"]


@pytest.mark.parametrize("entry", NETS, ids=[e["path"] for e in NETS])
@pytest.mark.parametrize("phase", ["TEST", "TRAIN"])
def test_product_parser_loads_reference_net(entry, phase, tmp_path):
    import caffe
    is_deploy = not entry["data_layers"]   # declares its inputs instead of reading them through VideoData layers
    if is_deploy and phase == "TRAIN":
        pytest.skip("deploy nets are TEST-phase definitions")
    text = reference_net_text(entry)
    assert tree_sha256(prototxt.parse(text)) == entry["sha256"]
    path = tmp_path / "net.prototxt"
    path.write_text(text)
    net = caffe.Net(str(path), caffe.TEST if phase == "TEST" else caffe.TRAIN)
    ref = refnet.RefNet(text, phase=phase)
    want_layers, want_blobs = ref.split_names()
    got_layers = list(net._layer_names)
    got_blobs = list(net._blob_names)
    assert got_layers == want_layers
    assert got_blobs == want_blobs
    # shapes of a few landmarks (SURVEY Appendix A): the r2Dto3D volume and the logits
    blobs = net.blobs
    if "res3a_2" in blobs:
        shp = tuple(blobs["res3a_2"].shape)
        assert len(shp) == 5 and shp[1] == 128 and shp[3:] == (28, 28)
    outs = list(net.outputs)
    assert outs, "net has no outputs"
    if is_deploy:
        assert len(outs) == 1 and len(blobs[outs[0]].shape) == 2
    else:
        # train/test definitions end in the loss (+ accuracy in TEST phase), scalars in caffe
        for o in outs:
            assert tuple(blobs[o].shape) == ()
