#!/usr/bin/env python
"""Describe every net definition the reference ships (models_ECO_*/**/*.prototxt, solvers excepted) as a call of
tools/gen_eco_prototxt.py, or of a backbone builder in tests/eco_testlib.py for the two pretrained backbones, and write
the descriptions to reference_nets.json.

    python tests/golden/make_reference_nets.py <root of the reference checkout>

The generator's arguments are read off the reference file (classifier name and width, dropout ratios, net name, input
batch).  A train/test net's header and VideoData layers are stored as text (tokens re-joined with single spaces), since
the generator replaces them by net inputs.  Each entry carries the SHA-256 of the reference file's parsed tree, and the
script stops unless the rebuilt text parses to exactly that tree.  tests/test_prototxt_gen.py and
tests/test_product_parser.py check against the JSON.
"""
import glob
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools"), os.path.dirname(HERE)]

from oracle import prototxt  # noqa: E402
from eco_testlib import reference_net_text, tree_sha256  # noqa: E402

OUT = os.path.join(HERE, "reference_nets.json")
BACKBONES = {"bn_inception_rgb_deploy.prototxt": "bn_inception_deploy",
             "112_c3d_resnet_18_train_val.prototxt": "c3d_resnet18_train"}


def generator_call(tree, train):
    layers = tree["layer"]
    fc = [l for l in layers if l["type"] == ["InnerProduct"]][0]
    drop = [l["dropout_param"][0]["dropout_ratio"][0] for l in layers if l["type"] == ["Dropout"]]
    kw = dict(segments=16, classes=fc["inner_product_param"][0]["num_output"][0], fc_name=fc["name"][0],
              net_name=tree["name"][0])
    if not train:
        kw["batch"] = tree["input_dim"][0] // kw["segments"]
    if any(l["name"] == ["global_pool2D"] for l in layers):
        kw.update(dropout2d=drop[0], dropout3d=drop[1])   # the 2-D stream's dropout comes first in the file
        return "eco_full_" + ("train" if train else "deploy"), kw
    kw["dropout"] = drop[0]
    return "eco_lite_" + ("train" if train else "deploy"), kw


def data_layers_text(text):
    """the top-level items in front of the first layer that is not a VideoData layer, re-joined token by token"""
    out, item, depth = [], [], 0
    toks = list(prototxt._tokens(text))
    for i, (kind, tok) in enumerate(toks):
        if depth == 0 and not item and kind == "atom" and tok == "layer":
            rest = prototxt.parse(" ".join(t if k != "str" else json.dumps(t) for k, t in toks[i:]))
            if rest["layer"][0]["type"] != ["VideoData"]:
                break
        item.append(json.dumps(tok) if kind == "str" else tok)
        if kind == "punct" and tok in "{<":
            depth += 1
        elif kind == "punct" and tok in "}>":
            depth -= 1
        if depth == 0 and kind != "atom" and not (kind == "punct" and tok in ":[],"):
            out.append(" ".join(item))
            item = []
    return "\n".join(out) + "\n"


def main():
    ref = sys.argv[1]
    nets = []
    for path in sorted(glob.glob(os.path.join(ref, "models_ECO_*", "**", "*.prototxt"), recursive=True)):
        if os.path.basename(path) == "solver.prototxt":
            continue
        text = open(path).read()
        tree = prototxt.parse(text)
        train = any(l["type"] == ["VideoData"] for l in tree["layer"])
        if os.path.basename(path) in BACKBONES:
            make, kw = BACKBONES[os.path.basename(path)], {}
        else:
            make, kw = generator_call(tree, train)
        entry = {"path": os.path.relpath(path, ref), "make": make, "kwargs": kw,
                 "data_layers": data_layers_text(text) if train else "",
                 "layers": len(tree["layer"]), "sha256": tree_sha256(tree)}
        got = prototxt.parse(reference_net_text(entry))
        if tree_sha256(got) != entry["sha256"]:
            raise SystemExit("%s: the generator does not rebuild this net" % entry["path"])
        nets.append(entry)
    with open(OUT, "w") as f:
        json.dump({"nets": nets}, f, indent=1)
        f.write("\n")
    print("wrote %s: %d nets" % (OUT, len(nets)))


if __name__ == "__main__":
    main()
