"""Shared helpers for the GPU parity tests: build a net from prototxt text through the product's
Python shim (-> C ABI -> CUDA), load the oracle's harness weights into it, and compare blobs.

Tolerance (written here once, used by every parity test): the device path stores bf16 and
accumulates in fp32; against the oracle run in its bf16-mirror mode (same rounding points,
DESIGN.md "Rounding contract") a blob must satisfy
    max|a-b| <= 1e-3 * max|b|   for single fused ops fed identical inputs, and
    ||a-b||_2 <= TOL_NET * ||b||_2 for whole networks (rounding-boundary flips accumulate).
"""
import hashlib
import json
import os

import numpy as np

TOL_OP = 1e-3     # fp32 blobs (fc, pooled vectors): max|a-b| <= TOL_OP * max|b|
FLIP_FRAC = 0.03  # bf16 blobs: at most this fraction of elements may sit on the neighbouring bf16 value
ATOL_REL = 1e-4   # bf16 blobs: fp32 accumulation-order noise near zero, relative to max|b|
TOL_NET = 4e-2    # free-running whole net, per-blob rel-L2.  Calibrated on the oracle itself: its bf16-mirror
                  # forward with a different fp32 summation order (naive conv vs im2col+SGEMM) already differs
                  # from itself by rel-L2 4e-4 (inception_3a) .. 1.6e-2 (res5b_bn), 4.4e-3 on fc8, because
                  # rounding-boundary flips of the bf16-stored maps are amplified through 32 conv layers
                  # (DESIGN.md section 4).  The tight statement is the teacher-forced per-layer check.
TOL_NET_FULL = 1e-1  # ECO-Full is 69 convs deep on the 2-D stream: oracle self-noise reaches 4.2e-2 at inception_5b_output
TOL_LOGITS = 2e-2 # free-running whole net, logits max|a-b| / max|b| (oracle self-noise: 4.2e-3)


def make_net(text, keep_all=True, a_mode=None, graph=False, persistent=True, dual_m=1, halo=0, stem_rows=None, **extra):
    import caffe
    opts = {"keep_all_blobs": 1 if keep_all else 0, "use_graph": 1 if graph else 0, "halo": halo,
            "persistent": 2 if persistent else 0, "dual_m": dual_m}
    if stem_rows is not None:
        opts["stem_rows"] = stem_rows
    opts.update(extra)
    if a_mode is not None:
        opts["a_mode"] = a_mode
    return caffe.Net.from_string(text, caffe.TEST, **opts)


def load_params(net, params):
    """params: {layer: [arrays]} from oracle.refnet.RefNet.params_dict()."""
    P = net.params
    for name, arrs in params.items():
        assert name in P, name
        assert len(P[name]) == len(arrs), (name, len(P[name]), len(arrs))
        for blob, a in zip(P[name], arrs):
            assert tuple(blob.shape) == tuple(a.shape), (name, blob.shape, a.shape)
            blob.data[...] = a


def rel_max(a, b):
    return float(np.abs(a.astype(np.float64) - b).max() / max(np.abs(b).max(), 1e-30))


def rel_l2(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-30))


def bf16_ulp(v):
    """spacing of bfloat16 (8 significant bits) at |v|"""
    a = np.maximum(np.abs(v.astype(np.float64)), 2.0 ** -120)
    return 2.0 ** (np.floor(np.log2(a)) - 7)


def check_bf16_blob(got, want, name=""):
    """Parity criterion for a blob the device stores as bf16: equal to the oracle's value rounded to
    bf16, except that an element may land on the adjacent bf16 value when the two fp32 sums (different
    summation order) straddle a rounding boundary.  Elementwise |d| <= 1 ulp + noise, few flips."""
    from oracle import refnet
    wr = refnet.round_bf16(want).astype(np.float64)
    d = np.abs(got.astype(np.float64) - wr)
    atol = ATOL_REL * max(np.abs(wr).max(), 1e-30)
    lim = 1.001 * bf16_ulp(wr) + atol
    ok = d <= lim
    flips = float((d > atol).mean())
    if not ok.all():
        excess = np.where(ok, 0.0, d / lim)
        idx = np.unravel_index(np.argmax(excess), excess.shape)
        raise AssertionError("%s: %d elements differ by more than one bf16 ulp; worst violation @%s got=%.9g want_bf16=%.9g "
                             "want_f32=%.9g ulp=%.3g atol=%.3g; %s" % (name, (~ok).sum(), idx, got[idx], wr[idx], want[idx],
                                                                      bf16_ulp(wr)[idx], atol, describe_mismatch(got, want, name)))
    assert flips <= FLIP_FRAC, "%s: %.4f of the elements differ from the oracle (limit %.2f)" % (name, flips, FLIP_FRAC)
    return flips


def teacher_blobs(ref, dev):
    """Device blobs the oracle may consume in a teacher-forced forward: everything except raw conv /
    eltwise sums, which the device's fused BN reads from the fp32 accumulator, not from the bf16 copy."""
    raw = set()
    for l in ref.layers:
        if l.type in ("Convolution", "Eltwise"):
            raw.update(l.tops)
    return {k: v for k, v in dev.items() if k not in raw}


def teacher_raw_blobs(ref, dev):
    """The raw sums as stored by the device: what its fused residual adds read back (older Eltwise operand)."""
    raw = set()
    for l in ref.layers:
        if l.type in ("Convolution", "Eltwise"):
            raw.update(l.tops)
    return {k: v for k, v in dev.items() if k in raw}


def check_f32_blob(got, want, name=""):
    assert rel_max(got, want) <= TOL_OP, describe_mismatch(got, want, name)


def describe_mismatch(a, b, name=""):
    d = np.abs(a.astype(np.float64) - b)
    idx = np.unravel_index(np.argmax(d), d.shape)
    bad = d > 1e-2 * max(np.abs(b).max(), 1e-30)
    return "%s shape=%s rel_max=%.3e rel_l2=%.3e worst@%s got=%.5f want=%.5f bad_frac=%.4f" % (
        name, a.shape, rel_max(a, b), rel_l2(a, b), idx, a[idx], b[idx], bad.mean())


# ---- the reference's net definitions, stored as generator calls (tests/golden/reference_nets.json) ----
# Every prototxt the reference ships under models_ECO_*/ is rebuilt from tools/gen_eco_prototxt.py (the two pretrained
# backbones from the builders below, made of its pieces) plus, for a train/test net, the text of its VideoData layers; the SHA-256 of the reference file's parsed tree pins the
# rebuilt text to the file (tests/golden/make_reference_nets.py writes the JSON and checks every rebuild).

def norm_tree(v):
    """a parsed prototxt with every number as float, so 1 and 1.0 compare equal"""
    from oracle import prototxt
    if isinstance(v, prototxt.Msg):
        return {k: [norm_tree(x) for x in vv] for k, vv in v.items()}
    if isinstance(v, (int, float)) and not isinstance(v, bool):
        return float(v)
    return v


def tree_sha256(tree):
    return hashlib.sha256(json.dumps(norm_tree(tree), sort_keys=True).encode()).hexdigest()


def reference_nets():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_nets.json")) as f:
        return json.load(f)["nets"]


def bn_inception_deploy():
    """the 2-D backbone the reference ships pretrained (models_ECO_Lite/kinetics/bn_inception_kinetics_rgb_pretrained):
    BN-Inception up to inception_5b, 400-way classifier"""
    import gen_eco_prototxt as gen
    o = gen._W()
    o.w('input: "data"')
    o.w("input_shape { dim: 1 dim: 3 dim: 224 dim: 224 }")
    t = gen._trunk_to_3c(o, "data")
    t = gen._inception(o, "3c", t, 0, 128, 160, 64, 96, 96, "MAX", 0, stride2=True)
    t = gen._inception(o, "4a", t, 224, 64, 96, 96, 128, 128, "AVE", 128)
    t = gen._inception(o, "4b", t, 192, 96, 128, 96, 128, 128, "AVE", 128)
    t = gen._inception(o, "4c", t, 160, 128, 160, 128, 160, 160, "AVE", 128)
    t = gen._inception(o, "4d", t, 96, 128, 192, 160, 192, 192, "AVE", 128)
    t = gen._inception(o, "4e", t, 0, 128, 192, 192, 256, 256, "MAX", 0, stride2=True)
    t = gen._inception(o, "5a", t, 352, 192, 320, 160, 224, 224, "AVE", 128)
    t = gen._inception(o, "5b", t, 352, 192, 320, 192, 224, 224, "MAX", 128)
    gen._pool(o, "global_pool", t, "AVE", 7, 1)
    o.w('layer { name: "dropout" type: "Dropout" bottom: "global_pool" top: "global_pool"')
    o.w("  dropout_param { dropout_ratio: 0.800000011921 } }")
    o.w('layer { name: "fc_action" type: "InnerProduct" bottom: "global_pool" top: "fc_action"')
    o.w("  param { lr_mult: 1 decay_mult: 1 } param { lr_mult: 1 decay_mult: 2 }")
    o.w('  inner_product_param { num_output: 400 weight_filler { type: "xavier" } bias_filler { type: "constant" value: 0 } } }')
    return o.f.getvalue()


def c3d_resnet18_train():
    """the 3-D backbone the reference ships pretrained (models_ECO_Lite/kinetics/112_c3d_resnet18_kinetics_rgb_pretrained):
    a 3-D ResNet-18 on 16 x 112 x 112 clips, 101-way classifier, behind the net inputs its VideoData layers produce"""
    import gen_eco_prototxt as gen
    o = gen._W()
    o.w('name: "C3D"')
    o.w('input: "data"')
    o.w("input_dim: 1\ninput_dim: 48\ninput_dim: 112\ninput_dim: 112")
    o.w('input: "label"')
    o.w("input_dim: 1\ninput_dim: 1\ninput_dim: 1\ninput_dim: 1")
    o.w('layer { name: "data_reshape" type: "Reshape" bottom: "data" top: "data_reshape"')
    o.w("  reshape_param { shape { dim: -1 dim: 3 dim: 16 dim: 112 dim: 112 } } }")
    o.w('layer { name: "conv1" type: "Convolution" bottom: "data_reshape" top: "conv1"')
    o.w("  convolution_param { num_output: 64 pad: [1, 3, 3] kernel_size: [3, 7, 7] stride: [2, 2, 2]")
    o.w('    weight_filler { type: "xavier" } bias_filler { type: "constant" value: 0 } }')
    o.w("  param { lr_mult: 1 decay_mult: 1 } param { lr_mult: 2 decay_mult: 0 } }")
    gen._bn3d(o, "conv1_bn", "conv1")
    o.w('layer { name: "relu1" type: "ReLU" bottom: "conv1_bn" top: "conv1_bn" }')
    t, shortcut = "conv1_bn", "conv1"
    for b in ("res2a", "res2b"):
        gen._conv3d(o, b + "_1", t, b + "_1", 64, 1)
        u = gen._bnrelu3d(o, b + "_1", b + "_1")
        gen._conv3d(o, b + "_2", u, b + "_2", 64, 1)
        gen._eltwise(o, b, *((shortcut, b + "_2") if b == "res2a" else (b + "_2", shortcut)))
        t, shortcut = gen._bnrelu3d(o, b, b), b
    for stage, ch in (("res3", 128), ("res4", 256), ("res5", 512)):   # the stages of gen._head3d's res4 / res5
        a, b = stage + "a", stage + "b"
        gen._conv3d(o, a + "_1", t, a + "_1", ch, 2)
        u = gen._bnrelu3d(o, a + "_1", a + "_1")
        gen._conv3d(o, a + "_2", u, a + "_2", ch, 1)
        gen._conv3d(o, a + "_down", t, a + "_down", ch, 2)
        gen._eltwise(o, a, a + "_2", a + "_down")
        t = gen._bnrelu3d(o, a, a)
        gen._conv3d(o, b + "_1", t, b + "_1", ch, 1)
        u = gen._bnrelu3d(o, b + "_1", b + "_1")
        gen._conv3d(o, b + "_2", u, b + "_2", ch, 1)
        gen._eltwise(o, b, b + "_2", a)
        t = gen._bnrelu3d(o, b, b)
    gen._tail3d(o, 4, 0.5)   # pools over a depth of 4 / 4 = 1: the 16 frames halved by conv1 and three stages
    gen._fc(o, "fc", "global_pool_reshape", 101)
    gen._loss_tail(o)
    return o.f.getvalue()


def reference_net_text(entry, text=None):
    """prototxt text with the same parsed tree as the reference file `entry` describes; `text` replaces the output of
    the generator call the entry stores (a function of tools/gen_eco_prototxt.py, or one of the backbone builders above)"""
    import gen_eco_prototxt as gen
    if text is None:
        make = getattr(gen, entry["make"], None) or globals()[entry["make"]]
        text = make(**entry["kwargs"])
    if entry["data_layers"]:
        # the generator's header declares the inputs a VideoData layer produces; the reference's header and data layers
        # take its place
        text = entry["data_layers"] + text[text.index("layer {"):]
    return text
