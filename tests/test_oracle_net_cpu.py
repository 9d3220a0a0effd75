"""CPU: the network oracle (oracle/net_cpu.py, "parity unpinned": TF 1.3 cannot run here) against an independently
written second restatement (oracle/net_alt.py: im2col matmul convs, reshape pooling, torch.nn.LSTM with permuted gate
columns and the forget bias folded into the bias).  A shared misreading of the reference graph is still possible; a slip
in only one of them (gate order, forget bias, padding phase, pool flooring, tap order, scan direction) is not."""
import numpy as np
import torch

from oracle import net_alt, net_cpu, synth


def _blob(seed, h, w):
    return (synth.make_image(seed, h, w).astype(np.float32) - net_cpu.PIXEL_MEANS).astype(np.float32)[None]


def test_two_independent_restatements_agree_in_float64():
    w = synth.make_weights(0)
    for seed, (h, wd) in [(0, (64, 96)), (1, (50, 83))]:            # even and odd sizes: pooling floors at every level
        blob = _blob(seed, h, wd)
        a = net_cpu.forward(blob, w, dtype=torch.float64)
        b = net_alt.forward(blob, w)
        for k in ("rpn_cls_score", "rpn_bbox_pred", "rpn_cls_prob_reshape"):
            assert a[k].shape == b[k].shape
            d = np.abs(a[k] - b[k]).max()
            assert d <= 1e-11 * max(1.0, np.abs(b[k]).max()), (k, d)


def test_restatements_agree_on_a_batch_and_reverse_direction_matters():
    w = synth.make_weights(3)
    blob = np.concatenate([_blob(5, 48, 64), _blob(6, 48, 64)])
    a = net_cpu.forward(blob, w, dtype=torch.float64)
    b = net_alt.forward(blob, w)
    assert np.abs(a["rpn_cls_score"] - b["rpn_cls_score"]).max() <= 1e-11
    # sanity of the check itself: swapping the two directions' weights must be visible
    w2 = dict(w)
    w2[net_cpu.LSTM_FW + "/kernel"], w2[net_cpu.LSTM_BW + "/kernel"] = w[net_cpu.LSTM_BW + "/kernel"], w[net_cpu.LSTM_FW + "/kernel"]
    c = net_alt.forward(blob, w2)
    assert np.abs(a["rpn_cls_score"] - c["rpn_cls_score"]).max() > 1e-3


# ---- the oracle against the reference's OWN graph code ---------------------------------------------------------------------
# tests/golden/reference_net_wiring*.npz: get_network("VGGnet_test") + test_ctpn + the py_func proposal layer, imported
# unmodified from /root/reference and executed on tests/golden/tf1_stub (numpy stand-ins for the TensorFlow functions that
# code calls).  Pins the wiring (layer order, variable names, row sequences, fw/bw concatenation, reshapes, pair softmax,
# blob / im_info handling); the per-op semantics inside the stub are a restatement, like the oracle's.
import glob  # noqa: E402
import os  # noqa: E402

import pytest  # noqa: E402

from oracle import postproc  # noqa: E402

WIRING = {}
for _part in sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_net_wiring*.npz"))):
    with np.load(_part) as _z:          # one fixture, split over files of less than 1 MB each (make_golden_net.py)
        WIRING.update(_z)
WIRING_TAGS = sorted(k[:-4] for k in WIRING if k.endswith("_cfg"))


def test_reference_graph_asks_for_exactly_the_variables_the_engine_requires():
    from ctpn_b200.engine import REQUIRED_VARIABLES
    assert sorted(REQUIRED_VARIABLES) == list(WIRING["variables_requested"]) and len(REQUIRED_VARIABLES) == 38
    assert sorted(synth.make_weights(0)) == sorted(REQUIRED_VARIABLES)


@pytest.mark.parametrize("tag", WIRING_TAGS)
def test_oracle_matches_the_reference_graph_code_on_the_tf_stub(tag):
    wseed = int(WIRING[tag + "_cfg"][0])
    w = synth.make_weights(wseed)
    names = {"conv1_1": "conv1_1", "conv1_2+pool": "pool1", "conv5_3": "conv5_3", "rpn_conv/3x3": "rpn_conv_3x3", "lstm_o": "lstm_o",
             "rpn_cls_score": "rpn_cls_score", "rpn_bbox_pred": "rpn_bbox_pred", "rpn_cls_prob_reshape": "rpn_cls_prob_reshape"}
    got = net_cpu.forward(WIRING[tag + "_blob"], w, taps=list(names))
    for ours, theirs in names.items():
        a, b = got[ours], WIRING["%s_%s" % (tag, theirs)]
        if theirs in ("conv1_1", "pool1"):
            a = a[:, ::5, ::5, :]                                     # the fixture keeps a strided sample of the large maps
        assert a.shape == b.shape, (ours, a.shape, b.shape)
        # float32 sums of up to 4608 products in two different orders: measured <= 3.1e-6 of the tensor's maximum
        assert np.abs(a - b).max() <= 2e-5 * max(1.0, np.abs(b).max()), (ours, float(np.abs(a - b).max()))
    info = WIRING[tag + "_im_info"]
    blob, _ = postproc.proposal_layer(got["rpn_cls_prob_reshape"], got["rpn_bbox_pred"], info, exp_mode="numpy")
    scores, boxes = blob[:, 0], blob[:, 1:5] / info[0, 2]            # test.py:54-57
    want_s, want_b = WIRING[tag + "_scores"], WIRING[tag + "_boxes"]
    # Here (same BLAS) the lists are equal row for row: same count, same order, scores within 4.4e-6, boxes within 1.2e-4 px.
    # Asserted order-insensitively with a little slack, so that another float32 summation order (a different oneDNN / BLAS
    # build) that swaps two near-equal scores or flips one NMS decision does not fail the wiring check.
    assert abs(len(scores) - len(want_s)) <= 2
    hit = 0
    for s_ref, b_ref in zip(want_s, want_b):
        close = np.abs(scores - s_ref) <= 2e-5
        hit += bool(close.any()) and bool((np.abs(boxes[close] - b_ref).max(axis=1) <= 1e-3).any())
    assert hit >= 0.98 * len(want_s), (hit, len(want_s))
