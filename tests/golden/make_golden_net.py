#!/usr/bin/env python
"""Generate tests/golden/reference_net_wiring*.npz by running the REFERENCE's own inference code -- get_network("VGGnet_test")
(lib/networks/factory.py, VGGnet_test.py, network.py), test_ctpn (lib/fast_rcnn/test.py) and, through tf.py_func, its
proposal layer -- imported unmodified from /root/reference, on top of tests/golden/tf1_stub (a numpy stand-in for the few
TensorFlow 1.x graph functions that code calls; TensorFlow 1.3 itself cannot be installed here).

This pins the WIRING of the network half of the oracle (oracle/net_cpu.py) to the reference's code; the per-op semantics in
the stub are a restatement of TensorFlow's documented behaviour (see the stub's docstring) -- that part stays unpinned.
Build container only:
    make -C oracle && python tests/golden/make_golden_net.py
cfg.TEST.SCALES / MAX_SIZE are reduced so that the numpy convolutions finish in seconds and the fixture stays small; the
weights are oracle/synth.py::make_weights(seed) keyed by the TF variable names."""
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "tf1_stub"))
import make_golden  # noqa: E402
import make_golden_train  # noqa: E402

CASES = [  # tag, weight seed, image seed, h, w, SCALES, MAX_SIZE
    ("identity", 0, 11, 96, 144, 96, 160),        # im_scale 1
    ("upscaled", 1, 12, 48, 80, 80, 160),         # short side 48 -> 80
    ("capped_odd", 2, 13, 70, 190, 100, 150),     # MAX_SIZE cap; odd feature-map sizes (pool flooring)
]
TAPS = ("conv1_1", "pool1", "conv5_3", "rpn_conv/3x3", "lstm_o", "rpn_cls_score", "rpn_bbox_pred", "rpn_cls_prob_reshape")
PART_BYTES = 1000000      # every fixture file stays below 1 MB: reference_net_wiring.npz, reference_net_wiring_2.npz, ...


def save_parts(out):
    """np.savez_compressed of `out` in key order, starting the next file before one would reach PART_BYTES."""
    parts, part = [], {}
    for k, v in out.items():
        part[k] = v
        buf = io.BytesIO()
        np.savez_compressed(buf, **part)
        if buf.tell() >= PART_BYTES and len(part) > 1:
            del part[k]
            parts.append(part)
            part = {k: v}
    parts.append(part)
    for i, arrays in enumerate(parts):
        path = os.path.join(HERE, "reference_net_wiring%s.npz" % ("_%d" % (i + 1) if i else ""))
        np.savez_compressed(path, **arrays)
        print("wrote", path, os.path.getsize(path), "bytes")


def main():
    cfg = make_golden.load_reference()[0]
    make_golden_train.load_bbox_module()       # network.py imports the training-side operator, which needs lib.utils.bbox
    import tensorflow as tf
    assert tf.__file__.startswith(HERE), "the stub must shadow any real tensorflow"
    from lib.networks.factory import get_network
    from lib.fast_rcnn import test as ref_test
    assert os.path.realpath(ref_test.__file__).startswith(make_golden.REF)
    from oracle import synth

    sess = tf.Session(config=tf.ConfigProto(allow_soft_placement=True))
    net = get_network("VGGnet_test")
    out = {"meta_reference_commit": np.array("c04a571e2593fc361c1aff3127e58dc13fdc4e5a"),
           "variables_requested": np.array(sorted(set(tf.requested_variables)))}
    print("%d variables requested by the graph" % len(set(tf.requested_variables)))
    for tag, wseed, iseed, h, w, scales, max_size in CASES:
        cfg.TEST.SCALES, cfg.TEST.MAX_SIZE = (scales,), max_size
        sess.load_variables(synth.make_weights(wseed))
        im = synth.make_image(iseed, h, w)
        scores, boxes = ref_test.test_ctpn(sess, net, im)
        # the same feed again for the intermediate tensors (test_ctpn fetches only the rois)
        blobs, im_scales = ref_test._get_blobs(im, None)
        info = np.array([[blobs["data"].shape[1], blobs["data"].shape[2], im_scales[0]]], dtype=np.float32)
        feed = {net.data: blobs["data"], net.im_info: info, net.keep_prob: 1.0}
        taps = sess.run([net.get_output(t) for t in TAPS], feed_dict=feed)
        out["%s_cfg" % tag] = np.array([wseed, iseed, h, w, scales, max_size], np.int64)
        out["%s_im_info" % tag] = info
        out["%s_blob" % tag] = blobs["data"]       # stored: cv2's float32 resize differs between OpenCV builds (IPP)
        out["%s_scores" % tag] = scores
        out["%s_boxes" % tag] = boxes
        for name, val in zip(TAPS, taps):
            val = np.asarray(val)
            if name in ("conv1_1", "pool1"):        # large maps: keep a strided sample (rows/cols 0, 5, 10, ...; all channels)
                val = val[:, ::5, ::5, :]
            out["%s_%s" % (tag, name.replace("/", "_"))] = val.astype(np.float32)
        print(tag, "blob", blobs["data"].shape, "scale %.4f" % im_scales[0], "rois", scores.shape[0],
              "heads", taps[TAPS.index("rpn_cls_score")].shape)
    save_parts(out)


if __name__ == "__main__":
    main()
