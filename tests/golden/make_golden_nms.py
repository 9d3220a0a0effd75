#!/usr/bin/env python
"""Generate tests/golden/reference_nms_kernel.npz: the keep lists of the REFERENCE's own CUDA NMS (lib/utils/nms_kernel.cu,
compiled unmodified by oracle/Makefile into oracle/_ref/libref_nms.so) on the score-sorted box sets that
tests/test_nms_gpu.py::test_against_the_reference_cuda_kernel compares the product's NMS with.
Needs a CUDA device and the oracle build:
    make -C oracle && python tests/golden/make_golden_nms.py [output directory, default tests/golden]
Only the case parameters, a SHA-256 of the input boxes and the keep lists are stored; the boxes come from oracle/synth.py."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import postproc, synth  # noqa: E402

CASES = [(3000, 0.7, False), (6000, 0.7, True), (2000, 0.2, True)]     # (boxes, IoU threshold, ctpn_like)


def case_tag(n, thresh, ctpn_like):
    return "n%d_t%g_%s" % (n, thresh, "ctpn" if ctpn_like else "generic")


def case_boxes(n, ctpn_like):
    dets = synth.make_boxes(77 + n % 5, n, ctpn_like=ctpn_like)
    return np.ascontiguousarray(dets[postproc.order_desc(dets[:, 4])])


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_nms.so"))
    lib.ref_nms.restype = None
    lib.ref_nms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int]
    out = {}
    for n, thresh, ctpn_like in CASES:
        tag = case_tag(n, thresh, ctpn_like)
        dets = case_boxes(n, ctpn_like)
        keep, num = np.zeros(n, np.int32), C.c_int(0)
        lib.ref_nms(keep.ctypes.data, C.byref(num), dets.ctypes.data, n, 5, np.float32(thresh), 0)
        out[tag + "_boxes_sha256"] = np.array(hashlib.sha256(dets.tobytes()).hexdigest())
        out[tag + "_keep"] = keep[:num.value].copy()
        print(tag, "kept", num.value)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "reference_nms_kernel.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
