"""GPU: NMS through the C ABI (ctpn_nms_host via the reference-named wrappers nms()/gpu_nms())
is bit-exact against the CPU oracle and the reference-generated golden keep lists."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from oracle import postproc, synth

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_postproc.npz"))
NMS_TAGS = sorted(k[4:-5] for k in G.files if k.startswith("nms_") and k.endswith("_keep"))
REF_KERNEL = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_nms_kernel.npz"))


@pytest.mark.parametrize("tag", NMS_TAGS)
def test_nms_matches_reference_golden(tag):
    from lib.fast_rcnn.nms_wrapper import nms
    seed, n, ctpn_like = (int(v) for v in G["nms_%s_cfg" % tag])
    dets = synth.make_boxes(seed, n, ctpn_like=bool(ctpn_like))
    keep = nms(dets, float(G["nms_%s_thresh" % tag]))
    np.testing.assert_array_equal(np.asarray(keep, np.int64), G["nms_%s_keep" % tag])


def test_nms_empty_and_single():
    from lib.fast_rcnn.nms_wrapper import nms
    assert nms(np.zeros((0, 5), np.float32), 0.7) == []
    assert nms(np.array([[1, 2, 30, 40, 0.5]], np.float32), 0.7) == [0]


@pytest.mark.parametrize("n,thresh,ctpn_like", [(12000, 0.7, True), (12000, 0.7, False), (5000, 0.2, True), (4097, 0.5, False)])
def test_nms_large_matches_oracle(n, thresh, ctpn_like):
    from lib.utils.gpu_nms import gpu_nms
    dets = synth.make_boxes(40 + n % 7, n, ctpn_like=ctpn_like)
    got = gpu_nms(dets, thresh)
    want = postproc.nms(dets, thresh)
    assert [int(v) for v in got] == want


def test_nms_with_ties_uses_canonical_order():
    from lib.utils.gpu_nms import gpu_nms
    dets = synth.make_boxes(3, 800)
    dets[:, 4] = np.round(dets[:, 4] * 20) / 20          # heavy score ties
    assert [int(v) for v in gpu_nms(dets, 0.5)] == postproc.nms(dets, 0.5)


def test_nms_sorted_batched_early_exit():
    """ctpn_nms_sorted on device pointers: batch of 3 images, ragged counts, max_keep early exit."""
    import torch
    from ctpn_b200 import _native as N
    dev = torch.device("cuda", 0)
    max_n, counts = 3000, [3000, 1777, 1]
    boxes = np.zeros((3, max_n, 4), np.float32)
    want = []
    for b, c in enumerate(counts):
        d = synth.make_boxes(60 + b, c, ctpn_like=(b == 1))
        d = d[postproc.order_desc(d[:, 4])]
        boxes[b, :c] = d[:, :4]
        want.append(postproc.nms_sorted(d, 0.7, max_keep=100))
    bt = torch.from_numpy(boxes).to(dev)
    ct = torch.tensor(counts, dtype=torch.int32, device=dev)
    keep = torch.full((3, 100), -1, dtype=torch.int32, device=dev)
    num = torch.zeros(3, dtype=torch.int32, device=dev)
    ws = torch.empty(N.lib.ctpn_nms_workspace_bytes(3, max_n), dtype=torch.uint8, device=dev)
    N.check(N.lib.ctpn_nms_sorted(N.ptr(bt), N.ptr(ct), 3, max_n, 0.7, 100, N.ptr(keep), N.ptr(num), N.ptr(ws), ws.numel(), N.stream_ptr()), "nms_sorted")
    torch.cuda.synchronize()
    for b in range(3):
        n = int(num[b])
        assert n == len(want[b])
        np.testing.assert_array_equal(keep[b, :n].cpu().numpy(), want[b])
    # too-small workspace is an error, not a crash
    rc = N.lib.ctpn_nms_sorted(N.ptr(bt), N.ptr(ct), 3, max_n, 0.7, 100, N.ptr(keep), N.ptr(num), N.ptr(ws), 1024, N.stream_ptr())
    assert rc == 3 and "workspace" in N.last_error()


@pytest.mark.parametrize("n,thresh,ctpn_like", [(3000, 0.7, False), (6000, 0.7, True), (2000, 0.2, True)])
def test_against_the_reference_cuda_kernel(n, thresh, ctpn_like):
    """ctpn_nms_host vs the reference's `_nms` on identical sorted boxes, through the keep lists that kernel produced on a
    B200 (tests/golden/make_golden_nms.py -> reference_nms_kernel.npz).  The reference kernel is compiled with nvcc's
    default FMA contraction, so an IoU within 1 ulp of the threshold may decide differently; everything else must agree."""
    from ctpn_b200 import _native as N
    tag = "n%d_t%g_%s" % (n, thresh, "ctpn" if ctpn_like else "generic")
    dets = synth.make_boxes(77 + n % 5, n, ctpn_like=ctpn_like)
    dets = np.ascontiguousarray(dets[postproc.order_desc(dets[:, 4])])
    assert hashlib.sha256(dets.tobytes()).hexdigest() == str(REF_KERNEL[tag + "_boxes_sha256"]), \
        "the boxes differ from those the stored keep list was computed on"
    keep_o = np.zeros(n, np.int32); num_o = C.c_int(0)
    N.check(N.lib.ctpn_nms_host(keep_o.ctypes.data, C.byref(num_o), dets.ctypes.data, n, 5, np.float32(thresh), 0), "ctpn_nms_host")
    a, b = REF_KERNEL[tag + "_keep"].tolist(), keep_o[:num_o.value].tolist()
    np.testing.assert_array_equal(np.asarray(b), postproc.nms_sorted(dets, thresh))      # ours == CPU oracle, always
    if a != b:
        sa, sb = set(a), set(b)
        assert len(sa ^ sb) <= max(2, n // 2000), "reference CUDA kernel and ours differ by more than FMA-rounding flips"
