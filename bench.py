#!/usr/bin/env python
"""bench.py -- images/sec of the CTPN detection hot path (BASELINE.json metric), one line of JSON.

    python bench.py [--config 2|3|4|5] --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 4 --warmup 1      # CPU reference arm (oracle port)
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR   # + the results of the last timed step as DIR/*.npy

--config selects the BASELINE.json configuration (SURVEY.md 8d); the default, 2, is the one the metric is quoted on:
  2  batch 32/GPU x 600x900, fp32-faithful conv arithmetic, DETECT_MODE H             (configs[1])
  3  batch 32/GPU x 600x900 (256 on 8 GPUs), bf16 conv operands / fp32 BiLSTM           (configs[2])
  4  batch 64 x 1200x1600, fp32-faithful, 75 000 anchors -> 12 000 into NMS              (configs[3])
  5  batch 32/GPU of mixed 600x900 / 900x600 images, DETECT_MODE O text lines            (configs[4])

One "step" = one pass of the hot path (uint8 image batch -> conv stack -> BiLSTM -> heads -> proposal layer incl. sort +
NMS -> rois [-> text lines in config 5]) over one batch of synthetic images per GPU; N GPUs process N independent shards
(weak scaling) and the per-image results are gathered with ONE all-gather per batch inside the timed region.
  value : whole-job images/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e   : same metric through the public streaming API with HOST buffers (pinned H2D of the uint8 images and D2H of
          the results inside the timed region; config 5 and `e2e_text_lines`: + the text-line connector on host threads)
  roofline : algorithmic conv FLOPs / CUDA-event time of the tcgen05 conv launches (measured live through the
          library's ctpn_prof_* hooks) vs MEASURED_PEAKS.json; roofline_extra: conv1_1 (HBM), BiLSTM recurrence (fp32 FMA)
  cpu_baseline : the CPU oracle (torch-CPU float32 network + numpy proposal layer, kind "port") timed on this host's
          cores on a bounded sample of the same workload; the same leg measures parity against the oracle and times the
          reference's own CUDA NMS (oracle/_ref) next to ours
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "text-detection-ctpn_b200")
sys.path.insert(0, ROOT)
sys.path.insert(0, PKG)

CONFIGS = {
    2: dict(tag="configs[1]", batch=32, shapes=[(600, 900)], mode="fp32", detect="H"),
    3: dict(tag="configs[2]", batch=32, shapes=[(600, 900)], mode="bf16", detect="H"),
    4: dict(tag="configs[3]", batch=64, shapes=[(1200, 1600)], mode="fp32", detect="H"),
    5: dict(tag="configs[4]", batch=32, shapes=[(600, 900), (900, 600)], mode="fp32", detect="O"),
}
# conv arithmetic modes of the engine (planes of Engine): what one algorithmic MAC costs in bf16-rate MMA units
MODES = {
    "bf16": dict(planes=1, units=1.0, dtype="bf16 operands, fp32 accumulate"),
    "bf16x2": dict(planes=2, units=3.0, dtype="fp32-faithful: bf16x2 split operands (3 tcgen05 MMAs per MAC), fp32 accumulate"),
    "f16f8": dict(planes=4, units=2.0, dtype="fp32-faithful: fp16 operands + e4m3 cross terms (1 kind::f16 + 1 kind::f8f6f4 tcgen05 MMA per 16 MACs: "
                                             "2 bf16-rate units per MAC), fp32 accumulate; matmuls around the BiLSTM on bf16x2"),
    "bf16x3": dict(planes=3, units=6.0, dtype="fp32-equivalent: bf16x3 split operands (6 tcgen05 MMAs per MAC), fp32 accumulate"),
}
FP32_MODE = os.environ.get("CTPN_BENCH_FP32_MODE", "f16f8")      # the float32-faithful mode configs 2/4/5 run in (bf16x2: the 3-unit one)
VGG = [("conv1_1", 3, 64, 0), ("conv1_2", 64, 64, 1), ("conv2_1", 64, 128, 0), ("conv2_2", 128, 128, 1), ("conv3_1", 128, 256, 0),
       ("conv3_2", 256, 256, 0), ("conv3_3", 256, 256, 1), ("conv4_1", 256, 512, 0), ("conv4_2", 512, 512, 0), ("conv4_3", 512, 512, 1),
       ("conv5_1", 512, 512, 0), ("conv5_2", 512, 512, 0), ("conv5_3", 512, 512, 0), ("rpn_conv/3x3", 512, 512, 0)]


def work_per_image(H, W):
    """Algorithmic FLOPs per image (SURVEY.md App. A.1): conv1_1, the 13 other 3x3 layers, GEMMs, recurrence."""
    h, w, conv = H, W, []
    for _name, cin, cout, pool in VGG:
        conv.append(2.0 * h * w * 9 * cin * cout)
        if pool:
            h, w = h // 2, w // 2
    cells = h * w
    return dict(conv1_1=conv[0], conv3x3=sum(conv[1:]), xproj=2.0 * cells * 512 * 1024, fc=2.0 * cells * 256 * 512,
                heads=2.0 * cells * 512 * 64, recurrent=2.0 * cells * 2 * 128 * 512, cells=cells, fh=h, fw=w)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=int(os.environ.get("CTPN_BENCH_CONFIG", "2")), choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the config's)")
    ap.add_argument("--mode", default="", choices=[""] + sorted(MODES), help="conv arithmetic (default: the config's)")
    ap.add_argument("--streams", type=int, default=int(os.environ.get("CTPN_BENCH_STREAMS", "1")), help="sub-batch streams per GPU")
    ap.add_argument("--alt-modes", type=int, default=1, help="config 2 on 1 GPU: also time the bf16x2 (3-unit) and bf16 (configs[2]) arithmetic")
    ap.add_argument("--cpu-sample", type=int, default=4, help="images in the cpu_baseline sample (0: skip that leg)")
    ap.add_argument("--connector-threads", type=int, default=8)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the timed path returned in its last step to DIR/*.npy (inputs are seeded: two builds compare file by file)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


class ClockSampler:
    """nvidia-smi clocks/throttle sampling during the timed region (B200_PROFILING.md recipe), every 50 ms."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for nme, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.f.name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def sources_sha256():
    """Content hash of the kernel sources: a committed ncu traffic figure is only valid for the code it was taken from."""
    h = hashlib.sha256()
    d = os.path.join(PKG, "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the only code here that touches oracle/)
def cpu_oracle_rate(n_images, shapes, detect, warmup=1):
    """images/s of the CPU oracle (network + proposal layer [+ O-mode text lines]) on n_images synthetic images."""
    import numpy as np
    import torch
    from oracle import net_cpu, postproc, synth, textline
    torch.set_num_threads(min(os.cpu_count() or 1, int(os.environ.get("CTPN_CPU_THREADS", "32"))))   # >32 threads is slower on the 128-core host
    w = synth.make_weights(0)

    def one(seed):
        H, W = shapes[seed % len(shapes)]
        info = np.array([[H, W, 1.0]], np.float32)
        im = synth.make_image(seed, H, W)
        blob = (im.astype(np.float32) - net_cpu.PIXEL_MEANS).astype(np.float32)[None]
        r = net_cpu.forward(blob, w)
        rois = postproc.proposal_layer(r["rpn_cls_prob_reshape"], r["rpn_bbox_pred"], info)[0]
        if detect == "O":
            textline.detect(rois[:, 1:5], rois[:, 0:1], (H, W), "O")
        return rois

    for i in range(warmup):
        one(1000 + i)
    t0 = time.perf_counter()
    for i in range(n_images):
        one(i)
    dt = time.perf_counter() - t0
    return n_images / dt, torch.get_num_threads(), dt


def parity_vs_oracle(eng, shapes, seed=7):
    """One image per shape through the engine and through the float32 CPU oracle: head-tensor and proposal deviations."""
    import numpy as np
    import torch
    from oracle import net_cpu, postproc, synth
    w = synth.make_weights(0)
    out = []
    for H, W in shapes:
        im = synth.make_image(seed, H, W)
        blob = (im.astype(np.float32) - net_cpu.PIXEL_MEANS).astype(np.float32)[None]
        ref = net_cpu.forward(blob, w)
        info = np.array([[H, W, 1.0]], np.float32)
        want = postproc.proposal_layer(ref["rpn_cls_prob_reshape"], ref["rpn_bbox_pred"], info)[0]
        cls, box = eng.forward_heads(torch.from_numpy(im[None]).to(eng.device))
        got = eng.rois_batch(im[None], info)[0]
        tol = 1e-3 * np.maximum(1.0, np.abs(want).max(axis=1))
        hit = 0
        for r, t in zip(want, tol):
            hit += bool((np.abs(got - r).max(axis=1) <= t).any()) if len(got) else 0
        out.append({"shape": [H, W], "head_cls_max_abs": float(np.abs(cls.cpu().numpy() - ref["rpn_cls_score"]).max()),
                    "head_bbox_max_abs": float(np.abs(box.cpu().numpy() - ref["rpn_bbox_pred"]).max()),
                    "oracle_rows": int(len(want)), "engine_rows": int(len(got)),
                    "oracle_rows_matched_within_1e-3": hit / max(len(want), 1)})
    return out


def nms_vs_reference(eng, n=12000, reps=5):
    """The reference's own CUDA NMS (lib/utils/nms_kernel.cu compiled into oracle/_ref) against ctpn_nms_host on the same
    12 000 sorted boxes (host in, host out, as gpu_nms.pyx calls it), plus our device-resident generic NMS and the whole
    batched proposal layer (decode + sort + column NMS + emit) per image."""
    import ctypes as C
    import numpy as np
    import torch
    from ctpn_b200 import _native as N
    from oracle import postproc, synth
    path = os.path.join(ROOT, "oracle", "_ref", "libref_nms.so")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/libref_nms.so not built"}
    ref = C.CDLL(path)
    ref.ref_nms.restype = None
    ref.ref_nms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int]
    res = {"boxes": n, "thresh": 0.7, "unit": "ms per call, best of %d" % reps}
    for tag, like in (("ctpn_structured", True), ("generic", False)):
        dets = synth.make_boxes(11, n, ctpn_like=like)
        dets = np.ascontiguousarray(dets[postproc.order_desc(dets[:, 4])])
        keep = np.zeros(n, np.int32)
        num = C.c_int(0)

        def best(fn):
            fn()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                fn()
                ts.append((time.perf_counter() - t0) * 1e3)
            return min(ts)

        t_ref = best(lambda: ref.ref_nms(keep.ctypes.data, C.byref(num), dets.ctypes.data, n, 5, np.float32(0.7), eng.device.index))
        kept_ref = num.value
        t_ours = best(lambda: N.check(N.lib.ctpn_nms_host(keep.ctypes.data, C.byref(num), dets.ctypes.data, n, 5, np.float32(0.7), eng.device.index), "nms"))
        bt = torch.from_numpy(np.ascontiguousarray(dets[:, :4])).to(eng.device)
        kd = torch.empty(n, dtype=torch.int32, device=eng.device)
        nd = torch.zeros(1, dtype=torch.int32, device=eng.device)
        ws = torch.empty(N.lib.ctpn_nms_workspace_bytes(1, n), dtype=torch.uint8, device=eng.device)

        def dev_call():
            N.check(N.lib.ctpn_nms_sorted(N.ptr(bt), None, 1, n, 0.7, 0, N.ptr(kd), N.ptr(nd), N.ptr(ws), ws.numel(), N.stream_ptr()), "nms_sorted")
            torch.cuda.synchronize()
        t_dev = best(dev_call)
        res[tag] = {"reference_nms_kernel_cu_ms": t_ref, "ctpn_nms_host_ms": t_ours, "ctpn_nms_sorted_device_ms": t_dev,
                    "kept": [kept_ref, num.value]}
    # the path the engine actually runs: batched decode + sort + column NMS + emit on head tensors, 32 images
    cls, box = synth.make_head_outputs(3, 37, 56)
    B = 32
    clsd = torch.from_numpy(np.repeat(cls, B, 0)).to(eng.device)
    boxd = torch.from_numpy(np.repeat(box, B, 0)).to(eng.device)
    info = torch.tensor([[600, 900, 1.0]] * B)
    for _ in range(2):
        eng.proposals(clsd, boxd, info, cls_is_logit=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.proposals(clsd, boxd, info, cls_is_logit=False)
    e1.record()
    torch.cuda.synchronize()
    res["proposal_layer_column_path_ms_per_image"] = e0.elapsed_time(e1) / reps / B
    return res


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, packed, shapes, per_shape, rows, world):
    """Results of one step as DIR/rois_<H>x<W>.npy (float32 [images, rows, 5] = score, x1, y1, x2, y2; rows past an image's
    count are zero, as the engine returns them) and DIR/count_<H>x<W>.npy (float64 [images]), images in rank order.
    Above DUMP_BYTES in all, a fixed seeded sample of the images of each shape is written, their indices in
    DIR/image_index_<H>x<W>.npy."""
    import numpy as np
    import torch
    flat = torch.cat([p.reshape(-1) for p in packed]).cpu().numpy().reshape(world, -1)
    n_img = world * per_shape
    keep = min(n_img, DUMP_BYTES // (len(shapes) * (rows * 5 * 4 + 8)))
    os.makedirs(out_dir, exist_ok=True)
    off = 0
    for H, W in shapes:
        n_rois = per_shape * rows * 5
        rois = flat[:, off:off + n_rois].reshape(n_img, rows, 5)
        count = np.ascontiguousarray(flat[:, off + n_rois:off + n_rois + per_shape]).view(np.int32).reshape(n_img)
        off += n_rois + per_shape
        if keep < n_img:
            idx = np.sort(np.random.RandomState(0).choice(n_img, keep, replace=False))
            rois, count = rois[idx], count[idx]
            np.save(os.path.join(out_dir, "image_index_%dx%d.npy" % (H, W)), idx.astype(np.float64))
        np.save(os.path.join(out_dir, "rois_%dx%d.npy" % (H, W)), np.ascontiguousarray(rois, dtype=np.float32))
        np.save(os.path.join(out_dir, "count_%dx%d.npy" % (H, W)), count.astype(np.float64))


def run_reference(a, cfg):
    """Reference arm: the reference's CPU path restated (oracle port; TF 1.3 cannot be installed),
    one image per step, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, cores, dt = cpu_oracle_rate(a.steps, cfg["shapes"], cfg["detect"], warmup=max(a.warmup, 1))
    line = {
        "impl": "reference", "metric": metric_name(cfg), "value": rate, "unit": "images/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1000.0 / rate, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"workload": workload(cfg, 1) + "; one image per step (bounded sample of the batch workload)", "baseline_config": cfg["tag"]},
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "%d images, torch-CPU float32 network + numpy proposal layer%s (oracle/), %.1f s" %
                                   (a.steps, " + O-mode text lines" if cfg["detect"] == "O" else "", dt)},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def metric_name(cfg):
    return "images/sec @%s" % "+".join("%dx%d" % s for s in cfg["shapes"])


def workload(cfg, B):
    shapes = " / ".join("%dx%dx3" % s for s in cfg["shapes"])
    out = "test_ctpn() rois" if cfg["detect"] == "H" else "TextDetector (DETECT_MODE O) text lines"
    return ("batch=%d/GPU %s uint8 synthetic%s, random-init VGG16+BiLSTM+heads (seed 0), proposal layer (12000 pre / 1000 post NMS); "
            "output = %s" % (B, shapes, " (equal shares, one shape bucket each)" if len(cfg["shapes"]) > 1 else "", out))


# ---------------------------------------------------------------------------------------------------------------------
def main():
    a = parse()
    cfg = dict(CONFIGS[a.config])
    if a.impl == "reference":
        return run_reference(a, cfg)
    import numpy as np
    import torch
    import torch.distributed as dist
    from ctpn_b200 import Engine, _native as N, synthetic as synth     # the product arm never touches oracle/

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The all-gather is tiny (0.64 MB per rank and step) and overlaps the next step's persistent, all-SM conv kernels: keep its
        # kernel small (few channels) and give the compute stream scheduling priority, so the collective fills the gaps between
        # kernels instead of holding SMs the conv CTAs are waiting for (measured on 4 GPUs, profiles/r2_multigpu.md)
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        os.environ.setdefault("NCCL_MIN_NCHANNELS", "1")
        dist.init_process_group("nccl", device_id=dev)
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=-1))
    mode = a.mode or (FP32_MODE if cfg["mode"] == "fp32" else cfg["mode"])
    M = MODES[mode]
    B, K = a.batch or cfg["batch"], a.steps
    shapes = cfg["shapes"]
    per_shape = B // len(shapes)
    B = per_shape * len(shapes)
    eng = Engine(synth.make_weights(0), planes=M["planes"], device=local, streams=a.streams)
    rs = np.random.RandomState(100 + rank)
    hosts, images, infos = [], [], []
    for (H, W) in shapes:      # one pinned host batch + one resident device batch per shape bucket
        h = torch.empty((per_shape, H, W, 3), dtype=torch.uint8).pin_memory()
        h.numpy()[...] = rs.randint(0, 256, size=(per_shape, H, W, 3), dtype=np.uint8)
        hosts.append(h)
        images.append(h.to(dev))
        infos.append(torch.tensor([[H, W, 1.0]] * per_shape, dtype=torch.float32, device=dev))
    post = eng.result_rows()

    gather_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    inflight = []            # (packed, gathered, work) of every step of the current region: released only after the region
    latest = []              # what the latest step returned (--dump-outputs)

    def step_device():
        outs = [eng.detect_packed(im, info) for im, info in zip(images, infos)]
        if world > 1:
            # the one collective of the path: all-gather of this step's packed results, issued asynchronously on a side stream
            # behind an event of the compute stream so that it overlaps the next step (drained before the timed region closes;
            # measured on 2 GPUs, tools/dbg_gather.py: +0.6 ms/step, a blocking gather on the compute stream +1.0 ms/step)
            packed = torch.cat(outs) if len(outs) > 1 else outs[0]
            done = torch.cuda.Event()
            done.record(torch.cuda.current_stream())
            with torch.cuda.stream(gather_stream):
                gather_stream.wait_event(done)
                gathered = torch.empty((world * packed.numel(),), dtype=packed.dtype, device=dev)
                work = dist.all_gather_into_tensor(gathered, packed, async_op=True)
            inflight.append((packed, gathered, work))
            outs = [gathered]
        latest[:] = outs
        return outs

    def drain():
        if gather_stream is not None:
            for _p, _g, work in inflight:
                work.wait()
            torch.cuda.current_stream().wait_stream(gather_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def host_stream(n):
        for _ in range(n):
            for h in hosts:
                yield h

    def e2e_rois(n):
        got = None
        for got in eng.rois_batches(host_stream(n), gather=world > 1):
            pass
        return got

    def e2e_lines(n):
        got = None
        for got in eng.detect_lines_batches(host_stream(n), mode=cfg["detect"], workers=a.connector_threads, gather=world > 1):
            pass
        return got

    W_ = max(a.warmup, 3)
    for _ in range(W_):
        step_device()
    drain()
    del inflight[:]
    sampler = ClockSampler(local) if rank == 0 else None
    # ---- value: device-resident inputs, CUDA events ----
    # per-kernel CUDA events (ctpn_prof_*): inside the timed region at N = 1; at N > 1 they perturb the overlap of the all-gather
    # with the next step (measured: -2 % at 2 GPUs), so the timed region runs without them and the per-kernel figures of the
    # roofline come from a separate K-step region right after it
    prof_inside = world == 1
    N.check(N.lib.ctpn_prof_enable(1 if prof_inside else 0), "prof")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        step_device()
    drain()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    timed_outs = list(latest)
    del inflight[:]
    if not prof_inside:
        N.check(N.lib.ctpn_prof_enable(1), "prof")
        for _ in range(K):
            step_device()
        drain()
        barrier()
        del inflight[:]
    prof = N.prof_report()
    N.check(N.lib.ctpn_prof_enable(0), "prof")
    value = world * B * K / (ms / 1e3)
    # ---- e2e: host buffers through the public streaming API ----
    primary = e2e_lines if cfg["detect"] == "O" else e2e_rois
    primary(2)
    barrier()
    t0 = time.perf_counter()
    res = primary(K)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    # second end-to-end figure: the whole ctpn() call chain (adds the text-line connector on host threads)
    lines_s = None
    if cfg["detect"] == "H":
        e2e_lines(2)
        barrier()
        t0 = time.perf_counter()
        e2e_lines(K)
        barrier()
        lines_s = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.stop() if sampler else None
    # single-image latency through the reference-shaped call (host image in, host rois out), 1 GPU only
    lat_ms = None
    if world == 1:
        one = hosts[0][:1]
        for _ in range(3):
            eng.rois_batch(one)
        t1 = time.perf_counter()
        for _ in range(10):
            eng.rois_batch(one)
        lat_ms = (time.perf_counter() - t1) / 10 * 1e3
    n_out = float(sum(len(r) for r in res)) / max(len(res), 1)

    # secondary measurements (config 2, 1 GPU, same box, same process): the other conv arithmetics; not the headline
    alt = None
    if world == 1 and a.config == 2 and a.alt_modes:
        alt = {}
        for m2 in ("bf16x2", "f16f8", "bf16"):
            if m2 == mode:
                continue
            eng1 = Engine(synth.make_weights(0), mode=m2, device=local)
            for _ in range(3):
                eng1.detect_packed(images[0], infos[0])
            N.check(N.lib.ctpn_prof_enable(1), "prof")
            torch.cuda.synchronize()
            e0.record()
            for _ in range(K):
                eng1.detect_packed(images[0], infos[0])
            e1.record()
            torch.cuda.synchronize()
            ms1 = e0.elapsed_time(e1)
            prof1 = N.prof_report()
            N.check(N.lib.ctpn_prof_enable(0), "prof")
            conv1_ms = sum(q["ms"] for q in prof1 if q["kernel"].startswith("conv_tc t9")) / K
            alt[m2] = {"dtype": MODES[m2]["dtype"] + (" (does NOT meet the 1e-3 parity bar; see --config 3 parity)" if m2 == "bf16" else ""),
                       "value": B * K / (ms1 / 1e3), "unit": "images/s", "ms_per_step": ms1 / K, "conv_ms_per_step": conv1_ms,
                       "conv_tflops": work_per_image(*shapes[0])["conv3x3"] * B / (conv1_ms / 1e3) / 1e12}
            del eng1
            torch.cuda.empty_cache()
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        hbm = peaks.get("hbm_gbs", 6500.0)
        peak_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md): 1.4 PFLOP/s sustained bf16, 6.5 TB/s HBM"
        works = [work_per_image(H, W) for H, W in shapes]
        conv = [p for p in prof if p["kernel"].startswith("conv_tc t9")]
        gemm = [p for p in prof if p["kernel"].startswith("conv_tc t1")]
        c11 = [p for p in prof if p["kernel"].startswith("conv1_1")]
        lstm = [p for p in prof if p["kernel"].startswith("bilstm")]
        conv_ms = sum(p["ms"] for p in conv) / K
        alg_flops = sum(w["conv3x3"] for w in works) * per_shape
        achieved = alg_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        traffic, traffic_note = None, "no ncu capture committed for this mode/config"
        try:        # DRAM bytes of the conv launches of one step from the committed ncu --set full capture -- only if it was
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_conv_traffic_cfg%d_%s.json" % (a.config, mode))))   # taken from THIS code
            if tj.get("sources_sha256") != sources_sha256():
                traffic_note = "committed capture is from other kernel sources (sha mismatch): not reported"
            elif tj.get("batch") == B and tj.get("launches") == int(sum(q["launches"] for q in conv)) // K:
                traffic, traffic_note = tj["dram_bytes_per_step"], "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of one step"
        except Exception:
            pass
        tc_launches = int(sum(p["launches"] for p in conv + gemm))
        other = [p for p in prof if not p["kernel"].startswith("conv_tc")]
        c11_ms = sum(p["ms"] for p in c11) / K
        lstm_ms = sum(p["ms"] for p in lstm) / K
        store_planes = 2 if mode == "f16f8" else M["planes"]          # F16F8 stores fp16 + 2 x e4m3 = the bytes of two bf16 planes
        c11_bytes = sum(H * W * (3 + 64 * store_planes * 2) for H, W in shapes) * per_shape
        lstm_flops = sum(w["recurrent"] for w in works) * per_shape
        lstm_bytes = sum(w["cells"] * (1024 * 4 + 256 * 2 * min(store_planes, 3)) for w in works) * per_shape
        fma_peak = 148 * 128 * 2 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / 1e12     # fp32 FMA lanes x 2 flop x max clock
        line = {
            "metric": metric_name(cfg), "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": M["dtype"], "data": "synthetic",
            "config": {"workload": workload(cfg, B), "baseline_config": "BASELINE.json %s (--config %d)" % (cfg["tag"], a.config),
                       "global_batch": world * B, "mode": mode, "planes": M["planes"], "streams": a.streams,
                       "parallelism": "dp%d (independent image shards, one NCCL all-gather of the packed results per batch)" % world,
                       "l2": "no explicit flush: every step streams >4 GB of activations through the 126 MB L2, nothing survives between steps"},
            "e2e": {"value": world * B * K / e2e_s, "unit": "images/s",
                    "h2d_bytes_per_step": sum(per_shape * H * W * 3 + per_shape * 12 for H, W in shapes),
                    "d2h_bytes_per_step": B * post * 5 * 4 + B * 4,
                    "api": "Engine.detect_lines_batches (rois -> host connector threads)" if cfg["detect"] == "O" else "Engine.rois_batches"},
            "gpu_launches": int(sum(p["launches"] for p in prof)) + K * len(shapes) * 6,   # + split_heads + decode/sort/nms/compact/emit
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "conv_tc_kernel (%d tcgen05 3x3 conv launches per step)" % (len(conv) and int(sum(p["launches"] for p in conv)) // K),
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                         "traffic_note": traffic_note, "peak_source": peak_src + " bf16_tflops_sustained", "ms_per_step": conv_ms,
                         "measured_in": "the timed region" if world == 1 else "a separate %d-step region after the timed one (per-kernel events perturb the all-gather overlap at N > 1)" % K,
                         "units_per_mac": M["units"], "executed_mma_tflops_bf16_equivalent": achieved * M["units"],
                         "note": "achieved = algorithmic conv FLOPs (%.2f GFLOP/step) / CUDA-event time of the conv launches; in mode %s "
                                 "each algorithmic MAC costs %.1f bf16-rate MMA units" % (alg_flops / 1e9, mode, M["units"])},
            "roofline_extra": [
                {"kernel": "conv1_tc_kernel (conv1_1)", "bound": "hbm", "achieved": c11_bytes / max(c11_ms, 1e-9) / 1e6, "peak": hbm, "unit": "GB/s",
                 "frac": c11_bytes / max(c11_ms, 1e-9) / 1e6 / hbm, "ms_per_step": c11_ms,
                 "note": "algorithmic bytes = 3 B in + 64 ch x %d planes x 2 B out per pixel" % store_planes},
                {"kernel": "bilstm_kernel (recurrence)", "bound": "fp32 FMA (latency-bound in practice)", "achieved": lstm_flops / max(lstm_ms, 1e-9) / 1e9,
                 "peak": fma_peak, "unit": "TFLOP/s", "frac": lstm_flops / max(lstm_ms, 1e-9) / 1e9 / fma_peak, "ms_per_step": lstm_ms,
                 "hbm_frac": lstm_bytes / max(lstm_ms, 1e-9) / 1e6 / hbm,
                 "note": "0.543 GFLOP/image of h.Wh at 600x900; peak = 148 SMs x 128 lanes x 2 x max SM clock; hbm_frac = (x-projection read + h write) / time / HBM peak"},
            ],
            "stage_ms_per_step": dict({"conv_tc 3x3": conv_ms, "conv_tc 1x1 GEMMs": sum(p["ms"] for p in gemm) / K},
                                      **{p["kernel"]: p["ms"] / K for p in other}),
            "outputs_per_image": n_out,
            "single_image_latency_ms": lat_ms,
            "layers": [{"kernel": q["kernel"], "ms": q["ms"] / K, "alg_tflops": q["work"] / max(q["ms"], 1e-9) / 1e9} for q in conv + gemm],
        }
        if lines_s is not None:
            line["e2e_text_lines"] = {"value": world * B * K / lines_s, "unit": "images/s", "connector_threads": a.connector_threads,
                                      "what": "uint8 host images -> rois -> TextDetector text lines (native host connector, DETECT_MODE H) "
                                              "per image: the whole ctpn() call chain minus file I/O"}
        if alt:
            line["alt_modes"] = alt
        if world == 1 and a.cpu_sample > 0:
            n_cpu = a.cpu_sample if shapes[0][0] < 1000 else max(2, a.cpu_sample // 2)
            rate, cores, dt = cpu_oracle_rate(n_cpu, shapes, cfg["detect"])
            line["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": cores, "kind": "port",
                                    "sample": "%d images of the same workload, torch-CPU float32 network + numpy proposal layer%s (oracle/), %.1f s" %
                                              (n_cpu, " + O-mode text lines" if cfg["detect"] == "O" else "", dt)}
            line["parity"] = {"mode": mode, "vs": "float32 CPU oracle, one synthetic image per shape", "images": parity_vs_oracle(eng, shapes)}
            if a.config == 2:
                line["nms_vs_reference"] = nms_vs_reference(eng)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, timed_outs, shapes, per_shape, post, world)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
