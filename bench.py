#!/usr/bin/env python
"""bench.py -- tracked frames/sec of the StrongSORT per-frame path on B200.

Metric (BASELINE.json): tracked frames/sec at 1080p, 100 dets/frame (config C2:
"1 stream 1080p synthetic, 100 dets/frame, OSNet-x0.25 ReID on 1xB200"), one
independent synthetic video stream per GPU (stream i -> GPU i, no data-path
collective: weak scaling, SURVEY.md 8e).

One step = one frame: detector post-process of that frame's raw YOLOv8 head (DFL decode + class-aware NMS +
scale_boxes, synthetic ``[144, 5040]`` head of the 384x640 letterboxed frame -- the backbone itself is out of
scope) + the tracker update (``StrongSORT.update(dets, img)``: OSNet ReID of every detection crop + Kalman
predict + gated appearance cost + IoU cost + two linear assignments + track-table update).  Seeded
random-weight OSNet (no pretrained file exists offline) and synthetic frames -- "data": "synthetic".

  value  : frames/s with frames and raw heads already resident in HBM, through the
           two-stage pipeline (``update_pipelined(lag=2)``: the OSNet of frame k on one stream
           overlaps the association of frame k-1 on another, rows come back two calls later so
           that no host round trip sits between frames; identical results), K frames
           timed as a whole with CUDA events; inputs rotate through W+K distinct frames
           (>= 5x the L2), ``detail.serial_flushed_ms_per_step`` is the one-frame-at-a-
           time figure with a 256 MiB L2 flush between steps
  e2e    : frames/s through the public streaming call ``StrongSORT.update_pipelined`` (what the
           CLI's frame loop calls) with the frame in pinned HOST memory (the raw head is what the
           detector backbone leaves on the device): H2D of the frame and the D2H of the result
           rows inside the timed region every step, the same ``lag=2``; ``e2e.lag1`` is the call
           at one frame of latency, ``e2e.synchronous`` the blocking ``StrongSORT.update`` (the reference's call
           shape: one host synchronisation per frame, nothing overlaps across frames)
  stages : per-stage microseconds of one serial frame (CUDA events between the kernels)
  roofline     : ReID forward (``ssb_reid``, the dominant kernels) timed alone with CUDA
                 events; algorithmic flops 2*82.3e6*N per frame vs the measured
                 bf16 peak in MEASURED_PEAKS.json; traffic = DRAM bytes of the same
                 forward from the committed ncu --set full capture
  cpu_baseline : the CPU oracle (oracle/: NumPy/SciPy tracker + fp32 torch
                 OSNet; the reference's own StrongSORT code is absent) on the
                 host cores over a bounded sample of the same stream
  clocks       : SM clock / throttle reasons polled through NVML during the timed region

``--workload C4`` runs BASELINE.json's configs[3]; ``--shared-gallery`` adds config C5's
per-frame cross-stream exchange (peer memory over NVLink, NCCL all-gather as the fallback) to the timed
region; at N > 1 the default line measures it in its ``shared_gallery`` block.
``--impl reference`` times that CPU oracle alone and prints the same line.
``--dump-outputs DIR`` saves what the timed loop returned for its last frame (track rows, and the detector
post-process output) as .npy files; the inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "tracked frames/sec at 1080p, 100 dets/frame"
UNIT = "frames/s"
REID_MACS_PER_CROP = 82314880          # oracle/osnet_torch.count_macs()
WORKLOAD = "C2: 1 stream/GPU, 1080p synthetic, 100 dets/frame, OSNet-x0.25 ReID + StrongSORT"
# --workload C4 (not the default bench line): BASELINE.json configs[3]
WORKLOADS = {
    "C2": (METRIC, WORKLOAD),
    "C4": ("tracked frames/sec at 4K, 500 dets/frame, 256 live tracks",
           "C4: 1 stream/GPU, 4K synthetic crowded scene, 500 dets/frame, 256 persistent tracks, "
           "OSNet-x0.25 ReID + StrongSORT"),
}
CFG = "C2"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


NET_HW = (384, 640)                    # 1080p letterboxed for the detector (stride-32 multiple)
NUM_CLASSES = 80


PIPE_LAG = 2      # update_pipelined(..., lag=2): rows come back two calls later, every inter-frame dependency is a device event


def gen_frames(stream_id, count, pin, heads=True):
    """Pre-generate `count` frames of the stream: host images (pinned torch tensors when `pin`), the
    detections a detector would report (class = identity mod 80, so that class-aware NMS keeps
    overlapping objects apart) and -- for the 1080p workload -- the RAW YOLOv8 head [144, 5040] whose
    decode + NMS + scale_boxes reproduces them (the backbone's output, SURVEY.md 8d)."""
    import torch
    from strongsort_yolo_b200 import synth, yolo
    st = synth.make_stream(CFG, stream_id=stream_id)
    rng = np.random.default_rng(1000 + stream_id)
    imgs, dets, raws = [], [], []
    for _ in range(count):
        fr = st.next_frame()
        d = fr.dets.copy()
        d[:, 5] = np.where(fr.gt_ids >= 0, fr.gt_ids % NUM_CLASSES, NUM_CLASSES - 1)
        t = torch.from_numpy(fr.img)
        imgs.append(t.pin_memory() if pin else t)
        dets.append(d)
        if heads and CFG == "C2":
            g, px, py = yolo.letterbox_params(NET_HW, fr.img.shape[:2])
            dn = d.copy()
            dn[:, [0, 2]] = dn[:, [0, 2]] * g + px
            dn[:, [1, 3]] = dn[:, [1, 3]] * g + py
            raws.append(yolo.synth_raw_head_v8(dn, NUM_CLASSES, NET_HW[0], NET_HW[1], rng=rng))
    return imgs, dets, raws


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: an NVML polling thread (every 20 ms,
    in-process, so even a 150 ms region gets several samples); falls back to `nvidia-smi -lms` if NVML
    cannot be loaded.  CUDA_VISIBLE_DEVICES is honoured through the device's UUID / PCI bus id."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, mode="nvml"):
        self.idx = gpu_index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = False
        self._thr = None
        self._smi = None
        self._nv = None
        self.mode = mode
        if mode == "off":
            return
        try:
            if mode == "smi":
                raise RuntimeError("nvidia-smi subprocess requested")
            import pynvml
            import torch
            pynvml.nvmlInit()
            props = torch.cuda.get_device_properties(gpu_index)
            h = None
            try:                                   # the CUDA device's UUID survives CUDA_VISIBLE_DEVICES remapping
                u = str(props.uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID((u if u.startswith("GPU-") else "GPU-" + u).encode())
            except Exception:
                h = None
            if h is None:
                try:
                    h = pynvml.nvmlDeviceGetHandleByPciBusId(
                        ("%08x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)).encode())
                except Exception:
                    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                    ids = [int(v) for v in vis.split(",") if v.strip().isdigit()]
                    h = pynvml.nvmlDeviceGetHandleByIndex(ids[gpu_index] if gpu_index < len(ids) else gpu_index)
            self._h = h
            self._nv = pynvml
        except Exception:
            self._nv = None

    def _poll(self):
        nv = self._nv
        bits = ((nv.nvmlClocksEventReasonHwSlowdown, "hw_slowdown"),
                (nv.nvmlClocksEventReasonHwThermalSlowdown, "hw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_thermal_slowdown"),
                (nv.nvmlClocksEventReasonSwPowerCap, "sw_power_cap"))
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for bit, name in bits:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.mode == "off":
            return
        if self._nv is not None:
            import threading
            try:
                self.max_mhz = float(self._nv.nvmlDeviceGetMaxClockInfo(self._h, self._nv.NVML_CLOCK_SM))
            except Exception:
                self.max_mhz = None
            self._thr = threading.Thread(target=self._poll, daemon=True)
            self._thr.start()
            return
        try:
            self._f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self._smi = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=self._f, stderr=subprocess.DEVNULL)
        except Exception:
            self._smi = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": None}
        if self._thr is not None:
            self._stop = True
            self._thr.join(timeout=2)
            src = "nvml"
            if not self.samples:                   # the poller never ran inside the region: one reading right after it
                try:
                    self.samples.append(float(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)))
                    src = "nvml (single reading right after the timed region)"
                except Exception:
                    pass
            if self.samples:
                out.update(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.max_mhz,
                           reasons=sorted(self.reasons), samples=len(self.samples), source=src)
            return out
        if self._smi is None:
            return out
        self._smi.terminate()
        try:
            self._smi.wait(timeout=5)
        except Exception:
            self._smi.kill()
        self._f.flush()
        rows = [r.strip().split(",") for r in open(self._f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self._f.name)
        sm, reasons = [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); out["sm_max_mhz"] = float(r[2])
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if sm:
            out["sm_mhz"] = float(np.median(sm))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        out["source"] = "nvidia-smi"
        return out


def base_config(world):
    """Identical in both arms (the driver compares the two `config` objects)."""
    cfg = {"workload": WORKLOAD, "streams_per_gpu": 1,
           "frame": [2160, 3840, 3] if CFG == "C4" else [1080, 1920, 3],
           "dets_per_frame_nominal": 500 if CFG == "C4" else 100,
           "detector_postprocess": "none (detections fed directly)" if CFG == "C4" else
           "raw YOLOv8 head [144,5040] -> DFL decode -> class-aware NMS (conf 0.3, iou 0.4) -> scale_boxes",
           "reid": "OSNet-x0.25, seeded random weights, BN calibrated on synthetic crops"}
    return cfg


def pick_threads(img, dets):
    """More threads is not faster for this oracle (small convs: 128 threads ran
    60x slower than 16 on the GPU box's host).  Time one ReID batch at a few
    thread counts and keep the fastest -- "all the host threads it can use"."""
    import torch
    from oracle import osnet_torch, strongsort_np
    from strongsort_yolo_b200 import weights
    ext = osnet_torch.OracleExtractor(weights.load_state_dict(), batch=128)
    xywh = strongsort_np.xyxy2xywh(dets[:, :4])
    boxes = np.asarray([strongsort_np.crop_box_xyxy(b, img.shape[1], img.shape[0]) for b in xywh])[:32]
    n = os.cpu_count() or 1
    best, best_t = 1, float("inf")
    for th in sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n}):
        torch.set_num_threads(th)
        ext(img, boxes[:4])
        t0 = time.perf_counter()
        ext(img, boxes)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = th, dt
        if dt > 4 * best_t:
            break
    return best


def run_oracle(frames_img, frames_dets, frames_raw, warm, timed, threads):
    """CPU oracle seconds per frame over frames [warm, warm+timed): detector post-process restatement
    (decode + NMS + scale_boxes, when raw heads are given) + the StrongSORT restatement."""
    import torch
    from oracle import nms_np, osnet_torch, strongsort_np, yolo_decode_np
    from strongsort_yolo_b200 import weights
    torch.set_num_threads(threads)
    ora = strongsort_np.StrongSORTOracle(
        osnet_torch.OracleExtractor(weights.load_state_dict(), batch=128))
    per = []
    for i in range(warm + timed):
        img = frames_img[i].numpy() if hasattr(frames_img[i], "numpy") else frames_img[i]
        t0 = time.perf_counter()
        if frames_raw:
            pred = yolo_decode_np.decode_v8(frames_raw[i], NUM_CLASSES, 0, NET_HW[0], NET_HW[1])
            rows = nms_np.yolo_nms(pred, NUM_CLASSES, 0, 0.3, 0.4, 1000, False)
            d = nms_np.scale_boxes(rows, NET_HW, img.shape[:2])[:, :6]
        else:
            d = frames_dets[i]
        ora.update(d, img)
        dt = time.perf_counter() - t0
        if i >= warm:
            per.append(dt)
    return per


def _ref_worker(job):
    """One CPU stream of the reference arm (its own process: N streams run concurrently at --gpus N)."""
    global CFG, METRIC, WORKLOAD
    stream_id, cfg, warm, steps, threads = job
    CFG = cfg
    METRIC, WORKLOAD = WORKLOADS[CFG]
    imgs, dets, raws = gen_frames(stream_id, warm + steps, pin=False)
    t0 = time.perf_counter()
    per = run_oracle(imgs, dets, raws, warm, steps, threads)
    return float(np.sum(per)), time.perf_counter() - t0


def impl_reference(args, rank):
    """The reference arm: the CPU restatement of the same path (detector post-process + StrongSORT with the
    fp32 torch OSNet) on the host cores -- the reference's own StrongSORT code is absent from /root/reference
    (SURVEY.md section 0).  At --gpus N it runs N independent CPU streams CONCURRENTLY (one process each,
    host threads divided between them), the like-for-like counterpart of N GPU streams."""
    if rank != 0:
        return
    import torch
    from multiprocessing import get_context
    n_streams = max(1, args.gpus)
    steps, warm = min(args.steps, 40), min(max(args.warmup, 1), 3)
    imgs, dets, raws = gen_frames(0, 2, pin=False)
    host = os.cpu_count() or 1
    best = pick_threads(imgs[0].numpy(), dets[0])
    threads = max(1, min(best, host // n_streams))
    if n_streams == 1:
        busy, wall = _ref_worker((0, CFG, warm, steps, threads))
        walls = [busy]
    else:
        with get_context("spawn").Pool(n_streams) as pool:
            res = pool.map(_ref_worker, [(i, CFG, warm, steps, threads) for i in range(n_streams)])
        walls = [r[0] for r in res]
    sec = max(walls)                          # slowest stream's timed seconds for `steps` frames
    fps = n_streams * steps / sec
    ms = 1000.0 * sec / steps
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 (torch OSNet, cosine) + f64 (Kalman, gating, LSAP)",
        "data": "synthetic", "config": base_config(n_streams),
        "detail": {"note": "CPU restatement of the path (reference StrongSORT code absent from the snapshot); "
                           f"{n_streams} concurrent CPU stream(s), {threads} torch threads each on {host} host threads"},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": int(threads * n_streams),
                         "kind": "port", "sample": f"{steps} frames after {warm} warm-up frames per stream, "
                         f"{n_streams} stream(s) concurrently"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


class DetectorPost:
    """The frame's detector post-process (yolo.YoloV8Post: one C call, 5 launches) with LOOK-AHEAD: ``get(i)``
    returns frame i's detections and has already submitted frame i+1's head, so in a stream loop the host never
    waits for a post-process it has just enqueued (the tracker's C-ABI takes the detection count as a host
    integer: one 16-byte read-back per frame, of work that finished a frame ago).  The slots of YoloV8Post rotate
    three deep: a frame's rows stay valid until two more frames have been submitted."""

    def __init__(self, device, frame_hw, raws_dev):
        import torch
        from strongsort_yolo_b200 import yolo
        self.post = yolo.YoloV8Post(NUM_CLASSES, 0, NET_HW[0], NET_HW[1], frame_hw, device=str(device), depth=4)
        self.raws = raws_dev
        self.stream = torch.cuda.Stream(device=device, priority=-1)
        self.pending = {}

    def submit(self, i):
        if 0 <= i < len(self.raws) and i not in self.pending:
            self.pending[i] = self.post.submit(self.raws[i], self.stream)

    def get(self, i, lookahead=True):
        self.submit(i)
        if lookahead:
            self.submit(i + 1)
        return self.post.result(self.pending.pop(i))[:, :6]


def run_gpu_config(args, device, rank, world, lib, barrier, max_over_ranks, K, W, want_cpu):
    """All measurements of one workload (CFG) on this rank's GPU; returns a dict."""
    import ctypes as C
    import torch
    from strongsort_yolo_b200 import _lib
    from strongsort_yolo_b200 import dist as ssb_dist
    from strongsort_yolo_b200.strong_sort import StrongSORT, _HDR_BYTES
    total = W + K
    imgs, dets, raws = gen_frames(rank, total, pin=True)
    use_post = bool(raws)
    H, Wd = imgs[0].shape[0], imgs[0].shape[1]
    trk_kw = dict(max_tracks=2048, max_dets=640) if CFG == "C4" else {}
    imgs_dev = [im.to(device) for im in imgs]
    dets_dev = [torch.from_numpy(d.astype(np.float32)).to(device) for d in dets]
    raws_dev = [torch.from_numpy(r).to(device) for r in raws]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    res = {}

    post = DetectorPost(device, (H, Wd), raws_dev) if use_post else None

    def frame_dets(i, stream=None, lookahead=True):
        """frame i's detections on the device; a serial caller (lookahead False) orders the post-process after its
        own stream (the L2 flush of the serial timing loop)"""
        if not use_post:
            return dets_dev[i]
        if not lookahead and stream is not None and i not in post.pending:
            post.stream.wait_stream(stream)
        return post.get(i, lookahead)

    if args.only_device:
        trk = StrongSORT(device=str(device), **trk_kw)
        pstream = torch.cuda.Stream(device=device)
        for i in range(W):
            trk.update_pipelined(frame_dets(i, pstream), imgs_dev[i], lag=PIPE_LAG)
        trk.flush_pipelined()
        barrier()
        torch.cuda.profiler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.ssb_launch_count()
        e0.record(trk.stream)
        for k in range(K):
            trk.update_pipelined(frame_dets(W + k, pstream), imgs_dev[W + k], lag=PIPE_LAG)
        trk.flush_pipelined()
        e1.record(trk.stream)
        barrier()
        torch.cuda.profiler.stop()
        print(json.dumps({"only_device": True, "ms_per_step": e0.elapsed_time(e1) / K, "steps": K, "warmup": W,
                          "gpu_launches": int(lib.ssb_launch_count() - l0)}), flush=True)
        sys.exit(0)

    # ---------------- (a) serial: one frame at a time, L2 flushed between steps; stage split -------------
    trk = StrongSORT(device=str(device), **trk_kw)
    st = trk.stream

    for i in range(W):
        trk.update(frame_dets(i, st), imgs_dev[i])
    barrier()
    KS = min(K, 30)
    _lib.check(lib.ssb_profile_enable(trk._h, 1))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(KS)]
    stage_ms = np.zeros((KS, 9), dtype=np.float64)
    buf = (C.c_float * 9)()
    for k in range(KS):
        with torch.cuda.stream(st):
            flush.fill_(k & 0xFF)                      # L2 flush, outside the timed events
            ev[k][0].record(st)
        d = frame_dets(W + k, st, lookahead=False)
        ev[k][1].record(st)
        trk.update(d, imgs_dev[W + k])
        ev[k][2].record(st)
        st.synchronize()
        _lib.check(lib.ssb_profile_read(trk._h, buf))
        stage_ms[k] = np.asarray(list(buf))
    _lib.check(lib.ssb_profile_enable(trk._h, 0))
    barrier()
    post_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev]))
    serial_ms = float(np.mean([e[0].elapsed_time(e[2]) for e in ev]))
    names = ["prep", "appearance", "gate", "lsap_a", "iou", "lsap_b", "kf_ema_update", "bookkeep", "gallery_append"]
    stages = {n: float(1000.0 * np.median(stage_ms[:, j])) for j, n in enumerate(names)}
    assoc_us = float(sum(stages.values()))
    res["serial_ms"] = serial_ms
    del trk

    # ---------------- (b) value: two-stage pipeline, device-resident inputs, K frames as a whole ----------
    trk = StrongSORT(device=str(device), **trk_kw)
    st = trk.stream
    sptr = C.c_void_p(st.cuda_stream)
    gal = ssb_dist.SharedGallery(trk) if args.shared_gallery else None
    pstream = torch.cuda.Stream(device=device)          # detector post-process of the next frame
    for i in range(W):
        trk.update_pipelined(frame_dets(i, pstream), imgs_dev[i], lag=PIPE_LAG)
        if gal is not None:
            gal.step()
    trk.flush_pipelined()
    barrier()
    clocks = ClockSampler(device.index, args.clock_sampler)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = lib.ssb_launch_count()
    e0.record(st)
    for k in range(K):
        d_last = frame_dets(W + k, pstream)
        trk.update_pipelined(d_last, imgs_dev[W + k], lag=PIPE_LAG)
        if gal is not None:
            gal.step()                     # export + exchange + cross-stream match, inside the timed region
    rows_last = trk.flush_pipelined()
    if gal is not None:
        st.wait_stream(gal.stream)
    e1.record(st)
    barrier()
    # what a caller of the timed path receives for the last timed frame (--dump-outputs); copied before the
    # detector post-process slots are reused below
    res["outputs"] = {"tracks": np.asarray(rows_last, dtype=np.float64)}
    if use_post:
        res["outputs"]["detections"] = d_last.cpu().numpy()
    launches = int(lib.ssb_launch_count() - l0)
    t_ms = max_over_ranks(e0.elapsed_time(e1))
    res["clocks"] = clocks.stop()
    res["ms_per_step"] = t_ms / K
    res["value"] = world * K / (t_ms / 1000.0)
    res["launches"] = launches
    final_next_id = int(trk.last_counts[3])
    res["n_cross"] = len(gal.report()) if gal is not None else None

    # ---------------- config C5's optional exchange, same invocation (N > 1): overhead of the shared gallery ----
    if world > 1 and not args.shared_gallery and CFG == "C2":
        trkg = StrongSORT(device=str(device), **trk_kw)
        galg = ssb_dist.SharedGallery(trkg)
        K2 = min(K, 60)
        for i in range(W):
            trkg.update_pipelined(frame_dets(i, pstream), imgs_dev[i], lag=PIPE_LAG)
            galg.step()
        trkg.flush_pipelined()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(trkg.stream)
        for k in range(K2):
            trkg.update_pipelined(frame_dets(W + k, pstream), imgs_dev[W + k], lag=PIPE_LAG)
            galg.step()
        trkg.flush_pipelined()
        trkg.stream.wait_stream(galg.stream)
        g1.record(trkg.stream)
        barrier()
        fps_g = world * K2 / (max_over_ranks(g0.elapsed_time(g1)) / 1000.0)
        res["gallery"] = {"value": fps_g, "unit": UNIT, "steps": K2,
                          "shared_gallery_overhead": 1.0 - fps_g / res["value"],
                          "exchange": ("peer memory: the match kernel pulls the other streams' packed exports "
                                       "[256 x 512 f32 features | 256 ids] over NVLink itself (symmetric memory + "
                                       "device-side barrier, no collective)" if galg.exchange == "peer" else
                                       "one all_gather_into_tensor (NCCL over NVLink) of the packed export "
                                       "[256 x 512 f32 features | 256 ids] per rank per frame") + ", on a side stream",
                          "nvlink_bytes_per_frame_per_rank": int((world - 1) * galg.t_max * (512 + 1) * 4),
                          "cross_stream_matches_last_frame_rank0": len(galg.report())}
        del trkg, galg

    # ---------------- ReID alone: roofline of the dominant kernels ------------------------------------
    i0 = W + K // 2
    n0 = int(dets_dev[i0].shape[0])
    boxes = torch.zeros((n0, 4), dtype=torch.int32, device=device)
    feats = torch.zeros((n0, 512), dtype=torch.float32, device=device)
    with torch.cuda.stream(st):
        _lib.check(lib.ssb_crop_boxes(_lib.ptr(dets_dev[i0]), n0, H, Wd, _lib.ptr(boxes), sptr))
        reps = 20
        rev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for r in range(3 + reps):
            if r >= 3:
                flush.fill_(r)
                rev[r - 3][0].record(st)
            _lib.check(lib.ssb_reid(trk._h, _lib.ptr(imgs_dev[i0]), H, Wd, 3 * Wd, _lib.ptr(boxes),
                                    n0, _lib.ptr(feats), sptr))
            if r >= 3:
                rev[r - 3][1].record(st)
    st.synchronize()
    res["reid_ms"] = float(np.mean([a.elapsed_time(b) for a, b in rev]))
    res["reid_n"] = n0
    res["tc_status"] = trk.reid_tc_status()
    del trk

    # ---------------- e2e: frame in pinned host memory through StrongSORT.update ------------------------
    trk2 = StrongSORT(device=str(device), **trk_kw)
    for i in range(W):
        trk2.update(frame_dets(i, trk2.stream), imgs[i])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(trk2.stream)
    t0 = time.perf_counter()
    n_seen = 0
    for k in range(K):
        trk2.prefetch(imgs[W + k])                 # the frame's H2D runs under the detector post-process
        d = frame_dets(W + k, pstream, lookahead=False)       # synchronous caller: this frame's head only
        n_seen += int(d.shape[0])
        trk2.update(d, imgs[W + k])
    e1.record(trk2.stream)
    barrier()
    e2e_s = max_over_ranks(max(time.perf_counter() - t0, e0.elapsed_time(e1) / 1000.0))
    res["e2e"] = world * K / e2e_s
    res["same_ids"] = int(trk2.last_counts[3]) == final_next_id
    res["dets_per_frame"] = n_seen / K
    res["h2d"] = int(imgs[0].numel() + (0 if use_post else np.mean([len(d) for d in dets]) * 24))
    res["d2h"] = int(trk2._out_bytes + (16 if use_post else 0))
    del trk2

    # ---------------- e2e, streaming call: update_pipelined with host frames -----------------------------
    trk3 = StrongSORT(device=str(device), **trk_kw)
    for i in range(W):
        trk3.update_pipelined(frame_dets(i, pstream), imgs[i], lag=PIPE_LAG)
    trk3.flush_pipelined()
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        trk3.update_pipelined(frame_dets(W + k, pstream), imgs[W + k], lag=PIPE_LAG)
    trk3.flush_pipelined()
    torch.cuda.synchronize()
    res["e2e_streaming"] = world * K / max_over_ranks(time.perf_counter() - t0)
    res["same_ids_streaming"] = int(trk3.last_counts[3]) == final_next_id
    del trk3
    trk3 = StrongSORT(device=str(device), **trk_kw)              # the same at one frame of latency
    for i in range(W):
        trk3.update_pipelined(frame_dets(i, pstream), imgs[i], lag=1)
    trk3.flush_pipelined()
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        trk3.update_pipelined(frame_dets(W + k, pstream), imgs[W + k], lag=1)
    trk3.flush_pipelined()
    torch.cuda.synchronize()
    res["e2e_streaming_lag1"] = world * K / max_over_ranks(time.perf_counter() - t0)
    del trk3

    res.update(stages_us=stages, assoc_us=assoc_us, post_us=1000.0 * post_ms, frames=total,
               frame_bytes=int(imgs[0].numel()), H=H, W=Wd, use_post=use_post)

    # ---------------- CPU baseline (rank 0, N=1 only) ---------------------------------------------------
    if want_cpu:
        img0 = imgs[0].numpy()
        cores = pick_threads(img0, dets[0])
        warm_c, timed_c = 3, args.cpu_frames
        per = run_oracle(imgs, dets, raws, warm_c, timed_c, cores)
        one = run_oracle(imgs, dets, raws, 1, 2, 1)
        res["cpu"] = {"value": 1.0 / float(np.mean(per)), "unit": UNIT, "cores": int(cores),
                      "kind": "port", "host_cores": os.cpu_count(),
                      "single_thread_value": 1.0 / float(np.mean(one)),
                      "sample": f"{timed_c} frames after {warm_c} warm-up frames of the same stream "
                                "(detector post-process + tracker), thread count = fastest of {4,8,16,32,64,all}; "
                                "single_thread_value: 2 frames after 1 warm-up at 1 thread; "
                                "CPU restatement of StrongSORT (reference code absent from the snapshot)"}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-sampler", default="nvml", choices=["nvml", "smi", "off"],
                    help="how the SM clock is sampled during the timed region (in-process NVML thread / nvidia-smi subprocess)")
    ap.add_argument("--cpu-frames", type=int, default=20)
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS),
                    help="C2 (default, the BASELINE.json metric) or C4 (4K, 500 dets/frame)")
    ap.add_argument("--no-c4", action="store_true", help="skip the appended C4 block of the N=1 line")
    ap.add_argument("--only-device", action="store_true",
                    help="profiling aid: only the device-resident pipelined loop (for ncu launch lists)")
    ap.add_argument("--shared-gallery", action="store_true",
                    help="config C5's optional exchange: every stream's confirmed-track features exchanged after each "
                         "frame and matched across streams (read-only), inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned for its last frame to DIR "
                         "(rank 0): tracks.npy, float64 [M,7] rows x1,y1,x2,y2,track_id,class_id,conf; "
                         "detections.npy, float32 [N,6] detector post-process output (C2 only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm has none")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    global CFG, METRIC, WORKLOAD
    CFG = args.workload
    METRIC, WORKLOAD = WORKLOADS[CFG]
    if args.impl == "reference":
        impl_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    from strongsort_yolo_b200 import dist as ssb_dist
    if world > 1:
        ssb_dist.init("nccl", device)
    import __graft_entry__ as ge
    if not os.path.exists(os.path.join(ROOT, "strongsort-yolo_b200", "libssb.so")):
        if local_rank == 0:
            ge.build()
        if world > 1:
            dist.barrier()
    from strongsort_yolo_b200 import _lib
    lib = _lib.load()
    peaks, peak_src = load_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        return ssb_dist.max_over_ranks(x, device)

    K, W = args.steps, max(args.warmup, 3)
    want_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline
    r = run_gpu_config(args, device, rank, world, lib, barrier, max_over_ranks, K, W, want_cpu)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in r["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    reid_flops = 2.0 * REID_MACS_PER_CROP * r["reid_n"]
    achieved_tf = reid_flops / (r["reid_ms"] * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    hbm = float(peaks.get("hbm_gbs", 6570.6))
    traffic = traffic_warm = None
    tpath = os.path.join(ROOT, "profiles", "reid_traffic_bytes.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get("dram_bytes_per_reid_forward")             # ncu --set full: caches flushed before every pass
            traffic_warm = tj.get("dram_bytes_per_reid_forward_warm")   # ncu application replay, caches left alone
        except Exception:
            traffic = traffic_warm = None
    n_conf = 256 if CFG == "C4" else 100
    app_bytes = (n_conf * 128 + 128 * ((r["reid_n"] + 127) // 128)) * 512 * 4      # operand planes the kernel streams
    app_gbs = app_bytes / max(r["stages_us"]["appearance"], 1e-3) / 1e3

    # ---- appended C4 block (N=1 only): BASELINE.json configs[3] through the same code
    c4 = None
    if world == 1 and CFG == "C2" and not args.no_c4:
        CFG = "C4"
        METRIC, WORKLOAD = WORKLOADS[CFG]
        K4, W4 = min(K, 30), min(W, 5)
        r4 = run_gpu_config(args, device, rank, world, lib, barrier, max_over_ranks, K4, W4, False)
        c4 = {"workload": WORKLOAD, "metric": METRIC, "value": r4["value"], "unit": UNIT, "steps": K4, "warmup": W4,
              "ms_per_step": r4["ms_per_step"], "e2e": r4["e2e_streaming"], "e2e_synchronous": r4["e2e"],
              "reid_ms": r4["reid_ms"], "assoc_us": r4["assoc_us"], "stages_us": r4["stages_us"],
              "serial_flushed_ms_per_step": r4["serial_ms"], "dets_per_frame": r4["dets_per_frame"],
              "e2e_ids_equal_device_run": bool(r4["same_ids"])}
        CFG = "C2"
        METRIC, WORKLOAD = WORKLOADS[CFG]

    if rank == 0:
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "fp16 hi/lo operand pairs (~22-bit mantissa) with fp32 accumulate on tcgen05 (ReID convs, appearance "
                     "cost) + fp32 (depthwise, decode, NMS) + f64 (Kalman, gating, IoU, LSAP)",
            "data": "synthetic",
            "config": base_config(world),
            "detail": {"streams": world, "dets_per_frame": r["dets_per_frame"],
                       "l2": f"not flushed: inputs rotate through {r['frames']} distinct frames "
                             f"({r['frames'] * r['frame_bytes'] / 1e6:.0f} MB > 126 MB L2)",
                       "pipeline": "detector post-process + embedding of frame k on stream 1 overlap the association of "
                                   "frame k-1 on stream 2 (ssb_embed / ssb_associate); results identical to the serial path",
                       "serial_flushed_ms_per_step": r["serial_ms"],
                       "e2e_ids_equal_device_run": bool(r["same_ids"]),
                       "e2e_streaming_ids_equal_device_run": bool(r["same_ids_streaming"]),
                       "reid_tc_status": r["tc_status"],
                       **({"shared_gallery": "per frame: export of [256,512] f32 + ids per rank, one packed exchange, "
                                             "cross-stream cosine match (read-only) on a side stream; inside the timed region",
                           "cross_stream_matches_last_frame_rank0": r["n_cross"]} if args.shared_gallery else {})},
            "e2e": {"value": r["e2e_streaming"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "call": "StrongSORT.update_pipelined(dets, img) with the frame in pinned host memory -- the call the "
                            "CLI's frame loop makes (yolo_multi_model.py); called with lag=2 it returns frame k-2's rows while "
                            "frames k-1 and k are in flight; every step copies its frame H2D and reads its result rows D2H",
                    "lag_frames": PIPE_LAG,
                    "lag1": {"value": r["e2e_streaming_lag1"], "unit": UNIT,
                             "call": "StrongSORT.update_pipelined(dets, img, lag=1) -- rows of the previous frame, host frame"},
                    "synchronous": {"value": r["e2e"], "unit": UNIT,
                                    "call": "StrongSORT.prefetch(img); dets = detector post-process; StrongSORT.update(dets, img) "
                                            "-- the reference's blocking call shape: one host synchronisation per frame, "
                                            "no overlap between frames"}},
            "gpu_launches": r["launches"],
            "clocks": r["clocks"],
            "stages": {"unit": "us per frame (serial, L2 flushed)", "detector_postprocess": r["post_us"],
                       "reid_forward": 1000.0 * r["reid_ms"], **r["stages_us"], "association_total": r["assoc_us"]},
            "roofline": {"bound": "tensor", "kernel": "OSNet ReID forward (all kernels of ssb_reid)",
                         "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf, "traffic": traffic, "traffic_not_flushed": traffic_warm,
                         "peak_source": peak_src,
                         "reid_ms": r["reid_ms"], "flops_per_launch": reid_flops},
            "roofline_cost": {"bound": "hbm", "kernel": "appearance_tc_kernel (cosine-NN cost over the gallery)",
                              "achieved": app_gbs, "peak": hbm, "unit": "GB/s", "frac": app_gbs / hbm,
                              "bytes_per_launch": app_bytes, "us": r["stages_us"]["appearance"]},
        }
        if "cpu" in r:
            line["cpu_baseline"] = r["cpu"]
        if "gallery" in r:
            line["shared_gallery"] = r["gallery"]
        if c4 is not None:
            line["configs"] = {"C4": c4}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
