#!/usr/bin/env python
"""K1 (letterbox / preprocess) and K5 (ReID crops) micro-benchmark against the HBM roofline.
64 x 1080p frames per launch (398 MB BGR / 199 MB NV12: larger than L2), CUDA events around each launch, L2 flushed
between launches by a 512 MB memset; reports the algorithmic bytes (DESIGN section 3) over the median time and the fraction
of MEASURED_PEAKS.json's copy bandwidth.
    python scripts/k1_bench.py [frames] [iters]"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from ai_camera_b200 import _lib  # noqa: E402
from ai_camera_b200._lib import check, ptr  # noqa: E402
from ai_camera_b200.config import tracked_class_mask  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 30
H, W = 1080, 1920
dev = torch.device("cuda:0")
lib = _lib.load()
peak = 6547.0
try:
    peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass
gen = torch.Generator(device=dev).manual_seed(1)
bgr = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=dev, generator=gen)
nv12 = torch.randint(0, 256, (B, H * 3 // 2, W), dtype=torch.uint8, device=dev, generator=gen)
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)


def timed(fn):
    ts = []
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts[3:]))


import subprocess  # noqa: E402
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                          text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:
    card = "%s (nvidia-smi: %s)" % (torch.cuda.get_device_name(0), e)
print("card: %s" % card)
print("K1 / K5 micro-benchmark: %d frames %dx%d, %d launches each, peak %.0f GB/s (MEASURED_PEAKS.json hbm_gbs)" % (B, H, W, iters, peak))
for fmt, name, out_bytes in ((3, "4x4 pixel blocks bf16 (engine input)", 640 * 640 * 8), (2, "2x2 pixel blocks bf16", 640 * 640 * 8), (1, "NHWC4 bf16", 640 * 640 * 8),
                             (0, "NCHW fp32 (reference layout)", 640 * 640 * 12)):
    out = torch.empty(B * out_bytes, dtype=torch.uint8, device=dev)
    for src, frames, fn, row_bytes in (("BGR", bgr, lib.aicam_preprocess, W * 3), ("NV12", nv12, lib.aicam_preprocess_nv12, W * 2)):
        ms = timed(lambda: check(fn(ptr(frames), B, H, W, fmt, ptr(out), None)))
        alg = B * (360 * row_bytes + out_bytes)
        print("K1 %-4s -> %-36s %7.1f us  %6.0f GB/s algorithmic = %4.1f %% of peak" % (src, name, ms * 1e3, alg / ms / 1e6, 100 * alg / ms / 1e6 / peak))

# K5: ~16 person-sized boxes per frame
K = 100
n_per = 16
boxes = torch.zeros((B, K, 4), dtype=torch.float32, device=dev)
cx = torch.rand((B, n_per), device=dev, generator=gen) * 1500 + 200
cy = torch.rand((B, n_per), device=dev, generator=gen) * 700 + 200
hh = torch.rand((B, n_per), device=dev, generator=gen) * 200 + 150
ww = hh * 0.4
boxes[:, :n_per] = torch.stack([cx - ww / 2, cy - hh / 2, cx + ww / 2, cy + hh / 2], dim=-1)
scores = torch.full((B, K), 0.9, dtype=torch.float32, device=dev)
labels = torch.zeros((B, K), dtype=torch.int32, device=dev)
num = torch.full((B,), n_per, dtype=torch.int32, device=dev)
max_crops = B * n_per
det_index = torch.zeros((B, K), dtype=torch.int32, device=dev)
det_count = torch.zeros((B,), dtype=torch.int32, device=dev)
crop_slot = torch.zeros((B, K), dtype=torch.int32, device=dev)
crop_rect = torch.zeros((max_crops, 5), dtype=torch.int32, device=dev)
crops = torch.empty((max_crops, 128, 64, 8), dtype=torch.bfloat16, device=dev)
crop_count = torch.zeros((2,), dtype=torch.int32, device=dev)
lo, hi = tracked_class_mask()
src_bytes = float((ww * hh).sum().item()) * 3  # BGR bytes under the boxes
for src, frames, fn in (("BGR", bgr, lib.aicam_reid_crops), ("NV12", nv12, lib.aicam_reid_crops_nv12)):
    ms = timed(lambda: check(fn(ptr(frames), B, H, W, ptr(boxes), ptr(scores), ptr(labels), ptr(num), K, 0.3, lo, hi, 2, max_crops,
                                ptr(det_index), ptr(det_count), ptr(crop_slot), ptr(crop_rect), ptr(crops), ptr(crop_count), None)))
    alg = src_bytes * (1.0 if src == "BGR" else 0.5) + max_crops * 128 * 64 * 16
    print("K5 %-4s filter + %d crops -> NHWC8 bf16            %7.1f us  %6.0f GB/s algorithmic = %4.1f %% of peak (two launches)" %
          (src, max_crops, ms * 1e3, alg / ms / 1e6, 100 * alg / ms / 1e6 / peak))


# ---- frame-table entry points (aicam_preprocess_table / aicam_reid_crops_table) next to the uniform ones ------------------
def timed_alternating(fns):
    """Median time of each fn, the fns launched in turn inside every iteration (L2 flushed before each launch)."""
    ts = [[] for _ in fns]
    for _ in range(iters):
        for k, fn in enumerate(fns):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    return [float(np.median(t[3:])) for t in ts]


def make_table(frames, bound):
    t = C.c_void_p()
    check(lib.aicam_frame_table_create(0, len(frames), bound[0], bound[1], C.byref(t)))
    descs = (_lib.FrameDesc * len(frames))()
    for d, f in zip(descs, frames):
        if f.dim() == 3:
            d.data, d.chroma, d.h, d.w, d.pitch, d.kind = f.data_ptr(), None, f.shape[0], f.shape[1], f.stride(0), 0
        else:
            h = f.shape[0] * 2 // 3
            d.data, d.chroma, d.h, d.w, d.pitch, d.kind = f.data_ptr(), f.data_ptr() + h * f.stride(0), h, f.shape[1], f.stride(0), 1
    check(lib.aicam_frame_table_set(t, descs, len(frames), None))
    torch.cuda.synchronize()
    return t


import ctypes as C  # noqa: E402
out3 = torch.empty(B * 640 * 640 * 8, dtype=torch.uint8, device=dev)
print("frame table vs uniform entry, alternating launches (median; table / uniform):")
for bound in ((1080, 1920), (2160, 3840)):
    for src, frames, fn, ffn in (("BGR", bgr, lib.aicam_preprocess, lib.aicam_reid_crops), ("NV12", nv12, lib.aicam_preprocess_nv12, lib.aicam_reid_crops_nv12)):
        t = make_table(list(frames), bound)
        u_ms, t_ms = timed_alternating([lambda: check(fn(ptr(frames), B, H, W, 3, ptr(out3), None)),
                                        lambda: check(lib.aicam_preprocess_table(t, 3, ptr(out3), None))])
        print("K1 %-4s format 3, table bound %dx%d: uniform %7.1f us  table %7.1f us  ratio %.3f" % (src, bound[0], bound[1], u_ms * 1e3, t_ms * 1e3, t_ms / u_ms))
        tail = (ptr(boxes), ptr(scores), ptr(labels), ptr(num), K, 0.3, lo, hi, 2, max_crops, ptr(det_index), ptr(det_count),
                ptr(crop_slot), ptr(crop_rect), ptr(crops), ptr(crop_count), None)
        u_ms, t_ms = timed_alternating([lambda: check(ffn(ptr(frames), B, H, W, *tail)),
                                        lambda: check(lib.aicam_reid_crops_table(t, *tail))])
        print("K5 %-4s filter + %d crops, table bound %dx%d: uniform %7.1f us  table %7.1f us  ratio %.3f" % (src, max_crops, bound[0], bound[1], u_ms * 1e3, t_ms * 1e3, t_ms / u_ms))
        lib.aicam_frame_table_destroy(t)


def touched_rows(h, w):
    """Source rows K1 reads for one frame: rows with a non-zero vertical tap (cv2 INTER_LINEAR tables, as preprocess.cu)."""
    r = min(640 / h, 640 / w, 1.0)
    nh = int(round(h * r))
    if nh == h:
        return h
    if h == 2 * nh and w == 2 * int(round(w * r)):
        return h
    rows = set()
    scale = 1.0 / (nh / h)
    for d in range(nh):
        f = np.float32((d + 0.5) * scale - 0.5)
        s = int(np.floor(f))
        f = np.float32(f - np.float32(s))
        w0, w1 = int(np.rint(np.float32(1.0 - f) * 2048)), int(np.rint(f * 2048))
        if w0:
            rows.add(min(max(s, 0), h - 1))
        if w1:
            rows.add(min(max(s + 1, 0), h - 1))
    return len(rows)


mixed_sizes = [(2160, 3840)] * 16 + [(1080, 1920)] * 16 + [(720, 1280)] * 16 + [(540, 960)] * 16
del bgr, nv12
mixed = [torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device=dev, generator=gen) for h, w in mixed_sizes]
t = make_table(mixed, (2160, 3840))
(t_ms,) = timed_alternating([lambda: check(lib.aicam_preprocess_table(t, 3, ptr(out3), None))])
alg = sum(touched_rows(h, w) * 3 * w + 640 * 640 * 8 for h, w in mixed_sizes)
print("K1 BGR mixed 16 x 2160x3840 + 16 x 1080x1920 + 16 x 720x1280 + 16 x 540x960 -> format 3: %7.1f us  %6.0f GB/s algorithmic = %4.1f %% of peak" %
      (t_ms * 1e3, alg / t_ms / 1e6, 100 * alg / t_ms / 1e6 / peak))
for hw in ((2160, 3840), (1080, 1920), (720, 1280), (540, 960)):
    print("   %dx%d: %d source rows touched per frame" % (hw[0], hw[1], touched_rows(*hw)))
lib.aicam_frame_table_destroy(t)
