"""Thin helpers for the -m gpu parity tests: every call goes through the C ABI of libaicam.so."""
import ctypes as C

import numpy as np
import torch

from ai_camera_b200 import _lib
from ai_camera_b200._lib import ConvDesc, NmsParams, TrackerConfig, check, ptr

DEV = torch.device("cuda:0")


def lib():
    return _lib.load()


def sync():
    torch.cuda.synchronize()


def bf16_round_np(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).float().numpy()


def conv2d(x_nhwc, w_oihw, bias, ksize, stride, act=0, res=None, res_mode=0, out_f32=False, n_dev=None, out=None):
    """x_nhwc: torch bf16 cuda [B,H,W,Cpad]; w_oihw/bias numpy fp32 (host).  n_dev: optional device int32 [1], the image
    count (B is then the capacity); out: optional output tensor to store into (kept as it is for images >= the count)."""
    B, H, W, _ = x_nhwc.shape
    cout, cin = w_oihw.shape[:2]
    ho = (H + 2 * (ksize // 2) - ksize) // stride + 1
    wo = (W + 2 * (ksize // 2) - ksize) // stride + 1
    if out is None:
        out = torch.empty((B, ho, wo, cout), dtype=torch.float32 if out_f32 else torch.bfloat16, device=DEV)
    d = ConvDesc(B, H, W, cin, cout, ksize, stride, act, res_mode, 1 if out_f32 else 0,
                 n_dev.data_ptr() if n_dev is not None else None)
    w = np.ascontiguousarray(w_oihw, np.float32)
    b = np.ascontiguousarray(bias, np.float32)
    check(lib().aicam_conv2d(C.byref(d), ptr(x_nhwc), ptr(w), ptr(b), ptr(res), ptr(out), None))
    return out


def preprocess(frames_u8, fmt):
    B, H, W, _ = frames_u8.shape
    if fmt == 0:
        out = torch.empty((B, 3, 640, 640), dtype=torch.float32, device=DEV)
    elif fmt == 1:
        out = torch.empty((B, 640, 640, 4), dtype=torch.bfloat16, device=DEV)
    elif fmt == 2:
        out = torch.empty((B, 320, 320, 16), dtype=torch.bfloat16, device=DEV)
    else:
        out = torch.empty((B, 160, 160, 64), dtype=torch.bfloat16, device=DEV)
    check(lib().aicam_preprocess(ptr(frames_u8), B, H, W, fmt, ptr(out), None))
    sync()
    return out


def nms(boxes, scores, labels, score_thr=0.3, iou_thr=0.5, topk=100, max_cand=1024, frame_hw=(0, 0)):
    """boxes [B,A,4] f32, scores [B,A] f32, labels [B,A] i32 (torch cuda) -> dict of numpy arrays."""
    B, A = scores.shape
    p = NmsParams(score_thr, iou_thr, topk, max_cand, frame_hw[0], frame_hw[1])
    ws = torch.empty(max(1, lib().aicam_decode_nms_workspace(B, A, C.byref(p))), dtype=torch.uint8, device=DEV)
    num = torch.empty(B, dtype=torch.int32, device=DEV)
    ob = torch.empty((B, topk, 4), dtype=torch.float32, device=DEV)
    oo = torch.empty((B, topk, 4), dtype=torch.float32, device=DEV)
    os_ = torch.empty((B, topk), dtype=torch.float32, device=DEV)
    ol = torch.empty((B, topk), dtype=torch.int32, device=DEV)
    ki = torch.empty((B, topk), dtype=torch.int32, device=DEV)
    check(lib().aicam_nms(ptr(boxes), ptr(scores), ptr(labels), B, A, C.byref(p), ptr(num), ptr(ob), ptr(oo),
                          ptr(os_), ptr(ol), ptr(ki), ptr(ws), ws.numel(), None))
    sync()
    return dict(num=num.cpu().numpy(), boxes=ob.cpu().numpy(), boxes_orig=oo.cpu().numpy(),
                scores=os_.cpu().numpy(), labels=ol.cpu().numpy(), keep=ki.cpu().numpy())


def decode(head):
    B, A, ch = head.shape
    boxes = torch.empty((B, A, 4), dtype=torch.float32, device=DEV)
    scores = torch.empty((B, A), dtype=torch.float32, device=DEV)
    labels = torch.empty((B, A), dtype=torch.int32, device=DEV)
    check(lib().aicam_decode(ptr(head), B, A, ch - 64, ptr(boxes), ptr(scores), ptr(labels), None))
    sync()
    return boxes, scores, labels


def lsap(costs):
    """costs numpy [n, nr, nc] float32 -> col_for_row [n, nr] int32."""
    n, nr, nc = costs.shape
    c = torch.from_numpy(np.ascontiguousarray(costs, np.float32)).to(DEV)
    out = torch.empty((n, nr), dtype=torch.int32, device=DEV)
    check(lib().aicam_lsap(ptr(c), n, nr, nc, ptr(out), None))
    sync()
    return out.cpu().numpy()


def kf_gating(state, meas):
    n, m = meas.shape[:2]
    s = torch.from_numpy(np.ascontiguousarray(state, np.float32)).to(DEV)
    z = torch.from_numpy(np.ascontiguousarray(meas, np.float32)).to(DEV)
    out = torch.empty((n, m), dtype=torch.float32, device=DEV)
    check(lib().aicam_kf_gating(ptr(s), ptr(z), n, m, ptr(out), None))
    sync()
    return out.cpu().numpy()


class Tracker:
    """n_streams device trackers fed with planted features (replaces the ReID net in tests)."""

    def __init__(self, n_streams=1, max_tracks=128, max_dets=128, feature_dim=512, max_cosine_distance=0.2,
                 max_iou_distance=0.7, max_age=70, n_init=3, nn_budget=100, stride_k=128, frame_hw=(1080, 1920)):
        self.cfg = TrackerConfig(n_streams, max_tracks, max_dets, feature_dim, max_cosine_distance,
                                 max_iou_distance, max_age, n_init, nn_budget, 0)
        self.h = C.c_void_p()
        check(lib().aicam_tracker_create(C.byref(self.cfg), C.byref(self.h)))
        self.S, self.K, self.F, self.T = n_streams, stride_k, feature_dim, max_tracks
        self.frame_hw = frame_hw
        S, K = self.S, self.K
        self.boxes = torch.zeros((S, K, 4), dtype=torch.float32, device=DEV)
        self.scores = torch.zeros((S, K), dtype=torch.float32, device=DEV)
        self.labels = torch.zeros((S, K), dtype=torch.int32, device=DEV)
        self.num = torch.zeros(S, dtype=torch.int32, device=DEV)
        self.det_index = torch.zeros((S, K), dtype=torch.int32, device=DEV)
        self.det_count = torch.zeros(S, dtype=torch.int32, device=DEV)
        self.crop_slot = torch.zeros((S, K), dtype=torch.int32, device=DEV)
        self.crop_rect = torch.zeros((S * K, 5), dtype=torch.int32, device=DEV)
        self.crop_count = torch.zeros(2, dtype=torch.int32, device=DEV)
        self.feats = torch.zeros((S * K, self.F), dtype=torch.float32, device=DEV)
        self.out_tracks = torch.zeros((S, max_tracks, 6), dtype=torch.int32, device=DEV)
        self.out_conf = torch.zeros((S, max_tracks), dtype=torch.float32, device=DEV)
        self.out_count = torch.zeros(S, dtype=torch.int32, device=DEV)

    def close(self):
        if self.h:
            lib().aicam_tracker_destroy(self.h)
            self.h = None

    def step(self, frames, probe=False, feats_null=False):
        """frames: list (one per stream) of dicts boxes/scores/classes/feats (numpy).  Returns, per
        stream, (out [n,6] int64, conf [n] float64).  probe=True: no step; returns, per stream,
        (track_ids [T], app_cost [T,D], gate_d2 [T,D]) from aicam_tracker_cost_probe, and sets
        self.probe_launches to the number of kernels that call launched."""
        from ai_camera_b200.config import tracked_class_mask
        S, K = self.S, self.K
        b = np.zeros((S, K, 4), np.float32)
        sc = np.zeros((S, K), np.float32)
        lb = np.zeros((S, K), np.int32)
        nm = np.zeros(S, np.int32)
        for s, f in enumerate(frames):
            n = len(f["boxes"])
            assert n <= K
            b[s, :n], sc[s, :n], lb[s, :n], nm[s] = f["boxes"], f["scores"], f["classes"], n
        self.boxes.copy_(torch.from_numpy(b))
        self.scores.copy_(torch.from_numpy(sc))
        self.labels.copy_(torch.from_numpy(lb))
        self.num.copy_(torch.from_numpy(nm))
        lo, hi = tracked_class_mask()
        H, W = self.frame_hw
        check(lib().aicam_reid_crops(None, S, H, W, ptr(self.boxes), ptr(self.scores), ptr(self.labels), ptr(self.num),
                                     K, 0.3, lo, hi, 1, S * K, ptr(self.det_index), ptr(self.det_count),
                                     ptr(self.crop_slot), ptr(self.crop_rect), None, ptr(self.crop_count), None))
        sync()
        di, dc, cs = self.det_index.cpu().numpy(), self.det_count.cpu().numpy(), self.crop_slot.cpu().numpy()
        feats = np.zeros((S * K, self.F), np.float32)
        for s, f in enumerate(frames):
            for k in range(dc[s]):
                if cs[s, k] >= 0:
                    feats[cs[s, k]] = f["feats"][di[s, k]]
        self.feats.copy_(torch.from_numpy(feats))
        if probe:
            Dm = self.cfg.max_dets
            app = torch.zeros((S, self.T, Dm), dtype=torch.float32, device=DEV)
            d2 = torch.zeros((S, self.T, Dm), dtype=torch.float32, device=DEV)
            ids = torch.zeros((S, self.T), dtype=torch.int32, device=DEV)
            nt = torch.zeros(S, dtype=torch.int32, device=DEV)
            launches = lib().aicam_launch_count()
            check(lib().aicam_tracker_cost_probe(self.h, ptr(self.boxes), K, ptr(self.det_index), ptr(self.det_count),
                                                 ptr(self.crop_slot), ptr(self.feats), ptr(app), ptr(d2), ptr(ids),
                                                 ptr(nt), None))
            self.probe_launches = lib().aicam_launch_count() - launches
            sync()
            app, d2, ids, nt = app.cpu().numpy(), d2.cpu().numpy(), ids.cpu().numpy(), nt.cpu().numpy()
            return [(ids[s, :nt[s]].astype(np.int64), app[s, :nt[s], :dc[s]], d2[s, :nt[s], :dc[s]]) for s in range(S)]
        check(lib().aicam_tracker_step(self.h, ptr(self.boxes), ptr(self.scores), ptr(self.labels), K,
                                       ptr(self.det_index), ptr(self.det_count), ptr(self.crop_slot),
                                       None if feats_null else ptr(self.feats),
                                       ptr(self.out_tracks), ptr(self.out_conf), ptr(self.out_count), None))
        sync()
        ot, oc, on = self.out_tracks.cpu().numpy(), self.out_conf.cpu().numpy(), self.out_count.cpu().numpy()
        return [(ot[s, :on[s]].astype(np.int64), oc[s, :on[s]].astype(np.float64)) for s in range(S)]

    def snapshot(self, s=0):
        ints = np.zeros((self.T, 7), np.int32)
        floats = np.zeros((self.T, 25), np.float32)
        n = lib().aicam_tracker_snapshot(self.h, s, ptr(ints), ptr(floats), self.T)
        if n < 0:
            check(n)
        return ints[:n].astype(np.int64), floats[:n]

    def overflow(self):
        f = np.zeros(self.S, np.int32)
        check(lib().aicam_tracker_overflow(self.h, ptr(f)))
        return f


def run_gpu_tracker(frames, frame_hw=(1080, 1920), feature_dim=512, **kw):
    """Single-stream scenario through the device tracker -> dict in the golden layout."""
    kmax = max(8, max(len(f["boxes"]) for f in frames))
    max_tracks = kw.pop("max_tracks", 256)
    trk = Tracker(1, max_tracks=max_tracks, max_dets=max(kmax, 8), feature_dim=feature_dim, stride_k=kmax,
                  frame_hw=frame_hw, **kw)
    outs, out_conf, out_off = [], [], [0]
    trk_i, trk_f, trk_off = [], [], [0]
    try:
        for f in frames:
            o, c = trk.step([f])[0]
            outs.extend(o.tolist())
            out_conf.extend(c.tolist())
            out_off.append(len(outs))
            ints, floats = trk.snapshot(0)
            trk_i.extend(ints.tolist())
            trk_f.extend(floats.tolist())
            trk_off.append(len(trk_i))
        assert not trk.overflow().any()
    finally:
        trk.close()
    return dict(out=np.asarray(outs, np.int64).reshape(-1, 6), out_conf=np.asarray(out_conf, np.float64),
                out_off=np.asarray(out_off, np.int64), trk_i=np.asarray(trk_i, np.int64).reshape(-1, 7),
                trk_f=np.asarray(trk_f, np.float32).reshape(-1, 25), trk_off=np.asarray(trk_off, np.int64))
