"""Both networks at the sizes the product runs them, under the device-side counts it passes (-m gpu).

ReID: one engine of capacity 4 096 (64 streams) through aicam_reid_forward_nhwc8, the call of a batched step, with the
crop count changing on the same buffers, eagerly and from a CUDA graph whose own kernel writes the count right before
the network (as the crop kernel writes crop_count inside a captured step).  YOLOv8n: a 64-entry frame table of 1080p
frames through aicam_preprocess_table format 3 and aicam_yolo_detect_table (4x4-block stem; fused decode at 80 classes,
the fp32 head tensor and decode_kernel at 20) with 64, 37, 1 and 64 present frames.  Everything past the count is
poisoned with NaN; what lies below it must be bit-identical with the full run, and samples must match the fp32 oracle
nets."""
import ctypes as C

import numpy as np
import pytest
import torch

from scenarios import synth_image

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
REID_CAP = 4096
REID_COUNTS = (4096, 1500, 1, 857, 129, 1115, 4096)
POOL = 512  # distinct crops; crop i is crop i % POOL shifted by i // POOL columns
SENTINEL = 7.25
TILES = (128, 256, 512)
# padded raster positions per crop of ReID layers 1 - 4 (shared border: (h + 1)(w + 1))
REID_RASTERS = (65 * 33, 33 * 17, 17 * 9, 9 * 5)


@pytest.fixture(scope="module")
def blobs(tmp_path_factory):
    from ai_camera_b200 import synth
    return synth.make_blobs(str(tmp_path_factory.mktemp("blobs")))


def _lib():
    from ai_camera_b200 import _lib as L
    return L.load()


def _check(rc):
    from ai_camera_b200 import _lib as L
    L.check(rc)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _crops():
    """(REID_CAP, 3, 128, 64) bf16 crops on the device, cut with image_ops.reid_batch from synthetic frames."""
    from oracle import image_ops
    rng = np.random.default_rng(2026)
    pool = []
    for _ in range(4):
        frame = synth_image(rng, 540, 960)
        rects = []
        for _ in range(POOL // 4):
            x, y = int(rng.integers(0, 900)), int(rng.integers(0, 480))
            rects.append((x, y, min(960, x + int(rng.integers(12, 160))), min(540, y + int(rng.integers(30, 300)))))
        pool.append(image_ops.reid_batch(frame, rects))
    pool = torch.from_numpy(np.concatenate(pool)).to(DEV)
    crops = torch.cat([torch.roll(pool, shifts=g, dims=3) for g in range(REID_CAP // POOL)])
    return crops.to(torch.bfloat16)


def _reid_sample(counts):
    """About 48 crops: the first and last of every count, and crops whose layer-1 to layer-4 rasters meet a tile or
    CTA-pair boundary."""
    s = {0}
    for n in counts:
        s |= {n - 1, min(n, REID_CAP - 1)}
    rng = np.random.default_rng(5)
    for R in REID_RASTERS:
        for T in TILES:
            for j in (1, 2, 3, *rng.integers(4, REID_CAP * R // T, 2)):
                s.add(min(REID_CAP - 1, int(j) * T // R))
    return sorted(s)[:48]


def test_reid_at_product_capacity_under_changing_counts(blobs):
    from oracle import nets
    _, reid = blobs
    lib = _lib()
    crops = _crops()
    nhwc8 = torch.zeros((REID_CAP, 128, 64, 8), dtype=torch.bfloat16, device=DEV)
    nhwc8[..., :3] = crops.permute(0, 2, 3, 1)
    h = C.c_void_p()
    _check(lib.aicam_engine_create(reid.encode(), 0, REID_CAP, C.byref(h)))
    try:
        assert lib.aicam_engine_accepts_nhwc8(h) == 1
        buf = torch.empty_like(nhwc8)
        feats = torch.empty((REID_CAP, 512), dtype=torch.float32, device=DEV)
        n_dev = torch.zeros(1, dtype=torch.int32, device=DEV)

        def stage(n):
            buf.copy_(nhwc8)  # (the crops a smaller count poisoned are back in place)
            buf[n:] = float("nan")
            feats.fill_(SENTINEL)

        def check_rows(n, got, want, tag):
            assert torch.equal(got[:n], want[:n]), "%s n=%d: rows < n differ from the full run (%d rows)" % (
                tag, n, int((got[:n] != want[:n]).any(1).sum()))
            assert bool((got[n:] == SENTINEL).all()), "%s n=%d: a feature row >= n was written" % (tag, n)

        full = None
        for n in REID_COUNTS:
            stage(n)
            n_dev.fill_(n)
            _check(lib.aicam_reid_forward_nhwc8(h, _ptr(buf), REID_CAP, _ptr(n_dev), _ptr(feats), None))
            torch.cuda.synchronize()
            if full is None:
                full = feats.clone()
                assert bool(torch.isfinite(full).all())
            check_rows(n, feats, full, "eager")

        # the count written by a kernel of the same graph, right before the network
        src = torch.zeros(1, dtype=torch.int32, device=DEV)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            torch.mul(src, 1, out=n_dev)
            _check(lib.aicam_reid_forward_nhwc8(h, _ptr(buf), REID_CAP, _ptr(n_dev), _ptr(feats),
                                                C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        for n in (1500, 1, 1115, 4096, 857, 129):
            stage(n)
            n_dev.fill_(REID_CAP)  # (a stale count the graph must overwrite)
            src.fill_(n)
            g.replay()
            torch.cuda.synchronize()
            check_rows(n, feats, full, "graph")
        del g
    finally:
        lib.aicam_engine_destroy(h)

    sample = _reid_sample(REID_COUNTS)
    x = crops[torch.tensor(sample, device=DEV)].float().cpu()
    want = nets.load_net(reid).forward(x).numpy()
    got = full[torch.tensor(sample, device=DEV)].cpu().numpy()
    cos = (got * want).sum(1) / (np.linalg.norm(got, axis=1) * np.linalg.norm(want, axis=1))
    print("reid at capacity %d: %d sampled crops, cosine min %.6f" % (REID_CAP, len(sample), cos.min()))
    assert cos.min() >= 0.999, [sample[i] for i in np.nonzero(cos < 0.999)[0]]


def test_yolov8n_frame_table_of_64_1080p_frames_under_present_counts(blobs):
    """80 classes: the decode runs inside the Detect-head epilogues."""
    _frame_table_under_present_counts(blobs[0], 80)


def test_yolov8n_frame_table_without_fused_decode(tmp_path):
    """20 classes: no fused decode, so the network writes the fp32 head tensor and decode_kernel reads it.  The dense
    arrays sit in the same workspace layout, so the checks are those of the 80-class run."""
    from ai_camera_b200 import weights as W
    yolo = str(tmp_path / "yolov8n_nc20.aicw")
    W.write_blob(yolo, *W.synth_yolov8_weights("n", nc=20, seed=0))
    _frame_table_under_present_counts(yolo, 20)


def _frame_table_under_present_counts(yolo, nc):
    from ai_camera_b200 import synth
    from ai_camera_b200.pipeline import BatchDetector, FrameTable
    from oracle import detect_post, image_ops
    from oracle.pipeline import Detector
    S, A = 64, 8400
    lib = _lib()
    det = BatchDetector(yolo, S)
    bias = synth.shifted_class_bias(yolo, -0.6)
    synth.apply_class_bias(det.engine, bias)
    e = det.engine
    assert det._s2d == 2 and e.fused_decode == (nc == 80) and (e._head is None) == (nc == 80)
    video = synth.SynthVideo(S, (1080, 1920), n_frames=1, device=DEV, seed=808)
    frames = [video.ring[0, s] for s in range(S)]
    table = FrameTable(DEV, S, (1080, 1920))
    rng = np.random.default_rng(37)
    some = np.zeros(S, bool)
    some[rng.choice(S, 37, replace=False)] = True
    one = np.zeros(S, bool)
    one[45] = True
    runs = []
    for present in (np.ones(S, bool), some, one, np.ones(S, bool)):
        table.set([f if p else None for f, p in zip(frames, present)])
        _check(lib.aicam_preprocess_table(table.handle, 3, _ptr(e._nhwc), None))
        count = int(present.sum())
        e._nhwc.view(torch.int16).view(S, -1)[count:] = 0x7FC0  # bf16 NaN in the input slots past the present count
        e._ws.fill_(0)
        det.num_dets.fill_(-1)
        _check(lib.aicam_yolo_detect_table(e.handle, _ptr(e._nhwc), 2, table.handle, C.byref(det._nms), _ptr(e._head),
                                           _ptr(det.num_dets), _ptr(det.boxes_lb), _ptr(det.boxes), _ptr(det.scores),
                                           _ptr(det.labels), _ptr(e._ws), e._ws.numel(), None))
        torch.cuda.synchronize()
        n = S * A
        dense = (e._ws[:n * 16].view(torch.float32).reshape(S, A, 4).clone(), e._ws[n * 16:n * 20].view(torch.float32).reshape(S, A).clone(),
                 e._ws[n * 20:n * 24].view(torch.int32).reshape(S, A).clone())
        rows = [t.clone() for t in (det.num_dets, det.boxes_lb, det.boxes, det.scores, det.labels)]
        runs.append((present, dense, rows))
    (_, dense0, rows0) = runs[0]
    assert int((rows0[0] > 0).sum()) >= S // 2, "too few frames with detections to compare"
    assert int(dense0[2].min()) >= 0 and int(dense0[2].max()) < nc and int(rows0[4].max()) < nc
    for present, dense, rows in runs[1:]:
        slots = np.nonzero(present)[0]
        for j, b in enumerate(slots):
            for d, d0 in zip(dense, dense0):
                assert torch.equal(d[j], d0[b]), "%d present: slot %d (frame %d) dense arrays differ" % (len(slots), j, b)
        for b in range(S):
            if present[b]:
                for r, r0 in zip(rows, rows0):
                    assert torch.equal(r[b], r0[b]), "%d present: NMS rows of frame %d differ" % (len(slots), b)
            else:
                assert int(rows[0][b]) == 0, "%d present: absent frame %d reports detections" % (len(slots), b)

    # four frames of the all-present run against the fp32 oracle (the bars of test_yolov8n_head_matches_oracle)
    net = Detector(yolo, bias_overrides=bias).net
    for b in (0, 21, 42, 63):
        x, _, _ = image_ops.preprocess_yolo_input(frames[b].cpu().numpy())
        want = net.head_flat(torch.from_numpy(x))[0].numpy()
        wb, ws, _ = detect_post.decode(want)
        gb, gs = dense0[0][b].cpu().numpy(), dense0[1][b].cpu().numpy()
        top = np.argsort(-ws)[:200]
        size = np.maximum(wb[top, 2] - wb[top, 0], wb[top, 3] - wb[top, 1])[:, None]
        box_err, score_err = (np.abs(gb[top] - wb[top]) / size).max(), np.abs(gs[top] - ws[top]).max()
        print("frame %d: max box err / size %.2e, max score err %.2e" % (b, box_err, score_err))
        assert box_err < 1e-2 and score_err < 2e-2, b
