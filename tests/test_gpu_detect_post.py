"""K3/K4 decode + class-aware bitmask NMS + detect() post-processing vs the oracle (-m gpu)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _planted(rng, A, n_hot, n_classes=6, dup=True):
    boxes = np.zeros((A, 4), np.float32)
    cx, cy = rng.uniform(0, 640, A), rng.uniform(0, 640, A)
    w, h = rng.uniform(8, 200, A), rng.uniform(8, 200, A)
    boxes[:, 0], boxes[:, 1], boxes[:, 2], boxes[:, 3] = cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2
    scores = rng.uniform(0.0, 0.29, A).astype(np.float32)
    hot = rng.choice(A, n_hot, replace=False)
    scores[hot] = rng.uniform(0.3, 0.99, n_hot).astype(np.float32)
    labels = rng.integers(0, n_classes, A).astype(np.int32)
    if dup and n_hot >= 8:  # exact score ties and duplicated boxes
        scores[hot[1]] = scores[hot[0]]
        boxes[hot[3]] = boxes[hot[2]]
        labels[hot[3]] = labels[hot[2]]
        scores[hot[5]] = np.float32(0.3)
    # clusters of near-duplicates around some hot boxes
    for k in hot[: n_hot // 3]:
        j = rng.choice(hot)
        boxes[j] = boxes[k] + rng.normal(0, 3, 4).astype(np.float32)
        labels[j] = labels[k]
    return boxes, scores, labels


@pytest.mark.parametrize("A,n_hot,topk,max_cand", [(8400, 0, 100, 1024), (8400, 1, 100, 1024), (8400, 300, 100, 1024),
                                                   (8400, 1500, 100, 1024), (8400, 1500, 300, 2048),
                                                   (8400, 8400, 100, 1024), (500, 200, 50, 64)])
def test_nms_keep_set_bit_exact(A, n_hot, topk, max_cand):
    import gpu_util as G
    from oracle import detect_post
    rng = np.random.default_rng(A + n_hot + topk)
    B = 3
    data = [_planted(rng, A, n_hot) for _ in range(B)]
    boxes = torch.from_numpy(np.stack([d[0] for d in data])).to(G.DEV)
    scores = torch.from_numpy(np.stack([d[1] for d in data])).to(G.DEV)
    labels = torch.from_numpy(np.stack([d[2] for d in data])).to(G.DEV)
    out = G.nms(boxes, scores, labels, 0.3, 0.5, topk, max_cand, frame_hw=(1080, 1920))
    from oracle import image_ops
    for b in range(B):
        keep, _ = detect_post.select_and_nms(*data[b], 0.3, 0.5, topk, max_cand)
        n = out["num"][b]
        assert n == len(keep)
        assert np.array_equal(out["keep"][b, :n], keep)
        assert np.array_equal(out["boxes"][b, :n], data[b][0][keep])
        assert np.array_equal(out["scores"][b, :n], data[b][1][keep])
        assert np.array_equal(out["labels"][b, :n], data[b][2][keep])
        assert not out["boxes"][b, n:].any() and not out["scores"][b, n:].any()
        p = image_ops.letterbox_params(1080, 1920)
        want = image_ops.scale_bboxes(data[b][0][keep], (1080, 1920), (p["r"], p["r"]), (p["dw"], p["dh"]))
        assert np.array_equal(out["boxes_orig"][b, :n].view(np.uint32), want.reshape(-1, 4).view(np.uint32))


def test_decode_matches_oracle():
    _check_decode(80)


@pytest.mark.parametrize("nc", [1, 3, 4, 12, 100, 601])
def test_decode_matches_oracle_at_class_count(nc):
    _check_decode(nc)


def _check_decode(nc):
    """decode_kernel at any class count: float4 loads when 64 + nc is a multiple of 4, scalar loads otherwise (head
    rows of 65, 67 or 665 floats).  Each thread of an anchor scans a quarter of the classes (`per` classes each);
    exact ties planted across the quarter boundaries must go to the lowest index."""
    import gpu_util as G
    from oracle import detect_post
    rng = np.random.default_rng(5 + nc)
    head = rng.normal(0, 2.0, (2, 8400, 64 + nc)).astype(np.float32)
    head[0, :, 64:] -= 3.0
    per = ((nc + 3) // 4 + 3) // 4 * 4
    starts = [q * per for q in range(1, 4) if q * per < nc]
    # class lists; the lowest of each must win
    ties = [[min(3, nc - 1), min(7, nc - 1)], [0, nc - 1], [0] + starts, starts, [nc - 1, nc // 2]]
    ties += [[s - 1, s] for s in starts] + [[s, min(nc - 1, s + per)] for s in starts]
    ties = [sorted(set(t)) for t in ties if len(set(t)) > 1]
    planted = []
    anchors = rng.choice(np.arange(6, 8400), len(ties), replace=False)
    for t, a in zip(ties, [5] + list(anchors[1:])):
        for b in range(2):
            head[b, a, 64:] = np.minimum(head[b, a, 64:], 8.0)
            head[b, a, [64 + c for c in t]] = 12.0
            planted.append((b, a, t[0]))
    boxes, scores, labels = G.decode(torch.from_numpy(head).to(G.DEV))
    for b in range(2):
        wb, ws, wl = detect_post.decode(head[b])
        assert np.array_equal(labels[b].cpu().numpy(), wl)
        assert np.allclose(scores[b].cpu().numpy(), ws, rtol=1e-5, atol=1e-6)
        assert np.allclose(boxes[b].cpu().numpy(), wb, rtol=1e-4, atol=1e-3)
    assert labels.min().item() >= 0 and labels.max().item() < nc
    assert planted or nc == 1
    for b, a, want in planted:
        assert labels[b, a].item() == want, (b, a, want)
