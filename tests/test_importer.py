"""Real-checkpoint importer (SURVEY.md 8f N4; replaces /root/reference/scripts/download_models.sh +
export_trt_engines.sh): ONNX initialisers / PyTorch state dicts with the public tensor names -> .aicw blob."""
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from ai_camera_b200 import importer, weights as W


def _unfused(specs, kind, seed, eps):
    """A checkpoint as the public repos save it: bias-free convolutions followed by BatchNorm (plus the plain
    biased 1x1 heads of YOLOv8)."""
    rng = np.random.default_rng(seed)
    t = OrderedDict()
    for name, cin, cout, k, s, act in specs:
        t[name + ".weight"] = rng.normal(0, 1.0 / np.sqrt(cin * k * k), (cout, cin, k, k)).astype(np.float32)
        bn = importer._bn_prefix(name, kind)
        if act == "none" and kind == W.KIND_YOLOV8:
            t[name + ".bias"] = rng.normal(0, 0.1, cout).astype(np.float32)
            continue
        t[bn + ".weight"] = rng.uniform(0.5, 1.5, cout).astype(np.float32)
        t[bn + ".bias"] = rng.normal(0, 0.1, cout).astype(np.float32)
        t[bn + ".running_mean"] = rng.normal(0, 0.1, cout).astype(np.float32)
        t[bn + ".running_var"] = rng.uniform(0.5, 1.5, cout).astype(np.float32)
        t[bn + ".num_batches_tracked"] = np.asarray(7.0, np.float32)
    return t


def _conv_bn(x, t, name, kind, k, s, eps):
    y = F.conv2d(x, torch.from_numpy(t[name + ".weight"]), None, stride=s, padding=k // 2)
    bn = importer._bn_prefix(name, kind)
    return F.batch_norm(y, torch.from_numpy(t[bn + ".running_mean"]), torch.from_numpy(t[bn + ".running_var"]),
                        torch.from_numpy(t[bn + ".weight"]), torch.from_numpy(t[bn + ".bias"]), False, 0.0, eps)


def test_reid_state_dict_import_matches_unfused_network(tmp_path):
    from oracle import nets
    ck = _unfused(W.reid_conv_specs(), W.KIND_REID, 3, 1e-5)
    ck["classifier.4.weight"] = np.zeros((751, 256), np.float32)  # ignored
    path = tmp_path / "ckpt.t7"
    torch.save({"net_dict": {k: torch.from_numpy(np.asarray(v)) for k, v in ck.items()}, "acc": 0.9}, path)
    blob = tmp_path / "reid.aicw"
    kind, params, out = importer.import_file(str(path), str(blob))
    assert kind == W.KIND_REID and len(out) == 2 * len(W.reid_conv_specs())
    net = nets.load_net(str(blob))
    x = torch.from_numpy(np.random.default_rng(0).normal(0, 1, (2, 3, 128, 64)).astype(np.float32))
    got = net.forward(x)

    def block(v, name, s):  # the unfused network, layer by layer (deep_sort_pytorch BasicBlock)
        y = F.relu(_conv_bn(v, ck, name + ".conv1", W.KIND_REID, 3, s, 1e-5))
        y = _conv_bn(y, ck, name + ".conv2", W.KIND_REID, 3, 1, 1e-5)
        if (name + ".downsample.0.weight") in ck:
            v = _conv_bn(v, ck, name + ".downsample.0", W.KIND_REID, 1, s, 1e-5)
        return F.relu(v + y)
    v = F.max_pool2d(F.relu(_conv_bn(x, ck, "conv.0", W.KIND_REID, 3, 1, 1e-5)), 3, 2, 1)
    for li in range(1, 5):
        v = block(v, "layer%d.0" % li, 2 if li > 1 else 1)
        v = block(v, "layer%d.1" % li, 1)
    v = F.avg_pool2d(v, (8, 4), 1).flatten(1)
    want = v / v.norm(p=2, dim=1, keepdim=True)
    assert torch.allclose(got, want, atol=2e-5), float((got - want).abs().max())


@pytest.mark.parametrize("scale", ["n", "s"])
def test_yolov8_onnx_import_named_and_unfused(tmp_path, scale):
    specs = W.yolov8_conv_specs(scale)
    ck = _unfused(specs, W.KIND_YOLOV8, 5, 1e-3)
    path = tmp_path / "yolo.onnx"
    importer.write_onnx_initializers(str(path), ck, use_float_data=("model.0.bn.weight", "model.22.cv2.0.2.bias"))
    read = importer.read_onnx_initializers(str(path))
    assert list(read) == list(ck) and all(np.array_equal(read[k], ck[k]) for k in ck)
    blob = tmp_path / "yolo.aicw"
    kind, params, out = importer.import_file(str(path), str(blob))
    D = W.yolov8_dims(scale)
    assert kind == W.KIND_YOLOV8 and params == D["c"] + [D["n_small"], D["n_large"], 80]
    k2, p2, back = W.read_blob(str(blob))
    assert k2 == kind and p2 == params and all(np.array_equal(back[n], out[n]) for n in out)
    # folded layers compute what conv + BatchNorm computes; the plain heads are copied
    x = torch.from_numpy(np.random.default_rng(1).normal(0, 1, (1, specs[1][1], 24, 24)).astype(np.float32))
    name, cin, cout, k, s, act = specs[1]
    got = F.conv2d(x, torch.from_numpy(back[name + ".weight"]), torch.from_numpy(back[name + ".bias"]), stride=s, padding=k // 2)
    assert torch.allclose(got, _conv_bn(x, ck, name, W.KIND_YOLOV8, k, s, 1e-3), atol=1e-5)
    assert np.array_equal(back["model.22.cv3.1.2.weight"], ck["model.22.cv3.1.2.weight"])
    assert np.array_equal(back["model.22.cv3.1.2.bias"], ck["model.22.cv3.1.2.bias"])


@pytest.mark.parametrize("nc", [1, 20, 601])
def test_yolov8_state_dict_import_at_class_count(tmp_path, nc):
    """A fine-tuned checkpoint carries its class count in model.22.cv3.0.2.weight: the blob header says nc, the class
    branch is cc = max(c3, min(nc, 100)) wide, and the oracle net gives (B, 8400, 64 + nc) head rows."""
    from oracle import nets
    specs = W.yolov8_conv_specs("n", nc)
    ck = _unfused(specs, W.KIND_YOLOV8, 11, 1e-3)
    path = tmp_path / "best.pt"
    torch.save({"model": {k: torch.from_numpy(np.asarray(v)) for k, v in ck.items()}}, path)
    blob = tmp_path / "yolo.aicw"
    kind, params, out = importer.import_file(str(path), str(blob))
    k2, p2, back = W.read_blob(str(blob))
    assert kind == k2 == W.KIND_YOLOV8 and p2 == params and params[7] == nc
    D = W.yolov8_dims("n", nc)
    cc = max(D["c"][2], min(nc, 100))  # c3 = 64: 64, 64, 100
    assert D["cc"] == cc
    for l, c in enumerate(D["c"][2:5]):
        assert back["model.22.cv3.%d.0.conv.weight" % l].shape == (cc, c, 3, 3)
        assert back["model.22.cv3.%d.1.conv.weight" % l].shape == (cc, cc, 3, 3)
        assert back["model.22.cv3.%d.2.weight" % l].shape == (nc, cc, 1, 1)
        assert back["model.22.cv3.%d.2.bias" % l].shape == (nc,)
        assert back["model.22.cv2.%d.2.weight" % l].shape == (64, D["cb"], 1, 1)
        assert np.array_equal(back["model.22.cv3.%d.2.weight" % l], ck["model.22.cv3.%d.2.weight" % l])
    x = torch.from_numpy(np.random.default_rng(2).normal(0, 1, (2, 3, 640, 640)).astype(np.float32))
    head = nets.load_net(str(blob)).head_flat(x)
    assert head.shape == (2, 8400, 64 + nc) and bool(torch.isfinite(head).all())


def test_fused_anonymous_onnx_is_matched_by_order(tmp_path):
    """Exports with Conv+BN fused rename the initialisers (onnx::Conv_<n>): layers are matched by order and shape."""
    kind, params, tensors = W.synth_yolov8_weights("n", seed=3)
    anon = OrderedDict()
    i = 100
    for name, cin, cout, k, s, act in W.yolov8_conv_specs("n"):
        anon["onnx::Conv_%d" % i] = tensors[name + ".weight"]
        anon["onnx::Conv_%d" % (i + 1)] = tensors[name + ".bias"]
        i += 3
    anon["/model.22/dfl/conv/Constant"] = np.arange(16, dtype=np.float32).reshape(1, 16, 1, 1)  # trailing non-layer initialiser
    path = tmp_path / "fused.onnx"
    importer.write_onnx_initializers(str(path), anon)
    k2, p2, out = importer.import_tensors(importer.read_onnx_initializers(str(path)))
    assert k2 == kind and p2 == params
    assert list(out) == list(tensors) and all(np.array_equal(out[n], tensors[n]) for n in tensors)
    # the ReID net the same way
    rk, rp, rt = W.synth_reid_weights(seed=2)
    anon = OrderedDict()
    for j, (name, *_r) in enumerate(W.reid_conv_specs()):
        anon["onnx::Conv_%d" % (2 * j)], anon["onnx::Conv_%d" % (2 * j + 1)] = rt[name + ".weight"], rt[name + ".bias"]
    k3, p3, out = importer.import_tensors(anon)
    assert k3 == rk and all(np.array_equal(out[n], rt[n]) for n in rt)


def test_import_errors(tmp_path):
    with pytest.raises(RuntimeError):
        importer.import_tensors({"model.0.conv.weight": np.zeros((16, 3, 3, 3), np.float32)})  # nothing to fold, layers missing
    bad = tmp_path / "x.onnx"
    bad.write_bytes(b"\x08\x08")
    with pytest.raises(RuntimeError):
        importer.read_onnx_initializers(str(bad))
