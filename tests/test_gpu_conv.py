"""tcgen05 implicit-GEMM convolution vs a PyTorch fp32 reference of the same op (-m gpu).

Operands are bf16 on the device; the reference convolves the same bf16-rounded values in fp32.
Tolerance: bf16 output rounding (2^-9 relative) plus fp32 accumulation-order noise."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

CASES = [
    # name, B, H, W, cin, cout, k, s, act, res_mode, out_f32
    ("1x1_16_32", 2, 20, 20, 16, 32, 1, 1, 1, 0, False),
    ("3x3_16_16_res1", 1, 24, 24, 16, 16, 3, 1, 1, 1, False),
    ("3x3s2_32_64", 2, 32, 32, 32, 64, 3, 2, 1, 0, False),
    ("stem_3_16", 2, 64, 64, 3, 16, 3, 2, 1, 0, False),
    ("stem_reid_3_64_s1", 3, 32, 16, 3, 64, 3, 1, 2, 0, False),
    ("cout80", 1, 20, 20, 64, 80, 3, 1, 1, 0, False),
    ("cout256_res2_relu", 5, 8, 4, 128, 256, 3, 1, 2, 2, False),
    ("cin48_1x1", 1, 40, 40, 48, 32, 1, 1, 1, 0, False),
    ("tail_7x9", 1, 7, 9, 32, 32, 3, 1, 1, 0, False),
    ("f32_out_1x1", 1, 20, 20, 64, 64, 1, 1, 0, 0, True),
    ("bigk_512", 4, 8, 4, 512, 512, 3, 1, 2, 0, False),
    ("1x1s2_down", 2, 16, 8, 64, 128, 1, 2, 0, 0, False),
    ("yolo_160_c32", 2, 160, 160, 32, 32, 3, 1, 1, 0, False),
    # unstaged epilogue: rows that are not a multiple of 16 bytes (Detect heads at class counts other than 80), stored
    # and, with a residual, read one channel at a time
    ("rows40B_3x3_20", 2, 20, 20, 32, 20, 3, 1, 1, 0, False),
    ("rows40B_1x1_20_res1", 2, 20, 20, 64, 20, 1, 1, 1, 1, False),
    ("rows200B_3x3_100_res1", 1, 20, 20, 100, 100, 3, 1, 1, 1, False),
    ("rows200B_1x1_100", 2, 20, 20, 100, 100, 1, 1, 1, 0, False),
    ("rows40B_3x3s2_20", 2, 33, 31, 32, 20, 3, 2, 1, 0, False),
    ("f32_rows4B_1x1_1", 2, 40, 40, 64, 1, 1, 1, 0, 0, True),
    ("f32_rows12B_1x1_3", 2, 20, 20, 100, 3, 1, 1, 0, 0, True),
    # window kernel (conv_win.cu): patch rasters with strips, every swizzle width, resident and
    # streamed weights, one and two accumulators per tile, residual modes, fp32 output
    ("win_reid_l1", 3, 64, 32, 64, 64, 3, 1, 2, 2, False),
    ("win_reid_l2", 3, 32, 16, 128, 128, 3, 1, 2, 2, False),
    ("win_c16_res1", 2, 40, 56, 16, 16, 3, 1, 1, 1, False),
    ("win_c32_wide", 1, 24, 200, 32, 32, 3, 1, 1, 0, False),
    ("win_80_80", 2, 20, 20, 80, 80, 3, 1, 1, 0, False),
    ("win_128_64_stream", 2, 40, 40, 128, 64, 3, 1, 1, 0, False),
    ("win_256_80_stream", 1, 20, 20, 256, 80, 3, 1, 1, 0, False),
    ("win_1x1_384_256", 2, 20, 20, 384, 256, 1, 1, 1, 0, False),
    ("win_1x1_48_32", 2, 40, 40, 48, 32, 1, 1, 1, 0, False),
    ("win_1x1_f32_80", 2, 40, 40, 80, 80, 1, 1, 0, 0, True),
    ("win_1x1_64_dfl_f32", 1, 80, 80, 64, 64, 1, 1, 0, 0, True),
    ("win_odd_13x17", 2, 13, 17, 64, 64, 3, 1, 1, 0, False),
    ("win_tall_300x9", 1, 300, 9, 32, 48, 3, 1, 2, 0, False),
    # im2col-TMA mode of the same kernel: stride 2, and 3x3 on maps too small for the window raster
    ("i2c_s2_64_128", 5, 64, 32, 64, 128, 3, 2, 2, 0, False),
    ("i2c_s2_odd_15x9", 3, 15, 9, 32, 32, 3, 2, 1, 0, False),
    ("i2c_s2_16_32_320", 1, 320, 320, 16, 32, 3, 2, 1, 0, False),
    ("i2c_1x1s2_256_512", 7, 16, 8, 256, 512, 1, 2, 0, 0, False),
    ("i2c_deep_256_res2", 9, 16, 8, 256, 256, 3, 1, 2, 2, False),
    ("i2c_deep_512_res2", 13, 8, 4, 512, 512, 3, 1, 2, 2, False),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_conv_matches_torch(case):
    import gpu_util as G
    name, B, H, W, cin, cout, k, s, act, res_mode, out_f32 = case
    rng = np.random.default_rng(abs(hash(name)) % (2 ** 31))
    cpad = 4 if cin <= 4 else (cin + 7) // 8 * 8
    x = G.bf16_round_np(rng.normal(0, 1, (B, H, W, cin)))
    xp = np.zeros((B, H, W, cpad), np.float32)
    xp[..., :cin] = x
    w = G.bf16_round_np(rng.normal(0, 1.0 / np.sqrt(cin * k * k), (cout, cin, k, k)))
    b = rng.normal(0, 0.5, cout).astype(np.float32)
    ho, wo = (H + 2 * (k // 2) - k) // s + 1, (W + 2 * (k // 2) - k) // s + 1
    res = G.bf16_round_np(rng.normal(0, 1, (B, ho, wo, cout))) if res_mode else None
    xd = torch.from_numpy(xp).to(G.DEV).to(torch.bfloat16)
    rd = torch.from_numpy(res).to(G.DEV).to(torch.bfloat16) if res_mode else None
    got = G.conv2d(xd, w, b, k, s, act, rd, res_mode, out_f32).float().cpu().numpy()

    y = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w), torch.from_numpy(b), stride=s,
                 padding=k // 2)
    r = torch.from_numpy(res).permute(0, 3, 1, 2) if res_mode else None
    if res_mode == 2:
        y = y + r
    y = F.silu(y) if act == 1 else (F.relu(y) if act == 2 else y)
    if res_mode == 1:
        y = y + r
    want = y.permute(0, 2, 3, 1).numpy()
    assert got.shape == want.shape
    err = np.abs(got - want)
    tol = 2e-2 + 1e-2 * np.abs(want) if not out_f32 else 2e-3 + 1e-3 * np.abs(want)
    bad = err > tol
    assert not bad.any(), "%s: %d/%d elements off, max abs err %.4g at %s (got %.5g want %.5g)" % (
        name, bad.sum(), bad.size, err.max(), np.unravel_index(err.argmax(), err.shape),
        got.flat[err.argmax()], want.flat[err.argmax()])


PADDED_CASES = [
    # name, B, H, W, cin, cout, k, s, act, res_mode, in_pad, out_pad
    # zero-bordered tensors (ReID layers 2-4): 3x3 stride 1 over the flat padded raster (conv_win.cu mode 4) ...
    ("pad_l2_128", 5, 32, 16, 128, 128, 3, 1, 2, 2, 1, 1),
    ("pad_l3_256", 9, 16, 8, 256, 256, 3, 1, 2, 2, 1, 1),
    ("pad_l3_256_nores", 3, 16, 8, 256, 256, 3, 1, 2, 0, 1, 1),
    # 16 x 8 maps take one image per tile (descriptor group stride = one raster row): narrower layers, act(conv) + res
    ("pad_16x8_64", 7, 16, 8, 64, 64, 3, 1, 1, 1, 1, 1),
    ("pad_16x8_128_to_96", 4, 16, 8, 128, 96, 3, 1, 2, 2, 1, 1),
    ("pad_l4_512", 13, 8, 4, 512, 512, 3, 1, 2, 2, 1, 1),
    ("pad_one_image", 1, 8, 4, 64, 64, 3, 1, 1, 1, 1, 1),
    ("pad_odd_13x7_c64_96", 4, 13, 7, 64, 96, 3, 1, 0, 0, 1, 1),
    # ... and the stride-2 layers that enter / leave the padded geometry (im2col mode)
    ("pad_out_s2_64_128", 5, 64, 32, 64, 128, 3, 2, 2, 0, 0, 1),
    ("pad_out_1x1s2_64_128", 5, 64, 32, 64, 128, 1, 2, 0, 0, 0, 1),
    ("pad_inout_s2_128_256", 7, 32, 16, 128, 256, 3, 2, 2, 0, 1, 1),
    ("pad_inout_1x1s2_256_512", 7, 16, 8, 256, 512, 1, 2, 0, 0, 1, 1),
    ("pad_in_s2_odd_15x9", 3, 15, 9, 32, 32, 3, 2, 1, 0, 1, 0),
]


@pytest.mark.parametrize("kind", [1, 2], ids=["symmetric", "shared"])
@pytest.mark.parametrize("case", PADDED_CASES, ids=[c[0] for c in PADDED_CASES])
def test_padded_conv_matches_torch(case, kind):
    """Same operator over zero-bordered tensors (border kind 1: [h+2][w+2] interior at (1,1); kind 2: shared border,
    [h+1][w+1] interior at (0,0)); the output border must stay exactly zero."""
    import ctypes as C
    import gpu_util as G
    from ai_camera_b200._lib import ConvDesc, check, ptr
    name, B, H, W, cin, cout, k, s, act, res_mode, ipad, opad = case
    ipad, opad = ipad * kind, opad * kind
    lo, ext = (1, 2) if kind == 1 else (0, 1)
    rng = np.random.default_rng(abs(hash(name)) % (2 ** 31))
    x = G.bf16_round_np(rng.normal(0, 1, (B, H, W, cin)))
    w = G.bf16_round_np(rng.normal(0, 1.0 / np.sqrt(cin * k * k), (cout, cin, k, k)))
    b = rng.normal(0, 0.5, cout).astype(np.float32)
    ho, wo = (H + 2 * (k // 2) - k) // s + 1, (W + 2 * (k // 2) - k) // s + 1
    res = G.bf16_round_np(rng.normal(0, 1, (B, ho, wo, cout))) if res_mode else None

    def padded(a, on):
        return np.pad(a, ((0, 0), (lo, ext - lo), (lo, ext - lo), (0, 0))) if on else a

    xd = torch.from_numpy(padded(x, ipad)).to(G.DEV).to(torch.bfloat16).contiguous()
    rd = torch.from_numpy(padded(res, opad)).to(G.DEV).to(torch.bfloat16).contiguous() if res_mode else None
    oe = ext if opad else 0
    out = torch.zeros((B, ho + oe, wo + oe, cout), dtype=torch.bfloat16, device=G.DEV)
    d = ConvDesc(B, H, W, cin, cout, k, s, act, res_mode, 0)
    check(G.lib().aicam_conv2d_padded(C.byref(d), ptr(xd), ptr(np.ascontiguousarray(w)), ptr(b), ptr(rd), ptr(out),
                                      ipad, opad, None))
    got = out.float().cpu().numpy()
    if opad:
        border = got.copy()
        border[:, lo:lo + ho, lo:lo + wo, :] = 0
        assert not border.any(), "%s: the zero border was written" % name
        got = got[:, lo:lo + ho, lo:lo + wo, :]
    y = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w), torch.from_numpy(b), stride=s,
                 padding=k // 2)
    r = torch.from_numpy(res).permute(0, 3, 1, 2) if res_mode else None
    if res_mode == 2:
        y = y + r
    y = F.silu(y) if act == 1 else (F.relu(y) if act == 2 else y)
    if res_mode == 1:
        y = y + r
    want = y.permute(0, 2, 3, 1).numpy()
    assert got.shape == want.shape
    err = np.abs(got - want)
    bad = err > 2e-2 + 1e-2 * np.abs(want)
    assert not bad.any(), "%s: %d/%d elements off, max abs err %.4g at %s (got %.5g want %.5g)" % (
        name, bad.sum(), bad.size, err.max(), np.unravel_index(err.argmax(), err.shape),
        got.flat[err.argmax()], want.flat[err.argmax()])


@pytest.mark.parametrize("shape", [(3, 128, 64), (2, 24, 40), (5, 6, 2)], ids=["reid_128x64", "odd_tiles_24x40", "tiny_6x2"])
def test_fused_stem_pool_matches_torch(shape):
    """stem_pool.cu: conv3x3(3->64) + bias + ReLU + maxpool(3, s2, p1) fused, vs torch fp32 on the same
    bf16-rounded operands.  The conv output is rounded to bf16 before pooling; max commutes with rounding."""
    import ctypes as C
    import gpu_util as G
    from ai_camera_b200._lib import check, ptr
    n, H, W = shape
    rng = np.random.default_rng(n * 1000 + H)
    x = G.bf16_round_np(rng.normal(0, 1, (n, H, W, 3)))
    xp = np.zeros((n, H, W, 4), np.float32)
    xp[..., :3] = x
    w = G.bf16_round_np(rng.normal(0, 1.0 / np.sqrt(27), (64, 3, 3, 3)))
    b = rng.normal(0, 0.5, 64).astype(np.float32)
    xd = torch.from_numpy(xp).to(G.DEV).to(torch.bfloat16)
    out = torch.empty((n, H // 2, W // 2, 64), dtype=torch.bfloat16, device=G.DEV)
    check(G.lib().aicam_reid_stem_pool(ptr(xd), n, H, W, ptr(np.ascontiguousarray(w)), ptr(b), ptr(out), None))
    got = out.float().cpu().numpy()
    y = F.relu(F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w), torch.from_numpy(b), padding=1))
    want = F.max_pool2d(y, 3, 2, 1).permute(0, 2, 3, 1).numpy()
    assert got.shape == want.shape
    err = np.abs(got - want)
    bad = err > 2e-2 + 1e-2 * np.abs(want)
    assert not bad.any(), "%d/%d elements off, max abs err %.4g at %s" % (
        bad.sum(), bad.size, err.max(), np.unravel_index(err.argmax(), err.shape))
