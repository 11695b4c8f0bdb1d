"""The convolution kernels under a device-side image count, as both engines run every layer (-m gpu).

The engines plan each launch for a capacity and read the number of images present (ReID crops, present frames) on the
device; every kernel clips its tile count there.  Per case, one set of buffers at the capacity runs the counts 1,
capacity - 1, capacity, the counts at which the raster (n (h + ext)(w + ext) padded positions, n ho wo output pixels)
ends 1 - 8 rows into, or 1 - 8 rows short of, a 128-, 256- or 512-row tile, and a few seeded ones.  Each run checks:

* images < n are bit-identical with the same images of the run at n = capacity (the plan depends on the capacity only
  and every accumulator row sums its K terms in a fixed order), and the run at the capacity matches torch fp32 on the
  same bf16-rounded operands (first and last image, and images whose rows meet a tile boundary);
* input and residual images >= n, border included, hold bf16 NaN: nothing below the count reads them into a stored
  value (junk accumulator rows of image n - 1's border do read image n, and the border must be stored as literal zeros);
* the output interior is pre-filled with a pattern: every interior position < n is overwritten;
* the zero border of a padded output stays exactly zero for every image up to the capacity;
* capacity -> small n -> larger n on the same buffers, with new inputs each time, equals fresh runs.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TILES = (128, 256, 512)
PATTERN = -31744.0  # exact in bf16 and far outside what a layer here can produce

# The ReID trunk (CTA pairs, weight-stationary 256-row tiles, image tiles, the 4-D stores of the stride-2 entry layers)
# in both border kinds, and the geometries of the randomised padded-convolution sweep (batches up to 300).
# name, H, W, cin, cout, k, s, act, res_mode, capacity
REID_CASES = [
    ("l1_64_pairs_ws", 64, 32, 64, 64, 3, 1, 2, 2, 300),
    ("l1_64_res1", 64, 32, 64, 64, 3, 1, 1, 1, 131),
    ("l2_128_pairs", 32, 16, 128, 128, 3, 1, 2, 2, 300),
    ("l2_64_to_128", 32, 16, 64, 128, 3, 1, 0, 0, 131),
    ("l2_128_to_64_res1", 32, 16, 128, 64, 3, 1, 1, 1, 131),
    ("l2_entry_s2_64_128", 64, 32, 64, 128, 3, 2, 2, 0, 300),
    ("l2_entry_1x1s2_64_128", 64, 32, 64, 128, 1, 2, 0, 0, 300),
    ("l3_entry_s2_128_256", 32, 16, 128, 256, 3, 2, 2, 0, 300),
    ("l3_entry_1x1s2_128_256", 32, 16, 128, 256, 1, 2, 0, 0, 300),
    ("l3_256_img_tiles", 16, 8, 256, 256, 3, 1, 2, 2, 300),
    ("l3_img_tiles_64_96_res1", 16, 8, 64, 96, 3, 1, 1, 1, 131),
    ("l3_img_tiles_128_64", 16, 8, 128, 64, 3, 1, 0, 0, 131),
    ("l4_entry_s2_256_512", 16, 8, 256, 512, 3, 2, 2, 0, 300),
    ("l4_entry_1x1s2_256_512", 16, 8, 256, 512, 1, 2, 0, 0, 300),
    ("l4_512", 8, 4, 512, 512, 3, 1, 2, 2, 300),
    ("l4_64_to_512_res1", 8, 4, 64, 512, 3, 1, 1, 1, 131),
]


def _sweep_cases(n=12, seed=20261019):
    """Seeded draws over the geometries of the randomised padded-convolution sweep: image tiles, 256-row tiles and pairs,
    the 4-D stores of the 1x1 stride-2 layers; capacities 1 - 300, either border kind."""
    geoms = [  # H, W, k, s, (cin choices), (cout choices)
        (16, 8, 3, 1, (64, 128, 256), (64, 96, 128, 256)),
        (64, 32, 3, 1, (64,), (64,)),
        (32, 16, 3, 1, (64, 128), (64, 128)),
        (8, 4, 3, 1, (64, 256), (64, 512)),
        (64, 32, 1, 2, (64,), (128,)), (32, 16, 1, 2, (128,), (256,)), (16, 8, 1, 2, (256,), (512,)),
        (64, 32, 3, 2, (64,), (128,)), (16, 8, 3, 2, (256,), (512,)),
    ]
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        H, W, k, s, cins, couts = geoms[int(rng.integers(len(geoms)))]
        cap = int(rng.choice([1, 2, 3, 5, 17, 40, 131, 300]))
        cin, cout = int(rng.choice(cins)), int(rng.choice(couts))
        act = int(rng.integers(0, 3))
        res_mode = int(rng.integers(0, 3)) if (k == 3 and s == 1) else 0
        kind = int(rng.integers(1, 3))
        name = "sweep%d_%dx%d_c%d_%d_k%ds%d_a%d_r%d_cap%d_kind%d" % (i, H, W, cin, cout, k, s, act, res_mode, cap, kind)
        out.append((name, H, W, cin, cout, k, s, act, res_mode, cap, kind))
    return out


SWEEP_CASES = _sweep_cases()

# YOLOv8 layers at the 640-input geometry, capacity 64 (unpadded: window, flat, im2col, the 2x2 window over the
# space-to-depth stem input, fp32 head outputs)
# name, H, W, cin, cout, k, s, act, res_mode, out_f32
YOLO_CASES = [
    ("yolo_win_160_c16_res1", 160, 160, 16, 16, 3, 1, 1, 1, False),
    ("yolo_win_80_c64", 80, 80, 64, 64, 3, 1, 1, 0, False),
    ("yolo_win_20_c128_res1", 20, 20, 128, 128, 3, 1, 1, 1, False),
    ("yolo_flat_160_48_32", 160, 160, 48, 32, 1, 1, 1, 0, False),
    ("yolo_flat_40_384_256", 40, 40, 384, 256, 1, 1, 1, 0, False),
    ("yolo_i2c_s2_160_32_64", 160, 160, 32, 64, 3, 2, 1, 0, False),
    ("yolo_i2c_s2_40_128_256", 40, 40, 128, 256, 3, 2, 1, 0, False),
    ("yolo_s2d_stem_640_3_16", 640, 640, 3, 16, 3, 2, 1, 0, False),
    ("yolo_s2d_320_16_32", 320, 320, 16, 32, 3, 2, 1, 0, False),
    ("yolo_head_f32_80_64", 80, 80, 64, 64, 1, 1, 0, 0, True),
    ("yolo_head_f32_20_80", 20, 20, 80, 80, 1, 1, 0, 0, True),
]
YOLO_CAPACITY = 64


def _geometry(H, W, k, s, kind):
    ho, wo = (H + 2 * (k // 2) - k) // s + 1, (W + 2 * (k // 2) - k) // s + 1
    lo, ext = ((1, 2) if kind == 1 else (0, 1)) if kind else (0, 0)
    return ho, wo, lo, ext


def _rasters(H, W, ho, wo, k, s, ext):
    """Raster rows per image the kernels tile: padded positions of a zero-bordered stride-1 layer, output pixels."""
    r = {ho * wo}
    if ext:
        r.add((ho + ext) * (wo + ext))
        if s == 1:
            r.add((H + ext) * (W + ext))
    return sorted(r)


def counts_for(cap, rows_per_image, seed):
    """1, cap - 1, cap, the counts whose raster ends 1 - 8 rows into / short of a tile, and three seeded ones."""
    out = {1, cap - 1, cap}
    boundary = set()
    for R in rows_per_image:
        for T in TILES:
            for r in range(1, 9):
                for want in (r, T - r):
                    for n in range(1, cap + 1):
                        if (n * R) % T == want:
                            boundary.add(n)
                            break
    out |= boundary
    rng = np.random.default_rng(seed)
    out |= {int(v) for v in rng.integers(1, cap + 1, 3)}
    return sorted(v for v in out if 1 <= v <= cap), sorted(boundary)


class Layer:
    """One convolution at a capacity, its device buffers, and the torch fp32 reference of chosen images."""

    def __init__(self, name, H, W, cin, cout, k, s, act, res_mode, cap, kind, out_f32=False):
        import gpu_util as G
        self.G = G
        self.name, self.H, self.W, self.cin, self.cout, self.k, self.s = name, H, W, cin, cout, k, s
        self.act, self.res_mode, self.cap, self.kind, self.out_f32 = act, res_mode, cap, kind, out_f32
        self.ho, self.wo, self.lo, self.ext = _geometry(H, W, k, s, kind)
        self.cpad = cin if kind else (4 if cin <= 4 else (cin + 7) // 8 * 8)
        self.seed = sum(map(ord, name)) * 7 + kind
        rng = np.random.default_rng(self.seed)
        self.w = G.bf16_round_np(rng.normal(0, 1.0 / np.sqrt(cin * k * k), (cout, cin, k, k)))
        self.b = rng.normal(0, 0.5, cout).astype(np.float32)
        dt = torch.float32 if out_f32 else torch.bfloat16
        e = self.ext
        self.x = torch.zeros((cap, H + e, W + e, self.cpad), dtype=torch.bfloat16, device=G.DEV)
        self.res = torch.zeros((cap, self.ho + e, self.wo + e, cout), dtype=torch.bfloat16, device=G.DEV) if res_mode else None
        self.out = torch.zeros((cap, self.ho + e, self.wo + e, cout), dtype=dt, device=G.DEV)
        self.n_dev = torch.zeros(1, dtype=torch.int32, device=G.DEV)
        interior = torch.zeros((cap, self.ho + e, self.wo + e, 1), dtype=torch.bool, device=G.DEV)
        interior[:, self.lo:self.lo + self.ho, self.lo:self.lo + self.wo] = True
        self.interior = interior

    def interior_of(self, t):
        return t[:, self.lo:self.lo + self.ho, self.lo:self.lo + self.wo]

    def fill(self, gen_seed):
        """New bf16 inputs (and residual) in every interior; the borders stay zero."""
        g = torch.Generator(device=self.G.DEV).manual_seed(gen_seed)
        xi = torch.randn((self.cap, self.H, self.W, self.cin), generator=g, device=self.G.DEV).to(torch.bfloat16)
        self.x.zero_()
        self.x[:, self.lo:self.lo + self.H, self.lo:self.lo + self.W, :self.cin] = xi
        if self.res is not None:
            ri = torch.randn((self.cap, self.ho, self.wo, self.cout), generator=g, device=self.G.DEV).to(torch.bfloat16)
            self.res.zero_()
            self.interior_of(self.res).copy_(ri)

    def poison(self, n):
        """Input and residual images >= n, border included, become bf16 NaN."""
        self.x[n:] = float("nan")
        if self.res is not None:
            self.res[n:] = float("nan")

    def prefill(self):
        """The interior of every output image holds PATTERN, the border zero."""
        self.out.zero_()
        self.interior_of(self.out).fill_(PATTERN)

    def run(self, n, out=None):
        G = self.G
        from ai_camera_b200._lib import ConvDesc, check, ptr
        out = self.out if out is None else out
        self.n_dev.fill_(n)
        w = np.ascontiguousarray(self.w)
        if self.kind:
            d = ConvDesc(self.cap, self.H, self.W, self.cin, self.cout, self.k, self.s, self.act, self.res_mode, 0, self.n_dev.data_ptr())
            check(G.lib().aicam_conv2d_padded(C.byref(d), ptr(self.x), ptr(w), ptr(self.b), ptr(self.res), ptr(out),
                                              self.kind, self.kind, None))
        else:
            G.conv2d(self.x, w, self.b, self.k, self.s, self.act, self.res, self.res_mode, self.out_f32, self.n_dev, out)
        G.sync()
        return out

    def check_against_torch(self, images):
        """Images of the last run (at the capacity) against torch fp32 on the same bf16-rounded operands."""
        idx = torch.tensor(sorted(images), dtype=torch.long, device=self.G.DEV)
        x = self.x[idx][:, self.lo:self.lo + self.H, self.lo:self.lo + self.W, :self.cin].float().cpu()
        y = F.conv2d(x.permute(0, 3, 1, 2), torch.from_numpy(self.w), torch.from_numpy(self.b), stride=self.s, padding=self.k // 2)
        if self.res_mode:
            r = self.interior_of(self.res)[idx].float().cpu().permute(0, 3, 1, 2)
        if self.res_mode == 2:
            y = y + r
        y = F.silu(y) if self.act == 1 else (F.relu(y) if self.act == 2 else y)
        if self.res_mode == 1:
            y = y + r
        want = y.permute(0, 2, 3, 1).numpy()
        got = self.interior_of(self.out)[idx].float().cpu().numpy()
        err = np.abs(got - want)
        tol = (2e-3 + 1e-3 * np.abs(want)) if self.out_f32 else (2e-2 + 1e-2 * np.abs(want))
        bad = err > tol
        assert not bad.any(), "%s: %d/%d elements off, max abs err %.4g at %s of images %s" % (
            self.name, bad.sum(), bad.size, err.max(), np.unravel_index(err.argmax(), err.shape), sorted(images))


def _sample_images(cap, rasters, boundary_counts):
    """First and last image, the image before a few boundary counts, images holding a tile boundary of the full raster."""
    s = {0, cap - 1}
    s |= {n - 1 for n in boundary_counts[::max(1, len(boundary_counts) // 6)]}
    for R in rasters:
        for T in TILES:
            for j in (1, 2, 3):
                s.add(min(cap - 1, j * T // R))
    return sorted(s)[:16]


def _exercise(L):
    rasters = _rasters(L.H, L.W, L.ho, L.wo, L.k, L.s, L.ext)
    counts, boundary = counts_for(L.cap, rasters, L.seed)
    cap = L.cap
    # the run at the capacity: reference of every smaller count, and checked against torch
    L.fill(L.seed)
    L.prefill()
    full = L.run(cap).clone()
    assert not (L.interior_of(full) == PATTERN).any(), "%s: an interior position was never written at n = capacity" % L.name
    if L.ext:
        assert not full[~L.interior.expand_as(full)].any(), "%s: the zero border was written" % L.name
    L.check_against_torch(_sample_images(cap, rasters, boundary))
    clean_x = L.x.clone()
    clean_r = L.res.clone() if L.res is not None else None
    for n in counts:
        L.x.copy_(clean_x)
        if clean_r is not None:
            L.res.copy_(clean_r)
        L.poison(n)
        L.prefill()
        got = L.run(n)
        head = got[:n]
        assert not torch.isnan(head).any(), "%s n=%d: NaN below the count (an image >= n was read)" % (L.name, n)
        assert not (L.interior_of(head) == PATTERN).any(), "%s n=%d: an interior position < n was not written" % (L.name, n)
        if not torch.equal(head, full[:n]):
            diff = (head != full[:n]).reshape(n, -1).any(1).nonzero().flatten().tolist()
            raise AssertionError("%s n=%d: images %s differ from the run at the capacity" % (L.name, n, diff[:8]))
        if L.ext:
            border = got[~L.interior.expand_as(got)]
            assert not border.any(), "%s n=%d: the zero border of an output image (< capacity) was written" % (L.name, n)
    # capacity -> small n -> larger n on the same buffers (no pre-fill), new inputs each time, against fresh runs
    small, large = (counts[1], counts[-2]) if len(counts) > 2 else (1, cap)
    for step, n in enumerate((cap, small, large)):
        L.fill(L.seed + 101 * (step + 1))
        got = L.run(n).clone()
        fresh = torch.zeros_like(L.out)
        L.run(cap, out=fresh)
        assert torch.equal(got[:n], fresh[:n]), "%s: count %d after %s differs from a fresh run" % (L.name, n, (cap, small, large)[:step])
        if L.ext:
            assert not got[~L.interior.expand_as(got)].any(), "%s: border written after the count changed to %d" % (L.name, n)
    return counts


@pytest.mark.parametrize("kind", [1, 2], ids=["symmetric", "shared"])
@pytest.mark.parametrize("case", REID_CASES, ids=[c[0] for c in REID_CASES])
def test_padded_conv_under_a_count(case, kind):
    name, H, W, cin, cout, k, s, act, res_mode, cap = case
    counts = _exercise(Layer(name, H, W, cin, cout, k, s, act, res_mode, cap, kind))
    print("%s kind %d: %d counts" % (name, kind, len(counts)))


@pytest.mark.parametrize("case", SWEEP_CASES, ids=[c[0] for c in SWEEP_CASES])
def test_padded_conv_sweep_under_a_count(case):
    name, H, W, cin, cout, k, s, act, res_mode, cap, kind = case
    _exercise(Layer(name, H, W, cin, cout, k, s, act, res_mode, cap, kind))


@pytest.mark.parametrize("case", YOLO_CASES, ids=[c[0] for c in YOLO_CASES])
def test_conv_under_a_count(case):
    name, H, W, cin, cout, k, s, act, res_mode, out_f32 = case
    counts = _exercise(Layer(name, H, W, cin, cout, k, s, act, res_mode, YOLO_CAPACITY, 0, out_f32))
    print("%s: %d counts" % (name, len(counts)))


def test_fallback_kernel_under_a_count():
    """conv_tc.cu clips its row count on the device too: the unpadded cases with every layer forced onto it (the switches
    are read once per process, hence the subprocess)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, AICAM_NO_WIN="1", AICAM_NO_S2D="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", "test_conv_under_a_count",
                        "-p", "no:cacheprovider"], env=env, capture_output=True, text=True, cwd=root)
    tail = (r.stdout + r.stderr)[-1500:]
    assert r.returncode == 0, tail
    assert "%d passed" % len(YOLO_CASES) in r.stdout, tail
