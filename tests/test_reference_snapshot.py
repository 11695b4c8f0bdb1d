"""The REAL reference tracker against the oracle restatement (CPU) and against the device tracker (GPU), on fresh
seeds - the golden fixtures pin the same thing on recorded seeds only.

The reference runs from oracle/_ref, a snapshot of the original AI-Camera sources that ``python oracle/build_ref.py
<checkout of the original project>`` makes.  The sources are not part of this repository and no output of the
reference on these seeds is stored, so without the snapshot these tests skip."""
import numpy as np
import pytest

from golden_util import assert_same_tracking, run_oracle
from scenarios import make_scenario


def _ref():
    from oracle import ref_bridge
    if not ref_bridge.available():
        pytest.skip("needs oracle/_ref, a snapshot of the original AI-Camera sources (python oracle/build_ref.py "
                    "<checkout of the original project>); no recorded output replaces it")
    return ref_bridge


@pytest.mark.parametrize("seed,n_objects,n_frames,kw", [
    (711, 8, 50, {}), (712, 30, 25, dict(size_range=(30.0, 120.0))), (713, 5, 40, dict(tracker_kw=dict(nn_budget=3, max_age=3, n_init=2)))])
def test_oracle_equals_real_reference_fresh_seeds(seed, n_objects, n_frames, kw):
    rb = _ref()
    tkw = kw.pop("tracker_kw", {})
    frames = make_scenario(seed=seed, n_frames=n_frames, n_objects=n_objects, **kw)
    assert_same_tracking(run_oracle(frames, **tkw), rb.run_tracker_scenario(frames, tracker_kw=tkw), "seed %d" % seed)


def test_reference_image_ops_equal_oracle():
    rb = _ref()
    from oracle import image_ops
    from scenarios import synth_image
    ip = rb.import_reference()[1]
    rng = np.random.default_rng(5)
    for (h, w) in [(1080, 1920), (540, 960), (333, 517)]:
        img = synth_image(rng, h, w)
        a, ra, pa = ip.preprocess_yolo_input(img, (640, 640))
        b, rb_, pb = image_ops.preprocess_yolo_input(img)
        assert np.array_equal(a, b) and tuple(ra) == tuple(rb_) and tuple(pa) == tuple(pb)
    crop = synth_image(rng, 211, 97)
    assert np.array_equal(ip.preprocess_reid_input(crop, (128, 64))[0], image_ops.reid_batch(crop, [(0, 0, 97, 211)])[0])


@pytest.mark.gpu
@pytest.mark.parametrize("seed,n_objects,n_frames", [(721, 20, 40), (722, 80, 12)])
def test_device_tracker_equals_real_reference(seed, n_objects, n_frames):
    rb = _ref()
    import gpu_util as G
    frames = make_scenario(seed=seed, n_frames=n_frames, n_objects=n_objects, size_range=(30.0, 150.0))
    assert_same_tracking(G.run_gpu_tracker(frames), rb.run_tracker_scenario(frames), "seed %d" % seed)
