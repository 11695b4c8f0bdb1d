"""Constants of the hot path, same names and values as the reference's ``src/config.py``
(:12-32, :36-53).  The engine paths name flat weight blobs (".aicw", see weights.py) instead
of serialized TensorRT engines."""
from pathlib import Path

PROJECT_ROOT = Path(__file__).resolve().parent.parent

YOLO_ENGINE_PATH = PROJECT_ROOT / "models/detection/yolov8n.aicw"
REID_ENGINE_PATH = PROJECT_ROOT / "models/reid/deepsort_reid.aicw"

YOLO_INPUT_SHAPE = (640, 640)
YOLO_CONF_THRESHOLD = 0.3
YOLO_NMS_THRESHOLD = 0.5
YOLO_TOPK = 100            # detections returned per frame by the engine's NMS
YOLO_MAX_CANDIDATES = 1024  # pre-NMS candidates per frame

DEEPSORT_MAX_DIST = 0.2
DEEPSORT_MIN_CONFIDENCE = 0.3
DEEPSORT_NMS_MAX_OVERLAP = 1.0
DEEPSORT_MAX_IOU_DISTANCE = 0.7
DEEPSORT_MAX_AGE = 70
DEEPSORT_N_INIT = 3
DEEPSORT_NN_BUDGET = 100

REID_INPUT_SHAPE = (128, 64)

CLASSES = (
    'person', 'bicycle', 'car', 'motorcycle', 'airplane', 'bus', 'train', 'truck', 'boat',
    'traffic light', 'fire hydrant', 'stop sign', 'parking meter', 'bench', 'bird', 'cat',
    'dog', 'horse', 'sheep', 'cow', 'elephant', 'bear', 'zebra', 'giraffe', 'backpack',
    'umbrella', 'handbag', 'tie', 'suitcase', 'frisbee', 'skis', 'snowboard', 'sports ball',
    'kite', 'baseball bat', 'baseball glove', 'skateboard', 'surfboard', 'tennis racket',
    'bottle', 'wine glass', 'cup', 'fork', 'knife', 'spoon', 'bowl', 'banana', 'apple',
    'sandwich', 'orange', 'broccoli', 'carrot', 'hot dog', 'pizza', 'donut', 'cake', 'chair',
    'couch', 'potted plant', 'bed', 'dining table', 'toilet', 'tv', 'laptop', 'mouse',
    'remote', 'keyboard', 'cell phone', 'microwave', 'oven', 'toaster', 'sink',
    'refrigerator', 'book', 'clock', 'vase', 'scissors', 'teddy bear', 'hair drier',
    'toothbrush'
)

CLASSES_TO_TRACK = {'person', 'car', 'bus', 'truck', 'motorcycle'}


def tracked_class_mask(classes=None):
    """(lo, hi) 64-bit masks of the COCO ids whose name is in ``classes`` (default CLASSES_TO_TRACK)."""
    classes = CLASSES_TO_TRACK if classes is None else classes
    lo = hi = 0
    for i, n in enumerate(CLASSES):
        if n in classes:
            if i < 64:
                lo |= 1 << i
            else:
                hi |= 1 << (i - 64)
    return lo, hi


# ---- visualisation (src/config.py:55-85) ----------------------------------------------------------------------------
# The reference draws one random BGR colour per class name, re-drawn at every start (its seed line is commented out,
# src/config.py:57); here the table is drawn once from a fixed seed so that runs - and overlay parity tests - agree.
def _class_colors():
    import random
    rng = random.Random(42)
    return {name: [rng.randint(0, 255) for _ in range(3)] for name in CLASSES}


CLASS_COLORS = _class_colors()
DEFAULT_TRACK_COLOR = (0, 255, 0)
FONT = 0                 # cv2.FONT_HERSHEY_SIMPLEX
FONT_SCALE_ID = 0.7
FONT_SCALE_INFO = 0.9
FONT_THICKNESS = 2
DEFAULT_OUTPUT_FPS = 30


def get_track_color(class_name):
    return CLASS_COLORS.get(class_name, DEFAULT_TRACK_COLOR)


def get_class_color(class_name):
    return CLASS_COLORS.get(class_name, (200, 200, 200))
