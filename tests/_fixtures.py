"""Shared helpers for the test-suite (fixtures under tests/golden)."""
import hashlib
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_DIR = os.path.join(HERE, "golden")


def golden(name="golden.json"):
    with open(os.path.join(GOLDEN_DIR, name)) as f:
        return json.load(f)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:32]


def out_digest(frame, text_box=(111, 620)):
    f = np.array(frame, copy=True)
    f[:text_box[0], :text_box[1]] = 0
    return sha(f)


def pix_digest(ly, lx, ry, rx):
    return sha(np.stack([np.asarray(ly), np.asarray(lx)]).astype(np.int64)) + ":" + \
        sha(np.stack([np.asarray(ry), np.asarray(rx)]).astype(np.int64))


def avg_xy_digest(t):
    return sha(np.concatenate([np.asarray(v, dtype=np.int64).ravel() for v in
                               (t.left_avg_y, t.left_avg_x, t.right_avg_y, t.right_avg_x)]))


def load_frame(name):
    """Decode a bundled test frame to RGB uint8 (cv2 is in the image; the decode
    is pinned by the 'frame' digest in golden.json)."""
    import cv2
    return cv2.cvtColor(cv2.imread(os.path.join(GOLDEN_DIR, "frames", name)), cv2.COLOR_BGR2RGB)


def frame_names():
    return sorted(golden()["images"].keys())
