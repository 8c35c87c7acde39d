"""tests/golden/make_orb_crops.py -- a fixed sample of the seven crazyhorse images (BASELINE configs[0]) with what OpenCV's ORB
returns on it, so that the ORB oracle can be checked on every one of the original photographs without them.

    python tests/golden/make_orb_crops.py <crazyhorse dataset directory>     (the directory holding the 7 *.JPG files)

The photographs (3 MB) do not travel with the repository.  Each is decoded like cv::imread (B,G,R), converted with
cvtColor(BGR2GRAY) -- what ORB does first with a colour image -- and cut to a 112 x 144 window centred on the median of that
image's cfg-1 key points (cfg1_crazyhorse.npz pts_i), where the textured object is; the window still has key points on pyramid
levels 0..3.  The key points [n, 6] (x, y, size, angle, response, octave) and descriptors are those of
`ORB::create(5000)->detectAndCompute` (the original's call) on each window, through the cv2 binding.

Writes orb_crazyhorse_crops.npz: files [7], rects [7, 4] (y0, y1, x0, x1), gray_i, kp_i, desc_i, cv2_version.
"""
import glob
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
H, W = 112, 144

files = sorted(glob.glob(os.path.join(sys.argv[1], "*.JPG")))
assert len(files) == 7, files
c1 = np.load(os.path.join(HERE, "cfg1_crazyhorse.npz"))
assert [os.path.basename(f) for f in files] == list(c1["files"]), c1["files"]
out = {"cv2_version": cv2.__version__, "files": np.array([os.path.basename(f) for f in files])}
rects = []
for i, f in enumerate(files):
    gray = cv2.cvtColor(cv2.imread(f), cv2.COLOR_BGR2GRAY)
    cx, cy = np.median(c1[f"pts_{i}"], 0)
    x0 = int(np.clip(round(cx) - W // 2, 0, gray.shape[1] - W)); y0 = int(np.clip(round(cy) - H // 2, 0, gray.shape[0] - H))
    g = np.ascontiguousarray(gray[y0:y0 + H, x0:x0 + W])
    k, d = cv2.ORB_create(5000).detectAndCompute(g, None)
    out[f"gray_{i}"] = g
    out[f"kp_{i}"] = np.array([(p.pt[0], p.pt[1], p.size, p.angle, p.response, p.octave) for p in k], np.float32).reshape(-1, 6)
    out[f"desc_{i}"] = d
    rects.append((y0, y0 + H, x0, x0 + W))
out["rects"] = np.array(rects, np.int32)
np.savez_compressed(os.path.join(HERE, "orb_crazyhorse_crops.npz"), **out)
print({k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items()})
