"""SURVEY.md section 8 row f-3: the ORB oracle (oracle/orb_oracle.py) pinned to OpenCV -- the committed cv2 goldens of a real crazyhorse
image (tests/golden/orb_golden.npz, make_orb.py) and cv2 itself on synthetic images: key points (all six fields, OpenCV's order) and
descriptors bit for bit, plus every stage on its own."""
import zlib

import numpy as np
import pytest

from orb_util import CASES, real_gray

from oracle import orb_oracle as O


@pytest.fixture(scope="module")
def gold(golden):
    return golden("orb_golden.npz")


def test_real_image_matches_cv2_golden(gold):
    g = real_gray()
    kp, desc = O.detect_and_compute(g, 5000)
    assert np.array_equal(kp, gold["kp_5000"]) and np.array_equal(desc, gold["desc_5000"])
    kp, desc = O.detect_and_compute(g, 1000)
    assert np.array_equal(kp, gold["kp_1000"]) and np.array_equal(desc, gold["desc_1000"])
    y0, y1, x0, x1 = gold["crop_rect"]
    kp, desc = O.detect_and_compute(np.ascontiguousarray(g[y0:y1, x0:x1]), 5000)
    assert np.array_equal(kp, gold["kp_crop"]) and np.array_equal(desc, gold["desc_crop"])


def test_real_image_is_the_cfg1_image(gold, golden):
    """The descriptors the cfg-1 matching goldens were made from (cfg1_crazyhorse.npz, cv2 on the BGR image) are these."""
    c1 = golden("cfg1_crazyhorse.npz")
    assert np.array_equal(c1["desc_0"], gold["desc_5000"]) and np.array_equal(c1["pts_0"], gold["kp_5000"][:, :2])


def test_stages_against_cv2_golden(gold):
    g = real_gray()
    assert np.array_equal(O.to_gray(gold["bgr_patch"]), gold["gray_patch"])
    imgs = O.pyramid(g)
    for l in range(1, 8):
        w, h, crc = gold["pyramid_crc"][l - 1]
        assert imgs[l].shape == (h, w) and zlib.crc32(imgs[l].tobytes()) == crc
    xs, ys, sc = O.fast_detect(g)
    assert np.array_equal(np.stack([xs, ys, sc], 1), gold["fast0"])
    assert np.array_equal(O.gaussian_kernel_7_2(), gold["gauss_kernel"])
    assert zlib.crc32(O.gaussian_blur_orb(g).tobytes()) == int(gold["blur0_crc"])
    yx = gold["atan_yx"]
    assert np.array_equal(O.fast_atan2(yx[:, 0], yx[:, 1]), gold["atan_deg"])
    assert O.umax_table() == [15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3]


@pytest.mark.parametrize("name,make,nf", CASES, ids=[c[0] for c in CASES])
def test_oracle_equals_cv2(name, make, nf):
    cv2 = pytest.importorskip("cv2")
    img = make()
    rk, rd = O.cv2_detect_and_compute(img, nf)
    kp, desc = O.detect_and_compute(img, nf)
    assert kp.shape == rk.shape and np.array_equal(kp, rk), name
    assert np.array_equal(desc, rd), name


def test_retain_best_keeps_ties_and_order():
    r = np.array([5, 7, 7, 3, 9, 7, 1, 7], np.float32)
    o = O.retain_best(r, 3)                      # threshold response 7: all four 7s stay
    assert sorted(r[o].tolist(), reverse=True) == [9, 7, 7, 7, 7]
    assert len(O.retain_best(r, 0)) == 0 and np.array_equal(O.retain_best(r, 20), np.arange(8))


def test_all_seven_crazyhorse_images_reproduce_the_cfg1_goldens(golden):
    """The oracle on each of the 7 original crazyhorse photographs gives exactly what cv2's ORB(5000) gave on it.  The photographs
    are too large to store, so each is represented by a fixed 112 x 144 grey window around its cfg-1 key points
    (orb_crazyhorse_crops.npz, make_orb_crops.py); image 0 in full is covered by the two tests above.  The window of image 0 is
    cut from the stored full grey image, which ties the windows to the photographs the cfg-1 goldens were made from."""
    cr = golden("orb_crazyhorse_crops.npz")
    assert len(cr["files"]) == 7 and list(cr["files"]) == list(golden("cfg1_crazyhorse.npz")["files"])
    y0, y1, x0, x1 = cr["rects"][0]
    assert np.array_equal(real_gray()[y0:y1, x0:x1], cr["gray_0"])
    for i in range(7):
        kp, desc = O.detect_and_compute(cr[f"gray_{i}"], 5000)
        assert len(kp) > 150 and len(np.unique(kp[:, 5])) >= 3, cr["files"][i]
        assert np.array_equal(kp, cr[f"kp_{i}"]) and np.array_equal(desc, cr[f"desc_{i}"]), cr["files"][i]
