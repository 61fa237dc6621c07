"""Generate tests/golden/{fixtures.npz,golden.json,reference_samples.npz} from the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY.  Run in the build container (where /root/reference
exists):  ``python -m oracle.gen_golden``.  It imports the reference's own
classes (oracle/ref_loader.py shims only argv / pointPolygonTest / np.load),
runs them on the reference's own data/ images and records

  * fixtures.npz -- the INPUTS the GPU box needs but cannot read from
    /root/reference: K, D, H of the four cameras (float64) and the encoded JPEG
    bytes of the fixture frames (decoded with cv2.imdecode at test time; same
    libjpeg-turbo in the same image => same pixels; the decoded-pixel hashes are
    recorded too so a decoder change is detected);
  * golden.json  -- SHA-256 prefixes (16 hex) of every output of the reference on
    those inputs: maps, masks, per-camera warps, BevGenerator at all flag
    combinations and at the rescaled configs of BASELINE.json;
  * reference_samples.npz -- values of the reference's BevGenerator(blend=True,
    balance=True) canvas (with car) and of each camera's BEV map at a fixed, seeded
    set of canvas pixels, so that tests compare against the reference's own numbers
    without the reference being installed.
"""
from __future__ import annotations

import hashlib
import json
import os
import runpy
import sys
import tempfile

import cv2
import numpy as np

from . import ref_loader as RL
from .cv2_path import padding

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
NAMES = ("front", "back", "left", "right")


def h16(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def main():
    assert RL.available(), "/root/reference is required to (re)generate golden vectors"
    os.makedirs(OUT, exist_ok=True)
    sb = RL.REF + "/SurroundBirdEyeView/data/"
    fx, gold = {}, {"decoded": {}, "cv2": cv2.__version__, "numpy": np.__version__}

    def add_jpeg(key, path):
        raw = np.fromfile(path, np.uint8)
        fx["jpg_" + key] = raw
        img = cv2.imdecode(raw, cv2.IMREAD_COLOR)
        assert (img == cv2.imread(path)).all()
        gold["decoded"][key] = h16(img)
        return img

    frames = {n: add_jpeg(n, sb + f"{n}/{n}.jpg") for n in NAMES}
    car_small = add_jpeg("car", sb + "car.jpg")
    raw0 = add_jpeg("raw0", RL.REF + "/IntrinsicCalibration/data/img_raw0.jpg")
    src_back = add_jpeg("src_back", RL.REF + "/ExtrinsicCalibration/data/img_src_back.jpg")
    for n in NAMES:
        for k in "KDH":
            fx[f"{k}_{n}"] = np.load(sb + f"{n}/camera_{n}_{k}.npy")

    # ---- native geometry: per-camera tables and warps (SURVEY App. B table 1) ----
    m = RL.surround()
    bev = RL.make_bev()
    cams = {}
    for n, cam in zip(NAMES, bev.cameras):
        u = cam.undistort(frames[n])
        cams[n] = {
            "und_map1": h16(cam.undistort_maps[0]), "und_map2": h16(cam.undistort_maps[1]),
            "bev_map1": h16(cam.bev_maps[0]), "bev_map2": h16(cam.bev_maps[1]),
            "undistort": h16(u), "raw2bev": h16(cam.raw2bev(frames[n])),
            "warp_undistort": h16(cam.warp_homography(u)),
        }
    gold["camera"] = cams
    gold["mask_plain"] = {n: h16(mk.mask) for n, mk in zip(NAMES, bev.masks)}
    car = m.padding(car_small, 1000, 1000)
    assert (car == padding(car_small, 1000, 1000)).all()
    gold["car_padded"] = h16(car)
    F = [frames[n] for n in NAMES]
    native = {}
    for blend in (False, True):
        for balance in (False, True):
            b = RL.make_bev(blend=blend, balance=balance)
            if blend:
                gold["mask_blend"] = {n: h16(mk.mask) for n, mk in zip(NAMES, b.masks)}
            native[f"blend{int(blend)}_balance{int(balance)}"] = {
                "nocar": h16(b(*F)), "car": h16(b(*F, car))}
    gold["native"] = native
    gold["main_py_variant"] = h16(RL.make_bev(CW=200, CH=350, blend=True, balance=True)(*F))  # main.py:79-84

    # ---- rescaled configs (SURVEY 8d) ----
    def resized(FW, FH):
        return [cv2.resize(f, (FW, FH), interpolation=cv2.INTER_LINEAR) for f in F]

    def cfg(FW, FH, BW, BH, blend, balance, with_car):
        CW, CH = int(250 * BW / 1000), int(400 * BH / 1000)
        b = RL.make_bev(FW, FH, BW, BH, CW, CH, blend=blend, balance=balance)
        c = m.padding(cv2.resize(car_small, (CW, CH)), BW, BH) if with_car else None
        return h16(b(*resized(FW, FH), c)) if with_car else h16(b(*resized(FW, FH)))

    gold["cfg"] = {
        "cfg2_1280x960_1000_plain": cfg(1280, 960, 1000, 1000, False, False, False),
        "cfg3_1920x1080_1200_blend_balance": cfg(1920, 1080, 1200, 1200, True, True, False),
        "cfg3_1920x1080_1200_blend_balance_car": cfg(1920, 1080, 1200, 1200, True, True, True),
        "1920x1080_1200_plain": cfg(1920, 1080, 1200, 1200, False, False, False),
        "cfg4_1920x1080_1000_blend": cfg(1920, 1080, 1000, 1000, True, False, False),
        "odd_1000x750_777x900_blend_balance_car": cfg(1000, 750, 777, 900, True, True, True),
        "cfg5size_3840x2160_2000_blend_balance": cfg(3840, 2160, 2000, 2000, True, True, False),
    }

    # ---- InCalibrator.undistort with injected front K,D (intrinsicCalib.py:193-195) ----
    ic = RL.intrinsic()
    a = ic.InCalibrator.get_args()
    a.FRAME_WIDTH, a.FRAME_HEIGHT, a.FOCAL_SCALE, a.SIZE_SCALE = 1280, 1024, 0.5, 1
    cal = ic.InCalibrator("fisheye")
    cal.camera.data.camera_mat = fx["K_front"]
    cal.camera.data.dist_coeff = fx["D_front"]
    cal.camera._get_undistort_maps()
    gold["incalib_fisheye_raw0"] = {"map1": h16(cal.camera.data.map1), "map2": h16(cal.camera.data.map2),
                                    "undistort": h16(cal.undistort(raw0))}
    # cfg1(b): 640x480 (BASELINE configs[0]); K rows scaled by (0.5, 480/1024)
    small = cv2.resize(raw0, (640, 480), interpolation=cv2.INTER_LINEAR)
    a.FRAME_WIDTH, a.FRAME_HEIGHT = 640, 480
    cal2 = ic.InCalibrator("fisheye")
    cal2.camera.data.camera_mat = np.diag([0.5, 480 / 1024, 1.0]) @ fx["K_front"]
    cal2.camera.data.dist_coeff = fx["D_front"]
    cal2.camera._get_undistort_maps()
    gold["incalib_fisheye_raw0_640x480"] = {"undistort": h16(cal2.undistort(small))}
    # pinhole ('normal') maps with a synthetic 5-coefficient vector (intrinsicCalib.py:158-163)
    a.FRAME_WIDTH, a.FRAME_HEIGHT = 1280, 1024
    d5 = np.array([[-0.28, 0.09, 0.0007, -0.0004, -0.014]])
    fx["D5_synth"] = d5
    caln = ic.InCalibrator("normal")
    caln.camera.data.camera_mat = fx["K_front"] * np.array([[2.0], [2.0], [1.0]])
    caln.camera.data.dist_coeff = d5
    caln.camera._get_undistort_maps()
    gold["incalib_normal_raw0"] = {"map1": h16(caln.camera.data.map1), "map2": h16(caln.camera.data.map2),
                                   "undistort": h16(caln.undistort(raw0))}

    # ---- ExCalibrator.warp (extrinsicCalib.py:166-169) with the shipped back H ----
    ec = RL.extrinsic()
    ex = ec.ExCalibrator()
    ex.src_img, ex.homography = src_back, fx["H_back"]
    ex.dst_img = np.zeros((1000, 1000, 3), np.uint8)
    gold["excalib_warp_back"] = h16(ex.warp())

    # ---- Tools/undistort.py main(), unmodified, through a temp dir (png = lossless) ----
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(td + "/in"), os.makedirs(td + "/out")
        np.save(td + "/K.npy", fx["K_front"]), np.save(td + "/D.npy", fx["D_front"])
        cv2.imwrite(td + "/in/front.png", frames["front"])
        argv = sys.argv
        sys.argv = ["undistort.py", "-path_read", td + "/in/", "-path_save", td + "/out/", "-path_k", td + "/K.npy",
                    "-path_d", td + "/D.npy", "-srcformat", "png", "-dstformat", "png", "-quality", "1"]
        try:
            runpy.run_path(RL.REF + "/Tools/undistort.py", run_name="__main__")
        finally:
            sys.argv = argv
        gold["tools_undistort_front"] = h16(cv2.imread(td + "/out/front.png"))

    np.savez(os.path.join(OUT, "fixtures.npz"), **fx)
    with open(os.path.join(OUT, "golden.json"), "w") as f:
        json.dump(gold, f, indent=1, sort_keys=True)
    print(json.dumps(gold, indent=1, sort_keys=True))
    write_reference_samples(F, car)


def write_reference_samples(frames, car, n_pixels=4096, seed=2024):
    """tests/golden/reference_samples.npz: the reference's blended, balanced canvas (with car) and every camera's BEV
    map (map1: integer source coordinates) at n_pixels canvas pixels drawn with a fixed seed."""
    b = RL.make_bev(blend=True, balance=True)
    bev = b(*frames, car)
    idx = np.sort(np.random.default_rng(seed).choice(bev.shape[0] * bev.shape[1], n_pixels, replace=False)).astype(np.int32)
    out = {"pixel_index": idx, "bev": bev.reshape(-1, 3)[idx]}
    for n, cam in zip(NAMES, b.cameras):
        out[f"bev_map1_{n}"] = cam.bev_maps[0].reshape(-1, 2)[idx]
    np.savez_compressed(os.path.join(OUT, "reference_samples.npz"), **out)


if __name__ == "__main__":
    main()
