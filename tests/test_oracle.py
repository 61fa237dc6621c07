"""CPU tests that PIN the oracle: restatement (oracle/restate.py) == the reference's
cv2 call sequence (oracle/cv2_path.py) == golden hashes made from the unmodified
reference (tests/golden/golden.json) == values recorded from the unmodified reference
(tests/golden/reference_samples.npz)."""
import os

import cv2
import numpy as np
import pytest

from oracle import cv2_path as C
from oracle import restate as R
from tests.helpers import GOLD, NAMES, h16


def test_fixture_decode_hashes(fx):
    for k, v in fx.gold["decoded"].items():
        assert h16(fx.img(k)) == v, k
    assert h16(fx.car()) == fx.gold["car_padded"]


@pytest.mark.parametrize("name", NAMES)
def test_camera_tables_and_warps(fx, name):
    g = fx.geometry()
    K, D, H = fx.calib[name]
    gold = fx.gold["camera"][name]
    P, (um1, um2), (bm1, bm2) = R.camera_tables(K, D, H, g.FW, g.FH, g.BW, g.BH)
    assert (h16(um1), h16(um2)) == (gold["und_map1"], gold["und_map2"])
    assert (h16(bm1), h16(bm2)) == (gold["bev_map1"], gold["bev_map2"])
    d1, d2 = R.fisheye_map(K, D, P, 2560, 2048, running=False)   # closed form used by the GPU kernel
    assert (d1 == um1).all() and (d2 == um2).all()
    img = fx.img(name)
    u = R.remap_linear(img, um1, um2)
    assert h16(u) == gold["undistort"]
    assert h16(R.remap_linear(img, bm1, bm2)) == gold["raw2bev"]
    assert h16(R.warp_perspective_u8(u, H, 1000, 1000)) == gold["warp_undistort"]
    # live cv2 (covers NEAREST, which the reference never uses and has no golden hash)
    assert (R.remap_nearest(img, bm1, bm2) == cv2.remap(img, bm1, bm2, cv2.INTER_NEAREST)).all()
    assert (R.remap_nearest(img, bm1, None) == cv2.remap(img, bm1, None, cv2.INTER_NEAREST)).all()
    assert (R.warp_perspective_u8(u, H, 1000, 1000, nearest=True)
            == cv2.warpPerspective(u, H, (1000, 1000), flags=cv2.INTER_NEAREST)).all()


def test_masks(fx):
    g = fx.geometry()
    for n in NAMES:
        assert h16(C.plain_mask(n, g)) == fx.gold["mask_plain"][n]
        assert h16(R.blend_mask(n, g.BW, g.BH, g.CW, g.CH)) == fx.gold["mask_blend"][n]


def test_blend_mask_loop_small():
    """restate.blend_mask == the reference's pointPolygonTest loop, at a small odd size."""
    g = C.Geometry(BW=203, BH=177, CW=51, CH=77)
    for n in NAMES:
        assert (R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) == C.blend_mask_loop(n, g)).all(), n


def test_remap_random_maps_and_channels():
    rng = np.random.default_rng(5)
    for ch in (1, 3, 4):
        shape = (97, 131) if ch == 1 else (97, 131, ch)
        src = rng.integers(0, 256, shape, dtype=np.uint8)
        m1 = rng.integers(-5, 140, (60, 75, 2)).astype(np.int16)
        m2 = rng.integers(0, 1024, (60, 75)).astype(np.uint16)
        assert (R.remap_linear(src, m1, m2) == cv2.remap(src, m1, m2, cv2.INTER_LINEAR)).all()
        assert (R.remap_nearest(src, m1, m2) == cv2.remap(src, m1, m2, cv2.INTER_NEAREST)).all()


def test_luminance_and_color_balance(fx):
    F = fx.frames()
    for a, b in zip(C.luminance_balance(F), R.luminance_balance(F)):
        assert (a == b).all()
    assert R.luminance_offsets(F)[0] == [6, -1, -6, 0]
    for W in (1279, 70, 33, 31):   # rows whose tail (<32 px) takes OpenCV's rounding scalar path
        Fw = [np.ascontiguousarray(f[:19, :W]) for f in F]
        for a, b in zip(C.luminance_balance(Fw), R.luminance_balance(Fw)):
            assert (a == b).all(), W
    cv = np.random.default_rng(0).integers(0, 256, (300, 200, 3), dtype=np.uint8)
    assert (C.color_balance(cv.copy()) == R.color_balance(cv)).all()


def test_hsv_exhaustive_roundtrip():
    """BGR->HSV over a 2^18 colour lattice + all V offsets used; HSV->BGR over all (h,s,v)."""
    v = np.arange(0, 256, 4, dtype=np.uint8)
    lat = np.stack(np.meshgrid(v, v, v, indexing="ij"), -1).reshape(-1, 64, 3)
    assert (np.stack(R.bgr2hsv(lat), -1) == cv2.cvtColor(lat, cv2.COLOR_BGR2HSV)).all()
    h, s, vv = np.meshgrid(np.arange(180, dtype=np.uint8), np.arange(256, dtype=np.uint8),
                           np.arange(256, dtype=np.uint8), indexing="ij")
    hsv = np.stack([h, s, vv], -1).reshape(-1, 256, 3)
    assert (R.hsv2bgr(hsv[..., 0], hsv[..., 1], hsv[..., 2]) == cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)).all()


@pytest.mark.parametrize("blend", [False, True])
@pytest.mark.parametrize("balance", [False, True])
def test_native_bev_golden(fx, blend, balance):
    g = fx.geometry()
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if blend else C.plain_mask(n, g) for n in NAMES]
    ref = C.RefBev(fx.calib, g, blend, balance, masks=masks)
    gold = fx.gold["native"][f"blend{int(blend)}_balance{int(balance)}"]
    F = fx.frames()
    assert h16(ref(*F)) == gold["nocar"]
    assert h16(ref(*F, fx.car())) == gold["car"]
    # pure-NumPy restatement end to end
    maps = [c.bev_maps for c in ref.cameras]
    assert h16(R.bev_generate(F, maps, masks, blend, balance, fx.car())) == gold["car"]


@pytest.mark.parametrize("key,FW,FH,BW,BH,blend,balance,car", [
    ("cfg2_1280x960_1000_plain", 1280, 960, 1000, 1000, False, False, False),
    ("cfg3_1920x1080_1200_blend_balance_car", 1920, 1080, 1200, 1200, True, True, True),
    ("cfg4_1920x1080_1000_blend", 1920, 1080, 1000, 1000, True, False, False),
    ("odd_1000x750_777x900_blend_balance_car", 1000, 750, 777, 900, True, True, True),
])
def test_rescaled_configs_golden(fx, key, FW, FH, BW, BH, blend, balance, car):
    g = fx.geometry(FW, FH, BW, BH)
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if blend else C.plain_mask(n, g) for n in NAMES]
    ref = C.RefBev(fx.scaled_calib(g), g, blend, balance, masks=masks)
    out = ref(*fx.frames(FW, FH), fx.car(BW, BH) if car else None)
    assert h16(out) == fx.gold["cfg"][key]


def test_incalib_excalib_tools_golden(fx):
    K, D, _ = fx.calib["front"]
    raw0 = fx.img("raw0")
    P = C.dst_camera_matrix(K, 1280, 1024, 0.5, 1)
    m1, m2 = R.fisheye_map(K, D, P, 1280, 1024)
    gi = fx.gold["incalib_fisheye_raw0"]
    assert (h16(m1), h16(m2)) == (gi["map1"], gi["map2"])
    assert h16(R.remap_linear(raw0, m1, m2)) == gi["undistort"]
    K2 = np.diag([0.5, 480 / 1024, 1.0]) @ K
    small = cv2.resize(raw0, (640, 480), interpolation=cv2.INTER_LINEAR)
    m1, m2 = R.fisheye_map(K2, D, C.dst_camera_matrix(K2, 640, 480, 0.5, 1), 640, 480)
    assert h16(R.remap_linear(small, m1, m2)) == fx.gold["incalib_fisheye_raw0_640x480"]["undistort"]
    Kn = K * np.array([[2.0], [2.0], [1.0]])
    m1, m2 = R.pinhole_map(Kn, fx.D5, C.dst_camera_matrix(Kn, 1280, 1024, 0.5, 1), 1280, 1024)
    gn = fx.gold["incalib_normal_raw0"]
    assert (h16(m1), h16(m2)) == (gn["map1"], gn["map2"])
    assert h16(R.remap_linear(raw0, m1, m2)) == gn["undistort"]
    assert h16(R.warp_perspective_u8(fx.img("src_back"), fx.calib["back"][2], 1000, 1000)) == fx.gold["excalib_warp_back"]
    m1, m2 = R.fisheye_map(K, D, C.dst_camera_matrix(K, 1280, 1024, 1, 1), 1280, 1024)
    assert h16(R.remap_linear(fx.img("front"), m1, m2)) == fx.gold["tools_undistort_front"]


def test_live_unmodified_reference(fx):
    """The unmodified reference's own outputs (canvas and BEV maps at seeded pixels, recorded by
    oracle/gen_golden.py into tests/golden/reference_samples.npz) agree with the oracle, whose full outputs
    agree with the golden file."""
    z = np.load(os.path.join(GOLD, "reference_samples.npz"))
    idx = z["pixel_index"]
    g = fx.geometry()
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) for n in NAMES]
    ref = C.RefBev(fx.calib, g, True, True, masks=masks)
    out = ref(*fx.frames(), fx.car())
    assert h16(out) == fx.gold["native"]["blend1_balance1"]["car"]
    assert (out.reshape(-1, 3)[idx] == z["bev"]).all()
    for n, cam in zip(NAMES, ref.cameras):
        assert h16(cam.bev_maps[0]) == fx.gold["camera"][n]["bev_map1"]
        assert (cam.bev_maps[0].reshape(-1, 2)[idx] == z[f"bev_map1_{n}"]).all(), n


def test_blend_weight_integer_identity_exhaustive():
    """The kernel's integer blend weighting == BlendMask.__call__'s float expression
    (surroundBEV.py:279-280) for every (pixel, mask) pair."""
    px = np.arange(256, dtype=np.uint8)[None, :].repeat(256, 0)
    mask = np.arange(256, dtype=np.uint8)[:, None].repeat(256, 1)
    ref = (px[..., None] * (np.repeat(mask[:, :, None], 1, axis=2) / 255.0).astype(np.float32)).astype(np.uint8)[..., 0]
    wm = mask.astype(np.int64) * 257 + (mask != 0)
    assert ((px.astype(np.int64) * wm) >> 16 == ref).all()
    assert (R.apply_blend(np.stack([px] * 3, -1), mask)[..., 0] == ref).all()
