"""The kernels' arithmetic, unit-tested on the CPU.  tests/host/kernel_math.cu includes the __host__ __device__
helpers of the CUDA sources and (a) checks the packed integer forms (interp_fast, sat_add_bgr, tile_row_word, lane_*)
against the scalar definitions of cv2.remap / BlendMask / cv2.add, (b) runs the FP64 coordinate code
(undistort_point, quantise_uv, warp_point, the closed-form 3x3 inverse) over whole maps, compared here with live cv2.
nvcc compiles it; only host code runs (no GPU, no CUDA runtime call)."""
import os
import re
import shutil
import subprocess

import cv2
import numpy as np
import pytest

from oracle import cv2_path as C
from oracle import restate as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    nvcc = next((c for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc") if c and os.path.exists(c)), None)
    if nvcc is None:
        pytest.skip("nvcc not found")
    out = tmp_path_factory.mktemp("host_math") / "kernel_math"
    src = os.path.join(ROOT, "tests", "host", "kernel_math.cu")
    # no FMA contraction on the host side either (x86-64 baseline has none; the flag makes it explicit)
    build = subprocess.run([nvcc, "-O2", "-std=c++17", "--fmad=false", "-Xcompiler", "-ffp-contract=off", "-gencode",
                            "arch=compute_100a,code=sm_100a", "-o", str(out), src], capture_output=True, text=True, timeout=600)
    assert build.returncode == 0, build.stdout + build.stderr
    return str(out)


def _run(exe, args, values):
    text = " ".join(float(v).hex() for v in values)
    r = subprocess.run([exe] + [str(a) for a in args], input=text, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)


def _maps(exe, tmp_path, model, K, D, P, w, h):
    d = np.zeros(5)
    dd = np.asarray(D, np.float64).ravel()
    d[:dd.size] = dd
    out = tmp_path / "maps.bin"
    _run(exe, ["maps", model, w, h, out], list(np.asarray(K, np.float64).ravel()) + list(d) + list(np.asarray(P, np.float64).ravel()))
    raw = np.fromfile(out, np.uint8)
    m1 = raw[:w * h * 4].view(np.int16).reshape(h, w, 2)
    m2 = raw[w * h * 4:].view(np.uint16).reshape(h, w)
    return m1, m2


def test_packed_kernel_arithmetic_on_the_host(exe):
    run = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout + run.stderr
    assert "fails=0" in run.stdout


def test_fisheye_and_pinhole_map_code_on_the_host(exe, tmp_path, fx):
    K, D, _ = fx.calib["front"]
    for (w, h, FS, SS) in ((1280, 1024, 0.5, 1), (2560, 2048, 1, 2)):     # InCalibrator / Camera geometries
        P = C.dst_camera_matrix(K, 1280, 1024, FS, SS)
        got, want = _maps(exe, tmp_path, 0, K, D, P, w, h), C.undistort_maps(K, D, P, w, h)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
    rng = np.random.default_rng(11)
    for _ in range(4):
        W, H = int(rng.integers(64, 500)), int(rng.integers(48, 400))
        Kr = np.array([[rng.uniform(80, 500), 0, W / 2 + rng.uniform(-20, 20)], [0, rng.uniform(80, 500), H / 2 + rng.uniform(-20, 20)],
                       [0, 0, 1.0]])
        P = C.dst_camera_matrix(Kr, W, H, rng.uniform(0.3, 1.5), 1, rng.uniform(-9, 9), rng.uniform(-9, 9))
        Dr = rng.uniform(-0.05, 0.05, (4, 1))
        got, want = _maps(exe, tmp_path, 0, Kr, Dr, P, W, H), C.undistort_maps(Kr, Dr, P, W, H)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
        D5 = np.array([rng.uniform(-0.3, 0.1), rng.uniform(-0.05, 0.1), rng.uniform(-1e-3, 1e-3), rng.uniform(-1e-3, 1e-3),
                       rng.uniform(-0.02, 0.02)])
        got, want = _maps(exe, tmp_path, 1, Kr, D5, P, W, H), C.pinhole_maps(Kr, D5[None, :], P, W, H)
        assert (got[0] == want[0]).all() and (got[1] == want[1]).all()


def test_warp_point_code_on_the_host(exe, tmp_path, fx):
    rng = np.random.default_rng(12)
    cases = [(fx.calib[n][2], 1000, 1000) for n in ("front", "left")]
    cases += [(np.eye(3) + rng.normal(0, [[0.3, 0.3, 40], [0.3, 0.3, 40], [6e-4, 6e-4, 0]]), 333, 177) for _ in range(3)]
    for Hm, w, h in cases:
        for unit in (32, 1):
            out = tmp_path / "warp.bin"
            _run(exe, ["warp", w, h, unit, out], list(np.asarray(Hm, np.float64).ravel()))
            xy = np.fromfile(out, np.int32).reshape(h, w, 2)
            X, Y = R.warp_coords(Hm, w, h, unit)
            assert (xy[..., 0] == X).all() and (xy[..., 1] == Y).all()
    # the coordinates are what cv2.warpPerspective itself uses: nearest-neighbour warp of an index image
    Hm = fx.calib["back"][2]
    out = tmp_path / "warp.bin"
    _run(exe, ["warp", 400, 300, 1, out], list(Hm.ravel()))
    xy = np.fromfile(out, np.int32).reshape(300, 400, 2)
    idx = (np.arange(2048 * 2560, dtype=np.int64) % 251).astype(np.uint8).reshape(2048, 2560)
    want = cv2.warpPerspective(idx, Hm, (400, 300), flags=cv2.INTER_NEAREST)
    sx, sy = xy[..., 0], xy[..., 1]
    inside = (sx >= 0) & (sx < 2560) & (sy >= 0) & (sy < 2048)
    got = np.where(inside, idx[np.clip(sy, 0, 2047), np.clip(sx, 0, 2559)], 0)
    assert (got == want).all()


def test_hsv_round_trip_code_on_the_host_all_colours(exe, tmp_path):
    """luminance_balance's 8-bit BGR -> HSV -> V+delta -> BGR (surroundBEV.py:57-79) for every one of the 2^24 colours:
    the kernels' hsv_roundtrip (host form) against cv2.cvtColor itself -- OpenCV's 32-pixel vector body (truncating)
    on a 4096-wide image, its scalar row tail (rounding) on 31-wide rows."""
    c = np.arange(1 << 24, dtype=np.uint32)
    colours = np.stack([c & 255, (c >> 8) & 255, c >> 16], axis=-1).astype(np.uint8)

    def cv2_round_trip(img, delta):
        h, s, v = cv2.split(cv2.cvtColor(img, cv2.COLOR_BGR2HSV))
        v = cv2.add(v, float(delta))                                            # the reference's saturating V shift (:74)
        return cv2.cvtColor(cv2.merge([h, s, v]), cv2.COLOR_HSV2BGR)

    for delta in (0, 6, -6, 100, -200):
        out = tmp_path / "hsv.bin"
        r = subprocess.run([exe, "hsv", str(delta), "0", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0
        got = np.fromfile(out, np.uint8).reshape(-1, 3)
        want = cv2_round_trip(colours.reshape(4096, 4096, 3), delta).reshape(-1, 3)
        assert (got == want).all(), (delta, int((got != want).any(axis=1).sum()))
    # scalar tail: rows of 31 pixels never enter the vector body
    n = (1 << 24) // 31 * 31
    out = tmp_path / "hsv_tail.bin"
    assert subprocess.run([exe, "hsv", "-6", "1", str(out)], capture_output=True, text=True, timeout=600).returncode == 0
    got = np.fromfile(out, np.uint8).reshape(-1, 3)[:n]
    want = cv2_round_trip(colours[:n].reshape(-1, 31, 3), -6).reshape(-1, 3)
    assert (got == want).all(), int((got != want).any(axis=1).sum())


def test_bev_lut_build_code_on_the_host(exe, tmp_path, fx):
    """Camera.get_bev_maps (surroundBEV.py:105-108) for all four fixture cameras through the code k_warp_maps<1> runs
    (undistort map evaluated at the taps, FP32 plane interpolation, cvRound + saturate), against cv2.warpPerspective of
    the cv2-built 2560x2048 map planes; and k_warp_maps<0> on given planes with a random homography."""
    g = fx.geometry(1280, 1024, 1000, 1000)
    for name in ("front", "back", "left", "right"):
        K, D, Hm = fx.calib[name]
        ref = C.RefCamera(K, D, Hm, g)
        out = tmp_path / "bev.bin"
        vals = list(K.ravel()) + list(np.asarray(D, np.float64).ravel()[:4]) + list(ref.P.ravel()) + list(Hm.ravel())
        _run(exe, ["bevmaps", 2560, 2048, 1000, 1000, out], vals)
        raw = np.fromfile(out, np.uint8)
        m1 = raw[:4000000].view(np.int16).reshape(1000, 1000, 2)
        m2 = raw[4000000:].view(np.uint16).reshape(1000, 1000)
        assert (m1 == ref.bev_maps[0]).all() and (m2 == ref.bev_maps[1]).all(), name
    rng = np.random.default_rng(13)
    p1 = rng.integers(-5, 500, (120, 160, 2)).astype(np.int16)
    p2 = rng.integers(0, 1024, (120, 160)).astype(np.uint16)
    Hm = np.eye(3) + rng.normal(0, [[0.2, 0.2, 20], [0.2, 0.2, 20], [5e-4, 5e-4, 0]])
    with open(tmp_path / "planes.bin", "wb") as f:
        f.write(p1.tobytes()); f.write(p2.tobytes())
    _run(exe, ["warpmaps", 160, 120, 140, 90, tmp_path / "planes.bin", tmp_path / "warped.bin"], list(Hm.ravel()))
    raw = np.fromfile(tmp_path / "warped.bin", np.uint8)
    n = 140 * 90
    assert (raw[:4 * n].view(np.int16).reshape(90, 140, 2) == cv2.warpPerspective(p1, Hm, (140, 90))).all()
    assert (raw[4 * n:].view(np.uint16).reshape(90, 140) == cv2.warpPerspective(p2, Hm, (140, 90))).all()


def test_blend_weight_code_on_the_host(exe, tmp_path):
    """BlendMask.get_blend_mask (surroundBEV.py:270-277): the k_blend_masks pixel code on the host against the oracle's
    restatement (itself pinned to the reference's pointPolygonTest loop in test_oracle.py), two geometries."""
    names = ("front", "back", "left", "right")
    for BW, BH, CW, CH in ((1000, 1000, 250, 400), (333, 257, 83, 102)):
        polys = np.stack([R.fill_poly(BW, BH, R.blend_polygon(n, BW, BH, CW, CH)) for n in names])
        L = R.blend_lines(BW, BH, CW, CH)
        lines = np.stack([np.asarray(L[k]).reshape(4) for k in ("FL", "FR", "BL", "BR", "LF", "LB", "RF", "RB")])
        (tmp_path / "polys.bin").write_bytes(polys.tobytes())
        _run(exe, ["blend", BW, BH, tmp_path / "polys.bin", tmp_path / "blend.bin"], list(lines.ravel()))
        got = np.fromfile(tmp_path / "blend.bin", np.uint8).reshape(4, BH, BW)
        for i, n in enumerate(names):
            assert (got[i] == R.blend_mask(n, BW, BH, CW, CH)).all(), (n, BW, BH)


def test_balance_scalar_code_on_the_host(exe, fx):
    """luminance_balance's offsets (surroundBEV.py:66-74) and color_balance's gains (:43-55) from exact integer sums:
    the k_delta / k_gain scalar code on the host against the reference's cv2 call sequence on the fixture frames."""
    frames = fx.frames()
    rng = np.random.default_rng(14)
    canvas = rng.integers(0, 256, (300, 400, 3), dtype=np.uint8)
    canvas[..., 1] //= 2                                         # distinct channel means -> gains away from 1
    vsum = [int(f.max(axis=2).astype(np.int64).sum()) for f in frames]
    csum = [int(canvas[..., c].astype(np.int64).sum()) for c in range(3)]
    vals = [frames[0].shape[0] * frames[0].shape[1], canvas.shape[0] * canvas.shape[1]] + vsum + csum
    r = subprocess.run([exe, "balance"], input=" ".join(float(v).hex() for v in vals), capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    rows = r.stdout.strip().split("\n")
    assert [int(t) for t in rows[0].split()] == R.luminance_offsets(frames)[0] == [6, -1, -6, 0]     # SURVEY 8a-11
    table = np.array([[int(t) for t in row.split()] for row in rows[1:4]], np.uint8)
    got = np.stack([table[c][canvas[..., c]] for c in range(3)], axis=-1)
    assert (got == C.color_balance(canvas.copy())).all()
    # the offsets are what the reference's float expression rounds to: V += (mean of means - own mean), cv2.add saturating
    hsv_v = [cv2.split(cv2.cvtColor(f, cv2.COLOR_BGR2HSV))[2] for f in frames]
    means = [np.mean(v) for v in hsv_v]
    vm = (means[0] + means[1] + means[2] + means[3]) / 4
    for v, m, d in zip(hsv_v, means, [int(t) for t in rows[0].split()]):
        assert (cv2.add(v, (vm - m)) == np.clip(v.astype(np.int32) + d, 0, 255)).all()


# ------------------------------------------------------------------ the whole BEV path on the CPU
from tests.helpers import NAMES, h16  # noqa: E402


def _bev_on_host(exe, tmp_path, fx, g, calib, masks, frames, car, balance, nearest=False):
    """Product plan compiler + plan interpreter (kernel_math bev): LUT planes built by the host form of the
    k_warp_maps<1> code, masks as given, one frame-set."""
    cams = [calib[n] for n in NAMES] if isinstance(calib, dict) else list(calib)
    blob = [np.array([len(cams), g.FW, g.FH, g.BW, g.BH, int(nearest), int(balance), int(car is not None)], np.int32).tobytes()]
    for (K, D, Hm), mask in zip(cams, masks):
        P = C.dst_camera_matrix(K, g.FW, g.FH, g.FS, g.SS)
        out = tmp_path / "lut.bin"
        vals = list(np.asarray(K).ravel()) + list(np.asarray(D, np.float64).ravel()[:4]) + list(P.ravel()) + list(np.asarray(Hm).ravel())
        _run(exe, ["bevmaps", int(g.FW * g.SS), int(g.FH * g.SS), g.BW, g.BH, out], vals)
        blob += [out.read_bytes(), np.ascontiguousarray(mask, np.uint8).tobytes()]
    blob += [np.ascontiguousarray(f).tobytes() for f in frames]
    if car is not None:
        blob.append(np.ascontiguousarray(car).tobytes())
    (tmp_path / "bev_in.bin").write_bytes(b"".join(blob))
    r = subprocess.run([exe, "bev", str(tmp_path / "bev_in.bin"), str(tmp_path / "bev_out.bin")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    out = np.fromfile(tmp_path / "bev_out.bin", np.uint8).reshape(g.BH, g.BW, 3)
    # the TMA-staged kernel's plan (bevk_plan_tma.cuh) through its own interpreter: boxes modelled as the tensor copy
    # delivers them (zeros outside the frame); several (stage size, entry groups per slot) settings: the library's own
    # (TMA_FS, TMA_EG), one that forces strip splits / multi-pass / GATHER items, three entry groups per slot
    # (4 groups = 3 + 1), single-group items.  info: the interpreters' output, the library's setting first.
    info = r.stdout
    for setting in (["shipped"], ["1536", "4"], ["4096", "3"], ["6144", "1"]):
        rt = subprocess.run([exe, "bevtma", str(tmp_path / "bev_in.bin"), str(tmp_path / "bevtma_out.bin"), *setting],
                            capture_output=True, text=True, timeout=600)
        assert rt.returncode == 0, (rt.returncode, rt.stdout, rt.stderr)
        out_t = np.fromfile(tmp_path / "bevtma_out.bin", np.uint8).reshape(g.BH, g.BW, 3)
        assert (out_t == out).all(), (setting, int((out_t != out).sum()), rt.stdout)
        info += rt.stdout
    return out, info


@pytest.mark.parametrize("blend", [False, True])
@pytest.mark.parametrize("balance", [False, True])
def test_bev_path_on_the_host_native_golden(exe, tmp_path, fx, blend, balance):
    """BevGenerator.__call__ (surroundBEV.py:312-325) at the reference's native geometry, all four flag combinations,
    with and without the car: plan compiler + per-entry kernel arithmetic on the CPU == golden hashes of the reference."""
    g = fx.geometry()
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if blend else C.plain_mask(n, g) for n in NAMES]
    gold = fx.gold["native"][f"blend{int(blend)}_balance{int(balance)}"]
    for car_key, car in (("car", fx.car()), ("nocar", None)):
        out, info = _bev_on_host(exe, tmp_path, fx, g, fx.calib, masks, fx.frames(), car, balance)
        assert h16(out) == gold[car_key], (car_key, info)
        # the library's plan at this geometry has every slot kind of k_bev_tma -- two- and four-pass items and GATHER
        # items -- so the GPU A/B of this geometry against the gather kernel runs all of them
        kinds = re.search(r"two_pass=(\d+) four_pass=(\d+) gather_items=(\d+)", info)
        assert kinds and all(int(n) > 0 for n in kinds.groups()), info


@pytest.mark.parametrize("key,FW,FH,BW,BH,blend,balance,car", [
    ("cfg2_1280x960_1000_plain", 1280, 960, 1000, 1000, False, False, False),
    ("cfg3_1920x1080_1200_blend_balance_car", 1920, 1080, 1200, 1200, True, True, True),
    ("odd_1000x750_777x900_blend_balance_car", 1000, 750, 777, 900, True, True, True),
])
def test_bev_path_on_the_host_config_golden(exe, tmp_path, fx, key, FW, FH, BW, BH, blend, balance, car):
    """BASELINE config shapes and an odd geometry (ragged edge tiles, row pitch 3000 = 8 mod 16, 777-px canvas rows)."""
    g = fx.geometry(FW, FH, BW, BH)
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if blend else C.plain_mask(n, g) for n in NAMES]
    out, _ = _bev_on_host(exe, tmp_path, fx, g, fx.scaled_calib(g), masks, fx.frames(FW, FH), fx.car(BW, BH) if car else None, balance)
    assert h16(out) == fx.gold["cfg"][key]


def test_bev_path_on_the_host_unaligned_pitch_and_nearest(exe, tmp_path, fx):
    """A frame width whose row pitch is not a multiple of 4 sends every entry through the per-tap checked path
    (sample_slow_core); INTER_NEAREST is compiled into the plan.  Both against the cv2 call sequence."""
    g = fx.geometry(333, 250, 203, 177)
    calib = fx.scaled_calib(g)
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) for n in NAMES]
    frames, car = fx.frames(333, 250), fx.car(203, 177)
    ref = C.RefBev(calib, g, True, True, masks=masks)
    out, _ = _bev_on_host(exe, tmp_path, fx, g, calib, masks, frames, car, True)
    assert (out == ref(*frames, car)).all()
    g2 = fx.geometry(640, 512, 500, 500)
    calib2 = fx.scaled_calib(g2)
    masks2 = [C.plain_mask(n, g2) for n in NAMES]
    frames2 = fx.frames(640, 512)
    cams = [C.RefCamera(*calib2[n], g2) for n in NAMES]
    want = np.zeros((500, 500, 3), np.uint8)
    for cam, m, f in zip(cams, masks2, frames2):
        want = cv2.add(want, R.apply_plain(cv2.remap(f, *cam.bev_maps, interpolation=cv2.INTER_NEAREST), m))
    out2, _ = _bev_on_host(exe, tmp_path, fx, g2, calib2, masks2, frames2, None, False, nearest=True)
    assert (out2 == want).all()


def test_stand_alone_gathers_on_the_host(exe, tmp_path, fx):
    """Tools/undistort.py / InCalibrator.undistort (fused form: camera model per pixel) and ExCalibrator.warp through
    the k_gather4 pixel code (gather_px) on the CPU, against the golden hashes of the reference."""
    K, D, _ = fx.calib["front"]
    d5 = list(np.asarray(D, np.float64).ravel()[:4]) + [0.0]
    front = fx.img("front")
    (tmp_path / "src.bin").write_bytes(front.tobytes())
    P = C.dst_camera_matrix(K, 1280, 1024, 1, 1)                                   # Tools/undistort.py defaults
    _run(exe, ["gather", 1, 1280, 1024, 1280, 1024, tmp_path / "src.bin", tmp_path / "und.bin"],
         list(K.ravel()) + d5 + list(P.ravel()) + [0.0])
    und = np.fromfile(tmp_path / "und.bin", np.uint8).reshape(1024, 1280, 3)
    assert h16(und) == fx.gold["tools_undistort_front"]
    raw0 = fx.img("raw0")
    (tmp_path / "src.bin").write_bytes(raw0.tobytes())
    P = C.dst_camera_matrix(K, 1280, 1024, 0.5, 1)                                 # InCalibrator: FOCAL_SCALE 0.5
    _run(exe, ["gather", 1, 1280, 1024, 1280, 1024, tmp_path / "src.bin", tmp_path / "und.bin"],
         list(K.ravel()) + d5 + list(P.ravel()) + [0.0])
    assert h16(np.fromfile(tmp_path / "und.bin", np.uint8).reshape(1024, 1280, 3)) == fx.gold["incalib_fisheye_raw0"]["undistort"]
    K2 = np.diag([0.5, 480 / 1024, 1.0]) @ K                                       # BASELINE cfg1b: 640x480
    small = cv2.resize(raw0, (640, 480), interpolation=cv2.INTER_LINEAR)
    (tmp_path / "src.bin").write_bytes(small.tobytes())
    _run(exe, ["gather", 1, 640, 480, 640, 480, tmp_path / "src.bin", tmp_path / "und.bin"],
         list(K2.ravel()) + d5 + list(C.dst_camera_matrix(K2, 640, 480, 0.5, 1).ravel()) + [0.0])
    assert h16(np.fromfile(tmp_path / "und.bin", np.uint8).reshape(480, 640, 3)) == fx.gold["incalib_fisheye_raw0_640x480"]["undistort"]
    Kn = K * np.array([[2.0], [2.0], [1.0]])                                        # InCalibrator('normal'): pinhole model
    (tmp_path / "src.bin").write_bytes(raw0.tobytes())
    _run(exe, ["gather", 1, 1280, 1024, 1280, 1024, tmp_path / "src.bin", tmp_path / "und.bin"],
         list(Kn.ravel()) + list(np.asarray(fx.D5, np.float64).ravel()) + list(C.dst_camera_matrix(Kn, 1280, 1024, 0.5, 1).ravel()) + [1.0])
    assert h16(np.fromfile(tmp_path / "und.bin", np.uint8).reshape(1024, 1280, 3)) == fx.gold["incalib_normal_raw0"]["undistort"]
    src = fx.img("src_back")
    Hm = fx.calib["back"][2]
    (tmp_path / "src.bin").write_bytes(src.tobytes())
    _run(exe, ["gather", 2, src.shape[1], src.shape[0], 1000, 1000, tmp_path / "src.bin", tmp_path / "warp.bin"], list(Hm.ravel()))
    assert h16(np.fromfile(tmp_path / "warp.bin", np.uint8).reshape(1000, 1000, 3)) == fx.gold["excalib_warp_back"]


def test_bev_path_on_the_host_eight_cameras(exe, tmp_path, fx):
    """BASELINE configs[4] semantics (SURVEY 8d.5) at a small size: 8 cameras, 8 angular wedge masks; oracle = the
    reference's Camera.raw2bev per camera + the N-way saturating compose."""
    g = fx.geometry(640, 512, 480, 480)
    calib4 = fx.scaled_calib(g)
    c, s_ = np.cos(np.pi / 4), np.sin(np.pi / 4)
    cx, cy = g.BW / 2, g.BH / 2
    Rot = np.array([[c, -s_, cx - c * cx + s_ * cy], [s_, c, cy - s_ * cx - c * cy], [0, 0, 1.0]])
    cams = [calib4[n] for n in NAMES] + [(calib4[n][0], calib4[n][1], Rot @ calib4[n][2]) for n in NAMES]
    ang = np.linspace(0, 2 * np.pi, 9)
    masks = []
    for i in range(8):
        tri = np.array([[cx, cy], [cx + g.BW * np.cos(ang[i]), cy + g.BW * np.sin(ang[i])],
                        [cx + g.BW * np.cos(ang[i + 1]), cy + g.BW * np.sin(ang[i + 1])]]).astype(np.int32)
        masks.append(cv2.fillPoly(np.zeros((g.BH, g.BW), np.uint8), [tri], 255))
    frames = fx.frames(g.FW, g.FH)
    frames8 = frames + [np.ascontiguousarray(f[:, ::-1]) for f in frames]
    want = np.zeros((g.BH, g.BW, 3), np.uint8)
    for (K, D, Hm), m, f in zip(cams, masks, frames8):
        want = R.sat_add(want, R.apply_plain(C.RefCamera(K, D, Hm, g).raw2bev(f), m))
    out, info = _bev_on_host(exe, tmp_path, fx, g, cams, masks, frames8, None, False)
    assert (out == want).all(), info


def _fuzz_case(rng, case):
    """Random geometry, maps (sometimes at the int16 extremes), masks and frames -> (input blob, cv2-based expectation)."""
    NC = int(rng.integers(1, 4))
    FW, FH = int(rng.integers(8, 90)), int(rng.integers(8, 70))
    BW, BH = int(rng.integers(5, 80)), int(rng.integers(5, 75))
    nearest = bool(case % 3 == 2)
    blob = [np.array([NC, FW, FH, BW, BH, int(nearest), 0, 0], np.int32).tobytes()]
    frames, maps, masks = [], [], []
    for _ in range(NC):
        lo, hi = (-6, 6) if case % 4 else (-40000, 40000)
        m1 = np.stack([rng.integers(lo, FW + hi, (BH, BW)), rng.integers(lo, FH + hi, (BH, BW))], -1).clip(-32768, 32767).astype(np.int16)
        m2 = rng.integers(0, 1024, (BH, BW)).astype(np.uint16)
        kind = rng.integers(0, 3)
        mask = (rng.integers(0, 2, (BH, BW)) * 255 if kind == 0 else rng.integers(0, 256, (BH, BW)) if kind == 1
                else np.full((BH, BW), 255)).astype(np.uint8)
        maps.append((m1, m2)); masks.append(mask)
        frames.append(rng.integers(0, 256, (FH, FW, 3), dtype=np.uint8))
        blob += [m1.tobytes(), m2.tobytes(), mask.tobytes()]
    blob += [f.tobytes() for f in frames]
    want = np.zeros((BH, BW, 3), np.uint8)
    for f, (m1, m2), mask in zip(frames, maps, masks):
        warped = cv2.remap(f, m1, m2, cv2.INTER_NEAREST if nearest else cv2.INTER_LINEAR)
        want = cv2.add(want, R.apply_blend(warped, mask))
    return b"".join(blob), want


def _run_fuzz(exe_path, tmp_path, n_cases, env=None):
    rng = np.random.default_rng(500)
    for case in range(n_cases):
        blob, want = _fuzz_case(rng, case)
        (tmp_path / "fz_in.bin").write_bytes(blob)
        r = subprocess.run([str(exe_path), "bev", str(tmp_path / "fz_in.bin"), str(tmp_path / "fz_out.bin")], capture_output=True,
                           text=True, timeout=300, env=env)
        assert r.returncode == 0, (case, r.stderr[-2000:])
        got = np.fromfile(tmp_path / "fz_out.bin", np.uint8).reshape(want.shape)
        assert (got == want).all(), (case, want.shape)


def test_plan_compiler_fuzz_arbitrary_maps(exe, tmp_path):
    """bevk_bev_set_maps accepts any CV_16SC2 + CV_16UC1 planes: random maps with taps far outside the frame, random
    masks (0, 255 and weights), 1-3 cameras, tiny ragged geometries, every pitch alignment, both interpolations --
    plan compiler + interpreter against cv2.remap + the mask / compose restatement."""
    _run_fuzz(exe, tmp_path, 48)


def test_plan_compiler_memory_safety_under_sanitizers(tmp_path, fx, exe):
    """The plan compiler and the interpreter again, built with AddressSanitizer + UBSan, on the geometry with ragged
    edge tiles and an unaligned pitch: no out-of-bounds plan index, same canvas as the plain build."""
    nvcc = next((c for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc") if c and os.path.exists(c)), None)
    san = tmp_path / "kernel_math_san"
    build = subprocess.run([nvcc, "-O1", "-g", "-std=c++17", "--fmad=false", "-Xcompiler",
                            "-ffp-contract=off,-fsanitize=address,-fsanitize=undefined,-fno-sanitize-recover=undefined,-fno-omit-frame-pointer",
                            "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(san),
                            os.path.join(ROOT, "tests", "host", "kernel_math.cu"), "-lasan", "-lubsan"],
                           capture_output=True, text=True, timeout=900)
    if build.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + build.stderr[-200:])
    g = fx.geometry(333, 250, 203, 177)
    calib = fx.scaled_calib(g)
    masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) for n in NAMES]
    frames, car = fx.frames(333, 250), fx.car(203, 177)
    want, _ = _bev_on_host(exe, tmp_path, fx, g, calib, masks, frames, car, True)
    env = dict(os.environ, ASAN_OPTIONS="protect_shadow_gap=0:detect_leaks=0")
    r = subprocess.run([str(san), "bev", str(tmp_path / "bev_in.bin"), str(tmp_path / "bev_san.bin")], capture_output=True, text=True,
                       timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert (np.fromfile(tmp_path / "bev_san.bin", np.uint8).reshape(g.BH, g.BW, 3) == want).all()
    _run_fuzz(san, tmp_path, 16, env=env)      # arbitrary maps (int16 extremes included) under the sanitizers too
