"""GPU parity tests of the TMA-staged fused kernel k_bev_tma (bevk_bev_tma.cuh): every check goes through the C ABI.

The kernel must (a) actually be the one that ran (bevk_bev_last_path == 2), (b) agree byte for byte with the
round-1 pointer-table gather kernel on the same inputs (BEVK_TMA=0 engine), and (c) agree with the oracle -- the
golden hashes of the unmodified reference and the reference's cv2 call sequence run live (oracle/cv2_path.py) -- at
the BASELINE sizes: cfg4 (4 x 1920x1080 -> 1000^2, blend) and cfg5 (8 cameras 3840x2160 -> 2000^2)."""
import os

import cv2
import numpy as np
import pytest

from oracle import cv2_path as C
from oracle import restate as R
from tests.helpers import NAMES, h16

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from cameracalibration_b200 import ops as o
    return o


def _engine(ops, fx, g, blend, calib=None, masks=None, tma=True, cams=None):
    """BevEngine for geometry g; tma=False builds it with BEVK_TMA=0 (read at finalize): the gather kernel only."""
    calib = calib or fx.scaled_calib(g)
    cams = cams or [calib[n] for n in NAMES]
    e = ops.BevEngine(len(cams), (g.FW, g.FH), (g.BW, g.BH))
    if masks is None:
        masks = [R.blend_mask(n, g.BW, g.BH, g.CW, g.CH) if blend else C.plain_mask(n, g) for n in NAMES]
    for i, (K, D, H) in enumerate(cams):
        e.set_camera(i, K, D, C.dst_camera_matrix(K, g.FW, g.FH, g.FS, g.SS), (int(g.FW * g.SS), int(g.FH * g.SS)), H)
        e.set_mask(i, masks[i])
    want = {"BEVK_TMA": "1" if tma else "0"}
    old = {k: os.environ.get(k) for k in want}
    os.environ.update(want)
    try:
        e.finalize()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return e, masks


def _stack(torch, dev, sets):
    """list (batch) of lists (cameras) of frames -> one uint8[batch][cam][FH][FW][3] device tensor (a frame stack)."""
    return torch.from_numpy(np.stack([np.stack(s) for s in sets])).to(dev)


def _run_stack(torch, e, d_all, car=None, balance=False):
    b, nc, FH, FW, _ = d_all.shape
    out = torch.empty((b, e.BH, e.BW, 3), dtype=torch.uint8, device=d_all.device)
    e.run_stack(d_all.data_ptr(), FH * FW * 3, b, out.data_ptr(), 0 if car is None else car.data_ptr(), balance)
    e.ctx.sync()
    return out.cpu().numpy()


@pytest.mark.parametrize("blend", [False, True])
def test_tma_kernel_native_goldens_and_ab(ops, fx, blend):
    """Reference geometry (1280x1024 -> 1000^2): goldens of the unmodified reference through the TMA kernel, all batch
    groupings (1: NB=1 variant; 4, 6: NB=4 with a ragged tail), with and without the car, balance on and off; the same
    inputs through the gather kernel must give the same bytes.  The plan has every slot kind -- one-, two- and four-pass
    TMA items and GATHER items (counted on the host by test_bev_path_on_the_host_native_golden) -- so the A/B covers all."""
    import torch
    g = fx.geometry()
    et, _ = _engine(ops, fx, g, blend, calib=fx.calib, tma=True)
    eg, _ = _engine(ops, fx, g, blend, calib=fx.calib, tma=False)
    info = et.tma_plan_info()
    assert info["items"] > 0 and info["tma_entries"] > 10 * info["gather_entries"] > 0, info
    assert eg.tma_plan_info()["items"] == 0
    dev = torch.device("cuda", et.ctx.device)
    F = fx.frames()
    rng = np.random.default_rng(5)
    sets = [F] + [[np.ascontiguousarray(np.roll(f, 13 * i + 5 * c, axis=1) ^ rng.integers(0, 16, f.shape, dtype=np.uint8))
                   for c, f in enumerate(F)] for i in range(1, 6)]
    car = torch.from_numpy(fx.car()).to(dev)
    for nb in (1, 4, 6):
        d_all = _stack(torch, dev, sets[:nb])
        for balance in (False, True):
            for c, ckey in ((car, "car"), (None, "nocar")):
                a = _run_stack(torch, et, d_all, c, balance)
                assert et.last_path() == "tma"
                b = _run_stack(torch, eg, d_all, c, balance)
                assert eg.last_path() == "gather"
                assert (a == b).all(), (nb, balance, ckey, int((a != b).sum()))
                assert h16(a[0]) == fx.gold["native"][f"blend{int(blend)}_balance{int(balance)}"][ckey], (nb, balance, ckey)


def test_tma_kernel_cfg4_size_vs_live_oracle(ops, fx):
    """BASELINE configs[3] shape (4 x 1920x1080 -> 1000^2, blend=True): the bench workload's geometry.  Frame-sets per
    SURVEY 8(d).4: fixture frames blended with seeded noise, one all-random set, one constant-255 set (saturation /
    rounding stress).  Oracle: the reference's cv2 call sequence, live."""
    import torch
    g = fx.geometry(1920, 1080, 1000, 1000)
    calib = fx.scaled_calib(g)
    et, masks = _engine(ops, fx, g, True, calib=calib)
    ref = C.RefBev(calib, g, True, False, masks=masks)
    dev = torch.device("cuda", et.ctx.device)
    rng = np.random.default_rng(99)
    sets = [fx.perturbed_frames(g.FW, g.FH, i) for i in range(3)]
    sets.append([rng.integers(0, 256, (g.FH, g.FW, 3), dtype=np.uint8) for _ in NAMES])
    sets.append([np.full((g.FH, g.FW, 3), 255, np.uint8) for _ in NAMES])
    car_h = fx.car(g.BW, g.BH)
    car = torch.from_numpy(car_h).to(dev)
    got = _run_stack(torch, et, _stack(torch, dev, sets), car)
    assert et.last_path() == "tma"
    for i, s in enumerate(sets):
        want = ref(*s, car_h)
        assert (got[i] == want).all(), (i, int((got[i] != want).sum()))
    # the host entry point (staging buffers are a frame stack too) and its pageable / page-locked ingest paths
    host = et.run(sets, car_h)
    assert et.last_path() == "tma" and (host == got).all()


def test_tma_kernel_camera_ranges_and_cam_sharded_compose(ops, fx):
    """Camera-per-GPU decomposition over a frame stack: partial canvases of camera ranges (bevk_bev_run_stack_cams)
    composed with the saturating sum equal the full canvas; ranges that skip the plan's first camera of a tile make a
    later camera the one that stores."""
    import torch
    g = fx.geometry()
    et, _ = _engine(ops, fx, g, True, calib=fx.calib)
    dev = torch.device("cuda", et.ctx.device)
    F = fx.frames()
    sets = [F, [np.ascontiguousarray(f[::-1]) for f in F], F, F, [np.ascontiguousarray(f[:, ::-1]) for f in F]]
    d_all = _stack(torch, dev, sets)
    full = _run_stack(torch, et, d_all)
    assert h16(full[0]) == fx.gold["native"]["blend1_balance0"]["nocar"]
    for ranges in ([(0, 1), (1, 2), (2, 3), (3, 4)], [(0, 3), (3, 4)], [(2, 4), (0, 2)]):
        parts = []
        for lo, hi in ranges:
            p = torch.empty((5, g.BH, g.BW, 3), dtype=torch.uint8, device=dev)
            et.run_stack_cams(d_all.data_ptr(), g.FH * g.FW * 3, 5, lo, hi, p.data_ptr())
            assert et.last_path() == "tma"
            parts.append(p)
        out = torch.empty_like(parts[0])
        et.sat_sum_device([p.data_ptr() for p in parts], out.numel(), out.data_ptr())
        et.ctx.sync()
        assert (out.cpu().numpy() == full).all(), ranges


def test_tma_kernel_cfg5_eight_cameras_4k(ops, fx):
    """BASELINE configs[4] as written: 8 cameras 3840x2160 -> 2000x2000 (SURVEY 8d.5): cameras 0-3 = the scaled fixtures,
    4-7 = the same four with H post-multiplied by a 45-degree rotation about the canvas centre; 8 angular wedge masks
    (cv2.fillPoly).  Oracle = the reference's Camera.raw2bev per camera (cv2 call sequence) + the N-way saturating
    compose.  Also the per-camera partial canvases (one camera per GPU) against the same oracle."""
    import torch
    g = fx.geometry(3840, 2160, 2000, 2000)
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
    et, _ = _engine(ops, fx, g, False, masks=masks, cams=cams)
    frames = fx.frames(g.FW, g.FH)
    frames8 = frames + [np.ascontiguousarray(f[:, ::-1]) for f in frames]
    want = np.zeros((g.BH, g.BW, 3), np.uint8)
    per_cam = []
    for (K, D, H), m, f in zip(cams, masks, frames8):
        per_cam.append(R.apply_plain(C.RefCamera(K, D, H, g).raw2bev(f), m))
        want = R.sat_add(want, per_cam[-1])
    dev = torch.device("cuda", et.ctx.device)
    d_all = _stack(torch, dev, [frames8])
    got = _run_stack(torch, et, d_all)
    assert et.last_path() == "tma"
    assert (got[0] == want).all(), int((got[0] != want).sum())
    for k in (0, 3, 6):
        p = torch.empty((1, g.BH, g.BW, 3), dtype=torch.uint8, device=dev)
        et.run_stack_cams(d_all.data_ptr(), g.FH * g.FW * 3, 1, k, k + 1, p.data_ptr())
        et.ctx.sync()
        assert (p.cpu().numpy()[0] == per_cam[k]).all(), k


def test_tma_falls_back_when_the_stack_is_not_16_byte_friendly(ops, fx):
    """A frame stack at an address or stride that is not a multiple of 16 bytes, and a row pitch that is not (640x480 is,
    1000x750 is not), take the pointer-table gather -- same bytes."""
    import torch
    g = fx.geometry(640, 512, 500, 500)
    et, _ = _engine(ops, fx, g, True)
    dev = torch.device("cuda", et.ctx.device)
    F = fx.frames(g.FW, g.FH)
    fb = g.FW * g.FH * 3
    want = et.run([F, F[::-1]])
    assert et.last_path() == "tma"
    raw = torch.zeros(8 * (fb + 4) + 64, dtype=torch.uint8, device=dev)
    for shift, stride in ((4, fb), (0, fb + 4), (16, fb)):
        view = raw[shift:shift + 8 * stride]
        for i, f in enumerate(F + F[::-1]):
            view[i * stride:i * stride + fb] = torch.from_numpy(f).reshape(-1).to(dev)
        out = torch.empty((2, g.BH, g.BW, 3), dtype=torch.uint8, device=dev)
        et.run_stack(view.data_ptr(), stride, 2, out.data_ptr())
        et.ctx.sync()
        aligned = (view.data_ptr() % 16 == 0) and stride % 16 == 0
        assert et.last_path() == ("tma" if aligned else "gather"), (shift, stride)
        assert (out.cpu().numpy() == want).all(), (shift, stride)
    g2 = fx.geometry(1000, 750, 777, 900)            # pitch 3000 B: no TMA plan at all
    e2, masks2 = _engine(ops, fx, g2, True)
    assert e2.tma_plan_info()["items"] == 0
    F2 = fx.frames(g2.FW, g2.FH)
    ref = C.RefBev(fx.scaled_calib(g2), g2, True, False, masks=masks2)
    assert (e2.run([F2])[0] == ref(*F2)).all() and e2.last_path() == "gather"


def test_cuda_graph_capture_of_the_device_entry_points(ops, fx):
    """bevk_graph_begin / end / launch: one frame-set batch (plain and BALANCE: memsets + five kernels) captured once and
    replayed; the replay on new frame contents gives what the direct call gives, and launches are counted per replay."""
    import torch
    from cameracalibration_b200 import _lib as L
    g = fx.geometry()
    et, _ = _engine(ops, fx, g, True, calib=fx.calib)
    dev = torch.device("cuda", et.ctx.device)
    F = fx.frames()
    d_all = _stack(torch, dev, [F, F[::-1], F, F, F[::-1]])
    car = torch.from_numpy(fx.car()).to(dev)
    for balance in (False, True):
        want = _run_stack(torch, et, d_all, car, balance)                   # also warms every buffer and table
        out = torch.zeros((5, g.BH, g.BW, 3), dtype=torch.uint8, device=dev)
        with et.ctx.graph_capture() as gr:
            et.run_stack(d_all.data_ptr(), g.FH * g.FW * 3, 5, out.data_ptr(), car.data_ptr(), balance)
        et.ctx.sync()
        assert not out.any().item()                                          # capturing executes nothing
        n0 = et.ctx.launches
        gr.launch(3)
        et.ctx.sync()
        assert et.ctx.launches - n0 == 3 * (5 if balance else 1)
        assert (out.cpu().numpy() == want).all()
        d_all.copy_(d_all.flip(0))                                           # same buffers, new contents
        torch.cuda.synchronize()
        gr.launch()
        et.ctx.sync()
        assert (out.cpu().numpy() == want[::-1]).all() if not balance else h16(out.cpu().numpy()[4]) == h16(want[0])
        d_all.copy_(d_all.flip(0))
        torch.cuda.synchronize()
        gr.destroy()
    # a call that has to build something inside the capture is reported, not silently dropped
    e2, _ = _engine(ops, fx, fx.geometry(640, 512, 500, 500), True)
    d2 = torch.zeros((1, 4, 512, 640, 3), dtype=torch.uint8, device=dev)
    o2 = torch.empty((1, 500, 500, 3), dtype=torch.uint8, device=dev)
    with pytest.raises(L.BevkError):
        with e2.ctx.graph_capture():
            e2.run_stack(d2.data_ptr(), 512 * 640 * 3, 1, o2.data_ptr())   # first call: tensor maps are built here
    e2.run_stack(d2.data_ptr(), 512 * 640 * 3, 1, o2.data_ptr())            # the ctx is usable afterwards
    e2.ctx.sync()
