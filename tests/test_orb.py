"""ORB descriptor stage (SURVEY.md 8f rank 3): oracle pinned against cv2 and the recorded reference output (CPU),
CUDA kernels against the oracle and cv2 live (GPU, through the C ABI)."""
import math
import os

import cv2
import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_golden
from oracle import c_oracle as co
from oracle import orb_oracle as oo
from slam_experiments_b200 import _native as nat
from slam_experiments_b200 import build as hm_build
from slam_experiments_b200 import synth

gpu = pytest.mark.gpu


def kp_arrays(kps):
    return (np.array([k.pt for k in kps], np.float32).reshape(-1, 2), np.array([k.angle for k in kps], np.float32),
            np.array([k.octave for k in kps], np.int32))


def golden_cases():
    g = load_golden(os.path.join(GOLDEN, "describe_sequence_orb.npz"))
    for name, (h, w, seed, ch, nf) in zip(g["cases"].tolist(), g["params"].tolist()):
        yield name, synth.textured_image(h, w, seed, ch), g[f"{name}_xy"], g[f"{name}_angle"], g[f"{name}_octave"], g[f"{name}_desc"], nf


# ---------------------------------------------------------------- CPU: the oracle is what cv2 computes
def test_pattern_table_files_agree():
    pts = oo.pattern31()
    assert pts.shape == (512, 2) and np.abs(pts).max() <= 15
    assert int((pts * np.arange(1, 1025).reshape(512, 2)).sum()) == -177504      # as printed by tools/extract_orb_pattern.py
    inc = open(os.path.join(ROOT, "slam_experiments_b200", "csrc", "hm_orb_pattern.inc")).read()
    import re
    c_pts = np.array(re.findall(r"\{(-?\d+), (-?\d+)\}", inc), dtype=np.int64)
    assert np.array_equal(c_pts, pts)


def test_oracle_resize_equals_cv2_linear_exact():
    for h, w, seed in ((480, 640, 1), (480, 752, 2), (333, 517, 3), (97, 131, 4)):
        prev = synth.textured_image(h, w, seed)
        for lv in range(1, 6 if h > 100 else 2):
            r, c = oo.level_size(h, w, lv)
            ref = cv2.resize(prev, (c, r), interpolation=cv2.INTER_LINEAR_EXACT)
            assert np.array_equal(oo.resize_linear_exact(prev, r, c), ref), (h, w, lv)
            prev = ref
    up = synth.textured_image(70, 90, 5)           # the edge rules (replicated first / last sample) need an upscale
    assert np.array_equal(oo.resize_linear_exact(up, 155, 201), cv2.resize(up, (201, 155), interpolation=cv2.INTER_LINEAR_EXACT))


def test_oracle_blur_equals_cv2_float_filter():
    """The float filter cv2 runs inside ORB (GaussianBlur on a sub-matrix = sepFilter2D with the float32 kernel), with
    its summation order; exact on AVX2 builds of the wheel (the order is a property of that code path)."""
    g = cv2.getGaussianKernel(7, 2, cv2.CV_32F).ravel()
    assert np.array_equal(g.view(np.uint32), oo.GAUSS7.view(np.uint32))
    rng = np.random.default_rng(3)
    diff = total = 0
    shapes = [(480, 640), (400, 533), (231, 309), (134, 179), (300, 127), (64, 67)]
    shapes += [(int(rng.integers(120, 260)), w) for w in range(40, 170)]       # every residue of the vector bodies' widths
    for h, w in shapes:
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        ref = cv2.sepFilter2D(img, cv2.CV_8U, g, g, borderType=cv2.BORDER_REFLECT_101)
        got = oo.blur_float7(np.pad(img, 3, mode="reflect"), h, w)
        diff += int((got != ref).sum())
        total += h * w
    if cv2.checkHardwareSupport(5):                # CV_CPU_AVX2
        assert diff == 0
    else:                                           # another dispatch of cv2's filter: rounding of a few pixels may differ
        assert diff <= total * 1e-5


def test_oracle_gray_equals_cv2():
    img = synth.textured_image(120, 160, 9, 3)
    assert np.array_equal(oo.to_gray(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))


def test_oracle_describe_equals_recorded_reference_output():
    """Fixture written by the unmodified reference's OrbFeatureDetector (tests/golden/make_golden_orb_describe.py)."""
    for name, img, xy, ang, octv, desc, nf in golden_cases():
        assert np.array_equal(oo.describe(img, xy, ang, octv), desc), name


def test_oracle_describe_equals_cv2_live():
    for h, w, seed, ch, nf in ((480, 640, 21, 1, 1500), (200, 260, 22, 3, 300)):
        img = synth.textured_image(h, w, seed, ch)
        orb = cv2.ORB.create(nfeatures=nf)
        kps, desc = orb.detectAndCompute(img, None)            # feature_detectors.py:26
        assert np.array_equal(oo.describe(img, *kp_arrays(kps)), desc)
        kps2, desc2 = orb.compute(img, orb.detect(img, None))  # detect + compute is the same computation
        assert np.array_equal(desc2, desc) and len(kps2) == len(kps)


def test_library_frame_rule_geometry_and_angles_without_a_device():
    """Level sizes and scales, the per-level frame rule (a level only has to be more than 32 pixels, so a 40-pixel
    side is accepted and a 32-pixel one is not), and the (cos, sin) arithmetic, all on the host."""
    hm_build.build()
    for h, w in ((480, 640), (480, 752), (333, 517), (1920, 2560), (1080, 1920)):
        for lv in range(8):
            r, c, inv = nat.orb_level_geometry(h, w, lv)
            assert (r, c) == oo.level_size(h, w, lv)
            assert np.float32(inv) == np.float32(1.0) / oo.level_scale(lv)
    assert nat.orb_level_geometry(40, 640, 0)[:2] == (40, 640)     # a level only has to hold the 32-pixel frame
    with pytest.raises(nat.NativeError):
        nat.orb_level_geometry(32, 640, 0)
    with pytest.raises(nat.NativeError):
        nat.orb_level_geometry(640, 32, 0)
    ang = np.concatenate([np.random.default_rng(0).random(200000).astype(np.float32) * np.float32(360), np.arange(0, 360, 0.5, dtype=np.float32)])
    rad = ang * np.float32(math.pi / np.float32(180.0))
    ref = np.stack([np.cos(rad.astype(np.float64)).astype(np.float32), np.sin(rad.astype(np.float64)).astype(np.float32)], 1)
    assert np.array_equal(nat.orb_angles_to_cs(ang), ref)


def test_angle_arithmetic_is_cv2s():
    """cv2 takes cos / sin in double and rounds to float; on the rare angles where that and cosf / sinf would sample a
    different pixel, its descriptors follow the double variant (so does hm_orb_angles_to_cs)."""
    rng = np.random.default_rng(1)
    ang = rng.random(400000).astype(np.float32) * np.float32(360)
    cs = nat.orb_angles_to_cs(ang)
    pat = oo.pattern31().astype(np.float32)
    img = rng.integers(0, 256, (200, 200), dtype=np.uint8)
    lv = oo.build_pyramid(img, 1)[0]
    orb = cv2.ORB.create()
    for i in range(0, 400000, 40000):
        _, d = orb.compute(img, [cv2.KeyPoint(100.0, 100.0, 31.0, float(ang[i]), 1.0, 0)])
        ix = np.rint(pat[:, 0] * cs[i, 0] - pat[:, 1] * cs[i, 1]).astype(int)
        iy = np.rint(pat[:, 0] * cs[i, 1] + pat[:, 1] * cs[i, 0]).astype(int)
        v = lv[132 + iy, 132 + ix].astype(int)
        assert np.array_equal(np.packbits((v[0::2] < v[1::2]).astype(np.uint8), bitorder="little"), d[0])


# ---------------------------------------------------------------- GPU: the kernels are what the oracle computes
def plane_layout(h, w, n_levels):
    """Byte layout of one pyramid plane inside the workspace (hm_orb.cu orb_geometry)."""
    out, off = [], 0
    for lv in range(n_levels):
        r, c = oo.level_size(h, w, lv)
        stride = (c + 64 + 15) // 16 * 16
        out.append((off, r, c, stride))
        off = (off + stride * (r + 64) + 255) // 256 * 256
    return out, off


@gpu
@pytest.mark.parametrize("h,w,seed,ch", [(480, 640, 7, 1), (480, 752, 11, 3), (333, 517, 13, 1), (120, 90, 5, 1)])
def test_device_pyramid_equals_oracle(h, w, seed, ch):
    img = synth.textured_image(h, w, seed, ch)
    n_levels = 8 if h >= 333 else 3
    ws = nat.orb_build_pyramid(torch.from_numpy(img).cuda(), n_levels).cpu().numpy()
    layout, plane = plane_layout(h, w, n_levels)
    levels = oo.build_pyramid(oo.to_gray(img), n_levels)
    for (off, r, c, stride), ref in zip(layout, levels):
        blurred = ws[256 + plane + off: 256 + plane + off + stride * (r + 64)].reshape(r + 64, stride)[:, :c + 64]
        assert np.array_equal(blurred, ref), (r, c)


@gpu
def test_device_descriptors_equal_reference_and_cv2():
    import slam_experiments_b200 as sx
    for name, img, xy, ang, octv, desc, nf in golden_cases():
        det = sx.OrbFeatureDetector(n_features=nf)
        kps, got = det.detect_and_compute(img, None)              # the reference's call, descriptors on the device
        ref_kps, ref = cv2.ORB.create(nfeatures=nf).detectAndCompute(img, None)
        assert [k.pt for k in kps] == [k.pt for k in ref_kps]
        assert np.array_equal(got, ref) and np.array_equal(got, desc), name
        dev = torch.device("cuda")
        ws = nat.orb_build_pyramid(torch.from_numpy(img).to(dev), 8)
        out = nat.orb_describe(ws, img.shape[:2], 8, torch.from_numpy(xy).to(dev), torch.from_numpy(nat.orb_angles_to_cs(ang)).to(dev),
                               torch.from_numpy(octv).to(dev))
        assert np.array_equal(out.cpu().numpy(), oo.describe(img, xy, ang, octv))
    det = sx.OrbFeatureDetector(n_features=50)
    flat = np.full((200, 200), 128, np.uint8)                     # no corners: cv2 returns ((), None)
    kps, d = det.detect_and_compute(flat, None)
    assert len(kps) == 0 and d is None


@gpu
def test_frames_described_on_device_match_like_cv2_frames():
    """frontend.py:245-249 + :181-187 end to end: two frames are detected by cv2, described on the device straight into
    the resident store, and matched there; equal to cv2 descriptors through the oracle pipeline."""
    import slam_experiments_b200 as sx
    a = synth.textured_image(480, 640, 31)
    b = np.roll(a, (3, 5), axis=(0, 1))
    det = sx.OrbFeatureDetector(n_features=1500)
    for kwargs in ({}, {"ratio": 0.75, "cross_check": True}):
        store = sx.FrameDescriptorStore(**kwargs)
        ka = det.detect_and_store(a, store, "a")
        kb = det.detect_and_store(b, store, "b")
        orb = cv2.ORB.create(nfeatures=1500)
        _, da = orb.compute(a, ka)
        _, db = orb.compute(b, kb)
        q, t, d = store.match_tensors("a", "b")
        eq, et, ed = co.pipeline(db, da, kwargs.get("ratio"), kwargs.get("cross_check", False))
        assert np.array_equal(q, eq) and np.array_equal(t, et) and np.array_equal(d, ed)
        sp, qp = store.matched_points("a", "b")
        pa = np.array([k.pt for k in ka], np.float32).astype(np.int32)
        pb = np.array([k.pt for k in kb], np.float32).astype(np.int32)
        assert np.array_equal(sp, pa[et]) and np.array_equal(qp, pb[eq])
    got = store.put_image("c", a, ka, want_descriptors=True)
    assert np.array_equal(got, da)
    with pytest.raises(nat.NativeError):
        store._ctx.frame_put_orb(0, a[:40], np.zeros((1, 2), np.float32), np.zeros(1, np.float32), np.zeros(1, np.int32))


def test_oracle_describe_random_keypoints_all_octaves():
    """Hand-made keypoints at arbitrary sub-pixel positions, angles and octaves (cv2.ORB.compute takes them as given):
    pins the coordinate rounding (pt * (1 / scale), half to even) and the rotation for angles the detector never emits."""
    img = synth.textured_image(480, 640, 77)
    rng = np.random.default_rng(0)
    kps = []
    for _ in range(400):
        o = int(rng.integers(0, 8))
        s = float(oo.level_scale(o))
        r, c = oo.level_size(480, 640, o)
        kps.append(cv2.KeyPoint(float(rng.uniform(31.5, c - 32.5)) * s, float(rng.uniform(31.5, r - 32.5)) * s, 31.0 * s,
                                float(rng.uniform(0, 360)), 1.0, o))
    kps.sort(key=lambda k: k.octave)
    k2, d = cv2.ORB.create(nfeatures=1000).compute(img, kps)
    assert len(k2) == len(kps)
    assert np.array_equal(oo.describe(img, *kp_arrays(k2)), d)


@gpu
def test_device_describe_random_keypoints_all_octaves():
    """The same hand-made keypoints through hm_orb_describe."""
    img = synth.textured_image(480, 640, 77)
    rng = np.random.default_rng(0)
    xy = np.empty((400, 2), np.float32)
    ang = rng.uniform(0, 360, 400).astype(np.float32)
    octv = np.sort(rng.integers(0, 8, 400)).astype(np.int32)
    for i, o in enumerate(octv):
        s = float(oo.level_scale(int(o)))
        r, c = oo.level_size(480, 640, int(o))
        xy[i] = (float(rng.uniform(31.5, c - 32.5)) * s, float(rng.uniform(31.5, r - 32.5)) * s)
    dev = torch.device("cuda")
    ws = nat.orb_build_pyramid(torch.from_numpy(img).to(dev), 8)
    out = nat.orb_describe(ws, img.shape[:2], 8, torch.from_numpy(xy).to(dev), torch.from_numpy(nat.orb_angles_to_cs(ang)).to(dev),
                           torch.from_numpy(octv).to(dev))
    assert np.array_equal(out.cpu().numpy(), oo.describe(img, xy, ang, octv))
