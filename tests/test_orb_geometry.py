"""ORB descriptor stage across geometry: which image sizes and level counts the library accepts (CPU), every pyramid
level of the device read back stage by stage against a cv2 chain (GPU), rBRIEF at the edges of the keypoint domain
against cv2.ORB.compute and the oracle (GPU), and the frontend calls on small and odd images against
cv2.ORB.detectAndCompute (GPU).

The rule the geometry follows: level L of a rows x cols image is round(rows / 1.2^L) x round(cols / 1.2^L) (float32,
half to even), and a pyramid of n levels is accepted when every level 0 .. n-1 is more than 32 pixels on both sides
(the 32-pixel reflect-101 frame must fit inside it), level 0 is at most 16384 on both sides and 1 <= n <= 16."""
import ctypes

import cv2
import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from oracle import orb_oracle as oo
from slam_experiments_b200 import _native as nat
from slam_experiments_b200 import build as hm_build
from slam_experiments_b200 import synth
from test_orb import kp_arrays, plane_layout

gpu = pytest.mark.gpu

B = oo.BORDER
MAX_LEVELS = 16
AVX2 = cv2.checkHardwareSupport(5)                 # CV_CPU_AVX2: the dispatch whose float blur order the kernels follow
G7 = cv2.getGaussianKernel(7, 2, cv2.CV_32F)


def levels_that_fit(side: int) -> int:
    """How many leading levels of one image side are more than 32 pixels (at most 16)."""
    n = 0
    while n < MAX_LEVELS and oo.level_size(side, side, n)[0] > B:
        n += 1
    return n


def max_levels(h: int, w: int) -> int:
    return min(levels_that_fit(h), levels_that_fit(w))


def smallest_side(n_levels: int) -> int:
    return next(s for s in range(B + 1, 1000) if levels_that_fit(s) >= n_levels)


# ---------------------------------------------------------------- A. host-side domain (no device)
SIDES = [-1, 0, 1] + list(range(28, 141)) + [167, 168, 201, 202, 241, 242, 500, 501, 1080, 1920, 4096, 16383, 16384, 16385]


def test_host_domain_is_every_level_wider_than_the_frame():
    hm_build.build()
    L = nat.lib()
    fit = {s: (levels_that_fit(s) if s <= 16384 else 0) for s in SIDES}
    size = {s: [oo.level_size(s, s, lv)[0] for lv in range(MAX_LEVELS)] for s in SIDES}
    inv = [np.float32(1.0) / oo.level_scale(lv) for lv in range(MAX_LEVELS)]
    r_, c_, inv_ = ctypes.c_int(), ctypes.c_int(), ctypes.c_float()
    exact = {33, 40, 64, 95, 117, 501, 1080}
    accepted = rejected = 0
    for r in SIDES:
        for c in SIDES:
            for n in range(-1, MAX_LEVELS + 2):
                ok = 1 <= n <= min(fit[r], fit[c])
                got = L.hm_orb_workspace_bytes(r, c, n)
                assert (got != 0) == ok, (r, c, n, got)
                if ok and r in exact and c in exact:
                    assert got == 256 + 2 * plane_layout(r, c, n)[1], (r, c, n)
                accepted += ok
                rejected += not ok
            for lv in range(-1, MAX_LEVELS + 1):
                ok = 0 <= lv < min(fit[r], fit[c])
                r_.value = c_.value = -7
                rc = L.hm_orb_level_geometry(r, c, lv, ctypes.byref(r_), ctypes.byref(c_), ctypes.byref(inv_))
                assert (rc == 0) == ok, (r, c, lv, rc)
                if ok:
                    assert (r_.value, c_.value) == (size[r][lv], size[c][lv]), (r, c, lv)
                    assert np.float32(inv_.value) == inv[lv], (r, c, lv)
    assert accepted > 50000 and rejected > 50000
    # the smallest accepted sides, and one less: every level count has its own boundary
    for n in range(1, MAX_LEVELS + 1):
        s = smallest_side(n)
        assert L.hm_orb_workspace_bytes(s, 4096, n) and L.hm_orb_workspace_bytes(4096, s, n)
        assert not L.hm_orb_workspace_bytes(s - 1, 4096, n) and not L.hm_orb_workspace_bytes(4096, s - 1, n)


# ---------------------------------------------------------------- B. the pyramid, stage by stage (GPU)
def cv2_pyramid(img: np.ndarray, n_levels: int):
    """(raw framed levels, blurred framed levels) computed by cv2: cvtColor, a chain of INTER_LINEAR_EXACT resizes each
    from the previous level, the reflect-101 frame, and the float sepFilter2D of the interior (the frame stays
    un-blurred).  Without AVX2 cv2 runs another dispatch of the float filter, so the blur comes from the oracle."""
    gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if img.ndim == 3 else np.ascontiguousarray(img)
    levels = [gray]
    for lv in range(1, n_levels):
        r, c = oo.level_size(gray.shape[0], gray.shape[1], lv)
        levels.append(cv2.resize(levels[-1], (c, r), interpolation=cv2.INTER_LINEAR_EXACT))
    raw = [cv2.copyMakeBorder(lv, B, B, B, B, cv2.BORDER_REFLECT_101) for lv in levels]
    if not AVX2:
        return raw, oo.build_pyramid(gray, n_levels)
    blurred = []
    for framed, lv in zip(raw, levels):
        b = framed.copy()
        b[B:-B, B:-B] = cv2.sepFilter2D(lv, cv2.CV_8U, G7, G7, borderType=cv2.BORDER_REFLECT_101)
        blurred.append(b)
    return raw, blurred


def device_planes(image: torch.Tensor, n_levels: int):
    """Both planes of the workspace hm_orb_build_pyramid filled: the raw framed levels at ws + 256 and the blurred ones
    at ws + 256 + plane_bytes, each level [rows + 64, cols + 64] (the row padding up to the stride is left out)."""
    h, w = int(image.shape[0]), int(image.shape[1])
    ws = nat.orb_build_pyramid(image, n_levels).cpu().numpy()
    layout, plane = plane_layout(h, w, n_levels)
    assert ws.size == 256 + 2 * plane
    raw, blurred = [], []
    for off, r, c, stride in layout:
        for base, dst in ((256, raw), (256 + plane, blurred)):
            dst.append(ws[base + off: base + off + stride * (r + 2 * B)].reshape(r + 2 * B, stride)[:, :c + 2 * B])
    return raw, blurred


def assert_same(got: np.ndarray, ref: np.ndarray, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bad = np.argwhere(got != ref)
    assert bad.shape[0] == 0, f"{what}: {bad.shape[0]} differing bytes, first at {tuple(bad[0])}"


def pyramid_cases():
    """(h, w, channels, n_levels, crop): crop > 0 makes the image a column slice of a tensor `crop` pixels wider."""
    cases = []
    for i, w in enumerate(range(64, 96)):              # level-0 widths: every residue mod 32 and mod 4
        h = 41 + 3 * i                                  # odd and even heights
        cases.append((h, w, 3 if i % 4 == 3 else 1, max_levels(h, w), 0))
    cases += [(333, 517, 1, 8, 0), (481, 777, 3, max_levels(481, 777), 0), (1080, 1920, 1, 16, 0), (1080, 1920, 3, 16, 0)]
    cases += [(531, 709, 1 + 2 * (n % 2), n, 0) for n in range(1, MAX_LEVELS + 1)]
    for n in (1, 2, 3, 4, 6, 8, 12, 16):                # the smallest accepted image for the level count
        s = smallest_side(n)
        cases += [(s, s, 1, n, 0), (s, 3 * s + 1, 3, n, 0)]
    cases += [(33, 4096, 1, 1, 0), (4096, 40, 1, 2, 0), (4096, 33, 3, 1, 0), (34, 2048, 3, 1, 0), (40, 3001, 1, 2, 0)]
    cases += [(97, 200, 1, max_levels(97, 200), 63), (150, 301, 3, max_levels(150, 301), 49), (1080, 1920, 1, 8, 80)]
    return cases


PYRAMID_CASES = pyramid_cases()


def test_pyramid_cases_cover_the_geometry_rules():
    """The device cases below reach every width residue of the blur's vector bodies (mod 32 for the row pass, mod 4
    for the column pass) on some level, odd and even level heights, every level count, BGR and strided input."""
    widths, heights = set(), set()
    for h, w, ch, n, crop in PYRAMID_CASES:
        assert 1 <= n <= max_levels(h, w), (h, w, n)
        for lv in range(n):
            r, c = oo.level_size(h, w, lv)
            widths.add(c)
            heights.add(r)
    assert {c % 32 for c in widths} == set(range(32))
    assert {r % 2 for r in heights} == {0, 1}
    assert {n for *_, n, _ in PYRAMID_CASES} == set(range(1, MAX_LEVELS + 1))
    assert {ch for _, _, ch, _, _ in PYRAMID_CASES} == {1, 3}
    assert any(crop for *_, crop in PYRAMID_CASES)


@gpu
@pytest.mark.parametrize("h,w,ch,n_levels,crop", PYRAMID_CASES,
                         ids=[f"{h}x{w}x{ch}_L{n}" + (f"_crop{c}" if c else "") for h, w, ch, n, c in PYRAMID_CASES])
def test_device_pyramid_equals_cv2_level_by_level(h, w, ch, n_levels, crop):
    full = np.ascontiguousarray(synth.textured_image(h, w + crop, h * 7919 + w + ch, ch))
    img = full[:, crop // 3: crop // 3 + w]
    image = torch.from_numpy(full).cuda()[:, crop // 3: crop // 3 + w]
    if crop:
        assert image.stride(0) > w * ch                 # the row stride reaches the kernel as it is
    raw, blurred = device_planes(image, n_levels)
    raw_ref, blurred_ref = cv2_pyramid(img, n_levels)
    for lv in range(n_levels):
        assert_same(raw[lv], raw_ref[lv], f"raw level {lv}")
        assert_same(blurred[lv], blurred_ref[lv], f"blurred level {lv}")
    if h * w <= 200000:
        for lv, ref in enumerate(oo.build_pyramid(oo.to_gray(img), n_levels)):
            assert_same(blurred[lv], ref, f"blurred level {lv} against the oracle")


@gpu
def test_device_gray_conversion_of_every_bgr_triple():
    """4096 x 4096 BGR holding each of the 2^24 (B, G, R) triples once: the raw level 0 is cv2.cvtColor, framed."""
    idx = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([idx & 255, (idx >> 8) & 255, idx >> 16], axis=1).astype(np.uint8).reshape(4096, 4096, 3)
    raw, _ = device_planes(torch.from_numpy(img).cuda(), 1)
    gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    assert_same(raw[0][B:-B, B:-B], gray, "gray interior")
    assert_same(raw[0], cv2.copyMakeBorder(gray, B, B, B, B, cv2.BORDER_REFLECT_101), "gray framed")


# ---------------------------------------------------------------- C. rBRIEF at the edges of the keypoint domain (GPU)
EH, EW = 1080, 1920                                 # every one of the 16 levels fits
EDGE_ANGLES = np.array([0, 45, 90, 135, 180, 225, 270, 315, 360, -0.0, 359.9999], np.float32)


def level_point(o: int, t, exact: bool) -> np.float32:
    """A float32 level-0 coordinate x with x * (1 / scale of level o) in float32 equal to t (exact) or rounding to t."""
    inv = np.float32(1.0) / oo.level_scale(o)
    base = np.float32(float(t) * float(oo.level_scale(o))).view(np.int32)
    for d in (0, -1, 1, -2, 2, -3, 3):
        x = np.int32(base + d).view(np.float32)
        p = x * inv
        if (p == np.float32(t)) if exact else (np.rint(p) == t):
            return x
    return None


def half_pixel_targets(size: int, o: int):
    """Level coordinates k + 0.5 that some float32 level-0 coordinate maps onto exactly: the first and last two with
    k even and with k odd (round half to even sends them to k and k + 1)."""
    inv = np.float32(1.0) / oo.level_scale(o)
    k = np.arange(B - 1, size - B)
    target = (k + 0.5).astype(np.float32)
    base = (target.astype(np.float64) * float(oo.level_scale(o))).astype(np.float32).view(np.int32)
    hit = np.zeros(k.shape, bool)
    for d in range(-3, 4):
        hit |= (np.int32(base + d).view(np.float32) * inv) == target
    out = []
    for parity in (0, 1):
        ks = k[hit & (k % 2 == parity)]
        out += sorted(set(ks[:2].tolist() + ks[-2:].tolist()))
    return [kk + 0.5 for kk in out]


def sort_by_octave(xy, ang, octv):
    o = np.argsort(octv, kind="stable")              # cv2.ORB.compute returns its keypoints grouped by octave
    return np.ascontiguousarray(xy[o]), np.ascontiguousarray(ang[o]), np.ascontiguousarray(octv[o])


def edge_keypoints():
    """Keypoints on every octave 0..15 of an EH x EW image: the nine combinations of {31, middle, size - 32} on both
    axes (the extremes cv2's detector can emit), exact half-pixel level positions on each axis, and every edge angle."""
    xy, ang, octv = [], [], []
    rng = np.random.default_rng(5)
    halves = {"x": 0, "y": 0, "even": 0, "odd": 0}

    def add(o, tx, ty, a, exact_x=False, exact_y=False):
        px, py = level_point(o, tx, exact_x), level_point(o, ty, exact_y)
        assert px is not None and py is not None, (o, tx, ty)
        xy.append((px, py)); ang.append(a); octv.append(o)

    for o in range(MAX_LEVELS):
        r, c = oo.level_size(EH, EW, o)
        for tx in (B - 1, c // 2, c - B):
            for ty in (B - 1, r // 2, r - B):
                add(o, tx, ty, np.float32(rng.uniform(0, 360)))
        for tx in half_pixel_targets(c, o):
            add(o, tx, r // 2, np.float32(rng.uniform(0, 360)), exact_x=True)
            halves["x"] += 1
            halves["even" if int(tx) % 2 == 0 else "odd"] += 1
        for ty in half_pixel_targets(r, o):
            add(o, c // 2 + 1, ty, np.float32(rng.uniform(0, 360)), exact_y=True)
            halves["y"] += 1
            halves["even" if int(ty) % 2 == 0 else "odd"] += 1
        for a in EDGE_ANGLES:
            add(o, c // 3, r // 3, a)
    xy, ang, octv = np.array(xy, np.float32), np.array(ang, np.float32), np.array(octv, np.int32)
    assert set(octv.tolist()) == set(range(MAX_LEVELS))
    assert min(halves.values()) >= 4 * MAX_LEVELS, halves
    return sort_by_octave(xy, ang, octv)


def random_keypoints(n: int, seed: int):
    """n keypoints on uniformly drawn octaves 0..15, anywhere cv2's detector could put one."""
    rng = np.random.default_rng(seed)
    octv = rng.integers(0, MAX_LEVELS, n).astype(np.int32)
    scale = np.array([oo.level_scale(o) for o in range(MAX_LEVELS)], np.float64)[octv]
    size = np.array([oo.level_size(EH, EW, o) for o in range(MAX_LEVELS)], np.float64)[octv]
    xl = rng.uniform(B - 1, size[:, 1] - B)
    yl = rng.uniform(B - 1, size[:, 0] - B)
    xy = np.stack([xl * scale, yl * scale], 1).astype(np.float32)
    return sort_by_octave(xy, rng.uniform(0, 360, n).astype(np.float32), octv)


def cv2_describe(img, xy, ang, octv):
    """cv2.ORB.compute of hand-made keypoints; cv2 must return exactly the keypoints it was given (its border filter
    removed none)."""
    kps = [cv2.KeyPoint(float(x), float(y), 31.0, float(a), 0.0, int(o)) for (x, y), a, o in zip(xy, ang, octv)]
    k2, desc = cv2.ORB.create(nlevels=MAX_LEVELS).compute(img, kps)
    assert len(k2) == len(kps)
    gxy, gang, goct = kp_arrays(k2)
    assert np.array_equal(gxy, xy) and np.array_equal(gang, ang) and np.array_equal(goct, octv)
    return desc


def test_oracle_equals_cv2_at_the_keypoint_edges():
    img = synth.textured_image(EH, EW, 41)
    xy, ang, octv = edge_keypoints()
    assert np.array_equal(oo.describe(img, xy, ang, octv), cv2_describe(img, xy, ang, octv))


@gpu
def test_device_describe_edges_equal_cv2_and_oracle():
    img = synth.textured_image(EH, EW, 41)
    dev = torch.device("cuda")
    ws = nat.orb_build_pyramid(torch.from_numpy(img).to(dev), MAX_LEVELS)
    sets = {"edges": edge_keypoints()}
    for n, seed in ((1, 1), (7, 2), (8, 3), (9, 4), (100003, 5)):    # 8 keypoints per block: tails and a large grid
        sets[f"n={n}"] = random_keypoints(n, seed)
    oracle_part = []
    for name, (xy, ang, octv) in sets.items():
        n = xy.shape[0]
        buf = torch.full((n + 9, 32), 0xA5, dtype=torch.uint8, device=dev)
        nat.orb_describe(ws, img.shape, MAX_LEVELS, torch.from_numpy(xy).to(dev), torch.from_numpy(nat.orb_angles_to_cs(ang)).to(dev),
                         torch.from_numpy(octv).to(dev), out=buf[:n])
        got = buf.cpu().numpy()
        assert (got[n:] == 0xA5).all(), f"{name}: rows past n written"
        assert_same(got[:n], cv2_describe(img, xy, ang, octv), f"{name} against cv2")
        keep = slice(None) if n < 1000 else slice(None, None, 97)     # the oracle is slow: a subset of the large set
        oracle_part.append((xy[keep], ang[keep], octv[keep], got[:n][keep]))
    xy, ang, octv, got = (np.concatenate(a) for a in zip(*oracle_part))
    assert_same(got, oo.describe(img, xy, ang, octv), "against the oracle")


# ---------------------------------------------------------------- D. drop-in on small and odd images (GPU)
def small_image(h, w, ch, kind, seed):
    if kind == "noise":                             # 63-pixel-tall textures give cv2 too few corners; noise gives plenty
        return np.random.default_rng(seed).integers(0, 256, (h, w) if ch == 1 else (h, w, 3), dtype=np.uint8)
    return np.ascontiguousarray(synth.textured_image(h, w, seed, ch))


SMALL_CASES = [(63, 300, 1, "noise", 0), (63, 640, 1, "noise", 0), (80, 80, 1, "texture", 0), (100, 130, 1, "texture", 0),
               (110, 640, 1, "texture", 0), (640, 70, 1, "texture", 0), (100, 130, 3, "texture", 0), (63, 400, 3, "noise", 0),
               (110, 640, 1, "texture", 37), (80, 80, 3, "noise", 11)]


@gpu
@pytest.mark.parametrize("h,w,ch,kind,crop", SMALL_CASES,
                         ids=[f"{h}x{w}x{ch}_{k}" + (f"_crop{c}" if c else "") for h, w, ch, k, c in SMALL_CASES])
def test_small_images_describe_like_cv2(h, w, ch, kind, crop):
    """OrbFeatureDetector and FrameDescriptorStore.put_image on images whose lower default levels do not fit: the
    pyramid has max(octave) + 1 levels, as cv2 builds it for given keypoints.  crop > 0 makes the image a numpy view
    with a padded row stride."""
    import slam_experiments_b200 as sx
    full = small_image(h, w + crop, ch, kind, h * 31 + w + ch)
    img = full[:, crop // 2: crop // 2 + w]
    assert img.strides[0] == (w + crop) * ch
    orb = cv2.ORB.create(nfeatures=500)
    ref_kps, ref = orb.detectAndCompute(img, None)
    assert len(ref_kps) > 0
    det = sx.OrbFeatureDetector(n_features=500)
    kps, got = det.detect_and_compute(img, None)
    assert [(k.pt, k.octave) for k in kps] == [(k.pt, k.octave) for k in ref_kps]
    assert_same(got, ref, "detect_and_compute")
    assert_same(det.compute(img, kps), ref, "compute")
    b = np.roll(img, (2, 3), axis=(0, 1))
    for kwargs in ({}, {"ratio": 0.75, "cross_check": True}):
        store = sx.FrameDescriptorStore(**kwargs)
        ka = det.detect_and_store(img, store, "a")
        kb = det.detect_and_store(b, store, "b")
        assert [k.pt for k in ka] == [k.pt for k in ref_kps] and len(kb) > 0
        assert_same(store.put_image("c", img, ka, want_descriptors=True), ref, "put_image")
        _, db = orb.compute(b, kb)
        q, t, d = store.match_tensors("a", "b")
        eq, et, ed = co.pipeline(db, ref, kwargs.get("ratio"), kwargs.get("cross_check", False))
        assert np.array_equal(q, eq) and np.array_equal(t, et) and np.array_equal(d, ed), kwargs
