"""The buffer contract of the C ABI: where the library reads and writes, not only what it computes.

The parity suites compare values.  They cannot see a launch that needs more workspace than its sizing function
reports (the cached workspace of ``_native.workspace`` always has slack behind it), a kernel that writes past an
output, a kernel that reads workspace it did not initialise in the same call, or one that reads input rows outside
the problem.  Every test here calls the library through ``nat.lib().hm_*`` on torch's current stream with buffers
the test lays out itself:

  - every workspace has exactly the size its sizing function reports, and every device buffer the library writes
    sits inside 1 MiB guard bands of seeded random bytes (``Guarded``) that must be byte-identical afterwards;
  - host outputs of the ``_host`` entry points sit between guard elements (``HostGuarded``);
  - workspaces start at offset 0 and at offset 16 modulo 256 (the 16-byte alignment the header promises), and are
    pre-filled with a seeded random pattern or with 0xFF: everything a kernel reads must be written by the same call;
  - inputs are compared with a copy after the call: the library never writes them;
  - poisoned inputs: tail rows, stride gaps, the padding rows of prepared images and the unselected rows of a
    selection hold rows that would win if a kernel read them.

Results are compared with oracle/c_oracle.py (or the ORB oracle) bit for bit.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from oracle import hamming_oracle as ho

gpu = pytest.mark.gpu
GUARD = 1 << 20                 # bytes of guard band on each side of a device buffer
HOST_GUARD = 1 << 16            # bytes of guard on each side of a host array
OFFSETS = (0, 16)
NO_MATCH = np.uint64(0xFFFFFFFFFFFFFFFF)
LOW32 = np.uint64(0xFFFFFFFF)
# (workspace offset, pre-fill) of the two runs every workspace case gets: each poison once, each offset once
POISONS = ((0, "random"), (16, 0xFF))
HM_ERR_WORKSPACE = -3


# =====================================================================================================================
# helpers
# =====================================================================================================================
def _pattern(n, seed, device):
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    return torch.randint(0, 256, (int(n),), dtype=torch.uint8, device=device, generator=g)


def _span(bad):
    return (int(bad[0]), int(bad[-1])) if bad.numel() else None


class Guarded:
    """A view of exactly ``nbytes`` inside one CUDA uint8 allocation, with a guard band of at least ``GUARD`` bytes of a
    seeded random pattern on each side.  The view starts at ``offset`` modulo 256.  Its own bytes hold the same kind of
    pattern unless ``fill`` is a byte value."""

    def __init__(self, nbytes, offset=0, seed=0, fill=None):
        self.nbytes, self.offset = int(nbytes), int(offset)
        self.raw = _pattern(2 * GUARD + 256 + self.nbytes, seed, "cuda")
        self.start = GUARD + ((self.offset - self.raw.data_ptr()) % 256)
        assert (self.raw.data_ptr() + self.start) % 256 == self.offset % 256
        self.end = self.start + self.nbytes
        self.view = self.raw[self.start:self.end]
        if fill not in (None, "random"):
            self.view.fill_(int(fill))
        self.front = self.raw[:self.start].clone()
        self.back = self.raw[self.end:].clone()

    @property
    def ptr(self):
        return self.view.data_ptr()

    def as_(self, dtype, shape):
        return self.view.view(dtype).view(shape)

    def check_guards(self, what=""):
        torch.cuda.synchronize()
        fb = torch.nonzero(self.raw[:self.start] != self.front).flatten() - self.start
        bb = torch.nonzero(self.raw[self.end:] != self.back).flatten()
        assert not fb.numel() and not bb.numel(), (
            f"{what}: guard bands of a {self.nbytes}-byte buffer (offset {self.offset}) overwritten: "
            f"before the start at {_span(fb)} (first, last byte relative to the start), "
            f"after the end at {_span(bb)} (first, last byte relative to the end)")


class HostGuarded:
    """numpy twin of ``Guarded``: an array of ``shape`` / ``dtype`` between ``HOST_GUARD`` bytes of seeded random
    bytes on each side (its own bytes hold the same pattern)."""

    def __init__(self, shape, dtype, seed=0):
        dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(shape)) * dtype.itemsize
        self.raw = np.random.default_rng(seed).integers(0, 256, 2 * HOST_GUARD + self.nbytes, dtype=np.uint8)
        self.pattern = self.raw.copy()
        self.a = self.raw[HOST_GUARD:HOST_GUARD + self.nbytes].view(dtype).reshape(shape)

    @property
    def ptr(self):
        return self.a.ctypes.data

    def check_guards(self, what=""):
        fb = np.flatnonzero(self.raw[:HOST_GUARD] != self.pattern[:HOST_GUARD]) - HOST_GUARD
        bb = np.flatnonzero(self.raw[HOST_GUARD + self.nbytes:] != self.pattern[HOST_GUARD + self.nbytes:])
        assert not fb.size and not bb.size, (
            f"{what}: host guards of a {self.nbytes}-byte array overwritten: before the start at "
            f"{(int(fb[0]), int(fb[-1])) if fb.size else None}, after the end at "
            f"{(int(bb[0]), int(bb[-1])) if bb.size else None}")


def lib():
    from slam_experiments_b200 import _native as nat
    return nat.lib()


def call(fn, *args):
    from slam_experiments_b200 import _native as nat
    rc = getattr(lib(), fn)(*args)
    assert rc == nat.HM_OK, f"{fn} returned {rc}: {nat.last_error()}"


def stream():
    return torch.cuda.current_stream().cuda_stream


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def with_ptr(t):
    return t, t.data_ptr()


class Frozen:
    """Copies of a call's inputs: ``check()`` asserts that the library wrote none of them."""

    def __init__(self, **inputs):
        self.items = {k: (v, v.clone()) for k, v in inputs.items()}

    def check(self, what=""):
        torch.cuda.synchronize()
        for k, (v, c) in self.items.items():
            assert torch.equal(v, c), f"{what}: the library wrote its input {k}"


def u64(t):
    return t.cpu().numpy().view(np.uint64)


def planted(nq, nt, seed, hi=256):
    """random train rows and queries of which half are train rows with a few bits flipped (clear nearest rows)"""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, hi, (nt, 32), dtype=np.uint8)
    q = rng.integers(0, hi, (nq, 32), dtype=np.uint8)
    m = nq // 2
    if nt and m:
        q[:m] = t[rng.integers(0, nt, m)] ^ (rng.integers(0, 16, (m, 32), dtype=np.uint8) == 0).astype(np.uint8)
    return q, t


def keys_equal(got, exp, what):
    bad = np.flatnonzero((got != exp).any(axis=-1).reshape(-1))
    assert bad.size == 0, f"{what}: {bad.size} rows differ from the oracle, first {bad[:5]}: got " \
                          f"{got.reshape(-1, 2)[bad[:2]].tolist()}, oracle {exp.reshape(-1, 2)[bad[:2]].tolist()}"


def matches_equal(got, exp, what):
    gq, gt, gd = got
    eq, et, ed = exp
    assert len(gq) == len(eq), f"{what}: {len(gq)} matches, oracle {len(eq)}"
    assert np.array_equal(gq, eq) and np.array_equal(gt, et) and np.array_equal(gd, ed), what


def variant_id(v):
    from slam_experiments_b200 import _native as nat
    return nat.variant_id(v)


def tensor_variant(v):
    from slam_experiments_b200 import _native as nat
    return nat.tensor_variant(v)


def padded_rows(n, v):
    from slam_experiments_b200 import _native as nat
    return lib().hm_prepared_bytes(n, v) // nat.PREPARED_ROW_BYTES[v]


def prepare(rows, v):
    from slam_experiments_b200 import _native as nat
    return nat.prepare(dev(rows), variant=v)


def poisoned_image(t, q, v):
    """The prepared image of ``t`` whose padding rows ``[nt, padded)`` hold the images of query rows, followed by the
    prepared image of the queries: a kernel that reads past row nt finds exact copies of the queries."""
    nt = t.shape[0]
    pad = padded_rows(nt, v) - nt
    img = prepare(np.concatenate([t, q[np.arange(pad) % q.shape[0]]]), v)
    assert img.numel() == lib().hm_prepared_bytes(nt, v)
    return torch.cat([img, prepare(q, v)])


def poisoned_rows(rows, filler, stride, tail=64):
    """``rows`` at ``stride`` bytes apart in a device buffer whose stride gaps and ``tail`` rows after the last one hold
    rows of ``filler`` (the gap of a 48-byte stride holds the first 16 bytes of one).  Returns (buffer, base pointer)."""
    n = rows.shape[0]
    fill = filler[np.arange(n + tail) % filler.shape[0]]
    slots = np.zeros((n + tail, stride), np.uint8)
    slots[:n, :32] = rows
    slots[n:, :32] = fill[n:]
    slots[:, 32:] = fill[:, :stride - 32]
    buf = dev(slots.reshape(-1))
    return buf, buf.data_ptr()


# =====================================================================================================================
# CPU: the checkers themselves
# =====================================================================================================================
def test_host_guards_report_the_overrun():
    g = HostGuarded((7, 2), np.int32, seed=3)
    g.a[:] = 5
    g.check_guards("in bounds")
    g.raw[HOST_GUARD + g.nbytes + 3] ^= 1
    with pytest.raises(AssertionError, match=r"after the end at \(3, 3\)"):
        g.check_guards("overrun")
    h = HostGuarded((4,), np.uint64, seed=4)
    h.raw[HOST_GUARD - 2] ^= 1
    with pytest.raises(AssertionError, match=r"before the start at \(-2, -2\)"):
        h.check_guards("underrun")


# =====================================================================================================================
# A + B + C: k-NN entry points
# =====================================================================================================================
def run_knn2(q, t, variant, offset, fill, seed=0, q_stride=32, t_stride=32, qbuf=None, tbuf=None):
    """hm_knn2 (2-D inputs) or hm_knn2_batched ([B, n, 32]) with an exact-size guarded workspace and guarded keys.
    ``qbuf`` / ``tbuf``: (buffer, pointer) of a strided device layout of q / t instead of contiguous copies."""
    batched = q.ndim == 3
    b = q.shape[0] if batched else 1
    nq, nt = q.shape[-2], t.shape[-2]
    v = variant_id(variant)
    qd, qp = qbuf if qbuf is not None else with_ptr(dev(q))
    td, tp = tbuf if tbuf is not None else with_ptr(dev(t))
    wsb = lib().hm_workspace_bytes(nq, nt, b, v)
    ws = Guarded(wsb, offset, seed, fill)
    out = Guarded(b * nq * 16, offset, seed + 1)
    frozen = Frozen(query=qd, train=td)
    if batched:
        call("hm_knn2_batched", qp, nq, 32, nq * 32, tp, nt, 32, nt * 32, b, out.ptr, v, ws.ptr, wsb, stream())
    else:
        call("hm_knn2", qp, nq, q_stride, tp, nt, t_stride, 0, out.ptr, v, ws.ptr, wsb, stream())
    what = f"hm_knn2 {b}x{nq}x{nt} {variant} offset={offset} fill={fill}"
    ws.check_guards(what + " workspace")
    out.check_guards(what + " keys")
    frozen.check(what)
    return u64(out.as_(torch.int64, (b, nq, 2) if batched else (nq, 2))), what


KNN_CASES = [(nq, nt, 1, v) for nq, nt in ((1, 1), (3, 1), (127, 129), (257, 255)) for v in ("popc", "i8", "f4", "auto")]
KNN_CASES += [(300, 40000, 1, v) for v in ("popc", "i8", "f4", "auto")]        # split launches, floor kernels
KNN_CASES += [(100, 100000, 1, "popc")]                                          # POPC splits
KNN_CASES += [(333, 20011, 3, v) for v in ("popc", "i8", "f4")]                  # batched
KNN_CASES += [(2000, 4000, 1, "auto"), (1999, 4000, 1, "auto")]                  # both sides of AUTO's 8e6 switch


@gpu
@pytest.mark.parametrize("nq,nt,batch,variant", KNN_CASES)
def test_knn2_exact_workspace(nq, nt, batch, variant):
    if (nq, nt) == (2000, 4000):
        from slam_experiments_b200 import _native as nat
        assert nat.select_variant(2000, 4000) == "f4" and nat.select_variant(1999, 4000) == "popc"
    rng = np.random.default_rng(nq * 7 + nt)
    if batch == 1:
        q, t = planted(nq, nt, nq + nt)
        exp = co.knn2_keys(q, t)
    else:
        pr = [planted(nq, nt, s) for s in range(batch)]
        q, t = np.stack([p[0] for p in pr]), np.stack([p[1] for p in pr])
        exp = np.stack([co.knn2_keys(q[i], t[i]) for i in range(batch)])
    for offset, fill in POISONS:
        got, what = run_knn2(q, t, variant, offset, fill, seed=int(rng.integers(1 << 30)))
        keys_equal(got, exp, what)


@gpu
def test_knn2_f4_cluster_pair_exact_workspace():
    from slam_experiments_b200 import _native as nat
    nq, nt = 2000, 2_500_000
    assert "cluster=2" in nat.describe_launch(nq, nt, 1, "f4"), nat.describe_launch(nq, nt, 1, "f4")
    q, t = planted(nq, nt, 99)
    exp = co.knn2_keys(q[::8], t)
    for offset, fill in POISONS:
        got, what = run_knn2(q, t, "f4", offset, fill, seed=5)
        keys_equal(got[::8], exp, what)


@gpu
@pytest.mark.parametrize("variant", ("popc", "i8", "f4", "auto"))
@pytest.mark.parametrize("stride", (48, 64))
@pytest.mark.parametrize("nq,nt", ((257, 255), (300, 40000), (2000, 4000)))
def test_knn2_ignores_rows_outside_its_inputs(nq, nt, stride, variant):
    """Train rows at ``stride`` bytes in a buffer whose gaps and tail hold copies of the queries; the queries likewise
    with copies of train rows: any read outside the nq x nt problem finds a row at distance 0."""
    q, t = planted(nq, nt, 3 * nq + nt)
    exp = co.knn2_keys(q, t)
    qb = poisoned_rows(q, t, stride)
    tb = poisoned_rows(t, q, stride)
    got, what = run_knn2(q, t, variant, 16, "random", seed=9, q_stride=stride, t_stride=stride, qbuf=qb, tbuf=tb)
    keys_equal(got, exp, what + f" stride={stride}")


# ---- hm_match_fused ----------------------------------------------------------------------------------------------
FLAG_SETS = [(ratio, cross, thr) for ratio in (None, 0.8) for cross in (False, True) for thr in (None, 12.5)]


def expected_fused(q, t, ratio, cross, thr):
    from test_pipeline_edges import expected
    return expected(q, t, ratio, cross, thr)


def run_fused(q, t, variant, ratio, cross, thr, want_keys, offset, fill, seed=0, strided=None):
    """hm_match_fused on [B, n, 32] problems, exact-size guarded workspace, every output guarded.  ``strided``:
    (stride) lays out batch-1 q / t as ``poisoned_rows`` views.  Returns [(q, t, d)] per problem and the keys."""
    from slam_experiments_b200 import _native as nat
    b, nq, nt = q.shape[0], q.shape[1], t.shape[1]
    v = variant_id(variant)
    if strided:
        qd, qp = poisoned_rows(q[0], t[0], strided)
        td, tp = poisoned_rows(t[0], q[0], strided)
        qs = ts = strided
    else:
        qd, td = dev(q), dev(t)
        qp, tp, qs, ts = qd.data_ptr(), td.data_ptr(), 32, 32
    flags = (nat.FLAG_RATIO if ratio is not None else 0) | (nat.FLAG_MUTUAL if cross else 0) | \
            (nat.FLAG_DIST_THRESHOLD if thr else 0)
    lut = nat.ratio_lut(ratio) if ratio is not None else None
    wsb = lib().hm_workspace_bytes(nq, nt, b, v)
    ws = Guarded(wsb, offset, seed, fill)
    outs = [Guarded(b * nq * 4, offset, seed + 1 + i) for i in range(3)]
    cnt = Guarded(b * 4, offset, seed + 4)
    keys = Guarded(b * nq * 16, offset, seed + 5) if want_keys else None
    frozen = Frozen(query=qd, train=td)
    call("hm_match_fused", qp, nq, qs, nq * qs, tp, nt, ts, nt * ts, b, flags,
         lut.ctypes.data if lut is not None else None, float(thr or 0.0), outs[0].ptr, outs[1].ptr, outs[2].ptr, cnt.ptr,
         keys.ptr if keys else None, v, ws.ptr, wsb, stream())
    what = f"hm_match_fused {b}x{nq}x{nt} {variant} ratio={ratio} cross={cross} thr={thr} keys={want_keys} " \
           f"offset={offset} fill={fill}"
    for g, name in zip([ws, *outs, cnt] + ([keys] if keys else []), ("workspace", "q", "t", "d", "count", "keys")):
        g.check_guards(f"{what} {name}")
    frozen.check(what)
    n = cnt.as_(torch.int32, (b,)).cpu().numpy()
    oq, ot, od = (o.as_(torch.int32, (b, nq)).cpu().numpy() for o in outs)
    res = [(oq[i, :n[i]], ot[i, :n[i]], od[i, :n[i]]) for i in range(b)]
    return res, (u64(keys.as_(torch.int64, (b, nq, 2))) if keys else None), what


def check_fused(q, t, variant, ratio, cross, thr, want_keys, seed=0, poisons=POISONS, strided=None):
    exp = [expected_fused(q[i], t[i], ratio, cross, thr) for i in range(q.shape[0])]
    kexp = np.stack([co.knn2_keys(q[i], t[i]) for i in range(q.shape[0])]) if want_keys else None
    for offset, fill in poisons:
        res, keys, what = run_fused(q, t, variant, ratio, cross, thr, want_keys, offset, fill, seed, strided)
        for i in range(q.shape[0]):
            matches_equal(res[i], exp[i], f"{what} problem {i}")
        if want_keys:
            keys_equal(keys, kexp, what)


@gpu
@pytest.mark.parametrize("variant", ("popc", "i8", "f4", "auto"))
@pytest.mark.parametrize("batch", (1, 3))
def test_match_fused_exact_workspace_every_flag_set(batch, variant):
    pr = [planted(300, 500, 40 + s) for s in range(batch)]
    q, t = np.stack([p[0] for p in pr]), np.stack([p[1] for p in pr])
    for i, (ratio, cross, thr) in enumerate(FLAG_SETS):
        for want_keys in (False, True):
            check_fused(q, t, variant, ratio, cross, thr, want_keys, seed=i)


@gpu
def test_match_fused_f4_candidate_pass_exact_workspace():
    pr = [planted(10000, 10000, 50 + s) for s in range(2)]
    q, t = np.stack([p[0] for p in pr]), np.stack([p[1] for p in pr])
    for ratio in (None, 0.8):
        check_fused(q, t, "f4", ratio, True, None, ratio is None, seed=7)


@gpu
def test_match_fused_auto_mixed_dispatch():
    """AUTO at 60000 x 150 with the mutual check: the forward pass resolves to POPC (nt < 256), the swapped 150 x 60000
    pass to the kind::mxf4 top-1 kernel."""
    from slam_experiments_b200 import _native as nat
    assert nat.select_variant(60000, 150) == "popc" and nat.select_variant(150, 60000) == "f4"
    q, t = planted(60000, 150, 61)
    for ratio in (None, 0.8):
        check_fused(q[None], t[None], "auto", ratio, True, None, True, seed=11)


@gpu
@pytest.mark.parametrize("variant", ("popc", "i8", "f4", "auto"))
@pytest.mark.parametrize("stride", (48, 64))
def test_match_fused_ignores_rows_outside_its_inputs(stride, variant):
    """the swapped pass scans the queries as columns: their gaps and tail hold train rows"""
    q, t = planted(700, 3000, 62)
    for ratio in (None, 0.8):
        check_fused(q[None], t[None], variant, ratio, True, None, True, seed=13, poisons=((16, "random"),),
                    strided=stride)


# ---- hm_prepare, hm_knn2_prepared, hm_knn2_prepared_partials, hm_merge_top2 ---------------------------------------
@gpu
@pytest.mark.parametrize("variant", ("i8", "f4"))
def test_prepare_writes_exactly_its_image(variant):
    v = tensor_variant(variant)
    rng = np.random.default_rng(70)
    for n in (1, 127, 128, 129, 255, 256, 257, 70001):
        bits = rng.integers(0, 256, (n, 32), dtype=np.uint8)
        ref = torch.zeros(lib().hm_prepared_bytes(n, v) + 4096, dtype=torch.uint8, device="cuda")
        bd = dev(bits)
        call("hm_prepare", bd.data_ptr(), n, 32, ref.data_ptr(), v, stream())
        ref = ref[:lib().hm_prepared_bytes(n, v)]
        for offset in OFFSETS:
            for stride in (32, 48):
                src, sp = (bd, bd.data_ptr()) if stride == 32 else poisoned_rows(bits, bits[::-1], stride)
                out = Guarded(lib().hm_prepared_bytes(n, v), offset, seed=n)
                frozen = Frozen(bits=src)
                call("hm_prepare", sp, n, stride, out.ptr, v, stream())
                what = f"hm_prepare n={n} {variant} stride={stride} offset={offset}"
                out.check_guards(what)
                frozen.check(what)
                assert torch.equal(out.view, ref), what


@gpu
@pytest.mark.parametrize("variant", ("i8", "f4"))
@pytest.mark.parametrize("nq,nt,split", ((20000, 500, False), (300, 40000, True)))
def test_knn2_prepared_and_partials_exact_workspace(nq, nt, split, variant):
    from slam_experiments_b200 import _native as nat
    v = tensor_variant(variant)
    grid = nat.describe_launch(nq, nt, 1, variant)
    assert (",1,1)" not in grid) == split, grid
    q, t = planted(nq, nt, nq + nt + 1)
    exp = co.knn2_keys(q, t)
    timg = poisoned_image(t, q, v)                  # padding rows of the train image hold query images
    qimg = prepare(q, v)
    wsb = lib().hm_prepared_workspace_bytes(nq, nt, v)
    for offset, fill in POISONS:
        what = f"{nq}x{nt} {variant} offset={offset} fill={fill}"
        ws = Guarded(wsb, offset, 1, fill)
        out = Guarded(nq * 16, offset, 2)
        frozen = Frozen(query=qimg, train=timg)
        call("hm_knn2_prepared", qimg.data_ptr(), nq, timg.data_ptr(), nt, 0, out.ptr, v, ws.ptr, wsb, stream())
        ws.check_guards("hm_knn2_prepared workspace " + what)
        out.check_guards("hm_knn2_prepared keys " + what)
        frozen.check("hm_knn2_prepared " + what)
        keys_equal(u64(out.as_(torch.int64, (nq, 2))), exp, "hm_knn2_prepared " + what)
        # partials: left in the workspace, merged by hm_merge_top2 into a guarded output
        ws = Guarded(wsb, offset, 3, fill)
        parts, groups = ctypes.c_void_p(), ctypes.c_int(0)
        call("hm_knn2_prepared_partials", qimg.data_ptr(), nq, timg.data_ptr(), nt, 0, v, ws.ptr, wsb, stream(),
             ctypes.byref(parts), ctypes.byref(groups))
        assert (groups.value > 1) == split, (what, groups.value)
        assert ws.ptr <= parts.value and parts.value + groups.value * nq * 16 <= ws.ptr + wsb, what
        out = Guarded(nq * 16, offset, 4)
        call("hm_merge_top2", parts.value, groups.value, nq, out.ptr, stream())
        ws.check_guards("hm_knn2_prepared_partials workspace " + what)
        out.check_guards("hm_merge_top2 keys " + what)
        frozen.check("hm_knn2_prepared_partials " + what)
        keys_equal(u64(out.as_(torch.int64, (nq, 2))), exp, "hm_knn2_prepared_partials + hm_merge_top2 " + what)


# ---- hm_knn2_resident ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("variant", ("i8", "f4"))
@pytest.mark.parametrize("nq", (1, 257, 2000, 4097))
def test_knn2_resident_exact_workspace(nq, variant):
    v = tensor_variant(variant)
    nt = 30000
    q, t = planted(nq, nt, nq + 80)
    exp = co.knn2_keys(q, t)
    timg = poisoned_image(t, q, v)
    wsb = lib().hm_resident_workspace_bytes(nq, nt, v)
    for stride in (32, 64):
        qd, qp = with_ptr(dev(q)) if stride == 32 else poisoned_rows(q, t, stride)
        for offset, fill in POISONS:
            what = f"hm_knn2_resident {nq}x{nt} {variant} q_stride={stride} offset={offset} fill={fill}"
            ws = Guarded(wsb, offset, 5, fill)
            out = Guarded(nq * 16, offset, 6)
            frozen = Frozen(query=qd, train=timg)
            call("hm_knn2_resident", qp, nq, stride, timg.data_ptr(), nt, 0, out.ptr, v, ws.ptr, wsb, stream())
            ws.check_guards(what + " workspace")
            out.check_guards(what + " keys")
            frozen.check(what)
            keys_equal(u64(out.as_(torch.int64, (nq, 2))), exp, what)


# ---- selections: hm_knn2_resident_runs, hm_knn2_runs --------------------------------------------------------------
def selection_problem(sizes, sel, nq, seed):
    """(queries, train rows, runs, selected rows): the unselected keyframes hold exact copies of the queries."""
    from slam_experiments_b200.keyframe_db import selection_mask, shard_runs
    rng = np.random.default_rng(seed)
    cat = rng.integers(0, 256, (int(sum(sizes)), 32), dtype=np.uint8)
    q = rng.integers(0, 256, (nq, 32), dtype=np.uint8)
    m = nq // 2
    q[:m] = cat[rng.integers(0, cat.shape[0], m)] ^ (rng.integers(0, 16, (m, 32), dtype=np.uint8) == 0)
    starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    mask = selection_mask(sel, len(sizes))
    runs = shard_runs(mask, starts, 0, len(sizes), 0)
    rows = np.concatenate([np.arange(lo, hi) for lo, hi in runs]) if runs.shape[0] else np.empty(0, np.int64)
    unsel = np.setdiff1d(np.arange(cat.shape[0]), rows)
    cat[unsel] = q[np.arange(unsel.size) % nq]
    return q, cat, runs, rows


def expected_runs(q, cat, rows):
    if rows.size == 0:
        return np.full((q.shape[0], 2), NO_MATCH, np.uint64)
    keys = co.knn2_keys(q, cat[rows])
    ok = keys != NO_MATCH
    mapped = (keys & np.uint64(0xFFFF_FFFF_0000_0000)) + rows[(keys & LOW32).astype(np.int64) * ok].astype(np.uint64)
    return np.where(ok, mapped, keys)


def run_runs(q, cat, runs, variant, prepared, offset, fill, timg=None, seed=0):
    from slam_experiments_b200 import _native as nat
    nq, nt = q.shape[0], cat.shape[0]
    runs = np.ascontiguousarray(runs, dtype=np.int64).reshape(-1, 2)
    v = tensor_variant(variant) if prepared else variant_id(variant)
    wsb = lib().hm_runs_workspace_bytes(nq, runs.ctypes.data, runs.shape[0], int(prepared), v)
    assert wsb > 0
    qd = dev(q)
    table = dev(nat.run_table(runs).view(np.uint8)) if runs.shape[0] else torch.zeros(32, dtype=torch.uint8, device="cuda")
    ws = Guarded(wsb, offset, seed, fill)
    out = Guarded(nq * 16, offset, seed + 1)
    what = f"{'hm_knn2_resident_runs' if prepared else 'hm_knn2_runs'} nq={nq} nt={nt} runs={runs.shape[0]} " \
           f"{variant} offset={offset} fill={fill}"
    if prepared:
        frozen = Frozen(query=qd, train=timg, runs=table)
        call("hm_knn2_resident_runs", qd.data_ptr(), nq, 32, timg.data_ptr(), nt, runs.ctypes.data, table.data_ptr(),
             runs.shape[0], 0, out.ptr, v, ws.ptr, wsb, stream())
    else:
        td = dev(cat)
        frozen = Frozen(query=qd, train=td, runs=table)
        call("hm_knn2_runs", qd.data_ptr(), nq, 32, td.data_ptr(), nt, 32, runs.ctypes.data, table.data_ptr(),
             runs.shape[0], 0, out.ptr, v, ws.ptr, wsb, stream())
    ws.check_guards(what + " workspace")
    out.check_guards(what + " keys")
    frozen.check(what)
    return u64(out.as_(torch.int64, (nq, 2))), what


def check_runs(sizes, selections, nq, variants_prepared, variants_packed, seed):
    for name, sel in selections.items():
        q, cat, runs, rows = selection_problem(sizes, sel, nq, seed)
        exp = expected_runs(q, cat, rows)
        for variant in variants_prepared:
            timg = poisoned_image(cat, q, tensor_variant(variant))
            for offset, fill in POISONS:
                got, what = run_runs(q, cat, runs, variant, True, offset, fill, timg)
                keys_equal(got, exp, f"{what} selection={name}")
        for variant in variants_packed:
            for offset, fill in POISONS:
                got, what = run_runs(q, cat, runs, variant, False, offset, fill)
                keys_equal(got, exp, f"{what} selection={name}")


@gpu
def test_runs_exact_workspace_selection_shapes():
    from test_keyframe_db_subset import SHAPE_SELECTIONS, SHAPE_SIZES
    check_runs(SHAPE_SIZES, SHAPE_SELECTIONS, 600, ("i8", "f4"), ("popc", "i8", "f4", "auto"), 31)


@gpu
def test_runs_exact_workspace_split_walk():
    from slam_experiments_b200 import _native as nat
    sizes = [64] * 4000 + [1, 77, 129, 3]
    sel = np.arange(0, len(sizes), 2)
    q, cat, runs, rows = selection_problem(sizes, sel, 2000, 34)
    assert int(nat.describe_runs_launch(2000, cat.shape[0], runs, "f4").split("grid=(")[1].split(",")[1]) > 1
    check_runs(sizes, {"every_other": sel}, 2000, ("i8", "f4"), ("f4",), 34)


# ---- hm_db_mutual_flags, hm_db_filter ------------------------------------------------------------------------------
def expected_flags(q, cat, keys, lo, rows, ratio):
    nq = q.shape[0]
    t1 = (keys[:, 0] & LOW32).astype(np.int64)
    own = (keys[:, 0] != NO_MATCH) & (t1 >= lo) & (t1 < lo + rows)
    if ratio is not None:
        d1 = (keys[:, 0] >> np.uint64(32)).astype(np.int64)
        has2 = keys[:, 1] != NO_MATCH
        d2 = np.where(has2, (keys[:, 1] >> np.uint64(32)).astype(np.int64), 0)
        own &= has2 & (d1 < ho.ratio_lut(ratio)[d2])
    flags = np.zeros(nq, np.uint8)
    if rows and own.any():
        col = co.colmin_keys(q, cat[lo:lo + rows])
        best_q = (col[t1[own] - lo] & LOW32).astype(np.int64)
        flags[np.flatnonzero(own)] = best_q == np.flatnonzero(own)
    return flags


def run_db_flags(keys_d, q, qd_ptr, q_stride, shard_d, shard_ptr, rows, t_stride, lo, ratio, variant, offset, fill,
                 seed=0):
    from slam_experiments_b200 import _native as nat
    nq = q.shape[0]
    v = variant_id(variant)
    flags = nat.FLAG_MUTUAL | (nat.FLAG_RATIO if ratio is not None else 0)
    lut = nat.ratio_lut(ratio) if ratio is not None else None
    wsb = lib().hm_db_mutual_workspace_bytes(nq, v)
    ws = Guarded(wsb, offset, seed, fill)
    out = Guarded(nq, offset, seed + 1)                         # the guard sits right after the nq flag bytes
    rc = lib().hm_db_mutual_flags(keys_d.data_ptr(), nq, qd_ptr, q_stride, shard_ptr, rows, t_stride, lo, flags,
                                  lut.ctypes.data if lut is not None else None, out.ptr, v, ws.ptr, wsb, stream())
    what = f"hm_db_mutual_flags nq={nq} shard=[{lo}, {lo + rows}) ratio={ratio} {variant} offset={offset} fill={fill}"
    ws.check_guards(what + " workspace")
    out.check_guards(what + " flags")
    return rc, out, what


DB_NQ = (1, 255, 256, 2000)


@gpu
@pytest.mark.parametrize("variant", ("popc", "i8", "f4", "auto"))
@pytest.mark.parametrize("nq", DB_NQ)
def test_db_mutual_flags_and_filter_exact_workspace(nq, variant):
    from slam_experiments_b200 import _native as nat
    q, cat = planted(nq, 6000, nq + 90)
    keys = co.knn2_keys(q, cat)
    keys_d, qd = dev(keys.view(np.int64)), dev(q)
    t1 = (keys[:, 0] & LOW32).astype(np.int64)
    free = np.setdiff1d(np.arange(cat.shape[0]), t1)
    shards = {"all": (0, cat.shape[0]), "some": (1500, 2500), "empty": (cat.shape[0], 0),
              "one_row_nobody_picks": (int(free[len(free) // 2]), 1)}
    for name, (lo, rows) in shards.items():
        sb = dev(cat[lo:lo + rows]) if rows else torch.zeros(32, dtype=torch.uint8, device="cuda")
        for ratio in (None, 0.8):
            exp = expected_flags(q, cat, keys, lo, rows, ratio)
            for offset, fill in ((0, "random"), (0, 0xFF)):
                frozen = Frozen(keys=keys_d, query=qd, shard=sb)
                rc, out, what = run_db_flags(keys_d, q, qd.data_ptr(), 32, sb, sb.data_ptr(), rows, 32, lo, ratio,
                                             variant, offset, fill)
                assert rc == nat.HM_OK, f"{what}: {rc} {nat.last_error()}"
                frozen.check(what)
                got = out.view.cpu().numpy()
                assert np.array_equal(got, exp), f"{what} ({name}): {int((got != exp).sum())} flags differ"
            # hm_db_mutual_flags promises 256-byte aligned workspaces only: offset 16 is rejected before any work
            rc, out, what = run_db_flags(keys_d, q, qd.data_ptr(), 32, sb, sb.data_ptr(), rows, 32, lo, ratio, variant,
                                         16, "random")
            assert rc == HM_ERR_WORKSPACE, f"{what}: {rc}"
    # hm_db_filter over the whole-database flags, with and without the ratio test
    for ratio in (None, 0.8):
        flags_h = expected_flags(q, cat, keys, 0, cat.shape[0], ratio)
        flags_d = dev(flags_h)
        for mutual in (False, True):
            k = (keys[:, 0] != NO_MATCH)
            if ratio is not None:
                d1 = (keys[:, 0] >> np.uint64(32)).astype(np.int64)
                d2 = (keys[:, 1] >> np.uint64(32)).astype(np.int64)
                k &= (keys[:, 1] != NO_MATCH) & (d1 < ho.ratio_lut(ratio)[np.clip(d2, 0, 256)])
            if mutual:
                k &= flags_h.astype(bool)
            qi = np.flatnonzero(k)
            exp = (qi.astype(np.int32), t1[qi].astype(np.int32), (keys[qi, 0] >> np.uint64(32)).astype(np.int32))
            fl = (nat.FLAG_RATIO if ratio is not None else 0) | (nat.FLAG_MUTUAL if mutual else 0)
            lut = nat.ratio_lut(ratio) if ratio is not None else None
            for offset in OFFSETS:
                outs = [Guarded(nq * 4, offset, 20 + i) for i in range(3)]
                cnt = Guarded(4, offset, 24)
                frozen = Frozen(keys=keys_d, flags=flags_d)
                call("hm_db_filter", keys_d.data_ptr(), nq, flags_d.data_ptr() if mutual else None, fl,
                     lut.ctypes.data if lut is not None else None, outs[0].ptr, outs[1].ptr, outs[2].ptr, cnt.ptr,
                     stream())
                what = f"hm_db_filter nq={nq} ratio={ratio} mutual={mutual} offset={offset}"
                for g in outs + [cnt]:
                    g.check_guards(what)
                frozen.check(what)
                n = int(cnt.as_(torch.int32, (1,)).item())
                got = tuple(o.as_(torch.int32, (nq,)).cpu().numpy()[:n] for o in outs)
                matches_equal(got, exp, what)


@gpu
@pytest.mark.parametrize("variant", ("popc", "i8", "f4", "auto"))
@pytest.mark.parametrize("stride", (48, 64))
def test_db_mutual_flags_ignores_rows_outside_its_inputs(stride, variant):
    """the flag pass scans the queries as columns: their gaps and tail hold database rows; the shard's hold queries"""
    from slam_experiments_b200 import _native as nat
    nq = 2000
    q, cat = planted(nq, 6000, 95)
    keys = co.knn2_keys(q, cat)
    keys_d = dev(keys.view(np.int64))
    for lo, rows in ((0, cat.shape[0]), (1500, 2500)):
        qd, qp = poisoned_rows(q, cat[lo:lo + rows], stride)
        sd, sp = poisoned_rows(cat[lo:lo + rows], q, stride)
        for ratio in (None, 0.8):
            exp = expected_flags(q, cat, keys, lo, rows, ratio)
            frozen = Frozen(keys=keys_d, query=qd, shard=sd)
            rc, out, what = run_db_flags(keys_d, q, qp, stride, sd, sp, rows, stride, lo, ratio, variant, 0, "random")
            assert rc == nat.HM_OK, f"{what}: {rc} {nat.last_error()}"
            frozen.check(what)
            got = out.view.cpu().numpy()
            assert np.array_equal(got, exp), f"{what} stride={stride}: {int((got != exp).sum())} flags differ"


# =====================================================================================================================
# outputs only: hm_filter_matches, hm_gather_points, hm_rasterize_mask
# =====================================================================================================================
@gpu
@pytest.mark.parametrize("offset", OFFSETS)
def test_filter_matches_writes_only_its_outputs(offset):
    from slam_experiments_b200 import _native as nat
    b, nq, nt = 2, 500, 300
    pr = [planted(nq, nt, 100 + s) for s in range(b)]
    fwd = np.stack([co.knn2_keys(p[0], p[1]) for p in pr])
    bwd = np.stack([co.knn2_keys(p[1], p[0]) for p in pr])
    fd, bd = dev(fwd.view(np.int64)), dev(bwd.view(np.int64))
    for i, (ratio, cross, thr) in enumerate(FLAG_SETS):
        flags = (nat.FLAG_RATIO if ratio is not None else 0) | (nat.FLAG_MUTUAL if cross else 0) | \
                (nat.FLAG_DIST_THRESHOLD if thr else 0)
        lut = nat.ratio_lut(ratio) if ratio is not None else None
        outs = [Guarded(b * nq * 4, offset, 30 + j) for j in range(3)]
        cnt = Guarded(b * 4, offset, 33)
        frozen = Frozen(fwd=fd, bwd=bd)
        call("hm_filter_matches", fd.data_ptr(), nq, bd.data_ptr(), nt, b, flags,
             lut.ctypes.data if lut is not None else None, float(thr or 0.0), outs[0].ptr, outs[1].ptr, outs[2].ptr,
             cnt.ptr, stream())
        what = f"hm_filter_matches ratio={ratio} cross={cross} thr={thr} offset={offset}"
        for g in outs + [cnt]:
            g.check_guards(what)
        frozen.check(what)
        n = cnt.as_(torch.int32, (b,)).cpu().numpy()
        oq, ot, od = (o.as_(torch.int32, (b, nq)).cpu().numpy() for o in outs)
        for j in range(b):
            matches_equal((oq[j, :n[j]], ot[j, :n[j]], od[j, :n[j]]), expected_fused(pr[j][0], pr[j][1], ratio, cross, thr),
                          f"{what} problem {j}")


@gpu
@pytest.mark.parametrize("offset", OFFSETS)
def test_gather_points_leaves_entries_past_count_untouched(offset):
    """``entries at m >= count[b] are left untouched`` (hm_matcher.h): count 0, partial and the whole stride"""
    rng = np.random.default_rng(110)
    b, stride, nq, nt = 3, 300, 400, 350
    counts = np.array([0, 137, stride], np.int32)
    # every index entry is valid, also past count[b] and one stride past the end, so that a kernel reading past
    # count[b] still reads memory the test owns
    qi = dev(rng.integers(0, nq, (b + 1) * stride).astype(np.int32))
    ti = dev(rng.integers(0, nt, (b + 1) * stride).astype(np.int32))
    qp = dev(rng.integers(-5000, 5000, (b, nq, 2)).astype(np.int32))
    tp = dev(rng.integers(-5000, 5000, (b, nt, 2)).astype(np.int32))
    cnt = dev(counts)
    oq, ot = Guarded(b * stride * 8, offset, 40), Guarded(b * stride * 8, offset, 41)
    before = [oq.as_(torch.int32, (b, stride, 2)).clone(), ot.as_(torch.int32, (b, stride, 2)).clone()]
    frozen = Frozen(q_idx=qi, t_idx=ti, query_pts=qp, train_pts=tp, count=cnt)
    call("hm_gather_points", qi.data_ptr(), ti.data_ptr(), cnt.data_ptr(), stride, b, qp.data_ptr(), nq, tp.data_ptr(),
         nt, oq.ptr, ot.ptr, stream())
    what = f"hm_gather_points offset={offset}"
    oq.check_guards(what + " query points")
    ot.check_guards(what + " train points")
    frozen.check(what)
    qi_h, ti_h = qi.cpu().numpy().reshape(-1, stride), ti.cpu().numpy().reshape(-1, stride)
    for out, pts, idx, prev, name in ((oq, qp, qi_h, before[0], "query"), (ot, tp, ti_h, before[1], "train")):
        got = out.as_(torch.int32, (b, stride, 2)).cpu().numpy()
        prev, pts = prev.cpu().numpy(), pts.cpu().numpy()
        for j in range(b):
            c = counts[j]
            assert np.array_equal(got[j, :c], pts[j][idx[j, :c]]), (what, name, j)
            assert np.array_equal(got[j, c:], prev[j, c:]), \
                f"{what}: {name} entries past count[{j}] = {c} written, first at " \
                f"{c + int(np.flatnonzero((got[j, c:] != prev[j, c:]).any(1))[0])}"


@gpu
@pytest.mark.parametrize("offset", OFFSETS)
@pytest.mark.parametrize("inner", (0, 1))
def test_rasterize_mask_leaves_row_gaps_untouched(inner, offset):
    rng = np.random.default_rng(120 + inner)
    h, w, row_stride, radius = 61, 77, 96, 3
    pts = np.concatenate([rng.integers(-5, 82, (40, 1)), rng.integers(-5, 66, (40, 1))], 1).astype(np.int32)
    pts[:4] = [[0, 0], [w - 1, h - 1], [-radius, h + radius], [w + radius, -radius]]
    pd = dev(pts)
    mask = Guarded(h * row_stride, offset, 50)
    before = mask.as_(torch.uint8, (h, row_stride)).clone().cpu().numpy()
    frozen = Frozen(points=pd)
    call("hm_rasterize_mask", pd.data_ptr(), pts.shape[0], radius, inner, mask.ptr, h, w, row_stride, stream())
    what = f"hm_rasterize_mask inner={inner} offset={offset}"
    mask.check_guards(what)
    frozen.check(what)
    got = mask.as_(torch.uint8, (h, row_stride)).cpu().numpy()
    exp = np.full((h, w), 0 if inner else 255, np.uint8)
    for x, y in pts:
        exp[max(0, y - radius):max(0, y + radius + 1), max(0, x - radius):max(0, x + radius + 1)] = 255 if inner else 0
    assert np.array_equal(got[:, :w], exp), what
    assert np.array_equal(got[:, w:], before[:, w:]), f"{what}: row gap bytes written"


# =====================================================================================================================
# ORB: hm_orb_build_pyramid (exact workspace), hm_orb_describe (strided output)
# =====================================================================================================================
def plane_layout(h, w, n_levels):
    """Byte layout of one pyramid plane inside the workspace (hm_orb.cu orb_geometry), as tests/test_orb.py reads it."""
    from oracle import orb_oracle as oo
    out, off = [], 0
    for lv in range(n_levels):
        r, c = oo.level_size(h, w, lv)
        stride = (c + 64 + 15) // 16 * 16
        out.append((off, r, c, stride))
        off = (off + stride * (r + 64) + 255) // 256 * 256
    return out, off


def orb_keypoints(h, w, n, seed):
    from oracle import orb_oracle as oo
    rng = np.random.default_rng(seed)
    xy = np.empty((n, 2), np.float32)
    ang = rng.uniform(0, 360, n).astype(np.float32)
    octv = np.sort(rng.integers(0, 8, n)).astype(np.int32)
    for i, o in enumerate(octv):
        s = float(oo.level_scale(int(o)))
        r, c = oo.level_size(h, w, int(o))
        xy[i] = (float(rng.uniform(31.5, c - 32.5)) * s, float(rng.uniform(31.5, r - 32.5)) * s)
    return xy, ang, octv


@gpu
@pytest.mark.parametrize("h,w,seed,ch", [(480, 640, 7, 1), (480, 752, 11, 3), (333, 517, 13, 1), (120, 90, 5, 1)])
def test_orb_pyramid_exact_workspace(h, w, seed, ch):
    from oracle import orb_oracle as oo
    from slam_experiments_b200 import synth
    img = synth.textured_image(h, w, seed, ch)
    n_levels = 8 if h >= 333 else 3
    wsb = lib().hm_orb_workspace_bytes(h, w, n_levels)
    levels = oo.build_pyramid(oo.to_gray(img), n_levels)
    layout, plane = plane_layout(h, w, n_levels)
    imd = dev(img)
    for offset, fill in POISONS:
        ws = Guarded(wsb, offset, seed, fill)
        frozen = Frozen(image=imd)
        call("hm_orb_build_pyramid", imd.data_ptr(), h, w, w * ch, ch, n_levels, ws.ptr, wsb, stream())
        what = f"hm_orb_build_pyramid {h}x{w}x{ch} offset={offset} fill={fill}"
        ws.check_guards(what)
        frozen.check(what)
        got = ws.view.cpu().numpy()
        for (off, r, c, stride), ref in zip(layout, levels):
            blurred = got[256 + plane + off: 256 + plane + off + stride * (r + 64)].reshape(r + 64, stride)[:, :c + 64]
            assert np.array_equal(blurred, ref), (what, r, c)


@gpu
@pytest.mark.parametrize("out_stride", (32, 48))
@pytest.mark.parametrize("offset", OFFSETS)
def test_orb_describe_leaves_stride_gaps_untouched(offset, out_stride):
    from slam_experiments_b200 import _native as nat
    from oracle import orb_oracle as oo
    from slam_experiments_b200 import synth
    h, w, n = 480, 640, 400
    img = synth.textured_image(h, w, 77)
    xy, ang, octv = orb_keypoints(h, w, n, 0)
    exp = oo.describe(img, xy, ang, octv)
    ws = nat.orb_build_pyramid(dev(img), 8)
    xyd, csd, od = dev(xy), dev(nat.orb_angles_to_cs(ang)), dev(octv)
    out = Guarded(n * out_stride, offset, 60)
    before = out.as_(torch.uint8, (n, out_stride)).cpu().numpy().copy()
    frozen = Frozen(workspace=ws, xy=xyd, cs=csd, octave=od)
    call("hm_orb_describe", ws.data_ptr(), h, w, 8, xyd.data_ptr(), csd.data_ptr(), od.data_ptr(), n, out.ptr, out_stride,
         stream())
    what = f"hm_orb_describe out_stride={out_stride} offset={offset}"
    out.check_guards(what)
    frozen.check(what)
    got = out.as_(torch.uint8, (n, out_stride)).cpu().numpy()
    assert np.array_equal(got[:, :32], exp), what
    assert np.array_equal(got[:, 32:], before[:, 32:]), f"{what}: stride gap bytes written"


# =====================================================================================================================
# host-buffer entry points: guard elements around every host output
# =====================================================================================================================
class Context:
    def __init__(self):
        self.h = ctypes.c_void_p()
        call("hm_context_create", ctypes.byref(self.h))

    def __enter__(self):
        return self.h

    def __exit__(self, *exc):
        lib().hm_context_destroy(self.h)


@gpu
@pytest.mark.parametrize("variant", ("auto", "popc", "f4"))
def test_host_entry_points_write_only_their_outputs(variant):
    from slam_experiments_b200 import _native as nat
    v = variant_id(variant)
    with Context() as ctx:
        for nq, nt in ((301, 400), (300, 401), (1501, 2000)):
            q, t = planted(nq, nt, nq + nt)
            # hm_knn2_host
            out = HostGuarded((nq, 2), np.uint64, 1)
            call("hm_knn2_host", ctx, q.ctypes.data, nq, t.ctypes.data, nt, out.ptr, v)
            out.check_guards(f"hm_knn2_host {nq}x{nt} {variant}")
            keys_equal(out.a, co.knn2_keys(q, t), f"hm_knn2_host {nq}x{nt} {variant}")
            # hm_match_host, three times (direct, graph capture, graph replay)
            for ratio, cross in ((None, False), (0.8, True)):
                flags = (nat.FLAG_RATIO if ratio else 0) | (nat.FLAG_MUTUAL if cross else 0)
                lut = nat.ratio_lut(ratio) if ratio else None
                exp = expected_fused(q, t, ratio, cross, None)
                for rep in range(3):
                    outs = [HostGuarded((nq,), np.int32, 2 + j) for j in range(3)]
                    cnt = HostGuarded((1,), np.int32, 5)
                    call("hm_match_host", ctx, q.ctypes.data, nq, 32, t.ctypes.data, nt, 32, flags,
                         lut.ctypes.data if lut is not None else None, 0.0, v, outs[0].ptr, outs[1].ptr, outs[2].ptr,
                         cnt.ptr)
                    what = f"hm_match_host {nq}x{nt} {variant} ratio={ratio} cross={cross} call {rep}"
                    for g in outs + [cnt]:
                        g.check_guards(what)
                    n = int(cnt.a[0])
                    matches_equal(tuple(o.a[:n] for o in outs), exp, what)
            # hm_frame_put + hm_frame_match with matched points (odd and even nq)
            rng = np.random.default_rng(nq)
            pq = rng.integers(0, 1000, (nq, 2)).astype(np.int32)
            pt = rng.integers(0, 1000, (nt, 2)).astype(np.int32)
            call("hm_frame_put", ctx, 0, t.ctypes.data, nt, 32, pt.ctypes.data)
            call("hm_frame_put", ctx, 1, q.ctypes.data, nq, 32, pq.ctypes.data)
            exp = expected_fused(q, t, 0.8, True, None)
            lut = nat.ratio_lut(0.8)
            for rep in range(3):
                outs = [HostGuarded((nq,), np.int32, 6 + j) for j in range(3)]
                pts = [HostGuarded((nq, 2), np.int32, 9 + j) for j in range(2)]
                cnt = HostGuarded((1,), np.int32, 11)
                call("hm_frame_match", ctx, 0, 1, nat.FLAG_RATIO | nat.FLAG_MUTUAL, lut.ctypes.data, 0.0, v,
                     outs[0].ptr, outs[1].ptr, outs[2].ptr, pts[0].ptr, pts[1].ptr, cnt.ptr)
                what = f"hm_frame_match {nq}x{nt} {variant} call {rep}"
                for g in outs + pts + [cnt]:
                    g.check_guards(what)
                n = int(cnt.a[0])
                matches_equal(tuple(o.a[:n] for o in outs), exp, what)
                assert np.array_equal(pts[0].a[:n], pq[exp[0]]) and np.array_equal(pts[1].a[:n], pt[exp[1]]), what
        # hm_resident_query_begin / _end against a prepared database
        tv = tensor_variant("f4" if variant == "f4" else "auto")
        for nq in (1, 257, 2000):
            q, t = planted(nq, 30000, nq + 7)
            timg = poisoned_image(t, q, tv)
            call("hm_resident_query_begin", ctx, q.ctypes.data, nq, 32, timg.data_ptr(), t.shape[0], 0, tv, 1, 0, None,
                 0, 0)
            out = HostGuarded((nq, 2), np.uint64, 12)
            call("hm_resident_query_end", ctx, nq, out.ptr)
            out.check_guards(f"hm_resident_query_end nq={nq}")
            keys_equal(out.a, co.knn2_keys(q, t), f"hm_resident_query nq={nq} variant={tv}")
        # hm_frame_put_orb with the descriptors copied back
        from oracle import orb_oracle as oo
        from slam_experiments_b200 import synth
        img = np.ascontiguousarray(synth.textured_image(480, 640, 78))
        xy, ang, octv = orb_keypoints(480, 640, 301, 1)
        out = HostGuarded((301, 32), np.uint8, 13)
        call("hm_frame_put_orb", ctx, 2, img.ctypes.data, 480, 640, 640, 1, 8, xy.ctypes.data, ang.ctypes.data,
             octv.ctypes.data, 301, None, out.ptr)
        out.check_guards("hm_frame_put_orb out_desc_host")
        assert np.array_equal(out.a, oo.describe(img, xy, ang, octv))


# =====================================================================================================================
# D: the grown keyframe database image
# =====================================================================================================================
@gpu
@pytest.mark.parametrize("variant", ("i8", "f4"))
def test_grown_database_image_equals_a_fresh_image(variant):
    """After every append_keyframe the resident image is byte-identical to hm_prepare of all rows, padding rows
    included, although everything past the image is filled with a pattern after each append: appends that re-expand
    from an odd multiple of 128 rows (200 -> 300 rows, 944 -> 1071) and the reallocation of the last one must rewrite
    every padding row."""
    from slam_experiments_b200 import _native as nat
    from slam_experiments_b200.keyframe_db import ShardedKeyframeDatabase
    sizes = [50, 150, 100, 1, 515, 0, 128, 127, 70000]
    rng = np.random.default_rng(130)
    kfs = [rng.integers(0, 256, (s, 32), dtype=np.uint8) for s in sizes]
    v = tensor_variant(variant)
    db = ShardedKeyframeDatabase(sizes[:1], kfs[:1], variant=variant)
    q = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    for i in range(1, len(sizes)):
        db.append_keyframe(kfs[i])
        sh = db.shard
        nt = sh["nt"]
        cat = np.concatenate(kfs[:i + 1])
        assert nt == cat.shape[0]
        nb = lib().hm_prepared_bytes(nt, v)
        want = prepare(cat, v)
        got = sh["prepared"][:nb]
        if not torch.equal(got, want):
            rb = nat.PREPARED_ROW_BYTES[v]
            bad = torch.nonzero(got != want).flatten() // rb
            pytest.fail(f"{variant}: after appending keyframe {i} ({nt} rows) image rows {int(bad[0])}..{int(bad[-1])} "
                        f"of {nb // rb} differ from hm_prepare of all rows")
        q[:100] = cat[rng.integers(0, nt, 100)]
        keys = db.knn2_keys_device(dev(q)).cpu().numpy().view(np.uint64)
        keys_equal(keys, co.knn2_keys(q, cat), f"{variant} grown to {nt} rows")
        if sh["pbuf"] is not None:
            tail = sh["pbuf"][nb:]
            tail.copy_(_pattern(tail.numel(), i, "cuda"))
