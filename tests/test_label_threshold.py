"""Edge labels at the curvature threshold, through every kernel that labels.

Every labelling kernel decides `curv > 0.1` (src/slam.c:11-61) with the fp32 filter of csrc/stencil_tile.cuh: the
curvature in fp32 together with a bound `err` on its error, and the reference's binary64 expression
(label_exact_at) only where fp32 is within `err` of the threshold or not finite.  The labels are the reference's
bit for bit only if that bound holds.  Synthetic room data rarely comes near the threshold, so this file builds
images whose points do:

  * every row is laid out as disjoint 5-column groups (the curvature of a column depends on columns c-2 .. c+2
    only); one coordinate of each group's centre is bisected until the centre's curvature is 0.1 + delta, delta
    log-uniform in +-[1e-15, 1e-3], or until the two ends are adjacent doubles whose labels differ (straddle pairs);
  * the groups span spacings from 2.5e-4 to 1e154 (the 1e-6 term of the denominator dominating, fp32 reciprocals
    going subnormal, fp32 squares and conversions overflowing, binary64 squares overflowing) and translations of
    0, 1e6 and 2^40 (binary64 differences already rounded); a few groups hold a duplicated neighbour, a zero
    (invalid) point, or a NaN / inf coordinate;
  * the group phase shifts from row to row, so the centres fall on every residue mod 256 (the CTA tiles), every
    residue mod 240 of the flattened batch index (the 1-D tiles of k_labels_tma) and on columns 2 and cols-3.

The CPU tests hold the numpy restatement of the reference's arithmetic to the oracle and the generator to stated
numbers of pixels per band of |curv - 0.1|.  The GPU tests run the same kind of images through every entry point
that labels and compare labels (and what depends on them) with the oracle bit for bit.  Around every call they
also read the exact-fallback counter and hold it between two bounds (fallback_bounds): at least every pixel within
half of the window the kernel's own `err` opens around the threshold (plus the non-finite and fp32-overflow cases),
so an `err` a few times too small fails even where fp32 happens to be right; at most the pixels within 1e-4 of the
threshold or with non-finite or huge inputs, so fp32 really decides the rest."""
import ctypes as C
import functools
import re

import numpy as np
import pytest

gpu = pytest.mark.gpu

F32_EPS6 = float(np.float32(1e-6))   # the reference's 1e-6f, promoted to double
SCALES = [2.5e-4, 1e-3, 1.0, 1e3, 1e5, 1e9, 2.0 ** 62, 9e18, 1.5e19, 1.8446e19, 2e19, 1e30, 1e39, 1e154]
SHIFTS = [0.0, 1e6, 2.0 ** 40]
TAPS = (-2, -1, 1, 2)
CANARY = 0xA5


# ------------------------------------------------------------------ the reference's arithmetic in numpy ----------
def _dist(a, b):
    d = a - b
    return np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])


def _curv_from_taps(d):
    """d: the four tap distances in tap order (-2, -1, +1, +2), stacked on the last axis."""
    s = ((d[..., 0] + d[..., 1]) + d[..., 2]) + d[..., 3]
    avg = s / 4
    var = np.zeros_like(avg)
    for k in range(4):
        e = d[..., k] - avg
        var = var + e * e
    out = var / 4 / (avg * avg + F32_EPS6)
    return np.where(avg > 0, out, 0.0)


def taps_np(cloud):
    """[..., rows, cols - 4, 4] binary64 tap distances of the evaluated columns 2 .. cols-3."""
    c = cloud.shape[-2]
    mid = cloud[..., 2:c - 2, :]
    return np.stack([_dist(mid, cloud[..., 2 + k:c - 2 + k, :]) for k in TAPS], axis=-1)


def curvature_np(cloud):
    """The reference's curvature of every pixel (0 on the two border columns each side), src/slam.c:18-55."""
    cloud = np.asarray(cloud, dtype=np.float64)
    out = np.zeros(cloud.shape[:-1])
    if cloud.shape[-2] >= 5:
        with np.errstate(all="ignore"):
            out[..., 2:-2] = _curv_from_taps(taps_np(cloud))
    return out


# ------------------------------------------------------------------ the generator ----------------------------------
def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _group_curv(cen, nb):
    """curvature of centres cen [n,3] with neighbours nb [n,4,3] (tap order)."""
    with np.errstate(all="ignore"):
        return _curv_from_taps(np.stack([_dist(cen, nb[:, k]) for k in range(4)], axis=-1))


def _tune(rng, n, n_pairs):
    """n group geometries; the first n_pairs are tuned to a straddle (adjacent doubles, labels differ), the rest
    to 0.1 + delta.  Returns centres lo/hi [n,3] (lo == hi where the scan found no bracket), neighbours [n,4,3],
    the tuned flags, the scale index and the duplicated-neighbour flags."""
    si = rng.integers(0, len(SCALES), n)
    s = np.array(SCALES)[si]
    shift = np.array(SHIFTS)[rng.integers(0, len(SHIFTS), n)]
    base = shift[:, None] * np.array([1.0, -0.75, 0.5]) + s[:, None] * rng.uniform(8, 12, (n, 3)) * \
        rng.choice([-1.0, 1.0], (n, 3))
    u = _unit(rng.normal(size=(n, 3)))
    # binary64 squares overflow above 1.34e154: at that scale the group is drawn 4x tighter, so that its taps fall
    # on both sides of the overflow
    s = np.where(s >= 1e154, 0.25 * s, s)
    jit = rng.uniform(0.0, 0.6, n)[:, None]
    pos = np.empty((n, 4))
    pos[:, 1] = -rng.uniform(0.3, 2.5, n)
    pos[:, 0] = pos[:, 1] - rng.uniform(0.3, 2.5, n)
    pos[:, 2] = rng.uniform(0.3, 2.5, n)
    pos[:, 3] = pos[:, 2] + rng.uniform(0.3, 2.5, n)
    with np.errstate(all="ignore"):
        nb = base[:, None, :] + s[:, None, None] * (pos[..., None] * u[:, None, :] +
                                                     jit[:, None] * rng.normal(size=(n, 4, 3)))
    dup = np.zeros(n, dtype=bool)
    dup[n_pairs:][rng.random(n - n_pairs) < 0.01] = True   # tap +1 sits on the centre: a zero distance
    axis = rng.integers(0, 3, n)
    mag = 10.0 ** np.where(rng.random(n) < 0.5, rng.uniform(-15, -3, n), rng.uniform(-8, -5, n))
    target = 0.1 + np.where(np.arange(n) < n_pairs, 0.0, mag * rng.choice([-1.0, 1.0], n))
    ii = np.arange(n)

    def above(x):   # label of the centre with coordinate `axis` set to x
        cen = base.copy()
        cen[ii, axis] = x
        b = nb.copy()
        b[dup, 2] = cen[dup]
        return _group_curv(cen, b) > target

    # scan the coordinate over base +- 3 s for the first sign change, then bisect to adjacent doubles
    x0 = base[ii, axis]
    grid = x0[:, None] + s[:, None] * np.linspace(-3.0, 3.0, 33)[None, :]
    sides = np.stack([above(grid[:, k]) for k in range(grid.shape[1])], axis=1)
    change = sides[:, 1:] != sides[:, :-1]
    ok = change.any(axis=1)
    k = np.argmax(change, axis=1)
    lo, hi = grid[ii, k].copy(), grid[ii, k + 1].copy()
    lo[~ok] = hi[~ok] = x0[~ok]
    lo_side = sides[ii, k]
    for _ in range(2000):
        mid = lo + (hi - lo) * 0.5
        live = ok & (mid != lo) & (mid != hi)
        if not live.any():
            break
        m_side = above(mid)
        move_lo = live & (m_side == lo_side)
        move_hi = live & (m_side != lo_side)
        lo = np.where(move_lo, mid, lo)
        hi = np.where(move_hi, mid, hi)
    cen_lo, cen_hi = base.copy(), base.copy()
    cen_lo[ii, axis] = lo
    cen_hi[ii, axis] = hi
    nb[dup, 2] = np.nan   # placeholder: filled with the centre at placement
    return cen_lo, cen_hi, nb, ok, si, dup


def group_slots(rows, cols, image):
    """(row, centre column) of every group of one image: centres at 2 + phase + 5k, phase = (row + 3*image) % 5
    (modulo fewer where a row is too short for that phase to hold a group)."""
    out = []
    for r in range(rows):
        ph = (r + 3 * image) % min(5, cols - 4)
        for c in range(2 + ph, cols - 2, 5):
            out.append((r, c))
    return out


def near_threshold_images(shape, n_images, seed, meta=False):
    """[n_images, rows, cols, 3] near-threshold images (see the module docstring).  meta: also return where the
    groups went -- image, row, centre column and scale index of every group, and the (lo, hi) group indices of
    every straddle pair that bracketed."""
    rows, cols = shape
    rng = np.random.default_rng(seed)
    img = rng.normal(0.0, 1000.0, (n_images, rows, cols, 3))   # background of the columns no group covers
    slots = [(i, r, c) for i in range(n_images) for r, c in group_slots(rows, cols, i)]
    m = len(slots)
    n_pairs = m // 10
    n = m - n_pairs
    cen_lo, cen_hi, nb, ok, si, dup = _tune(rng, n, n_pairs)
    # every straddle geometry gives two groups (its lo and its hi centre), every other one a group
    src = np.concatenate([np.arange(n_pairs), np.arange(n_pairs), np.arange(n_pairs, n)])
    use_hi = np.concatenate([np.zeros(n_pairs, bool), np.ones(n_pairs, bool), rng.random(n - n_pairs) < 0.5])
    order = rng.permutation(m)
    sl = np.array(slots)[order]
    cen = np.where(use_hi[:, None], cen_hi[src], cen_lo[src])
    b = nb[src].copy()
    b[dup[src], 2] = cen[dup[src]]
    i, r, c = sl[:, 0], sl[:, 1], sl[:, 2]
    img[i, r, c] = cen
    for k, t in enumerate(TAPS):
        img[i, r, c + t] = b[:, k]
    # a few groups with an invalid (zero) point or a NaN / +-inf coordinate
    special = rng.choice(m, size=min(m, 6 + m // 2000), replace=False)
    for j, g in enumerate(special):
        col = c[g] + rng.integers(-2, 3)
        if j % 4 == 0:
            img[i[g], r[g], col] = 0.0
        else:
            img[i[g], r[g], col, rng.integers(0, 3)] = (np.nan, np.inf, -np.inf)[j % 4 - 1]
    if not meta:
        return img
    pairs = np.stack([np.arange(n_pairs), n_pairs + np.arange(n_pairs)], axis=1)[ok[:n_pairs]]
    pairs = pairs[~np.isin(pairs, special).any(axis=1)]
    return img, {"image": i, "row": r, "col": c, "scale": si[src], "pairs": pairs}


# ------------------------------------------------------------------ bands and bounds ------------------------------
BANDS = [("<=1e-9", 0.0, 1e-9), ("(1e-9,1e-7]", 1e-9, 1e-7), ("(1e-7,1e-5]", 1e-7, 1e-5), ("(1e-5,1e-4]", 1e-5, 1e-4)]


def evaluated(a, cols):
    return a[..., 2:cols - 2]


def band_counts(cloud):
    """evaluated pixels per band of |curv - 0.1|"""
    cols = cloud.shape[-2]
    with np.errstate(all="ignore"):
        dev = np.abs(evaluated(curvature_np(cloud), cols) - 0.1)
    return {name: int(((dev > lo) & (dev <= hi)).sum() if lo > 0 else (dev <= hi).sum()) for name, lo, hi in BANDS}


def _fp32_square_overflows(cloud):
    """[..., rows, cols-4]: a tap's fp32 square sum (tile_dist32: fmaf(dx,dx, fmaf(dy,dy, dz*dz)) of the fp32
    differences) overflows"""
    c = cloud.shape[-2]
    mid = cloud[..., 2:c - 2, :]
    over = np.zeros(mid.shape[:-1], dtype=bool)
    with np.errstate(all="ignore"):
        for k in TAPS:
            d = (mid - cloud[..., 2 + k:c - 2 + k, :]).astype(np.float32).astype(np.float64)
            q = (d[..., 2] * d[..., 2]).astype(np.float32).astype(np.float64)
            q = (d[..., 1] * d[..., 1] + q).astype(np.float32).astype(np.float64)
            q = (d[..., 0] * d[..., 0] + q).astype(np.float32)
            over |= np.isinf(q)
    return over


# label_from_taps32 decides in fp32 only outside [0.0999999f - err, 0.1000001f + err]; the narrower side of the fixed
# margin, and u = 2^-24
MARGIN = 0.1 - float(np.float32(0.0999999))
U24 = 2.0 ** -24
THIN = 2e-7   # beyond MARGIN plus an err 64 times smaller than the kernel's (1u instead of 64u) near c = 0.1


def fallback_bounds(cloud):
    """(lower, upper, thin) for the exact re-evaluations the fp32 filter makes labelling `cloud` [..., rows, cols, 3].

    lower: the pixels the kernel must re-evaluate.  Its err = 64u (avg32 A32 / den32) + 64u c32 + 1e-9 with
    A32 >= sum |e_k| >= sqrt(V) = 2 sqrt(c den), so err >= g = 64u (2 sqrt(c) avg / sqrt(den) + c) + 1e-9 up to fp32
    rounding, and fp32 cannot decide a pixel whose c32 is within MARGIN + g of 0.1.  Every pixel with
    |c - 0.1| <= (MARGIN + g) / 2 therefore falls back as long as |c32 - c| stays below half of that window, which it
    does by a wide margin: sqrt.approx and rcp.approx are within 2^-22 and 2^-23 relative, and a relative error eps
    in each distance moves c by at most about 0.6 eps avg^2/den, below 1.6e-7, while half the window is at least
    (MARGIN + 64u c) / 2 = 2.4e-7 and grows with avg / sqrt(den).  So does every pixel with a non-finite curvature
    or an fp32 square that overflows.
    upper: the pixels within 1e-4 of the threshold, or with a non-finite curvature, a NaN / inf coordinate in the
    window or a tap of 2^60 or more; fp32 decides every other one (err <= 64u (4 sqrt(c) + c) + 1e-9 < 1e-5 near 0.1).
    thin: pixels of `lower` with finite curvature farther than THIN from 0.1 -- those an err 64 times too small would
    let fp32 decide, so that they drop out of the count."""
    cloud = np.asarray(cloud, dtype=np.float64)
    cols = cloud.shape[-2]
    if cols < 5:
        return 0, 0, 0
    curv = evaluated(curvature_np(cloud), cols)
    with np.errstate(all="ignore"):
        dev = np.abs(curv - 0.1)
        taps = taps_np(cloud)
        avg = (((taps[..., 0] + taps[..., 1]) + taps[..., 2]) + taps[..., 3]) / 4
        g = 64 * U24 * (2 * np.sqrt(curv) * avg / np.sqrt(avg * avg + F32_EPS6) + curv) + 1e-9
        window = dev <= 0.5 * (MARGIN + g)
    bad = ~np.isfinite(curv)
    over = _fp32_square_overflows(cloud)
    must = window | bad | over
    thin = window & (dev > THIN) & ~bad & ~over
    win = ~np.isfinite(cloud).all(axis=-1)
    win_bad = np.zeros(curv.shape, dtype=bool)
    for k in (-2, -1, 0, 1, 2):
        win_bad |= win[..., 2 + k:cols - 2 + k]
    may = (dev <= 1e-4) | bad | win_bad | (taps >= 2.0 ** 60).any(axis=-1)
    return int(must.sum()), int(may.sum()), int(thin.sum())


@functools.lru_cache(maxsize=None)
def _images(shape, n_images, seed):
    img = near_threshold_images(shape, n_images, seed)
    img.flags.writeable = False
    return img


def images(shape, n_images, seed):
    """a private copy of the cached near-threshold images"""
    return _images(shape, n_images, seed).copy()


def bounds_of(clouds):
    """fallback_bounds summed over several clouds"""
    return tuple(int(v) for v in np.sum([fallback_bounds(cl) for cl in clouds], axis=0))


def same_values(a, b):
    """bit for bit, except that a NaN matches any NaN (its payload follows the processor that formed it)"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.kind != "f":
        return a.tobytes() == b.tobytes()
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all()) and a[~na].tobytes() == b[~nb].tobytes()


# ------------------------------------------------------------------ 1-2. CPU: restatement and generator -----------
SHAPES = [(64, 2048), (1, 5), (2, 6), (3, 257), (2, 4100), (33, 1001)]
MAIN = ((64, 2048), 1, 1)   # the image the band counts are stated for
# evaluated pixels each band of MAIN must hold (measured about twice these)
MIN_BAND = {"<=1e-9": 3000, "(1e-9,1e-7]": 1500, "(1e-7,1e-5]": 2500, "(1e-5,1e-4]": 300}
MIN_PAIRS = 800
MIN_PER_SCALE = {"<=1e-9": 30, "<=1e-4": 150}   # group centres of every scale
MIN_THIN = 800   # pixels of MAIN that fallback_bounds counts as `thin` (measured 1120)
MAIN_EVALUATED = 64 * 2044


@pytest.mark.parametrize("shape", SHAPES)
def test_restatement_equals_oracle(oracle, shape):
    """curvature_np is the oracle's curvature bit for bit (NaN matching NaN) on near-threshold images."""
    for k, img in enumerate(images(shape, 2, 100 + shape[1])):
        assert same_values(curvature_np(img), oracle.curvature(img)), k


def test_generator_populates_every_band(oracle):
    img, meta = near_threshold_images(*MAIN, meta=True)
    img = img[0]
    assert same_values(curvature_np(img), oracle.curvature(img))
    counts = band_counts(img)
    for name, least in MIN_BAND.items():
        assert counts[name] >= least, (name, counts)
    # straddle pairs: one coordinate of the centre differs by one ulp and the labels differ
    r, c = meta["row"], meta["col"]
    lab = oracle.extract_feature(img)
    pairs = meta["pairs"]
    assert len(pairs) >= MIN_PAIRS
    a, b = img[r[pairs[:, 0]], c[pairs[:, 0]]], img[r[pairs[:, 1]], c[pairs[:, 1]]]
    diff = a != b
    assert (diff.sum(axis=1) == 1).all()
    assert (np.nextafter(a[diff], b[diff]) == b[diff]).all()
    assert (lab[r[pairs[:, 0]], c[pairs[:, 0]]] != lab[r[pairs[:, 1]], c[pairs[:, 1]]]).all()
    # every scale
    dev = np.abs(curvature_np(img)[r, c] - 0.1)
    for k, s in enumerate(SCALES):
        sel = meta["scale"] == k
        assert (dev[sel] <= 1e-9).sum() >= MIN_PER_SCALE["<=1e-9"], s
        assert (dev[sel] <= 1e-4).sum() >= MIN_PER_SCALE["<=1e-4"], s
    # the fallback bounds are ordered, and the lower one holds pixels only the kernel's own err sends to the
    # exact path
    lo, hi, thin = fallback_bounds(img)
    assert 0 < lo < hi and thin >= MIN_THIN, (lo, hi, thin)


@pytest.mark.parametrize("shape", SHAPES)
def test_group_centres_cover_every_tile_position(shape):
    """Across the images of one call the centres fall on every column residue mod 256, every flattened-index
    residue mod 240 (for images big enough to hold them), and on columns 2 and cols-3."""
    rows, cols = shape
    n = 4
    cen = np.array([(i, r, c) for i in range(n) for r, c in group_slots(rows, cols, i)])
    cc = set(cen[:, 2].tolist())
    assert 2 in cc and cols - 3 in cc
    flat = (cen[:, 0] * rows + cen[:, 1]) * cols + cen[:, 2]
    if cols - 4 >= 256:
        assert len(set((cen[:, 2] % 256).tolist())) == 256
    if n * rows * cols >= 5 * 240:
        assert len(set((flat % 240).tolist())) == 240


# ------------------------------------------------------------------ 3-4. GPU: every entry point that labels -------
GUARD = 4096   # bytes of canary on each side of a device output
POISON = 16    # NaN points on each side of a device input
Z6 = np.zeros(6)
STEP = np.array([46.0, 2.0, -1.0, 0.0, 0.0, 0.0])


def counted(ctx, fn):
    """(value of fn(), exact re-evaluations it caused): the context's 32-bit device counter, read synchronised on
    both sides of the call."""
    ctx.synchronize()
    before = ctx.exact_fallback_count()
    v = fn()
    ctx.synchronize()
    return v, (ctx.exact_fallback_count() - before) & 0xFFFFFFFF


def check_count(delta, clouds, what, floor=True):
    """delta within fallback_bounds of the clouds one call labelled.  floor: the clouds must also hold, per evaluated
    pixel, at least half of the band and thin-pixel counts stated for MAIN, so that the images reaching the kernels
    cannot silently become easy (off for calls on single tiny images; their totals are checked together)."""
    lo, hi, thin = bounds_of(clouds)
    if floor:
        print(f"{what}: {delta} exact re-evaluations, bounds [{lo}, {hi}]")
    assert lo <= delta <= hi, f"{what}: {delta} exact re-evaluations, expected [{lo}, {hi}]"
    if floor:
        n_eval = sum(cl[..., 2:-2, 0].size for cl in clouds)
        bands = {name: sum(band_counts(cl)[name] for cl in clouds) for name in MIN_BAND}
        for name, least in list(MIN_BAND.items()) + [("thin", MIN_THIN)]:
            got = thin if name == "thin" else bands[name]
            assert got >= int(0.5 * least * n_eval / MAIN_EVALUATED), (what, name, got, n_eval)


def kernels_run(torch, fn):
    """(value of fn(), names of the kernels it ran on the device), recorded with the CUDA profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        v = fn()
        torch.cuda.synchronize()
    return v, " ".join(e.name for e in prof.events())


def ran(names, kernel):
    """kernel (a name of csrc/, e.g. k_labels) among the profiled kernel names -- k_labels is not k_labels_tma"""
    return re.search(r"\b" + kernel + r"\b(?!_)", names) is not None


_CUDART = None


def dev_to_numpy(p, dtype, count):
    """copy `count` elements from a raw device pointer (buffers the context owns) to numpy"""
    global _CUDART
    if _CUDART is None:
        _CUDART = C.CDLL("libcudart.so")
    out = np.empty(count, dtype=dtype)
    rc = _CUDART.cudaMemcpy(C.c_void_p(out.ctypes.data), C.c_void_p(p), C.c_size_t(out.nbytes), C.c_int(2))
    assert rc == 0, rc
    return out


def unpack_mask(words, c):
    """label masks uint32 [..., ceil(c/16)] (bit i of word b = column 16 b + i) -> int32 labels [..., c]"""
    w = np.asarray(words).view(np.uint32)
    bits = (w[..., None] >> np.arange(16, dtype=np.uint32)) & 1
    return bits.reshape(w.shape[:-1] + (-1,))[..., :c].astype(np.int32)


class Guarded:
    """A device buffer of `nbytes` with canary guard bands on both sides."""

    def __init__(self, torch, nbytes):
        self.buf = torch.full((nbytes + 2 * GUARD,), CANARY, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()

    def ptr(self):
        return self.buf.data_ptr() + GUARD

    def get(self, dtype, shape):
        return self.buf.cpu().numpy()[GUARD:-GUARD].view(dtype).reshape(shape)

    def guards_intact(self):
        b = self.buf.cpu().numpy()
        return bool((b[:GUARD] == CANARY).all() and (b[-GUARD:] == CANARY).all())


def pinned(pkg, a):
    """page-lock a numpy array in place (nav_host_register); the caller unregisters it"""
    L = pkg.load_library()
    assert a.flags.c_contiguous
    assert L.nav_host_register(a.ctypes.data, a.nbytes) == 0, L.nav_last_error()
    return a


def unpin(pkg, a):
    pkg.load_library().nav_host_unregister(a.ctypes.data)


@gpu
@pytest.mark.parametrize("shape", [(64, 2048), (1, 5), (2, 6), (3, 257), (2, 4100)])
def test_extract_feature_and_curvature(pkg, oracle, shape):
    """nav_extract_feature (k_labels: 547 1-D tiles at 64x2048, too few for the TMA kernel) and nav_curvature
    (k_curvature, binary64 throughout) on near-threshold images: one at 64x2048, up to 64 of the smaller shapes
    (64 groups at 1x5, 128 at 2x6, about 460 in three 3x257 images), one call per image."""
    torch = pytest.importorskip("torch")
    n = max(1, min(64, 2500 // (shape[0] * shape[1])))
    imgs = images(shape, n, 200 + shape[1])
    ctx = pkg.Context(*shape, device=0)
    try:
        total = 0
        for k, img in enumerate(imgs):
            labels = lambda: counted(ctx, lambda: ctx.extract_feature(img))  # noqa: E731
            curvature = lambda: counted(ctx, lambda: ctx.curvature(img))  # noqa: E731
            if k == 0:   # the kernels reached, from the first image
                (got, delta), names = kernels_run(torch, labels)
                assert ran(names, "k_labels"), names
            else:
                got, delta = labels()
            assert np.array_equal(got, oracle.extract_feature(img)), k
            check_count(delta, [img], f"nav_extract_feature {shape[0]}x{shape[1]} image {k}", floor=False)
            total += delta
            if k == 0:
                (curv, delta), names = kernels_run(torch, curvature)
                assert ran(names, "k_curvature"), names
            else:
                curv, delta = curvature()
            assert same_values(curv, oracle.curvature(img)), k
            assert delta == 0   # the exact kernel has no fallback to count
        check_count(total, list(imgs), f"nav_extract_feature {shape[0]}x{shape[1]} x{n}")
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("shape,n,offset,kernel", [((64, 2048), 4, 0, "k_labels_tma"),
                                                   ((33, 1001), 5, 0, "k_labels_tma"),
                                                   ((64, 2048), 4, 8, "k_labels")])
def test_batch_labels(pkg, oracle, shape, n, offset, kernel):
    """nav_extract_feature_batch_dev: the 1-D tiles of k_labels_tma cross row and image boundaries (an odd point
    count at 5x33x1001: the last bulk copy ends on a hand-stored double); a cloud 8 bytes off the 16-byte rule
    goes to k_labels.  The batch sits between NaN points, so that a read past either end that fed an evaluated
    column would change a label, and the labels between canary guard bands."""
    torch = pytest.importorskip("torch")
    rows, cols = shape
    imgs = images(shape, n, 300 + cols + offset)
    n_pts = imgs.size // 3
    first = POISON * 3 + offset // 8
    buf = torch.full((2 * POISON * 3 + n_pts * 3 + 1,), float("nan"), dtype=torch.float64, device="cuda")
    buf[first:first + n_pts * 3] = torch.from_numpy(imgs.reshape(-1)).cuda()
    labels = Guarded(torch, n_pts * 4)
    ctx = pkg.Context(rows, cols, device=0)
    try:
        ctx.set_stream(torch.cuda.current_stream().cuda_stream)
        call = lambda: ctx.extract_feature_batch_dev(buf.data_ptr() + first * 8, n, labels.ptr())  # noqa: E731
        (_, delta), names = kernels_run(torch, lambda: counted(ctx, call))
        ctx.set_stream(None)
        assert ran(names, kernel), names
        assert labels.guards_intact()
        got = labels.get(np.int32, imgs.shape[:-1])
        for k in range(n):
            assert np.array_equal(got[k], oracle.extract_feature(imgs[k])), k
        check_count(delta, list(imgs), f"nav_extract_feature_batch_dev ({kernel})")
    finally:
        ctx.close()


@gpu
@pytest.mark.parametrize("n_seq", [1, 2])
def test_frontend_frame(pkg, oracle, n_seq):
    """nav_frontend_frame (k_frame_match, labels fused): labels, nn_idx, nn_dist and the global cloud of two
    near-threshold frames against a near-threshold map."""
    torch = pytest.importorskip("torch")
    shape = (64, 2048)
    r, c = shape
    frames = [images(shape, n_seq, 400 + 10 * n_seq + f) for f in range(3)]
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    slams = [oracle.slam(r, c, 1) for _ in range(n_seq)]
    one = (lambda a: a[0]) if n_seq == 1 else (lambda a: a)
    try:
        pos = np.stack([np.array([10.0 * s, -20.0, 5.0, 1.0, -2.0, 30.0]) for s in range(n_seq)])
        g = ctx.slam_init(one(pos), one(frames[0])).reshape(n_seq, r, c, 3)
        for s in range(n_seq):
            assert same_values(g[s], slams[s].init(pos[s], frames[0][s]))
        last = pos
        for f in (1, 2):
            pred = last + STEP + np.array([1.0, -0.5, 0.0, 0.0, 0.0, 0.1])
            final = pred + np.array([0.5, -0.5, 0.1, 0.0, 0.0, 0.0])
            cl = one(frames[f])
            (out, delta), names = kernels_run(torch, lambda: counted(ctx, lambda: ctx.frontend_frame(
                cl, one(pred), one(last), one(final))))
            assert ran(names, "k_frame_match"), names
            feat, idx, dist = (a.reshape(n_seq, r, c) for a in out[:3])
            glob = out[3].reshape(n_seq, r, c, 3)
            for s in range(n_seq):
                ofeat, oidx, odist, og = slams[s].frontend_frame(frames[f][s], pred[s], last[s], final[s])
                assert np.array_equal(feat[s], ofeat), (f, s)
                assert np.array_equal(idx[s], oidx), (f, s)
                assert same_values(dist[s], odist), (f, s)
                assert same_values(glob[s], og), (f, s)
            check_count(delta, list(frames[f]), "nav_frontend_frame")
            last = final
    finally:
        ctx.close()
        for s in slams:
            s.close()


def pose_chain(k, n_seq):
    """pred, last, final [k][n_seq][6] for frames 1..k; frame 0 is mapped at zero"""
    final = np.array([[(f + 1) * STEP + np.array([0.0, 0.5 * s, 0, 0, 0, 0]) for s in range(n_seq)] for f in range(k)])
    last = np.concatenate([np.zeros((1, n_seq, 6)), final[:-1]])
    pred = last + STEP + np.array([1.0, -0.5, 0.0, 0.0, 0.0, 0.1])
    return pred, last, final


@gpu
@pytest.mark.parametrize("shape,k,kernel", [((64, 2048), 6, "k_frame_seq"), ((2, 4100), 6, "k_frame_match")])
def test_sequence_out(pkg, oracle, shape, k, kernel):
    """nav_frontend_sequence_out_dev over k near-threshold frames: one k_frame_seq launch (double-buffered tiles)
    at 64x2048, one k_frame_match launch per frame for rows wider than a cluster.  Every frame's label mask,
    nn_idx and nn_dist against the oracle driven along the same poses."""
    torch = pytest.importorskip("torch")
    r, c = shape
    frames = np.stack([images(shape, 1, 500 + c + f) for f in range(k + 1)])   # [k+1][1][r][c][3]
    pred, last, final = pose_chain(k, 1)
    d_frames = torch.from_numpy(frames).cuda()
    nch = -(-c // 16)
    mask = torch.zeros((k, 1, r, nch), dtype=torch.int32, device="cuda")
    idx = torch.zeros((k, 1, r, c), dtype=torch.int32, device="cuda")
    dist = torch.zeros((k, 1, r, c), dtype=torch.float64, device="cuda")
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    try:
        ctx.slam_init_dev(d_frames[0].data_ptr(), np.zeros((1, 6)))
        call = lambda: ctx.frontend_sequence_out_dev(  # noqa: E731
            d_frames[1].data_ptr(), k, pred.reshape(-1, 6), last.reshape(-1, 6), final.reshape(-1, 6),
            label_mask=mask.data_ptr(), nn_idx=idx.data_ptr(), nn_dist=dist.data_ptr())
        (_, delta), names = kernels_run(torch, lambda: counted(ctx, call))
        assert ran(names, kernel), names
        mask, idx, dist = mask.cpu().numpy(), idx.cpu().numpy(), dist.cpu().numpy()
        slam.init(Z6, frames[0, 0])
        for f in range(k):
            ofeat, oidx, odist, _ = slam.frontend_frame(frames[f + 1, 0], pred[f, 0], last[f, 0], final[f, 0])
            lab = ofeat == 1
            assert np.array_equal(unpack_mask(mask[f, 0], c), ofeat), f
            assert np.array_equal(idx[f, 0][lab], oidx[lab]), f
            assert same_values(dist[f, 0][lab], odist[lab]), f
            assert (idx[f, 0][~lab] == -1).all() and (dist[f, 0][~lab] == -1.0).all(), f
        check_count(delta, [frames[f + 1, 0] for f in range(k)], f"nav_frontend_sequence_out_dev ({kernel})")
    finally:
        ctx.close()
        slam.close()


def deltas_of(k, n_seq, seed):
    rng = np.random.default_rng(seed)
    d = np.tile(STEP, (k, n_seq, 1)) + rng.uniform(-3.0, 3.0, (k, n_seq, 6)) * np.array([1, 1, 1, 0, 0, 0])
    d[..., 5] += rng.uniform(-0.4, 0.4, (k, n_seq))
    return d


@gpu
def test_slam_run(pkg, oracle):
    """nav_slam_run over k near-threshold frames: the labels of every frame come from the prefetch (k_labels),
    k_loop_step matches and fits.  Per frame the correspondence count equals the oracle's at the returned poses;
    the last frame's labels (the map's edge masks) and global cloud equal the oracle's."""
    torch = pytest.importorskip("torch")
    shape, k = (64, 2048), 4
    r, c = shape
    frames = np.ascontiguousarray(np.stack([images(shape, 1, 600 + f)[0] for f in range(k + 1)]))
    deltas = deltas_of(k, 1, 7)[:, 0]
    ctx = pkg.Context(r, c, device=0)
    slam = oracle.slam(r, c, 1)
    pinned(pkg, frames)
    try:
        ctx.slam_init(Z6, frames[0], want_global=False)
        call = lambda: ctx.slam_run([frames[f].ctypes.data for f in range(1, k + 1)], deltas, Z6)  # noqa: E731
        ((poses, _, n_corr), delta), names = kernels_run(torch, lambda: counted(ctx, call))
        assert ran(names, "k_labels") and ran(names, "k_loop_step"), names
        res = ctx.frame_results_dev()
        map_mask = dev_to_numpy(res.map_mask, np.uint32, r * -(-c // 16)).reshape(r, -1)
        glob = dev_to_numpy(res.global_, np.float64, r * c * 3).reshape(r, c, 3)
        slam.init(Z6, frames[0])
        last = Z6
        for t in range(k):
            _, corr, _, _ = slam.localize(frames[t + 1], last + deltas[t], last)
            assert n_corr[t] == corr.shape[0], t
            og = slam.map(poses[t], frames[t + 1])
            last = poses[t]
        assert n_corr.sum() > 0
        assert np.array_equal(unpack_mask(map_mask, c), oracle.extract_feature(frames[k]))
        assert same_values(glob, og)
        check_count(delta, list(frames[1:]), "nav_slam_run")
    finally:
        unpin(pkg, frames)
        ctx.close()
        slam.close()


@gpu
@pytest.mark.parametrize("shape,n_seq", [((64, 2048), 1), ((16, 1800), 3)])
def test_slam_run_dev(pkg, oracle, shape, n_seq):
    """nav_slam_run_dev over k near-threshold frames: the device variant of k_loop_step labels every frame itself.
    Per frame and sequence fit_stats[t][s][0] equals the oracle's correspondence count at the device's poses; the
    last frame's labels (nav_frame_results_dev) equal the oracle's."""
    torch = pytest.importorskip("torch")
    k = 4
    r, c = shape
    frames = np.ascontiguousarray(np.stack([images(shape, n_seq, 700 + 10 * n_seq + f) for f in range(k + 1)]))
    deltas = deltas_of(k, n_seq, 11)
    start = np.zeros((n_seq, 6))
    d_frames = torch.from_numpy(frames).cuda()
    poses = torch.full((k, n_seq, 6), -7.0, dtype=torch.float64, device="cuda")
    stats = torch.full((k, n_seq, 5), -7.0, dtype=torch.float64, device="cuda")
    ctx = pkg.Context(r, c, device=0, n_seq=n_seq)
    slams = [oracle.slam(r, c, 1) for _ in range(n_seq)]
    try:
        ctx.slam_init(start if n_seq > 1 else start[0], frames[0] if n_seq > 1 else frames[0, 0], want_global=False)
        call = lambda: ctx.slam_run_dev(d_frames[1].data_ptr(), k, deltas.reshape(-1, 6), start,  # noqa: E731
                                        poses.data_ptr(), None, stats.data_ptr())
        (_, delta), names = kernels_run(torch, lambda: counted(ctx, call))
        assert ran(names, "k_loop_step"), names
        assert not ran(names, "k_labels") and not ran(names, "k_labels_tma"), names
        poses, stats = poses.cpu().numpy(), stats.cpu().numpy()
        labels = dev_to_numpy(ctx.frame_results_dev().labels, np.int32, n_seq * r * c).reshape(n_seq, r, c)
        for s in range(n_seq):
            slams[s].init(start[s], frames[0, s])
            last = start[s]
            for t in range(k):
                _, corr, _, _ = slams[s].localize(frames[t + 1, s], last + deltas[t, s], last)
                assert stats[t, s, 0] == corr.shape[0], (t, s)
                slams[s].map(poses[t, s], frames[t + 1, s])
                last = poses[t, s]
            assert np.array_equal(labels[s], oracle.extract_feature(frames[k, s])), s
        assert stats[:, :, 0].sum() > 0
        check_count(delta, [frames[t, s] for t in range(1, k + 1) for s in range(n_seq)], "nav_slam_run_dev")
    finally:
        ctx.close()
        for s in slams:
            s.close()
