"""The large-map kd build (csrc/kdbuild.cu) against the exact reference tree, on every path the build can take.

The tree is fully defined, ties included (kdbuild.cu:4-14): the node of [lo,hi) is the element of rank (hi-lo)/2 in
the order (key on the split axis, build index), the axis is level % 3 (cyclic rule) or the axis of the widest extent
of the segment's key box (widest rule, split_of: NaN extents and ties keep the lowest axis).  `ref_tree` restates
that in numpy, level by level, and the GPU tests compare `KdTree.export(with_axes=True)` with it bit for bit: nodes
as uint64 views (NaN payloads and the sign of zero count), build indices and axes.

Which kernels order a segment depends on its size: above mid_cap points (16 384, or NAV_KD_MIDCAP, read once per
process) the multi-CTA kernels k_kd_hist / k_kd_hist2 / k_kd_partition / k_kd_resolve, above kFinSeg = 2048
k_kd_level_cta, below that k_kd_finish.  Inside those, counting_argsort takes a one-level count, a second-level
subdivision or the bitonic network; a crowded median bin takes a second selection round, then narrowing rounds on the
key and on the point index; bin_range clips a bin's upper key where it would pass 2^64.  `census` restates the bin
arithmetic of every one of those decisions on the CPU, and the CPU tests hold the point families below to a stated
number of segments per branch, so a family that stops reaching its branch fails here rather than silently testing
less.  The GPU tests run every family at the sizes where the paths switch, at 1 M points with both split rules on
the host and the device-pointer entry points, through a worker process per NAV_KD_MIDCAP value (2049: every level
above the finisher on the multi-CTA kernels; 2^30: whole large segments in one CTA), and once at 10 M points, and
check the answers of every 1 M / 10 M tree against the fp64 brute force.

Some of those decisions only choose between correct orderings, so no tree can tell them apart: the kBucketMax
threshold (one-level count, second level or bitonic: all three order exactly), the pre = shift - 52 rescale (shift is
at most 53 and a bucket holds at most 2048 points, so (low * n_b) fits in 64 bits without it, and any monotone
sub-bucket map orders correctly) and the clamp sub = min(sub, nb - 1) (low < 2^shift keeps sub below nb).  The census
still counts them, so that a rewrite that makes one of those branches wrong is caught by the families that reach it."""
import functools
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIGN = np.uint64(1 << 63)
K_BINS, K_BIN_BITS, K_CAP, K_FIN_SEG, K_BUCKET_MAX, K_CHUNK = 2048, 11, 2048, 2048, 48, 4096
MID_CAP = 16384
U64_MAX = (1 << 64) - 1

# families of the existing exact tests, plus ones aimed at single branches (see family())
FAMILIES = ["uniform", "clustered", "duplicates", "integer", "planes", "slab", "ties49", "special", "all_equal",
            "int_walls", "far_dense", "top_crowd", "walls"]
NO_NAN = [f for f in FAMILIES if f != "special"]


# ------------------------------------------------------------------ restatement of the build ----------------------
def order_keys(pts):
    """order_key of kdbuild.cu on float64.view(uint64): (3, n) keys, monotone in the coordinate, -NaN lowest,
    +NaN highest, -0 below +0."""
    b = np.ascontiguousarray(np.asarray(pts, dtype=np.float64).reshape(-1, 3)).view(np.uint64).T
    return np.ascontiguousarray(np.where((b >> np.uint64(63)) != 0, ~b, b | SIGN))


def key_value(k):
    k = np.asarray(k, dtype=np.uint64)
    return np.where((k >> np.uint64(63)) != 0, k & ~SIGN, ~k).view(np.float64)


def bin_shift(r):
    """smallest shift with (r >> shift) < kBins, elementwise"""
    r = np.atleast_1d(np.asarray(r, dtype=np.uint64))
    bits = np.zeros(r.shape, np.int64)
    for b in range(64):
        bits[(r >> np.uint64(b)) != 0] = b + 1
    return np.maximum(bits - K_BIN_BITS, 0)


def levels_of(n, mid_cap=MID_CAP):
    """(level0, top_levels) of kd_build: levels < top_levels take the multi-CTA kernels, the rest below level0
    k_kd_level_cta, level0 the finisher"""
    level0 = 0
    while (n >> level0) > K_FIN_SEG:
        level0 += 1
    top = 0
    while top < level0 and (n >> top) > mid_cap:
        top += 1
    return level0, top


def launches_of(n, mid_cap=MID_CAP):
    """kernel launches of one kd_build: init + keys, four per multi-CTA level, one per level_cta level, finisher"""
    if n == 0:
        return 0
    level0, top = levels_of(n, mid_cap)
    return 2 + 4 * top + (level0 - top) + 1


def widest_axis(lo_key, hi_key):
    """split_of's widest rule on (3, s) key boxes: extent in value space, NaN extents and ties keep the lowest axis"""
    with np.errstate(invalid="ignore", over="ignore"):
        e = key_value(hi_key) - key_value(lo_key)
        axis = np.zeros(e.shape[1], np.int64)
        axis[e[1] > e[0]] = 1
        axis[e[2] > e[axis, np.arange(e.shape[1])]] = 2
    return axis


BRANCHES = ["fin_count1", "fin_count2", "fin_bitonic", "res_count1", "res_count2", "res_bitonic", "pre",
            "crowded", "round2_key", "round2_index", "crowded_after_round2", "level_cta_crowded", "narrow_index",
            "clip", "clip_narrow"]


def _counting(keys, klo, khi):
    """counting_argsort's choice on keys (uint64) with the key range [klo, khi]: 'count1', 'count2' or 'bitonic',
    and whether the second level rescaled by pre = shift - 52"""
    shift = int(bin_shift(np.uint64(khi - klo))[0])
    off = keys - np.uint64(klo)
    bins = (off >> np.uint64(shift)).astype(np.int64)
    h = np.bincount(bins, minlength=K_BINS)
    if h.max() <= K_BUCKET_MAX:
        return "count1", False
    start = np.concatenate([[0], np.cumsum(h)[:-1]])
    pre = shift - 52 if shift > 52 else 0
    nb = h[bins].astype(np.uint64)
    low = off & np.uint64((1 << shift) - 1)
    sub = ((low >> np.uint64(pre)) * nb) >> np.uint64(shift - pre)
    sub = np.minimum(sub, nb - np.uint64(1)).astype(np.int64)
    h2 = np.bincount(start[bins] + sub, minlength=K_BINS)
    return ("bitonic" if h2.max() > K_BUCKET_MAX else "count2"), pre > 0


def _pick(sub, r):
    """bin holding rank r of a monotone bin sequence: (bin, below, count)"""
    b = int(sub[r])
    below = int(np.searchsorted(sub, b, "left"))
    return b, below, int(np.searchsorted(sub, b, "right")) - below


def _narrow(keys, ids, r, klo, khi):
    """resolve_region's narrowing rounds over more than kCap candidates (keys / ids in (key, index) order); True
    when they reach the round on the point index"""
    cnt, by_id, ilo, ihi = len(keys), False, 0, 0x7FFFFFFF
    while cnt > K_CAP:
        if not by_id and klo == khi:
            by_id = True
        if not by_id:
            sh = int(bin_shift(np.uint64(khi - klo))[0])
            sel = (keys >= np.uint64(klo)) & (keys <= np.uint64(khi))
            sub = ((keys[sel] - np.uint64(klo)) >> np.uint64(sh)).astype(np.int64)
        else:
            sh = int(bin_shift(np.uint64(ihi - ilo))[0])
            sel = (keys == np.uint64(klo)) & (ids >= ilo) & (ids <= ihi)
            sub = (ids[sel] - ilo) >> sh
        b2, below2, cnt = _pick(sub, r)
        r -= below2
        if not by_id:
            klo += b2 << sh
            khi = min(khi, klo + (1 << sh) - 1)
        else:
            ilo += b2 << sh
            ihi = min(ihi, ilo + (1 << sh) - 1)
    return by_id


def _census_level(stats, skeys, sids, starts, sizes, base, hi_key, shift, multi, n):
    """the selection of one level above the finisher, per segment: skeys / sids are the live points in (segment,
    key, index) order, base / hi_key / shift the split of every segment"""
    for s in range(len(starts)):
        a, m = int(starts[s]), int(sizes[s])
        keys, ids = skeys[a:a + m], sids[a:a + m]
        sh, bse = int(shift[s]), int(base[s])
        b, below, cnt = _pick(((keys - np.uint64(bse)) >> np.uint64(sh)).astype(np.int64), m >> 1)
        klo, span = bse + (b << sh), (1 << sh) - 1
        clipped = klo + span > U64_MAX    # bin_range's khi would not fit in 64 bits
        stats["clip"] += clipped
        khi = klo + span if int(hi_key[s]) - klo > span else int(hi_key[s])
        ck, ci = keys[below:below + cnt], ids[below:below + cnt]
        r = (m >> 1) - below
        if multi and cnt > K_CAP:
            stats["crowded"] += 1
            if sh == 0:      # one key value: second round on the leading bits of the point index
                stats["round2_index"] += 1
                id_bits = max(n - 1, 1).bit_length()
                sub = ci >> max(id_bits - K_BIN_BITS, 0)
            else:
                stats["round2_key"] += 1
                sh2 = max(sh - K_BIN_BITS, 0)
                sub = ((ck - np.uint64(klo)) >> np.uint64(sh2)).astype(np.int64)
            b2, below2, cnt = _pick(sub, r)
            if sh != 0:
                lo2, span2 = klo + (b2 << sh2), (1 << sh2) - 1
                khi = lo2 + span2 if khi - lo2 > span2 else khi
                klo = lo2
            ck, ci, r = ck[below2:below2 + cnt], ci[below2:below2 + cnt], r - below2
            if cnt > K_CAP:
                stats["crowded_after_round2"] += 1
        elif cnt > K_CAP:
            stats["level_cta_crowded"] += 1
        if cnt > K_CAP:
            stats["narrow_index"] += _narrow(ck, ci, r, klo, khi)
            stats["clip_narrow"] += clipped
        else:
            outcome, pre = _counting(ck, klo, khi)
            stats["res_" + outcome] += 1
            stats["pre"] += pre


def ref_tree(pts, split, mid_cap=MID_CAP, stats=None):
    """The exact tree of kdbuild.cu: (nodes, oidx, axes) as KdTree.export(with_axes=True) returns them.  With a
    dict `stats`, also counts the segments (and finisher axes) that take each branch of BRANCHES on the paths
    that mid_cap selects."""
    pts = np.ascontiguousarray(np.asarray(pts, dtype=np.float64).reshape(-1, 3))
    n = pts.shape[0]
    axes = np.zeros(n, np.int32)
    if n == 0:
        return pts.copy(), np.zeros(0, np.int32), axes
    K = order_keys(pts)
    ar = np.arange(n, dtype=np.int64)
    order = np.stack([np.lexsort((ar, K[d])) for d in range(3)])     # (key, index) order per axis
    rank = np.empty((3, n), np.int64)
    for d in range(3):
        rank[d, order[d]] = ar
    perm = ar.copy()                    # position -> build index
    level0, top = levels_of(n, mid_cap)
    seg_lo, seg_hi = np.array([0]), np.array([n])
    fin_m = None                        # size of the finisher segment a segment lies in (levels >= level0)
    level = 0
    while len(seg_lo):
        sizes = seg_hi - seg_lo
        starts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
        mark = np.zeros(n + 1, np.int64)
        np.add.at(mark, seg_lo, 1)
        np.add.at(mark, seg_hi, -1)
        live = np.nonzero(np.cumsum(mark)[:n])[0]
        g = np.repeat(np.arange(len(seg_lo)), sizes)
        lp = perm[live]
        lo_key = np.empty((3, len(seg_lo)), np.uint64)
        hi_key = np.empty((3, len(seg_lo)), np.uint64)
        for d in range(3):
            r = rank[d, lp]
            lo_key[d] = K[d, order[d, np.minimum.reduceat(r, starts)]]
            hi_key[d] = K[d, order[d, np.maximum.reduceat(r, starts)]]
        if split == "cyclic":
            axis = np.full(len(seg_lo), level % 3, np.int64)
        else:
            axis = widest_axis(lo_key, hi_key)
        if level == level0:
            fin_m = sizes.copy()
        if level >= level0:   # the finisher sets no axis once its largest sub-segment holds a single point
            axis = np.where((fin_m >> (level - level0)) >= 2, axis, 0)
        comp = g * n + rank[axis[g], lp]
        lp = lp[np.argsort(comp)]
        perm[live] = lp
        mid = seg_lo + sizes // 2
        axes[mid] = axis
        if stats is not None:
            sg = np.arange(len(seg_lo))
            if level < level0:
                skeys = K[axis[g], lp]
                span = hi_key[axis, sg] - lo_key[axis, sg]
                _census_level(stats, skeys, lp, starts, sizes, lo_key[axis, sg], hi_key[axis, sg], bin_shift(span),
                              level < top, n)
            elif level == level0:
                for s in range(len(seg_lo)):
                    seg = lp[starts[s]:starts[s] + sizes[s]]
                    for d in range(3):
                        outcome, pre = _counting(K[d, seg], int(lo_key[d, s]), int(hi_key[d, s]))
                        stats["fin_" + outcome] += 1
                        stats["pre"] += pre
        lo2 = np.stack([seg_lo, mid + 1], 1).ravel()
        hi2 = np.stack([mid, seg_hi], 1).ravel()
        keep = hi2 > lo2
        if fin_m is not None:
            fin_m = np.repeat(fin_m, 2)[keep]
        seg_lo, seg_hi = lo2[keep], hi2[keep]
        level += 1
    return pts[perm], perm.astype(np.int32), axes


def census(pts, split, mid_cap=MID_CAP):
    stats = dict.fromkeys(BRANCHES, 0)
    ref_tree(pts, split, mid_cap, stats)
    return stats


# ------------------------------------------------------------------ point families -------------------------------
def special_values(rng, size):
    """+-1e300, +-inf, NaN of both signs with two payloads, +-0 and subnormals"""
    v = np.array([1e300, -1e300, np.inf, -np.inf, 0.0, -0.0, 5e-324, -5e-324, 2.2e-308, -1e-310])
    nans = np.array([0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000001, 0xFFF4000000000123],
                    dtype=np.uint64).view(np.float64)
    return rng.choice(np.concatenate([v, nans]), size)


@functools.lru_cache(maxsize=None)
def _family(kind, n):
    rng = np.random.default_rng([FAMILIES.index(kind), n])
    if kind == "uniform":
        pts = rng.uniform(0.0, 1.0, (n, 3)) * np.array([1e5, 1e5, 1e4])
    elif kind == "clustered":   # surfaces of 64 boxes: many nearly equal coordinates on one axis
        c = rng.uniform(0.0, 1.0, (64, 3)) * np.array([1e5, 1e5, 1e4])
        half = rng.uniform(500.0, 4000.0, (64, 3))
        which, face = rng.integers(0, 64, n), rng.integers(0, 6, n)
        u = rng.uniform(-1.0, 1.0, (n, 3))
        u[np.arange(n), face // 2] = np.where(face % 2 == 0, -1.0, 1.0)
        pts = c[which] + half[which] * u + rng.normal(0.0, 5.0, (n, 3))
    elif kind == "duplicates":  # four copies of every point, at scattered build indices
        pts = np.repeat(rng.normal(0, 100, ((n + 3) // 4, 3)), 4, axis=0)[:n][rng.permutation(n)]
    elif kind == "integer":
        pts = rng.integers(0, 40, (n, 3)).astype(np.float64)
    elif kind == "planes":      # one coordinate on a wall per point
        pts = rng.uniform(-4000, 4000, (n, 3))
        pts[np.arange(n), rng.integers(0, 3, n)] = rng.choice([-4000.0, 4000.0], n)
    elif kind == "slab":
        # a thin slab (z within 1 mm) plus far outliers: the outliers stretch the key range of every segment they
        # are in, so the slab lands in a few first-level bins of the counting sort (second-level subdivision)
        pts = np.stack([rng.uniform(0, 8000, n), rng.uniform(0, 8000, n), 1000.0 + rng.uniform(0, 1, n)], 1)
        out = rng.random(n) < 0.02
        pts[out, 2] = rng.choice([-1.0, 1.0], int(out.sum())) * rng.uniform(1e5, 1e6, int(out.sum()))
    elif kind == "ties49":      # 8 values per axis: hundreds of equal keys in every finisher segment (bitonic)
        pts = rng.integers(0, 8, (n, 3)).astype(np.float64) * 250.0
    elif kind == "special":
        # a dense cluster near 0 mixed with special values on single coordinates: key ranges of 2^63 and more
        # (pre, bin_range clipping), NaN and inf extents under the widest rule
        pts = rng.normal(0.0, 1.0, (n, 3))
        hit = rng.random((n, 3)) < 0.06
        pts[hit] = special_values(rng, int(hit.sum()))
    elif kind == "all_equal":
        pts = np.full((n, 3), 3.25)
    elif kind == "int_walls":   # integer millimetres, two thirds of the points on four walls
        pts = np.rint(rng.uniform(-8000, 8000, (n, 3)))
        wall = rng.random(n) < 0.67
        ax = rng.integers(0, 2, n)
        pts[np.arange(n)[wall], ax[wall]] = rng.choice([-8000.0, 8000.0], int(wall.sum()))
    elif kind == "far_dense":   # a 1e4 mm lattice with 1 mm jitter centred at (1e9, -1e9, 5e8)
        k = int(np.ceil(n ** (1 / 3)))
        gr = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), -1).reshape(-1, 3)[rng.permutation(k ** 3)[:n]]
        pts = np.array([1e9, -1e9, 5e8]) + (gr + 0.5) * (1e4 / k) - 5e3 + rng.normal(0, 1, (n, 3))
    elif kind == "top_crowd":
        # x: more than half of the points at the largest finite double, the rest spread, one -NaN and one +NaN
        # stretching the key box to (almost) 2^64: the median bin is the top one, whose upper key bin_range clips,
        # and it holds more candidates than fit in shared memory
        pts = rng.normal(0.0, 1e3, (n, 3))
        top = rng.random(n) < 0.6
        pts[top, 0] = np.finfo(np.float64).max
        if n >= 2:
            pts[:2, 0] = np.array([0x7FF8000000000000, 0xFFF8000000000000], np.uint64).view(np.float64)
    elif kind == "walls":       # uniform in a 100 m x 100 m x 10 m volume, 40 % of the points on eight walls
        pts = rng.uniform(0.0, 1.0, (n, 3)) * np.array([1e5, 1e5, 1e4])
        wall = np.nonzero(rng.random(n) < 0.4)[0]
        pts[wall, rng.integers(0, 2, wall.size)] = rng.choice([0.0, 2.5e4, 7.5e4, 1e5], wall.size)
    else:
        raise ValueError(kind)
    pts = np.ascontiguousarray(pts, dtype=np.float64)
    pts.setflags(write=False)
    return pts


def family(kind, n):
    return _family(kind, n)


@functools.lru_cache(maxsize=None)
def _ref(kind, n, split):
    return ref_tree(family(kind, n), split)


def _check_ordered(nodes_keys, oidx, axes, split, n):
    """in-order layout with the strict (key, index) order: every element left of a node is smaller, every element
    right of it larger; the axis follows the rule"""
    stack = [(0, n, 0)]
    while stack:
        lo, hi, d = stack.pop()
        if hi - lo <= 1:
            continue
        mid = lo + (hi - lo) // 2
        a = int(axes[mid])
        if split == "cyclic":
            assert a == d % 3
        else:
            assert a == int(widest_axis(nodes_keys[:, lo:hi].min(axis=1, keepdims=True),
                                        nodes_keys[:, lo:hi].max(axis=1, keepdims=True))[0])
        k, i = nodes_keys[a, mid], oidx[mid]
        kl, il = nodes_keys[a, lo:mid], oidx[lo:mid]
        kr, ir = nodes_keys[a, mid + 1:hi], oidx[mid + 1:hi]
        assert ((kl < k) | ((kl == k) & (il < i))).all()
        assert ((kr > k) | ((kr == k) & (ir > i))).all()
        stack.append((lo, mid, d + 1))
        stack.append((mid + 1, hi, d + 1))


def assert_same_tree(got, want):
    nodes, oidx, axes = got
    wn, wi, wa = want
    assert nodes.shape == wn.shape
    bad = np.nonzero((nodes.view(np.uint64) != wn.view(np.uint64)).any(axis=1) | (oidx != wi) | (axes != wa))[0]
    assert bad.size == 0, f"{bad.size} nodes differ, first at {bad[:8]}: got idx {oidx[bad[:4]]} axis " \
                          f"{axes[bad[:4]]}, want idx {wi[bad[:4]]} axis {wa[bad[:4]]}"


# ------------------------------------------------------------------ CPU: the restatement ----------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 17, 1000, 2049, 5000, 40000])
def test_reference_equals_oracle_tree(oracle, n):
    """distinct keys, cyclic rule: the reference's recursive median split (utils/kdtree.c:65-82) leaves the same
    in-order array"""
    pts = family("uniform", n)
    h, want = oracle.tree_build(pts)
    oracle.tree_free(h)
    nodes, oidx, axes = ref_tree(pts, "cyclic")
    assert np.array_equal(nodes, want)
    assert np.array_equal(nodes, pts[oidx])


@pytest.mark.parametrize("split", ["widest", "cyclic"])
@pytest.mark.parametrize("kind", NO_NAN)
def test_reference_is_ordered(kind, split):
    """every family without NaN: a permutation, the strict (key, index) in-order property, the split rule"""
    n = 20000
    pts = family(kind, n)
    nodes, oidx, axes = ref_tree(pts, split)
    assert np.array_equal(np.sort(oidx), np.arange(n))
    assert np.array_equal(nodes.view(np.uint64), pts[oidx].view(np.uint64))
    _check_ordered(order_keys(nodes), oidx, axes, split, n)


def test_reference_keys_and_axis_rule():
    """order_key is monotone over the special values, key_value its exact inverse; the widest rule keeps the lowest
    axis on ties and NaN extents"""
    rng = np.random.default_rng(1)
    v = np.concatenate([special_values(rng, 200), rng.normal(0, 1e3, 200)])
    pts = np.stack([v, v[::-1], -v], 1)
    assert np.array_equal(key_value(order_keys(pts)).T.view(np.uint64), pts.view(np.uint64))
    fin = v[~np.isnan(v)]
    kf = order_keys(np.repeat(fin, 3))[0]
    f = fin[np.argsort(kf, kind="stable")]
    assert (f[1:] >= f[:-1]).all()
    assert order_keys([-0.0, 0.0, 0.0])[0, 0] < order_keys([0.0, 0.0, 0.0])[0, 0]
    lo = order_keys(np.array([[0.0, 0.0, 0.0], [0.0, -np.inf, 0.0], [0.0, 0.0, 0.0]]))
    hi = order_keys(np.array([[1.0, 1.0, 1.0], [np.nan, np.inf, 1.0], [1.0, np.nan, 5.0]]))
    assert list(widest_axis(lo, hi)) == [0, 0, 2]
    assert list(widest_axis(order_keys([[0.0, 0.0, -np.inf]]), order_keys([[0.0, 0.0, np.inf]]))) == [2]


def test_launch_formula():
    assert launches_of(2048) == 3 and launches_of(2049) == 4
    assert launches_of(16384) == 2 + 3 + 1 and launches_of(16385) == 2 + 4 + 2 + 1
    assert launches_of(1 << 20) == 2 + 4 * 6 + 3 + 1
    assert launches_of(1 << 20, mid_cap=2049) == 2 + 4 * 9 + 1
    assert launches_of(1 << 20, mid_cap=1 << 30) == 2 + 9 + 1


# ------------------------------------------------------------------ CPU: every branch is reached ----------------------
# (family, n, split, mid_cap) -> stated minimum number of segments (finisher: segment axes) per branch.  The minima
# sit well below the counts the families give, so a family that stops reaching a branch fails here.
BRANCH_CASES = [
    (("uniform", 1 << 20, "widest", MID_CAP), {"fin_count1": 1000, "res_count1": 300}),
    (("slab", 1 << 20, "cyclic", MID_CAP), {"fin_count1": 500, "fin_count2": 15, "crowded_after_round2": 10,
                                            "level_cta_crowded": 50}),
    (("clustered", 300000, "cyclic", MID_CAP), {"res_count2": 3, "fin_count2": 100}),
    (("ties49", 100000, "widest", MID_CAP), {"fin_bitonic": 100, "res_bitonic": 20, "level_cta_crowded": 4,
                                             "narrow_index": 5}),
    (("special", 1 << 20, "widest", MID_CAP), {"pre": 500, "fin_count2": 400, "narrow_index": 10}),
    (("special", 1 << 20, "cyclic", MID_CAP), {"fin_bitonic": 300, "level_cta_crowded": 100}),
    (("all_equal", 1 << 20, "cyclic", MID_CAP), {"crowded": 30, "round2_index": 30, "level_cta_crowded": 200,
                                                 "narrow_index": 200, "fin_bitonic": 1000, "res_bitonic": 30}),
    (("int_walls", 1 << 20, "widest", MID_CAP), {"crowded": 15, "round2_key": 15, "crowded_after_round2": 5,
                                                 "fin_bitonic": 200, "fin_count2": 70}),
    (("int_walls", 1 << 20, "widest", 2049), {"crowded": 60, "crowded_after_round2": 5, "narrow_index": 5}),
    (("top_crowd", 100000, "cyclic", 1 << 30), {"clip": 1, "level_cta_crowded": 5, "clip_narrow": 1}),
    (("top_crowd", 100000, "cyclic", 2049), {"clip": 1, "crowded": 5, "round2_key": 5, "round2_index": 1,
                                              "crowded_after_round2": 1, "clip_narrow": 1}),
]


@pytest.mark.parametrize("case,least", BRANCH_CASES, ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else "")
def test_families_reach_every_branch(case, least):
    kind, n, split, mid_cap = case
    got = census(family(kind, n), split, mid_cap)
    for branch, m in least.items():
        assert got[branch] >= m, (branch, got)


def test_every_branch_is_in_a_case():
    assert set(BRANCHES) == {b for _, least in BRANCH_CASES for b in least}


# ------------------------------------------------------------------ GPU: the kernels against the reference ----------
SWITCH_SIZES = [2047, 2048, 2049, 4095, 4096, 4097, 16384, 16385, 32769]   # level0, kChunkElems and mid_cap steps
POW20 = [(1 << 20) - 1, 1 << 20, (1 << 20) + 1]
POW20_FAMILIES = ["uniform", "special", "int_walls", "all_equal"]
BIG = 1_000_000


def gpu_tree(pkg, pts, split, stream=None):
    """(export, launch count) of a build from the host, or, with a torch stream, from device memory on that stream"""
    if stream is None:
        tree = pkg.KdTree(pts, device=0, split=split)
    else:
        import torch
        d_pts = torch.from_numpy(pts.copy()).cuda()
        stream.wait_stream(torch.cuda.current_stream())
        tree = pkg.KdTree(dev_ptr=d_pts.data_ptr(), n=pts.shape[0], stream=stream.cuda_stream, device=0, split=split)
        d_pts.record_stream(stream)
    try:
        return tree.export(with_axes=True), tree.launch_count()
    finally:
        tree.close()


@gpu
@pytest.mark.parametrize("split", ["widest", "cyclic"])
@pytest.mark.parametrize("kind", FAMILIES)
@pytest.mark.parametrize("n", SWITCH_SIZES)
def test_tree_at_switch_sizes(pkg, kind, n, split):
    got, launches = gpu_tree(pkg, family(kind, n), split)
    assert_same_tree(got, ref_tree(family(kind, n), split))
    assert launches == launches_of(n)


@gpu
@pytest.mark.parametrize("split", ["widest", "cyclic"])
@pytest.mark.parametrize("kind", POW20_FAMILIES)
@pytest.mark.parametrize("n", POW20)
def test_tree_at_2pow20(pkg, kind, n, split):
    got, launches = gpu_tree(pkg, family(kind, n), split)
    assert_same_tree(got, ref_tree(family(kind, n), split))
    assert launches == launches_of(n)


def queries_for(pts, nq=4096, seed=0):
    """near-copies, exact copies and far points, around the finite points of a set (scaled by their spread about
    the median, so that sets with outliers at 1e300 or at the largest double still get finite queries)"""
    rng = np.random.default_rng(seed)
    fin = pts[np.isfinite(pts).all(axis=1)]
    med = np.quantile(fin, 0.5, axis=0, method="lower")
    scale = np.maximum(np.quantile(np.abs(fin - med), 0.5, axis=0, method="lower"), 1.0)
    q = fin[rng.integers(0, fin.shape[0], nq)] + rng.normal(0.0, 1e-2, (nq, 3)) * scale
    q[: nq // 4] = fin[rng.integers(0, fin.shape[0], nq // 4)]
    q[nq - nq // 8:] = med + scale * rng.uniform(-20.0, 20.0, (nq // 8, 3))
    assert np.isfinite(q).all()
    return np.ascontiguousarray(q)


def check_answers(pkg, oracle, pts, split):
    """nn_batch and nn_batch_dev of the tree against the fp64 brute-force kernel bit for bit, 64 queries against the
    oracle"""
    import torch
    q = queries_for(pts)
    nq = q.shape[0]
    tree = pkg.KdTree(pts, device=0, split=split)
    try:
        idx, dist, _ = tree.nn_batch(q, want_nearest=False)
        d_pts, d_q = torch.from_numpy(pts.copy()).cuda(), torch.from_numpy(q).cuda()
        d_idx = torch.empty(nq, dtype=torch.int32, device="cuda")
        d_dist = torch.empty(nq, dtype=torch.float64, device="cuda")
        b_idx, b_dist = torch.empty_like(d_idx), torch.empty_like(d_dist)
        stream = torch.cuda.current_stream().cuda_stream
        tree.nn_batch_dev(d_q.data_ptr(), nq, d_idx.data_ptr(), d_dist.data_ptr(), stream=stream)
        pkg.bruteforce_nn_dev(0, d_pts.data_ptr(), pts.shape[0], d_q.data_ptr(), nq, b_idx.data_ptr(),
                              b_dist.data_ptr(), stream=stream)
        torch.cuda.synchronize()
    finally:
        tree.close()
    bi, bd = b_idx.cpu().numpy(), b_dist.cpu().numpy()
    assert np.array_equal(idx, bi) and np.array_equal(dist.view(np.uint64), bd.view(np.uint64))
    assert np.array_equal(d_idx.cpu().numpy(), bi) and np.array_equal(d_dist.cpu().numpy().view(np.uint64),
                                                                      bd.view(np.uint64))
    oi, od = oracle.nn_brute(pts, q[::64])
    assert np.array_equal(oi, bi[::64]) and np.array_equal(od.view(np.uint64), bd[::64].view(np.uint64))


@gpu
@pytest.mark.parametrize("kind", FAMILIES)
def test_tree_1m(pkg, oracle, kind):
    """1 M points, both split rules, from the host and from device memory on a user stream; then the answers"""
    torch = pytest.importorskip("torch")
    pts = family(kind, BIG)
    for split in ("widest", "cyclic"):
        want = _ref(kind, BIG, split)
        got, launches = gpu_tree(pkg, pts, split)
        assert_same_tree(got, want)
        assert launches == launches_of(BIG)
        got, launches = gpu_tree(pkg, pts, split, stream=torch.cuda.Stream())
        assert_same_tree(got, want)
        assert launches == launches_of(BIG)
        check_answers(pkg, oracle, pts, split)


@gpu
def test_tree_10m(pkg, oracle):
    """config 5b's map size, 10 M points of the walls family, widest rule: the exact tree and the answers"""
    n = 10_000_000
    pts = family("walls", n)
    got, launches = gpu_tree(pkg, pts, "widest")
    assert_same_tree(got, _ref("walls", n, "widest"))
    assert launches == launches_of(n)
    check_answers(pkg, oracle, pts, "widest")


@gpu
def test_two_streams_give_identical_exports(pkg):
    """two device-pointer builds of one tie-heavy set in flight at once on two streams: byte-identical exports"""
    torch = pytest.importorskip("torch")
    pts = family("int_walls", BIG)
    d_pts = torch.from_numpy(pts.copy()).cuda()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    trees = []
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
        trees.append(pkg.KdTree(dev_ptr=d_pts.data_ptr(), n=BIG, stream=s.cuda_stream, device=0, split="widest"))
    try:
        a, b = (t.export(with_axes=True) for t in trees)
    finally:
        for t in trees:
            t.close()
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    assert_same_tree(a, _ref("int_walls", BIG, "widest"))


@gpu
@pytest.mark.parametrize("kind", ["duplicates", "int_walls", "all_equal", "special"])
def test_permuted_input(pkg, kind):
    """a permutation of the input is a different set of (point, index) pairs: the tree of the permuted set"""
    pts = family(kind, 100000)
    perm = np.random.default_rng(7).permutation(pts.shape[0])
    got, _ = gpu_tree(pkg, pts[perm], "widest")
    assert_same_tree(got, ref_tree(pts[perm], "widest"))


WORKER_SIZES = [4097, 32769, BIG]


def worker_cases(mid_cap):
    cases = [(k, n, s) for k in FAMILIES for n in WORKER_SIZES for s in ("widest", "cyclic")]
    if mid_cap == 2049:
        cases.append(("walls", 10_000_000, "widest"))
    return cases


@gpu
@pytest.mark.parametrize("mid_cap", [2049, 1 << 30])
def test_every_path_selection(mid_cap):
    """NAV_KD_MIDCAP is read once per process: a worker builds every family with 2049 (every level above the finisher
    on the multi-CTA kernels: 256 segments per launch at 1 M, 4096 at 10 M) or 2^30 (whole large segments through
    k_kd_level_cta and its in-CTA narrowing), and the trees are held to the reference"""
    cases = worker_cases(mid_cap)
    with tempfile.TemporaryDirectory() as tmp:
        src, dst = os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.npz")
        np.savez(src, kind=[c[0] for c in cases], n=[c[1] for c in cases], split=[c[2] for c in cases])
        res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "kd_build_worker.py"), src, dst],
                             env=dict(os.environ, NAV_KD_MIDCAP=str(mid_cap)), capture_output=True, text=True,
                             timeout=1800)
        assert res.returncode == 0, res.stderr[-4000:]
        out = np.load(dst)
        for i, (kind, n, split) in enumerate(cases):
            want = _ref(kind, n, split) if n >= BIG else ref_tree(family(kind, n), split)
            assert_same_tree((out[f"nodes_{i}"], out[f"oidx_{i}"], out[f"axes_{i}"]), want)
            assert int(out[f"launches_{i}"]) == launches_of(n, mid_cap), (kind, n, split)
