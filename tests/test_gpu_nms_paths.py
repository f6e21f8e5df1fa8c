"""GPU parity of the int16 NMS kernel (nms_i16_kernel, csrc/nms.cu) on every code path it selects, against the oracle.

Each image's CTA picks its candidate-vs-kept pair test from the threshold and the image's boxes:
  packed    threshold p/q (q <= 1000), every box valid, 3 * side^2 * max(p, q) < 2^31 - 1, coordinates in [0, 16000):
            16-bit packed intersections, 32-bit products
  small     as packed, but some coordinate is negative or >= 16000 (screen_small_valid)
  rational  threshold p/q, and some box is invalid (x2 < x1 or y2 < y1) or has a side above the 32-bit bound
            (screen_rational, 64-bit products; the exact predicate decides unions <= 0)
  fixed     1e-6 < t < 1 and t is not such a ratio: 64-bit fixed-point screen (screen_i16); the exact predicate decides
            pairs inside its band and unions <= 0
  exact     t <= 1e-6 or t >= 1: the exact predicate only (suppressed_i16)
The intra-tile test follows the same choice, so every path has an in-tile and a cross-tile form (kept box and candidate
in the same or in different tiles of 64 visited candidates).  The kernel also picks a load path (one bulk copy when the
scores are strictly descending and the rows are 16-byte aligned, a plain copy when they are not aligned, a sort
otherwise) and a cluster size from max_boxes, the batch and the SM count.  `kernel_path`, `load_path` and
`cluster_size` restate those choices.  Every case is tagged with the path it is meant to reach, and
test_case_table_reaches_every_path checks, without a GPU, that the tags hold and that the table covers every path in both
forms, every load path and every cluster size of a 148-SM B200.  The GPU tests take their batch sizes from the device's
own SM count.

Oracle domain: oracle.frcnn_oracle.greedy_nms follows the input dtype, so int16 boxes get int16 areas, intersections
and unions, which numpy wraps past 32767, while the kernel computes them as exact integers.  Cases compared with the
int16 oracle therefore stay where nothing wraps (`assert_oracle_domain`).  Cases with large boxes (sides up to 32767,
which reach the side bound of the 32-bit products and the 64-bit products) are compared with greedy_nms on the same
boxes as int64, which is the exact integer arithmetic the kernel implements.
"""
import math
from collections import namedtuple

import numpy as np
import pytest

from helpers import dev, host
from oracle import frcnn_oracle as O

B200_SMS = 148
TILE = 64
LIVE_PATHS = ("packed", "small", "rational", "fixed", "exact")
NEXT_UP, NEXT_DOWN = math.nextafter(0.7, 1.0), math.nextafter(0.7, 0.0)
INVALID_THRESHOLDS = (0.71234, NEXT_UP, 0.3141, 0.7, -0.5, 1e-7, 1.5)
INVALID_PATHS = ("fixed", "fixed", "fixed", "rational", "exact", "exact", "exact")


# ------------------------------------------------------------------------------------------------
# The kernel's choices, restated
# ------------------------------------------------------------------------------------------------
def rational(t):
    """launch_nms_i16's search: (p, q) with p / q == t as doubles and 2 <= q <= 1000, else (0, 0)."""
    if not 1e-6 < t < 1.0:
        return 0, 0
    for q in range(2, 1001):
        p = float(round(t * q))                      # nearbyint: round half to even, as round() does
        if 1.0 <= p < q and p / q == t:
            return int(p), q
    return 0, 0


def fits_32bit(side, p, q):
    """the kernel's per-image test for 32-bit pair products"""
    return 3.0 * side * side * max(p, q) < 2147483647.0


def side_bound(p, q):
    """largest box side that still takes the 32-bit pair test for the threshold p/q"""
    s = int(math.sqrt(2147483647.0 / (3.0 * max(p, q))))
    while fits_32bit(s + 1, p, q):
        s += 1
    while not fits_32bit(s, p, q):
        s -= 1
    return s


def kernel_path(boxes, thresh):
    """the candidate-vs-kept pair test the kernel picks for one image (`boxes` = its first n rows)"""
    if not 1e-6 < thresh < 1.0:
        return "exact"
    p, q = rational(thresh)
    if q == 0:
        return "fixed"
    b = np.asarray(boxes, np.int64).reshape(-1, 4)
    maxdim = maxabs = 0
    if len(b):
        maxdim = int(np.max(np.maximum(np.abs(b[:, 2] - b[:, 0]), np.abs(b[:, 3] - b[:, 1])))) + 1
        maxabs = int(np.abs(b).max())
        if np.any(b[:, 0] < 0) or np.any(b[:, 1] < 0):
            maxabs = 1 << 20
        if np.any(b[:, 2] < b[:, 0]) or np.any(b[:, 3] < b[:, 1]):
            maxdim = 1 << 20
    if not fits_32bit(maxdim, p, q):
        return "rational"
    return "packed" if maxabs < 16000 else "small"


def load_path(probs, n, row):
    """'sort' unless the first n scores are strictly descending; then 'bulk' when the n rows are a multiple of 16 bytes
    and start 16-byte aligned (`row` = image * n_max rows into an aligned allocation), else 'copy'"""
    s = np.asarray(probs[:n], np.float32)
    if n > 1 and not np.all(s[:-1] > s[1:]):
        return "sort"
    return "bulk" if n > 0 and (n * 8) % 16 == 0 and (row * 8) % 16 == 0 else "copy"


def cluster_size(n_max, max_boxes, batch, sm_count):
    """launch_nms_i16's CTAs per image"""
    max_keep = min(max_boxes, n_max)
    cap = 16 if max_keep >= 1024 else 8 if max_keep >= 256 else 1
    cl = 1
    while cl < cap and batch * cl * 2 <= sm_count:
        cl <<= 1
    return cl


def batch_for(cl, n_max, max_boxes, sm_count):
    """a batch size that gets `cl` CTAs per image: the largest one for cl > 1, the smallest one of at least 4 for cl = 1"""
    fits = [b for b in range(1, 2 * sm_count + 2) if cluster_size(n_max, max_boxes, b, sm_count) == cl]
    assert fits, "no batch gives %d CTAs per image at n_max %d, max_boxes %d, %d SMs" % (cl, n_max, max_boxes, sm_count)
    return max(fits) if cl > 1 else min(b for b in fits if b >= 4)


# ------------------------------------------------------------------------------------------------
# Oracle
# ------------------------------------------------------------------------------------------------
def assert_oracle_domain(boxes):
    """every value the int16 oracle forms fits int16: coordinate differences, sides, areas, the intersection extents
    of any pair and area_i + area_j of any pair (a positive intersection is at most the smaller area, and the union is
    then between the larger area and the sum)"""
    b = np.asarray(boxes, np.int64).reshape(-1, 4)
    if len(b) == 0:
        return
    vals = [b[:, 2] - b[:, 0], b[:, 3] - b[:, 1], b[:, 2] - b[:, 0] + 1, b[:, 3] - b[:, 1] + 1]
    area = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
    vals.append(area)
    for lo, hi in ((0, 2), (1, 3)):
        vals.append(np.array([b[:, hi].max() - b[:, lo].min() + 1, b[:, hi].min() - b[:, lo].max()]))
    if len(b) > 1:
        a = np.sort(area)
        vals.append(np.array([a[0] + a[1], a[-1] + a[-2]]))
    v = np.concatenate(vals)
    assert v.min() >= -32768 and v.max() <= 32767, "case leaves the int16 oracle's domain"


def oracle_pick(boxes, probs, thresh, max_boxes, wide):
    if not wide:
        assert_oracle_domain(boxes)
    return O.greedy_nms(np.asarray(boxes, np.int64) if wide else boxes, probs, thresh, max_boxes)


def pair_kinds(boxes, probs, pick):
    """{'in', 'cross'}: whether the sweep tests a kept box against a later candidate of the same / of another tile for
    a pair whose answer is not the trivial disjoint one (intersection > 0 or union <= 0)"""
    n = len(boxes)
    if len(pick) == 0:
        return set()
    order = np.argsort(probs, kind="stable")[::-1]
    rank = np.empty(n, np.int64)
    rank[order] = np.arange(n)
    b = np.asarray(boxes, np.int64)[order]
    area = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
    kept = rank[np.asarray(pick)]
    end = min(n, (int(kept.max()) // TILE + 1) * TILE)         # the sweep stops after the tile of the last keep
    kinds = set()
    for r in kept:
        j = np.arange(r + 1, end)
        iw = np.maximum(0, np.minimum(b[r, 2], b[j, 2]) - np.maximum(b[r, 0], b[j, 0]) + 1)
        ih = np.maximum(0, np.minimum(b[r, 3], b[j, 3]) - np.maximum(b[r, 1], b[j, 1]) + 1)
        inter = iw * ih
        live = (inter > 0) | (area[r] + area[j] - inter <= 0)
        same = j // TILE == r // TILE
        if np.any(live & same):
            kinds.add("in")
        if np.any(live & ~same):
            kinds.add("cross")
    return kinds


# ------------------------------------------------------------------------------------------------
# Inputs
# ------------------------------------------------------------------------------------------------
def _scores(rng, n, order):
    """float32 scores: 'desc' strictly descending, 'perm' distinct in random order, 'ties' few distinct values"""
    if order == "desc":
        return (np.arange(n, 0, -1) / max(n, 1)).astype(np.float32)
    if order == "perm":
        return ((rng.permutation(n) + 0.5) / max(n, 1)).astype(np.float32)
    return (rng.integers(0, 5, n) / 5).astype(np.float32)


def _valid(rng, n, dx=0, dy=0, max_side=40):
    """valid boxes at a density that gives both suppressions and survivors"""
    span = max(8, int(12 * math.sqrt(n)))
    x1, y1 = dx + rng.integers(0, span, n), dy + rng.integers(0, span, n)
    w, h = rng.integers(1, max_side + 1, n), rng.integers(1, max_side + 1, n)
    return np.stack([x1, y1, x1 + w - 1, y1 + h - 1], 1)


def _with_invalid(rng, b, frac=0.15):
    """turn a fraction of the boxes (always the first) into invalid ones: width or height in [-10, 0]"""
    b = b.copy()
    bad = rng.random(len(b)) < frac
    bad[0] = True
    for k in np.where(bad)[0]:
        c = int(rng.integers(0, 2))                            # 0: x, 1: y
        b[k, c + 2] = b[k, c] - int(rng.integers(1, 12))      # side = x2 - x1 + 1 in [-10, 0]
    return b


def _small_invalid(rng, n):
    """boxes in +-40 with sides -11..31: zero and negative areas, zero and negative unions everywhere"""
    x1, y1 = rng.integers(-40, 41, n), rng.integers(-40, 41, n)
    w, h = rng.integers(-11, 32, n), rng.integers(-11, 32, n)
    return np.stack([x1, y1, x1 + w - 1, y1 + h - 1], 1)


def _disjoint(k, start=0, x0=200):
    """k pairwise disjoint 2 x 2 boxes in a row"""
    return [[x0 + 3 * i, 0, x0 + 3 * i + 1, 1] for i in range(start, start + k)]


SWEEP_BOXES = {
    "packed": lambda rng, n: _valid(rng, n),
    "small": lambda rng, n: _valid(rng, n, dx=16000),
    "rational": lambda rng, n: _with_invalid(rng, _valid(rng, n)),
    "fixed": lambda rng, n: _valid(rng, n, dx=-20, dy=-7),
    "exact": lambda rng, n: _valid(rng, n),
}
SWEEP_THRESH = {"packed": 0.7, "small": 0.7, "rational": 0.7, "fixed": 0.65432, "exact": 1e-7}


def _case_sweep(path, n, order):
    def make():
        rng = np.random.default_rng([LIVE_PATHS.index(path), n, order == "desc"])
        return SWEEP_BOXES[path](rng, n).astype(np.int16), _scores(rng, n, order)
    return make


def _case_exact_ratio(cross, dx=0, invalid=False):
    """pairs with inter/union = 7/10 exactly and pairs just above it, once all in one tile, once spread over three"""
    kept = [[0, 0, 9, 9], [20, 0, 39, 9]]                      # areas 100 and 200
    at = [[0, 3, 9, 9], [20, 0, 33, 9]]                        # 70 / 100 and 140 / 200 against the kept boxes
    over = [[0, 2, 9, 9], [20, 0, 34, 9]]                      # 80 / 100 and 150 / 200
    if cross:
        rows = kept + _disjoint(62) + at + _disjoint(62, 62) + over
    else:
        rows = kept + at + over + _disjoint(20)
    if invalid:
        rows = rows + [[1000, 1000, 999, 1000]]                # zero width: takes the image off the 32-bit paths

    def make():
        b = np.array(rows, np.int64)
        b[:, [0, 2]] += dx
        return b.astype(np.int16), _scores(None, len(b), "desc")
    return make


def _case_corner(maxc=None, neg=False):
    """valid boxes whose largest coordinate is `maxc`, or with one coordinate at -1"""
    def make():
        rng = np.random.default_rng([7, maxc or 0, neg])
        b = _valid(rng, 150, dx=(maxc - 200) if maxc else 0, max_side=60)
        if maxc:
            b[:, 2] = np.minimum(b[:, 2], maxc)
            b[0, 2] = maxc
        if neg:
            b[0, 0] = -1
        return b.astype(np.int16), _scores(rng, 150, "perm")
    return make


def _case_side(side):
    """thin boxes (height 1, so the areas stay in the oracle domain), the longest of side `side`"""
    def make():
        rng = np.random.default_rng([11, side])
        n = 150
        x1, y = rng.integers(0, 6000, n), rng.integers(0, 4, n)
        length = rng.integers(1000, side + 1, n)
        length[5] = side
        b = np.stack([x1, y, x1 + length - 1, y], 1)
        return b.astype(np.int16), _scores(rng, n, "perm")
    return make


def _case_wide(invalid):
    """sides up to 32767: past the 32-bit bound, 64-bit products, unions up to 2^31 (int64 oracle)"""
    def make():
        rng = np.random.default_rng([13, invalid])
        n = 200
        x1, y1 = rng.integers(-16000, 1, n), rng.integers(-16000, 1, n)
        w, h = rng.integers(1, 32768, n), rng.integers(1, 32768, n)
        b = np.stack([x1, y1, x1 + w - 1, y1 + h - 1], 1)
        if invalid:                                            # a third of them with a side in [-16000, 0]
            bad = np.where(rng.random(n) < 0.33)[0]
            c = rng.integers(0, 2, len(bad))
            b[bad, c] = rng.integers(0, 16001, len(bad))
            b[bad, c + 2] = b[bad, c] + rng.integers(-16000, 1, len(bad)) - 1
        return b.astype(np.int16), _scores(rng, n, "perm")
    return make


def _case_invalid():
    """crafted pairs across tiles -- zero areas (x2 = x1 - 1), negative areas, a box with both sides negative, zero
    unions (0 / 0 is NaN, which suppresses) and negative unions (0 / -5 = -0.0, which survives t >= 0) -- around 190
    random boxes with sides -11..31"""
    heads = [[0, 0, -1, 5], [10, 10, 7, 14], [60, 60, 57, 58]]          # areas 0, -10 and (-2) * (-1) = 2
    tails = [[50, 50, 49, 50], [100, 100, 101, 104], [100, 100, 100, 104], [60, 60, 60, 60]]   # 0, 10, 5, 1

    def make():
        rng = np.random.default_rng(17)
        b = np.concatenate([np.array(heads), _small_invalid(rng, 190), np.array(tails)])
        return b.astype(np.int16), _scores(rng, len(b), "desc")
    return make


def regression_negative_union():
    """box A (width -2, area -10) is kept first; B (area 5) is in the next tile and their union is -5: 0 / -5 = -0.0
    is <= t, so B survives.  The fixed-point screen used to wrap the negative union and suppress B."""
    a = [10, 10, 7, 14]
    fill = [[200 + 3 * i, 0, 201 + 3 * i, 1] for i in range(63)]
    b = [100, 100, 100, 104]
    boxes = np.array([a] + fill + [b], np.int16)
    probs = (np.arange(65, 0, -1) / 65).astype(np.float32)
    return boxes, probs


Case = namedtuple("Case", "id make thresh max_boxes path wide")
P, Q = rational(0.7)
SIDE = side_bound(P, Q)

CASES = (
    [Case("sweep-%s-n%d-%s" % (p, n, o), _case_sweep(p, n, o), SWEEP_THRESH[p], 2000, p, False)
     for p in LIVE_PATHS for n in (1, 63, 64, 65, 129, 3000) for o in ("perm", "desc")]
    + [Case("ratio-packed-" + f, _case_exact_ratio(f == "cross"), 0.7, 300, "packed", False) for f in ("in", "cross")]
    + [Case("ratio-small-" + f, _case_exact_ratio(f == "cross", dx=16000), 0.7, 300, "small", False) for f in ("in", "cross")]
    + [Case("ratio-rational-" + f, _case_exact_ratio(f == "cross", invalid=True), 0.7, 300, "rational", False)
       for f in ("in", "cross")]
    + [Case("ratio-fixed-%s-%s" % (d, f), _case_exact_ratio(f == "cross"), t, 300, "fixed", False)
       for d, t in (("up", NEXT_UP), ("down", NEXT_DOWN)) for f in ("in", "cross")]
    + [Case("corner-15999", _case_corner(maxc=15999), 0.7, 300, "packed", False),
       Case("corner-16000", _case_corner(maxc=16000), 0.7, 300, "small", False),
       Case("corner-minus1", _case_corner(neg=True), 0.7, 300, "small", False),
       Case("side-%d" % SIDE, _case_side(SIDE), 0.7, 300, "packed", False),
       Case("side-%d" % (SIDE + 1), _case_side(SIDE + 1), 0.7, 300, "rational", False),
       Case("wide-0.7", _case_wide(False), 0.7, 300, "rational", True),
       Case("wide-0.71234", _case_wide(False), 0.71234, 300, "fixed", True),
       Case("wide-invalid-0.7", _case_wide(True), 0.7, 300, "rational", True),
       Case("wide-invalid-0.71234", _case_wide(True), 0.71234, 300, "fixed", True),
       Case("wide-invalid-1.5", _case_wide(True), 1.5, 300, "exact", True)]
    + [Case("invalid-%r" % t, _case_invalid(), t, 300, path, False) for t, path in zip(INVALID_THRESHOLDS, INVALID_PATHS)]
)

# one launch per cluster size: (id, CTAs per image, n_max, max_boxes, threshold, box makers of the distinct images)
ClusterCase = namedtuple("ClusterCase", "id cl n_max max_boxes thresh kinds")
CLUSTER_CASES = [
    ClusterCase("cl1-200", 1, 700, 200, 0.7, ("packed",)),
    ClusterCase("cl1-300", 1, 1000, 300, 0.7, ("packed", "small")),
    ClusterCase("cl2-300", 2, 1000, 300, 0.71234, ("invalid", "fixed")),
    ClusterCase("cl4-300-mixed", 4, 1000, 300, 0.7, ("packed", "small", "rational")),
    ClusterCase("cl8-300", 8, 1000, 300, 1e-7, ("exact",)),
    ClusterCase("cl8-2000", 8, 2500, 2000, 0.7, ("rational", "packed")),
    ClusterCase("cl16-2000", 16, 3000, 2000, 0.65432, ("fixed", "invalid")),
]
IMAGE_BOXES = dict(SWEEP_BOXES, invalid=_small_invalid)


def cluster_images(case):
    """four distinct images (box kind, per-image n, score order), one of them empty; image i of a batch is image i % 4"""
    out = []
    for d, (cut, order) in enumerate(((0, "perm"), (37, "desc"), (100, "perm"), (case.n_max, "desc"))):
        rng = np.random.default_rng([19, case.cl, case.max_boxes, d])
        kind = case.kinds[d % len(case.kinds)]
        boxes = IMAGE_BOXES[kind](rng, case.n_max).astype(np.int16)
        out.append((boxes, _scores(rng, case.n_max, order), case.n_max - cut))
    return out


def load_images():
    """odd n_max with strictly descending scores: image 0 (n even, aligned) takes the bulk copy, image 1 (n even, its
    rows 8 bytes off alignment) and image 2 (n odd) the plain copy, image 3 (ties) the sort"""
    n_max, rng = 301, np.random.default_rng(23)
    imgs = []
    for n, order in ((300, "desc"), (300, "desc"), (301, "desc"), (301, "ties")):
        probs = np.zeros(n_max, np.float32)
        probs[:n] = _scores(rng, n, order)
        imgs.append((_valid(rng, n_max).astype(np.int16), probs, n))
    return n_max, imgs


# ------------------------------------------------------------------------------------------------
# Coverage of the table (no GPU)
# ------------------------------------------------------------------------------------------------
def test_case_table_reaches_every_path():
    reached, loads = set(), set()
    for c in CASES:
        boxes, probs = c.make()
        assert kernel_path(boxes, c.thresh) == c.path, c.id
        pick = oracle_pick(boxes, probs, c.thresh, c.max_boxes, c.wide)
        reached |= {(c.path, k) for k in pair_kinds(boxes, probs, pick)}
        loads.add(load_path(probs, len(probs), 0))
    assert reached == {(p, k) for p in LIVE_PATHS for k in ("in", "cross")}, sorted(reached)
    n_max, imgs = load_images()
    assert [load_path(p, n, i * n_max) for i, (_, p, n) in enumerate(imgs)] == ["bulk", "copy", "copy", "sort"]
    assert loads == {"bulk", "copy", "sort"}

    sizes, mixed = set(), False
    for c in CLUSTER_CASES:
        batch = batch_for(c.cl, c.n_max, c.max_boxes, B200_SMS)
        assert cluster_size(c.n_max, c.max_boxes, batch, B200_SMS) == c.cl, c.id
        sizes.add(c.cl)
        paths = {kernel_path(b[:n], c.thresh) for b, _, n in cluster_images(c) if n > 0}
        mixed |= len(paths) > 1
    assert sizes == {1, 2, 4, 8, 16} and mixed
    # the exact-ratio pairs sit on the threshold: they decide between the two sides of 0.7
    boxes, probs = _case_exact_ratio(True)()
    assert len(O.greedy_nms(boxes, probs, 0.7)) == len(O.greedy_nms(boxes, probs, NEXT_DOWN)) + 2


def test_helpers_restate_the_launcher():
    assert rational(0.7) == (7, 10) and rational(0.75) == (3, 4) and rational(0.999) == (999, 1000)
    assert rational(0.71234) == (0, 0) and rational(NEXT_UP) == (0, 0) and rational(0.5555) == (0, 0)
    assert rational(1e-7) == (0, 0) and rational(1.0) == (0, 0)
    assert fits_32bit(SIDE, 7, 10) and not fits_32bit(SIDE + 1, 7, 10)
    assert [cluster_size(3000, 2000, b, 148) for b in (1, 9, 10, 18, 19, 37, 38, 74, 75)] == [16, 16, 8, 8, 4, 4, 2, 2, 1]
    assert [cluster_size(1000, 300, b, 148) for b in (1, 18, 19, 37, 38, 74, 75)] == [8, 8, 4, 4, 2, 2, 1]
    assert cluster_size(700, 200, 1, 148) == 1
    assert kernel_path(np.zeros((0, 4)), 0.7) == "packed"


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ops():
    from faster_rcnn_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def assert_keep(out, i, boxes, probs, pick, what):
    """image i of an nms_i16 result equals the oracle's pick: index, boxes, score bits, then -1 / zero padding"""
    ki, kc, kb, ks = out
    m = len(pick)
    assert kc[i] == m, "%s: kept %d, oracle %d" % (what, kc[i], m)
    assert np.array_equal(ki[i, :m], pick), "%s: first difference at keep %d" % (
        what, int(np.argmax(ki[i, :m] != pick)) if m else -1)
    assert np.all(ki[i, m:] == -1), what
    assert np.array_equal(kb[i, :m], boxes[pick]) and not np.any(kb[i, m:]), what
    assert np.array_equal(ks[i, :m].view(np.int32), probs[pick].view(np.int32)) and not np.any(ks[i, m:].view(np.int32)), what


def run_nms(ops, boxes, probs, n, thresh, max_boxes):
    """boxes (B, n_max, 4) i16, probs (B, n_max) f32, n (B,) i32 or None -> host copies of the four outputs"""
    out = ops.nms_i16(dev(boxes), dev(probs), None if n is None else dev(np.asarray(n, np.int32)), thresh, max_boxes)
    return tuple(host(t) for t in out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_nms_path_vs_oracle(ops, case):
    boxes, probs = case.make()
    pick = oracle_pick(boxes, probs, case.thresh, case.max_boxes, case.wide)
    out = run_nms(ops, boxes[None], probs[None], None, case.thresh, case.max_boxes)
    assert_keep(out, 0, boxes, probs, pick, case.id)


@pytest.mark.gpu
@pytest.mark.parametrize("thresh", [0.71234, NEXT_UP, 0.7], ids=["0.71234", "nextafter-0.7-up", "0.7"])
def test_nms_negative_union_across_tiles_survives(ops, thresh):
    boxes, probs = regression_negative_union()
    pick = oracle_pick(boxes, probs, thresh, 300, False)
    assert len(pick) == 65
    assert_keep(run_nms(ops, boxes[None], probs[None], None, thresh, 300), 0, boxes, probs, pick, "65 boxes")


@pytest.mark.gpu
@pytest.mark.parametrize("thresh", [0.7, 0.71234])
def test_nms_room_cut_in_second_tile(ops, thresh):
    """tile 0 keeps k = 5 boxes (59 duplicates of its first box go), tile 1 holds 64 disjoint boxes; max_boxes = k + 1
    ... k + 64 cuts tile 1 at every position, in both 32-bit halves of its keep mask"""
    k = 5
    rows = _disjoint(1) + _disjoint(1) * 59 + _disjoint(k - 1, 1) + _disjoint(64, k)
    boxes, probs = np.array(rows, np.int16), _scores(None, len(rows), "desc")
    assert kernel_path(boxes, thresh) == ("packed" if thresh == 0.7 else "fixed")
    for max_boxes in range(k + 1, k + 65):
        pick = oracle_pick(boxes, probs, thresh, max_boxes, False)
        assert len(pick) == max_boxes
        out = run_nms(ops, boxes[None], probs[None], None, thresh, max_boxes)
        assert_keep(out, 0, boxes, probs, pick, "max_boxes %d" % max_boxes)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CLUSTER_CASES, ids=[c.id for c in CLUSTER_CASES])
def test_nms_cluster_sizes(ops, sm_count, case):
    batch = batch_for(case.cl, case.n_max, case.max_boxes, sm_count)
    imgs = cluster_images(case)
    picks = [oracle_pick(b[:n], p[:n], case.thresh, case.max_boxes, False) for b, p, n in imgs]
    idx = [i % len(imgs) for i in range(batch)]
    out = run_nms(ops, np.stack([imgs[d][0] for d in idx]), np.stack([imgs[d][1] for d in idx]),
                  [imgs[d][2] for d in idx], case.thresh, case.max_boxes)
    for i, d in enumerate(idx):
        b, p, n = imgs[d]
        assert_keep(out, i, b[:n], p[:n], picks[d], "%s image %d of %d" % (case.id, i, batch))


@pytest.mark.gpu
def test_nms_load_paths_in_one_batch(ops):
    n_max, imgs = load_images()
    out = run_nms(ops, np.stack([b for b, _, _ in imgs]), np.stack([p for _, p, _ in imgs]), [n for _, _, n in imgs], 0.7, 300)
    for i, (b, p, n) in enumerate(imgs):
        assert_keep(out, i, b[:n], p[:n], oracle_pick(b[:n], p[:n], 0.7, 300, False), "image %d" % i)


@pytest.mark.gpu
def test_det_util_nms_with_invalid_rows():
    from faster_rcnn_b200 import det_util
    boxes, probs = _case_invalid()()
    probs = probs[np.random.default_rng(29).permutation(len(probs))]
    got_b, got_p = det_util.nms(boxes, probs, 0.71234, 300)
    want_b, want_p = O.nms(boxes, probs, 0.71234, 300)
    assert got_b.dtype == np.int16 and np.array_equal(got_b, want_b) and np.array_equal(got_p, want_p)
