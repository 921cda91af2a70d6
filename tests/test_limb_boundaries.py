"""Limb scoring (K2, `limb_score_kernel`, csrc/og_limbs.cu) and the row preparation fused behind it
(`prepare_limb_rows`, csrc/og_prep.cuh) at the values where they decide.

Every scene is built at test time from isolated single-pixel peaks (top-K order = peak value order),
one construction per (image, limb type), so each from-candidate's nearest to-candidate is the
intended one.  Families:

  A  near ties: to-candidates whose float32 squared distances differ by 1 or 2 ulps yet round to
     one root (the reference's Tensor.min takes the FIRST index of the smallest rounded distance,
     even when its squared distance is the larger one: the "order trap"), 2-ulp pairs in the even
     binade [256, 512) that only a 2^-20 re-evaluation window catches, 1-ulp controls whose roots
     differ (the later candidate wins), exact 2- and 3-way ties (the first wins), and a pair whose
     decision changes when d^2 is evaluated in another order (sq2's operands swapped, sq4
     contracted into fused multiply-adds); 2-D offsets
     (sqrt(fma(dy, dy, dx*dx))) and 4-D cat_flip_offs (left-to-right sum of squares).  Every pair
     is certified with exact rational arithmetic (`fractions`).
  B  threshold shift: from- and to-scores at thre_hmp and one float32 step below.
  C  len = max(norm, min_len) with the norm at min_len (3-4-5) and min_len one step either side.
  D  gate: min_dist at dist_max and one step either side; with use_scale scale_t = min_dist,
     scale_t = dist_max, scale_t one step above min_dist and a NaN scale; endpoints in row / column
     0 against 1; jitter moving x1 or y1 to exactly 0 and from 0 to above it.
  E  jitter refinement bounds: guided x or y in (-1, 0), at -1 and just below W or H on maps with
     H < W and H > W, covering the four regions (inside / outside the reference's bounds check) x
     (inside / outside the [x, y]-as-[row, col] indexed plane).
  F  K = 31 ... 128 around the CTA sizes 32 / 64 / 128, full and partly empty candidate lists.
  G  NaN limb scores (min_len = 0, from- and to-candidate on one pixel, zero offset).

Three routes: K2 alone (`limb_score` on the oracle's own top-K lists), K1 -> K2 + prep -> K3
(`decode_maps` + `last_intermediates`), and prep + K3 on the oracle's limb table (`group`)."""
import functools
from fractions import Fraction as Fr

import numpy as np
import pytest

import golden_io as gio
from oracle import c_oracle as co
from oracle import ref_oracle as ro

F32 = np.float32
RTOL = 1e-5
THRE = F32(0.25)
PERSON_THRE = 0.05
C = 4
SK = [(0, 1), (2, 3)]                 # two limb types on disjoint channels: two constructions per image
L = len(SK)
WINDOW = 1 + 2.0 ** -20               # K2's pass-2 window factor (1.00000095367431640625f)


def _up(v):
    return np.nextafter(F32(v), F32(np.inf))


def _down(v):
    return np.nextafter(F32(v), F32(-np.inf))


# =========================================================================== exact arithmetic
def _round32(q):
    """The float32 nearest to the rational q (ties to even)."""
    c = F32(float(q))
    best = None
    for v in (_down(c), c, _up(c)):
        key = (abs(Fr(float(v)) - q), int(np.array(v).view(np.uint32)) & 1)
        if best is None or key < best[0]:
            best = (key, v)
    return best[1]


def exact_sq2(dx, dy):
    """fma(dy, dy, dx * dx) in float32, each rounding done exactly."""
    xx = _round32(Fr(float(dx)) ** 2)
    return _round32(Fr(float(dy)) ** 2 + Fr(float(xx)))


def exact_sq4(a, b, c, d):
    """((a*a + b*b) + c*c) + d*d in float32, every product and sum rounded."""
    sq = [_round32(Fr(float(v)) ** 2) for v in (a, b, c, d)]
    acc = _round32(Fr(float(sq[0])) + Fr(float(sq[1])))
    acc = _round32(Fr(float(acc)) + Fr(float(sq[2])))
    return _round32(Fr(float(acc)) + Fr(float(sq[3])))


def exact_root(v):
    """The correctly rounded float32 square root of the float32 v, certified: v lies between the
    squares of the midpoints to its neighbours."""
    q = Fr(float(v))
    r0 = F32(np.sqrt(np.float64(v)))
    for r in (_down(r0), r0, _up(r0)):
        lo = (Fr(float(_down(r))) + Fr(float(r))) / 2
        hi = (Fr(float(r)) + Fr(float(_up(r)))) / 2
        if lo * lo <= q <= hi * hi:
            return r
    raise AssertionError(v)


def _ulps(a, b):
    return abs(int(np.array(F32(a)).view(np.int32)) - int(np.array(F32(b)).view(np.int32)))


# =========================================================================== scenes
def build_scene(sites, n_img, h, w, nd=2, topk=8):
    """Heat maps (n, C, h, w) and offsets (n, nd * L, h, w) of `sites`, site i on image i // L,
    limb type i % L.  A site is a dict: `frm` (x, y), `off` (nd components), `to` [(x, y), ...] in
    top-K order, optional `fs` / `ts` peak values (default 0.9, then 0.8, 0.75, ...)."""
    assert len(sites) <= n_img * L
    heat = np.zeros((n_img, C, h, w), F32)
    offs = np.zeros((n_img, nd * L, h, w), F32)
    for i, s in enumerate(sites):
        n, l = divmod(i, L)
        jf, jt = SK[l]
        x1, y1 = s['frm']
        heat[n, jf, y1, x1] = s.get('fs', F32(0.9))
        for c, v in enumerate(s['off']):
            offs[n, nd * l + c, y1, x1] = v
        ts = s.get('ts') or [F32(0.8 - 0.05 * r) for r in range(len(s['to']))]
        for (x, y), v in zip(s['to'], ts):
            assert heat[n, jt, y, x] == 0, 'two to-candidates on one pixel'
            heat[n, jt, y, x] = v
    for n in range(n_img):                      # peaks are isolated: no two within one pixel
        for c in range(C):
            ys, xs = np.nonzero(heat[n, c])
            for a in range(len(ys)):
                for b in range(a + 1, len(ys)):
                    assert max(abs(ys[a] - ys[b]), abs(xs[a] - xs[b])) >= 2, (n, c)
            assert len(ys) <= topk
    return heat, offs


def site_of(i):
    return divmod(i, L)


# =========================================================================== A: near ties
A_BASE = (32, 32)                       # guided point = A_BASE + fraction; 64 x 64 maps
A_FROM = (30, 29)
A_HW = 64


def _a_vectors(lo, hi):
    """Integer vectors (i, j), |i|, |j| <= 31, grouped by i^2 + j^2 in [lo, hi)."""
    groups = {}
    for i in range(-31, 32):
        for j in range(-31, 32):
            if lo <= i * i + j * j < hi:
                groups.setdefault(i * i + j * j, []).append((i, j))
    return [g for _, g in sorted(groups.items()) if len(g) > 1]


def _a_diffs(v, f):
    """Components of guided - to for integer vector v and fraction f (2 or 4 values)."""
    if len(f) == 2:
        return (F32(v[0] + f[0]), F32(v[1] + f[1]))
    return (F32(v[0] + f[0]), F32(v[1] + f[1]), F32(v[0] + f[2]), F32(v[1] + f[3]))


def _a_sq(d):
    return exact_sq2(*d) if len(d) == 2 else exact_sq4(*d)


def _approx_sq(d, alt=False):
    """Float squared distance (`alt`: the other evaluation order, see _alt_sq) for the search's
    pre-filter only: not certified."""
    d = [np.float64(F32(v)) for v in d]
    if len(d) == 2:
        a, b = (d[1], d[0]) if alt else (d[0], d[1])
        return F32(b * b + np.float64(F32(a * a)))
    if alt:
        acc = F32(d[1] * d[1] + np.float64(F32(d[0] * d[0])))
        acc = F32(d[2] * d[2] + np.float64(acc))
        return F32(d[3] * d[3] + np.float64(acc))
    acc = F32(np.float64(F32(d[0] * d[0])) + np.float64(F32(d[1] * d[1])))
    acc = F32(np.float64(acc) + np.float64(F32(d[2] * d[2])))
    return F32(np.float64(acc) + np.float64(F32(d[3] * d[3])))


def _alt_sq(d):
    """The squared distance evaluated the other way: sq2's operands swapped (fma(dx, dx, dy*dy)),
    sq4 contracted into fused multiply-adds."""
    return _sq2_swapped(*d) if len(d) == 2 else _sq4_fma(*d)


def _decision(sq):
    """(index, rounded distance) the reference takes from squared distances `sq`."""
    roots = [F32(np.sqrt(v)) for v in sq]
    m = roots.index(min(roots))
    return m, float(roots[m])


def _pair_kind(a, b):
    """(ulps apart, roots equal) of two exact squared distances."""
    return _ulps(a, b), exact_root(a) == exact_root(b)


@functools.lru_cache(maxsize=None)
def near_tie_sites(nd):
    """Certified near-tie constructions: list of (tag, fraction, [vectors in top-K order],
    expected winner).  Guided - to of vector v is v + fraction."""
    rng = np.random.RandomState(20 + nd)
    s = 1 if nd == 2 else 2                     # 4-D: d^2 is twice the vector's i^2 + j^2
    groups = _a_vectors(256 // s, 1024 // s)
    narrow = _a_vectors(256 // s, 384 // s)     # where the 2-ulp trap tells the windows apart
    want = ['trap1', 'plain1', 'trap2_even', 'plain2', 'control', 'formula']
    found = {}
    if nd == 2:                 # the pair the near-tie analysis verified by hand, translated
        found['issue'] = ((2.0 ** -13, 2.0 ** -15), [(18, 11), (21, -2)], 0)
    step = 2.0 ** -15
    for _ in range(200000):
        if all(k in found for k in want):
            break
        pool = narrow if ('trap2_even' not in found and _ % 2) else groups
        g = pool[rng.randint(len(pool))]
        a, b = rng.choice(len(g), 2, replace=False)
        p, q = g[a], g[b]
        if max(abs(p[0] - q[0]), abs(p[1] - q[1])) < 2:         # peaks must stay isolated
            continue
        if _ % 3 == 2:      # fractions with more bits: the evaluation order of d^2 then matters
            f = tuple(float(rng.randint(-2 ** 13, 2 ** 13) * 2.0 ** -14) for _ in range(nd))
        else:
            f = tuple(float(rng.randint(-8, 9) * step) for _ in range(nd))
        # float pre-filter, then exact certification
        dp, dq = _a_diffs(p, f), _a_diffs(q, f)
        ap, aq = _approx_sq(dp), _approx_sq(dq)
        if 'formula' not in found and _decision([ap, aq]) != _decision([_approx_sq(dp, True), _approx_sq(dq, True)]):
            ref = [_a_sq(dp), _a_sq(dq)]
            if _decision(ref) != _decision([_alt_sq(dp), _alt_sq(dq)]):
                found['formula'] = (f, [p, q], reference_pick(ref))
        if abs(int(ap.view(np.int32)) - int(aq.view(np.int32))) not in (1, 2, 3):
            continue
        sp, sq = _a_sq(dp), _a_sq(dq)
        if sp == sq:
            continue
        gap, same = _pair_kind(sp, sq)
        lo, hi = (p, q) if sp < sq else (q, p)
        small = min(sp, sq)
        if same and gap == 1:
            found.setdefault('trap1', (f, [hi, lo], 0))
            found.setdefault('plain1', (f, [lo, hi], 0))
        elif same and gap == 2:
            if 256 <= small < 384:      # there 1 + 2^-23 widens the window by one ulp only
                found.setdefault('trap2_even', (f, [hi, lo], 0))
            found.setdefault('plain2', (f, [lo, hi], 0))
        elif not same and gap == 1:
            found.setdefault('control', (f, [hi, lo], 1))
    assert all(k in found for k in want), sorted(found)
    z = (0.0,) * nd
    ties = [('tie2', z if nd == 4 else (2.0 ** -14, 2.0 ** -14), [(12, 16), (16, 12)], 0),
            ('tie3', z, [(20, 0), (12, 16), (16, 12)], 0)]
    out = [(k,) + found[k] for k in (['issue'] if nd == 2 else []) + want]
    return out + ties


def near_tie_scene(nd):
    """Sites of family A: each construction once as listed and once behind a far decoy that
    takes the first top-K slot (so the pair sits at other indices)."""
    sites, meta = [], []
    bx, by = A_BASE
    for tag, f, vecs, win in near_tie_sites(nd):
        for decoy in (False, True):
            off = [F32(bx - A_FROM[0] + f[0]), F32(by - A_FROM[1] + f[1])]
            if nd == 4:
                off += [F32(bx - A_FROM[0] + f[2]), F32(by - A_FROM[1] + f[3])]
            to = [(bx - v[0], by - v[1]) for v in vecs]
            if decoy:
                to = [(1, 62) if to[0] != (1, 62) else (62, 1)] + to
            sites.append(dict(frm=A_FROM, off=off, to=to))
            meta.append((tag, f, vecs, win + (1 if decoy else 0)))
    n = (len(sites) + L - 1) // L
    heat, offs = build_scene(sites, n, A_HW, A_HW, nd)
    return heat, offs, meta


def two_pass_model(sq, k_live, factor, first_break=True):
    """Pass 1 (minimum squared distance) and pass 2 (first index whose rounded root equals the
    minimum's, searched within best2 * factor) over exact float32 squared distances `sq`."""
    best2 = sq[0]
    for d in sq[1:k_live]:
        if d < best2:
            best2 = d
    best = exact_root(best2)
    window = _round32(Fr(float(best2)) * Fr(factor)) if factor != 1 else best2
    pick = 0
    for m in range(k_live):
        if sq[m] <= window and exact_root(sq[m]) == best:
            pick = m
            if first_break:
                break
    return pick


def _sq2_swapped(dx, dy):
    return exact_sq2(dy, dx)


def _sq4_fma(a, b, c, d):
    acc = _round32(Fr(float(b)) ** 2 + Fr(float(_round32(Fr(float(a)) ** 2))))
    acc = _round32(Fr(float(c)) ** 2 + Fr(float(acc)))
    return _round32(Fr(float(d)) ** 2 + Fr(float(acc)))


def reference_pick(sq):
    """Tensor.min over the rounded roots: the first index of the smallest."""
    roots = [exact_root(v) for v in sq]
    return roots.index(min(roots))


# =========================================================================== CPU tests
@pytest.mark.parametrize('nd', [2, 4])
def test_near_tie_constructions_reach_their_regime(nd):
    """No GPU.  Family A as certified with fractions: the near-tie pairs have distinct squared
    distances and one root, an order trap (the first candidate has the larger squared distance) and
    a 2-ulp pair with d^2 in [256, 512) are present, the controls' roots differ, the ties are exact;
    the oracle picks the expected candidate in every site."""
    tags = {}
    for tag, f, vecs, win in near_tie_sites(nd):
        sq = [_a_sq(_a_diffs(v, f)) for v in vecs]
        tags[tag] = sq
        assert reference_pick(sq) == win, tag
        if tag.startswith('tie'):
            assert len(set(float(v) for v in sq)) == 1
            continue
        if tag == 'formula':        # d^2 evaluated the other way picks another candidate or distance
            assert _decision(sq) != _decision([_alt_sq(_a_diffs(v, f)) for v in vecs])
            continue
        gap, same = _pair_kind(sq[0], sq[1])
        assert gap in (1, 2) and same == (tag != 'control'), (tag, gap, same)
        if tag.startswith('trap') or tag in ('issue', 'control'):
            assert sq[0] > sq[1], tag
        if tag == 'trap2_even':
            assert gap == 2 and 256 <= min(sq) < 512
    assert len(tags['tie3']) == 3
    if nd == 2:       # the hand-verified pair: d^2 = 445.0050048828125 / 445.00506591796875, root 21.095142
        assert float(tags['issue'][0]) == 445.00506591796875 and float(tags['issue'][1]) == 445.0050048828125
        assert abs(float(exact_root(tags['issue'][0])) - 21.095142) < 1e-5
    heat, offs, meta = near_tie_scene(nd)
    lim = ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1, vector_nd=nd)
    ds, di, _, _ = ro.joint_dets(heat, 8)
    for i, (tag, f, vecs, win) in enumerate(meta):
        n, l = site_of(i)
        jt = SK[l][1]
        row = lim[n, l, 0]
        picked = int(row[7]) - jt * A_HW * A_HW
        assert picked == di[n, jt, win], (tag, i)


@pytest.mark.parametrize('nd', [2, 4])
def test_two_pass_search_model(nd):
    """No GPU.  A model of K2's two-pass search over the exact squared distances picks the
    reference's index on every family-A construction with the window factor 1 + 2^-20; with no
    pass 2 (factor 1), a one-ulp window (1 + 2^-23), pass 2 without its break, or the squared
    distance evaluated the other way round (sq2's operands swapped, sq4 contracted into fma) it
    misses on some construction."""
    misses = {'best2': 0, 'ulp': 0, 'nobreak': 0, 'formula': 0}
    for tag, f, vecs, win in near_tie_sites(nd):
        d = [_a_diffs(v, f) for v in vecs]
        sq = [_a_sq(x) for x in d]
        ref = reference_pick(sq)
        assert two_pass_model(sq, len(sq), WINDOW) == ref, tag
        misses['best2'] += two_pass_model(sq, len(sq), 1) != ref
        misses['ulp'] += two_pass_model(sq, len(sq), 1 + 2.0 ** -23) != ref
        misses['nobreak'] += two_pass_model(sq, len(sq), WINDOW, first_break=False) != ref
        alt = [_alt_sq(x) for x in d]
        pick = two_pass_model(alt, len(alt), WINDOW)
        misses['formula'] += (pick != ref) or (exact_root(alt[pick]) != exact_root(sq[ref]))
    assert all(v > 0 for v in misses.values()), misses


# ---- B, C, D, E, G scenes
B_HW = 48


def threshold_scene():
    """Family B: (site tag, site).  From- or to-score at thre or one step below; the to-candidate
    at thre competes with a farther one well above thre."""
    lo = _down(THRE)
    sites = []
    for tag, fs, ts in (('from_at', THRE, [F32(0.8)]), ('from_below', lo, [F32(0.8)]),
                        ('to_at', F32(0.9), [THRE, F32(0.8)]), ('to_below', F32(0.9), [lo, F32(0.8)])):
        sites.append((tag, dict(frm=(10, 12), off=[F32(6.25), F32(5.5)], to=[(16, 18), (30, 36)][:len(ts)],
                                fs=fs, ts=ts)))
    return sites


def len_scene():
    """Family C: to-candidate at (+3, +4) of the from-candidate (norm exactly 5), guided off by
    (0.5, 0.25) so that the score depends on len."""
    return [dict(frm=(10, 10), off=[F32(3.5), F32(4.25)], to=[(13, 14)]),
            dict(frm=(20, 30), off=[F32(3.5), F32(4.25)], to=[(23, 34), (3, 3)])]


def gate_distance_scene():
    """Family D, distance and scale: min_dist exactly 5 (guided point at (+3, +4) of the
    to-candidate).  Returns sites and the scale_t of each (None: no scale map there: 0)."""
    scales = [None, F32(5), 'dist_max', _up(5), F32(np.nan), F32(4)]
    sites = [dict(frm=(10, 10), off=[F32(8), F32(10)], to=[(15, 16)]) for _ in scales]
    return sites, scales


def gate_border_scene():
    """Family D, borders and jitter: (tag, site, from jitter (jx, jy)).  Endpoints in row / column
    0 against 1 (kept only off 0), jitter moving x1 or y1 from 1 to exactly 0 and from 0 to 0.5."""
    out = []
    for tag, frm, to, jit in (
            ('x1_0', (0, 10), (6, 14), None), ('x1_1', (1, 10), (7, 14), None),
            ('y1_0', (10, 0), (14, 6), None), ('y1_1', (10, 1), (14, 7), None),
            ('x2_0', (6, 10), (0, 14), None), ('x2_1', (6, 10), (1, 14), None),
            ('y2_0', (10, 6), (14, 0), None), ('y2_1', (10, 6), (14, 1), None),
            ('jx_to_0', (1, 10), (7, 14), (F32(-1), F32(0))), ('jy_to_0', (10, 1), (14, 7), (F32(0), F32(-1))),
            ('jx_from_0', (0, 10), (6, 14), (F32(0.5), F32(0))), ('jy_from_0', (10, 0), (14, 6), (F32(0), F32(0.5)))):
        off = [F32(to[0] - frm[0] + 0.25), F32(to[1] - frm[1] - 0.5)]
        out.append((tag, dict(frm=frm, off=off, to=[to]), jit))
    return out


E_SHAPES = {'h_lt_w': (40, 64), 'h_gt_w': (64, 40)}


def jitter_bound_scene(h, w):
    """Family E: (tag, site) with guided points at the limits of the refinement's bounds.  The
    to-candidate sits next to the guided point; the jitter maps are dense."""
    out = []

    def add(tag, gx, gy):
        x1 = int(np.clip(np.floor(gx) + 3, 0, w - 1)) if gx < w / 2 else int(np.clip(np.floor(gx) - 3, 0, w - 1))
        y1 = int(np.clip(np.floor(gy) + 3, 0, h - 1)) if gy < h / 2 else int(np.clip(np.floor(gy) - 3, 0, h - 1))
        tx = int(np.clip(np.round(gx), 0, w - 1))
        ty = int(np.clip(np.round(gy), 0, h - 1))
        out.append((tag, dict(frm=(x1, y1), off=[F32(gx - x1), F32(gy - y1)], to=[(tx, ty)])))
    mid_y, mid_x = 20.25, 12.5
    add('gx_neg', -0.5, mid_y)
    add('gy_neg', mid_x, -0.75)
    add('gx_m1', -1.0, mid_y)
    add('gy_m1', mid_x, -1.0)
    add('gx_below_w', w - 0.25, mid_y)
    add('gy_below_h', mid_x, h - 0.25)
    add('inside', mid_x + 3, mid_y + 2)
    lo, hi = min(h, w), max(h, w)
    if w > h:         # x in [h, w): inside the reference's check, outside the plane's rows
        add('x_off_plane', (lo + hi) / 2 + 0.5, mid_y)
    else:             # x in [w, h): outside the check, inside the plane's rows
        add('x_off_check', (lo + hi) / 2 + 0.5, mid_y)
    if h > w:         # y in [w, h): inside the check, outside the plane's columns
        add('y_off_plane', mid_x, (lo + hi) / 2 + 0.5)
    else:             # y in [h, w): outside the check, inside the plane's columns
        add('y_off_check', mid_x, (lo + hi) / 2 + 0.5)
    return out


def jitter_maps(n, h, w, seed):
    """Dense jitter offsets, multiples of 1/32 in [-1/4, 1/4], nonzero everywhere."""
    rng = np.random.RandomState(seed)
    v = rng.randint(1, 9, size=(n, 2, h, w)) * rng.choice([-1, 1], size=(n, 2, h, w))
    return (v / 32.0).astype(F32)


def _guided(site):
    return site['frm'][0] + float(site['off'][0]), site['frm'][1] + float(site['off'][1])


def _regions(gx, gy, h, w):
    """(inside the reference's bounds check, inside the indexed plane) of a guided point."""
    xi, yi = int(np.trunc(gx)), int(np.trunc(gy))
    return 0 <= xi < w and 0 <= yi < h, 0 <= xi < h and 0 <= yi < w


def nan_scene():
    """Family G on the chain skeleton GSK (min_len = 0): (image, description).  Image 0: a NaN row
    (from- and to-candidate on one pixel, zero offset) starts a person that the next limb extends.
    Image 1: a person started by a finite row at limb 0 matches a NaN row at limb 1.  Image 2: a
    NaN row shares its to-id with a finite row."""
    h = w = 32
    heat = np.zeros((3, 3, h, w), F32)
    offs = np.zeros((3, 4, h, w), F32)
    # image 0: keypoints 0 and 1 on (10, 10); keypoint 2 at (14, 13), guided from 1 by (4, 3.5)
    heat[0, 0, 10, 10], heat[0, 1, 10, 10], heat[0, 2, 13, 14] = 0.9, 0.8, 0.7
    offs[0, 2, 10, 10], offs[0, 3, 10, 10] = 4, 3.5
    # image 1: 0 at (5, 6) guided to 1 at (9, 8); 2 on 1's pixel, zero offset
    heat[1, 0, 6, 5], heat[1, 1, 8, 9], heat[1, 2, 8, 9] = 0.9, 0.8, 0.7
    offs[1, 0, 6, 5], offs[1, 1, 6, 5] = 4.25, 2
    # image 2: 0 at (20, 20) and (12, 12); 1 on (20, 20); the (12, 12) candidate is guided there
    heat[2, 0, 20, 20], heat[2, 0, 12, 12], heat[2, 1, 20, 20] = 0.9, 0.85, 0.8
    offs[2, 0, 12, 12], offs[2, 1, 12, 12] = 8.5, 7.75
    return heat, offs


GSK = [(0, 1), (1, 2)]


def drop_nan_rows(limbs):
    """The limb table as `prepare_limb_rows` sees it: rows with a NaN limb score never pass."""
    out = limbs.copy()
    out[np.isnan(out[..., 10]), 8] = np.inf
    return out


def test_boundary_constructions_reach_their_regimes():
    """No GPU.  The oracle's limbs show that each construction of families B, C, D, E and G sits
    exactly where it is meant to."""
    # B: the from-candidate at thre keeps its position, one step below is moved off the image;
    # a to-candidate at thre is the nearest one, one step below it is moved away
    sites = [s for _, s in threshold_scene()]
    heat, offs = build_scene(sites, 2, B_HW, B_HW)
    lim = ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1)
    assert lim[0, 0, 0, 0] == 10 and lim[0, 1, 0, 0] == 10 - 100000
    assert lim[1, 0, 0, 3] == 16 and lim[1, 0, 0, 8] < 1
    assert lim[1, 1, 0, 3] == 30 and lim[1, 1, 0, 8] > 10
    # C: the norm is exactly 5 and the score depends on len
    heat, offs = build_scene(len_scene(), 1, B_HW, B_HW)
    for ml, want in ((_down(5), F32(5)), (F32(5), F32(5)), (_up(5), _up(5))):
        lim = ro.generate_limbs(heat, offs, SK, 8, THRE, ml, 1, 1)
        assert np.all(lim[0, :, 0, 9] == want) and np.all(lim[0, :, 0, 8] > 0)
    # D: min_dist is exactly 5
    sites, _ = gate_distance_scene()
    heat, offs = build_scene(sites, 3, B_HW, B_HW)
    lim = ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1)
    assert np.all(lim[:, :, 0, 8] == 5)
    # D: the border endpoints and the jitter-moved ones land on 0 or 1 / 0.5
    rows = gate_border_scene()
    heat, offs = build_scene([s for _, s, _ in rows], 6, B_HW, B_HW)
    jom = gate_jitter(rows, 6, B_HW, B_HW)
    lim = ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1, jomps_hr=jom, use_jitter=True)
    col = {'x1': 0, 'y1': 1, 'x2': 3, 'y2': 4}
    for i, (tag, s, jit) in enumerate(rows):
        r = lim[site_of(i)][0]
        assert r[7] == SK[site_of(i)[1]][1] * B_HW * B_HW + s['to'][0][1] * B_HW + s['to'][0][0], tag
        if tag.startswith('j'):
            c = 0 if tag[1] == 'x' else 1
            assert r[c] == (0 if tag.endswith('to_0') else 0.5), tag
        else:
            assert r[col[tag[:2]]] == int(tag[-1]), tag
        assert r[8] < 2 and all(r[c] >= 0 for c in (0, 1, 3, 4)), tag
    # E: every region is present on both shapes
    for name, (h, w) in E_SHAPES.items():
        seen = set()
        for tag, s in jitter_bound_scene(h, w):
            gx, gy = _guided(s)
            seen.add(_regions(gx, gy, h, w))
            if tag.endswith('_neg'):
                assert -1 < (gx if tag[1] == 'x' else gy) < 0
            if tag.endswith('_m1'):
                assert (gx if tag[1] == 'x' else gy) == -1
        assert {(True, True), (True, False), (False, False)} <= seen, (name, seen)
    both = set()
    for h, w in E_SHAPES.values():
        both |= {_regions(*_guided(s), h, w) for _, s in jitter_bound_scene(h, w)}
    assert len(both) == 4
    # G: NaN rows where intended, and the reference's grouping differs from the NaN-free one
    heat, offs = nan_scene()
    with np.errstate(invalid='ignore'):
        lim = ro.generate_limbs(heat, offs, GSK, 8, THRE, 0.0, 1, 1)
    nan = np.isnan(lim[..., 10]) & (lim[..., 2] >= THRE)
    assert nan[0, 0, 0] and nan[1, 1, 0] and nan[2, 0, 0] and nan.sum() == 3
    assert lim[2, 0, 0, 7] == lim[2, 0, 1, 7]          # the NaN row shares the finite row's to-id
    full = [ro.group_skeletons(lim[i], GSK, 3, PERSON_THRE, 2, 20, True) for i in range(3)]
    pinned = [ro.group_skeletons(drop_nan_rows(lim)[i], GSK, 3, PERSON_THRE, 2, 20, True) for i in range(3)]
    assert full[0].shape == (1, 3, 6) and full[0][0, 0, 5] > 0 and np.isnan(full[0][0, 0, 4])
    assert pinned[0][0, 0, 5] == 0                      # without the NaN row keypoint 0 is unset
    for i in (1, 2):
        gio.compare_poses(pinned[i], full[i])


def gate_jitter(rows, n, h, w):
    """Jitter maps of the border scene: the listed jitter at each from-candidate, 0 elsewhere."""
    jom = np.zeros((n, 2, h, w), F32)
    for i, (_, s, jit) in enumerate(rows):
        if jit is not None:
            x, y = s['frm']
            jom[site_of(i)[0], :, y, x] = jit
    return jom


def test_jitter_oracle_raises_off_the_plane():
    """No GPU.  The oracle's jitter refinement raises IndexError for a guided point inside the
    reference's bounds check but outside the [x, y]-as-[row, col] indexed plane, as the reference
    does; with `unrefined_off_plane` it leaves that point unrefined."""
    for h, w in E_SHAPES.values():
        rows = jitter_bound_scene(h, w)
        heat, offs = build_scene([s for _, s in rows], (len(rows) + 1) // 2, h, w)
        jom = jitter_maps(heat.shape[0], h, w, 5)
        with pytest.raises(IndexError):
            ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1, jomps_hr=jom, use_jitter=True)
        ro.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1, jomps_hr=jom, use_jitter=True,
                          unrefined_off_plane=True)


def test_nan_scores_rank_last_in_both_oracles():
    """No GPU.  Limb scores [0.5, NaN, 0.7, 0.5] (distinct to-ids) rank [2, 0, 3, 1] in the numpy
    oracle, the stable form of np.argsort(-s); the C oracle groups that table the same way."""
    limbs = np.zeros((1, 4, 13), F32)
    for k, s in enumerate([0.5, np.nan, 0.7, 0.5]):
        limbs[0, k] = [2 + 3 * k, 2, 0.9, 3 + 3 * k, 4, 0.8, 100 + k, 200 + k, 1, 2, s, 4, 4]
    assert ro.delete_reconns(limbs[0], ro.valid_limb_rows(limbs[0], 20, False)) == [2, 0, 3, 1]
    assert list(np.argsort(-limbs[0, :, 10], kind='stable')) == [2, 0, 3, 1]
    # rows 0 and 2 share a to-id with the NaN row: the finite rows win wherever they stand
    limbs[0, :, 7] = [200, 200, 201, 201]
    assert ro.delete_reconns(limbs[0], ro.valid_limb_rows(limbs[0], 20, False)) == [2, 0]
    limbs[0, :, 7] = [200, 201, 202, 201]
    kept = ro.delete_reconns(limbs[0], ro.valid_limb_rows(limbs[0], 20, False))
    assert kept == [2, 0, 3]
    skel = [(0, 1)]
    for table in (limbs, np.ascontiguousarray(limbs[:, ::-1])):
        ref = ro.group_skeletons(table, skel, 2, 0.01, 2, 20, False)
        got = co.group_batch(table[None], skel, 2, 0.01, 2, 20, False)[0]
        assert ref.shape[0] == 3
        gio.compare_poses(got, ref)


# =========================================================================== GPU
@pytest.fixture(scope='module')
def engines(cuda_device):
    """Engines by configuration, made on first use."""
    from offsetguided_b200.engine import DecoderEngine
    made = {}

    def get(topk=8, min_len=0.5, dist_max=20.0, use_scale=True, skeleton=SK, n_keypoints=C):
        key = (topk, float(min_len), float(dist_max), use_scale, tuple(skeleton))
        if key not in made:
            made[key] = DecoderEngine(n_keypoints, skeleton, topk=topk, thre_hmp=float(THRE), min_len=float(min_len),
                                      resize_factor=1.0, dist_max=float(dist_max), use_scale=use_scale,
                                      person_thre=PERSON_THRE, sort_dim=2)
        return made[key]
    yield get
    for e in made.values():
        e.close()


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda() if a is not None else None


def assert_limbs(got, ref, rows=None):
    """Columns other than the limb score bit for bit (NaN equal to NaN), the score to RTOL."""
    if rows is not None:
        got, ref = got[rows], ref[rows]
    cols = [c for c in range(13) if c != 10]
    for c in cols:
        assert np.array_equal(got[..., c], ref[..., c], equal_nan=True), f'limb column {c} differs'
    np.testing.assert_allclose(got[..., 10], ref[..., 10], rtol=RTOL, atol=0, equal_nan=True)


def oracle_limbs(heat, offs, k, min_len=0.5, nd=2, scales=None, jomps=None, use_jitter=False, skel=SK):
    with np.errstate(invalid='ignore', divide='ignore'):
        return ro.generate_limbs(heat, offs, skel, k, THRE, min_len, 1, 1, scmps_hr=scales, jomps_hr=jomps,
                                 use_jitter=use_jitter, vector_nd=nd, unrefined_off_plane=True)


def route_k2(eng, heat, offs, k, nd=2, jomps=None, use_jitter=False):
    """K2 alone on the oracle's own top-K lists (fillers and sub-threshold candidates included)."""
    ds, di, _, _ = ro.joint_dets(heat, k)
    return eng.limb_score(_t(ds), _t(di.astype(np.int32)), _t(offs), jomps=_t(jomps), vector_nd=nd,
                          use_jitter=use_jitter).cpu().numpy()


def route_decode(eng, heat, offs, nd=2, scales=None, jomps=None, use_jitter=False):
    """K1 -> K2 + prep -> K3: (poses per image, limbs)."""
    poses = eng.decode_maps(_t(heat), _t(offs), _t(scales), jomps=_t(jomps), vector_nd=nd, use_jitter=use_jitter)
    _, _, lb = eng.last_intermediates(heat.shape[0])
    return poses, lb.cpu().numpy()


def live_rows(ref):
    """Rows of listed candidates: from-candidate >= thre (K1 lists no others)."""
    return ref[..., 2] >= THRE


def check_decode(eng, heat, offs, ref, skel=SK, dist_max=20.0, use_scale=True, **kw):
    """Decode path against the oracle: limbs of live from-candidates whose matched to-candidate is
    live bit for bit, inert rows far away; poses equal to both oracles' grouping of `ref`."""
    poses, lb = route_decode(eng, heat, offs, **kw)
    live = live_rows(ref)
    to_live = live & (ref[..., 5] >= THRE)
    assert np.array_equal(live, lb[..., 2] >= THRE)
    assert_limbs(lb, ref, to_live)
    assert np.all(lb[live & ~to_live][:, 8] > 5e4)
    check_poses(poses, ref, skel, dist_max, use_scale)
    return poses, lb


def check_poses(poses, ref, skel=SK, dist_max=20.0, use_scale=True, n_kp=None):
    n_kp = n_kp or max(max(a, b) for a, b in skel) + 1
    want = co.group_batch(ref, skel, n_kp, PERSON_THRE, 2, dist_max, use_scale)
    assert len(poses) == len(want) == ref.shape[0]
    for i, (p, r) in enumerate(zip(poses, want)):
        gio.compare_poses(p, ro.group_skeletons(ref[i], skel, n_kp, PERSON_THRE, 2, dist_max, use_scale), RTOL)
        gio.compare_poses(p, r, RTOL)


@pytest.mark.gpu
@pytest.mark.parametrize('nd', [2, 4])
def test_near_ties(engines, nd):
    """Family A: K2 picks the reference's first index of the smallest rounded distance, alone and
    on the decode path; 2-D against the C oracle as well."""
    heat, offs, meta = near_tie_scene(nd)
    eng = engines()
    ref = oracle_limbs(heat, offs, 8, nd=nd)
    got = route_k2(eng, heat, offs, 8, nd)
    assert_limbs(got, ref)
    if nd == 2:
        assert_limbs(got, co.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1))
    check_decode(eng, heat, offs, ref, nd=nd)


@pytest.mark.gpu
def test_threshold_shift(engines):
    """Family B: a candidate at thre stays, one a float32 step below moves off the image."""
    heat, offs = build_scene([s for _, s in threshold_scene()], 2, B_HW, B_HW)
    eng = engines()
    ref = oracle_limbs(heat, offs, 8)
    assert_limbs(route_k2(eng, heat, offs, 8), ref)
    assert_limbs(route_k2(eng, heat, offs, 8), co.generate_limbs(heat, offs, SK, 8, THRE, 0.5, 1, 1))
    check_decode(eng, heat, offs, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('min_len', ['below', 'at', 'above'])
def test_len_at_min_len(engines, min_len):
    """Family C: len = max(norm, min_len) with the norm 5 and min_len = 5 and one step either side."""
    ml = {'below': _down(5), 'at': F32(5), 'above': _up(5)}[min_len]
    heat, offs = build_scene(len_scene(), 1, B_HW, B_HW)
    eng = engines(min_len=ml)
    ref = oracle_limbs(heat, offs, 8, min_len=ml)
    assert_limbs(route_k2(eng, heat, offs, 8), ref)
    check_decode(eng, heat, offs, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('dist_max', ['below', 'at', 'above'])
def test_gate_distance_and_scale(engines, dist_max):
    """Family D: min_dist = 5 against dist_max = 5 and one step either side, without scale maps and
    with scale_t = min_dist, = dist_max, one step above min_dist, NaN and 4; a row is kept only
    when min_dist < max(dist_max, scale_t) strictly, and never with a NaN scale."""
    dm = {'below': _down(5), 'at': F32(5), 'above': _up(5)}[dist_max]
    sites, scale_t = gate_distance_scene()
    n = (len(sites) + 1) // 2
    heat, offs = build_scene(sites, n, B_HW, B_HW)
    eng = engines(dist_max=dm)
    ref = oracle_limbs(heat, offs, 8)
    check_decode(eng, heat, offs, ref, dist_max=dm)            # no scale maps: scale_t = 4
    scales = np.zeros_like(heat)
    for i, (s, v) in enumerate(zip(sites, scale_t)):
        n_, l = site_of(i)
        x, y = s['to'][0]
        scales[n_, SK[l][1], y, x] = dm if isinstance(v, str) else (0 if v is None else v)
    ref = oracle_limbs(heat, offs, 8, scales=scales)
    poses, _ = check_decode(eng, heat, offs, ref, dist_max=dm, scales=scales)
    kept = [len(p) for p in poses]
    assert sum(kept) == (5 if dist_max == 'above' else 1), kept    # scale_t = next(5) always, the rest but NaN above
    got = eng.group(_t(ref))
    check_poses(got, ref, dist_max=dm)


@pytest.mark.gpu
def test_gate_borders_and_jitter(engines):
    """Family D: endpoints in row / column 0 fail the gate, in row / column 1 pass; jitter that
    moves x1 or y1 to exactly 0 fails it, jitter from 0 to 0.5 passes."""
    rows = gate_border_scene()
    heat, offs = build_scene([s for _, s, _ in rows], 6, B_HW, B_HW)
    eng = engines()
    ref = oracle_limbs(heat, offs, 8)
    poses, _ = check_decode(eng, heat, offs, ref)
    check_poses(eng.group(_t(ref)), ref)
    jom = gate_jitter(rows, 6, B_HW, B_HW)
    ref = oracle_limbs(heat, offs, 8, jomps=jom, use_jitter=True)
    poses, _ = check_decode(eng, heat, offs, ref, jomps=jom, use_jitter=True)
    check_poses(eng.group(_t(ref)), ref)
    assert sum(len(p) for p in poses) == 6            # *_1 (4) and jitter from 0 (2) keep their row


@pytest.mark.gpu
@pytest.mark.parametrize('shape', list(E_SHAPES))
def test_jitter_bounds(engines, shape):
    """Family E: the guided point is refined at column 0 for x in (-1, 0) (truncation), not at -1,
    just below W / H only inside the indexed plane; maps with H < W and H > W."""
    h, w = E_SHAPES[shape]
    rows = jitter_bound_scene(h, w)
    heat, offs = build_scene([s for _, s in rows], (len(rows) + 1) // 2, h, w)
    jom = jitter_maps(heat.shape[0], h, w, 5)
    eng = engines()
    ref = oracle_limbs(heat, offs, 8, jomps=jom, use_jitter=True)
    assert_limbs(route_k2(eng, heat, offs, 8, jomps=jom, use_jitter=True), ref)
    check_decode(eng, heat, offs, ref, jomps=jom, use_jitter=True)


KS = (31, 32, 33, 63, 64, 65, 127, 128)


def many_candidates(k, nd, seed):
    """Family F: two images; image 0 lists exactly K live candidates per channel, image 1 K - 7.
    From-candidates on a 4-px grid, to-candidates at (+1, +2) of them, offsets (1, 2) +- up to
    1/2 in steps of 1/16 (4-D: both vectors)."""
    rng = np.random.RandomState(seed)
    h = w = 60
    grid = [(x, y) for y in range(2, h - 3, 4) for x in range(2, w - 3, 4)]
    heat = np.zeros((2, C, h, w), F32)
    offs = np.zeros((2, nd * L, h, w), F32)
    for n, live in ((0, k), (1, k - 7)):
        for l, (jf, jt) in enumerate(SK):
            pick = rng.choice(len(grid), live, replace=False)
            vals = rng.choice(np.arange(1, 3001), 2 * live, replace=False) / 3001.0 * 0.7 + 0.28
            for a, g in enumerate(pick):
                x, y = grid[g]
                heat[n, jf, y, x] = vals[a]
                heat[n, jt, y + 2, x + 1] = vals[live + a]
                for c in range(nd):
                    offs[n, nd * l + c, y, x] = (1, 2)[c % 2] + rng.randint(-8, 9) / 16.0
    return heat, offs


@pytest.mark.gpu
@pytest.mark.parametrize('nd', [2, 4])
@pytest.mark.parametrize('k', KS)
def test_k_around_cta_sizes(engines, k, nd):
    """Family F: every K around the 32 / 64 / 128-thread CTAs, full and partly empty lists: K2
    alone, the decode path (K2's fused prep) and the stand-alone prep + K3 on the oracle's table."""
    heat, offs = many_candidates(k, nd, 1000 + k)
    eng = engines(topk=k)
    ref = oracle_limbs(heat, offs, k, nd=nd)
    assert_limbs(route_k2(eng, heat, offs, k, nd), ref)
    if nd == 2:
        assert_limbs(route_k2(eng, heat, offs, k, nd), co.generate_limbs(heat, offs, SK, k, THRE, 0.5, 1, 1))
    poses, _ = check_decode(eng, heat, offs, ref, nd=nd)
    assert min(len(p) for p in poses) > 0
    check_poses(eng.group(_t(ref)), ref)


@pytest.mark.gpu
def test_nan_limb_scores_are_dropped(engines):
    """Family G (min_len = 0): a limb whose from- and to-candidate share a pixel and whose offset is
    exactly zero scores 0 * exp(-0 / 0) = NaN.  The reference keeps such a row (sorted last) and
    lets it start a person; `prepare_limb_rows` drops it (DESIGN.md section 3).  Pinned here: the
    decode path and the stand-alone grouping equal both oracles on the table without the NaN rows,
    and the NaN rows themselves are the reference's."""
    heat, offs = nan_scene()
    eng = engines(min_len=0.0, skeleton=GSK, n_keypoints=3)
    ref = oracle_limbs(heat, offs, 8, min_len=0.0, skel=GSK)
    poses, lb = route_decode(eng, heat, offs)
    live = live_rows(ref) & (ref[..., 5] >= THRE)
    assert_limbs(lb, ref, live)
    assert (np.isnan(lb[..., 10]) & live).sum() == 3
    pinned = drop_nan_rows(ref)
    check_poses(poses, pinned, GSK, n_kp=3)
    check_poses(eng.group(_t(ref)), pinned, GSK, n_kp=3)
    full = ro.group_skeletons(ref[0], GSK, 3, PERSON_THRE, 2, 20, True)
    assert full[0, 0, 5] > 0 and poses[0][0, 0, 5] == 0        # the documented deviation
