"""Result rows of the grouping kernels' epilogue (SURVEY 8f-2) on every grouping path and call route.

When image frames are staged, both grouping kernels (the one-warp kernel and the CTA kernel it hands
oversized images to) end with ``coco_joint``: every joint is moved back into its image's frame as
(x + offset) / scale, each step in float64 rounded to float32, rounded to two decimals in float32
(x * 100, rint, / 100) and flagged x > 0 or y > 0; every person is scored with the float64
left-to-right mean of its C keypoint scores.  The rows must equal the reference's loops
(``ro.coco_result_rows``) run on the same poses, bit for bit.

Frames are per image, so one joint per image and axis can be steered onto any value: with scale 1
and offset v - x (exact in float64) a joint lands on any float32 v, with scale 8 and an odd x1 on a
multiple of 1/8.  The constructions below put joints where a subtly different epilogue gives other
rows (ties of the rounding, float32 products that are ties while the exact ones are not, float32
cancellation and division next to a rounding boundary, zero and negative-zero flags, unset joints);
a numpy model of ``coco_joint`` and its mutants shows, with and without a GPU, that they do.

The GPU tests decode each batch once without frames and then with frames: the poses must not
change, and the rows must equal the reference loops and ``results.coco_results``.  They run on the
warp kernel, the CTA kernel, both in one call, the regroup into a worst-case result buffer and the
candidate-list overflow redo, through replayed graphs, kernel-by-kernel launches, pinned host maps
of several image ranges, full-resolution maps and the materialising path; and they follow the
frames through graph replays, alternating calls, growing batches and refused calls."""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import ref_oracle as ro
from oracle import scenes
from offsetguided_b200 import config as cfg
from offsetguided_b200 import results
from test_gpu_parity import _lowres_scene
from test_k3_crowds import CHAIN, _chain_maps, _crowd_scenes

F32, F64 = np.float32, np.float64
HUNDRED = F32(100)
SKEL = cfg.COCO_PERSON_SKELETON
KW = dict(topk=16, thre_hmp=0.05, min_len=0.5, dist_max=40, use_scale=True, person_thre=0.05)
MUTANTS = ('float_add', 'float_divide', 'reciprocal', 'product_f64', 'roundf', 'flag_unrounded', 'flag_ge',
           'score_f32', 'score_set_joints')


# --------------------------------------------------------------------------- model of coco_joint
def _round2(v, mutants=()):
    """np.around(v, 2) of float32 values as the epilogue computes it: x * 100 in float32, rint, / 100."""
    v = np.asarray(v, F32)
    if 'product_f64' in mutants:
        return (np.rint(v.astype(F64) * 100.0) / 100.0).astype(F32)
    p = v * HUNDRED
    if 'roundf' in mutants:                        # halves away from zero
        t = np.trunc(p)
        r = np.where(np.abs(p - t) >= F32(0.5), t + np.sign(p), t).astype(F32)
    else:
        r = np.rint(p)
    return (r / HUNDRED).astype(F32)


def _axis(v, offset, scale, mutants):
    v = np.asarray(v, F32)
    if 'float_add' in mutants:
        v1 = (v + F32(offset)).astype(F32)
    else:
        v1 = (v.astype(F64) + F64(offset)).astype(F32)
    if 'float_divide' in mutants:
        return (v1 / F32(scale)).astype(F32)
    if 'reciprocal' in mutants:
        return (v1 * F32(1.0 / scale)).astype(F32)
    return (v1.astype(F64) / F64(scale)).astype(F32)


def _joint(x, y, frame, mutants=()):
    """coco_joint (og_group.cu) on arrays of pose coordinates: (x3, y3, flag, x2, y2)."""
    x2 = _axis(x, frame[0], frame[2], mutants)
    y2 = _axis(y, frame[1], frame[3], mutants)
    x3, y3 = _round2(x2, mutants), _round2(y2, mutants)
    fx, fy = (x2, y2) if 'flag_unrounded' in mutants else (x3, y3)
    flag = ((fx >= 0) | (fy >= 0)) if 'flag_ge' in mutants else ((fx > 0) | (fy > 0))
    return x3, y3, flag.astype(F32), x2, y2


def _score(v, mutants=()):
    """sum(v) / len(v) of the keypoint scores, float64 left to right (evaluate.py:250)."""
    c = v.shape[1]
    if 'score_f32' in mutants:
        acc = np.zeros(len(v), F32)
        for j in range(c):
            acc = (acc + v[:, j]).astype(F32)
        return acc.astype(F64) / c
    acc = np.zeros(len(v), F64)
    for j in range(c):
        acc = acc + v[:, j].astype(F64)
    if 'score_set_joints' in mutants:
        return acc / np.maximum((v != 0).sum(axis=1), 1)
    return acc / c


def _model_rows(poses, frames, mutants=()):
    """(keypoints (T, 3C) float32, scores (T,) float64, image index (T,)) of the model."""
    kp, sc, im = [], [], []
    for i, (p, f) in enumerate(zip(poses, frames)):
        c = p.shape[1]
        if len(p) == 0:
            kp.append(np.zeros((1, 3 * c), F32))
            sc.append(np.array([0.01]))
            im.append(np.array([i]))
            continue
        x3, y3, flag, _, _ = _joint(p[:, :, 0], p[:, :, 1], f, mutants)
        kp.append(np.stack([x3, y3, flag], axis=2).reshape(len(p), 3 * c))
        sc.append(_score(p[:, :, 2], mutants))
        im.append(np.full(len(p), i))
    return np.concatenate(kp), np.concatenate(sc).astype(F64), np.concatenate(im)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view({4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def _same(a, b):
    """Equal bit for bit (so -0.0 differs from 0.0), shapes and types included."""
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(_bits(a), _bits(b))


def _rows_as_arrays(rows, ids):
    kp = np.array([r['keypoints'] for r in rows], F64).astype(F32)
    sc = np.array([r['score'] for r in rows], F64)
    im = np.array([ids.index(r['image_id']) for r in rows])
    return kp, sc, im


def _reference(poses, metas):
    return _rows_as_arrays(*ro.coco_result_rows(poses, metas))


# --------------------------------------------------------------------------- constructions
@functools.lru_cache(maxsize=None)
def _float32_ties():
    """Positive float32 v whose float32 product with 100 is exactly k + 1/2 while the exact product is
    not, so that rint of the float32 product and rounding of the exact one disagree (0.915f: 0.92
    against 0.91).  Found with exact rational arithmetic."""
    out = []
    for k in range(1, 3000):
        tie = Fraction(2 * k + 1, 200)
        v = F32(float(tie))
        for v in (np.nextafter(np.nextafter(v, F32(0)), F32(0)), np.nextafter(v, F32(0)), v,
                  np.nextafter(v, F32(1e9)), np.nextafter(np.nextafter(v, F32(1e9)), F32(1e9))):
            p = v * HUNDRED
            exact = Fraction(float(v)) * 100
            if Fraction(float(p)) == Fraction(2 * k + 1, 2) and exact != Fraction(2 * k + 1, 2) \
                    and int(np.rint(p)) != math.floor(exact + Fraction(1, 2)):
                out.append(F32(v))
        if len(out) >= 4:
            return tuple(out)
    raise AssertionError('no float32 product ties found')


def _boundary(k):
    """The 0.01 rounding boundary (k + 1/2) / 100 (k may be negative)."""
    return (k + 0.5) / 100.0


def _cancel_offset(x, k):
    """Offset o ~ -x with a full-precision fraction: the exact sum x + o lands just beside the
    boundary _boundary(k), and adding in float32 (x + fl32(o)) lands on its other side."""
    x = F32(x)
    o = (_boundary(k) + np.arange(-600, 601) * 1e-8) - F64(x)
    good = _round2((F64(x) + o).astype(F32))
    bad = _round2((x + o.astype(F32)).astype(F32))
    hit = np.nonzero(good != bad)[0]
    return float(o[hit[len(hit) // 2]]) if hit.size else 0.123456789 - float(x)


def _division_scale(v1, k):
    """Scale s (float64): fl32(v1 / s) lies beside the boundary _boundary(k), and both v1 / fl32(s) in
    float32 and v1 * fl32(1 / s) land on its other side (either one when both cannot)."""
    v1 = F32(v1)
    s = F64(v1) / (_boundary(k) * (1.0 + np.arange(-400, 401) * 2.0 ** -27))
    good = _round2((F64(v1) / s).astype(F32))
    fdiv = _round2((v1 / s.astype(F32)).astype(F32))
    recip = _round2((v1 * (1.0 / s).astype(F32)).astype(F32))
    for mask in ((good != fdiv) & (good != recip), (good != fdiv) | (good != recip)):
        hit = np.nonzero(mask)[0]
        if hit.size:
            return float(s[hit[0]])
    return 1.7


def _families():
    """(name, x axis, y axis) of the steered joint of an image.  Axis specs: ('at', v) lands on
    float32 v (scale 1), ('eighth', m) on m / 8 (odd m, scale 8), ('cancel', k) and ('div', v1, k)
    beside boundary k, ('fixed', offset, scale) leaves the joint where the frame puts it."""
    t = _float32_ties()
    return [
        ('tie', ('at', 0.125), ('at', -0.625)),                   # 12.5 and -62.5: rint 12 / -62, roundf 13 / -63
        ('tie', ('eighth', 9), ('eighth', -1)),                   # 1.125 and -0.125 through a division by 8
        ('tie', ('eighth', 5), ('eighth', -9)),
        ('tie32', ('at', t[0]), ('at', -t[1])),
        ('tie32', ('at', t[2]), ('at', -t[3])),
        ('cancel', ('cancel', 12), ('cancel', -31)),
        ('cancel', ('cancel', 3), ('cancel', 47)),
        ('div', ('div', 37.0, 41), ('div', -23.0, -18)),
        ('div', ('div', 311.0, 5), ('div', 129.0, 73)),
        ('zero', ('at', 0.003), ('at', -2.0)),                    # x2 in (0, 0.005): x3 = 0, flag 0
        ('zero', ('at', 0.0), ('at', 0.01)),                      # x3 = 0, y3 = 0.01: flag 1
        ('zero', ('at', -0.003), ('at', -1.0)),                   # x3 = -0.0, flag 0
        ('zero', ('at', 0.0), ('at', -0.004)),                    # x3 = 0, y3 = -0.0: flag 0
    ]


UNSET = [('unset0', ('fixed', 0.0, 1.3), ('fixed', 0.0, 0.7)),   # unset joints stay (0, 0, 0)
         ('unset+', ('fixed', 3.5, 1.5), ('fixed', 2.25, 0.75))]  # unset joints at (2.33, 3), flag 1


def _axis_frame(spec, coord):
    kind = spec[0]
    if kind == 'at':
        return F64(F32(spec[1])) - F64(coord), 1.0
    if kind == 'eighth':
        return F64(spec[1]) - F64(coord), 8.0
    if kind == 'cancel':
        return _cancel_offset(coord, spec[1]), 1.0
    if kind == 'div':
        return F64(spec[1]) - F64(coord), _division_scale(spec[1], spec[2])
    return spec[1], spec[2]


def _generic(rng):
    return [-float(rng.randint(0, 90)) + rng.uniform(0, 1), -float(rng.randint(0, 60)) + rng.uniform(0, 1),
            rng.uniform(0.4, 1.7), rng.uniform(0.4, 1.7)]


def _frames_for(poses, seed, constructed=True):
    """(n, 4) float64 frames for decoded poses and the family of every image.  Images with unset
    joints take the unset families first, images with persons the steering families in turn, the
    others (and everything when not ``constructed``) a random frame like the reference's metas."""
    rng = np.random.RandomState(seed)
    fams, unset = list(_families()), list(UNSET)
    frames, names = [], []
    for p in poses:
        if not constructed or len(p) == 0:
            frames.append(_generic(rng))
            names.append('generic' if len(p) else 'empty')
            continue
        if unset and (p[:, :, 2] == 0).any():
            name, xs, ys = unset.pop(0)
        else:
            name, xs, ys = fams.pop(0) if fams else ('generic', None, None)
        if xs is None:
            frames.append(_generic(rng))
            names.append(name)
            continue
        j = int(np.nonzero((p[0, :, 2] > 0) & (p[0, :, 0] >= 1) & (p[0, :, 1] >= 1))[0][0])
        (ox, sx), (oy, sy) = _axis_frame(xs, p[0, j, 0]), _axis_frame(ys, p[0, j, 1])
        frames.append([ox, oy, sx, sy])
        names.append(name)
    return np.array(frames, F64).reshape(-1, 4), names


def _metas(frames):
    return [{'offset': np.array(f[:2], F64), 'scale': np.array(f[2:], F64), 'hflip': False,
             'width_height': (640, 480), 'image_id': 1000 + i} for i, f in enumerate(frames)]


def _regimes(poses, frames):
    """Which limits the rows of these poses and frames reach; the mutants that change them."""
    seen = set()
    for p, f in zip(poses, frames):
        if len(p) == 0:
            seen.add('empty')
            continue
        x3, y3, flag, x2, y2 = _joint(p[:, :, 0], p[:, :, 1], f)
        unset = p[:, :, 2] == 0
        for v2, v3 in ((x2, x3), (y2, y3)):
            prod = v2 * HUNDRED
            # a tie that rint takes towards zero, where roundf goes away from it
            tie = (prod - np.floor(prod) == F32(0.5)) & (np.abs(np.rint(prod)) < np.abs(prod))
            if (tie & (prod > 0)).any():
                seen.add('tie+')
            if (tie & (prod < 0)).any():
                seen.add('tie-')
            if (tie & (v2.astype(F64) * 100.0 != prod.astype(F64))).any():
                seen.add('tie32')
            if ((v3 == 0) & np.signbit(v3)).any():
                seen.add('-0.0')
        if ((x2 > 0) & (x2 < F32(0.005)) & (flag == 0)).any():
            seen.add('x2 in (0, 0.005), flag 0')
        if ((x3 == 0) & (y3 < 0) & (flag == 0)).any():
            seen.add('x3 = 0, y3 < 0')
        if ((x3 == 0) & (y3 == F32(0.01)) & (flag == 1)).any():
            seen.add('x3 = 0, y3 = 0.01')
        if (unset & (x3 == 0) & (y3 == 0) & (flag == 0)).any():
            seen.add('unset (0, 0, 0)')
        if (unset & (flag == 1)).any():
            seen.add('unset, flag 1')
    ref = _model_rows(poses, frames)
    for m in MUTANTS:
        got = _model_rows(poses, frames, (m,))
        if not (_same(got[0], ref[0]) and _same(got[1], ref[1])):
            seen.add(m)
    return seen


REGIMES = {'tie+', 'tie-', 'tie32', '-0.0', 'x2 in (0, 0.005), flag 0', 'x3 = 0, y3 < 0', 'x3 = 0, y3 = 0.01',
           'unset (0, 0, 0)', 'unset, flag 1', 'empty'} | set(MUTANTS)


# --------------------------------------------------------------------------- CPU
def _synthetic_poses(rng, n, c=17):
    out = []
    for i in range(n):
        m = 0 if i % 9 == 4 else rng.randint(1, 4)
        p = np.zeros((m, c, 6), F32)
        p[:, :, 0] = rng.randint(1, 640, size=(m, c))
        p[:, :, 1] = rng.randint(1, 480, size=(m, c))
        p[:, :, 2] = rng.uniform(0.05, 1.0, size=(m, c))
        p[:, :, 3] = rng.uniform(1, 8, size=(m, c))
        p[:, :, 4] = rng.uniform(0.05, 1.0, size=(m, c))
        p[:, :, 5] = rng.randint(0, 4096, size=(m, c))
        if i % 5 == 2 and m:
            p[:, rng.randint(1, c), :] = 0                      # an unset joint: all six columns zero
        out.append(p)
    return out


def test_constructions_reach_their_regimes():
    """No GPU: on synthetic integer poses the constructions reach every limit, the numpy model of
    coco_joint equals the reference's loops (and results.coco_results) bit for bit, and every value
    mutant of the epilogue changes some row."""
    rng = np.random.RandomState(812)
    poses = _synthetic_poses(rng, 30)
    frames, names = _frames_for(poses, 7)
    assert {n for n, _, _ in _families()} <= set(names) and {'unset0', 'unset+'} <= set(names)
    metas = _metas(frames)
    ref = _reference(poses, metas)
    model = _model_rows(poses, frames)
    assert _same(model[0], ref[0]) and _same(model[1], ref[1]) and np.array_equal(model[2], ref[2])
    host = _rows_as_arrays(*results.coco_results(poses, metas)[:2])
    assert _same(host[0], ref[0]) and _same(host[1], ref[1])
    seen = _regimes(poses, frames)
    assert REGIMES <= seen, sorted(REGIMES - seen)
    # each steering family reaches its own limit on its own images
    for fam in ('cancel', 'div'):
        idx = [i for i, n in enumerate(names) if n == fam]
        sub = _regimes([poses[i] for i in idx], frames[idx])
        assert {'cancel': {'float_add'}, 'div': {'float_divide', 'reciprocal'}}[fam] <= sub, (fam, sub)


def test_float32_ties_are_exact_rational_findings():
    """The float32 product ties are ties only in float32: 0.015f = 0.01499999966... times 100 is 1.5 in
    float32, which rint takes to 2 (0.02), while the float64 product 1.49999996... gives 0.01; numpy's
    around agrees with the float32 form on every value found."""
    v = F32(0.015)
    assert v in _float32_ties()
    assert _round2(v) == F32(0.02) and _round2(v, ('product_f64',)) == F32(0.01)
    for t in _float32_ties():
        assert _round2(t) != _round2(t, ('product_f64',))
        assert np.around(np.array([t, -t], F32), 2).tolist() == [_round2(t), -_round2(t)]


# --------------------------------------------------------------------------- GPU helpers
def _check_rows(rows, poses, metas, c):
    """GPU rows (engine.last_result_rows) against the reference's loops and results.coco_results."""
    assert rows is not None, 'no result rows'
    kp, sc, im = results.result_arrays(rows, c)
    rk, rs, ri = _reference(poses, metas)
    assert len(kp) == len(rk) == sum(max(len(p), 1) for p in poses)
    assert np.array_equal(im, ri), 'image order'
    bad = np.nonzero((_bits(kp) != _bits(rk)).any(axis=1))[0]
    assert bad.size == 0, ('keypoint triples differ', bad[:5], kp[bad[:2]], rk[bad[:2]])
    assert _same(sc, rs), ('scores differ', np.nonzero(_bits(sc) != _bits(rs))[0][:5])
    empty = [i for i, p in enumerate(poses) if len(p) == 0]
    assert all(sc[im == i].tolist() == [0.01] for i in empty)
    hk, hs, hi = _rows_as_arrays(*results.coco_results(poses, metas)[:2])
    assert _same(hk, kp) and _same(hs, sc) and np.array_equal(hi, im)


def _same_poses(a, b):
    return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))


def _engine(c=17, skel=SKEL, **over):
    from offsetguided_b200.engine import DecoderEngine
    kw = dict(KW, **over)
    return DecoderEngine(c, skel, **kw)


def _tables(flip):
    if not flip:
        return None
    return (cfg.heatmap_hflip(cfg.COCO_KEYPOINTS),) + tuple(cfg.offset_hflip(cfg.COCO_KEYPOINTS, SKEL))


@functools.lru_cache(maxsize=None)
def _batch(n, flip, kind='plain'):
    """Network-resolution maps (stride 4) of n images, mirrored copies appended when ``flip``.
    Image 1 holds nobody; images 2 and 3 lack both elbows (unset joints).  ``kind``: 'crowd' puts
    three rendered crowds of 35-60 persons last (their mirrored halves are W-reversed copies),
    'noise' turns one heat-map plane of image 0 into noise: at 160 x 160 its ~5000 peaks overflow the
    candidate list (80 x 80 holds ~1300, which fit)."""
    crowd = kind == 'crowd'
    m = n - 3 if crowd else n
    hmp, omp = _lowres_scene(7100 + n, m, flip, edge={'crowd': 512, 'noise': 640}.get(kind, 320))
    if crowd:
        _, ch, co = _crowd_scenes(scenes.TEMPLATE_COCO)
        halves = [(hmp[:m], omp[:m], ch, co)]
        if flip:
            halves.append((hmp[m:], omp[m:], ch[..., ::-1], co[..., ::-1]))
        hmp = np.concatenate([np.concatenate([a, c_]) for a, _, c_, _ in halves])
        omp = np.concatenate([np.concatenate([b, d]) for _, b, _, d in halves])
    hmp = np.ascontiguousarray(hmp, F32)
    omp = np.ascontiguousarray(omp, F32)
    for half in range(2 if flip else 1):
        hmp[half * n + 1] = 0
        hmp[half * n + 2:half * n + 4, 7:9] = 0
    if kind == 'noise':
        hmp[0, 5] = np.random.RandomState(9).uniform(0, 1, size=hmp.shape[2:]).astype(F32)
    return hmp, omp


ROUTES = {'graph', 'kernels', 'host', 'materialising'}


def _inputs(route, hmp, omp):
    import torch
    h, o = torch.from_numpy(hmp), torch.from_numpy(omp)
    return (h.pin_memory(), o.pin_memory()) if route == 'host' else (h.cuda(), o.cuda())


def _decode(eng, route, maps, flip, frames=None):
    eng.set_graph(route != 'kernels')
    if eng._fused != (route != 'materialising'):
        eng.set_fused(route != 'materialising')
    return eng.decode_features(maps[0], maps[1], 4, 4, 'bicubic', _tables(flip), frames=frames)


PATH_ENV = {'warp': {}, 'cta': {'OG_K3_WARP_ROWS': '0'}, 'warp+cta': {'OG_K3_WARP_ROWS': '8'},
            'regroup': {'OG_RESULT_ROWS': '1'}, 'redo': {}}
PATH_BATCH = {'warp+cta': 'crowd', 'redo': 'noise'}


def _cases():
    out = []
    for path in PATH_ENV:                                   # every grouping path on the graph and host routes
        for route, n in (('graph', 20), ('host', 20)):
            out += [(path, route, n, flip) for flip in (False, True)]
    for path in ('warp', 'cta'):                            # the other routes on both kernels
        out += [(path, 'kernels', 20, False), (path, 'host', 8, True), (path, 'host', 8, False),
                (path, 'materialising', 20, True)]
    return out


# --------------------------------------------------------------------------- A: the limits on the GPU
@pytest.mark.gpu
def test_constructed_rows_on_the_gpu(cuda_device):
    """PostProcess.generate_results on a 26-image batch whose frames were built from its frame-less
    decode: every limit is reached on the decoded poses, every mutant of the model changes a row,
    and the GPU rows equal the reference's loops bit for bit."""
    import torch
    from offsetguided_b200 import decoder
    from test_gpu_parity import _args
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.05, person_thre=0.05, dist_max=40))
    hmp, omp = _batch(26, False)
    feats = [[[torch.from_numpy(hmp).cuda()], [[]], [[]]], [[torch.from_numpy(omp).cuda()], [[]], [[]]]]
    plain = pp.generate_poses(feats)
    assert sum(len(p) for p in plain) > 40
    frames, names = _frames_for(plain, 26)
    assert {n for n, _, _ in _families()} <= set(names), names
    seen = _regimes(plain, frames)
    assert REGIMES <= seen, sorted(REGIMES - seen)
    metas = _metas(frames)
    for _ in range(2):                                       # the second call replays the captured graph
        poses, kp, sc, img = pp.generate_results(feats, metas)
        assert _same_poses(poses, plain)
        eng = pp._engine(torch.device('cuda', 0))
        _check_rows(eng.last_result_rows, poses, metas, 17)
        ref = _reference(poses, metas)
        assert _same(kp, ref[0]) and _same(sc, ref[1]) and np.array_equal(img, ref[2])


# --------------------------------------------------------------------------- B: paths x routes
@pytest.mark.gpu
@pytest.mark.parametrize('path,route,n,flip', _cases())
def test_rows_on_every_grouping_path_and_route(cuda_device, monkeypatch, path, route, n, flip):
    """Frames-less decode, then three decodes with frames (random ones, the constructions, other
    random ones) on a fresh handle: same poses, rows equal to the reference loops.  The warp + CTA
    path runs the CTA kernel at fetch time on single-range calls (k3_redo_count) and eagerly per
    range on host calls of several ranges; the regroup path outgrows a one-row-per-image buffer;
    the redo path overflows a candidate list on every call."""
    for k, v in PATH_ENV[path].items():
        monkeypatch.setenv(k, v)
    hmp, omp = _batch(n, flip, PATH_BATCH.get(path, 'plain'))
    maps = _inputs(route, hmp, omp)
    plain = _decode(_engine(), route, maps, flip)
    assert len(plain) == n and len(plain[1]) == 0
    total = sum(len(p) for p in plain)
    if path == 'regroup':
        assert total > n
    eng = _engine()                                          # its first call is one with frames
    for call, frames in enumerate((_frames_for(plain, 1, False)[0], _frames_for(plain, 2)[0],
                                   _frames_for(plain, 3, False)[0])):
        k3, redo, (replays, builds) = eng.k3_redo_count, eng.fused_redo_count, eng.graph_counts
        poses = _decode(eng, route, maps, flip, frames)
        assert _same_poses(poses, plain), f'call {call}'
        _check_rows(eng.last_result_rows, poses, _metas(frames), 17)
        lazy = route != 'host'                               # host calls here are several ranges
        if path != 'redo':                                   # a noise plane may outgrow the warp kernel too
            assert eng.k3_redo_count - k3 == (1 if path == 'warp+cta' and lazy else 0)
        assert eng.fused_redo_count - redo == (1 if path == 'redo' and route != 'materialising' else 0)
        if route == 'graph' and call == 2:
            assert eng.graph_counts == (replays + 1, builds)
    if path == 'warp+cta':
        assert max(len(p) for p in plain) > 8


@pytest.mark.gpu
@pytest.mark.parametrize('rows', ['64', '0'])
def test_rows_from_full_resolution_maps(cuda_device, monkeypatch, rows):
    """engine.stage_frames + decode_maps on full-resolution chain maps (K1 -> K2 -> K3, one range),
    on the warp kernel and on the CTA kernel alone."""
    import torch
    monkeypatch.setenv('OG_K3_WARP_ROWS', rows)
    counts = [3, 0, 6, 1, 9, 2, 4, 5, 7, 1, 2, 8, 3, 5, 6, 4, 2, 3]
    heat, offs = _chain_maps(counts, 16)
    heat[1::4, 2] = 0                                        # images without joint 2: unset joints
    hd, od = torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda()
    kw = dict(topk=16, thre_hmp=0.06, min_len=0.5, dist_max=40, use_scale=True, person_thre=0.06)
    plain = _engine(5, CHAIN, **kw).decode_maps(hd, od)
    assert [len(p) for p in plain][:3] == [3, 0, 6]
    eng = _engine(5, CHAIN, **kw)
    for seed, constructed in ((4, True), (5, False)):
        frames, names = _frames_for(plain, seed, constructed)
        eng.stage_frames(frames)
        poses = eng.decode_maps(hd, od)
        assert _same_poses(poses, plain)
        _check_rows(eng.last_result_rows, poses, _metas(frames), 5)
    assert {'tie', 'zero', 'unset0'} <= set(_frames_for(plain, 4)[1])


# --------------------------------------------------------------------------- C: the frames' lifecycle
def _device_batch(n=6, flip=True):
    import torch
    hmp, omp = _batch(n, flip)
    return torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()


@pytest.mark.gpu
def test_replayed_graph_rows_follow_each_calls_frames(cuda_device):
    hd, od = _device_batch()
    plain = _engine().decode_features(hd, od, 4, 4, 'bicubic', _tables(True))
    eng = _engine()
    eng.decode_features(hd, od, 4, 4, 'bicubic', _tables(True), frames=_frames_for(plain, 10)[0])
    replays, builds = eng.graph_counts
    for call in range(5):
        frames = _frames_for(plain, 11 + call, constructed=call % 2 == 0)[0]
        poses = eng.decode_features(hd, od, 4, 4, 'bicubic', _tables(True), frames=frames)
        assert _same_poses(poses, plain)
        _check_rows(eng.last_result_rows, poses, _metas(frames), 17)
    assert eng.graph_counts == (replays + 5, builds)


@pytest.mark.gpu
@pytest.mark.parametrize('route', ['graph', 'kernels', 'host'])
def test_rows_only_for_calls_with_frames(cuda_device, route):
    """Frames, none, frames again on the same buffers: rows appear only where frames were staged
    and the poses never change."""
    hmp, omp = _batch(6, True)
    maps = _inputs(route, hmp, omp)
    eng = _engine()
    plain = _decode(eng, route, maps, True)
    for call, staged in enumerate((True, False, True, False, True)):
        frames = _frames_for(plain, 20 + call)[0] if staged else None
        poses = _decode(eng, route, maps, True, frames)
        assert _same_poses(poses, plain)
        if staged:
            _check_rows(eng.last_result_rows, poses, _metas(frames), 17)
        else:
            assert eng.last_result_rows is None


@pytest.mark.gpu
def test_frames_buffers_grow_on_every_slot(cuda_device):
    """Two rounds of 16 calls in flight, one per result slot, the second round with larger batches
    than the first: every slot grows its frames buffer, and every call's rows are its own."""
    from offsetguided_b200 import _lib
    hd, od = _device_batch(32, False)
    ref_eng = _engine()
    sizes = [list(range(1, 17)), list(range(17, 33))]
    plains = {n: ref_eng.decode_features(hd[:n], od[:n], 4, 4, 'bicubic') for s in sizes for n in s}
    eng = _engine()
    for rnd, ns in enumerate(sizes):
        frames = {n: _frames_for(plains[n], 100 * rnd + n, constructed=n % 3 != 0)[0] for n in ns}
        for n in ns:
            assert eng.decode_features(hd[:n], od[:n], 4, 4, 'bicubic', fetch=False, frames=frames[n]) == n
        assert eng.pending == _lib.OG_MAX_IN_FLIGHT
        for n in ns:
            poses = eng.fetch()
            assert _same_poses(poses, plains[n])
            _check_rows(eng.last_result_rows, poses, _metas(frames[n]), 17)


@pytest.mark.gpu
def test_refused_calls_discard_their_frames(cuda_device):
    """A call refused before it runs — by the Python checks, by the library's argument checks, with
    every result slot in flight, or because the frames are for another number of images — drops
    its frames: the next call decodes without rows."""
    import torch
    from offsetguided_b200 import _lib, decoder
    from test_gpu_parity import _args
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.05, person_thre=0.05, dist_max=40))
    hd, od = _device_batch(6, False)
    feats = lambda h_, o_: [[[h_], [[]], [[]]], [[o_], [[]], [[]]]]
    eng = pp._engine(torch.device('cuda', 0))
    plain = pp.generate_poses(feats(hd, od))
    plain4 = pp.generate_poses(feats(hd[:4], od[:4]))
    metas = _metas(_frames_for(plain, 30)[0])

    def unaffected():
        got = pp.generate_poses(feats(hd[:4], od[:4]))           # another image count than the refused call
        assert _same_poses(got, plain4) and eng.last_result_rows is None
        poses, kp, sc, img = pp.generate_results(feats(hd, od), metas)
        assert _same_poses(poses, plain)
        _check_rows(eng.last_result_rows, poses, metas, 17)

    with pytest.raises(ValueError):                             # mismatched heads: refused in Python
        pp.generate_results(feats(hd, od[:, :30]), metas)
    unaffected()
    with pytest.raises(_lib.OgError):                           # heat and offset strides differ: refused by the library
        eng.decode_features(hd, od, 4, 2, 'bicubic', frames=_frames_for(plain, 31)[0])
    unaffected()
    for _ in range(_lib.OG_MAX_IN_FLIGHT):                      # every result slot in flight
        eng.decode_features(hd[:4], od[:4], 4, 4, 'bicubic', fetch=False)
    with pytest.raises(_lib.OgError):
        eng.decode_features(hd, od, 4, 4, 'bicubic', fetch=False, frames=_frames_for(plain, 32)[0])
    for _ in range(_lib.OG_MAX_IN_FLIGHT):
        assert _same_poses(eng.fetch(), plain4) and eng.last_result_rows is None
    unaffected()
    eng.stage_frames(_frames_for(plain, 33)[0][:-1])             # frames for n - 1 images
    with pytest.raises(_lib.OgError, match='staged 5 image frames'):
        eng.decode_features(hd, od, 4, 4, 'bicubic')
    unaffected()
    eng.set_graph(False)
    eng.stage_frames(_frames_for(plain, 34)[0][:-1])
    with pytest.raises(_lib.OgError, match='staged 5 image frames'):
        eng.decode_features(hd, od, 4, 4, 'bicubic')
    unaffected()


@pytest.mark.gpu
@pytest.mark.parametrize('host', [False, True])
def test_empty_batch_has_no_rows(cuda_device, host):
    """generate_results on zero images returns empty arrays, as the reference's loops make no row;
    the next call is unaffected."""
    import torch
    from offsetguided_b200 import decoder
    from test_gpu_parity import _args
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.05, person_thre=0.05, dist_max=40))
    hmp, omp = _batch(6, False)
    h_, o_ = torch.from_numpy(hmp), torch.from_numpy(omp)
    h_, o_ = (h_.pin_memory(), o_.pin_memory()) if host else (h_.cuda(), o_.cuda())
    feats = lambda a, b: [[[a], [[]], [[]]], [[b], [[]], [[]]]]
    poses, kp, sc, img = pp.generate_results(feats(h_[:0], o_[:0]), [])
    assert poses == [] and kp.shape == (0, 51) and kp.dtype == F32 and sc.shape == (0,) and img.shape == (0,)
    assert ro.coco_result_rows([], []) == ([], [])
    plain = pp.generate_poses(feats(h_, o_))
    metas = _metas(_frames_for(plain, 40)[0])
    poses, kp, sc, img = pp.generate_results(feats(h_, o_), metas)
    assert _same_poses(poses, plain)
    _check_rows(pp._engine(torch.device('cuda', 0)).last_result_rows, poses, metas, 17)
