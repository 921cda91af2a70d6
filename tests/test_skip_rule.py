"""The fused path's skip rule at its limits.

K1f's activity scan (`amax_scan_kernel` for planar maps, `amax_scan_nhwc_kernel` for channels-last
maps) flags a work block only when a network-resolution cell within the tap halo of the block
(2 cells bicubic, 1 bilinear: `scan_halo`) reaches |v| >= thre / 1.95 (bicubic) or thre / 1.001
(bilinear: `scan_limit`); unflagged blocks are never interpolated.  Two constructions pin both
constants of that rule:

  A  outer ring: every cell of a block and of its inner ring (Chebyshev distance < halo) is at
     most 3/128 in magnitude (below thre / 1.95 at thre = 0.05), yet a pixel in the block's corner
     cell is an NMS peak >= thre, reached only through the outer ring (distance = halo).  A scan whose
     halo is one cell short never interpolates that block.  The cells come from a linear program
     over the exact tap weights (`derive_outer_ring`), rounded and committed as `A_CELLS`; each is
     mirrored to all four corners of a block, which puts hot cells on both sides of the 4-cell
     load groups and the peak (bicubic, and bilinear at S = 2) on lane 0 or lane 31 of the block
     kernel, next to the ring pixels it evaluates on demand.
  B  tight bound: a 4 x 4 bicubic checker patch of +-1/32 whose interpolated peak is r_S / 32,
     r_S the largest ratio of an interpolated NMS peak to max |cell| (1.6416 / 1.8267 / 1.8745 for
     S = 2 / 4 / 8), decoded with thre set to that peak: a limit of thre / f with f < r_S loses it.
     Bilinear: a 2 x 2 plateau of 1/16 at thre = 1/16, lost by any limit above thre.

Every plane holds fewer survivors than K = 128, so the decoder's dets are the oracle's complete
thresholded candidate set: a lost candidate cannot hide behind the top-K cut or the overflow redo.
`test_constructions_pin_the_skip_rule` proves on the CPU, with a numpy model of the scan, that the
exact rule loses nothing and each defect loses every construction's peak; the GPU matrix decodes
them with every element type, scale, resize mode, flip setting and activity scan."""
import functools

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import ref_oracle as ro
from test_fused_matrix import (BLOCK_H, C, DTYPES, FL, KP, L2, RS, _assert_same, _decode_both, _device_views,
                               _engine, _torch_dtype, oracle_dets, scan_flags, scan_uses_vector_loads)

THRE = 0.05
TOPK = 128                        # the largest top-K: every plane's whole candidate set is listed
SCALES = (2, 4, 8)
MODES = ('bicubic', 'bilinear')
# the largest ratio of an interpolated NMS peak to max |cell| (A = -0.75 bicubic); 1 for bilinear
R_S = {2: 1.6416, 4: 1.8267, 8: 1.8745}
# scan variants: shape (h, w) of the maps; `vector` and `scalar` are planar, `nhwc` channels-last
SCANS = {'vector': (37, 44), 'scalar': (37, 47), 'nhwc': (37, 47)}
CORNERS = ((False, False), (False, True), (True, False), (True, True))   # (mirrored in y, in x)
SITES = ('interior', 'last_col', 'last_row', 'last_both')
MARGIN = 1.0 / 512                # A: the peak beats thre and each of its 8 neighbours by this much


def _halo(mode):
    return 2 if mode == 'bicubic' else 1


# =========================================================================== A: derivation
def _axis_weights(scale, cubic, n):
    """[pixel, cell] interpolation weights of one axis of n cells (ATen's float32 weights)."""
    idx, wts = ro._resize_taps(n, scale, cubic)
    m = np.zeros((n * scale, n))
    for i, w in zip(idx, wts):
        np.add.at(m, (np.arange(n * scale), i), np.broadcast_to(np.asarray(w, np.float64), (n * scale,)))
    return m


def derive_outer_ring(scale, mode):
    """Cells around the top-left corner of a work block, rows and columns -halo .. 2 relative to
    it, the first row and column the outer ring, holding a pixel within the block's first cell
    that is an NMS peak >= thre.  linprog (HiGHS) first maximises the margin m by which the pixel
    beats thre and its 8 neighbours, then minimises sum |cell| at m / 2; the result is rounded to
    multiples of 1/128 within +-3/128 inside and 1/64 outside (1/16 beyond 4, exact in bf16).
    Returns (dy, dx, cells in units of 1/128): the first pixel (by dy + dx) where a peak exists.
    A bilinear peak sits where its four taps change (phase S/2 - 1 at S = 8) and needs the outer
    cell opposite the block at about -6 or below, so S = 8 bilinear gets a bound of 16, not 4."""
    from scipy.optimize import linprog
    cubic = mode == 'bicubic'
    halo = _halo(mode)
    hot_bound = 16.0 if (scale, mode) == (8, 'bilinear') else 4.0
    n, c0 = 16, 8
    m = _axis_weights(scale, cubic, n)[:, c0 - halo:c0 + 3]
    nw = m.shape[1]
    nv = nw * nw
    hot = np.zeros((nw, nw), bool)
    hot[0, :] = hot[:, 0] = True
    cell_bounds = [(-hot_bound, hot_bound) if t else (-3 / 128, 3 / 128) for t in hot.ravel()]

    def solve(y, x, need):
        # variables: cells (nv), |cells| (nv), margin
        p = np.outer(m[y], m[x]).ravel()
        rows, rhs = [], []

        def add(cells, margin, b):
            rows.append(np.concatenate((cells, np.zeros(nv), [margin])))
            rhs.append(b)
        add(-p, 1.0, -THRE)
        for ey in (-1, 0, 1):
            for ex in (-1, 0, 1):
                if ey or ex:
                    add(np.outer(m[y + ey], m[x + ex]).ravel() - p, 1.0, 0.0)
        eye = np.eye(nv)
        a_ub = np.concatenate((np.array(rows), np.block([[eye, -eye, np.zeros((nv, 1))],
                                                         [-eye, -eye, np.zeros((nv, 1))]])))
        b_ub = np.concatenate((rhs, np.zeros(2 * nv)))
        cost = np.zeros(2 * nv + 1)
        if need is None:
            cost[-1] = -1.0
            last = (0.0, 1.0)
        else:
            cost[nv:2 * nv] = 1.0
            last = (need, need)
        r = linprog(cost, A_ub=a_ub, b_ub=b_ub, bounds=cell_bounds + [(0, None)] * nv + [last], method='highs')
        return r.x if r.status == 0 else None

    y0 = c0 * scale
    for dy, dx in sorted(((a, b) for a in range(scale) for b in range(scale)), key=lambda t: (t[0] + t[1], t)):
        r = solve(y0 + dy, y0 + dx, None)
        if r is None or r[-1] <= 1e-6:
            continue
        cells = solve(y0 + dy, y0 + dx, r[-1] / 2)[:nv].reshape(nw, nw)
        step = np.where(hot, np.where(np.abs(cells) > 4, 8, 2), 1)
        units = (np.round(cells * 128 / step) * step).astype(np.int64)
        units[~hot] = np.clip(units[~hot], -3, 3)
        return dy, dx, units
    raise AssertionError('no outer-ring peak for S = %d %s' % (scale, mode))


# (dy, dx, cells in units of 1/128) from derive_outer_ring
A_CELLS = {
    (2, 'bicubic'): (0, 0, np.array([[0, 0, -140, 244, 0], [366, -3, 0, -3, 0], [-118, 0, 3, -3, 0],
                                     [316, -3, -3, 3, 0], [0, 0, 0, 0, 0]])),
    (4, 'bicubic'): (0, 0, np.array([[0, 20, -54, 182, 0], [0, -3, -3, -3, 0], [-50, -3, 3, -3, 0],
                                     [210, -3, -3, 3, 0], [0, 0, 0, 0, 0]])),
    (8, 'bicubic'): (0, 0, np.array([[0, 0, -58, 116, 0], [-14, -3, -3, -3, 0], [-52, -3, 3, -3, 0],
                                     [164, -3, -3, 3, 0], [0, 0, 0, 0, 0]])),
    (2, 'bilinear'): (0, 0, np.array([[-268, 90, -238, 0], [90, 3, 0, 0], [-238, 0, 0, 0], [0, 0, 0, 0]])),
    (4, 'bilinear'): (1, 1, np.array([[-336, 50, -246, 0], [50, 3, -3, 0], [-246, -3, 0, 0], [0, 0, 0, 0]])),
    (8, 'bilinear'): (3, 3, np.array([[-1400, 90, -1000, 0], [90, 3, -3, 0], [-1000, -3, 0, 0], [0, 0, 0, 0]])),
}


# =========================================================================== planes
def _blocks(scale, h, w):
    bw = 32 // scale
    return bw, (w + bw - 1) // bw, (h + BLOCK_H - 1) // BLOCK_H


def _site_block(site, scale, h, w, mirror_y=False, mirror_x=False):
    """Target block (bx, by) of a site.  A construction whose outer ring lies right of (below) the
    block takes the block before the last column (row), its ring then in the last one."""
    _, bxs, bys = _blocks(scale, h, w)
    bx = bxs - 1 if site in ('last_col', 'last_both') else 1
    by = bys - 1 if site in ('last_row', 'last_both') else 1
    if mirror_x:
        bx = min(bx, bxs - 2)
    if mirror_y:
        by = min(by, bys - 2)
    return bx, by


def outer_ring_plane(scale, mode, h, w, site, mirror_y, mirror_x):
    """Construction A at one site and corner: (plane, (Y, X) of its peak pixel, target block)."""
    dy, dx, units = A_CELLS[(scale, mode)]
    cells = units.astype(np.float32) / np.float32(128)
    halo = _halo(mode)
    bw = 32 // scale
    bx, by = _site_block(site, scale, h, w, mirror_y, mirror_x)
    p = np.zeros((h, w), np.float32)
    n = cells.shape[0]
    Y = by * BLOCK_H * scale + dy
    X = bx * 32 + dx
    y_lo, x_lo = by * BLOCK_H - halo, bx * bw - halo
    if mirror_y:                       # mirrored about the block's centre row
        cells = cells[::-1]
        y_lo = (by + 1) * BLOCK_H - 1 + halo - (n - 1)
        Y = (by + 1) * BLOCK_H * scale - 1 - dy
    if mirror_x:
        cells = cells[:, ::-1]
        x_lo = (bx + 1) * bw - 1 + halo - (n - 1)
        X = (bx + 1) * 32 - 1 - dx
    p[y_lo:y_lo + n, x_lo:x_lo + n] = cells
    return p, (Y, X), (bx, by)


def checker_patch():
    """4 x 4 cells of +-1/32: the signs of the A = -0.75 bicubic weights' outer product, negated
    twice.  Its four central pixels reach r_S / 32 at every S."""
    s = np.array([1.0, -1.0, -1.0, 1.0], np.float32)
    return (np.outer(s, s) / np.float32(32)).astype(np.float32)


def tight_plane(scale, mode, h, w, site):
    """Construction B at one site: the checker patch (bicubic), its first cell one cell up and left
    of the target block's first cell, or a 2 x 2 plateau of 1/16 (bilinear) on that first cell;
    either way the peaks lie in the target block."""
    bw = 32 // scale
    bx, by = _site_block(site, scale, h, w)
    p = np.zeros((h, w), np.float32)
    if mode == 'bicubic':
        p[by * BLOCK_H - 1:by * BLOCK_H + 3, bx * bw - 1:bx * bw + 3] = checker_patch()
    else:
        p[by * BLOCK_H:by * BLOCK_H + 2, bx * bw:bx * bw + 2] = np.float32(1.0 / 16)
    return p, (bx, by)


@functools.lru_cache(maxsize=None)
def tight_thre(scale, mode):
    """thre of construction B: the exact oracle peak of the patch (bicubic), 1/16 (bilinear)."""
    if mode == 'bilinear':
        return np.float32(1.0 / 16)
    p = np.zeros((16, 16), np.float32)
    p[6:10, 6:10] = checker_patch()
    return ro.hmp_nms(co.resize(p[None, None], scale, mode)).max()


@functools.lru_cache(maxsize=None)
def skip_inputs(kind, scale, mode, h, w, flip):
    """float32 heat maps [n, C, h, w] of 2 images (+ their mirrored copies with flip) and the
    constructions' records.  kind 'A': channel 4 * corner + site holds construction A at that
    corner and site; kind 'B': channel `site` holds construction B.  Image 1 holds image 0's
    channels in reverse order.  With flip the partner channel KP[c] of the flipped image holds
    the W-mirror of channel c, so the flip-fused planes equal the originals exactly."""
    hm = np.zeros((2, C, h, w), np.float32)
    recs = []
    if kind == 'A':
        for k, (my, mx) in enumerate(CORNERS):
            for j, site in enumerate(SITES):
                p, peak, blk = outer_ring_plane(scale, mode, h, w, site, my, mx)
                hm[0, 4 * k + j] = p
                recs.append((4 * k + j, peak, blk))
    else:
        for j, site in enumerate(SITES):
            p, blk = tight_plane(scale, mode, h, w, site)
            hm[0, j] = p
            recs.append((j, None, blk))
    hm[1] = hm[0, ::-1]
    if flip:
        mh = np.empty_like(hm)
        mh[:, KP] = hm[:, :, :, ::-1]
        hm = np.concatenate((hm, mh))
    return np.ascontiguousarray(hm), tuple(recs)


def _thre(kind, scale, mode):
    return np.float32(THRE) if kind == 'A' else tight_thre(scale, mode)


def _dtype_exact(hm):
    """The cells are exact in every element type."""
    import torch
    return all(np.array_equal(torch.from_numpy(hm).to(_torch_dtype(d)).float().numpy(), hm) for d in DTYPES)


def lost_peaks(hm, scale, mode, flip, thre, variant='exact', factor=None):
    """Oracle survivors >= thre (image, channel, flat index) in the blocks the modelled scan leaves
    unflagged, and all survivors: (lost set, survivor set)."""
    n = hm.shape[0] // 2 if flip else hm.shape[0]
    nms = ro.hmp_nms(co.resize(hm[:n], scale, mode))
    W = hm.shape[3] * scale
    bw = 32 // scale
    lost, every = set(), set()
    for i in range(n):
        for c in range(C):
            flat = np.flatnonzero(nms[i, c] >= thre)
            if flat.size == 0:
                continue
            flags = scan_flags(hm[i, c], hm[n + i, KP[c]] if flip else None, scale, mode, variant, thre, factor)
            for f in flat:
                every.add((i, c, int(f)))
                if not flags[(f // W) // scale // BLOCK_H, (f % W) // scale // bw]:
                    lost.add((i, c, int(f)))
    return lost, every


# =========================================================================== CPU
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('scale', SCALES)
def test_constructions_pin_the_skip_rule(scale, mode):
    """No GPU.  On the cells as every element type holds them, with the C / numpy oracles and the
    numpy model of the activity scan, for every scan shape and flip setting:
      * every plane has fewer than K = 128 survivors >= thre, each construction at least one;
      * A: the designated pixel is a peak >= thre + MARGIN that beats its 8 neighbours by MARGIN,
        in the target block, and the block's cells and inner ring are below thre / 1.95;
      * B: thre is the patch's exact peak, r_S / 32 (bicubic), or 1/16 (bilinear);
      * the exact scan loses nothing; a halo one cell short loses every A peak; a bound factor
        of 0.999 r_S (bilinear: a limit of thre / 0.999) loses every B survivor, while 1.001 r_S
        (bilinear: thre itself) loses none: the bound is tight."""
    if mode == 'bicubic':
        assert abs(float(tight_thre(scale, mode)) * 32 - R_S[scale]) < 1e-4
    for scan, (h, w) in SCANS.items():
        for flip in (False, True):
            for kind in ('A', 'B'):
                hm, recs = skip_inputs(kind, scale, mode, h, w, flip)
                n = 2
                assert _dtype_exact(hm)
                thre = _thre(kind, scale, mode)
                if flip:      # the flip-fused planes are the originals
                    fused = ((hm[:n] + hm[n:, :, :, ::-1][:, KP]) * np.float32(0.5)).astype(np.float32)
                    assert np.array_equal(fused, hm[:n])
                lost, every = lost_peaks(hm, scale, mode, flip, thre)
                assert not lost, (scan, flip, kind)
                counts = np.zeros((n, C), int)
                for i, c, _ in every:
                    counts[i, c] += 1
                assert counts.max() < TOPK
                for c, _, _ in recs:
                    assert counts[0, c] >= 1 and counts[1, C - 1 - c] >= 1, (scan, flip, kind, c)
                if kind == 'A':
                    _check_outer_ring(hm, recs, scale, mode)
                    lost, _ = lost_peaks(hm, scale, mode, flip, thre, 'halo')
                    W = w * scale
                    for c, (Y, X), _ in recs:
                        assert (0, c, Y * W + X) in lost and (1, C - 1 - c, Y * W + X) in lost, (scan, flip, c)
                else:
                    r = R_S[scale] if mode == 'bicubic' else 1.0
                    lost, _ = lost_peaks(hm, scale, mode, flip, thre, factor=0.999 * r)
                    assert lost == every, (scan, flip)
                    lost, _ = lost_peaks(hm, scale, mode, flip, thre, factor=1.001 * r if mode == 'bicubic' else 1.0)
                    assert not lost, (scan, flip)


def _check_outer_ring(hm, recs, scale, mode):
    full = co.resize(hm[:1], scale, mode)[0]
    limit = np.float32(THRE) / np.float32(1.95)
    halo = _halo(mode)
    bw = 32 // scale
    for c, (Y, X), (bx, by) in recs:
        assert (X // 32, Y // (BLOCK_H * scale)) == (bx, by)
        v = full[c, Y, X]
        nb = full[c, Y - 1:Y + 2, X - 1:X + 2].copy()
        nb[1, 1] = -np.inf
        assert v >= THRE + MARGIN and v >= nb.max() + MARGIN, (c, v, nb.max())
        inner = hm[0, c, max(by * BLOCK_H - halo + 1, 0):(by + 1) * BLOCK_H + halo - 1,
                   max(bx * bw - halo + 1, 0):(bx + 1) * bw + halo - 1]
        assert np.abs(inner).max() <= 3.0 / 128 < limit


def test_outer_ring_cells_come_from_the_lp():
    """No GPU.  `derive_outer_ring` reproduces the committed cells of construction A."""
    pytest.importorskip('scipy')
    for (scale, mode), (dy, dx, units) in A_CELLS.items():
        gy, gx, gu = derive_outer_ring(scale, mode)
        assert (gy, gx) == (dy, dx) and np.array_equal(gu, units), (scale, mode)


# =========================================================================== GPU
@pytest.fixture(scope='module')
def engines(cuda_device):
    """Engines by thre, K = 128, made on first use."""
    made = {}

    def get(thre):
        key = float(thre)
        if key not in made:
            made[key] = _engine(topk=TOPK, thre_hmp=key, person_thre=key)
        return made[key]
    yield get
    for e in made.values():
        e.close()


def _views(hm, scan, dtype):
    """Heat maps in `dtype` on the GPU, planar or channels-last, and zero offsets alike."""
    import torch
    from offsetguided_b200.engine import _channels_last_view
    om = np.zeros((hm.shape[0], L2) + hm.shape[2:], np.float32)
    if scan != 'nhwc':
        hv, ov = _device_views(hm, om, 'dense', dtype)
        assert scan_uses_vector_loads(hm.shape[3], hv.data_ptr(), hv.stride(0), hv.element_size()) == (scan == 'vector')
        return hv, ov
    td = _torch_dtype(dtype)
    hv, ov = [torch.from_numpy(a).to(td).cuda().contiguous(memory_format=torch.channels_last) for a in (hm, om)]
    assert _channels_last_view(hv) is not None
    return hv, ov


def _decode_complete(engines, kind, dtype, scale, mode, flip, scan):
    """Decode one construction set fused and materialising: no overflow redo, the two paths equal
    bit for bit, the dets equal the oracle's complete candidate set >= thre.  Returns the dets'
    indices and the constructions' records."""
    h, w = SCANS[scan]
    hm, recs = skip_inputs(kind, scale, mode, h, w, flip)
    n = 2
    hv, ov = _views(hm, scan, dtype)
    thre = _thre(kind, scale, mode)
    fused, f_int, staged, s_int, redo = _decode_both(engines(thre), hv, ov, scale, mode, flip, n)
    assert redo == 0
    _assert_same(fused, f_int, staged, s_int)
    ref_s, ref_i, _ = oracle_dets(hm[:n], scale, mode, TOPK)      # the flip-fused planes are hm[:n]
    live = ref_s >= thre
    assert (live.sum(axis=-1) < TOPK).all()
    ds, di, _ = f_int
    assert np.array_equal(di[live], ref_i[live]) and np.array_equal(ds[live], ref_s[live])
    assert np.all(di[~live] == -1)
    return di, recs


@pytest.mark.gpu
@pytest.mark.parametrize('scan', list(SCANS))
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('scale', SCALES)
@pytest.mark.parametrize('dtype', DTYPES)
def test_outer_ring_peaks(engines, dtype, scale, mode, flip, scan):
    """Construction A at the four corners of interior blocks and of blocks in or next to the last
    partial block column and row: every peak reached only through the outer tap ring is found."""
    di, recs = _decode_complete(engines, 'A', dtype, scale, mode, flip, scan)
    W = SCANS[scan][1] * scale
    for c, (Y, X), _ in recs:
        assert Y * W + X in di[0, c] and Y * W + X in di[1, C - 1 - c], (c, Y, X)


@pytest.mark.gpu
@pytest.mark.parametrize('scan', list(SCANS))
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('scale', SCALES)
@pytest.mark.parametrize('dtype', DTYPES)
def test_tight_bound_peaks(engines, dtype, scale, mode, flip, scan):
    """Construction B decoded at thre = its exact peak (bicubic r_S / 32, bilinear 1/16): the
    peaks, equal to thre, are found in interior blocks and in the last partial column and row."""
    di, recs = _decode_complete(engines, 'B', dtype, scale, mode, flip, scan)
    for c, _, _ in recs:
        assert (di[0, c] >= 0).sum() >= 4 and (di[1, C - 1 - c] >= 0).sum() >= 4, c
