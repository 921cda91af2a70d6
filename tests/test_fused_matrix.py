"""The fused network-resolution path (K1f) over its whole template matrix, and the selection at
the limits of its candidate lists.

K1f streams the network-resolution heat maps once (`amax_scan_kernel`: vector loads when the
rows, the base pointer and the image stride allow them, scalar loads otherwise), lists the work
blocks that can hold a candidate (`block_list_kernel`) and interpolates + NMS-tests only those
(`fused_block_kernel<T, S, kCubic, kFlip>`); `select_topk_kernel` ranks each plane's candidate
list (one warp up to 128 candidates, the whole CTA up to 2048, more raise the overflow flag and the
plane is materialised and selected exactly when the call is fetched).  Every element type,
scale, resize mode, flip setting and input layout is decoded here and compared with the
materialising path on dense float32 copies and with the oracles.

The heat maps carry, besides rendered persons, constructions that only a correct kernel decodes:
  * spikes on both sides of work-block boundaries and a plateau across one;
  * a ring of -1 cells around a zero interior: bicubic overshoot gives peaks of about 0.22
    although no cell is positive (the activity scan must test |cell|);
  * a checkerboard of 2 x 2 tiles of +-1/32: bicubic peaks above thre = 0.05 from cells all
    below it (the scan's limit must be thre / 1.95, not thre);
  * probes for the 4-cell vector loads: a short wall of -1 cells on a block boundary (its
    overshoot peak lies in the block to the left, flagged only through the wall's halo) and
    dipoles (+v, -v) inside one 4-cell group, which cancel when the mirrored copy of a
    flip-test is paired with the wrong lane.
`test_constructions_reach_their_regimes` proves on the CPU, with a numpy model of the scan, that
each construction does what it is there for.  The selection boundaries use "L" shapes of three
cells, each of which leaves exactly one NMS survivor, to put exact candidate counts (0, 1, 127,
128, 129, 2047, 2048, 2049) into planes."""
import functools

import numpy as np
import pytest

import golden_io as gio
from oracle import c_oracle as co
from oracle import ref_oracle as ro
from oracle import scenes
from offsetguided_b200 import config as cfg

RTOL = 1e-5
THRE = 0.05
TOPK = 32
SKEL = cfg.COCO_PERSON_SKELETON
KP = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
FL, RS = cfg.offset_hflip(cfg.COCO_KEYPOINTS, SKEL)
C, L2 = 17, 2 * len(SKEL)
KSUB = 4                          # cells per vector load of the activity scan
BLOCK_H = 8                       # cell rows of a work block
CAND_CAP = 2048                   # candidate-list capacity of a plane
SMALL_CAND = 128                  # candidates one warp of the selection ranks
DTYPES = ('f32', 'bf16', 'f16')
LAYOUTS = ('dense', 'odd', 'packed_shift', 'packed_stride', 'packed_aligned')
SHAPES = {'dense': (40, 48), 'odd': (37, 47)}
# construction channels (the persons keep channels 0 - 11)
SPIKES, PROBES, RING, CHECKER = 12, 13, 15, 16


def _itemsize(dtype):
    return 4 if dtype == 'f32' else 2


def _torch_dtype(dtype):
    import torch
    return {'f32': torch.float32, 'bf16': torch.bfloat16, 'f16': torch.float16}[dtype]


# --------------------------------------------------------------------------- layouts
def _layout_geometry(layout, h, w):
    """(element offset of the heat view in its buffer, image stride in elements) of a layout in
    which heat and offsets are views of one buffer, the heat after the offsets.  `dense` and
    `odd` are separate contiguous tensors: offset 0, stride C * h * w."""
    hw = h * w
    if layout in ('dense', 'odd'):
        return 0, C * hw
    if layout == 'packed_shift':          # heat starts 3 cells past a 4-cell boundary
        return L2 * hw + 3, (C + L2) * hw + 4
    if layout == 'packed_stride':         # image stride 2 cells past a multiple of 4
        return L2 * hw, (C + L2) * hw + 2
    return L2 * hw, (C + L2) * hw          # packed_aligned


def scan_uses_vector_loads(w, heat_byte_addr, img_stride, itemsize):
    """og_fused.cu launch_fused_t: the activity scan loads 4 cells at once when rows are whole
    4-cell groups, the base pointer is aligned to the load size and so is every image."""
    vec_bytes = KSUB * itemsize
    return w % KSUB == 0 and heat_byte_addr % vec_bytes == 0 and (img_stride * itemsize) % vec_bytes == 0


def _expected_vector(layout, h, w, dtype):
    """The predicate for a layout, for a buffer that starts on a 256-byte boundary (every CUDA
    allocation does)."""
    off, stride = _layout_geometry(layout, h, w)
    return scan_uses_vector_loads(w, off * _itemsize(dtype), stride, _itemsize(dtype))


def _device_views(hmp, omp, layout, dtype):
    """Heat and offset maps of `layout` on the GPU, in `dtype`, holding hmp / omp rounded to it."""
    import torch
    n, _, h, w = hmp.shape
    td = _torch_dtype(dtype)
    if layout in ('dense', 'odd'):
        return torch.from_numpy(hmp).cuda().to(td), torch.from_numpy(omp).cuda().to(td)
    off, stride = _layout_geometry(layout, h, w)
    buf = torch.zeros(n * stride + 8, dtype=td, device='cuda')
    hv = torch.as_strided(buf, (n, C, h, w), (stride, h * w, w, 1), off)
    ov = torch.as_strided(buf, (n, L2, h, w), (stride, h * w, w, 1), 0)
    hv.copy_(torch.from_numpy(hmp).to(td))
    ov.copy_(torch.from_numpy(omp).to(td))
    return hv, ov


# --------------------------------------------------------------------------- content
def _spike_and_plateau_plane(rng, h, w, bw):
    """Spikes on both sides of every work-block boundary (dyadic values, exact in bf16 and f16)
    and a 2-cell plateau across a vertical boundary."""
    p = np.zeros((h, w), np.float32)
    for by in range(BLOCK_H, h, BLOCK_H):
        for bx in range(bw, w, bw):
            if rng.rand() < 0.6:
                y = by - 1 if rng.rand() < 0.5 else by
                x = bx - 1 if rng.rand() < 0.5 else bx
                p[y, x] = rng.randint(20, 64) / np.float32(64)
    p[0, 0], p[h - 1, w - 1] = 0.75, 0.625
    y = 2 * BLOCK_H + 4
    p[y, bw - 1:bw + 1] = 0.625
    return p


def _probe_plane(h, w, bw):
    """Constructions aimed at the lane order of the 4-cell vector loads, one per block row so that
    no other hot cell flags their blocks:
      block row 0: a wall of three -1 cells in column bw (a block boundary, lane 0 of its group);
                   the bicubic overshoot peak left of it lies in the block before, which only the
                   wall's 2-cell halo flags;
      block row 2: a dipole +v, -v in lanes 0 and 1 of one group (v = 1/2);
      block row 4: a dipole +v, -v in lanes 0 and 3 of one group.
    A flip-test whose mirrored copy is paired with the wrong lane averages +v with -v there."""
    p = np.zeros((h, w), np.float32)
    p[2:5, bw] = -1.0
    x0 = 4 * (w // 8)
    p[2 * BLOCK_H + 3, x0], p[2 * BLOCK_H + 3, x0 + 1] = 0.5, -0.5
    if h > 4 * BLOCK_H + 3:
        p[4 * BLOCK_H + 3, x0 - 4], p[4 * BLOCK_H + 3, x0 - 1] = 0.5, -0.5
    return p


def _ring_plane(h, w):
    """-1 cells on the border of a 9 x 9 square, zeros inside and outside."""
    p = np.zeros((h, w), np.float32)
    y0, x0 = 10, 12
    p[y0:y0 + 9, x0:x0 + 9] = -1.0
    p[y0 + 1:y0 + 8, x0 + 1:x0 + 8] = 0.0
    return p


def _checker_plane(h, w):
    """2 x 2 tiles of +-1/32 in a checkerboard: the signs follow the bicubic weights' signs, so
    interpolated peaks reach 1.64 (S = 2) to 1.87 (S = 8) times the cells."""
    p = np.zeros((h, w), np.float32)
    yy, xx = np.mgrid[0:h, 0:w]
    sign = np.where(((yy // 2) + (xx // 2)) % 2 == 0, 1.0, -1.0)
    inside = (yy >= 4) & (yy < h - 4) & (xx >= 4) & (xx < w - 4)
    p[inside] = (sign[inside] / 32.0).astype(np.float32)
    return p


@functools.lru_cache(maxsize=None)
def matrix_inputs(h, w, scale, flip):
    """(hmp, omp) float32 at network resolution, 2 images (+ their mirrored copies with flip).
    Persons are rendered for a stride-4 network; the flipped half holds the exact mirror of the
    original half plus its own noise on the persons' channels, so the flip-fused construction
    channels equal the originals."""
    n = 2
    bw = 32 // scale
    W, H = 4 * w, 4 * h
    hs, os_ = [], []
    for i in range(n):
        rng = np.random.RandomState(1000 * h + 10 * scale + i)
        p = scenes.make_persons(rng, 3, W, H, scale_range=(W / 48.0, W / 30.0))
        hm = scenes.render_heatmaps(p, W, H) + rng.uniform(0, 0.02, size=(C, h, w)).astype(np.float32)
        hm[SPIKES] = _spike_and_plateau_plane(rng, h, w, bw)
        hm[PROBES] = _probe_plane(h, w, bw)
        hm[14] = 0.0                       # the probes' mirrored partner: empty
        hm[RING] = _ring_plane(h, w)
        hm[CHECKER] = _checker_plane(h, w)
        om = scenes.render_offsets(p, W, H, SKEL)
        om[~np.isfinite(om)] = 0
        hs.append(hm)
        os_.append(om)
    hmp, omp = np.stack(hs), np.stack(os_)
    if flip:
        rng = np.random.RandomState(h + w + scale)
        mh = np.empty_like(hmp)
        mh[:, KP] = hmp[:, :, :, ::-1]
        for c in range(SPIKES):
            mh[:, KP[c]] += rng.uniform(0, 0.02, size=(n, h, w)).astype(np.float32)
        mo = rng.uniform(-6, 6, size=omp.shape).astype(np.float32)
        hmp, omp = np.concatenate((hmp, mh)), np.concatenate((omp, mo))
    return hmp.astype(np.float32), omp.astype(np.float32)


def _fused_heat(hmp, flip):
    """The flip-fused heat maps as the reference computes them."""
    if not flip:
        return hmp
    n = hmp.shape[0] // 2
    return ((hmp[:n] + hmp[n:, :, :, ::-1][:, KP]) * np.float32(0.5)).astype(np.float32)


def oracle_dets(heat_lo, scale, mode, k):
    """Top-K of the thresholded NMS map of the resized maps: (scores, indices, full-res NMS map)."""
    nms = ro.hmp_nms(co.resize(heat_lo, scale, mode))
    cut = nms.copy()
    cut[cut < np.float32(THRE)] = -1.0
    s, i, _, _ = ro.topk_channel(cut, k)
    return s, i, nms


# --------------------------------------------------------------------------- scan model
def scan_flags(a, b, scale, mode, variant='exact'):
    """numpy model of amax_scan_kernel's vector path for one plane: the work blocks it flags.
    `a` is the plane, `b` the mirrored partner plane of a flip-test (None without flip).
    `variant` models a kernel defect:
      'no_abs'   the scan tests v instead of |v|;
      'limit'    the scan's limit is thre instead of thre / 1.95 (bicubic) or thre / 1.001;
      'lanes01'  lanes 0 and 1 of each 4-cell load swapped (both inputs);
      'halves'   the two 2-cell halves of each 4-cell load swapped (both inputs);
      'mirror'   the mirrored copy's lanes 0 and 3 paired with the wrong cells."""
    h, w = a.shape
    cubic = mode == 'bicubic'
    halo = 2 if cubic else 1
    limit = np.float32(THRE) if variant == 'limit' else np.float32(THRE / (1.95 if cubic else 1.001))
    perm = {'lanes01': (1, 0, 2, 3), 'halves': (2, 3, 0, 1)}.get(variant, (0, 1, 2, 3))
    g = a.reshape(h, w // KSUB, KSUB)
    va = g[:, :, list(perm)]
    if b is None:
        f = va
    else:
        # vb[i] = b[w - 4 - x0 + perm[i]]: the mirrored group, in load order
        gb = b[:, ::-1].reshape(h, w // KSUB, KSUB)[:, :, ::-1]        # gb[.., x0 / 4, i] = b[w - 4 - x0 + i]
        vb = gb[:, :, list(perm)]
        pair = (0, 2, 1, 3) if variant == 'mirror' else (3, 2, 1, 0)
        f = ((va + vb[:, :, list(pair)]) * np.float32(0.5)).astype(np.float32)
    f = f.reshape(h, w)
    hot = (f >= limit) if variant == 'no_abs' else ~(np.abs(f) < limit)
    bw = 32 // scale
    bxs, bys = (w + bw - 1) // bw, (h + BLOCK_H - 1) // BLOCK_H
    flags = np.zeros((bys, bxs), bool)
    for y, x in zip(*np.nonzero(hot)):
        flags[max(y - halo, 0) // BLOCK_H:min((y + halo) // BLOCK_H, bys - 1) + 1,
              max(x - halo, 0) // bw:min((x + halo) // bw, bxs - 1) + 1] = True
    return flags


def lost_topk(hmp, scale, mode, flip, variant, channels):
    """Oracle top-K dets of `channels` that lie in blocks the modelled scan `variant` leaves
    unflagged (the dets a kernel with that defect would lose)."""
    n = hmp.shape[0] // 2 if flip else hmp.shape[0]
    fused = _fused_heat(hmp, flip)
    s, i, _ = oracle_dets(fused[:, channels], scale, mode, TOPK)
    W = hmp.shape[3] * scale
    bw = 32 // scale
    lost = 0
    for img in range(n):
        for j, c in enumerate(channels):
            b = hmp[n + img, KP[c]] if flip else None
            flags = scan_flags(hmp[img, c], b, scale, mode, variant)
            for sc, idx in zip(s[img, j], i[img, j]):
                if sc >= np.float32(THRE) and not flags[(idx // W) // scale // BLOCK_H, (idx % W) // scale // bw]:
                    lost += 1
    return lost


# --------------------------------------------------------------------------- L shapes
def l_plane(h, w, count, rng, spacing=6):
    """A plane holding `count` L shapes (a, a / 2 to its right, a / 4 below), spaced `spacing`
    cells apart on a grid; amplitudes are multiples of 1/16 in [1/2, 1), exact in bf16 and f16,
    and repeat, so equal peaks are ranked by their index."""
    p = np.zeros((h, w), np.float32)
    sites = [(y, x) for y in range(2, h - 3, spacing) for x in range(2, w - 3, spacing)]
    assert count <= len(sites), (count, len(sites))
    for (y, x) in [sites[j] for j in rng.permutation(len(sites))[:count]]:
        a = np.float32(rng.randint(8, 16) / 16.0)
        p[y, x], p[y, x + 1], p[y + 1, x] = a, a / 2, a / 4
    return p


L_COUNTS = [2049, 0, 1, 127, 128, 129, 2, 5, 2048, 1, 128, 129, 2047, 0, 127, 3, 64]
L_SHAPE = (256, 320)            # 2226 grid sites of 6 x 6 cells


@functools.lru_cache(maxsize=None)
def l_inputs(counts):
    rng = np.random.RandomState(sum(counts) % 1000)
    h, w = L_SHAPE
    return np.stack([l_plane(h, w, c, rng) for c in counts])[None]


def survivors(plane_lo, scale, mode):
    nms = ro.hmp_nms(co.resize(plane_lo[None, None], scale, mode))
    return int((nms >= np.float32(THRE)).sum())


# =========================================================================== CPU
def test_constructions_reach_their_regimes():
    """No GPU.  (1) L shapes leave exactly one NMS survivor each, so the planes hold the intended
    candidate counts (at every scale and mode for small planes, at S = 4 bicubic for the planes
    of the boundary test); (2) the ring and the checkerboard give bicubic survivors >= thre while
    every cell is below thre; (3) the vector / scalar scan choice of every layout, both reached by
    every element type (the matrix runs each layout with and without flip); (4) the numpy model of the scan loses
    top-K dets of the construction channels under each modelled defect and none when exact."""
    rng = np.random.RandomState(0)
    for scale in (2, 4, 8):
        for mode in ('bicubic', 'bilinear'):
            for count in (0, 1, 7, 30):
                assert survivors(l_plane(40, 48, count, rng), scale, mode) == count, (scale, mode, count)
    edges = {0, 1, SMALL_CAND - 1, SMALL_CAND, SMALL_CAND + 1, CAND_CAP - 1, CAND_CAP, CAND_CAP + 1}
    assert edges <= set(L_COUNTS)
    big = l_inputs(tuple(L_COUNTS))[0]
    nms = ro.hmp_nms(co.resize(big[None], 4, 'bicubic'))[0]
    assert [int((p >= np.float32(THRE)).sum()) for p in nms] == L_COUNTS

    for scale in (2, 4, 8):
        h, w = SHAPES['dense']
        for plane in (_ring_plane(h, w), _checker_plane(h, w)):
            assert np.abs(plane).max() < 1.0 + 1e-6 and plane.max() < THRE
            s = ro.hmp_nms(co.resize(plane[None, None], scale, 'bicubic'))
            assert (s >= np.float32(THRE)).sum() >= 4, scale

    for dtype in DTYPES:
        seen = set()
        for layout in LAYOUTS:
            h, w = SHAPES['odd' if layout == 'odd' else 'dense']
            vec = _expected_vector(layout, h, w, dtype)
            assert vec == (layout in ('dense', 'packed_aligned')), (dtype, layout)
            seen.add(vec)
        assert seen == {True, False}

    for scale in (2, 4, 8):
        for flip in (False, True):
            hmp, _ = matrix_inputs(*SHAPES['dense'], scale, flip)
            for mode in ('bicubic', 'bilinear'):
                assert lost_topk(hmp, scale, mode, flip, 'exact', list(range(C))) == 0
            # tested |v|: only the ring (all cells <= 0) loses its peaks
            assert lost_topk(hmp, scale, 'bicubic', flip, 'no_abs', [RING]) > 0
            assert lost_topk(hmp, scale, 'bicubic', flip, 'limit', [CHECKER]) > 0
            assert lost_topk(hmp, scale, 'bicubic', flip, 'halves', [PROBES]) > 0
            if flip:
                assert lost_topk(hmp, scale, 'bicubic', flip, 'lanes01', [PROBES]) > 0
                assert lost_topk(hmp, scale, 'bicubic', flip, 'mirror', [PROBES]) > 0


# =========================================================================== GPU
def _engine(**over):
    from offsetguided_b200.engine import DecoderEngine
    kw = dict(topk=TOPK, thre_hmp=THRE, min_len=0.5, dist_max=40, use_scale=True, person_thre=THRE)
    kw.update(over)
    return DecoderEngine(C, SKEL, **kw)


def _tables(flip):
    return (KP, FL, RS) if flip else None


def _decode_both(eng, hv, ov, scale, mode, flip, n):
    """Fused decode of the given views, then the materialising path on dense float32 copies:
    (fused poses, fused intermediates, staged poses, staged intermediates)."""
    eng.set_fused(True)
    r0 = eng.fused_redo_count
    fused = eng.decode_features(hv, ov, scale, scale, mode, _tables(flip))
    f_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    redo = eng.fused_redo_count - r0
    eng.set_fused(False)
    staged = eng.decode_features(hv.float().contiguous(), ov.float().contiguous(), scale, scale, mode, _tables(flip))
    s_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    eng.set_fused(True)
    return fused, f_int, staged, s_int, redo


def _assert_same(fused, f_int, staged, s_int):
    for a, b in zip(f_int, s_int):
        assert np.array_equal(a, b)
    assert len(fused) == len(staged)
    for a, b in zip(fused, staged):
        assert np.array_equal(a, b)


def _assert_dets_equal_oracle(ds, di, ref_s, ref_i):
    live = ref_s >= np.float32(THRE)
    assert np.array_equal(di[live], ref_i[live]) and np.array_equal(ds[live], ref_s[live])
    assert np.all(di[~live] == -1)


@functools.lru_cache(maxsize=None)
def _matrix_oracle(dtype, h, w, scale, mode, flip):
    """Oracle results on the widened maps of a matrix case (shared by the layouts of one shape)."""
    import torch
    hmp, omp = matrix_inputs(h, w, scale, flip)
    td = _torch_dtype(dtype)
    wh = torch.from_numpy(hmp).to(td).float().numpy()
    wo = torch.from_numpy(omp).to(td).float().numpy()
    fused = _fused_heat(wh, flip)
    s, i, nms = oracle_dets(fused, scale, mode, TOPK)
    poses = co.generate_poses(wh, wo, SKEL, C, topk=TOPK, thre_hmp=THRE, min_len=0.5, person_thre=THRE,
                              dist_max=40.0, use_scale=True, hmp_stride=scale, off_stride=scale,
                              resize_mode=mode, flip_test=flip, kp_flips=KP, limb_flips=FL, limb_reserve=RS)
    return s, i, fused, poses


@pytest.mark.gpu
@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('mode', ['bicubic', 'bilinear'])
@pytest.mark.parametrize('scale', [2, 4, 8])
@pytest.mark.parametrize('dtype', DTYPES)
def test_fused_instantiation_matrix(cuda_device, dtype, scale, mode, flip, layout):
    """One case per fused_block_kernel<T, S, kCubic, kFlip> x scan variant: dets, limbs and poses
    equal the materialising path on dense float32 copies bit for bit, dets equal the oracle's
    top-K exactly, poses the C oracle's; the ring and checkerboard channels (bicubic) produce
    dets >= thre from cells all below thre."""
    h, w = SHAPES['odd' if layout == 'odd' else 'dense']
    hmp, omp = matrix_inputs(h, w, scale, flip)
    n = hmp.shape[0] // 2 if flip else hmp.shape[0]
    hv, ov = _device_views(hmp, omp, layout, dtype)
    vec = scan_uses_vector_loads(w, hv.data_ptr(), hv.stride(0), hv.element_size())
    assert vec == _expected_vector(layout, h, w, dtype)
    eng = _engine()
    fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, scale, mode, flip, n)
    assert redo == 0
    _assert_same(fused, f_int, staged, s_int)
    ref_s, ref_i, fused_lo, ref_poses = _matrix_oracle(dtype, h, w, scale, mode, flip)
    ds, di, _ = f_int
    _assert_dets_equal_oracle(ds, di, ref_s, ref_i)
    assert len(fused) == len(ref_poses)
    for p, r in zip(fused, ref_poses):
        gio.compare_poses(p, r, rtol=RTOL)
    assert sum(len(p) for p in fused) >= 1
    assert (ds[:, SPIKES] >= THRE).sum() >= 4 and (ds[:, PROBES] >= THRE).sum() >= 2
    if mode == 'bicubic':
        for c in (RING, CHECKER):
            assert np.abs(fused_lo[:, c]).max() <= 1.0 and fused_lo[:, c].max() < THRE
            assert (ds[:, c] >= THRE).all(axis=-1).any(), c          # a full top-K list from sub-threshold cells
    eng.close()


# --------------------------------------------------------------------------- overflow redo
@pytest.mark.gpu
@pytest.mark.parametrize('scale', [2, 4, 8])
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('dtype', DTYPES)
def test_overflow_redo_per_dtype(cuda_device, dtype, flip, scale):
    """One noise plane in a clean batch overflows its candidate list: the fetch redoes that plane
    alone (fuse_planes_kernel<T>, resize, radix selection) and the call equals the materialising
    path on float32 copies."""
    import bench
    import torch
    hmp, omp = bench.lowres_inputs(606 + scale, 2, 640, flip)
    rng = np.random.RandomState(scale)
    hmp[1, 6] = rng.uniform(0, 1, size=hmp.shape[2:]).astype(np.float32)
    omp[~np.isfinite(omp)] = 0
    td = _torch_dtype(dtype)
    hv, ov = torch.from_numpy(hmp).cuda().to(td), torch.from_numpy(omp).cuda().to(td)
    eng = _engine()
    fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, scale, 'bicubic', flip, 2)
    assert redo == 1
    _assert_same(fused, f_int, staged, s_int)
    assert sum(len(p) for p in fused) >= 4 and (f_int[0][1, 6] > 0).all()
    eng.close()


@pytest.mark.gpu
def test_overflow_redo_in_several_groups(cuda_device):
    """2 images x 17 noise planes of 512 x 512 at S = 4: 34 overflowed planes of 2048 x 2048,
    redone 16 per group (256 MB of full-resolution planes), in three groups.  Every plane equals
    the materialising path, and a few the C oracle."""
    import torch
    rng = np.random.RandomState(17)
    hmp = rng.uniform(0, 1, size=(2, C, 512, 512)).astype(np.float32)
    omp = rng.uniform(-8, 8, size=(2, L2, 512, 512)).astype(np.float32)
    hv, ov = torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()
    eng = _engine()
    fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, 4, 'bicubic', False, 2)
    assert redo == 1
    _assert_same(fused, f_int, staged, s_int)
    ds, di, _ = f_int
    assert (ds > 0).all()
    for img, c in ((0, 0), (0, 15), (1, 0), (1, 16)):
        s, i, _ = oracle_dets(hmp[img:img + 1, c:c + 1], 4, 'bicubic', TOPK)
        assert np.array_equal(di[img, c], i[0, 0]) and np.array_equal(ds[img, c], s[0, 0]), (img, c)
    del hv, ov
    eng.close()


@pytest.mark.gpu
def test_host_flip_overflow_in_last_range(cuda_device):
    """Host API, flip-test, 16 images over four image ranges: a noise plane in the last image
    (its mirrored partner in the last image of the flipped half) overflows; the call equals the
    device-maps call on the materialising path."""
    import bench
    import torch
    n = 16
    hmp, omp = bench.lowres_inputs(2468, n, 640, True)
    rng = np.random.RandomState(3)
    hmp[n - 1, 4] = rng.uniform(0, 1, size=hmp.shape[2:]).astype(np.float32)
    hmp[2 * n - 1, KP[4]] = rng.uniform(0, 1, size=hmp.shape[2:]).astype(np.float32)
    th, to = torch.from_numpy(hmp), torch.from_numpy(omp)
    eng = _engine()
    r0 = eng.fused_redo_count
    got = eng.decode_features(th.pin_memory(), to.pin_memory(), 4, 4, 'bicubic', _tables(True))
    g_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    assert eng.fused_redo_count - r0 == 1
    eng.set_fused(False)
    ref = eng.decode_features(th.cuda(), to.cuda(), 4, 4, 'bicubic', _tables(True))
    r_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    _assert_same(got, g_int, ref, r_int)
    assert (g_int[0][n - 1, 4] > 0).all() and sum(len(p) for p in got) >= n * 3
    eng.close()


# --------------------------------------------------------------------------- candidate counts
@pytest.mark.gpu
def test_candidate_count_boundaries(cuda_device):
    """Planes with exactly 0, 1, 127, 128, 129, 2047, 2048 and 2049 candidates, small planes in the
    same select CTA as big ones.  Fused path: only the call whose image holds the 2049-candidate
    plane redoes it; dets equal the materialising path and the oracle.  K1 on the oracle's
    full-resolution maps lists the same counts."""
    import torch
    lo_a = l_inputs(tuple(L_COUNTS))
    counts_b = tuple(2048 if c == 2049 else c for c in L_COUNTS[::-1])
    lo_b = l_inputs(counts_b)
    eng = _engine()
    for lo, redo_want in ((lo_a, 1), (lo_b, 0), (np.concatenate((lo_b, lo_a)), 1)):
        n = lo.shape[0]
        hv = torch.from_numpy(lo).cuda()
        ov = torch.zeros((n, L2) + lo.shape[2:], device='cuda')
        fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, 4, 'bicubic', False, n)
        assert redo == redo_want
        _assert_same(fused, f_int, staged, s_int)
        ref_s, ref_i, nms = oracle_dets(lo, 4, 'bicubic', TOPK)
        _assert_dets_equal_oracle(f_int[0], f_int[1], ref_s, ref_i)
        # K1's own candidate lists on the full-resolution maps
        s, i, cnt = eng.nms_topk(torch.from_numpy(co.resize(lo, 4, 'bicubic')).cuda())
        assert np.array_equal(cnt.cpu().numpy(), np.minimum((nms >= np.float32(THRE)).sum(axis=(2, 3)), TOPK))
        _assert_dets_equal_oracle(s.cpu().numpy(), i.cpu().numpy(), ref_s, ref_i)
    eng.close()


@pytest.mark.gpu
def test_topk_channel_large_k(cuda_device):
    """decoder.topK_channel beyond the 128-candidate warp path and up to the 2048 limit, and with
    K = H * W on a small map, against the oracle (ties by index)."""
    import torch
    from offsetguided_b200 import decoder
    rng = np.random.RandomState(21)
    big = (rng.randint(0, 64, size=(1, 3, 96, 128)) / np.float32(64)).astype(np.float32)
    small = rng.uniform(-1, 1, size=(2, 2, 9, 11)).astype(np.float32)
    small[0, 1, 2:5, 3:6] = 0.25
    for maps, ks in ((big, (129, 2048)), (small, (99,))):
        for k in ks:
            ts, ti, ty, tx = decoder.topK_channel(torch.from_numpy(maps).cuda(), K=k)
            rs, ri, ry, rx = ro.topk_channel(maps, k)
            assert np.array_equal(ti.cpu().numpy(), ri) and np.array_equal(ts.cpu().numpy(), rs), k
            assert np.array_equal(ty.cpu().numpy(), ry) and np.array_equal(tx.cpu().numpy(), rx), k
