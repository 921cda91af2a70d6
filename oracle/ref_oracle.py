"""TEST INFRASTRUCTURE — CPU restatement (numpy + explicit Python loops) of the
reference's post-network decoding path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module.  The product package never does: it fails loudly
when the CUDA library is missing.

Parity pinning: the reference has no tests or golden vectors for this path
(SURVEY.md 8c), so this oracle is pinned against *outputs of the reference itself*,
produced inside the build container by ``tests/golden/make_golden.py`` (which
imports /root/reference) and committed under ``tests/golden/``;
``tests/test_oracle_golden.py`` replays them.

Documented deviations from the mounted reference source (both from SURVEY.md 8c):
  * ``topk_channel`` uses ``ys = idx // w`` — the reference's ``idx / w``
    (decoder/heatmap.py:47) is integer division only under its pinned torch 1.3.1;
  * where the reference leaves the order of *equal* keys to the library
    (``torch.topk``, ``np.argsort``), the canonical order is
    (value desc, flat index asc) and (limb score desc, row asc).

All citations are relative to /root/reference.
"""
import numpy as np

F32 = np.float32


# --------------------------------------------------------------------------- #
# decoder/heatmap.py
# --------------------------------------------------------------------------- #
def hmp_nms(heat):
    """decoder/heatmap.py:15-35 — zero-pad 1, 3x3 stride-1 max, keep == max.

    heat: (N, C, H, W) float32.  Border pixels see the padded zeros, so a negative
    value on the border is never a peak; plateaus survive entirely."""
    heat = np.asarray(heat, dtype=F32)
    n, c, h, w = heat.shape
    pad = np.zeros((n, c, h + 2, w + 2), dtype=F32)
    pad[:, :, 1:-1, 1:-1] = heat
    hmax = pad[:, :, 0:h, 0:w].copy()
    for dy in range(3):
        for dx in range(3):
            np.maximum(hmax, pad[:, :, dy:dy + h, dx:dx + w], out=hmax)
    return heat * (hmax == heat).astype(F32)


def topk_channel(scores, k):
    """decoder/heatmap.py:38-49 — per-(n, c) top-K over the flattened plane,
    sorted by (value desc, flat index asc).  Returns (scores f32, inds i64,
    ys i64, xs i64), each (N, C, K)."""
    scores = np.asarray(scores, dtype=F32)
    n, c, h, w = scores.shape
    flat = scores.reshape(n * c, h * w)
    out_s = np.zeros((n * c, k), dtype=F32)
    out_i = np.zeros((n * c, k), dtype=np.int64)
    for r in range(n * c):
        row = flat[r]
        kth = np.partition(row, row.size - k)[row.size - k]
        above = np.flatnonzero(row > kth)
        equal = np.flatnonzero(row == kth)[:k - above.size]
        sel = np.concatenate((above, equal))
        order = np.lexsort((sel, -row[sel].astype(np.float64)))
        sel = sel[order]
        out_s[r] = row[sel]
        out_i[r] = sel
    out_s = out_s.reshape(n, c, k)
    out_i = out_i.reshape(n, c, k)
    return out_s, out_i, out_i // w, out_i % w


def joint_dets(hmps, k):
    """decoder/heatmap.py:52-59."""
    return topk_channel(hmp_nms(hmps), k)


# --------------------------------------------------------------------------- #
# decoder/offset.py
# --------------------------------------------------------------------------- #
def pack_jtypes(skeleton):
    """decoder/offset.py:46-51."""
    return [a for a, _ in skeleton], [b for _, b in skeleton]


def _sumpool(x, k):
    """k x k stride-1 sum pooling with zero padding on the last two dims
    (avg_pool2d(divisor_override=1), decoder/offset.py:31-40).  Accumulated in the
    row-major window order ATen's CPU kernel uses."""
    p = (k - 1) // 2
    h, w = x.shape[-2:]
    pad = np.zeros(x.shape[:-2] + (h + 2 * p, w + 2 * p), dtype=F32)
    pad[..., p:p + h, p:p + w] = x
    acc = np.zeros_like(x, dtype=F32)
    for dy in range(k):
        for dx in range(k):
            acc = acc + pad[..., dy:dy + h, dx:dx + w]
    return acc


def scored_offset(hmp, off, jtypes_f, jtypes_t, kernel_size=7):
    """decoder/offset.py:8-43 — heat-weighted local re-averaging of the offsets.
    (n must be >= 2 in the reference, whose squeeze() at :31 drops a batch of 1;
    this restatement accepts any n.)"""
    hmp = np.asarray(hmp, dtype=F32)
    off = np.asarray(off, dtype=F32)
    n, l2, h, w = off.shape
    score = hmp[:, jtypes_f][:, :, None]                       # (n, L, 1, h, w)
    somap = score * off.reshape(n, -1, 2, h, w)                # (n, L, 2, h, w)
    mean_score = _sumpool(score[:, :, 0], kernel_size)         # (n, L, h, w)
    somap_sum = _sumpool(somap.reshape(n, -1, h, w), kernel_size)
    out = somap_sum.reshape(n, -1, 2, h, w) / (mean_score[:, :, None] + F32(1e-6))
    return out.reshape(n, -1, h, w).astype(F32)


# --------------------------------------------------------------------------- #
# decoder/collect.py
# --------------------------------------------------------------------------- #
def channel_dets(dets, jtypes, thresh):
    """decoder/collect.py:247-254 — per-limb candidate tables; candidates with
    score < thresh are moved 100000 px off the image (integer arithmetic)."""
    scores, inds, ys, xs = [d[:, jtypes, :] for d in dets]     # (N, L, K)
    xy = np.stack((xs, ys), axis=-1).astype(np.int64)          # (N, L, K, 2)
    xy[scores < F32(thresh)] -= 100000
    return inds.astype(np.int64), scores.astype(F32), xy.astype(F32)


def _norm2(dx, dy):
    """Tensor.norm(dim=-1) over an (x, y) pair as ATen's CPU kernel evaluates it:
    sqrt(fma(dy, dy, dx*dx)) in float32 (probed bit-for-bit against the reference's
    torch; the fused multiply-add is emulated through float64, whose product of two
    float32 values is exact)."""
    dx = np.asarray(dx, dtype=F32)
    dy = np.asarray(dy, dtype=F32)
    with np.errstate(over='ignore', invalid='ignore'):
        xx = (dx * dx).astype(np.float64)
        return np.sqrt((dy.astype(np.float64) * dy.astype(np.float64) + xx).astype(F32))


def _norm4(a, b, c, d):
    """Tensor.norm over 4 components as ATen's CPU kernel evaluates it (probed): plain
    left-to-right float32 sum of squares, no fused multiply-add."""
    acc = (a * a + b * b).astype(F32)
    acc = (acc + c * c).astype(F32)
    acc = (acc + d * d).astype(F32)
    return np.sqrt(acc)


def generate_limbs(hmps_hr, offs_hr, skeleton, topk, thre_hmp, min_len,
                   hmp_s=4, off_s=4, scmps_hr=None, return_dets=False, jomps_hr=None,
                   use_jitter=True, vector_nd=2):
    """decoder/collect.py:62-236 with include_scale / include_jitter_offset off
    unless ``scmps_hr`` (the scale gather of :111-116, 257-262) / ``jomps_hr`` (jitter offsets,
    :127-138, 158-165, 213-218) are given; ``vector_nd = 4`` is the cat_flip_offs layout.

    Returns limbs (N, L, K, 13) float32 =
    [x1, y1, v1, x2, y2, v2, ind1, ind2, min_dist, len, limb_score, scale1, scale2].
    """
    hmps_hr = np.asarray(hmps_hr, dtype=F32)
    offs_hr = np.asarray(offs_hr, dtype=F32)
    assert hmps_hr.shape[-2:] == offs_hr.shape[-2:], 'spatial resolution should be equal'
    n, c, h, w = hmps_hr.shape
    nl = len(skeleton)
    jf, jt = pack_jtypes(skeleton)
    dets = joint_dets(hmps_hr, topk)                                          # :93
    ind_f, s_f, xy_f = channel_dets(dets, jf, thre_hmp)                       # :100
    ind_t, s_t, xy_t = channel_dets(dets, jt, thre_hmp)                       # :105

    if scmps_hr is not None:                                                  # :111-116
        sc = np.asarray(scmps_hr, dtype=F32).reshape(n, c, h * w)
        scale_f = np.take_along_axis(sc[:, jf], ind_f, axis=-1)
        scale_t = np.take_along_axis(sc[:, jt], ind_t, axis=-1)
    else:                                                                     # :117-122
        scale_f = np.full(s_f.shape, 4, dtype=F32)
        scale_t = np.full(s_t.shape, 4, dtype=F32)

    flat_off = offs_hr.reshape(n, nl, vector_nd, h * w)                       # :143-144
    off_f = np.take_along_axis(flat_off, ind_f[:, :, None, :], axis=-1)       # (N,L,nd,K)
    off_f = np.transpose(off_f, (0, 1, 3, 2))                                 # (N,L,K,nd)
    guid = np.tile(xy_f, (1, 1, 1, vector_nd // 2)) + off_f * F32(off_s / hmp_s)   # :152

    if jomps_hr is not None:                                                  # :127-138
        jm = np.asarray(jomps_hr, dtype=F32)
        jflat = jm.reshape(n, 2, h * w)
        jit_f = np.stack([np.take_along_axis(jflat[:, None, c_], ind_f, axis=-1) for c_ in (0, 1)], -1)
        jit_t = np.stack([np.take_along_axis(jflat[:, None, c_], ind_t, axis=-1) for c_ in (0, 1)], -1)
        if use_jitter:                                                        # :158-165
            assert vector_nd == 2, 'the reference cannot refine 4-D vectors'
            gi = guid.astype(np.int32)                                        # .int(): toward zero
            for i in range(n):
                for j in range(nl):
                    for k in range(topk):
                        gx_, gy_ = int(gi[i, j, k, 0]), int(gi[i, j, k, 1])
                        if 0 <= gx_ < w and 0 <= gy_ < h:
                            guid[i, j, k] += jm[i, :, gx_, gy_]               # [x, y] as [row, col]
    else:
        jit_f = jit_t = None

    xy_t_nd = np.tile(xy_t, (1, 1, 1, vector_nd // 2))
    diff = guid[:, :, :, None, :] - xy_t_nd[:, :, None, :, :]                 # (N,L,K,M,nd)
    if vector_nd == 2:
        dist = _norm2(diff[..., 0], diff[..., 1])                             # :175
    else:
        dist = _norm4(diff[..., 0], diff[..., 1], diff[..., 2], diff[..., 3])
    min_ind = np.argmin(dist, axis=-1)                                        # :177 first index on ties
    min_dist = np.take_along_axis(dist, min_ind[..., None], axis=-1)[..., 0]

    m_s_t = np.take_along_axis(s_t, min_ind, axis=-1)                         # :185-189
    m_xy_t = np.take_along_axis(xy_t, min_ind[..., None], axis=2)
    m_ind_t = np.take_along_axis(ind_t, min_ind, axis=-1)
    m_scale_t = np.take_along_axis(scale_t, min_ind, axis=-1)

    page_f = (np.asarray(jf, dtype=np.int64) * (h * w))[None, :, None]        # :194-199
    page_t = (np.asarray(jt, dtype=np.int64) * (h * w))[None, :, None]
    g_ind_f = ind_f + page_f
    g_ind_t = m_ind_t + page_t

    d = xy_f - m_xy_t                                                         # :204-205
    length = np.maximum(_norm2(d[..., 0], d[..., 1]), F32(min_len))
    limb_score = s_f * m_s_t * np.exp(-min_dist / length)                     # :208

    if jit_f is not None and use_jitter:                                      # :211-218
        m_jit_t = np.take_along_axis(jit_t, min_ind[..., None], axis=2)
        xy_f = xy_f + jit_f
        m_xy_t = m_xy_t + m_jit_t
    limbs = np.stack((xy_f[..., 0], xy_f[..., 1], s_f,
                      m_xy_t[..., 0], m_xy_t[..., 1], m_s_t,
                      g_ind_f.astype(F32), g_ind_t.astype(F32),
                      min_dist, length, limb_score, scale_f, m_scale_t),
                     axis=-1).astype(F32)                                     # :223-233
    if return_dets:
        return limbs, dets
    return limbs


# --------------------------------------------------------------------------- #
# decoder/group.py
# --------------------------------------------------------------------------- #
def valid_limb_rows(conns, dist_max, use_scale):
    """decoder/group.py:64-76 — rows that pass the distance gate and lie strictly
    inside the image (x, y > 0 for both endpoints)."""
    dmax = F32(dist_max)
    rows = []
    for k in range(conns.shape[0]):
        r = conns[k]
        lim = np.maximum(dmax, r[12]) if use_scale else dmax
        if r[8] < lim and r[0] > 0 and r[4] > 0 and r[3] > 0 and r[1] > 0:
            rows.append(k)
    return rows


def delete_reconns(conns, rows):
    """decoder/group.py:222-240 — sort by limb score desc (canonical: stable) and
    keep the best row per distinct to-joint id."""
    rows = sorted(rows, key=lambda k: -float(conns[k, 10]))   # Python sort is stable
    seen, kept = set(), []
    for k in rows:
        t = int(conns[k, 7])
        if t not in seen:
            seen.add(t)
            kept.append(k)
    return kept


def person_score(row, index):
    """decoder/group.py:207-208 — float32 sum over entries > 0 (numpy pairwise
    summation) divided by their float64 count."""
    vals = np.ascontiguousarray(row[row[:, index] > 0, index], dtype=F32)
    with np.errstate(invalid='ignore', divide='ignore'):
        return vals.sum() / np.float64(vals.size)


def group_skeletons(limbs, skeleton, n_keypoints, person_thre, sort_dim=2,
                    dist_max=10, use_scale=False, stats=None, trace=None):
    """decoder/group.py:39-185 for ONE image, written as explicit sequential
    loops so that every numpy fancy-indexing subtlety of the reference is spelled
    out (last write wins, right-hand sides read the pre-update state, mask_sum
    resets only when at least one pair passed, column-sum cancellation).

    ``trace`` (a list) receives one tuple (li, mm, kk, n_new, n_merged) per limb
    step that has kept rows: persons at the start of the step, kept rows, persons
    the step starts and persons it merges away.  The sum of n_new is the number of
    person rows a table that never recycles rows needs.

    limbs: (L, K, 13) float32.  Returns (M, C, 6) float32
    [x, y, v, s, limb_score, ind]."""
    limbs = np.asarray(limbs, dtype=F32)
    assert len(limbs) == len(skeleton), 'check the skeleton config and input limbs Tensor'
    c = n_keypoints
    subset = []                                   # list of (C, 6) float32 rows, unset = -1
    if stats is None:
        stats = {}
    for key in ('case2', 'case1', 'dup_person_write', 'merge', 'share3', 'cancel_new'):
        stats.setdefault(key, 0)

    for li, (jf, jt) in enumerate(skeleton):
        conns = limbs[li]
        kept = delete_reconns(conns, valid_limb_rows(conns, dist_max, use_scale))
        kk, mm = len(kept), len(subset)
        if kk == 0:                                                          # :84-85
            continue
        ind1 = [int(conns[k, 6]) for k in kept]
        ind2 = [int(conns[k, 7]) for k in kept]
        score = [conns[k, 10] for k in kept]                                 # np.float32 scalars
        # snapshots taken before any update of this limb type (:87-88)
        id_f = [int(r[jf, 5]) for r in subset]
        id_t = [int(r[jt, 5]) for r in subset]
        sc_f = [r[jf, 4] for r in subset]
        sc_t = [r[jt, 4] for r in subset]
        msum = [[(id_f[m] == ind1[k]) + (id_t[m] == ind2[k]) for k in range(kk)]
                for m in range(mm)]                                          # :103-104
        repl = [[bool(score[k] > sc_t[m]) or bool(score[k] > sc_f[m]) for k in range(kk)]
                for m in range(mm)]                                          # :108-109

        # -- both endpoints already belong to person m (:114-119)
        pairs = [(m, k) for m in range(mm) for k in range(kk) if msum[m][k] == 2 and repl[m][k]]
        if pairs:
            stats['case2'] += len(pairs)
            rhs = [np.maximum(score[k], subset[m][jf, 4]) for m, k in pairs]
            for (m, k), v in zip(pairs, rhs):
                subset[m][jf, 4] = v
            rhs = [np.maximum(score[k], subset[m][jt, 4]) for m, k in pairs]
            for (m, k), v in zip(pairs, rhs):
                subset[m][jt, 4] = v
            for m in range(mm):
                for k in range(kk):
                    if msum[m][k] == 2:
                        msum[m][k] = -1

        # -- exactly one endpoint belongs to person m (:124-135)
        pairs = [(m, k) for m in range(mm) for k in range(kk) if msum[m][k] == 1 and repl[m][k]]
        if pairs:
            stats['case1'] += len(pairs)
            stats['dup_person_write'] += len(pairs) - len({m for m, _ in pairs})
            for m, k in pairs:                      # ids, then x, y, v, s; last pair wins
                row = conns[kept[k]]
                subset[m][jf, 5] = row[6]
                subset[m][jt, 5] = row[7]
            for m, k in pairs:
                row = conns[kept[k]]
                subset[m][jf, 0:4] = (row[0], row[1], row[2], row[11])
                subset[m][jt, 0:4] = (row[3], row[4], row[5], row[12])
            rhs = [np.maximum(score[k], subset[m][jf, 4]) for m, k in pairs]
            for (m, k), v in zip(pairs, rhs):
                subset[m][jf, 4] = v
            rhs = [np.maximum(score[k], subset[m][jt, 4]) for m, k in pairs]
            for (m, k), v in zip(pairs, rhs):
                subset[m][jt, 4] = v
            for m in range(mm):
                for k in range(kk):
                    if msum[m][k] == 1:
                        msum[m][k] = -1

        # -- merge persons that now share exactly two keypoints (:140-161)
        n_merged = 0
        if mm >= 2:
            ids = [[int(v) for v in r[:, 5]] for r in subset]
            mpairs = []
            for a in range(mm):
                for b in range(a + 1, mm):
                    shared = sum(1 for j in range(c) if ids[a][j] == ids[b][j] and ids[a][j] != -1)
                    if shared == 2:
                        mpairs.append((a, b))
                    elif shared >= 3:
                        stats['share3'] += 1
            if mpairs:
                stats['merge'] += len(mpairs)
                rhs = [np.maximum(subset[a], subset[b]) for a, b in mpairs]   # pre-update state
                for (a, b), v in zip(mpairs, rhs):
                    subset[a] = v
                gone = {b for _, b in mpairs}
                subset = [r for m, r in enumerate(subset) if m not in gone]
                n_merged = len(gone)

        # -- limbs no existing person claimed start new persons (:166-177)
        n_new = 0
        for k in range(kk):
            col = sum(msum[m][k] for m in range(mm))
            if col == 0:
                if mm and any(msum[m][k] != 0 for m in range(mm)):
                    stats['cancel_new'] += 1
                row = conns[kept[k]]
                new = np.full((c, 6), -1, dtype=F32)
                new[jf, 5], new[jt, 5] = row[6], row[7]
                new[jf, 0:4] = (row[0], row[1], row[2], row[11])
                new[jt, 0:4] = (row[3], row[4], row[5], row[12])
                new[jf, 4] = new[jt, 4] = row[10]
                subset.append(new)
                n_new += 1
        if trace is not None:
            trace.append((li, mm, kk, n_new, n_merged))

    return delete_sort(subset, c, person_thre, sort_dim)


def delete_sort(subset, n_keypoints, thre, index):
    """decoder/group.py:188-219 — drop persons scoring below ``thre``, stable
    descending sort, then every -1 becomes 0."""
    kept, scores = [], []
    for r in subset:
        s = person_score(r, index)
        if s < thre:            # NaN (no positive entry) is kept, as in the reference
            continue
        kept.append(r)
        scores.append(s)
    order = sorted(range(len(kept)), key=lambda i: scores[i], reverse=True)
    out = np.zeros((len(kept), n_keypoints, 6), dtype=F32)
    for dst, src in enumerate(order):
        out[dst] = kept[src]
    out[out == -1] = 0
    return out


# --------------------------------------------------------------------------- #
# decoder/factory.py
# --------------------------------------------------------------------------- #
def flip_average(x2n, perm=None, negate_even=False):
    """(orig + sign * flip_W(flipped)[perm]) / 2 — heat / scale / jitter maps
    (decoder/factory.py:101-113, 141-144)."""
    x2n = np.asarray(x2n, dtype=F32)
    n = x2n.shape[0] // 2
    fl = x2n[n:, :, :, ::-1].copy()
    if perm is not None:
        fl = fl[:, perm]
    if negate_even:
        fl[:, ::2] *= F32(-1)
    return ((x2n[:n] + fl) / F32(2)).astype(F32)


def flip_cat_offsets(offs, limb_flips, limb_reserve):
    """decoder/factory.py:115-127 — (2N, 2L, h, w) -> (N, 4L, h, w): per limb the original
    vector followed by the mirrored limb's vector (x negated); reserved limbs repeat theirs."""
    offs = np.asarray(offs, dtype=F32)
    n2, l2, h, w = offs.shape
    n = n2 // 2
    o = offs.reshape(n2, -1, 2, h, w)
    orig = o[:n]
    fl = o[n:, :, :, :, ::-1].copy()
    fl[:, :, 0] *= F32(-1.0)
    out = np.concatenate((orig, fl[:, limb_flips]), axis=2)
    out[:, limb_reserve, 2:] = orig[:, limb_reserve]
    return out.reshape(n, -1, h, w).astype(F32)


def flip_augment(hmps, offs, kp_flips, limb_flips, limb_reserve):
    """decoder/factory.py:98-146, default (vector addition) branch.
    hmps (2N, C, h, w), offs (2N, 2L, h, w): originals then W-flipped copies."""
    hmps = np.asarray(hmps, dtype=F32)
    offs = np.asarray(offs, dtype=F32)
    n2, l2, h, w = offs.shape
    n = n2 // 2
    flip_h = hmps[n:, :, :, ::-1][:, kp_flips]
    out_h = (hmps[:n] + flip_h) / F32(2)                                     # :101-106
    o = offs.reshape(n2, -1, 2, h, w)
    orig = o[:n]
    flip_o = o[n:, :, :, :, ::-1].copy()
    flip_o[:, :, 0] *= F32(-1.0)                                             # :132
    out_o = (orig + flip_o[:, limb_flips]) / F32(2)                          # :133
    out_o[:, limb_reserve] = orig[:, limb_reserve]                           # :134
    return out_h.astype(F32), out_o.reshape(n, -1, h, w).astype(F32)


def _fma(a, b, c):
    """float32 fused multiply-add emulated through float64 (the product of two
    float32 values is exact in float64; the final double rounding is harmless at
    the sizes this numpy oracle is used for — oracle/og_oracle.c uses fmaf)."""
    return (np.asarray(a, dtype=np.float64) * np.asarray(b, dtype=np.float64)
            + np.asarray(c, dtype=np.float64)).astype(F32)


def _cubic_weights(t):
    """ATen get_cubic_upsample_coefficients, A = -0.75 (UpSample.h)."""
    a = F32(-0.75)

    def inner(x):      # |x| <= 1
        return ((a + F32(2)) * x - (a + F32(3))) * x * x + F32(1)

    def outer(x):      # 1 < |x| < 2
        return ((a * x - F32(5) * a) * x + F32(8) * a) * x - F32(4) * a
    return [outer(t + F32(1)), inner(t), inner(F32(1) - t), outer(F32(2) - t)]


def _resize_taps(n_in, scale, cubic):
    """Source indices and weights of one axis for F.interpolate(scale_factor=scale,
    align_corners=False): src = (dst + 0.5) / scale - 0.5, clamped at 0 for
    bilinear only; taps clamped to the image (ATen UpSampleKernel.cpp
    HelperInterpLinear / HelperInterpCubic)."""
    n_out = int(n_in * scale)
    dst = np.arange(n_out, dtype=F32)
    real = F32(1.0 / scale) * (dst + F32(0.5)) - F32(0.5)
    if not cubic:
        real = np.maximum(real, F32(0))
    base = np.floor(real).astype(np.int64)
    lam = np.clip(real - base.astype(F32), 0, 1).astype(F32)
    if cubic:
        return [np.clip(base + j - 1, 0, n_in - 1) for j in range(4)], \
               [w.astype(F32) for w in _cubic_weights(lam)]
    return [np.minimum(base, n_in - 1), np.minimum(base + 1, n_in - 1)], [F32(1) - lam, lam]


def _combine_taps(terms, weights):
    """Accumulation order of ATen's generic CPU interpolation loop as compiled
    with FMA contraction: round(t1*w1), then fma(t0, w0, .), fma(t2, w2, .), ...
    (probed bit-for-bit against torch 2.11 CPU, see tests/golden/make_golden.py)."""
    acc = (terms[1] * weights[1]).astype(F32)
    acc = _fma(terms[0], weights[0], acc)
    for k in range(2, len(terms)):
        acc = _fma(terms[k], weights[k], acc)
    return acc


def resize(x, scale, mode):
    """F.interpolate(x, scale_factor=scale, mode=mode) for mode in
    {'bicubic', 'bilinear'}, align_corners=False (decoder/factory.py:74-78), as
    ATen's generic CPU kernel computes it (the path taken when output H + W > 128):
    rows are interpolated along x first, then combined along y."""
    x = np.asarray(x, dtype=F32)
    cubic = (mode == 'bicubic')
    h, w = x.shape[-2:]
    iy, wy = _resize_taps(h, scale, cubic)
    ix, wx = _resize_taps(w, scale, cubic)
    rows = []
    for j in range(len(iy)):
        xr = x[..., iy[j], :]
        terms = [xr[..., ix[i]] for i in range(len(ix))]
        wts = [np.broadcast_to(wx[i], terms[0].shape) for i in range(len(ix))]
        rows.append(_combine_taps(terms, wts))
    wts = [np.broadcast_to(wy[j][:, None], rows[0].shape) for j in range(len(iy))]
    return _combine_taps(rows, wts)


def generate_poses(hmps, offs, skeleton, n_keypoints, *, topk, thre_hmp, min_len, person_thre,
                   sort_dim=2, dist_max=20, use_scale=True, hmp_stride=4, off_stride=4,
                   resize_mode='bicubic', flip_test=False, kp_flips=None, limb_flips=None,
                   limb_reserve=None, return_limbs=False, scmps=None, jomps=None, use_jitter=True,
                   cat_flip_offs=False):
    """decoder/factory.py:52-96 on network-resolution maps: optional flip fusion, x stride
    resize, limb collection, greedy grouping; ``scmps`` / ``jomps`` are the optional
    keypoint-scale and jitter-offset heads, ``cat_flip_offs`` the 4-D offset variant."""
    vector_nd = 2
    if flip_test:
        if cat_flip_offs:
            offs = flip_cat_offsets(offs, limb_flips, limb_reserve)
            hmps = flip_average(hmps, kp_flips)
            vector_nd = 4
        else:
            hmps, offs = flip_augment(hmps, offs, kp_flips, limb_flips, limb_reserve)
        if jomps is not None:
            jomps = flip_average(jomps, None, True)
        if scmps is not None:
            scmps = flip_average(scmps, kp_flips)
    hmps_hr = resize(hmps, hmp_stride, resize_mode)
    offs_hr = resize(offs, off_stride, 'bilinear')
    scmps_hr = resize(scmps, off_stride, resize_mode) if scmps is not None else None
    jomps_hr = resize(jomps, hmp_stride, 'bilinear') if jomps is not None else None
    limbs = generate_limbs(hmps_hr, offs_hr, skeleton, topk, thre_hmp, min_len,
                           hmp_stride, off_stride, scmps_hr=scmps_hr, jomps_hr=jomps_hr,
                           use_jitter=use_jitter, vector_nd=vector_nd)
    poses = [group_skeletons(l, skeleton, n_keypoints, person_thre, sort_dim, dist_max, use_scale)
             for l in limbs]
    if return_limbs:
        return poses, limbs
    return poses


# --------------------------------------------------------------------------- #
# caller side: transforms/preprocess.py, evaluate.py
# --------------------------------------------------------------------------- #
def annotations_inverse(keypoints, meta):
    """transforms/preprocess.py:33-63 (hflip metas raise in the reference)."""
    k = np.array(keypoints, copy=True)
    k[:, :, 0] += meta['offset'][0]
    k[:, :, 1] += meta['offset'][1]
    k[:, :, 0] /= meta['scale'][0]
    k[:, :, 1] /= meta['scale'][1]
    k[:, :, 3] /= np.sqrt(np.prod(meta['scale']))
    if meta['hflip']:
        raise Exception('this should not happen. please have a check here, not implemented actually!')
    return k


def coco_result_rows(batch_poses, metas):
    """evaluate.py:227-265 — explicit loops, as the reference writes them."""
    rows, ids = [], []
    for poses, meta in zip(batch_poses, metas):
        subset = annotations_inverse(poses, meta)
        ids.append(meta['image_id'])
        subset[:, :, :2] = np.around(subset[:, :, :2], 2)
        for person in subset.astype(float):
            kps, v = [], []
            for xyv in person[:, :3]:
                v.append(xyv[2])
                kps += [xyv[0], xyv[1], 1 if xyv[0] > 0 or xyv[1] > 0 else 0]
            rows.append({'image_id': meta['image_id'], 'category_id': 1, 'keypoints': kps,
                         'score': sum(v) / len(v)})
        if not len(subset):
            rows.append({'image_id': meta['image_id'], 'category_id': 1,
                         'keypoints': np.zeros((subset.shape[1] * 3,)).tolist(), 'score': 0.01})
    return rows, ids
