"""Grouping (K3) on crowded images and at top-K values that are not powers of two.

The one-warp grouping kernel takes one of two code paths in every limb step: the register
path while the step starts with at most 32 persons and the limb type has at most 32 kept rows,
the general path (shared-memory work arrays) above that, up to the `warp_rows` person rows of
its table.  An image that needs more rows is regrouped by the CTA kernel.  The tables below
are built to land in every one of these regimes — the oracle's trace of each limb step
(persons, kept rows, new and merged persons) proves which — and the kernels are compared
with the oracles bit for bit.  The end-to-end tests decode rendered crowds of 35-60 persons
through K1 -> K2 -> K3 at top-K 1 ... 128."""
import functools

import numpy as np
import pytest

import golden_io as gio
from oracle import c_oracle as co
from oracle import ref_oracle as ro
from oracle import scenes
from offsetguided_b200 import config as cfg

RTOL = 1e-5
LANES = 32                          # register path: at most this many persons and kept rows
COCO = cfg.COCO_PERSON_SKELETON
CHAIN = [(0, 1), (1, 2), (2, 3), (3, 4)]
# limb 2 joins the persons of limbs 0 and 1 at both ends: they share two ids and merge
TWICE = [(0, 1), (2, 3), (1, 3), (3, 4)]
CLOSING = [(0, 1), (1, 2), (0, 2), (2, 3)]
THRE = 0.06
DIST_MAX = 40
ID0 = 1 << 23                       # candidate ids of the generated tables; exact in float32, apart from
                                    # the ids of the committed fuzz tables (below 17 * 409600)


# --------------------------------------------------------------------------- tables
def _table(rng, skel, n_kp, k, rows, ties=False, same_v=False, decoys=True, lift=None, scores=None):
    """(L, k, 13) limb table whose kept rows are exactly ``rows[l]``: a list of (a, b) pairs
    linking candidate a of the from-joint to candidate b of the to-joint of limb type l, the b
    distinct.  Candidate p of joint j has id ID0 + j * 4096 + p.  The free rows of the table become
    decoys that the gate or the best-row-per-to-id rule removes: rows beyond the distance
    gate, rows outside the image, and rows repeating a kept to-id at a score no higher (with
    equal scores the row that sorts first is kept, so the rank order of ties decides which).
    Rows from ``lift`` on score above the others; ``scores[l]`` gives the scores explicitly."""
    pool = 1 + max([max(max(a, b) for a, b in r) for r in rows if r] + [0])
    xy = rng.randint(1, 600, size=(n_kp, pool, 2)).astype(np.float32)
    t = np.zeros((len(skel), k, 13), np.float32)
    t[:, :, 8] = 1000.0                                    # unused rows fail the distance gate
    for l, (jf, jt) in enumerate(skel):
        pairs = list(rows[l])
        assert len(pairs) <= k and len({b for _, b in pairs}) == len(pairs)
        n = len(pairs)
        if ties:
            sc = (rng.randint(1, 4, size=n) / np.float32(8)).astype(np.float32)
        else:
            sc = ((rng.permutation(n) + rng.uniform(0.1, 0.9, size=n)) / max(n, 1)).astype(np.float32)
        if lift is not None:
            sc[lift:] += np.float32(1)
        if scores is not None:
            sc = np.asarray(scores[l], np.float32)
        slots = rng.permutation(k)
        for r, (a, b) in enumerate(pairs):
            v1, v2 = (0.5, 0.5) if same_v else (0.5, 0.6)
            t[l, slots[r]] = (xy[jf, a, 0], xy[jf, a, 1], v1, xy[jt, b, 0], xy[jt, b, 1], v2,
                              ID0 + jf * 4096 + a, ID0 + jt * 4096 + b, rng.uniform(0, DIST_MAX - 1), 10, sc[r], 4, 4)
        if not decoys:
            continue
        for s in slots[n:]:
            kind = rng.randint(3)
            if kind == 0 or n == 0:
                continue                                   # beyond the gate
            r = rng.randint(n)
            a, b = pairs[r]
            t[l, s] = t[l, slots[r]]
            if kind == 1:                                  # outside the image
                t[l, s, 0] = 0.0
            else:                                          # same to-id, another from-candidate
                a2 = rng.randint(pool)
                t[l, s, 0:2] = xy[jf, a2]
                t[l, s, 6] = ID0 + jf * 4096 + a2
                t[l, s, 10] = sc[r] if ties else sc[r] * np.float32(rng.uniform(0.5, 1.0))
    return t


def _links(rng, n_rows, share, from_pool=None):
    """Kept rows of one limb type: to-candidates 0 .. n_rows - 1.  The row ending at b starts
    at candidate b of the from-joint (the links of one person) while b < ``from_pool``; with
    probability ``share``, and for every b >= ``from_pool``, at a random candidate below
    ``from_pool`` instead (crossed links: shared ids, merges, duplicate from-ids)."""
    from_pool = from_pool or n_rows
    return [(b if (b < from_pool and rng.uniform() >= share) else int(rng.randint(from_pool)), b)
            for b in range(n_rows)]


def _opening(skel):
    """Limb types whose to-joint no earlier type has seen: there a person's to-joint is unset,
    so every row a person matches passes the replacement test and the last one wins."""
    seen, out = set(), []
    for l, (jf, jt) in enumerate(skel):
        if jf in seen and jt not in seen:
            out.append(l)
        seen |= {jf, jt}
    return out


def _crowd(rng, kk, persons, share, k, skel=COCO, n_kp=17, **kw):
    """Table of ``persons`` persons in which the opening limb types have ``kk`` kept rows: the
    rows beyond the persons' own start at a joint one of them holds and score above the own
    rows, so the own row (last in score order) wins.  They are matched, so they start nobody:
    the table stays near ``persons`` per skeleton component while kk exceeds the lane count."""
    opening = _opening(skel)
    rows = [_links(rng, kk if l in opening else persons, share, persons) for l in range(len(skel))]
    return _table(rng, skel, n_kp, k, rows, lift=persons, **kw)


def _crowd_tables():
    """The generated set: (name, skeleton, n_keypoints, k, table).  Every entry is seeded."""
    rng = np.random.RandomState(4848)
    out = []
    nl = len(COCO)
    # kept rows per limb type around the lane count and far above it; 16 / 30 persons, whose
    # second component (limb type 5 on) doubles the table before the merges join them up
    for kk in (31, 32, 33, 48, 64, 128):
        k = 48 if kk <= 48 else kk
        for persons, share in ((16, 0.03), (30, 0.0), (24, 0.06)):
            out.append((f'kk{kk}_p{persons}_s{share}', COCO, 17, k,
                        _crowd(rng, kk, persons, share, k, ties=share > 0.05)))
    # one component only (limb type 5 has no rows) of 40 persons, all with the same score: the
    # stable rank of equal scores across the 32-lane strides
    for ties in (False, True):
        rows = [_links(rng, 40, 0.05 if ties else 0.0) for _ in range(nl)]
        rows[5] = []
        out.append((f'tied_scores_{ties}', COCO, 17, 48, _table(rng, COCO, 17, 48, rows, ties=ties, same_v=True)))
    # register -> general -> register: 20 persons, two opening steps of 48 / 40 rows
    rows = [_links(rng, 20, 0.03) for _ in range(nl)]
    rows[1] = _links(rng, 48, 0.03, from_pool=20)
    rows[9] = _links(rng, 40, 0.03, from_pool=20)
    out.append(('reg_gen_reg', COCO, 17, 48, _table(rng, COCO, 17, 48, rows, ties=True, lift=20)))
    # heavy sharing: most rows cross between persons
    for persons in (12, 24):
        out.append((f'shared_p{persons}', COCO, 17, 48, _crowd(rng, 40, persons, 0.6, 48, ties=True)))
    # the committed fuzz tables with a cancellation person and persons sharing three ids,
    # next to 30 more persons (other ids, rows in the first limb types only, so that they add
    # no case to the later steps): the same steps, taken on the general path
    fuzz = gio.load_group_fuzz()
    for i in (0, 1, 2, 3):
        pad = _table(rng, COCO, 17, 32, [_links(rng, 30, 0.0) if l in (0, 1, 3, 4) else [] for l in range(nl)])
        out.append((f'fuzz{i}_padded', COCO, 17, 48, np.concatenate([fuzz[i]['limbs'], pad], axis=1)))
    # hand-off from the general path to the register path: in the general step (limb type 2,
    # 36 kept rows) the row 0:x -> 2:x is held at both ends by X and at one end by Y and Z, none
    # of them replacing, while W replaces: the column sum 2 * 1 - 2 cancels and the row starts
    # a person sharing exactly two ids with X.  The next step only fills in Y's joint 3 — no id
    # is rewritten — and must still merge that pair (group.py compares all pairs every step).
    rows = [[(0, 0), (0, 1), (0, 2), (3, 3)], [(0, 0), (1, 1), (2, 2), (3, 3)],
            [(0, 0)] + [(3, b) for b in range(4, 39)], [(1, 1)]]
    scores = [[0.9] * 4, [0.9] * 4, [0.1] + [0.95] * 35, [0.9]]
    out.append(('handoff', CLOSING, 4, 48, _table(rng, CLOSING, 4, 48, rows, scores=scores)))
    # outgrow the warp kernel's 64 rows: the CTA kernel finishes these
    for kk in (33, 48):
        rows = [_links(rng, kk, 0.15) for _ in range(nl)]
        out.append((f'overflow_kk{kk}', COCO, 17, 48, _table(rng, COCO, 17, 48, rows, ties=True)))
    # CrowdPose skeleton, 14 keypoints: one component
    for kk, persons in ((36, 36), (56, 24)):
        out.append((f'crowdpose_kk{kk}_p{persons}', cfg.CROWDPOSE_PERSON_SKELETON, 14, 64,
                    _crowd(rng, kk, persons, 0.1, 64, cfg.CROWDPOSE_PERSON_SKELETON, 14)))
    return out


def _boundary_tables(r):
    """Tables whose grouping allocates exactly ``r`` and ``r + 1`` person rows:
    (name, skeleton, k, allocations, table)."""
    rng = np.random.RandomState(1000 + r)
    k = 48 if r < 48 else 128
    out = []
    for n in (r, r + 1):
        # a chain of n persons: all of them start in the first step
        out.append((f'chain{n}', CHAIN, k, n, _table(rng, CHAIN, 5, k, [_links(rng, n, 0.0)] * 4)))
    # r - 1 persons, the last step starts one or two more: the overflow comes late
    for extra in (1, 2):
        rows = [_links(rng, r - 1, 0.0)] * 3 + [_links(rng, r - 1 + extra, 0.0)]
        out.append((f'late{r - 1 + extra}', CHAIN, k, r - 1 + extra, _table(rng, CHAIN, 5, k, rows)))
    # two halves of r / 2 persons merge in step 2 (merged rows are not reused), then the last
    # step starts zero or one more
    h = r // 2
    for extra in (0, 1):
        rows = [_links(rng, h, 0.0)] * 3 + [_links(rng, h + extra, 0.0)]
        out.append((f'merged{2 * h + extra}', TWICE, k, 2 * h + extra, _table(rng, TWICE, 5, k, rows)))
    return out


@functools.lru_cache(maxsize=None)
def _traces(which):
    """Numpy-oracle poses and trace of every table of a generated set."""
    tables = _crowd_tables() if which == 'crowd' else _boundary_tables(which)
    out = []
    for entry in tables:
        skel, t = entry[1], entry[-1]
        c = entry[2] if which == 'crowd' else 5
        tr = []
        poses = ro.group_skeletons(t, skel, c, THRE, 2, DIST_MAX, True, trace=tr)
        out.append((poses, tr))
    return out


def _register(step):
    _, mm, kk, _, _ = step
    return mm <= LANES and kk <= LANES


def _allocated(trace):
    return sum(s[3] for s in trace)


def _person_scores(poses):
    return [ro.person_score(p, 2) for p in poses]


def _paths(trace):
    return ''.join('R' if _register(s) else 'G' for s in trace)


# --------------------------------------------------------------------------- CPU
def test_trace_leaves_results_unchanged():
    for c in gio.load_group_fuzz():
        args = (c['limbs'], c['skeleton'], c['n_keypoints'], c['person_thre'], c['sort_dim'], 40, c['use_scale'])
        trace = []
        got = ro.group_skeletons(*args, trace=trace)
        assert np.array_equal(got, c['poses'])
        assert np.array_equal(got, ro.group_skeletons(*args))
        assert all(s[2] > 0 for s in trace) and [s[0] for s in trace] == sorted({s[0] for s in trace})
        # persons at the start of a step = those of the step before, minus merged, plus new
        for a, b in zip(trace, trace[1:]):
            assert b[1] == a[1] - a[4] + a[3]


@pytest.mark.parametrize('rows', [64, 128])
def test_generated_tables_cover_every_regime(rows):
    """Every regime the warp kernel has, on tables it finishes itself (at most ``rows`` person
    rows allocated); and tables it must hand to the CTA kernel."""
    tables, traces = _crowd_tables(), _traces('crowd')
    fit = [(e, p, tr) for e, (p, tr) in zip(tables, traces) if _allocated(tr) <= rows]
    steps = [(e, s) for e, _, tr in fit for s in tr]
    assert {31, 32, 33, 48, 64, 128} <= {s[2] for _, s in steps}
    assert any(_register(s) and s[2] in (31, 32) for _, s in steps)
    assert any(not _register(s) and s[1] > LANES for _, s in steps)                 # many persons
    assert any(not _register(s) and s[1] <= LANES and s[2] > LANES for _, s in steps)   # many rows
    assert any(not _register(s) and s[4] > 0 for _, s in steps)                       # general-path merge
    assert any(not _register(s) and s[1] > 48 for _, s in steps)
    assert any('RG' in _paths(tr) and 'GR' in _paths(tr)[_paths(tr).index('RG'):] for _, _, tr in fit)
    # a register step right after a general step merges persons without rewriting any id
    handoff = [(e, tr) for e, _, tr in fit if e[0] == 'handoff'][0][1]
    assert _paths(handoff) == 'RRGR' and handoff[2][3] == 1 and handoff[3][4] == 1
    # sharing patterns on tables whose every step takes the general path
    general = [(e, tr) for e, _, tr in fit if 'R' not in _paths(tr)]
    seen = dict(case2=0, case1=0, dup_person_write=0, merge=0, share3=0, cancel_new=0)
    dup_from = 0
    for (name, skel, c, k, t), tr in general:
        st = {}
        ro.group_skeletons(t, skel, c, THRE, 2, DIST_MAX, True, stats=st)
        for key in seen:
            seen[key] += st[key]
        for li, _, _, _, _ in tr:
            kept = ro.delete_reconns(t[li], ro.valid_limb_rows(t[li], DIST_MAX, True))
            ids = [int(t[li, r, 6]) for r in kept]
            dup_from += len(ids) > len(set(ids))
    assert all(v > 0 for v in seen.values()), seen
    assert dup_from > 0
    # more than 32 kept persons with equal scores (their order is the stable one)
    assert any(max(np.unique(_person_scores(p), return_counts=True)[1]) > LANES for _, p, _ in fit)
    # and images that outgrow the table
    assert any(_allocated(tr) > rows for tr in (t for _, t in traces))


@pytest.mark.parametrize('r', [40, 64])
def test_boundary_tables_allocate_r_and_r_plus_one(r):
    for (name, skel, k, n, t), (poses, tr) in zip(_boundary_tables(r), _traces(r)):
        assert _allocated(tr) == n, name
        assert 'G' in _paths(tr), name
        assert len(poses) == n - sum(s[4] for s in tr), name
    allocs = [e[3] for e in _boundary_tables(r)]
    assert allocs.count(r) >= 2 and allocs.count(r + 1) >= 2


def test_c_oracle_equals_numpy_oracle_on_generated_tables():
    """The GPU tests check most tables against the C oracle only."""
    for (name, skel, c, k, t), (poses, _) in zip(_crowd_tables(), _traces('crowd')):
        assert np.array_equal(co.group_skeletons(t, skel, c, THRE, 2, DIST_MAX, True), poses), name
    for r in (40, 64):
        for (name, skel, k, n, t), (poses, _) in zip(_boundary_tables(r), _traces(r)):
            assert np.array_equal(co.group_skeletons(t, skel, 5, THRE, 2, DIST_MAX, True), poses), name


# --------------------------------------------------------------------------- GPU
def _group(monkeypatch, warp_rows, skel, c, stack):
    """GreedyGroup.group_batch with the warp kernel's table at ``warp_rows`` rows (0: CTA kernel
    only); the handle reads OG_K3_WARP_ROWS when it is created."""
    from offsetguided_b200 import decoder
    monkeypatch.setenv('OG_K3_WARP_ROWS', str(warp_rows))
    g = decoder.GreedyGroup(THRE, sort_dim=2, dist_max=DIST_MAX, use_scale=True,
                            keypoints=list(range(c)), skeleton=skel)
    return g.group_batch(stack)


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [64, 128])
@pytest.mark.parametrize('batch', [100, 400])          # fewer images than SMs / several per SM
def test_crowd_tables_warp_cta_and_oracles(cuda_device, monkeypatch, rows, batch):
    tables, traces = _crowd_tables(), _traces('crowd')
    groups = {}
    for i, (name, skel, c, k, t) in enumerate(tables):
        groups.setdefault((tuple(skel), c, k), []).append(i)
    for (skel, c, k), idx in groups.items():
        order = [idx[j % len(idx)] for j in range(batch)]
        stack = np.stack([tables[i][4] for i in order])
        warp = _group(monkeypatch, rows, list(skel), c, stack)
        cta = _group(monkeypatch, 0, list(skel), c, stack)
        ref = {i: co.group_skeletons(tables[i][4], list(skel), c, THRE, 2, DIST_MAX, True) for i in idx}
        for j, i in enumerate(order):
            name = tables[i][0]
            assert warp[j].shape == ref[i].shape and np.array_equal(warp[j], ref[i]), f'{name} warp rows={rows}'
            assert cta[j].shape == ref[i].shape and np.array_equal(cta[j], ref[i]), f'{name} CTA'
        for i in idx:                                   # numpy oracle (the traced one)
            assert np.array_equal(warp[order.index(i)], traces[i][0]), tables[i][0]


def _chain_maps(counts, k):
    """Full-resolution maps of CHAIN persons, one image per entry of ``counts``: joint j of
    person p is an isolated peak 4 px right of joint j - 1, and the offset at joint j points at
    joint j + 1 exactly.  Every person is one limb row per limb type: the grouping allocates
    exactly ``count`` person rows."""
    h, w = 64, 208
    assert max(counts) <= k and max(counts) <= 8 * 14
    heat = np.zeros((len(counts), 5, h, w), np.float32)
    offs = np.zeros((len(counts), 8, h, w), np.float32)
    for i, n in enumerate(counts):
        for p in range(n):
            x0, y0 = 4 + (p % 8) * 25, 4 + (p // 8) * 4
            for j in range(5):
                heat[i, j, y0, x0 + 4 * j] = 0.5 + 0.01 * ((3 * p + j) % 7)
                if j < 4:
                    offs[i, 2 * j, y0, x0 + 4 * j] = 4.0
    return heat, offs


@pytest.mark.gpu
@pytest.mark.parametrize('r', [40, 64])
def test_boundary_tables_at_warp_rows(cuda_device, monkeypatch, r):
    """Tables that allocate exactly r and r + 1 person rows, with the warp kernel's table at r
    rows: the first are finished by the warp kernel, the others by the CTA kernel, and all
    equal the oracle.  On the decode path the CTA kernel runs only for a batch with an image
    that outgrew the table, which k3_redo_count counts."""
    import torch
    from offsetguided_b200.engine import DecoderEngine
    entries, traces = _boundary_tables(r), _traces(r)
    for skel in (CHAIN, TWICE):
        idx = [i for i, e in enumerate(entries) if e[1] is skel]
        stack = np.stack([entries[i][4] for i in idx])
        for rows in (r, 0):
            got = _group(monkeypatch, rows, skel, 5, stack)
            for j, i in enumerate(idx):
                assert np.array_equal(got[j], traces[i][0]), f'{entries[i][0]} rows={rows}'
    k = entries[0][2]
    monkeypatch.setenv('OG_K3_WARP_ROWS', str(r))
    eng = DecoderEngine(5, CHAIN, topk=k, thre_hmp=THRE, min_len=0.5, dist_max=DIST_MAX, use_scale=True,
                        person_thre=THRE)
    for counts, redo in (([r, r - 1], 0), ([r, r + 1], 1), ([r + 1], 1), ([r], 0)):
        heat, offs = _chain_maps(counts, k)
        before = eng.k3_redo_count
        got = eng.decode_maps(torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda())
        assert eng.k3_redo_count - before == redo, counts
        limbs = co.generate_limbs(heat, offs, CHAIN, k, THRE, 0.5, 1, 1)
        _, _, lb = eng.last_intermediates(len(counts))
        assert gio.compare_limbs(lb.cpu().numpy(), limbs, THRE, rtol=RTOL) == 4 * sum(counts)
        for p, lim, n in zip(got, limbs, counts):
            ref = ro.group_skeletons(lim, CHAIN, 5, THRE, 2, DIST_MAX, True)
            assert len(ref) == n
            gio.compare_poses(p, ref, rtol=RTOL)


def _crowd_scenes(template):
    skel = COCO if template is scenes.TEMPLATE_COCO else cfg.CROWDPOSE_PERSON_SKELETON
    hs, os_ = [], []
    for i, n in enumerate((35, 48, 60)):
        h, o = scenes.render_batch(5100 + 10 * i, 1, n, 512, 512, skel, template=template, noise=0.02,
                                   scale_range=(6.0, 12.0))
        hs.append(h)
        os_.append(o)
    return skel, np.concatenate(hs), np.concatenate(os_)


@functools.lru_cache(maxsize=None)
def _scene_reference(template_name, topk):
    template = getattr(scenes, template_name)
    skel, hmp, omp = _crowd_scenes(template)
    c = template.shape[0]
    poses, limbs = co.generate_poses(hmp, omp, skel, c, topk=topk, thre_hmp=THRE, min_len=0.5, person_thre=THRE,
                                     dist_max=float(DIST_MAX), use_scale=True, return_limbs=True)
    traces = []
    for lim in limbs:
        tr = []
        ro.group_skeletons(lim, skel, c, THRE, 2, DIST_MAX, True, trace=tr)
        traces.append(tr)
    return skel, hmp, omp, poses, limbs, traces


@pytest.mark.gpu
@pytest.mark.parametrize('template', ['TEMPLATE_COCO', 'TEMPLATE_CROWDPOSE'])
@pytest.mark.parametrize('topk', [1, 33, 48, 64, 100, 128])
def test_crowd_scenes_end_to_end(cuda_device, monkeypatch, template, topk):
    """Rendered crowds of 35, 48 and 60 persons, decoded through K1 -> K2 -> K3 on the fused
    and on the materialising path, with the warp kernel's table at 64 (default) and 128 rows:
    limbs and poses equal the C oracle.  From top-K 33 on every image takes the general path
    in some step.  The images whose trace allocates more rows than the table are the ones the
    CTA kernel finishes: every COCO crowd at 64 rows (its skeleton has two components, so
    every person is allocated twice before the merges), some CrowdPose crowds at 64 rows and
    some COCO crowds at 128."""
    import torch
    from offsetguided_b200.engine import DecoderEngine
    skel, hmp, omp, ref, ref_limbs, traces = _scene_reference(template, topk)
    c, n = hmp.shape[1], hmp.shape[0]
    if topk >= 33:
        assert all('G' in _paths(tr) for tr in traces), [_paths(tr) for tr in traces]
    finished = {}
    for rows in (64, 128):
        monkeypatch.setenv('OG_K3_WARP_ROWS', str(rows))
        eng = DecoderEngine(c, skel, topk=topk, thre_hmp=THRE, min_len=0.5, dist_max=DIST_MAX, use_scale=True,
                            person_thre=THRE)
        outgrown = [_allocated(tr) > rows for tr in traces]
        finished[rows] = ['CTA' if o else 'warp' for o in outgrown]
        for fused in (True, False):
            eng.set_fused(fused)
            before = eng.k3_redo_count
            got = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), 4, 4, 'bicubic')
            assert eng.k3_redo_count - before == (1 if any(outgrown) else 0)
            _, _, lb = eng.last_intermediates(n)
            assert gio.compare_limbs(lb.cpu().numpy(), ref_limbs, THRE, rtol=RTOL) >= n * min(topk, 35)
            assert len(got) == n
            for p, r in zip(got, ref):
                gio.compare_poses(p, r, rtol=RTOL)
    if topk >= 48:
        assert 'warp' in finished[64 if template == 'TEMPLATE_CROWDPOSE' else 128]
    print(f'{template} topk={topk}: persons {[len(r) for r in ref]}, rows allocated '
          f'{[_allocated(tr) for tr in traces]}, finished by {finished}')


@pytest.mark.gpu
def test_ring_64_keypoints_at_largest_k(cuda_device):
    """64 keypoints / 64 limbs (a ring) at K = 96, the largest top-K the library accepts for this
    skeleton (K = 97 is refused): the warp kernel's table is halved to 32 rows to fit 96 KB of
    shared memory, so 24 persons stay in it and 40 go to the CTA kernel."""
    import torch
    from offsetguided_b200 import _lib
    from offsetguided_b200.engine import DecoderEngine
    c = 64
    ring = [(j, (j + 1) % c) for j in range(c)]
    rng = np.random.RandomState(6464)
    h, w = 260, 380
    with pytest.raises(_lib.OgError):
        DecoderEngine(c, ring, topk=97, thre_hmp=0.05)
    eng = DecoderEngine(c, ring, topk=96, thre_hmp=0.05, min_len=0.5, dist_max=DIST_MAX, use_scale=True,
                        person_thre=0.05)
    for persons, redo in ((24, 0), (40, 1)):
        heat = rng.uniform(0, 0.02, size=(1, c, h, w)).astype(np.float32)
        offs = np.zeros((1, 2 * c, h, w), np.float32)
        for p in range(persons):
            x0, y0 = 8 + (p % 4) * 90 + rng.randint(0, 3), 8 + (p // 4) * 25
            pts = [(x0 + (j % 16) * 5, y0 + (j // 16) * 5 + rng.randint(0, 2)) for j in range(c)]
            for j, (x, y) in enumerate(pts):
                heat[0, j, y, x] = 0.9 - 0.01 * (p % 10) + 0.001 * j
            for l, (a, b) in enumerate(ring):
                (xa, ya), (xb, yb) = pts[a], pts[b]
                offs[0, 2 * l, ya, xa] = xb - xa
                offs[0, 2 * l + 1, ya, xa] = yb - ya
        before = eng.k3_redo_count
        got = eng.decode_maps(torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda())
        assert eng.k3_redo_count - before == redo
        limbs = co.generate_limbs(heat, offs, ring, 96, 0.05, 0.5, 1, 1)
        tr = []
        ref = ro.group_skeletons(limbs[0], ring, c, 0.05, 2, DIST_MAX, True, trace=tr)
        assert len(ref) == persons and _allocated(tr) == persons
        gio.compare_poses(got[0], ref, rtol=RTOL)
