"""GPU suite (-m gpu): the CUDA path, called through the C ABI, against the oracle on
seeded inputs and against the committed reference outputs (tests/golden).

Bar (BASELINE.json north_star): peak coordinates, top-K indices and person
assignments bit-exact; keypoint / limb / person scores within 1e-5 relative."""
import numpy as np
import pytest
import torch

import golden_io as gio
from oracle import ref_oracle as ro
from oracle import scenes
from offsetguided_b200 import config as cfg
from offsetguided_b200 import decoder
from offsetguided_b200.engine import DecoderEngine

pytestmark = pytest.mark.gpu

RTOL = 1e-5      # tolerance north_star states for floating-point scores


def _engine(d, c, skeleton, **over):
    kw = dict(topk=d['topk'], thre_hmp=d['thre_hmp'], min_len=d['min_len'], resize_factor=1.0,
              dist_max=d['dist_max'], use_scale=True, person_thre=d['person_thre'], sort_dim=2)
    kw.update(over)
    return DecoderEngine(c, skeleton, **kw)


# --------------------------------------------------------------------------- K1
@pytest.mark.parametrize('name', ['limbs_coco_a', 'limbs_coco_noise', 'limbs_crowdpose'])
def test_k1_matches_reference_dets(cuda_device, name):
    d = gio.load_limbs_case(name)
    eng = _engine(d, d['n_keypoints'], d['skeleton'])
    s, i, cnt = eng.nms_topk(torch.from_numpy(d['heat']).cuda())
    s, i, cnt = s.cpu().numpy(), i.cpu().numpy(), cnt.cpu().numpy()
    live = d['det_scores'] >= np.float32(d['thre_hmp'])
    assert np.array_equal(cnt, live.sum(-1))
    assert np.array_equal(s[live], d['det_scores'][live])
    assert np.array_equal(i[live], d['det_inds'][live])
    assert np.all(i[~live] == -1) and np.all(s[~live] == 0)


def test_k1_exact_joint_dets_radix_path(cuda_device):
    """thre = -inf: every pixel qualifies, all planes take the radix path; the result
    must be the exact top-K of the NMS map including zero filler by lowest index."""
    rng = np.random.RandomState(0)
    heat = rng.uniform(0, 1, size=(2, 3, 70, 90)).astype(np.float32)
    heat[0, 1] = 0                      # constant plane: all ties
    heat[1, 2, 10:20, 10:30] = 0.5      # plateau block
    eng = DecoderEngine(3, [(0, 1), (1, 2)], topk=40)
    s, i, _ = eng.nms_topk(torch.from_numpy(heat).cuda(), thre=float('-inf'))
    ref_s, ref_i, _, _ = ro.joint_dets(heat, 40)
    assert np.array_equal(i.cpu().numpy(), ref_i)
    assert np.array_equal(s.cpu().numpy(), ref_s)


@pytest.mark.parametrize('thre', [0.0, -0.5, float('-inf')])
def test_k1_non_positive_threshold_lists_peaks_then_zeros(cuda_device, thre):
    """thre <= 0: pass 1 lists the positive peaks, the selection completes the top-K with the
    zeros of the non-peaks (lowest index first); planes without enough of them — constant
    negative planes, whose interior is all peaks — take the radix selection, which then also
    ranks the negative peaks above the threshold."""
    rng = np.random.RandomState(11)
    heat = np.zeros((2, 4, 48, 64), np.float32)
    for c in range(4):                                   # a few positive and negative isolated peaks
        for _ in range(5):
            y, x = rng.randint(2, 46), rng.randint(2, 62)
            heat[0, c, y, x] = rng.uniform(0.1, 1.0)
            heat[1, c, y, x] = -rng.uniform(0.1, 1.0)
    heat[0, 3] = rng.uniform(-1, 1, size=(48, 64))       # dense mixed-sign noise
    heat[1, 3] = -0.25                                   # constant negative: zeros on the border ring only
    small = np.full((1, 2, 3, 4), -0.25, np.float32)     # 10 border zeros, 2 interior peaks, K = 12
    small[0, 1, 1, 1] = -0.75
    for maps, k in ((heat, 40), (small, 12)):
        eng = DecoderEngine(maps.shape[1], [(0, 1)], topk=k)
        s, i, cnt = eng.nms_topk(torch.from_numpy(maps).cuda(), thre=thre)
        nms = ro.hmp_nms(maps)
        nms[nms < np.float32(thre)] = -np.inf
        ref_s, ref_i, _, _ = ro.topk_channel(nms, k)
        live = ref_s >= np.float32(thre)
        assert np.array_equal(cnt.cpu().numpy(), live.sum(-1))
        assert np.array_equal(i.cpu().numpy()[live], ref_i[live])
        assert np.array_equal(s.cpu().numpy()[live], ref_s[live])


def test_k1_overflow_planes_fall_back_to_radix(cuda_device):
    """Noise maps: > 2048 peaks per plane above the threshold."""
    rng = np.random.RandomState(1)
    heat = rng.uniform(0, 1, size=(1, 17, 200, 256)).astype(np.float32)
    eng = DecoderEngine(17, cfg.COCO_PERSON_SKELETON, topk=32, thre_hmp=0.04)
    s, i, cnt = eng.nms_topk(torch.from_numpy(heat).cuda())
    ref_s, ref_i, _, _ = ro.joint_dets(heat, 32)
    assert np.array_equal(i.cpu().numpy(), ref_i) and np.array_equal(s.cpu().numpy(), ref_s)
    assert np.all(cnt.cpu().numpy() == 32)


@pytest.mark.parametrize('shape', [(1, 2, 5, 7), (1, 1, 1, 1), (2, 3, 33, 130), (1, 2, 64, 128),
                                   (1, 1, 65, 129), (1, 2, 130, 516), (1, 1, 3, 1030)])
def test_k1_ragged_shapes_and_borders(cuda_device, shape):
    rng = np.random.RandomState(sum(shape))
    heat = rng.uniform(-0.2, 1, size=shape).astype(np.float32)
    heat[..., 0, :] = rng.uniform(-1, 1, size=shape[:2] + (shape[3],))     # border values
    heat[..., :, -1] = rng.uniform(-1, 1, size=shape[:3])
    k = min(16, shape[2] * shape[3])
    eng = DecoderEngine(shape[1], [(0, 0)], topk=k, thre_hmp=0.3)
    s, i, cnt = eng.nms_topk(torch.from_numpy(heat).cuda())
    nms = ro.hmp_nms(heat)
    nms[nms < np.float32(0.3)] = -1          # threshold first
    ref_s, ref_i, _, _ = ro.topk_channel(nms, k)
    live = ref_s >= np.float32(0.3)
    assert np.array_equal(cnt.cpu().numpy(), live.sum(-1))
    assert np.array_equal(i.cpu().numpy()[live], ref_i[live])
    assert np.array_equal(s.cpu().numpy()[live], ref_s[live])
    # the stand-alone API on the same map
    out = decoder.hmp_NMS(torch.from_numpy(heat).cuda())
    assert np.array_equal(out.cpu().numpy(), ro.hmp_nms(heat))
    ts, ti, ty, tx = decoder.topK_channel(out, K=k)
    rs, ri, ry, rx = ro.topk_channel(ro.hmp_nms(heat), k)
    assert np.array_equal(ti.cpu().numpy(), ri) and np.array_equal(ts.cpu().numpy(), rs)
    assert np.array_equal(ty.cpu().numpy(), ry) and np.array_equal(tx.cpu().numpy(), rx)
    assert ti.dtype == torch.int64


def test_k1_unaligned_base_pointer(cuda_device):
    rng = np.random.RandomState(5)
    buf = torch.from_numpy(rng.uniform(0, 1, size=(1 + 2 * 40 * 64,)).astype(np.float32)).cuda()
    heat = buf[1:].view(1, 2, 40, 64)          # 4-byte aligned only
    assert heat.data_ptr() % 16 != 0
    eng = DecoderEngine(2, [(0, 1)], topk=8, thre_hmp=0.5)
    s, i, _ = eng.nms_topk(heat)
    nms = ro.hmp_nms(heat.cpu().numpy())
    rs, ri, _, _ = ro.topk_channel(nms, 8)
    assert np.array_equal(i.cpu().numpy(), ri) and np.array_equal(s.cpu().numpy(), rs)


# --------------------------------------------------------------------------- K2
@pytest.mark.parametrize('name', ['limbs_coco_a', 'limbs_coco_noise', 'limbs_crowdpose'])
def test_k2_limbs_match_reference(cuda_device, name):
    d = gio.load_limbs_case(name)
    lc = decoder.LimbsCollect(1, 1, topk=d['topk'], thre_hmp=d['thre_hmp'], min_len=d['min_len'],
                              keypoints=list(range(d['n_keypoints'])), skeleton=d['skeleton'])
    limbs = lc.generate_limbs(torch.from_numpy(d['heat']).cuda(), [], torch.from_numpy(d['offs']).cuda(), [])
    assert limbs.is_cuda and tuple(limbs.shape) == d['limbs'].shape
    got = limbs.cpu().numpy()
    assert gio.compare_limbs(got, d['limbs'], d['thre_hmp'], rtol=RTOL) > 100
    both = (d['limbs'][..., 2] >= np.float32(d['thre_hmp'])) & (d['limbs'][..., 5] >= np.float32(d['thre_hmp']))
    # distances follow ATen's fma formula: bit-exact
    assert np.array_equal(got[both][:, 8], d['limbs'][both][:, 8])
    assert np.array_equal(got[both][:, 9], d['limbs'][both][:, 9])


def test_k2_scale_maps_and_float32_ids(cuda_device):
    """include_scale gather (collect.py:111-116) and global ids above 2**24 stored as
    rounded float32 (SURVEY.md config 4)."""
    rng = np.random.RandomState(9)
    h, w = 1024, 1024
    skel = [(0, 16), (16, 1)]
    heat = np.zeros((1, 17, h, w), np.float32)
    offs = np.zeros((1, 4, h, w), np.float32)
    sc = rng.uniform(1, 30, size=(1, 17, h, w)).astype(np.float32)
    pts = rng.randint(5, 1000, size=(6, 2))
    for (x, y) in pts:
        heat[0, 0, y, x] = rng.uniform(0.3, 1)
        heat[0, 16, y + 3, x + 2] = rng.uniform(0.3, 1)
        heat[0, 1, y + 5, x - 3] = rng.uniform(0.3, 1)
        offs[0, 0, y, x], offs[0, 1, y, x] = 2.25, 2.75
        offs[0, 2, y + 3, x + 2], offs[0, 3, y + 3, x + 2] = -5.5, 2.5
    eng = DecoderEngine(17, skel, topk=8, thre_hmp=0.1, min_len=0.5)
    s, i, _ = eng.nms_topk(torch.from_numpy(heat).cuda())
    got = eng.limb_score(s, i, torch.from_numpy(offs).cuda(), torch.from_numpy(sc).cuda()).cpu().numpy()
    ref = ro.generate_limbs(heat, offs, skel, 8, 0.1, 0.5, 1, 1, scmps_hr=sc)
    assert gio.compare_limbs(got, ref, 0.1, rtol=RTOL) >= 10
    assert got[0, 1, :6, 6].max() > 2 ** 24       # ids of channel 16 exceed 2**24


# --------------------------------------------------------------------------- K3
def test_k3_group_fuzz_bit_exact(cuda_device):
    cases = gio.load_group_fuzz()
    for ci, c in enumerate(cases):
        g = decoder.GreedyGroup(c['person_thre'], sort_dim=c['sort_dim'], dist_max=40,
                                use_scale=c['use_scale'], keypoints=list(range(c['n_keypoints'])),
                                skeleton=c['skeleton'])
        got = g.group_skeletons(c['limbs'])
        assert got.dtype == np.float32
        assert got.shape == c['poses'].shape, f'case {ci}: person count {got.shape} vs {c["poses"].shape}'
        assert np.array_equal(got, c['poses']), f'case {ci}'


@pytest.mark.parametrize('name', ['limbs_coco_a', 'limbs_coco_noise', 'limbs_crowdpose'])
def test_k3_on_reference_limbs_bit_exact(cuda_device, name):
    d = gio.load_limbs_case(name)
    g = decoder.GreedyGroup(d['person_thre'], sort_dim=2, dist_max=d['dist_max'], use_scale=True,
                            keypoints=list(range(d['n_keypoints'])), skeleton=d['skeleton'])
    got = g.group_batch(d['limbs'])
    for p, r in zip(got, gio.split_poses(d['poses'], d['pose_counts'])):
        gio.compare_poses(p, r, exact=True)


def test_k3_random_tables_against_oracle(cuda_device):
    """Fresh seeded fuzz (not from the fixture), incl. pure-noise tables that outgrow the warp
    kernel's person table and are regrouped by the CTA kernel."""
    rng = np.random.RandomState(77)
    skel = cfg.COCO_PERSON_SKELETON
    for case in range(40):
        k = int(rng.choice([8, 32, 64]))
        pool = int(rng.choice([3, 8, 400]))
        limbs = np.zeros((19, k, 13), np.float32)
        xy = rng.randint(1, 600, size=(17, pool, 2)).astype(np.float32)
        ids = rng.randint(0, 640 * 640, size=(17, pool))
        for l, (jf, jt) in enumerate(skel):
            sc = (rng.permutation(k) + rng.uniform(0.1, 0.9, size=k)).astype(np.float32) / k
            for r in range(k):
                a, b = rng.randint(pool), rng.randint(pool)
                limbs[l, r] = (xy[jf, a, 0], xy[jf, a, 1], 0.5, xy[jt, b, 0], xy[jt, b, 1], 0.6,
                               ids[jf, a] + jf * 409600, ids[jt, b] + jt * 409600,
                               rng.uniform(0, 50), 10, sc[r], 4, 4)
        g = decoder.GreedyGroup(0.06, sort_dim=2, dist_max=40, use_scale=True)
        got = g.group_skeletons(limbs)
        ref = ro.group_skeletons(limbs, skel, 17, 0.06, 2, 40, True)
        assert got.shape == ref.shape and np.array_equal(got, ref), f'case {case} k={k} pool={pool}'


def test_k3_large_batch_with_warp_overflow_against_oracle(cuda_device):
    """A batch of 400 images, some of whose tables outgrow the warp kernel's person table and are
    regrouped by the CTA kernel: every image equals the oracle, as in a batch of 12."""
    rng = np.random.RandomState(123)
    skel = cfg.COCO_PERSON_SKELETON
    tables = []
    for case in range(12):
        k, pool = 32, int(rng.choice([4, 10, 400]))         # pool 400: ~100+ persons, outgrows 64 rows
        limbs = np.zeros((19, k, 13), np.float32)
        xy = rng.randint(1, 600, size=(17, pool, 2)).astype(np.float32)
        ids = rng.randint(0, 640 * 640, size=(17, pool))
        for l, (jf, jt) in enumerate(skel):
            sc = (rng.permutation(k) + rng.uniform(0.1, 0.9, size=k)).astype(np.float32) / k
            for r in range(k):
                a, b = rng.randint(pool), rng.randint(pool)
                limbs[l, r] = (xy[jf, a, 0], xy[jf, a, 1], 0.5, xy[jt, b, 0], xy[jt, b, 1], 0.6,
                               ids[jf, a] + jf * 409600, ids[jt, b] + jt * 409600,
                               rng.uniform(0, 50), 10, sc[r], 4, 4)
        tables.append(limbs)
    g = decoder.GreedyGroup(0.06, sort_dim=2, dist_max=40, use_scale=True)
    small = g.group_batch(np.stack(tables))
    ref = [ro.group_skeletons(t, skel, 17, 0.06, 2, 40, True) for t in tables]
    assert max(len(r) for r in ref) > 100
    for a, r in zip(small, ref):
        assert a.shape == r.shape and np.array_equal(a, r)
    order = rng.randint(0, len(tables), size=400)
    big = g.group_batch(np.stack([tables[i] for i in order]))
    assert len(big) == 400
    for got, i in zip(big, order):
        assert got.shape == ref[i].shape and np.array_equal(got, ref[i])


def _random_limb_tables(rng, count, skel, n_kp):
    """Limb tables with tiny keypoint pools: persons share ids, kept rows start at the same joint,
    slots are overwritten — everything the merge step of group.py:140-155 can meet."""
    tables = []
    for _ in range(count):
        k = int(rng.choice([4, 8, 16, 32]))
        pool = int(rng.choice([2, 3, 4, 5, 6, 8, 12, 20]))
        limbs = np.zeros((len(skel), 32, 13), np.float32)
        xy = rng.randint(1, 600, size=(n_kp, pool, 2)).astype(np.float32)
        ids = rng.randint(0, 640 * 640, size=(n_kp, pool))
        for l, (jf, jt) in enumerate(skel):
            sc = (rng.permutation(k) + rng.uniform(0.1, 0.9, size=k)).astype(np.float32) / k
            for r in range(k):
                a, b = rng.randint(pool), rng.randint(pool)
                limbs[l, r] = (xy[jf, a, 0], xy[jf, a, 1], 0.5, xy[jt, b, 0], xy[jt, b, 1], 0.6,
                               ids[jf, a] + jf * 409600, ids[jt, b] + jt * 409600,
                               rng.uniform(0, 55), 10, sc[r], 4, 4)
            limbs[l, k:, 8] = 1000.0                       # rows beyond k fail the distance gate
        tables.append(limbs)
    return np.stack(tables)


def test_k3_warp_kernel_skips_no_merge(cuda_device, monkeypatch):
    """The one-warp kernel runs the all-pairs merge test only in steps where a pair's number of
    shared ids can have changed; the CTA kernel runs it in every step like the reference.  2000
    random tables with tiny keypoint pools (shared ids, duplicate from-joints, overwritten slots,
    cancellation persons) must come out identically from both, and a sample equals the oracle."""
    rng = np.random.RandomState(2025)
    skel = cfg.COCO_PERSON_SKELETON
    tables = _random_limb_tables(rng, 2000, skel, 17)
    warp = decoder.GreedyGroup(0.06, sort_dim=2, dist_max=40, use_scale=True).group_batch(tables)
    monkeypatch.setenv('OG_K3_WARP_ROWS', '0')
    cta = decoder.GreedyGroup(0.06, sort_dim=2, dist_max=40, use_scale=True).group_batch(tables)
    merged = 0
    for i, (a, b) in enumerate(zip(warp, cta)):
        assert a.shape == b.shape and np.array_equal(a, b), f'table {i}'
    for i in range(0, 2000, 40):
        ref = ro.group_skeletons(tables[i], skel, 17, 0.06, 2, 40, True)
        assert warp[i].shape == ref.shape and np.array_equal(warp[i], ref), f'table {i}'
        merged += 1
    assert merged == 50


def test_k3_empty_and_degenerate(cuda_device):
    g = decoder.GreedyGroup(0.06, sort_dim=2, dist_max=40, use_scale=False)
    out = g.group_skeletons(np.zeros((19, 4, 13), np.float32))
    assert out.shape == (0, 17, 6) and out.dtype == np.float32
    with pytest.raises(AssertionError):
        g.group_skeletons(np.zeros((18, 4, 13), np.float32))


# --------------------------------------------------------------------------- maps
def test_resize_and_flip_bit_exact(cuda_device):
    from offsetguided_b200 import _lib
    from offsetguided_b200.engine import _ptr, _stream_ptr
    lib = _lib.load()
    d = gio.load('resize_small')
    for key, xk, scale, mode in (('bicubic4', 'x', 4, 1), ('bilinear4', 'x', 4, 0),
                                 ('bicubic2', 'x2', 2, 1), ('bilinear2', 'x2', 2, 0),
                                 ('bicubic8', 'x8', 8, 1), ('bilinear8', 'x8', 8, 0)):
        x = torch.from_numpy(d[xk]).cuda()
        n, c, h, w = x.shape
        out = torch.empty((n, c, h * scale, w * scale), device='cuda')
        _lib.check(lib.og_resize_f32(_ptr(x), _ptr(out), n * c, h, w, scale, mode, _stream_ptr(x.device)))
        assert np.array_equal(out.cpu().numpy(), d[key]), key      # == ATen CPU, bit for bit
    # flip fusion vs the oracle
    rng = np.random.RandomState(2)
    hm = rng.uniform(0, 1, size=(4, 17, 12, 20)).astype(np.float32)
    om = rng.uniform(-9, 9, size=(4, 38, 12, 20)).astype(np.float32)
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, cfg.COCO_PERSON_SKELETON)
    eng = DecoderEngine(17, cfg.COCO_PERSON_SKELETON, topk=4)
    fh = torch.empty((2, 17, 12, 20), device='cuda')
    fo = torch.empty((2, 38, 12, 20), device='cuda')
    hm_d, om_d = torch.from_numpy(hm).cuda(), torch.from_numpy(om).cuda()
    _lib.check(lib.og_flip_fuse_f32(eng._h, _ptr(hm_d), _ptr(om_d),
                                    _lib.int32_array(kp), _lib.int32_array(fl), _lib.int32_array(rs), len(rs),
                                    2, 12, 20, _ptr(fh), _ptr(fo), _stream_ptr(fh.device)))
    rh, rr = ro.flip_augment(hm, om, kp, fl, rs)
    assert np.array_equal(fh.cpu().numpy(), rh) and np.array_equal(fo.cpu().numpy(), rr)


def test_flip_augment_method_matches_reference_semantics(cuda_device):
    """PostProcess.flip_augment keeps the reference's signature and return tuple
    (decoder/factory.py:98-146): default branch against the oracle, cat_flip_offs branch against
    the reference's own tensor expressions."""
    rng = np.random.RandomState(8)
    n, h, w = 2, 12, 20
    hm = rng.uniform(0, 1, size=(2 * n, 17, h, w)).astype(np.float32)
    om = rng.uniform(-9, 9, size=(2 * n, 38, h, w)).astype(np.float32)
    pp = decoder.decoder_factory(_args())
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, cfg.COCO_PERSON_SKELETON)
    th, to = torch.from_numpy(hm).cuda(), torch.from_numpy(om).cuda()
    fh, fj, fo, fs, nd = pp.flip_augment(th, [], to, [], False, 2)
    rh, ro_ = ro.flip_augment(hm, om, kp, fl, rs)
    assert nd == 2 and fj == [] and fs == []
    assert np.array_equal(fh.cpu().numpy(), rh) and np.array_equal(fo.cpu().numpy(), ro_)
    ch, _, co_, _, nd = pp.flip_augment(th, [], to, [], True, 2)
    o5 = torch.from_numpy(om).view(2 * n, -1, 2, h, w)
    orig = o5[:n]
    reserve = o5[:n, rs].clone()
    flip = torch.flip(o5[n:], [-1]).clone()
    flip[:, :, ::2] *= -1.0
    cat = torch.cat((orig, flip[:, fl]), dim=2)
    cat[:, rs, 2:] = reserve
    assert nd == 4 and np.array_equal(co_.cpu().numpy(), cat.reshape(n, -1, h, w).numpy())
    assert np.array_equal(ch.cpu().numpy(), rh)
    assert th.shape[0] == 2 * n and np.array_equal(th.cpu().numpy(), hm)          # inputs untouched


def test_scored_offset_matches_reference(cuda_device):
    """decoder.scored_offset against the reference's own output (tests/golden/scored_offset.npz,
    decoder/offset.py:8-43), k = 3 (the call site) and 7 (the default); 1e-5 relative."""
    d = gio.load('scored_offset')
    jf, jt = ro.pack_jtypes(cfg.COCO_PERSON_SKELETON)
    for tag in ('a', 'b'):
        hm, om = torch.from_numpy(d['hmp_' + tag]).cuda(), torch.from_numpy(d['off_' + tag]).cuda()
        for ks in (3, 7):
            got = decoder.scored_offset(hm, om, jf, jt, ks).cpu().numpy()
            ref = d['out_%s_k%d' % (tag, ks)]
            np.testing.assert_allclose(got, ref, rtol=RTOL, atol=1e-6)
            assert np.array_equal(got, ro.scored_offset(d['hmp_' + tag], d['off_' + tag], jf, jt, ks))


# --------------------------------------------------------------------------- whole path
@pytest.mark.parametrize('name', ['limbs_coco_a', 'limbs_coco_noise', 'limbs_crowdpose'])
def test_decode_maps_matches_reference(cuda_device, name):
    d = gio.load_limbs_case(name)
    eng = _engine(d, d['n_keypoints'], d['skeleton'])
    poses = eng.decode_maps(torch.from_numpy(d['heat']).cuda(), torch.from_numpy(d['offs']).cuda())
    ref = gio.split_poses(d['poses'], d['pose_counts'])
    assert len(poses) == len(ref)
    for p, r in zip(poses, ref):
        gio.compare_poses(p, r, rtol=RTOL)


def _args(**over):
    import argparse
    p = argparse.ArgumentParser()
    decoder.decoder_cli(p)
    a = p.parse_args([])
    a.headnets, a.strides, a.batch_size = ['hmp', 'omp'], [4, 4], 8
    a.include_scale = a.include_jitter_offset = False
    for k, v in over.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize('name,host', [('poses_cfg1', False), ('poses_cfg2_flip', False),
                                       ('poses_cfg1', True), ('poses_cfg2_flip', True),
                                       ('poses_inf_background', False), ('poses_inf_background', True),
                                       ('poses_inf_background_flip', False),
                                       ('poses_inf_background_flip', True),
                                       ('poses_bilinear_flip', False), ('poses_bilinear_flip', True)])
def test_generate_poses_matches_reference(cuda_device, name, host):
    """BASELINE configs 1 and 2 through the reference-facing API, device and host inputs."""
    d = gio.load_poses_case(name)
    pp = decoder.decoder_factory(_args(topk=d['topk'], thre_hmp=d['thre_hmp'], person_thre=d['person_thre'],
                                       dist_max=d['dist_max'], resize_mode=d['resize_mode']))
    hmp, omp = torch.from_numpy(d['hmp']), torch.from_numpy(d['omp'])
    if host:
        hmp, omp = hmp.pin_memory(), omp.pin_memory()
    else:
        hmp, omp = hmp.cuda(), omp.cuda()
    feats = [[[hmp], [[]], [[]]], [[omp], [[]], [[]]]]
    poses = pp.generate_poses(feats, flip_test=d['flip_test'])
    ref = gio.split_poses(d['poses'], d['pose_counts'])
    assert len(poses) == len(ref)
    lr, da, pr = gio.tolerances(name, RTOL)
    for p, r in zip(poses, ref):
        assert p.dtype == np.float32
        gio.compare_poses(p, r, rtol=pr)
    n = len(ref)
    ds, di, lb = pp._engine(torch.device('cuda', 0)).last_intermediates(n)
    live = d['det_scores'] >= np.float32(d['thre_hmp'])
    assert np.array_equal(di.cpu().numpy()[live], d['det_inds'][live])         # bit-exact peaks
    assert np.array_equal(ds.cpu().numpy()[live], d['det_scores'][live])       # after bicubic x4
    assert gio.compare_limbs(lb.cpu().numpy(), d['limbs'], d['thre_hmp'], rtol=lr, dist_atol=da) > 50


def test_generate_poses_scored_off_and_last_partial_batch(cuda_device):
    d = gio.load_poses_case('poses_cfg2_flip')
    pp = decoder.decoder_factory(_args(topk=32, thre_hmp=0.04, person_thre=0.04, dist_max=40))
    hmp, omp = torch.from_numpy(d['hmp']).cuda(), torch.from_numpy(d['omp']).cuda()
    feats = [[[hmp], [[]], [[]]], [[omp], [[]], [[]]]]
    got = pp.generate_poses(feats, flip_test=True, scored_off=True)
    # the reference's own generate_poses(flip_test=True, scored_off=True) on these inputs
    s = gio.load('poses_scored_off')
    ref = gio.split_poses(s['poses'], s['pose_counts'])
    assert len(got) == len(ref) == 2
    for p, r in zip(got, ref):
        gio.compare_poses(p, r, rtol=RTOL)
    # a smaller last batch through the same PostProcess
    feats1 = [[[hmp[[0, 2]]], [[]], [[]]], [[omp[[0, 2]]], [[]], [[]]]]
    one = pp.generate_poses(feats1, flip_test=True)
    two = pp.generate_poses(feats, flip_test=True)
    assert len(one) == 1 and np.array_equal(one[0], two[0])


def test_decode_full_size_properties(cuda_device):
    """BASELINE sizes (640x640, batch 8): oracle comparison on 2 images plus
    size-independent properties on all: determinism, batch-order equivariance,
    dets sorted, persons sorted by score."""
    skel = cfg.COCO_PERSON_SKELETON
    heat, offs = scenes.synth_hires_batch(123, 8, 6, 640, 640, skel)
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, min_len=0.5, dist_max=40,
                        use_scale=True, person_thre=0.04)
    th, to = torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda()
    poses = eng.decode_maps(th, to)
    ds, di, lb = eng.last_intermediates(8)
    again = eng.decode_maps(th, to)
    perm = [3, 1, 7, 0, 5, 2, 6, 4]
    shuffled = eng.decode_maps(th[perm], to[perm])
    for i in range(8):
        assert np.array_equal(poses[i], again[i])
        assert np.array_equal(shuffled[i], poses[perm[i]])
        v = poses[i][:, :, 2]
        sc = np.array([r[r > 0].mean() for r in v])
        assert np.all(np.diff(sc) <= 1e-6)
        assert len(poses[i]) >= 5
    s = ds.cpu().numpy()
    assert np.all(np.diff(s, axis=-1) <= 0)
    ref_limbs = ro.generate_limbs(heat[:2], offs[:2], skel, 32, 0.04, 0.5, 1, 1)
    assert gio.compare_limbs(lb.cpu().numpy()[:2], ref_limbs, 0.04, rtol=RTOL) > 150
    for i in range(2):
        ref = ro.group_skeletons(ref_limbs[i], skel, 17, 0.04, 2, 40, True)
        gio.compare_poses(poses[i], ref, rtol=RTOL)


# --------------------------------------------------------------------------- fused path
@pytest.mark.parametrize('shape,stride,mode,flip', [
    ((2, 40, 56), 4, 'bicubic', False), ((2, 45, 70), 4, 'bicubic', True),
    ((1, 33, 31), 2, 'bicubic', False), ((2, 48, 64), 4, 'bilinear', True),
    ((1, 20, 24), 8, 'bicubic', True), ((1, 17, 35), 4, 'bicubic', False)])
def test_fused_path_equals_materialising_path(cuda_device, shape, stride, mode, flip):
    """flip fusion + resize + NMS fused over network-resolution maps must give the very same
    dets, limbs and poses as flip -> resize -> K1 on materialised maps (bit for bit)."""
    n, h, w = shape
    skel = cfg.COCO_PERSON_SKELETON
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    W, H = w * 4, h * 4                      # scenes are rendered for a stride-4 network
    hs, os_ = [], []
    for half in range(2 if flip else 1):
        for i in range(n):
            rng = np.random.RandomState(100 * h + i)
            p = scenes.make_persons(rng, 3, W, H, scale_range=(W / 40.0, W / 24.0))
            if half:
                p = scenes.mirror_persons(p, W, kp)
            hm = scenes.render_heatmaps(p, W, H) + rng.uniform(0, 0.02, size=(17, h, w)).astype(np.float32)
            om = scenes.render_offsets(p, W, H, skel)
            om[~np.isfinite(om)] = 0
            hs.append(hm)
            os_.append(om)
    hmp = torch.from_numpy(np.stack(hs).astype(np.float32)).cuda()
    omp = torch.from_numpy(np.stack(os_).astype(np.float32)).cuda()
    tables = (kp, fl, rs) if flip else None
    eng = DecoderEngine(17, skel, topk=16, thre_hmp=0.05, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.05)
    fused = eng.decode_features(hmp, omp, stride, stride, mode, tables)
    f_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    assert eng.fused_redo_count == 0
    eng.set_fused(False)
    staged = eng.decode_features(hmp, omp, stride, stride, mode, tables)
    s_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    assert sum(len(p) for p in staged) >= 1
    for a, b in zip(f_int, s_int):
        assert np.array_equal(a, b)
    for a, b in zip(fused, staged):
        assert np.array_equal(a, b)
    # and against the oracle
    ref = ro.generate_poses(np.stack(hs), np.stack(os_), skel, 17, topk=16, thre_hmp=0.05, min_len=0.5,
                            person_thre=0.05, dist_max=40, use_scale=True, hmp_stride=stride,
                            off_stride=stride, resize_mode=mode, flip_test=flip, kp_flips=kp,
                            limb_flips=fl, limb_reserve=rs)
    for p, r in zip(fused, ref):
        gio.compare_poses(p, r, rtol=RTOL)


@pytest.mark.parametrize('stride,mode,flip', [(4, 'bicubic', False), (4, 'bicubic', True), (2, 'bicubic', False),
                                              (8, 'bicubic', True), (4, 'bilinear', False), (2, 'bilinear', True),
                                              (8, 'bilinear', False)])
def test_fused_candidates_at_block_and_image_borders(cuda_device, stride, mode, flip):
    """K1f corner cases, compared with flip -> resize -> K1 on the materialised map: spikes on both
    sides of every work-block boundary (the 3 x 3 test then needs the pixel ring outside the block,
    lanes 0 / 31 and the rows above / below), in the image corners and on the borders (tap clamping,
    bilinear's src < 0 clamp, zero padding of the NMS window), 2-cell plateaus straddling a boundary
    (tied peaks in two blocks), values that land exactly on the threshold, and negative lobes."""
    h, w = 37, 70
    bw = 32 // stride                       # cells per work block along x; 8 cell rows per block
    rng = np.random.RandomState(stride * 7 + len(mode))
    n_in = 4 if flip else 2
    hmp = np.zeros((n_in, 17, h, w), np.float32)
    for img in range(n_in):
        for c in range(17):
            pts = [(0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (0, w // 2), (h // 2, 0), (h - 1, 5), (9, w - 1)]
            for by in (8, 16, 24, 32):
                for bx in range(bw, w, bw):
                    pts.append((by - 1 if rng.rand() < 0.5 else by, bx - 1 if rng.rand() < 0.5 else bx))
            picks = [pts[i] for i in rng.choice(len(pts), size=10, replace=False)]
            for (y, x) in picks:
                hmp[img, c, y, x] = rng.uniform(0.3, 1.0)
            # plateaus across a vertical and a horizontal block boundary
            hmp[img, c, 20, bw - 1:bw + 1] = 0.625
            hmp[img, c, 15:17, 3 * bw // 2] = 0.75
            hmp[img, c, 28, 40] = -0.5                       # negative lobe next to positives
            hmp[img, c, 28, 41] = 0.5
    hmp[0, 0] = 0
    hmp[0, 0, 12, 12] = 0.05                                 # an exact-threshold plane (see thre below)
    omp = np.zeros((n_in, 38, h, w), np.float32)
    skel = cfg.COCO_PERSON_SKELETON
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    tables = (kp, fl, rs) if flip else None
    # threshold = the exact interpolated peak value of plane (0, 0), so ">= thre" is hit with equality
    up = co_resize_plane(hmp, kp, flip, stride, mode)
    thre = float(up.max())
    assert 0.01 < thre < 0.6
    eng = DecoderEngine(17, skel, topk=64, thre_hmp=thre, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.05)
    th, to = torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()
    eng.decode_features(th, to, stride, stride, mode, tables)
    assert eng.fused_redo_count == 0
    f_s, f_i, _ = [t.cpu().numpy() for t in eng.last_intermediates(n_in // 2 if flip else n_in)]
    eng.set_fused(False)
    eng.decode_features(th, to, stride, stride, mode, tables)
    s_s, s_i, _ = [t.cpu().numpy() for t in eng.last_intermediates(n_in // 2 if flip else n_in)]
    assert (s_i >= 0).sum() > 17 * 4
    assert np.array_equal(f_i, s_i) and np.array_equal(f_s, s_s)
    assert (f_s[0, 0] == np.float32(thre)).any()              # the equality case was really exercised


def co_resize_plane(hmp, kp, flip, stride, mode):
    """Full-resolution values of plane (image 0, channel 0) as the reference computes them."""
    from oracle import c_oracle as co
    n = hmp.shape[0] // 2 if flip else hmp.shape[0]
    plane = hmp[:1, :1].copy()
    if flip:
        plane = ((hmp[:1, :1] + hmp[n:n + 1, kp[0]:kp[0] + 1, :, ::-1]) * np.float32(0.5)).astype(np.float32)
    return co.resize(np.ascontiguousarray(plane), stride, mode)[0, 0]


def test_random_maps_small_skeleton_full_decode(cuda_device):
    """Random full decodes with a 4-keypoint / 4-limb skeleton and its own flip tables (nothing
    COCO-specific in the kernels): fused path against the numpy oracle, strides 2 / 4, both resize
    modes, plateaus, negative border values."""
    rng = np.random.RandomState(11)
    skel = [(0, 1), (1, 2), (0, 2), (2, 3)]
    kp_flips, limb_flips, limb_reserve = [0, 2, 1, 3], [2, 1, 0, 3], [1]
    for case in range(6):
        stride = int(rng.choice([2, 4]))
        mode = str(rng.choice(['bicubic', 'bilinear']))
        flip = bool(case % 2)
        n, h, w = 2, int(rng.randint(20, 30)), int(rng.randint(40, 52))
        hmp = np.zeros((2 * n if flip else n, 4, h, w), np.float32)
        for img in range(hmp.shape[0]):
            for c in range(4):
                for _ in range(5):
                    y, x = rng.randint(0, h), rng.randint(0, w)
                    hmp[img, c, y, x] = rng.uniform(0.2, 1.0)
                hmp[img, c, 3, 5:7] = 0.5
        hmp[:, :, 0, :] -= rng.uniform(0, 0.3, size=(hmp.shape[0], 4, w)).astype(np.float32)
        omp = rng.uniform(-12, 12, size=(hmp.shape[0], 8, h, w)).astype(np.float32)
        eng = DecoderEngine(4, skel, topk=8, thre_hmp=0.1, min_len=0.5, dist_max=30.0, use_scale=True,
                            person_thre=0.1)
        tables = (kp_flips, limb_flips, limb_reserve) if flip else None
        got = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), stride, stride,
                                  mode, tables)
        assert eng.fused_redo_count == 0
        _, _, lb = eng.last_intermediates(n)
        ref, ref_limbs = ro.generate_poses(hmp, omp, skel, 4, topk=8, thre_hmp=0.1, min_len=0.5, person_thre=0.1,
                                           dist_max=30.0, use_scale=True, hmp_stride=stride, off_stride=stride,
                                           resize_mode=mode, flip_test=flip, kp_flips=kp_flips,
                                           limb_flips=limb_flips, limb_reserve=limb_reserve, return_limbs=True)
        assert gio.compare_limbs(lb.cpu().numpy(), ref_limbs, 0.1, rtol=RTOL) >= 4, case
        assert sum(len(p) for p in ref) >= 2
        _pose_lists_equal(got, ref)
        eng.close()


@pytest.mark.parametrize('thre', [0.0, -1.0])
def test_non_positive_threshold_takes_the_exact_path(cuda_device, thre):
    """thre_hmp <= 0 makes every NMS survivor (also the zero plateau) a candidate: the fused path is
    not eligible, the materialising path selects with the exact radix selection, and the result
    equals the oracle's top-K with its canonical tie order."""
    skel = cfg.COCO_PERSON_SKELETON
    hmp, omp = scenes.render_batch(77, 2, 3, 256, 192, skel)
    eng = DecoderEngine(17, skel, topk=16, thre_hmp=thre, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.05)
    got = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), 4, 4, 'bicubic', None)
    ds, di, _ = [t.cpu().numpy() for t in eng.last_intermediates(2)]
    ref = ro.generate_poses(hmp, omp, skel, 17, topk=16, thre_hmp=thre, min_len=0.5, person_thre=0.05,
                            dist_max=40, use_scale=True)
    heat = ro.resize(hmp, 4, 'bicubic')
    rs, ri, _, _ = ro.topk_channel(ro.hmp_nms(heat), 16)
    assert np.array_equal(di, ri) and np.array_equal(ds, rs)
    assert sum(len(p) for p in ref) >= 4
    _pose_lists_equal(got, ref)


def test_fused_path_overflow_reruns_exactly(cuda_device):
    """Noise heat maps overflow the per-plane candidate lists; the overflowed planes are then
    materialised and selected exactly when the batch is fetched, and the result must equal the
    materialising path."""
    rng = np.random.RandomState(3)
    hmp = torch.from_numpy(rng.uniform(0, 1, size=(1, 17, 160, 200)).astype(np.float32)).cuda()
    omp = torch.from_numpy(rng.uniform(-8, 8, size=(1, 38, 160, 200)).astype(np.float32)).cuda()
    eng = DecoderEngine(17, cfg.COCO_PERSON_SKELETON, topk=32, thre_hmp=0.04, dist_max=40,
                        use_scale=True, person_thre=0.04)
    fused = eng.decode_features(hmp, omp, 4, 4, 'bicubic', None)
    assert eng.fused_redo_count == 1
    f_int = [t.cpu().numpy() for t in eng.last_intermediates(1)]
    eng.set_fused(False)
    staged = eng.decode_features(hmp, omp, 4, 4, 'bicubic', None)
    s_int = [t.cpu().numpy() for t in eng.last_intermediates(1)]
    for a, b in zip(f_int, s_int):
        assert np.array_equal(a, b)
    assert np.array_equal(fused[0], staged[0]) and len(fused[0]) > 10


@pytest.mark.parametrize('flip', [False, True])
def test_fused_path_redoes_only_the_overflowed_planes(cuda_device, flip):
    """One noisy plane in a clean batch (flip-test too: its mirrored partner is another channel of
    the second half): the fetch materialises that plane alone, the dets of every other plane are
    the fused kernel's, and dets / limbs / poses equal the materialising path."""
    import bench
    skel = cfg.COCO_PERSON_SKELETON
    hmp, omp = bench.lowres_inputs(777, 3, 640, flip)
    rng = np.random.RandomState(9)
    hmp[1, 5] = rng.uniform(0, 1, size=hmp.shape[2:]).astype(np.float32)
    tables = (cfg.heatmap_hflip(cfg.COCO_KEYPOINTS),) + tuple(cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)) if flip else None
    th, to = torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, dist_max=40, use_scale=True, person_thre=0.04)
    l0 = eng.launch_count
    fused = eng.decode_features(th, to, 4, 4, 'bicubic', tables)
    # K1f x3, select, K2, K3 + the redo: fuse, resize, radix select of ONE plane, K2, K3
    assert eng.fused_redo_count == 1 and eng.launch_count - l0 == 6 + 5
    f_int = [t.cpu().numpy() for t in eng.last_intermediates(3)]
    eng.set_fused(False)
    staged = eng.decode_features(th, to, 4, 4, 'bicubic', tables)
    s_int = [t.cpu().numpy() for t in eng.last_intermediates(3)]
    for a, b in zip(f_int, s_int):
        assert np.array_equal(a, b)
    assert sum(len(p) for p in fused) >= 6
    for a, b in zip(fused, staged):
        assert np.array_equal(a, b)


def test_overflow_redo_after_graph_replay_reads_the_calls_own_buffers(cuda_device):
    """A result slot replays the graph captured for buffers A after it has served buffers B in
    between; when that replay overflows a plane, the redo at fetch time must materialise the plane
    from A (the call's own buffers), not from whatever the slot decoded last."""
    import bench
    skel = cfg.COCO_PERSON_SKELETON
    (ha, oa), (hb, ob) = bench.lowres_inputs(31, 2, 640, False), bench.lowres_inputs(32, 2, 640, False)
    a_h, a_o = torch.from_numpy(ha).cuda(), torch.from_numpy(oa).cuda()
    b_h, b_o = torch.from_numpy(hb).cuda(), torch.from_numpy(ob).cuda()
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, dist_max=40, use_scale=True, person_thre=0.04)
    eng.decode_features(a_h, a_o, 4, 4, 'bicubic', None)          # captures the chain for A
    eng.decode_features(b_h, b_o, 4, 4, 'bicubic', None)          # the same slot now serves B
    assert eng.fused_redo_count == 0
    rng = np.random.RandomState(4)
    a_h[1, 3] = torch.from_numpy(rng.uniform(0, 1, size=ha.shape[2:]).astype(np.float32)).cuda()
    replays = eng.graph_counts[0]
    got = eng.decode_features(a_h, a_o, 4, 4, 'bicubic', None)    # replay of A's graph, plane (1, 3) overflows
    assert eng.graph_counts[0] == replays + 1 and eng.fused_redo_count == 1
    g_int = [t.cpu().numpy() for t in eng.last_intermediates(2)]
    eng.set_fused(False)
    ref = eng.decode_features(a_h, a_o, 4, 4, 'bicubic', None)
    r_int = [t.cpu().numpy() for t in eng.last_intermediates(2)]
    for x, y in zip(g_int, r_int):
        assert np.array_equal(x, y)
    for x, y in zip(got, ref):
        assert np.array_equal(x, y)


def test_device_call_after_host_call_on_the_same_slot(cuda_device):
    """A result slot serves a host-maps call (several image ranges, counters cleared by memsets) and
    then a device-maps call (one chain that expects its counters at zero): the second call must not
    see the active-block count the first one left behind (found by profiles/tools/soak.py)."""
    import bench
    skel = cfg.COCO_PERSON_SKELETON
    tables = (cfg.heatmap_hflip(cfg.COCO_KEYPOINTS),) + tuple(cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel))
    hmp, omp = bench.lowres_inputs(808, 16, 320, True)
    th_d, to_d = torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()
    th_h, to_h = torch.from_numpy(hmp).pin_memory(), torch.from_numpy(omp).pin_memory()
    kw = dict(topk=32, thre_hmp=0.04, dist_max=40, use_scale=True, person_thre=0.04)
    ref = DecoderEngine(17, skel, **kw).decode_features(th_d, to_d, 4, 4, 'bicubic', tables)
    assert sum(len(p) for p in ref) >= 16 * 4
    eng = DecoderEngine(17, skel, **kw)
    for rep in range(3):
        host = eng.decode_features(th_h, to_h, 4, 4, 'bicubic', tables)
        dev = eng.decode_features(th_d, to_d, 4, 4, 'bicubic', tables)        # captured, then replayed
        for a, b, r in zip(host, dev, ref):
            assert np.array_equal(a, r) and np.array_equal(b, r), rep


def test_host_offsets_stay_on_the_host(cuda_device):
    """Host API, fused path: pinned offset maps are not copied (K2 gathers its samples over
    PCIe); pageable maps are copied as a whole; after a candidate overflow the overflowed planes
    are redone exactly and K2 samples the host-resident offsets once more.  All three give the
    results of the device-resident call."""
    import bench
    skel = cfg.COCO_PERSON_SKELETON
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    hmp, omp = bench.lowres_inputs(777, 3, 320, True)
    th, to = torch.from_numpy(hmp), torch.from_numpy(omp)
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, dist_max=40, use_scale=True, person_thre=0.04)
    ref = eng.decode_features(th.cuda(), to.cuda(), 4, 4, 'bicubic', (kp, fl, rs))
    ref_int = [t.cpu().numpy() for t in eng.last_intermediates(3)]
    assert sum(len(p) for p in ref) >= 12 and eng.zero_copy_count == 0
    pinned = eng.decode_features(th.pin_memory(), to.pin_memory(), 4, 4, 'bicubic', (kp, fl, rs))
    pin_int = [t.cpu().numpy() for t in eng.last_intermediates(3)]
    assert eng.zero_copy_count == 1
    pageable = eng.decode_features(th, to, 4, 4, 'bicubic', (kp, fl, rs))
    assert eng.zero_copy_count == 1
    eng.set_zero_copy(False)
    copied = eng.decode_features(th.pin_memory(), to.pin_memory(), 4, 4, 'bicubic', (kp, fl, rs))
    assert eng.zero_copy_count == 1 and eng.fused_redo_count == 0
    for a, b in zip(ref_int, pin_int):
        assert np.array_equal(a, b)
    for r, a, b, c in zip(ref, pinned, pageable, copied):
        assert np.array_equal(r, a) and np.array_equal(r, b) and np.array_equal(r, c)
    # overflow of the candidate lists with the offsets still on the host
    eng.set_zero_copy(True)
    rng = np.random.RandomState(5)
    nh = torch.from_numpy(rng.uniform(0, 1, size=(1, 17, 160, 200)).astype(np.float32))
    no = torch.from_numpy(rng.uniform(-8, 8, size=(1, 38, 160, 200)).astype(np.float32))
    over = eng.decode_features(nh.pin_memory(), no.pin_memory(), 4, 4, 'bicubic', None)
    assert eng.fused_redo_count == 1 and eng.zero_copy_count == 2
    eng.set_fused(False)
    staged = eng.decode_features(nh.cuda(), no.cuda(), 4, 4, 'bicubic', None)
    assert np.array_equal(over[0], staged[0]) and len(over[0]) > 5


@pytest.mark.parametrize('dtype,flip', [('bf16', True), ('bf16', False), ('f32', True), ('f16', True)])
def test_packed_head_output_decoded_in_place(cuda_device, dtype, flip):
    """SURVEY 8f-4 / BASELINE config 5 hand-over: one packed [2N, 17 + 38, h, w] head output, bf16 or
    float32, its two channel slices decoded in place (no split, no float32 copy).  A bf16 value
    widens exactly, so dets / limbs / poses equal those of the dense float32 copies bit for bit,
    and the oracle on the converted maps agrees."""
    import bench
    skel = cfg.COCO_PERSON_SKELETON
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    n = 3
    hmp, omp = bench.lowres_inputs(4321, n, 384, flip)
    packed = torch.from_numpy(np.concatenate((hmp, omp), axis=1)).cuda()
    if dtype != 'f32':
        packed = packed.to(torch.bfloat16 if dtype == 'bf16' else torch.float16)
    h_view, o_view = packed[:, :17], packed[:, 17:]
    assert not h_view.is_contiguous()
    pp = decoder.decoder_factory(_args(topk=32, thre_hmp=0.04, person_thre=0.04, dist_max=40))
    eng = pp._engine(torch.device('cuda', 0))
    feats = [[[h_view], [[]], [[]]], [[o_view], [[]], [[]]]]
    l0 = eng.launch_count
    got = pp.generate_poses(feats, flip_test=flip)
    assert eng.launch_count - l0 == 6          # K1f x3, select, K2, K3: no conversion kernel of ours
    got_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    h32, o32 = h_view.float().contiguous(), o_view.float().contiguous()
    ref = pp.generate_poses([[[h32], [[]], [[]]], [[o32], [[]], [[]]]], flip_test=flip)
    ref_int = [t.cpu().numpy() for t in eng.last_intermediates(n)]
    assert sum(len(p) for p in ref) >= 3 * 4
    for a, b in zip(got_int, ref_int):
        assert np.array_equal(a, b)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)
    orc = ro.generate_poses(h32.cpu().numpy(), o32.cpu().numpy(), skel, 17, topk=32, thre_hmp=0.04,
                            min_len=0.5, person_thre=0.04, dist_max=40, use_scale=True, hmp_stride=4,
                            off_stride=4, resize_mode='bicubic', flip_test=flip, kp_flips=kp,
                            limb_flips=fl, limb_reserve=rs)
    for p, r in zip(got, orc):
        gio.compare_poses(p, r, rtol=RTOL)


def test_config5_handover_batch32_bf16(cuda_device):
    """BASELINE config 5 per-GPU share (batch 256 over 8 GPUs = 32 images, flip-test: 64 network
    outputs): the hourglass head hands over one packed bf16 [64, 55, 160, 160] tensor.  With
    random-init weights (normal(0, 0.001), models/networks.py:147-173) the heat maps are ~0 and no
    person may come out; with persons rendered into the same tensor every image must decode as the
    float32 copies do (C oracle)."""
    import bench
    from oracle import c_oracle as co
    skel = cfg.COCO_PERSON_SKELETON
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    n = 32
    pp = decoder.decoder_factory(_args(topk=32, thre_hmp=0.04, person_thre=0.04, dist_max=40, batch_size=n))
    g = torch.Generator(device='cuda').manual_seed(5)
    empty = (torch.randn((2 * n, 55, 160, 160), generator=g, device='cuda') * 0.001).to(torch.bfloat16)
    out = pp.generate_poses([[[empty[:, :17]], [[]], [[]]], [[empty[:, 17:]], [[]], [[]]]], flip_test=True)
    assert len(out) == n and all(p.shape == (0, 17, 6) and p.dtype == np.float32 for p in out)
    hmp, omp = bench.lowres_inputs(31337, n, 640, True)
    packed = torch.from_numpy(np.concatenate((hmp, omp), axis=1)).cuda().to(torch.bfloat16)
    got = pp.generate_poses([[[packed[:, :17]], [[]], [[]]], [[packed[:, 17:]], [[]], [[]]]], flip_test=True)
    wide = packed.float().cpu().numpy()
    ref = co.generate_poses(np.ascontiguousarray(wide[:, :17]), np.ascontiguousarray(wide[:, 17:]), skel, 17,
                            topk=32, thre_hmp=0.04, min_len=0.5, person_thre=0.04, dist_max=40.0,
                            use_scale=True, flip_test=True, kp_flips=kp, limb_flips=fl, limb_reserve=rs)
    assert sum(len(p) for p in ref) >= n * 4
    _pose_lists_equal(got, ref)


def test_bf16_overflow_redo_and_odd_shapes(cuda_device):
    """bf16 maps with an odd width (scalar loads) and a noise batch whose candidate lists overflow
    (exact redo after an on-device conversion to dense float32)."""
    skel = cfg.COCO_PERSON_SKELETON
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, dist_max=40, use_scale=True, person_thre=0.04)
    rng = np.random.RandomState(11)
    for shape, redo in (((2, 55, 37, 45), 0), ((1, 55, 160, 200), 1)):
        packed = torch.from_numpy(rng.uniform(0, 1, size=shape).astype(np.float32))
        packed[:, 17:] = packed[:, 17:] * 16 - 8
        if not redo:
            packed[:, :17] *= torch.from_numpy(rng.uniform(0, 1, size=(shape[0], 17) + shape[2:]) > 0.97)
        packed = packed.cuda().to(torch.bfloat16)
        r0 = eng.fused_redo_count
        got = eng.decode_features(packed[:, :17], packed[:, 17:], 4, 4, 'bicubic', None)
        assert eng.fused_redo_count - r0 == redo
        eng.set_fused(False)
        ref = eng.decode_features(packed[:, :17].float(), packed[:, 17:].float(), 4, 4, 'bicubic', None)
        eng.set_fused(True)
        assert sum(len(p) for p in ref) > 3
        for a, b in zip(got, ref):
            assert np.array_equal(a, b)


def test_dev_ex_argument_errors(cuda_device):
    """og_decode_features_dev_ex refuses what it cannot decode in place (loudly, no fallback):
    reduced-precision maps without the fused path, image strides shorter than an image, unknown
    element types; the Python mirror converts to dense float32 itself in the first case."""
    import ctypes
    from offsetguided_b200 import _lib
    from offsetguided_b200.engine import _ptr, _stream_ptr
    skel = cfg.COCO_PERSON_SKELETON
    eng = DecoderEngine(17, skel, topk=8, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    packed = torch.zeros((2, 55, 16, 24), dtype=torch.bfloat16, device='cuda')
    hv, ov = packed[:, :17], packed[:, 17:]

    def call(dtype, hs, os_, stride=4):
        return eng.lib.og_decode_features_dev_ex(eng._h, _ptr(hv), _ptr(ov), dtype, hs, os_, 2, 16, 24, stride,
                                                 stride, 1, 0, None, None, None, 0, _stream_ptr(eng.device))
    per = 55 * 16 * 24
    assert call(_lib.OG_DTYPE_BF16, per, per) == 0 and eng.fetch(2)[0].shape == (0, 17, 6)
    assert call(7, per, per) != 0 and b'dtype' in eng.lib.og_last_error()
    assert call(_lib.OG_DTYPE_BF16, 100, per) != 0 and b'hmp_image_stride' in eng.lib.og_last_error()
    assert call(_lib.OG_DTYPE_BF16, per, per, stride=3) != 0          # stride 3: no fused kernel
    eng.set_fused(False)
    assert call(_lib.OG_DTYPE_BF16, per, per) != 0 and b'fused path' in eng.lib.og_last_error()
    assert eng.pending == 0
    out = eng.decode_features(hv, ov, 4, 4, 'bicubic', None)           # mirror: dense float32 copy
    assert len(out) == 2 and out[0].shape == (0, 17, 6)


def test_handles_with_different_table_sizes_coexist(cuda_device):
    """K3's dynamic shared memory attribute is per kernel, not per handle: a handle with a small
    person table created later must not shrink it for an earlier, larger one."""
    skel = cfg.COCO_PERSON_SKELETON
    heat, offs = scenes.synth_hires_batch(99, 2, 4, 320, 256, skel)
    th, to = torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda()
    big = DecoderEngine(17, skel, topk=32, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    first = big.decode_maps(th, to)
    small = DecoderEngine(17, skel[:4], topk=2, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    small.decode_maps(th, to[:, :8].contiguous())
    again = big.decode_maps(th, to)
    for a, b in zip(first, again):
        assert np.array_equal(a, b)


def test_decodes_in_flight(cuda_device):
    """The handle queues up to OG_MAX_IN_FLIGHT decode calls; results come back oldest first and
    equal the synchronous results; one more un-fetched call is refused, and a synchronous call
    while others are pending raises instead of handing out somebody else's result."""
    from offsetguided_b200 import _lib
    skel = cfg.COCO_PERSON_SKELETON
    heat, offs = scenes.synth_hires_batch(321, 4, 4, 320, 256, skel)
    th, to = torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda()
    eng = DecoderEngine(17, skel, topk=16, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    eng.enable_stage_timing(True)
    cuts = [slice(0, 3), slice(3, 4), slice(1, 3), slice(0, 4), slice(2, 3), slice(0, 1), slice(1, 4), slice(0, 2)]
    cuts = (cuts * _lib.OG_MAX_IN_FLIGHT)[:_lib.OG_MAX_IN_FLIGHT]
    refs = [eng.decode_maps(th[c], to[c]) for c in cuts]
    assert eng.pending == 0
    for c in cuts:
        eng.decode_maps(th[c], to[c], fetch=False)
    assert eng.pending == _lib.OG_MAX_IN_FLIGHT
    with pytest.raises(_lib.OgError):
        eng.decode_maps(th[:1], to[:1], fetch=False)
    with pytest.raises(_lib.OgError):
        eng.decode_maps(th[:1], to[:1])                        # fetch=True behind pending calls
    got = [eng.fetch()]
    t_a = eng.last_stage_times_ms()
    eng.decode_maps(th[:0], to[:0], fetch=False)               # empty batch in the queue
    got += [eng.fetch() for _ in cuts[1:]]
    assert eng.fetch() == [] and eng.pending == 0
    for c, g, r in zip(cuts, got, refs):
        assert len(g) == len(r) == c.stop - c.start
        for a_, b_ in zip(g, r):
            assert np.array_equal(a_, b_)
    assert t_a['k1_stream'] > 0 and t_a['k3'] > 0
    with pytest.raises(_lib.OgError):
        eng.fetch()


def _lowres_scene(seed, n, flip, edge=320):
    """Network-resolution maps (stride 4) of n images, mirrored copies appended when flip."""
    kp = cfg.heatmap_hflip(cfg.COCO_KEYPOINTS)
    skel = cfg.COCO_PERSON_SKELETON
    hs, os_, hf, of = [], [], [], []
    for i in range(n):
        rng = np.random.RandomState(seed + i)
        p = scenes.make_persons(rng, 4, edge, edge, scale_range=(edge / 64.0, edge / 27.0))
        hs.append(scenes.render_heatmaps(p, edge, edge) + rng.uniform(0, 0.02, size=(17, edge // 4, edge // 4)).astype(np.float32))
        os_.append(scenes.render_offsets(p, edge, edge, skel))
        if flip:
            pf = scenes.mirror_persons(p, edge, kp)
            hf.append(scenes.render_heatmaps(pf, edge, edge))
            of.append(scenes.render_offsets(pf, edge, edge, skel))
    hmp = np.stack(hs + hf).astype(np.float32)
    omp = np.stack(os_ + of).astype(np.float32)
    omp[~np.isfinite(omp)] = 0
    return hmp, omp


def test_graph_replay_and_recapture(cuda_device):
    """Device path: the chain of a result slot is captured once and replayed while pointers and
    shapes stay the same; other buffers / batch sizes re-capture; every result equals the
    kernel-by-kernel launch (og_set_graph(0)) and the host path."""
    skel = cfg.COCO_PERSON_SKELETON
    tables = (cfg.heatmap_hflip(cfg.COCO_KEYPOINTS),) + tuple(cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel))
    hmp, omp = _lowres_scene(77, 3, True)
    hd, od = torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()
    eng = DecoderEngine(17, skel, topk=16, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    eng.set_graph(False)
    ref = eng.decode_features(hd, od, 4, 4, 'bicubic', tables)
    assert sum(len(p) for p in ref) >= 6 and eng.graph_counts == (0, 0)
    eng.set_graph(True)
    for _ in range(17):                             # a synchronous caller stays on one slot: one capture, then replays
        got = eng.decode_features(hd, od, 4, 4, 'bicubic', tables)
        for g, r in zip(got, ref):
            assert np.array_equal(g, r)
    replays, builds = eng.graph_counts
    assert builds == 1 and replays == 17
    for _ in range(3):                              # three in flight: two more slots capture
        eng.decode_features(hd, od, 4, 4, 'bicubic', tables, fetch=False)
    for _ in range(3):
        assert all(np.array_equal(g, r) for g, r in zip(eng.fetch(), ref))
    assert eng.graph_counts[1] == 3
    # the same maps in other buffers, and a smaller batch: re-captured, same answers
    hd2, od2 = hd.clone(), od.clone()
    got = eng.decode_features(hd2, od2, 4, 4, 'bicubic', tables)
    assert eng.graph_counts[1] == 4 and all(np.array_equal(g, r) for g, r in zip(got, ref))
    sub = [0, 1, 3, 4]
    got = eng.decode_features(hd[sub], od[sub], 4, 4, 'bicubic', tables)
    assert all(np.array_equal(g, r) for g, r in zip(got, ref[:2]))
    host = eng.decode_features(torch.from_numpy(hmp).pin_memory(), torch.from_numpy(omp).pin_memory(), 4, 4,
                               'bicubic', tables)
    assert all(np.array_equal(g, r) for g, r in zip(host, ref))
    # a prepared plan: one foreign call per launch / fetch
    plan = eng.plan_features(hd, od, 4, 4, 'bicubic', tables)
    for _ in range(3):
        plan.launch()
    for _ in range(3):
        assert all(np.array_equal(g, r) for g, r in zip(plan.fetch(), ref))


def test_calls_in_flight_from_different_streams(cuda_device):
    """Every call owns its scratch (candidate lists, block flags, work list): decode calls launched
    from alternating caller streams with several in flight equal the synchronous results."""
    skel = cfg.COCO_PERSON_SKELETON
    eng = DecoderEngine(17, skel, topk=16, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    batches = []
    for i in range(4):
        hmp, omp = _lowres_scene(500 + 10 * i, 2 + i % 2, False)
        batches.append((torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda()))
    refs = [eng.decode_features(h_, o_, 4, 4, 'bicubic') for h_, o_ in batches]
    streams = [torch.cuda.Stream() for _ in range(3)]
    torch.cuda.synchronize()
    for rep in range(6):
        for graph in (True, False):
            eng.set_graph(graph)
            for i, (h_, o_) in enumerate(batches):
                with torch.cuda.stream(streams[(i + rep) % 3]):
                    eng.decode_features(h_, o_, 4, 4, 'bicubic', fetch=False)
            for r in refs:
                got = eng.fetch()
                assert len(got) == len(r) and all(np.array_equal(a_, b_) for a_, b_ in zip(got, r))


def test_mismatched_heads_are_rejected(cuda_device):
    """Channel counts / resolutions that do not fit the configuration raise before the library is
    called (the C ABI infers the channel counts from the configuration)."""
    skel = cfg.COCO_PERSON_SKELETON
    eng = DecoderEngine(17, skel, topk=8, thre_hmp=0.05, dist_max=40, use_scale=True, person_thre=0.05)
    z = lambda *s_: torch.zeros(s_, device='cuda')
    with pytest.raises(ValueError):
        eng.decode_features(z(2, 17, 16, 16), z(2, 62, 16, 16), 4, 4)          # omp31 maps, 19-limb skeleton
    with pytest.raises(ValueError):
        eng.decode_features(z(2, 14, 16, 16), z(2, 38, 16, 16), 4, 4)
    with pytest.raises(ValueError):
        eng.decode_features(z(2, 17, 16, 16), z(2, 38, 32, 32), 4, 4)
    with pytest.raises(ValueError):
        eng.decode_features(z(2, 17, 16, 16), z(4, 38, 16, 16), 4, 4)
    tables = (cfg.heatmap_hflip(cfg.COCO_KEYPOINTS),) + tuple(cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel))
    with pytest.raises(ValueError):
        eng.decode_features(z(3, 17, 16, 16), z(3, 38, 16, 16), 4, 4, 'bicubic', tables)    # odd flip batch
    with pytest.raises(ValueError):
        eng.decode_maps(z(1, 17, 32, 32), z(1, 38, 16, 16))
    assert eng.pending == 0 and eng.decode_features(z(2, 17, 16, 16), z(2, 38, 16, 16), 4, 4)[0].shape == (0, 17, 6)


@pytest.mark.parametrize('env', [{'OG_K3_WARP_ROWS': '0'}, {'OG_K3_WARP_ROWS': '8'}, {'OG_RESULT_ROWS': '1'}])
def test_k3_kernel_variants_agree(cuda_device, env, monkeypatch):
    """The one-warp-per-image grouping kernel, the CTA kernel it hands oversized images to
    (OG_K3_WARP_ROWS = 8: most fuzz tables overflow 8 person rows; 0: CTA kernel only) and the
    regroup into a worst-case result buffer (OG_RESULT_ROWS = 1) all reproduce the reference."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    cases = gio.load_group_fuzz()
    for c in cases[::3]:
        g = decoder.GreedyGroup(c['person_thre'], sort_dim=c['sort_dim'], dist_max=40, use_scale=c['use_scale'],
                                keypoints=list(range(c['n_keypoints'])), skeleton=c['skeleton'])
        stack = np.stack([c['limbs']] * 3)
        for got in g.group_batch(stack):
            gio.compare_poses(got, c['poses'], exact=True)
    d = gio.load_limbs_case('limbs_crowdpose')
    eng = _engine(d, d['n_keypoints'], d['skeleton'])
    poses = eng.decode_maps(torch.from_numpy(d['heat']).cuda(), torch.from_numpy(d['offs']).cuda())
    for p, r in zip(poses, gio.split_poses(d['poses'], d['pose_counts'])):
        gio.compare_poses(p, r, rtol=RTOL)
    # on the decode path the CTA kernel runs at fetch time, and only for batches that need it
    assert eng.k3_redo_count == (1 if env.get('OG_K3_WARP_ROWS') == '8' else 0)


# --------------------------------------------------------------------------- BASELINE sizes
def _pose_lists_equal(got, ref):
    assert len(got) == len(ref)
    for p, r in zip(got, ref):
        gio.compare_poses(p, r, rtol=RTOL)


def test_bench_workload_batch64_matches_c_oracle(cuda_device):
    """The bench workload itself (BASELINE configs[1] settings, batch 64, flip-test fusion,
    160x160 -> 640x640) decoded through the reference-facing API from pinned host maps, every
    image compared with the C oracle: person count / order, x, y, ids exact, scores 1e-5."""
    import bench
    from oracle import c_oracle as co
    hmp, omp = bench.lowres_inputs(5000, 64, 640, True)
    pp = decoder.decoder_factory(_args(topk=32, thre_hmp=0.04, person_thre=0.04, dist_max=40.0, batch_size=64))
    feats = [[[torch.from_numpy(hmp).pin_memory()], [[]], [[]]], [[torch.from_numpy(omp).pin_memory()], [[]], [[]]]]
    got = pp.generate_poses(feats, flip_test=True)
    eng = pp._engine(torch.device('cuda', 0))
    assert eng.fused_redo_count == 0
    ds, di, lb = [t.cpu().numpy() for t in eng.last_intermediates(64)]
    skel = cfg.COCO_PERSON_SKELETON
    fl, rs = cfg.offset_hflip(cfg.COCO_KEYPOINTS, skel)
    ref, ref_limbs = co.generate_poses(hmp, omp, skel, 17, topk=32, thre_hmp=0.04, min_len=0.5,
                                       person_thre=0.04, dist_max=40.0, use_scale=True, flip_test=True,
                                       kp_flips=cfg.heatmap_hflip(cfg.COCO_KEYPOINTS), limb_flips=fl,
                                       limb_reserve=rs, return_limbs=True)
    assert sum(len(p) for p in ref) >= 64 * 5
    assert gio.compare_limbs(lb, ref_limbs, 0.04, rtol=RTOL) > 64 * 90
    _pose_lists_equal(got, ref)
    # the hot path on the materialised maps of the same batch gives the same persons
    hm_f, om_f = co.flip_augment(hmp, omp, cfg.heatmap_hflip(cfg.COCO_KEYPOINTS), fl, rs)
    heat = torch.from_numpy(co.resize(hm_f[:16], 4, 'bicubic')).cuda()
    offs = torch.from_numpy(co.resize(om_f[:16], 4, 'bilinear')).cuda()
    hot = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.04).decode_maps(heat, offs)
    for p, r in zip(hot, got[:16]):
        assert np.array_equal(p, r)


def test_config4_1024_long_edge(cuda_device):
    """BASELINE config 4 sizes: 256x256 maps -> 1024x1024, ids of the last channels exceed 2**24
    and are stored as rounded float32 exactly like the reference (collect.py:227-228)."""
    from oracle import c_oracle as co
    skel = cfg.COCO_PERSON_SKELETON
    n = 4
    hmp, omp = scenes.render_batch(4242, n, 8, 1024, 1024, skel, noise=0.02, scale_range=(16.0, 38.0))
    eng = DecoderEngine(17, skel, topk=32, thre_hmp=0.04, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.04)
    got = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), 4, 4, 'bicubic')
    _, _, lb = eng.last_intermediates(n)
    ref, ref_limbs = co.generate_poses(hmp, omp, skel, 17, topk=32, thre_hmp=0.04, min_len=0.5,
                                       person_thre=0.04, dist_max=40.0, use_scale=True, return_limbs=True)
    assert gio.compare_limbs(lb.cpu().numpy(), ref_limbs, 0.04, rtol=RTOL) > n * 100
    _pose_lists_equal(got, ref)
    ids = np.concatenate([p[..., 5].ravel() for p in got])
    assert ids.max() > 2 ** 24
    eng.set_fused(False)
    staged = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), 4, 4, 'bicubic')
    for a, b in zip(got, staged):
        assert np.array_equal(a, b)


def test_maximum_sizes(cuda_device):
    """The ABI's upper bounds: topk = OG_MAX_TOPK (128) on crowded scenes, and a skeleton with
    OG_MAX_KEYPOINTS = 64 keypoints and OG_MAX_LIMBS = 64 limbs (a ring), both against the oracle."""
    skel = cfg.COCO_PERSON_SKELETON
    heat, offs = scenes.synth_hires_batch(909, 2, 20, 320, 256, skel)
    eng = DecoderEngine(17, skel, topk=128, thre_hmp=0.04, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.04)
    got = eng.decode_maps(torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda())
    ref_limbs = ro.generate_limbs(heat, offs, skel, 128, 0.04, 0.5, 1, 1)
    _, _, lb = eng.last_intermediates(2)
    assert gio.compare_limbs(lb.cpu().numpy(), ref_limbs, 0.04, rtol=RTOL) > 300
    for i in range(2):
        gio.compare_poses(got[i], ro.group_skeletons(ref_limbs[i], skel, 17, 0.04, 2, 40, True), rtol=RTOL)
        assert len(got[i]) >= 15
    # 64 keypoints / 64 limbs: joint j sits at a fixed offset from joint j - 1
    c = 64
    ring = [(j, (j + 1) % c) for j in range(c)]
    rng = np.random.RandomState(64)
    h, w = 96, 128
    heat = rng.uniform(0, 0.02, size=(1, c, h, w)).astype(np.float32)
    offs = np.zeros((1, 2 * c, h, w), np.float32)
    for person in range(3):
        x0, y0 = rng.randint(10, 40), rng.randint(10, 30) + 25 * person
        pts = [(x0 + (j % 16) * 5 + rng.randint(0, 2), y0 + (j // 16) * 5) for j in range(c)]
        for j, (x, y) in enumerate(pts):
            heat[0, j, y, x] = 0.9 - 0.1 * person + 0.001 * j
        for l, (a, b) in enumerate(ring):
            (xa, ya), (xb, yb) = pts[a], pts[b]
            offs[0, 2 * l, ya, xa] = xb - xa
            offs[0, 2 * l + 1, ya, xa] = yb - ya
    eng = DecoderEngine(c, ring, topk=8, thre_hmp=0.05, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.05)
    got = eng.decode_maps(torch.from_numpy(heat).cuda(), torch.from_numpy(offs).cuda())
    ref_limbs = ro.generate_limbs(heat, offs, ring, 8, 0.05, 0.5, 1, 1)
    ref = ro.group_skeletons(ref_limbs[0], ring, c, 0.05, 2, 40, True)
    assert len(ref) == 3 and (ref[:, :, 2] > 0).all()
    gio.compare_poses(got[0], ref, rtol=RTOL)
    from offsetguided_b200 import _lib
    with pytest.raises(_lib.OgError):
        DecoderEngine(17, skel, topk=129, thre_hmp=0.05)
    with pytest.raises(_lib.OgError):
        DecoderEngine(65, [(0, 1)], topk=8, thre_hmp=0.05)


def test_config3_crowdpose_batch32(cuda_device):
    """BASELINE config 3: 14 keypoints, builder-supplied skeleton, 20 persons, K = 64, batch 32."""
    from oracle import c_oracle as co
    skel = cfg.CROWDPOSE_PERSON_SKELETON
    hmp, omp = scenes.render_batch(777, 32, 20, 512, 512, skel, template=scenes.TEMPLATE_CROWDPOSE,
                                   noise=0.02, scale_range=(7.0, 16.0))
    eng = DecoderEngine(14, skel, topk=64, thre_hmp=0.06, min_len=0.5, dist_max=40, use_scale=True,
                        person_thre=0.06)
    got = eng.decode_features(torch.from_numpy(hmp).cuda(), torch.from_numpy(omp).cuda(), 4, 4, 'bicubic')
    ref = co.generate_poses(hmp, omp, skel, 14, topk=64, thre_hmp=0.06, min_len=0.5, person_thre=0.06,
                            dist_max=40.0, use_scale=True)
    assert sum(len(p) for p in ref) > 32 * 15
    _pose_lists_equal(got, ref)


@pytest.mark.parametrize('name', list(gio.OPTIONAL_VARIANTS))
def test_optional_heads_match_reference(cuda_device, name):
    """include_scale / include_jitter_offset / use_jitter_offset / cat_flip_offs through
    decoder_factory(args).generate_poses against the reference's own output."""
    d = gio.load_optional_heads()
    inc_scale, inc_jit, use_jit, flip, cat = gio.OPTIONAL_VARIANTS[name]
    n = d['hmp'].shape[0] // 2
    sel = slice(None) if flip else slice(0, n)
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.06, person_thre=0.06, dist_max=40, batch_size=n,
                                       include_scale=inc_scale, include_jitter_offset=inc_jit,
                                       use_jitter_offset=use_jit))
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    feats = [[[dev(d['hmp'][sel])], [[]], [dev(d['jom'][sel]) if inc_jit else []]],
             [[dev(d['omp'][sel])], [[]], [dev(d['scm'][sel]) if inc_scale else []]]]
    got = pp.generate_poses(feats, flip_test=flip, cat_flip_offs=cat)
    ref = gio.split_poses(d[name + '_poses'], d[name + '_counts'])
    assert len(got) == len(ref)
    for p, r in zip(got, ref):
        assert p.shape == r.shape and np.array_equal(p[..., 5], r[..., 5])
        np.testing.assert_allclose(p, r, rtol=RTOL, atol=1e-5)
        if not (inc_jit and use_jit):
            assert np.array_equal(p[..., :2], r[..., :2])
    # that was the fused path (K2 interpolates the optional heads at the candidate pixels); the
    # stage-by-stage path on materialised maps gives the same poses bit for bit
    eng = pp._engine(torch.device('cuda', 0))
    l0 = eng.launch_count
    pp.generate_poses(feats, flip_test=flip, cat_flip_offs=cat)
    assert eng.launch_count - l0 == 6 and eng.fused_redo_count == 0
    eng.set_fused(False)
    staged = pp.generate_poses(feats, flip_test=flip, cat_flip_offs=cat)
    for p, q in zip(got, staged):
        assert np.array_equal(p, q)


def test_tied_peaks_tie_aware_against_reference(cuda_device):
    """Bicubic x4 plateaus: equal-valued above-threshold peaks within a channel (SURVEY 8c).  Dets are
    compared with the reference's own torch.topk output as sets within tied groups; final poses must
    equal the reference's (the generator verified they do not depend on the order of the tie)."""
    d = gio.load('poses_tied_peaks')
    thre = float(d['thre_hmp'])
    pp = decoder.decoder_factory(_args(topk=int(d['topk']), thre_hmp=thre, person_thre=float(d['person_thre']),
                                       dist_max=float(d['dist_max'])))
    for host in (False, True):
        hmp, omp = torch.from_numpy(d['hmp']), torch.from_numpy(d['omp'])
        hmp, omp = (hmp.pin_memory(), omp.pin_memory()) if host else (hmp.cuda(), omp.cuda())
        poses = pp.generate_poses([[[hmp], [[]], [[]]], [[omp], [[]], [[]]]])
        ref = gio.split_poses(d['poses'], d['pose_counts'])
        assert len(poses) == len(ref)
        for p, r in zip(poses, ref):
            gio.compare_poses(p, r, rtol=RTOL)
        ds, di, _ = pp._engine(torch.device('cuda', 0)).last_intermediates(len(ref))
        groups = gio.compare_dets_tie_aware(ds.cpu().numpy(), di.cpu().numpy(), d['det_scores'], d['det_inds'], thre)
        assert groups >= int(d['ties'])


def test_submit_collect_equals_generate_poses(cuda_device):
    """PostProcess.submit / collect (the pipelined form of generate_poses): same results as the
    synchronous call, in launch order, for device maps (cached plan, replayed graph — also when
    the buffers are refilled with other images), packed bf16 slices and pinned host maps."""
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.05, person_thre=0.05, dist_max=40))
    batches = [_lowres_scene(900 + 7 * i, 2, True) for i in range(3)]
    refs = []
    for hmp, omp in batches:
        feats = [[[torch.from_numpy(hmp).cuda()], [[]], [[]]], [[torch.from_numpy(omp).cuda()], [[]], [[]]]]
        refs.append(pp.generate_poses(feats, flip_test=True))
    assert sum(len(p) for r in refs for p in r) > 10
    # the same two device buffers refilled batch after batch (what a network does)
    hd = torch.empty_like(torch.from_numpy(batches[0][0])).cuda()
    od = torch.empty_like(torch.from_numpy(batches[0][1])).cuda()
    for rep in range(3):
        for i, (hmp, omp) in enumerate(batches):
            hd.copy_(torch.from_numpy(hmp))
            od.copy_(torch.from_numpy(omp))
            torch.cuda.synchronize()
            pp.submit([[[hd.view_as(hd)], [[]], [[]]], [[od.view_as(od)], [[]], [[]]]], flip_test=True)
            got = pp.collect()
            assert all(np.array_equal(g, r) for g, r in zip(got, refs[i])) and len(got) == len(refs[i])
    assert len(pp._plans) == 1
    # several in flight, distinct buffers, plus a pinned-host and a packed bf16 submission
    dev = [(torch.from_numpy(h_).cuda(), torch.from_numpy(o_).cuda()) for h_, o_ in batches]
    for h_, o_ in dev:
        pp.submit([[[h_], [[]], [[]]], [[o_], [[]], [[]]]], flip_test=True)
    host = (torch.from_numpy(batches[1][0]).pin_memory(), torch.from_numpy(batches[1][1]).pin_memory())
    pp.submit([[[host[0]], [[]], [[]]], [[host[1]], [[]], [[]]]], flip_test=True)
    for i in range(3):
        got = pp.collect()
        assert all(np.array_equal(g, r) for g, r in zip(got, refs[i]))
    got = pp.collect()
    assert all(np.array_equal(g, r) for g, r in zip(got, refs[1]))
    packed = torch.cat((dev[2][0], dev[2][1]), dim=1).to(torch.bfloat16)
    f32 = packed.float()
    ref_bf = pp.generate_poses([[[f32[:, :17].contiguous()], [[]], [[]]], [[f32[:, 17:].contiguous()], [[]], [[]]]],
                               flip_test=True)
    pp.submit([[[packed[:, :17]], [[]], [[]]], [[packed[:, 17:]], [[]], [[]]]], flip_test=True)
    got = pp.collect()
    assert len(got) == len(ref_bf) and all(np.array_equal(g, r) for g, r in zip(got, ref_bf))


def test_result_rows_on_the_gpu_equal_the_reference_loops(cuda_device):
    """PostProcess.generate_results: poses back-projected and formatted by the grouping kernel
    equal the reference's loops (oracle restatement of preprocess.annotations_inverse +
    evaluate.py:227-265) value for value, incl. an image without persons, through the graph
    replay, the kernel-by-kernel launch and the host-input path."""
    from offsetguided_b200 import results
    pp = decoder.decoder_factory(_args(topk=16, thre_hmp=0.05, person_thre=0.05, dist_max=40))
    hmp, omp = _lowres_scene(4242, 3, True)
    hmp[1] = 0
    hmp[4] = 0                                            # image 1 (and its mirrored copy): nobody there
    rng = np.random.RandomState(5)
    metas = [{'offset': np.array([-float(rng.randint(0, 90)), -float(rng.randint(0, 60))]),
              'scale': np.array([rng.uniform(0.4, 1.7), rng.uniform(0.4, 1.7)]), 'hflip': False,
              'width_height': (640, 480), 'image_id': 70 + i} for i in range(3)]
    eng = pp._engine(torch.device('cuda', 0))
    for mode in ('graph', 'kernels', 'host'):
        eng.set_graph(mode == 'graph')
        h_, o_ = torch.from_numpy(hmp), torch.from_numpy(omp)
        h_, o_ = (h_.pin_memory(), o_.pin_memory()) if mode == 'host' else (h_.cuda(), o_.cuda())
        feats = [[[h_], [[]], [[]]], [[o_], [[]], [[]]]]
        for _ in range(2):
            poses, kp, sc, img = pp.generate_results(feats, metas, flip_test=True)
        ref_rows, ref_ids = ro.coco_result_rows(poses, metas)
        rows = results.rows_from_arrays(kp, sc, img, metas)
        assert len(poses[1]) == 0 and len(poses[0]) > 0 and len(rows) == len(ref_rows)
        for a, b in zip(rows, ref_rows):
            assert a['image_id'] == b['image_id'] and a['keypoints'] == b['keypoints'] and a['score'] == b['score']
        plain = pp.generate_poses(feats, flip_test=True)              # no frames staged: no result rows
        assert eng.last_result_rows is None and all(np.array_equal(a, b) for a, b in zip(plain, poses))
