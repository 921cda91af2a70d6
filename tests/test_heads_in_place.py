"""The optional heads (keypoint-scale and jitter-offset maps) decoded in place on the device path.

A network built with ``--include-scale`` / ``--include-jitter-offset`` leaves four maps behind: heat,
offsets, keypoint scales and jitter offsets, often as channel slices of one packed output, in
bf16 / f16 under AMP and channels-last when the network runs in ``torch.channels_last``.
``engine._heads_in_place`` decides whether ``decode_features_heads`` hands them to
``og_decode_features_heads_dev_strided`` where they are; K2 then samples the heads through their
element strides.  Every case must equal, bit for bit, ``og_decode_features_heads_dev`` on dense
float32 copies of the same values."""
import ctypes

import numpy as np
import pytest

import golden_io as gio
from oracle import ref_oracle as ro
from test_fused_matrix import C, DTYPES, KP, FL, RS, L2, SHAPES, SKEL, THRE, TOPK, RTOL, matrix_inputs, _torch_dtype
from test_channels_last import _bench_packed

LAYOUTS = ('dense', 'planar_packed', 'cl_separate', 'cl_packed', 'mixed')
HEADS = {                       # name: (scale head, jitter head, use_jitter)
    'scale': (True, False, True),
    'jitter': (False, True, True),
    'jitter_unused': (False, True, False),
    'both': (True, True, True),
}
FLIPS = ('noflip', 'flip', 'flip_cat')
# cat_flip_offs with used jitter is refused (the reference raises): those pairs are not decoded
CASES = [(hd, fl) for hd in HEADS for fl in FLIPS if not (fl == 'flip_cat' and HEADS[hd][1] and HEADS[hd][2])]
PACKED = C + L2 + C + 2          # heat, offsets, keypoint scales, jitter offsets of one head output


# =========================================================================== CPU: the routing
class _OnDevice(object):
    """A CPU tensor's shape, strides and element type, presented as those of a CUDA tensor (the
    router looks at nothing else)."""

    def __init__(self, t):
        self.shape, self.dtype, self.is_cuda, self._st = t.shape, t.dtype, True, t.stride()

    def stride(self):
        return self._st


def _split(buf):
    return buf[:, :C], buf[:, C:C + L2], buf[:, C + L2:2 * C + L2], buf[:, 2 * C + L2:]


def test_heads_routing():
    """No GPU.  Which four-map sets go in place, with which element strides, and which are
    converted."""
    import torch
    from offsetguided_b200.engine import _heads_in_place
    n, h, w = 4, 6, 10
    hw = h * w
    dev = lambda ts: tuple(_OnDevice(t) if t is not None else None for t in ts)
    chans = (C, L2, C, 2)

    def planar(ch, image_stride=None):
        return (image_stride or ch * hw, hw, w, 1)

    # dense, separate: bf16 / f16 in place with planar strides; dense float32 is already what the
    # library reads, so it keeps the dense entry point
    for dt in (torch.bfloat16, torch.float16):
        maps = tuple(torch.zeros(n, ch, h, w, dtype=dt) for ch in chans)
        assert _heads_in_place(dev(maps)) == [planar(ch) for ch in chans]
        assert _heads_in_place(dev(maps[:2] + (None, maps[3]))) == [planar(C), planar(L2), None, planar(2)]
    maps32 = tuple(torch.zeros(n, ch, h, w) for ch in chans)
    assert _heads_in_place(dev(maps32)) is None
    # image-strided slices of one packed planar [2N, C + 2L + C + 2, h, w] output
    packed = torch.zeros(2 * n, PACKED, h, w, dtype=torch.bfloat16)
    assert _heads_in_place(dev(_split(packed))) == [planar(ch, PACKED * hw) for ch in chans]
    assert _heads_in_place(dev(_split(packed.float()))) == [planar(ch, PACKED * hw) for ch in chans]
    # channels-last, separate
    sep = tuple(t.contiguous(memory_format=torch.channels_last) for t in maps32)
    assert _heads_in_place(dev(sep)) == [(hw * ch, 1, w * ch, ch) for ch in chans]
    # channels-last packed slices: pixel stride = the channel count of the whole output
    cl = packed.contiguous(memory_format=torch.channels_last)
    assert _heads_in_place(dev(_split(cl))) == [(hw * PACKED, 1, w * PACKED, PACKED)] * 4
    # padded channels-last (80 channels, offsets first, every other image of the buffer)
    pad = torch.zeros(4 * n, 80, h, w, dtype=torch.float16).contiguous(memory_format=torch.channels_last)[::2]
    pv = (pad[:, L2:L2 + C], pad[:, :L2], pad[:, L2 + C:L2 + 2 * C], pad[:, L2 + 2 * C:L2 + 2 * C + 2])
    assert [t.shape[1] for t in pv] == list(chans)
    assert _heads_in_place(dev(pv)) == [(2 * hw * 80, 1, w * 80, 80)] * 4
    # heat channels-last, the rest planar
    mixed = (sep[0],) + maps32[1:]
    assert _heads_in_place(dev(mixed)) == [(hw * C, 1, w * C, C), planar(L2), planar(C), planar(2)]
    # converted: mixed element types, rows that are not dense, host tensors, an empty batch
    assert _heads_in_place(dev(maps32[:3] + (maps32[3].half(),))) is None
    assert _heads_in_place(dev((maps32[0].half(),) + maps32[1:])) is None
    wide = torch.zeros(n, C, h, 2 * w, dtype=torch.bfloat16)[..., ::2]
    assert _heads_in_place(dev((wide,) + tuple(t.bfloat16() for t in maps32[1:]))) is None
    assert _heads_in_place(dev(_split(packed)[:3] + (torch.zeros(n * 2, 2, h, 2 * w, dtype=torch.bfloat16)[..., ::2],))) is None
    assert _heads_in_place(_split(packed)) is None
    assert _heads_in_place(dev(tuple(torch.zeros(0, ch, h, w, dtype=torch.bfloat16) for ch in chans))) is None


# =========================================================================== GPU
def _cl(t):
    import torch
    return t.contiguous(memory_format=torch.channels_last)


def _heads_inputs(h, w, scale, flip):
    """(hmp, omp, scm, jom) float32 at network resolution: the fused-matrix scenes plus keypoint
    scales in [2, 60) and jitter offsets in [-1.5, 1.5) (the range of the reference fixture)."""
    hmp, omp = matrix_inputs(h, w, scale, flip)
    rng = np.random.RandomState(7 * h + scale + (100 if flip else 0))
    scm = rng.uniform(2, 60, size=(hmp.shape[0], C, h, w)).astype(np.float32)
    jom = rng.uniform(-1.5, 1.5, size=(hmp.shape[0], 2, h, w)).astype(np.float32)
    return hmp, omp, scm, jom


def _views(arrays, layout, dtype):
    """The four maps of `layout` on the GPU in `dtype`."""
    import torch
    td = _torch_dtype(dtype)
    ts = [torch.from_numpy(a).to(td).cuda() for a in arrays]
    if layout == 'dense':
        return tuple(ts)
    if layout == 'cl_separate':
        return tuple(_cl(t) for t in ts)
    buf = torch.cat(ts, dim=1)
    if layout == 'planar_packed':
        return _split(buf)
    if layout == 'cl_packed':
        return _split(_cl(buf))
    rest = torch.cat(ts[1:], dim=1)            # mixed: heat channels-last, the heads planar slices
    return (_cl(ts[0]), rest[:, :L2], rest[:, L2:L2 + C], rest[:, L2 + C:])


def _tables(flip):
    return (KP, FL, RS) if flip else None


def _decode(eng, maps, scale, mode, flip, cat, use_jitter, n):
    """Poses and (dets, indices, limbs) of one decode_features_heads call."""
    got = eng.decode_features_heads(*maps, hmp_stride=scale, off_stride=scale, resize_mode=mode,
                                    flip_tables=_tables(flip), cat_flip_offs=cat, use_jitter=use_jitter)
    return got, [t.cpu().numpy() for t in eng.last_intermediates(n)]


def _dense32(maps):
    return tuple(t.float().contiguous() if t is not None else None for t in maps)


def _assert_same(a, b):
    (pa, ia), (pb, ib) = a, b
    for x, y in zip(ia, ib):
        assert np.array_equal(x, y)
    assert len(pa) == len(pb)
    for x, y in zip(pa, pb):
        assert np.array_equal(x, y)


@pytest.fixture(scope='module')
def eng(cuda_device):
    from test_fused_matrix import _engine
    e = _engine()
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize('scale_case', ['s4', 's2or8'])
@pytest.mark.parametrize('heads,flips', CASES)
@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('dtype', DTYPES)
def test_heads_matrix(eng, dtype, layout, heads, flips, scale_case):
    """Dets, limbs and poses of the heads read in place equal og_decode_features_heads_dev on dense
    float32 copies bit for bit (bicubic at S = 4, bilinear at S = 2 or 8)."""
    from offsetguided_b200.engine import _heads_in_place
    inc_scale, inc_jit, use_jit = HEADS[heads]
    flip, cat = flips != 'noflip', flips == 'flip_cat'
    if scale_case == 's4':
        scale, mode = 4, 'bicubic'
    else:
        scale, mode = (2, 8)[(DTYPES.index(dtype) + LAYOUTS.index(layout)) % 2], 'bilinear'
    h, w = SHAPES['dense']
    arrays = _heads_inputs(h, w, scale, flip)
    n = arrays[0].shape[0] // 2 if flip else arrays[0].shape[0]
    hv, ov, sv, jv = _views(arrays, layout, dtype)
    maps = (hv, ov, sv if inc_scale else None, jv if inc_jit else None)
    assert (_heads_in_place(maps) is None) == (dtype == 'f32' and layout == 'dense')
    r0 = eng.fused_redo_count
    got = _decode(eng, maps, scale, mode, flip, cat, use_jit, n)
    want = _decode(eng, _dense32(maps), scale, mode, flip, cat, use_jit, n)
    assert eng.fused_redo_count == r0
    _assert_same(got, want)
    assert sum(len(p) for p in got[0]) >= 1


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', DTYPES)
def test_heads_sample_against_oracle(eng, dtype):
    """One channels-last packed case per element type, both heads, flip-test, against the reference
    oracle on the widened maps (the C oracle has no optional heads).  Square maps: the reference's
    jitter refinement indexes [x, y] as [row, col] and raises for x >= H on wider maps."""
    h = w = 40
    arrays = _heads_inputs(h, w, 4, True)
    maps = _views(arrays, 'cl_packed', dtype)
    got, _ = _decode(eng, maps, 4, 'bicubic', True, False, True, 2)
    wide = [t.float().cpu().numpy() for t in maps]
    ref = ro.generate_poses(np.ascontiguousarray(wide[0]), np.ascontiguousarray(wide[1]), SKEL, C, topk=TOPK,
                            thre_hmp=THRE, min_len=0.5, person_thre=THRE, dist_max=40.0, use_scale=True,
                            flip_test=True, kp_flips=KP, limb_flips=FL, limb_reserve=RS,
                            scmps=np.ascontiguousarray(wide[2]), jomps=np.ascontiguousarray(wide[3]),
                            use_jitter=True)
    assert len(got) == len(ref) == 2 and sum(len(p) for p in ref) >= 2
    for p, r in zip(got, ref):
        assert p.shape == r.shape and np.array_equal(p[..., 5], r[..., 5])
        np.testing.assert_allclose(p, r, rtol=RTOL, atol=1e-5)


def _post(**over):
    import argparse
    from offsetguided_b200 import decoder
    p = argparse.ArgumentParser()
    decoder.decoder_cli(p)
    a = p.parse_args([])
    a.headnets, a.strides, a.batch_size = ['hmp', 'omp'], [4, 4], 8
    a.include_scale = a.include_jitter_offset = False
    for k, v in over.items():
        setattr(a, k, v)
    return decoder.decoder_factory(a)


@pytest.mark.gpu
@pytest.mark.parametrize('layout', ['cl_packed', 'planar_packed', 'cl_separate'])
@pytest.mark.parametrize('name', list(gio.OPTIONAL_VARIANTS))
def test_reference_fixture_in_new_layouts(cuda_device, name, layout):
    """The optional-heads reference fixture, float32 but laid out channels-last or as packed slices,
    through decoder_factory(args).generate_poses: read in place, equal to the reference's poses
    and to the decode of the dense maps."""
    import torch
    from offsetguided_b200.engine import _heads_in_place
    d = gio.load_optional_heads()
    inc_scale, inc_jit, use_jit, flip, cat = gio.OPTIONAL_VARIANTS[name]
    n = d['hmp'].shape[0] // 2
    sel = slice(None) if flip else slice(0, n)
    pp = _post(topk=16, thre_hmp=0.06, person_thre=0.06, dist_max=40, batch_size=n, include_scale=inc_scale,
               include_jitter_offset=inc_jit, use_jitter_offset=use_jit)

    def feats(maps):
        hv, ov, sv, jv = maps
        return [[[hv], [[]], [jv if inc_jit else []]], [[ov], [[]], [sv if inc_scale else []]]]
    arrays = [np.ascontiguousarray(d[k][sel]) for k in ('hmp', 'omp', 'scm', 'jom')]
    maps = _views(arrays, layout, 'f32')
    assert _heads_in_place((maps[0], maps[1], maps[2] if inc_scale else None, maps[3] if inc_jit else None))
    got = pp.generate_poses(feats(maps), flip_test=flip, cat_flip_offs=cat)
    ref = gio.split_poses(d[name + '_poses'], d[name + '_counts'])
    assert len(got) == len(ref)
    for p, r in zip(got, ref):
        assert p.shape == r.shape and np.array_equal(p[..., 5], r[..., 5])
        np.testing.assert_allclose(p, r, rtol=RTOL, atol=1e-5)
        if not (inc_jit and use_jit):
            assert np.array_equal(p[..., :2], r[..., :2])
    dense = pp.generate_poses(feats(tuple(torch.from_numpy(a).cuda() for a in arrays)), flip_test=flip,
                              cat_flip_offs=cat)
    assert all(np.array_equal(a, b) for a, b in zip(got, dense))


def _bench_heads(seed, n, edge, flip, dtype='bf16'):
    """A packed channels-last [n or 2n, C + 2L + C + 2, h, w] head output of rendered scenes with
    keypoint-scale and jitter-offset channels."""
    import torch
    buf = _bench_packed(seed, n, edge, flip, dtype)
    rng = np.random.RandomState(seed)
    n_in, _, h, w = buf.shape
    scm = torch.from_numpy(rng.uniform(2, 60, size=(n_in, C, h, w)).astype(np.float32))
    jom = torch.from_numpy(rng.uniform(-1.5, 1.5, size=(n_in, 2, h, w)).astype(np.float32))
    heads = torch.cat((scm, jom), dim=1).to(buf.dtype).cuda()
    return _cl(torch.cat((buf, heads), dim=1))


@pytest.mark.gpu
def test_heads_decoded_in_place(eng):
    """No conversion copy: torch allocates nothing during a call (peak included), and a call is as
    many launches as the dense-float32 call, with graph replay and kernel by kernel."""
    import torch
    buf = _bench_heads(41, 8, 640, True)
    maps = _split(buf)
    dense = _dense32(maps)
    kw = dict(hmp_stride=4, off_stride=4, resize_mode='bicubic', flip_tables=(KP, FL, RS), use_jitter=True)
    ref = eng.decode_features_heads(*dense, **kw)
    for graph in (True, False):
        eng.set_graph(graph)
        eng.decode_features_heads(*maps, **kw)         # warm-up: the slot's channels-last scratch exists now
        eng.decode_features_heads(*dense, **kw)
        torch.cuda.synchronize()
        l0 = eng.launch_count
        eng.decode_features_heads(*dense, **kw)
        dense_launches = eng.launch_count - l0
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        l0 = eng.launch_count
        got = eng.decode_features_heads(*maps, **kw)
        assert eng.launch_count - l0 == dense_launches == 6
        torch.cuda.synchronize()
        assert torch.cuda.memory_allocated() == before and torch.cuda.max_memory_allocated() == before
        assert len(got) == len(ref) and all(np.array_equal(a, b) for a, b in zip(got, ref))
    eng.set_graph(True)
    assert sum(len(p) for p in ref) >= 8


@pytest.mark.gpu
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
def test_heads_overflow_redo(eng, flip):
    """A noise plane of more than 2048 candidates in a bf16 channels-last batch with both heads: the
    fetch redoes it and K2 samples the same in-place heads again; the call equals the dense-float32
    decode."""
    import torch
    buf = _bench_heads(808, 2, 640, flip)
    rng = np.random.RandomState(12)
    buf[1, 6] = torch.from_numpy(rng.uniform(0, 1, size=buf.shape[2:]).astype(np.float32)).to(buf.dtype).cuda()
    maps = _split(buf)
    r0 = eng.fused_redo_count
    got = _decode(eng, maps, 4, 'bicubic', flip, False, True, 2)
    assert eng.fused_redo_count == r0 + 1
    want = _decode(eng, _dense32(maps), 4, 'bicubic', flip, False, True, 2)
    _assert_same(got, want)
    assert sum(len(p) for p in got[0]) >= 4 and (got[1][0][1, 6] > 0).all()


@pytest.mark.gpu
def test_graph_key_includes_the_heads(eng):
    """Same pointers, another element type or head layout or head stride: the graph is re-captured
    and the result is that of the new maps; the same call again replays."""
    import torch
    n_in, h, w = 4, 40, 48
    hw = h * w
    arrays = _heads_inputs(h, w, 4, True)
    kw = dict(hmp_stride=4, off_stride=4, resize_mode='bicubic', flip_tables=(KP, FL, RS), use_jitter=True)
    raw = [torch.empty(n_in * 4 * ch * hw * 2, dtype=torch.uint8, device='cuda') for ch in (C, L2, C, 2)]

    def place(dtype, scale_cl=False, jitter_image=2):
        """The four maps in `raw`: planar, dense unless noted (scale head channels-last, jitter images
        `jitter_image` planes apart)."""
        td = _torch_dtype(dtype)
        views = []
        for i, (a, ch) in enumerate(zip(arrays, (C, L2, C, 2))):
            base = raw[i].view(td)
            st = (ch * hw, hw, w, 1)
            if i == 2 and scale_cl:
                st = (ch * hw, 1, w * ch, ch)
            if i == 3:
                st = (jitter_image * hw, hw, w, 1)
            v = torch.as_strided(base, (n_in, ch, h, w), st)
            v.copy_(torch.from_numpy(a).to(td))
            views.append(v)
        return tuple(views)

    def decode(maps):
        return eng.decode_features_heads(*maps, **kw)
    cases = [('bf16', False, 2), ('f16', False, 2), ('f16', True, 2), ('f16', True, 3)]
    for case in cases:
        maps = place(*case)
        assert all(m.data_ptr() == r.data_ptr() for m, r in zip(maps, raw))
        want = decode(_dense32(maps))
        r0, b0 = eng.graph_counts
        got = decode(maps)
        r1, b1 = eng.graph_counts
        assert b1 == b0 + 1 and r1 == r0 + 1, case
        assert len(got) == len(want) and all(np.array_equal(a, b) for a, b in zip(got, want)), case
        again = decode(maps)
        assert eng.graph_counts == (r1 + 1, b1), case
        assert all(np.array_equal(a, b) for a, b in zip(again, want)), case
    assert sum(len(p) for p in want) >= 1


@pytest.mark.gpu
def test_bad_heads_are_refused_before_any_launch(eng):
    """og_decode_features_heads_dev_strided refuses bad head strides, a head with the wrong channel
    count, an unknown element type, a missing stride array and cat_flip_offs with used jitter on the
    host: nothing is launched and nothing is queued.  The Python layer refuses a head of the wrong
    shape and converts heads of mixed element types."""
    from offsetguided_b200 import _lib
    from offsetguided_b200.engine import _ptr, _stream_ptr
    buf = _bench_heads(3, 2, 128, True)
    hv, ov, sv, jv = _split(buf)
    n_in, _, h, w = hv.shape
    p = PACKED
    good = (h * w * p, 1, w * p, p)
    tables = [ctypes.cast(_lib.int32_array(t), _lib.c_int32_p) for t in (KP, FL, RS)]

    def call(ss=good, js=good, dtype=_lib.OG_DTYPE_BF16, cat=0, use_jitter=1, scale_ptr=sv, jitter_ptr=jv):
        arr = lambda s: _lib.int64_array(s) if s is not None else None
        return eng.lib.og_decode_features_heads_dev_strided(
            eng._h, _ptr(hv), _ptr(ov), _ptr(scale_ptr), _ptr(jitter_ptr), dtype, arr(good), arr(good), arr(ss),
            arr(js), n_in // 2, h, w, 4, 4, 1, 1, cat, use_jitter, *tables, len(RS), _stream_ptr(eng.device))
    bad = [dict(ss=(h * w * p, 1, w * p + 1, p)),           # row stride != w * p
           dict(js=(h * w * p, 2, w * p, p)),               # channel stride 2
           dict(ss=(h * w * p - 1, 1, w * p, p)),           # images overlap
           dict(js=(2 * h * w - 1, h * w, w, 1)),           # planar images overlap
           dict(ss=(h * w * 2, 1, w * 2, 2)),               # a 2-channel map as the C keypoint scales
           dict(dtype=3),                                   # no such element type
           dict(ss=None),                                   # a map without strides
           dict(cat=1, use_jitter=1)]                       # jitter refinement of 4-D vectors
    l0 = eng.launch_count
    for kw in bad:
        assert call(**kw) == 1, kw
    assert eng.launch_count == l0 and eng.pending == 0
    assert call(cat=1, use_jitter=0) == 0
    assert len(eng.fetch()) == n_in // 2
    assert call(ss=None, scale_ptr=None) == 0
    assert len(eng.fetch()) == n_in // 2
    with pytest.raises(ValueError):
        eng.decode_features_heads(hv, ov, sv[:, :C - 1], jv, flip_tables=(KP, FL, RS))
    mixed = (hv, ov, sv.float(), jv)
    want = eng.decode_features_heads(*_dense32(mixed), flip_tables=(KP, FL, RS), use_jitter=True)
    got = eng.decode_features_heads(*mixed, flip_tables=(KP, FL, RS), use_jitter=True)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
