"""Channels-last (NHWC) network outputs decoded in place on the fused path.

A network run in ``torch.channels_last`` leaves its head output with the channels of a pixel
adjacent: element (i, c, y, x) at i * s_n + (y * w + x) * p + c, p >= C the channel count of the
whole packed tensor.  ``engine._channels_last_view`` recognises such a view (also a channel slice
of one packed output) and the library reads it where it is: the transposing activity scan
(`amax_scan_nhwc_kernel`) reads each heat cell once, writes the flip-fused planes as dense float32
scratch and flags the work blocks; K2 samples the offsets with pixel / plane strides; the overflow
redo reads the maps with the same strides.  Every case must equal, bit for bit, the decode of dense
float32 copies of the same tensors, and the oracles."""
import ctypes

import numpy as np
import pytest

import golden_io as gio
from oracle import c_oracle as co
from test_fused_matrix import (C, DTYPES, KP, FL, RS, L2, SHAPES, SKEL, THRE, TOPK, RTOL, PROBES, SPIKES, RING,
                               CHECKER, matrix_inputs, _decode_both, _matrix_oracle, _assert_same, _torch_dtype)

LAYOUTS = ('cl_separate', 'cl_packed', 'cl_offsets_first_padded', 'cl_odd', 'mixed')


# =========================================================================== CPU: the classifier
def test_channels_last_classifier():
    """No GPU.  Which tensors are read in place as channels-last, and with which element strides."""
    import torch
    from offsetguided_b200.engine import _channels_last_view, _image_strided
    n, h, w = 4, 6, 10
    planar = torch.zeros(n, C, h, w)
    assert _channels_last_view(planar) is None
    sep = planar.contiguous(memory_format=torch.channels_last)
    assert _channels_last_view(sep) == (h * w * C, 1, w * C, C)
    packed = torch.zeros(n, 55, h, w).contiguous(memory_format=torch.channels_last)
    assert _channels_last_view(packed[:, :17]) == (h * w * 55, 1, w * 55, 55)
    assert _channels_last_view(packed[:, 17:]) == (h * w * 55, 1, w * 55, 55)
    assert packed[:, 17:].storage_offset() == 17
    padded = torch.zeros(n, 64, h, w).contiguous(memory_format=torch.channels_last)
    assert _channels_last_view(padded[:, 38:55]) == (h * w * 64, 1, w * 64, 64)
    big = torch.zeros(2 * n, 64, h, w).contiguous(memory_format=torch.channels_last)
    assert _channels_last_view(big[::2, :38]) == (2 * h * w * 64, 1, w * 64, 64)
    # ambiguous layouts resolve to planar (and _image_strided passes them through)
    one = torch.zeros(1, C, h, w)
    assert _channels_last_view(one) is None and _image_strided(one)[0] is one
    dot = torch.zeros(n, C, 1, 1).contiguous(memory_format=torch.channels_last)
    assert _channels_last_view(dot) is None and _image_strided(dot)[0] is dot
    # every other column of a channels-last tensor is channels-last with twice the pixel stride
    assert _channels_last_view(packed[..., ::2]) == (h * w * 55, 1, (w // 2) * 110, 110)
    # neither family: copied (non-dense rows, W-major, channels 2 elements apart)
    for t in (planar[..., ::2], sep[:, :, ::2], packed[:, :17, ::2], torch.zeros(n, C, w, h).transpose(2, 3),
              torch.zeros(n, h, w, 2 * C)[..., ::2].permute(0, 3, 1, 2)):
        assert _channels_last_view(t) is None
        _, stride = _image_strided(t)
        assert stride == t.shape[1] * t.shape[2] * t.shape[3]


# =========================================================================== GPU
def _cl(t):
    import torch
    return t.contiguous(memory_format=torch.channels_last)


def _views(hmp, omp, layout, dtype):
    """Heat and offset maps of `layout` on the GPU in `dtype`."""
    import torch
    td = _torch_dtype(dtype)
    th, to = torch.from_numpy(hmp).to(td), torch.from_numpy(omp).to(td)
    n = hmp.shape[0]
    if layout in ('cl_separate', 'cl_odd'):
        return _cl(th.cuda()), _cl(to.cuda())
    if layout == 'mixed':
        return _cl(th.cuda()), to.cuda()
    if layout == 'cl_packed':             # heat first, P = 55; the offsets start at element 17
        buf = _cl(torch.cat((th, to), dim=1).cuda())
        return buf[:, :C], buf[:, C:]
    # offsets first, heat at element 38, P = 64: padding channels NaN, every other image of a
    # buffer twice as long (the images in between NaN too)
    buf = _cl(torch.full((2 * n, 64) + hmp.shape[2:], float('nan'), dtype=td, device='cuda'))
    hv, ov = buf[::2, L2:L2 + C], buf[::2, :L2]
    hv.copy_(th)
    ov.copy_(to)
    return hv, ov


def _engine():
    from test_fused_matrix import _engine as make
    return make()


@pytest.fixture(scope='module')
def eng(cuda_device):
    e = _engine()
    yield e
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('mode', ['bicubic', 'bilinear'])
@pytest.mark.parametrize('scale', [2, 4, 8])
@pytest.mark.parametrize('dtype', DTYPES)
def test_channels_last_matrix(eng, dtype, scale, mode, flip, layout):
    """Dets, limbs and poses of channels-last views equal the materialising path on dense float32
    copies bit for bit; dets equal the oracle's top-K, poses the C oracle's; the ring and
    checkerboard channels (bicubic) give dets >= thre from cells all below it."""
    from offsetguided_b200.engine import _channels_last_view
    h, w = SHAPES['odd' if layout == 'cl_odd' else 'dense']
    hmp, omp = matrix_inputs(h, w, scale, flip)
    n = hmp.shape[0] // 2 if flip else hmp.shape[0]
    hv, ov = _views(hmp, omp, layout, dtype)
    assert _channels_last_view(hv) is not None
    assert (_channels_last_view(ov) is None) == (layout == 'mixed')
    fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, scale, mode, flip, n)
    assert redo == 0
    _assert_same(fused, f_int, staged, s_int)
    ref_s, ref_i, fused_lo, ref_poses = _matrix_oracle(dtype, h, w, scale, mode, flip)
    ds, di, _ = f_int
    live = ref_s >= np.float32(THRE)
    assert np.array_equal(di[live], ref_i[live]) and np.array_equal(ds[live], ref_s[live])
    assert np.all(di[~live] == -1)
    assert len(fused) == len(ref_poses)
    for p, r in zip(fused, ref_poses):
        gio.compare_poses(p, r, rtol=RTOL)
    assert sum(len(p) for p in fused) >= 1
    assert (ds[:, SPIKES] >= THRE).sum() >= 4 and (ds[:, PROBES] >= THRE).sum() >= 2
    if mode == 'bicubic':
        for c in (RING, CHECKER):
            assert np.abs(fused_lo[:, c]).max() <= 1.0 and fused_lo[:, c].max() < THRE
            assert (ds[:, c] >= THRE).all(axis=-1).any(), c


def _bench_packed(seed, n, edge, flip, dtype='bf16'):
    """A packed [n or 2n, 55, h, w] channels_last head output of rendered scenes."""
    import bench
    import torch
    hmp, omp = bench.lowres_inputs(seed, n, edge, flip)
    omp[~np.isfinite(omp)] = 0
    buf = _cl(torch.cat((torch.from_numpy(hmp), torch.from_numpy(omp)), dim=1).to(_torch_dtype(dtype)).cuda())
    return buf


@pytest.mark.gpu
def test_decoded_in_place(eng):
    """No transposing copy: a call is 6 kernels (graph replay and kernel by kernel), and torch's
    peak allocation during a call grows by less than one heat slice."""
    import torch
    buf = _bench_packed(31, 8, 640, True)
    hv, ov = buf[:, :C], buf[:, C:]
    slice_bytes = hv.shape[0] * C * hv.shape[2] * hv.shape[3] * hv.element_size()
    ref = eng.decode_features(hv.float().contiguous(), ov.float().contiguous(), 4, 4, 'bicubic', (KP, FL, RS))
    for graph in (True, False):
        eng.set_graph(graph)
        eng.decode_features(hv, ov, 4, 4, 'bicubic', (KP, FL, RS))
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        l0 = eng.launch_count
        got = eng.decode_features(hv, ov, 4, 4, 'bicubic', (KP, FL, RS))
        assert eng.launch_count - l0 == 6
        assert torch.cuda.max_memory_allocated() - before < slice_bytes
        assert len(got) == len(ref) and all(np.array_equal(a, b) for a, b in zip(got, ref))
    eng.set_graph(True)
    assert sum(len(p) for p in ref) >= 8


@pytest.mark.gpu
@pytest.mark.parametrize('flip', [False, True], ids=['noflip', 'flip'])
@pytest.mark.parametrize('dtype', DTYPES)
def test_channels_last_overflow_redo(eng, dtype, flip):
    """One noise plane in a channels-last batch overflows its candidate list: the fetch redoes it
    from the strided maps and the call equals the materialising path."""
    import torch
    buf = _bench_packed(707, 2, 640, flip, dtype)
    rng = np.random.RandomState(11)
    noise = torch.from_numpy(rng.uniform(0, 1, size=buf.shape[2:]).astype(np.float32))
    buf[1, 6] = noise.to(buf.dtype).cuda()
    hv, ov = buf[:, :C], buf[:, C:]
    fused, f_int, staged, s_int, redo = _decode_both(eng, hv, ov, 4, 'bicubic', flip, 2)
    assert redo == 1
    _assert_same(fused, f_int, staged, s_int)
    assert sum(len(p) for p in fused) >= 4 and (f_int[0][1, 6] > 0).all()


@pytest.mark.gpu
def test_graph_key_includes_the_layout(eng):
    """The same channels-last buffers replay their graph; a planar view of the same storage,
    address and shape re-captures and decodes as that view's contiguous copy."""
    import torch
    buf = _bench_packed(55, 2, 320, True)
    hv = _cl(buf[:, :C].clone())
    ov = buf[:, C:]
    tables = (KP, FL, RS)
    first = eng.decode_features(hv, ov, 4, 4, 'bicubic', tables)
    r0, b0 = eng.graph_counts
    again = eng.decode_features(hv, ov, 4, 4, 'bicubic', tables)
    r1, b1 = eng.graph_counts
    assert b1 == b0 and r1 == r0 + 1
    assert all(np.array_equal(a, b) for a, b in zip(first, again))
    n, c, h, w = hv.shape
    planar = torch.as_strided(hv, hv.shape, (c * h * w, h * w, w, 1), hv.storage_offset())
    assert planar.data_ptr() == hv.data_ptr() and planar.shape == hv.shape
    got = eng.decode_features(planar, ov, 4, 4, 'bicubic', tables)
    assert eng.graph_counts[1] == b1 + 1
    want = eng.decode_features(planar.contiguous(), ov, 4, 4, 'bicubic', tables)
    assert len(got) == len(want) and all(np.array_equal(a, b) for a, b in zip(got, want))


def _post(topk=TOPK):
    import argparse
    from offsetguided_b200 import decoder
    p = argparse.ArgumentParser()
    decoder.decoder_cli(p)
    a = p.parse_args(['--topk', str(topk), '--thre-hmp', str(THRE), '--person-thre', str(THRE),
                      '--dist-max', '40', '--min-len', '0.5'])
    a.headnets, a.strides, a.batch_size = ['hmp', 'omp'], [4, 4], 8
    a.include_scale = a.include_jitter_offset = False
    return decoder.decoder_factory(a)


def _feats(h, o):
    return [[[h], [[]], [[]]], [[o], [[]], [[]]]]


@pytest.mark.gpu
def test_callers_decode_channels_last(cuda_device):
    """submit / collect, plan_features and generate_results on channels-last slices equal their
    results on contiguous copies."""
    import torch
    pp = _post()
    bufs = [_bench_packed(300 + i, 2, 320, True) for i in range(4)]
    refs = [pp.generate_poses(_feats(b[:, :C].contiguous(), b[:, C:].contiguous()), flip_test=True) for b in bufs]
    assert sum(len(p) for r in refs for p in r) >= 8
    for i in range(16):
        b = bufs[i % 4]
        pp.submit(_feats(b[:, :C], b[:, C:]), flip_test=True)
    for i in range(16):
        got = pp.collect()
        assert len(got) == len(refs[i % 4]) and all(np.array_equal(a, r) for a, r in zip(got, refs[i % 4]))
    eng = pp._engine(torch.device('cuda', 0))
    plan = eng.plan_features(bufs[0][:, :C], bufs[0][:, C:], 4, 4, 'bicubic', pp._flip_tables)
    assert plan.in_place
    plan.launch()
    got = plan.fetch()
    assert all(np.array_equal(a, r) for a, r in zip(got, refs[0]))
    rng = np.random.RandomState(2)
    metas = [{'offset': np.array([-float(rng.randint(0, 90)), -float(rng.randint(0, 60))]),
              'scale': np.array([rng.uniform(0.4, 1.7), rng.uniform(0.4, 1.7)]), 'hflip': False,
              'width_height': (640, 480), 'image_id': 90 + i} for i in range(2)]
    b = bufs[1]
    want = pp.generate_results(_feats(b[:, :C].contiguous(), b[:, C:].contiguous()), metas, flip_test=True)
    got = pp.generate_results(_feats(b[:, :C], b[:, C:]), metas, flip_test=True)
    assert all(np.array_equal(a, r) for a, r in zip(got[0], want[0]))
    for a, r in zip(got[1:], want[1:]):
        assert np.array_equal(a, r)


@pytest.mark.gpu
def test_bad_strides_are_refused_before_any_launch(eng):
    """og_decode_features_dev_strided / og_plan_features_strided refuse strides outside the two
    layouts on the host: nothing is launched and nothing is queued."""
    from offsetguided_b200 import _lib
    from offsetguided_b200.engine import _ptr, _stream_ptr
    buf = _bench_packed(3, 2, 128, False)
    hv, ov = buf[:, :C], buf[:, C:]
    n, _, h, w = hv.shape
    good_h, good_o = (h * w * 55, 1, w * 55, 55), (h * w * 55, 1, w * 55, 55)

    def call(hs, os_):
        return eng.lib.og_decode_features_dev_strided(
            eng._h, _ptr(hv), _ptr(ov), _lib.OG_DTYPE_BF16, _lib.int64_array(hs), _lib.int64_array(os_), n, h, w,
            4, 4, 1, 0, None, None, None, 0, _stream_ptr(eng.device))

    def plan(hs, os_):
        pid = ctypes.c_int32(-1)
        return eng.lib.og_plan_features_strided(
            eng._h, _ptr(hv), _ptr(ov), _lib.OG_DTYPE_BF16, _lib.int64_array(hs), _lib.int64_array(os_), n, h, w,
            4, 4, 1, 0, None, None, None, 0, ctypes.byref(pid))
    bad = [((h * w * 55, 1, w * 55 + 1, 55), good_o),        # row stride != w * p
           ((h * w * 55, 1, w * 16, 16), good_o),             # p < C
           ((h * w * 55, 2, w * 55, 55), good_o),             # channel stride 2
           (good_h, (h * w * 55, 1, w * 30, 30)),             # p < 2L
           ((h * w * 55 - 1, 1, w * 55, 55), good_o),         # images overlap
           ((C * h * w - 1, h * w, w, 1), good_o)]            # planar images overlap
    l0 = eng.launch_count
    for hs, os_ in bad:
        assert call(hs, os_) == 1, (hs, os_)
        assert plan(hs, os_) == 1, (hs, os_)
    assert eng.launch_count == l0 and eng.pending == 0
    assert call(good_h, good_o) == 0
    assert len(eng.fetch()) == n


@pytest.mark.gpu
def test_config5_handover(cuda_device):
    """A bf16 1 x 1 convolution head run channels-last (like the stand-in network of config 5),
    rendered persons added, batch 32 with flip-test: decoded in place, equal to the C oracle on
    the widened maps."""
    import bench
    import torch
    torch.manual_seed(0)
    n, edge = 32, 256
    hmp, omp = bench.lowres_inputs(5151, n, edge, True)
    omp[~np.isfinite(omp)] = 0
    synth = torch.cat((torch.from_numpy(hmp), torch.from_numpy(omp)), dim=1).cuda().to(torch.bfloat16)
    head = torch.nn.Conv2d(32, C + L2, 1).cuda().to(torch.bfloat16).to(memory_format=torch.channels_last)
    with torch.no_grad():
        head.weight.mul_(1e-3)
        x = _cl(torch.randn(2 * n, 32, edge // 4, edge // 4, device='cuda', dtype=torch.bfloat16))
        y = head(x)
        y.add_(_cl(synth))
    from offsetguided_b200.engine import _channels_last_view
    assert _channels_last_view(y[:, :C]) == (y.stride(0), 1, y.stride(2), C + L2)
    pp = _post()
    got = pp.generate_poses(_feats(y[:, :C], y[:, C:]), flip_test=True)
    wide = y.float().cpu().numpy()
    ref = co.generate_poses(np.ascontiguousarray(wide[:, :C]), np.ascontiguousarray(wide[:, C:]), SKEL, C,
                            topk=TOPK, thre_hmp=THRE, min_len=0.5, person_thre=THRE, dist_max=40.0, use_scale=True,
                            hmp_stride=4, off_stride=4, resize_mode='bicubic', flip_test=True, kp_flips=KP,
                            limb_flips=FL, limb_reserve=RS)
    assert len(got) == len(ref) == n and sum(len(p) for p in got) >= n
    for p, r in zip(got, ref):
        gio.compare_poses(p, r, rtol=RTOL)
