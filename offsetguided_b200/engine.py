"""Host-side owner of one ``og_handle`` (one GPU, one decoder configuration).

PyTorch is used for device memory, streams and the numpy bridge only; every
computation is a call into libogdecoder.so through ``_lib``.
"""
import collections
import ctypes

import numpy as np
import torch

from . import _lib


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def as_cuda_f32(t, device=None):
    """Contiguous float32 CUDA view/copy of a tensor (CPU tensors are uploaded)."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    if not t.is_cuda:
        if not torch.cuda.is_available():
            raise _lib.OgError('a CUDA device is required: the decoder has no CPU fallback')
        t = t.to(device if device is not None else 'cuda')
    return t.contiguous().float()


_DTYPES = {torch.float32: _lib.OG_DTYPE_F32, torch.bfloat16: _lib.OG_DTYPE_BF16,
           torch.float16: _lib.OG_DTYPE_F16}


def _view(pointer, ctype, count, dtype):
    """numpy view of `count` elements behind a ctypes pointer (cheaper than np.ctypeslib.as_array)."""
    return np.frombuffer((ctype * count).from_address(ctypes.addressof(pointer.contents)), dtype=dtype)


def _image_strided(t):
    """(tensor, elements between images) for an NCHW tensor whose planes are dense and contiguous
    within an image (a channel slice of a packed head output qualifies); other layouts are
    made contiguous first."""
    n, c, h, w = t.shape
    st = t.stride()
    if st[3] == 1 and st[2] == w and st[1] == h * w and (n <= 1 or st[0] >= c * h * w):
        return t, (st[0] if n > 1 else c * h * w)
    return t.contiguous(), c * h * w


def _channels_last_view(t):
    """Element strides (s_n, 1, w * p, p) of an NCHW tensor stored channels-last: the channels of a
    pixel adjacent, pixels p >= c elements apart, rows dense (a channel slice of a packed
    ``channels_last`` head output qualifies; p is then the channel count of the whole tensor).
    None for any other layout and for one that is also planar (n = 1 contiguous, h = w = 1), which
    ``_image_strided`` handles.  Strides of size-1 dimensions are arbitrary and are not looked at."""
    n, c, h, w = t.shape
    st = t.stride()
    if ((w == 1 or st[3] == 1) and (h == 1 or st[2] == w) and (c == 1 or st[1] == h * w)
            and (n <= 1 or st[0] >= c * h * w)):
        return None
    if w > 1:
        p = st[3]
    elif h > 1:
        p = st[2]
    else:
        return None
    if p < c or (h > 1 and st[2] != w * p) or (c > 1 and st[1] != 1) or (n > 1 and st[0] < h * w * p):
        return None
    return (st[0] if n > 1 else h * w * p, 1, w * p, p)


def _planar_strides(t, image_stride):
    _, _, h, w = t.shape
    return (image_stride, h * w, w, 1)


class DecoderEngine(object):
    """One configured decoder bound to one CUDA device."""

    def __init__(self, n_keypoints, skeleton, *, topk, thre_hmp=0.06, min_len=0.5,
                 resize_factor=1.0, dist_max=20.0, use_scale=True, person_thre=0.06,
                 sort_dim=2, device=None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.OgError('a CUDA device is required: the decoder has no CPU fallback')
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None \
            else torch.device(device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.n_keypoints = int(n_keypoints)
        self.skeleton = [(int(a), int(b)) for a, b in skeleton]
        self.n_limbs = len(self.skeleton)
        self.topk = int(topk)
        self._from = _lib.int32_array([a for a, _ in self.skeleton])
        self._to = _lib.int32_array([b for _, b in self.skeleton])
        cfg = _lib.OgConfig(
            n_keypoints=self.n_keypoints, n_limbs=self.n_limbs,
            limb_from=ctypes.cast(self._from, _lib.c_int32_p),
            limb_to=ctypes.cast(self._to, _lib.c_int32_p),
            topk=self.topk, thre_hmp=float(thre_hmp), min_len=float(min_len),
            resize_factor=float(resize_factor), dist_max=float(dist_max),
            use_scale=1 if use_scale else 0, person_thre=float(person_thre),
            sort_dim=int(sort_dim), device=self.device.index, max_images=0)
        self.thre_hmp = float(thre_hmp)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_create(ctypes.byref(cfg), ctypes.byref(handle)))
        self._h = handle
        # input tensors of the decode calls in flight: K2 reads the offset maps on the handle's
        # stream after the call has returned, so they must outlive the call (until its fetch)
        self._inflight = collections.deque()
        self._fused = True
        self._flip_cache = {}
        self._result = _lib.OgResult()
        self._result_ref = ctypes.byref(self._result)
        # prepared ctypes argument tuples of device-path decodes, keyed by buffers / shapes / flags
        self._arg_cache = collections.OrderedDict()
        self._views = {}
        self._fetch_fn = self.lib.og_fetch_result
        self.last_result_rows = None

    def close(self):
        if getattr(self, '_h', None):
            with torch.cuda.device(self.device):
                self.lib.og_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self):
        return int(self.lib.og_launch_count(self._h))

    # ---- single stages -----------------------------------------------------
    def nms_topk(self, heat, thre=None):
        """K1.  heat (N, C, H, W) CUDA f32 -> scores (N, C, K) f32, inds (N, C, K) i32,
        counts (N, C) i32."""
        heat = as_cuda_f32(heat, self.device)
        n, c, h, w = heat.shape
        assert c == self.n_keypoints, 'heat map channel count differs from the keypoint list'
        scores = torch.empty((n, c, self.topk), dtype=torch.float32, device=self.device)
        inds = torch.empty((n, c, self.topk), dtype=torch.int32, device=self.device)
        counts = torch.empty((n, c), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_nms_topk_f32(
                self._h, _ptr(heat), n, h, w, float(self.thre_hmp if thre is None else thre),
                _ptr(scores), _ptr(inds), _ptr(counts), _stream_ptr(self.device)))
        return scores, inds, counts

    def topk_channel(self, scores_map, k):
        scores_map = as_cuda_f32(scores_map, self.device)
        n, c, h, w = scores_map.shape
        scores = torch.empty((n, c, k), dtype=torch.float32, device=self.device)
        inds = torch.empty((n, c, k), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_topk_channel_f32(
                self._h, _ptr(scores_map), n, c, h, w, int(k), _ptr(scores), _ptr(inds),
                _stream_ptr(self.device)))
        return scores, inds

    def limb_score(self, det_scores, det_inds, offs, scales=None, jomps=None, vector_nd=2,
                   use_jitter=False):
        """K2.  -> limbs (N, L, K, 13) CUDA f32.  ``jomps`` (N, 2, H, W) jitter-offset maps and
        ``vector_nd=4`` (cat_flip_offs offsets, 4L channels) are the optional variants."""
        offs = as_cuda_f32(offs, self.device)
        n, l2, h, w = offs.shape
        assert l2 == vector_nd * self.n_limbs, 'offset map channel count differs from vector_nd * limbs'
        det_scores = as_cuda_f32(det_scores, self.device)
        det_inds = det_inds.to(self.device, torch.int32).contiguous()
        if scales is not None:
            scales = as_cuda_f32(scales, self.device)
        if jomps is not None:
            jomps = as_cuda_f32(jomps, self.device)
        limbs = torch.empty((n, self.n_limbs, self.topk, _lib.OG_LIMB_COLS),
                            dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_limb_score_ex_f32(
                self._h, _ptr(det_scores), _ptr(det_inds), _ptr(offs), _ptr(scales), _ptr(jomps),
                int(vector_nd), 1 if use_jitter else 0, n, h, w, _ptr(limbs),
                _stream_ptr(self.device)))
        return limbs

    def group(self, limbs):
        """K3.  limbs (N, L, K, 13) -> list of N numpy arrays (M_i, C, 6)."""
        limbs = as_cuda_f32(limbs, self.device)
        n = limbs.shape[0]
        assert tuple(limbs.shape[1:]) == (self.n_limbs, self.topk, _lib.OG_LIMB_COLS), \
            'check the skeleton config and input limbs Tensor'
        if n == 0:
            return []
        cap = max(1, n * self.n_limbs * self.topk)
        poses = torch.empty((cap, self.n_keypoints, _lib.OG_POSE_COLS), dtype=torch.float32,
                            device=self.device)
        meta = torch.empty((2 * n + 1,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_group_f32(
                self._h, _ptr(limbs), n, _ptr(poses), cap, _ptr(meta[:n]), _ptr(meta[n:2 * n]),
                _ptr(meta[2 * n:]), _stream_ptr(self.device)))
        meta_h = meta.cpu().numpy()
        total = int(meta_h[2 * n])
        poses_h = poses[:total].cpu().numpy()
        return [poses_h[meta_h[i]:meta_h[i] + meta_h[n + i]].copy() for i in range(n)]

    # ---- whole path ----------------------------------------------------------
    def _fetch(self):
        """Result of the OLDEST decode call in flight: list of (M_i, C, 6) arrays, one per image
        of that call (the library reports the image count of the slot it hands out)."""
        if torch._C._cuda_getDevice() == self.device.index:
            st = self._fetch_fn(self._h, self._result_ref)
        else:
            with torch.cuda.device(self.device):
                st = self._fetch_fn(self._h, self._result_ref)
        if st != 0:
            _lib.check(st)
        if self._inflight:
            self._inflight.popleft()
        r = self._result
        n, total, c = r.n_images, r.total_rows, self.n_keypoints
        self.last_result_rows = None
        if r.coco_keypoints:
            # (keypoints (T, 3C) float32, scores (T,) float64, image index (T,) int32, persons per image (n,))
            if total:
                kp = np.frombuffer((ctypes.c_float * (total * 3 * c)).from_address(
                    ctypes.cast(r.coco_keypoints, ctypes.c_void_p).value), dtype=np.float32).reshape(total, 3 * c).copy()
                sc = np.frombuffer((ctypes.c_double * total).from_address(
                    ctypes.cast(r.coco_scores, ctypes.c_void_p).value), dtype=np.float64).copy()
                im = np.frombuffer((ctypes.c_int32 * total).from_address(
                    ctypes.cast(r.coco_images, ctypes.c_void_p).value), dtype=np.int32).copy()
            else:
                kp, sc, im = np.zeros((0, 3 * c), np.float32), np.zeros((0,), np.float64), np.zeros((0,), np.int32)
            cn = np.frombuffer((ctypes.c_int32 * n).from_address(
                ctypes.cast(r.counts, ctypes.c_void_p).value), dtype=np.int32).copy() if n else np.zeros((0,), np.int32)
            self.last_result_rows = (kp, sc, im, cn)
        if n == 0:
            return []
        if total == 0:
            return [np.zeros((0, c, _lib.OG_POSE_COLS), dtype=np.float32) for _ in range(n)]
        # numpy views over the result slot's pinned buffers are made once per (buffer, batch size):
        # buffer_id changes when the library has re-allocated the buffer, and the pose rows start
        # behind a header whose size depends on n
        per_row = c * _lib.OG_POSE_COLS
        view_key = (r.buffer_id, n)
        views = self._views.get(view_key)
        if views is None or views[1].size < total * per_row:
            addr = ctypes.cast(r.offsets, ctypes.c_void_p).value
            paddr = ctypes.cast(r.poses, ctypes.c_void_p).value
            grow = max(total, 64 * n) * per_row
            views = (np.frombuffer((ctypes.c_int32 * (2 * n)).from_address(addr), dtype=np.int32),
                     np.frombuffer((ctypes.c_float * grow).from_address(paddr), dtype=np.float32))
            if len(self._views) > 4 * _lib.OG_MAX_IN_FLIGHT:          # buffers the library has replaced
                self._views.clear()
            self._views[view_key] = views
        meta, pool = views
        offs = meta[:n].tolist()
        cnts = meta[n:2 * n].tolist()
        # one copy out of the handle's pinned buffer; the per-image arrays are views of it
        rows = pool[:total * per_row].copy().reshape(total, c, _lib.OG_POSE_COLS)
        return [rows[o:o + k] for o, k in zip(offs, cnts)]

    def _finish(self, keep_alive, fetch, n):
        """Book-keeping after a decode launch: the inputs stay referenced until the call is
        fetched; a synchronous call drains the queue IN ORDER and returns its own result."""
        self._inflight.append(keep_alive)
        if not fetch:
            return n
        if len(self._inflight) > 1:
            raise _lib.OgError('fetch=True while %d earlier decode calls are pending: fetch() them first '
                               '(results are handed out in launch order)' % (len(self._inflight) - 1))
        return self._fetch()

    def decode_maps(self, heat, offs, scales=None, fetch=True, jomps=None, vector_nd=2,
                    use_jitter=False):
        """generate_limbs + group_skeletons on full-resolution maps (K1 -> K2 -> K3).
        With ``fetch=False`` the call only launches (up to OG_MAX_IN_FLIGHT calls may be in
        flight); ``fetch()`` later returns the oldest pending result."""
        heat = as_cuda_f32(heat, self.device)
        offs = as_cuda_f32(offs, self.device)
        if scales is not None:
            scales = as_cuda_f32(scales, self.device)
        if jomps is not None:
            jomps = as_cuda_f32(jomps, self.device)
        n, c, h, w = heat.shape
        self._check_heads(heat.shape, offs.shape, vector_nd, False)
        if scales is not None and tuple(scales.shape) != tuple(heat.shape):
            raise ValueError('keypoint-scale maps %s do not match the heat maps %s'
                             % (tuple(scales.shape), tuple(heat.shape)))
        if jomps is not None and tuple(jomps.shape) != (n, 2, h, w):
            raise ValueError('jitter-offset maps must be (N, 2, H, W) = %s, got %s'
                             % ((n, 2, h, w), tuple(jomps.shape)))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_decode_maps_ex(self._h, _ptr(heat), _ptr(offs), _ptr(scales),
                                                  _ptr(jomps), int(vector_nd), 1 if use_jitter else 0,
                                                  n, h, w, _stream_ptr(self.device)))
            return self._finish((heat, offs, scales, jomps), fetch, n)

    def _check_heads(self, hmp_shape, off_shape, vector_nd, flip):
        """The C ABI takes one (n, h, w) and infers the channel counts from the configuration, so a
        mismatched head would read out of bounds on the device: validate here (the reference
        asserts the spatial part at decoder/collect.py:81)."""
        if len(hmp_shape) != 4 or len(off_shape) != 4:
            raise ValueError('heat / offset maps must be 4-D (N, C, H, W) tensors')
        if hmp_shape[1] != self.n_keypoints:
            raise ValueError('heat maps have %d channels but the decoder is configured for %d keypoints'
                             % (hmp_shape[1], self.n_keypoints))
        if off_shape[1] != vector_nd * self.n_limbs:
            raise ValueError('offset maps have %d channels but the skeleton has %d limbs (x %d components)'
                             % (off_shape[1], self.n_limbs, vector_nd))
        if tuple(off_shape[-2:]) != tuple(hmp_shape[-2:]):
            raise ValueError('spatial resolution should be equal: heat %s vs offsets %s'
                             % (tuple(hmp_shape[-2:]), tuple(off_shape[-2:])))
        if off_shape[0] != hmp_shape[0]:
            raise ValueError('heat and offset maps hold different numbers of images: %d vs %d'
                             % (hmp_shape[0], off_shape[0]))
        if flip and hmp_shape[0] % 2:
            raise ValueError('flip-test inputs hold the originals followed by their mirrored copies: '
                             'the batch must be even, got %d' % hmp_shape[0])

    def stage_frames(self, frames):
        """Image frames of the NEXT decode call: (n, 4) float64 rows (offset_x, offset_y, scale_x,
        scale_y) = meta['offset'], meta['scale'] of every image.  That call then also produces the
        back-projected result rows on the GPU (``last_result_rows`` after its fetch)."""
        frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(-1, 4)
        _lib.check(self.lib.og_set_frames(self._h, frames.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                          frames.shape[0]))

    def decode_features(self, hmp, off, hmp_stride, off_stride, resize_mode='bicubic',
                        flip_tables=None, fetch=True, frames=None):
        """PostProcess.generate_poses on network-resolution maps.  ``hmp`` / ``off`` are
        either CUDA tensors or CPU tensors (pinned memory gives asynchronous copies).
        ``flip_tables`` = (kp_flips, limb_flips, limb_reserve) enables flip fusion; the
        inputs then hold the originals followed by the W-flipped copies.  ``frames``: see
        ``stage_frames``."""
        if frames is not None:
            self.stage_frames(frames)
        on_host = not hmp.is_cuda
        flip = flip_tables is not None
        if not on_host:
            # Device maps, the call evaluate.py makes after model(images): a network writes its
            # outputs to the same buffers batch after batch, so everything that depends only on
            # (buffers, shapes, flags) — validation, layout analysis, ctypes conversion — is done
            # once and looked up afterwards; the library replays its CUDA graph for the same key.
            key = (hmp.data_ptr(), off.data_ptr(), hmp.shape, off.shape, hmp.stride(), off.stride(),
                   hmp.dtype, off.dtype, hmp_stride, off_stride, resize_mode, id(flip_tables))
            hit = self._arg_cache.get(key)
            if hit is not None and (not flip or hit[3] is flip_tables):
                fn, args, n, _ = hit
                stream = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
                if torch.cuda.current_device() == self.device.index:
                    st = fn(*args, stream)
                else:
                    with torch.cuda.device(self.device):
                        st = fn(*args, stream)
                if st != 0:
                    _lib.check(st)
                return self._finish((hmp, off), fetch, n)
        mode = {'bilinear': 0, 'bicubic': 1}[resize_mode]
        assert hmp.is_cuda == off.is_cuda, 'heat and offset maps must live on the same side'
        self._check_heads(hmp.shape, off.shape, 2, flip)
        args = self._flip_args(flip_tables) if flip else (None, None, None, 0)
        # Device maps as a reduced-precision network leaves them (bf16 / f16, channel slices of
        # one packed head output, channels-last) are decoded in place on the fused path; anything
        # else becomes dense float32.
        in_place = (not on_host and self._fused and self.thre_hmp > 0 and int(hmp_stride) in (2, 4, 8)
                    and hmp.shape[0] > 0 and hmp.dtype == off.dtype
                    and hmp.dtype in _DTYPES)
        src_hmp, src_off = hmp, off
        hcl = ocl = None
        if in_place:
            # channels-last maps (a network run in torch.channels_last) are read in place; the
            # other map of the pair may be planar
            hcl, ocl = _channels_last_view(hmp), _channels_last_view(off)
            if hcl is None:
                hmp, hmp_is = _image_strided(hmp)
            if ocl is None:
                off, off_is = _image_strided(off)
            in_place = (hcl is not None or ocl is not None or hmp.dtype != torch.float32
                        or hmp_is != hmp.shape[1] * hmp.shape[2] * hmp.shape[3]
                        or off_is != off.shape[1] * off.shape[2] * off.shape[3])
        if not in_place:
            hmp = hmp.contiguous().float()
            off = off.contiguous().float()
        n_in, c, h, w = hmp.shape
        n = n_in // 2 if flip else n_in
        if in_place and (hcl is not None or ocl is not None):
            fn = self.lib.og_decode_features_dev_strided
            hs = _lib.int64_array(hcl if hcl is not None else _planar_strides(hmp, hmp_is))
            os_ = _lib.int64_array(ocl if ocl is not None else _planar_strides(off, off_is))
            call = (self._h, _ptr(hmp), _ptr(off), _DTYPES[hmp.dtype], hs, os_, n, h, w,
                    int(hmp_stride), int(off_stride), mode, 1 if flip else 0) + tuple(args)
        elif in_place:
            fn = self.lib.og_decode_features_dev_ex
            call = (self._h, _ptr(hmp), _ptr(off), _DTYPES[hmp.dtype], hmp_is, off_is, n, h, w,
                    int(hmp_stride), int(off_stride), mode, 1 if flip else 0) + tuple(args)
        else:
            fn = self.lib.og_decode_features_host if on_host else self.lib.og_decode_features_dev
            call = (self._h, _ptr(hmp), _ptr(off), n, h, w, int(hmp_stride), int(off_stride),
                    mode, 1 if flip else 0) + tuple(args)
        with torch.cuda.device(self.device):
            _lib.check(fn(*call, _stream_ptr(self.device)))
        if not on_host and hmp is src_hmp and off is src_off:
            # the library was handed the caller's own buffers: the conversion can be reused
            self._arg_cache[key] = (fn, call, n, flip_tables)
            while len(self._arg_cache) > 64:
                self._arg_cache.popitem(last=False)
        return self._finish((hmp, off), fetch, n)

    def decode_features_heads(self, hmp, off, scales=None, jomps=None, hmp_stride=4, off_stride=4,
                              resize_mode='bicubic', flip_tables=None, cat_flip_offs=False,
                              use_jitter=False, fetch=True):
        """decode_features with the optional heads on the fused path: keypoint-scale maps and
        jitter-offset maps at NETWORK resolution are interpolated by K2 at the candidate pixels
        (flip-test averages fused in), ``cat_flip_offs`` scores limbs on the 4-D [original,
        mirrored] offset vectors.  Device-resident maps (anything else is converted to dense
        float32 on the device first)."""
        flip = flip_tables is not None
        self._check_heads(hmp.shape, off.shape, 2, flip)
        mode = {'bilinear': 0, 'bicubic': 1}[resize_mode]
        hmp = as_cuda_f32(hmp, self.device)
        off = as_cuda_f32(off, self.device)
        n_in, c, h, w = hmp.shape
        keep = [hmp, off]
        for t, ch in ((scales, c), (jomps, 2)):
            if t is not None and tuple(t.shape) != (n_in, ch, h, w):
                raise ValueError('optional head of shape %s, expected %s' % (tuple(t.shape), (n_in, ch, h, w)))
        scales = as_cuda_f32(scales, self.device) if scales is not None else None
        jomps = as_cuda_f32(jomps, self.device) if jomps is not None else None
        keep += [scales, jomps]
        args = self._flip_args(flip_tables) if flip else (None, None, None, 0)
        n = n_in // 2 if flip else n_in
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_decode_features_heads_dev(
                self._h, _ptr(hmp), _ptr(off), _ptr(scales) if scales is not None else None,
                _ptr(jomps) if jomps is not None else None, n, h, w, int(hmp_stride), int(off_stride), mode,
                1 if flip else 0, 1 if cat_flip_offs else 0, 1 if use_jitter else 0, *args,
                _stream_ptr(self.device)))
        return self._finish(tuple(keep), fetch, n)

    def plan_features(self, hmp, off, hmp_stride, off_stride, resize_mode='bicubic', flip_tables=None):
        """A prepared decode of DEVICE-resident network-resolution maps for callers that decode the
        same buffers batch after batch (a network writes its outputs in place): shapes are
        validated and every ctypes argument is converted once; ``plan.launch()`` is then one
        foreign call (a CUDA-graph replay inside the library) and ``plan.fetch()`` another."""
        return FeaturePlan(self, hmp, off, hmp_stride, off_stride, resize_mode, flip_tables)

    def _flip_args(self, flip_tables):
        """ctypes views of (kp_flips, limb_flips, limb_reserve), built once per table set."""
        key = tuple(id(t) for t in flip_tables)          # the tables are long-lived config lists
        hit = self._flip_cache.get(key)
        if hit is None or any(a is not b for a, b in zip(hit[0], flip_tables)):
            arrays = tuple(_lib.int32_array(t) for t in flip_tables)
            hit = (tuple(flip_tables), arrays,
                   tuple(ctypes.cast(a, _lib.c_int32_p) for a in arrays) + (len(flip_tables[2]),))
            self._flip_cache[key] = hit
        return hit[2]

    def fetch(self, n=None):
        """Result of the oldest decode call launched with ``fetch=False`` (``n`` is accepted for
        compatibility; the library knows the image count of every call in flight)."""
        return self._fetch()

    @property
    def pending(self):
        return int(self.lib.og_pending(self._h))

    def set_fused(self, on=True):
        """Enable / disable the fused network-resolution path of decode_features."""
        _lib.check(self.lib.og_set_fused(self._h, 1 if on else 0))
        self._fused = bool(on)
        self._arg_cache.clear()

    @property
    def fused_redo_count(self):
        return int(self.lib.og_fused_redo_count(self._h))

    @property
    def k3_redo_count(self):
        """Fetches that ran the CTA grouping kernel for images whose person table outgrew the warp kernel's."""
        return int(self.lib.og_k3_redo_count(self._h))

    def set_graph(self, on=True):
        """Device path: replay a captured CUDA graph per result slot (default) or launch kernel by kernel."""
        _lib.check(self.lib.og_set_graph(self._h, 1 if on else 0))

    @property
    def graph_counts(self):
        """(replays, captures) of the device-path graphs."""
        return int(self.lib.og_graph_replay_count(self._h)), int(self.lib.og_graph_build_count(self._h))

    def set_zero_copy(self, on=True):
        """Host inputs on the fused path: leave the offset maps in pinned host memory and let K2
        gather its samples over PCIe (default), or copy them as a whole."""
        _lib.check(self.lib.og_set_zero_copy(self._h, 1 if on else 0))

    @property
    def zero_copy_count(self):
        return int(self.lib.og_zero_copy_count(self._h))

    def enable_stage_timing(self, on=True):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_enable_stage_timing(self._h, 1 if on else 0))

    def last_stage_times_ms(self):
        """{prep, k1_stream, k1_select, k2, k3, d2h} of the last decode call, in ms."""
        out = (ctypes.c_float * 6)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_last_stage_times_ms(self._h, out))
        return dict(zip(('prep', 'k1_stream', 'k1_select', 'k2', 'k3', 'd2h'), [float(v) for v in out]))

    def last_intermediates(self, n):
        """Copies of the last decode call's dets (scores, indices) and limbs."""
        c, k, l = self.n_keypoints, self.topk, self.n_limbs
        ds = torch.empty((n, c, k), dtype=torch.float32, device=self.device)
        di = torch.empty((n, c, k), dtype=torch.int32, device=self.device)
        lb = torch.empty((n, l, k, _lib.OG_LIMB_COLS), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.og_copy_intermediates(self._h, n, _ptr(ds), _ptr(di), _ptr(lb),
                                                      _stream_ptr(self.device)))
        return ds, di, lb


class FeaturePlan(object):
    """See DecoderEngine.plan_features.  The plan holds converted arguments only: ``launch(keep)``
    takes the tensors to keep referenced until the call has been fetched (default: the ones the
    plan was made from)."""

    def __init__(self, eng, hmp, off, hmp_stride, off_stride, resize_mode, flip_tables):
        if not (hmp.is_cuda and off.is_cuda):
            raise ValueError('plan_features takes device-resident maps; host maps go through decode_features')
        flip = flip_tables is not None
        eng._check_heads(hmp.shape, off.shape, 2, flip)
        mode = {'bilinear': 0, 'bicubic': 1}[resize_mode]
        args = eng._flip_args(flip_tables) if flip else (None, None, None, 0)
        src = (hmp, off)
        if hmp.dtype != off.dtype or hmp.dtype not in _DTYPES:
            hmp, off = hmp.float(), off.float()
        hcl, ocl = _channels_last_view(hmp), _channels_last_view(off)
        if hcl is None:
            hmp, hmp_is = _image_strided(hmp)
        if ocl is None:
            off, off_is = _image_strided(off)
        n_in, _, h, w = hmp.shape
        self.n = n_in // 2 if flip else n_in
        self.eng = eng
        self.in_place = hmp is src[0] and off is src[1]      # the library reads the caller's own buffers
        self.keep = (hmp, off)
        self.flip_tables = flip_tables
        self.stream_ptr = torch.cuda.current_stream(eng.device).cuda_stream
        plan_id = ctypes.c_int32(-1)
        with torch.cuda.device(eng.device):
            if hcl is not None or ocl is not None:
                hs = _lib.int64_array(hcl if hcl is not None else _planar_strides(hmp, hmp_is))
                os_ = _lib.int64_array(ocl if ocl is not None else _planar_strides(off, off_is))
                _lib.check(eng.lib.og_plan_features_strided(
                    eng._h, _ptr(hmp), _ptr(off), _DTYPES[hmp.dtype], hs, os_, self.n, h, w, int(hmp_stride),
                    int(off_stride), mode, 1 if flip else 0, *args, ctypes.byref(plan_id)))
            else:
                _lib.check(eng.lib.og_plan_features(
                    eng._h, _ptr(hmp), _ptr(off), _DTYPES[hmp.dtype], hmp_is, off_is, self.n, h, w,
                    int(hmp_stride), int(off_stride), mode, 1 if flip else 0, *args, ctypes.byref(plan_id)))
        self._fn = eng.lib.og_plan_launch
        self._handle = eng._h
        self._id = plan_id.value
        self._stream = ctypes.c_void_p(self.stream_ptr)
        self._append = eng._inflight.append

    def launch(self, keep=None):
        """Launch one decode of the planned buffers on the stream that was current when the plan
        was made (the CUDA device of the engine must be current)."""
        st = self._fn(self._handle, self._id, self._stream)
        if st != 0:
            _lib.check(st)
        self._append(self.keep if keep is None else keep)

    def release(self):
        """Drop the references to the planned tensors (a cached plan is launched with the caller's
        current tensor objects as ``keep``)."""
        self.keep = None
        return self

    def fetch(self):
        return self.eng._fetch()
