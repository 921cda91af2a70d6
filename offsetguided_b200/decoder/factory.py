"""Post-processing entry point (reference decoder/factory.py): ``decoder_cli``,
``decoder_factory(args)`` -> ``PostProcess``, ``PostProcess.generate_poses``."""
import argparse
import collections
import logging
import re

import numpy as np
import torch

from .. import config
from ..config import (COCO_KEYPOINTS, COCO_PERSON_SKELETON,
                      COCO_PERSON_WITH_REDUNDANT_SKELETON, DENSER_COCO_PERSON_SKELETON,
                      REDUNDANT_CONNECTIONS, KINEMATIC_TREE_SKELETON)
from ..engine import DecoderEngine
from .collect import LimbsCollect
from .group import GreedyGroup
from . import offset as _offset

LOG = logging.getLogger(__name__)


def boolean_string(s):
    """'False' / 'True' command-line values (reference utils/util.py:4-8)."""
    if s not in {'False', 'True'}:
        raise ValueError('Not a valid boolean string')
    return s == 'True'


class PostProcess(torch.nn.Module):
    """Network outputs -> per-image pose arrays (reference decoder/factory.py:21-96).

    Constructor arguments are the reference's.  No worker pool is forked: grouping runs
    on the GPU (one CTA per image) in the same stream as the rest of the decoder.
    """

    def __init__(self, batch_size, hmp_stride, off_stride, inter_mode, keypoints, skeleton,
                 limb_collector, limb_grouper, include_scale=False, include_jitter_offset=False,
                 hmp_index=0, omp_index=1, feat_stage=-1):
        super(PostProcess, self).__init__()
        self.batch_size = batch_size
        self.inter_mode = inter_mode
        self.hmp_stride = hmp_stride
        self.off_stride = off_stride
        self.keypoints = keypoints
        self.skeleton = skeleton
        self.limb_collect = limb_collector
        self.limb_group = limb_grouper
        self.hmp_index = hmp_index
        self.omp_index = omp_index
        self.feat_stage = feat_stage
        self.include_scale = include_scale
        self.include_jitter_offset = include_jitter_offset
        self.keypoints_flips = config.heatmap_hflip(keypoints)
        self.limbs_flips = config.offset_hflip(keypoints, skeleton)
        self.worker_pool = None          # the reference forks Pool(batch_size) here
        self._engines = {}
        self._flip_tables = (self.keypoints_flips, self.limbs_flips[0], self.limbs_flips[1])
        self._submitted = collections.deque()
        self._plans = {}
        LOG.info('use the inferred feature maps at stage %d, heatmap index is %d, offsetmap index '
                 'is %d, interpolate the predicted heatmaps using %s, grouping on the GPU',
                 feat_stage, hmp_index, omp_index, inter_mode)

    def _engine(self, device):
        key = (device.type, device.index)
        if key not in self._engines:
            lc, lg = self.limb_collect, self.limb_group
            self._engines[key] = DecoderEngine(
                len(self.keypoints), self.skeleton, topk=lc.K, thre_hmp=lc.thre_hmp,
                min_len=lc.min_len, resize_factor=lc.resize_factor, dist_max=lg.dist_max,
                use_scale=lg.use_scale, person_thre=lg.person_thre, sort_dim=lg.sort_dim,
                device=device)
        return self._engines[key]

    def generate_poses(self, features, flip_test=False, cat_flip_offs=False, scored_off=False):
        """Decode a batch (reference decoder/factory.py:52-96).

        ``features[hmp_index] = (out_hmps, out_bghmp, out_jomps)`` and
        ``features[omp_index] = (out_offsets, out_spreads, out_scales)``, each a list over
        stacks; stage ``feat_stage`` is used.  With ``flip_test`` the batch holds the
        originals followed by their W-flipped copies.  Tensors may live on the GPU (the
        normal case, right after ``model(images)``) or on the host.

        Returns a list with one (M_i, C, 6) float32 array per image.
        """
        out_hmps, out_bghmp, out_jomps = features[self.hmp_index]
        out_offsets, out_spreads, out_scales = features[self.omp_index]
        hmps = out_hmps[self.feat_stage]
        jomps = out_jomps[self.feat_stage]
        offs = out_offsets[self.feat_stage]
        scmps = out_scales[self.feat_stage]

        lc = self.limb_collect
        use_scale_maps = self.include_scale and lc.include_scale and isinstance(scmps, torch.Tensor)
        use_jitter_maps = (self.include_jitter_offset and lc.include_jitter_offset
                           and isinstance(jomps, torch.Tensor))
        device = hmps.device if hmps.is_cuda else torch.device('cuda', torch.cuda.current_device())
        eng = self._engine(device)
        tables = self._flip_tables if flip_test else None
        if scored_off or use_scale_maps or use_jitter_maps or (flip_test and cat_flip_offs):
            jomps = jomps if use_jitter_maps else None
            scmps = scmps if use_scale_maps else None
            fused_ok = (eng._fused and eng.thre_hmp > 0 and int(self.hmp_stride) in (2, 4, 8)
                        and int(self.hmp_stride) == int(self.off_stride) and hmps.shape[0] > 0)
            if not fused_ok:
                return self._generate_poses_staged(hmps, jomps, offs, scmps, flip_test, cat_flip_offs, scored_off)
            return self._generate_poses_heads(eng, hmps, jomps, offs, scmps, flip_test, cat_flip_offs, scored_off)
        return eng.decode_features(hmps, offs, self.hmp_stride, self.off_stride, self.inter_mode, tables)

    def generate_results(self, features, metas, flip_test=False):
        """generate_poses plus the caller's next step on the GPU: every pose back-projected into
        its original image frame and turned into the evaluation's result row (reference
        transforms/preprocess.py:33-63 + evaluate.py:227-265, per-image / per-person /
        per-keypoint Python loops there).  ``metas``: the batch's meta dictionaries ('offset',
        'scale', 'hflip', 'image_id').  Returns (batch_poses, keypoints (T, 3C) float32,
        scores (T,) float64, image_index (T,)): rows ordered by image then person rank, an image
        without persons holds the reference's all-zero row with score 0.01;
        ``results.rows_from_arrays`` turns the arrays into the COCO dictionaries."""
        from .. import results
        hmps = features[self.hmp_index][0][self.feat_stage]
        offs = features[self.omp_index][0][self.feat_stage]
        device = hmps.device if hmps.is_cuda else torch.device('cuda', torch.cuda.current_device())
        eng = self._engine(device)
        tables = self._flip_tables if flip_test else None
        poses = eng.decode_features(hmps, offs, self.hmp_stride, self.off_stride, self.inter_mode, tables,
                                    frames=results.frames_of(metas))
        rows = eng.last_result_rows
        if rows is None and not poses:
            # an empty batch runs no kernel, so nothing wrote rows; the reference's loops make none
            c = len(self.keypoints)
            rows = (np.zeros((0, 3 * c), np.float32), np.zeros((0,), np.float64), np.zeros((0,), np.int32),
                    np.zeros((0,), np.int32))
        return (poses,) + results.result_arrays(rows, len(self.keypoints))

    # ---- pipelined form of generate_poses ------------------------------------------------------
    # The reference call is synchronous: the host waits for every batch.  A decode of a few images
    # is ~0.05 ms of latency-bound kernels, so a caller that shards a batch over several GPUs (or
    # decodes while the network already runs the next batch) keeps several calls in flight:
    # submit() launches and returns at once, collect() returns the oldest result.
    def submit(self, features, flip_test=False):
        """generate_poses without the wait: launch the decode of ``features`` (default heads, no
        scored_off / cat_flip_offs) and return the number of calls now in flight (at most
        ``engine.OG_MAX_IN_FLIGHT``).  The tensors must stay unmodified until ``collect()``."""
        hmps = features[self.hmp_index][0][self.feat_stage]
        offs = features[self.omp_index][0][self.feat_stage]
        # A network writes its outputs to the same ADDRESSES batch after batch (new tensor objects,
        # same allocator blocks): the prepared call (validated shapes, converted arguments) is looked
        # up by buffer address + shape and launched with one foreign call, a CUDA-graph replay
        # inside the library.  A plan keeps no reference to the tensors it was made from.
        if hmps.is_cuda:
            key = (hmps.data_ptr(), offs.data_ptr(), hmps.shape, offs.shape, hmps.stride(), offs.stride(),
                   hmps.dtype, offs.dtype, flip_test, torch._C._cuda_getCurrentRawStream(hmps.device.index))
            plan = self._plans.get(key)
            if plan is not None and torch._C._cuda_getDevice() == plan.eng.device.index:
                plan.launch((hmps, offs))
                self._submitted.append(plan.eng)
                return len(self._submitted)
        device = hmps.device if hmps.is_cuda else torch.device('cuda', torch.cuda.current_device())
        eng = self._engine(device)
        tables = self._flip_tables if flip_test else None
        if (hmps.is_cuda and offs.is_cuda and hmps.is_contiguous() and offs.is_contiguous() and eng._fused
                and eng.thre_hmp > 0 and int(self.hmp_stride) in (2, 4, 8) and hmps.shape[0] > 0
                and hmps.dtype == offs.dtype and hmps.dtype in (torch.float32, torch.bfloat16, torch.float16)):
            with torch.cuda.device(device):
                plan = eng.plan_features(hmps, offs, self.hmp_stride, self.off_stride, self.inter_mode, tables)
                plan.launch()
                if plan.in_place:
                    if len(self._plans) >= 256:
                        self._plans.clear()
                    self._plans[key] = plan.release()
        else:
            eng.decode_features(hmps, offs, self.hmp_stride, self.off_stride, self.inter_mode, tables, fetch=False)
        self._submitted.append(eng)
        return len(self._submitted)

    def collect(self):
        """Poses of the oldest submitted batch: list of (M_i, C, 6) float32 arrays."""
        return self._submitted.popleft().fetch()

    def flip_augment(self, hmps, jomps, offs, scmps, cat_flip_offs, vector_nd):
        """Fuse the outputs of the original and the W-flipped images (reference
        decoder/factory.py:98-146; same arguments and return tuple).  ``hmps`` (2N, C, h, w) and
        ``offs`` (2N, 2L, h, w) hold the originals followed by the flipped copies; ``jomps`` /
        ``scmps`` are tensors only when the matching optional head is enabled.  Returns
        ``(hmps, jomps, offs, scmps, vector_nd)`` for N images; ``cat_flip_offs`` builds the 4-D
        offset vectors (vector_nd = 4) instead of averaging."""
        from .. import _lib
        from ..engine import as_cuda_f32, _ptr, _stream_ptr
        lib = _lib.load()
        hmps = as_cuda_f32(hmps)
        device = hmps.device
        offs = as_cuda_f32(offs, device)
        use_jomps = self.include_jitter_offset and isinstance(jomps, torch.Tensor)
        use_scmps = self.include_scale and isinstance(scmps, torch.Tensor)
        eng = self._engine(device)
        with torch.cuda.device(device):
            s = _stream_ptr(device)

            def flip_average(x, perm, negate_even):
                x = as_cuda_f32(x, device)
                n2, ch, h, w = x.shape
                out = torch.empty((n2 // 2, ch, h, w), dtype=torch.float32, device=device)
                _lib.check(lib.og_flip_average_f32(_ptr(x), _lib.int32_array(perm) if perm else None,
                                                   1 if negate_even else 0, n2 // 2, ch, h, w,
                                                   _ptr(out), s))
                return out

            n2, _, h, w = hmps.shape
            lf = _lib.int32_array(self.limbs_flips[0])
            lr = _lib.int32_array(self.limbs_flips[1])
            if cat_flip_offs:                                       # factory.py:115-127
                out = torch.empty((n2 // 2, 4 * len(self.skeleton), h, w), dtype=torch.float32,
                                  device=device)
                _lib.check(lib.og_flip_cat_offsets_f32(_ptr(offs), lf, lr, len(self.limbs_flips[1]),
                                                       n2 // 2, len(self.skeleton), h, w, _ptr(out), s))
                offs, vector_nd = out, 4
                hmps = flip_average(hmps, self.keypoints_flips, False)
            else:                                                   # factory.py:128-139
                fh = torch.empty((n2 // 2,) + tuple(hmps.shape[1:]), dtype=torch.float32, device=device)
                fo = torch.empty((n2 // 2,) + tuple(offs.shape[1:]), dtype=torch.float32, device=device)
                _lib.check(lib.og_flip_fuse_f32(eng._h, _ptr(hmps), _ptr(offs),
                                                _lib.int32_array(self.keypoints_flips), lf, lr,
                                                len(self.limbs_flips[1]), n2 // 2, h, w,
                                                _ptr(fh), _ptr(fo), s))
                hmps, offs = fh, fo
            if use_jomps:                                           # factory.py:109-113
                jomps = flip_average(jomps, None, True)
            if use_scmps:                                           # factory.py:141-144
                scmps = flip_average(scmps, self.keypoints_flips, False)
        return hmps, jomps, offs, scmps, vector_nd

    def _generate_poses_heads(self, eng, hmps, jomps, offs, scmps, flip_test, cat_flip_offs, scored_off):
        """The optional heads and flags on the fused path: no map is resized.  K2 interpolates the
        keypoint-scale / jitter-offset maps at the candidate pixels and combines the flip-test
        halves on the fly.  ``scored_off`` re-averages the offsets at NETWORK resolution
        (decoder/offset.py:8-43 runs before the resize, factory.py:67-69), so the flip-test
        halves are combined first, exactly as flip_augment does."""
        tables = self._flip_tables if flip_test else None
        if scored_off:
            if flip_test and cat_flip_offs:
                raise ValueError('scored_off cannot be combined with cat_flip_offs')
            vector_nd = 2
            if flip_test:
                hmps, jomps, offs, scmps, vector_nd = self.flip_augment(hmps, jomps, offs, scmps, False, vector_nd)
            jf, jt = _offset.pack_jtypes(self.skeleton)
            offs = _offset.scored_offset(hmps, offs, jf, jt, kernel_size=3)
            tables, cat_flip_offs = None, False
        return eng.decode_features_heads(hmps, offs, scmps, jomps, self.hmp_stride, self.off_stride,
                                         self.inter_mode, tables, cat_flip_offs,
                                         self.limb_collect.use_jitter_offset)

    def _generate_poses_staged(self, hmps, jomps, offs, scmps, flip_test, cat_flip_offs, scored_off):
        """The optional heads and flags (scored_off, keypoint-scale maps, jitter-offset maps,
        cat_flip_offs): the same kernels, called stage by stage through the C ABI on
        materialised maps (reference decoder/factory.py:67-91)."""
        from .. import _lib
        from ..engine import as_cuda_f32, _ptr, _stream_ptr
        lib = _lib.load()
        hmps = as_cuda_f32(hmps)
        device = hmps.device
        offs = as_cuda_f32(offs, device)
        scmps = as_cuda_f32(scmps, device) if scmps is not None else None
        jomps = as_cuda_f32(jomps, device) if jomps is not None else None
        eng = self._engine(device)
        mode = {'bilinear': 0, 'bicubic': 1}[self.inter_mode]
        vector_nd = 2
        if flip_test:
            hmps, jomps, offs, scmps, vector_nd = self.flip_augment(hmps, jomps, offs, scmps,
                                                                    cat_flip_offs, vector_nd)
        with torch.cuda.device(device):
            s = _stream_ptr(device)
            if scored_off:
                if vector_nd != 2:
                    raise ValueError('scored_off cannot be combined with cat_flip_offs')
                jf, jt = _offset.pack_jtypes(self.skeleton)
                offs = _offset.scored_offset(hmps, offs, jf, jt, kernel_size=3)

            def up(x, stride, m):
                if x is None or stride == 1:
                    return x
                n, c, h, w = x.shape
                out = torch.empty((n, c, h * stride, w * stride), dtype=torch.float32, device=device)
                _lib.check(lib.og_resize_f32(_ptr(x.contiguous()), _ptr(out), n * c, h, w, stride, m, s))
                return out
            hmps_hr = up(hmps, self.hmp_stride, mode)                   # factory.py:74-88
            offs_hr = up(offs, self.off_stride, 0)
            scmps_hr = up(scmps, self.off_stride, mode)
            jomps_hr = up(jomps, self.hmp_stride, 0)
            return eng.decode_maps(hmps_hr, offs_hr, scmps_hr, jomps=jomps_hr, vector_nd=vector_nd,
                                   use_jitter=self.limb_collect.use_jitter_offset)


def decoder_cli(parser):
    """Command-line flags of the decoder: the flag names, types, choices and defaults of the
    reference (decoder/factory.py:149-188), so that its launch commands keep working."""
    collect_flags = parser.add_argument_group('limb collections in post-processing')
    add = collect_flags.add_argument
    add('--resize-mode', default='bicubic', choices=['bilinear', 'bicubic'], type=str,
        help='how the heat maps are brought to decode resolution (offset maps are always bilinear)')
    add('--topk', default=48, type=int,
        help='peaks kept per heat-map channel = limb candidates per limb type (at most 128)')
    add('--thre-hmp', default=0.06, type=float,
        help='peaks scoring less than this are parked off-image and never form a limb')
    add('--min-len', default=0.5, type=float,
        help='lower clamp (pixels) of a limb length, guards the score of zero-length limbs')
    add('--feat-stage', default=-1, type=int,
        help='index of the network stack whose output maps are decoded')

    group_flags = parser.add_argument_group('greedy grouping in post-processing')
    add = group_flags.add_argument
    add('--person-thre', default=0.06, type=float,
        help='persons whose mean score falls below this are dropped')
    add('--sort-dim', default=2, choices=[2, 4], type=int,
        help='pose column the person score averages: 2 = keypoint score, 4 = limb score')
    add('--dist-max', default=20, type=float,
        help='largest distance (pixels) between a guided limb end and its matched keypoint; with '
             '--use-scale the keypoint scale takes over whenever it is larger')
    add('--use-scale', default=True, type=boolean_string,
        help='gate limbs by the regressed keypoint scale (needs a network built with --include-scale)')
    add('--use-jitter-offset', default=True, type=boolean_string,
        help='refine keypoint positions with the regressed jitter offsets (needs '
             '--include-jitter-offset)')


_OMP_SKELETONS = {
    'omp': COCO_PERSON_SKELETON, 'omp19': COCO_PERSON_SKELETON, 'omps': COCO_PERSON_SKELETON,
    'offset': COCO_PERSON_SKELETON, 'offsets': COCO_PERSON_SKELETON,
    'omp16': KINEMATIC_TREE_SKELETON,
    'omp31': COCO_PERSON_WITH_REDUNDANT_SKELETON,
    'omp44': DENSER_COCO_PERSON_SKELETON,
    'omp25': REDUNDANT_CONNECTIONS, 'omps25': REDUNDANT_CONNECTIONS,
}


def parse_heads(head_name, stride):
    """Head name -> keypoints / skeleton and stride (reference decoder/factory.py:191-231).
    Unlike the reference, 'hmp17' / 'hmps17' resolve to the COCO keypoints instead of
    leaving the variable unbound."""
    m = re.match('hmp[s]?([0-9]+)$', head_name)
    if head_name in ('hmp', 'hmps', 'heatmap', 'heatmaps') or m is not None:
        if m is not None:
            n_keypoints = int(m.group(1))
            assert n_keypoints == 17, f'{n_keypoints} keypoints not supported'
        return {'keypoints': COCO_KEYPOINTS, 'hmp_stride': stride}
    if head_name in _OMP_SKELETONS:
        return {'skeleton': _OMP_SKELETONS[head_name], 'omp_stride': stride}
    if re.match('omp[s]?([0-9]+)$', head_name) is not None:
        raise Exception('unknown skeleton type of head')
    raise Exception('unknown head to create an encoder: {}'.format(head_name))


def decoder_factory(args):
    """Build the PostProcess of a parsed command line (reference decoder/factory.py:234-267).
    Reads args.headnets, strides, topk, thre_hmp, min_len, include_jitter_offset,
    include_scale, use_jitter_offset, person_thre, sort_dim, dist_max, use_scale,
    batch_size, resize_mode, feat_stage."""
    temp_dic = {}
    for hd_name, stride in zip(args.headnets, args.strides):
        temp_dic.update(parse_heads(hd_name, stride))

    limb_handler = LimbsCollect(temp_dic['hmp_stride'], temp_dic['omp_stride'],
                                topk=args.topk, thre_hmp=args.thre_hmp, min_len=args.min_len,
                                include_jitter_offset=args.include_jitter_offset,
                                include_scale=args.include_scale,
                                use_jitter_offset=args.use_jitter_offset,
                                keypoints=temp_dic['keypoints'], skeleton=temp_dic['skeleton'])
    skeleton_grouper = GreedyGroup(args.person_thre, sort_dim=args.sort_dim,
                                   dist_max=args.dist_max, use_scale=args.use_scale,
                                   keypoints=temp_dic['keypoints'], skeleton=temp_dic['skeleton'])
    return PostProcess(args.batch_size, temp_dic['hmp_stride'], temp_dic['omp_stride'],
                       args.resize_mode, keypoints=temp_dic['keypoints'],
                       skeleton=temp_dic['skeleton'], limb_collector=limb_handler,
                       limb_grouper=skeleton_grouper, include_scale=args.include_scale,
                       include_jitter_offset=args.include_jitter_offset,
                       feat_stage=args.feat_stage)


def debug_parse_args():
    """Decoder flags at their defaults plus ``--for-debug`` (reference decoder/factory.py:270-280)."""
    parser = argparse.ArgumentParser(description='Test decoder')
    parser.add_argument('--for-debug', default=False, action='store_true',
                        help='this parse is only for debug the code')
    decoder_cli(parser)
    return parser.parse_args(['--for-debug'])
