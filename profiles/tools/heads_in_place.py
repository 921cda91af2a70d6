"""Hand-over of the optional heads (keypoint scales, jitter offsets) to the decoder.

Workload: bench.py's config 2 (batch 64, flip-test, COCO 17 keypoints / 19 limbs, 160 x 160 maps)
plus a keypoint-scale head (17 channels) and a jitter-offset head (2 channels), all four maps in
float16 as an AMP network leaves them, once as four separate planar tensors and once as four
channels-last tensors.  Two arms through PostProcess.generate_poses with --include-scale and
--include-jitter-offset:
  a_convert   explicit `.contiguous().float()` copies of the four maps (the hand-over before the
              heads were read in place),
  b_in_place  the maps themselves.
Each call is timed with CUDA events around the synchronous generate_poses (it ends with the fetch);
the arms alternate after a warm-up until each has run for at least `--seconds`.  Medians and the
10th / 90th percentiles per call are reported with the card's name and power limit.

`--k2-stage --tree DIR` instead records the K2 stage time (og_enable_stage_timing) of the
default-heads decode of the bench workload (bf16 planar maps, no optional heads) with the package in
DIR, so that two commits can be compared in one session.

    python profiles/tools/heads_in_place.py [--seconds S] > out.json
    python profiles/tools/heads_in_place.py --k2-stage --tree DIR [--calls N]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ', power limit not read'


def make_post(w, heads):
    from offsetguided_b200 import decoder
    ap = argparse.ArgumentParser()
    decoder.decoder_cli(ap)
    dargs = ap.parse_args(['--topk', str(w['topk']), '--thre-hmp', str(w['thre_hmp']),
                           '--person-thre', str(w['person_thre']), '--dist-max', str(w['dist_max'])])
    dargs.headnets, dargs.strides, dargs.batch_size = ['hmp', 'omp'], [4, 4], w['batch']
    dargs.include_scale = dargs.include_jitter_offset = heads
    return decoder.decoder_factory(dargs)


def workload():
    import bench

    class _Args(object):
        workload, no_flip, batch, long_edge = 'cfg2', False, 0, 0
    return bench.workload(_Args())


def heads_inputs(w):
    """(hmp, omp, scm, jom) float32 numpy maps of the workload with flip-test."""
    import numpy as np
    import bench
    hmp, omp = bench.lowres_inputs(4100, w['batch'], w['edge'], True, w)
    omp[~np.isfinite(omp)] = 0
    rng = np.random.RandomState(4101)
    n2, _, h, ww = hmp.shape
    scm = rng.uniform(2, 60, size=(n2, w['c'], h, ww)).astype(np.float32)
    jom = rng.uniform(-1.5, 1.5, size=(n2, 2, h, ww)).astype(np.float32)
    return hmp, omp, scm, jom


def feats(maps):
    hv, ov, sv, jv = maps
    return [[[hv], [[]], [jv]], [[ov], [[]], [sv]]]


def measure(post, maps, label, seconds, warmup=5, min_rounds=30):
    import numpy as np
    import torch

    def convert():
        return post.generate_poses(feats(tuple(t.contiguous().float() for t in maps)), flip_test=True)

    def in_place():
        return post.generate_poses(feats(maps), flip_test=True)

    arms = (('a_convert', convert), ('b_in_place', in_place))
    ref = {name: fn() for name, fn in arms}
    same = len(ref['a_convert']) == len(ref['b_in_place']) and all(
        np.array_equal(x, y) for x, y in zip(ref['a_convert'], ref['b_in_place']))
    for _ in range(warmup):
        for _, fn in arms:
            fn()
    times = {name: [] for name, _ in arms}
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while min(sum(v) for v in times.values()) < seconds * 1e3 or len(times['a_convert']) < min_rounds:
        for name, fn in arms:
            torch.cuda.synchronize()
            start.record()
            fn()
            end.record()
            end.synchronize()
            times[name].append(start.elapsed_time(end))
    elements = sum(t.numel() for t in maps)
    return {
        'layout': label, 'dtype': 'f16', 'flip_test': True, 'shapes': [list(t.shape) for t in maps],
        'elements_m': round(elements / 1e6, 1),
        'conversion_bytes_mb': {'read': round(elements * 2 / 1e6, 1), 'written': round(elements * 4 / 1e6, 1)},
        'persons': sum(len(p) for p in ref['b_in_place']), 'results_equal': bool(same),
        'calls_per_arm': len(times['a_convert']),
        'seconds_per_arm': {k: round(sum(v) / 1e3, 3) for k, v in times.items()},
        'median_ms': {k: round(float(np.median(v)), 4) for k, v in times.items()},
        'p10_p90_ms': {k: [round(float(np.percentile(v, 10)), 4), round(float(np.percentile(v, 90)), 4)]
                       for k, v in times.items()},
    }


def k2_stage(calls):
    """Median K2 stage time of the default-heads decode of the bench workload (bf16 planar maps)."""
    import numpy as np
    import torch
    import bench
    w = workload()
    post = make_post(w, False)
    hmp, omp = bench.lowres_inputs(4000, w['batch'], w['edge'], True, w)
    omp[~np.isfinite(omp)] = 0
    hv, ov = (torch.from_numpy(a).to(torch.bfloat16).cuda() for a in (hmp, omp))
    eng = post._engine(hv.device)
    eng.enable_stage_timing(True)
    k2 = []
    for i in range(calls + 10):
        post.generate_poses([[[hv], [[]], [[]]], [[ov], [[]], [[]]]], flip_test=True)
        if i >= 10:
            k2.append(eng.last_stage_times_ms()['k2'])
    return {'k2_median_ms': round(float(np.median(k2)), 5),
            'k2_p10_p90_ms': [round(float(np.percentile(k2, 10)), 5), round(float(np.percentile(k2, 90)), 5)],
            'calls': calls}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--seconds', type=float, default=1.0, help='least timed seconds per arm and layout')
    ap.add_argument('--k2-stage', action='store_true')
    ap.add_argument('--tree', default=ROOT, help='repository tree whose package is measured (--k2-stage)')
    ap.add_argument('--calls', type=int, default=200)
    args = ap.parse_args()
    tree = os.path.abspath(args.tree)
    sys.path.insert(0, tree)
    import torch
    assert torch.cuda.is_available(), 'needs a CUDA device'
    import offsetguided_b200
    assert os.path.dirname(os.path.dirname(os.path.abspath(offsetguided_b200.__file__))) == tree
    if args.k2_stage:
        out = dict(card=card(), tree=os.path.basename(tree), **k2_stage(args.calls))
        print(json.dumps(out))
        return
    w = workload()
    post = make_post(w, True)
    arrays = heads_inputs(w)
    separate = tuple(torch.from_numpy(a).to(torch.float16).cuda() for a in arrays)
    channels_last = tuple(t.contiguous(memory_format=torch.channels_last) for t in separate)
    out = {'card': card(), 'torch': torch.__version__,
           'workload': 'bench config 2 (batch 64, flip-test, 160x160 maps) + keypoint-scale and jitter-offset heads',
           'results': [measure(post, separate, 'separate planar', args.seconds),
                       measure(post, channels_last, 'separate channels-last', args.seconds)]}
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
