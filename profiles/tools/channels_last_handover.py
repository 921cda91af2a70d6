"""Hand-over of a channels-last head output to the decoder: (a) `.contiguous()` of the NHWC heat and
offset slices, then generate_poses (what a caller had to do before channels-last maps were read in
place), against (b) generate_poses on the NHWC slices themselves.  One packed bf16
[2N, 55, h, w] channels_last buffer per shape, flip-test; each call is timed with CUDA events
around the synchronous generate_poses (which ends with the fetch), the two variants alternating
after a warm-up; the medians per call are reported with the card's name and power limit.

    python profiles/tools/channels_last_handover.py [rounds] > out.json
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np      # noqa: E402
import torch            # noqa: E402
import bench            # noqa: E402

SHAPES = (('cfg2 (bench shape)', 'cfg2'), ('cfg4', 'cfg4'))


class _Args(object):
    no_flip = False
    batch = 0
    long_edge = 0

    def __init__(self, workload):
        self.workload = workload


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ', power limit not read'


def measure(label, workload, rounds, warmup=5):
    w = bench.workload(_Args(workload))
    n, edge = w['batch'], w['edge']
    post = bench.make_post(w, n)
    hmp, omp = bench.lowres_inputs(4000, n, edge, True, w)
    buf = torch.cat((torch.from_numpy(hmp), torch.from_numpy(omp)), dim=1).to(torch.bfloat16).cuda()
    buf = buf.contiguous(memory_format=torch.channels_last)
    c = w['c']

    def copied():
        return post.generate_poses([[[buf[:, :c].contiguous()], [[]], [[]]], [[buf[:, c:].contiguous()], [[]], [[]]]],
                                   flip_test=True)

    def in_place():
        return post.generate_poses([[[buf[:, :c]], [[]], [[]]], [[buf[:, c:]], [[]], [[]]]], flip_test=True)

    variants = (('a_contiguous_copy', copied), ('b_in_place', in_place))
    ref = {name: fn() for name, fn in variants}
    same = all(np.array_equal(x, y) for x, y in zip(ref['a_contiguous_copy'], ref['b_in_place']))
    for _ in range(warmup):
        for _, fn in variants:
            fn()
    times = {name: [] for name, _ in variants}
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for name, fn in variants:
            torch.cuda.synchronize()
            start.record()
            fn()
            end.record()
            end.synchronize()
            times[name].append(start.elapsed_time(end))
    heat_mb = buf.shape[0] * c * buf.shape[2] * buf.shape[3] * 2 / 1e6
    return {
        'shape': label, 'buffer': list(buf.shape), 'dtype': 'bf16', 'flip_test': True,
        'buffer_mb': round(buf.numel() * 2 / 1e6, 1), 'heat_slice_mb': round(heat_mb, 1),
        'persons': sum(len(p) for p in ref['b_in_place']), 'results_equal': bool(same), 'rounds': rounds,
        'median_ms': {k: round(float(np.median(v)), 4) for k, v in times.items()},
        'p10_p90_ms': {k: [round(float(np.percentile(v, 10)), 4), round(float(np.percentile(v, 90)), 4)]
                       for k, v in times.items()},
    }


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 30
    assert torch.cuda.is_available(), 'needs a CUDA device'
    out = {'card': card(), 'torch': torch.__version__, 'results': [measure(l, wl, rounds) for l, wl in SHAPES]}
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
