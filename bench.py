#!/usr/bin/env python
"""Benchmark of the OffsetGuided post-network decoder on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload cfg2|cfg3|cfg4] [--batch B] [--long-edge E] [--dump-outputs DIR]

One "step" decodes ONE GLOBAL BATCH of synthetic network outputs, sharded by image over the N
ranks (strong scaling: ceil(B / N) images per GPU, no collective on the data path).  Default
workload: BASELINE.json configs[1] settings (COCO skeleton, flip-test fusion, x4 bicubic resize
to 640x640, topk 32, thre-hmp 0.04, person-thre 0.04, dist-max 40) at the north-star batch of 64.
`--workload cfg4` is configs[3] (long edge 1024, batch 64), `--workload cfg3` configs[2]
(CrowdPose 14 keypoints, 20 persons per image, topk 64, batch 32).

  value     images/s of the PRODUCT PATH, the same work the reference arm does: device-resident
            network-resolution maps (what evaluate.py holds after model(images)) -> flip fusion
            + x4 resize + NMS + top-K -> limb scoring -> grouping -> poses in host memory,
            through PostProcess.submit / collect (the pipelined form of generate_poses) with
            up to eight batches in flight; max over ranks of the timed region;
  e2e       the same through the reference's own synchronous call
            PostProcess.generate_poses(features, flip_test) with HOST (pinned) maps: H2D copy
            of this rank's shard, decode and the poses' way back are inside the timed region;
  roofline  K1 on MATERIALISED full-resolution maps (SURVEY 8d's definition: N*C*H*W*4 bytes per
            launch over the CUDA-event duration of nms_candidates + select, batch B per GPU)
            against the measured HBM copy peak (MEASURED_PEAKS.json);
  roofline_fused   the product path's own K1f: network-resolution bytes over scan + list + blocks;
  cpu_baseline     the oracle port of the reference decoder on the host cores (N = 1 only).

`--impl reference` times the CPU oracle port alone on the same global batch (rank 0 only).

`--dump-outputs DIR` writes, after the timed steps, the poses the timed path returned for its last
step: one (M_i, C, 6) float32 array per image as DIR/poses_<global image index>.npy.  The inputs are
seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'decoded images/s @640 long-edge'
UNIT = 'images/s'
MIN_LEN = 0.5
L2_BYTES = 126e6
DUMP_BYTES = 64 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=['cfg2', 'cfg3', 'cfg4'])
    ap.add_argument('--batch', type=int, default=0, help='GLOBAL batch per step (0 = the workload default)')
    ap.add_argument('--long-edge', type=int, default=0, help='0 = the workload default')
    ap.add_argument('--no-flip', action='store_true', help='no flip-test inputs')
    ap.add_argument('--cpu-sample', type=int, default=0, help='images of the CPU sample (0 = auto)')
    ap.add_argument('--hot-only', action='store_true',
                    help='run only the HBM-resident full-resolution hot path (for ncu captures; no bench line)')
    ap.add_argument('--lean', action='store_true', help='skip the extra legs (weak scaling, sustained run, baselines)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the poses of the last timed step as DIR/poses_<image>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    return args


def workload(args):
    from offsetguided_b200 import config as cfg
    from oracle import scenes
    if args.workload == 'cfg3':
        w = dict(tag='BASELINE configs[2]: CrowdPose 14 keypoints / 15 limbs, 20 persons per image',
                 keypoints=cfg.CROWDPOSE_KEYPOINTS, skeleton=cfg.CROWDPOSE_PERSON_SKELETON,
                 template=scenes.TEMPLATE_CROWDPOSE, topk=64, persons=20, edge=640, batch=32)
    else:
        w = dict(tag='BASELINE configs[1] settings: COCO 17 keypoints / 19 limbs, 6 persons per image'
                 if args.workload == 'cfg2' else
                 'BASELINE configs[3]: long edge 1024 (256x256 maps), COCO 17 keypoints / 19 limbs, 6 persons per image',
                 keypoints=cfg.COCO_KEYPOINTS, skeleton=cfg.COCO_PERSON_SKELETON,
                 template=scenes.TEMPLATE_COCO, topk=32, persons=6,
                 edge=1024 if args.workload == 'cfg4' else 640, batch=64)
    w.update(thre_hmp=0.04, person_thre=0.04, dist_max=40.0, flip=not args.no_flip)
    if args.batch:
        w['batch'] = args.batch
    if args.long_edge:
        w['edge'] = args.long_edge
    w['c'] = len(w['keypoints'])
    w['l'] = len(w['skeleton'])
    w['kp_flips'] = cfg.heatmap_hflip(w['keypoints'])
    w['limb_flips'], w['limb_reserve'] = cfg.offset_hflip(w['keypoints'], w['skeleton'])
    return w


def workload_config(w, n_gpus, per_gpu):
    e = w['edge']
    return {
        'workload': '%s; network maps %dx%d (x4 -> %dx%d), %s, topk=%d, thre_hmp=%.2f, person_thre=%.2f, '
                    'dist_max=%d' % (w['tag'], e // 4, e // 4, e, e, 'flip-test fusion' if w['flip'] else 'no flip',
                                     w['topk'], w['thre_hmp'], w['person_thre'], int(w['dist_max'])),
        'global_batch': w['batch'],
        'images_per_gpu_per_step': per_gpu,
        'parallelism': 'one global batch image-sharded x%d (ceil(B / N) per GPU), no collective' % n_gpus,
        'l2_policy': 'every step decodes another input buffer of a ring whose total size exceeds 2x the 126 MB L2 '
                     '(network-resolution heat maps: %.0f MB per GPU per step); the full-resolution K1 roofline leg '
                     'streams %.2f GB per launch' % (per_gpu * (2 if w['flip'] else 1) * w['c'] * (e // 4) ** 2 * 4 / 1e6,
                                                     w['batch'] * w['c'] * e * e * 4 / 1e9),
        'persons_per_image': w['persons'],
    }


def dump_outputs(out_dir, poses, first, n_images, w):
    """Write `poses` (the per-image results of images first, first + 1, ... of a batch of `n_images`)
    as out_dir/poses_<image>.npy.  An image has at most L * K persons; when that bound allows more
    than DUMP_BYTES in all, a fixed seeded sample of the images is written, chosen from the arguments
    alone so that every build writes the same files."""
    images = np.arange(n_images)
    cap = DUMP_BYTES // (w['l'] * w['topk'] * w['c'] * 6 * 4)
    if n_images > cap:
        images = np.sort(np.random.RandomState(0).permutation(n_images)[:cap])
    os.makedirs(out_dir, exist_ok=True)
    for g in images:
        if first <= g < first + len(poses):
            np.save(os.path.join(out_dir, 'poses_%05d.npy' % g), np.asarray(poses[g - first], dtype=np.float32))


# --------------------------------------------------------------------------- inputs
def lowres_inputs(seed, n, long_edge, flip, w=None):
    """Network-resolution maps as the reference encoder renders them (oracle/scenes.py
    restates encoder/heatmap.py and encoder/offset.py); flipped half from mirrored persons."""
    from oracle import scenes
    from offsetguided_b200 import config as cfg
    if w is None:
        w = dict(skeleton=cfg.COCO_PERSON_SKELETON, keypoints=cfg.COCO_KEYPOINTS, template=scenes.TEMPLATE_COCO,
                 persons=6, c=17)
    skel = w['skeleton']
    kp = cfg.heatmap_hflip(w['keypoints'])
    c = len(w['keypoints'])
    distinct = min(n, 16)
    hs, os_, hf, of = [], [], [], []
    for i in range(distinct):
        rng = np.random.RandomState(seed + i)
        p = scenes.make_persons(rng, w['persons'], long_edge, long_edge, w['template'],
                                scale_range=(long_edge / 64.0, long_edge / 27.0))
        hs.append(scenes.render_heatmaps(p, long_edge, long_edge) +
                  rng.uniform(0, 0.02, size=(c, long_edge // 4, long_edge // 4)).astype(np.float32))
        os_.append(scenes.render_offsets(p, long_edge, long_edge, skel))
        if flip:
            pf = scenes.mirror_persons(p, long_edge, kp)
            hf.append(scenes.render_heatmaps(pf, long_edge, long_edge) +
                      rng.uniform(0, 0.02, size=(c, long_edge // 4, long_edge // 4)).astype(np.float32))
            of.append(scenes.render_offsets(pf, long_edge, long_edge, skel))
    reps = (n + distinct - 1) // distinct

    def tile(lst):
        return np.concatenate([np.stack(lst)] * reps)[:n]
    hmp = tile(hs)
    omp = tile(os_)
    if flip:
        hmp = np.concatenate((hmp, tile(hf)))
        omp = np.concatenate((omp, tile(of)))
    omp[~np.isfinite(omp)] = 0
    return hmp.astype(np.float32), omp.astype(np.float32)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons of one GPU during the timed region."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None,
                'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------- CPU arm
def cpu_decode_fn(w):
    """The oracle port of the reference decoder: multi-threaded C restatement when it has
    been built (oracle/og_oracle.c), else the numpy restatement (single thread)."""
    kw = dict(topk=w['topk'], thre_hmp=w['thre_hmp'], min_len=MIN_LEN, person_thre=w['person_thre'],
              dist_max=w['dist_max'], use_scale=True, kp_flips=w['kp_flips'], limb_flips=w['limb_flips'],
              limb_reserve=w['limb_reserve'])
    try:
        from oracle import c_oracle
        c_oracle.load()
        cores = c_oracle.num_threads()

        def run(hmp, omp, flip, stage_seconds=None):
            return c_oracle.generate_poses(hmp, omp, w['skeleton'], w['c'], flip_test=flip,
                                           stage_seconds=stage_seconds, **kw)
        return run, cores, 'oracle/og_oracle.c (C + OpenMP restatement of the reference decoder)'
    except Exception:
        from oracle import ref_oracle as ro

        def run(hmp, omp, flip, stage_seconds=None):
            return ro.generate_poses(hmp, omp, w['skeleton'], w['c'], flip_test=flip, **kw)
        return run, 1, 'oracle/ref_oracle.py (numpy restatement of the reference decoder)'


def time_cpu(w, n_images, repeats):
    run, cores, what = cpu_decode_fn(w)
    flip = w['flip']
    hmp, omp = lowres_inputs(9000, n_images, w['edge'], flip, w)
    run(hmp[:1] if not flip else np.concatenate((hmp[:1], hmp[n_images:n_images + 1])),
        omp[:1] if not flip else np.concatenate((omp[:1], omp[n_images:n_images + 1])), flip)   # warm
    times, stage_runs = [], []
    for _ in range(repeats):
        stage = {}
        t0 = time.perf_counter()
        poses = run(hmp, omp, flip, stage)
        times.append(time.perf_counter() - t0)
        stage_runs.append(stage)
        assert len(poses) == n_images
    best = min(times)
    stage_ms = {k: 1e3 * v / n_images for k, v in stage_runs[times.index(best)].items()}
    return n_images / best, cores, what, times, stage_ms


def run_reference(args):
    """The reference arm: the CPU port of the reference decoder with all host threads, one step =
    the whole global batch (the same unit of work as the B200 arm), same warm-up."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    w = workload(args)
    run, cores, what = cpu_decode_fn(w)
    n_images = args.cpu_sample or (w['batch'] if cores > 1 else 1)
    flip = w['flip']
    hmp, omp = lowres_inputs(5000, n_images, w['edge'], flip, w)
    for _ in range(args.warmup):
        run(hmp, omp, flip)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        poses = run(hmp, omp, flip)
    dt = time.perf_counter() - t0
    value = n_images * args.steps / dt
    sample = '%d images per step (the global batch is %d), %d steps after %d warm-up steps, %s' % (
        n_images, w['batch'], args.steps, args.warmup, what)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'config': workload_config(w, args.gpus, -(-w['batch'] // args.gpus)),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, poses, 0, n_images, w)


# --------------------------------------------------------------------------- B200 arm
def make_post(w, batch):
    """PostProcess of the workload: decoder_factory(args) for the COCO heads (the reference's own
    construction path); the CrowdPose table is not reachable through parse_heads (it asserts 17
    keypoints, decoder/factory.py:204), so config 3 builds the same classes directly."""
    from offsetguided_b200 import decoder
    if w['c'] == 17:
        ap = argparse.ArgumentParser()
        decoder.decoder_cli(ap)
        dargs = ap.parse_args(['--topk', str(w['topk']), '--thre-hmp', str(w['thre_hmp']),
                               '--person-thre', str(w['person_thre']), '--dist-max', str(w['dist_max'])])
        dargs.headnets, dargs.strides, dargs.batch_size = ['hmp', 'omp'], [4, 4], batch
        dargs.include_scale = dargs.include_jitter_offset = False
        return decoder.decoder_factory(dargs)
    from offsetguided_b200.decoder.factory import PostProcess
    lc = decoder.LimbsCollect(4, 4, topk=w['topk'], thre_hmp=w['thre_hmp'], min_len=MIN_LEN,
                              keypoints=w['keypoints'], skeleton=w['skeleton'])
    lg = decoder.GreedyGroup(w['person_thre'], sort_dim=2, dist_max=w['dist_max'], use_scale=True,
                             keypoints=w['keypoints'], skeleton=w['skeleton'])
    return PostProcess(batch, 4, 4, 'bicubic', keypoints=w['keypoints'], skeleton=w['skeleton'],
                       limb_collector=lc, limb_grouper=lg)


def pipelined(post, feats_ring, flip, steps, depth, probe=None):
    """`steps` decodes through submit / collect with up to `depth` in flight; every batch's poses
    are collected.  Returns the last result.  `probe` (a dict) receives the median host
    microseconds of a submit and of a collect (diagnostic passes only)."""
    depth = max(1, min(depth, steps))
    nb = len(feats_ring)
    out = None
    for i in range(depth - 1):
        post.submit(feats_ring[i % nb], flip_test=flip)
    if probe is None:
        for i in range(depth - 1, steps):
            post.submit(feats_ring[i % nb], flip_test=flip)
            out = post.collect()
    else:
        ts, tc = [], []
        for i in range(depth - 1, steps):
            a = time.perf_counter()
            post.submit(feats_ring[i % nb], flip_test=flip)
            b = time.perf_counter()
            out = post.collect()
            tc.append(time.perf_counter() - b)
            ts.append(b - a)
        probe['submit_us'] = round(1e6 * statistics.median(ts), 2)
        probe['collect_us'] = round(1e6 * statistics.median(tc), 2)
        probe['collect_us_max'] = round(1e6 * max(tc), 2)
    for _ in range(depth - 1):
        out = post.collect()
    return out


def pin_to_own_core(local, local_world):
    """One physical core per rank (both hardware threads): a step of the sharded batch is ~20 us of
    host work, so two ranks sharing the sibling threads of one core show up in the max over ranks."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        cores = {}
        for cpu in allowed:
            try:
                with open('/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list' % cpu) as f:
                    sib = f.read().strip()
            except OSError:
                sib = str(cpu)
            cores.setdefault(sib, []).append(cpu)
        groups = sorted(cores.values())
        if len(groups) >= 2 * local_world:           # leave the other cores to samplers / NCCL threads
            os.sched_setaffinity(0, set(groups[(2 * local + 1) % len(groups)]))
            return groups[(2 * local + 1) % len(groups)]
    except (AttributeError, OSError):
        pass
    return None


def run_b200(args):
    import torch
    import torch.distributed as dist
    from offsetguided_b200 import _lib, sharding
    from offsetguided_b200.engine import DecoderEngine
    from oracle import scenes

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    # Spread the ranks over the PCIe tree: with fewer ranks than GPUs, neighbouring ordinals share
    # upstream links (profiles/r1_topo_8gpu.txt), so rank r takes GPU r * (G / N).
    ndev = torch.cuda.device_count()
    local_world = int(os.environ.get('LOCAL_WORLD_SIZE', str(world)))
    dev_index = local * (ndev // local_world) if (ndev >= local_world and ndev % local_world == 0) else local
    torch.cuda.set_device(dev_index)
    dev = torch.device('cuda', dev_index)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # This image exports NCCL_DEBUG=VERSION, which makes NCCL print its version banner on
        # STDOUT (also at WARN; probed) — stdout carries the one JSON line only.  Any other explicit
        # setting of the caller (INFO, TRACE) is left alone.
        if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
            os.environ.pop('NCCL_DEBUG')
        dist.init_process_group('nccl', device_id=dev)
    n_gpus = world

    w = workload(args)
    skel, C, L, E, B, flip = w['skeleton'], w['c'], w['l'], w['edge'], w['batch'], w['flip']
    start_i, stop_i = sharding.partition(B, world)[rank]
    n_local = stop_i - start_i
    per_gpu = -(-B // world)
    tables = (w['kp_flips'], w['limb_flips'], w['limb_reserve']) if flip else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    post = make_post(w, per_gpu)
    eng = post._engine(dev)
    torch.set_num_threads(1)

    # ---- ONE global batch, the same on every rank (same seed); this rank decodes its shard
    hmp_np, omp_np = lowres_inputs(5000, B, E, flip, w)
    feats_global = [[[torch.from_numpy(hmp_np)], [[]], [[]]], [[torch.from_numpy(omp_np)], [[]], [[]]]]
    shard = sharding.shard_features(feats_global, rank, world, flip_test=flip)
    hmp_h = shard[0][0][0].contiguous().pin_memory()
    omp_h = shard[1][0][0].contiguous().pin_memory()
    del hmp_np, omp_np, feats_global, shard
    step_bytes = hmp_h.numel() * 4
    ring = 1
    while ring * step_bytes < 2 * L2_BYTES and ring < 16:
        ring *= 2
    feats_ring = []
    for _ in range(ring):
        feats_ring.append([[[hmp_h.to(dev)], [[]], [[]]], [[omp_h.to(dev)], [[]], [[]]]])

    # ---- hot path on HBM-resident full-resolution maps (K1 roofline; B images on every GPU)
    hot_n = B
    distinct = min(hot_n, 8)
    heat_np, offs_np = scenes.synth_hires_batch(1000 * (rank + 1), distinct, w['persons'], E, E, skel, n_channels=C)
    reps = (hot_n + distinct - 1) // distinct
    heat = torch.from_numpy(heat_np).to(dev).repeat(reps, 1, 1, 1)[:hot_n].contiguous()
    offs = torch.from_numpy(offs_np).to(dev).repeat(reps, 1, 1, 1)[:hot_n].contiguous()
    del heat_np, offs_np
    hot_eng = DecoderEngine(C, skel, topk=w['topk'], thre_hmp=w['thre_hmp'], min_len=MIN_LEN,
                            dist_max=w['dist_max'], use_scale=True, person_thre=w['person_thre'], device=dev)
    hot_eng.enable_stage_timing(True)
    for _ in range(max(3, args.warmup)):
        hot_eng.decode_maps(heat, offs)
    hot_eng.decode_maps(heat, offs, fetch=False)           # the timed loop keeps two calls in flight: warm both slots
    hot_eng.decode_maps(heat, offs, fetch=False)
    hot_eng.fetch()
    hot_eng.fetch()
    hot_steps = max(4, min(args.steps, 10))
    torch.cuda.synchronize(dev)
    hot_l0 = hot_eng.launch_count
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    hot_stages = []
    h0.record()
    hot_eng.decode_maps(heat, offs, fetch=False)
    for _ in range(hot_steps - 1):
        hot_eng.decode_maps(heat, offs, fetch=False)
        hot_eng.fetch()
        hot_stages.append(hot_eng.last_stage_times_ms())
    hot_eng.fetch()
    hot_stages.append(hot_eng.last_stage_times_ms())
    h1.record()
    torch.cuda.synchronize(dev)
    hot_ms = h0.elapsed_time(h1) / hot_steps
    hot_launches = hot_eng.launch_count - hot_l0
    if args.hot_only:
        print('hot-only: %.3f ms/step, stages %s' % (hot_ms, hot_stages[-1]), file=sys.stderr)
        return
    del heat, offs
    hot_eng.close()
    torch.cuda.empty_cache()

    # ---- stage times of the product path (kernel by kernel, stage events; graphs are off meanwhile)
    eng.enable_stage_timing(True)
    dev_stages = []
    for i in range(max(3, min(args.warmup, 5)) + 4):
        post.generate_poses(feats_ring[i % ring], flip_test=flip)
        dev_stages.append(eng.last_stage_times_ms())
    dev_stages = dev_stages[-4:]
    eng.enable_stage_timing(False)

    # ---- value: the product path, pipelined, one global batch per step
    depth = _lib.OG_MAX_IN_FLIGHT
    if os.environ.get('OG_BENCH_DEPTH'):                      # tuning aid
        depth = max(1, min(int(os.environ['OG_BENCH_DEPTH']), _lib.OG_MAX_IN_FLIGHT))
    persons = pipelined(post, feats_ring, flip, args.warmup + 2 * depth, depth)      # warm-up: every slot has its graphs
    n_persons = sum(len(p) for p in persons)
    sampler = ClockSampler(dev_index).start()
    pinned_cpus = pin_to_own_core(local, local_world) if world > 1 else None
    host_probe = {}
    pipelined(post, feats_ring, flip, 4 * depth, depth, host_probe)
    barrier()
    l0 = eng.launch_count
    v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    v0.record()
    last_poses = pipelined(post, feats_ring, flip, args.steps, depth)
    v1.record()
    torch.cuda.synchronize(dev)
    value_wall_ms = (time.perf_counter() - t0) * 1e3
    value_ms = v0.elapsed_time(v1)
    barrier()
    value_launches = eng.launch_count - l0
    graph_counts = eng.graph_counts

    # ---- e2e: the reference's synchronous call on pinned HOST maps (this rank's shard)
    feats_host = [[[hmp_h], [[]], [[]]], [[omp_h], [[]], [[]]]]
    eng.enable_stage_timing(True)
    for _ in range(max(3, args.warmup)):
        out = post.generate_poses(feats_host, flip_test=flip)
    e2e_l0 = eng.launch_count
    barrier()
    t0 = time.perf_counter()
    e2e_stages = []
    for _ in range(args.steps):
        out = post.generate_poses(feats_host, flip_test=flip)
        e2e_stages.append(eng.last_stage_times_ms())
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    eng.enable_stage_timing(False)
    e2e_launches = eng.launch_count - e2e_l0
    d2h = sum(p.nbytes for p in out) + (2 * n_local + 2) * 4
    zero_copy = eng.zero_copy_count > 0
    _, det_idx, _ = eng.last_intermediates(n_local)
    per_joint = (det_idx >= 0).sum(dim=2).cpu().numpy()                     # (n_local, C)
    gathered = 0
    for l, (jf, _jt) in enumerate(skel):
        maps = 2 if (flip and l not in w['limb_reserve']) else 1
        gathered += int(per_joint[:, jf].sum()) * 2 * 4 * 4 * maps
    h2d_full = hmp_h.numel() * 4 + omp_h.numel() * 4
    h2d = hmp_h.numel() * 4 + gathered if zero_copy else h2d_full
    # pinned host -> device peak of this rank's link (the e2e roofline denominator), all ranks at once
    probe_h = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    probe_d = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    barrier()
    best = 0.0
    for _ in range(5):
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        probe_d.copy_(probe_h, non_blocking=True)
        p1.record()
        torch.cuda.synchronize(dev)
        best = max(best, probe_h.numel() / (p0.elapsed_time(p1) * 1e-3) / 1e9)
    h2d_peak = best
    del probe_h, probe_d
    clocks = sampler.stop()

    # ---- extras: weak scaling (B images per GPU), a sustained run, the baselines
    weak_block = sustained = sustained_strong = None
    if not args.lean:
        hw_np, ow_np = lowres_inputs(7000 + 100 * rank, B, E, flip, w)
        hw_d, ow_d = torch.from_numpy(hw_np).to(dev), torch.from_numpy(ow_np).to(dev)
        del hw_np, ow_np
        weak_ring = [[[[hw_d], [[]], [[]]], [[ow_d], [[]], [[]]]]]
        if hw_d.numel() * 4 < 2 * L2_BYTES:
            weak_ring.append([[[hw_d.clone()], [[]], [[]]], [[ow_d.clone()], [[]], [[]]]])
        pipelined(post, weak_ring, flip, 3 * depth, depth)
        barrier()
        wk0, wk1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wk0.record()
        pipelined(post, weak_ring, flip, args.steps, depth)
        wk1.record()
        torch.cuda.synchronize(dev)
        weak_ms = wk0.elapsed_time(wk1)
        barrier()
        # sustained: >= 1 s of the product path back to back, clocks sampled meanwhile
        s_sampler = ClockSampler(dev_index).start()
        s_steps = max(args.steps, int(1.2e3 / max(weak_ms / args.steps, 1e-3)))
        t0 = time.perf_counter()
        pipelined(post, weak_ring, flip, s_steps, depth)
        torch.cuda.synchronize(dev)
        s_ms = (time.perf_counter() - t0) * 1e3
        s_clocks = s_sampler.stop()
        weak_t = torch.tensor([weak_ms, s_ms / s_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(weak_t, op=dist.ReduceOp.MAX)
        weak_ms, s_step_ms = [float(v) for v in weak_t.cpu()]
        weak_block = {'value': n_gpus * B * args.steps / (weak_ms * 1e-3), 'unit': UNIT,
                      'ms_per_step': weak_ms / args.steps, 'images_per_gpu_per_step': B,
                      'note': 'the same product path with %d images on EVERY GPU per step (round 1\'s scaling mode)' % B}
        sustained = {'value': n_gpus * B / (s_step_ms * 1e-3), 'unit': UNIT, 'seconds': s_ms * 1e-3,
                     'steps': s_steps, 'ms_per_step': s_step_ms, 'clocks': s_clocks,
                     'note': 'product path, %d images per GPU per step, back to back for >= 1 s' % B}
        del hw_d, ow_d, weak_ring
        if world > 1:
            # the sharded batch in steady state: this rank's shard back to back for >= 0.5 s (the
            # 20-step window of `value` contains the fill and drain of the ~75 us kernel chain)
            ss_steps = max(args.steps, int(0.6e3 / max(value_ms / args.steps, 1e-3)))
            barrier()
            t0 = time.perf_counter()
            pipelined(post, feats_ring, flip, ss_steps, depth)
            torch.cuda.synchronize(dev)
            ss_t = torch.tensor([(time.perf_counter() - t0) * 1e3 / ss_steps], dtype=torch.float64, device=dev)
            dist.all_reduce(ss_t, op=dist.ReduceOp.MAX)
            ss_step_ms = float(ss_t.cpu()[0])
            sustained_strong = {'value': B / (ss_step_ms * 1e-3), 'unit': UNIT, 'steps': ss_steps,
                                'ms_per_step': ss_step_ms, 'images_per_gpu_per_step': per_gpu,
                                'note': 'the sharded global batch (`value`) back to back for >= 0.5 s, max over ranks'}

    eager_block = None
    if rank == 0 and world == 1 and not args.lean and C == 17 and not os.environ.get('OG_BENCH_SKIP_EAGER'):
        try:
            from oracle import torch_eager
            hmp_d, omp_d = feats_ring[0][0][0][0], feats_ring[0][1][0][0]
            eager_kw = dict(topk=w['topk'], thre_hmp=w['thre_hmp'], min_len=MIN_LEN, person_thre=w['person_thre'],
                            dist_max=w['dist_max'], use_scale=True, stride=4, resize_mode='bicubic', flip_test=flip,
                            kp_flips=tables[0] if flip else None, limb_flips=tables[1] if flip else None,
                            limb_reserve=tables[2] if flip else None)
            with torch.no_grad():
                eager_out = torch_eager.generate_poses(hmp_d, omp_d, skel, 17, **eager_kw)      # warm-up
                torch.cuda.synchronize(dev)
                eager_steps = max(2, args.steps // 5)
                t0 = time.perf_counter()
                for _ in range(eager_steps):
                    eager_out = torch_eager.generate_poses(hmp_d, omp_d, skel, 17, **eager_kw)
                torch.cuda.synchronize(dev)
                eager_ms = (time.perf_counter() - t0) * 1e3 / eager_steps
            eager_block = {'value': B / (eager_ms * 1e-3), 'unit': UNIT, 'ms_per_step': eager_ms,
                           'steps': eager_steps, 'persons_per_step': sum(len(p) for p in eager_out),
                           'note': 'stock PyTorch operators on the same GPU, device-resident network-resolution '
                                   'maps (the same work as `value`), grouping on the host cores with the C '
                                   'oracle; one GPU (rank 0), not part of the timed arms'}
            del eager_out
            torch.cuda.empty_cache()
        except Exception as exc:                      # a baseline must never break the bench line
            eager_block = {'unavailable': repr(exc)[:200]}

    # ---- max over ranks
    rank_ms = torch.zeros(world, dtype=torch.float64, device=dev)
    rank_ms[rank] = value_ms / args.steps
    if world > 1:
        dist.all_reduce(rank_ms, op=dist.ReduceOp.SUM)
    rank_ms = [round(float(v), 5) for v in rank_ms.cpu()]
    times = torch.tensor([value_ms, value_wall_ms, e2e_ms, hot_ms], dtype=torch.float64, device=dev)
    sums = torch.tensor([float(value_launches + e2e_launches + hot_launches), float(h2d), float(d2h), float(n_persons),
                         h2d_peak], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    value_ms, value_wall_ms, e2e_ms, hot_ms = [float(v) for v in times.cpu()]
    launches_all, h2d_all, d2h_all, persons_all, h2d_peak_all = [float(v) for v in sums.cpu()]

    if rank == 0:
        def mean_stage(stages):
            return {k: statistics.mean(s[k] for s in stages) for k in stages[0]}
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
        try:
            mp = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
            peak, peak_src = float(mp['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
        hot_stage = mean_stage(hot_stages)
        k1_ms = hot_stage['k1_stream'] + hot_stage['k1_select']
        alg_bytes = hot_n * C * E * E * 4 + hot_n * C * w['topk'] * 8
        achieved = alg_bytes / (k1_ms * 1e-3) / 1e9
        traffic = None
        if args.workload == 'cfg2' and B == 64 and E == 640:
            try:
                traffic = json.load(open(os.path.join(ROOT, 'profiles', 'k1_traffic.json')))['dram_bytes_per_launch']
            except Exception:
                pass
        dev_stage = mean_stage(dev_stages)
        fused_bytes = hmp_h.numel() * 4
        fused_gbs = fused_bytes / (dev_stage['k1_stream'] * 1e-3) / 1e9
        e2e_step_ms = e2e_ms / args.steps
        cpu_block = None          # timed on rank 0 at N = 1 only (bench contract)
        if n_gpus == 1 and not args.lean:
            run, cores, what = cpu_decode_fn(w)
            cpu_n = args.cpu_sample or (16 if cores > 1 else 1)
            cpu_value, cores, what, cpu_times, cpu_stage = time_cpu(w, cpu_n, 2 if cores > 1 else 1)
            cpu_block = {'value': cpu_value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d images of the same workload (flip fusion + x4 resize + NMS/top-K '
                                   '+ limbs + grouping), best of %d, %s' % (cpu_n, len(cpu_times), what),
                         'stage_ms_per_image': cpu_stage,
                         # second baseline of the same leg: the path with stock PyTorch operators on this GPU
                         'eager_torch_gpu': eager_block}
        line = {
            'metric': METRIC, 'value': B * args.steps / (value_ms * 1e-3), 'unit': UNIT,
            'n_gpus': n_gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': value_ms / args.steps, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(w, n_gpus, per_gpu),
            'value_detail': {
                'api': 'decoder_factory(args) -> PostProcess.submit(features, flip_test=%s) / collect(): the pipelined '
                       'form of generate_poses, device-resident network-resolution maps -> poses in host memory' % flip,
                'calls_in_flight': depth, 'input_buffers_in_rotation': ring,
                'wall_ms_per_step': value_wall_ms / args.steps,
                'ms_per_step_of_every_rank': rank_ms,
                'host_cores_of_rank0': pinned_cpus, 'host_call_us_rank0': host_probe,
                'graph_replays_and_captures': list(graph_counts),
                'persons_per_step': persons_all,
                'stage_ms': dev_stage,
                'stage_note': 'per-call device times of one rank\'s shard, taken kernel by kernel with stage events '
                              'in a separate pass (the timed loop replays CUDA graphs)'},
            'e2e': {'value': B * args.steps / (e2e_ms * 1e-3), 'unit': UNIT,
                    'h2d_bytes_per_step': int(h2d_all), 'd2h_bytes_per_step': int(d2h_all),
                    'ms_per_step': e2e_step_ms,
                    'stage_ms': mean_stage(e2e_stages),
                    'fused_redos': eng.fused_redo_count,
                    'api': 'decoder_factory(args).generate_poses(features, flip_test=%s) (synchronous), pinned host '
                           'maps of this rank\'s shard' % flip,
                    'roofline': {'bound': 'pcie', 'achieved': h2d_all / (e2e_step_ms * 1e-3) / 1e9,
                                 'peak': h2d_peak_all, 'unit': 'GB/s',
                                 'frac': h2d_all / (e2e_step_ms * 1e-3) / 1e9 / h2d_peak_all,
                                 'peak_source': 'sum over ranks of a 256 MB pinned host -> device copy, best of 5, '
                                                'all ranks copying at once'},
                    'h2d_detail': {'heat_maps_copied': int(h2d_all) - (gathered if zero_copy else 0) if n_gpus == 1 else None,
                                   'offset_samples_read_over_pcie_rank0': gathered if zero_copy else 0,
                                   'offset_maps_left_on_host_rank0': omp_h.numel() * 4 if zero_copy else 0,
                                   'note': 'fused path: K2 needs 2*L*K bilinear samples per image, so pinned '
                                           'offset maps are read in place (zero-copy) instead of copied'}},
            'gpu_launches': int(launches_all),
            'gpu_launches_detail': {'note': 'kernels of this library launched inside the three timed regions, all ranks; '
                                            'a graph replay counts its 6 kernel nodes',
                                    'value_rank0': value_launches, 'e2e_rank0': e2e_launches,
                                    'k1_roofline_leg_rank0': hot_launches},
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                         'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                         'kernel': 'K1 = nms_candidates_kernel + select_topk_kernel on materialised %dx%d maps, '
                                   '%d images per launch (SURVEY 8d definition)' % (E, E, hot_n),
                         'algorithmic_bytes_per_launch': alg_bytes, 'ms_per_launch': k1_ms,
                         'stream_pass_only_gbs': alg_bytes / (hot_stage['k1_stream'] * 1e-3) / 1e9,
                         'hot_path_ms_per_step': hot_ms, 'hot_path_stage_ms': hot_stage,
                         'hot_path_images_per_s_per_gpu': hot_n / (hot_ms * 1e-3)},
            'roofline_fused': {'bound': 'hbm', 'achieved': fused_gbs, 'peak': peak, 'unit': 'GB/s',
                               'frac': fused_gbs / peak, 'kernel': 'K1f = amax_scan + block_list + fused_block '
                               '(flip fusion + x4 resize + NMS over network-resolution maps), one rank\'s shard',
                               'algorithmic_bytes_per_launch': fused_bytes, 'ms_per_launch': dev_stage['k1_stream']},
            'weak_scaling': weak_block,
            'sustained': sustained,
            'sustained_strong': sustained_strong,
            'cpu_baseline': cpu_block,
            'clocks': clocks,
        }
        print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_poses, start_i, B, w)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
