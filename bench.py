#!/usr/bin/env python
"""Benchmark of the detection hot path (BASELINE.json metric: images/sec).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload frcnn_r50|frcnn_r101|ssd] [--impl ours|reference]
                  [--dump-outputs DIR]

A "step" = one pass of the forward hot path over one batch of synthetic images
(N=1 workload: BASELINE.json configs[1] -- Faster R-CNN ResNet-50, COCO config,
batch 8 of 600x1024).  N>1: one process per GPU under torchrun, per-GPU batch
fixed (weak scaling, BASELINE configs[4]); rank 0 broadcasts the weights over
NCCL once, every step all-gathers the padded detection records.

`value`  : images/s with the input batch resident in HBM (device timed, CUDA events
           on the engine's stream, max over ranks).
`e2e`    : the same through the public host-buffer call (pinned host images ->
           H2D -> forward -> D2H of boxes/scores/labels/counts inside the timed region).
`--impl reference`: the CPU oracle port of the reference forward (the original needs
           TensorFlow 1) on all host cores, one image of the batch per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    'frcnn_r50': dict(model='fasterrcnn', batch=8, h=600, w=1024,
                      overrides=['model.base_network.architecture=resnet_v1_50', 'model.network.num_classes=80'],
                      name='Faster R-CNN ResNet-50 (reference COCO config: 80 classes, post_nms_top_n 2000), '
                           'batch 8 x 600x1024x3 synthetic uint8'),
    'frcnn_r101': dict(model='fasterrcnn', batch=8, h=600, w=1024,
                       overrides=['model.base_network.architecture=resnet_v1_101', 'model.network.num_classes=80',
                                  'model.rpn.proposals.post_nms_top_n=300', 'model.rcnn.proposals.min_prob_threshold=0.0'],
                       name='Faster R-CNN ResNet-101, 300 proposals/img, 80 classes (NMS stress), batch 8 x 600x1024x3'),
    'ssd': dict(model='ssd', batch=32, h=300, w=300, overrides=[],
                name='SSD VGG-16 300x300 (VOC config, 20 classes), batch 32 synthetic uint8'),
    # contract self-test only (tests/test_bench_contract.py): seconds on a CPU, not a benchmark
    'tiny': dict(model='fasterrcnn', batch=2, h=96, w=128,
                 overrides=['model.base_network.architecture=resnet_v1_50', 'model.network.num_classes=5',
                            'model.rpn.proposals.post_nms_top_n=50'],
                 name='contract self-test: Faster R-CNN ResNet-50, 5 classes, batch 2 x 96x128'),
}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('hbm_gbs', 6650.0), d.get('bf16_tflops_sustained', 1400.0), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 1400.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(',')])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm = [float(s[0]) for s in self.samples if len(s) >= 6 and s[0].replace('.', '').isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 6 and s[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(s) >= 6 and s[2 + i].lower().startswith('active') for s in self.samples)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


def conv_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of the conv_tc launches of one step.  ncu cannot run inside a
    timed bench, so the figure comes from the committed `ncu --set full` capture of `bench.py --ncu-range`
    (scripts/gpu_evidence.sh -> scripts/ncu_step_summary.py) and is stamped with the commit and date of that capture,
    so a stale profile is visible as stale; None if this workload was never captured."""
    here = os.path.dirname(os.path.abspath(__file__))
    for name in ('r2_ncu_step_summary.json', 'r1_ncu_step_summary.json'):
        try:
            j = json.load(open(os.path.join(here, 'profiles', name)))
            d = j[workload]['conv_tc_kernel']
            stamp = j.get('_capture', {})
            return d['dram_bytes'], ('sum of dram__bytes_read+write over the %d conv_tc launches of one step '
                                     '(profiles/%s, captured at commit %s on %s)'
                                     % (d['launches'], name, stamp.get('commit', 'round-1 final'), stamp.get('date', '2026-09-22')))
        except Exception:
            continue
    return None, 'not captured'


def write_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per output, floats as float32, integers as float64 (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + '.npy'), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def build_config(wl):
    from luminoth_b200 import default_config
    return default_config(wl['model'], wl['overrides'])


def best_thread_count(cfg, wts, wl):
    """The oracle's convolutions run on torch's CPU thread pool; more threads is not always faster (128 threads on
    the GPU box measured 2x SLOWER than torchrun's OMP_NUM_THREADS=1 default).  Give the CPU arm its best setting:
    time one small forward per candidate and keep the fastest."""
    import torch
    from luminoth_b200 import synth
    from oracle import predict as opredict
    ncpu = os.cpu_count() or 1
    cands = sorted({max(1, c) for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8, 1) if c <= ncpu}, reverse=True)
    h, w = (wl['h'], wl['w']) if wl['model'] == 'ssd' else (wl['h'] // 2, wl['w'] // 2)
    img = synth.make_images(1, h, w, seed=7)[0]
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        opredict.network_outputs(img, wts, cfg)
        t0 = time.perf_counter()
        opredict.network_outputs(img, wts, cfg)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_oracle_images_per_s(cfg, wts, wl, n_images, threads):
    """The CPU restatement of the reference forward (oracle/), timed one image at a time."""
    import torch
    from luminoth_b200 import synth
    from oracle import predict as opredict
    torch.set_num_threads(threads)
    imgs = synth.make_images(n_images + 1, wl['h'], wl['w'], seed=123)
    opredict.network_outputs(imgs[0], wts, cfg)                 # warm-up
    t0 = time.perf_counter()
    for i in range(n_images):
        opredict.network_outputs(imgs[1 + i], wts, cfg)
    dt = time.perf_counter() - t0
    return n_images / dt, dt


def run_reference(args, wl):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from luminoth_b200 import synth
    from oracle import predict as opredict
    cfg = build_config(wl)
    wts = synth.make_weights(cfg, seed=0, profile='peaky')
    threads = best_thread_count(cfg, wts, wl)
    imgs = synth.make_images(max(1, min(args.steps + args.warmup, 4)), wl['h'], wl['w'], seed=123)
    budget_s = 240.0
    t_start = time.perf_counter()
    for i in range(args.warmup):
        opredict.network_outputs(imgs[i % len(imgs)], wts, cfg)
        if time.perf_counter() - t_start > budget_s / 3:
            break
    t0 = time.perf_counter()
    for i in range(args.steps):
        objects, labels, probs, _ = opredict.network_outputs(imgs[i % len(imgs)], wts, cfg)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    if args.dump_outputs:       # the engine's layout: a batch of one image, detections in the first counts[0] rows
        write_outputs(args.dump_outputs, {'boxes': objects[None], 'scores': probs[None], 'labels': labels[None],
                                          'counts': np.array([len(probs)])})
    line = {'impl': 'reference', 'metric': 'images/sec', 'value': v, 'unit': 'images/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * dt / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'sample': '1 image of the batch per step'},
            'cpu_baseline': {'value': v, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
                             'sample': '%d images, one per step (oracle port of the reference forward; TF1 not '
                                       'installable); thread count picked as the fastest of a calibration sweep up to '
                                       '%d host threads' % (args.steps, os.cpu_count() or 1)},
            'e2e': {'value': v, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    from luminoth_b200 import synth
    from luminoth_b200.engine import Engine

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # rank 0 prints ONE JSON line on stdout: NCCL's version banner (printed at NCCL_DEBUG=VERSION *and* WARN) and any
        # other NCCL log line go to stderr
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    cfg = build_config(wl)
    B, H, W = (args.per_gpu_batch or wl['batch']), wl['h'], wl['w']

    # ---- weights: rank 0 owns them, NCCL broadcast to the other GPUs (once, outside the step)
    eng = Engine(cfg, device=local, max_batch=B, max_h=H, max_w=W)
    from luminoth_b200 import parallel as P
    specs = eng.weight_specs()
    wts = synth.make_weights(cfg, seed=0, profile='peaky') if rank == 0 else None
    bcast_ms = 0.0
    if world > 1:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        wts = P.broadcast_weights(wts, specs, dev, src=0)
        torch.cuda.synchronize()
        bcast_ms = (time.perf_counter() - t0) * 1e3
    eng.load_weights(wts).finalize()

    # ---- inputs: NROT distinct batches (rotated so the input is never L2-hot), device + pinned host copies
    NROT = 12 if wl['model'] == 'fasterrcnn' else 16
    imgs_host = [torch.from_numpy(synth.make_images(B, H, W, seed=1000 * rank + i)).pin_memory() for i in range(NROT)]
    imgs_dev = [t.to(dev) for t in imgs_host]
    K = eng.max_detections
    boxes = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((B, K), dtype=torch.float32, device=dev)
    labels = torch.empty((B, K), dtype=torch.int32, device=dev)
    counts = torch.empty((B,), dtype=torch.int32, device=dev)
    rec = torch.empty((B, 1 + 6 * K), dtype=torch.float32, device=dev)
    gathered = torch.empty((world * B, 1 + 6 * K), dtype=torch.float32, device=dev) if world > 1 else None
    # host-side (pinned) outputs for the end-to-end path
    hb = torch.empty((B, K, 4), dtype=torch.float32).pin_memory()
    hs = torch.empty((B, K), dtype=torch.float32).pin_memory()
    hl = torch.empty((B, K), dtype=torch.int32).pin_memory()
    hc = torch.empty((B,), dtype=torch.int32).pin_memory()
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)

    import ctypes
    lib = eng._lib

    if world > 1:
        # the detection kernel itself writes the packed {count, boxes, scores, labels} row of every image into `rec`
        # (lumi_set_record_output): the only multi-GPU work on the step path is ONE ncclAllGather
        eng.set_record_output(rec)

    def step_device(i):
        eng.predict_device(imgs_dev[i % NROT], boxes, scores, labels, counts)
        if world > 1:           # detections all-gather (fixed-size padded record per image), on the engine's stream
            with torch.cuda.stream(stream):
                P.all_gather_detections(rec, out=gathered)

    def step_host(i):
        x = imgs_host[i % NROT]
        rc = lib.lumi_predict(eng._h, ctypes.c_void_p(x.data_ptr()), 0, B, H, W, ctypes.c_void_p(hb.data_ptr()),
                              ctypes.c_void_p(hs.data_ptr()), ctypes.c_void_p(hl.data_ptr()),
                              ctypes.c_void_p(hc.data_ptr()), 0)
        if rc != 0:
            raise RuntimeError(lib.lumi_last_error(eng._h).decode())
        if world > 1:           # `rec` was written on the device by the same call
            with torch.cuda.stream(stream):
                P.all_gather_detections(rec, out=gathered)
            stream.synchronize()

    def timed(step_fn, steps, warmup):
        for i in range(warmup):
            step_fn(i)
        eng.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            step_fn(warmup + i)
        e1.record(stream)
        eng.synchronize()
        torch.cuda.synchronize()
        local_ms = e0.elapsed_time(e1)
        ms = torch.tensor([local_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        torch.cuda.synchronize()
        timed.local_ms = local_ms              # this rank's own time (the returned value is the max over ranks)
        return float(ms.item())

    if args.ncu_range:
        # evidence mode for `ncu --profile-from-start off`: warm up, then expose exactly ONE step to the profiler.
        # --ncu-unpiped: single stream, whole batch per launch -- the configuration of the per-category event
        # profile that `roofline.achieved` comes from (ncu serialises kernels anyway)
        if args.ncu_unpiped:
            eng.set_pipeline(False)
        for i in range(args.warmup):
            step_device(i)
        eng.synchronize()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_device(args.warmup)
        eng.synchronize()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        del imgs_dev, imgs_host, boxes, scores, labels, counts, rec, gathered, hb, hs, hl, hc, stream
        torch.cuda.synchronize()
        eng.close()
        return

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    ms_dev = timed(step_device, args.steps, args.warmup)
    ms_dev_local = timed.local_ms
    launches = eng.last_launch_count
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:     # the last timed step's results, before later passes overwrite them
        dump = {k: t.cpu().numpy() for k, t in
                (('boxes', boxes), ('scores', scores), ('labels', labels), ('counts', counts))}
        for i, k in enumerate(dump['counts']):      # rows past an image's count carry no detection
            dump['boxes'][i, k:] = 0
            dump['scores'][i, k:] = 0
            dump['labels'][i, k:] = 0
        write_outputs(args.dump_outputs, dump)
    ms_e2e = timed(step_host, args.steps, max(3, args.warmup))

    # ---- per-kernel-category device time (events around our own kernels) for the roofline
    eng.profile(True)
    eng.profile_read()
    for i in range(args.steps):
        eng.predict_device(imgs_dev[i % NROT], boxes, scores, labels, counts)
    prof = eng.profile_read()
    layer_prof = eng.profile_read_layers()
    eng.profile(False)

    # every rank reports its own step time and per-category kernel time (a slow rank, or one whose conv kernels slow
    # down under a shared power / clock domain, must be visible -- VERDICT r1 item 5)
    per_rank = None
    if world > 1:
        mine = {'rank': rank, 'ms_per_step': ms_dev_local / args.steps,
                'category_ms_per_step': {k: v_[1] / args.steps for k, v_ in prof.items() if v_[1] > 0}}
        try:
            import pynvml
            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByIndex(local)
            mine['sm_mhz_now'] = pynvml.nvmlDeviceGetClockInfo(hnd, pynvml.NVML_CLOCK_SM)
            mine['power_w_now'] = pynvml.nvmlDeviceGetPowerUsage(hnd) / 1000.0
        except Exception:
            pass
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    if rank == 0:
        hbm, tf, src = peaks()
        total_imgs = B * world
        v = total_imgs * args.steps / (ms_dev / 1e3)
        e2e_v = total_imgs * args.steps / (ms_e2e / 1e3)
        cat_ms = {k: v_[1] / args.steps for k, v_ in prof.items()}
        tc_spans, tc_ms, tc_flops = prof['conv_tc']
        roof = None
        if tc_ms > 0:
            ach = tc_flops / (tc_ms * 1e-3) / 1e12
            roof = {'kernel': 'conv_tc_kernel (tcgen05 implicit-GEMM conv, all instances of one step)',
                    'bound': 'tensor', 'achieved': ach, 'peak': tf, 'unit': 'TFLOP/s', 'frac': ach / tf,
                    'peak_source': src + ', bf16 sustained', 'traffic': conv_traffic(args.workload)[0],
                    'traffic_note': conv_traffic(args.workload)[1],
                    'launches_per_step': tc_spans / args.steps,
                    'algorithmic_gflop_per_step': tc_flops / args.steps / 1e9,
                    'ms_per_step': tc_ms / args.steps,
                    'note': 'fp32-class accuracy is bought with 3 kind::f16 MMAs per algorithmic MAC '
                            '(fp16x2 operand split): the tensor pipe does 3x the algorithmic FLOPs, so frac <= 1/3'}
            for cat, key, note in (('roi_pool', 'roi_pool_hbm', 'ROI crop+max-pool(+mean) kernel; gather is L1/issue-bound, not HBM-bound'),
                                   ('rpn_proposals', 'rpn_nms_hbm', 'RPN decode+sort+bitmask NMS chain (bitmask-algorithm bytes)')):
                rs, rms, rbytes = prof.get(cat, (0, 0.0, 0.0))
                if rms > 0 and rbytes > 0:
                    roof[key] = {'achieved_GBs': rbytes / (rms * 1e-3) / 1e9, 'peak_GBs': hbm,
                                 'frac': rbytes / (rms * 1e-3) / 1e9 / hbm, 'ms_per_step': rms / args.steps,
                                 'algorithmic_MB_per_step': rbytes / args.steps / 1e6, 'note': note}
        out = {
            'metric': 'images/sec', 'value': v, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32 (fp16x2-split operands on tcgen05 kind::f16, fp32 accumulate)',
            'data': 'synthetic',
            'config': {'workload': wl['name'] + (' [batch overridden to %d]' % B if args.per_gpu_batch else ''),
                       'global_batch': total_imgs, 'per_gpu_batch': B,
                       'parallelism': 'dp%d (images sharded, NCCL weight broadcast + detection all-gather)' % world,
                       'l2': 'inputs rotate over %d distinct batches (%.0f MB > 126 MB L2); per-step activation '
                             'working set is several GB' % (NROT, NROT * B * H * W * 3 / 1e6),
                       'weights': 'random-init (synthetic, seed 0, "peaky" profile)'},
            'e2e': {'value': e2e_v, 'unit': 'images/s', 'h2d_bytes_per_step': B * H * W * 3,
                    'd2h_bytes_per_step': B * K * 24 + B * 4, 'ms_per_step': ms_e2e / args.steps},
            'gpu_launches': launches * args.steps,
            'clocks': clocks,
            'category_ms_per_step': cat_ms,
            'per_rank': per_rank,
            'weight_bcast_ms': bcast_ms,
            'roofline': roof,
        }
        if args.layers:      # per-conv-layer live timing (events around each launch, single stream, whole batch)
            out['conv_layers'] = [{'layer': n, 'us': ms_ * 1e3 / c, 'gflop': w_ / c / 1e9,
                                   'tflops': (w_ / c) / (ms_ / c * 1e-3) / 1e12 if ms_ > 0 else None}
                                  for n, c, ms_, w_ in layer_prof]
        if world == 1 and not args.no_cpu_baseline:
            if wts is None:
                wts = synth.make_weights(cfg, seed=0, profile='peaky')
            threads = best_thread_count(cfg, wts, wl)
            n_cpu = 2 if wl['model'] == 'fasterrcnn' else 8
            cv, cdt = cpu_oracle_images_per_s(cfg, wts, wl, n_cpu, threads)
            out['cpu_baseline'] = {'value': cv, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
                                   'sample': '%d images of the same workload, one at a time, %.1f s (oracle port of the '
                                             'reference forward; TF1 not installable; thread count = fastest of a sweep up '
                                             'to %d host threads)' % (n_cpu, cdt, os.cpu_count() or 1)}
        print(json.dumps(out), flush=True)
    # teardown order matters: tensors that lived on the engine's (external) stream must be released, and the
    # process group torn down, BEFORE the engine destroys that stream
    eng.synchronize()
    del imgs_dev, imgs_host, boxes, scores, labels, counts, rec, gathered, hb, hs, hl, hc, stream
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='frcnn_r50', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--per-gpu-batch', type=int, default=0,
                    help='override the workload batch (latency studies; the headline number uses the default)')
    ap.add_argument('--layers', action='store_true', help='add a per-conv-layer timing table to the JSON line')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step (boxes, scores, labels, counts) as DIR/<name>.npy; '
                         'the inputs depend only on the arguments, so two builds can be compared output for output')
    ap.add_argument('--ncu-unpiped', action='store_true', help='with --ncu-range: single-stream forward')
    ap.add_argument('--ncu-range', action='store_true',
                    help='run warm-up, then one step inside cudaProfilerStart/Stop (for ncu --profile-from-start off)')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == 'reference':
        run_reference(args, wl)
    else:
        from luminoth_b200.engine import load_library
        load_library()          # fail loudly if the CUDA library is missing
        run_ours(args, wl)
        # normal interpreter exit: the library shares torch's CUDA runtime (-cudart shared, luminoth_b200/build.py),
        # every engine / tensor / process group was released above, so atexit hooks (and the driver's) run


if __name__ == '__main__':
    main()
