#!/usr/bin/env python
"""Benchmark of the SipMask inference hot path (BASELINE.json metric: images/sec @ 800x1333, bs=1/GPU).

    python bench.py --gpus N --steps K --warmup W                      # this repo's sm_100a path, workload A (config 2)
    python bench.py --workload A101 | B                                 # R101 (config 3) | 544x544 bs=32 (config 4)
    python bench.py --impl reference --gpus N --steps K --warmup W      # the reference's CPU forward (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR             # + the last timed step's outputs as DIR/*.npy

One "step" = one pass of the whole hot path (image -> backbone/FPN -> head -> decode/NMS -> mask assembly ->
bit-packed masks) over one synthetic image per GPU (workload B: one 32-image batch per GPU).  Prints ONE JSON line (rank 0).
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

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration `metric` is quoted on
    'A': dict(name='SipMask R50-FPN-GN 4conv, 800x1333 (padded 800x1344), bs=1/GPU, synthetic image + seeded synthetic weights',
              depth=50, stacked=4, gn=True, ssd=False, H=800, W=1344, img_w=1333, batch=1, score_thr=0.05, in_flight=6),
    # configs[2]: R101 backbone, one image per GPU
    'A101': dict(name='SipMask R101-FPN-GN 4conv, 800x1333 (padded 800x1344), bs=1/GPU, synthetic image + seeded synthetic weights',
                 depth=101, stacked=4, gn=True, ssd=False, H=800, W=1344, img_w=1333, batch=1, score_thr=0.05, in_flight=6),
    # configs[3]: real-time SSD-style head (2 convs, no GN, fast_nms), 544x544, bs=32 per forward (throughput mode)
    'B': dict(name='SipMask R50-FPN SSD-style head (2conv, no GN, fast_nms), 544x544, bs=32 per forward, synthetic images + '
                   'seeded synthetic weights', depth=50, stacked=2, gn=False, ssd=True, H=544, W=544, img_w=544, batch=32,
              score_thr=0.1, in_flight=1),
    # configs[4]: SipMask-VIS frame path (3-conv towers, 40 classes, tracking branch, fast_nms max 10), 360x640 padded to
    # 384x640; frames are sharded one per GPU per step, records + 512-d track features are gathered once at the end and the
    # tracker association runs on the host in frame order (inside the timed region)
    'C': dict(name='SipMask-VIS R50-FPN-GN 3conv + track branch, 360x640 (padded 384x640), one frame per GPU per step, '
                   'synthetic frames + seeded synthetic weights', depth=50, stacked=3, gn=True, ssd=False, vis=True, H=384, W=640,
              img_w=640, img_h=360, batch=1, score_thr=0.03, in_flight=6, nms_pre=200, max_per_img=10, num_classes=41),
}
CLS_BIAS = -5.0
ROLL = 500          # untimed pre/post-roll steps around the timed region while nvidia-smi samples clocks


def test_cfg(wl):
    return dict(nms_pre=wl.get('nms_pre', 1000), score_thr=wl['score_thr'], nms=dict(type='nms', iou_thr=0.5),
                max_per_img=wl.get('max_per_img', 100))


# workload A's constants under their round-1 names (tools/*.py import them)
H, W, IMG_W = WORKLOADS['A']['H'], WORKLOADS['A']['W'], WORKLOADS['A']['img_w']
TEST_CFG = test_cfg(WORKLOADS['A'])


def state_dict_for(wl):
    from sipmask_b200 import synth
    if wl.get('vis'):
        sd = {}
        sd.update(synth.backbone_state_dict(wl['depth'], 1))
        sd.update(synth.neck_state_dict(2))
        sd.update(synth.head_state_dict(3, num_classes=wl['num_classes'], stacked_convs=wl['stacked'], gn=True, cls_bias=CLS_BIAS,
                                        track=True))
        return sd
    return synth.detector_state_dict(wl['depth'], stacked_convs=wl['stacked'], gn=wl['gn'], seed=1, cls_bias=CLS_BIAS)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured'
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0), 'fallback'


def ncu_traffic():
    """Per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the roofline kernels, read from the committed
    ncu --set full summary of this round (profiles/r02_ncu_traffic.json; bench.py itself never runs under a profiler)."""
    try:
        return json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')))
    except Exception:
        return {}


def host_threads():
    """Threads the CPU arm may really use: CPU affinity capped by the cgroup CPU quota (os.cpu_count() is the machine's
    core count, 128 on the B200 hosts, of which a container usually owns a fraction - r1's CPU numbers moved 66x between
    boxes because 128 threads were started on a few cores)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if q != 'max':
            quota = float(q) / float(p)
    except Exception:
        try:
            q = float(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            p = float(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    n = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-6)) or 1))
    return n, dict(cpu_count=os.cpu_count(), affinity=aff, cgroup_quota=quota, used=n)


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md 'clocks line')."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index),
                 '--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
                 'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
                 'clocks_event_reasons.sw_power_cap', '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ----------------------------------------------------------------------------------------------- CPU reference arm
def build_oracle(wl, threads):
    import torch
    from oracle import model as M
    from oracle import ops as O
    from sipmask_b200 import synth
    torch.set_num_threads(threads)
    O.USE_TORCHVISION_DCN = True
    O.USE_C_CROP_SPLIT = True
    net = M.SipMaskDetector(wl['depth'], stacked_convs=wl['stacked'], gn=wl['gn'], ssd_flag=wl['ssd'])
    if wl.get('vis'):
        net.bbox_head = M.SipMaskVISHead(num_classes=wl['num_classes'], stacked_convs=wl['stacked'])
    net.load_state_dict(state_dict_for(wl), strict=True)
    net.eval()
    return net


def oracle_step(net, img, wl):
    """The reference's forward on host cores: backbone -> FPN -> head -> get_bboxes (decode, per-class NMS with the
    compiled C oracle, dense 4x matmul/sigmoid/stack/CropSplit mask assembly, x2 upsample + threshold), ONE image."""
    import numpy as np
    import torch
    from oracle import cbind, postproc as P
    from oracle import ops as O
    if wl.get('vis'):
        with torch.no_grad():
            outs = net.bbox_head(net.extract_feat(img))
        shape = (wl['img_h'], wl['img_w'], 3)
        meta = dict(img_shape=shape, ori_shape=shape, scale_factor=1.0, is_first=False)
        det, lab, masks, ids = P.vis_get_bboxes(outs, meta, test_cfg(wl), oracle_step.tracker, rescale=True)
        return dict(det_bboxes=det)
    t0 = time.perf_counter()
    with torch.no_grad():                                  # per-stage split of the CPU forward (SURVEY 8d)
        c = net.backbone(img)
        t1 = time.perf_counter()
        p = net.neck(c)
        t2 = time.perf_counter()
        cls, box, ctr, cof, fm = net.bbox_head(p)
    t3 = time.perf_counter()
    real_nms = O.nms
    O.nms = lambda dets, thr, cmp_ge=False, plus_one=True: cbind.nms(dets, thr, int(cmp_ge), int(plus_one))
    shape = (wl['H'], wl['img_w'], 3)
    sf = np.ones(4, dtype=np.float32) if wl['ssd'] else 1.0
    post = {}
    try:
        res = P.get_bboxes_single([t[0] for t in cls], [t[0] for t in box], [t[0] for t in ctr], [t[0] for t in cof], fm[0],
                                  (8, 16, 32, 64, 128), shape, shape, sf, test_cfg(wl), rescale=True, ssd_flag=wl['ssd'], timing=post)
    finally:
        O.nms = real_nms
    res['stage_s'] = dict(backbone=t1 - t0, fpn=t2 - t1, head=t3 - t2, decode_nms=post.get('decode_nms', 0.0),
                          mask_assembly=post.get('mask_assembly', 0.0), paste=post.get('paste', 0.0))
    return res


def cpu_reference(wl, steps, warmup, threads, budget_s=None):
    """Times WHOLE images only (r1's row-strip extrapolation was refuted by its own numbers): `warmup` untimed images, then
    `steps` timed ones.  With `budget_s` (the bounded CPU sample beside the GPU arm) the first image is a probe and both
    counts shrink to what fits the time budget, at least one warm-up and one timed image.  Returns (seconds per image,
    detections, images timed, per-image times, warm-up images)."""
    if wl.get('vis'):
        from oracle import postproc as P
        oracle_step.tracker = P.VISTracker()
    from sipmask_b200 import synth
    net = build_oracle(wl, threads)
    img = synth.synthetic_image(wl['H'], wl['W'], seed=0)
    n_warm, n_timed = max(0, warmup), steps
    if budget_s is not None:
        t0 = time.perf_counter()
        oracle_step(net, img, wl)                         # probe = first warm-up image
        t_probe = max(time.perf_counter() - t0, 1e-3)
        n_warm = 1 + max(0, min(warmup - 1, int(0.2 * budget_s / t_probe)))
        n_timed = max(1, min(steps, int(0.8 * budget_s / t_probe)))
    for _ in range(n_warm - (budget_s is not None)):
        oracle_step(net, img, wl)
    ts, stages = [], []
    for _ in range(n_timed):
        t0 = time.perf_counter()
        res = oracle_step(net, img, wl)
        ts.append(time.perf_counter() - t0)
        stages.append(res.get('stage_s'))
    cpu_reference.stage_split = None
    if all(stages):                                        # median per stage over the timed images (not for the VIS workload)
        cpu_reference.stage_split = {k: round(statistics.median(st[k] for st in stages), 4) for k in stages[0]}
    return statistics.median(ts), int(res['det_bboxes'].shape[0]), n_timed, ts, n_warm


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    threads, tinfo = host_threads()
    sec, ndet, n_timed, ts, n_warm = cpu_reference(wl, args.steps, args.warmup, threads)
    val = 1.0 / sec
    sample = ('%d whole %dx%d images timed (median) after %d warm-up image(s), through the '
              'oracle = PyTorch CPU fp32 restatement of the reference forward incl. get_bboxes on %d threads; the literal '
              'reference cannot run on CPU (DeformConv / CropSplit are CUDA-only)' % (n_timed, wl['H'], wl['W'], n_warm, threads))
    line = dict(impl='reference', metric='images/sec', value=val, unit='images/s', n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='f32', data='synthetic',
                config=dict(workload=wl['name'], detections=ndet, images_timed=n_timed, step_times_s=[round(t, 3) for t in ts],
                            images_per_step_per_gpu=1, host_threads=tinfo),
                cpu_baseline=dict(value=val, unit='images/s', cores=threads, kind='port', sample=sample,
                                  stage_split_s=cpu_reference.stage_split, torch=__import__('torch').__version__),
                e2e=dict(value=val, unit='images/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sipmask_b200 import dist as sdist
    from sipmask_b200 import ops, synth
    from sipmask_b200.serving import PipelinedRunner, EnginePool, make_engines

    wl = WORKLOADS[args.workload]
    H, W, IMG_W, B = wl['H'], wl['W'], wl['img_w'], wl['batch']
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (there is no CPU fallback for the product path)'
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')        # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)

    sd = state_dict_for(wl)
    vis = bool(wl.get('vis'))
    IMG_H = wl.get('img_h', H)
    nfl = max(1, args.in_flight if args.in_flight > 0 else wl['in_flight'])
    cfg = test_cfg(wl)
    sf = np.ones(4, dtype=np.float32) if wl['ssd'] else 1.0
    ekw = dict(depth=wl['depth'], stacked_convs=wl['stacked'], gn=wl['gn'], ssd_flag=wl['ssd'], batch=B, test_cfg=cfg,
               img_shape=(IMG_H, IMG_W, 3), scale_factor=sf, use_graph=True, device=dev, vis=vis,
               num_classes=wl.get('num_classes', 81))
    # nfl forwards in flight per GPU: nfl engines (shared weights, private activations + CUDA graph)
    engs = make_engines(sd, (H, W), in_flight=nfl, **ekw)
    eng = engs[0]
    img_host = torch.cat([synth.synthetic_image(H, W, seed=rank * B + b) for b in range(B)], 0).pin_memory()   # weak scaling
    for e in engs:
        e.img.copy_(img_host, non_blocking=True)
    torch.cuda.synchronize()
    pool = EnginePool(engs)
    # the single collective of the path (SURVEY.md 8e): records are logged locally per image and gathered ONCE at the end
    # of the run, inside the timed region
    # one STEP = one image (batch) through EVERY forward in flight: nfl * B images per GPU (workload A: 6 images, ~5 ms),
    # so the timed region of K = 20 steps is ~0.1 s instead of ~17 ms and the end-of-run gather / rank skew are measured
    # against a region long enough to resolve them (VERDICT r1: "run-to-run noise ... same order as the scaling loss")
    ips = nfl * B
    log = sdist.RecordLog(max(args.steps, 1) * ips, eng.max_num, dev, feat_dim=512 if vis else 0)
    gathered = torch.empty((world,) + tuple(log.buf.shape), dtype=torch.float32, device=dev) if world > 1 else None
    if vis:
        from sipmask_b200.tracker import Tracker
        tracker = Tracker()

    def consume(out):
        for b in range(B):
            log.append(out['det_bboxes'][b], out['det_labels'][b], out['count'][b:b + 1],
                       out['track_feats'][b] if vis else None)

    def finish_records():
        n_local = min(log.n, log.cap)
        g = log.gather(out=gathered)           # world == 1: a view, no communication
        if vis:                                # association in frame order on the gathered records (host, rank-replicated)
            tracker.reset()
            sdist.track_gathered(g, n_local * world, tracker)
        log.reset()

    def step():
        for _ in range(nfl):
            pool.step(consume)

    def step_finish():
        pool.flush(consume)
        finish_records()

    # end-to-end through the public serving API: pinned-host uint8 image in (the decoder's output; resize / normalise / pad /
    # layout run in one kernel on the device), pinned-host record + bit-packed masks out; upload / replay / download of
    # consecutive images overlap on their own streams (sipmask_b200/serving.py)
    raw = (B == 1 and not vis)
    if raw:
        g = torch.Generator().manual_seed(rank)
        img_u8 = (torch.rand(H, IMG_W, 3, generator=g) * 255.0).to(torch.uint8).pin_memory()
        runner = PipelinedRunner(engs, raw_hw=(H, IMG_W))
        e2e_in = img_u8
    else:
        runner = PipelinedRunner(engs)
        e2e_in = img_host
    copy_done = []

    def step_e2e():
        for _ in range(nfl):
            copy_done.append(runner.step(e2e_in, consume))
        del copy_done[:-1]

    def e2e_finish():
        runner.flush(consume)                  # the timed region ends when the last result is on the host
        finish_records()

    def timed(fn, steps, sample_clocks=False, finish=None, after=None):
        """K steps between barrier+synchronize, CUDA events, max over ranks.  nvidia-smi samples clocks every 100 ms;
        a short timed region would get no sample, so ROLL untimed steps of the same load run before and after it and
        the sampler stays on throughout (clocks.window says so).  `after` runs once the timed steps are complete, before
        the untimed steps after them overwrite their outputs."""
        sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
        roll = max(1, ROLL // ips)
        if sample_clocks:
            # nvidia-smi needs ~0.3 s to start and samples every 100 ms: make each roll last >= 0.8 s of the same load
            # (short steps - workloads B / C - got no sample with a fixed count); every rank uses the same count
            t0 = time.perf_counter()
            for _ in range(3):
                fn()
            if finish is not None:
                finish()
            torch.cuda.synchronize()
            per = max(1e-5, (time.perf_counter() - t0) / 3)
            need = torch.tensor([max(roll, int(0.8 / per) + 1)], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(need, op=dist.ReduceOp.MAX)
            roll = int(need.item())
        if sampler:
            sampler.start()
        if sample_clocks:
            for _ in range(roll):                       # fixed count: every rank must issue the same collectives
                fn()
            if finish is not None:
                finish()
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()                                # joins the images in flight / downloads and issues the end-of-run gather
        e1.record()
        torch.cuda.synchronize()
        if after is not None:
            after()
        if world > 1:
            dist.barrier()
        if sample_clocks:
            for _ in range(roll):
                fn()
            if finish is not None:
                finish()
            torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        if clocks is not None:
            clocks['window'] = 'timed region plus %d untimed steps of the identical load before and after it' % roll
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), clocks

    for _ in range(max(args.warmup, 3)):
        step()
    step_finish()
    torch.cuda.synchronize()
    last_step = {}
    total_ms, clocks = timed(step, args.steps, sample_clocks=True, finish=step_finish,
                             after=(lambda: last_step.update(step_outputs(engs))) if args.dump_outputs and rank == 0 else None)
    if last_step:
        write_outputs(args.dump_outputs, last_step)
    ms_per_step = total_ms / args.steps
    value = world * ips * 1000.0 / ms_per_step
    for _ in range(3):
        step_e2e()
    e2e_finish()
    e2e_ms, _ = timed(step_e2e, args.steps, finish=e2e_finish)
    e2e_value = world * ips * 1000.0 / (e2e_ms / args.steps)
    last = runner.result(copy_done[-1])
    assert int(last['cnt'][0]) > 0
    h2d, d2h = runner.h2d_bytes * nfl, runner.d2h_bytes * nfl
    ndet = int(eng.count[0].item())

    line = dict(metric='images/sec', value=value, unit='images/s', n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                ms_per_step=ms_per_step, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f16',
                data='synthetic',
                config=dict(workload=wl['name'],
                            parallelism='dp%d (%d forward(s) in flight per GPU, one image batch through each per step; detection '
                                        'records logged on the device and all-gathered ONCE at the end of the run, inside the '
                                        'timed region)' % (world, nfl),
                            detections_per_image=ndet, cuda_graph=True, forwards_in_flight=nfl, batch_per_forward=B,
                            images_per_step_per_gpu=ips,
                            l2='no flush: one step streams >= 1.3 GB of activations/masks through a 126 MB L2, so nothing but '
                               'weights can survive from the previous step'),
                clocks=clocks, e2e=dict(value=e2e_value, unit='images/s', h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                                        ms_per_step=e2e_ms / args.steps,
                                        input='uint8 BGR HWC image from pinned host memory (resize/normalise/pad on the device)'
                                              if raw else 'fp32 NCHW batch from pinned host memory'),
                gpu_launches=eng.n_launch * nfl * args.steps)
    torch.cuda.synchronize()

    if rank == 0:
        pk, pk_kind = peaks()
        traffic = ncu_traffic()
        # ---- roofline of the dominant kernel (conv_gemm_kernel): the conv launches of one step of EVERY engine in flight,
        # captured per engine (same stream schedule as in the step) and replayed concurrently on the pool's streams
        graphs = []
        for e, st in zip(engs, pool.streams):
            with torch.cuda.stream(st):
                e._run_ops(only={'conv'})
                st.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    e._run_ops(only={'conv'})
            graphs.append(g)
        torch.cuda.synchronize()

        def conv_round():
            for g, st in zip(graphs, pool.streams):
                with torch.cuda.stream(st):
                    g.replay()

        for _ in range(3):
            conv_round()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(3, min(args.steps, 20))
        e0.record()
        for st in pool.streams:
            st.wait_event(e0)
        for _ in range(reps):
            conv_round()
        pool.join()
        e1.record()
        torch.cuda.synchronize()
        conv_ms = e0.elapsed_time(e1) / (reps * nfl)                      # per forward
        tf = eng.conv_flops / (conv_ms * 1e-3) / 1e12
        peak_tf = float(pk.get('bf16_tflops_sustained', pk.get('bf16_tflops', 1400.0)))
        tr = traffic.get('conv_gemm_kernel', {})
        line['roofline'] = dict(bound='tensor', kernel='conv_gemm_kernel (%d launches/step)' % len(eng.conv_plans),
                                achieved=tf, peak=peak_tf, unit='TFLOP/s', frac=tf / peak_tf,
                                traffic=tr.get('dram_bytes_per_step') * nfl if tr.get('dram_bytes_per_step') else None,
                                traffic_source=tr.get('source'),
                                peak_source=pk_kind + ' bf16_tflops_sustained', algorithmic_gflop_per_step=eng.conv_flops * nfl / 1e9,
                                ms_per_step=conv_ms * nfl, share_of_step=conv_ms * nfl / ms_per_step,
                                ms_per_forward=conv_ms,
                                note='conv launches of %d forwards in flight replayed concurrently (one step = %d forwards)'
                                     % (nfl, nfl))
        del graphs
        # ---- strictly serial reference point: ONE engine tuned for a single stream, one forward at a time
        if nfl > 1:
            e1s = make_engines(sd, (H, W), in_flight=1, **ekw)[0]
            e1s.img.copy_(img_host, non_blocking=True)
            for _ in range(5):
                e1s.forward(None)
            torch.cuda.synchronize()
            e0.record()
            nser = max(args.steps, 20)
            for _ in range(nser):
                e1s.forward(None)
            e1.record()
            torch.cuda.synchronize()
            sms = e0.elapsed_time(e1) / nser
            line['serial'] = dict(ms_per_step=sms, value=B * 1000.0 / sms, unit='images/s',
                                  note='one forward in flight (latency-optimal planner settings), same GPU, N=1 rank only')
            del e1s
        if args.workload == 'A':
            mask_rooflines(line, eng, pk, pk_kind, traffic, H, IMG_W)
            line['e2e_dropin'] = dropin_timing(eng, sd, cfg, H, IMG_W)
            if not args.no_library_baseline:
                line['library_gpu_baseline'] = library_baseline(wl, img_host, dev)
        # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload on the host cores
        if world == 1 and not args.no_cpu_baseline:
            threads, tinfo = host_threads()
            sec, _, n_timed, ts, n_warm = cpu_reference(wl, 3, 1, threads, budget_s=25.0)
            line['cpu_baseline'] = dict(value=1.0 / sec, unit='images/s', cores=threads, kind='port', host_threads=tinfo,
                                        stage_split_s=cpu_reference.stage_split, torch=torch.__version__,
                                        sample='%d whole %dx%d image(s) timed (median) after %d warm-up, through the oracle (PyTorch '
                                               'CPU fp32 restatement of the reference forward incl. get_bboxes)' % (n_timed, H, W, n_warm))
        else:
            line['cpu_baseline'] = None
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 48 << 20      # --dump-outputs writes at most this much


def step_outputs(engs):
    """What the last forward of every engine returned (the record EnginePool.consume hands to its caller), one row per
    image in engine order, as float32 / float64 numpy arrays: count [I]; det_bboxes [I,max,5], det_labels and idxs_keep
    [I,max], track_feats [I,max,512] (VIS only), with the rows at and past count zeroed (no forward writes them).  The
    bit-packed masks [I,max,H,ceil(W/32)] int32 are kept as a fixed, seeded sample of their words (all of them when they
    fit in DUMP_BYTES): mask_bits_sample [I,K] holds the words at the flat per-image positions mask_bits_index [K]."""
    import numpy as np
    import torch
    recs = [e._result() for e in engs]

    def cat(k):
        return torch.cat([r[k] for r in recs], 0)

    count = cat('count').long()
    n_img, max_num = count.shape[0], recs[0]['det_bboxes'].shape[1]
    valid = torch.arange(max_num, device=count.device).view(1, max_num) < count.view(n_img, 1)

    def rows(t):
        keep = valid.view(n_img, max_num, *([1] * (t.dim() - 2)))
        return torch.where(keep, t, torch.zeros((), dtype=t.dtype, device=t.device))

    out = dict(count=count.float(), det_bboxes=rows(cat('det_bboxes')), det_labels=rows(cat('det_labels')).float(),
               idxs_keep=rows(cat('idxs_keep')).double())
    if 'track_feats' in recs[0]:
        out['track_feats'] = rows(cat('track_feats'))
    bits = rows(cat('mask_bits')).view(n_img, -1)
    per_img = bits.shape[1]
    k = (DUMP_BYTES - sum(t.numel() * t.element_size() for t in out.values())) // (8 * (n_img + 1))
    idx = np.arange(per_img) if per_img <= k else np.sort(np.random.RandomState(0).choice(per_img, k, replace=False))
    out['mask_bits_sample'] = bits.index_select(1, torch.from_numpy(idx).to(bits.device)).double()
    out['mask_bits_index'] = torch.from_numpy(idx.astype(np.float64))
    return {name: t.cpu().numpy() for name, t in out.items()}


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def mask_rooflines(line, eng, pk, pk_kind, traffic, H, IMG_W):
    """Mask assembly (BASELINE metric part 2): HBM GB/s at N = max_per_img detections with 32-512 px boxes, L2 flushed
    between launches.  Each number is the whole ABI call (zero-fill memset node + kernel)."""
    import torch
    from sipmask_b200 import ops
    dev = eng.dev
    N = eng.max_num
    Hm, Wm = eng.protos.shape[1], eng.protos.shape[2]
    gen = torch.Generator().manual_seed(0)
    cofs = torch.randn(N, 128, generator=gen).to(dev)
    cx, cy = torch.rand(N, generator=gen) * IMG_W, torch.rand(N, generator=gen) * H
    bw, bh = torch.rand(N, generator=gen) * 480 + 32, torch.rand(N, generator=gen) * 480 + 32
    boxes = torch.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1).clamp(min=0).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    pos = torch.empty((N, Hm, Wm), dtype=torch.float32, device=dev)
    bits = torch.empty((N, H, (IMG_W + 31) // 32), dtype=torch.int32, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_kernel(fn):
        ts = []
        for i in range(10):
            flush.fill_(i)                                 # evict L2 between timed launches
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts[2:])

    protos = eng.protos[0]
    tensor_dot = ops.set_mask_tensor_dot(None)             # the family the engine runs (fp16 prototypes)
    fam = 'mma.sync dot products' if tensor_dot else 'scalar fmaf dot products'
    # the other family, same inputs, for the record
    ops.set_mask_tensor_dot(not tensor_dot)
    other = dict(kernels='scalar fmaf' if tensor_dot else 'mma.sync',
                 dense_ms=time_kernel(lambda: ops.mask_assemble(protos, cofs, boxes, 0.5, layout='hwc', out=pos)),
                 fused_ms=time_kernel(lambda: ops.mask_assemble_pack(protos, cofs, boxes, 0.5, (H, IMG_W), 0.4, layout='hwc', out=bits)))
    ops.set_mask_tensor_dot(tensor_dot)
    # (a) the reference-shaped output: dense pos_masks [N,Hm,Wm] fp32 (what CropSplit returns, permuted)
    ma_ms = time_kernel(lambda: ops.mask_assemble(protos, cofs, boxes, 0.5, layout='hwc', out=pos))
    ma_bytes = Hm * Wm * 32 * 2 + N * 128 * 4 + N * 16 + N * Hm * Wm * 4
    gbs = ma_bytes / (ma_ms * 1e-3) / 1e9
    tr = traffic.get('mask_assemble', {})
    line['roofline_mask_assembly'] = dict(bound='hbm', kernel='mask_assemble%s_kernel, %s (writes every output element; no memset)'
                                                              % ('_mma' if tensor_dot else '', fam), achieved=gbs,
                                          peak=float(pk['hbm_gbs']), unit='GB/s', frac=gbs / float(pk['hbm_gbs']),
                                          traffic=tr.get('dram_bytes_per_launch'), traffic_source=tr.get('source'), ms=ma_ms,
                                          algorithmic_bytes=ma_bytes, peak_source=pk_kind + ' hbm_gbs',
                                          note='protos fp16 HWC read once + fp32 pos_masks [100,400,672] written; L2 flushed between launches')
    # (b) the path the engine runs: fused assembly + bilinear resize + threshold + bit-pack (no pos_masks traffic)
    mf_ms = time_kernel(lambda: ops.mask_assemble_pack(protos, cofs, boxes, 0.5, (H, IMG_W), 0.4, layout='hwc', out=bits))
    mf_bytes = Hm * Wm * 32 * 2 + N * 128 * 4 + N * 16 + bits.numel() * 4
    mgbs = mf_bytes / (mf_ms * 1e-3) / 1e9
    tr = traffic.get('mask_fused', {})
    line['roofline_mask_fused'] = dict(bound='hbm', kernel='smb_mask_assemble_pack = memset + mask_fused_pack%s_kernel, %s'
                                                           % ('_mma' if tensor_dot else '', fam), achieved=mgbs,
                                       peak=float(pk['hbm_gbs']), unit='GB/s', frac=mgbs / float(pk['hbm_gbs']),
                                       traffic=tr.get('dram_bytes_per_launch'), traffic_source=tr.get('source'), ms=mf_ms,
                                       algorithmic_bytes=mf_bytes, peak_source=pk_kind + ' hbm_gbs',
                                       note='protos fp16 read once + bit-packed [100,800,42] int32 masks written')
    line['roofline_mask_assembly']['other_family'] = dict(kernels=other['kernels'], ms=other['dense_ms'])
    line['roofline_mask_fused']['other_family'] = dict(kernels=other['kernels'], ms=other['fused_ms'])


def dropin_timing(eng, sd, cfg, H, IMG_W):
    """The reference's call pattern through the drop-in module (detectors/single_stage.py:75-93): SipMaskHead.forward(feats)
    + get_bboxes(..., rescale=True) -> python result with COCO RLE strings on the host; wall clock per image.  The five FPN
    maps are the engine's own (NCHW fp32 copies, as the reference's neck would hand them over)."""
    import torch
    from sipmask_b200.head import SipMaskHead

    class Cfg(dict):
        __getattr__ = dict.get
    head = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=4, strides=[8, 16, 32, 64, 128])
    head.load_state_dict({k[len('bbox_head.'):]: v for k, v in sd.items() if k.startswith('bbox_head.')}, strict=True)
    head = head.to(eng.dev).eval()
    feats = tuple(f.permute(0, 3, 1, 2).float().contiguous() for f in eng.fpn_outs)
    tcfg = Cfg(cfg)
    tcfg['nms'] = Cfg(cfg['nms'])
    meta = dict(img_shape=(H, IMG_W, 3), ori_shape=(H, IMG_W, 3), scale_factor=1.0)
    ts = []
    k = 0
    for i in range(7):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        outs = head(feats)
        det, lab, segms = head.get_bboxes(*outs, [meta], tcfg, rescale=True)[0]
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        k = int(det.shape[0])
    ms = statistics.median(ts[2:]) * 1e3
    return dict(ms_per_image=ms, value=1000.0 / ms, unit='images/s (head + post-processing only)', detections=k,
                note='wall clock of SipMaskHead.forward + get_bboxes (eager launches, one host sync per image, RLE strings built '
                     'on the host from device run lengths); backbone / neck are the caller\'s on this path')


def library_baseline(wl, img_host, dev):
    """Informational: the same network through the library path on this GPU (PyTorch eager: cuDNN / cuBLAS convolutions,
    ATen GroupNorm / interpolate, torchvision deform_conv2d), fp16 channels_last, forward only (no post-processing)."""
    import torch
    try:
        from oracle import model as M
        from oracle import ops as O
        from sipmask_b200 import synth
        O.USE_TORCHVISION_DCN = True
        net = M.SipMaskDetector(wl['depth'], stacked_convs=wl['stacked'], gn=wl['gn'], ssd_flag=wl['ssd'])
        net.load_state_dict(synth.detector_state_dict(wl['depth'], stacked_convs=wl['stacked'], gn=wl['gn'], seed=1,
                                                      cls_bias=CLS_BIAS), strict=True)
        net = net.to(dev).half().to(memory_format=torch.channels_last).eval()
        x = img_host.to(dev).half().contiguous(memory_format=torch.channels_last)
        torch.backends.cudnn.benchmark = True
        with torch.no_grad():
            for _ in range(5):
                net(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = 20
            for _ in range(n):
                net(x)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        return dict(ms_per_image=ms, value=1000.0 / ms, unit='images/s',
                    note='oracle SipMaskDetector on CUDA, fp16 channels_last, cudnn.benchmark, eager; network forward ONLY '
                         '(decode / NMS / mask assembly excluded, so this favours the library path)')
    except Exception as ex:                                    # informational leg: never fail the bench line
        return dict(unavailable='%s: %s' % (type(ex).__name__, str(ex)[:200]))
    finally:
        try:
            O.USE_TORCHVISION_DCN = False
        except Exception:
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='A', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-library-baseline', action='store_true')
    ap.add_argument('--in-flight', type=int, default=int(os.environ.get('SMB_IN_FLIGHT', '0')),
                    help='forwards in flight per GPU (independent forwards on separate streams); 0 = the workload default, '
                         '1 = strictly serial')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (rank 0, see step_outputs) to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
