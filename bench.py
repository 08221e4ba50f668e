#!/usr/bin/env python
"""bench.py -- the hot path's headline metric on synthetic data.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp16|fp32] [--impl reference] [--scaling weak|strong]

Metric (BASELINE.json): img/s of res101_coco 550x550, batch 64, eval forward + fused post-process (decode + Fast-NMS +
top-k); Fast-NMS us/img reported alongside.  One "step" = one pass of the hot path over one batch per GPU.  For N > 1 the
driver launches one rank per GPU with torch.distributed.run; images shard across ranks (no data-path collective) and the
detection records are all-gathered over NCCL once per step, overlapped with the next step's forward.

Rank 0 prints ONE JSON line:
  value / ms_per_step  device-resident inputs, per-op profiling OFF, CUDA events, max over ranks; `--scaling weak` (default): 64
                       images per GPU; the same line carries `strong_scaling` (BASELINE configs[2] as stated: GLOBAL batch 64,
                       64/N images per GPU) measured in the same run.  `--scaling strong` makes that leg the line's `value`.
  e2e                  N = 1: the C ABI with HOST buffers (yb_net_submit_host / collect_host: pinned host input, H2D + forward +
                       post-process + D2H of the records in the timed region); N > 1: the package's public calls (pinned host
                       tensor -> .to(device) -> Yolact.forward -> detect_batched -> dist.gather_detections -> D2H of the
                       gathered records), i.e. the collective is inside the timed region.
  roofline             per-launch CUDA-event timing of every layer in a SEPARATE profiling pass; `traffic` = measured DRAM
                       bytes per k_conv_tc launch from the committed ncu pass over all launches of one step (profiles/).
  gpu_eager_baseline   N = 1: the reference's own GPU path on the same box -- its unmodified modules ($YOLACT_REFERENCE, else the
                       torch restatement in oracle/) .cuda().eval(), cudnn.benchmark=True (eval.py:122-125), TF32 default and
                       bf16 autocast, same batch, CUDA events -- with ours / eager ratios.
  cpu_baseline         N = 1: the reference's CPU path on the host cores, bounded sample.
  parity               the TIMED B=64 output itself: images 0/31/63 vs the fp32 oracle and bit-wise vs B=1 runs; N > 1: the
                       gathered records vs rank 0 re-running every rank's batch on one GPU, bit-for-bit.
  other_configs        BASELINE configs[1] (res50 bs32), configs[4] (swin_tiny bs32) and the 544 variants, N = 1.
  mask_stage           after_nms for 100 detections at 480x640 (float32 / uint8 / bit-packed masks), mask IoU and RLE on the packed masks, N = 1.
  training             BASELINE configs[3]: res101 550x550 training step (native engine forward + backward + SGD), bs 2 per GPU, DDP over
                       NCCL at N > 1; at N = 1 beside the same step on torch autograd / cuDNN.
`--impl reference` times the reference's CPU implementation of the path (the reference itself when $YOLACT_REFERENCE names a
checkout of it, else the port).
`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32 / float64): the
detection records det_count, det_cls, det_anchor, det_score, det_box, det_coef (rank 0; all ranks' records at N > 1), and the
network outputs cls, box, coef, proto (rank 0's shard; arrays above DUMP_SAMPLE elements as a fixed seeded sample of flat
positions).  Inputs and weights are seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ARCH, IMG, BATCH = 'res101', 550, 64
# SURVEY.md section 6: algorithmic 2*MAC of the reference forward per image
GFLOPS = {('res101', 550): 164.68, ('res101', 544): 157.16, ('res50', 550): 118.28, ('res50', 544): 113.38,
          ('swin_tiny', 550): 123.43, ('swin_tiny', 544): 119.19}


def host_cores():
    """CPU threads this process can actually use: min(affinity, cgroup cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(int(q) / int(per))))
    except (OSError, ValueError):
        pass
    return n


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf=d['bf16_tflops'], tf_sustained=d['bf16_tflops_sustained'], src='measured')
    return dict(hbm=6650.0, tf=1590.0, tf_sustained=1400.0, src='fallback')


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self, t0=None, t1=None):
        """Summarise the samples taken between wall-clock times t0 and t1 (the timed region)."""
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(2)
        import datetime
        sm, pw, mx, reasons = [], [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(',')]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.05):
                    continue
                sm.append(float(f[1])); mx = float(f[2]); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx, 'power_w_max': max(pw) if pw else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU path (eval forward + nms() per image), fp32, all host threads
# ----------------------------------------------------------------------------------------------------
def cpu_reference_sample(arch, img_size, n_img, reps, threads):
    """Returns (img_per_s, seconds, fast_nms_us_per_img, kind).  kind = 'reference' when the unmodified reference is available
    ($YOLACT_REFERENCE: its Yolact.forward + utils/output_utils.nms, FPN run-time patch for sizes % 32 != 0), else 'port' (oracle/)."""
    import torch
    from oracle import synth, forward_torch as ft, postprocess_np as pp, ref_loader
    torch.set_num_threads(threads)
    sd = ft.synth_state_dict(arch, seed=0)
    img = torch.from_numpy(synth.image_batch(1, n_img, img_size))
    t_nms = 0.0
    if ref_loader.available():
        kind = 'reference'
        net, cfg = ref_loader.build_net(arch, img_size, sd)
        rnms = ref_loader.load()[2].nms
        with torch.no_grad():
            net(img[:1])                                                # warm-up
            t0 = time.perf_counter()
            for _ in range(reps):
                cls, box, coef, proto = net(img)
                t1 = time.perf_counter()
                for b in range(n_img):                                  # the reference's nms() is batch-1 (output_utils.py:127-130)
                    rnms(cls[b:b + 1], box[b:b + 1], coef[b:b + 1], proto[b:b + 1], net.anchors, cfg)
                t_nms += time.perf_counter() - t1
            dt = time.perf_counter() - t0
    else:
        kind = 'port'
        anchors = pp.make_anchors(img_size)
        ft.forward(img[:1], sd, arch)                                   # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            cls, box, coef, proto = [t.numpy() for t in ft.forward(img, sd, arch)]
            t1 = time.perf_counter()
            for b in range(n_img):
                pp.nms(cls[b], box[b], anchors)
            t_nms += time.perf_counter() - t1
        dt = time.perf_counter() - t0
    return n_img * reps / dt, dt, 1e6 * t_nms / (n_img * reps), kind


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = host_cores()
    n_img = 4
    vals, t_all, nms_us, kind = [], 0.0, 0.0, 'port'
    steps = max(1, min(args.steps, 20))                             # bounded: each step is a 4-image sample
    for _ in range(steps):
        v, dt, nu, kind = cpu_reference_sample(ARCH, IMG, n_img, 1, cores)
        vals.append(v); t_all += dt; nms_us = nu
    value = float(np.mean(vals))
    what = ('the UNMODIFIED reference ($YOLACT_REFERENCE: Yolact.forward + utils/output_utils.nms' + (', FPN interpolate-to-size run-time patch for 550' if IMG % 32 else '') + ')'
            if kind == 'reference' else 'CPU port of the reference path (oracle/)')
    line = {'impl': 'reference', 'metric': 'img/s', 'value': value, 'unit': 'img/s', 'n_gpus': args.gpus, 'steps': steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * t_all / steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'{ARCH}_coco {IMG}x{IMG} eval forward + Fast-NMS on the host CPU: {what}, '
                                   f'bounded sample of {n_img} images per step (full workload: bs={BATCH})'},
            'cpu_baseline': {'value': value, 'unit': 'img/s', 'cores': cores, 'kind': kind,
                             'sample': f'{steps} x {n_img} images, torch fp32 CPU forward + nms() per image'},
            'fast_nms_us_per_img': nms_us,
            'e2e': {'value': value, 'unit': 'img/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
def cuda_time(fn, reps):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps                                  # ms per call


DUMP_SAMPLE = 1 << 20     # elements kept of each network output by --dump-outputs: 4 x 4 MB, beside ~1 MB of detection records


def dump_outputs(dirname, outs, det):
    """--dump-outputs: the network outputs (cls, box, coef, proto) and the detection records (det_*) of one step as .npy files.
    An output above DUMP_SAMPLE elements is written as the values at the sorted flat positions np.unique of DUMP_SAMPLE draws
    from default_rng(0), the same positions in every run of the same shape."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    arrays = {}
    for name, t in zip(('cls', 'box', 'coef', 'proto'), outs):
        if t.numel() > DUMP_SAMPLE:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_SAMPLE))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        arrays[name] = t.float().cpu().numpy()
    for k in ('count', 'cls', 'anchor', 'score', 'box', 'coef'):
        a = det[k].cpu().numpy()
        arrays['det_' + k] = a.astype(np.float64 if a.dtype.kind in 'iu' else np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), a)


def gpu_eager_baseline(arch, img_size, batch, dev, our_img_s, steps=5):
    """The reference's own GPU path, on this box: eager PyTorch / cuDNN, as eval.py:122-125 runs it."""
    import torch
    from oracle import forward_torch as ft, ref_loader
    sd = ft.synth_state_dict(arch, seed=0)
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    out = {'batch': batch, 'steps': steps, 'what': 'eval forward only (the reference has no batched post-process: its nms() is batch-1 Python); '
                                                   'ours / eager compares OUR forward + post-process step against it'}
    x = torch.randn(batch, 3, img_size, img_size, device=dev)
    try:
        if ref_loader.available():
            net, _ = ref_loader.build_net(arch, img_size, sd)
            net = net.to(dev)
            fwd = lambda: net(x)
            out['impl'] = 'unmodified reference modules ($YOLACT_REFERENCE)' + (' + FPN interpolate-to-size run-time patch' if img_size % 32 else '')
        else:
            sdd = {k: v.to(dev) for k, v in sd.items()}
            fwd = lambda: ft.forward(x, sdd, arch)
            out['impl'] = 'torch restatement of the reference forward (oracle/forward_torch.py; bit-identical to the reference on CPU)'
        for name, ctx in (('tf32', None), ('bf16_autocast', torch.autocast('cuda', dtype=torch.bfloat16))):
            torch.backends.cudnn.allow_tf32 = True
            torch.backends.cuda.matmul.allow_tf32 = True

            def run(_):
                with torch.no_grad():
                    if ctx is None:
                        fwd()
                    else:
                        with ctx:
                            fwd()
            for i in range(3):
                run(i)
            torch.cuda.synchronize()
            ms = cuda_time(run, steps)
            out[name] = {'img_per_s': batch / (ms / 1e3), 'ms_per_step': ms, 'ours_over_eager': our_img_s / (batch / (ms / 1e3))}
    except Exception as e:                                          # a baseline leg must not take the bench line down
        out['error'] = repr(e)[:300]
    finally:
        torch.backends.cudnn.benchmark = prev
    torch.cuda.empty_cache()
    return out


def build_net(arch, img_size, batch, precision, dev):
    from oracle import forward_torch as ft
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.modules.yolact import Yolact
    cfg = make_config(arch + '_coco', img_size)
    cfg.precision, cfg.max_batch = precision, batch
    net = Yolact(cfg)
    net.load_state_dict(ft.synth_state_dict(arch, seed=0), strict=True)
    net = net.to(dev).eval()
    return net, cfg, net.engine(batch)


def measure_config(arch, img_size, batch, precision, dev, steps, pk):
    """Device-resident img/s of another BASELINE configuration (single GPU), same step definition."""
    import torch
    from yolact_minimal_b200.utils.output_utils import detect_batched
    net, cfg, eng = build_net(arch, img_size, batch, precision, dev)
    anchors = torch.from_numpy(eng.anchors()).to(dev)
    gen = torch.Generator().manual_seed(99)
    imgs = [torch.randn(batch, 3, img_size, img_size, generator=gen).to(dev) for _ in range(2)]

    def step(i):
        with torch.no_grad():
            cls, box, coef, proto = net(imgs[i & 1])
        return detect_batched(cls, box, coef, anchors, cfg)
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    ms = cuda_time(step, steps)
    v = batch / (ms / 1e3)
    gf = GFLOPS.get((arch, img_size))
    del net, eng, imgs
    torch.cuda.empty_cache()
    return {'workload': f'{arch}_coco {img_size}x{img_size} bs={batch}', 'value': v, 'unit': 'img/s', 'ms_per_step': ms, 'steps': steps,
            'tensor_frac_of_peak': v * gf * 1e9 / (pk['tf_sustained'] * 1e12) if gf else None}


def mask_stage_leg(dev, pk, img_size=550, img_h=480, img_w=640, reps=20):
    """after_nms (mask assembly: proto @ coef^T, sigmoid, crop, up-sampling to the image, threshold) for the 100 detections of one image,
    in the reference's float32 mask format and in the byte / bit-packed formats, then the stage the reference's evaluation loop runs on
    the masks (mask IoU against ground truth, COCO RLE).  Output-write bound: the roofline is the mask bytes written per image."""
    import torch
    from oracle import synth, postprocess_np as pp
    from yolact_minimal_b200.utils.output_utils import after_nms
    from yolact_minimal_b200.utils import mask_utils as mu
    anchors = pp.make_anchors(img_size)
    cls, box, coef = synth.head_outputs(5, anchors.shape[0], 81, 'realistic')
    proto = synth.proto(5, (img_size + 3) // 4)
    ids, scores, boxes, aidx = pp.nms(cls, box, anchors)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    args = (t(ids), t(scores), t(boxes), t(coef[aidx]), t(proto), img_h, img_w)
    d = len(ids)
    out = {'detections': d, 'image': f'{img_h}x{img_w}', 'proto': int(proto.shape[0])}
    for name, dt, bpp in (('float32', torch.float32, 4.0), ('uint8', torch.uint8, 1.0), ('bits', 'bits', 0.125)):
        for _ in range(3):
            after_nms(*args, mask_dtype=dt)
        ms = cuda_time(lambda i: after_nms(*args, mask_dtype=dt), reps)
        wbytes = d * img_h * img_w * bpp
        out[name] = {'ms_per_image': ms, 'mask_bytes_per_image': wbytes, 'write_gbs': wbytes / (ms * 1e-3) / 1e9, 'frac_of_hbm_peak': wbytes / (ms * 1e-3) / 1e9 / pk['hbm']}
        try:                                                        # the same call replayed from a CUDA graph: device time without the Python / launch gaps
            g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
            with torch.cuda.stream(st):
                after_nms(*args, mask_dtype=dt)
                torch.cuda.synchronize()
                with torch.cuda.graph(g, stream=st):
                    keep = after_nms(*args, mask_dtype=dt)
            torch.cuda.synchronize()
            gms = cuda_time(lambda i: g.replay(), reps)
            out[name].update({'graph_ms_per_image': gms, 'graph_write_gbs': wbytes / (gms * 1e-3) / 1e9, 'graph_frac_of_hbm_peak': wbytes / (gms * 1e-3) / 1e9 / pk['hbm']})
            del g, keep
        except Exception as e:
            out[name]['graph_error'] = repr(e)[:200]
    bits = after_nms(*args, mask_dtype='bits')[3]
    gt = bits[:20].contiguous()
    for _ in range(3):
        mu.mask_iou_bits(bits, gt)
    out['mask_iou_100x20_ms'] = cuda_time(lambda i: mu.mask_iou_bits(bits, gt), reps)
    t0 = time.perf_counter()
    for _ in range(5):
        mu.encode_rle(bits, img_h, img_w)
    out['rle_100_masks_ms_incl_host_string'] = (time.perf_counter() - t0) / 5 * 1e3
    return out


TRAIN_LR = 2e-4   # config.py:97 uses 2e-3 with warm-up on real data; random-init weights on random targets diverge at that rate within ~50 steps


def training_leg(arch, img_size, per_gpu, steps, dev, rank, world, eager_only=False):
    """BASELINE.json configs[3]: res101_coco 550x550 training, bs per GPU = 2 (DDP 8x2 at N = 8), synthetic targets (3 boxes per image,
    seed 1 + rank), SGD lr TRAIN_LR momentum 0.9 wd 5e-4 (config.py:97-100), `steps` timed steps.  The step is Yolact.forward in train mode
    (native engine: forward + targets + losses) + loss.backward() (native backward) + optimizer.step(); under torchrun the module is
    wrapped in DistributedDataParallel (train.py:76) and the gradient all-reduce runs over NCCL.  Beside it, at N = 1: the same step
    on the reference's own GPU path (torch autograd over cuDNN: oracle/train_torch.py, TF32 default, cudnn.benchmark)."""
    import torch
    import torch.distributed as dist
    from oracle import synth, forward_torch as ft, train_torch as tt
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.modules.yolact import Yolact

    def make():
        cfg = make_config(arch + '_coco', img_size, mode='train', train_bs=per_gpu)
        net = Yolact(cfg)
        net.load_state_dict(ft.synth_state_dict(arch, seed=0, train=True), strict=True)
        return net.to(dev).train()
    img = torch.from_numpy(synth.image_batch(100 + rank, per_gpu, img_size)).to(dev)
    tg, mk = synth.train_targets(1 + rank, per_gpu, img_size)
    tgt = [torch.from_numpy(t).to(dev) for t in tg]
    mks = [torch.from_numpy(m).to(dev) for m in mk]
    out = {'workload': f'{arch}_coco {img_size}x{img_size} training, bs={per_gpu}/GPU x {world} GPU(s), synthetic targets, SGD', 'steps': steps}

    def run(net, fwd, n):
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index], broadcast_buffers=True) if world > 1 else net
        opt = torch.optim.SGD(model.parameters(), lr=TRAIN_LR, momentum=0.9, weight_decay=5e-4)
        first = None

        def step(_):
            nonlocal first
            losses = fwd(model)
            if first is None:
                first = [float(l.detach()) for l in losses]
            opt.zero_grad(set_to_none=True)
            sum(losses).backward()
            opt.step()
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = cuda_time(step, n)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), first
    try:
        if eager_only:                                              # child process (see below)
            torch.backends.cudnn.benchmark = True
            torch.backends.cudnn.allow_tf32 = True
            torch.backends.cuda.matmul.allow_tf32 = True
            ems, efirst = run(make(), lambda m: tt.training_step_forward(m, img, tgt, mks), max(5, steps // 5))
            return {'impl': 'torch autograd over cuDNN / ATen (oracle/train_torch.py: the reference training branch restated), TF32, cudnn.benchmark',
                    'img_per_s': per_gpu / (ems / 1e3), 'ms_per_step': ems, 'first_step_losses': efirst}
        net = make()
        ms, first = run(net, lambda m: m(img, tgt, mks), steps)
        out.update(value=world * per_gpu / (ms / 1e3), unit='img/s', ms_per_step=ms, first_step_losses=first, dtype='bf16 tensor-core operands, f32 accumulation / statistics / master weights',
                   launches_per_step=next(iter(net._train_engines.values())).launches_per_step())
        del net
        torch.cuda.empty_cache()
        if world == 1:
            # the eager baseline runs in a CHILD process: ATen's loss kernels device-assert on a NaN (a diverged run), and a device-side
            # assert would take this process's CUDA context -- and every later leg of the bench line -- with it
            import subprocess
            r = subprocess.run([sys.executable, os.path.abspath(__file__), '--eager-train-leg', '--arch', arch, '--img', str(img_size), '--batch', str(per_gpu),
                                '--steps', str(steps)], capture_output=True, text=True, timeout=600)
            js = [l for l in r.stdout.splitlines() if l.startswith('{')]
            if r.returncode == 0 and js:
                eb = json.loads(js[-1])
                eb['ours_over_eager'] = (per_gpu / (ms / 1e3)) / eb['img_per_s']
                out['gpu_eager_baseline'] = eb
            else:
                out['gpu_eager_baseline'] = {'error': (r.stderr or r.stdout)[-300:]}
    except Exception as e:
        out['error'] = repr(e)[:400]
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from oracle import synth, forward_torch as ft, postprocess_np as pp        # cpu_baseline leg, parity gate, synthetic inputs only
    from yolact_minimal_b200 import _lib, dist as ydist
    from yolact_minimal_b200.utils.output_utils import detect_batched

    rank, world, local = ydist.init_from_env()
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    K, W = args.steps, max(args.warmup, 3)
    pk = peaks()
    GFLOP_PER_IMG = GFLOPS.get((ARCH, IMG), float('nan'))

    net, cfg, eng = build_net(ARCH, IMG, BATCH, args.precision, dev)
    anchors = torch.from_numpy(eng.anchors()).to(dev)
    # two distinct resident input batches (232 MB each > 126 MB L2), alternated between steps
    seed_of = lambda r: 1234 + r
    gen = torch.Generator().manual_seed(seed_of(rank))
    host = [torch.randn(BATCH, 3, IMG, IMG, generator=gen).pin_memory() for _ in range(2)]     # ~N(0,1) like normalised RGB
    imgs = [h.to(dev) for h in host]

    def make_step(b):
        """forward + post-process of b images per GPU; at N > 1 the record all-gather of step i overlaps the forward of i+1."""
        state = {'pending': None, 'outs': None, 'det': None}

        def step(i):
            with torch.no_grad():
                outs = net(imgs[i & 1][:b])
            det = detect_batched(outs[0], outs[1], outs[2], anchors, cfg)
            if world > 1:
                if state['pending'] is not None:
                    state['pending'].wait()                          # orders this stream after the PREVIOUS step's collective
                state['pending'] = ydist.gather_detections(det, async_op=True)
            state['outs'], state['det'] = outs, det

        def drain():
            if state['pending'] is not None:
                state['pending'].wait()
            return state
        return step, drain

    def timed(step, drain, K):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        wall0 = time.time()
        ev0.record()
        for i in range(K):
            step(i)
        drain()
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        wall1 = time.time()
        t = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), wall0, wall1

    sampler = ClockSampler(local)
    sampler.start()                                                 # nvidia-smi needs ~0.5 s to start: begin before warm-up
    per_gpu = {'weak': BATCH, 'strong': max(1, BATCH // world)}
    main_mode = args.scaling
    step, drain = make_step(per_gpu[main_mode])
    for i in range(W):
        step(i)
    drain()
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs, per-op profiling OFF ----------------------------------
    l0 = _lib.launch_count()
    torch.cuda.nvtx.range_push('timed')                       # ncu --nvtx --nvtx-include "timed/" isolates these K steps
    ms, wall0, wall1 = timed(step, drain, K)
    torch.cuda.nvtx.range_pop()
    clocks = sampler.stop(wall0, wall1)
    launches = _lib.launch_count() - l0
    state = drain()
    outs, det = state['outs'], state['det']
    gathered = state['pending'].result() if world > 1 else det
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs, gathered)
    value = world * per_gpu[main_mode] * K / (ms / 1e3)

    # ---- the other scaling mode in the same run (N > 1) -------------------------------------------------
    other_scaling = None
    if world > 1:
        om = 'strong' if main_mode == 'weak' else 'weak'
        s2, d2 = make_step(per_gpu[om])
        for i in range(3):
            s2(i)
        d2()
        ms2, _, _ = timed(s2, d2, K)
        other_scaling = {'scaling': om, 'global_batch': per_gpu[om] * world, 'images_per_gpu': per_gpu[om],
                         'value': world * per_gpu[om] * K / (ms2 / 1e3), 'unit': 'img/s', 'ms_per_step': ms2 / K, 'steps': K,
                         'tensor_frac_of_peak': world * per_gpu[om] * K / (ms2 / 1e3) * GFLOP_PER_IMG * 1e9 / (world * pk['tf_sustained'] * 1e12)}

    # ---- multi-GPU result parity: gathered records == one GPU running every rank's batch (SURVEY.md 8(e)) ----
    gather_parity = None
    if world > 1:
        last = (K - 1) & 1                                           # the input batch of the last timed step
        b = per_gpu[main_mode]
        if rank == 0:
            ok, ndet = True, 0
            for r in range(world):
                g = torch.Generator().manual_seed(seed_of(r))
                hb = [torch.randn(BATCH, 3, IMG, IMG, generator=g) for _ in range(2)][last][:b].to(dev)
                with torch.no_grad():
                    o = net(hb)
                d1 = detect_batched(o[0], o[1], o[2], anchors, cfg)
                for k in ('count', 'cls', 'anchor', 'score', 'box', 'coef'):
                    ok = ok and torch.equal(gathered[k][r * b:(r + 1) * b].view(torch.int32), d1[k].view(torch.int32))
                ndet += int(d1['count'].sum())
            gather_parity = {'gathered_equals_single_gpu_bit_exact': bool(ok), 'images': world * b, 'detections': ndet}
        dist.barrier()

    # ---- per-kernel profiling pass (separate from the timed region) ---------------------------------------
    eng.set_profiling(True)
    eng.profile()
    s3, d3 = make_step(BATCH)
    for i in range(3):
        s3(i)
    d3()
    torch.cuda.synchronize()
    prof = eng.profile()
    eng.set_profiling(False)

    # ---- Fast-NMS alone (decode + Fast-NMS + top-k), CUDA events -----------------------------------
    def time_detect(cls, box, coef, reps=10):
        for _ in range(3):
            detect_batched(cls, box, coef, anchors, cfg)
        return 1e3 * cuda_time(lambda i: detect_batched(cls, box, coef, anchors, cfg), reps) / cls.shape[0]      # us / img
    nms_us = {'network_output': time_detect(*outs[:3])}
    A = anchors.shape[0]
    for regime in ('stress', 'realistic'):
        c, b_, k_ = synth.head_outputs(7, A, 81, regime)
        rep = lambda a: torch.from_numpy(a).to(dev)[None].expand(BATCH, *a.shape).contiguous()
        nms_us[regime] = time_detect(rep(c), rep(b_), rep(k_))
    pp_bytes = A * 81 * 4 + A * 16 + A * 16 + 100 * (128 + 156)          # SURVEY.md 8(d): algorithmic bytes / img

    # ---- e2e ------------------------------------------------------------------------------------------
    D = cfg.max_detections
    rec_bytes = BATCH * (4 + D * (4 + 4 + 4 + 16 + 128))
    if world == 1:
        # the C ABI with host buffers: yb_net_submit_host / yb_net_collect_host (two batches in flight)
        p = _lib.DetectParams(cfg.nms_score_thre, cfg.nms_iou_thre, cfg.top_k, cfg.max_detections, cfg.num_classes, 32, 0, float(IMG))
        host_np = [h.numpy() for h in host]
        for i in range(2):
            eng.detect_host(host_np[i & 1], p)
        for i in range(3):                                                   # both pipeline slots: buffers, graphs, events
            a_ = eng.submit_host(host_np[0], p); b_ = eng.submit_host(host_np[1], p)
            eng.collect_host(a_); eng.collect_host(b_)
        t0 = time.perf_counter()
        pending = eng.submit_host(host_np[0], p)
        for i in range(1, K):
            nxt = eng.submit_host(host_np[i & 1], p)
            r = eng.collect_host(pending)
            pending = nxt
        r = eng.collect_host(pending)
        e2e_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        for i in range(K):
            r = eng.detect_host(host_np[i & 1], p)
        e2e_sync_s = time.perf_counter() - t0
        e2e = {'value': BATCH * K / e2e_s, 'unit': 'img/s', 'h2d_bytes_per_step': BATCH * 3 * IMG * IMG * 4, 'd2h_bytes_per_step': rec_bytes,
               'api': 'yb_net_submit_host / yb_net_collect_host (pinned host input, 2 batches in flight)',
               'synchronous_call_value': BATCH * K / e2e_sync_s}
    else:
        # the package's public calls with the collective inside: pinned host -> device -> forward -> post-process -> all-gather -> D2H
        b = per_gpu[main_mode]

        # software pipeline, as the single-GPU C entry points do it: the H2D copy of batch i+1 runs on a copy stream under the compute of
        # batch i, and the gathered records of batch i-1 are read back after batch i has been launched
        main_s, copy_s = torch.cuda.current_stream(), torch.cuda.Stream()
        xbuf = [torch.empty(b, 3, IMG, IMG, device=dev) for _ in range(2)]
        ev_up = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            with torch.cuda.stream(copy_s):
                copy_s.wait_event(ev_free[i & 1])                            # the forward that read this buffer last has finished with it
                xbuf[i & 1].copy_(host[i & 1][:b], non_blocking=True)
                ev_up[i & 1].record(copy_s)

        def launch(i):
            main_s.wait_event(ev_up[i & 1])
            with torch.no_grad():
                o = net(xbuf[i & 1])
            ev_free[i & 1].record(main_s)
            d_ = detect_batched(o[0], o[1], o[2], anchors, cfg)
            return ydist.gather_detections(d_, async_op=True)

        def e2e_run(n):
            for e in ev_free:
                e.record(main_s)
            upload(0)
            prev = None
            for i in range(n):
                if i + 1 < n:
                    upload(i + 1)
                g = launch(i)
                if prev is not None:
                    prev.wait().out.cpu()                                    # D2H of the gathered records (synchronises)
                prev = g
            return prev.wait().out.cpu()
        e2e_run(3)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e2e_run(K)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {'value': world * b * K / float(t.item()), 'unit': 'img/s', 'h2d_bytes_per_step': b * 3 * IMG * IMG * 4,
               'd2h_bytes_per_step': world * b * (4 + D * (4 + 4 + 4 + 16 + 128)),
               'api': 'pinned host tensor -> (copy stream) device -> Yolact.forward -> detect_batched -> dist.gather_detections (NCCL, async) -> D2H of the gathered records; '
                      'two batches in flight'}

    training = None
    if world > 1 and not os.environ.get('YB_BENCH_QUICK') and (ARCH, IMG) == ('res101', 550):
        del imgs
        torch.cuda.empty_cache()
        training = training_leg(ARCH, IMG, 2, 50, dev, rank, world)           # every rank takes part (DDP all-reduce)
        imgs = [h.to(dev) for h in host]
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return

    # ---- parity gate on the TIMED output (oracle on images 0 / mid / last of the last timed batch) ------------
    last = (K - 1) & 1
    b = per_gpu[main_mode]
    sd = ft.synth_state_dict(ARCH, seed=0)
    parity = {'images_checked': [], 'max_abs_err_vs_fp32_oracle': {n: 0.0 for n in ('cls', 'box', 'coef', 'proto')},
              'batch_output_equals_b1_runs_bitwise': True, 'fast_nms_indices_exact': True}
    for bi in sorted({0, b // 2 - 1 if b > 1 else 0, b - 1}):
        ref = [r.numpy() for r in ft.forward(host[last][bi:bi + 1], sd, ARCH)]
        with torch.no_grad():
            one = [o.clone() for o in net(imgs[last][bi:bi + 1])]
        for n, f, o, r in zip(('cls', 'box', 'coef', 'proto'), outs, one, ref):
            parity['batch_output_equals_b1_runs_bitwise'] &= bool(torch.equal(f[bi:bi + 1], o))
            parity['max_abs_err_vs_fp32_oracle'][n] = max(parity['max_abs_err_vs_fp32_oracle'][n], float(np.abs(f[bi:bi + 1].cpu().numpy() - r).max()))
        o = pp.nms(outs[0][bi].cpu().numpy(), outs[1][bi].cpu().numpy(), eng.anchors())
        d = int(det['count'][bi])
        parity['fast_nms_indices_exact'] &= bool(o is not None and d == len(o[0]) and np.array_equal(det['cls'][bi, :d].cpu().numpy(), o[0]) and
                                                 np.array_equal(det['anchor'][bi, :d].cpu().numpy(), o[3]))
        parity['images_checked'].append(bi)
    parity['gather'] = gather_parity

    # ---- roofline of the dominant kernel (from the profiling pass) ----
    tc = prof['conv_tc'] if prof['conv_tc']['launches'] else prof['conv_simt']
    dom = 'k_conv_tc' if prof['conv_tc']['launches'] else 'k_conv_simt'
    achieved = tc['flops'] / (tc['ms'] * 1e-3) / 1e12 if tc['ms'] else 0.0
    total_ms = sum(v['ms'] for v in prof.values())
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if os.path.exists(tpath) and dom == 'k_conv_tc' and (ARCH, IMG, BATCH) == ('res101', 550, 64):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get('dram_bytes_per_launch_avg'), tj.get('source')
    roofline = {'kernel': dom, 'bound': 'tensor', 'achieved': achieved, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s',
                'frac': achieved / pk['tf_sustained'], 'traffic': traffic, 'traffic_source': traffic_src,
                'alg_bytes_per_launch': tc['bytes'] / max(1, tc['launches']), 'peak_source': pk['src'] + ' (sustained bf16 cuBLAS)',
                'launches_per_step': tc['launches'] / max(1, tc['forwards']),
                'share_of_forward': tc['ms'] / total_ms if total_ms else None,
                'alg_flops_per_launch': tc['flops'] / max(1, tc['launches']),
                'avg_launch_ms': tc['ms'] / max(1, tc['launches']), 'timing': 'CUDA events per launch, separate profiling pass (3 steps)'}
    roofline_fused = None
    fz = prof.get('bneck_tc')
    if fz and fz['launches']:
        fa = fz['flops'] / (fz['ms'] * 1e-3) / 1e12
        ft_ = None
        if os.path.exists(tpath) and (ARCH, IMG, BATCH) == ('res101', 550, 64):
            ft_ = (json.load(open(tpath)).get('fused') or {}).get('dram_bytes_per_launch_avg')
        roofline_fused = {'kernel': 'k_bneck_tc (conv3 + residual + ReLU of a bottleneck chained into the next block\'s conv1 through shared memory)',
                          'bound': 'tensor', 'achieved': fa, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s', 'frac': fa / pk['tf_sustained'],
                          'traffic': ft_, 'alg_bytes_per_launch': fz['bytes'] / fz['launches'], 'alg_flops_per_launch': fz['flops'] / fz['launches'],
                          'launches_per_step': fz['launches'] / max(1, fz['forwards']), 'avg_launch_ms': fz['ms'] / fz['launches'],
                          'share_of_forward': fz['ms'] / total_ms if total_ms else None,
                          'hbm_gbs': fz['bytes'] / (fz['ms'] * 1e-3) / 1e9, 'hbm_frac': fz['bytes'] / (fz['ms'] * 1e-3) / 1e9 / pk['hbm']}
        both = (tc['flops'] + fz['flops']) / ((tc['ms'] + fz['ms']) * 1e-3) / 1e12
        roofline['tcgen05_kernels_together'] = {'achieved': both, 'frac': both / pk['tf_sustained'], 'share_of_forward': (tc['ms'] + fz['ms']) / total_ms}
    breakdown = {k: {'ms_per_step': v['ms'] / max(1, v['forwards']), 'launches_per_step': v['launches'] / max(1, v['forwards']),
                     'alg_tflops': (v['flops'] / (v['ms'] * 1e-3) / 1e12) if v['ms'] and v['flops'] else None,
                     'alg_gbs': (v['bytes'] / (v['ms'] * 1e-3) / 1e9) if v['ms'] else None}
                 for k, v in prof.items() if v['launches']}
    pp_roof = {'kernel': 'post-process (decode + Fast-NMS + top-k)', 'bound': 'hbm',
               'achieved': pp_bytes / (nms_us['stress'] * 1e-6) / 1e9, 'peak': pk['hbm'], 'unit': 'GB/s',
               'frac': pp_bytes / (nms_us['stress'] * 1e-6) / 1e9 / pk['hbm'], 'alg_bytes_per_img': pp_bytes, 'regime': 'stress'}

    line = {'metric': 'img/s', 'value': value, 'unit': 'img/s', 'n_gpus': world, 'steps': K, 'warmup': W, 'ms_per_step': ms / K,
            'higher_is_better': True, 'scaling': main_mode, 'vs_baseline': None,
            'dtype': {'fp16': 'f16', 'bf16': 'bf16', 'fp32': 'f32'}[args.precision], 'dtype_detail': 'tensor-core operands in that type, f32 accumulation; fp32 inputs and outputs',
            'data': 'synthetic',
            'config': {'workload': f'{ARCH}_coco {IMG}x{IMG} bs={per_gpu[main_mode]}/GPU eval forward + decode/Fast-NMS/top-k (BASELINE.json configs[2]), random-init weights',
                       'global_batch': per_gpu[main_mode] * world,
                       'parallelism': f'dp{world} (image shards, NCCL all-gather of detection records overlapped with the next forward)' if world > 1 else 'single GPU',
                       'l2_policy': 'inputs (232 MB/step, two alternating batches) larger than the 126 MB L2'},
            'tensor_frac_of_peak': value * GFLOP_PER_IMG * 1e9 / (world * pk['tf_sustained'] * 1e12),
            'gflop_per_img': GFLOP_PER_IMG,
            'fast_nms_us_per_img': nms_us, 'roofline': roofline, 'roofline_fused': roofline_fused, 'roofline_postprocess': pp_roof, 'kernel_breakdown': breakdown,
            'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks, 'parity': parity}
    if other_scaling:
        line[other_scaling['scaling'] + '_scaling'] = other_scaling
    if training:
        line['training'] = training

    if world == 1 and not os.environ.get('YB_BENCH_QUICK'):
        # the reference's own GPU path on this box, then the other BASELINE configurations, then the CPU baseline
        del imgs
        torch.cuda.empty_cache()
        line['gpu_eager_baseline'] = gpu_eager_baseline(ARCH, IMG, BATCH, dev, value)
        if (ARCH, IMG, BATCH) == ('res101', 550, 64):
            oc = []
            for a_, s_, b_ in (('res101', 544, 64), ('res50', 550, 32), ('res50', 544, 32), ('swin_tiny', 550, 32), ('swin_tiny', 544, 32)):
                try:
                    oc.append(measure_config(a_, s_, b_, args.precision, dev, 10, pk))
                except Exception as e:
                    oc.append({'workload': f'{a_}_coco {s_}x{s_} bs={b_}', 'error': repr(e)[:200]})
            line['other_configs'] = oc
            line['training'] = training_leg(ARCH, IMG, 2, 50, dev, 0, 1)
            try:
                line['mask_stage'] = mask_stage_leg(dev, pk)
            except Exception as e:
                line['mask_stage'] = {'error': repr(e)[:300]}
        cores = host_cores()
        cpu_v, cpu_s, cpu_nms_us, kind = cpu_reference_sample(ARCH, IMG, 4, 6, cores)
        line['cpu_baseline'] = {'value': cpu_v, 'unit': 'img/s', 'cores': cores, 'kind': kind,
                                'sample': f'6 reps x 4 images ({cpu_s:.1f} s): torch fp32 CPU forward + nms() per image', 'fast_nms_us_per_img': cpu_nms_us}
    else:
        line['cpu_baseline'] = None
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--precision', default=os.environ.get('YOLACT_B200_PRECISION', 'fp16'), choices=['fp16', 'bf16', 'fp32'])
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--eager-train-leg', action='store_true', help=argparse.SUPPRESS)     # internal: training_leg's eager baseline in a child process
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'], help='N > 1: images per GPU fixed at --batch (weak) or global batch fixed (strong); '
                    'the other mode is measured in the same run and reported beside it')
    ap.add_argument('--arch', default=ARCH, choices=['res101', 'res50', 'swin_tiny'], help='default: the BASELINE metric config')
    ap.add_argument('--img', type=int, default=IMG)
    ap.add_argument('--batch', type=int, default=BATCH, help='images per GPU (weak) / global batch (strong)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    ARCH, IMG, BATCH = args.arch, args.img, args.batch
    if args.eager_train_leg:
        import torch
        print(json.dumps(training_leg(args.arch, args.img, args.batch, args.steps, torch.device('cuda', 0), 0, 1, eager_only=True)))
        sys.exit(0)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
