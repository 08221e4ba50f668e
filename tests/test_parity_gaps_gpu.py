"""GPU parity holes named by the round-1 review, closed here:

  * the BENCHMARKED configuration (res101_coco 550x550, B=64, fp16 operands) is parity-checked itself:
    images 0 / 31 / 63 of the B=64 output vs the fp32 oracle (<= 1e-2, north_star's 16-bit bound) and
    bit-wise vs B=1 runs of the same images (persistent tile scheduling, CTA-pair tails and arena reuse
    only show their bugs at large B);
  * N-rank sharded inference: the NCCL-gathered detection records equal the single-GPU detections of the
    concatenated batch bit-for-bit (SURVEY.md 8(e)); needs >= 2 GPUs, skipped otherwise;
  * Fast-NMS decisions within a few ulps of IoU == threshold (SURVEY.md App. B; the kernel decides with a
    reciprocal estimate unless it is within 4e-6 of the threshold, postprocess.cu);
  * fp16 range: activations scaled toward 65504 stay within the relative 16-bit bound, and beyond it the
    stores saturate to +-65504 (cvt.satfinite) instead of producing inf / NaN.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth, forward_torch as ft, postprocess_np as pp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _net(arch, S, precision, cuda, max_batch):
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.modules.yolact import Yolact
    cfg = make_config(arch + '_coco', S)
    cfg.precision, cfg.max_batch = precision, max_batch
    net = Yolact(cfg)
    sd = ft.synth_state_dict(arch, seed=0)
    net.load_state_dict(sd, strict=True)
    return net.to(cuda).eval(), sd


def test_bench_config_b64_res101_550_fp16(cuda):
    B, S, arch = 64, 550, 'res101'
    net, sd = _net(arch, S, 'fp16', cuda, B)
    gen = torch.Generator().manual_seed(1234)                      # bench.py's rank-0 input batch
    img = torch.randn(B, 3, S, S, generator=gen)
    x = img.to(cuda)
    with torch.no_grad():
        full = [o.clone() for o in net(x)]
    torch.cuda.synchronize()
    assert all(torch.isfinite(o).all() for o in full)
    for b in (0, 31, 63):
        ref = [r.numpy() for r in ft.forward(img[b:b + 1], sd, arch)]
        with torch.no_grad():
            one = net(x[b:b + 1])
        for name, f, o, r in zip(('cls', 'box', 'coef', 'proto'), full, one, ref):
            assert torch.equal(f[b:b + 1], o), f'image {b} {name}: B=64 output differs bit-wise from the B=1 run'
            err = float(np.abs(f[b:b + 1].cpu().numpy() - r).max())
            assert err < 1e-2, f'image {b} {name}: max abs err {err} vs the fp32 oracle'
    # the timed step's second half: detections of the B=64 batch == detections of the B=1 runs, and index-exact vs the oracle
    from yolact_minimal_b200.utils.output_utils import detect_batched
    det = detect_batched(full[0], full[1], full[2], net.anchors, net.cfg)
    anchors = net.engine(B).anchors()
    for b in (0, 31, 63):
        o = pp.nms(full[0][b].cpu().numpy(), full[1][b].cpu().numpy(), anchors)
        d = int(det['count'][b])
        assert o is not None and d == len(o[0])
        assert np.array_equal(det['cls'][b, :d].cpu().numpy(), o[0]) and np.array_equal(det['anchor'][b, :d].cpu().numpy(), o[3])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_two_rank_gather_equals_single_gpu(tmp_path):
    out = tmp_path / 'gather.json'
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', '29621', os.path.join(ROOT, 'tests', 'dist_gpu_worker.py'), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    import json
    res = json.load(open(out))
    assert res['bit_exact'] and res['images'] == res['world'] * res['per_rank'] and res['detections'] > 0, res


def _pair_iou(a0, a1):
    """fp32 IoU of two (cx,cy,w,h) anchors after the reference's decode with zero regressions (output_utils.py:148-153)."""
    c = pp.decode(np.zeros((2, 4), np.float32), np.stack([a0, a1]).astype(np.float32))
    return pp.box_iou(c[None, 0:1], c[None, 1:2])[0, 0, 0]


def _near_threshold_case(thr):
    """Pairs of boxes whose fp32 IoU (box_utils.py:28-36 op order) sits within a few ulps of `thr`, on both sides: the second box
    of a pair is the first shifted in x by d ~ w (1-thr)/(1+thr) (IoU = (w-d)/(w+d)); the exact fp32 crossing is searched one
    ulp of cx at a time and the pair is then placed -3 .. +3 ulps from it.  One pair per (class, slot) so that pairs do not
    interact; box regressions are 0, so the anchors ARE the decoded boxes."""
    rng = np.random.RandomState(5)
    anchors, cls_rows, ious = [], [], []
    per_cls = 6
    up, down = np.float32(2.0), np.float32(-2.0)
    for c in range(80):
        for j in range(per_cls):
            w = np.float32(0.05 + 0.02 * rng.rand()); h = np.float32(0.05 + 0.03 * rng.rand())
            cx = np.float32(0.08 + 0.14 * j + 0.01 * rng.rand()); cy = np.float32(0.1 + 0.8 * rng.rand())
            a0 = np.asarray([cx, cy, w, h], np.float32)
            a1 = a0.copy()
            a1[0] = np.float32(cx + w * np.float32((1 - thr) / (1 + thr)))
            for _ in range(200):                                   # walk to the crossing: largest shift with IoU > thr
                if _pair_iou(a0, a1) > np.float32(thr):
                    a1[0] = np.nextafter(a1[0], up)
                else:
                    break
            for _ in range(200):
                if not _pair_iou(a0, a1) > np.float32(thr):
                    a1[0] = np.nextafter(a1[0], down)
                else:
                    break
            steps = (c * per_cls + j) % 7 - 3                      # > 0: IoU <= thr (kept), <= 0: IoU > thr (suppressed)
            for _ in range(abs(steps)):
                a1[0] = np.nextafter(a1[0], up if steps > 0 else down)
            ious.append(_pair_iou(a0, a1))
            for (a, sc) in ((a0, 0.9 - 0.001 * j), (a1, 0.6 - 0.001 * j)):
                anchors.append(a.copy())
                row = np.zeros(81, np.float32); row[c + 1] = sc; row[0] = 1 - sc
                cls_rows.append(row)
    anchors = np.asarray(anchors, np.float32)
    cls = np.asarray(cls_rows, np.float32)
    box = np.zeros((len(anchors), 4), np.float32)
    coef = synth.normal(9, 1, (len(anchors), 32)).astype(np.float32)
    return anchors, cls, box, coef, np.asarray(ious, np.float32)


@pytest.mark.parametrize('thr', [0.5, 0.3])
def test_fast_nms_iou_within_ulps_of_threshold(cuda, thr):
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.utils.output_utils import detect_batched
    anchors, cls, box, coef, iou = _near_threshold_case(thr)
    # the case must really sit on the threshold, on both sides
    assert np.abs(iou - np.float32(thr)).max() < 2e-5 and (np.abs(iou - np.float32(thr)) < 1e-6).sum() > 100
    assert (iou > np.float32(thr)).sum() > 100 and (iou <= np.float32(thr)).sum() > 100
    cfg = make_config('res101_coco', 544)
    cfg.nms_iou_thre, cfg.top_k, cfg.max_detections = thr, 200, 256
    # four images of 20 classes each (240 boxes <= max_det), so that EVERY keep/drop decision is visible in the output
    n = len(anchors)
    owner = (np.arange(n) // 12) // 20                              # 12 boxes per class
    cls_b = np.repeat(cls[None], 4, 0)
    for g in range(4):
        off = owner != g
        cls_b[g, off, 1:] = 0; cls_b[g, off, 0] = 1
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    r = detect_batched(t(cls_b), t(np.repeat(box[None], 4, 0)), t(np.repeat(coef[None], 4, 0)), t(anchors), cfg)
    kept = set()
    for g in range(4):
        o = pp.nms(cls_b[g], box, anchors, iou_thre=thr, top_k=200, max_det=256)
        d = int(r['count'][g])
        assert o is not None and d == len(o[0])                           # (zero-score entries of the other classes fill the tail up to max_det)
        assert np.array_equal(r['cls'][g, :d].cpu().numpy(), o[0])
        assert np.array_equal(r['anchor'][g, :d].cpu().numpy(), o[3])    # every keep/drop decision at the threshold agrees
        assert np.array_equal(r['score'][g, :d].cpu().numpy(), o[1])
        sc = r['score'][g, :d].cpu().numpy()
        assert (sc > 0).sum() < 256                                           # every real (non-zero score) survivor made the max_det cut
        kept |= {int(a) for a, s_ in zip(r['anchor'][g, :d].cpu().numpy(), sc) if s_ > 0}
    second = np.arange(1, n, 2)
    assert all(int(a) in kept for a in range(0, n, 2))              # the higher-scored box of every pair survives
    assert np.array_equal(np.asarray([int(a) in kept for a in second]), iou <= np.float32(thr))


def test_fp16_range_relative_error_and_saturation(cuda):
    """One tcgen05 conv layer (yb_conv2d) with trained-weight-like magnitudes: |y| up to ~3e4 keeps the 16-bit relative accuracy;
    |y| beyond 65504 saturates (finite), never inf / NaN."""
    import torch.nn.functional as F
    from test_conv_gpu import run_conv
    B, Cin, H, Cout, k = 2, 256, 35, 256, 3
    x = synth.normal(21, 1, (B, Cin, H, H)).astype(np.float32)
    w = (synth.normal(21, 2, (Cout, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = np.zeros(Cout, np.float32)
    q = lambda t: torch.from_numpy(t).to(cuda).half().double()
    for scale, wscale, saturates in ((6.0e3, 1.0, False), (1.0e4, 4.0, True)):      # inputs stay inside the fp16 range, outputs may not
        xs = (x * np.float32(scale)).astype(np.float32)
        ws = (w * np.float32(wscale)).astype(np.float32)
        y = run_conv(cuda, xs, ws, b, None, k, 1, 0, 2, 1).double()
        ref = F.conv2d(q(xs), q(ws), None, padding=1)
        assert torch.isfinite(y).all()
        if not saturates:
            assert float(ref.abs().max()) > 2.0e4                              # the case really is near the top of the range
            assert float((y - ref).abs().max() / ref.abs().max()) < 2e-3
        else:
            over = ref.abs() > 65504
            assert over.any()
            assert torch.equal(y[over], torch.sign(ref[over]) * 65504.0)       # clamped, not inf
            ok = ref.abs() < 6.0e4
            assert float(((y - ref)[ok]).abs().max() / 6.0e4) < 2e-3
