"""GPU parity: the CUDA forward (through yb_net_* via the Yolact module) vs the oracle
(oracle/forward_torch.py on CPU, fp32) and the golden vectors minted from the reference.
Tolerances (absolute, on softmaxed class scores / box regressions / tanh coefficients / proto):
  fp32 mode  (CUDA cores)                       <= 1e-3 vs the fp32 oracle      (north_star)
  fp16 mode  (tcgen05, fp32 accumulate)         <= 1e-2 vs the fp32 oracle      (north_star's 16-bit bound)
  bf16 mode  (tcgen05, fp32 accumulate)         NOT an inference parity mode: an 8-bit-mantissa pipeline of ~100 layers sits at
             1-2e-2 from the fp32 oracle on box / coef / proto (oracle/forward_torch.forward_emulated shows the same deviation
             on the CPU, independent of these kernels), so it makes no 1e-2 claim and has no bench arm.  The kernels themselves
             are still pinned in that type (the training path computes in bf16): <= 4e-2 x scale vs the bf16-EMULATED oracle,
             i.e. "the kernels compute exactly the 16-bit pipeline"."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import synth, forward_torch as ft, postprocess_np as pp

pytestmark = pytest.mark.gpu

TOL = {'fp32': 1e-3, 'fp16': 1e-2}


def make_net(arch, S, precision, cuda, max_batch=0):
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.modules.yolact import Yolact
    cfg = make_config(arch + '_coco', S)
    cfg.precision = precision
    cfg.max_batch = max_batch
    net = Yolact(cfg)
    sd = ft.synth_state_dict(arch, seed=0)
    net.load_state_dict(sd, strict=True)
    return net.to(cuda).eval(), sd


def run(net, img, cuda):
    with torch.no_grad():
        out = net(torch.from_numpy(img).to(cuda))
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in out]


def rel_err(a, b):
    return float(np.abs(a - b).max()), float(np.abs(a - b).max() / (np.abs(b).max() + 1e-12))


@pytest.mark.parametrize('arch,S,B', [('res50', 64, 2), ('res101', 64, 1), ('res50', 128, 2), ('swin_tiny', 96, 2), ('swin_tiny', 224, 1)])
def test_forward_fp32_small_vs_oracle_golden_and_taps(cuda, arch, S, B):
    net, sd = make_net(arch, S, 'fp32', cuda)
    img = synth.image_batch(11, B, S)
    mine = run(net, img, cuda)
    ref, inter = ft.forward(torch.from_numpy(img), sd, arch, return_intermediates=True)
    ref = [r.numpy() for r in ref]
    for name, m, r in zip(('cls', 'box', 'coef', 'proto'), mine, ref):
        assert m.shape == r.shape, name
        assert np.abs(m - r).max() < TOL['fp32'], (name, rel_err(m, r))
    for tap in ('c3', 'c4', 'c5', 'p3', 'p4', 'p5', 'p6', 'p7'):
        t = net.engine(B).read_activation(tap, B).cpu().numpy()
        r = inter[tap].numpy()
        assert t.shape == r.shape, tap
        assert np.abs(t - r).max() < 1e-3 * max(1.0, np.abs(r).max()), (tap, rel_err(t, r))
    g = load_golden('forward.npz')
    key = f'{arch}_S{S}_B{B}'
    sub, psub = int(g[key + '/sub']), int(g[key + '/psub'])
    assert np.abs(mine[0][:, ::sub] - g[key + '/cls']).max() < TOL['fp32']
    assert np.abs(mine[1][:, ::sub] - g[key + '/box']).max() < TOL['fp32']
    assert np.abs(mine[2][:, ::sub] - g[key + '/coef']).max() < TOL['fp32']
    assert np.abs(mine[3][:, ::psub, ::psub] - g[key + '/proto']).max() < TOL['fp32']
    assert np.array_equal(net.engine(B).anchors(), pp.make_anchors(S))


@pytest.mark.parametrize('arch,S', [('res50', 400), ('res101', 544), ('res101', 550), ('swin_tiny', 550)])
def test_forward_fp32_full_size_vs_golden(cuda, arch, S):
    """BASELINE sizes incl. the odd 550/400 (reference needs the FPN patch there)."""
    net, sd = make_net(arch, S, 'fp32', cuda)
    img = synth.image_batch(11, 1, S)
    mine = run(net, img, cuda)
    g = load_golden('forward.npz')
    key = f'{arch}_S{S}_B1'
    sub, psub = int(g[key + '/sub']), int(g[key + '/psub'])
    assert mine[0].shape[1] == int(g[key + '/shapes'][0]) and mine[3].shape[1] == int(g[key + '/shapes'][1])
    for m, name in ((mine[0][:, ::sub], 'cls'), (mine[1][:, ::sub], 'box'), (mine[2][:, ::sub], 'coef'), (mine[3][:, ::psub, ::psub], 'proto')):
        assert np.abs(m - g[f'{key}/{name}']).max() < TOL['fp32'], (name, rel_err(m, g[f'{key}/{name}']))


def test_forward_fp32_batch_invariance_and_softmax(cuda):
    net, sd = make_net('res50', 96, 'fp32', cuda, max_batch=4)
    img = synth.image_batch(3, 3, 96)
    full = run(net, img, cuda)
    for b in range(3):
        one = run(net, img[b:b + 1], cuda)
        for f, o in zip(full, one):
            assert np.array_equal(f[b:b + 1], o)          # images are independent, bitwise
    assert np.allclose(full[0].sum(-1), 1.0, atol=1e-5)   # softmax rows
    assert np.abs(full[2]).max() <= 1.0 and full[3].min() >= 0.0


@pytest.mark.parametrize('arch,S,B', [('res50', 128, 2), ('res101', 256, 1), ('res101', 550, 1), ('swin_tiny', 96, 2), ('swin_tiny', 550, 1)])
@pytest.mark.parametrize('precision', ['fp16', 'bf16'])
def test_forward_16bit_vs_oracle(cuda, arch, S, B, precision):
    net, sd = make_net(arch, S, precision, cuda)
    img = synth.image_batch(11, B, S)
    mine = run(net, img, cuda)
    ref = [r.numpy() for r in ft.forward(torch.from_numpy(img), sd, arch)]
    act = torch.float16 if precision == 'fp16' else torch.bfloat16
    emu = [r.numpy() for r in ft.forward_emulated(torch.from_numpy(img), sd, arch, act=act)]
    for name, m, r, e in zip(('cls', 'box', 'coef', 'proto'), mine, ref, emu):
        err, err_emu = np.abs(m - r).max(), np.abs(m - e).max()
        print(f'{precision} {arch}@{S} {name}: max abs err vs fp32 oracle {err:.3e}, vs 16-bit emulation {err_emu:.3e} '
              f'(ref max {np.abs(r).max():.3f})')
        if precision == 'fp16':
            assert err < TOL['fp16'], (name, rel_err(m, r))
        # same rounding points as the emulation: only summation order / 1-ulp flips remain
        assert err_emu < (4e-2 if precision == 'bf16' else 4e-3) * max(1.0, np.abs(r).max()), (name, rel_err(m, e))


def test_forward_tc_vs_simt_same_precision(cuda, monkeypatch):
    """tcgen05 path == CUDA-core path in the same 16-bit precision (up to summation order)."""
    img = synth.image_batch(5, 2, 128)
    outs = {}
    for no_tc in ('', '1'):
        if no_tc:
            monkeypatch.setenv('YOLACT_B200_NO_TC', '1')
        else:
            monkeypatch.delenv('YOLACT_B200_NO_TC', raising=False)
        net, sd = make_net('res50', 128, 'fp16', cuda)
        outs[no_tc] = run(net, img, cuda)
    for a, b in zip(outs[''], outs['1']):
        assert np.abs(a - b).max() < 2e-3


def test_strict_load_and_error_paths(cuda):
    from yolact_minimal_b200 import _lib
    from yolact_minimal_b200.config import make_config
    from yolact_minimal_b200.modules.yolact import Yolact
    cfg = make_config('res50_coco', 64)
    net = Yolact(cfg)
    sd = ft.synth_state_dict('res50')
    bad = dict(sd); bad.pop('fpn.lat_layers.0.bias')
    with pytest.raises(RuntimeError):
        net.load_state_dict(bad, strict=True)
    net.load_state_dict(sd, strict=True)
    with pytest.raises(RuntimeError):
        net.eval()(torch.zeros(1, 3, 64, 64))                          # CPU input: no fallback
    net = net.to(cuda)
    with pytest.raises(ValueError):
        net.eval()(torch.zeros(1, 3, 96, 96, device=cuda))


def test_detect_host_end_to_end(cuda):
    """yb_net_detect_host (host buffers in, detections out) == forward + detect on device."""
    from yolact_minimal_b200 import _lib
    from yolact_minimal_b200.utils.output_utils import detect_batched
    net, sd = make_net('res50', 128, 'fp32', cuda, max_batch=2)
    img = synth.image_batch(21, 2, 128)
    with torch.no_grad():
        cls, box, coef, proto = net(torch.from_numpy(img).to(cuda))
    r = detect_batched(cls, box, coef, net.anchors, net.cfg)
    p = _lib.DetectParams(0.05, 0.5, 200, 100, 81, 32, 0, 128.0)
    h = net.engine(2).detect_host(img, p)
    for k in ('count', 'cls', 'anchor', 'score', 'box', 'coef'):
        assert np.array_equal(h[k], r[k].cpu().numpy()), k
    assert int(h['count'].min()) > 0
    # pipelined submit/collect: two batches in flight, results identical to the synchronous call
    eng = net.engine(2)
    img2 = np.ascontiguousarray(img[::-1])
    t0 = eng.submit_host(img, p)
    t1 = eng.submit_host(img2, p)
    with pytest.raises(_lib.YolactB200Error):
        eng.submit_host(img, p)                                        # a third submission must be refused, not queued
    a, b = eng.collect_host(t0), eng.collect_host(t1)
    h2 = eng.detect_host(img2, p)
    for k in ('count', 'cls', 'anchor', 'score', 'box', 'coef'):
        assert np.array_equal(a[k], h[k]) and np.array_equal(b[k], h2[k]), k
