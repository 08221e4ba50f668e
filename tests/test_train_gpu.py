"""GPU: the native training path (SURVEY.md 8 rows a12 / f3) vs its checkers.

  * the fused loss kernels (yb_losses) on the reference-minted stage goldens (tests/golden/train_stages.npz): match() labels and
    matched indices bit-exact, SSD offsets, OHEM negatives, the four losses; their gradients w.r.t. the five network outputs vs
    torch autograd over oracle/train_torch.py (fp32);
  * the training engine (yb_train_*, through Yolact.forward in train mode + loss.backward()) vs the fp32 torch-autograd checker
    from identical parameters and inputs: losses (also vs the reference-minted tests/golden/train.npz), activations and activation
    gradients at named taps, EVERY parameter gradient, BatchNorm running statistics.  The engine computes the convolutions with
    bf16 tensor-core operands and fp32 accumulation, so the bounds are those of a 16-bit training pipeline (a few 1e-2 relative on
    gradients), not fp32 identity.
  * an SGD step moves the loss; DDP over NCCL (needs >= 2 GPUs)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden
import train_checks as tc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_native_losses_match_reference_stage_goldens(cuda):
    from yolact_minimal_b200.config import make_config
    g = load_golden('train_stages.npz')
    tg, mk, class_p, box_p, coef_p, proto_p, seg_p = tc.stage_inputs(g)
    cfg = make_config('res50_coco', tc.S_ST, mode='train', train_bs=tc.B_ST)
    r = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p)
    assert np.array_equal(r['labels'], g['labels'])                       # match(): bit-exact labels (pos / neutral / bg by IoU thresholds)
    assert np.array_equal(r['matched_idx'], g['matched_idx'])
    pos = g['labels'] > 0
    assert np.allclose(r['offsets'][pos], g['offsets'][pos], rtol=1e-5, atol=1e-6)
    assert (r['neg'].astype(bool) != g['ohem_neg']).sum() <= 2            # OHEM set (expf / logf may flip an exact boundary tie)
    assert np.allclose(r['losses'], [g['loss_c'], g['loss_b'], g['loss_m'], g['loss_s']], rtol=2e-5)
    ref_l, ref_g = tc.torch_losses_and_grads(cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p)
    for k in ('d_cls', 'd_box', 'd_coef', 'd_proto', 'd_seg'):
        assert tc.rel(r[k], ref_g[k]) < 1e-5, (k, tc.rel(r[k], ref_g[k]))
    # loss weights on the gradient side (what autograd hands to backward), and losses-only mode
    w = (0.5, 2.0, 0.25, 3.0)
    r2 = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p, grad_scale=w)
    _, ref_g2 = tc.torch_losses_and_grads(cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p, grad_scale=w)
    for k in ('d_cls', 'd_box', 'd_coef', 'd_proto', 'd_seg'):
        assert tc.rel(r2[k], ref_g2[k]) < 1e-5, k
    r3 = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p, grads=False)
    assert np.array_equal(r3['losses'], r['losses'])


def test_native_losses_random_subset_when_many_positives(cuda):
    """More positives than masks_to_train: a random subset of exactly masks_to_train masks, re-weighted by n_all / n (yolact.py:261-286)."""
    from yolact_minimal_b200.config import make_config
    g = load_golden('train_stages.npz')
    tg, mk, class_p, box_p, coef_p, proto_p, seg_p = tc.stage_inputs(g)
    cfg = make_config('res50_coco', tc.S_ST, mode='train', train_bs=tc.B_ST)
    full = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p)
    npos = (g['labels'] > 0).sum(1)
    cfg.masks_to_train = int(npos.max()) - 2
    a = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p, seed=1)
    b = tc.run_native_losses(cuda, cfg, g['anchors'], tg, mk, class_p, box_p, coef_p, proto_p, seg_p, seed=2)
    assert np.array_equal(a['losses'][[0, 1, 3]], full['losses'][[0, 1, 3]])                 # only the mask loss samples
    assert a['losses'][2] != full['losses'][2] and a['losses'][2] != b['losses'][2]          # a subset, and a different one per seed
    assert abs(a['losses'][2] / full['losses'][2] - 1) < 0.5                                 # re-weighted: same scale
    nz = lambda r: (np.abs(r['d_coef']).sum(-1) > 0).sum(1)
    assert (nz(a) <= cfg.masks_to_train).all() and nz(a).max() == cfg.masks_to_train         # exactly masks_to_train masks get a gradient


@pytest.mark.parametrize('arch,S,B,precision', [('res50', 128, 2, 'bf16'), ('res50', 128, 2, 'fp16'), ('res101', 96, 2, 'bf16')])
def test_training_engine_backward_at_its_own_activations(cuda, arch, S, B, precision):
    """The strict check of the BACKWARD pass: the torch-autograd checker is evaluated AT the engine's stored activations (every conv
    output, BN / ReLU output, FPN level ...: identical ReLU masks and batch statistics), so that what is compared is the engine's
    gradient arithmetic -- dgrad convolutions, weight-gradient GEMMs, BatchNorm / max-pool / bilinear / stride-2 backward, bias sums,
    loss gradients -- against fp32 autograd.  Measured: median relative error of a parameter gradient 1.2e-2 (bf16) / 1.2e-3 (fp16:
    8x more mantissa, 8x less error -- rounding, not logic), worst parameter 7e-2 / 7e-3."""
    o = tc.engine_vs_checker(arch, S, B, cuda, precision, mode='subst')
    assert o['substituted'] > 100
    assert np.allclose(o['losses'], o['ref_losses'], rtol=1e-4), (o['losses'], o['ref_losses'])      # same activations -> same losses
    rels = o['grads']
    assert not any(np.isnan(v[0]) for v in rels.values()), [n for n, v in rels.items() if np.isnan(v[0])]
    worst = sorted(rels.items(), key=lambda kv: -kv[1][0])[:5]
    print(f'{arch}@{S} {precision}: worst parameter gradients (rel err, cosine, |ref|):', worst, 'launches/step', o['launches'])
    tol_max, tol_med = (0.15, 3e-2) if precision == 'bf16' else (2e-2, 4e-3)
    for n, (r, c, nr) in rels.items():
        assert r < tol_max and c > 0.99, (n, r, c, nr)                                             # EVERY parameter of the network
    assert float(np.median([v[0] for v in rels.values()])) < tol_med
    for name, e in o['gact'].items():
        if name not in ('c3', 'c4', 'c5'):                     # (the checker's c3..c5 taps sit on the FPN branch only in this mode)
            assert e < (6e-2 if precision == 'bf16' else 1e-2), ('activation gradient', name, e)


@pytest.mark.parametrize('arch,S,B', [('res50', 128, 2), ('res101', 96, 2)])
def test_training_engine_vs_fp32_reference(cuda, arch, S, B):
    """How far the 16-bit training step is from the reference's fp32 arithmetic: losses (also vs the reference-minted
    tests/golden/train.npz), forward activations, BatchNorm statistics, gradient direction.  Gradients of a 16-bit forward differ from
    fp32 ones mostly through ReLU masks that flip where an activation is within rounding noise of zero (relative L2 error ~ sqrt of the
    flipped fraction, 0.2-0.5 with bf16 activations at this depth) -- inherent to any mixed-precision training step; the backward
    arithmetic itself is pinned by the test above."""
    o = tc.engine_vs_checker(arch, S, B, cuda, 'bf16', mode='fp32')
    g = load_golden('train.npz')
    gold = g[f'{arch}_S{S}_B{B}/losses']
    print('losses', o['losses'], 'checker', o['ref_losses'], 'reference golden', gold.tolist())
    assert np.allclose(o['ref_losses'], gold, rtol=2e-3)                                     # the checker is the reference
    assert np.allclose(o['losses'], gold, rtol=5e-2), (o['losses'], gold.tolist())           # bf16 forward: losses within 5 %
    for name in ('stem.z', 'pool', 'c2'):
        assert o['act'][name] < 2e-2, (name, o['act'][name])
    assert all(isinstance(e, float) and e < 0.25 for e in o['act'].values()), o['act']
    coss = np.asarray([v[1] for v in o['grads'].values()])
    assert not np.isnan(coss).any() and float(np.median(coss)) > (0.85 if S >= 128 else 0.4), float(np.median(coss))
    for n, e in o['bn'].items():
        if n.endswith('num_batches_tracked'):
            assert e == 0, n
        else:
            assert e < 6e-2, (n, e)


def test_sgd_steps_reduce_the_loss(cuda):
    from oracle import synth
    net = tc.make_train_net('res50', 128, 2, cuda)
    opt = torch.optim.SGD(net.parameters(), lr=3e-4, momentum=0.9, weight_decay=5e-4)
    img = torch.from_numpy(synth.image_batch(11, 2, 128)).to(cuda)
    tg, mk = synth.train_targets(5, 2, 128)
    tgt = [torch.from_numpy(t).to(cuda) for t in tg]
    mks = [torch.from_numpy(m).to(cuda) for m in mk]
    hist = []
    for _ in range(8):
        losses = net(img, tgt, mks)
        total = sum(losses)
        opt.zero_grad()
        total.backward()
        opt.step()
        hist.append(float(total.detach()))
    assert all(np.isfinite(hist)) and min(hist[4:]) < 0.6 * hist[0], hist        # (measured at lr 1e-3: 147 -> 118 -> 80 -> 62 -> 31 -> 23)
    # the engine keeps serving: eval forward after training uses the updated parameters and running statistics
    net.eval()
    with torch.no_grad():
        out = net(img)
    assert all(torch.isfinite(t).all() for t in out)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs >= 2 GPUs')
def test_ddp_training_two_ranks_nccl(tmp_path):
    out = tmp_path / 'ddp.json'
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', '29631', os.path.join(ROOT, 'tests', 'ddp_train_worker.py'), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    import json
    res = json.load(open(out))
    assert res['weights_equal_across_ranks'] and res['finite'] and res['loss_last'] < res['loss_first'], res
