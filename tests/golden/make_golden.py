#!/usr/bin/env python
"""Golden-vector generator (TEST INFRASTRUCTURE).  Needs a checkout of the reference, named by
$YOLACT_REFERENCE; the fixtures it writes next to this file are committed, so the tests never
need the reference itself.

  YOLACT_REFERENCE=<checkout> python tests/golden/make_golden.py            # regenerate every fixture

It imports the UNMODIFIED reference modules (modules.yolact.Yolact, utils.output_utils.nms /
after_nms, utils.box_utils.make_anchors) and, for the traditional-NMS path, a copy of
cython_nms.pyx built into the git-ignored oracle/_ref/ with the 2-token numpy-2 patch
(np.int_t -> np.int64_t, np.int -> np.int64; SURVEY.md App. E.2).  Inputs come from
oracle/synth.py so the tests can rebuild them bit-for-bit.
"""
import os
import subprocess
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ['YOLACT_REFERENCE']
REFBUILD = os.path.join(ROOT, 'oracle', '_ref')
sys.path.insert(0, ROOT)

from oracle import synth, postprocess_np as pp, forward_torch as ft  # noqa: E402


def build_cython_nms():
    os.makedirs(REFBUILD, exist_ok=True)
    src = open(os.path.join(REF, 'cython_nms.pyx')).read()
    src = src.replace('np.int_t', 'np.int64_t').replace('dtype=np.int)', 'dtype=np.int64)')
    open(os.path.join(REFBUILD, 'cython_nms.pyx'), 'w').write(src)
    open(os.path.join(REFBUILD, 'setup.py'), 'w').write(
        "from distutils.core import setup\nfrom Cython.Build import cythonize\nimport numpy\n"
        "setup(ext_modules=cythonize('cython_nms.pyx', language_level=3), include_dirs=[numpy.get_include()])\n")
    subprocess.check_call([sys.executable, 'setup.py', '-q', 'build_ext', '--inplace'], cwd=REFBUILD)


def import_reference():
    scratch = '/tmp/yolact_ref_cwd'
    os.makedirs(scratch, exist_ok=True)
    os.chdir(scratch)                      # config.py mkdirs in CWD on import (config.py:6-15)
    sys.path.insert(0, REFBUILD)
    sys.path.insert(0, REF)
    import cython_nms  # noqa: F401  (the patched build)
    import config as rcfg
    from modules import yolact as ryolact
    from utils import output_utils as rout
    from utils import box_utils as rbox
    return rcfg, ryolact, rout, rbox


def ref_cfg(rcfg, name, img_size, mode='detect', traditional=False):
    ns = types.SimpleNamespace(cfg=name, img_size=544, weight=None, traditional_nms=traditional,
                               visual_thre=0.0, save_lincomb=False, no_crop=False, image=None, video=None,
                               hide_mask=False, hide_bbox=False, hide_score=False, cutout=False,
                               real_time=False, val_num=-1, coco_api=False)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        cfg = rcfg.get_config(ns, mode)
    cfg.img_size = img_size                                   # bypass config.py:75 for 550/400
    cfg.scales = [int(img_size / 544 * a) for a in (24, 48, 96, 192, 384)]
    return cfg


# ----------------------------------------------------------------------------- post-process
def nms_cases():
    """(name, img_size for anchors, regime, seed, mutation)"""
    cases = []
    for S in (128, 256):
        for regime in ('stress', 'realistic', 'sparse'):
            for seed in (1, 2):
                cases.append((f'{regime}_S{S}_s{seed}', S, regime, seed, None))
    cases.append(('stress_S544_s1', 544, 'stress', 1, None))
    cases.append(('realistic_S544_s1', 544, 'realistic', 1, None))
    cases.append(('realistic_S550_s3', 550, 'realistic', 3, None))
    for mut in ('dup_boxes', 'zero_area', 'few', 'none', 'one'):
        cases.append((f'adv_{mut}', 128, 'stress', 7, mut))
    return cases


def build_nms_inputs(S, regime, seed, mut):
    anchors = pp.make_anchors(S)
    A = anchors.shape[0]
    cls, box, coef = synth.head_outputs(seed, A, 81, regime)
    if mut == 'dup_boxes':                 # identical boxes+anchors -> IoU exactly 1 / NaN-free dup handling
        box[1::2] = box[0::2][:box[1::2].shape[0]]
        anchors = anchors.copy(); anchors[1::2] = anchors[0::2][:anchors[1::2].shape[0]]
    elif mut == 'zero_area':               # push boxes outside [0,1] -> clip gives zero-area -> 0/0 = NaN IoU
        box[:, :2] += 40.0
    elif mut in ('few', 'none', 'one'):    # n < top_k, n == 0, n == 1
        keep_n = {'few': 37, 'none': 0, 'one': 1}[mut]
        cls[:] = 0.0; cls[:, 0] = 1.0
        src, _, _ = synth.head_outputs(seed + 1, A, 81, 'stress')
        rows = (np.arange(keep_n) * 23 + 5) % A
        cls[rows] = src[rows]
    return anchors, cls, box, coef


def gen_postprocess(rcfg, rout):
    out = {}
    cfg = ref_cfg(rcfg, 'res101_coco', 544)
    for name, S, regime, seed, mut in nms_cases():
        anchors, cls, box, coef = build_nms_inputs(S, regime, seed, mut)
        A = anchors.shape[0]
        idxcoef = torch.arange(A, dtype=torch.float32).view(1, A, 1).repeat(1, 1, 2)   # App. E.4
        proto = torch.zeros(1, 4, 4, 2)
        for trad in (False, True):
            if trad and (S > 256 or regime == 'stress' and S > 128):
                continue                                       # cython path is O(n^2) python-free but slow
            cfg.traditional_nms = trad
            cfg.img_size = S
            try:
                r = rout.nms(torch.from_numpy(cls)[None], torch.from_numpy(box)[None], idxcoef, proto,
                             torch.from_numpy(anchors), cfg)
            except RuntimeError as e:                         # torch.cat([]) in traditional_nms with no survivors
                r = (None,) * 5
            key = f'{name}/{"trad" if trad else "fast"}'
            if r[0] is None:
                out[key + '/count'] = np.int64(0)
                continue
            ids, scores, boxes, ic, _ = r
            out[key + '/count'] = np.int64(ids.numel())
            out[key + '/class'] = ids.numpy().astype(np.int64)
            out[key + '/anchor'] = ic[:, 0].long().numpy()
            out[key + '/score'] = scores.numpy()
            out[key + '/box'] = boxes.numpy()
            # oracle vs reference, here and now
            o = pp.nms(cls, box, anchors, traditional=trad, img_size=S)
            assert o is not None and np.array_equal(o[0], out[key + '/class']), key
            assert np.array_equal(o[3], out[key + '/anchor']), key
            assert np.array_equal(o[1], out[key + '/score']), key
            assert np.allclose(o[2], out[key + '/box'], rtol=0, atol=2.4e-7), key
            print(f'  nms {key}: {ids.numel()} dets, oracle == reference')
    np.savez_compressed(os.path.join(HERE, 'postprocess.npz'), **out)


def gen_hard_nms():
    import cython_nms
    out = {}
    for seed, n in ((1, 1), (2, 17), (3, 300), (4, 1500)):
        xy = synth.uniform(seed, 11, (n, 2)) * 400
        wh = synth.uniform(seed, 12, (n, 2)) * 120 + 1
        sc = synth.uniform(seed, 13, (n, 1))
        dets = np.concatenate([xy, xy + wh, sc], 1).astype(np.float32)
        for thr in (0.3, 0.5):
            keep = cython_nms.nms(dets, np.float32(thr))
            assert np.array_equal(keep, pp.hard_nms(dets, thr))
            out[f's{seed}_n{n}_t{thr}'] = keep.astype(np.int64)
    np.savez_compressed(os.path.join(HERE, 'hard_nms.npz'), **out)
    print('  hard_nms goldens written, oracle == reference')


def gen_after_nms(rcfg, rout):
    out = {}
    for name, S, h, w, seed in (('S128_80x120', 128, 80, 120, 5), ('S128_97x64', 128, 97, 64, 6),
                                ('S256_60x60', 256, 60, 60, 7)):
        anchors = pp.make_anchors(S)
        cls, box, coef = synth.head_outputs(seed, anchors.shape[0], 81, 'realistic')
        proto = synth.proto(seed, S // 4)
        r = pp.nms(cls, box, anchors)
        ids, scores, boxes, aidx = r
        coefs = coef[aidx]
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
        rid, rsc, rbx, rmask = rout.after_nms(t(ids), t(scores), t(boxes.copy()), t(coefs), t(proto), h, w)
        o = pp.after_nms(ids, scores, boxes, coefs, proto, h, w)
        mism = float((o[3] != rmask.numpy()).mean())
        assert np.array_equal(o[2], rbx.numpy()), name
        assert mism < 2e-4, (name, mism)
        out[name + '/boxes_px'] = rbx.numpy().astype(np.int32)
        out[name + '/mask_bits'] = np.packbits(rmask.numpy().astype(np.uint8))
        out[name + '/mask_shape'] = np.asarray(rmask.shape, dtype=np.int64)
        print(f'  after_nms {name}: masks {tuple(rmask.shape)}, oracle mismatch {mism:.2e}')
    np.savez_compressed(os.path.join(HERE, 'after_nms.npz'), **out)


def gen_numpy_twins(rcfg, rout):
    """The ONNX / TRT callers' numpy post-process (utils/output_utils.py:46-81,:166-197,:236-273), run by the reference itself:
    nms_numpy (no clip of the decoded boxes) and after_nms_numpy (cv2 resize, boolean masks)."""
    out = {}
    cfg = ref_cfg(rcfg, 'res101_coco', 544)
    cfg.traditional_nms = False
    for name, S, regime, seed, h, w in (('stress_S128', 128, 'stress', 1, 80, 120), ('realistic_S256', 256, 'realistic', 2, 97, 64),
                                        ('wild_S128', 128, 'stress', 4, 60, 60)):
        anchors = pp.make_anchors(S)
        cls, box, coef = synth.head_outputs(seed, anchors.shape[0], 81, regime)
        if name.startswith('wild'):
            box = (box * 3).astype(np.float32)                   # boxes far outside [0,1]: the missing clip matters
        proto = synth.proto(seed, S // 4)
        r = rout.nms_numpy(cls[None], box[None], coef[None], proto[None], anchors.reshape(-1).tolist(), cfg)
        ids, scores, boxes, coefs, _ = r
        out[name + '/class'] = np.asarray(ids, np.int64); out[name + '/score'] = np.asarray(scores, np.float32)
        out[name + '/box'] = np.asarray(boxes, np.float64); out[name + '/coef'] = np.asarray(coefs, np.float32)
        o = pp.nms_numpy(cls, box, anchors)
        assert np.array_equal(o[0], out[name + '/class']) and np.array_equal(o[1], out[name + '/score']), name
        assert np.allclose(o[2], out[name + '/box'], rtol=0, atol=1e-5), name
        rid, rsc, rbx, rmask = rout.after_nms_numpy(ids, scores, np.asarray(boxes, np.float32).copy(), coefs, proto, h, w, cfg)
        out[name + '/boxes_px'] = rbx.astype(np.int32)
        out[name + '/mask_bits'] = np.packbits(rmask.astype(np.uint8)); out[name + '/mask_shape'] = np.asarray(rmask.shape, np.int64)
        print(f'  numpy twins {name}: {len(ids)} dets, box range [{float(np.min(boxes)):.2f}, {float(np.max(boxes)):.2f}], masks {rmask.shape}, oracle == reference')
    np.savez_compressed(os.path.join(HERE, 'numpy_twins.npz'), **out)


def gen_anchors(rcfg, ryolact):
    out = {}
    for S in (128, 384, 400, 544, 550, 576):
        cfg = ref_cfg(rcfg, 'res50_coco', S)
        ref = []
        import math
        from utils.box_utils import make_anchors
        for i, size in enumerate([math.ceil(S / s) for s in (8, 16, 32, 64, 128)]):
            ref += make_anchors(cfg, size, size, cfg.scales[i])
        ref = torch.tensor(ref).reshape(-1, 4).numpy()
        mine = pp.make_anchors(S)
        assert np.array_equal(ref, mine), S
        out[f'S{S}/count'] = np.int64(ref.shape[0])
        out[f'S{S}/rows'] = ref[:: max(1, ref.shape[0] // 64)]
        out[f'S{S}/sum64'] = ref.astype(np.float64).sum(0)
    np.savez_compressed(os.path.join(HERE, 'anchors.npz'), **out)
    print('  anchors goldens written, oracle == reference')


# ----------------------------------------------------------------------------- forward
def patch_fpn(ryolact):
    """SURVEY.md App. E.3: interpolate-to-lateral-size so 550/400 run."""
    import torch.nn.functional as F

    def forward(self, outs):
        p5_1 = self.lat_layers[2](outs[2])
        l4 = self.lat_layers[1](outs[1])
        p4_1 = l4 + F.interpolate(p5_1, size=l4.shape[2:], mode='bilinear', align_corners=False)
        l3 = self.lat_layers[0](outs[0])
        p3_1 = l3 + F.interpolate(p4_1, size=l3.shape[2:], mode='bilinear', align_corners=False)
        p5 = self.pred_layers[2](p5_1); p4 = self.pred_layers[1](p4_1); p3 = self.pred_layers[0](p3_1)
        p6 = self.downsample_layers[0](p5); p7 = self.downsample_layers[1](p6)
        return p3, p4, p5, p6, p7
    orig = ryolact.FPN.forward
    ryolact.FPN.forward = forward
    return orig


def gen_forward(rcfg, ryolact):
    # strides keep the fixture small: about 40 anchor rows (every aspect ratio: sub is not a multiple of 3) and a 6 x 6
    # grid of proto pixels per image
    out = {}
    cases = [('res50', 64, 2, 7, 3, False), ('res101', 64, 1, 7, 3, False), ('res50', 128, 2, 25, 5, False),
             ('res50', 400, 1, 250, 17, True), ('res101', 544, 1, 463, 23, False), ('res101', 550, 1, 481, 23, True),
             ('swin_tiny', 96, 2, 14, 4, False), ('swin_tiny', 224, 1, 79, 9, False), ('swin_tiny', 550, 1, 481, 23, True)]
    for arch, S, B, sub, psub, need_patch in cases:
        cfg = ref_cfg(rcfg, arch + '_coco', S)
        sd = ft.synth_state_dict(arch, seed=0)
        net = ryolact.Yolact(cfg)
        net.load_state_dict(sd, strict=True)         # also proves state-dict key compatibility
        net.eval()
        img = torch.from_numpy(synth.image_batch(11, B, S))
        orig = patch_fpn(ryolact) if need_patch else None
        with torch.no_grad():
            ref = net(img)
        if orig is not None:
            ryolact.FPN.forward = orig
        mine = ft.forward(img, sd, arch)
        errs = [float((a - b).abs().max()) for a, b in zip(ref, mine)]
        assert max(errs) < (2e-5 if arch == 'swin_tiny' else 2e-6), (arch, S, errs)
        key = f'{arch}_S{S}_B{B}'
        cls, box, coef, proto = [t.numpy() for t in ref]
        out[key + '/sub'] = np.int64(sub)
        out[key + '/psub'] = np.int64(psub)
        out[key + '/cls'] = cls[:, ::sub]
        out[key + '/box'] = box[:, ::sub]
        out[key + '/coef'] = coef[:, ::sub]
        out[key + '/proto'] = proto[:, ::psub, ::psub]
        out[key + '/shapes'] = np.asarray([cls.shape[1], proto.shape[1]], dtype=np.int64)
        print(f'  forward {key}: A={cls.shape[1]} P={proto.shape[1]} oracle-vs-reference max err {max(errs):.2e}')
    np.savez_compressed(os.path.join(HERE, 'forward.npz'), **out)


def gen_val_aug():
    """Pre-process goldens from the reference's own val_aug (cv2)."""
    sys.path.insert(0, REF)
    from utils.augmentations import val_aug as ref_val_aug
    out = {}
    for name, h, w, S, seed in (('97x64_S96', 97, 64, 96, 1), ('120x160_S128', 120, 160, 128, 2), ('200x200_S64', 200, 200, 64, 3),
                                ('375x500_S550', 375, 500, 550, 4)):
        img = (synth.uniform(seed, 21, (h, w, 3)) * 256).astype(np.uint8)
        ref = ref_val_aug(img, S).astype(np.float32)
        mine = pp.val_aug(img, S)
        err = float(np.abs(ref - mine).max())
        assert err < 2e-4, (name, err)      # cv2's (IPP) float resize differs from the textbook formula by ~1e-4
        sub = 1 if S <= 128 else 11
        out[name + '/sub'] = np.int64(sub)
        out[name + '/out'] = ref[:, ::sub, ::sub]
        out[name + '/sum'] = ref.astype(np.float64).sum(axis=(1, 2))
        print(f'  val_aug {name}: oracle-vs-reference max err {err:.2e}')
    np.savez_compressed(os.path.join(HERE, 'val_aug.npz'), **out)


def gen_train(rcfg, ryolact):
    """Training-branch goldens: the reference's 4 losses, a few gradient norms and BN statistics after
    one forward/backward on CPU (train mode, synthetic targets)."""
    import contextlib, io, types
    out = {}
    for arch, S, B in (('res50', 128, 2), ('res101', 96, 2)):
        ns = types.SimpleNamespace(cfg=arch + '_coco', img_size=S, weight=None, traditional_nms=False, resume=None, train_bs=B,
                                   val_interval=-1, val_num=-1, coco_api=False)
        with contextlib.redirect_stdout(io.StringIO()):
            cfg = rcfg.get_config(ns, 'train')
        sd = ft.synth_state_dict(arch, seed=0, train=True)
        net = ryolact.Yolact(cfg)
        net.load_state_dict(sd, strict=True)
        net.train()
        img = torch.from_numpy(synth.image_batch(11, B, S))
        tg, mk = synth.train_targets(5, B, S)
        losses = net(img, [torch.from_numpy(t) for t in tg], [torch.from_numpy(m) for m in mk])
        sum(losses).backward()
        key = f'{arch}_S{S}_B{B}'
        out[key + '/losses'] = np.asarray([float(l) for l in losses], dtype=np.float64)
        named = dict(net.named_parameters())
        for pn in ('backbone.conv1.weight', 'backbone.layers.2.0.conv2.weight', 'fpn.lat_layers.0.bias', 'proto_net.proto2.2.weight',
                   'prediction_layers.conf_layer.weight', 'semantic_seg_conv.weight'):
            out[f'{key}/grad/{pn}'] = np.float64(named[pn].grad.double().norm())
        out[key + '/bn1_mean'] = net.backbone.bn1.running_mean.detach().numpy().copy()
        print(f'  train {key}: losses {[round(float(l), 5) for l in losses]}')
    np.savez_compressed(os.path.join(HERE, 'train.npz'), **out)


def gen_train_stages(rcfg, ryolact, rbox):
    """Stage-by-stage goldens of the training branch (oracle/train_np.py): the reference's match(), the OHEM selection
    recovered from category_loss's internals, each of the four losses on synthetic head outputs, and mask_iou."""
    import contextlib, io, types
    from oracle import train_np as tn
    out = {}
    S, B = 128, 3
    ns = types.SimpleNamespace(cfg='res50_coco', img_size=S, weight=None, traditional_nms=False, resume=None, train_bs=B,
                               val_interval=-1, val_num=-1, coco_api=False)
    with contextlib.redirect_stdout(io.StringIO()):
        cfg = rcfg.get_config(ns, 'train')
    net = ryolact.Yolact(cfg)
    anchors = torch.tensor(net.anchors).reshape(-1, 4)
    A, P = anchors.shape[0], S // 4
    tg, mk = synth.train_targets(9, B, S, n=4)
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
    class_p = f32(synth.normal(21, 1, (B, A, cfg.num_classes)) * 2)
    box_p = f32(synth.normal(21, 2, (B, A, 4)) * 0.5)
    coef_p = torch.tanh(f32(synth.normal(21, 3, (B, A, 32))))
    proto_p = torch.relu(f32(synth.normal(21, 4, (B, P, P, 32))))
    seg_p = f32(synth.normal(21, 5, (B, cfg.num_classes - 1, S // 8, S // 8)))
    offs, labs, mgt, midx = [], [], [], []
    for i in range(B):
        t = torch.from_numpy(tg[i])
        o, c, g, m = rbox.match(cfg, t[:, :4], anchors, t[:, 4].long())
        offs.append(o); labs.append(c); mgt.append(g); midx.append(m)
    offs, labs, mgt, midx = torch.stack(offs), torch.stack(labs), torch.stack(mgt), torch.stack(midx)
    pos = labs > 0
    out['anchors'] = anchors.numpy(); out['offsets'] = offs.numpy(); out['labels'] = labs.numpy()
    out['matched'] = mgt.numpy(); out['matched_idx'] = midx.numpy()
    out['loss_c'] = np.float64(net.category_loss(class_p, labs, pos))
    out['loss_b'] = np.float64(net.box_loss(box_p, offs, pos))
    out['loss_m'] = np.float64(net.lincomb_mask_loss(pos, midx, coef_p, proto_p, [torch.from_numpy(m) for m in mk], mgt))
    out['loss_s'] = np.float64(net.semantic_seg_loss(seg_p, [torch.from_numpy(m) for m in mk], [torch.from_numpy(t[:, 4]).long() for t in tg]))
    # the OHEM negatives, recomputed exactly as category_loss does (modules/yolact.py:205-225)
    bc = class_p.reshape(-1, cfg.num_classes); mx = bc.max()
    mark = (torch.log(torch.sum(torch.exp(bc - mx), 1)) + mx - bc[:, 0]).reshape(B, -1)
    mark[pos] = 0; mark[labs < 0] = 0
    _, idx = mark.sort(1, descending=True); _, rank = idx.sort(1)
    neg = rank < torch.clamp(3 * pos.long().sum(1, keepdim=True), max=A - 1)
    neg[pos] = 0; neg[labs < 0] = 0
    out['ohem_neg'] = neg.numpy()
    m1 = torch.from_numpy((synth.uniform(31, 1, (5, 400)) > 0.5).astype(np.float32))
    m2 = torch.from_numpy((synth.uniform(31, 2, (7, 400)) > 0.6).astype(np.float32))
    out['mask_iou'] = rbox.mask_iou(m1, m2).numpy()
    # the oracle must reproduce all of it before the fixture is written
    o2, l2, g2, i2 = zip(*[tn.match(tg[i][:, :4], anchors.numpy(), tg[i][:, 4], cfg.pos_iou_thre, cfg.neg_iou_thre) for i in range(B)])
    assert np.array_equal(np.stack(l2), out['labels']) and np.array_equal(np.stack(i2), out['matched_idx'])
    assert np.allclose(np.stack(o2)[out['labels'] > 0], out['offsets'][out['labels'] > 0], rtol=1e-5, atol=1e-6)
    assert np.array_equal(tn.ohem_negatives(class_p.numpy(), out['labels']), out['ohem_neg'])
    print('  train stages: pos', int(pos.sum()), 'neg', int(neg.sum()), 'losses', [round(float(out[k]), 5) for k in ('loss_c', 'loss_b', 'loss_m', 'loss_s')])
    np.savez_compressed(os.path.join(HERE, 'train_stages.npz'), **out)


def gen_surface(rcfg, ryolact):
    """Drop-in surface of the reference: state-dict layout (name, shape, dtype) of Yolact for every backbone in eval and
    train mode, and the config attributes the hot path reads (SURVEY.md 8b), per config name and mode."""
    import contextlib, io, json, types
    out = {'state_dict': {}, 'config': {}}
    for arch in ('res50', 'res101', 'swin_tiny'):
        for mode in ('detect', 'train'):
            ns = types.SimpleNamespace(cfg=arch + '_coco', img_size=544, weight=None, traditional_nms=False, resume=None, train_bs=2,
                                       val_interval=-1, val_num=-1, coco_api=False, visual_thre=0.0, save_lincomb=False, no_crop=False,
                                       image=None, video=None, hide_mask=False, hide_bbox=False, hide_score=False, cutout=False,
                                       real_time=False)
            with contextlib.redirect_stdout(io.StringIO()):
                cfg = rcfg.get_config(ns, mode)
            net = ryolact.Yolact(cfg)
            out['state_dict'][f'{arch}/{mode}'] = [[k, list(v.shape), str(v.dtype).replace('torch.', '')] for k, v in net.state_dict().items()]
            keep = ('num_classes', 'aspect_ratios', 'img_size', 'scales', 'mode', 'nms_score_thre', 'nms_iou_thre', 'top_k', 'max_detections',
                    'traditional_nms', 'pos_iou_thre', 'neg_iou_thre', 'masks_to_train', 'conf_alpha', 'bbox_alpha', 'mask_alpha',
                    'semantic_alpha', 'visual_thre', 'lr', 'warmup_until', 'warmup_init', 'momentum', 'decay', 'bs_per_gpu')
            out['config'][f'{arch}_coco/{mode}'] = {k: getattr(cfg, k) for k in keep if hasattr(cfg, k)}
    json.dump(out, open(os.path.join(HERE, 'surface.json'), 'w'), indent=0, sort_keys=True)
    print('  surface:', {k: len(v) for k, v in out['state_dict'].items()})


if __name__ == '__main__':
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())
    build_cython_nms()
    rcfg, ryolact, rout, rbox = import_reference()
    which = sys.argv[1:] or ['anchors', 'hard', 'post', 'after', 'forward', 'valaug', 'train', 'surface', 'stages', 'twins']
    if 'anchors' in which: gen_anchors(rcfg, ryolact)
    if 'hard' in which: gen_hard_nms()
    if 'post' in which: gen_postprocess(rcfg, rout)
    if 'after' in which: gen_after_nms(rcfg, rout)
    if 'forward' in which: gen_forward(rcfg, ryolact)
    if 'valaug' in which: gen_val_aug()
    if 'train' in which: gen_train(rcfg, ryolact)
    if 'surface' in which: gen_surface(rcfg, ryolact)
    if 'stages' in which: gen_train_stages(rcfg, ryolact, rbox)
    if 'twins' in which: gen_numpy_twins(rcfg, rout)
    print('done')
