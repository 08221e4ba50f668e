"""CPU: the oracle (numpy / torch restatements) reproduces every golden vector minted from the
reference itself (tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from cases import nms_cases, build_nms_inputs
from oracle import synth, postprocess_np as pp, forward_torch as ft


def test_anchors_golden():
    g = load_golden('anchors.npz')
    for S in (128, 384, 400, 544, 550, 576):
        a = pp.make_anchors(S)
        assert a.shape[0] == int(g[f'S{S}/count'])
        assert np.array_equal(a[:: max(1, a.shape[0] // 64)], g[f'S{S}/rows'])
        assert np.array_equal(a.astype(np.float64).sum(0), g[f'S{S}/sum64'])
    assert pp.make_anchors(550).shape[0] == 19248 and pp.make_anchors(544).shape[0] == 18525


def test_hard_nms_golden():
    g = load_golden('hard_nms.npz')
    for seed, n in ((1, 1), (2, 17), (3, 300), (4, 1500)):
        xy = synth.uniform(seed, 11, (n, 2)) * 400
        wh = synth.uniform(seed, 12, (n, 2)) * 120 + 1
        sc = synth.uniform(seed, 13, (n, 1))
        dets = np.concatenate([xy, xy + wh, sc], 1).astype(np.float32)
        for thr in (0.3, 0.5):
            assert np.array_equal(pp.hard_nms(dets, thr), g[f's{seed}_n{n}_t{thr}'])


@pytest.mark.parametrize('case', nms_cases(), ids=lambda c: c[0])
def test_nms_golden(case):
    g = load_golden('postprocess.npz')
    name, S, regime, seed, mut = case
    anchors, cls, box, coef = build_nms_inputs(S, regime, seed, mut)
    for trad in (False, True):
        key = f'{name}/{"trad" if trad else "fast"}'
        if key + '/count' not in g:
            continue
        r = pp.nms(cls, box, anchors, traditional=trad, img_size=S)
        if int(g[key + '/count']) == 0:
            assert r is None or len(r[0]) == 0
            continue
        assert np.array_equal(r[0], g[key + '/class'])
        assert np.array_equal(r[3], g[key + '/anchor'])
        assert np.array_equal(r[1], g[key + '/score'])
        # boxes: reference uses SLEEF expf, oracle the correctly-rounded exp: <= 1 ulp at <= 1.0
        assert np.allclose(r[2], g[key + '/box'], rtol=0, atol=2.4e-7)


def test_after_nms_golden():
    g = load_golden('after_nms.npz')
    for name, S, h, w, seed in (('S128_80x120', 128, 80, 120, 5), ('S128_97x64', 128, 97, 64, 6), ('S256_60x60', 256, 60, 60, 7)):
        anchors = pp.make_anchors(S)
        cls, box, coef = synth.head_outputs(seed, anchors.shape[0], 81, 'realistic')
        proto = synth.proto(seed, S // 4)
        ids, scores, boxes, aidx = pp.nms(cls, box, anchors)
        o = pp.after_nms(ids, scores, boxes, coef[aidx], proto, h, w)
        shape = tuple(g[name + '/mask_shape'])
        ref = np.unpackbits(g[name + '/mask_bits'])[:int(np.prod(shape))].reshape(shape)
        assert o[3].shape == shape
        assert np.array_equal(o[2], g[name + '/boxes_px'])
        assert (o[3] != ref).mean() < 2e-4


@pytest.mark.parametrize('key', ['res50_S64_B2', 'res101_S64_B1', 'res50_S128_B2'])
def test_forward_golden_small(key):
    g = load_golden('forward.npz')
    arch, S, B = key.split('_')
    S, B = int(S[1:]), int(B[1:])
    sub, psub = int(g[key + '/sub']), int(g[key + '/psub'])
    sd = ft.synth_state_dict(arch, seed=0)
    img = torch.from_numpy(synth.image_batch(11, B, S))
    cls, box, coef, proto = [t.numpy() for t in ft.forward(img, sd, arch)]
    assert cls.shape[1] == int(g[key + '/shapes'][0]) and proto.shape[1] == int(g[key + '/shapes'][1])
    for mine, name in ((cls[:, ::sub], 'cls'), (box[:, ::sub], 'box'), (coef[:, ::sub], 'coef'), (proto[:, ::psub, ::psub], 'proto')):
        assert np.allclose(mine, g[f'{key}/{name}'], rtol=0, atol=2e-6), name


def test_c_hard_nms_matches_numpy_oracle_and_golden():
    """oracle/hard_nms.c (plain-C restatement of cython_nms.pyx) == numpy oracle == reference goldens."""
    import ctypes, os, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(['make', '-s', '-C', os.path.join(root, 'oracle')])
    lib = ctypes.CDLL(os.path.join(root, 'oracle', '_build', 'liboracle_hard_nms.so'))
    lib.oracle_hard_nms.restype = ctypes.c_int
    lib.oracle_hard_nms.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_void_p]
    g = load_golden('hard_nms.npz')
    for seed, n in ((1, 1), (2, 17), (3, 300), (4, 1500)):
        xy = synth.uniform(seed, 11, (n, 2)) * 400
        wh = synth.uniform(seed, 12, (n, 2)) * 120 + 1
        sc = synth.uniform(seed, 13, (n, 1))
        dets = np.ascontiguousarray(np.concatenate([xy, xy + wh, sc], 1).astype(np.float32))
        for thr in (0.3, 0.5):
            keep = np.zeros(n, np.uint8)
            kept = lib.oracle_hard_nms(dets.ctypes.data, n, thr, keep.ctypes.data)
            idx = np.nonzero(keep)[0]
            assert kept == len(idx)
            assert np.array_equal(idx, g[f's{seed}_n{n}_t{thr}'])
            assert np.array_equal(idx, pp.hard_nms(dets, thr))


VAL_AUG_CASES = (('97x64_S96', 97, 64, 96, 1), ('120x160_S128', 120, 160, 128, 2), ('200x200_S64', 200, 200, 64, 3),
                 ('375x500_S550', 375, 500, 550, 4))


def test_val_aug_golden():
    """numpy restatement of val_aug vs the reference's cv2 pipeline (cv2's IPP resize differs from the
    textbook bilinear formula by ~1e-4 on normalised values)."""
    g = load_golden('val_aug.npz')
    for name, h, w, S, seed in VAL_AUG_CASES:
        img = (synth.uniform(seed, 21, (h, w, 3)) * 256).astype(np.uint8)
        out = pp.val_aug(img, S)
        sub = int(g[name + '/sub'])
        assert out.shape == (3, S, S)
        assert np.abs(out[:, ::sub, ::sub] - g[name + '/out']).max() < 2e-4
        assert np.allclose(out.astype(np.float64).sum(axis=(1, 2)), g[name + '/sum'], rtol=0, atol=0.05)
