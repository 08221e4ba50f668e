"""oracle/ref_loader.py -- TEST INFRASTRUCTURE (see oracle/__init__.py).

Imports the UNMODIFIED reference (feiyuhuahuo/Yolact_minimal) for bench.py's reference arm and the golden-vector scripts:

  * location: $YOLACT_REFERENCE (unset: the reference is not available and callers use the restatements in oracle/);
  * config.py mkdirs in the CWD on import (config.py:6-15) -> imported from a scratch CWD;
  * utils/output_utils.py:7 imports cython_nms unconditionally; cython_nms.pyx does not compile with Cython 3 / numpy 2
    (np.int_t, dtype=np.int) -> the 2-token-patched build in oracle/_ref is used when present, else a stub module (only
    --traditional_nms calls it);
  * sizes that are not multiples of 32 (550, 400) need the 3-line FPN change of SURVEY.md App. E.3 (interpolate to the lateral's
    size instead of scale_factor=2): `patch_fpn()` installs it at run time, the reference's files stay untouched.

Nothing under yolact_minimal_b200/ imports this module.
"""
import contextlib
import io
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFBUILD = os.path.join(ROOT, 'oracle', '_ref')


def locate():
    p = os.environ.get('YOLACT_REFERENCE')
    if p and os.path.exists(os.path.join(p, 'modules', 'yolact.py')):
        return p
    return None


def available():
    return locate() is not None


def build_cython_nms(src):
    """Build the reference's cython_nms.pyx (with the 2-token numpy-2 patch: np.int_t -> np.int64_t, np.int -> np.int64) into
    the git-ignored oracle/_ref/.  Outputs only; the patched copy of the .pyx is a build intermediate and is not tracked."""
    import subprocess
    pyx = os.path.join(src, 'cython_nms.pyx')
    if not os.path.exists(pyx):
        return False
    os.makedirs(REFBUILD, exist_ok=True)
    text = open(pyx).read().replace('np.int_t', 'np.int64_t').replace('dtype=np.int)', 'dtype=np.int64)')
    dst = os.path.join(REFBUILD, 'cython_nms.pyx')
    if not (os.path.exists(dst) and open(dst).read() == text and any(f.startswith('cython_nms.') and f.endswith('.so') for f in os.listdir(REFBUILD))):
        open(dst, 'w').write(text)
        open(os.path.join(REFBUILD, 'setup.py'), 'w').write(
            "from distutils.core import setup\nfrom Cython.Build import cythonize\nimport numpy\n"
            "setup(ext_modules=cythonize('cython_nms.pyx', language_level=3), include_dirs=[numpy.get_include()])\n")
        subprocess.check_call([sys.executable, 'setup.py', '-q', 'build_ext', '--inplace'], cwd=REFBUILD,
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    return True


_cache = {}


def load():
    """-> (config module, modules.yolact, utils.output_utils, utils.box_utils) of the reference."""
    if 'mods' in _cache:
        return _cache['mods']
    ref = locate()
    if ref is None:
        raise RuntimeError('reference not available: set YOLACT_REFERENCE to a checkout of it')
    scratch = '/tmp/yolact_ref_cwd'
    os.makedirs(scratch, exist_ok=True)
    cwd = os.getcwd()
    os.chdir(scratch)
    try:
        if os.path.isdir(REFBUILD):
            sys.path.insert(0, REFBUILD)
        try:
            import cython_nms  # noqa: F401  (the patched build of the reference's .pyx)
        except ImportError:
            stub = types.ModuleType('cython_nms')
            stub.nms = lambda *a, **k: (_ for _ in ()).throw(RuntimeError('cython_nms is not built in this environment'))
            sys.modules['cython_nms'] = stub
        # the reference's top-level names (config, modules, utils) must win over anything already imported
        for name in [m for m in sys.modules if m == 'config' or m.split('.')[0] in ('modules', 'utils')]:
            del sys.modules[name]
        sys.path.insert(0, ref)
        import config as rcfg
        from modules import yolact as ryolact
        from utils import output_utils as rout
        from utils import box_utils as rbox
    finally:
        os.chdir(cwd)
    _cache['mods'] = (rcfg, ryolact, rout, rbox)
    return _cache['mods']


def ref_cfg(name, img_size, mode='detect', traditional=False):
    rcfg = load()[0]
    ns = types.SimpleNamespace(cfg=name, img_size=544, weight=None, traditional_nms=traditional, visual_thre=0.0,
                               save_lincomb=False, no_crop=False, image=None, video=None, hide_mask=False, hide_bbox=False,
                               hide_score=False, cutout=False, real_time=False, val_num=-1, coco_api=False)
    cwd = os.getcwd()
    os.chdir('/tmp/yolact_ref_cwd')
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            cfg = rcfg.get_config(ns, mode)
    finally:
        os.chdir(cwd)
    cfg.img_size = img_size                                   # bypass config.py:75 for 550/400
    cfg.scales = [int(img_size / 544 * a) for a in (24, 48, 96, 192, 384)]
    return cfg


def patch_fpn():
    """SURVEY.md App. E.3: interpolate-to-lateral-size so that 550 / 400 run.  Returns the original forward."""
    import torch.nn.functional as F
    ryolact = load()[1]

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


def build_net(arch, img_size, state_dict):
    """The reference's Yolact(cfg) in eval mode with `state_dict` loaded strictly (FPN patched when img_size % 32 != 0)."""
    ryolact = load()[1]
    cfg = ref_cfg(arch + '_coco', img_size)
    net = ryolact.Yolact(cfg)
    net.load_state_dict(state_dict, strict=True)
    if img_size % 32 != 0:
        patch_fpn()
    return net.eval(), cfg
