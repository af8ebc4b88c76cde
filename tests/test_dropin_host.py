"""Host-side drop-in logic (CPU, no GPU): install_as_reference_modules() against a reference-shaped checkout,
and the ownership rules of nn.DataParallel replicas of the engine-backed KVNET (ADVICE r1)."""
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import torch

from tests import cases
from tests.conftest import ROOT

# A stand-in for the `code/` directory of an NVlabs/neuralrgbd checkout: the module names, the symbols the patches
# touch or must keep, and the cross-imports that matter to the install (warping.homography imports warping.View by
# `from warping import View`; mutils.misc, models.KVNET, the data loaders and the inference step import the reference
# modules by their top-level names). Bodies are placeholders: only where each name resolves is checked.
STUB_CHECKOUT = {
    'warping/__init__.py': '',
    'warping/View.py': 'def normalised_pixel_to_ray_array(width=320, height=240, hfov=60, vfov=45, normalize_z=True):\n'
                       '    raise NotImplementedError\n',
    'warping/homography.py': 'from warping import View\n' + ''.join(
        'def %s(*args, **kwargs):\n    raise NotImplementedError\n' % n
        for n in ('est_swp_volume_v4', 'warp_img_feats_v3', 'warp_img_feats_mgpu', 'resample_vol_cuda', 'get_rel_extrinsicM',
                  'back_warp_th_Rt', 'back_warp_th_Rt_msrc')),
    'mutils/__init__.py': '',
    'mutils/misc.py': 'import warping.View as View\nimport warping.homography as warp_homo\n' + ''.join(
        'def %s(*args, **kwargs):\n    raise NotImplementedError\n' % n
        for n in ('depth_val_regression', 'valid_dpv', 'get_entries_list_dict', 'm_makedir', 'save_ScenePathInfo',
                  'split_frame_list')),
    'models/__init__.py': '',
    'models/KVNET.py': 'import warping.homography as warp_homo\nimport mutils.misc as m_misc\n\n\nclass KVNET:\n    pass\n',
    'mdataloader/__init__.py': '',
    'mdataloader/scanNet.py': 'import warping.View as View\n',
    'test_utils/__init__.py': '',
    'test_utils/test_KVNet.py': 'import warping.homography as warp_homo\nimport mutils.misc as m_misc\n\n\n'
                                'def test(*args, **kwargs):\n    return warp_homo.resample_vol_cuda(*args, **kwargs)\n',
}


def _stub_checkout(root):
    code = os.path.join(str(root), 'code')
    for rel, text in STUB_CHECKOUT.items():
        os.makedirs(os.path.dirname(os.path.join(code, rel)), exist_ok=True)
        with open(os.path.join(code, rel), 'w') as f:
            f.write(text)
    return code


INSTALL_PROBE = r'''
import json, sys
sys.path.insert(0, %(root)r)
import neuralrgbd_b200
ns = neuralrgbd_b200.install_as_reference_modules(%(ref)r)
out = {}
import warping.homography as warp_homo, warping.View, mutils.misc as m_misc, models.KVNET as m_kvnet
import test_utils.test_KVNet as ref_test            # the reference's own inference step, unmodified
import mdataloader.scanNet                          # imports warping.View (broke when the package was replaced)
out['homography_file'] = warp_homo.__file__
out['misc_file'] = m_misc.__file__
out['step_file'] = ref_test.__file__
for mod, names in (('h', ['est_swp_volume_v4', 'warp_img_feats_v3', 'warp_img_feats_mgpu', 'resample_vol_cuda']),):
    out['patched_h'] = [getattr(warp_homo, n).__module__ for n in names]
out['patched_misc'] = m_misc.depth_val_regression.__module__
out['patched_kvnet'] = m_kvnet.KVNET.__module__
out['kept'] = [hasattr(m_misc, n) for n in ('get_entries_list_dict', 'm_makedir', 'save_ScenePathInfo', 'split_frame_list')]
out['view'] = hasattr(warping.View, 'normalised_pixel_to_ray_array')
out['step_sees_patch'] = ref_test.warp_homo.resample_vol_cuda.__module__
neuralrgbd_b200.uninstall_reference_patches()
out['restored'] = warp_homo.resample_vol_cuda.__module__
print(json.dumps(out))
'''


def test_install_patches_the_reference_modules_in_place(tmp_path):
    REF_CODE = _stub_checkout(tmp_path)
    r = subprocess.run([sys.executable, '-c', INSTALL_PROBE % dict(root=ROOT, ref=REF_CODE)], capture_output=True, text=True,
                       timeout=600, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out['homography_file'].startswith(REF_CODE) and out['misc_file'].startswith(REF_CODE)      # reference modules stay
    assert out['step_file'].startswith(REF_CODE)
    assert all(m == 'neuralrgbd_b200.warping.homography' for m in out['patched_h'])
    assert out['patched_misc'] == 'neuralrgbd_b200.mutils.misc' and out['patched_kvnet'] == 'neuralrgbd_b200.models.KVNET'
    assert all(out['kept']) and out['view']
    assert out['step_sees_patch'] == 'neuralrgbd_b200.warping.homography'
    assert out['restored'] == 'warping.homography'


def test_install_without_a_checkout_registers_the_mirrors():
    code = ('import sys; sys.path.insert(0, %r); import neuralrgbd_b200 as n; n.install_as_reference_modules(); '
            'import warping.homography as w, models.KVNET as k, mutils.misc as m; '
            'print(w.__name__, k.KVNET.__module__, m.__name__)' % ROOT)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=600, cwd='/tmp')
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == ['neuralrgbd_b200.warping.homography', 'neuralrgbd_b200.models.KVNET', 'neuralrgbd_b200.mutils.misc']


def _fake_replicate(m):
    """What torch.nn.parallel.replicate does to a module tree, minus the CUDA broadcast."""
    modules = list(m.modules())
    idx = {mod: i for i, mod in enumerate(modules)}
    reps = [mod._replicate_for_data_parallel() for mod in modules]
    for i, mod in enumerate(modules):
        r = reps[i]
        for k, ch in mod._modules.items():
            r._modules[k] = None if ch is None else reps[idx[ch]]
        for k, p in mod._parameters.items():
            if p is not None:
                setattr(r, k, p.detach().clone())          # plain tensor attribute: replica._parameters stays empty
        for k, b in mod._buffers.items():
            r._buffers[k] = None if b is None else b.clone()
    return reps[0]


def test_dataparallel_replica_resolves_parameters_and_never_owns_handles(monkeypatch):
    from neuralrgbd_b200.models import KVNET as K
    from neuralrgbd_b200 import camera
    cam = camera.make_cam_intrinsics(cases.FX, cases.FY, cases.CX, cases.CY, [64, 64])
    with contextlib.redirect_stdout(io.StringIO()):
        m = K.KVNET(64, cam, np.linspace(0.1, 5, 8), 10., 64, None, t_win_r=2)
    rep = _fake_replicate(m)
    assert getattr(rep, '_is_replica', False) and len(dict(rep.named_parameters())) == 0
    plist = rep._param_list()                                   # raised KeyError in round 1
    base = dict(m._param_list())
    assert len(plist) == len(base) and all(t.shape == base[n].shape for n, t in plist)
    assert rep._engines is m._engines                           # one engine table, keyed by device

    destroyed = []

    class FakeLib:
        def nrgbd_kvnet_destroy(self, h):
            destroyed.append(h)
    monkeypatch.setattr(K._lib, 'lib', lambda: FakeLib())
    m._engines[('fake',)] = {'h': 'HANDLE'}
    rep.__del__()
    assert destroyed == [] and ('fake',) in m._engines          # a replica never frees the owner's engines
    m.__del__()
    assert destroyed == ['HANDLE'] and not m._engines           # the owner frees each handle exactly once
    m.__del__()
    assert destroyed == ['HANDLE']


def test_batches_tracked_counters_follow_the_reference():
    """kv_net BatchNorm3d counters advance only on forwards that ran K-Net (ADVICE r1, KVNET.py:138-143)."""
    from neuralrgbd_b200.models import KVNET as K
    from neuralrgbd_b200 import camera
    cam = camera.make_cam_intrinsics(cases.FX, cases.FY, cases.CX, cases.CY, [64, 64])
    with contextlib.redirect_stdout(io.StringIO()):
        m = K.KVNET(64, cam, np.linspace(0.1, 5, 8), 10., 64, None, t_win_r=2)
    m.__dict__['_nb_pending'] = 5          # five forwards ...
    m.__dict__['_nb_pending_kv'] = 3       # ... three of them with a valid prior
    sd = m.state_dict()
    nb = {k: int(v) for k, v in sd.items() if k.endswith('num_batches_tracked')}
    assert len(nb) == 15
    assert all(v == 3 for k, v in nb.items() if k.startswith('kv_net.'))
    assert all(v == 5 for k, v in nb.items() if not k.startswith('kv_net.'))
