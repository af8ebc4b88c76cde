"""Drop-in boundary on the GPU (SURVEY 8b; VERDICT r1 weak #4, ADVICE r1 high):
 * the inference step `test_utils.test_KVNet.test` streams frames on a KVNET built through the reference's
   `models.KVNET` name (install_as_reference_modules()) and nn.DataParallel, and reproduces the live-reference fixtures;
 * a real nn.DataParallel replica (torch.nn.parallel.replicate) of the engine-backed KVNET runs a forward, and
   freeing it leaves the owner's engines usable.
"""
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import planesweep_oracle as O
from tests import cases
from tests.conftest import ROOT, maxabs

pytestmark = pytest.mark.gpu


def test_reference_inference_step_runs_on_the_engine():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'dropin_driver.py'), 'kvnet_256_d16'],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out['class'] == 'neuralrgbd_b200.models.KVNET' and out['launches'] > 100
    assert len(out['steps']) == 3
    for i, s in enumerate(out['steps']):
        tol = 1e-4 if i == 0 else 5e-4          # free-running K-Net steps: see tests/test_gpu_configs.py
        assert s['deterministic']
        assert s['dmap_refined'] <= tol and s['DPV'] <= tol and s['prior_next'] <= 5e-4, out


def test_dataparallel_replica_forward_and_ownership():
    from neuralrgbd_b200.models.KVNET import KVNET
    from torch.nn.parallel import replicate
    c = cases.kvnet_case('kvnet_256x320_d8')
    cam = cases.cam_for(O.make_cam_intrinsics, c['W'] // 4, c['H'] // 4)
    cam = dict(cam, unit_ray_array_2D=torch.from_numpy(cam['unit_ray_array_2D']), intrinsic_M_cuda=torch.from_numpy(cam['intrinsic_M_cuda']))
    with contextlib.redirect_stdout(io.StringIO()):
        m = KVNET(64, cam, c['d'], c['sigma'], 64, None, t_win_r=2)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in c['sd'].items()})
    m = m.cuda()
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()     # noqa: E731
    ref_f, src_f, poses = cases.window(c, 2)
    args = (T(ref_f), T(src_f), T(poses), torch.zeros(1))
    with torch.no_grad():
        base = m(*args, cam_intrinsics=[cam], BV_predict=None)
        for _ in range(2):                                  # what DataParallel.forward does on a multi-GPU box, every call
            rep = replicate(m, [0])[0]
            assert getattr(rep, '_is_replica', False)
            got = rep(*args, cam_intrinsics=[cam], BV_predict=None)
            assert torch.equal(got[2], base[2]) and torch.equal(got[0], base[0])
            del rep, got
        again = m(*args, cam_intrinsics=[cam], BV_predict=None)        # owner's engine still alive after the replicas died
    assert torch.equal(again[2], base[2])
    gold = np.load(os.path.join(ROOT, 'tests', 'golden', 'reference_outputs.npz'))
    assert maxabs(np.exp(cases.subsample(base[2].cpu().numpy())), np.exp(gold['kvnet/kvnet_256x320_d8/step0/BV_cur'])) <= 1e-4
