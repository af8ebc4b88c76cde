"""Runs the inference step of the streaming loop (neuralrgbd_b200.test_utils.test_KVNet.test, the engine's restatement of
the reference's test_utils/test_KVNet.py:test) on a KVNET built through the reference's import names, the way the
reference's test_KVNet.py:159-168,190-250 does: install_as_reference_modules() with no checkout registers the engine
under `models.KVNET`, the model is constructed by keyword, wrapped in nn.DataParallel, .cuda(), loaded with weights,
then frames are streamed feeding each step the prior the previous one returned. Prints one JSON line with the outputs'
deviation from the committed live-reference fixtures. Executed as a subprocess by tests/test_gpu_dropin.py (keeps the
reference's top-level module names out of the test process)."""
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    case_name = sys.argv[1] if len(sys.argv) > 1 else 'kvnet_256_d16'
    import neuralrgbd_b200
    neuralrgbd_b200.install_as_reference_modules()
    import models.KVNET as m_kvnet                     # the reference's module name, registered to the engine
    from neuralrgbd_b200.test_utils import test_KVNet as ref_step
    from oracle import planesweep_oracle as O
    from tests import cases
    c = cases.kvnet_case(case_name)
    cam = cases.cam_for(O.make_cam_intrinsics, c['W'] // 4, c['H'] // 4)
    cam = dict(cam, unit_ray_array_2D=torch.from_numpy(cam['unit_ray_array_2D']),
               intrinsic_M_cuda=torch.from_numpy(cam['intrinsic_M_cuda']))
    with contextlib.redirect_stdout(io.StringIO()):
        model = m_kvnet.KVNET(feature_dim=64, cam_intrinsics=cam, d_candi=c['d'], sigma_soft_max=c['sigma'],
                              KVNet_feature_dim=64, d_upsample_ratio_KV_net=None, t_win_r=2, if_refined=True)   # test_KVNet.py:159-162
    model = torch.nn.DataParallel(model)                # :163
    model.cuda()                                        # :164
    model.module.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in c['sd'].items()})
    gold = np.load(os.path.join(ROOT, 'tests', 'golden', 'reference_outputs.npz'))
    out = {'class': type(model.module).__module__, 'steps': []}
    bv = None
    for step in range(len(c['frames']) - 4):
        ref_f, src_f, poses = cases.window(c, 2 + step)
        Ref_Dats = [{'img': torch.from_numpy(ref_f)}]
        Src_Dats = [[{'img': torch.from_numpy(src_f[0, v:v + 1])} for v in range(src_f.shape[1])]]
        poses_t = torch.from_numpy(poses).cuda()
        dmap, bv_next = ref_step.test(model, c['d'], [cam], 2, Ref_Dats, Src_Dats, poses_t, bv, R_net=True)
        kv, bv_next2 = ref_step.test(model, c['d'], [cam], 2, Ref_Dats, Src_Dats, poses_t, bv, R_net=False)
        key = 'kvnet/%s/step%d' % (case_name, step)
        e = lambda a, k: float(np.abs(np.exp(cases.subsample(a.cpu().numpy())) - np.exp(gold[k])).max())      # noqa: E731
        out['steps'].append({'dmap_refined': e(dmap, key + '/dmap_refined'), 'DPV': e(kv, key + '/DPV'),
                             'prior_next': e(bv_next, key + '/BV_predict_next'),
                             'deterministic': bool(torch.equal(bv_next, bv_next2))})
        bv = bv_next                                    # free-running, as the driver loop does (test_KVNet.py:224-236)
    from neuralrgbd_b200 import _lib
    out['launches'] = int(_lib.lib().nrgbd_launch_count())
    print(json.dumps(out))


if __name__ == '__main__':
    main()
