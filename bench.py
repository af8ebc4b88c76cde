#!/usr/bin/env python
"""bench.py - depth frames/s of the plane-sweep DPV hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1..c5] [--impl engine|reference|reference-gpu]
                    [--dump-outputs DIR]

Workloads = BASELINE.json configs (SURVEY 8d). `--config` picks one; the default c2 is the configuration the metric is
quoted on (the driver's BENCH / SCALE runs use it), the others write the same JSON line for their shape:
  c1  single 320x256 reference + 1 source pair, 32 planes, C = 67: warping.homography.est_swp_volume_v4 only
  c2  640x480, 64 planes, 4 source views, D-Net DPV + R-Net = first-window KVNET.forward           (default)
  c3  c2's shape, full KVNet (D-Net + K-Net Bayesian filter + 2x R-Net + DPV propagation), streaming 30-frame window
  c4  1248x376 (the reference CNN rejects 1242x375), 128 KITTI planes, full KVNet streaming, frame chunks sharded over ranks
  c5  1920x1080, 256 planes, 8 source views, first-window KVNET.forward (the 1/2/4/8-GPU throughput sweep)
One step = one depth frame (c1: one cost volume). Synthetic seeded frames / poses / random-init weights of the reference
architecture (no datasets or checkpoints offline).

value  : whole-job frames/s with the inputs already resident in HBM (engine C ABI, device pointers).
e2e    : the same metric through the public Python surface with pinned HOST buffers inside the timed region, every step:
         c1/c2/c5 upload the float window + poses and read back the full-resolution depth + confidence maps;
         c3/c4 stream ONE decoded uint8 frame per step into the resident FrameWindow (mdataloader mirror, SURVEY f-4),
         run the reference-named inference step (test_utils.test_KVNet.test: forward + DPV propagation) and read back the
         depth map and the confidence map (export_res mirror, f-2).
roofline: the dominant kernel family (conv_h2_kernel, tcgen05 kind::f16 on split-fp16 pairs) timed with CUDA events around
         every launch on the launching stream, in eager frames with ONE frame in flight run right after the timed region;
         the frames/s of that same regime is reported next to it (roofline.regime). achieved = algorithmic fp32 FLOPs /
         kernel time against the measured bf16 tensor peak (MEASURED_PEAKS.json; the kernel issues 3 f16 MMAs per
         product: its MMA rate is 3x the algorithmic rate). The geometry kernels' HBM fractions are listed in config.hbm_kernels.
cpu_baseline / --impl reference: the UNMODIFIED reference (baseline/_ref, copied by baseline/fetch_reference.py) through its
         own models.KVNET.KVNET.forward / test_utils.test_KVNet.test on the host cores (the 4-line .cuda() shim of SURVEY
         8c; kind "reference"); oracle/torch_port.py (kind "port") only when baseline/_ref is absent.
--impl reference-gpu: the same unmodified reference, unshimmed, eager ATen/cuDNN on the same B200 (SURVEY 8d ii), with
         cudnn.benchmark as test_KVNet.py:10 sets it; also records its TF32-default vs fp32 deviation (the noise floor
         the reference itself has on this GPU).

N > 1 (torchrun): one process per GPU; frames (c1, c2, c5) / trajectory chunks (c3, c4) shard across ranks, weights are
broadcast once over NCCL, no per-frame collective; value = all ranks' frames / max-over-ranks time.

--dump-outputs DIR (engine arm, rank 0): what the last timed step returned, as DIR/<name>.npy in float32 - c1 the cost
         volume; c2/c5 dmap_cur_refined, bv_cur, depth_lowres; c3/c4 the maps of the last streamed frame and the prior it
         propagated (bv_predict_next). Inputs and weights are seeded, so the same arguments give the same inputs on every
         run and two builds can be compared output for output.
"""
import argparse
import contextlib
import ctypes
import io
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF_CODE = os.path.join(ROOT, 'baseline', '_ref', 'code')

SCANNET = dict(fx=585.0, fy=585.0, cx=320.0, cy=240.0, d=(0.1, 5.0))          # DSO/cam_info_7scenes.mat, test_KVNet.py ScanNet planes
CONFIGS = {
    'c1': dict(kind='sweep', h=256, w=320, V=1, D=32, C=67, intr=SCANNET,
               workload='pair320x256_d32_c67_plane_sweep_cost (BASELINE.json configs[0]; SURVEY C1)',
               metric='plane-sweep cost volumes/sec at 320x256x32-plane x1-view (C=67)'),
    'c2': dict(kind='first', H=480, W=640, D=64, V=4, r=2, intr=SCANNET, inflight=3,
               workload='scannet640x480_d64_v4_dnet_dpv_plus_rnet (BASELINE.json configs[1]; SURVEY C2)',
               metric='depth frames/sec at 640x480x64-plane x4-view'),
    'c3': dict(kind='stream', H=480, W=640, D=64, V=4, r=2, intr=SCANNET, n_stream=30, inflight=2,
               workload='scannet640x480_d64_v4_full_kvnet_stream30 (BASELINE.json configs[2]; SURVEY C3)',
               metric='depth frames/sec at 640x480x64-plane x4-view, full KVNet (D-Net + K-Net + 2x R-Net + propagation), streaming'),
    'c4': dict(kind='stream', H=376, W=1248, D=128, V=4, r=2, intr=dict(fx=721.5377, fy=721.5377, cx=624.0, cy=188.0, d=(1.0, 60.0)), n_stream=12, inflight=2,
               workload='kitti1248x376_d128_v4_full_kvnet_stream (BASELINE.json configs[3]; 1242x375 is rejected by the reference CNN; SURVEY C4)',
               metric='depth frames/sec at 1248x376x128-plane x4-view, full KVNet, streaming'),
    'c5': dict(kind='first', H=1080, W=1920, D=256, V=8, r=4, intr=dict(fx=1755.0, fy=1755.0, cx=960.0, cy=540.0, d=(0.1, 5.0)), inflight=2,
               workload='synthetic1920x1080_d256_v8_dnet_dpv_plus_rnet (BASELINE.json configs[4]; SURVEY C5)',
               metric='depth frames/sec at 1920x1080x256-plane x8-view'),
}


def read_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j['hbm_gbs'], bf16=j['bf16_tflops'], bf16_sustained=j.get('bf16_tflops_sustained', j['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16=1590.0, bf16_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop = False

    def run(self):
        while not self.stop:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]) if self.rows[0][1].replace('.', '').isdigit() else None,
                'samples': len(self.rows), 'reasons': sorted(reasons)}


def conv_traffic_per_launch():
    """dram__bytes_read.sum + dram__bytes_write.sum per conv launch (mean over the conv launches of one c2 frame) from the ncu
    capture of this round's kernels, profiles/r2_conv_dram_traffic.json; None if the file is missing."""
    try:
        return float(json.load(open(os.path.join(ROOT, 'profiles', 'r2_conv_dram_traffic.json')))['traffic_bytes_per_launch'])
    except Exception:
        return None


DUMP_BYTES = 64 << 20


def sample_outputs(arrays):
    """{name: CUDA tensor} -> {name: float32 host array} for --dump-outputs. The arrays share DUMP_BYTES (less 1 MiB for the
    .npy headers); one larger than its share becomes a 1-D sample of its flattened elements at positions drawn by a fixed
    seed and sorted, i.e. the same positions for the same shape on every run."""
    import torch
    cap = (DUMP_BYTES - (1 << 20)) // (4 * len(arrays))
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[name] = t.float().cpu().numpy()
    return out


def write_outputs(path, host_arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in host_arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def make_video(cfg, n_frames, seed):
    from neuralrgbd_b200 import synth
    frames, rng = synth.video(seed, n_frames, cfg['H'], cfg['W'])
    exts = synth.camera_track(rng, n_frames)
    return frames, exts


def make_windows(cfg, n_windows, seed=7):
    """n_windows seeded windows: frames [V+1,3,H,W] (sources then reference, basic.py:245) and relative poses [V,4,4]."""
    from neuralrgbd_b200 import synth
    r = cfg['r']
    frames, exts = make_video(cfg, n_windows + 2 * r, seed)
    wins = []
    for i in range(n_windows):
        poses, idx = synth.window_rel_poses(exts, r + i, r)
        f = np.stack([frames[j] for j in idx] + [frames[r + i]])
        wins.append((np.ascontiguousarray(f, np.float32), np.ascontiguousarray(poses, np.float32)))
    return wins


def cam_of(cfg, make_cam, quarter=True):
    i = cfg['intr']
    if cfg['kind'] == 'sweep':
        return make_cam(i['fx'], i['fy'], i['cx'], i['cy'], [cfg['w'], cfg['h']])
    return make_cam(i['fx'], i['fy'], i['cx'], i['cy'], [cfg['W'] // 4, cfg['H'] // 4])


# ==============================================================================================
# reference arms: the unmodified reference (baseline/_ref) on the host cores / on the same GPU
# ==============================================================================================
def pick_cpu_threads():
    """Thread count for the CPU arm: the fastest of {all cores, 64, 32, 16, 8} on a short calibration over the three conv
    shapes that dominate the frame (on many-core hosts torch's intra-op pool oversubscribes: 128 threads ran this path 6x
    slower than 8, and which count wins differs from host to host)."""
    import torch
    import torch.nn.functional as F
    n_all = os.cpu_count() or 1
    cands = sorted({c for c in (n_all, 64, 32, 16, 8) if c <= n_all})
    work = [(torch.randn(5, 64, 120, 160), torch.randn(64, 64, 3, 3)), (torch.randn(5, 128, 120, 160), torch.randn(128, 128, 3, 3)),
            (torch.randn(5, 32, 240, 320), torch.randn(32, 32, 3, 3))]
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        for x, w in work:
            F.conv2d(x, w, padding=1)
        if best_t is not None and time.perf_counter() - t0 > 4 * best_t:
            continue
        t0 = time.perf_counter()
        for _ in range(2):
            for x, w in work:
                F.conv2d(x, w, padding=1)
        t = time.perf_counter() - t0
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def reference_runner(cfg, on_gpu):
    """-> (step(i) -> seconds, description). Drives the unmodified reference (or, without baseline/_ref, the torch port)."""
    import torch
    from neuralrgbd_b200 import arch, synth
    from oracle import planesweep_oracle as O
    have_ref = os.path.isdir(REF_CODE)
    scale = 1.0
    crop = None
    if cfg['kind'] != 'sweep' and not on_gpu and cfg['H'] * cfg['W'] * cfg['D'] > 1248 * 376 * 128:
        # bounded CPU sample of the biggest configuration: a centred half-size crop (1/4 of the pixels), fps scaled by 1/4
        crop = dict(cfg, H=cfg['H'] // 2 // 4 * 4, W=cfg['W'] // 2 // 4 * 4)
        crop['intr'] = dict(cfg['intr'], cx=crop['W'] / 2.0, cy=crop['H'] / 2.0)
        scale = (crop['H'] * crop['W']) / float(cfg['H'] * cfg['W'])
        cfg = crop
    i = cfg['intr']
    d = synth.d_candidates(cfg['D'], i['d'][0], i['d'][1])
    camn = cam_of(cfg, O.make_cam_intrinsics)
    cam = dict(camn, unit_ray_array_2D=torch.from_numpy(camn['unit_ray_array_2D']), intrinsic_M_cuda=torch.from_numpy(camn['intrinsic_M_cuda']))
    dev = torch.device('cuda:0') if on_gpu else torch.device('cpu')
    if not on_gpu and have_ref:                      # SURVEY 8c: the reference hard-codes .cuda()
        torch.Tensor.cuda = lambda s, *a, **k: s
        torch.nn.Module.cuda = lambda s, *a, **k: s
        torch.cuda.current_device = lambda: 0
        torch.Tensor.get_device = lambda s: 0
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    if cfg['kind'] == 'sweep':
        from tests import cases
        c = cases.sweep_case('c1_320x256_v1_d32_c67')
        if have_ref:
            sys.path.insert(0, REF_CODE)
            import warping.homography as wh                     # reference
            args = (T(c['ref']), T(c['src']), c['d'], T(c['R']), T(c['t']), cam, c['sigma'])

            def step(k):
                t0 = time.perf_counter()
                out = wh.est_swp_volume_v4(*args)
                if on_gpu:
                    torch.cuda.synchronize()
                assert torch.isfinite(out).all()
                return time.perf_counter() - t0
            return step, 'unmodified reference warping.homography.est_swp_volume_v4 (baseline/_ref)', 'reference', 1.0
        from oracle import torch_port as TP

        def step(k):
            t0 = time.perf_counter()
            TP.est_swp_volume_v4(torch.from_numpy(c['ref']), torch.from_numpy(c['src']), c['d'], torch.from_numpy(c['R']), torch.from_numpy(c['t']), camn, c['sigma'])
            return time.perf_counter() - t0
        return step, 'CPU torch port of est_swp_volume_v4 (baseline/_ref absent)', 'port', 1.0
    r = cfg['r']
    sd = arch.synth_state_dict(5, 64, cfg['D'], r, 64)
    n_frames = 2 * r + 4
    frames, exts = make_video(cfg, n_frames, 7)
    if not have_ref:
        if cfg['kind'] != 'first' or on_gpu:
            raise RuntimeError('baseline/_ref is not present: only the first-window CPU port is available')
        from oracle import torch_port as TP
        P = TP._P(sd)

        def step(k):
            poses, idx = synth.window_rel_poses(exts, r + k % 3, r)
            f = np.stack([frames[j] for j in idx] + [frames[r + k % 3]])
            t0 = time.perf_counter()
            TP.kvnet_first_window(P, f[-1:], f[None, :-1], poses[None], camn, d, 10.)
            return time.perf_counter() - t0
        return step, 'CPU torch port of the reference path (oracle/torch_port.py; baseline/_ref absent)', 'port', scale
    sys.path.insert(0, REF_CODE)
    import models.KVNET as m_kvnet                              # reference
    import test_utils.test_KVNet as ref_step                    # reference
    if on_gpu:
        import torch.backends.cudnn as cudnn
        cudnn.benchmark = True                                  # test_KVNet.py:10
    with contextlib.redirect_stdout(io.StringIO()):
        model = m_kvnet.KVNET(feature_dim=64, cam_intrinsics=cam, d_candi=d, sigma_soft_max=10., KVNet_feature_dim=64,
                              d_upsample_ratio_KV_net=None, t_win_r=r, if_refined=True)
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    model = torch.nn.DataParallel(model)
    model.cuda()
    state = {'bv': None}

    def window(k):
        poses, idx = synth.window_rel_poses(exts, r + k, r)
        Ref = [{'img': torch.from_numpy(frames[r + k][None])}]
        Src = [[{'img': torch.from_numpy(frames[j][None])} for j in idx]]
        return Ref, Src, T(poses[None])

    if cfg['kind'] == 'first':
        def step(k):
            Ref, Src, poses = window(k % 3)
            t0 = time.perf_counter()
            out, _ = ref_step.test(model, d, [cam], r, Ref, Src, poses, None, R_net=True)
            if on_gpu:
                torch.cuda.synchronize()
            assert torch.isfinite(out).all()
            return time.perf_counter() - t0
    else:
        def step(k):
            if state['bv'] is None:                              # untimed first window seeds the recursion
                Ref, Src, poses = window(0)
                _, state['bv'] = ref_step.test(model, d, [cam], r, Ref, Src, poses, None, R_net=True)
            Ref, Src, poses = window(1 + k % 3)
            t0 = time.perf_counter()
            out, bv = ref_step.test(model, d, [cam], r, Ref, Src, poses, state['bv'], R_net=True)
            if on_gpu:
                torch.cuda.synchronize()
            assert torch.isfinite(out).all()
            state['bv'] = bv
            return time.perf_counter() - t0
    what = 'unmodified reference (baseline/_ref): models.KVNET.KVNET.forward + resample_vol_cuda through its own test_utils.test_KVNet.test'
    if crop is not None:
        what += ', on a centred %dx%d crop (%.3f of the pixels; frames/s scaled by that factor)' % (cfg['W'], cfg['H'], scale)
    return step, what, 'reference', scale


def run_reference(args, cfg, on_gpu):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    cores = 0
    if not on_gpu:
        cores = pick_cpu_threads()
    step, what, kind, scale = reference_runner(cfg, on_gpu)
    n_warm = (2 if on_gpu else 1) if args.warmup > 0 else 0
    cap = args.steps if on_gpu else min(args.steps, 3 if cfg['kind'] != 'sweep' else 10)      # CPU frames cost seconds each: bounded sample
    with torch.no_grad():
        for k in range(n_warm):
            step(k)
        ts = [step(n_warm + k) for k in range(max(1, cap))]
    sec = float(np.mean(ts))
    val = scale / sec
    line = {
        'impl': 'reference-gpu' if on_gpu else 'reference', 'metric': cfg['metric'], 'value': val, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': len(ts), 'warmup': n_warm, 'ms_per_step': sec * 1e3 / scale, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 (cuDNN/cuBLAS TF32 defaults of torch, as the reference runs)' if on_gpu else 'f32', 'data': 'synthetic',
        'config': {'workload': cfg['workload'], 'name': args.config},
        'e2e': {'value': val, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    if on_gpu:
        line['config']['what'] = what + '; eager ATen/cuDNN on cuda:0, cudnn.benchmark=True, frames uploaded inside the timed step by the reference itself'
    else:
        line['cpu_baseline'] = {'value': val, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
                                'sample': '%s; %d step(s) after %d warm-up, torch.set_num_threads(%d) (fastest of a calibration over {all=%d,64,32,16,8})'
                                          % (what, len(ts), n_warm, cores, os.cpu_count())}
    _emit(json.dumps(line))


def cpu_baseline_subprocess(args):
    """The CPU arm as a child process (the reference needs torch's .cuda() patched away, which must not happen in the process
    that drives the GPU). Returns the child's cpu_baseline object or an error note."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--config', args.config, '--steps', '1', '--warmup', '1'],
                           capture_output=True, text=True, timeout=1500, env=dict(os.environ, RANK='0', WORLD_SIZE='1'))
        line = [l for l in r.stdout.splitlines() if l.startswith('{')]
        return json.loads(line[-1])['cpu_baseline'] if line else {'error': (r.stderr or 'no output')[-300:]}
    except Exception as e:          # noqa: BLE001
        return {'error': repr(e)[:300]}


# ==============================================================================================
# the engine arm
# ==============================================================================================
def dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)          # NCCL_DEBUG is left alone: fd 1 points at stderr until the result line
    return world, rank, local, dev


def max_ms(ms, world, dev):
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_sweep(args, cfg):
    """c1: the fused plane-sweep cost kernel through warping.homography.est_swp_volume_v4 (public mirror)."""
    import torch
    import torch.distributed as dist
    import neuralrgbd_b200.warping.homography as Hm
    from neuralrgbd_b200 import _lib, camera
    from tests import cases
    world, rank, local, dev = dist_setup()
    L = _lib.lib()
    peaks = read_peaks()
    K, Wm = args.steps, args.warmup
    c = cases.sweep_case('c1_320x256_v1_d32_c67')
    i = cfg['intr']
    cam = camera.make_cam_intrinsics(i['fx'], i['fy'], i['cx'], i['cy'], [cfg['w'], cfg['h']])
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)      # noqa: E731
    ref, src, R, t = T(c['ref']), T(c['src']), T(c['R']), T(c['t'])
    pin = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (c['ref'], c['src'], c['R'], c['t'])]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    host_out = torch.empty((1, cfg['D'], cfg['h'], cfg['w'])).pin_memory()
    for _ in range(Wm):
        Hm.est_swp_volume_v4(ref, src, c['d'], R, t, cam, c['sigma'])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    barrier()
    L.nrgbd_reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        flush.zero_()
        cost = Hm.est_swp_volume_v4(ref, src, c['d'], R, t, cam, c['sigma'])
    e1.record()
    barrier()
    launches = int(L.nrgbd_launch_count())
    ms = max_ms(e0.elapsed_time(e1), world, dev)
    dumped = sample_outputs({'cost_volume': cost}) if args.dump_outputs and rank == 0 else None
    del cost
    # kernel-only time of the sweep (events around each call, no flush in between the event pair)
    ks = []
    for _ in range(10):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); Hm.est_swp_volume_v4(ref, src, c['d'], R, t, cam, c['sigma']); b.record(); torch.cuda.synchronize()
        ks.append(a.elapsed_time(b))
    barrier()
    e0.record()
    for _ in range(K):
        flush.zero_()
        dr, ds, dR, dt = [p.to(dev, non_blocking=True) for p in pin]
        out = Hm.est_swp_volume_v4(dr, ds, c['d'], dR, dt, cam, c['sigma'])
        host_out.copy_(out, non_blocking=True)
        torch.cuda.synchronize()
    e1.record()
    barrier()
    ms_e2e = max_ms(e0.elapsed_time(e1), world, dev)
    sampler.stop = True
    if rank == 0:
        hw = cfg['h'] * cfg['w']
        alg_bytes = ((1 + cfg['V']) * cfg['C'] + cfg['D'] + 3) * hw * 4.0
        call_ms = float(np.median(ks))
        gbs = alg_bytes / (call_ms * 1e-3) / 1e9
        line = {
            'metric': cfg['metric'], 'value': world * K / (ms * 1e-3), 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
            'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': cfg['workload'], 'name': args.config, 'l2': 'explicit 256 MiB flush write before every step (inside the timed region)',
                       'parallelism': 'dp%d (independent pairs)' % world},
            'e2e': {'value': world * K / (ms_e2e * 1e-3), 'unit': 'frames/s', 'h2d_bytes_per_step': sum(p.numel() * 4 for p in pin),
                    'd2h_bytes_per_step': host_out.numel() * 4},
            'gpu_launches': launches, 'clocks': sampler.summary(),
            'roofline': {'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'], 'traffic': None,
                         'kernel': 'est_swp_volume_v4 mirror = pack_features x2 + sweep set-up + plane_sweep kernel + transpose, %.1f us per call '
                                   '(CUDA events around the call, median of 10); algorithmic bytes (1+V) C hw 4 + D hw 4 + 3 hw 4 = %.1f MB. At C = 67 the '
                                   'kernel is gather / FFMA bound, not HBM bound (SURVEY 8d)' % (call_ms * 1e3, alg_bytes / 1e6),
                         'peak_source': peaks['source'] + ', HBM copy'},
        }
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline_subprocess(args)
        if dumped:
            write_outputs(args.dump_outputs, dumped)
        _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_engine(args, cfg):
    import torch
    import torch.distributed as dist
    from neuralrgbd_b200 import _lib, arch, camera, sharding, synth
    from neuralrgbd_b200._lib import ptr, check
    from neuralrgbd_b200.models.KVNET import KVNET
    from neuralrgbd_b200.mutils import misc
    from neuralrgbd_b200.mdataloader import m_preprocess
    from neuralrgbd_b200.test_utils import test_KVNet as step_mod
    from neuralrgbd_b200.test_utils import export_res

    world, rank, local, dev = dist_setup()
    L = _lib.lib()
    if args.dev_bn_unroll:
        _lib.dev_lib().nrgbd_dev_set_bn_unroll(args.dev_bn_unroll)
    if args.dev_smem_cap_kb:
        _lib.dev_lib().nrgbd_dev_conv_h2_set_smem_cap_kb(args.dev_smem_cap_kb)
    peaks = read_peaks()
    K, Wm = args.steps, args.warmup
    H_IMG, W_IMG, D_PLANES, V_SRC, R_WIN = cfg['H'], cfg['W'], cfg['D'], cfg['V'], cfg['r']
    stream_mode = cfg['kind'] == 'stream'
    ii = cfg['intr']
    cam = camera.make_cam_intrinsics(ii['fx'], ii['fy'], ii['cx'], ii['cy'], [W_IMG // 4, H_IMG // 4])
    d = synth.d_candidates(D_PLANES, ii['d'][0], ii['d'][1])

    def new_model():
        with contextlib.redirect_stdout(io.StringIO()):
            return KVNET(64, cam, d, 10., 64, None, t_win_r=R_WIN)
    model = new_model()
    # random-init weights of the reference architecture: rank 0 generates, NCCL broadcasts (weights only)
    if rank == 0:
        sd = arch.synth_state_dict(5, 64, D_PLANES, R_WIN, 64)
        model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    model = model.to(dev)
    model.conv_math = args.conv_math
    sharding.broadcast_module(model, src=0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    h, w = H_IMG // 4, W_IMG // 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ms_c, wk_c, n_c = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    sampler = ClockSampler(local)
    inflight = 1
    if not stream_mode:
        # ------------------------------------------------------------------ first-window frames (c2, c5)
        n_win = 4 if H_IMG * W_IMG <= 640 * 480 else 2
        wins = make_windows(cfg, n_win, seed=7 + rank)           # every rank owns its own windows (frames shard naturally)
        dev_frames = [torch.from_numpy(f).to(dev) for f, _ in wins]
        dev_poses = [torch.from_numpy(p).to(dev) for _, p in wins]
        pin_frames = [torch.from_numpy(f).pin_memory() for f, _ in wins]
        pin_poses = [torch.from_numpy(p).pin_memory() for _, p in wins]
        h2d_bytes = pin_frames[0].numel() * 4 + pin_poses[0].numel() * 4
        d2h_bytes = 2 * H_IMG * W_IMG * 4
        # `inflight` independent engines (own buffers, shared read-only weights) run consecutive frames on their own
        # streams so that one frame's kernels fill the other's tail waves
        inflight = max(1, args.inflight if args.inflight > 0 else cfg.get('inflight', 1))
        models = [model]
        for _ in range(inflight - 1):
            m2 = new_model()
            m2.load_state_dict(model.state_dict())
            m2 = m2.to(dev); m2.conv_math = args.conv_math
            models.append(m2)
        streams = [torch.cuda.current_stream()] + [torch.cuda.Stream(device=dev) for _ in range(inflight - 1)]
        hnds = []
        for m_, s_ in zip(models, streams):
            with torch.cuda.stream(s_), torch.no_grad():
                m_(dev_frames[0][-1:], dev_frames[0][None, :-1], dev_poses[0][None], torch.zeros(1), cam_intrinsics=[cam], BV_predict=None)
            hnds.append(m_._engine(H_IMG, W_IMG, V_SRC, dev)['h'])
        torch.cuda.synchronize()
        hnd, stream = hnds[0], streams[0]
        outs = [(torch.empty((D_PLANES, H_IMG, W_IMG), device=dev), torch.empty((D_PLANES, h, w), device=dev), torch.empty((h, w), device=dev))
                for _ in range(inflight)]

        def step_resident(i):
            k = i % inflight
            sk = streams[k]
            with torch.cuda.stream(sk):
                if k == 0:
                    flush.zero_()
                check(L.nrgbd_kvnet_forward(hnds[k], ptr(dev_frames[i % n_win]), ptr(dev_poses[i % n_win]), None, ptr(outs[k][0]), None,
                                            ptr(outs[k][1]), None, ptr(outs[k][2]), None, ctypes.c_void_p(sk.cuda_stream)))
        n_prime = inflight * n_win // math.gcd(inflight, n_win)
        for i in range(n_prime):          # untimed priming: every (engine, window) pointer tuple gets its CUDA graph captured
            step_resident(i)
        torch.cuda.synchronize()
        for i in range(Wm):
            step_resident(i)
        if rank == 0:
            sampler.start()
        barrier()
        L.nrgbd_reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for s_ in streams[1:]:
            s_.wait_stream(stream)
        for i in range(K):
            step_resident(Wm + i)
        for s_ in streams[1:]:
            stream.wait_stream(s_)
        e1.record(stream)
        barrier()
        launches = int(L.nrgbd_launch_count())
        ms_value = max_ms(e0.elapsed_time(e1), world, dev)
        if args.dump_outputs and rank == 0:
            last = outs[(Wm + K - 1) % inflight]
            dumped = sample_outputs({'dmap_cur_refined': last[0], 'bv_cur': last[1], 'depth_lowres': last[2]})

        def eager_frame(i):
            flush.zero_()
            check(L.nrgbd_kvnet_forward(hnd, ptr(dev_frames[i % n_win]), ptr(dev_poses[i % n_win]), None, ptr(outs[0][0]), None,
                                        ptr(outs[0][1]), None, ptr(outs[0][2]), None, ctypes.c_void_p(stream.cuda_stream)))
    else:
        # ------------------------------------------------------------------ streaming full KVNet (c3, c4)
        n_stream = cfg['n_stream']
        # `inflight` independent trajectory chunks stream concurrently on their own engines / CUDA streams (the same chunks
        # sharding.chunk_trajectory hands to different ranks at N > 1): one chunk's HBM-bound BatchNorm passes overlap the other's
        # tensor-bound K-Net convolutions. Every chunk keeps its own sequential recursion.
        inflight = max(1, args.inflight if args.inflight > 0 else cfg.get('inflight', 1))
        models = [model]
        for _ in range(inflight - 1):
            m2 = new_model()
            m2.load_state_dict(model.state_dict())
            m2 = m2.to(dev); m2.conv_math = args.conv_math
            models.append(m2)
        streams = [torch.cuda.current_stream()] + [torch.cuda.Stream(device=dev) for _ in range(inflight - 1)]
        trajs = []
        for t in range(inflight):
            frames, exts = make_video(cfg, n_stream + 2 * R_WIN, seed=7 + rank + 1000 * t)   # every rank / chunk streams its own trajectory
            dev_f = [torch.from_numpy(f[None]).to(dev) for f in frames]
            u8 = [np.ascontiguousarray(np.clip((f.transpose(1, 2, 0) * 0.226 + 0.45) * 255.0, 0, 255).astype(np.uint8)) for f in frames]
            tr = dict(exts=exts, pin_u8=[torch.from_numpy(a).pin_memory() for a in u8], win=[], pose=[], nxt=[])
            for i in range(n_stream):
                poses, idx = synth.window_rel_poses(exts, R_WIN + i, R_WIN)
                tr['win'].append(torch.cat([dev_f[j] for j in idx] + [dev_f[R_WIN + i]], 0).contiguous())
                tr['pose'].append(torch.from_numpy(np.ascontiguousarray(poses, np.float32)).to(dev))
                tr['nxt'].append(torch.from_numpy(np.linalg.inv(poses[R_WIN].astype(np.float64)).astype(np.float32)).to(dev))   # inverse of the (t+1) pose
            with torch.cuda.stream(streams[t]), torch.no_grad():
                models[t](tr['win'][0][-1:], tr['win'][0][None, :-1], tr['pose'][0][None], torch.zeros(1), cam_intrinsics=[cam], BV_predict=None)
            ent = models[t]._engine(H_IMG, W_IMG, V_SRC, dev)
            models[t]._set_camera(ent, 1, cam=cam)         # per-call intrinsics (K-Net image warp, propagation): the same camera here
            tr['h'] = ent['h']
            tr['o_ref'] = torch.empty((D_PLANES, H_IMG, W_IMG), device=dev)
            tr['o_cur'] = torch.empty((D_PLANES, H_IMG, W_IMG), device=dev)
            tr['o_dpv'] = torch.empty((D_PLANES, h, w), device=dev)
            tr['o_dep'] = torch.empty((h, w), device=dev)
            tr['priors'] = [torch.empty((D_PLANES, h, w), device=dev) for _ in range(2)]
            trajs.append(tr)
        torch.cuda.synchronize()
        pin_u8, exts = trajs[0]['pin_u8'], trajs[0]['exts']
        h2d_bytes = pin_u8[0].numel() + V_SRC * 64
        d2h_bytes = 2 * H_IMG * W_IMG * 4
        hnd = trajs[0]['h']
        stream = streams[0]

        def stream_step(i, have_prior):
            """One depth frame of one chunk's stream on resident inputs: forward (K-Net when a prior exists) + propagation."""
            t = i % inflight
            j = i // inflight
            k = j % n_stream
            tr = trajs[t]
            sp = ctypes.c_void_p(streams[t].cuda_stream)
            with torch.cuda.stream(streams[t]):
                if t == 0:
                    flush.zero_()
                if k == 0 or not have_prior:
                    check(L.nrgbd_kvnet_forward(tr['h'], ptr(tr['win'][k]), ptr(tr['pose'][k]), None, ptr(tr['o_ref']), None, None, None,
                                                ptr(tr['o_dep']), None, sp))
                else:
                    # both refined maps, like models/KVNET.py:93-185 returns them (R-Net runs on BV_cur AND on the K-Net DPV)
                    check(L.nrgbd_kvnet_forward(tr['h'], ptr(tr['win'][k]), ptr(tr['pose'][k]), ptr(tr['priors'][j % 2]), ptr(tr['o_cur']), ptr(tr['o_ref']),
                                                None, ptr(tr['o_dpv']), ptr(tr['o_dep']), None, sp))
                check(L.nrgbd_kvnet_propagate(tr['h'], None, ptr(tr['nxt'][k]), ptr(tr['priors'][(j + 1) % 2]), sp))
        for i in range(inflight):
            stream_step(i, False)
        for i in range(inflight, (3 + Wm) * inflight):     # warm-up: first window + steady-state graph capture
            stream_step(i, True)
        torch.cuda.synchronize()
        if rank == 0:
            sampler.start()
        barrier()
        L.nrgbd_reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for s_ in streams[1:]:
            s_.wait_stream(stream)
        base = (3 + Wm) * inflight
        for i in range(K):
            stream_step(base + i, True)                # a 30-frame window: the recursion restarts (first-window frame) every n_stream frames
        for s_ in streams[1:]:
            stream.wait_stream(s_)
        e1.record(stream)
        barrier()
        launches = int(L.nrgbd_launch_count())
        ms_value = max_ms(e0.elapsed_time(e1), world, dev)
        if args.dump_outputs and rank == 0:
            i = base + K - 1                            # the last timed step: which chunk, frame and prior slot stream_step used
            tr, j = trajs[i % inflight], i // inflight
            if j % n_stream == 0:
                last = {'dmap_cur_refined': tr['o_ref'], 'depth_lowres': tr['o_dep']}
            else:
                last = {'dmap_cur_refined': tr['o_cur'], 'dmap_refined': tr['o_ref'], 'dpv': tr['o_dpv'], 'depth_lowres': tr['o_dep']}
            last['bv_predict_next'] = tr['priors'][(j + 1) % 2]
            dumped = sample_outputs(last)

        def eager_frame(i):
            stream_step((1 + i % (n_stream - 1)) * inflight, True)      # chunk 0, a steady-state frame

    # ---------------- roofline pass: per-kernel CUDA events, eager, ONE frame in flight, right after the timed region -----------
    P_PROF = 4 if H_IMG * W_IMG * D_PLANES <= 1248 * 376 * 128 else 2
    check(L.nrgbd_kvnet_set_option(hnd, b'profile', 1))
    for cat in (0, 1, 2):
        L.nrgbd_kvnet_profile_read(hnd, cat, ctypes.byref(ms_c), ctypes.byref(wk_c), ctypes.byref(n_c))   # clear
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for i in range(P_PROF):
        eager_frame(i)
    p1.record(stream)
    torch.cuda.synchronize()
    prof_ms_total = p0.elapsed_time(p1)
    layer_rows = None
    if rank == 0:
        buf = ctypes.create_string_buffer(1 << 16)
        check(L.nrgbd_kvnet_profile_table(hnd, 0, buf, len(buf)))
        layer_rows = []
        for ln in buf.value.decode().splitlines():
            tag, n, ms, work = ln.split(';')
            layer_rows.append({'layer': tag, 'launches_per_frame': int(n) / P_PROF, 'ms_per_frame': float(ms) / P_PROF,
                               'algorithmic_tflops': float(work) / (float(ms) * 1e-3) / 1e12})
        layer_rows.sort(key=lambda r_: -r_['ms_per_frame'])
        if args.layer_table:
            with open(args.layer_table, 'w') as f:
                json.dump({'note': 'conv launches of one %s frame (%s), CUDA events around each launch in %d eager frames, one frame in flight'
                                   % (args.config, args.conv_math, P_PROF), 'frame_ms_eager': prof_ms_total / P_PROF, 'layers': layer_rows}, f, indent=1)
    check(L.nrgbd_kvnet_profile_read(hnd, 0, ctypes.byref(ms_c), ctypes.byref(wk_c), ctypes.byref(n_c)))
    conv_ms, conv_flops, conv_n = ms_c.value, wk_c.value, n_c.value
    check(L.nrgbd_kvnet_profile_read(hnd, 1, ctypes.byref(ms_c), ctypes.byref(wk_c), ctypes.byref(n_c)))
    sw_ms, sw_bytes, sw_n = ms_c.value, wk_c.value, n_c.value
    check(L.nrgbd_kvnet_set_option(hnd, b'profile', 0))
    value = world * K / (ms_value * 1e-3)

    # ---------------- e2e: public Python surface, pinned host buffers inside the timed region ----------------
    if not stream_mode:
        h_depth = [torch.empty((1, H_IMG, W_IMG)).pin_memory() for _ in range(inflight)]
        h_conf = [torch.empty((1, H_IMG, W_IMG)).pin_memory() for _ in range(inflight)]
        done_ev = [None] * inflight

        def consume(k):
            if done_ev[k] is not None:
                done_ev[k].synchronize()              # the user reads the depth map on the host

        def step_e2e(i):
            k = i % inflight
            consume(k)
            sk = streams[k]
            with torch.cuda.stream(sk):
                if k == 0:
                    flush.zero_()
                f = pin_frames[i % n_win].to(dev, non_blocking=True)
                p = pin_poses[i % n_win].to(dev, non_blocking=True)
                with torch.no_grad():
                    out = models[k](f[-1:], f[None, :-1], p[None], torch.zeros(1), cam_intrinsics=[cam], BV_predict=None)
                    dep, conf = misc.depth_val_regression(out[0], d, BV_log=True, return_conf=True)
                h_depth[k].copy_(dep, non_blocking=True)
                h_conf[k].copy_(conf, non_blocking=True)
                ev = torch.cuda.Event(); ev.record(sk); done_ev[k] = ev
        for i in range(n_prime + Wm):
            step_e2e(i)
        for k in range(inflight):
            consume(k); done_ev[k] = None
        barrier()
        e0.record(stream)
        for s_ in streams[1:]:
            s_.wait_stream(stream)
        for i in range(K):
            step_e2e(Wm + i)
        for k in range(inflight):
            consume(k)
        for s_ in streams[1:]:
            stream.wait_stream(s_)
        e1.record(stream)
        barrier()
        host_depth = h_depth[0]
    else:
        # the reference's streaming loop (test_KVNet.py:190-250) on the mirrors: one new decoded frame per step and chunk
        fws = [m_preprocess.FrameWindow(t_win_r=R_WIN, img_size=None, device=dev) for _ in range(inflight)]
        h_depths = [torch.empty((H_IMG, W_IMG)).pin_memory() for _ in range(inflight)]
        h_confs = [torch.empty((H_IMG, W_IMG)).pin_memory() for _ in range(inflight)]
        states = [{'bv': None, 'pos': 0, 'ev': None} for _ in range(inflight)]

        def consume(t):
            if states[t]['ev'] is not None:
                states[t]['ev'].synchronize()          # the user reads this chunk's maps on the host before its next frame arrives
                states[t]['ev'] = None

        def step_e2e(i):
            t = i % inflight
            consume(t)
            state, fw, tr = states[t], fws[t], trajs[t]
            with torch.cuda.stream(streams[t]):
                if t == 0:
                    flush.zero_()
                if state['pos'] == 0 or state['pos'] >= len(tr['pin_u8']):      # new trajectory chunk: refill the window, restart the recursion
                    fw.frames.clear(); state['bv'] = None
                    for j in range(2 * R_WIN):
                        fw.push(tr['pin_u8'][j], tr['exts'][j])
                    state['pos'] = 2 * R_WIN
                k = state['pos']; state['pos'] += 1
                fw.push(tr['pin_u8'][k], tr['exts'][k])       # H2D: ONE decoded uint8 frame; the other 2r frames of the window are resident
                fds = fw.frame_dicts()
                ref_d, src_d = fds[R_WIN], [fd for j, fd in enumerate(fds) if j != R_WIN]
                inv_ref = np.linalg.inv(ref_d['extM'])
                poses = np.stack([fd['extM'].dot(inv_ref) for fd in src_d]).astype(np.float32)      # warping.homography.get_rel_extrinsicM
                poses_t = torch.from_numpy(poses[None]).to(dev, non_blocking=True)
                dmap, bv = step_mod.test(models[t], d, [cam], R_WIN, [ref_d], [src_d], poses_t, state['bv'], R_net=True)
                maps = export_res.depth_conf_maps(dmap, d, want_float=True, want_u16=False)
                h_depths[t].copy_(maps['dmap'], non_blocking=True)
                h_confs[t].copy_(maps['conf'], non_blocking=True)
                ev = torch.cuda.Event(); ev.record(streams[t]); state['ev'] = ev
                state['bv'] = bv
        for i in range((3 + Wm) * inflight):
            step_e2e(i)
        for t in range(inflight):
            consume(t)
        barrier()
        e0.record(stream)
        for s_ in streams[1:]:
            s_.wait_stream(stream)
        for i in range(K):
            step_e2e((3 + Wm) * inflight + i)
        for t in range(inflight):
            consume(t)
        for s_ in streams[1:]:
            stream.wait_stream(s_)
        e1.record(stream)
        barrier()
        h_depth = h_depths[0]
        host_depth = h_depth
    e2e_value = world * K / (max_ms(e0.elapsed_time(e1), world, dev) * 1e-3)
    sampler.stop = True
    assert np.isfinite(host_depth.numpy()).all()

    if rank == 0:
        conv_tflops = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        sweep_gbs = sw_bytes / (sw_ms * 1e-3) / 1e9 if sw_ms > 0 else 0.0
        peak_tf = peaks['bf16_sustained']       # kernels timed inside a long step -> sustained figure
        kname = {'f16x3': 'conv_h2_kernel (tcgen05 kind::f16 on split-fp16 operand pairs, halo tile, persistent CTAs; algorithmic fp32 FLOPs, the MMA rate is 3x this)',
                 'tf32x3': 'conv_tc2_kernel (tcgen05 3xTF32 implicit GEMM; algorithmic fp32 FLOPs, the MMA rate is 3x this)',
                 'fp32': 'conv_igemm_kernel<128,{32,64}> (fp32 FFMA implicit GEMM)'}[args.conv_math]
        dtype = {'f16x3': 'f32 (split-fp16 pair products: 22-bit significands, fp32 accumulate)', 'tf32x3': 'f32 (3xTF32 error-compensated products, fp32 accumulate)',
                 'fp32': 'f32'}[args.conv_math]
        line = {
            'metric': cfg['metric'], 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': Wm, 'ms_per_step': ms_value / K,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': dtype, 'data': 'synthetic',
            'config': {'workload': cfg['workload'], 'name': args.config, 'conv_math': args.conv_math, 'planes': D_PLANES, 'views': V_SRC, 'frame': [H_IMG, W_IMG],
                       'parallelism': 'dp%d (%s sharded, weights NCCL-broadcast once)' % (world, 'trajectory chunks' if stream_mode else 'frames'),
                       'l2': 'explicit 256 MiB flush write before every %s step (inside the timed region)' % ('' if inflight == 1 else '%d-th' % inflight),
                       'frames_in_flight': inflight,
                       'in_flight_unit': 'independent trajectory chunks, each with its own sequential recursion' if stream_mode else 'independent first-window frames',
                       'weights': 'random init of the reference architecture (arch.synth_state_dict seed 5)',
                       'hbm_kernels': {'plane_sweep': {'avg_us': 1e3 * sw_ms / max(sw_n, 1), 'algorithmic_GBps': sweep_gbs, 'frac_of_hbm_peak': sweep_gbs / peaks['hbm_gbs'],
                                                       'note': 'fused plane-sweep (+ log-softmax) kernel; at C = 67 it is gather / FFMA bound, not HBM bound (SURVEY 8d)'}},
                       'conv_share_of_step': conv_ms / prof_ms_total if prof_ms_total > 0 else None,
                       'cuda_graph': 'each frame is one cudaGraphLaunch (captured per I/O pointer tuple after an eager warm-up)'},
            'e2e': {'value': e2e_value, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': d2h_bytes},
            'gpu_launches': launches,
            'clocks': sampler.summary(),
            'roofline': {'bound': 'tensor', 'achieved': conv_tflops, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': conv_tflops / peak_tf,
                         'traffic': conv_traffic_per_launch() if (args.conv_math == 'f16x3' and args.config == 'c2') else None,
                         'kernel': kname + ', %d launches/step, avg %.1f us' % (conv_n // P_PROF, 1e3 * conv_ms / max(conv_n, 1)),
                         'regime': {'what': 'CUDA events around every conv launch in %d eager frames, ONE frame in flight, run right after the timed region' % P_PROF,
                                    'frames_per_s_in_this_regime': 1e3 * P_PROF / prof_ms_total, 'frame_ms': prof_ms_total / P_PROF},
                         'traffic_note': 'bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum, mean over the conv launches of one c2 frame, ncu capture of this '
                                         "round's kernels (profiles/r2_conv_dram_traffic.json)",
                         'peak_source': peaks['source'] + ', sustained bf16'},
        }
        if args.conv_math in ('f16x3', 'tf32x3'):
            # `achieved` counts each fp32 product ONCE (the algorithmic FLOPs the contract asks for); the tensor pipe executes three
            # half-precision (or TF32) products per algorithmic one, so its own utilisation is three times `frac` (f16) - reported
            # here so that both readings are on the line
            mult = 3.0
            mma_peak = peak_tf if args.conv_math == 'f16x3' else peak_tf / 2.0
            line['roofline']['mma_issue_rate'] = {'achieved': mult * conv_tflops, 'peak': mma_peak, 'unit': 'TFLOP/s', 'frac': mult * conv_tflops / mma_peak,
                                                  'note': 'executed tensor-core FLOPs (3 error-compensating MMAs per fp32 product) against the dense %s rate'
                                                          % ('f16/bf16' if args.conv_math == 'f16x3' else 'tf32 (half the bf16)')}
        if layer_rows:
            line['config']['top_conv_layers'] = [{'layer': r_['layer'], 'n': r_['launches_per_frame'], 'ms': round(r_['ms_per_frame'], 4),
                                                  'tflops': round(r_['algorithmic_tflops'], 1)} for r_ in layer_rows[:4]]
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline_subprocess(args)
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dumped)
        _emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


_emit = print


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='engine', choices=['engine', 'reference', 'reference-gpu'])
    ap.add_argument('--config', default='c2', choices=sorted(CONFIGS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--layer-table', default=None, help='write the per-shape conv table of the roofline pass to this JSON file')
    ap.add_argument('--inflight', type=int, default=0, help='independent frames (first-window configs) or trajectory chunks (streaming configs) in flight on separate CUDA streams; 0 = the config default')
    ap.add_argument('--dev-bn-unroll', type=int, default=0, help='development: vectors in flight per thread in the BatchNorm pass')
    ap.add_argument('--dev-smem-cap-kb', type=int, default=0, help='development: cap conv_h2 shared memory (co-residency experiment)')
    ap.add_argument('--conv-math', default='f16x3', choices=['fp32', 'tf32x3', 'f16x3'],
                    help='f16x3: tcgen05 kind::f16 on split-fp16 pairs (default); tf32x3: tcgen05 3xTF32; fp32: exact CUDA-core FFMA implicit GEMM')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write what the last timed step returned to DIR/<name>.npy (float32, at most 64 MB in all; larger outputs as a fixed seeded sample)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'engine':
        ap.error('--dump-outputs applies to the engine arm')
    cfg = CONFIGS[args.config]
    args.warmup = max(args.warmup, 3) if args.impl == 'engine' else args.warmup
    # stdout carries exactly one JSON line: anything a library prints there meanwhile (e.g. NCCL's version banner with
    # NCCL_DEBUG set) is sent to stderr by pointing fd 1 at fd 2 until the result line is written to the real stdout
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    _emit = lambda text: os.write(real_stdout, (text + '\n').encode())      # noqa: E731
    if args.impl == 'reference':
        # the CPU arm must not see a GPU: with visible devices nn.DataParallel (test_KVNet.py:163) scatters the inputs to cuda:0
        # while the .cuda() shim keeps everything else on the host
        os.environ['CUDA_VISIBLE_DEVICES'] = ''
        run_reference(args, cfg, on_gpu=False)
    elif args.impl == 'reference-gpu':
        run_reference(args, cfg, on_gpu=True)
    elif cfg['kind'] == 'sweep':
        run_sweep(args, cfg)
    else:
        run_engine(args, cfg)


if __name__ == '__main__':
    main()
