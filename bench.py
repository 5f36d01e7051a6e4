#!/usr/bin/env python
"""Benchmark of the GIMS matcher forward path on B200 — BASELINE.json metric: image pairs/sec at
2048 keypoints/image (configs[1]: fp32, 100 Sinkhorn iterations, r/p/m = 25/7/8).

  python bench.py --gpus N --steps K --warmup W            our CUDA path
  python bench.py --impl reference ...                     the reference's own CPU implementation on the host cores:
                                                           the UNMODIFIED reference modules (oracle/_ref, a git-ignored
                                                           copy made by __graft_entry__.build(), or GIMS_REFERENCE_ROOT;
                                                           run under oracle/ref_shims) or, if absent, the oracle port
  --kpts N                                                 keypoints per image (BASELINE configs[3] = 4096, configs[4] = 8192)
  --weights random|damped                                  random-init weights (degenerate scores: mean 0.3, std 0.002) or
                                                           the non-degenerate "damped" set (scores ~ 90 +- 2.6 like a trained net)
A step = one batch of `--pairs-per-step` synthetic pairs per GPU through the whole hot path
(AGC graphs -> SAGE -> kenc -> 18 attention layers -> scores -> Sinkhorn -> matches).
`value`   : pairs/s, inputs already resident in HBM, pairs issued over several CUDA streams.
`e2e`     : pairs/s through the reference-facing call `Matching(config)(data)` with pinned HOST tensors
            (H2D of keypoints/descriptors/scores and D2H of matches/scores inside the timed region), issued by
            `--e2e-threads` host threads with one CUDA stream each; `single_thread_value` = one caller.
`roofline`: dominant kernel, timed live with CUDA events inside the library on its own stream.
Multi-GPU: one process per GPU (torchrun), pairs sharded, no collective on the data path (weak scaling).
`--dump-outputs DIR` writes what the last timed step returned (see `dump_outputs`) so that two builds can be compared
output for output: the inputs depend only on the arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from gims_b200.synth import make_pair, make_state_dict  # noqa: E402

UNIT = 'pairs/s'
FALLBACK_PEAKS = {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}
DUMP_LIMIT_BYTES = 64 * 10 ** 6           # --dump-outputs, all files


def metric_name(kpts):
    return 'image_pairs_per_sec_%dkp' % kpts


def workload_name(args):
    cfg = {2048: 'configs[1]', 4096: 'configs[3]', 8192: 'configs[4]'}.get(args.kpts, 'custom size')
    return ('BASELINE %s: GMatcher forward, %d kp/image, fp32, 100 Sinkhorn it, AGC r/p/m 25/7/8, %s weights'
            % (cfg, args.kpts, 'random-init' if args.weights == 'random' else 'random-init "damped" (non-degenerate)'))


def adjust_sizes(args):
    """Keep the step (and the per-stream workspaces) bounded at the large configs; both arms call this."""
    if args.kpts > 2048:
        scale = (args.kpts // 2048) ** 2
        args.pairs_per_step = max(4, args.pairs_per_step // scale)
        args.streams = max(2, min(args.streams, args.pairs_per_step))
        args.pool = max(8, args.pool // scale)


def pair_input_bytes(kpts):
    return 2 * (kpts * 2 + 256 * kpts + kpts) * 4


def base_config(args, world):
    """The `config` object of the JSON line — identical for `--impl ours` and `--impl reference`."""
    return {'workload': workload_name(args), 'kpts_per_image': args.kpts, 'weights': args.weights,
            'sinkhorn_iterations': 100, 'agc_radius_percentile_minsize': [25, 7, 8],
            'pairs_per_step_per_gpu': args.pairs_per_step, 'streams': args.streams,
            'pairs_per_launch': args.pairs_per_launch,
            'l2': 'input pool of %d distinct pairs (%.0f MB) > L2' % (args.pool, args.pool * pair_input_bytes(args.kpts) / 1e6),
            'parallelism': 'pair-parallel x%d, no collective' % world}


def ncu_traffic(kernel):
    """dram__bytes_read + write per launch of `kernel` from the newest committed `ncu --set full` summary under
    profiles/ (lines `<kernel> dram_bytes_read=<n> dram_bytes_write=<n>`); None if there is no such capture."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_ncu_full_metrics.txt')), reverse=True):
        with open(path) as fh:
            for ln in fh:
                m = re.match(r'\s*%s\S*\s.*dram_bytes_read=(\d+)\s+dram_bytes_write=(\d+)' % re.escape(kernel), ln)
                if m:
                    return int(m.group(1)) + int(m.group(2)), os.path.relpath(path, ROOT)
    return None, None


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        d['_source'] = 'measured'
        return d
    d = dict(FALLBACK_PEAKS)
    d['_source'] = 'fallback'
    return d


def projection_flops(n0, n1, layers=18, d=256):
    """Algorithmic FLOPs of the per-node linear maps of one pair (q/k/v/merge, MLP, kenc, SAGE, final_proj)."""
    per_node = layers * (4 * 2 * d * d + 2 * (2 * d) * (2 * d) + 2 * (2 * d) * d) + 2 * 108608 + \
        2 * (2 * 256 * 128 + 2 * 128 * 128 + 2 * 128 * 256) + 2 * d * d
    return per_node * (n0 + n1)


def pair_flops(n0, n1, layers=18, d=256):
    """Algorithmic FLOPs of one pair (SURVEY.md §8d), N = surviving keypoints per image."""
    per_node = layers * (4 * 2 * d * d + 2 * (2 * d) * (2 * d) + 2 * (2 * d) * d) + 2 * 108608 + \
        2 * (2 * 256 * 128 + 2 * 128 * 128 + 2 * 128 * 256) + 2 * d * d
    attn = 0
    for l in range(layers):
        cross = l % 2 == 1
        attn += 2 * 2 * d * (n0 * (n1 if cross else n0) + n1 * (n0 if cross else n1))
    return per_node * (n0 + n1) + attn + 2 * n0 * n1 * d


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every 2 ms from a
    host thread; falls back to an `nvidia-smi -lms` child process if NVML is not usable."""

    REASONS = ((0x4, 'sw_power_cap'), (0x8, 'hw_slowdown'), (0x20, 'sw_thermal_slowdown'), (0x40, 'hw_thermal_slowdown'),
               (0x80, 'hw_power_brake_slowdown'))

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []
        self.mask = 0
        self.stop_flag = False

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith('GPU-'):
                uuid = 'GPU-' + uuid
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, 'encode') else uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def _poll(self):
        pynvml, h = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        try:
            self.nvml = self._nvml_handle()
            pynvml, h = self.nvml
            self.smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            sm = sorted(self.samples)
            return {'sm_mhz': float(sm[len(sm) // 2]) if sm else None, 'sm_min_mhz': float(sm[0]) if sm else None,
                    'sm_max_mhz': float(self.smax), 'reasons': [n for b, n in self.REASONS if self.mask & b],
                    'samples': len(sm), 'source': 'nvml, 2 ms period'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {'sm_mhz': med, 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi'}


def dump_outputs(path, outs, kpts):
    """Write what one step of `PairBatchRunner.run` returned to its caller, pairs in step order, as `path/<name>.npy`:
      counts.npy            (P, 8) float64  the library's per-pair counters: N' of both images, edges, components, status
      matches0.npy          (sum of N'0,) float64  per pair, for each kept keypoint of image 0: the index of its match
                            among the kept keypoints of image 1, or -1; pairs one after the other (counts[:, 0] splits them)
      matching_scores0.npy  (sum of N'0,) float32  laid out like matches0
      pair_index.npy        (P,) float64  position of each pair in the step
    When the pairs could exceed DUMP_LIMIT_BYTES, a fixed seeded sample of them is written instead."""
    import numpy as np
    per_pair = 9 * 8 + kpts * (8 + 4)                  # N'0 <= kpts
    room = DUMP_LIMIT_BYTES - 4 * 128                   # .npy headers
    idx = np.arange(len(outs))
    if len(outs) * per_pair > room:
        idx = np.sort(np.random.default_rng(0).choice(len(outs), room // per_pair, replace=False))
    counts = np.stack([outs[i]['n_kept_dev'].cpu().numpy() for i in idx]).astype(np.float64)
    kept = [int(c) for c in counts[:, 0]]
    matches = np.concatenate([outs[i]['matches0'][:n].cpu().numpy() for i, n in zip(idx, kept)]).astype(np.float64)
    scores = np.concatenate([outs[i]['mscores0'][:n].cpu().numpy() for i, n in zip(idx, kept)]).astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for name, arr in (('counts', counts), ('matches0', matches), ('matching_scores0', scores),
                      ('pair_index', idx.astype(np.float64))):
        np.save(os.path.join(path, name + '.npy'), arr)


def measure_tf32_peak(dev):
    """Dense TF32 tensor throughput of this GPU (cuBLAS, 8192^3), measured like MEASURED_PEAKS.json's bf16 number
    (SURVEY.md 8d asks for it: the file has no TF32 entry).  Used only as a roofline denominator."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(8192, 8192, device=dev)
        b = torch.randn(8192, 8192, device=dev)
        for _ in range(3):
            c = a @ b
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            c = a @ b
        e1.record()
        torch.cuda.synchronize(dev)
        del c
        return 10 * 2.0 * 8192 ** 3 / (e0.elapsed_time(e1) / 1e3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def _reference_runner(args):
    """Callable one(seed) that runs one pair of the bench workload through the reference's CPU implementation, and
    a description of what it is.  Preferred: the unmodified reference modules (ref_shims.REFERENCE_ROOT: the
    git-ignored copy in oracle/_ref made by __graft_entry__.build(), or GIMS_REFERENCE_ROOT) imported under
    oracle/ref_shims.py.  Fallback: the oracle port."""
    import contextlib
    import io
    sd = make_state_dict(0, damped=(args.weights == 'damped'))
    cfg = {'sinkhorn_iterations': 100, 'match_threshold': 0.2}
    from oracle import ref_shims
    if ref_shims.reference_available() and not os.environ.get('GIMS_BENCH_FORCE_PORT'):
        _, gm = ref_shims.load_reference()
        model = gm.GMatcher(cfg)
        model.load_state_dict(sd)
        model.eval()

        def one(seed):
            data = make_pair(args.kpts, seed=seed)
            data.update({'radius': 25, 'percentile': 7, 'min_size': 8, 'device': torch.device('cpu')})
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                return model(data)
        return one, 'reference', 'unmodified reference models/{agc,gmatcher}.py under oracle/ref_shims.py'
    from oracle import gims_oracle as orc

    def one(seed):
        data = make_pair(args.kpts, seed=seed)
        data.update({'radius': 25, 'percentile': 7, 'min_size': 8})
        with torch.no_grad():
            return orc.gmatcher_forward(sd, data, cfg)
    return one, 'port', 'oracle/gims_oracle.py (port of the reference)'


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    one, kind, what = _reference_runner(args)
    # each step is one pair on the host (seconds at 2048 keypoints, most of a minute at 8192)
    steps = args.steps
    for w in range(args.warmup):
        one(1000 + w)
    t0 = time.perf_counter()
    for s in range(steps):
        one(2000 + s)
    dt = time.perf_counter() - t0
    val = steps / dt
    line = {
        'impl': 'reference', 'metric': metric_name(args.kpts), 'value': val, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': base_config(args, world),
        'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': kind,
                         'sample': 'one pair per step, %d steps timed, %s, torch %d threads' % (steps, what, cores)},
        'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def cpu_baseline(args):
    """Rank 0, N = 1: the CPU arm on a bounded sample (10-60 s) of the same workload, timed beside the GPU number."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    one, kind, what = _reference_runner(args)
    n = 3 if args.kpts <= 2048 else 1
    if args.kpts <= 4096:
        one(1000)
    t0 = time.perf_counter()
    for s in range(n):
        one(2000 + s)
    dt = time.perf_counter() - t0
    return {'value': n / dt, 'unit': UNIT, 'cores': cores, 'kind': kind,
            'sample': '%d pair(s) at %d kp, %s, torch %d threads' % (n, args.kpts, what, cores)}


def load_caller_carhynet(dev):
    """The CALLER's descriptor object of the pipeline config: the reference's CAR_HyNet (random init — the trained
    weights are not in the reference tree) from the reference under oracle/ref_shims.py's REFERENCE_ROOT, wrapped like
    carhynet/models.py:639-670 `HyNetnetFeature2D` (whose __init__ hard-loads ./weights/car_hynet.pth)."""
    from oracle import ref_shims
    ref_root = ref_shims.REFERENCE_ROOT
    if not os.path.isfile(os.path.join(ref_root, 'carhynet', 'models.py')):
        return None
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    import importlib
    hm = importlib.import_module('carhynet.models')
    torch.manual_seed(0)
    car = object.__new__(hm.HyNetnetFeature2D)
    car.G_dim, car.do_cuda, car.device, car.batch_size = 128, True, dev, 512
    car.model = hm.CAR_HyNet().to(dev).eval()
    return car


def run_pipeline(args):
    """BASELINE configs[2].  One JSON line: pairs/s of the whole `matching({'image0', 'image1', 'carhynet', ...})` call
    (eval_homography.py:177: AGC r/p/m 15/2/7, 20 Sinkhorn iterations) and its stage split."""
    from gims_b200 import Matching, _lib, frontend
    from gims_b200.synth import make_textured_image, warp_image
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', 0)))
    torch.cuda.set_device(dev)
    car = load_caller_carhynet(dev)
    if car is None:
        print(json.dumps({'metric': 'pipeline_pairs_per_sec_800x600', 'unavailable': 'the reference\'s carhynet/ is missing '
                          '(run __graft_entry__.build() with GIMS_REFERENCE_ROOT set to a reference checkout)'}))
        return
    max_kp = args.kpts
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.2, 'max_keypoints': max_kp})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=(args.weights == 'damped')))
    matching = matching.eval().to(dev)
    n_pairs = args.steps
    pairs = []
    for i in range(n_pairs + 1):
        img0 = make_textured_image(600, 800, seed=100 + i)
        img1, _ = warp_image(img0, seed=200 + i)
        pairs.append((img0[None], img1[None]))                 # (1, H, W, 3) as frame2tensor(color=True) gives
    def call(p):
        with torch.no_grad():
            pred = matching({'delaunay': False, 'image0': p[0], 'image1': p[1], 'carhynet': car, 'device': dev,
                             'radius': 15, 'percentile': 2, 'min_size': 7})
        out = {k: v[0].cpu().numpy() for k, v in pred.items()}       # eval_homography.py:181
        return out
    call(pairs[0])
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    kept = []
    for p in pairs[1:]:
        out = call(p)
        kept.append((int(out['keypoints0'].shape[0]), int(out['keypoints1'].shape[0]), int((out['matches0'] >= 0).sum())))
    torch.cuda.synchronize(dev)
    dt = (time.perf_counter() - t0) / n_pairs
    # stage split on the last pair
    t = {}
    a = time.perf_counter()
    kps = [frontend.detect(im[0], max_kp) for im in pairs[-1]]
    t['sift_detect_host_ms'] = 1e3 * (time.perf_counter() - a)
    a = time.perf_counter()
    levels = [frontend.gaussian_pyramid(im[0]) for im in pairs[-1]]
    t['pyramid_host_ms'] = 1e3 * (time.perf_counter() - a)
    host_patches = os.environ.get('GIMS_HOST_PATCHES') == '1'
    a = time.perf_counter()
    if host_patches:
        patches = [frontend.extract_patches(k, lv) for k, lv in zip(kps, levels)]
        t['patches_host_ms'] = 1e3 * (time.perf_counter() - a)
    else:
        patches = [frontend.extract_patches_device(k, lv, dev) for k, lv in zip(kps, levels)]
        torch.cuda.synchronize(dev)
        t['patches_gpu_ms_incl_pyramid_upload'] = 1e3 * (time.perf_counter() - a)
    torch.cuda.synchronize(dev)
    a = time.perf_counter()
    descs = [frontend.describe(p, car, dev) for p in patches]
    torch.cuda.synchronize(dev)
    t['carhynet_gpu_ms'] = 1e3 * (time.perf_counter() - a)
    data = {'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7, 'image0': pairs[-1][0], 'image1': pairs[-1][1]}
    for s, (k, d) in enumerate(zip(kps, descs)):
        data['keypoints%d' % s] = torch.tensor([x.pt for x in k], device=dev)[None]
        data['scores%d' % s] = torch.tensor([x.response for x in k], device=dev)[None]
        data['descriptors%d' % s] = torch.cat([d, d], 1).t()[None].contiguous()
    with torch.no_grad():
        matching(dict(data))
    torch.cuda.synchronize(dev)
    a = time.perf_counter()
    for _ in range(5):
        with torch.no_grad():
            pred = matching(dict(data))
        pred['matches0'].cpu()
    t['matcher_gpu_ms'] = 1e3 * (time.perf_counter() - a) / 5
    print(json.dumps({
        'metric': 'pipeline_pairs_per_sec_800x600', 'value': 1.0 / dt, 'unit': UNIT, 'n_gpus': 1, 'steps': n_pairs,
        'ms_per_pair': 1e3 * dt, 'higher_is_better': True, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'BASELINE configs[2]: eval_homography-shaped pipeline, synthetic 800x600 colour image pairs, '
                               'cv2 SIFT (max_keypoints %d) + Gaussian pyramid on the host, 64->32 px patches %s, random-init '
                               'CAR_HyNet on the GPU, matcher with AGC r/p/m 15/2/7 and 20 Sinkhorn iterations; one caller, '
                               'sequential pairs' % (max_kp, 'on the host (cv2 per keypoint)' if host_patches else
                                                     'on the GPU (gims_extract_patches, bit-identical to cv2)')},
        'kept_keypoints_and_matches': kept, 'stage_ms_last_pair': {k: round(v, 2) for k, v in t.items()},
        'reference_published': '14.2-17.2 s per pair (README.md:116-120, unstated GPU, trained weights, all keypoints)'}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--kpts', type=int, default=2048)
    ap.add_argument('--pairs-per-step', type=int, default=24)
    ap.add_argument('--streams', type=int, default=12)
    ap.add_argument('--e2e-threads', type=int, default=8)
    ap.add_argument('--pool', type=int, default=40, help='distinct resident input pairs (> L2 in total)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--prof-kernel', default='attention')
    ap.add_argument('--weights', default='random', choices=['random', 'damped'])
    ap.add_argument('--pairs-per-launch', type=int, default=2,
                    help='pairs stacked into one gims_forward_pairs call (shared GEMM / attention launches)')
    ap.add_argument('--gemm-mode', default=None, choices=['simt', 'tf32', 'f16', 'bf16'],
                    help='arithmetic of the dense contractions (default: f16 = fp16 hi+lo attention operands, fp32 parity); '
                         'bf16 is the separately reported bf16 variant')
    ap.add_argument('--pipeline', action='store_true',
                    help='BASELINE configs[2]: eval_homography-shaped pipeline (synthetic 800x600 image pairs -> SIFT + '
                         'patches on the host -> CAR-HyNet on the GPU -> matcher), the literal call of eval_homography.py:177')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.pipeline or args.impl != 'ours'):
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours, without --pipeline)')
    if args.pipeline:
        run_pipeline(args)
        return
    METRIC = metric_name(args.kpts)
    adjust_sizes(args)

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch.distributed as dist
    from gims_b200 import Matching, _lib
    from gims_b200.engine import PairBatchRunner

    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    L = _lib.lib()
    if args.gemm_mode:
        L.gims_set_gemm_mode(_lib.GEMM_MODES[args.gemm_mode])
    gemm_mode_name = {0: 'simt (fp32 CUDA cores)', 1: 'tf32x3', 2: 'fp16 hi+lo operands (3 MMAs per fp32 product) in attention and projections',
                      3: 'bf16 attention operands + fp16 hi+lo projections (bf16 variant, not fp32 parity)'}[L.gims_get_gemm_mode()]

    cfg = {'sinkhorn_iterations': 100, 'match_threshold': 0.2}
    matching = Matching(cfg)
    matching.gmodel.load_state_dict(make_state_dict(0, damped=(args.weights == 'damped')))
    matching = matching.eval().to(dev)
    gm = matching.gmodel

    # resident input pool: distinct pairs, total bytes > L2 so no step re-reads inputs from cache
    P = args.pairs_per_step
    pool_host = [make_pair(args.kpts, seed=10000 * (rank + 1) + i) for i in range(args.pool)]
    pool = []
    for d in pool_host:
        pool.append({'keypoints0': d['keypoints0'][0].to(dev), 'keypoints1': d['keypoints1'][0].to(dev),
                     'descriptors0': d['descriptors0'][0].to(dev), 'descriptors1': d['descriptors1'][0].to(dev),
                     'scores0': d['scores0'][0].to(dev), 'scores1': d['scores1'][0].to(dev),
                     'shape0': d['image0'].shape, 'shape1': d['image1'].shape})
    in_bytes = sum(v.numel() * 4 for k, v in pool[0].items() if torch.is_tensor(v))
    runner = PairBatchRunner(gm, n_streams=args.streams, pairs_per_launch=args.pairs_per_launch)
    cursor = [0]

    def step():
        batch = [pool[(cursor[0] + i) % len(pool)] for i in range(P)]
        cursor[0] += P
        return runner.run(batch)

    for _ in range(args.warmup):
        outs = step()
    torch.cuda.synchronize(dev)
    counts = outs[0]['n_kept_dev'].cpu().tolist()
    if counts[6] & _lib.STATUS_ERROR_MASK:
        raise RuntimeError('error status %#x in the benchmark workload' % counts[6])
    sink_path = 'fast (exp-free scaled-kernel iteration)' if counts[6] & _lib.STATUS_SINKHORN_FAST else \
        'exact (log-sum-exp iteration)'
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.gims_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        outs = step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = L.gims_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, args.kpts)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * P * args.steps / (ms / 1e3)

    # --- roofline of the dominant kernel: CUDA events inside the library, same workload, one stream ----------
    import ctypes as C
    roof = None
    if rank == 0:
        peaks = load_peaks()
        L.gims_profile_begin(_lib.PROF[args.prof_kernel], 4096)
        torch.cuda.synchronize(dev)
        outs1 = PairBatchRunner(gm, n_streams=1, pairs_per_launch=args.pairs_per_launch).run([pool[i % len(pool)] for i in range(2 * args.pairs_per_launch)])
        torch.cuda.synchronize(dev)
        tot, cnt = C.c_double(0), C.c_int(0)
        L.gims_profile_end(C.byref(tot), C.byref(cnt))
        c = outs1[0]['n_kept_dev'].cpu().tolist()
        n0k, n1k = c[0], c[1]
        if cnt.value:
            avg_s = tot.value / cnt.value / 1e3
            if args.prof_kernel == 'attention':
                try:
                    tf32_peak = measure_tf32_peak(dev)
                except Exception:      # noqa: BLE001 - the extra denominator is optional
                    tf32_peak = None
                # QK^T + PV over 4 heads x 64: 4*D*nq*nk per image; averaged over self / cross layers
                flops = 2.0 * 256 * (n0k + n1k) ** 2 * args.pairs_per_launch     # one launch serves the whole batch
                ach = flops / avg_s / 1e12
                mode = L.gims_get_gemm_mode()
                kname = 'k_attention_tc' if mode == _lib.GEMM_TC else 'k_attention_f16'
                traffic, traffic_src = (None, None)
                if args.kpts == 2048 and args.pairs_per_launch == 2 and mode == _lib.GEMM_TC_F16:
                    traffic, traffic_src = ncu_traffic(kname)
                peak = peaks['bf16_tflops_sustained']
                # fp32 parity = error-compensated products: 3 kind::f16 MMAs per product (fp16 hi + lo planes) -> an
                # fp32-exact kernel cannot exceed 1/3 of the bf16 peak (1/6 with the 3xTF32 kernels, 1 for the bf16 variant);
                # `frac` is against the full bf16 peak as the contract asks
                mmas = {_lib.GEMM_TC: 6.0, _lib.GEMM_TC_F16: 3.0, _lib.GEMM_BF16: 1.0}.get(mode, 3.0)
                roof = {'kernel': kname, 'bound': 'tensor', 'achieved': ach, 'peak': peak,
                        'unit': 'TFLOP/s', 'frac': ach / peak, 'traffic': traffic,
                        'traffic_source': ('dram__bytes_read+write per launch, %s (algorithmic per 2-pair launch: Q fp32 8.4 MB + '
                                           'K and Vt fp16 hi/lo planes 16.8 MB)' % traffic_src) if traffic else
                                          'no ncu capture for this configuration',
                        'ceiling_frac': 1.0 / mmas, 'frac_of_ceiling': ach / peak * mmas,
                        'tf32_dense_tflops_measured': tf32_peak,
                        'ceiling_note': '%d bf16-rate-equivalent MMAs per fp32 product (error compensation); tensor-pipe work '
                                        'actually issued = achieved x %d = %.0f TFLOP/s' % (mmas, mmas, ach * mmas),
                        'peak_source': peaks['_source'] + ' bf16 sustained', 'launches_timed': cnt.value,
                        'avg_launch_ms': avg_s * 1e3, 'flops_per_launch': flops, 'pairs_per_launch': args.pairs_per_launch}
            elif args.prof_kernel == 'sinkhorn':
                byts = 4.0 * (n0k + 1) * (n1k + 1)
                ach = byts / avg_s / 1e9
                peak = peaks['hbm_gbs']
                traffic, traffic_src = ncu_traffic('k_sinkhorn') if args.kpts == 2048 else (None, None)
                roof = {'kernel': 'k_sinkhorn', 'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                        'frac': ach / peak, 'traffic': traffic,
                        'traffic_source': ('dram__bytes_read+write per launch, %s' % traffic_src) if traffic else None,
                        'peak_source': peaks['_source'],
                        'launches_timed': cnt.value, 'avg_launch_ms': avg_s * 1e3, 'bytes_per_launch': byts}

    # --- the other kernel classes, timed the same way (one stream, CUDA events inside the library) -------------
    other = {}
    if rank == 0 and roof is not None:
        npair = 2 * args.pairs_per_launch
        d = 256
        for cls in ('gemm', 'sinkhorn', 'cosine'):
            L.gims_profile_begin(_lib.PROF[cls], 4096)
            torch.cuda.synchronize(dev)
            PairBatchRunner(gm, n_streams=1, pairs_per_launch=args.pairs_per_launch).run([pool[i % len(pool)] for i in range(npair)])
            torch.cuda.synchronize(dev)
            tot, cnt = C.c_double(0), C.c_int(0)
            L.gims_profile_end(C.byref(tot), C.byref(cnt))
            if not cnt.value:
                continue
            ent = {'launches_per_pair': cnt.value / npair, 'ms_per_pair': tot.value / npair}
            if cls == 'gemm':
                # every per-node linear map of a pair (the reference's count: the merge conv that we fold away included)
                fl = float(projection_flops(n0k, n1k))
                ent.update({'bound': 'tensor', 'achieved': fl / (tot.value / npair / 1e3) / 1e12, 'unit': 'TFLOP/s',
                            'flops_per_pair': fl})
                ent['frac'] = ent['achieved'] / peaks['bf16_tflops_sustained']
                # fp32 parity costs 3 MMAs per product: fp16 hi+lo planes at the bf16 rate (ceiling 1/3), tf32 planes at half (1/6)
                ent['ceiling_frac'] = 1.0 / 6.0 if L.gims_get_gemm_mode() == _lib.GEMM_TC else 1.0 / 3.0
                ent['frac_of_ceiling'] = ent['frac'] / ent['ceiling_frac']
            elif cls == 'sinkhorn':
                e_bytes = 4.0 * (n0k + 1) * (n1k + 1)
                us_it = tot.value / cnt.value * 1e3 / 100.0
                if n1k + 1 > 2051 or n0k + 1 > 2368:
                    # streamed regime: the scaled matrix E is read once per iteration (from L2 while it fits, else HBM)
                    ent.update({'bound': 'hbm' if e_bytes > 100e6 else 'l2', 'us_per_iteration': us_it,
                                'bytes_per_iteration': e_bytes, 'achieved': e_bytes / us_it / 1e3, 'unit': 'GB/s',
                                'peak': peaks['hbm_gbs'], 'frac': e_bytes / us_it / 1e3 / peaks['hbm_gbs'], 'path': sink_path,
                                'note': 'frac is against the measured HBM copy bandwidth; iterations include the grid-wide exchange'})
                else:
                    ent.update({'bound': 'latency (100 grid-wide exchanges through L2; the matrix stays on chip)',
                                'us_per_iteration': us_it, 'hbm_bytes_per_launch': e_bytes, 'sms_used': 74, 'path': sink_path})
            elif cls == 'cosine':
                fl = 2.0 * d * (n0k * (n0k + 1) / 2 + n1k * (n1k + 1) / 2)
                ent.update({'bound': 'fp64 pipe', 'achieved': fl / (tot.value / npair / 1e3) / 1e12, 'unit': 'TFLOP/s (fp64)',
                            'flops_per_pair': fl})
            other[cls] = ent

    # --- e2e: the reference-facing call with pinned host tensors ------------------------------------------
    e2e = None
    if not args.no_e2e:
        # long enough that the ramp and the tail (one pair latency under load, ~20 ms) are a few per cent of the region
        n_e2e = max(8, min(4 * P * args.steps, 512))
        pinned = []
        for d in pool_host:
            h = {k: (v.pin_memory() if torch.is_tensor(v) and k != 'image0' and k != 'image1' else v) for k, v in d.items()}
            h['device'] = dev
            pinned.append(h)
        host = [pinned[i % len(pinned)] for i in range(n_e2e)]     # every call copies its inputs from pinned host memory
        # T host threads (one CUDA stream each) issue sequential Matching(data) calls — the reference-facing call,
        # as a server handling concurrent requests would make it; ctypes / torch release the GIL while they wait
        T = max(1, min(args.e2e_threads, n_e2e))
        e2e_streams = [torch.cuda.Stream(device=dev) for _ in range(T)]
        d2h_box = [0]
        errors = []

        # the results of a call are read into pinned host buffers (a pageable .cpu() makes the driver stage the copy under
        # a lock the other caller threads need for their launches)
        res_m = [torch.empty(args.kpts, dtype=torch.int64).pin_memory() for _ in range(T)]
        res_s = [torch.empty(args.kpts, dtype=torch.float32).pin_memory() for _ in range(T)]

        def e2e_worker(tid, items):
            try:
                torch.cuda.set_device(dev)
                with torch.no_grad(), torch.cuda.stream(e2e_streams[tid]):
                    for h in items:
                        pred = matching(dict(h))
                        m0, s0 = pred['matches0'][0], pred['matching_scores0'][0]
                        res_m[tid][:m0.numel()].copy_(m0, non_blocking=True)
                        res_s[tid][:s0.numel()].copy_(s0, non_blocking=True)
                        e2e_streams[tid].synchronize()
                        d2h_box[0] = m0.numel() * 8 + s0.numel() * 4
            except Exception as exc:      # noqa: BLE001 - reported below
                errors.append(exc)

        def e2e_round(items):
            ths = [threading.Thread(target=e2e_worker, args=(t, items[t::T])) for t in range(T)]
            for th in ths:
                th.start()
            for th in ths:
                th.join()
            torch.cuda.synchronize(dev)
            if errors:
                raise errors[0]

        e2e_round(host[:2 * T])                          # warm-up: workspaces, pinned staging, allocator
        t0 = time.perf_counter()                         # for reference: one thread, one pair in flight (latency-bound)
        e2e_worker(0, host[:8])
        torch.cuda.synchronize(dev)
        single = 8 / (time.perf_counter() - t0)
        if errors:
            raise errors[0]
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        e2e_round(host)
        dt = time.perf_counter() - t0
        d2h = d2h_box[0]
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {'value': world * n_e2e / dt, 'unit': UNIT, 'h2d_bytes_per_step': in_bytes * P, 'd2h_bytes_per_step': d2h * P,
               'pairs_timed': n_e2e, 'host_threads': T, 'single_thread_value': single,
               'note': '%d host threads x sequential Matching(data) calls on pinned host tensors, one stream each; '
                       'wall clock incl. H2D/D2H, max over ranks' % T}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': base_config(args, world), 'kept_keypoints': counts[:2], 'sinkhorn_path': sink_path,
            'arithmetic': gemm_mode_name,
            'cuda_device_max_connections': os.environ.get('CUDA_DEVICE_MAX_CONNECTIONS'),   # set by `import gims_b200`
            'clocks': clocks, 'e2e': e2e, 'gpu_launches': int(launches) * world, 'gpu_launches_per_rank': int(launches),
            'roofline': roof, 'roofline_other': other,
            'pair_gflop': pair_flops(counts[0], counts[1]) / 1e9,
            'model_tflops': value / world * pair_flops(counts[0], counts[1]) / 1e12,
        }
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = cpu_baseline(args)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
