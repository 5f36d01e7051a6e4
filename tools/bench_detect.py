"""SIFT detection on the device (`detect_device`, csrc/sift.cu) against cv2 on the host, and the image-input `Matching`
call (BASELINE configs[2], eval_homography.py:177) with 'detector': 'opencv' against 'device'.

    python tools/bench_detect.py [--pairs 24] [--kpts 2048] [--reps 50]

One JSON line: per 800 x 600 colour image the cv2 detect time (with cv2's host thread count) and the device detect time
(CUDA events over --reps warm calls, upload of the image and the read-back of count and records included), the
agreement of the two keypoint sets (tests/test_sift_cpu.py's tolerance), and ms per pair of the whole `Matching` call
with images for both detectors, in one process, alternated pair by pair.  The descriptor network is the reference's
CAR_HyNet (random init) when oracle/_ref has it, else the stand-in of tools/bench_frontend.py; the line says which.  The
GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def _stats(t):
    return {'median': round(float(np.median(t)), 2), 'mean': round(float(np.mean(t)), 2), 'min': round(float(np.min(t)), 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pairs', type=int, default=24)
    ap.add_argument('--kpts', type=int, default=2048)
    ap.add_argument('--reps', type=int, default=50)
    args = ap.parse_args()
    import cv2

    import bench
    from bench_frontend import StandInNet, gpu_info
    from gims_b200 import Matching, frontend as fe
    from gims_b200.synth import make_state_dict, make_textured_image, warp_image
    from test_sift_cpu import agreement, records
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    info = gpu_info()
    car = bench.load_caller_carhynet(dev)
    net = 'CAR_HyNet (reference, random init)'
    if car is None:
        torch.manual_seed(0)
        car = type('Car', (), {})()
        car.model, car.batch_size = StandInNet().to(dev).eval(), 512
        net = 'stand-in Conv2d(3, 8, 5, stride=3) network of tests/test_gpu_frontend.py (reference CAR_HyNet not found)'

    # -- detection alone ----------------------------------------------------------------------------------------------
    img = make_textured_image(600, 800, seed=100)
    for _ in range(5):
        fe.detect_device(img, dev)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.reps):
        dk = fe.detect_device(img, dev)
    e1.record()
    torch.cuda.synchronize(dev)
    dev_ms = e0.elapsed_time(e1) / args.reps
    fe.detect(img)
    a = time.perf_counter()
    for _ in range(5):
        kps = fe.detect(img)
    host_ms = 1e3 * (time.perf_counter() - a) / 5
    got = {'pt': dk.pt.cpu().numpy(), 'size': dk.size.cpu().numpy(), 'angle': dk.angle.cpu().numpy(),
           'octave': dk.octave.cpu().numpy()}
    want = records(kps)

    # -- the whole image-input call, both detectors, alternated ---------------------------------------------------------
    routes = {}
    for name in ('opencv', 'device'):
        m = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.2, 'max_keypoints': args.kpts, 'detector': name})
        m.gmodel.load_state_dict(make_state_dict(0))
        routes[name] = m.eval().to(dev)
    knobs = {'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7}

    def call(name, p):
        with torch.no_grad():
            pred = routes[name]({**knobs, 'image0': p[0], 'image1': p[1], 'carhynet': car})
        return {k: v[0].cpu() for k, v in pred.items()}

    pairs = []
    for i in range(args.pairs + 2):
        i0 = make_textured_image(600, 800, seed=100 + i)
        i1, _ = warp_image(i0, seed=200 + i)
        pairs.append((i0[None], i1[None]))
    for p in pairs[:2]:
        call('opencv', p)
        call('device', p)
    times = {'opencv': [], 'device': []}
    for k, p in enumerate(pairs[2:]):
        for name in (('opencv', 'device') if k % 2 == 0 else ('device', 'opencv')):
            torch.cuda.synchronize(dev)
            a = time.perf_counter()
            call(name, p)
            torch.cuda.synchronize(dev)
            times[name].append(1e3 * (time.perf_counter() - a))
    print(json.dumps({
        'metric': 'frontend_detect_800x600', 'gpu': info, 'network': net, 'kpts': args.kpts, 'pairs': args.pairs,
        'cv2_detect_ms_per_image': round(host_ms, 2), 'cv2_threads': cv2.getNumThreads(), 'host_cpus': os.cpu_count(),
        'device_detect_ms_per_image_incl_upload_and_readback': round(dev_ms, 3), 'device_detect_reps': args.reps,
        'keypoints_cv2': len(kps), 'keypoints_device': len(dk),
        'agreement_device_in_cv2': round(agreement(got, want), 4), 'agreement_cv2_in_device': round(agreement(want, got), 4),
        'pipeline_ms_per_pair_opencv': _stats(times['opencv']), 'pipeline_ms_per_pair_device': _stats(times['device'])}))


if __name__ == '__main__':
    main()
