"""Front end of the image-input pipeline (BASELINE configs[2], eval_homography.py:177): the Gaussian pyramid built on the
device (`gaussian_pyramid_device`) against the host pyramid (OpenCV) whose levels `extract_patches_device` uploads.

    python tools/bench_frontend.py [--pairs 24] [--kpts 2048]

One JSON line: the device pyramid per image (CUDA events, upload of the image included), the host pyramid per image,
the bytes each route uploads per image, and ms per pair of the whole `Matching` call with images for the old route
(host pyramid, the levels carrying keypoints uploaded) against the new one, in one process, alternated pair by pair.
The descriptor network is the reference's CAR_HyNet (random init) when oracle/_ref has it, else a small stand-in; the
line says which.  The GPU's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class StandInNet(torch.nn.Module):
    """The stand-in descriptor network of tests/test_gpu_frontend.py."""

    def __init__(self):
        super().__init__()
        self.c = torch.nn.Conv2d(3, 8, 5, stride=3)

    def forward(self, x):
        return torch.nn.functional.normalize(self.c(x).flatten(1)[:, :128], dim=1)


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pairs', type=int, default=24)
    ap.add_argument('--kpts', type=int, default=2048)
    args = ap.parse_args()
    import bench
    from gims_b200 import Matching, frontend as fe
    from gims_b200.synth import make_state_dict, make_textured_image, warp_image
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    car = bench.load_caller_carhynet(dev)
    net = 'CAR_HyNet (reference, random init)'
    if car is None:
        torch.manual_seed(0)
        car = type('Car', (), {})()
        car.model, car.batch_size = StandInNet().to(dev).eval(), 512
        net = 'stand-in Conv2d(3, 8, 5, stride=3) network of tests/test_gpu_frontend.py (reference CAR_HyNet not found)'
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.2, 'max_keypoints': args.kpts})
    matching.gmodel.load_state_dict(make_state_dict(0))
    matching = matching.eval().to(dev)
    knobs = {'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7}

    # -- the pyramid alone ------------------------------------------------------------------------------------------
    img = make_textured_image(600, 800, seed=100)
    for _ in range(5):
        fe.gaussian_pyramid_device(img, dev)
    torch.cuda.synchronize(dev)
    reps = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        pyr = fe.gaussian_pyramid_device(img, dev)
    e1.record()
    torch.cuda.synchronize(dev)
    dev_pyr_ms = e0.elapsed_time(e1) / reps
    a = time.perf_counter()
    for _ in range(5):
        levels = fe.gaussian_pyramid(img)
    host_pyr_ms = 1e3 * (time.perf_counter() - a) / 5
    kps = fe.detect(img, args.kpts)
    used = sorted(set(fe.patch_maps(kps)[0].tolist()))
    old_bytes = int(sum(levels[i].size for i in used))
    new_bytes = int(img.size + 16 * len(pyr))
    same = all(np.array_equal(pyr.level(i).cpu().numpy(), lv) for i, lv in enumerate(levels))

    # -- the whole image-input call, old route against new, alternated -------------------------------------------------
    def old_route(p):
        """Matching.forward as it was: detection and the host pyramid side by side, levels uploaded per image."""
        device_pyramid = fe._use_device_pyramid
        fe._use_device_pyramid = lambda image, device, detector: False
        try:
            staged = fe.stage_images([p[0], p[1]], dev, args.kpts)
        finally:
            fe._use_device_pyramid = device_pyramid
        data = dict(knobs)
        for s, imgs in (('0', p[0]), ('1', p[1])):
            f = fe.sift_forward({'image': imgs, 'max_keypoints': args.kpts, 'carhynet': car}, dev, staged=staged[int(s)])
            for k, v in f.items():
                data[k + s] = torch.stack(v)
        data['image0'], data['image1'] = p
        with torch.no_grad():
            pred = matching(data)
        return {k: v[0].cpu() for k, v in pred.items()}

    def new_route(p):
        with torch.no_grad():
            pred = matching({**knobs, 'image0': p[0], 'image1': p[1], 'carhynet': car})
        return {k: v[0].cpu() for k, v in pred.items()}

    pairs = []
    for i in range(args.pairs + 2):
        i0 = make_textured_image(600, 800, seed=100 + i)
        i1, _ = warp_image(i0, seed=200 + i)
        pairs.append((i0[None], i1[None]))
    for p in pairs[:2]:                                                 # warm-up of both routes
        old_route(p)
        new_route(p)
    t_old, t_new, equal = [], [], True
    for k, p in enumerate(pairs[2:]):
        order = (('old', old_route), ('new', new_route)) if k % 2 == 0 else (('new', new_route), ('old', old_route))
        outs = {}
        for name, fn in order:
            torch.cuda.synchronize(dev)
            a = time.perf_counter()
            outs[name] = fn(p)
            torch.cuda.synchronize(dev)
            (t_old if name == 'old' else t_new).append(1e3 * (time.perf_counter() - a))
        equal = equal and all(torch.equal(outs['old'][x], outs['new'][x]) for x in ('keypoints0', 'keypoints1', 'matches0', 'matches1'))
    print(json.dumps({
        'metric': 'frontend_pyramid_800x600', 'gpu': gpu_info(), 'network': net, 'kpts': args.kpts, 'pairs': args.pairs,
        'device_pyramid_ms_per_image_incl_upload': round(dev_pyr_ms, 3), 'host_pyramid_ms_per_image': round(host_pyr_ms, 2),
        'device_pyramid_levels_equal_host': bool(same), 'levels': len(levels),
        'upload_bytes_per_image_old': old_bytes, 'upload_bytes_per_image_new': new_bytes,
        'pipeline_ms_per_pair_old': {'median': round(float(np.median(t_old)), 2), 'mean': round(float(np.mean(t_old)), 2),
                                     'min': round(float(np.min(t_old)), 2)},
        'pipeline_ms_per_pair_new': {'median': round(float(np.median(t_new)), 2), 'mean': round(float(np.mean(t_new)), 2),
                                     'min': round(float(np.min(t_new)), 2)},
        'old_and_new_keypoints_and_matches_equal': bool(equal)}))


if __name__ == '__main__':
    main()
