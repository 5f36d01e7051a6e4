"""RANSAC homographies of a batch of pairs on the device (`postprocess.find_homographies`, csrc/homography.cu) against
cv2.findHomography(..., cv2.RANSAC, 3) on the host.

    python tools/bench_homography.py [--pairs 199] [--reps 10] [--out FILE]

Workloads: --pairs synthetic pairs (199 = the size of eval_homography's image set) at 300 and 2048 matches with inlier
ratios 0.8 / 0.5 / 0.2 (noise 1 px, outliers uniform over 800 x 600).  Device: the batched call timed with CUDA events
over --reps warm calls, and the single-pair latency (one pair per call, the median over the first 20 pairs).  Host: cv2
over the same pairs sequentially, and in a thread pool of one thread per host core.  One JSON line per workload, with
the GPU's name and power limit and the host core count read in the same run; --out also appends the lines to FILE."""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--pairs', type=int, default=199)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import cv2
    from bench_frontend import gpu_info
    from gims_b200 import postprocess as pp
    from gims_b200.synth import make_correspondences
    if not torch.cuda.is_available():
        raise SystemExit('bench_homography needs a CUDA device')
    dev = torch.device('cuda')
    gpu, cores = gpu_info(), os.cpu_count()
    cv2.setNumThreads(1)                      # one pair per host thread; the pool supplies the parallelism
    lines = []
    for m in (300, 2048):
        for ratio in (0.8, 0.5, 0.2):
            pairs = [make_correspondences(m, ratio, noise=1.0, seed=10000 * m + 100 * int(ratio * 10) + i)[:2]
                     for i in range(args.pairs)]
            src = [torch.from_numpy(s).to(dev) for s, _ in pairs]
            dst = [torch.from_numpy(d).to(dev) for _, d in pairs]
            pp.find_homographies(src, dst)                               # warm-up
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.reps):
                H, n_in, _ = pp.find_homographies(src, dst)
            t1.record()
            torch.cuda.synchronize()
            batch_ms = t0.elapsed_time(t1) / args.reps
            single = []
            for i in range(min(20, args.pairs)):
                t0.record()
                pp.find_homographies([src[i]], [dst[i]])
                t1.record()
                torch.cuda.synchronize()
                single.append(t0.elapsed_time(t1))
            found = int((H[:, 2, 2] != 0).sum())
            t = time.perf_counter()
            for s, d in pairs:
                cv2.findHomography(s, d, cv2.RANSAC, 3.0)
            seq_ms = (time.perf_counter() - t) * 1e3
            with ThreadPoolExecutor(cores) as ex:
                list(ex.map(lambda sd: cv2.findHomography(sd[0], sd[1], cv2.RANSAC, 3.0), pairs[:8]))   # warm-up
                t = time.perf_counter()
                list(ex.map(lambda sd: cv2.findHomography(sd[0], sd[1], cv2.RANSAC, 3.0), pairs))
                pool_ms = (time.perf_counter() - t) * 1e3
            line = {'metric': 'ransac_homography', 'gpu': gpu, 'host_cores': cores, 'pairs': args.pairs, 'matches': m,
                    'inlier_ratio': ratio, 'device_batch_ms': round(batch_ms, 3),
                    'device_single_pair_ms_median': round(float(np.median(single)), 3),
                    'cv2_sequential_ms': round(seq_ms, 2), 'cv2_pool_ms': round(pool_ms, 2), 'cv2_pool_threads': cores,
                    'speedup_vs_pool': round(pool_ms / batch_ms, 2), 'device_found': found,
                    'device_mean_inliers': round(float(n_in.double().mean()), 1)}
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, 'a') as fh:
            for line in lines:
                fh.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
