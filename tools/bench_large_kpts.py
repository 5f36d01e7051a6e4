"""One pair at 8192 .. 65536 keypoints per image: time, stage split and peak device memory.

    python tools/bench_large_kpts.py [--sizes 8192,16384,32768,49152,65536] [--reps 3] [--out FILE]

Per size, one JSON line: the whole forward (`GMatcher.run_pair`, `damped` weights, 100 Sinkhorn iterations, radius 25,
percentile 7, min_size 8) in ms (host clock around enqueue + device synchronise, median of --reps warm calls); the stage
split from the library's CUDA-event profiler (`gims_profile_begin`, one warm call per class: the AGC cosine matrix, the
projection / MLP GEMMs, flash attention, the score GEMM, the Sinkhorn launch or launches); the graph construction of one
image alone (`gims_agc_build`, CUDA events; in the forward the two images' chains run side by side); which Sinkhorn path
ran; and the peak of `torch.cuda.max_memory_allocated` over one call with an empty allocator.  The GPU's name and power
limit are read in the same run."""
import argparse
import ctypes as C
import gc
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

CLASSES = ('cosine', 'gemm', 'attention', 'score', 'sinkhorn')


def _geometry(n):
    """Image size of a synthetic pair with the keypoint density of the 16384-keypoint test (2400 x 1800)."""
    s = (n / 16384) ** 0.5
    return int(2400 * s), int(1800 * s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--sizes', default='8192,16384,32768,49152,65536')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    from bench_frontend import gpu_info
    from gims_b200 import GMatcher, _lib
    from gims_b200.synth import make_pair, make_state_dict
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    gpu = gpu_info()
    lines = []
    for n in [int(x) for x in args.sizes.split(',')]:
        w, h = _geometry(n)
        data = make_pair(n, n, seed=900 + n % 997, width=w, height=h)
        ins = [data[k][0].to(dev).contiguous() for k in ('keypoints0', 'descriptors0', 'scores0',
                                                         'keypoints1', 'descriptors1', 'scores1')]
        model = GMatcher({'sinkhorn_iterations': 100, 'match_threshold': 0.2})
        model.load_state_dict(make_state_dict(0, damped=True))
        model = model.to(dev).eval()

        def call():
            with torch.no_grad():
                return model.run_pair(*ins, data['image0'].shape, data['image1'].shape, 25, 7, 8)

        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        r = call()
        torch.cuda.synchronize(dev)
        peak = torch.cuda.max_memory_allocated(dev)
        cnt = r['n_kept_dev'].cpu().tolist()
        status = int(cnt[6])
        assert status & _lib.STATUS_ERROR_MASK == 0, 'status %#x' % status
        times = []
        for _ in range(args.reps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            r = call()
            torch.cuda.synchronize(dev)
            times.append((time.perf_counter() - t0) * 1e3)
        split = {}
        for cls in CLASSES:
            L.gims_profile_begin(_lib.PROF[cls], 100000)
            call()
            torch.cuda.synchronize(dev)
            tot, k = C.c_double(0), C.c_int(0)
            L.gims_profile_end(C.byref(tot), C.byref(k))
            split[cls] = {'ms': round(tot.value, 3), 'launches': k.value}
        # graph construction of image 0 alone
        from gims_b200.gmatcher import GMatcher as G
        cap = max(1024, int(model.edge_cap_factor) * n)
        ws = torch.empty(L.gims_agc_workspace_bytes(n, cap), dtype=torch.uint8, device=dev)
        kept = torch.empty(n, dtype=torch.int32, device=dev)
        cbuf = torch.zeros(4, dtype=torch.int32, device=dev)
        indptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
        indices = torch.empty(cap, dtype=torch.int32, device=dev)
        kpo, fo, so, thr = (torch.empty(n, 2, device=dev), torch.empty(n, 256, device=dev), torch.empty(n, device=dev),
                            torch.zeros(1, device=dev))
        st = torch.cuda.current_stream(dev)

        def agc():
            _lib.check(L.gims_agc_build(_lib.ptr(ins[0]), _lib.ptr(ins[1]), 1, _lib.ptr(ins[2]), n, 25.0, G._k_rank(n, 7), 8,
                                        _lib.ptr(ws), ws.numel(), _lib.ptr(kept), C.c_void_p(cbuf.data_ptr()), _lib.ptr(indptr),
                                        _lib.ptr(indices), cap, C.c_void_p(cbuf.data_ptr() + 4), _lib.ptr(kpo), _lib.ptr(fo),
                                        _lib.ptr(so), _lib.ptr(thr), C.c_void_p(cbuf.data_ptr() + 8),
                                        C.c_void_p(cbuf.data_ptr() + 12), C.c_void_p(st.cuda_stream)), 'gims_agc_build')

        agc()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record(st)
        for _ in range(args.reps):
            agc()
        ev[1].record(st)
        torch.cuda.synchronize(dev)
        agc_ms = ev[0].elapsed_time(ev[1]) / args.reps
        path = 'wide' if status & _lib.STATUS_SINKHORN_WIDE else ('fast' if status & _lib.STATUS_SINKHORN_FAST else 'exact')
        line = {'kpts_per_image': n, 'kept': cnt[:2], 'gpu': gpu, 'forward_ms': round(float(np.median(times)), 2),
                'forward_ms_all': [round(t, 2) for t in times], 'sinkhorn_iterations': 100, 'sinkhorn_path': path,
                'stages_ms': split, 'agc_one_image_ms': round(agc_ms, 3),
                'peak_memory_gb': round(peak / 1e9, 2), 'weights': 'damped'}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del model, r, ws, ins, data, kept, indptr, indices, kpo, fo, so
        gc.collect()
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, 'w') as fh:
            for line in lines:
                fh.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
