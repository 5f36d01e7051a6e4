"""TEST INFRASTRUCTURE — generate `tests/golden/*.npz` by running the UNMODIFIED reference.

Needs a checkout of the reference:   GIMS_REFERENCE_ROOT=<songxf1024/GIMS checkout> python -m oracle.make_golden
Each fixture holds the synthetic-input recipe (sizes, seed, knobs — inputs are regenerated from
`gims_b200.synth`, not stored) and the reference's outputs at that boundary:
  * graph fixtures (`agc_*.npz`): kept indices + relabelled CSR per image, from
    models/agc.py:682-709 `build_optimize_graph_with_cosine_similarity`;
  * forward fixtures (`fwd_*.npz`): kept/CSR, pre-Sinkhorn scores (sub-sampled), Z (sub-sampled),
    potentials u/v (re-derived from the captured couplings with the reference's own
    `log_sinkhorn_iterations` lines, gmatcher.py:41-47), pre-threshold argmax indices, matches,
    matching scores and mdesc (sub-sampled), from models/gmatcher.py:219-307 `GMatcher.forward`.
"""
import contextlib
import io
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from gims_b200.synth import make_pair, make_state_dict  # noqa: E402
from oracle.ref_shims import load_reference  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')

# name -> recipe
AGC_CASES = {
    'agc_n512_dense': dict(n0=512, n1=512, seed=11, width=400, height=300, radius=25, percentile=7, min_size=8),
    'agc_n512_sparse': dict(n0=512, n1=480, seed=12, width=800, height=600, radius=25, percentile=7, min_size=8),
    'agc_n1024_eval': dict(n0=1024, n1=1000, seed=13, width=800, height=600, radius=15, percentile=2, min_size=7),
    'agc_n2048': dict(n0=2048, n1=2048, seed=14, width=800, height=600, radius=25, percentile=7, min_size=8),
    'agc_n2048_eval': dict(n0=2048, n1=2048, seed=15, width=800, height=600, radius=15, percentile=2, min_size=7),
    'agc_n4096': dict(n0=4096, n1=4096, seed=16, width=800, height=600, radius=25, percentile=7, min_size=8),
    'agc_n300_p50': dict(n0=300, n1=333, seed=17, width=320, height=240, radius=20, percentile=50, min_size=5),
    'agc_n64_tiny': dict(n0=64, n1=40, seed=18, width=100, height=80, radius=12, percentile=10, min_size=3),
}
FWD_CASES = {
    'fwd_n512': dict(n0=512, n1=512, seed=21, width=400, height=300, radius=25, percentile=7, min_size=8,
                     wseed=0, peaked=False, damped=False, iters=100, image_style='tensor', match_threshold=0.2),
    'fwd_n512_peaked': dict(n0=512, n1=512, seed=22, width=400, height=300, radius=25, percentile=7, min_size=8,
                            wseed=0, peaked=True, damped=False, iters=100, image_style='tensor',
                            match_threshold=0.0005),
    'fwd_n512_damped': dict(n0=512, n1=500, seed=26, width=400, height=300, radius=25, percentile=7, min_size=8,
                            wseed=2, peaked=False, damped=True, iters=100, image_style='tensor',
                            match_threshold=0.01),
    'fwd_ragged_eval': dict(n0=300, n1=257, seed=23, width=320, height=240, radius=15, percentile=2, min_size=7,
                            wseed=1, peaked=True, damped=False, iters=20, image_style='eval', match_threshold=0.001),
    'fwd_n512_sparse': dict(n0=512, n1=512, seed=24, width=800, height=600, radius=25, percentile=7, min_size=8,
                            wseed=0, peaked=False, damped=True, iters=100, image_style='tensor',
                            match_threshold=0.01),
    'fwd_n2048_damped': dict(n0=2048, n1=2048, seed=25, width=800, height=600, radius=25, percentile=7,
                             min_size=8, wseed=0, peaked=False, damped=True, iters=100, image_style='tensor',
                             match_threshold=0.005),
    # BASELINE configs[3] / configs[4] sizes (L2-resident and HBM-streaming Sinkhorn regimes), non-degenerate weights
    'fwd_n4096_damped': dict(n0=4096, n1=4096, seed=27, width=800, height=600, radius=25, percentile=7,
                             min_size=8, wseed=0, peaked=False, damped=True, iters=100, image_style='tensor',
                             match_threshold=0.005),
    'fwd_n4096_ragged_peaked': dict(n0=4096, n1=3500, seed=28, width=800, height=600, radius=15, percentile=2,
                                    min_size=7, wseed=1, peaked=True, damped=False, iters=20, image_style='eval',
                                    match_threshold=0.0005),
    'fwd_n8192_damped': dict(n0=8192, n1=8192, seed=29, width=1600, height=1200, radius=25, percentile=7,
                             min_size=8, wseed=0, peaked=False, damped=True, iters=100, image_style='tensor',
                             match_threshold=0.005),
}
SUB = 48   # rows/cols kept of dense matrices


def _csr_from_shim_graph(g):
    n = g.num_nodes()
    src = g.src.numpy()
    dst = g.dst.numpy()
    order = np.lexsort((src, dst))           # rows = dst (in-edges; graph is symmetric), neighbours ascending
    dst_s, src_s = dst[order], src[order]
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.add.at(indptr, dst_s + 1, 1)
    return np.cumsum(indptr), src_s.astype(np.int64)


def run_agc(rec):
    agc, _ = load_reference()
    data = make_pair(rec['n0'], rec['n1'], seed=rec['seed'], width=rec['width'], height=rec['height'])
    out = {}
    for s in ('0', '1'):
        with contextlib.redirect_stdout(io.StringIO()):
            graphs, kept = agc.build_optimize_graph_with_cosine_similarity(
                data['keypoints' + s], data['descriptors' + s], data['scores' + s], radius=rec['radius'],
                percentile=rec['percentile'], min_size=rec['min_size'], device=torch.device('cpu'),
                image=None, show=False)
        indptr, indices = _csr_from_shim_graph(graphs[0])
        out['kept' + s] = np.asarray(kept[0], dtype=np.int64)
        out['csr_indptr' + s] = indptr
        out['csr_indices' + s] = indices
    return out


def run_fwd(rec):
    _, gm = load_reference()
    data = make_pair(rec['n0'], rec['n1'], seed=rec['seed'], width=rec['width'], height=rec['height'],
                     image_style=rec['image_style'])
    data.update({'device': torch.device('cpu'), 'radius': rec['radius'], 'percentile': rec['percentile'],
                 'min_size': rec['min_size']})
    sd = make_state_dict(rec['wseed'], peaked=rec['peaked'], damped=rec['damped'])
    model = gm.GMatcher({'sinkhorn_iterations': rec['iters'], 'match_threshold': rec['match_threshold']})
    model.load_state_dict(sd)
    model.eval()
    cap = {}
    orig = gm.log_optimal_transport

    def spy(scores, alpha, iters):
        cap['scores'] = scores.clone()
        z = orig(scores, alpha, iters)
        cap['Z'] = z.clone()
        return z

    gm.log_optimal_transport = spy
    try:
        with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
            pred = model(data)
    finally:
        gm.log_optimal_transport = orig
    out = {}
    for s in ('0', '1'):
        indptr, indices = _csr_from_shim_graph(data['graph' + s][0])
        out['kept' + s] = np.asarray(data['kept_kpts%s_indices' % s][0], dtype=np.int64)
        out['csr_indptr' + s] = indptr
        out['csr_indices' + s] = indices
    scores, z = cap['scores'], cap['Z']
    # potentials: the reference's own five lines (gmatcher.py:41-47) on the captured couplings
    b, m, n = scores.shape
    alpha = model.bin_score.detach()
    coup = torch.cat([torch.cat([scores, alpha.expand(b, m, 1)], -1),
                      torch.cat([alpha.expand(b, 1, n), alpha.expand(b, 1, 1)], -1)], 1)
    norm = -torch.tensor(float(m + n)).log()
    log_mu = torch.cat([norm.expand(m), torch.tensor(float(n)).log()[None] + norm])[None]
    log_nu = torch.cat([norm.expand(n), torch.tensor(float(m)).log()[None] + norm])[None]
    u, v = torch.zeros_like(log_mu), torch.zeros_like(log_nu)
    for _ in range(rec['iters']):
        u = log_mu - torch.logsumexp(coup + v.unsqueeze(1), dim=2)
        v = log_nu - torch.logsumexp(coup + u.unsqueeze(2), dim=1)
    assert torch.equal(coup + u.unsqueeze(2) + v.unsqueeze(1) - norm, z)
    zi = z[:, :-1, :-1]
    out.update({
        'scores_sub': scores[0, :SUB, :SUB].numpy(), 'scores_mean': np.float64(scores.double().mean()),
        'scores_std': np.float64(scores.double().std()), 'scores_absmax': np.float64(scores.abs().max()),
        'Z_sub': z[0, :SUB, :SUB].numpy(), 'Z_lastrow': z[0, -1, :].numpy(), 'Z_lastcol': z[0, :, -1].numpy(),
        'Z_rowmax': zi.max(2).values[0].numpy(), 'Z_colmax': zi.max(1).values[0].numpy(),
        'u': u[0].numpy(), 'v': v[0].numpy(),
        'indices0': zi.max(2).indices[0].numpy(), 'indices1': zi.max(1).indices[0].numpy(),
        'matches0': pred['matches0'][0].numpy(), 'matches1': pred['matches1'][0].numpy(),
        'matching_scores0': pred['matching_scores0'][0].numpy(),
        'matching_scores1': pred['matching_scores1'][0].numpy(),
        'mdesc0_sub': pred['mdesc0'][:SUB].numpy(), 'mdesc1_sub': pred['mdesc1'][:SUB].numpy(),
        'mdesc0_rownorm': pred['mdesc0'].norm(dim=1).numpy(), 'mdesc1_rownorm': pred['mdesc1'].norm(dim=1).numpy(),
        'keypoints0': pred['keypoints0'][0].numpy(), 'keypoints1': pred['keypoints1'][0].numpy(),
    })
    return out


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.manual_seed(0)
    only = set(sys.argv[1:])          # optional: fixture names to (re)generate; default all
    for name, rec in AGC_CASES.items():
        if only and name not in only:
            continue
        out = run_agc(rec)
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + '.npz'), recipe=np.array(repr(rec)), **out)
        print(name, {k: v.shape for k, v in out.items() if k.startswith('kept')})
    for name, rec in FWD_CASES.items():
        if only and name not in only:
            continue
        out = run_fwd(rec)
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + '.npz'), recipe=np.array(repr(rec)), **out)
        print(name, 'kept', out['kept0'].shape, out['kept1'].shape,
              'mutual matches', int((out['matches0'] >= 0).sum()))


if __name__ == '__main__':
    main()
