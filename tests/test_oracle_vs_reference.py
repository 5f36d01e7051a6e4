"""CPU: the oracle restatement against the UNMODIFIED reference run live (oracle/ref_shims.py), on inputs that are not
among the committed fixtures.  The reference is not part of the repository: these tests run where it is installed
(oracle/_ref, copied by __graft_entry__.build() from GIMS_REFERENCE_ROOT, or GIMS_REFERENCE_ROOT itself)."""
import contextlib
import io

import numpy as np
import pytest
import torch

from gims_b200.synth import make_pair, make_state_dict
from oracle import gims_oracle as orc
from oracle.ref_shims import REFERENCE_ROOT, load_reference, reference_available

pytestmark = pytest.mark.skipif(not reference_available(), reason='needs the original GIMS code (oracle/_ref or GIMS_REFERENCE_ROOT)')


@pytest.mark.parametrize('n0,n1,seed,r,p,m', [(260, 231, 901, 25, 7, 8), (400, 400, 902, 15, 2, 7), (150, 90, 903, 30, 20, 3)])
def test_graph_equals_live_reference(n0, n1, seed, r, p, m):
    """models/agc.py:682-709 run unchanged vs oracle.agc_build: kept indices and edge sets identical."""
    agc, _ = load_reference()
    data = make_pair(n0, n1, seed=seed, width=300, height=240)
    for s in ('0', '1'):
        with contextlib.redirect_stdout(io.StringIO()):
            graphs, kept = agc.build_optimize_graph_with_cosine_similarity(
                data['keypoints' + s], data['descriptors' + s], data['scores' + s], radius=r, percentile=p, min_size=m,
                device=torch.device('cpu'), image=None, show=False)
        out = orc.agc_build(data['keypoints' + s][0].numpy(), data['descriptors' + s][0].t().contiguous().numpy(), r, p, m)
        assert np.array_equal(np.asarray(kept[0], dtype=np.int64), out['kept'])
        g = graphs[0]
        ref_edges = set(zip(g.dst.tolist(), g.src.tolist()))
        rows = np.repeat(np.arange(len(out['kept'])), np.diff(out['indptr']))
        assert ref_edges == set(zip(rows.tolist(), out['indices'].tolist()))


def test_forward_equals_live_reference():
    """models/gmatcher.py:219-307 run unchanged vs oracle.gmatcher_forward on a ragged pair."""
    _, gm = load_reference()
    data = make_pair(333, 290, seed=904, width=320, height=250)
    data.update({'radius': 25, 'percentile': 7, 'min_size': 8})
    sd = make_state_dict(5, damped=True)
    cfg = {'sinkhorn_iterations': 30, 'match_threshold': 0.01}
    model = gm.GMatcher(cfg)
    model.load_state_dict(sd)
    model.eval()
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        ref = model({**data, 'device': torch.device('cpu')})
        got = orc.gmatcher_forward(sd, dict(data), cfg)
    assert torch.equal(ref['keypoints0'], got['keypoints0']) and torch.equal(ref['keypoints1'], got['keypoints1'])
    assert (ref['matches0'] == got['matches0']).float().mean() >= 0.999
    assert (ref['matches1'] == got['matches1']).float().mean() >= 0.999
    assert torch.allclose(ref['matching_scores0'], got['matching_scores0'], atol=1e-5)
    assert torch.allclose(ref['mdesc0'], got['mdesc0'], rtol=1e-4, atol=1e-4 * float(ref['mdesc0'].abs().max()))
    assert int((ref['matches0'] >= 0).sum()) > 10          # the case is not degenerate


def test_gt_matches_equal_live_reference():
    """utils/preprocess_utils.py:98-132 run unchanged vs oracle.find_gt_matches (row f-3)."""
    import importlib
    import sys
    load_reference()
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            pu = importlib.import_module('utils.preprocess_utils')
    except Exception as e:                         # albumentations / pycocotools are not in this image
        pytest.skip('utils.preprocess_utils cannot be imported here: %s' % e)
    g = torch.Generator().manual_seed(77)
    k0 = torch.rand(300, 2, generator=g) * 400
    H = torch.tensor([[1.02, 0.03, 5.0], [-0.02, 0.98, -3.0], [1e-5, -2e-5, 1.0]])
    k1 = orc.warp_keypoints(k0, H)[torch.randperm(300, generator=g)[:260]] + torch.randn(260, 2, generator=g) * 1.5
    ref = pu.torch_find_matches(k0, k1, H, dist_thresh=3, n_iters=3)
    got = orc.find_gt_matches(k0, k1, H, dist_thresh=3, n_iters=3)
    for a, b in zip(ref, got):
        assert torch.equal(a, b)
    assert len(got[0]) > 100
