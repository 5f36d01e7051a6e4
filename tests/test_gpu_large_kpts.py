"""More than 16384 keypoints per image (GIMS_MAX_KPTS = 65536): graph construction bit-exact on both sides of the
component search's 16-bit switch, the wide Sinkhorn path against float64, the score matrix past 2^31 / 2^32 elements,
whole forwards at 32768 and 65536, and the image-input call above 16384 keypoints.

Every test drops its model and buffers and empties the caching allocator: the matcher's per-stream workspace is
grow-only and holds tens of GB at these sizes."""
import ctypes as C
import gc
import types

import numpy as np
import pytest
import torch

from golden_util import index_agreement
from gims_b200.synth import make_pair, make_state_dict

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _release_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(1.0, np.abs(b))


# ---- 1. graph construction above 16384 nodes -------------------------------------------------------------------------
@pytest.mark.parametrize('n,seed', [(16384, 701), (20000, 702)])
def test_agc_above_16384_vs_oracle(n, seed):
    """gims_agc_build against the oracle (kept ids, CSR, threshold, component count bit for bit).  16384 nodes is the
    largest problem of the 32-bit union-find parents, 20000 runs the 16-bit ones."""
    from oracle import gims_oracle as orc
    from test_gpu_parity import _agc_only
    rec = dict(radius=25, percentile=7, min_size=8)
    data = make_pair(n, n - 17, seed=seed, width=2600, height=1900)
    outs = _agc_only(data, rec)
    for s, o in zip(('0', '1'), outs):
        ref = orc.agc_build(data['keypoints' + s][0].numpy(), data['descriptors' + s][0].t().contiguous().numpy(), 25, 7, 8)
        assert np.float32(o['thr']) == ref['thr']
        assert np.array_equal(o['kept'], ref['kept'])
        assert np.array_equal(o['indptr'], ref['indptr'])
        assert np.array_equal(o['indices'], ref['indices'])
        assert o['n_comp'] == ref['n_components']


# ---- 2. / 3. the wide Sinkhorn path -----------------------------------------------------------------------------------
def _sinkhorn(cbuf, ld, n0m, n1m, n0, n1, iters, threshold=0.0):
    from gims_b200 import _lib
    L = _lib.lib()
    dev = cbuf.device
    nd = torch.tensor([n0, n1], dtype=torch.int32, device=dev)
    ws = torch.empty(L.gims_sinkhorn_workspace_bytes(n0m, n1m), dtype=torch.uint8, device=dev)
    o = dict(u=torch.zeros(n0m + 1, device=dev), v=torch.zeros(n1m + 1, device=dev),
             i0=torch.zeros(n0m, dtype=torch.int32, device=dev), i1=torch.zeros(n1m, dtype=torch.int32, device=dev),
             m0=torch.zeros(n0m, dtype=torch.int64, device=dev), m1=torch.zeros(n1m, dtype=torch.int64, device=dev),
             s0=torch.zeros(n0m, device=dev), s1=torch.zeros(n1m, device=dev),
             status=torch.zeros(1, dtype=torch.int32, device=dev))
    _lib.check(L.gims_sinkhorn_match(_lib.ptr(cbuf), ld, n0m, n1m, _lib.ptr(nd), iters, threshold, _lib.ptr(ws), ws.numel(),
                                     _lib.ptr(o['u']), _lib.ptr(o['v']), _lib.ptr(o['i0']), _lib.ptr(o['i1']),
                                     _lib.ptr(o['m0']), _lib.ptr(o['m1']), _lib.ptr(o['s0']), _lib.ptr(o['s1']),
                                     _lib.ptr(o['status']), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
               'gims_sinkhorn_match')
    torch.cuda.synchronize()
    return {k: t.cpu() for k, t in o.items()}


@pytest.mark.parametrize('n0,n1,iters,scale,offset,aligned', [
    (300, 60000, 20, 2.0, 0.0, True),
    (300, 60000, 0, 2.0, 0.0, True),          # no iteration: zero potentials, only the final pass
    (300, 60000, 10, 1.0, 50.0, False),
    (1000, 65536, 10, 3.0, 0.0, True),
    (1000, 65536, 5, 1.0, 90.0, False),
])
def test_wide_sinkhorn_vs_float64(n0, n1, iters, scale, offset, aligned):
    """Problems the shared-memory kernels cannot hold: the wide path against the reference's iteration in float64, with
    capacities above the live counts and an aligned or unaligned pitch; run twice, bit-identical.  The status bit shows
    that the wide path ran (the shared-memory kernels cannot hold more than about 56 k columns on a B200)."""
    from gims_b200 import _lib
    from oracle import gims_oracle as orc
    L = _lib.lib()
    g = torch.Generator().manual_seed(n0 * 7 + n1 + int(offset))
    scores = torch.randn(1, n0, n1, generator=g) * scale + offset
    alpha = torch.tensor(0.7)
    dev = torch.device('cuda')
    z, u, v, coup = orc.log_optimal_transport(scores.double().to(dev), alpha.double().to(dev), iters)
    z, u, v, coup = z.float().cpu(), u.float().cpu(), v.float().cpu(), coup.float()
    m = orc.extract_matches(z, 0.0)
    n0m, n1m = n0 + 3, n1 + 5
    ld = L.gims_couplings_ld(n1m) if aligned else n1m + 1
    cbuf = torch.zeros(n0m + 1, ld, device=dev)
    cbuf[:n0 + 1, :n1 + 1] = coup[0]
    del coup
    got = _sinkhorn(cbuf, ld, n0m, n1m, n0, n1, iters)
    again = _sinkhorn(cbuf, ld, n0m, n1m, n0, n1, iters)
    del cbuf
    st = int(got['status'])
    assert st & _lib.STATUS_ERROR_MASK == 0, 'status %#x' % st
    assert st & _lib.STATUS_SINKHORN_WIDE and not st & (_lib.STATUS_SINKHORN_FAST | _lib.STATUS_SINKHORN_EXACT)
    for k in ('u', 'v', 'i0', 'i1', 'm0', 'm1', 's0', 's1'):
        assert torch.equal(got[k], again[k]), k                     # no float atomics: bit-identical run to run
    eu = _rel(got['u'][:n0 + 1].numpy(), u[0].numpy()).max()
    ev = _rel(got['v'][:n1 + 1].numpy(), v[0].numpy()).max()
    zi = z[0, :-1, :-1].numpy()
    i0, i1 = got['i0'][:n0].numpy(), got['i1'][:n1].numpy()
    a0 = index_agreement(i0, m['indices0'][0].numpy(), zi.max(1), zi[np.arange(n0), i0])
    a1 = index_agreement(i1, m['indices1'][0].numpy(), zi.max(0), zi[i1, np.arange(n1)])
    ours_ms, ref_ms = got['s0'][:n0].numpy(), m['matching_scores0'][0].numpy()
    flip = np.nonzero((ours_ms > 0) != (ref_ms > 0))[0]
    for i in flip:
        col = np.sort(zi[:, int(m['indices0'][0, i])])
        assert col[-1] - col[-2] < 1e-3, 'mutual status of row %d differs without a tie' % i
    keep = np.ones(n0, dtype=bool)
    keep[flip] = False
    ems = np.abs(ours_ms - ref_ms)[keep].max() if keep.any() else 0.0
    print('\n[wide %dx%d it=%d status %#x] du %.2e dv %.2e agree %.4f/%.4f exact %.4f/%.4f dms %.2e tie-flips %d' %
          (n0, n1, iters, st, eu, ev, a0, a1, (i0 == m['indices0'][0].numpy()).mean(),
           (i1 == m['indices1'][0].numpy()).mean(), ems, len(flip)))
    assert eu <= 1e-4 and ev <= 1e-4
    assert a0 >= 0.999 and a1 >= 0.999
    assert len(flip) <= max(8, n0 // 100)
    assert ems <= 1e-4 * max(1e-3, float(m['matching_scores0'].max())) + 1e-6
    assert (got['m0'][:n0] == m['matches0'][0]).numpy()[keep].mean() >= 0.999


def _structured_reference(a, b, perm, c, alpha, iters):
    """The reference's iteration in float64 on z_ij = a_i + b_j + c [j = perm(i)] with a dustbin score alpha: every
    log-sum-exp over a row or a column reduces to two running sums, O(N + M) per iteration."""
    from scipy.special import logsumexp
    n0, n1 = a.size, b.size
    inv = np.empty_like(perm)
    inv[perm] = np.arange(n0)
    norm = -np.log(n0 + n1)
    lmu = np.full(n0 + 1, norm); lmu[-1] = np.log(n1) + norm
    lnu = np.full(n1 + 1, norm); lnu[-1] = np.log(n0) + norm
    lc = np.log(np.expm1(c))                 # the diagonal adds (e^c - 1) exp(term) to the plain sum
    u, v = np.zeros(n0 + 1), np.zeros(n1 + 1)
    for _ in range(iters):
        w = b + v[:n1]
        W = logsumexp(w)
        u[:n0] = lmu[:n0] - np.logaddexp(a + np.logaddexp(W, w[perm] + lc), alpha + v[n1])
        u[n0] = lmu[n0] - (alpha + logsumexp(v))
        t = a + u[:n0]
        A = logsumexp(t)
        v[:n1] = lnu[:n1] - np.logaddexp(b + np.logaddexp(A, t[inv] + lc), alpha + u[n0])
        v[n1] = lnu[n1] - (alpha + logsumexp(u))
    return u, v, inv


def test_wide_sinkhorn_full_size_structured():
    """65536 x 65536 (17.2 GB of couplings, element offsets past 2^32) on a matrix whose float64 answer costs O(N + M)
    per iteration: the potentials match it and the argmax of every row / column is the planted permutation."""
    from gims_b200 import _lib
    L = _lib.lib()
    n, iters, c, alpha = 65536, 30, 12.0, 0.5
    rng = np.random.default_rng(77)
    a, b = rng.normal(0, 1, n), rng.normal(0, 1, n)
    perm = rng.permutation(n)
    dev = torch.device('cuda')
    ld = L.gims_couplings_ld(n)
    cbuf = torch.empty(n + 1, ld, device=dev)
    at, bt = torch.tensor(a, dtype=torch.float32, device=dev), torch.tensor(b, dtype=torch.float32, device=dev)
    for r0 in range(0, n, 4096):
        cbuf[r0:r0 + 4096, :n] = at[r0:r0 + 4096, None] + bt[None, :]
    rows = torch.arange(n, device=dev)
    pt = torch.tensor(perm, device=dev)
    cbuf[rows, pt] += c
    cbuf[n, :n + 1] = alpha
    cbuf[:n + 1, n] = alpha
    # the host reference sees the matrix as stored (fp32 entries), in float64
    a32 = at.double().cpu().numpy()
    b32 = bt.double().cpu().numpy()
    c_eff = (cbuf[rows, pt].double() - (at.double() + bt[pt].double())).cpu().numpy()
    assert np.abs(c_eff - c).max() < 1e-5
    got = _sinkhorn(cbuf, ld, n, n, n, n, iters)
    del cbuf, rows, pt
    st = int(got['status'])
    assert st & _lib.STATUS_ERROR_MASK == 0 and st & _lib.STATUS_SINKHORN_WIDE, 'status %#x' % st
    u, v, inv = _structured_reference(a32, b32, perm, c, np.float64(np.float32(alpha)), iters)
    eu, ev = _rel(got['u'].numpy(), u).max(), _rel(got['v'].numpy(), v).max()
    print('\n[wide 65536^2 structured] du %.2e dv %.2e' % (eu, ev))
    assert eu <= 1e-4 and ev <= 1e-4
    assert np.array_equal(got['i0'].numpy(), perm)
    assert np.array_equal(got['i1'].numpy(), inv)
    assert np.array_equal(got['m0'].numpy(), perm) and np.array_equal(got['m1'].numpy(), inv)


# ---- 4. / 5. whole forwards ------------------------------------------------------------------------------------------
def _check_properties(pred, data, n):
    """The size-independent properties test_forward_at_maximum_size_properties checks."""
    n0, n1 = pred['matches0'].shape[1], pred['matches1'].shape[1]
    assert 0.9 * n <= n0 <= n and 0.9 * n <= n1 <= n
    k0 = torch.tensor(data['kept_kpts0_indices'][0])
    assert (k0[1:] > k0[:-1]).all() and k0.numel() == n0
    indptr, indices = [t.cpu().long() for t in data['graph0'][0]]
    assert indptr[0] == 0 and indptr[-1] == indices.numel() and (indptr[1:] >= indptr[:-1]).all()
    rows = torch.repeat_interleave(torch.arange(n0), indptr[1:] - indptr[:-1])
    assert (rows != indices).all()
    key = rows * n0 + indices
    assert (key[1:] > key[:-1]).all()
    assert torch.equal(torch.sort(indices * n0 + rows).values, key)
    m0, m1 = pred['matches0'][0].cpu(), pred['matches1'][0].cpu()
    i = torch.nonzero(m0 >= 0).squeeze(1)
    assert i.numel() > 100 and (m1[m0[i]] == i).all()
    j = torch.nonzero(m1 >= 0).squeeze(1)
    assert (m0[m1[j]] == j).all() and i.numel() == j.numel()
    s0 = pred['matching_scores0'][0].cpu()
    assert torch.isfinite(s0).all() and (s0[i] > 0).all() and (s0 <= 1.0 + 1e-5).all() and (s0[m0 < 0] == 0).all()


def test_forward_at_32768_properties():
    """Between the old limit and the wide path: 32769 columns still fit the exact shared-memory kernel."""
    from gims_b200 import Matching
    n = 32768
    m = Matching({'sinkhorn_iterations': 5, 'match_threshold': 0.0})
    m.gmodel.load_state_dict(make_state_dict(3, damped=True))
    m = m.eval().to('cuda')
    data = make_pair(n, n, seed=641, width=3400, height=2500)
    data.update({'radius': 25, 'percentile': 7, 'min_size': 8, 'device': 'cuda'})
    with torch.no_grad():
        pred = m.gmodel(data)
    torch.cuda.synchronize()
    _check_properties(pred, data, n)
    del m, pred


def test_score_matrix_past_32bit_offsets():
    """The forward at 65536 keypoints with the couplings returned (debug): rows at the start, the end and around element
    offsets 2^31 and 2^32 equal mdesc0 . mdesc1^T / 16 in float64, and the dustbin border holds bin_score."""
    from gims_b200 import GMatcher, _lib
    n = _lib.MAX_KPTS
    sd = make_state_dict(3, damped=True)
    model = GMatcher({'sinkhorn_iterations': 3, 'match_threshold': 0.0})
    model.load_state_dict(sd)
    model = model.cuda().eval()
    data = make_pair(n, n, seed=642, width=4800, height=3600)
    dev = torch.device('cuda')
    with torch.no_grad():
        r = model.run_pair(data['keypoints0'][0].to(dev), data['descriptors0'][0].to(dev), data['scores0'][0].to(dev),
                           data['keypoints1'][0].to(dev), data['descriptors1'][0].to(dev), data['scores1'][0].to(dev),
                           data['image0'].shape, data['image1'].shape, 25, 7, 1, debug=True)    # min_size 1: nothing pruned
    torch.cuda.synchronize()
    cnt = r['n_kept_dev'].cpu().numpy()
    assert cnt[6] & 0xff == 0, 'error status %#x' % cnt[6]
    assert cnt[6] & _lib.STATUS_SINKHORN_WIDE
    n0, n1 = int(cnt[0]), int(cnt[1])
    assert n0 == n and n1 == n
    ld = r['couplings_buf'].shape[1]
    assert (n0 + 1) * ld > 2 ** 32
    want_rows = sorted({0, 1, 2 ** 31 // ld, 2 ** 31 // ld + 1, 2 ** 32 // ld, min(2 ** 32 // ld + 1, n0 - 1), n0 - 1})
    md = r['mdesc'].double()
    md0, md1 = md[:n0], md[n:n + n1]
    rows = torch.tensor(want_rows, device=dev)
    want = (md0[rows] @ md1.t() / 16).cpu().numpy()
    got = r['couplings_buf'][rows, :n1].cpu().numpy()
    err = _rel(got, want).max()
    print('\n[score rows %s] rel err %.2e' % (want_rows, err))
    assert err <= 2e-5
    bs = float(sd['bin_score'])
    coup = r['couplings_buf']
    assert bool((coup[n0, :n1 + 1] == bs).all()) and bool((coup[:n0 + 1, n1] == bs).all())
    assert bool(torch.isfinite(r['u'][:n0 + 1]).all()) and bool(torch.isfinite(r['v'][:n1 + 1]).all())
    del model, r, md, md0, md1, coup


# ---- 6. the image-input call above 16384 keypoints --------------------------------------------------------------------
class _Net(torch.nn.Module):
    """The stand-in descriptor network of test_gpu_pyramid.py / test_gpu_sift.py."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Sequential(torch.nn.Conv2d(3, 32, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(32, 64, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(64, 128, 8))

    def forward(self, x):
        return torch.nn.functional.normalize(self.body(x).flatten(1), dim=1)


def test_image_input_above_16384_keypoints():
    pytest.importorskip('cv2')
    from gims_b200 import Matching
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image, warp_image
    dev = torch.device('cuda:0')
    k = 24576
    torch.manual_seed(0)
    car = types.SimpleNamespace(model=_Net().to(dev).eval(), batch_size=2048)
    img0 = make_textured_image(1800, 2400, seed=91, n_shapes=2400)
    img1, _ = warp_image(img0, seed=92)
    for img in (img0, img1):
        assert fe.detect_device(img, dev, 0).n > k                 # more keypoints than the call keeps
    # threshold 0: every mutual pair is a match (the stand-in network's descriptors give weak evidence at this size)
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.0, 'max_keypoints': k, 'detector': 'device'})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to(dev)
    knobs = {'device': dev, 'radius': 25, 'percentile': 7, 'min_size': 1}
    with torch.no_grad():
        pred = matching({**knobs, 'image0': img0[None], 'image1': img1[None], 'carhynet': car})
    torch.cuda.synchronize()
    assert pred['keypoints0'].shape[1] == k and pred['keypoints1'].shape[1] == k
    m0, m1 = pred['matches0'][0].cpu(), pred['matches1'][0].cpu()
    i = torch.nonzero(m0 >= 0).squeeze(1)
    print('\n[image input, %d keypoints per image] %d mutual matches' % (k, i.numel()))
    assert i.numel() > 0 and (m1[m0[i]] == i).all()
    j = torch.nonzero(m1 >= 0).squeeze(1)
    assert (m0[m1[j]] == j).all() and i.numel() == j.numel()
    del matching, pred, car


# ---- 7. the limit itself ------------------------------------------------------------------------------------------------
def test_matcher_rejects_65537_keypoints():
    from gims_b200 import GMatcher, _lib
    model = GMatcher({}).cuda().eval()
    data = make_pair(_lib.MAX_KPTS + 1, 10, seed=643)
    with pytest.raises(ValueError, match='more than 65536'):
        model.run_pair(data['keypoints0'][0], data['descriptors0'][0], data['scores0'][0], data['keypoints1'][0],
                       data['descriptors1'][0], data['scores1'][0], data['image0'].shape, data['image1'].shape)
