"""GPU parity tests (run on the B200 box: `pytest -m gpu`).

The CUDA path (libgims_b200.so through the C ABI, driven by gims_b200.GMatcher) is compared
  * with the committed golden fixtures produced by the unmodified reference (tests/golden), and
  * with the CPU oracle (oracle/gims_oracle.py) on the same seeded inputs, stage by stage.
Bars (SURVEY.md §8c): kept indices + CSR bit-exact; |dscores| <= 2e-5*max(1,|s|); |dZ|,|du|,|dv| <= 1e-4
(scaled by max(1,|.|)); pre-threshold argmax agreement >= 99.9 % (tie-aware); matching scores within
1e-4*max + 1e-7.
"""
import numpy as np
import pytest
import torch

from golden_util import golden_names, index_agreement, inputs_for, load_golden, weights_for
from gims_b200.synth import make_pair, make_state_dict

pytestmark = pytest.mark.gpu


def _model(sd, cfg):
    from gims_b200 import GMatcher
    m = GMatcher(cfg)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _run_pair(model, data, debug=True):
    dev = torch.device('cuda')
    r = model.run_pair(data['keypoints0'][0].to(dev), data['descriptors0'][0].to(dev), data['scores0'][0].to(dev),
                       data['keypoints1'][0].to(dev), data['descriptors1'][0].to(dev), data['scores1'][0].to(dev),
                       data['image0'].shape, data['image1'].shape, data.get('radius', 25), data.get('percentile', 7),
                       data.get('min_size', 8), debug=debug)
    torch.cuda.synchronize()
    cnt = r['n_kept_dev'].cpu().numpy()
    assert cnt[6] & 0xff == 0, 'error status %#x' % cnt[6]
    return r, cnt


def _csr(r, s, cnt):
    n, e = int(cnt[s]), int(cnt[2 + s])
    return (r['kept_idx%d' % s][:n].cpu().numpy().astype(np.int64),
            r['csr_indptr%d' % s][:n + 1].cpu().numpy().astype(np.int64),
            r['csr_indices%d' % s][:e].cpu().numpy().astype(np.int64))


def _agc_only(data, rec):
    """gims_agc_build through the C ABI for both images."""
    import ctypes as C
    from gims_b200 import _lib
    from gims_b200.gmatcher import GMatcher
    L = _lib.lib()
    dev = torch.device('cuda')
    outs = []
    for s in ('0', '1'):
        kp = data['keypoints' + s][0].to(dev).contiguous()
        de = data['descriptors' + s][0].to(dev).contiguous()
        sc = data['scores' + s][0].to(dev).contiguous()
        n = kp.shape[0]
        cap = max(1024, 64 * n)
        ws = torch.empty(L.gims_agc_workspace_bytes(n, cap), dtype=torch.uint8, device=dev)
        kept = torch.empty(n, dtype=torch.int32, device=dev)
        cnt = torch.zeros(4, dtype=torch.int32, device=dev)       # n_kept, n_edges, n_comp, status
        indptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
        indices = torch.empty(cap, dtype=torch.int32, device=dev)
        kpo = torch.empty(n, 2, device=dev)
        fo = torch.empty(n, 256, device=dev)
        so = torch.empty(n, device=dev)
        thr = torch.zeros(1, device=dev)
        st = torch.cuda.current_stream()
        _lib.check(L.gims_agc_build(_lib.ptr(kp), _lib.ptr(de), 1, _lib.ptr(sc), n, float(rec['radius']),
                                    GMatcher._k_rank(n, rec['percentile']), int(rec['min_size']), _lib.ptr(ws), ws.numel(),
                                    _lib.ptr(kept), C.c_void_p(cnt.data_ptr()), _lib.ptr(indptr), _lib.ptr(indices), cap,
                                    C.c_void_p(cnt.data_ptr() + 4), _lib.ptr(kpo), _lib.ptr(fo), _lib.ptr(so), _lib.ptr(thr),
                                    C.c_void_p(cnt.data_ptr() + 8), C.c_void_p(cnt.data_ptr() + 12),
                                    C.c_void_p(st.cuda_stream)), 'gims_agc_build')
        torch.cuda.synchronize()
        c = cnt.cpu().numpy()
        assert c[3] == 0
        nk, ne = int(c[0]), int(c[1])
        outs.append(dict(kept=kept[:nk].cpu().numpy().astype(np.int64), indptr=indptr[:nk + 1].cpu().numpy().astype(np.int64),
                         indices=indices[:ne].cpu().numpy().astype(np.int64), n_comp=int(c[2]), thr=float(thr.cpu()),
                         kpts=kpo[:nk].cpu(), feat=fo[:nk].cpu(), scores=so[:nk].cpu()))
    return outs


@pytest.mark.parametrize('name', golden_names('agc_'))
def test_agc_golden_bit_exact(name):
    """a-1..a-7 against the reference's own graphs (tests/golden/agc_*.npz)."""
    rec, g = load_golden(name)
    data = inputs_for(rec)
    outs = _agc_only(data, rec)
    for s, o in zip(('0', '1'), outs):
        assert np.array_equal(o['kept'], g['kept' + s]), 'kept indices differ (image %s)' % s
        assert np.array_equal(o['indptr'], g['csr_indptr' + s]), 'indptr differs (image %s)' % s
        assert np.array_equal(o['indices'], g['csr_indices' + s]), 'indices differ (image %s)' % s
        kept = torch.from_numpy(o['kept'])
        assert torch.equal(o['kpts'], data['keypoints' + s][0][kept])
        assert torch.equal(o['feat'], data['descriptors' + s][0].t()[kept])
        assert torch.equal(o['scores'], data['scores' + s][0][kept])


@pytest.mark.parametrize('n,width,height,r,p,m,seed', [
    (700, 500, 400, 25, 7, 8, 101), (333, 300, 300, 10, 30, 2, 102), (1500, 800, 600, 15, 2, 7, 103),
    (2048, 640, 480, 25, 7, 8, 104), (97, 60, 60, 9, 0, 1, 105), (512, 2000, 2000, 25, 7, 8, 106),
])
def test_agc_vs_oracle(n, width, height, r, p, m, seed):
    """a-1..a-7 against the oracle, including the threshold value and the component count."""
    from oracle import gims_oracle as orc
    rec = dict(radius=r, percentile=p, min_size=m)
    data = make_pair(n, max(2, n - 17), seed=seed, width=width, height=height)
    outs = _agc_only(data, rec)
    for s, o in zip(('0', '1'), outs):
        ref = orc.agc_build(data['keypoints' + s][0].numpy(), data['descriptors' + s][0].t().contiguous().numpy(), r, p, m)
        assert np.float32(o['thr']) == ref['thr'], 'cosine threshold differs'
        assert np.array_equal(o['kept'], ref['kept'])
        assert np.array_equal(o['indptr'], ref['indptr'])
        assert np.array_equal(o['indices'], ref['indices'])
        assert o['n_comp'] == ref['n_components']


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(1.0, np.abs(b))


def _sinkhorn_f64(coup, iters):
    """The reference's iteration (gmatcher.py:41-69) in float64 on the GPU, on OUR couplings: the exact-arithmetic
    yardstick for the potentials."""
    z = coup.double()
    n0, n1 = z.shape[0] - 1, z.shape[1] - 1
    norm = -np.log(n0 + n1)
    lmu = torch.full((n0 + 1,), norm, dtype=torch.float64, device=z.device)
    lnu = torch.full((n1 + 1,), norm, dtype=torch.float64, device=z.device)
    lmu[-1] = np.log(n1) + norm
    lnu[-1] = np.log(n0) + norm
    u, v = torch.zeros_like(lmu), torch.zeros_like(lnu)
    for _ in range(iters):
        u = lmu - torch.logsumexp(z + v[None, :], 1)
        v = lnu - torch.logsumexp(z + u[:, None], 0)
    return u.cpu().numpy(), v.cpu().numpy()


def _check_forward(rec, data, sd, cfg, ref, label):
    """ref: dict with the reference/oracle values (full or sub-sampled)."""
    model = _model(sd, cfg)
    r, cnt = _run_pair(model, data)
    n0, n1 = int(cnt[0]), int(cnt[1])
    n0_in = data['keypoints0'].shape[1]
    msgs = []
    for s in (0, 1):
        kept, indptr, indices = _csr(r, s, cnt)
        assert np.array_equal(kept, ref['kept%d' % s]), label + ': kept%d' % s
        assert np.array_equal(indices, ref['csr_indices%d' % s]), label + ': csr%d' % s
    coup = r['couplings'].cpu().numpy()
    scores = coup[:n0, :n1]
    assert np.all(coup[n0, :n1 + 1] == float(sd['bin_score'])) and np.all(coup[:n0 + 1, n1] == float(sd['bin_score']))
    sub = ref['scores_sub'].shape
    e_sc = _rel(scores[:sub[0], :sub[1]], ref['scores_sub']).max()
    msgs.append('scores %.2e' % e_sc)
    u, v = r['u'].cpu().numpy()[:n0 + 1], r['v'].cpu().numpy()[:n1 + 1]
    # Potentials.  u and v are individually ill-conditioned: shifting every u_r by +c and every v_j by -c is a
    # neutrally stable mode of the iteration (only u_r + v_j, i.e. Z, is well determined), so fp32 rounding drifts
    # along it — the reference's own fp32 potentials deviate from a float64 run of the same iteration by up to
    # ~6e-4 when the scores sit near 90.  Bars: (1) ours within 1e-4 * max(1, |.|) of the float64 iteration on our
    # couplings; (2) ours within 1e-4 * max(1, |.|) + (the reference's own distance from that float64 run) of the reference.
    u64, v64 = _sinkhorn_f64(r['couplings'][:n0 + 1, :n1 + 1], cfg['sinkhorn_iterations'])
    e_u64, e_v64 = _rel(u, u64).max(), _rel(v, v64).max()
    ref_u64, ref_v64 = np.abs(ref['u'] - u64).max(), np.abs(ref['v'] - v64).max()
    e_u = (np.maximum(np.abs(u - ref['u']) - ref_u64, 0) / np.maximum(1.0, np.abs(ref['u']))).max()
    e_v = (np.maximum(np.abs(v - ref['v']) - ref_v64, 0) / np.maximum(1.0, np.abs(ref['v']))).max()
    msgs.append('u,v vs f64 %.2e %.2e; vs reference raw %.2e %.2e (reference vs f64: %.2e %.2e abs)' %
                (e_u64, e_v64, _rel(u, ref['u']).max(), _rel(v, ref['v']).max(), ref_u64, ref_v64))
    assert e_u64 <= 1e-4 and e_v64 <= 1e-4, msgs
    # Z of ours from our own potentials (the fused kernel never materialises it)
    norm = -np.log(np.float32(n0 + n1))
    z_ours = (coup[:n0 + 1, :n1 + 1] + u[:, None]) + v[None, :] - norm
    e_z = _rel(z_ours[:sub[0], :sub[1]], ref['Z_sub']).max()
    msgs.append('Z %.2e' % e_z)
    i0, i1 = r['indices0'][:n0].cpu().numpy(), r['indices1'][:n1].cpu().numpy()
    # tie-aware agreement, judged on our Z (close to the reference's within e_z)
    zi = z_ours[:n0, :n1]
    a0 = index_agreement(i0, ref['indices0'], zi[np.arange(n0), i0], zi[np.arange(n0), ref['indices0']])
    a1 = index_agreement(i1, ref['indices1'], zi[i1, np.arange(n1)], zi[ref['indices1'], np.arange(n1)])
    raw0, raw1 = (i0 == ref['indices0']).mean(), (i1 == ref['indices1']).mean()
    msgs.append('argmax agree raw %.4f/%.4f tie-aware %.4f/%.4f' % (raw0, raw1, a0, a1))
    m0, m1 = r['matches0'][:n0].cpu().numpy(), r['matches1'][:n1].cpu().numpy()
    ms0, ms1 = r['mscores0'][:n0].cpu().numpy(), r['mscores1'][:n1].cpu().numpy()
    am0, am1 = (m0 == ref['matches0']).mean(), (m1 == ref['matches1']).mean()
    tol_ms = 1e-4 * max(ref['matching_scores0'].max(), 1e-3) + 1e-7
    # scores of keypoints whose mutual status agrees
    same0 = (ms0 > 0) == (ref['matching_scores0'] > 0)
    e_ms = np.abs(ms0 - ref['matching_scores0'])[same0].max() if same0.any() else 0.0
    msgs.append('matches agree %.4f/%.4f, mscores err %.2e (tol %.2e), mutual-status agree %.4f' %
                (am0, am1, e_ms, tol_ms, same0.mean()))
    md = r['mdesc'].cpu().numpy()
    e_md = (np.abs(md[:sub[0]] - ref['mdesc0_sub']).max() / max(1e-6, np.abs(ref['mdesc0_sub']).max()))
    msgs.append('mdesc rel %.2e' % e_md)
    print('\n[%s] N\'=(%d,%d) ' % (label, n0, n1) + '; '.join(msgs))
    assert e_sc <= 2e-5, msgs
    assert e_u <= 1e-4 and e_v <= 1e-4 and e_z <= 1e-4, msgs
    assert a0 >= 0.999 and a1 >= 0.999, msgs
    assert am0 >= 0.999 and am1 >= 0.999, msgs
    assert e_ms <= tol_ms and same0.mean() >= 0.999, msgs
    assert e_md <= 2e-5, msgs
    assert r['matches0'].dtype == torch.int64 and r['mscores0'].dtype == torch.float32
    return r, cnt


@pytest.mark.parametrize('name', golden_names('fwd_'))
def test_forward_golden(name):
    """Whole forward (a-1..a-15) against the reference's outputs (tests/golden/fwd_*.npz)."""
    rec, g = load_golden(name)
    data = inputs_for(rec)
    sd = weights_for(rec)
    cfg = {'sinkhorn_iterations': rec['iters'], 'match_threshold': rec['match_threshold']}
    ref = {k: g[k] for k in g.files if k != 'recipe'}
    _check_forward(rec, data, sd, cfg, ref, name)


def test_forward_stages_vs_oracle():
    """Stage-by-stage against the oracle on a ragged pair: SAGE+kenc, every attention layer's output,
    mdesc, scores, potentials, matches."""
    from oracle import gims_oracle as orc
    data = make_pair(600, 555, seed=301, width=420, height=330)
    data.update({'radius': 25, 'percentile': 7, 'min_size': 8})
    sd = make_state_dict(3, damped=True)
    cfg = {'sinkhorn_iterations': 50, 'match_threshold': 0.01}
    with torch.no_grad():
        out = orc.gmatcher_forward(sd, data, cfg, stages=True)
    st = out['_stages']
    ref = {'scores_sub': st['scores'][0].numpy(), 'Z_sub': st['Z'][0, :-1, :-1].numpy(), 'u': st['u'][0].numpy(),
           'v': st['v'][0].numpy(), 'indices0': st['indices0'][0].numpy(), 'indices1': st['indices1'][0].numpy(),
           'matches0': out['matches0'][0].numpy(), 'matches1': out['matches1'][0].numpy(),
           'matching_scores0': out['matching_scores0'][0].numpy(), 'matching_scores1': out['matching_scores1'][0].numpy(),
           'mdesc0_sub': out['mdesc0'].numpy()}
    for s in (0, 1):
        ref['kept%d' % s] = st['graph%d' % s]['kept']
        ref['csr_indices%d' % s] = st['graph%d' % s]['indices']
    r, cnt = _check_forward(None, data, sd, cfg, ref, 'stages')
    n0, n1, n0_in = int(cnt[0]), int(cnt[1]), 600
    din = r['desc_in'].cpu()
    for s, (a, b) in enumerate(((0, n0), (n0_in, n0_in + n1))):
        want = st['desc_in%d' % s][0].t()
        err = (din[a:b] - want).abs().max() / want.abs().max()
        print('desc_in%d rel err %.2e' % (s, err))
        assert err <= 1e-5
    dg = r['desc_gnn'].cpu()
    for s, (a, b) in enumerate(((0, n0), (n0_in, n0_in + n1))):
        want = st['desc_out%d' % s][0].t()
        err = (dg[a:b] - want).abs().max() / want.abs().max()
        print('desc_gnn%d rel err %.2e' % (s, err))
        assert err <= 2e-5


@pytest.mark.parametrize('n0,n1,iters,scale,aligned,offset', [
    (1, 1, 3, 1.0, True, 0.0), (5, 9, 100, 1.0, True, 0.0), (300, 257, 20, 5.0, True, 0.0), (2048, 2048, 100, 1.0, True, 0.0),
    (2048, 2040, 100, 2.6, True, 90.0),       # trained-like: scores ~ 90 +- 2.6 against a dustbin score of 0.7
    (1000, 3100, 10, 30.0, True, 0.0), (4500, 4000, 4, 1.0, True, 0.0), (4500, 4000, 100, 3.0, True, 90.0),
    (8200, 8100, 30, 1.0, True, 0.0),
    (1500, 11000, 10, 2.0, True, 50.0),       # > 10240 columns: nine column groups per thread, rows re-read from the stage,
                                              # one-row blocks (the widest streaming instantiation)
    (600, 15000, 5, 1.0, True, 0.0),          # no room for two stages next to v and w: the exact kernel
    (3000, 2500, 10, 2.0, False, 50.0),       # unaligned pitch: the exact kernel
    (700, 650, 30, 60.0, True, 0.0),          # very spread scores
])
def test_sinkhorn_vs_oracle(n0, n1, iters, scale, aligned, offset):
    """a-14/a-15 alone on random couplings: register-resident, streamed (L2 / HBM) and exact kernels, ragged, tiny."""
    import ctypes as C
    from gims_b200 import _lib
    from oracle import gims_oracle as orc
    L = _lib.lib()
    g = torch.Generator().manual_seed(n0 * 7 + n1)
    scores = torch.randn(1, n0, n1, generator=g) * scale + offset
    alpha = torch.tensor(0.7)
    # yardstick: the reference's iteration evaluated in float64 on the same fp32 couplings (its fp32 evaluation drifts
    # along the neutral u + c / v - c mode by more than our tolerance when the scores are large, see _check_forward)
    z, u, v, coup = orc.log_optimal_transport(scores.double(), alpha.double(), iters)
    z, u, v, coup = z.float(), u.float(), v.float(), coup.float()
    m = orc.extract_matches(z, 0.0)
    dev = torch.device('cuda')
    # exercise device-side counts: allocate for larger maxima than the live sizes
    n0m, n1m = n0 + 3, n1 + 5
    ld = L.gims_couplings_ld(n1m) if aligned else n1m + 1
    cbuf = torch.zeros(n0m + 1, ld, device=dev)
    cbuf[:n0 + 1, :n1 + 1] = coup[0].to(dev)
    cbuf = cbuf.contiguous()
    nd = torch.tensor([n0, n1], dtype=torch.int32, device=dev)
    ws = torch.empty(L.gims_sinkhorn_workspace_bytes(n0m, n1m), dtype=torch.uint8, device=dev)
    uo, vo = torch.zeros(n0m + 1, device=dev), torch.zeros(n1m + 1, device=dev)
    i0, i1 = torch.zeros(n0m, dtype=torch.int32, device=dev), torch.zeros(n1m, dtype=torch.int32, device=dev)
    m0, m1 = torch.zeros(n0m, dtype=torch.int64, device=dev), torch.zeros(n1m, dtype=torch.int64, device=dev)
    s0, s1 = torch.zeros(n0m, device=dev), torch.zeros(n1m, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(L.gims_sinkhorn_match(_lib.ptr(cbuf), ld, n0m, n1m, _lib.ptr(nd), iters, 0.0, _lib.ptr(ws), ws.numel(),
                                     _lib.ptr(uo), _lib.ptr(vo), _lib.ptr(i0), _lib.ptr(i1), _lib.ptr(m0), _lib.ptr(m1),
                                     _lib.ptr(s0), _lib.ptr(s1), _lib.ptr(status),
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream)),
               'gims_sinkhorn_match')
    torch.cuda.synchronize()
    st_word = int(status.cpu())
    assert st_word & _lib.STATUS_ERROR_MASK == 0, 'status %#x' % st_word
    assert st_word & (_lib.STATUS_SINKHORN_FAST | _lib.STATUS_SINKHORN_EXACT)
    eu = _rel(uo[:n0 + 1].cpu().numpy(), u[0].numpy()).max()
    ev = _rel(vo[:n1 + 1].cpu().numpy(), v[0].numpy()).max()
    zi = z[0, :-1, :-1].numpy()
    a0 = index_agreement(i0[:n0].cpu().numpy(), m['indices0'][0].numpy(), zi.max(1),
                         zi[np.arange(n0), i0[:n0].cpu().numpy()])
    a1 = index_agreement(i1[:n1].cpu().numpy(), m['indices1'][0].numpy(), zi.max(0),
                         zi[i1[:n1].cpu().numpy(), np.arange(n1)])
    # mutual status may legitimately flip where a column has an (almost) exact tie between two rows:
    # such rows are excused only if the oracle's own column gap is below 1e-3
    ours_ms, ref_ms = s0[:n0].cpu().numpy(), m['matching_scores0'][0].numpy()
    flip = np.nonzero((ours_ms > 0) != (ref_ms > 0))[0]
    for i in flip:
        col = np.sort(zi[:, int(m['indices0'][0, i])])
        assert col[-1] - col[-2] < 1e-3, 'mutual status of row %d differs without a tie' % i
    keep = np.ones(n0, dtype=bool)
    keep[flip] = False
    ems = np.abs(ours_ms - ref_ms)[keep].max() if keep.any() else 0.0
    print('\n[sinkhorn %dx%d it=%d status %#x] du %.2e dv %.2e agree %.4f/%.4f dms %.2e tie-flips %d' %
          (n0, n1, iters, st_word, eu, ev, a0, a1, ems, len(flip)))
    assert eu <= 1e-4 and ev <= 1e-4
    assert a0 >= 0.999 and a1 >= 0.999
    # (the column sums are float atomics: which of two tied rows wins varies from run to run, 2 .. 6 flips seen at 700 x 650)
    assert len(flip) <= max(8, n0 // 100)
    assert ems <= 1e-4 * max(1e-3, float(m['matching_scores0'].max())) + 1e-6
    same = (m0[:n0].cpu() == m['matches0'][0]).numpy()[keep].mean()
    assert same >= 0.999


def test_drop_in_call_signature():
    """The reference-facing call: Matching(config)(data) with host tensors, dict in / dict out, the
    side effects of gmatcher.py:244-252, dtypes and shapes of matching.py / gmatcher.py:296-307."""
    from gims_b200 import Matching
    rec, g = load_golden('fwd_n512_damped')
    data = inputs_for(rec)
    data['device'] = 'cuda'
    matching = Matching({'sinkhorn_iterations': rec['iters'], 'match_threshold': rec['match_threshold']})
    matching.gmodel.load_state_dict(weights_for(rec))
    matching = matching.eval().to('cuda')
    with torch.no_grad():
        pred = matching(data)
    n0, n1 = len(g['kept0']), len(g['kept1'])
    assert pred['keypoints0'].shape == (1, n0, 2) and pred['descriptors0'].shape == (1, 256, n0)
    assert pred['matches0'].shape == (1, n0) and pred['matches0'].dtype == torch.int64
    assert pred['matches1'].shape == (1, n1) and pred['matching_scores1'].shape == (1, n1)
    assert pred['mdesc0'].shape == (n0, 256) and pred['mdesc1'].shape == (n1, 256)
    assert (pred['matches0'][0].cpu().numpy() == g['matches0']).mean() >= 0.999
    assert np.allclose(pred['keypoints0'][0].cpu().numpy(), g['keypoints0'])
    pred_np = {k: v[0].cpu().numpy() for k, v in pred.items()}       # what eval_homography.py:181 does
    assert pred_np['matches0'].shape == (n0,)


def test_edge_cap_overflow_retry():
    """gmatcher.py host loop: an edge list that does not fit makes the kernels report an EMPTY graph + the overflow bit
    (nothing downstream walks the unwritten CSR); forward() retries with 4x the capacity until it fits and then returns
    the same result as a roomy first attempt."""
    from gims_b200 import Matching, _lib
    rec, g = load_golden('fwd_n512_damped')
    data = inputs_for(rec)
    data['device'] = 'cuda'
    matching = Matching({'sinkhorn_iterations': rec['iters'], 'match_threshold': rec['match_threshold']})
    matching.gmodel.load_state_dict(weights_for(rec))
    matching = matching.eval().to('cuda')
    # the raw single attempt with a capacity that cannot hold the graph: status bit set, graph reported empty
    gm = matching.gmodel
    dev = torch.device('cuda')
    r = gm.run_pair(data['keypoints0'][0].to(dev), data['descriptors0'][0].to(dev), data['scores0'][0].to(dev),
                    data['keypoints1'][0].to(dev), data['descriptors1'][0].to(dev), data['scores1'][0].to(dev),
                    data['image0'].shape, data['image1'].shape, rec['radius'], rec['percentile'], rec['min_size'],
                    edge_cap=256)
    torch.cuda.synchronize()
    cnt = r['n_kept_dev'].cpu().numpy()
    assert cnt[6] & _lib.STATUS_EDGE_OVERFLOW
    assert cnt[0] == 0 or cnt[1] == 0
    # the reference-facing call recovers by itself
    gm.edge_cap_factor = 0           # -> initial capacity 1024 directed edges (the graph has several thousand)
    with torch.no_grad():
        pred = matching(dict(data))
    torch.cuda.synchronize()
    assert pred['keypoints0'].shape[1] == len(g['kept0'])
    assert (pred['matches0'][0].cpu().numpy() == g['matches0']).mean() >= 0.999
    assert (pred['matches1'][0].cpu().numpy() == g['matches1']).mean() >= 0.999


def test_all_pruned_image():
    """gmatcher.py:257-264: when AGC removes every keypoint of an image the reference returns int32 -1 matches and
    zero scores of shape (B, 0) / (B, N1')."""
    from gims_b200 import Matching
    data = make_pair(200, 180, seed=611, width=2000, height=2000)     # sparse: no component reaches min_size
    data.update({'radius': 5, 'percentile': 7, 'min_size': 50, 'device': 'cuda'})
    matching = Matching({'sinkhorn_iterations': 10}).eval().to('cuda')
    with torch.no_grad():
        pred = matching.gmodel(data)      # GMatcher mutates ITS argument (Matching passes it a copy, matching.py:25)
    torch.cuda.synchronize()
    assert set(pred) == {'matches0', 'matches1', 'matching_scores0', 'matching_scores1'}
    assert pred['matches0'].shape == (1, 0) and pred['matches0'].dtype == torch.int32
    assert pred['matching_scores1'].shape == (1, 0) and float(pred['matching_scores1'].sum()) == 0.0
    assert data['keypoints0'].shape == (1, 0, 2) and data['kept_kpts0_indices'] == [[]]


def test_other_network_configuration_vs_oracle():
    """The constructor config is honoured (gmatcher.py:166-176, 136-140): 4 attention layers in the order self / self /
    cross / cross and a 3-conv keypoint encoder (its last conv is K = 64 -> N = 256: one k-block per tile in the persistent
    GEMM), against the oracle run on the same weights and inputs."""
    from gims_b200 import Matching
    from oracle import gims_oracle as orc
    cfg = {'transformer_layers': ['self', 'self', 'cross', 'cross'], 'keypoint_encoder': [32, 64],
           'sinkhorn_iterations': 25, 'match_threshold': 0.01}
    sd = make_state_dict(13, damped=True, config=cfg)
    data = make_pair(420, 390, seed=633, width=360, height=280)
    data.update({'radius': 25, 'percentile': 7, 'min_size': 8})
    with torch.no_grad():
        want = orc.gmatcher_forward(sd, dict(data), cfg)
    m = Matching(cfg)
    m.gmodel.load_state_dict(sd)
    m = m.eval().to('cuda')
    with torch.no_grad():
        got = m({**data, 'device': 'cuda'})
    torch.cuda.synchronize()
    assert torch.equal(got['keypoints0'].cpu(), want['keypoints0']) and torch.equal(got['keypoints1'].cpu(), want['keypoints1'])
    assert (got['matches0'].cpu() == want['matches0']).float().mean().item() >= 0.999
    assert (got['matches1'].cpu() == want['matches1']).float().mean().item() >= 0.999
    scale = max(1e-3, float(want['matching_scores0'].max()))
    assert (got['matching_scores0'].cpu() - want['matching_scores0']).abs().max().item() <= 1e-4 * scale + 1e-6
    md = want['mdesc0']
    assert torch.allclose(got['mdesc0'].cpu(), md, rtol=1e-4, atol=1e-4 * float(md.abs().max()))
    assert int((want['matches0'] >= 0).sum()) > 10


@pytest.mark.parametrize('n0,n1,seed', [(2, 2, 650), (3, 9, 651), (17, 5, 652)])
def test_tiny_forward_vs_oracle(n0, n1, seed):
    """The smallest inputs the reference accepts (two keypoints: one candidate pair for the percentile) through the whole
    path, nothing pruned (min_size 1): one partial row tile, one key tile, a Sinkhorn slab of a single CTA."""
    from gims_b200 import Matching
    from oracle import gims_oracle as orc
    cfg = {'sinkhorn_iterations': 15, 'match_threshold': 0.0}
    sd = make_state_dict(2, damped=True)
    data = make_pair(n0, n1, seed=seed, width=60, height=50)
    data.update({'radius': 40, 'percentile': 7, 'min_size': 1})
    with torch.no_grad():
        want = orc.gmatcher_forward(sd, dict(data), cfg)
    m = Matching(cfg)
    m.gmodel.load_state_dict(sd)
    m = m.eval().to('cuda')
    with torch.no_grad():
        got = m({**data, 'device': 'cuda'})
    torch.cuda.synchronize()
    assert got['keypoints0'].shape == want['keypoints0'].shape and got['keypoints1'].shape == want['keypoints1'].shape
    assert torch.equal(got['keypoints0'].cpu(), want['keypoints0'])
    assert torch.equal(got['matches0'].cpu(), want['matches0']) and torch.equal(got['matches1'].cpu(), want['matches1'])
    assert torch.allclose(got['matching_scores0'].cpu(), want['matching_scores0'], atol=1e-5)
    md = want['mdesc0']
    assert torch.allclose(got['mdesc0'].cpu(), md, rtol=1e-4, atol=1e-4 * float(md.abs().max()))


def test_forward_at_maximum_size_properties():
    """GIMS_MAX_KPTS = 16384 keypoints per image (the CPU reference needs tens of minutes there): size-independent
    properties of the result — status clean, kept indices ascending, CSR sorted / symmetric / loop-free, matches mutual,
    scores in (0, 1], potentials finite.  16385 columns exceed the streaming kernel's shared-memory budget: this is the
    exact Sinkhorn kernel at full size."""
    from gims_b200 import Matching, _lib
    n = _lib.MAX_KPTS
    cfg = {'sinkhorn_iterations': 5, 'match_threshold': 0.0}
    m = Matching(cfg)
    m.gmodel.load_state_dict(make_state_dict(3, damped=True))
    m = m.eval().to('cuda')
    data = make_pair(n, n, seed=640, width=2400, height=1800)
    data.update({'radius': 25, 'percentile': 7, 'min_size': 8, 'device': 'cuda'})
    with torch.no_grad():
        pred = m.gmodel(data)
    torch.cuda.synchronize()
    n0, n1 = pred['matches0'].shape[1], pred['matches1'].shape[1]
    assert 0.9 * n <= n0 <= n and 0.9 * n <= n1 <= n
    k0 = torch.tensor(data['kept_kpts0_indices'][0])
    assert (k0[1:] > k0[:-1]).all() and k0.numel() == n0
    indptr, indices = [t.cpu().long() for t in data['graph0'][0]]
    assert indptr[0] == 0 and indptr[-1] == indices.numel() and (indptr[1:] >= indptr[:-1]).all()
    rows = torch.repeat_interleave(torch.arange(n0), indptr[1:] - indptr[:-1])
    assert (rows != indices).all()                                            # no self loops
    key = rows * n0 + indices
    assert (key[1:] > key[:-1]).all()                                         # rows ascending, neighbours ascending, no duplicates
    assert torch.equal(torch.sort(indices * n0 + rows).values, key)           # every edge has its reverse
    m0, m1 = pred['matches0'][0].cpu(), pred['matches1'][0].cpu()
    i = torch.nonzero(m0 >= 0).squeeze(1)
    assert i.numel() > 100 and (m1[m0[i]] == i).all()                         # mutual
    j = torch.nonzero(m1 >= 0).squeeze(1)
    assert (m0[m1[j]] == j).all() and i.numel() == j.numel()
    s0 = pred['matching_scores0'][0].cpu()
    assert torch.isfinite(s0).all() and (s0[i] > 0).all() and (s0 <= 1.0 + 1e-5).all() and (s0[m0 < 0] == 0).all()


def test_batch_of_two_equal_sizes():
    """Batch > 1 works in the reference only when every item keeps the same N' (torch.stack, gmatcher.py:244-249);
    with min_size = 1 nothing is pruned.  Each item must equal its own single call."""
    from gims_b200 import Matching
    cfg = {'sinkhorn_iterations': 20, 'match_threshold': 0.005}
    matching = Matching(cfg)
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to('cuda')
    items = [make_pair(300, 280, seed=620 + k, width=300, height=240) for k in range(2)]
    knobs = {'radius': 25, 'percentile': 7, 'min_size': 1, 'device': 'cuda'}
    batch = {k: (torch.cat([it[k] for it in items]) if torch.is_tensor(items[0][k]) else items[0][k]) for k in items[0]}
    batch.update(knobs)
    with torch.no_grad():
        pb = matching(batch)
        singles = [matching({**it, **knobs}) for it in items]
    torch.cuda.synchronize()
    assert pb['matches0'].shape == (2, 300) and pb['descriptors1'].shape == (2, 256, 280)
    assert pb['mdesc0'].shape == (2, 300, 256)
    for k, ps in enumerate(singles):
        assert torch.equal(pb['matches0'][k], ps['matches0'][0]) and torch.equal(pb['matches1'][k], ps['matches1'][0])
        assert torch.allclose(pb['matching_scores0'][k], ps['matching_scores0'][0], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize('name', ['fwd_n512_damped', 'fwd_n2048_damped'])
def test_bf16_variant_report(name):
    """The bf16 variant (GIMS_GEMM_BF16: attention operands in bf16) is NOT an fp32-parity path: its agreement with the
    reference's fixtures is measured and printed ("reported separately", BASELINE.json north_star); only sanity is
    asserted."""
    from gims_b200 import _lib
    rec, g = load_golden(name)
    data = inputs_for(rec)
    model = _model(weights_for(rec), {'sinkhorn_iterations': rec['iters'], 'match_threshold': rec['match_threshold']})
    dev = torch.device('cuda')
    r = model.run_pair(data['keypoints0'][0].to(dev), data['descriptors0'][0].to(dev), data['scores0'][0].to(dev),
                       data['keypoints1'][0].to(dev), data['descriptors1'][0].to(dev), data['scores1'][0].to(dev),
                       data['image0'].shape, data['image1'].shape, rec['radius'], rec['percentile'], rec['min_size'],
                       debug=True, gemm_mode=_lib.GEMM_BF16)
    torch.cuda.synchronize()
    cnt = r['n_kept_dev'].cpu().numpy()
    n0, n1 = int(cnt[0]), int(cnt[1])
    assert cnt[6] & 0xff == 0
    sub = g['scores_sub'].shape
    sc = r['couplings'].cpu().numpy()[:sub[0], :sub[1]]
    e_sc = _rel(sc, g['scores_sub']).max()
    i0 = r['indices0'][:n0].cpu().numpy()
    m0 = r['matches0'][:n0].cpu().numpy()
    ms0 = r['mscores0'][:n0].cpu().numpy()
    agree_idx, agree_m = (i0 == g['indices0']).mean(), (m0 == g['matches0']).mean()
    both = (m0 >= 0) & (g['matches0'] >= 0)
    e_ms = np.abs(ms0 - g['matching_scores0'])[both].max() if both.any() else 0.0
    print('\n[bf16 variant %s] N\'=(%d,%d): scores rel err %.2e (fp32 path: 5e-6); argmax agreement %.4f; matches agreement '
          '%.4f (%d reference matches); matching-score err on common matches %.2e' %
          (name, n0, n1, e_sc, agree_idx, agree_m, int((g['matches0'] >= 0).sum()), e_ms))
    assert agree_idx >= 0.9 and agree_m >= 0.9


class _PatchNet(torch.nn.Module):
    """Stands in for the caller's CAR-HyNet (whose definition lives in the reference, not here): colour 32x32 patches ->
    unit-norm 128-d descriptors, random init.  The front-end treats the caller's network as opaque."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Sequential(torch.nn.Conv2d(3, 32, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(32, 64, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(64, 128, 8))

    def forward(self, x):
        return torch.nn.functional.normalize(self.body(x).flatten(1), dim=1)


def test_eval_homography_literal_call():
    """§8f row 1: the call every script of the reference makes (eval_homography.py:177) — images + the caller's descriptor
    network, no keypoints — against the same call with the front-end run by hand and fed in as keypoints / descriptors.
    The network is `_PatchNet`, a stand-in, not the reference's CAR-HyNet: both calls run the same network, which is all
    the comparison needs."""
    import types
    pytest.importorskip('cv2')
    from gims_b200 import Matching, frontend
    from gims_b200.synth import make_textured_image, warp_image
    dev = torch.device('cuda')
    torch.manual_seed(0)
    car = types.SimpleNamespace(model=_PatchNet().to(dev).eval(), batch_size=512)   # the wrapper's fields describe() reads
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.01, 'max_keypoints': 700})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to(dev)
    img0 = make_textured_image(300, 400, seed=7)
    img1, _ = warp_image(img0, seed=8)
    knobs = {'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7}
    with torch.no_grad():
        pred = matching({**knobs, 'image0': img0[None], 'image1': img1[None], 'carhynet': car})
    out = {k: v[0].cpu().numpy() for k, v in pred.items()}                 # eval_homography.py:181
    assert out['keypoints0'].shape[1] == 2 and out['matches0'].shape[0] == out['keypoints0'].shape[0]
    assert pred['descriptors0'].is_cuda and pred['descriptors0'].shape[1] == 256
    # the same through the keypoint interface
    feats = frontend.sift_forward({'image': img0[None], 'max_keypoints': 700, 'carhynet': car}, dev)
    feats1 = frontend.sift_forward({'image': img1[None], 'max_keypoints': 700, 'carhynet': car}, dev)
    data = {**knobs, 'image0': img0[None], 'image1': img1[None]}
    for s, f in (('0', feats), ('1', feats1)):
        data['keypoints' + s] = torch.stack(f['keypoints'])
        data['scores' + s] = torch.stack(f['scores'])
        data['descriptors' + s] = torch.stack(f['descriptors'])
    with torch.no_grad():
        pred2 = matching(data)
    assert torch.equal(pred['matches0'], pred2['matches0']) and torch.equal(pred['keypoints1'], pred2['keypoints1'])
    d = feats['descriptors'][0]
    assert torch.equal(d[:128], d[128:]) and abs(float(d[:128, 0].norm()) - 1.0) < 1e-4


def test_batched_pairs_equal_single():
    """gims_forward_pairs: a batch of pairs of different sizes, stacked into shared launches, must give what the same pairs
    give one by one (same kernels, same arithmetic per row: bit-identical up to the fp32 atomics of the Sinkhorn)."""
    cfg = {'sinkhorn_iterations': 30, 'match_threshold': 0.005}
    model = _model(make_state_dict(0, damped=True), cfg)
    dev = torch.device('cuda')
    sizes = [(300, 280), (513, 450), (128, 190), (700, 700)]
    items = []
    for k, (a, b) in enumerate(sizes):
        d = make_pair(a, b, seed=700 + k, width=400, height=300)
        items.append((d['keypoints0'][0].to(dev), d['descriptors0'][0].to(dev), d['scores0'][0].to(dev),
                      d['keypoints1'][0].to(dev), d['descriptors1'][0].to(dev), d['scores1'][0].to(dev),
                      d['image0'].shape, d['image1'].shape))
    singles = [model.run_pair(*it, debug=True) for it in items]
    torch.cuda.synchronize()
    for nb in (4, 3, 2):
        batch = model.run_pairs(items[:nb], debug=True)
        torch.cuda.synchronize()
        for k in range(nb):
            a, b = singles[k], batch[k]
            ca, cb = a['n_kept_dev'].cpu(), b['n_kept_dev'].cpu()
            assert torch.equal(ca[:6], cb[:6]) and int(cb[6]) & 0xff == 0
            n0, n1 = int(ca[0]), int(ca[1])
            assert torch.equal(a['kept_idx0'][:n0], b['kept_idx0'][:n0])
            live = torch.cat([torch.arange(n0), sizes[k][0] + torch.arange(n1)]).to(dev)     # rows past N' are scratch
            assert torch.equal(a['desc_gnn'][live], b['desc_gnn'][live])          # same kernels, same per-row arithmetic
            assert torch.equal(a['mdesc'][live], b['mdesc'][live])
            assert torch.equal(a['couplings'][:n0 + 1, :n1 + 1], b['couplings'][:n0 + 1, :n1 + 1])
            assert torch.equal(a['matches0'][:n0], b['matches0'][:n0]) and torch.equal(a['matches1'][:n1], b['matches1'][:n1])
            assert torch.allclose(a['mscores0'][:n0], b['mscores0'][:n0], rtol=1e-4, atol=1e-6)


def test_concurrent_callers_match_sequential():
    """Several host threads calling Matching(data) at once (one CUDA stream each, host inputs) — how bench.py measures
    `e2e` — must give what the same calls give one after the other: per-stream workspaces, the locked
    cooperative-launch chain and the thread-local error state are what this exercises."""
    import threading
    from gims_b200 import Matching
    cfg = {'sinkhorn_iterations': 20, 'match_threshold': 0.005}
    matching = Matching(cfg)
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to('cuda')
    items = []
    for k in range(8):
        d = make_pair(300 + 37 * k, seed=500 + k)
        d['device'] = 'cuda'
        items.append(d)

    def call(d):
        with torch.no_grad():
            pred = matching(dict(d))
        return {k: pred[k][0].cpu() for k in ('matches0', 'matches1', 'matching_scores0', 'keypoints0')}

    sequential = [call(d) for d in items]
    results = [None] * len(items)
    errors = []

    def worker(tid):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for rep in range(3):                                  # several calls per thread, interleaved with the others
                    for k in range(tid, len(items), 4):
                        results[k] = call(items[k])
        except Exception as exc:                                      # noqa: BLE001
            errors.append(exc)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    torch.cuda.synchronize()
    assert not errors, errors
    for a, b in zip(sequential, results):
        assert torch.equal(a['keypoints0'], b['keypoints0'])          # same graphs, same pruning
        assert (a['matches0'] == b['matches0']).float().mean() >= 0.999
        assert (a['matches1'] == b['matches1']).float().mean() >= 0.999
        # fp32 atomics in the Sinkhorn column sums make the last bits order dependent
        assert torch.allclose(a['matching_scores0'], b['matching_scores0'], rtol=1e-4, atol=1e-6)


def test_round_trip_properties_full_size():
    """BASELINE config 2 (2048 kp, 100 Sinkhorn iterations): size-independent properties.
    * marginals: exp(Z) rows/cols sum to the prescribed masses (Sinkhorn fixed point, last update is v)
    * matches are mutual and consistent: matches1[matches0[i]] == i
    * permutation equivariance: shuffling image-1 keypoints permutes matches0 accordingly."""
    data = make_pair(2048, seed=77)
    sd = make_state_dict(0, damped=True)
    cfg = {'sinkhorn_iterations': 100, 'match_threshold': 0.005}
    model = _model(sd, cfg)
    r, cnt = _run_pair(model, data)
    n0, n1 = int(cnt[0]), int(cnt[1])
    coup = r['couplings'][:n0 + 1, :n1 + 1].double()
    u, v = r['u'][:n0 + 1].double(), r['v'][:n1 + 1].double()
    logp = coup + u[:, None] + v[None, :]
    col = torch.logsumexp(logp, 0)
    norm = -np.log(n0 + n1)
    log_nu = torch.full((n1 + 1,), norm, dtype=torch.float64, device=col.device)
    log_nu[-1] = np.log(n0) + norm
    assert (col - log_nu).abs().max() < 1e-4                        # v was updated last: columns are exact
    row = torch.logsumexp(logp, 1)
    log_mu = torch.full((n0 + 1,), norm, dtype=torch.float64, device=col.device)
    log_mu[-1] = np.log(n1) + norm
    assert (row - log_mu).abs().max() < 1.0                         # rows: converging, not exact
    m0, m1 = r['matches0'][:n0], r['matches1'][:n1]
    idx = torch.nonzero(m0 >= 0)[:, 0]
    assert idx.numel() > 50
    assert torch.equal(m1[m0[idx]], idx)
    perm = torch.randperm(2048, generator=torch.Generator().manual_seed(5))
    data2 = dict(data)
    data2['keypoints1'] = data['keypoints1'][:, perm]
    data2['descriptors1'] = data['descriptors1'][:, :, perm]
    data2['scores1'] = data['scores1'][:, perm]
    r2, cnt2 = _run_pair(model, data2)
    assert int(cnt2[0]) == n0 and int(cnt2[1]) == n1
    kept1 = r['kept_idx1'][:n1].cpu()
    kept1b = r2['kept_idx1'][:n1].cpu()
    # original ids matched by each image-0 keypoint must coincide
    inv = torch.empty(2048, dtype=torch.long)
    inv[torch.arange(2048)] = perm
    a = torch.where(m0.cpu() >= 0, kept1[m0.cpu().clamp(min=0)].long(), torch.full_like(m0.cpu(), -1))
    mb = r2['matches0'][:n0].cpu()
    b = torch.where(mb >= 0, perm[kept1b[mb.clamp(min=0)].long()], torch.full_like(mb, -1))
    assert (a == b).float().mean() >= 0.995
