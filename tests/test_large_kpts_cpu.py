"""CPU: the 65536-keypoint limit on the host side — workspace queries at full size hold their buffers without wrapping
around, and the argument checks reject 65537 keypoints before any CUDA call."""
import ctypes as C

import pytest

N = 65536


@pytest.fixture(scope='module')
def lib():
    from gims_b200 import build, _lib
    build.build()
    return _lib.lib()


def test_limit_matches_header():
    import os
    from gims_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'gims_b200.h')).read()
    assert '#define GIMS_MAX_KPTS    65536' in hdr
    assert _lib.MAX_KPTS == N
    assert '#define GIMS_STATUS_SINKHORN_WIDE   0x400u' in hdr and _lib.STATUS_SINKHORN_WIDE == 0x400


def test_workspace_queries_at_65536(lib):
    edge_cap = 16 * N
    agc = lib.gims_agc_workspace_bytes(N, edge_cap)
    assert agc >= N * N * 4 + 2 * N * 256 * 4 + edge_cap * 4       # cosine matrix S (16 GiB) + descriptors + edges
    assert agc < N * N * 4 + (1 << 30)                                 # and nothing near a second copy of S
    assert lib.gims_agc_workspace_bytes(N // 2, edge_cap) < agc // 3
    # the wide Sinkhorn path keeps (max, sum) partials of 256 row blocks per column, and no scaled-matrix scratch:
    # the couplings-sized buffer E ((N + 1) x ld floats, 17.2 GB) is not reserved
    sink = lib.gims_sinkhorn_workspace_bytes(N, N)
    ld = lib.gims_couplings_ld(N)
    assert sink >= 256 * (N + 1) * 8
    assert sink < (N + 1) * ld * 4 // 16
    # problems that may stream still reserve it
    assert lib.gims_sinkhorn_workspace_bytes(8192, 8192) > 8193 * lib.gims_couplings_ld(8192) * 4
    pair = lib.gims_pair_workspace_bytes(None, N, N, edge_cap)
    coup = (N + 1) * ld * 4
    assert coup > 2 ** 34
    assert pair >= 2 * agc + coup + sink                               # two graph chains + the couplings + Sinkhorn
    n0 = (C.c_int * 1)(N)
    assert lib.gims_batch_workspace_bytes(1, n0, n0, edge_cap) == pair


def _agc_call(lib, n):
    z = C.c_void_p(0)
    return lib.gims_agc_build(z, z, 1, z, n, 25.0, 0, 8, z, 0, z, z, z, z, 1024, z, z, z, z, z, z, z, z)


def test_agc_rejects_65537_before_any_cuda_call(lib):
    from gims_b200 import _lib
    assert _agc_call(lib, N + 1) == -1                                  # GIMS_ERR_ARG
    assert b'n=65537' in lib.gims_last_error()
    assert _agc_call(lib, N) == -1                                      # 65536 passes the size check ...
    assert b'null pointer' in lib.gims_last_error()                    # ... and stops at the missing buffers
    assert _lib.MAX_KPTS + 1 == N + 1


def test_forward_pair_rejects_65537(lib):
    from gims_b200 import _lib
    pin, po = _lib.PairInputs(), _lib.PairOutputs()
    pin.n[0], pin.n[1] = N + 1, 100
    pin.edge_cap = 1024
    dummy = C.create_string_buffer(64)
    rc = lib.gims_forward_pair(C.cast(dummy, C.c_void_p), C.byref(pin), C.byref(po), C.cast(dummy, C.c_void_p), 64,
                               C.c_void_p(0))
    assert rc == -1
    assert b'(65537, 100)' in lib.gims_last_error()
