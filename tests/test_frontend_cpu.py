"""CPU: gims_b200.frontend.sift_forward against the UNMODIFIED reference `sift_forward` (utils/common.py:837-893) with
the reference's own CAR_HyNet (random init) on a synthetic textured image.  The reference is not part of the repository:
these tests run where it is installed (oracle/_ref, copied by __graft_entry__.build() from GIMS_REFERENCE_ROOT, or
GIMS_REFERENCE_ROOT itself)."""
import contextlib
import io
import sys

import numpy as np
import pytest
import torch

from oracle.ref_shims import REFERENCE_ROOT, _install_stubs, reference_available

cv2 = pytest.importorskip('cv2')
pytestmark = pytest.mark.skipif(not reference_available(), reason='needs the original GIMS code (oracle/_ref or GIMS_REFERENCE_ROOT)')


def _textured(h, w, seed, color=True):
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w, 3), dtype=np.float32)
    for _ in range(60):
        c = (int(rng.integers(0, w)), int(rng.integers(0, h)))
        col = tuple(float(x) for x in rng.integers(40, 255, 3))
        if rng.random() < 0.5:
            cv2.circle(img, c, int(rng.integers(4, 30)), col, -1)
        else:
            cv2.rectangle(img, c, (c[0] + int(rng.integers(5, 50)), c[1] + int(rng.integers(5, 50))), col, -1)
    img = cv2.GaussianBlur(img, (0, 0), 1.0) + rng.normal(0, 3, img.shape).astype(np.float32)
    img = np.clip(img, 0, 255).astype(np.uint8)
    return img if color else cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)


def _reference_modules():
    _install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    return importlib.import_module('utils.common'), importlib.import_module('carhynet.models')


def test_sift_forward_equals_reference():
    common, hm = _reference_modules()
    from gims_b200.frontend import sift_forward
    torch.manual_seed(3)
    car = object.__new__(hm.HyNetnetFeature2D)           # the wrapper's __init__ hard-loads ./weights/car_hynet.pth
    car.G_dim, car.do_cuda, car.device, car.batch_size = 128, False, torch.device('cpu'), 512
    car.model = hm.CAR_HyNet().eval()
    img = _textured(240, 320, 5)
    data = {'image': img[None], 'max_keypoints': 300, 'carhynet': car}
    with contextlib.redirect_stdout(io.StringIO()):
        ref = common.sift_forward(dict(data), device=torch.device('cpu'))
    got = sift_forward(dict(data), device=torch.device('cpu'))
    assert len(got['keypoints']) == 1 and got['keypoints'][0].shape[0] == 300
    assert torch.equal(got['keypoints'][0], ref['keypoints'][0])
    assert torch.equal(got['scores'][0], ref['scores'][0])
    assert got['descriptors'][0].shape == ref['descriptors'][0].shape == (256, 300)
    assert torch.allclose(got['descriptors'][0], ref['descriptors'][0], atol=1e-6)
    assert torch.equal(got['descriptors'][0][:128], got['descriptors'][0][128:])       # the 128 -> 256 duplication


def test_patches_equal_reference():
    common, _ = _reference_modules()
    import importlib
    lib = importlib.import_module('utils.library')
    from gims_b200 import frontend
    img = _textured(200, 260, 9)
    kps = frontend.detect(img, 150)
    want = np.array([cv2.resize(p, (32, 32), interpolation=cv2.INTER_AREA)
                     for p in lib.ComputePatches(kps, lib.buildGaussianPyramid(img, 6, graydesc=False), radius_size=64)]) / 255.0
    got = frontend.extract_patches(kps, frontend.gaussian_pyramid(img))
    assert got.shape == want.shape == (150, 32, 32, 3)
    assert np.array_equal(got, want.astype(np.float32)) or np.allclose(got, want, atol=1e-6)
