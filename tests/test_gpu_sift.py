"""SIFT detection on the GPU (gims_sift_detect, csrc/sift.cu): every record bit-identical to the numpy restatement
(oracle/cv_sift_oracle.py), within tolerance of cv2, deterministic across calls and threads, the overflow retry, the
patches cut for device keypoints, and the image-input Matching call with 'detector': 'device'."""
import threading
import types

import numpy as np
import pytest
import torch

from test_sift_cpu import BAR, IMAGES, agreement, records, sift_image, top

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip('cv2')
DEV = 'cuda:0'


def _device_records(dk):
    return {'pt': dk.pt.cpu().numpy(), 'size': dk.size.cpu().numpy(), 'angle': dk.angle.cpu().numpy(),
            'response': dk.response.cpu().numpy(), 'octave': dk.octave.cpu().numpy()}


def _assert_same_records(got, want):
    assert len(got['pt']) == len(want['pt'])
    for k in ('pt', 'size', 'angle', 'response', 'octave'):
        g, w = got[k], want[k]
        assert g.dtype == w.dtype and np.array_equal(g, w), (k, int(np.sum(g != w)))


@pytest.mark.parametrize('h,w,channels,seed', IMAGES)
def test_device_equals_oracle_and_agrees_with_cv2(h, w, channels, seed):
    from gims_b200 import frontend as fe
    from oracle import cv_sift_oracle as so
    img = sift_image(h, w, channels, seed)
    got = _device_records(fe.detect_device(img, DEV))
    _assert_same_records(got, so.detect(img))
    want = records(fe.detect(img))
    assert min(agreement(got, want), agreement(want, got)) >= BAR
    assert min(agreement(top(got, 2048), top(want, 2048)), agreement(top(want, 2048), top(got, 2048))) >= BAR


@pytest.mark.parametrize('max_kp', [2048, 300])
def test_device_max_keypoints_equals_oracle(max_kp):
    from gims_b200 import frontend as fe
    from oracle import cv_sift_oracle as so
    img = sift_image(600, 800, 3, 100)
    got = _device_records(fe.detect_device(img, DEV, max_kp))
    _assert_same_records(got, so.detect(img, max_kp))


def test_one_channel_image_equals_grey():
    from gims_b200 import frontend as fe
    img = sift_image(240, 320, 1, 3)
    _assert_same_records(_device_records(fe.detect_device(img[:, :, None], DEV)),
                         _device_records(fe.detect_device(img, DEV)))


def test_repeat_and_threads_are_bit_identical():
    from gims_b200 import frontend as fe
    imgs = [sift_image(600, 800, 3, 100 + k) for k in range(4)]
    single = [_device_records(fe.detect_device(im, DEV)) for im in imgs]
    _assert_same_records(_device_records(fe.detect_device(imgs[0], DEV)), single[0])
    out = [None] * len(imgs)
    errors = []

    def worker(t):
        try:
            with torch.cuda.stream(torch.cuda.Stream(DEV)):
                for k in range(t, len(imgs), 2):
                    out[k] = _device_records(fe.detect_device(imgs[k], DEV))
        except Exception as exc:                                      # noqa: BLE001
            errors.append(exc)
    threads = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for a, b in zip(out, single):
        _assert_same_records(a, b)


def test_overflow_retries_with_larger_capacity():
    from gims_b200 import frontend as fe
    img = sift_image(301, 417, 3, 5)
    small = fe.detect_enqueue(img, DEV, kp_cap=8)
    got = _device_records(small.result())
    _assert_same_records(got, _device_records(fe.detect_device(img, DEV)))
    assert len(got['pt']) > 8


def test_patches_for_device_keypoints_equal_host_route():
    from gims_b200 import frontend as fe
    img = sift_image(600, 800, 3, 2)
    pyr = fe.gaussian_pyramid_device(img, DEV)
    dk = fe.detect_device(img, DEV, 2048, pyramid=pyr)
    kps = dk.keypoints()
    assert len(kps) == len(dk) == 2048
    got = fe.extract_patches_device(dk, pyr, DEV)
    want = fe.extract_patches(kps, fe.gaussian_pyramid(img))
    assert torch.equal(got.cpu(), torch.from_numpy(want.astype(np.float32)))
    level, inv = fe.patch_maps(kps)
    level2, inv2 = fe.patch_maps_from_arrays(*dk.host())
    assert np.array_equal(level, level2) and np.array_equal(inv, inv2)


class _Net(torch.nn.Module):
    """The stand-in descriptor network of test_gpu_pyramid.py."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Sequential(torch.nn.Conv2d(3, 32, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(32, 64, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(64, 128, 8))

    def forward(self, x):
        return torch.nn.functional.normalize(self.body(x).flatten(1), dim=1)


def test_matching_device_detector_equals_keypoint_input_call(monkeypatch):
    from gims_b200 import Matching
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_state_dict, make_textured_image, warp_image
    dev = torch.device(DEV)
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)
    monkeypatch.setattr(torch.backends.cudnn, 'benchmark', False)
    torch.manual_seed(0)
    car = types.SimpleNamespace(model=_Net().to(dev).eval(), batch_size=512)
    cfg = {'sinkhorn_iterations': 20, 'match_threshold': 0.01, 'max_keypoints': 700}
    matching = Matching({**cfg, 'detector': 'device'})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to(dev)
    img0 = make_textured_image(320, 400, seed=31)
    img1, _ = warp_image(img0, seed=61)
    knobs = {'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7}
    with torch.no_grad():
        got = matching({**knobs, 'image0': img0[None], 'image1': img1[None], 'carhynet': car})
    data = dict(knobs)
    for s, img in (('0', img0), ('1', img1)):
        pyr = fe.gaussian_pyramid_device(img, dev)
        dk = fe.detect_device(img, dev, 700, pyramid=pyr)
        with torch.no_grad():
            d = fe.describe(fe.extract_patches_device(dk, pyr, dev), car, dev)
        data['keypoints' + s] = dk.pt[None]
        data['scores' + s] = dk.response[None]
        data['descriptors' + s] = torch.cat([d, d], dim=1).t().contiguous()[None]
        data['image' + s] = img[None]
    with torch.no_grad():
        want = matching(data)
    # the matcher returns its own keypoints / descriptors / matches; the scores are the detector's, passed through
    for s in '01':
        assert torch.equal(got['scores' + s][0], data['scores' + s][0])
    exact = {'keypoints0', 'keypoints1', 'matches0', 'matches1'}
    shared = [k for k in want if k in got]
    assert exact <= set(shared)
    for k in shared:
        if k in exact or not got[k].is_floating_point():
            assert torch.equal(got[k], want[k]), k
        else:
            assert torch.allclose(got[k], want[k], rtol=0, atol=1e-6), k
    assert int((got['matches0'] >= 0).sum()) > 0


def test_bad_inputs_and_options_raise():
    from gims_b200 import Matching, _lib
    from gims_b200 import frontend as fe
    with pytest.raises(ValueError):
        Matching({'detector': 'sift-gpu'})
    img = sift_image(120, 160, 3, 1)
    with pytest.raises(_lib.GimsError):
        fe.detect_device(img.astype(np.float32), DEV)
    with pytest.raises(_lib.GimsError):
        fe.detect_device(np.zeros((120, 160, 4), np.uint8), DEV)
    with pytest.raises(_lib.GimsError):
        fe.detect_device(img, 'cpu')
    m = Matching({'detector': 'device'}).eval().to(DEV)
    with pytest.raises(_lib.GimsError):
        m({'image0': img[None].astype(np.float32), 'image1': img[None], 'carhynet': None, 'device': torch.device(DEV)})
