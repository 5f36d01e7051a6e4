"""Row f-2 on the GPU: gims_extract_patches against the host path (cv2.warpAffine per keypoint + INTER_AREA resize, as
utils/library.py:84-110 / utils/common.py:882-884 do it) — every patch bit-identical — and the whole front end."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip('cv2')


@pytest.mark.parametrize('h,w,channels,nkp,seed', [(300, 400, 3, 600, 1), (600, 800, 3, 2048, 2), (240, 320, 1, 300, 3)])
def test_device_patches_equal_host_patches(h, w, channels, nkp, seed):
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image
    img = make_textured_image(h, w, seed=seed)
    if channels == 1:
        img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    kps = fe.detect(img, nkp)
    levels = fe.gaussian_pyramid(img)
    want = fe.extract_patches(kps, levels)
    got = fe.extract_patches_device(kps, levels, 'cuda:0')
    assert got.is_cuda and tuple(got.shape) == want.shape
    same = torch.equal(got.cpu(), torch.from_numpy(want.astype(np.float32)))
    if not same:
        d = (got.cpu().numpy() - want).reshape(len(kps), -1)
        print('patches that differ: %d of %d, max |d| %.3g' % (int((np.abs(d).max(1) > 0).sum()), len(kps), np.abs(d).max()))
    assert same
    # keypoints near the border produce patches that hang over the image: the constant border must be there too
    assert float(got.min()) == 0.0


def test_sift_forward_device_patches_equal_host_patches(monkeypatch):
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image

    class Net(torch.nn.Module):                         # any descriptor network: the two paths must feed it the same patches
        def __init__(self):
            super().__init__()
            self.c = torch.nn.Conv2d(3, 8, 5, stride=3)

        def forward(self, x):
            return torch.nn.functional.normalize(self.c(x).flatten(1)[:, :128], dim=1)

    torch.manual_seed(0)
    car = type('Car', (), {})()
    car.model = Net().cuda().eval()
    car.batch_size = 256
    img = make_textured_image(300, 400, seed=7)
    data = {'image': img[None], 'max_keypoints': 500, 'carhynet': car}
    got = fe.sift_forward(dict(data), torch.device('cuda:0'))
    monkeypatch.setenv('GIMS_HOST_PATCHES', '1')
    want = fe.sift_forward(dict(data), torch.device('cuda:0'))
    assert torch.equal(got['keypoints'][0], want['keypoints'][0])
    assert got['descriptors'][0].shape == (256, 500)
    assert torch.allclose(got['descriptors'][0], want['descriptors'][0], atol=1e-6)


def test_keypoint_outside_the_pyramid_raises():
    from gims_b200 import _lib
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image
    img = make_textured_image(240, 320, seed=3)
    kps = fe.detect(img, 50)
    host = fe.gaussian_pyramid(img)
    sources = {'host levels': host, 'device pyramid': fe.gaussian_pyramid_device(img, 'cuda:0')}
    past = len(host) // (fe.LAYERS + 3) - 1                   # the octave after the coarsest one: level len(host)
    for octave in (0xFE, past):                               # 0xFE unpacks to octave -2: level -6
        bad = kps + [cv2.KeyPoint(100, 100, 8, 0, 1, octave)]
        for name, levels in sources.items():
            with pytest.raises(_lib.GimsError, match='level'):
                fe.extract_patches_device(bad, levels, 'cuda:0')
    for name, levels in sources.items():                     # the good keypoints still go through
        assert fe.extract_patches_device(kps, levels, 'cuda:0').shape[0] == len(kps), name
