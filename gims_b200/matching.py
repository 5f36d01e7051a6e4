"""Host-side mirror of the reference's `Matching` front-end (models/matching.py:8-30)."""
import torch

from .frontend import sift_forward, stage_images
from .gmatcher import GMatcher


class Matching(torch.nn.Module):
    """Image Matching Frontend — same constructor and dict-in/dict-out call as the reference.

    With `keypoints{0,1}` in `data` the matcher runs on them directly (matching.py:17,21); without, the images go
    through `sift_forward` first (matching.py:18-24 -> utils/common.py:837-893; here gims_b200/frontend.py: OpenCV SIFT
    on the host while the Gaussian pyramid is built on the device, patches and the caller's CAR-HyNet on the device,
    descriptors never leave it).

    `config['detector']` picks the keypoint detector of that route: 'opencv' (the default, cv2 SIFT on the host) or
    'device' (the same SIFT on the GPU, csrc/sift.cu: within a tolerance of cv2, not bit for bit; the keypoints and
    scores never pass through the host).
    """

    DETECTORS = ('opencv', 'device')

    def __init__(self, config={}):
        super().__init__()
        self.detector = config.get('detector', 'opencv')
        if self.detector not in self.DETECTORS:
            raise ValueError("Matching: config['detector'] must be one of %s (got %r)" % (self.DETECTORS, self.detector))
        self.gmodel = GMatcher(config)
        self.max_keypoints = config.get('max_keypoints', -1)

    def forward(self, data):
        pred = {}
        need = [s for s in ('0', '1') if 'keypoints' + s not in data]
        dev = data.get('device', self.gmodel.bin_score.device)
        # both images are staged at once: the device work of both is enqueued first, then the host work of the two runs
        # side by side (the reference does image 0, then image 1)
        staged = stage_images([data['image' + s] for s in need], dev, self.max_keypoints, self.detector) if need else []
        for s, st in zip(need, staged):
            out = sift_forward({'image': data['image' + s], 'max_keypoints': self.max_keypoints,
                                'carhynet': data['carhynet']}, device=dev, staged=st)
            pred = {**pred, **{k + s: v for k, v in out.items()}}
        data = {**data, **pred}
        for k in data:
            if isinstance(data[k], (list, tuple)):
                data[k] = torch.stack(data[k])
        pred = {**pred, **self.gmodel(data)}
        return pred
