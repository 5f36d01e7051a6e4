"""Host-side mirror of the reference's `Matching` front-end (models/matching.py:8-30)."""
import numpy as np
import torch

from . import _lib
from .frontend import detect_enqueue, device_pyramids, gaussian_pyramid_device, host_stages, sift_forward
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

    def _device_stages(self, images, dev):
        """Pyramid and detection of every image enqueued on the device, then one wait: per set, (keypoints, pyramid)."""
        if torch.device(dev).type != 'cuda':
            raise _lib.GimsError("Matching: 'detector': 'device' needs a CUDA device (got %s)" % dev)
        pending = []
        for imgs in images:
            row = []
            for img in imgs:
                pyr = gaussian_pyramid_device(img, dev)
                row.append((detect_enqueue(img, dev, self.max_keypoints, pyramid=pyr), pyr))
            pending.append(row)
        return [[(p.result(), pyr) for p, pyr in row] for row in pending]

    def forward(self, data):
        pred = {}
        need = [s for s in ('0', '1') if 'keypoints' + s not in data]
        dev = data.get('device', self.gmodel.bin_score.device)
        # the pyramids go onto the caller's stream first (uint8 grey / colour images, CUDA device); the OpenCV stages of
        # both images then run side by side (the reference does image 0, then image 1)
        images = [[np.asarray(img) for img in data['image' + s]] for s in need]
        if self.detector == 'device':
            staged = dict(zip(need, self._device_stages(images, dev)))
        else:
            pyramids = [device_pyramids(imgs, dev) for imgs in images]
            staged = dict(zip(need, host_stages(images, self.max_keypoints, pyramids))) if need else {}
        for s in need:
            out = sift_forward({'image': data['image' + s], 'max_keypoints': self.max_keypoints,
                                'carhynet': data['carhynet']}, device=dev, staged=staged[s])
            pred = {**pred, **{k + s: v for k, v in out.items()}}
        data = {**data, **pred}
        for k in data:
            if isinstance(data[k], (list, tuple)):
                data[k] = torch.stack(data[k])
        pred = {**pred, **self.gmodel(data)}
        return pred
