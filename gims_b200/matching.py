"""Host-side mirror of the reference's `Matching` front-end (models/matching.py:8-30)."""
import numpy as np
import torch

from .frontend import device_pyramids, host_stages, sift_forward
from .gmatcher import GMatcher


class Matching(torch.nn.Module):
    """Image Matching Frontend — same constructor and dict-in/dict-out call as the reference.

    With `keypoints{0,1}` in `data` the matcher runs on them directly (matching.py:17,21); without, the images go
    through `sift_forward` first (matching.py:18-24 -> utils/common.py:837-893; here gims_b200/frontend.py: OpenCV SIFT
    on the host while the Gaussian pyramid is built on the device, patches and the caller's CAR-HyNet on the device,
    descriptors never leave it).
    """

    def __init__(self, config={}):
        super().__init__()
        self.gmodel = GMatcher(config)
        self.max_keypoints = config.get('max_keypoints', -1)

    def forward(self, data):
        pred = {}
        need = [s for s in ('0', '1') if 'keypoints' + s not in data]
        dev = data.get('device', self.gmodel.bin_score.device)
        # the pyramids go onto the caller's stream first (uint8 grey / colour images, CUDA device); the OpenCV stages of
        # both images then run side by side (the reference does image 0, then image 1)
        images = [[np.asarray(img) for img in data['image' + s]] for s in need]
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
