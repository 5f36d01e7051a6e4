"""Synthetic keypoints / descriptors / weights for parity tests and the benchmark (SURVEY.md §8d).

There is no network and the reference ships no weights or images, so every test and bench input
is generated here from fixed seeds.  Nothing in this file touches the GPU or the oracle.
"""
import math

import torch

from .config import DEFAULT_CONFIG, state_dict_schema


def _random_homography(gen, width, height):
    """Mild random homography about the image centre (rotation, scale, shear-free perspective, shift)."""
    u = torch.rand(6, generator=gen, dtype=torch.float64)
    ang = math.radians(float(u[0]) * 30.0 - 15.0)
    sc = 0.9 + 0.2 * float(u[1])
    tx = (float(u[2]) - 0.5) * 0.1 * width
    ty = (float(u[3]) - 0.5) * 0.1 * height
    px = (float(u[4]) - 0.5) * 2e-4
    py = (float(u[5]) - 0.5) * 2e-4
    cx, cy = width / 2.0, height / 2.0
    c, s = math.cos(ang) * sc, math.sin(ang) * sc
    to_c = torch.tensor([[1, 0, -cx], [0, 1, -cy], [0, 0, 1]], dtype=torch.float64)
    rot = torch.tensor([[c, -s, 0], [s, c, 0], [px, py, 1]], dtype=torch.float64)
    back = torch.tensor([[1, 0, cx + tx], [0, 1, cy + ty], [0, 0, 1]], dtype=torch.float64)
    return back @ rot @ to_c


def make_pair(n0, n1=None, seed=0, width=800, height=600, desc_dim=256, image_style='tensor'):
    """One synthetic image pair in the layout `Matching.forward` receives (matching.py:15-29).

    keypoints{0,1} (1,N,2) fp32 pixel xy, descriptors{0,1} (1,D,N) fp32 channel-major with the
    128-d unit vector duplicated to 256-d as utils/common.py:891 does, scores{0,1} (1,N) fp32.
    70 % of image-1 keypoints are homography images of image-0 keypoints (+0.5 px noise) with
    perturbed descriptors; the rest are fresh.  `image_style='tensor'` gives a (1,1,H,W) image
    tensor, `'eval'` the (1,H,W,3) numpy layout of eval_homography.py:169-178 (shape quirk of
    gmatcher.py:28).
    """
    n1 = n0 if n1 is None else n1
    gen = torch.Generator().manual_seed(int(seed))
    half = desc_dim // 2
    size = torch.tensor([width, height], dtype=torch.float32)
    k0 = torch.rand(n0, 2, generator=gen) * size
    d0 = torch.nn.functional.normalize(torch.randn(n0, half, generator=gen), dim=1)
    n_corr = min(int(0.7 * n1), n0)
    src = torch.randperm(n0, generator=gen)[:n_corr]
    hmat = _random_homography(gen, width, height)
    p = torch.cat([k0[src].double(), torch.ones(n_corr, 1, dtype=torch.float64)], 1) @ hmat.T
    kc = (p[:, :2] / p[:, 2:3]).float() + 0.5 * torch.randn(n_corr, 2, generator=gen)
    dc = torch.nn.functional.normalize(d0[src] + 0.05 * torch.randn(n_corr, half, generator=gen), dim=1)
    kf = torch.rand(n1 - n_corr, 2, generator=gen) * size
    df = torch.nn.functional.normalize(torch.randn(n1 - n_corr, half, generator=gen), dim=1)
    k1 = torch.cat([kc, kf], 0)
    d1 = torch.cat([dc, df], 0)
    perm = torch.randperm(n1, generator=gen)
    k1, d1 = k1[perm], d1[perm]
    s0 = torch.rand(n0, generator=gen)
    s1 = torch.rand(n1, generator=gen)
    if image_style == 'tensor':
        img0 = torch.zeros(1, 1, height, width)
        img1 = torch.zeros(1, 1, height, width)
    elif image_style == 'eval':
        import numpy as np
        img0 = np.zeros((1, height, width, 3), dtype=np.float32)
        img1 = np.zeros((1, height, width, 3), dtype=np.float32)
    else:
        raise ValueError(image_style)
    return {
        'keypoints0': k0[None].contiguous(), 'keypoints1': k1[None].contiguous(),
        'descriptors0': torch.cat([d0, d0], 1).t()[None].contiguous(),
        'descriptors1': torch.cat([d1, d1], 1).t()[None].contiguous(),
        'scores0': s0[None].contiguous(), 'scores1': s1[None].contiguous(),
        'image0': img0, 'image1': img1,
    }


def make_state_dict(seed=0, peaked=False, damped=False, config=None):
    """Random-init weights with the reference's key set (config.state_dict_schema).

    Conv/Linear weights ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)) like torch's default init; the last
    bias of kenc and of every layer MLP is zero as in gmatcher.py:92,121; BatchNorm running stats
    are randomised (mean ~ N(0,0.1), var ~ U(0.5,1.5), affine weight ~ U(0.8,1.2), bias ~ N(0,0.05))
    so BN folding is exercised.  `peaked=True` multiplies `final_proj.weight` by 16 (SURVEY.md §7),
    which makes the assignment non-degenerate under random weights.  `damped=True` scales every layer's
    last MLP conv by 0.05 and `final_proj.weight` by 64, so the input descriptors' similarity survives the
    random attention stack and a useful share of keypoints gets confident mutual matches.
    """
    cfg = {**DEFAULT_CONFIG, **(config or {})}
    gen = torch.Generator().manual_seed(int(seed) + 7919)
    sd = {}
    for key, shape in state_dict_schema(cfg).items():
        leaf = key.rsplit('.', 1)[-1]
        if key == 'bin_score':
            t = torch.tensor(1.0)
        elif leaf == 'num_batches_tracked':
            t = torch.tensor(100, dtype=torch.long)
        elif leaf == 'running_mean':
            t = 0.1 * torch.randn(shape, generator=gen)
        elif leaf == 'running_var':
            t = 0.5 + torch.rand(shape, generator=gen)
        elif len(shape) >= 2:
            fan_in = shape[1]
            bound = 1.0 / math.sqrt(fan_in)
            t = (torch.rand(shape, generator=gen) * 2 - 1) * bound
        else:  # 1-d: conv bias, BN affine, SAGE bias
            parent = key.rsplit('.', 1)[0]
            is_bn = (parent + '.running_mean') in state_dict_schema(cfg)
            if is_bn and leaf == 'weight':
                t = 0.8 + 0.4 * torch.rand(shape, generator=gen)
            elif is_bn:
                t = 0.05 * torch.randn(shape, generator=gen)
            else:
                t = (torch.rand(shape, generator=gen) * 2 - 1) * 0.05
        sd[key] = t
    nk = 3 * (len(cfg['keypoint_encoder']))
    sd['kenc.encoder.%d.bias' % nk].zero_()
    for l in range(len(cfg['transformer_layers'])):
        sd['gnn.layers.%d.mlp.3.bias' % l].zero_()
    if peaked:
        sd['final_proj.weight'] = sd['final_proj.weight'] * 16.0
    if damped:
        for l in range(len(cfg['transformer_layers'])):
            sd['gnn.layers.%d.mlp.3.weight' % l] = sd['gnn.layers.%d.mlp.3.weight' % l] * 0.05
        sd['final_proj.weight'] = sd['final_proj.weight'] * 64.0
    return sd


def make_textured_image(height=600, width=800, seed=0, n_shapes=260, noise=0.6):
    """Synthetic colour image (H, W, 3) uint8 with enough structure for a few thousand SIFT keypoints — stands in for
    the COCO images of eval_homography.py (BASELINE configs[2]; there is no dataset offline)."""
    import cv2
    import numpy as np
    rng = np.random.default_rng(seed)
    img = np.full((height, width, 3), 40.0, dtype=np.float32)
    for _ in range(n_shapes):
        c = (int(rng.integers(0, width)), int(rng.integers(0, height)))
        col = tuple(float(x) for x in rng.integers(30, 255, 3))
        kind = rng.random()
        if kind < 0.4:
            cv2.circle(img, c, int(rng.integers(3, 28)), col, -1)
        elif kind < 0.8:
            cv2.rectangle(img, c, (c[0] + int(rng.integers(4, 60)), c[1] + int(rng.integers(4, 60))), col, -1)
        else:
            cv2.line(img, c, (int(rng.integers(0, width)), int(rng.integers(0, height))), col, int(rng.integers(1, 4)))
    img = cv2.GaussianBlur(img, (0, 0), 0.8) + rng.normal(0, noise, img.shape).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def warp_image(img, seed=0):
    """The second image of a homography pair (eval_homography.py warps image0 with a random homography)."""
    import cv2
    import numpy as np
    h, w = img.shape[:2]
    hmat = _random_homography(torch.Generator().manual_seed(int(seed)), w, h).numpy()
    return cv2.warpPerspective(img, hmat, (w, h)), hmat.astype(np.float32)


def make_correspondences(m, inlier_ratio, noise=1.0, seed=0, width=800, height=600):
    """Matched points of one synthetic pair for the homography estimator: (src, dst) float32 (m, 2) and the true H (3, 3)
    float64.  round(m * inlier_ratio) matches follow H with Gaussian noise of `noise` px on the destination; the others
    are uniform over the image on both sides.  The matches are in random order."""
    import numpy as np
    hmat = _random_homography(torch.Generator().manual_seed(int(seed)), width, height).numpy()
    rng = np.random.default_rng(int(seed) + 7919)
    n_in = int(round(m * inlier_ratio))
    wh = np.array([width, height], dtype=np.float64)
    src = rng.random((m, 2)) * wh
    proj = np.concatenate([src, np.ones((m, 1))], axis=1) @ hmat.T
    dst = proj[:, :2] / proj[:, 2:] + rng.normal(0.0, noise, (m, 2))
    dst[n_in:] = rng.random((m - n_in, 2)) * wh
    perm = rng.permutation(m)
    return src[perm].astype(np.float32), dst[perm].astype(np.float32), hmat
