"""Front-end hand-off (SURVEY.md §8f row 1): keypoints + CAR-HyNet descriptors for `Matching.forward` when the caller
passes images instead of keypoints — the call every script of the reference makes (eval_homography.py:177,
eval_matches.py:152-156, tools/parameter_search.py:150-154).

Mirrors `sift_forward` (utils/common.py:837-893): OpenCV SIFT detection, OpenCV-SIFT Gaussian pyramid
(utils/library.py:234-293), one oriented 64x64 patch per keypoint taken from the pyramid level the keypoint was found on
(utils/library.py:84-110), resized to 32x32 (INTER_AREA) and scaled to [0, 1], CAR-HyNet descriptor of every patch, the
128-d descriptor duplicated to 256-d (utils/common.py:891).

What is different from the reference, and why:
  * detection stays on the host (OpenCV) by default; `Matching({'detector': 'device'})` detects on the GPU instead
    (`detect_device`, csrc/sift.cu: within a tolerance of cv2, not bit for bit, see DESIGN.md §9); the Gaussian pyramid of a uint8 grey or colour image is built on the device,
    byte for byte what OpenCV builds (`gaussian_pyramid_device`, csrc/pyramid.cu), while the host detects; the per-keypoint patch loop (§8f row 2: cv2.warpAffine
    + resize per keypoint, 200-500 ms per image) runs as ONE kernel on the device that reproduces OpenCV's fixed-point
    cubic warp bit for bit (`extract_patches_device`, csrc/patches.cu; GIMS_HOST_PATCHES=1 keeps the host loop);
  * the descriptor network runs on the device the matcher lives on and its output NEVER leaves it: the reference
    round-trips every batch through `.cpu().detach().numpy()` (carhynet/models.py:656-665) and uploads again at
    utils/common.py:890-892.  The 128 -> 256 duplication and the (N, D) -> (D, N) layout of `descriptors{0,1}` are
    views / one small device copy.
The caller's `carhynet` object is used as it is: anything with a `.model` (the torch module) is run directly; an object
that only offers the reference's `compute_sift(patches, kps, color)` is called through that method.
"""
import math
import os

import numpy as np
import torch

# the constants sift_forward hard-codes (utils/common.py:838-848)
SIFT_CONFIG = dict(nfeatures=None, nOctaveLayers=3, contrastThreshold=0.001, edgeThreshold=80, sigma=1.6)
PATCH_SUPPORT = 64      # ComputePatches(radius_size=64): side of the sampled window
PATCH_SIZE = 32         # CAR-HyNet input
FIRST_OCTAVE = -1       # OpenCV SIFT doubles the image first
LAYERS = 3              # nOctaveLayers


def _cv2():
    import cv2
    return cv2


def detect(image, max_keypoints=-1):
    """cv2 SIFT keypoints of one image (H, W[, 3]), strongest `max_keypoints` first if that limit is positive
    (utils/common.py:851-861, 710-718)."""
    cv2 = _cv2()
    sift = cv2.SIFT_create(nfeatures=SIFT_CONFIG['nfeatures'], nOctaveLayers=SIFT_CONFIG['nOctaveLayers'],
                           contrastThreshold=SIFT_CONFIG['contrastThreshold'], edgeThreshold=SIFT_CONFIG['edgeThreshold'],
                           sigma=SIFT_CONFIG['sigma'])
    kps = sift.detect(image, None)
    if 0 < max_keypoints < len(kps):
        order = np.argsort([k.response for k in kps])[::-1]
        kps = [kps[i] for i in order[:max_keypoints]]
    return kps


def gaussian_pyramid(image):
    """The scale space OpenCV's SIFT builds (utils/library.py:234-293): the image doubled (linear), then per octave
    LAYERS + 3 levels, level i blurred from level i-1 with the incremental sigma, each next octave seeded by the
    nearest-neighbour decimation of level LAYERS of the previous one.  Colour images keep their channels."""
    cv2 = _cv2()
    base = cv2.resize(image, (0, 0), fx=2, fy=2, interpolation=cv2.INTER_LINEAR_EXACT)
    rows, cols = base.shape[:2]
    n_octaves = int(np.round(np.log(np.float32(min(cols, rows))) / np.log(2.0) - 2) - FIRST_OCTAVE)
    per_octave = LAYERS + 3
    k = np.float32(2.0 ** (1.0 / LAYERS))
    sigma0 = SIFT_CONFIG['sigma']
    inc = [sigma0]
    for i in range(1, per_octave):
        prev = (k ** np.float32(i - 1)) * sigma0
        total = prev * k
        inc.append(math.sqrt(total * total - prev * prev))
    levels = []
    for o in range(n_octaves):
        for i in range(per_octave):
            if o == 0 and i == 0:
                img = base
            elif i == 0:
                img = cv2.resize(levels[(o - 1) * per_octave + LAYERS], (0, 0), fx=0.5, fy=0.5, interpolation=cv2.INTER_NEAREST)
            else:
                img = cv2.GaussianBlur(levels[o * per_octave + i - 1], (0, 0), sigmaX=inc[i], sigmaY=inc[i])
            levels.append(img)
    return levels


def _unpack_octave(kp):
    """cv2 packs octave / layer into KeyPoint.octave (utils/library.py:16-35)."""
    octave = kp.octave & 0xFF
    layer = (kp.octave >> 8) & 0xFF
    if octave >= 128:
        octave -= 256
    scale = 1.0 / (1 << octave) if octave >= 0 else float(1 << -octave)
    return octave, layer, scale


def extract_patches(kps, levels, support=PATCH_SUPPORT, out_size=PATCH_SIZE):
    """(N, out_size, out_size[, C]) float32 in [0, 1]: for each keypoint the window of half-width size*scale/2 * (support-1)/2
    around it on its own pyramid level, rotated by its orientation (bicubic, constant border), then area-resampled
    (utils/library.py:84-110, utils/common.py:882-884)."""
    cv2 = _cv2()
    r = (support - 1) / 2
    dim = int(2 * r + 1)
    out = []
    for kp in kps:
        octave, layer, scale = _unpack_octave(kp)
        step = kp.size * scale * 0.5
        centre = np.array(kp.pt) * scale
        angle = 360.0 - kp.angle
        if abs(angle - 360.0) < 1.19209e-07:
            angle = 0.0
        phi = np.deg2rad(angle)
        s, c = np.sin(phi), np.cos(phi)
        rot = np.float32([[c, -s], [s, c]]) / step
        shift = np.matmul(rot, centre)
        affine = np.hstack([rot, [[r - shift[0]], [r - shift[1]]]])
        level = levels[(octave - FIRST_OCTAVE) * (LAYERS + 3) + layer]
        patch = cv2.warpAffine(level, affine, (dim, dim), flags=cv2.INTER_CUBIC, borderMode=cv2.BORDER_CONSTANT)
        out.append(cv2.resize(patch.astype(np.float32), (out_size, out_size), interpolation=cv2.INTER_AREA))
    if not out:
        return np.zeros((0, out_size, out_size), dtype=np.float32)
    return np.array(out) / 255.0


def keypoint_arrays(kps):
    """(pt float64 [N, 2], size, angle float64 [N], octave int64 [N]) of a list of cv2.KeyPoint."""
    n = len(kps)
    return (np.array([k.pt for k in kps], dtype=np.float64).reshape(n, 2),
            np.array([k.size for k in kps], dtype=np.float64).reshape(n),
            np.array([k.angle for k in kps], dtype=np.float64).reshape(n),
            np.array([k.octave for k in kps], dtype=np.int64).reshape(n))


def patch_maps(kps):
    """`patch_maps_from_arrays` of a list of cv2.KeyPoint."""
    return patch_maps_from_arrays(*keypoint_arrays(kps))


def patch_maps_from_arrays(pt, size, angle, octave):
    """Per keypoint: the pyramid level index and the 2 x 3 matrix `extract_patches` hands to cv2.warpAffine
    (utils/library.py:84-110), vectorised over the keypoints with the reference's dtypes (float32 rotation / step, float64
    shift), then inverted the way cv::warpAffine inverts its argument (imgwarp.cpp).  `pt` (N, 2), `size`, `angle`,
    `octave` (N,) as cv2.KeyPoint holds them.  Returns (level int32 [N], inverse map float64 [N, 6])."""
    n = len(size)
    r = (PATCH_SUPPORT - 1) / 2
    octv = np.asarray(octave, dtype=np.int64).reshape(n)
    octave = octv & 0xFF
    layer = (octv >> 8) & 0xFF
    octave = np.where(octave >= 128, octave - 256, octave)
    scale = np.where(octave >= 0, 1.0 / (1 << np.maximum(octave, 0)), (1 << np.maximum(-octave, 0)).astype(np.float64))
    size = np.asarray(size, dtype=np.float64).reshape(n)
    pt = np.asarray(pt, dtype=np.float64).reshape(n, 2)
    ang = np.asarray(angle, dtype=np.float64).reshape(n)
    step = size * scale * 0.5
    centre = pt * scale[:, None]
    angle = 360.0 - ang
    angle = np.where(np.abs(angle - 360.0) < 1.19209e-07, 0.0, angle)
    phi = np.deg2rad(angle)
    s, c = np.sin(phi), np.cos(phi)
    step32 = step.astype(np.float32)
    r00 = (c.astype(np.float32) / step32).astype(np.float64)
    r01 = ((-s).astype(np.float32) / step32).astype(np.float64)
    r10 = (s.astype(np.float32) / step32).astype(np.float64)
    r11 = r00
    m2 = r - (r00 * centre[:, 0] + r01 * centre[:, 1])
    m5 = r - (r10 * centre[:, 0] + r11 * centre[:, 1])
    # cv::warpAffine without WARP_INVERSE_MAP
    det = r00 * r11 - r01 * r10
    with np.errstate(divide='ignore'):
        d = np.where(det != 0, 1.0 / det, 0.0)
    a11, a22 = r11 * d, r00 * d
    i0, i1, i3, i4 = a11, r01 * (-d), r10 * (-d), a22
    b1 = -i0 * m2 - i1 * m5
    b2 = -i3 * m2 - i4 * m5
    inv = np.stack([i0, i1, b1, i3, i4, b2], axis=1)
    level = ((octave - FIRST_OCTAVE) * (LAYERS + 3) + layer).astype(np.int32)
    return level, np.ascontiguousarray(inv, dtype=np.float64)


_STAGING = __import__('threading').local()


def _pinned_staging(nbytes):
    """Grow-only pinned host buffer of the calling thread (pinning 40 MB per call cost more than the copy itself)."""
    ev = getattr(_STAGING, 'event', None)
    if ev is not None:
        ev.synchronize()                          # the previous upload from this buffer has left the host
    buf = getattr(_STAGING, 'buf', None)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8).pin_memory()
        _STAGING.buf = buf
    return buf


class DevicePyramid:
    """The Gaussian pyramid of one image on the device (`gaussian_pyramid_device`): every level in one uint8 buffer and
    the level table `gims_extract_patches` reads.  `buffer` uint8, `offset` int64, `height` / `width` int32 are device
    tensors; `shapes` is the host copy of the level sizes; `image` is the uploaded image (uint8, on the device), which
    `detect_device` reuses."""

    def __init__(self, buffer, offset, height, width, shapes, offsets, channels, image=None):
        self.buffer, self.offset, self.height, self.width = buffer, offset, height, width
        self.shapes, self.offsets, self.channels, self.image = shapes, offsets, channels, image

    def __len__(self):
        return len(self.shapes)

    def level(self, i):
        """Level i as a (H, W[, C]) uint8 device tensor (a view of the buffer); the same shape as the host level."""
        h, w = self.shapes[i]
        o = int(self.offsets[i])
        v = self.buffer[o:o + h * w * self.channels]
        return v.view(h, w, self.channels) if self.channels == 3 else v.view(h, w)


_PYR_WS = {}                    # (device, stream, thread) -> grow-only uint8 workspace of gims_gaussian_pyramid
_PYR_WS_LOCK = __import__('threading').Lock()


def pyramid_on_device(image):
    """True if `gaussian_pyramid_device` can build this image's pyramid: uint8, grey or 3-channel colour."""
    a = np.asarray(image)
    return a.dtype == np.uint8 and (a.ndim == 2 or (a.ndim == 3 and a.shape[2] in (1, 3))) and a.size > 0


def gaussian_pyramid_device(image, device):
    """`gaussian_pyramid` on the GPU, byte for byte the same levels (csrc/pyramid.cu follows OpenCV's 8-bit fixed-point
    resize and blur).  Only the image travels: it is copied through the calling thread's pinned staging buffer and the
    pyramid is enqueued on the current stream of `device`; nothing waits for it.  Returns a `DevicePyramid`, which
    `extract_patches_device` takes in place of host levels.  The level buffer belongs to the returned object (the
    pyramids of several images may be alive at once); the row-pass workspace is cached per (device, stream, thread),
    grow-only, and its reuse is ordered by the stream."""
    import ctypes as C
    from . import _lib
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise _lib.GimsError('gaussian_pyramid_device needs a CUDA device')
    img = np.asarray(image)
    if not pyramid_on_device(img):
        raise _lib.GimsError('gaussian_pyramid_device: need a uint8 (H, W), (H, W, 1) or (H, W, 3) image (got %s %s)'
                             % (img.dtype, img.shape))
    h, w = img.shape[:2]
    cn = 3 if img.ndim == 3 and img.shape[2] == 3 else 1
    L = _lib.lib()
    n = C.c_int(0)
    _lib.check(L.gims_pyramid_layout(h, w, cn, C.byref(n), None, None, None), 'gims_pyramid_layout')
    offs = np.zeros(max(n.value, 1), dtype=np.int64)
    hs = np.zeros(max(n.value, 1), dtype=np.int32)
    ws = np.zeros(max(n.value, 1), dtype=np.int32)
    _lib.check(L.gims_pyramid_layout(h, w, cn, C.byref(n), offs.ctypes.data, hs.ctypes.data, ws.ctypes.data),
               'gims_pyramid_layout')
    nl = n.value
    offs, hs, ws = offs[:nl], hs[:nl], ws[:nl]
    total = int(offs[-1]) + int(hs[-1]) * int(ws[-1]) * cn if nl else 0
    shapes = [(int(a), int(b)) for a, b in zip(hs, ws)]
    # one upload: the level table (int64 offsets, int32 heights, int32 widths), then the image at a 256-byte boundary
    img_at = (16 * nl + 255) // 256 * 256
    st = torch.cuda.current_stream(dev)
    with torch.cuda.device(dev):
        buf = torch.empty(max(total, 1), dtype=torch.uint8, device=dev)
        flat = _pinned_staging(img_at + img.size)
        fl = flat.numpy()
        fl[:8 * nl].view(np.int64)[:] = offs
        fl[8 * nl:12 * nl].view(np.int32)[:] = hs
        fl[12 * nl:16 * nl].view(np.int32)[:] = ws
        np.copyto(fl[img_at:img_at + img.size].reshape(img.shape), img)
        up = flat[:img_at + img.size].to(dev, non_blocking=True)
        _STAGING.event = torch.cuda.Event()
        _STAGING.event.record(st)                 # the staging buffer is reused by this thread's next call
        d_off, d_h, d_w = up[:8 * nl].view(torch.int64), up[8 * nl:12 * nl].view(torch.int32), up[12 * nl:16 * nl].view(torch.int32)
        if nl:
            need = int(L.gims_pyramid_workspace_bytes(h, w, cn))
            key = (str(dev), st.cuda_stream, __import__('threading').get_ident())
            with _PYR_WS_LOCK:
                wsp = _PYR_WS.get(key)
            if wsp is None or wsp.numel() < need:
                wsp = torch.empty(need, dtype=torch.uint8, device=dev)
                with _PYR_WS_LOCK:
                    _PYR_WS[key] = wsp
            _lib.check(L.gims_gaussian_pyramid(_lib.ptr(up[img_at:]), h, w, cn, _lib.ptr(buf), _lib.ptr(wsp), wsp.numel(),
                                               C.c_void_p(st.cuda_stream)), 'gims_gaussian_pyramid')
    return DevicePyramid(buf, d_off, d_h, d_w, shapes, offs, cn, up[img_at:])


def extract_patches_device(kps, levels, device):
    """`extract_patches` on the GPU: (N, 32, 32[, C]) float32 ON `device`, bit-identical to the host path (the kernel follows
    OpenCV's 8-bit fixed-point cubic warp, csrc/patches.cu).  `levels`: the host pyramid (a list of uint8 arrays; the
    levels that carry keypoints are uploaded) or a `DevicePyramid` of the same device (nothing is uploaded).  `kps`: a list
    of cv2.KeyPoint or the `DeviceKeypoints` of `detect_device`."""
    import ctypes as C
    from . import _lib
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise _lib.GimsError('extract_patches_device needs a CUDA device')
    n = len(kps)
    on_device = isinstance(levels, DevicePyramid)
    if on_device:
        pdev = levels.buffer.device
        if dev.index is not None and dev.index != pdev.index:
            raise _lib.GimsError('extract_patches_device: the pyramid is on %s, not %s' % (pdev, dev))
        dev, cn = pdev, levels.channels
        grey = cn == 1
    else:
        cn = levels[0].shape[2] if levels[0].ndim == 3 else 1
        grey = levels[0].ndim != 3
    shape = (n, PATCH_SIZE, PATCH_SIZE) if grey else (n, PATCH_SIZE, PATCH_SIZE, cn)
    out = torch.empty(shape, dtype=torch.float32, device=dev)
    if n == 0:
        return out
    level, inv = patch_maps_from_arrays(*kps.host()) if isinstance(kps, DeviceKeypoints) else patch_maps(kps)
    st = torch.cuda.current_stream(dev)
    if on_device:
        if int(level.max()) >= len(levels):
            raise _lib.GimsError('extract_patches_device: a keypoint names level %d of a %d-level pyramid'
                                 % (int(level.max()), len(levels)))
        with torch.cuda.device(dev):
            d_level = torch.from_numpy(level).to(dev)
            d_inv = torch.from_numpy(inv).to(dev)
            _lib.check(_lib.lib().gims_extract_patches(_lib.ptr(levels.buffer), _lib.ptr(levels.offset),
                                                       _lib.ptr(levels.height), _lib.ptr(levels.width), len(levels), cn,
                                                       _lib.ptr(d_level), _lib.ptr(d_inv), n, _lib.ptr(out),
                                                       C.c_void_p(st.cuda_stream)), 'gims_extract_patches')
        return out
    # only the levels that carry keypoints travel (the coarse octaves are small, the unused fine ones are not)
    used = np.zeros(len(levels), dtype=bool)
    used[level] = True
    sizes = [int(l.size) if u else 0 for l, u in zip(levels, used)]
    offs = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    total = int(sum(sizes))
    flat = _pinned_staging(total)
    fl = flat.numpy()
    for l, o, u in zip(levels, offs, used):
        if not u:
            continue
        if l.dtype != np.uint8:
            raise _lib.GimsError('extract_patches_device: pyramid levels must be uint8 (got %s)' % l.dtype)
        np.copyto(fl[o:o + l.size].reshape(l.shape), l)
    with torch.cuda.device(dev):
        d_lv = flat[:total].to(dev, non_blocking=True)
        _STAGING.event = torch.cuda.Event()
        _STAGING.event.record(st)                 # the staging buffer is reused by this thread's next call
        d_off = torch.from_numpy(offs).to(dev)
        d_h = torch.tensor([l.shape[0] for l in levels], dtype=torch.int32, device=dev)
        d_w = torch.tensor([l.shape[1] for l in levels], dtype=torch.int32, device=dev)
        d_level = torch.from_numpy(level).to(dev)
        d_inv = torch.from_numpy(inv).to(dev)
        _lib.check(_lib.lib().gims_extract_patches(_lib.ptr(d_lv), _lib.ptr(d_off), _lib.ptr(d_h), _lib.ptr(d_w), len(levels), cn,
                                                   _lib.ptr(d_level), _lib.ptr(d_inv), n, _lib.ptr(out),
                                                   C.c_void_p(st.cuda_stream)), 'gims_extract_patches')
        # the staging buffers may be freed once the stream has passed this point
        for t in (d_lv, d_off, d_h, d_w, d_level, d_inv):
            t.record_stream(st)
    return out


def describe(patches, carhynet, device, batch_size=512):
    """(N, 128) descriptors ON `device`.  `patches`: (N, 32, 32, 3) colour or (N, 32, 32) grey, float in [0, 1]; a numpy
    array (host path) or a tensor that is already on the device (extract_patches_device)."""
    n = len(patches)
    model = getattr(carhynet, 'model', None)
    if not isinstance(model, torch.nn.Module) and isinstance(carhynet, torch.nn.Module):
        model = carhynet
    if model is None:
        # only the reference's host interface is available (carhynet/models.py:667-670): use it, upload once
        if torch.is_tensor(patches):
            patches = patches.cpu().numpy()
        _, d = carhynet.compute_sift(patches, list(range(n)), patches.ndim == 4)
        return torch.as_tensor(np.asarray(d, dtype=np.float32).reshape(n, -1), device=device)
    batch_size = int(getattr(carhynet, 'batch_size', batch_size))
    p = next(model.parameters(), None)
    mdev = p.device if p is not None else torch.device(device)
    x = patches if torch.is_tensor(patches) else torch.from_numpy(np.ascontiguousarray(patches, dtype=np.float32))
    x = x.permute(0, 3, 1, 2) if x.dim() == 4 else x.unsqueeze(1)
    outs = []
    with torch.no_grad():
        for i in range(0, n, batch_size):
            chunk = x[i:i + batch_size]
            if chunk.device != mdev:
                chunk = chunk.pin_memory().to(mdev, non_blocking=True) if (mdev.type == 'cuda' and not chunk.is_cuda) else chunk.to(mdev)
            outs.append(model(chunk).reshape(chunk.shape[0], -1))
    d = torch.cat(outs) if outs else torch.zeros(0, 128, device=mdev)
    return d.to(device)


def device_pyramids(images, device):
    """Enqueue `gaussian_pyramid_device` for every image of `images` that it takes (uint8, 1 or 3 channels) when `device`
    is a CUDA device and GIMS_HOST_PATCHES is not 1; None for the others, whose pyramid stays on the host."""
    on_gpu = torch.device(device).type == 'cuda' and os.environ.get('GIMS_HOST_PATCHES') != '1'
    return [gaussian_pyramid_device(img, device) if on_gpu and pyramid_on_device(img) else None for img in images]


def host_stages(image_sets, max_kp=-1, pyramids=None):
    """The OpenCV stages (SIFT detection + Gaussian pyramid) of several images side by side — OpenCV releases the GIL, and
    the reference runs image 0 and image 1 one after the other (matching.py:18-24).  `image_sets`: a list of iterables of
    images (each what `data['image']` is); returns, per set, a list of (keypoints, pyramid levels).  `pyramids`, if given,
    holds per set and image a pyramid already built (a `DevicePyramid`) or None: only the None ones are built here."""
    flat = [np.asarray(img) for imgs in image_sets for img in imgs]
    counts = [len(imgs) for imgs in image_sets]
    pyrs = [p for ps in pyramids for p in ps] if pyramids is not None else [None] * len(flat)

    def stage(args):
        img, pyr = args
        return detect(img, max_kp), (gaussian_pyramid(img) if pyr is None else pyr)
    if len(flat) > 1:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(flat), 8)) as pool:
            done = list(pool.map(stage, zip(flat, pyrs)))
    else:
        done = [stage(a) for a in zip(flat, pyrs)]
    out, i = [], 0
    for c in counts:
        out.append(done[i:i + c])
        i += c
    return out


SIFT_KP_CAP = 16384             # first keypoint capacity of detect_device; 4x more on each overflow
_SIFT_WS = {}                   # (device, stream, thread) -> grow-only uint8 workspace of gims_sift_detect
_SIFT_WS_LOCK = __import__('threading').Lock()


class DeviceKeypoints:
    """The keypoints `detect_device` found in one image, on the device: `pt` (N, 2), `size`, `angle`, `response` float32
    and `octave` int32 (packed as cv2.KeyPoint.octave), in cv2's order (see gims_sift_detect).  `host()` gives the same
    records as numpy arrays (pt, size, angle, octave), read back once with the count."""

    def __init__(self, n, pt, size, angle, response, octave, host):
        self.n, self.pt, self.size, self.angle, self.response, self.octave = n, pt, size, angle, response, octave
        self._host = host

    def __len__(self):
        return self.n

    def host(self):
        return self._host

    def keypoints(self):
        """The records as a list of cv2.KeyPoint."""
        cv2 = _cv2()
        pt, size, angle, octave = self._host
        resp = self.response.cpu().numpy()
        return [cv2.KeyPoint(float(pt[i, 0]), float(pt[i, 1]), float(size[i]), float(angle[i]), float(resp[i]),
                             int(octave[i])) for i in range(self.n)]


class _PendingDetect:
    """A detection enqueued by `detect_enqueue`: the device outputs and their pinned host copy, not yet waited for."""

    def __init__(self, image, h, w, cn, dev, max_keypoints, kp_cap):
        import ctypes as C
        from . import _lib
        self.args = (image, h, w, cn, dev, max_keypoints)
        self.cap = kp_cap
        L = _lib.lib()
        st = torch.cuda.current_stream(dev)
        with torch.cuda.device(dev):
            # one buffer: count, status, 2 spare ints, then pt [cap][2], size, angle, response, octave
            out = torch.zeros(4 + 6 * kp_cap, dtype=torch.int32, device=dev)
            f = out.view(torch.float32)
            self.pt = f[4:4 + 2 * kp_cap].view(kp_cap, 2)
            self.size, self.angle, self.response = (f[4 + k * kp_cap:4 + (k + 1) * kp_cap] for k in (2, 3, 4))
            self.octave = out[4 + 5 * kp_cap:]
            need = int(L.gims_sift_workspace_bytes(h, w, cn, kp_cap))
            key = (str(dev), st.cuda_stream, __import__('threading').get_ident())
            with _SIFT_WS_LOCK:
                wsp = _SIFT_WS.get(key)
            if wsp is None or wsp.numel() < need:
                wsp = torch.empty(need, dtype=torch.uint8, device=dev)
                with _SIFT_WS_LOCK:
                    _SIFT_WS[key] = wsp
            _lib.check(L.gims_sift_detect(_lib.ptr(image), h, w, cn, max_keypoints, kp_cap, _lib.ptr(wsp), wsp.numel(),
                                          _lib.ptr(self.pt), _lib.ptr(self.size), _lib.ptr(self.angle),
                                          _lib.ptr(self.response), _lib.ptr(self.octave), _lib.ptr(out[0:1]),
                                          _lib.ptr(out[1:2]), C.c_void_p(st.cuda_stream)), 'gims_sift_detect')
            self.host = torch.empty(out.numel(), dtype=torch.int32, pin_memory=True)
            self.host.copy_(out, non_blocking=True)
            self.done = torch.cuda.Event()
            self.done.record(st)
        self.out = out

    def result(self):
        """Wait for the read-back; on GIMS_STATUS_KEYPOINT_OVERFLOW run again with 4x the capacity."""
        from . import _lib
        self.done.synchronize()
        hv = self.host.numpy()
        status = int(hv[1])
        if status & _lib.STATUS_KEYPOINT_OVERFLOW:
            return _PendingDetect(*self.args, kp_cap=4 * self.cap).result()
        if status & _lib.STATUS_ERROR_MASK:
            raise _lib.GimsError('gims_sift_detect: status 0x%x' % status)
        n, cap = int(hv[0]), self.cap
        hf = hv.view(np.float32)
        host = (hf[4:4 + 2 * n].reshape(n, 2).astype(np.float64), hf[4 + 2 * cap:4 + 2 * cap + n].astype(np.float64),
                hf[4 + 3 * cap:4 + 3 * cap + n].astype(np.float64), hv[4 + 5 * cap:4 + 5 * cap + n].astype(np.int64))
        return DeviceKeypoints(n, self.pt[:n], self.size[:n], self.angle[:n], self.response[:n], self.octave[:n], host)


def detect_enqueue(image, device, max_keypoints=-1, pyramid=None, kp_cap=SIFT_KP_CAP):
    """Enqueue `detect_device` on the current stream of `device` without waiting; `.result()` of the returned object
    waits and gives the `DeviceKeypoints`.  `pyramid`: the `DevicePyramid` of the same image, whose uploaded copy is
    reused (otherwise the image is uploaded here)."""
    from . import _lib
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise _lib.GimsError('detect_device needs a CUDA device')
    img = np.asarray(image)
    if not pyramid_on_device(img):
        raise _lib.GimsError('detect_device: need a uint8 (H, W), (H, W, 1) or (H, W, 3) image (got %s %s)'
                             % (img.dtype, img.shape))
    h, w = img.shape[:2]
    cn = 3 if img.ndim == 3 and img.shape[2] == 3 else 1
    if pyramid is not None and pyramid.image is not None:
        d_img = pyramid.image
        dev = d_img.device
    else:
        with torch.cuda.device(dev):
            d_img = torch.from_numpy(np.ascontiguousarray(img).reshape(-1)).pin_memory().to(dev, non_blocking=True)
    return _PendingDetect(d_img, h, w, cn, dev, int(max_keypoints), int(kp_cap))


def detect_device(image, device, max_keypoints=-1, pyramid=None):
    """`detect` on the GPU (csrc/sift.cu): SIFT keypoints of a uint8 grey or colour image as `DeviceKeypoints`, the
    strongest `max_keypoints` first if that limit is positive.  Not bit-identical to cv2 (cv2 is not bit-identical to
    itself): the records equal oracle/cv_sift_oracle.py bit for bit and agree with cv2 within 0.01 px, 1e-3 relative size
    and 0.5 degrees for more than 99 % of keypoints.  Waits for the count and the records (one read-back)."""
    return detect_enqueue(image, device, max_keypoints, pyramid).result()


def sift_forward(data, device, staged=None):
    """Same dict in / dict out as utils/common.py:837-893: `data['image']` iterates over images, `data['carhynet']` is the
    caller's descriptor object; returns lists (one entry per image) of device tensors
    `keypoints` (N, 2) fp32 pixel xy, `scores` (N,) fp32 SIFT responses, `descriptors` (256, N) fp32.
    `staged`: the (keypoints, pyramid) pairs of the images if `host_stages` has already produced them.  On a CUDA device
    the pyramid of a uint8 grey or colour image is built there (enqueued before detection starts, so the two overlap)."""
    max_kp = data.get('max_keypoints', -1)
    kpts, scores, descs = [], [], []
    images = [np.asarray(img) for img in data['image']]
    if staged is None:
        staged = host_stages([images], max_kp, [device_pyramids(images, device)])[0]
    for img, (kps, levels) in zip(images, staged):
        if isinstance(levels, DevicePyramid):
            patches = extract_patches_device(kps, levels, device)
        else:
            on_gpu = torch.device(device).type == 'cuda' and levels[0].dtype == np.uint8 and os.environ.get('GIMS_HOST_PATCHES') != '1'
            patches = extract_patches_device(kps, levels, device) if on_gpu else extract_patches(kps, levels)
        d = describe(patches, data['carhynet'], device)                        # (N, 128), on the device
        if isinstance(kps, DeviceKeypoints):
            kpts.append(kps.pt)
            scores.append(kps.response)
        else:
            pts = np.array([k.pt for k in kps], dtype=np.float32).reshape(-1, 2)
            resp = np.array([k.response for k in kps], dtype=np.float32)
            kpts.append(torch.from_numpy(pts).to(device))
            scores.append(torch.from_numpy(resp).to(device))
        descs.append(torch.cat([d, d], dim=1).t().contiguous())                # utils/common.py:891
    return {'keypoints': kpts, 'scores': scores, 'descriptors': descs}
