"""Caller-side result consumption on the device (SURVEY.md §8f row 3) — what eval_homography.py:180-229 does with a
matcher result, without moving it to the host first.

  torch_find_matches(kpts0, kpts1, homography, dist_thresh, n_iters)
      same signature and results as utils/preprocess_utils.py:98-132: (match_list_1, match_list_2, missing_1, missing_2),
      int64 device tensors, the pairs ordered by round and then by image-1 index as the reference produces them.
      One C-ABI call (gims_gt_matches: projection + n_iters rounds of mutual nearest neighbours) instead of
      n_iters x (N0 x N1 distance matrix, two argmin, unique / cat bookkeeping).
  gt_match_vector(...)   the dense form eval_homography.py:210-211 builds: gt[i] = partner index in image 1 or -1.
  precision_recall(pred, gt0)   eval_homography.py:224-228 as three device-side counts.
  matched_points(pred)   eval_homography.py:187-189: the matched keypoint pairs and confidences, still on the device.
  find_homographies(src_list, dst_list, ...)   cv2.findHomography(..., cv2.RANSAC, ...) of eval_homography.py and
      eval_matches.py for a batch of pairs in one C-ABI call (gims_find_homographies); device tensors in and out.
  find_homography(srcPoints, dstPoints, method, ...)   the drop-in for that cv2 call: numpy in, (H, mask) numpy out.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import GimsError


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def gt_match_vector(kpts0, kpts1, homography, dist_thresh=3, n_iters=1):
    """(gt0 int32 [N0], gt1 int32 [N1], round0 int32 [N0]) on the device of `kpts0`."""
    dev = kpts0.device
    if dev.type != 'cuda':
        raise GimsError('gims_b200.postprocess runs on a CUDA device only (no CPU fallback)')
    L = _lib.lib()
    k0 = kpts0.detach().to(torch.float32).contiguous()
    k1 = kpts1.detach().to(device=dev, dtype=torch.float32).contiguous()
    n0, n1 = k0.shape[0], k1.shape[0]
    if n0 < 1 or n1 < 1:
        raise GimsError('torch_find_matches: empty keypoint set')          # the reference raises inside torch.argmin
    h = torch.as_tensor(homography).detach().to(device=dev, dtype=torch.float32).contiguous().reshape(9)
    ws = torch.empty(L.gims_gt_workspace_bytes(n0, n1), dtype=torch.uint8, device=dev)
    gt0 = torch.empty(n0, dtype=torch.int32, device=dev)
    gt1 = torch.empty(n1, dtype=torch.int32, device=dev)
    rnd = torch.empty(n0, dtype=torch.int32, device=dev)
    _lib.check(L.gims_gt_matches(_lib.ptr(k0), n0, _lib.ptr(k1), n1, _lib.ptr(h), float(dist_thresh), int(n_iters),
                                 _lib.ptr(ws), ws.numel(), _lib.ptr(gt0), _lib.ptr(gt1), _lib.ptr(rnd), _stream(dev)),
               'gims_gt_matches')
    return gt0, gt1, rnd


def torch_find_matches(src_keypoints1, src_keypoints2, homography, dist_thresh=3, n_iters=1):
    """Drop-in for utils/preprocess_utils.py:98-132."""
    gt0, gt1, rnd = gt_match_vector(src_keypoints1, src_keypoints2, homography, dist_thresh, n_iters)
    n1 = gt1.numel()
    idx0 = torch.nonzero(gt0 >= 0).squeeze(1)
    partner = gt0[idx0].long()
    order = torch.argsort(rnd[idx0].long() * n1 + partner)                # by round, then by image-1 index
    match_1, match_2 = idx0[order], partner[order]
    missing_1 = torch.nonzero(gt0 < 0).squeeze(1)
    missing_2 = torch.nonzero(gt1 < 0).squeeze(1)
    return match_1, match_2, missing_1, missing_2


def precision_recall(pred, gt0):
    """eval_homography.py:224-228 for one pair: `pred` is the matcher's output dict (matches0 (1, N0') int64 on the device),
    `gt0` the vector of gt_match_vector.  Returns (precision, recall, counts) — counts = device int32 [tp, predicted, missed];
    the two ratios are device scalars (0-d tensors), nothing is synchronised here."""
    m0 = pred['matches0'] if torch.is_tensor(pred) is False else pred
    m0 = m0.reshape(-1).contiguous()
    dev = m0.device
    if dev.type != 'cuda':
        raise GimsError('gims_b200.postprocess runs on a CUDA device only (no CPU fallback)')
    if m0.dtype != torch.int64 or gt0.dtype != torch.int32 or gt0.numel() != m0.numel():
        raise GimsError('precision_recall: matches0 must be int64 and gt0 int32 of the same length')
    L = _lib.lib()
    counts = torch.empty(3, dtype=torch.int32, device=dev)
    _lib.check(L.gims_match_counts(_lib.ptr(m0), _lib.ptr(gt0.contiguous()), m0.numel(), None, _lib.ptr(counts), _stream(dev)),
               'gims_match_counts')
    c = counts.to(torch.float64)
    return c[0] / c[1], c[0] / (c[0] + c[2]), counts


def matched_points(pred):
    """eval_homography.py:187-189 on the device: (mkpts0, mkpts1, mconf) of the pairs with matches0 > -1."""
    kpts0, kpts1 = pred['keypoints0'][0], pred['keypoints1'][0]
    matches, conf = pred['matches0'][0], pred['matching_scores0'][0]
    valid = matches > -1
    return kpts0[valid], kpts1[matches[valid]], conf[valid]


RANSAC = 8          # cv2.RANSAC, the only method find_homography implements


def _check_ransac_args(threshold, max_iters, confidence):
    if not (float(threshold) > 0.0 and np.isfinite(float(threshold))):
        raise GimsError('find_homographies: threshold must be > 0, got %r' % (threshold,))
    if not 0.0 < float(confidence) < 1.0:
        raise GimsError('find_homographies: confidence must be in (0, 1), got %r' % (confidence,))
    if int(max_iters) < 1:
        raise GimsError('find_homographies: max_iters must be >= 1, got %r' % (max_iters,))


def find_homographies_packed(src, dst, offsets, threshold=3.0, max_iters=2000, confidence=0.995, seed=0):
    """The C-ABI form: src, dst (T, 2) float32 and offsets (P+1,) int32 on one CUDA device, pair p owning rows
    offsets[p]:offsets[p+1].  Returns device tensors (H (P, 3, 3) float64, n_inliers (P,) int32, mask (T,) uint8,
    n_iters (P,) int32).  "Not found" is n_inliers = 0 with H = 0.  Enqueued on the current stream, not synchronised."""
    dev = src.device
    if dev.type != 'cuda':
        raise GimsError('gims_b200.postprocess runs on a CUDA device only (no CPU fallback)')
    _check_ransac_args(threshold, max_iters, confidence)
    if src.dim() != 2 or src.shape[1] != 2 or src.shape != dst.shape or src.dtype != torch.float32 or \
            dst.dtype != torch.float32 or dst.device != dev or offsets.device != dev or offsets.dtype != torch.int32 or \
            offsets.dim() != 1 or offsets.numel() < 1:
        raise GimsError('find_homographies_packed: src, dst (T, 2) float32 and offsets (P+1,) int32 on one device')
    src, dst, offsets = src.contiguous(), dst.contiguous(), offsets.contiguous()
    L = _lib.lib()
    P, T = offsets.numel() - 1, src.shape[0]
    ws = torch.empty(L.gims_homography_workspace_bytes(P, T), dtype=torch.uint8, device=dev)
    H = torch.empty((max(P, 1), 3, 3), dtype=torch.float64, device=dev)
    n_in = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
    n_it = torch.empty(max(P, 1), dtype=torch.int32, device=dev)
    mask = torch.empty(max(T, 1), dtype=torch.uint8, device=dev)
    if T == 0:                       # the C ABI wants real buffers even when every pair is empty
        src = dst = torch.zeros((1, 2), dtype=torch.float32, device=dev)
    _lib.check(L.gims_find_homographies(_lib.ptr(src), _lib.ptr(dst), _lib.ptr(offsets), P, float(threshold),
                                        int(max_iters), float(confidence), int(seed) & 0xFFFFFFFFFFFFFFFF, _lib.ptr(ws),
                                        ws.numel(), _lib.ptr(H), _lib.ptr(mask), _lib.ptr(n_in), _lib.ptr(n_it),
                                        _stream(dev)), 'gims_find_homographies')
    return H[:P], n_in[:P], mask[:T], n_it[:P]


def find_homographies(src_list, dst_list, threshold=3.0, max_iters=2000, confidence=0.995, seed=0):
    """cv2.findHomography(src, dst, cv2.RANSAC, threshold, maxIters=max_iters, confidence=confidence) for a batch of
    pairs in one launch.  src_list[p], dst_list[p]: (M_p, 2) tensors on one CUDA device (M_p may be 0..3: "not found").
    Returns device tensors (H (P, 3, 3) float64, n_inliers (P,) int32, masks: list of (M_p,) uint8).  A pair's result
    does not depend on the rest of the batch.  Nothing is synchronised."""
    if len(src_list) != len(dst_list):
        raise GimsError('find_homographies: %d source and %d destination point sets' % (len(src_list), len(dst_list)))
    if len(src_list) == 0:
        raise GimsError('find_homographies: no pairs')
    dev = src_list[0].device
    sizes = []
    for s, d in zip(src_list, dst_list):
        if not (torch.is_tensor(s) and torch.is_tensor(d)) or s.device != dev or d.device != dev:
            raise GimsError('find_homographies: every point set must be a tensor on %s' % dev)
        if s.dim() != 2 or s.shape[1] != 2 or s.shape != d.shape:
            raise GimsError('find_homographies: point sets must be (M, 2) with the same M on both sides, got %s and %s'
                            % (tuple(s.shape), tuple(d.shape)))
        sizes.append(int(s.shape[0]))
    offs = np.zeros(len(sizes) + 1, dtype=np.int32)
    np.cumsum(sizes, out=offs[1:])
    offsets = torch.from_numpy(offs).pin_memory().to(dev, non_blocking=True) if dev.type == 'cuda' else torch.from_numpy(offs)
    src = torch.cat([s.detach().to(torch.float32) for s in src_list]).contiguous()
    dst = torch.cat([d.detach().to(torch.float32) for d in dst_list]).contiguous()
    H, n_in, mask, _ = find_homographies_packed(src, dst, offsets, threshold, max_iters, confidence, seed)
    return H, n_in, [mask[offs[p]:offs[p + 1]] for p in range(len(sizes))]


def find_homography(srcPoints, dstPoints, method=RANSAC, ransacReprojThreshold=3.0, mask=None, maxIters=2000,
                    confidence=0.995):
    """Drop-in for `cv2.findHomography(srcPoints, dstPoints, cv2.RANSAC, ransacReprojThreshold)` of eval_homography.py
    and eval_matches.py, computed on the current CUDA device.  Takes numpy arrays or tensors of shape (M, 2) (or
    (M, 1, 2)) and returns what cv2 returns: (H float64 (3, 3), mask uint8 (M, 1)), or (None, zeros (M, 1)) when no
    homography is found.  Raises GimsError for M < 4, where cv2 raises, and for any method other than cv2.RANSAC: there
    is no CPU fallback.  `mask` is accepted for signature compatibility and ignored, as cv2's Python binding does."""
    if method != RANSAC:
        raise GimsError('find_homography: only cv2.RANSAC (8) is implemented, got method %r' % (method,))
    _check_ransac_args(ransacReprojThreshold, maxIters, confidence)
    pts = []
    for a in (srcPoints, dstPoints):
        t = a.detach() if torch.is_tensor(a) else torch.from_numpy(np.asarray(a))
        if t.dim() == 3 and t.shape[1] == 1:
            t = t[:, 0]
        if t.dim() != 2 or t.shape[1] != 2:
            raise GimsError('find_homography: points must be (M, 2), got %s' % (tuple(t.shape),))
        pts.append(t)
    if pts[0].shape[0] != pts[1].shape[0]:
        raise GimsError('find_homography: %d source and %d destination points' % (pts[0].shape[0], pts[1].shape[0]))
    m = pts[0].shape[0]
    if m < 4:
        raise GimsError('find_homography: at least 4 correspondences are needed, got %d' % m)
    dev = pts[0].device if pts[0].is_cuda else torch.device('cuda', torch.cuda.current_device())
    H, n_in, masks = find_homographies([pts[0].to(dev)], [pts[1].to(dev)], ransacReprojThreshold, maxIters, confidence)
    H = H[0].cpu().numpy()
    out_mask = masks[0].cpu().numpy().reshape(m, 1)
    if H[2, 2] == 0.0:
        return None, np.zeros((m, 1), dtype=np.uint8)
    return H, out_mask
