"""oracle/seeding.py -- TEST INFRASTRUCTURE ONLY.

Plain-torch restatement of the reference's temporal-CAM max and seed selection, line by line, so that the
CUDA kernels (tcam_seed_select / tcam_seed_labels) can be compared with it bit for bit on the same random
stream.  It runs on whatever device its inputs are on and uses the very same torch calls as the reference
(``torch.sort(stable=True)``, ``nonzero``, ``Tensor.multinomial``), in the same order:

  temporal_max         <- dlib/datasets/wsol_loader.py:591-600   (chain of torch.maximum)
  sample_fg            <- _SFG.forward      dlib/cams/tcam_seeding.py:498-544
  sample_bg            <- _SBG.forward      dlib/cams/tcam_seeding.py:555-592
  one_sample           <- _OneSample.forward  tcam_seeding.py:453-487   (roi given or unused)
  flat_dilation        <- kornia==0.6.4 kornia.morphology.dilation with a ones kernel (third-party, not in
                          /root/reference; requirements.txt:36): out = max over the ksz x ksz window whose
                          origin is (ksz//2, ksz//2), positions outside the image ignored (geodesic border)
  tcam_seeder_forward  <- TCAMSeeder.forward  tcam_seeding.py:178-256

Parity of flat_dilation and of torch 2.11's multinomial/sort against the versions the reference pins
(torch 1.11, kornia 0.6.4) is UNPINNED: no reference test fixes them and those packages are not installed
here (SURVEY.md §8c).  Their documented semantics are restated.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

SEED_UNIFORM = 'seed_uniform'
SEED_WEIGHTED = 'seed_weighted'


def temporal_max(cams: torch.Tensor) -> torch.Tensor:
    """cams [B,T,...] -> [B,...]: std_cam = maximum(std_cam, cam_t) frame after frame."""
    out = cams[:, 0]
    for t in range(1, cams.shape[1]):
        out = torch.maximum(out, cams[:, t])
    return out


def re_normalize_cam(cam: torch.Tensor, h: float) -> torch.Tensor:
    """dlib/datasets/wsol_loader.py:630-635, line by line."""
    _cam = cam + 1e-6
    e = torch.exp(_cam * h)
    e = e / e.max()  # in [0, 1]
    e = torch.nan_to_num(e, nan=0.0, posinf=1., neginf=0.0)
    return e


def temporal_max_renorm(cams: torch.Tensor, h: float) -> torch.Tensor:
    """cams [B,T,...]: the loader's loop (wsol_loader.py:591-600) with re_normalize_cam on every frame."""
    outs = []
    for b in range(cams.shape[0]):
        std = None
        for t in range(cams.shape[1]):
            c = re_normalize_cam(cams[b, t], h) if h > 0 else cams[b, t]
            std = c if std is None else torch.maximum(std, c)
        outs.append(std)
    return torch.stack(outs)


def prepare_std_cams_disq(std_cams: torch.Tensor, image_size) -> torch.Tensor:
    """dlib/learning/train_wsol.py:417-432, line by line."""
    cams = std_cams.detach()
    cams = torch.nan_to_num(cams, nan=0.0, posinf=1., neginf=0.0)
    cams = torch.nn.functional.interpolate(cams, image_size, mode='bilinear', align_corners=False)
    cams = torch.nan_to_num(cams, nan=0.0, posinf=1., neginf=0.0)
    return cams


def fg_candidates(cam, roi, max_p):
    """The first half of _SFG.forward (tcam_seeding.py:498-530): (n, _cam, tmp) with n the number of candidates, _cam
    the scores (cam*roi + 1e-8 or cam + 1e-8) and tmp [h,w] 1 at the n largest scores (stable sort: ties to the
    lower pixel index), 0 elsewhere."""
    h, w = cam.shape
    if roi is not None:
        n = roi.sum()
        _cam = cam * roi
        _cam = _cam + 1e-8
    else:
        n = h * w
        _cam = cam + 1e-8
    n = int(max_p * n)
    _cam_flatten = _cam.view(h * w)
    val, idx_ = torch.sort(_cam_flatten, dim=0, descending=True, stable=True)
    tmp = _cam_flatten * 0.
    tmp[idx_[:n]] = 1
    return n, _cam, tmp.view(h, w)


def bg_candidates(cam, min_p):
    """The first half of _SBG.forward (tcam_seeding.py:555-580): (n, tmp) with tmp [h,w] 1 at the n smallest
    cam + 1e-8 (stable sort), 0 elsewhere."""
    h, w = cam.shape
    n = int(min_p * h * w)
    _cam = cam + 1e-8
    _cam_flatten = _cam.view(h * w)
    val, idx_ = torch.sort(_cam_flatten, dim=0, descending=False, stable=True)
    tmp = _cam_flatten * 0.
    tmp[idx_[:n]] = 1
    return n, tmp.view(h, w)


def sample_fg(cam, roi, fg, max_p, max_, seed_tech):
    n, _cam, tmp = fg_candidates(cam, roi, max_p)
    if (n > 0) and (max_ > 0):
        _idx = torch.nonzero(tmp, as_tuple=True)
        if seed_tech == SEED_UNIFORM:
            probs = torch.ones(n, dtype=torch.float, device=cam.device)
        elif seed_tech == SEED_WEIGHTED:
            probs = _cam[_idx[0], _idx[1]]
            assert probs.numel() == n
        else:
            raise NotImplementedError(seed_tech)
        selected = probs.multinomial(num_samples=min(max_, n), replacement=False)
        fg[_idx[0][selected], _idx[1][selected]] = 1
    return fg


def sample_bg(cam, bg, min_p, min_):
    n, tmp = bg_candidates(cam, min_p)
    if (n > 0) and (min_ > 0):
        _idx = torch.nonzero(tmp, as_tuple=True)
        probs = torch.ones(n, dtype=torch.float, device=cam.device)   # _SBG is always built with SEED_UNIFORM
        selected = probs.multinomial(num_samples=min(min_, n), replacement=False)
        bg[_idx[0][selected], _idx[1][selected]] = 1
    return bg


def one_sample(cam, roi, *, min_p, max_p, min_, max_, seed_tech, use_roi):
    h, w = cam.shape
    fg = torch.zeros((h, w), dtype=torch.long, device=cam.device)
    bg = torch.zeros((h, w), dtype=torch.long, device=cam.device)
    if cam.min() == cam.max():
        return fg, bg
    _roi = roi if use_roi else None
    fg = sample_fg(cam, _roi, fg, max_p, max_, seed_tech)
    bg = sample_bg(cam, bg, min_p, min_)
    return fg, bg


def flat_dilation(x: torch.Tensor, ksz: int) -> torch.Tensor:
    """x [B,1,H,W] (0/1) -> same shape: flat ksz x ksz dilation, window origin ksz//2, outside ignored."""
    if ksz == 1:
        return x
    o = ksz // 2
    padded = F.pad(x.float(), (o, ksz - o - 1, o, ksz - o - 1), value=float('-inf'))
    return F.max_pool2d(padded, kernel_size=ksz, stride=1).to(x.dtype)


def tcam_seeder_forward(x, roi=None, *, seed_tech, min_, max_, min_p, max_p, ksz, ignore_idx, use_roi):
    b, d, h, w = x.shape
    assert d == 1
    out = torch.zeros((b, h, w), dtype=torch.long, device=x.device) + ignore_idx
    all_fg = torch.zeros((b, h, w), dtype=torch.long, device=x.device)
    all_bg = torch.zeros((b, h, w), dtype=torch.long, device=x.device)
    for i in range(b):
        _roi = roi[i].squeeze() if roi is not None else None
        all_fg[i], all_bg[i] = one_sample(x[i].squeeze(), _roi, min_p=min_p, max_p=max_p, min_=min_, max_=max_,
                                          seed_tech=seed_tech, use_roi=use_roi)
    all_fg = flat_dilation(all_fg.unsqueeze(1), ksz).squeeze(1)
    all_bg = flat_dilation(all_bg.unsqueeze(1), ksz).squeeze(1)
    outer = all_fg + all_bg
    all_fg[outer == 2] = 0
    all_bg[outer == 2] = 0
    out[all_fg == 1] = 1
    out[all_bg == 1] = 0
    return out.detach()


# --------------------------------------------------------------------------------------------------
# ROI by Otsu (numpy, like the reference runs it on the CPU)
# --------------------------------------------------------------------------------------------------
def threshold_otsu_skimage(image, nbins=256):
    """scikit-image 0.17.2 ``skimage.filters.threshold_otsu`` restated (third-party, requirements.txt:83;
    not installed here -> parity UNPINNED against the real package).  ``histogram(image.ravel(), nbins,
    source_range='image')`` is ``np.histogram(image, bins=nbins)`` plus bin centres for float images."""
    import numpy as np
    first_pixel = image.ravel()[0]
    if np.all(image == first_pixel):
        return first_pixel
    hist, bin_edges = np.histogram(image.ravel(), bins=nbins, range=None)
    bin_centers = (bin_edges[:-1] + bin_edges[1:]) / 2.
    hist = hist.astype(float)
    weight1 = np.cumsum(hist)
    weight2 = np.cumsum(hist[::-1])[::-1]
    mean1 = np.cumsum(hist * bin_centers) / weight1
    mean2 = (np.cumsum((hist * bin_centers)[::-1]) / weight2[::-1])[::-1]
    variance12 = weight1[:-1] * weight2[1:] * (mean1[:-1] - mean2[1:]) ** 2
    idx = np.argmax(variance12)
    return bin_centers[:-1][idx]


def roi_all_single_cam(cam):
    """GetRoiSingleCam(roi_method='roi_all').__call__ + get_thresh (dlib/cams/tcam_seeding.py:325-345,419-430)
    for one CAM given as a float32 numpy array [h,w]; returns (roi int64 [h,w], threshold on the 0..255 scale)."""
    import numpy as np
    _cam = np.asarray(cam, dtype=np.float32)
    cam_ = np.floor(_cam * 255.)
    if cam_.min() == cam_.max():
        th = 0.
    else:
        th = threshold_otsu_skimage(cam_)
    blobs = (_cam * 255. >= th).astype(int)
    return blobs.astype(np.int64), float(th)


def roi_components_single_cam(cam, roi_method, p_min_area_roi, thresh=None):
    """GetRoiSingleCam.__call__ for roi_method 'roi_high_density' / 'largest' (dlib/cams/tcam_seeding.py:325-417),
    line by line, with the two third-party calls restated:
      * skimage.measure.label(blobs, background=0, connectivity=1) -> scipy.ndimage.label with the 4-neighbour
        structure (same components; both number them in raster order of their first pixel);
      * cv2.findContours(RETR_EXTERNAL) + cv2.boundingRect on ONE 4-connected component -> its bounding rectangle
        (x, y, w, h) = (min col, min row, extent, extent), then dlib/utils/wsol.py:133-137.
    Returns (final_roi int64 [h,w], bbox_mask float32 [h,w], bbox [1,4] x0y0x1y1)."""
    import numpy as np
    from scipy import ndimage
    _cam = np.asarray(cam, dtype=np.float32)
    h, w = _cam.shape
    if thresh is None:
        cam_ = np.floor(_cam * 255.)
        _thresh = 0. if cam_.min() == cam_.max() else threshold_otsu_skimage(cam_)
    else:
        _thresh = thresh * 255.
    blobs = (_cam * 255. >= np.float32(_thresh)).astype(int)
    four = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]])
    blobs_labels, _ = ndimage.label(blobs, structure=four)
    labels = np.unique(blobs_labels)
    if labels.size == 1:
        final_roi = blobs.astype(float)
    else:
        label_density, label_area = dict(), dict()
        min_area = (h * w) * p_min_area_roi
        for l in labels:
            if l == 0:
                continue
            s_roi = (blobs_labels == l).astype(float)
            s_cam = _cam * s_roi
            s_roi_area = s_roi.sum()
            label_density[l] = s_cam.sum() / s_roi_area
            label_area[l] = s_roi_area
        if roi_method == 'roi_high_density':
            l_roi = max(label_density, key=label_density.get)
            if label_area[l_roi] < min_area:
                l_roi = max(label_area, key=label_area.get)
        elif roi_method == 'largest':
            l_roi = max(label_area, key=label_area.get)
        else:
            raise NotImplementedError(roi_method)
        final_roi = (blobs_labels == l_roi).astype(float)
    ys, xs = np.nonzero(final_roi > 0.5)
    if ys.size == 0:
        bbox = np.array([[0, 0, 0, 0]])
    else:
        x, y, bw, bh = xs.min(), ys.min(), xs.max() - xs.min() + 1, ys.max() - ys.min() + 1
        bbox = np.array([[x, y, min(x + bw, w - 1), min(y + bh, h - 1)]])
    bbox_mask = np.zeros((h, w), dtype=np.float32)
    x0, y0, x1, y1 = bbox.flatten()
    bbox_mask[y0:y1, x0:x1] = 1.
    return final_roi.astype(np.int64), bbox_mask, bbox.astype(np.float32)
