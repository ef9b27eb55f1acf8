"""TCAMSeeder -- drop-in for ``dlib/cams/tcam_seeding.py::TCAMSeeder`` of the reference.

Same constructor arguments, same ``forward(x, roi=None)`` contract (``x`` CAMs ``[B,1,H,W]`` in [0,1],
``roi`` long ``[B,1,H,W]``; returns long ``[B,H,W]`` in {ignore, 0 bg, 1 fg}), ``set_seed_tech``,
``use_all_roi`` and ``extra_repr``.  The reference loops over the samples in Python and, per sample, runs two
full stable sorts, ``nonzero``, ``multinomial`` and several host syncs (tcam_seeding.py:232-237,453-592);
here the whole batch is ONE kernel launch (``tcam_seed_fused``, csrc/seed.cuh: a thread-block cluster per sample does
the temporal max, the candidate counts, both selections and the label map; frames too large for an SM's shared memory
take ``tcam_seed_select`` + ``tcam_seed_labels``) and, with ``rng_parity=True``, ONE host sync (to size the random
draws exactly like the reference does).

Random draws.  ``torch.multinomial(probs, k, replacement=False)`` is ``topk(probs / q)`` with
``q = empty_like(probs).exponential_(1)``.  With ``rng_parity=True`` (default) the draws are taken from the
current torch CUDA generator with the same sizes and in the same order as the reference's calls
(sample 0 fg, sample 0 bg, sample 1 fg, ...), so for the same seed the seeds are bit-identical to the
reference's.  ``rng_parity=False`` makes the Exp(1) draws inside the kernel (Philox4x32-10, keyed by two words taken
from torch's CUDA generator per call: ``torch.manual_seed`` still makes runs repeatable; same distribution, different
stream), only for the candidates: no host sync, no draw tensor, capturable in a CUDA graph.

``use_roi=True`` with ``roi=None``: the reference computes the ROI on the CPU with scikit-image's Otsu, one
sample at a time (tcam_seeding.py:476-479); here ``roi_method='roi_all'`` runs as one kernel for the batch
(``tcam_otsu_roi``, SURVEY.md §8f.2) and the two connected-component modes (``roi_high_density``, ``largest``)
as one kernel too (``tcam_roi_components``).
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops

__all__ = ['TCAMSeeder', 'SparseSeeds', 'GetRoiSingleCam', 'SEED_UNIFORM', 'SEED_WEIGHTED', 'ROI_ALL', 'ROI_H_DENSITY', 'ROI_LARGEST']

# dlib/configure/constants.py:352-354,368-372
SEED_UNIFORM = 'seed_uniform'
SEED_WEIGHTED = 'seed_weighted'
SEED_TECHS = [SEED_UNIFORM, SEED_WEIGHTED]
ROI_ALL = 'roi_all'
ROI_H_DENSITY = 'roi_high_density'
ROI_LARGEST = 'largest'
ROI_SELECT = [ROI_ALL, ROI_H_DENSITY, ROI_LARGEST]


class SparseSeeds(object):
    """The seeder's output before it is painted into a label map: the selected pixel indices ``sel`` [B,2,kmax] int32
    (side 0 = foreground, 1 = background, -1 = unused) with the dilation size and the ignore index that turn them into
    labels.  Unused slots are trailing: ``dense()`` (``seed_labels_kernel``) stops reading a side at its first -1.  ``SelfLearningTcams`` / ``FusedTcamLosses`` take it as ``seeds`` and compute the cross-entropy from the
    2*kmax*ksz^2 labelled pixels per sample directly (the map is 99.96 % ignore with the README recipe); ``dense()``
    paints the reference's [B,H,W] long map when something else needs it."""

    def __init__(self, sel: torch.Tensor, ksz: int, ignore_idx: int, h: int, w: int):
        self.sel, self.ksz, self.ignore_idx, self.h, self.w = sel, int(ksz), int(ignore_idx), int(h), int(w)

    @property
    def kmax(self) -> int:
        return int(self.sel.shape[2])

    def dense(self) -> torch.Tensor:
        lib = _lib.load()
        b = self.sel.shape[0]
        out = torch.empty((b, self.h, self.w), dtype=torch.long, device=self.sel.device)
        with torch.cuda.device(self.sel.device):
            _lib.check(lib.tcam_seed_labels(self.sel.data_ptr(), self.kmax, b, self.h, self.w, self.ksz, self.ignore_idx,
                                            out.data_ptr(), torch.cuda.current_stream(self.sel.device).cuda_stream),
                       'tcam_seed_labels')
        return out


class TCAMSeeder(nn.Module):
    def __init__(self,
                 seed_tech: str,
                 min_: int,
                 max_: int,
                 max_p: float,
                 min_p: float,
                 fg_erode_k: int,
                 fg_erode_iter: int,
                 ksz: int,
                 support_background: bool,
                 multi_label_flag: bool,
                 seg_ignore_idx: int,
                 cuda_id: int,
                 roi_method: str,
                 p_min_area_roi: float,
                 use_roi: bool,
                 rng_parity: bool = True
                 ):
        super(TCAMSeeder, self).__init__()
        assert seed_tech in SEED_TECHS, seed_tech
        self.seed_tech = seed_tech
        assert not multi_label_flag
        assert isinstance(cuda_id, int)
        assert cuda_id >= 0, cuda_id
        self._device = torch.device('cuda', cuda_id)
        assert isinstance(ksz, int)
        assert ksz > 0
        self.ksz = ksz
        assert isinstance(min_, int)
        assert isinstance(max_, int)
        assert min_ >= 0
        assert max_ >= 0
        assert min_ + max_ > 0
        self.min_ = min_
        self.max_ = max_
        assert isinstance(min_p, float)
        assert 0. <= min_p <= 1.
        self.min_p = min_p
        assert isinstance(max_p, float)
        assert 0. <= max_p <= 1.
        self.max_p = max_p
        assert isinstance(fg_erode_k, int)
        assert fg_erode_k >= 1
        self.fg_erode_k = fg_erode_k
        assert isinstance(fg_erode_iter, int)
        assert fg_erode_iter >= 0
        self.fg_erode_iter = fg_erode_iter
        self.support_background = support_background
        self.multi_label_flag = multi_label_flag
        self.ignore_idx = seg_ignore_idx
        assert roi_method in ROI_SELECT, roi_method
        self.roi_method = roi_method
        assert 0. < p_min_area_roi < 1., p_min_area_roi
        self.p_min_area_roi = p_min_area_roi
        self.use_roi = use_roi
        self.rng_parity = rng_parity

    def set_seed_tech(self, seed_tech):
        assert seed_tech in SEED_TECHS, seed_tech
        self.seed_tech = seed_tech

    # -- helpers -----------------------------------------------------------------------------------
    def _erode(self, roi: torch.Tensor) -> torch.Tensor:
        """fg_erode_iter flat erosions of a binary map [B,1,H,W] (kornia.morphology.erosion with a ones
        kernel and the geodesic border = min over the part of the window that lies inside the image)."""
        if self.fg_erode_iter == 0:
            return roi
        assert self.fg_erode_k > 1
        k = self.fg_erode_k
        o = k // 2
        out = roi.float()
        for _ in range(self.fg_erode_iter):
            padded = F.pad(-out, (o, k - o - 1, o, k - o - 1), value=float('-inf'))
            out = -F.max_pool2d(padded, kernel_size=k, stride=1)
        return out.to(roi.dtype)

    def _candidate_counts(self, x: torch.Tensor, roi: Optional[torch.Tensor]) -> Tuple[np.ndarray, np.ndarray]:
        """Per-sample numbers of fg / bg candidates, computed like the reference (one host sync)."""
        b, _, h, w = x.shape
        flat = x.reshape(b, -1)
        degenerate = (flat.amin(dim=1) == flat.amax(dim=1)).long()       # tcam_seeding.py:465
        if roi is not None:
            stats = torch.stack([degenerate, roi.reshape(b, -1).sum(dim=1).long()], dim=1).cpu().numpy()
        else:
            stats = torch.stack([degenerate, torch.zeros_like(degenerate)], dim=1).cpu().numpy()
        n_bg = int(self.min_p * h * w)                                    # tcam_seeding.py:567
        counts = np.zeros((b, 2), dtype=np.int32)
        for i in range(b):
            if stats[i, 0]:
                continue                                                   # flat CAM: no seeds at all
            if roi is not None:
                # int(max_p * roi.sum()): a python float times a 0-dim long tensor is a float32 product
                n_fg = int(np.float32(self.max_p) * np.float32(stats[i, 1]))   # tcam_seeding.py:510,519
            else:
                n_fg = int(self.max_p * (h * w))                          # tcam_seeding.py:515,519
            counts[i, 0] = n_fg if self.max_ > 0 else 0
            counts[i, 1] = n_bg if self.min_ > 0 else 0
        return counts, stats

    def _candidate_counts_device(self, x: torch.Tensor, roi: Optional[torch.Tensor]) -> torch.Tensor:
        """The same counts as _candidate_counts, as an int32 [B,2] tensor that never leaves the GPU (no host sync).
        Only usable when the draws need not line up with the reference's random stream (rng_parity=False)."""
        b, _, h, w = x.shape
        flat = x.reshape(b, -1)
        alive = flat.amin(dim=1) != flat.amax(dim=1)                     # tcam_seeding.py:465
        if roi is not None:
            # int(max_p * roi.sum()): float32 product, truncated (tcam_seeding.py:510,519)
            n_fg = (roi.reshape(b, -1).sum(dim=1).float() * float(np.float32(self.max_p))).to(torch.int32)
        else:
            n_fg = torch.full((b,), int(self.max_p * (h * w)), dtype=torch.int32, device=x.device)
        n_bg = torch.full((b,), int(self.min_p * h * w), dtype=torch.int32, device=x.device)
        if self.max_ <= 0:
            n_fg = torch.zeros_like(n_fg)
        if self.min_ <= 0:
            n_bg = torch.zeros_like(n_bg)
        return (torch.stack([n_fg, n_bg], dim=1) * alive.to(torch.int32).unsqueeze(1)).contiguous()

    def _draws(self, counts: np.ndarray, device: torch.device) -> Tuple[torch.Tensor, np.ndarray]:
        offsets = np.zeros_like(counts)
        total = 0
        for i in range(counts.shape[0]):
            for c in range(2):
                offsets[i, c] = total
                total += int(counts[i, c])
        q = torch.empty(max(total, 1), dtype=torch.float32, device=device)
        if total == 0:
            return q, offsets
        if self.rng_parity:
            # same sizes, same order as the reference's multinomial calls (fg then bg, sample by sample)
            for i in range(counts.shape[0]):
                for c in range(2):
                    n = int(counts[i, c])
                    if n > 0:
                        q[offsets[i, c]:offsets[i, c] + n].exponential_(1)
        else:
            q.exponential_(1)
        return q, offsets

    def _select(self, cams: torch.Tensor, roi: Optional[torch.Tensor], counts, sparse: bool = False):
        """cams [B,T,H,W] float32 CUDA -> (labels [B,H,W] long, cam_max [B,H,W]).  counts: numpy [B,2] (draws sized and
        ordered like the reference's multinomial calls) or None (no host round trip: counts and draws are made by the
        kernel)."""
        lib = _lib.load()
        b, t, h, w = cams.shape
        device = cams.device
        kmax = max(self.max_, self.min_, 1)
        with torch.cuda.device(device):
            fused = bool(lib.tcam_seed_fused_supported(h * w, kmax))   # answers for the current device
            n_fg_fixed = int(self.max_p * (h * w)) if self.max_ > 0 else 0       # tcam_seeding.py:515,519
            n_bg = int(self.min_p * h * w) if self.min_ > 0 else 0                # tcam_seeding.py:567
            rng = q = q_off = n_cand = None
            if counts is None and fused:
                # two words from torch's CUDA generator key the in-kernel Philox stream of this call
                rng = torch.randint(0, 2 ** 31 - 1, (2,), dtype=torch.int32, device=device)
            else:
                if counts is None:
                    counts_t = self._candidate_counts_device(cams.amax(dim=1, keepdim=True) if t > 1 else cams, roi)
                    q = torch.empty(b * 2 * h * w, dtype=torch.float32, device=device).exponential_(1)
                    q_off = torch.arange(2 * b, dtype=torch.int32, device=device) * (h * w)
                    n_cand = counts_t.reshape(-1)
                else:
                    q, offsets = self._draws(counts, device)
                    meta = torch.from_numpy(np.concatenate([offsets.reshape(-1), counts.reshape(-1)]).astype(np.int32)).to(device)
                    q_off, n_cand = meta[: 2 * b], meta[2 * b:]
            cam_max = torch.empty((b, h, w), dtype=torch.float32, device=device)
            sel = torch.empty((b, 2, kmax), dtype=torch.int32, device=device)
            out = None if sparse else torch.empty((b, h, w), dtype=torch.long, device=device)
            stream = torch.cuda.current_stream(device).cuda_stream
            if fused:
                _lib.check(lib.tcam_seed_fused(
                    cams.data_ptr(), t, roi.data_ptr() if roi is not None else None,
                    q.data_ptr() if q is not None else None, q_off.data_ptr() if q is not None else None,
                    n_cand.data_ptr() if n_cand is not None else None, rng.data_ptr() if rng is not None else None,
                    float(np.float32(self.max_p)), n_fg_fixed, n_bg, self.max_, self.min_,
                    1 if self.seed_tech == SEED_WEIGHTED else 0, b, h, w, self.ksz, int(self.ignore_idx),
                    cam_max.data_ptr(), sel.data_ptr(), kmax, out.data_ptr() if out is not None else None, stream),
                    'tcam_seed_fused')
            else:
                scratch = torch.empty((b, 2, h * w), dtype=torch.float32, device=device)
                _lib.check(lib.tcam_seed_select(cams.data_ptr(), t, roi.data_ptr() if roi is not None else None,
                                                q.data_ptr(), q_off.data_ptr(), n_cand.data_ptr(), self.max_, self.min_,
                                                1 if self.seed_tech == SEED_WEIGHTED else 0, b, h * w,
                                                cam_max.data_ptr(), scratch.data_ptr(), sel.data_ptr(), kmax, stream),
                           'tcam_seed_select')
                if out is not None:
                    _lib.check(lib.tcam_seed_labels(sel.data_ptr(), kmax, b, h, w, self.ksz, int(self.ignore_idx),
                                                    out.data_ptr(), stream), 'tcam_seed_labels')
        self._last_sel = sel
        if sparse:
            return SparseSeeds(sel, self.ksz, int(self.ignore_idx), h, w), cam_max
        return out, cam_max

    def _prep(self, x: torch.Tensor, roi: Optional[torch.Tensor]):
        assert isinstance(x, torch.Tensor)
        assert x.ndim == 4
        if not x.is_cuda:
            raise _lib.TcamCrfError('TCAMSeeder needs CUDA tensors: this package has no CPU path')
        if roi is not None:
            assert torch.is_tensor(roi)
            assert roi.ndim == 4  # b, 1, h, w
            assert roi.shape[0] == x.shape[0], f'{roi.shape[0]}, {x.shape[0]}'
            assert roi.shape[1] == 1, roi.shape[1]
            assert roi.shape[2:] == x.shape[2:]
        if self.ksz < 1:
            raise ValueError
        _roi = None
        if self.use_roi:
            if roi is None:
                # the reference falls back to GetRoiSingleCam on the CPU here (tcam_seeding.py:476-479)
                if self.roi_method == ROI_ALL:
                    roi, _ = ops.otsu_roi(x)
                else:
                    roi, _, _ = ops.roi_components(x, self.roi_method == ROI_LARGEST, self.p_min_area_roi)
            _roi = self._erode(roi.to(x.device)).long().contiguous()
        return x.detach().float().contiguous(), _roi

    # -- reference API -----------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, roi: torch.Tensor = None, sparse: bool = False):
        """``sparse=True`` (extension): return the ``SparseSeeds`` instead of painting the [B,H,W] label map."""
        x, _roi = self._prep(x, roi)
        b, d, h, w = x.shape
        assert d == 1, d  # todo multilabel.
        counts = self._candidate_counts(x, _roi)[0] if self.rng_parity else None
        out, _ = self._select(x, _roi, counts, sparse=sparse)
        return out if sparse else out.detach()

    def forward_stack(self, cams: torch.Tensor, roi: torch.Tensor = None, sparse: bool = False):
        """Fused temporal max + seeding: cams [B,T,H,W] (current frame and its neighbours' CAMs at the same
        resolution).  Returns (seeds [B,H,W] long, cam_max [B,H,W]); identical to
        ``forward(cams.max-chain over T)`` (dlib/datasets/wsol_loader.py:591-600 followed by TCAMSeeder)."""
        assert cams.ndim == 4
        cams = cams.detach().float().contiguous()
        if self.rng_parity:
            # the draws must be sized like the reference's multinomial calls: the counts go through the host
            x_max, _roi = self._prep(ops.temporal_cam_max(cams).unsqueeze(1), roi)
            counts = self._candidate_counts(x_max, _roi)[0]
        else:
            counts = None
            if self.use_roi and roi is None:   # the ROI is computed from the temporal max
                _, _roi = self._prep(ops.temporal_cam_max(cams).unsqueeze(1), None)
            elif self.use_roi:
                assert torch.is_tensor(roi) and roi.ndim == 4 and roi.shape[1] == 1
                assert roi.shape[0] == cams.shape[0] and roi.shape[2:] == cams.shape[2:]
                _roi = self._erode(roi.to(cams.device)).long().contiguous()
            else:
                _roi = None
        out, cam_max = self._select(cams, _roi, counts, sparse=sparse)
        return (out if sparse else out.detach()), cam_max

    def use_all_roi(self, x: torch.Tensor, roi: torch.Tensor = None) -> torch.Tensor:
        """Every roi pixel becomes foreground, everything else ignore (tcam_seeding.py:258-299)."""
        assert isinstance(x, torch.Tensor)
        assert x.ndim == 4
        assert roi is not None
        assert roi.ndim == 4
        assert roi.shape[0] == x.shape[0] and roi.shape[1] == 1 and roi.shape[2:] == x.shape[2:]
        b, d, h, w = x.shape
        assert d == 1, d
        out = torch.zeros((b, h, w), dtype=torch.long, requires_grad=False, device=x.device) + self.ignore_idx
        out[roi.squeeze(1) == 1] = 1
        return out.detach()

    def extra_repr(self):
        return f'min_={self.min_}, max_={self.max_}, min_p={self.min_p},' \
               f'max_p={self.max_p}, ksz={self.ksz}, fg_erode_k: ' \
               f'{self.fg_erode_k}, fg_erode_iter: {self.fg_erode_iter}' \
               f'support_background={self.support_background},' \
               f'multi_label_flag={self.multi_label_flag}, ' \
               f'seg_ignore_idx={self.ignore_idx}, seed_tech={self.seed_tech}'


class GetRoiSingleCam(object):
    """ROI of ONE cam [H,W] (dlib/cams/tcam_seeding.py:316-430) on the GPU: Otsu threshold (or `thresh` in [0,1]),
    then the whole thresholded map ('roi_all') or one connected component ('roi_high_density', 'largest').
    Returns (final_roi long [H,W], bbox_mask float [H,W], bbox float [1,4] = x0,y0,x1,y1) on the cam's device
    (the reference returns CPU tensors).  For a batch use ops.otsu_roi / ops.roi_components directly."""

    def __init__(self, roi_method: str, p_min_area_roi: float):
        assert roi_method in ROI_SELECT, roi_method
        self.roi_method = roi_method
        assert 0 < p_min_area_roi < 1., p_min_area_roi
        self.p_min_area_roi = p_min_area_roi

    def __call__(self, cam: torch.Tensor, thresh: float = None):
        assert torch.is_tensor(cam)
        assert cam.ndim == 2, cam.ndim
        if not cam.is_cuda:
            raise _lib.TcamCrfError('GetRoiSingleCam needs a CUDA tensor: this package has no CPU path')
        h, w = cam.shape
        x = cam.detach().float().reshape(1, h, w)
        if self.roi_method == ROI_ALL:
            if thresh is None:
                roi, _ = ops.otsu_roi(x)
            else:
                assert thresh >= 0, thresh
                roi = ((x * 255.) >= torch.tensor(thresh * 255., dtype=torch.float32, device=x.device)).long()
            # "not used" box of the reference: [0, 0, h - 1, w - 1] read back as x0, y0, x1, y1 (tcam_seeding.py:345,408)
            bbox = torch.tensor([[0, 0, h - 1, w - 1]], dtype=torch.float32, device=x.device)
            mask = torch.zeros((h, w), dtype=torch.float32, device=x.device)
            mask[0:w - 1, 0:h - 1] = 1.
            return roi[0], mask, bbox
        roi, mask, bbox = ops.roi_components(x, self.roi_method == ROI_LARGEST, self.p_min_area_roi, thresh)
        return roi[0], mask[0], bbox.reshape(1, 4)

    @staticmethod
    def get_thresh(cam: torch.Tensor) -> float:
        """Otsu threshold on floor(cam*255), 0 for a flat cam (tcam_seeding.py:419-430); in [0, 255]."""
        _, th = ops.otsu_roi(cam.detach().float().reshape(1, *cam.shape[-2:]))
        return float(th.item())
