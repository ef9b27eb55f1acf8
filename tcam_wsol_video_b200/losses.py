"""The loss-side callers of the CRF op, mirroring ``dlib/losses/tcam.py`` / ``dlib/losses/core.py``.

Only what sits on the hot path (SURVEY.md §8 a12, a13, a19): ``ConRanFieldTcams`` (5-D DenseCRF loss on
softmax(fcams)), ``RgbJointConRanFieldTcams`` (colour-only lattice over the width-concatenated frames of each
clip) and ``SelfLearningTcams`` (cross-entropy on the seeds; plain torch, it only consumes the seeder's
output).  ``ElementaryLoss`` keeps the reference's epoch gating and naming so ``MasterLoss``-style code can
hold these objects unchanged.
"""
from __future__ import annotations

import re
from typing import List, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .color_dense_crf_loss import ColorDenseCRFLoss
from .dense_crf_loss import (CrfAndSeedCEFromLogitsFunction, DenseCRFLoss, DenseCRFLossFromLogits,
                             SeedCrossEntropyFunction, _folded_weight)
from .tcam_seeding import SparseSeeds

__all__ = ['ElementaryLoss', 'ConRanFieldTcams', 'RgbJointConRanFieldTcams', 'SelfLearningTcams', 'FusedTcamLosses',
           'group_ordered_frames']


def group_ordered_frames(seq_iter: torch.Tensor, frm_iter: torch.Tensor) -> List[List[int]]:
    """Indices of the batch grouped by clip (``seq_iter``) and ordered by frame number (``frm_iter``);
    dlib/losses/tcam.py:32-45.  Done on the host in one transfer instead of one ``nonzero`` per clip."""
    seq = seq_iter.detach().cpu().tolist()
    frm = frm_iter.detach().cpu().tolist()
    groups = {}
    for i, s in enumerate(seq):
        groups.setdefault(s, []).append(i)
    out = []
    for s in sorted(groups):
        out.append(sorted(groups[s], key=lambda i: frm[i]))   # sorted() is stable, like the reference's
    return out


def _probabilities(fcams: torch.Tensor) -> torch.Tensor:
    """softmax over classes, or (1-sigmoid, sigmoid) for a single-channel map (tcam.py:109-113)."""
    if fcams.shape[1] > 1:
        return F.softmax(fcams, dim=1)
    p = torch.sigmoid(fcams)
    return torch.cat((1. - p, p), dim=1)


class ElementaryLoss(nn.Module):
    """dlib/losses/core.py:21-120: holds lambda, the CRF bandwidths and the epoch window of a loss term."""

    def __init__(self, cuda_id, name=None, lambda_=1., elb=None, support_background=False, multi_label_flag=False,
                 sigma_rgb=15., sigma_xy=100., scale_factor=0.5, start_epoch=None, end_epoch=None,
                 seg_ignore_idx=-255):
        super(ElementaryLoss, self).__init__()
        self._name = name
        self.lambda_ = lambda_
        self.elb = elb if elb is not None else nn.Identity()
        self.support_background = support_background
        assert not multi_label_flag
        self.multi_label_flag = multi_label_flag
        self.sigma_rgb = sigma_rgb
        self.sigma_xy = sigma_xy
        self.scale_factor = scale_factor
        if end_epoch == -1:
            end_epoch = None
        self.start_epoch = start_epoch
        self.end_epoch = end_epoch
        self.c_epoch = 0
        self.loss = None
        self._device = torch.device('cuda', cuda_id) if isinstance(cuda_id, int) else torch.device(cuda_id)
        self._zero = torch.tensor([0.0], device=self._device, requires_grad=False, dtype=torch.float)
        self.seg_ignore_idx = seg_ignore_idx

    def is_on(self, _epoch=None):
        c_epoch = self.c_epoch if _epoch is None else _epoch
        if (self.start_epoch is None) and (self.end_epoch is None):
            return True
        if all(isinstance(z, int) for z in (c_epoch, self.start_epoch, self.end_epoch)):
            return self.start_epoch <= c_epoch <= self.end_epoch
        if self.start_epoch is None and isinstance(self.end_epoch, int):
            return c_epoch <= self.end_epoch
        if isinstance(self.start_epoch, int) and self.end_epoch is None:
            return c_epoch >= self.start_epoch
        return False

    @property
    def __name__(self):
        if self._name is None:
            name = self.__class__.__name__
            s1 = re.sub('(.)([A-Z][a-z]+)', r'\1_\2', name)
            return re.sub('([a-z0-9])([A-Z])', r'\1_\2', s1).lower()
        return self._name

    def forward(self, epoch=0, **kwargs):
        self.c_epoch = epoch


def _check_seeds(seeds: SparseSeeds, fcams: torch.Tensor) -> None:
    """SparseSeeds label pixels by index: seeds made for other frames (another resolution or batch) would label the
    wrong pixels, where the reference's cross-entropy raises on the mismatched target."""
    if (seeds.h, seeds.w) != tuple(fcams.shape[2:]) or seeds.sel.shape[0] != fcams.shape[0]:
        raise ValueError(f'seeds were made for {seeds.sel.shape[0]} frames of {seeds.h}x{seeds.w}, the maps are '
                         f'{tuple(fcams.shape)}')


class SelfLearningTcams(ElementaryLoss):
    """Cross-entropy of the decoder's maps against the sampled seeds (tcam.py:48-77)."""

    def __init__(self, **kwargs):
        super(SelfLearningTcams, self).__init__(**kwargs)
        self.loss = nn.CrossEntropyLoss(reduction="mean", ignore_index=self.seg_ignore_idx).to(self._device)

    def forward(self, epoch=0, fcams=None, seeds=None, **kwargs):
        """``seeds``: the reference's [B,H,W] long map, or (extension) the seeder's ``SparseSeeds``: the same loss and
        gradient computed from the labelled pixels alone."""
        super(SelfLearningTcams, self).forward(epoch=epoch)
        if not self.is_on():
            return self._zero
        if isinstance(seeds, SparseSeeds):
            if seeds.ignore_idx != self.seg_ignore_idx:
                raise ValueError('seeds were made with another ignore index')
            _check_seeds(seeds, fcams)
            return SeedCrossEntropyFunction.apply(fcams, seeds.sel, seeds.ksz) * self.lambda_
        return self.loss(input=fcams, target=seeds) * self.lambda_


class ConRanFieldTcams(ElementaryLoss):
    """DenseCRF loss over the decoder's class probabilities (tcam.py:80-115)."""

    def __init__(self, fuse_softmax: bool = False, **kwargs):
        """``fuse_softmax=True`` (extension, off by default): the softmax over the classes and its backward run
        inside the CRF kernels (``DenseCRFLossFromLogits``); needs scale_factor == 1 and more than one channel,
        otherwise the unfused path is taken."""
        super(ConRanFieldTcams, self).__init__(**kwargs)
        self.loss = DenseCRFLoss(weight=self.lambda_, sigma_rgb=self.sigma_rgb, sigma_xy=self.sigma_xy,
                                 scale_factor=self.scale_factor).to(self._device)
        self.loss_from_logits = None
        if fuse_softmax and self.scale_factor == 1.0:
            self.loss_from_logits = DenseCRFLossFromLogits(weight=self.lambda_, sigma_rgb=self.sigma_rgb,
                                                           sigma_xy=self.sigma_xy, scale_factor=1.0).to(self._device)

    def forward(self, epoch=0, fcams=None, raw_img=None, **kwargs):
        super(ConRanFieldTcams, self).forward(epoch=epoch)
        if not self.is_on():
            return self._zero
        if self.loss_from_logits is not None and fcams.shape[1] > 1:
            return self.loss_from_logits(images=raw_img, logits=fcams)
        return self.loss(images=raw_img, segmentations=_probabilities(fcams))


class FusedTcamLosses(nn.Module):
    """``SelfLearningTcams`` + ``ConRanFieldTcams`` as one autograd node (extension; same value and gradient as the sum
    of the two modules, tests/test_gpu_losses.py::test_fused_tcam_losses).  Takes the two loss objects (their lambdas,
    bandwidths and epoch windows are honoured) and, per step, the decoder's logits, the raw frames and the seeder's
    ``SparseSeeds``.  Falls back to the separate modules whenever a term is off, the CRF rescales its inputs, the
    weights are not plain numbers or the maps have a single channel."""

    def __init__(self, self_learning: SelfLearningTcams, con_ran_field: ConRanFieldTcams):
        super(FusedTcamLosses, self).__init__()
        self.sl = self_learning
        self.crf = con_ran_field

    def forward(self, epoch=0, fcams=None, raw_img=None, seeds=None, **kwargs):
        self.sl.c_epoch = epoch
        self.crf.c_epoch = epoch
        w_crf, w_sl = _folded_weight(self.crf.lambda_), _folded_weight(self.sl.lambda_)
        fusable = (self.sl.is_on() and self.crf.is_on() and isinstance(seeds, SparseSeeds) and fcams.shape[1] > 1
                   and self.crf.scale_factor == 1.0 and w_crf is not None and w_sl is not None
                   and seeds.ignore_idx == self.sl.seg_ignore_idx)
        if not fusable:
            return self.sl(epoch=epoch, fcams=fcams, seeds=seeds) + self.crf(epoch=epoch, fcams=fcams, raw_img=raw_img)
        _check_seeds(seeds, fcams)
        total, self.last_crf, ce = CrfAndSeedCEFromLogitsFunction.apply(
            raw_img, fcams, self.crf.sigma_rgb, self.crf.sigma_xy, w_crf, seeds.sel, seeds.ksz, w_sl)
        self.last_ce = ce           # the unweighted cross-entropy; last_crf is the weighted CRF term (for logging)
        return total


class RgbJointConRanFieldTcams(ElementaryLoss):
    """Colour-only CRF that couples the frames of each clip (tcam.py:154-232).

    The reference concatenates the frames of one clip along the width and calls the colour filter once per
    clip in a Python loop, averaging over the clips.  The colour-only lattice has no position features, so
    all clips with the same number of frames go through ONE batched call here (one lattice per clip, built in
    the same launch); the mean over clips is unchanged."""

    def __init__(self, **kwargs):
        super(RgbJointConRanFieldTcams, self).__init__(**kwargs)
        self.loss = ColorDenseCRFLoss(weight=self.lambda_, sigma_rgb=self.sigma_rgb,
                                      scale_factor=self.scale_factor).to(self._device)

    def forward(self, epoch=0, fcams=None, raw_img=None, seq_iter=None, frm_iter=None, **kwargs):
        super(RgbJointConRanFieldTcams, self).forward(epoch=epoch)
        if not self.is_on():
            return self._zero
        fcams_n = _probabilities(fcams)
        clips = [item for item in group_ordered_frames(seq_iter, frm_iter) if len(item) >= 2]
        if not clips:
            return self._zero   # (the reference divides by zero here; tcam.py:204-205 "todo")
        by_len = {}
        for item in clips:
            by_len.setdefault(len(item), []).append(item)
        total = self._zero
        for t, items in by_len.items():
            imgs, cams = self.pair_clips(items, raw_img, fcams_n)
            # ColorDenseCRFLoss divides by its batch size (= number of clips in this group)
            total = total + self.loss(images=imgs, segmentations=cams) * float(len(items))
        return total / float(len(clips))

    @staticmethod
    def pair_clips(items: List[List[int]], imgs: torch.Tensor, prob_cams: torch.Tensor):
        """[len(items), C, H, T*W] tensors: frames of each clip side by side along the width (tcam.py:207-232)."""
        assert imgs.ndim == 4 and imgs.shape[1] == 3
        assert prob_cams.ndim == 4
        idx = torch.as_tensor(items, dtype=torch.long)                       # [clips, T]
        c, t = idx.shape
        gi = imgs[idx.reshape(-1).to(imgs.device)]                             # [c*t, 3, H, W]
        gp = prob_cams[idx.reshape(-1).to(prob_cams.device)]
        h, w = gi.shape[2:]
        gi = gi.view(c, t, gi.shape[1], h, w).permute(0, 2, 3, 1, 4).reshape(c, gi.shape[1], h, t * w)
        gp = gp.view(c, t, gp.shape[1], h, w).permute(0, 2, 3, 1, 4).reshape(c, gp.shape[1], h, t * w)
        return gi.contiguous(), gp.contiguous()

    @staticmethod
    def pair_samples(o_idx: list, imgs: torch.Tensor, prob_cams: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """One clip, the reference's signature (tcam.py:207-232)."""
        assert len(o_idx) > 1, len(o_idx)
        return RgbJointConRanFieldTcams.pair_clips([list(o_idx)], imgs, prob_cams)
