"""DenseCRFLoss -- drop-in for ``dlib/crf/dense_crf_loss.py`` of the reference.

Same constructor, same ``forward(images, segmentations)`` keywords, same ``extra_repr``,
same value and gradient (``loss = -sum(S*AS)/N``, ``dS = -2*g*AS/N``,
dense_crf_loss.py:63-74), but the bilateral filter runs on the GPU through
``libtcamcrf.so`` instead of the SWIG/OpenMP C++ module, with no device synchronisation
and no device->host->device round trip of the segmentations.

``images`` may be what the reference's trainer passes (a CPU float32 tensor holding 0..255,
train_wsol.py:1128) or, to skip the host copy, a CUDA float32 / uint8 tensor.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function

from . import _lib, ops

__all__ = ['DenseCRFLoss', 'DenseCRFLossFunction', 'DenseCRFLossFromLogits', 'DenseCRFLossFromLogitsFunction',
           'SeedCrossEntropyFunction', 'CrfAndSeedCEFromLogitsFunction']


def _scale_images(images: torch.Tensor, scale_factor: float) -> torch.Tensor:
    if scale_factor == 1.0:
        return images  # nearest-neighbour resampling at scale 1 is the identity
    x = images if images.is_floating_point() else images.float()
    return F.interpolate(x, scale_factor=scale_factor, mode='nearest', recompute_scale_factor=False)


def _scale_segs(segmentations: torch.Tensor, scale_factor: float) -> torch.Tensor:
    if scale_factor == 1.0:
        return segmentations
    return F.interpolate(segmentations, scale_factor=scale_factor, mode='bilinear',
                         recompute_scale_factor=False, align_corners=False)


def _folded_weight(weight):
    """The module's weight as a python float when it can be folded into the loss kernels (cfg.loss_weight and the
    weighted backward: same two roundings as ``weight * loss`` and its autograd backward, three launches less per
    step), else None (tensor weights, zero): the caller then multiplies like the reference does."""
    if isinstance(weight, bool) or not isinstance(weight, (int, float)):
        return None
    w = float(weight)
    if w == 0.0 or w != w or w in (float('inf'), float('-inf')):
        return None
    return w


class DenseCRFLossFunction(Function):

    @staticmethod
    @torch.amp.custom_fwd(device_type='cuda')
    def forward(ctx, images, segmentations, sigma_rgb, sigma_xy, exact_gradient=False, weight=1.0, batch_size=None):
        # the reference divides by the local batch (dense_crf_loss.py:64); `batch_size` replaces it (a shard of a
        # larger batch reports its share of the global mean, dist.ShardedCRFLoss)
        n = segmentations.shape[0] if batch_size is None else batch_size
        cfg = _lib.make_config(ops.FEAT_XY_RGB, 3, sigma_rgb, sigma_xy, loss_weight=weight)
        _lib.require_key_range(cfg, segmentations.shape[2], segmentations.shape[3])
        ctx.N = n
        ctx.weight = float(weight)
        ctx.exact = bool(exact_gradient)
        if ctx.exact and segmentations.shape[0] <= ops.lattice_capacity(cfg, segmentations.shape[1],
                                                                         *segmentations.shape[2:]):
            # keep the lattice: the backward pass runs the transposed filter on it (blur axes in reverse order)
            ctx.lattice = ops.Lattice(images, cfg, segmentations.shape[1], device=segmentations.device)
            ctx.segs = segmentations.detach()
            ctx.AS, loss = ctx.lattice.apply(ctx.segs, want_loss=True, n_norm=float(n))
            return loss
        as_t, loss, _ = ops.crf_forward(images, segmentations.detach(), cfg, want_loss=True, n_norm=float(n))
        ctx.AS = as_t
        if ctx.exact:   # more frames than one lattice holds: the backward pass rebuilds it
            ctx.lattice = None
            ctx.images = images
            ctx.segs = segmentations.detach()
            ctx.sigmas = (sigma_rgb, sigma_xy)
        return loss

    @staticmethod
    @torch.amp.custom_bwd(device_type='cuda')
    def backward(ctx, grad_output):
        if ctx.exact:
            # d/dS [-S.(A S)/N] = -(A + A^T) S / N.  The reference uses -2 A S / N (dense_crf_loss.py:73), which is
            # exact only for a symmetric A; the blur axes are applied in a fixed order, so A != A^T in general.
            if ctx.lattice is not None:
                ats = ctx.lattice.apply(ctx.segs, transposed=True)
                ctx.lattice = None   # releases the workspace
            else:
                cfg = _lib.make_config(ops.FEAT_XY_RGB, 3, ctx.sigmas[0], ctx.sigmas[1])
                ats = ops.crf_filter_transposed(ctx.images, ctx.segs, cfg)
            grad_segmentation = ops.crf_backward((ctx.AS + ats) * 0.5, grad_output, float(ctx.N), ctx.weight)
        else:
            grad_segmentation = ops.crf_backward(ctx.AS, grad_output, float(ctx.N), ctx.weight)
        return None, grad_segmentation, None, None, None, None, None


class DenseCRFLoss(nn.Module):
    def __init__(self, weight, sigma_rgb, sigma_xy, scale_factor, exact_gradient=False):
        """
        :param weight: float. lambda of the CRF loss.
        :param sigma_rgb: float. colour bandwidth of the bilateral kernel.
        :param sigma_xy: float. spatial bandwidth of the bilateral kernel.
        :param scale_factor: float. images and segmentations are rescaled by it first.
        :param exact_gradient: bool, extension, OFF by default (reference behaviour: grad = -2*g*AS/N).  When on,
            the backward pass runs the transposed filter and returns the true gradient -g*(A + A^T)S/N.
        """
        super(DenseCRFLoss, self).__init__()
        self.weight = weight
        self.sigma_rgb = sigma_rgb
        self.sigma_xy = sigma_xy
        self.scale_factor = scale_factor
        self.exact_gradient = exact_gradient

    accepts_batch_size = True   # forward(..., batch_size=): see dist.ShardedCRFLoss

    def forward(self, images, segmentations, batch_size=None):
        """
        :param images: N*3*H*W tensor with values in [0, 255]; CPU float32 (as in the reference) or CUDA float32/uint8.
        :param segmentations: softmaxed logits, N*K*H*W, CUDA.
        :param batch_size: extension, None by default (reference behaviour: divide by N).  The batch size the sum is
            divided by when these N frames are a shard of a larger batch.
        :return: loss tensor of shape [1] on segmentations.device.
        """
        scaled_images = _scale_images(images, self.scale_factor)
        scaled_segs = _scale_segs(segmentations, self.scale_factor)
        w = _folded_weight(self.weight)
        if w is not None:   # weight * loss formed inside the loss kernels (same roundings, no extra launches)
            return DenseCRFLossFunction.apply(
                scaled_images, scaled_segs, self.sigma_rgb, self.sigma_xy * self.scale_factor, self.exact_gradient, w,
                batch_size)
        val = self.weight * DenseCRFLossFunction.apply(
            scaled_images, scaled_segs, self.sigma_rgb, self.sigma_xy * self.scale_factor, self.exact_gradient, 1.0,
            batch_size)
        return val

    def extra_repr(self):
        return 'sigma_rgb={}, sigma_xy={}, weight={}, scale_factor={}'.format(
            self.sigma_rgb, self.sigma_xy, self.weight, self.scale_factor
        )


class DenseCRFLossFromLogitsFunction(Function):
    """``DenseCRFLossFunction`` applied to ``softmax(logits, dim=1)`` with the softmax (forward and backward)
    fused into the CRF kernels -- the probabilities are never written to memory (SURVEY.md §8f.1).

    float16 and bfloat16 logits (what a model run under autocast produces) are read as they are and get their
    gradient in their own dtype: no float32 copy, no cast of the gradient.  The computation is float32 throughout, so
    the gradient has the bits of the float32 path on the widened logits cast back.  Other dtypes are cast to float32
    (ops.library_logits); this holds for the three logits Functions below."""

    @staticmethod
    @torch.amp.custom_fwd(device_type='cuda')
    def forward(ctx, images, logits, sigma_rgb, sigma_xy, weight=1.0):
        n = logits.shape[0]
        cfg = _lib.make_config(ops.FEAT_XY_RGB, 3, sigma_rgb, sigma_xy, loss_weight=weight)
        _lib.require_key_range(cfg, logits.shape[2], logits.shape[3])
        logits = ops.library_logits(logits.detach())
        as_t, loss, _ = ops.crf_forward_logits(images, logits, cfg, n_norm=float(n))
        ctx.AS = as_t
        ctx.logits = logits
        ctx.N = n
        ctx.weight = float(weight)
        return loss

    @staticmethod
    @torch.amp.custom_bwd(device_type='cuda')
    def backward(ctx, grad_output):
        return (None, ops.crf_backward_logits(ctx.AS, ctx.logits, grad_output, float(ctx.N), ctx.weight), None, None,
                None)


class DenseCRFLossFromLogits(nn.Module):
    """Same value and gradient as ``DenseCRFLoss(...)(images, F.softmax(logits, dim=1))`` (what
    ``ConRanFieldTcams.forward`` computes, dlib/losses/tcam.py:109-115) without materialising the softmax.
    Only for ``scale_factor == 1`` (the reference rescales the probabilities, not the logits) and K >= 2."""

    def __init__(self, weight, sigma_rgb, sigma_xy, scale_factor=1.0):
        super(DenseCRFLossFromLogits, self).__init__()
        if scale_factor != 1.0:
            raise ValueError('DenseCRFLossFromLogits supports scale_factor == 1 only')
        self.weight = weight
        self.sigma_rgb = sigma_rgb
        self.sigma_xy = sigma_xy
        self.scale_factor = scale_factor

    def forward(self, images, logits):
        w = _folded_weight(self.weight)
        if w is not None:
            return DenseCRFLossFromLogitsFunction.apply(images, logits, self.sigma_rgb, self.sigma_xy, w)
        return self.weight * DenseCRFLossFromLogitsFunction.apply(images, logits, self.sigma_rgb, self.sigma_xy)

    def extra_repr(self):
        return 'sigma_rgb={}, sigma_xy={}, weight={}, scale_factor={}, fused_softmax=True'.format(
            self.sigma_rgb, self.sigma_xy, self.weight, self.scale_factor
        )


class SeedCrossEntropyFunction(Function):
    """``F.cross_entropy(logits, seeds, ignore_index=ignore)`` for seeds given as ``SparseSeeds`` (tcam_seeding.py): the
    loss and its gradient come from the labelled pixels alone (csrc/seed.cuh, seed_ce_*_kernel)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type='cuda')
    def forward(ctx, logits, sel, ksz):
        logits = ops.library_logits(logits.detach())
        loss, count, _ = ops.seed_ce_forward(logits, sel, ksz)
        ctx.logits, ctx.sel, ctx.ksz, ctx.count = logits, sel, int(ksz), count
        return loss

    @staticmethod
    @torch.amp.custom_bwd(device_type='cuda')
    def backward(ctx, grad_output):
        grad = torch.zeros_like(ctx.logits)
        ops.seed_ce_backward_(grad, ctx.logits, ctx.sel, ctx.ksz, ctx.count, grad_output)
        return grad, None, None


class CrfAndSeedCEFromLogitsFunction(Function):
    """``crf_weight * DenseCRFLoss(softmax(logits)) + ce_weight * cross_entropy(logits, seeds)`` as ONE autograd node:
    the two terms of TCAM's loss that read the decoder's logits (dlib/losses/tcam.py:48-115).  The backward pass writes
    the CRF gradient through the softmax (one kernel) and adds the cross-entropy's on the handful of labelled pixels
    in place -- no second dense gradient, no accumulation pass.  Returns (total, crf term, unweighted cross-entropy);
    only the total carries a gradient."""

    @staticmethod
    @torch.amp.custom_fwd(device_type='cuda')
    def forward(ctx, images, logits, sigma_rgb, sigma_xy, crf_weight, sel, ksz, ce_weight):
        n = logits.shape[0]
        cfg = _lib.make_config(ops.FEAT_XY_RGB, 3, sigma_rgb, sigma_xy, loss_weight=crf_weight)
        _lib.require_key_range(cfg, logits.shape[2], logits.shape[3])
        logits = ops.library_logits(logits.detach())
        as_t, crf_loss, _ = ops.crf_forward_logits(images, logits, cfg, n_norm=float(n))
        # the kernel that finishes the cross-entropy also forms total = crf + ce_weight * ce: no torch glue launches
        ce_loss, count, total = ops.seed_ce_forward(logits, sel, ksz, add=crf_loss, weight=float(ce_weight))
        ctx.AS, ctx.logits, ctx.N = as_t, logits, n
        ctx.crf_weight, ctx.ce_weight = float(crf_weight), float(ce_weight)
        ctx.sel, ctx.ksz, ctx.count = sel, int(ksz), count
        ctx.mark_non_differentiable(crf_loss, ce_loss)
        return total, crf_loss, ce_loss

    @staticmethod
    @torch.amp.custom_bwd(device_type='cuda')
    def backward(ctx, grad_total, _g_crf, _g_ce):
        grad = ops.crf_seed_ce_backward(ctx.AS, ctx.logits, ctx.sel, ctx.ksz, ctx.count, grad_total, float(ctx.N),
                                        ctx.crf_weight, ctx.ce_weight)
        return None, grad, None, None, None, None, None, None
