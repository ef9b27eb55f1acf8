"""torch-facing wrappers over the device API of libtcamcrf.so.

PyTorch is plumbing here: it owns device memory (inputs, outputs, workspace) and the
stream; all compute happens in the hand-written CUDA kernels behind the C ABI.
"""
from __future__ import annotations

import os
from ctypes import byref, c_int
from typing import Dict, Optional, Tuple

import torch

from . import _lib
from ._lib import FEAT_COLOR, FEAT_XY_RGB, TcamCrfError

_workspaces: Dict[Tuple[int, int], torch.Tensor] = {}

STRICT = os.environ.get("TCAMCRF_STRICT", "0") == "1"


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise TcamCrfError(f"{name} must be a CUDA tensor: this package has no CPU path")


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream_ptr(device))
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        # grow geometrically; the old buffer is released to torch's caching allocator (stream-safe)
        ws = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def release_workspaces() -> None:
    """Drops the cached per-(device, stream) buffers: the CRF workspaces and the seed cross-entropy scratch."""
    _workspaces.clear()
    _seed_ce_scratch.clear()


def _prep_images(images: torch.Tensor, device: torch.device) -> Tuple[torch.Tensor, bool]:
    """Bring the image batch onto `device` as contiguous float32 or uint8 [N,C,H,W]."""
    if images.dtype == torch.uint8:
        u8 = True
    else:
        u8 = False
        if images.dtype != torch.float32:
            images = images.float()
    if images.device != device:
        if images.device.type == 'cpu' and not images.is_pinned():
            _warn_pageable_once(images)
        images = images.to(device, non_blocking=True)
    return images.contiguous(), u8


_warned_pageable = False


def _warn_pageable_once(images: torch.Tensor) -> None:
    """Pageable host frames work (it is what the reference's trainer passes, train_wsol.py:1128) but the copy is
    staged by the driver and blocks the host; pinned uint8 frames take the overlapped path at a quarter of the
    bytes.  Said once per process."""
    global _warned_pageable
    if _warned_pageable:
        return
    _warned_pageable = True
    import warnings
    warnings.warn(
        "tcam_wsol_video_b200: images arrive in pageable host memory (%s, %.1f MB per call): the copy blocks the "
        "host and cannot overlap the lattice build.  Pin the loader's frames (DataLoader(pin_memory=True)) and keep "
        "them uint8 to take the overlapped path (tcamcrf_loss_forward_host_frames)."
        % (str(images.dtype).replace('torch.', ''), images.numel() * images.element_size() / 1e6),
        RuntimeWarning, stacklevel=4)


def _host_frames(images: torch.Tensor, device: torch.device) -> bool:
    """Frames the trainer left on the CPU (train_wsol.py:1128), in the layout the library copies from directly:
    float32 (or uint8), contiguous, pinned.  They take tcamcrf_loss_forward_host_frames (the copy overlaps the lattice build)."""
    return (images.device.type == 'cpu' and device.type == 'cuda' and images.dtype in (torch.float32, torch.uint8)
            and images.is_contiguous() and images.is_pinned() and images.numel() > 0)


_pending_host_frames = []   # (event, tensor): host frames whose asynchronous copy may still be in flight


def _keep_until_done(frames: torch.Tensor, device: torch.device) -> None:
    """torch does not know about the library's copy stream: hold a reference to the pinned tensor until the work
    queued behind the copy has completed, so the host allocator cannot hand its memory out again meanwhile."""
    if torch.cuda.is_current_stream_capturing():
        return   # a captured graph re-reads the tensor on every replay: its owner keeps it alive
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(device))
    _pending_host_frames.append((ev, frames))
    while _pending_host_frames and _pending_host_frames[0][0].query():
        _pending_host_frames.pop(0)


def workspace_status(ws: torch.Tensor) -> Tuple[int, int]:
    """(device status bits, vertex count of the last chunk); synchronises the stream."""
    lib = _lib.load()
    st, m = c_int(0), c_int(0)
    _lib.check(lib.tcamcrf_workspace_status(ws.data_ptr(), _stream_ptr(ws.device), byref(st), byref(m)),
               "tcamcrf_workspace_status")
    return st.value, m.value


def _raise_on_status(ws: torch.Tensor) -> None:
    st, _ = workspace_status(ws)
    if st:
        why = [n for b, n in ((1, "hash table full"), (2, "vertex pool full"), (4, "lattice coordinate out of key range")) if st & b]
        raise TcamCrfError("device status 0x%x: %s" % (st, ", ".join(why)))


def crf_forward(images: torch.Tensor, segs: torch.Tensor, cfg: _lib.Config, want_loss: bool = True,
                n_norm: Optional[float] = None, check: Optional[bool] = None):
    """Runs build+splat+blur+slice (and the loss reduction) on the current stream.

    images [N,C,H,W] float32 0..255 or uint8 (any device; moved to segs.device), segs [N,K,H,W] float32 CUDA.
    Returns (AS [N,K,H,W], loss [1] or None, workspace tensor).
    """
    lib = _lib.load()
    _require_cuda(segs, "segmentations")
    device = segs.device
    if segs.dtype != torch.float32:
        segs = segs.float()
    segs = segs.contiguous()
    n, k, h, w = segs.shape
    host_frames = images if _host_frames(images, device) else None
    if host_frames is not None:
        u8 = host_frames.dtype == torch.uint8
        with torch.cuda.device(device):
            images = torch.empty(host_frames.shape, dtype=host_frames.dtype, device=device)   # staging buffer
    else:
        images, u8 = _prep_images(images, device)
    if images.ndim != 4 or images.shape[0] != n or tuple(images.shape[2:]) != (h, w):
        raise TcamCrfError(f"images {tuple(images.shape)} do not match segmentations {tuple(segs.shape)}")
    if images.shape[1] < cfg.channels:
        raise TcamCrfError(f"images have {images.shape[1]} planes, config needs {cfg.channels}")
    cfg.image_stride_planes = images.shape[1]
    with torch.cuda.device(device):
        nbytes = lib.tcamcrf_workspace_bytes(byref(cfg), n, k, h, w)
        if nbytes == 0:
            raise TcamCrfError("tcamcrf_workspace_bytes: " + _lib.last_error())
        ws = _workspace(device, nbytes)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256
        ws_bytes = ws.numel() - (ws_ptr - ws.data_ptr())
        as_out = torch.empty_like(segs)
        stream = _stream_ptr(device)
        if host_frames is not None:
            loss = torch.empty(1, dtype=torch.float32, device=device) if want_loss else None
            rc = lib.tcamcrf_loss_forward_host_frames(
                byref(cfg), host_frames.data_ptr(), images.data_ptr(), 1 if u8 else 0, segs.data_ptr(),
                as_out.data_ptr(), loss.data_ptr() if want_loss else None, 0, n, k, h, w, float(n if n_norm is None else n_norm),
                ws_ptr, ws_bytes, stream)
            _keep_until_done(host_frames, device)
        elif want_loss:
            loss = torch.empty(1, dtype=torch.float32, device=device)
            fn = lib.tcamcrf_loss_forward_u8 if u8 else lib.tcamcrf_loss_forward
            rc = fn(byref(cfg), images.data_ptr(), segs.data_ptr(), as_out.data_ptr(), loss.data_ptr(), n, k, h, w,
                    float(n if n_norm is None else n_norm), ws_ptr, ws_bytes, stream)
        else:
            loss = None
            fn = lib.tcamcrf_filter_u8 if u8 else lib.tcamcrf_filter
            rc = fn(byref(cfg), images.data_ptr(), segs.data_ptr(), as_out.data_ptr(), n, k, h, w, ws_ptr, ws_bytes,
                    stream)
        _lib.check(rc, "tcamcrf forward")
        if STRICT if check is None else check:
            _raise_on_status(ws if ws_ptr == ws.data_ptr() else ws[ws_ptr - ws.data_ptr():])
    return as_out, loss, ws


def crf_filter_transposed(images: torch.Tensor, segs: torch.Tensor, cfg: _lib.Config) -> torch.Tensor:
    """A^T segs (blur axes in reverse order) on the current stream; see tcamcrf_filter_transposed."""
    lib = _lib.load()
    _require_cuda(segs, "segmentations")
    device = segs.device
    segs = segs.detach().float().contiguous()
    n, k, h, w = segs.shape
    images, u8 = _prep_images(images, device)
    cfg.image_stride_planes = images.shape[1]
    with torch.cuda.device(device):
        nbytes = lib.tcamcrf_workspace_bytes(byref(cfg), n, k, h, w)
        if nbytes == 0:
            raise TcamCrfError("tcamcrf_workspace_bytes: " + _lib.last_error())
        ws = _workspace(device, nbytes)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256
        out = torch.empty_like(segs)
        _lib.check(lib.tcamcrf_filter_transposed(byref(cfg), images.data_ptr(), 1 if u8 else 0, segs.data_ptr(),
                                                 out.data_ptr(), n, k, h, w, ws_ptr,
                                                 ws.numel() - (ws_ptr - ws.data_ptr()), _stream_ptr(device)),
                   "tcamcrf_filter_transposed")
    return out


def lattice_capacity(cfg: _lib.Config, k: int, h: int, w: int) -> int:
    """Most frames one lattice (one pass of the library) holds for this problem: 64 unless the frames are large."""
    cap = _lib.load().tcamcrf_chunk_frames(byref(cfg), 1 << 20, int(k), int(h), int(w))
    if cap <= 0:
        raise TcamCrfError("tcamcrf_chunk_frames: " + _lib.last_error())
    return cap


class Lattice:
    """The permutohedral lattice of a batch of frames, built once and applied many times.

    Owns its workspace (the lattice lives in it).  `apply(segs)` = A segs, `apply(segs, transposed=True)` = A^T segs
    (blur axes in reverse order).  Mirrors what the reference does per image inside bilateralfilter() -- one
    Permutohedral::init, K computes (bilateralfilter.cpp:28-37) -- and backs the exact-gradient backward and the
    mean-field iterations of DenseCRFFilter.  At most `lattice_capacity(...)` frames per lattice (64 unless large).
    """

    def __init__(self, images: torch.Tensor, cfg: _lib.Config, k: int, device: Optional[torch.device] = None):
        lib = _lib.load()
        device = torch.device(device) if device is not None else images.device
        if device.type != "cuda":
            raise TcamCrfError("Lattice needs a CUDA device: this package has no CPU path")
        images, u8 = _prep_images(images, device)
        if images.ndim != 4:
            raise TcamCrfError(f"images must be [N,C,H,W], got {tuple(images.shape)}")
        n, c, h, w = images.shape
        if c < cfg.channels:
            raise TcamCrfError(f"images have {c} planes, config needs {cfg.channels}")
        self.cfg = _lib.Config(cfg.feat, cfg.channels, c, cfg.sigma_rgb, cfg.sigma_xy, cfg.hash_load,
                               cfg.pool_factor, cfg.chunk_frames, cfg.loss_weight)
        self.shape = (n, int(k), h, w)
        self.device = device
        with torch.cuda.device(device):
            nbytes = lib.tcamcrf_workspace_bytes(byref(self.cfg), n, int(k), h, w)
            if nbytes == 0:
                raise TcamCrfError("tcamcrf_workspace_bytes: " + _lib.last_error())
            self._ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
            self._ws_ptr = (self._ws.data_ptr() + 255) // 256 * 256
            self._ws_bytes = self._ws.numel() - (self._ws_ptr - self._ws.data_ptr())
            _lib.check(lib.tcamcrf_lattice_build(byref(self.cfg), images.data_ptr(), 1 if u8 else 0, n, int(k), h, w,
                                                 self._ws_ptr, self._ws_bytes, _stream_ptr(device)),
                       "tcamcrf_lattice_build")
            # the build reads `images` asynchronously; tie their lifetime to this stream
            images.record_stream(torch.cuda.current_stream(device))

    def apply(self, segs: torch.Tensor, transposed: bool = False, want_loss: bool = False,
              n_norm: Optional[float] = None):
        """Returns A segs (or A^T segs); with want_loss also -sum(segs * out) / n_norm as a [1] tensor."""
        lib = _lib.load()
        _require_cuda(segs, "segmentations")
        if segs.device != self.device:
            raise TcamCrfError(f"segmentations on {segs.device}, lattice on {self.device}")
        if tuple(segs.shape) != self.shape:
            raise TcamCrfError(f"segmentations {tuple(segs.shape)} do not match the lattice {self.shape}")
        segs = segs.detach().float().contiguous()
        n, k, h, w = self.shape
        with torch.cuda.device(self.device):
            out = torch.empty_like(segs)
            loss = torch.empty(1, dtype=torch.float32, device=self.device) if want_loss else None
            _lib.check(lib.tcamcrf_lattice_apply(byref(self.cfg), segs.data_ptr(), out.data_ptr(),
                                                 loss.data_ptr() if want_loss else None, n, k, h, w,
                                                 float(n if n_norm is None else n_norm), 1 if transposed else 0,
                                                 self._ws_ptr, self._ws_bytes, _stream_ptr(self.device)),
                       "tcamcrf_lattice_apply")
        return (out, loss) if want_loss else out

    def status(self) -> Tuple[int, int]:
        """(device status bits, vertex count); synchronises the stream."""
        ws = self._ws if self._ws_ptr == self._ws.data_ptr() else self._ws[self._ws_ptr - self._ws.data_ptr():]
        return workspace_status(ws)


# logits the kernels read as they are (TCAMCRF_DTYPE_*): float32, and the two autocast dtypes
_LOGIT_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}


def library_logits(logits: torch.Tensor) -> torch.Tensor:
    """`logits` as the library reads them: float32, float16 and bfloat16 as they are (no copy when contiguous), any
    other dtype cast to float32; contiguous."""
    if logits.dtype not in _LOGIT_DTYPES:
        logits = logits.float()
    return logits.contiguous()


def _logits_code(logits: torch.Tensor) -> int:
    """TCAMCRF_DTYPE_* of logits about to be handed to the library: 4-D, contiguous, CUDA, of a dtype it reads."""
    _require_cuda(logits, "logits")
    if logits.ndim != 4:
        raise TcamCrfError(f"logits must be [B,K,H,W], got {tuple(logits.shape)}")
    if not logits.is_contiguous():
        raise TcamCrfError("logits must be contiguous")
    if logits.dtype not in _LOGIT_DTYPES:
        raise TcamCrfError(f"logits must be float32, float16 or bfloat16, got {logits.dtype}")
    return _LOGIT_DTYPES[logits.dtype]


def crf_forward_logits(images: torch.Tensor, logits: torch.Tensor, cfg: _lib.Config, n_norm: Optional[float] = None,
                       check: Optional[bool] = None):
    """Like crf_forward(want_loss=True) with segs = softmax(logits, dim=1) formed inside the kernels.
    float16 and bfloat16 logits are read as they are (see library_logits).  Returns (AS float32, loss [1], workspace)."""
    lib = _lib.load()
    _require_cuda(logits, "logits")
    device = logits.device
    logits = library_logits(logits)
    dtype = _logits_code(logits)
    n, k, h, w = logits.shape
    if k < 2:
        raise TcamCrfError("the fused softmax needs at least two classes")
    host_frames = images if _host_frames(images, device) else None
    if host_frames is not None:
        u8 = host_frames.dtype == torch.uint8
        with torch.cuda.device(device):
            images = torch.empty(host_frames.shape, dtype=host_frames.dtype, device=device)   # staging buffer
    else:
        images, u8 = _prep_images(images, device)
    if images.ndim != 4 or images.shape[0] != n or tuple(images.shape[2:]) != (h, w):
        raise TcamCrfError(f"images {tuple(images.shape)} do not match logits {tuple(logits.shape)}")
    if images.shape[1] < cfg.channels:
        raise TcamCrfError(f"images have {images.shape[1]} planes, config needs {cfg.channels}")
    cfg.image_stride_planes = images.shape[1]
    with torch.cuda.device(device):
        nbytes = lib.tcamcrf_workspace_bytes(byref(cfg), n, k, h, w)
        if nbytes == 0:
            raise TcamCrfError("tcamcrf_workspace_bytes: " + _lib.last_error())
        ws = _workspace(device, nbytes)
        ws_ptr = (ws.data_ptr() + 255) // 256 * 256
        ws_bytes = ws.numel() - (ws_ptr - ws.data_ptr())
        as_out = torch.empty(logits.shape, dtype=torch.float32, device=device)
        loss = torch.empty(1, dtype=torch.float32, device=device)
        if host_frames is not None:
            rc = lib.tcamcrf_loss_forward_host_frames_typed(
                byref(cfg), host_frames.data_ptr(), images.data_ptr(), 1 if u8 else 0, logits.data_ptr(), dtype,
                as_out.data_ptr(), loss.data_ptr(), n, k, h, w, float(n if n_norm is None else n_norm), ws_ptr, ws_bytes,
                _stream_ptr(device))
            _keep_until_done(host_frames, device)
        else:
            rc = lib.tcamcrf_loss_forward_logits_typed(byref(cfg), images.data_ptr(), 1 if u8 else 0, logits.data_ptr(),
                                                       dtype, as_out.data_ptr(), loss.data_ptr(), n, k, h, w,
                                                       float(n if n_norm is None else n_norm), ws_ptr, ws_bytes,
                                                       _stream_ptr(device))
        _lib.check(rc, "tcamcrf_loss_forward_logits")
        if STRICT if check is None else check:
            _raise_on_status(ws if ws_ptr == ws.data_ptr() else ws[ws_ptr - ws.data_ptr():])
    return as_out, loss, ws


def crf_backward_logits(as_t: torch.Tensor, logits: torch.Tensor, grad_output: torch.Tensor, n_norm: float,
                        weight: float = 1.0):
    """Gradient w.r.t. the logits (CRF gradient chained through the softmax) in one kernel; `weight`: the module's
    weight when it was folded into the forward (cfg.loss_weight).  The gradient has the dtype the library read the
    logits in (library_logits): float16 / bfloat16 logits get theirs, rounded once from the float32 value."""
    lib = _lib.load()
    _require_cuda(as_t, "AS")
    n, k, h, w = as_t.shape
    logits = library_logits(logits.detach())
    dtype = _logits_code(logits)
    _check_as(as_t, logits)
    g = grad_output.detach().reshape(-1)[:1].to(device=as_t.device, dtype=torch.float32).contiguous()
    grad = torch.empty_like(logits)
    with torch.cuda.device(as_t.device):
        _lib.check(lib.tcamcrf_loss_backward_logits_typed(as_t.data_ptr(), logits.data_ptr(), dtype, g.data_ptr(),
                                                          grad.data_ptr(), n, k, h, w, float(n_norm), float(weight),
                                                          _stream_ptr(as_t.device)),
                   "tcamcrf_loss_backward_logits_typed")
    return grad


def _check_as(as_t: torch.Tensor, logits: torch.Tensor) -> None:
    if as_t.dtype != torch.float32 or not as_t.is_contiguous() or as_t.shape != logits.shape or \
            as_t.device != logits.device:
        raise TcamCrfError(f"AS must be contiguous float32 {tuple(logits.shape)} on {logits.device}, got "
                           f"{as_t.dtype} {tuple(as_t.shape)} on {as_t.device}")


def crf_backward(as_t: torch.Tensor, grad_output: torch.Tensor, n_norm: float, weight: float = 1.0) -> torch.Tensor:
    """grad_seg = ((-2*(g*weight)) * AS) / n_norm on the current stream (dlib/crf/dense_crf_loss.py:73; `weight`: the
    module's weight when it was folded into the forward, cfg.loss_weight)."""
    lib = _lib.load()
    _require_cuda(as_t, "AS")
    g = grad_output.detach().reshape(-1)[:1].to(device=as_t.device, dtype=torch.float32).contiguous()
    grad = torch.empty_like(as_t)
    with torch.cuda.device(as_t.device):
        _lib.check(lib.tcamcrf_loss_backward_weighted(as_t.data_ptr(), g.data_ptr(), grad.data_ptr(), as_t.numel(),
                                                      float(n_norm), float(weight), _stream_ptr(as_t.device)),
                   "tcamcrf_loss_backward_weighted")
    return grad


_seed_ce_scratch: Dict[Tuple[int, int, int], torch.Tensor] = {}


def _check_seeds(logits: torch.Tensor, sel: torch.Tensor) -> None:
    """sel: the int32 [B,2,kmax] seeds of the B samples of `logits`, contiguous, on their device."""
    if sel.dtype != torch.int32 or sel.ndim != 3 or sel.shape[0] != logits.shape[0] or sel.shape[1] != 2 or \
            sel.shape[2] < 1 or sel.device != logits.device or not sel.is_contiguous():
        raise TcamCrfError(f"sel must be contiguous int32 [{logits.shape[0]},2,kmax] on {logits.device}, got "
                           f"{sel.dtype} {tuple(sel.shape)} on {sel.device}")


def seed_ce_forward(logits: torch.Tensor, sel: torch.Tensor, ksz: int, add: Optional[torch.Tensor] = None,
                    weight: float = 1.0):
    """Cross-entropy of `logits` [B,K,H,W] on the seeds `sel` [B,2,kmax] (see tcam_seed_ce_forward): returns
    (loss [1], count [1] float32 = labelled pixels, total [1] = add + weight * loss or None without `add`).
    float16 and bfloat16 logits are read as they are, other dtypes cast to float32 (library_logits); the results are
    float32."""
    lib = _lib.load()
    _require_cuda(logits, "logits")
    if logits.dtype not in _LOGIT_DTYPES:
        logits = logits.float()
    dtype = _logits_code(logits)
    _check_seeds(logits, sel)
    b, k, h, w = logits.shape
    device = logits.device
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream_ptr(device), b)
    scratch = _seed_ce_scratch.get(key)
    if scratch is None or torch.cuda.is_current_stream_capturing():
        scratch = torch.zeros(1 + 2 * b, dtype=torch.float32, device=device)    # ticket + per-sample partials
        if not torch.cuda.is_current_stream_capturing():
            _seed_ce_scratch[key] = scratch
    out = torch.empty(3, dtype=torch.float32, device=device)     # loss, count, total
    with torch.cuda.device(device):
        _lib.check(lib.tcam_seed_ce_forward_typed(logits.data_ptr(), dtype, sel.data_ptr(), int(sel.shape[2]), b, k, h,
                                                  w, int(ksz), scratch.data_ptr(), out.data_ptr(), out.data_ptr() + 4,
                                                  add.data_ptr() if add is not None else None, float(weight),
                                                  out.data_ptr() + 8 if add is not None else None, _stream_ptr(device)),
                   "tcam_seed_ce_forward")
    return out[0:1], out[1:2], (out[2:3] if add is not None else None)


def _check_grad(grad_logits: torch.Tensor, logits: torch.Tensor) -> None:
    if grad_logits.dtype != logits.dtype or grad_logits.shape != logits.shape or \
            grad_logits.device != logits.device or not grad_logits.is_contiguous():
        raise TcamCrfError(f"the gradient buffer must be contiguous {logits.dtype} {tuple(logits.shape)} on "
                           f"{logits.device}, got {grad_logits.dtype} {tuple(grad_logits.shape)} on {grad_logits.device}")


def seed_ce_backward_(grad_logits: torch.Tensor, logits: torch.Tensor, sel: torch.Tensor, ksz: int, count: torch.Tensor,
                      grad_output: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """grad_logits += (grad_output * scale) * d CE / d logits, in place on the labelled pixels.  grad_logits has the
    dtype the library reads the logits in (library_logits); a float16 / bfloat16 element is rounded once from the
    float32 sum."""
    lib = _lib.load()
    _require_cuda(logits, "logits")
    if logits.dtype not in _LOGIT_DTYPES:
        logits = logits.float()
    dtype = _logits_code(logits)
    _check_seeds(logits, sel)
    _check_grad(grad_logits, logits)
    b, k, h, w = logits.shape
    g = grad_output.detach().reshape(-1)[:1].to(device=logits.device, dtype=torch.float32).contiguous()
    with torch.cuda.device(logits.device):
        _lib.check(lib.tcam_seed_ce_backward_typed(logits.data_ptr(), dtype, sel.data_ptr(), int(sel.shape[2]), b, k, h,
                                                   w, int(ksz), count.data_ptr(), g.data_ptr(), float(scale),
                                                   grad_logits.data_ptr(), _stream_ptr(logits.device)),
                   "tcam_seed_ce_backward")
    return grad_logits


def crf_seed_ce_backward(as_t: torch.Tensor, logits: torch.Tensor, sel: torch.Tensor, ksz: int, count: torch.Tensor,
                         grad_output: torch.Tensor, n_norm: float, crf_weight: float, ce_weight: float) -> torch.Tensor:
    """Gradient w.r.t. the logits of crf_weight * CRF(softmax(logits)) + ce_weight * CE(logits, seeds)
    (tcam_crf_seed_ce_backward_typed): crf_backward_logits with the cross-entropy's gradient added on the labelled
    pixels, every element rounded once to the dtype the library read the logits in."""
    lib = _lib.load()
    _require_cuda(as_t, "AS")
    logits = library_logits(logits.detach())
    dtype = _logits_code(logits)
    _check_as(as_t, logits)
    _check_seeds(logits, sel)
    b, k, h, w = logits.shape
    g = grad_output.detach().reshape(-1)[:1].to(device=logits.device, dtype=torch.float32).contiguous()
    grad = torch.empty_like(logits)
    with torch.cuda.device(logits.device):
        _lib.check(lib.tcam_crf_seed_ce_backward_typed(as_t.data_ptr(), logits.data_ptr(), dtype, sel.data_ptr(),
                                                       int(sel.shape[2]), int(ksz), count.data_ptr(), g.data_ptr(), b,
                                                       k, h, w, float(n_norm), float(crf_weight), float(ce_weight),
                                                       grad.data_ptr(), _stream_ptr(logits.device)),
                   "tcam_crf_seed_ce_backward_typed")
    return grad


def temporal_cam_max(cams: torch.Tensor, renorm_h: float = 0.0) -> torch.Tensor:
    """max over dim 1 of a CUDA float32 stack [B,T,...] -> [B,...] with torch.maximum's NaN propagation.

    Mirrors the chain of ``torch.maximum`` calls in dlib/datasets/wsol_loader.py:591-600.  With renorm_h > 0
    (the loader's ``sl_tc_knn_t``) every frame first goes through ``re_normalize_cam`` (:630-635):
    ``nan_to_num(exp((cam + 1e-6) * h) / max over the frame)``, in the same kernel."""
    lib = _lib.load()
    _require_cuda(cams, "cams")
    if cams.dtype != torch.float32:
        raise TcamCrfError("cams must be float32")
    cams = cams.contiguous()
    b, t = cams.shape[0], cams.shape[1]
    rest = cams.shape[2:]
    hw = 1
    for s in rest:
        hw *= s
    out = torch.empty((b,) + tuple(rest), dtype=torch.float32, device=cams.device)
    with torch.cuda.device(cams.device):
        if renorm_h > 0:
            _lib.check(lib.tcam_temporal_max_renorm(cams.data_ptr(), out.data_ptr(), b, t, hw, float(renorm_h),
                                                    _stream_ptr(cams.device)), "tcam_temporal_max_renorm")
        else:
            _lib.check(lib.tcam_temporal_max(cams.data_ptr(), out.data_ptr(), b, t, hw, _stream_ptr(cams.device)),
                       "tcam_temporal_max")
    return out


def prepare_std_cams(std_cams: torch.Tensor, image_size) -> torch.Tensor:
    """nan_to_num -> bilinear resize (align_corners=False) -> nan_to_num in one kernel.

    std_cams [B,1,h,w] CUDA float32 -> [B,1,H,W]; Trainer.prepare_std_cams_disq, dlib/learning/train_wsol.py:417-432."""
    lib = _lib.load()
    _require_cuda(std_cams, "std_cams")
    if std_cams.ndim != 4 or std_cams.shape[1] != 1:
        raise TcamCrfError(f"std_cams must be [B,1,h,w], got {tuple(std_cams.shape)}")
    x = std_cams.detach().float().contiguous()
    bsz, _, h, w = x.shape
    big_h, big_w = (int(image_size), int(image_size)) if isinstance(image_size, int) else (int(image_size[0]), int(image_size[1]))
    out = torch.empty((bsz, 1, big_h, big_w), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tcam_prepare_std_cams(x.data_ptr(), out.data_ptr(), bsz, h, w, big_h, big_w,
                                             _stream_ptr(x.device)), "tcam_prepare_std_cams")
    return out


def otsu_roi(cams: torch.Tensor):
    """ROI masks by Otsu's threshold for a batch of CAMs [B,1,H,W] or [B,H,W] (float32, CUDA).
    Returns (roi long, same shape as cams; thresholds float32 [B] on the 0..255 scale).
    GPU version of GetRoiSingleCam with roi_method='roi_all' (dlib/cams/tcam_seeding.py:316-345)."""
    lib = _lib.load()
    _require_cuda(cams, "cams")
    x = cams.detach().float().contiguous()
    b = x.shape[0]
    hw = x[0].numel()
    roi = torch.empty(x.shape, dtype=torch.long, device=x.device)
    th = torch.empty(b, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tcam_otsu_roi(x.data_ptr(), roi.data_ptr(), th.data_ptr(), b, hw, _stream_ptr(x.device)),
                   "tcam_otsu_roi")
    return roi, th


def roi_components(cams: torch.Tensor, largest_only: bool, p_min_area: float, thresh: Optional[float] = None):
    """ROI = one 4-connected component of ``cam*255 >= thresh`` per sample: the densest one ('roi_high_density',
    falling back to the largest when it covers less than p_min_area of the frame) or the largest ('largest').

    cams [B,1,H,W] or [B,H,W] float32 CUDA; thresh in [0,1] or None (Otsu per sample, like get_thresh).
    Returns (roi long, same shape as cams; bbox_mask float32 [B,H,W]; bbox float32 [B,4] = x0,y0,x1,y1).
    GPU version of GetRoiSingleCam.__call__ (dlib/cams/tcam_seeding.py:347-412)."""
    lib = _lib.load()
    _require_cuda(cams, "cams")
    x = cams.detach().float().contiguous()
    if x.ndim == 4:
        assert x.shape[1] == 1
    b, h, w = x.shape[0], x.shape[-2], x.shape[-1]
    if thresh is None:
        _, th = otsu_roi(x)
    else:
        assert thresh >= 0, thresh
        th = torch.full((b,), float(thresh) * 255.0, dtype=torch.float32, device=x.device)
    roi = torch.empty(x.shape, dtype=torch.long, device=x.device)
    mask = torch.empty((b, h, w), dtype=torch.float32, device=x.device)
    bbox = torch.empty((b, 4), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device):
        nbytes = lib.tcam_roi_components_scratch_bytes(b, h, w)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        _lib.check(lib.tcam_roi_components(x.data_ptr(), th.data_ptr(), roi.data_ptr(), mask.data_ptr(),
                                           bbox.data_ptr(), b, h, w, 1 if largest_only else 0, float(p_min_area),
                                           scratch.data_ptr(), nbytes, _stream_ptr(x.device)),
                   "tcam_roi_components")
    return roi, mask, bbox.float()


__all__ = ["Lattice", "library_logits", "seed_ce_forward", "seed_ce_backward_", "crf_seed_ce_backward", "otsu_roi", "roi_components", "crf_filter_transposed", "crf_forward", "crf_backward", "crf_forward_logits", "crf_backward_logits", "temporal_cam_max", "prepare_std_cams", "workspace_status", "release_workspaces",
           "FEAT_COLOR", "FEAT_XY_RGB"]
