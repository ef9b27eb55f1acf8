"""oracle/ -- CPU checkers for the DenseCRF-loss hot path.  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package; the product package
(``tcam_wsol_video_b200``) never does and has no CPU fallback.

Two checkers live here:

* **port** -- ``permuto_oracle.c``: a plain-C restatement of the reference's
  permutohedral filter (file header cites the reference lines it follows).  It
  can be rebuilt anywhere gcc exists, so it travels to the GPU box.
* **ref** -- ``_ref/libref_{bilateralfilter,colorbilateralfilter}.so``: the
  reference's own C++ (``dlib/crf/crfwrapper/*``) compiled unmodified, in place,
  with a ctypes shim (``ref_shim.cpp``).  Built only where ``/root/reference`` is
  mounted; the git-ignored binaries travel to the GPU box with the snapshot.

The python functions below restate the few numpy/torch lines that surround the
native call in the reference (``dlib/crf/dense_crf_loss.py:56-74``,
``dlib/crf/color_dense_crf_loss.py:58-76``) and the temporal-CAM max / seed
selection (``oracle/seeding.py``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_float, c_int, c_void_p
from typing import Callable, Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PORT_SO = os.path.join(_HERE, "liboracle_permuto.so")
_REF_BF_SO = os.path.join(_HERE, "_ref", "libref_bilateralfilter.so")
_REF_CBF_SO = os.path.join(_HERE, "_ref", "libref_colorbilateralfilter.so")

_fp = POINTER(c_float)
_ip = POINTER(c_int)


def build(verbose: bool = False) -> None:
    """Compile the C restatement, and the reference's own C++ when its tree is mounted."""
    res = subprocess.run(["make", "-C", _HERE, "all"], capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("oracle build failed")


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _ptr(a: np.ndarray, typ=_fp):
    return a.ctypes.data_as(typ)


# --------------------------------------------------------------------------
# port (C restatement)
# --------------------------------------------------------------------------
_port = None


def load_port():
    global _port
    if _port is None:
        if not os.path.exists(_PORT_SO):
            build()
        lib = ctypes.CDLL(_PORT_SO)
        lib.po_bilateralfilter_batch.argtypes = [_fp, _fp, _fp, c_int, c_int, c_int, c_int, c_float, c_float]
        lib.po_bilateralfilter_batch.restype = c_int
        lib.po_colorbilateralfilter_batch.argtypes = [_fp, _fp, _fp, c_int, c_int, c_int, c_int, c_float, c_int]
        lib.po_colorbilateralfilter_batch.restype = c_int
        lib.po_lattice_bilateral.argtypes = [_fp, c_int, c_int, c_float, c_float]
        lib.po_lattice_bilateral.restype = c_void_p
        lib.po_lattice_color.argtypes = [_fp, c_int, c_int, c_float, c_int]
        lib.po_lattice_color.restype = c_void_p
        lib.po_build.argtypes = [_fp, c_int, c_int]
        lib.po_build.restype = c_void_p
        lib.po_filter.argtypes = [c_void_p, _fp, _fp]
        lib.po_filter.restype = c_int
        lib.po_free.argtypes = [c_void_p]
        lib.po_free.restype = None
        lib.po_num_vertices.argtypes = [c_void_p]
        lib.po_num_vertices.restype = c_int
        for name, typ in (("po_offsets", POINTER(ctypes.c_int32)), ("po_barycentric", _fp),
                          ("po_neighbours", POINTER(ctypes.c_int32)), ("po_keys", POINTER(ctypes.c_int16))):
            getattr(lib, name).argtypes = [c_void_p]
            getattr(lib, name).restype = typ
        lib.po_scale_factors.argtypes = [c_int, _fp]
        lib.po_scale_factors.restype = None
        _port = lib
    return _port


def port_bilateralfilter_batch(images, segs, N, K, H, W, sigma_rgb, sigma_xy) -> np.ndarray:
    """AS = filter(segs) with the 5-D lattice; flat float32 arrays in, [N*K*H*W] out."""
    lib = load_port()
    images, segs = _f32(images).ravel(), _f32(segs).ravel()
    out = np.zeros(N * K * H * W, dtype=np.float32)
    rc = lib.po_bilateralfilter_batch(_ptr(images), _ptr(segs), _ptr(out), N, K, H, W, sigma_rgb, sigma_xy)
    if rc:
        raise RuntimeError("po_bilateralfilter_batch failed")
    return out


def port_colorbilateralfilter_batch(images, segs, N, K, H, W, sigma_rgb, DIM) -> np.ndarray:
    lib = load_port()
    images, segs = _f32(images).ravel(), _f32(segs).ravel()
    out = np.zeros(N * K * H * W, dtype=np.float32)
    rc = lib.po_colorbilateralfilter_batch(_ptr(images), _ptr(segs), _ptr(out), N, K, H, W, sigma_rgb, DIM)
    if rc:
        raise RuntimeError("po_colorbilateralfilter_batch failed")
    return out


class Lattice:
    """Plain-numpy view of one built lattice (offset, bary, nbr, keys, M)."""

    def __init__(self, d, n, m, offset, bary, nbr, keys=None):
        self.d, self.n, self.m = d, n, m
        self.offset, self.bary, self.nbr, self.keys = offset, bary, nbr, keys


def _port_lattice_from_handle(lib, h, d, n) -> Lattice:
    if not h:
        raise RuntimeError("oracle lattice build failed")
    try:
        m = lib.po_num_vertices(h)
        cnt = n * (d + 1)
        offset = np.ctypeslib.as_array(lib.po_offsets(h), shape=(cnt,)).copy().reshape(n, d + 1)
        bary = np.ctypeslib.as_array(lib.po_barycentric(h), shape=(cnt,)).copy().reshape(n, d + 1)
        nbr = np.ctypeslib.as_array(lib.po_neighbours(h), shape=((d + 1) * max(m, 1) * 2,)).copy()
        nbr = nbr[: (d + 1) * m * 2].reshape(d + 1, m, 2)
        keys = np.ctypeslib.as_array(lib.po_keys(h), shape=(max(m, 1) * d,)).copy()[: m * d].reshape(m, d)
    finally:
        lib.po_free(h)
    return Lattice(d, n, m, offset, bary, nbr, keys)


def port_lattice_bilateral(image, H, W, sigma_rgb, sigma_xy) -> Lattice:
    lib = load_port()
    image = _f32(image).ravel()
    h = lib.po_lattice_bilateral(_ptr(image), H, W, sigma_rgb, sigma_xy)
    return _port_lattice_from_handle(lib, h, 5, H * W)


def port_lattice_color(image, H, W, sigma_rgb, DIM) -> Lattice:
    lib = load_port()
    image = _f32(image).ravel()
    h = lib.po_lattice_color(_ptr(image), H, W, sigma_rgb, DIM)
    return _port_lattice_from_handle(lib, h, DIM, H * W)


def port_lattice_features(features) -> Lattice:
    """The lattice of explicit per-pixel features [n, d] (already divided by their sigmas): Permutohedral::init
    (permutohedral.cpp:115-297), for layouts the two wrappers do not build (x, y + 1, 2 or 4 planes)."""
    lib = load_port()
    features = _f32(features)
    n, d = features.shape
    return _port_lattice_from_handle(lib, lib.po_build(_ptr(features.ravel()), d, n), d, n)


def port_filter_features(features, planes) -> np.ndarray:
    """Filters `planes` [K, n] through the lattice of explicit per-pixel features [n, d] (already divided by
    their sigmas): Permutohedral::init + one compute per plane (permutohedral.cpp:115-297, 507-572).
    Covers feature layouts the two reference wrappers do not build themselves (x, y, gray; d = 4)."""
    lib = load_port()
    features = _f32(features)
    n, d = features.shape
    planes = _f32(planes).reshape(-1, n)
    h = lib.po_build(_ptr(features.ravel()), d, n)
    if not h:
        raise RuntimeError("po_build failed")
    out = np.zeros_like(planes)
    try:
        for k in range(planes.shape[0]):
            src = np.ascontiguousarray(planes[k])
            dst = np.zeros(n, dtype=np.float32)
            if lib.po_filter(h, _ptr(src), _ptr(dst)):
                raise RuntimeError("po_filter failed")
            out[k] = dst
    finally:
        lib.po_free(h)
    return out


def xy_features(H: int, W: int, sigma_xy: float, planes, sigma_rgb: float) -> np.ndarray:
    """[H*W, 2 + C] features (col/sigma_xy, row/sigma_xy, plane_c/sigma_rgb ...) in float32, the arithmetic of
    initializePermutohedral (bilateralfilter.cpp:4-19) for any number of image planes C."""
    planes = _f32(planes).reshape(-1, H * W)
    col = np.tile(np.arange(W, dtype=np.float32), H)
    row = np.repeat(np.arange(H, dtype=np.float32), W)
    feats = [col / np.float32(sigma_xy), row / np.float32(sigma_xy)]
    feats += [planes[c] / np.float32(sigma_rgb) for c in range(planes.shape[0])]
    return np.ascontiguousarray(np.stack(feats, axis=1).astype(np.float32))


def port_scale_factors(d: int) -> np.ndarray:
    lib = load_port()
    sf = np.zeros(d, dtype=np.float32)
    lib.po_scale_factors(d, _ptr(sf))
    return sf


# --------------------------------------------------------------------------
# ref (the reference's own C++, compiled in place)
# --------------------------------------------------------------------------
_ref_bf = None
_ref_cbf = None


def have_ref() -> bool:
    return os.path.exists(_REF_BF_SO) and os.path.exists(_REF_CBF_SO)


def load_ref():
    global _ref_bf, _ref_cbf
    if _ref_bf is None:
        if not have_ref():
            raise FileNotFoundError("oracle/_ref is not built (needs /root/reference; run `make -C oracle`)")
        bf = ctypes.CDLL(_REF_BF_SO)
        bf.ref_bilateralfilter_batch.argtypes = [_fp, _fp, _fp, c_int, c_int, c_int, c_int, c_float, c_float]
        bf.ref_bilateralfilter_batch.restype = None
        bf.ref_lattice_bilateral.argtypes = [_fp, c_int, c_int, c_float, c_float, _ip, _fp, _ip]
        bf.ref_lattice_bilateral.restype = c_int
        bf.ref_omp_max_threads.restype = c_int
        bf.ref_omp_set_threads.argtypes = [c_int]
        cbf = ctypes.CDLL(_REF_CBF_SO)
        cbf.ref_colorbilateralfilter_batch.argtypes = [_fp, _fp, _fp, c_int, c_int, c_int, c_int, c_float, c_int]
        cbf.ref_colorbilateralfilter_batch.restype = None
        cbf.ref_lattice_color.argtypes = [_fp, c_int, c_int, c_float, c_int, _ip, _fp, _ip]
        cbf.ref_lattice_color.restype = c_int
        cbf.ref_omp_max_threads.restype = c_int
        cbf.ref_omp_set_threads.argtypes = [c_int]
        _ref_bf, _ref_cbf = bf, cbf
    return _ref_bf, _ref_cbf


def ref_bilateralfilter_batch(images, segs, N, K, H, W, sigma_rgb, sigma_xy) -> np.ndarray:
    bf, _ = load_ref()
    images, segs = _f32(images).ravel().copy(), _f32(segs).ravel().copy()
    out = np.zeros(N * K * H * W, dtype=np.float32)
    bf.ref_bilateralfilter_batch(_ptr(images), _ptr(segs), _ptr(out), N, K, H, W, sigma_rgb, sigma_xy)
    return out


def ref_colorbilateralfilter_batch(images, segs, N, K, H, W, sigma_rgb, DIM) -> np.ndarray:
    _, cbf = load_ref()
    images, segs = _f32(images).ravel().copy(), _f32(segs).ravel().copy()
    out = np.zeros(N * K * H * W, dtype=np.float32)
    cbf.ref_colorbilateralfilter_batch(_ptr(images), _ptr(segs), _ptr(out), N, K, H, W, sigma_rgb, DIM)
    return out


def ref_lattice_bilateral(image, H, W, sigma_rgb, sigma_xy) -> Lattice:
    bf, _ = load_ref()
    image = _f32(image).ravel().copy()
    d, n = 5, H * W
    offset = np.zeros(n * (d + 1), dtype=np.int32)
    bary = np.zeros(n * (d + 1), dtype=np.float32)
    m = bf.ref_lattice_bilateral(_ptr(image), H, W, sigma_rgb, sigma_xy, _ptr(offset, _ip), _ptr(bary), None)
    nbr = np.zeros((d + 1) * m * 2, dtype=np.int32)
    bf.ref_lattice_bilateral(_ptr(image), H, W, sigma_rgb, sigma_xy, None, None, _ptr(nbr, _ip))
    return Lattice(d, n, m, offset.reshape(n, d + 1), bary.reshape(n, d + 1), nbr.reshape(d + 1, m, 2))


def ref_lattice_color(image, H, W, sigma_rgb, DIM) -> Lattice:
    _, cbf = load_ref()
    image = _f32(image).ravel().copy()
    d, n = DIM, H * W
    offset = np.zeros(n * (d + 1), dtype=np.int32)
    bary = np.zeros(n * (d + 1), dtype=np.float32)
    m = cbf.ref_lattice_color(_ptr(image), H, W, sigma_rgb, DIM, _ptr(offset, _ip), _ptr(bary), None)
    nbr = np.zeros((d + 1) * m * 2, dtype=np.int32)
    cbf.ref_lattice_color(_ptr(image), H, W, sigma_rgb, DIM, None, None, _ptr(nbr, _ip))
    return Lattice(d, n, m, offset.reshape(n, d + 1), bary.reshape(n, d + 1), nbr.reshape(d + 1, m, 2))


def ref_set_threads(n: int) -> None:
    bf, cbf = load_ref()
    bf.ref_omp_set_threads(n)
    cbf.ref_omp_set_threads(n)


# --------------------------------------------------------------------------
# the python lines around the native call
# --------------------------------------------------------------------------
def best_filter(color: bool = False) -> Tuple[Callable, str]:
    """(filter function, kind): the reference build when present, else the port."""
    if have_ref():
        return (ref_colorbilateralfilter_batch if color else ref_bilateralfilter_batch), "reference"
    return (port_colorbilateralfilter_batch if color else port_bilateralfilter_batch), "port"


def densecrf_loss_fwd_bwd(images, segs, sigma_rgb, sigma_xy, grad_output: float = 1.0,
                          filter_fn: Optional[Callable] = None):
    """Restates DenseCRFLossFunction.forward/backward (dlib/crf/dense_crf_loss.py:56-74).

    images [N,3,H,W] float32 0..255, segs [N,K,H,W] float32.
    Returns (loss float32 scalar, grad_seg [N,K,H,W] float32, AS [N,K,H,W] float32).
    """
    segs = _f32(segs)
    N, K, H, W = segs.shape
    fn = filter_fn or best_filter(False)[0]
    AS = fn(images, segs, N, K, H, W, float(sigma_rgb), float(sigma_xy))
    n_fp32 = np.float32(N)
    loss = np.float32(-(segs.ravel() * AS).sum(dtype=np.float32)) / n_fp32
    AS = AS.reshape(N, K, H, W)
    grad = (np.float32(-2.0) * np.float32(grad_output)) * AS / n_fp32
    return np.float32(loss), grad.astype(np.float32), AS


def color_densecrf_loss_fwd_bwd(images, segs, sigma_rgb, grad_output: float = 1.0,
                                filter_fn: Optional[Callable] = None):
    """Restates ColorDenseCRFLossFunction (dlib/crf/color_dense_crf_loss.py:58-76).

    DIM is images.shape[1] (``nbr_p``, color_dense_crf_loss.py:47)."""
    segs = _f32(segs)
    images = _f32(images)
    N, K, H, W = segs.shape
    DIM = images.shape[1]
    fn = filter_fn or best_filter(True)[0]
    AS = fn(images, segs, N, K, H, W, float(sigma_rgb), int(DIM))
    n_fp32 = np.float32(N)
    loss = np.float32(-(segs.ravel() * AS).sum(dtype=np.float32)) / n_fp32
    AS = AS.reshape(N, K, H, W)
    grad = (np.float32(-2.0) * np.float32(grad_output)) * AS / n_fp32
    return np.float32(loss), grad.astype(np.float32), AS
