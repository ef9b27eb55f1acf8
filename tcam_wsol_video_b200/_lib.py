"""ctypes binding of csrc/libtcamcrf.so (C ABI: include/tcamcrf.h).

The library is built in-tree by ``build()`` (called from ``__graft_entry__.build``)
with ``nvcc -gencode arch=compute_100a,code=sm_100a``.  Loading never falls back to
anything else: a missing library or a failed call raises ``TcamCrfError``.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libtcamcrf.so")
SOURCES = [os.path.join(CSRC, "tcamcrf.cu")]
HEADERS = [os.path.join(CSRC, "lattice.cuh"), os.path.join(CSRC, "seed.cuh"), os.path.join(os.path.dirname(_HERE), "include", "tcamcrf.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]

FEAT_XY_RGB = 0
FEAT_COLOR = 1

STAGES = ("build", "neighbour", "splat", "blur", "slice", "loss", "backward", "prepare", "seed")

# element types of logits (TCAMCRF_DTYPE_*)
DTYPE_F32 = 0
DTYPE_F16 = 1
DTYPE_BF16 = 2

DEV_TABLE_FULL = 1
DEV_POOL_FULL = 2
DEV_KEY_RANGE = 4


class TcamCrfError(RuntimeError):
    pass


class Config(Structure):
    """Mirror of ``tcamcrf_config`` (include/tcamcrf.h)."""

    _fields_ = [
        ("feat", c_int),
        ("channels", c_int),
        ("image_stride_planes", c_int),
        ("sigma_rgb", c_float),
        ("sigma_xy", c_float),
        ("hash_load", c_float),
        ("pool_factor", c_float),
        ("chunk_frames", c_int),
        ("loss_weight", c_float),
    ]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise TcamCrfError("nvcc not found; cannot build libtcamcrf.so")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/tcamcrf.cu into csrc/libtcamcrf.so with NVCC_FLAGS only (sm_100a; cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + ["-o", LIB_PATH] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(" ".join(cmd))
        print(res.stdout + res.stderr)
    if res.returncode != 0:
        raise TcamCrfError("nvcc failed building libtcamcrf.so")
    return LIB_PATH


_lib = None

_fp = POINTER(c_float)
_cfgp = POINTER(Config)

# name -> (restype, argtypes); every symbol include/tcamcrf.h declares
SIGNATURES = {
    "tcamcrf_version": (c_int, []),
    "tcamcrf_last_error": (c_char_p, []),
    "tcamcrf_device_count": (c_int, []),
    "tcamcrf_workspace_bytes": (c_size_t, [_cfgp, c_int, c_int, c_int, c_int]),
    "tcamcrf_chunk_frames": (c_int, [_cfgp, c_int, c_int, c_int, c_int]),
    "tcamcrf_key_range_ok": (c_int, [_cfgp, c_int, c_int, c_float]),
    "tcamcrf_filter": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_filter_transposed": (c_int, [_cfgp, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_lattice_build": (c_int, [_cfgp, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_lattice_apply": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_filter_u8": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_forward": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_forward_host_frames": (c_int, [_cfgp, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_forward_u8": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_forward_logits": (c_int, [_cfgp, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_backward_logits": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "tcamcrf_loss_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_void_p]),
    "tcamcrf_loss_backward_weighted": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_void_p]),
    "tcamcrf_loss_backward_logits_weighted": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p]),
    "tcamcrf_workspace_status": (c_int, [c_void_p, c_void_p, POINTER(c_int), POINTER(c_int)]),
    "tcamcrf_debug_lattice": (c_int, [_cfgp, c_void_p, c_int, c_int, c_void_p, c_void_p, POINTER(c_int), c_void_p, c_size_t]),
    "tcam_debug_seed_draws": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "tcam_debug_exp_draws": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "bilateralfilter": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_float, c_float]),
    "bilateralfilter_batch": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float]),
    "colorbilateralfilter": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_float, c_int]),
    "colorbilateralfilter_batch": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int]),
    "tcamcrf_loss_fwd_bwd_host": (c_int, [_cfgp, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float]),
    "tcamcrf_set_tuning": (c_int, [c_char_p, c_int]),
    "tcamcrf_profile_enable": (None, [c_int]),
    "tcamcrf_profile_read": (c_int, [POINTER(ctypes.c_double), POINTER(ctypes.c_longlong), c_int]),
    "tcamcrf_launch_count": (ctypes.c_longlong, []),
    "tcam_temporal_max": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tcam_roi_components_scratch_bytes": (c_size_t, [c_int, c_int, c_int]),
    "tcam_roi_components": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_void_p, c_size_t, c_void_p]),
    "tcam_temporal_max_renorm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p]),
    "tcam_prepare_std_cams": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "tcam_seed_select": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                 c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "tcam_otsu_roi": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "tcam_seed_labels": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, ctypes.c_longlong, c_void_p, c_void_p]),
    "tcam_seed_ce_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "tcam_seed_ce_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                      c_float, c_void_p, c_void_p]),
    "tcamcrf_loss_forward_logits_typed": (c_int, [_cfgp, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int,
                                                  c_int, c_int, c_float, c_void_p, c_size_t, c_void_p]),
    "tcamcrf_loss_forward_host_frames_typed": (c_int, [_cfgp, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                                       c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_size_t,
                                                       c_void_p]),
    "tcamcrf_loss_backward_logits_typed": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                                   c_int, c_float, c_float, c_void_p]),
    "tcam_seed_ce_forward_typed": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "tcam_seed_ce_backward_typed": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                            c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "tcam_crf_seed_ce_backward_typed": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                                c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_void_p,
                                                c_void_p]),
    "tcam_seed_fused_supported": (c_int, [c_int, c_int]),
    "tcam_seed_fused": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int, c_int,
                                c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.c_longlong, c_void_p, c_void_p,
                                c_int, c_void_p, c_void_p]),
}


def load():
    """Load libtcamcrf.so (building it first if the sources are newer). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if needs_build():
        build()
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as exc:  # pragma: no cover - depends on the box
        raise TcamCrfError(f"cannot load {LIB_PATH}: {exc}") from exc
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and the header drift apart
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    return load().tcamcrf_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise TcamCrfError(f"{what} failed (status {rc}): {last_error()}")


def set_tuning(name: str, value: int = -1) -> None:
    """Sets a tuning knob of the library at run time (the TCAMCRF_<NAME> environment variables are read once, at
    first use); value < 0 restores the default.  Sweeps and tests only."""
    check(load().tcamcrf_set_tuning(name.encode(), int(value)), "tcamcrf_set_tuning")


_key_range_seen = {}


def require_key_range(cfg: Config, h: int, w: int, max_value: float = 255.0) -> None:
    """Raises a clear error when frames holding 0..max_value could leave the packed-key range of the lattice for this
    configuration (sigma too small for the lattice dimension, or more than 6 feature dimensions) instead of letting
    the call come back with a NaN loss.  Host arithmetic only; cached per configuration."""
    key = (cfg.feat, cfg.channels, float(cfg.sigma_rgb), float(cfg.sigma_xy), int(h), int(w), float(max_value))
    ok = _key_range_seen.get(key)
    if ok is None:
        ok = bool(load().tcamcrf_key_range_ok(ctypes.byref(cfg), int(h), int(w), float(max_value)))
        if len(_key_range_seen) < 256:
            _key_range_seen[key] = ok
    if not ok:
        d = cfg.channels + (2 if cfg.feat == FEAT_XY_RGB else 0)
        raise TcamCrfError(
            f"lattice configuration out of range: d={d} (supported: 1..6), sigma_rgb={cfg.sigma_rgb:g}, "
            f"sigma_xy={cfg.sigma_xy:g}, {h}x{w} frames with values up to {max_value:g} would leave the packed "
            f"64-bit vertex keys; use a larger sigma or fewer image planes")


def make_config(feat: int, channels: int, sigma_rgb: float, sigma_xy: float = 1.0, image_stride_planes: int = 0,
                hash_load: float = 0.0, pool_factor: float = 0.0, chunk_frames: int = 0,
                loss_weight: float = 0.0) -> Config:
    return Config(feat, channels, image_stride_planes or channels, float(sigma_rgb), float(sigma_xy),
                  float(hash_load), float(pool_factor), int(chunk_frames), float(loss_weight))
