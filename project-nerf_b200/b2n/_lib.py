"""ctypes binding of libb2nerf.so (C ABI declared in include/b2nerf.h).

The library is built in-tree by ``project-nerf_b200/build.py`` and is the only
compute path of this package: if it is missing the import FAILS -- there is no
CPU or eager-PyTorch fallback.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libb2nerf.so")

ABI_VERSION = 19

P, L, I, F = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float

# name -> argtypes (all functions return int unless listed in _RESTYPES)
SIGNATURES = {
    "b2n_abi_version": [],
    "b2n_last_error": [],
    "b2n_set_active_rows": [P],
    "b2n_occ_pack_bits": [P, L, P, P],
    "b2n_occ_active_mask": [P, L, P, I, F, F, P, P],
    "b2n_occ_update": [P, P, L, I, F, F, P, P, P, P],
    "b2n_march_mask": [P, P, P, P, P, P, P, I, F, F, L, I, P, P, P, P],
    "b2n_march_scan_scratch": [L],
    "b2n_march_scan": [P, P, I, L, P, P, P, P],
    "b2n_march_compact": [P, P, P, P, P, P, L, I, P, P, P, P, P],
    "b2n_composite_fwd": [P, P, P, P, P, P, I, P, P, L, I, P, P, P, P, P],
    "b2n_composite_bwd": [P, P, P, P, P, P, I, P, P, L, I, P, P, P, P, P, P, P, P],
    "b2n_pe_fwd": [P, L, I, P, I, P, I, I, P],
    "b2n_pe_bwd": [P, L, I, P, I, P, I, I, P, I, P],
    "b2n_hash_fwd": [P, L, F, P, P, I, I, P, I, I, P],
    "b2n_hash_bwd": [P, L, F, P, P, I, I, P, I, I, P, P, I, I, I, P],
    "b2n_hash_order_scratch": [L],
    "b2n_hash_order": [P, L, F, P, P, P, P],
    "b2n_hash_fwd_ordered": [P, P, L, F, P, P, I, I, P, I, I, P],
    "b2n_hash_bwd_ordered": [P, P, L, F, P, P, I, I, P, I, I, P, I, I, P],
    "b2n_hash_tri_fwd": [P, P, L, F, P, P, P, P, I, P, I, P],
    "b2n_hash_tri_bwd": [P, P, L, F, P, I, P, I, P, P, P, P],
    "b2n_linear_fwd": [P, I, P, I, P, P, I, L, I, I, I, P],
    "b2n_linear_dgrad": [P, I, P, I, P, I, I, P, I, L, I, I, I, P],
    "b2n_linear_wgrad": [P, I, P, I, P, I, P, L, I, I, P],
    "b2n_act_bwd": [P, I, P, I, L, I, I, P],
    "b2n_sigma_head_fwd": [P, I, L, P, P],
    "b2n_sigma_head_bwd": [P, I, L, P, P, I, P],
    "b2n_instant_mlp_fwd_tc": [P, I, I, P, P, I, P, P, L, P, P, F, P, P],
    "b2n_instant_mlp_bwd_tc": [P, I, I, P, P, I, P, P, L, P, P, P, I, P, P, P, F, P, P],
    "b2n_fmlp_in_pad": [I],
    "b2n_fmlp_out_pad": [I],
    "b2n_fmlp_fwd": [P, I, I, P, I, I, I, I, P, P, P, I, I, L, P, I, P, P, P],
    "b2n_fmlp_bwd": [I, I, I, I, P, P, I, I, L, P, I, P, I, P, P, P, P, I, P, I, P, P],
    "b2n_fmlp_wgrad_tc": [P, P, P, P, L, I, I, I, P, P, P, P, P, P, P],
    "b2n_fmlp_wgrad": [I, P, P, P, P, P, P, P, P, P, P, P, L, P, P],
    "b2n_nerf_mlp_wgrad": [P, P, P, I, P, L, P, P, P, P, P, P, P, P],
    "b2n_nerf_mlp_dx": [P, P, P, I, P, I, I, L, P, I, P],
    "b2n_nerf_mlp_head_wgrad": [P, P, P, L, P, P, P, P],
    "b2n_nerf_mlp_packed_bytes": [],
    "b2n_nerf_mlp_pack": [P, P, P, I, I, P, P],
    "b2n_nerf_mlp_fwd": [P, I, P, I, P, P, P, P, P, L, P, P, P, P, P, P],
    "b2n_pad_bf16": [P, L, I, I, P, P],
    "b2n_opt_prepare": [P, I, P, P, P],
    "b2n_opt_adamw": [P, I, P, I, P, P, P, P, P],
    "b2n_sample_rays": [P, P, P, P, P, P, L, I, I, I, F, F, P, P, P, P, P],
    "b2n_nerf_mlp_packed_bwd_bytes": [],
    "b2n_nerf_mlp_pack_bwd": [P, P, P, I, I, P, P],
    "b2n_nerf_mlp_bwd": [P, P, P, P, P, P, P, P, L, P, P, P, P],
    "b2n_mesh_scratch": [I],
    "b2n_mesh_count": [P, I, F, P, P, P],
    "b2n_mesh_emit": [P, P, I, F, P, L, L, P, P, P],
    "b2n_render_scratch": [L],
    "b2n_render_begin": [P, L, I, P, P, P, P, P],
    "b2n_render_emit": [P, P, P, P, P, L, I, P, P, L, I, P, P, P, P, P, P, P],
    "b2n_render_composite": [P, P, P, P, L, I, F, P, P, L, P, P, P, P, P],
    "b2n_render_finish": [P, L, P, I, P, P, P, P],
    "b2n_importance_sample": [P, P, P, P, P, L, I, I, P, P, P, P],
}
# development / measurement entry points (include/b2nerf_debug.h): bound like the rest, never called by a product path
DEBUG_SIGNATURES = {
    "b2n_debug_mlp256_prof": [P],
    "b2n_debug_mlp256_flags": [ctypes.c_int],
    "b2n_debug_mlp256_set_pair": [ctypes.c_int],
    "b2n_debug_hash_variant": [I, I],
    "b2n_debug_hash_config": [P, P],
    "b2n_debug_instant_bwd_groups": [I],
    "b2n_debug_instant_fwd_slots": [I],
    "b2n_debug_gather_bench": [P, L, I, I, P, P],
    "b2n_debug_red_bench": [P, L, I, I, I, P],
    "b2n_debug_mnmajor_probe": [P, P, P, I, I, I, I, P],
}
_RESTYPES = {"b2n_last_error": ctypes.c_char_p, "b2n_march_scan_scratch": ctypes.c_size_t, "b2n_hash_order_scratch": ctypes.c_size_t,
             "b2n_mesh_scratch": ctypes.c_size_t, "b2n_render_scratch": ctypes.c_size_t,
             "b2n_nerf_mlp_packed_bytes": ctypes.c_size_t, "b2n_nerf_mlp_packed_bwd_bytes": ctypes.c_size_t}


class HashLevelC(ctypes.Structure):
    """mirror of b2n_hash_level"""
    _fields_ = [("scale", ctypes.c_float), ("res", ctypes.c_uint32), ("size", ctypes.c_uint32),
                ("offset", ctypes.c_uint32), ("hashed", ctypes.c_uint32)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA extension first (python project-nerf_b200/build.py). "
            "This package has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in list(SIGNATURES.items()) + list(DEBUG_SIGNATURES.items()):
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, ctypes.c_int)
    v = lib.b2n_abi_version()
    if v != ABI_VERSION:
        raise ImportError(f"libb2nerf.so ABI {v} != binding ABI {ABI_VERSION}: rebuild")
    return lib


lib = _load()

# launch accounting for bench.py ("gpu_launches"): every successful C-ABI call adds the
# number of kernels that entry point launches.
LAUNCHES = {"count": 0}
_KERNELS_PER_CALL = {"b2n_march_scan": 3, "b2n_hash_order": 5, "b2n_mesh_count": 2, "b2n_mesh_emit": 2, "b2n_render_begin": 3, "b2n_render_emit": 3, "b2n_render_composite": 3, "b2n_linear_wgrad": 2, "b2n_instant_mlp_bwd_tc": 2, "b2n_fmlp_bwd": 2}   # 16-bit MLP backwards: |g|-max pre-pass + kernel


def ptr(t):
    """device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


class Profiler:
    """Per-entry-point device timing with CUDA events on the launching stream (bench.py uses it
    inside the timed region to get the dominant kernel's average duration for the roofline).
    ``work`` is (algorithmic_bytes, flops) of the call as computed by the op wrapper."""

    def __init__(self):
        self.records = []        # (name, bytes, flops, start_event, end_event)

    def summary(self):
        """name -> dict(calls, ms, bytes, flops); call after torch.cuda.synchronize()."""
        out = {}
        for name, nbytes, flops, e0, e1 in self.records:
            d = out.setdefault(name, dict(calls=0, ms=0.0, bytes=0.0, flops=0.0))
            d["calls"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["bytes"] += nbytes
            d["flops"] += flops
        return out


PROFILER = None      # set to a Profiler() to time every C-ABI call
# the ordered hash-grid entries compute what the plain ones compute: timed and counted under the same name
_PROFILE_AS = {"b2n_hash_fwd_ordered": "b2n_hash_fwd", "b2n_hash_bwd_ordered": "b2n_hash_bwd"}


def call(name: str, *args, work=(0.0, 0.0)):
    prof = PROFILER
    if prof is not None:
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = getattr(lib, name)(*args)
    if prof is not None:
        e1.record()
        prof.records.append((_PROFILE_AS.get(name, name), float(work[0]), float(work[1]), e0, e1))
    _raise_on(name, rc)
    LAUNCHES["count"] += _KERNELS_PER_CALL.get(name, 1)


def _raise_on(name, rc):
    if rc != 0:
        msg = lib.b2n_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError(f"{name}: {msg}")
        raise RuntimeError(f"{name} failed ({rc}): {msg}")


def hash_config():
    """(variant, merge_res) the F = 2 hash-grid kernels currently run with (include/b2nerf_debug.h)"""
    v, m = ctypes.c_int(), ctypes.c_int()
    _raise_on("b2n_debug_hash_config", lib.b2n_debug_hash_config(ctypes.byref(v), ctypes.byref(m)))
    return v.value, m.value


class hash_variant:
    """``with hash_variant(variant, merge_res):`` -- the F = 2 hash-grid kernels run in that A/B configuration
    (b2n_debug_hash_variant); the configuration found on entry is restored on exit."""

    def __init__(self, variant, merge_res):
        self.cfg = (variant, merge_res)

    def __enter__(self):
        self.prev = hash_config()
        _raise_on("b2n_debug_hash_variant", lib.b2n_debug_hash_variant(*self.cfg))
        return self

    def __exit__(self, *exc):
        _raise_on("b2n_debug_hash_variant", lib.b2n_debug_hash_variant(*self.prev))
        return False


# ---- device-side row count (b2n_set_active_rows): see march.march(static=True)
_ROWS = [None]


def current_rows():
    """the int32[1] device tensor holding the number of valid rows of the compact sample buffers, or None"""
    return _ROWS[0]


class active_rows:
    """``with active_rows(n_dev):`` -- every kernel launched inside treats rows >= n_dev[0] of its point-indexed
    arguments as absent (they are neither read nor written); ``None`` restores the host-side counts."""

    def __init__(self, n_dev):
        self.n_dev = n_dev

    def __enter__(self):
        self.prev = _ROWS[0]
        _ROWS[0] = self.n_dev
        lib.b2n_set_active_rows(ptr(self.n_dev))
        return self

    def __exit__(self, *exc):
        _ROWS[0] = self.prev
        lib.b2n_set_active_rows(ptr(self.prev))
        return False


def with_ctx_rows(backward):
    """decorator for autograd ``backward`` static methods: re-installs the row count that was active in the forward"""
    import functools

    @functools.wraps(backward)
    def wrapped(ctx, *grads):
        rows = getattr(ctx, "rows", None)
        if rows is None and _ROWS[0] is None:
            return backward(ctx, *grads)
        with active_rows(rows):
            return backward(ctx, *grads)
    return wrapped


def require_cuda(*tensors):
    """Every tensor handed to a kernel must live on ONE CUDA device, and that device must be the current one: the
    kernels launch on ``torch.cuda.current_stream()`` of the current device, so a tensor on another GPU would be read
    through a foreign pointer (an illegal address that poisons the context) instead of failing in Python."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise ValueError("b2n ops need CUDA tensors: there is no CPU path in this package")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError(f"b2n ops need all tensors on one device (got {dev} and {t.device})")
    if dev is not None and dev.index != torch.cuda.current_device():
        raise ValueError(f"tensors live on {dev} but the current CUDA device is cuda:{torch.cuda.current_device()}: "
                         f"call torch.cuda.set_device({dev.index}) (one process per GPU) or wrap the call in "
                         f"torch.cuda.device({dev.index})")
