"""ctypes binding of libneuradar_b200.so (the C ABI declared in include/neuradar_b200.h).

There is deliberately no fallback: if the shared library is missing, `load()` raises, and every op in this
package goes through it.  PyTorch only supplies device memory and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libneuradar_b200.so")

MAX_LEVELS = 16
MAX_MLP_LAYERS = 4
MAX_MLP_WIDTH = 64
MAX_SAMPLES = 256

c_float_p = C.POINTER(C.c_float)


class Grid(C.Structure):
    _fields_ = [
        ("table", C.c_void_p),
        ("scalings", C.c_float * MAX_LEVELS),
        ("num_levels", C.c_int32),
        ("features_per_level", C.c_int32),
        ("log2_hashmap_size", C.c_int32),
    ]


class Rays(C.Structure):
    _fields_ = [
        ("origins", C.c_void_p),
        ("directions", C.c_void_p),
        ("pixel_area", C.c_void_p),
        ("nears", C.c_void_p),
        ("fars", C.c_void_p),
        ("num_rays", C.c_int64),
    ]


class Intervals(C.Structure):
    _fields_ = [
        ("starts", C.c_void_p),
        ("ends", C.c_void_p),
        ("row_stride", C.c_int64),
        ("num_samples", C.c_int32),
    ]


class Mlp(C.Structure):
    _fields_ = [
        ("weights", C.c_void_p * MAX_MLP_LAYERS),
        ("biases", C.c_void_p * MAX_MLP_LAYERS),
        ("dims", C.c_int32 * (MAX_MLP_LAYERS + 1)),
        ("num_layers", C.c_int32),
    ]


class MlpGrad(C.Structure):
    _fields_ = [
        ("weights", C.c_void_p * MAX_MLP_LAYERS),
        ("biases", C.c_void_p * MAX_MLP_LAYERS),
    ]


class FieldMlp(C.Structure):
    _fields_ = [
        ("weights", C.c_void_p * 5),
        ("biases", C.c_void_p * 5),
        ("beta", C.c_void_p),
        ("beta_min", C.c_float),
    ]


class FieldFusedSaved(C.Structure):  # nrb_field_fused_saved_t
    _fields_ = [("ximg", C.c_void_p), ("masks", C.c_void_p), ("ld", C.c_int64)]


class FieldFusedBwdIn(C.Structure):
    _fields_ = [("saved", FieldFusedSaved)] + [
        (n, C.c_void_p) for n in ("sh", "sdf", "alpha", "dfeature", "dfeat_ray", "weights", "dsdf", "dalpha", "actor_grid_id",
                                  "actor_dirs")
    ]


MAX_ACTORS = 256  # NRB_MAX_ACTORS: the length of ActorGrids.tables, checked against the library in load()


class ActorGrids(C.Structure):  # nrb_actor_grids_t
    _fields_ = [("tables", C.c_void_p * MAX_ACTORS), ("scalings", C.c_float * MAX_LEVELS), ("num_levels", C.c_int32),
                ("features_per_level", C.c_int32), ("log2_hashmap_size", C.c_int32), ("num_grids", C.c_int32)]


class ActorSamples(C.Structure):  # nrb_actor_samples_t
    _fields_ = [("grid_id", C.c_void_p), ("pos", C.c_void_p), ("std", C.c_void_p), ("dirs", C.c_void_p)]


class FieldFusedBwdOut(C.Structure):
    _fields_ = [("dximg", C.c_void_p), ("dweights", C.c_void_p * 5), ("dbiases", C.c_void_p * 5), ("dbeta", C.c_void_p)]


class Spacing(C.Structure):
    _fields_ = [("lam", C.c_float), ("scaling", C.c_float)]


class AdamCfg(C.Structure):  # nrb_adam_t
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("decoupled_weight_decay", C.c_int32), ("step", C.c_int32),
                ("grad_mult", C.c_float), ("zero_grad", C.c_int32)]


_P = C.c_void_p
_I32 = C.c_int32
_I64 = C.c_int64
_F = C.c_float

# name -> argtypes; every function returns int unless listed in _RESTYPES.  Mirrors include/neuradar_b200.h.
SIGNATURES = {
    "nrb_version": [],
    "nrb_max_actors": [],
    "nrb_last_error_string": [],
    "nrb_launch_count": [],
    "nrb_hash_fwd": [C.POINTER(Grid), _P, _P, _P, _I64, _P],
    "nrb_hash_indices": [C.POINTER(Grid), _P, _P, _I64, _P],
    "nrb_hash_bwd_workspace_bytes": [C.POINTER(Grid), _I64],
    "nrb_hash_bwd": [C.POINTER(Grid), _P, _P, _P, _P, _P, _I64, _P, _I64, _P],
    "nrb_frustum_gaussians": [C.POINTER(Rays), C.POINTER(Intervals), _F, _P, _P, _P],
    "nrb_mlp_fwd": [C.POINTER(Mlp), _P, _P, _P, _I64, _P],
    "nrb_mlp_bwd": [C.POINTER(Mlp), _P, _P, _P, _P, C.POINTER(MlpGrad), _I64, _P],
    "nrb_sh16": [_P, _P, _I64, _I32, _P],
    "nrb_weighted_depth_fwd": [_P, C.POINTER(Intervals), _I64, _P, _P],
    "nrb_weighted_depth_bwd": [C.POINTER(Intervals), _P, _I64, _P, _P],
    "nrb_peer_all_reduce": [_P, _P, C.c_uint64, _I32, _I32, _I32, _I64, _I64, _F, _I32, _P],
    "nrb_radar_rays": [_P, _P, _P, _P, _P, _P, _P, _P, _I32, _I64, _P, _P, _P, _P, _P, _P, _P],
    "nrb_tc_linear": [_P, _P, _P, _I32, _I32, _I32, _I64, _P, _P],
    "nrb_field_saved_ld": [_I64],
    "nrb_field_fused_image_bytes": [_I64],
    "nrb_field_fused_fwd": [C.POINTER(FieldMlp), C.POINTER(Grid), _P, _P, _P, _P, _I32, _I64, _P, _P, _P,
                            C.POINTER(FieldFusedSaved), C.POINTER(ActorGrids), C.POINTER(ActorSamples), _P],
    "nrb_field_fused_bwd": [C.POINTER(FieldMlp), C.POINTER(FieldFusedBwdIn), C.POINTER(FieldFusedBwdOut), _I32, _I64, _P],
    "nrb_hash_bwd_image": [C.POINTER(Grid), _P, _P, _P, _P, _P, _I64, _P, _I64, _P],
    "nrb_actor_assign": [C.POINTER(Rays), C.POINTER(Intervals), _P, _P, _P, _P, _I32, _P, _F, _P, _P, _P, _P, _P, _P],
    "nrb_actor_scatter": [C.POINTER(ActorGrids), C.POINTER(C.c_void_p), C.POINTER(ActorSamples), _P, _P, _I64, _P],
    "nrb_actor_pose_grad": [C.POINTER(Rays), C.POINTER(Intervals), _P, _I32, _P, _P, _F, C.POINTER(ActorGrids),
                            C.POINTER(ActorSamples), _P, _P, _P],
    "nrb_spaced_bins": [C.POINTER(Rays), Spacing, _P, _P, _I32, _I32, _P, _P, _P],
    "nrb_pdf_sample": [C.POINTER(Rays), Spacing, _P, _P, _I32, _P, _P, _I32, _F, _F, _P, _P, _P, _P, _P],
    "nrb_density_weights_fwd": [_P, C.POINTER(Intervals), _I64, _P, _P],
    "nrb_density_weights_bwd": [_P, C.POINTER(Intervals), _P, _I64, _P, _P],
    "nrb_alpha_composite_fwd": [_P, _P, C.POINTER(Intervals), _I64, _I32, _F, _I32, _P, _P, _P, _P, _P, _P],
    "nrb_accumulate_fwd": [_P, _P, _I64, _I32, _I32, _P, _P],
    "nrb_accumulate_bwd": [_P, _P, _P, _I64, _I32, _I32, _P, _P, _P],
    "nrb_alpha_composite_bwd": [_P, _P, C.POINTER(Intervals), _I64, _I32, _F, _I32, _P, _P, _P, _P, _P, _P, _P],
    "nrb_point_heads_fwd": [_P, _P, _P, _P, _P, _P, _P, _I64, _P],
    "nrb_point_heads_bwd": [_P, _P, _P, _P, _P, _P, _I64, _P],
    "nrb_lidar_carving": [C.POINTER(Intervals), _I64, _P, _P, _P, _F, _F, _P, _P, _P, _P, _P],
    "nrb_adam_step": [_P, _P, _P, _P, _I64, C.POINTER(AdamCfg), _P, _P, _P, _P],
    "nrb_grad_check": [_P, _I64, _P, _P],
    "nrb_distortion_loss": [_P, _I64, _P, _I64, _I32, _P, _P, _P],
    "nrb_interlevel_loss": [_P, _I64, _P, _I32, _P, _I64, _P, _I32, _F, _I64, _P, _P, _P],
    "nrb_proposal_fwd": [C.POINTER(Rays), C.POINTER(Grid), _P, _F, C.POINTER(Intervals), _P, _P, _P, _P,
                         C.POINTER(ActorGrids), C.POINTER(ActorSamples), _P],
    "nrb_proposal_bwd": [C.POINTER(Rays), C.POINTER(Grid), _P, _F, C.POINTER(Intervals), _P, _P, _P, _P, _P, _P, _P, _I64,
                         C.POINTER(ActorGrids), C.POINTER(ActorSamples), C.POINTER(C.c_void_p), _P],
}
_RESTYPES = {"nrb_max_actors": C.c_int32, "nrb_last_error_string": C.c_char_p, "nrb_launch_count": C.c_int64, "nrb_hash_bwd_workspace_bytes": C.c_int64, "nrb_field_saved_ld": C.c_int64,
             "nrb_field_fused_image_bytes": C.c_int64}

_lib: Optional[C.CDLL] = None


class NeuradarB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built: there is no other code path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NeuradarB200Error(
            f"{LIB_PATH} not found. Build it with `python -m neuradar_b200.build` (needs nvcc); "
            "neuradar_b200 has no CPU or pure-PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    if lib.nrb_max_actors() != MAX_ACTORS:  # every ActorGrids field after `tables` would be misplaced
        raise NeuradarB200Error(f"{LIB_PATH} was built with NRB_MAX_ACTORS = {lib.nrb_max_actors()}, the binding expects "
                                f"{MAX_ACTORS}; rebuild it with `python -m neuradar_b200.build`")
    _lib = lib
    return lib


class KernelTimer:
    """Optional per-kernel CUDA-event timing on the launching stream (used by bench.py for the roofline figure).
    Install with `_lib.TIMER = KernelTimer()`; `summary()` synchronises and returns {name: (launches, mean ms)}."""

    def __init__(self):
        self.events = {}

    def start(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def stop(self, name, e0):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self.events.setdefault(name, []).append((e0, e1))

    def reset(self):
        self.events = {}

    def summary(self):
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v) / len(v)) for k, v in self.events.items()}


TIMER: Optional[KernelTimer] = None
_EMPTY_SENTINEL = 256  # non-null, 16-byte aligned, never dereferenced (only passed together with a zero size)


def call(name: str, *args, tag: Optional[str] = None) -> None:
    """Invoke one C-ABI entry point, raising on a non-zero return code."""
    fn = getattr(load(), name)
    timer = TIMER
    if timer is None:
        rc = fn(*args)
    else:
        e0 = timer.start()
        rc = fn(*args)
        timer.stop(tag or name, e0)
    check(rc, name)


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().nrb_last_error_string()
        raise NeuradarB200Error(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def launch_count() -> int:
    return int(load().nrb_launch_count())


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a contiguous fp32/int64 CUDA tensor (None passes through as NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NeuradarB200Error("neuradar_b200 ops need CUDA tensors; there is no CPU path")
    if not t.is_contiguous():
        raise NeuradarB200Error("internal error: non-contiguous tensor reached the C ABI")
    if t.numel() == 0:
        return _EMPTY_SENTINEL  # empty tensors have a null data_ptr; sizes of 0 make every entry point a no-op
    return t.data_ptr()


def f32c(t: torch.Tensor) -> torch.Tensor:
    """fp32 + contiguous (no copy when already so)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()
