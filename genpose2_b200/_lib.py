"""ctypes binding of libgenpose_b200.so (the C ABI declared in include/genpose_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or a call
fails, this module raises.  PyTorch is used only for device memory and streams: every call
passes `tensor.data_ptr()` and `torch.cuda.current_stream().cuda_stream`.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgenpose_b200.so")

c_int, c_float, c_double, c_size_t, c_void_p = (
    ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_size_t, ctypes.c_void_p)


class TrunkParams(ctypes.Structure):
    """gp_trunk_params"""
    _fields_ = [
        ("pose_w0", c_void_p), ("pose_b0", c_void_p), ("pose_w1", c_void_p), ("pose_b1", c_void_p),
        ("fourier_w", c_void_p), ("t_w", c_void_p), ("t_b", c_void_p),
        ("head_w0", c_void_p * 3), ("head_b0", c_void_p * 3),
        ("head_w1", c_void_p * 3), ("head_b1", c_void_p * 3),
    ]


class ScaleNetParams(ctypes.Structure):
    """gp_scalenet_params"""
    _fields_ = [(n, c_void_p) for n in (
        "axes_w0", "axes_b0", "axes_w1", "axes_b1", "tail_w0", "tail_b0", "tail_w1", "tail_b1")]


# name -> (restype, argtypes); must list every symbol include/genpose_b200.h declares
SIGNATURES = {
    "gp_version": (c_int, []),
    "gp_last_error": (ctypes.c_char_p, []),
    "gp_launch_count": (ctypes.c_longlong, []),
    "gp_launch_count_reset": (None, []),
    "gp_fps": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gp_fps_chain": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gp_gather": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gp_ball_query": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p]),
    "gp_ball_query2": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p,
                               c_float, c_int, c_void_p, c_void_p]),
    "gp_ball_query2_tails": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                     c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gp_group": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gp_query_group": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p]),
    "gp_group_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                              c_void_p, c_void_p]),
    "gp_maxpool_rows": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gp_sa_small_mlp": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p),
                                ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gp_sa_small_mlp_hostw": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p),
                                ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gp_sa_small_mlp_hostw_tail": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p),
                                ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "gp_zero": (c_int, [c_void_p, c_size_t, c_void_p]),
    "gp_gemm_packed_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gp_gemm_pack": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "gp_gemm_bias_relu": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                                  c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gp_gemm_linear": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int,
                               c_void_p]),
    "gp_gemm_gather_bias_relu": (c_int, [c_void_p, c_int, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int,
                                         c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                         c_void_p, c_int, c_void_p]),
    "gp_centre_term": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "gp_centre_term_tail": (c_int, [c_void_p, ctypes.c_longlong, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                    c_void_p, c_int, c_void_p]),
    "gp_sa_mlp2_fused_xyz": (c_int, [c_void_p, c_void_p, c_int, c_void_p, ctypes.c_longlong, c_int, c_int, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                     c_int, c_void_p]),
    "gp_sa_mlp2_fused": (c_int, [c_void_p, c_int, c_int, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int,
                                 c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                 c_int, c_void_p]),
    "gp_trunk_packed_bytes": (c_size_t, []),
    "gp_trunk_pack": (c_int, [ctypes.POINTER(TrunkParams), c_void_p, c_void_p]),
    "gp_trunk_pack_tf32": (c_int, [ctypes.POINTER(TrunkParams), c_void_p, c_void_p]),
    "gp_trunk_project": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "gp_scorenet_eval": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gp_scorenet_ode_workspace_bytes": (c_size_t, [c_int]),
    "gp_scorenet_ode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double,
                                c_double, c_double, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                c_size_t, c_int, c_void_p]),
    "gp_scorenet_ode_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double,
                                      c_double, c_double, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                      c_size_t, c_int, c_void_p]),
    "gp_scorenet_ode_objects_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gp_scorenet_ode_objects": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double,
                                        c_double, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                        c_int, c_void_p]),
    "gp_scorenet_ode_dense_objects": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double,
                                              c_double, c_double, c_double, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                              c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "gp_scorenet_ode_objects_t0": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_double,
                                           c_double, c_double, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "gp_object_noise": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gp_traj_finalize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gp_scorenet_pc_workspace_bytes": (c_size_t, [c_int]),
    "gp_scorenet_pc": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                               c_int, c_double, c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "gp_energy": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gp_aggregate": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_int, c_void_p,
                             c_void_p, c_void_p, c_void_p]),
    "gp_pose_to_quat": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "gp_scalenet": (c_int, [ctypes.POINTER(ScaleNetParams), c_void_p, c_int, c_int, c_void_p, c_int,
                            c_void_p, c_void_p]),
}

GP_STAT_COUNT = 32
STAT_NFEV, STAT_ACCEPTED, STAT_REJECTED, STAT_STATUS, STAT_T_FINAL, STAT_H_INITIAL, STAT_H_LAST = range(7)

_lib = None


def load():
    """Load the library (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C genpose2_b200/csrc`).  genpose2_b200 has no CPU / PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().gp_last_error().decode("utf-8", "replace")


def launch_count():
    return int(load().gp_launch_count())


def reset_launch_count():
    load().gp_launch_count_reset()


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)  # ~50x cheaper than current_stream()


def stream_ptr(index=None):
    """cudaStream_t of torch's current stream on the current (or the given) device."""
    if _raw_stream is not None:
        return c_void_p(_raw_stream(torch.cuda.current_device() if index is None else index))
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def call(name, *args, device=None):
    """Invoke `name` on torch's current stream, raising RuntimeError (with gp_last_error) on a non-zero status."""
    lib = _lib if _lib is not None else load()
    fn = getattr(lib, name)
    cur = torch.cuda.current_device()
    if device is not None and device.index is not None and device.index != cur:
        with torch.cuda.device(device):
            rc = fn(*args, stream_ptr(device.index))
    else:
        rc = fn(*args, stream_ptr(cur))
    if rc != 0:
        raise RuntimeError(f"{name} failed with status {rc}: {last_error()}")


def check_cuda(t, name, dtype=None, rows=False):
    """rows=True: a 2-D row-major matrix that may be a column slice (unit column stride, any row stride)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (genpose2_b200 has no CPU path)")
    if rows:
        if t.dim() != 2 or t.stride(1) != 1:
            raise RuntimeError(f"{name} must be a row-major matrix (or a column slice of one)")
    elif not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t
