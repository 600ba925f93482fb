"""ctypes binding of libsmoke_sm100.so (the C ABI declared in include/smoke_b200.h).

There is no fallback: if the shared object is missing or a call fails, this raises.
"""
import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libsmoke_sm100.so")

c_f, c_i32, c_i64, c_p = C.c_float, C.c_int32, C.c_int64, C.c_void_p


class Grid(C.Structure):                     # smk_grid_t
    _fields_ = [("h", c_i32), ("w", c_i32), ("batch", c_i32),
                ("pitch_u", c_i32), ("pitch_v", c_i32), ("pitch_c", c_i32),
                ("stride_u", c_i64), ("stride_v", c_i64), ("stride_c", c_i64),
                ("row0", c_i32), ("gh", c_i32)]


class SlabCheck(C.Structure):                # smk_slab_check_t
    _fields_ = [("need_lo", c_i32), ("need_hi", c_i32), ("valid_lo", c_i32), ("valid_hi", c_i32),
                ("overflow_flag", c_p)]


class Source(C.Structure):                   # smk_source_t
    _fields_ = [("x", c_i32), ("y", c_i32), ("radius", c_i32), ("intensity", c_f)]


class State(C.Structure):                    # smk_state_t
    _fields_ = [("u", c_p * 2), ("v", c_p * 2), ("d", c_p * 2), ("p", c_p * 2), ("div", c_p),
                ("cur_u", c_i32), ("cur_v", c_i32), ("cur_d", c_i32), ("cur_p", c_i32)]


class Params(C.Structure):                   # smk_params_t
    _fields_ = [("dt", c_f), ("c_uv", c_f), ("c_d", c_f), ("decay", c_f),
                ("jacobi_iters", c_i32), ("sweeps_per_launch", c_i32), ("step_kernel", c_i32)]


STEP_KERNELS = {"auto": 0, "phases": 1, "fused": 2}           # SMK_STEP_AUTO / _PHASES / _FUSED

# element type of the frames smk_step_ex / smk_run_steps_ex write: SMK_FRAME_F32 / _F16 / _BF16
FRAME_FORMATS = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def frame_format(dtype):
    """SMK_FRAME_* code of a torch dtype; ValueError for anything but float32, float16 and bfloat16."""
    fmt = FRAME_FORMATS.get(dtype)
    if fmt is None:
        raise ValueError("frame dtype must be one of torch.float32, torch.float16, torch.bfloat16; got %r" % (dtype,))
    return fmt


class HaloBlock(C.Structure):                # smk_halo_block_t
    _fields_ = [("ptr", c_p), ("count", c_i64), ("peer", c_i32), ("is_send", c_i32)]


class PeerLink(C.Structure):                 # smk_peer_link_t
    _fields_ = [("remote_mailbox", c_p), ("remote_flag", c_p), ("local_mailbox", c_p), ("local_flag", c_p),
                ("send_off", c_i64 * 4), ("send_count", c_i64 * 4), ("recv_off", c_i64 * 4), ("recv_count", c_i64 * 4)]


class PeerComm(C.Structure):                 # smk_peer_comm_t
    _fields_ = [("link", PeerLink * 2), ("field_stride", c_i64), ("parity_stride", c_i64), ("seq", c_p)]


GP, SP, PP = C.POINTER(Grid), C.POINTER(State), C.POINTER(Params)

# name -> argtypes; every function returns int except smk_last_error_string.  Kept in one table so
# tests can check it against the header and the exported symbols.
SIGNATURES = {
    "smk_version": [],
    "smk_device_info": [C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32)],
    "smk_launch_count": [C.POINTER(c_i64)],
    "smk_set_device": [c_i32],
    "smk_reload_env": [],
    "smk_profile_begin": [c_i32],
    "smk_profile_end": [C.POINTER(C.c_double), C.POINTER(c_i64), c_i32],
    "smk_splat_sources": [GP, c_p, c_p, c_p, c_p],
    "smk_diffuse": [c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i64, c_f, c_p],
    "smk_forces_diffuse_div": [GP, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_p],
    "smk_divergence": [GP, c_p, c_p, c_p, c_f, c_p],
    "smk_jacobi": [GP, c_p, c_p, c_p, c_i32, c_i32, C.POINTER(c_i32), c_p],
    "smk_project": [GP, c_p, c_p, c_p, c_f, c_p],
    "smk_bilerp": [c_p, c_i32, c_i32, c_i32, c_p, c_p, c_p, c_i64, c_i32, c_p],
    "smk_advect": [GP, c_p, c_p, c_i32, c_i32, c_i32, c_i64, c_p, c_p, c_f, c_f, c_p, c_i64, c_p, c_p],
    "smk_advect_slab": [GP, c_p, c_p, c_i32, c_i32, c_i32, c_p, c_p, c_f, c_f, C.POINTER(SlabCheck), c_p],
    "smk_step": [GP, SP, PP, c_p, c_i64, c_p, c_p],
    "smk_run_steps": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_p],
    "smk_step_ex": [GP, SP, PP, c_p, c_i64, c_p, c_i32, c_p],
    "smk_run_steps_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p],
    "smk_run_steps_reset_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p, c_p, C.POINTER(c_i32), c_p],
    "smk_run_steps_src_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p, c_p, c_i32, c_p, c_p, C.POINTER(c_i32), c_p],
    "smk_run_steps_sched_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p, c_p, c_i32, c_i32, c_p, c_p, C.POINTER(c_i32),
                               c_p],
    "smk_run_steps_force_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p, c_p, c_i32, c_p, c_p, c_i32, c_i32, c_p, c_p,
                               C.POINTER(c_i32), c_p],
    "smk_run_steps_obst_ex": [GP, SP, PP, c_i32, c_p, c_i64, c_i64, c_p, c_i32, c_p, c_p, c_i32, c_p, c_p, c_i32, c_p, c_i64, c_i32, c_p,
                              c_p, C.POINTER(c_i32), c_p],
    "smk_jacobi_obst": [GP, c_p, c_p, c_p, c_p, c_i64, c_i32, c_i32, C.POINTER(c_i32), c_p],
    "smk_jacobi_residual_ex": [GP, c_p, c_p, c_p, c_i64, c_p, c_p],
    "smk_add_forcing": [GP, c_p, c_p, c_p, c_p, c_p],
    "smk_project_ex": [GP, c_p, c_p, c_p, c_f, c_p, c_i64, c_p],
    "smk_obstacle_faces": [GP, c_p, c_p, c_p, c_p, c_i64, c_f, c_p],
    "smk_obstacle_cells": [GP, c_p, c_p, c_i64, c_i32, c_p, c_i64, c_p],
    "smk_step_is_fused": [GP, PP, c_i32, C.POINTER(c_i32)],
    "smk_fused_plan": [c_i32, c_i32, c_i32, C.POINTER(c_i32), c_i32, C.POINTER(c_i32)],
    "smk_div_norms": [GP, c_p, c_p, c_p, c_p],
    "smk_jacobi_residual": [GP, c_p, c_p, c_p, c_p],
    "smk_fractal_fields": [c_p, c_p, c_p, c_i32, c_i32, c_i32, c_f, c_i32, c_p, c_p, c_p, c_p, c_p],
    "smk_frame_features": [c_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_p, c_i32, c_f, c_f, c_p, c_p, c_p, c_p],
    "smk_frame_distances": [c_p, c_i64, c_i32, c_i32, c_i32, c_i32, c_p, c_p],
    "smk_apply_mul": [c_p, c_p, c_p, c_i32, c_i32, c_i32, c_i32, c_i64, c_p],
    "smk_nccl_load": [C.c_char_p, C.POINTER(c_i32)],
    "smk_nccl_unique_id": [c_p],
    "smk_nccl_comm_init": [c_p, c_i32, c_i32, C.POINTER(c_p)],
    "smk_nccl_comm_destroy": [c_p],
    "smk_nccl_exchange": [c_p, C.POINTER(HaloBlock), c_i32, c_p],
    "smk_ipc_export": [c_p, c_p, C.POINTER(c_i64)],
    "smk_ipc_open": [c_p, c_i64, C.POINTER(c_p)],
    "smk_ipc_close": [c_p, c_i64],
    "smk_peer_push": [C.POINTER(PeerComm), C.POINTER(c_p), c_p],
    "smk_peer_unpack": [C.POINTER(PeerComm), C.POINTER(c_p), c_p],
    "smk_slab_step": [GP, SP, PP, C.POINTER(PeerComm), c_i32, C.POINTER(SlabCheck), C.POINTER(SlabCheck), C.POINTER(SlabCheck), c_p],
    "smk_project_advect": [GP, SP, PP, C.POINTER(SlabCheck), C.POINTER(SlabCheck), C.POINTER(SlabCheck), c_p],
    "smk_advect_adjoint": [GP, c_p, c_i32, c_i32, c_i32, c_i64, c_p, c_p, c_f, c_f, c_p, c_p, c_i64, c_p, c_p, c_i32, c_p, c_p,
                           c_p, c_p],
    "smk_project_adjoint": [GP, c_p, c_p, c_p, c_p, c_f, c_p],
    "smk_jacobi_adjoint": [GP, c_p, c_p, c_p, c_i32, c_i32, c_p, c_p],
    "smk_forces_diffuse_div_adjoint": [GP, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_p],
    "smk_project_adjoint_ex": [GP, c_p, c_p, c_p, c_p, c_f, c_p, c_i64, c_p],
    "smk_jacobi_adjoint_ex": [GP, c_p, c_p, c_p, c_i32, c_i32, c_p, c_p, c_i64, c_p],
    "smk_forces_diffuse_div_adjoint_ex": [GP, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_f, c_p, c_i64, c_p],
    "smk_splat_sources_adjoint": [GP, c_p, c_p, c_p, c_i32, c_p, c_p],
    "smk_splat_sources_adjoint_ex": [GP, c_p, c_p, c_p, c_i32, c_i32, c_p, c_p],
}

_lib = None


class SmokeLibraryError(RuntimeError):
    pass


def load():
    """Load libsmoke_sm100.so (built by smokephysai_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise SmokeLibraryError(
            "%s is missing: build it with `python -m smokephysai_b200.build` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for the smoke step." % SO_PATH)
    lib = C.CDLL(SO_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.smk_last_error_string.argtypes = []
    lib.smk_last_error_string.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().smk_last_error_string()
        raise SmokeLibraryError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def call(name, *args):
    check(getattr(load(), name)(*args), name)


_tls = threading.local()


def stream_on(device):
    """torch's current stream on `device` (a torch.device with an index); binds the library's own (statically linked)
    CUDA runtime to that device the first time this thread launches there.  Callers whose device may differ from the
    thread's current one wrap the launches in `on_device(device)`."""
    import torch
    idx = device.index
    if getattr(_tls, "bound", None) != idx:
        call("smk_set_device", idx)
        _tls.bound = idx
    return torch.cuda.current_stream(device).cuda_stream


class on_device:
    """Scope in which `device` is the thread's current CUDA device, for torch and for the library alike; the previous
    device is restored on exit, so a simulator built on cuda:1 never changes the process's current device behind the
    caller's back (both runtimes share the driver's per-thread current context).  Free when `device` already is current."""

    def __init__(self, device):
        self.idx = device.index
        self.prev = None

    def __enter__(self):
        import torch
        cur = torch.cuda.current_device()
        if cur != self.idx:
            self.prev = cur
            torch.cuda.set_device(self.idx)
            call("smk_set_device", self.idx)
            _tls.bound = self.idx
        return self

    def __exit__(self, *exc):
        if self.prev is not None:
            import torch
            call("smk_set_device", self.prev)
            torch.cuda.set_device(self.prev)
            _tls.bound = self.prev
        return False


def scoped(fn):
    """Method decorator: run with self._cuda as the current device (see on_device)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with on_device(self._cuda):
            return fn(self, *args, **kwargs)
    return wrapper


def reload_env():
    """Make the library read its SMK_* environment switches again (it reads them once per process otherwise)."""
    call("smk_reload_env")


def launch_count():
    """Kernels launched by the library in this process so far."""
    n = c_i64(0)
    call("smk_launch_count", C.byref(n))
    return n.value


PHASES = ("splat", "forces_diffuse_div", "jacobi", "project", "advect_u", "advect_v", "advect_d", "other", "step_fused", "halo",
          "project_advect_u", "halo_unpack")


def profile_begin(max_records=4096):
    call("smk_profile_begin", int(max_records))


def profile_end():
    """-> {phase: (total_ms, launches)} of every kernel launched since profile_begin()."""
    n = len(PHASES)
    ms = (C.c_double * n)()
    cnt = (c_i64 * n)()
    call("smk_profile_end", ms, cnt, n)
    return {PHASES[k]: (ms[k], cnt[k]) for k in range(n)}
