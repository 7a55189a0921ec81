"""ctypes mirror of the reference's AEROBULK_MODEL interface (src/mod_aerobulk.f90:176-230)
on top of the C ABI of libaerobulk_gpu.so.  Same argument names, meaning and optional
arguments; Fortran STOPs become :class:`AerobulkError`."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# AEROBULK_GPU_LIB selects an experiment build (see aerobulk_b200/build.py); default: the in-tree library
_SO = os.environ.get("AEROBULK_GPU_LIB") or os.path.join(_HERE, "libaerobulk_gpu.so")
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_lib = None
NSTATS = 64


class AerobulkError(RuntimeError):
    """The reference would have STOPped here (ctl_stop / STOP); `code` is an AEROBULK_GPU_ERR_* value."""

    def __init__(self, code: int, message: str):
        super().__init__(f"[aerobulk_gpu rc={code}] {message}")
        self.code = code
        self.message = message


def lib():
    """Load libaerobulk_gpu.so (built in-tree by `python -m aerobulk_b200.build`). No fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise ImportError(f"{_SO} is missing: build it with `python -m aerobulk_b200.build` "
                          "(aerobulk_b200 has no CPU or PyTorch fallback)")
    L = C.CDLL(_SO)
    model_args = ([C.c_int, C.c_int, C.c_char_p, C.c_double, C.c_double, C.c_int, C.c_int] + [C.c_void_p] * 11 +
                  [_ip, _ip, C.c_void_p, C.c_void_p, C.c_void_p])
    for name in ("aerobulk_gpu_model", "aerobulk_gpu_model_device", "aerobulk_gpu_model_f32", "aerobulk_gpu_model_device_f32"):
        f = getattr(L, name)
        f.restype = C.c_int
        f.argtypes = model_args
    L.aerobulk_gpu_synchronize.restype = C.c_int
    L.aerobulk_gpu_init_local_stats.restype = C.c_int
    L.aerobulk_gpu_init_local_stats.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 7 + [_dp]
    L.aerobulk_gpu_stats_reduce_op.restype = C.c_int
    L.aerobulk_gpu_stats_reduce_op.argtypes = [C.c_int]
    L.aerobulk_gpu_init_from_stats.restype = C.c_int
    L.aerobulk_gpu_init_from_stats.argtypes = [C.c_int, C.c_char_p, _ip, C.c_int, _dp]
    L.aerobulk_gpu_init_local_stats_device.restype = C.c_int
    L.aerobulk_gpu_init_local_stats_device.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 8
    L.aerobulk_gpu_init_from_gathered_stats.restype = C.c_int
    L.aerobulk_gpu_init_from_gathered_stats.argtypes = [C.c_int, C.c_char_p, _ip, C.c_int, C.c_void_p, C.c_int]
    L.aerobulk_gpu_init.restype = C.c_int
    L.aerobulk_gpu_init.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_int] + [C.c_void_p] * 6 + [_ip, C.c_void_p, C.c_void_p]
    L.aerobulk_gpu_bye.restype = None
    L.aerobulk_gpu_set_async.argtypes = [C.c_int]
    L.aerobulk_gpu_set_kernel_timing.argtypes = [C.c_int]
    L.aerobulk_gpu_kernel_times.restype = C.c_int
    L.aerobulk_gpu_kernel_times.argtypes = [_dp, C.c_int]
    L.aerobulk_gpu_set_rdt.argtypes = [C.c_double]
    L.aerobulk_gpu_set_gdept.argtypes = [C.c_double]
    L.aerobulk_gpu_set_nb_iter.argtypes = [C.c_int]
    L.aerobulk_gpu_get_humidity_type.restype = C.c_char_p
    L.aerobulk_gpu_set_device.argtypes = [C.c_int]
    L.aerobulk_gpu_set_devices.restype = C.c_int
    L.aerobulk_gpu_set_devices.argtypes = [C.c_int]
    L.aerobulk_gpu_get_devices.restype = C.c_int
    L.aerobulk_gpu_shard_plan.restype = C.c_int
    L.aerobulk_gpu_shard_plan.argtypes = [C.c_longlong, C.c_int, C.POINTER(C.c_longlong)]
    L.aerobulk_gpu_set_stream.argtypes = [C.c_void_p]
    L.aerobulk_gpu_set_error_mode.argtypes = [C.c_int]
    L.aerobulk_gpu_set_verbose.argtypes = [C.c_int]
    L.aerobulk_gpu_last_error.restype = C.c_char_p
    L.aerobulk_gpu_get_state.restype = C.c_long
    L.aerobulk_gpu_get_state.argtypes = [C.c_int, _dp, C.c_long]
    L.aerobulk_gpu_set_state.restype = C.c_long
    L.aerobulk_gpu_set_state.argtypes = [C.c_int, _dp, C.c_long]
    L.aerobulk_gpu_launch_count.restype = C.c_long
    L.aerobulk_gpu_measure_fp64_peak.restype = C.c_double
    L.aerobulk_gpu_work_per_point.restype = C.c_double
    L.aerobulk_gpu_work_per_point.argtypes = [C.c_char_p, C.c_int, C.c_int]
    L.aerobulk_gpu_bytes_per_point.restype = C.c_double
    L.aerobulk_gpu_bytes_per_point.argtypes = [C.c_char_p, C.c_int]
    L.aerobulk_gpu_kernel_info.restype = C.c_int
    L.aerobulk_gpu_kernel_info.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.aerobulk_gpu_version.restype = C.c_char_p
    L.aerobulk_gpu_turb.restype = C.c_int
    L.aerobulk_gpu_turb.argtypes = ([C.c_char_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int] + [C.c_void_p] * 5 +
                                    [C.c_int, C.c_int] + [C.c_void_p] * 6 + [C.c_void_p] * 3 + [C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_int])
    L.aerobulk_gpu_set_nitend.argtypes = [C.c_int]
    L.aerobulk_gpu_turb_ice.restype = C.c_int
    L.aerobulk_gpu_turb_ice.argtypes = ([C.c_char_p, C.c_double, C.c_double, C.c_int, C.c_int] + [C.c_void_p] * 14 + [C.c_int])
    L.aerobulk_gpu_oce_ice.restype = C.c_int
    L.aerobulk_gpu_oce_ice.argtypes = ([C.c_char_p, C.c_char_p, C.c_double, C.c_double, C.c_longlong] + [C.c_void_p] * 4 +
                                       [C.c_int] + [C.c_void_p] * 5 + [C.c_int])
    L.aerobulk_gpu_set_ice_form_drag_per_point.argtypes = [C.c_int]
    L.aerobulk_gpu_flux_diagnostics.restype = C.c_int
    L.aerobulk_gpu_flux_diagnostics.argtypes = [C.c_longlong] + [C.c_void_p] * 6 + [_dp, C.c_int]
    L.aerobulk_gpu_diag_reduce_op.restype = C.c_int
    L.aerobulk_gpu_diag_reduce_op.argtypes = [C.c_int]
    L.aerobulk_gpu_host_register.restype = C.c_int
    L.aerobulk_gpu_host_register.argtypes = [C.c_void_p, C.c_size_t]
    L.aerobulk_gpu_host_unregister.restype = C.c_int
    L.aerobulk_gpu_host_unregister.argtypes = [C.c_void_p]
    L.aerobulk_gpu_series_ice.restype = C.c_int
    L.aerobulk_gpu_series_ice.argtypes = ([C.c_char_p, C.c_double, C.c_double, C.c_longlong] + [C.c_void_p] * 4 + [C.c_int] +
                                          [C.c_void_p] * 4 + [C.c_void_p, C.c_int])
    L.aerobulk_gpu_series.restype = C.c_int
    L.aerobulk_gpu_series.argtypes = ([C.c_char_p, C.c_int, C.c_longlong, C.c_double, C.c_double] + [C.c_void_p] * 5 +
                                      [C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int])
    L.aerobulk_gpu_series_csv.restype = C.c_int
    L.aerobulk_gpu_series_csv.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_double, C.c_double, C.c_int]
    L.aerobulk_gpu_probe.restype = C.c_int
    L.aerobulk_gpu_probe.argtypes = [C.c_int, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
    L.aerobulk_cxx_skin.restype = None
    L.aerobulk_cxx_no_skin.restype = None
    # language bindings get return codes instead of the reference's fail-stop
    L.aerobulk_gpu_set_error_mode(1)
    L.aerobulk_gpu_set_verbose(0)
    _lib = L
    return L


def _check(rc: int):
    if rc != 0:
        raise AerobulkError(rc, lib().aerobulk_gpu_last_error().decode(errors="replace"))


def _f64(a, shape=None):
    """float64 array in the ONE layout the library indexes: column-major (Fortran) for 2-D fields -- the flat index
    ji + Ni*jj of the reference's (Ni,Nj) arrays -- and contiguous for 1-D.  A C-ordered 2-D array (numpy's default)
    is copied; arrays already in that layout (pinned slabs, views of torch tensors) pass through untouched."""
    a = np.asarray(a, dtype=np.float64)
    if a.ndim >= 2:
        if not a.flags.f_contiguous:
            a = np.asfortranarray(a)
    elif not a.flags.c_contiguous:
        a = np.ascontiguousarray(a)
    if shape is not None and a.shape != shape:
        raise AerobulkError(101, f"AEROBULK_INIT => arrays do not agree in shape: {a.shape} vs {shape}")
    return a


def _f32(a, shape=None):
    """A float32 input of aerobulk_model_f32 in the layout of _f64; any other dtype is refused, never cast."""
    if not isinstance(a, np.ndarray) or a.dtype != np.float32:
        raise AerobulkError(101, f"aerobulk_model_f32 needs float32 numpy arrays, got {getattr(a, 'dtype', type(a).__name__)}")
    if a.ndim >= 2:
        if not a.flags.f_contiguous:
            a = np.asfortranarray(a)
    elif not a.flags.c_contiguous:
        a = np.ascontiguousarray(a)
    if shape is not None and a.shape != shape:
        raise AerobulkError(101, f"AEROBULK_INIT => arrays do not agree in shape: {a.shape} vs {shape}")
    return a


def _check_out(name, a, shape, dtype=np.float64):
    """A caller-supplied output array must be exactly what the library writes: `dtype`, the grid's shape, column-major
    (2-D) or contiguous (1-D), writeable -- anything else would silently pair different grid points across fields."""
    if not isinstance(a, np.ndarray) or a.dtype != dtype:
        raise AerobulkError(101, f"out['{name}'] must be a {np.dtype(dtype).name} numpy array")
    if a.shape != shape:
        raise AerobulkError(101, f"out['{name}'] has shape {a.shape}, the fields have {shape}")
    if not (a.flags.f_contiguous if a.ndim >= 2 else a.flags.c_contiguous):
        raise AerobulkError(101, f"out['{name}'] must be {'column-major (order=F)' if a.ndim >= 2 else 'contiguous'}")
    if not a.flags.writeable:
        raise AerobulkError(101, f"out['{name}'] is read-only")
    return a


def _shape2(shape):
    if len(shape) == 1:
        return shape[0], 1
    if len(shape) == 2:
        return shape[0], shape[1]
    raise AerobulkError(101, "fields must be 1-D or 2-D (Ni,Nj)")


def aerobulk_model(jt: int, Nt: int, calgo: str, zt: float, zu: float, sst, t_zt, hum_zt, U_zu, V_zu, slp,
                   Niter: Optional[int] = None, l_use_skin: Optional[bool] = None, rad_sw=None, rad_lw=None,
                   out: Optional[dict] = None) -> dict:
    """AEROBULK_MODEL with HOST (numpy) arrays, Fortran order (Ni,Nj).

    Returns {"QL","QH","Tau_x","Tau_y","Evap"[,"T_s"]}; T_s is present iff rad_sw and rad_lw
    are given (mod_aerobulk.f90:246-253).  `out` may hold preallocated (e.g. pinned) arrays.
    """
    return _model_host(lib().aerobulk_gpu_model, _f64, np.float64, jt, Nt, calgo, zt, zu,
                       (sst, t_zt, hum_zt, U_zu, V_zu, slp), Niter, l_use_skin, rad_sw, rad_lw, out)


def aerobulk_model_f32(jt: int, Nt: int, calgo: str, zt: float, zu: float, sst, t_zt, hum_zt, U_zu, V_zu, slp,
                       Niter: Optional[int] = None, l_use_skin: Optional[bool] = None, rad_sw=None, rad_lw=None,
                       out: Optional[dict] = None) -> dict:
    """:func:`aerobulk_model` on float32 numpy arrays (Fortran order), returning float32 arrays.

    Every output is the FP64 call on the exactly widened inputs, rounded once to nearest: bit for bit
    ``aerobulk_model(..., x.astype(float64), ...)[k].astype(float32)``.  The warm-layer state stays FP64 on the device,
    so float32 and float64 calls may alternate within one session.  Arrays of any other dtype raise
    AerobulkError(101); nothing is cast.  `out` may hold preallocated (e.g. pinned) float32 arrays.
    """
    return _model_host(lib().aerobulk_gpu_model_f32, _f32, np.float32, jt, Nt, calgo, zt, zu,
                       (sst, t_zt, hum_zt, U_zu, V_zu, slp), Niter, l_use_skin, rad_sw, rad_lw, out)


def _model_host(fn, prep, dtype, jt, Nt, calgo, zt, zu, fields, Niter, l_use_skin, rad_sw, rad_lw, out):
    sst = prep(fields[0])
    shape = sst.shape
    Ni, Nj = _shape2(shape)
    ins = [sst] + [prep(a, shape) for a in fields[1:]]
    rs = None if rad_sw is None else prep(rad_sw, shape)
    rl = None if rad_lw is None else prep(rad_lw, shape)
    names = ["QL", "QH", "Tau_x", "Tau_y", "Evap"] + (["T_s"] if (rs is not None and rl is not None) else [])
    res = {}
    for k in names:
        if out is not None and k in out:
            res[k] = _check_out(k, out[k], shape, dtype)
        else:
            res[k] = np.empty(shape, dtype=dtype, order="F")
    ni = None if Niter is None else C.byref(C.c_int(int(Niter)))
    ls = None if l_use_skin is None else C.byref(C.c_int(int(bool(l_use_skin))))
    ptr = lambda a: None if a is None else a.ctypes.data
    rc = fn(int(jt), int(Nt), calgo.encode(), float(zt), float(zu), Ni, Nj,
            *[ptr(a) for a in ins], *[ptr(res[k]) for k in names[:5]],
            ni, ls, ptr(rs), ptr(rl), ptr(res.get("T_s")))
    _check(rc)
    return res


def aerobulk_model_device(jt: int, Nt: int, calgo: str, zt: float, zu: float, sst, t_zt, hum_zt, U_zu, V_zu, slp,
                          out: dict, Niter: Optional[int] = None, l_use_skin: Optional[bool] = None,
                          rad_sw=None, rad_lw=None, shape=None) -> dict:
    """AEROBULK_MODEL on DEVICE-resident torch.float64 CUDA tensors (no host<->device traffic).

    `out` holds preallocated CUDA tensors QL, QH, Tau_x, Tau_y, Evap (and T_s with radiation).
    Tensors are flat buffers in Fortran (column-major) point order; `shape=(Ni,Nj)` names the
    grid (default (numel,1)).  The launch goes to the stream set by :func:`set_stream`
    (default: the library's own).
    """
    return _model_device(lib().aerobulk_gpu_model_device, "float64", jt, Nt, calgo, zt, zu,
                         (sst, t_zt, hum_zt, U_zu, V_zu, slp), out, Niter, l_use_skin, rad_sw, rad_lw, shape)


def aerobulk_model_device_f32(jt: int, Nt: int, calgo: str, zt: float, zu: float, sst, t_zt, hum_zt, U_zu, V_zu, slp,
                              out: dict, Niter: Optional[int] = None, l_use_skin: Optional[bool] = None,
                              rad_sw=None, rad_lw=None, shape=None) -> dict:
    """:func:`aerobulk_model_device` on contiguous torch.float32 CUDA tensors, `out` included (see
    :func:`aerobulk_model_f32` for what the outputs are).  Tensors of any other dtype raise AerobulkError(101)."""
    return _model_device(lib().aerobulk_gpu_model_device_f32, "float32", jt, Nt, calgo, zt, zu,
                         (sst, t_zt, hum_zt, U_zu, V_zu, slp), out, Niter, l_use_skin, rad_sw, rad_lw, shape)


def _model_device(fn, dtype, jt, Nt, calgo, zt, zu, tensors, out, Niter, l_use_skin, rad_sw, rad_lw, shape):
    tensors = list(tensors)
    n = tensors[0].numel()
    for t in tensors + [x for x in (rad_sw, rad_lw) if x is not None] + list(out.values()):
        if (not t.is_cuda) or str(t.dtype) != f"torch.{dtype}" or not t.is_contiguous() or t.numel() != n:
            raise AerobulkError(101, f"device API needs contiguous {dtype} CUDA tensors of one size")
    Ni, Nj = (n, 1) if shape is None else (int(shape[0]), int(shape[1]))
    if Ni * Nj != n:
        raise AerobulkError(101, f"shape {shape} does not match {n} points")
    ni = None if Niter is None else C.byref(C.c_int(int(Niter)))
    ls = None if l_use_skin is None else C.byref(C.c_int(int(bool(l_use_skin))))
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = fn(int(jt), int(Nt), calgo.encode(), float(zt), float(zu), Ni, Nj,
            *[ptr(t) for t in tensors],
            *[ptr(out[k]) for k in ("QL", "QH", "Tau_x", "Tau_y", "Evap")],
            ni, ls, ptr(rad_sw), ptr(rad_lw), ptr(out.get("T_s")))
    _check(rc)
    return out


def init_local_stats(sst, t_zt, hum_zt, U_zu, V_zu, slp, rad_lw=None) -> np.ndarray:
    """Row-block statistics of AEROBULK_INIT on flat DEVICE tensors (see include/aerobulk_gpu.h)."""
    L = lib()
    Ni, Nj = sst.numel(), 1
    st = np.zeros(NSTATS, dtype=np.float64)
    ptr = lambda t: None if t is None else t.data_ptr()
    _check(L.aerobulk_gpu_init_local_stats(Ni, Nj, ptr(sst), ptr(t_zt), ptr(hum_zt), ptr(U_zu), ptr(V_zu), ptr(slp),
                                           ptr(rad_lw), st.ctypes.data_as(_dp)))
    return st


def stats_reduce_ops() -> np.ndarray:
    L = lib()
    return np.array([L.aerobulk_gpu_stats_reduce_op(i) for i in range(NSTATS)], dtype=np.int64)


def init_from_stats(Nt: int, calgo: str, l_use_skin: Optional[bool], have_rad: bool, stats: np.ndarray):
    L = lib()
    st = np.ascontiguousarray(stats, dtype=np.float64)
    ls = None if l_use_skin is None else C.byref(C.c_int(int(bool(l_use_skin))))
    _check(L.aerobulk_gpu_init_from_stats(int(Nt), calgo.encode(), ls, int(bool(have_rad)), st.ctypes.data_as(_dp)))


def aerobulk_init(Nt: int, calgo: str, psst, pta, pha, pU, pV, pslp, l_use_skin: Optional[bool] = None, prsw=None, prlw=None):
    """AEROBULK_INIT on HOST (numpy) arrays -- the reference's public routine of the same name
    (src/mod_aerobulk.f90:24-160): flags, mask, humidity type and unit checks; raises AerobulkError where it STOPs."""
    L = lib()
    sst = _f64(psst)
    shape = sst.shape
    Ni, Nj = _shape2(shape)
    ins = [sst] + [_f64(a, shape) for a in (pta, pha, pU, pV, pslp)]
    rs = None if prsw is None else _f64(prsw, shape)
    rl = None if prlw is None else _f64(prlw, shape)
    ls = None if l_use_skin is None else C.byref(C.c_int(int(bool(l_use_skin))))
    ptr = lambda a: None if a is None else a.ctypes.data
    _check(L.aerobulk_gpu_init(int(Nt), calgo.encode(), Ni, Nj, *[ptr(a) for a in ins], ls, ptr(rs), ptr(rl)))


def aerobulk_bye():
    lib().aerobulk_gpu_bye()


def init_local_stats_device(sst, t_zt, hum_zt, U_zu, V_zu, slp, rad_lw=None, out=None):
    """Row-block statistics of AEROBULK_INIT written to DEVICE memory (`out`: 64-double CUDA tensor, created if None) on
    the session stream -- no host copy, no synchronisation (aerobulk_gpu_init_local_stats_device)."""
    import torch
    L = lib()
    if out is None:
        out = torch.empty(NSTATS, dtype=torch.float64, device=sst.device)
    ptr = lambda t: None if t is None else t.data_ptr()
    _check(L.aerobulk_gpu_init_local_stats_device(sst.numel(), 1, ptr(sst), ptr(t_zt), ptr(hum_zt), ptr(U_zu), ptr(V_zu),
                                                  ptr(slp), ptr(rad_lw), ptr(out)))
    return out


def init_from_gathered_stats(Nt: int, calgo: str, l_use_skin: Optional[bool], have_rad: bool, gathered, nranks: int):
    """AEROBULK_INIT from the all-gathered [nranks, 64] DEVICE tensor of row-block statistics: combined and judged on the
    device, asynchronously (aerobulk_gpu_init_from_gathered_stats)."""
    L = lib()
    if (not gathered.is_cuda) or str(gathered.dtype) != "torch.float64" or not gathered.is_contiguous() or gathered.numel() != nranks * NSTATS:
        raise AerobulkError(101, "init_from_gathered_stats needs a contiguous float64 CUDA tensor of nranks * 64 values")
    ls = None if l_use_skin is None else C.byref(C.c_int(int(bool(l_use_skin))))
    _check(L.aerobulk_gpu_init_from_gathered_stats(int(Nt), calgo.encode(), ls, int(bool(have_rad)), gathered.data_ptr(), int(nranks)))


def synchronize():
    _check(lib().aerobulk_gpu_synchronize())


def set_stream(cuda_stream_handle: Optional[int]):
    """Run on a caller-owned CUDA stream (e.g. ``torch.cuda.current_stream().cuda_stream``).
    None: the library's own stream.  Handle 0 is torch's legacy default stream -> cudaStreamLegacy (0x1)."""
    if cuda_stream_handle is None:
        lib().aerobulk_gpu_set_stream(None)
    else:
        lib().aerobulk_gpu_set_stream(C.c_void_p(cuda_stream_handle if cuda_stream_handle != 0 else 1))


def set_device(device: int):
    _check(lib().aerobulk_gpu_set_device(int(device)))


def set_devices(n: int):
    """Split every host-array aerobulk_model call over n GPUs inside the library (aerobulk_gpu_set_devices)."""
    _check(lib().aerobulk_gpu_set_devices(int(n)))


def get_devices() -> int:
    return lib().aerobulk_gpu_get_devices()


def shard_plan(n: int, n_dev: int) -> list:
    """Shard boundaries (flat point indices) of an n-point field on n_dev devices."""
    start = (C.c_longlong * 17)()
    k = lib().aerobulk_gpu_shard_plan(int(n), int(n_dev), start)
    if k < 0:
        raise ValueError("shard_plan: bad arguments")
    return [int(start[i]) for i in range(k + 1)]


def set_async(on: bool): lib().aerobulk_gpu_set_async(int(bool(on)))
def set_kernel_timing(on: bool): lib().aerobulk_gpu_set_kernel_timing(int(bool(on)))


def kernel_times(max_n: int = 65536) -> np.ndarray:
    """Durations [ms] of the flux-kernel launches recorded since the last call (set_kernel_timing(True))."""
    buf = np.zeros(max_n, dtype=np.float64)
    k = lib().aerobulk_gpu_kernel_times(buf.ctypes.data_as(_dp), max_n)
    return buf[:k].copy()


def set_rdt(v: float): lib().aerobulk_gpu_set_rdt(float(v))
def set_gdept(v: float): lib().aerobulk_gpu_set_gdept(float(v))
def set_nb_iter(v: int): lib().aerobulk_gpu_set_nb_iter(int(v))
def set_verbose(on: bool): lib().aerobulk_gpu_set_verbose(int(bool(on)))
def set_sort(mode: int): lib().aerobulk_gpu_set_sort(int(mode))
def nb_iter() -> int: return lib().aerobulk_gpu_get_nb_iter()
def use_skin() -> bool: return bool(lib().aerobulk_gpu_get_use_skin())
def humidity_type() -> str: return lib().aerobulk_gpu_get_humidity_type().decode()
def last_error() -> str: return lib().aerobulk_gpu_last_error().decode(errors="replace")
def reset(): lib().aerobulk_gpu_reset()
def new_session(): lib().aerobulk_gpu_new_session()
def launch_count() -> int: return lib().aerobulk_gpu_launch_count()
def reset_launch_count(): lib().aerobulk_gpu_reset_launch_count()
def measure_fp64_peak() -> float: return lib().aerobulk_gpu_measure_fp64_peak()
def work_per_point(calgo: str, skin: bool, nb: int) -> float: return lib().aerobulk_gpu_work_per_point(calgo.encode(), int(skin), int(nb))
def bytes_per_point(calgo: str, skin: bool) -> float: return lib().aerobulk_gpu_bytes_per_point(calgo.encode(), int(skin))


def kernel_info(calgo: str, skin: bool = False, zt_eq_zu: bool = False) -> dict:
    """Registers per thread, local (spill) bytes per thread and resident blocks per SM of the flux kernel that a call
    with (algo, skin, zt == zu) launches (aerobulk_gpu_kernel_info)."""
    r, l, b = C.c_int(0), C.c_int(0), C.c_int(0)
    _check(lib().aerobulk_gpu_kernel_info(calgo.encode(), int(skin), int(zt_eq_zu), C.byref(r), C.byref(l), C.byref(b)))
    return {"registers": r.value, "local_bytes": l.value, "blocks_per_sm": b.value, "warps_per_sm": b.value * 8}


def get_state(which: int, n: int) -> Optional[np.ndarray]:
    """Copy of the device-resident warm-layer state (0 dT_wl, 1 Hz_wl, 2 Qnt_ac, 3 Tau_ac)."""
    out = np.empty(n, dtype=np.float64)
    got = lib().aerobulk_gpu_get_state(int(which), out.ctypes.data_as(_dp), n)
    return out if got == n else None


def set_state(which: int, values) -> bool:
    v = np.ascontiguousarray(values, dtype=np.float64).ravel()
    return lib().aerobulk_gpu_set_state(int(which), v.ctypes.data_as(_dp), v.size) == v.size


TURB_OPTIONAL = ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "pdT_cs", "pdT_wl", "pHz_wl")


def set_nitend(v: int): lib().aerobulk_gpu_set_nitend(int(v))


def turb(calgo: str, kt: int, zt: float, zu: float, T_s, t_zt, q_s, q_zt, U_zu, l_use_cs: bool = False,
         l_use_wl: bool = False, Qsw=None, rad_lw=None, slp=None, isecday_utc: int = 0, plong=None, want=()) -> dict:
    """Direct TURB_* call on HOST (numpy) arrays, mirroring e.g. TURB_COARE3P6 (src/mod_blk_coare3p6.f90:123-127).
    Returns {"T_s","q_s","Cd","Ch","Ce","t_zu","q_zu","Ubzu"} plus the optional outputs named in `want`."""
    L = lib()
    Ts = np.array(T_s, dtype=np.float64, order="F", copy=True)
    shape = Ts.shape
    Ni, Nj = _shape2(shape)
    qs = np.array(q_s, dtype=np.float64, order="F", copy=True)
    ins = [_f64(a, shape) for a in (t_zt, q_zt, U_zu)]
    opt_in = [None if a is None else _f64(a, shape) for a in (Qsw, rad_lw, slp, plong)]
    outs = {k: np.empty(shape, dtype=np.float64, order="F") for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")}
    optv = {k: np.zeros(shape, dtype=np.float64, order="F") for k in want}
    ptr = lambda a: None if a is None else a.ctypes.data
    arr = (C.c_void_p * 10)(*[ptr(optv.get(k)) for k in TURB_OPTIONAL])
    rc = L.aerobulk_gpu_turb(calgo.encode(), int(kt), float(zt), float(zu), Ni, Nj, ptr(Ts), ptr(ins[0]), ptr(qs),
                             ptr(ins[1]), ptr(ins[2]), int(bool(l_use_cs)), int(bool(l_use_wl)),
                             *[ptr(outs[k]) for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")],
                             ptr(opt_in[0]), ptr(opt_in[1]), ptr(opt_in[2]), int(isecday_utc), ptr(opt_in[3]),
                             C.cast(arr, C.c_void_p), 0)
    _check(rc)
    outs.update(optv)
    outs["T_s"], outs["q_s"] = Ts, qs
    return outs


# ---------------------------------------------------------------------------
# station time series (SURVEY.md 8f row 3)
# ---------------------------------------------------------------------------
SERIES_OUT = ("rho_zu", "QL", "QH", "Qlw", "QNS", "Qsw", "dT_cs", "dT_wl", "TAU", "dT", "Hz_wl", "Qnt_ac", "Tau_ac",
              "Cd", "Ce", "Ch", "theta_zu", "q_zu", "t_zu", "RiB", "z0", "u_star", "L", "UN10", "Ts", "Evap", "q_zt",
              "theta_zt")
HUM_KINDS = {"q": 0, "sh": 0, "dp": 1, "rh": 2}


def series(calgo: str, zt: float, zu: float, isecday_utc, lon, sst, t_zt, hum_zt, wind, slp, rad_sw, rad_lw,
           hum_kind="q", l_use_skin: bool = True, want=SERIES_OUT) -> dict:
    """The time loop of src/tests/test_aerobulk_buoy_series_oce.f90:364-537 for S stations in one launch.
    Inputs are (Nt, S) C-ordered numpy arrays (station index fastest), `isecday_utc` (Nt,) ints, `lon` (S,).
    Returns the series named in `want`, each (Nt, S)."""
    L = lib()
    isd = np.ascontiguousarray(isecday_utc, dtype=np.int32)
    Nt = isd.shape[0]
    lon = np.ascontiguousarray(lon, dtype=np.float64).reshape(-1)
    S = lon.shape[0]
    ins = []
    for a in (sst, t_zt, hum_zt, wind, slp, rad_sw, rad_lw):
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.size != Nt * S:
            raise ValueError(f"series input of {a.size} values, expected Nt*S = {Nt}*{S}")
        ins.append(a)
    outs = {k: np.zeros((Nt, S), dtype=np.float64) for k in want}
    ptr = lambda a: None if a is None else a.ctypes.data
    arr = (C.c_void_p * len(SERIES_OUT))(*[ptr(outs.get(k)) for k in SERIES_OUT])
    hk = HUM_KINDS[hum_kind] if isinstance(hum_kind, str) else int(hum_kind)
    rc = L.aerobulk_gpu_series(calgo.encode(), Nt, S, float(zt), float(zu), ptr(isd), ptr(lon),
                               *[ptr(a) for a in ins[:3]], hk, *[ptr(a) for a in ins[3:]],
                               int(bool(l_use_skin)), C.cast(arr, C.c_void_p), 0)
    _check(rc)
    return outs


def series_device(calgo: str, zt: float, zu: float, isecday_utc, lon, sst, t_zt, hum_zt, wind, slp, rad_sw, rad_lw,
                  out: dict, hum_kind="q", l_use_skin: bool = True) -> dict:
    """:func:`series` on DEVICE-resident torch.float64 CUDA tensors ((Nt, S) contiguous; `lon` (S,)); `out` maps
    names of SERIES_OUT to preallocated (Nt, S) CUDA tensors.  `isecday_utc` stays a host int array.  Blocking."""
    L = lib()
    isd = np.ascontiguousarray(isecday_utc, dtype=np.int32)
    Nt, S = isd.shape[0], lon.numel()
    ins = [sst, t_zt, hum_zt, wind, slp, rad_sw, rad_lw]
    for t in ins + list(out.values()):
        if (not t.is_cuda) or str(t.dtype) != "torch.float64" or not t.is_contiguous() or t.numel() != Nt * S:
            raise AerobulkError(101, "series_device needs contiguous float64 CUDA tensors of Nt*S values")
    arr = (C.c_void_p * len(SERIES_OUT))(*[out[k].data_ptr() if k in out else None for k in SERIES_OUT])
    hk = HUM_KINDS[hum_kind] if isinstance(hum_kind, str) else int(hum_kind)
    rc = L.aerobulk_gpu_series(calgo.encode(), Nt, S, float(zt), float(zu), isd.ctypes.data, lon.data_ptr(),
                               *[t.data_ptr() for t in ins[:3]], hk, *[t.data_ptr() for t in ins[3:]],
                               int(bool(l_use_skin)), C.cast(arr, C.c_void_p), 1)
    _check(rc)
    return out


def series_csv(path_in: str, path_out: str, calgo: str, zt: float, zu: float, l_use_skin: bool = True) -> None:
    """One station, CSV in / CSV out (see include/aerobulk_gpu.h: aerobulk_gpu_series_csv)."""
    _check(lib().aerobulk_gpu_series_csv(os.fsencode(path_in), os.fsencode(path_out), calgo.encode(), float(zt),
                                         float(zu), int(bool(l_use_skin))))


# ---------------------------------------------------------------------------
# sea ice (SURVEY.md 8f row 4)
# ---------------------------------------------------------------------------
ICE_ALGORITHMS = ("nemo", "easy", "an05", "lu12", "lg15", "lg15_io")
ICE_OPTIONAL = ("CdN", "ChN", "CeN", "xz0", "xu_star", "xL", "xUN10", "CdN_frm")
OCE_ICE_OUT = tuple([k + "_i" for k in ("Cd", "Ch", "Ce", "theta_zu", "q_zu", "t_zu", "Ub", "RiB", "z0", "u_star", "L", "UN10",
                                         "rho_zu", "Tau", "QH", "QL", "Evap")] +
                    [k + "_w" for k in ("Cd", "Ch", "Ce", "theta_zu", "q_zu", "Ub", "z0", "u_star", "L", "UN10", "Tau", "QH",
                                         "QL", "Evap")] + ["Tau", "QH", "QL", "Evap"])


def set_ice_form_drag_per_point(on: bool):
    lib().aerobulk_gpu_set_ice_form_drag_per_point(int(bool(on)))


def turb_ice(calgo: str, zt: float, zu: float, Ts_i, t_zt, qs_i, q_zt, U_zu, frice=None, cxn=None, want=()) -> dict:
    """Direct TURB_ICE_<calgo> call on HOST (numpy) arrays (src/ice/mod_blk_ice_*.f90).
    Returns {"Cd","Ch","Ce","t_zu","q_zu","Ubzu"} plus the optional outputs named in `want`."""
    L = lib()
    Ts = _f64(Ts_i)
    shape = Ts.shape
    Ni, Nj = _shape2(shape)
    ins = [Ts] + [_f64(a, shape) for a in (t_zt, qs_i, q_zt, U_zu)] + [None if frice is None else _f64(frice, shape)]
    cx = None if cxn is None else np.ascontiguousarray(cxn, dtype=np.float64)
    outs = {k: np.empty(shape, dtype=np.float64, order="F") for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")}
    optv = {k: np.zeros(shape, dtype=np.float64, order="F") for k in want}
    ptr = lambda a: None if a is None else a.ctypes.data
    arr = (C.c_void_p * 8)(*[ptr(optv.get(k)) for k in ICE_OPTIONAL])
    rc = L.aerobulk_gpu_turb_ice(calgo.encode(), float(zt), float(zu), Ni, Nj, *[ptr(a) for a in ins], ptr(cx),
                                 *[ptr(outs[k]) for k in ("Cd", "Ch", "Ce", "t_zu", "q_zu", "Ubzu")],
                                 C.cast(arr, C.c_void_p), 0)
    _check(rc)
    outs.update(optv)
    return outs


def oce_ice(calgo_ice: str, calgo_oce, zt: float, zu: float, sit, sst, t_zt, hum_zt, wind, slp, frice, hum_kind="q",
            cxn=None, want=OCE_ICE_OUT) -> dict:
    """Ice + leads fluxes on HOST (numpy) 1-D arrays: the computation of src/ice/test_aerobulk_oce+ice.f90:225-412.
    `calgo_oce` None skips the leads.  Returns the series named in `want` (see OCE_ICE_OUT)."""
    L = lib()
    f = lambda a: None if a is None else np.ascontiguousarray(np.ravel(a, order="F"), dtype=np.float64)
    ins = [f(a) for a in (sit, sst, t_zt, hum_zt, wind, slp, frice)]
    n = ins[0].size
    cx = None if cxn is None else np.ascontiguousarray(cxn, dtype=np.float64)
    outs = {k: np.zeros(n, dtype=np.float64) for k in want}
    ptr = lambda a: None if a is None else a.ctypes.data
    arr = (C.c_void_p * len(OCE_ICE_OUT))(*[ptr(outs.get(k)) for k in OCE_ICE_OUT])
    hk = HUM_KINDS[hum_kind] if isinstance(hum_kind, str) else int(hum_kind)
    rc = L.aerobulk_gpu_oce_ice(calgo_ice.encode(), None if calgo_oce is None else calgo_oce.encode(), float(zt), float(zu),
                                n, ptr(ins[0]), ptr(ins[1]), ptr(ins[2]), ptr(ins[3]), hk, ptr(ins[4]), ptr(ins[5]),
                                ptr(ins[6]), ptr(cx), C.cast(arr, C.c_void_p), 0)
    _check(rc)
    return outs


SERIES_ICE_OUT = ("rho_zu", "QL", "QH", "Qlw", "QNS", "Qsw", "TAU", "SBLM", "Cd_i", "Ch_i", "Ce_i", "z0", "RiB_zt", "RiB_zu", "CdN",
                  "u_star", "L", "UN10", "theta_zu", "q_zu", "Ublk")


def series_ice(calgo: str, zt: float, zu: float, sic, sit, t_zt, hum_zt, wind, slp, rad_sw, rad_lw, hum_kind="q",
               want=SERIES_ICE_OUT) -> dict:
    """Sea-ice station series on HOST (numpy) arrays of any common shape: the per-record computation of
    src/ice/test_aerobulk_buoy_series_ice.f90:326-470 (records without ice read 0).  Returns the series named in `want`."""
    L = lib()
    shape = np.shape(sic)
    f = lambda a: np.ascontiguousarray(np.ravel(a), dtype=np.float64)
    ins = [f(a) for a in (sic, sit, t_zt, hum_zt, wind, slp, rad_sw, rad_lw)]
    n = ins[0].size
    if any(a.size != n for a in ins):
        raise ValueError("series_ice inputs differ in size")
    outs = {k: np.zeros(n, dtype=np.float64) for k in want}
    ptr = lambda a: None if a is None else a.ctypes.data
    arr = (C.c_void_p * len(SERIES_ICE_OUT))(*[ptr(outs.get(k)) for k in SERIES_ICE_OUT])
    hk = HUM_KINDS[hum_kind] if isinstance(hum_kind, str) else int(hum_kind)
    rc = L.aerobulk_gpu_series_ice(calgo.encode(), float(zt), float(zu), n, *[ptr(a) for a in ins[:4]], hk,
                                   *[ptr(a) for a in ins[4:]], C.cast(arr, C.c_void_p), 0)
    _check(rc)
    return {k: v.reshape(shape) for k, v in outs.items()}


# ---------------------------------------------------------------------------
# optional global flux diagnostics (SURVEY.md 8e)
# ---------------------------------------------------------------------------
NDIAG = 19
DIAG_FIELDS = ("QL", "QH", "Tau_x", "Tau_y", "Evap", "T_s")


def flux_diagnostics(fields: dict) -> np.ndarray:
    """Row-block sum / min / max of the flux fields named in DIAG_FIELDS (numpy arrays or CUDA torch tensors; missing
    ones are skipped): the 19-double vector of aerobulk_gpu_flux_diagnostics, to be combined across ranks with
    :func:`diag_reduce_ops` (0 sum, 1 min, 2 max)."""
    L = lib()
    present = [fields[k] for k in DIAG_FIELDS if k in fields and fields[k] is not None]
    on_dev = bool(present) and hasattr(present[0], "data_ptr")
    keep, ptrs, n = [], [], 0
    for k in DIAG_FIELDS:
        a = fields.get(k)
        if a is None:
            ptrs.append(None)
        elif on_dev:
            ptrs.append(a.data_ptr())
            n = a.numel()
        else:
            a = np.ascontiguousarray(np.ravel(a, order="F"), dtype=np.float64)
            keep.append(a)
            ptrs.append(a.ctypes.data)
            n = a.size
    st = np.zeros(NDIAG, dtype=np.float64)
    _check(L.aerobulk_gpu_flux_diagnostics(n, *ptrs, st.ctypes.data_as(_dp), int(on_dev)))
    return st


def diag_reduce_ops() -> np.ndarray:
    L = lib()
    return np.array([L.aerobulk_gpu_diag_reduce_op(i) for i in range(NDIAG)], dtype=np.int64)


def diagnostics_summary(st: np.ndarray) -> dict:
    """{"n": count, field: {"mean", "min", "max"}} from a (combined) diagnostics vector."""
    out = {"n": int(st[0])}
    for f, k in enumerate(DIAG_FIELDS):
        s_, lo, hi = st[1 + 3 * f: 4 + 3 * f]
        if hi >= lo:
            out[k] = {"mean": float(s_ / max(st[0], 1.0)), "min": float(lo), "max": float(hi)}
    return out


PROBE = {"e_sat": 1, "q_sat": 2, "theta_from_z_P0_T_q": 3, "rho_air": 4, "visc_air": 5, "L_vap": 6, "cp_air": 7,
         "gamma_moist": 8, "alpha_sw": 9, "qlw_net": 10, "one_on_L": 11, "Ri_bulk": 12, "q_air_rh": 13, "q_air_dp": 14,
         "psi_m_ncar": 20, "psi_h_ncar": 21, "psi_m_coare": 22, "psi_h_coare": 23, "psi_m_ecmwf": 24, "psi_h_ecmwf": 25,
         "psi_m_andreas": 26, "psi_h_andreas": 27, "z0tq_LKB": 30, "cd_n10_ncar": 31, "charn_coare3p0": 32,
         "charn_coare3p6": 33, "cs_coare": 34, "cs_ecmwf": 35, "exp": 40, "exp10": 41, "log": 42, "atan": 43, "sqrt": 44,
         "rsqrt": 45, "cbrt": 46, "rcbrt": 47, "pow075": 48, "rcp": 49, "powr": 50}


def probe(func: str, *args) -> np.ndarray:
    """One __device__ building block of the hot path evaluated on the GPU for arrays of arguments
    (aerobulk_gpu_probe; the per-function unit tests of tests/test_gpu_functions.py)."""
    cols = np.broadcast_arrays(*[np.asarray(a, dtype=np.float64) for a in args])
    n = cols[0].size
    packed = np.ascontiguousarray(np.stack([c.ravel() for c in cols], axis=0))
    out = np.empty(n, dtype=np.float64)
    _check(lib().aerobulk_gpu_probe(PROBE[func], n, len(cols), packed.ctypes.data, out.ctypes.data))
    return out.reshape(cols[0].shape)


def host_register(a: np.ndarray):
    """Page-lock an existing numpy array so that host-array calls take the zero-copy path (release with host_unregister
    before the array is freed)."""
    _check(lib().aerobulk_gpu_host_register(a.ctypes.data, a.nbytes))


def host_unregister(a: np.ndarray):
    _check(lib().aerobulk_gpu_host_unregister(a.ctypes.data))
