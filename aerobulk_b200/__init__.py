"""aerobulk_b200 -- B200-native (sm_100a) implementation of AeroBulk's `aerobulk_model` hot path.

The product is the CUDA shared library ``libaerobulk_gpu.so`` (C ABI in
``include/aerobulk_gpu.h``, C++ API in ``include/aerobulk.hpp``, Fortran shims in
``aerobulk_b200/fortran/``).  This Python package is a thin ctypes mirror of the
reference's ``aerobulk_model`` interface used by the tests and by ``bench.py``.
There is no CPU fallback: importing :mod:`aerobulk_b200.model` without the built
library raises, and every compute call fails without a CUDA device.
"""
from .model import (AerobulkError, aerobulk_model, aerobulk_model_device, aerobulk_model_f32, aerobulk_model_device_f32,
                    get_state, set_state, humidity_type,
                    last_error, launch_count, lib, measure_fp64_peak, nb_iter, reset, set_gdept, set_nb_iter,
                    set_rdt, set_stream, set_verbose, synchronize, use_skin, work_per_point, bytes_per_point, kernel_info,
                    set_nitend, turb, series, series_csv, series_device, SERIES_OUT, turb_ice, oce_ice,
                    set_ice_form_drag_per_point, ICE_ALGORITHMS, OCE_ICE_OUT, set_sort, flux_diagnostics,
                    diag_reduce_ops, diagnostics_summary, host_register, host_unregister, series_ice, SERIES_ICE_OUT, probe, set_devices, get_devices, shard_plan, init_local_stats_device,
                    init_from_gathered_stats, new_session, set_async, set_kernel_timing, kernel_times, aerobulk_init,
                    aerobulk_bye)

ALGORITHMS = ("coare3p0", "coare3p6", "ncar", "ecmwf", "andreas")
__all__ = ["ALGORITHMS", "AerobulkError", "aerobulk_model", "aerobulk_model_device", "aerobulk_model_f32",
           "aerobulk_model_device_f32", "get_state", "set_state", "humidity_type",
           "last_error", "launch_count", "lib", "measure_fp64_peak", "nb_iter", "reset", "set_gdept", "set_nb_iter",
           "set_rdt", "set_stream", "set_verbose", "synchronize", "use_skin", "work_per_point", "bytes_per_point", "kernel_info",
           "set_nitend", "turb", "series", "series_csv", "series_device", "SERIES_OUT", "turb_ice", "oce_ice",
           "set_ice_form_drag_per_point", "ICE_ALGORITHMS", "OCE_ICE_OUT", "set_sort", "flux_diagnostics",
           "diag_reduce_ops", "diagnostics_summary", "host_register", "host_unregister", "series_ice", "SERIES_ICE_OUT", "probe", "set_devices", "get_devices", "shard_plan", "init_local_stats_device",
           "init_from_gathered_stats", "new_session", "set_async", "set_kernel_timing", "kernel_times", "aerobulk_init", "aerobulk_bye"]
