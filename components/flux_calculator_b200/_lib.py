"""ctypes binding of libfluxcalc_b200.so (C ABI: include/fluxcalc.h).

The CUDA library is the product; this module only loads it.  There is no Python/NumPy fallback:
if the shared library is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FLUXCALC_LIB") or os.path.join(_HERE, "libfluxcalc_b200.so")   # env: tuning builds only

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "libfluxcalc_b200.so not found at %s -- build it with `make -C components/flux_calculator_b200/csrc` "
        "(or python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback." % LIB_PATH)

lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_int32_p = C.POINTER(C.c_int32)
ctx_p = C.c_void_p
dp = C.c_void_p          # double* passed as raw address (host or device)
i64 = C.c_int64
stream_t = C.c_void_p

# every exported symbol of include/fluxcalc.h: name -> (restype, argtypes)
SIGNATURES = {
    "fc_version": (C.c_int, []),
    "fc_last_error": (C.c_char_p, [ctx_p]),
    "fc_device_count": (C.c_int, []),
    "fc_var_index": (C.c_int, [C.c_char_p]),
    "fc_var_name": (C.c_char_p, [C.c_int]),
    "fc_current_month": (C.c_int, [C.c_int, i64]),
    "fc_shard_range": (C.c_int, [i64, C.c_int, C.c_int, i64, c_int64_p, c_int64_p]),
    "fc_device_malloc": (C.c_int, [C.c_int, i64, C.POINTER(C.c_void_p)]),
    "fc_device_free": (C.c_int, [C.c_int, C.c_void_p]),
    "fc_host_malloc_pinned": (C.c_int, [i64, C.POINTER(C.c_void_p)]),
    "fc_host_free_pinned": (C.c_int, [C.c_void_p]),
    "fc_memcpy_h2d": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, i64]),
    "fc_memcpy_d2h": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, i64]),
    "fc_device_memset": (C.c_int, [C.c_int, C.c_void_p, C.c_int, i64]),
    # level 1
    "fc_spec_vapor_surface_cclm": (C.c_int, [dp, dp, dp, dp, i64, c_double_p, c_double_p, stream_t]),
    "fc_flux_mass_evap_cclm": (C.c_int, [dp] * 8 + [i64, c_double_p, c_double_p, c_double_p, stream_t]),
    "fc_flux_mass_evap_mom5": (C.c_int, [dp] * 8 + [i64, stream_t]),
    "fc_flux_mass_evap_rco": (C.c_int, [dp] * 5 + [i64, stream_t]),
    "fc_flux_heat_latent_ice": (C.c_int, [dp, dp, i64, c_double_p, stream_t]),
    "fc_flux_heat_latent_water": (C.c_int, [dp, dp, i64, c_double_p, stream_t]),
    "fc_flux_heat_sensible_cclm": (C.c_int, [dp] * 9 + [i64, c_double_p, c_double_p, c_double_p, c_double_p, stream_t]),
    "fc_flux_heat_sensible_mom5": (C.c_int, [dp] * 9 + [i64, stream_t]),
    "fc_flux_heat_sensible_rco": (C.c_int, [dp] * 5 + [i64, stream_t]),
    "fc_flux_momentum_cclm": (C.c_int, [dp] * 8 + [i64, c_double_p, c_double_p, stream_t]),
    "fc_flux_momentum_mom5": (C.c_int, [dp] * 8 + [i64, stream_t]),
    "fc_flux_momentum_rco": (C.c_int, [dp] * 4 + [i64, stream_t]),
    "fc_flux_radiation_blackbody_StBo": (C.c_int, [dp, dp, i64, c_double_p, stream_t]),
    "fc_distribute_radiation_flux": (C.c_int, [dp, dp, dp, dp, i64, stream_t]),
    # level 2
    "fc_create": (C.c_int, [C.POINTER(ctx_p), c_int64_p, C.c_int, C.c_int]),
    "fc_destroy": (C.c_int, [ctx_p]),
    "fc_set_allocated": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "fc_create_from_namelist": (C.c_int, [C.POINTER(ctx_p), C.c_char_p, C.c_int, c_int64_p, C.c_int]),
    "fc_num_input_fields": (C.c_int, [ctx_p]),
    "fc_num_output_fields": (C.c_int, [ctx_p]),
    "fc_input_field": (C.c_int, [ctx_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                 C.POINTER(C.c_void_p), c_int64_p]),
    "fc_output_field": (C.c_int, [ctx_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_void_p), c_int64_p]),
    "fc_field_pointer": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p), c_int64_p]),
    "fc_namelist_registry": (C.c_int, [C.c_char_p, C.c_int, c_int64_p, C.c_char_p, i64]),
    "fc_mark_static": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "fc_mark_dirty": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int]),
    "fc_bind_thread_to_device_numa": (C.c_int, [C.c_int]),
    "fc_bind_field": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, dp, i64]),
    "fc_set_method": (C.c_int, [ctx_p, C.c_char_p, C.c_int, C.c_char_p]),
    "fc_set_distribute_shortwave": (C.c_int, [ctx_p, C.c_int]),
    "fc_set_corrections": (C.c_int, [ctx_p, C.c_int, dp, i64, C.c_int, C.c_int]),
    "fc_add_output_field": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int]),
    "fc_set_area": (C.c_int, [ctx_p, C.c_int, dp, i64]),
    "fc_set_time": (C.c_int, [ctx_p, i64]),
    "fc_prepare": (C.c_int, [ctx_p, C.c_int]),
    "fc_calc_spec_vapor_surface": (C.c_int, [ctx_p, C.c_int]),
    "fc_calc_flux_mass_evap": (C.c_int, [ctx_p]),
    "fc_calc_flux_heat_latent": (C.c_int, [ctx_p]),
    "fc_calc_flux_heat_sensible": (C.c_int, [ctx_p]),
    "fc_calc_flux_momentum_east": (C.c_int, [ctx_p, C.c_int]),
    "fc_calc_flux_momentum_north": (C.c_int, [ctx_p, C.c_int]),
    "fc_calc_flux_radiation_blackbody": (C.c_int, [ctx_p]),
    "fc_distribute_shortwave_radiation_flux": (C.c_int, [ctx_p]),
    "fc_average_across_surface_types": (C.c_int, [ctx_p, C.c_int, C.c_int]),
    "fc_step_early": (C.c_int, [ctx_p, i64]),
    "fc_step_normal": (C.c_int, [ctx_p, i64]),
    "fc_step_all": (C.c_int, [ctx_p, i64]),
    "fc_run_steps": (C.c_int, [ctx_p, i64, i64, C.c_int]),
    "fc_synchronize": (C.c_int, [ctx_p]),
    "fc_get_stream": (C.c_void_p, [ctx_p]),
    "fc_event_record": (C.c_int, [ctx_p, C.c_int]),
    "fc_event_elapsed_ms": (C.c_int, [ctx_p, c_double_p]),
    "fc_kernel_time_ms": (C.c_int, [ctx_p, c_double_p, c_int64_p]),
    "fc_set_option": (C.c_int, [ctx_p, C.c_char_p, i64]),
    "fc_get_info": (i64, [ctx_p, C.c_char_p]),
    "fc_get_diagnostics": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, c_double_p]),
    "fc_get_diagnostics_history": (C.c_int, [ctx_p, C.c_int, C.c_int, C.c_int, i64, i64, c_double_p]),
    "fc_comm_get_unique_id": (C.c_int, [C.c_char_p]),
    "fc_comm_init": (C.c_int, [ctx_p, C.c_char_p, C.c_int, C.c_int]),
    "fc_configure_from_namelist": (C.c_int, [ctx_p, C.c_char_p, C.c_int]),
    "fc_load_corrections": (C.c_int, [ctx_p, C.c_char_p, i64, C.c_int]),
    "fc_last_warning": (C.c_char_p, [ctx_p]),
    "fc_namelist_get": (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, c_int64_p, C.c_int, c_int64_p, C.c_char_p, C.c_int]),
    "fc_nc_read_var_double": (C.c_int, [C.c_char_p, C.c_char_p, i64, i64, c_double_p, c_double_p, C.POINTER(C.c_int)]),
    "fc_comm_p2p_handle": (C.c_int, [ctx_p, C.c_char_p]),
    "fc_comm_p2p_connect": (C.c_int, [ctx_p, C.c_char_p, C.c_int, C.c_int]),
    "fc_allreduce_diagnostics": (C.c_int, [ctx_p]),
    "fc_set_regrid_matrix": (C.c_int, [ctx_p, C.c_int, i64, c_int32_p, c_int32_p, c_double_p]),
    "fc_regrid": (C.c_int, [ctx_p, C.c_int, dp, dp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _f = getattr(lib, _name)     # AttributeError here == header/library mismatch: fail loudly
    _f.restype = _res
    _f.argtypes = _args


class FluxCalcError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("fluxcalc error %d: %s" % (code, message))
        self.code = code
        self.message = message


def check(rc, ctx=None):
    if rc != 0:
        msg = lib.fc_last_error(ctx)
        raise FluxCalcError(rc, msg.decode() if msg else "")
    return rc
