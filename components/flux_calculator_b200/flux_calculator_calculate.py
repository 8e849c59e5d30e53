"""Host-side mirror of the reference's `MODULE flux_calculator_calculate`
(flux_calculator_calculate.F90:25-385) on top of the C ABI (include/fluxcalc.h).

`FluxCalculator` plays the role of the reference's module state: local_field(0:10,3)%var(35)
(flux_calculator.F90:159), the which_* method arrays of namelist /input/ (:99-107), the bias
corrections (bias_corrections.F90:26-33) and the send list.  The nine calculators keep the reference's
names and meaning; `step_early/step_normal/step_all` are the fused replacements of the inlined sequence
in the time loop (flux_calculator.F90:902, :972-991).  All arithmetic happens in the CUDA library.
"""
import ctypes as C

import numpy as np

from ._lib import lib, check, FluxCalcError
from .fields import IDX, VARNAMES, METHODS, var_index
from .memory import DeviceArray


class FluxCalculator:
    def __init__(self, grid_size, num_surface_types=1, device=0):
        gs = (C.c_int64 * 3)(*[int(x) for x in grid_size])
        self._ctx = C.c_void_p()
        check(lib.fc_create(C.byref(self._ctx), gs, int(num_surface_types), int(device)))
        self.grid_size = tuple(int(x) for x in grid_size)
        self.num_surface_types = int(num_surface_types)
        self.device = int(device)
        self._keep = {}       # (type, grid, idx) -> array object (keeps host memory alive, like the Fortran host)
        self._misc = []

    # ---- life cycle -------------------------------------------------------------------------
    def close(self):
        if self._ctx:
            lib.fc_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        return check(rc, self._ctx)

    # ---- registry ---------------------------------------------------------------------------
    def bind_field(self, surface_type, grid, var, array):
        """local_field(surface_type, grid)%var(idx_<var>)%field => array   (None: nullify)"""
        idx = var_index(var)
        if array is None:
            self._check(lib.fc_bind_field(self._ctx, surface_type, grid, idx, None, 0))
            self._keep.pop((surface_type, grid, idx), None)
            return
        if isinstance(array, DeviceArray):
            ptr, n = array.ptr, array.n
        else:
            if not (isinstance(array, np.ndarray) and array.dtype == np.float64 and array.flags.c_contiguous):
                raise TypeError("fields must be contiguous float64 NumPy arrays or DeviceArrays")
            ptr, n = array.ctypes.data, array.size
        self._check(lib.fc_bind_field(self._ctx, surface_type, grid, idx, ptr, n))
        self._keep[(surface_type, grid, idx)] = array

    def set_allocated(self, surface_type, grid, var, allocated):
        """local_field(surface_type, grid)%var(idx_<var>)%allocated as the host's registry has it (None: infer)"""
        self._check(lib.fc_set_allocated(self._ctx, surface_type, grid, var_index(var),
                                         -1 if allocated is None else int(bool(allocated))))

    def mark_static(self, surface_type, grid, var, is_static=True):
        """the host does not rewrite this bound array between steps (a namelist constant): uploaded once"""
        self._check(lib.fc_mark_static(self._ctx, surface_type, grid, var_index(var), int(bool(is_static))))

    def mark_dirty(self, surface_type, grid, var):
        self._check(lib.fc_mark_dirty(self._ctx, surface_type, grid, var_index(var)))

    def field(self, surface_type, grid, var):
        return self._keep.get((surface_type, grid, var_index(var)))

    def set_method(self, which, surface_type, method):
        self._check(lib.fc_set_method(self._ctx, which.encode(), surface_type, method.encode()))

    def set_distribute_shortwave(self, on):
        self._check(lib.fc_set_distribute_shortwave(self._ctx, -1 if on is None else int(bool(on))))

    def set_corrections(self, corrections, enabled=True, init_date=19610101):
        """corrections: Fortran array corrections(1,12,n) flattened in Fortran order, i.e. shape (n,12) C-order,
        NumPy or DeviceArray (bias_corrections.F90:29-30,191)"""
        if corrections is None:
            self._check(lib.fc_set_corrections(self._ctx, 1, None, 0, 0, int(init_date)))
            return
        if isinstance(corrections, DeviceArray):
            ptr, n = corrections.ptr, corrections.n // 12
        else:
            corrections = np.ascontiguousarray(corrections, dtype=np.float64)
            ptr, n = corrections.ctypes.data, corrections.size // 12
        self._misc.append(corrections)
        self._check(lib.fc_set_corrections(self._ctx, 1, ptr, n, int(bool(enabled)), int(init_date)))

    def add_output_field(self, surface_type, grid, var):
        self._check(lib.fc_add_output_field(self._ctx, surface_type, grid, var_index(var)))

    def set_area(self, grid, area):
        if isinstance(area, DeviceArray):
            ptr, n = area.ptr, area.n
        else:
            area = np.ascontiguousarray(area, dtype=np.float64)
            ptr, n = area.ctypes.data, area.size
        self._misc.append(area)
        self._check(lib.fc_set_area(self._ctx, grid, ptr, n))

    def set_time(self, seconds):
        self._check(lib.fc_set_time(self._ctx, int(seconds)))

    def set_option(self, name, value):
        self._check(lib.fc_set_option(self._ctx, name.encode(), int(value)))

    def info(self, name):
        return int(lib.fc_get_info(self._ctx, name.encode()))

    def prepare(self, strict=False):
        self._check(lib.fc_prepare(self._ctx, int(bool(strict))))

    # ---- the nine calculators (same names as the reference) ---------------------------------
    def calc_spec_vapor_surface(self, which_grid):
        self._check(lib.fc_calc_spec_vapor_surface(self._ctx, which_grid))

    def calc_flux_mass_evap(self):
        self._check(lib.fc_calc_flux_mass_evap(self._ctx))

    def calc_flux_heat_latent(self):
        self._check(lib.fc_calc_flux_heat_latent(self._ctx))

    def calc_flux_heat_sensible(self):
        self._check(lib.fc_calc_flux_heat_sensible(self._ctx))

    def calc_flux_momentum_east(self, which_grid=2):
        self._check(lib.fc_calc_flux_momentum_east(self._ctx, which_grid))

    def calc_flux_momentum_north(self, which_grid=3):
        self._check(lib.fc_calc_flux_momentum_north(self._ctx, which_grid))

    def calc_flux_radiation_blackbody(self):
        self._check(lib.fc_calc_flux_radiation_blackbody(self._ctx))

    def distribute_shortwave_radiation_flux(self):
        self._check(lib.fc_distribute_shortwave_radiation_flux(self._ctx))

    def average_across_surface_types(self, which_grid, var):
        self._check(lib.fc_average_across_surface_types(self._ctx, which_grid, var_index(var)))

    # ---- fused phases -------------------------------------------------------------------------
    def step_early(self, current_step_time=0):
        self._check(lib.fc_step_early(self._ctx, int(current_step_time)))

    def step_normal(self, current_step_time=0):
        self._check(lib.fc_step_normal(self._ctx, int(current_step_time)))

    def step_all(self, current_step_time=0):
        self._check(lib.fc_step_all(self._ctx, int(current_step_time)))

    def run_steps(self, t0, timestep, nsteps):
        self._check(lib.fc_run_steps(self._ctx, int(t0), int(timestep), int(nsteps)))

    def synchronize(self):
        self._check(lib.fc_synchronize(self._ctx))

    def event_record(self, which):
        self._check(lib.fc_event_record(self._ctx, int(which)))

    def event_elapsed_ms(self):
        ms = C.c_double()
        self._check(lib.fc_event_elapsed_ms(self._ctx, C.byref(ms)))
        return ms.value

    def kernel_time_ms(self):
        ms, cnt = C.c_double(), C.c_int64()
        self._check(lib.fc_kernel_time_ms(self._ctx, C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    @property
    def stream(self):
        return lib.fc_get_stream(self._ctx)

    # ---- diagnostics / multi-GPU -------------------------------------------------------------
    def diagnostics(self, surface_type, grid, var):
        out = (C.c_double * 3)()
        self._check(lib.fc_get_diagnostics(self._ctx, surface_type, grid, var_index(var), out))
        return tuple(out)

    def diagnostics_history(self, surface_type, grid, var, first=None, count=None):
        """(count, 3) float64 array: row j = diagnostics(surface_type, grid, var) as it was right after step first + j
        (NaN where that step did not compute the field); needs option "diagnostics_history" > 0.  Default: every
        retained step; with only count given, the last count steps."""
        total = self.info("diagnostics_history_steps")
        if first is None:
            first = max(0, total - self.info("diagnostics_history")) if count is None else total - count
        if count is None:
            count = total - first
        out = np.empty((max(int(count), 0), 3), dtype=np.float64)
        self._check(lib.fc_get_diagnostics_history(self._ctx, surface_type, grid, var_index(var), int(first), int(count),
                                                   out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def comm_init(self, unique_id, rank, nranks):
        self._check(lib.fc_comm_init(self._ctx, unique_id, rank, nranks))

    def comm_p2p_handle(self):
        """CUDA IPC handle of this rank's diagnostics mailbox (64 bytes); all-gather them and call comm_p2p_connect"""
        buf = C.create_string_buffer(64)
        self._check(lib.fc_comm_p2p_handle(self._ctx, buf))
        return buf.raw

    def comm_p2p_connect(self, handles, rank, nranks):
        """handles: the ranks' 64-byte handles in rank order; afterwards every step posts its diagnostics to all ranks"""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * nranks
        self._check(lib.fc_comm_p2p_connect(self._ctx, blob, rank, nranks))

    def allreduce_diagnostics(self):
        self._check(lib.fc_allreduce_diagnostics(self._ctx))

    # ---- the reference's configuration files ("next" rows 3-4) ---------------------------------
    def configure_from_namelist(self, nml_path, bottom_model=1):
        """&input which_* and &correctionsctl of a flux_calculator.nml (flux_calculator.F90:99-130, bias_corrections.F90:60-76)"""
        self._check(lib.fc_configure_from_namelist(self._ctx, str(nml_path).encode(), int(bottom_model)))

    def load_corrections(self, root_dir, grid_offset=0, reference_start_quirk=False):
        """initialize_bias_corrections (bias_corrections.F90:165-249); returns the loader's warnings"""
        self._check(lib.fc_load_corrections(self._ctx, str(root_dir).encode(), int(grid_offset), int(bool(reference_start_quirk))))
        return lib.fc_last_warning(self._ctx).decode()

    # ---- regridding ("next" row) ---------------------------------------------------------------
    def set_regrid_matrix(self, direction, src_index, dst_index, weight):
        s = np.ascontiguousarray(src_index, dtype=np.int32)
        d = np.ascontiguousarray(dst_index, dtype=np.int32)
        w = np.ascontiguousarray(weight, dtype=np.float64)
        self._check(lib.fc_set_regrid_matrix(self._ctx, direction, s.size, s.ctypes.data_as(C.POINTER(C.c_int32)),
                                             d.ctypes.data_as(C.POINTER(C.c_int32)),
                                             w.ctypes.data_as(C.POINTER(C.c_double))))

    def regrid(self, direction, dst, src):
        dp = dst.ptr if isinstance(dst, DeviceArray) else dst.ctypes.data
        sp = src.ptr if isinstance(src, DeviceArray) else src.ctypes.data
        self._check(lib.fc_regrid(self._ctx, direction, dp, sp))


def namelist_registry(nml_path, bottom_model, grid_size):
    """the registry flux_calculator.nml describes (what fc_create_from_namelist builds), parsed from the library's JSON text"""
    import json
    gs = (C.c_int64 * 3)(*[int(x) for x in grid_size])
    buf = C.create_string_buffer(1 << 22)
    check(lib.fc_namelist_registry(str(nml_path).encode(), int(bottom_model), gs, buf, len(buf)))
    return json.loads(buf.value.decode())


class NamelistCalculator(FluxCalculator):
    """a FluxCalculator whose registry, methods and field lists come from a flux_calculator.nml (fc_create_from_namelist):
    the library owns the host arrays; `inputs` / `outputs` list (name, grid, early, surface type, variable, NumPy view)"""

    def __init__(self, nml_path, grid_size, bottom_model=1, device=0):
        gs = (C.c_int64 * 3)(*[int(x) for x in grid_size])
        self._ctx = C.c_void_p()
        check(lib.fc_create_from_namelist(C.byref(self._ctx), str(nml_path).encode(), int(bottom_model), gs, int(device)))
        self.grid_size = tuple(int(x) for x in grid_size)
        self.device = int(device)
        self._keep, self._misc = {}, []
        self.inputs = self._fields(lib.fc_num_input_fields, lib.fc_input_field)
        self.outputs = self._fields(lib.fc_num_output_fields, lib.fc_output_field)
        self.num_surface_types = max([f["type"] for f in self.inputs + self.outputs] + [1])

    def _fields(self, count, getter):
        res = []
        for j in range(count(self._ctx)):
            name = C.create_string_buffer(16)
            g, e, t, v = C.c_int(), C.c_int(), C.c_int(), C.c_int()
            p, n = C.c_void_p(), C.c_int64()
            self._check(getter(self._ctx, j, name, C.byref(g), C.byref(e), C.byref(t), C.byref(v), C.byref(p), C.byref(n)))
            res.append({"name": name.value.decode(), "grid": g.value, "early": bool(e.value), "type": t.value, "var": VARNAMES[v.value - 1],
                        "array": self._view(p.value, n.value)})
        return res

    @staticmethod
    def _view(ptr, n):
        if not ptr or n <= 0:
            return np.empty(0)
        return np.frombuffer((C.c_double * n).from_address(ptr), dtype=np.float64, count=n)

    def array(self, surface_type, grid, var):
        p, n = C.c_void_p(), C.c_int64()
        self._check(lib.fc_field_pointer(self._ctx, surface_type, grid, var_index(var), C.byref(p), C.byref(n)))
        return self._view(p.value, n.value) if p.value else None


def namelist_get(nml_path, group, name, shape=(), index=()):
    """one element of a namelist array (1-based index, declared shape) as text, None if the namelist does not set it"""
    rank = len(shape)
    shp = (C.c_int64 * max(rank, 1))(*shape)
    idx = (C.c_int64 * max(rank, 1))(*index)
    out = C.create_string_buffer(256)
    rc = lib.fc_namelist_get(str(nml_path).encode(), group.encode(), name.encode(), shp, rank, idx, out, 256)
    if rc == 20:
        return None
    check(rc)
    return out.value.decode()


def nc_read_var(path, varname, start, count):
    """elements [start, start+count) of a NetCDF classic variable as float64, plus its _FillValue (or None)"""
    out = np.empty(count, dtype=np.float64)
    fill, has = C.c_double(), C.c_int()
    rc = lib.fc_nc_read_var_double(str(path).encode(), varname.encode(), int(start), int(count),
                                   out.ctypes.data_as(C.POINTER(C.c_double)), C.byref(fill), C.byref(has))
    if rc:
        raise OSError(rc, lib.fc_last_error(None).decode())
    return out, (fill.value if has.value else None)


def comm_get_unique_id():
    buf = C.create_string_buffer(128)
    check(lib.fc_comm_get_unique_id(buf))
    return buf.raw


def current_month(init_date, seconds):
    """pyfort/datetime_helpers.py:4-13 replacement"""
    return int(lib.fc_current_month(int(init_date), int(seconds)))


def shard_range(n, rank, nranks, align=32):
    off, size = C.c_int64(), C.c_int64()
    check(lib.fc_shard_range(int(n), int(rank), int(nranks), int(align), C.byref(off), C.byref(size)))
    return off.value, size.value
