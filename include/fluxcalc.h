/*
 * fluxcalc.h -- C ABI of the B200-native flux calculator hot path (libfluxcalc_b200.so).
 *
 * Drop-in boundary for the per-exchange-grid-cell flux computation of
 * iow-esm/components.flux_calculator.  A Fortran host binds these entry points with
 * ISO_C_BINDING (shim sources: components/flux_calculator_b200/fortran/, recipe: INTEGRATION.md).
 * Plain pointers and sizes only; no C++/torch types.  Reference citations are file:line relative
 * to /root/reference/src.
 *
 * Two levels, mirroring the reference:
 *   Level 1  flux_lib: the 14 public routines of module flux_library (flux_lib/flux_library.F90:32-45),
 *            here in array ("batched") form with the SAME argument order as the Fortran dummies.
 *   Level 2  flux_calculator_calculate: the 9 per-step calculators (flux_calculator_calculate.F90:25-385)
 *            acting on a context that plays the role of local_field(0:MAX_SURFACE_TYPES,3)%var(35)
 *            (flux_calculator_basic.F90:86-103, flux_calculator.F90:159), plus fused per-phase steps
 *            replacing the inlined sequence of the time loop (flux_calculator.F90:902, :972-991 and the
 *            averaging triggers of the send loops :912-919, :1002-1009).
 *
 * Pointer arguments may be HOST pointers (pageable or pinned; staged through device mirrors, results
 * are valid on the host when the call returns) or DEVICE pointers (used in place, asynchronous on the
 * context's stream until fc_synchronize).  All arithmetic is binary64.  There is no CPU fallback: every
 * compute entry point returns FC_ERR_CUDA if no sm_100 device is usable.
 *
 * Every function returns an int status (0 = FC_OK), following the reference's only C-interop
 * precedent (pyfort/call_python.f90:13-16: non-zero C return -> stop).
 */
#ifndef FLUXCALC_H
#define FLUXCALC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FC_VERSION 100

/* limits: flux_calculator_basic.F90:27-32, :40 */
#define FC_MAX_SURFACE_TYPES 10
#define FC_MAX_VARNAMES      35

/* status codes */
enum {
    FC_OK = 0,
    FC_ERR_ARG = 1,      /* bad argument (index out of range, NULL, size mismatch) */
    FC_ERR_METHOD = 2,   /* unknown method string (prepare.F90:70-73 "Method ... is not known") */
    FC_ERR_MISSING = 3,  /* a required input is not bound (prepare.F90:29-33 "we are lacking ...") */
    FC_ERR_CUDA = 4,     /* CUDA runtime error / no usable device */
    FC_ERR_NCCL = 5,     /* NCCL error or libnccl.so.2 not loadable */
    FC_ERR_STATE = 6,    /* call sequence error (e.g. step before binding) */
    FC_ERR_NOMEM = 7
};

/* variable indices, 1-based, identical to idx_* (flux_calculator_basic.F90:42-51, :526-568) */
enum {
    FC_ALBE = 1, FC_ALBA, FC_AMOI, FC_AMOM, FC_FARE, FC_FICE, FC_PATM, FC_PSUR,
    FC_QATM, FC_TATM, FC_TSUR, FC_UATM, FC_VATM, FC_U10M, FC_V10M,
    FC_CMOM, FC_CMOI, FC_CHEA,
    FC_QSUR,
    FC_HLAT, FC_HSEN,
    FC_MEVA, FC_MPRE, FC_MRAI, FC_MSNO,
    FC_RBBR, FC_RLWD, FC_RLWU, FC_RSID, FC_RSIU, FC_RSIN, FC_RSDD, FC_RSDR,
    FC_UMOM, FC_VMOM
};

/* grids: 1 = t_grid, 2 = u_grid, 3 = v_grid (flux_calculator_basic.F90:63) */

typedef struct fc_context fc_context;
typedef void *fc_stream_t;          /* a cudaStream_t, or NULL for the default stream */

/* ------------------------------------------------------------------------------------------------
 * Utilities
 * ---------------------------------------------------------------------------------------------- */
int         fc_version(void);
/* last error message of ctx (or of the calling thread when ctx == NULL); never NULL */
const char *fc_last_error(const fc_context *ctx);
/* number of usable CUDA devices with compute capability 10.x; <0 on error */
int         fc_device_count(void);
/* idx (1..35) of a 4-character variable name, 0 if unknown (init_varname_idx, basic.F90:526-568) */
int         fc_var_index(const char *name);
const char *fc_var_name(int var_idx);
/* replaces pyfort/datetime_helpers.py:4-13 + call_python (calculate.F90:67-73):
 * month (1..12) of  date(init_date as YYYYMMDD) + seconds, proleptic Gregorian calendar */
int         fc_current_month(int init_date, int64_t seconds);
/* contiguous 1-D decomposition of n cells over nranks (decomp_def.F90:14-31 APPLE rule with the part
 * size rounded down to a multiple of `align` cells; the last rank takes the remainder) */
int         fc_shard_range(int64_t n, int rank, int nranks, int64_t align, int64_t *offset, int64_t *size);
/* device / pinned memory helpers for hosts that want device-resident fields */
int         fc_device_malloc(int device, int64_t nbytes, void **dptr);
int         fc_device_free(int device, void *dptr);
int         fc_host_malloc_pinned(int64_t nbytes, void **hptr);
int         fc_host_free_pinned(void *hptr);
int         fc_memcpy_h2d(int device, void *dst_device, const void *src_host, int64_t nbytes);
int         fc_memcpy_d2h(int device, void *dst_host, const void *src_device, int64_t nbytes);
/* write nbytes of zeros over a scratch device buffer (bench: L2 flush between timed steps) */
int         fc_device_memset(int device, void *dptr, int value, int64_t nbytes);

/* ------------------------------------------------------------------------------------------------
 * Level 1: flux_lib in array form.  Result array(s) first, then inputs in the Fortran dummy order,
 * then n, then the Fortran OPTIONAL constants as pointers to ONE host double (NULL = not PRESENT =
 * default_values, flux_lib/constants/flux_constants.F90:13-32), then the stream.
 * ---------------------------------------------------------------------------------------------- */
/* flux_lib/auxiliaries/flux_aux_vapor.F90:20-70 */
int fc_spec_vapor_surface_cclm(double *specific_vapor_content_surface, const double *fraction_ice,
                               const double *pressure_surface, const double *temperature_surface, int64_t n,
                               const double *gas_constant_air_new, const double *gas_constant_vapor_new,
                               fc_stream_t stream);
/* flux_lib/mass/flux_mass_evap.F90:22-85 */
int fc_flux_mass_evap_cclm(double *flux_mass_evap, const double *diffusion_coefficient_moisture,
                           const double *pressure_surface, const double *specific_vapor_content_atmos,
                           const double *specific_vapor_content_surface, const double *temperature_surface,
                           const double *u_atmos, const double *v_atmos, int64_t n, const double *u_min_evap_new,
                           const double *gas_constant_air_new, const double *gas_constant_vapor_new,
                           fc_stream_t stream);
/* flux_lib/mass/flux_mass_evap.F90:87-118 */
int fc_flux_mass_evap_mom5(double *flux_mass_evap, const double *diffusion_coefficient_moisture,
                           const double *pressure_surface, const double *specific_vapor_content_atmos,
                           const double *specific_vapor_content_surface, const double *temperature_surface,
                           const double *u_atmos, const double *v_atmos, int64_t n, fc_stream_t stream);
/* flux_lib/mass/flux_mass_evap.F90:120-158 */
int fc_flux_mass_evap_rco(double *flux_mass_evap, const double *specific_vapor_content_atmos,
                          const double *temperature_surface, const double *u_atmos, const double *v_atmos,
                          int64_t n, fc_stream_t stream);
/* flux_lib/heat/flux_heat_latent.F90:23-43 */
int fc_flux_heat_latent_ice(double *flux_heat_latent, const double *flux_mass_evap, int64_t n,
                            const double *latent_heat_sublimation_new, fc_stream_t stream);
/* flux_lib/heat/flux_heat_latent.F90:47-67 */
int fc_flux_heat_latent_water(double *flux_heat_latent, const double *flux_mass_evap, int64_t n,
                              const double *latent_heat_vaporization_new, fc_stream_t stream);
/* flux_lib/heat/flux_heat_sensible.F90:24-99 */
int fc_flux_heat_sensible_cclm(double *flux_heat_sensible, const double *diffusion_coefficient_moisture,
                               const double *pressure_atmos, const double *pressure_surface,
                               const double *specific_vapor_content_surface, const double *temperature_atmos,
                               const double *temperature_surface, const double *u_atmos, const double *v_atmos,
                               int64_t n, const double *heat_capacity_air_new, const double *u_min_evap_new,
                               const double *gas_constant_air_new, const double *gas_constant_vapor_new,
                               fc_stream_t stream);
/* flux_lib/heat/flux_heat_sensible.F90:101-135 */
int fc_flux_heat_sensible_mom5(double *flux_heat_sensible, const double *diffusion_coefficient_moisture,
                               const double *pressure_atmos, const double *pressure_surface,
                               const double *specific_vapor_content_surface, const double *temperature_atmos,
                               const double *temperature_surface, const double *u_atmos, const double *v_atmos,
                               int64_t n, fc_stream_t stream);
/* flux_lib/heat/flux_heat_sensible.F90:137-167 */
int fc_flux_heat_sensible_rco(double *flux_heat_sensible, const double *temperature_atmos,
                              const double *temperature_surface, const double *u_atmos, const double *v_atmos,
                              int64_t n, fc_stream_t stream);
/* flux_lib/momentum/flux_momentum.F90:22-76.  Either result may be NULL: the reference's callers pass
 * a scalar `dummy` for the component they do not need (calculate.F90:223,233,276,285). */
int fc_flux_momentum_cclm(double *flux_momentum_east, double *flux_momentum_north,
                          const double *diffusion_coefficient_momentum, const double *pressure_surface,
                          const double *specific_vapor_content_surface, const double *temperature_surface,
                          const double *u_atmos, const double *v_atmos, int64_t n,
                          const double *gas_constant_air_new, const double *gas_constant_vapor_new,
                          fc_stream_t stream);
/* flux_lib/momentum/flux_momentum.F90:78-108 */
int fc_flux_momentum_mom5(double *flux_momentum_east, double *flux_momentum_north,
                          const double *diffusion_coefficient_momentum, const double *pressure_surface,
                          const double *specific_vapor_content_surface, const double *temperature_surface,
                          const double *u_atmos, const double *v_atmos, int64_t n, fc_stream_t stream);
/* flux_lib/momentum/flux_momentum.F90:110-138 */
int fc_flux_momentum_rco(double *flux_momentum_east, double *flux_momentum_north, const double *u_atmos,
                         const double *v_atmos, int64_t n, fc_stream_t stream);
/* flux_lib/radiation/flux_radiation_blackbody.F90:22-42 */
int fc_flux_radiation_blackbody_StBo(double *flux_radiation_blackbody, const double *temperature_surface,
                                     int64_t n, const double *stefan_boltzmann_constant_new, fc_stream_t stream);
/* flux_lib/radiation/distribute_radiation_flux.F90:12-26 (the two albedo arguments are accepted and,
 * exactly as in the reference, unused; they may be NULL) */
int fc_distribute_radiation_flux(double *flux_radiation_surface_type, const double *flux_radiation_averaged,
                                 const double *albedo_averaged, const double *albedo_surface_type, int64_t n,
                                 fc_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Level 2: context == local_field registry + namelist method strings + bias corrections
 * ---------------------------------------------------------------------------------------------- */
/* grid_size[3] = local cell counts of t/u/v grid (flux_calculator_io.F90:77-107);
 * num_surface_types as in namelist /input/ (flux_calculator.F90:116); device = CUDA ordinal */
int fc_create(fc_context **ctx, const int64_t grid_size[3], int num_surface_types, int device);
int fc_destroy(fc_context *ctx);

/* local_field(surface_type, grid)%var(var_idx)%field => p(1:n)   (surface_type 0..10, grid 1..3).
 * Binding the same p to several slots reproduces the reference's pointer aliasing
 * (distribute_input_field basic.F90:334-358; method 'copy' prepare.F90:36-38; uniform outputs
 * basic.F90:203-207): one buffer.  A surface-type-0 slot counts as "%allocated" (own storage, the
 * condition average_across_surface_types tests, calculate.F90:376) iff no slot of a surface type >= 1
 * is bound to the same p.  p == NULL unbinds (NULLIFY).  n must equal grid_size[grid-1]. */
int fc_bind_field(fc_context *ctx, int surface_type, int grid, int var_idx, double *p, int64_t n);
/* local_field(surface_type, grid)%var(var_idx)%allocated (flux_calculator_basic.F90:88), the flag
 * average_across_surface_types tests (calculate.F90:376): 1 / 0 as the host's registry has it (set by allocate_localvar
 * basic.F90:299, do_prepare_calculation prepare.F90:41, add_output_field basic.F90:226,239,259; NOT set for pointer
 * aliases), -1 = infer from the aliasing as described above (the default).  The Fortran shim passes the real flag. */
int fc_set_allocated(fc_context *ctx, int surface_type, int grid, int var_idx, int allocated);

/* Host-pointer mode moves every bound array across PCIe every step unless told otherwise:
 *   fc_mark_static : the host will not rewrite this array between steps (the reference's own idiom: fields given as a
 *                    constant in the namelist, val_bottom_var_* / val_atmos_var_*, flux_calculator.F90:444-449, are
 *                    written once by init_localvar) -> uploaded once;  fc_mark_dirty: ... it did change, upload it again.
 *   option "download" = 1 : only fields registered with fc_add_output_field come back (what the reference hands to
 *                    oasis_put); intermediates such as QSUR stay on the device. */
int fc_mark_static(fc_context *ctx, int surface_type, int grid, int var_idx, int is_static);
int fc_mark_dirty(fc_context *ctx, int surface_type, int grid, int var_idx);
/* pins the calling thread to the CPUs next to `device` (sysfs local_cpulist of its PCI function), so that host buffers
 * allocated afterwards are local to the GPU's socket; one rank per GPU calls it before allocating its fields */
int fc_bind_thread_to_device_numa(int device);

/* Method string of one namelist array for one surface type (flux_calculator.F90:99-107):
 *   which = "which_spec_vapor_surface_t" | "_u" | "_v"  : none copy CCLM
 *           "which_flux_mass_evap"                      : none zero copy CCLM MOM5 RCO
 *           "which_flux_heat_latent"                    : none zero copy water ice
 *           "which_flux_heat_sensible"                  : none zero copy CCLM MOM5 RCO
 *           "which_flux_momentum"                       : none zero copy CCLM MOM5 RCO
 *           "which_flux_radiation_blackbody"            : none zero copy StBo
 * Unknown strings -> FC_ERR_METHOD (prepare.F90 "Method ... is not known"). */
int fc_set_method(fc_context *ctx, const char *which, int surface_type, const char *method);

/* distribute_shortwave_radiation_flux runs unconditionally in the reference (flux_calculator.F90:991)
 * and is undefined if RSDD(0)/RSDR(i) do not exist; here it runs iff enabled (default: enabled when
 * RSDD(0,t) and RSDR(i,t) are bound for every surface type at prepare time). on: 0 / 1 / -1 = auto */
int fc_set_distribute_shortwave(fc_context *ctx, int on);

/* bias_corrections.F90:26-33, :191: corrections(which, 12, n) in FORTRAN element order, i.e. element
 * (1, month, j) at corr[(month-1) + 12*(j-1)]; which = 1 (E_MASS_EVAP_CORRECTION); enabled ==
 * lcorrections(which); init_date = YYYYMMDD.  The array is copied (re-laid-out as [month][cell]). */
int fc_set_corrections(fc_context *ctx, int which, const double *corrections_fortran, int64_t n, int enabled,
                       int init_date);

/* add_output_field (basic.F90:170-283): registers a field that will be sent, so that the send loops'
 * averaging trigger (flux_calculator.F90:912-919, :1002-1009) is reproduced for surface_type 0.
 * early/normal phase is derived from the variable (RBBR,TSUR,FICE,ALBE are early: basic.F90:271-273). */
int fc_add_output_field(fc_context *ctx, int surface_type, int grid, int var_idx);

/* grid cell areas (grid_area, flux_calculator_io.F90:63-64) for the area-weighted diagnostics */
int fc_set_area(fc_context *ctx, int grid, const double *area, int64_t n);

/* current_step_time (flux_calculator_basic.F90:125), seconds since start of this instance */
int fc_set_time(fc_context *ctx, int64_t current_step_time);

/* prepare_* (flux_calculator_prepare.F90): validates methods against bound fields and builds the
 * launch plan.  strict != 0 reproduces the reference's required-input lists INCLUDING their quirks
 * (SURVEY App. F 1-3); strict == 0 checks what the formulae really read.  Called implicitly (strict=0)
 * by the first calculator/step call after any change. */
int fc_prepare(fc_context *ctx, int strict);

/* The 9 calculators, same names and meaning as flux_calculator_calculate.F90.  In host-pointer mode
 * each call uploads what it reads and downloads what it writes (host arrays stay authoritative). */
int fc_calc_spec_vapor_surface(fc_context *ctx, int which_grid);          /* :25-50 */
int fc_calc_flux_mass_evap(fc_context *ctx);                              /* :54-120 (incl. bias add) */
int fc_calc_flux_heat_latent(fc_context *ctx);                            /* :124-154 */
int fc_calc_flux_heat_sensible(fc_context *ctx);                          /* :156-208 */
int fc_calc_flux_momentum_east(fc_context *ctx, int which_grid);          /* :212-263 */
int fc_calc_flux_momentum_north(fc_context *ctx, int which_grid);         /* :265-316 */
int fc_calc_flux_radiation_blackbody(fc_context *ctx);                    /* :320-345 */
int fc_distribute_shortwave_radiation_flux(fc_context *ctx);              /* :347-364 */
int fc_average_across_surface_types(fc_context *ctx, int which_grid, int var_idx); /* :368-385 */

/* Fused phases of one coupling step (one kernel launch each):
 *   early  = flux_calculator.F90:902  + averaging of early outputs (:912-919)
 *   normal = flux_calculator.F90:972-991 + averaging of normal outputs (:1002-1009)
 *   all    = early then normal in a single pass (standalone / benchmark use)           */
int fc_step_early(fc_context *ctx, int64_t current_step_time);
int fc_step_normal(fc_context *ctx, int64_t current_step_time);
int fc_step_all(fc_context *ctx, int64_t current_step_time);
/* nsteps consecutive fc_step_all at t0, t0+dt, ... without host synchronisation in between (device-resident fields
 * only) -- the time loop of flux_calculator.F90:859-1028 for a host that keeps its fields on the device.  The steps of one
 * calendar month differ in nothing (the month selects the bias slab, calculate.F90:66-73): they are issued as replays of
 * one CUDA graph of 32 step launches per month, the remainder directly.  Results are bit-identical to nsteps calls of
 * fc_step_all.  With diagnostics only the LAST step's values can be read afterwards. */
int fc_run_steps(fc_context *ctx, int64_t t0, int64_t timestep, int nsteps);

int fc_synchronize(fc_context *ctx);
/* the context's CUDA stream (cudaStream_t), so callers can record events on the launching stream */
fc_stream_t fc_get_stream(fc_context *ctx);

/* CUDA-event timing on the context's stream: record event `which` (0 = start, 1 = stop); elapsed
 * waits for event 1.  fc_kernel_time_ms returns the summed device time and the number of fused-kernel
 * launches bracketed by event pairs since the last call (needs option "profile_kernel" = n >= 1: every n-th
 * fused launch is bracketed; an event between two launches disables their programmatic overlap). */
int fc_event_record(fc_context *ctx, int which);
int fc_event_elapsed_ms(fc_context *ctx, double *ms);
int fc_kernel_time_ms(fc_context *ctx, double *total_ms, int64_t *count);

/* options: "early_loads" (0/1, default 1: a step that directly follows another step of this context on its stream may
 *          fill its shared-memory ring before the previous step has finished -- steps write no input array; set
 *          "stream_touched" = 1 after enqueuing own work that writes bound arrays on fc_get_stream()),
 *          "dyn_min_tiles" (tiles per CTA from which the specialised kernel without diagnostics claims tiles dynamically;
 *          0 = default: 48 with one surface type, never with two),
 *          "force_generic" (0/1: use the op-list interpreter kernels instead of the fused kernel),
 *          "pin_host" (0/1: cudaHostRegister bound host arrays), "h2d_chunks" (pipeline depth of the
 *          host-pointer path), "diagnostics" (0 off, 1 area-weighted sums, 2 sums + min/max),
 *          "profile_kernel" (0 off, n: time every n-th fused launch), "staged" (specialised persistent kernel: 0 never,
 *          >= 1 (default) whenever the plan fits) */
int fc_set_option(fc_context *ctx, const char *name, int64_t value);
int64_t fc_get_info(const fc_context *ctx, const char *name);
/* info names: "launches" (kernel launches issued so far), "fused" (1 if the fused kernel serves
 * fc_step_*), "bytes_per_cell" (algorithmic bytes of fc_step_all per t/u/v cell triple),
 * "h2d_bytes_per_step", "d2h_bytes_per_step", "exact_path_calls" (threads of the specialised kernel / warps of the generic
 * fused kernel that left the lock-step fast path and recomputed their cells with the IEEE routines; 0 for physical data) */

/* ------------------------------------------------------------------------------------------------
 * Diagnostics (new, additive; reproduce the reference's debug "range =" lines, flux_calculator.F90:881,
 * :923,:951,:1013, plus area-weighted sums) and their multi-GPU reduction
 * ---------------------------------------------------------------------------------------------- */
/* after a step with option diagnostics >= 1: out[0] = sum_j area_j * x_j; with diagnostics == 2 also
 * out[1] = min_j x_j, out[2] = max_j x_j (NaN at level 1), over the LOCAL cells (or over all ranks after
 * fc_allreduce_diagnostics).  The sums are reproducible run to run (fixed trees); their last bits depend on the
 * summation tree, i.e. on the kernel that served the step and, in host-pointer mode, on the pipeline depth
 * ("h2d_chunks": one partial vector per chunk, combined in chunk order) -- min and max do not. */
int fc_get_diagnostics(fc_context *ctx, int surface_type, int grid, int var_idx, double out[3]);

#define FC_UNIQUE_ID_BYTES 128
int fc_comm_get_unique_id(char id[FC_UNIQUE_ID_BYTES]);                  /* ncclGetUniqueId */
int fc_comm_init(fc_context *ctx, const char id[FC_UNIQUE_ID_BYTES], int rank, int nranks);
int fc_allreduce_diagnostics(fc_context *ctx);                           /* ncclAllReduce sum / min / max */

/* Peer-memory exchange fused into the step (preferred on one NVLink/NVSwitch node, one process per GPU): every
 * rank exports its mailbox (fc_comm_p2p_handle), the host all-gathers the handles (MPI_Allgather of
 * FC_P2P_HANDLE_BYTES per rank) and passes the rank-ordered array to fc_comm_p2p_connect.  From then on
 * fc_allreduce_diagnostics launches nothing: it numbers an EXCHANGE, and the kernel that folds the step's diagnostics
 * rows (the next step's kernel, or a small fold kernel when the host asks first) stores the rank's vector into the
 * mailbox of every rank over NVLink as self-validating 8-byte words.  fc_get_diagnostics folds the ranks' records in
 * rank order (bit-identical on all ranks).  Mailboxes are keyed by exchange (slot = exchange mod 8): steps whose
 * global values nobody asked for post nothing, and the values of an exchange can be read until eight further
 * exchanges were issued.  If fc_comm_p2p_connect fails (no IPC / no peer access) use fc_comm_init (NCCL) instead. */
#define FC_P2P_HANDLE_BYTES 64
int fc_comm_p2p_handle(fc_context *ctx, char handle[FC_P2P_HANDLE_BYTES]);
int fc_comm_p2p_connect(fc_context *ctx, const char *handles /* nranks x FC_P2P_HANDLE_BYTES */, int rank, int nranks);

/* ------------------------------------------------------------------------------------------------
 * "Next" row: do_regridding (flux_calculator_basic.F90:463-522), COO sparse mat-vec with the
 * reference's sequential accumulation order per destination cell.  direction: 0 = u->t, 1 = v->t,
 * 2 = t->u, 3 = t->v.  Indices are 1-based like the Fortran arrays.
 * ---------------------------------------------------------------------------------------------- */
int fc_set_regrid_matrix(fc_context *ctx, int direction, int64_t num_elements, const int32_t *src_index,
                         const int32_t *dst_index, const double *weight);
/* dst(1:n_dst) = M * src for one array pair (host or device pointers) */
int fc_regrid(fc_context *ctx, int direction, double *dst, const double *src);

/* ------------------------------------------------------------------------------------------------
 * "Next" rows 3-4: the reference's own configuration files (host code, frontend.cu)
 * ---------------------------------------------------------------------------------------------- */
/* Reads the method selection of bottom model `bottom_model` (1-based first index of the which_* arrays,
 * flux_calculator.F90:99-107, NAMELIST /input/ :109-130) for surface types 1..S from a flux_calculator.nml and applies
 * it with fc_set_method (unset entries keep the declared default 'none'); reads &correctionsctl init_date and
 * lcorrections(1) (bias_corrections.F90:60-76) for fc_load_corrections.  Standard Fortran namelist input: comments,
 * r*c repeats, null values, element / section subscripts, array element order. */
int fc_configure_from_namelist(fc_context *ctx, const char *nml_path, int bottom_model);
/* The WHOLE &input group drives a context: what the reference's main program does between reading the namelist and the
 * time loop (flux_calculator.F90 STEP 1.4-1.7, :340-768, with allocate_localvar / init_localvar / distribute_input_field /
 * add_input_field / add_output_field / prepare_regridding of flux_calculator_basic.F90 and the prepare_* routines of
 * flux_calculator_prepare.F90, required-input quirks and error messages included).  The context owns the (page-locked)
 * host arrays a Fortran host would ALLOCATE; val_* constants are written once and marked static; 'copy' methods, uniform
 * outputs and the distribution of atmosphere fields over the surface types are pointer aliases; the %allocated flags, the
 * OASIS names (R/S + model letter + variable + surface type), the early flags and the regridding requests
 * (regrid_t_to_u ...) are the reference's.  A namelist the reference would stop on returns its message (FC_ERR_MISSING,
 * FC_ERR_METHOD); one it would run into undefined behaviour with (more sent fields than it allocates room for) is refused.
 * The host then fills the received fields (fc_input_field), sets regridding matrices if the namelist asks for any
 * (fc_set_regrid_matrix) and steps: fc_step_early / fc_step_normal regrid the received fields of their phase first
 * (do_regridding, flux_calculator.F90:891-896, :961-966) and computed ones after their calculator (:975-989). */
int fc_create_from_namelist(fc_context **ctx, const char *nml_path, int bottom_model, const int64_t grid_size[3], int device);
int fc_num_input_fields(const fc_context *ctx);       /* -1 unless created from a namelist */
int fc_num_output_fields(const fc_context *ctx);
/* field j (0-based, the reference's order): OASIS name (<= 8 characters + NUL), grid, early flag, surface type, variable
 * index, the bound host array and its length; any out pointer may be NULL */
int fc_input_field(fc_context *ctx, int j, char name[16], int *grid, int *early, int *surface_type, int *var_idx, double **field,
                   int64_t *n);
int fc_output_field(fc_context *ctx, int j, char name[16], int *grid, int *early, int *surface_type, int *var_idx, double **field,
                    int64_t *n);
int fc_field_pointer(fc_context *ctx, int surface_type, int grid, int var_idx, double **field, int64_t *n);
/* the registry that namelist describes as JSON text (no device needed): slots with storage group, %allocated, constant,
 * regridding flags; input and output field lists */
int fc_namelist_registry(const char *nml_path, int bottom_model, const int64_t grid_size[3], char *out, int64_t outlen);

/* initialize_bias_corrections (bias_corrections.F90:165-249): if lcorrections is set, reads variable 'mass_evap' of
 * <root_dir>/corrections/mass_evap-01.nc ... -12.nc (NetCDF classic CDF-1/2/5), cells [grid_offset, grid_offset + n_t),
 * replaces _FillValue by 0 and hands the (1,12,n_t) array to fc_set_corrections.  A month whose file, variable or
 * _FillValue attribute is missing stays zero with a line in fc_last_warning ("... Unset correction.", like the
 * reference).  reference_start_quirk = 1 reproduces the reference's use of the 0-based offset as 1-based NetCDF start
 * (SURVEY App. F-8: rank 0 reads nothing, other ranks read shifted by one cell); 0 reads the intended cells. */
int fc_load_corrections(fc_context *ctx, const char *root_dir, int64_t grid_offset, int reference_start_quirk);
const char *fc_last_warning(const fc_context *ctx);
/* the two parsers on their own (no device needed).  fc_namelist_get: value of element index[0..rank) (1-based) of an
 * array declared with `shape` (rank 0: scalar) as text; returns FC_NML_UNSET if the namelist does not set it.
 * fc_nc_read_var_double: elements [start0, start0+count) of a variable in row-major order converted to double;
 * returns 0, or 101 cannot open, 102 not NetCDF classic, 103 no such variable, 104 range. */
#define FC_NML_UNSET 20
int fc_namelist_get(const char *nml_path, const char *group, const char *name, const int64_t *shape, int rank,
                    const int64_t *index, char *out, int outlen);
int fc_nc_read_var_double(const char *path, const char *varname, int64_t start0, int64_t count, double *out,
                          double *fill_value, int *has_fill_value);

#ifdef __cplusplus
}
#endif
#endif /* FLUXCALC_H */
