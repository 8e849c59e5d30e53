// context.cu -- Level 2 of the C ABI: the context (local_field registry), the plan builder that turns
// namelist method strings + bound fields into launch plans, and the per-step calculators.
// Reference paths relative to /root/reference/src.
#include "context.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cctype>
#include <sched.h>
#include <set>

using namespace fc;

namespace fc {
thread_local std::string g_last_error;
int nccl_allreduce_diag(fc_context *ctx);   // nccl_dyn.cu
void p2p_destroy(fc_context *ctx);          // p2p_comm.cu
void p2p_make_post(fc_context *ctx, PeerPost &post);
int p2p_fetch(fc_context *ctx, double *planes, int n_active, int level);
void nccl_destroy(fc_context *ctx);
}  // namespace fc

// ---------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------
static const char *kVarNames[FC_MAX_VARNAMES + 1] = {
    "",     "ALBE", "ALBA", "AMOI", "AMOM", "FARE", "FICE", "PATM", "PSUR", "QATM", "TATM", "TSUR",
    "UATM", "VATM", "U10M", "V10M", "CMOM", "CMOI", "CHEA", "QSUR", "HLAT", "HSEN", "MEVA", "MPRE",
    "MRAI", "MSNO", "RBBR", "RLWD", "RLWU", "RSID", "RSIU", "RSIN", "RSDD", "RSDR", "UMOM", "VMOM"};   // basic.F90:43-51
static const char *kGridNames[4] = {"", "t_grid", "u_grid", "v_grid"};                                 // basic.F90:63

namespace fc {
int fail(fc_context *ctx, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (ctx) ctx->err = buf;
    return code;
}

int classify_pointer(const void *p, bool *is_device, bool *is_pinned, int *device)
{
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *is_device = false;
        *is_pinned = false;
        return 0;
    }
    *is_device = (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged);
    *is_pinned = (a.type == cudaMemoryTypeHost);
    if (device && *is_device) *device = a.device;
    return 0;
}
}  // namespace fc

static int parse_method(const char *s)
{
    // trailing blanks are insignificant (Fortran trim(method), calculate.F90:38)
    std::string m(s ? s : "");
    while (!m.empty() && m.back() == ' ') m.pop_back();
    if (m == "none") return M_NONE;
    if (m == "zero") return M_ZERO;
    if (m == "copy") return M_COPY;
    if (m == "CCLM") return M_CCLM;
    if (m == "MOM5") return M_MOM5;
    if (m == "RCO") return M_RCO;
    if (m == "water") return M_WATER;
    if (m == "ice") return M_ICE;
    if (m == "StBo") return M_STBO;
    return M_INVALID;
}

static bool method_allowed(int q, int m)
{
    switch (q) {
        case Q_QSUR_T: case Q_QSUR_U: case Q_QSUR_V: return m == M_NONE || m == M_COPY || m == M_CCLM;       // prepare.F90:57-73
        case Q_MEVA: case Q_HSEN: case Q_MOM:
            return m == M_NONE || m == M_ZERO || m == M_COPY || m == M_CCLM || m == M_MOM5 || m == M_RCO;   // :86-114
        case Q_HLAT: return m == M_NONE || m == M_ZERO || m == M_COPY || m == M_WATER || m == M_ICE;         // :130-144
        case Q_RBBR: return m == M_NONE || m == M_ZERO || m == M_COPY || m == M_STBO;                        // :288-298
    }
    return false;
}

static inline int slot_of(const fc_context *c, int i, int g, int idx) { return c->slot[i][g][idx]; }

// "%allocated" (basic.F90:88) of a surface-type-0 slot: it owns its storage iff no slot of a surface type
// >= 1 is bound to the same array (otherwise it is a pointer alias such as a uniform output,
// basic.F90:203-207, or an atmosphere field distributed to the surface types, basic.F90:349)
static bool slot_owns(const fc_context *c, int i, int g, int idx)
{
    const int b = c->slot[i][g][idx];
    if (b < 0) return false;
    if (c->alloc_flag[i][g][idx] >= 0) return c->alloc_flag[i][g][idx] != 0;      // the host said so (fc_set_allocated)
    for (int ii = 1; ii <= FC_MAX_SURFACE_TYPES; ++ii)
        for (int gg = 1; gg <= 3; ++gg)
            for (int v = 1; v <= FC_MAX_VARNAMES; ++v)
                if (!(ii == i && gg == g && v == idx) && c->slot[ii][gg][v] == b) return false;
    return true;
}

// ---------------------------------------------------------------------------------------------
// utilities of the ABI
// ---------------------------------------------------------------------------------------------
extern "C" int fc_version(void) { return FC_VERSION; }

extern "C" const char *fc_last_error(const fc_context *ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

extern "C" int fc_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, d) == cudaSuccess && p.major == 10) ++ok;
    }
    return ok;
}

extern "C" int fc_var_index(const char *name)
{
    if (!name) return 0;
    for (int i = 1; i <= FC_MAX_VARNAMES; ++i)
        if (strncmp(name, kVarNames[i], 4) == 0 && (name[4] == 0 || name[4] == ' ')) return i;
    return 0;
}

extern "C" const char *fc_var_name(int idx) { return (idx >= 1 && idx <= FC_MAX_VARNAMES) ? kVarNames[idx] : ""; }

// days since 1970-01-01 of a proleptic Gregorian civil date
static int64_t days_from_civil(int64_t y, int m, int d)
{
    y -= m <= 2;
    const int64_t era = (y >= 0 ? y : y - 399) / 400;
    const int64_t yoe = y - era * 400;
    const int64_t doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
    const int64_t doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
    return era * 146097 + doe - 719468;
}

// pyfort/datetime_helpers.py:4-13 without Python: strptime(init_date, "%Y%m%d") + timedelta(seconds) -> month
extern "C" int fc_current_month(int init_date, int64_t seconds)
{
    const int y = init_date / 10000, m = (init_date / 100) % 100, d = init_date % 100;
    // datetime.strptime(init_date, "%Y%m%d") raises on a date that does not exist (year 1..9999, day within the month)
    static const int mdays[12] = {31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31};
    if (init_date < 10101 || y < 1 || y > 9999 || m < 1 || m > 12 || d < 1) return 0;
    const bool leap = (y % 4 == 0 && y % 100 != 0) || y % 400 == 0;
    if (d > mdays[m - 1] + ((m == 2 && leap) ? 1 : 0)) return 0;
    const int64_t shift = seconds >= 0 ? seconds / 86400 : -((-seconds + 86399) / 86400);
    const int64_t z = days_from_civil(y, m, d) + shift + 719468;
    const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
    const int64_t doe = z - era * 146097;
    const int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    const int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const int64_t mp = (5 * doy + 2) / 153;
    return (int)(mp < 10 ? mp + 3 : mp - 9);
}

// decomp_def.F90:14-31 (APPLE) on a 1-D grid; part size rounded down to `align` cells so that every
// shard start stays vector aligned; the last rank takes the remainder (decomp_def.F90:27-30)
extern "C" int fc_shard_range(int64_t n, int rank, int nranks, int64_t align, int64_t *offset, int64_t *size)
{
    if (n < 0 || nranks < 1 || rank < 0 || rank >= nranks || !offset || !size) return fail(nullptr, FC_ERR_ARG, "fc_shard_range: bad argument");
    if (align < 1) align = 1;
    int64_t part = n / nranks;
    // the APPLE rule never leaves a rank empty when n >= nranks (decomp_def.F90:23-30): if rounding to `align` would, round to
    // the largest power-of-two fraction of it that does not (down to single cells; such starts take the guarded tile path)
    while (align > 1 && part - part % align == 0 && part > 0) align /= 2;
    part -= part % align;
    *offset = rank * part;
    *size = rank < nranks - 1 ? part : n - rank * part;
    return FC_OK;
}

extern "C" int fc_device_malloc(int device, int64_t nbytes, void **dptr)
{
    if (!dptr || nbytes < 0) return fail(nullptr, FC_ERR_ARG, "fc_device_malloc: bad argument");
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, cudaMalloc(dptr, (size_t)std::max<int64_t>(nbytes, 8)));
    return FC_OK;
}
extern "C" int fc_device_free(int device, void *dptr)
{
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, cudaFree(dptr));
    return FC_OK;
}
extern "C" int fc_host_malloc_pinned(int64_t nbytes, void **hptr)
{
    if (!hptr || nbytes < 0) return fail(nullptr, FC_ERR_ARG, "fc_host_malloc_pinned: bad argument");
    CUDA_TRY(nullptr, cudaHostAlloc(hptr, (size_t)std::max<int64_t>(nbytes, 8), cudaHostAllocPortable));
    return FC_OK;
}
extern "C" int fc_host_free_pinned(void *hptr)
{
    CUDA_TRY(nullptr, cudaFreeHost(hptr));
    return FC_OK;
}
extern "C" int fc_memcpy_h2d(int device, void *dst, const void *src, int64_t nbytes)
{
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, cudaMemcpy(dst, src, (size_t)nbytes, cudaMemcpyHostToDevice));
    return FC_OK;
}
extern "C" int fc_memcpy_d2h(int device, void *dst, const void *src, int64_t nbytes)
{
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, cudaMemcpy(dst, src, (size_t)nbytes, cudaMemcpyDeviceToHost));
    return FC_OK;
}
extern "C" int fc_device_memset(int device, void *dptr, int value, int64_t nbytes)
{
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, cudaMemsetAsync(dptr, value, (size_t)nbytes, nullptr));
    return FC_OK;
}

// ---------------------------------------------------------------------------------------------
// context life cycle and registry
// ---------------------------------------------------------------------------------------------
extern "C" int fc_create(fc_context **out, const int64_t grid_size[3], int num_surface_types, int device)
{
    if (!out || !grid_size) return fail(nullptr, FC_ERR_ARG, "fc_create: NULL argument");
    if (num_surface_types < 1 || num_surface_types > FC_MAX_SURFACE_TYPES)
        return fail(nullptr, FC_ERR_ARG, "fc_create: num_surface_types must be 1..%d (MAX_SURFACE_TYPES, basic.F90:28)",
                    FC_MAX_SURFACE_TYPES);
    for (int g = 0; g < 3; ++g)
        if (grid_size[g] < 0) return fail(nullptr, FC_ERR_ARG, "fc_create: negative grid size");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, FC_ERR_CUDA, "fc_create: no CUDA device available (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev) return fail(nullptr, FC_ERR_ARG, "fc_create: device %d out of range (0..%d)", device, ndev - 1);
    cudaDeviceProp prop;
    CUDA_TRY(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(nullptr, FC_ERR_CUDA, "fc_create: device %d is sm_%d%d; the kernels are built for sm_100a only", device,
                    prop.major, prop.minor);
    CUDA_TRY(nullptr, cudaSetDevice(device));
    fc_context *c = new fc_context();
    c->device = device;
    c->S = num_surface_types;
    for (int g = 1; g <= 3; ++g) c->n[g] = grid_size[g - 1];
    for (auto &a : c->slot)
        for (auto &b : a)
            for (auto &v : b) v = -1;
    for (auto &a : c->alloc_flag)
        for (auto &b : a)
            for (auto &v : b) v = -1;
    for (auto &q : c->method)
        for (auto &m : q) m = M_NONE;   // namelist defaults 'none' (flux_calculator.F90:99-107)
    c->consts = make_consts();
    CUDA_TRY(nullptr, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    for (int k = 0; k < 3; ++k) {
        CUDA_TRY(nullptr, cudaStreamCreateWithFlags(&c->pipe[k], cudaStreamNonBlocking));
        CUDA_TRY(nullptr, cudaEventCreateWithFlags(&c->pipe_done[k], cudaEventDisableTiming));
    }
    *out = c;
    return FC_OK;
}

static void free_regrid(RegridMatrix &m)
{
    cudaFree(m.row_ptr);
    cudaFree(m.src_idx);
    cudaFree(m.weight);
    m = RegridMatrix();
}

extern "C" int fc_destroy(fc_context *c)
{
    if (!c) return FC_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    nccl_destroy(c);
    for (auto &b : c->bufs) {
        if (b.registered) cudaHostUnregister(b.user);
        if (!b.user_is_device && b.dev) cudaFree(b.dev);
    }
    cudaFree(c->corr_dev);
    for (int g = 1; g <= 3; ++g)
        if (c->area_owned[g]) cudaFree(c->area_dev[g]);
    cudaFree(c->diag_partials);
    cudaFree(c->diag_chunk_out);
    cudaFree(c->tile_ctr);
    cudaFree(c->chain_done);
    for (auto &g : c->step_graph)
        if (g) cudaGraphExecDestroy(g);
    p2p_destroy(c);
    for (int b = 0; b < 2; ++b) {
        cudaFree(c->diag_buf[b]);
        if (c->ev_fin[b]) cudaEventDestroy(c->ev_fin[b]);
        if (c->ev_comm[b]) cudaEventDestroy(c->ev_comm[b]);
    }
    if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
    if (c->diag_host) cudaFreeHost(c->diag_host);
    for (auto &m : c->regrid) free_regrid(m);
    for (cudaEvent_t e : c->prof_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : c->user_ev)
        if (e) cudaEventDestroy(e);
    for (int k = 0; k < 3; ++k) {
        cudaStreamDestroy(c->pipe[k]);
        cudaEventDestroy(c->pipe_done[k]);
    }
    cudaStreamDestroy(c->stream);
    if (c->sa) {
        standalone_free(*c->sa);
        delete c->sa;
    }
    delete c;
    return FC_OK;
}

static void release_buffer(fc_context *c, int b)
{
    Buffer &B = c->bufs[b];
    if (--B.refs > 0) return;
    if (B.registered) cudaHostUnregister(B.user);
    if (!B.user_is_device && B.dev) cudaFree(B.dev);
    B = Buffer();   // tombstone (indices of other buffers stay valid)
}

extern "C" int fc_bind_field(fc_context *c, int i, int g, int idx, double *p, int64_t n)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "fc_bind_field: NULL context");
    if (i < 0 || i > FC_MAX_SURFACE_TYPES || g < 1 || g > 3 || idx < 1 || idx > FC_MAX_VARNAMES)
        return fail(c, FC_ERR_ARG, "fc_bind_field: index out of range (surface_type %d, grid %d, var %d)", i, g, idx);
    cudaSetDevice(c->device);
    c->dirty = true;
    if (c->slot[i][g][idx] >= 0) {
        release_buffer(c, c->slot[i][g][idx]);
        c->slot[i][g][idx] = -1;
    }
    if (!p) {      // NULLIFY
        c->alloc_flag[i][g][idx] = -1;
        return FC_OK;
    }
    if (n != c->n[g])
        return fail(c, FC_ERR_ARG, "fc_bind_field: %s on %s has %lld elements, grid_size is %lld", kVarNames[idx], kGridNames[g],
                    (long long)n, (long long)c->n[g]);
    for (size_t b = 0; b < c->bufs.size(); ++b)
        if (c->bufs[b].user == p) {
            if (c->bufs[b].grid != g) return fail(c, FC_ERR_ARG, "fc_bind_field: array already bound on another grid");
            c->bufs[b].refs++;
            c->slot[i][g][idx] = (int)b;
            return FC_OK;
        }
    Buffer B;
    B.user = p;
    B.n = n;
    B.grid = g;
    B.refs = 1;
    classify_pointer(p, &B.user_is_device, &B.user_is_pinned, nullptr);
    if (B.user_is_device) {
        B.dev = p;
    } else {
        CUDA_TRY(c, cudaMalloc(&B.dev, (size_t)std::max<int64_t>(n, 1) * sizeof(double)));
        if (c->pin_host && !B.user_is_pinned && n > 0) {
            if (cudaHostRegister(p, (size_t)n * sizeof(double), cudaHostRegisterPortable) == cudaSuccess) B.registered = true;
            else cudaGetLastError();
        }
    }
    // reuse a tombstone if there is one
    for (size_t b = 0; b < c->bufs.size(); ++b)
        if (c->bufs[b].user == nullptr && c->bufs[b].refs == 0) {
            c->bufs[b] = B;
            c->slot[i][g][idx] = (int)b;
            return FC_OK;
        }
    c->bufs.push_back(B);
    c->slot[i][g][idx] = (int)c->bufs.size() - 1;
    return FC_OK;
}

extern "C" int fc_set_allocated(fc_context *c, int i, int g, int idx, int allocated)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "fc_set_allocated: NULL context");
    if (i < 0 || i > FC_MAX_SURFACE_TYPES || g < 1 || g > 3 || idx < 1 || idx > FC_MAX_VARNAMES)
        return fail(c, FC_ERR_ARG, "fc_set_allocated: index out of range (surface_type %d, grid %d, var %d)", i, g, idx);
    c->alloc_flag[i][g][idx] = (signed char)(allocated < 0 ? -1 : (allocated ? 1 : 0));
    c->dirty = true;
    return FC_OK;
}

static int mark_slot(fc_context *c, int i, int g, int idx, const char *fn, Buffer **B)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "%s: NULL context", fn);
    if (i < 0 || i > FC_MAX_SURFACE_TYPES || g < 1 || g > 3 || idx < 1 || idx > FC_MAX_VARNAMES)
        return fail(c, FC_ERR_ARG, "%s: index out of range (surface_type %d, grid %d, var %d)", fn, i, g, idx);
    if (c->slot[i][g][idx] < 0) return fail(c, FC_ERR_STATE, "%s: %s of surface_type %d on grid %d is not bound", fn, kVarNames[idx], i, g);
    *B = &c->bufs[c->slot[i][g][idx]];
    return FC_OK;
}

extern "C" int fc_mark_static(fc_context *c, int i, int g, int idx, int is_static)
{
    Buffer *B = nullptr;
    if (int rc = mark_slot(c, i, g, idx, "fc_mark_static", &B)) return rc;
    B->is_static = is_static != 0;
    B->dev_valid = false;
    return FC_OK;
}

extern "C" int fc_mark_dirty(fc_context *c, int i, int g, int idx)
{
    Buffer *B = nullptr;
    if (int rc = mark_slot(c, i, g, idx, "fc_mark_dirty", &B)) return rc;
    B->dev_valid = false;
    return FC_OK;
}

// CPUs next to the device's PCIe root: pinned buffers allocated (first touched) afterwards land in that NUMA node, and
// the copies of eight ranks do not all cross the socket interconnect
extern "C" int fc_bind_thread_to_device_numa(int device)
{
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, FC_ERR_CUDA, "fc_bind_thread_to_device_numa: no PCI bus id for device %d", device);
    }
    for (char *q = bus; *q; ++q) *q = (char)tolower(*q);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/local_cpulist", bus);
    FILE *f = fopen(path, "r");
    if (!f) return fail(nullptr, FC_ERR_STATE, "fc_bind_thread_to_device_numa: cannot read %s", path);
    char line[4096] = {0};
    const bool got = fgets(line, sizeof line, f) != nullptr;
    fclose(f);
    if (!got) return fail(nullptr, FC_ERR_STATE, "fc_bind_thread_to_device_numa: %s is empty", path);
    cpu_set_t set, allowed;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return fail(nullptr, FC_ERR_STATE, "sched_getaffinity failed");
    int ncpu = 0;
    for (char *tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int lo = 0, hi = 0;
        const int k = sscanf(tok, "%d-%d", &lo, &hi);
        if (k == 1) hi = lo;
        if (k < 1) continue;
        for (int cpu = lo; cpu <= hi && cpu < CPU_SETSIZE; ++cpu)
            if (CPU_ISSET(cpu, &allowed)) {      // stay inside what the job was given (cgroup / taskset)
                CPU_SET(cpu, &set);
                ++ncpu;
            }
    }
    if (ncpu == 0) return fail(nullptr, FC_ERR_STATE, "fc_bind_thread_to_device_numa: none of the device's local CPUs is available to this process");
    if (sched_setaffinity(0, sizeof set, &set) != 0) return fail(nullptr, FC_ERR_STATE, "sched_setaffinity failed");
    return FC_OK;
}

extern "C" int fc_set_method(fc_context *c, const char *which, int i, const char *method)
{
    if (!c || !which || !method) return fail(c, FC_ERR_ARG, "fc_set_method: NULL argument");
    if (i < 1 || i > FC_MAX_SURFACE_TYPES) return fail(c, FC_ERR_ARG, "fc_set_method: surface_type %d out of range 1..%d", i, FC_MAX_SURFACE_TYPES);
    static const struct { const char *name; int q; } table[] = {
        {"which_spec_vapor_surface_t", Q_QSUR_T}, {"which_spec_vapor_surface_u", Q_QSUR_U},
        {"which_spec_vapor_surface_v", Q_QSUR_V}, {"which_flux_mass_evap", Q_MEVA},
        {"which_flux_heat_latent", Q_HLAT},       {"which_flux_heat_sensible", Q_HSEN},
        {"which_flux_momentum", Q_MOM},           {"which_flux_radiation_blackbody", Q_RBBR}};   // flux_calculator.F90:99-107
    int q = -1;
    for (auto &t : table)
        if (strcmp(which, t.name) == 0) q = t.q;
    if (q < 0) return fail(c, FC_ERR_ARG, "fc_set_method: unknown namelist array '%s'", which);
    const int m = parse_method(method);
    if (m == M_INVALID || !method_allowed(q, m)) {
        static const char *vn[] = {"QSUR", "QSUR", "QSUR", "MEVA", "HLAT", "HSEN", "UMOM/VMOM", "RBBR"};
        return fail(c, FC_ERR_METHOD, "Error calculating %s for surface_type %d: Method %s is not known.", vn[q], i, method);
    }
    c->method[q][i] = m;
    c->dirty = true;
    return FC_OK;
}

extern "C" int fc_set_distribute_shortwave(fc_context *c, int on)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    c->dist_sw = on < 0 ? -1 : (on ? 1 : 0);
    c->dirty = true;
    return FC_OK;
}

extern "C" int fc_set_corrections(fc_context *c, int which, const double *corr, int64_t n, int enabled, int init_date)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (which != 1) return fail(c, FC_ERR_ARG, "fc_set_corrections: only correction 1 (E_MASS_EVAP_CORRECTION) exists (bias_corrections.F90:16-19)");
    cudaSetDevice(c->device);
    c->dirty = true;
    c->corr_enabled = false;
    c->init_date = init_date;
    if (!enabled) return FC_OK;
    if (!corr || n != c->n[1]) return fail(c, FC_ERR_ARG, "fc_set_corrections: need corrections(1,12,%lld)", (long long)c->n[1]);
    if (fc_current_month(init_date, 0) == 0) return fail(c, FC_ERR_ARG, "fc_set_corrections: init_date %d is not YYYYMMDD", init_date);
    if (!c->corr_dev) CUDA_TRY(c, cudaMalloc(&c->corr_dev, (size_t)std::max<int64_t>(corr_stride(n), 2) * 12 * sizeof(double)));
    if (n > 0) {
        bool is_dev, is_pin;
        classify_pointer(corr, &is_dev, &is_pin, nullptr);
        const double *src = corr;
        struct Tmp {      // freed on every path out of this block
            double *p = nullptr;
            ~Tmp() { cudaFree(p); }
        } tmp;
        if (!is_dev) {
            CUDA_TRY(c, cudaMalloc(&tmp.p, (size_t)n * 12 * sizeof(double)));
            CUDA_TRY(c, cudaMemcpyAsync(tmp.p, corr, (size_t)n * 12 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
            src = tmp.p;
        }
        if (launch_transpose_corrections(src, c->corr_dev, n, corr_stride(n), c->stream)) return fail(c, FC_ERR_CUDA, "transpose_corrections launch failed");
        c->launches++;
        c->tail_own_step = false;
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    c->corr_enabled = true;
    return FC_OK;
}

extern "C" int fc_add_output_field(fc_context *c, int i, int g, int idx)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (i < 0 || i > FC_MAX_SURFACE_TYPES || g < 1 || g > 3 || idx < 1 || idx > FC_MAX_VARNAMES)
        return fail(c, FC_ERR_ARG, "fc_add_output_field: index out of range");
    OutputField o{i, g, idx, idx == FC_RBBR || idx == FC_TSUR || idx == FC_FICE || idx == FC_ALBE};   // basic.F90:271-273
    c->outputs.push_back(o);
    c->dirty = true;
    return FC_OK;
}

extern "C" int fc_set_area(fc_context *c, int g, const double *area, int64_t n)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (g < 1 || g > 3 || !area || n != c->n[g]) return fail(c, FC_ERR_ARG, "fc_set_area: bad argument");
    cudaSetDevice(c->device);
    bool is_dev, is_pin;
    classify_pointer(area, &is_dev, &is_pin, nullptr);
    if (c->area_owned[g]) cudaFree(c->area_dev[g]);
    c->area_owned[g] = false;
    if (is_dev) {
        c->area_dev[g] = const_cast<double *>(area);
    } else {
        CUDA_TRY(c, cudaMalloc(&c->area_dev[g], (size_t)std::max<int64_t>(n, 1) * sizeof(double)));
        c->area_owned[g] = true;
        CUDA_TRY(c, cudaMemcpy(c->area_dev[g], area, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
    }
    c->dirty = true;
    return FC_OK;
}

extern "C" int fc_set_time(fc_context *c, int64_t t)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    c->time = t;
    return FC_OK;
}

extern "C" int fc_set_option(fc_context *c, const char *name, int64_t value)
{
    if (!c || !name) return fail(c, FC_ERR_ARG, "fc_set_option: NULL argument");
    if (!strcmp(name, "force_generic")) c->force_generic = value != 0;
    else if (!strcmp(name, "pin_host")) c->pin_host = value != 0;
    else if (!strcmp(name, "h2d_chunks")) c->h2d_chunks = (int)std::max<int64_t>(0, std::min<int64_t>(value, 256));
    else if (!strcmp(name, "diagnostics")) c->diagnostics = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2));
    else if (!strcmp(name, "staged")) c->use_staged = (int)std::max<int64_t>(0, std::min<int64_t>(value, 2));
    else if (!strcmp(name, "early_loads")) c->early_loads = value != 0;
    else if (!strcmp(name, "chain")) c->chain_steps = value != 0;
    else if (!strcmp(name, "download")) c->download_sent_only = value != 0;
    else if (!strcmp(name, "dyn_min_tiles")) c->dyn_min_tiles = (int)std::max<int64_t>(0, std::min<int64_t>(value, 1 << 30));
    else if (!strcmp(name, "stream_touched")) {      // the caller enqueued own work on fc_get_stream(): no shortcut across it
        c->tail_own_step = false;
        return FC_OK;
    }
    else if (!strcmp(name, "profile_kernel")) {
        c->profile_kernel = (int)std::max<int64_t>(0, std::min<int64_t>(value, 1 << 20));   // 0 off, n: every n-th launch
        c->prof_seq = 0;
        c->prof_used = 0;
        return FC_OK;
    }
    else return fail(c, FC_ERR_ARG, "fc_set_option: unknown option '%s'", name);
    c->dirty = true;
    return FC_OK;
}

extern "C" fc_stream_t fc_get_stream(fc_context *c) { return c ? (fc_stream_t)c->stream : nullptr; }

extern "C" int fc_synchronize(fc_context *c)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    cudaSetDevice(c->device);
    if (int rc = flush_fold(c)) return rc;      // the last step's diagnostics rows -> its result vector (and the peers' mailboxes)
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    if (c->comm_stream) CUDA_TRY(c, cudaStreamSynchronize(c->comm_stream));
    return FC_OK;
}

// ---------------------------------------------------------------------------------------------
// op generation: the reference's pass sequence (flux_calculator_calculate.F90)
// ---------------------------------------------------------------------------------------------
namespace {

struct Gen {
    fc_context *c;
    std::vector<HOp> ops;
    std::string missing;     // accumulated like prepare.F90's missing_field
    bool strict;

    int need(int i, int g, int idx, const char *label = nullptr)
    {
        const int b = slot_of(c, i, g, idx);
        if (b < 0) {
            missing += " ";
            missing += label ? label : kVarNames[idx];
        }
        return b;
    }
};

int report_missing(Gen &G, const char *var, int i, int g, const char *method)
{
    // wording follows prepare.F90:29-31
    return fail(G.c, FC_ERR_MISSING,
                "Error calculating %s for surface_type %d on the grid %s: For method %s we are lacking the following variables:%s",
                var, i, kGridNames[g], method, G.missing.c_str());
}

const char *method_name(int m)
{
    static const char *n[] = {"none", "zero", "copy", "CCLM", "MOM5", "RCO", "water", "ice", "StBo"};
    return (m >= 0 && m <= M_STBO) ? n[m] : "?";
}

HOp mk(int code, int g, int out, std::initializer_list<int> ins, double cst = 0.0, int out2 = -1)
{
    HOp o;
    o.code = code;
    o.grid = g;
    o.out = out;
    o.out2 = out2;
    o.cst = cst;
    int k = 0;
    for (int b : ins) o.in[k++] = b;
    o.n_in = k;
    return o;
}

// calc_spec_vapor_surface, calculate.F90:25-50
int gen_qsur(Gen &G, int g)
{
    fc_context *c = G.c;
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_QSUR_T + (g - 1)][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        if (m == M_COPY) {
            if (slot_of(c, 1, g, FC_QSUR) < 0) G.missing = " QSUR for surface_type=1";   // prepare.F90:58-59
            if (!G.missing.empty()) return report_missing(G, "QSUR", i, g, "copy");
            continue;
        }
        const int out = G.need(i, g, FC_QSUR, "QSUR(output)");
        const int f = G.need(i, g, FC_FICE), p = G.need(i, g, FC_PSUR), t = G.need(i, g, FC_TSUR);   // prepare.F90:61-63
        if (!G.missing.empty()) return report_missing(G, "QSUR", i, g, method_name(m));
        G.ops.push_back(mk(OP_QSUR_CCLM, g, out, {f, p, t}));
    }
    return FC_OK;
}

// calc_flux_mass_evap, calculate.F90:54-120
int gen_meva(Gen &G)
{
    fc_context *c = G.c;
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_MEVA][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        int out = -1;
        if (m == M_COPY) {
            if (slot_of(c, 1, 1, FC_MEVA) < 0) G.missing = " MEVA for surface_type=1";
            out = slot_of(c, i, 1, FC_MEVA);
            if (out < 0 && c->corr_enabled) G.missing += " MEVA(output)";
        } else {
            out = G.need(i, 1, FC_MEVA, "MEVA(output)");
        }
        if (m == M_ZERO) {
            if (!G.missing.empty()) return report_missing(G, "MEVA", i, 1, "zero");
            G.ops.push_back(mk(OP_ZERO, 1, out, {}));
        } else if (m == M_CCLM || m == M_MOM5) {
            const int a = G.need(i, 1, m == M_CCLM ? FC_AMOI : FC_CMOI);      // :83 / :94
            const int ps = G.need(i, 1, FC_PSUR), qa = G.need(i, 1, FC_QATM), qs = G.need(i, 1, FC_QSUR);
            const int ta = G.need(i, 1, FC_TATM);                             // T slot <- TATM (:87, :98)
            const int u = G.need(i, 1, FC_UATM), v = G.need(i, 1, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, "MEVA", i, 1, method_name(m));
            G.ops.push_back(mk(OP_MEVA_CCLM, 1, out, {a, ps, qa, qs, ta, u, v}));
        } else if (m == M_RCO) {
            const int qa = G.need(i, 1, FC_QATM);
            if (G.strict && slot_of(c, i, 1, FC_QSUR) < 0) G.missing += " TSUR";   // prepare.F90:107 tests QSUR, says TSUR
            const int ts = G.need(i, 1, FC_TSUR);                             // what :104-108 really reads
            const int u = G.need(i, 1, FC_UATM), v = G.need(i, 1, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, "MEVA", i, 1, "RCO");
            G.ops.push_back(mk(OP_MEVA_RCO, 1, out, {qa, ts, u, v}));
        } else if (!G.missing.empty()) {
            return report_missing(G, "MEVA", i, 1, "copy");
        }
        if (c->corr_enabled) {                                                 // :112-116, also after 'zero' and 'copy'
            HOp o = mk(OP_ADD, 1, out, {-1});
            o.in0_is_bias = true;
            G.ops.push_back(o);
        }
    }
    return FC_OK;
}

// calc_flux_heat_latent, calculate.F90:124-154
int gen_hlat(Gen &G)
{
    fc_context *c = G.c;
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_HLAT][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        if (m == M_COPY) {
            // prepare.F90:132 tests HSEN of type 1 (quirk); the sane check is HLAT of type 1
            if (slot_of(c, 1, 1, G.strict ? FC_HSEN : FC_HLAT) < 0) G.missing = " HLAT for surface_type=1";
            if (!G.missing.empty()) return report_missing(G, "HLAT", i, 1, "copy");
            continue;
        }
        const int out = G.need(i, 1, FC_HLAT, "HLAT(output)");
        if (m == M_ZERO) {
            if (!G.missing.empty()) return report_missing(G, "HLAT", i, 1, "zero");
            G.ops.push_back(mk(OP_ZERO, 1, out, {}));
            continue;
        }
        const int e = G.need(i, 1, FC_MEVA);                                  // prepare.F90:136,138
        if (!G.missing.empty()) return report_missing(G, "HLAT", i, 1, method_name(m));
        G.ops.push_back(mk(OP_SCALE, 1, out, {e},
                           m == M_WATER ? c->consts.latent_heat_vaporization : c->consts.latent_heat_sublimation));
    }
    return FC_OK;
}

// calc_flux_heat_sensible, calculate.F90:156-208
int gen_hsen(Gen &G)
{
    fc_context *c = G.c;
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_HSEN][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        if (m == M_COPY) {
            if (slot_of(c, 1, 1, FC_HSEN) < 0) G.missing = " HSEN for surface_type=1";
            if (!G.missing.empty()) return report_missing(G, "HSEN", i, 1, "copy");
            continue;
        }
        const int out = G.need(i, 1, FC_HSEN, "HSEN(output)");
        if (m == M_ZERO) {
            if (!G.missing.empty()) return report_missing(G, "HSEN", i, 1, "zero");
            G.ops.push_back(mk(OP_ZERO, 1, out, {}));
        } else if (m == M_CCLM || m == M_MOM5) {
            const int a = G.need(i, 1, m == M_CCLM ? FC_AMOI : FC_CHEA);      // :175 / :187
            const int pa = G.need(i, 1, FC_PATM), ps = G.need(i, 1, FC_PSUR);
            if (G.strict && slot_of(c, i, 1, FC_QSUR) < 0) G.missing += " QSUR";   // prepare.F90:166 (never read)
            const int qa = G.need(i, 1, FC_QATM);                             // q_s slot <- QATM (:178, :190)
            const int ta = G.need(i, 1, FC_TATM), ts = G.need(i, 1, FC_TSUR);
            const int u = G.need(i, 1, FC_UATM), v = G.need(i, 1, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, "HSEN", i, 1, method_name(m));
            G.ops.push_back(mk(OP_HSEN_CCLM, 1, out, {a, pa, ps, qa, ta, ts, u, v}));
        } else {   // RCO
            const int ta = G.need(i, 1, FC_TATM), ts = G.need(i, 1, FC_TSUR);
            const int u = G.need(i, 1, FC_UATM), v = G.need(i, 1, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, "HSEN", i, 1, "RCO");
            G.ops.push_back(mk(OP_HSEN_RCO, 1, out, {ta, ts, u, v}));
        }
    }
    return FC_OK;
}

// calc_flux_momentum_east (north=0) / _north (north=1), calculate.F90:212-316
int gen_mom(Gen &G, int g, int north)
{
    fc_context *c = G.c;
    const int ovar = north ? FC_VMOM : FC_UMOM;
    const char *oname = north ? "VMOM" : "UMOM";
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_MOM][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        if (m == M_COPY) {
            if (slot_of(c, 1, g, ovar) < 0) G.missing = std::string(" ") + oname + " for surface_type=1";
            if (!G.missing.empty()) return report_missing(G, oname, i, g, "copy");
            continue;
        }
        const int out = G.need(i, g, ovar, north ? "VMOM(output)" : "UMOM(output)");
        if (m == M_ZERO) {
            if (!G.missing.empty()) return report_missing(G, oname, i, g, "zero");
            G.ops.push_back(mk(OP_ZERO, g, out, {}));
        } else if (m == M_CCLM || m == M_MOM5) {
            const int a = G.need(i, g, m == M_CCLM ? FC_AMOM : FC_CMOM);
            const int ps = G.need(i, g, FC_PSUR), qs = G.need(i, g, FC_QSUR);
            if (G.strict && slot_of(c, i, g, FC_TATM) < 0) G.missing += " TATM TSUR";   // prepare.F90:214-215 (TATM is never read)
            const int ts = G.need(i, g, FC_TSUR);
            const int u = G.need(i, g, FC_UATM), v = G.need(i, g, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, oname, i, g, method_name(m));
            G.ops.push_back(north ? mk(OP_MOM_CCLM, g, -1, {a, ps, qs, ts, u, v}, 0.0, out)
                                  : mk(OP_MOM_CCLM, g, out, {a, ps, qs, ts, u, v}));
        } else {   // RCO
            const int u = G.need(i, g, FC_UATM), v = G.need(i, g, FC_VATM);
            if (!G.missing.empty()) return report_missing(G, oname, i, g, "RCO");
            G.ops.push_back(north ? mk(OP_MOM_RCO, g, -1, {u, v}, 0.0, out) : mk(OP_MOM_RCO, g, out, {u, v}));
        }
    }
    return FC_OK;
}

// calc_flux_radiation_blackbody, calculate.F90:320-345
int gen_rbbr(Gen &G)
{
    fc_context *c = G.c;
    for (int i = 1; i <= c->S; ++i) {
        const int m = c->method[Q_RBBR][i];
        if (m == M_NONE) continue;
        G.missing.clear();
        if (m == M_COPY) {
            if (slot_of(c, 1, 1, FC_RBBR) < 0) G.missing = " RBBR for surface_type=1";
            if (!G.missing.empty()) return report_missing(G, "RBBR", i, 1, "copy");
            continue;
        }
        const int out = G.need(i, 1, FC_RBBR, "RBBR(output)");
        if (m == M_ZERO) {
            if (!G.missing.empty()) return report_missing(G, "RBBR", i, 1, "zero");
            G.ops.push_back(mk(OP_ZERO, 1, out, {}));
            continue;
        }
        const int ts = G.need(i, 1, FC_TSUR);                                 // prepare.F90:293
        if (!G.missing.empty()) return report_missing(G, "RBBR", i, 1, "StBo");
        G.ops.push_back(mk(OP_RBBR, 1, out, {ts}, c->consts.stefan_boltzmann_constant));
    }
    return FC_OK;
}

bool shortwave_enabled(const fc_context *c)
{
    if (c->dist_sw == 0) return false;
    bool all = slot_of(c, 0, 1, FC_RSDD) >= 0;
    for (int i = 1; i <= c->S; ++i) all = all && slot_of(c, i, 1, FC_RSDR) >= 0;
    return c->dist_sw == 1 ? true : all;
}

// distribute_shortwave_radiation_flux, calculate.F90:347-364 (ALBA/ALBE are passed but unused)
int gen_rsdr(Gen &G, bool explicit_call)
{
    fc_context *c = G.c;
    if (!explicit_call && !shortwave_enabled(c)) return FC_OK;
    for (int i = 1; i <= c->S; ++i) {
        G.missing.clear();
        const int out = G.need(i, 1, FC_RSDR, "RSDR(output)");
        const int in = G.need(0, 1, FC_RSDD, "RSDD(surface_type 0)");
        if (!G.missing.empty()) return report_missing(G, "RSDR", i, 1, "distribute");
        G.ops.push_back(mk(OP_COPY, 1, out, {in}));
    }
    return FC_OK;
}

// average_across_surface_types, calculate.F90:368-385
int gen_avg(Gen &G, int g, int idx)
{
    fc_context *c = G.c;
    if (slot_of(c, 0, g, idx) < 0 || !slot_owns(c, 0, g, idx)) return FC_OK;   // :376 "%allocated"
    const int out = slot_of(c, 0, g, idx);
    G.missing.clear();
    std::vector<HOp> acc;
    for (int i = 1; i <= c->S; ++i) {
        const int x = G.need(i, g, idx), f = G.need(i, g, FC_FARE);
        acc.push_back(mk(OP_MULADD, g, out, {x, f}));
    }
    if (!G.missing.empty())
        return fail(c, FC_ERR_MISSING, "Error averaging %s on the grid %s: lacking per-surface-type arrays:%s", kVarNames[idx],
                    kGridNames[g], G.missing.c_str());
    G.ops.push_back(mk(OP_ZERO, g, out, {}));                                 // :377
    for (auto &o : acc) G.ops.push_back(o);                                   // :378-383
    return FC_OK;
}

// send loops: flux_calculator.F90:909-919 (early) / :999-1009 (normal)
int gen_send(Gen &G, bool early, std::vector<OutputField> *fused_candidates = nullptr)
{
    fc_context *c = G.c;
    for (int g = 1; g <= 3; ++g)
        for (const OutputField &o : c->outputs) {
            if (o.grid != g || o.early != early || o.surface_type != 0) continue;
            if (slot_of(c, 0, g, o.idx) < 0 || slot_of(c, 2, g, o.idx) < 0) continue;   // :913-914
            if (fused_candidates) {
                fused_candidates->push_back(o);
                continue;
            }
            if (int rc = gen_avg(G, g, o.idx)) return rc;
        }
    return FC_OK;
}

int gen_early(Gen &G)
{
    if (int rc = gen_rbbr(G)) return rc;        // flux_calculator.F90:902
    return gen_send(G, true);
}

int gen_normal(Gen &G)
{
    int rc;
    if ((rc = gen_qsur(G, 1))) return rc;       // :972
    if ((rc = gen_qsur(G, 2))) return rc;       // :973
    if ((rc = gen_qsur(G, 3))) return rc;       // :974
    if ((rc = gen_meva(G))) return rc;          // :977
    if ((rc = gen_hlat(G))) return rc;          // :980
    if ((rc = gen_hsen(G))) return rc;          // :983
    if ((rc = gen_mom(G, 2, 0))) return rc;     // :986
    if ((rc = gen_mom(G, 3, 1))) return rc;     // :988
    if ((rc = gen_rsdr(G, false))) return rc;   // :991
    return gen_send(G, false);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// executing an op sequence with the interpreter kernel
// ---------------------------------------------------------------------------------------------
static const double *bias_slab(fc_context *c)
{
    const int month = fc_current_month(c->init_date, c->time);   // calculate.F90:66-73
    return c->corr_dev + (size_t)(month - 1) * (size_t)corr_stride(c->n[1]);
}

static int run_ops(fc_context *c, const std::vector<HOp> &ops)
{
    if (ops.empty()) return FC_OK;
    cudaSetDevice(c->device);
    c->tail_own_step = false;
    // host-pointer mode: upload every buffer that is read before it is written, download what is written
    std::vector<int> up, down;
    {
        std::set<int> written, ups, downs;
        for (const HOp &o : ops) {
            for (int k = 0; k < o.n_in; ++k) {
                const int b = o.in[k];
                if (b >= 0 && !written.count(b)) ups.insert(b);
            }
            if ((o.code == OP_ADD || o.code == OP_MULADD)) {
                if (o.out >= 0 && !written.count(o.out)) ups.insert(o.out);
            }
            for (int b : {o.out, o.out2})
                if (b >= 0) {
                    written.insert(b);
                    downs.insert(b);
                }
        }
        for (int b : ups)
            if (!c->bufs[b].user_is_device) up.push_back(b);
        for (int b : downs)
            if (!c->bufs[b].user_is_device) down.push_back(b);
    }
    for (int b : up) {
        const Buffer &B = c->bufs[b];
        CUDA_TRY(c, cudaMemcpyAsync(B.dev, B.user, (size_t)B.n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        c->h2d_bytes += B.n * (int64_t)sizeof(double);
    }
    for (int g = 1; g <= 3; ++g) {
        OpList L;
        L.n = 0;
        L.pad = 0;
        auto flush = [&]() -> int {
            if (L.n == 0) return FC_OK;
            if (launch_oplist(L, c->consts, c->n[g], c->stream)) return fail(c, FC_ERR_CUDA, "oplist launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            if (c->n[g] > 0) c->launches++;
            L.n = 0;
            return FC_OK;
        };
        for (const HOp &o : ops) {
            if (o.grid != g) continue;
            Op d;
            memset(&d, 0, sizeof d);
            d.code = o.code;
            d.cst = o.cst;
            d.out = o.out >= 0 ? c->bufs[o.out].dev : nullptr;
            d.out2 = o.out2 >= 0 ? c->bufs[o.out2].dev : nullptr;
            for (int k = 0; k < o.n_in; ++k) d.in[k] = o.in[k] >= 0 ? c->bufs[o.in[k]].dev : nullptr;
            if (o.in0_is_bias) d.in[0] = bias_slab(c);
            L.ops[L.n++] = d;
            if (L.n == kMaxOps)
                if (int rc = flush()) return rc;
        }
        if (int rc = flush()) return rc;
    }
    for (int b : down) {
        const Buffer &B = c->bufs[b];
        CUDA_TRY(c, cudaMemcpyAsync(B.user, B.dev, (size_t)B.n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        c->d2h_bytes += B.n * (int64_t)sizeof(double);
    }
    if (!down.empty() || !up.empty()) CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return FC_OK;
}

// ---------------------------------------------------------------------------------------------
// fused plan builder
// ---------------------------------------------------------------------------------------------

// chunks of the host-pointer pipeline.  Its depth: the first chunk's upload and the last chunk's download are exposed, so even
// a small shard (the 8-GPU share of a 10^7-cell grid is 1.25 * 10^6 cells) gets at least 8 chunks; tiny grids are not worth
// splitting
static int pipeline_chunks(const fc_context *c)
{
    const int64_t nmax = std::max(c->n[1], std::max(c->n[2], c->n[3]));
    return c->h2d_chunks > 0 ? std::min(c->h2d_chunks, kMaxChunks)
                             : (nmax < 65536 ? 1 : (int)std::min<int64_t>(kMaxChunks, std::max<int64_t>(8, nmax / 262144)));
}

// chunk boundaries of the host-pointer pipeline: 256-byte aligned starts, the last chunk takes the remainder
static void chunk_range(const fc_context *c, int k, int K, int64_t c0[4], int64_t c1[4])
{
    for (int g = 1; g <= 3; ++g) {
        c0[g] = (K == 1) ? 0 : ((c->n[g] * k / K) & ~int64_t(31));
        c1[g] = (k == K - 1) ? c->n[g] : ((c->n[g] * (k + 1) / K) & ~int64_t(31));
    }
}

// how the plan launches as one device-resident step and as the chunks of the host-pointer pipeline
static void resolve_bundle(const fc_context *c, FusedBundle &F)
{
    const int64_t zero[3] = {0, 0, 0}, n[3] = {c->n[1], c->n[2], c->n[3]};
    F.step = resolve_fused(F.plan, zero, n, c->use_staged, c->dyn_min_tiles);
    const int K = pipeline_chunks(c);
    for (int k = 0; k < K; ++k) {
        int64_t c0[4], c1[4];
        chunk_range(c, k, K, c0, c1);
        const int64_t first[3] = {c0[1], c0[2], c0[3]}, cells[3] = {c1[1] - c0[1], c1[2] - c0[2], c1[3] - c0[3]};
        F.chunks.push_back(resolve_fused(F.plan, first, cells, c->use_staged, c->dyn_min_tiles));
    }
}

static bool build_fused(fc_context *c, bool do_early, bool do_normal, FusedBundle &F)
{
    F = FusedBundle();
    FusedPlan &P = F.plan;
    memset(&P, 0, sizeof P);
    P.S = c->S;
    P.do_early = do_early;
    P.do_normal = do_normal;
    P.c = c->consts;
    P.t.n = c->n[1];
    P.uv[0].n = c->n[2];
    P.uv[1].n = c->n[3];
    P.uv[0].north = 0;
    P.uv[1].north = 1;

    std::set<int> ins, outs;
    bool ok = true;
    auto in = [&](int i, int g, int idx) -> const double * {
        const int b = slot_of(c, i, g, idx);
        if (b < 0) {
            ok = false;
            return nullptr;
        }
        ins.insert(b);
        return c->bufs[b].dev;
    };
    auto out = [&](int i, int g, int idx) -> double * {
        const int b = slot_of(c, i, g, idx);
        if (b < 0 || outs.count(b)) {   // unbound, or two results into one array (aliasing) -> generic path
            ok = false;
            return nullptr;
        }
        outs.insert(b);
        return c->bufs[b].dev;
    };
    const bool rsdr = do_normal && shortwave_enabled(c);
    if (rsdr) P.t.rsdd = in(0, 1, FC_RSDD);
    const bool bias = do_normal && c->corr_enabled;

    for (int i = 1; i <= c->S && ok; ++i) {
        FusedTType &T = P.t.ty[i - 1];
        T.m_qsur = T.m_meva = T.m_hlat = T.m_hsen = T.m_rbbr = M_NONE;
        if (do_normal) {
            const int mq = c->method[Q_QSUR_T][i], me = c->method[Q_MEVA][i], ml = c->method[Q_HLAT][i], mh = c->method[Q_HSEN][i];
            if (mq == M_COPY || me == M_COPY || ml == M_COPY || mh == M_COPY) return false;
            T.m_qsur = mq;
            T.m_meva = me;
            T.m_hlat = ml;
            T.m_hsen = mh;
            const bool need_q = (me == M_CCLM || me == M_MOM5);
            if (mq == M_CCLM) {
                T.fice = in(i, 1, FC_FICE);
                T.psur = in(i, 1, FC_PSUR);
                T.tsur = in(i, 1, FC_TSUR);
                T.qsur = out(i, 1, FC_QSUR);
            } else if (need_q) {
                T.qsur_in = in(i, 1, FC_QSUR);
            }
            if (me == M_CCLM || me == M_MOM5) {
                T.a_evap = in(i, 1, me == M_CCLM ? FC_AMOI : FC_CMOI);
                T.psur = in(i, 1, FC_PSUR);
                T.qatm = in(i, 1, FC_QATM);
                T.tatm = in(i, 1, FC_TATM);
                T.uatm = in(i, 1, FC_UATM);
                T.vatm = in(i, 1, FC_VATM);
            } else if (me == M_RCO) {
                T.qatm = in(i, 1, FC_QATM);
                T.tsur = in(i, 1, FC_TSUR);
                T.uatm = in(i, 1, FC_UATM);
                T.vatm = in(i, 1, FC_VATM);
            }
            if (me != M_NONE) T.meva = out(i, 1, FC_MEVA);
            if (ml == M_WATER || ml == M_ICE) {
                if (me == M_NONE) return false;   // MEVA would be an input array: generic path
                T.latent_heat = ml == M_WATER ? c->consts.latent_heat_vaporization : c->consts.latent_heat_sublimation;
            }
            if (ml != M_NONE) T.hlat = out(i, 1, FC_HLAT);
            if (mh == M_CCLM || mh == M_MOM5) {
                T.a_sens = in(i, 1, mh == M_CCLM ? FC_AMOI : FC_CHEA);
                T.patm = in(i, 1, FC_PATM);
                T.psur = in(i, 1, FC_PSUR);
                T.qatm = in(i, 1, FC_QATM);
                T.tatm = in(i, 1, FC_TATM);
                T.tsur = in(i, 1, FC_TSUR);
                T.uatm = in(i, 1, FC_UATM);
                T.vatm = in(i, 1, FC_VATM);
            } else if (mh == M_RCO) {
                T.tatm = in(i, 1, FC_TATM);
                T.tsur = in(i, 1, FC_TSUR);
                T.uatm = in(i, 1, FC_UATM);
                T.vatm = in(i, 1, FC_VATM);
            }
            if (mh != M_NONE) T.hsen = out(i, 1, FC_HSEN);
            if (rsdr) T.rsdr = out(i, 1, FC_RSDR);
            for (int g = 0; g < 2; ++g) {
                FusedUVType &U = P.uv[g].ty[i - 1];
                const int gg = g + 2;
                const int mqs = c->method[Q_QSUR_U + g][i], mm = c->method[Q_MOM][i];
                if (mqs == M_COPY || mm == M_COPY) return false;
                U.m_qsur = mqs;
                U.m_mom = mm;
                const bool needq = (mm == M_CCLM || mm == M_MOM5);
                if (mqs == M_CCLM) {
                    U.fice = in(i, gg, FC_FICE);
                    U.psur = in(i, gg, FC_PSUR);
                    U.tsur = in(i, gg, FC_TSUR);
                    U.qsur = out(i, gg, FC_QSUR);
                } else if (needq) {
                    U.qsur_in = in(i, gg, FC_QSUR);
                }
                if (mm == M_CCLM || mm == M_MOM5) {
                    U.a_mom = in(i, gg, mm == M_CCLM ? FC_AMOM : FC_CMOM);
                    U.psur = in(i, gg, FC_PSUR);
                    U.tsur = in(i, gg, FC_TSUR);
                    U.uatm = in(i, gg, FC_UATM);
                    U.vatm = in(i, gg, FC_VATM);
                } else if (mm == M_RCO) {
                    U.uatm = in(i, gg, FC_UATM);
                    U.vatm = in(i, gg, FC_VATM);
                }
                if (mm != M_NONE) U.mom = out(i, gg, g == 0 ? FC_UMOM : FC_VMOM);
            }
        }
        if (do_early) {
            const int mr = c->method[Q_RBBR][i];
            if (mr == M_COPY) return false;
            T.m_rbbr = mr;
            if (mr == M_STBO) T.tsur = in(i, 1, FC_TSUR);
            if (mr != M_NONE) T.rbbr = out(i, 1, FC_RBBR);
        }
    }
    if (!ok) return false;

    // averaging of sent type-0 fields (send loops)
    Gen G{c, {}, "", false};
    std::vector<OutputField> cand;
    if (do_early) gen_send(G, true, &cand);
    if (do_normal) gen_send(G, false, &cand);
    for (const OutputField &o : cand) {
        if (!slot_owns(c, 0, o.grid, o.idx)) continue;
        double **dst = nullptr;
        bool computed_all = true;
        auto all = [&](auto pred) {
            bool a = true;
            for (int i = 1; i <= c->S; ++i) a = a && pred(i);
            return a;
        };
        if (o.grid == 1) {
            switch (o.idx) {
                case FC_QSUR: dst = &P.t.avg_qsur; computed_all = all([&](int i) { return P.t.ty[i - 1].m_qsur == M_CCLM; }); break;
                case FC_MEVA: dst = &P.t.avg_meva; computed_all = all([&](int i) { return P.t.ty[i - 1].m_meva != M_NONE; }); break;
                case FC_HLAT: dst = &P.t.avg_hlat; computed_all = all([&](int i) { return P.t.ty[i - 1].m_hlat != M_NONE; }); break;
                case FC_HSEN: dst = &P.t.avg_hsen; computed_all = all([&](int i) { return P.t.ty[i - 1].m_hsen != M_NONE; }); break;
                case FC_RBBR: dst = &P.t.avg_rbbr; computed_all = all([&](int i) { return P.t.ty[i - 1].m_rbbr != M_NONE; }); break;
                case FC_RSDR: dst = &P.t.avg_rsdr; computed_all = rsdr; break;
                default: break;
            }
        } else {
            FusedUV &U = P.uv[o.grid - 2];
            if (o.idx == FC_QSUR) {
                dst = &U.avg_qsur;
                computed_all = all([&](int i) { return U.ty[i - 1].m_qsur == M_CCLM; });
            } else if (o.idx == (o.grid == 2 ? FC_UMOM : FC_VMOM)) {
                dst = &U.avg_mom;
                computed_all = all([&](int i) { return U.ty[i - 1].m_mom != M_NONE; });
            }
        }
        if (dst && computed_all) {
            if (*dst) continue;   // listed twice
            *dst = out(0, o.grid, o.idx);
            for (int i = 1; i <= c->S; ++i) {
                const double *f = in(i, o.grid, FC_FARE);
                if (o.grid == 1) P.t.ty[i - 1].fare = f;
                else P.uv[o.grid - 2].ty[i - 1].fare = f;
            }
        } else {
            // pass-through variable (TSUR, FICE, ALBE, ...) or partially computed: averaged by ops after the launch
            Gen GA{c, {}, "", false};
            if (gen_avg(GA, o.grid, o.idx)) return false;
            for (auto &h : GA.ops) {
                F.extra.push_back(h);
                // an averaged array that the fused kernel writes would be a read-after-write across kernels: fine
                // (same stream), but an averaged array the fused kernel ALSO averages would be a conflict
                if (h.out >= 0 && outs.count(h.out)) return false;
            }
        }
    }
    if (!ok) return false;
    // no array may be both read and written by the fused pass (in-place aliasing -> generic path)
    for (int b : outs)
        if (ins.count(b)) return false;
    if (bias) P.t.bias = c->corr_dev;   // month slab patched per step

    // diagnostics slots
    P.diag = 0;
    memset(P.diag_map, 0xff, sizeof P.diag_map);
    if (c->diagnostics) {
        for (int g = 1; g <= 3; ++g)
            if ((g == 1 || do_normal) && !c->area_dev[g] && c->n[g] > 0) return false;   // reported by prepare
        P.t.area = c->area_dev[1];
        P.uv[0].area = c->area_dev[2];
        P.uv[1].area = c->area_dev[3];
        P.diag = c->diagnostics;
        memset(P.diag_map, 0xff, sizeof P.diag_map);
        auto act = [&](int type, int q) {
            const int s = type * DQ_COUNT + q;
            P.diag_map[s] = (signed char)F.diag_slots.size();
            F.diag_slots.push_back(s);
        };
        for (int i = 1; i <= c->S; ++i) {
            const FusedTType &T = P.t.ty[i - 1];
            if (do_normal) {
                if (T.m_qsur == M_CCLM) act(i, DQ_QSUR_T);
                if (T.m_meva != M_NONE) act(i, DQ_MEVA);
                if (T.m_hlat != M_NONE) act(i, DQ_HLAT);
                if (T.m_hsen != M_NONE) act(i, DQ_HSEN);
                if (rsdr) act(i, DQ_RSDR);
                if (P.uv[0].ty[i - 1].m_qsur == M_CCLM) act(i, DQ_QSUR_U);
                if (P.uv[0].ty[i - 1].m_mom != M_NONE) act(i, DQ_UMOM);
                if (P.uv[1].ty[i - 1].m_qsur == M_CCLM) act(i, DQ_QSUR_V);
                if (P.uv[1].ty[i - 1].m_mom != M_NONE) act(i, DQ_VMOM);
            }
            if (do_early && T.m_rbbr != M_NONE) act(i, DQ_RBBR);
        }
        if (P.t.avg_qsur) act(0, DQ_QSUR_T);
        if (P.t.avg_meva) act(0, DQ_MEVA);
        if (P.t.avg_hlat) act(0, DQ_HLAT);
        if (P.t.avg_hsen) act(0, DQ_HSEN);
        if (P.t.avg_rbbr) act(0, DQ_RBBR);
        if (P.t.avg_rsdr) act(0, DQ_RSDR);
        if (P.uv[0].avg_qsur) act(0, DQ_QSUR_U);
        if (P.uv[0].avg_mom) act(0, DQ_UMOM);
        if (P.uv[1].avg_qsur) act(0, DQ_QSUR_V);
        if (P.uv[1].avg_mom) act(0, DQ_VMOM);
        P.diag_n = (int)F.diag_slots.size();
        if (P.diag_n == 0) P.diag = 0;
    }
    F.in_bufs.assign(ins.begin(), ins.end());
    F.out_bufs.assign(outs.begin(), outs.end());
    resolve_bundle(c, F);
    F.ok = true;
    return true;
}

// ---------------------------------------------------------------------------------------------
// prepare
// ---------------------------------------------------------------------------------------------
static int prepare_impl(fc_context *c, int strict)
{
    cudaSetDevice(c->device);
    if (int rc = flush_fold(c)) return rc;
    c->tail_own_step = false;
    c->chain_key = nullptr;
    c->strict = strict != 0;
    // validation == generating the full pass sequence once (reports what is lacking)
    {
        Gen G{c, {}, "", c->strict};
        if (int rc = gen_early(G)) return rc;
    }
    {
        Gen G{c, {}, "", c->strict};
        if (int rc = gen_normal(G)) return rc;
    }
    if (c->diagnostics)
        for (int g = 1; g <= 3; ++g)
            if (!c->area_dev[g] && c->n[g] > 0)
                return fail(c, FC_ERR_MISSING, "diagnostics are enabled but fc_set_area was not called for the %s", kGridNames[g]);
    if (c->corr_enabled && !c->corr_dev) return fail(c, FC_ERR_STATE, "corrections enabled without data");
    for (int k = 0; k < 3; ++k) c->fused[k] = FusedBundle();
    for (auto &g : c->step_graph)
        if (g) {
            cudaGraphExecDestroy(g);
            g = nullptr;
        }
    if (!c->force_generic) {
        build_fused(c, true, false, c->fused[0]);
        build_fused(c, false, true, c->fused[1]);
        build_fused(c, true, true, c->fused[2]);
    }
    c->dirty = false;
    return FC_OK;
}

extern "C" int fc_prepare(fc_context *c, int strict)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    return prepare_impl(c, strict);
}

static int ensure_prepared(fc_context *c)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (c->dirty) return prepare_impl(c, c->strict ? 1 : 0);
    return FC_OK;
}

// ---------------------------------------------------------------------------------------------
// the 9 calculators (unfused, reference pass structure; interpreter kernel)
// ---------------------------------------------------------------------------------------------
#define CALC_PROLOGUE()                       \
    if (int rc_ = ensure_prepared(c)) return rc_; \
    c->h2d_bytes = c->d2h_bytes = 0;          \
    Gen G{c, {}, "", false};

extern "C" int fc_calc_spec_vapor_surface(fc_context *c, int g)
{
    CALC_PROLOGUE();
    if (g < 1 || g > 3) return fail(c, FC_ERR_ARG, "which_grid must be 1..3");
    if (int rc = gen_qsur(G, g)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_mass_evap(fc_context *c)
{
    CALC_PROLOGUE();
    if (int rc = gen_meva(G)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_heat_latent(fc_context *c)
{
    CALC_PROLOGUE();
    if (int rc = gen_hlat(G)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_heat_sensible(fc_context *c)
{
    CALC_PROLOGUE();
    if (int rc = gen_hsen(G)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_momentum_east(fc_context *c, int g)
{
    CALC_PROLOGUE();
    if (g < 1 || g > 3) return fail(c, FC_ERR_ARG, "which_grid must be 1..3");
    if (int rc = gen_mom(G, g, 0)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_momentum_north(fc_context *c, int g)
{
    CALC_PROLOGUE();
    if (g < 1 || g > 3) return fail(c, FC_ERR_ARG, "which_grid must be 1..3");
    if (int rc = gen_mom(G, g, 1)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_calc_flux_radiation_blackbody(fc_context *c)
{
    CALC_PROLOGUE();
    if (int rc = gen_rbbr(G)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_distribute_shortwave_radiation_flux(fc_context *c)
{
    CALC_PROLOGUE();
    if (int rc = gen_rsdr(G, true)) return rc;
    return run_ops(c, G.ops);
}
extern "C" int fc_average_across_surface_types(fc_context *c, int g, int idx)
{
    CALC_PROLOGUE();
    if (g < 1 || g > 3 || idx < 1 || idx > FC_MAX_VARNAMES) return fail(c, FC_ERR_ARG, "bad grid / variable index");
    if (int rc = gen_avg(G, g, idx)) return rc;
    return run_ops(c, G.ops);
}

// ---------------------------------------------------------------------------------------------
// fused steps
// ---------------------------------------------------------------------------------------------
// Diagnostics storage for a step issued as K launches (K = 1: device-resident; K > 1: chunks of the host-pointer
// pipeline, which run concurrently on three streams): every chunk owns its partial rows, its reduce scratch, its
// last-CTA counter and its result vector; diag_combine folds the K vectors in chunk order into a.diag_out.
static int ensure_diag_storage(fc_context *c, const FusedPlan &P, const FusedLaunch *L, int K, FusedStepArgs &a)
{
    int64_t rows = 1;
    for (int k = 0; k < K; ++k) rows = std::max(rows, L[k].diag_rows);
    const int planes = P.diag >= 2 ? 3 : 1;
    const size_t stride = (size_t)planes * P.diag_n * (size_t)rows + (size_t)diag_tmp_doubles(rows, P.diag_n);
    // K = 1: two sets, alternating by step -- the rows of step k are folded while step k + 1 writes its own (DiagFold)
    const size_t need = stride * sizeof(double) * (size_t)std::max(K, 2);
    if (need > c->diag_partials_cap) {
        if (int rc = flush_fold(c)) return rc;
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        cudaFree(c->diag_partials);
        c->diag_partials = nullptr;
        CUDA_TRY(c, cudaMalloc(&c->diag_partials, need));
        c->diag_partials_cap = need;
    }
    c->diag_chunk_stride = stride;
    for (int b = 0; b < 2; ++b)
        if (!c->diag_buf[b]) {
            CUDA_TRY(c, cudaMalloc(&c->diag_buf[b], sizeof(double) * kDiagSlots * 3));
            CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_fin[b], cudaEventDisableTiming));
            CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_comm[b], cudaEventDisableTiming));
        }
    if (!c->diag_host) CUDA_TRY(c, cudaHostAlloc(&c->diag_host, sizeof(double) * kDiagSlots * 3 * 2, cudaHostAllocDefault));
    if (!c->diag_chunk_out) {
        CUDA_TRY(c, cudaMalloc(&c->diag_chunk_out, sizeof(double) * kDiagSlots * 3 * kMaxChunks));
        CUDA_TRY(c, cudaMemsetAsync(c->diag_chunk_out, 0, sizeof(double) * kDiagSlots * 3 * kMaxChunks, c->stream));
    }
    a.diag_partials = c->diag_partials;
    a.diag_rows = rows;
    if (K == 1) c->diag_rows_1 = rows;
    // result buffer of this step; if its previous all-reduce is still in flight on the side stream, wait for it
    const int b = c->diag_cur ^ 1;
    if (c->comm_busy[b]) {
        CUDA_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_comm[b], 0));
        c->comm_busy[b] = false;
    }
    a.diag_out = c->diag_buf[b];
    return FC_OK;
}

// chunk k's view of the diagnostics storage
static void diag_chunk_view(const fc_context *c, const FusedStepArgs &a, int k, int K, FusedStepArgs &q)
{
    q.diag_partials = c->diag_partials + (size_t)k * c->diag_chunk_stride;
    q.diag_rows = a.diag_rows;
    q.diag_out = (K == 1) ? a.diag_out : c->diag_chunk_out + (size_t)k * 3 * kDiagSlots;
}

static double *diag_tmp(const FusedPlan &P, const FusedStepArgs &a)
{
    const int planes = P.diag >= 2 ? 3 : 1;
    return a.diag_partials + (size_t)planes * P.diag_n * (size_t)a.diag_rows;
}

// partial rows of a generic launch -> a.diag_out, on the stream it was launched on
static int finalize_chunk(fc_context *c, const FusedPlan &P, const FusedLaunch &L, const FusedStepArgs &a, cudaStream_t s)
{
    int nl = 0;
    if (launch_diag_finalize(P, L, a, diag_tmp(P, a), s, &nl)) return fail(c, FC_ERR_CUDA, "diag finalize launch failed");
    c->launches += nl;
    return FC_OK;
}

// the rows a specialised launch leaves behind, as a fold request
static DiagFold make_fold(const FusedPlan &P, const FusedLaunch &L, const FusedStepArgs &a)
{
    DiagFold f;
    memset(&f, 0, sizeof f);
    f.rows = a.diag_partials;
    f.row_stride = a.diag_rows;
    f.plane = (int64_t)P.diag_n * a.diag_rows;
    f.nrows = (int)L.diag_rows;
    f.nslots = P.diag_n;
    f.level = P.diag;
    f.out = a.diag_out;
    return f;
}

namespace fc {
// fold the rows of the last specialised step now (stand-alone kernel) if no later step has done it yet
int flush_fold(fc_context *c)
{
    if (!c->fold_pending) return FC_OK;
    cudaSetDevice(c->device);
    if (launch_diag_fold(c->fold, c->stream)) return fail(c, FC_ERR_CUDA, "diag fold launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    c->launches += 1;
    c->fold_pending = false;
    c->tail_own_step = false;
    return FC_OK;
}
}  // namespace fc

// bookkeeping once the step's result vector (diag_buf[next]) is issued
static void diag_step_done(fc_context *c, const FusedBundle &F)
{
    c->diag_cur ^= 1;
    c->diag_active = F.diag_slots;
    c->diag_valid = false;
    c->diag_global = false;
    c->diag_level = F.plan.diag;
}

static int ensure_tile_counters(fc_context *c)
{
    if (!c->tile_ctr) {
        CUDA_TRY(c, cudaMalloc(&c->tile_ctr, sizeof(unsigned int) * (kMaxChunks + 2)));
        CUDA_TRY(c, cudaMemset(c->tile_ctr, 0, sizeof(unsigned int) * (kMaxChunks + 2)));
        memset(c->tile_base, 0, sizeof c->tile_base);
    }
    return FC_OK;
}

// dynamic schedule: give launch L claim counter `slot` (the caller advances the counter's base by L.claims)
static int attach_tile_counter(fc_context *c, const FusedLaunch &L, FusedStepArgs &a, int slot)
{
    if (L.claims == 0) return FC_OK;
    if (int rc = ensure_tile_counters(c)) return rc;
    a.tile_counter = c->tile_ctr + slot;
    a.tile_base = c->tile_base[slot];
    return FC_OK;
}

// one device-resident step on the context's stream.  Which kernel runs and how it is scheduled was decided when the plan
// was prepared (F.step, kernels.cu: resolve_fused); what is left here is this step's arguments.  gstep < 0: an ordinary
// step.  gstep >= 0: step number gstep of a sequence that is being captured into a CUDA graph (fc_run_steps): nothing here
// may depend on state that changes between two launches of that graph -- no fold of the previous step's rows (only the
// last step's diagnostics are ever read; the caller registers them after the graph), one row set, tile counters that the
// graph's leading memset node zeroes (step s uses counter s mod 2 at base (s / 2) * claims), no event records, no allocation.
static int launch_resident(fc_context *c, const FusedBundle &F, const double *bias, int gstep)
{
    const bool graph = gstep >= 0;
    const FusedPlan &P = F.plan;
    const FusedLaunch &L = F.step;
    const bool spec = L.spec;
    FusedStepArgs a{};
    a.bias = bias;
    int nlaunch = 0;
    // rows of the previous specialised step that nobody folded yet: this launch folds them while its ring fills,
    // unless it is not that kind of launch
    if (!graph && c->fold_pending && !(spec && P.diag))
        if (int rc = flush_fold(c)) return rc;
    if (P.diag) {
        if (!graph)
            if (int rc = ensure_diag_storage(c, P, &L, 1, a)) return rc;
        const int b = c->diag_cur ^ 1;
        a.diag_partials = c->diag_partials;
        a.diag_rows = c->diag_rows_1;
        a.diag_out = c->diag_buf[b];
        diag_chunk_view(c, a, graph ? 0 : (c->row_set ^= 1), 1, a);
        if (!graph && c->fold_pending) a.fold_prev = c->fold;
    }
    a.early_loads = (spec && c->early_loads && (graph ? gstep > 0 : c->tail_own_step)) ? 1 : 0;
    // dynamic schedule: consecutive steps alternate between two counters, because the producers of a step may claim
    // while the previous step still runs.  That holds for at most two steps at a time only if this step's grid
    // fills the device (a third step finds no room before the first has left); smaller grids wait first.
    const unsigned int claims = L.claims;
    const int tslot = kMaxChunks + (graph ? (gstep & 1) : (c->tile_par ^= 1));
    if (claims && !graph)
        if (int rc = ensure_tile_counters(c)) return rc;
    if (claims) {
        a.tile_counter = c->tile_ctr + tslot;
        a.tile_base = graph ? (unsigned int)(gstep >> 1) * claims : c->tile_base[tslot];
    }
    if (claims && !L.fills) a.early_loads = 0;
    // static schedule: record per-CTA completion, and hand over per CTA if the previous launch of the stream was this plan
    if (spec && !claims && !graph) {
        if (!c->chain_done) {
            const size_t nb = sizeof(unsigned int) * (size_t)std::max(spec_capacity(1), spec_capacity(2));
            CUDA_TRY(c, cudaMalloc(&c->chain_done, nb));
            CUDA_TRY(c, cudaMemsetAsync(c->chain_done, 0, nb, c->stream));
            c->tail_own_step = false;
        }
        a.chain_done = c->chain_done;
        a.chain_seq = ++c->chain_seq;
        a.chain = (c->chain_steps && c->early_loads && c->tail_own_step && c->chain_key == (const void *)&F && L.fills) ? 1 : 0;
        if (!a.chain && !c->tail_own_step) a.early_loads = 0;
    }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (!graph && c->profile_kernel && c->prof_used < 8192 && (c->prof_seq++ % c->profile_kernel) == 0) {
        while (c->prof_ev.size() < c->prof_used + 2) {
            cudaEvent_t e;
            CUDA_TRY(c, cudaEventCreate(&e));
            c->prof_ev.push_back(e);
        }
        e0 = c->prof_ev[c->prof_used];
        e1 = c->prof_ev[c->prof_used + 1];
        c->prof_used += 2;
        CUDA_TRY(c, cudaEventRecord(e0, c->stream));
    }
    if (launch_fused(P, L, a, c->stream, &nlaunch)) return fail(c, FC_ERR_CUDA, "fused launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (e1) CUDA_TRY(c, cudaEventRecord(e1, c->stream));
    c->launches += nlaunch;
    if (!graph) {
        c->tile_base[tslot] += claims;
        c->fold_pending = false;      // (the launch took the previous step's rows along)
        c->tail_own_step = spec;
        c->chain_key = (spec && !claims) ? (const void *)&F : nullptr;
    }
    if (P.diag) {
        if (spec) {
            if (!graph) {
                c->fold = make_fold(P, L, a);
                c->fold_pending = true;
            }
        } else if (int rc = finalize_chunk(c, P, L, a, c->stream)) {
            return rc;
        }
        if (!graph) diag_step_done(c, F);
    }
    if (!F.extra.empty())
        if (int rc = run_ops(c, F.extra)) return rc;
    return FC_OK;
}

static int run_fused(fc_context *c, FusedBundle &F, bool async_device_only)
{
    const FusedPlan &P = F.plan;
    const double *bias = P.t.bias ? bias_slab(c) : nullptr;
    bool any_host = false;
    for (int b : F.in_bufs) any_host = any_host || !c->bufs[b].user_is_device;
    for (int b : F.out_bufs) any_host = any_host || !c->bufs[b].user_is_device;
    for (const HOp &h : F.extra)
        for (int b : {h.out, h.in[0], h.in[1]})
            if (b >= 0) any_host = any_host || !c->bufs[b].user_is_device;
    if (async_device_only && any_host) return fail(c, FC_ERR_STATE, "fc_run_steps needs device-resident fields (bind device pointers)");
    int nlaunch = 0;

    if (!any_host) return launch_resident(c, F, bias, -1);

    // host-pointer mode: chunked H2D -> kernel -> D2H pipeline over three streams (copy engines
    // and SMs overlap; inputs of chunk k+1 travel while chunk k computes and chunk k-1 returns)
    const int K = (int)F.chunks.size();
    // what travels: inputs the host may have rewritten (everything not marked static, and static arrays not uploaded
    // yet), results the host will read (everything computed, or with option "download" = 1 only the registered output
    // fields -- what the reference hands to oasis_put, flux_calculator.F90:909-936,999-1026)
    std::vector<int> up, down;
    for (int b : F.in_bufs) {
        const Buffer &B = c->bufs[b];
        if (!B.user_is_device && !(B.is_static && B.dev_valid)) up.push_back(b);
    }
    {
        std::set<int> sent;
        const bool sent_only = c->download_sent_only && F.extra.empty();
        if (sent_only)
            for (const OutputField &o : c->outputs)
                if (c->slot[o.surface_type][o.grid][o.idx] >= 0) sent.insert(c->slot[o.surface_type][o.grid][o.idx]);
        for (int b : F.out_bufs)
            if (!c->bufs[b].user_is_device && (!sent_only || sent.count(b))) down.push_back(b);
    }
    FusedStepArgs a{};
    a.bias = bias;
    if (int rc = flush_fold(c)) return rc;
    if (P.diag)
        if (int rc = ensure_diag_storage(c, P, F.chunks.data(), K, a)) return rc;
    c->tail_own_step = false;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    for (int k = 0; k < K; ++k) {
        cudaStream_t s = c->pipe[k % 3];
        int64_t c0[4], c1[4];
        chunk_range(c, k, K, c0, c1);
        for (int b : up) {
            const Buffer &B = c->bufs[b];
            const int64_t cnt = c1[B.grid] - c0[B.grid];
            if (cnt <= 0) continue;
            CUDA_TRY(c, cudaMemcpyAsync(B.dev + c0[B.grid], B.user + c0[B.grid], (size_t)cnt * sizeof(double), cudaMemcpyHostToDevice, s));
            c->h2d_bytes += cnt * (int64_t)sizeof(double);
        }
        const FusedLaunch &L = F.chunks[(size_t)k];
        FusedStepArgs q = a;
        if (P.diag) diag_chunk_view(c, a, k, K, q);
        if (int rc = attach_tile_counter(c, L, q, k)) return rc;
        c->tile_base[k] += L.claims;
        if (launch_fused(P, L, q, s, &nlaunch)) return fail(c, FC_ERR_CUDA, "fused launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (P.diag) {
            if (L.spec) {      // the chunk's rows -> the chunk's result vector, right behind it on its stream
                if (launch_diag_fold(make_fold(P, L, q), s)) return fail(c, FC_ERR_CUDA, "diag fold launch failed");
                nlaunch += 1;
            } else if (int rc = finalize_chunk(c, P, L, q, s)) {
                return rc;
            }
        }
        for (int b : down) {
            const Buffer &B = c->bufs[b];
            const int64_t cnt = c1[B.grid] - c0[B.grid];
            if (cnt <= 0) continue;
            CUDA_TRY(c, cudaMemcpyAsync(B.user + c0[B.grid], B.dev + c0[B.grid], (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, s));
            c->d2h_bytes += cnt * (int64_t)sizeof(double);
        }
    }
    c->launches += nlaunch;
    for (int k = 0; k < 3; ++k) CUDA_TRY(c, cudaStreamSynchronize(c->pipe[k]));
    for (int b : up) c->bufs[b].dev_valid = true;
    if (P.diag) {
        if (K > 1) {      // fold the chunks' result vectors in chunk order
            if (launch_diag_combine(c->diag_chunk_out, K, a.diag_out, c->stream)) return fail(c, FC_ERR_CUDA, "diag combine launch failed");
            c->launches += 1;
        }
        diag_step_done(c, F);
    }
    if (!F.extra.empty())
        if (int rc = run_ops(c, F.extra)) return rc;
    return FC_OK;
}

// do_regridding (flux_calculator_basic.F90:463-522) of variable idx for surface type st (0 = all), in the reference's
// order u->t, v->t, t->u, t->v, for a context that knows the namelist's regridding requests (fc_create_from_namelist)
static int sa_regrid_var(fc_context *c, int idx, int st)
{
    static const int from[4] = {2, 3, 1, 1}, to[4] = {1, 1, 2, 3};
    Standalone &R = *c->sa;
    for (int j = 1; j <= FC_MAX_SURFACE_TYPES; ++j) {
        if (!(j == st || st == 0)) continue;
        for (int d = 0; d < 4; ++d) {
            const SaSlot &src = R.slot[j][from[d]][idx], &dst = R.slot[j][to[d]][idx];
            if (!src.put[to[d]] || src.arr < 0 || dst.arr < 0) continue;
            if (!c->regrid[d].set)
                return fail(c, FC_ERR_STATE, "the namelist asks for regridding %s from the %s to the %s but no matrix was set (fc_set_regrid_matrix, direction %d)",
                            kVarNames[idx], kGridNames[from[d]], kGridNames[to[d]], d);
            if (int rc = fc_regrid(c, d, R.arrays[(size_t)dst.arr].host, R.arrays[(size_t)src.arr].host)) return rc;
        }
    }
    return FC_OK;
}

// received fields of one phase (flux_calculator.F90:891-896 early, :961-966 normal)
static int sa_regrid_inputs(fc_context *c, bool early)
{
    for (const SaField &f : c->sa->in)
        if (f.early == early)
            if (int rc = sa_regrid_var(c, f.idx, f.type)) return rc;
    return FC_OK;
}

static int step_impl(fc_context *c, int which, int64_t t, bool async_device_only)
{
    if (int rc = ensure_prepared(c)) return rc;
    cudaSetDevice(c->device);
    c->time = t;                       // current_step_time (flux_calculator.F90:861)
    c->h2d_bytes = c->d2h_bytes = 0;
    if (c->sa && !c->sa->regrid.empty()) {
        if (which == 0 || which == 2)
            if (int rc = sa_regrid_inputs(c, true)) return rc;
        if (which == 1 || which == 2)
            if (int rc = sa_regrid_inputs(c, false)) return rc;
        if (c->sa->regrid.size() > c->sa->n_input_regrid) {
            // a COMPUTED field is regridded between two calculators (flux_calculator.F90:903, :975-989): the reference's pass
            // sequence, one calculator at a time
            if (c->diagnostics) return fail(c, FC_ERR_STATE, "diagnostics need the fused path, but regridding of computed fields requires the pass sequence");
            auto pass = [&](int (*gen)(Gen &), int idx) -> int {
                Gen G{c, {}, "", false};
                if (int rc = gen(G)) return rc;
                if (int rc = run_ops(c, G.ops)) return rc;
                return idx ? sa_regrid_var(c, idx, 0) : FC_OK;
            };
            if (which == 0 || which == 2) {
                if (int rc = pass([](Gen &G) { return gen_rbbr(G); }, FC_RBBR)) return rc;
                if (int rc = pass([](Gen &G) { return gen_send(G, true); }, 0)) return rc;
            }
            if (which == 1 || which == 2) {
                if (int rc = pass([](Gen &G) { int r = gen_qsur(G, 1); if (!r) r = gen_qsur(G, 2); if (!r) r = gen_qsur(G, 3); return r; }, FC_QSUR)) return rc;
                if (int rc = pass([](Gen &G) { return gen_meva(G); }, FC_MEVA)) return rc;
                if (int rc = pass([](Gen &G) { return gen_hlat(G); }, FC_HLAT)) return rc;
                if (int rc = pass([](Gen &G) { return gen_hsen(G); }, FC_HSEN)) return rc;
                if (int rc = pass([](Gen &G) { return gen_mom(G, 2, 0); }, FC_UMOM)) return rc;
                if (int rc = pass([](Gen &G) { return gen_mom(G, 3, 1); }, FC_VMOM)) return rc;
                if (int rc = pass([](Gen &G) { int r = gen_rsdr(G, false); if (!r) r = gen_send(G, false); return r; }, 0)) return rc;
            }
            return FC_OK;
        }
    }
    FusedBundle &F = c->fused[which];
    if (F.ok) return run_fused(c, F, async_device_only);
    if (async_device_only) {
        for (auto &B : c->bufs)
            if (B.user && !B.user_is_device) return fail(c, FC_ERR_STATE, "fc_run_steps needs device-resident fields (bind device pointers)");
    }
    if (c->diagnostics) return fail(c, FC_ERR_STATE, "diagnostics need the fused path, but this configuration requires the generic path");
    Gen G{c, {}, "", false};
    if (which == 0 || which == 2)
        if (int rc = gen_early(G)) return rc;
    if (which == 1 || which == 2)
        if (int rc = gen_normal(G)) return rc;
    return run_ops(c, G.ops);
}

extern "C" int fc_step_early(fc_context *c, int64_t t) { return step_impl(c, 0, t, false); }
extern "C" int fc_step_normal(fc_context *c, int64_t t) { return step_impl(c, 1, t, false); }
extern "C" int fc_step_all(fc_context *c, int64_t t) { return step_impl(c, 2, t, false); }

// ---------------------------------------------------------------------------------------------
// fc_run_steps: consecutive coupling steps as CUDA graphs (the time loop of flux_calculator.F90:859-1028 with the
// fields resident on the device).  The only thing that changes from step to step is the month slab of the bias
// corrections (calculate.F90:66-73,112-116), so the steps of one calendar month are replays of ONE captured graph of
// kGraphSteps step launches (programmatic dependent launch edges between them are captured as such); what is left
// over at the end of a month is issued directly.  Graphs are kept per (month, length) until the next fc_prepare.
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int kGraphSteps = 32;      // step launches per graph (even: the tile counters alternate)

int capture_steps(fc_context *c, const FusedBundle &F, int month, int nsteps, cudaGraphExec_t *exec)
{
    const double *bias = F.plan.t.bias ? c->corr_dev + (size_t)(month - 1) * (size_t)corr_stride(c->n[1]) : nullptr;
    // everything that allocates or synchronises happens before the capture
    if (int rc = flush_fold(c)) return rc;
    if (F.step.claims)
        if (int rc = ensure_tile_counters(c)) return rc;
    if (F.plan.diag) {
        FusedStepArgs unused{};
        if (int rc = ensure_diag_storage(c, F.plan, &F.step, 1, unused)) return rc;
    }
    cudaGraph_t graph = nullptr;
    CUDA_TRY(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    int rc = FC_OK;
    if (F.step.claims && cudaMemsetAsync(c->tile_ctr + kMaxChunks, 0, 2 * sizeof(unsigned int), c->stream) != cudaSuccess)
        rc = fail(c, FC_ERR_CUDA, "fc_run_steps: memset node failed");
    for (int s = 0; s < nsteps && rc == FC_OK; ++s) rc = launch_resident(c, F, bias, s);
    const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
    if (rc != FC_OK) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    if (e != cudaSuccess || !graph) return fail(c, FC_ERR_CUDA, "fc_run_steps: stream capture failed: %s", cudaGetErrorString(e));
    const cudaError_t ei = cudaGraphInstantiate(exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) return fail(c, FC_ERR_CUDA, "fc_run_steps: cudaGraphInstantiate failed: %s", cudaGetErrorString(ei));
    return FC_OK;
}
}  // namespace

extern "C" int fc_run_steps(fc_context *c, int64_t t0, int64_t dt, int nsteps)
{
    if (!c || nsteps < 0) return fail(c, FC_ERR_ARG, "fc_run_steps: bad argument");
    if (int rc = ensure_prepared(c)) return rc;
    cudaSetDevice(c->device);
    FusedBundle &F = c->fused[2];
    bool resident = F.ok;
    if (resident) {
        for (int b : F.in_bufs) resident = resident && c->bufs[b].user_is_device;
        for (int b : F.out_bufs) resident = resident && c->bufs[b].user_is_device;
        for (const HOp &h : F.extra)
            for (int b : {h.out, h.in[0], h.in[1]})
                if (b >= 0) resident = resident && c->bufs[b].user_is_device;
    }
    const bool graphs = resident && !c->profile_kernel;
    int k = 0;
    while (k < nsteps) {
        const int64_t t = t0 + (int64_t)k * dt;
        const int month = F.ok && F.plan.t.bias ? fc_current_month(c->init_date, t) : 1;
        int run = 1;      // steps k .. k + run - 1 share the month
        while (k + run < nsteps && (!(F.ok && F.plan.t.bias) || fc_current_month(c->init_date, t0 + (int64_t)(k + run) * dt) == month)) ++run;
        while (graphs && run >= kGraphSteps) {
            cudaGraphExec_t &g = c->step_graph[month];
            if (!g)
                if (int rc = capture_steps(c, F, month, kGraphSteps, &g)) return rc;
            if (int rc = flush_fold(c)) return rc;      // (a directly issued step before this graph left its rows)
            CUDA_TRY(c, cudaGraphLaunch(g, c->stream));
            c->graph_launches += 1;
            c->launches += (int64_t)kGraphSteps * (1 + (F.extra.empty() ? 0 : 1));
            k += kGraphSteps;
            run -= kGraphSteps;
            // state as the graph leaves it: time, tile counters, the last step's diagnostics rows (set 0) not folded yet
            c->time = t0 + (int64_t)(k - 1) * dt;
            if (F.step.claims) c->tile_base[kMaxChunks] = c->tile_base[kMaxChunks + 1] = (unsigned int)(kGraphSteps / 2) * F.step.claims;
            c->tail_own_step = F.step.spec && F.extra.empty();
            c->chain_key = nullptr;
            if (F.plan.diag) {
                FusedStepArgs a{};
                a.diag_partials = c->diag_partials;
                a.diag_rows = c->diag_rows_1;
                a.diag_out = c->diag_buf[c->diag_cur ^ 1];
                c->row_set = 0;
                if (F.step.spec) {
                    c->fold = make_fold(F.plan, F.step, a);
                    c->fold_pending = true;
                }
                diag_step_done(c, F);
            }
        }
        for (int r = 0; r < run; ++r, ++k)
            if (int rc = step_impl(c, 2, t0 + (int64_t)k * dt, true)) return rc;
    }
    return FC_OK;
}

// CUDA-event timing on the context's stream (the stream the kernels are launched on)
extern "C" int fc_event_record(fc_context *c, int which)
{
    if (!c || which < 0 || which > 1) return fail(c, FC_ERR_ARG, "fc_event_record: bad argument");
    cudaSetDevice(c->device);
    if (!c->user_ev[which]) CUDA_TRY(c, cudaEventCreate(&c->user_ev[which]));
    for (int b = 0; b < 2; ++b)      // an event on the main stream also covers all-reduces still running on the side stream
        if (c->comm_busy[b]) {
            CUDA_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_comm[b], 0));
            c->comm_busy[b] = false;
        }
    CUDA_TRY(c, cudaEventRecord(c->user_ev[which], c->stream));
    return FC_OK;
}

extern "C" int fc_event_elapsed_ms(fc_context *c, double *ms)
{
    if (!c || !ms || !c->user_ev[0] || !c->user_ev[1]) return fail(c, FC_ERR_ARG, "fc_event_elapsed_ms: record events 0 and 1 first");
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaEventSynchronize(c->user_ev[1]));
    float f = 0.f;
    CUDA_TRY(c, cudaEventElapsedTime(&f, c->user_ev[0], c->user_ev[1]));
    *ms = f;
    return FC_OK;
}

extern "C" int fc_kernel_time_ms(fc_context *c, double *total_ms, int64_t *count)
{
    if (!c || !total_ms || !count) return fail(c, FC_ERR_ARG, "fc_kernel_time_ms: NULL argument");
    cudaSetDevice(c->device);
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    double t = 0.0;
    for (size_t k = 0; k + 1 < c->prof_used; k += 2) {
        float f = 0.f;
        CUDA_TRY(c, cudaEventElapsedTime(&f, c->prof_ev[k], c->prof_ev[k + 1]));
        t += f;
    }
    *total_ms = t;
    *count = (int64_t)(c->prof_used / 2);
    c->prof_used = 0;
    return FC_OK;
}

extern "C" int64_t fc_get_info(const fc_context *c, const char *name)
{
    if (!c || !name) return -1;
    if (!strcmp(name, "launches")) return c->launches;
    if (!strcmp(name, "graph_launches")) return c->graph_launches;
    if (!strcmp(name, "exact_path_calls")) {   // threads that recomputed their cells with the IEEE routines (process-wide)
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        return (int64_t)read_exact_calls();
    }
    if (!strcmp(name, "fused")) return (!c->dirty && c->fused[2].ok) ? 1 : 0;
    if (!strcmp(name, "spec_kernel")) {   // fc_step_all runs on the specialised persistent kernel (spec_kernel.cu)
        return (!c->dirty && c->fused[2].ok && c->fused[2].step.spec) ? 1 : 0;
    }
    if (!strcmp(name, "fused_early")) return (!c->dirty && c->fused[0].ok) ? 1 : 0;
    if (!strcmp(name, "fused_normal")) return (!c->dirty && c->fused[1].ok) ? 1 : 0;
    if (!strcmp(name, "h2d_bytes_per_step")) return c->h2d_bytes;
    if (!strcmp(name, "d2h_bytes_per_step")) return c->d2h_bytes;
    if (!strcmp(name, "bytes_per_cell")) {
        // algorithmic bytes of fc_step_all per (t,u,v) cell triple: 8 * (unique arrays read + arrays written)
        if (c->dirty || !c->fused[2].ok) return 0;
        const FusedBundle &F = c->fused[2];
        int64_t arrays = (int64_t)F.in_bufs.size() + (int64_t)F.out_bufs.size();
        if (F.plan.t.bias) arrays += 1;
        if (F.plan.diag) arrays += 3;
        return 8 * arrays;
    }
    return -1;
}

// ---------------------------------------------------------------------------------------------
// diagnostics
// ---------------------------------------------------------------------------------------------
static int diag_slot_for(int i, int g, int idx)
{
    int q = -1;
    if (g == 1) {
        switch (idx) {
            case FC_QSUR: q = DQ_QSUR_T; break;
            case FC_MEVA: q = DQ_MEVA; break;
            case FC_HLAT: q = DQ_HLAT; break;
            case FC_HSEN: q = DQ_HSEN; break;
            case FC_RBBR: q = DQ_RBBR; break;
            case FC_RSDR: q = DQ_RSDR; break;
        }
    } else if (g == 2) {
        if (idx == FC_QSUR) q = DQ_QSUR_U;
        if (idx == FC_UMOM) q = DQ_UMOM;
    } else if (g == 3) {
        if (idx == FC_QSUR) q = DQ_QSUR_V;
        if (idx == FC_VMOM) q = DQ_VMOM;
    }
    return q < 0 ? -1 : i * DQ_COUNT + q;
}

namespace fc {
int diag_fetch(fc_context *c)
{
    if (c->diag_valid) return FC_OK;
    if (c->diag_active.empty()) return fail(c, FC_ERR_STATE, "no diagnostics available: enable option 'diagnostics' and run a step");
    cudaSetDevice(c->device);
    if (int rc = flush_fold(c)) return rc;
    const int b = c->diag_cur;
    if (c->comm_busy[b]) {      // the all-reduce of this buffer runs on the side stream
        CUDA_TRY(c, cudaStreamWaitEvent(c->stream, c->ev_comm[b], 0));
        c->comm_busy[b] = false;
    }
    double *planes = c->diag_host + kDiagSlots * 3;
    if (c->p2p && c->diag_global) {      // global values from the peer mailboxes, folded in rank order
        if (int rc = p2p_fetch(c, planes, (int)c->diag_active.size(), c->diag_level)) return rc;
    } else {
        CUDA_TRY(c, cudaMemcpyAsync(planes, c->diag_buf[b], sizeof(double) * kDiagSlots * 3, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    for (size_t k = 0; k < c->diag_active.size(); ++k)
        for (int j = 0; j < 3; ++j) c->diag_host[c->diag_active[k] * 3 + j] = planes[j * kDiagSlots + k];
    c->diag_valid = true;
    return FC_OK;
}
}  // namespace fc

extern "C" int fc_get_diagnostics(fc_context *c, int i, int g, int idx, double out[3])
{
    if (!c || !out) return fail(c, FC_ERR_ARG, "fc_get_diagnostics: NULL argument");
    const int s = (i >= 0 && i <= FC_MAX_SURFACE_TYPES) ? diag_slot_for(i, g, idx) : -1;
    if (s < 0) return fail(c, FC_ERR_ARG, "fc_get_diagnostics: no diagnostics slot for this field");
    if (std::find(c->diag_active.begin(), c->diag_active.end(), s) == c->diag_active.end())
        return fail(c, FC_ERR_STATE, "fc_get_diagnostics: %s of surface_type %d was not computed by the last step", kVarNames[idx], i);
    if (int rc = diag_fetch(c)) return rc;
    for (int j = 0; j < 3; ++j) out[j] = c->diag_host[s * 3 + j];
    if (c->diag_level < 2) out[1] = out[2] = nan("");   // min/max only at diagnostics level 2
    return FC_OK;
}

extern "C" int fc_allreduce_diagnostics(fc_context *c)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (c->diag_active.empty()) return fail(c, FC_ERR_STATE, "no diagnostics to reduce");
    if (c->p2p) {
        // one more exchange: its record goes into every rank's mailbox together with the fold of the step's rows -- by the
        // next step's kernel, or by fc_get_diagnostics / fc_synchronize, whichever comes first -- or right now if the
        // result vector is already complete (generic kernels, host-pointer pipeline)
        PeerPost post;
        p2p_make_post(c, post);
        if (c->fold_pending) {
            c->fold.post = post;
        } else {
            cudaSetDevice(c->device);
            if (launch_diag_post(c->diag_buf[c->diag_cur], post, (int)c->diag_active.size(), c->stream)) return fail(c, FC_ERR_CUDA, "diag post launch failed");
            c->launches += 1;
            c->tail_own_step = false;
        }
        c->diag_valid = false;
        c->diag_global = true;
        return FC_OK;
    }
    if (c->nranks <= 1 || !c->nccl_comm) return FC_OK;   // single rank: local == global
    c->diag_valid = false;
    if (int rc = flush_fold(c)) return rc;
    return nccl_allreduce_diag(c);
}

// ---------------------------------------------------------------------------------------------
// regridding ("next" row): do_regridding, basic.F90:463-522
// ---------------------------------------------------------------------------------------------
extern "C" int fc_set_regrid_matrix(fc_context *c, int dir, int64_t nnz, const int32_t *src_index, const int32_t *dst_index,
                                    const double *weight)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (dir < 0 || dir > 3 || nnz < 0 || (nnz > 0 && (!src_index || !dst_index || !weight)))
        return fail(c, FC_ERR_ARG, "fc_set_regrid_matrix: bad argument");
    cudaSetDevice(c->device);
    static const int src_grid[4] = {2, 3, 1, 1}, dst_grid[4] = {1, 1, 2, 3};   // u->t, v->t, t->u, t->v
    RegridMatrix &M = c->regrid[dir];
    free_regrid(M);
    M.nnz = nnz;
    M.n_src = c->n[src_grid[dir]];
    M.n_dst = c->n[dst_grid[dir]];
    // stable counting sort by destination keeps the reference's per-cell accumulation order (:483-486)
    std::vector<int64_t> row_ptr(M.n_dst + 1, 0);
    for (int64_t k = 0; k < nnz; ++k) {
        const int64_t d = dst_index[k], s = src_index[k];
        if (d < 1 || d > M.n_dst || s < 1 || s > M.n_src)
            return fail(c, FC_ERR_ARG, "fc_set_regrid_matrix: element %lld has index out of range (src %lld, dst %lld)", (long long)k,
                        (long long)s, (long long)d);
        row_ptr[d]++;
    }
    for (int64_t r = 0; r < M.n_dst; ++r) row_ptr[r + 1] += row_ptr[r];
    std::vector<int32_t> s_sorted(nnz);
    std::vector<double> w_sorted(nnz);
    {
        std::vector<int64_t> cur(row_ptr.begin(), row_ptr.end() - 1);
        for (int64_t k = 0; k < nnz; ++k) {
            const int64_t pos = cur[dst_index[k] - 1]++;
            s_sorted[pos] = src_index[k] - 1;
            w_sorted[pos] = weight[k];
        }
    }
    CUDA_TRY(c, cudaMalloc(&M.row_ptr, sizeof(int64_t) * (M.n_dst + 1)));
    CUDA_TRY(c, cudaMalloc(&M.src_idx, sizeof(int32_t) * std::max<int64_t>(nnz, 1)));
    CUDA_TRY(c, cudaMalloc(&M.weight, sizeof(double) * std::max<int64_t>(nnz, 1)));
    CUDA_TRY(c, cudaMemcpy(M.row_ptr, row_ptr.data(), sizeof(int64_t) * (M.n_dst + 1), cudaMemcpyHostToDevice));
    if (nnz) {
        CUDA_TRY(c, cudaMemcpy(M.src_idx, s_sorted.data(), sizeof(int32_t) * nnz, cudaMemcpyHostToDevice));
        CUDA_TRY(c, cudaMemcpy(M.weight, w_sorted.data(), sizeof(double) * nnz, cudaMemcpyHostToDevice));
    }
    M.set = true;
    return FC_OK;
}

extern "C" int fc_regrid(fc_context *c, int dir, double *dst, const double *src)
{
    if (!c) return fail(nullptr, FC_ERR_ARG, "NULL context");
    if (dir < 0 || dir > 3 || !dst || !src) return fail(c, FC_ERR_ARG, "fc_regrid: bad argument");
    RegridMatrix &M = c->regrid[dir];
    if (!M.set) return fail(c, FC_ERR_STATE, "fc_regrid: matrix %d not set", dir);
    cudaSetDevice(c->device);
    c->tail_own_step = false;
    bool sd, sp, dd, dp;
    classify_pointer(src, &sd, &sp, nullptr);
    classify_pointer(dst, &dd, &dp, nullptr);
    const double *s_dev = src;
    double *d_dev = dst, *ts = nullptr, *td = nullptr;
    if (!sd) {
        CUDA_TRY(c, cudaMalloc(&ts, sizeof(double) * std::max<int64_t>(M.n_src, 1)));
        CUDA_TRY(c, cudaMemcpyAsync(ts, src, sizeof(double) * M.n_src, cudaMemcpyHostToDevice, c->stream));
        s_dev = ts;
    }
    if (!dd) {
        CUDA_TRY(c, cudaMalloc(&td, sizeof(double) * std::max<int64_t>(M.n_dst, 1)));
        d_dev = td;
    }
    if (launch_regrid_csr(M.row_ptr, M.src_idx, M.weight, s_dev, d_dev, M.n_dst, c->stream))
        return fail(c, FC_ERR_CUDA, "regrid launch failed");
    if (M.n_dst > 0) c->launches++;
    if (!dd) CUDA_TRY(c, cudaMemcpyAsync(dst, td, sizeof(double) * M.n_dst, cudaMemcpyDeviceToHost, c->stream));
    if (!dd || !sd) {
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
        cudaFree(ts);
        cudaFree(td);
    }
    return FC_OK;
}
