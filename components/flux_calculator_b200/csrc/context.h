// context.h -- host-side state behind fc_context: the local_field registry, method strings,
// bias corrections, send list, and the plans derived from them.
#pragma once

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../../include/fluxcalc.h"
#include "plan.h"

struct fc_context;

namespace fc {

struct Buffer {
    double *user = nullptr;      // pointer the host bound (host or device memory)
    double *dev = nullptr;       // device pointer the kernels use (== user for device memory)
    int64_t n = 0;
    int grid = 0;
    bool user_is_device = false;
    bool user_is_pinned = false;
    bool registered = false;     // we called cudaHostRegister on it
    bool is_static = false;      // fc_mark_static: the host does not rewrite it between steps (a namelist constant, val_*)
    bool dev_valid = false;      // ... and the device mirror already holds it
    int refs = 0;
};

// host-side op: device pointers are resolved from buffer ids at launch time
struct HOp {
    int code = 0;
    double cst = 0.0;
    int grid = 1;
    int out = -1, out2 = -1;     // buffer ids (-1: none)
    int in[8] = {-1, -1, -1, -1, -1, -1, -1, -1};
    int n_in = 0;
    bool in0_is_bias = false;    // in[0] is the month slab of the corrections
};

struct OutputField {
    int surface_type, grid, idx;
    bool early;
};

struct RegridMatrix {
    bool set = false;
    int64_t nnz = 0, n_dst = 0, n_src = 0;
    int64_t *row_ptr = nullptr;  // device, n_dst+1
    int32_t *src_idx = nullptr;  // device, 0-based, grouped by destination in original element order
    double *weight = nullptr;    // device
};

constexpr int kMaxChunks = 16;   // chunks of the host-pointer pipeline (measured on C4: 8 -> 38.3 ms, 16 -> 37.7 ms, 32 -> 38.7 ms per step)

enum Quantity { Q_QSUR_T = 0, Q_QSUR_U, Q_QSUR_V, Q_MEVA, Q_HLAT, Q_HSEN, Q_MOM, Q_RBBR, Q_COUNT };

struct FusedBundle {
    bool ok = false;
    FusedPlan plan;
    FusedLaunch step;                     // how the plan launches as a device-resident step (kernels.cu: resolve_fused)
    std::vector<FusedLaunch> chunks;      // ... and as the chunks of the host-pointer pipeline
    std::vector<int> in_bufs, out_bufs;   // buffers to upload / download in host-pointer mode
    std::vector<HOp> extra;               // averaging of pass-through variables (run after the fused launch)
    // diagnostics slot -> (surface type, grid, var) of the active slots, compact order
    std::vector<int> diag_slots;
};

// what fc_create_from_namelist builds from flux_calculator.nml (frontend.cu): the arrays a Fortran host would ALLOCATE and the
// reference's registry / field lists on top of them
struct SaArray {
    int grid = 1;
    double *host = nullptr;      // page-locked, owned by the context
    double fill = 0.0;           // constant from the namelist (val_*), or default value of a flux nobody computes (val_flux_*)
    bool has_fill = false, constant = false;
};
struct SaSlot {
    int arr = -1;                // index into arrays (-1: disassociated); aliases share it
    bool allocated = false;      // %allocated (basic.F90:88)
    bool put[4] = {false, false, false, false};      // put_to_t/u/v_grid (basic.F90:89-91), index = destination grid
};
struct SaField {
    std::string name;            // OASIS name: R|S + model letter + variable + two-digit surface type (basic.F90:149, :266)
    int grid = 1, type = 0, idx = 0;
    bool early = false;
};
struct SaRegrid {
    int type, idx, from, to;
};
struct Standalone {
    int S = 0;
    char letter = 'M';
    int64_t n[4] = {0, 0, 0, 0};
    std::vector<SaArray> arrays;
    SaSlot slot[FC_MAX_SURFACE_TYPES + 1][4][FC_MAX_VARNAMES + 1];
    std::vector<SaField> in, out;
    std::vector<SaRegrid> regrid;        // in the order prepare_regridding creates them: first those of received fields ...
    size_t n_input_regrid = 0;           // ... then those of computed ones
    std::string method[8][FC_MAX_SURFACE_TYPES + 1];
    std::string warnings;
};
void standalone_free(Standalone &R);

extern thread_local std::string g_last_error;
int fail(fc_context *ctx, int code, const char *fmt, ...);
int classify_pointer(const void *p, bool *is_device, bool *is_pinned, int *device);
int diag_fetch(fc_context *c);
int flush_fold(fc_context *c);

}  // namespace fc

#define CUDA_TRY(ctx, call)                                                                                  \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess)                                                                               \
            return fc::fail(ctx, FC_ERR_CUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, \
                            __LINE__, #call);                                                                \
    } while (0)

struct fc_context {
    int device = 0;
    int S = 1;
    int64_t n[4] = {0, 0, 0, 0};
    cudaStream_t stream = nullptr;
    cudaStream_t pipe[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t pipe_done[3] = {nullptr, nullptr, nullptr};

    std::vector<fc::Buffer> bufs;
    int slot[FC_MAX_SURFACE_TYPES + 1][4][FC_MAX_VARNAMES + 1];
    signed char alloc_flag[FC_MAX_SURFACE_TYPES + 1][4][FC_MAX_VARNAMES + 1];   // %allocated as stated by the host: -1 = infer from aliasing
    int method[fc::Q_COUNT][FC_MAX_SURFACE_TYPES + 1];
    int dist_sw = -1;            // -1 auto, 0 off, 1 on

    // bias corrections, month-major [12][n_t] on the device
    double *corr_dev = nullptr;
    bool corr_enabled = false;
    int init_date = 19000101;
    double *area_dev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool area_owned[4] = {false, false, false, false};

    std::vector<fc::OutputField> outputs;
    int64_t time = 0;

    // options
    bool force_generic = false;
    bool pin_host = false;
    int diagnostics = 0;         // 0 off, 1 area-weighted sums, 2 sums + min/max
    int h2d_chunks = 0;          // 0 = auto
    int use_staged = 1;          // specialised persistent kernel (spec_kernel.cu): 0 never, >= 1 whenever the plan fits

    // derived
    bool dirty = true;
    bool strict = false;
    fc::Consts consts;
    fc::FusedBundle fused[3];    // 0 early, 1 normal, 2 all

    // diagnostics storage
    double *diag_partials = nullptr;
    size_t diag_partials_cap = 0;
    fc::DiagFold fold;                      // rows of the last specialised step (device-resident path), not folded yet
    bool fold_pending = false;
    int row_set = 0;                        // which of the two row sets the last device-resident step wrote
    bool tail_own_step = false;             // the last operation enqueued on `stream` is a specialised step kernel
    bool early_loads = true;                // option: let such a step's successor fill its ring before griddepcontrol.wait
    // dynamic tile schedule (specialised kernel without diagnostics): monotonic claim counters, one per chunk of the host
    // pipeline plus two that alternate between consecutive device-resident steps (a step's producers may start claiming
    // while the previous step still runs); tile_base = what each counter will read before its next launch
    unsigned int *tile_ctr = nullptr;
    unsigned int tile_base[fc::kMaxChunks + 2] = {};
    int tile_par = 0;
    // chained static steps (spec_kernel.cu): per-CTA completion records, the running launch number, and which bundle issued the
    // last recorded launch (a step chains to its predecessor only if that was the same plan, directly before it on the stream)
    unsigned int *chain_done = nullptr;
    unsigned int chain_seq = 0;
    const void *chain_key = nullptr;
    bool chain_steps = true;                // option "chain"
    double *diag_chunk_out = nullptr;       // [kMaxChunks][sum|min|max][kDiagSlots]: per-chunk results (host-pointer pipeline)
    size_t diag_chunk_stride = 0;           // doubles of partial rows + reduce scratch per chunk
    int64_t diag_rows_1 = 0;                // row stride of the device-resident (one launch per step) layout
    double *diag_buf[2] = {nullptr, nullptr};   // [sum|min|max][kDiagSlots] compact slots, double buffered by step
    int diag_cur = 0;                    // buffer the last step wrote
    cudaStream_t comm_stream = nullptr;  // NCCL all-reduce runs here, overlapped with the next step
    cudaEvent_t ev_fin[2] = {nullptr, nullptr}, ev_comm[2] = {nullptr, nullptr};
    bool comm_busy[2] = {false, false};
    double *diag_host = nullptr;         // pinned copy, expanded to [kDiagSlots][3]
    std::vector<int> diag_active;        // slot ids in compact order (of the last step)
    bool diag_valid = false;
    int diag_level = 0;                  // level of the last step

    // NCCL
    void *nccl_comm = nullptr;
    int rank = 0, nranks = 1;
    // peer-memory exchange (p2p_comm.cu)
    fc::DiagMail *mailbox = nullptr;           // own mailbox [kMailDepth][nranks]
    fc::DiagMail *peer_mail[fc::kMaxPeers] = {};   // every rank's mailbox as mapped here (peer_mail[rank] == mailbox)
    bool p2p = false;                          // connected
    unsigned long long diag_seq = 0;           // number of exchanges so far (fc_allreduce_diagnostics calls, a collective)
    bool diag_global = false;                  // fc_allreduce_diagnostics was called for the last step

    fc::RegridMatrix regrid[4];

    // live timing of the fused kernel (option "profile_kernel" = n): event pairs around every n-th launch
    int profile_kernel = 0;
    int64_t prof_seq = 0;
    std::vector<cudaEvent_t> prof_ev;    // start/stop pairs, recycled
    size_t prof_used = 0;
    cudaEvent_t user_ev[2] = {nullptr, nullptr};

    fc::Standalone *sa = nullptr;        // set by fc_create_from_namelist
    // front end (frontend.cu): &correctionsctl of the last namelist read, warnings of the corrections loader
    bool nml_read = false;
    bool nml_lcorrections = false;
    std::string warning;

    // fc_run_steps: one instantiated graph of kGraphSteps step launches per calendar month (index 1..12)
    cudaGraphExec_t step_graph[13] = {};
    bool download_sent_only = false;        // option "download" = 1: only registered output fields travel back to the host
    int dyn_min_tiles = 0;                  // option: tiles per CTA from which the specialised kernel schedules dynamically (0: default)
    int64_t graph_launches = 0;
    int64_t launches = 0;
    int64_t h2d_bytes = 0, d2h_bytes = 0;   // of the last step call
    std::string err;
};
