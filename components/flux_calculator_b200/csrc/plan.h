// plan.h -- launch plans shared by the host-side plan builder and the kernels.
//
// Two kinds of plan are built from the context (bound fields + method strings):
//   * OpList    : the reference's pass sequence (flux_calculator_calculate.F90) as a list of per-cell
//                 ops on device pointers.  Executed by the op-list interpreter kernel.  Exact reference
//                 semantics for every configuration, including pointer aliasing ('copy', uniform
//                 outputs) because each op reads/writes global memory in the reference's order.
//   * FusedPlan : the same work for "canonical" configurations (no aliased outputs) as ONE pass over
//                 SoA fields with every intermediate in registers.
// How a FusedPlan is launched over a cell range -- specialised or generic kernel, grid, schedule, diagnostics rows -- is
// decided in one place, resolve_fused (kernels.cu, with spec_resolve in spec_kernel.cu for the specialised kernel), once
// per prepared plan; the result is a FusedLaunch.  A step fills in its FusedStepArgs and calls launch_fused.
#pragma once

#include <stdint.h>
#include <string.h>

#include "formulas.cuh"

namespace fc {

enum Method : int {
    M_NONE = 0,
    M_ZERO,
    M_COPY,
    M_CCLM,
    M_MOM5,
    M_RCO,
    M_WATER,
    M_ICE,
    M_STBO,
    M_INVALID = -1
};

constexpr int kMaxSurfaceTypes = 10;
constexpr int kMaxVars = 35;

// ---------------------------------------------------------------------------------------------
// op-list interpreter
// ---------------------------------------------------------------------------------------------
enum OpCode : int {
    OP_ZERO = 0,      // out = 0.0
    OP_COPY,          // out = in0                                     (distribute_radiation_flux)
    OP_QSUR_CCLM,     // out = q_s(in0=FICE, in1=PSUR, in2=TSUR)
    OP_MEVA_CCLM,     // out = evap(in0=a, in1=PSUR, in2=QATM, in3=QSUR, in4=T, in5=U, in6=V)
    OP_MEVA_RCO,      // out = evap(in0=QATM, in1=TSUR, in2=U, in3=V)
    OP_ADD,           // out = out + in0                               (bias correction)
    OP_SCALE,         // out = in0 * cst                               (latent heat)
    OP_HSEN_CCLM,     // out = hsen(in0=a, in1=PATM, in2=PSUR, in3=q, in4=TATM, in5=TSUR, in6=U, in7=V)
    OP_HSEN_RCO,      // out = hsen(in0=TATM, in1=TSUR, in2=U, in3=V)
    OP_MOM_CCLM,      // out/out2 = tau(in0=a, in1=PSUR, in2=QSUR, in3=TSUR, in4=U, in5=V)
    OP_MOM_RCO,       // out/out2 = tau(in0=U, in1=V)
    OP_RBBR,          // out = cst * in0**4
    OP_MULADD         // out = out + in0*in1                           (average_across_surface_types)
};

struct Op {
    int code;
    int pad;
    double cst;
    double *out;
    double *out2;          // second result of the momentum routines (north), may be null
    const double *in[8];
};

constexpr int kMaxOps = 160;   // 10 types x (<=9 calculators + bias) + averaging of a few fields

struct OpList {
    int n;
    int pad;
    Op ops[kMaxOps];
};

// ---------------------------------------------------------------------------------------------
// fused plan
// ---------------------------------------------------------------------------------------------
struct FusedTType {     // one surface type on the t grid
    const double *fice, *psur, *tsur, *qatm, *tatm, *patm, *uatm, *vatm;
    const double *a_evap;    // AMOI (CCLM) or CMOI (MOM5)
    const double *a_sens;    // AMOI (CCLM) or CHEA (MOM5)
    const double *qsur_in;   // QSUR when it is an input (method 'none' but bound)
    const double *fare;
    double *qsur, *meva, *hlat, *hsen, *rbbr, *rsdr;
    int m_qsur, m_meva, m_hlat, m_hsen, m_rbbr, pad;
    double latent_heat;      // L_v (water) or L_s (ice)
};

struct FusedUVType {    // one surface type on the u or v grid
    const double *fice, *psur, *tsur, *a_mom, *uatm, *vatm, *qsur_in, *fare;
    double *qsur, *mom;      // mom = UMOM on the u grid, VMOM on the v grid
    int m_qsur, m_mom;
};

struct FusedT {
    int64_t n;
    const double *rsdd;      // RSDD of surface type 0 (null: no shortwave distribution)
    const double *bias;      // corrections[month-1][0..n) or null
    const double *area;      // cell areas (diagnostics) or null
    // type-0 area-fraction averages (null = not averaged)
    double *avg_qsur, *avg_meva, *avg_hlat, *avg_hsen, *avg_rbbr, *avg_rsdr;
    FusedTType ty[kMaxSurfaceTypes];
};

struct FusedUV {
    int64_t n;
    int north;               // 0: east component (u grid), 1: north component (v grid)
    int pad;
    const double *area;
    double *avg_qsur, *avg_mom;
    FusedUVType ty[kMaxSurfaceTypes];
};

// Peer-memory exchange of the diagnostics (p2p_comm.cu): every rank owns a mailbox [parity][source rank] of DiagMail
// records; the last CTA of a step's kernel stores the rank's result vector into the mailbox of EVERY rank over
// NVLink.  Every double travels as two self-validating 8-byte words (32 data bits + the step's 32-bit sequence number,
// the layout of NCCL's LL protocol): an aligned 8-byte store is single-copy atomic, so no fence, no barrier and no
// separate flag store are needed on the writer's side -- the stores just drain when the kernel ends -- and a reader
// accepts a word only if its tag equals the sequence number it is waiting for.  Readers fold the records in rank
// order, so all ranks obtain bit-identical global values.
constexpr int kMaxPeers = 16;
constexpr int kDiagSlotsFwd = (kMaxSurfaceTypes + 1) * 10;
struct DiagMail {
    unsigned long long w[3][kDiagSlotsFwd][2];      // [sum|min|max][compact slot][lo|hi]: (seq32 << 32) | 32 bits of the double
};
__host__ __device__ inline void diag_mail_pack(double x, unsigned int seq32, unsigned long long out[2])
{
    unsigned long long b;
    memcpy(&b, &x, 8);
    out[0] = ((unsigned long long)seq32 << 32) | (b & 0xffffffffull);
    out[1] = ((unsigned long long)seq32 << 32) | (b >> 32);
}
constexpr int kMailDepth = 8;       // mailbox records per source rank: the record of exchange e lives in slot e mod kMailDepth
struct PeerPost {
    int nranks, rank;                // nranks <= 1: off
    int slot, pad;                   // seq mod kMailDepth
    unsigned long long seq;          // number of the exchange (fc_allreduce_diagnostics calls so far), the words' tag
    DiagMail *mail[kMaxPeers];       // mailbox base of every rank (the own one included), mapped into this process
};

// Rows of a specialised launch (one per CTA) that still have to be folded into that step's result vector.  The
// specialised kernel does not fold its own rows: the CTAs just leave their row and exit, and the fold runs where it
// costs nothing -- in the producer warps of the NEXT step's kernel while its ring fills (griddepcontrol.wait orders
// it after the rows) -- or in a one-warp-per-slot kernel when the host asks for the values first.  Same function,
// same order, same bits either way.
struct DiagFold {
    const double *rows;              // [plane][compact slot][row_stride]
    int64_t row_stride, plane;       // plane = nslots * row_stride
    int nrows, nslots;               // rows written per slot (= grid of that launch); nslots == 0: nothing to fold
    int level, pad;                  // 1: sums, 2: sums + min/max
    double *out;                     // [sum|min|max][kDiagSlots]
    PeerPost post;                   // nranks > 1: also post the result to every rank's mailbox
};

struct FusedPlan {
    int S;                   // num_surface_types
    int do_early;            // RBBR (+ its average) in this launch
    int do_normal;           // everything else
    int diag;                // accumulate diagnostics
    Consts c;
    FusedT t;
    FusedUV uv[2];           // [0] = u grid, [1] = v grid
    double *diag_partials;   // [plane: sum|min|max][diag_n][diag_rows]
    int64_t diag_rows;       // warp rows of one fused step (row stride of the partials)
    int diag_n;              // number of active diagnostics slots
    signed char diag_map[(kMaxSurfaceTypes + 1) * 10];   // slot -> compact index, -1 = inactive
};

// diagnostics slot layout: slot(type 0..10, quantity)
enum DiagQuantity { DQ_QSUR_T = 0, DQ_MEVA, DQ_HLAT, DQ_HSEN, DQ_RBBR, DQ_RSDR, DQ_QSUR_U, DQ_UMOM, DQ_QSUR_V, DQ_VMOM, DQ_COUNT };
constexpr int kDiagSlots = (kMaxSurfaceTypes + 1) * DQ_COUNT;
static_assert(kDiagSlots == kDiagSlotsFwd, "DiagMail layout");

constexpr int kFusedThreads = 256;
constexpr int kFusedMinBlocks = 2;                           // __launch_bounds__ occupancy target
constexpr int kFusedVec = 2;                                  // cells per thread (128-bit accesses)
constexpr int kFusedCellsPerBlock = kFusedThreads * kFusedVec;

// FULL = true : every thread owns V whole cells and every array is 16-byte aligned (128-bit accesses only);
//               launched over floor(cells/V) cell vectors per grid.
// FULL = false: guarded scalar accesses; launched over the ragged remainder (cells % V) of each grid, or over
//               everything when a bound array is not 16-byte aligned.  first[] = first cell of this launch.
struct LaunchGeom {
    int nb_t, nb_u;          // blocks of the t / u grid (the rest is the v grid)
    int64_t first[3];        // first cell handled by this launch on each grid
    int64_t count[3];        // cells handled by this launch on each grid
    int64_t row0;            // first diagnostics row of this launch
};

// parameter block of the specialised persistent kernel (spec_kernel.cu)
constexpr int kSpecMaxSlots = 16;
constexpr int kSpecMaxNS = 2;                            // surface types the specialised kernel handles
constexpr int kSpecBiasSlot = 6;                         // src[0] slot of the bias month slab (spec_kernel.cu: Lay::BIAS)
struct SpecPlan {
    Consts c;
    int64_t first[3];                 // first cell of the range on each grid
    int64_t end[3];                   // one past its last cell
    int ntiles[3];                    // ceil(cells / tile): the last tile of a grid may be partial (guarded path)
    int rot[3];                       // static schedule: CTA that takes tile 0 of each grid
    int ns;                           // number of surface types (the kernel has it as NS)
    int t_stages, u_stages;           // the two carvings of the ring
    int t_stage_bytes, u_stage_bytes;
    int t_bars, u_bars;               // lcm(teams, stages): tile i uses barrier i mod bars (one per (team, stage) pair) in phase i / bars
    int do_early;                     // RBBR in this launch
    int has_bias, has_rsdr;
    int any_avg_t;                    // some t-grid flux is area-fraction averaged (FARE is staged)
    int ase_slot;                     // bulk: slot of the sensible-heat transfer coefficient (AEV for CCLM, ASE for MOM5)
    int diag;
    double latent_heat[kSpecMaxNS];
    const double *src[3][kSpecMaxSlots];   // per grid: source array of each stage slot (null: slot unused)
    uint32_t tx_bytes[3];             // bytes one tile of that grid brings in
    const double *area[3];
    double *out[kSpecMaxNS + 1][DQ_COUNT];   // [surface type, 0 = average][quantity] (null: not produced)
    double *partials;                 // [plane][compact slot][row]; rows [0, grid) are this kernel's (one per CTA)
    int64_t rows, plane;
    DiagFold prev;                    // rows of the previous launch, folded here while the ring fills (nslots == 0: none)
    int early_loads;                  // first bulk copies before griddepcontrol.wait (previous kernel = own step)
    int dyn;                          // this launch uses the dynamic schedule
    int chain;                        // static schedule: the previous launch of the stream is the same plan -> per-CTA hand-over
    unsigned int seq;                 // number of this launch in the context's sequence of static launches
    unsigned int *done;               // [CTA]: seq of the last launch whose CTA of that index has stored everything (null: not recorded)
    int area_ahead;                   // fetch the cell areas one tile ahead (pays while the launch is latency bound: few tiles per CTA)
    unsigned int tile_base;           // dynamic schedule: value of *tile_counter before this launch's first claim
    unsigned int *tile_counter;       // dynamic schedule: tiles are claimed with atomicAdd (never reset: the host tracks the base)
    signed char dmap[(kSpecMaxNS + 1) * DQ_COUNT];   // type * DQ_COUNT + quantity -> compact diagnostics slot (-1: inactive)
};

// A fused plan resolved for one cell range (resolve_fused): which kernel serves it, its launch geometry and schedule.
// All of it follows from the plan, the range and the options "staged" and "dyn_min_tiles", so it is worked out once
// per prepared plan; a step adds only its FusedStepArgs.
struct FusedLaunch {
    bool spec;               // the specialised persistent kernel serves the whole range in one launch
    // generic kernel: the 128-bit kernel over whole 512-cell blocks, the guarded kernel over the ragged rest (or over
    // everything if an array is misaligned); a launch with no blocks is skipped
    LaunchGeom main, tail;
    int nb_main, nb_tail;
    // specialised kernel: its formula set (spec_kernel.cu: SpecSet), grid, and parameter block without the per-step fields
    int spec_set, spec_grid;
    SpecPlan sp;
    int64_t diag_rows;       // diagnostics rows the launch writes (one per warp; one per CTA of the specialised kernel)
    unsigned int claims;     // dynamic schedule: by how much a launch advances its tile counter (0: static schedule)
    bool fills;              // the specialised launch occupies every CTA slot of the device
};

// what changes from one launch of a resolved plan to the next
struct FusedStepArgs {
    const double *bias;      // month slab of the corrections (null: the plan has none)
    double *diag_partials;   // [plane][compact slot][diag_rows]
    int64_t diag_rows;       // row stride of the partials
    double *diag_out;        // [sum|min|max][kDiagSlots] result of this step
    // specialised kernel only
    DiagFold fold_prev;      // rows of the previous specialised launch of the stream, folded by this launch (nslots == 0: none)
    int early_loads;         // the previous operation of the stream is this library's own step kernel (which writes no
                             // input): the producers may start their first bulk copies before griddepcontrol.wait
    int chain;               // static schedule: the previous launch of the stream was this very plan -> its CTA b hands over to this
    unsigned int chain_seq;  //   launch's CTA b (spec_kernel.cu); number of this launch, and where the CTAs record it
    unsigned int *chain_done;
    unsigned int tile_base;  // dynamic schedule: the counter's value before this launch (it is never reset, see spec_kernel.cu)
    unsigned int *tile_counter;
};

// launchers (kernels.cu)
int launch_oplist(const OpList &ops, const Consts &c, int64_t n, cudaStream_t stream);
FusedLaunch resolve_fused(const FusedPlan &plan, const int64_t first[3], const int64_t cells[3], int staged, int dyn_min_tiles);
int launch_fused(const FusedPlan &plan, const FusedLaunch &L, const FusedStepArgs &a, cudaStream_t stream, int *launches);
int launch_diag_finalize(const FusedPlan &plan, const FusedLaunch &L, const FusedStepArgs &a, double *tmp, cudaStream_t stream, int *launches);
int launch_diag_post(const double *diag_out, const PeerPost &post, int n_active, cudaStream_t stream);
int launch_diag_fold(const DiagFold &fold, cudaStream_t stream);      // spec_kernel.cu: the stand-alone fold
int launch_diag_combine(const double *chunk_out, int nchunks, double *diag_out, cudaStream_t stream);
int diag_tmp_doubles(int64_t rows, int nslots);
unsigned long long read_exact_calls();
// specialised persistent kernel (spec_kernel.cu)
bool spec_resolve(const FusedPlan &plan, const int64_t first[3], const int64_t cells[3], int dyn_min_tiles, FusedLaunch &L);
int spec_launch(const SpecPlan &sp, int set, int grid, cudaStream_t stream);
int spec_capacity(int num_surface_types);
unsigned long long read_spec_exact_calls();
int launch_transpose_corrections(const double *corr_fortran, double *corr_month_major, int64_t n, int64_t stride, cudaStream_t stream);
inline int64_t corr_stride(int64_t n) { return (n + 1) & ~int64_t(1); }      // cells between two month slabs: even, so that each slab is 16-byte aligned
int launch_regrid_csr(const int64_t *row_ptr, const int32_t *src_idx, const double *weight, const double *src,
                      double *dst, int64_t n_dst, cudaStream_t stream);

}  // namespace fc
