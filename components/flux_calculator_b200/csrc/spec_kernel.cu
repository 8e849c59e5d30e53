// spec_kernel.cu -- the fast path of the fused coupling step: one persistent, formula-set-specialised kernel for
// the canonical configurations with one or two surface types (every configuration BASELINE.json benchmarks).
//
//   * persistent CTAs: one producer warp + TEAMS x 8 consumer warps.  One surface type: 2 CTAs per SM, one team
//     each.  Two surface types (15-16 input arrays per t tile): 1 CTA per SM with two teams that share one ring, so
//     that three 60 KB stages serve two tiles in work and one in flight;
//   * the producer streams the input arrays of 512-cell tiles into a shared-memory ring with cp.async.bulk,
//     completion counted on mbarriers.  The ring bytes are carved twice: into t stages (all arrays of a t-grid
//     tile) and into smaller u/v stages, so the light u/v tiles get about twice as many stages out of the same
//     bytes; the switch from t tiles to u/v tiles needs no drain (the first use of a u/v stage waits for the last
//     t tile of every t stage it overlaps);
//   * consumers read operands from shared memory at the point of use (LDS.128 with an immediate offset: the slot
//     of every array is a compile-time constant of the formula set), two cells per thread in lock step, results
//     leave through 128-bit global stores; nothing but the running quantities lives in registers;
//   * formula set and number of surface types are template parameters -- no method dispatch inside the kernel;
//     area-fraction averages over the surface types (average_across_surface_types) are formed in registers;
//   * diagnostics: per-thread running sums (and min/max at level 2) over all tiles of a thread, one warp tree per
//     quantity per kernel, the CTA's warps combined in shared memory into one row per CTA -- and that is all a CTA
//     does at its end: no fence, no atomic, no last-CTA reduction on the tail of the step.  The rows are folded
//     into the step's result vector (and posted to the peer GPUs' mailboxes over NVLink) by the producer warps of
//     the NEXT step's kernel while its ring fills, or by a one-warp-per-slot kernel when the host asks first
//     (DiagFold, plan.h).  Static schedule + fixed trees: reproducible sums;
//   * cells whose operands leave the range in which the lock-step division / sqrt / exp / log sequences are
//     proven (vmath.cuh) are NOT handled inline: the warp notes the tile, and a cold, out-of-line epilogue
//     recomputes those tiles with the IEEE routines from global memory and rebuilds the warp's diagnostics
//     from the stored outputs.  The hot loop carries no call, no stack frame and no spill;
//   * the ragged remainder of a grid (cells mod 512) is one more tile of the schedule, taken by its CTA before
//     the ring tiles with guarded global loads/stores -- same chain code, no second launch;
//   * launched with programmatic stream serialisation: the next step's CTAs become resident and set up their
//     barriers while this step drains; consumers wait (griddepcontrol.wait) before touching global memory, and
//     when the previous kernel of the stream is this library's own step (which writes no input array) the
//     producer fills the ring BEFORE it waits, so the fill overlaps the previous step's tail.
//
// Everything else (S > 2, 'zero'/'none' mixes, averaged QSUR, misaligned arrays, early-only phase) runs on the
// generic kernels of kernels.cu, instantiated from the same formula templates.
#include "plan.h"

#include <cuda_runtime.h>
#include <float.h>
#include <string.h>

namespace fc {

constexpr int kSpecV = 2;
// CTA geometry per number of surface types.  One type: 2 CTAs per SM, one team of 8 consumer warps, 512-cell tiles.
// Two types (15-16 input arrays per t tile): 1 CTA per SM, two teams of 8 warps sharing three 60 KB t stages (two in
// work, one in flight).  Lane 0 of the producer warp issues all bulk copies of a tile.  Measured on one B200
// (profiles/run18.sh, 3 repetitions each, C5 = 10^7 cells, two types) against four teams of 4 warps on 256-cell tiles
// (7 stages of 30 KB) and against a producer in which lane a issues the copy of slot a:
//   teams x producer          2 x one lane   2 x lane per slot   4 x one lane   4 x lane per slot
//   C5 ms / step              0.852-0.861    0.892-0.905         1.054-1.058    0.898-0.906
//   C4 ms / step (one type)   0.434-0.445    0.437               0.435-0.444    0.437
// Registers per thread, 96 for both:
//   one type: 2 CTAs x 9 warps per SM (112 would still fit the register file on paper, but measured 0.57 ms instead of
//   0.43 ms on C4: the second CTA no longer becomes resident);
//   two types: 17 warps.  One of the four SM sub-partitions (16384 registers each) holds five of them: 5 x 32 x 96 fits,
//   5 x 32 x 104 does not ("too many resources requested for launch" at 112 and 120).
template <int NS>
struct SpecGeom {
    static constexpr int kTeams = (NS == 1) ? 1 : 2;
    static constexpr int kTeamWarps = 8;                     // consumer warps of one team = one tile per pass
    static constexpr int kTeamThreads = kTeamWarps * 32;
    static constexpr int kTile = kTeamThreads * kSpecV;      // cells per tile
    static constexpr int kSlotBytes = kTile * 8;             // one array of one tile
    static constexpr int kConsumers = kTeams * kTeamThreads;
    static constexpr int kThreads = kConsumers + 32;         // + producer warp
    static constexpr int kWarps = kTeams * kTeamWarps;
    static constexpr int kCtasPerSm = (NS == 1) ? 2 : 1;
    static constexpr int kMaxRegs = 96;                      // registers per thread (see above)
};
constexpr int kSpecMaxStages = 16;
constexpr int kSpecMaxBars = 32;                         // barriers per set: lcm(teams, stages) <= 2 * 16
constexpr int kSpecBadCap = 16;                          // flagged tiles remembered per warp and phase; more -> all

using S2 = Vd<kSpecV>;

enum SpecSet { SET_BULK = 0, SET_RCO = 1 };

// Slots of the shared-memory stage: shared (atmosphere / bottom-model) arrays first, then the per-surface-type
// arrays (FICE, TSUR and, with two types, FARE), then the MOM5-only second transfer coefficient.
//   SET_BULK: CCLM / MOM5 formulae (the MOM5 routines forward to the CCLM ones, flux_mass_evap.F90:107-115)
//   SET_RCO : Meier et al. 1999 formulae; QSUR on the t grid is still the CCLM routine (App. F-1)
template <int SET, int NS>
struct Lay {
    static constexpr int kPer = (NS == 1) ? 2 : 3;       // per-type arrays: FICE, TSUR (, FARE)
    // t grid
    static constexpr int PSUR = 0, QATM = 1, TATM = 2, UATM = 3, VATM = 4, RSDD = 5, BIAS = 6;
    static constexpr int AEV = 7, PATM = 8;              // bulk only
    static constexpr int kShared = (SET == SET_BULK) ? 9 : 7;
    __host__ __device__ static constexpr int FICE(int i) { return kShared + kPer * i; }
    __host__ __device__ static constexpr int TSUR(int i) { return kShared + kPer * i + 1; }
    __host__ __device__ static constexpr int FARE(int i) { return kShared + kPer * i + 2; }
    static constexpr int ASE = kShared + kPer * NS;      // bulk/MOM5 only (CHEA != CMOI)
    static constexpr int NT = ASE + (SET == SET_BULK ? 1 : 0);
    // u / v grid
    static constexpr int U_UATM = 0, U_VATM = 1, U_PSUR = 2, U_AMOM = 3;
    static constexpr int kUShared = (SET == SET_BULK) ? 4 : 2;
    __host__ __device__ static constexpr int U_FICE(int i) { return kUShared + kPer * i; }       // bulk only
    __host__ __device__ static constexpr int U_TSUR(int i) { return kUShared + kPer * i + 1; }   // bulk only
    __host__ __device__ static constexpr int U_FARE(int i) { return (SET == SET_BULK) ? kUShared + kPer * i + 2 : kUShared + i; }
    static constexpr int NUV = (SET == SET_BULK) ? kUShared + kPer * NS : kUShared + (NS == 1 ? 0 : NS);
};
static_assert(Lay<SET_BULK, 2>::NT <= kSpecMaxSlots && Lay<SET_BULK, 1>::NT == 12 && Lay<SET_BULK, 1>::NUV == 6, "");
static_assert(Lay<SET_BULK, 1>::BIAS == kSpecBiasSlot && Lay<SET_RCO, 2>::BIAS == kSpecBiasSlot, "plan.h: kSpecBiasSlot");

template <int NS, int DIAG>
struct WarpSums {    // per-CTA staging of the consumer warps' diagnostics
    static constexpr int kWarps = SpecGeom<NS>::kWarps;
    static constexpr int kSlots = (NS == 1 ? 1 : NS + 1) * DQ_COUNT;
    double v[DIAG >= 2 ? 3 : 1][kSlots][kWarps];
};
// staging index of (surface type, quantity): with one type only that type's quantities exist
template <int NS>
__device__ __forceinline__ constexpr int ws_index(int type, int q) { return NS == 1 ? q : type * DQ_COUNT + q; }

// ---------------------------------------------------------------------------------------------
// mbarrier / bulk-copy primitives (PTX ISA: mbarrier, cp.async.bulk)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.release.cta.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    asm volatile("{\n\t.reg .pred P_OUT;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 P_OUT, [%1], %2;\n\t"
                 "selp.b32 %0, 1, 0, P_OUT;\n\t}"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------------------------------------
// operand sources, result sinks, diagnostics accumulators
// ---------------------------------------------------------------------------------------------
// hot path: this thread's 16 bytes of each slot of the current stage
template <int SLOT_BYTES>
struct LdStage {
    const char *base;
    __device__ __forceinline__ S2 operator()(int slot) const
    {
        const double2 t = *reinterpret_cast<const double2 *>(base + slot * SLOT_BYTES);
        S2 r;
        r.v[0] = t.x;
        r.v[1] = t.y;
        return r;
    }
};
struct StPair {
    int64_t j;
    __device__ __forceinline__ void operator()(double *p, const S2 &x) const
    {
        *reinterpret_cast<double2 *>(p + j) = make_double2(x.v[0], x.v[1]);
    }
};
// partial tile: guarded global accesses, nv = 0, 1 or 2 valid cells
struct LdPairGuard {
    const double *const *src;
    int64_t j;
    int nv;
    __device__ __forceinline__ S2 operator()(int slot) const
    {
        S2 r;
#pragma unroll
        for (int k = 0; k < kSpecV; ++k) r.v[k] = (k < nv) ? __ldg(src[slot] + j + k) : 1.0;
        return r;
    }
};
struct StPairGuard {
    int64_t j;
    int nv;
    __device__ __forceinline__ void operator()(double *p, const S2 &x) const
    {
#pragma unroll
        for (int k = 0; k < kSpecV; ++k)
            if (k < nv) p[j + k] = x.v[k];
    }
};
// cold path: one cell from global memory
struct LdCell {
    const double *const *src;
    int64_t j;
    __device__ __forceinline__ Vd<1> operator()(int slot) const
    {
        Vd<1> r;
        r.v[0] = src[slot][j];
        return r;
    }
};
struct StCell {
    int64_t j;
    __device__ __forceinline__ void operator()(double *p, const Vd<1> &x) const { p[j] = x.v[0]; }
};
struct NoDiag {
    template <class T>
    __device__ __forceinline__ void operator()(int, int, const T &) const {}
};

// acc = acc + (area0*x0 + area1*x1): the one definition both the hot loop and the rebuild of the cold epilogue use
__device__ __forceinline__ void diag_pair(double &s, double &mn, double &mx, int level, double a0, double a1, double x0, double x1)
{
    s = add(s, add(mul(a0, x0), mul(a1, x1)));
    if (level >= 2) {
        mn = fmin(fmin(mn, x0), x1);
        mx = fmax(fmax(mx, x0), x1);
    }
}
// nv valid cells (partial tile); identical to diag_pair for nv == 2
__device__ __forceinline__ void diag_cells(double &s, double &mn, double &mx, int level, double a0, double a1, double x0, double x1, int nv)
{
    if (nv >= 2) {
        diag_pair(s, mn, mx, level, a0, a1, x0, x1);
    } else if (nv == 1) {
        s = add(s, mul(a0, x0));
        if (level >= 2) {
            mn = fmin(mn, x0);
            mx = fmax(mx, x0);
        }
    }
}

// warp tree of one quantity; lane 0 leaves the warp's value in the CTA's staging area
template <int NS, int DIAG>
__device__ __forceinline__ void diag_flush_one(WarpSums<NS, DIAG> &ws, int wsi, double s, double mn, double mx)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s = add(s, __shfl_down_sync(0xffffffffu, s, off));
        if (DIAG >= 2) {
            mn = fmin(mn, __shfl_down_sync(0xffffffffu, mn, off));
            mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, off));
        }
    }
    if ((threadIdx.x & 31) == 0) {
        const int w = threadIdx.x >> 5;
        ws.v[0][wsi][w] = s;
        if constexpr (DIAG >= 2) {
            ws.v[1][wsi][w] = mn;
            ws.v[2][wsi][w] = mx;
        }
    }
}

// Running diagnostics of one phase: NQ quantities (Q0 ..) of every surface type (and of the averages with two types).
//   REG = true  (one surface type): per-THREAD running values in registers over all tiles of the thread, one warp
//                tree per quantity at the end of the phase;
//   REG = false (two surface types: 17 sums, or 51 values with min/max, do not fit the register file next to the
//                chain): one warp tree per quantity per TILE, lane 0 accumulates the warp's value in shared memory.
// Both are deterministic (static tile schedule, fixed trees).
constexpr int kDiagAccMax = (kSpecMaxNS + 1) * 6;      // accumulators of the t phase with two types
template <int NS, int DIAG, int NQ, int Q0, bool REG = (NS == 1)>
struct DiagAcc;

template <int NS, int DIAG, int NQ, int Q0>
struct DiagAcc<NS, DIAG, NQ, Q0, true> {
    static constexpr int kN = NQ;
    double s[kN], mn[DIAG >= 2 ? kN : 1], mx[DIAG >= 2 ? kN : 1];
    S2 area;
    static __device__ __forceinline__ constexpr int idx(int, int q) { return q - Q0; }
    __device__ __forceinline__ void init(double *) {}
    __device__ __forceinline__ void reset()
    {
#pragma unroll
        for (int k = 0; k < kN; ++k) {
            s[k] = 0.0;
            if (DIAG >= 2) {
                mn[k] = DBL_MAX;
                mx[k] = -DBL_MAX;
            }
        }
    }
    __device__ __forceinline__ void add_cells(int type, int q, const S2 &x, int nv)      // nv valid cells (2 except in the partial tile)
    {
        if (DIAG == 0) return;
        const int k = idx(type, q);
        if constexpr (DIAG >= 2) {
            diag_cells(s[k], mn[k], mx[k], DIAG, area.v[0], area.v[1], x.v[0], x.v[1], nv);
        } else {
            double dm = 0.0, dM = 0.0;
            diag_cells(s[k], dm, dM, DIAG, area.v[0], area.v[1], x.v[0], x.v[1], nv);
        }
    }
    __device__ __forceinline__ void operator()(int type, int q, const S2 &x) { add_cells(type, q, x, kSpecV); }
    // end of the phase: q0 = first quantity of the phase in the staging area (DQ_QSUR_T / _U / _V)
    __device__ __forceinline__ void flush(WarpSums<NS, DIAG> &ws, int q0)
    {
#pragma unroll
        for (int q = 0; q < NQ; ++q)
            diag_flush_one<NS, DIAG>(ws, ws_index<NS>(1, q0 + q), s[q], DIAG >= 2 ? mn[DIAG >= 2 ? q : 0] : 0.0, DIAG >= 2 ? mx[DIAG >= 2 ? q : 0] : 0.0);
    }
};

template <int NS, int DIAG, int NQ, int Q0>
struct DiagAcc<NS, DIAG, NQ, Q0, false> {
    static constexpr int kN = (NS + 1) * NQ;
    static_assert(kN <= kDiagAccMax && kN <= 32, "one lane per accumulator at reset / flush");
    double *acc;      // this warp's [plane][kDiagAccMax] in shared memory
    S2 area;
    static __device__ __forceinline__ constexpr int idx(int type, int q) { return type * NQ + (q - Q0); }
    __device__ __forceinline__ void init(double *warp_rows) { acc = warp_rows; }
    __device__ __forceinline__ void reset()
    {
        if (DIAG == 0) return;
        const int lane = threadIdx.x & 31;
        if (lane < kN) {
            acc[lane] = 0.0;
            if (DIAG >= 2) {
                acc[kDiagAccMax + lane] = DBL_MAX;
                acc[2 * kDiagAccMax + lane] = -DBL_MAX;
            }
        }
        __syncwarp();
    }
    __device__ __forceinline__ void add_cells(int type, int q, const S2 &x, int nv)
    {
        if (DIAG == 0) return;
        const int k = idx(type, q);
        double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
        diag_cells(s, mn, mx, DIAG, area.v[0], area.v[1], x.v[0], x.v[1], nv);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s = add(s, __shfl_down_sync(0xffffffffu, s, off));
            if (DIAG >= 2) {
                mn = fmin(mn, __shfl_down_sync(0xffffffffu, mn, off));
                mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, off));
            }
        }
        if ((threadIdx.x & 31) == 0) {
            acc[k] = add(acc[k], s);
            if (DIAG >= 2) {
                acc[kDiagAccMax + k] = fmin(acc[kDiagAccMax + k], mn);
                acc[2 * kDiagAccMax + k] = fmax(acc[2 * kDiagAccMax + k], mx);
            }
        }
    }
    __device__ __forceinline__ void operator()(int type, int q, const S2 &x) { add_cells(type, q, x, kSpecV); }
    __device__ __forceinline__ void flush(WarpSums<NS, DIAG> &ws, int q0)
    {
        __syncwarp();
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (lane < kN) {
            const int wsi = ws_index<NS>(lane / NQ, q0 + lane % NQ);
            ws.v[0][wsi][w] = acc[lane];
            if constexpr (DIAG >= 2) {
                ws.v[1][wsi][w] = acc[kDiagAccMax + lane];
                ws.v[2][wsi][w] = acc[2 * kDiagAccMax + lane];
            }
        }
        __syncwarp();
    }
};

template <int NS, int DIAG, int NQ, int Q0>
struct DiagAccGuard {    // the same accumulators fed from a partial tile
    DiagAcc<NS, DIAG, NQ, Q0> &a;
    int nv;
    __device__ __forceinline__ void operator()(int type, int q, const S2 &x) { a.add_cells(type, q, x, nv); }
};

template <int NS>
__device__ __forceinline__ void consumer_barrier()
{
    asm volatile("bar.sync 1, %0;" ::"n"(SpecGeom<NS>::kConsumers) : "memory");
}

// one warp folds the rows of compact slot cs into the result vector (and the step's history row): lane-strided rows, then
// a tree -- a fixed order, the same in the next step's kernel and in the stand-alone fold kernel -- and posts the result
// to the peers' mailboxes
__device__ __forceinline__ void diag_fold_slot(const DiagFold &f, int cs)
{
    const int lane = threadIdx.x & 31;
    const double *col = f.rows + (int64_t)cs * f.row_stride;
    const bool mm = f.level >= 2;
    double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
    constexpr int kPer = 10;      // rows per lane fetched at once (2 CTAs x 148 SMs = 296 rows -> one round)
    for (int r0 = 0; r0 < f.nrows; r0 += 32 * kPer) {
        double vs[kPer], vn[kPer], vx[kPer];
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int r = r0 + k * 32 + lane;
            vs[k] = (r < f.nrows) ? __ldcg(col + r) : 0.0;
            vn[k] = (mm && r < f.nrows) ? __ldcg(col + f.plane + r) : DBL_MAX;
            vx[k] = (mm && r < f.nrows) ? __ldcg(col + 2 * f.plane + r) : -DBL_MAX;
        }
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            s = add(s, vs[k]);
            mn = fmin(mn, vn[k]);
            mx = fmax(mx, vx[k]);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s = add(s, __shfl_down_sync(0xffffffffu, s, off));
        mn = fmin(mn, __shfl_down_sync(0xffffffffu, mn, off));
        mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, off));
    }
    s = __shfl_sync(0xffffffffu, s, 0);
    mn = __shfl_sync(0xffffffffu, mn, 0);
    mx = __shfl_sync(0xffffffffu, mx, 0);
    if (lane == 0 && f.out) {
        f.out[0 * kDiagSlots + cs] = s;
        f.out[1 * kDiagSlots + cs] = mn;
        f.out[2 * kDiagSlots + cs] = mx;
    }
    if (lane == 0 && f.hist.ring) {
        double *h = diag_hist_row(f.hist);
        h[0 * kDiagSlots + cs] = s;
        h[1 * kDiagSlots + cs] = mn;
        h[2 * kDiagSlots + cs] = mx;
    }
    // compute -> exchange without a collective launch: the result goes straight into every rank's mailbox over NVLink
    // as self-validating 8-byte words (no fence, no flag store: see DiagMail); one lane per (rank, plane)
    if (f.post.nranks > 1) {
        for (int e = lane; e < f.post.nranks * 3; e += 32) {
            const int r = e / 3, pl = e - 3 * r;
            unsigned long long w[2];
            diag_mail_pack(pl == 0 ? s : (pl == 1 ? mn : mx), (unsigned int)f.post.seq, w);
            DiagMail *m = f.post.mail[r] + (size_t)f.post.slot * f.post.nranks + f.post.rank;
            __stcg(&m->w[pl][cs][0], w[0]);
            __stcg(&m->w[pl][cs][1], w[1]);
        }
    }
}

__global__ void __launch_bounds__(32) diag_fold_kernel(const __grid_constant__ DiagFold f) { diag_fold_slot(f, (int)blockIdx.x); }

int launch_diag_fold(const DiagFold &f, cudaStream_t stream)
{
    if (f.nslots <= 0) return 0;
    diag_fold_kernel<<<f.nslots, 32, 0, stream>>>(f);
    return (int)cudaGetLastError();
}

// end of kernel, consumer warps only: warps -> one row per CTA.  Nothing else: the rows are folded after this grid
// completed (DiagFold), so neither a fence nor a counter is needed here.
template <int NS, int DIAG>
__device__ __forceinline__ void diag_finish(const SpecPlan &p, WarpSums<NS, DIAG> &ws)
{
    constexpr int kWarps = WarpSums<NS, DIAG>::kWarps;
    constexpr int kSlots = WarpSums<NS, DIAG>::kSlots;
    const int tid = threadIdx.x;
    consumer_barrier<NS>();
    if (tid < kSlots) {
        const int cs = p.dmap[NS == 1 ? DQ_COUNT + tid : tid];      // one type: staging holds surface type 1
        if (cs >= 0) {
            double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) {
                s = add(s, ws.v[0][tid][w]);
                if constexpr (DIAG >= 2) {
                    mn = fmin(mn, ws.v[1][tid][w]);
                    mx = fmax(mx, ws.v[2][tid][w]);
                }
            }
            double *o = p.partials + (int64_t)cs * p.rows + blockIdx.x;
            o[0] = s;
            if (DIAG >= 2) {
                o[p.plane] = mn;
                o[2 * p.plane] = mx;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// the chains, written once over (arithmetic policy, operand source, result sink, diagnostics sink)
// ---------------------------------------------------------------------------------------------
// acc = acc + x*fare, separate multiply and add (average_across_surface_types, calculate.F90:379-382)
template <class M>
__device__ __forceinline__ void avg_add(typename M::T &acc, const typename M::T &x, const typename M::T &fare)
{
    acc = M::add(acc, M::mul(x, fare));
}

// t grid, per surface type: QSUR -> MEVA (+bias) -> HLAT, HSEN, RBBR, RSDR; then the type-0 averages.
// Call-site wiring of calculate.F90 (App. A.2): the evaporation routine gets TATM in its temperature slot (:87), the
// sensible-heat routine gets QATM in its q_s slot (:178).
template <int SET, int NS, class M, class LD, class ST, class DG>
__device__ __forceinline__ void spec_t_chain(M &m, const SpecPlan &p, const LD &ld, const ST &st, DG &dg)
{
    using T = typename M::T;
    using L = Lay<SET, NS>;
    const Consts &c = p.c;
    const T vel = wind_speed(m, ld(L::UATM), ld(L::VATM));
    T aM = M::bc(0.0), aL = M::bc(0.0), aH = M::bc(0.0), aR = M::bc(0.0), aS = M::bc(0.0);
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        const int ty = i + 1;
        // calc_spec_vapor_surface (calculate.F90:25-50)
        const T qsur = spec_vapor_surface_cclm(m, ld(L::FICE(i)), ld(L::PSUR), ld(L::TSUR(i)), c);
        st(p.out[ty][DQ_QSUR_T], qsur);
        dg(ty, DQ_QSUR_T, qsur);
        // calc_flux_mass_evap (calculate.F90:54-120) + bias (:112-116)
        T meva;
        if (SET == SET_BULK) meva = flux_mass_evap_cclm(m, ld(L::AEV), ld(L::PSUR), ld(L::QATM), qsur, ld(L::TATM), vel, c);
        else meva = flux_mass_evap_rco(m, ld(L::QATM), ld(L::TSUR(i)), vel);
        if (p.has_bias) meva = M::add(meva, ld(L::BIAS));
        st(p.out[ty][DQ_MEVA], meva);
        dg(ty, DQ_MEVA, meva);
        // calc_flux_heat_latent (calculate.F90:124-154): the corrected MEVA
        const T hlat = M::mul(meva, M::bc(p.latent_heat[i]));
        st(p.out[ty][DQ_HLAT], hlat);
        dg(ty, DQ_HLAT, hlat);
        // calc_flux_heat_sensible (calculate.F90:156-208)
        T hsen;
        if (SET == SET_BULK)
            hsen = flux_heat_sensible_cclm(m, ld(p.ase_slot), ld(L::PATM), ld(L::PSUR), ld(L::QATM), ld(L::TATM), ld(L::TSUR(i)), vel, c);
        else
            hsen = flux_heat_sensible_rco<M>(ld(L::TATM), ld(L::TSUR(i)), vel);
        st(p.out[ty][DQ_HSEN], hsen);
        dg(ty, DQ_HSEN, hsen);
        T fare;
        if (NS > 1 && p.any_avg_t) {
            fare = ld(L::FARE(i));
            if (p.out[0][DQ_MEVA]) avg_add<M>(aM, meva, fare);
            if (p.out[0][DQ_HLAT]) avg_add<M>(aL, hlat, fare);
            if (p.out[0][DQ_HSEN]) avg_add<M>(aH, hsen, fare);
        }
        // calc_flux_radiation_blackbody (calculate.F90:320-345), early phase
        if (p.do_early) {
            const T rbbr = flux_radiation_blackbody_StBo<M>(ld(L::TSUR(i)), c.stefan_boltzmann_constant);
            st(p.out[ty][DQ_RBBR], rbbr);
            dg(ty, DQ_RBBR, rbbr);
            if (NS > 1 && p.out[0][DQ_RBBR]) avg_add<M>(aR, rbbr, fare);
        }
        // distribute_shortwave_radiation_flux (calculate.F90:347-364): a copy
        if (p.has_rsdr) {
            const T rsdr = ld(L::RSDD);
            st(p.out[ty][DQ_RSDR], rsdr);
            dg(ty, DQ_RSDR, rsdr);
            if (NS > 1 && p.out[0][DQ_RSDR]) avg_add<M>(aS, rsdr, fare);
        }
    }
    if (NS > 1) {      // average_across_surface_types (calculate.F90:368-385) of the sent fluxes
        if (p.out[0][DQ_MEVA]) { st(p.out[0][DQ_MEVA], aM); dg(0, DQ_MEVA, aM); }
        if (p.out[0][DQ_HLAT]) { st(p.out[0][DQ_HLAT], aL); dg(0, DQ_HLAT, aL); }
        if (p.out[0][DQ_HSEN]) { st(p.out[0][DQ_HSEN], aH); dg(0, DQ_HSEN, aH); }
        if (p.do_early && p.out[0][DQ_RBBR]) { st(p.out[0][DQ_RBBR], aR); dg(0, DQ_RBBR, aR); }
        if (p.has_rsdr && p.out[0][DQ_RSDR]) { st(p.out[0][DQ_RSDR], aS); dg(0, DQ_RSDR, aS); }
    }
}

// u / v grid: QSUR on that grid (bulk sets) -> momentum flux, east component on the u grid, north on the v grid
template <int SET, int NS, class M, class LD, class ST, class DG>
__device__ __forceinline__ void spec_uv_chain(M &m, const SpecPlan &p, int north, const LD &ld, const ST &st, DG &dg)
{
    using T = typename M::T;
    using L = Lay<SET, NS>;
    const Consts &c = p.c;
    const int qQ = north ? DQ_QSUR_V : DQ_QSUR_U, qM = north ? DQ_VMOM : DQ_UMOM;
    const T vel = wind_speed(m, ld(L::U_UATM), ld(L::U_VATM));
    const T wind = ld(north ? L::U_VATM : L::U_UATM);
    T aM = M::bc(0.0);
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        const int ty = i + 1;
        T mom;
        if (SET == SET_BULK) {
            const T qsur = spec_vapor_surface_cclm(m, ld(L::U_FICE(i)), ld(L::U_PSUR), ld(L::U_TSUR(i)), c);
            st(p.out[ty][qQ], qsur);
            dg(ty, DQ_QSUR_U, qsur);      // phase-local index: the u/v accumulators start at DQ_QSUR_U for both grids
            const T fa = momentum_flux_air_cclm(m, ld(L::U_AMOM), ld(L::U_PSUR), qsur, ld(L::U_TSUR(i)), vel, c);
            mom = momentum_component<M>(fa, wind);
        } else {
            mom = momentum_component<M>(momentum_flux_air_rco<M>(vel), wind);
        }
        st(p.out[ty][qM], mom);
        dg(ty, DQ_UMOM, mom);
        if (NS > 1 && p.out[0][qM]) avg_add<M>(aM, mom, ld(L::U_FARE(i)));
    }
    if (NS > 1 && p.out[0][qM]) {
        st(p.out[0][qM], aM);
        dg(0, DQ_UMOM, aM);
    }
}

// ---------------------------------------------------------------------------------------------
// cold epilogue of one phase of one warp: recompute the flagged tiles with the IEEE routines (scalar, from global
// memory), then rebuild this warp's diagnostics of the phase from the stored outputs in the hot loop's order:
// the partial tile (jpart >= 0) first, then the ring tiles j0, j0 + jstride, ...
// flagged[]: ring-tile numbers, -1 = the partial tile.
// ---------------------------------------------------------------------------------------------
__device__ unsigned long long g_spec_exact_calls = 0ull;

unsigned long long read_spec_exact_calls()
{
    unsigned long long v = 0;
    cudaMemcpyFromSymbol(&v, g_spec_exact_calls, sizeof v);
    return v;
}

template <int SET, int NS>
__device__ __forceinline__ void spec_fix_pair(const SpecPlan &p, int ph, int64_t j)
{
    atomicAdd(&g_spec_exact_calls, 1ull);
    for (int k = 0; k < kSpecV; ++k) {
        if (j + k >= p.end[ph]) break;      // partial tile
        ExactVec<1> m;
        const LdCell ld{p.src[ph], j + k};
        const StCell st{j + k};
        NoDiag nd;
        if (ph == 0) spec_t_chain<SET, NS>(m, p, ld, st, nd);
        else spec_uv_chain<SET, NS>(m, p, ph - 1, ld, st, nd);
    }
}

template <int SET, int NS, int DIAG>
__device__ __noinline__ void spec_cold_phase(const SpecPlan &p, int ph, int64_t jpart, int64_t j0, int64_t jstride, int ntiles,
                                             const int *flagged, int nflag, WarpSums<NS, DIAG> &ws)
{
    const bool all = nflag > kSpecBadCap;
    for (int i = -1; i < ntiles; ++i) {
        if (i < 0 && jpart < 0) continue;
        bool f = all;
        for (int e = 0; e < nflag && e < kSpecBadCap; ++e) f = f || (flagged[e] == i);
        if (f) spec_fix_pair<SET, NS>(p, ph, i < 0 ? jpart : j0 + (int64_t)i * jstride);
    }
    if (DIAG == 0) return;
    const int q0 = (ph == 0) ? DQ_QSUR_T : (ph == 1 ? DQ_QSUR_U : DQ_QSUR_V);
    const int nq = (ph == 0) ? 6 : 2;
    for (int ty = (NS == 1 ? 1 : 0); ty <= NS; ++ty)
        for (int q = q0; q < q0 + nq; ++q) {
            const double *x = p.out[ty][q];
            if (p.dmap[ty * DQ_COUNT + q] < 0 || x == nullptr) continue;      // uniform
            double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
            for (int i = -1; i < ntiles; ++i) {
                if (i < 0 && jpart < 0) continue;
                const int64_t j = i < 0 ? jpart : j0 + (int64_t)i * jstride;
                const int64_t left = p.end[ph] - j;
                const int nv = left >= 2 ? 2 : (left > 0 ? (int)left : 0);
                if (nv == 2) diag_pair(s, mn, mx, DIAG, p.area[ph][j], p.area[ph][j + 1], x[j], x[j + 1]);
                else if (nv == 1) diag_cells(s, mn, mx, DIAG, p.area[ph][j], 0.0, x[j], 0.0, 1);
            }
            diag_flush_one<NS, DIAG>(ws, ws_index<NS>(ty, q), s, mn, mx);
        }
}


// ---------------------------------------------------------------------------------------------
// dynamic tile schedule (the instantiations without diagnostics)
// ---------------------------------------------------------------------------------------------
// With the static round-robin schedule every CTA owns the same number of tiles, but the SMs do not stream at the
// same speed (ncu: sm__cycles_active min / avg / max = 0.68 / 0.84 / 1.0 of the kernel for the RCO set, 0.84 / 0.92 / 1.0
// for CCLM without diagnostics): the step ends when the slowest SM ends, with DRAM far from saturated on the tail.
// Without diagnostics nothing depends on WHICH CTA computes a tile, so the producers claim tiles one by one from a global
// counter (atomicAdd; claims are monotonic per CTA, hence every CTA still sees t tiles first, then u, then v and the
// two ring carvings need no change) and hand the tile number to the consumers through shared memory, published by
// the same mbarrier phase that publishes the tile's bytes.  A phase ends with one sentinel per team.  Partial tiles
// are claimed like all others and read straight from global memory.  The counter is never reset: every producer
// makes exactly two failing claims (two are kept in flight), so a launch advances it by (units + 2 CTAs) and the host
// keeps the base.  Small grids (few tiles per CTA: nothing to balance, and the claims' latency shows) and launches
// with diagnostics (the per-thread running sums need a reproducible tile -> thread map) use the static schedule.
constexpr int kDynPartial = 1 << 30;      // tile id flag: partial tile, nothing in the stage
constexpr unsigned kDynUvBatch = 4;       // u/v tiles per claim

template <int SET, int NS>
__device__ __noinline__ void spec_cold_dyn(const SpecPlan &p, int uv, const int *ids, int n, int ttid)
{
    using GEO = SpecGeom<NS>;
    for (int e = 0; e < n; ++e) {
        const int id = ids[e] & ~kDynPartial;
        const int ph = uv ? 1 + (id & 1) : 0;
        const int64_t tile = uv ? (id >> 1) : id;
        spec_fix_pair<SET, NS>(p, ph, p.first[ph] + tile * GEO::kTile + ttid * kSpecV);
    }
}

template <int SET, int NS>
__device__ __forceinline__ void spec_dynamic_body(const SpecPlan &p, char *ring, uint64_t *fullT, uint64_t *emptyT, uint64_t *fullU,
                                                  uint64_t *emptyU, int *tileT, int *tileU, int (*flagged)[kSpecBadCap], int *nflagged)
{
    using GEO = SpecGeom<NS>;
    using L = Lay<SET, NS>;
    constexpr int TEAMS = GEO::kTeams;
    const int NT = p.t_stages, NUS = p.u_stages, LT = p.t_bars, LU = p.u_bars;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned nt0 = (unsigned)p.ntiles[0], nt1 = (unsigned)p.ntiles[1], nt2 = (unsigned)p.ntiles[2];
    const bool partial[3] = {(p.end[0] - p.first[0]) % GEO::kTile != 0, (p.end[1] - p.first[1]) % GEO::kTile != 0,
                             (p.end[2] - p.first[2]) % GEO::kTile != 0};

    if (warp == GEO::kWarps) {
        // ---------------- producer: one lane claims, publishes and fetches ----------------
        if (lane != 0) return;
        // work units: unit u < nt0 is t tile u; unit nt0 + q is the kDynUvBatch consecutive tiles 4q .. 4q+3 of the list
        // [u tiles | v tiles] (they are light: a claim per tile would cost more than the tile).  Two claims are kept in
        // flight so that the atomic's round trip overlaps the issue of the previous unit's copies.
        const unsigned nuv = nt1 + nt2, units = nt0 + (nuv + kDynUvBatch - 1) / kDynUvBatch;
        unsigned g = atomicAdd(p.tile_counter, 1u) - p.tile_base;
        unsigned g_ahead = atomicAdd(p.tile_counter, 1u) - p.tile_base;
        auto claim = [&]() {      // unconditional: every producer ends with exactly two failing claims, whatever it got before
            g = g_ahead;
            g_ahead = atomicAdd(p.tile_counter, 1u) - p.tile_base;
        };
        int i = 0;
        {   // t tiles: local tile i -> stage i mod NT, barrier i mod LT
            int st = 0, bi = 0, pb = 0, puse = 0;
            auto slot = [&]() {      // wait until local tile i - NT (and with it every earlier one) is released, i.e. stage and id slot are free
                if (i >= NT) {
                    mbar_wait(&emptyT[pb], puse & 1);
                    if (++pb == LT) {
                        pb = 0;
                        ++puse;
                    }
                }
            };
            auto next = [&]() {
                if (++st == NT) st = 0;
                if (++bi == LT) bi = 0;
                ++i;
            };
            while (g < nt0) {
                slot();
                const bool part = partial[0] && g == nt0 - 1;
                tileT[bi] = part ? (int)(g | kDynPartial) : (int)g;
                if (part) {
                    mbar_arrive(&fullT[bi]);
                } else {
                    const int64_t cell = p.first[0] + (int64_t)g * GEO::kTile;
                    mbar_expect_tx(&fullT[bi], p.tx_bytes[0]);
                    char *dst = ring + (size_t)st * p.t_stage_bytes;
#pragma unroll 1
                    for (int a = 0; a < L::NT; ++a)
                        if (p.src[0][a]) bulk_g2s(dst + a * GEO::kSlotBytes, p.src[0][a] + cell, GEO::kSlotBytes, &fullT[bi]);
                }
                next();
                claim();
            }
            const int ring0 = i;      // t tiles this CTA took
            for (int t = 0; t < TEAMS; ++t) {      // end of the t phase, once per team
                slot();
                tileT[bi] = -1;
                mbar_arrive(&fullT[bi]);
                next();
            }
            i = ring0;
        }
        {   // u and v tiles: local tile k -> stage k mod NUS of the u/v carving, barrier k mod LU
            const int ring0 = i;
            int st = 0, bi = 0, pb = 0, puse = 0, k = 0;
            auto slot = [&]() {
                if (k >= NUS) {
                    mbar_wait(&emptyU[pb], puse & 1);
                    if (++pb == LU) {
                        pb = 0;
                        ++puse;
                    }
                } else {      // first use of these bytes as a u/v stage: the last t tile of every t stage they overlap must be done
                    const int lo = (st * p.u_stage_bytes) / p.t_stage_bytes, hi = ((st + 1) * p.u_stage_bytes - 1) / p.t_stage_bytes;
                    for (int s = lo; s <= hi && s < NT; ++s)
                        if (ring0 > s) {
                            const int last = s + ((ring0 - 1 - s) / NT) * NT;
                            mbar_wait(&emptyT[last % LT], (last / LT) & 1);
                        }
                }
            };
            auto next = [&]() {
                if (++st == NUS) st = 0;
                if (++bi == LU) bi = 0;
                ++k;
            };
            while (g < units) {
                const unsigned w0 = (g - nt0) * kDynUvBatch, w1 = (w0 + kDynUvBatch < nuv) ? w0 + kDynUvBatch : nuv;
                for (unsigned w = w0; w < w1; ++w) {
                    const int ph = w < nt1 ? 1 : 2;
                    const unsigned tile = ph == 1 ? w : w - nt1;
                    slot();
                    const bool part = partial[ph] && tile == (ph == 1 ? nt1 : nt2) - 1;
                    tileU[bi] = (int)((tile << 1) | (unsigned)(ph - 1)) | (part ? kDynPartial : 0);
                    if (part) {
                        mbar_arrive(&fullU[bi]);
                    } else {
                        const int64_t cell = p.first[ph] + (int64_t)tile * GEO::kTile;
                        mbar_expect_tx(&fullU[bi], p.tx_bytes[ph]);
                        char *dst = ring + (size_t)st * p.u_stage_bytes;
#pragma unroll 1
                        for (int a = 0; a < L::NUV; ++a)
                            if (p.src[ph][a]) bulk_g2s(dst + a * GEO::kSlotBytes, p.src[ph][a] + cell, GEO::kSlotBytes, &fullU[bi]);
                    }
                    next();
                }
                claim();
            }
            for (int t = 0; t < TEAMS; ++t) {      // end of the step, once per team
                slot();
                tileU[bi] = -1;
                mbar_arrive(&fullU[bi]);
                next();
            }
        }
        return;
    }

    // ---------------- consumers: team t takes local tiles t, t + TEAMS, ... of each phase ----------------
    const int team = (TEAMS == 1) ? 0 : warp / GEO::kTeamWarps;
    const int ttid = threadIdx.x - team * GEO::kTeamThreads;
    const int toff = ttid * (kSpecV * 8);
    NoDiag nd;
    auto note = [&](int id, int uv) {      // a cell left the proven range: remember the tile; a full list is worked off at once
        if (lane == 0) {
            const int n = nflagged[warp];
            flagged[warp][n] = id;
            nflagged[warp] = n + 1;
        }
        __syncwarp();
        if (nflagged[warp] == kSpecBadCap) {
            spec_cold_dyn<SET, NS>(p, uv, flagged[warp], kSpecBadCap, ttid);
            __syncwarp();
            if (lane == 0) nflagged[warp] = 0;
            __syncwarp();
        }
    };
#pragma unroll 1
    for (int uv = 0; uv < 2; ++uv) {
        uint64_t *full = uv ? fullU : fullT, *empty = uv ? emptyU : emptyT;
        const int *ids = uv ? tileU : tileT;
        const int NS_ = uv ? NUS : NT, LB = uv ? LU : LT, sbytes = uv ? p.u_stage_bytes : p.t_stage_bytes;
        int s = team % NS_, bi = team % LB, use = team / LB;
        for (;;) {
            mbar_wait(&full[bi], use & 1);
            const int id = ids[bi];
            if (id < 0) break;
            const int tid_ = id & ~kDynPartial;
            const int north = uv ? (tid_ & 1) : 0, ph = uv ? 1 + north : 0;
            const int64_t j = p.first[ph] + (int64_t)(uv ? (tid_ >> 1) : tid_) * GEO::kTile + ttid * kSpecV;
            FastVec<kSpecV> m;
            bool bad;
            if (!(id & kDynPartial)) {
                const StPair st{j};
                if (uv) {
                    const LdStage<GEO::kSlotBytes> ld{ring + (size_t)s * sbytes + toff};
                    spec_uv_chain<SET, NS>(m, p, north, ld, st, nd);
                } else {
                    const LdStage<GEO::kSlotBytes> ld{ring + (size_t)s * sbytes + toff};
                    spec_t_chain<SET, NS>(m, p, ld, st, nd);
                }
                bad = m.bad();
            } else {
                const int64_t left = p.end[ph] - j;
                const int nv = left >= 2 ? 2 : (left > 0 ? (int)left : 0);
                const LdPairGuard ld{p.src[ph], j, nv};
                const StPairGuard st{j, nv};
                if (uv) spec_uv_chain<SET, NS>(m, p, north, ld, st, nd);
                else spec_t_chain<SET, NS>(m, p, ld, st, nd);
                bad = nv > 0 && m.bad();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[bi]);
            if (__any_sync(0xffffffffu, bad)) note(id, uv);
            s += TEAMS;
            while (s >= NS_) s -= NS_;
            bi += TEAMS;
            while (bi >= LB) {
                bi -= LB;
                ++use;
            }
        }
        __syncwarp();
        const int nf = nflagged[warp];
        if (nf) {
            spec_cold_dyn<SET, NS>(p, uv, flagged[warp], nf, ttid);
            __syncwarp();
            if (lane == 0) nflagged[warp] = 0;
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
template <int SET, int NS, int DIAG, bool DYN>
__global__ void __launch_bounds__(SpecGeom<NS>::kThreads) __maxnreg__(SpecGeom<NS>::kMaxRegs) flux_spec_kernel(const __grid_constant__ SpecPlan p)
{
    using GEO = SpecGeom<NS>;
    constexpr int TEAMS = GEO::kTeams;
    extern __shared__ __align__(128) char ring[];
    // Tile i of a phase lives in stage i mod NT and is consumed by team i mod TEAMS.  With two teams alternating on a
    // stage each team would skip every other phase of a per-stage barrier, which mbarrier parity cannot tell apart; so
    // there is one barrier per (team, stage) pair: index i mod LT (LT = lcm(TEAMS, NT)), phase i / LT.
    __shared__ uint64_t fullT[kSpecMaxBars], emptyT[kSpecMaxBars], fullU[kSpecMaxBars], emptyU[kSpecMaxBars];
    __shared__ int flagged[GEO::kWarps][kSpecBadCap];
    __shared__ int nflagged[GEO::kWarps];
    static_assert(!DYN || DIAG == 0, "the dynamic schedule exists without diagnostics only");
    __shared__ int tileT[DYN ? kSpecMaxBars : 1], tileU[DYN ? kSpecMaxBars : 1];      // dynamic schedule: tile of each barrier slot
    __shared__ WarpSums<NS, DIAG> ws;
    __shared__ double wacc[(NS > 1 && DIAG) ? GEO::kWarps : 1][(NS > 1 && DIAG) ? (DIAG >= 2 ? 3 : 1) * kDiagAccMax : 1];

    const int NT = p.t_stages, NUS = p.u_stages, LT = p.t_bars, LU = p.u_bars;
    if (threadIdx.x < kSpecMaxBars) {      // lane s arms the barriers of index s -- only those in use (a CTA's set-up is on the critical
        const int s = threadIdx.x;          // path between two steps: the SM is full, so the next step's CTA starts when this slot frees)
        if (s < LT) {
            mbar_init(&fullT[s], 1);                // one expect_tx arrival + the bytes
            mbar_init(&emptyT[s], GEO::kTeamWarps);      // one arrival per consumer warp of the team that took the tile
        }
        if (s < LU) {
            mbar_init(&fullU[s], 1);
            mbar_init(&emptyU[s], GEO::kTeamWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x < GEO::kWarps) nflagged[threadIdx.x] = 0;
    if (DIAG) {
        constexpr int kE = WarpSums<NS, DIAG>::kSlots * WarpSums<NS, DIAG>::kWarps;
        for (int e = threadIdx.x; e < kE; e += blockDim.x) {
            (&ws.v[0][0][0])[e] = 0.0;
            if constexpr (DIAG >= 2) {
                (&ws.v[1][0][0])[e] = DBL_MAX;
                (&ws.v[2][0][0])[e] = -DBL_MAX;
            }
        }
    }
    __syncthreads();
    // programmatic dependent launch: everything above overlapped the previous kernel of the stream.  From here on
    // global memory is touched, so wait for that kernel to complete (no-op without the launch attribute) -- except for
    // the producer warp when the host vouches that the previous kernel is this library's own step, which writes none
    // of the arrays the producer reads: it fills the ring first and waits afterwards (before it folds that step's rows)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool producer_warp = (threadIdx.x >> 5) == GEO::kWarps;
    const bool early_producer = p.early_loads && producer_warp;
    // chained steps (static schedule, same plan as the previous launch of the stream): CTA b writes exactly the cells CTA b
    // of the previous step wrote, so it only has to wait for THAT CTA, not for the whole grid -- the previous step's slow SMs
    // no longer hold up the fast ones, the steps flow into each other per SM.  Everything that does need the whole previous
    // grid (its diagnostics rows) still waits for it, but at the END of this CTA's work, when it has long completed.
    const bool chain = !DYN && p.chain;
    if (!early_producer && !chain) asm volatile("griddepcontrol.wait;" ::: "memory");
    if (chain && !producer_warp) {
        if (threadIdx.x == 0) {
            const unsigned int want = p.seq - 1u;
            unsigned int v;
            // (bounded: the CTA waited for is resident and never waits for this one, so the bound -- about a second --
            // is never reached; it is there so that a host-side sequencing error cannot turn into a hung device)
            for (unsigned int spins = 0; spins < (1u << 24); ++spins) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p.done + blockIdx.x) : "memory");
                if ((int)(v - want) >= 0) break;
                __nanosleep(64);
            }
        }
        consumer_barrier<NS>();
    }
    if constexpr (DYN) {      // (its producer never has to wait: it reads input arrays and the tile counter only)
        spec_dynamic_body<SET, NS>(p, ring, fullT, emptyT, fullU, emptyU, tileT, tileU, flagged, nflagged);
        return;
    } else {

    // static schedule: this CTA takes positions b, b+G, b+2G, ... of the tile list [t tiles | u tiles | v tiles]
    const int G = gridDim.x, b = blockIdx.x;
    // (scalars, not arrays: a runtime-indexed local array would live in local memory)
    int cnt0, cnt1, cnt2;
    int64_t tl0, tl1, tl2;      // first tile of this CTA inside each grid
    {
        // grid g's tiles go round the CTAs starting at CTA rot[g]: CTA b takes tiles (b - rot[g]) mod G, + G, + 2G, ...  With
        // rot = {0, nt, nt + nu} (what the host sets) this is "positions b, b + G, ... of the concatenated list"
        auto sched = [&](int rot, int64_t n, int &cnt, int64_t &tl) {
            tl = (b - rot + G) % G;
            cnt = (tl < n) ? (int)((n - tl + G - 1) / G) : 0;
        };
        sched(p.rot[0], p.ntiles[0], cnt0, tl0);
        sched(p.rot[1], p.ntiles[1], cnt1, tl1);
        sched(p.rot[2], p.ntiles[2], cnt2, tl2);
    }
    // the last tile of a grid may be partial: its CTA takes it before the ring tiles, through guarded global accesses
    auto partial = [&](int ph, int cnt, int64_t tl) {
        return cnt > 0 && tl + (int64_t)(cnt - 1) * G == p.ntiles[ph] - 1 && (p.end[ph] - p.first[ph]) % GEO::kTile != 0;
    };
    const int part0 = partial(0, cnt0, tl0), part1 = partial(1, cnt1, tl1), part2 = partial(2, cnt2, tl2);
    const int ring0 = cnt0 - part0, ring1 = cnt1 - part1, ring2 = cnt2 - part2;      // tiles that travel through the ring
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == GEO::kWarps) {
        // ---------------- producer warp: lane 0 waits, arms the barrier and issues the bulk copies ----------------
        {   // t tiles: tile i -> stage i mod NT, barrier i mod LT
            int st = 0, bi = 0, use = 0;          // of tile i
            int pb = 0, puse = 0;                 // of tile i - NT, the previous tenant of the stage
            const int nfill = ring0 < NT ? ring0 : NT;      // the first pass over the stages waits for nobody
            for (int i = 0;; ++i) {
                if (i == nfill) {
                    // the ring is filling: now (a) honour the stream order if the fill ran ahead of it, (b) fold the previous
                    // step's diagnostics rows -- CTA b takes compact slots b, b + G, ... with the whole warp -- and
                    // (c) retire the lanes that issue nothing.  Chained steps fold at the very end instead (the previous
                    // grid has to be complete for it), so the lanes of a folding warp stay.
                    if (!chain) {
                        if (early_producer) asm volatile("griddepcontrol.wait;" ::: "memory");
                        __syncwarp();
                        for (int cs = b; cs < p.prev.nslots; cs += G) diag_fold_slot(p.prev, cs);
                    }
                    if (lane != 0 && !(chain && b < p.prev.nslots)) return;
                }
                if (i >= ring0) break;
                if (i >= NT) {
                    if (lane == 0) mbar_wait(&emptyT[pb], puse & 1);
                    if (++pb == LT) {
                        pb = 0;
                        ++puse;
                    }
                }
                const int64_t cell = p.first[0] + (tl0 + (int64_t)i * G) * GEO::kTile;
                if (lane == 0) mbar_expect_tx(&fullT[bi], p.tx_bytes[0]);
                __syncwarp();
                char *dst = ring + (size_t)st * p.t_stage_bytes;
                if (lane == 0) {
#pragma unroll 1
                    for (int a = 0; a < Lay<SET, NS>::NT; ++a)
                        if (p.src[0][a]) bulk_g2s(dst + a * GEO::kSlotBytes, p.src[0][a] + cell, GEO::kSlotBytes, &fullT[bi]);
                }
                if (++st == NT) st = 0;
                if (++bi == LT) {
                    bi = 0;
                    ++use;
                }
            }
        }
        {   // u then v tiles: tile k (counted across both grids) -> stage k mod NUS of the u/v carving, barrier k mod LU
            int st = 0, bi = 0, k = 0;
            int pb = 0, puse = 0;
#pragma unroll 1
            for (int ph = 1; ph < 3; ++ph) {
                const int cnt_ph = ph == 1 ? ring1 : ring2;
                const int64_t tl_ph = ph == 1 ? tl1 : tl2;
                for (int i = 0; i < cnt_ph; ++i, ++k) {
                    if (k >= NUS) {
                        if (lane == 0) mbar_wait(&emptyU[pb], puse & 1);
                        if (++pb == LU) {
                            pb = 0;
                            ++puse;
                        }
                    } else if (lane == 0) {      // first use of these bytes as a u/v stage: the last t tile of every t stage they overlap must be done
                        const int lo = (st * p.u_stage_bytes) / p.t_stage_bytes, hi = ((st + 1) * p.u_stage_bytes - 1) / p.t_stage_bytes;
                        for (int s = lo; s <= hi && s < NT; ++s)
                            if (ring0 > s) {
                                const int last = s + ((ring0 - 1 - s) / NT) * NT;      // last t tile that lived in stage s
                                mbar_wait(&emptyT[last % LT], (last / LT) & 1);
                            }
                    }
                    const int64_t cell = p.first[ph] + (tl_ph + (int64_t)i * G) * GEO::kTile;
                    if (lane == 0) mbar_expect_tx(&fullU[bi], p.tx_bytes[ph]);
                    __syncwarp();
                    char *dst = ring + (size_t)st * p.u_stage_bytes;
                    if (lane == 0) {
#pragma unroll 1
                        for (int a = 0; a < Lay<SET, NS>::NUV; ++a)
                            if (p.src[ph][a]) bulk_g2s(dst + a * GEO::kSlotBytes, p.src[ph][a] + cell, GEO::kSlotBytes, &fullU[bi]);
                    }
                    if (++st == NUS) st = 0;
                    if (++bi == LU) bi = 0;
                }
            }
        }
        if (chain && b < p.prev.nslots) {      // chained step: the previous step's rows, now that its grid is certainly complete
            asm volatile("griddepcontrol.wait;" ::: "memory");
            __syncwarp();
            for (int cs = b; cs < p.prev.nslots; cs += G) diag_fold_slot(p.prev, cs);
        }
        return;
    }

    // ---------------- consumer warps: team = warp / 8 takes ring tiles team, team + TEAMS, ... ----------------
    const int team = (TEAMS == 1) ? 0 : warp / GEO::kTeamWarps;
    const int ttid = threadIdx.x - team * GEO::kTeamThreads;
    const int toff = ttid * (kSpecV * 8);
    const int64_t jstride = (int64_t)G * GEO::kTile;
    {   // t phase
        DiagAcc<NS, DIAG, 6, DQ_QSUR_T> dg;
        dg.init(wacc[(NS > 1 && DIAG) ? warp : 0]);
        dg.reset();
        const int64_t jbase = p.first[0] + tl0 * GEO::kTile + ttid * kSpecV;      // this thread's cells of ring tile 0
        int64_t jpart = -1;
        if (part0 && team == 0) {      // the partial tile first: its (slow, guarded) global loads overlap the filling of the ring
            const int64_t j = jbase + (int64_t)(cnt0 - 1) * jstride;
            jpart = j;
            const int64_t left = p.end[0] - j;
            const int nv = left >= 2 ? 2 : (left > 0 ? (int)left : 0);
            if (DIAG) {
                dg.area.v[0] = nv > 0 ? __ldg(p.area[0] + j) : 0.0;
                dg.area.v[1] = nv > 1 ? __ldg(p.area[0] + j + 1) : 0.0;
            }
            FastVec<kSpecV> m;
            const LdPairGuard ld{p.src[0], j, nv};
            const StPairGuard st{j, nv};
            DiagAccGuard<NS, DIAG, 6, DQ_QSUR_T> dgg{dg, nv};
            spec_t_chain<SET, NS>(m, p, ld, st, dgg);
            if (__any_sync(0xffffffffu, nv > 0 && m.bad()) && lane == 0) {
                const int n = nflagged[warp];
                if (n < kSpecBadCap) flagged[warp][n] = -1;
                nflagged[warp] = n + 1;
            }
        }
        int s = team % NT, bi = team % LT, use = team / LT, mine = 0;
        int64_t j = jbase + (int64_t)team * jstride;
        // the cell areas do not travel through the ring: each thread fetches its 16 bytes ONE TILE AHEAD, so that the
        // load's latency hides behind the chain of the current tile instead of in front of it
        double2 a_next = make_double2(0.0, 0.0);
        const int64_t ahead = p.area_ahead ? TEAMS * jstride : 0;
        if (DIAG && p.area_ahead && team < ring0) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[0] + j));
        for (int i = team; i < ring0; i += TEAMS, j += TEAMS * jstride, ++mine) {
            if (DIAG) {
                if (!p.area_ahead) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[0] + j));
                dg.area.v[0] = a_next.x;
                dg.area.v[1] = a_next.y;
                if (p.area_ahead && i + TEAMS < ring0) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[0] + j + ahead));
            }
            mbar_wait(&fullT[bi], use & 1);
            FastVec<kSpecV> m;
            const LdStage<GEO::kSlotBytes> ld{ring + (size_t)s * p.t_stage_bytes + toff};
            const StPair st{j};
            spec_t_chain<SET, NS>(m, p, ld, st, dg);
            __syncwarp();
            if (lane == 0) mbar_arrive(&emptyT[bi]);
            if (__any_sync(0xffffffffu, m.bad()) && lane == 0) {
                const int n = nflagged[warp];
                if (n < kSpecBadCap) flagged[warp][n] = mine;
                nflagged[warp] = n + 1;
            }
            s += TEAMS;
            while (s >= NT) s -= NT;
            bi += TEAMS;
            while (bi >= LT) {
                bi -= LT;
                ++use;
            }
        }
        __syncwarp();
        const int nf = nflagged[warp];
        if (nf) {
            spec_cold_phase<SET, NS, DIAG>(p, 0, jpart, jbase + (int64_t)team * jstride, TEAMS * jstride, mine, flagged[warp], nf, ws);
            __syncwarp();
            if (lane == 0) nflagged[warp] = 0;
            __syncwarp();
        } else if (DIAG) {
            dg.flush(ws, DQ_QSUR_T);
        }
    }
    {   // u phase, then v phase: same code, same carving, tile counter k runs across both grids
        int kbase = 0;      // ring tiles of this CTA before the current grid
#pragma unroll 1
        for (int ph = 1; ph < 3; ++ph) {
            DiagAcc<NS, DIAG, 2, DQ_QSUR_U> dg;
            dg.init(wacc[(NS > 1 && DIAG) ? warp : 0]);
            dg.reset();
            const int north = ph - 1;
            const int cnt_ph = ph == 1 ? cnt1 : cnt2, ring_ph = ph == 1 ? ring1 : ring2;
            const int64_t jbase = p.first[ph] + (ph == 1 ? tl1 : tl2) * GEO::kTile + ttid * kSpecV;
            int64_t jpart = -1;
            if (ring_ph != cnt_ph && team == 0) {      // partial tile of this grid, before its ring tiles
                const int64_t j = jbase + (int64_t)(cnt_ph - 1) * jstride;
                jpart = j;
                const int64_t left = p.end[ph] - j;
                const int nv = left >= 2 ? 2 : (left > 0 ? (int)left : 0);
                if (DIAG) {
                    dg.area.v[0] = nv > 0 ? __ldg(p.area[ph] + j) : 0.0;
                    dg.area.v[1] = nv > 1 ? __ldg(p.area[ph] + j + 1) : 0.0;
                }
                FastVec<kSpecV> m;
                const LdPairGuard ld{p.src[ph], j, nv};
                const StPairGuard st{j, nv};
                DiagAccGuard<NS, DIAG, 2, DQ_QSUR_U> dgg{dg, nv};
                spec_uv_chain<SET, NS>(m, p, north, ld, st, dgg);
                if (__any_sync(0xffffffffu, nv > 0 && m.bad()) && lane == 0) {
                    const int n = nflagged[warp];
                    if (n < kSpecBadCap) flagged[warp][n] = -1;
                    nflagged[warp] = n + 1;
                }
            }
            // this team's first tile of the grid: the smallest i >= 0 with (kbase + i) mod TEAMS == team
            const int i0 = (TEAMS == 1) ? 0 : ((team - kbase) % TEAMS + TEAMS) % TEAMS;
            int h = (kbase + i0) % NUS, bi = (kbase + i0) % LU, use = (kbase + i0) / LU, mine = 0;
            const int64_t jfirst = jbase + (int64_t)i0 * jstride;
            int64_t j = jfirst;
            double2 a_next = make_double2(0.0, 0.0);
            const int64_t ahead = p.area_ahead ? TEAMS * jstride : 0;
            if (DIAG && p.area_ahead && i0 < ring_ph) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[ph] + j));
            for (int i = i0; i < ring_ph; i += TEAMS, j += TEAMS * jstride, ++mine) {
                if (DIAG) {
                    if (!p.area_ahead) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[ph] + j));
                    dg.area.v[0] = a_next.x;
                    dg.area.v[1] = a_next.y;
                    if (p.area_ahead && i + TEAMS < ring_ph) a_next = __ldg(reinterpret_cast<const double2 *>(p.area[ph] + j + ahead));
                }
                mbar_wait(&fullU[bi], use & 1);
                FastVec<kSpecV> m;
                const LdStage<GEO::kSlotBytes> ld{ring + (size_t)h * p.u_stage_bytes + toff};
                const StPair st{j};
                spec_uv_chain<SET, NS>(m, p, north, ld, st, dg);
                __syncwarp();
                if (lane == 0) mbar_arrive(&emptyU[bi]);
                if (__any_sync(0xffffffffu, m.bad()) && lane == 0) {
                    const int n = nflagged[warp];
                    if (n < kSpecBadCap) flagged[warp][n] = mine;
                    nflagged[warp] = n + 1;
                }
                h += TEAMS;
                while (h >= NUS) h -= NUS;
                bi += TEAMS;
                while (bi >= LU) {
                    bi -= LU;
                    ++use;
                }
            }
            kbase += ring_ph;
            __syncwarp();
            const int nf = nflagged[warp];
            if (nf) {
                spec_cold_phase<SET, NS, DIAG>(p, ph, jpart, jfirst, TEAMS * jstride, mine, flagged[warp], nf, ws);
                __syncwarp();
                if (lane == 0) nflagged[warp] = 0;
                __syncwarp();
            } else if (DIAG) {
                dg.flush(ws, north ? DQ_QSUR_V : DQ_QSUR_U);
            }
        }
    }
    // hand-over to the same CTA of the next step: every consumer warp has issued its last store
    consumer_barrier<NS>();
    if (threadIdx.x == 0 && p.done) {
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p.done + blockIdx.x), "r"(p.seq) : "memory");
    }
    if (DIAG) {
        if (chain) asm volatile("griddepcontrol.wait;" ::: "memory");      // the rows go where the step before the previous one left its own
        diag_finish<NS, DIAG>(p, ws);
    }
    }      // static schedule
}

// ---------------------------------------------------------------------------------------------
// host side: does the fused plan fit the specialised kernel?  If so, build its plan and launch.
// ---------------------------------------------------------------------------------------------
static int spec_num_sms()
{
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}

static bool is_bulk(int m) { return m == M_CCLM || m == M_MOM5; }

template <int SET, int NS>
static bool spec_fill(const FusedPlan &p, SpecPlan &sp)
{
    using L = Lay<SET, NS>;
    const FusedT &t = p.t;
    const FusedTType &T0 = t.ty[0];
    const double **s = sp.src[0];
    s[L::PSUR] = T0.psur; s[L::QATM] = T0.qatm; s[L::TATM] = T0.tatm; s[L::UATM] = T0.uatm; s[L::VATM] = T0.vatm;
    s[L::RSDD] = t.rsdd; s[L::BIAS] = t.bias;
    if (SET == SET_BULK) {
        s[L::AEV] = T0.a_evap;
        s[L::PATM] = T0.patm;
        if (T0.a_sens == T0.a_evap) {
            sp.ase_slot = L::AEV;
        } else {
            s[L::ASE] = T0.a_sens;
            sp.ase_slot = L::ASE;
        }
        if (!T0.a_evap || !T0.patm || !T0.a_sens) return false;
    }
    if (!T0.psur || !T0.qatm || !T0.tatm || !T0.uatm || !T0.vatm) return false;
    bool any_avg_t = false, any_avg_uv[2] = {false, false};
    for (int q = DQ_MEVA; q <= DQ_RSDR; ++q) any_avg_t = any_avg_t || sp.out[0][q] != nullptr;
    sp.any_avg_t = any_avg_t;
    any_avg_uv[0] = sp.out[0][DQ_UMOM] != nullptr;
    any_avg_uv[1] = sp.out[0][DQ_VMOM] != nullptr;
    for (int i = 0; i < NS; ++i) {
        const FusedTType &T = t.ty[i];
        // the atmosphere / shared bottom fields must be the SAME arrays for every surface type (basic.F90:334-358)
        if (T.psur != T0.psur || T.qatm != T0.qatm || T.tatm != T0.tatm || T.uatm != T0.uatm || T.vatm != T0.vatm) return false;
        if (SET == SET_BULK && (T.a_evap != T0.a_evap || T.a_sens != T0.a_sens || T.patm != T0.patm)) return false;
        s[L::FICE(i)] = T.fice;
        s[L::TSUR(i)] = T.tsur;
        if (!T.fice || !T.tsur) return false;
        if (NS > 1 && any_avg_t) {
            s[L::FARE(i)] = T.fare;
            if (!T.fare) return false;
        }
    }
    for (int g = 0; g < 2; ++g) {
        const FusedUVType &Y0 = p.uv[g].ty[0];
        const double **u = sp.src[g + 1];
        u[L::U_UATM] = Y0.uatm;
        u[L::U_VATM] = Y0.vatm;
        if (!Y0.uatm || !Y0.vatm) return false;
        if (SET == SET_BULK) {
            u[L::U_PSUR] = Y0.psur;
            u[L::U_AMOM] = Y0.a_mom;
            if (!Y0.psur || !Y0.a_mom) return false;
        }
        for (int i = 0; i < NS; ++i) {
            const FusedUVType &Y = p.uv[g].ty[i];
            if (Y.uatm != Y0.uatm || Y.vatm != Y0.vatm) return false;
            if (SET == SET_BULK) {
                if (Y.psur != Y0.psur || Y.a_mom != Y0.a_mom) return false;
                u[L::U_FICE(i)] = Y.fice;
                u[L::U_TSUR(i)] = Y.tsur;
                if (!Y.fice || !Y.tsur) return false;
            }
            if (NS > 1 && any_avg_uv[g]) {
                u[L::U_FARE(i)] = Y.fare;
                if (!Y.fare) return false;
            }
        }
    }
    // the two carvings of the ring: as many stages as fit (2 CTAs per SM with one type, the whole SM with two)
    int t_slots = 0, u_slots = 0;
    for (int a = 0; a < L::NT; ++a)
        if (sp.src[0][a]) t_slots = a + 1;
    for (int g = 1; g < 3; ++g)
        for (int a = 0; a < L::NUV; ++a)
            if (sp.src[g][a]) u_slots = (a + 1 > u_slots) ? a + 1 : u_slots;
    // 227 KB per SM, 1 KB reserved per CTA, static shared memory: barriers + flag lists (2 KB) and the diagnostics
    // staging (one type: <= 2 KB; two types: 6 KB with sums, 18 KB with min/max)
    const int budget = (NS == 1) ? 108 * 1024 : (sp.diag >= 2 ? 204 * 1024 : 216 * 1024);
    sp.t_stage_bytes = t_slots * SpecGeom<NS>::kSlotBytes;
    sp.u_stage_bytes = u_slots * SpecGeom<NS>::kSlotBytes;
    sp.t_stages = budget / sp.t_stage_bytes;
    sp.u_stages = budget / sp.u_stage_bytes;
    if (sp.t_stages > kSpecMaxStages) sp.t_stages = kSpecMaxStages;
    if (sp.u_stages > kSpecMaxStages) sp.u_stages = kSpecMaxStages;
    auto lcm = [](int a, int b) {
        int x = a, y = b;
        while (y) {
            const int t = x % y;
            x = y;
            y = t;
        }
        return a / x * b;
    };
    const int teams = SpecGeom<NS>::kTeams;
    // one barrier per (team, stage) pair: lcm(teams, stages) of them; give up a stage if that exceeds the barrier arrays
    while (sp.t_stages > 2 && lcm(teams, sp.t_stages) > kSpecMaxBars) --sp.t_stages;
    while (sp.u_stages > 2 && lcm(teams, sp.u_stages) > kSpecMaxBars) --sp.u_stages;
    sp.t_bars = lcm(teams, sp.t_stages);
    sp.u_bars = lcm(teams, sp.u_stages);
    return sp.t_stages >= 2 && sp.u_stages >= 2 && sp.t_bars <= kSpecMaxBars && sp.u_bars <= kSpecMaxBars;
}

// cells[g] cells starting at first[g] (every bound array 16-byte aligned there: decided by the caller)
static bool spec_build(const FusedPlan &p, const int64_t first[3], const int64_t cells[3], SpecPlan &sp, int *set_out)
{
    if (p.S < 1 || p.S > kSpecMaxNS || !p.do_normal) return false;
    const FusedT &t = p.t;
    if (t.avg_qsur || p.uv[0].avg_qsur || p.uv[1].avg_qsur) return false;
    if (p.S == 1 && (t.avg_meva || t.avg_hlat || t.avg_hsen || t.avg_rbbr || t.avg_rsdr || p.uv[0].avg_mom || p.uv[1].avg_mom)) return false;
    int set = -1;
    for (int i = 0; i < p.S; ++i) {
        const FusedTType &T = t.ty[i];
        const FusedUVType &U = p.uv[0].ty[i], &W = p.uv[1].ty[i];
        if (T.m_qsur != M_CCLM || T.qsur_in || U.qsur_in || W.qsur_in) return false;
        if (T.m_hlat != M_WATER && T.m_hlat != M_ICE) return false;
        if (p.do_early ? (T.m_rbbr != M_STBO) : (T.m_rbbr != M_NONE)) return false;
        int si;
        if (is_bulk(T.m_meva) && is_bulk(T.m_hsen) && U.m_qsur == M_CCLM && W.m_qsur == M_CCLM && is_bulk(U.m_mom) && is_bulk(W.m_mom))
            si = SET_BULK;
        else if (T.m_meva == M_RCO && T.m_hsen == M_RCO && U.m_qsur == M_NONE && W.m_qsur == M_NONE && U.m_mom == M_RCO && W.m_mom == M_RCO)
            si = SET_RCO;
        else
            return false;
        if (set >= 0 && si != set) return false;
        set = si;
    }
    if (p.diag && !(t.area && p.uv[0].area && p.uv[1].area)) return false;

    memset(&sp, 0, sizeof sp);
    sp.c = p.c;
    sp.ns = p.S;
    for (int g = 0; g < 3; ++g) {
        sp.first[g] = first[g];
        sp.end[g] = first[g] + cells[g];
        const int tile = (p.S == 1) ? SpecGeom<1>::kTile : SpecGeom<2>::kTile;
        sp.ntiles[g] = (int)((cells[g] + tile - 1) / tile);
    }
    sp.do_early = p.do_early;
    sp.has_bias = t.bias != nullptr;
    sp.has_rsdr = t.rsdd != nullptr;
    sp.diag = p.diag;
    for (int i = 0; i < p.S; ++i) {
        const FusedTType &T = t.ty[i];
        const FusedUVType &U = p.uv[0].ty[i], &W = p.uv[1].ty[i];
        double **o = sp.out[i + 1];
        sp.latent_heat[i] = T.latent_heat;
        o[DQ_QSUR_T] = T.qsur; o[DQ_MEVA] = T.meva; o[DQ_HLAT] = T.hlat; o[DQ_HSEN] = T.hsen;
        o[DQ_RBBR] = p.do_early ? T.rbbr : nullptr;
        o[DQ_RSDR] = sp.has_rsdr ? T.rsdr : nullptr;
        o[DQ_QSUR_U] = U.qsur; o[DQ_UMOM] = U.mom; o[DQ_QSUR_V] = W.qsur; o[DQ_VMOM] = W.mom;
        if (!T.qsur || !T.meva || !T.hlat || !T.hsen || !U.mom || !W.mom) return false;
        if (set == SET_BULK && (!U.qsur || !W.qsur)) return false;
        if (p.do_early && !T.rbbr) return false;
        if (sp.has_rsdr && !T.rsdr) return false;
    }
    sp.out[0][DQ_MEVA] = t.avg_meva; sp.out[0][DQ_HLAT] = t.avg_hlat; sp.out[0][DQ_HSEN] = t.avg_hsen;
    sp.out[0][DQ_RBBR] = p.do_early ? t.avg_rbbr : nullptr;
    sp.out[0][DQ_RSDR] = sp.has_rsdr ? t.avg_rsdr : nullptr;
    sp.out[0][DQ_UMOM] = p.uv[0].avg_mom;
    sp.out[0][DQ_VMOM] = p.uv[1].avg_mom;
    if (!p.do_early && t.avg_rbbr) return false;
    bool ok;
    if (set == SET_BULK) ok = (p.S == 1) ? spec_fill<SET_BULK, 1>(p, sp) : spec_fill<SET_BULK, 2>(p, sp);
    else ok = (p.S == 1) ? spec_fill<SET_RCO, 1>(p, sp) : spec_fill<SET_RCO, 2>(p, sp);
    if (!ok) return false;
    for (int g = 0; g < 3; ++g) {
        int n = 0;
        for (int k = 0; k < kSpecMaxSlots; ++k) n += sp.src[g][k] != nullptr;
        sp.tx_bytes[g] = (uint32_t)n * (uint32_t)((p.S == 1) ? SpecGeom<1>::kSlotBytes : SpecGeom<2>::kSlotBytes);
    }
    sp.area[0] = t.area;
    sp.area[1] = p.uv[0].area;
    sp.area[2] = p.uv[1].area;
    for (int k = 0; k < (kSpecMaxNS + 1) * DQ_COUNT; ++k) sp.dmap[k] = p.diag ? p.diag_map[k] : (signed char)-1;
    *set_out = set;
    return true;
}

static int SpecGeomCtas(int ns) { return ns == 1 ? SpecGeom<1>::kCtasPerSm : SpecGeom<2>::kCtasPerSm; }

static int spec_grid(const SpecPlan &sp)
{
    const int64_t total = (int64_t)sp.ntiles[0] + sp.ntiles[1] + sp.ntiles[2];
    const int cap = SpecGeomCtas(sp.ns) * spec_num_sms();
    return (int)(total < cap ? total : cap);
}

// CTAs of the specialised kernel the device holds at once
int spec_capacity(int num_surface_types) { return SpecGeomCtas(num_surface_types) * spec_num_sms(); }

// tiles per CTA from which the dynamic schedule is used: below, the static one has nothing to lose to imbalance and the
// claims would only add latency (measured, RCO set at 10^6 cells = 20 tiles per CTA: 29.2 us static, 32.7 us dynamic)
constexpr int kSpecDynMinTiles = 48;
static bool spec_wants_dyn(const SpecPlan &sp, int dyn_min_tiles)
{
    if (sp.diag) return false;
    // Two surface types keep the static schedule unless the caller asks (option dyn_min_tiles): a t tile is 128 KB of traffic
    // and ~9 us of a team's time there, claims are coarse against 132 tiles per CTA, and consecutive static steps hand over
    // per CTA -- measured on C5 (10^7 cells, call 14, two repetitions): static 0.908 / 0.909 ms, dynamic 0.922 / 0.926 ms.
    if (sp.ns > 1 && dyn_min_tiles <= 0) return false;
    const int64_t min_tiles = dyn_min_tiles > 0 ? dyn_min_tiles : kSpecDynMinTiles;
    return (int64_t)sp.ntiles[0] + sp.ntiles[1] + sp.ntiles[2] >= min_tiles * spec_grid(sp);
}

// the specialised half of resolve_fused (kernels.cu): if the plan fits the specialised kernel over this range, L gets the
// kernel's parameter block without the per-step fields, its formula set, grid and schedule
bool spec_resolve(const FusedPlan &p, const int64_t first[3], const int64_t cells[3], int dyn_min_tiles, FusedLaunch &L)
{
    SpecPlan &sp = L.sp;
    int set = 0;
    if (cells[0] + cells[1] + cells[2] <= 0 || !spec_build(p, first, cells, sp, &set)) return false;
    const int grid = spec_grid(sp);
    sp.dyn = spec_wants_dyn(sp, dyn_min_tiles) ? 1 : 0;
    // static schedule: the three grids follow each other round the CTAs (positions b, b + G, ... of the concatenated list).
    // (Choosing the starts so that the CTAs with one tile more spread evenly over the SMs by bytes was tried for the chained
    // 8-GPU shards -- 2480 vs 2404 KB per SM with plain succession -- and measured no gain: 61.2 vs 60.2 us, within the
    // box-to-box spread; profiles/README.md.)
    sp.rot[0] = 0;
    sp.rot[1] = grid > 0 ? sp.ntiles[0] % grid : 0;
    sp.rot[2] = grid > 0 ? (int)(((int64_t)sp.ntiles[0] + sp.ntiles[1]) % grid) : 0;
    // cell areas one tile ahead while there are few tiles per CTA (8-GPU shard of C4, 25 tiles per CTA: 61.3 -> 58.3 us);
    // with many the kernel is DRAM bound and the earlier loads only synchronise the warps (10^7 cells: 0.433 -> 0.455 ms)
    sp.area_ahead = ((int64_t)sp.ntiles[0] + sp.ntiles[1] + sp.ntiles[2] < (int64_t)64 * grid) ? 1 : 0;
    L.spec_set = set;
    L.spec_grid = grid;
    // dynamic schedule: every tile is claimed once, every CTA's producer makes one failing claim
    const unsigned nuv = (unsigned)(sp.ntiles[1] + sp.ntiles[2]);
    L.claims = sp.dyn ? (unsigned int)sp.ntiles[0] + (nuv + kDynUvBatch - 1) / kDynUvBatch + 2u * (unsigned)grid : 0u;
    return true;
}

template <int SET, int NS, int DIAG, bool DYN>
static cudaError_t spec_launch_t(const SpecPlan &sp, int grid, cudaStream_t stream)
{
    const size_t tb = (size_t)sp.t_stages * sp.t_stage_bytes, ub = (size_t)sp.u_stages * sp.u_stage_bytes;
    const size_t smem = tb > ub ? tb : ub;
    static size_t configured = 0;
    if (smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(flux_spec_kernel<SET, NS, DIAG, DYN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(flux_spec_kernel<SET, NS, DIAG, DYN>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        configured = smem;
    }
    // programmatic stream serialisation: this launch may become resident while the previous kernel of the stream
    // drains; the kernel itself waits (griddepcontrol.wait) before its first global access
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(SpecGeom<NS>::kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, flux_spec_kernel<SET, NS, DIAG, DYN>, sp);
}

template <int SET, int NS>
static cudaError_t spec_launch_d(const SpecPlan &sp, int grid, cudaStream_t stream)
{
    if (sp.diag >= 2) return spec_launch_t<SET, NS, 2, false>(sp, grid, stream);
    if (sp.diag == 1) return spec_launch_t<SET, NS, 1, false>(sp, grid, stream);
    if (sp.dyn) return spec_launch_t<SET, NS, 0, true>(sp, grid, stream);
    return spec_launch_t<SET, NS, 0, false>(sp, grid, stream);
}

// sp: a resolved parameter block (spec_resolve) with the per-step fields filled in
int spec_launch(const SpecPlan &sp, int set, int grid, cudaStream_t stream)
{
    if (sp.diag && !sp.partials) return (int)cudaErrorInvalidValue;
    if (sp.dyn && !sp.tile_counter) return (int)cudaErrorInvalidValue;
    cudaError_t e;
    if (set == SET_BULK) e = (sp.ns == 1) ? spec_launch_d<SET_BULK, 1>(sp, grid, stream) : spec_launch_d<SET_BULK, 2>(sp, grid, stream);
    else e = (sp.ns == 1) ? spec_launch_d<SET_RCO, 1>(sp, grid, stream) : spec_launch_d<SET_RCO, 2>(sp, grid, stream);
    return (int)e;
}

}  // namespace fc
