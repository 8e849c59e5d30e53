// kernels.cu -- hand-written sm_100a kernels of the flux calculator hot path.
//
//  fused_step_kernel   generic fused pass (any number of surface types, any method mix, averaging): t-, u-
//                      and v-grid chains of every surface type in one pass over SoA fields, intermediates in
//                      registers, 128-bit coalesced loads/stores, per-warp diagnostics partials.  Also the
//                      guarded variant for ragged remainders / misaligned arrays.  The chain is a template over the
//                      arithmetic policy: the hot instantiation flags operands outside the proven range, the warp
//                      then re-runs it out of line with the IEEE policy.  The specialised persistent kernel of
//                      spec_kernel.cu takes over for the canonical plans with one or two surface types.
//  oplist_kernel       interpreter for the reference's pass sequence (exact semantics for aliased
//                      outputs / unfused calc_* calls / the Level-1 flux_lib array routines).
//  diag_finalize, transpose_corrections, regrid_csr: small helpers.
//
// The path is elementwise FP64 streaming: HBM-bound, no reuse across cells, so no tensor cores.
#include "plan.h"

#include <cuda_runtime.h>
#include <float.h>
#include <stdio.h>
#include <stdlib.h>

namespace fc {

// ---------------------------------------------------------------------------------------------
// vector helpers
// ---------------------------------------------------------------------------------------------
constexpr int V = kFusedVec;
using V2 = Vd<V>;
using Fast = FastVec<V>;
using Exact = ExactVec<V>;

// Loader policies: where a thread's V cells of an input array come from, and how results are stored.
//   LdGlobal : 128-bit global loads/stores (every array 16-byte aligned, all V cells valid)
//   LdGuard  : guarded scalar accesses (ragged tail of a grid, misaligned arrays)
struct LdGlobal {
    static constexpr bool kFull = true;
    int64_t j;
    __device__ __forceinline__ V2 load(const double *__restrict__ p) const
    {
        static_assert(V == 2, "128-bit path assumes 2 cells per thread");
        const double2 t = __ldg(reinterpret_cast<const double2 *>(p + j));
        V2 r;
        r.v[0] = t.x;
        r.v[1] = t.y;
        return r;
    }
    __device__ __forceinline__ void store(double *p, const V2 &x) const
    {
        *reinterpret_cast<double2 *>(p + j) = make_double2(x.v[0], x.v[1]);
    }
};

struct LdGuard {
    static constexpr bool kFull = false;
    int64_t j;
    int nv;
    __device__ __forceinline__ V2 load(const double *__restrict__ p) const
    {
        V2 r;
#pragma unroll
        for (int k = 0; k < V; ++k) r.v[k] = (k < nv) ? __ldg(p + j + k) : 1.0;
        return r;
    }
    __device__ __forceinline__ void store(double *p, const V2 &x) const
    {
#pragma unroll
        for (int k = 0; k < V; ++k)
            if (k < nv) p[j + k] = x.v[k];
    }
};

// a field loaded at most once per distinct pointer: atmosphere fields are aliased into every
// surface type (distribute_input_field, basic.F90:334-358), so consecutive types usually share them
template <class LD>
struct Cached {
    const double *ptr = nullptr;
    V2 val;
    __device__ __forceinline__ const V2 &get(const LD &ld, const double *p)
    {
        if (p != ptr) {
            ptr = p;
            if (p) val = ld.load(p);
        }
        return val;
    }
};

__device__ __forceinline__ V2 vzero()
{
    V2 r;
#pragma unroll
    for (int k = 0; k < V; ++k) r.v[k] = 0.0;
    return r;
}

// acc = acc + x*fare, separate multiply and add (average_across_surface_types, calculate.F90:379-382)
__device__ __forceinline__ void avg_acc(V2 &acc, const V2 &x, const V2 &fare)
{
#pragma unroll
    for (int k = 0; k < V; ++k) acc.v[k] = add(acc.v[k], mul(x.v[k], fare.v[k]));
}

// ---------------------------------------------------------------------------------------------
// diagnostics: DIAG == 1: sum_j area_j*x_j ; DIAG == 2: additionally min_j x_j and max_j x_j.
// thread partial -> warp shuffle tree -> lane 0 stores the warp's partial to global memory:
// partials[plane][compact slot][warp row], planes = (sum, min, max).  No shared memory, no CTA barrier;
// two tiny deterministic kernels combine the rows afterwards (diag_reduce_rows / diag_reduce_final).
// ---------------------------------------------------------------------------------------------
struct DiagCtx {
    double *base;        // partials
    int64_t rows;        // row stride (total warp rows of the launch)
    int64_t row;         // this warp's row
    int64_t plane;       // slots * rows
};

template <int DIAG>
__device__ __forceinline__ void diag_commit(const FusedPlan &p, DiagCtx &d, int base, int q, const V2 &x, const V2 &area, int nv)
{
    const int slot = base + q;
    double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
#pragma unroll
    for (int k = 0; k < V; ++k)
        if (k < nv) {
            s = add(s, mul(area.v[k], x.v[k]));
            if (DIAG >= 2) {
                mn = fmin(mn, x.v[k]);
                mx = fmax(mx, x.v[k]);
            }
        }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s = add(s, __shfl_down_sync(0xffffffffu, s, off));
        if (DIAG >= 2) {
            mn = fmin(mn, __shfl_down_sync(0xffffffffu, mn, off));
            mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, off));
        }
    }
    if ((threadIdx.x & 31) == 0) {
        double *o = d.base + (int64_t)p.diag_map[slot] * d.rows + d.row;
        o[0] = s;
        if (DIAG >= 2) {
            o[d.plane] = mn;
            o[2 * d.plane] = mx;
        }
    }
}
#define DIAG_COMMIT(base, q, x) diag_commit<DIAG>(p, dg, (base), (q), (x), area, nv)

// ---------------------------------------------------------------------------------------------
// per-surface-type arithmetic of the t grid, instantiated with the fast and the exact policy
// ---------------------------------------------------------------------------------------------
// inputs of one surface type, preloaded into registers
struct TIn {
    V2 fice_, psur_, tsur_, qatm_, tatm_, patm_, uatm_, vatm_, aev_, ase_, qsur_in_, bias_;
    __device__ __forceinline__ const V2 &fice() const { return fice_; }
    __device__ __forceinline__ const V2 &psur() const { return psur_; }
    __device__ __forceinline__ const V2 &tsur() const { return tsur_; }
    __device__ __forceinline__ const V2 &qatm() const { return qatm_; }
    __device__ __forceinline__ const V2 &tatm() const { return tatm_; }
    __device__ __forceinline__ const V2 &patm() const { return patm_; }
    __device__ __forceinline__ const V2 &uatm() const { return uatm_; }
    __device__ __forceinline__ const V2 &vatm() const { return vatm_; }
    __device__ __forceinline__ const V2 &aev() const { return aev_; }
    __device__ __forceinline__ const V2 &ase() const { return ase_; }
    __device__ __forceinline__ const V2 &qsur_in() const { return qsur_in_; }
    __device__ __forceinline__ const V2 &bias() const { return bias_; }
};
struct TOut {
    V2 qsur, meva, hlat, hsen, rbbr;
};

template <class M, class IN>
__device__ __forceinline__ bool t_type_math(const FusedPlan &p, const FusedTType &ty, const IN &in, bool has_bias, TOut &o)
{
    M m;
    const Consts &c = p.c;
    if (p.do_normal) {
        // --- QSUR: calc_spec_vapor_surface (calculate.F90:25-50)
        if (ty.m_qsur == M_CCLM) o.qsur = spec_vapor_surface_cclm(m, in.fice(), in.psur(), in.tsur(), c);
        else if (ty.qsur_in) o.qsur = in.qsur_in();
        V2 vel;
        if (ty.m_meva >= M_CCLM || ty.m_hsen >= M_CCLM) vel = wind_speed(m, in.uatm(), in.vatm());
        // --- MEVA: calc_flux_mass_evap (calculate.F90:54-120); T slot <- TATM (:87,:98)
        if (ty.m_meva != M_NONE) {
            if (ty.m_meva == M_CCLM || ty.m_meva == M_MOM5)
                o.meva = flux_mass_evap_cclm(m, in.aev(), in.psur(), in.qatm(), o.qsur, in.tatm(), vel, c);
            else if (ty.m_meva == M_RCO)
                o.meva = flux_mass_evap_rco(m, in.qatm(), in.tsur(), vel);
            else
                o.meva = vzero();                                              // 'zero' (:79)
            if (has_bias) o.meva = M::add(o.meva, in.bias());                    // :112-116
        }
        // --- HLAT: calc_flux_heat_latent (calculate.F90:124-154), sees the corrected MEVA
        if (ty.m_hlat != M_NONE)
            o.hlat = (ty.m_hlat == M_ZERO) ? vzero() : M::mul(o.meva, M::bc(ty.latent_heat));   // heat_latent.F90:41,65
        // --- HSEN: calc_flux_heat_sensible (calculate.F90:156-208); q_s slot <- QATM (:178,:190)
        if (ty.m_hsen != M_NONE) {
            if (ty.m_hsen == M_CCLM || ty.m_hsen == M_MOM5)
                o.hsen = flux_heat_sensible_cclm(m, in.ase(), in.patm(), in.psur(), in.qatm(), in.tatm(), in.tsur(), vel, c);
            else if (ty.m_hsen == M_RCO)
                o.hsen = flux_heat_sensible_rco<M>(in.tatm(), in.tsur(), vel);
            else
                o.hsen = vzero();
        }
    }
    // --- RBBR: calc_flux_radiation_blackbody (calculate.F90:320-345), early phase
    if (p.do_early && ty.m_rbbr != M_NONE)
        o.rbbr = (ty.m_rbbr == M_ZERO) ? vzero() : flux_radiation_blackbody_StBo<M>(in.tsur(), c.stefan_boltzmann_constant);
    return m.bad();
}

// how often the recompute path ran (per warp here, per thread in the specialised kernel); fc_get_info("exact_path_calls")
__device__ unsigned long long g_exact_calls = 0ull;

unsigned long long read_exact_calls()
{
    unsigned long long v = 0;
    cudaMemcpyFromSymbol(&v, g_exact_calls, sizeof v);
    return v + read_spec_exact_calls();
}

// The chain of one thread's V cells, written over the arithmetic policy M: the hot instantiation (Fast) returns whether an
// operand left the range in which the lock-step sequences are proven; the kernel then re-runs the SAME chain with the IEEE
// policy for the whole warp (fused_cold_warp): no by-value call, no stack frame on the hot path.
template <class M, int SS, int DIAG, class LD>
__device__ __forceinline__ bool t_chain(const FusedPlan &p, const LD &ld, int nv, DiagCtx &dg)
{
    const FusedT &t = p.t;
    bool bad = false;
    const int S = SS ? SS : p.S;
    Cached<LD> cPSUR, cQATM, cTATM, cPATM, cUATM, cVATM, cAEV, cASE, cFICE, cTSUR;
    TIn in;
    V2 rsdd, area;
    const bool has_bias = p.do_normal && t.bias != nullptr;
    const bool has_rsdr = p.do_normal && t.rsdd != nullptr;
    if (has_bias) in.bias_ = ld.load(t.bias);
    if (has_rsdr) rsdd = ld.load(t.rsdd);
    if (DIAG) area = ld.load(t.area);
    V2 aQ = vzero(), aM = vzero(), aL = vzero(), aH = vzero(), aR = vzero(), aS = vzero();   // type-0 averages

    auto per_type = [&](const int i) {
        const FusedTType &ty = t.ty[i];
        V2 fare;
        TOut o;
        if (LD::kFull || nv) {
            // all loads of this surface type up front (memory-level parallelism), then arithmetic
            if (ty.fare) fare = ld.load(ty.fare);
            in.tsur_ = cTSUR.get(ld, ty.tsur);
            if (p.do_normal) {
                in.psur_ = cPSUR.get(ld, ty.psur);
                in.qatm_ = cQATM.get(ld, ty.qatm);
                in.tatm_ = cTATM.get(ld, ty.tatm);
                in.uatm_ = cUATM.get(ld, ty.uatm);
                in.vatm_ = cVATM.get(ld, ty.vatm);
                in.fice_ = cFICE.get(ld, ty.fice);
                in.aev_ = cAEV.get(ld, ty.a_evap);
                in.ase_ = cASE.get(ld, ty.a_sens);
                in.patm_ = cPATM.get(ld, ty.patm);
                if (ty.qsur_in) in.qsur_in_ = ld.load(ty.qsur_in);
            }
            bad |= t_type_math<M>(p, ty, in, has_bias, o);
            if (p.do_normal) {
                if (ty.m_qsur == M_CCLM) ld.store(ty.qsur, o.qsur);
                if (ty.m_meva != M_NONE) ld.store(ty.meva, o.meva);
                if (ty.m_hlat != M_NONE) ld.store(ty.hlat, o.hlat);
                if (ty.m_hsen != M_NONE) ld.store(ty.hsen, o.hsen);
                if (has_rsdr) ld.store(ty.rsdr, rsdd);                 // calculate.F90:347-364
            }
            if (p.do_early && ty.m_rbbr != M_NONE) ld.store(ty.rbbr, o.rbbr);
            if (t.avg_qsur) avg_acc(aQ, o.qsur, fare);
            if (t.avg_meva) avg_acc(aM, o.meva, fare);
            if (t.avg_hlat) avg_acc(aL, o.hlat, fare);
            if (t.avg_hsen) avg_acc(aH, o.hsen, fare);
            if (t.avg_rbbr) avg_acc(aR, o.rbbr, fare);
            if (t.avg_rsdr) avg_acc(aS, rsdd, fare);
        }
        if (DIAG) {
            const int base = (i + 1) * DQ_COUNT;
            if (p.do_normal) {
                if (ty.m_qsur == M_CCLM) DIAG_COMMIT(base, DQ_QSUR_T, o.qsur);
                if (ty.m_meva != M_NONE) DIAG_COMMIT(base, DQ_MEVA, o.meva);
                if (ty.m_hlat != M_NONE) DIAG_COMMIT(base, DQ_HLAT, o.hlat);
                if (ty.m_hsen != M_NONE) DIAG_COMMIT(base, DQ_HSEN, o.hsen);
                if (has_rsdr) DIAG_COMMIT(base, DQ_RSDR, rsdd);
            }
            if (p.do_early && ty.m_rbbr != M_NONE) DIAG_COMMIT(base, DQ_RBBR, o.rbbr);
        }
    };
    if constexpr (SS > 0) {
#pragma unroll
        for (int i = 0; i < SS; ++i) per_type(i);
    } else {
#pragma unroll 1
        for (int i = 0; i < S; ++i) per_type(i);
    }
    if (LD::kFull || nv) {
        if (t.avg_qsur) ld.store(t.avg_qsur, aQ);
        if (t.avg_meva) ld.store(t.avg_meva, aM);
        if (t.avg_hlat) ld.store(t.avg_hlat, aL);
        if (t.avg_hsen) ld.store(t.avg_hsen, aH);
        if (t.avg_rbbr) ld.store(t.avg_rbbr, aR);
        if (t.avg_rsdr) ld.store(t.avg_rsdr, aS);
    }
    if (DIAG) {
        if (t.avg_qsur) DIAG_COMMIT(0, DQ_QSUR_T, aQ);
        if (t.avg_meva) DIAG_COMMIT(0, DQ_MEVA, aM);
        if (t.avg_hlat) DIAG_COMMIT(0, DQ_HLAT, aL);
        if (t.avg_hsen) DIAG_COMMIT(0, DQ_HSEN, aH);
        if (t.avg_rbbr) DIAG_COMMIT(0, DQ_RBBR, aR);
        if (t.avg_rsdr) DIAG_COMMIT(0, DQ_RSDR, aS);
    }
    return bad;
}

// ---------------------------------------------------------------------------------------------
// u / v grid
// ---------------------------------------------------------------------------------------------
struct UVIn {
    V2 fice_, psur_, tsur_, amom_, uatm_, vatm_, qsur_in_;
    __device__ __forceinline__ const V2 &fice() const { return fice_; }
    __device__ __forceinline__ const V2 &psur() const { return psur_; }
    __device__ __forceinline__ const V2 &tsur() const { return tsur_; }
    __device__ __forceinline__ const V2 &amom() const { return amom_; }
    __device__ __forceinline__ const V2 &uatm() const { return uatm_; }
    __device__ __forceinline__ const V2 &vatm() const { return vatm_; }
    __device__ __forceinline__ const V2 &qsur_in() const { return qsur_in_; }
};
struct UVOut {
    V2 qsur, mom;
};

template <class M, class IN>
__device__ __forceinline__ bool uv_type_math(const FusedPlan &p, const FusedUVType &ty, const IN &in, int north, UVOut &o)
{
    M m;
    const Consts &c = p.c;
    // --- QSUR on this grid (calculate.F90:25-50, called for grids 2 and 3)
    if (ty.m_qsur == M_CCLM) o.qsur = spec_vapor_surface_cclm(m, in.fice(), in.psur(), in.tsur(), c);
    else if (ty.qsur_in) o.qsur = in.qsur_in();
    // --- momentum: calc_flux_momentum_east / _north (calculate.F90:212-316)
    if (ty.m_mom != M_NONE) {
        if (ty.m_mom == M_ZERO) {
            o.mom = vzero();
        } else {
            const V2 vel = wind_speed(m, in.uatm(), in.vatm());
            const V2 fa = (ty.m_mom == M_RCO) ? momentum_flux_air_rco<M>(vel)
                                              : momentum_flux_air_cclm(m, in.amom(), in.psur(), o.qsur, in.tsur(), vel, c);
            o.mom = momentum_component<M>(fa, north ? in.vatm() : in.uatm());
        }
    }
    return m.bad();
}

template <class M, int SS, int DIAG, class LD>
__device__ __forceinline__ bool uv_chain(const FusedPlan &p, const FusedUV &g, int which, const LD &ld, int nv, DiagCtx &dg)
{
    const int S = SS ? SS : p.S;
    bool bad = false;
    Cached<LD> cPSUR, cUATM, cVATM, cAMOM, cFICE, cTSUR;
    UVIn in;
    V2 area;
    if (DIAG) area = ld.load(g.area);
    V2 aQ = vzero(), aM = vzero();

    auto per_type = [&](const int i) {
        const FusedUVType &ty = g.ty[i];
        V2 fare;
        UVOut o;
        if (LD::kFull || nv) {
            if (ty.fare) fare = ld.load(ty.fare);
            in.fice_ = cFICE.get(ld, ty.fice);
            in.psur_ = cPSUR.get(ld, ty.psur);
            in.tsur_ = cTSUR.get(ld, ty.tsur);
            in.uatm_ = cUATM.get(ld, ty.uatm);
            in.vatm_ = cVATM.get(ld, ty.vatm);
            in.amom_ = cAMOM.get(ld, ty.a_mom);
            if (ty.qsur_in) in.qsur_in_ = ld.load(ty.qsur_in);
            bad |= uv_type_math<M>(p, ty, in, g.north, o);
            if (ty.m_qsur == M_CCLM) ld.store(ty.qsur, o.qsur);
            if (ty.m_mom != M_NONE) ld.store(ty.mom, o.mom);
            if (g.avg_qsur) avg_acc(aQ, o.qsur, fare);
            if (g.avg_mom) avg_acc(aM, o.mom, fare);
        }
        if (DIAG) {
            const int base = (i + 1) * DQ_COUNT;
            if (which == 1) {
                if (ty.m_qsur == M_CCLM) DIAG_COMMIT(base, DQ_QSUR_U, o.qsur);
                if (ty.m_mom != M_NONE) DIAG_COMMIT(base, DQ_UMOM, o.mom);
            } else {
                if (ty.m_qsur == M_CCLM) DIAG_COMMIT(base, DQ_QSUR_V, o.qsur);
                if (ty.m_mom != M_NONE) DIAG_COMMIT(base, DQ_VMOM, o.mom);
            }
        }
    };
    if constexpr (SS > 0) {
#pragma unroll
        for (int i = 0; i < SS; ++i) per_type(i);
    } else {
#pragma unroll 1
        for (int i = 0; i < S; ++i) per_type(i);
    }
    if (LD::kFull || nv) {
        if (g.avg_qsur) ld.store(g.avg_qsur, aQ);
        if (g.avg_mom) ld.store(g.avg_mom, aM);
    }
    if (DIAG) {
        if (which == 1) {
            if (g.avg_qsur) DIAG_COMMIT(0, DQ_QSUR_U, aQ);
            if (g.avg_mom) DIAG_COMMIT(0, DQ_UMOM, aM);
        } else {
            if (g.avg_qsur) DIAG_COMMIT(0, DQ_QSUR_V, aQ);
            if (g.avg_mom) DIAG_COMMIT(0, DQ_VMOM, aM);
        }
    }
    return bad;
}

// cold, out of line: every lane of the warp that called recomputes its V cells with the IEEE policy (identical bits for the
// lanes whose operands were in range: ExactVec's exp / pow fall back to the lock-step sequences there) and, with
// diagnostics, the warp's row is rebuilt by the same trees.  Scalars only: nothing of the hot path's state is passed.
template <int SS, int DIAG, bool FULL>
__device__ __noinline__ void fused_cold_warp(const FusedPlan &p, int which, int64_t j, int nv, int64_t row)
{
    atomicAdd(&g_exact_calls, 1ull);
    DiagCtx dg;
    if (DIAG) {
        dg.base = p.diag_partials;
        dg.rows = p.diag_rows;
        dg.plane = (int64_t)p.diag_n * p.diag_rows;
        dg.row = row;
    }
    if (FULL) {
        const LdGlobal ld{j};
        if (which == 0) t_chain<Exact, SS, DIAG>(p, ld, V, dg);
        else uv_chain<Exact, SS, DIAG>(p, p.uv[which - 1], which, ld, V, dg);
    } else {
        const LdGuard ld{j, nv};
        if (which == 0) t_chain<Exact, SS, DIAG>(p, ld, nv, dg);
        else uv_chain<Exact, SS, DIAG>(p, p.uv[which - 1], which, ld, nv, dg);
    }
}

template <int SS, int DIAG, bool FULL>
__global__ void __launch_bounds__(kFusedThreads, kFusedMinBlocks)
fused_step_kernel(const __grid_constant__ FusedPlan p, const __grid_constant__ LaunchGeom geo)
{
    const int b = blockIdx.x;
    const int which = (b < geo.nb_t) ? 0 : (b < geo.nb_t + geo.nb_u ? 1 : 2);
    const int blk = (which == 0) ? b : (which == 1 ? b - geo.nb_t : b - geo.nb_t - geo.nb_u);
    const int64_t end = geo.first[which] + geo.count[which];
    const int64_t j = geo.first[which] + ((int64_t)blk * kFusedThreads + threadIdx.x) * V;
    const int nv = (j >= end) ? 0 : (end - j >= V ? V : (int)(end - j));
    DiagCtx dg;
    if (DIAG) {
        dg.base = p.diag_partials;
        dg.rows = p.diag_rows;
        dg.plane = (int64_t)p.diag_n * p.diag_rows;
        dg.row = geo.row0 + (int64_t)b * (kFusedThreads / 32) + (threadIdx.x >> 5);
    }
    bool bad;
    if (FULL) {        // whole 512-cell blocks only: every thread owns V valid cells
        const LdGlobal ld{j};
        if (which == 0) bad = t_chain<Fast, SS, DIAG>(p, ld, V, dg);
        else bad = uv_chain<Fast, SS, DIAG>(p, p.uv[which - 1], which, ld, V, dg);
    } else {
        if (!DIAG && nv == 0) return;      // with DIAG even empty threads take part in the warp reductions
        const LdGuard ld{j, nv};
        if (which == 0) bad = t_chain<Fast, SS, DIAG>(p, ld, nv, dg);
        else bad = uv_chain<Fast, SS, DIAG>(p, p.uv[which - 1], which, ld, nv, dg);
        bad = bad && nv > 0;
    }
    // an operand of some lane left the proven range (never with physical data): the warp redoes its cells with the IEEE
    // routines -- same chain, same order, from global memory -- and overwrites its outputs and its diagnostics row
    if (__any_sync(__activemask(), bad)) fused_cold_warp<SS, DIAG, FULL>(p, which, j, nv, DIAG ? dg.row : 0);
}

// diagnostics reduction, deterministic (fixed tree, independent of scheduling):
//   stage 1: grid (chunks, slots): CTA sums kDiagChunk warp rows of one slot -> tmp[plane][slot][chunk]
//   stage 2: grid (slots): sums the chunks -> out[slot][3] (sum, min, max)
constexpr int kDiagChunk = 4096;

struct DiagRanges {
    int64_t row_begin[3], row_end[3];     // main-launch rows of the t / u / v blocks
    int64_t tail_begin[3], tail_end[3];   // tail-launch rows
    signed char grid_of_slot[kDiagSlots]; // compact slot -> 0/1/2
};

__device__ __forceinline__ void block_combine(double &s, double &mn, double &mx, int planes)
{
    __shared__ double sh[3][256];
    sh[0][threadIdx.x] = s;
    sh[1][threadIdx.x] = mn;
    sh[2][threadIdx.x] = mx;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
            sh[0][threadIdx.x] = add(sh[0][threadIdx.x], sh[0][threadIdx.x + w]);
            if (planes > 1) {
                sh[1][threadIdx.x] = fmin(sh[1][threadIdx.x], sh[1][threadIdx.x + w]);
                sh[2][threadIdx.x] = fmax(sh[2][threadIdx.x], sh[2][threadIdx.x + w]);
            }
        }
        __syncthreads();
    }
    s = sh[0][0];
    mn = sh[1][0];
    mx = sh[2][0];
}

__global__ void __launch_bounds__(256)
diag_reduce_rows_kernel(const double *__restrict__ part, int64_t rows, int nslots, int planes,
                        const __grid_constant__ DiagRanges R, double *__restrict__ tmp, int nchunks)
{
    const int slot = blockIdx.y, chunk = blockIdx.x;
    const int g = R.grid_of_slot[slot];
    const int64_t plane = (int64_t)nslots * rows;
    const double *col = part + (int64_t)slot * rows;
    double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
    constexpr int per = kDiagChunk / 256;
    const int64_t r0 = (int64_t)chunk * kDiagChunk + threadIdx.x * per;
#pragma unroll 4
    for (int k = 0; k < per; ++k) {
        const int64_t r = r0 + k;
        const bool in = (r >= R.row_begin[g] && r < R.row_end[g]) || (r >= R.tail_begin[g] && r < R.tail_end[g]);
        if (in) {
            s = add(s, col[r]);
            if (planes > 1) {
                mn = fmin(mn, col[plane + r]);
                mx = fmax(mx, col[2 * plane + r]);
            }
        }
    }
    block_combine(s, mn, mx, planes);
    if (threadIdx.x == 0) {
        double *o = tmp + ((int64_t)slot * nchunks + chunk) * 3;
        o[0] = s;
        o[1] = mn;
        o[2] = mx;
    }
}

__global__ void __launch_bounds__(256)
diag_reduce_final_kernel(const double *__restrict__ tmp, int nchunks, int planes, double *__restrict__ out,
                         const __grid_constant__ DiagHist hist)
{
    const int slot = blockIdx.x;
    double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
    const int per = (nchunks + 255) / 256;
    for (int k = 0; k < per; ++k) {
        const int c = threadIdx.x * per + k;
        if (c < nchunks) {
            const double *q = tmp + ((int64_t)slot * nchunks + c) * 3;
            s = add(s, q[0]);
            mn = fmin(mn, q[1]);
            mx = fmax(mx, q[2]);
        }
    }
    block_combine(s, mn, mx, planes);
    if (threadIdx.x == 0) {      // plane-major [sum | min | max][kDiagSlots]: each plane is one NCCL all-reduce
        out[0 * kDiagSlots + slot] = s;
        out[1 * kDiagSlots + slot] = mn;
        out[2 * kDiagSlots + slot] = mx;
        if (hist.ring) {
            double *h = diag_hist_row(hist);
            h[0 * kDiagSlots + slot] = s;
            h[1 * kDiagSlots + slot] = mn;
            h[2 * kDiagSlots + slot] = mx;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// op-list interpreter: one cell per thread, ops in the reference's order, every op reads and
// writes global memory (a thread always observes its own earlier writes), so aliased arrays
// behave exactly like the Fortran pointer aliases.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) oplist_kernel(const __grid_constant__ OpList L, const __grid_constant__ Consts c,
                                                     int64_t n)
{
    using M = ExactScalar;
    M m;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        for (int o = 0; o < L.n; ++o) {
            const Op &op = L.ops[o];
            switch (op.code) {
                case OP_ZERO: op.out[j] = 0.0; break;
                case OP_COPY: op.out[j] = op.in[0][j]; break;
                case OP_QSUR_CCLM:
                    op.out[j] = spec_vapor_surface_cclm(m, op.in[0][j], op.in[1][j], op.in[2][j], c);
                    break;
                case OP_MEVA_CCLM:
                    op.out[j] = flux_mass_evap_cclm(m, op.in[0][j], op.in[1][j], op.in[2][j], op.in[3][j], op.in[4][j],
                                                    wind_speed(m, op.in[5][j], op.in[6][j]), c);
                    break;
                case OP_MEVA_RCO:
                    op.out[j] = flux_mass_evap_rco(m, op.in[0][j], op.in[1][j], wind_speed(m, op.in[2][j], op.in[3][j]));
                    break;
                case OP_ADD: op.out[j] = add(op.out[j], op.in[0][j]); break;
                case OP_SCALE: op.out[j] = mul(op.in[0][j], op.cst); break;
                case OP_HSEN_CCLM:
                    op.out[j] = flux_heat_sensible_cclm(m, op.in[0][j], op.in[1][j], op.in[2][j], op.in[3][j], op.in[4][j],
                                                        op.in[5][j], wind_speed(m, op.in[6][j], op.in[7][j]), c);
                    break;
                case OP_HSEN_RCO:
                    op.out[j] = flux_heat_sensible_rco<M>(op.in[0][j], op.in[1][j], wind_speed(m, op.in[2][j], op.in[3][j]));
                    break;
                case OP_MOM_CCLM: {
                    const double u = op.in[4][j], v = op.in[5][j];
                    const double fa = momentum_flux_air_cclm(m, op.in[0][j], op.in[1][j], op.in[2][j], op.in[3][j],
                                                             wind_speed(m, u, v), c);
                    if (op.out) op.out[j] = momentum_component<M>(fa, u);
                    if (op.out2) op.out2[j] = momentum_component<M>(fa, v);
                    break;
                }
                case OP_MOM_RCO: {
                    const double u = op.in[0][j], v = op.in[1][j];
                    const double fa = momentum_flux_air_rco<M>(wind_speed(m, u, v));
                    if (op.out) op.out[j] = momentum_component<M>(fa, u);
                    if (op.out2) op.out2[j] = momentum_component<M>(fa, v);
                    break;
                }
                case OP_RBBR: op.out[j] = flux_radiation_blackbody_StBo<M>(op.in[0][j], op.cst); break;
                case OP_MULADD: op.out[j] = add(op.out[j], mul(op.in[0][j], op.in[1][j])); break;
                default: break;
            }
        }
    }
}

// corrections(1,12,n) Fortran order (month fastest) -> [12][n] month-major (bias_corrections.F90:29-30,191)
// corrections(1,12,n) (month fastest) -> [12][stride] (stride >= n: every month slab starts 16-byte aligned)
__global__ void transpose_corrections_kernel(const double *__restrict__ src, double *__restrict__ dst, int64_t n, int64_t stride)
{
    __shared__ double tile[12][65];
    const int64_t j0 = (int64_t)blockIdx.x * 64;
    for (int e = threadIdx.x; e < 12 * 64; e += blockDim.x) {
        const int64_t g = j0 * 12 + e;   // contiguous read
        if (g < n * 12) tile[e % 12][e / 12] = src[g];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 12 * 64; e += blockDim.x) {
        const int m = e / 64, jj = e % 64;
        if (j0 + jj < n) dst[(int64_t)m * stride + j0 + jj] = tile[m][jj];
    }
}

// do_regridding (basic.F90:476-486) with the COO elements grouped by destination (stable), one thread
// per destination cell, accumulation in the reference's element order: acc = acc + src*w
__global__ void regrid_csr_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ src_idx,
                                  const double *__restrict__ weight, const double *__restrict__ src,
                                  double *__restrict__ dst, int64_t n_dst)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_dst) return;
    double acc = 0.0;
    for (int64_t k = row_ptr[r]; k < row_ptr[r + 1]; ++k) acc = add(acc, mul(src[src_idx[k]], weight[k]));
    dst[r] = acc;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
static bool plan_aligned(const FusedPlan &p, const int64_t first[3])
{
    auto ok = [](const void *q, int64_t cell0) { return q == nullptr || ((reinterpret_cast<uintptr_t>(q) + cell0 * 8) & 15) == 0; };
    bool a = true;
    const FusedT &t = p.t;
    const int64_t c0 = first[0];
    a = a && ok(t.rsdd, c0) && ok(t.bias, c0) && ok(t.area, c0) && ok(t.avg_qsur, c0) && ok(t.avg_meva, c0) &&
        ok(t.avg_hlat, c0) && ok(t.avg_hsen, c0) && ok(t.avg_rbbr, c0) && ok(t.avg_rsdr, c0);
    for (int i = 0; i < p.S; ++i) {
        const FusedTType &y = t.ty[i];
        const void *ps[] = {y.fice, y.psur, y.tsur, y.qatm, y.tatm, y.patm, y.uatm, y.vatm, y.a_evap, y.a_sens,
                            y.qsur_in, y.fare, y.qsur, y.meva, y.hlat, y.hsen, y.rbbr, y.rsdr};
        for (const void *q : ps) a = a && ok(q, c0);
    }
    for (int g = 0; g < 2; ++g) {
        const FusedUV &u = p.uv[g];
        const int64_t cg = first[g + 1];
        a = a && ok(u.area, cg) && ok(u.avg_qsur, cg) && ok(u.avg_mom, cg);
        for (int i = 0; i < p.S; ++i) {
            const FusedUVType &y = u.ty[i];
            const void *ps[] = {y.fice, y.psur, y.tsur, y.a_mom, y.uatm, y.vatm, y.qsur_in, y.fare, y.qsur, y.mom};
            for (const void *q : ps) a = a && ok(q, cg);
        }
    }
    return a;
}

// The one place that decides how plan p is launched over cells[g] cells from first[g] on: whole 512-cell blocks through
// the 128-bit kernel (specialised persistent kernel or generic direct-load kernel), the ragged remainder (or everything,
// if an array is misaligned) through the guarded kernel.  The bias slab's alignment is part of the decision; it holds for
// every month, because corr_stride keeps each month slab 16-byte aligned.
FusedLaunch resolve_fused(const FusedPlan &p, const int64_t first[3], const int64_t cells_in[3], int staged, int dyn_min_tiles)
{
    FusedLaunch L;
    memset(&L, 0, sizeof L);
    const bool al = plan_aligned(p, first);
    int nbm[3], nbt[3];
    for (int g = 0; g < 3; ++g) {
        const bool active = (g == 0) ? (p.do_early || p.do_normal) : (p.do_normal != 0);
        const int64_t cells = active ? cells_in[g] : 0;
        const int64_t whole = al ? (cells / kFusedCellsPerBlock) : 0;
        nbm[g] = (int)whole;
        L.main.first[g] = first[g];
        L.main.count[g] = whole * kFusedCellsPerBlock;
        L.tail.first[g] = first[g] + whole * kFusedCellsPerBlock;
        L.tail.count[g] = cells - whole * kFusedCellsPerBlock;
        nbt[g] = (int)((L.tail.count[g] + kFusedCellsPerBlock - 1) / kFusedCellsPerBlock);
    }
    L.main.nb_t = nbm[0];
    L.main.nb_u = nbm[1];
    L.nb_main = nbm[0] + nbm[1] + nbm[2];
    L.tail.nb_t = nbt[0];
    L.tail.nb_u = nbt[1];
    L.nb_tail = nbt[0] + nbt[1] + nbt[2];
    L.main.row0 = 0;
    L.tail.row0 = (int64_t)L.nb_main * (kFusedThreads / 32);
    L.diag_rows = L.tail.row0 + (int64_t)L.nb_tail * (kFusedThreads / 32);
    // specialised persistent kernel for the canonical plans with one or two surface types, whatever the grid size (20 000 cells:
    // 6 us per step against 20 us on the generic kernels); it takes the ragged remainder along: one launch, one diagnostics
    // row per CTA
    if (al && p.S <= 2 && staged >= 1 && L.nb_main + L.nb_tail > 0) {
        int64_t spec_cells[3];
        for (int g = 0; g < 3; ++g) spec_cells[g] = L.main.count[g] + L.tail.count[g];
        if (spec_resolve(p, L.main.first, spec_cells, dyn_min_tiles, L)) {
            L.spec = true;
            L.diag_rows = L.spec_grid;
            L.fills = L.spec_grid >= spec_capacity(p.S);
        }
    }
    return L;
}

template <int SS, int DIAG>
static void launch_fused_t(const FusedPlan &p, const FusedLaunch &L, cudaStream_t stream, int *launches)
{
    if (L.nb_tail) {
        fused_step_kernel<SS, DIAG, false><<<L.nb_tail, kFusedThreads, 0, stream>>>(p, L.tail);
        if (launches) *launches += 1;
    }
    if (L.nb_main) {
        fused_step_kernel<SS, DIAG, true><<<L.nb_main, kFusedThreads, 0, stream>>>(p, L.main);
        if (launches) *launches += 1;
    }
}

template <int SS>
static void launch_fused_s(const FusedPlan &p, const FusedLaunch &L, cudaStream_t stream, int *launches)
{
    if (p.diag >= 2) launch_fused_t<SS, 2>(p, L, stream, launches);
    else if (p.diag == 1) launch_fused_t<SS, 1>(p, L, stream, launches);
    else launch_fused_t<SS, 0>(p, L, stream, launches);
}

// one launch of a resolved plan: its parameter block with this step's fields filled in
int launch_fused(const FusedPlan &plan, const FusedLaunch &L, const FusedStepArgs &a, cudaStream_t stream, int *launches)
{
    if (L.spec) {
        SpecPlan sp = L.sp;
        if (sp.has_bias) sp.src[0][kSpecBiasSlot] = a.bias;
        sp.partials = a.diag_partials;
        sp.rows = a.diag_rows;
        sp.plane = (int64_t)plan.diag_n * a.diag_rows;
        sp.prev = a.fold_prev;
        sp.early_loads = a.early_loads;
        sp.chain = sp.dyn ? 0 : a.chain;
        sp.seq = a.chain_seq;
        sp.done = a.chain_done;
        sp.tile_base = a.tile_base;
        sp.tile_counter = a.tile_counter;
        if (const int e = spec_launch(sp, L.spec_set, L.spec_grid, stream)) return e;
        if (launches) *launches += 1;
        return (int)cudaGetLastError();
    }
    if (L.nb_main + L.nb_tail == 0) return 0;
    FusedPlan p = plan;
    if (p.t.bias) p.t.bias = a.bias;
    p.diag_partials = a.diag_partials;
    p.diag_rows = a.diag_rows;
    switch (p.S) {
        case 1: launch_fused_s<1>(p, L, stream, launches); break;
        case 2: launch_fused_s<2>(p, L, stream, launches); break;
        default: launch_fused_s<0>(p, L, stream, launches); break;
    }
    return (int)cudaGetLastError();
}

// partials written by a generic launch of a resolved plan -> a.diag_out[compact slot][3] (a specialised launch leaves one row
// per CTA, folded later: DiagFold)
int launch_diag_finalize(const FusedPlan &p, const FusedLaunch &L, const FusedStepArgs &a, double *tmp, cudaStream_t stream, int *launches)
{
    if (!p.diag || p.diag_n <= 0) return 0;
    const int w = kFusedThreads / 32;
    DiagRanges R;
    memset(&R, 0, sizeof R);
    const int nbm[3] = {L.main.nb_t, L.main.nb_u, L.nb_main - L.main.nb_t - L.main.nb_u};
    const int nbt[3] = {L.tail.nb_t, L.tail.nb_u, L.nb_tail - L.tail.nb_t - L.tail.nb_u};
    int64_t rm = 0, rt = L.tail.row0;
    for (int g = 0; g < 3; ++g) {
        R.row_begin[g] = rm;
        rm += (int64_t)nbm[g] * w;
        R.row_end[g] = rm;
        R.tail_begin[g] = rt;
        rt += (int64_t)nbt[g] * w;
        R.tail_end[g] = rt;
    }
    for (int s = 0; s < kDiagSlots; ++s) {
        const int q = s % DQ_COUNT;
        const int g = (q == DQ_QSUR_U || q == DQ_UMOM) ? 1 : ((q == DQ_QSUR_V || q == DQ_VMOM) ? 2 : 0);
        if (p.diag_map[s] >= 0 && p.diag_map[s] < kDiagSlots) R.grid_of_slot[p.diag_map[s]] = (signed char)g;
    }
    const int64_t rows = a.diag_rows;
    const int nchunks = (int)((rows + kDiagChunk - 1) / kDiagChunk);
    const int planes = p.diag >= 2 ? 3 : 1;
    diag_reduce_rows_kernel<<<dim3(nchunks, p.diag_n), 256, 0, stream>>>(a.diag_partials, rows, p.diag_n, planes, R, tmp, nchunks);
    diag_reduce_final_kernel<<<p.diag_n, 256, 0, stream>>>(tmp, nchunks, planes, a.diag_out, a.hist);
    if (launches) *launches += 2;
    return (int)cudaGetLastError();
}

// result vectors [sum|min|max][kDiagSlots] of the chunks of one step -> one vector, in chunk order
__global__ void diag_combine_kernel(const double *__restrict__ chunk_out, int nchunks, double *__restrict__ out,
                                    const __grid_constant__ DiagHist hist)
{
    const int t = threadIdx.x;
    if (t >= kDiagSlots) return;
    double s = 0.0, mn = DBL_MAX, mx = -DBL_MAX;
    for (int k = 0; k < nchunks; ++k) {
        const double *q = chunk_out + (size_t)k * 3 * kDiagSlots;
        s = add(s, q[t]);
        mn = fmin(mn, q[kDiagSlots + t]);
        mx = fmax(mx, q[2 * kDiagSlots + t]);
    }
    out[t] = s;
    out[kDiagSlots + t] = mn;
    out[2 * kDiagSlots + t] = mx;
    if (hist.ring) {
        double *h = diag_hist_row(hist);
        h[t] = s;
        h[kDiagSlots + t] = mn;
        h[2 * kDiagSlots + t] = mx;
    }
}

// peer exchange of a finished result vector (generic kernel / chunked host pipeline; the specialised kernel does it itself)
__global__ void diag_post_kernel(const double *__restrict__ diag_out, const __grid_constant__ PeerPost post, int n_active)
{
    const int t = threadIdx.x;
    if (t >= n_active) return;
    unsigned long long w[3][2];
    for (int pl = 0; pl < 3; ++pl) diag_mail_pack(diag_out[pl * kDiagSlots + t], (unsigned int)post.seq, w[pl]);
    for (int r = 0; r < post.nranks; ++r) {
        DiagMail *m = post.mail[r] + (size_t)post.slot * post.nranks + post.rank;
        for (int pl = 0; pl < 3; ++pl) {
            __stcg(&m->w[pl][t][0], w[pl][0]);
            __stcg(&m->w[pl][t][1], w[pl][1]);
        }
    }
}

int launch_diag_post(const double *diag_out, const PeerPost &post, int n_active, cudaStream_t stream)
{
    diag_post_kernel<<<1, 128, 0, stream>>>(diag_out, post, n_active);
    return (int)cudaGetLastError();
}

int launch_diag_combine(const double *chunk_out, int nchunks, double *diag_out, const DiagHist &hist, cudaStream_t stream)
{
    diag_combine_kernel<<<1, 128, 0, stream>>>(chunk_out, nchunks, diag_out, hist);
    return (int)cudaGetLastError();
}

// number of the first step of the graph that is replayed next (DiagHist::base), in stream order before the replay
__global__ void diag_hist_base_kernel(int64_t *word, int64_t base) { *word = base; }

int launch_diag_hist_base(int64_t *word, int64_t base, cudaStream_t stream)
{
    diag_hist_base_kernel<<<1, 1, 0, stream>>>(word, base);
    return (int)cudaGetLastError();
}

int diag_tmp_doubles(int64_t rows, int nslots) { return (int)(((rows + kDiagChunk - 1) / kDiagChunk) * nslots * 3); }

int launch_oplist(const OpList &ops, const Consts &c, int64_t n, cudaStream_t stream)
{
    if (n <= 0 || ops.n == 0) return 0;
    int64_t nb = (n + 255) / 256;
    if (nb > 148 * 64) nb = 148 * 64;
    oplist_kernel<<<(int)nb, 256, 0, stream>>>(ops, c, n);
    return (int)cudaGetLastError();
}

int launch_transpose_corrections(const double *src, double *dst, int64_t n, int64_t stride, cudaStream_t stream)
{
    if (n <= 0) return 0;
    transpose_corrections_kernel<<<(int)((n + 63) / 64), 256, 0, stream>>>(src, dst, n, stride);
    return (int)cudaGetLastError();
}

int launch_regrid_csr(const int64_t *row_ptr, const int32_t *src_idx, const double *weight, const double *src,
                      double *dst, int64_t n_dst, cudaStream_t stream)
{
    if (n_dst <= 0) return 0;
    regrid_csr_kernel<<<(int)((n_dst + 255) / 256), 256, 0, stream>>>(row_ptr, src_idx, weight, src, dst, n_dst);
    return (int)cudaGetLastError();
}

}  // namespace fc
