// vmath_probe.cu -- test-only entry points into the arithmetic policies of csrc/vmath.cuh.
//
// tests/test_gpu_vmath.py compiles this file into a temporary directory and loads it with ctypes.  It adds no
// arithmetic of its own: every result comes from a policy of vmath.cuh, or, in the on-device sweeps, from CUDA's
// IEEE __ddiv_rn / __dsqrt_rn, whose correctly rounded answer is unique.
//
//   vp_run    one operation (div, sqrt, exp, log, powc) under one policy over n operands, host arrays in and out;
//             the per-thread bad() flag is written to every cell of that thread
//   vp_sweep  FastVec<2>::div / ::sqrt against __ddiv_rn / __dsqrt_rn on operands drawn from a counter hash,
//             exponents uniform in [-500, 499]; returns the mismatch count and the first mismatching operands
#include <stdint.h>

#include "vmath.cuh"

using namespace fc;

enum { OP_DIV = 0, OP_SQRT = 1, OP_EXP = 2, OP_LOG = 3, OP_POWC = 4 };
enum { POL_FAST1 = 0, POL_FAST2 = 1, POL_EXACTVEC2 = 2, POL_EXACTSCALAR = 3 };

// ExactScalar in the shape of the vector policies (one cell per thread, no flag)
struct ScalarAsVec {
    using T = Vd<1>;
    ExactScalar s;
    __device__ T div(const T &a, const T &b) { T r; r.v[0] = s.div(a.v[0], b.v[0]); return r; }
    __device__ T sqrt(const T &a) { T r; r.v[0] = s.sqrt(a.v[0]); return r; }
    __device__ T exp(const T &a) { T r; r.v[0] = s.exp(a.v[0]); return r; }
    __device__ T powc(const T &a, double c) { T r; r.v[0] = s.powc(a.v[0], c); return r; }
    __device__ bool bad() const { return false; }
};

template <int OP, class P, int V>
__global__ void vp_kernel(const double *x, const double *y, double c, double *out, unsigned char *bad, int64_t n)
{
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * V;
    if (i0 >= n) return;
    Vd<V> a, b;
#pragma unroll
    for (int k = 0; k < V; ++k) {      // a ragged last thread fills its spare lanes with 1.0, inside every range
        a.v[k] = i0 + k < n ? x[i0 + k] : 1.0;
        b.v[k] = i0 + k < n ? y[i0 + k] : 1.0;
    }
    P p;
    Vd<V> r;
    if constexpr (OP == OP_DIV) r = p.div(a, b);
    else if constexpr (OP == OP_SQRT) r = p.sqrt(a);
    else if constexpr (OP == OP_EXP) r = p.exp(a);
    else if constexpr (OP == OP_LOG) r = p.log(a);
    else r = p.powc(a, c);
    const unsigned char f = p.bad() ? 1 : 0;
#pragma unroll
    for (int k = 0; k < V; ++k)
        if (i0 + k < n) {
            out[i0 + k] = r.v[k];
            bad[i0 + k] = f;
        }
}

template <int OP, class P, int V>
static cudaError_t launch(const double *x, const double *y, double c, double *out, unsigned char *bad, int64_t n)
{
    const int64_t threads = (n + V - 1) / V;
    vp_kernel<OP, P, V><<<(unsigned)((threads + 255) / 256), 256>>>(x, y, c, out, bad, n);
    return cudaGetLastError();
}

template <int OP>
static cudaError_t launch_policy(int policy, const double *x, const double *y, double c, double *out, unsigned char *bad,
                                 int64_t n)
{
    switch (policy) {
    case POL_FAST1: return launch<OP, FastVec<1>, 1>(x, y, c, out, bad, n);
    case POL_FAST2: return launch<OP, FastVec<2>, 2>(x, y, c, out, bad, n);
    case POL_EXACTVEC2:
        if constexpr (OP != OP_LOG) return launch<OP, ExactVec<2>, 2>(x, y, c, out, bad, n);
        break;
    case POL_EXACTSCALAR:
        if constexpr (OP != OP_LOG) return launch<OP, ScalarAsVec, 1>(x, y, c, out, bad, n);
        break;
    }
    return cudaErrorInvalidValue;      // log exists in FastVec only; unknown policy
}

// Frees whatever was allocated, on every return path.
struct DevBuffers {
    void *p[4] = {nullptr, nullptr, nullptr, nullptr};
    ~DevBuffers()
    {
        for (void *q : p)
            if (q) cudaFree(q);
    }
};

// Returns a cudaError_t value (0 = success); out and bad are written only on success.
extern "C" int vp_run(int op, int policy, const double *x, const double *y, double c, double *out, unsigned char *bad,
                      int64_t n)
{
    if (n <= 0 || op < OP_DIV || op > OP_POWC) return (int)cudaErrorInvalidValue;
    DevBuffers d;
    const size_t bytes = (size_t)n * sizeof(double);
    cudaError_t e;
    for (int i = 0; i < 3; ++i)
        if ((e = cudaMalloc(&d.p[i], bytes)) != cudaSuccess) return (int)e;
    if ((e = cudaMalloc(&d.p[3], (size_t)n)) != cudaSuccess) return (int)e;
    double *dx = (double *)d.p[0], *dy = (double *)d.p[1], *dout = (double *)d.p[2];
    unsigned char *dbad = (unsigned char *)d.p[3];
    if ((e = cudaMemcpy(dx, x, bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(dy, y, bytes, cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    switch (op) {
    case OP_DIV: e = launch_policy<OP_DIV>(policy, dx, dy, c, dout, dbad, n); break;
    case OP_SQRT: e = launch_policy<OP_SQRT>(policy, dx, dy, c, dout, dbad, n); break;
    case OP_EXP: e = launch_policy<OP_EXP>(policy, dx, dy, c, dout, dbad, n); break;
    case OP_LOG: e = launch_policy<OP_LOG>(policy, dx, dy, c, dout, dbad, n); break;
    default: e = launch_policy<OP_POWC>(policy, dx, dy, c, dout, dbad, n); break;
    }
    if (e != cudaSuccess) return (int)e;
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(out, dout, bytes, cudaMemcpyDeviceToHost)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(bad, dbad, (size_t)n, cudaMemcpyDeviceToHost)) != cudaSuccess) return (int)e;
    return (int)cudaSuccess;
}

// ---------------------------------------------------------------------------------------------
// On-device sweeps
static constexpr int kSweepKeep = 8;   // mismatching operands returned (a, b pairs)

__device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// operand number i of the stream `seed`: random mantissa, exponent uniform in [-500, 499], random sign if `sign`
__device__ __forceinline__ double sweep_operand(uint64_t seed, uint64_t i, bool sign)
{
    const uint64_t h = splitmix64(seed ^ splitmix64(i));
    const uint64_t g = splitmix64(h);
    const uint64_t e = (uint64_t)(1023 - 500) + (g >> 32) % 1000u;
    const uint64_t s = sign ? (g & 1u) << 63 : 0u;
    return __longlong_as_double((long long)(s | (e << 52) | (h & 0x000fffffffffffffull)));
}

__device__ __forceinline__ void sweep_note(unsigned long long *count, double *keep, double a, double b)
{
    const unsigned long long slot = atomicAdd(count, 1ull);
    if (slot < (unsigned long long)kSweepKeep) {
        keep[2 * slot] = a;
        keep[2 * slot + 1] = b;
    }
}

template <int OP>
__global__ void vp_sweep_kernel(uint64_t seed, uint64_t pairs, unsigned long long *count, double *keep)
{
    // each thread evaluates two operands per iteration in lock step, as the production kernels do
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; 2 * t < pairs; t += stride) {
        Vd<2> a, b, q;
        FastVec<2> m;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            a.v[k] = sweep_operand(seed, 2 * (2 * t + k), OP == OP_DIV);
            b.v[k] = sweep_operand(seed, 2 * (2 * t + k) + 1, true);
        }
        if constexpr (OP == OP_DIV) q = m.div(a, b);
        else q = m.sqrt(a);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const double ref = OP == OP_DIV ? __ddiv_rn(a.v[k], b.v[k]) : __dsqrt_rn(a.v[k]);
            if (m.bad() || __double_as_longlong(q.v[k]) != __double_as_longlong(ref))
                sweep_note(count, keep, a.v[k], OP == OP_DIV ? b.v[k] : 0.0);
        }
    }
}

// op: OP_DIV or OP_SQRT; evaluates `count` operands (rounded up to even).  *mismatches gets the number of results that
// differ from the IEEE routine or whose thread was flagged; keep[0 .. 2*kSweepKeep) the first (a, b) pairs of those.
extern "C" int vp_sweep(int op, uint64_t seed, uint64_t count, unsigned long long *mismatches, double *keep)
{
    if (op != OP_DIV && op != OP_SQRT) return (int)cudaErrorInvalidValue;
    DevBuffers d;
    cudaError_t e;
    if ((e = cudaMalloc(&d.p[0], sizeof(unsigned long long))) != cudaSuccess) return (int)e;
    if ((e = cudaMalloc(&d.p[1], 2 * kSweepKeep * sizeof(double))) != cudaSuccess) return (int)e;
    unsigned long long *dcount = (unsigned long long *)d.p[0];
    double *dkeep = (double *)d.p[1];
    if ((e = cudaMemset(dcount, 0, sizeof(unsigned long long))) != cudaSuccess) return (int)e;
    if ((e = cudaMemset(dkeep, 0, 2 * kSweepKeep * sizeof(double))) != cudaSuccess) return (int)e;
    int dev = 0, sms = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return (int)e;
    const uint64_t pairs = count + (count & 1u);
    if (op == OP_DIV) vp_sweep_kernel<OP_DIV><<<sms * 8, 256>>>(seed, pairs, dcount, dkeep);
    else vp_sweep_kernel<OP_SQRT><<<sms * 8, 256>>>(seed, pairs, dcount, dkeep);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(mismatches, dcount, sizeof(unsigned long long), cudaMemcpyDeviceToHost)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(keep, dkeep, 2 * kSweepKeep * sizeof(double), cudaMemcpyDeviceToHost)) != cudaSuccess) return (int)e;
    return (int)cudaSuccess;
}

extern "C" int vp_sweep_keep(void) { return kSweepKeep; }
