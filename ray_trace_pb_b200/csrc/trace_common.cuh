// trace_common.cuh -- pieces shared by the fp64-exact and the fp32 trace kernels: refractive-index evaluation,
// ray I/O (256-bit row accesses), the on-device ray sources and the fused reductions.
#pragma once

#include <cmath>
#include <math_constants.h>

#include "exact_math.cuh"
#include "rtb_device.cuh"
#include "surface_steps.cuh"

namespace rtb {
namespace {

// Material.n (materials.py:39-51); Constant.n (materials.py:72-79) ignores the wavelength, NaN included
__device__ __forceinline__ double eval_index(const DevMaterial &m, double wl)
{
    if (m.kind == RTB_MAT_CONSTANT) return m.n_const;
    if (m.kind == RTB_MAT_TABLE_ONLY) return nan64(); // only the host knows this medium
    const double w2 = wl * wl;
    const double acc = (xm::div(m.b0 * w2, w2 - m.c0) + xm::div(m.b1 * w2, w2 - m.c1)) + xm::div(m.b2 * w2, w2 - m.c2);
    return xm::sqrt(acc + 1.0);
}

// a ray whose wavelength is not in the host table (the table may be built from a sample of the batch)
static __device__ __noinline__ double index_for_unlisted(const DevMaterial *m, double wl) { return eval_index(*m, wl); }

// the row of the index tables that lists wavelength wl (bit for bit), or P.n_wl -- the NaN-wavelength row -- when none does
__device__ __forceinline__ int wavelength_row(const TraceParams &P, double wl)
{
    int row = P.n_wl;
    const long long bits = __double_as_longlong(wl);
#pragma unroll 1
    for (int k = 0; k < P.n_wl; k++)
        if (__double_as_longlong(P.wl[k]) == bits) row = k;
    return row;
}

// a reciprocal 1/den usable by the optimistic steps: finite, |den| < 2^52, and a reciprocal that is an ordinary normal
// number
__device__ __forceinline__ bool usable_rcp(double den, double rcp)
{
    return xm::den_ok(den) && fabs(den) < 4503599627370496.0 && xm::quo_ok(rcp);
}

__device__ __forceinline__ bool non_finite(double v) { return (__double2hiint(v) & 0x7ff00000) == 0x7ff00000; }

// ---- ray I/O ---------------------------------------------------------------------------------------------
// Two layouts (rtb_trace_opts.flags): rows of 8 doubles -- the reference's (N, 8), moved as two 256-bit accesses per
// ray so every 32-byte sector is used whole -- or planes (8, N), where each of the eight accesses of a warp is one
// contiguous 256-byte run.
__device__ __forceinline__ void load_ray(const double *base, long long i, long long n, bool planes, Ray &r)
{
    if (planes) {
        r.ox = __ldg(base + i);         r.oy = __ldg(base + n + i);     r.oz = __ldg(base + 2 * n + i);
        r.dx = __ldg(base + 3 * n + i); r.dy = __ldg(base + 4 * n + i); r.dz = __ldg(base + 5 * n + i);
        r.ph = __ldg(base + 6 * n + i); r.wl = __ldg(base + 7 * n + i);
        return;
    }
    const double *p = base + 8 * i;
    ld256_stream(p, r.ox, r.oy, r.oz, r.dx);
    ld256_stream(p + 4, r.dy, r.dz, r.ph, r.wl);
}

__device__ __forceinline__ void store_ray(double *base, long long i, long long n, bool planes, const Ray &r)
{
    if (planes) {
        base[i] = r.ox;         base[n + i] = r.oy;     base[2 * n + i] = r.oz;
        base[3 * n + i] = r.dx; base[4 * n + i] = r.dy; base[5 * n + i] = r.dz;
        base[6 * n + i] = r.ph; base[7 * n + i] = r.wl;
        return;
    }
    double *p = base + 8 * i;
    st256(p, r.ox, r.oy, r.oz, r.dx);
    st256(p + 4, r.dy, r.dz, r.ph, r.wl);
}

// on-device ray sources (raytrace.py:45-161 and this library's Cartesian grid); see rtb_source in rtb.h
__device__ __forceinline__ double linspace_at(long long i, long long n, double start, double step, double stop)
{
    // explicit roundings: this header is also compiled into the fp32 mode's translation unit, where FMA contraction
    // is on, and the sources must produce the same rays in both modes (np.linspace: arange(n) * step + start)
    const double v = __dadd_rn(__dmul_rn((double)i, step), start);
    return (n > 1 && i == n - 1) ? stop : v;
}

// idx = hi * n + lo with 0 <= lo < n; 32-bit division when both fit (the 64-bit one is a ~100-instruction routine)
__device__ __forceinline__ void split_index(long long idx, long long n, long long &lo, long long &hi)
{
    if ((((unsigned long long)idx | (unsigned long long)n) >> 32) == 0) {
        const unsigned q = (unsigned)idx / (unsigned)n;
        hi = q;
        lo = (unsigned)idx - q * (unsigned)n;
    } else {
        hi = idx / n;
        lo = idx - hi * n;
    }
}

__device__ __noinline__ Ray make_ray(const DevSource &g, long long idx)
{
    Ray r;
    r.ph = 0.0;
    r.wl = g.wavelength;
    if (g.kind == RTB_SRC_GRID) {
        long long iu, iv;
        split_index(idx, g.n_a, iu, iv);
        const double u = linspace_at(iu, g.n_a, g.a_start, g.a_step, g.a_stop);
        const double v = linspace_at(iv, g.n_b, g.b_start, g.b_step, g.b_stop);
        r.ox = __dadd_rn(__dadd_rn(g.px, __dmul_rn(g.e1x, u)), __dmul_rn(g.e2x, v));
        r.oy = __dadd_rn(__dadd_rn(g.py, __dmul_rn(g.e1y, u)), __dmul_rn(g.e2y, v));
        r.oz = __dadd_rn(__dadd_rn(g.pz, __dmul_rn(g.e1z, u)), __dmul_rn(g.e2z, v));
        r.dx = g.axx; r.dy = g.axy; r.dz = g.axz;
    } else if (g.kind == RTB_SRC_COLLIMATED) {
        long long ip, id;
        split_index(idx, g.n_b, ip, id);
        const double off = linspace_at(id, g.n_a, g.a_start, g.a_step, g.a_stop);
        const double phi = __dadd_rn(__dmul_rn((double)ip, kTwoPi) / (double)g.n_b, g.b_start);
        double sp, cp;
        sincos(phi, &sp, &cp);
        const double a = __dmul_rn(off, cp), b = __dmul_rn(off, sp);
        r.ox = __dadd_rn(__dadd_rn(g.px, __dmul_rn(g.e1x, a)), __dmul_rn(g.e2x, b));
        r.oy = __dadd_rn(__dadd_rn(g.py, __dmul_rn(g.e1y, a)), __dmul_rn(g.e2y, b));
        r.oz = __dadd_rn(__dadd_rn(g.pz, __dmul_rn(g.e1z, a)), __dmul_rn(g.e2z, b));
        r.dx = g.axx; r.dy = g.axy; r.dz = g.axz;
    } else {
        long long it, ip;
        split_index(idx, g.n_a, it, ip);
        const double theta = linspace_at(it, g.n_a, g.a_start, g.a_step, g.a_stop);
        const double phi = ((double)ip * kTwoPi) / (double)g.n_b;
        double st, ct, sp, cp;
        sincos(theta, &st, &ct);
        sincos(phi, &sp, &cp);
        r.ox = g.px; r.oy = g.py; r.oz = g.pz;
        r.dx = __dadd_rn(__dadd_rn(__dmul_rn(g.axx, ct), __dmul_rn(__dmul_rn(g.e1x, cp), st)), __dmul_rn(__dmul_rn(g.e2x, sp), st));
        r.dy = __dadd_rn(__dadd_rn(__dmul_rn(g.axy, ct), __dmul_rn(__dmul_rn(g.e1y, cp), st)), __dmul_rn(__dmul_rn(g.e2y, sp), st));
        r.dz = __dadd_rn(__dadd_rn(__dmul_rn(g.axz, ct), __dmul_rn(__dmul_rn(g.e1z, cp), st)), __dmul_rn(__dmul_rn(g.e2z, sp), st));
    }
    return r;
}

// ---- sweeps (rtb_trace_sources): the block's source and reduction bucket, staged in shared memory ------------------
template <bool SWEEP>
struct SweepShared {
    char unused;
};
template <>
struct SweepShared<true> {
    DevSource src;
    DevReduce red;
};

__device__ __forceinline__ void sweep_setup(const TraceParams &, SweepShared<false> &) {}
__device__ __forceinline__ const DevSource &sweep_source(const TraceParams &P, const SweepShared<false> &) { return P.src; }
__device__ __forceinline__ const DevReduce &sweep_reduce(const TraceParams &P, const SweepShared<false> &) { return P.red; }
__device__ __forceinline__ const DevSource &sweep_source(const TraceParams &, const SweepShared<true> &s) { return s.src; }
__device__ __forceinline__ const DevReduce &sweep_reduce(const TraceParams &, const SweepShared<true> &s) { return s.red; }

__device__ __forceinline__ void sweep_setup(const TraceParams &P, SweepShared<true> &s)
{
    if (threadIdx.x == 0) {
        s.src = P.src_list[blockIdx.y];
        s.red = P.red;
        if (s.red.stats) s.red.stats += (long long)blockIdx.y * RTB_N_STATS;
        if (s.red.grid) s.red.grid += (long long)blockIdx.y * 3 * s.red.grid_n * s.red.grid_n;
        finish_reduce(s.red);
    }
}

// ---- fused reductions (rtb_reduce in rtb.h) -----------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ void atomic_min_f64(double *addr, double v)
{
    unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *a;
    while (v < __longlong_as_double((long long)old)) {
        const unsigned long long prev = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (prev == old) break;
        old = prev;
    }
}
__device__ __forceinline__ void atomic_max_f64(double *addr, double v)
{
    unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *a;
    while (v > __longlong_as_double((long long)old)) {
        const unsigned long long prev = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (prev == old) break;
        old = prev;
    }
}

// Running sums of one thread, flushed once per thread block at the end of the kernel.
struct Tally {
    double cnt, su, sv, suu, svv, suv, sp, spp, umin, umax, vmin, vmax;
};

__device__ __forceinline__ void tally_init(Tally &t)
{
    t.cnt = t.su = t.sv = t.suu = t.svv = t.suv = t.sp = t.spp = 0.0;
    t.umin = t.vmin = CUDART_INF;
    t.umax = t.vmax = -CUDART_INF;
}

__device__ __noinline__ void reduce_sample(const DevReduce &R, const Ray r, Tally &t)
{
    const double px = r.ox - R.ox, py = r.oy - R.oy, pz = r.oz - R.oz;
    const double u = dot3(px, py, pz, R.e1x, R.e1y, R.e1z);
    const double v = dot3(px, py, pz, R.e2x, R.e2y, R.e2z);
    const double ph = r.ph - R.phase_ref;
    if (!(isfinite(u) && isfinite(v) && isfinite(ph))) return;
    if (R.stats) {
        t.cnt += 1.0;
        t.su += u; t.sv += v;
        t.suu += u * u; t.svv += v * v; t.suv += u * v;
        t.sp += ph; t.spp += ph * ph;
        t.umin = fmin(t.umin, u); t.umax = fmax(t.umax, u);
        t.vmin = fmin(t.vmin, v); t.vmax = fmax(t.vmax, v);
    }
    if (R.grid) {
        const double fu = floor((u + R.half_width) * R.inv_cell);
        const double fv = floor((v + R.half_width) * R.inv_cell);
        const double g = (double)R.grid_n;
        if (fu >= 0.0 && fu < g && fv >= 0.0 && fv < g) {
            const long long cell = (long long)fv * R.grid_n + (long long)fu;
            const long long plane = (long long)R.grid_n * R.grid_n;
            double s, c;
            sincos(ph, &s, &c);
            // the grid is always global memory: a plain reduction, no generic-address dispatch, nothing returned
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid + cell), "d"(c) : "memory");
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid + plane + cell), "d"(s) : "memory");
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid + 2 * plane + cell), "d"(1.0) : "memory");
        }
    }
}

__device__ __noinline__ void tally_flush(const DevReduce &R, Tally &t)
{
    if (!R.stats) return;
    __shared__ double part[12][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    double v[12] = {warp_sum(t.cnt), warp_sum(t.su),  warp_sum(t.sv),  warp_sum(t.suu),
                    warp_sum(t.svv), warp_sum(t.suv), warp_sum(t.sp),  warp_sum(t.spp),
                    warp_min(t.umin), warp_max(t.umax), warp_min(t.vmin), warp_max(t.vmax)};
    if (lane == 0)
        for (int k = 0; k < 12; k++) part[k][warp] = v[k];
    __syncthreads();
    if (warp == 0) {
        for (int k = 0; k < 12; k++) {
            double x;
            if (k < 8) {
                x = (lane < nwarp) ? part[k][lane] : 0.0;
                x = warp_sum(x);
                if (lane == 0 && x != 0.0) atomicAdd(R.stats + k, x);
            } else if (k == 8 || k == 10) {
                x = (lane < nwarp) ? part[k][lane] : CUDART_INF;
                x = warp_min(x);
                if (lane == 0 && x < CUDART_INF) atomic_min_f64(R.stats + k, x);
            } else {
                x = (lane < nwarp) ? part[k][lane] : -CUDART_INF;
                x = warp_max(x);
                if (lane == 0 && x > -CUDART_INF) atomic_max_f64(R.stats + k, x);
            }
        }
    }
}


} // namespace
} // namespace rtb
