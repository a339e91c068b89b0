// rtb_device.cuh -- device-side records and small helpers shared by the kernels and the C-ABI front end.
//
// Data layout in HBM
//   rays     : (N, 8) float64 rows of 64 B (x y z dx dy dz phase wavelength), the reference's own layout
//              (raytrace.py:1-5).  One thread owns one ray; a row moves as two 256-bit vector accesses, so a
//              warp touches 2 KB of contiguous memory with every 32-B sector fully used.
//   history  : (n_slabs, N, 8), slab-major like the NumPy array System.ray_trace returns.
//   the prescription (surfaces, media, refractive-index table) lives in the kernel parameter block
//   (__grid_constant__, constant bank 0): it is read warp-uniformly and is private to each launch, so concurrent
//   traces of different systems on different streams cannot interfere.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/rtb.h"

namespace rtb {

constexpr int kMaxSurfaces = RTB_MAX_SURFACES;
constexpr int kMaxMedia = RTB_MAX_SURFACES + 1;
constexpr int kMaxWavelengths = RTB_MAX_WAVELENGTHS;
constexpr int kMaxSlabs = 2 * RTB_MAX_SURFACES + 1;
constexpr int kMaxDevices = 64;       // device indices the C ABI accepts

// sets rtb_last_error() and returns `code` (rtb_api.cu; every translation unit of the C ABI reports errors through it)
int api_fail(int code, const char *fmt, ...);

// launch shape of the trace kernels: 128-thread blocks, register budget for kTraceMinBlocks resident blocks per SM
#ifndef RTB_TRACE_THREADS
#define RTB_TRACE_THREADS 128
#endif
constexpr int kTraceThreads = RTB_TRACE_THREADS;
#ifndef RTB_TRACE_MIN_BLOCKS
#define RTB_TRACE_MIN_BLOCKS 7
#endif
constexpr int kTraceMinBlocks = RTB_TRACE_MIN_BLOCKS;

struct DevSurface {
    double cx, cy, cz;    // center
    double nx, ny, nz;    // geometric normal (flat / mirror / lens)
    double ax, ay, az;    // input axis (front-side cull, sphere aperture)
    double radius, radius_sq, abs_radius;
    double aperture;
    double focal_len;
    double nfx, nfy, nfz; // normal * focal_len
    double sin_alpha;
    // exact squared-domain thresholds, computed on the host (rtb_api.cu: pack_thresholds) so that the kernel can
    // test  norm <= aperture  and  | norm - |R| | < 1e-12  without taking the square root:
    //   in_aperture  <=>  s <= ap_sq_max          (s = the left-associated sum of squares the reference feeds to sqrt)
    //   on_sphere    <=>  on_sq_lo <= s <= on_sq_hi
    double ap_sq_max;
    double on_sq_lo, on_sq_hi;
    int32_t kind;
    int8_t z_normal; // +-1 when normal == (0, 0, +-1) exactly, else 0   (shortcuts of the Optimistic policy)
    int8_t z_axis;   // +-1 when input_axis == (0, 0, +-1) exactly, else 0
    int8_t degenerate_hint; // rtb_surface.hints & RTB_HINT_DEGENERATE (flat surfaces: zero forms in the hot loop)
    int8_t pad;
};

struct DevMaterial {
    double b0, b1, b2;
    double c0, c1, c2;
    double n_const;
    int32_t kind;
    int32_t pad;
};

struct DevReduce {
    double ox, oy, oz;
    double e1x, e1y, e1z;
    double e2x, e2y, e2z;
    double phase_ref;
    double half_width;
    double inv_cell; // G / (2 * half_width), host computed
    double *stats;
    double *grid;
    int32_t slab; // -1 = no reduction
    int32_t grid_n;
    // derived (finish_reduce): the sin and count planes of the grid, grid_n as a double
    double *grid_sin;
    double *grid_count;
    double grid_n_f;
};

__host__ __device__ inline void finish_reduce(DevReduce &r)
{
    const long long plane = (long long)r.grid_n * r.grid_n;
    r.grid_sin = r.grid ? r.grid + plane : nullptr;
    r.grid_count = r.grid ? r.grid + 2 * plane : nullptr;
    r.grid_n_f = (double)r.grid_n;
}

struct DevSource {
    double a_start, a_step, a_stop; // linspace pieces: value(i) = i*a_step + a_start, last forced to a_stop
    double b_start, b_step, b_stop; // GRID: second linspace; FAN / COLLIMATED: azimuth = i * b_step + b_start
    double px, py, pz;
    double axx, axy, axz;
    double e1x, e1y, e1z;
    double e2x, e2y, e2z;
    double wavelength;
    long long n_a, n_b;
    long long first;
    int32_t kind; // -1 = rays come from memory
    int32_t pad;
};

// Everything one trace launch needs.  ~26 KB: inside the 32,764-byte kernel parameter limit of CUDA 12.1+.
struct TraceParams {
    const double *rays_in;
    double *out;
    long long n_rays;
    long long out_stride;       // doubles between output slabs (= 8 * n_rays of the *output* buffer)
    int32_t n_surf;
    int32_t n_wl;               // > 0: refractive indices come from n_tab
    int32_t store_last_only;    // RTB_KEEP_LAST fast flag
    int32_t any_store;
    int32_t flags;              // RTB_FLAG_*
    int32_t pad0;
    int16_t slab_pos[kMaxSlabs + 3]; // output slab position of trace slab j, -1 = not stored
    uint8_t slab_act[kMaxSurfaces];  // per surface: bit 0 store at-slab, 1 store after-slab, 2 reduce at, 3 reduce after
    DevReduce red;
    DevSource src;
    // a sweep (rtb_trace_sources): n_src > 0 sources in global memory, one per blockIdx.y, each tracing n_rays rays
    // into rows [y * n_rays, (y + 1) * n_rays) of the output and into bucket y of the reductions
    const DevSource *src_list;
    int32_t n_src;
    int32_t pad1;
    // the lean kernel (trace_lean.cu): results of its probe launch, [source][surface][2] = {rays that reached the
    // surface, rays whose lean step failed there}; surfaces that run the general steps whatever the probe says; and,
    // for the probe launch itself, the sampling stride through the n_rays_total rays of the real launch
    const unsigned *lean_counts;
    unsigned long long lean_general;
    long long lean_probe_stride;
    long long lean_probe_total;
    // runs of consecutive surfaces that take the same step (StepCode in trace_lean.cu), decided by the launcher: the
    // hot loops' control flow depends on kernel parameters only, which keeps their index in a uniform register
    int32_t lean_n_runs;
    int32_t lean_sample_run;         // the reduction samples after this run (-1: no reduction)
    int32_t lean_pure;               // the launcher vouches for every surface's lean step: the pure instantiations
    int32_t lean_pad;
    uint8_t lean_run_end[kMaxSurfaces + 2];
    uint8_t lean_run_code[kMaxSurfaces + 2];
    DevSurface surf[kMaxSurfaces];
    DevMaterial mat[kMaxMedia];
    double wl[kMaxWavelengths];
    double n_tab[(kMaxWavelengths + 1) * kMaxMedia]; // row-major [wavelength row][medium], row n_wl = NaN answer
    double ratio_tab[(kMaxWavelengths + 1) * kMaxMedia]; // [row][k] = n_tab[row][k] / n_tab[row][k+1] (host IEEE division)
};

static_assert(sizeof(TraceParams) < 32764, "TraceParams must fit the kernel parameter space");

// 256-bit global accesses (sm_100+): one ray row = two of these.
__device__ __forceinline__ void ld256_stream(const double *p, double &a, double &b, double &c, double &d)
{
    asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(a), "=d"(b), "=d"(c), "=d"(d)
                 : "l"(p));
}

__device__ __forceinline__ void st256(double *p, double a, double b, double c, double d)
{
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

} // namespace rtb
