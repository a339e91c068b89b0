// trace_fast.cu -- the two fast modes: fp32 geometry (RTB_F32_FAST) and FMA fp64 (RTB_F64_FAST).
//
// Same sequential trace, same slab / NaN conventions and the same I/O (float64 (N, 8) rows) as the exact mode, but
// built for speed instead of bit parity with NumPy:
//   * directions, normals and Snell's law in fp32 with FMA, using the direct vector form
//         d' = mu * d_t + sign(n.d) * sqrt(1 - mu^2 |d_t|^2) * n,   d_t = d - (n.d) n
//     (algebraically the reference's (normal, nb, nc) construction, raytrace.py:1203-1216, without the two cross
//     products and six divisions);
//   * positions, the sphere's quadratic coefficients and the phase stay in fp64 -- the far-sphere quadratic
//     (b ~ 600, c ~ 600^2) cancels catastrophically in fp32 and the phase reaches 1e7 rad (SURVEY.md section 7) --
//     which costs ~25 FP64 instructions per surface instead of ~190;
//   * a point produced by the intersection is on the surface by construction, so the reference's absolute 1e-12
//     on-surface test (meaningless in fp32) reduces to "the intersection exists"; the aperture test is kept.
//
// The same code instantiated with T = double is the RTB_F64_FAST mode: all arithmetic fp64 with FMA and the direct
// Snell form, ~3x fewer FP64 instructions than the exact mode.  It agrees with the reference to ~1e-13 (tolerance
// below) but NOT in the validity masks of knife-edge rays: the reference's absolute 1e-12 on-surface test culls a few
// rays in 1e5 purely on round-off (SURVEY.md section 0), which only the exact mode reproduces.
//
// Stated tolerances against the exact mode (asserted in tests/test_gpu_parity.py::test_fast_modes_tolerance and on every
// kernel route in tests/test_gpu_fast_modes.py; the classes and the knife-edge rules are tests/fast_tolerance.py):
//   RTB_F64_FAST: positions 1e-11 * L, directions 1e-12, phase 1e-12 relative (100x looser for high-NA perfect-lens
//                 systems); NaN masks equal except knife-edge rays.
//   RTB_F32_FAST:
//   positions  |dp| <= 2e-6 * L   (L = 1000 mm, the length scale of the traced systems: 2 nm per mm of path)
//   directions |dd| <= 2e-6
//   phase      |dphi| <= 2e-6 * |phi|  (i.e. optical path length to 2e-6 relative)
//   (10x looser, 2e-5, for high-NA perfect-lens systems such as the ideal OPM, where sin(theta) reaches 0.96 and the
//   fp32 direction error is amplified by 1/cos(theta)); phase 10x looser where fp32 t meets a small accumulated
//   phase: long trains of large spheres (the fp32 root, <= |R|, is off by up to |R| 2^-22) and systems of long-focal-
//   length perfect lenses (two plane steps per lens with fp32 t, |t| ~ n f): tests/fast_tolerance.py PHASE_F32
//   validity   identical NaN masks except for rays within the position tolerance of an aperture edge, of a
//              grazing / missing intersection or of the critical angle.
// This translation unit is compiled with FMA contraction enabled (see Makefile).
#include <cmath>
#include <math_constants.h>

#include "rtb_device.cuh"
#include "trace_common.cuh"

namespace rtb {

namespace {

// T = float: fp32 directions / normals; T = double: everything fp64
template <typename T>
struct RayT {
    double ox, oy, oz; // position (fp64)
    T dx, dy, dz;      // direction
    double ph;         // phase (fp64)
    double wl;
};

__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float sqrt_t(float x) { return sqrtf(x); }
__device__ __forceinline__ double sqrt_t(double x) { return xm::sqrt(x); }
__device__ __forceinline__ float div_t(float a, float b) { return a / b; }
__device__ __forceinline__ double div_t(double a, double b) { return xm::div(a, b); }
__device__ __forceinline__ float abs_t(float x) { return fabsf(x); }
__device__ __forceinline__ double abs_t(double x) { return fabs(x); }

template <typename T>
__device__ __forceinline__ T dot3f(T ax, T ay, T az, T bx, T by, T bz)
{
    return fma_t(az, bz, fma_t(ay, by, ax * bx));
}

template <typename T>
__device__ __forceinline__ void set_nan(RayT<T> &r)
{
    const double q = CUDART_NAN;
    r.ox = q; r.oy = q; r.oz = q;
    r.dx = (T)q; r.dy = (T)q; r.dz = (T)q;
    r.ph = q;
    r.wl = q;
}

template <typename T>
__device__ __forceinline__ Ray widen(const RayT<T> &r)
{
    Ray o;
    o.ox = r.ox; o.oy = r.oy; o.oz = r.oz;
    o.dx = (double)r.dx; o.dy = (double)r.dy; o.dz = (double)r.dz;
    o.ph = r.ph;
    o.wl = r.wl;
    return o;
}

// per-surface constants in the working precision
template <typename T>
struct SurfF {
    T nx, ny, nz, ax, ay, az;
    T focal_len, sin_alpha;
};

template <typename T>
__device__ __forceinline__ SurfF<T> surf_consts(const DevSurface &s)
{
    SurfF<T> f;
    f.nx = (T)s.nx; f.ny = (T)s.ny; f.nz = (T)s.nz;
    f.ax = (T)s.ax; f.ay = (T)s.ay; f.az = (T)s.az;
    f.focal_len = (T)s.focal_len;
    f.sin_alpha = (T)s.sin_alpha;
    return f;
}

// ray -> plane through (cx, cy, cz) with normal n; t in fp32, position and phase in fp64.  Returns t.
template <typename T>
__device__ __forceinline__ T to_plane_f(const RayT<T> &in, T nx, T ny, T nz, double cx, double cy, double cz, double k_n,
                                        double &px, double &py, double &pz, double &ph)
{
    const T rx = (T)(in.ox - cx), ry = (T)(in.oy - cy), rz = (T)(in.oz - cz);
    const T t = div_t(-dot3f(rx, ry, rz, nx, ny, nz), dot3f(in.dx, in.dy, in.dz, nx, ny, nz));
    const double td = (double)t;
    px = fma((double)in.dx, td, in.ox);
    py = fma((double)in.dy, td, in.oy);
    pz = fma((double)in.dz, td, in.oz);
    ph = fma(td, k_n, in.ph); // |d t| sign(t) k n with |d| = 1
    return t;
}

// refraction / reflection of unit d at unit normal n; mu = n1/n2 (mu < 0 selects reflection)
template <typename T>
__device__ __forceinline__ void bend(T dx, T dy, T dz, T nx, T ny, T nz, T mu, bool reflect, T &ex, T &ey, T &ez)
{
    const T c = dot3f(nx, ny, nz, dx, dy, dz);
    if (reflect) {
        ex = fma_t((T)-2 * c, nx, dx);
        ey = fma_t((T)-2 * c, ny, dy);
        ez = fma_t((T)-2 * c, nz, dz);
        return;
    }
    const T tx = fma_t(-c, nx, dx), ty = fma_t(-c, ny, dy), tz = fma_t(-c, nz, dz);
    const T s2 = mu * mu * dot3f(tx, ty, tz, tx, ty, tz);
    const T root = sqrt_t((T)1 - s2);                          // NaN beyond the critical angle
    const T w = (c > (T)0) ? root : ((c < (T)0) ? -root : (T)0 * root);
    ex = fma_t(mu, tx, w * nx);
    ey = fma_t(mu, ty, w * ny);
    ez = fma_t(mu, tz, w * nz);
}

// PerfectLens.propagate (raytrace.py:1601-1801)
template <typename T>
__device__ __forceinline__ bool lens_step(const DevSurface &s, const RayT<T> &in, double k, double n1, double n2,
                                          bool as_get_intersect, RayT<T> &before, RayT<T> &after)
{
    const SurfF<T> f = surf_consts<T>(s);
    const double fx = fma(-s.nfx, n1, s.cx), fy = fma(-s.nfy, n1, s.cy), fz = fma(-s.nfz, n1, s.cz);
    const double gx = fma(s.nfx, n2, s.cx), gy = fma(s.nfy, n2, s.cy), gz = fma(s.nfz, n2, s.cz);
    double ax, ay, az, ph_ffp;
    to_plane_f(in, f.nx, f.ny, f.nz, fx, fy, fz, k * n1, ax, ay, az, ph_ffp);

    const T rnd = dot3f(in.dx, in.dy, in.dz, f.nx, f.ny, f.nz);
    const T qx = fma_t(-rnd, f.nx, in.dx), qy = fma_t(-rnd, f.ny, in.dy), qz = fma_t(-rnd, f.nz, in.dz);
    T px = qx, py = qy, pz = qz;
    const T pn = sqrt_t(dot3f(px, py, pz, px, py, pz));
    if (pn > (T)1e-12) {
        const T inv = div_t((T)1, pn);
        px *= inv; py *= inv; pz *= inv;
    }
    const T hx = (T)(ax - fx), hy = (T)(ay - fy), hz = (T)(az - fz);
    const T hn = sqrt_t(dot3f(hx, hy, hz, hx, hy, hz));
    T ux = hx, uy = hy, uz = hz;
    if (hn != (T)0) {
        const T inv = div_t((T)1, hn);
        ux *= inv; uy *= inv; uz *= inv;
    }
    // sin(theta1) = p.d with p the unit transverse direction; p is perpendicular to n, so p.d = p.q (q = d - (d.n) n,
    // the transverse part itself).  p.q, not p.d: the rounding of q leaves p a component ~eps / |q| along n, which
    // p.d multiplies by d.n ~ 1 -- in fp32, 2e-5 for |q| = 2.5e-3, i.e. 1e-3 of sin(theta1) and mm-scale 1e-3 errors
    // in the image-side position n1 f sin(theta1)
    const T sin_t1 = dot3f(px, py, pz, qx, qy, qz);

    RayT<T> rb;
    const double scale = n1 * s.focal_len * (double)sin_t1;
    rb.ox = fma(scale, (double)px, gx);
    rb.oy = fma(scale, (double)py, gy);
    rb.oz = fma(scale, (double)pz, gz);
    const T sin_t2 = div_t(div_t(-hn, f.focal_len), (T)n2);
    const T cos_t2 = sqrt_t((T)1 - sin_t2 * sin_t2);
    rb.dx = fma_t(sin_t2, ux, cos_t2 * f.nx);
    rb.dy = fma_t(sin_t2, uy, cos_t2 * f.ny);
    rb.dz = fma_t(sin_t2, uz, cos_t2 * f.nz);
    rb.wl = in.wl;
    const bool culled = (abs_t(sin_t1) > f.sin_alpha) || (abs_t(sin_t2) > f.sin_alpha);
    if (culled) set_nan(rb);
    // the phase stays fp64: the plane-wave term from the fp64 focal-plane height and the widened direction
    const double plane_wave = fma(az - fz, (double)in.dz, fma(ay - fy, (double)in.dy, (ax - fx) * (double)in.dx));
    rb.ph = (ph_ffp - (k * n1) * plane_wave) + k * ((n1 * n1) * s.focal_len + (n2 * n2) * s.focal_len);

    to_plane_f(rb, f.nx, f.ny, f.nz, s.cx, s.cy, s.cz, k * n2, after.ox, after.oy, after.oz, after.ph);
    after.dx = rb.dx; after.dy = rb.dy; after.dz = rb.dz;
    after.wl = rb.wl;
    before = in;
    const T tb = to_plane_f(in, f.nx, f.ny, f.nz, s.cx, s.cy, s.cz, k * n1, before.ox, before.oy, before.oz,
                                before.ph);
    if (as_get_intersect && tb < (T)0) set_nan(before);
    return culled;
}

// SWEEP (FROM_SOURCE only): blockIdx.y picks the source, its output rows and its reduction bucket (rtb_trace_sources)
// LAST = 1: the launch keeps nothing but the final slab and reduces nothing (the common fast-mode call): no per-surface
// slab bookkeeping, a dead ray leaves the surface loop.  LAST = 2: the final slab or nothing, plus the fused reduction
// at one slab behind the launch rays (the analysis launches: spot statistics, pupil grids) -- no slab stores in the loop.
template <typename T, bool USE_TABLE, bool FROM_SOURCE, bool SWEEP = false, int LAST = 0>
__global__ void __launch_bounds__(128, sizeof(T) == 8 ? 4 : 6) trace_fast_kernel(const __grid_constant__ TraceParams P)
{
    static_assert(!SWEEP || FROM_SOURCE, "sweeps generate their rays");
    __shared__ double s_ntab[USE_TABLE ? (kMaxWavelengths + 1) * kMaxMedia : 1];
    __shared__ double s_ratio[USE_TABLE ? (kMaxWavelengths + 1) * kMaxMedia : 1];
    // per-surface fp32 constants and the fp32 copy of n1/n2, converted once per block (conversions run on the
    // quarter-rate XU pipe, so they must not be repeated per ray)
    __shared__ T s_geo[kMaxSurfaces][8];   // normal xyz, axis xyz, 1/R, aperture^2 (unused slot)
    __shared__ T s_ratio_f[USE_TABLE ? (kMaxWavelengths + 1) * kMaxMedia : 1];
    __shared__ SweepShared<SWEEP> s_sweep;
    if (SWEEP) sweep_setup(P, s_sweep);     // visible after the __syncthreads below
    const int n_med = P.n_surf + 1;
    if (USE_TABLE) {
        const int count = (P.n_wl + 1) * n_med;
        for (int k = threadIdx.x; k < count; k += blockDim.x) {
            s_ntab[k] = P.n_tab[k];
            s_ratio[k] = P.ratio_tab[k];
            s_ratio_f[k] = (T)P.ratio_tab[k];
        }
    }
    for (int k = threadIdx.x; k < P.n_surf; k += blockDim.x) {
        const DevSurface &s = P.surf[k];
        s_geo[k][0] = (T)s.nx; s_geo[k][1] = (T)s.ny; s_geo[k][2] = (T)s.nz;
        s_geo[k][3] = (T)s.ax; s_geo[k][4] = (T)s.ay; s_geo[k][5] = (T)s.az;
        s_geo[k][6] = (T)(1.0 / s.radius);
        s_geo[k][7] = (T)0;
    }
    __syncthreads();
    const DevSource &source = sweep_source(P, s_sweep);
    const DevReduce &red = sweep_reduce(P, s_sweep);
    const long long row0 = SWEEP ? (long long)blockIdx.y * P.n_rays : 0;
    const bool reducing = LAST != 1 && P.red.slab >= 0;
    const bool intersect_only = !LAST && (P.flags & RTB_FLAG_INTERSECT_ONLY) != 0;
    Tally tally;
    tally_init(tally);

    const bool planes_in = (P.flags & RTB_FLAG_PLANES_IN) != 0, planes_out = (P.flags & RTB_FLAG_PLANES_OUT) != 0;
    const long long out_rows = P.out_stride / 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P.n_rays; i += stride) {
        Ray first;
        if (FROM_SOURCE)
            first = make_ray(source, source.first + i);
        else
            load_ray(P.rays_in, i, P.n_rays, planes_in, first);
        if (!LAST && P.slab_pos[0] >= 0)
            store_ray(P.out + P.slab_pos[0] * P.out_stride, row0 + i, out_rows, planes_out, first);
        if (reducing && P.red.slab == 0) reduce_sample(red, first, tally);

        // the ray, in registers: position / phase fp64, direction fp32; the wavelength only ever turns NaN with the
        // whole ray (dead)
        double ox = first.ox, oy = first.oy, oz = first.oz, ph = first.ph;
        T dx = (T)first.dx, dy = (T)first.dy, dz = (T)first.dz;
        const double wl0 = first.wl;
        const double k = kTwoPi / wl0;
        int row = 0;
        bool unlisted = false;
        if (USE_TABLE) {
            row = wavelength_row(P, wl0);
            unlisted = (row == P.n_wl) && (wl0 == wl0);
            row *= n_med;
        }
        double n1 = !USE_TABLE ? eval_index(P.mat[0], wl0) : (unlisted ? index_for_unlisted(&P.mat[0], wl0) : s_ntab[row]);
        bool dead = false;           // every column NaN from here on
#pragma unroll 1
        for (int q = 0; q < P.n_surf; q++) {
            const DevSurface &s = P.surf[q];
            const double n2 = !USE_TABLE ? eval_index(P.mat[q + 1], wl0)
                                         : (unlisted ? index_for_unlisted(&P.mat[q + 1], wl0) : s_ntab[row + q + 1]);
            if (LAST && dead) break;
            const int act = LAST == 1 ? 0 : (LAST == 2 ? (P.slab_act[q] & 12) : P.slab_act[q]);
            auto emit = [&](bool at_slab, const Ray &w) {
                const int pos = P.slab_pos[2 * q + (at_slab ? 1 : 2)];
                if (act & (at_slab ? 1 : 2)) store_ray(P.out + pos * P.out_stride, row0 + i, out_rows, planes_out, w);
                if (act & (at_slab ? 4 : 8)) reduce_sample(red, w, tally);
            };
            if (dead) {
                if (act) {
                    Ray w;
                    set_nan(w);
                    if (act & 5) emit(true, w);
                    if (act & 10) emit(false, w);
                }
            } else if (s.kind == RTB_SURF_PERFECT_LENS) {
                RayT<T> cur, at, after;
                cur.ox = ox; cur.oy = oy; cur.oz = oz; cur.dx = dx; cur.dy = dy; cur.dz = dz; cur.ph = ph;
                cur.wl = wl0;
                dead = lens_step(s, cur, k, n1, n2, intersect_only, at, after);
                if (act & 5) emit(true, widen(at));
                if (act & 10) emit(false, widen(after));
                ox = after.ox; oy = after.oy; oz = after.oz; dx = after.dx; dy = after.dy; dz = after.dz; ph = after.ph;
            } else {
                // ---- flat / sphere refraction and plane mirror (raytrace.py:1160-1303) ----
                const bool mirror = s.kind == RTB_SURF_MIRROR;
                const double ddx = (double)dx, ddy = (double)dy, ddz = (double)dz;
                const T snx = s_geo[q][0], sny = s_geo[q][1], snz = s_geo[q][2];
                double px, py, pz, ph_at;
                T nx, ny, nz;
                bool kill = false, on;
                if (s.kind == RTB_SURF_SPHERE) {
                    // quadratic in fp64 (raytrace.py:1497-1509), root in fp32
                    const double qx = ox - s.cx, qy = oy - s.cy, qz = oz - s.cz;
                    const double b = fma(ddz, qz, fma(ddy, qy, ddx * qx));
                    const double cq = fma(qz, qz, fma(qy, qy, qx * qx)) - s.radius_sq;
                    const double root = (double)sqrt_t((T)fma(b, b, -cq));
                    const double t1 = root - b, t2 = -b - root;
                    double t = (t2 < 0.0) ? t1 : t2;
                    t = (t1 < 0.0 || root != root) ? CUDART_NAN : t;
                    px = fma(ddx, t, ox);
                    py = fma(ddy, t, oy);
                    pz = fma(ddz, t, oz);
                    ph_at = fma(t, k * n1, ph);
                    const T inv_r = s_geo[q][6];
                    nx = (T)(px - s.cx) * inv_r;
                    ny = (T)(py - s.cy) * inv_r;
                    nz = (T)(pz - s.cz) * inv_r;
                    // aperture measured from the axis through the origin (raytrace.py:1530-1533); fp64 is cheaper
                    // here than three more conversions
                    const double along = fma(pz, s.az, fma(py, s.ay, px * s.ax));
                    const double ux = fma(-along, s.ax, px), uy = fma(-along, s.ay, py), uz = fma(-along, s.az, pz);
                    on = fma(uz, uz, fma(uy, uy, ux * ux)) <= s.aperture * s.aperture;
                } else {
                    const T rx = (T)(ox - s.cx), ry = (T)(oy - s.cy), rz = (T)(oz - s.cz);
                    const T t = div_t(-dot3f(rx, ry, rz, snx, sny, snz), dot3f(dx, dy, dz, snx, sny, snz));
                    const double td = (double)t;
                    px = fma(ddx, td, ox);
                    py = fma(ddy, td, oy);
                    pz = fma(ddz, td, oz);
                    ph_at = fma(td, k * n1, ph);
                    kill = t < (T)0;
                    nx = snx; ny = sny; nz = snz;
                    const double ux = px - s.cx, uy = py - s.cy, uz = pz - s.cz;
                    on = fma(uz, uz, fma(uy, uy, ux * ux)) <= s.aperture * s.aperture;
                }
                if (!intersect_only && !mirror)
                    kill = kill || (dot3f(dx, dy, dz, s_geo[q][3], s_geo[q][4], s_geo[q][5]) < (T)0);
                on = on && !kill;
                if (act & 5) {
                    Ray w;
                    w.ox = px; w.oy = py; w.oz = pz; w.dx = ddx; w.dy = ddy; w.dz = ddz; w.ph = ph_at;
                    w.wl = wl0;
                    if (kill) set_nan(w);
                    emit(true, w);
                }
                const T ratio = (USE_TABLE && !unlisted) ? s_ratio_f[row + q] : (T)(n1 / n2);
                T ex, ey, ez;
                bend(dx, dy, dz, nx, ny, nz, ratio, mirror, ex, ey, ez);
                dead = !on;
                const bool no_dir = ex != ex;             // beyond the critical angle: position blanked too
                ox = no_dir ? CUDART_NAN : px;
                oy = no_dir ? CUDART_NAN : py;
                oz = no_dir ? CUDART_NAN : pz;
                dx = ex; dy = ey; dz = ez;
                ph = ph_at;
                if (act & 10) {
                    Ray w;
                    w.ox = ox; w.oy = oy; w.oz = oz; w.dx = (double)ex; w.dy = (double)ey; w.dz = (double)ez; w.ph = ph;
                    w.wl = wl0;
                    if (dead) set_nan(w);
                    emit(false, w);
                }
            }
            n1 = n2;
        }
        if (LAST && P.any_store) {
            // the final slab's row (slab_pos[2 S] = 0): the ray as it left the last surface, blank when it died
            Ray w;
            w.ox = ox; w.oy = oy; w.oz = oz; w.dx = (double)dx; w.dy = (double)dy; w.dz = (double)dz; w.ph = ph;
            w.wl = wl0;
            if (dead) set_nan(w);
            store_ray(P.out, row0 + i, out_rows, planes_out, w);
        }
    }
    if (reducing) tally_flush(red, tally);
}

template <typename T, int LAST>
cudaError_t launch_fast(const TraceParams &P, unsigned b, int threads, cudaStream_t stream)
{
    const bool table = P.n_wl > 0;
    const bool source = P.src.kind >= 0;
    if (P.n_src > 0) {
        const dim3 grid(b, (unsigned)P.n_src);
        if (table)
            trace_fast_kernel<T, true, true, true, LAST><<<grid, threads, 0, stream>>>(P);
        else
            trace_fast_kernel<T, false, true, true, LAST><<<grid, threads, 0, stream>>>(P);
        return cudaGetLastError();
    }
    if (table && source)
        trace_fast_kernel<T, true, true, false, LAST><<<b, threads, 0, stream>>>(P);
    else if (table)
        trace_fast_kernel<T, true, false, false, LAST><<<b, threads, 0, stream>>>(P);
    else if (source)
        trace_fast_kernel<T, false, true, false, LAST><<<b, threads, 0, stream>>>(P);
    else
        trace_fast_kernel<T, false, false, false, LAST><<<b, threads, 0, stream>>>(P);
    return cudaGetLastError();
}

} // namespace

cudaError_t launch_trace_fast(const TraceParams &P, int precision, int sm_count, cudaStream_t stream)
{
    if (P.n_rays <= 0) return cudaSuccess;
    const int threads = 128;
    long long blocks = (P.n_rays + threads - 1) / threads;
    long long max_blocks = (long long)sm_count * 32;
    if (P.n_src > 0) max_blocks = (max_blocks + P.n_src - 1) / P.n_src;   // the cap is for the whole grid
    if (blocks > max_blocks) blocks = max_blocks;
    // nothing but the final slab (or nothing at all) and at most one reduction behind the launch rays: the
    // instantiations without per-surface slab bookkeeping
    const bool plain = (P.flags & RTB_FLAG_INTERSECT_ONLY) == 0 && P.n_surf > 0;
    const int last = !plain ? 0
                     : (P.store_last_only && P.red.slab < 0) ? 1
                     : ((P.store_last_only || !P.any_store) && P.red.slab >= 1) ? 2 : 0;
    if (precision == RTB_F64_FAST)
        return last == 1 ? launch_fast<double, 1>(P, (unsigned)blocks, threads, stream)
               : last == 2 ? launch_fast<double, 2>(P, (unsigned)blocks, threads, stream)
                           : launch_fast<double, 0>(P, (unsigned)blocks, threads, stream);
    return last == 1 ? launch_fast<float, 1>(P, (unsigned)blocks, threads, stream)
           : last == 2 ? launch_fast<float, 2>(P, (unsigned)blocks, threads, stream)
                       : launch_fast<float, 0>(P, (unsigned)blocks, threads, stream);
}

} // namespace rtb
