// trace_lean.cu -- the fused fp64 trace for the workloads that keep nothing but the final slab and / or ONE fused
// reduction (spot statistics, pupil grid) after a surface: BASELINE configs 2-5, the bench step, every sweep.
// Same results, bit for bit, as trace_f64.cu (tests/test_gpu_parity.py runs both); what differs is how the work is laid
// out for the B200's operand-read port (lean_steps.cuh, DESIGN.md section 4a):
//
//   * The surface loop's trip count and index are warp-uniform -- a dead ray idles through the remaining surfaces instead
//     of leaving the loop -- so the prescription is read through uniform registers / constant-bank operands.
//   * The ray is updated in place by steps that carry no exact-zero handling and no second copy of the state.  A ray
//     whose domain flag fails anywhere is re-traced from its launch state, once, after the loop, by the careful
//     per-surface machinery of surface_steps.cuh (redo_ray, out of line).
//   * Surfaces at which WHOLE BUNDLES fail the lean step (a collimated beam at its first lens: d x n has an exact zero
//     component ray after ray; a source on the first flat; a beam along a flat's normal) are found by a probe launch of
//     this same kernel over a sample of <= 2048 rays per source, which counts per surface the rays that reached it and the
//     rays whose lean step failed; the main launch reads the counts and runs the zero-tolerant general steps
//     (surface_steps.cuh, OptimisticZ) at those surfaces.  No host round trip: probe and trace are two launches on the
//     caller's stream.  Hints (rtb_surface.hints) are therefore not needed by this kernel.
//   * Spot statistics are tallied per thread in shared memory (touched once per ray) instead of in 24 registers.
//
// THIS TRANSLATION UNIT MUST BE COMPILED WITH -fmad=false (see trace_f64.cu).
#include <cmath>
#include <math_constants.h>

#include "exact_math.cuh"
#include "lean_steps.cuh"
#include "rtb_device.cuh"
#include "surface_steps.cuh"
#include "trace_common.cuh"

namespace rtb {

namespace {

#ifndef RTB_LEAN_THREADS
#define RTB_LEAN_THREADS 128
#endif
#ifndef RTB_LEAN_MIN_BLOCKS
#define RTB_LEAN_MIN_BLOCKS 7
#endif
constexpr int kLeanThreads = RTB_LEAN_THREADS;
constexpr int kLeanMinBlocks = RTB_LEAN_MIN_BLOCKS;
constexpr int kProbeRays = 2048;          // sample size of the probe launch, per source
constexpr unsigned kProbeOneIn = 200;     // a surface runs the general steps when more than 1 in 200 probe rays failed

// which step a surface runs (decided once per block: kind, axes, the reciprocal radius, the probe's counts)
enum StepCode : int { kLeanSphere = 0, kLeanFlat = 1, kGeneralRefracting = 2, kGeneralMirror = 3, kGeneralLens = 4,
                      kMixedRun = 5, kLeanFlatAny = 6, kLeanLens = 7, kLeanFlatZ = 8 };

// the step a surface runs: lean where one exists (spheres on a z axis; flats, on the axis or tilted; perfect lenses),
// the general step of its kind otherwise or when `general` says so (probe result, unusable reciprocal)
__host__ __device__ inline int step_code(const DevSurface &s, bool general)
{
    const int fallback = (s.kind == RTB_SURF_MIRROR) ? kGeneralMirror
                                                     : (s.kind == RTB_SURF_PERFECT_LENS) ? kGeneralLens : kGeneralRefracting;
    // (an on-axis flat keeps a lean step when the probe overrides it: the zero-tolerant form, which takes every bundle
    // the general step takes)
    if (s.kind == RTB_SURF_FLAT && s.z_axis != 0 && s.z_normal != 0) return general ? kLeanFlatZ : kLeanFlat;
    if (general) return fallback;
    if (s.kind == RTB_SURF_SPHERE) return s.z_axis != 0 ? kLeanSphere : fallback;
    if (s.kind == RTB_SURF_FLAT) return kLeanFlatAny;
    if (s.kind == RTB_SURF_PERFECT_LENS) return kLeanLens;
    return fallback;
}

__host__ __device__ inline bool has_lean_step(const DevSurface &s) { return step_code(s, false) < kGeneralRefracting || step_code(s, false) > kMixedRun; }

// per-surface facts every ray needs, decided once per block: one 16-byte shared-memory read per surface
struct __align__(16) SurfaceShared {
    double rcp;                           // refined 1/R (1/f for perfect lenses)
    int code;                             // StepCode
    int rcp_ok;                           // that reciprocal is usable by the optimistic steps
};

struct LeanShared {
    SurfaceShared surf[kMaxSurfaces];
    double2 near_one[xm::kNearOneEntries];  // (sqrt(s), 1/sqrt(s)) for |c|^2 = s near 1 (exact_math.cuh)
    int run_clean[kMaxSurfaces + 2];      // the probe overrode no surface of this run (see TraceParams::lean_run_*)
};

// ---- the careful whole-ray trace: a ray whose lean flag failed starts over here --------------------------------------
// Returns the final slab's row (blanked when the ray is dead) and the row of slab 2 * k_sample + 2 (or, sample_at,
// 2 * k_sample + 1).
template <bool USE_TABLE>
static __device__ __noinline__ void redo_ray(const TraceParams *P, Ray cur, int k_sample, bool sample_at, Ray *final_row,
                                             Ray *sample_row)
{
    const int n_med = P->n_surf + 1;
    const double wl0 = cur.wl;
    int row = 0;
    bool unlisted = false;
    if (USE_TABLE) {
        row = P->n_wl;
        const long long bits = __double_as_longlong(wl0);
        for (int k = 0; k < P->n_wl; k++)
            if (__double_as_longlong(P->wl[k]) == bits) row = k;
        unlisted = (row == P->n_wl) && (wl0 == wl0);
        row *= n_med;
    }
    auto index_of = [&](int medium) {
        return !USE_TABLE ? eval_index(P->mat[medium], wl0)
                          : (unlisted ? index_for_unlisted(&P->mat[medium], wl0) : P->n_tab[row + medium]);
    };
    double n1 = index_of(0);
    bool dead = false;
    Ray blank;
    set_nan(blank);
    *sample_row = blank;
    for (int k = 0; k < P->n_surf; k++) {
        if (!dead) {
            const DevSurface *s = &P->surf[k];
            const double n2 = index_of(k + 1);
            StepResult res;
            if (s->kind == RTB_SURF_FLAT || s->kind == RTB_SURF_SPHERE) {
                const double ratio = (USE_TABLE && !unlisted) ? P->ratio_tab[row + k] : xm::div(n1, n2);
                res = careful_refracting(s, cur, n1, ratio, true);
            } else if (s->kind == RTB_SURF_MIRROR) {
                res = careful_mirror(s, cur, n1);
            } else {
                res = careful_lens(s, cur, n1, n2, false);
            }
            if (k == k_sample && sample_at) *sample_row = res.at;
            cur = res.after;
            dead = res.dead;
            n1 = n2;
        }
        if (k == k_sample && !sample_at) *sample_row = dead ? blank : cur;
    }
    *final_row = dead ? blank : cur;
}

// ---- fused reductions: rtb_reduce in rtb.h (same arithmetic as reduce_sample in trace_common.cuh) --------------------
// The per-thread tally lives in shared memory as six (statistic 2j, statistic 2j + 1) pairs, [pair][thread]: one 128-bit
// load and store per pair.  u, v and the phase are finite where it is touched, so the extrema are plain compares (fmin /
// fmax would carry their NaN handling), the cell is the truncation of a non-negative number (floor(x) >= 0 <=> x >= 0,
// floor(x) < G <=> x < G for an integer G) and fits 32 bits (G <= 32768).
__device__ __forceinline__ void accumulate(const DevReduce &R, double ox, double oy, double oz, double phase, double *tally)
{
    const double px = ox - R.ox, py = oy - R.oy, pz = oz - R.oz;
    const double u = dot3(px, py, pz, R.e1x, R.e1y, R.e1z);
    const double v = dot3(px, py, pz, R.e2x, R.e2y, R.e2z);
    const double ph = phase - R.phase_ref;
    if (!(isfinite(u) && isfinite(v) && isfinite(ph))) return;
    if (R.stats) {
        double2 *t = reinterpret_cast<double2 *>(tally) + threadIdx.x;
        constexpr int W = kLeanThreads;
        double2 a = t[0 * W], b = t[1 * W], c = t[2 * W], d = t[3 * W], e = t[4 * W], f = t[5 * W];
        a.x += 1.0;
        a.y += u;
        b.x += v;
        b.y += u * u;
        c.x += v * v;
        c.y += u * v;
        d.x += ph;
        d.y += ph * ph;
        e.x = u < e.x ? u : e.x;
        e.y = u > e.y ? u : e.y;
        f.x = v < f.x ? v : f.x;
        f.y = v > f.y ? v : f.y;
        t[0 * W] = a; t[1 * W] = b; t[2 * W] = c; t[3 * W] = d; t[4 * W] = e; t[5 * W] = f;
    }
    if (R.grid) {
        const double xu = (u + R.half_width) * R.inv_cell;
        const double xv = (v + R.half_width) * R.inv_cell;
        const double g = R.grid_n_f;
        if (xu >= 0.0 && xu < g && xv >= 0.0 && xv < g) {
            const unsigned cell = (unsigned)__double2int_rz(xv) * (unsigned)R.grid_n + (unsigned)__double2int_rz(xu);
            double s, c;
            sincos(ph, &s, &c);
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid + cell), "d"(c) : "memory");
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid_sin + cell), "d"(s) : "memory");
            asm volatile("red.global.add.f64 [%0], %1;" ::"l"(R.grid_count + cell), "d"(1.0) : "memory");
        }
    }
}

// statistic k of thread `thread` in that layout
__device__ __forceinline__ int tally_index(int k, int thread) { return ((k >> 1) * kLeanThreads + thread) * 2 + (k & 1); }

__device__ __noinline__ void flush_tally(const DevReduce &R, const double *tally)
{
    if (!R.stats) return;
    __shared__ double part[12][kLeanThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = 0; k < 12; k++) {
        double x = tally[tally_index(k, threadIdx.x)];
        x = (k < 8) ? warp_sum(x) : ((k == 8 || k == 10) ? warp_min(x) : warp_max(x));
        if (lane == 0) part[k][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < 12) {
        const int k = threadIdx.x;
        double x = part[k][0];
        for (int w = 1; w < kLeanThreads / 32; w++)
            x = (k < 8) ? x + part[k][w] : ((k == 8 || k == 10) ? fmin(x, part[k][w]) : fmax(x, part[k][w]));
        if (k < 8) {
            if (x != 0.0) atomicAdd(R.stats + k, x);
        } else if (k == 8 || k == 10) {
            if (x < CUDART_INF) atomic_min_f64(R.stats + k, x);
        } else {
            if (x > -CUDART_INF) atomic_max_f64(R.stats + k, x);
        }
    }
}

// the general steps of surface_steps.cuh with their zero forms in line, on the lean kernel's in-place state
__device__ __forceinline__ bool general_step(const DevSurface &s, int code, double rcp_y, bool rcp_ok, lean::State &r, double n1,
                                             double n2, double ratio, double wl0, double wl_rcp, bool &ok, bool &kill)
{
    OptimisticZ m;
    xm::Rcp rcp_wl, rcp_k;
    rcp_wl.b = wl0; rcp_wl.y = wl_rcp; rcp_wl.ok = true;
    rcp_k.b = (code == kGeneralLens) ? s.focal_len : s.radius;
    rcp_k.y = rcp_y;
    rcp_k.ok = rcp_ok;
    Ray in, after;
    in.ox = r.ox; in.oy = r.oy; in.oz = r.oz; in.dx = r.dx; in.dy = r.dy; in.dz = r.dz; in.ph = r.ph;
    in.wl = wl0;
    AtRaw raw;
    bool dead;
    if (code == kGeneralRefracting)
        dead = refracting_step<OptimisticZ, true>(m, s, in, n1, ratio, rcp_wl, rcp_k, true, raw, after);
    else if (code == kGeneralMirror)
        dead = mirror_step<OptimisticZ, true>(m, s, in, n1, rcp_wl, raw, after);
    else
        dead = perfect_lens_step<OptimisticZ>(m, s, in, n1, n2, rcp_wl, rcp_k, false, false, raw, after);
    ok = m.ok;
    kill = raw.kill;       // (a perfect lens's "at" slab is not offered as a sample: lean_eligible)
    r.ox = after.ox; r.oy = after.oy; r.oz = after.oz;
    r.dx = after.dx; r.dy = after.dy; r.dz = after.dz;
    r.ph = after.ph;
    return !dead;
}

// ---- the kernel --------------------------------------------------------------------------------------------------
// USE_TABLE / FROM_SOURCE as in trace_f64.cu.  SWEEP: blockIdx.y picks the source, its output rows and its reduction
// bucket (rtb_trace_sources).  PROBE: the probe launch -- a strided sample of the rays, per-surface recovery, counts only.
// KINDS   0: the instantiation for systems of spheres and on-axis flats only (lens trains: the relay, doublets, the
//            achromat systems) -- it does not carry the perfect-lens, tilted-flat and mirror steps, whose mere presence
//            costs the sphere loop 2 % through register allocation; 1: every step.  2 / 3: the PURE forms of 0 / of
//            "every lean step": no general steps, no probe counts -- the launcher has made sure (from an earlier probe's
//            verdict on the same system, rtb_api.cu) that every surface can run its lean step.  Nothing in them branches on
//            a value loaded from memory, which lets ptxas keep the loop indices in uniform registers and read the
//            prescription through the uniform datapath (operands that cost no operand-port cycle, DESIGN.md 4a).
template <bool USE_TABLE, bool FROM_SOURCE, bool SWEEP, bool PROBE, int KINDS>
__global__ void __launch_bounds__(kLeanThreads, kLeanMinBlocks) trace_lean_kernel(const __grid_constant__ TraceParams P,
                                                                                  unsigned *probe_counts)
{
    static_assert(!SWEEP || FROM_SOURCE, "sweeps generate their rays");
    // dynamic shared memory: {n, n1/n2} pairs per (wavelength row, surface), then the per-thread tallies
    extern __shared__ __align__(16) double s_dyn[];
    const int n_med = P.n_surf + 1;
    double *const s_pair = s_dyn;
    double *const s_tally = s_dyn + (USE_TABLE ? 2 * (P.n_wl + 1) * n_med : 0);
    __shared__ LeanShared s_c;
    __shared__ SweepShared<SWEEP> s_sweep;
    if (SWEEP) sweep_setup(P, s_sweep);
    if (USE_TABLE) {
        const int count = (P.n_wl + 1) * n_med;
        for (int k = threadIdx.x; k < count; k += blockDim.x) {
            s_pair[2 * k] = P.n_tab[k];
            s_pair[2 * k + 1] = P.ratio_tab[k];
        }
    }
    const bool reducing = !PROBE && P.red.slab >= 0;
    if (reducing && P.red.stats) {
        for (int k = 0; k < 12; k++)
            s_tally[tally_index(k, threadIdx.x)] = (k < 8) ? 0.0 : ((k == 8 || k == 10) ? CUDART_INF : -CUDART_INF);
    }
    for (int k = threadIdx.x; k < xm::kNearOneEntries; k += blockDim.x) s_c.near_one[k] = xm::near_one_entry(k);
    for (int k = threadIdx.x; k < P.n_surf; k += blockDim.x) {
        const DevSurface &s = P.surf[k];
        const double den = (s.kind == RTB_SURF_PERFECT_LENS) ? s.focal_len : s.radius;
        const double rcp = xm::refine_rcp(den);
        const bool sane = xm::den_ok(den) && fabs(den) < 4503599627370496.0 && xm::quo_ok(rcp);
        s_c.surf[k].rcp = rcp;
        s_c.surf[k].rcp_ok = sane;
        // a sphere / lens whose reciprocal radius / focal length is unusable goes through the general step (which flags
        // it for the careful path)
        bool general = ((P.lean_general >> k) & 1ull) != 0 ||
                       (!sane && (s.kind == RTB_SURF_SPHERE || s.kind == RTB_SURF_PERFECT_LENS));
        if (!PROBE && KINDS < 2 && P.lean_counts) {
            const unsigned *cnt = P.lean_counts + ((size_t)(SWEEP ? blockIdx.y : 0) * kMaxSurfaces + k) * 2;
            general |= (unsigned long long)cnt[1] * kProbeOneIn > (unsigned long long)cnt[0];
        }
        s_c.surf[k].code = step_code(s, general);
    }
    __syncthreads();
    for (int run = threadIdx.x; KINDS < 2 && run < P.lean_n_runs; run += blockDim.x) {
        bool clean = true;
        for (int k = run > 0 ? P.lean_run_end[run - 1] : 0; k < P.lean_run_end[run]; k++)
            clean &= s_c.surf[k].code == P.lean_run_code[run];
        s_c.run_clean[run] = clean;
    }
    __syncthreads();

    const DevSource &source = sweep_source(P, s_sweep);
    const DevReduce &red = sweep_reduce(P, s_sweep);
    const long long row0 = SWEEP ? (long long)blockIdx.y * P.n_rays : 0;
    // the sample is the slab after surface k_red (even slab) or at it (odd slab)
    const int k_red = reducing ? ((P.red.slab - 1) >> 1) : -1;
    const bool sample_at = reducing && (P.red.slab & 1) != 0;
    const bool planes_in = (P.flags & RTB_FLAG_PLANES_IN) != 0, planes_out = (P.flags & RTB_FLAG_PLANES_OUT) != 0;
    const long long out_rows = P.out_stride / 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned *const my_counts = PROBE ? probe_counts + (size_t)(SWEEP ? blockIdx.y : 0) * kMaxSurfaces * 2 : nullptr;

    // warp-uniform trip count: every lane of a warp runs the same iterations, lanes past the end idle
    for (long long base = (long long)blockIdx.x * blockDim.x; base < P.n_rays; base += stride) {
        long long i = base + threadIdx.x;
        const bool valid = i < P.n_rays;
        if (PROBE) {
            // the probe's ray `i` of the sample is ray i * stride + jitter of the real launch (the jitter keeps the sample
            // off the rows / columns of a Cartesian source)
            const long long st = P.lean_probe_stride;
            i = i * st + (long long)((unsigned)(i * 2654435761u) % (unsigned long long)st);
            if (i >= P.lean_probe_total) i = P.lean_probe_total - 1;
        }
        Ray cur;
        set_nan(cur);
        if (valid) {
            if (FROM_SOURCE)
                cur = make_ray(source, source.first + i);
            else
                load_ray(P.rays_in, i, PROBE ? P.lean_probe_total : P.n_rays, planes_in, cur);
        }
        const double wl0 = cur.wl;
        const double wl_rcp = xm::refine_rcp(wl0);
        int row = 0;
        bool listed = true;
        if (USE_TABLE) {
            row = P.n_wl;
            const long long bits = __double_as_longlong(wl0);
#pragma unroll 1
            for (int k = 0; k < P.n_wl; k++)
                if (__double_as_longlong(P.wl[k]) == bits) row = k;
            listed = row != P.n_wl;              // NaN and unlisted wavelengths take the careful route
        }
        const double *pair = s_pair + 2 * row * n_med;
        // The lean and optimistic steps assume finite geometry and a wavelength in [2^-100, 2^100] (then no phase
        // quotient can leave the normal range); anything else is the careful route's business.
        auto non_finite = [](double v) { return (__double2hiint(v) & 0x7ff00000) == 0x7ff00000; };
        const unsigned wl_exp = ((unsigned)__double2hiint(wl0) >> 20) & 0x7ffu;
        const bool fit = valid && listed && (wl_exp - 923u <= 200u) &&
                         !(non_finite(cur.ox) | non_finite(cur.oy) | non_finite(cur.oz) | non_finite(cur.dx) |
                           non_finite(cur.dy) | non_finite(cur.dz) | non_finite(cur.ph));
        bool failed = valid && !fit;             // to be re-traced by redo_ray
        bool alive = fit;
        bool sampled = false, at_valid = false;
        lean::State r = {cur.ox, cur.oy, cur.oz, cur.dx, cur.dy, cur.dz, cur.ph};
        double n1 = 0.0;
        if (!USE_TABLE) n1 = eval_index(P.mat[0], wl0);

        if (!PROBE) {
            // ---- the hot loop: warp-convergent from top to bottom.  Every lane runs every surface -- a dead or failed
            // ray's lane computes on with whatever it holds (nothing it computes is used; it has no side effects) -- so
            // the loop index is warp-uniform where the compiler can see it and the prescription is read through the
            // uniform datapath / constant bank instead of vector registers.  Whole warps of dead rays leave early.
            // (each run's loop has its own induction variable, defined from kernel parameters only: the general steps
            // branch on values loaded through theirs, which makes it a vector register; the lean loops' stay uniform)
            for (int run = 0; run < P.lean_n_runs; run++) {
                const int begin = run > 0 ? P.lean_run_end[run - 1] : 0;
                const int end = P.lean_run_end[run];
                // (a run is "clean" when the probe left every surface of it on the launcher's step)
                // (an overridden run goes through the loop that dispatches per surface)
                const int code = (KINDS >= 2 || s_c.run_clean[run]) ? P.lean_run_code[run] : kMixedRun;
                if (code == kLeanSphere) {
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;      // (the surface that would have been sampled is not reached)
                            break;
                        }
                        if (USE_TABLE) {
                            n1 = pair[0];
                            pair += 2;
                        }
                        const double n2 = USE_TABLE ? 0.0 : eval_index(P.mat[k + 1], wl0);
                        const double ratio = USE_TABLE ? pair[-1] : xm::div(n1, n2);
                        bool ok = true, kill;
                        const bool on = lean::sphere_axial(ok, P.surf[k], s_c.surf[k].rcp, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if (code == kLeanFlat) {
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;      // (the surface that would have been sampled is not reached)
                            break;
                        }
                        if (USE_TABLE) {
                            n1 = pair[0];
                            pair += 2;
                        }
                        const double n2 = USE_TABLE ? 0.0 : eval_index(P.mat[k + 1], wl0);
                        const double ratio = USE_TABLE ? pair[-1] : xm::div(n1, n2);
                        bool ok = true, kill;
                        const bool on = lean::flat_axial<false>(ok, P.surf[k], r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if (KINDS >= 2 && code == kLeanFlatZ) {
                    // (pure kernels only: the zero-tolerant on-axis flat where the cached verdict asks for it; the
                    // probe-driven kernels reach this step through their dispatching loop)
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;
                            break;
                        }
                        if (USE_TABLE) {
                            n1 = pair[0];
                            pair += 2;
                        }
                        const double n2 = USE_TABLE ? 0.0 : eval_index(P.mat[k + 1], wl0);
                        const double ratio = USE_TABLE ? pair[-1] : xm::div(n1, n2);
                        bool ok = true, kill;
                        const bool on = lean::flat_axial<true>(ok, P.surf[k], r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if ((KINDS == 1 || KINDS == 3) && code == kLeanFlatAny) {
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;
                            break;
                        }
                        if (USE_TABLE) {
                            n1 = pair[0];
                            pair += 2;
                        }
                        const double n2 = USE_TABLE ? 0.0 : eval_index(P.mat[k + 1], wl0);
                        const double ratio = USE_TABLE ? pair[-1] : xm::div(n1, n2);
                        bool ok = true, kill;
                        const bool on = lean::flat_any(ok, P.surf[k], r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if ((KINDS == 1 || KINDS == 3) && code == kLeanLens) {
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;
                            break;
                        }
                        double n2;
                        if (USE_TABLE) {
                            n1 = pair[0];
                            n2 = pair[2];
                            pair += 2;
                        } else {
                            n2 = eval_index(P.mat[k + 1], wl0);
                        }
                        bool ok = true;
                        const bool on = lean::lens_any(ok, P.surf[k], s_c.surf[k].rcp, r, n1, n2, wl0, wl_rcp);
                        failed = failed | (alive & !ok);
                        at_valid = false;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if (KINDS == 1 && code == kGeneralLens) {
                    // a run of perfect lenses: its own loop, so that the hot code of a lens train (the OPM: 4f relays of
                    // perfect lenses and flats) is this step and the flats' -- not every step the kernel knows
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;
                            break;
                        }
                        const DevSurface &s = P.surf[k];
                        const SurfaceShared ss = s_c.surf[k];
                        double ratio, n2;
                        if (USE_TABLE) {
                            n1 = pair[0];
                            ratio = pair[1];
                            n2 = pair[2];
                            pair += 2;
                        } else {
                            n2 = eval_index(P.mat[k + 1], wl0);
                            ratio = xm::div(n1, n2);
                        }
                        bool ok = true, kill;
                        const bool on = general_step(s, kGeneralLens, ss.rcp, ss.rcp_ok != 0, r, n1, n2, ratio, wl0, wl_rcp, ok, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if (KINDS < 2 && code == kGeneralRefracting) {
                    // tilted / decentred flats and spheres, or ones the launcher keeps off the lean steps
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;
                            break;
                        }
                        const DevSurface &s = P.surf[k];
                        const SurfaceShared ss = s_c.surf[k];
                        double ratio, n2 = 0.0;
                        if (USE_TABLE) {
                            n1 = pair[0];
                            ratio = pair[1];
                            pair += 2;
                        } else {
                            n2 = eval_index(P.mat[k + 1], wl0);
                            ratio = xm::div(n1, n2);
                        }
                        bool ok = true, kill;
                        const bool on = general_step(s, kGeneralRefracting, ss.rcp, ss.rcp_ok != 0, r, n1, n2, ratio, wl0, wl_rcp, ok, kill);
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                } else if (KINDS < 2) {
                    for (int k = begin; k < end; k++) {
                        if (!__any_sync(0xffffffffu, alive)) {
                            at_valid = false;      // (the surface that would have been sampled is not reached)
                            break;
                        }
                        const DevSurface &s = P.surf[k];
                        const SurfaceShared ss = s_c.surf[k];
                        double ratio, n2 = 0.0;
                        if (USE_TABLE) {
                            n1 = pair[0];
                            ratio = pair[1];
                            n2 = pair[2];
                            pair += 2;
                        } else {
                            n2 = eval_index(P.mat[k + 1], wl0);
                            ratio = xm::div(n1, n2);
                        }
                        bool ok = true, kill;
                        bool on;
                        if (ss.code == kLeanSphere) {
                            on = lean::sphere_axial(ok, s, ss.rcp, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        } else if (ss.code == kLeanFlat) {
                            on = lean::flat_axial<false>(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        } else if (ss.code == kLeanFlatZ) {
                            on = lean::flat_axial<true>(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        } else if (KINDS == 1 && ss.code == kLeanFlatAny) {
                            on = lean::flat_any(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                        } else if (KINDS == 1 && ss.code == kLeanLens) {
                            on = lean::lens_any(ok, s, ss.rcp, r, n1, n2, wl0, wl_rcp);
                            kill = false;
                        } else {
                            // (KINDS = 0: the launcher has made sure that only refracting surfaces get here)
                            on = general_step(s, KINDS == 1 ? ss.code : (int)kGeneralRefracting, ss.rcp, ss.rcp_ok != 0, r, n1,
                                              n2, ratio, wl0, wl_rcp, ok, kill);
                        }
                        failed = failed | (alive & !ok);
                        at_valid = alive & ok & !kill;
                        alive = alive & ok & on;
                        if (!USE_TABLE) n1 = n2;
                    }
                }
                // the sample: the slab after the run's last surface, or (odd slab) the one at it -- whose position and
                // phase the step has left in the ray, valid unless the ray was culled there
                if (run == P.lean_sample_run && (sample_at ? at_valid : alive)) {
                    accumulate(red, r.ox, r.oy, r.oz, r.ph, s_tally);
                    sampled = true;
                }
            }
        } else {
            // ---- the probe: per-surface recovery, so that every surface is probed with the rays that really reach it
            for (int k = 0; k < P.n_surf; k++) {
                if (!alive) break;
                const DevSurface &s = P.surf[k];
                const SurfaceShared ss = s_c.surf[k];
                const int code = ss.code;
                double ratio, n2;
                if (USE_TABLE) {
                    n1 = pair[0];
                    ratio = pair[1];
                    n2 = pair[2];
                    pair += 2;
                } else {
                    n2 = eval_index(P.mat[k + 1], wl0);
                    ratio = xm::div(n1, n2);
                }
                const lean::State before = r;
                bool ok = true, on, kill;
                if (code == kLeanSphere)
                    on = lean::sphere_axial(ok, s, ss.rcp, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                else if (code == kLeanFlat)
                    on = lean::flat_axial<false>(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                else if (code == kLeanFlatZ)
                    on = lean::flat_axial<true>(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                else if (code == kLeanFlatAny)
                    on = lean::flat_any(ok, s, r, n1, ratio, wl0, wl_rcp, s_c.near_one, kill);
                else if (code == kLeanLens)
                    on = lean::lens_any(ok, s, ss.rcp, r, n1, n2, wl0, wl_rcp);
                else
                    on = general_step(s, code, ss.rcp, ss.rcp_ok != 0, r, n1, n2, ratio, wl0, wl_rcp, ok, kill);
                atomicAdd(my_counts + 2 * k, 1u);
                if (!ok) {
                    atomicAdd(my_counts + 2 * k + 1, 1u);
                    Ray in;
                    in.ox = before.ox; in.oy = before.oy; in.oz = before.oz;
                    in.dx = before.dx; in.dy = before.dy; in.dz = before.dz;
                    in.ph = before.ph; in.wl = wl0;
                    StepResult res;
                    if (s.kind == RTB_SURF_FLAT || s.kind == RTB_SURF_SPHERE)
                        res = careful_refracting(&s, in, n1, ratio, true);
                    else if (s.kind == RTB_SURF_MIRROR)
                        res = careful_mirror(&s, in, n1);
                    else
                        res = careful_lens(&s, in, n1, n2, false);
                    r.ox = res.after.ox; r.oy = res.after.oy; r.oz = res.after.oz;
                    r.dx = res.after.dx; r.dy = res.after.dy; r.dz = res.after.dz;
                    r.ph = res.after.ph;
                    on = !res.dead;
                }
                alive = on;
                if (!USE_TABLE) n1 = n2;
            }
        }
        if (PROBE) continue;

        Ray out;
        out.ox = r.ox; out.oy = r.oy; out.oz = r.oz; out.dx = r.dx; out.dy = r.dy; out.dz = r.dz; out.ph = r.ph;
        out.wl = wl0;
        if (!alive) set_nan(out);
        if (failed) {
            // start over from the launch state (reloaded: it was not kept in registers)
            // (`redone`, not `out`, goes to the call: a row whose address is taken lives in local memory, for every ray)
            Ray launch, sample, redone;
            if (FROM_SOURCE)
                launch = make_ray(source, source.first + i);
            else
                load_ray(P.rays_in, i, P.n_rays, planes_in, launch);
            redo_ray<USE_TABLE>(&P, launch, k_red, sample_at, &redone, &sample);
            out = redone;
            if (reducing && !sampled) accumulate(red, sample.ox, sample.oy, sample.oz, sample.ph, s_tally);
        }
        if (valid && P.any_store) store_ray(P.out, row0 + i, out_rows, planes_out, out);
    }
    if (reducing) flush_tally(red, s_tally);
}

// systems of spheres and on-axis flats only
bool refracting_only(const TraceParams &P)
{
    for (int k = 0; k < P.n_surf; k++) {
        const DevSurface &s = P.surf[k];
        if (!(s.kind == RTB_SURF_SPHERE || (s.kind == RTB_SURF_FLAT && s.z_axis != 0 && s.z_normal != 0))) return false;
    }
    return true;
}

template <bool T, bool S, bool W, bool PR>
cudaError_t launch_lean_one(const TraceParams &P, unsigned blocks, unsigned n_y, unsigned *probe_counts, cudaStream_t stream)
{
    size_t dyn = T ? 2 * sizeof(double) * (size_t)(P.n_wl + 1) * (size_t)(P.n_surf + 1) : 0;
    if (!PR && P.red.slab >= 0 && P.red.stats) dyn += sizeof(double) * 12 * kLeanThreads;
    const bool pure = !PR && P.lean_pure != 0;
    // With lazy module loading (the CUDA default) a kernel is loaded at its first launch, which stalls the host for
    // milliseconds with the GPU idle -- and the verdict cache launches the pure instantiations for the first time in the
    // middle of a run of launches.  Load the whole family when its first member is launched.
    static const bool loaded = [] {
        cudaFuncAttributes a;
        cudaFuncGetAttributes(&a, trace_lean_kernel<T, S, W, false, 0>);
        cudaFuncGetAttributes(&a, trace_lean_kernel<T, S, W, false, 1>);
        cudaFuncGetAttributes(&a, trace_lean_kernel<T, S, W, false, 2>);
        cudaFuncGetAttributes(&a, trace_lean_kernel<T, S, W, false, 3>);
        cudaFuncGetAttributes(&a, trace_lean_kernel<T, S, W, true, 1>);
        cudaGetLastError();
        return true;
    }();
    (void)loaded;
    if (pure && refracting_only(P))
        trace_lean_kernel<T, S, W, false, 2><<<dim3(blocks, n_y), kLeanThreads, dyn, stream>>>(P, probe_counts);
    else if (pure)
        trace_lean_kernel<T, S, W, false, 3><<<dim3(blocks, n_y), kLeanThreads, dyn, stream>>>(P, probe_counts);
    else if (!PR && refracting_only(P))
        trace_lean_kernel<T, S, W, PR, 0><<<dim3(blocks, n_y), kLeanThreads, dyn, stream>>>(P, probe_counts);
    else
        trace_lean_kernel<T, S, W, PR, 1><<<dim3(blocks, n_y), kLeanThreads, dyn, stream>>>(P, probe_counts);
    return cudaGetLastError();
}

template <bool PR>
cudaError_t launch_lean_pick(const TraceParams &P, unsigned blocks, unsigned *probe_counts, cudaStream_t stream)
{
    const bool table = P.n_wl > 0, source = P.src.kind >= 0, sweep = P.n_src > 0;
    const unsigned n_y = sweep ? (unsigned)P.n_src : 1u;
#ifdef RTB_LEAN_ONLY_ONE   // experiments: one instantiation, seconds to compile
    return launch_lean_one<true, false, false, PR>(P, blocks, 1, probe_counts, stream);
#endif
    if (sweep)
        return table ? launch_lean_one<true, true, true, PR>(P, blocks, n_y, probe_counts, stream)
                     : launch_lean_one<false, true, true, PR>(P, blocks, n_y, probe_counts, stream);
    if (table)
        return source ? launch_lean_one<true, true, false, PR>(P, blocks, 1, probe_counts, stream)
                      : launch_lean_one<true, false, false, PR>(P, blocks, 1, probe_counts, stream);
    return source ? launch_lean_one<false, true, false, PR>(P, blocks, 1, probe_counts, stream)
                  : launch_lean_one<false, false, false, PR>(P, blocks, 1, probe_counts, stream);
}

} // namespace

// share of surfaces with a lean step below which a system stays with trace_f64.cu (rtb_tune "lean_min_share_pct")
int g_lean_min_share_pct = 75;
void set_lean_min_share_pct(int pct) { g_lean_min_share_pct = pct; }

// What the lean kernel traces: fp64 exact, nothing stored but the final slab (or nothing at all), no reduction or one at
// an after-surface slab, not the intersect-only operator.
bool lean_eligible(const TraceParams &P)
{
    if (P.flags & RTB_FLAG_INTERSECT_ONLY) return false;
    if (P.any_store && !P.store_last_only) return false;
    if (P.red.slab == 0) return false;                       // the launch rays themselves: nothing to trace for
    // (an odd slab is the one AT a surface: the steps leave its position and phase in the ray -- except a perfect lens,
    // whose "at" slab is a fourth plane propagation)
    if (P.red.slab > 0 && (P.red.slab & 1) != 0 && P.surf[(P.red.slab - 1) >> 1].kind == RTB_SURF_PERFECT_LENS) return false;
    // worth it when most surfaces have a lean step (on-axis spheres and flats); trains of perfect lenses, mirrors and
    // tilted surfaces stay with trace_f64.cu, whose loops are built around the general steps
    int n_lean = 0;
    for (int k = 0; k < P.n_surf; k++) {
        const DevSurface &s = P.surf[k];
        n_lean += has_lean_step(s);
    }
    if (100 * n_lean < g_lean_min_share_pct * P.n_surf) return false;
    if (P.red.slab < 0 && !P.any_store) return false;      // nothing to do: leave it to the general kernel's conventions
    return P.n_surf > 0;
}

// The probe's rule, for the host: bit k is set when more than 1 in kProbeOneIn of the probe rays that reached surface k
// failed their lean step there, in any source (`counts`: n_src x kMaxSurfaces x {reached, failed}, the probe's output).
unsigned long long lean_verdict_from_counts(const unsigned *counts, int n_src, int n_surf)
{
    unsigned long long general = 0ull;
    for (int j = 0; j < n_src; j++)
        for (int k = 0; k < n_surf; k++) {
            const unsigned *cnt = counts + ((size_t)j * kMaxSurfaces + k) * 2;
            if ((unsigned long long)cnt[1] * kProbeOneIn > (unsigned long long)cnt[0]) general |= 1ull << k;
        }
    return general;
}

namespace {
bool sane_reciprocal(const DevSurface &s)
{
    const double den = (s.kind == RTB_SURF_PERFECT_LENS) ? s.focal_len : s.radius;
    const bool needs_rcp = s.kind == RTB_SURF_SPHERE || s.kind == RTB_SURF_PERFECT_LENS;
    return !needs_rcp || (std::isfinite(den) && fabs(den) > 1e-150 && fabs(den) < 4503599627370496.0);
}

// runs of equal step codes, split where the reduction samples; `general`: surfaces kept off their plain lean step.
// Returns whether every surface ended up on a lean step.
bool build_runs(TraceParams &P, unsigned long long general)
{
    const int k_red = P.red.slab >= 0 ? (P.red.slab - 1) >> 1 : -1;
    bool all_lean = P.n_surf > 0;
    P.lean_n_runs = 0;
    P.lean_sample_run = -1;
    int prev = -1;
    for (int k = 0; k < P.n_surf; k++) {
        const DevSurface &s = P.surf[k];
        const int code = step_code(s, ((general >> k) & 1ull) != 0 || !sane_reciprocal(s));
        all_lean &= code < kGeneralRefracting || code > kMixedRun;
        if (code != prev) P.lean_n_runs++;
        P.lean_run_code[P.lean_n_runs - 1] = (uint8_t)code;
        P.lean_run_end[P.lean_n_runs - 1] = (uint8_t)(k + 1);
        prev = code;
        if (k == k_red) {
            P.lean_sample_run = P.lean_n_runs - 1;
            prev = -1;
        }
    }
    return all_lean;
}
} // namespace

// `counts`: device scratch of n_sources * kMaxSurfaces * 2 unsigned for the probe (zeroed here), owned by the caller for
// the duration of both launches.  *launches is increased by the number of kernels launched.
// `pure_mode` 0: the probe-driven kernels.  1: the pure kernels, if the system allows, with `verdict_general` = the
// surfaces at which an EARLIER probe of the same system and bundle found bundle-wide failures of the plain lean step
// (rtb_api.cu's cache; on-axis flats among them run the zero-tolerant lean flat, anything else sends the launch back to the
// probe-driven kernels).  2: the pure kernels with no verdict (tests: whatever fails is re-traced by redo_ray).  The probe
// runs in every mode but one (see probe_optional) -- in the pure modes its counts only feed the caller's next verdict.
// *pure_used says what ran.
// `probe_optional`: the verdict is final for this launch (rays that are a pure function of the cache key): when the pure
// kernels take it, the probe -- which would only confirm it -- is not launched.  *probed says whether it was.
cudaError_t launch_trace_lean(const TraceParams &P_in, unsigned *counts, int sm_count, cudaStream_t stream, int *launches,
                              int pure_mode, unsigned long long verdict_general, bool *pure_used, bool probe_optional,
                              bool *probed)
{
    if (pure_used) *pure_used = false;
    if (probed) *probed = false;
    if (P_in.n_rays <= 0) return cudaSuccess;
    TraceParams P = P_in;
    const bool sweep = P.n_src > 0;
    const int n_sources = sweep ? P.n_src : 1;
    // surfaces without a lean step (tilted / decentred axes, mirrors, lenses) run the general steps
    P.lean_general = 0ull;
    for (int k = 0; k < P.n_surf; k++) {
        const DevSurface &s = P.surf[k];
        if (!has_lean_step(s)) P.lean_general |= 1ull << k;
    }
    P.lean_pure = 0;
    if (pure_mode != 0 && P.lean_general == 0ull && build_runs(P, pure_mode == 1 ? verdict_general : 0ull))
        P.lean_pure = 1;
    else
        build_runs(P, P.lean_general);
    if (pure_used) *pure_used = P.lean_pure != 0;
    if (P.lean_pure != 0 && probe_optional) counts = nullptr;
    if (probed) *probed = counts != nullptr;
    cudaError_t e;
    P.lean_counts = nullptr;
    if (counts) {
        e = cudaMemsetAsync(counts, 0, sizeof(unsigned) * 2 * kMaxSurfaces * (size_t)n_sources, stream);
        if (e != cudaSuccess) return e;
        TraceParams Q = P;
        const long long n_probe = P.n_rays < kProbeRays ? P.n_rays : kProbeRays;
        Q.lean_probe_total = P.n_rays;
        Q.lean_probe_stride = P.n_rays / n_probe;
        Q.n_rays = n_probe;
        Q.red.slab = -1;
        Q.any_store = 0;
        const unsigned pb = (unsigned)((n_probe + kLeanThreads - 1) / kLeanThreads);
        e = launch_lean_pick<true>(Q, pb, counts, stream);
        if (e != cudaSuccess) return e;
        if (launches) ++*launches;
        P.lean_counts = counts;
    }
    long long blocks = (P.n_rays + kLeanThreads - 1) / kLeanThreads;
    long long max_blocks = (long long)sm_count * kLeanMinBlocks * 4;
    if (sweep) max_blocks = (max_blocks + P.n_src - 1) / P.n_src;
    if (blocks > max_blocks) blocks = max_blocks;
    e = launch_lean_pick<false>(P, (unsigned)blocks, nullptr, stream);
    if (e == cudaSuccess && launches) ++*launches;
    return e;
}

} // namespace rtb
