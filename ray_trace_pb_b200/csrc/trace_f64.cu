// trace_f64.cu -- the fused fp64 sequential trace: one thread carries one ray in registers through every surface.
//
// Replaces the Python loop of System.ray_trace (reference raytrace.py:641-661) and the whole-array NumPy bodies
// of RefractingSurface.propagate (1160-1234), ReflectingSurface.propagate (1238-1303), PerfectLens.propagate
// (1601-1801), propagate_ray2plane (241-306), SphericalSurface.get_intersect / get_normal / is_pt_on_surface
// (1467-1535), FlatSurface / PlaneMirror geometry (1323-1347, 1392-1412) and Material.n (materials.py:39-51).
//
// THIS TRANSLATION UNIT MUST BE COMPILED WITH -fmad=false.
// The fp64 mode promises results bit-identical to the NumPy path (values and NaN masks), because the reference's
// validity tests use an absolute 1e-12 tolerance that flips on last-bit differences (SURVEY.md section 0).  That
// needs every + - * rounded on its own (no FMA contraction), 3-term sums associated left to right, IEEE / and
// sqrt, and NaN-aware selects written in the reference's polarity.  Only value-preserving rewrites are used:
//   * x*2*pi == x*(2*pi) (scaling by 2 is exact); norm*(+-1) done as a sign flip; sqrt(disc) evaluated once;
//   * n(lambda) looked up / evaluated once per medium per ray, n1/n2 taken from a host-divided table;
//   * divisions by one denominator share the Newton-refined reciprocal (exact_math.cuh: same bits as IEEE `/`);
//   * `norm <= aperture` and `|norm - |R|| < 1e-12` are tested on the squared sum against host-computed exact
//     thresholds (monotonicity of the correctly rounded sqrt), so those square roots are never taken;
//   * the NaN fills of culled rays are applied once, where a slab is stored or feeds the next surface;
//   * each surface runs branch-free ("Optimistic") with one domain flag and is redone by the self-checking
//     ("Careful") instantiation when the flag fails; terms multiplied by the exact zeros of a z-aligned normal or
//     axis are dropped when all operands are known finite (surface_steps.cuh).
#include <cmath>
#include <type_traits>
#include <math_constants.h>

#include "exact_math.cuh"
#include "rtb_device.cuh"
#include "surface_steps.cuh"
#include "trace_common.cuh"

#ifndef RTB_TU_VARIANT
#define RTB_TU_VARIANT 0
#endif

namespace rtb {

namespace {

// per-block shared prescription-derived constants
struct SharedConsts {
    double rcp_radius[kMaxSurfaces]; // refined 1/R per spherical surface (1/f for perfect lenses)
    unsigned long long rcp_ok;       // bit k: that reciprocal is usable by the Optimistic steps (see below)
};

struct RayLoop {       // the loop-carried state of one ray
    Ray cur;
    double n1, n2;     // refractive index before / after the current surface
    double wl0;        // launch wavelength
    xm::Rcp rcp_wl;
    int row;           // this ray's row of the index tables (times the number of media)
    bool unlisted;     // valid wavelength that the host table does not list
    bool dead;
    bool force_careful;
};

// the refractive index after surface kk
template <bool USE_TABLE>
__device__ __forceinline__ double index_after(const TraceParams &P, const double *s_ntab, int kk, const RayLoop &st)
{
    return !USE_TABLE ? eval_index(P.mat[kk + 1], st.wl0)
                      : (st.unlisted ? index_for_unlisted(&P.mat[kk + 1], st.wl0) : s_ntab[st.row + kk + 1]);
}

// 1/R (1/f for a perfect lens) of surface kk
__device__ __forceinline__ xm::Rcp radius_rcp(const DevSurface &s, const SharedConsts &s_c, int kk)
{
    xm::Rcp r;
    r.b = (s.kind == RTB_SURF_PERFECT_LENS) ? s.focal_len : s.radius;
    r.y = s_c.rcp_radius[kk];
    r.ok = (s_c.rcp_ok >> kk) & 1ull;
    return r;
}

// One surface with nothing to keep.  It runs optimistically; one flag says whether every intermediate stayed in the fast
// paths' domain, otherwise the surface is redone with the Careful arithmetic (surface_steps.cuh).  (Each kind's redo
// sits in its own branch: one careful_step after the branches costs the final-slab kernels 34 FP64 instructions and
// spill traffic.)
// A FUNCTION: it must be inlined at every call site -- out of line, the prescription would be read through generic
// pointers into the parameter block, at half the speed -- and only functions can be forced.
template <class OPT, bool USE_TABLE, bool INTERSECT_ONLY>
__device__ __forceinline__ void plain_surface_step(const TraceParams &P, const double *s_ntab, const double *s_ratio,
                                                   const SharedConsts &s_c, int kk, RayLoop &st)
{
    const DevSurface &s = P.surf[kk];
    st.n2 = index_after<USE_TABLE>(P, s_ntab, kk, st);
    const xm::Rcp rcp_k = radius_rcp(s, s_c, kk);
    OPT m;
    m.ok = !st.force_careful;
    st.force_careful = false;
    AtRaw raw;
    Ray after;
    if (s.kind == RTB_SURF_FLAT || s.kind == RTB_SURF_SPHERE) {
        const double ratio = (USE_TABLE && !st.unlisted) ? s_ratio[st.row + kk] : xm::div(st.n1, st.n2);
        st.dead = refracting_step<OPT, false>(m, s, st.cur, st.n1, ratio, st.rcp_wl, rcp_k, !INTERSECT_ONLY, raw, after);
        if (!m.ok) {
            const StepResult redo = careful_refracting(&s, st.cur, st.n1, ratio, !INTERSECT_ONLY);
            after = redo.after;
            st.dead = redo.dead;
        }
    } else if (s.kind == RTB_SURF_MIRROR) {
        st.dead = mirror_step<OPT, false>(m, s, st.cur, st.n1, st.rcp_wl, raw, after);
        if (!m.ok) {
            const StepResult redo = careful_mirror(&s, st.cur, st.n1);
            after = redo.after;
            st.dead = redo.dead;
        }
    } else {
        st.dead = perfect_lens_step<OPT>(m, s, st.cur, st.n1, st.n2, st.rcp_wl, rcp_k, INTERSECT_ONLY, false, raw, after);
        if (!m.ok) {
            const StepResult redo = careful_lens(&s, st.cur, st.n1, st.n2, INTERSECT_ONLY);
            after = redo.after;
            st.dead = redo.dead;
        }
    }
    st.cur = after;
    st.n1 = st.n2;
}

// ---- the kernel --------------------------------------------------------------------------------------------
// USE_TABLE   refractive indices (and n1/n2) from the host table (any material), else in-register Sellmeier.
// FROM_SOURCE rays are produced by the on-device source instead of being read from memory.
// MODE        0: only the final slab is stored; 1: general (any slab selection, fused reductions); 2: general, as a
//             sweep over P.n_src sources (FROM_SOURCE only): blockIdx.y picks the source, its output rows and its
//             reduction bucket; 3: general with RTB_FLAG_INTERSECT_ONLY (Surface.get_intersect: no front-side cull);
//             4: the final slab (or nothing) is stored and ONE after-surface slab is reduced -- the pupil-grid /
//             spot-statistics workload -- on the final-slab kernel's loop, run in two legs around the sample.
// VARIANT     0: the plain hot loop (Optimistic); 1: the launch carries surface hints (rtb_surface.hints): the hot loop
//             runs on OptimisticFlatZ; 2: every normal / axis of the system is exactly +-z: OptimisticAxial.
template <bool USE_TABLE, bool FROM_SOURCE, int MODE, int VARIANT>
__global__ void __launch_bounds__(kTraceThreads, kTraceMinBlocks) trace_f64_kernel(const __grid_constant__ TraceParams P)
{
    using Optimistic = std::conditional_t<VARIANT == 1, OptimisticFlatZ,
                                          std::conditional_t<VARIANT == 2, OptimisticAxial, rtb::Optimistic>>;
    constexpr bool FINAL_RED = MODE == 4;
    constexpr bool GENERAL = MODE >= 1 && MODE <= 3;
    constexpr bool SWEEP = MODE == 2;
    static_assert(!SWEEP || FROM_SOURCE, "sweeps generate their rays");
    // the index tables are sized at launch ((n_wl + 1) * (n_surf + 1) doubles each, typically a few hundred bytes):
    // shared memory comes out of the L1 that the kernel's spill slots live in
    extern __shared__ double s_tables[];
    double *const s_ntab = s_tables;
    double *const s_ratio = s_tables + (USE_TABLE ? (P.n_wl + 1) * (P.n_surf + 1) : 0);
    __shared__ SharedConsts s_c;
    __shared__ SweepShared<SWEEP> s_sweep;
    if (SWEEP) sweep_setup(P, s_sweep);     // visible after the first __syncthreads below
    const int n_med = P.n_surf + 1;
    if (USE_TABLE) {
        const int count = (P.n_wl + 1) * n_med;
        for (int k = threadIdx.x; k < count; k += blockDim.x) {
            s_ntab[k] = P.n_tab[k];
            s_ratio[k] = P.ratio_tab[k];
        }
    }
    if (threadIdx.x == 0) s_c.rcp_ok = 0ull;
    __syncthreads();
    for (int k = threadIdx.x; k < P.n_surf; k += blockDim.x) {
        const DevSurface &s = P.surf[k];
        const double den = (s.kind == RTB_SURF_PERFECT_LENS) ? s.focal_len : s.radius;
        s_c.rcp_radius[k] = xm::refine_rcp(den);
        if (usable_rcp(den, s_c.rcp_radius[k])) atomicOr(&s_c.rcp_ok, 1ull << k);
    }
    __syncthreads();

    const DevSource &source = sweep_source(P, s_sweep);
    const DevReduce &red = sweep_reduce(P, s_sweep);
    const long long row0 = SWEEP ? (long long)blockIdx.y * P.n_rays : 0;
    const bool reducing = (GENERAL || FINAL_RED) && P.red.slab >= 0;
    // (a compile-time fact, not a flag test: the front-side cull it switches sits in the middle of every refracting
    // step, and a warp-uniform branch there splits the step's basic block -- 1.4 % of the general kernel, 4 % of the OPM)
    constexpr bool intersect_only = MODE == 3;
    Tally tally;
    if (GENERAL || FINAL_RED) tally_init(tally);

    const bool planes_in = (P.flags & RTB_FLAG_PLANES_IN) != 0, planes_out = (P.flags & RTB_FLAG_PLANES_OUT) != 0;
    const long long out_rows = P.out_stride / 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P.n_rays; i += stride) {
        Ray cur;
        if (FROM_SOURCE)
            cur = make_ray(source, source.first + i);
        else
            load_ray(P.rays_in, i, P.n_rays, planes_in, cur);

        // refractive indices are functions of the launch wavelength; see DESIGN.md ("n is taken at launch")
        RayLoop st;
        st.cur = cur;
        st.wl0 = cur.wl;
        st.rcp_wl = xm::make_rcp(st.wl0);
        st.row = 0;
        st.unlisted = false;
        if (USE_TABLE) {
            const int row = wavelength_row(P, st.wl0);
            // a valid wavelength the table does not list: evaluate Sellmeier / constant media for this ray
            st.unlisted = (row == P.n_wl) && (st.wl0 == st.wl0);
            st.row = row * n_med;
        }
        if (GENERAL) {
            if (P.slab_pos[0] >= 0) store_ray(P.out + P.slab_pos[0] * P.out_stride, row0 + i, out_rows, planes_out, cur);
            if (reducing && P.red.slab == 0) reduce_sample(red, cur, tally);
        }

        st.n1 = !USE_TABLE ? eval_index(P.mat[0], st.wl0)
                           : (st.unlisted ? index_for_unlisted(&P.mat[0], st.wl0) : s_ntab[st.row]);
        st.n2 = st.n1;
        // Live rays run the surface loop; a ray that dies (leaves a surface all-NaN) drops out of it and only has
        // its remaining slabs blanked below -- an all-NaN ray stays all-NaN through every kind of surface.
        st.dead = false;
        // The optimistic steps may assume finite geometry (that is what licenses their shortcuts), and inside a trace
        // it always is -- the reference blanks x, y, z together.  Only a ray that ARRIVES with an inf/NaN in some
        // position or direction column could break that, so such a ray takes the careful path at its first surface.
        st.force_careful = non_finite(cur.ox) | non_finite(cur.oy) | non_finite(cur.oz) | non_finite(cur.dx) |
                           non_finite(cur.dy) | non_finite(cur.dz);
        int k = 0;
        // act (uniform per surface): bit 0 store "at", 1 store "after", 2 reduce "at", 3 reduce "after"
        auto emit_after = [&](int kk, int act) {
            Ray out = st.cur;
            if (st.dead) set_nan(out); // the optimistic step leaves a culled ray's values un-blanked
            if (act & 2) store_ray(P.out + P.slab_pos[2 * kk + 2] * P.out_stride, row0 + i, out_rows, planes_out, out);
            if (act & 8) reduce_sample(red, out, tally);
        };
        // One surface whose "at" slab is stored or reduced.  (Each kind's redo sits in its own branch, as in
        // plain_surface_step: one careful_step after the branches costs the general kernel FP64 instructions and spills.)
        auto observed_surface = [&](int kk, int act) {
            const DevSurface &s = P.surf[kk];
            st.n2 = index_after<USE_TABLE>(P, s_ntab, kk, st);
            const xm::Rcp rcp_k = radius_rcp(s, s_c, kk);
            const bool need_at = (act & 5) != 0;
            auto emit_at = [&](const Ray &at) {
                if (act & 1) store_ray(P.out + P.slab_pos[2 * kk + 1] * P.out_stride, row0 + i, out_rows, planes_out, at);
                if (act & 4) reduce_sample(red, at, tally);
            };
            Optimistic m;
            m.ok = !st.force_careful;
            st.force_careful = false;
            AtRaw raw;
            Ray after;
            if (s.kind == RTB_SURF_FLAT || s.kind == RTB_SURF_SPHERE) {
                const double ratio = (USE_TABLE && !st.unlisted) ? s_ratio[st.row + kk] : xm::div(st.n1, st.n2);
                st.dead = refracting_step<Optimistic, true>(m, s, st.cur, st.n1, ratio, st.rcp_wl, rcp_k, !intersect_only,
                                                            raw, after);
                if (!m.ok) {
                    const StepResult redo = careful_refracting(&s, st.cur, st.n1, ratio, !intersect_only);
                    if (need_at) emit_at(redo.at);
                    after = redo.after;
                    st.dead = redo.dead;
                }
            } else if (s.kind == RTB_SURF_MIRROR) {
                st.dead = mirror_step<Optimistic, true>(m, s, st.cur, st.n1, st.rcp_wl, raw, after);
                if (!m.ok) {
                    const StepResult redo = careful_mirror(&s, st.cur, st.n1);
                    if (need_at) emit_at(redo.at);
                    after = redo.after;
                    st.dead = redo.dead;
                }
            } else {
                st.dead = perfect_lens_step<Optimistic>(m, s, st.cur, st.n1, st.n2, st.rcp_wl, rcp_k, intersect_only, need_at,
                                                        raw, after);
                if (!m.ok) {
                    const StepResult redo = careful_lens(&s, st.cur, st.n1, st.n2, intersect_only);
                    if (need_at) emit_at(redo.at);
                    after = redo.after;
                    st.dead = redo.dead;
                }
            }
            if (m.ok && need_at) {
                Ray at;
                fill_at(raw, st.cur, at);
                emit_at(at);
            }
            st.cur = after;
            st.n1 = st.n2;
        };
        if (FINAL_RED) {
            const int k_red = (P.red.slab - 2) >> 1;        // the sample is the slab after surface k_red
#pragma unroll 1
            for (; k <= k_red && !st.dead; k++) plain_surface_step<Optimistic, USE_TABLE, false>(P, s_ntab, s_ratio, s_c, k, st);
            if (!st.dead) reduce_sample(red, st.cur, tally);
#pragma unroll 1
            for (; k < P.n_surf && !st.dead; k++) plain_surface_step<Optimistic, USE_TABLE, false>(P, s_ntab, s_ratio, s_c, k, st);
        } else if (!GENERAL) {
            // two surfaces per trip: the ray's registers ping-pong between the two copies of the body instead of
            // being moved back at the end of every surface (+3 % here; the general mode's loop loses by it)
            for (; k < P.n_surf && !st.dead; k += 2) {
                plain_surface_step<Optimistic, USE_TABLE, false>(P, s_ntab, s_ratio, s_c, k, st);
                if (k + 1 < P.n_surf && !st.dead) plain_surface_step<Optimistic, USE_TABLE, false>(P, s_ntab, s_ratio, s_c, k + 1, st);
            }
        } else {
            // runs of surfaces whose "at" slab is not needed go through the same tight loop as the final-slab-only kernel
            while (k < P.n_surf && !st.dead) {
#pragma unroll 1
                for (; k < P.n_surf && !st.dead && (P.slab_act[k] & 5) == 0; k++) {
                    plain_surface_step<Optimistic, USE_TABLE, intersect_only>(P, s_ntab, s_ratio, s_c, k, st);
                    const int act = P.slab_act[k];
                    if (act & 10) emit_after(k, act);
                }
                if (k < P.n_surf && !st.dead) {
                    const int act = P.slab_act[k];
                    observed_surface(k, act);
                    if (act & 10) emit_after(k, act);
                    k++;
                }
            }
        }
        if (GENERAL && st.dead) {
            // blank what is left of a dead ray's history (reductions skip NaN samples, nothing to add there)
            Ray blank;
            set_nan(blank);
#pragma unroll 1
            for (; k < P.n_surf; k++) {
                const int act = P.slab_act[k];
                if (act & 1) store_ray(P.out + P.slab_pos[2 * k + 1] * P.out_stride, row0 + i, out_rows, planes_out, blank);
                if (act & 2) store_ray(P.out + P.slab_pos[2 * k + 2] * P.out_stride, row0 + i, out_rows, planes_out, blank);
            }
        }
        if (!GENERAL && (!FINAL_RED || P.any_store)) {
            if (st.dead) set_nan(st.cur);
            store_ray(P.out, i, out_rows, planes_out, st.cur);
        }
    }
    if ((GENERAL || FINAL_RED) && reducing) tally_flush(red, tally);
}

// MODE 4's shape: no sweep, no intersect-only, the final slab or nothing stored, one reduction at an after-surface slab
bool final_slab_plus_one_reduction(const TraceParams &P)
{
    return P.n_src == 0 && (P.flags & RTB_FLAG_INTERSECT_ONLY) == 0 && P.red.slab >= 2 && (P.red.slab & 1) == 0 &&
           (P.store_last_only || !P.any_store);
}

template <bool T, bool S, int M>
cudaError_t launch_one(const TraceParams &P, unsigned blocks, cudaStream_t stream)
{
    const size_t tables = T ? 2 * sizeof(double) * (size_t)(P.n_wl + 1) * (size_t)(P.n_surf + 1) : 0;
    const dim3 grid(blocks, M == 2 ? (unsigned)P.n_src : 1u);
    trace_f64_kernel<T, S, M, RTB_TU_VARIANT><<<grid, kTraceThreads, tables, stream>>>(P);
    return cudaGetLastError();
}

} // namespace

// launchers used by rtb_api.cu.  This file is compiled three times (Makefile): RTB_TU_VARIANT = 0 gives the plain kernels
// (and launch_trace_f64, which picks), 1 those of launches that carry surface hints, 2 the final-slab kernels (MODE 0
// and MODE 4) for systems whose every normal and axis is exactly +-z -- three translation units that build in parallel.
#if RTB_TU_VARIANT == 1
cudaError_t launch_trace_f64_hinted(const TraceParams &P, int sm_count, cudaStream_t stream)
#elif RTB_TU_VARIANT == 2
cudaError_t launch_trace_f64_axial(const TraceParams &P, int sm_count, cudaStream_t stream)
#else
cudaError_t launch_trace_f64_hinted(const TraceParams &P, int sm_count, cudaStream_t stream);
cudaError_t launch_trace_f64_axial(const TraceParams &P, int sm_count, cudaStream_t stream);
static cudaError_t launch_trace_f64_plain(const TraceParams &P, int sm_count, cudaStream_t stream);

cudaError_t launch_trace_f64(const TraceParams &P, int sm_count, cudaStream_t stream)
{
    bool hinted = false, axial = P.n_surf > 0;
    for (int k = 0; k < P.n_surf; k++) {
        const DevSurface &s = P.surf[k];
        hinted |= s.degenerate_hint != 0;
        // spheres use their axis only; flats also cull by it; mirrors and lenses use the normal only
        const bool needs_normal = s.kind != RTB_SURF_SPHERE, needs_axis = s.kind == RTB_SURF_SPHERE || s.kind == RTB_SURF_FLAT;
        axial &= (!needs_normal || s.z_normal != 0) && (!needs_axis || s.z_axis != 0);
    }
    if (hinted) return launch_trace_f64_hinted(P, sm_count, stream);
    // (only the final-slab kernel gains from the axial form: +2.8 %; the general kernel loses 1.7 % and keeps the plain one)
    const bool final_slab_only = P.n_src == 0 && P.store_last_only && P.red.slab < 0 && (P.flags & RTB_FLAG_INTERSECT_ONLY) == 0;
    if (axial && (final_slab_only || final_slab_plus_one_reduction(P))) return launch_trace_f64_axial(P, sm_count, stream);
    return launch_trace_f64_plain(P, sm_count, stream);
}

static cudaError_t launch_trace_f64_plain(const TraceParams &P, int sm_count, cudaStream_t stream)
#endif
{
    if (P.n_rays <= 0) return cudaSuccess;
    long long blocks = (P.n_rays + kTraceThreads - 1) / kTraceThreads;
    // a whole number of waves over the SMs, grid-stride inside
    long long max_blocks = (long long)sm_count * kTraceMinBlocks * 4;
    const bool sweep = P.n_src > 0;
    if (sweep) max_blocks = (max_blocks + P.n_src - 1) / P.n_src;   // the cap is for the whole grid
    if (blocks > max_blocks) blocks = max_blocks;
    const bool table = P.n_wl > 0;
    const bool source = P.src.kind >= 0;
#if RTB_TU_VARIANT != 2
    if (sweep && (P.flags & RTB_FLAG_INTERSECT_ONLY)) return cudaErrorNotSupported;   // (refused by rtb_trace_sources)
    if (sweep)
        return table ? launch_one<true, true, 2>(P, (unsigned)blocks, stream)
                     : launch_one<false, true, 2>(P, (unsigned)blocks, stream);
#endif
    const bool fast = P.store_last_only && P.red.slab < 0 && (P.flags & RTB_FLAG_INTERSECT_ONLY) == 0;
    const unsigned b = (unsigned)blocks;
#if RTB_TU_VARIANT == 2
    // (measured: +6 % on axial systems; on tilted or hinted ones the general kernel is 5 % faster and keeps the job)
    if (final_slab_plus_one_reduction(P)) {
        if (table) return source ? launch_one<true, true, 4>(P, b, stream) : launch_one<true, false, 4>(P, b, stream);
        return source ? launch_one<false, true, 4>(P, b, stream) : launch_one<false, false, 4>(P, b, stream);
    }
#endif
    if (fast) {
        if (table) return source ? launch_one<true, true, 0>(P, b, stream) : launch_one<true, false, 0>(P, b, stream);
        return source ? launch_one<false, true, 0>(P, b, stream) : launch_one<false, false, 0>(P, b, stream);
    }
#if RTB_TU_VARIANT != 2
    if (P.flags & RTB_FLAG_INTERSECT_ONLY) {
        if (table) return source ? launch_one<true, true, 3>(P, b, stream) : launch_one<true, false, 3>(P, b, stream);
        return source ? launch_one<false, true, 3>(P, b, stream) : launch_one<false, false, 3>(P, b, stream);
    }
    if (table) return source ? launch_one<true, true, 1>(P, b, stream) : launch_one<true, false, 1>(P, b, stream);
    return source ? launch_one<false, true, 1>(P, b, stream) : launch_one<false, false, 1>(P, b, stream);
#else
    return cudaErrorInvalidValue;   // the axial translation unit only carries the final-slab kernels
#endif
}

} // namespace rtb
