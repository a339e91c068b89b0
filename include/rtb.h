/*
 * rtb.h -- C ABI of librtb.so, the B200 (sm_100a) batch ray tracer behind the `raytrace.raytrace` Python API.
 *
 * The reference (QI2lab/ray_trace_pb) has no FFI of its own: its boundary is the Python call
 *     System.ray_trace(rays, initial_material, final_material)            src/raytrace/raytrace.py:641-661
 * which loops `surface.propagate(...)` (raytrace.py:1160-1234, 1238-1303, 1601-1801) over whole NumPy arrays.
 * Every entry point below replaces one such Python-level operator; the reference lines it stands in for are cited
 * next to it.  Bindings: plain pointers and sizes only, no torch / numpy types.  INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - A ray is 8 contiguous doubles (x, y, z, dx, dy, dz, phase[rad], wavelength[um])      raytrace.py:1-5
 *   - Ray batches are row-major (N, 8); histories are (n_slabs, N, 8).
 *   - Slab index j of a trace through S surfaces: 0 = launch rays, 2k+1 = at surface k, 2k+2 = just after surface k.
 *   - Numerical invalidity is in-band NaN, never an error code (raytrace.py:303-304, 1192, 1221, 1226, 1760).
 *   - Return value: 0 on success; negative rtb_status for structural problems (mapped to ValueError /
 *     NotImplementedError / RuntimeError by the Python host).  rtb_last_error() gives the text (thread local).
 *   - "dev" pointers are CUDA device pointers on the given device; "host" pointers are ordinary host memory.
 *   - The caller owns every buffer.  The library never frees or writes its inputs.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device entry points only enqueue
 *     work; host entry points return after the results are in the host buffers.
 *   - There is no CPU fallback anywhere in this library.
 */
#ifndef RTB_H
#define RTB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_ABI_VERSION 5 /* 2: rtb_surface.hints, rtb_measure_dfma_chain_rate; 3: rtb_tune; 4: rtb_comm_*; 5: rtb_pure_launch_count */
/* per launch (the prescription travels in the kernel parameter block); the host layer chains longer systems */
#define RTB_MAX_SURFACES 64
#define RTB_MAX_WAVELENGTHS 8 /* rows of the host refractive-index table (one extra row answers NaN wavelengths) */
#define RTB_MAX_KEEP (2 * RTB_MAX_SURFACES + 1)

typedef enum rtb_status {
    RTB_OK = 0,
    RTB_ERR_INVALID = -1,     /* structurally invalid argument (-> ValueError)              */
    RTB_ERR_UNSUPPORTED = -2, /* valid but not implemented on the device (-> NotImplementedError) */
    RTB_ERR_CUDA = -3,        /* CUDA runtime failure (-> RuntimeError)                     */
    RTB_ERR_NOMEM = -4
} rtb_status;

/* raytrace.py:1306 FlatSurface, :1435 SphericalSurface, :1377 PlaneMirror, :1558 PerfectLens */
typedef enum rtb_surface_kind {
    RTB_SURF_FLAT = 0,
    RTB_SURF_SPHERE = 1,
    RTB_SURF_MIRROR = 2,
    RTB_SURF_PERFECT_LENS = 3
} rtb_surface_kind;

/* materials.py:59 Constant, :6 Material (Sellmeier), anything else = host table only */
typedef enum rtb_material_kind {
    RTB_MAT_CONSTANT = 0,
    RTB_MAT_SELLMEIER = 1,
    RTB_MAT_TABLE_ONLY = 2
} rtb_material_kind;

/*
 * One optical surface.  All derived scalars are computed on the host by the same Python expressions the
 * reference uses, so that the device arithmetic starts from bit-identical constants:
 *   radius_sq = radius**2, abs_radius = abs(radius)                  raytrace.py:1499, 1528
 *   normal_f  = normal * focal_len                                   raytrace.py:1683
 *   sin_alpha = np.sin(alpha)                                        raytrace.py:1758
 * `normal` is the geometric plane normal (flat / mirror / perfect lens; raytrace.py:1320, 1389, 1576), `input_axis`
 * the axis used by the "ray comes from the front" cull and the sphere's aperture test (raytrace.py:1189, 1531).
 * System.reverse() flips only the latter (raytrace.py:409-411), so both are carried.
 */
/*
 * rtb_surface.hints (optional, 0 = none).  Hints never change a result -- every route computes the same bits -- only
 * which code path gets there first.
 * RTB_HINT_DEGENERATE  on a flat refracting surface: the bundle meets it with exact zeros ray after ray (the rays
 *                      start on the plane, t = +-0, or run exactly along its normal, d x n = 0 -- what the reference's
 *                      scripts do with their first surface).  The hot loop then handles those zeros in line instead of
 *                      redoing every ray out of line.  Costs a few percent at that surface when the bundle is ordinary.
 */
#define RTB_HINT_DEGENERATE 1

typedef struct rtb_surface {
    int32_t kind; /* rtb_surface_kind */
    int32_t hints; /* RTB_HINT_* */
    double center[3];
    double normal[3];
    double input_axis[3];
    double radius;
    double radius_sq;
    double abs_radius;
    double aperture_rad;
    double focal_len;
    double normal_f[3];
    double sin_alpha;
} rtb_surface;

/* Sellmeier: n = sqrt(((b0 w^2/(w^2-c0) + b1 w^2/(w^2-c1)) + b2 w^2/(w^2-c2)) + 1)      materials.py:39-51 */
typedef struct rtb_material {
    int32_t kind; /* rtb_material_kind */
    int32_t reserved;
    double b[3];
    double c[3];
    double n_const;
} rtb_material;

/*
 * A sequential system: S surfaces and the S+1 media around them, i.e. the list
 * [initial_material] + system.materials + [final_material] of raytrace.py:653.
 *
 * Refractive indices come from one of two places:
 *   n_wavelengths > 0 : `wavelengths[n_wavelengths]` lists every distinct wavelength bit pattern of the batch and
 *        `n_table[(n_wavelengths + 1) * (S + 1)]` (row-major, row = wavelength, column = medium) holds material.n()
 *        evaluated on the host by the user's own Python objects; the extra last row is the answer for a NaN
 *        wavelength.  Works for every material kind, bit exact by construction.  A ray whose (valid) wavelength
 *        is not listed is evaluated in the kernel like the n_wavelengths == 0 case, so the list may be a sample
 *        of the batch UNLESS a RTB_MAT_TABLE_ONLY medium is present (then it must be complete: such a ray's
 *        index would be NaN).
 *   n_wavelengths == 0: the kernel evaluates Constant / Sellmeier media per ray; RTB_MAT_TABLE_ONLY media are
 *        then refused with RTB_ERR_UNSUPPORTED.
 */
typedef struct rtb_system {
    int32_t n_surfaces;
    int32_t n_wavelengths;
    const rtb_surface *surfaces;   /* host, n_surfaces */
    const rtb_material *materials; /* host, n_surfaces + 1 */
    const double *wavelengths;     /* host, n_wavelengths (may be NULL when 0) */
    const double *n_table;         /* host, (n_wavelengths + 1) * (n_surfaces + 1) (may be NULL when 0) */
} rtb_system;

typedef enum rtb_precision {
    RTB_F64_EXACT = 0, /* reference operation order, no FMA contraction: bit-identical to the NumPy path */
    RTB_F32_FAST = 1,  /* fp32 geometry, fp64 positions / phase; tolerance stated in DESIGN.md section 8 */
    RTB_F64_FAST = 2   /* all fp64 with FMA and the direct Snell form: ~1e-13 from the reference, but the
                          round-off-dependent validity of knife-edge rays is not reproduced              */
} rtb_precision;

typedef enum rtb_keep_mode {
    RTB_KEEP_ALL = 0,  /* out = (2S+1, N, 8): what System.ray_trace returns (raytrace.py:1229-1232)   */
    RTB_KEEP_LAST = 1, /* out = (1, N, 8): slab 2S only                                               */
    RTB_KEEP_LIST = 2, /* out = (n_keep, N, 8): slabs keep_slabs[0..n_keep), strictly increasing      */
    RTB_KEEP_NONE = 3  /* no ray output (reductions only)                                             */
} rtb_keep_mode;

/*
 * Optional fused reductions evaluated at one slab of the trace (the "ray fan -> pupil phase -> PSF accumulation"
 * and the spot statistics of BASELINE.json).  Coordinates are taken in a plane basis:
 *     u = (p - origin) . e1,   v = (p - origin) . e2
 * A ray contributes when u, v and phase are all finite (not NaN).
 *
 *   stats_dev  (RTB_N_STATS doubles, accumulated with atomics -- zero it first):
 *       [0] count  [1] sum u  [2] sum v  [3] sum u^2  [4] sum v^2  [5] sum u v
 *       [6] sum (phase - phase_ref)  [7] sum (phase - phase_ref)^2  [8] min u [9] max u [10] min v [11] max v
 *       (min/max slots must be initialised to +inf / -inf by the caller; rtb_reduce_init does all of this)
 *   grid_dev   (3 * grid_n * grid_n doubles, accumulated with atomics):
 *       plane 0: sum cos(phase - phase_ref), plane 1: sum sin(phase - phase_ref), plane 2: count,
 *       cell (iu, iv) at [plane * G*G + iv * G + iu], iu = floor((u + grid_half_width) * (G / (2*grid_half_width)));
 *       rays outside [-half, half) are counted in stats only.
 */
#define RTB_N_STATS 12
typedef struct rtb_reduce {
    int32_t slab;   /* slab index in [0, 2S] at which (p, phase) are sampled */
    int32_t grid_n; /* G, 0 = no grid */
    double origin[3];
    double e1[3];
    double e2[3];
    double phase_ref;
    double grid_half_width;
    double *stats_dev; /* device, RTB_N_STATS, or NULL */
    double *grid_dev;  /* device, 3*G*G, or NULL       */
} rtb_reduce;

/* rtb_trace_opts.flags */
#define RTB_FLAG_INTERSECT_ONLY 1 /* the "at surface" slab is Surface.get_intersect's result (raytrace.py:1331-1337,
                                     1398-1403, 1479-1516, 1580-1584): no front-side cull; a perfect lens blanks
                                     rays that would have to travel backwards.  Used by the per-surface operator. */

#define RTB_FLAG_PLANES_IN 2      /* device entry points only: rays_in_dev is (8, N) -- one plane per column           */
#define RTB_FLAG_PLANES_OUT 4     /* device entry points only: out_dev is (n_slabs, 8, N)                              */

typedef struct rtb_trace_opts {
    int32_t precision; /* rtb_precision */
    int32_t keep_mode; /* rtb_keep_mode */
    int32_t n_keep;
    int32_t flags;
    const int32_t *keep_slabs; /* host, n_keep entries, for RTB_KEEP_LIST */
    const rtb_reduce *reduce;  /* host, optional */
} rtb_trace_opts;

/* On-device ray sources, so that 1e8..1e9-ray batches never exist on the host. */
typedef enum rtb_source_kind {
    RTB_SRC_COLLIMATED = 0, /* get_collimated_rays, raytrace.py:99-161:  index = i_disp * n_b + i_phi      */
    RTB_SRC_FAN = 1,        /* get_ray_fan,         raytrace.py:45-96 :  index = i_phi  * n_a + i_theta    */
    RTB_SRC_GRID = 2        /* Cartesian grid of parallel rays: index = i_v * n_a + i_u (this library's own) */
} rtb_source_kind;

/*
 * kind COLLIMATED: a = displacement (n_a values, linspace(-a_max, a_max, n_a)), b = azimuth (n_b values,
 *                  arange(n_b)*2pi/n_b + b_start); position = pt + e1*(a cos b) + e2*(a sin b), direction = axis.
 * kind FAN:        a = polar angle theta (linspace(-a_max, a_max, n_a)), b = azimuth phi (arange(n_b)*2pi/n_b);
 *                  position = pt, direction = axis cos(theta) + e1 cos(phi) sin(theta) + e2 sin(phi) sin(theta).
 * kind GRID:       u = linspace(-a_max, a_max, n_a), v = linspace(-b_max, b_max, n_b);
 *                  position = (pt + e1*u) + e2*v, direction = axis.
 * e1, e2 are the transverse unit vectors, computed on the host exactly as the reference does (raytrace.py:79-81,
 * 135-144).  phase = 0, wavelength = `wavelength` for every ray.
 */
typedef struct rtb_source {
    int32_t kind;
    int32_t reserved;
    int64_t n_a;
    int64_t n_b;
    double a_max;
    double b_max;   /* GRID only */
    double b_start; /* COLLIMATED: phi_start */
    double pt[3];
    double axis[3];
    double e1[3];
    double e2[3];
    double wavelength;
} rtb_source;

/* ---- library ------------------------------------------------------------------------------------------ */
int rtb_abi_version(void);
const char *rtb_last_error(void);
/* number of CUDA devices visible (0 if none); negative rtb_status if the runtime cannot be initialised */
int rtb_device_count(void);
/* kernels launched by this library in this process so far (for bench.py's gpu_launches claim) */
int64_t rtb_launch_count(void);
/* lean launches so far that ran the pure kernel instantiations (picked by the verdict cache, see rtb_tune "lean_pure") */
int64_t rtb_pure_launch_count(void);

/*
 * Tuning knobs (never change a result, only which kernel gets there).  The environment variables named below set
 * initial values; they are read when the library is loaded, and rtb_tune overrides them.
 *   "lean_min_rays"  launches of at least this many rays that keep only the final slab and / or one after-surface
 *                    reduction run the probe + lean kernel pair (csrc/trace_lean.cu); default 32768, negative = never.
 *                    The environment variable RTB_LEAN_MIN_RAYS sets the initial value.
 *   "lean_min_share_pct"  that kernel pair takes a system only when at least this share (per cent, default 75) of its
 *                    surfaces are on-axis spheres / flats, the ones it has lean steps for (RTB_LEAN_MIN_SHARE_PCT).
 *   "psf_dmma"       1 (default): the PSF contraction runs on the FP64 tensor path (mma.sync.m8n8k4.f64); 0: the SIMT
 *                    register-tiled kernel.  Same sums in a different order (agreement ~1e-13 relative).
 *   "lean_pure"      which lean kernel traces a system whose every surface has a lean step.  1 (default): the "pure"
 *                    instantiations -- no general steps, control flow from kernel parameters only, the prescription read
 *                    through the uniform datapath, +4 % -- once the probe of an EARLIER launch of the same system (and,
 *                    for on-device sources, the same source description) has found no surface where whole bundles fail
 *                    the lean step; every launch's probe counts are read back asynchronously for the next one, nothing
 *                    synchronises (launches from on-device sources, whose rays the key determines, drop the probe once
 *                    their verdict is in).  0: the probe-driven kernels always.  2: the pure kernels whatever the bundle (tests).
 *                    RTB_LEAN_PURE sets the initial value.  A stale verdict costs time only: failing rays are re-traced.
 *                    Setting the mode forgets every cached verdict.
 *   "sweep_split_rays" rtb_trace_sources traces sweeps of at least this many rays per source (default 2^24) as one launch
 *                    per source -- source and reduction bucket in the kernel parameters -- instead of one launch for all;
 *                    negative = never.  RTB_SWEEP_SPLIT_RAYS sets the initial value.  Same rows, same buckets.
 *   "keep_probe_counts" test hook: 1 = every lean launch synchronises and keeps its probe's per-surface counts for
 *                    rtb_last_probe_counts().
 *   "host_fail_chunk" test hook: rtb_trace_host returns RTB_ERR_CUDA when it is about to launch chunk n (0-based) of a
 *                    call (negative = off), after draining every copy already in flight.
 */
int rtb_tune(const char *key, int64_t value);
/* out[2k] = probe rays that reached surface k, out[2k+1] = those whose lean step failed there (last lean launch made
   with "keep_probe_counts" on; first source of a sweep) */
int rtb_last_probe_counts(uint32_t *out, int n_surfaces);

/* ---- the hot path: replaces System.ray_trace, raytrace.py:641-661 --------------------------------------- */
/*
 * rays_in_dev : (N, 8) device.  out_dev : (n_out_slabs, N, 8) device, n_out_slabs per opts->keep_mode
 * (may be NULL for RTB_KEEP_NONE).  In RTB_KEEP_ALL / RTB_KEEP_LIST slab 0 is a copy of the input rows.
 * Enqueues on `stream` and returns; no host synchronisation.
 */
int rtb_trace_device(const rtb_system *sys, const double *rays_in_dev, int64_t n_rays, double *out_dev,
                     const rtb_trace_opts *opts, int device, void *stream);

/*
 * Same trace with HOST buffers (the drop-in call): rays_in_host (N, 8), out_host (n_out_slabs, N, 8).
 * The library stages chunks through pinned memory on its own streams (copy-in, kernel, copy-out overlapped) and
 * returns when out_host is complete.  opts->reduce buffers, if given, stay device pointers.
 */
int rtb_trace_host(const rtb_system *sys, const double *rays_in_host, int64_t n_rays, double *out_host,
                   const rtb_trace_opts *opts, int device);

/*
 * Trace rays produced on the device by `src` (ray indices [first_ray, first_ray + n_rays) of the source's index
 * space), fused as the prologue of the trace kernel: no input bytes.  out_dev as for rtb_trace_device.
 */
int rtb_trace_source(const rtb_system *sys, const rtb_source *src, int64_t first_ray, int64_t n_rays,
                     double *out_dev, const rtb_trace_opts *opts, int device, void *stream);

/*
 * A sweep in ONE launch (field points, wavelengths, defocus ... : the per-wavelength loop of
 * scripts/2022_08_04_ACT508-100-B.py:120-150, BASELINE configs 2 and 3): n_src sources, each
 * tracing ray indices [first_ray, first_ray + n_rays_each) of its own index space through the same system.
 * Source k's rays occupy rows [k * n_rays_each, (k + 1) * n_rays_each) of every output slab (out_dev is
 * (n_out_slabs, n_src * n_rays_each, 8)), and its reductions go to bucket k of opts->reduce: statistics at
 * stats_dev + k * RTB_N_STATS, grid at grid_dev + k * 3 * grid_n * grid_n (initialise every bucket with
 * rtb_reduce_init).  sys must tabulate the sources' wavelengths (at most RTB_MAX_WAVELENGTHS distinct ones; more are
 * fine when every medium is CONSTANT / SELLMEIER).
 */
int rtb_trace_sources(const rtb_system *sys, const rtb_source *srcs, int32_t n_src, int64_t first_ray,
                      int64_t n_rays_each, double *out_dev, const rtb_trace_opts *opts, int device, void *stream);

/* ---- ray sources: replace get_collimated_rays / get_ray_fan, raytrace.py:45-161 --------------------------- */
int rtb_generate_device(const rtb_source *src, int64_t first_ray, int64_t n_rays, double *rays_out_dev,
                        int device, void *stream);

/* ---- reductions ------------------------------------------------------------------------------------------- */
/* zero / initialise the stats vector and grid referenced by `red` (count=0, min=+inf, max=-inf) */
int rtb_reduce_init(const rtb_reduce *red, int device, void *stream);

/*
 * Pupil grid -> PSF (the tail of scripts/2022_02_06_perfect_imaging_system_psf.py:90-105 as a dense complex contraction).
 * grid_dev is the (3, G, G) accumulator of rtb_reduce; P[v,u] = grid[0] + i grid[1] (divided by grid[2] where non-empty
 * if normalize_by_count).  Output: n_samples x n_samples samples of E = A P B^T and/or |E|^2 with
 *   B[k,u] = exp(-2 pi i f_k x_u),  f_k = (k - (n_samples-1)/2) * df,  x_u = (u + 0.5) * (2 half/G) - half  (same for A).
 * psf_out_dev (n*n) and/or field_re_dev + field_im_dev (n*n each) may be NULL.  scratch_dev: at least
 * rtb_psf_scratch_doubles() doubles of device memory.
 */
int64_t rtb_psf_scratch_doubles(int grid_n, int n_samples, int normalize_by_count);
int rtb_psf_from_grid_device(const double *grid_dev, int grid_n, double grid_half_width, int n_samples, double df,
                             int normalize_by_count, double *scratch_dev, int64_t scratch_doubles, double *psf_out_dev,
                             double *field_re_dev, double *field_im_dev, int device, void *stream);

/* ---- multi-GPU: the one exchange step of the path (SURVEY.md 8e) --------------------------------------------------
 * Rays shard by contiguous index range over one process per GPU (the reference has no counterpart: its loop,
 * raytrace.py:641-661, is single-process); the trace never communicates.  What is exchanged afterwards are the reduced
 * products of rtb_reduce: the pupil grid (summed) and the statistics vectors (8 sums, 2 minima, 2 maxima per bucket).
 * These entry points wrap NCCL (resolved at run time from libnccl.so.2; RTB_ERR_UNSUPPORTED when it is absent) so that
 * a binder without PyTorch can do the reduction.  Bootstrapping: rank 0 calls rtb_comm_unique_id and hands the
 * RTB_COMM_ID_BYTES bytes to every rank (MPI, a file, a socket ...); then every rank calls rtb_comm_init, which blocks
 * until all n_ranks have joined.  The collectives enqueue on `stream` and return; every rank must call them in the same
 * order.  One communicator per (process, device); not thread safe.
 */
#define RTB_COMM_ID_BYTES 128
typedef struct rtb_comm rtb_comm;
/* NCCL's version code (e.g. 22809) when the library could be loaded, 0 otherwise */
int rtb_comm_available(void);
int rtb_comm_unique_id(void *id_out, size_t id_bytes);
int rtb_comm_init(rtb_comm **comm_out, int n_ranks, int rank, const void *unique_id, int device);
/* number of ranks of the communicator (negative rtb_status on error) */
int rtb_comm_size(const rtb_comm *comm);
/* in-place sum over the ranks of n_doubles doubles: the (3, G, G) grid of rtb_reduce, all buckets at once */
int rtb_comm_allreduce_grid(rtb_comm *comm, double *grid_dev, int64_t n_doubles, void *stream);
/* in-place merge over the ranks of n_buckets statistics vectors (RTB_N_STATS doubles each): one all-gather and a
   merge kernel; sums are accumulated in rank order, so the result is the same on every rank and run to run */
int rtb_comm_allreduce_stats(rtb_comm *comm, double *stats_dev, int n_buckets, void *stream);
int rtb_comm_destroy(rtb_comm *comm);

/* ---- after the trace: replaces intersect_rays, raytrace.py:164-238 ----------------------------------------- */
/* ray1_dev, ray2_dev : (N, 8) device; pts_out_dev : (N, 3) device. n1 or n2 may be 1 (broadcast). */
int rtb_intersect_rays_device(const double *ray1_dev, int64_t n1, const double *ray2_dev, int64_t n2,
                              double *pts_out_dev, int device, void *stream);

/*
 * replaces propagate_ray2plane, raytrace.py:241-306, with per-ray planes:
 * rays_dev (N,8); normal_dev (n_normal,3) and center_dev (n_center,3) with n_* in {1, N}; index_dev (N) = the
 * medium's n(wavelength) per ray (evaluated by the caller's material object); rays_out_dev (N,8); ts_out_dev (N).
 */
int rtb_ray2plane_device(const double *rays_dev, int64_t n_rays, const double *normal_dev, int64_t n_normal,
                         const double *center_dev, int64_t n_center, const double *index_dev,
                         int exclude_backward, double *rays_out_dev, double *ts_out_dev, int device, void *stream);

/*
 * Distinct non-NaN wavelength bit patterns of a device ray batch (column 7), for building the host
 * refractive-index table of a device-resident batch.  table_dev: RTB_MAX_WAVELENGTHS + 1 doubles of scratch on the
 * device.  On return (after a stream synchronise done inside) wavelengths_host[0..*n_found) holds them in ascending
 * order; *n_found = RTB_MAX_WAVELENGTHS + 1 means "more than RTB_MAX_WAVELENGTHS".
 */
int rtb_distinct_wavelengths_device(const double *rays_dev, int64_t n_rays, double *table_dev,
                                    double *wavelengths_host, int32_t *n_found, int device, void *stream);

/* The same for a host batch (multi-threaded scan of column 7); wavelengths_out holds RTB_MAX_WAVELENGTHS + 1 doubles. */
int rtb_distinct_wavelengths_host(const double *rays_host, int64_t n_rays, double *wavelengths_out, int32_t *n_found);

/* page-locked host memory for zero-staging transfers in rtb_trace_host (NULL on failure) */
void *rtb_host_alloc(size_t bytes);
void rtb_host_free(void *p);

/*
 * Self-test of the library's factored IEEE division / square root (csrc/exact_math.cuh) against the built-in
 * operators on n_cases pseudo-random operand sets (raw bit patterns, moderate magnitudes, special values).
 * mismatches[0] = scalar divisions, [1] = three-way divisions, [2] = square roots that differ in any bit.
 */
int rtb_selftest_exact_math(int device, uint64_t seed, int64_t n_cases, uint64_t mismatches[3]);

/* ---- measurement helpers ------------------------------------------------------------------------------------ */
/*
 * Register-only dependent-chain DFMA micro-benchmark: the FP64-pipe roofline denominator (SURVEY.md 8d).
 * *dfma_per_s = thread-level DFMA instructions per second on `device` (x2 for FLOP/s), best of 5 launches.
 */
int rtb_measure_dfma_rate(int device, double *dfma_per_s, double *elapsed_ms);
/*
 * The same measurement for latency-bound code: `chains` (1, 2, 4 or 8) independent dependent-DFMA chains per thread at
 * the trace kernels' occupancy (7 warps of 32 per SM sub-partition).  On the B200 the FP64 pipe takes an instruction
 * that follows one of the same warp after 2 cycles and one that follows another warp's after 3, so chains = 1 -- what
 * one ray through one surface looks like -- tops out at 2/3 of the chains = 8 rate (DESIGN.md 4a).
 */
int rtb_measure_dfma_chain_rate(int device, int chains, double *dfma_per_s, double *elapsed_ms);
/* device-to-device copy bandwidth (read+write bytes / s) over `bytes` bytes, for cross-checking MEASURED_PEAKS */
int rtb_measure_copy_bandwidth(int device, int64_t bytes, double *bytes_per_s);

#ifdef __cplusplus
}
#endif
#endif /* RTB_H */
