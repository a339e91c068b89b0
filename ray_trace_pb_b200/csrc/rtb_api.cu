// rtb_api.cu -- the C ABI declared in include/rtb.h: argument checking, prescription packing, launches and the
// pinned-memory host pipeline.  No ray arithmetic happens here and nothing here runs a trace on the CPU.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "rtb_device.cuh"

namespace rtb {
cudaError_t launch_trace_f64(const TraceParams &P, int sm_count, cudaStream_t stream);
cudaError_t launch_trace_fast(const TraceParams &P, int precision, int sm_count, cudaStream_t stream);
bool lean_takes(const TraceParams &P, int precision);
size_t lean_scratch_bytes(int n_sources);
cudaError_t launch_lean(const TraceParams &P, int device, int sm_count, cudaStream_t stream, cudaMemPool_t pool,
                        void *scratch, const DevSource *sources, int *launches);
void lean_forget_verdicts();
cudaError_t launch_generate(const DevSource &src, long long n_rays, double *out, int sm_count, cudaStream_t stream);
cudaError_t launch_reduce_init(const DevReduce &red, int sm_count, cudaStream_t stream);
cudaError_t launch_intersect(const double *r1, long long n1, const double *r2, long long n2, double *out,
                             cudaStream_t stream);
cudaError_t launch_ray2plane(const double *rays, long long n, const double *normal, long long n_normal,
                             const double *center, long long n_center, const double *index, int exclude_backward,
                             double *out, double *ts, cudaStream_t stream);
cudaError_t run_distinct_wavelengths(const double *rays, long long n, double *table_dev, int capacity,
                                     double *host_out, int *n_found, int sm_count, cudaStream_t stream);
long long psf_scratch_doubles(int G, int M, int normalize);
cudaError_t launch_psf(const double *grid, int G, double half_width, int M, double df, int normalize, double *scratch,
                       double *psf_out, double *field_re, double *field_im, int sm_count, cudaStream_t stream, int *launches);
cudaError_t run_exact_math_selftest(unsigned long long seed, long long n, unsigned long long *bad_host, int sm_count);
cudaError_t run_dfma_probe(int sm_count, double *dfma_per_s, double *elapsed_ms);
cudaError_t run_dfma_chain_probe(int sm_count, int chains, double *dfma_per_s, double *elapsed_ms);
cudaError_t run_copy_probe(long long bytes, double *bytes_per_s);
// the tuning knobs of trace_lean.cu and psf_kernels.cu
extern std::atomic<long long> g_lean_min_rays, g_lean_min_share_pct, g_lean_pure, g_keep_probe_counts, g_psf_dmma;
} // namespace rtb

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};
// test hook: rtb_trace_host fails (RTB_ERR_CUDA, "injected") when it is about to launch chunk number n (0-based) of a
// call; negative = off.  rtb_tune("host_fail_chunk", n).  Lets the tests check that an error return leaves no copy in flight.
std::atomic<long long> g_host_fail_chunk{-1};
// rtb_trace_sources traces sweeps of at least this many rays per source as one launch PER SOURCE (each with its source and
// its reduction bucket in the kernel parameters, i.e. warp-uniform operands) instead of one launch whose blocks fetch
// theirs from shared memory.  Measured: 3 x 16.8 M rays +3.6 % (BASELINE config 2: 65.3 -> 67.7 G ray*surf/s), but
// 32 x 4.2 M rays -5.7 % (config 3: each launch pays its own probe and its own tail), so only really big sources are
// split.  rtb_tune("sweep_split_rays", n); RTB_SWEEP_SPLIT_RAYS; negative = never.
std::atomic<long long> g_sweep_split_rays{1 << 24};

// rtb_tune's keys (include/rtb.h): the knob each sets, the environment variable that sets its initial value, and the
// values it takes
struct Knob {
    const char *key;
    const char *env;                  // (NULL: none)
    std::atomic<long long> *value;
    long long lo = LLONG_MIN, hi = LLONG_MAX;
};
const Knob kKnobs[] = {
    {"lean_min_rays", "RTB_LEAN_MIN_RAYS", &rtb::g_lean_min_rays},
    {"lean_min_share_pct", "RTB_LEAN_MIN_SHARE_PCT", &rtb::g_lean_min_share_pct},
    {"lean_pure", "RTB_LEAN_PURE", &rtb::g_lean_pure, 0, 2},
    {"psf_dmma", nullptr, &rtb::g_psf_dmma},
    {"sweep_split_rays", "RTB_SWEEP_SPLIT_RAYS", &g_sweep_split_rays},
    {"keep_probe_counts", nullptr, &rtb::g_keep_probe_counts},
    {"host_fail_chunk", nullptr, &g_host_fail_chunk},
};

// The environment is read when the library is loaded, before any rtb_tune call, which therefore always wins.  (An
// environment value outside the knob's range is clamped.)
const bool g_knobs_from_env = [] {
    for (const Knob &k : kKnobs)
        if (const char *env = k.env ? getenv(k.env) : nullptr)
            k.value->store(std::min(k.hi, std::max(k.lo, (long long)atoll(env))), std::memory_order_relaxed);
    return true;
}();

} // namespace

namespace rtb {
int api_fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
} // namespace rtb

namespace {

constexpr auto &fail = rtb::api_fail;

// The tail of an entry point that ran a launcher: RTB_ERR_CUDA ("<what>: <CUDA error>") if the launcher failed, else
// its `n_kernels` kernels join rtb_launch_count().
int launched(cudaError_t e, const char *what, long long n_kernels)
{
    if (e != cudaSuccess) return fail(RTB_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
    g_launches.fetch_add(n_kernels, std::memory_order_relaxed);
    return RTB_OK;
}

#define RTB_CUDA(call)                                                                                     \
    do {                                                                                                   \
        cudaError_t e_ = (call);                                                                           \
        if (e_ != cudaSuccess)                                                                             \
            return fail(RTB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---- per-device context: SM count, streams and staging buffers of the host pipeline ------------------------
constexpr int kSlots = 4;

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    cudaEvent_t copied_in = nullptr;   // this slot's copy-in has landed (the previous chunk's copy-out waits for it)
    void *lean_scratch = nullptr;      // probe scratch of the lean kernel for this slot's chunks
    double *dev_in = nullptr;
    double *dev_out = nullptr;
    double *pin_in = nullptr;
    double *pin_out = nullptr;
    size_t dev_in_bytes = 0, dev_out_bytes = 0, pin_in_bytes = 0, pin_out_bytes = 0;
};

struct DeviceCtx {
    bool ready = false;
    int sm_count = 0;
    Slot slot[kSlots];
    std::mutex host_path; // one host-buffer trace at a time per device
    cudaMemPool_t pool = nullptr; // small stream-ordered allocations (sweep source lists); keeps its memory
};

DeviceCtx g_ctx[rtb::kMaxDevices];
std::mutex g_ctx_mutex;

int get_ctx(int device, DeviceCtx **out)
{
    if (device < 0 || device >= rtb::kMaxDevices) return fail(RTB_ERR_INVALID, "device index %d out of range", device);
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(RTB_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
    if (device >= n) return fail(RTB_ERR_INVALID, "device index %d but only %d device(s) visible", device, n);
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    DeviceCtx &c = g_ctx[device];
    if (!c.ready) {
        RTB_CUDA(cudaDeviceGetAttribute(&c.sm_count, cudaDevAttrMultiProcessorCount, device));
        c.ready = true;
    }
    *out = &c;
    return RTB_OK;
}

// The device of an entry point: its context, and the device made current for the rest of the call (the caller's
// current device comes back when this goes out of scope).
struct OnDevice {
    DeviceCtx *ctx = nullptr;
    int device = -1, prev = -1;
    bool changed = false;
    int enter(int dev)
    {
        if (int rc = get_ctx(dev, &ctx)) return rc;
        device = dev;
        RTB_CUDA(cudaGetDevice(&prev));
        if (prev != device) {
            RTB_CUDA(cudaSetDevice(device));
            changed = true;
        }
        return RTB_OK;
    }
    ~OnDevice()
    {
        if (changed) cudaSetDevice(prev);
    }
};

// ---- exact squared-domain thresholds (see DevSurface in rtb_device.cuh) ------------------------------------------
// fl(sqrt(.)) is monotone, so  fl(sqrt(s)) <= r  <=>  s <= sq_upper(r)  and  fl(sqrt(s)) >= r  <=>  s >= sq_lower(r).
double sq_upper(double r) // largest s with fl(sqrt(s)) <= r
{
    if (std::isnan(r)) return r;
    if (r < 0) return -1.0;
    if (std::isinf(r)) return r;
    double c = r * r;
    while (std::sqrt(c) > r) c = std::nextafter(c, -INFINITY);
    for (;;) {
        const double n = std::nextafter(c, INFINITY);
        if (std::isinf(n) || !(std::sqrt(n) <= r)) break;
        c = n;
    }
    return c;
}

double sq_lower(double r) // smallest s >= 0 with fl(sqrt(s)) >= r
{
    if (std::isnan(r)) return r;
    if (r <= 0) return 0.0;
    if (std::isinf(r)) return r;
    double c = r * r;
    while (std::sqrt(c) < r) c = std::nextafter(c, INFINITY);
    for (;;) {
        const double n = std::nextafter(c, -INFINITY);
        if (n < 0 || !(std::sqrt(n) >= r)) break;
        c = n;
    }
    return c;
}

// | fl(norm - abs_radius) | < tol   <=>   lo <= norm <= hi   (fl(x - a) is monotone in x)
void on_sphere_window(double abs_radius, double tol, double &lo, double &hi)
{
    if (!std::isfinite(abs_radius)) {
        lo = INFINITY;
        hi = -INFINITY;
        return;
    }
    double r = abs_radius - tol;
    while (!((r - abs_radius) > -tol)) r = std::nextafter(r, INFINITY);
    while ((std::nextafter(r, -INFINITY) - abs_radius) > -tol) r = std::nextafter(r, -INFINITY);
    lo = r;
    r = abs_radius + tol;
    while (!((r - abs_radius) < tol)) r = std::nextafter(r, -INFINITY);
    while ((std::nextafter(r, INFINITY) - abs_radius) < tol) r = std::nextafter(r, INFINITY);
    hi = r;
}

// ---- packing ------------------------------------------------------------------------------------------------
int n_out_slabs(const rtb_system *sys, const rtb_trace_opts *opts)
{
    switch (opts->keep_mode) {
    case RTB_KEEP_ALL: return 2 * sys->n_surfaces + 1;
    case RTB_KEEP_LAST: return 1;
    case RTB_KEEP_LIST: return opts->n_keep;
    default: return 0;
    }
}

int pack_params(const rtb_system *sys, const rtb_trace_opts *opts, rtb::TraceParams &P)
{
    if (!sys || !opts) return fail(RTB_ERR_INVALID, "system / options pointer is NULL");
    const int S = sys->n_surfaces;
    if (S < 0 || S > RTB_MAX_SURFACES)
        return fail(RTB_ERR_INVALID, "n_surfaces = %d outside [0, %d]", S, RTB_MAX_SURFACES);
    if (S > 0 && (!sys->surfaces)) return fail(RTB_ERR_INVALID, "surfaces pointer is NULL");
    if (!sys->materials) return fail(RTB_ERR_INVALID, "materials pointer is NULL (need n_surfaces + 1 media)");
    if (sys->n_wavelengths < 0 || sys->n_wavelengths > RTB_MAX_WAVELENGTHS)
        return fail(RTB_ERR_INVALID, "n_wavelengths = %d outside [0, %d]", sys->n_wavelengths, RTB_MAX_WAVELENGTHS);
    if (sys->n_wavelengths > 0 && (!sys->wavelengths || !sys->n_table))
        return fail(RTB_ERR_INVALID, "n_wavelengths > 0 needs wavelengths and n_table");

    memset(&P, 0, sizeof(P));
    P.n_surf = S;
    P.n_wl = sys->n_wavelengths;
    for (int k = 0; k < S; k++) {
        const rtb_surface &a = sys->surfaces[k];
        if (a.kind < RTB_SURF_FLAT || a.kind > RTB_SURF_PERFECT_LENS)
            return fail(RTB_ERR_UNSUPPORTED, "surface %d has unknown kind %d", k, a.kind);
        rtb::DevSurface &d = P.surf[k];
        d.kind = a.kind;
        d.cx = a.center[0]; d.cy = a.center[1]; d.cz = a.center[2];
        d.nx = a.normal[0]; d.ny = a.normal[1]; d.nz = a.normal[2];
        d.ax = a.input_axis[0]; d.ay = a.input_axis[1]; d.az = a.input_axis[2];
        d.radius = a.radius; d.radius_sq = a.radius_sq; d.abs_radius = a.abs_radius;
        d.aperture = a.aperture_rad;
        d.focal_len = a.focal_len;
        d.nfx = a.normal_f[0]; d.nfy = a.normal_f[1]; d.nfz = a.normal_f[2];
        d.sin_alpha = a.sin_alpha;
        auto z_aligned = [](const double v[3]) -> int8_t {
            if (v[0] == 0.0 && v[1] == 0.0 && (v[2] == 1.0 || v[2] == -1.0)) return v[2] > 0 ? 1 : -1;
            return 0;
        };
        d.z_normal = z_aligned(a.normal);
        d.z_axis = z_aligned(a.input_axis);
        d.degenerate_hint = (a.hints & RTB_HINT_DEGENERATE) ? 1 : 0;
        d.ap_sq_max = sq_upper(a.aperture_rad);
        double lo, hi;
        on_sphere_window(a.abs_radius, 1e-12, lo, hi);
        d.on_sq_lo = sq_lower(lo);
        d.on_sq_hi = sq_upper(hi);
    }
    for (int k = 0; k <= S; k++) {
        const rtb_material &a = sys->materials[k];
        if (a.kind < RTB_MAT_CONSTANT || a.kind > RTB_MAT_TABLE_ONLY)
            return fail(RTB_ERR_INVALID, "medium %d has unknown kind %d", k, a.kind);
        if (a.kind == RTB_MAT_TABLE_ONLY && sys->n_wavelengths == 0)
            return fail(RTB_ERR_UNSUPPORTED,
                        "medium %d can only be evaluated by its host n(); supply a wavelength table "
                        "(at most %d distinct wavelengths per batch)", k, RTB_MAX_WAVELENGTHS);
        rtb::DevMaterial &d = P.mat[k];
        d.kind = a.kind;
        d.b0 = a.b[0]; d.b1 = a.b[1]; d.b2 = a.b[2];
        d.c0 = a.c[0]; d.c1 = a.c[1]; d.c2 = a.c[2];
        d.n_const = a.n_const;
    }
    for (int k = 0; k < sys->n_wavelengths; k++) P.wl[k] = sys->wavelengths[k];
    if (sys->n_wavelengths > 0) {
        memcpy(P.n_tab, sys->n_table, sizeof(double) * (size_t)(sys->n_wavelengths + 1) * (size_t)(S + 1));
        // n1 / n2 per (wavelength row, surface): the host's IEEE division gives the bits the kernel's would
        for (int r = 0; r <= sys->n_wavelengths; r++)
            for (int k = 0; k < S; k++)
                P.ratio_tab[r * (S + 1) + k] = P.n_tab[r * (S + 1) + k] / P.n_tab[r * (S + 1) + k + 1];
    }

    // which slabs go where
    const int n_slabs = 2 * S + 1;
    for (int j = 0; j < rtb::kMaxSlabs + 3; j++) P.slab_pos[j] = -1;
    switch (opts->keep_mode) {
    case RTB_KEEP_ALL:
        for (int j = 0; j < n_slabs; j++) P.slab_pos[j] = (int16_t)j;
        P.any_store = 1;
        break;
    case RTB_KEEP_LAST:
        P.slab_pos[n_slabs - 1] = 0;
        P.store_last_only = 1;
        P.any_store = 1;
        break;
    case RTB_KEEP_LIST: {
        if (opts->n_keep < 1 || opts->n_keep > n_slabs || !opts->keep_slabs)
            return fail(RTB_ERR_INVALID, "keep list needs 1..%d slab indices", n_slabs);
        int prev = -1;
        for (int q = 0; q < opts->n_keep; q++) {
            const int j = opts->keep_slabs[q];
            if (j < 0 || j >= n_slabs) return fail(RTB_ERR_INVALID, "keep_slabs[%d] = %d outside [0, %d]", q, j, n_slabs - 1);
            if (j <= prev) return fail(RTB_ERR_INVALID, "keep_slabs must be strictly increasing");
            P.slab_pos[j] = (int16_t)q;
            prev = j;
        }
        P.any_store = 1;
        break;
    }
    case RTB_KEEP_NONE:
        break;
    default:
        return fail(RTB_ERR_INVALID, "unknown keep_mode %d", opts->keep_mode);
    }
    if (opts->precision != RTB_F64_EXACT && opts->precision != RTB_F32_FAST && opts->precision != RTB_F64_FAST)
        return fail(RTB_ERR_INVALID, "unknown precision %d", opts->precision);

    P.flags = opts->flags;
    P.red.slab = -1;
    if (opts->reduce) {
        const rtb_reduce &r = *opts->reduce;
        if (r.slab < 0 || r.slab >= n_slabs) return fail(RTB_ERR_INVALID, "reduce slab %d outside [0, %d]", r.slab, n_slabs - 1);
        if (r.grid_n < 0 || r.grid_n > 32768) return fail(RTB_ERR_INVALID, "reduce grid_n %d outside [0, 32768]", r.grid_n);
        if (r.grid_n > 0 && !(r.grid_half_width > 0)) return fail(RTB_ERR_INVALID, "reduce grid_half_width must be > 0");
        if (r.grid_n > 0 && !r.grid_dev) return fail(RTB_ERR_INVALID, "reduce grid_n > 0 but grid_dev is NULL");
        rtb::DevReduce &d = P.red;
        d.slab = r.slab;
        d.grid_n = r.grid_n;
        d.ox = r.origin[0]; d.oy = r.origin[1]; d.oz = r.origin[2];
        d.e1x = r.e1[0]; d.e1y = r.e1[1]; d.e1z = r.e1[2];
        d.e2x = r.e2[0]; d.e2y = r.e2[1]; d.e2z = r.e2[2];
        d.phase_ref = r.phase_ref;
        d.half_width = r.grid_half_width;
        d.inv_cell = r.grid_n > 0 ? (double)r.grid_n / (2.0 * r.grid_half_width) : 0.0;
        d.stats = r.stats_dev;
        d.grid = r.grid_n > 0 ? r.grid_dev : nullptr;
        if (!d.stats && !d.grid) d.slab = -1;
        rtb::finish_reduce(d);
    }
    for (int k = 0; k < S; k++) {
        int act = 0;
        if (P.slab_pos[2 * k + 1] >= 0) act |= 1;
        if (P.slab_pos[2 * k + 2] >= 0) act |= 2;
        if (P.red.slab == 2 * k + 1) act |= 4;
        if (P.red.slab == 2 * k + 2) act |= 8;
        P.slab_act[k] = (uint8_t)act;
    }
    P.src.kind = -1;
    P.src_list = nullptr;
    P.n_src = 0;
    P.pad1 = 0;
    return RTB_OK;
}

int pack_source(const rtb_source *src, long long first, long long count, rtb::DevSource &d)
{
    if (!src) return fail(RTB_ERR_INVALID, "source pointer is NULL");
    if (src->kind < RTB_SRC_COLLIMATED || src->kind > RTB_SRC_GRID)
        return fail(RTB_ERR_INVALID, "unknown source kind %d", src->kind);
    if (src->n_a < 1 || src->n_b < 1) return fail(RTB_ERR_INVALID, "source needs n_a >= 1 and n_b >= 1");
    const long long total = src->n_a * src->n_b;
    if (first < 0 || count < 0 || first + count > total)
        return fail(RTB_ERR_INVALID, "ray range [%lld, %lld) outside the source's %lld rays", first, first + count, total);
    memset(&d, 0, sizeof(d));
    d.kind = src->kind;
    d.n_a = src->n_a;
    d.n_b = src->n_b;
    d.first = first;
    // np.linspace(-m, m, n): step = (stop - start) / (n - 1); y = arange(n) * step + start; y[-1] = stop
    auto lin = [](double m, long long n, double &start, double &step, double &stop) {
        start = -m;
        stop = m;
        const double delta = stop - start;
        step = (n > 1) ? delta / (double)(n - 1) : delta;
    };
    lin(src->a_max, src->n_a, d.a_start, d.a_step, d.a_stop);
    if (src->kind == RTB_SRC_GRID)
        lin(src->b_max, src->n_b, d.b_start, d.b_step, d.b_stop);
    else
        d.b_start = (src->kind == RTB_SRC_COLLIMATED) ? src->b_start : 0.0;
    d.px = src->pt[0]; d.py = src->pt[1]; d.pz = src->pt[2];
    d.axx = src->axis[0]; d.axy = src->axis[1]; d.axz = src->axis[2];
    d.e1x = src->e1[0]; d.e1y = src->e1[1]; d.e1z = src->e1[2];
    d.e2x = src->e2[0]; d.e2y = src->e2[1]; d.e2z = src->e2[2];
    d.wavelength = src->wavelength;
    return RTB_OK;
}

int ensure_pool(DeviceCtx *ctx, int device)
{
    std::lock_guard<std::mutex> lock(g_ctx_mutex);
    if (!ctx->pool) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        RTB_CUDA(cudaMemPoolCreate(&ctx->pool, &props));
        unsigned long long keep = ~0ull;    // never hand the (few KB of) memory back between calls
        RTB_CUDA(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    return RTB_OK;
}

// `lean_scratch`: the lean kernel's probe scratch, owned by the caller (the host pipeline's slots), or NULL to take it from
// the device's stream-ordered pool for the duration of this launch.  `sources`: the host copy of the source
// description(s) of a launch from on-device sources (the lean kernel's verdict cache keys on them).
int launch(const rtb::TraceParams &P, int precision, const OnDevice &on, cudaStream_t stream,
           void *lean_scratch = nullptr, const rtb::DevSource *sources = nullptr)
{
    DeviceCtx *ctx = on.ctx;
    if (rtb::lean_takes(P, precision)) {
        int rc, launches = 0;
        if (!lean_scratch && (rc = ensure_pool(ctx, on.device))) return rc;
        const cudaError_t e = rtb::launch_lean(P, on.device, ctx->sm_count, stream, lean_scratch ? nullptr : ctx->pool,
                                               lean_scratch, sources, &launches);
        if (e == cudaErrorMemoryAllocation)
            return fail(RTB_ERR_NOMEM, "stream-ordered allocation of the lean kernel's probe scratch failed");
        return launched(e, "trace kernel launch failed", launches);
    }
    const cudaError_t e = (precision == RTB_F64_EXACT) ? rtb::launch_trace_f64(P, ctx->sm_count, stream)
                                                       : rtb::launch_trace_fast(P, precision, ctx->sm_count, stream);
    return launched(e, "trace kernel launch failed", P.n_rays > 0 ? 1 : 0);
}

int grow_dev(double **p, size_t *have, size_t want)
{
    if (*have >= want) return RTB_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    if (cudaMalloc(p, want) != cudaSuccess) return fail(RTB_ERR_NOMEM, "cudaMalloc of %zu bytes failed", want);
    *have = want;
    return RTB_OK;
}

int grow_pin(double **p, size_t *have, size_t want)
{
    if (*have >= want) return RTB_OK;
    if (*p) cudaFreeHost(*p);
    *p = nullptr;
    *have = 0;
    if (cudaHostAlloc(p, want, cudaHostAllocDefault) != cudaSuccess)
        return fail(RTB_ERR_NOMEM, "cudaHostAlloc of %zu bytes failed", want);
    *have = want;
    return RTB_OK;
}

// Staging copies between pageable caller memory and the pinned slots: one core moves ~10 GB/s, a fifth of the link, so
// copies of 4 MiB and more are split over a few threads (RTB_HOST_COPY_THREADS, default 4, 1 = plain memcpy).
void staging_copy(void *dst, const void *src, size_t bytes)
{
    static const int n_threads = [] {
        int n = 4;
        if (const char *env = getenv("RTB_HOST_COPY_THREADS")) n = atoi(env);
        const int hw = (int)std::thread::hardware_concurrency();
        if (hw > 0) n = std::min(n, hw);
        return std::max(1, std::min(n, 16));
    }();
    if (n_threads == 1 || bytes < ((size_t)4 << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    const size_t part = ((bytes / n_threads) + 4095) & ~(size_t)4095;
    std::vector<std::thread> workers;
    for (int t = 1; t < n_threads; t++) {
        const size_t lo = std::min(bytes, part * t), hi = std::min(bytes, part * (t + 1));
        if (hi > lo) workers.emplace_back([=] { memcpy((char *)dst + lo, (const char *)src + lo, hi - lo); });
    }
    memcpy(dst, src, std::min(bytes, part));
    for (std::thread &w : workers) w.join();
}

// RTB_HOST_LAG=0: the host pipeline without the lagged copy-out (see rtb_trace_host)
bool lag_default()
{
    static const bool lag = !(getenv("RTB_HOST_LAG") && atoi(getenv("RTB_HOST_LAG")) == 0);
    return lag;
}

bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

} // namespace

extern "C" {

int rtb_abi_version(void) { return RTB_ABI_VERSION; }

const char *rtb_last_error(void) { return g_err; }

int rtb_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int64_t rtb_launch_count(void) { return g_launches.load(); }

int rtb_tune(const char *key, int64_t value)
{
    if (!key) return fail(RTB_ERR_INVALID, "key is NULL");
    for (const Knob &k : kKnobs) {
        if (strcmp(key, k.key) != 0) continue;
        if (value < k.lo || value > k.hi) return fail(RTB_ERR_INVALID, "%s takes %lld .. %lld", key, k.lo, k.hi);
        k.value->store(value, std::memory_order_relaxed);
        // (setting the mode also forgets every cached verdict: tests start from a known state)
        if (k.value == &rtb::g_lean_pure) rtb::lean_forget_verdicts();
        return RTB_OK;
    }
    return fail(RTB_ERR_INVALID, "unknown tuning key '%s'", key);
}

int rtb_trace_device(const rtb_system *sys, const double *rays_in_dev, int64_t n_rays, double *out_dev,
                     const rtb_trace_opts *opts, int device, void *stream)
{
    rtb::TraceParams P;
    int rc = pack_params(sys, opts, P);
    if (rc) return rc;
    if (n_rays < 0) return fail(RTB_ERR_INVALID, "n_rays = %lld is negative", (long long)n_rays);
    if (n_rays > 0 && !rays_in_dev) return fail(RTB_ERR_INVALID, "rays_in_dev is NULL");
    if (n_rays > 0 && P.any_store && !out_dev) return fail(RTB_ERR_INVALID, "out_dev is NULL but the keep mode stores rays");
    OnDevice on;
    if ((rc = on.enter(device))) return rc;
    P.rays_in = rays_in_dev;
    P.out = out_dev;
    P.n_rays = n_rays;
    P.out_stride = 8 * (long long)n_rays;
    return launch(P, opts->precision, on, (cudaStream_t)stream);
}

int rtb_trace_source(const rtb_system *sys, const rtb_source *src, int64_t first_ray, int64_t n_rays,
                     double *out_dev, const rtb_trace_opts *opts, int device, void *stream)
{
    rtb::TraceParams P;
    int rc = pack_params(sys, opts, P);
    if (rc) return rc;
    if ((rc = pack_source(src, first_ray, n_rays, P.src))) return rc;
    if (n_rays > 0 && P.any_store && !out_dev) return fail(RTB_ERR_INVALID, "out_dev is NULL but the keep mode stores rays");
    OnDevice on;
    if ((rc = on.enter(device))) return rc;
    P.rays_in = nullptr;
    P.out = out_dev;
    P.n_rays = n_rays;
    P.out_stride = 8 * (long long)n_rays;
    return launch(P, opts->precision, on, (cudaStream_t)stream, nullptr, &P.src);
}

int rtb_trace_sources(const rtb_system *sys, const rtb_source *srcs, int32_t n_src, int64_t first_ray,
                      int64_t n_rays_each, double *out_dev, const rtb_trace_opts *opts, int device, void *stream)
{
    rtb::TraceParams P;
    int rc = pack_params(sys, opts, P);
    if (rc) return rc;
    if (!srcs) return fail(RTB_ERR_INVALID, "source list pointer is NULL");
    if (n_src < 1 || n_src > 65535) return fail(RTB_ERR_INVALID, "n_src = %d, expected 1 .. 65535", n_src);
    if (opts->flags & RTB_FLAG_PLANES_IN) return fail(RTB_ERR_INVALID, "RTB_FLAG_PLANES_IN has no meaning for sources");
    if (opts->flags & RTB_FLAG_INTERSECT_ONLY)
        return fail(RTB_ERR_UNSUPPORTED, "RTB_FLAG_INTERSECT_ONLY is not offered for sweeps (one source per call: rtb_trace_source)");
    std::vector<rtb::DevSource> list((size_t)n_src);
    for (int k = 0; k < n_src; k++)
        if ((rc = pack_source(srcs + k, first_ray, n_rays_each, list[(size_t)k]))) return rc;
    if (n_rays_each == 0) return RTB_OK;
    if (P.any_store && !out_dev) return fail(RTB_ERR_INVALID, "out_dev is NULL but the keep mode stores rays");
    OnDevice on;
    if ((rc = on.enter(device))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const long long split = g_sweep_split_rays.load(std::memory_order_relaxed);
    if (n_src > 1 && split >= 0 && n_rays_each >= split) {
        // one launch per source: rows [k n, (k + 1) n) of every kept slab, bucket k of the reductions
        const bool planes_out = (opts->flags & RTB_FLAG_PLANES_OUT) != 0;
        for (int k = 0; k < n_src; k++) {
            rtb::TraceParams Q = P;
            Q.src = list[(size_t)k];
            Q.src_list = nullptr;
            Q.n_src = 0;
            Q.rays_in = nullptr;
            Q.out = out_dev ? out_dev + (size_t)k * (size_t)n_rays_each * (planes_out ? 1 : 8) : nullptr;
            Q.n_rays = n_rays_each;
            Q.out_stride = 8 * (long long)n_rays_each * n_src;
            if (Q.red.stats) Q.red.stats += (long long)k * RTB_N_STATS;
            if (Q.red.grid) Q.red.grid += (long long)k * 3 * Q.red.grid_n * Q.red.grid_n;
            rtb::finish_reduce(Q.red);
            if ((rc = launch(Q, opts->precision, on, st, nullptr, &list[(size_t)k]))) return rc;
        }
        return RTB_OK;
    }
    // the list lives in stream-ordered device memory for exactly this launch (pageable source: the copy has staged
    // it by the time the call returns, so the vector may go out of scope)
    rtb::DevSource *list_dev = nullptr;
    const size_t bytes = sizeof(rtb::DevSource) * (size_t)n_src;
    if ((rc = ensure_pool(on.ctx, device))) return rc;
    if (cudaMallocFromPoolAsync((void **)&list_dev, bytes, on.ctx->pool, st) != cudaSuccess)
        return fail(RTB_ERR_NOMEM, "stream-ordered allocation of %zu bytes for the source list failed", bytes);
    cudaError_t e = cudaMemcpyAsync(list_dev, list.data(), bytes, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) {
        cudaFreeAsync(list_dev, st);
        return fail(RTB_ERR_CUDA, "copying the source list failed: %s", cudaGetErrorString(e));
    }
    P.src = list[0];
    P.src_list = list_dev;
    P.n_src = n_src;
    P.rays_in = nullptr;
    P.out = out_dev;
    P.n_rays = n_rays_each;
    P.out_stride = 8 * (long long)n_rays_each * n_src;
    rc = launch(P, opts->precision, on, st, nullptr, list.data());
    cudaFreeAsync(list_dev, st);
    return rc;
}

int rtb_trace_host(const rtb_system *sys, const double *rays_in_host, int64_t n_rays, double *out_host,
                   const rtb_trace_opts *opts, int device)
{
    rtb::TraceParams P;
    int rc = pack_params(sys, opts, P);
    if (rc) return rc;
    if (n_rays < 0) return fail(RTB_ERR_INVALID, "n_rays = %lld is negative", (long long)n_rays);
    if (n_rays == 0) return RTB_OK;
    if (!rays_in_host) return fail(RTB_ERR_INVALID, "rays_in_host is NULL");
    if (opts->flags & (RTB_FLAG_PLANES_IN | RTB_FLAG_PLANES_OUT))
        return fail(RTB_ERR_UNSUPPORTED, "the plane (8, N) layouts are offered by the device entry points only");
    const int slabs = n_out_slabs(sys, opts);
    if (slabs > 0 && !out_host) return fail(RTB_ERR_INVALID, "out_host is NULL but the keep mode stores rays");
    OnDevice on;
    if ((rc = on.enter(device))) return rc;
    DeviceCtx *ctx = on.ctx;
    std::lock_guard<std::mutex> lock(ctx->host_path);

    // chunk so that one chunk's output is ~64 MiB (RTB_HOST_CHUNK_MIB overrides; 8-128 MiB measured within 15%): big enough for PCIe efficiency,
    // small enough that the un-overlapped first copy-in and last copy-out stay a few per cent of the call
    const size_t row = 64;
    size_t target = (size_t)(slabs <= 1 && lag_default() ? 16 : 64) << 20;
    if (const char *env = getenv("RTB_HOST_CHUNK_MIB")) {
        const long v = atol(env);
        if (v >= 1 && v <= 4096) target = (size_t)v << 20;
    }
    long long chunk = (long long)(target / (row * (size_t)std::max(slabs, 1)));
    chunk = std::max<long long>(chunk, 1 << 14);
    chunk = std::min<long long>(chunk, 1 << 22);
    chunk = std::min<long long>(chunk, n_rays);
    chunk = (chunk + 127) / 128 * 128;

    const bool in_pinned = is_pinned(rays_in_host);
    const bool out_pinned = slabs > 0 && is_pinned(out_host);

    for (int s = 0; s < kSlots; s++) {
        Slot &sl = ctx->slot[s];
        if (!sl.stream) RTB_CUDA(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        if (!sl.done) RTB_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
        if (!sl.copied_in) RTB_CUDA(cudaEventCreateWithFlags(&sl.copied_in, cudaEventDisableTiming));
        if (!sl.lean_scratch) RTB_CUDA(cudaMalloc(&sl.lean_scratch, rtb::lean_scratch_bytes(1)));
        if ((rc = grow_dev(&sl.dev_in, &sl.dev_in_bytes, (size_t)chunk * row))) return rc;
        if (slabs > 0 && (rc = grow_dev(&sl.dev_out, &sl.dev_out_bytes, (size_t)chunk * row * slabs))) return rc;
        if (!in_pinned && (rc = grow_pin(&sl.pin_in, &sl.pin_in_bytes, (size_t)chunk * row))) return rc;
        if (slabs > 0 && !out_pinned && (rc = grow_pin(&sl.pin_out, &sl.pin_out_bytes, (size_t)chunk * row * slabs)))
            return rc;
    }

    struct Pending {
        bool active = false;
        long long r0 = 0, cnt = 0;
    } pending[kSlots];

    auto retire = [&](int s) -> int {
        Pending &pd = pending[s];
        if (!pd.active) return RTB_OK;
        Slot &sl = ctx->slot[s];
        RTB_CUDA(cudaEventSynchronize(sl.done));
        if (slabs > 0 && !out_pinned) {
            for (int j = 0; j < slabs; j++)
                staging_copy(out_host + ((size_t)j * n_rays + pd.r0) * 8, sl.pin_out + (size_t)j * pd.cnt * 8,
                             (size_t)pd.cnt * row);
        }
        pd.active = false;
        return RTB_OK;
    };

    // cudaMemcpy2DAsync refuses pitches above cudaDevAttrMaxPitch (2^31 - 1 bytes: N >= 2^25 rays); then, and for a
    // single slab, each slab's rows go out as one contiguous copy
    int max_pitch = 0;
    if (cudaDeviceGetAttribute(&max_pitch, cudaDevAttrMaxPitch, device) != cudaSuccess) max_pitch = 0;
    const bool strided_copy_ok = slabs > 1 && (size_t)n_rays * row <= (size_t)max_pitch;

    // Every error return below goes through drain(): copies into the caller's buffers that are still in flight must
    // have landed (or failed) before the call returns, whatever it returns.
    auto drain = [&]() {
        for (int s = 0; s < kSlots; s++)
            if (ctx->slot[s].stream) cudaStreamSynchronize(ctx->slot[s].stream);
    };
    auto cuda_failed = [&](cudaError_t e, const char *what) -> int {
        if (e == cudaSuccess) return RTB_OK;
        drain();
        return fail(RTB_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
    };
    // The copy-out of chunk c is issued BEHIND THE COPY-IN OF CHUNK c + 1 (an event wait on its own stream): a chunk's two
    // copies then no longer meet through the compute engine at every step -- the copy-out engine always has a finished
    // chunk waiting when it ends one, instead of idling through the next chunk's kernels (tools/ubench/copy_pipeline.cu
    // <chunk> <streams> 1 1 0 <lag>: 16 MiB chunks on 4 streams 24.15 -> 22.75 ms per 2 GiB, the rate of the same pipeline
    // WITHOUT kernels; RTB_HOST_LAG=0 switches it off).
    const bool lag = lag_default();
    auto copy_out = [&](long long c) -> int {
        const int s = (int)(c % kSlots);
        Slot &sl = ctx->slot[s];
        const long long r0 = c * chunk;
        const long long cnt = std::min<long long>(chunk, n_rays - r0);
        if (slabs > 0) {
            cudaError_t e = cudaSuccess;
            if (!out_pinned) {
                e = cudaMemcpyAsync(sl.pin_out, sl.dev_out, (size_t)cnt * row * slabs, cudaMemcpyDeviceToHost, sl.stream);
            } else if (strided_copy_ok) {
                // (slabs, cnt, 8) device -> rows [r0, r0+cnt) of every slab of the (slabs, N, 8) host array
                e = cudaMemcpy2DAsync(out_host + (size_t)r0 * 8, (size_t)n_rays * row, sl.dev_out, (size_t)cnt * row,
                                      (size_t)cnt * row, (size_t)slabs, cudaMemcpyDeviceToHost, sl.stream);
            } else {
                for (int j = 0; j < slabs && e == cudaSuccess; j++)
                    e = cudaMemcpyAsync(out_host + ((size_t)j * n_rays + r0) * 8, sl.dev_out + (size_t)j * cnt * 8,
                                        (size_t)cnt * row, cudaMemcpyDeviceToHost, sl.stream);
            }
            if ((rc = cuda_failed(e, "copy-out"))) return rc;
        }
        if ((rc = cuda_failed(cudaEventRecord(sl.done, sl.stream), "cudaEventRecord"))) return rc;
        pending[s].active = true;
        pending[s].r0 = r0;
        pending[s].cnt = cnt;
        return RTB_OK;
    };
    auto run_pipeline = [&]() -> int {
        // (equal chunks: ones that taper towards both ends of the call -- to shrink the copy-in and copy-out that have
        // nothing to overlap with -- were measured twice, rounds 1 and 2, and change nothing: DESIGN.md section 8)
        const long long n_chunks = (n_rays + chunk - 1) / chunk;
        for (long long c = 0; c < n_chunks; c++) {
            const int s = (int)(c % kSlots);
            if ((rc = retire(s))) return rc;
            Slot &sl = ctx->slot[s];
            const long long r0 = c * chunk;
            const long long cnt = std::min<long long>(chunk, n_rays - r0);
            const double *src = rays_in_host + (size_t)r0 * 8;
            if (!in_pinned) {
                staging_copy(sl.pin_in, src, (size_t)cnt * row);
                src = sl.pin_in;
            }
            if ((rc = cuda_failed(cudaMemcpyAsync(sl.dev_in, src, (size_t)cnt * row, cudaMemcpyHostToDevice, sl.stream),
                                  "copy-in")))
                return rc;
            if (lag && (rc = cuda_failed(cudaEventRecord(sl.copied_in, sl.stream), "cudaEventRecord"))) return rc;
            P.rays_in = sl.dev_in;
            P.out = sl.dev_out;
            P.n_rays = cnt;
            P.out_stride = 8 * cnt;
            if (c == g_host_fail_chunk.load(std::memory_order_relaxed))
                return fail(RTB_ERR_CUDA, "injected failure before the launch of chunk %lld (rtb_tune host_fail_chunk)", c);
            if ((rc = launch(P, opts->precision, on, sl.stream, sl.lean_scratch))) return rc;
            if (!lag) {
                if ((rc = copy_out(c))) return rc;
            } else if (c > 0) {
                if ((rc = cuda_failed(cudaStreamWaitEvent(ctx->slot[(c - 1) % kSlots].stream, sl.copied_in, 0),
                                      "cudaStreamWaitEvent")))
                    return rc;
                if ((rc = copy_out(c - 1))) return rc;
            }
        }
        if (lag && n_chunks > 0 && (rc = copy_out(n_chunks - 1))) return rc;
        // drain in issue order
        for (long long c = n_chunks; c < n_chunks + kSlots; c++)
            if ((rc = retire((int)(c % kSlots)))) return rc;
        return RTB_OK;
    };
    rc = run_pipeline();
    if (rc) drain();
    return rc;
}

int rtb_generate_device(const rtb_source *src, int64_t first_ray, int64_t n_rays, double *rays_out_dev, int device,
                        void *stream)
{
    rtb::DevSource d;
    int rc = pack_source(src, first_ray, n_rays, d);
    if (rc) return rc;
    if (n_rays == 0) return RTB_OK;
    if (!rays_out_dev) return fail(RTB_ERR_INVALID, "rays_out_dev is NULL");
    OnDevice on;
    if ((rc = on.enter(device))) return rc;
    return launched(rtb::launch_generate(d, n_rays, rays_out_dev, on.ctx->sm_count, (cudaStream_t)stream),
                    "generator launch failed", 1);
}

int rtb_reduce_init(const rtb_reduce *red, int device, void *stream)
{
    if (!red) return fail(RTB_ERR_INVALID, "reduce pointer is NULL");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    rtb::DevReduce d;
    memset(&d, 0, sizeof(d));
    d.stats = red->stats_dev;
    d.grid = red->grid_n > 0 ? red->grid_dev : nullptr;
    d.grid_n = red->grid_n;
    rtb::finish_reduce(d);
    if (!d.stats && !d.grid) return RTB_OK;
    return launched(rtb::launch_reduce_init(d, on.ctx->sm_count, (cudaStream_t)stream), "reduce-init launch failed", 1);
}

int rtb_intersect_rays_device(const double *ray1_dev, int64_t n1, const double *ray2_dev, int64_t n2,
                              double *pts_out_dev, int device, void *stream)
{
    if (n1 < 0 || n2 < 0) return fail(RTB_ERR_INVALID, "negative ray count");
    if (!(n1 == n2 || n1 == 1 || n2 == 1)) return fail(RTB_ERR_INVALID, "ray1 and ray2 must be the same length");
    if (n1 == 0 || n2 == 0) return RTB_OK;
    if (!ray1_dev || !ray2_dev || !pts_out_dev) return fail(RTB_ERR_INVALID, "NULL device pointer");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    return launched(rtb::launch_intersect(ray1_dev, n1, ray2_dev, n2, pts_out_dev, (cudaStream_t)stream),
                    "intersect launch failed", 1);
}

int rtb_ray2plane_device(const double *rays_dev, int64_t n_rays, const double *normal_dev, int64_t n_normal,
                         const double *center_dev, int64_t n_center, const double *index_dev, int exclude_backward,
                         double *rays_out_dev, double *ts_out_dev, int device, void *stream)
{
    if (n_rays < 0) return fail(RTB_ERR_INVALID, "n_rays is negative");
    if (n_rays == 0) return RTB_OK;
    if (!(n_normal == 1 || n_normal == n_rays) || !(n_center == 1 || n_center == n_rays))
        return fail(RTB_ERR_INVALID, "normal / center must have 1 or n_rays rows");
    if (!rays_dev || !normal_dev || !center_dev || !index_dev || !rays_out_dev || !ts_out_dev)
        return fail(RTB_ERR_INVALID, "NULL device pointer");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    return launched(rtb::launch_ray2plane(rays_dev, n_rays, normal_dev, n_normal, center_dev, n_center, index_dev,
                                          exclude_backward, rays_out_dev, ts_out_dev, (cudaStream_t)stream),
                    "ray2plane launch failed", 1);
}

int rtb_distinct_wavelengths_device(const double *rays_dev, int64_t n_rays, double *table_dev,
                                    double *wavelengths_host, int32_t *n_found, int device, void *stream)
{
    if (n_rays < 0) return fail(RTB_ERR_INVALID, "n_rays is negative");
    if (!table_dev || !wavelengths_host || !n_found) return fail(RTB_ERR_INVALID, "NULL pointer");
    if (n_rays > 0 && !rays_dev) return fail(RTB_ERR_INVALID, "rays_dev is NULL");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    int found = 0;
    double vals[RTB_MAX_WAVELENGTHS + 1];
    if ((rc = launched(rtb::run_distinct_wavelengths(rays_dev, n_rays, table_dev, RTB_MAX_WAVELENGTHS + 1, vals, &found,
                                                     on.ctx->sm_count, (cudaStream_t)stream),
                       "distinct-wavelength scan failed", n_rays > 0 ? 2 : 1)))
        return rc;
    std::sort(vals, vals + found);
    for (int k = 0; k < found; k++) wavelengths_host[k] = vals[k];
    *n_found = found;
    return RTB_OK;
}

int rtb_distinct_wavelengths_host(const double *rays_host, int64_t n_rays, double *wavelengths_out, int32_t *n_found)
{
    if (n_rays < 0 || !wavelengths_out || !n_found) return fail(RTB_ERR_INVALID, "bad arguments");
    if (n_rays > 0 && !rays_host) return fail(RTB_ERR_INVALID, "rays_host is NULL");
    constexpr int cap = RTB_MAX_WAVELENGTHS + 1;
    unsigned hw = std::thread::hardware_concurrency();
    int n_threads = (int)std::min<int64_t>(std::max(1u, std::min(hw, 16u)), std::max<int64_t>(1, n_rays / 65536));
    struct Local {
        uint64_t v[cap];
        int n = 0;
    };
    std::vector<Local> found(n_threads);
    auto scan = [&](int t) {
        Local &L = found[t];
        const int64_t lo = n_rays * t / n_threads, hi = n_rays * (t + 1) / n_threads;
        uint64_t last = 0;
        bool have_last = false;
        for (int64_t i = lo; i < hi && L.n < cap; i++) {
            const double w = rays_host[8 * i + 7];
            if (w != w) continue;
            uint64_t bits;
            memcpy(&bits, &w, 8);
            if (have_last && bits == last) continue;
            last = bits;
            have_last = true;
            int k = 0;
            while (k < L.n && L.v[k] != bits) k++;
            if (k == L.n) L.v[L.n++] = bits;
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < n_threads; t++) pool.emplace_back(scan, t);
    scan(0);
    for (auto &th : pool) th.join();
    uint64_t all[cap];
    int n = 0;
    for (int t = 0; t < n_threads && n < cap; t++)
        for (int k = 0; k < found[t].n && n < cap; k++) {
            int j = 0;
            while (j < n && all[j] != found[t].v[k]) j++;
            if (j == n) all[n++] = found[t].v[k];
        }
    double vals[cap];
    for (int k = 0; k < n; k++) memcpy(&vals[k], &all[k], 8);
    std::sort(vals, vals + n);
    for (int k = 0; k < n; k++) wavelengths_out[k] = vals[k];
    *n_found = n;
    return RTB_OK;
}

int64_t rtb_psf_scratch_doubles(int grid_n, int n_samples, int normalize_by_count)
{
    if (grid_n <= 0 || n_samples <= 0) return 0;
    return rtb::psf_scratch_doubles(grid_n, n_samples, normalize_by_count);
}

int rtb_psf_from_grid_device(const double *grid_dev, int grid_n, double grid_half_width, int n_samples, double df,
                             int normalize_by_count, double *scratch_dev, int64_t scratch_doubles, double *psf_out_dev,
                             double *field_re_dev, double *field_im_dev, int device, void *stream)
{
    if (!grid_dev || grid_n <= 0 || n_samples <= 0 || !(grid_half_width > 0) || !(df > 0))
        return fail(RTB_ERR_INVALID, "psf: need a grid, grid_n > 0, n_samples > 0, grid_half_width > 0, df > 0");
    if (!psf_out_dev && !(field_re_dev && field_im_dev)) return fail(RTB_ERR_INVALID, "psf: no output requested");
    if (!scratch_dev || scratch_doubles < rtb::psf_scratch_doubles(grid_n, n_samples, normalize_by_count))
        return fail(RTB_ERR_INVALID, "psf: scratch buffer too small (see rtb_psf_scratch_doubles)");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    int launches = 0;
    cudaError_t e = rtb::launch_psf(grid_dev, grid_n, grid_half_width, n_samples, df, normalize_by_count, scratch_dev,
                                    psf_out_dev, field_re_dev, field_im_dev, on.ctx->sm_count, (cudaStream_t)stream,
                                    &launches);
    return launched(e, "psf launch failed", launches);
}

int rtb_selftest_exact_math(int device, uint64_t seed, int64_t n_cases, uint64_t mismatches[3])
{
    if (!mismatches || n_cases < 0) return fail(RTB_ERR_INVALID, "bad arguments");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    unsigned long long bad[3] = {0, 0, 0};
    if ((rc = launched(rtb::run_exact_math_selftest(seed, n_cases, bad, on.ctx->sm_count),
                       "exact-math self-test failed to run", 1)))
        return rc;
    for (int k = 0; k < 3; k++) mismatches[k] = bad[k];
    return RTB_OK;
}

int rtb_measure_dfma_rate(int device, double *dfma_per_s, double *elapsed_ms)
{
    if (!dfma_per_s) return fail(RTB_ERR_INVALID, "dfma_per_s is NULL");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    double ms = 0;
    if ((rc = launched(rtb::run_dfma_probe(on.ctx->sm_count, dfma_per_s, &ms), "DFMA probe failed", 0))) return rc;
    if (elapsed_ms) *elapsed_ms = ms;
    return RTB_OK;
}

int rtb_measure_dfma_chain_rate(int device, int chains, double *dfma_per_s, double *elapsed_ms)
{
    if (!dfma_per_s) return fail(RTB_ERR_INVALID, "dfma_per_s is NULL");
    if (chains != 1 && chains != 2 && chains != 4 && chains != 8) return fail(RTB_ERR_INVALID, "chains must be 1, 2, 4 or 8");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    double ms = 0;
    if ((rc = launched(rtb::run_dfma_chain_probe(on.ctx->sm_count, chains, dfma_per_s, &ms), "DFMA chain probe failed", 0)))
        return rc;
    if (elapsed_ms) *elapsed_ms = ms;
    return RTB_OK;
}

int rtb_measure_copy_bandwidth(int device, int64_t bytes, double *bytes_per_s)
{
    if (!bytes_per_s || bytes <= 0) return fail(RTB_ERR_INVALID, "bad arguments");
    OnDevice on;
    int rc;
    if ((rc = on.enter(device))) return rc;
    return launched(rtb::run_copy_probe(bytes, bytes_per_s), "copy probe failed", 0);
}

void *rtb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        fail(RTB_ERR_NOMEM, "cudaHostAlloc of %zu bytes failed", bytes);
        return nullptr;
    }
    return p;
}

void rtb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

} // extern "C"
