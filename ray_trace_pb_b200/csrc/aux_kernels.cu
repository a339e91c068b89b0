// aux_kernels.cu -- the small kernels around the fused trace: stand-alone ray sources, reduction buffers,
// intersect_rays, and the two roofline probes.  Compiled with -fmad=false like the trace (the bit-exact kernels
// rely on it; the DFMA probe asks for fused multiply-adds explicitly).
#include <cmath>
#include <math_constants.h>

#include "exact_math.cuh"
#include "rtb_device.cuh"

namespace rtb {

namespace {

constexpr double kTwoPi = 6.283185307179586;

__device__ __forceinline__ double linspace_at(long long i, long long n, double start, double step, double stop)
{
    const double v = (double)i * step + start;
    return (n > 1 && i == n - 1) ? stop : v;
}

// Stand-alone version of the trace kernel's ray source (get_ray_fan raytrace.py:45-96, get_collimated_rays 99-161,
// Cartesian grid).  Same index conventions and operation order as make_ray() in trace_f64.cu.
__global__ void __launch_bounds__(256) generate_kernel(const __grid_constant__ DevSource g, long long n_rays,
                                                       double *__restrict__ out)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_rays; i += stride) {
        const long long idx = g.first + i;
        double ox, oy, oz, dx, dy, dz;
        if (g.kind == RTB_SRC_GRID) {
            const long long iu = idx % g.n_a, iv = idx / g.n_a;
            const double u = linspace_at(iu, g.n_a, g.a_start, g.a_step, g.a_stop);
            const double v = linspace_at(iv, g.n_b, g.b_start, g.b_step, g.b_stop);
            ox = (g.px + g.e1x * u) + g.e2x * v;
            oy = (g.py + g.e1y * u) + g.e2y * v;
            oz = (g.pz + g.e1z * u) + g.e2z * v;
            dx = g.axx; dy = g.axy; dz = g.axz;
        } else if (g.kind == RTB_SRC_COLLIMATED) {
            const long long ip = idx % g.n_b, id = idx / g.n_b;
            const double off = linspace_at(id, g.n_a, g.a_start, g.a_step, g.a_stop);
            const double phi = ((double)ip * kTwoPi) / (double)g.n_b + g.b_start;
            double sp, cp;
            sincos(phi, &sp, &cp);
            const double a = off * cp, b = off * sp;
            ox = (g.px + g.e1x * a) + g.e2x * b;
            oy = (g.py + g.e1y * a) + g.e2y * b;
            oz = (g.pz + g.e1z * a) + g.e2z * b;
            dx = g.axx; dy = g.axy; dz = g.axz;
        } else {
            const long long it = idx % g.n_a, ip = idx / g.n_a;
            const double theta = linspace_at(it, g.n_a, g.a_start, g.a_step, g.a_stop);
            const double phi = ((double)ip * kTwoPi) / (double)g.n_b;
            double st, ct, sp, cp;
            sincos(theta, &st, &ct);
            sincos(phi, &sp, &cp);
            ox = g.px; oy = g.py; oz = g.pz;
            dx = (g.axx * ct + (g.e1x * cp) * st) + (g.e2x * sp) * st;
            dy = (g.axy * ct + (g.e1y * cp) * st) + (g.e2y * sp) * st;
            dz = (g.axz * ct + (g.e1z * cp) * st) + (g.e2z * sp) * st;
        }
        double *p = out + 8 * i;
        st256(p, ox, oy, oz, dx);
        st256(p + 4, dy, dz, 0.0, g.wavelength);
    }
}

__global__ void reduce_init_kernel(DevReduce r)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r.stats && tid < RTB_N_STATS) {
        double v = 0.0;
        if (tid == 8 || tid == 10) v = CUDART_INF;
        if (tid == 9 || tid == 11) v = -CUDART_INF;
        r.stats[tid] = v;
    }
    if (r.grid) {
        const long long n = 3LL * r.grid_n * r.grid_n;
        for (long long i = tid; i < n; i += stride) r.grid[i] = 0.0;
    }
}

// intersect_rays (raytrace.py:164-238); either input may be a single ray broadcast against the other (175-182)
__global__ void __launch_bounds__(256) intersect_kernel(const double *__restrict__ r1, long long n1,
                                                        const double *__restrict__ r2, long long n2,
                                                        double *__restrict__ out, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *a = r1 + 8 * (n1 == 1 ? 0 : i);
    const double *b = r2 + 8 * (n2 == 1 ? 0 : i);
    const double x1 = a[0], y1 = a[1], z1 = a[2], dx1 = a[3], dy1 = a[4], dz1 = a[5];
    const double x2 = b[0], y2 = b[1], z2 = b[2], dx2 = b[3], dy2 = b[4], dz2 = b[5];
    const double nan = CUDART_NAN;

    // distance along ray 2 from whichever 2x2 sub-system is non-singular (raytrace.py:205-217)
    const double det_xz = dx2 * dz1 - dz2 * dx1;
    const double det_xy = dx2 * dy1 - dy2 * dx1;
    const double det_yz = dz2 * dy1 - dy2 * dz1;
    const bool use_xz = det_xz != 0.0;
    const bool use_xy = !use_xz && (det_xy != 0.0);
    const bool use_yz = !use_xz && !use_xy && (det_yz != 0.0);
    double s = nan;
    if (use_xz) s = ((z2 - z1) * dx1 - (x2 - x1) * dz1) / det_xz;
    if (use_xy) s = ((y2 - y1) * dx1 - (x2 - x1) * dy1) / det_xy;
    if (use_yz) s = ((y2 - y1) * dz1 - (z2 - z1) * dy1) / det_yz;

    // distance along ray 1 (raytrace.py:220-228)
    const bool use_z = dz1 != 0.0;
    const bool use_y = !use_z && (dy1 != 0.0);
    double t;
    if (use_z)
        t = ((z2 + s * dz2) - z1) / dz1;
    else if (use_y)
        t = ((y2 + s * dy2) - y1) / dy1;
    else
        t = ((x2 + s * dx2) - x1) / dx1;

    double px = x1 + t * dx1, py = y1 + t * dy1, pz = z1 + t * dz1;
    const double qx = x2 + s * dx2, qy = y2 + s * dy2, qz = z2 + s * dz2;
    // np.max propagates NaN and NaN > 1e-12 is False (raytrace.py:234-236)
    const double ex = fabs(px - qx), ey = fabs(py - qy), ez = fabs(pz - qz);
    double m = ex;
    m = (ey > m) ? ey : m;
    m = (ez > m) ? ez : m;
    const bool any_nan = (ex != ex) || (ey != ey) || (ez != ez);
    if (!any_nan && m > 1e-12) {
        px = nan; py = nan; pz = nan;
    }
    out[3 * i] = px;
    out[3 * i + 1] = py;
    out[3 * i + 2] = pz;
}

// propagate_ray2plane (raytrace.py:241-306) with per-ray plane normal / centre and a per-ray refractive index
__global__ void __launch_bounds__(256) ray2plane_kernel(const double *__restrict__ rays, long long n,
                                                        const double *__restrict__ normal, long long n_normal,
                                                        const double *__restrict__ center, long long n_center,
                                                        const double *__restrict__ index, int exclude_backward,
                                                        double *__restrict__ out, double *__restrict__ ts)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *r = rays + 8 * i;
    const double *nm = normal + 3 * (n_normal == 1 ? 0 : i);
    const double *c = center + 3 * (n_center == 1 ? 0 : i);
    const double ox = r[0], oy = r[1], oz = r[2], dx = r[3], dy = r[4], dz = r[5], ph = r[6], wl = r[7];
    const double num = ((ox - c[0]) * nm[0] + (oy - c[1]) * nm[1]) + (oz - c[2]) * nm[2];
    const double den = (dx * nm[0] + dy * nm[1]) + dz * nm[2];
    const double t = (-num) / den;
    const double vx = dx * t, vy = dy * t, vz = dz * t;
    double len = sqrt((vx * vx + vy * vy) + vz * vz);
    len = (t < 0.0) ? -len : len;
    const bool kill = exclude_backward && (t < 0.0);
    const double q = CUDART_NAN;
    double *o = out + 8 * i;
    o[0] = kill ? q : ox + vx;
    o[1] = kill ? q : oy + vy;
    o[2] = kill ? q : oz + vz;
    o[3] = kill ? q : dx;
    o[4] = kill ? q : dy;
    o[5] = kill ? q : dz;
    o[6] = kill ? q : ph + ((len * kTwoPi) / wl) * index[i];
    o[7] = kill ? q : wl;
    ts[i] = t;
}

// Collect the distinct non-NaN wavelength bit patterns of a batch into a small table (slots start as kEmptySlot).
constexpr unsigned long long kEmptySlot = 0x7FF8C0DEC0DEC0DEull; // a NaN payload no wavelength can equal
__global__ void __launch_bounds__(256) distinct_wavelengths_kernel(const double *__restrict__ rays, long long n,
                                                                   unsigned long long *table, int capacity)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double w = rays[8 * i + 7];
        if (w != w) continue;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(w);
        int slot = 0;
        for (; slot < capacity; slot++) {
            unsigned long long cur = *((volatile unsigned long long *)(table + slot));
            if (cur == bits) break;
            if (cur == kEmptySlot) {
                cur = atomicCAS(table + slot, kEmptySlot, bits);
                if (cur == kEmptySlot || cur == bits) break;
            }
        }
        // slot == capacity: more distinct values than the table holds; the last slot then stays full and the host
        // sees "capacity" entries, which it reports as overflow (capacity = RTB_MAX_WAVELENGTHS + 1).
    }
}

__global__ void fill_u64_kernel(unsigned long long *p, int n, unsigned long long v)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ---- self-test of exact_math.cuh against the built-in IEEE operators ------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__device__ __forceinline__ double test_operand(unsigned long long h, int category)
{
    const double specials[16] = {0.0, -0.0, 1.0, -1.0, CUDART_INF, -CUDART_INF, CUDART_NAN, 4.9406564584124654e-324,
                                 2.2250738585072014e-308, 1.7976931348623157e308, 1e-300, 1e300, 0.5, 3.0,
                                 1.0000000000000002, 6.283185307179586};
    if (category == 0) return __longlong_as_double((long long)h);                 // raw bits: every class of double
    if (category == 2) return specials[h & 15];
    // moderate magnitudes: random mantissa and sign, exponent within 2^-40 .. 2^40 (category 1) or 2^-3..2^3 (3)
    const int span = (category == 1) ? 81 : 7;
    const unsigned long long expo = 1023ull - span / 2 + (h >> 52) % span;
    return __longlong_as_double((long long)((h & 0x800FFFFFFFFFFFFFull) | (expo << 52)));
}

__device__ __forceinline__ bool same_bits(double a, double b)
{
    return (a != a && b != b) || (__double_as_longlong(a) == __double_as_longlong(b));
}

__global__ void __launch_bounds__(256) exact_math_selftest_kernel(unsigned long long seed, long long n,
                                                                  unsigned long long *bad)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long bad_div = 0, bad_div3 = 0, bad_sqrt = 0;
    __shared__ double2 near_one_tab[xm::kNearOneEntries];
    for (int k = threadIdx.x; k < xm::kNearOneEntries; k += blockDim.x) near_one_tab[k] = xm::near_one_entry(k);
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int cat = (int)(i & 3);
        const unsigned long long h0 = splitmix64(seed ^ (unsigned long long)(4 * i));
        const double b = test_operand(splitmix64(h0), cat);
        double a0 = test_operand(splitmix64(h0 + 1), cat);
        double a1 = test_operand(splitmix64(h0 + 2), cat == 3 ? 2 : cat);       // zeros next to ordinary numbers
        double a2 = test_operand(splitmix64(h0 + 3), cat);
        if (cat == 3 && (h0 & 8)) a2 = b * 1.0000000000000002;                   // quotients next to 1
        bad_div += !same_bits(xm::div(a0, b), a0 / b);
        const xm::Rcp r = xm::make_rcp(b);
        bad_div += !same_bits(xm::div(a1, r), a1 / b);
        double x = a0, y = a1, z = a2;
        xm::div3(x, y, z, r);
        bad_div3 += !(same_bits(x, a0 / b) && same_bits(y, a1 / b) && same_bits(z, a2 / b));
        bad_sqrt += !same_bits(xm::sqrt(a0), sqrt(a0));
        bad_sqrt += !same_bits(xm::sqrt(fabs(a2)), sqrt(fabs(a2)));
        // the near-one table: every s = bits(1.0) + k, k in [-128, 127], passes, and a numerator of moderate size (those
        // of lean_steps.cuh are components of a vector of norm sqrt(s)) is divided by it as c / sqrt(s) divides; the
        // doubles next to either end of the table fail
        const long long k = (long long)((i >> 2) & (xm::kNearOneEntries - 1)) - xm::kNearOneEntries / 2;
        const double s = __longlong_as_double(0x3FF0000000000000ll + k);
        const double c = (cat & 1) ? a0 : test_operand(splitmix64(h0 + 4), 1);
        bool in = true, below = true, above = true;
        const double2 lr = xm::near_one(in, s, near_one_tab);
        xm::near_one(below, __longlong_as_double(0x3FF0000000000000ll - xm::kNearOneEntries / 2 - 1), near_one_tab);
        xm::near_one(above, __longlong_as_double(0x3FF0000000000000ll + xm::kNearOneEntries / 2), near_one_tab);
        bad_div += !in | below | above;
        if (xm::num_ok(c)) bad_div += !same_bits(xm::div_core(c, lr.x, lr.y), c / sqrt(s));
    }
    if (bad_div) atomicAdd(bad + 0, bad_div);
    if (bad_div3) atomicAdd(bad + 1, bad_div3);
    if (bad_sqrt) atomicAdd(bad + 2, bad_sqrt);
}

// Register-only DFMA throughput: 8 independent chains per thread, explicit fused multiply-adds.
__global__ void __launch_bounds__(256) dfma_probe_kernel(double *sink, int iters, double seed)
{
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
           a7 = a0 + 7;
    const double m = 0.999999, c = 1e-9;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            a0 = __fma_rn(a0, m, c); a1 = __fma_rn(a1, m, c); a2 = __fma_rn(a2, m, c); a3 = __fma_rn(a3, m, c);
            a4 = __fma_rn(a4, m, c); a5 = __fma_rn(a5, m, c); a6 = __fma_rn(a6, m, c); a7 = __fma_rn(a7, m, c);
        }
    }
    const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456) sink[0] = r; // never true; keeps the chains alive
}

// FP64 issue rate of latency-bound code: CHAINS independent dependent-DFMA chains per thread at the trace kernels' own
// occupancy (7 warps per scheduler).  One chain per warp is what a ray through a surface looks like to the pipe: every
// FP64 instruction then follows one of ANOTHER warp, which costs 3 cycles instead of 2 (DESIGN.md 4a).
template <int CHAINS>
__global__ void __launch_bounds__(128) dfma_chain_probe_kernel(double *sink, int iters, double m, double c)
{
    double a[CHAINS];
#pragma unroll
    for (int k = 0; k < CHAINS; k++) a[k] = 1.0 + threadIdx.x * 1e-9 + k;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
#pragma unroll
            for (int k = 0; k < CHAINS; k++) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(a[k]) : "d"(m), "d"(c));
        }
    }
    double r = 0.0;
#pragma unroll
    for (int k = 0; k < CHAINS; k++) r += a[k];
    if (r == 123.456) sink[0] = r; // never true; keeps the chains alive
}

__global__ void copy_probe_kernel(const double4 *__restrict__ in, double4 *__restrict__ out, long long n)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = in[i];
}

} // namespace

cudaError_t launch_generate(const DevSource &src, long long n_rays, double *out, int sm_count, cudaStream_t stream)
{
    if (n_rays <= 0) return cudaSuccess;
    long long blocks = (n_rays + 255) / 256;
    blocks = blocks > (long long)sm_count * 8 ? (long long)sm_count * 8 : blocks;
    generate_kernel<<<(unsigned)blocks, 256, 0, stream>>>(src, n_rays, out);
    return cudaGetLastError();
}

cudaError_t launch_reduce_init(const DevReduce &red, int sm_count, cudaStream_t stream)
{
    reduce_init_kernel<<<sm_count * 4, 256, 0, stream>>>(red);
    return cudaGetLastError();
}

cudaError_t launch_intersect(const double *r1, long long n1, const double *r2, long long n2, double *out,
                             cudaStream_t stream)
{
    const long long n = n1 > n2 ? n1 : n2;
    if (n <= 0) return cudaSuccess;
    intersect_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(r1, n1, r2, n2, out, n);
    return cudaGetLastError();
}

cudaError_t launch_ray2plane(const double *rays, long long n, const double *normal, long long n_normal,
                             const double *center, long long n_center, const double *index, int exclude_backward,
                             double *out, double *ts, cudaStream_t stream)
{
    if (n <= 0) return cudaSuccess;
    ray2plane_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(rays, n, normal, n_normal, center, n_center,
                                                                      index, exclude_backward, out, ts);
    return cudaGetLastError();
}

// table_dev: capacity slots.  Returns the distinct values (unsorted) in host_out and their count in *n_found.
cudaError_t run_distinct_wavelengths(const double *rays, long long n, double *table_dev, int capacity,
                                     double *host_out, int *n_found, int sm_count, cudaStream_t stream)
{
    unsigned long long *tab = reinterpret_cast<unsigned long long *>(table_dev);
    fill_u64_kernel<<<1, 64, 0, stream>>>(tab, capacity, kEmptySlot);
    if (n > 0) {
        long long blocks = (n + 255) / 256;
        blocks = blocks > (long long)sm_count * 8 ? (long long)sm_count * 8 : blocks;
        distinct_wavelengths_kernel<<<(unsigned)blocks, 256, 0, stream>>>(rays, n, tab, capacity);
    }
    unsigned long long host[64];
    cudaError_t e = cudaMemcpyAsync(host, tab, sizeof(unsigned long long) * capacity, cudaMemcpyDeviceToHost, stream);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return e;
    int count = 0;
    for (int k = 0; k < capacity; k++)
        if (host[k] != kEmptySlot) host_out[count++] = __builtin_bit_cast(double, host[k]);
    *n_found = count;
    return cudaGetLastError();
}

cudaError_t run_exact_math_selftest(unsigned long long seed, long long n, unsigned long long *bad_host, int sm_count)
{
    unsigned long long *bad = nullptr;
    cudaError_t e = cudaMalloc(&bad, 3 * sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    cudaMemset(bad, 0, 3 * sizeof(unsigned long long));
    exact_math_selftest_kernel<<<sm_count * 8, 256>>>(seed, n, bad);
    e = cudaMemcpy(bad_host, bad, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    cudaFree(bad);
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t run_dfma_probe(int sm_count, double *dfma_per_s, double *elapsed_ms)
{
    double *sink = nullptr;
    cudaError_t e = cudaMalloc(&sink, sizeof(double));
    if (e != cudaSuccess) return e;
    cudaEvent_t t0, t1;
    cudaEventCreate(&t0);
    cudaEventCreate(&t1);
    const int blocks = sm_count * 8, threads = 256, iters = 4096;
    dfma_probe_kernel<<<blocks, threads>>>(sink, 64, 1.0); // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(t0);
        dfma_probe_kernel<<<blocks, threads>>>(sink, iters, 1.0);
        cudaEventRecord(t1);
        e = cudaEventSynchronize(t1);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(sink);
    if (e != cudaSuccess) return e;
    const double ops = (double)blocks * threads * (double)iters * 64.0;
    *dfma_per_s = ops / (best * 1e-3);
    *elapsed_ms = best;
    return cudaGetLastError();
}

cudaError_t run_dfma_chain_probe(int sm_count, int chains, double *dfma_per_s, double *elapsed_ms)
{
    double *sink = nullptr;
    cudaError_t e = cudaMalloc(&sink, sizeof(double));
    if (e != cudaSuccess) return e;
    cudaEvent_t t0, t1;
    cudaEventCreate(&t0);
    cudaEventCreate(&t1);
    const int blocks = sm_count * 7, threads = 128, iters = 8192 / chains;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(t0);
        switch (chains) {
        case 1: dfma_chain_probe_kernel<1><<<blocks, threads>>>(sink, iters, 0.999999, 1e-9); break;
        case 2: dfma_chain_probe_kernel<2><<<blocks, threads>>>(sink, iters, 0.999999, 1e-9); break;
        case 4: dfma_chain_probe_kernel<4><<<blocks, threads>>>(sink, iters, 0.999999, 1e-9); break;
        default: dfma_chain_probe_kernel<8><<<blocks, threads>>>(sink, iters, 0.999999, 1e-9); break;
        }
        cudaEventRecord(t1);
        e = cudaEventSynchronize(t1);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(sink);
    if (e != cudaSuccess) return e;
    *dfma_per_s = (double)blocks * threads * (double)iters * 16.0 * chains / (best * 1e-3);
    *elapsed_ms = best;
    return cudaGetLastError();
}

cudaError_t run_copy_probe(long long bytes, double *bytes_per_s)
{
    const long long n = bytes / 32;
    double4 *a = nullptr, *b = nullptr;
    cudaError_t e = cudaMalloc(&a, n * 32);
    if (e != cudaSuccess) return e;
    e = cudaMalloc(&b, n * 32);
    if (e != cudaSuccess) {
        cudaFree(a);
        return e;
    }
    cudaMemset(a, 0, n * 32);
    cudaEvent_t t0, t1;
    cudaEventCreate(&t0);
    cudaEventCreate(&t1);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    float best = 1e30f;
    for (int rep = 0; rep < 6; rep++) {
        cudaEventRecord(t0);
        copy_probe_kernel<<<sms * 16, 256>>>(a, b, n);
        cudaEventRecord(t1);
        e = cudaEventSynchronize(t1);
        if (e != cudaSuccess) break;
        float ms = 0;
        cudaEventElapsedTime(&ms, t0, t1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(t0);
    cudaEventDestroy(t1);
    cudaFree(a);
    cudaFree(b);
    if (e != cudaSuccess) return e;
    *bytes_per_s = 2.0 * (double)n * 32.0 / (best * 1e-3);
    return cudaGetLastError();
}

// the fast modes live in trace_fast.cu

} // namespace rtb
