// psf_kernels.cu -- pupil grid -> PSF as a dense complex contraction (the "ray fan -> pupil phase -> PSF" tail of
// BASELINE.json; SURVEY.md 8f row 2).
//
// The reference only has this at script level (scripts/2022_02_06_perfect_imaging_system_psf.py:90-105): scattered
// pupil phases -> scipy griddata -> exp(i phi) -> mask -> fftshift(fft2(ifftshift(.))) -> |.|^2.  Here the pupil
// function is what the trace kernel accumulated per cell, P[v,u] = sum_rays exp(i (phi - phi_ref)) (optionally divided
// by the ray count of the cell), and the field at M x M image-plane sample points is the separable matrix product
//     E = A P B^T,   B[k,u] = exp(-2 pi i fx_k x_u),  A[l,v] = exp(-2 pi i fy_l y_v),   PSF = |E|^2
// with x_u, y_v the cell centres and fx_k, fy_l = (k - (M-1)/2) * df spatial frequencies (for a lens of focal length f:
// image coordinate = lambda f fx).  A "zoomed DFT": any sampling and window, no padding; for odd G, M = G and
// df = 1/(G*cell) it is exactly fftshift(fft2(ifftshift(P))) (odd M puts a sample on the zero frequency).
// fp64 throughout: tcgen05 has no f64 kind, so this runs on the FP64 pipe (64x64 register-tiled, K-split complex GEMM).
#include <atomic>
#include <cmath>
#include <math_constants.h>

#include "rtb_device.cuh"

namespace rtb {

// which contraction kernel runs: 1 = DMMA (mma.sync.m8n8k4.f64), 0 = the SIMT register-tiled one (rtb_tune "psf_dmma")
std::atomic<long long> g_psf_dmma{1};

namespace {

// P = (sum cos + i sum sin) / count, zero where the cell is empty.  Planar output (re plane, im plane).
__global__ void normalize_pupil_kernel(const double *__restrict__ grid, long long cells, double *__restrict__ re,
                                       double *__restrict__ im)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += stride) {
        const double c = grid[2 * cells + i];
        const double inv = c > 0.0 ? 1.0 / c : 0.0;
        re[i] = grid[i] * inv;
        im[i] = grid[cells + i] * inv;
    }
}

// D[k, u] = exp(-2 pi i f_k x_u), f_k = (k - (M-1)/2) df, x_u = (u + 0.5) cell - half.  Planar (M x G).
__global__ void dft_matrix_kernel(int M, int G, double df, double cell, double half, double *__restrict__ re,
                                  double *__restrict__ im)
{
    const long long n = (long long)M * G;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int k = (int)(i / G), u = (int)(i % G);
        const double f = ((double)k - 0.5 * (double)(M - 1)) * df;
        const double x = ((double)u + 0.5) * cell - half;
        double s, c;
        sincospi(-2.0 * f * x, &s, &c);
        re[i] = c;
        im[i] = s;
    }
}

// C[m, n] (+)= sum_{k in this block's K range} X[m, k] * Y[n, k]   (complex, planar, row-major; X is Mx x K, Y is Ny x K)
// 64 x 64 tile per block, 16 x 16 threads, 4 x 4 complex accumulators each; thread (ty, tx) owns rows ty + 16 a and
// columns tx + 16 b, so shared-memory reads are conflict-free (x: broadcast, y: consecutive doubles) and the stores
// of a warp are contiguous.  gridDim.z splits K: the output tiles of a 257 x 2048 or 257 x 257 product are far too
// few to fill 148 SMs (160 and 25), so each tile's K loop is shared by several blocks; block z writes its partial sums
// to slice z of `part` and sum_partials_kernel adds the slices in order -- the PSF is the same bits run to run (the
// first version added them with atomics, in whatever order the blocks finished).
constexpr int kTile = 64, kStep = 16;
__global__ void __launch_bounds__(256) zgemm_nt_kernel(int Mx, int Ny, int K, int k_chunk,
                                                       const double *__restrict__ x_re, const double *__restrict__ x_im,
                                                       const double *__restrict__ y_re, const double *__restrict__ y_im,
                                                       double *__restrict__ c_re, double *__restrict__ c_im)
{
    __shared__ double sxr[kStep][kTile + 1], sxi[kStep][kTile + 1], syr[kStep][kTile + 1], syi[kStep][kTile + 1];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int m0 = blockIdx.y * kTile, n0 = blockIdx.x * kTile;
    const int k_begin = blockIdx.z * k_chunk, k_end = min(K, k_begin + k_chunk);
    double ar[4][4] = {}, ai[4][4] = {};
    for (int k0 = k_begin; k0 < k_end; k0 += kStep) {
        // stage 64 x 16 of X and of Y: k is fastest in memory, so 16 consecutive threads read one 128-byte row piece;
        // the row stride of 65 doubles keeps the transposed shared-memory write conflict-free
        for (int e = threadIdx.x; e < kTile * kStep; e += 256) {
            const int r = e / kStep, kk = e % kStep;
            const int k = k0 + kk;
            const bool kin = k < k_end;
            const int m = m0 + r, n = n0 + r;
            sxr[kk][r] = (kin && m < Mx) ? x_re[(long long)m * K + k] : 0.0;
            sxi[kk][r] = (kin && m < Mx) ? x_im[(long long)m * K + k] : 0.0;
            syr[kk][r] = (kin && n < Ny) ? y_re[(long long)n * K + k] : 0.0;
            syi[kk][r] = (kin && n < Ny) ? y_im[(long long)n * K + k] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kStep; kk++) {
            double xr[4], xi[4], yr[4], yi[4];
#pragma unroll
            for (int a = 0; a < 4; a++) {
                xr[a] = sxr[kk][ty + 16 * a];
                xi[a] = sxi[kk][ty + 16 * a];
                yr[a] = syr[kk][tx + 16 * a];
                yi[a] = syi[kk][tx + 16 * a];
            }
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    ar[a][b] = fma(xr[a], yr[b], fma(-xi[a], yi[b], ar[a][b]));
                    ai[a][b] = fma(xr[a], yi[b], fma(xi[a], yr[b], ai[a][b]));
                }
        }
        __syncthreads();
    }
    // (split: c_re / c_im point at the partial-sum slices, slice stride = 2 * Mx * Ny doubles: re plane, im plane)
    const long long slice = (long long)blockIdx.z * 2 * Mx * Ny;
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int m = m0 + ty + 16 * a, n = n0 + tx + 16 * b;
            if (m < Mx && n < Ny) {
                const long long o = (long long)m * Ny + n;
                c_re[slice + o] = ar[a][b];
                c_im[slice + o] = ai[a][b];
            }
        }
}

// The same product on the FP64 tensor path: mma.sync.m8n8k4.f64 (DMMA).  64 x 64 tile per block, 8 warps as 4 (m) x 2 (n),
// each warp 16 x 32 = 2 x 4 fragments of 8 x 8; per k-step of 4 a warp loads 4 A fragments (X re / im of its two row
// groups) and 8 B fragments from shared memory and issues 32 DMMAs (re += Xr Yr; re += (-Xi) Yi; im += Xr Yi; im += Xi Yr).
// A DMMA does the work of eight DFMAs with four register operands, which is what the operand-read port (DESIGN.md 4a)
// leaves room for.  Shared tiles are k-major with a row stride of 68 doubles: a fragment read touches 16 distinct
// 8-byte banks per half warp.
constexpr int kPad = 68;
__device__ __forceinline__ void dmma(double &d0, double &d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) zgemm_nt_dmma_kernel(int Mx, int Ny, int K, int k_chunk,
                                                            const double *__restrict__ x_re, const double *__restrict__ x_im,
                                                            const double *__restrict__ y_re, const double *__restrict__ y_im,
                                                            double *__restrict__ c_re, double *__restrict__ c_im)
{
    __shared__ double sxr[kStep][kPad], sxi[kStep][kPad], syr[kStep][kPad], syi[kStep][kPad];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm = warp >> 1, wn = warp & 1;               // this warp's 16 x 32 piece of the tile
    const int g = lane >> 2, t = lane & 3;                 // fragment coordinates: group (row / column), thread in group (k)
    const int m0 = blockIdx.y * kTile, n0 = blockIdx.x * kTile;
    const int k_begin = blockIdx.z * k_chunk, k_end = min(K, k_begin + k_chunk);
    double cr[2][4][2] = {}, ci[2][4][2] = {};
    for (int k0 = k_begin; k0 < k_end; k0 += kStep) {
        for (int e = threadIdx.x; e < kTile * kStep; e += 256) {
            const int r = e / kStep, kk = e % kStep;
            const int k = k0 + kk;
            const bool kin = k < k_end;
            const int m = m0 + r, n = n0 + r;
            sxr[kk][r] = (kin && m < Mx) ? x_re[(long long)m * K + k] : 0.0;
            sxi[kk][r] = (kin && m < Mx) ? x_im[(long long)m * K + k] : 0.0;
            syr[kk][r] = (kin && n < Ny) ? y_re[(long long)n * K + k] : 0.0;
            syi[kk][r] = (kin && n < Ny) ? y_im[(long long)n * K + k] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kStep; kk += 4) {
            double ar[2], ai[2], an[2], br[4], bi[4];
#pragma unroll
            for (int a = 0; a < 2; a++) {
                ar[a] = sxr[kk + t][16 * wm + 8 * a + g];
                ai[a] = sxi[kk + t][16 * wm + 8 * a + g];
                an[a] = -ai[a];
            }
#pragma unroll
            for (int b = 0; b < 4; b++) {
                br[b] = syr[kk + t][32 * wn + 8 * b + g];
                bi[b] = syi[kk + t][32 * wn + 8 * b + g];
            }
#pragma unroll
            for (int a = 0; a < 2; a++)
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    dmma(cr[a][b][0], cr[a][b][1], ar[a], br[b]);
                    dmma(cr[a][b][0], cr[a][b][1], an[a], bi[b]);
                    dmma(ci[a][b][0], ci[a][b][1], ar[a], bi[b]);
                    dmma(ci[a][b][0], ci[a][b][1], ai[a], br[b]);
                }
        }
        __syncthreads();
    }
    const long long slice = (long long)blockIdx.z * 2 * Mx * Ny;
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 4; b++)
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int m = m0 + 16 * wm + 8 * a + g, n = n0 + 32 * wn + 8 * b + 2 * t + j;
                if (m < Mx && n < Ny) {
                    const long long o = (long long)m * Ny + n;
                    c_re[slice + o] = cr[a][b][j];
                    c_im[slice + o] = ci[a][b][j];
                }
            }
}

// C = sum over the K-split slices, in slice order
__global__ void sum_partials_kernel(const double *__restrict__ part, int split, long long n, double *__restrict__ c_re,
                                    double *__restrict__ c_im)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double re = 0.0, im = 0.0;
        for (int z = 0; z < split; z++) {
            re += part[(long long)z * 2 * n + i];
            im += part[(long long)z * 2 * n + n + i];
        }
        c_re[i] = re;
        c_im[i] = im;
    }
}

__global__ void abs2_kernel(const double *__restrict__ re, const double *__restrict__ im, long long n,
                            double *__restrict__ out)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = fma(re[i], re[i], im[i] * im[i]);
}

// K split so that the grid is at least ~4 waves of blocks (each block still loops over >= 4 k-steps)
int zgemm_split(int Mx, int Ny, int K, int sm_count, int *k_chunk_out)
{
    const int tiles = ((Mx + kTile - 1) / kTile) * ((Ny + kTile - 1) / kTile);
    int split = (4 * sm_count + tiles - 1) / tiles;
    split = max(1, min(split, K / (4 * kStep)));
    const int k_chunk = ((K + split - 1) / split + kStep - 1) / kStep * kStep;
    if (k_chunk_out) *k_chunk_out = k_chunk;
    return (K + k_chunk - 1) / k_chunk;
}

// `part`: scratch for split * 2 * Mx * Ny doubles (unused when the product is not split)
cudaError_t launch_zgemm(int Mx, int Ny, int K, const double *x_re, const double *x_im, const double *y_re,
                         const double *y_im, double *c_re, double *c_im, double *part, int sm_count, cudaStream_t stream,
                         int *launches)
{
    int k_chunk = K;
    const int split = zgemm_split(Mx, Ny, K, sm_count, &k_chunk);
    dim3 grid((Ny + kTile - 1) / kTile, (Mx + kTile - 1) / kTile, split);
    const long long n = (long long)Mx * Ny;
    const bool tensor = g_psf_dmma.load(std::memory_order_relaxed) != 0;
    if (split == 1) {
        if (tensor)
            zgemm_nt_dmma_kernel<<<grid, 256, 0, stream>>>(Mx, Ny, K, k_chunk, x_re, x_im, y_re, y_im, c_re, c_im);
        else
            zgemm_nt_kernel<<<grid, 256, 0, stream>>>(Mx, Ny, K, k_chunk, x_re, x_im, y_re, y_im, c_re, c_im);
        if (launches) (*launches)++;
        return cudaGetLastError();
    }
    if (tensor)
        zgemm_nt_dmma_kernel<<<grid, 256, 0, stream>>>(Mx, Ny, K, k_chunk, x_re, x_im, y_re, y_im, part, part + n);
    else
        zgemm_nt_kernel<<<grid, 256, 0, stream>>>(Mx, Ny, K, k_chunk, x_re, x_im, y_re, y_im, part, part + n);
    sum_partials_kernel<<<(unsigned)min((long long)sm_count * 8, (n + 255) / 256), 256, 0, stream>>>(part, split, n, c_re, c_im);
    if (launches) (*launches) += 2;
    return cudaGetLastError();
}

} // namespace

// scratch layout (doubles): [0, 2MG) DFT matrix D (re, im) ; [2MG, 4MG) Wt (re, im) ; [4MG, 4MG + 2MM) the field E when
// the caller does not take it ; then 2GG for the normalised pupil ; then the K-split partial sums of the larger product
long long psf_partials_doubles(int G, int M, int sm_count)
{
    const long long a = (long long)zgemm_split(M, G, G, sm_count, nullptr) * 2 * M * G;
    const long long b = (long long)zgemm_split(M, M, G, sm_count, nullptr) * 2 * M * M;
    return a > b ? a : b;
}

long long psf_scratch_doubles(int G, int M, int normalize)
{
    // (sized for the split a 1-SM .. 256-SM device would choose: the split count only falls as the SM count does)
    return 4LL * M * G + 2LL * M * M + (normalize ? 2LL * G * G : 0LL) + psf_partials_doubles(G, M, 256);
}

cudaError_t launch_psf(const double *grid, int G, double half_width, int M, double df, int normalize, double *scratch,
                       double *psf_out, double *field_re, double *field_im, int sm_count, cudaStream_t stream, int *launches)
{
    const long long cells = (long long)G * G, mg = (long long)M * G, mm = (long long)M * M;
    double *d_re = scratch, *d_im = scratch + mg, *w_re = scratch + 2 * mg, *w_im = scratch + 3 * mg;
    double *e_re = scratch + 4 * mg, *e_im = e_re + mm;
    const double *p_re = grid, *p_im = grid + cells;
    double *part = scratch + 4 * mg + 2 * mm + (normalize ? 2 * cells : 0);
    int n = 0;
    if (normalize) {
        double *q_re = scratch + 4 * mg + 2 * mm, *q_im = q_re + cells;
        normalize_pupil_kernel<<<sm_count * 8, 256, 0, stream>>>(grid, cells, q_re, q_im);
        p_re = q_re;
        p_im = q_im;
        n++;
    }
    const double cell = 2.0 * half_width / (double)G;
    dft_matrix_kernel<<<sm_count * 8, 256, 0, stream>>>(M, G, df, cell, half_width, d_re, d_im);
    n++;
    // Wt[k, v] = sum_u D[k, u] P[v, u]
    cudaError_t e = launch_zgemm(M, G, G, d_re, d_im, p_re, p_im, w_re, w_im, part, sm_count, stream, &n);
    if (e != cudaSuccess) return e;
    // E[l, k] = sum_v D[l, v] Wt[k, v]   (square pupil grid: the same DFT matrix serves both axes)
    if (field_re && field_im) {
        e_re = field_re;
        e_im = field_im;
    }
    e = launch_zgemm(M, M, G, d_re, d_im, w_re, w_im, e_re, e_im, part, sm_count, stream, &n);
    if (e != cudaSuccess) return e;
    if (psf_out) {
        abs2_kernel<<<min((long long)sm_count * 8, (mm + 255) / 256), 256, 0, stream>>>(e_re, e_im, mm, psf_out);
        n++;
    }
    if (launches) *launches = n;
    return cudaGetLastError();
}

} // namespace rtb
