// Across-member statistics of an ensemble (mean, standard deviation, minimum, maximum per (time, cell)), accumulated
// on the device one member at a time so that no member's grid has to leave HBM for them.
//
// State per (time, cell), fp64, month-major [ntime][ld], packed as two double2 arrays for 16-byte accesses:
//   d_sm = (sum, m2)  sequential sum in member order; Welford's sum of squared deviations around the running mean sum/n
//   d_mm = (min, max) NaN-propagating, like numpy.min / numpy.max (fmin / fmax would skip NaN)
// Only + - * / sqrt are used and the library is built with -fmad=false: every kernel is bitwise equal to the numpy
// restatement of the same operation order in oracle/ensemble_stats.py.
#include "common.cuh"

namespace xan {

constexpr int ES_BLOCK = 256;

// np.minimum / np.maximum semantics: a NaN on either side wins
__device__ __forceinline__ double nan_min(double a, double x) { return (x < a || isnan(x)) ? x : a; }
__device__ __forceinline__ double nan_max(double a, double x) { return (x > a || isnan(x)) ? x : a; }

// n = members seen including this one.  n == 1 initialises (there is no previous mean: 0/0).
__global__ void __launch_bounds__(ES_BLOCK)
    ens_stats_update_kernel(const double *__restrict__ x, double2 *__restrict__ sm, double2 *__restrict__ mm,
                            int ncell, int ld, int n) {
    const int c = blockIdx.x * ES_BLOCK + threadIdx.x;
    if (c >= ncell) return;
    const size_t i = (size_t)blockIdx.y * ld + c;
    const double v = ldg_stream(x + i);
    if (n == 1) {
        sm[i] = make_double2(v, 0.0 * v);   // 0 * NaN = NaN: a NaN member makes all four NaN
        mm[i] = make_double2(v, v);
        return;
    }
    double2 a = sm[i], b = mm[i];
    const double mean_old = a.x / (double)(n - 1);
    a.x = a.x + v;
    const double mean_new = a.x / (double)n;
    a.y = a.y + (v - mean_old) * (v - mean_new);
    b.x = nan_min(b.x, v);
    b.y = nan_max(b.y, v);
    sm[i] = a;
    mm[i] = b;
}

// Chan et al.'s pairwise combination: partial a (na members) absorbs partial b (nb members), in place.
__global__ void __launch_bounds__(ES_BLOCK)
    ens_stats_merge_kernel(double2 *__restrict__ sm_a, double2 *__restrict__ mm_a, const double2 *__restrict__ sm_b,
                           const double2 *__restrict__ mm_b, int ncell, int ld, double na, double nb) {
    const int c = blockIdx.x * ES_BLOCK + threadIdx.x;
    if (c >= ncell) return;
    const size_t i = (size_t)blockIdx.y * ld + c;
    double2 a = sm_a[i], b = mm_a[i];
    const double2 p = sm_b[i], q = mm_b[i];
    const double n = na + nb;
    const double delta = p.x / nb - a.x / na;
    a.x = a.x + p.x;
    a.y = a.y + p.y + delta * delta * na * nb / n;
    b.x = nan_min(b.x, q.x);
    b.y = nan_max(b.y, q.y);
    sm_a[i] = a;
    mm_a[i] = b;
}

// mean = sum / n, std = sqrt(m2 / (n - ddof)), min, max -> cell-major [ncell][ntime] (the layout of the host arrays),
// transposed through shared-memory tiles as in to_cell_major_kernel.  Any output pointer may be NULL.
constexpr int FT = 32;
constexpr int FROWS = 8;

__global__ void __launch_bounds__(FT *FROWS)
    ens_stats_finalize_kernel(const double2 *__restrict__ sm, const double2 *__restrict__ mm, int ncell, int ntime,
                              int ld, double n, double dof, double *__restrict__ mean, double *__restrict__ std_,
                              double *__restrict__ mn, double *__restrict__ mx) {
    __shared__ double tile[4][FT][FT + 1];
    const int c0 = blockIdx.x * FT;
    const int t0 = blockIdx.y * FT;
    for (int r = threadIdx.y; r < FT; r += FROWS) {
        const int t = t0 + r, c = c0 + threadIdx.x;
        if (c < ncell && t < ntime) {
            const size_t i = (size_t)t * ld + c;
            const double2 a = sm[i], b = mm[i];
            tile[0][r][threadIdx.x] = a.x / n;
            tile[1][r][threadIdx.x] = sqrt(a.y / dof);
            tile[2][r][threadIdx.x] = b.x;
            tile[3][r][threadIdx.x] = b.y;
        }
    }
    __syncthreads();
    double *const outs[4] = {mean, std_, mn, mx};
    for (int r = threadIdx.y; r < FT; r += FROWS) {
        const int c = c0 + r, t = t0 + threadIdx.x;
        if (c < ncell && t < ntime) {
            const size_t o = (size_t)c * ntime + t;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (outs[k]) stg_stream(outs[k] + o, tile[k][threadIdx.x][r]);
        }
    }
}

}  // namespace xan

using namespace xan;

extern "C" {

int xan_ens_stats_update(const double *d_x, double *d_sm, double *d_mm, int ncell, int ntime, int ld, int n,
                         void *stream) {
    XAN_REQUIRE(d_x && d_sm && d_mm, "xan_ens_stats_update: null pointer");
    XAN_REQUIRE(ncell > 0 && ntime > 0 && ntime <= 65535 && ld >= ncell && n >= 1,
                "xan_ens_stats_update: bad shape %d x %d (ld %d) or member count %d", ncell, ntime, ld, n);
    XAN_REQUIRE(((uintptr_t)d_sm | (uintptr_t)d_mm) % 16 == 0, "xan_ens_stats_update: state not 16-byte aligned");
    dim3 grid(ceil_div(ncell, ES_BLOCK), ntime);
    ens_stats_update_kernel<<<grid, ES_BLOCK, 0, (cudaStream_t)stream>>>(d_x, (double2 *)d_sm, (double2 *)d_mm, ncell,
                                                                        ld, n);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_ens_stats_merge(double *d_sm_a, double *d_mm_a, const double *d_sm_b, const double *d_mm_b, int ncell,
                        int ntime, int ld, int na, int nb, void *stream) {
    XAN_REQUIRE(d_sm_a && d_mm_a && d_sm_b && d_mm_b, "xan_ens_stats_merge: null pointer");
    XAN_REQUIRE(ncell > 0 && ntime > 0 && ntime <= 65535 && ld >= ncell && na >= 1 && nb >= 1,
                "xan_ens_stats_merge: bad shape %d x %d (ld %d) or member counts %d, %d", ncell, ntime, ld, na, nb);
    XAN_REQUIRE(((uintptr_t)d_sm_a | (uintptr_t)d_mm_a | (uintptr_t)d_sm_b | (uintptr_t)d_mm_b) % 16 == 0,
                "xan_ens_stats_merge: state not 16-byte aligned");
    dim3 grid(ceil_div(ncell, ES_BLOCK), ntime);
    ens_stats_merge_kernel<<<grid, ES_BLOCK, 0, (cudaStream_t)stream>>>(
        (double2 *)d_sm_a, (double2 *)d_mm_a, (const double2 *)d_sm_b, (const double2 *)d_mm_b, ncell, ld, (double)na,
        (double)nb);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_ens_stats_finalize(const double *d_sm, const double *d_mm, int ncell, int ntime, int ld, int n, int ddof,
                           double *d_mean, double *d_std, double *d_min, double *d_max, void *stream) {
    XAN_REQUIRE(d_sm && d_mm, "xan_ens_stats_finalize: null pointer");
    XAN_REQUIRE(ncell > 0 && ntime > 0 && ld >= ncell && n >= 1 && ddof >= 0,
                "xan_ens_stats_finalize: bad shape %d x %d (ld %d), member count %d or ddof %d", ncell, ntime, ld, n,
                ddof);
    XAN_REQUIRE(((uintptr_t)d_sm | (uintptr_t)d_mm) % 16 == 0, "xan_ens_stats_finalize: state not 16-byte aligned");
    dim3 grid(ceil_div(ncell, FT), ceil_div(ntime, FT)), block(FT, FROWS);
    ens_stats_finalize_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
        (const double2 *)d_sm, (const double2 *)d_mm, ncell, ntime, ld, (double)n, (double)(n - ddof), d_mean, d_std,
        d_min, d_max);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

}  // extern "C"
