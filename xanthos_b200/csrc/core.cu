// Library plumbing + layout kernels (transposes at the reference boundary, yearly aggregation).
#include "common.cuh"

#include <cstring>

namespace xan {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// Stream-ordered scratch memory.  The default memory pool of a device returns its memory to the driver
// at every synchronisation (release threshold 0), so a 3 GB scratch buffer would be cudaMalloc'ed and
// freed on every call (tens of milliseconds).  The threshold is raised once per device; scratch then
// stays cached in the pool between calls.
cudaError_t scratch_alloc(void **p, size_t bytes, cudaStream_t s) {
    static thread_local int configured_dev = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (configured_dev != dev) {
        cudaMemPool_t pool;
        e = cudaDeviceGetDefaultMemPool(&pool, dev);
        if (e != cudaSuccess) return e;
        unsigned long long keep = ~0ull;
        e = cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        if (e != cudaSuccess) return e;
        configured_dev = dev;
    }
    return cudaMallocAsync(p, bytes, s);
}

// ---------------------------------------------------------------------------------------------
// Transposes.  The reference keeps every field as [ncell][nmonths] (data_load.py:288-340); the
// kernels of this library want [nmonths][ld] so that a warp reads 32 consecutive cells of one
// month.  32x32 fp64 tiles through padded shared memory: both sides coalesced, HBM-bound
// (16 B per element).
// ---------------------------------------------------------------------------------------------
constexpr int TILE = 32;
constexpr int TROWS = 8;

template <bool NAN_TO_NUM, typename SRC = double>
__global__ void __launch_bounds__(TILE *TROWS)
    to_month_major_kernel(const SRC *__restrict__ src, double *__restrict__ dst, int ncell,
                          int nmonths, int ld) {
    __shared__ double tile[TILE][TILE + 1];
    const int c0 = blockIdx.x * TILE;  // cell tile
    const int m0 = blockIdx.y * TILE;  // month tile
    // read: rows = cells, contiguous along months
    for (int r = threadIdx.y; r < TILE; r += TROWS) {
        const int c = c0 + r, m = m0 + threadIdx.x;
        if (c < ncell && m < nmonths) {
            double v = (double)ldg_stream(src + (size_t)c * nmonths + m);   // float -> double is exact
            if (NAN_TO_NUM) v = nan_to_num(v);
            tile[r][threadIdx.x] = v;
        }
    }
    __syncthreads();
    // write: rows = months, contiguous along cells
    for (int r = threadIdx.y; r < TILE; r += TROWS) {
        const int m = m0 + r, c = c0 + threadIdx.x;
        if (c < ncell && m < nmonths) dst[(size_t)m * ld + c] = tile[threadIdx.x][r];
    }
}

__global__ void __launch_bounds__(TILE *TROWS)
    to_cell_major_kernel(const double *__restrict__ src, double *__restrict__ dst, int ncell,
                         int nmonths, int ld) {
    __shared__ double tile[TILE][TILE + 1];
    const int c0 = blockIdx.x * TILE;
    const int m0 = blockIdx.y * TILE;
    for (int r = threadIdx.y; r < TILE; r += TROWS) {
        const int m = m0 + r, c = c0 + threadIdx.x;
        if (c < ncell && m < nmonths) tile[r][threadIdx.x] = ldg_stream(src + (size_t)m * ld + c);
    }
    __syncthreads();
    for (int r = threadIdx.y; r < TILE; r += TROWS) {
        const int c = c0 + r, m = m0 + threadIdx.x;
        if (c < ncell && m < nmonths) stg_stream(dst + (size_t)c * nmonths + m, tile[threadIdx.x][r]);
    }
}

// OutWriter.agg_to_year (out_writer.py:237-248): sum (mean for avgchflow) of each block of 12 months, NaN skipped.
__global__ void agg_to_year_kernel(const double *__restrict__ src, double *__restrict__ dst,
                                   int ncell, int nyears, int ld, int take_mean) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (c >= ncell || y >= nyears) return;
    // pandas' groupby sum / mean skip NaN: an all-NaN year sums to 0.0 and averages to NaN
    double v[12], acc = 0.0;
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < 12; ++k) v[k] = ldg_stream(src + (size_t)(y * 12 + k) * ld + c);
#pragma unroll
    for (int k = 0; k < 12; ++k)
        if (!isnan(v[k])) {
            acc += v[k];
            ++cnt;
        }
    if (take_mean) acc = acc / (double)cnt;   // 0 / 0 = NaN
    dst[(size_t)y * ld + c] = acc;
}

// OutWriter's mm -> km3 conversion (out_writer.py:114-115): every time row times a per-cell factor (src may be dst)
__global__ void scale_cells_kernel(const double *src, const double *__restrict__ scale, int ncell, int ld,
                                   double *dst) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const size_t i = (size_t)blockIdx.y * ld + c;
    dst[i] = src[i] * scale[c];
}

}  // namespace xan

using namespace xan;

extern "C" {

int xan_version(void) { return 100; }

const char *xan_last_error(void) { return g_err; }

int xan_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    XAN_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    XAN_CUDA_CHECK(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return XAN_OK;
}

int xan_to_month_major(const double *d_src, double *d_dst, int ncell, int nmonths, int ld,
                       int nan_to_num_flag, void *stream) {
    XAN_REQUIRE(d_src && d_dst, "xan_to_month_major: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && ld >= ncell, "xan_to_month_major: bad shape %d x %d (ld %d)",
                ncell, nmonths, ld);
    dim3 grid(ceil_div(ncell, TILE), ceil_div(nmonths, TILE)), block(TILE, TROWS);
    cudaStream_t s = (cudaStream_t)stream;
    if (nan_to_num_flag)
        to_month_major_kernel<true><<<grid, block, 0, s>>>(d_src, d_dst, ncell, nmonths, ld);
    else
        to_month_major_kernel<false><<<grid, block, 0, s>>>(d_src, d_dst, ncell, nmonths, ld);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_to_month_major_f32(const float *d_src, double *d_dst, int ncell, int nmonths, int ld, int nan_to_num_flag,
                           void *stream) {
    XAN_REQUIRE(d_src && d_dst, "xan_to_month_major_f32: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && ld >= ncell, "xan_to_month_major_f32: bad shape %d x %d (ld %d)", ncell,
                nmonths, ld);
    dim3 grid(ceil_div(ncell, TILE), ceil_div(nmonths, TILE)), block(TILE, TROWS);
    cudaStream_t s = (cudaStream_t)stream;
    if (nan_to_num_flag)
        to_month_major_kernel<true, float><<<grid, block, 0, s>>>(d_src, d_dst, ncell, nmonths, ld);
    else
        to_month_major_kernel<false, float><<<grid, block, 0, s>>>(d_src, d_dst, ncell, nmonths, ld);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_to_cell_major(const double *d_src, double *d_dst, int ncell, int nmonths, int ld, void *stream) {
    XAN_REQUIRE(d_src && d_dst, "xan_to_cell_major: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && ld >= ncell, "xan_to_cell_major: bad shape %d x %d (ld %d)",
                ncell, nmonths, ld);
    dim3 grid(ceil_div(ncell, TILE), ceil_div(nmonths, TILE)), block(TILE, TROWS);
    to_cell_major_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(d_src, d_dst, ncell, nmonths, ld);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_agg_to_year(const double *d_src, double *d_dst, int ncell, int nmonths, int ld, int take_mean,
                    void *stream) {
    XAN_REQUIRE(d_src && d_dst, "xan_agg_to_year: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && nmonths % 12 == 0 && ld >= ncell,
                "xan_agg_to_year: bad shape %d x %d (ld %d)", ncell, nmonths, ld);
    dim3 grid(ceil_div(ncell, 256), nmonths / 12);
    agg_to_year_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_src, d_dst, ncell, nmonths / 12, ld,
                                                              take_mean);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_scale_cells(const double *d_src, const double *d_scale, int ncell, int ntime, int ld, double *d_dst,
                    void *stream) {
    XAN_REQUIRE(d_src && d_scale && d_dst, "xan_scale_cells: null pointer");
    XAN_REQUIRE(ncell > 0 && ntime > 0 && ntime <= 65535 && ld >= ncell, "xan_scale_cells: bad shape %d x %d (ld %d)",
                ncell, ntime, ld);
    dim3 grid(ceil_div(ncell, 256), ntime);
    scale_cells_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_src, d_scale, ncell, ld, d_dst);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

}  // extern "C"
