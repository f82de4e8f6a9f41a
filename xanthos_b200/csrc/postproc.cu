// Post-processing scans on the device-resident [month][cell] fields (SURVEY.md section 8, row f3).
//
//   * drought_scan_kernel       - DroughtStats.droughtstats   (xanthos/drought/drought_stats.py:85-148), and the
//                                 ensemble runner's drought counts and member summaries in the same scan
//   * drought_thresholds_kernel - DroughtStats.getthresh      (drought_stats.py:150-171, numpy.percentile "linear")
//   * group_sum_kernel          - Aggregation_Map             (xanthos/diagnostics/time_series.py:126-138) and the
//                                 basin aggregation of AccessibleWater (xanthos/accessible/accessible.py:41-51)
//   * year_sum_scaled_kernel    - mm/month -> km3/year        (accessible.py:34-39)
//
// All of them keep the reference's operation order (the library is compiled with -fmad=false), so the results
// are bit-identical to numpy: plain IEEE subtract / divide / add, numpy's pairwise order for the 12-month sum,
// numpy's two-sided linear interpolation for the percentile, and cell-index order for the group sums.
#include "common.cuh"

namespace xan {

// ---------------------------------------------------------------------------------------------
// Severity / intensity / duration.  thread = cell, months in sequence, (S, D) of the previous month in
// registers; reads and writes are coalesced rows of the month-major fields.  HBM-bound: 8 B read (the
// K <= 12 threshold rows stay in L2 / L1) + 24 B written per cell-month.
// Quirk kept: month 0 uses threshold row 0 and intensity == severity there (drought_stats.py:121-123);
// later months use row t % K (:130).
//
// FIELDS writes S / I / D.  ACCUM is the ensemble accumulation: count[t][c] += dry (int32, the number of members in
// drought so far) and, per cell, the member summary [4][ld] = (D > 0).sum(0), (D == 1).sum(0), D.max(0), S.max(0)
// (NaN-propagating like np.max).  Without FIELDS the traffic is 8 B read + at most 4 + 4 B of count per cell-month:
// the count is added in L2 by a reduction without return value, only in dry months.  The accumulation arguments
// come last, so FIELDS-only compiles to the code of the kernel before it had them (same SASS, 60 registers).
// ---------------------------------------------------------------------------------------------
constexpr int DS_BATCH = 8;   // months loaded ahead of the scan (the scan itself is a dependent chain per cell)

template <bool FIELDS, bool ACCUM>
__global__ void __launch_bounds__(128)
    drought_scan_kernel(const double *__restrict__ hydro, const double *__restrict__ thresh, int ncell, int nmonths,
                        int ld, int ld_t, int nthresh, double *__restrict__ S, double *__restrict__ I,
                        double *__restrict__ D, int *__restrict__ count, double *__restrict__ summary) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    double s = 0.0, d = 0.0;
    int n_dry = 0, n_events = 0;
    float longest = 0.0f;           // a whole number of months: exact in float, one register fewer
    double peak = -INFINITY;        // np.max: the first severity replaces it (a -inf severity leaves it equal)
    // both groups: one month fewer in flight keeps the kernel within 64 registers (8 blocks per SM, as FIELDS alone)
    constexpr int B = FIELDS && ACCUM ? DS_BATCH - 1 : DS_BATCH;
    for (int t0 = 0; t0 < nmonths; t0 += B) {
        double h[B], th[B];
#pragma unroll
        for (int k = 0; k < B; ++k) {                      // all loads of the batch in flight together
            const int t = min(t0 + k, nmonths - 1);
            h[k] = ldg_stream(hydro + (size_t)t * ld + c);
            th[k] = thresh[(size_t)(t % nthresh) * ld_t + c];
        }
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const int t = t0 + k;
            if (t >= nmonths) break;
            const bool dry = h[k] < th[k];                          // false for NaN, like numpy
            const double deficit = (th[k] - h[k]) / th[k];          // off the chain: depends on the inputs only
            double it;
            if (t == 0) {
                d = dry ? 1.0 : 0.0;
                s = dry ? deficit : 0.0;
                it = s;
            } else {
                d = dry ? d + 1.0 : 0.0;
                s = dry ? s + deficit : 0.0;
                it = dry ? s / d : 0.0;
            }
            if constexpr (FIELDS) {
                stg_stream(S + (size_t)t * ld + c, s);
                stg_stream(I + (size_t)t * ld + c, it);
                stg_stream(D + (size_t)t * ld + c, d);
            }
            if constexpr (ACCUM) {
                if (dry) atomicAdd(count + (size_t)t * ld + c, 1);   // result unused: a RED, no register, no wait
                n_dry += dry ? 1 : 0;
                n_events += (d == 1.0) ? 1 : 0;
                longest = fmaxf(longest, (float)d);                 // d is never NaN
                if (!isnan(peak) && !(s <= peak)) peak = s;         // a NaN severity sticks, as in np.max
            }
        }
    }
    if constexpr (ACCUM) {
        summary[c] = (double)n_dry;
        summary[(size_t)ld + c] = (double)n_events;
        summary[2 * (size_t)ld + c] = (double)longest;
        summary[3 * (size_t)ld + c] = peak;
    }
}

// ---------------------------------------------------------------------------------------------
// Quantile thresholds.  thread = (cell, period): the nyear values hist[y * nper + p][cell] are sorted by
// insertion (nyear is a few dozen) and numpy's "linear" rule is applied with the
// virtual index (prev, gamma) computed on the host exactly as numpy does.  A NaN anywhere in the sample
// gives NaN (numpy sorts NaN last and then tests the last element).
// ---------------------------------------------------------------------------------------------
constexpr int MAX_YEARS = 1024;   // samples per (period, cell): 85 years of monthly data with a single period
constexpr int THR_BLOCK = 128;
constexpr int THR_SMEM_YEARS = 96;   // up to this many samples per thread the sort runs in shared memory

// SMEM = true: the samples of a thread live in shared memory as v[y * THR_BLOCK + thread] (conflict-free); a
// thread-private array in local memory costs 2 KB per thread of DRAM write-back (ncu: 447 MB for a 6.5 MB result).
template <bool SMEM>
__global__ void __launch_bounds__(THR_BLOCK)
    drought_thresholds_kernel(const double *__restrict__ hist, int ncell, int nyear, int nper, int ld, int prev,
                              double gamma, double *__restrict__ out, int ld_out) {
    extern __shared__ double s_v[];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = blockIdx.y;
    if (c >= ncell) return;
    double local_v[SMEM ? 1 : MAX_YEARS];
    double *v = SMEM ? s_v + threadIdx.x : local_v;
    const int st = SMEM ? THR_BLOCK : 1;
    bool has_nan = false;
    for (int y = 0; y < nyear; ++y) {
        const double x = hist[(size_t)(y * nper + p) * ld + c];
        has_nan = has_nan || isnan(x);
        int k = y;
        while (k > 0 && v[(k - 1) * st] > x) {
            v[k * st] = v[(k - 1) * st];
            --k;
        }
        v[k * st] = x;
    }
    double r;
    if (has_nan) {
        r = nan("");
    } else {
        const int nxt = min(prev + 1, nyear - 1);
        r = numpy_lerp(v[prev * st], v[nxt * st], gamma);
    }
    out[(size_t)p * ld_out + c] = r;
}

// ---------------------------------------------------------------------------------------------
// Group sums in cell-index order.  thread = (time step, group): walks the cells of its group in ascending
// index (`order` is the stable sort of the cells by group id) and adds the non-NaN values, exactly like
// the reference's double loop.  The 32 lanes of a warp are 32 consecutive time steps of one group and
// read the same columns of 32 different rows.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    group_sum_kernel(const double *__restrict__ src, const int *__restrict__ order, const int *__restrict__ offsets,
                     int ngroups, int ntime, int ld, double *__restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int g = blockIdx.y;
    if (t >= ntime) return;
    const double *row = src + (size_t)t * ld;
    double acc = 0.0;
    // The additions are a dependent chain in cell order (bit-exactness), so the time of the kernel is the largest group
    // times the latency per cell: GB loads are kept in flight and the indices of the next batch are fetched while the
    // values of this one arrive.
    constexpr int GB = 16;
    const int end = offsets[g + 1];
    int k = offsets[g];
    if (k >= end) {          // a group without cells
        out[(size_t)g * ntime + t] = 0.0;
        return;
    }
    int idx[GB];
#pragma unroll
    for (int j = 0; j < GB; ++j) idx[j] = order[min(k + j, end - 1)];
    for (; k + GB <= end; k += GB) {
        double x[GB];
#pragma unroll
        for (int j = 0; j < GB; ++j) x[j] = row[idx[j]];
#pragma unroll
        for (int j = 0; j < GB; ++j) idx[j] = order[min(k + GB + j, end - 1)];
#pragma unroll
        for (int j = 0; j < GB; ++j)
            if (!isnan(x[j])) acc = acc + x[j];
    }
    for (int j = 0; k + j < end; ++j) {      // tail: its indices are already in idx[]
        const double x = row[idx[j]];
        if (!isnan(x)) acc = acc + x;
    }
    out[(size_t)g * ntime + t] = acc;   // [group][time], the reference's orientation
}

// numpy.sum over 12 contiguous months (pairwise order) times a per-cell factor: [nmonths][ld] -> [nyears][ld]
__global__ void __launch_bounds__(256)
    year_sum_scaled_kernel(const double *__restrict__ src, const double *__restrict__ scale, int ncell, int nyears,
                           int ld, double *__restrict__ dst) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (c >= ncell) return;
    const double *p = src + (size_t)y * 12 * ld + c;
    const double s = numpy_pairwise_sum(12, [&](int i) { return p[(size_t)i * ld]; });
    dst[(size_t)y * ld + c] = scale ? s * scale[c] : s;
}

}  // namespace xan

using namespace xan;

extern "C" {

int xan_drought_stats(const double *d_hydro, const double *d_thresh, int ncell, int nmonths, int ld, int nthresh,
                      int ld_thresh, double *d_severity, double *d_intensity, double *d_duration, void *stream) {
    XAN_REQUIRE(d_hydro && d_thresh && d_severity && d_intensity && d_duration, "xan_drought_stats: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && nthresh > 0 && ld >= ncell && ld_thresh >= ncell,
                "xan_drought_stats: bad shape ncell=%d nmonths=%d nthresh=%d ld=%d ld_thresh=%d", ncell, nmonths,
                nthresh, ld, ld_thresh);
    drought_scan_kernel<true, false><<<ceil_div(ncell, 128), 128, 0, (cudaStream_t)stream>>>(
        d_hydro, d_thresh, ncell, nmonths, ld, ld_thresh, nthresh, d_severity, d_intensity, d_duration, nullptr,
        nullptr);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_drought_scan(const double *d_hydro, const double *d_thresh, int ncell, int nmonths, int ld, int nthresh,
                     int ld_thresh, double *d_severity, double *d_intensity, double *d_duration, int *d_count,
                     double *d_summary, void *stream) {
    const bool fields = d_severity || d_intensity || d_duration, accum = d_count || d_summary;
    XAN_REQUIRE(d_hydro && d_thresh, "xan_drought_scan: null pointer");
    XAN_REQUIRE(!fields || (d_severity && d_intensity && d_duration),
                "xan_drought_scan: severity, intensity and duration are written together");
    XAN_REQUIRE(!accum || (d_count && d_summary), "xan_drought_scan: count and summary are accumulated together");
    XAN_REQUIRE(fields || accum, "xan_drought_scan: no output requested");
    XAN_REQUIRE(ncell > 0 && nmonths > 0 && nthresh > 0 && ld >= ncell && ld_thresh >= ncell,
                "xan_drought_scan: bad shape ncell=%d nmonths=%d nthresh=%d ld=%d ld_thresh=%d", ncell, nmonths,
                nthresh, ld, ld_thresh);
    const dim3 grid(ceil_div(ncell, 128));
    cudaStream_t st = (cudaStream_t)stream;
    if (fields && accum)
        drought_scan_kernel<true, true><<<grid, 128, 0, st>>>(d_hydro, d_thresh, ncell, nmonths, ld, ld_thresh, nthresh,
                                                              d_severity, d_intensity, d_duration, d_count, d_summary);
    else if (fields)
        drought_scan_kernel<true, false><<<grid, 128, 0, st>>>(d_hydro, d_thresh, ncell, nmonths, ld, ld_thresh,
                                                               nthresh, d_severity, d_intensity, d_duration, nullptr,
                                                               nullptr);
    else
        drought_scan_kernel<false, true><<<grid, 128, 0, st>>>(d_hydro, d_thresh, ncell, nmonths, ld, ld_thresh,
                                                               nthresh, nullptr, nullptr, nullptr, d_count, d_summary);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_drought_thresholds(const double *d_hist, int ncell, int ntime, int ld, int nper, int prev_index, double gamma,
                           double *d_out, int ld_out, void *stream) {
    XAN_REQUIRE(d_hist && d_out, "xan_drought_thresholds: null pointer");
    XAN_REQUIRE(ncell > 0 && nper > 0 && ntime >= nper && ntime % nper == 0 && ld >= ncell && ld_out >= ncell,
                "xan_drought_thresholds: %d time steps are not a multiple of %d periods (ncell=%d ld=%d)", ntime, nper,
                ncell, ld);
    const int nyear = ntime / nper;
    XAN_REQUIRE(nyear <= MAX_YEARS, "xan_drought_thresholds: reference period of %d years per period (max %d)", nyear,
                MAX_YEARS);
    XAN_REQUIRE(prev_index >= 0 && prev_index < nyear && gamma >= 0.0 && gamma <= 1.0,
                "xan_drought_thresholds: bad virtual index %d + %g for %d samples", prev_index, gamma, nyear);
    dim3 grid(ceil_div(ncell, THR_BLOCK), nper);
    if (nyear <= THR_SMEM_YEARS) {
        const size_t smem = sizeof(double) * THR_BLOCK * (size_t)nyear;
        XAN_CUDA_CHECK(cudaFuncSetAttribute(drought_thresholds_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)(sizeof(double) * THR_BLOCK * THR_SMEM_YEARS)));
        drought_thresholds_kernel<true><<<grid, THR_BLOCK, smem, (cudaStream_t)stream>>>(d_hist, ncell, nyear, nper, ld,
                                                                                          prev_index, gamma, d_out, ld_out);
    } else {
        drought_thresholds_kernel<false><<<grid, THR_BLOCK, 0, (cudaStream_t)stream>>>(d_hist, ncell, nyear, nper, ld,
                                                                                        prev_index, gamma, d_out, ld_out);
    }
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_group_sum(const double *d_src, const int *d_order, const int *d_offsets, int ngroups, int ntime, int ld,
                  double *d_out, void *stream) {
    XAN_REQUIRE(d_src && d_order && d_offsets && d_out, "xan_group_sum: null pointer");
    XAN_REQUIRE(ngroups > 0 && ngroups <= 65535 && ntime > 0 && ld > 0, "xan_group_sum: bad shape ngroups=%d ntime=%d",
                ngroups, ntime);
    dim3 grid(ceil_div(ntime, 128), ngroups);
    group_sum_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_src, d_order, d_offsets, ngroups, ntime, ld, d_out);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

int xan_year_sum_scaled(const double *d_src, const double *d_scale, int ncell, int nmonths, int ld, double *d_dst,
                        void *stream) {
    XAN_REQUIRE(d_src && d_dst, "xan_year_sum_scaled: null pointer");
    XAN_REQUIRE(ncell > 0 && nmonths >= 12 && ld >= ncell, "xan_year_sum_scaled: bad shape %d x %d (ld %d)", ncell,
                nmonths, ld);
    dim3 grid(ceil_div(ncell, 256), nmonths / 12);   // int(nmonths / 12): a trailing partial year is dropped
    year_sum_scaled_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_src, d_scale, ncell, nmonths / 12, ld, d_dst);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

}  // extern "C"
