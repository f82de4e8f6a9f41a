// ABCD runoff kernels (xanthos/runoff/abcd.py) and the batched calibration objective
// (xanthos/calibrate/calibrate_abcd.py).  fp64, month-major fields, compiled with -fmad=false.
//
// Structure of one run (ABCD.emulate, abcd.py:305-311):
//   1. abcd_spinup_kernel   - thread per cell, state (snowpack, SW, G) in registers for the whole
//                             spin-up; only the three "December" snapshots leave the SM.
//   2. abcd_reinit_kernel   - block per basin, deterministic nanmean over the basin's cells
//                             (set_vals, abcd.py:246-282).
//   3. abcd_sim_kernel      - thread per cell, state in registers, streams AET / Q / SW out.
#include "common.cuh"

#include <type_traits>

#include <cstring>
#include <vector>
#include <algorithm>
#include <numeric>

struct xan_abcd_plan {
    int ncell = 0;
    int n_basins = 0;
    int max_basin_cells = 0;
    std::vector<int> h_offsets;   // [n_basins + 1]
    std::vector<int> h_order;     // cells sorted by basin (stable)
    int *d_basin_idx = nullptr;   // [ncell] row of the parameter table, < 0 = not simulated
    int *d_order = nullptr;       // [n_live]
    int *d_offsets = nullptr;     // [n_basins + 1]
};

namespace xan {

constexpr double TRAIN = 2.5;   // abcd.py:103
constexpr double TSNOW = 0.6;   // abcd.py:104
constexpr double SW_INIT = 100.0, GW_INIT = 500.0;   // abcd.py:82-84

// Division by a per-cell constant d whose correctly rounded reciprocal `inv` is known:
//   q0 = n * inv;  r = fma(-q0, d, n) (exact);  q = fma(r, inv, q0)
// is the correctly rounded quotient n / d (Markstein's theorem: q0 is within one ulp, the residual is
// exact, the correction rounds once), i.e. bit-identical to the `/` of numpy - in 3 dependent
// instructions instead of the ~10 of div.rn.f64.  The division sits in the middle of the
// month-to-month recurrence that bounds this kernel (14 warps per SM; before: fp64 pipe 33 %, DRAM 27 %).
// Not covered by the theorem: divisors whose significand is all ones (`exact_ok` is then false and the
// plain division is used) and n = +-inf (does not occur; NaN propagates as in the reference).
// The formula is ill conditioned where w ~ b and a ~ 1 (y = x - sqrt(x^2 - w b / a)), so a 1-ulp
// shortcut such as n * inv alone shows up as 1e-7 in runoff; this one does not change a bit.
struct AbcdPar {
    double a2, b, b_over_a, c, d, d1, m, inv_a2, inv_b, inv_d1;
    bool exact_ok;
};
constexpr double TSPAN_C = 2.5 - 0.6;            // TRAIN - TSNOW as numpy evaluates it
constexpr double INV_TSPAN = 1.0 / TSPAN_C;

__device__ __forceinline__ bool significand_all_ones(double d) {
    return (__double_as_longlong(d) & 0x000fffffffffffffLL) == 0x000fffffffffffffLL;
}
__device__ __forceinline__ double div_const(double n, double d, double inv, bool ok) {
    if (!ok) return n / d;
    const double q0 = n * inv;
    const double r = fma(-q0, d, n);
    return fma(r, inv, q0);
}
// FAST: the caller has established that the divisor is covered (par.exact_ok): no test, and above all no copy of the
// ~30-instruction division inlined at every call site of the month step.
template <bool FAST>
__device__ __forceinline__ double div_par(double n, double d, double inv, bool ok) {
    if (FAST) {
        const double q0 = n * inv;
        const double r = fma(-q0, d, n);
        return fma(r, inv, q0);
    }
    return div_const(n, d, inv, ok);
}

__device__ __forceinline__ AbcdPar load_par(const double *__restrict__ pars, int row, bool snow) {
    AbcdPar q;
    const double a = pars[row * 5 + 0];
    q.b = pars[row * 5 + 1] * 1000;   // :48
    q.c = pars[row * 5 + 2];
    q.d = pars[row * 5 + 3];
    q.m = snow ? pars[row * 5 + 4] : 0.0;
    q.a2 = a * 2;                     // :54
    q.b_over_a = q.b / a;             // :55
    q.d1 = q.d + 1;                   // :56
    q.inv_a2 = 1.0 / q.a2;
    q.inv_b = 1.0 / q.b;
    q.inv_d1 = 1.0 / q.d1;
    q.exact_ok = !(significand_all_ones(q.a2) || significand_all_ones(q.b) || significand_all_ones(q.d1));
    return q;
}

// numpy.maximum / numpy.minimum propagate NaN (abcd.py:223-224)
__device__ __forceinline__ double np_maximum(double a, double b) {
    return (isnan(a) || isnan(b)) ? (a + b) : (a >= b ? a : b);
}
__device__ __forceinline__ double np_minimum(double a, double b) {
    return (isnan(a) || isnan(b)) ? (a + b) : (a <= b ? a : b);
}

// One month of ABCD.abcd_dist (abcd.py:171-228) for one cell.  `snowpack` must start at 0 (SN0, abcd.py:79).
// Straight-line code: the rain / snow partition (set_rain_and_snow, :140-169) and the melt (:183-192) are selects, not
// branches - as `if / else if` they were 13 % of the executed instructions (BSSY / BRA / BSYNC) of the passes.
template <bool SNOW, bool FASTDIV = false>
__device__ __forceinline__ void abcd_step(bool first, double p, double e, double t, const AbcdPar &par,
                                          double &snowpack, double &sw, double &g, double &aet_out,
                                          double &q_out) {
    double rain = p, snm = 0.0;
    if (SNOW) {
        const bool allrain = t > TRAIN;
        const bool mixed = (t <= TRAIN) && (t >= TSNOW);
        const bool allsnow = t < TSNOW;                                        // a NaN temperature is none of the three
        const double dtr = TRAIN - t;
        const double frac = div_const(dtr, TSPAN_C, INV_TSPAN, true);
        const double snow_mixed = div_const(p * dtr, TSPAN_C, INV_TSPAN, true);   // :154
        const double snow = mixed ? snow_mixed : (allsnow ? p : 0.0);
        rain = mixed ? (p - snow_mixed) : (allrain ? p : 0.0);                 // :156-166
        snowpack = snowpack + snow;                                            // :178-181 (SN0 = 0)
        const double sm = snowpack * par.m;
        snm = allrain ? sm : (mixed ? sm * frac : 0.0);                        // :189-192
        snowpack = snowpack - snm;                                             // :195
    }
    const double w = (rain + sw) + (first ? 0.0 : snm);                        // :198-201 (x + 0.0 == x here)
    const double x = div_par<FASTDIV>(w + par.b, par.a2, par.inv_a2, par.exact_ok);  // :204-205
    const double y = x - sqrt(x * x - (w * par.b_over_a));                    // :206
    const double swt = y * exp(div_par<FASTDIV>(-e, par.b, par.inv_b, par.exact_ok));   // :209
    const double awet = w - y;                                                // :212
    const double c_awet = par.c * awet;                                       // :213
    g = div_par<FASTDIV>(g + c_awet, par.d1, par.inv_d1, par.exact_ok);       // :216-219
    double aet = y - swt;                                                     // :222
    aet = np_maximum(0.0, aet);                                               // :223
    aet = np_minimum(e, aet);                                                 // :224
    sw = y - aet;                                                             // :225
    q_out = (awet - c_awet) + par.d * g;                                      // :226
    aet_out = aet;
}

// Forcing of one cell, months 0 .. n-1, through `body(month, p, e, t)`.
// Every thread owns a column of a small ring in shared memory: ABCD_STAGES stages of ABCD_SM months x 3 fields,
// filled with 8-byte cp.async (a warp's 32 copies are one 256-byte segment of a month row) ABCD_STAGES - 1 stages
// ahead of the stage being stepped through.  The data never pass through registers before they are needed, so the
// month loop is ROLLED: the month step exists once per stage position instead of once per prefetched month - with the
// register double buffer of 2 x 6 months the kernel was 63 KB of code and stalled on instruction fetch for a quarter of
// its issue slots (ncu: no_instruction 0.95 per issued instruction).  No block-level synchronisation: a thread reads
// only what it copied itself.
constexpr int ABCD_SM = 4;        // months per stage
constexpr int ABCD_STAGES = 4;    // stages in the ring: 3 x 4 months x 3 fields x 8 B = 288 B in flight per thread
constexpr int ABCD_BLOCK = 128;

template <bool SNOW>
__device__ __forceinline__ void abcd_stage_load(double *ring, const double *__restrict__ pet,
                                                const double *__restrict__ precip, const double *__restrict__ tmin,
                                                int c, int ld, int stage, int i0, int n) {
#pragma unroll
    for (int u = 0; u < ABCD_SM; ++u) {
        if (i0 + u < n) {                                  // uniform over the block
            const size_t off = (size_t)(i0 + u) * ld + c;
            double *dst = ring + ((size_t)(stage * ABCD_SM + u) * 3) * ABCD_BLOCK + threadIdx.x;
            const unsigned d0 = (unsigned)__cvta_generic_to_shared(dst);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d0), "l"(precip + off) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d0 + ABCD_BLOCK * 8), "l"(pet + off) : "memory");
            if (SNOW)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d0 + 2 * ABCD_BLOCK * 8), "l"(tmin + off)
                             : "memory");
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

template <bool SNOW, typename Body>
__device__ __forceinline__ void abcd_stream(const double *__restrict__ pet, const double *__restrict__ precip,
                                            const double *__restrict__ tmin, int c, int ld, int n, Body body,
                                            int begin = 0) {
    extern __shared__ double abcd_ring[];   // [ABCD_STAGES][ABCD_SM][3][ABCD_BLOCK]
#pragma unroll
    for (int st = 0; st < ABCD_STAGES - 1; ++st)
        abcd_stage_load<SNOW>(abcd_ring, pet, precip, tmin, c, ld, st, begin + st * ABCD_SM, n);
    int stage = 0;
#pragma unroll 1
    for (int i = begin; i < n; i += ABCD_SM) {
        // the stage ABCD_STAGES - 1 ahead goes into the slot that was consumed in the previous iteration
        abcd_stage_load<SNOW>(abcd_ring, pet, precip, tmin, c, ld, (stage + ABCD_STAGES - 1) % ABCD_STAGES,
                              i + (ABCD_STAGES - 1) * ABCD_SM, n);
        asm volatile("cp.async.wait_group %0;" ::"n"(ABCD_STAGES - 1) : "memory");   // this stage has landed
        const double *col = abcd_ring + ((size_t)stage * ABCD_SM * 3) * ABCD_BLOCK + threadIdx.x;
#pragma unroll
        for (int u = 0; u < ABCD_SM; ++u) {
            if (i + u < n) {
                const double p = col[(u * 3 + 0) * ABCD_BLOCK], e = col[(u * 3 + 1) * ABCD_BLOCK];
                const double t = SNOW ? col[(u * 3 + 2) * ABCD_BLOCK] : 0.0;
                body(i + u, p, e, t);
            }
        }
        stage = (stage + 1) % ABCD_STAGES;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
constexpr size_t ABCD_RING_BYTES = sizeof(double) * ABCD_STAGES * ABCD_SM * 3 * ABCD_BLOCK;   // 48 KB per block

// Sets of parameter tables over one forcing (xan_abcd_run_sets): a thread steps K sets through every month it reads from
// the ring, so each forcing value is read once per K sets, and the K recurrences are independent (instruction-level
// parallelism in the latency-bound month chain).  blockIdx.y = group of K sets; the last group of a call may be short
// (nk < K): its spare slots repeat the group's last set and write nothing.  xan_abcd_run is the K = 1 instance.
// K = 2 (B200, tools/parameter_ensemble_bench.py, DESIGN.md section 6): 0.334 ms per set at 8 sets per call against
// 0.405 with K = 1 and 0.525 for single-set calls; K = 4 spills under the 128-register budget of 4 blocks per SM.
constexpr int ABCD_SETS_PER_THREAD = 2;
static_assert(XAN_ABCD_MAX_SETS % ABCD_SETS_PER_THREAD == 0, "whole groups at the largest call");

struct AbcdSetOut {   // device output pointers of every set, passed by value in the kernel parameters
    double *aet[XAN_ABCD_MAX_SETS], *q[XAN_ABCD_MAX_SETS], *sav[XAN_ABCD_MAX_SETS];
};

// Parameters of the K sets of this thread; true when every divisor of every set is covered by the fast division.
// A thread whose sets are not all covered takes the generic template, in which div_const decides per set: both give
// the same bits, so a set's result does not depend on the sets it is grouped with.
template <int K>
__device__ __forceinline__ bool load_pars(const double *__restrict__ pars, int n_rows, int s0, int nk, int row,
                                          bool snow, AbcdPar (&par)[K]) {
    bool ok = true;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        par[j] = load_par(pars + (size_t)(s0 + min(j, nk - 1)) * n_rows * 5, row, snow);
        ok = ok && par[j].exact_ok;
    }
    return ok;
}

// 4 blocks of 128 threads per SM (<= 128 registers): 67,420 cells are 527 blocks = 3.6 per SM, one wave
template <bool SNOW, int K>
__global__ void __launch_bounds__(128, 4)
    abcd_spinup_kernel(const double *__restrict__ pet, const double *__restrict__ precip,
                       const double *__restrict__ tmin, const int *__restrict__ basin_idx,
                       const double *__restrict__ pars, int n_rows, int n_sets, int ncell, int spinup, int ld,
                       double *__restrict__ snap /* [n_sets][6][ncell]: SW x3, G x3 */) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const int row = basin_idx[c];
    if (row < 0) return;
    const int s0 = blockIdx.y * K, nk = min(K, n_sets - s0);
    AbcdPar par[K];
    const bool fast_all = load_pars<K>(pars, n_rows, s0, nk, row, SNOW, par);
    double snowpack[K], sw[K], g[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        snowpack[j] = 0.0;
        sw[j] = SW_INIT;
        g[j] = GW_INIT;
    }
    const int s1 = spinup - 25, s2 = spinup - 13, s3 = spinup - 1;   // Decembers -25, -13, -1 (:255)
    // three segments ending at the three Decembers whose state is kept: no per-month test for the snapshot months
    auto run = [&](auto fast) {
        int begin = 0;
#pragma unroll 1
        for (int seg = 0; seg < 3; ++seg) {
            const int last = seg == 0 ? s1 : (seg == 1 ? s2 : s3);
            abcd_stream<SNOW>(pet, precip, tmin, c, ld, last + 1, [&](int k, double p, double e, double t) {
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    double aet, q;
                    abcd_step<SNOW, decltype(fast)::value>(k == 0, p, e, t, par[j], snowpack[j], sw[j], g[j], aet, q);
                }
            }, begin);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (j < nk) {
                    double *sn = snap + (size_t)(s0 + j) * 6 * ncell;
                    sn[(2 - seg) * (size_t)ncell + c] = sw[j];
                    sn[(5 - seg) * (size_t)ncell + c] = g[j];
                }
            }
            begin = last + 1;
        }
    };
    if (fast_all) run(std::true_type{});      // practically always: no divisor with an all-ones significand
    else run(std::false_type{});
}

// Deterministic block reduction of (sum, count) pairs; result valid in thread 0.
template <int NT>
__device__ __forceinline__ void block_reduce2(double &s, double &n, double *scratch /* [2 * NT/32] */) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        n += __shfl_down_sync(0xffffffffu, n, o);
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) {
        scratch[2 * w] = s;
        scratch[2 * w + 1] = n;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ts = 0.0, tn = 0.0;
        for (int k = 0; k < NT / 32; ++k) {
            ts += scratch[2 * k];
            tn += scratch[2 * k + 1];
        }
        s = ts;
        n = tn;
    }
}

// set_vals (abcd.py:246-282): per basin, mean over the 3 Decembers of nanmean over cells.  blockIdx.y = parameter set.
__global__ void __launch_bounds__(256)
    abcd_reinit_kernel(const double *__restrict__ snap /* [n_sets][6][ncell] */, const int *__restrict__ order,
                       const int *__restrict__ offsets, int ncell, double *__restrict__ init /* [n_sets][nb][2] */) {
    __shared__ double scratch[16];
    const int b = blockIdx.x;
    snap += (size_t)blockIdx.y * 6 * ncell;
    init += (size_t)blockIdx.y * 2 * gridDim.x;
    const int beg = offsets[b], end = offsets[b + 1];
    double mean3[2];
    for (int v = 0; v < 2; ++v) {
        double acc = 0.0;   // only meaningful in thread 0
        for (int k = 0; k < 3; ++k) {
            double s = 0.0, n = 0.0;
            const double *src = snap + (size_t)(v * 3 + k) * ncell;
            for (int j = beg + threadIdx.x; j < end; j += blockDim.x) {
                const double x = src[order[j]];
                if (!isnan(x)) {
                    s += x;
                    n += 1.0;
                }
            }
            block_reduce2<256>(s, n, scratch);
            acc = acc + s / n;   // nanmean; 0/0 -> NaN like numpy
        }
        mean3[v] = acc / 3.0;
    }
    if (threadIdx.x == 0) {
        init[2 * b] = mean3[0];
        init[2 * b + 1] = mean3[1];
    }
}

template <bool SNOW, int K>
__global__ void __launch_bounds__(128, 4)
    abcd_sim_kernel(const double *__restrict__ pet, const double *__restrict__ precip,
                    const double *__restrict__ tmin, const int *__restrict__ basin_idx,
                    const double *__restrict__ pars, int n_rows, int n_sets,
                    const double *__restrict__ init /* [n_sets][nb][2] */, int n_basins, int ncell, int nmonths,
                    int ld, const AbcdSetOut out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const int s0 = blockIdx.y * K, nk = min(K, n_sets - s0);
    double *aet_o[K], *q_o[K], *sav_o[K];     // NULL: not requested, or a spare slot of a short group
#pragma unroll
    for (int j = 0; j < K; ++j) {
        aet_o[j] = j < nk ? out.aet[s0 + j] : nullptr;
        q_o[j] = j < nk ? out.q[s0 + j] : nullptr;
        sav_o[j] = j < nk ? out.sav[s0 + j] : nullptr;
    }
    const int row = basin_idx[c];
    if (row < 0) {
        // not simulated: the reference leaves these rows uninitialised (abcd.py:384-389)
        const double nanv = __longlong_as_double(0x7ff8000000000000LL);
        for (int i = 0; i < nmonths; ++i) {
            const size_t off = (size_t)i * ld + c;
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (aet_o[j]) aet_o[j][off] = nanv;
                if (q_o[j]) q_o[j][off] = nanv;
                if (sav_o[j]) sav_o[j][off] = nanv;
            }
        }
        return;
    }
    AbcdPar par[K];
    const bool fast_all = load_pars<K>(pars, n_rows, s0, nk, row, SNOW, par);
    double snowpack[K], sw[K], g[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const double *in = init + ((size_t)(s0 + min(j, nk - 1)) * n_basins + row) * 2;
        snowpack[j] = 0.0;
        sw[j] = in[0];
        g[j] = in[1];
    }
    auto run = [&](auto fast) {
        abcd_stream<SNOW>(pet, precip, tmin, c, ld, nmonths, [&](int k, double p, double e, double t) {
            const size_t off = (size_t)k * ld + c;
#pragma unroll
            for (int j = 0; j < K; ++j) {
                double aet, q;
                abcd_step<SNOW, decltype(fast)::value>(k == 0, p, e, t, par[j], snowpack[j], sw[j], g[j], aet, q);
                if (aet_o[j]) stg_stream(aet_o[j] + off, aet);
                if (q_o[j]) stg_stream(q_o[j] + off, q);
                if (sav_o[j]) stg_stream(sav_o[j] + off, sw[j]);
            }
        });
    };
    if (fast_all) run(std::true_type{});
    else run(std::false_type{});
}

// ---------------------------------------------------------------------------------------------
// Calibration objective, batched over parameter sets (calibrate_abcd.py:134-162, 176-213).
// block = (parameter set p, basin slot i).  Every thread owns the cells j = tid, tid + NT, ... of
// the basin; their (snowpack, SW, G) live in shared memory; months are the outer loop, so the
// forcing of the basin is streamed once per block and re-used from L2 by the other parameter
// sets of the same basin (blockIdx.x = p is the fastest index).
// ---------------------------------------------------------------------------------------------
constexpr int KGE_NT = 128;

template <bool SNOW>
__global__ void __launch_bounds__(KGE_NT)
    abcd_kge_kernel(const double *__restrict__ pet, const double *__restrict__ precip,
                    const double *__restrict__ tmin, const double *__restrict__ area,
                    const int *__restrict__ order, const int *__restrict__ offsets,
                    const int *__restrict__ slot_basin /* [nb] plan row, sorted by size desc */,
                    const int *__restrict__ slot_out /* [nb] caller slot */, const double *__restrict__ pars,
                    const double *__restrict__ obs, int npar, int nmonths, int spinup, int ld, int unit_km3,
                    double *__restrict__ ed_out, double *__restrict__ series_out) {
    extern __shared__ double smem[];
    const int p = blockIdx.x;
    const int b = slot_basin[blockIdx.y];
    const int slot = slot_out[blockIdx.y];
    const int beg = offsets[b], nb = offsets[b + 1] - beg;
    constexpr int NW = KGE_NT / 32;
    double *st_sw = smem;                 // [nb]
    double *st_g = st_sw + nb;            // [nb]
    double *st_sn = st_g + nb;            // [nb]
    double *part = st_sn + nb;            // [NW][nmonths] per-warp partial basin sums
    double *scratch = part + (size_t)NW * nmonths;   // [16]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const AbcdPar par = load_par(pars, slot * npar + p, SNOW);

    // ---- spin-up ------------------------------------------------------------------------------
    for (int j = threadIdx.x; j < nb; j += KGE_NT) {
        st_sw[j] = SW_INIT;
        st_g[j] = GW_INIT;
        st_sn[j] = 0.0;
    }
    const int s1 = spinup - 25, s2 = spinup - 13, s3 = spinup - 1;
    double dsum[6] = {0, 0, 0, 0, 0, 0}, dcnt[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < spinup; ++i) {
        const size_t off = (size_t)i * ld;
        const int which = (i == s3) ? 0 : (i == s2) ? 1 : (i == s1) ? 2 : -1;
        for (int j = threadIdx.x; j < nb; j += KGE_NT) {
            const int c = order[beg + j];
            double sn = st_sn[j], sw = st_sw[j], g = st_g[j], aet, q;
            abcd_step<SNOW>(i == 0, __ldg(precip + off + c), __ldg(pet + off + c),
                            SNOW ? __ldg(tmin + off + c) : 0.0, par, sn, sw, g, aet, q);
            st_sn[j] = sn;
            st_sw[j] = sw;
            st_g[j] = g;
            if (which >= 0) {
                if (!isnan(sw)) { dsum[which] += sw; dcnt[which] += 1.0; }
                if (!isnan(g)) { dsum[3 + which] += g; dcnt[3 + which] += 1.0; }
            }
        }
    }
    // ---- basin re-initialisation (set_vals with all cells in one basin, :143) --------------------
    __shared__ double init_sw, init_g;
    {
        double m_sw = 0.0, m_g = 0.0;
        for (int k = 0; k < 3; ++k) {
            double s = dsum[k], n = dcnt[k];
            block_reduce2<KGE_NT>(s, n, scratch);
            m_sw = m_sw + s / n;
            s = dsum[3 + k];
            n = dcnt[3 + k];
            block_reduce2<KGE_NT>(s, n, scratch);
            m_g = m_g + s / n;
        }
        if (threadIdx.x == 0) {
            init_sw = m_sw / 3.0;
            init_g = m_g / 3.0;
        }
        __syncthreads();
    }
    for (int j = threadIdx.x; j < nb; j += KGE_NT) {
        st_sw[j] = init_sw;
        st_g[j] = init_g;
        st_sn[j] = 0.0;
    }
    // ---- simulation + basin aggregation (nansum over cells, :159 / :162) -------------------------
    for (int i = 0; i < nmonths; ++i) {
        const size_t off = (size_t)i * ld;
        double acc = 0.0;
        for (int j = threadIdx.x; j < nb; j += KGE_NT) {
            const int c = order[beg + j];
            double sn = st_sn[j], sw = st_sw[j], g = st_g[j], aet, q;
            abcd_step<SNOW>(i == 0, __ldg(precip + off + c), __ldg(pet + off + c),
                            SNOW ? __ldg(tmin + off + c) : 0.0, par, sn, sw, g, aet, q);
            st_sn[j] = sn;
            st_sw[j] = sw;
            st_g[j] = g;
            const double v = unit_km3 ? (q * __ldg(area + c) * 1e-6) : q;
            if (!isnan(v)) acc += v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
        if (lane == 0) part[(size_t)warp * nmonths + i] = acc;
    }
    __syncthreads();
    // ---- KGE distance (:197-211) --------------------------------------------------------------
    const double *ob = obs + (size_t)slot * nmonths;
    double sm = 0.0, so = 0.0;
    for (int i = threadIdx.x; i < nmonths; i += KGE_NT) {
        double m = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) m += part[(size_t)w * nmonths + i];
        part[i] = m;   // warp 0's row now holds the basin series
        if (series_out) series_out[((size_t)slot * npar + p) * nmonths + i] = m;
        sm += m;
        so += ob[i];
    }
    block_reduce2<KGE_NT>(sm, so, scratch);
    __shared__ double mean_m, mean_o;
    if (threadIdx.x == 0) {
        mean_m = sm / nmonths;
        mean_o = so / nmonths;
    }
    __syncthreads();
    double vm = 0.0, vo = 0.0, cov = 0.0;
    for (int i = threadIdx.x; i < nmonths; i += KGE_NT) {
        const double dm = part[i] - mean_m, dob = ob[i] - mean_o;
        vm += dm * dm;
        vo += dob * dob;
        cov += dm * dob;
    }
    double dummy = 0.0;
    block_reduce2<KGE_NT>(vm, vo, scratch);
    block_reduce2<KGE_NT>(cov, dummy, scratch);
    if (threadIdx.x == 0) {
        const double sd_m = sqrt(vm / nmonths), sd_o = sqrt(vo / nmonths);
        const double relvar = sd_m / sd_o;
        const double bias = mean_m / mean_o;
        double r = cov / sqrt(vm * vo);
        // np.corrcoef clips to [-1, 1] with np.clip, which keeps NaN (a constant series): fmax(NaN, -1) would give -1
        r = r < -1.0 ? -1.0 : (r > 1.0 ? 1.0 : r);
        ed_out[(size_t)slot * npar + p] =
            sqrt(((r - 1) * (r - 1)) + ((relvar - 1) * (relvar - 1)) + ((bias - 1) * (bias - 1)));
    }
}

// ---------------------------------------------------------------------------------------------
// Calibration objective, population layout (used when a generation has >= 16 candidates).
// lane = candidate parameter set, warp = a chunk of KC cells of one basin.  The 32 candidates of a
// warp read the SAME forcing (one broadcast load serves 32 evaluations), every lane keeps the state of
// its KC cells in registers for the whole pass (KC independent recurrences per thread = ILP).  Per chunk
// and candidate the spin-up pass leaves 12 partial (sum, count) values for the basin re-initialisation;
// the simulation pass adds the monthly partial basin sums of the KQ chunks of a block in shared memory (one
// barrier per month) and leaves one value per block, month and candidate; two small kernels add the blocks
// of a basin in index order (deterministic) and finish the KGE.
//   kge_pop_pass<.., false> -> kge_pop_reinit_kernel -> kge_pop_pass<.., true> -> kge_pop_series_kernel -> kge_pop_finish_kernel
// ---------------------------------------------------------------------------------------------
constexpr int KC = 4;   // cells per warp-chunk
constexpr int KQ = 4;   // chunks (warps) per block

struct KgeChunk {
    int slot;    // caller's basin slot
    int beg;     // first index into `order`
    int n;       // cells in this chunk (1..KC)
};

template <bool SNOW, bool SIM>
__global__ void __launch_bounds__(128)
    kge_pop_pass_kernel(const double *__restrict__ pet, const double *__restrict__ precip,
                        const double *__restrict__ tmin, const double *__restrict__ area,
                        const int *__restrict__ order, const KgeChunk *__restrict__ chunks, int nchunks,
                        const double *__restrict__ pars, const double *__restrict__ init /* [nb][npar][2], SIM */,
                        int npar, int npad, int nsteps, int ld, int unit_km3,
                        double *__restrict__ out /* SIM: [nchunks / KQ][nsteps][npad]; else [nchunks][12][npad] */) {
    // block = 4 consecutive chunks of ONE basin (the host pads every basin to a multiple of 4 chunks; a padding chunk
    // has n == 0) for one group of 32 candidates: the four partial basin sums of a month are added in chunk order in
    // shared memory, so only one value per (4 chunks, month, candidate) goes to global memory.
    __shared__ double s_acc[2][KQ][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ngroups = npad >> 5;
    const int quad = blockIdx.x / ngroups, grp = blockIdx.x - quad * ngroups;
    const int ch = quad * KQ + warp;
    const KgeChunk c = chunks[ch];
    const int p = grp * 32 + lane;
    const int pp = min(p, npar - 1);                       // padding lanes repeat the last candidate
    const AbcdPar par = load_par(pars, c.slot * npar + pp, SNOW);
    int cell[KC];
    double sn[KC], sw[KC], g[KC];
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        cell[k] = order[c.beg + max(min(k, c.n - 1), 0)];  // short / padding chunks repeat a cell (masked below)
        sn[k] = 0.0;
        sw[k] = SIM ? init[((size_t)c.slot * npar + pp) * 2] : SW_INIT;
        g[k] = SIM ? init[((size_t)c.slot * npar + pp) * 2 + 1] : GW_INIT;
    }
    const int s1 = nsteps - 25, s2 = nsteps - 13, s3 = nsteps - 1;   // Decembers -25, -13, -1 (abcd.py:255)
    double *o = SIM ? out + (size_t)quad * nsteps * npad + p : out + (size_t)ch * 12 * npad + p;
    // block-uniform choice of the division: the fast form needs every divisor of every candidate of the block covered
    const bool fast_all = __syncthreads_and(par.exact_ok ? 1 : 0) != 0;
    auto months = [&](auto fastc) {
    for (int i = 0; i < nsteps; ++i) {
        const size_t off = (size_t)i * ld;
        double e[KC], pr[KC], t[KC];
#pragma unroll
        for (int k = 0; k < KC; ++k) {                     // warp-uniform addresses: one broadcast per load
            pr[k] = __ldg(precip + off + cell[k]);
            e[k] = __ldg(pet + off + cell[k]);
            t[k] = SNOW ? __ldg(tmin + off + cell[k]) : 0.0;
        }
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            double aet, q;
            abcd_step<SNOW, decltype(fastc)::value>(i == 0, pr[k], e[k], t[k], par, sn[k], sw[k], g[k], aet, q);
            if (SIM) {
                const double v = unit_km3 ? (q * __ldg(area + cell[k]) * 1e-6) : q;   // rsim * area * 1e-6 (:159)
                if (k < c.n && !isnan(v)) acc += v;
            }
        }
        if (SIM) {
            s_acc[i & 1][warp][lane] = acc;
            __syncthreads();       // one barrier per month: the two buffers alternate
            if (warp == 0)
                o[(size_t)i * npad] = ((s_acc[i & 1][0][lane] + s_acc[i & 1][1][lane]) + s_acc[i & 1][2][lane]) +
                                      s_acc[i & 1][3][lane];
        } else if (i == s1 || i == s2 || i == s3) {
            const int which = (i == s3) ? 0 : (i == s2) ? 1 : 2;
            double ssw = 0.0, nsw = 0.0, sg = 0.0, ng = 0.0;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                if (k < c.n) {
                    if (!isnan(sw[k])) { ssw += sw[k]; nsw += 1.0; }
                    if (!isnan(g[k])) { sg += g[k]; ng += 1.0; }
                }
            }
            o[(size_t)(which) * npad] = ssw;
            o[(size_t)(3 + which) * npad] = nsw;
            o[(size_t)(6 + which) * npad] = sg;
            o[(size_t)(9 + which) * npad] = ng;
        }
    }
    };
    if (fast_all) months(std::true_type{});
    else months(std::false_type{});
}

// set_vals with every cell of the basin in one group (calibrate_abcd.py:143): mean over the three Decembers
// of the nanmean over cells.  thread = (slot, candidate); chunks of the slot are added in index order.
__global__ void __launch_bounds__(256)
    kge_pop_reinit_kernel(const double *__restrict__ snap /* [nchunks][12][npad] */, const int *__restrict__ slot_chunk0,
                          int npar, int npad, double *__restrict__ init /* [nb][npar][2] */) {
    extern __shared__ double s_acc[];   // [12][npad]
    const int slot = blockIdx.x;
    const int c0 = slot_chunk0[slot], c1 = slot_chunk0[slot + 1];
    const int total = 12 * npad;
    // thread = (snapshot value j, candidate p): the chunks are added in index order, 8 loads in flight
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
        double acc = 0.0;
        int c = c0;
        for (; c + 8 <= c1; c += 8) {
            double x[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) x[k] = snap[(size_t)(c + k) * total + idx];
#pragma unroll
            for (int k = 0; k < 8; ++k) acc += x[k];
        }
        for (; c < c1; ++c) acc += snap[(size_t)c * total + idx];
        s_acc[idx] = acc;
    }
    __syncthreads();
    for (int p = threadIdx.x; p < npar; p += blockDim.x) {
        double m_sw = 0.0, m_g = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            m_sw = m_sw + s_acc[k * npad + p] / s_acc[(3 + k) * npad + p];       // nanmean; 0/0 -> NaN like numpy
            m_g = m_g + s_acc[(6 + k) * npad + p] / s_acc[(9 + k) * npad + p];
        }
        init[((size_t)slot * npar + p) * 2] = m_sw / 3.0;
        init[((size_t)slot * npar + p) * 2 + 1] = m_g / 3.0;
    }
}

// series[slot][m][p] = sum over the 4-chunk blocks of the slot (index order) of part[block][m][p]
__global__ void __launch_bounds__(256)
    kge_pop_series_kernel(const double *__restrict__ part, const int *__restrict__ slot_chunk0, int nmonths, int npad,
                          double *__restrict__ series /* [nb][nmonths][npad] */) {
    const int slot = blockIdx.x;
    const int c0 = slot_chunk0[slot] / KQ, c1 = slot_chunk0[slot + 1] / KQ;
    const int total = nmonths * npad;
    for (int idx = blockIdx.y * blockDim.x + threadIdx.x; idx < total; idx += gridDim.y * blockDim.x) {
        double a = 0.0;
        for (int c = c0; c < c1; ++c) a += part[(size_t)c * total + idx];
        series[(size_t)slot * total + idx] = a;
    }
}

// KGE distance (calibrate_abcd.py:197-211); thread = (slot, candidate), sequential over months.
__global__ void __launch_bounds__(64)
    kge_pop_finish_kernel(const double *__restrict__ series /* [nb][nmonths][npad] */, const double *__restrict__ obs,
                          int npar, int npad, int nmonths, double *__restrict__ ed_out, double *__restrict__ series_out) {
    const int slot = blockIdx.x;
    const double *ob = obs + (size_t)slot * nmonths;
    for (int p = threadIdx.x; p < npar; p += blockDim.x) {
        const double *sr = series + (size_t)slot * nmonths * npad + p;
        double sm = 0.0, so = 0.0;
        for (int i = 0; i < nmonths; ++i) {
            const double m = sr[(size_t)i * npad];
            if (series_out) series_out[((size_t)slot * npar + p) * nmonths + i] = m;
            sm += m;
            so += ob[i];
        }
        const double mean_m = sm / nmonths, mean_o = so / nmonths;
        double vm = 0.0, vo = 0.0, cov = 0.0;
        for (int i = 0; i < nmonths; ++i) {
            const double dm = sr[(size_t)i * npad] - mean_m, dob = ob[i] - mean_o;
            vm += dm * dm;
            vo += dob * dob;
            cov += dm * dob;
        }
        const double sd_m = sqrt(vm / nmonths), sd_o = sqrt(vo / nmonths);
        const double relvar = sd_m / sd_o;
        const double bias = mean_m / mean_o;
        double r = cov / sqrt(vm * vo);
        r = r < -1.0 ? -1.0 : (r > 1.0 ? 1.0 : r);   // np.clip keeps NaN, as in abcd_kge_kernel
        ed_out[(size_t)slot * npar + p] =
            sqrt(((r - 1) * (r - 1)) + ((relvar - 1) * (relvar - 1)) + ((bias - 1) * (bias - 1)));
    }
}

// out[m][b] = nansum over the cells of basin b of src[m][c] * w[c]; one warp per (basin, month).
__global__ void __launch_bounds__(256)
    basin_sum_kernel(const double *__restrict__ src, const double *__restrict__ w, const int *__restrict__ order,
                     const int *__restrict__ offsets, int n_basins, int nmonths, int ld,
                     double *__restrict__ out) {
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m = blockIdx.y * (blockDim.x >> 5) + warp;
    if (m >= nmonths) return;
    const int beg = offsets[b], end = offsets[b + 1];
    double acc = 0.0;
    for (int j = beg + lane; j < end; j += 32) {
        const int c = order[j];
        double v = src[(size_t)m * ld + c];
        if (w) v = v * w[c];
        if (!isnan(v)) acc += v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if (lane == 0) out[(size_t)m * n_basins + b] = acc;
}

}  // namespace xan

using namespace xan;

// The three launches of n_sets tables, K sets per thread of the two passes.
template <int K>
static int abcd_launch(const xan_abcd_plan *pl, int n_sets, int n_rows, const double *d_pet, const double *d_precip,
                       const double *d_tmin, const double *d_pars, int nmonths, int spinup, int ld,
                       const AbcdSetOut &out, cudaStream_t s) {
    const int ncell = pl->ncell;
    double *snap = nullptr, *init = nullptr;
    XAN_CUDA_CHECK(scratch_alloc(&snap, sizeof(double) * 6 * (size_t)ncell * n_sets, s));
    XAN_CUDA_CHECK(scratch_alloc(&init, sizeof(double) * 2 * (size_t)pl->n_basins * n_sets, s));
    const dim3 grid(ceil_div(ncell, ABCD_BLOCK), ceil_div(n_sets, K));
    {   // 4 blocks x 48 KB of ring per SM: ask for the large shared-memory carve-out (otherwise the 527 blocks of the
        // 0.5 degree grid do not fit in one wave)
        static bool once = false;
        if (!once) {
            once = true;
            cudaFuncSetAttribute(abcd_spinup_kernel<true, K>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            cudaFuncSetAttribute(abcd_spinup_kernel<false, K>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            cudaFuncSetAttribute(abcd_sim_kernel<true, K>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            cudaFuncSetAttribute(abcd_sim_kernel<false, K>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        }
    }
    if (d_tmin)
        abcd_spinup_kernel<true, K><<<grid, ABCD_BLOCK, ABCD_RING_BYTES, s>>>(d_pet, d_precip, d_tmin, pl->d_basin_idx,
                                                                              d_pars, n_rows, n_sets, ncell, spinup, ld,
                                                                              snap);
    else
        abcd_spinup_kernel<false, K><<<grid, ABCD_BLOCK, ABCD_RING_BYTES, s>>>(d_pet, d_precip, d_tmin, pl->d_basin_idx,
                                                                               d_pars, n_rows, n_sets, ncell, spinup, ld,
                                                                               snap);
    abcd_reinit_kernel<<<dim3(pl->n_basins, n_sets), 256, 0, s>>>(snap, pl->d_order, pl->d_offsets, ncell, init);
    if (d_tmin)
        abcd_sim_kernel<true, K><<<grid, ABCD_BLOCK, ABCD_RING_BYTES, s>>>(d_pet, d_precip, d_tmin, pl->d_basin_idx,
                                                                           d_pars, n_rows, n_sets, init, pl->n_basins,
                                                                           ncell, nmonths, ld, out);
    else
        abcd_sim_kernel<false, K><<<grid, ABCD_BLOCK, ABCD_RING_BYTES, s>>>(d_pet, d_precip, d_tmin, pl->d_basin_idx,
                                                                            d_pars, n_rows, n_sets, init, pl->n_basins,
                                                                            ncell, nmonths, ld, out);
    XAN_CUDA_CHECK(cudaGetLastError());
    XAN_CUDA_CHECK(cudaFreeAsync(snap, s));
    XAN_CUDA_CHECK(cudaFreeAsync(init, s));
    return XAN_OK;
}

static int abcd_check_spinup(int spinup) {
    if (spinup < 25) {
        // ABCD.set_vals indexes month -25 of the spin-up arrays (abcd.py:255-266)
        set_error("Spin-up steps must produce at least 10 years spin-up. Your spin-up only consist of %d months. "
                  "Please reconfigure and try again.", spinup);
        return XAN_E_SPINUP;
    }
    return XAN_OK;
}

extern "C" {

xan_abcd_plan *xan_abcd_plan_create(const int *h_basin_idx, int ncell, int n_basins) {
    if (!h_basin_idx || ncell <= 0 || n_basins <= 0) {
        set_error("xan_abcd_plan_create: bad arguments (ncell=%d, n_basins=%d)", ncell, n_basins);
        return nullptr;
    }
    auto *pl = new xan_abcd_plan();
    pl->ncell = ncell;
    pl->n_basins = n_basins;
    pl->h_offsets.assign(n_basins + 1, 0);
    for (int c = 0; c < ncell; ++c) {
        const int b = h_basin_idx[c];
        if (b >= n_basins) {
            set_error("xan_abcd_plan_create: basin index %d of cell %d >= n_basins %d", b, c, n_basins);
            delete pl;
            return nullptr;
        }
        if (b >= 0) pl->h_offsets[b + 1]++;
    }
    for (int b = 0; b < n_basins; ++b) {
        pl->max_basin_cells = std::max(pl->max_basin_cells, pl->h_offsets[b + 1]);
        pl->h_offsets[b + 1] += pl->h_offsets[b];
    }
    const int n_live = pl->h_offsets[n_basins];
    pl->h_order.assign(std::max(n_live, 1), 0);
    std::vector<int> cur(pl->h_offsets.begin(), pl->h_offsets.end() - 1);
    for (int c = 0; c < ncell; ++c) {
        const int b = h_basin_idx[c];
        if (b >= 0) pl->h_order[cur[b]++] = c;
    }
    bool ok = cudaMalloc(&pl->d_basin_idx, sizeof(int) * ncell) == cudaSuccess &&
              cudaMalloc(&pl->d_order, sizeof(int) * std::max(n_live, 1)) == cudaSuccess &&
              cudaMalloc(&pl->d_offsets, sizeof(int) * (n_basins + 1)) == cudaSuccess &&
              cudaMemcpy(pl->d_basin_idx, h_basin_idx, sizeof(int) * ncell, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(pl->d_order, pl->h_order.data(), sizeof(int) * std::max(n_live, 1),
                         cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(pl->d_offsets, pl->h_offsets.data(), sizeof(int) * (n_basins + 1),
                         cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok) {
        set_error("xan_abcd_plan_create: CUDA allocation/copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        xan_abcd_plan_destroy(pl);
        return nullptr;
    }
    return pl;
}

void xan_abcd_plan_destroy(xan_abcd_plan *pl) {
    if (!pl) return;
    cudaFree(pl->d_basin_idx);
    cudaFree(pl->d_order);
    cudaFree(pl->d_offsets);
    delete pl;
}

int xan_abcd_run(const xan_abcd_plan *pl, const double *d_pet, const double *d_precip, const double *d_tmin,
                 const double *d_pars, int nmonths, int spinup, int ld, double *d_aet, double *d_q,
                 double *d_sav, void *stream) {
    XAN_REQUIRE(pl && d_pet && d_precip && d_pars, "xan_abcd_run: null pointer");
    XAN_REQUIRE(nmonths > 0 && ld >= pl->ncell, "xan_abcd_run: bad shape nmonths=%d ld=%d", nmonths, ld);
    if (abcd_check_spinup(spinup) != XAN_OK) return XAN_E_SPINUP;
    XAN_REQUIRE(spinup <= nmonths, "xan_abcd_run: spinup (%d) exceeds the %d months of forcing", spinup, nmonths);
    AbcdSetOut out{};
    out.aet[0] = d_aet;
    out.q[0] = d_q;
    out.sav[0] = d_sav;
    return abcd_launch<1>(pl, 1, pl->n_basins, d_pet, d_precip, d_tmin, d_pars, nmonths, spinup, ld, out,
                          (cudaStream_t)stream);
}

int xan_abcd_run_sets(const xan_abcd_plan *pl, int n_sets, int n_rows, const double *d_pet, const double *d_precip,
                      const double *d_tmin, const double *d_pars, int nmonths, int spinup, int ld,
                      double *const *h_aet, double *const *h_q, double *const *h_sav, void *stream) {
    XAN_REQUIRE(pl && d_pet && d_precip && d_pars, "xan_abcd_run_sets: null pointer");
    XAN_REQUIRE(n_sets >= 1 && n_sets <= XAN_ABCD_MAX_SETS, "xan_abcd_run_sets: n_sets=%d outside 1 .. %d", n_sets,
                XAN_ABCD_MAX_SETS);
    XAN_REQUIRE(n_rows >= 1, "xan_abcd_run_sets: n_rows=%d", n_rows);
    XAN_REQUIRE(nmonths > 0 && ld >= pl->ncell, "xan_abcd_run_sets: bad shape nmonths=%d ld=%d", nmonths, ld);
    if (abcd_check_spinup(spinup) != XAN_OK) return XAN_E_SPINUP;
    XAN_REQUIRE(spinup <= nmonths, "xan_abcd_run_sets: spinup (%d) exceeds the %d months of forcing", spinup,
                nmonths);
    int max_row = -1;   // the last row the plan maps a live cell to: every table must have it
    for (int b = 0; b < pl->n_basins; ++b)
        if (pl->h_offsets[b + 1] > pl->h_offsets[b]) max_row = b;
    XAN_REQUIRE(max_row < n_rows, "xan_abcd_run_sets: the plan maps cells to row %d, the tables have %d rows",
                max_row, n_rows);
    AbcdSetOut out{};
    for (int k = 0; k < n_sets; ++k) {
        out.aet[k] = h_aet ? h_aet[k] : nullptr;
        out.q[k] = h_q ? h_q[k] : nullptr;
        out.sav[k] = h_sav ? h_sav[k] : nullptr;
    }
    // one set alone takes the K = 1 instance: a group of K would step its spare slot through every month for nothing
    if (n_sets == 1)
        return abcd_launch<1>(pl, 1, n_rows, d_pet, d_precip, d_tmin, d_pars, nmonths, spinup, ld, out,
                              (cudaStream_t)stream);
    return abcd_launch<ABCD_SETS_PER_THREAD>(pl, n_sets, n_rows, d_pet, d_precip, d_tmin, d_pars, nmonths, spinup,
                                             ld, out, (cudaStream_t)stream);
}

// Population layout of the calibration objective (see kge_pop_pass_kernel).
static int kge_population(const xan_abcd_plan *pl, const int *h_basins, int nb, int npar, const double *d_pet,
                          const double *d_precip, const double *d_tmin, const double *d_area, const double *d_pars,
                          const double *d_obs, int nmonths, int spinup, int ld, int unit_km3, double *d_ed,
                          double *d_series, cudaStream_t s) {
    const int npad = (npar + 31) / 32 * 32;
    XAN_REQUIRE(npad <= 512, "xan_abcd_kge_batch: at most 512 parameter sets per basin and call (got %d)", npar);
    std::vector<KgeChunk> chunks;
    std::vector<int> slot_chunk0(nb + 1, 0);
    for (int i = 0; i < nb; ++i) {
        const int beg = pl->h_offsets[h_basins[i]], end = pl->h_offsets[h_basins[i] + 1];
        slot_chunk0[i] = (int)chunks.size();
        for (int b = beg; b < end; b += KC) chunks.push_back(KgeChunk{i, b, std::min(KC, end - b)});
        while (chunks.size() % KQ) chunks.push_back(KgeChunk{i, beg, 0});   // padding chunks: no cell counts
    }
    slot_chunk0[nb] = (int)chunks.size();
    const int nch = (int)chunks.size();
    KgeChunk *d_chunks = nullptr;
    int *d_slot0 = nullptr;
    double *snap = nullptr, *init = nullptr, *part = nullptr, *series = nullptr;
    XAN_CUDA_CHECK(scratch_alloc(&d_chunks, sizeof(KgeChunk) * nch, s));
    XAN_CUDA_CHECK(scratch_alloc(&d_slot0, sizeof(int) * (nb + 1), s));
    XAN_CUDA_CHECK(scratch_alloc(&snap, sizeof(double) * 12 * (size_t)nch * npad, s));
    XAN_CUDA_CHECK(scratch_alloc(&init, sizeof(double) * 2 * (size_t)nb * npar, s));
    XAN_CUDA_CHECK(scratch_alloc(&part, sizeof(double) * (size_t)(nch / KQ) * nmonths * npad, s));
    XAN_CUDA_CHECK(scratch_alloc(&series, sizeof(double) * (size_t)nb * nmonths * npad, s));
    XAN_CUDA_CHECK(cudaMemcpyAsync(d_chunks, chunks.data(), sizeof(KgeChunk) * nch, cudaMemcpyHostToDevice, s));
    XAN_CUDA_CHECK(cudaMemcpyAsync(d_slot0, slot_chunk0.data(), sizeof(int) * (nb + 1), cudaMemcpyHostToDevice, s));
    const int grid = (nch / KQ) * (npad / 32);
    if (d_tmin)
        kge_pop_pass_kernel<true, false><<<grid, 128, 0, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, d_chunks, nch,
                                                              d_pars, nullptr, npar, npad, spinup, ld, unit_km3, snap);
    else
        kge_pop_pass_kernel<false, false><<<grid, 128, 0, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, d_chunks, nch,
                                                               d_pars, nullptr, npar, npad, spinup, ld, unit_km3, snap);
    kge_pop_reinit_kernel<<<nb, 256, sizeof(double) * 12 * npad, s>>>(snap, d_slot0, npar, npad, init);
    if (d_tmin)
        kge_pop_pass_kernel<true, true><<<grid, 128, 0, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, d_chunks, nch,
                                                             d_pars, init, npar, npad, nmonths, ld, unit_km3, part);
    else
        kge_pop_pass_kernel<false, true><<<grid, 128, 0, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, d_chunks, nch,
                                                              d_pars, init, npar, npad, nmonths, ld, unit_km3, part);
    kge_pop_series_kernel<<<dim3(nb, 8), 256, 0, s>>>(part, d_slot0, nmonths, npad, series);
    kge_pop_finish_kernel<<<nb, 64, 0, s>>>(series, d_obs, npar, npad, nmonths, d_ed, d_series);
    XAN_CUDA_CHECK(cudaGetLastError());
    // (the host tables are pageable: cudaMemcpyAsync has staged them before it returned)
    XAN_CUDA_CHECK(cudaFreeAsync(d_chunks, s));
    XAN_CUDA_CHECK(cudaFreeAsync(d_slot0, s));
    XAN_CUDA_CHECK(cudaFreeAsync(snap, s));
    XAN_CUDA_CHECK(cudaFreeAsync(init, s));
    XAN_CUDA_CHECK(cudaFreeAsync(part, s));
    XAN_CUDA_CHECK(cudaFreeAsync(series, s));
    return XAN_OK;
}

int xan_abcd_kge_batch(const xan_abcd_plan *pl, const int *h_basins, int nb, int npar, const double *d_pet,
                       const double *d_precip, const double *d_tmin, const double *d_area, const double *d_pars,
                       const double *d_obs, int nmonths, int spinup, int ld, int unit_km3, double *d_ed,
                       double *d_series, void *stream) {
    XAN_REQUIRE(pl && h_basins && d_pet && d_precip && d_pars && d_obs && d_ed, "xan_abcd_kge_batch: null pointer");
    XAN_REQUIRE(!unit_km3 || d_area, "xan_abcd_kge_batch: km3_per_mth needs the cell areas");
    XAN_REQUIRE(nb > 0 && npar > 0 && nmonths > 0 && ld >= pl->ncell, "xan_abcd_kge_batch: bad shape");
    if (spinup < 25) {
        set_error("Spin-up steps must produce at least 10 years spin-up. Your spin-up only consist of %d months. "
                  "Please reconfigure and try again.", spinup);
        return XAN_E_SPINUP;
    }
    XAN_REQUIRE(spinup <= nmonths, "xan_abcd_kge_batch: spinup (%d) exceeds the %d months of forcing", spinup,
                nmonths);
    cudaStream_t s = (cudaStream_t)stream;
    for (int i = 0; i < nb; ++i) {
        XAN_REQUIRE(h_basins[i] >= 0 && h_basins[i] < pl->n_basins, "xan_abcd_kge_batch: basin row %d out of range",
                    h_basins[i]);
        XAN_REQUIRE(pl->h_offsets[h_basins[i] + 1] > pl->h_offsets[h_basins[i]],
                    "xan_abcd_kge_batch: basin row %d has no cells", h_basins[i]);
    }
    {
        const char *env = getenv("XANTHOS_KGE_LAYOUT");   // "block" forces the block-per-(candidate, basin) kernel
        const bool force_block = env && !strcmp(env, "block"), force_pop = env && !strcmp(env, "population");
        if (!force_block && (npar >= 16 || force_pop))
            return kge_population(pl, h_basins, nb, npar, d_pet, d_precip, d_tmin, d_area, d_pars, d_obs, nmonths,
                                  spinup, ld, unit_km3, d_ed, d_series, s);
    }
    // schedule big basins first (longest-processing-time order)
    std::vector<int> slots(nb);
    std::iota(slots.begin(), slots.end(), 0);
    int max_cells = 0;
    for (int i = 0; i < nb; ++i) {
        XAN_REQUIRE(h_basins[i] >= 0 && h_basins[i] < pl->n_basins, "xan_abcd_kge_batch: basin row %d out of range",
                    h_basins[i]);
        const int n = pl->h_offsets[h_basins[i] + 1] - pl->h_offsets[h_basins[i]];
        XAN_REQUIRE(n > 0, "xan_abcd_kge_batch: basin row %d has no cells", h_basins[i]);
        max_cells = std::max(max_cells, n);
    }
    std::stable_sort(slots.begin(), slots.end(), [&](int x, int y) {
        const int nx = pl->h_offsets[h_basins[x] + 1] - pl->h_offsets[h_basins[x]];
        const int ny = pl->h_offsets[h_basins[y] + 1] - pl->h_offsets[h_basins[y]];
        return nx > ny;
    });
    std::vector<int> h_meta(2 * nb);
    for (int i = 0; i < nb; ++i) {
        h_meta[i] = h_basins[slots[i]];
        h_meta[nb + i] = slots[i];
    }
    const size_t smem = sizeof(double) * (3 * (size_t)max_cells + (KGE_NT / 32) * (size_t)nmonths + 16);
    XAN_REQUIRE(smem <= 227 * 1024, "xan_abcd_kge_batch: basin with %d cells x %d months needs %zu B of shared memory",
                max_cells, nmonths, smem);
    int *d_meta = nullptr;
    XAN_CUDA_CHECK(scratch_alloc(&d_meta, sizeof(int) * 2 * nb, s));
    XAN_CUDA_CHECK(cudaMemcpyAsync(d_meta, h_meta.data(), sizeof(int) * 2 * nb, cudaMemcpyHostToDevice, s));
    dim3 grid(npar, nb);
    if (d_tmin) {
        XAN_CUDA_CHECK(cudaFuncSetAttribute(abcd_kge_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        abcd_kge_kernel<true><<<grid, KGE_NT, smem, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, pl->d_offsets,
                                                         d_meta, d_meta + nb, d_pars, d_obs, npar, nmonths, spinup, ld,
                                                         unit_km3, d_ed, d_series);
    } else {
        XAN_CUDA_CHECK(cudaFuncSetAttribute(abcd_kge_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        abcd_kge_kernel<false><<<grid, KGE_NT, smem, s>>>(d_pet, d_precip, d_tmin, d_area, pl->d_order, pl->d_offsets,
                                                          d_meta, d_meta + nb, d_pars, d_obs, npar, nmonths, spinup, ld,
                                                          unit_km3, d_ed, d_series);
    }
    XAN_CUDA_CHECK(cudaGetLastError());
    XAN_CUDA_CHECK(cudaFreeAsync(d_meta, s));
    return XAN_OK;
}

int xan_basin_sum(const xan_abcd_plan *pl, const double *d_src, const double *d_w, int nmonths, int ld,
                  double *d_out, void *stream) {
    XAN_REQUIRE(pl && d_src && d_out, "xan_basin_sum: null pointer");
    XAN_REQUIRE(nmonths > 0 && ld >= pl->ncell, "xan_basin_sum: bad shape");
    dim3 grid(pl->n_basins, ceil_div(nmonths, 8));
    basin_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_src, d_w, pl->d_order, pl->d_offsets, pl->n_basins,
                                                            nmonths, ld, d_out);
    XAN_CUDA_CHECK(cudaGetLastError());
    return XAN_OK;
}

}  // extern "C"
