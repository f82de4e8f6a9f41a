/*
 * xanthos_b200.h - C ABI of libxanthos_b200.so, the B200 (sm_100a) implementation of the
 * Xanthos per-month grid hot path: PET (Penman-Monteith, Hargreaves-Samani, Thornthwaite),
 * ABCD runoff, MRTM river routing and the ABCD calibration objective.
 *
 * This is the drop-in boundary.  The reference (JGCRI/xanthos v2.4.1) is pure Python: its
 * "plug-in API" is the set of module-level functions that xanthos/components.py calls
 * (components.py:189-296, 486-497).  Every entry point below replaces the body of one of those
 * functions; the reference-side binding is a ctypes stub (see INTEGRATION.md).
 *
 * Conventions
 *   - d_* pointers are DEVICE pointers, h_* pointers are HOST pointers.
 *   - Field arrays are fp64, month-major: element (month m, cell c) lives at ptr[m * ld + c],
 *     ld >= ncell.  The reference's own layout is [ncell][nmonths] (cell-major); use
 *     xan_to_month_major / xan_to_cell_major at the boundary.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - Return value: 0 on success, a negative XAN_E_* code otherwise; xan_last_error() gives the
 *     message of the last failure on the calling thread.
 *   - No CPU fallback exists: if no CUDA device is usable every compute entry point fails.
 */
#ifndef XANTHOS_B200_H
#define XANTHOS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XAN_OK 0
#define XAN_E_INVALID (-1)  /* bad argument (maps to ValidationException / ValueError)          */
#define XAN_E_CUDA (-2)     /* CUDA runtime failure (maps to RuntimeError)                      */
#define XAN_E_SPINUP (-3)   /* ABCD spin-up shorter than 25 months (maps to IndexError,         */
                            /* xanthos/runoff/abcd.py:253-266)                                  */
#define XAN_E_NOMEM (-4)

#define XAN_PM_MAX_CLASSES 32

/* ---- library ------------------------------------------------------------------------------ */
int xan_version(void);
const char *xan_last_error(void);
/* number of SMs / compute capability of the current device (fails without a GPU) */
int xan_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* ---- layout at the boundary (reference arrays are [ncell][nmonths], data_load.py:288-340) -- */
/* nan_to_num != 0 applies numpy.nan_to_num (NaN->0, +-inf->+-DBL_MAX) on the fly, as the loader
 * does for the PM forcings, Thornthwaite tas and ABCD tmin (data_load.py:120-125, 138, 194). */
int xan_to_month_major(const double *d_src, double *d_dst, int ncell, int nmonths, int ld,
                       int nan_to_num, void *stream);
/* the same from a single-precision source: forcing whose values are single precision (NetCDF float variables of
 * the ESMs, widened to float64 by the loader) can cross the host-device link at half the bytes; float -> double
 * is exact, so the month-major field is bit-identical to the one made from the float64 array */
int xan_to_month_major_f32(const float *d_src, double *d_dst, int ncell, int nmonths, int ld,
                           int nan_to_num, void *stream);
int xan_to_cell_major(const double *d_src, double *d_dst, int ncell, int nmonths, int ld,
                      void *stream);

/* ---- PET ---------------------------------------------------------------------------------- */
/* Hargreaves-Samani; replaces hargreaves_samani.execute (xanthos/pet/hargreaves_samani.py:91-119,
 * per-element formula :31-65).  Month k is calendar month k % 12 of year start_year + k / 12
 * (Gregorian month lengths, :18-28). */
int xan_hs_pet(const double *d_tas, const double *d_tmax, const double *d_tmin,
               const double *d_lat_deg, double *d_pet, int ncell, int nmonths, int ld,
               int start_year, void *stream);

/* Thornthwaite; replaces thornthwaite.execute (xanthos/pet/thornthwaite.py:47-130) including the
 * np.repeat day-length tiling of :110.  NaN / negative temperatures count as 0 (:82). */
int xan_thornthwaite_pet(const double *d_tas, const double *d_lat_rad, double *d_pet, int ncell,
                         int nmonths, int ld, int start_year, void *stream);

/* Monthly mean day length; replaces calc_daylight_hours (thornthwaite.py:18-44) for a 365-day
 * year (rows 0..11 of d_hours) and a 366-day year (rows 12..23); d_hours is [24][ncell]. */
int xan_thornthwaite_daylight(const double *d_lat_rad, double *d_hours, int ncell, void *stream);

/* Penman-Monteith; replaces run_pmpet (xanthos/pet/penman_monteith.py:394-477).
 * Per-class vectors and [nlcs][12] tables are HOST pointers (data_load.py:94-117). */
typedef struct xan_pm_tables {
    int nlcs;      /* number of land classes, 7 <= nlcs <= XAN_PM_MAX_CLASSES (rows 0 and 6 of
                      alpha are hard-wired to water and snow, penman_monteith.py:361, 377)     */
    int water_idx; /* class whose ET is replaced by et_water (:459-460)                        */
    int snow_idx;  /* class whose ET is replaced by et_snow  (:462-464)                        */
    const double *cL, *beta, *rslimit, *Tminopen, *Tminclose, *VPDclose, *VPDopen, *RBLmin,
        *RBLmax, *rc, *emiss;                /* [nlcs]     */
    const double *alpha, *lai, *laimin, *laimax; /* [nlcs][12] */
} xan_pm_tables;

/* d_lct: [n_lc_years][nlcs][ld] (land-cover percentages, class-major per year);
 * h_lc_index[y] = land-cover slice used for year start_year + y (SetData, :32-43);
 * d_prev_idx: optional [ncell] index of the cell whose tair is "tairprev" (data_load.py:128-129);
 *             NULL means cell c uses cell c-1 and cell 0 uses 0.0; an entry < 0 also means 0.0.
 *             Indices may address halo columns ncell <= j < ld of d_tair. */
int xan_pm_pet(const double *d_tair, const double *d_tmin, const double *d_rhs,
               const double *d_wind, const double *d_rsds, const double *d_rlds,
               const double *d_lct, const double *d_elev, const int *d_prev_idx,
               const xan_pm_tables *h_tables, const int *h_lc_index, double *d_pet, int ncell,
               int nmonths, int ld, int start_year, void *stream);

/* ---- ABCD runoff -------------------------------------------------------------------------- */
/* A plan holds the basin -> cells ordering used by the deterministic per-basin re-initialisation
 * (ABCD.set_vals, xanthos/runoff/abcd.py:246-282).  h_basin_idx[c] = 0-based row of the
 * parameter table for cell c, or < 0 for cells that are not simulated (they come back as NaN;
 * the reference leaves them uninitialised, :384-389). */
typedef struct xan_abcd_plan xan_abcd_plan;
xan_abcd_plan *xan_abcd_plan_create(const int *h_basin_idx, int ncell, int n_basins);
void xan_abcd_plan_destroy(xan_abcd_plan *plan);

/* Replaces abcd_execute / ABCD.emulate (abcd.py:394-422, :305-311): spin-up over the first
 * `spinup` months from SW0=100, GW0=500, per-basin re-initialisation from the last three
 * Decembers, then `nmonths` simulated months.  d_tmin may be NULL (no snow, m = 0).
 * d_pars: [n_basins][5] = a, b, c, d, m.  Outputs month-major; any of them may be NULL. */
int xan_abcd_run(const xan_abcd_plan *plan, const double *d_pet, const double *d_precip,
                 const double *d_tmin, const double *d_pars, int nmonths, int spinup, int ld,
                 double *d_aet, double *d_q, double *d_sav, void *stream);

/* n_sets parameter tables over the same forcing in one call.  d_pars: [n_sets][n_rows][5], n_rows = the rows of
 * ONE table (its stride; the rows the plan maps live cells to must be < n_rows, as for xan_abcd_run).
 * h_aet / h_q / h_sav: HOST arrays of n_sets DEVICE pointers; the arrays and any entry may be NULL.
 * Set s is bit-identical to xan_abcd_run(plan, ..., d_pars + s * n_rows * 5, ...).  1 <= n_sets <= XAN_ABCD_MAX_SETS. */
#define XAN_ABCD_MAX_SETS 8
int xan_abcd_run_sets(const xan_abcd_plan *plan, int n_sets, int n_rows, const double *d_pet,
                      const double *d_precip, const double *d_tmin, const double *d_pars, int nmonths,
                      int spinup, int ld, double *const *h_aet, double *const *h_q, double *const *h_sav,
                      void *stream);

/* Calibration objective for a batch of parameter sets; replaces objective_kge + basin_runoff
 * (xanthos/calibrate/calibrate_abcd.py:134-162, 176-213) evaluated `npar` times per basin.
 * For basin b = h_basins[i] (row of the plan) and parameter set p:
 *   mod[t] = nansum_cells(q[t][c] * w[c]),  w = area * 1e-6 (km3_per_mth) or 1 (mm_per_mth)
 *   ed     = sqrt((r-1)^2 + (std(mod)/std(obs)-1)^2 + (mean(mod)/mean(obs)-1)^2)
 * d_pars: [nb][npar][5]; d_obs: [nb][nmonths]; d_ed: [nb][npar];
 * d_series (optional): [nb][npar][nmonths] modelled basin series. */
int xan_abcd_kge_batch(const xan_abcd_plan *plan, const int *h_basins, int nb, int npar,
                       const double *d_pet, const double *d_precip, const double *d_tmin,
                       const double *d_area, const double *d_pars, const double *d_obs,
                       int nmonths, int spinup, int ld, int unit_km3, double *d_ed,
                       double *d_series, void *stream);

/* ---- MRTM routing ------------------------------------------------------------------------- */
/* Integer topology, bit-exact, host-side (no device needed).
 * xan_mrtm_downstream replaces downstream (xanthos/routing/mrtm.py:85-120 with make_flowdirgrid
 * :233-258): h_coords [ncell][5] = id, lon, lat, ilon, ilat (1-based), h_flow_dir D8 codes
 * (-9999 = missing) -> h_dsid [ncell] (1-based id, -1 = outlet).
 * xan_mrtm_upstream replaces upstream (mrtm.py:123-191): -> h_upid [ncell][9], the 8 neighbour
 * ids with the inflowing ones first (stable) and their count in column 8. */
int xan_mrtm_downstream(const double *h_coords, const double *h_flow_dir, int ncell, int nrow,
                        int ncol, int64_t *h_dsid);
int xan_mrtm_upstream(const double *h_coords, const int64_t *h_dsid, int ncell, int nrow, int ncol,
                      int64_t *h_upid);

/* Execution plan; replaces upstream_genmatrix (mrtm.py:194-230): from h_upid [ncell][9] it
 * builds the rows of UM = UP - I, checks that the flow graph is a forest, cuts large river trees
 * into pieces of at most 31 lanes and packs them into warps (lane 31 of every warp stays empty).
 * block_threads: multiple of 32, <= 640; <= 0 picks the default 640 (20 warps, one block per SM,
 * 96 registers).  chunk_substeps: kept for ABI stability (1..1024, <= 0 = default) and otherwise
 * unused - warps hand their cut-edge series over once per month.  At launch the packed warps are
 * assigned to SM sub-partitions by cost and loop variant (see mrtm_sched_kernel;
 * XANTHOS_MRTM_SCHED=static binds packed warp w to grid warp w instead).  Plan
 * creation is host-side integer work and needs no device; the device tables are uploaded by the
 * first xan_mrtm_route call. */
typedef struct xan_mrtm_plan xan_mrtm_plan;
xan_mrtm_plan *xan_mrtm_plan_create(const int64_t *h_upid, int ncell, int block_threads,
                                    int chunk_substeps);
void xan_mrtm_plan_destroy(xan_mrtm_plan *plan);
/* rows of UM = UP - I in CSR form (mrtm.py:194-230): indptr [ncell+1], indices/data [nnz] */
int xan_mrtm_plan_um_nnz(const xan_mrtm_plan *plan);
int xan_mrtm_plan_um(const xan_mrtm_plan *plan, int64_t *h_indptr, int64_t *h_indices,
                     int64_t *h_data);
/* info[0]=is_forest info[1]=n_components info[2]=max_component info[3]=n_warps
 * info[4]=n_cut_edges info[5]=n_levels info[6]=block_threads info[7]=max ghost lanes of a warp */
int xan_mrtm_plan_info(const xan_mrtm_plan *plan, int *info8);
/* diagnostic export of the warp-kernel packing: lane_cell [n_warps * 32] (cell index or -1),
 * edge_prod / edge_cons [n_cut_edges] (warp indices).  Any pointer may be NULL. */
int xan_mrtm_plan_packing(const xan_mrtm_plan *plan, int *h_lane_cell, int *h_edge_prod,
                          int *h_edge_cons);

/* diagnostic export of the skew-kernel plan (csrc/mrtm_skew.cu; built on first use).
 * info[0]=K (cells per lane) [1]=n_warps [2]=n_cut_edges [3]=n_levels [4]=max ghost entries of a warp
 * [5]=max lag [6]=n_pieces [7]=row-term sources per lane [8]=index of the all-zero table entry
 * [9]=ghost entries per warp [10]=export entries per warp [11]=iterations a cell lags its tributaries;
 * all zero if the graph has no skew plan.
 * Tables (any pointer may be NULL): cell, lag [n_warps][32 K]; src [n_warps][32][info[7]];
 * ghost_edge, ghost_lag [n_warps][info[9]]; exp_edge, exp_place [n_warps][info[10]]; Dw [n_warps];
 * edge_prod, edge_cons [n_cut_edges]. */
int xan_mrtm_skew_info(xan_mrtm_plan *plan, int *info12);
/* Pacing window the skew kernel would use for this plan: out4[0] = effective window in months for a requested window
 * (0 = off; any other value is raised to the smallest deadlock-free one: pipeline depth of the linked warps + ring
 * capacity, in months of nt_min sub-steps), [1] = sub-steps per hand-over chunk, [2] = ring entries per cut edge,
 * [3] = default requested window.  Host only. */
int xan_mrtm_skew_window(xan_mrtm_plan *plan, int requested, int nt_min, int *out4);
int xan_mrtm_skew_tables(xan_mrtm_plan *plan, int *cell, int *lag, int *src, int *ghost_edge,
                         int *ghost_lag, int *exp_edge, int *exp_place, int *Dw, int *edge_prod,
                         int *edge_cons);

#define XAN_MRTM_AUTO 0  /* skew kernel if the flow graph is a forest and the calendar allows it,
                          * else the warp-dataflow kernel, else the grid kernel              */
#define XAN_MRTM_GRID 1  /* cooperative grid-sync kernel (any graph)            */
#define XAN_MRTM_TREE 2  /* force the warp-dataflow kernel (fails if not a forest) */
#define XAN_MRTM_SKEW 3  /* force the skew kernel (fails if it is not available)   */

/* Replaces the routing loops of Components.calculate_routing (xanthos/components.py:262-296)
 * around streamrouting (mrtm.py:16-82): `spinup_months` months of spin-up over the first months
 * of d_runoff starting from d_chs_prev (NULL = zeros), then nmonths months continuing from the
 * spun-up storage.  h_ndays[m] = days of month m (mod-4 leap rule, utils/general.py:15-50);
 * dt in seconds (reference: 3 * 3600, components.py:91).
 * Outputs: d_chs, d_avg month-major [nmonths][ld] (either may be NULL); d_instream [ncell] =
 * instantaneous flow after the last sub-step (may be NULL). */
int xan_mrtm_route(xan_mrtm_plan *plan, const double *d_runoff, const double *d_flow_dist,
                   const double *d_velocity, const double *d_area, const double *d_chs_prev,
                   const int *h_ndays, int nmonths, int spinup_months, int ld, double dt,
                   int method, double *d_chs, double *d_avg, double *d_instream, void *stream);

/* Ensemble variant of xan_mrtm_route: n_members independent scenarios (same topology, same static
 * fields, same calendar) in one call.  The h_* arguments are HOST arrays of n_members DEVICE
 * pointers (h_chs_prev, h_chs, h_avg, h_instream and any of their entries may be NULL).  On a river
 * forest two members share one launch of the skew kernel: their thread blocks are co-resident on
 * every SM and fill each other's idle issue slots (31 against 43 ms per member on the 0.5 degree
 * world; XANTHOS_MRTM_SKEW_MEMBERS=1 routes one member per launch, =3 three where they fit).  With
 * the warp-dataflow kernel (XANTHOS_MRTM_AUTO=tree) members are advanced one after the other (two
 * members per warp measured slower: 69 against 54 ms per member; XANTHOS_MRTM_MEMBERS=2 keeps that
 * path testable).  Results are bit-identical to n_members calls of xan_mrtm_route.  Concurrent calls
 * on one plan from different streams are allowed: rings and counters are per-launch scratch. */
int xan_mrtm_route_batch(xan_mrtm_plan *plan, int n_members, const double *const *h_runoff,
                         const double *d_flow_dist, const double *d_velocity, const double *d_area,
                         const double *const *h_chs_prev, const int *h_ndays, int nmonths,
                         int spinup_months, int ld, double dt, int method, double *const *h_chs,
                         double *const *h_avg, double *const *h_instream, void *stream);

/* ---- step-wise (legacy v1) path: Hargreaves PET + GWAM runoff ------------------------------- */
/* Replaces hargreaves.calculate_pet (xanthos/pet/hargreaves.py:17-73), which Components.simulation
 * calls once per month (components.py:329-340), for the whole series in one launch.  d_temp / d_dtr
 * month-major [nmonths][ld] (NaN -> 0 and negative dtr -> 0 are applied inside, components.py:143-176,
 * hargreaves.py:32); h_solar_dec / h_dr [nmonths] from calc_sinusoidal_factor
 * (utils/general.py:53-90); h_days [nmonths] days per month (mod-4 leap rule). */
int xan_hargreaves_pet(const double *d_temp, const double *d_dtr, const double *d_lat_rad,
                       const double *h_solar_dec, const double *h_dr, const int *h_days,
                       double *d_pet, int ncell, int nmonths, int ld, void *stream);
/* Replaces the month loop around gwam.runoffgen (xanthos/runoff/gwam.py:18-88; components.py:358-366)
 * including the spin-up pass of ConfigRunner.run (configurations.py:106-113): `spinup_months` months
 * from d_sm_prev that only carry the soil moisture over, then nmonths months from month 0.
 * d_sm_max [ncell]: maximum soil moisture, 999 = water body, 0 = no soil.  Outputs month-major
 * [nmonths][ld] (any may be NULL); d_sm_after_spinup / d_sm_last [ncell] (may be NULL) are the carried
 * soil moisture after the spin-up pass and after the last month. */
int xan_gwam_run(const double *d_pet, const double *d_precip, const double *d_sm_max,
                 const double *d_sm_prev, int ncell, int nmonths, int spinup_months, int ld,
                 double *d_aet, double *d_q, double *d_sav, double *d_sm_after_spinup,
                 double *d_sm_last, void *stream);

/* ---- device-resident output staging (OutWriter, xanthos/data_writer/out_writer.py:237-265) -- */
/* sums (or means) every 12 consecutive months: [nmonths][ld] -> [nmonths/12][ld] */
int xan_agg_to_year(const double *d_src, double *d_dst, int ncell, int nmonths, int ld,
                    int take_mean, void *stream);
/* basin aggregate: out[m][b] = nansum_{c in basin b} src[m][c] * w[c] (w may be NULL = 1) */
int xan_basin_sum(const xan_abcd_plan *plan, const double *d_src, const double *d_w,
                  int nmonths, int ld, double *d_out, void *stream);
/* mm -> km3 (out_writer.py:114-115): dst[t][c] = src[t][c] * scale[c] over [ntime][ld]; d_dst may be d_src */
int xan_scale_cells(const double *d_src, const double *d_scale, int ncell, int ntime, int ld,
                    double *d_dst, void *stream);

/* ---- across-member statistics of an ensemble (csrc/ensemble_stats.cu) ------------------------- */
/* State per (time, cell), month-major [ntime][ld], 16-byte aligned: d_sm = (sum, m2) and d_mm = (min, max) as
 * interleaved pairs of doubles ([ntime][ld][2] each).  Operations are + - * / sqrt only (no FMA contraction), so the
 * results are bitwise those of oracle/ensemble_stats.py.
 *   xan_ens_stats_update    adds member number n (1-based, member order) with values d_x [ntime][ld]: n == 1
 *                           initialises (sum = x, m2 = 0, min = max = x); later members add x to the sequential sum
 *                           (numpy.mean(stack, axis=0) = sum / n bitwise), update m2 by Welford with the running mean
 *                           sum / n, and min / max propagate NaN like numpy.min / numpy.max.
 *   xan_ens_stats_merge     Chan et al.: partial a of na members absorbs partial b of nb members in place:
 *                           sum = sa + sb, m2 = m2a + m2b + d * d * na * nb / (na + nb) with d = sb / nb - sa / na.
 *   xan_ens_stats_finalize  numpy.mean, numpy.std(ddof) = sqrt(m2 / (n - ddof)), numpy.min, numpy.max over the n
 *                           members, written cell-major [ncell][ntime]; any output may be NULL. */
int xan_ens_stats_update(const double *d_x, double *d_sm, double *d_mm, int ncell, int ntime, int ld, int n,
                         void *stream);
int xan_ens_stats_merge(double *d_sm_a, double *d_mm_a, const double *d_sm_b, const double *d_mm_b, int ncell,
                        int ntime, int ld, int na, int nb, void *stream);
int xan_ens_stats_finalize(const double *d_sm, const double *d_mm, int ncell, int ntime, int ld, int n, int ddof,
                           double *d_mean, double *d_std, double *d_min, double *d_max, void *stream);
/* numpy.quantile(stack, levels, axis=0) with method 'linear' over n members, all levels in one pass.
 * d_x points at time step t0 of member 0 of a month-major stack: member i, step t in [t0, t1) is
 * d_x[i * member_stride + (t - t0) * ld + c].  lo / gamma (host arrays of nq) are numpy's virtual index (n - 1) q of
 * every level split into floor and fraction; the result interpolates the sorted members lo and lo + 1 (clamped) with
 * numpy's two-sided rule.  A NaN member gives NaN at every level of its (cell, step).  d_out is cell-major
 * [nq][ncell][ntime]; the call writes columns [t0, t1). */
#define XAN_ENS_MAX_MEMBERS 256
#define XAN_ENS_MAX_LEVELS 64
int xan_ens_quantiles(const double *d_x, long long member_stride, int n, int ncell, int ld, int t0, int t1,
                      int ntime, int nq, const int *lo, const double *gamma, double *d_out, void *stream);

/* ---- post-processing scans on the resident fields (SURVEY.md section 8 row f3) -------------- */
/* DroughtStats.droughtstats (xanthos/drought/drought_stats.py:85-148): d_hydro [nmonths][ld],
 * d_thresh [nthresh][ld_thresh] (row t % nthresh applies to month t) -> severity, intensity,
 * duration [nmonths][ld].  Bit-identical to the numpy loop. */
int xan_drought_stats(const double *d_hydro, const double *d_thresh, int ncell, int nmonths, int ld,
                      int nthresh, int ld_thresh, double *d_severity, double *d_intensity,
                      double *d_duration, void *stream);
/* The same scan with optional outputs (the ensemble runner's drought statistics).  Severity / intensity /
 * duration as xan_drought_stats when all three are given, skipped when all three are null.  With d_count and
 * d_summary (both or neither): d_count[t][c] += (hydro < threshold) for every month (int32 [nmonths][ld], the
 * members in drought so far), and d_summary[4][ld] = the member's drought months (D > 0).sum(0), events
 * (D == 1).sum(0), longest duration D.max(0) and peak severity S.max(0) (NaN if any severity is NaN, like
 * np.max).  At least one of the two groups is required. */
int xan_drought_scan(const double *d_hydro, const double *d_thresh, int ncell, int nmonths, int ld, int nthresh,
                     int ld_thresh, double *d_severity, double *d_intensity, double *d_duration, int *d_count,
                     double *d_summary, void *stream);
/* DroughtStats.getthresh (drought_stats.py:150-171): numpy.percentile(..., method "linear") over the
 * ntime / nper samples of every (period, cell); the caller passes numpy's virtual index
 * ((n - 1) q, split into floor and fraction).  d_out [nper][ld_out]. */
int xan_drought_thresholds(const double *d_hist, int ncell, int ntime, int ld, int nper,
                           int prev_index, double gamma, double *d_out, int ld_out, void *stream);
/* Aggregation_Map (xanthos/diagnostics/time_series.py:126-138) / basin aggregation of
 * AccessibleWater (xanthos/accessible/accessible.py:41-51): out[g][t] = sum over the cells of group g
 * in ascending cell index of the non-NaN src[t][cell].  d_order = cells sorted (stable) by group,
 * d_offsets [ngroups + 1] = group boundaries in d_order; cells with id <= 0 are left out by the
 * caller.  d_out is [ngroups][ntime] (the reference's orientation). */
int xan_group_sum(const double *d_src, const int *d_order, const int *d_offsets, int ngroups,
                  int ntime, int ld, double *d_out, void *stream);
/* accessible.py:34-39: dst[y][c] = numpy.sum(src[12 y .. 12 y + 11][c]) * scale[c] (scale may be
 * NULL); a trailing partial year is dropped like int(nmonths / 12). */
int xan_year_sum_scaled(const double *d_src, const double *d_scale, int ncell, int nmonths, int ld,
                        double *d_dst, void *stream);

/* ---- differential evolution on the device (SURVEY.md section 8 row f4) ----------------------- */
/* The generation logic of scipy.optimize.differential_evolution as calibrate_abcd.py:103-110 uses
 * it (best1bin, Latin-hypercube init, dither, binomial crossover with one forced gene, out-of-bounds
 * genes redrawn, deferred updating, convergence std(E) <= atol + tol |mean(E)|) for many independent
 * problems in lock step.  d_pop [n_problems][pop_size][n_dims] holds scaled vectors in [0, 1],
 * d_energy [n_problems][pop_size]; d_active [n_active] lists the problems a call works on (trial
 * arrays are compact: [n_active][pop_size][...]).  Random numbers are Philox4x32-10 keyed by `seed`
 * and indexed by (generation, problem, member): reproducible for any launch geometry.
 *   xan_de_init    Latin hypercube
 *   xan_de_trial   trial vectors of generation `generation` (>= 1): scaled (d_trial_x) and in parameter
 *                  units lo + x * span with n_par_cols >= n_dims columns, the extra ones 0 (d_trial_par -
 *                  what xan_abcd_kge_batch takes)
 *   xan_de_select  keep trial where its energy <= the member's (NaN = +inf), then the convergence test:
 *                  d_converged[problem] = generation at which it first held (-1: already at
 *                  initialisation; 0: not yet); converged problems are frozen.  d_trial_x == NULL:
 *                  only the test. */
int xan_de_init(double *d_pop, int n_problems, int pop_size, int n_dims, unsigned long long seed,
                void *stream);
int xan_de_trial(const double *d_pop, const double *d_energy, const int *d_active, int n_active,
                 int pop_size, int n_dims, int n_par_cols, const double *d_lo, const double *d_span,
                 unsigned long long seed, int generation, double mutation_lo, double mutation_hi,
                 double recombination, double *d_trial_x, double *d_trial_par, void *stream);
int xan_de_select(double *d_pop, double *d_energy, const int *d_active, int n_active, int pop_size,
                  int n_dims, const double *d_trial_x, const double *d_trial_energy, double tol,
                  double atol, int generation, int *d_converged, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* XANTHOS_B200_H */
