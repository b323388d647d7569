/*
 * ufair.h -- C ABI of libufair.so, the B200 (sm_100a) ensemble integrator for
 * the 5-equation Universal-FaIR model.
 *
 * What this replaces in the reference (stujen/fiveEqSCM):
 *   - U_FaIR/concentrations.py:4-5  `calculate_hfc_conc(emissions, time, lifetime)`
 *     -> ufair_hfc_pulse_f64()   (bit-for-bit the same expression, batched)
 *   - the functions the reference only NAMES (.coveragerc:12-19):
 *       step_conc, step_forc, step_temp, g_1, g_0, alpha_val, k_q, oxfair
 *     -> ufair_run_f64()/ufair_run_f32() (oxfair = the driver loop; the step_*
 *        functions are fused inside one kernel launch), ufair_g1g0_f64()
 *        (g_1, g_0) and ufair_kq_f64() (k_q).
 * The reference has no FFI of its own (it is 3 lines of numpy); the binding a
 * maintainer would add is the ctypes stub shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain C, no torch types. All pointers are DEVICE pointers unless the
 *     entry point says "host". The library never allocates or frees memory the
 *     caller can see; ufair_run_host_* keeps private staging buffers inside an
 *     opaque workspace.
 *   - every [..][member] array has the member axis fastest, with one common row
 *     pitch `ld_member` (elements). Time is the axis above it
 *     (reference: time is axis 0 of `emissions`, U_FaIR/concentrations.py:5).
 *   - rows must be 16-byte aligned: base pointers 16-B aligned and ld_member a
 *     multiple of 2 (f64) / 4 (f32). Violations return UFAIR_ERR_ALIGN -- the
 *     kernel streams emission rows with TMA bulk copies.  The rule is on the
 *     run's element size also with float32 outputs (out_type below), whose rows
 *     are then only 8-byte aligned; nothing that reads or writes them needs more.
 *   - every entry point returns 0 on success or a negative UFAIR_ERR_*;
 *     ufair_last_error() gives the message (thread-local). Nothing aborts.
 *   - `stream` is a cudaStream_t passed as void*. Calls are asynchronous on it.
 *
 * The same descriptor drives the CPU oracle (oracle/ufair_oracle.c) with host
 * pointers; that is test infrastructure, not part of this library.
 */
#ifndef UFAIR_H_
#define UFAIR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UFAIR_ABI_VERSION 5

#define UFAIR_MAX_GAS 4
#define UFAIR_N_POOL 4
#define UFAIR_MAX_STAT_GROUPS 256 /* cap of ufair_desc.n_stat_groups */

/* rows of gas_params[n_gas][UFAIR_GP_COUNT][ld_member] */
enum {
  UFAIR_GP_A0 = 0,   /* pool fractions a_1..a_4                       */
  UFAIR_GP_TAU0 = 4, /* pool lifetimes tau_1..tau_4 (yr)              */
  UFAIR_GP_R0 = 8,   /* iIRF100 = r0 + rU*G_u + rT*T + rA*G_a         */
  UFAIR_GP_RU = 9,
  UFAIR_GP_RT = 10,
  UFAIR_GP_RA = 11,
  UFAIR_GP_C0 = 12,  /* pre-industrial concentration                  */
  UFAIR_GP_EMIS2CONC = 13, /* c: emission unit -> concentration unit */
  UFAIR_GP_F1 = 14,  /* F = f1 ln(C/C0) + f2 (C-C0) + f3 (sqrt C - sqrt C0) */
  UFAIR_GP_F2 = 15,
  UFAIR_GP_F3 = 16,
  UFAIR_GP_COUNT = 17
};

/* rows of thermal_params[UFAIR_TP_COUNT][ld_member] */
enum { UFAIR_TP_Q1 = 0, UFAIR_TP_Q2 = 1, UFAIR_TP_D1 = 2, UFAIR_TP_D2 = 3, UFAIR_TP_COUNT = 4 };

/* rows of state_in/state_out[UFAIR_STATE_ROWS(n_gas)][ld_member]:
 *   per gas g: rows 5g..5g+3 = pools R_1..R_4 (concentration units above C0),
 *              row  5g+4     = cumulative emissions G_cum
 *   then S_1, S_2 (thermal boxes, K) and T_prev (the T the next alpha sees). */
#define UFAIR_STATE_ROWS(n_gas) (5 * (n_gas) + 3)

enum { UFAIR_E_MEMBER = 0,    /* emissions[n_gas][n_t][ld_member]                   */
       UFAIR_E_SCENARIO = 1   /* emissions[n_gas][n_t][n_scen] + scen_idx (+e_scale) */ };
enum { UFAIR_FEXT_NONE = 0,
       UFAIR_FEXT_SCENARIO = 1, /* f_ext[n_t][n_scen] (n_scen==1, scen_idx NULL: shared) */
       UFAIR_FEXT_MEMBER = 2    /* f_ext[n_t][ld_member]                                 */ };
enum { UFAIR_ALPHA_EXP = 0,    /* alpha = g0 * exp(iIRF/g1)      (the "derived functional form") */
       UFAIR_ALPHA_SINH = 1,   /* alpha = g0 * sinh(iIRF/g1), g0 = 1/sinh(.)                     */
       UFAIR_ALPHA_NEWTON = 2, /* EXP seed + newton_iters Newton steps on iIRF100(alpha)=iIRF    */
       UFAIR_ALPHA_ONE = 3     /* alpha == 1: no state dependence (HFC-style fixed lifetime)     */ };
enum { UFAIR_T_MID = 0,  /* T = sum_j (S_j + S_j')/2 */
       UFAIR_T_END = 1   /* T = sum_j S_j'           */ };
enum { UFAIR_OUT_C = 1, UFAIR_OUT_RF = 2, UFAIR_OUT_T = 4, UFAIR_OUT_ALPHA = 8, UFAIR_OUT_E = 16 };

/* out_type: the element type of out_C, out_RF and out_T.
 *   UFAIR_OUTTYPE_RUN (0, the default): the run's precision, as ufair_run_f64 / ufair_run_f32 say.
 *   UFAIR_OUTTYPE_F32 (1): float32.  The integration stays in the run's precision; with ufair_run_f64 every
 *     element of out_C, out_RF and out_T is the round-to-nearest-even float32 (cvt.rn.f32.f64) of the double
 *     the same descriptor stores with UFAIR_OUTTYPE_RUN -- bit for bit, period means (out_every >= 2) included:
 *     their sum and their product with (Real)(1.0 / k) stay in FP64, and the mean is rounded once, at the store.
 *     Half the bytes cross HBM and the host link, and the outputs take half the device memory.
 *     state_out stays in the run's precision, so a run split into time chunks gives the float32 rows of one call.
 *     The statistics (stats == 1) bin the T rows the integrator stored: here float32 T, with ufair_stats_pass_f64
 *     running the FP32 pass -- FP32 binning rule, FP64 moments of the float32 values.  The histogram is thus a
 *     recount of the stored float32 T, not of the FP64 T: a member within about 1e-7 relative of a bin edge can
 *     land in the neighbouring bin.  A statistics-only call (stats == 1 without UFAIR_OUT_T) needs a float32
 *     out_T scratch of n_out rows.
 *     Not supported (UFAIR_ERR_UNSUPPORTED) with ufair_run_f64: the UFAIR_OUT_ALPHA and UFAIR_OUT_E diagnostics
 *     and concentration-driven gases (conc_driven != 0).  With ufair_run_f32 it is accepted and changes nothing.
 *   Any other value: UFAIR_ERR_ARG.  No combination widens the outputs. */
enum { UFAIR_OUTTYPE_RUN = 0, UFAIR_OUTTYPE_F32 = 1 };

/* gas_form[g]: what gas g actually uses, so that the library may pick a kernel that skips the rest.
 * 0 = unspecified (four pools, all three forcing terms).  Otherwise UFAIR_FORM(n_pool, terms):
 * only pools 1..n_pool carry mass (a_i == 0 and zero initial state for the others) and only the
 * forcing terms in `terms` have non-zero coefficients -- for EVERY member of the call.  It is a
 * promise by the caller (ufair_detect_form_* derives it from the parameter arrays); results are
 * those of the unspecialised kernel.  One-pool gases are the reference's own case
 * (U_FaIR/concentrations.py:4-5 is a single box). */
enum { UFAIR_TERM_LOG = 1, UFAIR_TERM_LIN = 2, UFAIR_TERM_SQRT = 4 };
#define UFAIR_FORM(n_pool, terms) ((uint8_t)((n_pool) | ((terms) << 4)))

/* moments_private / moments rows */
enum { UFAIR_MOM_SUM = 0, UFAIR_MOM_SUMSQ = 1, UFAIR_MOM_MIN = 2, UFAIR_MOM_MAX = 3, UFAIR_MOM_COUNT = 4 };

enum {
  UFAIR_OK = 0,
  UFAIR_ERR_ARG = -1,    /* bad dims / mode / NULL where required */
  UFAIR_ERR_ALIGN = -2,  /* pointer or ld_member alignment        */
  UFAIR_ERR_CUDA = -3,   /* a CUDA runtime call failed            */
  UFAIR_ERR_UNSUPPORTED = -4,
  UFAIR_ERR_NOMEM = -5
};

typedef struct ufair_desc {
  uint32_t struct_size; /* = sizeof(ufair_desc); checked */
  int32_t out_type;     /* UFAIR_OUTTYPE_*: element type of out_C / out_RF / out_T (see above) */

  /* ---- dimensions ---- */
  int32_t n_gas;     /* 1..UFAIR_MAX_GAS */
  int32_t n_t;       /* time steps in this call */
  int64_t n_member;  /* members in this call */
  int64_t ld_member; /* row pitch (elements) of every [..][member] array */
  int32_t n_scen;    /* columns of scenario-shared arrays (>=1) */

  /* ---- modes ---- */
  int32_t e_mode;       /* UFAIR_E_* */
  int32_t fext_mode;    /* UFAIR_FEXT_* */
  int32_t alpha_mode;   /* UFAIR_ALPHA_* */
  int32_t newton_iters; /* UFAIR_ALPHA_NEWTON only, 0..8 */
  int32_t t_mode;       /* UFAIR_T_* */
  int32_t out_mask;     /* UFAIR_OUT_* bits; outputs not selected may be NULL */
  int32_t stats;        /* 0 = none, 1 = per-output-row T histogram + moments */

  double dt;       /* step length (yr) */
  double iirf_h;   /* iIRF horizon, 100 */
  double iirf_max; /* clamp iIRF <= iirf_max; <= 0 or inf disables */

  /* ---- inputs ---- */
  const void* emissions;      /* see e_mode; emission RATE during each step */
  const int32_t* scen_idx;    /* [n_member] or NULL (all members use column 0) */
  const void* e_scale;        /* [n_gas][ld_member] or NULL; UFAIR_E_SCENARIO only */
  const void* f_ext;          /* see fext_mode */
  const void* gas_params;     /* [n_gas][UFAIR_GP_COUNT][ld_member] */
  const void* thermal_params; /* [UFAIR_TP_COUNT][ld_member] */
  const void* state_in;       /* [UFAIR_STATE_ROWS][ld_member] or NULL (= all zero) */

  /* ---- outputs ---- */
  void* out_C;     /* [n_gas][n_out][ld_member]; n_out = n_t, or n_t / out_every (period means below); out_type */
  void* out_RF;    /* [n_gas][n_out][ld_member]; out_type */
  void* out_T;     /* [n_out][ld_member]; out_type */
  void* out_alpha; /* [n_gas][n_t][ld_member] (diagnostic) */
  void* state_out; /* [UFAIR_STATE_ROWS][ld_member] or NULL; always the run's precision */

  /* ---- ensemble statistics (stats == 1) ----
   * bin(T) = clamp(floor((T - hist_lo) * (hist_bins / (hist_hi - hist_lo))), 0, hist_bins-1),
   * evaluated in the precision of the stored T rows: the run's, or float32 with UFAIR_OUTTYPE_F32.  Non-finite T: NaN is neither counted in the histogram nor
   * taken into min / max, but it makes its row's sum and sum of squares NaN (a mean / std computed
   * from them flags the step); +inf and -inf are counted in the last and first bin and enter every
   * moment.  A row with no value other than NaN keeps the min / max sentinels +inf / -inf.
   * The integrator only writes the T rows (so out_T must be non-NULL when stats == 1, whether or
   * not UFAIR_OUT_T is set); ufair_stats_pass_*() then reads them once at HBM speed and adds member
   * slice c of every row into copy c of hist_private / moments_private (counts; sum, sum of
   * squares, min, max) in a fixed order.  ufair_stats_reset() initialises the private buffers
   * once; they may keep accumulating over several run + pass pairs (member chunks);
   * ufair_stats_finalize() folds the copies.
   *
   * Grouped statistics (n_stat_groups, stat_group at the end of the struct): with stat_group != NULL
   * every member m carries a label, and the pass builds one histogram and one set of moments per
   * group.  Let G = max(1, n_stat_groups):
   *   0 <= stat_group[m] < G  member m is counted in group stat_group[m];
   *   stat_group[m] < 0       member m is counted nowhere (neither histogram nor moments);
   *   stat_group[m] >= G      not counted either (the library does not check labels: that would
   *                           need a synchronise; the Python layer rejects them).
   * stat_group may be the scen_idx pointer itself: per-scenario statistics.  Group g, step t lives in
   * row g * hist_rows + hist_t0 + t, so every statistics buffer has G times the rows:
   *   hist_private[hist_copies][G * hist_rows][hist_bins], moments_private[hist_copies][G * hist_rows][4],
   *   and the finalised hist / moments (and the packed sums / ext) [G][hist_rows][..].
   * With stat_group == NULL (n_stat_groups 0 or 1) the pass is the pooled one, unchanged.
   * The binning rule and the NaN handling are those of the pooled pass; counts are exact and the
   * moments deterministic (fixed order, no floating-point atomics); one group with every label 0
   * gives the pooled pass's histogram and moments bit for bit.  Memory: the private histogram is
   * G times the pooled one (16 copies x 4 groups x 736 steps x 1024 bins x 4 B = 193 MB); fewer
   * hist_copies reduce it.  Measured on a B200 (1000 W), T of 1.25e6 members x 736 steps f64: pooled 1.37 ms,
   * 4 scenario groups 4.59 ms, 16 random groups 23.7 ms (DESIGN.md 4.2). */
  int32_t hist_bins;
  int32_t hist_copies;
  double hist_lo, hist_hi;
  int32_t hist_t0;          /* row offset: output row t of this call lands in row hist_t0 + t */
  int32_t hist_rows;        /* rows allocated per copy (>= hist_t0 + n_out) */
  uint32_t* hist_private;   /* [hist_copies][hist_rows][hist_bins] */
  double* moments_private;  /* [hist_copies][hist_rows][UFAIR_MOM_COUNT]: member slice c of every
                               row is folded into copy c, in a fixed order (deterministic) */

  /* ---- optional per-gas specialisation (see UFAIR_FORM) ---- */
  uint8_t gas_form[UFAIR_MAX_GAS];

  /* ---- concentration-driven gases (the inverse of step_conc) ----
   * bit g set: rows emissions[g][..] hold the CONCENTRATION gas g must have at the end of each step;
   * the integrator diagnoses the emission rate that produces it -- step_conc is linear in E:
   *   E = (C_target - C0 - sum_i R_i (1 - m_i)) / (c sum_i a_i alpha tau_i m_i)
   * -- and carries on with it (pools, G_cum, forcing, temperature).  out_E (UFAIR_OUT_E) receives
   * the emission rate of every gas: diagnosed where the bit is set, the input otherwise. */
  int32_t conc_driven;
  void* out_E; /* [n_gas][n_t][ld_member] */

  /* ---- grouped statistics (see the statistics block above; stats == 1 only) ---- */
  int32_t n_stat_groups;      /* 0 or 1 = pooled; up to UFAIR_MAX_STAT_GROUPS */

  /* ---- period means ----
   * out_every = k: 0 or 1 writes one row of C, RF and T per step (n_out = n_t).  k >= 2 writes one row per
   * period of k steps instead: n_t must be a multiple of k (else UFAIR_ERR_ARG), n_out = n_t / k, and row p of
   * out_C, out_RF ([n_gas][n_out][ld_member]) and out_T ([n_out][ld_member]) is the mean of that output over
   * steps p k .. p k + k - 1, defined bit for bit as
   *   s = 0;  s = s + x_t for t = p k .. p k + k - 1 in step order (the run's precision);  mean = s * (Real)(1.0 / k)
   * with no contraction into FMAs.  Inputs (emissions, f_ext) stay per step; state_out is the state at the end
   * of the call.  A run split into calls of whole periods (state_in / state_out) gives the rows of one call.
   * The statistics bin the period-mean T rows: hist_t0 counts output rows and hist_rows >= hist_t0 + n_out.
   * With k >= 2 the diagnostics UFAIR_OUT_ALPHA and UFAIR_OUT_E and concentration-driven gases
   * (conc_driven != 0) are not supported: UFAIR_ERR_UNSUPPORTED. */
  int32_t out_every;
  const int32_t* stat_group;  /* [n_member] group labels, or NULL */
} ufair_desc;

/* ---- version / errors ---- */
int ufair_abi_version(void);
const char* ufair_last_error(void);

/* Members per CTA of the integrator (informational: chunk sizes that are a multiple of it
 * waste no lanes; the run functions accept any n_member). */
int64_t ufair_block_members(void);

/* ---- the hot path: oxfair (driver loop) with step_conc/alpha_val/step_forc/step_temp fused ---- */
int ufair_run_f64(const ufair_desc* d, void* stream);
int ufair_run_f32(const ufair_desc* d, void* stream);

/* Derive gas_form from the descriptor's DEVICE parameter arrays (gas_params, state_in): scans every
 * member, writes n_gas bytes to the HOST array `form` and synchronises `stream`.
 * `scratch` is a device buffer of at least UFAIR_MAX_GAS int32. */
int ufair_detect_form_f64(const ufair_desc* d, int32_t* scratch, uint8_t* form, void* stream);
int ufair_detect_form_f32(const ufair_desc* d, int32_t* scratch, uint8_t* form, void* stream);

/* Which integrator variant ufair_run_* launches for this descriptor (informational / tests):
 * *form = the specialised per-gas form in use, packed one UFAIR_FORM byte per gas (0 = the general
 * kernel), *gases_per_lane and *members_per_warp = the lane mapping, *loop = UFAIR_LOOP_*: which
 * instantiation of the time loop (all of them give bit-identical results; the plain ones carry no
 * run-time switches for features that are off).  elem_size: 8 (f64) or 4 (f32).  Out-pointers may be NULL.
 * Float32 outputs of an FP64 run (UFAIR_OUTTYPE_F32) always run all gases per lane. */
enum { UFAIR_LOOP_GENERAL = 0,      /* every run-time option                                         */
       UFAIR_LOOP_CONC_DRIVEN = 1,  /* concentration-driven gases / emissions output                 */
       UFAIR_LOOP_PLAIN = 2,        /* no f_ext, no iIRF ceiling, outputs exactly C + RF + T         */
       UFAIR_LOOP_PLAIN_FEXT = 3,   /* the same with external forcing (default alpha mode)           */
       UFAIR_LOOP_PLAIN_SUBSET = 4, /* a subset of C, RF, T (e.g. T + statistics only), with or
                                       without external forcing (default alpha mode)                */
       UFAIR_LOOP_PERIOD_MEAN = 5   /* out_every >= 2: period means of C, RF, T (every alpha mode)   */ };
int ufair_kernel_variant(const ufair_desc* d, int32_t elem_size, uint32_t* form, int32_t* gases_per_lane,
                         int32_t* members_per_warp, int32_t* loop);

/* Zero (and initialise the min/max sentinels of) the private statistics buffers. */
int ufair_stats_reset(const ufair_desc* d, void* stream);
/* The statistics pass: per-row histogram and moments of the T rows ufair_run_* just wrote
 * (d->out_T, n_out rows: per step, or per period with out_every >= 2; same descriptor, same stream).
 * One call per ufair_run_* call when stats == 1.  The _f64 / _f32 suffix names the run's precision; the
 * rows are read in the descriptor's out_type (float32 rows of an FP64 run take the FP32 pass). */
int ufair_stats_pass_f64(const ufair_desc* d, void* stream);
int ufair_stats_pass_f32(const ufair_desc* d, void* stream);
/* Fold the private copies: hist[G][hist_rows][hist_bins] (uint64 counts) and
 * moments[G][hist_rows][UFAIR_MOM_COUNT] (sum, sumsq, min, max as doubles); G = max(1, n_stat_groups).
 * Here and in ufair_stats_finalize_packed, "hist_rows" below stands for G * hist_rows. */
int ufair_stats_finalize(const ufair_desc* d, uint64_t* hist, double* moments, void* stream);

/* The same fold in the layout the cross-GPU reduction uses -- two buffers, two collectives:
 *   sums[hist_rows][hist_bins + 2]: the counts as doubles (integers below 2^53 add exactly in any order,
 *     so the reduced histogram is bitwise independent of the GPU count), then sum T and sum T^2 -> all-reduce SUM
 *   ext[hist_rows][2]: max T, -min T                                                            -> all-reduce MAX
 * and back: ufair_stats_unpack() turns the reduced buffers into hist (uint64) and moments. */
int ufair_stats_finalize_packed(const ufair_desc* d, double* sums, double* ext, void* stream);
int ufair_stats_unpack(const double* sums, const double* ext, int32_t rows, int32_t bins, uint64_t* hist,
                       double* moments, void* stream);

/* Percentiles read off the (reduced) per-step histogram CDF, linear inside the bin:
 * out[row][j] = percentile pcts[j] (0..100) of row `row`; hist: [rows][bins] counts, pcts: [n_pct]
 * (device), out: [rows][n_pct] (device).  Bit-identical to the oracle's percentiles_from_hist. */
int ufair_hist_percentiles(const uint64_t* hist, int32_t rows, int32_t bins, double lo, double hi,
                           const double* pcts, int32_t n_pct, double* out, void* stream);

/* ---- parameter preparation (g_1, g_0, k_q in the reference's naming) ---- */
/* a, tau: [4][ld]; out g1, g0: [ld]. alpha_mode selects the g0 form (EXP/NEWTON vs SINH). */
int ufair_g1g0_f64(const double* a, const double* tau, int64_t n_member, int64_t ld_member,
                   double iirf_h, int32_t alpha_mode, double* g1, double* g0, void* stream);
/* tcr, ecs, d1, d2: [n]; out q1, q2: [n]. */
int ufair_kq_f64(const double* tcr, const double* ecs, const double* d1, const double* d2,
                 double f2x, int64_t n_member, double* q1, double* q2, void* stream);

/* ---- on-device ensemble sampler (SURVEY 8f-3: parameter / scenario sampling next to the path) ----
 * Fills gas_params, thermal_params, e_scale and scen_idx for members first_member ..
 * first_member + n_member - 1 of the ensemble that (sampler, seed) defines.  A member's values
 * depend only on the seed and its GLOBAL index, so any split of the member axis over calls or GPUs
 * yields the same ensemble, bit for bit.
 *
 * Random stream (counter-based, Philox4x32-10 of Salmon et al. 2011; key = seed low, seed high;
 * counter = member low, member high, block, 0x55464152):  the four output words x0..x3 give
 *   u_a = (((x1 << 32 | x0) >> 11) + 0.5) 2^-53,  u_b likewise from x3, x2          (both in (0, 1))
 *   z_even = sqrt(-2 ln u_a) cos(2 pi u_b),  z_odd = sqrt(-2 ln u_a) sin(2 pi u_b)  (Box-Muller)
 * and slot s of a member is z_{s & 1} of block s >> 1.  Slots: gas g row r -> 18 g + r;
 * e_scale[g] -> 18 g + 17; thermal row k -> 72 + k; scen_idx = (x0 of block 38 * n_scen) >> 32.
 * A row with distribution UFAIR_DIST_LOGNORMAL is base * exp(sigma z), UFAIR_DIST_NORMAL is
 * base * (1 + sigma z), UFAIR_DIST_FIXED is base; the four pool fractions of a gas are then
 * renormalised to sum 1; e_scale = 1 + e_scale_sigma z.  Everything is evaluated in double; the
 * _f32 entry point rounds once on store.  Output pointers may be NULL (that array is skipped). */
enum { UFAIR_DIST_FIXED = 0, UFAIR_DIST_LOGNORMAL = 1, UFAIR_DIST_NORMAL = 2 };

typedef struct ufair_sampler {
  uint32_t struct_size; /* = sizeof(ufair_sampler); checked */
  int32_t n_gas;
  uint64_t seed;
  int32_t n_scen;       /* scen_idx in [0, n_scen) */
  int32_t reserved;
  double e_scale_sigma;
  double gas_base[UFAIR_MAX_GAS][UFAIR_GP_COUNT];
  double gas_sigma[UFAIR_MAX_GAS][UFAIR_GP_COUNT];
  double thermal_base[UFAIR_TP_COUNT];
  double thermal_sigma[UFAIR_TP_COUNT];
  uint8_t gas_dist[UFAIR_MAX_GAS][24]; /* UFAIR_DIST_* per row (first UFAIR_GP_COUNT entries used) */
  uint8_t thermal_dist[8];             /* first UFAIR_TP_COUNT entries used */
} ufair_sampler;

int ufair_sample_f64(const ufair_sampler* s, int64_t first_member, int64_t n_member, int64_t ld_member,
                     double* gas_params, double* thermal_params, double* e_scale, int32_t* scen_idx,
                     void* stream);
int ufair_sample_f32(const ufair_sampler* s, int64_t first_member, int64_t n_member, int64_t ld_member,
                     float* gas_params, float* thermal_params, float* e_scale, int32_t* scen_idx,
                     void* stream);

/* ---- the one function the reference ships (U_FaIR/concentrations.py:4-5) ----
 * out[i] = e0[i] * exp(-time[i]) over n already-broadcast elements. */
int ufair_hfc_pulse_f64(const double* e0, const double* time, double* out, int64_t n, void* stream);

/* ---- host-buffer pipeline (HOST pointers inside `d`, same meaning otherwise) ----
 * Splits the member axis into chunks, and overlaps H2D copies, the kernel and
 * D2H copies on three streams with double-buffered device staging.
 * Statistics, when requested, are finalised into host `hist`/`moments`. */
typedef struct ufair_workspace ufair_workspace;
int ufair_workspace_create(int device, int64_t chunk_members, ufair_workspace** ws);
int ufair_workspace_destroy(ufair_workspace* ws);
int ufair_run_host_f64(ufair_workspace* ws, const ufair_desc* d, uint64_t* hist, double* moments);
int ufair_run_host_f32(ufair_workspace* ws, const ufair_desc* d, uint64_t* hist, double* moments);

/* ---- host-link probe (measurement support: the ceiling bench.py states e2e against) ----
 * Times `reps` rounds of copies between a page-locked host buffer (allocated and kept by the probe) and
 * device memory on `device`: bytes_up bytes host -> device and bytes_down bytes device -> host per round,
 * the two directions at once on two streams (either may be 0: that direction alone).  rows <= 1:
 * contiguous cudaMemcpyAsync; rows > 1: one pitched cudaMemcpy2DAsync of `rows` rows per copy (host pitch =
 * twice the row width: the shape of a member-chunk copy).  Wall clock from the first enqueue to each
 * stream's completion: gbs[0] = host -> device GB/s, gbs[1] = device -> host GB/s, *seconds (may be NULL)
 * = until both are done.  bytes_up <= 0 and bytes_down <= 0 releases the probe's buffers. */
int ufair_link_probe(int device, int64_t bytes_up, int64_t bytes_down, int32_t rows, int32_t reps, double* gbs,
                     double* seconds);

/* ---- device-math probe (test support): y[i] = op(x[i]) with the kernel's own math routines.
 * op: 0 decay(x)=1-exp(-x), 1 exp, 2 rcp, 3 sqrt, 4 log, 5 sinh. */
int ufair_math_probe_f64(int op, const double* x, double* y, int64_t n, void* stream);
int ufair_math_probe_f32(int op, const float* x, float* y, int64_t n, void* stream);

/* ---- measured-peak microbenchmarks used by bench.py for the roofline denominators ---- */
/* Runs `iters` dependent-chain DFMA (or FFMA / MUFU.EX2) per thread over a full grid and
 * returns the elapsed milliseconds and the operation count through the out-params. */
int ufair_peak_fp64(int iters, double* ms, double* flops, void* stream);
int ufair_peak_fp32(int iters, double* ms, double* flops, void* stream);
int ufair_peak_mufu(int iters, double* ms, double* ops, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UFAIR_H_ */
