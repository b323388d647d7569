// ufair_abi.cu -- extern "C" entry points of libufair.so (include/ufair.h): argument checking,
// dispatch to the fused integrator instantiations, and the small kernels either side of it
// (statistics reset/finalise, g_1/g_0, k_q, the reference's one-box pulse, peak microbenchmarks).
#include <stdlib.h>
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>

#include "../../include/ufair.h"
#include "ufair_internal.h"
#include "ufair_kernel.cuh"

namespace ufair {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int cuda_error(cudaError_t e, const char* what) {
  return set_error(UFAIR_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

// ---- descriptor validation ---------------------------------------------------------------------
static bool misaligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }

// the grouped-statistics fields (shared by the run / pass validation and the statistics-buffer entry points)
static int check_stat_groups(const ufair_desc* d) {
  if (d->n_stat_groups < 0 || d->n_stat_groups > UFAIR_MAX_STAT_GROUPS)
    return set_error(UFAIR_ERR_ARG, "n_stat_groups %d outside 0..%d", d->n_stat_groups, UFAIR_MAX_STAT_GROUPS);
  if (d->n_stat_groups > 1 && !d->stat_group)
    return set_error(UFAIR_ERR_ARG, "n_stat_groups %d needs stat_group labels (NULL)", d->n_stat_groups);
  if (d->stat_group && !d->stats) return set_error(UFAIR_ERR_ARG, "stat_group set but stats == 0");
  if ((int64_t)stat_groups(d) * d->hist_rows > (int64_t)INT32_MAX)
    return set_error(UFAIR_ERR_ARG, "n_stat_groups %d x hist_rows %d rows do not fit in 32 bits", d->n_stat_groups,
                     d->hist_rows);
  return UFAIR_OK;
}

// period means (out_every, include/ufair.h): the step count, and what the mean loop does not support
static int check_out_every(const ufair_desc* d) {
  if (d->out_every < 0) return set_error(UFAIR_ERR_ARG, "out_every %d < 0", d->out_every);
  if (d->out_every < 2) return UFAIR_OK;
  if (d->n_t % d->out_every != 0)
    return set_error(UFAIR_ERR_ARG, "n_t %d is not a multiple of out_every %d", d->n_t, d->out_every);
  if (d->out_mask & (UFAIR_OUT_ALPHA | UFAIR_OUT_E))
    return set_error(UFAIR_ERR_UNSUPPORTED, "out_every %d: the alpha and emissions outputs are per step only", d->out_every);
  if (d->conc_driven != 0)
    return set_error(UFAIR_ERR_UNSUPPORTED, "out_every %d: concentration-driven gases are not supported", d->out_every);
  return UFAIR_OK;
}

// the outputs' element type (out_type, include/ufair.h), and what float32 outputs of an FP64 run do not support
static int check_out_type(const ufair_desc* d, size_t elem) {
  if (d->out_type != UFAIR_OUTTYPE_RUN && d->out_type != UFAIR_OUTTYPE_F32)
    return set_error(UFAIR_ERR_ARG, "out_type %d is not UFAIR_OUTTYPE_RUN (0) or UFAIR_OUTTYPE_F32 (1)", d->out_type);
  if (out_elem(d, elem) == elem) return UFAIR_OK;
  if (d->out_mask & (UFAIR_OUT_ALPHA | UFAIR_OUT_E))
    return set_error(UFAIR_ERR_UNSUPPORTED, "float32 outputs: the alpha and emissions outputs are in the run's precision only");
  if (d->conc_driven != 0)
    return set_error(UFAIR_ERR_UNSUPPORTED, "float32 outputs: concentration-driven gases are not supported");
  return UFAIR_OK;
}

// the private statistics buffers: what the statistics pass adds into, and what ufair_stats_reset / _finalize /
// _finalize_packed work on
static int check_stat_buffers(const ufair_desc* d) {
  if (d->hist_copies < 1 || !d->hist_private || !d->moments_private)
    return set_error(UFAIR_ERR_ARG, "stats requested but histogram spec/buffers incomplete");
  return UFAIR_OK;
}

// The run rules say what the caller asked for; they hold for host and device arrays alike.  The placement rules
// (placement == true) say how device arrays must be laid out for this library's kernels: the 16-byte rows of the TMA
// bulk copies, and the statistics buffers, row offset and T rows of the statistics pass.  The pitch rule comes before
// the other run rules, so that misaligned rows are reported before missing arrays.
static int check_desc(const ufair_desc* d, size_t elem, bool placement) {
  if (!d) return set_error(UFAIR_ERR_ARG, "descriptor is NULL");
  if (d->struct_size != sizeof(ufair_desc))
    return set_error(UFAIR_ERR_ARG, "struct_size %u != sizeof(ufair_desc) %zu (header/binding mismatch)",
                     d->struct_size, sizeof(ufair_desc));
  if (d->n_gas < 1 || d->n_gas > UFAIR_MAX_GAS)
    return set_error(UFAIR_ERR_ARG, "n_gas %d outside 1..%d", d->n_gas, UFAIR_MAX_GAS);
  if (d->n_t < 0 || d->n_member < 0) return set_error(UFAIR_ERR_ARG, "negative n_t / n_member");
  if (d->ld_member < d->n_member) return set_error(UFAIR_ERR_ARG, "ld_member < n_member");
  // TMA box coordinates and the warp index arithmetic are 32-bit: one launch takes at most 2^31 - 1 members per row
  if (d->ld_member > (int64_t)INT32_MAX)
    return set_error(UFAIR_ERR_ARG, "ld_member %lld > %d: split the member axis over several calls", (long long)d->ld_member,
                     INT32_MAX);
  if (placement && d->n_member > 0 && (d->ld_member * (int64_t)elem) % 16 != 0)
    return set_error(UFAIR_ERR_ALIGN, "ld_member %lld: rows must be a multiple of 16 bytes", (long long)d->ld_member);
  if (d->e_mode != UFAIR_E_MEMBER && d->e_mode != UFAIR_E_SCENARIO) return set_error(UFAIR_ERR_ARG, "bad e_mode");
  if (d->fext_mode < UFAIR_FEXT_NONE || d->fext_mode > UFAIR_FEXT_MEMBER) return set_error(UFAIR_ERR_ARG, "bad fext_mode");
  if (d->alpha_mode < UFAIR_ALPHA_EXP || d->alpha_mode > UFAIR_ALPHA_ONE) return set_error(UFAIR_ERR_ARG, "bad alpha_mode");
  if (d->t_mode != UFAIR_T_MID && d->t_mode != UFAIR_T_END) return set_error(UFAIR_ERR_ARG, "bad t_mode");
  if (d->alpha_mode == UFAIR_ALPHA_NEWTON && (d->newton_iters < 0 || d->newton_iters > 8))
    return set_error(UFAIR_ERR_ARG, "newton_iters %d outside 0..8", d->newton_iters);
  if (d->n_scen < 1) return set_error(UFAIR_ERR_ARG, "n_scen must be >= 1");
  if (!(d->dt > 0.0) || !(d->iirf_h > 0.0)) return set_error(UFAIR_ERR_ARG, "dt and iirf_h must be > 0");
  int rc = check_stat_groups(d);
  if (rc != UFAIR_OK) return rc;
  if ((rc = check_out_every(d)) != UFAIR_OK) return rc;
  if ((rc = check_out_type(d, elem)) != UFAIR_OK) return rc;
  if (d->n_member == 0 || d->n_t == 0) return UFAIR_OK;
  if (!d->emissions || !d->gas_params || !d->thermal_params)
    return set_error(UFAIR_ERR_ARG, "emissions / gas_params / thermal_params must not be NULL");
  if (d->fext_mode != UFAIR_FEXT_NONE && !d->f_ext) return set_error(UFAIR_ERR_ARG, "fext_mode set but f_ext is NULL");
  if ((d->out_mask & UFAIR_OUT_C) && !d->out_C) return set_error(UFAIR_ERR_ARG, "out_C requested but NULL");
  if ((d->out_mask & UFAIR_OUT_RF) && !d->out_RF) return set_error(UFAIR_ERR_ARG, "out_RF requested but NULL");
  if ((d->out_mask & UFAIR_OUT_T) && !d->out_T) return set_error(UFAIR_ERR_ARG, "out_T requested but NULL");
  if ((d->out_mask & UFAIR_OUT_ALPHA) && !d->out_alpha) return set_error(UFAIR_ERR_ARG, "out_alpha requested but NULL");
  if ((d->out_mask & UFAIR_OUT_E) && !d->out_E) return set_error(UFAIR_ERR_ARG, "out_E requested but NULL");
  if (d->conc_driven < 0 || d->conc_driven >= (1 << d->n_gas))
    return set_error(UFAIR_ERR_ARG, "conc_driven 0x%x names a gas >= n_gas %d", d->conc_driven, d->n_gas);
  if (d->stats && (d->hist_bins < 1 || !(d->hist_hi > d->hist_lo)))
    return set_error(UFAIR_ERR_ARG, "stats requested but histogram spec/buffers incomplete");
  if (!placement) return UFAIR_OK;
  // TMA bulk-copy sources
  if (d->e_mode == UFAIR_E_MEMBER && misaligned(d->emissions))
    return set_error(UFAIR_ERR_ALIGN, "emissions must be 16-byte aligned");
  if (d->fext_mode == UFAIR_FEXT_MEMBER && misaligned(d->f_ext))
    return set_error(UFAIR_ERR_ALIGN, "f_ext must be 16-byte aligned");
  if (d->stats) {
    if ((rc = check_stat_buffers(d)) != UFAIR_OK) return rc;
    if (!d->out_T) return set_error(UFAIR_ERR_ARG, "stats need out_T (the moments pass reads the T rows)");
    if (d->hist_t0 < 0 || d->hist_rows < d->hist_t0 + out_rows(d))
      return set_error(UFAIR_ERR_ARG, "hist_rows %d < hist_t0 %d + output rows %d", d->hist_rows, d->hist_t0, out_rows(d));
  }
  return UFAIR_OK;
}
int validate_desc(const ufair_desc* d, size_t elem) { return check_desc(d, elem, true); }
int check_run(const ufair_desc* d, size_t elem) { return check_desc(d, elem, false); }

template <typename Real, typename Out> static KArgs<Real, Out> make_args(const ufair_desc* d) {
  KArgs<Real, Out> a;
  a.n_gas = d->n_gas;
  a.n_t = d->n_t;
  a.n_member = d->n_member;
  a.ld = d->ld_member;
  a.n_scen = d->n_scen;
  a.e_mode = d->e_mode;
  a.fext_mode = d->fext_mode;
  a.t_mode = d->t_mode;
  a.w_old = d->t_mode == UFAIR_T_MID ? (Real)0.5 : (Real)0;
  a.w_new = d->t_mode == UFAIR_T_MID ? (Real)0.5 : (Real)1;
  a.out_mask = d->out_mask;
  a.stats = d->stats;
  a.newton_iters = d->newton_iters;
#ifdef UFAIR_DEBUG_BOUNDS
  {  // negative control of the in-kernel bounds checks: UFAIR_DEBUG_TRIP=1 must make a full-length run fail
    const char* trip = getenv("UFAIR_DEBUG_TRIP");
    a.dbg_cut = (trip && trip[0] == '1') ? 1 : 0;
    a.dbg_cut_hits = nullptr;
  }
#else
  a.dbg_cut = 0;
#endif
  a.clamp = (d->iirf_max > 0.0 && isfinite(d->iirf_max)) ? 1 : 0;
  a.dt = d->dt;
  a.h = d->iirf_h;
  a.iirf_max = d->iirf_max;
  a.E = (const Real*)d->emissions;
  a.scen_idx = d->scen_idx;
  a.e_scale = (const Real*)d->e_scale;
  a.fext = (const Real*)d->f_ext;
  a.gp = (const Real*)d->gas_params;
  a.tp = (const Real*)d->thermal_params;
  a.state_in = (const Real*)d->state_in;
  a.oC = (Out*)d->out_C;
  a.oRF = (Out*)d->out_RF;
  a.oT = (Out*)d->out_T;
  a.oA = (Real*)d->out_alpha;
  a.oE = (Real*)d->out_E;
  a.conc_driven = d->conc_driven;
  a.state_out = (Real*)d->state_out;
  a.out_every = d->out_every >= 2 ? d->out_every : 1;
  a.n_out = out_rows(d);
  a.inv_every = (Real)(1.0 / a.out_every);
  return a;
}

// ---- tensor maps for the per-warp TMA pipelines (cuTensorMapEncodeTiled via the runtime's driver
// entry point, so libufair.so does not link libcuda) ---------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// emissions [n_gas][n_t][ld] -> rank-3 map, box = MW members x tile_steps steps x n_gas gases;
// f_ext [n_t][ld] -> rank-2 map, box = MW x tile_steps.  Out-of-range parts of a box are zero-filled.
int make_tensor_maps(const ufair_desc* d, size_t elem, int mw_members, int tile_steps, CUtensorMap* tmE,
                     CUtensorMap* tmF) {
  memset(tmE, 0, sizeof(*tmE));
  memset(tmF, 0, sizeof(*tmF));
  const bool e_member = d->e_mode == UFAIR_E_MEMBER, f_member = d->fext_mode == UFAIR_FEXT_MEMBER;
  if (!e_member && !f_member) return UFAIR_OK;
  EncodeTiledFn enc = encode_tiled();
  if (!enc) return set_error(UFAIR_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
  const CUtensorMapDataType dt = elem == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const cuuint32_t mw = (cuuint32_t)mw_members;
  const cuuint64_t row = (cuuint64_t)d->ld_member * elem;
  const cuuint32_t ones[3] = {1, 1, 1};
  if (e_member) {
    const cuuint64_t dims[3] = {(cuuint64_t)d->ld_member, (cuuint64_t)d->n_t, (cuuint64_t)d->n_gas};
    const cuuint64_t strides[2] = {row, row * (cuuint64_t)d->n_t};
    const cuuint32_t box[3] = {mw, (cuuint32_t)tile_steps, (cuuint32_t)d->n_gas};
    CUresult r = enc(tmE, dt, 3, const_cast<void*>(d->emissions), dims, strides, box, ones, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(UFAIR_ERR_CUDA, "cuTensorMapEncodeTiled(emissions) failed: %d", (int)r);
  }
  if (f_member) {
    const cuuint64_t dims[2] = {(cuuint64_t)d->ld_member, (cuuint64_t)d->n_t};
    const cuuint64_t strides[1] = {row};
    const cuuint32_t box[2] = {mw, (cuuint32_t)tile_steps};
    CUresult r = enc(tmF, dt, 2, const_cast<void*>(d->f_ext), dims, strides, box, ones, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(UFAIR_ERR_CUDA, "cuTensorMapEncodeTiled(f_ext) failed: %d", (int)r);
  }
  return UFAIR_OK;
}

// ---- statistics of T: second pass over the T rows the integrator just wrote ----------------------
// The moments of a set of values; the members are in the UFAIR_MOM_* slot order, so a Moments is one row of a moments
// buffer and at() views a stored row as one.  take() and merge() are the only statement of the merge rule; every fold
// applies them in a fixed order, so the moments are deterministic.
struct Moments {
  double sum, sumsq, min, max;
  __device__ static Moments identity() { return {0.0, 0.0, INFINITY, -INFINITY}; }
  __device__ static Moments& at(double* row) { return *reinterpret_cast<Moments*>(row); }
  __device__ static const Moments& at(const double* row) { return *reinterpret_cast<const Moments*>(row); }
  __device__ void take(double v) {
    sum += v;
    sumsq = fma(v, v, sumsq);
    min = fmin(min, v);
    max = fmax(max, v);
  }
  // a value of integer weight w > 0, with wv = (double)w * v: with w == 1 the operations of take(v)
  __device__ void take(double v, double wv) {
    sum += wv;
    sumsq = fma(wv, v, sumsq);
    min = fmin(min, v);
    max = fmax(max, v);
  }
  __device__ void merge(const Moments& o) {
    sum += o.sum;
    sumsq += o.sumsq;
    min = fmin(min, o.min);
    max = fmax(max, o.max);
  }
  __device__ Moments shfl_xor(int off) const {
    return {__shfl_xor_sync(0xffffffffu, sum, off), __shfl_xor_sync(0xffffffffu, sumsq, off),
            __shfl_xor_sync(0xffffffffu, min, off), __shfl_xor_sync(0xffffffffu, max, off)};
  }
};
static_assert(offsetof(Moments, sum) == UFAIR_MOM_SUM * sizeof(double) &&
                  offsetof(Moments, sumsq) == UFAIR_MOM_SUMSQ * sizeof(double) &&
                  offsetof(Moments, min) == UFAIR_MOM_MIN * sizeof(double) &&
                  offsetof(Moments, max) == UFAIR_MOM_MAX * sizeof(double) &&
                  sizeof(Moments) == UFAIR_MOM_COUNT * sizeof(double),
              "a Moments is one moments row");

// CTA (x = t * n_tiles + z, y = c) handles member slice c of row t for the groups [z NGT, z NGT + ngt) of tile z.
//   LABELS false: the pooled pass, one group, no labels read, x = t.
//   LABELS true (stat_group, e.g. per scenario): a tile of NGT groups.  The tiles of one row slice are neighbours on the
//   fastest grid axis, so they run together and all but the first find the slice in L2 (with one tile, T streams past
//   L2 as in the pooled pass, which keeps the label slice -- shared by every step of slice c, and those CTAs run
//   together -- resident).  A label outside [0, n_groups) is counted nowhere; one tile still reads the labels, so a
//   single group skips the negative ones.
//   histogram: bin = clamp(floor((T - lo) * invw), 0, bins - 1) in the run's precision (subtract and multiply rounded
//   separately, NaN not counted); counts go to a shared-memory histogram [ngt][bins] (per-thread run-length merging,
//   keyed by group and bin, in front of the atomics), then are added to row g * hist_rows + hist_t0 + t of
//   hist_private copy c -- rows this CTA alone owns, so no global atomics.  With more than kStatsSmemBins slots the
//   counts go straight to those rows with global atomics.
//   moments: strided per-thread partials (per group in registers: unrolled predicated updates), shuffle tree, warps in
//   order, merged into the same row of moments_private: no atomics, deterministic.  One group with every label 0
//   performs the pooled pass's operations in the same order, so it reproduces the pooled pass bit for bit.
//   WEIGHTS (ufair_stats_pass_weighted_*): member m adds weight[m] to its bin instead of 1 and takes
//   Moments::take(v, w * v); weight 0 counts the member nowhere, like a negative label.  Weights of 1 perform the
//   unweighted operations, so they reproduce the unweighted pass bit for bit.
constexpr int kStatsThreads = 256;
constexpr int kStatsSmemBins = 16384;  // 64 KB of dynamic shared memory at most

// The label arguments come after the pooled pass's, and the weights after them: each instantiation then keeps the
// parameter offsets of the arguments it shares with the pooled pass, and with them its instruction schedule.
template <typename Real, int NGT, bool LABELS, bool WEIGHTS>
__global__ void __launch_bounds__(kStatsThreads)
    stats_pass_kernel(const Real* __restrict__ T, long long ld, long long n_member, int t0_row, int rows, int bins,
                      Real lo, Real invw, int smem_hist, unsigned int* __restrict__ hp, double* mp,
                      const int32_t* __restrict__ labels, int n_groups, int n_tiles,
                      const uint32_t* __restrict__ weight) {
  static_assert(LABELS || NGT == 1, "without labels every member is in the one group");
  using M = Math<Real>;
  extern __shared__ unsigned int sh[];
  const int c = blockIdx.y, copies = gridDim.y;
  int t = blockIdx.x, g0 = 0, ngt = 1;  // t on x: no 65535 limit on the step count
  if constexpr (LABELS) {
    t = (int)(blockIdx.x / (unsigned)n_tiles);
    g0 = ((int)blockIdx.x - t * n_tiles) * NGT;
    ngt = min(NGT, n_groups - g0);
  }
  const long long m_lo = n_member * c / copies, m_hi = n_member * (c + 1) / copies;
  const Real* src = T + (long long)t * ld + m_lo;
  // rows per copy; one group's rows
  const size_t copy_rows = (size_t)(LABELS ? n_groups : 1) * rows, gstride = (size_t)rows * bins;
  unsigned int* grow = hp + ((size_t)c * copy_rows + (size_t)g0 * rows + t0_row + t) * bins;  // group g0 + j: + j gstride
  if (smem_hist) {
    for (int i = threadIdx.x; i < ngt * bins; i += blockDim.x) sh[i] = 0u;
    __syncthreads();
  }
  const int bins_m1 = bins - 1;
  Moments mom[NGT];
#pragma unroll
  for (int j = 0; j < NGT; ++j) mom[j] = Moments::identity();
  // four independent streaming loads in flight per thread; counts are run-length merged per thread
  // (a thread flushes one atomic when its group or bin changes), so a row whose members sit in one or two bins
  // issues almost no atomics and a spread-out row issues conflict-free ones
  const long long span = m_hi - m_lo;
  int last_g = -1, last_b = -1;
  unsigned run = 0;
  unsigned int* const hdst = smem_hist ? sh : grow;  // chosen once: a choice per flush costs the pooled FP32 pass a register
  auto flush = [&]() {
    if (!run) return;
    if constexpr (LABELS)
      atomicAdd(smem_hist ? sh + last_g * bins + last_b : grow + last_g * gstride + last_b, run);
    else
      atomicAdd(hdst + last_b, run);
  };
  auto take = [&](Real x, int label, unsigned wt) {
    int sel = 0;  // the member's group in this tile, -1 for none
    if constexpr (LABELS) {
      const int gl = label - g0;
      sel = (unsigned)gl < (unsigned)ngt ? gl : -1;
    }
    if constexpr (WEIGHTS)
      if (wt == 0u) sel = -1;  // skipped, not multiplied by 0: 0 * NaN and 0 * inf are NaN
    const double v = (double)x;
    if constexpr (WEIGHTS) {
      const double wv = (double)wt * v;
#pragma unroll
      for (int j = 0; j < NGT; ++j)
        if (sel == j) mom[j].take(v, wv);
    } else {
#pragma unroll
      for (int j = 0; j < NGT; ++j)
        if (sel == j) mom[j].take(v);
    }
    const Real q = M::bin_x(x, lo, invw);
    const int b = (sel >= 0 && q == q) ? max(0, min(bins_m1, M::floor_to_int(q))) : -1;
    if (b != last_b || (LABELS && sel != last_g)) {
      flush();
      last_g = sel;
      last_b = b;
      run = 0;
    }
    if constexpr (WEIGHTS)
      run += b >= 0 ? wt : 0u;  // the sum of a call's weights fits in 32 bits (include/ufair.h)
    else
      run += (b >= 0);
  };
  // one tile: stream T past L2; several: keep it for the sibling tiles.  The addresses are src + k + offset: with
  // src + (k + offset) nvcc unrolls the pooled FP64 loop differently (40 registers and 14 loads instead of 48 and 30).
  const bool keep = LABELS && n_tiles > 1;
  auto load = [&](const Real* p) { return keep ? __ldg(p) : __ldcs(p); };
  auto label = [&](long long i) {
    if constexpr (LABELS)
      return __ldg(labels + m_lo + i);
    else
      return 0;
  };
  // the weight slice, like the label slice, is shared by every row of copy c: __ldg keeps it in L2
  auto wgt = [&](long long i) {
    if constexpr (WEIGHTS)
      return __ldg(weight + m_lo + i);
    else
      return 1u;
  };
  long long k = threadIdx.x;
  for (; k + 3 * kStatsThreads < span; k += 4 * kStatsThreads) {
    const Real x0 = load(src + k), x1 = load(src + k + kStatsThreads), x2 = load(src + k + 2 * kStatsThreads),
               x3 = load(src + k + 3 * kStatsThreads);
    const int l0 = label(k), l1 = label(k + kStatsThreads), l2 = label(k + 2 * kStatsThreads),
              l3 = label(k + 3 * kStatsThreads);
    const unsigned w0 = wgt(k), w1 = wgt(k + kStatsThreads), w2 = wgt(k + 2 * kStatsThreads),
                   w3 = wgt(k + 3 * kStatsThreads);
    take(x0, l0, w0);
    take(x1, l1, w1);
    take(x2, l2, w2);
    take(x3, l3, w3);
  }
  for (; k < span; k += kStatsThreads) take(load(src + k), label(k), wgt(k));
  flush();
#pragma unroll
  for (int j = 0; j < NGT; ++j)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mom[j].merge(mom[j].shfl_xor(off));
  __shared__ Moments red[kStatsThreads / 32][NGT];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0)
#pragma unroll
    for (int j = 0; j < NGT; ++j) red[w][j] = mom[j];
  __syncthreads();
  if (smem_hist)
    for (int i = threadIdx.x; i < ngt * bins; i += blockDim.x)
      if (sh[i]) grow[LABELS ? (size_t)(i / bins) * gstride + i % bins : (size_t)i] += sh[i];
  if (threadIdx.x < ngt) {  // thread j folds group g0 + j, warps in order
    const int j = threadIdx.x;
    Moments& o = Moments::at(mp + ((size_t)c * copy_rows + (size_t)(g0 + j) * rows + t0_row + t) * UFAIR_MOM_COUNT);
    Moments m = o;
    for (int k = 0; k < (int)(blockDim.x >> 5); ++k) m.merge(red[k][j]);
    o = m;
  }
}

// Real here is the element type of the stored T rows (out_type), not necessarily the run's precision
template <typename Real, int NGT, bool LABELS, bool WEIGHTS>
static int launch_stats_pass(const ufair_desc* d, const uint32_t* weight, cudaStream_t stream) {
  const int G = LABELS ? stat_groups(d) : 1, n_tiles = (G + NGT - 1) / NGT;
  if (d->hist_copies > 65535) return set_error(UFAIR_ERR_ARG, "hist_copies %d > 65535", d->hist_copies);
  const int rows = out_rows(d);  // the T rows the integrator wrote
  if ((int64_t)rows * n_tiles > (int64_t)INT32_MAX) return set_error(UFAIR_ERR_ARG, "output rows x group tiles too large");
  const int smem_hist = (int64_t)NGT * d->hist_bins <= kStatsSmemBins ? 1 : 0;
  const size_t smem = smem_hist ? (size_t)NGT * d->hist_bins * sizeof(unsigned int) : 0;
  cudaError_t e = cudaSuccess;
  if (smem > 48 * 1024)
    e = cudaFuncSetAttribute(stats_pass_kernel<Real, NGT, LABELS, WEIGHTS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)smem);
  if (e != cudaSuccess) return cuda_error(e, "cudaFuncSetAttribute(stats_pass_kernel)");
  const Real lo = (Real)d->hist_lo;
  const Real invw = (Real)((Real)d->hist_bins / ((Real)d->hist_hi - (Real)d->hist_lo));
  stats_pass_kernel<Real, NGT, LABELS, WEIGHTS>
      <<<dim3((unsigned)(rows * n_tiles), (unsigned)d->hist_copies), kStatsThreads, smem, stream>>>(
          (const Real*)d->out_T, d->ld_member, d->n_member, d->hist_t0, d->hist_rows, d->hist_bins, lo, invw, smem_hist,
          d->hist_private, d->moments_private, d->stat_group, G, n_tiles, weight);
  e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "stats_pass_kernel launch");
}

// the launcher of the descriptor's gas count and alpha mode (validate_desc bounds both); v picks the kernel
template <typename Real, typename Out>
static int dispatch(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v, cudaStream_t s) {
  switch (4 * d->n_gas + d->alpha_mode) {
#define UFAIR_GAS(G)                                                                                      \
  case 4 * G + UFAIR_ALPHA_EXP: return launch_integrate<Real, Out, G, UFAIR_ALPHA_EXP>(d, a, v, s);       \
  case 4 * G + UFAIR_ALPHA_SINH: return launch_integrate<Real, Out, G, UFAIR_ALPHA_SINH>(d, a, v, s);     \
  case 4 * G + UFAIR_ALPHA_NEWTON: return launch_integrate<Real, Out, G, UFAIR_ALPHA_NEWTON>(d, a, v, s); \
  case 4 * G + UFAIR_ALPHA_ONE: return launch_integrate<Real, Out, G, UFAIR_ALPHA_ONE>(d, a, v, s);
    UFAIR_GAS(1) UFAIR_GAS(2) UFAIR_GAS(3) UFAIR_GAS(4)
#undef UFAIR_GAS
  }
  return set_error(UFAIR_ERR_UNSUPPORTED, "no integrator for %d gases in alpha mode %d", d->n_gas, d->alpha_mode);
}

#ifdef UFAIR_DEBUG_BOUNDS
// the negative control of the store check (a.dbg_cut > 0): run, then report every store the check found in the
// rows it pretends are missing as an error of this call
template <typename Real, typename Out>
static int run_cut_control(const ufair_desc* d, KArgs<Real, Out> a, Variant v, cudaStream_t stream) {
  cudaError_t e = cudaMalloc(&a.dbg_cut_hits, sizeof(unsigned long long));
  if (e != cudaSuccess) return cuda_error(e, "cudaMalloc(dbg_cut_hits)");
  unsigned long long hits = 0;
  int rc = UFAIR_OK;
  if ((e = cudaMemsetAsync(a.dbg_cut_hits, 0, sizeof(hits), stream)) != cudaSuccess) rc = cuda_error(e, "cudaMemsetAsync(dbg_cut_hits)");
  if (rc == UFAIR_OK) rc = dispatch<Real, Out>(d, a, v, stream);
  if (rc == UFAIR_OK && (e = cudaMemcpyAsync(&hits, a.dbg_cut_hits, sizeof(hits), cudaMemcpyDeviceToHost, stream)) != cudaSuccess)
    rc = cuda_error(e, "cudaMemcpyAsync(dbg_cut_hits)");
  if (rc == UFAIR_OK && (e = cudaStreamSynchronize(stream)) != cudaSuccess) rc = cuda_error(e, "cudaStreamSynchronize");
  cudaFree(a.dbg_cut_hits);
  if (rc == UFAIR_OK && hits)
    rc = set_error(UFAIR_ERR_ARG, "debug bounds check: %llu output stores in the last %d row(s) that UFAIR_DEBUG_TRIP cut off",
                   hits, a.dbg_cut);
  return rc;
}
#endif

// the run with outputs of element type Out
template <typename Real, typename Out> static int run_with(const ufair_desc* d, Variant v, cudaStream_t stream) {
  const KArgs<Real, Out> a = make_args<Real, Out>(d);
#ifdef UFAIR_DEBUG_BOUNDS
  if (a.dbg_cut) return run_cut_control<Real, Out>(d, a, v, stream);
#endif
  return dispatch<Real, Out>(d, a, v, stream);
}

template <typename Real> int run_device(const ufair_desc* d, cudaStream_t stream) {
  int rc = validate_desc(d, sizeof(Real));
  if (rc != UFAIR_OK) return rc;
  if (d->n_member == 0 || d->n_t == 0) return UFAIR_OK;
  const Variant v = choose_variant(d, sizeof(Real));
  if constexpr (sizeof(Real) == 8)
    if (v.out == UFAIR_OUTTYPE_F32) return run_with<Real, float>(d, v, stream);
  return run_with<Real, Real>(d, v, stream);
}

// ---- gas_form detection: which pools carry mass, which forcing terms exist, over all members -------
// flags[g]: bit q (q = 1..3) pool q+1 in use (a != 0 or initial state != 0); bits 4..6 f1 / f2 / f3 != 0
template <typename Real>
__global__ void detect_form_kernel(const Real* gp, const Real* state_in, int n_gas, long long n_member, long long ld,
                                   int* flags) {
  const int g = blockIdx.y;
  int f = 0;
  for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < n_member; m += (long long)gridDim.x * blockDim.x) {
    const Real* p = gp + (long long)g * UFAIR_GP_COUNT * ld + m;
    for (int q = 1; q < 4; ++q) {
      if (p[(UFAIR_GP_A0 + q) * ld] != Real(0)) f |= 1 << q;
      if (state_in && state_in[(long long)(5 * g + q) * ld + m] != Real(0)) f |= 1 << q;
    }
    if (p[UFAIR_GP_F1 * ld] != Real(0)) f |= 16;
    if (p[UFAIR_GP_F2 * ld] != Real(0)) f |= 32;
    if (p[UFAIR_GP_F3 * ld] != Real(0)) f |= 64;
  }
  f = __reduce_or_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0 && f) atomicOr(flags + g, f);
}

template <typename Real> int detect_form(const ufair_desc* d, int32_t* scratch, uint8_t* form, cudaStream_t stream) {
  int rc = validate_desc(d, sizeof(Real));
  if (rc != UFAIR_OK) return rc;
  if (!scratch || !form) return set_error(UFAIR_ERR_ARG, "ufair_detect_form: scratch / form must not be NULL");
  for (int g = 0; g < d->n_gas; ++g) form[g] = UFAIR_FORM(1, UFAIR_TERM_LIN);  // no members: nothing is used
  if (d->n_member == 0) return UFAIR_OK;
  cudaError_t e = cudaMemsetAsync(scratch, 0, UFAIR_MAX_GAS * sizeof(int32_t), stream);
  if (e != cudaSuccess) return cuda_error(e, "cudaMemsetAsync(scratch)");
  const unsigned bx = (unsigned)((d->n_member + 255) / 256 < 592 ? (d->n_member + 255) / 256 : 592);
  detect_form_kernel<Real><<<dim3(bx, (unsigned)d->n_gas), 256, 0, stream>>>(
      (const Real*)d->gas_params, (const Real*)d->state_in, d->n_gas, d->n_member, d->ld_member, scratch);
  if ((e = cudaGetLastError()) != cudaSuccess) return cuda_error(e, "detect_form_kernel launch");
  int32_t flags[UFAIR_MAX_GAS];
  if ((e = cudaMemcpyAsync(flags, scratch, sizeof(flags), cudaMemcpyDeviceToHost, stream)) != cudaSuccess)
    return cuda_error(e, "cudaMemcpyAsync(flags)");
  if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return cuda_error(e, "cudaStreamSynchronize");
  for (int g = 0; g < d->n_gas; ++g) {
    const int n_pool = (flags[g] & 8) ? 4 : (flags[g] & 4) ? 3 : (flags[g] & 2) ? 2 : 1;
    int terms = (flags[g] >> 4) & 7;
    if (terms == 0) terms = UFAIR_TERM_LIN;  // no forcing at all: the linear term (with f2 == 0) is the cheapest
    form[g] = UFAIR_FORM(n_pool, terms);
  }
  return UFAIR_OK;
}

// the pass over T rows of element type Rows, with or without member weights
template <typename Rows, bool WEIGHTS>
static int stats_pass_rows(const ufair_desc* d, const uint32_t* weight, cudaStream_t stream) {
  if (!d->stat_group) return launch_stats_pass<Rows, 1, false, WEIGHTS>(d, weight, stream);
  // up to four groups a tile of four: half the registers and predicated updates of a tile of eight
  return stat_groups(d) <= 4 ? launch_stats_pass<Rows, 4, true, WEIGHTS>(d, weight, stream)
                             : launch_stats_pass<Rows, 8, true, WEIGHTS>(d, weight, stream);
}
template <typename Rows> static int stats_pass_rows(const ufair_desc* d, const uint32_t* weight, cudaStream_t stream) {
  return weight ? stats_pass_rows<Rows, true>(d, weight, stream) : stats_pass_rows<Rows, false>(d, nullptr, stream);
}

// weight: the member weights of the weighted pass, NULL for the unweighted one
template <typename Real> int run_stats_pass(const ufair_desc* d, const uint32_t* weight, cudaStream_t stream) {
  int rc = validate_desc(d, sizeof(Real));
  if (rc != UFAIR_OK) return rc;
  if (!d->stats) return set_error(UFAIR_ERR_ARG, "ufair_stats_pass: descriptor has stats == 0");
  if (d->n_member == 0 || d->n_t == 0) return UFAIR_OK;
  // the T rows the integrator stored: float32 outputs of an FP64 run take the FP32 pass (include/ufair.h out_type)
  return out_elem(d, sizeof(Real)) == sizeof(float) ? stats_pass_rows<float>(d, weight, stream)
                                                    : stats_pass_rows<Real>(d, weight, stream);
}
template int run_stats_pass<double>(const ufair_desc*, const uint32_t*, cudaStream_t);
template int run_stats_pass<float>(const ufair_desc*, const uint32_t*, cudaStream_t);
template int run_device<double>(const ufair_desc*, cudaStream_t);
template int run_device<float>(const ufair_desc*, cudaStream_t);

// ---- statistics buffers -------------------------------------------------------------------------
__global__ void stats_reset_kernel(unsigned int* hist, size_t n_hist, double* mom, size_t n_rows) {
  const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = i0; i < n_hist; i += stride) hist[i] = 0u;
  for (size_t i = i0; i < n_rows; i += stride) Moments::at(mom + i * UFAIR_MOM_COUNT) = Moments::identity();
}

// The fold of the private copies, copies in order (deterministic): put_count(i, count) for every histogram slot i
// of the [rows][bins] result, put_moments(r, moments) for every row r.  The moments merge straight from the stored
// rows: copying each row out first reorders the unrolled loads and made the finalize kernels 14 % slower.
template <typename PutCount, typename PutMoments>
__device__ void fold_copies(const unsigned int* hp, const double* mp, int copies, int rows, int bins, PutCount put_count,
                            PutMoments put_moments) {
  const size_t n = (size_t)rows * bins;
  const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = i0; i < n; i += stride) {
    unsigned long long s = 0;
    for (int c = 0; c < copies; ++c) s += hp[(size_t)c * n + i];
    put_count(i, s);
  }
  for (size_t r = i0; r < (size_t)rows; r += stride) {
    Moments m = Moments::identity();
    for (int c = 0; c < copies; ++c) m.merge(Moments::at(mp + ((size_t)c * rows + r) * UFAIR_MOM_COUNT));
    put_moments(r, m);
  }
}

__global__ void stats_finalize_kernel(const unsigned int* hp, const double* mp, int copies, int rows, int bins,
                                      unsigned long long* hist, double* mom) {
  fold_copies(
      hp, mp, copies, rows, bins, [&](size_t i, unsigned long long s) { hist[i] = s; },
      [&](size_t r, const Moments& m) { Moments::at(mom + r * UFAIR_MOM_COUNT) = m; });
}

// The same fold, written in the layout the cross-GPU reduction wants: ONE buffer that is summed
// (sums[row][0 .. bins) = the counts as doubles -- integers below 2^53 add exactly in any order, so the
// reduced histogram stays bitwise independent of the GPU count --, sums[row][bins] = sum T,
// sums[row][bins + 1] = sum T^2) and ONE buffer that is max-reduced (ext[row] = {max T, -min T}).
__global__ void stats_finalize_packed_kernel(const unsigned int* hp, const double* mp, int copies, int rows, int bins,
                                             double* sums, double* ext) {
  const int pitch = bins + 2;
  fold_copies(
      hp, mp, copies, rows, bins, [&](size_t i, unsigned long long s) { sums[(i / bins) * pitch + (i % bins)] = (double)s; },
      [&](size_t r, const Moments& m) {
        sums[r * pitch + bins] = m.sum;
        sums[r * pitch + bins + 1] = m.sumsq;
        ext[2 * r] = m.max;
        ext[2 * r + 1] = -m.min;
      });
}

__global__ void stats_unpack_kernel(const double* sums, const double* ext, int rows, int bins, unsigned long long* hist,
                                    double* mom) {
  const int pitch = bins + 2;
  const size_t n = (size_t)rows * bins;
  const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = i0; i < n; i += stride) hist[i] = (unsigned long long)sums[(i / bins) * pitch + (i % bins)];
  for (size_t r = i0; r < (size_t)rows; r += stride) {
    double* o = mom + r * UFAIR_MOM_COUNT;
    o[UFAIR_MOM_SUM] = sums[r * pitch + bins];
    o[UFAIR_MOM_SUMSQ] = sums[r * pitch + bins + 1];
    o[UFAIR_MOM_MAX] = ext[2 * r];
    o[UFAIR_MOM_MIN] = -ext[2 * r + 1];
  }
}

// one thread per (row, percentile): walk the row's CDF (exact integers), interpolate inside the bin.
// Same operations in the same order as oracle/ufair_oracle.py percentiles_from_hist (no FMA).
__global__ void percentiles_kernel(const unsigned long long* __restrict__ hist, int rows, int bins, double lo, double hi,
                                   const double* __restrict__ pcts, int n_pct, double* __restrict__ out) {
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (long long)rows * n_pct) return;
  const int row = (int)(id / n_pct), j = (int)(id % n_pct);
  const unsigned long long* h = hist + (size_t)row * bins;
  unsigned long long tot = 0;
  for (int b = 0; b < bins; ++b) tot += h[b];
  const double target = __dmul_rn((double)tot, __ddiv_rn(pcts[j], 100.0));
  unsigned long long cum = 0, prev = 0;
  int k = bins - 1;
  for (int b = 0; b < bins; ++b) {  // k = number of bins whose CDF is < target, capped at bins - 1
    prev = cum;
    cum += h[b];
    if (!((double)cum < target)) {
      k = b;
      break;
    }
  }
  if (k == bins - 1 && (double)cum < target) {  // ran off the end: recompute prev for the last bin
    prev = cum - h[bins - 1];
  }
  const double cnt = (double)h[k];
  double frac = cnt > 0.0 ? __ddiv_rn(__dsub_rn(target, (double)prev), cnt) : 0.0;
  frac = fmin(fmax(frac, 0.0), 1.0);
  const double w = __ddiv_rn(__dsub_rn(hi, lo), (double)bins);
  out[id] = __dadd_rn(lo, __dmul_rn(__dadd_rn((double)k, frac), w));
}

static int check_stats_desc(const ufair_desc* d) {
  if (!d || d->struct_size != sizeof(ufair_desc)) return set_error(UFAIR_ERR_ARG, "bad descriptor");
  if (d->hist_bins < 1 || d->hist_rows < 1) return set_error(UFAIR_ERR_ARG, "histogram spec/buffers incomplete");
  const int rc = check_stat_buffers(d);
  return rc != UFAIR_OK ? rc : check_stat_groups(d);
}

// ---- parameter preparation ------------------------------------------------------------------------
__global__ void g1g0_kernel(const double* a, const double* tau, long long n, long long ld, double h, int mode,
                            double* g1o, double* g0o) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  double g1 = 0.0, s = 0.0;
  for (int i = 0; i < 4; ++i) {
    const double ai = a[i * ld + m], ti = tau[i * ld + m];
    const double z = h / ti, ez = exp(-z);
    g1 += ai * ti * (1.0 - (1.0 + z) * ez);
    s += ai * ti * (1.0 - ez);
  }
  s /= g1;
  g1o[m] = g1;
  g0o[m] = (mode == UFAIR_ALPHA_SINH) ? 1.0 / sinh(s) : exp(-s);
}

__global__ void kq_kernel(const double* tcr, const double* ecs, const double* d1, const double* d2, double f2x,
                          long long n, double* q1, double* q2) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  const double k1 = 1.0 - (d1[m] / 70.0) * (1.0 - exp(-70.0 / d1[m]));
  const double k2 = 1.0 - (d2[m] / 70.0) * (1.0 - exp(-70.0 / d2[m]));
  const double den = f2x * (k1 - k2);
  q1[m] = (tcr[m] - ecs[m] * k2) / den;
  q2[m] = (ecs[m] * k1 - tcr[m]) / den;
}

// reference U_FaIR/concentrations.py:5 -- emissions[0] * np.exp(-time), on broadcast operands.
// __dmul_rn: the product is rounded on its own, exactly like numpy's separate multiply.
__global__ void hfc_pulse_kernel(const double* e0, const double* time, double* out, long long n) {
  const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
  for (long long i = i0; i < n; i += stride) out[i] = __dmul_rn(e0[i], exp(-time[i]));
}

// ---- device-math probe (tests/test_gpu_math.py) ---------------------------------------------------
template <typename Real> __global__ void math_probe_kernel(int op, const Real* x, Real* y, long long n) {
  using M = Math<Real>;
  __shared__ __align__(16) unsigned char tbl[512];  // the exponential table, as the integrator's warps hold it
  const uint32_t tb = (uint32_t)__cvta_generic_to_shared(tbl);
  if (threadIdx.x < 32) M::fill_table(tb, (int)threadIdx.x);
  __syncthreads();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Real v = x[i];
  Real r;
  switch (op) {
    case 0: r = M::decay(v, tb); break;
    case 1: r = M::exp_(v, tb); break;
    case 2: r = M::rcp(v); break;
    case 3: r = M::sqrt_(v); break;
    case 4: r = M::log_(v); break;
    default: r = M::sinh_pair(v, tb); break;
  }
  y[i] = r;
}

// ---- peak microbenchmarks ---------------------------------------------------------------------------
template <typename T> __global__ void __launch_bounds__(256) peak_fma_kernel(int iters, T* sink) {
  T a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = T(1) + T(threadIdx.x + j) * T(1e-6);
  const T b = T(0.999999), c = T(1e-7);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = fma(a[j], b, c);  // one FMA per line (written out: the library builds with -fmad=false)
  }
  T s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += a[j];
  if (s == T(-12345)) sink[0] = s;  // never true; keeps the chains alive
}
__global__ void __launch_bounds__(256) peak_mufu_kernel(int iters, float* sink) {
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = 0.001f * (threadIdx.x + j);
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int j = 0; j < 8; ++j) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(a[j]));
  }
  float s = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) s += a[j];
  if (s == -12345.f) sink[0] = s;
}

template <typename Launch> static int time_kernel(Launch&& launch, cudaStream_t s, double* ms) {
  cudaEvent_t e0, e1;
  cudaError_t e;
  if ((e = cudaEventCreate(&e0)) != cudaSuccess) return cuda_error(e, "cudaEventCreate");
  if ((e = cudaEventCreate(&e1)) != cudaSuccess) return cuda_error(e, "cudaEventCreate");
  launch();  // warm-up
  cudaEventRecord(e0, s);
  launch();
  cudaEventRecord(e1, s);
  e = cudaEventSynchronize(e1);
  float t = 0.f;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&t, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (e != cudaSuccess) return cuda_error(e, "peak kernel");
  *ms = t;
  return UFAIR_OK;
}

static int peak_grid() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms * 8;
}

}  // namespace ufair

using namespace ufair;

extern "C" {

int ufair_abi_version(void) { return UFAIR_ABI_VERSION; }
const char* ufair_last_error(void) { return g_err; }
int64_t ufair_block_members(void) { return kWarps * 32; }

int ufair_run_f64(const ufair_desc* d, void* stream) { return run_device<double>(d, (cudaStream_t)stream); }
int ufair_run_f32(const ufair_desc* d, void* stream) { return run_device<float>(d, (cudaStream_t)stream); }

int ufair_stats_pass_f64(const ufair_desc* d, void* stream) {
  return run_stats_pass<double>(d, nullptr, (cudaStream_t)stream);
}
int ufair_stats_pass_f32(const ufair_desc* d, void* stream) {
  return run_stats_pass<float>(d, nullptr, (cudaStream_t)stream);
}
int ufair_stats_pass_weighted_f64(const ufair_desc* d, const uint32_t* weight, void* stream) {
  if (!weight) return set_error(UFAIR_ERR_ARG, "ufair_stats_pass_weighted: weight is NULL");
  return run_stats_pass<double>(d, weight, (cudaStream_t)stream);
}
int ufair_stats_pass_weighted_f32(const ufair_desc* d, const uint32_t* weight, void* stream) {
  if (!weight) return set_error(UFAIR_ERR_ARG, "ufair_stats_pass_weighted: weight is NULL");
  return run_stats_pass<float>(d, weight, (cudaStream_t)stream);
}

int ufair_detect_form_f64(const ufair_desc* d, int32_t* scratch, uint8_t* form, void* stream) {
  return detect_form<double>(d, scratch, form, (cudaStream_t)stream);
}
int ufair_detect_form_f32(const ufair_desc* d, int32_t* scratch, uint8_t* form, void* stream) {
  return detect_form<float>(d, scratch, form, (cudaStream_t)stream);
}

int ufair_kernel_variant(const ufair_desc* d, int32_t elem_size, uint32_t* form, int32_t* gpl, int32_t* mw,
                         int32_t* loop) {
  if (elem_size != 8 && elem_size != 4) return set_error(UFAIR_ERR_ARG, "elem_size must be 8 or 4");
  const int rc = validate_desc(d, (size_t)elem_size);
  if (rc != UFAIR_OK) return rc;
  const Variant v = choose_variant(d, elem_size);
  if (form) *form = v.form;
  if (gpl) *gpl = v.gpl;
  if (mw) *mw = members_per_warp(elem_size, d->n_gas, v.gpl);
  if (loop) *loop = v.loop;
  return UFAIR_OK;
}

int ufair_stats_reset(const ufair_desc* d, void* stream) {
  int rc = check_stats_desc(d);
  if (rc != UFAIR_OK) return rc;
  const size_t rows = (size_t)d->hist_copies * stat_groups(d) * d->hist_rows;
  stats_reset_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(d->hist_private, rows * d->hist_bins, d->moments_private, rows);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "stats_reset_kernel");
}

int ufair_stats_finalize(const ufair_desc* d, uint64_t* hist, double* moments, void* stream) {
  int rc = check_stats_desc(d);
  if (rc != UFAIR_OK) return rc;
  if (!hist || !moments) return set_error(UFAIR_ERR_ARG, "hist / moments output is NULL");
  stats_finalize_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(d->hist_private, d->moments_private, d->hist_copies,
                                                               stat_groups(d) * d->hist_rows, d->hist_bins,
                                                               (unsigned long long*)hist, moments);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "stats_finalize_kernel");
}

int ufair_stats_finalize_packed(const ufair_desc* d, double* sums, double* ext, void* stream) {
  int rc = check_stats_desc(d);
  if (rc != UFAIR_OK) return rc;
  if (!sums || !ext) return set_error(UFAIR_ERR_ARG, "sums / ext output is NULL");
  stats_finalize_packed_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(d->hist_private, d->moments_private, d->hist_copies,
                                                                      stat_groups(d) * d->hist_rows, d->hist_bins, sums, ext);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "stats_finalize_packed_kernel");
}

int ufair_stats_unpack(const double* sums, const double* ext, int32_t rows, int32_t bins, uint64_t* hist, double* moments,
                       void* stream) {
  if (rows < 0 || bins < 1) return set_error(UFAIR_ERR_ARG, "bad rows / bins");
  if (rows == 0) return UFAIR_OK;
  if (!sums || !ext || !hist || !moments) return set_error(UFAIR_ERR_ARG, "NULL pointer");
  stats_unpack_kernel<<<592, 256, 0, (cudaStream_t)stream>>>(sums, ext, rows, bins, (unsigned long long*)hist, moments);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "stats_unpack_kernel");
}

int ufair_g1g0_f64(const double* a, const double* tau, int64_t n, int64_t ld, double h, int32_t mode, double* g1,
                   double* g0, void* stream) {
  if (n < 0 || ld < n || !(h > 0.0)) return set_error(UFAIR_ERR_ARG, "bad n / ld / h");
  if (n == 0) return UFAIR_OK;
  if (!a || !tau || !g1 || !g0) return set_error(UFAIR_ERR_ARG, "NULL pointer");
  g1g0_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a, tau, n, ld, h, mode, g1, g0);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "g1g0_kernel");
}

int ufair_kq_f64(const double* tcr, const double* ecs, const double* d1, const double* d2, double f2x, int64_t n,
                 double* q1, double* q2, void* stream) {
  if (n < 0) return set_error(UFAIR_ERR_ARG, "bad n");
  if (n == 0) return UFAIR_OK;
  if (!tcr || !ecs || !d1 || !d2 || !q1 || !q2) return set_error(UFAIR_ERR_ARG, "NULL pointer");
  kq_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(tcr, ecs, d1, d2, f2x, n, q1, q2);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "kq_kernel");
}

int ufair_hfc_pulse_f64(const double* e0, const double* time, double* out, int64_t n, void* stream) {
  if (n < 0) return set_error(UFAIR_ERR_ARG, "bad n");
  if (n == 0) return UFAIR_OK;
  if (!e0 || !time || !out) return set_error(UFAIR_ERR_ARG, "NULL pointer");
  const unsigned grid = (unsigned)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  hfc_pulse_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(e0, time, out, n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "hfc_pulse_kernel");
}

int ufair_hist_percentiles(const uint64_t* hist, int32_t rows, int32_t bins, double lo, double hi, const double* pcts,
                           int32_t n_pct, double* out, void* stream) {
  if (rows < 0 || bins < 1 || n_pct < 0 || !(hi > lo)) return set_error(UFAIR_ERR_ARG, "bad histogram spec");
  if (rows == 0 || n_pct == 0) return UFAIR_OK;
  if (!hist || !pcts || !out) return set_error(UFAIR_ERR_ARG, "NULL pointer");
  const long long n = (long long)rows * n_pct;
  percentiles_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)hist, rows, bins, lo, hi, pcts, n_pct, out);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "percentiles_kernel");
}

int ufair_math_probe_f64(int op, const double* x, double* y, int64_t n, void* stream) {
  if (n <= 0) return UFAIR_OK;
  math_probe_kernel<double><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(op, x, y, n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "math_probe_kernel");
}
int ufair_math_probe_f32(int op, const float* x, float* y, int64_t n, void* stream) {
  if (n <= 0) return UFAIR_OK;
  math_probe_kernel<float><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(op, x, y, n);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "math_probe_kernel");
}

int ufair_peak_fp64(int iters, double* ms, double* flops, void* stream) {
  if (iters < 1 || !ms || !flops) return set_error(UFAIR_ERR_ARG, "bad args");
  double* sink = nullptr;
  cudaError_t e = cudaMalloc(&sink, sizeof(double));
  if (e != cudaSuccess) return cuda_error(e, "cudaMalloc");
  const int grid = peak_grid();
  int rc = time_kernel([&] { peak_fma_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink); },
                       (cudaStream_t)stream, ms);
  cudaFree(sink);
  *flops = 2.0 * 8.0 * (double)iters * 256.0 * grid;
  return rc;
}
int ufair_peak_fp32(int iters, double* ms, double* flops, void* stream) {
  if (iters < 1 || !ms || !flops) return set_error(UFAIR_ERR_ARG, "bad args");
  float* sink = nullptr;
  cudaError_t e = cudaMalloc(&sink, sizeof(float));
  if (e != cudaSuccess) return cuda_error(e, "cudaMalloc");
  const int grid = peak_grid();
  int rc = time_kernel([&] { peak_fma_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink); },
                       (cudaStream_t)stream, ms);
  cudaFree(sink);
  *flops = 2.0 * 8.0 * (double)iters * 256.0 * grid;
  return rc;
}
int ufair_peak_mufu(int iters, double* ms, double* ops, void* stream) {
  if (iters < 1 || !ms || !ops) return set_error(UFAIR_ERR_ARG, "bad args");
  float* sink = nullptr;
  cudaError_t e = cudaMalloc(&sink, sizeof(float));
  if (e != cudaSuccess) return cuda_error(e, "cudaMalloc");
  const int grid = peak_grid();
  int rc = time_kernel([&] { peak_mufu_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(iters, sink); },
                       (cudaStream_t)stream, ms);
  cudaFree(sink);
  *ops = 8.0 * (double)iters * 256.0 * grid;
  return rc;
}

}  // extern "C"
