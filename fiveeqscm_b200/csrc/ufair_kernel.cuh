// ufair_kernel.cuh -- the fused Universal-FaIR time-stepping kernel (sm_100a).
//
// Work decomposition.  A WARP owns MW consecutive ensemble members and runs its own TMA pipeline
// (its own shared-memory ring and mbarriers); warps never wait for each other -- there is NO
// block-level synchronisation anywhere in the kernel.  Inside the warp a lane integrates either
//   GPL = NGAS : ALL gases of one member  (MW = 32: no idle lanes, no shuffles, one thermal step per member; the
//                                          default for FP32, for the specialised forms, and since round 2 for FP64
//                                          ensembles above UFAIR_SMALL_ENSEMBLE members), or
//   GPL = 1    : ONE gas of one member    (MW = 32, 16, 10, 8 members per warp for 1..4 gases; the NGAS lanes of
//                                          a member add up their forcings with warp shuffles; 3.2x as many warps,
//                                          which is what small FP64 ensembles in the default alpha mode need).
//   Pools, cumulative emissions and the two thermal boxes stay in REGISTERS across the serial time
//   loop.  The derived per-member constants sit in registers too where the register budget allows (all of
//   them in the FP64 kernels: 226-230 registers at 8 warps per SM in the all-gases-per-lane ones), and
//   otherwise in shared memory ([param][lane], conflict-free LDS.64 at base + immediate).  Which ones, the
//   tile length and the occupancy target of each class of kernel are one row of kTuning; LaneConsts places them.
//   Why: the loop is chains of dependent DFMAs (Horner polynomials); it is bound by the warp
//   schedulers' issue rate and dependent-issue latency, not by HBM.  ncu history (profiles/):
//     v1 thread per member, everything in regs (255), 2 warps/SMSP: FP64 pipe 35 %, IPC 0.37
//     v2 warp per gas + named barrier, 96 regs:      FP64 42 %, 61 % of issue slots non-FP64
//     v3 + constants in c[3], params in smem:        FP64 52 %, 19 % of samples in barrier stalls
//     v4 lanes = (member, gas), shuffles, no barrier: IPC 0.69, 413 instr / 10-member warp-step,
//        ~40 of them per-row TMA issue (R2UR + UBLKCP, 12 rows per tile)
//     v5 one 3-D tensor-map TMA per warp-tile, pinned smem addresses, running pointers: 335 instr
//        per 10-member warp-step, IPC 0.69 at 5 warps/SMSP -> 38.7 ms (41.8 with statistics)
//     v6 = GPL_ALL: a lane integrates all gases of its member again, now with smem constants (no
//        redundant thermal step, no shuffles, no idle lanes: 22.6 instr per member-step instead of
//        28.2).  First measured at 47.8 ms -- but that build was capped at 8 warps/SM by its 28 KB of
//        shared memory per warp (8-step tiles x 32 members), not by its 155 registers; with 2-step
//        tiles (11 warps/SM) it runs the dense case in 35.5 ms, a tie with GPL = 1 (35.3 ms), which
//        stays the FP64 default.  FP32, with half-width state, runs GPL = NGAS (26.4 -> 13.3 ms), and
//        so do the specialised per-gas forms (DESIGN.md 4.1b).
//     final round 1: cheaper rcp / sqrt / log, single-constant decay reduction, single-warp CTAs,
//        TT = 8; histogram moved out of the loop into the statistics pass (36.4 -> 33.7 ms); the plain
//        instantiation without run-time switches (-> 32.9); the 17 hottest per-lane constants in
//        registers at 16 warps/SM (-> 31.8 ms alone, 32-33.5 ms sustained): 221 instr per warp-step,
//        143 of them FP64, FP64 pipe 72 %.
//     round 2: the "2 N_FP64 + N_other" cost model of round 1 was wrong (tools/micro/: the pipes issue
//        independently; a DFMA reading three different registers holds the FP64 pipe 3 cycles, everything else 2;
//        dependent-issue latency 8 cycles).  Branch-free logarithm (its special-case branch had put every gas in
//        a basic block of its own), all gases per lane again (33.1 -> 29.6 ms), every per-lane constant in
//        registers at 8 warps/SM (-> 27.0), 8-step tiles (-> 26.0-27.2 ms, 0.69-0.72 of the FP64 roofline):
//        569 instr per 32-member warp-step, 407 of them FP64, FP64 pipe 80 % (profiles/r2_final_summary.md).
//   The loop body is alpha_val -> step_conc -> step_forc -> step_temp, the names the reference
//   reserves in .coveragerc:12-19; `oxfair` is ONE launch.
//   Which instantiation runs -- loop (VAR), lane mapping (GPL), per-gas form (FORM) -- is decided once per launch
//   by choose_variant (end of this file); launch_integrate runs it and ufair_kernel_variant reports it.
//
// Memory system
//   * per-member emissions [gas][t][member] are streamed into the warp's shared-memory ring one
//     tile of TT time steps ahead by ONE tensor-map TMA per tile
//     (cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes, box =
//     MW members x TT steps x NGAS gases; out-of-range rows/columns are zero-filled by the
//     hardware, which is what makes ragged tails free), double-buffered on two mbarriers per warp.
//     Per-member external forcing rides the same way through a 2-D map.
//   * C / RF / T are written straight from registers with streaming 64-bit stores (STG.E.EF.64): with all
//     gases of a member in one lane a warp writes one 256-byte run per row, with one gas per lane three
//     80-byte runs; L2 merges them into full sectors (DRAM traffic 1.01x the algorithmic bytes, ncu) --
//     nothing is re-read.  With float32 outputs of an FP64 run (UFAIR_OUTTYPE_F32, Out = float) each value is
//     rounded once at its store (cvt.rn.f32.f64) and a warp writes one 128-byte run per row (32-bit stores).
//   * optional statistics: the per-step histogram and the moments both come from a second,
//     HBM-speed pass over the T rows this kernel writes (stats_pass_kernel, ufair_abi.cu; one kernel for
//     pooled and per-label statistics, the pooled instantiation reading no labels): block-level
//     shared-memory histograms behind per-thread run-length merging.  Measured: the in-loop version (one
//     RED.ADD.U32 per member-step + the binning arithmetic in every lane) cost 2 ms of the 38 ms launch,
//     the extra work in the pass costs 0.3 ms.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include <utility>

#include "../../include/ufair.h"
#include "ufair_internal.h"
#include "ufair_math.cuh"

// FP64, default alpha mode: ensembles of at most this many members run one gas per lane (3.2x as many
// warps: a 10^4-member ensemble fills a third of the GPU's schedulers with 32-member warps, all of them
// with 10-member warps), larger ones all gases per lane.  Both give bit-identical results.  Measured (ms per
// launch, 3 gases x 736 steps; one gas per lane | all gases per lane): 10^4 members 0.38 | 0.65, 2*10^4
// 0.64 | 0.99, 4*10^4 1.07 | 1.38, 8*10^4 2.07 | 2.22, 1.6*10^5 4.05 | 3.88, 6.4*10^5 16.2 | 14.7.
#ifndef UFAIR_SMALL_ENSEMBLE
#define UFAIR_SMALL_ENSEMBLE 100000
#endif
#ifndef UFAIR_WARPS
#define UFAIR_WARPS 1  // warps per CTA.  A CTA is only a launch / shared-memory grouping (warps never
#endif                 // synchronise); single-warp CTAs measured ~2 % faster than 4 (finer refill)

namespace ufair {

constexpr int kWarps = UFAIR_WARPS;
constexpr int kStages = 2;  // tile ring depth

// ---- per-gas specialisation ("form"): 8 bits per gas, the descriptor's gas_form byte ------------
// bits 0-2: pools in use (0 = all four), bits 4-6: forcing terms present (0 = all three).  A form is
// the caller's promise that the other pools have a_i = 0 and zero initial state and that the other
// forcing coefficients are zero for every member; the specialised kernels then never touch them.
// Results are those of the dense kernel (adding exact zeros), only cheaper.
constexpr unsigned form_byte(int n_pool, unsigned terms) { return (unsigned)n_pool | (terms << 4); }
constexpr unsigned kGasFull = 0u;
constexpr unsigned kGasOneSqrt = form_byte(1, UFAIR_TERM_LIN | UFAIR_TERM_SQRT);  // CH4 / N2O-like
constexpr unsigned kGasOneLin = form_byte(1, UFAIR_TERM_LIN);                     // HFC-like
constexpr unsigned pack_form(unsigned g0, unsigned g1 = 0, unsigned g2 = 0, unsigned g3 = 0) {
  return g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
}
__host__ __device__ constexpr int form_pools(unsigned form, int g) {
  const int n = (int)((form >> (8 * g)) & 7u);
  return n ? n : 4;
}
__host__ __device__ constexpr unsigned form_terms(unsigned form, int g) {
  const unsigned t = (form >> (8 * g + 4)) & 7u;
  return t ? t : 7u;
}
// does the instantiated form `have` do everything the requested form `want` needs?
inline bool form_covers(unsigned have, unsigned want, int n_gas) {
  for (int g = 0; g < n_gas; ++g)
    if (form_pools(have, g) < form_pools(want, g) || (form_terms(have, g) & form_terms(want, g)) != form_terms(want, g))
      return false;
  return true;
}
// the specialised forms that are instantiated, per gas count, most specific first; a row ends at its
// first 0 (the dense kernel, never a specialised form)
constexpr int kMaxForms = 2;
constexpr unsigned kForms[UFAIR_MAX_GAS + 1][kMaxForms] = {
    {},
    {pack_form(kGasOneLin), pack_form(kGasOneSqrt)},
    {pack_form(kGasFull, kGasOneSqrt)},
    {pack_form(kGasFull, kGasOneSqrt, kGasOneSqrt)},
    {pack_form(kGasFull, kGasOneSqrt, kGasOneSqrt, kGasOneLin)}};
constexpr int n_forms(int n_gas) {
  int n = 0;
  while (n < kMaxForms && kForms[n_gas][n] != 0) ++n;
  return n;
}

// A lane integrates all gases of its member: no idle lanes, no shuffles, one thermal step per member (with
// the branch-free logarithm this wins in FP64 too, 31.3 -> 28.6 ms), and a specialised form must (its per-gas
// code differs, so gases cannot share a warp's instruction stream).  The dense FP64 kernels of the default
// alpha mode also exist with one gas per lane, for small ensembles (UFAIR_SMALL_ENSEMBLE).
// Float32 outputs (UFAIR_OUTTYPE_F32) have all gases per lane only: both mappings give the same bits.
constexpr bool has_small_variant(int elem_size, int n_gas, int amode, int var, int out_type) {
  return elem_size == 8 && n_gas > 1 && amode == UFAIR_ALPHA_EXP && var != UFAIR_LOOP_CONC_DRIVEN &&
         var != UFAIR_LOOP_PERIOD_MEAN && out_type == UFAIR_OUTTYPE_RUN;
}
// members per warp: rows of MW elements must be a multiple of 16 bytes for the TMA box
constexpr int members_per_warp(int elem_size, int n_gas, int gpl) {
  const int q = 16 / elem_size;    // elements per 16 bytes
  const int groups = n_gas / gpl;  // lanes per member
  return (32 / groups) / q * q;
}

// Out: the element type of the C / RF / T outputs (Real, or float for UFAIR_OUTTYPE_F32 outputs of an FP64 run);
// every other array, the state included, is in the run's precision
template <typename Real, typename Out = Real> struct KArgs {
  int n_gas, n_t;
  long long n_member, ld;
  int n_scen;
  int e_mode, fext_mode, t_mode, out_mask, stats, newton_iters, clamp;
  double dt, h, iirf_max;
  Real w_old, w_new;  // T = w_old (S1 + S2)_old + w_new (S1 + S2)_new; operands straight from the constant bank
  const Real* E;
  const int* scen_idx;
  const Real* e_scale;
  const Real* fext;
  const Real* gp;
  const Real* tp;
  const Real* state_in;
  Out* oC;
  Out* oRF;
  Out* oT;
  Real* oA;
  Real* oE;
  int conc_driven;  // bit g: gas g's input rows are target concentrations (INV kernels only)
  int dbg_cut;      // UFAIR_DEBUG_BOUNDS builds only: rows the store check pretends are missing (its negative control)
#ifdef UFAIR_DEBUG_BOUNDS
  unsigned long long* dbg_cut_hits;  // stores the check found in those rows (counted, not trapped)
#endif
  Real* state_out;
  int out_every, n_out;  // kVarMean: steps per output row (>= 2) and output rows
  Real inv_every;        // (Real)(1.0 / out_every)
};

// ---- PTX wrappers: mbarrier, tensor-map TMA, shared-space loads/stores with 32-bit addresses ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ double lds(uint32_t a, double) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds(uint32_t a, float) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts(uint32_t a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void sts(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
// keep a loop-invariant value in a register (stops the compiler from re-deriving it every step)
__device__ __forceinline__ void pin(uint32_t& x) { asm volatile("" : "+r"(x)); }

// a streaming store of v as an Out: with Out = float and Real = double the one rounding, to nearest even
template <typename Out, typename Real> __device__ __forceinline__ void st_stream(Out* p, Real v) { __stcs(p, (Out)v); }
// p - q for the diagnostic outputs (alpha, E), which are addressed relative to out_C: they exist only when the
// outputs have the run's element type (validate_desc rejects them otherwise)
template <typename P, typename Q> __device__ __forceinline__ long long diag_offset(P* p, Q* q) {
  if constexpr (std::is_same<P, Q>::value)
    return p - q;
  else
    return 0;
}

// -DUFAIR_DEBUG_BOUNDS (libufair_dbg.so, `make debug`; tests/test_gpu_guard.py runs the ragged cases on it):
// every output store must land inside its array, in a column below n_member, and every read of the
// shared-memory rings inside the box the TMA delivered for the current stage -- otherwise the kernel traps.
// compute-sanitizer is closed on the GPU pool this was developed on; this is the in-kernel stand-in.
// Its negative control (dbg_cut > 0) pretends the last rows of every output array are missing: stores the
// check finds there are counted in dbg_cut_hits and reported by the host, so the control never faults the device.
#ifdef UFAIR_DEBUG_BOUNDS
#define UFAIR_CHECK_ST(base, nrows, p)                                                                    \
  do {                                                                                                    \
    const long long off_ = (long long)((p) - (base));                                                     \
    if ((base) == nullptr || off_ < 0 || off_ >= (long long)(nrows) * ld || off_ % ld >= a.n_member) __trap(); \
    if (off_ >= ((long long)(nrows) - a.dbg_cut) * ld) atomicAdd(a.dbg_cut_hits, 1ull);                \
  } while (0)
#define UFAIR_CHECK_RING(addr, ring0, stage_bytes, box_bytes)                                             \
  do {                                                                                                    \
    const uint32_t off_ = (addr) - (ring0);                                                               \
    if ((addr) < (ring0) || off_ >= (uint32_t)kStages * (stage_bytes) || off_ % (stage_bytes) + ES > (box_bytes)) __trap(); \
  } while (0)
#else
#define UFAIR_CHECK_ST(base, nrows, p) ((void)0)
#define UFAIR_CHECK_RING(addr, ring0, stage_bytes, box_bytes) ((void)0)
#endif

// per-lane derived constants, by logical row: the G_* rows once per gas the lane integrates, the T_* rows once
// per lane.  Where each one lives is LaneConsts' business (below).
enum { H_RHO0 = 0, H_RHOU, H_WR, H_RHOT, H_UMAX, H_COUNT };  // u = rho0 + rhoU Gcum + wR sumR + rhoT T, capped at umax
enum {
  G_KA0 = 0,  // c a_i tau_i: equilibrium pool per unit (E alpha)
  G_K0 = 4,   // dt / tau_i   (ALPHA_ONE: m_i = 1 - exp(-dt/tau_i))
  G_C0 = 8,
  G_INVC0,
  G_SQRTC0,
  G_F1,
  G_F2,
  G_F3,
  G_HOT,                  // = 14: alpha_val's five, needed first in a step (on the critical path into alpha)
  G_X0 = G_HOT + H_COUNT  // SINH: g0; NEWTON: g1, ln g0, 1/c
};
enum { T_QM0 = 0, T_QM1, T_DEC0, T_DEC1, T_COUNT };  // q_j (1 - e^{-dt/d_j}),  e^{-dt/d_j}

// VAR, the instantiation of the time loop: kVarGeneral | kVarInverse (concentration-driven gases: diagnose the
// emissions, emissions output) | kVarPlain (no external forcing, no iIRF ceiling, outputs among C, RF, T only: the
// run-time switches for those cost ~38 of the general loop's 282 instructions, issued every step even when
// predicated off -- measured 35.6 -> 34.1 ms) | kVarPlainFx (the same with external forcing, shared
// or per member: the usual production configuration; default alpha mode only)
// | kVarPlainSub (any subset of C, RF, T -- typically T + statistics only -- as three lane predicates
// fixed before the loop; external forcing optional; default alpha mode only)
// | kVarMean (out_every >= 2: the general loop's options but alpha / E outputs, with C, RF and T summed in
// per-lane registers over a period of out_every steps and stored once per period, times 1 / out_every)
enum { kVarGeneral = UFAIR_LOOP_GENERAL, kVarInverse = UFAIR_LOOP_CONC_DRIVEN, kVarPlain = UFAIR_LOOP_PLAIN,
       kVarPlainFx = UFAIR_LOOP_PLAIN_FEXT, kVarPlainSub = UFAIR_LOOP_PLAIN_SUBSET, kVarMean = UFAIR_LOOP_PERIOD_MEAN };

// ---- per-instantiation tuning: one row per class of kernel ---------------------------------------------
// A class is a precision, dense or specialised form, and one gas or several per lane (GPL is 1 or NGAS, so the
// one-gas kernels -- NGAS = 1, or the FP64 small-ensemble mapping -- share a row).  A row gives the time steps per
// shared-memory tile, the resident warps per SM the register allocator must allow (__launch_bounds__), and which
// per-lane constants live in registers instead of shared memory -- the five alpha_val ones, the eight pool ones
// (G_KA0.., G_K0..), the four thermal ones: fewer LDS against more registers.  A tuning experiment edits one row.
// Measurements are ms per launch at [constants in registers (a alpha_val, p pools, t thermal, - none), warps/SM].
struct Tuning {
  int tile_steps;
  int warps_per_sm;
  bool alpha_reg, pool_reg, therm_reg;
  constexpr int min_blocks() const { return warps_per_sm / kWarps; }  // __launch_bounds__ counts CTAs
};
// classes by precision, then dense / specialised form, then several gases / one gas per lane; the period-mean loop
// (seven more FP64 values per lane in the 3-gas kernel) has rows of its own where the register budget needs them
enum { kF64Dense, kF64Dense1, kF64Form, kF64Form1, kF32Dense, kF32Dense1, kF32Form, kF32Form1, kF64DenseMean, kF64FormMean,
       kClasses };
constexpr int tuning_class(int elem_size, int gpl, unsigned form, int var) {
  return (var == kVarMean && elem_size == 8 && gpl > 1) ? (form != 0 ? kF64FormMean : kF64DenseMean)
                                                        : (elem_size == 8 ? 0 : 4) + (form != 0 ? 2 : 0) + (gpl == 1 ? 1 : 0);
}
constexpr Tuning kTuning[kClasses] = {
    // kF64Dense: all gases of a member in one lane, 2-4 gases.  Occupancy buys nothing here -- 16, 14, 12, 10 and
    // 8 resident warps per SM were all measured, and what sets the time is the length of each warp's own
    // instruction stream -- so the constants go to registers as far as the 255-register limit allows: [-,16] 29.5,
    // [-,12] 29.2, [t,12] 29.1, [at,12] 28.3, [at,10] 27.5, [pt,8] 28.0, [apt,8] 27.0 (226 registers; 21 LDS per
    // step left).  At 8 warps per SM shared memory is no constraint on the tile: 1 step 27.1 ms, 2: 27.2, 4: 26.8,
    // 8: 26.5.
    {8, 8, true, true, true},
    // kF64Dense1: one gas per lane (the small-ensemble mapping, and NGAS = 1).  Measured on the plain kernel:
    // [-,20] 34.5, [p,20] 34.0, [p,18] 33.8, [pt,18] 33.4, [ap,18] 33.0, [apt,18] 33.2 (spills), [apt,16] 32.6
    // (118 registers, 229 instructions per warp-step); 8-step tiles measured ~2 % faster than 4.
    {8, 16, true, true, true},
    // kF64Form: specialised forms, 2-4 gases.  Literature parameters: [-,12] 19.8-20.4, [p,12] 19.6, [pt,12] 19.6,
    // [apt,10] 19.0 (157 registers).  Short tiles: with 32 members per warp they are 3.2x as wide as the one-gas-
    // per-lane kernel's, and shared memory, not registers, would otherwise cap the occupancy.
    {2, 10, true, true, true},
    // kF64Form1: specialised forms of one gas: the row above with 8-step tiles (not measured on its own)
    {8, 10, true, true, true},
    // kF32Dense: 2-4 gases: [a,16] 9.7, [ap,16] 9.7, [apt,16] 9.5, [ap,12] 9.3, [apt,12] 9.1 (128 registers, 295
    // instructions per 32-member warp-step)
    {8, 12, true, true, true},
    // kF32Dense1: one gas: every constant in shared memory (not measured on its own)
    {8, 12, false, false, false},
    // kF32Form: specialised forms, 2-4 gases
    {8, 16, true, false, false},
    // kF32Form1: specialised forms of one gas: every constant in shared memory (not measured on its own)
    {8, 16, false, false, false},
    // kF64DenseMean: the period-mean loop, 2-4 gases: kF64Dense's row with the pool constants back in shared memory,
    // which makes room for the accumulators (on the plain loop that move measured 2 %: [at,10] 27.5 ms, [apt,8] 27.0;
    // 1.33x the plain loop's time at equal work, DESIGN.md 4.1)
    {8, 8, true, false, true},
    // kF64FormMean: the period-mean loop, specialised forms of 2-4 gases: kF64Form's row at 8 warps per SM (255
    // registers instead of 168: the 4-gas kernel spills at 10)
    {2, 8, true, true, true}};
constexpr Tuning tuning(int elem_size, int gpl, unsigned form, int var) {
  return kTuning[tuning_class(elem_size, gpl, form, var)];
}

constexpr int extra_rows(int amode) { return amode == UFAIR_ALPHA_NEWTON ? 3 : (amode == UFAIR_ALPHA_SINH ? 1 : 0); }
constexpr size_t round128(size_t b) { return (b + 127) / 128 * 128; }

// parameter rows of one gas when only its first `np` pools exist (the absent pools' KA / K0 rows are
// not allocated), and the compact row of row k of the per-gas block (LaneConsts::slot)
__host__ __device__ constexpr int gas_rows(int pg, int np) { return pg - 2 * (4 - np); }
__host__ __device__ constexpr int compact_row(int np, int k) { return k < 4 ? k : (k < 8 ? np + (k - 4) : 2 * np + (k - 8)); }

// per-WARP shared memory, in bytes (every piece 128-byte aligned: tensor-map TMA destinations)
template <typename Real, int NGAS, int AMODE, int GPL, unsigned FORM, int VAR> struct WarpSmem {
  static constexpr Tuning TUNE = tuning(sizeof(Real), GPL, FORM, VAR);
  static constexpr int TT = TUNE.tile_steps;  // time steps per tile
  static constexpr int MW = members_per_warp(sizeof(Real), NGAS, GPL);
  // rows per gas: register-resident alpha_val constants own none
  static constexpr int PG = G_X0 - (TUNE.alpha_reg ? H_COUNT : 0) + extra_rows(AMODE);
  // first row of gas gl / of the thermal block, and the row of logical row k of gas gl
  static __host__ __device__ constexpr int gas_base(int gl) {
    int b = 0;
    for (int g = 0; g < gl; ++g) b += gas_rows(PG, form_pools(FORM, g));
    return b;
  }
  static __host__ __device__ constexpr int row(int gl, int k) { return gas_base(gl) + compact_row(form_pools(FORM, gl), k); }
  static constexpr int T_BASE = gas_base(GPL);
  static constexpr int ROWS = T_BASE + T_COUNT;
  static constexpr uint32_t e_box = (uint32_t)(NGAS * TT * MW * sizeof(Real));  // bytes one E box delivers
  static constexpr uint32_t f_box = (uint32_t)(TT * MW * sizeof(Real));         // bytes one f_ext box delivers
  static constexpr uint32_t e_stage = (uint32_t)round128(e_box);
  static constexpr uint32_t f_stage = (uint32_t)round128(f_box);
  static constexpr uint32_t off_e = 0;
  static constexpr uint32_t off_f = off_e + kStages * e_stage;
  static constexpr uint32_t par_bytes = (uint32_t)round128(ROWS * 32 * sizeof(Real));
  // the f_ext ring exists only when external forcing is per member (decided at launch)
  static __host__ __device__ constexpr uint32_t off_par(bool fx_member) {
    return off_f + (fx_member ? kStages * f_stage : 0u);
  }
  static constexpr uint32_t tbl_bytes = sizeof(Real) == 8 ? kExpTableBytes : 0u;  // exp table copy (ufair_math.cuh)
  static __host__ __device__ constexpr uint32_t off_tbl(bool fx_member) { return off_par(fx_member) + par_bytes; }
  static __host__ __device__ constexpr uint32_t off_bar(bool fx_member) { return off_tbl(fx_member) + tbl_bytes; }
  static __host__ __device__ constexpr uint32_t bytes(bool fx_member) { return off_bar(fx_member) + 128u; }
};

// One lane's per-lane constants: its column of the warp's parameter block ([row][lane] in shared memory) and its
// register copies (the kernel's own arrays, declared where the compiler has always seen them).  The prologue sets
// each gas constant once through at(), the step reads every constant through get() / get_t(), both by logical row;
// which constants sit in registers is decided here and nowhere else:
//   * a register-resident alpha_val constant is set directly and owns no shared-memory row;
//   * register-resident pool and thermal constants still own a row: the prologue writes them there and load(),
//     after the prologue's __syncwarp, reads them into registers once;
//   * any other constant is read from its row at every use.
// The thermal constants are written to their rows (T_BASE + k) by the prologue itself: they own a row in every
// kernel, so there is nothing to decide, and through any helper call the FP32 specialised-form kernels compile to
// different code.
// A gas constant is named by a row K and an offset q inside K's block (the pool index for G_KA0 / G_K0, H_* for
// G_HOT, the position after G_X0).  Only K decides where it lives: K is a constant at every call site, and q, a
// loop index there, must not enter the decision -- it would stay a run-time test until the loops are unrolled
// and change how the compiler unrolls the Newton iteration around them.  at() returns the place before the value
// is computed, as a plain store computes its address first: a setter taking the value as an argument reorders the
// prologue (and changes the code of the FP32 sinh kernels).
template <typename Real, int NGAS, int AMODE, int GPL, unsigned FORM, int VAR> struct LaneConsts {
  using WS = WarpSmem<Real, NGAS, AMODE, GPL, FORM, VAR>;
  static constexpr bool kAlphaReg = WS::TUNE.alpha_reg, kPoolReg = WS::TUNE.pool_reg, kThermReg = WS::TUNE.therm_reg;
  uint32_t col;  // row 0 of this lane's column
  // register copies; only the rows in_reg() names are used, and of k0 / ka only the lane's pools (q < NP)
  Real (&hot)[GPL][H_COUNT];
  Real (&k0)[GPL][4];
  Real (&ka)[GPL][4];
  Real (&t)[T_COUNT];

  static __device__ __forceinline__ constexpr bool in_reg(int K) {
    return (K == G_HOT) ? kAlphaReg : (K == G_KA0 || K == G_K0) && kPoolReg;
  }
  // shared-memory row of logical gas row K: without alpha_val rows the extra rows move up
  static __device__ __forceinline__ constexpr int slot(int K) { return (kAlphaReg && K >= G_X0) ? K - H_COUNT : K; }
  __device__ __forceinline__ uint32_t gas_addr(int gl, int K, int q) const {
    return col + (uint32_t)WS::row(gl, slot(K) + q) * 32u * (uint32_t)sizeof(Real);
  }
  __device__ __forceinline__ uint32_t therm_addr(int k) const {
    return col + (uint32_t)(WS::T_BASE + k) * 32u * (uint32_t)sizeof(Real);
  }
  __device__ __forceinline__ Real reg(int gl, int K, int q) const {
    return K == G_HOT ? hot[gl][q] : K == G_KA0 ? ka[gl][q] : k0[gl][q];
  }

  struct Place {
    Real* reg;
    uint32_t addr;
    template <typename V> __device__ __forceinline__ void set(V v) const {
      if (reg)
        *reg = (Real)v;
      else
        sts(addr, (Real)v);
    }
  };
  __device__ __forceinline__ Place at(int gl, int K, int q = 0) {
    return (K == G_HOT && kAlphaReg) ? Place{&hot[gl][q], 0u} : Place{nullptr, gas_addr(gl, K, q)};
  }
  __device__ __forceinline__ void load() {
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        k0[gl][q] = (kPoolReg && q < form_pools(FORM, gl)) ? lds(gas_addr(gl, G_K0, q), Real()) : Real(0);
        ka[gl][q] = (kPoolReg && q < form_pools(FORM, gl)) ? lds(gas_addr(gl, G_KA0, q), Real()) : Real(0);
      }
#pragma unroll
    for (int k = 0; k < T_COUNT; ++k) t[k] = kThermReg ? lds(therm_addr(k), Real()) : Real(0);
  }
  __device__ __forceinline__ Real get(int gl, int K, int q = 0) const {
    return in_reg(K) ? reg(gl, K, q) : lds(gas_addr(gl, K, q), Real());
  }
  __device__ __forceinline__ Real get_t(int k) const { return kThermReg ? t[k] : lds(therm_addr(k), Real()); }
};

// EMEM: per-member emissions (TMA-staged tile) vs scenario-shared (read-only path + register prefetch)
// pool sum in the dense kernel's association, (R1 + R2) + (R3 + R4), without the absent pools
template <typename Real> __device__ __forceinline__ Real sum_pools(const Real (&R)[4], int np) {
  if (np >= 4) return (R[0] + R[1]) + (R[2] + R[3]);
  if (np == 3) return (R[0] + R[1]) + R[2];
  if (np == 2) return R[0] + R[1];
  return R[0];
}

// GPL: gases per lane (1 or NGAS); FORM: per-gas specialisation (0 = dense; needs GPL == NGAS);
// VAR: the loop (enum kVar* above the tuning table); Out: the element type of C / RF / T (KArgs)
template <typename Real, int NGAS, int AMODE, bool EMEM, int GPL, unsigned FORM, int VAR, typename Out = Real>
__global__ void __launch_bounds__(kWarps * 32, tuning(sizeof(Real), GPL, FORM, VAR).min_blocks())
    ufair_integrate_kernel(const __grid_constant__ KArgs<Real, Out> a, const __grid_constant__ CUtensorMap tmE,
                           const __grid_constant__ CUtensorMap tmF) {
  static_assert(FORM == 0 || GPL == NGAS, "a per-gas form needs all gases of a member in one lane");
  constexpr bool INV = (VAR == kVarInverse), PLAIN = (VAR >= kVarPlain && VAR != kVarMean), NOFX = (VAR == kVarPlain),
                 ALLOUT = (VAR == kVarPlain || VAR == kVarPlainFx),  // C, RF and T all written: no output predicates
                 MEAN = (VAR == kVarMean),  // period means: sums in registers, one store per period and output
                 DIAG = std::is_same<Out, Real>::value;  // the alpha / E outputs exist (outputs in the run's precision)
  static_assert(DIAG || !INV, "the inverse loop has no float32-output instantiation");
  using M = Math<Real>;
  using WS = WarpSmem<Real, NGAS, AMODE, GPL, FORM, VAR>;
  constexpr int kTT = WS::TT;            // time steps per tile
  constexpr int GROUPS = NGAS / GPL;     // lanes per member
  constexpr int MW = WS::MW;             // members per warp
  constexpr int NACT = MW * GROUPS;      // working lanes
  constexpr unsigned FULL = 0xffffffffu;
  constexpr uint32_t ES = sizeof(Real);
  constexpr uint32_t GROW = (uint32_t)(kTT * MW) * ES;  // bytes between two gases inside an E stage
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long wg = (long long)blockIdx.x * kWarps + warp;  // global warp index
  const long long m0 = wg * MW;                                // first member of this warp
  if (m0 >= a.n_member) return;  // whole warp: nothing to do (no CTA-wide sync exists)

  const int grp = min(lane / MW, GROUPS - 1);  // spare lanes shadow the last group
  const int i = min(lane - grp * MW, MW - 1);  // this lane's member inside the warp
  const int g0 = grp * GPL;                    // first gas of this lane
  const long long m_raw = m0 + i;
  const bool active = (lane < NACT) && (m_raw < a.n_member);
  const long long m = min(m_raw, a.n_member - 1);
  const long long ld = a.ld;
  const int n_t = a.n_t;

  const bool fx_member = !NOFX && (a.fext_mode == UFAIR_FEXT_MEMBER);
  const bool fx_scen = !NOFX && (a.fext_mode == UFAIR_FEXT_SCENARIO);
  const bool fx_any = fx_member || fx_scen;
  const bool use_tma = EMEM || fx_member;

  const uint32_t wbase = smem_u32(smem_raw) + (uint32_t)warp * WS::bytes(fx_member);
  uint32_t e_addr = wbase + WS::off_e + (uint32_t)(g0 * kTT * MW + i) * ES;  // this lane's E element: stage 0, tt 0
  uint32_t f_addr = wbase + WS::off_f + (uint32_t)i * ES;
  uint32_t par = wbase + WS::off_par(fx_member) + (uint32_t)lane * ES;       // this lane's parameter column
  const uint32_t bar0 = wbase + WS::off_bar(fx_member);
  uint32_t tb = wbase + WS::off_tbl(fx_member);  // this warp's copy of the exponential table
  M::fill_table(tb, lane);
  pin(e_addr);
  pin(f_addr);
  pin(par);
  pin(tb);

  const int n_tile = (n_t + kTT - 1) / kTT;
  if (lane == 0 && use_tma) {
    for (int s = 0; s < kStages; ++s) mbar_init(bar0 + 8u * s, 1);
    fence_barrier_init();
  }
  __syncwarp();
  auto issue_tile = [&](int k) {  // lane 0 only: one bulk tensor copy per tile (two with per-member f_ext)
    const uint32_t s = (uint32_t)(k % kStages);
    const uint32_t bar = bar0 + 8u * s;
    mbar_expect_tx(bar, (EMEM ? WS::e_box : 0u) + (fx_member ? WS::f_box : 0u));
    if (EMEM) tma_load_3d(wbase + WS::off_e + s * WS::e_stage, &tmE, (int)m0, k * kTT, 0, bar);
    if (fx_member) tma_load_2d(wbase + WS::off_f + s * WS::f_stage, &tmF, (int)m0, k * kTT, bar);
  };
  if (use_tma && lane == 0 && n_tile > 0) issue_tile(0);

  // ---------------- prologue: raw parameters -> derived constants, in double for both precisions
  // (g_1 and g_0 of .coveragerc:15-16 are fused here; in FP32 they would cancel catastrophically
  // for the 10^6-year pool, so the one-off prologue always runs in FP64 and rounds once)
  Real R[GPL][4], Gcum[GPL], sumR[GPL];
  Real hot[GPL][H_COUNT], k0[GPL][4], ka[GPL][4], tr[T_COUNT];  // LaneConsts' register copies
  LaneConsts<Real, NGAS, AMODE, GPL, FORM, VAR> cst{par, hot, k0, ka, tr};
  unsigned mk3[GPL];
  int nmin[GPL];  // lowest exponent alpha may take (Math::alpha_floor_exp)
  bool need_log[GPL], need_sqrt[GPL];
#pragma unroll
  for (int gl = 0; gl < GPL; ++gl) {
    const int g = g0 + gl;
    const int NP = form_pools(FORM, gl);         // pools this gas uses (4 unless specialised)
    const unsigned TERMS = form_terms(FORM, gl);  // forcing terms this gas has
    const Real* p = a.gp + (long long)g * UFAIR_GP_COUNT * ld + m;
    double av[4], tau[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      av[q] = (q < NP) ? (double)p[(UFAIR_GP_A0 + q) * ld] : 0.0;
      tau[q] = (q < NP) ? (double)p[(UFAIR_GP_TAU0 + q) * ld] : 1.0;
    }
    const double r0 = p[UFAIR_GP_R0 * ld], rU = p[UFAIR_GP_RU * ld], rT = p[UFAIR_GP_RT * ld], rA = p[UFAIR_GP_RA * ld];
    const double C0d = p[UFAIR_GP_C0 * ld], c = p[UFAIR_GP_EMIS2CONC * ld];
    double g1 = 0.0, sden = 0.0, k0max = 0.0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (q < NP) {
        k0max = fmax(k0max, a.dt / tau[q]);
        const double z = a.h / tau[q];
        const double ez = exp(-z);
        g1 += av[q] * tau[q] * (1.0 - (1.0 + z) * ez);
        sden += av[q] * tau[q] * (1.0 - ez);
      }
    }
    const double sarg = sden / g1;
    const double inv_g1 = 1.0 / g1, invc = 1.0 / c;
    const double lng0 = -sarg;
    const double fold = (AMODE == UFAIR_ALPHA_SINH) ? 0.0 : lng0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (q < NP) {
        cst.at(gl, G_KA0, q).set(c * av[q] * tau[q]);
        cst.at(gl, G_K0, q).set((AMODE == UFAIR_ALPHA_ONE) ? -expm1(-a.dt / tau[q]) : a.dt / tau[q]);
      }
    }
    const double hv[H_COUNT] = {r0 * inv_g1 + fold, rU * inv_g1, (rA - rU) * inv_g1 * invc, rT * inv_g1,
                                a.clamp ? (a.iirf_max * inv_g1 + fold) : (double)INFINITY};
#pragma unroll
    for (int q = 0; q < H_COUNT; ++q) cst.at(gl, G_HOT, q).set(hv[q]);
    nmin[gl] = M::alpha_floor_exp(k0max, AMODE == UFAIR_ALPHA_NEWTON ? 8 : 0);
    pin(reinterpret_cast<uint32_t&>(nmin[gl]));
    const Real f1v = p[UFAIR_GP_F1 * ld], f3v = p[UFAIR_GP_F3 * ld];
    cst.at(gl, G_C0).set(C0d);
    // the logarithm's argument is 1 + sumR / C0; a gas WITHOUT the log term (f1 == 0) gets 1 / C0 := 0 here,
    // so its argument is exactly 1, its logarithm exactly 0 and the term exactly zero -- also for C0 = 0
    // gases, where 1 / C0 is infinite -- with no mask or test in the loop
    cst.at(gl, G_INVC0).set(f1v != Real(0) ? 1.0 / C0d : 0.0);
    cst.at(gl, G_SQRTC0).set(sqrt(C0d));
    cst.at(gl, G_F1).set(f1v);
    cst.at(gl, G_F2).set(p[UFAIR_GP_F2 * ld]);
    cst.at(gl, G_F3).set(f3v);
    if (AMODE == UFAIR_ALPHA_SINH) cst.at(gl, G_X0).set(1.0 / sinh(sarg));
    if (AMODE == UFAIR_ALPHA_NEWTON) {
      cst.at(gl, G_X0).set(g1);
      cst.at(gl, G_X0, 1).set(lng0);
      cst.at(gl, G_X0, 2).set(invc);
    }
    // a zero forcing coefficient means a zero term; the log / sqrt is skipped only when no lane of
    // the warp needs it (voted once, outside the loop; with all gases in one lane this is per gas)
    // (PLAIN: no vote, no branch in the loop -- the masks below still zero an absent term)
    need_log[gl] = (TERMS & UFAIR_TERM_LOG) && (PLAIN || __any_sync(FULL, f1v != Real(0)));
    need_sqrt[gl] = (TERMS & UFAIR_TERM_SQRT) && (PLAIN || __any_sync(FULL, f3v != Real(0)));
    mk3[gl] = (f3v != Real(0)) ? 0xffffffffu : 0u;
    pin(mk3[gl]);
    const Real* si = a.state_in;
#pragma unroll
    for (int q = 0; q < 4; ++q) R[gl][q] = (si && q < NP) ? si[(long long)(5 * g + q) * ld + m] : Real(0);
    Gcum[gl] = si ? si[(long long)(5 * g + 4) * ld + m] : Real(0);
    sumR[gl] = sum_pools(R[gl], NP);
  }
  Real S0, S1, Tprev;
  {
    const Real* tp = a.tp + m;
    const Real* si = a.state_in;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const double qq = tp[(UFAIR_TP_Q1 + q) * ld], d = tp[(UFAIR_TP_D1 + q) * ld];
      const double mj = -expm1(-a.dt / d);
      // the thermal rows (see LaneConsts)
      sts(cst.col + (uint32_t)(WS::T_BASE + (T_QM0 + q)) * 32u * ES, (Real)(qq * mj));
      sts(cst.col + (uint32_t)(WS::T_BASE + (T_DEC0 + q)) * 32u * ES, (Real)(1.0 - mj));
    }
    S0 = si ? si[(long long)(5 * NGAS + 0) * ld + m] : Real(0);
    S1 = si ? si[(long long)(5 * NGAS + 1) * ld + m] : Real(0);
    Tprev = si ? si[(long long)(5 * NGAS + 2) * ld + m] : Real(0);
  }
  Real Ssum = S0 + S1;  // carried so that the mid-step mean costs one add
  __syncwarp();
  cst.load();

  const int scen = (a.scen_idx != nullptr) ? a.scen_idx[m] : 0;
  const Real dt = (Real)a.dt;
  const Real hdt = (Real)(a.h / a.dt);
  // T = wOld (S1 + S2)_old + wNew (S1 + S2)_new: (1/2, 1/2) is the mid-step mean, (0, 1) the end value;
  // bit-identical to the select it replaces because scaling by 1/2 is exact
  const Real wOld = a.w_old, wNew = a.w_new;
  const bool clamp = !PLAIN && a.clamp != 0;

  // Whether this lane stores an output this launch.  The general loops test a bit of wm, which packs all the
  // decisions in one register on purpose.  The plain loops have no alpha or E output and keep C, RF and T as lane
  // predicates fixed before the loop, not bits re-tested every step; in the loops that write all three those are
  // just `active` and `owner`.  Each store site picks its form inline: through a helper lambda the compiler
  // schedules several loops differently.
  const bool owner = active && (g0 == 0);  // the lane that owns the member's T / histogram count
  unsigned wm = (active ? (unsigned)(a.out_mask & (UFAIR_OUT_C | UFAIR_OUT_RF | UFAIR_OUT_ALPHA | (INV ? UFAIR_OUT_E : 0))) : 0u) |
                ((owner && ((a.out_mask & UFAIR_OUT_T) || a.stats)) ? (unsigned)UFAIR_OUT_T : 0u);
  const bool st_c = active && (a.out_mask & UFAIR_OUT_C) != 0, st_rf = active && (a.out_mask & UFAIR_OUT_RF) != 0,
             st_t = owner && ((a.out_mask & UFAIR_OUT_T) != 0 || a.stats != 0);
  pin(wm);
  // running output pointers (gas g0; + gl * gstride); the mean loop's advance once per period
  const long long gstride = (long long)(MEAN ? a.n_out : n_t) * ld;
  const long long o_gas = (long long)g0 * gstride + m_raw;
  Out* pC = a.oC + o_gas;
  Out* pRF = a.oRF + o_gas;
  const long long dA = diag_offset(a.oA, a.oC);  // the (diagnostic) alpha output is addressed relative to pC
  const long long dE = INV ? diag_offset(a.oE, a.oC) : 0;  // and so is the emissions output
  Out* pT = a.oT + m_raw;

  // scenario-mode inputs: register prefetch one step ahead through the read-only path
  Real e_next[GPL], esc[GPL], fx_next = 0;
  const Real* e_scen = a.E + ((long long)g0 * n_t) * a.n_scen + scen;
  const long long scen_gstride = (long long)n_t * a.n_scen;
  const Real* fx_scen_p = a.fext + scen;
#pragma unroll
  for (int gl = 0; gl < GPL; ++gl) {
    esc[gl] = (!EMEM && a.e_scale) ? a.e_scale[(long long)(g0 + gl) * ld + m] : Real(1);
    e_next[gl] = (!EMEM && n_t > 0) ? __ldg(e_scen + gl * scen_gstride) : Real(0);
  }
  if (fx_scen && n_t > 0) fx_next = __ldg(fx_scen_p);
  // the mean loop's period sums (s = 0; s = s + x every step; stored as s * (1 / out_every)) and its step counter
  // inside the period, the same in every lane
  Real sC[GPL], sRF[GPL], sT;
  int kk;
  if constexpr (MEAN) {
    sT = Real(0);
    kk = 0;
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) sC[gl] = sRF[gl] = Real(0);
  }

  // ---------------- one time step ------------------------------------------------------------------
  auto step = [&](const int t, const uint32_t tt_off) {
    Real fx = 0;
    if (fx_any) {  // one uniform branch when there is no external forcing at all
      if (fx_member) {
        UFAIR_CHECK_RING(f_addr + tt_off, wbase + WS::off_f, WS::f_stage, WS::f_box);
        fx = lds(f_addr + tt_off, Real());
      }
      if (fx_scen) {
        fx = fx_next;
        fx_next = __ldg(fx_scen_p + (long long)min(t + 1, n_t - 1) * a.n_scen);
      }
    }
    // The step runs in three passes over the gases of the lane -- alpha_val for every gas, then step_conc
    // for every gas, then step_forc for every gas -- instead of gas by gas: the gases are independent until
    // their forcings are added, and with the same stage of all of them next to each other in one basic
    // block the scheduler interleaves their dependent FP64 chains (with one gas per lane the passes are
    // the old gas-by-gas order).
    Real Fg[GPL], e[GPL], alpha[GPL], inva[GPL], Cg[GPL];
    bool bad = false;  // some logarithm of this step has an argument outside the fast path's domain
    // ---- inputs + alpha_val: state at t-1 -> alpha, 1/alpha
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) {
      const int NP = form_pools(FORM, gl);
      if (EMEM) {
        UFAIR_CHECK_RING(e_addr + tt_off + (uint32_t)gl * GROW, wbase + WS::off_e, WS::e_stage, WS::e_box);
        e[gl] = lds(e_addr + tt_off + (uint32_t)gl * GROW, Real());
      } else {
        e[gl] = e_next[gl] * esc[gl];
        e_next[gl] = __ldg(e_scen + gl * scen_gstride + (long long)min(t + 1, n_t - 1) * a.n_scen);
      }
      if (AMODE == UFAIR_ALPHA_ONE) {
        alpha[gl] = Real(1);
        inva[gl] = Real(1);
      } else {
        const Real rho0 = cst.get(gl, G_HOT, H_RHO0);
        const Real rhoU = cst.get(gl, G_HOT, H_RHOU);
        const Real wR = cst.get(gl, G_HOT, H_WR);
        const Real rhoT = cst.get(gl, G_HOT, H_RHOT);
        Real u = fma(rhoU, Gcum[gl], fma(wR, sumR[gl], fma(rhoT, Tprev, rho0)));
        if (clamp) {  // uniform: the iIRF ceiling costs nothing when it is switched off
          const Real umax = cst.get(gl, G_HOT, H_UMAX);
          u = (u > umax) ? umax : u;
        }
        Real al = (AMODE == UFAIR_ALPHA_SINH) ? cst.get(gl, G_X0) * M::sinh_pair(u, tb, nmin[gl]) : M::exp_(u, tb, nmin[gl]);
        if (AMODE == UFAIR_ALPHA_NEWTON) {
          const Real iirf = (u - cst.get(gl, G_X0, 1)) * cst.get(gl, G_X0);
          const Real invc = cst.get(gl, G_X0, 2);
          for (int it = 0; it < a.newton_iters; ++it) {
            const Real ia = M::rcp(al);
            Real f = -iirf, fp = 0;
#pragma unroll
            for (int q = 0; q < NP; ++q) {
              const Real z = cst.get(gl, G_K0, q) * hdt * ia;
              const Real mz = M::decay(z, tb);
              const Real at = cst.get(gl, G_KA0, q) * invc;  // a_i tau_i
              f = fma(at * al, mz, f);
              fp = fma(at, mz - z * (Real(1) - mz), fp);
            }
            const Real an = al - f * M::rcp(fp);
            al = M::fmax_(an, Real(0.5) * al);
          }
        }
        alpha[gl] = al;
        inva[gl] = M::rcp(al);
      }
    }
    // ---- step_conc: relax each pool toward its equilibrium  E alpha c a_i tau_i
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) {
      const int NP = form_pools(FORM, gl);
      Real mq[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q < NP) mq[q] = (AMODE == UFAIR_ALPHA_ONE) ? cst.get(gl, G_K0, q) : M::decay(cst.get(gl, G_K0, q) * inva[gl], tb);
      if (INV) {
        // concentration-driven gas: `e` is the target C; step_conc is linear in E, so
        //   E = (C_target - C0 - sum R_i (1 - m_i)) / (alpha sum m_i c a_i tau_i)
        Real keep = 0, gain = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (q < NP) {
            keep += fma(-mq[q], R[gl][q], R[gl][q]);
            gain = fma(mq[q], cst.get(gl, G_KA0, q), gain);
          }
        const Real e_inv = ((e[gl] - cst.get(gl, G_C0)) - keep) * M::rcp(gain * alpha[gl]);
        if ((a.conc_driven >> (g0 + gl)) & 1) e[gl] = e_inv;
        if constexpr (DIAG)
          if (wm & UFAIR_OUT_E) {
            UFAIR_CHECK_ST(a.oE, (long long)NGAS * n_t, pC + dE + gl * gstride);
            st_stream(pC + dE + gl * gstride, e[gl]);
          }
      }
      const Real ea = e[gl] * alpha[gl];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q < NP) R[gl][q] = fma(mq[q], fma(ea, cst.get(gl, G_KA0, q), -R[gl][q]), R[gl][q]);
      Gcum[gl] = fma(e[gl], dt, Gcum[gl]);
      sumR[gl] = sum_pools(R[gl], NP);
      Cg[gl] = cst.get(gl, G_C0) + sumR[gl];
      if constexpr (MEAN) {
        sC[gl] = sC[gl] + Cg[gl];
      } else if (ALLOUT ? active : PLAIN ? st_c : (wm & UFAIR_OUT_C) != 0) {
        UFAIR_CHECK_ST(a.oC, (long long)NGAS * n_t, pC + gl * gstride);
        st_stream(pC + gl * gstride, Cg[gl]);
      }
      if constexpr (DIAG && !PLAIN && !MEAN)
        if (wm & UFAIR_OUT_ALPHA) {
          UFAIR_CHECK_ST(a.oA, (long long)NGAS * n_t, pC + dA + gl * gstride);
          st_stream(pC + dA + gl * gstride, alpha[gl]);
        }
    }
    // ---- step_forc: F = f2 (C - C0) + f1 ln(C / C0) + f3 (sqrt C - sqrt C0), with C - C0 = sumR and
    // C / C0 = 1 + sumR / C0.  The logarithm runs its branch-free fast path for every gas (a special-case
    // branch per logarithm would split the gases into separate basic blocks); arguments outside its domain
    // are patched after the loop.  The sqrt VALUE is masked, not the product, so that a zero coefficient
    // with a NaN function value still contributes exactly zero.
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) {
      const unsigned TERMS = form_terms(FORM, gl);
      Real F = (TERMS & UFAIR_TERM_LIN) ? cst.get(gl, G_F2) * sumR[gl] : Real(0);
      if (need_log[gl]) {
        const Real y = fma(sumR[gl], cst.get(gl, G_INVC0), Real(1));
        F = fma(cst.get(gl, G_F1), M::log_fast(y), F);
        bad = bad || M::not_normal(y);
      }
      if (need_sqrt[gl]) F = fma(cst.get(gl, G_F3), M::mask(M::sqrt_(Cg[gl]) - cst.get(gl, G_SQRTC0), mk3[gl]), F);
      Fg[gl] = F;
    }
    if (__builtin_expect(bad, 0)) {  // never on a physical trajectory: redo those gases' forcing with the special values
#pragma unroll
      for (int gl = 0; gl < GPL; ++gl) {
        const unsigned TERMS = form_terms(FORM, gl);
        if (need_log[gl]) {
          const Real y = fma(sumR[gl], cst.get(gl, G_INVC0), Real(1));
          if (M::not_normal(y)) {
            Real F = (TERMS & UFAIR_TERM_LIN) ? cst.get(gl, G_F2) * sumR[gl] : Real(0);
            F = fma(cst.get(gl, G_F1), M::log_special(y), F);
            if (need_sqrt[gl])
              F = fma(cst.get(gl, G_F3), M::mask(M::sqrt_(cst.get(gl, G_C0) + sumR[gl]) - cst.get(gl, G_SQRTC0), mk3[gl]), F);
            Fg[gl] = F;
          }
        }
      }
    }
    Real Fsum = 0;
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) {
      if constexpr (MEAN) {
        sRF[gl] = sRF[gl] + Fg[gl];
      } else if (ALLOUT ? active : PLAIN ? st_rf : (wm & UFAIR_OUT_RF) != 0) {
        UFAIR_CHECK_ST(a.oRF, (long long)NGAS * n_t, pRF + gl * gstride);
        st_stream(pRF + gl * gstride, Fg[gl]);
      }
      Fsum = (gl == 0) ? Fg[gl] : Fsum + Fg[gl];
    }
    if constexpr (!MEAN) {
      pC += ld;
      pRF += ld;
    }
    // ---- total forcing of the member, gases in fixed order; external forcing last (as the oracle)
    Real Ftot;
    if (GROUPS == 1) {
      Ftot = Fsum + fx;
    } else {
      Ftot = __shfl_sync(FULL, Fsum, i);
#pragma unroll
      for (int gg = 1; gg < GROUPS; ++gg) Ftot += __shfl_sync(FULL, Fsum, gg * MW + i);
      Ftot += fx;
    }
    // ---- step_temp (with GROUPS > 1 computed redundantly, bit-identically, by a member's lanes)
    const Real s0 = fma(cst.get_t(T_QM0), Ftot, S0 * cst.get_t(T_DEC0));
    const Real s1 = fma(cst.get_t(T_QM1), Ftot, S1 * cst.get_t(T_DEC1));
    const Real Snew = s0 + s1;
    const Real T = fma(wNew, Snew, wOld * Ssum);
    S0 = s0;
    S1 = s1;
    Ssum = Snew;
    Tprev = T;
    if constexpr (MEAN) {
      sT = sT + T;
      if (++kk == a.out_every) {  // uniform: the last step of a period stores its means and starts the next sums
        kk = 0;
        const Real w = a.inv_every;
#pragma unroll
        for (int gl = 0; gl < GPL; ++gl) {
          if (st_c) {
            UFAIR_CHECK_ST(a.oC, (long long)NGAS * a.n_out, pC + gl * gstride);
            st_stream(pC + gl * gstride, sC[gl] * w);
          }
          if (st_rf) {
            UFAIR_CHECK_ST(a.oRF, (long long)NGAS * a.n_out, pRF + gl * gstride);
            st_stream(pRF + gl * gstride, sRF[gl] * w);
          }
          sC[gl] = sRF[gl] = Real(0);
        }
        if (st_t) {
          UFAIR_CHECK_ST(a.oT, (long long)a.n_out, pT);
          st_stream(pT, sT * w);
        }
        sT = Real(0);
        pC += ld;
        pRF += ld;
        pT += ld;
      }
    } else {
      if (ALLOUT ? owner : PLAIN ? st_t : (wm & UFAIR_OUT_T) != 0) {
        UFAIR_CHECK_ST(a.oT, (long long)n_t, pT);
        st_stream(pT, T);
      }
      pT += ld;
    }
  };

  // ---------------- the time loop --------------------------------------------------------------------
  for (int k = 0; k < n_tile; ++k) {
    const uint32_t s = (uint32_t)(k % kStages);
    const int t0 = k * kTT;
    if (use_tma) {
      if (lane == 0 && k + 1 < n_tile) issue_tile(k + 1);  // that stage was drained before the last __syncwarp
      mbar_wait(bar0 + 8u * s, (uint32_t)((k / kStages) & 1));
    }
    // not unrolled on purpose: the 24 FP64 polynomial / reduction constants stay hoisted in uniform
    // registers only while the body is a single copy (unrolling x4 spilled them back to LDC + moves)
    const int nt = min(kTT, n_t - t0);
    uint32_t tt_off = s * WS::e_stage;
    const uint32_t f_adj = s * WS::f_stage - s * WS::e_stage;  // f_addr + tt_off + f_adj addresses the f_ext stage
    f_addr += f_adj;
#pragma unroll 1
    for (int tt = 0; tt < nt; ++tt) {
      step(t0 + tt, tt_off);
      tt_off += (uint32_t)MW * ES;
    }
    f_addr -= f_adj;
    __syncwarp();  // every lane is done with stage s before lane 0 refills it
  }

  // ---------------- epilogue: final state (checkpoint / resume) ---------------------------------
  if (a.state_out && active) {
    Real* so = a.state_out;
#pragma unroll
    for (int gl = 0; gl < GPL; ++gl) {
#pragma unroll
      for (int q = 0; q < 4; ++q) so[(long long)(5 * (g0 + gl) + q) * ld + m] = R[gl][q];
      so[(long long)(5 * (g0 + gl) + 4) * ld + m] = Gcum[gl];
    }
    if (g0 == 0) {
      so[(long long)(5 * NGAS + 0) * ld + m] = S0;
      so[(long long)(5 * NGAS + 1) * ld + m] = S1;
      so[(long long)(5 * NGAS + 2) * ld + m] = Tprev;
    }
  }
}

// ---- the choice of instantiation, and its launch ----------------------------------------------------
int make_tensor_maps(const ufair_desc* d, size_t elem, int mw_members, int tile_steps, CUtensorMap* tmE,
                     CUtensorMap* tmF);

template <typename Real, int NGAS, int AMODE, int GPL, unsigned FORM, int VAR, typename Out>
int launch_variant(const ufair_desc* d, const KArgs<Real, Out>& a, cudaStream_t stream) {
  using WS = WarpSmem<Real, NGAS, AMODE, GPL, FORM, VAR>;
  CUtensorMap tmE, tmF;  // box = WS::MW members x WS::TT steps (x NGAS gases): depends on the variant
  const int rc = make_tensor_maps(d, sizeof(Real), WS::MW, WS::TT, &tmE, &tmF);
  if (rc != UFAIR_OK) return rc;
  const size_t smem = (size_t)WS::bytes(a.fext_mode == UFAIR_FEXT_MEMBER) * kWarps;
  auto kern = (a.e_mode == UFAIR_E_MEMBER) ? ufair_integrate_kernel<Real, NGAS, AMODE, true, GPL, FORM, VAR, Out>
                                            : ufair_integrate_kernel<Real, NGAS, AMODE, false, GPL, FORM, VAR, Out>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return cuda_error(e, "cudaFuncSetAttribute(ufair_integrate_kernel)");
  const long long n_warp = (a.n_member + WS::MW - 1) / WS::MW;
  const unsigned grid = (unsigned)((n_warp + kWarps - 1) / kWarps);
  kern<<<grid, kWarps * 32, smem, stream>>>(a, tmE, tmF);
  e = cudaGetLastError();
  return e == cudaSuccess ? UFAIR_OK : cuda_error(e, "ufair_integrate_kernel launch");
}

// the descriptor's gas_form bytes, packed like the FORM template argument
inline unsigned requested_form(const ufair_desc* d) {
  unsigned f = 0;
  for (int g = 0; g < d->n_gas; ++g) f |= (unsigned)d->gas_form[g] << (8 * g);
  return f;
}

// concentration-driven gases / the emissions output run on the INV instantiation of the general kernel
inline bool wants_inverse(const ufair_desc* d) { return d->conc_driven != 0 || (d->out_mask & UFAIR_OUT_E) != 0; }

// the element type of the C / RF / T outputs an instantiation stores
template <typename Real, typename Out>
constexpr int kOutType = std::is_same<Out, Real>::value ? UFAIR_OUTTYPE_RUN : UFAIR_OUTTYPE_F32;

// the loops each alpha mode has: the plain loops with external forcing (kVarPlainFx) or with a subset of
// the outputs (kVarPlainSub) exist in the default alpha mode only, and float32 outputs have every loop but
// the inverse one (validate_desc rejects what needs it) ...
constexpr bool loop_instantiated(int amode, int loop, int out_type) {
  return (amode == UFAIR_ALPHA_EXP || (loop != kVarPlainFx && loop != kVarPlainSub)) &&
         (out_type == UFAIR_OUTTYPE_RUN || loop != kVarInverse);
}
// ... and so do the specialised forms, for every loop but the inverse one
constexpr bool forms_instantiated(int amode, int loop) { return amode == UFAIR_ALPHA_EXP && loop != kVarInverse; }

// which instantiation of ufair_integrate_kernel runs a descriptor (EMEM follows e_mode)
struct Variant {
  unsigned form;  // FORM: an entry of kForms[n_gas], 0 = the dense kernel
  int loop;       // VAR: kVar* = UFAIR_LOOP_*
  int gpl;        // GPL: gases per lane, 1 or n_gas
  int out;        // Out: UFAIR_OUTTYPE_RUN (Out = Real) or UFAIR_OUTTYPE_F32 (Out = float, FP64 runs only)
};

// The only statement of the choice: run_device launches it and ufair_kernel_variant reports it.
inline Variant choose_variant(const ufair_desc* d, int elem_size) {
  // float32 outputs of an FP32 run are its own outputs
  const int out = (elem_size == 8 && d->out_type == UFAIR_OUTTYPE_F32) ? UFAIR_OUTTYPE_F32 : UFAIR_OUTTYPE_RUN;
  // the plain loops: no iIRF ceiling, outputs among C, RF, T only, emission-driven
  const int crt = UFAIR_OUT_C | UFAIR_OUT_RF | UFAIR_OUT_T;
  int loop = d->out_every >= 2 ? kVarMean
             : wants_inverse(d) ? kVarInverse
             : ((d->iirf_max > 0.0 && isfinite(d->iirf_max)) || (d->out_mask & UFAIR_OUT_ALPHA)) ? kVarGeneral
             : (d->out_mask & crt) != crt ? kVarPlainSub
             : d->fext_mode == UFAIR_FEXT_NONE ? kVarPlain
                                              : kVarPlainFx;
  if (!loop_instantiated(d->alpha_mode, loop, out)) loop = kVarGeneral;
  unsigned form = 0;  // the first instantiated form that covers the requested one
  const unsigned want = requested_form(d);
  if (want != 0 && forms_instantiated(d->alpha_mode, loop))
    for (int k = 0; k < n_forms(d->n_gas) && form == 0; ++k)
      if (form_covers(kForms[d->n_gas][k], want, d->n_gas)) form = kForms[d->n_gas][k];
  const bool small = form == 0 && has_small_variant(elem_size, d->n_gas, d->alpha_mode, loop, out) &&
                     d->n_member <= UFAIR_SMALL_ENSEMBLE;
  return {form, loop, small ? 1 : d->n_gas, out};
}

// launches <GPL, FORM, LOOP, Out> if that is v
template <typename Real, typename Out, int NGAS, int AMODE, int LOOP, int GPL, unsigned FORM>
bool launch_if(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v, cudaStream_t stream, int& rc) {
  if (v.loop != LOOP || v.gpl != GPL || v.form != FORM || v.out != kOutType<Real, Out>) return false;
  rc = launch_variant<Real, NGAS, AMODE, GPL, FORM, LOOP, Out>(d, a, stream);
  return true;
}
// the instantiations of one loop: dense with one gas per lane, dense with all of them, and the forms kForms[NGAS][K]
template <typename Real, typename Out, int NGAS, int AMODE, int LOOP, size_t... K>
bool launch_loop(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v, cudaStream_t stream, int& rc,
                 std::index_sequence<K...>) {
  constexpr int OUT = kOutType<Real, Out>;
  if constexpr (loop_instantiated(AMODE, LOOP, OUT)) {
    if constexpr (has_small_variant(sizeof(Real), NGAS, AMODE, LOOP, OUT))
      if (launch_if<Real, Out, NGAS, AMODE, LOOP, 1, 0u>(d, a, v, stream, rc)) return true;
    return launch_if<Real, Out, NGAS, AMODE, LOOP, NGAS, 0u>(d, a, v, stream, rc) ||
           (launch_if<Real, Out, NGAS, AMODE, LOOP, NGAS, kForms[NGAS][K]>(d, a, v, stream, rc) || ...);
  }
  return false;
}
// every instantiation of one (Real, Out, NGAS, AMODE) in turn: exactly those choose_variant can return; one that is
// not there is an error, never another kernel
template <typename Real, typename Out, int NGAS, int AMODE, int... LOOP>
int launch_chosen(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v, cudaStream_t stream,
                  std::integer_sequence<int, LOOP...>) {
  int rc = UFAIR_OK;
  if ((launch_loop<Real, Out, NGAS, AMODE, LOOP>(
           d, a, v, stream, rc, std::make_index_sequence<forms_instantiated(AMODE, LOOP) ? n_forms(NGAS) : 0>()) ||
       ...))
    return rc;
  return set_error(UFAIR_ERR_UNSUPPORTED,
                   "no integrator for %d gases, alpha mode %d, form 0x%x, %d gases per lane, loop %d, output type %d", NGAS,
                   AMODE, v.form, v.gpl, v.loop, v.out);
}

// The launcher of one (precision, output type, gas count, alpha mode): runs the instantiation v names.
// UFAIR_INSTANTIATE defines the four of a (precision, gas count) with outputs in the run's precision, and
// UFAIR_INSTANTIATE_OUT those of another output type (float32 outputs of FP64 runs), one ufair_inst_*.cu per
// (precision, gas count), so the kernels compile in parallel.
template <typename Real, typename Out, int NGAS, int AMODE>
int launch_integrate(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v, cudaStream_t stream);

#define UFAIR_LAUNCHER(Real, Out, NGAS, AMODE)                                                                  \
  template <>                                                                                                   \
  int launch_integrate<Real, Out, NGAS, AMODE>(const ufair_desc* d, const KArgs<Real, Out>& a, Variant v,      \
                                               cudaStream_t s) {                                                \
    return launch_chosen<Real, Out, NGAS, AMODE>(                                                               \
        d, a, v, s,                                                                                             \
        std::integer_sequence<int, kVarGeneral, kVarInverse, kVarPlain, kVarPlainFx, kVarPlainSub, kVarMean>()); \
  }
#define UFAIR_INSTANTIATE_OUT(Real, Out, NGAS)                                                                  \
  UFAIR_LAUNCHER(Real, Out, NGAS, UFAIR_ALPHA_EXP)                                                              \
  UFAIR_LAUNCHER(Real, Out, NGAS, UFAIR_ALPHA_SINH)                                                             \
  UFAIR_LAUNCHER(Real, Out, NGAS, UFAIR_ALPHA_NEWTON)                                                           \
  UFAIR_LAUNCHER(Real, Out, NGAS, UFAIR_ALPHA_ONE)
#define UFAIR_INSTANTIATE(Real, NGAS) UFAIR_INSTANTIATE_OUT(Real, Real, NGAS)

}  // namespace ufair
