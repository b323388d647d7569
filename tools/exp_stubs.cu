// tools/exp_stubs.cu -- perf-experiment builds only (never in the shipped library): stands in for every
// integrator instantiation except <double, 3 gases>, so that a tuning variant of the headline kernel
// links in seconds.  Usage: see tools/build_variant.sh.
#include "../fiveeqscm_b200/csrc/ufair_kernel.cuh"
namespace ufair {
#define STUB(Real, NGAS, AMODE)                                                                        \
  template <> int launch_integrate<Real, NGAS, AMODE>(const ufair_desc*, const KArgs<Real>&, Variant, cudaStream_t) { \
    return set_error(UFAIR_ERR_UNSUPPORTED, "experiment build: only <double, 3 gases> is instantiated"); \
  }
#define STUB4(Real, NGAS) STUB(Real, NGAS, UFAIR_ALPHA_EXP) STUB(Real, NGAS, UFAIR_ALPHA_SINH) STUB(Real, NGAS, UFAIR_ALPHA_NEWTON) STUB(Real, NGAS, UFAIR_ALPHA_ONE)
STUB4(double, 1) STUB4(double, 2) STUB4(double, 4)
STUB4(float, 1) STUB4(float, 2) STUB4(float, 3) STUB4(float, 4)
}  // namespace ufair
