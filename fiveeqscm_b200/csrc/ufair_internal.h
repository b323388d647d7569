// ufair_internal.h -- shared between the translation units of libufair.so (not installed).
#pragma once
#include <cuda_runtime.h>

#include "../../include/ufair.h"

namespace ufair {
int set_error(int code, const char* fmt, ...);
int cuda_error(cudaError_t e, const char* what);
// A run's descriptor: validate_desc checks the run rules and the placement rules of device arrays (every device entry
// point), check_run the run rules alone (ufair_run_host_* on the caller's descriptor of host arrays).
int validate_desc(const ufair_desc* d, size_t elem);
int check_run(const ufair_desc* d, size_t elem);
// statistics groups G: every statistics buffer holds G x hist_rows rows (include/ufair.h)
inline int stat_groups(const ufair_desc* d) { return d->n_stat_groups > 1 ? d->n_stat_groups : 1; }
// output rows of C, RF and T: one per step, or one per period of out_every >= 2 steps (include/ufair.h)
inline int out_rows(const ufair_desc* d) { return d->out_every >= 2 ? d->n_t / d->out_every : d->n_t; }
// bytes per element of out_C / out_RF / out_T in a run of element size elem (out_type, include/ufair.h)
inline size_t out_elem(const ufair_desc* d, size_t elem) { return d->out_type == UFAIR_OUTTYPE_F32 ? sizeof(float) : elem; }
template <typename Real> int run_device(const ufair_desc* d, cudaStream_t stream);
// the statistics pass; weight: [n_member] member weights (ufair_stats_pass_weighted_*), NULL for the unweighted pass
template <typename Real> int run_stats_pass(const ufair_desc* d, const uint32_t* weight, cudaStream_t stream);
}  // namespace ufair
