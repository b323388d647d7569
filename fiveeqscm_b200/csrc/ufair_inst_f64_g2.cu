// the fused integrator's launchers and kernels for double, 2 gas(es): every alpha mode, loop and instantiated form
#include "ufair_kernel.cuh"
namespace ufair {
UFAIR_INSTANTIATE(double, 2)
}  // namespace ufair
