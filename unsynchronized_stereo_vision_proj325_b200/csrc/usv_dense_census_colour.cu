// usv_dense_census_colour.cu — the three-plane census variants of the sliding-window sweep (usv_dense.cu): census frames
// split into planes by the launcher, every plane swept into the same accumulators.
#include "usv_dense_kernel.cuh"

namespace usv {

template DenseKernel dense_kernel<3, 4, true>(int, int, bool);
template DenseKernel dense_kernel<3, 8, true>(int, int, bool);

}  // namespace usv
