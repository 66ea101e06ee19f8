// usv_dense_colour.cu — the three-plane variants of the sliding-window SAD kernel (usv_dense.cu): interleaved colour frames,
// split into planes by the launcher, every plane swept into the same accumulators.
#include "usv_dense_kernel.cuh"

namespace usv {

template DenseKernel dense_kernel<3, 4>(int, int, bool);
template DenseKernel dense_kernel<3, 8>(int, int, bool);

}  // namespace usv
