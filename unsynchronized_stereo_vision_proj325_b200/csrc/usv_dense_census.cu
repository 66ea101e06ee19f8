// usv_dense_census.cu — the one-plane census variants (JT = 4 and 8) of the sliding-window sweep (usv_dense.cu): the
// Hamming arm of usv_dense_kernel.cuh, compiled apart from the SAD variants so that the build stays parallel.
#include "usv_dense_kernel.cuh"

namespace usv {

template DenseKernel dense_kernel<1, 4, true>(int, int, bool);
template DenseKernel dense_kernel<1, 8, true>(int, int, bool);

}  // namespace usv
