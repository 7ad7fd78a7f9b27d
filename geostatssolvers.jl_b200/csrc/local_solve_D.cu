// local_solve_D.cu — instantiates K3 for <G, R, W, RS, NT> = <32, 3, 8, 72, 128> (see local_solve.cuh): k <= 64 with more than 6 drift terms
#include "local_solve.cuh"
cudaError_t gsk_local_launch_D(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols) {
  return cols ? gsk_local::launch_cfg<32, 3, 8, 72, 128, true>(a, *cols, e, st) : gsk_local::launch_cfg<32, 3, 8, 72, 128>(a, GskColArgs{}, e, st);
}
