// local_solve_A.cu — instantiates K3 for <G, R, W, RS, NT> = <4, 3, 4, 12, 128> (see local_solve.cuh)
#include "local_solve.cuh"
cudaError_t gsk_local_launch_A(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols) {
  return cols ? gsk_local::launch_cfg<4, 3, 4, 12, 128, true>(a, *cols, e, st) : gsk_local::launch_cfg<4, 3, 4, 12, 128>(a, GskColArgs{}, e, st);
}
