// local_solve_C.cu — instantiates K3 for <G, R, W, RS, NT> = <8, 5, 8, 40, 64> (see local_solve.cuh)
#include "local_solve.cuh"
cudaError_t gsk_local_launch_C(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols) {
  return cols ? gsk_local::launch_cfg<8, 5, 8, 40, 64, true>(a, *cols, e, st) : gsk_local::launch_cfg<8, 5, 8, 40, 64>(a, GskColArgs{}, e, st);
}
