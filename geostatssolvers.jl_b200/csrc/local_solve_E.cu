// local_solve_E.cu — instantiates K3 for <G, R, W, RS, NT> = <32, 4, 8, 112, 128> (see local_solve.cuh)
#include "local_solve.cuh"
cudaError_t gsk_local_launch_E(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols) {
  return cols ? gsk_local::launch_cfg<32, 4, 8, 112, 128, true>(a, *cols, e, st) : gsk_local::launch_cfg<32, 4, 8, 112, 128>(a, GskColArgs{}, e, st);
}
