// ntt_pass_stark_t11.cu -- one instantiation of the NTT pass kernel (ntt.cuh): radix-8 rounds, 2048-element tiles.
// Each instantiation has its own translation unit so that the heavy kernels compile in parallel.
#include "ntt.cuh"

using namespace stk;

int stk_launch_pass_stark_t11(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  return launch_pass_r<StarkField, 3, 256, 2, 0>(c, s, P, StarkField());
}
