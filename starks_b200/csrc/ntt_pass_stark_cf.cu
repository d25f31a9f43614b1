// ntt_pass_stark_cf.cu -- one instantiation of the NTT pass kernel (ntt.cuh): final pass of a
// coset transform (interleaved store), 1024-element tiles.
// Each instantiation has its own translation unit so that the heavy kernels compile in parallel.
#include "ntt.cuh"

using namespace stk;

int stk_launch_pass_stark_cf(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  return launch_pass_r<StarkField, 3, 128, 4, 2>(c, s, P, StarkField());
}
