// ntt_pass_stark_zs.cu -- one instantiation of the NTT pass kernel (ntt.cuh): first pass of a
// zero-padded transform (expansion round or coset scaling on load), 1024-element tiles.
// Each instantiation has its own translation unit so that the heavy kernels compile in parallel.
#include "ntt.cuh"

using namespace stk;

int stk_launch_pass_stark_zs(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  return launch_pass_r<StarkField, 3, 128, 4, 1>(c, s, P, StarkField());
}
