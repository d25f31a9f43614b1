// ntt_pass_mont.cu -- one instantiation of the NTT pass kernel (ntt.cuh): run-time modulus
// (Montgomery), radix-4 rounds, 1024-element tiles.
// Each instantiation has its own translation unit so that the heavy kernels compile in parallel.
#include "ntt.cuh"

using namespace stk;

int stk_launch_pass_mont(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  return launch_pass_r<MontField, 2, 256, 2, 0>(c, s, P, c->mont);
}
