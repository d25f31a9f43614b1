// ntt_pass_stark.cu -- one instantiation of the NTT pass kernel (ntt.cuh): radix-8 rounds, 1024-element tiles.
// Each instantiation has its own translation unit so that the heavy kernels compile in parallel.
#include "ntt.cuh"

using namespace stk;

// resident CTAs per SM the kernel is compiled for (register budget 65536 / (128 * STK_MINB)); the
// A/B builds of tools/gpu_minb_ab.sh override it
#ifndef STK_MINB
#define STK_MINB 4
#endif
int stk_launch_pass_stark(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  return launch_pass_r<StarkField, 3, 128, STK_MINB, 0>(c, s, P, StarkField());
}
