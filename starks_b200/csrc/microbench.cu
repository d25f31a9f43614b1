// microbench.cu -- K0: measured integer-pipe issue rates on this B200 (the roofline
// denominators MEASURED_PEAKS.json does not carry) and in-register throughput of the
// field multiply / NTT butterfly built from them.
#include "ctx.h"
#include "field_exp.cuh"

using namespace stk;

namespace {

constexpr int kIlp = 8;

// Each thread keeps kIlp independent dependency chains so the pipe, not latency, bounds it.
template <int WHICH>
__global__ void __launch_bounds__(256) int_pipe_kernel(uint32_t* out, uint32_t seed, uint64_t iters) {
  uint32_t a[kIlp], b[kIlp];
  unsigned long long acc64[kIlp];
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
  for (int i = 0; i < kIlp; ++i) {
    a[i] = seed + t * 2654435761u + i;
    b[i] = (seed ^ t) * 40503u + 7u * i + 1u;
    acc64[i] = ((unsigned long long)a[i] << 32) | b[i];
  }
  uint32_t k = seed | 1u;
  double da[kIlp], dk = 1.0 + (double)(seed & 7u) * 0x1p-40, dc = 0x1p-30;
#pragma unroll
  for (int i = 0; i < kIlp; ++i) da[i] = 1.0 + (double)i * 0x1p-20 + (double)(t & 255u) * 0x1p-30;
  for (uint64_t it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (WHICH == 9) {  // 8-limb carry chain a += b (IADD3 with predicate carries)
        asm volatile("add.cc.u32 %0, %0, %1;" : "+r"(a[0]) : "r"(b[0]));
#pragma unroll
        for (int i = 1; i < kIlp - 1; ++i) asm volatile("addc.cc.u32 %0, %0, %1;" : "+r"(a[i]) : "r"(b[i]));
        asm volatile("addc.u32 %0, %0, %1;" : "+r"(a[kIlp - 1]) : "r"(b[kIlp - 1]));
        asm volatile("add.cc.u32 %0, %0, %1;" : "+r"(b[0]) : "r"(a[0]));
#pragma unroll
        for (int i = 1; i < kIlp - 1; ++i) asm volatile("addc.cc.u32 %0, %0, %1;" : "+r"(b[i]) : "r"(a[i]));
        asm volatile("addc.u32 %0, %0, %1;" : "+r"(b[kIlp - 1]) : "r"(a[kIlp - 1]));
        continue;
      }
      if (WHICH == 10) {  // two rows of 4 IMAD.WIDE.U32.X each (the mul512 inner pattern)
        asm volatile("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(a[0]), "+r"(a[1]) : "r"(b[0]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(a[2]), "+r"(a[3]) : "r"(b[2]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(a[4]), "+r"(a[5]) : "r"(b[4]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.u32 %1, %2, %3, %1;" : "+r"(a[6]), "+r"(a[7]) : "r"(b[6]), "r"(k));
        asm volatile("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(b[0]), "+r"(b[1]) : "r"(a[1]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(b[2]), "+r"(b[3]) : "r"(a[3]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(b[4]), "+r"(b[5]) : "r"(a[5]), "r"(k));
        asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.u32 %1, %2, %3, %1;" : "+r"(b[6]), "+r"(b[7]) : "r"(a[7]), "r"(k));
        continue;
      }
#pragma unroll
      for (int i = 0; i < kIlp; ++i) {
        if (WHICH == 0) {  // IMAD (32-bit multiply-add, low half)
          asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(a[i]) : "r"(k), "r"(b[i]));
        } else if (WHICH == 1) {  // IMAD.WIDE.U32 accumulate (32x32+64 -> 64)
          asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc64[i]) : "r"((uint32_t)acc64[i]), "r"(k));
        } else if (WHICH == 2) {  // IADD3
          asm volatile("add.u32 %0, %0, %1; add.u32 %0, %0, %2;" : "+r"(a[i]) : "r"(b[i]), "r"(k));
        } else if (WHICH == 3) {  // IMAD.HI.U32
          asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(a[i]) : "r"(k), "r"(b[i]));
        } else if (WHICH == 4) {  // BLAKE2s-like G quarter: add3, xor, rotate
          a[i] = a[i] + b[i] + k;
          b[i] = __funnelshift_r(b[i] ^ a[i], b[i] ^ a[i], 12);
        } else if (WHICH == 7) {  // IMAD + IADD3 on independent chains
          asm volatile("mad.lo.u32 %0, %0, %1, %1;" : "+r"(a[i]) : "r"(k));
          asm volatile("add.u32 %0, %0, %1; add.u32 %0, %0, %1;" : "+r"(b[i]) : "r"(k));
        } else if (WHICH == 11) {  // DFMA (FP64 pipe)
          asm volatile("fma.rz.f64 %0, %0, %1, %2;" : "+d"(da[i]) : "d"(dk), "d"(dc));
        } else if (WHICH == 12) {  // DFMA + IMAD.WIDE on independent chains
          asm volatile("fma.rz.f64 %0, %0, %1, %2;" : "+d"(da[i]) : "d"(dk), "d"(dc));
          asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc64[i]) : "r"((uint32_t)acc64[i]), "r"(k));
        } else if (WHICH == 13) {  // DFMA + two IADD3 on independent chains
          asm volatile("fma.rz.f64 %0, %0, %1, %2;" : "+d"(da[i]) : "d"(dk), "d"(dc));
          asm volatile("add.u32 %0, %0, %1; add.u32 %0, %0, %1;" : "+r"(b[i]) : "r"(k));
        } else if (WHICH == 8) {  // IMAD.WIDE + IADD3 on independent chains
          asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc64[i]) : "r"((uint32_t)acc64[i]), "r"(k));
          asm volatile("add.u32 %0, %0, %1; add.u32 %0, %0, %1;" : "+r"(b[i]) : "r"(k));
        }
      }
    }
  }
  uint32_t acc = 0;
#pragma unroll
  for (int i = 0; i < kIlp; ++i)
    acc ^= a[i] ^ b[i] ^ (uint32_t)acc64[i] ^ (uint32_t)(acc64[i] >> 32) ^ (uint32_t)__double2loint(da[i]) ^
           (uint32_t)__double2hiint(da[i]);
  out[t] = acc;
}

// ops per inner step (per chain for the per-chain kinds), as counted in the returned `ops`
__host__ double ops_per_iter(int which) {
  switch (which) {
    case 4: return 4.0 * kIlp * 3;   // IADD3 + LOP3 + SHF
    case 7: case 8: case 12: case 13: return 4.0 * kIlp * 2;
    case 9: return 4.0 * 2 * kIlp;   // two 8-limb add chains
    case 10: return 4.0 * 8;         // eight wide multiply-adds
    default: return 4.0 * kIlp;
  }
}

template <class F, int WHICH>
__global__ void __launch_bounds__(256) field_kernel(fe* out, const fe* in, uint64_t iters, const F f) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  fe x0 = fe_load(in + (t & 1023)), x1 = fe_load(in + ((t + 1) & 1023));
  fe y0 = fe_load(in + ((t + 2) & 1023)), y1 = fe_load(in + ((t + 3) & 1023));
  fe w = fe_load(in + ((t + 4) & 1023));
  for (uint64_t it = 0; it < iters; ++it) {
    if (WHICH == 5) {  // 4 independent multiplies
      x0 = f.mul_tw(x0, w); x1 = f.mul_tw(x1, w); y0 = f.mul_tw(y0, w); y1 = f.mul_tw(y1, w);
    } else {  // 2 DIF butterflies
      fe s0 = f.add(x0, y0), d0 = f.sub(x0, y0);
      fe s1 = f.add(x1, y1), d1 = f.sub(x1, y1);
      x0 = s0; y0 = f.mul_tw(d0, w);
      x1 = s1; y1 = f.mul_tw(d1, w);
    }
  }
  fe r = f.add(f.add(x0, x1), f.add(y0, y1));
  fe_store(out + t, r);
}

}  // namespace

STK_API int stk_microbench(stk_ctx* c, int which, uint64_t iters, float* ms, double* ops) {
  if (!c || !ms || !ops || which < 0 || which > 13) return STK_EINVAL;
  const unsigned blocks = (unsigned)c->sm_count * 8, threads = 256;
  void* buf;
  STK_TRY(stk_scratch(c, kSlotStage, (uint64_t)blocks * threads * sizeof(fe) + 1024 * sizeof(fe), &buf));
  fe* out = (fe*)buf;
  fe* in = out + (uint64_t)blocks * threads;
  if (which == 5 || which == 6) {
    std::vector<fe> h(1024);
    for (int i = 0; i < 1024; ++i)
      for (int l = 0; l < 8; ++l) h[i].v[l] = (uint32_t)(2654435761u * (i * 8 + l + 1)) & (l == 7 ? 0x7FFFFFFFu : 0xFFFFFFFFu);
    STK_CUDA(c, cudaMemcpyAsync(in, h.data(), 1024 * sizeof(fe), cudaMemcpyHostToDevice, c->stream));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  cudaEvent_t e0, e1;
  STK_CUDA(c, cudaEventCreate(&e0));
  STK_CUDA(c, cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; ++rep) {  // first repetition warms up
    STK_CUDA(c, cudaEventRecord(e0, c->stream));
    switch (which) {
#define IPK(W) case W: int_pipe_kernel<W><<<blocks, threads, 0, c->stream>>>((uint32_t*)out, 12345u, iters); break;
      IPK(0) IPK(1) IPK(2) IPK(3) IPK(4) IPK(7) IPK(8) IPK(9) IPK(10) IPK(11) IPK(12) IPK(13)
#undef IPK
      case 5:
        STK_TRY(stk_with_field(c, [&](auto f) {
          field_kernel<decltype(f), 5><<<blocks, threads, 0, c->stream>>>(out, in, iters, f);
        }));
        break;
      default:
        STK_TRY(stk_with_field(c, [&](auto f) {
          field_kernel<decltype(f), 6><<<blocks, threads, 0, c->stream>>>(out, in, iters, f);
        }));
        break;
    }
    STK_CUDA(c, cudaEventRecord(e1, c->stream));
    STK_CUDA(c, cudaEventSynchronize(e1));
  }
  STK_CUDA(c, cudaGetLastError());
  STK_CUDA(c, cudaEventElapsedTime(ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  double nthreads = (double)blocks * threads;
  if (which == 5) *ops = nthreads * (double)iters * 4.0;
  else if (which == 6) *ops = nthreads * (double)iters * 2.0;
  else *ops = nthreads * (double)iters * ops_per_iter(which);
  return STK_OK;
}

// A/B of the experimental multiply (field_exp.cuh) against the production one, in registers:
// which = 5 (four independent multiplies per iteration) or 6 (two DIF butterflies); variant 0 is
// the production StarkField, bit 0 = accumulators without zero-initialisation, bit 1 = aligned
// 351*H rows.  *mismatches = how many of the kernel's outputs differ from the production
// kernel's on the same inputs (must be 0: both are exact).
template <int V>
static int run_variant(stk_ctx* c, int which, uint64_t iters, unsigned blocks, unsigned threads, fe* out, const fe* in) {
  if (which == 5) field_kernel<StarkFieldX<V>, 5><<<blocks, threads, 0, c->stream>>>(out, in, iters, StarkFieldX<V>());
  else field_kernel<StarkFieldX<V>, 6><<<blocks, threads, 0, c->stream>>>(out, in, iters, StarkFieldX<V>());
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

STK_API int stk_microbench_variant(stk_ctx* c, int variant, int which, uint64_t iters, float* ms, double* ops,
                                   uint64_t* mismatches) {
  if (!c || !ms || !ops || !mismatches || (which != 5 && which != 6) || variant < 0 || variant > 3) return STK_EINVAL;
  if (!c->is_stark) return stk_fail(c, STK_EUNSUPPORTED, "the experimental multiply is for the STARK prime");
  const unsigned blocks = (unsigned)c->sm_count * 8, threads = 256;
  const uint64_t nthr = (uint64_t)blocks * threads;
  void* buf;
  STK_TRY(stk_scratch(c, kSlotStage, (2 * nthr + 1024) * sizeof(fe), &buf));
  fe* out = (fe*)buf;
  fe* ref = out + nthr;
  fe* in = ref + nthr;
  std::vector<fe> h(1024);
  for (int i = 0; i < 1024; ++i)
    for (int l = 0; l < 8; ++l) h[i].v[l] = (uint32_t)(2654435761u * (i * 8 + l + 1)) & (l == 7 ? 0x7FFFFFFFu : 0xFFFFFFFFu);
  // a few saturated operands so that the carry limbs of every row are exercised
  for (int l = 0; l < 8; ++l) { h[5].v[l] = 0xFFFFFFFFu; h[6].v[l] = l == 0 ? 0u : (l == 1 ? 0xFFFFFEA1u : 0xFFFFFFFFu); }
  h[5] = StarkField().reduce(h[5]);
  STK_CUDA(c, cudaMemcpyAsync(in, h.data(), 1024 * sizeof(fe), cudaMemcpyHostToDevice, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  const uint64_t check_iters = iters < 64 ? iters : 64;
  if (which == 5) field_kernel<StarkField, 5><<<blocks, threads, 0, c->stream>>>(ref, in, check_iters, StarkField());
  else field_kernel<StarkField, 6><<<blocks, threads, 0, c->stream>>>(ref, in, check_iters, StarkField());
  STK_CUDA(c, cudaGetLastError());
#define RUNV(IT) \
  do { \
    switch (variant) { \
      case 0: STK_TRY(run_variant<0>(c, which, IT, blocks, threads, out, in)); break; \
      case 1: STK_TRY(run_variant<1>(c, which, IT, blocks, threads, out, in)); break; \
      case 2: STK_TRY(run_variant<2>(c, which, IT, blocks, threads, out, in)); break; \
      default: STK_TRY(run_variant<3>(c, which, IT, blocks, threads, out, in)); break; \
    } \
  } while (0)
  RUNV(check_iters);
  std::vector<fe> ho(nthr), hr(nthr);
  STK_CUDA(c, cudaMemcpyAsync(ho.data(), out, nthr * sizeof(fe), cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaMemcpyAsync(hr.data(), ref, nthr * sizeof(fe), cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  uint64_t bad = 0;
  for (uint64_t i = 0; i < nthr; ++i) bad += fe_eq(ho[i], hr[i]) ? 0 : 1;
  *mismatches = bad;
  cudaEvent_t e0, e1;
  STK_CUDA(c, cudaEventCreate(&e0));
  STK_CUDA(c, cudaEventCreate(&e1));
  for (int rep = 0; rep < 2; ++rep) {
    STK_CUDA(c, cudaEventRecord(e0, c->stream));
    RUNV(iters);
    STK_CUDA(c, cudaEventRecord(e1, c->stream));
    STK_CUDA(c, cudaEventSynchronize(e1));
  }
#undef RUNV
  STK_CUDA(c, cudaEventElapsedTime(ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ops = (double)nthr * (double)iters * (which == 5 ? 4.0 : 2.0);
  return STK_OK;
}
