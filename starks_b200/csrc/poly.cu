// poly.cu -- dense polynomial product and long division in coefficient form (Polynomial.__mul__ and
// Polynomial.__divmod__, starks/polynomial.py:110-143) in O(n log n).
//
// Every product picks one of two routes from the modulus: the transform route (forward transforms
// of length L through stk_ntt_dev, a pointwise product, a scaled inverse) wherever Z/p has a root of
// unity of order L, and otherwise the direct route, one thread per output coefficient.  Division is
// Newton iteration on the reversed divisor, g <- g(2 - f g), fused into one pointwise kernel on the
// transform route.
#include <string.h>
#include <algorithm>
#include "ctx.h"

using namespace stk;

// scratch slots of this file (ctx.h): the transform route's evaluations, and divmod's temporaries
static const int kSlotEvals = 12, kSlotDiv = 13;

static uint64_t pow2_at_least(uint64_t x) {
  uint64_t L = 1;
  while (L < x) L <<= 1;
  return L;
}

static bool overlaps(const void* x, uint64_t nx, const void* y, uint64_t ny) {
  if (!nx || !ny) return false;
  const uintptr_t x0 = (uintptr_t)x, y0 = (uintptr_t)y;
  return x0 < y0 + ny * sizeof(fe) && y0 < x0 + nx * sizeof(fe);
}

// Roots of unity of power-of-two order for the current modulus: w[s] = z^((p-1)/2^s) for
// s <= smax, z = 7 for the STARK prime (as everywhere else in the library) and otherwise the first
// z in [2, 64] with z^((p-1)/2) = -1.  w[1] = -1 gives every w[s] the exact order 2^s; without such
// a z only the trivial root w[0] = 1 exists and every longer product takes the direct route.
struct PolyRoots {
  int smax = 0;
  fe w[31];   // transforms are limited to 2^30
};

static PolyRoots poly_roots(stk_ctx* c) {
  PolyRoots R;
  const fe p = c->p, one = host::reduce(host::from_u64(1), p);
  R.w[0] = one;
  fe pm1;
  sub8(pm1.v, p.v, one.v);
  int v = 0;
  while (v < 30 && !((pm1.v[v >> 5] >> (v & 31)) & 1u)) ++v;
  if (v == 0) return R;
  fe e = pm1;   // (p-1) >> v
  for (int i = 0; i < 8; ++i) e.v[i] = (pm1.v[i] >> v) | (i < 7 && v ? pm1.v[i + 1] << (32 - v) : 0);
  for (uint64_t z = c->is_stark ? 7 : 2; z <= (c->is_stark ? 7 : 64); ++z) {
    fe w[31];
    w[v] = host::powmod(host::reduce(host::from_u64(z), p), e, p);
    for (int s = v; s > 1; --s) w[s - 1] = stk_h_mul(c, w[s], w[s]);
    if (fe_eq(w[1], pm1)) {
      for (int s = 1; s <= v; ++s) R.w[s] = w[s];
      R.smax = v;
      break;
    }
  }
  return R;
}

template <class F>
__global__ void poly_mul_direct_kernel(const fe* __restrict__ a, uint64_t na, const fe* __restrict__ b, uint64_t nb,
                                       fe* __restrict__ out, uint64_t nout, const F f) {
  const uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (k >= nout) return;
  const uint64_t i0 = k + 1 > nb ? k + 1 - nb : 0, i1 = k + 1 < na ? k + 1 : na;
  fe acc = fe_zero();
  for (uint64_t i = i0; i < i1; ++i) acc = f.add(acc, f.mul_tw(fe_load(a + i), fe_load(b + (k - i))));
  if constexpr (F::kMontgomery) acc = f.mul_tw(acc, f.r2);  // the sum of a_i b_j / R, times R
  fe_store(out + k, acc);
}

// One Newton step of the reciprocal on evaluations: G <- G (2 - F G)
template <class F>
__global__ void newton_recip_kernel(const fe* __restrict__ Fv, fe* __restrict__ G, uint64_t n, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe two = fe_zero();
  two.v[0] = 2;
  const fe g = fe_load(G + i);
  fe_store(G + i, f_mul(f, g, f.sub(two, f_mul(f, fe_load(Fv + i), g))));
}

// The same step's middle term on coefficients (direct route): t <- 2 - t
template <class F>
__global__ void two_minus_kernel(fe* t, uint64_t n, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe x = fe_zero();
  if (i == 0) x.v[0] = 2;
  fe_store(t + i, f.sub(x, fe_load(t + i)));
}

__global__ void reverse_kernel(const fe* __restrict__ src, uint64_t n, fe* __restrict__ dst) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) fe_store(dst + i, fe_load(src + (n - 1 - i)));
}

static unsigned blocks_for(uint64_t n, unsigned t) { return (unsigned)((n + t - 1) / t); }

static int reverse(stk_ctx* c, const fe* src, uint64_t n, fe* dst) {
  reverse_kernel<<<blocks_for(n, 256), 256, 0, c->stream>>>(src, n, dst);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

// Transforms are limited to 2^30 (ntt_api.cu); the STARK prime has roots of every order up to there,
// so only run-time moduli ever take the direct route.
static int check_length(stk_ctx* c, int s) {
  return s > 30 ? stk_fail(c, STK_EUNSUPPORTED, "polynomial product longer than 2^30") : STK_OK;
}

// out[0 .. nout) = (a * b) mod X^nout, zero beyond na + nb - 1; na, nb, nout >= 1; out overlaps
// neither input.
static int mul_low(stk_ctx* c, const PolyRoots& R, const fe* a, uint64_t na, const fe* b, uint64_t nb, fe* out,
                   uint64_t nout) {
  na = std::min(na, nout);
  nb = std::min(nb, nout);
  const uint64_t L = pow2_at_least(na + nb - 1);
  const int s = __builtin_ctzll(L);
  STK_TRY(check_length(c, s));
  if (s > R.smax) {
    poly_mul_direct_kernel<MontField><<<blocks_for(nout, 128), 128, 0, c->stream>>>(a, na, b, nb, out, nout, c->mont);
    STK_CUDA(c, cudaGetLastError());
    return STK_OK;
  }
  void* t;
  STK_TRY(stk_scratch(c, kSlotEvals, 2 * L * sizeof(fe), &t));
  fe* A = (fe*)t;
  fe* B = A + L;
  STK_TRY(stk_ntt_dev(c, a, na, na, A, L, L, 1, R.w[s], 0, 0));
  STK_TRY(stk_ntt_dev(c, b, nb, nb, B, L, L, 1, R.w[s], 0, 0));
  STK_TRY(stk_vec_op(c, 2, (const uint32_t*)A, (const uint32_t*)B, (uint32_t*)A, L));
  if (nout == L) return stk_ntt_dev(c, A, L, L, out, L, L, 1, R.w[s], 1, 1);
  STK_TRY(stk_ntt_dev(c, A, L, L, B, L, L, 1, R.w[s], 1, 1));
  const uint64_t m = std::min(nout, L);
  STK_CUDA(c, cudaMemcpyAsync(out, B, m * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
  if (nout > m) STK_CUDA(c, cudaMemsetAsync(out + m, 0, (nout - m) * sizeof(fe), c->stream));
  return STK_OK;
}

extern "C" __attribute__((visibility("default"))) int stk_poly_mul(stk_ctx* c, const uint32_t* d_a, uint64_t na,
                                                                    const uint32_t* d_b, uint64_t nb, uint32_t* d_out) {
  if (!c) return STK_EINVAL;
  if (!na || !nb) return STK_OK;
  if (!d_a || !d_b || !d_out) return stk_fail(c, STK_EINVAL, "null pointer");
  const uint64_t m = na + nb - 1;
  if (overlaps(d_out, m, d_a, na) || overlaps(d_out, m, d_b, nb))
    return stk_fail(c, STK_EINVAL, "the product must not overlap either factor");
  const PolyRoots R = poly_roots(c);
  return mul_low(c, R, (const fe*)d_a, na, (const fe*)d_b, nb, (fe*)d_out, m);
}

extern "C" __attribute__((visibility("default"))) int stk_poly_divmod(stk_ctx* c, const uint32_t* d_a, uint64_t na,
                                                                       const uint32_t* d_b, uint64_t nb, uint32_t* d_q,
                                                                       uint32_t* d_r) {
  if (!c) return STK_EINVAL;
  if (nb == 0 || !d_b) return stk_fail(c, STK_EINVAL, "the divisor has no coefficients");
  const uint64_t k = na >= nb ? na - nb + 1 : 0, nr = nb - 1;
  if ((na && !d_a) || (k && !d_q) || (nr && !d_r)) return stk_fail(c, STK_EINVAL, "null pointer");
  if (overlaps(d_q, k, d_a, na) || overlaps(d_q, k, d_b, nb) || overlaps(d_r, nr, d_a, na) ||
      overlaps(d_r, nr, d_b, nb) || overlaps(d_q, k, d_r, nr))
    return stk_fail(c, STK_EINVAL, "quotient and remainder must overlap neither each other nor an input");
  fe lead;
  STK_CUDA(c, cudaMemcpyAsync(&lead, d_b + 8 * (nb - 1), sizeof(fe), cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  lead = host::reduce(lead, c->p);
  const fe one = host::reduce(host::from_u64(1), c->p);
  const fe inv = stk_h_inv(c, lead);
  if (!fe_eq(stk_h_mul(c, lead, inv), one))
    return stk_fail(c, STK_EINVAL, "the divisor's leading coefficient is zero (or not invertible mod p)");
  const fe* a = (const fe*)d_a;
  const fe* b = (const fe*)d_b;
  if (k == 0) {  // deg a < deg b: q = 0, r = a
    if (na) STK_CUDA(c, cudaMemcpyAsync(d_r, a, na * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
    if (nr > na) STK_CUDA(c, cudaMemsetAsync((fe*)d_r + na, 0, (nr - na) * sizeof(fe), c->stream));
    return STK_OK;
  }
  const PolyRoots R = poly_roots(c);
  // f = rev(b) mod X^k, g = f^-1 mod X^k, ra = rev(a) mod X^k; t holds a product of length <= k
  const uint64_t nf = std::min(nb, k);
  void* scr;
  STK_TRY(stk_scratch(c, kSlotDiv, (nf + 3 * k) * sizeof(fe), &scr));
  fe* f = (fe*)scr;
  fe* g = f + nf;
  fe* ra = g + k;
  fe* t = ra + k;
  STK_TRY(reverse(c, b + (nb - nf), nf, f));
  STK_CUDA(c, cudaMemcpyAsync(g, &inv, sizeof(fe), cudaMemcpyHostToDevice, c->stream));
  for (uint64_t l = 1; l < k;) {  // g is f^-1 mod X^l; the step doubles l
    const uint64_t l2 = std::min(2 * l, k), nf2 = std::min(nf, l2);
    const uint64_t L = pow2_at_least(std::max(nf2 + 2 * l - 2, l2));  // g (2 - f g) in full: no wrap-around
    const int s = __builtin_ctzll(L);
    STK_TRY(check_length(c, s));
    if (s <= R.smax) {
      void* e;
      STK_TRY(stk_scratch(c, kSlotEvals, 2 * L * sizeof(fe), &e));
      fe* Fv = (fe*)e;
      fe* Gv = Fv + L;
      STK_TRY(stk_ntt_dev(c, f, nf2, nf2, Fv, L, L, 1, R.w[s], 0, 0));
      STK_TRY(stk_ntt_dev(c, g, l, l, Gv, L, L, 1, R.w[s], 0, 0));
      if (c->is_stark) newton_recip_kernel<StarkField><<<blocks_for(L, 256), 256, 0, c->stream>>>(Fv, Gv, L, StarkField());
      else newton_recip_kernel<MontField><<<blocks_for(L, 256), 256, 0, c->stream>>>(Fv, Gv, L, c->mont);
      STK_CUDA(c, cudaGetLastError());
      STK_TRY(stk_ntt_dev(c, Gv, L, L, Fv, L, L, 1, R.w[s], 1, 1));
      STK_CUDA(c, cudaMemcpyAsync(g + l, Fv + l, (l2 - l) * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
    } else {
      STK_TRY(mul_low(c, R, f, nf2, g, l, t, l2));
      two_minus_kernel<MontField><<<blocks_for(l2, 256), 256, 0, c->stream>>>(t, l2, c->mont);
      STK_CUDA(c, cudaGetLastError());
      STK_TRY(mul_low(c, R, g, l, t, l2, ra, l2));
      STK_CUDA(c, cudaMemcpyAsync(g + l, ra + l, (l2 - l) * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
    }
    l = l2;
  }
  // q = rev(rev(a) g mod X^k)
  STK_TRY(reverse(c, a + (na - k), k, ra));
  STK_TRY(mul_low(c, R, ra, k, g, k, t, k));
  STK_TRY(reverse(c, t, k, (fe*)d_q));
  // r = (a - b q) mod X^(nb-1)
  if (nr) {
    STK_TRY(mul_low(c, R, b, nb, (const fe*)d_q, k, (fe*)d_r, nr));
    STK_TRY(stk_vec_op(c, 1, d_a, d_r, d_r, nr));
  }
  return STK_OK;
}
