// poly.cu -- dense polynomial arithmetic in coefficient form: product and long division
// (Polynomial.__mul__ and Polynomial.__divmod__, starks/polynomial.py:110-143), composition a(b(X))
// (Polynomial.__call__ on a polynomial) and multivariate polynomials evaluated at polynomials
// (MultivariatePolynomial.__call__, starks/multivariate_polynomial.py:329-338), in O(n log n).
//
// Every product picks one of two routes from the modulus: the transform route (forward transforms
// of length L through stk_ntt_dev, a pointwise product, a scaled inverse) wherever Z/p has a root of
// unity of order L, and otherwise the direct route, one thread per output coefficient.  Division is
// Newton iteration on the reversed divisor, g <- g(2 - f g), fused into one pointwise kernel on the
// transform route.
#include <string.h>
#include <algorithm>
#include <vector>
#include "ctx.h"

using namespace stk;

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
  const fe p = c->p, one = stk_h_one(c);
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
  STK_TRY(stk_scratch(c, kSlotPolyEvals, 2 * L * sizeof(fe), &t));
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

STK_API int stk_poly_mul(stk_ctx* c, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                         uint32_t* d_out) {
  if (!c) return STK_EINVAL;
  if (!na || !nb) return STK_OK;
  if (!d_a || !d_b || !d_out) return stk_fail(c, STK_EINVAL, "null pointer");
  const uint64_t m = na + nb - 1;
  if (overlaps(d_out, m, d_a, na) || overlaps(d_out, m, d_b, nb))
    return stk_fail(c, STK_EINVAL, "the product must not overlap either factor");
  const PolyRoots R = poly_roots(c);
  return mul_low(c, R, (const fe*)d_a, na, (const fe*)d_b, nb, (fe*)d_out, m);
}

STK_API int stk_poly_divmod(stk_ctx* c, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                            uint32_t* d_q, uint32_t* d_r) {
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
  const fe inv = stk_h_inv(c, lead);
  if (!fe_eq(stk_h_mul(c, lead, inv), stk_h_one(c)))
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
  STK_TRY(stk_scratch(c, kSlotPolyDiv, (nf + 3 * k) * sizeof(fe), &scr));
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
      STK_TRY(stk_scratch(c, kSlotPolyEvals, 2 * L * sizeof(fe), &e));
      fe* Fv = (fe*)e;
      fe* Gv = Fv + L;
      STK_TRY(stk_ntt_dev(c, f, nf2, nf2, Fv, L, L, 1, R.w[s], 0, 0));
      STK_TRY(stk_ntt_dev(c, g, l, l, Gv, L, L, 1, R.w[s], 0, 0));
      STK_TRY(stk_with_field(c, [&](auto f) {
        newton_recip_kernel<<<blocks_for(L, 256), 256, 0, c->stream>>>(Fv, Gv, L, f);
      }));
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

// ---------------------------------------------------------------- composition a(b(X))

static const uint64_t kMaxOut = 1ull << 30;   // transforms are limited to 2^30 (ntt_api.cu)

// out[k] = a[k] alpha^k.  Each thread owns kScaleChunk coefficients: it raises alpha to its first
// index by square-and-multiply and multiplies along the chunk (alpha_tw in twiddle form).
static const int kScaleChunk = 16;
template <class F>
__global__ void scale_powers_kernel(const fe* __restrict__ a, uint64_t n, const fe alpha_tw, fe* __restrict__ out,
                                    const F f) {
  const uint64_t k0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) * kScaleChunk;
  if (k0 >= n) return;
  fe pw = f.one_tw();
  for (int bit = k0 ? 63 - __clzll(k0) : -1; bit >= 0; --bit) {
    pw = f.mul_tw(pw, pw);
    if ((k0 >> bit) & 1) pw = f.mul_tw(pw, alpha_tw);
  }
  for (uint64_t k = k0; k < n && k < k0 + kScaleChunk; ++k) {
    fe_store(out + k, f.mul_tw(fe_load(a + k), pw));
    pw = f.mul_tw(pw, alpha_tw);
  }
}

// Level 0 of the composition: chunk i = a_{2i} + a_{2i+1} b (nb coefficients), a zero past na.
template <class F>
__global__ void compose_level0_kernel(const fe* __restrict__ a, uint64_t na, const fe* __restrict__ b, uint64_t nb,
                                      fe* __restrict__ r, uint64_t nchunks, const F f) {
  const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (idx >= nchunks * nb) return;
  const uint64_t i = idx / nb, k = idx - i * nb;
  fe v = fe_zero();
  if (2 * i + 1 < na) v = f_mul(f, fe_load(a + 2 * i + 1), fe_load(b + k));
  if (k == 0 && 2 * i < na) v = f.add(v, fe_load(a + 2 * i));
  fe_store(r + idx, v);
}

// T[c*L + i] *= Bv[i*step] for every column c (L a power of two)
template <class F>
__global__ void mul_bcast_kernel(fe* __restrict__ T, uint64_t L, uint64_t total, const fe* __restrict__ Bv,
                                 uint64_t step, const F f) {
  const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  fe_store(T + idx, f_mul(f, fe_load(T + idx), fe_load(Bv + (idx & (L - 1)) * step)));
}

// out chunk i (nn coefficients) = T chunk i (stride ts) + previous chunk 2i (np coefficients)
template <class F>
__global__ void compose_combine_kernel(const fe* __restrict__ prev, uint64_t np, const fe* __restrict__ T, uint64_t ts,
                                       fe* __restrict__ out, uint64_t nn, uint64_t batch, const F f) {
  const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (idx >= batch * nn) return;
  const uint64_t i = idx / nn, k = idx - i * nn;
  fe v = fe_load(T + i * ts + k);
  if (k < np) v = f.add(v, fe_load(prev + 2 * i * np + k));
  fe_store(out + idx, v);
}

// `batch` transforms of length n (columns at in_stride, n_in coefficients each, zero-padded) into
// out at stride n; the inverse is scaled.  Multi-pass transforms take at most 65535 columns per
// launch (ntt.cuh), so large batches go in groups: stk_ntt_dev only groups transforms longer than
// 2048, and a run-time modulus already takes two passes at 2048 (1024-element tiles).
static int ntt_cols(stk_ctx* c, const fe* in, uint64_t n_in, uint64_t in_stride, fe* out, uint64_t n, uint64_t batch,
                    const fe& root, int inverse) {
  for (uint64_t b0 = 0; b0 < batch; b0 += 32768) {
    const uint64_t g = std::min<uint64_t>(batch - b0, 32768);
    STK_TRY(stk_ntt_dev(c, in + b0 * in_stride, n_in, in_stride, out + b0 * n, n, n, g, root, inverse, inverse));
  }
  return STK_OK;
}

// a(b(X)) for na >= 2, nb >= 2, bottom up: with a padded to N = 2^levels coefficients, level 0
// forms the N/2 chunks a_{2i} + a_{2i+1} b and level j >= 1 forms r_i <- r_{2i} + b^(2^j) r_{2i+1}.
// Below the top a level-j chunk has P_j = (2^(j+1) - 1)(nb - 1) + 1 coefficients; the top level
// writes only the nout the unpadded a has (the padding adds zeros above them).  On the transform
// route a level is one batched forward transform of the odd chunks, a product with the transform
// of b^(2^j) broadcast over the batch, one batched inverse and the add; b^(2^(j+1)) is the square
// of a transform of b^(2^j) long enough for it, whose even points are the level's own.  Without
// roots of the needed order a level runs through mul_low chunk by chunk.
static int compose_general(stk_ctx* c, const fe* a, uint64_t na, const fe* b, uint64_t nb, fe* out, uint64_t nout) {
  const PolyRoots R = poly_roots(c);
  const uint64_t d = nb - 1, N = pow2_at_least(na);
  const int levels = __builtin_ctzll(N);
  if (levels == 1) {
    return stk_with_field(c, [&](auto f) {
      compose_level0_kernel<<<blocks_for(nb, 256), 256, 0, c->stream>>>(a, na, b, nb, out, 1, f);
    });
  }
  auto chunk = [&](int j) -> uint64_t { return j + 1 == levels ? nout : ((2ull << j) - 1) * d + 1; };
  uint64_t cur_max = (N / 2) * nb, t_max = 0, b_max = 2 * d + 1;
  for (int j = 1; j < levels; ++j) {
    const uint64_t batch = N >> (j + 1), nbp = (1ull << j) * d + 1;
    const uint64_t L = pow2_at_least(chunk(j));
    if (j + 1 < levels) cur_max = std::max(cur_max, batch * chunk(j));
    t_max = std::max(t_max, batch * L);
    b_max = std::max(b_max, j + 1 < levels ? pow2_at_least(2 * nbp - 1) : L);
  }
  void* s1;
  void* s2;
  STK_TRY(stk_scratch(c, kSlotPolyA, 2 * cur_max * sizeof(fe), &s1));
  STK_TRY(stk_scratch(c, kSlotPolyB, (t_max + 2 * b_max) * sizeof(fe), &s2));
  fe* cur = (fe*)s1;
  fe* nxt = cur + cur_max;
  fe* T = (fe*)s2;
  fe* Bp = T + t_max;   // coefficients of b^(2^j)
  fe* Bv = Bp + b_max;  // its transform (product route: the next power)
  STK_TRY(stk_with_field(c, [&](auto f) {
    compose_level0_kernel<<<blocks_for((N / 2) * nb, 256), 256, 0, c->stream>>>(a, na, b, nb, cur, N / 2, f);
  }));
  STK_TRY(mul_low(c, R, b, nb, b, nb, Bp, 2 * d + 1));
  uint64_t np = nb;
  for (int j = 1; j < levels; ++j) {
    const bool top = j + 1 == levels;
    const uint64_t batch = N >> (j + 1), nn = chunk(j), nbp = (1ull << j) * d + 1;
    const uint64_t L = pow2_at_least(nn), Lb = top ? L : pow2_at_least(2 * nbp - 1);
    const int s = __builtin_ctzll(L), sb = __builtin_ctzll(Lb);
    fe* dst = top ? out : nxt;
    uint64_t ts = nn;
    if (sb <= R.smax) {
      ts = L;
      STK_TRY(ntt_cols(c, cur + np, np, 2 * np, T, L, batch, R.w[s], 0));
      STK_TRY(stk_ntt_dev(c, Bp, nbp, nbp, Bv, Lb, Lb, 1, R.w[sb], 0, 0));
      STK_TRY(stk_with_field(c, [&](auto f) {
        mul_bcast_kernel<<<blocks_for(batch * L, 256), 256, 0, c->stream>>>(T, L, batch * L, Bv, Lb / L, f);
      }));
      STK_TRY(ntt_cols(c, T, L, L, T, L, batch, R.w[s], 1));
      if (!top) {
        STK_TRY(stk_vec_op(c, 2, (const uint32_t*)Bv, (const uint32_t*)Bv, (uint32_t*)Bv, Lb));
        STK_TRY(stk_ntt_dev(c, Bv, Lb, Lb, Bp, Lb, Lb, 1, R.w[sb], 1, 1));
      }
    } else {
      for (uint64_t i = 0; i < batch; ++i) STK_TRY(mul_low(c, R, cur + (2 * i + 1) * np, np, Bp, nbp, T + i * nn, nn));
      if (!top) {
        STK_TRY(mul_low(c, R, Bp, nbp, Bp, nbp, Bv, 2 * nbp - 1));
        std::swap(Bp, Bv);
      }
    }
    STK_TRY(stk_with_field(c, [&](auto f) {
      compose_combine_kernel<<<blocks_for(batch * nn, 256), 256, 0, c->stream>>>(cur, np, T, ts, dst, nn, batch, f);
    }));
    std::swap(cur, nxt);
    np = nn;
  }
  return STK_OK;
}

STK_API int stk_poly_compose(stk_ctx* c, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                             uint32_t* d_out) {
  if (!c) return STK_EINVAL;
  if (nb < 2) return stk_fail(c, STK_EINVAL, "the inner polynomial needs at least two coefficients");
  if (!na) return STK_OK;
  if (!d_a || !d_b || !d_out) return stk_fail(c, STK_EINVAL, "null pointer");
  if (na - 1 > (kMaxOut - 1) / (nb - 1)) return stk_fail(c, STK_EUNSUPPORTED, "composition longer than 2^30");
  const uint64_t m = (na - 1) * (nb - 1) + 1;
  if (overlaps(d_out, m, d_a, na) || overlaps(d_out, m, d_b, nb))
    return stk_fail(c, STK_EINVAL, "the composition must not overlap either input");
  const fe* a = (const fe*)d_a;
  const fe* b = (const fe*)d_b;
  if (na == 1) {
    STK_CUDA(c, cudaMemcpyAsync(d_out, a, sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
    return STK_OK;
  }
  if (nb == 2) {  // b = alpha X: a pointwise scaling
    fe b01[2];
    STK_CUDA(c, cudaMemcpyAsync(b01, b, sizeof b01, cudaMemcpyDeviceToHost, c->stream));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
    if (fe_eq(host::reduce(b01[0], c->p), fe_zero())) {
      const fe alpha_tw = stk_h_to_tw(c, host::reduce(b01[1], c->p));
      const uint64_t threads = (na + kScaleChunk - 1) / kScaleChunk;
      return stk_with_field(c, [&](auto f) {
        scale_powers_kernel<<<blocks_for(threads, 256), 256, 0, c->stream>>>(a, na, alpha_tw, (fe*)d_out, f);
      });
    }
  }
  return compose_general(c, a, na, b, nb, (fe*)d_out, m);
}

// ---------------------------------------------------------------- multivariate evaluation

struct PolyMonomial {
  fe coeff_tw;        // coefficient in twiddle form
  uint32_t exp[12];   // exponent of each argument (width <= 12)
};

// One thread per evaluation point: the arguments' values are loaded once, every monomial is
// coeff * prod_k v_k^e_k with each power by left-to-right square-and-multiply (all in twiddle
// form).  Monomials of output j are monos[first[j] .. first[j+1]).
template <class F>
__global__ void __launch_bounds__(128) multivar_eval_kernel(const fe* __restrict__ A, uint64_t L, uint32_t width,
                                                            const PolyMonomial* __restrict__ monos,
                                                            const uint32_t* __restrict__ first, uint32_t nout,
                                                            fe* __restrict__ E, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= L) return;
  fe v[12];
  for (uint32_t k = 0; k < width; ++k) v[k] = f.to_tw(fe_load(A + k * L + i));
  for (uint32_t j = 0; j < nout; ++j) {
    fe acc = fe_zero();
    for (uint32_t m = first[j]; m < first[j + 1]; ++m) {
      fe term = monos[m].coeff_tw;
      for (uint32_t k = 0; k < width; ++k) {
        const uint32_t e = monos[m].exp[k];
        if (!e) continue;
        fe r = v[k];
        for (int bit = 30 - __clz((int)e); bit >= 0; --bit) {
          r = f.mul_tw(r, r);
          if ((e >> bit) & 1) r = f.mul_tw(r, v[k]);
        }
        term = f.mul_tw(term, r);
      }
      acc = f.add(acc, term);
    }
    fe_store(E + j * L + i, f.from_tw(acc));
  }
}

// Product route of stk_poly_eval_multivar (no root of order L): every monomial from mul_low
// products, powers by left-to-right square-and-multiply; out column j accumulates its monomials.
// W holds 3 * (D+1) elements of workspace, h_coeffs the canonical coefficients on the device.
static int multivar_products(stk_ctx* c, const fe* polys, const uint64_t* lens, uint64_t in_stride, uint64_t width,
                             const uint32_t* h_out, const fe* d_coeffs, const uint32_t* h_exps,
                             const std::vector<uint64_t>& order, fe* out, uint64_t out_len, fe* W) {
  const PolyRoots R = poly_roots(c);
  fe* term = W;
  fe* pw = W + out_len;
  fe* tmp = pw + out_len;
  for (uint64_t m : order) {
    STK_CUDA(c, cudaMemcpyAsync(term, d_coeffs + m, sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
    uint64_t nt = 1;
    for (uint64_t k = 0; k < width; ++k) {
      const uint32_t e = h_exps[m * width + k];
      if (!e) continue;
      const fe* x = polys + k * in_stride;
      const uint64_t nx = lens[k];
      STK_CUDA(c, cudaMemcpyAsync(pw, x, nx * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
      uint64_t np = nx;
      for (int bit = 30 - __builtin_clz(e); bit >= 0; --bit) {
        STK_TRY(mul_low(c, R, pw, np, pw, np, tmp, 2 * np - 1));
        np = 2 * np - 1;
        if ((e >> bit) & 1) {
          STK_TRY(mul_low(c, R, tmp, np, x, nx, pw, np + nx - 1));
          np += nx - 1;
        } else {
          STK_CUDA(c, cudaMemcpyAsync(pw, tmp, np * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
        }
      }
      STK_TRY(mul_low(c, R, term, nt, pw, np, tmp, nt + np - 1));
      nt += np - 1;
      std::swap(term, tmp);
    }
    fe* col = out + h_out[m] * out_len;
    STK_TRY(stk_vec_op(c, 0, (const uint32_t*)col, (const uint32_t*)term, (uint32_t*)col, nt));
  }
  return STK_OK;
}

STK_API int stk_poly_eval_multivar(stk_ctx* c, const uint32_t* d_polys, const uint64_t* h_lens, uint64_t in_stride,
                                   uint64_t width, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                                   const uint32_t* h_mono_exps, uint64_t nmono, uint64_t nout, uint32_t* d_out,
                                   uint64_t out_len) {
  if (!c) return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "width must be in 1..12");
  if (!h_lens || (nmono && (!h_mono_out || !h_mono_coeffs || !h_mono_exps)))
    return stk_fail(c, STK_EINVAL, "null pointer");
  if (nout > 0xffffffffull) return stk_fail(c, STK_EUNSUPPORTED, "too many outputs");
  uint64_t maxlen = 0;
  for (uint64_t k = 0; k < width; ++k) maxlen = std::max(maxlen, h_lens[k]);
  if (maxlen && !d_polys) return stk_fail(c, STK_EINVAL, "null pointer");
  // D = max over the monomials that do not vanish of sum_k e_k (len_k - 1)
  unsigned __int128 D = 0;
  for (uint64_t m = 0; m < nmono; ++m) {
    if (h_mono_out[m] >= nout) return stk_fail(c, STK_EINVAL, "monomial output index out of range");
    unsigned __int128 deg = 0;
    bool vanishes = false;
    for (uint64_t k = 0; k < width; ++k) {
      const uint32_t e = h_mono_exps[m * width + k];
      if (e && !h_lens[k]) vanishes = true;
      else if (e) deg += (unsigned __int128)e * (h_lens[k] - 1);
    }
    if (!vanishes) D = std::max(D, deg);
  }
  if (D + 1 > kMaxOut) return stk_fail(c, STK_EUNSUPPORTED, "evaluation longer than 2^30");
  if (out_len != (uint64_t)D + 1) return stk_fail(c, STK_EINVAL, "out_len must be D + 1 = %llu", (unsigned long long)D + 1);
  if (!nout) return STK_OK;
  if (!d_out) return stk_fail(c, STK_EINVAL, "null pointer");
  if (nout > (1ull << 62) / out_len) return stk_fail(c, STK_EUNSUPPORTED, "output too large");
  for (uint64_t k = 0; k < width; ++k)
    if (overlaps(d_out, nout * out_len, d_polys + 8 * k * in_stride, h_lens[k]))
      return stk_fail(c, STK_EINVAL, "the outputs must not overlap an argument");
  // monomials grouped by output (stable), the ones that vanish dropped
  std::vector<uint64_t> order;
  std::vector<uint32_t> first(nout + 1, 0);
  for (uint64_t m = 0; m < nmono; ++m) {
    bool vanishes = false;
    for (uint64_t k = 0; k < width; ++k) vanishes |= h_mono_exps[m * width + k] && !h_lens[k];
    if (!vanishes) {
      order.push_back(m);
      ++first[h_mono_out[m] + 1];
    }
  }
  std::stable_sort(order.begin(), order.end(), [&](uint64_t x, uint64_t y) { return h_mono_out[x] < h_mono_out[y]; });
  for (uint64_t j = 0; j < nout; ++j) first[j + 1] += first[j];
  const uint64_t L = pow2_at_least(out_len);
  const int s = __builtin_ctzll(L);
  const PolyRoots R = poly_roots(c);
  fe* out = (fe*)d_out;
  if (s > R.smax) {
    std::vector<fe> coeffs(nmono ? nmono : 1);
    for (uint64_t m = 0; m < nmono; ++m) coeffs[m] = host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p);
    const uint64_t coeff_bytes = coeffs.size() * sizeof(fe);
    void* w;
    void* cf;
    STK_TRY(stk_scratch(c, kSlotPolyA, 3 * out_len * sizeof(fe), &w));
    STK_TRY(stk_stage(c, kSlotPolyB, coeff_bytes, {{0, coeffs.data(), coeff_bytes}}, &cf));
    STK_CUDA(c, cudaMemsetAsync(out, 0, nout * out_len * sizeof(fe), c->stream));
    return multivar_products(c, (const fe*)d_polys, h_lens, in_stride, width, h_mono_out, (const fe*)cf, h_mono_exps,
                             order, out, out_len, (fe*)w);
  }
  // transform route: the arguments (cut to L coefficients: a longer one appears with exponent 0
  // only) staged at one stride with zero padding, one batched forward, the pointwise kernel, one
  // batched scaled inverse
  const uint64_t ms = std::max<uint64_t>(std::min(maxlen, L), 1);
  std::vector<PolyMonomial> hm(order.size() ? order.size() : 1);
  for (size_t t = 0; t < order.size(); ++t) {
    const uint64_t m = order[t];
    hm[t].coeff_tw = stk_h_to_tw(c, host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p));
    for (uint64_t k = 0; k < 12; ++k) hm[t].exp[k] = k < width ? h_mono_exps[m * width + k] : 0;
  }
  const uint64_t stage_bytes = width * ms * sizeof(fe), mono_bytes = hm.size() * sizeof(PolyMonomial);
  const uint64_t first_bytes = first.size() * sizeof(uint32_t);
  void* s1;
  void* s2;
  STK_TRY(stk_scratch(c, kSlotPolyA, (width + nout) * L * sizeof(fe), &s1));
  STK_TRY(stk_stage(c, kSlotPolyB, stage_bytes + mono_bytes + first_bytes,
                    {{stage_bytes, hm.data(), mono_bytes}, {stage_bytes + mono_bytes, first.data(), first_bytes}},
                    &s2));
  fe* Av = (fe*)s1;
  fe* E = Av + width * L;
  fe* stage = (fe*)s2;
  const PolyMonomial* d_monos = (const PolyMonomial*)((char*)s2 + stage_bytes);
  const uint32_t* d_first = (const uint32_t*)((char*)s2 + stage_bytes + mono_bytes);
  STK_CUDA(c, cudaMemsetAsync(stage, 0, stage_bytes, c->stream));
  for (uint64_t k = 0; k < width; ++k) {
    const uint64_t nk = std::min(h_lens[k], ms);
    if (nk)
      STK_CUDA(c, cudaMemcpyAsync(stage + k * ms, (const fe*)d_polys + k * in_stride, nk * sizeof(fe),
                                  cudaMemcpyDeviceToDevice, c->stream));
  }
  STK_TRY(ntt_cols(c, stage, ms, ms, Av, L, width, R.w[s], 0));
  STK_TRY(stk_with_field(c, [&](auto f) {
    multivar_eval_kernel<<<blocks_for(L, 128), 128, 0, c->stream>>>(Av, L, (uint32_t)width, d_monos, d_first,
                                                                    (uint32_t)nout, E, f);
  }));
  STK_TRY(ntt_cols(c, E, L, L, E, L, nout, R.w[s], 1));
  for (uint64_t j = 0; j < nout; ++j)
    STK_CUDA(c, cudaMemcpyAsync(out + j * out_len, E + j * L, out_len * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
  return STK_OK;
}
