// stark.cu -- the prover's polynomial constructions between the commitments, in
// O(n log n) evaluation/NTT form.  The reference builds them in coefficient form with
// O(n^2) Horner composition and schoolbook long division (starks/stark.py:38-104,
// starks/polynomial.py:128-143); arithmetic is exact mod p, so the polynomials -- and hence
// every committed evaluation -- are identical (SURVEY.md App. C.1-C.2).
//
//   constraint evaluations   C_j(x_i) = P_j(G1*x_i) - step_j(P_1(x_i), ..., P_w(x_i))
//                            with P_j(G1*x_i) = Pev_j[(i+ext) mod N]        (stark.py:38-55)
//   quotient by Z            D_j = C_j*(X-last) / (X^steps - 1)             (stark.py:57-78)
//   division by X - r        quotient coefficients as geometric suffix sums (stark.py:80-104,
//                            B_j = (P_j - I_j) / ((X-1)(X-last)))
//   linear combination       l = sum_c weight_c * column_c                  (stark.py:130-177)
#include <vector>
#include "ctx.h"

using namespace stk;

namespace {

struct Monomial {
  fe coeff_tw;       // coefficient in twiddle form
  uint32_t out;      // which constraint it belongs to
  uint8_t exp[12];   // exponent of each state variable (width <= 12)
};

// step_j(P_1(x_i), ..., P_w(x_i)) from the state in twiddle form: every monomial of output j is
// coeff * prod_k P_k^e_k by repeated multiplication (degrees are tiny: <= extension factor).
template <class F>
__device__ __forceinline__ fe step_poly(const Monomial* __restrict__ monos, uint32_t nmono, uint32_t width, uint32_t j,
                                        const fe* st_tw, const F& f) {
  fe acc = fe_zero();
  for (uint32_t m = 0; m < nmono; ++m) {
    if (monos[m].out != j) continue;
    fe term = f.from_tw(monos[m].coeff_tw);  // plain coefficient
    for (uint32_t k = 0; k < width; ++k)
      for (uint32_t e = 0; e < monos[m].exp[k]; ++e) term = f.mul_tw(term, st_tw[k]);
    acc = f.add(acc, term);
  }
  return acc;
}

// One thread per evaluation point; the state values P_k(x_i) are loaded once.
template <class F>
__global__ void __launch_bounds__(128) constraint_eval_kernel(const fe* __restrict__ pev, uint64_t n, uint64_t ext,
                                                              uint32_t width, uint64_t col_stride,
                                                              const Monomial* __restrict__ monos, uint32_t nmono,
                                                              fe* __restrict__ cev, uint64_t out_stride, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe st[12], st_tw[12];
  for (uint32_t k = 0; k < width; ++k) {
    st[k] = fe_load(pev + k * col_stride + i);
    st_tw[k] = f.to_tw(st[k]);
  }
  const uint64_t inext = (i + ext) % n;
  for (uint32_t j = 0; j < width; ++j) {
    const fe acc = step_poly(monos, nmono, width, j, st_tw, f);
    fe nxt = fe_load(pev + j * col_stride + inext);
    fe_store(cev + j * out_stride + i, f.sub(nxt, acc));
  }
}

// D = C / Z on the evaluation domain itself (x_i = G2^i), pointwise wherever Z(x_i) != 0:
// Z(x) = (x^steps - 1)/(x - last) and x_i^steps = omega^(i mod ext) (omega = G2^steps has order
// ext), so D(x_i) = C(x_i) * (x_i - last) * inv[i mod ext] with the ext-1 constants
// inv[r] = (omega^r - 1)^-1.  At i = 0 mod ext both C and Z vanish; those values (D on the
// subgroup <G1>) come from D's coefficients through a small transform (dsub).  Replaces the
// size-N transform of D for 7/8 of the points.
struct QuotInv { fe v[16]; };  // inv[r] plain, r < ext <= 16
template <class F>
__global__ void __launch_bounds__(128) quotient_eval_kernel(const fe* __restrict__ pev, uint64_t n, uint64_t ext,
                                                            uint32_t width, uint64_t col_stride,
                                                            const Monomial* __restrict__ monos, uint32_t nmono,
                                                            const fe* __restrict__ X, int xshift, fe last_tw,
                                                            const QuotInv inv, const fe* __restrict__ dsub,
                                                            uint64_t dsub_stride, uint64_t sub_step,
                                                            fe* __restrict__ dev, uint64_t out_stride, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t r = i % ext;
  if (r == 0) {
    const uint64_t k = (i / ext) * sub_step;
    for (uint32_t j = 0; j < width; ++j) fe_store(dev + j * out_stride + i, fe_load(dsub + j * dsub_stride + k));
    return;
  }
  fe st_tw[12];
  for (uint32_t k = 0; k < width; ++k) st_tw[k] = f.to_tw(fe_load(pev + k * col_stride + i));
  const uint64_t inext = (i + ext) % n;
  // (x_i - last) * inv[r], back in twiddle form for the final product
  const fe xm = f.sub(fe_load_ro(X + (i << xshift)), last_tw);
  const fe fac_tw = f.to_tw(f.mul_tw(inv.v[r], xm));
  for (uint32_t j = 0; j < width; ++j) {
    const fe acc = step_poly(monos, nmono, width, j, st_tw, f);
    const fe cval = f.sub(fe_load(pev + j * col_stride + inext), acc);
    fe_store(dev + j * out_stride + i, f.mul_tw(cval, fac_tw));
  }
}

// ---- B = (P - I) / ((X - 1)(X - last)) on the evaluation domain, pointwise (STARK prime) ----
// 1/(x_i - a) for a = G2^e in the domain is a^-1 * T[(i - e) mod n] with ONE cached table
// T[i] = (G2^i - 1)^-1, i >= 1 (built once per (G2, n) by chunked batch inversion).
constexpr int kInvChunk = 32;
__device__ __forceinline__ fe stark_inv(const StarkField& f, const fe& a) {  // a^(p-2)
  fe e = StarkField::modulus();  // limbs {1, 0xFFFFFEA1, ...}: p - 2 borrows out of limb 0
  e.v[0] = 0xFFFFFFFFu;
  e.v[1] -= 1u;
  fe r = fe_zero();
  r.v[0] = 1;
  fe base = a;
  for (int i = 0; i < 256; ++i) {
    if ((e.v[i >> 5] >> (i & 31)) & 1u) r = f.mul_tw(r, base);
    base = f.mul_tw(base, base);
  }
  return r;
}
// T[i] = (X[i] - 1)^-1 for i in [1, n); T[0] = 0.  One thread per chunk of kInvChunk entries:
// prefix products parked in T itself, one inversion, then the backward sweep (Montgomery's trick).
__global__ void __launch_bounds__(128) invtable_kernel(const fe* __restrict__ X, int xshift, uint64_t n, fe* __restrict__ T) {
  const StarkField f;
  const uint64_t c0 = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) * kInvChunk;
  if (c0 >= n) return;
  const uint64_t c1 = c0 + kInvChunk < n ? c0 + kInvChunk : n;
  fe one = fe_zero();
  one.v[0] = 1;
  fe acc = one;
  for (uint64_t i = c0; i < c1; ++i) {
    const fe v = i ? f.sub(fe_load_ro(X + (i << xshift)), one) : one;
    acc = f.mul_tw(acc, v);
    fe_store(T + i, acc);
  }
  fe inv = stark_inv(f, acc);
  for (uint64_t i = c1; i-- > c0;) {
    const fe v = i ? f.sub(fe_load_ro(X + (i << xshift)), one) : one;
    const fe prev = i > c0 ? fe_load(T + i - 1) : one;
    fe_store(T + i, i ? f.mul_tw(inv, prev) : fe_zero());
    inv = f.mul_tw(inv, v);
  }
}
struct BoundaryInterp { fe i0[12], i1[12]; };
__global__ void __launch_bounds__(128) boundary_eval_kernel(const fe* __restrict__ pev, uint64_t n, uint64_t ext, uint32_t width,
                                                            uint64_t col_stride, const fe* __restrict__ X, int xshift,
                                                            const fe* __restrict__ T, uint64_t last_index, fe last_inv,
                                                            const BoundaryInterp I, const fe* __restrict__ bsub,
                                                            uint64_t bsub_stride, fe* __restrict__ bev, uint64_t out_stride) {
  const StarkField f;
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (i % ext == 0) {
    for (uint32_t j = 0; j < width; ++j) fe_store(bev + j * out_stride + i, fe_load(bsub + j * bsub_stride + i / ext));
    return;
  }
  const fe x = fe_load_ro(X + (i << xshift));
  const uint64_t il = i >= last_index ? i - last_index : i + n - last_index;  // != 0: last_index is a multiple of ext
  // 1/((x - 1)(x - last)) = T[i] * last^-1 * T[i - last_index]
  const fe inv = f.mul_tw(f.mul_tw(fe_load(T + i), fe_load(T + il)), last_inv);
  for (uint32_t j = 0; j < width; ++j) {
    const fe ix = f.add(I.i0[j], f.mul_tw(I.i1[j], x));
    const fe num = f.sub(fe_load(pev + j * col_stride + i), ix);
    fe_store(bev + j * out_stride + i, f.mul_tw(num, inv));
  }
}

// E = C*(X - last) has coefficients e[i] = c[i-1] - last*c[i] (c[-1] = c[n] = 0, i <= n).
template <class F>
__device__ __forceinline__ fe e_coeff(const fe* c, uint64_t n, uint64_t i, const fe& last_tw, const F& f) {
  fe lo = (i >= 1 && i - 1 < n) ? fe_load(c + i - 1) : fe_zero();
  fe hi = (i < n) ? f.mul_tw(fe_load(c + i), last_tw) : fe_zero();
  return f.sub(lo, hi);
}

// D = E / (X^steps - 1): d[i] = e[i+steps] + d[i+steps], high to low; one thread per
// residue r = i mod steps walks its chain (length n/steps).  Remainder e[r] + d[r] must be 0
// (the reference asserts `cp % z == 0`, stark.py:74-75): violations are counted.
template <class F>
__global__ void __launch_bounds__(256) quotient_z_kernel(const fe* __restrict__ c, uint64_t n, uint64_t steps,
                                                         fe last_tw, fe* __restrict__ d, uint32_t* __restrict__ bad,
                                                         const F f) {
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (r >= steps) return;
  const uint64_t chain = n / steps;  // e has n+1 coefficients: indices r + m*steps, m <= chain (only r = 0 reaches n)
  fe acc = fe_zero();                // d[r + m*steps] for the m above
  // top: indices i = r + m*steps with i + steps > n have d[i] = 0
  for (uint64_t m = chain; m-- > 0;) {
    const uint64_t i = r + m * steps;  // computing d[i] = e[i+steps] + d[i+steps]
    fe e = (i + steps <= n) ? e_coeff(c, n, i + steps, last_tw, f) : fe_zero();
    acc = f.add(e, acc);
    fe_store(d + i, acc);
  }
  fe rem = f.add(e_coeff(c, n, r, last_tw, f), acc);
  if (!fe_is_zero(rem)) atomicAdd(bad, 1u);
}

// ---- geometric suffix sums: out[k] = sum_{i>k} a[i] * r^(i-k-1),  k < n-1 ------------------
// With a'[i] = a[i]*r^i this is r^-(k+1) * S[k], S the exclusive suffix sum of a'.
constexpr int kScanChunk = 8;      // elements per thread
constexpr int kScanThreads = 256;  // threads per block -> 2048 elements per block

template <class F>
__device__ __forceinline__ fe scan_load(const fe* a, const fe* rpow, uint64_t rs, uint64_t n, uint64_t i, const F& f) {
  if (i >= n) return fe_zero();
  fe v = fe_load(a + i);
  return rpow ? f.mul_tw(v, fe_load_ro(rpow + i * rs)) : v;
}

// phase 1: block totals
template <class F>
__global__ void __launch_bounds__(kScanThreads) scan_block_totals_kernel(const fe* __restrict__ a, const fe* __restrict__ rpow,
                                                                         uint64_t rs, uint64_t n, fe* __restrict__ totals, const F f) {
  __shared__ fe sh[kScanThreads];
  const uint64_t base = ((uint64_t)blockIdx.x * kScanThreads + threadIdx.x) * kScanChunk;
  fe s = fe_zero();
#pragma unroll
  for (int u = 0; u < kScanChunk; ++u) s = f.add(s, scan_load(a, rpow, rs, n, base + u, f));
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int off = kScanThreads / 2; off > 0; off >>= 1) {
    if (threadIdx.x < off) sh[threadIdx.x] = f.add(sh[threadIdx.x], sh[threadIdx.x + off]);
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = sh[0];
}

// phase 2: exclusive suffix scan of the block totals, one CTA: each thread walks a contiguous
// chunk, a Hillis-Steele suffix scan combines the chunk sums, then the chunk is rewritten.
template <class F>
__global__ void __launch_bounds__(kScanThreads) scan_totals_kernel(fe* totals, uint64_t nblocks, const F f) {
  __shared__ fe sh[kScanThreads];
  const uint64_t per = (nblocks + kScanThreads - 1) / kScanThreads;
  const uint64_t lo = threadIdx.x * per, hi = (lo + per < nblocks) ? lo + per : nblocks;
  fe s = fe_zero();
  for (uint64_t b = lo; b < hi; ++b) s = f.add(s, totals[b]);
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < kScanThreads; off <<= 1) {
    fe t = fe_zero();
    bool has = threadIdx.x + off < kScanThreads;
    if (has) t = sh[threadIdx.x + off];
    __syncthreads();
    if (has) sh[threadIdx.x] = f.add(sh[threadIdx.x], t);
    __syncthreads();
  }
  fe run = (threadIdx.x + 1 < kScanThreads) ? sh[threadIdx.x + 1] : fe_zero();  // all chunks after mine
  for (uint64_t b = hi; b-- > lo;) {
    fe t = totals[b];
    totals[b] = run;  // sum of all blocks after b
    run = f.add(run, t);
  }
}

// phase 3: exclusive suffix sums inside each block + block offset, then unscale
template <class F>
__global__ void __launch_bounds__(kScanThreads) scan_finish_kernel(const fe* __restrict__ a, const fe* __restrict__ rpow, uint64_t rs,
                                                                   const fe* __restrict__ rinvpow, uint64_t ris, uint64_t n,
                                                                   const fe* __restrict__ totals, fe* __restrict__ out,
                                                                   const F f) {
  __shared__ fe sh[kScanThreads];
  const uint64_t base = ((uint64_t)blockIdx.x * kScanThreads + threadIdx.x) * kScanChunk;
  fe v[kScanChunk];
  fe s = fe_zero();
#pragma unroll
  for (int u = 0; u < kScanChunk; ++u) { v[u] = scan_load(a, rpow, rs, n, base + u, f); s = f.add(s, v[u]); }
  sh[threadIdx.x] = s;
  __syncthreads();
  // inclusive suffix scan over thread sums (Hillis-Steele)
  for (int off = 1; off < kScanThreads; off <<= 1) {
    fe t = fe_zero();
    bool has = threadIdx.x + off < kScanThreads;
    if (has) t = sh[threadIdx.x + off];
    __syncthreads();
    if (has) sh[threadIdx.x] = f.add(sh[threadIdx.x], t);
    __syncthreads();
  }
  // sum of everything after this thread's chunk
  fe after = (threadIdx.x + 1 < kScanThreads) ? sh[threadIdx.x + 1] : fe_zero();
  after = f.add(after, totals[blockIdx.x]);
  // walk the chunk from its top: S[k] = sum_{i>k} a'[i]
#pragma unroll
  for (int u = kScanChunk - 1; u >= 0; --u) {
    const uint64_t k = base + u;
    if (k + 1 < n) {
      fe r = after;
      if (rinvpow) r = f.mul_tw(r, fe_load_ro(rinvpow + ((k + 1) % n) * ris));  // r^-(k+1)
      fe_store(out + k, r);
    }
    after = f.add(after, v[u]);
  }
}

template <class F>
__global__ void __launch_bounds__(256) lincomb_kernel(const fe* __restrict__ cols, uint64_t n, uint32_t ncols,
                                                      uint64_t col_stride, const fe* __restrict__ weights_tw,
                                                      fe* __restrict__ out, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe acc = fe_zero();
  for (uint32_t c = 0; c < ncols; ++c)
    acc = f.add(acc, f.mul_tw(fe_load(cols + c * col_stride + i), fe_load_ro(weights_tw + c)));
  fe_store(out + i, acc);
}

// The monomial list of the step polynomials: for monomial m, out[m] = constraint index,
// coeffs[8*m..] = coefficient limbs (canonical), exps[width*m + k] = exponent of X_{k+1}.
int pack_monomials(stk_ctx* c, uint64_t width, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                   const uint8_t* h_mono_exps, uint64_t nmono, std::vector<Monomial>& ms) {
  ms.resize(nmono ? nmono : 1);
  for (uint64_t m = 0; m < nmono; ++m) {
    if (h_mono_out[m] >= width) return stk_fail(c, STK_EINVAL, "monomial output index out of range");
    ms[m].coeff_tw = stk_h_to_tw(c, host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p));
    ms[m].out = h_mono_out[m];
    for (uint64_t k = 0; k < 12; ++k) ms[m].exp[k] = k < width ? h_mono_exps[width * m + k] : 0;
  }
  return STK_OK;
}

}  // namespace

// step polynomials as a monomial list (pack_monomials)
STK_API int stk_constraint_eval(stk_ctx* c, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                                uint64_t col_stride, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                                const uint8_t* h_mono_exps, uint64_t nmono, uint32_t* d_cev, uint64_t out_stride) {
  if (!c || !d_pev || !d_cev || (!nmono ? false : (!h_mono_out || !h_mono_coeffs || !h_mono_exps))) return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  std::vector<Monomial> ms;
  STK_TRY(pack_monomials(c, width, h_mono_out, h_mono_coeffs, h_mono_exps, nmono, ms));
  const uint64_t mono_bytes = ms.size() * sizeof(Monomial);
  void* t;
  STK_TRY(stk_stage(c, kSlotStage, mono_bytes, {{0, ms.data(), mono_bytes}}, &t));
  unsigned blocks = (unsigned)((n + 127) / 128);
  return stk_with_field(c, [&](auto f) {
    constraint_eval_kernel<<<blocks, 128, 0, c->stream>>>((const fe*)d_pev, n, ext, (uint32_t)width, col_stride,
                                                          (const Monomial*)t, (uint32_t)nmono, (fe*)d_cev, out_stride,
                                                          f);
  });
}

// construct_remainder_polynomials (stark.py:57-78) in evaluation form on the size-n domain <g2>:
// d_dev[j][i] = D_j(g2^i) from the trace evaluations d_pev (n per column) wherever Z does not
// vanish, and from d_dsub (D_j on a subgroup of order sub_n containing <g2^ext>, e.g. the forward
// transform of D's coefficients) at i = 0 mod ext.  ext <= 16.
STK_API int stk_quotient_eval(stk_ctx* c, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                              uint64_t col_stride, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                              const uint8_t* h_mono_exps, uint64_t nmono, const uint32_t g2[8], const uint32_t last[8],
                              const uint32_t* d_dsub, uint64_t sub_n, uint64_t dsub_stride, uint32_t* d_dev,
                              uint64_t out_stride) {
  if (!c || !d_pev || !d_dev || !d_dsub || !g2 || !last || (nmono && (!h_mono_out || !h_mono_coeffs || !h_mono_exps)))
    return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  if (ext < 2 || ext > 16 || n % ext) return stk_fail(c, STK_EUNSUPPORTED, "extension factor must be in 2..16 and divide n");
  const uint64_t steps = n / ext;
  if (sub_n == 0 || sub_n % steps) return stk_fail(c, STK_EINVAL, "d_dsub must cover a subgroup containing <g2^ext>");
  std::vector<Monomial> ms;
  STK_TRY(pack_monomials(c, width, h_mono_out, h_mono_coeffs, h_mono_exps, nmono, ms));
  const fe G2 = host::reduce(stk_load_fe(g2), c->p);
  const fe one = stk_h_one(c);
  if (!fe_eq(stk_h_pow(c, G2, n), one)) return stk_fail(c, STK_EINVAL, "g2^n != 1");
  const fe omega = stk_h_pow(c, G2, steps);
  QuotInv inv;
  for (int r = 0; r < 16; ++r) inv.v[r] = fe_zero();
  fe wr = omega;
  for (uint64_t r = 1; r < ext; ++r) {
    fe den = host::submod(wr, one, c->p);
    if (fe_is_zero(den)) return stk_fail(c, STK_EINVAL, "g2^steps has order below ext");
    inv.v[r] = stk_h_inv(c, den);
    wr = stk_h_mul(c, wr, omega);
  }
  const fe* X;
  int xshift;
  STK_TRY(stk_get_table_shift(c, G2, n, &X, &xshift));
  const uint64_t mono_bytes = ms.size() * sizeof(Monomial);
  void* t;
  STK_TRY(stk_stage(c, kSlotStage, mono_bytes, {{0, ms.data(), mono_bytes}}, &t));
  const fe last_tw = stk_h_to_tw(c, host::reduce(stk_load_fe(last), c->p));
  unsigned blocks = (unsigned)((n + 127) / 128);
  return stk_with_field(c, [&](auto f) {
    quotient_eval_kernel<<<blocks, 128, 0, c->stream>>>((const fe*)d_pev, n, ext, (uint32_t)width, col_stride,
                                                        (const Monomial*)t, (uint32_t)nmono, X, xshift, last_tw, inv,
                                                        (const fe*)d_dsub, dsub_stride, sub_n / steps, (fe*)d_dev,
                                                        out_stride, f);
  });
}

// construct_boundary_polynomials (stark.py:80-104) in evaluation form on the size-n domain <g2>
// (STARK prime only): d_bev[j][i] = (P_j(x_i) - (i0_j + i1_j x_i)) / ((x_i - 1)(x_i - last)) with
// last = g2^last_index (a multiple of ext), pointwise wherever the denominator is non-zero; the
// values at i = 0 mod ext come from d_bsub = B_j on <g2^ext> (transform of B's coefficients).
void stk_stark_release(stk_ctx* c) {
  for (auto& t : c->invtables) cudaFree(t.d);
  c->invtables.clear();
}
STK_API int stk_boundary_eval(stk_ctx* c, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                              uint64_t col_stride, const uint32_t g2[8], uint64_t last_index, const uint32_t* h_interp,
                              const uint32_t* d_bsub, uint64_t bsub_stride, uint32_t* d_bev, uint64_t out_stride) {
  if (!c || !d_pev || !d_bev || !d_bsub || !g2 || !h_interp) return STK_EINVAL;
  if (!c->is_stark) return stk_fail(c, STK_EUNSUPPORTED, "pointwise boundary quotient is built for the STARK prime");
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  if (ext < 2 || n % ext || last_index % ext || last_index >= n || last_index == 0)
    return stk_fail(c, STK_EINVAL, "last_index must be a non-zero multiple of ext below n");
  const fe G2 = host::reduce(stk_load_fe(g2), c->p);
  if (!stk_h_primitive(c, G2, n)) return stk_fail(c, STK_EINVAL, "g2 is not a primitive n-th root of unity");
  const fe* X;
  int xshift;
  STK_TRY(stk_get_table_shift(c, G2, n, &X, &xshift));
  // per-context cache (least recently used first), bounded by kInvTableCacheBytes; only this
  // context's own stream can still be reading an evicted table, and it is synchronised first
  fe* T = nullptr;
  for (size_t i = 0; i < c->invtables.size(); ++i)
    if (c->invtables[i].n == n && fe_eq(c->invtables[i].root, G2)) {
      stk_invtable t = c->invtables[i];
      c->invtables.erase(c->invtables.begin() + i);
      c->invtables.push_back(t);
      T = t.d;
      break;
    }
  if (!T) {
    uint64_t held = 0;
    for (auto& t : c->invtables) held += t.n * sizeof(fe);
    bool synced = false;
    while (!c->invtables.empty() && (c->invtables.size() >= 8 || held + n * sizeof(fe) > kInvTableCacheBytes)) {
      if (!synced) { STK_CUDA(c, cudaStreamSynchronize(c->stream)); synced = true; }
      held -= c->invtables.front().n * sizeof(fe);
      cudaFree(c->invtables.front().d);
      c->invtables.erase(c->invtables.begin());
    }
    STK_CUDA(c, cudaMalloc(&T, n * sizeof(fe)));
    const uint64_t chunks = (n + kInvChunk - 1) / kInvChunk;
    invtable_kernel<<<(unsigned)((chunks + 127) / 128), 128, 0, c->stream>>>(X, xshift, n, T);
    STK_CUDA(c, cudaGetLastError());
    c->invtables.push_back({G2, n, T});
  }
  BoundaryInterp I;
  for (uint64_t j = 0; j < 12; ++j) {
    I.i0[j] = j < width ? host::reduce(stk_load_fe(h_interp + 16 * j), c->p) : fe_zero();
    I.i1[j] = j < width ? host::reduce(stk_load_fe(h_interp + 16 * j + 8), c->p) : fe_zero();
  }
  const fe last_inv = stk_h_inv(c, stk_h_pow(c, G2, last_index));
  boundary_eval_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>((const fe*)d_pev, n, ext, (uint32_t)width, col_stride,
                                                                          X, xshift, T, last_index, last_inv, I,
                                                                          (const fe*)d_bsub, bsub_stride, (fe*)d_bev, out_stride);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

// D = C * (X - last) / (X^steps - 1) on coefficient vectors of length n (n a multiple of
// steps).  *h_bad receives the number of non-zero remainder coefficients (0 = exact).
STK_API int stk_quotient_z(stk_ctx* c, const uint32_t* d_ccoef, uint64_t n, uint64_t steps, const uint32_t last[8],
                           uint32_t* d_dcoef, uint32_t* h_bad) {
  if (!c || !d_ccoef || !d_dcoef || !last || steps == 0 || n % steps) return STK_EINVAL;
  void* t;
  STK_TRY(stk_scratch(c, kSlotStage, 64, &t));
  STK_CUDA(c, cudaMemsetAsync(t, 0, 4, c->stream));
  fe last_tw = stk_h_to_tw(c, host::reduce(stk_load_fe(last), c->p));
  unsigned blocks = (unsigned)((steps + 255) / 256);
  STK_TRY(stk_with_field(c, [&](auto f) {
    quotient_z_kernel<<<blocks, 256, 0, c->stream>>>((const fe*)d_ccoef, n, steps, last_tw, (fe*)d_dcoef, (uint32_t*)t,
                                                     f);
  }));
  if (h_bad) {
    STK_CUDA(c, cudaMemcpyAsync(h_bad, t, 4, cudaMemcpyDeviceToHost, c->stream));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return STK_OK;
}

// Quotient of a (n coefficients, low -> high) by (X - r): out[k] = sum_{i>k} a[i] r^(i-k-1),
// k < n-1 (out[n-1] is not written).  r must be 1 or an element whose order divides n... the
// powers r^i and r^-i (i < n) are taken from the cached tables of r and r^-1.
STK_API int stk_div_linear(stk_ctx* c, const uint32_t* d_a, uint64_t n, const uint32_t r[8], uint64_t r_order,
                           uint32_t* d_out) {
  if (!c || !d_a || !d_out || !r || n < 2) return STK_EINVAL;
  fe rr = host::reduce(stk_load_fe(r), c->p);
  fe one = stk_h_one(c);
  const fe* rpow = nullptr;
  const fe* rinvpow = nullptr;
  uint64_t rs = 1, ris = 1;
  if (!fe_eq(rr, one)) {
    if (r_order < n) return stk_fail(c, STK_EINVAL, "order of r must be at least the coefficient count");
    if (!fe_eq(stk_h_pow(c, rr, r_order), one)) return stk_fail(c, STK_EINVAL, "r^order != 1");
    STK_TRY(stk_get_table_strided(c, rr, r_order, &rpow, &rs));
    STK_TRY(stk_get_table_strided(c, stk_h_inv(c, rr), r_order, &rinvpow, &ris));
  }
  const fe* a = (const fe*)d_a;
  fe* out = (fe*)d_out;
  const uint64_t per_block = (uint64_t)kScanChunk * kScanThreads;
  const uint64_t nblocks = (n + per_block - 1) / per_block;
  void* t;
  STK_TRY(stk_scratch(c, kSlotStage, nblocks * sizeof(fe), &t));
  fe* totals = (fe*)t;
  return stk_with_field(c, [&](auto f) {
    scan_block_totals_kernel<<<(unsigned)nblocks, kScanThreads, 0, c->stream>>>(a, rpow, rs, n, totals, f);
    scan_totals_kernel<<<1, kScanThreads, 0, c->stream>>>(totals, nblocks, f);
    scan_finish_kernel<<<(unsigned)nblocks, kScanThreads, 0, c->stream>>>(a, rpow, rs, rinvpow, ris, n, totals, out, f);
  });
}

// out[i] = sum_c weights[c] * cols[c][i]
STK_API int stk_lincomb(stk_ctx* c, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                        const uint32_t* h_weights, uint32_t* d_out) {
  if (!c || !d_cols || !d_out || !h_weights || ncols == 0) return STK_EINVAL;
  std::vector<fe> w(ncols);
  for (uint64_t i = 0; i < ncols; ++i) w[i] = stk_h_to_tw(c, host::reduce(stk_load_fe(h_weights + 8 * i), c->p));
  void* t;
  STK_TRY(stk_stage(c, kSlotStage, ncols * sizeof(fe), {{0, w.data(), ncols * sizeof(fe)}}, &t));
  unsigned blocks = (unsigned)((n + 255) / 256);
  return stk_with_field(c, [&](auto f) {
    lincomb_kernel<<<blocks, 256, 0, c->stream>>>((const fe*)d_cols, n, (uint32_t)ncols, col_stride, (const fe*)t,
                                                  (fe*)d_out, f);
  });
}
