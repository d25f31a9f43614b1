// trace.cu -- execution traces on the device (starks/air.py:31-52 get_computational_trace + the
// witness transposition of AIR.generate_witness, :124): state[i+1][j] = step_poly_j(state[i]).
//
// One trace is a sequential chain of `steps` links, so the parallelism has to come from
// somewhere else:
//   * MANY independent traces (different inputs, same step polynomials): one thread per trace.
//   * ONE trace of an AIR whose step polynomials have degree <= 1 (Fibonacci-style, affine):
//     the state is a linear image of the previous one, (s, 1)' = A (s, 1), so the state at step
//     c*L is A^(cL) (s0, 1).  The host squares the (w+1) x (w+1) companion matrix log2 L times,
//     walks the `steps/L` chunk starts with one matrix-vector product each (a prefix over powers
//     of A: ~(w+1)^2 host multiplies per chunk), and the device runs every chunk's L links in
//     its own thread.  Exact arithmetic: the trace is the sequential one bit for bit.
//   * ONE trace of a non-linear AIR stays a single dependency chain: stk_trace_generate (host)
//     or stk_trace_generate_upload below, which hides the host recurrence behind the
//     upload of the blocks already generated.
// Witness layout on the device: d_witness[(t*width + dim)*stride + step], ABI elements.
#include <algorithm>
#include <vector>
#include "ctx.h"

using namespace stk;

namespace {

struct TraceMono {
  fe coeff_tw;       // coefficient, twiddle form
  uint32_t out;      // which state component it contributes to
  uint32_t unit;     // coefficient == 1 and total degree == 1: the term is a copy
  uint8_t exp[12];
  uint32_t pad;
};

// thread = (trace, chunk): runs min(L, steps - chunk*L) links from the chunk's start state
template <class F>
__global__ void __launch_bounds__(128) trace_chunk_kernel(const fe* __restrict__ starts, uint64_t nthreads,
                                                          uint64_t nchunks, uint64_t L, uint64_t steps, uint32_t width,
                                                          const TraceMono* __restrict__ monos, uint32_t nmono,
                                                          fe* __restrict__ out, uint64_t stride, const F f) {
  const uint64_t id = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (id >= nthreads) return;
  const uint64_t t = id / nchunks, c = id % nchunks;
  const uint64_t i0 = c * L;
  const uint64_t cnt = i0 >= steps ? 0 : (steps - i0 < L ? steps - i0 : L);
  fe st[12], nx[12];
  for (uint32_t k = 0; k < width; ++k) st[k] = fe_load(starts + id * width + k);
  for (uint64_t i = 0; i < cnt; ++i) {
    for (uint32_t k = 0; k < width; ++k) fe_store(out + (t * width + k) * stride + i0 + i, st[k]);
    if (i + 1 == cnt) break;
    for (uint32_t j = 0; j < width; ++j) nx[j] = fe_zero();
    for (uint32_t m = 0; m < nmono; ++m) {
      const TraceMono& M = monos[m];
      fe term;
      if (M.unit) {
        term = fe_zero();
        for (uint32_t k = 0; k < width; ++k)
          if (M.exp[k]) term = st[k];
      } else {
        term = f.from_tw(M.coeff_tw);
        for (uint32_t k = 0; k < width; ++k) {
          if (!M.exp[k]) continue;
          const fe sk = f.to_tw(st[k]);
          for (uint32_t e = 0; e < M.exp[k]; ++e) term = f.mul_tw(term, sk);
        }
      }
      nx[M.out] = f.add(nx[M.out], term);
    }
    for (uint32_t j = 0; j < width; ++j) st[j] = nx[j];
  }
}

// counts elements that are not canonical residues (>= p)
__global__ void noncanonical_kernel(const fe* __restrict__ a, uint64_t n, fe p, uint32_t* bad) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe x = fe_load(a + i);
  if (geq8(x.v, p.v)) atomicAdd(bad, 1u);
}

struct HostMat {            // (w+1) x (w+1), Montgomery domain, 4 x u64 limbs
  int d;
  std::vector<uint64_t> v;  // d*d*4
  uint64_t* at(int r, int c) { return &v[(size_t)(r * d + c) * 4]; }
  const uint64_t* at(int r, int c) const { return &v[(size_t)(r * d + c) * 4]; }
};

inline void add64m(const host::HostMont& H, const uint64_t* a, const uint64_t* b, uint64_t* r) {
  typedef unsigned __int128 u128;
  u128 cy = 0;
  uint64_t t[4];
  for (int i = 0; i < 4; ++i) { cy += (u128)a[i] + b[i]; t[i] = (uint64_t)cy; cy >>= 64; }
  bool ge = cy != 0;
  if (!ge) {
    ge = true;
    for (int i = 3; i >= 0; --i) { if (t[i] > H.m[i]) break; if (t[i] < H.m[i]) { ge = false; break; } }
  }
  if (ge) {
    uint64_t bw = 0;
    for (int i = 0; i < 4; ++i) { u128 d = (u128)t[i] - H.m[i] - bw; t[i] = (uint64_t)d; bw = (uint64_t)(d >> 64) & 1; }
  }
  for (int i = 0; i < 4; ++i) r[i] = t[i];
}

HostMat mat_mul(const host::HostMont& H, const HostMat& A, const HostMat& B) {
  HostMat C;
  C.d = A.d;
  C.v.assign((size_t)A.d * A.d * 4, 0);
  uint64_t t[4];
  for (int r = 0; r < A.d; ++r)
    for (int c = 0; c < A.d; ++c)
      for (int k = 0; k < A.d; ++k) {
        host::mont64(H, A.at(r, k), B.at(k, c), t);
        add64m(H, C.at(r, c), t, C.at(r, c));
      }
  return C;
}

int pack_monomials(stk_ctx* c, uint64_t width, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                   const uint8_t* h_mono_exps, uint64_t nmono, std::vector<TraceMono>& monos, bool* linear) {
  monos.resize(nmono ? nmono : 1);
  memset(monos.data(), 0, monos.size() * sizeof(TraceMono));
  *linear = true;
  const fe one = stk_h_one(c);
  for (uint64_t m = 0; m < nmono; ++m) {
    if (h_mono_out[m] >= width) return stk_fail(c, STK_EINVAL, "monomial output index out of range");
    const fe co = host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p);
    monos[m].coeff_tw = stk_h_to_tw(c, co);
    monos[m].out = h_mono_out[m];
    uint32_t deg = 0;
    for (uint64_t k = 0; k < width; ++k) { monos[m].exp[k] = h_mono_exps[width * m + k]; deg += monos[m].exp[k]; }
    monos[m].unit = (deg == 1 && fe_eq(co, one)) ? 1u : 0u;
    if (deg > 1) *linear = false;
  }
  return STK_OK;
}

}  // namespace

// *h_bad = number of elements of d_vals[0..n) that are >= p (0: every one is a canonical
// residue, which the add/sub/multiply kernels assume of their operands).  sync = 0: h_bad must be
// pinned host memory and is valid after the stream is next synchronised.
STK_API int stk_count_noncanonical(stk_ctx* c, const uint32_t* d_vals, uint64_t n, uint32_t* h_bad, int sync) {
  if (!c || !d_vals || !h_bad) return STK_EINVAL;
  *h_bad = 0;
  if (!n) return STK_OK;
  void* t;
  STK_TRY(stk_scratch(c, kSlotCounter, 64, &t));
  STK_CUDA(c, cudaMemsetAsync(t, 0, 4, c->stream));
  noncanonical_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>((const fe*)d_vals, n, c->p, (uint32_t*)t);
  STK_CUDA(c, cudaGetLastError());
  STK_CUDA(c, cudaMemcpyAsync(h_bad, t, 4, cudaMemcpyDeviceToHost, c->stream));
  if (sync) STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}

STK_API int stk_trace_generate_dev(stk_ctx* c, const uint32_t* h_inp, uint64_t ntraces, uint64_t steps, uint64_t width,
                                   const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                                   const uint8_t* h_mono_exps, uint64_t nmono, uint32_t* d_witness, uint64_t stride) {
  if (!c || !h_inp || !d_witness || steps == 0 || ntraces == 0 || stride < steps ||
      (nmono && (!h_mono_out || !h_mono_coeffs || !h_mono_exps)))
    return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  std::vector<TraceMono> monos;
  bool linear = false;
  STK_TRY(pack_monomials(c, width, h_mono_out, h_mono_coeffs, h_mono_exps, nmono, monos, &linear));
  // chunking: only an affine AIR can start a chunk without running the links before it
  uint64_t L = steps, nchunks = 1;
  if (linear && steps >= 4096) {
    uint64_t want = std::max<uint64_t>(1, 8192 / ntraces);   // ~8192 threads in flight
    L = std::max<uint64_t>(64, (steps + want - 1) / want);
    uint64_t l2 = 1;
    while (l2 < L) l2 <<= 1;                                 // A^L by squarings only
    L = l2;
    nchunks = (steps + L - 1) / L;
  }
  const uint64_t nthreads = ntraces * nchunks;
  std::vector<fe> starts(nthreads * width);
  const host::HostMont& H = host::host_mont(c->p);
  const uint64_t one_plain[4] = {1, 0, 0, 0};
  if (nchunks == 1) {
    for (uint64_t t = 0; t < ntraces; ++t)
      for (uint64_t k = 0; k < width; ++k)
        starts[t * width + k] = host::reduce(stk_load_fe(h_inp + (t * width + k) * 8), c->p);
  } else {
    const int d = (int)width + 1;
    HostMat A;
    A.d = d;
    A.v.assign((size_t)d * d * 4, 0);
    uint64_t one_m[4];
    host::mont64(H, one_plain, H.r2, one_m);                 // 1 in the Montgomery domain
    memcpy(A.at(d - 1, d - 1), one_m, 32);
    for (uint64_t m = 0; m < nmono; ++m) {
      uint64_t co[4], com[4];
      host::to64(host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p), co);
      host::mont64(H, co, H.r2, com);
      int col = d - 1;                                       // constant term unless a variable appears
      for (uint64_t k = 0; k < width; ++k)
        if (h_mono_exps[width * m + k]) col = (int)k;
      add64m(H, A.at((int)h_mono_out[m], col), com, A.at((int)h_mono_out[m], col));
    }
    HostMat AL = A;
    for (uint64_t l = 1; l < L; l <<= 1) AL = mat_mul(H, AL, AL);
    std::vector<uint64_t> v((size_t)d * 4), nv((size_t)d * 4);
    uint64_t t4[4];
    for (uint64_t t = 0; t < ntraces; ++t) {
      for (uint64_t k = 0; k < width; ++k) {
        uint64_t x[4];
        host::to64(host::reduce(stk_load_fe(h_inp + (t * width + k) * 8), c->p), x);
        host::mont64(H, x, H.r2, &v[k * 4]);
      }
      memcpy(&v[(size_t)width * 4], one_m, 32);
      for (uint64_t ch = 0; ch < nchunks; ++ch) {
        for (uint64_t k = 0; k < width; ++k) {
          uint64_t plain[4];
          host::mont64(H, &v[k * 4], one_plain, plain);
          starts[(t * nchunks + ch) * width + k] = host::from64(plain);
        }
        if (ch + 1 == nchunks) break;
        std::fill(nv.begin(), nv.end(), 0);
        for (int r = 0; r < d; ++r)
          for (int k = 0; k < d; ++k) {
            host::mont64(H, AL.at(r, k), &v[(size_t)k * 4], t4);
            add64m(H, &nv[(size_t)r * 4], t4, &nv[(size_t)r * 4]);
          }
        v.swap(nv);
      }
    }
  }
  void* dm;
  const uint64_t mono_bytes = monos.size() * sizeof(TraceMono);
  const uint64_t start_bytes = starts.size() * sizeof(fe), mono_off = ((start_bytes + 63) / 64) * 64;
  STK_TRY(stk_stage(c, kSlotStage, mono_bytes + start_bytes + 64,
                    {{0, starts.data(), start_bytes}, {mono_off, monos.data(), mono_bytes}}, &dm));
  const fe* d_starts = (const fe*)dm;
  const TraceMono* d_monos = (const TraceMono*)((char*)dm + mono_off);
  const unsigned blocks = (unsigned)((nthreads + 127) / 128);
  return stk_with_field(c, [&](auto f) {
    trace_chunk_kernel<<<blocks, 128, 0, c->stream>>>(d_starts, nthreads, nchunks, L, steps, (uint32_t)width, d_monos,
                                                      (uint32_t)nmono, (fe*)d_witness, stride, f);
  });
}

// get_computational_trace (starks/air.py:31-52) + the witness transposition of AIR.generate_witness
// (:124): state[i+1][j] = step_poly_j(state[i]).  The recurrence is sequential by nature (one
// 256-bit dependency chain of `steps` links), so it runs on one host core in the Montgomery
// domain (hostmath.h) and writes witness[dim][step] in the ABI element layout -- pinned memory
// from stk_host_alloc makes the following upload a single DMA.  Same monomial encoding as
// stk_trace_generate_dev.
STK_API int stk_trace_generate(stk_ctx* c, const uint32_t* h_inp, uint64_t steps, uint64_t width,
                               const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs, const uint8_t* h_mono_exps,
                               uint64_t nmono, uint32_t* h_witness) {
  if (!c || !h_inp || !h_witness || steps == 0 || (nmono && (!h_mono_out || !h_mono_coeffs || !h_mono_exps)))
    return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  const host::HostMont& H = host::host_mont(c->p);
  struct M64 { uint64_t v[4]; };
  auto to_mont = [&](const fe& x) { M64 a, r; host::to64(x, a.v); host::mont64(H, a.v, H.r2, r.v); return r; };
  const uint64_t one_plain[4] = {1, 0, 0, 0};
  std::vector<M64> coef(nmono ? nmono : 1);
  for (uint64_t m = 0; m < nmono; ++m) {
    if (h_mono_out[m] >= width) return stk_fail(c, STK_EINVAL, "monomial output index out of range");
    coef[m] = to_mont(host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p));
  }
  M64 st[12], nx[12];
  for (uint64_t k = 0; k < width; ++k) st[k] = to_mont(host::reduce(stk_load_fe(h_inp + 8 * k), c->p));
  for (uint64_t i = 0; i < steps; ++i) {
    for (uint64_t k = 0; k < width; ++k) {  // leave the Montgomery domain on the way out
      uint64_t plain[4];
      host::mont64(H, st[k].v, one_plain, plain);
      fe o = host::from64(plain);
      memcpy(h_witness + (k * steps + i) * 8, o.v, 32);
    }
    if (i + 1 == steps) break;
    for (uint64_t j = 0; j < width; ++j) memset(nx[j].v, 0, 32);
    for (uint64_t m = 0; m < nmono; ++m) {
      M64 t = coef[m];
      for (uint64_t k = 0; k < width; ++k)
        for (uint32_t e = 0; e < h_mono_exps[width * m + k]; ++e) host::mont64(H, t.v, st[k].v, t.v);
      add64m(H, nx[h_mono_out[m]].v, t.v, nx[h_mono_out[m]].v);
    }
    for (uint64_t j = 0; j < width; ++j) st[j] = nx[j];
  }
  return STK_OK;
}

// One trace on the host (any AIR) with the upload hidden behind the recurrence: the trace is
// generated in blocks of 2^15 steps into h_witness (pinned memory from stk_host_alloc) and every
// finished block is copied to d_witness[dim*stride + step] asynchronously while the next block
// is computed.  Returns with the copies enqueued on the context's stream.
STK_API int stk_trace_generate_upload(stk_ctx* c, const uint32_t* h_inp, uint64_t steps, uint64_t width,
                                      const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                                      const uint8_t* h_mono_exps, uint64_t nmono, uint32_t* h_witness,
                                      uint32_t* d_witness, uint64_t stride) {
  if (!c || !h_inp || !h_witness || !d_witness || steps == 0 || stride < steps ||
      (nmono && (!h_mono_out || !h_mono_coeffs || !h_mono_exps)))
    return STK_EINVAL;
  if (width == 0 || width > 12) return stk_fail(c, STK_EUNSUPPORTED, "state width must be in 1..12");
  const host::HostMont& H = host::host_mont(c->p);
  struct M64 { uint64_t v[4]; };
  const uint64_t one_plain[4] = {1, 0, 0, 0};
  std::vector<M64> coef(nmono ? nmono : 1);
  for (uint64_t m = 0; m < nmono; ++m) {
    if (h_mono_out[m] >= width) return stk_fail(c, STK_EINVAL, "monomial output index out of range");
    uint64_t x[4];
    host::to64(host::reduce(stk_load_fe(h_mono_coeffs + 8 * m), c->p), x);
    host::mont64(H, x, H.r2, coef[m].v);
  }
  M64 st[12], nx[12];
  for (uint64_t k = 0; k < width; ++k) {
    uint64_t x[4];
    host::to64(host::reduce(stk_load_fe(h_inp + 8 * k), c->p), x);
    host::mont64(H, x, H.r2, st[k].v);
  }
  const uint64_t B = 1ull << 15;
  for (uint64_t b0 = 0; b0 < steps; b0 += B) {
    const uint64_t b1 = std::min(steps, b0 + B);
    for (uint64_t i = b0; i < b1; ++i) {
      for (uint64_t k = 0; k < width; ++k) {
        uint64_t plain[4];
        host::mont64(H, st[k].v, one_plain, plain);
        fe o = host::from64(plain);
        memcpy(h_witness + (k * steps + i) * 8, o.v, 32);
      }
      if (i + 1 == steps) break;
      for (uint64_t j = 0; j < width; ++j) memset(nx[j].v, 0, 32);
      for (uint64_t m = 0; m < nmono; ++m) {
        M64 t = coef[m];
        for (uint64_t k = 0; k < width; ++k)
          for (uint32_t e = 0; e < h_mono_exps[width * m + k]; ++e) host::mont64(H, t.v, st[k].v, t.v);
        add64m(H, nx[h_mono_out[m]].v, t.v, nx[h_mono_out[m]].v);
      }
      for (uint64_t j = 0; j < width; ++j) st[j] = nx[j];
    }
    for (uint64_t k = 0; k < width; ++k)
      STK_CUDA(c, cudaMemcpyAsync((fe*)d_witness + k * stride + b0, h_witness + (k * steps + b0) * 8,
                                  (b1 - b0) * sizeof(fe), cudaMemcpyHostToDevice, c->stream));
  }
  return STK_OK;
}
