// ntt_api.cu -- context, twiddle tables, NTT plans and the NTT entry points of the C ABI.
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include "ctx.h"
#include "ntt.cuh"

using namespace stk;

// ------------------------------------------------------------------ small helpers

fe stk_load_fe(const uint32_t* w) {
  fe r;
  for (int i = 0; i < 8; ++i) r.v[i] = w[i];
  return r;
}
fe stk_h_mul(stk_ctx* c, const fe& a, const fe& b) { return host::mulmod(a, b, c->p); }
fe stk_h_pow(stk_ctx* c, const fe& a, uint64_t e) { return host::pow_u64(a, e, c->p); }
fe stk_h_inv(stk_ctx* c, const fe& a) { return host::invmod(a, c->p); }
fe stk_h_to_tw(stk_ctx* c, const fe& a) { return c->is_stark ? a : host::mulmod(a, c->mont.rone, c->p); }
fe stk_h_one(stk_ctx* c) { return host::reduce(host::from_u64(1), c->p); }
bool stk_h_primitive(stk_ctx* c, const fe& root, uint64_t n) {
  const fe one = stk_h_one(c);
  return fe_eq(stk_h_pow(c, root, n), one) && !fe_eq(stk_h_pow(c, root, n / 2), one);
}

void stk_stark_release(stk_ctx* c);  // stark.cu: per-context inverse tables

static int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return s && *s ? atoi(s) : dflt;
}

int stk_scratch(stk_ctx* c, int slot, uint64_t bytes, void** out) {
  if (c->scratch_bytes[slot] < bytes) {
    if (c->scratch[slot]) {
      STK_CUDA(c, cudaStreamSynchronize(c->stream));
      STK_CUDA(c, cudaFree(c->scratch[slot]));
      c->scratch[slot] = nullptr;
      c->scratch_bytes[slot] = 0;
    }
    STK_CUDA(c, cudaMalloc(&c->scratch[slot], bytes));
    c->scratch_bytes[slot] = bytes;
  }
  *out = c->scratch[slot];
  return STK_OK;
}

int stk_stage(stk_ctx* c, int slot, uint64_t bytes, std::initializer_list<stk_upload> ups, void** out) {
  STK_TRY(stk_scratch(c, slot, bytes, out));
  for (const stk_upload& u : ups)
    STK_CUDA(c, cudaMemcpyAsync((char*)*out + u.off, u.h, u.bytes, cudaMemcpyHostToDevice, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}

// ------------------------------------------------------------------ context

STK_API int stk_version(void) { return 1; }

STK_API int stk_init(int device, stk_ctx** out) {
  if (!out) return STK_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return STK_ECUDA;
  stk_ctx* c = new stk_ctx();
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete c; return STK_ECUDA; }
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return STK_ECUDA; }
  c->stream = c->own_stream;
  for (int i = 0; i < 3; ++i) cudaStreamCreateWithFlags(&c->copy_streams[i], cudaStreamNonBlocking);
  for (int i = 0; i < 8; ++i) cudaEventCreateWithFlags(&c->ev[i], cudaEventDisableTiming);
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
  c->is_stark = true;
  c->p = StarkField::modulus();
  *out = c;
  return STK_OK;
}

STK_API void stk_destroy(stk_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& t : c->tables) cudaFree(t.d);
  stk_stark_release(c);
  for (int i = 0; i < kScratchSlots; ++i) if (c->scratch[i]) cudaFree(c->scratch[i]);
  for (int i = 0; i < 8; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (int i = 0; i < 3; ++i) if (c->copy_streams[i]) cudaStreamDestroy(c->copy_streams[i]);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

STK_API const char* stk_last_error(stk_ctx* c) { return c ? c->err.c_str() : "no context"; }

STK_API int stk_set_stream(stk_ctx* c, void* s) {
  if (!c) return STK_EINVAL;
  cudaStream_t next = s ? (cudaStream_t)s : c->own_stream;
  if (next != c->stream) {
    // work enqueued on the old stream may still read cached tables and scratch buffers that the new
    // stream's calls are free to evict or regrow: drain it once, at the switch
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stream = next;
  }
  return STK_OK;
}

STK_API int stk_sync(stk_ctx* c) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}

STK_API int stk_field_set(stk_ctx* c, const uint32_t p32[8]) {
  if (!c || !p32) return STK_EINVAL;
  fe p = stk_load_fe(p32);
  if (fe_eq(p, c->p)) return STK_OK;
  // tables are per field: drop them
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  for (auto& t : c->tables) cudaFree(t.d);
  c->tables.clear();
  stk_stark_release(c);   // the inverse tables are per field too
  c->ntt_consts.clear();
  ++c->table_gen;
  if (host::is_stark_prime(p)) {
    c->is_stark = true;
    c->p = p;
    return STK_OK;
  }
  MontField F;
  if (!host::mont_setup(&F, p)) return stk_fail(c, STK_EUNSUPPORTED, "modulus must be odd and > 1");
  c->mont = F;
  c->is_stark = false;
  c->p = p;
  return STK_OK;
}

// ------------------------------------------------------------------ memory helpers

STK_API int stk_dev_alloc(stk_ctx* c, uint64_t bytes, void** d) {
  if (!c || !d) return STK_EINVAL;
  STK_CUDA(c, cudaMalloc(d, bytes ? bytes : 1));
  return STK_OK;
}
STK_API int stk_dev_free(stk_ctx* c, void* d) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  STK_CUDA(c, cudaFree(d));
  return STK_OK;
}
STK_API int stk_host_alloc(stk_ctx* c, uint64_t bytes, void** h) {
  if (!c || !h) return STK_EINVAL;
  STK_CUDA(c, cudaHostAlloc(h, bytes ? bytes : 1, cudaHostAllocDefault));
  return STK_OK;
}
STK_API int stk_host_free(stk_ctx* c, void* h) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaFreeHost(h));
  return STK_OK;
}
STK_API int stk_memcpy_h2d(stk_ctx* c, void* d, const void* h, uint64_t bytes) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c->stream));
  return STK_OK;
}
STK_API int stk_memcpy_d2h(stk_ctx* c, void* h, const void* d, uint64_t bytes) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}
STK_API int stk_memcpy_d2d(stk_ctx* c, void* dd, const void* ds, uint64_t bytes) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaMemcpyAsync(dd, ds, bytes, cudaMemcpyDeviceToDevice, c->stream));
  return STK_OK;
}
STK_API int stk_memset(stk_ctx* c, void* d, int value, uint64_t bytes) {
  if (!c) return STK_EINVAL;
  STK_CUDA(c, cudaMemsetAsync(d, value, bytes, c->stream));
  return STK_OK;
}

// ------------------------------------------------------------------ twiddle tables

// Cache discipline: `tables` is kept least-recently-used first; a hit moves its entry to the
// back.  An insertion evicts from the front while the cache holds 48 entries or more than
// kTableCacheBytes, but never the most recently used entry -- so a caller may hold the pointer
// of ONE earlier lookup across the next lookup (stk_div_linear holds r's table while fetching
// r^-1's).
static void table_touch(stk_ctx* c, size_t i) {
  if (i + 1 == c->tables.size()) return;
  stk_table t = c->tables[i];
  c->tables.erase(c->tables.begin() + i);
  c->tables.push_back(t);
}

int stk_get_table(stk_ctx* c, const fe& root, uint64_t n, const fe** d_table) {
  for (size_t i = 0; i < c->tables.size(); ++i)
    if (c->tables[i].n == n && fe_eq(c->tables[i].root, root)) {
      *d_table = c->tables[i].d;
      table_touch(c, i);
      return STK_OK;
    }
  const uint64_t need = std::max<uint64_t>(n, 1) * sizeof(fe);
  uint64_t held = 0;
  for (auto& t : c->tables) held += std::max<uint64_t>(t.n, 1) * sizeof(fe);
  bool synced = false;
  while (c->tables.size() > 1 && (c->tables.size() >= 48 || held + need > kTableCacheBytes)) {
    if (!synced) { STK_CUDA(c, cudaStreamSynchronize(c->stream)); synced = true; }
    held -= std::max<uint64_t>(c->tables.front().n, 1) * sizeof(fe);
    cudaFree(c->tables.front().d);
    c->tables.erase(c->tables.begin());
    ++c->table_gen;
  }
  stk_table t;
  t.root = root; t.n = n; t.mont = !c->is_stark; t.d = nullptr;
  STK_CUDA(c, cudaMalloc(&t.d, std::max<uint64_t>(n, 1) * sizeof(fe)));
  fe one = stk_h_to_tw(c, stk_h_one(c));
  STK_CUDA(c, cudaMemcpyAsync(t.d, &one, sizeof(fe), cudaMemcpyHostToDevice, c->stream));
  STK_TRY(stk_with_field(c, [&](auto f) {
    fe wm = root;  // root^m, plain
    for (uint64_t m = 1; m < n; m <<= 1) {
      uint64_t cnt = std::min<uint64_t>(m, n - m);
      unsigned blocks = (unsigned)((cnt + 255) / 256);
      twiddle_extend_kernel<<<blocks, 256, 0, c->stream>>>(t.d, m, n, stk_h_to_tw(c, wm), f);
      wm = stk_h_mul(c, wm, wm);
    }
  }));
  c->tables.push_back(t);
  *d_table = t.d;
  return STK_OK;
}

int stk_get_table_strided(stk_ctx* c, const fe& root, uint64_t n, const fe** d_table, uint64_t* stride) {
  *stride = 1;
  for (size_t i = 0; i < c->tables.size(); ++i)
    if (c->tables[i].n == n && fe_eq(c->tables[i].root, root)) {
      *d_table = c->tables[i].d;
      table_touch(c, i);
      return STK_OK;
    }
  for (size_t i = 0; i < c->tables.size(); ++i) {
    const stk_table& t = c->tables[i];
    if (t.n > n && t.n % n == 0) {
      uint64_t s = t.n / n;
      if (fe_eq(stk_h_pow(c, t.root, s), root)) {
        *d_table = t.d;
        *stride = s;
        table_touch(c, i);
        return STK_OK;
      }
    }
  }
  return stk_get_table(c, root, n, d_table);
}

int stk_get_table_shift(stk_ctx* c, const fe& root, uint64_t n, const fe** d_table, int* shift) {
  uint64_t stride;
  STK_TRY(stk_get_table_strided(c, root, n, d_table, &stride));
  *shift = stk_ilog2(stride);
  if ((1ull << *shift) == stride) return STK_OK;
  *shift = 0;
  return stk_get_table(c, root, n, d_table);
}

// ------------------------------------------------------------------ NTT plan

// log2 radix of the STARK-prime rounds; radix-4 measured no faster: profiles/r01_ntt_radix_sweep.txt
static const int kStarkRadix = 3;

// Rounds of a pass.  Where the remainder round (k mod R levels) goes was measured
// (profiles/r01_ntt_round_order.txt): last in non-final passes and in 1024-element final
// passes, first in 2048-element final passes; the spread is 1-3 %.
static void fill_rounds(NttPass& P, int R) {
  int k = P.k, rem = k % R, full = k / R, idx = 0;
  const int pos = (P.final_pass && P.logT > 10) ? 0 : full;
  for (int i = 0; i <= full; ++i) {
    if (i == pos && rem) P.r[idx++] = rem;
    if (i < full) P.r[idx++] = R;
  }
  P.nrounds = idx;
}

// Cuts the n index bits into passes (top bits first) and fixes each pass's tile geometry.
static int build_plan(int n, uint64_t batch, std::vector<NttPass>& plan, int rmax) {
  // 1024-element tiles (4 CTAs/SM) unless 2048-element tiles (2 CTAs/SM) save a whole pass
  // over HBM (n = 11, 21, 22): profiles/r01_ntt_plan_sweep2.txt.  Run-time moduli: 1024 only.
  int logT = ((n + 10) / 11 < (n + 9) / 10) ? 11 : 10;
  if (rmax < 3) logT = 10;
  const int kmax = logT;  // butterfly levels per pass: at most one whole tile
  plan.clear();
  if (n <= kmax) {
    NttPass P;
    memset(&P, 0, sizeof P);
    P.n = n; P.n_tw = n; P.lo = 0; P.k = n;
    P.logC = std::min(logT - n, stk_ilog2(batch));
    P.logT = P.k + P.logC;
    P.c_is_col = 1; P.cb = 0; P.nl = 0; P.sl = 0; P.sh = 0;
    P.final_pass = 1;
    fill_rounds(P, rmax);
    plan.push_back(P);
    return STK_OK;
  }
  int npass = (n + kmax - 1) / kmax;
  int hi = n;
  for (int i = 0; i < npass; ++i) {
    int k = (hi + (npass - i) - 1) / (npass - i);  // spread the remaining bits evenly
    NttPass P;
    memset(&P, 0, sizeof P);
    P.n = n; P.n_tw = n; P.k = k; P.lo = hi - k;
    P.final_pass = (i == npass - 1);
    P.c_is_col = 0;
    P.logC = logT - k;
    if (!P.final_pass) {
      if (P.logC > P.lo) P.logC = P.lo;
      P.cb = 0;
      P.nl = P.lo - P.logC; P.sl = P.logC; P.sh = P.lo + P.k;
    } else {
      if (P.logC > n - k) P.logC = n - k;
      P.cb = n - P.logC;
      P.nl = n - P.logC - k; P.sl = k; P.sh = 0;
    }
    P.logT = P.k + P.logC;
    fill_rounds(P, rmax);
    plan.push_back(P);
    hi -= k;
  }
  return STK_OK;
}

// The pass kernel and its launcher (ntt.cuh) are instantiated in their own translation units
// (ntt_pass_*.cu) so that they compile in parallel; this file only sees the launchers.
int stk_launch_pass_stark(stk_ctx* c, cudaStream_t s, const NttPass& P);      // radix-8 rounds
int stk_launch_pass_stark_zs(stk_ctx* c, cudaStream_t s, const NttPass& P);   // + zero-skip levels
int stk_launch_pass_stark_t11(stk_ctx* c, cudaStream_t s, const NttPass& P);     // 2048-element tiles
int stk_launch_pass_stark_t11_zs(stk_ctx* c, cudaStream_t s, const NttPass& P);
int stk_launch_pass_stark_cf(stk_ctx* c, cudaStream_t s, const NttPass& P);      // coset transform, final pass
int stk_launch_pass_stark_t11_cf(stk_ctx* c, cudaStream_t s, const NttPass& P);
int stk_launch_pass_mont(stk_ctx* c, cudaStream_t s, const NttPass& P);       // run-time modulus, radix-4

static int launch_pass(stk_ctx* c, cudaStream_t s, const NttPass& P) {
  if (!c->is_stark) return stk_launch_pass_mont(c, s, P);
  const bool zs = P.zbit < 32 || (P.cshift && !P.in_virtual);  // expansion round / coset scaling on load
  const bool cf = !zs && P.cshift && (P.final_pass || P.cskip0);  // interleaved store / skipped r = 0 columns
  if (P.logT > 10)
    return zs ? stk_launch_pass_stark_t11_zs(c, s, P) : cf ? stk_launch_pass_stark_t11_cf(c, s, P) : stk_launch_pass_stark_t11(c, s, P);
  else
    return zs ? stk_launch_pass_stark_zs(c, s, P) : cf ? stk_launch_pass_stark_cf(c, s, P) : stk_launch_pass_stark(c, s, P);
}

// direct DFT for orders that are not a power of two >= 8 (_simple_ft, starks/fft.py:287-300)
template <class F>
__global__ void dft_generic_kernel(const fe* in, uint64_t n_in, uint64_t in_stride, fe* out, uint64_t out_stride,
                                   uint64_t n, uint64_t batch, const fe* W, uint64_t wstride, int do_scale, fe scale,
                                   const F f) {
  uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (idx >= n * batch) return;
  uint64_t k = idx % n, col = idx / n;
  const fe* src = in + col * in_stride;
  fe acc = fe_zero();
  for (uint64_t j = 0; j < n_in; ++j) {
    uint64_t e = (j * k) % n;
    acc = f.add(acc, f.mul_tw(fe_load(src + j), fe_load_ro(W + e * wstride)));
  }
  if (do_scale) acc = f.mul_tw(acc, scale);
  fe_store(out + col * out_stride + k, acc);
}

static int launch_dft(stk_ctx* c, cudaStream_t s, const fe* in, uint64_t n_in, uint64_t in_stride, fe* out,
                      uint64_t out_stride, uint64_t n, uint64_t batch, const fe* W, uint64_t wstride, int do_scale,
                      const fe& scale_tw) {
  const unsigned blocks = (unsigned)((n * batch + 127) / 128);
  return stk_with_field(c, [&](auto f) {
    dft_generic_kernel<<<blocks, 128, 0, s>>>(in, n_in, in_stride, out, out_stride, n, batch, W, wstride, do_scale,
                                              scale_tw, f);
  });
}

// out[col][8K] = canonical(r0[col][K]): the residue-0 coset of an 8x extension is the input domain
__global__ void r0_copy_kernel(const fe* __restrict__ r0, uint64_t r0_stride, fe* __restrict__ out, uint64_t out_stride,
                               uint64_t ns, uint64_t batch) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= ns * batch) return;
  const uint64_t col = i / ns, K = i % ns;
  fe v = fe_load(r0 + col * r0_stride + K);
  StarkField::canon(v.v);
  fe_store(out + col * out_stride + 8 * K, v);
}

// optional peer scatter of a transform's final pass (stk_ntt_dev_peer)
struct stk_peer_leaf {
  int g;                      // log2 of the rank count
  uint32_t col0;              // global index of this rank's first column
  const uint64_t* ptrs;       // nranks exchange buffers (columns_total x N/G elements each)
};

static int ntt_dev_on(stk_ctx* c, cudaStream_t s, int scratch_slot, const fe* d_in, uint64_t n_in, uint64_t in_stride,
                      fe* d_out, uint64_t out_stride, uint64_t n, uint64_t batch, const fe& root, int inverse,
                      int scale, const stk_peer_leaf* peer = nullptr, const fe* r0 = nullptr,
                      uint64_t r0_stride = 0) {
  if (n == 0 || batch == 0) return STK_OK;
  if (n_in > n) return stk_fail(c, STK_EINDEX, "input length %llu exceeds the order %llu of the root",
                                (unsigned long long)n_in, (unsigned long long)n);
  if (n > (1ull << 30)) return stk_fail(c, STK_EUNSUPPORTED, "transform length above 2^30");
  // multi-pass launches put the column index in gridDim.y (<= 65535): wider batches run as
  // consecutive column groups on the same stream (the scratch buffer is reused in stream order)
  if (batch > 32768 && n > 2048 && !peer) {
    for (uint64_t b0 = 0; b0 < batch; b0 += 32768) {
      const uint64_t nb = std::min<uint64_t>(32768, batch - b0);
      STK_TRY(ntt_dev_on(c, s, scratch_slot, d_in + b0 * in_stride, n_in, in_stride, d_out + b0 * out_stride,
                         out_stride, n, nb, root, inverse, scale, nullptr, r0 ? r0 + b0 * r0_stride : nullptr,
                         r0_stride));
    }
    return STK_OK;
  }
  stk_ntt_consts* K = nullptr;
  for (auto& e : c->ntt_consts)
    if (e.n == n && e.inverse == (inverse ? 1 : 0) && fe_eq(e.root, root)) { K = &e; break; }
  if (!K) {
    // odd orders (the direct DFT) are held to root^n == 1 only
    if (n % 2 ? !fe_eq(stk_h_pow(c, root, n), stk_h_one(c)) : !stk_h_primitive(c, root, n))
      return stk_fail(c, STK_EINVAL, "root is not a primitive n-th root of unity");
    stk_ntt_consts e;
    e.root = root; e.n = n; e.inverse = inverse ? 1 : 0;
    e.w = inverse ? stk_h_inv(c, root) : root;
    e.scale_tw = fe_zero();
    if (inverse) e.scale_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(n), c->p)));
    if (c->ntt_consts.size() >= 64) c->ntt_consts.erase(c->ntt_consts.begin());
    c->ntt_consts.push_back(e);
    K = &c->ntt_consts.back();
  }
  const bool pow2 = (n & (n - 1)) == 0;
  if (K->table_gen != c->table_gen || !K->W) {
    const fe* Wt = nullptr;
    uint64_t ws = 1;
    if (pow2) {  // the pass kernels index by shift
      int shift;
      STK_TRY(stk_get_table_shift(c, K->w, n, &Wt, &shift));
      ws = 1ull << shift;
    } else {
      STK_TRY(stk_get_table_strided(c, K->w, n, &Wt, &ws));
    }
    K->W = Wt; K->wstride = ws; K->table_gen = c->table_gen;
  }
  const fe* W = K->W;
  const uint64_t wstride = K->wstride;
  const int do_scale = inverse && scale;
  const fe scale_tw = K->scale_tw;
  if (!pow2 || n < 8) {
    if (n > 4096) return stk_fail(c, STK_EUNSUPPORTED, "non power-of-two order above 4096");
    const fe* src = d_in;
    if ((const void*)d_in == (const void*)d_out) {  // every output reads the whole column
      void* tmp;
      STK_TRY(stk_scratch(c, scratch_slot, batch * n_in * sizeof(fe), &tmp));
      for (uint64_t b = 0; b < batch; ++b)
        STK_CUDA(c, cudaMemcpyAsync((fe*)tmp + b * n_in, d_in + b * in_stride, n_in * sizeof(fe),
                                    cudaMemcpyDeviceToDevice, s));
      src = (const fe*)tmp;
      in_stride = n_in;
    }
    return launch_dft(c, s, src, n_in, in_stride, d_out, out_stride, n, batch, W, wstride, do_scale, scale_tw);
  }
  int logn = stk_ilog2(n);
  std::vector<NttPass> plan;
  // Zero-padded forward transform (LDE, n_in <= N/8): eight coset transforms of order N/8 over
  // <w^8> as 8*batch virtual columns (ntt.cuh, cshift) -- the sub-transform's passes split its
  // own bits evenly (2^18: 9+9, 2^20: 10+10) instead of the long transform's (11+10, 8+8+7).
  if (c->is_stark && !inverse && !peer && n_in > 0 && n_in * 8 <= n && logn >= 6 &&
      (const void*)d_in != (const void*)d_out && env_int("STK_LDE_COSET", 1)) {
    const int logns = logn - 3;
    const uint64_t ns = n >> 3, vb = batch * 8;
    STK_TRY(build_plan(logns, vb, plan, kStarkRadix));
    std::vector<NttPass> whole;
    STK_TRY(build_plan(logn, batch, whole, kStarkRadix));
    // only where it saves a pass over HBM (N >= 2^23): at equal pass counts the two routes time the
    // same on one GPU (2^21: 17.87 ms both) and the coset route measured slower inside the NCCL
    // sharded commit (profiles/r01b_dist_2gpu.txt), so the long transform keeps the expansion round
    const bool fewer_passes = plan.size() < whole.size() || env_int("STK_LDE_COSET", 1) > 1;
    // with the input's own evaluations at hand (r0: the trace of an 8x LDE) the r = 0 coset is a copy:
    // one eighth of the transform is not computed at all, which pays at every size
    const bool use_r0 = r0 && n_in * 8 == n && env_int("STK_LDE_R0", 1);
    if ((fewer_passes || use_r0) && vb <= 0x7fffffffull && (plan.size() == 1 || vb <= 65535)) {
      fe* tmpc = nullptr;
      if (plan.size() > 1) {
        void* t;
        STK_TRY(stk_scratch(c, scratch_slot, batch * n * sizeof(fe), &t));
        tmpc = (fe*)t;
      }
      for (size_t i = 0; i < plan.size(); ++i) {
        NttPass& P = plan[i];
        P.batch = (uint32_t)vb;
        P.W = W;
        P.cs_shift = stk_ilog2(wstride);
        P.tw_shift = P.cs_shift + 3;
        P.cshift = 3;
        P.in_virtual = i > 0;
        P.cskip0 = use_r0 ? 1 : 0;
        P.zbit = 32;
        if (i == 0) { P.in = d_in; P.in_col_stride = in_stride; P.n_in = (uint32_t)n_in; }
        else { P.in = tmpc; P.in_col_stride = ns; P.n_in = (uint32_t)ns; }
        if (P.final_pass) { P.out = d_out; P.out_col_stride = out_stride; }
        else { P.out = tmpc; P.out_col_stride = ns; }
        STK_TRY(launch_pass(c, s, P));
      }
      if (use_r0) {
        const uint64_t tot = ns * batch;
        r0_copy_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(r0, r0_stride, d_out, out_stride, ns, batch);
        STK_CUDA(c, cudaGetLastError());
      }
      return STK_OK;
    }
  }
  STK_TRY(build_plan(logn, batch, plan, c->is_stark ? kStarkRadix : 2));
  fe* tmp = nullptr;
  if (peer && (plan.size() < 2 || logn - 2 - peer->g < plan.back().logC))
    return stk_fail(c, STK_EUNSUPPORTED, "peer scatter needs a multi-pass transform (N >= 2^11) and N/4G >= tile width");
  bool need_tmp = plan.size() > 1 || (const void*)d_in == (const void*)d_out;
  if (need_tmp) {
    void* t;
    STK_TRY(stk_scratch(c, scratch_slot, batch * n * sizeof(fe), &t));
    tmp = (fe*)t;
  }
  for (size_t i = 0; i < plan.size(); ++i) {
    NttPass& P = plan[i];
    P.batch = (uint32_t)batch;
    P.W = W;
    P.tw_shift = stk_ilog2(wstride);
    P.do_scale = (P.final_pass && do_scale) ? 1 : 0;
    P.scale = scale_tw;
    P.zbit = 32;
    if (i == 0 && n_in > 0 && n_in * 8 <= n && P.k >= 3 && c->is_stark) {
      // the top three levels only scale-and-copy: run them as the first (radix-8) round
      P.zbit = stk_ilog2(n_in);             // 2^zbit >= n_in, and 2^zbit <= N/8
      if (P.r[0] != 3) {                    // remainder round goes last in this pass
        int rem = P.r[0];
        for (int q = 0; q + 1 < P.nrounds; ++q) P.r[q] = P.r[q + 1];
        P.r[P.nrounds - 1] = rem;
      }
    }
    if (plan.size() == 1) {
      if (need_tmp) {  // in place: stage the input
        for (uint64_t b = 0; b < batch; ++b)
          STK_CUDA(c, cudaMemcpyAsync(tmp + b * n, d_in + b * in_stride, n_in * sizeof(fe),
                                      cudaMemcpyDeviceToDevice, s));
        P.in = tmp; P.in_col_stride = n;
      } else {
        P.in = d_in; P.in_col_stride = in_stride;
      }
      P.n_in = (uint32_t)n_in;
      P.out = d_out; P.out_col_stride = out_stride;
    } else if (i == 0) {
      P.in = d_in; P.in_col_stride = in_stride; P.n_in = (uint32_t)n_in;
      P.out = tmp; P.out_col_stride = n;
    } else if (!P.final_pass) {
      P.in = tmp; P.in_col_stride = n; P.n_in = (uint32_t)n;
      P.out = tmp; P.out_col_stride = n;
    } else {
      P.in = tmp; P.in_col_stride = n; P.n_in = (uint32_t)n;
      P.out = d_out; P.out_col_stride = out_stride;
      if (peer) {
        P.peer_on = 2; P.peer_g = peer->g; P.peer_col0 = peer->col0;
        for (int r2 = 0; r2 < (1 << peer->g); ++r2) P.peer_out[r2] = (fe*)(uintptr_t)peer->ptrs[r2];
      }
    }
    STK_TRY(launch_pass(c, s, P));
  }
  return STK_OK;
}

int stk_ntt_dev_peer(stk_ctx* c, const fe* d_in, uint64_t n_in, uint64_t in_stride, uint64_t n, uint64_t batch,
                     const fe& root, uint64_t nranks, uint64_t col_base, const uint64_t* ptrs) {
  const stk_peer_leaf peer = {stk_ilog2(nranks), (uint32_t)col_base, ptrs};
  // d_out is never written in peer mode; any distinct non-null pointer keeps the in-place logic off
  return ntt_dev_on(c, c->stream, kSlotNtt, d_in, n_in, in_stride, (fe*)(uintptr_t)16, n, n, batch, root, 0, 0,
                    &peer);
}

// Forward transform of coefficient rows whose values on the order-n/8 subgroup are already known
// (r0: the trace an 8x low-degree extension started from): see NttPass::cskip0.
int stk_ntt_dev_r0(stk_ctx* c, const fe* d_in, uint64_t n_in, uint64_t in_stride, fe* d_out, uint64_t out_stride,
                   uint64_t n, uint64_t batch, const fe& root, const fe* r0, uint64_t r0_stride) {
  return ntt_dev_on(c, c->stream, kSlotNtt, d_in, n_in, in_stride, d_out, out_stride, n, batch, root, 0, 0, nullptr,
                    r0, r0_stride);
}

int stk_ntt_dev(stk_ctx* c, const fe* d_in, uint64_t n_in, uint64_t in_stride, fe* d_out, uint64_t out_stride,
                uint64_t n, uint64_t batch, const fe& root, int inverse, int scale) {
  return ntt_dev_on(c, c->stream, kSlotNtt, d_in, n_in, in_stride, d_out, out_stride, n, batch, root, inverse,
                    scale);
}

STK_API int stk_ntt(stk_ctx* c, const uint32_t* d_in, uint64_t n_in, uint64_t in_stride, uint32_t* d_out,
                    uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse) {
  if (!c || !d_out || !root || (!d_in && n_in)) return STK_EINVAL;
  return stk_ntt_dev(c, (const fe*)d_in, n_in, in_stride, (fe*)d_out, out_stride, n, batch, stk_load_fe(root),
                     inverse, 1);
}

// _simple_ft (starks/fft.py:287-300) as its own entry point: the direct O(n^2) sum for ANY order
// n <= 4096 (stk_ntt routes orders that are not a power of two >= 8 here on its own).
STK_API int stk_dft_generic(stk_ctx* c, const uint32_t* d_in, uint64_t n_in, uint64_t in_stride, uint32_t* d_out,
                            uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse) {
  if (!c || !d_out || !root || (!d_in && n_in)) return STK_EINVAL;
  if (n == 0 || batch == 0) return STK_OK;
  if (n_in > n) return stk_fail(c, STK_EINDEX, "input length exceeds the order of the root");
  if (n > 4096) return stk_fail(c, STK_EUNSUPPORTED, "direct DFT is limited to orders <= 4096");
  if ((const void*)d_in == (const void*)d_out) return stk_fail(c, STK_EINVAL, "direct DFT works out of place");
  fe r = host::reduce(stk_load_fe(root), c->p);
  if (!fe_eq(stk_h_pow(c, r, n), stk_h_one(c))) return stk_fail(c, STK_EINVAL, "root^n != 1");
  fe w = inverse ? stk_h_inv(c, r) : r;
  const fe* W = nullptr;
  uint64_t ws = 1;
  STK_TRY(stk_get_table_strided(c, w, n, &W, &ws));
  fe scale_tw = fe_zero();
  if (inverse) scale_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(n), c->p)));
  return launch_dft(c, c->stream, (const fe*)d_in, n_in, in_stride, (fe*)d_out, out_stride, n, batch, W, ws,
                    inverse ? 1 : 0, scale_tw);
}

// Host buffers: columns stream through three device slots, each with its own stream, so that
// the H2D copy of chunk i+1, the transform of chunk i and the D2H copy of chunk i-1 overlap
// (PCIe is full duplex; the transform itself is ~5x faster than either copy).
STK_API int stk_ntt_host(stk_ctx* c, const uint32_t* h_in, uint64_t n_in, uint64_t in_stride, uint32_t* h_out,
                         uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse) {
  if (!c || !h_out || !root || (!h_in && n_in)) return STK_EINVAL;
  if (n_in > n) return stk_fail(c, STK_EINDEX, "input length exceeds the order of the root");
  if (n == 0 || batch == 0) return STK_OK;
  fe r = stk_load_fe(root);
  constexpr int kSlots = 3;
  const uint64_t col_bytes = n * sizeof(fe);
  uint64_t chunk = std::max<uint64_t>(1, ((uint64_t)64 << 20) / col_bytes);  // 64 MiB of output per slot
  chunk = std::min(chunk, batch);
  // slot buffers: in (n_in per column, packed) and out (n per column)
  void* bufs;
  const uint64_t in_b = chunk * std::max<uint64_t>(n_in, 1) * sizeof(fe), out_b = chunk * col_bytes;
  STK_TRY(stk_scratch(c, kSlotHostNttBufs, kSlots * (in_b + out_b), &bufs));
  char* base = (char*)bufs;
  fe* din[kSlots];
  fe* dout[kSlots];
  for (int i = 0; i < kSlots; ++i) {
    din[i] = (fe*)(base + i * in_b);
    dout[i] = (fe*)(base + kSlots * in_b + i * out_b);
  }
  // tables (and the per-slot NTT scratch) must exist before the streams fork
  {
    const fe* W;
    fe w = inverse ? stk_h_inv(c, r) : r;
    STK_TRY(stk_get_table(c, w, n, &W));
    void* t;
    for (int i = 0; i < kSlots; ++i) STK_TRY(stk_scratch(c, kSlotHostNtt + i, chunk * col_bytes, &t));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  int slot = 0;
  for (uint64_t b0 = 0; b0 < batch; b0 += chunk, slot = (slot + 1) % kSlots) {
    uint64_t nb = std::min(chunk, batch - b0);
    cudaStream_t s = c->copy_streams[slot];
    if (n_in) {
      if (in_stride == n_in)
        STK_CUDA(c, cudaMemcpyAsync(din[slot], h_in + b0 * in_stride * 8, nb * n_in * sizeof(fe),
                                    cudaMemcpyHostToDevice, s));
      else
        STK_CUDA(c, cudaMemcpy2DAsync(din[slot], n_in * sizeof(fe), h_in + b0 * in_stride * 8,
                                      in_stride * sizeof(fe), n_in * sizeof(fe), nb, cudaMemcpyHostToDevice, s));
    }
    STK_TRY(ntt_dev_on(c, s, kSlotHostNtt + slot, din[slot], n_in, n_in, dout[slot], n, n, nb, r, inverse, 1));
    if (out_stride == n)
      STK_CUDA(c, cudaMemcpyAsync(h_out + b0 * out_stride * 8, dout[slot], nb * col_bytes, cudaMemcpyDeviceToHost, s));
    else
      STK_CUDA(c, cudaMemcpy2DAsync(h_out + b0 * out_stride * 8, out_stride * sizeof(fe), dout[slot], col_bytes,
                                    col_bytes, nb, cudaMemcpyDeviceToHost, s));
  }
  for (int i = 0; i < kSlots; ++i) STK_CUDA(c, cudaStreamSynchronize(c->copy_streams[i]));
  return STK_OK;
}

// ------------------------------------------------------------------ multi-GPU four-step phases
// A transform of order N = G * L over G ranks, one all-to-all (SURVEY.md App. C.4):
//   input   cyclic: rank r holds x[r + G*m], m < L
//   phase 0 (in place, no communication): the top log2(L) butterfly levels of the DIF act inside
//           one residue class r -- a partial transform of the local array whose global index
//           is (m << g) | r;
//   all-to-all + local transpose (done by the caller): rank r' then holds the block
//           J in [r'*L, (r'+1)*L) of the partially transformed global array, low g bits fastest;
//   phase 1: the last g = log2(G) levels and the bit-reversed store; the output index K has
//           K mod G = bitrev_g(r'), and rank r' keeps X[K] at local position K >> g
//           (cyclic output, k2-sharded as in App. C.4).
static int dist_phase_impl(stk_ctx* c, int phase, const uint32_t* d_in, uint32_t* d_out, uint64_t local_n, uint64_t batch,
                           uint64_t stride, const uint32_t root[8], uint64_t nranks, uint64_t rank, int inverse,
                           const uint64_t* peer_ptrs, int rotated_input) {
  if (!c || !d_in || !d_out || !root || local_n == 0 || batch == 0) return STK_EINVAL;
  if ((local_n & (local_n - 1)) || (nranks & (nranks - 1)) || nranks < 2 || rank >= nranks || nranks > 8)
    return stk_fail(c, STK_EINVAL, "local length and rank count must be powers of two (2..8 ranks)");
  if (phase != 0 && phase != 1) return STK_EINVAL;
  const int nloc = stk_ilog2(local_n), g = stk_ilog2(nranks), n = nloc + g;
  if (n > 30 || nloc < 3) return stk_fail(c, STK_EUNSUPPORTED, "distributed transform needs 2^3 <= local length and N <= 2^30");
  if (phase == 0 && d_in != d_out) return stk_fail(c, STK_EINVAL, "phase 0 works in place");
  if (phase == 1 && (const void*)d_in == (const void*)d_out) return stk_fail(c, STK_EINVAL, "phase 1 works out of place");
  fe r = stk_load_fe(root);
  const uint64_t N = local_n * nranks;
  if (!stk_h_primitive(c, r, N))
    return stk_fail(c, STK_EINVAL, "root is not a primitive (G*L)-th root of unity");
  fe w = inverse ? stk_h_inv(c, r) : r;
  const fe* W = nullptr;
  STK_TRY(stk_get_table(c, w, N, &W));
  std::vector<NttPass> plan;
  if (phase == 0) {
    STK_TRY(build_plan(nloc, batch, plan, c->is_stark ? kStarkRadix : 2));
    for (auto& P : plan) {
      P.final_pass = 0;  // keep the tile geometry, store in place
      P.n_tw = n; P.j_shift = g; P.j_or = (uint32_t)rank; P.out_shift = 0;
    }
    if (peer_ptrs) {  // the last pass scatters straight into the peers' exchange buffers
      if (batch != 1) return stk_fail(c, STK_EUNSUPPORTED, "peer scatter handles one column");
      NttPass& L = plan.back();
      L.peer_on = 1; L.peer_log_chunk = nloc - g; L.peer_self = (uint32_t)rank;
      for (uint64_t r2 = 0; r2 < nranks; ++r2) L.peer_out[r2] = (fe*)(uintptr_t)peer_ptrs[r2];
    }
  } else {
    // last g levels: bits [0, g) of the local index; final-pass geometry (batch bits on top)
    const int logT = 10;
    NttPass P;
    memset(&P, 0, sizeof P);
    P.n = nloc; P.k = g; P.lo = 0; P.final_pass = 1; P.c_is_col = 0;
    P.logC = std::min(logT - g, nloc - g);
    P.cb = nloc - P.logC;
    P.nl = nloc - P.logC - g; P.sl = g; P.sh = 0;
    P.logT = P.k + P.logC;
    fill_rounds(P, c->is_stark ? kStarkRadix : 2);
    P.n_tw = n; P.j_shift = 0; P.j_or = (uint32_t)(rank << nloc); P.out_shift = g;
    P.in_rot = rotated_input ? g : 0;
    plan.push_back(P);
  }
  fe scale_tw = fe_zero();
  int do_scale = 0;
  if (inverse && phase == 1) {
    scale_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(N), c->p)));
    do_scale = 1;
  }
  for (auto& P : plan) {
    P.batch = (uint32_t)batch;
    P.W = W;
    P.zbit = 32;
    P.n_in = (uint32_t)local_n;
    P.in = (const fe*)d_in; P.in_col_stride = stride;
    P.out = (fe*)d_out; P.out_col_stride = stride;
    P.do_scale = (P.final_pass && do_scale) ? 1 : 0;
    P.scale = scale_tw;
    STK_TRY(launch_pass(c, c->stream, P));
  }
  return STK_OK;
}

STK_API int stk_ntt_dist_phase(stk_ctx* c, int phase, const uint32_t* d_in, uint32_t* d_out, uint64_t local_n,
                               uint64_t batch, uint64_t stride, const uint32_t root[8], uint64_t nranks, uint64_t rank,
                               int inverse) {
  if (phase == 2)  // phase 1 on the untransposed exchange layout [source rank][m]
    return dist_phase_impl(c, 1, d_in, d_out, local_n, batch, stride, root, nranks, rank, inverse, nullptr, 1);
  return dist_phase_impl(c, phase, d_in, d_out, local_n, batch, stride, root, nranks, rank, inverse, nullptr, 0);
}

// Phase 0 fused with the transpose: the last pass stores every element directly into the
// owning rank's exchange buffer over NVLink (peer_ptrs[r] = rank r's buffer mapped into this
// process, e.g. torch symmetric memory), so no separate all-to-all or transpose pass runs.
// The caller orders it with a cross-rank barrier before stk_ntt_dist_phase(phase = 2).
STK_API int stk_ntt_dist_phase0_p2p(stk_ctx* c, uint32_t* d_inout, uint64_t local_n, const uint32_t root[8],
                                    uint64_t nranks, uint64_t rank, int inverse, const uint64_t* peer_ptrs) {
  if (!peer_ptrs) return STK_EINVAL;
  return dist_phase_impl(c, 0, d_inout, d_inout, local_n, 1, local_n, root, nranks, rank, inverse, peer_ptrs, 0);
}

// ------------------------------------------------------------------ pointwise helpers

template <class F>
__global__ void vec_op_kernel(int op, const fe* a, const fe* b, fe* out, uint64_t n, const F f) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe x = fe_load(a + i), y = fe_load(b + i), r;
  if (op == 0) r = f.add(x, y);
  else if (op == 1) r = f.sub(x, y);
  else r = f_mul(f, x, y);
  fe_store(out + i, r);
}

STK_API int stk_vec_op(stk_ctx* c, int op, const uint32_t* d_a, const uint32_t* d_b, uint32_t* d_out, uint64_t n) {
  if (!c || op < 0 || op > 2) return STK_EINVAL;
  if (!n) return STK_OK;
  unsigned blocks = (unsigned)((n + 255) / 256);
  return stk_with_field(c, [&](auto f) {
    vec_op_kernel<<<blocks, 256, 0, c->stream>>>(op, (const fe*)d_a, (const fe*)d_b, (fe*)d_out, n, f);
  });
}

STK_API int stk_mul_polys(stk_ctx* c, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                          uint32_t* d_out, uint64_t n, const uint32_t root[8]) {
  if (!c || !d_out || !root) return STK_EINVAL;
  if (na > n || nb > n) return stk_fail(c, STK_EINDEX, "operand longer than the order of the root");
  fe r = stk_load_fe(root);
  void* t;
  STK_TRY(stk_scratch(c, kSlotStage, 2 * n * sizeof(fe), &t));
  fe* x1 = (fe*)t;
  fe* x2 = x1 + n;
  STK_TRY(stk_ntt_dev(c, (const fe*)d_a, na, na, x1, n, n, 1, r, 0, 0));
  STK_TRY(stk_ntt_dev(c, (const fe*)d_b, nb, nb, x2, n, n, 1, r, 0, 0));
  STK_TRY(stk_vec_op(c, 2, (const uint32_t*)x1, (const uint32_t*)x2, (uint32_t*)x1, n));
  // _fft(..., rootz[:0:-1]) without the 1/n factor (starks/fft.py:345)
  STK_TRY(stk_ntt_dev(c, x1, n, n, (fe*)d_out, n, n, 1, r, 1, 0));
  return STK_OK;
}

template <class F>
__global__ void from_tw_kernel(const fe* W, fe* out, uint64_t n, const F f) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i < n) fe_store(out + i, f.from_tw(fe_load(W + i)));
}

STK_API int stk_power_cycle(stk_ctx* c, const uint32_t r32[8], uint64_t n, uint32_t* d_out) {
  if (!c || !r32 || !d_out) return STK_EINVAL;
  if (!n) return STK_OK;
  const fe* W;
  STK_TRY(stk_get_table(c, stk_load_fe(r32), n, &W));
  if (c->is_stark) {
    STK_CUDA(c, cudaMemcpyAsync(d_out, W, n * sizeof(fe), cudaMemcpyDeviceToDevice, c->stream));
  } else {
    unsigned blocks = (unsigned)((n + 255) / 256);
    from_tw_kernel<MontField><<<blocks, 256, 0, c->stream>>>(W, (fe*)d_out, n, c->mont);
    STK_CUDA(c, cudaGetLastError());
  }
  return STK_OK;
}
