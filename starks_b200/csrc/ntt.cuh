// ntt.cuh -- batched radix-2 NTT over Z/p as shared-memory-staged radix-8 passes.
//
// Replaces the reference's recursive decimation-in-time `_fft` / `fft_1d`
// (starks/fft.py:303-331): natural-order input, natural-order output,
// out[k] = sum_j in[j] * w^(jk).  All arithmetic is exact mod p, so any correct
// factorisation is bit-identical to the reference.
//
// Factorisation used here: plain decimation-in-frequency over the global index J
// (n = log2 N bits), cut into 1-3 passes.  A pass owns `k` consecutive index bits
// [lo, lo+k); a CTA stages a tile of C * 2^k elements in shared memory (two planes of
// 16-byte half-elements, XOR-swizzled so every radix-8 round is bank-conflict free), runs the k butterfly levels
// as in-register radix-8 (2^R) rounds -- the first round reads global memory directly, the
// last one writes it directly -- and the final pass stores to the bit-reversed index, which
// makes the output natural-order without a separate permutation pass.  The C "batch"
// positions of a tile are chosen so that global accesses come in C*32-byte runs: the
// lowest index bits in non-final passes, the highest ones (lowest after bit reversal)
// in the final pass, or C whole columns when one pass covers the transform.
//
// Butterfly at level with half-size H:  (a, b) -> (a + b, (a - b) * w^((J mod H) * N/(2H))).
// Twiddles come from one table W[e] = w^e (e < N) kept in HBM in "twiddle form".
#pragma once
#include <algorithm>
#include "ctx.h"
#include "field.cuh"

namespace stk {

struct NttPass {
  int n;         // log2 N
  int lo;        // lowest index bit of this pass
  int k;         // butterfly levels in this pass
  int logC;      // log2 tile batch width
  int logT;      // k + logC
  int c_is_col;  // batch positions are whole columns (single-pass transforms)
  int cb;        // index bit position of the batch bits (when !c_is_col)
  int nl, sl, sh;  // deposit of blockIdx.x into the remaining index bits
  int nrounds;
  int r[8];      // log2 radix of each round
  int final_pass;  // bit-reversed store
  int do_scale;    // multiply by `scale` on the final store (inverse transform)
  uint32_t n_in;   // valid input elements per column; above that the input is zero
  uint32_t batch;  // number of columns
  unsigned long long in_col_stride, out_col_stride;  // elements
  // distributed (multi-GPU four-step) use: the local array holds the elements of a longer
  // transform of order 2^n_tw whose global index is (J << j_shift) | j_or; the final store
  // goes to local position bitrev_{n_tw}(global J) >> out_shift.  Single-GPU: n_tw = n, rest 0.
  // zero-padded inputs (LDE, n_in <= N/8): the first radix-8 round of the first pass sees one
  // non-zero element per group and becomes x[m] = x[0] * w^(J*rev3(m)).  zbit = log2 of the
  // padded input length (32 disables the shortcut).
  int zbit;
  // LDE by cosets (zero-padded input, n_in <= N/8): the transform of order 8*2^n over <w> is run as
  // 8 independent transforms of order 2^n over <w^8>, one per residue r of the OUTPUT index:
  // out[8K + r] = sum_j (c_j * w^(r*j)) * (w^8)^(jK).  Virtual column vc = 8*col + r: real column
  // vc >> cshift for the first pass's input and the final pass's output, residue r = vc mod 8; the
  // first round multiplies c_j by W[(r*j) << cs_shift] (ZS instantiations only) and the final store
  // goes to index (K << cshift) | r.  cshift = 0 everywhere else.
  int cshift;
  int cs_shift;
  int in_virtual;  // this pass reads the virtual columns (not the first pass of a coset transform)
  // LDE with N = 8*n_in: the residue-0 coset <w^8> IS the trace domain <G1>, so out[8K] = trace[K]
  // (starks/stark.py:217-224: no coset shift) and the r = 0 virtual columns need no transform at
  // all -- their CTAs leave at once (ZS instantiations) and the caller copies the trace in.
  int cskip0;
  int tw_shift;  // the table is a longer one: entry e lives at W[e << tw_shift]
  int n_tw;
  int j_shift;
  uint32_t j_or;
  int out_shift;
  // fused transpose of the four-step transform: a non-final pass with peer_on stores element
  // K not locally but into rank (K >> peer_log_chunk)'s buffer, at [this rank][K mod chunk]
  // (P2P stores over NVLink, contiguous 256-byte runs per thread); in_rot makes the next
  // phase read that [source rank][m] layout as if it were [m][source rank].
  // peer_on = 2 (sharded Merkle commit): the FINAL pass stores output row K of column
  // peer_col0 + col into the rank that owns K's leaf range under permute4
  // (starks/merkle_tree.py:11-23): with q = N/4, K = j4*q + d*(q/G) + i goes to rank d, local
  // row j4*(q/G) + i of a (columns x N/G) buffer -- the rows of a local tree in permute4 order.
  int peer_on;
  int peer_log_chunk;
  uint32_t peer_self;
  int peer_g;
  uint32_t peer_col0;
  int in_rot;
  fe* peer_out[8];
  const fe* in;
  fe* out;
  const fe* W;
  fe scale;  // twiddle form
};

// Shared-memory tile: two planes of 16-byte half-elements (limbs 0-3, limbs 4-7), accessed with
// LDS.128 / STS.128.  A 128-bit access is served per quarter-warp, so eight consecutive lanes
// must hit eight different 16-byte bank groups; XOR-ing position bits [3,6) into [0,3) does
// that for every radix-8 round (consecutive lanes differ in bits [0,q) and [q+3, ...)).
__device__ __forceinline__ uint32_t sm_phys(uint32_t pos) { return pos ^ ((pos >> 3) & 7u); }

// TRIV: the round's lowest level has global stride 1 (last round of the final pass of a whole
// transform), so its exponent base is 0 and every mm == 0 twiddle is w^0 = 1: 7 of the 12
// multiplies of a radix-8 round (3 of 4 for radix-4, the only one for radix-2) are skipped.
// ZS: 0 = plain pass; 1 = first pass of a zero-padded transform (expansion round or coset scaling
// on load, real input column = virtual >> cshift; also the interleaved store, for single-pass
// coset transforms); 2 = final pass of a coset transform (interleaved store only).  The plain
// instantiation carries none of this: even a few extra integer instructions in its load / store
// paths cost 2 % on the 64 x 2^20 transform (measured, tools/gpu_altlib.py).
template <class F, int R, int ZS, bool TRIV>
__device__ __forceinline__ void ntt_round(const NttPass& A, const F& f, uint32_t* sm, uint32_t T,
                                          uint32_t Jcta, uint32_t col0, int a, bool first, bool last) {
  constexpr int M = 1 << R;
  const int logS = a + A.logC;
  const uint32_t S = 1u << logS;
  const uint32_t Cm = (1u << A.logC) - 1u;
  const uint32_t ngroups = T >> R;
  const int gshift = A.lo + a;  // global index stride of m is 2^gshift
  uint4* sm4 = reinterpret_cast<uint4*>(sm);
  for (uint32_t g = threadIdx.x; g < ngroups; g += blockDim.x) {
    const uint32_t pos0 = ((g >> logS) << (logS + R)) | (g & (S - 1u));
    const uint32_t j0 = pos0 >> A.logC, c0 = pos0 & Cm;
    const uint32_t J0 = Jcta | (j0 << A.lo) | (A.c_is_col ? 0u : (c0 << A.cb));
    const uint32_t col = A.c_is_col ? (col0 + c0) : col0;
    const bool col_ok = col < A.batch;
    fe x[M];
    if (first) {
      const uint32_t icol = (ZS == 1 && !A.in_virtual) ? (col >> A.cshift) : col;
      const fe* src = A.in + (unsigned long long)icol * A.in_col_stride;
#pragma unroll
      for (int m = 0; m < M; ++m) {
        uint32_t J = J0 + ((uint32_t)m << gshift);
        uint32_t Jm = A.in_rot ? (((J & ((1u << A.in_rot) - 1u)) << (A.n - A.in_rot)) | (J >> A.in_rot)) : J;
        x[m] = (col_ok && J < A.n_in) ? fe_load(src + Jm) : fe_zero();
      }
      if (ZS == 1 && A.cshift && !A.in_virtual) {  // coset scaling c_j * w^(r*j); r = 0 needs none
        const uint32_t r = col & ((1u << A.cshift) - 1u);
        if (r) {
#pragma unroll
          for (int m = 0; m < M; ++m) {
            const uint32_t J = J0 + ((uint32_t)m << gshift);
            x[m] = f.mul_tw(x[m], fe_load_ro(A.W + ((unsigned long long)(r * J) << A.cs_shift)));
          }
        }
      }
    } else {
#pragma unroll
      for (int m = 0; m < M; ++m) {
        uint32_t ph = sm_phys(pos0 + (uint32_t)m * S);
        uint4 lo = sm4[ph], hi = sm4[T + ph];
        x[m].v[0] = lo.x; x[m].v[1] = lo.y; x[m].v[2] = lo.z; x[m].v[3] = lo.w;
        x[m].v[4] = hi.x; x[m].v[5] = hi.y; x[m].v[6] = hi.z; x[m].v[7] = hi.w;
      }
    }
    // exponent of the last (smallest-half) level of this round
    if (ZS == 1 && first && R == 3 && gshift >= A.zbit && gshift == A.n - 3) {
      // Zero-padded input (LDE, N = 8 * n_in): only x[0] is non-zero and the three levels of
      // this round reduce to x[m] = x[0] * w^(J0 * rev3(m)) -- seven multiplies, no add/sub,
      // instead of twelve butterflies on mostly-zero data.
      if (J0 < (1u << A.zbit)) {
        const fe x0 = x[0];
#pragma unroll
        for (int m = 1; m < M; ++m) {
          const uint32_t r3 = ((m & 1) << 2) | (m & 2) | ((m >> 2) & 1);
          x[m] = f.mul_tw(x0, fe_load_ro(A.W + ((unsigned long long)(J0 * r3) << A.tw_shift)));
        }
      }
    } else {
    const int ggs = gshift + A.j_shift;  // log2 of the global index stride of m
    const uint32_t Jl = ((J0 << A.j_shift) | A.j_or) & ((1u << ggs) - 1u);
    const uint32_t er = Jl << (A.n_tw - 1 - ggs);
#pragma unroll
    for (int lv = 0; lv < R; ++lv) {
      const int lh = R - 1 - lv;  // log2 of half size in m units
      const int hm = 1 << lh;
#pragma unroll
      for (int mm = 0; mm < hm; ++mm) {
        const bool unit = TRIV && mm == 0;  // er == 0 here
        const uint32_t e = (er >> lh) + ((uint32_t)mm << (A.n_tw - 1 - lh));
        fe tw;
        if (!unit) tw = fe_load_ro(A.W + ((unsigned long long)e << A.tw_shift));
#pragma unroll
        for (int blk = 0; blk < (M >> (lh + 1)); ++blk) {
          const int i0 = blk * 2 * hm + mm, i1 = i0 + hm;
          fe s = f.add(x[i0], x[i1]);
          fe d = f.sub(x[i0], x[i1]);
          x[i0] = s;
          x[i1] = unit ? d : f.mul_tw(d, tw);
        }
      }
    }
    }  // butterfly levels
    if (last && !A.peer_on) {
      if (col_ok) {
        const bool ovirt = ZS == 0 || !A.final_pass || !A.cshift;  // non-final passes keep virtual columns apart
        fe* dst = A.out + (unsigned long long)(ovirt ? col : (col >> A.cshift)) * A.out_col_stride;
#pragma unroll
        for (int m = 0; m < M; ++m) {
          uint32_t J = J0 + ((uint32_t)m << gshift);
          uint32_t K = A.final_pass ? ((__brev((J << A.j_shift) | A.j_or) >> (32 - A.n_tw)) >> A.out_shift) : J;
          if (!ovirt) K = (K << A.cshift) | (col & ((1u << A.cshift) - 1u));
          fe v = x[m];
          if (A.do_scale) v = f.mul_tw(v, A.scale);
          fe_store(dst + K, v);
        }
      }
    } else {
#pragma unroll
      for (int m = 0; m < M; ++m) {
        uint32_t ph = sm_phys(pos0 + (uint32_t)m * S);
        sm4[ph] = make_uint4(x[m].v[0], x[m].v[1], x[m].v[2], x[m].v[3]);
        sm4[T + ph] = make_uint4(x[m].v[4], x[m].v[5], x[m].v[6], x[m].v[7]);
      }
    }
  }
}

template <class F, int MAXR, int MAXT = (4096 >> MAXR), int MINB = 1, int ZS = 0>
__global__ void __launch_bounds__(MAXT, MINB) ntt_pass_kernel(const NttPass A, const F f) {
  extern __shared__ __align__(16) uint32_t sm[];
  const uint32_t T = 1u << A.logT;
  // single-pass transforms put the column groups on grid.x (no 65535 limit), tiles otherwise
  const uint32_t bx = blockIdx.x, by = blockIdx.y;
  const uint32_t xb = A.c_is_col ? 0u : bx;
  const uint32_t Jcta = ((xb & ((1u << A.nl) - 1u)) << A.sl) | ((xb >> A.nl) << A.sh);
  const uint32_t col0 = A.c_is_col ? (bx << A.logC) : by;
  if (ZS != 0 && A.cskip0 && !A.c_is_col && (col0 & ((1u << A.cshift) - 1u)) == 0u) return;  // whole CTA
  int a = A.k;
  for (int rd = 0; rd < A.nrounds; ++rd) {
    const int r = A.r[rd];
    a -= r;
    const bool first = rd == 0, last = rd == A.nrounds - 1;
    if (last && A.lo + a + A.j_shift == 0) {  // global stride 1: unit twiddles (see TRIV)
      if (MAXR >= 3 && r == 3) ntt_round<F, (MAXR >= 3 ? 3 : 2), ZS, true>(A, f, sm, T, Jcta, col0, a, first, last);
      else if (r == 2) ntt_round<F, 2, ZS, true>(A, f, sm, T, Jcta, col0, a, first, last);
      else ntt_round<F, 1, ZS, true>(A, f, sm, T, Jcta, col0, a, first, last);
    } else if (MAXR >= 3 && r == 3) ntt_round<F, (MAXR >= 3 ? 3 : 2), ZS, false>(A, f, sm, T, Jcta, col0, a, first, last);
    else if (r == 2) ntt_round<F, 2, ZS, false>(A, f, sm, T, Jcta, col0, a, first, last);
    else ntt_round<F, 1, ZS, false>(A, f, sm, T, Jcta, col0, a, first, last);
    if (!last) __syncthreads();
  }
  if (A.peer_on == 2) {
    // Fused leaf exchange of the sharded commit: rows leave for their leaf owners, consecutive
    // lanes on consecutive 16-byte chunks of consecutive output rows (runs of C rows).
    __syncthreads();
    const uint4* s4 = reinterpret_cast<const uint4*>(sm);
    const uint32_t Cm = (1u << A.logC) - 1u;
    const int qb = A.n - 2 - A.peer_g;  // log2 of rows per (quarter, owner)
    for (uint32_t q = threadIdx.x; q < 2u * T; q += blockDim.x) {
      const uint32_t e = q >> 1, h = q & 1u;
      const uint32_t jr = e >> A.logC, cr = e & Cm;
      const uint32_t c = A.logC ? (__brev(cr) >> (32 - A.logC)) : 0u;
      const uint32_t j = __brev(jr) >> (32 - A.k);
      const uint32_t J = Jcta | (j << A.lo) | (c << A.cb);
      const uint32_t K = __brev(J) >> (32 - A.n);
      const uint32_t j4 = K >> (A.n - 2), rem = K & ((1u << (A.n - 2)) - 1u);
      const uint32_t d = rem >> qb, i = rem & ((1u << qb) - 1u);
      const unsigned long long off =
          ((unsigned long long)(A.peer_col0 + col0) << (A.n - A.peer_g)) + ((j4 << qb) | i);
      reinterpret_cast<uint4*>(A.peer_out[d] + off)[h] = s4[h * T + sm_phys((j << A.logC) | c)];
    }
  } else if (A.peer_on) {
    // Fused exchange: the finished tile sits in shared memory; write it to the owning ranks'
    // buffers with consecutive lanes on consecutive 16-byte chunks, so every warp store is a
    // contiguous 512-byte run over NVLink (a direct per-thread store would issue 16/32-byte
    // fragments 256 bytes apart and reach a quarter of the link rate).
    __syncthreads();
    const uint4* s4 = reinterpret_cast<const uint4*>(sm);
    const uint32_t Lm = (1u << A.k) - 1u, cmask = (1u << A.peer_log_chunk) - 1u;
    for (uint32_t q = threadIdx.x; q < 2u * T; q += blockDim.x) {
      const uint32_t e = q >> 1, h = q & 1u;
      const uint32_t c = e >> A.k, j = e & Lm;
      const uint32_t J = Jcta | (j << A.lo) | (A.c_is_col ? 0u : (c << A.cb));
      const uint4 v = s4[h * T + sm_phys((j << A.logC) | c)];
      fe* pd = A.peer_out[J >> A.peer_log_chunk];
      reinterpret_cast<uint4*>(pd + ((A.peer_self << A.peer_log_chunk) | (J & cmask)))[h] = v;
    }
  }
}

// Host-side launcher of one ntt_pass_kernel instantiation, whose tiles hold up to (1 << MAXR) * MAXT
// elements.  Each ntt_pass_*.cu instantiates one so that nvcc compiles the heavy kernels in parallel.
template <class F, int MAXR, int MAXT, int MINB, int ZS>
static int launch_pass_r(stk_ctx* c, cudaStream_t s, const NttPass& P, const F& f) {
  static bool attr_done[64] = {};  // cudaFuncSetAttribute is per device
  if (!attr_done[c->device & 63]) {
    STK_CUDA(c, cudaFuncSetAttribute(ntt_pass_kernel<F, MAXR, MAXT, MINB, ZS>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * (1 << MAXR) * MAXT));
    attr_done[c->device & 63] = true;
  }
  const uint32_t T = 1u << P.logT;
  if (T > (1u << MAXR) * MAXT) return stk_fail(c, STK_EUNSUPPORTED, "tile larger than this instantiation");
  unsigned threads = std::max(1u, T >> MAXR);
  uint64_t tiles = P.c_is_col ? 1 : ((1ull << P.n) >> P.logT);
  uint64_t cols = P.c_is_col ? ((P.batch + (1u << P.logC) - 1) >> P.logC) : P.batch;
  if (!P.c_is_col && cols > 65535) return stk_fail(c, STK_EUNSUPPORTED, "more than 65535 columns of a multi-pass transform");
  if (cols > 0x7fffffffull) return stk_fail(c, STK_EUNSUPPORTED, "batch too large");
  dim3 grid(P.c_is_col ? (unsigned)cols : (unsigned)tiles, P.c_is_col ? 1u : (unsigned)cols);
  size_t smem = (P.nrounds > 1 || P.peer_on) ? (size_t)32 * T : 0;
  ntt_pass_kernel<F, MAXR, MAXT, MINB, ZS><<<grid, threads, smem, s>>>(P, f);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

// W[m + i] = W[i] * wm  for i < m  (table doubling; both operands in twiddle form)
template <class F>
__global__ void twiddle_extend_kernel(fe* W, unsigned long long m, unsigned long long total, fe wm, const F f) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  if (i < m && m + i < total) fe_store(W + m + i, f.mul_tw(fe_load(W + i), wm));
}

}  // namespace stk
