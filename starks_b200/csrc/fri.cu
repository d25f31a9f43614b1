// fri.cu -- FRI fold-by-4 (the "column" of one FRI layer).  Replaces the per-row Lagrange
// interpolation of SmoothSubgroupFRI.generate_proximity_proof (starks/fri.py:236-242) via
// multi_interp_4 / multi_inv (starks/poly_utils.py:301-320, 412-440) and Polynomial.__call__
// (starks/polynomial.py:158-164) by its closed form (SURVEY.md App. C.3):
//
//   q = n/4, iota = w^q (primitive 4th root), t = x * w^(-i)
//   column[i] = 1/4 * sum_k t^k * sum_j values[i + q*j] * iota^(-jk)
//
// i.e. a 4-point inverse DFT in the variable X / w^i (multiplications by iota only) followed
// by Horner at t.  Exact arithmetic mod p, hence bit-identical to the interpolation route.
#include <algorithm>
#include "ctx.h"

using namespace stk;

namespace {

// i0: index of this launch's first quad in the WHOLE layer (0 unless the layer is sharded by
// leaf range: a rank then holds the quads i0 .. i0 + q - 1 as four runs of q rows each).
template <class F>
__global__ void __launch_bounds__(256) fri_fold4_kernel(const fe* __restrict__ vals, uint64_t q, uint64_t i0,
                                                        const fe* __restrict__ Winv, uint64_t wstride, fe x_plain, fe iota_tw,
                                                        fe quarter_tw, fe* __restrict__ out, const F f) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (i >= q) return;
  fe v0 = fe_load(vals + i), v1 = fe_load(vals + i + q), v2 = fe_load(vals + i + 2 * q), v3 = fe_load(vals + i + 3 * q);
  fe s02 = f.add(v0, v2), d02 = f.sub(v0, v2), s13 = f.add(v1, v3), d13 = f.sub(v1, v3);
  fe m = f.mul_tw(d13, iota_tw);
  fe c0 = f.add(s02, s13), c2 = f.sub(s02, s13);  // 4*b0, 4*b2
  fe c1 = f.sub(d02, m), c3 = f.add(d02, m);      // 4*b1, 4*b3
  fe t = f.mul_tw(x_plain, fe_load_ro(Winv + (i0 + i) * wstride));  // x * w^-(i0+i), plain
  fe t_tw = f.to_tw(t);
  fe r = f.add(f.mul_tw(c3, t_tw), c2);
  r = f.add(f.mul_tw(r, t_tw), c1);
  r = f.add(f.mul_tw(r, t_tw), c0);
  fe_store(out + i, f.mul_tw(r, quarter_tw));
}

}  // namespace

// launch only: w a primitive n-th root (checked by the caller), winv = w^-1, x reduced
// the layer has n points; this launch folds the q_run quads i0 .. i0 + q_run - 1, held at d_vals as
// four runs of q_run values (q_run = n/4, i0 = 0: the whole layer)
static int fri_fold4_launch(stk_ctx* c, const uint32_t* d_vals, uint64_t n, const fe& w, const fe& winv, const fe& x,
                            const fe& quarter_tw, uint32_t* d_out, uint64_t q_run = 0, uint64_t i0 = 0) {
  const uint64_t q = n / 4;
  if (!q_run) q_run = q;
  const fe* Winv;
  uint64_t wstride = 1;
  STK_TRY(stk_get_table_strided(c, winv, n, &Winv, &wstride));
  fe iota_tw = stk_h_to_tw(c, stk_h_pow(c, w, q));
  unsigned blocks = (unsigned)((q_run + 255) / 256);
  return stk_with_field(c, [&](auto f) {
    fri_fold4_kernel<<<blocks, 256, 0, c->stream>>>((const fe*)d_vals, q_run, i0, Winv, wstride, x, iota_tw, quarter_tw,
                                                    (fe*)d_out, f);
  });
}

STK_API int stk_fri_fold4(stk_ctx* c, const uint32_t* d_vals, uint64_t n, const uint32_t root[8],
                          const uint32_t special_x[8], uint32_t* d_out) {
  if (!c || !d_vals || !d_out || !root || !special_x) return STK_EINVAL;
  if (n == 0 || (n & 3)) return stk_fail(c, STK_EINVAL, "fold-by-4 needs a length divisible by 4");
  fe w = stk_load_fe(root);
  if (!stk_h_primitive(c, w, n))
    return stk_fail(c, STK_EINVAL, "root is not a primitive n-th root of unity");
  fe x = host::reduce(stk_load_fe(special_x), c->p);  // fri.py:229 does not reduce; products do
  fe quarter_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(4), c->p)));
  return fri_fold4_launch(c, d_vals, n, w, stk_h_inv(c, w), x, quarter_tw, d_out);
}

// stk_fri_fold4 for a layer sharded by leaf range (SURVEY.md 8e: "shard layer 0 by index range
// aligned to fold quads"): d_rows holds the four runs {j*q + i0 + t : t < q_run}, j < 4, of the
// n-point layer back to back (the row order of a rank's local tree under permute4), d_out
// receives column[i0 .. i0 + q_run).
STK_API int stk_fri_fold4_rows(stk_ctx* c, const uint32_t* d_rows, uint64_t n, const uint32_t root[8],
                               const uint32_t special_x[8], uint64_t q_run, uint64_t i0, uint32_t* d_out) {
  if (!c || !d_rows || !d_out || !root || !special_x) return STK_EINVAL;
  if (n == 0 || (n & 3) || q_run == 0 || i0 + q_run > n / 4)
    return stk_fail(c, STK_EINVAL, "fold-by-4 rows: need n divisible by 4 and i0 + q_run <= n/4");
  fe w = stk_load_fe(root);
  if (!stk_h_primitive(c, w, n))
    return stk_fail(c, STK_EINVAL, "root is not a primitive n-th root of unity");
  fe x = host::reduce(stk_load_fe(special_x), c->p);
  fe quarter_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(4), c->p)));
  return fri_fold4_launch(c, d_rows, n, w, stk_h_inv(c, w), x, quarter_tw, d_out, q_run, i0);
}

// ------------------------------------------------------------------------------------------
// Whole commit phase of SmoothSubgroupFRI.generate_proximity_proof (starks/fri.py:189-266) in
// one call: per layer the fold, the column's tree, the Fiat-Shamir indices (host BLAKE2s of
// the 32-byte root, starks/utils.py:60-90) and the branch gathers, with ONE host
// synchronisation per layer (the root the next challenge is derived from) and one download of
// all opened branches at the end.
//
// Output (h_out, packed), for every fold layer in order:
//   root2 (32 B) | k records of the column tree (branch of y) | 4k records of the layer's own
//   tree (branches of y, y+q, y+2q, y+3q for each y, in that order)
// followed by the final layer's values as 32-byte big-endian words (fri.py:212-214).  A record
// is what stk_merkle_paths returns: leaf | sibling leaf | sibling nodes up to the root.
// k = security for the first layer and 40 below it (the reference's recursive call does not
// forward the argument, fri.py:262-266).
// ------------------------------------------------------------------------------------------
#include <vector>
#include "hostblake2s.h"

namespace {

// get_pseudorandom_indices (starks/utils.py:60-90)
int fri_indices(stk_ctx* c, const uint8_t root[32], uint64_t modulus, uint64_t count, uint64_t exclude,
                std::vector<uint64_t>& out) {
  if (modulus >= (1ull << 24)) return stk_fail(c, STK_EINVAL, "index modulus must be below 2^24 (utils.py:69)");
  std::vector<uint8_t> data(root, root + 32);
  while (data.size() < 4 * count) {
    uint8_t d[32];
    host::blake2s_256(data.data() + data.size() - 32, 32, d);
    data.insert(data.end(), d, d + 32);
  }
  out.resize(count);
  const uint64_t real = exclude ? modulus * (exclude - 1) / exclude : modulus;
  if (real == 0) return stk_fail(c, STK_EINVAL, "empty index range");
  for (uint64_t i = 0; i < count; ++i) {
    const uint8_t* w = data.data() + 4 * i;
    uint64_t x = (((uint64_t)w[0] << 24) | ((uint64_t)w[1] << 16) | ((uint64_t)w[2] << 8) | w[3]) % real;
    out[i] = exclude ? x + 1 + x / (exclude - 1) : x;
  }
  return STK_OK;
}

uint64_t rec_bytes_for(uint64_t n) { return 64 + 32ull * (stk_ilog2(n) - 1); }

}  // namespace

// get_pseudorandom_indices (starks/utils.py:60-90) exactly as the FRI driver derives them; needs no
// device (ctx may be NULL), so the host BLAKE2s and the index rule are testable on a CPU-only box.
STK_API int stk_pseudorandom_indices(stk_ctx* c, const uint8_t entropy[32], uint64_t modulus, uint64_t count,
                                     uint64_t exclude_multiples_of, uint64_t* h_out) {
  if (!entropy || !h_out) return STK_EINVAL;
  if (exclude_multiples_of == 1) return stk_fail(c, STK_EINVAL, "exclude_multiples_of = 1 leaves no positions");
  std::vector<uint64_t> v;
  STK_TRY(fri_indices(c, entropy, modulus, count, exclude_multiples_of, v));
  for (uint64_t i = 0; i < count; ++i) h_out[i] = v[i];
  return STK_OK;
}

STK_API int stk_fri_prove(stk_ctx* c, const uint32_t* d_vals0, uint64_t n0, const uint8_t* d_nodes0,
                          const uint8_t* h_root0, const uint32_t root[8], uint64_t maxdeg_plus_1, uint64_t exclude,
                          uint64_t security, uint8_t* h_out, uint64_t out_cap, uint64_t* out_len) {
  if (!c || !d_vals0 || !root || !h_out || !out_len || (d_nodes0 && !h_root0)) return STK_EINVAL;
  if (n0 < 4 || (n0 & (n0 - 1))) return stk_fail(c, STK_EUNSUPPORTED, "FRI driver needs a power-of-two domain");
  if (exclude == 1) return stk_fail(c, STK_EINVAL, "exclude_multiples_of = 1 leaves no positions");
  // layer geometry
  struct Layer { uint64_t n, q, k, rec1, rec2, idx_off, out_off; };
  std::vector<Layer> L;
  uint64_t n = n0, md = maxdeg_plus_1, k = security, store = 0, stage = 0, total = 0;
  while (md > 16) {
    if (n < 16) return stk_fail(c, STK_EUNSUPPORTED, "layer of %llu values cannot be folded and committed", (unsigned long long)n);
    Layer l;
    l.n = n; l.q = n / 4; l.k = k;
    l.rec1 = rec_bytes_for(n); l.rec2 = rec_bytes_for(l.q);
    l.idx_off = stage; stage += 5 * k * 8;
    l.out_off = stage; stage += k * l.rec2 + 4 * k * l.rec1;
    total += 32 + k * l.rec2 + 4 * k * l.rec1;
    store += 2 * l.q * 32;
    L.push_back(l);
    n /= 4; md /= 4; k = 40;
  }
  const uint64_t n_final = n;
  total += 32 * n_final;
  *out_len = total;
  if (out_cap < total) return stk_fail(c, STK_EINVAL, "output buffer too small: need %llu bytes", (unsigned long long)total);
  void *sv, *st;
  STK_TRY(stk_scratch(c, kSlotFriLayers, std::max<uint64_t>(store + (d_nodes0 ? 0 : 32 * n0), 32), &sv));
  STK_TRY(stk_scratch(c, kSlotFriStage, std::max<uint64_t>(stage, 32), &st));
  uint8_t* sbase = (uint8_t*)sv;
  uint8_t* stg = (uint8_t*)st;
  const uint32_t* vals = d_vals0;
  const uint8_t* nodes = d_nodes0;
  uint8_t cur_root[32];
  if (nodes) memcpy(cur_root, h_root0, 32);
  else {
    uint8_t* nb = sbase + store;
    STK_TRY(stk_merkle_commit(c, vals, n0, 1, n0, nb, cur_root));   // m = merkelize(values), fri.py:224
    nodes = nb;
  }
  fe w = host::reduce(stk_load_fe(root), c->p);
  if (!stk_h_primitive(c, w, n0)) return stk_fail(c, STK_EINVAL, "root is not a primitive n-th root of unity");
  fe winv = stk_h_inv(c, w);  // layer l folds with w^(4^l): both follow by two squarings
  const fe quarter_tw = stk_h_to_tw(c, stk_h_inv(c, host::reduce(host::from_u64(4), c->p)));
  std::vector<uint8_t> roots(32 * L.size());
  std::vector<uint64_t> ys, idx;
  uint64_t soff = 0;
  for (size_t li = 0; li < L.size(); ++li) {
    const Layer& l = L[li];
    uint32_t sx[8];  // special_x = the root read as a big-endian integer, unreduced (fri.py:229)
    for (int i = 0; i < 8; ++i)
      sx[i] = ((uint32_t)cur_root[28 - 4 * i] << 24) | ((uint32_t)cur_root[29 - 4 * i] << 16) |
              ((uint32_t)cur_root[30 - 4 * i] << 8) | cur_root[31 - 4 * i];
    uint32_t* col = (uint32_t*)(sbase + soff);
    uint8_t* colnodes = sbase + soff + l.q * 32;
    soff += 2 * l.q * 32;
    fe sxe;
    for (int i = 0; i < 8; ++i) sxe.v[i] = sx[i];
    STK_TRY(fri_fold4_launch(c, vals, l.n, w, winv, host::reduce(sxe, c->p), quarter_tw, col));  // fri.py:236-242
    uint8_t* root2 = roots.data() + 32 * li;
    STK_TRY(stk_merkle_commit(c, col, l.q, 1, l.q, colnodes, root2));          // :243 (synchronises)
    STK_TRY(fri_indices(c, root2, l.q, l.k, exclude, ys));                     // :246-247
    idx.resize(5 * l.k);
    for (uint64_t i = 0; i < l.k; ++i) {
      idx[i] = ys[i];
      for (uint64_t j = 0; j < 4; ++j) idx[l.k + 4 * i + j] = ys[i] + l.q * j;
    }
    uint64_t* d_idx = (uint64_t*)(stg + l.idx_off);
    // pageable source: the copy is staged before the call returns, idx can be reused
    STK_CUDA(c, cudaMemcpyAsync(d_idx, idx.data(), 5 * l.k * 8, cudaMemcpyHostToDevice, c->stream));
    uint32_t* rec = (uint32_t*)(stg + l.out_off);
    STK_TRY(stk_merkle_paths_dev(c, (const fe*)col, l.q, 1, l.q, colnodes, d_idx, l.k, rec, l.rec2));
    STK_TRY(stk_merkle_paths_dev(c, (const fe*)vals, l.n, 1, l.n, nodes, d_idx + l.k, 4 * l.k,
                                 (uint32_t*)((uint8_t*)rec + l.k * l.rec2), l.rec1));
    vals = col; nodes = colnodes;
    memcpy(cur_root, root2, 32);
    w = stk_h_pow(c, w, 4);
    winv = stk_h_pow(c, winv, 4);
  }
  // one download: every layer's records, then the final values (big-endian on the way out)
  uint8_t* o = h_out;
  for (size_t li = 0; li < L.size(); ++li) {
    const Layer& l = L[li];
    memcpy(o, roots.data() + 32 * li, 32);
    o += 32;
    const uint64_t bytes = l.k * l.rec2 + 4 * l.k * l.rec1;
    STK_CUDA(c, cudaMemcpyAsync(o, stg + l.out_off, bytes, cudaMemcpyDeviceToHost, c->stream));
    o += bytes;
  }
  std::vector<uint32_t> fin(8 * n_final);
  STK_CUDA(c, cudaMemcpyAsync(fin.data(), vals, 32 * n_final, cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  for (uint64_t i = 0; i < n_final; ++i)
    for (int lb = 0; lb < 8; ++lb) {
      const uint32_t v = fin[8 * i + 7 - lb];
      o[32 * i + 4 * lb] = (uint8_t)(v >> 24); o[32 * i + 4 * lb + 1] = (uint8_t)(v >> 16);
      o[32 * i + 4 * lb + 2] = (uint8_t)(v >> 8); o[32 * i + 4 * lb + 3] = (uint8_t)v;
    }
  return STK_OK;
}
