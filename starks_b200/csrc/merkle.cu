// merkle.cu -- BLAKE2s Merkle commitment over evaluation columns, level-by-level reduction
// and branch extraction.  Replaces merkelize / permute4 / merkelize_polynomial_evaluations /
// mk_branch of starks/merkle_tree.py:11-68, 94-119.
//
// Tree layout (identical to the reference's list): heap order, root at index 1, internal
// node i = BLAKE2s(node 2i || node 2i+1), leaves (NOT hashed) at indices [n, 2n) in
// permute4 order: leaf position l holds original row (l mod 4) * n/4 + l div 4.  On the
// device only the n internal nodes are stored (32 bytes each, entry 0 unused); leaves stay
// where they are -- in the evaluation columns -- and are serialised on the fly:
// leaf(row) = concat over columns of the 32-byte big-endian value (merkle_tree.py:116-118).
#include <algorithm>
#include "blake2s.cuh"
#include "ctx.h"

using namespace stk;

namespace {

// Bottom level over column leaves.  One thread per node i in [n/2, n): hashes
// leaf(2i-n) || leaf(2i-n+1) = 2*ncols values = ncols 64-byte blocks.
__global__ void __launch_bounds__(256) merkle_leaf_pairs_cols_kernel(const fe* __restrict__ cols, uint64_t n,
                                                                      uint32_t ncols, uint64_t col_stride,
                                                                      uint32_t* __restrict__ nodes) {
  const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t half = n >> 1, q = n >> 2;
  if (i >= half) return;
  const uint64_t l0 = 2 * i;
  const uint64_t x0 = (l0 & 3) * q + (l0 >> 2), x1 = x0 + q;
  uint32_t h[8];
  b2s_init(h);
  const uint32_t nblk = ncols;  // 2*ncols values, two per block
  for (uint32_t b = 0; b < nblk; ++b) {
    uint32_t m[16];
#pragma unroll
    for (int half_blk = 0; half_blk < 2; ++half_blk) {
      uint32_t s = 2 * b + half_blk;
      const fe* src = (s < ncols) ? (cols + (uint64_t)s * col_stride + x0)
                                  : (cols + (uint64_t)(s - ncols) * col_stride + x1);
      fe v = fe_load(src);
#pragma unroll
      for (int k = 0; k < 8; ++k) m[8 * half_blk + k] = bswap32(v.v[7 - k]);
    }
    b2s_compress(h, m, 64u * (b + 1), b + 1 == nblk);
  }
  uint4* dst = reinterpret_cast<uint4*>(nodes + 8 * (half + i));
  dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
  dst[1] = make_uint4(h[4], h[5], h[6], h[7]);
}

// Bottom level over raw byte leaves of any width (merkelize on bytes, merkle_tree.py:46-53).
// Leaves are given in ORIGINAL order; np = 4*(n/4) leaves enter the tree.
__global__ void __launch_bounds__(128) merkle_leaf_pairs_raw_kernel(const uint8_t* __restrict__ leaves, uint64_t np,
                                                                     uint64_t leaf_len, uint64_t first,
                                                                     uint64_t count, uint32_t* __restrict__ nodes) {
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= count) return;
  const uint64_t i = first + t;  // node whose children are leaves: 2i >= np
  const uint64_t q = np >> 2;
  const uint64_t l0 = 2 * i - np;
  const uint64_t x0 = (l0 & 3) * q + (l0 >> 2), x1 = ((l0 + 1) & 3) * q + ((l0 + 1) >> 2);
  const uint64_t total = 2 * leaf_len;
  uint32_t h[8];
  b2s_init(h);
  uint64_t off = 0;
  do {
    uint32_t m[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) m[k] = 0;
    uint64_t take = total - off < 64 ? total - off : 64;
    for (uint64_t bi = 0; bi < take; ++bi) {
      uint64_t pos = off + bi;
      uint8_t byte = pos < leaf_len ? leaves[x0 * leaf_len + pos] : leaves[x1 * leaf_len + (pos - leaf_len)];
      m[bi >> 2] |= (uint32_t)byte << (8 * (bi & 3));
    }
    off += take;
    b2s_compress(h, m, (uint32_t)off, off == total);
  } while (off < total);
#pragma unroll
  for (int k = 0; k < 8; ++k) nodes[8 * i + k] = h[k];
}

// One heap level: node i = H(node 2i || node 2i+1) for i in [first, first+count).
__global__ void __launch_bounds__(256) merkle_level_kernel(uint32_t* __restrict__ nodes, uint64_t first, uint64_t count) {
  const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (t >= count) return;
  const uint64_t i = first + t;
  const uint4* src = reinterpret_cast<const uint4*>(nodes + 16 * i);
  uint4 a = src[0], b = src[1], c = src[2], d = src[3];
  uint32_t m[16] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
  uint32_t h[8];
  b2s_init(h);
  b2s_compress(h, m, 64u, true);
  uint4* dst = reinterpret_cast<uint4*>(nodes + 8 * i);
  dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
  dst[1] = make_uint4(h[4], h[5], h[6], h[7]);
}

// All levels below `top` (a power of two <= 1024) in one CTA: nodes [1, top).
__global__ void __launch_bounds__(512) merkle_top_kernel(uint32_t* __restrict__ nodes, uint32_t top, uint64_t np) {
  for (uint32_t lo = top >> 1; lo >= 1; lo >>= 1) {
    for (uint32_t i = lo + threadIdx.x; i < 2 * lo && i < np; i += blockDim.x) {
      if (2ull * i >= np) continue;  // children are leaves: done by the leaf kernel
      uint32_t m[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) m[k] = nodes[16 * i + k];
      uint32_t h[8];
      b2s_init(h);
      b2s_compress(h, m, 64u, true);
#pragma unroll
      for (int k = 0; k < 8; ++k) nodes[8 * i + k] = h[k];
    }
    __syncthreads();
  }
}

// Branches (mk_branch, merkle_tree.py:59-68) for column-leaf trees.  Output record per
// query, as 32-bit words: own leaf (8*ncols) | sibling leaf (8*ncols) | sibling nodes up
// to the root (8 words each).
__global__ void __launch_bounds__(128) merkle_paths_cols_kernel(const fe* __restrict__ cols, uint64_t n, uint32_t ncols,
                                                                 uint64_t col_stride, const uint32_t* __restrict__ nodes,
                                                                 const uint64_t* __restrict__ idx, uint32_t* __restrict__ out,
                                                                 uint64_t rec_words) {
  const uint64_t qi = blockIdx.x;
  const uint64_t x = idx[qi], ld4 = n >> 2;
  const uint64_t perm = x / ld4 + 4 * (x % ld4);
  const uint64_t index = perm + n;
  uint32_t* o = out + qi * rec_words;
  const uint32_t lw = 8 * ncols;
  for (uint32_t w = threadIdx.x; w < 2 * lw; w += blockDim.x) {
    uint32_t which = w / lw, ww = w % lw, c = ww >> 3, k = ww & 7;
    uint64_t lp = which ? (perm ^ 1) : perm;
    uint64_t row = (lp & 3) * ld4 + (lp >> 2);
    o[w] = bswap32(cols[(uint64_t)c * col_stride + row].v[7 - k]);
  }
  uint32_t d = 1;
  for (uint64_t id = index >> 1; id > 1; id >>= 1, ++d) {
    if (threadIdx.x < 8) o[2 * lw + 8 * (d - 1) + threadIdx.x] = nodes[8 * (id ^ 1) + threadIdx.x];
  }
}

// verify_branch (starks/merkle_tree.py:71-86) for many branches of one tree: one thread per
// record (own leaf | sibling leaf | sibling nodes up to the root), ok[r] = recomputed root == root.
__global__ void __launch_bounds__(128) verify_branches_kernel(const uint32_t* __restrict__ rec, uint64_t rec_words,
                                                               const uint64_t* __restrict__ idx, uint64_t k, uint64_t n,
                                                               uint32_t leaf_words, uint32_t depth,
                                                               const uint32_t* __restrict__ root, uint8_t* __restrict__ ok) {
  const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  if (r >= k) return;
  const uint32_t* R = rec + r * rec_words;
  const uint64_t x = idx[r], q = n >> 2;
  uint64_t index = x / q + 4 * (x % q) + n;   // get_index_in_permuted + leaf offset (:26-33, :73-78)
  uint32_t h[8];
  b2s_init(h);
  const uint32_t* first = (index & 1) ? R + leaf_words : R;   // odd: sibling || own
  const uint32_t* second = (index & 1) ? R : R + leaf_words;
  const uint32_t total = 2 * leaf_words;  // a multiple of 16 words (leaves are 32*ncols bytes)
  for (uint32_t w0 = 0; w0 < total; w0 += 16) {
    uint32_t m[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const uint32_t w = w0 + j;
      m[j] = w < leaf_words ? first[w] : second[w - leaf_words];
    }
    b2s_compress(h, m, 4u * (w0 + 16), w0 + 16 == total);
  }
  index >>= 1;
  for (uint32_t d = 0; d + 1 < depth; ++d, index >>= 1) {
    const uint32_t* sib = R + 2 * leaf_words + 8 * d;
    uint32_t m[16];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      m[j] = (index & 1) ? sib[j] : h[j];
      m[8 + j] = (index & 1) ? h[j] : sib[j];
    }
    b2s_init(h);
    b2s_compress(h, m, 64u, true);
  }
  uint32_t diff = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) diff |= h[j] ^ root[j];
  ok[r] = diff == 0;
}

// D consecutive levels in one launch: CTA b owns the subtree under node R = roots + b of the level
// with `roots` nodes, stages the subtree's 2^D already-computed descendants (nodes R*2^D ...) in
// shared memory and writes the D levels above them.  Used where a level is too small to fill the
// GPU (< 2^16 nodes): there a launch per level costs more than its compressions (FRI layers,
// upper halves of every tree).
__global__ void __launch_bounds__(64) merkle_mid_kernel(uint32_t* __restrict__ nodes, uint32_t roots, int D) {
  __shared__ uint4 sm[2 * 128];                       // up to 2^7 nodes of two uint4 each
  const uint64_t R = (uint64_t)roots + blockIdx.x;
  const uint32_t nin = 1u << D;
  const uint4* src = reinterpret_cast<const uint4*>(nodes + 8 * (R << D));
  for (uint32_t i = threadIdx.x; i < 2 * nin; i += blockDim.x) sm[i] = src[i];
  __syncthreads();
  for (int lv = 1; lv <= D; ++lv) {
    const uint32_t cnt = nin >> lv;                   // nodes of this level inside the subtree
    const uint32_t t = threadIdx.x;
    uint32_t h[8];
    if (t < cnt) {
      const uint4 a = sm[4 * t], b = sm[4 * t + 1], cc = sm[4 * t + 2], d = sm[4 * t + 3];
      uint32_t m[16] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, cc.x, cc.y, cc.z, cc.w, d.x, d.y, d.z, d.w};
      b2s_init(h);
      b2s_compress(h, m, 64u, true);
    }
    __syncthreads();                                  // every pair is read before any slot is reused
    if (t < cnt) {
      const uint4 lo4 = make_uint4(h[0], h[1], h[2], h[3]), hi4 = make_uint4(h[4], h[5], h[6], h[7]);
      sm[2 * t] = lo4;
      sm[2 * t + 1] = hi4;
      uint4* dst = reinterpret_cast<uint4*>(nodes + 8 * ((R << (D - lv)) + t));
      dst[0] = lo4;
      dst[1] = hi4;
    }
    __syncthreads();
  }
}

// Power-of-two trees: nodes [1, np/2) have node children; levels go bottom-up.  Levels of 2^16
// nodes and more get one launch each; below that one launch covers up to 7 levels in shared
// memory, and the last (at most 512-node) levels run inside one CTA.
int reduce_levels(stk_ctx* c, uint32_t* nodes, uint64_t np) {
  if (np < 4) return STK_OK;
  uint64_t lo = np >> 2;
  for (; lo >= 65536; lo >>= 1)
    merkle_level_kernel<<<(unsigned)((lo + 255) / 256), 256, 0, c->stream>>>(nodes, lo, lo);
  while (lo >= 1024) {                                // lo < 2^16: 2..7 levels at once, down to a 512-node level
    const int loglo = stk_ilog2(lo);
    const int D = loglo - 8 > 7 ? 7 : loglo - 8;      // levels lo, lo/2, ..., lo >> (D-1)
    const uint32_t roots = (uint32_t)(lo >> (D - 1));
    merkle_mid_kernel<<<roots, 64, 0, c->stream>>>(nodes, roots, D);
    lo = roots >> 1;
  }
  if (lo >= 1) merkle_top_kernel<<<1, 512, 0, c->stream>>>(nodes, (uint32_t)(2 * lo), np);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

}  // namespace

int stk_merkle_paths_dev(stk_ctx* c, const fe* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                         const uint8_t* d_nodes, const uint64_t* d_idx, uint64_t k, uint32_t* d_out, uint64_t rec_bytes) {
  if (!k) return STK_OK;
  const uint64_t np = 4 * (n / 4);
  if (np == 0 || (np & (np - 1))) return stk_fail(c, STK_EUNSUPPORTED, "branch extraction needs a power-of-two tree");
  merkle_paths_cols_kernel<<<(unsigned)k, 128, 0, c->stream>>>(d_cols, np, (uint32_t)ncols, col_stride,
                                                               (const uint32_t*)d_nodes, d_idx, d_out, rec_bytes / 4);
  STK_CUDA(c, cudaGetLastError());
  return STK_OK;
}

STK_API int stk_merkle_commit(stk_ctx* c, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                              uint8_t* d_nodes, uint8_t* h_root) {
  if (!c || !d_cols || !d_nodes || ncols == 0) return STK_EINVAL;
  const uint64_t np = 4 * (n / 4);
  if (np == 0) return stk_fail(c, STK_EINVAL, "fewer than 4 leaves: the reference's permute4 yields an empty tree");
  if (np & (np - 1)) {
    // heap levels of a non power-of-two tree mix leaf parents and node parents; the column
    // fast path keeps to the power-of-two sizes the prover produces
    return stk_fail(c, STK_EUNSUPPORTED, "column commit needs a power-of-two row count (use stk_merkle_commit_raw)");
  }
  STK_CUDA(c, cudaMemsetAsync(d_nodes, 0, 32, c->stream));
  const uint64_t half = np >> 1;
  merkle_leaf_pairs_cols_kernel<<<(unsigned)((half + 255) / 256), 256, 0, c->stream>>>(
      (const fe*)d_cols, np, (uint32_t)ncols, col_stride, (uint32_t*)d_nodes);
  STK_CUDA(c, cudaGetLastError());
  STK_TRY(reduce_levels(c, (uint32_t*)d_nodes, np));
  if (h_root) {
    STK_CUDA(c, cudaMemcpyAsync(h_root, d_nodes + 32, 32, cudaMemcpyDeviceToHost, c->stream));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return STK_OK;
}

STK_API int stk_merkle_commit_raw(stk_ctx* c, const uint8_t* d_leaves, uint64_t n, uint64_t leaf_len, uint8_t* d_nodes,
                                  uint8_t* h_root) {
  if (!c || !d_leaves || !d_nodes || leaf_len == 0) return STK_EINVAL;
  const uint64_t np = 4 * (n / 4);
  if (np == 0) return stk_fail(c, STK_EINVAL, "fewer than 4 leaves: the reference's permute4 yields an empty tree");
  STK_CUDA(c, cudaMemsetAsync(d_nodes, 0, 32, c->stream));
  // nodes whose children are leaves: i in [np/2, np)
  const uint64_t first = np >> 1, count = np - first;
  merkle_leaf_pairs_raw_kernel<<<(unsigned)((count + 127) / 128), 128, 0, c->stream>>>(d_leaves, np, leaf_len, first,
                                                                                       count, (uint32_t*)d_nodes);
  STK_CUDA(c, cudaGetLastError());
  // remaining nodes [1, np/2) by heap level, deepest first (any np, merkle_tree.py:54-55)
  uint64_t lo = 1;
  while (lo * 2 < first) lo *= 2;  // deepest level start: largest power of two < np/2 ... or == when pow2
  if (first > 1) {
    for (;; lo >>= 1) {
      uint64_t hi = std::min<uint64_t>(2 * lo, first);
      if (hi > lo) {
        uint64_t cnt = hi - lo;
        merkle_level_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>((uint32_t*)d_nodes, lo, cnt);
      }
      if (lo == 1) break;
    }
    STK_CUDA(c, cudaGetLastError());
  }
  if (h_root) {
    STK_CUDA(c, cudaMemcpyAsync(h_root, d_nodes + 32, 32, cudaMemcpyDeviceToHost, c->stream));
    STK_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return STK_OK;
}

STK_API int stk_merkle_paths(stk_ctx* c, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                             const uint8_t* d_nodes, const uint64_t* h_indices, uint64_t k, uint8_t* h_out,
                             uint64_t rec_bytes) {
  if (!c || !d_cols || !d_nodes || (!h_indices && k) || (!h_out && k)) return STK_EINVAL;
  if (!k) return STK_OK;
  const uint64_t np = 4 * (n / 4);
  if (np == 0 || (np & (np - 1))) return stk_fail(c, STK_EUNSUPPORTED, "branch extraction needs a power-of-two tree");
  const uint32_t depth = stk_ilog2(np);
  const uint64_t need = 2 * 32 * ncols + 32ull * (depth - 1);
  if (rec_bytes < need || (rec_bytes & 3)) return stk_fail(c, STK_EINVAL, "record size %llu < %llu", (unsigned long long)rec_bytes, (unsigned long long)need);
  for (uint64_t i = 0; i < k; ++i)
    if (h_indices[i] >= np) return stk_fail(c, STK_EINDEX, "branch index out of range");
  void* buf;
  STK_TRY(stk_scratch(c, kSlotStage, k * 8 + k * rec_bytes, &buf));
  uint64_t* d_idx = (uint64_t*)buf;
  uint32_t* d_out = (uint32_t*)((char*)buf + k * 8);
  STK_CUDA(c, cudaMemcpyAsync(d_idx, h_indices, k * 8, cudaMemcpyHostToDevice, c->stream));
  merkle_paths_cols_kernel<<<(unsigned)k, 128, 0, c->stream>>>((const fe*)d_cols, np, (uint32_t)ncols, col_stride,
                                                               (const uint32_t*)d_nodes, d_idx, d_out, rec_bytes / 4);
  STK_CUDA(c, cudaGetLastError());
  STK_CUDA(c, cudaMemcpyAsync(h_out, d_out, k * rec_bytes, cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}

// verify_branch (starks/merkle_tree.py:71-86) for k branches of ONE tree of n leaves (a power of
// two) whose leaves are leaf_len bytes (a multiple of 32): records as stk_merkle_paths returns
// them.  h_ok[r] = 1 when branch r hashes up to `root`.
STK_API int stk_verify_branches(stk_ctx* c, const uint8_t root[32], uint64_t n, uint64_t leaf_len,
                                const uint64_t* h_indices, uint64_t k, const uint8_t* h_records, uint64_t rec_bytes,
                                uint8_t* h_ok) {
  if (!c || !root || !h_indices || !h_records || !h_ok) return STK_EINVAL;
  if (!k) return STK_OK;
  if (n < 4 || (n & (n - 1))) return stk_fail(c, STK_EUNSUPPORTED, "branch verification needs a power-of-two tree");
  if (leaf_len == 0 || (leaf_len & 31)) return stk_fail(c, STK_EINVAL, "leaf length must be a multiple of 32 bytes");
  const uint32_t depth = stk_ilog2(n);
  if (rec_bytes != 2 * leaf_len + 32ull * (depth - 1)) return stk_fail(c, STK_EINVAL, "record size does not match the tree depth");
  for (uint64_t i = 0; i < k; ++i)
    if (h_indices[i] >= n) return stk_fail(c, STK_EINDEX, "branch index out of range");
  const uint64_t rb = k * rec_bytes, ib = k * 8;
  void* buf;
  STK_TRY(stk_scratch(c, kSlotStage, rb + ib + 32 + k + 64, &buf));
  uint8_t* base = (uint8_t*)buf;
  uint32_t* d_rec = (uint32_t*)base;
  uint64_t* d_idx = (uint64_t*)(base + ((rb + 7) & ~7ull));
  uint32_t* d_root = (uint32_t*)((uint8_t*)d_idx + ib);
  uint8_t* d_ok = (uint8_t*)d_root + 32;
  STK_CUDA(c, cudaMemcpyAsync(d_rec, h_records, rb, cudaMemcpyHostToDevice, c->stream));
  STK_CUDA(c, cudaMemcpyAsync(d_idx, h_indices, ib, cudaMemcpyHostToDevice, c->stream));
  STK_CUDA(c, cudaMemcpyAsync(d_root, root, 32, cudaMemcpyHostToDevice, c->stream));
  verify_branches_kernel<<<(unsigned)((k + 127) / 128), 128, 0, c->stream>>>(d_rec, rec_bytes / 4, d_idx, k, n,
                                                                            (uint32_t)(leaf_len / 4), depth, d_root, d_ok);
  STK_CUDA(c, cudaGetLastError());
  STK_CUDA(c, cudaMemcpyAsync(h_ok, d_ok, k, cudaMemcpyDeviceToHost, c->stream));
  STK_CUDA(c, cudaStreamSynchronize(c->stream));
  return STK_OK;
}
