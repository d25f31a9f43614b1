// lde.cu -- low-degree extension of trace columns and the LDE -> Merkle commit pipeline.
// Replaces construct_trace_polynomials (starks/stark.py:27-36: inverse NTT of each witness
// column over <G1>) followed by the evaluation loop of mk_proof (starks/stark.py:254-256:
// forward NTT over <G2>, G1 = G2^ext) and merkelize_polynomial_evaluations (:257).  There is
// no coset shift in the reference: the evaluation domain is the subgroup <G2> itself, so
// evals[i*ext] == trace[i].
#include <algorithm>
#include <vector>
#include "ctx.h"

using namespace stk;

// Coefficients (optional output, cols x steps) and evaluations (cols x steps*ext).
STK_API int stk_lde(stk_ctx* c, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                    uint64_t cols, const uint32_t g2[8], uint32_t* d_coeffs, uint64_t coeff_stride, uint32_t* d_evals,
                    uint64_t eval_stride) {
  if (!c || !d_trace || !d_evals || !g2 || steps == 0 || ext == 0 || cols == 0) return STK_EINVAL;
  const uint64_t n = steps * ext;
  // The coefficients may replace the trace in its own buffer (same start and stride: the inverse
  // transform runs in place); any other overlap would overwrite trace values still to be read.
  const bool in_place = (const void*)d_coeffs == (const void*)d_trace && coeff_stride == trace_stride;
  if (d_coeffs && !in_place) {
    const uint64_t t0 = (uint64_t)d_trace, t1 = t0 + ((cols - 1) * trace_stride + steps) * sizeof(fe);
    const uint64_t c0 = (uint64_t)d_coeffs, c1 = c0 + ((cols - 1) * coeff_stride + steps) * sizeof(fe);
    if (c0 < t1 && t0 < c1) return stk_fail(c, STK_EINVAL, "coefficient rows overlap the trace rows");
  }
  fe G2 = stk_load_fe(g2);
  fe G1 = stk_h_pow(c, G2, ext);
  fe* coef = (fe*)d_coeffs;
  if (!coef) {
    void* t;
    STK_TRY(stk_scratch(c, kSlotLdeCoeffs, cols * steps * sizeof(fe), &t));
    coef = (fe*)t;
    coeff_stride = steps;
  }
  STK_TRY(stk_ntt_dev(c, (const fe*)d_trace, steps, trace_stride, coef, coeff_stride, steps, cols, G1, 1, 1));
  // ext = 8: evals[8K] = trace[K] (the evaluation domain contains the trace domain unshifted), so
  // the residue-0 coset of the forward transform is copied instead of computed -- unless the
  // coefficients have just overwritten the trace
  if (ext == 8 && c->is_stark && !in_place && (const void*)d_trace != (const void*)d_evals)
    return stk_ntt_dev_r0(c, coef, steps, coeff_stride, (fe*)d_evals, eval_stride, n, cols, G2, (const fe*)d_trace,
                          trace_stride);
  STK_TRY(stk_ntt_dev(c, coef, steps, coeff_stride, (fe*)d_evals, eval_stride, n, cols, G2, 0, 0));
  return STK_OK;
}

STK_API int stk_lde_commit(stk_ctx* c, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                           uint64_t cols, const uint32_t g2[8], uint32_t* d_evals, uint64_t eval_stride,
                           uint8_t* d_nodes, uint8_t* h_root) {
  if (!c || !d_trace || !d_evals || !d_nodes || !g2 || steps == 0 || ext == 0 || cols == 0) return STK_EINVAL;
  STK_TRY(stk_lde(c, d_trace, steps, trace_stride, ext, cols, g2, nullptr, 0, d_evals, eval_stride));
  return stk_merkle_commit(c, d_evals, steps * ext, cols, eval_stride, d_nodes, h_root);
}

// stk_lde whose final NTT pass stores every evaluation row directly into the rank that owns
// the row's Merkle leaf (P2P stores over NVLink; see ntt.cuh, peer_on = 2): the column-sharded
// LDE and the column->leaf-range exchange of the sharded commit in one kernel.  peer_ptrs[r] is
// rank r's (cols_total x N/nranks) row buffer mapped into this process.
STK_API int stk_lde_p2p(stk_ctx* c, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                        uint64_t cols, const uint32_t g2[8], uint64_t nranks, uint64_t col_base,
                        const uint64_t* peer_ptrs) {
  if (!c || !d_trace || !g2 || !peer_ptrs || steps == 0 || ext == 0 || cols == 0) return STK_EINVAL;
  if (nranks < 2 || nranks > 8 || (nranks & (nranks - 1))) return stk_fail(c, STK_EINVAL, "2, 4 or 8 ranks");
  const uint64_t n = steps * ext;
  if (n & (n - 1)) return stk_fail(c, STK_EINVAL, "steps*ext must be a power of two");
  fe G2 = stk_load_fe(g2);
  fe G1 = stk_h_pow(c, G2, ext);
  void* t;
  STK_TRY(stk_scratch(c, kSlotLdeCoeffs, cols * steps * sizeof(fe), &t));
  fe* coef = (fe*)t;
  STK_TRY(stk_ntt_dev(c, (const fe*)d_trace, steps, trace_stride, coef, steps, steps, cols, G1, 1, 1));
  return stk_ntt_dev_peer(c, coef, steps, steps, n, cols, G2, nranks, col_base, peer_ptrs);
}

// Forward transform of COEFFICIENT rows (n_in coefficients each, implicitly zero-padded to n)
// whose final pass scatters every evaluation row to its leaf owner, like stk_lde_p2p: the
// sharded prover hands each rank a slice of the 3w coefficient vectors P_1..P_w, D_1..D_w,
// B_1..B_w (starks/stark.py:247, 254-256).  cols may be 0 (a rank without columns still takes
// part in the barriers and hashes its leaf range).
STK_API int stk_ntt_p2p(stk_ctx* c, const uint32_t* d_coeffs, uint64_t n_in, uint64_t in_stride, uint64_t n,
                        uint64_t cols, const uint32_t root[8], uint64_t nranks, uint64_t col_base,
                        const uint64_t* peer_ptrs) {
  if (!c || !root || !peer_ptrs || n == 0) return STK_EINVAL;
  if (cols == 0) return STK_OK;
  if (!d_coeffs) return STK_EINVAL;
  if (nranks < 2 || nranks > 8 || (nranks & (nranks - 1))) return stk_fail(c, STK_EINVAL, "2, 4 or 8 ranks");
  if (n & (n - 1)) return stk_fail(c, STK_EINVAL, "the transform length must be a power of two");
  return stk_ntt_dev_peer(c, (const fe*)d_coeffs, n_in, in_stride, n, cols, stk_load_fe(root), nranks, col_base,
                          peer_ptrs);
}

// stk_lde_commit with the trace in HOST memory (pinned: stk_host_alloc) -- the end-to-end form of
// BASELINE's "LDE + Merkle-commit" metric (trace on the host -> root on the host).  Columns are
// independent until the leaves are hashed, so the upload is pipelined with the transforms: column
// groups stream through two staging slots on a copy stream while the previous group's inverse
// and forward transforms run on the compute stream; only the first group's copy is exposed.
STK_API int stk_lde_commit_host(stk_ctx* c, const uint32_t* h_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                                uint64_t cols, const uint32_t g2[8], uint32_t* d_evals, uint64_t eval_stride,
                                uint8_t* d_nodes, uint8_t* h_root) {
  if (!c || !h_trace || !d_evals || !d_nodes || !g2 || steps == 0 || ext == 0 || cols == 0 || trace_stride < steps)
    return STK_EINVAL;
  const uint64_t n = steps * ext;
  const uint64_t col_bytes = steps * sizeof(fe);
  // Group sizes grow geometrically (x1.5): only the FIRST group's copy is exposed, so it is small
  // (~16 MiB), and a column uploads faster than it transforms (PCIe ~50 GB/s against ~0.28 ms per
  // 2^18-step column), so a group up to 1.7x the previous one still arrives in time; larger
  // groups keep the per-launch overheads of the transforms down.  Capped at 128 MiB per slot.
  const uint64_t first = std::max<uint64_t>(1, ((uint64_t)16 << 20) / col_bytes);
  const uint64_t cap = std::max<uint64_t>(first, ((uint64_t)128 << 20) / col_bytes);
  std::vector<uint64_t> groups;
  for (uint64_t done = 0, g = first; done < cols; g = std::min(cap, g + (g + 1) / 2)) {
    const uint64_t nb = std::min(g, cols - done);
    groups.push_back(nb);
    done += nb;
  }
  const uint64_t slot_cols = std::min(cap, cols);
  void* st;
  STK_TRY(stk_scratch(c, kSlotLdeHost, 2 * slot_cols * col_bytes, &st));
  fe* slot[2] = {(fe*)st, (fe*)st + slot_cols * steps};
  cudaStream_t cp = c->copy_streams[0];
  // the staging slots may still be read by transforms of an earlier call on the compute stream
  STK_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  STK_CUDA(c, cudaStreamWaitEvent(cp, c->ev[0], 0));
  uint64_t b0 = 0;
  for (size_t gi = 0; gi < groups.size(); ++gi) {
    const int k = (int)(gi & 1);
    const uint64_t nb = groups[gi];
    cudaEvent_t up = c->ev[1 + k], done = c->ev[3 + k];
    if (gi >= 2) STK_CUDA(c, cudaStreamWaitEvent(cp, done, 0));   // slot k's previous group is transformed
    if (trace_stride == steps)
      STK_CUDA(c, cudaMemcpyAsync(slot[k], h_trace + b0 * trace_stride * 8, nb * col_bytes, cudaMemcpyHostToDevice, cp));
    else
      STK_CUDA(c, cudaMemcpy2DAsync(slot[k], col_bytes, h_trace + b0 * trace_stride * 8, trace_stride * sizeof(fe),
                                    col_bytes, nb, cudaMemcpyHostToDevice, cp));
    STK_CUDA(c, cudaEventRecord(up, cp));
    STK_CUDA(c, cudaStreamWaitEvent(c->stream, up, 0));
    STK_TRY(stk_lde(c, (const uint32_t*)slot[k], steps, steps, ext, nb, g2, nullptr, 0,
                    d_evals + b0 * eval_stride * 8, eval_stride));
    STK_CUDA(c, cudaEventRecord(done, c->stream));
    b0 += nb;
  }
  return stk_merkle_commit(c, d_evals, n, cols, eval_stride, d_nodes, h_root);
}
