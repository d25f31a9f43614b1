/*
 * starks_b200.h -- C ABI of libstarks_b200.so, the B200-native drop-in for the STARK
 * prover's data-parallel hot path of computablelabs/starks.
 *
 * The reference is pure Python and has no FFI; the boundary it offers is the module
 * surface of starks/fft.py, starks/merkle_tree.py and starks/fri.py as consumed by
 * starks/stark.py:4-17,31-35,225,254-276.  Each entry point below names the reference
 * function (file:line, relative to the upstream repository root) it replaces; the Python
 * shim in starks_b200/ (ctypes) rebinds those functions onto these symbols, see
 * INTEGRATION.md.
 *
 * Conventions
 *   - A field element is 8 little-endian uint32 limbs holding the canonical residue
 *     (IntegerModP.n, starks/modp.py:36).  The 32-byte big-endian form
 *     (IntegerModP.to_bytes, starks/modp.py:94-95) exists only inside hashed bytes.
 *   - Columns are contiguous arrays of elements; `*_stride` arguments are in elements.
 *   - Pointers named d_* are device pointers (cudaMalloc / torch.Tensor.data_ptr());
 *     pointers named h_* are host pointers (pinned memory makes the copies asynchronous).
 *   - Every call returns 0 on success or an STK_E* code; stk_last_error() gives the text.
 *   - Calls are asynchronous on the context's stream unless they return data to the host.
 *   - There is no CPU fallback: without a CUDA device stk_init fails.
 */
#ifndef STARKS_B200_H
#define STARKS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct stk_ctx stk_ctx;

enum {
  STK_OK = 0,
  STK_EINVAL = 1,      /* bad argument (maps to ValueError / TypeError)          */
  STK_ECUDA = 2,       /* CUDA runtime failure                                   */
  STK_EUNSUPPORTED = 3,/* size / modulus outside what the kernels implement      */
  STK_EINDEX = 4       /* input longer than the order of the root: the reference
                          raises IndexError there (starks/fft.py:303-314)        */
};

/* ---- context ------------------------------------------------------------------ */
int stk_version(void);
int stk_init(int device, stk_ctx** ctx);
void stk_destroy(stk_ctx* ctx);
const char* stk_last_error(stk_ctx* ctx);
/* Use an existing CUDA stream (e.g. torch.cuda.current_stream().cuda_stream); 0 = the
 * context's own stream.  Switching to a different stream first drains the old one (its work may
 * still read cached tables / scratch the new stream's calls are free to evict); setting the
 * stream already in use costs nothing. */
int stk_set_stream(stk_ctx* ctx, void* cuda_stream);
int stk_sync(stk_ctx* ctx);
/* Modulus of IntegersModP(p) (starks/modp.py:25-106).  p = 2^256 - 351*2^32 + 1 selects
 * the fast path; any other odd p < 2^256 runs 8-limb Montgomery. */
int stk_field_set(stk_ctx* ctx, const uint32_t p[8]);

/* ---- memory helpers (so a host language needs no CUDA binding of its own) -------- */
int stk_dev_alloc(stk_ctx* ctx, uint64_t bytes, void** d_ptr);
int stk_dev_free(stk_ctx* ctx, void* d_ptr);
int stk_host_alloc(stk_ctx* ctx, uint64_t bytes, void** h_ptr); /* pinned */
int stk_host_free(stk_ctx* ctx, void* h_ptr);
int stk_memcpy_h2d(stk_ctx* ctx, void* d_dst, const void* h_src, uint64_t bytes);
int stk_memcpy_d2h(stk_ctx* ctx, void* h_dst, const void* d_src, uint64_t bytes); /* synchronous */
int stk_memcpy_d2d(stk_ctx* ctx, void* d_dst, const void* d_src, uint64_t bytes);
int stk_memset(stk_ctx* ctx, void* d_dst, int value, uint64_t bytes);

/* ---- NTT ------------------------------------------------------------------------ */
/* fft_1d (starks/fft.py:316-331) for `batch` columns.  Column c reads n_in elements at
 * d_in + c*in_stride (zero padded up to n, :323-324; n_in > n -> STK_EINDEX) and writes n
 * elements at d_out + c*out_stride.  out[k] = sum_j in[j] * root^(jk); inverse uses
 * root^-1 and scales by n^-1 (:327-328).  n must be the multiplicative order of root:
 * powers of two >= 8 run the shared-memory radix-8 passes, anything else (n <= 4096, e.g.
 * the reference test's n = 6 over p = 31) the direct DFT kernel (_simple_ft, :287-300). */
int stk_ntt(stk_ctx* ctx, const uint32_t* d_in, uint64_t n_in, uint64_t in_stride, uint32_t* d_out,
            uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse);
/* _simple_ft (starks/fft.py:287-300) on its own: the direct O(n^2) DFT for any order n <= 4096
 * (powers of two included -- an independent cross-check of the fast path). */
int stk_dft_generic(stk_ctx* ctx, const uint32_t* d_in, uint64_t n_in, uint64_t in_stride, uint32_t* d_out,
                    uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse);
/* Same, host buffers; columns are streamed through the device in chunks with the copies
 * overlapping the transforms. */
int stk_ntt_host(stk_ctx* ctx, const uint32_t* h_in, uint64_t n_in, uint64_t in_stride, uint32_t* h_out,
                 uint64_t out_stride, uint64_t n, uint64_t batch, const uint32_t root[8], int inverse);
/* mul_polys (starks/fft.py:334-345): NTT(a) .* NTT(b) through the inverse-root transform
 * WITHOUT the 1/n scaling, exactly as the reference. */
int stk_mul_polys(stk_ctx* ctx, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                  uint32_t* d_out, uint64_t n, const uint32_t root[8]);
/* Polynomial.__mul__ (starks/polynomial.py:110-121): d_out[0 .. na+nb-1) = a * b (linear, not
 * cyclic; coefficients low -> high).  na == 0 or nb == 0 writes nothing.  d_out must not
 * overlap either input (STK_EINVAL).  Asynchronous.  Forward transforms, a pointwise product and
 * a scaled inverse where Z/p has a root of unity of the power-of-two order the product needs
 * (the STARK prime always; otherwise z^((p-1)/L) for a quadratic non-residue z); a direct
 * O(na*nb) kernel where it has none (e.g. p = 31).  Products longer than 2^30: STK_EUNSUPPORTED. */
int stk_poly_mul(stk_ctx* ctx, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                 uint32_t* d_out);
/* Polynomial.__divmod__ (starks/polynomial.py:128-143): a = b*q + r with deg r < deg b.
 * d_q receives max(na-nb+1, 0) coefficients; d_r receives nb-1 (zero-padded when na < nb-1).
 * nb >= 1 and b[nb-1] != 0, otherwise STK_EINVAL.  The call reads b's leading coefficient,
 * so it synchronises the stream.  Outputs must not overlap inputs or each other.  Newton
 * iteration on the reversed divisor (g <- g(2 - f g), doubling the precision), with products
 * routed as in stk_poly_mul. */
int stk_poly_divmod(stk_ctx* ctx, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                    uint32_t* d_q, uint32_t* d_r);
/* Polynomial.__call__ on a polynomial (starks/polynomial.py:158-164): d_out[0 .. (na-1)(nb-1)+1)
 * = a(b(X)).  na == 0 writes nothing; nb < 2 returns STK_EINVAL (a constant b is a scalar
 * evaluation).  d_out must not overlap either input (STK_EINVAL); an output longer than 2^30
 * returns STK_EUNSUPPORTED and writes nothing.  With nb == 2 the call reads b[0] and b[1], so it
 * synchronises the stream; b = alpha X (b[0] == 0, the prover's P(G1 X)) is then one pointwise
 * kernel, out[k] = a[k] alpha^k.  Any other b: divide and conquer over a padded to a power of two,
 * r_i <- r_2i + b^(2^j) r_2i+1 per level, each level one batched forward transform, a broadcast
 * pointwise product, one batched inverse and an add; levels without a root of the needed order
 * run through the products of stk_poly_mul (direct kernel).  Asynchronous for nb > 2. */
int stk_poly_compose(stk_ctx* ctx, const uint32_t* d_a, uint64_t na, const uint32_t* d_b, uint64_t nb,
                     uint32_t* d_out);
/* MultivariatePolynomial.__call__ on polynomials (starks/multivariate_polynomial.py:329-338):
 * argument k has h_lens[k] coefficients at d_polys + 8*k*in_stride (k < width <= 12, else
 * STK_EUNSUPPORTED).  Monomial m contributes coeffs[m] * prod_k X_k^exps[m*width+k] to output
 * h_mono_out[m] < nout (the list form of stk_constraint_eval with uint32 exponents).  An exponent
 * of 0 is a factor of 1 even on an empty argument; a positive one on an empty argument makes the
 * monomial vanish.  D = max over the remaining monomials of sum_k e_k (h_lens[k] - 1) (0 if none);
 * out_len must equal D + 1 (STK_EINVAL otherwise), D + 1 > 2^30 returns STK_EUNSUPPORTED.
 * Output j is written at d_out + 8*j*out_len, zero-padded; outputs must not overlap an argument.
 * Transform route (a root of order L = 2^ceil(log2(D+1)) exists): one batched forward transform of
 * the arguments, one pointwise kernel (every monomial by square-and-multiply), one batched scaled
 * inverse.  Otherwise the monomials are built from stk_poly_mul products.  Synchronises the stream
 * once to stage the monomial list. */
int stk_poly_eval_multivar(stk_ctx* ctx, const uint32_t* d_polys, const uint64_t* h_lens, uint64_t in_stride,
                           uint64_t width, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                           const uint32_t* h_mono_exps, uint64_t nmono, uint64_t nout, uint32_t* d_out,
                           uint64_t out_len);
/* Pointwise helpers on device columns: out[i] = a[i] (op) b[i]; op 0 add, 1 sub, 2 mul. */
int stk_vec_op(stk_ctx* ctx, int op, const uint32_t* d_a, const uint32_t* d_b, uint32_t* d_out, uint64_t n);
/* get_power_cycle (starks/utils.py:30-38): out[i] = r^i, i < n (n = order of r). */
int stk_power_cycle(stk_ctx* ctx, const uint32_t r[8], uint64_t n, uint32_t* d_out);

/* One large transform over G = nranks GPUs (four-step, one all-to-all; SURVEY.md App. C.4;
 * replaces a single fft_1d call, starks/fft.py:316-331, whose column does not fit or is
 * sharded).  Order N = nranks * local_n.  Input is cyclic (rank r holds x[r + G*m]).
 *   phase 0: in place, the butterfly levels that stay inside one residue class;
 *   caller:  all-to-all of equal contiguous chunks, then a local [r][m] -> [m][r] transpose;
 *   phase 1: the last log2(G) levels + bit-reversed store; rank r' ends with X[K] for
 *            K mod G = bitrev(r'), at local position K / G. */
int stk_ntt_dist_phase(stk_ctx* ctx, int phase, const uint32_t* d_in, uint32_t* d_out, uint64_t local_n,
                       uint64_t batch, uint64_t stride, const uint32_t root[8], uint64_t nranks, uint64_t rank,
                       int inverse);
/* Phase 0 FUSED with the exchange: the last pass of phase 0 stores each element straight into
 * the owning rank's buffer through peer pointers (peer_ptrs[r] = rank r's exchange buffer
 * mapped into this process; NVLink P2P stores, 256-byte runs), laid out [source rank][m].
 * After a cross-rank barrier, stk_ntt_dist_phase(phase = 2, ...) runs phase 1 directly on
 * that layout: no all-to-all and no transpose pass. */
int stk_ntt_dist_phase0_p2p(stk_ctx* ctx, uint32_t* d_inout, uint64_t local_n, const uint32_t root[8],
                            uint64_t nranks, uint64_t rank, int inverse, const uint64_t* peer_ptrs);

/* ---- LDE ------------------------------------------------------------------------ */
/* construct_trace_polynomials + evaluation loop (starks/stark.py:27-36, 254-256): per column
 * inverse NTT of `steps` trace values over <G1>, G1 = g2^ext, then forward NTT of the
 * coefficients over <g2> (order steps*ext).  d_coeffs may be NULL (scratch is used), or equal
 * to d_trace with coeff_stride == trace_stride: the coefficients then replace the trace (with
 * ext = 8 the evaluations are computed in full instead of copying residue 0 from the trace).
 * Any other overlap of the coefficient rows with the trace rows returns STK_EINVAL. */
int stk_lde(stk_ctx* ctx, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
            uint64_t cols, const uint32_t g2[8], uint32_t* d_coeffs, uint64_t coeff_stride, uint32_t* d_evals,
            uint64_t eval_stride);
/* stk_lde followed by stk_merkle_commit over the extended columns (stark.py:254-257). */
int stk_lde_commit(stk_ctx* ctx, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                   uint64_t cols, const uint32_t g2[8], uint32_t* d_evals, uint64_t eval_stride, uint8_t* d_nodes,
                   uint8_t* h_root);

/* stk_lde_commit with the trace in HOST memory (pinned, stk_host_alloc): column groups are uploaded
 * on a copy stream while the previous group is transformed, so only the first group's copy is
 * exposed.  The end-to-end form of "LDE + Merkle commit": trace on the host -> root on the host. */
int stk_lde_commit_host(stk_ctx* ctx, const uint32_t* h_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                        uint64_t cols, const uint32_t g2[8], uint32_t* d_evals, uint64_t eval_stride,
                        uint8_t* d_nodes, uint8_t* h_root);

/* stk_lde for a column shard with the commit's exchange fused in: the final pass of the forward
 * transform stores every evaluation row straight into the rank that owns the row's leaf range
 * (peer_ptrs[r] = rank r's (cols_total x N/nranks) row buffer mapped into this process; rows
 * arrive in the order of a local tree under permute4, merkle_tree.py:11-23).  After a
 * cross-rank barrier each rank runs stk_merkle_commit on its buffer (global node nranks + r). */
int stk_lde_p2p(stk_ctx* ctx, const uint32_t* d_trace, uint64_t steps, uint64_t trace_stride, uint64_t ext,
                uint64_t cols, const uint32_t g2[8], uint64_t nranks, uint64_t col_base, const uint64_t* peer_ptrs);
/* Forward transform of `cols` COEFFICIENT rows (n_in coefficients, zero-padded to n) with the same
 * fused row scatter: the sharded prover's evaluation of its slice of P, D, B (starks/stark.py:247,
 * 254-256).  cols = 0 is a no-op. */
int stk_ntt_p2p(stk_ctx* ctx, const uint32_t* d_coeffs, uint64_t n_in, uint64_t in_stride, uint64_t n,
                uint64_t cols, const uint32_t root[8], uint64_t nranks, uint64_t col_base,
                const uint64_t* peer_ptrs);

/* ---- Merkle ---------------------------------------------------------------------- */
/* merkelize_polynomial_evaluations + merkelize (starks/merkle_tree.py:36-56, 94-119) over
 * `ncols` device columns of n rows (n a power of two >= 4): leaf(row) = concatenation of the
 * columns' 32-byte big-endian values, leaves in permute4 order (:11-23), unhashed; node i =
 * BLAKE2s(node 2i || node 2i+1).  d_nodes receives 32*n bytes (node i at byte 32*i, i in
 * [1, n); entry 0 zero).  h_root (optional) receives node 1.  One column gives
 * merkelize(values). */
int stk_merkle_commit(stk_ctx* ctx, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                      uint8_t* d_nodes, uint8_t* h_root);
/* merkelize (merkle_tree.py:36-56) over n raw leaves of leaf_len bytes in ORIGINAL order;
 * any n >= 4 (the heap formula is applied as is, e.g. n = 144 in test_merkle_tree.py:32-38;
 * n mod 4 trailing leaves are dropped exactly as permute4 does). */
int stk_merkle_commit_raw(stk_ctx* ctx, const uint8_t* d_leaves, uint64_t n, uint64_t leaf_len, uint8_t* d_nodes,
                          uint8_t* h_root);
/* mk_branch (merkle_tree.py:59-68) for k original indices of a column tree.  Record per
 * query (rec_bytes each, host memory): leaf (32*ncols) | sibling leaf (32*ncols) | sibling
 * nodes bottom-up (32 bytes each, log2(n)-1 of them). */
int stk_merkle_paths(stk_ctx* ctx, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                     const uint8_t* d_nodes, const uint64_t* h_indices, uint64_t k, uint8_t* h_out,
                     uint64_t rec_bytes);
/* verify_branch (starks/merkle_tree.py:71-86) for k branches of ONE tree of n leaves (a power
 * of two, leaves of leaf_len bytes, a multiple of 32): h_records holds k stk_merkle_paths
 * records (leaf | sibling leaf | sibling nodes), h_ok[r] = 1 when branch r hashes up to root. */
int stk_verify_branches(stk_ctx* ctx, const uint8_t root[32], uint64_t n, uint64_t leaf_len,
                        const uint64_t* h_indices, uint64_t k, const uint8_t* h_records, uint64_t rec_bytes,
                        uint8_t* h_ok);

/* ---- FRI ------------------------------------------------------------------------- */
/* The `column` of one FRI layer (starks/fri.py:236-242; multi_interp_4,
 * starks/poly_utils.py:412-440): out[i], i < n/4, is the degree<4 interpolant through
 * (root^(i+jn/4), vals[i+jn/4]), j<4, evaluated at special_x (any 256-bit integer; the
 * reference does not reduce it, fri.py:229). */
int stk_fri_fold4(stk_ctx* ctx, const uint32_t* d_vals, uint64_t n, const uint32_t root[8],
                  const uint32_t special_x[8], uint32_t* d_out);
/* get_pseudorandom_indices (starks/utils.py:60-90) as the FRI driver derives them (host BLAKE2s
 * chain over the 32-byte entropy, 4-byte big-endian words).  Host only: ctx may be NULL. */
/* The same fold for a layer sharded by leaf range (one proof over several GPUs, SURVEY.md 8e):
 * d_rows = the four runs {j*n/4 + i0 + t : t < q_run}, j < 4, back to back; d_out receives
 * column[i0 .. i0 + q_run). */
int stk_fri_fold4_rows(stk_ctx* ctx, const uint32_t* d_rows, uint64_t n, const uint32_t root[8],
                       const uint32_t special_x[8], uint64_t q_run, uint64_t i0, uint32_t* d_out);
int stk_pseudorandom_indices(stk_ctx* ctx, const uint8_t entropy[32], uint64_t modulus, uint64_t count,
                             uint64_t exclude_multiples_of, uint64_t* h_out);
/* The whole commit phase of SmoothSubgroupFRI.generate_proximity_proof (starks/fri.py:189-266)
 * for evaluations already on the device: per layer fold, column tree, Fiat-Shamir indices
 * (starks/utils.py:60-90) and branch gathers, one host synchronisation per layer.  d_nodes0 /
 * h_root0: the tree over d_vals0 if the caller has built it (both NULL: built here).
 * h_out receives, per fold layer: root2 (32 B) | k column-tree records (branch of y) | 4k
 * records of the layer's own tree (y, y+q, y+2q, y+3q per y); then the last layer's values
 * as 32-byte big-endian words.  k = security for the first layer, 40 below it (fri.py:262-266).
 * Records are stk_merkle_paths records.  *out_len = bytes needed / written; n0 a power of two. */
int stk_fri_prove(stk_ctx* ctx, const uint32_t* d_vals0, uint64_t n0, const uint8_t* d_nodes0,
                  const uint8_t* h_root0, const uint32_t root[8], uint64_t maxdeg_plus_1,
                  uint64_t exclude_multiples_of, uint64_t security, uint8_t* h_out, uint64_t out_cap,
                  uint64_t* out_len);

/* ---- prover constructions between the commitments (starks/stark.py:38-177) ---------- */
/* construct_constraint_polynomials in evaluation form (stark.py:38-55):
 * cev[j][i] = pev[j][(i+ext) mod n] - step_j(pev[0][i], ..., pev[width-1][i]).  The step
 * polynomials arrive as a monomial list (the reference's MultiVarPoly is a dict
 * monomial -> coefficient, starks/multivariate_polynomial.py): monomial m contributes
 * coeffs[m] * prod_k X_{k+1}^exps[width*m+k] to constraint out[m].  width <= 12. */
int stk_constraint_eval(stk_ctx* ctx, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                        uint64_t col_stride, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                        const uint8_t* h_mono_exps, uint64_t nmono, uint32_t* d_cev, uint64_t out_stride);
/* construct_remainder_polynomials (stark.py:57-78) in EVALUATION form on the size-n domain <g2>:
 * d_dev[j][i] = D_j(g2^i).  Where Z(x_i) != 0 (i != 0 mod ext) it is pointwise,
 * D = C * (x - last) / (x^steps - 1) with x_i^steps one of ext constants; at i = 0 mod ext
 * (both C and Z vanish) it is read from d_dsub = D_j on a subgroup of order sub_n containing
 * <g2^ext> (the forward transform of D's coefficients, stk_quotient_z).  Saves 7/8 of D's
 * size-n transform.  ext in 2..16; monomial list as stk_constraint_eval. */
int stk_quotient_eval(stk_ctx* ctx, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                      uint64_t col_stride, const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs,
                      const uint8_t* h_mono_exps, uint64_t nmono, const uint32_t g2[8], const uint32_t last[8],
                      const uint32_t* d_dsub, uint64_t sub_n, uint64_t dsub_stride, uint32_t* d_dev,
                      uint64_t out_stride);
/* construct_boundary_polynomials (stark.py:80-104) in EVALUATION form on the size-n domain <g2>
 * (STARK prime): d_bev[j][i] = (P_j(x_i) - (i0_j + i1_j*x_i)) / ((x_i - 1)(x_i - last)),
 * last = g2^last_index (a non-zero multiple of ext), pointwise wherever the denominator is
 * non-zero -- 1/(x_i - g2^e) = g2^-e * T[(i - e) mod n] with one cached table
 * T[i] = (g2^i - 1)^-1 -- and from d_bsub (B_j on <g2^ext>, n/ext values per column) at
 * i = 0 mod ext.  h_interp: width x {i0, i1} (8 limbs each).  Saves 7/8 of B's size-n transform. */
int stk_boundary_eval(stk_ctx* ctx, const uint32_t* d_pev, uint64_t n, uint64_t ext, uint64_t width,
                      uint64_t col_stride, const uint32_t g2[8], uint64_t last_index, const uint32_t* h_interp,
                      const uint32_t* d_bsub, uint64_t bsub_stride, uint32_t* d_bev, uint64_t out_stride);
/* construct_remainder_polynomials (stark.py:57-78) on coefficient vectors of length n:
 * D = C / Z with Z = (X^steps - 1)/(X - last), computed as C*(X-last) / (X^steps - 1).
 * *h_bad = number of non-zero remainder coefficients (the reference asserts divisibility). */
int stk_quotient_z(stk_ctx* ctx, const uint32_t* d_ccoef, uint64_t n, uint64_t steps, const uint32_t last[8],
                   uint32_t* d_dcoef, uint32_t* h_bad);
/* Quotient of a polynomial (n coefficients, low -> high) by (X - r), as Polynomial.__divmod__
 * (starks/polynomial.py:128-143) yields it: out[k] = sum_{i>k} a[i] r^(i-k-1), k < n-1.
 * r = 1, or r of multiplicative order r_order >= n (its power tables are cached). */
int stk_div_linear(stk_ctx* ctx, const uint32_t* d_a, uint64_t n, const uint32_t r[8], uint64_t r_order,
                   uint32_t* d_out);
/* compute_pseudorandom_linear_combination (stark.py:130-177) in evaluation form:
 * out[i] = sum_c weights[c] * cols[c][i]. */
int stk_lincomb(stk_ctx* ctx, const uint32_t* d_cols, uint64_t n, uint64_t ncols, uint64_t col_stride,
                const uint32_t* h_weights, uint32_t* d_out);
/* get_computational_trace (starks/air.py:31-52) with the witness transposition of
 * AIR.generate_witness (:124): h_witness[dim][step] (width x steps elements, host memory --
 * ideally from stk_host_alloc), state[0] = h_inp, state[i+1][j] = step_poly_j(state[i]).  Step
 * polynomials as the monomial list of stk_constraint_eval.  Sequential recurrence: runs on the
 * calling host thread. */
int stk_trace_generate(stk_ctx* ctx, const uint32_t* h_inp, uint64_t steps, uint64_t width,
                       const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs, const uint8_t* h_mono_exps,
                       uint64_t nmono, uint32_t* h_witness);

/* The same trace generated ON THE DEVICE (trace.cu): d_witness[(t*width + dim)*stride + step]
 * for `ntraces` independent traces with inputs h_inp[t][dim].  Parallel over traces (one thread
 * each) and, for AIRs whose step polynomials have degree <= 1, over chunks of one trace: the
 * chunk-start states come from powers of the (width+1)^2 companion matrix (a prefix over A^L on
 * the host, ~(width+1)^2 multiplies per chunk), every chunk's links run in their own thread.
 * Asynchronous on the context's stream. */
int stk_trace_generate_dev(stk_ctx* ctx, const uint32_t* h_inp, uint64_t ntraces, uint64_t steps, uint64_t width,
                           const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs, const uint8_t* h_mono_exps,
                           uint64_t nmono, uint32_t* d_witness, uint64_t stride);
/* stk_trace_generate into h_witness (pinned) with every finished block of 2^15 steps copied to
 * d_witness[dim*stride + step] while the next block is computed (upload hidden behind the
 * recurrence).  Returns with the copies enqueued. */
int stk_trace_generate_upload(stk_ctx* ctx, const uint32_t* h_inp, uint64_t steps, uint64_t width,
                              const uint32_t* h_mono_out, const uint32_t* h_mono_coeffs, const uint8_t* h_mono_exps,
                              uint64_t nmono, uint32_t* h_witness, uint32_t* d_witness, uint64_t stride);
/* *h_bad = number of elements of d_vals[0..n) that are not canonical residues (>= p): the kernels
 * assume canonical operands (IntegerModP.__init__ reduces, starks/modp.py:35-36).  sync != 0:
 * returns with *h_bad written; sync == 0: h_bad must be pinned host memory (stk_host_alloc) and
 * holds the count once the context's stream has been synchronised. */
int stk_count_noncanonical(stk_ctx* ctx, const uint32_t* d_vals, uint64_t n, uint32_t* h_bad, int sync);

/* ---- K0: integer-pipe microbenchmarks (roofline denominators) ---------------------- */
/* which: 0 IMAD, 1 IMAD.WIDE, 2 IADD3, 3 IMAD.HI, 4 IADD3+LOP3+SHF (BLAKE2s mix),
 * 5 field multiply, 6 NTT butterfly, 7 IMAD+IADD3, 8 IMAD.WIDE+IADD3, 9 carry-chain adds,
 * 10 IMAD.WIDE.X carry rows.  Returns elapsed milliseconds and the number of
 * operations (of the kind named) executed. */
int stk_microbench(stk_ctx* ctx, int which, uint64_t iters, float* ms, double* ops);
/* A/B of the experimental multiply (csrc/field_exp.cuh) in registers: which = 5 | 6 as above,
 * variant 0 = production, bit 0 = accumulators without zero-initialisation, bit 1 = aligned
 * 351*H rows.  *mismatches counts outputs that differ from the production kernel's (must be 0). */
int stk_microbench_variant(stk_ctx* ctx, int variant, int which, uint64_t iters, float* ms, double* ops,
                           uint64_t* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* STARKS_B200_H */
