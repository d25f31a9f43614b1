"""Drop-in for the prover/verifier driver of starks/stark.py: STARK(field, steps,
extension_factor, width, step_polys).mk_proof(witness, boundary) / .verify_proof(proof,
witness, boundary), get_pseudorandom_ks and the construct_* helpers' results.

mk_proof keeps every column on the device from the witness upload to the last FRI layer:
LDE (stk_lde), constraint evaluations (stk_constraint_eval), quotients (stk_quotient_z,
stk_div_linear), Merkle commitments (stk_merkle_commit), linear combination (stk_lincomb),
branch gathers (stk_merkle_paths) and FRI folds (stk_fri_fold4).  Only 32-byte roots, the
Fiat-Shamir scalars and the opened branches cross to the host.  The proof object
[m_root, l_root, branches, fri_proof] (stark.py:270-277) is bit-identical to the reference's.
verify_proof is host-side glue (80 positions + FRI checks) mirroring stark.py:281-372."""
import ctypes
import os
import time
from hashlib import blake2s

import numpy as np

from .air import _monomial_arrays
from .engine import P_STARK, DevBuf, _u32, default_engine
from .fri import FRI, DeviceLayer
from .limbs import int_to_limbs, ints_to_limbs, limbs_to_ints
from .merkle_tree import unpack_merkle_leaf, verify_branch
from .modp import element_to_int
from .polynomial import monomials_of
from .utils import get_pseudorandom_indices

blake = lambda x: blake2s(x).digest()
E = 32                                    # bytes per field element on the device


def get_pseudorandom_ks(m_root: bytes, num: int):
  """starks/stark.py:106-126: k_i = BLAKE2s(m_root | salt_i) as integers.  The salts are ASCII
  strings: b'0x01'.. for num <= 4, b'0x00'.. (a different numbering) for 5 <= num < 10, and the
  reference returns None for ten or more (SURVEY.md A.15)."""
  if num < 0 or num >= 10:
    return None
  first = 1 if num <= 4 else 0
  return [int.from_bytes(blake(m_root + b"0x0%d" % (first + i)), "big") for i in range(num)]


def lincomb_weights(m_root, width, steps, precision, G2, p):
  """compute_pseudorandom_linear_combination (:130-177) in evaluation form: the weights of l over
  the 3w committed rows P_1..P_w, D_1..D_w, B_1..B_w, in that order."""
  k1, k2, k3, k4 = get_pseudorandom_ks(m_root, 4)
  l_ks = get_pseudorandom_ks(m_root, width)
  c = pow(pow(G2, steps, p), precision - 1, p)     # powers[i] with the leaked i = precision-1 (:153-160)
  wP, wD, wB = [], [], []
  for j in range(width):
    aj = (1 + l_ks[j] * c) % p
    wD.append(aj)
    wP.append(aj * ((k1 + k2 * c) % p) % p)
    wB.append(aj * ((k3 + k4 * c) % p) % p)
  return wP + wD + wB


def interleave_branches(mb, lb):
  """compute_merkle_spot_checks' order (:390-402): for each position, the m-tree branches at pos and
  pos + ext (mb[2i], mb[2i+1]), then the l-tree branch at pos (lb[i])."""
  return [b for i in range(len(lb)) for b in (mb[2 * i], mb[2 * i + 1], lb[i])]


def raise_if_noncanonical(check):
  """check: None or a pending Engine.count_noncanonical of the witness, read once the stream has
  been synchronised."""
  if check is not None and check():
    raise ValueError("witness holds elements >= p; reduce them mod p first")


def _interp2(p, x0, x1, y0, y1):
  """lagrange_interp_2 (starks/poly_utils.py:397-410) -> coefficients [i0, i1]."""
  eq0, eq1 = [(-x1) % p, 1], [(-x0) % p, 1]
  e0, e1 = (eq0[0] + x0) % p, (eq1[0] + x1) % p
  invall = pow(e0 * e1 % p, -1, p)
  inv_y0 = y0 * invall % p * e1 % p
  inv_y1 = y1 * invall % p * e0 % p
  return [(eq0[i] * inv_y0 + eq1[i] * inv_y1) % p for i in range(2)]


class STARK(object):
  """Generates and verifies STARKs (starks/stark.py:179-402)."""

  def __init__(self, field, steps, extension_factor, width, step_polys, spot_check_security_factor=80,
               engine=None):
    self.field = field
    self.width = width
    self.steps = steps
    self.step_polys = step_polys
    self.extension_factor = extension_factor
    self.precision = steps * extension_factor
    self.spot_check_security_factor = spot_check_security_factor
    self._engine = engine
    p = self.field.p
    self.G2 = field(7)**((p - 1) // self.precision)                      # :217
    self.G1 = self.G2**extension_factor                                  # :220
    self.last_step_position = self.G2**((steps - 1) * extension_factor)  # xs[(steps-1)*ext], :223-224
    self._monomials = [monomials_of(sp, width, p) for sp in step_polys]
    self._mono_arrays = _monomial_arrays(step_polys, width, p)   # the constraint kernels' form of them
    # The constraint subgroup <G_M>, G_M = G2^(N/M): deg C <= d*(steps-1) < M = steps*2^ceil(log2 d),
    # so C (and D = C/Z) are recovered exactly from M evaluations.
    mult = 1
    while mult < max(self.get_degree(), 1):
      mult *= 2
    self.M = min(self.precision, steps * mult)
    self.GM = pow(int(self.G2), self.precision // self.M, p)
    self.timings = {}

  @property
  def xs(self):
    from .utils import get_power_cycle
    return get_power_cycle(self.G2, self.field, engine=self._engine)

  def get_degree(self):
    return max(max([sum(k) for k, _ in m] or [0]) for m in self._monomials)  # :230-231

  # ----------------------------------------------------------------- prover
  def _witness(self, eng, witness):
    """The witness on the device, from any of its three forms: a list of w columns of field
    elements (reduced mod p like IntegerModP.__init__, modp.py:35-36), (w, steps, 8) uint32 limbs,
    or a DevBuf holding those (air.witness_device / stk_trace_generate_dev).
    Returns (d_trace, owned, noncanonical): the caller frees d_trace when it owns it.  Limbs are used
    as they are, but the kernels' add/sub/reduce assume canonical residues: for both limb forms
    noncanonical is a pending count of the elements >= p, for raise_if_noncanonical; None for a list."""
    p, w, steps = self.field.p, self.width, self.steps
    listed = not isinstance(witness, (DevBuf, np.ndarray))
    if isinstance(witness, DevBuf):
      assert witness.nbytes >= w * steps * E
      d_trace, owned = witness, False
    else:
      if listed:
        assert len(witness) == w
        limbs = np.stack([ints_to_limbs([element_to_int(v) % p for v in col]) for col in witness])
      else:
        limbs = np.ascontiguousarray(witness, dtype=np.uint32)
      assert limbs.shape == (w, steps, 8)
      # no wait: a caller's pinned array copies while the host enqueues; a pageable one has been
      # staged by the time the call returns
      d_trace, owned = eng.alloc(w * steps * E).upload(limbs, wait=False), True
    return d_trace, owned, None if listed else eng.count_noncanonical(d_trace.ptr, w * steps, wait=False)

  def _last_row(self, witness):
    """The witness's last row (the boundary outputs) as ints, from any form _witness takes.  For a
    DevBuf the copies wait for the stream."""
    if isinstance(witness, DevBuf):
      s = self.steps
      return limbs_to_ints(np.stack([witness.download((1, 8), byte_offset=(j * s + s - 1) * E)[0]
                                     for j in range(self.width)]))
    if isinstance(witness, np.ndarray):
      return limbs_to_ints(witness[:, -1, :])
    return [element_to_int(col[-1]) % self.field.p for col in witness]

  def _boundary_interpolants(self, boundary, outputs):
    """I_j, the line through (1, input_j) and (last, output_j), for every column (construct_boundary_polynomials,
    :80-104): [i0_1, i1_1, i0_2, i1_2, ...]."""
    p, last = self.field.p, int(self.last_step_position)
    interps = []
    for j, out in enumerate(outputs):
      (_, _, input_value) = boundary[j]
      interps += _interp2(p, 1, last, element_to_int(input_value) % p, out)
    return interps

  def _d_coefficients(self, eng, cols, src, dst, dst_stride, witness_check=None):
    """construct_remainder_polynomials (:57-78) for the columns `cols`: D_j = C_j / Z, from C_j's M
    coefficients at src + j*M into dst + j*dst_stride.  stk_quotient_z synchronises the stream, so a
    pending witness_check is read here, before a witness with elements >= p fails the divisibility
    assert instead."""
    M, steps = self.M, self.steps
    last_l = int_to_limbs(int(self.last_step_position))
    bad = ctypes.c_uint32(0)
    for j in cols:
      eng._check(eng.lib.stk_quotient_z(eng.ctx, src + j * M * E, M, steps, _u32(last_l),
                                        dst + j * dst_stride * E, ctypes.byref(bad)))
      raise_if_noncanonical(witness_check)
      assert bad.value == 0, "constraint polynomial is not divisible by Z (stark.py:74-75)"

  def _b_coefficients(self, eng, cols, d_coef, cs, d_interp, scratch, dst, dst_stride, clear):
    """construct_boundary_polynomials (:80-104) for the columns `cols`: B_j = (P_j - I_j) / ((X - 1)(X - last))
    from P_j's coefficients at d_coef + j*cs and I_j's two at d_interp + 2j, into the steps - 2 coefficients
    at dst + j*dst_stride; clear: zero the two stale ones above them.  scratch: steps elements per column
    whose last reader is already enqueued."""
    steps = self.steps
    one_l, last_l = int_to_limbs(1), int_to_limbs(int(self.last_step_position))
    for j in cols:
      a, q1 = dst + j * dst_stride * E, scratch + j * steps * E
      eng._check(eng.lib.stk_memcpy_d2d(eng.ctx, a, d_coef + j * cs * E, steps * E))
      eng._check(eng.lib.stk_vec_op(eng.ctx, 1, a, d_interp + 2 * j * E, a, 2))
      eng._check(eng.lib.stk_div_linear(eng.ctx, a, steps, _u32(one_l), 1, q1))
      eng._check(eng.lib.stk_div_linear(eng.ctx, q1, steps - 1, _u32(last_l), steps, a))
      if clear:
        eng._check(eng.lib.stk_memset(eng.ctx, a + (steps - 2) * E, 0, 2 * E))

  def coefficient_rows(self, eng, d_trace_ptr, boundary, out_vals, want=None, witness_check=None):
    """The 3w polynomials mk_proof commits to -- P_1..P_w (stark.py:27-36), D_1..D_w (:38-78),
    B_1..B_w (:80-104), in the leaf order of :247 -- as COEFFICIENT rows on the device: returns
    (buffer, row stride cs), row r at byte r*cs*32, zero-padded to cs >= deg + 1.  The sharded
    prover (dist.ShardedProver) evaluates slices of these rows on different GPUs; mk_proof itself
    takes shortcuts (pointwise quotients) that this form does not need.
    want: the rows the caller will read (global row numbers 0..3w-1; default all).  Only those --
    and what they depend on -- are computed: a rank that evaluates one column of a Fibonacci proof
    runs one or two transforms of size `steps` here instead of four.
    witness_check: the pending count from _witness, if any; ValueError when it finds elements >= p."""
    w, steps, M, GM = self.width, self.steps, self.M, self.GM
    G1 = pow(int(self.G2), self.extension_factor, self.field.p)
    want = set(range(3 * w)) if want is None else set(int(c) for c in want)
    nm, h_out, h_coef, h_exp = self._mono_arrays
    cs = M
    want_d = sorted(c - w for c in want if w <= c < 2 * w)
    want_b = sorted(c - 2 * w for c in want if c >= 2 * w)
    # P's coefficients: for its own rows, for B_j, and -- unless the constraint subgroup is the trace
    # domain itself -- for every column (C_j needs all of P on that subgroup)
    need_p = set(c for c in want if c < w) | set(want_b)
    if want_d and M != steps:
      need_p = set(range(w))
    d_coef = eng.alloc(3 * w * cs * E)
    eng._check(eng.lib.stk_memset(eng.ctx, d_coef.ptr, 0, 3 * w * cs * E))
    if len(need_p) == w:
      eng.ntt(d_trace_ptr, steps, steps, d_coef.ptr, cs, steps, w, G1, inverse=True)
    else:
      for j in sorted(need_p):
        eng.ntt(d_trace_ptr + j * steps * E, steps, steps, d_coef.at(j * cs * E), cs, steps, 1, G1, inverse=True)
    held = []
    d_t1 = eng.alloc(w * M * E)
    held.append(d_t1)
    if want_d:
      if M == steps:
        pev_ptr, pev_stride = d_trace_ptr, steps     # P_j on <G1> is the witness column itself
      else:
        d_t2 = eng.alloc(w * M * E)
        held.append(d_t2)
        eng.ntt(d_coef.ptr, steps, cs, d_t2.ptr, M, M, w, GM)
        pev_ptr, pev_stride = d_t2.ptr, M
      eng._check(eng.lib.stk_constraint_eval(eng.ctx, pev_ptr, M, M // steps, w, pev_stride, h_out.ctypes.data,
                                             h_coef.ctypes.data, h_exp.ctypes.data, nm, d_t1.ptr, M))
      d_t3 = eng.alloc(w * M * E)
      held.append(d_t3)
      if len(want_d) == w:
        eng.ntt(d_t1.ptr, M, M, d_t3.ptr, M, M, w, GM, inverse=True)
      else:
        for j in want_d:
          eng.ntt(d_t1.at(j * M * E), M, M, d_t3.at(j * M * E), M, M, 1, GM, inverse=True)
      self._d_coefficients(eng, want_d, d_t3.ptr, d_coef.at(w * cs * E), cs, witness_check)
    if want_b:
      d_i = eng.alloc(2 * w * E).upload(ints_to_limbs(self._boundary_interpolants(boundary, out_vals)))
      held.append(d_i)
      self._b_coefficients(eng, want_b, d_coef.ptr, cs, d_i.ptr, d_t1.ptr, d_coef.at(2 * w * cs * E), cs, clear=True)
    eng.sync()   # the scratch rows go back to the pool
    for b in held:
      b.free()
    raise_if_noncanonical(witness_check)
    return d_coef, cs

  def mk_proof(self, witness, boundary, keep_device=False):
    """stark.py:233-279."""
    t_start = time.time()
    marks = [("start", t_start)]
    mark = lambda name: marks.append((name, time.time()))
    eng = self._engine or default_engine()
    p = self.field.p
    eng.set_field(p)
    w, steps, ext, N, M, GM = self.width, self.steps, self.extension_factor, self.precision, self.M, self.GM
    G2, last = int(self.G2), int(self.last_step_position)
    nm, h_out, h_coef, h_exp = self._mono_arrays
    d_trace, owned, noncanonical = self._witness(eng, witness)
    d_cols = eng.alloc(3 * w * N * E)        # rows: P_1..P_w, D_1..D_w, B_1..B_w (stark.py:247)
    d_t1 = eng.alloc(w * N * E)
    d_t2 = eng.alloc(w * N * E)
    mark("upload")
    # construct_constraint_polynomials (:38-55), evaluation form -- on the constraint subgroup <G_M>,
    # the smallest that determines C; only D's final evaluation runs at size N.
    # On <G_M>, P_j(G1*x_k) is the evaluation M/steps places further on.
    # When every coefficient vector is short enough for the zero-padded transform (M <= N/8) the
    # 3w columns P, D, B are evaluated by ONE batched transform at the end; otherwise P goes
    # first (the constraints may need its size-N evaluations) and D, B follow on their own.
    merged = M * 8 <= N
    cs = M if merged else steps                 # coefficient row stride
    d_coef = eng.alloc((3 * w if merged else w) * cs * E)
    if merged and cs > steps:
      eng._check(eng.lib.stk_memset(eng.ctx, d_coef.ptr, 0, 3 * w * cs * E))
    # D's evaluations can be taken pointwise from P's wherever Z does not vanish (stk_quotient_eval):
    # then only P and B go through the size-N transform
    pointwise_d = M < N and 2 <= ext <= 16 and os.environ.get("STK_PROOF_POINTWISE", "1") != "0"
    # Where the coefficient rows of D and B live (pointer, row stride), and the scratch buffer that
    # takes each one's evaluations on its subgroup.  Unmerged, D and B sit in the scratch buffers,
    # which keeps this route at about 5 w N elements of device memory (d_cols, d_t1, d_t2).
    if merged:
      d_rows, d_stride, d_sub = d_coef.at(w * cs * E), cs, d_t1
      b_rows, b_stride, b_sub = d_coef.at(2 * w * cs * E), cs, d_t2
    else:
      d_rows, d_stride, d_sub = d_t1.ptr, M, d_t2
      b_rows, b_stride, b_sub = d_t2.ptr, steps, d_t1
    if (not merged or pointwise_d) and ext == 8 and p == P_STARK:
      # construct_trace_polynomials (:27-36) and the evaluation of P (:254-256) in one call: with an
      # 8x blowup the evaluations at every 8th point ARE the trace, so stk_lde copies that coset
      # instead of computing it (one eighth of the forward transform)
      eng.lde(d_trace.ptr, steps, steps, ext, w, G2, d_cols.ptr, N, d_coeffs=d_coef.ptr, coeff_stride=cs)
    else:
      # construct_trace_polynomials (:27-36): inverse transform over <G1>
      eng.ntt(d_trace.ptr, steps, steps, d_coef.ptr, cs, steps, w, pow(G2, ext, p), inverse=True)
      if not merged or pointwise_d:
        eng.ntt(d_coef.ptr, steps, cs, d_cols.ptr, N, N, w, G2)          # evaluation of P (:254-256)
    if M == N:
      pev_ptr, pev_stride = d_cols.ptr, N
    elif M == steps:
      pev_ptr, pev_stride = d_trace.ptr, steps   # P_j on <G1> is the witness column itself
    else:
      eng.ntt(d_coef.ptr, steps, cs, d_t2.ptr, M, M, w, GM)
      pev_ptr, pev_stride = d_t2.ptr, M
    eng._check(eng.lib.stk_constraint_eval(eng.ctx, pev_ptr, M, M // steps, w, pev_stride, h_out.ctypes.data,
                                           h_coef.ctypes.data, h_exp.ctypes.data, nm, d_t1.ptr, M))
    eng.ntt(d_t1.ptr, M, M, d_t2.ptr, M, M, w, GM, inverse=True)        # C's coefficients
    self._d_coefficients(eng, range(w), d_t2.ptr, d_rows, d_stride, noncanonical)
    if pointwise_d:
      # D on <G_M> (contains <G1>, where Z vanishes) from its coefficients, everything else pointwise
      eng.ntt(d_rows, M, d_stride, d_sub.ptr, M, M, w, GM)
      eng._check(eng.lib.stk_quotient_eval(eng.ctx, d_cols.ptr, N, ext, w, N, h_out.ctypes.data, h_coef.ctypes.data,
                                           h_exp.ctypes.data, nm, _u32(int_to_limbs(G2)), _u32(int_to_limbs(last)),
                                           d_sub.ptr, M, M, d_cols.at(w * N * E), N))
    elif not merged:
      eng.ntt(d_rows, M, d_stride, d_cols.at(w * N * E), N, N, w, G2)
    # construct_boundary_polynomials (:80-104)
    h_interp = ints_to_limbs(self._boundary_interpolants(boundary, self._last_row(witness)))
    d_i = eng.alloc(2 * w * E).upload(h_interp)
    # B's quotient has steps-2 coefficients; merged, the two stale ones above it would be transformed
    self._b_coefficients(eng, range(w), d_coef.ptr, cs, d_i.ptr, d_t1.ptr, b_rows, b_stride, clear=merged)
    if pointwise_d and p == P_STARK and steps >= 4:
      # B on <G1> (holds x = 1 and x = last, where the denominator vanishes) from its coefficients,
      # everything else pointwise from P's evaluations (stk_boundary_eval)
      eng.ntt(b_rows, steps - 2, b_stride, b_sub.ptr, steps, steps, w, pow(G2, ext, p))
      eng._check(eng.lib.stk_boundary_eval(eng.ctx, d_cols.ptr, N, ext, w, N, _u32(int_to_limbs(G2)),
                                           (steps - 1) * ext, h_interp.ctypes.data, b_sub.ptr, steps,
                                           d_cols.at(2 * w * N * E), N))
    elif pointwise_d and merged:
      eng.ntt(b_rows, cs, b_stride, d_cols.at(2 * w * N * E), N, N, w, G2)   # evaluation of B
    elif merged:
      eng.ntt(d_coef.ptr, cs, cs, d_cols.ptr, N, N, 3 * w, G2)           # evaluation of P, D, B (:254-256)
    else:
      eng.ntt(b_rows, steps - 2, b_stride, d_cols.at(2 * w * N * E), N, N, w, G2)
    mark("enqueue_polys")
    # merkelize_polynomial_evaluations (:257)
    d_mnodes = eng.alloc(32 * N)
    m_root = eng.merkle_commit(d_cols.ptr, N, 3 * w, N, d_mnodes.ptr)
    mark("m_root")
    d_l = eng.alloc(N * E)
    eng.lincomb(d_cols.ptr, N, 3 * w, N, lincomb_weights(m_root, w, steps, N, G2, p), d_l.ptr)
    d_lnodes = eng.alloc(32 * N)
    l_root = eng.merkle_commit(d_l.ptr, N, 1, N, d_lnodes.ptr)           # :262-263
    mark("l_root")
    # compute_merkle_spot_checks (:390-402), samples = 80
    positions = get_pseudorandom_indices(l_root, N, 80, exclude_multiples_of=ext)
    mb = eng.merkle_paths(d_cols.ptr, N, 3 * w, N, d_mnodes.ptr,
                          [x for pos in positions for x in (pos, (pos + ext) % N)])
    lb = eng.merkle_paths(d_l.ptr, N, 1, N, d_lnodes.ptr, positions)
    branches = interleave_branches(mb, lb)
    mark("spot_checks")
    # FRI on l (:267-276); its first layer's tree is l_mtree
    fri = FRI(self.field, engine=eng)
    fri_proof = fri.prove_from_device(DeviceLayer(eng, d_l.ptr, N, d_lnodes.ptr, l_root), G2,
                                      steps * self.get_degree(), exclude_multiples_of=ext)
    proof = [m_root, l_root, branches, fri_proof]
    mark("fri")
    self.timings = {"mk_proof_s": time.time() - t_start}
    for (a, ta), (b, tb) in zip(marks[:-1], marks[1:]):
      self.timings[b + "_ms"] = (tb - ta) * 1e3
    if keep_device:
      self.device = dict(cols=d_cols, pcoef=d_coef, l=d_l, mnodes=d_mnodes, lnodes=d_lnodes)
    else:
      for b in (d_coef, d_i, d_cols, d_t1, d_t2, d_mnodes, d_l, d_lnodes) + ((d_trace,) if owned else ()):
        b.free()
    return proof

  # --------------------------------------------------------------- verifier
  def verify_proof(self, proof, witness, boundary):
    """stark.py:281-317 (host-side; the reference hands the verifier the witness, :370)."""
    m_root, l_root, branches, fri_proof = proof
    fri = FRI(self.field, engine=self._engine)
    assert fri.verify_proximity_proof(fri_proof, l_root, self.G2, self.steps * self.get_degree(),
                                      exclude_multiples_of=self.extension_factor)
    samples = self.spot_check_security_factor
    positions = get_pseudorandom_indices(l_root, self.precision, samples,
                                         exclude_multiples_of=self.extension_factor)
    ks = get_pseudorandom_ks(m_root, 4)
    N, ext = self.precision, self.extension_factor
    leaves = None
    if self._engine is not None and N >= 4 and N & (N - 1) == 0:
      # all 3 * samples branches re-hashed in two kernels (stk_verify_branches)
      ml = self._engine.verify_branches(m_root, [x for pos in positions for x in (pos, (pos + ext) % N)],
                                        [branches[3 * i + d] for i in range(len(positions)) for d in (0, 1)])
      self._engine.verify_branches(l_root, positions, [branches[3 * i + 2] for i in range(len(positions))])
      leaves = ml
    interps = self._boundary_interpolants(boundary, self._last_row(witness))
    for i, pos in enumerate(positions):
      self.verify_proof_at_position(witness, boundary, ks, proof, i, pos,
                                    checked_leaves=None if leaves is None else leaves[2 * i:2 * i + 2],
                                    interps=interps)
    return True

  def _step(self, j, state, p):
    acc = 0
    for exps, c in self._monomials[j]:
      t = c
      for k, e in enumerate(exps):
        t = t * pow(state[k], e, p) % p
      acc = (acc + t) % p
    return acc

  def verify_proof_at_position(self, witness, boundary, ks, proof, i, pos, checked_leaves=None, interps=None):
    """stark.py:319-372.  checked_leaves: the two m-tree leaves of this position when their
    branches (and the l-tree branch) have already been verified in a batch.  interps: the boundary
    interpolants, when the caller has already read them from the witness."""
    if interps is None:
      interps = self._boundary_interpolants(boundary, self._last_row(witness))
    p, width = self.field.p, self.width
    m_root, l_root, branches, fri_proof = proof
    G2, last = int(self.G2), int(self.last_step_position)
    x = pow(G2, pos, p)
    if checked_leaves is not None:
      leaf1, leaf2 = (unpack_merkle_leaf(v, width, 3) for v in checked_leaves)
    else:
      leaf1 = unpack_merkle_leaf(verify_branch(m_root, pos, branches[i * 3]), width, 3)
      leaf2 = unpack_merkle_leaf(verify_branch(m_root, (pos + self.extension_factor) % self.precision,
                                               branches[i * 3 + 1]), width, 3)
      verify_branch(l_root, pos, branches[i * 3 + 2], output_as_int=True)
    f_ = lambda b: int.from_bytes(b, "big")   # field(bytes) does not reduce; values are canonical
    p_of_x = [f_(v) for v in leaf1[:width]]
    p_of_g1x = [f_(v) for v in leaf2[:width]]
    d_of_x = [f_(v) for v in leaf1[width:2 * width]]
    b_of_x = [f_(v) for v in leaf1[2 * width:]]
    zvalue = (pow(x, self.steps, p) - 1) * pow((x - last) % p, -1, p) % p
    for dim in range(width):                                             # transition constraints
      assert (p_of_g1x[dim] - self._step(dim, p_of_x, p) - zvalue * d_of_x[dim]) % p == 0
    zeropoly2_x = (x - 1) * (x - last) % p
    for dim in range(width):                                             # boundary constraints
      i0, i1 = interps[2 * dim:2 * dim + 2]
      assert (p_of_x[dim] - b_of_x[dim] * zeropoly2_x - (i0 + i1 * x)) % p == 0
