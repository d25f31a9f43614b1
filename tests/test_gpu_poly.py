"""GPU parity of the coefficient-form polynomial product and long division (stk_poly_mul,
stk_poly_divmod, and Polynomial.__mul__ / __divmod__ on top of them) against the CPU oracle's
schoolbook routines, element for element.

Both calls route every product by the modulus: forward transforms, a pointwise product and a
scaled inverse where Z/p has a root of unity of the power-of-two order the product needs, a direct
kernel where it has none (p = 31 and 7 at any useful length, p = 97 above 32).  Division runs
Newton iteration on the reversed divisor.  Inputs are uniform over the whole field [0, p) with
every limb random, and start with the values where carries and reductions turn over (0, 1, p-1,
2^255, ...).  Every output sits between canaries: nothing beyond the documented lengths may be
written, and the inputs must come back unchanged."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 2**256 - 351 * 2**32 + 1
BN254_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
BLS12_381_R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
PAT = 0xA5C35A3C
GUARD = 256          # elements of canary before and after every output
slow = pytest.mark.slow


@pytest.fixture(scope="module")
def eng():
  from starks_b200 import Engine
  e = Engine(0)
  yield e
  e.close()


def limbs(ints):
  if not len(ints):
    return np.zeros((0, 8), np.uint32)
  return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in ints), dtype="<u4").reshape(-1, 8).copy()


def ints(arr):
  b = np.ascontiguousarray(arr, dtype="<u4").tobytes()
  return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def edge_values(p):
  b = p.bit_length()
  cand = [0, 1, p - 1, p - 2, 2**255, 2**255 - 1, 2**256 - 2**64, 2**(b - 1), 2**(b - 1) - 1]
  out = []
  for v in cand:
    if v < p and v not in out:
      out.append(v)
  return out


def full_range(rng, n, p=P, lead=True):
  """n residues uniform over [0, p) (all limbs random, rejection on the top one), starting with
  edge_values(p) rotated by a random offset; lead=True makes the last one non-zero."""
  top = (1 << ((p.bit_length() - 1) % 32 + 1)) - 1
  out = [int(x) for x in rng.integers(0, p, size=n)] if p < 2**63 else []
  while len(out) < n:
    a = np.frombuffer(rng.bytes(max(n, 16) * 32), dtype=np.uint32).reshape(-1, 8).copy()
    a[:, 7] &= top
    out += [x for x in ints(a) if x < p]
  out = out[:n]
  E = edge_values(p)
  r = int(rng.integers(len(E)))
  E = E[r:] + E[:r]
  out[:min(len(E), n)] = E[:n]
  if lead and n and out[-1] == 0:
    out[-1] = p - 1
  return out


def padded(xs, n):
  assert len(xs) <= n
  return list(xs) + [0] * (n - len(xs))


class Guarded(object):
  """`elems` elements between two guards, everything pre-filled with the pattern."""

  def __init__(self, eng, elems):
    self.eng, self.elems = eng, elems
    self.buf = eng.alloc((elems + 2 * GUARD) * 32)
    self.buf.upload(np.full((elems + 2 * GUARD, 8), PAT, dtype=np.uint32))
    self.ptr = self.buf.ptr + GUARD * 32

  def body(self):
    got = self.buf.download((self.elems + 2 * GUARD, 8))
    assert (got[:GUARD] == PAT).all(), "write BELOW the output"
    assert (got[GUARD + self.elems:] == PAT).all(), "write ABOVE the output's documented length"
    return ints(got[GUARD:GUARD + self.elems])

  def free(self):
    self.buf.free()


def upload(eng, xs):
  A = limbs(xs)
  d = eng.alloc(max(A.nbytes, 32))
  if len(xs):
    d.upload(A)
  return d, A


def unchanged(d, A):
  if len(A):
    assert (d.download(A.shape) == A).all(), "an input was modified"
  d.free()


def dev_mul(eng, a, b):
  da, A = upload(eng, a)
  db, B = upload(eng, b)
  out = Guarded(eng, len(a) + len(b) - 1 if a and b else 0)
  eng.poly_mul(da.ptr, len(a), db.ptr, len(b), out.ptr)
  got = out.body()
  unchanged(da, A)
  unchanged(db, B)
  out.free()
  return got


def dev_divmod(eng, a, b):
  da, A = upload(eng, a)
  db, B = upload(eng, b)
  q = Guarded(eng, max(len(a) - len(b) + 1, 0))
  r = Guarded(eng, len(b) - 1)
  eng.poly_divmod(da.ptr, len(a), db.ptr, len(b), q.ptr, r.ptr)
  got = q.body(), r.body()
  unchanged(da, A)
  unchanged(db, B)
  q.free()
  r.free()
  return got


def check_mul(eng, oracle, p, a, b):
  eng.set_field(p)
  got = dev_mul(eng, a, b)
  want = padded(oracle.poly_mul(p, a, b), len(a) + len(b) - 1)
  bad = [i for i in range(len(want)) if got[i] != want[i]]
  assert not bad, "%d of %d coefficients differ, first at %s" % (len(bad), len(want), bad[:4])


def check_divmod(eng, oracle, p, a, b):
  eng.set_field(p)
  q, r = dev_divmod(eng, a, b)
  wq, wr = oracle.poly_divmod(p, a, b)
  assert q == padded(wq, len(q)), "quotient differs"
  assert r == padded(wr, len(r)), "remainder differs"
  return q, r


# ----------------------------------------------------------------------- products, STARK prime

MUL_SHAPES = [(1, 1), (1, 4097), (2, 3), (7, 9), (1000, 1), (1 << 10, 1 << 10), ((1 << 13) + 3, (1 << 12) - 1),
              (1 << 14, 1 << 14),
              (1 << 11, (1 << 11) + 1),         # na + nb - 1 = 2^12 exactly
              ((1 << 11) + 1, (1 << 11) + 1),   # 2^12 + 1
              (1 << 8, 1 << 8), (1 << 8, (1 << 8) + 1)]  # 2^9 - 1 and 2^9


@pytest.mark.parametrize("na,nb", MUL_SHAPES, ids=["%dx%d" % s for s in MUL_SHAPES])
def test_mul_stark(eng, oracle, na, nb):
  rng = np.random.default_rng(na * 7919 + nb)
  check_mul(eng, oracle, P, full_range(rng, na), full_range(rng, nb))


def test_mul_empty_writes_nothing(eng):
  eng.set_field(P)
  assert dev_mul(eng, [], [1, 2, 3]) == []
  da, _ = upload(eng, [1, 2])
  out = Guarded(eng, 0)
  eng.poly_mul(da.ptr, 2, 0, 0, out.ptr)
  assert out.body() == []
  out.free()
  da.free()


# ----------------------------------------------------------------------- division, STARK prime

def test_divmod_by_a_constant(eng, oracle):
  rng = np.random.default_rng(1)
  q, r = check_divmod(eng, oracle, P, full_range(rng, 300), [P - 2])
  assert len(q) == 300 and r == []


def test_divmod_linear_matches_div_linear(eng, oracle):
  """nb = 2: X - w with w of order 2^13, also against stk_div_linear (the prover's divisor)."""
  from starks_b200.engine import _u32
  from starks_b200.limbs import int_to_limbs
  n = 1 << 12
  w = pow(7, (P - 1) // (1 << 13), P)
  a = full_range(np.random.default_rng(2), n)
  q, r = check_divmod(eng, oracle, P, a, [(-w) % P, 1])
  da, A = upload(eng, a)
  out = eng.alloc((n - 1) * 32)
  eng._check(eng.lib.stk_div_linear(eng.ctx, da.ptr, n, _u32(int_to_limbs(w)), 1 << 13, out.ptr))
  assert ints(out.download((n - 1, 8))) == q
  assert r == [sum(c * pow(w, i, P) for i, c in enumerate(a)) % P]   # remainder theorem
  da.free()
  out.free()


def test_divmod_boundary_zerofier(eng, oracle):
  """nb = 3: (X - 1)(X - last), the divisor of the boundary quotient."""
  steps, ext = 1 << 9, 8
  g2 = pow(7, (P - 1) // (steps * ext), P)
  last = pow(g2, (steps - 1) * ext, P)
  b = oracle.poly_mul(P, [P - 1, 1], [(-last) % P, 1])
  check_divmod(eng, oracle, P, full_range(np.random.default_rng(3), steps), b)


@pytest.mark.parametrize("na,nb", [(0, 1), (0, 5), (3, 9), (8, 9), (9, 9), (10, 9), (1 << 14, 5),
                                   (1 << 14, (1 << 13) + 1), (5000, 4999), (4097, 2048), (1 << 12, 1)])
def test_divmod_shapes(eng, oracle, na, nb):
  rng = np.random.default_rng(na * 31 + nb)
  a, b = full_range(rng, na, lead=False), full_range(rng, nb)
  if na < nb:
    q, r = dev_divmod(eng, a, b)
    assert q == [] and r == padded(a, nb - 1)   # zero-padded when na < nb - 1
  else:
    check_divmod(eng, oracle, P, a, b)


def test_divmod_exact(eng, oracle):
  rng = np.random.default_rng(4)
  b, q0 = full_range(rng, 300), full_range(rng, 1700)
  a = oracle.poly_mul(P, b, q0)
  eng.set_field(P)
  q, r = dev_divmod(eng, a, b)
  assert q == q0 and r == [0] * 299


def test_divmod_constraint_by_transition_zerofier(eng, oracle):
  """mk_proof's Z = (X^steps - 1) / (X - last), built on the device, divided into the constraint
  polynomial the oracle's prover builds for a two-register AIR (starks/stark.py:38-78)."""
  steps, ext = 1 << 8, 8
  sp = [{(0, 1): 1}, {(1, 0): 1, (0, 2): 1}]
  S = oracle.StarkOracle(steps, ext, 2, sp)
  last = S.last_step_position
  z, zr = check_divmod(eng, oracle, P, [P - 1] + [0] * (steps - 1) + [1], [(-last) % P, 1])
  assert zr == [0]
  witness = oracle.computational_trace(P, [2, 3], steps, sp)
  tps = [oracle._strip(oracle.fft_1d(P, w, S.G1, inv=True, order=steps)) for w in witness]
  nxt = [oracle._strip([c * pow(S.G1, i, P) % P for i, c in enumerate(tp)]) for tp in tps]
  _, ds, _ = S.intermediates(witness, [(0, 0, 2), (0, 1, 3)])
  for j in range(2):
    cp = oracle.poly_sub(P, nxt[j], oracle.eval_step_poly_on_polys(P, sp[j], tps))
    q, r = check_divmod(eng, oracle, P, cp, z)
    assert oracle._strip(q) == ds[j] and r == [0] * len(r)


# ----------------------------------------------------------------------- large sizes

def points(n):
  rng = np.random.default_rng(16)
  return full_range(rng, n)


@slow
def test_mul_2_20(eng, oracle):
  rng = np.random.default_rng(20)
  n = 1 << 20
  a, b = full_range(rng, n), full_range(rng, n)
  eng.set_field(P)
  ab = dev_mul(eng, a, b)
  xs = points(16)
  ea, eb, eab = oracle.poly_eval(P, a, xs), oracle.poly_eval(P, b, xs), oracle.poly_eval(P, ab, xs)
  assert all(z == x * y % P for x, y, z in zip(ea, eb, eab))


@slow
def test_divmod_2_21_by_2_20(eng, oracle):
  rng = np.random.default_rng(21)
  a, b = full_range(rng, 1 << 21), full_range(rng, 1 << 20)
  eng.set_field(P)
  q, r = dev_divmod(eng, a, b)
  assert len(q) == (1 << 20) + 1 and len(r) == (1 << 20) - 1
  xs = points(16)
  ea, eb, eq, er = (oracle.poly_eval(P, v, xs) for v in (a, b, q, r))
  assert all(x == (y * z + w) % P for x, y, z, w in zip(ea, eb, eq, er))


# ----------------------------------------------------------------------- run-time moduli

TRANSFORM_FIELDS = [("bn254", BN254_R), ("bls12_381", BLS12_381_R)]
RT_SHAPES = [(1, 1), (3, 5), (100, 37), (1 << 11, (1 << 11) + 1), ((1 << 11) + 1, (1 << 11) + 1)]


@pytest.mark.parametrize("name,p", TRANSFORM_FIELDS, ids=[n for n, _ in TRANSFORM_FIELDS])
@pytest.mark.parametrize("na,nb", RT_SHAPES, ids=["%dx%d" % s for s in RT_SHAPES])
def test_mul_transform_route_runtime_modulus(eng, oracle, name, p, na, nb):
  rng = np.random.default_rng(na + nb)
  check_mul(eng, oracle, p, full_range(rng, na, p), full_range(rng, nb, p))


@pytest.mark.parametrize("name,p", TRANSFORM_FIELDS, ids=[n for n, _ in TRANSFORM_FIELDS])
@pytest.mark.parametrize("na,nb", [(1 << 12, 3), (1 << 12, (1 << 11) + 1), (1000, 1), (700, 699)])
def test_divmod_transform_route_runtime_modulus(eng, oracle, name, p, na, nb):
  rng = np.random.default_rng(na + nb)
  check_divmod(eng, oracle, p, full_range(rng, na, p), full_range(rng, nb, p))


# p = 31 and 7 have roots of order 2 only; p = 97 up to 32 (96 = 3 * 2^5)
DIRECT = [(31, 5, 7), (31, 40, 60), (31, 300, 200), (7, 9, 4), (7, 130, 70),
          (97, 16, 17), (97, 16, 18), (97, 20, 30), (97, 200, 150)]


@pytest.mark.parametrize("p,na,nb", DIRECT, ids=["p%d-%dx%d" % s for s in DIRECT])
def test_mul_small_moduli(eng, oracle, p, na, nb):
  rng = np.random.default_rng(p * na + nb)
  check_mul(eng, oracle, p, full_range(rng, na, p), full_range(rng, nb, p))


@pytest.mark.parametrize("p,na,nb", [(31, 50, 7), (31, 300, 120), (7, 100, 1), (7, 64, 33),
                                     (97, 40, 10), (97, 60, 30), (97, 400, 150)])
def test_divmod_small_moduli(eng, oracle, p, na, nb):
  rng = np.random.default_rng(p * na + nb)
  check_divmod(eng, oracle, p, full_range(rng, na, p), full_range(rng, nb, p))


# ----------------------------------------------------------------------- interface

def test_overlapping_outputs_raise(eng):
  eng.set_field(P)
  buf = eng.alloc(64 * 32)
  buf.upload(limbs(range(1, 65)))
  at = lambda i: buf.ptr + 32 * i
  with pytest.raises(ValueError):
    eng.poly_mul(at(0), 8, at(8), 8, at(15))          # product overlaps b
  with pytest.raises(ValueError):
    eng.poly_mul(at(20), 8, at(40), 8, at(10))        # ... overlaps a
  with pytest.raises(ValueError):
    eng.poly_divmod(at(0), 20, at(20), 5, at(30), at(45))   # q [30, 46) overlaps r [45, 49)
  with pytest.raises(ValueError):
    eng.poly_divmod(at(0), 20, at(20), 5, at(22), at(50))   # q overlaps b
  with pytest.raises(ValueError):
    eng.poly_divmod(at(0), 20, at(20), 5, at(30), at(18))   # r overlaps a and b
  buf.free()


def test_zero_leading_coefficient_raises(eng):
  eng.set_field(P)
  da, _ = upload(eng, [1, 2, 3, 4])
  db, _ = upload(eng, [5, 0])
  q, r = eng.alloc(64), eng.alloc(64)
  with pytest.raises(ValueError):
    eng.poly_divmod(da.ptr, 4, db.ptr, 2, q.ptr, r.ptr)
  with pytest.raises(ValueError):
    eng.poly_divmod(da.ptr, 4, db.ptr, 0, q.ptr, r.ptr)
  for x in (da, db, q, r):
    x.free()


# ----------------------------------------------------------------------- Polynomial

@pytest.mark.parametrize("p", [P, BN254_R, 97, 31])
def test_polynomial_arithmetic(eng, oracle, p):
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over
  F = IntegersModP(p)
  Poly = polynomials_over(F)
  rng = np.random.default_rng(p % 1000)
  a, b = full_range(rng, 150, p), full_range(rng, 61, p)
  A, B = Poly(a), Poly(b)
  prod = A * B
  assert type(prod) is Poly and prod == Poly(oracle.poly_mul(p, a, b))
  q, r = divmod(A, B)
  wq, wr = oracle.poly_divmod(p, a, b)
  assert type(q) is Poly and type(r) is Poly and q == Poly(wq) and r == Poly(wr)
  assert q.coefficients[-1] != 0 and all(isinstance(c, F) for c in q.coefficients + r.coefficients)
  assert A + B == Poly(oracle.poly_add(p, a, b)) and A - B == Poly(oracle.poly_sub(p, a, b))
  assert -A == Poly([(-x) % p for x in a]) and (A - A).is_zero()
  # ints and field elements act as constants, on either side
  assert A * 3 == 3 * A == A * F(3) == Poly([3 * x % p for x in a])
  assert A + 1 == 1 + A == Poly([(a[0] + 1) % p] + a[1:])
  assert 1 - A == Poly([(1 - a[0]) % p] + [(-x) % p for x in a[1:]])
  assert (A * 0).is_zero() and (A * Poly([])).is_zero()
  q5, r5 = divmod(A, 5)
  assert q5 == Poly([x * pow(5, -1, p) % p for x in a]) and r5.is_zero()
  qs, rs = divmod(B, A)                               # deg B < deg A
  assert qs.is_zero() and rs == B
  with pytest.raises(ZeroDivisionError):
    divmod(A, Poly([]))
  with pytest.raises(ZeroDivisionError):
    divmod(A, 0)
