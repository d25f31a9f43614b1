"""GPU parity of polynomial composition, powers and multivariate polynomials evaluated at
polynomials (stk_poly_compose, stk_poly_eval_multivar, and Polynomial.__call__ / __pow__,
MultiVarPoly.__call__ and eval_at_polynomials on top of them) against the CPU oracle.

Composition takes the scaling route for b = alpha X (one pointwise kernel) and divide and conquer
over a padded to a power of two for any other b; multivariate evaluation runs forward transforms,
one pointwise kernel and an inverse where Z/p has a root of the needed order, and products through
the direct kernel where it has none (p = 31, p = 97 past 32).  Inputs are drawn over all of [0, p)
starting with edge values; every output sits between canaries and every input must come back
unchanged."""
import numpy as np
import pytest

from test_gpu_poly import BLS12_381_R, BN254_R, P, Guarded, full_range, ints, limbs, padded, unchanged, upload

pytestmark = pytest.mark.gpu
slow = pytest.mark.slow


@pytest.fixture(scope="module")
def eng():
  from starks_b200 import Engine
  e = Engine(0)
  yield e
  e.close()


def horner_compose(oracle, p, a, b):
  acc = []
  for c in reversed(a):
    acc = oracle.poly_add(p, oracle.poly_mul(p, acc, b), [c])
  return acc


def dev_compose(eng, a, b):
  da, A = upload(eng, a)
  db, B = upload(eng, b)
  out = Guarded(eng, (len(a) - 1) * (len(b) - 1) + 1 if a else 0)
  eng.poly_compose(da.ptr, len(a), db.ptr, len(b), out.ptr)
  got = out.body()
  unchanged(da, A)
  unchanged(db, B)
  out.free()
  return got


def inner(rng, kind, p):
  """b = alpha X, alpha X + beta (beta != 0), or nb coefficients."""
  if kind == "ax":
    return [0, full_range(rng, 2, p)[1]]       # the last draw is non-zero
  if kind == "ax+b":
    ab = full_range(rng, 2, p)
    return [ab[0] or 1, ab[1]]
  return full_range(rng, kind, p)


def check_compose(eng, oracle, p, a, b):
  eng.set_field(p)
  got = dev_compose(eng, a, b)
  want = padded(horner_compose(oracle, p, a, b), len(got))
  bad = [i for i in range(len(want)) if got[i] != want[i]]
  assert not bad, "%d of %d coefficients differ, first at %s" % (len(bad), len(want), bad[:4])


def dev_multivar(eng, args, monomials, nout, out_len):
  """stk_poly_eval_multivar on guarded outputs; args at one stride."""
  stride = max([len(a) for a in args] + [1])
  buf = eng.alloc(len(args) * stride * 32)
  rows = np.zeros((len(args), stride, 8), dtype=np.uint32)
  for k, a in enumerate(args):
    rows[k, :len(a)] = limbs(a)
  buf.upload(rows)
  out = Guarded(eng, nout * out_len)
  eng.poly_eval_multivar(buf.ptr, [len(a) for a in args], stride, monomials, nout, out.ptr, out_len)
  got = out.body()
  assert (buf.download(rows.shape) == rows).all(), "an argument was modified"
  buf.free()
  out.free()
  return [got[j * out_len:(j + 1) * out_len] for j in range(nout)]


def out_len_of(args, step_polys):
  from starks_b200.polynomial import _out_len
  return _out_len([len(a) for a in args], [(0, 1, e) for sp in step_polys for e in sp])


def check_multivar(eng, oracle, p, args, step_polys):
  eng.set_field(p)
  monomials = [(j, c, e) for j, sp in enumerate(step_polys) for e, c in sp.items()]
  n = out_len_of(args, step_polys)
  got = dev_multivar(eng, args, monomials, len(step_polys), n)
  for j, sp in enumerate(step_polys):
    want = oracle.eval_step_poly_on_polys(p, {e: c % p for e, c in sp.items()}, args)
    assert got[j] == padded(want, n), "output %d differs" % j


# ----------------------------------------------------------------------- composition, STARK prime

# (na, inner): every na with alpha X, alpha X + beta, nb = 3 and 5; nb = 17 to na = 257 and
# nb = 64, 65 to na = 33 (the Horner oracle's cost grows as (na nb)^2).  na = 32 pads to exactly
# 2^5 and 33 to 2^6; (2, 64) and (2, 65) write 2^6 and 2^6 + 1 coefficients, (33, 3) 2^6 + 1.
NAS = [1, 2, 3, 31, 32, 33, 257, 1000]
COMPOSE = ([(na, k) for na in NAS for k in ("ax", "ax+b", 3, 5)] + [(na, 17) for na in NAS if na <= 257] +
           [(na, k) for na in NAS if na <= 33 for k in (64, 65)])


@pytest.mark.parametrize("na,kind", COMPOSE, ids=["%dx%s" % s for s in COMPOSE])
def test_compose_stark(eng, oracle, na, kind):
  rng = np.random.default_rng(na * 131 + (kind if isinstance(kind, int) else len(kind)))
  check_compose(eng, oracle, P, full_range(rng, na), inner(rng, kind, P))


def test_compose_alpha_zero_and_empty(eng, oracle):
  """b = 0 X (scaling by 0^k) leaves a_0; na = 0 writes nothing."""
  a = full_range(np.random.default_rng(5), 40)
  eng.set_field(P)
  assert dev_compose(eng, a, [0, 0]) == [a[0]] + [0] * 39
  check_compose(eng, oracle, P, a, [7, 0, 0])   # constant b with explicit zeros: a(7), padded
  assert dev_compose(eng, [], [1, 2, 3]) == []


@slow
@pytest.mark.parametrize("logn", [16, 20])
def test_compose_scaling_at_size(eng, logn):
  rng = np.random.default_rng(logn)
  n = 1 << logn
  a = full_range(rng, n)
  alpha = full_range(rng, 3)[2] or 3
  eng.set_field(P)
  got = dev_compose(eng, a, [0, alpha])
  pw = 1
  for k in range(n):
    assert got[k] == a[k] * pw % P, "coefficient %d differs" % k
    pw = pw * alpha % P


def points(n):
  return full_range(np.random.default_rng(16), n)


@pytest.mark.parametrize("na,nb", [(1 << 12, (1 << 6) + 1), (1 << 16, 2)])
def test_compose_general_at_size(eng, oracle, na, nb):
  rng = np.random.default_rng(na + nb)
  a, b = full_range(rng, na), full_range(rng, nb)
  if nb == 2 and b[0] == 0:
    b[0] = 5
  eng.set_field(P)
  got = dev_compose(eng, a, b)
  assert len(got) == (na - 1) * (nb - 1) + 1
  xs = points(16)
  assert oracle.poly_eval(P, got, xs) == oracle.poly_eval(P, a, oracle.poly_eval(P, b, xs))


# ----------------------------------------------------------------------- powers

def repeated(oracle, p, a, e):
  acc = [1]
  for _ in range(e):
    acc = oracle.poly_mul(p, acc, a)
  return acc


@pytest.mark.parametrize("e", [0, 1, 2, 3, 8, 255, 256, 1000])
@pytest.mark.parametrize("n", [1, 2, 3])
def test_pow_small(eng, oracle, n, e):
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over
  Poly = polynomials_over(IntegersModP(P))
  a = full_range(np.random.default_rng(n * 1000 + e), n)
  got = Poly(a) ** e
  assert type(got) is Poly and got == Poly(repeated(oracle, P, a, e))
  # the same through the entry point, between canaries
  eng.set_field(P)
  [raw] = dev_multivar(eng, [a], [(0, 1, (e,))], 1, e * (n - 1) + 1)
  assert raw == padded(repeated(oracle, P, a, e), e * (n - 1) + 1)


def test_pow_edges():
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over
  Poly = polynomials_over(IntegersModP(P))
  assert Poly([]) ** 0 == Poly([1]) and Poly([3, 4]) ** 0 == Poly([1])
  assert (Poly([]) ** 5).is_zero()
  assert Poly([0, 1]) ** 300 == Poly([0] * 300 + [1])
  with pytest.raises(ValueError):
    Poly([1, 2]) ** -1


def test_pow_2_14_by_8(oracle):
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over
  Poly = polynomials_over(IntegersModP(P))
  a = full_range(np.random.default_rng(14), 1 << 14)
  got = Poly(a) ** 8
  assert len(got) == 8 * ((1 << 14) - 1) + 1
  xs = points(16)
  assert oracle.poly_eval(P, [int(c) for c in got], xs) == [pow(v, 8, P) for v in oracle.poly_eval(P, a, xs)]


# ----------------------------------------------------------------------- multivariate

def deg_air(d):
  return [{(0, 1): 1}, {(1, 0): 1, (0, d): 1, (0, 0): 5}]


STEP_POLYS = [
    ("fibonacci", [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}]),
    ("cubic+const", [{(3,): 1, (1,): 2, (0,): 5}]),
    *[("degree-%d" % d, deg_air(d)) for d in range(2, 9)],
    ("3-wide", [{(0, 1, 0): 1}, {(0, 0, 1): 1}, {(1, 1, 0): 7, (0, 0, 2): P - 1, (0, 0, 0): 9}]),
    ("4-wide", [{(0, 1, 0, 0): 1}, {(0, 0, 1, 1): 1}, {(2, 1, 0, 0): 1, (0, 0, 0, 1): 1},
                {(1, 0, 0, 0): 1, (0, 1, 1, 0): 3}]),
    ("6-wide", [{(0, 1, 0, 0, 0, 0): 1}, {(0, 0, 1, 0, 0, 0): 2}, {(0, 0, 0, 1, 1, 0): 1},
                {(0, 0, 0, 0, 1, 0): 1, (3, 0, 0, 0, 0, 0): 4}, {(0, 0, 0, 0, 0, 1): 1, (0, 2, 0, 0, 0, 1): 1},
                {(1, 1, 1, 1, 1, 1): P - 3, (0, 0, 0, 0, 0, 0): 1}]),
]


@pytest.mark.parametrize("name,sp", STEP_POLYS, ids=[n for n, _ in STEP_POLYS])
def test_multivar_step_polys(eng, oracle, name, sp):
  """Arguments of different lengths per variable."""
  rng = np.random.default_rng(len(name) * 17 + len(sp))
  width = len(next(iter(sp[0])))
  args = [full_range(rng, 37 + 29 * k) for k in range(width)]
  check_multivar(eng, oracle, P, args, sp)


def test_multivar_zero_and_constant_arguments(eng, oracle):
  rng = np.random.default_rng(9)
  a, c = full_range(rng, 50), [full_range(rng, 1)[0] or 2]
  # zero argument with exponent 0 (a factor of 1) and with exponent > 0 (the monomial vanishes)
  sp = [{(2, 0, 0): 3, (1, 0, 1): 5}, {(0, 1, 2): 1, (1, 0, 0): 4}, {(0, 0, 3): 1}, {(0, 1, 0): 2}]
  for args in ([a, [], c], [c, c, a], [[], [], c]):
    check_multivar(eng, oracle, P, args, sp)
  # no monomial at all: zero outputs of one coefficient
  assert dev_multivar(eng, [a], [], 2, 1) == [[0], [0]]


def test_multivar_polynomial_interface(eng, oracle):
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import MultiVarPoly, eval_at_polynomials, polynomials_over
  F = IntegersModP(P)
  Poly = polynomials_over(F)
  rng = np.random.default_rng(12)
  a, b = full_range(rng, 33), full_range(rng, 20)
  sp = {(1, 0): 1, (0, 2): 3, (1, 1): P - 1}
  m = MultiVarPoly(F, 2, sp)
  got = m([Poly(a), Poly(b)])
  assert type(got) is Poly and got == Poly(oracle.eval_step_poly_on_polys(P, sp, [a, b]))
  assert m([Poly(a), 7]) == m([Poly(a), F(7)]) == Poly(oracle.eval_step_poly_on_polys(P, sp, [a, [7]]))
  y = m([3, 5])                                       # no polynomial: the host path, a field element
  assert isinstance(y, F) and int(y) == (3 + 3 * 25 - 15) % P
  outs = eval_at_polynomials([m, MultiVarPoly(F, 2, {(0, 1): 1}), MultiVarPoly(F, 2, {})], [Poly(a), Poly(b)])
  assert outs[0] == got and outs[1] == Poly(b) and outs[2].is_zero()


# ----------------------------------------------------------------------- the reference's constraint step

AIRS = [("fibonacci", [0, 1], [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}]),
        ("degree-3", [3], [{(3,): 1, (1,): 2, (0,): 5}]),
        ("4-wide-mixed", [1, 2, 3, 4], [{(0, 1, 0, 0): 1}, {(0, 0, 1, 1): 1}, {(2, 1, 0, 0): 1, (0, 0, 0, 1): 1},
                                        {(1, 0, 0, 0): 1, (0, 1, 1, 0): 3}])]


@pytest.mark.parametrize("steps", [32, 256, 1024])
@pytest.mark.parametrize("name,inp,sp", AIRS, ids=[n for n, _, _ in AIRS])
def test_constraint_polynomials_end_to_end(oracle, name, inp, sp, steps):
  """C_j = P_j(G1 X) - step_j(P) through the Polynomial API (starks/stark.py:38-55), and
  divmod(C_j, Z) equal to the oracle's D_j with a zero remainder (:57-78)."""
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import MultiVarPoly, eval_at_polynomials, polynomials_over
  F = IntegersModP(P)
  Poly = polynomials_over(F)
  width = len(inp)
  S = oracle.StarkOracle(steps, 8, width, sp)
  witness = oracle.computational_trace(P, inp, steps, sp)
  tps, ds, _ = S.intermediates(witness, [(0, j, inp[j]) for j in range(width)])
  trace = [Poly(tp) for tp in tps]
  G1X = Poly([0, S.G1])
  stepped = eval_at_polynomials([MultiVarPoly(F, width, s) for s in sp], trace)
  z, zr = divmod(Poly([P - 1] + [0] * (steps - 1) + [1]), Poly([(-S.last_step_position) % P, 1]))
  assert zr.is_zero()
  for j in range(width):
    c = trace[j](G1X) - stepped[j]
    q, r = divmod(c, z)
    assert q == Poly(ds[j]) and r.is_zero(), "D_%d differs" % j


# ----------------------------------------------------------------------- other fields

TRANSFORM_FIELDS = [("bn254", BN254_R), ("bls12_381", BLS12_381_R)]


@pytest.mark.parametrize("name,p", TRANSFORM_FIELDS, ids=[n for n, _ in TRANSFORM_FIELDS])
@pytest.mark.parametrize("na,kind", [(1, 3), (33, "ax"), (33, "ax+b"), (40, 5), (100, 17)])
def test_compose_runtime_modulus(eng, oracle, name, p, na, kind):
  rng = np.random.default_rng(na + len(name))
  check_compose(eng, oracle, p, full_range(rng, na, p), inner(rng, kind, p))


@pytest.mark.parametrize("name,p", TRANSFORM_FIELDS, ids=[n for n, _ in TRANSFORM_FIELDS])
def test_multivar_runtime_modulus(eng, oracle, name, p):
  rng = np.random.default_rng(len(name))
  sp = [{(0, 1): 1}, {(1, 0): 1, (0, 3): p - 2, (0, 0): 7}, {(2, 2): 1}]
  check_multivar(eng, oracle, p, [full_range(rng, 30, p), full_range(rng, 17, p)], sp)
  check_multivar(eng, oracle, p, [full_range(rng, 3, p)], [{(256,): 1}, {(300,): 2, (1,): 1}])


def test_multivar_outputs_beyond_a_grid_dimension(eng):
  """The batched inverse transform of multivariate evaluation has one column per output.  Over
  BN254's scalar field a transform of length 2048 takes two passes, whose launches hold at most
  65535 columns: 65 537 outputs (j + 1) x of a 1025-coefficient x must come back whole on both
  sides of every column group."""
  import torch
  p, n, nout = BN254_R, 1025, 65537
  x = full_range(np.random.default_rng(11), n, p)
  eng.set_field(p)
  dx = torch.from_numpy(limbs(x).view(np.int32)).cuda()
  out = torch.empty((nout, n, 8), dtype=torch.int32, device="cuda")
  torch.cuda.synchronize()
  eng.poly_eval_multivar(dx.data_ptr(), [n], n, [(j, j + 1, (1,)) for j in range(nout)], nout, out.data_ptr(), n)
  eng.sync()
  for j in (0, 1, 32767, 32768, 65535, 65536):
    assert ints(out[j].cpu().numpy().view(np.uint32)) == [(j + 1) * v % p for v in x], j
  del dx, out
  torch.cuda.empty_cache()


# p = 31 has roots of order 2 only, p = 97 up to 32: the product / direct route, na > p included
SMALL = [(31, 40, 3), (31, 40, "ax+b"), (31, 70, "ax"), (97, 20, 5), (97, 120, 3), (97, 130, "ax+b"), (97, 9, 17)]


@pytest.mark.parametrize("p,na,kind", SMALL, ids=["p%d-%dx%s" % s for s in SMALL])
def test_compose_small_moduli(eng, oracle, p, na, kind):
  rng = np.random.default_rng(p * na)
  check_compose(eng, oracle, p, full_range(rng, na, p), inner(rng, kind, p))


@pytest.mark.parametrize("p", [31, 97])
def test_multivar_small_moduli(eng, oracle, p):
  rng = np.random.default_rng(p)
  sp = [{(0, 1): 1}, {(1, 0): 1, (0, 3): p - 2, (0, 0): 7}, {(5, 2): 3}]
  check_multivar(eng, oracle, p, [full_range(rng, 12, p), full_range(rng, 9, p)], sp)
  check_multivar(eng, oracle, p, [full_range(rng, 2, p), []], [{(40, 0): 1, (0, 1): 1}, {(0, 0): 3}])


# ----------------------------------------------------------------------- errors

def test_compose_errors(eng):
  from starks_b200 import StarksB200Error
  eng.set_field(P)
  buf = eng.alloc(64 * 32)
  buf.upload(limbs(range(1, 65)))
  at = lambda i: buf.ptr + 32 * i
  with pytest.raises(ValueError):
    eng.poly_compose(at(0), 8, at(8), 1, at(20))      # nb < 2
  with pytest.raises(ValueError):
    eng.poly_compose(at(0), 8, at(8), 0, at(20))
  with pytest.raises(ValueError):
    eng.poly_compose(at(0), 8, at(8), 3, at(5))       # output overlaps a
  with pytest.raises(ValueError):
    eng.poly_compose(at(0), 8, at(20), 3, at(10))     # output [10, 25) overlaps b
  buf.free()
  # (2^16)(2^14 + 1) coefficients: past 2^30, nothing written
  da, _ = upload(eng, [1, 2])
  out = Guarded(eng, 16)
  with pytest.raises(StarksB200Error):
    eng.poly_compose(da.ptr, (1 << 16) + 1, da.ptr, (1 << 14) + 1, out.ptr)
  assert out.body() == [int.from_bytes(np.full(8, 0xA5C35A3C, "<u4").tobytes(), "little")] * 16
  out.free()
  da.free()


def test_multivar_errors(eng):
  from starks_b200 import StarksB200Error
  eng.set_field(P)
  d, _ = upload(eng, list(range(1, 14 * 4 + 1)))
  out = eng.alloc(64 * 32)
  with pytest.raises(StarksB200Error):                # width > 12
    eng.poly_eval_multivar(d.ptr, [4] * 13, 4, [(0, 1, (1,) * 13)], 1, out.ptr, 13 * 3 + 1)
  with pytest.raises(ValueError):                     # out_len must be D + 1 = 7
    eng.poly_eval_multivar(d.ptr, [4, 4], 4, [(0, 1, (2, 0))], 1, out.ptr, 8)
  with pytest.raises(ValueError):
    eng.poly_eval_multivar(d.ptr, [4, 4], 4, [(0, 1, (2, 0))], 1, out.ptr, 6)
  with pytest.raises(ValueError):                     # output index out of range
    eng.poly_eval_multivar(d.ptr, [4, 4], 4, [(1, 1, (2, 0))], 1, out.ptr, 7)
  with pytest.raises(ValueError):                     # output overlaps an argument
    eng.poly_eval_multivar(d.ptr, [4, 4], 4, [(0, 1, (2, 0))], 1, d.ptr + 32 * 6, 7)
  with pytest.raises(StarksB200Error):                # D + 1 past 2^30
    eng.poly_eval_multivar(d.ptr, [4], 4, [(0, 1, (1 << 29,))], 1, out.ptr, 3 * (1 << 29) + 1)
  d.free()
  out.free()
