"""Minimal dense-polynomial value types mirroring what the hot path touches of
starks/polynomial.py (coefficient list low -> high, trailing zeros stripped, :58; Horner
__call__, :158-164; products and long division, :110-143) and of
starks/multivariate_polynomial.py (dict monomial -> coefficient, __call__ :329-338).  Products,
divisions, composition, powers and multivariate polynomials evaluated at polynomials run on the
device (stk_poly_mul, stk_poly_divmod, stk_poly_compose, stk_poly_eval_multivar); the rest is
host-side glue."""
import functools
import itertools

import numpy as np

from .engine import default_engine
from .limbs import ints_to_limbs, limbs_to_ints
from .modp import element_to_int


def _upload(eng, coeffs):
  buf = eng.alloc(max(len(coeffs), 1) * 32)
  if coeffs:
    buf.upload(ints_to_limbs(element_to_int(x) for x in coeffs))
  return buf


class _Polynomial(object):
  """Common base of the classes polynomials_over makes, so that MultiVarPoly can tell a
  polynomial argument from a constant."""


def _out_len(lens, monomials):
  """D + 1 of stk_poly_eval_multivar: D = max over the monomials that do not vanish (no positive
  exponent on an empty argument) of sum_k e_k (len_k - 1), 0 if none."""
  D = 0
  for _, _, exps in monomials:
    if not any(e and not n for e, n in zip(exps, lens)):
      D = max(D, sum(e * (n - 1) for e, n in zip(exps, lens) if e))
  return D + 1


def _eval_multivar(poly_cls, args, monomials, nout):
  """Device evaluation of nout multivariate polynomials (monomials: (output, int coefficient,
  exponent tuple)) at the polynomial arguments args; returns nout poly_cls."""
  lens = [len(a) for a in args]
  stride = max(lens + [1])
  out_len = _out_len(lens, monomials)
  eng = poly_cls._engine()
  buf = eng.alloc(len(args) * stride * 32)
  dout = eng.alloc(max(nout, 1) * out_len * 32)
  try:
    rows = np.zeros((len(args), stride, 8), dtype=np.uint32)
    for k, a in enumerate(args):
      if lens[k]:
        rows[k, :lens[k]] = ints_to_limbs(element_to_int(x) for x in a.coefficients)
    buf.upload(rows)
    eng.poly_eval_multivar(buf.ptr, lens, stride, monomials, nout, dout.ptr, out_len)
    got = limbs_to_ints(dout.download((nout, out_len, 8)).reshape(-1, 8)) if nout else []
    return [poly_cls([poly_cls.ring(v) for v in got[j * out_len:(j + 1) * out_len]]) for j in range(nout)]
  finally:
    buf.free()
    dout.free()


@functools.lru_cache(maxsize=None)
def polynomials_over(ring):
  class Polynomial(_Polynomial):
    def __init__(self, c):
      if isinstance(c, Polynomial):
        coeffs = list(c.coefficients)
      elif hasattr(c, "__iter__"):
        coeffs = [x if isinstance(x, ring) else ring(x) for x in c]
      else:
        coeffs = [c if isinstance(c, ring) else ring(c)]
      while coeffs and int(coeffs[-1]) == 0:         # polynomial.py:58
        coeffs.pop()
      self.coefficients = coeffs

    @classmethod
    def factory(cls, L):
      return Polynomial(L)

    def is_zero(self):
      return self.coefficients == []

    def degree(self):
      return len(self.coefficients) - 1

    def __len__(self):
      return len(self.coefficients)

    def __iter__(self):
      return iter(self.coefficients)

    def __eq__(self, other):
      oc = getattr(other, "coefficients", None)
      if oc is None:
        return False
      return [int(x) for x in self.coefficients] == [element_to_int(x) for x in oc]

    def __call__(self, x):                           # polynomial.py:158-164
      if isinstance(x, Polynomial):                  # a(x(X)): stk_poly_compose
        if len(x) < 2:
          return Polynomial([self(x.coefficients[0] if len(x) else ring(0))])
        na, nb = len(self), len(x)
        if not na:
          return Polynomial([])
        eng = Polynomial._engine()
        da, db = _upload(eng, self.coefficients), _upload(eng, x.coefficients)
        n = (na - 1) * (nb - 1) + 1
        dout = eng.alloc(n * 32)
        try:
          eng.poly_compose(da.ptr, na, db.ptr, nb, dout.ptr)
          return Polynomial._download(dout, n)
        finally:
          for b in (da, db, dout):
            b.free()
      acc = ring(0)
      for c in reversed(self.coefficients):
        acc = acc * x + c
      return acc

    def __pow__(self, e):                            # one variable, one monomial: stk_poly_eval_multivar
      if not isinstance(e, int):
        return NotImplemented
      if e < 0:
        raise ValueError("a polynomial has no negative powers")
      return _eval_multivar(Polynomial, [self], [(0, 1, (e,))], 1)[0]

    @staticmethod
    def _lift(other):
      """Anything the constructor accepts: an int or a field element is a constant."""
      return other if isinstance(other, Polynomial) else Polynomial(other)

    def __add__(self, other):
      o = Polynomial._lift(other)
      zero = ring(0)
      return Polynomial([x + y for x, y in itertools.zip_longest(self.coefficients, o.coefficients,
                                                                  fillvalue=zero)])
    __radd__ = __add__

    def __neg__(self):
      return Polynomial([-x for x in self.coefficients])

    def __sub__(self, other):
      return self + (-Polynomial._lift(other))

    def __rsub__(self, other):
      return Polynomial._lift(other) + (-self)

    @staticmethod
    def _engine():
      eng = default_engine()
      eng.set_field(ring.p)
      return eng

    @staticmethod
    def _download(buf, n):
      return Polynomial([ring(v) for v in limbs_to_ints(buf.download((n, 8)))])

    def __mul__(self, other):                        # polynomial.py:110-121, stk_poly_mul
      o = Polynomial._lift(other)
      na, nb = len(self), len(o)
      if not na or not nb:
        return Polynomial([])
      eng = Polynomial._engine()
      da, db = _upload(eng, self.coefficients), _upload(eng, o.coefficients)
      dout = eng.alloc((na + nb - 1) * 32)
      try:
        eng.poly_mul(da.ptr, na, db.ptr, nb, dout.ptr)
        return Polynomial._download(dout, na + nb - 1)
      finally:
        for x in (da, db, dout):
          x.free()
    __rmul__ = __mul__

    def __divmod__(self, divisor):                   # polynomial.py:128-143, stk_poly_divmod
      d = Polynomial._lift(divisor)
      if d.is_zero():
        raise ZeroDivisionError("polynomial division by zero")
      na, nb = len(self), len(d)
      nq, nr = max(na - nb + 1, 0), nb - 1
      eng = Polynomial._engine()
      da, db = _upload(eng, self.coefficients), _upload(eng, d.coefficients)
      dq, dr = eng.alloc(max(nq, 1) * 32), eng.alloc(max(nr, 1) * 32)
      try:
        eng.poly_divmod(da.ptr, na, db.ptr, nb, dq.ptr, dr.ptr)
        return Polynomial._download(dq, nq), Polynomial._download(dr, nr)
      finally:
        for x in (da, db, dq, dr):
          x.free()

    def __repr__(self):
      return "Polynomial(%r)" % ([int(c) for c in self.coefficients],)

  Polynomial.ring = ring
  return Polynomial


class MultiVarPoly(object):
  """Sparse multivariate polynomial {exponent tuple: coefficient} over Z/p, enough to write
  AIR step functions (X_1 + X_2**3 ...) and to evaluate them on states."""

  def __init__(self, field, num_vars, coefficients):
    self.field, self.num_vars = field, num_vars
    self.coefficients = {tuple(k): (v if isinstance(v, field) else field(v))
                         for k, v in coefficients.items() if int(v if not hasattr(v, "n") else v.n) % field.p}

  def _lift(self, other):
    if isinstance(other, MultiVarPoly):
      return other
    return MultiVarPoly(self.field, self.num_vars, {(0,) * self.num_vars: self.field(other)})

  def __add__(self, other):
    o = self._lift(other)
    out = dict(self.coefficients)
    for k, v in o.coefficients.items():
      out[k] = out.get(k, self.field(0)) + v
    return MultiVarPoly(self.field, self.num_vars, out)
  __radd__ = __add__

  def __neg__(self):
    return MultiVarPoly(self.field, self.num_vars, {k: -v for k, v in self.coefficients.items()})

  def __sub__(self, other):
    return self + (-self._lift(other))

  def __mul__(self, other):
    o = self._lift(other)
    out = {}
    for k1, v1 in self.coefficients.items():
      for k2, v2 in o.coefficients.items():
        k = tuple(a + b for a, b in zip(k1, k2))
        out[k] = out.get(k, self.field(0)) + v1 * v2
    return MultiVarPoly(self.field, self.num_vars, out)
  __rmul__ = __mul__

  def __pow__(self, e):
    r = MultiVarPoly(self.field, self.num_vars, {(0,) * self.num_vars: self.field(1)})
    for _ in range(int(e)):
      r = r * self
    return r

  def degree(self):
    return max([sum(k) for k in self.coefficients] or [0])

  def __call__(self, vals):                          # multivariate_polynomial.py:329-338
    assert len(vals) == self.num_vars
    if any(isinstance(v, _Polynomial) for v in vals):
      return eval_at_polynomials([self], vals)[0]
    y = self.field(0)
    for k in sorted(self.coefficients):
      prod = self.field(1)
      for i, power in enumerate(k):
        prod = prod * vals[i]**power
      y = y + self.coefficients[k] * prod
    return y


def eval_at_polynomials(mvps, polys):
  """[m(polys) for m in mvps] in one device call (stk_poly_eval_multivar): the reference's
  step_j(P_1, ..., P_w) for every j (starks/stark.py:49).  At least one of polys is a Polynomial;
  ints and field elements among them are constants.  Returns Polynomials of that class."""
  poly_cls = next(type(v) for v in polys if isinstance(v, _Polynomial))
  args = [v if isinstance(v, poly_cls) else poly_cls(v) for v in polys]
  monomials = []
  for j, m in enumerate(mvps):
    monomials += [(j, c, exps) for exps, c in monomials_of(m, len(args), poly_cls.ring.p)]
  return _eval_multivar(poly_cls, args, monomials, len(mvps))


def generate_Xi_s(field, width):
  """starks/utils.py:40-57: the index polynomials X_1 .. X_width."""
  return [MultiVarPoly(field, width, {tuple(1 if j == i else 0 for j in range(width)): field(1)})
          for i in range(width)]


def monomials_of(step_poly, width, p):
  """Normalises a step polynomial (MultiVarPoly here, the reference's MultivariatePolynomial,
  or a plain dict) to a list of (exponent tuple, int coefficient)."""
  coeffs = step_poly if isinstance(step_poly, dict) else step_poly.coefficients
  out = []
  for k in sorted(coeffs):
    assert len(k) == width
    c = element_to_int(coeffs[k]) % p
    if c:
      out.append((tuple(int(e) for e in k), c))
  return out
