"""Minimal dense-polynomial value types mirroring what the hot path touches of
starks/polynomial.py (coefficient list low -> high, trailing zeros stripped, :58; Horner
__call__, :158-164; products and long division, :110-143) and of
starks/multivariate_polynomial.py (dict monomial -> coefficient, __call__ :329-338).  Products
and divisions run on the device (stk_poly_mul, stk_poly_divmod); the rest is host-side glue."""
import functools
import itertools

from .engine import default_engine
from .limbs import ints_to_limbs, limbs_to_ints
from .modp import element_to_int


def _upload(eng, coeffs):
  buf = eng.alloc(max(len(coeffs), 1) * 32)
  if coeffs:
    buf.upload(ints_to_limbs(element_to_int(x) for x in coeffs))
  return buf


@functools.lru_cache(maxsize=None)
def polynomials_over(ring):
  class Polynomial(object):
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
      acc = ring(0)
      for c in reversed(self.coefficients):
        acc = acc * x + c
      return acc

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
    y = self.field(0)
    for k in sorted(self.coefficients):
      prod = self.field(1)
      for i, power in enumerate(k):
        prod = prod * vals[i]**power
      y = y + self.coefficients[k] * prod
    return y


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
