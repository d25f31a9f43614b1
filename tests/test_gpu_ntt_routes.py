"""GPU parity of every route ntt_dev_on (ntt_api.cu) picks for a transform, and of stk_lde's call
shapes, element for element against the CPU oracle (fft_1d restatement).

ntt_dev_on chooses by size, padding, direction and aliasing: the plain transform (1024- or
2048-element tiles, one to three passes), the expansion round of a zero-padded forward transform,
the eight coset transforms over <w^8> (with or without the copied residue-0 coset), the padded
inverse, the in-place transform and the run-time (Montgomery) modulus.  Each case id names the
route and the plan it exercises.  Inputs are uniform over the whole field [0, p) with every limb
random, and each column starts with the values where carries and reductions turn over (0, 1, p-1,
p-2, 2^255, ...).  The cases above 2^22 are also marked `slow`: the oracle needs tens of seconds
per column there."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 2**256 - 351 * 2**32 + 1
# scalar fields of two pairing curves, as run-time moduli: (p, a quadratic non-residue)
BN254_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001      # 2-adicity 28
BLS12_381_R = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001  # 2-adicity 32
NT = max(1, min(os.cpu_count() or 1, 16))   # oracle threads (one column each)
slow = pytest.mark.slow


@pytest.fixture(scope="module")
def eng():
  from starks_b200 import Engine
  e = Engine(0)
  yield e
  e.close()


def limbs(ints):
  return np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in ints), dtype="<u4").reshape(-1, 8).copy()


def ge(a, p):
  """a >= p for every element of a (..., 8) little-endian limb array."""
  pl = limbs([p])[0]
  res = np.ones(a.shape[:-1], dtype=bool)   # all limbs equal: a == p
  open_ = np.ones(a.shape[:-1], dtype=bool)
  for i in range(7, -1, -1):
    gt, lt = a[..., i] > pl[i], a[..., i] < pl[i]
    res[open_ & lt] = False
    open_ &= ~(gt | lt)
  return res


def edge_values(p):
  b = p.bit_length()
  cand = [0, 1, p - 1, p - 2, 2**255, 2**255 - 1, 2**256 - 2**64, 2**(b - 1), 2**(b - 1) - 1]
  out = []
  for v in cand:
    if v < p and v not in out:
      out.append(v)
  return out


def full_range(rng, cols, n, p=P):
  """(cols, n, 8) uniform residues in [0, p): all eight limbs random (the top one masked to the
  bit length of p, then rejection), and edge_values(p) at the start of every column, rotated by the
  column index so that no two short columns are equal."""
  top = (1 << ((p.bit_length() - 1) % 32 + 1)) - 1
  a = np.frombuffer(rng.bytes(cols * n * 32), dtype=np.uint32).reshape(cols, n, 8).copy()
  a[..., 7] &= top
  bad = ge(a, p)
  while bad.any():
    k = int(bad.sum())
    r = np.frombuffer(rng.bytes(k * 32), dtype=np.uint32).reshape(k, 8).copy()
    r[:, 7] &= top
    a[bad] = r
    bad = ge(a, p)
  E = limbs(edge_values(p))
  k = min(len(E), n)
  idx = (np.arange(k)[None, :] + np.arange(cols)[:, None]) % len(E)
  a[:, :k] = E[idx]
  assert not ge(a, p).any()
  return a


def root(n, p=P, g=7):
  w = pow(g, (p - 1) // n, p)
  assert pow(w, n // 2, p) == p - 1
  return w


def ntt(eng, x, n, w, inverse=False):
  """Out-of-place device transform of the (cols, n_in, 8) columns in x, contiguous rows."""
  cols, n_in, _ = x.shape
  d_in = eng.alloc(max(x.nbytes, 32)).upload(x)
  d_out = eng.alloc(cols * n * 32)
  eng._check(eng.lib.stk_memset(eng.ctx, d_out.ptr, 0xA5, cols * n * 32))   # no stale results
  eng.ntt(d_in.ptr, n_in, n_in, d_out.ptr, n, n, cols, w, inverse=inverse)
  out = d_out.download((cols, n, 8))
  d_in.free()
  d_out.free()
  return out


def diff(got, want):
  """Assertion message: how many elements differ and where the first few are (column, index)."""
  bad = np.argwhere((got != want).any(-1))
  return "%d of %d elements differ, first at %s" % (len(bad), got.size // 8, bad[:4].tolist())


def pad(x, n):
  out = np.zeros((x.shape[0], n, 8), np.uint32)
  out[:, :x.shape[1]] = x
  return out


# ---------------------------------------------------------------- plain transforms (n_in = N)

PLAIN = [(17, 4, "stark-2pass"), (18, 4, "stark-2pass"), (19, 4, "stark-2pass"), (21, 4, "t11-2pass"),
         (22, 4, "t11-2pass"), (23, 1, "stark-3pass"), (25, 1, "stark-3pass")]


@pytest.mark.parametrize("logn,cols,inverse", [
    pytest.param(l, c, inv, id="%s-plain-2^%d-%s" % ("inv" if inv else "fwd", l, t), marks=[slow] if l > 22 else [])
    for l, c, t in PLAIN for inv in (False, True)])
def test_plain(eng, oracle, logn, cols, inverse):
  n = 1 << logn
  w = root(n)
  eng.set_field(P)
  x = full_range(np.random.default_rng(1000 + logn), cols, n)
  got = ntt(eng, x, n, w, inverse)
  want = oracle.fft_limbs(P, w, x, n, inv=inverse, nthreads=NT)
  assert (got == want).all(), diff(got, want)


# ------------------------------------------------- zero-padded forward (n_in <= N/8): two routes

# expansion: the long transform's first round scales-and-copies (ZS); coset: eight transforms of
# order N/8 over <w^8>, chosen where that saves a pass (zs first pass, cf final pass)
PAD_FWD = [(11, "expansion-t11-1pass"), (17, "expansion-stark-2pass"), (22, "expansion-t11-2pass"),
           (13, "coset-stark-1pass"), (14, "coset-t11-1pass"),
           (23, "coset-stark-2pass"), (24, "coset-t11-2pass"), (25, "coset-t11-2pass")]


@pytest.mark.parametrize("logn", [pytest.param(l, id="fwd-pad-2^%d-%s" % (l, t), marks=[slow] if l > 22 else [])
                                  for l, t in PAD_FWD])
def test_padded_forward(eng, oracle, logn):
  """n_in = N/8, N/8 - 1 and 5 against the oracle; above 2^22 also against the plain route run on
  the same input padded with explicit zeros (pinned to the oracle in test_plain)."""
  n = 1 << logn
  w = root(n)
  eng.set_field(P)
  cols = 2 if logn <= 22 else 1
  rng = np.random.default_rng(2000 + logn)
  xs = [full_range(rng, cols, n_in) for n_in in (n // 8, n // 8 - 1, 5)]
  gots = [ntt(eng, x, n, w) for x in xs]
  want = oracle.fft_limbs(P, w, np.concatenate([pad(x, n // 8) for x in xs]), n, nthreads=NT)
  for i, (x, got) in enumerate(zip(xs, gots)):
    assert (got == want[i * cols:(i + 1) * cols]).all(), (x.shape[1], diff(got, want[i * cols:(i + 1) * cols]))
    if logn > 22:
      plain = ntt(eng, pad(x, n), n, w)
      assert (got == plain).all(), (x.shape[1], diff(got, plain))


# ------------------------------------------------------------- zero-padded inverse (n_in <= N/8)

PAD_INV = [(8, "stark-1pass"), (11, "t11-1pass"), (16, "stark-2pass"), (21, "t11-2pass")]


@pytest.mark.parametrize("logn", [pytest.param(l, id="inv-pad-2^%d-%s" % (l, t)) for l, t in PAD_INV])
def test_padded_inverse(eng, oracle, logn):
  """The expansion round followed by the 1/N scale of the final pass."""
  n = 1 << logn
  w = root(n)
  eng.set_field(P)
  rng = np.random.default_rng(3000 + logn)
  xs = [full_range(rng, 2, n_in) for n_in in (n // 8, n // 8 - 1, 5)]
  gots = [ntt(eng, x, n, w, inverse=True) for x in xs]
  want = oracle.fft_limbs(P, w, np.concatenate([pad(x, n // 8) for x in xs]), n, inv=True, nthreads=NT)
  for i, (x, got) in enumerate(zip(xs, gots)):
    assert (got == want[2 * i:2 * i + 2]).all(), (x.shape[1], diff(got, want[2 * i:2 * i + 2]))


# --------------------------------------------------------------------- in place, padded, strided

INPLACE = [(10, "stark-1pass"), (16, "stark-2pass"), (21, "t11-2pass")]


@pytest.mark.parametrize("logn,inverse", [
    pytest.param(l, inv, id="%s-inplace-pad-2^%d-%s" % ("inv" if inv else "fwd", l, t))
    for l, t in INPLACE for inv in (False, True)])
def test_in_place_padded(eng, oracle, logn, inverse):
  """d_in == d_out with n_in = N/8 - 3 and a row stride of N + 24: rows hold other data past n_in,
  which the transform must read as zeros, and past N, which it must leave alone."""
  n = 1 << logn
  n_in, stride, cols = n // 8 - 3, n + 24, 2
  w = root(n)
  eng.set_field(P)
  x = full_range(np.random.default_rng(4000 + logn), cols, stride)
  d = eng.alloc(x.nbytes).upload(x)
  eng.ntt(d.ptr, n_in, stride, d.ptr, stride, n, cols, w, inverse=inverse)
  got = d.download((cols, stride, 8))
  d.free()
  want = oracle.fft_limbs(P, w, np.ascontiguousarray(x[:, :n_in]), n, inv=inverse, nthreads=NT)
  assert (got[:, :n] == want).all(), diff(got[:, :n], want)
  assert (got[:, n:] == x[:, n:]).all(), diff(got[:, n:], x[:, n:])


# ----------------------------------------------------------------------------------------- LDE

def lde(eng, trace, ext, g2, trace_stride=None, coeff_stride=None, eval_stride=None):
  """stk_lde with separate, optionally strided buffers -> (coefficients, evaluations)."""
  cols, steps, _ = trace.shape
  n = steps * ext
  ts, cs, es = trace_stride or steps, coeff_stride or steps, eval_stride or n
  tr = np.zeros((cols, ts, 8), np.uint32)
  tr[:, :steps] = trace
  d_tr = eng.alloc(tr.nbytes).upload(tr)
  d_co, d_ev = eng.alloc(cols * cs * 32), eng.alloc(cols * es * 32)
  eng._check(eng.lib.stk_memset(eng.ctx, d_ev.ptr, 0xA5, cols * es * 32))
  eng.lde(d_tr.ptr, steps, ts, ext, cols, g2, d_ev.ptr, es, d_coeffs=d_co.ptr, coeff_stride=cs)
  co = d_co.download((cols, cs, 8))[:, :steps]
  ev = d_ev.download((cols, es, 8))[:, :n]
  for b in (d_tr, d_co, d_ev):
    b.free()
  return co, ev


def check_lde(oracle, trace, ext, g2, co, ev):
  steps = trace.shape[1]
  want_co = oracle.fft_limbs(P, pow(g2, ext, P), trace, steps, inv=True, nthreads=NT)
  assert (co == want_co).all(), diff(co, want_co)
  want_ev = oracle.fft_limbs(P, g2, want_co, steps * ext, nthreads=NT)
  assert (ev == want_ev).all(), diff(ev, want_ev)


LDE = [(6, 2, "plain-1pass"), (6, 4, "plain-1pass"), (6, 16, "expansion-1pass"), (6, 32, "expansion-t11-1pass"),
       (14, 2, "plain-2pass"), (14, 4, "plain-2pass"), (14, 16, "expansion-2pass"), (14, 32, "expansion-2pass")]


@pytest.mark.parametrize("logsteps,ext", [pytest.param(s, e, id="lde-ext%d-2^%d-steps-%s" % (e, s, t))
                                          for s, e, t in LDE])
def test_lde_other_blowups(eng, oracle, logsteps, ext):
  """ext != 8: no residue-0 copy.  2 and 4 run the partially padded plain transform, 16 and 32 the
  expansion round.  Strided trace, coefficient and evaluation rows."""
  steps = 1 << logsteps
  n = steps * ext
  g2 = root(n)
  eng.set_field(P)
  trace = full_range(np.random.default_rng(5000 + 64 * logsteps + ext), 3, steps)
  co, ev = lde(eng, trace, ext, g2, steps + 3, steps + 1, n + 5)
  check_lde(oracle, trace, ext, g2, co, ev)


@slow
@pytest.mark.parametrize("logsteps", [pytest.param(21, id="lde-ext8-2^21-steps-coset-r0-t11-2pass")])
def test_lde_copied_coset_vs_oracle(eng, oracle, logsteps):
  """ext = 8 at N = 2^24: the coset route with the copied residue 0, whose final pass is the
  2048-tile interleaved store (t11_cf)."""
  steps, ext = 1 << logsteps, 8
  g2 = root(steps * ext)
  eng.set_field(P)
  trace = full_range(np.random.default_rng(6000 + logsteps), 1, steps)
  co, ev = lde(eng, trace, ext, g2)
  check_lde(oracle, trace, ext, g2, co, ev)


@slow
def test_lde_wider_than_a_grid_dimension(eng, oracle):
  """8200 columns of 2^12 steps: 8 * 8200 virtual coset columns exceed gridDim.y (65535), so the
  LDE falls back from the coset route to the expansion route.  Sampled columns equal their own
  single-column LDE (which takes the coset route) and, for two of them, the oracle."""
  steps, ext, cols = 1 << 12, 8, 8200
  n = steps * ext
  g2 = root(n)
  eng.set_field(P)
  trace = full_range(np.random.default_rng(7000), cols, steps)
  d_tr = eng.alloc(trace.nbytes).upload(trace)
  d_ev = eng.alloc(cols * n * 32)
  eng.lde(d_tr.ptr, steps, steps, ext, cols, g2, d_ev.ptr, n)
  d_one = eng.alloc(n * 32)
  for c in (0, 1, 4095, 8191, cols - 1):
    eng.lde(d_tr.at(c * steps * 32), steps, steps, ext, 1, g2, d_one.ptr, n)
    one = d_one.download((n, 8))
    assert (d_ev.download((n, 8), byte_offset=c * n * 32) == one).all(), c
    if c in (1, cols - 1):
      co = oracle.fft_limbs(P, pow(g2, ext, P), trace[c:c + 1], steps, inv=True)
      assert (one == oracle.fft_limbs(P, g2, co, n)[0]).all(), c
  for b in (d_tr, d_ev, d_one):
    b.free()


@pytest.mark.parametrize("logsteps,ext", [pytest.param(6, 8, id="lde-alias-ext8-2^6-steps-coset-r0-1pass"),
                                          pytest.param(12, 8, id="lde-alias-ext8-2^12-steps-coset-r0-2pass"),
                                          pytest.param(12, 4, id="lde-alias-ext4-2^12-steps-plain-2pass")])
def test_lde_coefficients_over_the_trace(eng, oracle, logsteps, ext):
  """d_coeffs == d_trace with equal strides: the inverse transform overwrites the trace with the
  coefficients, so the evaluations must not copy residue 0 from that buffer.  Same evaluations as
  with separate buffers, and the coefficients left in the trace's place.  Any other overlap of the
  two ranges is rejected."""
  steps, cols = 1 << logsteps, 3
  n = steps * ext
  stride = steps + 2
  g2 = root(n)
  eng.set_field(P)
  trace = full_range(np.random.default_rng(8000 + logsteps + ext), cols, steps)
  want_co, want_ev = lde(eng, trace, ext, g2, stride, stride)
  check_lde(oracle, trace, ext, g2, want_co, want_ev)
  tr = np.zeros((cols, stride, 8), np.uint32)
  tr[:, :steps] = trace
  d = eng.alloc(2 * tr.nbytes).upload(tr)   # room for every overlapping coefficient range below
  d_ev = eng.alloc(cols * n * 32)
  eng.lde(d.ptr, steps, stride, ext, cols, g2, d_ev.ptr, n, d_coeffs=d.ptr, coeff_stride=stride)
  ev = d_ev.download((cols, n, 8))
  bad = np.argwhere((ev != want_ev).any(-1))
  assert not len(bad), "%d evaluations differ, at residues %s mod %d" % (len(bad), sorted({int(r) for r in bad[:, 1] % ext}), ext)
  assert (d.download((cols, stride, 8))[:, :steps] == want_co).all()
  for co_ptr, cs in ((d.ptr + 32, stride), (d.ptr, stride + 1), (d.ptr + (cols - 1) * stride * 32, stride)):
    with pytest.raises(ValueError):
      eng.lde(d.ptr, steps, stride, ext, cols, g2, d_ev.ptr, n, d_coeffs=co_ptr, coeff_stride=cs)
  d.free()
  d_ev.free()


# ------------------------------------------------------------------ run-time (Montgomery) modulus

MONT_P = [("bn254", BN254_R, 5), ("bls12_381", BLS12_381_R, 7)]
MONT_N = [(3, "1pass"), (10, "1pass"), (11, "2pass"), (16, "2pass"), (21, "3pass")]


@pytest.mark.parametrize("logn", [pytest.param(l, id="2^%d-mont-%s" % (l, t)) for l, t in MONT_N])
@pytest.mark.parametrize("name,p,g", [pytest.param(*m, id=m[0]) for m in MONT_P])
def test_runtime_modulus(eng, oracle, name, p, g, logn):
  """Radix-4 Montgomery passes (1024-element tiles) over 254- and 255-bit primes, forward and
  inverse, inputs over the whole field."""
  n = 1 << logn
  w = root(n, p, g)
  cols = 4 if logn <= 16 else 2
  x = full_range(np.random.default_rng(9000 + logn + p % 1000), cols, n, p)
  try:
    eng.set_field(p)
    for inverse in (False, True):
      got = ntt(eng, x, n, w, inverse)
      want = oracle.fft_limbs(p, w, x, n, inv=inverse, nthreads=NT)
      assert (got == want).all(), (name, inverse, diff(got, want))
  finally:
    eng.set_field(P)
