"""CPU tests of the host-side logic above the C ABI (no GPU): value types, limb conversions,
Fiat-Shamir helpers, Merkle index arithmetic and the verifier -- exercised on proofs made by
the CPU oracle."""
import hashlib

import numpy as np
import pytest

from conftest import load_golden

P = 2**256 - 351 * 2**32 + 1


def test_limbs_roundtrip():
  from starks_b200.limbs import ints_to_limbs, limbs_to_ints, limbs_to_be_bytes, be_bytes_to_limbs, int_to_limbs
  vals = [0, 1, P - 1, 2**255 + 12345, 0xdeadbeef << 100]
  L = ints_to_limbs(vals)
  assert L.shape == (5, 8) and limbs_to_ints(L) == vals
  be = limbs_to_be_bytes(L)
  assert [be[i].tobytes() for i in range(5)] == [v.to_bytes(32, "big") for v in vals]
  assert (be_bytes_to_limbs(be) == L).all()
  assert (int_to_limbs(P) == np.array([1, 0xFFFFFEA1] + [0xFFFFFFFF] * 6, dtype=np.uint32)).all()


def test_modp_mirror():
  from starks_b200.modp import IntegersModP
  F = IntegersModP(P)
  assert IntegersModP(P) is F
  a, b = F(2)**256, F(7)
  assert int(a) == 351 * 2**32 - 1                      # starks/test/test_modpy.py:28-35
  e = (P - 1) // 2
  assert int(b**e) == pow(7, e, P) == P - 1            # :54-61
  assert int(a * b + 1 - b) == (int(a) * 7 + 1 - 7) % P
  assert int((a / b) * b) == int(a) and int(b.inverse() * b) == 1
  assert F(b"\xff" * 32).n == 2**256 - 1                # bytes ctor does not reduce (modp.py:33-34)
  assert b.to_bytes() == (7).to_bytes(32, "big") and isinstance(a + 1, F) and (1 + a) == (a + 1)
  with pytest.raises(TypeError):
    F("x")


def test_polynomial_mirrors():
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over, generate_Xi_s, monomials_of
  F = IntegersModP(31)
  poly = polynomials_over(F).factory([0, 1, 2, 3, 0, 0])
  assert [int(c) for c in poly.coefficients] == [0, 1, 2, 3] and poly.degree() == 3
  assert int(poly(F(2))) == (2 + 8 + 24) % 31
  assert polynomials_over(F).factory([0, 0]).coefficients == []
  X = generate_Xi_s(F, 2)
  sp = X[0] + 2 * X[1]**2
  assert monomials_of(sp, 2, 31) == [((0, 2), 2), ((1, 0), 1)] and sp.degree() == 2
  assert int(sp([F(3), F(4)])) == (3 + 2 * 16) % 31
  assert monomials_of({(1, 1): 34}, 2, 31) == [((1, 1), 3)]


def test_utils_host():
  from starks_b200.utils import multiplicative_order, get_pseudorandom_indices, is_a_power_of_2
  assert multiplicative_order(pow(3, 5, 31), 31) == 6
  assert multiplicative_order(pow(7, (P - 1) // 2**20, P), P) == 2**20
  assert multiplicative_order(1, P) == 1 and multiplicative_order(P - 1, P) == 2
  g = load_golden("field_utils.json")
  for e in g["indices"]:
    assert get_pseudorandom_indices(bytes.fromhex(e["seed"]), e["modulus"], e["count"], e["exclude"]) == e["out"]
  with pytest.raises(AssertionError):
    get_pseudorandom_indices(b"\0" * 32, 2**24, 4)
  assert is_a_power_of_2(64) and not is_a_power_of_2(48)
  from starks_b200.stark import get_pseudorandom_ks
  for e in g["ks"]:
    assert [("%064x" % k) for k in get_pseudorandom_ks(bytes.fromhex(e["root"]), e["num"])] == e["out"]
  assert get_pseudorandom_ks(b"\0" * 32, 10) is None


def test_merkle_host_helpers(oracle):
  import starks_b200.merkle_tree as mt
  assert mt.permute4(list(range(8))) == [0, 2, 4, 6, 1, 3, 5, 7]
  assert mt.permute4([1, 2, 3]) == []
  t = oracle.merkelize([x.to_bytes(32, "big") for x in range(128)])
  assert mt.verify_branch(t[1], 59, mt.mk_branch(t, 59), output_as_int=True) == 59
  with pytest.raises(AssertionError):
    mt.verify_branch(t[1], 58, mt.mk_branch(t, 59))
  assert mt.blake(b"abc").hex() == "508c5e8c327c14e2e1a72ba34eeb452f37458b209ed63a294d999b4c86675982"
  leaf = b"".join(bytes([i]) * 32 for i in range(6))
  assert mt.unpack_merkle_leaf(leaf, 2, 3) == [bytes([i]) * 32 for i in range(6)]


def test_verifier_accepts_oracle_proofs_and_rejects_tampering(oracle):
  """STARK.verify_proof / FRI.verify_proximity_proof (host mirrors of stark.py:281-372,
  fri.py:268-366) on proofs produced by the CPU oracle."""
  from starks_b200.modp import IntegersModP
  from starks_b200.stark import STARK
  from starks_b200.fri import FRI
  F = IntegersModP(P)
  sp = [{(0, 1): 1}, {(1, 0): 1, (0, 2): 2}]
  steps = 64
  witness = oracle.computational_trace(P, [2, 5], steps, sp)
  boundary = [(0, 0, 2), (0, 1, 5)]
  proof = oracle.StarkOracle(steps, 8, 2, sp).mk_proof(witness, boundary)
  S = STARK(F, steps, 8, 2, sp)
  assert S.get_degree() == 2
  assert S.verify_proof(proof, witness, boundary)
  bad = [proof[0], proof[1], list(proof[2]), proof[3]]
  leaf = bytearray(bad[2][0][0]); leaf[40] ^= 1
  bad[2][0] = [bytes(leaf)] + list(bad[2][0][1:])
  with pytest.raises(AssertionError):
    S.verify_proof(bad, witness, boundary)
  # FRI alone
  n, deg = 1 << 10, 128
  w = pow(7, (P - 1) // n, P)
  f = [oracle.synth(9, i) for i in range(deg)]
  prf = oracle.fri_prove(P, f, w, deg, exclude_multiples_of=8)
  root = oracle.merkelize(oracle.fft_1d(P, f, w, order=n))[1]
  assert FRI(F).verify_proximity_proof(prf, root, F(w), deg, exclude_multiples_of=8)
  with pytest.raises(AssertionError):
    FRI(F).verify_proximity_proof(prf, b"\1" * 32, F(w), deg, exclude_multiples_of=8)


# A stand-in for the upstream `starks` package: the module attributes install() replaces, `from x
# import y` aliases of them in starks.fri and starks.stark (as in stark.py:4-17, fri.py:6-8,17), and
# the FRI class present as oracle/pyref.py restores it.  Bodies are irrelevant: nothing is called.
_UPSTREAM_STAND_IN = {
    "__init__": "",
    "fft": ("def fft_1d(field, vals, modulus, root_of_unity, inv=False): raise NotImplementedError\n"
            "def mul_polys(a, b, root_of_unity): raise NotImplementedError\n"
            "class NonBinaryFFT(object): pass\n"),
    "merkle_tree": ("def merkelize(L): raise NotImplementedError\n"
                    "def merkelize_polynomial_evaluations(dims, polynomial_evals): raise NotImplementedError\n"),
    "utils": "def get_power_cycle(r, field): raise NotImplementedError\n",
    "fri": ("from starks.merkle_tree import merkelize\n"
            "class SmoothSubgroupFRI(object): pass\n"
            "FRI = SmoothSubgroupFRI\n"),
    "stark": ("from starks.merkle_tree import merkelize\n"
              "from starks.fri import FRI\n"
              "from starks.utils import get_power_cycle\n"
              "class STARK(object):\n"
              "  def mk_proof(self, witness, boundary): raise NotImplementedError\n"),
}


def test_install_rebinds_reference_when_present(tmp_path, monkeypatch):
  """install() rebinds the upstream hot-path names and their aliases; uninstall() puts every one
  back.  Runs on a stand-in package with the upstream module surface (the upstream source is not
  part of this repository), so it needs neither the reference tree nor a GPU."""
  import sys
  pkg = tmp_path / "starks"
  pkg.mkdir()
  for name, src in _UPSTREAM_STAND_IN.items():
    (pkg / (name + ".py")).write_text(src)
  for m in [m for m in sys.modules if m == "starks" or m.startswith("starks.")]:
    monkeypatch.delitem(sys.modules, m)     # a reference loaded by another test comes back afterwards
  monkeypatch.syspath_prepend(str(tmp_path))
  try:
    _install_rebinds_and_restores()
  finally:
    for m in [m for m in sys.modules if m == "starks" or m.startswith("starks.")]:
      del sys.modules[m]


def _install_rebinds_and_restores():
  import sys
  import starks.stark, starks.fft, starks.merkle_tree, starks.fri
  before = {m: dict(vars(sys.modules[m])) for m in ("starks.fft", "starks.merkle_tree", "starks.fri", "starks.stark", "starks.utils")}
  saved_mk = starks.stark.STARK.mk_proof
  import starks_b200.install as shim
  import starks_b200.fft as bfft, starks_b200.merkle_tree as bmt, starks_b200.fri as bfri
  import starks_b200.utils as butils
  try:
    assert shim.install()
    assert starks.fft.fft_1d is bfft.fft_1d and starks.merkle_tree.merkelize is bmt.merkelize
    assert starks.stark.merkelize is bmt.merkelize and starks.stark.FRI is bfri.FRI
    assert starks.fri.merkelize is bmt.merkelize and starks.fri.SmoothSubgroupFRI is bfri.SmoothSubgroupFRI
    assert starks.utils.get_power_cycle is butils.get_power_cycle
    assert starks.stark.get_power_cycle is butils.get_power_cycle
    assert starks.stark.STARK.mk_proof is not saved_mk
    # function-level mode: the upstream prover body stays, only its callees are rebound
    assert shim.install(replace_prover=False)
    assert starks.stark.STARK.mk_proof is saved_mk and starks.stark.merkelize is bmt.merkelize
  finally:
    shim.uninstall()
  assert not shim.installed()
  assert starks.stark.STARK.mk_proof is saved_mk
  for m, d in before.items():
    now = vars(sys.modules[m])
    for k, v in d.items():
      assert now.get(k) is v, (m, k)


def test_compression_mirror(oracle):
  """starks/compression.py mirror vs values produced by the reference's own functions
  (tests/golden/compression.json) on oracle-made proofs; round trips as upstream asserts."""
  from starks_b200.compression import (compress_fri, decompress_fri, compress_branches, decompress_branches,
                                       bin_length)
  g = load_golden("compression.json")
  n, deg = 1 << 10, 128
  w = pow(7, (P - 1) // n, P)
  prf = oracle.fri_prove(P, [oracle.synth(9, i) for i in range(deg)], w, deg, exclude_multiples_of=8)
  c = compress_fri(prf)
  e = g["fri_2^10"]
  assert (len(c), bin_length(c), hashlib.blake2s(b"|".join(c)).hexdigest()) == (e["n_objects"], e["bin_length"], e["digest"])
  assert decompress_fri(c) == prf and bin_length(c) > 0          # test_compression.py:18-42
  sp = [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}]
  wit = oracle.computational_trace(P, [0, 1], 32, sp)
  proof = oracle.StarkOracle(32, 8, 2, sp).mk_proof(wit, [(0, 0, 0), (0, 1, 1)])
  cb = compress_branches(proof[2])
  e = g["stark_fib32_branches"]
  assert (len(cb), bin_length(cb), hashlib.blake2s(b"|".join(cb)).hexdigest()) == (e["n_objects"], e["bin_length"], e["digest"])
  assert decompress_branches(cb) == proof[2]


def test_verifier_closed_forms_equal_lagrange_interpolation():
  """The FRI verifier's fold check and final-layer check use closed forms; both must equal the
  literal interpolation (multi_interp_4 / lagrange_interp + evaluation, starks/poly_utils.py:337-440)."""
  import random
  from starks_b200.fri import _fold4_eval, _interp_weights, _lagrange_eval, _weighted_eval
  P = 2**256 - 351 * 2**32 + 1
  rnd = random.Random(5)
  for p, g, sizes in ((P, 7, (16, 4096, 1 << 23)), (97, 5, (4, 8, 32))):
    for n in sizes:
      root = pow(g, (p - 1) // n, p)
      quartic = [pow(root, n * j // 4, p) for j in range(4)]
      for _ in range(10):
        y = rnd.randrange(n // 4)
        x1 = pow(root, y, p)
        xs = [quartic[j] * x1 % p for j in range(4)]
        row = [rnd.randrange(p) for _ in range(4)]
        sx = rnd.randrange(2**256)   # fri.py:229: the challenge is not reduced
        t = sx * pow(root, n - y, p) % p
        assert _fold4_eval(row, t, quartic[3], pow(4, -1, p), p) == _lagrange_eval(xs, row, sx, p)
  xs = rnd.sample(range(1, 97), 16)
  ys = [rnd.randrange(97) for _ in range(16)]
  ws = _interp_weights(xs, 97)
  for x in range(97):
    assert _weighted_eval(xs, ws, ys, x, 97) == _lagrange_eval(xs, ys, x, 97)


def test_opened_value_checker_accepts_oracle_proofs(oracle):
  """tests/proofcheck.py (used on the GPU at 2^20 steps) against oracle-made proofs: it accepts
  them, and it notices a wrong linear combination -- which upstream's verifier would not
  (starks/stark.py:374-381 is commented out)."""
  from proofcheck import check_opened_values
  import numpy as np
  for steps, inp, sp in ((256, [0, 1], [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}]),
                         (64, [2, 3], [{(0, 1): 1}, {(1, 0): 1, (0, 2): 1}])):
    wit = oracle.computational_trace(P, inp, steps, sp)
    proof = oracle.StarkOracle(steps, 8, 2, sp).mk_proof(wit, [(0, 0, inp[0]), (0, 1, inp[1])])
    limbs = np.stack([oracle.to_limbs(col) for col in wit])
    assert check_opened_values(oracle, proof, limbs, inp, steps, 8, sp) == 80
  # a proof whose l-tree opens something else at one position
  bad = [proof[0], proof[1], [list(b) for b in proof[2]], proof[3]]
  other = proof[2][5]
  bad[2][2] = list(other)
  with pytest.raises(AssertionError):
    check_opened_values(oracle, bad, limbs, inp, steps, 8, sp)
