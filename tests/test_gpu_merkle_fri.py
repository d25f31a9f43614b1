"""GPU parity: Merkle commitment (column and raw leaves), branches, LDE + commit and the
FRI fold vs the CPU oracle and the golden vectors.  Bit-exact."""
import hashlib

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

P = 2**256 - 351 * 2**32 + 1


@pytest.fixture(scope="module")
def eng():
  from starks_b200 import Engine
  e = Engine(0)
  yield e
  e.close()


def H(ints):
  return hashlib.blake2s(b"".join(x.to_bytes(32, "big") for x in ints)).hexdigest()


def rand_cols(rng, ncols, n):
  a = rng.integers(0, 2**32, size=(ncols, n, 8), dtype=np.uint64).astype(np.uint32)
  a[:, :, 7] &= 0x7FFFFFFF
  return a


def _leaves(entry):
  n, ll = entry["n"], entry["leaf_len"]
  if entry["leaves_rule"] == "range":
    return [x.to_bytes(32, "big") for x in range(n)]
  return [bytes(hashlib.blake2s(b"%d-%d-%d" % (n, i, k)).digest()[0] for k in range(ll)) for i in range(n)]


def test_raw_trees_golden(eng, oracle):
  for e in load_golden("merkle.json")["trees"]:
    L = _leaves(e)
    n, ll = e["n"], e["leaf_len"]
    np_ = 4 * (n // 4)
    if np_ == 0:
      with pytest.raises(ValueError):
        d = eng.alloc(n * ll); nodes = eng.alloc(32)
        eng.merkle_commit_raw(d.ptr, n, ll, nodes.ptr)
      continue
    d = eng.alloc(n * ll)
    d.upload(np.frombuffer(b"".join(L), dtype=np.uint8))
    nodes = eng.alloc(32 * np_)
    root = eng.merkle_commit_raw(d.ptr, n, ll, nodes.ptr)
    assert root.hex() == e["root"], e["tag"]
    got_nodes = nodes.download((np_, 32), np.uint8)
    want = oracle.merkelize(L)
    assert [got_nodes[i].tobytes() for i in range(1, np_)] == want[1:np_], e["tag"]


@pytest.mark.parametrize("n,ncols", [(4, 1), (8, 1), (64, 1), (1024, 1), (4096, 1), (2048, 2), (256, 3), (512, 6), (128, 64), (1 << 15, 5)])
def test_column_trees_match_oracle(eng, oracle, n, ncols):
  rng = np.random.default_rng(n * 131 + ncols)
  cols = rand_cols(rng, ncols, n)
  d = eng.alloc(cols.nbytes).upload(cols)
  nodes = eng.alloc(32 * n)
  root = eng.merkle_commit(d.ptr, n, ncols, n, nodes.ptr)
  leaves = oracle.pack_leaves([oracle.from_limbs(c) for c in cols]) if n <= 4096 else None
  if leaves is None:
    from starks_b200.limbs import limbs_to_be_bytes
    leaves = np.concatenate([limbs_to_be_bytes(c) for c in cols], axis=1)
  perm, want_nodes = oracle.merkelize_bytes(leaves, 4)
  got = nodes.download((n, 32), np.uint8)
  assert (got[1:] == want_nodes[1:]).all()
  assert root == want_nodes[1].tobytes()
  # branches
  tree = [b""] + [want_nodes[i].tobytes() for i in range(1, n)] + [perm[i].tobytes() for i in range(n)]
  idx = sorted(set([0, 1, n // 4, n // 2 + 1, n - 1, (n * 3) // 7]))
  got_br = eng.merkle_paths(d.ptr, n, ncols, n, nodes.ptr, idx)
  for i, br in zip(idx, got_br):
    assert br == oracle.mk_branch(tree, i), (n, ncols, i)
    if n >= 8:
      assert oracle.verify_branch(root, i, br) == perm[oracle.get_index_in_permuted(i, n)].tobytes()
  with pytest.raises(IndexError):
    eng.merkle_paths(d.ptr, n, ncols, n, nodes.ptr, [n])


def test_golden_fft_roots_and_lde_commit(eng, oracle):
  g = load_golden("fft.json")
  for s in g["synth"]:
    n = 1 << s["logn"]
    if n < 8:
      continue
    cols = oracle.to_limbs([oracle.synth(0, i) for i in range(n)]).reshape(1, n, 8)
    ev = eng.ntt_host(cols, n, int(s["w"], 16))
    d = eng.alloc(ev.nbytes).upload(ev)
    nodes = eng.alloc(32 * n)
    assert eng.merkle_commit(d.ptr, n, 1, n, nodes.ptr).hex() == s["root"]
  e = load_golden("merkle.json")["lde_commit"]
  steps, ext, ncols = e["steps"], e["ext"], e["cols"]
  N = steps * ext
  G2 = pow(7, (P - 1) // N, P)
  trace = np.stack([oracle.to_limbs([oracle.synth(c, i) for i in range(steps)]) for c in range(ncols)])
  d_tr = eng.alloc(trace.nbytes).upload(trace)
  d_ev = eng.alloc(ncols * N * 32)
  nodes = eng.alloc(32 * N)
  root = eng.lde_commit(d_tr.ptr, steps, steps, ext, ncols, G2, d_ev.ptr, N, nodes.ptr)
  assert root.hex() == e["root"]
  evs = d_ev.download((ncols, N, 8))
  for c in range(ncols):
    assert H(oracle.from_limbs(evs[c])) == e["H_cols"][c]
    assert (evs[c, ::ext] == trace[c]).all()
  br = eng.merkle_paths(d_ev.ptr, N, ncols, N, nodes.ptr, [5])[0]
  assert [b.hex() for b in br] == e["branch5"]


def test_lde_commit_larger_vs_oracle(eng, oracle):
  steps, ext, ncols = 1 << 12, 8, 6
  N = steps * ext
  G2 = pow(7, (P - 1) // N, P)
  G1 = pow(G2, ext, P)
  rng = np.random.default_rng(5)
  trace = rand_cols(rng, ncols, steps)
  d_tr = eng.alloc(trace.nbytes).upload(trace)
  d_ev = eng.alloc(ncols * N * 32)
  nodes = eng.alloc(32 * N)
  root = eng.lde_commit(d_tr.ptr, steps, steps, ext, ncols, G2, d_ev.ptr, N, nodes.ptr)
  coef = oracle.fft_limbs(P, G1, trace, steps, inv=True, nthreads=4)
  want = oracle.fft_limbs(P, G2, coef, N, nthreads=4)
  assert (d_ev.download((ncols, N, 8)) == want).all()
  from starks_b200.limbs import limbs_to_be_bytes
  leaves = np.concatenate([limbs_to_be_bytes(c) for c in want], axis=1)
  _, want_nodes = oracle.merkelize_bytes(leaves, 4)
  assert root == want_nodes[1].tobytes()


def test_fri_fold(eng, oracle):
  g = load_golden("fri.json")["fold64"]
  n = g["n"]
  vals = oracle.to_limbs([oracle.synth(g["col"], i) for i in range(n)])
  d = eng.alloc(vals.nbytes).upload(vals)
  o = eng.alloc(n // 4 * 32)
  eng.fri_fold4(d.ptr, n, int(g["root"], 16), int(g["special_x"], 16), o.ptr)
  assert [("%064x" % c) for c in oracle.from_limbs(o.download((n // 4, 8)))] == g["column"]
  rng = np.random.default_rng(11)
  for logn in (2, 3, 5, 8, 12, 14):
    n = 1 << logn
    w = pow(7, (P - 1) // n, P)
    vals = rand_cols(rng, 1, n)[0]
    sx = int.from_bytes(rng.bytes(32), "big")  # may exceed p, like field(m[1]) in fri.py:229
    if logn == 3:
      sx = P + 5
    d = eng.alloc(vals.nbytes).upload(vals)
    o = eng.alloc(max(n // 4, 1) * 32)
    eng.fri_fold4(d.ptr, n, w, sx, o.ptr)
    want = oracle.fri_fold(P, w, oracle.from_limbs(vals), sx)
    assert oracle.from_limbs(o.download((n // 4, 8))) == want, logn
  with pytest.raises(ValueError):
    eng.fri_fold4(d.ptr, 6, w, 1, o.ptr)


def test_full_size_commit_properties(eng, oracle):
  """BASELINE config 3 shape at reduced column count (the oracle cannot hash 4 GiB in
  seconds): 2^21 rows x 8 columns.  Checks: root recomputed from a branch (verify_branch),
  leaf bytes equal the big-endian values, and the root changes when one value changes."""
  from starks_b200.limbs import limbs_to_be_bytes
  n, ncols = 1 << 21, 8
  rng = np.random.default_rng(21)
  cols = rand_cols(rng, ncols, n)
  d = eng.alloc(cols.nbytes).upload(cols)
  nodes = eng.alloc(32 * n)
  root = eng.merkle_commit(d.ptr, n, ncols, n, nodes.ptr)
  idx = [0, 7, n // 4 + 3, n // 2, n - 1, 1234567]
  for i, br in zip(idx, eng.merkle_paths(d.ptr, n, ncols, n, nodes.ptr, idx)):
    leaf = oracle.verify_branch(root, i, br)
    assert leaf == b"".join(limbs_to_be_bytes(cols[c, i:i + 1]).tobytes() for c in range(ncols))
    assert len(br) == 22
  cols[3, 99, 0] ^= 1
  d.upload(cols)
  assert eng.merkle_commit(d.ptr, n, ncols, n, nodes.ptr) != root


def test_fri_driver_matches_layer_loop(eng, oracle):
  """stk_fri_prove (whole commit phase in the library) must produce the same proof object as the
  per-layer Python loop over the same kernels (starks/fri.py:189-266)."""
  from starks_b200.fri import FRI, DeviceLayer
  from starks_b200.modp import IntegersModP
  fri = FRI(IntegersModP(P), engine=eng)
  rng = np.random.default_rng(31)
  for logn, maxdeg, excl, sec, with_tree in ((6, 17, 0, 40, False), (10, 128, 8, 40, True), (13, 1024, 8, 10, False),
                                             (16, 8192, 0, 40, True), (12, 64, 4, 3, False)):
    n = 1 << logn
    w = pow(7, (P - 1) // n, P)
    vals = rand_cols(rng, 1, n)[0]
    d = eng.alloc(vals.nbytes).upload(vals)
    nodes, root = None, None
    if with_tree:
      nodes = eng.alloc(32 * n)
      root = eng.merkle_commit(d.ptr, n, 1, n, nodes.ptr)
    mk = lambda: DeviceLayer(eng, d.ptr, n, nodes.ptr if nodes else None, root)
    a = fri.prove_from_device(mk(), w, maxdeg, exclude_multiples_of=excl, security=sec, use_driver=True)
    b = fri.prove_from_device(mk(), w, maxdeg, exclude_multiples_of=excl, security=sec, use_driver=False)
    assert a == b, (logn, maxdeg, excl, sec)
    assert len(a) >= 2 and len(a[0][1]) == sec
    d.free()
    if nodes:
      nodes.free()


def test_batched_branch_verification(eng, oracle):
  """stk_verify_branches == verify_branch (starks/merkle_tree.py:71-86) on every branch, and a
  single flipped bit anywhere in a record is rejected."""
  from starks_b200.merkle_tree import verify_branch
  rng = np.random.default_rng(41)
  for logn, ncols in ((2, 1), (5, 1), (10, 6), (14, 3), (12, 64)):
    n = 1 << logn
    cols = rand_cols(rng, ncols, n)
    d = eng.alloc(cols.nbytes).upload(cols)
    nodes = eng.alloc(32 * n)
    root = eng.merkle_commit(d.ptr, n, ncols, n, nodes.ptr)
    idx = sorted(set([0, 1, n // 4, n // 2, n - 1] + [int(x) for x in rng.integers(0, n, size=20)]))
    brs = eng.merkle_paths(d.ptr, n, ncols, n, nodes.ptr, idx)
    leaves = eng.verify_branches(root, idx, brs)
    assert leaves == [verify_branch(root, i, b) for i, b in zip(idx, brs)]
    for which in range(len(brs[0])):          # flip one bit in each part of one record
      bad = [list(b) for b in brs]
      part = bytearray(bad[len(idx) // 2][which])
      part[len(part) // 2] ^= 0x10
      bad[len(idx) // 2][which] = bytes(part)
      with pytest.raises(AssertionError):
        eng.verify_branches(root, idx, bad)
    with pytest.raises(AssertionError):       # right branches, wrong positions
      eng.verify_branches(root, idx[1:] + idx[:1], brs)
    # Same committed bytes, element boundaries shifted: the packed record still hashes to the root,
    # but b[0] is no longer the committed leaf -- must be refused (the reference hashes exactly the
    # proof[0] it returns, merkle_tree.py:71-86).
    if len(idx) > 1:
      for cut in (1, 31, 32):
        bad = [list(b) for b in brs]
        b = bad[1]
        bad[1] = [b[0][:-cut], b[0][-cut:] + b[1]] + b[2:]
        with pytest.raises(AssertionError):
          eng.verify_branches(root, idx, bad)
      bad = [list(b) for b in brs]
      if len(bad[1]) > 3:
        b = bad[1]
        bad[1] = b[:2] + [b[2] + b[3][:1], b[3][1:]] + b[4:]
        with pytest.raises(AssertionError):
          eng.verify_branches(root, idx, bad)
    d.free(); nodes.free()


def test_lde_commit_from_host_trace(eng, oracle):
  """stk_lde_commit_host (upload pipelined with the transforms) == stk_lde_commit on the same
  trace: root, nodes and evaluations; ragged last column group, strided host rows."""
  rng = np.random.default_rng(77)
  for steps, ncols in ((1 << 10, 3), (1 << 14, 70), (1 << 17, 9)):
    ext = 8
    n = steps * ext
    g2 = pow(7, (P - 1) // n, P)
    pin = eng.pinned((ncols, steps, 8))
    pin.array[...] = rand_cols(rng, ncols, steps)
    d_tr = eng.alloc(pin.array.nbytes).upload(pin.array)
    ev_a, ev_b = eng.alloc(ncols * n * 32), eng.alloc(ncols * n * 32)
    no_a, no_b = eng.alloc(32 * n), eng.alloc(32 * n)
    want = eng.lde_commit(d_tr.ptr, steps, steps, ext, ncols, g2, ev_a.ptr, n, no_a.ptr)
    for rep in range(2):
      got = eng.lde_commit_host(pin.array, ext, g2, ev_b.ptr, n, no_b.ptr)
      assert got == want
    assert (no_a.download((n, 32), np.uint8)[1:] == no_b.download((n, 32), np.uint8)[1:]).all()
    for c in (0, ncols - 1):
      assert (ev_a.download((n, 8), byte_offset=c * n * 32) == ev_b.download((n, 8), byte_offset=c * n * 32)).all()
    for b in (d_tr, ev_a, ev_b, no_a, no_b):
      b.free()
    pin.free()


def test_lde_copied_coset_equals_full_transform(eng, oracle, monkeypatch):
  """With an 8x blowup evals[8K] == trace[K], so stk_lde copies that coset instead of computing it
  (NttPass::cskip0).  Same evaluations as the full transform (STK_LDE_R0=0) at single-pass, two-pass
  and three-pass sizes, with strided rows and a ragged column count; and the oracle's where cheap."""
  rng = np.random.default_rng(123)
  for logsteps, ncols in ((3, 2), (6, 5), (8, 3), (11, 9), (14, 4), (18, 3), (21, 1)):
    steps, ext = 1 << logsteps, 8
    n = steps * ext
    g2 = pow(7, (P - 1) // n, P)
    trace = rand_cols(rng, ncols, steps)
    d_tr = eng.alloc(trace.nbytes).upload(trace)
    ev_a, ev_b, co = eng.alloc(ncols * n * 32), eng.alloc(ncols * n * 32), eng.alloc(ncols * steps * 32)
    eng.lde(d_tr.ptr, steps, steps, ext, ncols, g2, ev_a.ptr, n, d_coeffs=co.ptr, coeff_stride=steps)
    monkeypatch.setenv("STK_LDE_R0", "0")
    eng.lde(d_tr.ptr, steps, steps, ext, ncols, g2, ev_b.ptr, n)
    monkeypatch.delenv("STK_LDE_R0")
    a, b = ev_a.download((ncols, n, 8)), ev_b.download((ncols, n, 8))
    assert (a == b).all(), logsteps
    assert (a[:, ::ext] == trace).all()
    if logsteps <= 14:
      coeffs = oracle.fft_limbs(P, pow(g2, ext, P), trace, steps, inv=True)
      assert (co.download((ncols, steps, 8)) == coeffs).all()
      assert (a == oracle.fft_limbs(P, g2, coeffs, n)).all()
    for x in (d_tr, ev_a, ev_b, co):
      x.free()
