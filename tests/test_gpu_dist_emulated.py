"""The multi-GPU kernels under the single-GPU `-m gpu` run: G ranks are emulated one after
another on cuda:0 (no kernel waits on another), the all-to-all is a host-side regrouping of
the ranks' buffers.  Checks stk_ntt_dist_phase (four-step NTT) and the sharded Merkle commit
geometry against the single-GPU transform / tree.  The NCCL path itself is exercised by
tools/gpu_dist_check.py under torchrun (profiles/r01_dist_*gpu.txt) and the index logic by
tests/test_dist_gloo.py on CPU."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

P = 2**256 - 351 * 2**32 + 1


@pytest.fixture(scope="module")
def eng():
  from starks_b200 import Engine
  e = Engine(0)
  yield e
  e.close()


def rand(n, seed):
  rng = np.random.default_rng(seed)
  a = rng.integers(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
  a[:, 7] &= 0x7FFFFFFF
  return a


@pytest.mark.parametrize("world,logn", [(2, 6), (2, 13), (4, 14), (8, 12), (8, 21), (4, 22)])
@pytest.mark.parametrize("inverse", [False, True])
def test_four_step_emulated(eng, world, logn, inverse):
  n = 1 << logn
  L = n // world
  g = world.bit_length() - 1
  w = pow(7, (P - 1) // n, P)
  x = rand(n, logn * 10 + world)
  ref = eng.ntt_host(x.reshape(1, n, 8), n, w, inverse=inverse)[0]
  d_a, d_b = eng.alloc(L * 32), eng.alloc(L * 32)
  # phase 0 on every rank's cyclic shard
  y = []
  for r in range(world):
    d_a.upload(np.ascontiguousarray(x[r::world]))
    eng.ntt_dist_phase(0, d_a.ptr, d_a.ptr, L, 1, L, w, world, r, inverse)
    y.append(d_a.download((L, 8)))
  # all-to-all of contiguous chunks + local [r][m] -> [m][r] transpose
  chunk = L // world
  out = np.empty((n, 8), dtype=np.uint32)
  for rp in range(world):
    recv = np.stack([y[r][rp * chunk:(rp + 1) * chunk] for r in range(world)])      # [r][m_local]
    z = np.ascontiguousarray(recv.transpose(1, 0, 2)).reshape(L, 8)                   # [m_local][r]
    d_a.upload(z)
    eng.ntt_dist_phase(1, d_a.ptr, d_b.ptr, L, 1, L, w, world, rp, inverse)
    res = d_b.download((L, 8))
    rho = int(format(rp, "0%db" % g)[::-1], 2)
    out[rho::world] = res                                                             # X[K], K mod G = bitrev(r')
  assert (out == ref).all()
  d_a.free()
  d_b.free()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_commit_emulated(eng, world):
  """Each emulated rank commits the rows pack_rows_for_leaf_owners gives it; its nodes must be
  the global tree's subtree G + r and the combined top levels must give the global root."""
  import torch
  from starks_b200.dist import pack_rows_for_leaf_owners, combine_subtree_roots
  n, ncols = 1 << 12, 8
  rng = np.random.default_rng(world)
  cols = rng.integers(0, 2**32, size=(ncols, n, 8), dtype=np.uint64).astype(np.uint32)
  cols[:, :, 7] &= 0x7FFFFFFF
  d = eng.alloc(cols.nbytes).upload(cols)
  nodes = eng.alloc(32 * n)
  root = eng.merkle_commit(d.ptr, n, ncols, n, nodes.ptr)
  full = nodes.download((n, 32), np.uint8)
  cl = ncols // world
  packed = [pack_rows_for_leaf_owners(torch.from_numpy(cols[s * cl:(s + 1) * cl].view(np.int32).copy()), world)
            for s in range(world)]
  roots = []
  n_local = n // world
  for r in range(world):
    rows = torch.cat([packed[s][r] for s in range(world)], dim=0).numpy().view(np.uint32)   # (ncols, n/G, 8)
    dr = eng.alloc(rows.nbytes).upload(np.ascontiguousarray(rows))
    ln = eng.alloc(32 * n_local)
    roots.append(eng.merkle_commit(dr.ptr, n_local, ncols, n_local, ln.ptr))
    loc = ln.download((n_local, 32), np.uint8)
    for i in (1, 2, 3, n_local // 2, n_local - 1):
      dd = i.bit_length() - 1
      gi = (world + r) * (1 << dd) + (i - (1 << dd))
      assert (loc[i] == full[gi]).all()
    dr.free()
    ln.free()
  top = combine_subtree_roots(roots)
  assert top[1] == root
  for i in range(1, 2 * world):
    assert top[i] == full[i].tobytes()


@pytest.mark.parametrize("world,logn", [(2, 9), (4, 14), (8, 16), (8, 21)])
def test_four_step_fused_exchange_emulated(eng, world, logn):
  """stk_ntt_dist_phase0_p2p: the last pass of phase 0 scatters into the ranks' exchange
  buffers (here G buffers on one GPU stand in for the peers), phase 2 reads that layout."""
  n = 1 << logn
  L = n // world
  g = world.bit_length() - 1
  w = pow(7, (P - 1) // n, P)
  x = rand(n, 77 + logn)
  ref = eng.ntt_host(x.reshape(1, n, 8), n, w)[0]
  recv = [eng.alloc(L * 32) for _ in range(world)]
  work, outb = eng.alloc(L * 32), eng.alloc(L * 32)
  for r in range(world):
    work.upload(np.ascontiguousarray(x[r::world]))
    eng.ntt_dist_phase0_p2p(work.ptr, L, w, world, r, [b.ptr for b in recv])
  out = np.empty((n, 8), dtype=np.uint32)
  for rp in range(world):
    eng.ntt_dist_phase(2, recv[rp].ptr, outb.ptr, L, 1, L, w, world, rp)
    rho = int(format(rp, "0%db" % g)[::-1], 2)
    out[rho::world] = outb.download((L, 8))
  assert (out == ref).all()
  for b in recv + [work, outb]:
    b.free()


@pytest.mark.parametrize("world,logsteps,ncols", [(2, 9, 4), (4, 10, 8), (8, 12, 8)])
def test_lde_with_fused_leaf_exchange_emulated(eng, world, logsteps, ncols):
  """stk_lde_p2p: every emulated rank's LDE scatters its rows into the owners' buffers (G
  buffers on one GPU); each owner's subtree must be the single-GPU tree's subtree G + r."""
  from starks_b200.dist import combine_subtree_roots
  steps, ext = 1 << logsteps, 8
  n = steps * ext
  g2 = pow(7, (P - 1) // n, P)
  rng = np.random.default_rng(world + logsteps)
  trace = rng.integers(0, 2**32, size=(ncols, steps, 8), dtype=np.uint64).astype(np.uint32)
  trace[:, :, 7] &= 0x7FFFFFFF
  d_tr = eng.alloc(trace.nbytes).upload(trace)
  d_ev = eng.alloc(ncols * n * 32)
  nodes = eng.alloc(32 * n)
  root = eng.lde_commit(d_tr.ptr, steps, steps, ext, ncols, g2, d_ev.ptr, n, nodes.ptr)
  full = nodes.download((n, 32), np.uint8)
  n_local, cl = n // world, ncols // world
  bufs = [eng.alloc(ncols * n_local * 32) for _ in range(world)]
  for r in range(world):
    eng.lde_p2p(d_tr.at(r * cl * steps * 32), steps, steps, ext, cl, g2, world, r * cl, [b.ptr for b in bufs])
  roots = []
  ln = eng.alloc(32 * n_local)
  for r in range(world):
    roots.append(eng.merkle_commit(bufs[r].ptr, n_local, ncols, n_local, ln.ptr))
    loc = ln.download((n_local, 32), np.uint8)
    for i in (1, 2, n_local // 2 + 1, n_local - 1):
      dd = i.bit_length() - 1
      gi = (world + r) * (1 << dd) + (i - (1 << dd))
      assert (loc[i] == full[gi]).all(), (r, i)
  assert combine_subtree_roots(roots)[1] == root


@pytest.mark.parametrize("world,logsteps,air", [(2, 9, "fib"), (4, 10, "fib"), (8, 11, "fib"), (4, 9, "quad"),
                                                (8, 9, "w4")])
def test_sharded_prover_emulated(oracle, world, logsteps, air):
  """dist.ShardedProver -- ONE proof over G ranks (BASELINE config 5 "on 8 x B200") -- with the
  ranks emulated as G threads on cuda:0 (dist.ThreadComm: every exchange is a host-side barrier
  after a stream synchronisation): column-sharded evaluation of P, D, B with the row scatter of
  stk_ntt_p2p (uneven splits: 6 columns over 8 ranks), subtrees + replicated top levels, the
  linear combination and FRI layer 0 on leaf ranges, branches cut by their owners.  The proof
  must be the one-GPU proof, object for object; the NCCL / symmetric-memory plumbing of the same
  class runs in tests/test_gpu_multi.py."""
  import threading
  import torch
  from starks_b200 import Engine
  from starks_b200.dist import ShardedProver, ThreadComm
  from starks_b200.modp import IntegersModP
  from starks_b200.stark import STARK
  steps = 1 << logsteps
  F = IntegersModP(P)
  if air == "fib":
    width, sp, inp = 2, [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}], [0, 1]
  elif air == "quad":
    width, sp, inp = 2, [{(0, 1): 1}, {(1, 0): 1, (0, 2): 2}], [2, 5]
  else:
    width, inp = 4, [1, 2, 3, 4]
    sp = [{(0, 1, 0, 0): 1}, {(0, 0, 1, 1): 1}, {(2, 1, 0, 0): 1, (0, 0, 0, 1): 1}, {(1, 0, 0, 0): 1, (0, 1, 1, 0): 3}]
  wit = oracle.computational_trace(P, inp, steps, sp)
  bnd = [(0, j, inp[j]) for j in range(width)]
  e0 = Engine(0)
  want = STARK(F, steps, 8, width, sp, engine=e0).mk_proof(wit, bnd)
  e0.close()
  dev = torch.device("cuda", 0)
  shared = ThreadComm.Shared(world)
  results, errors = [None] * world, []

  def run(r):
    try:
      torch.cuda.set_device(0)
      eng = Engine(0)
      prover = ShardedProver(eng, F, steps, 8, width, sp, dev, comm=ThreadComm(shared, r, dev))
      first = prover.mk_proof(wit, bnd)
      results[r] = prover.mk_proof(wit, bnd)     # second proof: the row buffers are reused
      assert first == results[r]
      eng.close()
    except BaseException as ex:  # noqa: BLE001
      errors.append((r, repr(ex)))
      shared.bar.abort()

  threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
  for t in threads:
    t.start()
  for t in threads:
    t.join(timeout=600)
  assert not errors, errors
  assert results[0] == want, "sharded proof differs from the one-GPU proof"
  assert all(x is None for x in results[1:])


@pytest.mark.parametrize("world", [2, 8])
def test_sharded_prover_rejects_noncanonical_limbs_emulated(oracle, world):
  """Limbs >= p are not field elements: every rank of the sharded prover refuses them with the
  error STARK.mk_proof raises, whether it derives D rows (whose divisibility check would fail
  first), only P or B rows, or none (8 ranks, 6 rows)."""
  import threading
  import torch
  from starks_b200 import Engine
  from starks_b200.dist import ShardedProver, ThreadComm
  from starks_b200.limbs import ints_to_limbs
  from starks_b200.modp import IntegersModP
  steps, width, sp, inp = 1 << 9, 2, [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}], [0, 1]
  bad = np.stack([ints_to_limbs(col) for col in oracle.computational_trace(P, inp, steps, sp)])
  bad[1, 5] = np.array([0xFFFFFFFF] * 8, dtype=np.uint32)
  bnd = [(0, j, inp[j]) for j in range(width)]
  dev = torch.device("cuda", 0)
  shared = ThreadComm.Shared(world)
  outcome = [None] * world

  def run(r):
    try:
      torch.cuda.set_device(0)
      eng = Engine(0)
      prover = ShardedProver(eng, IntegersModP(P), steps, 8, width, sp, dev, comm=ThreadComm(shared, r, dev))
      try:
        prover.mk_proof(bad, bnd)
        outcome[r] = "returned"
      except ValueError as ex:
        outcome[r] = str(ex)
      eng.close()
    except BaseException as ex:  # noqa: BLE001
      outcome[r] = repr(ex)
      shared.bar.abort()

  threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
  for t in threads:
    t.start()
  for t in threads:
    t.join(timeout=600)
  assert outcome == ["witness holds elements >= p; reduce them mod p first"] * world, outcome
