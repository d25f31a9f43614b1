"""Multi-GPU plumbing on one 8 x B200 box: one process per GPU, torch.distributed (NCCL over
NVLink/NVSwitch on GPUs, gloo in the CPU tests).  Only the two steps of the path that need
an exchange use a collective (SURVEY.md section 8e); everything else shards with none.

  * ShardedCommit   LDE of a column shard + Merkle commit over ALL columns' leaves:
                    column-sharded evaluations -> (all-to-all) -> leaf-range-sharded rows,
                    one subtree per rank, all-gather of the 32-byte subtree roots, top
                    log2(G) levels replicated (merkle_tree.py:36-56 heap layout is kept:
                    rank r's subtree root is global node G + r).
  * dist_ntt        one large transform over G ranks, four-step with ONE all-to-all
                    (stk_ntt_dist_phase), cyclic in / cyclic out.

The data-movement helpers take and return torch tensors and never compute field arithmetic,
so they are exercised on CPU tensors with gloo (tests/test_dist_gloo.py); the compute hooks
are the engine's device kernels."""
from hashlib import blake2s

import numpy as np
import torch
import torch.distributed as dist


def _world(group=None):
  return dist.get_world_size(group), dist.get_rank(group)


def _adopt_stream(engine, t: torch.Tensor):
  """Run the engine's kernels on torch's current stream so that they are ordered with the
  collectives and tensor ops torch enqueues there (no host synchronisation needed)."""
  if t.is_cuda:
    handle = torch.cuda.current_stream(t.device).cuda_stream
    # torch's default stream has handle 0, which stk_set_stream reads as "the context's own
    # stream"; name the legacy default stream explicitly (cudaStreamLegacy == 1)
    engine.set_stream(handle if handle else 1)


# ---------------------------------------------------------------- leaf exchange (commit)

def pack_rows_for_leaf_owners(evals: torch.Tensor, world: int) -> torch.Tensor:
  """evals: (cols_local, N, 8) column-sharded evaluations.  Returns (world, cols_local, N/world, 8):
  block d holds, for every local column, the rows rank d needs for its N/world permuted
  leaves: rows {j*q + d*q/G + i : j < 4, i < q/G}, q = N/4, ordered (j, i) -- which is
  exactly the row order of a local tree of N/world rows under permute4
  (starks/merkle_tree.py:11-23)."""
  cl, n, limbs = evals.shape
  q = n // 4
  assert n % (4 * world) == 0
  v = evals.view(cl, 4, world, q // world, limbs)      # [c][j][d][i]
  return v.permute(2, 0, 1, 3, 4).contiguous().view(world, cl, n // world, limbs)


def exchange_leaf_rows(evals: torch.Tensor, group=None) -> torch.Tensor:
  """All-to-all of pack_rows_for_leaf_owners: returns (world*cols_local, N/world, 8), i.e. ALL
  columns (global column order: source rank major) for this rank's leaf range."""
  world, _ = _world(group)
  send = pack_rows_for_leaf_owners(evals, world)
  recv = torch.empty_like(send)
  dist.all_to_all_single(recv, send, group=group)
  cl, n_local, limbs = send.shape[1], send.shape[2], send.shape[3]
  return recv.view(world * cl, n_local, limbs)


def combine_subtree_roots(roots):
  """Top log2(G) levels of the heap from the G subtree roots (global nodes G .. 2G-1):
  node i = BLAKE2s(node 2i || node 2i+1) (merkle_tree.py:54-55).  Returns {index: digest}."""
  g = len(roots)
  assert g & (g - 1) == 0
  nodes = {g + r: bytes(roots[r]) for r in range(g)}
  for i in range(g - 1, 0, -1):
    nodes[i] = blake2s(nodes[2 * i] + nodes[2 * i + 1]).digest()
  return nodes


def allgather_roots(root: bytes, group=None, device="cpu"):
  world, _ = _world(group)
  mine = torch.tensor(list(root), dtype=torch.uint8, device=device)
  out = [torch.empty_like(mine) for _ in range(world)]
  dist.all_gather(out, mine, group=group)
  return [bytes(t.cpu().tolist()) for t in out]


def allgather_roots_from_nodes(nodes: torch.Tensor, group=None):
  """Subtree roots straight from the ranks' node buffers (node 1 of each local heap): one
  all-gather of 32 bytes per rank and ONE device-to-host copy, without the round trip through the
  host that a root returned by stk_merkle_commit would take."""
  world, _ = _world(group)
  out = torch.empty(world * 32, dtype=torch.uint8, device=nodes.device)   # flat: the shape every backend accepts
  dist.all_gather_into_tensor(out, nodes[1].contiguous(), group=group)
  host = out.cpu().numpy().reshape(world, 32)
  return [host[r].tobytes() for r in range(world)]


class ShardedCommit(object):
  """LDE + Merkle commitment with the trace columns sharded over the ranks of `group`."""

  def __init__(self, engine, group=None):
    self.eng, self.group = engine, group
    self.world, self.rank = _world(group)

  def lde_commit(self, trace: torch.Tensor, ext: int, g2: int):
    """trace: (cols_local, steps, 8) int32 CUDA tensor (this rank's columns).
    Returns (root, top_nodes, evals_local, rows_all_columns, local_nodes)."""
    import time
    cl, steps, _ = trace.shape
    n = steps * ext
    dev = trace.device
    _adopt_stream(self.eng, trace)
    marks = [("start", time.perf_counter())]
    evals = torch.empty((cl, n, 8), dtype=torch.int32, device=dev)
    marks.append(("alloc_evals", time.perf_counter()))
    self.eng.lde(trace.data_ptr(), steps, steps, ext, cl, g2, evals.data_ptr(), n)
    marks.append(("lde_enqueued", time.perf_counter()))
    if self.world == 1:
      nodes = torch.empty((n, 32), dtype=torch.uint8, device=dev)
      root = self.eng.merkle_commit(evals.data_ptr(), n, cl, n, nodes.data_ptr())
      return root, {1: root}, evals, evals, nodes
    rows = exchange_leaf_rows(evals, self.group)            # (cols_total, n/G, 8)
    marks.append(("exchange_enqueued", time.perf_counter()))
    n_local = n // self.world
    nodes = torch.empty((n_local, 32), dtype=torch.uint8, device=dev)
    sub_root = self.eng.merkle_commit(rows.data_ptr(), n_local, rows.shape[0], n_local, nodes.data_ptr())
    marks.append(("subtree_root_on_host", time.perf_counter()))
    roots = allgather_roots(sub_root, self.group, device=dev)
    marks.append(("roots_gathered", time.perf_counter()))
    top = combine_subtree_roots(roots)
    # host-side timeline of the last call (ms since entry): where the calling thread was held up
    self.timings = {name: round((t - marks[0][1]) * 1e3, 3) for name, t in marks[1:]}
    return top[1], top, evals, rows, nodes


# ---------------------------------------------------------------- four-step NTT

def block_to_cyclic(x: torch.Tensor, group=None) -> torch.Tensor:
  """x: (L, 8) block-distributed (rank s holds indices [s*L, (s+1)*L)) -> cyclic (rank r holds
  indices r + G*m).  One all-to-all."""
  world, _ = _world(group)
  L, limbs = x.shape
  send = x.view(L // world, world, limbs).permute(1, 0, 2).contiguous()   # [r][t] = x[s*L + r + G*t]
  recv = torch.empty_like(send)
  dist.all_to_all_single(recv, send, group=group)
  return recv.view(L, limbs)                                               # [s][t] -> m = s*L/G + t


def cyclic_to_block(x: torch.Tensor, group=None) -> torch.Tensor:
  """Inverse of block_to_cyclic."""
  world, _ = _world(group)
  L, limbs = x.shape
  recv = torch.empty_like(x)
  dist.all_to_all_single(recv, x.contiguous(), group=group)                # [s][t]: from rank s its chunk for me
  return recv.view(world, L // world, limbs).permute(1, 0, 2).contiguous().view(L, limbs)


def transpose_exchange(y: torch.Tensor, group=None) -> torch.Tensor:
  """The four-step transpose: rank r holds y[(m << g) | r] at position m; afterwards rank r'
  holds the contiguous global block [r'*L, (r'+1)*L), low g bits fastest."""
  world, _ = _world(group)
  L, limbs = y.shape
  recv = torch.empty_like(y)
  dist.all_to_all_single(recv, y.contiguous(), group=group)                # [r][m_local]
  return recv.view(world, L // world, limbs).permute(1, 0, 2).contiguous().view(L, limbs)


def output_owner(k: int, world: int):
  """(rank, local position) holding output index k after dist_ntt."""
  g = world.bit_length() - 1
  rho = k % world
  r = int(format(rho, "0%db" % g)[::-1], 2) if g else 0
  return r, k // world


def dist_ntt(engine, x_cyclic: torch.Tensor, root: int, inverse=False, group=None) -> torch.Tensor:
  """x_cyclic: (L, 8) int32 CUDA tensor, rank r holding x[r + G*m].  Returns (L, 8): rank r'
  holds X[K] for K mod G = bitrev(r') at position K // G (see output_owner)."""
  world, rank = _world(group)
  L = x_cyclic.shape[0]
  if world == 1:
    _adopt_stream(engine, x_cyclic)
    out = torch.empty_like(x_cyclic)
    engine.ntt(x_cyclic.data_ptr(), L, L, out.data_ptr(), L, L, 1, root, inverse=inverse)
    return out
  _adopt_stream(engine, x_cyclic)
  y = x_cyclic.clone()
  engine.ntt_dist_phase(0, y.data_ptr(), y.data_ptr(), L, 1, L, root, world, rank, inverse)
  z = transpose_exchange(y, group)
  out = torch.empty_like(z)
  engine.ntt_dist_phase(1, z.data_ptr(), out.data_ptr(), L, 1, L, root, world, rank, inverse)
  return out


class FourStepP2P(object):
  """dist_ntt with the exchange fused into the compute kernel: the last pass of phase 0 stores
  its results directly into the destination ranks' exchange buffers over NVLink (peer
  pointers from torch symmetric memory), so neither an NCCL all-to-all nor a transpose pass
  runs; two device-side barriers order the exchange.  One column of L = N/G elements per rank."""

  def __init__(self, engine, local_n: int, device, group=None):
    import torch.distributed._symmetric_memory as symm_mem
    self.eng, self.L = engine, local_n
    self.group = group if group is not None else dist.group.WORLD
    self.world, self.rank = _world(group)
    self.recv = symm_mem.empty((local_n, 8), dtype=torch.int32, device=device)
    self.hdl = symm_mem.rendezvous(self.recv, self.group)
    self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]

  def ntt(self, x_cyclic: torch.Tensor, root: int, inverse=False) -> torch.Tensor:
    _adopt_stream(self.eng, x_cyclic)
    y = x_cyclic.clone()
    self.hdl.barrier(channel=0)          # every rank is done reading its exchange buffer
    self.eng.ntt_dist_phase0_p2p(y.data_ptr(), self.L, root, self.world, self.rank, self.ptrs, inverse)
    self.hdl.barrier(channel=1)          # every rank's stores have landed
    out = torch.empty_like(x_cyclic)
    self.eng.ntt_dist_phase(2, self.recv.data_ptr(), out.data_ptr(), self.L, 1, self.L, root, self.world, self.rank,
                            inverse)
    return out


class ShardedCommitP2P(object):
  """ShardedCommit with the exchange fused into the LDE: the final pass of every rank's forward
  transform stores each evaluation row directly into the leaf owner's row buffer over NVLink
  (stk_lde_p2p), so the column-sharded evaluations never exist and no all-to-all runs."""

  def __init__(self, engine, cols_total: int, n: int, device, group=None):
    import torch.distributed._symmetric_memory as symm_mem
    self.eng, self.n, self.cols_total = engine, n, cols_total
    self.group = group if group is not None else dist.group.WORLD
    self.world, self.rank = _world(group)
    self.n_local = n // self.world
    self.rows = symm_mem.empty((cols_total, self.n_local, 8), dtype=torch.int32, device=device)
    self.hdl = symm_mem.rendezvous(self.rows, self.group)
    self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
    self.nodes = torch.empty((self.n_local, 32), dtype=torch.uint8, device=device)

  def lde_commit(self, trace: torch.Tensor, ext: int, g2: int):
    """trace: (cols_local, steps, 8) int32 CUDA tensor.  Returns (root, top_nodes); the rows of
    this rank's leaf range (all columns) stay in self.rows, its subtree nodes in self.nodes."""
    cl, steps, _ = trace.shape
    assert steps * ext == self.n and cl * self.world == self.cols_total
    _adopt_stream(self.eng, trace)
    self.hdl.barrier(channel=0)          # nobody still reads the previous commit's rows
    self.eng.lde_p2p(trace.data_ptr(), steps, steps, ext, cl, g2, self.world, self.rank * cl, self.ptrs)
    self.hdl.barrier(channel=1)          # all rows have landed
    return self._commit_rows()

  def _commit_rows(self):
    self.eng.merkle_commit(self.rows.data_ptr(), self.n_local, self.cols_total, self.n_local, self.nodes.data_ptr(),
                           want_root=False)
    top = combine_subtree_roots(allgather_roots_from_nodes(self.nodes, self.group))
    return top[1], top

  def lde_commit_host(self, h_trace: torch.Tensor, d_stage: torch.Tensor, ext: int, g2: int):
    """The same commit with this rank's columns in pinned HOST memory (h_trace: (cols_local, steps,
    8) int32 CPU tensor, d_stage: a device tensor of the same shape): columns are uploaded in
    geometrically growing groups on a side stream while the previous group is transformed and
    scattered, so only the first group's copy is exposed (the end-to-end form of the metric)."""
    cl, steps, _ = h_trace.shape
    assert steps * ext == self.n and cl * self.world == self.cols_total and d_stage.shape == h_trace.shape
    _adopt_stream(self.eng, d_stage)
    main = torch.cuda.current_stream(d_stage.device)
    if not hasattr(self, "_copy_stream"):
      self._copy_stream = torch.cuda.Stream(device=d_stage.device)
    side = self._copy_stream
    side.wait_stream(main)               # d_stage may still be read by the previous call's transforms
    groups, done, g = [], 0, max(1, cl // 8)
    while done < cl:
      nb = min(g, cl - done)
      groups.append((done, nb))
      done += nb
      g = g + (g + 1) // 2
    events = []
    with torch.cuda.stream(side):
      for c0, nb in groups:
        d_stage[c0:c0 + nb].copy_(h_trace[c0:c0 + nb], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(side)
        events.append(ev)
    self.hdl.barrier(channel=0)
    for (c0, nb), ev in zip(groups, events):
      main.wait_event(ev)
      self.eng.lde_p2p(d_stage[c0:c0 + nb].data_ptr(), steps, steps, ext, nb, g2, self.world, self.rank * cl + c0,
                       self.ptrs)
    self.hdl.barrier(channel=1)
    return self._commit_rows()


# ---------------------------------------------------------------- one proof over all ranks

def split_columns(ncols: int, world: int):
  """Contiguous column ranges, sizes differing by at most one: [(c0, c1), ...] per rank (a rank
  may get none: 6 columns over 8 ranks)."""
  base, extra = divmod(ncols, world)
  out, c = [], 0
  for r in range(world):
    k = base + (1 if r < extra else 0)
    out.append((c, c + k))
    c += k
  return out


def leaf_owner(x: int, n: int, world: int):
  """Row x of an n-row tree sharded by leaf range -> (owner rank, row index in the owner's local
  buffer).  Rank d holds rows {j*q + d*q/G + t : j < 4, t < q/G} (q = n/4) in (j, t) order --
  the rows of a local tree of n/G leaves whose permute4 order is the global one restricted to
  the subtree under global node G + d (starks/merkle_tree.py:11-33)."""
  q = n // 4
  lq = q // world
  j, i = divmod(x, q)
  d, t = divmod(i, lq)
  return d, j * lq + t


def extend_branch(local_branch, top_nodes, world: int, d: int):
  """mk_branch (merkle_tree.py:59-68) of the global tree from the branch inside rank d's
  subtree: the siblings above the subtree root (global node G + d) come from the replicated
  top levels."""
  out = list(local_branch)
  g = world + d
  while g > 1:
    out.append(top_nodes[g ^ 1])
    g //= 2
  return out


class NcclComm(object):
  """The sharded prover's exchanges over NCCL + torch symmetric memory (one process per GPU)."""

  def __init__(self, device, group=None):
    self.group = group if group is not None else dist.group.WORLD
    self.world, self.rank = _world(group)
    self.device = device
    self.hdl = None

  def shared_rows(self, shape):
    """A buffer every rank can store into: (tensor, [peer pointers])."""
    import torch.distributed._symmetric_memory as symm_mem
    t = symm_mem.empty(shape, dtype=torch.int32, device=self.device)
    self.hdl = symm_mem.rendezvous(t, self.group)
    return t, [int(p) for p in self.hdl.buffer_ptrs]

  def rows_barrier(self, engine, channel):
    self.hdl.barrier(channel=channel)     # device-side, on torch's current stream

  def commit_roots(self, engine, rows, n_local, ncols, nodes):
    """Local subtree over `rows` + the roots of every rank's subtree."""
    engine.merkle_commit(rows.data_ptr(), n_local, ncols, n_local, nodes.data_ptr(), want_root=False)
    return allgather_roots_from_nodes(nodes, self.group)

  def allreduce_bytes(self, buf):
    t = torch.from_numpy(buf).to(self.device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
    return t.cpu().numpy()

  def allgather_column(self, engine, column, col_local):
    dist.all_gather_into_tensor(column, col_local, group=self.group)


class ThreadComm(object):
  """The same exchanges between G emulated ranks that are THREADS of one process sharing one
  GPU (each with its own Engine): every exchange is a host-side barrier after a stream
  synchronisation, so no kernel ever waits on another (tests/test_gpu_dist_emulated.py)."""

  class Shared(object):
    def __init__(self, world):
      import threading
      self.world = world
      self.bar = threading.Barrier(world, timeout=300)   # a failed rank must not hang the others
      self.slots = [None] * world

  def __init__(self, shared, rank, device):
    self.sh, self.rank, self.world, self.device = shared, rank, shared.world, device

  def _exchange(self, value):
    self.sh.slots[self.rank] = value
    self.sh.bar.wait()
    out = list(self.sh.slots)
    self.sh.bar.wait()
    return out

  def shared_rows(self, shape):
    t = torch.empty(shape, dtype=torch.int32, device=self.device)
    return t, self._exchange(t.data_ptr())

  def rows_barrier(self, engine, channel):
    engine.sync()
    self.sh.bar.wait()

  def commit_roots(self, engine, rows, n_local, ncols, nodes):
    root = engine.merkle_commit(rows.data_ptr(), n_local, ncols, n_local, nodes.data_ptr())
    return self._exchange(bytes(root))

  def allreduce_bytes(self, buf):
    parts = self._exchange(buf)
    out = parts[0].copy()
    for x in parts[1:]:
      out += x
    return out

  def allgather_column(self, engine, column, col_local):
    engine.sync()
    parts = self._exchange(col_local)
    column.copy_(torch.cat(parts, dim=0))
    torch.cuda.synchronize()
    self.sh.bar.wait()


class ShardedProver(object):
  """STARK.mk_proof (starks/stark.py:233-279) for ONE proof over the G ranks of `group`
  (BASELINE config 5 "on 8 x B200"; SURVEY.md 8e):

    * every rank derives the 3w coefficient rows P, D, B (STARK.coefficient_rows: transforms of
      size `steps` and M <= d*steps, replicated -- a few per cent of the work);
    * the 3w size-N evaluations are split by COLUMN over the ranks and every transform's final
      pass stores its rows straight into the leaf owner's buffer over NVLink (stk_ntt_p2p): after
      one barrier every rank holds ALL columns for its leaf range;
    * leaf hashing, the linear combination l (pointwise), l's tree and FRI layer 0's fold (whole
      quads {i, i+q, i+2q, i+3q} are local under the permute4 ranges) run on N/G rows per rank;
      the two commitments are subtrees + an all-gather of 32-byte roots;
    * opened branches are cut from the local subtrees by the owner of each position and summed
      into one buffer (every record has exactly one owner);
    * the folded column (N/4 values) is all-gathered and FRI layers >= 1 run on rank 0
      (their sizes shrink 4x per layer and every challenge depends on the previous root).

  The proof object (rank 0) is bit-identical to the one-GPU STARK.mk_proof's."""

  def __init__(self, engine, field, steps, extension_factor, width, step_polys, device, group=None, comm=None):
    from .stark import STARK
    self.eng = engine
    self.S = STARK(field, steps, extension_factor, width, step_polys, engine=engine)
    self.comm = comm if comm is not None else NcclComm(device, group)
    self.world, self.rank = self.comm.world, self.comm.rank
    self.device = device
    N, G, w = self.S.precision, self.world, width
    assert N % (4 * G) == 0
    self.n_local = N // G
    self.rows, self.ptrs = self.comm.shared_rows((3 * w, self.n_local, 8))
    u8 = dict(dtype=torch.uint8, device=device)
    i32 = dict(dtype=torch.int32, device=device)
    self.nodes_m = torch.empty((self.n_local, 32), **u8)
    self.nodes_l = torch.empty((self.n_local, 32), **u8)
    self.l_rows = torch.empty((self.n_local, 8), **i32)
    q = N // 4
    self.col_local = torch.empty((q // G, 8), **i32)
    self.column = torch.empty((q, 8), **i32)
    self.nodes2 = torch.empty((q, 32), **u8)
    self.timings = {}

  # -- opened branches of a tree sharded by leaf range -------------------------------------
  def _branches(self, specs):
    """specs: [(rows tensor, ncols, nodes tensor, top nodes, [global positions]), ...] ->
    [[branch, ...], ...] on every rank.  Each rank cuts the branches whose leaves it owns; one
    all-reduce (sum of byte buffers with exactly one non-zero contributor per record) shares them."""
    N, G = self.S.precision, self.world
    depth = N.bit_length() - 1
    recs, total = [], 0
    for rows, ncols, nodes, top, pos in specs:
      L = 32 * ncols
      rec = 2 * L + 32 * (depth - 1)
      recs.append((L, rec, total))
      total += rec * len(pos)
    buf = np.zeros(total, dtype=np.uint8)
    for (rows, ncols, nodes, top, pos), (L, rec, off) in zip(specs, recs):
      mine = [(k, leaf_owner(x, N, G)) for k, x in enumerate(pos)]
      mine = [(k, loc) for k, (d, loc) in mine if d == self.rank]
      if not mine:
        continue
      local = self.eng.merkle_paths(rows.data_ptr(), self.n_local, ncols, self.n_local, nodes.data_ptr(),
                                    [loc for _, loc in mine])
      for (k, _), br in zip(mine, local):
        full = extend_branch(br, top, G, self.rank)
        b = b"".join(full)
        assert len(b) == rec
        buf[off + k * rec:off + (k + 1) * rec] = np.frombuffer(b, dtype=np.uint8)
    data = self.comm.allreduce_bytes(buf).tobytes()
    out = []
    from .engine import _path_struct
    for (rows, ncols, nodes, top, pos), (L, rec, off) in zip(specs, recs):
      S = _path_struct(L, depth)
      out.append([list(x) for x in S.iter_unpack(data[off:off + rec * len(pos)])])
    return out

  def mk_proof(self, witness, boundary):
    """Same arguments as STARK.mk_proof; every rank passes the same witness.  Returns the proof
    on rank 0 (None elsewhere)."""
    import time
    from .fri import FRI, DeviceLayer
    from .stark import interleave_branches, lincomb_weights
    from .utils import get_pseudorandom_indices
    t0 = time.perf_counter()
    marks = []
    mark = lambda name: marks.append((name, time.perf_counter()))
    S, eng, G, rank = self.S, self.eng, self.world, self.rank
    p = S.field.p
    eng.set_field(p)
    w, steps, ext, N = S.width, S.steps, S.extension_factor, S.precision
    G2 = int(S.G2)
    if isinstance(self.comm, NcclComm):
      _adopt_stream(eng, self.rows)   # order the engine's kernels with torch's collectives
    d_trace, owned, noncanonical = S._witness(eng, witness)
    c0, c1 = split_columns(3 * w, G)[rank]
    d_coef, cs = S.coefficient_rows(eng, d_trace.ptr, boundary, S._last_row(witness), want=range(c0, c1),
                                    witness_check=noncanonical)
    mark("coefficients")
    self.comm.rows_barrier(eng, 0)       # nobody still reads the previous proof's rows
    eng.ntt_p2p(d_coef.at(c0 * cs * 32), cs, cs, N, c1 - c0, G2, G, c0, self.ptrs)
    self.comm.rows_barrier(eng, 1)       # all rows have landed
    top_m = combine_subtree_roots(self.comm.commit_roots(eng, self.rows, self.n_local, 3 * w, self.nodes_m))
    m_root = top_m[1]
    mark("m_root")
    eng.lincomb(self.rows.data_ptr(), self.n_local, 3 * w, self.n_local, lincomb_weights(m_root, w, steps, N, G2, p),
                self.l_rows.data_ptr())
    top_l = combine_subtree_roots(self.comm.commit_roots(eng, self.l_rows, self.n_local, 1, self.nodes_l))
    l_root = top_l[1]
    mark("l_root")
    positions = get_pseudorandom_indices(l_root, N, 80, exclude_multiples_of=ext)
    # (the spot-check branches are cut together with FRI layer 0's below: one exchange for both)
    # FRI layer 0 (fri.py:217-256) on the sharded l, the rest on rank 0
    maxdeg = steps * S.get_degree()
    assert maxdeg > 16, "the sharded prover needs at least one FRI fold layer"
    q = N // 4
    lq = q // G
    eng.fri_fold4_rows(self.l_rows.data_ptr(), N, G2, int.from_bytes(l_root, "big"), lq, rank * lq,
                       self.col_local.data_ptr())
    self.comm.allgather_column(eng, self.column, self.col_local)
    root2 = eng.merkle_commit(self.column.data_ptr(), q, 1, q, self.nodes2.data_ptr())
    ys = get_pseudorandom_indices(root2, q, 40, exclude_multiples_of=ext)
    mb, lb, lb0 = self._branches([
        (self.rows, 3 * w, self.nodes_m, top_m, [x for pos in positions for x in (pos, (pos + ext) % N)]),
        (self.l_rows, 1, self.nodes_l, top_l, positions),
        (self.l_rows, 1, self.nodes_l, top_l, [y + q * j for y in ys for j in range(4)])])
    branches = interleave_branches(mb, lb)
    mark("fri_layer0_and_branches")
    proof = None
    if rank == 0:
      cb = eng.merkle_paths(self.column.data_ptr(), q, 1, q, self.nodes2.data_ptr(), ys)
      rest = FRI(S.field, engine=eng).prove_from_device(
          DeviceLayer(eng, self.column.data_ptr(), q, self.nodes2.data_ptr(), root2), pow(G2, 4, p), maxdeg // 4,
          exclude_multiples_of=ext)
      fri_proof = [[root2, [[cb[i]] + lb0[4 * i:4 * i + 4] for i in range(len(ys))]]] + rest
      proof = [m_root, l_root, branches, fri_proof]
    mark("fri_rest")
    eng.sync()
    if owned:
      d_trace.free()
    d_coef.free()
    self.timings = {"mk_proof_s": time.perf_counter() - t0}
    prev = t0
    for name, t in marks:
      self.timings[name + "_ms"] = (t - prev) * 1e3
      prev = t
    return proof
