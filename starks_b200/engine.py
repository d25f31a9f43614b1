"""Engine: one libstarks_b200 context (one GPU, one stream) with numpy-facing helpers.

Host code above the C ABI.  Device memory is owned either by the library
(`Engine.alloc`) or by torch tensors whose `data_ptr()` is passed straight through;
nothing here computes on the CPU."""
import ctypes
import functools
import struct
import threading

import numpy as np

from . import _lib
from .limbs import int_to_limbs, ints_to_limbs

P_STARK = 2**256 - 351 * 2**32 + 1


class DevBuf:
  """A device allocation made through stk_dev_alloc.  Freed buffers go back to a per-engine
  pool keyed by (rounded) size: cudaMalloc/cudaFree of GiB-sized buffers cost milliseconds and
  cudaFree synchronises the device, which would dominate a 20 ms proof.  Reuse is safe because
  every kernel of an engine runs on one stream (stream order = reuse order)."""

  _GRAN = 1 << 16

  def __init__(self, eng, nbytes):
    self.eng, self.nbytes = eng, int(nbytes)
    self.cap = max(self._GRAN, (self.nbytes + self._GRAN - 1) // self._GRAN * self._GRAN)
    pool = eng._pool.get(self.cap)
    if pool:
      self.ptr = pool.pop()
      return
    p = ctypes.c_void_p()
    rc = eng.lib.stk_dev_alloc(eng.ctx, self.cap, ctypes.byref(p))
    if rc != 0:  # out of memory: drop the pool and retry once
      eng.release_pool()
      eng._check(eng.lib.stk_dev_alloc(eng.ctx, self.cap, ctypes.byref(p)))
    self.ptr = p.value

  def free(self):
    if self.ptr is not None and self.eng.ctx is not None:
      self.eng._pool.setdefault(self.cap, []).append(self.ptr)
    self.ptr = None

  def __del__(self):
    try:
      self.free()
    except Exception:
      pass

  def at(self, byte_offset):
    return self.ptr + int(byte_offset)

  def upload(self, arr, byte_offset=0, wait=True):
    """wait=False: the caller keeps `arr` alive and unchanged until the stream is next synchronised
    (pinned sources then copy while the host goes on enqueueing)."""
    arr = np.ascontiguousarray(arr)
    assert byte_offset + arr.nbytes <= self.nbytes
    self.eng._check(self.eng.lib.stk_memcpy_h2d(self.eng.ctx, self.ptr + byte_offset, arr.ctypes.data, arr.nbytes))
    if wait:
      self.eng.sync()  # pageable source: keep it alive until the copy is done
    return self

  def download(self, shape, dtype=np.uint32, byte_offset=0):
    out = np.empty(shape, dtype=dtype)
    assert byte_offset + out.nbytes <= self.nbytes, (byte_offset, out.nbytes, self.nbytes)
    self.eng._check(self.eng.lib.stk_memcpy_d2h(self.eng.ctx, out.ctypes.data, self.ptr + byte_offset, out.nbytes))
    return out


class PinnedBuf:
  """Pinned host memory (stk_host_alloc) exposed as a numpy array."""

  def __init__(self, eng, shape, dtype=np.uint32):
    self.eng = eng
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = ctypes.c_void_p()
    eng._check(eng.lib.stk_host_alloc(eng.ctx, n, ctypes.byref(p)))
    self.ptr = p.value
    buf = (ctypes.c_uint8 * n).from_address(self.ptr)
    self.array = np.frombuffer(buf, dtype=dtype).reshape(shape)

  def free(self):
    if self.ptr is not None:
      self.array = None
      self.eng.lib.stk_host_free(self.eng.ctx, self.ptr)
      self.ptr = None


class Engine:
  """Owns a stk_ctx.  Raises if the library is not built or no CUDA device exists."""

  def __init__(self, device=0):
    self.lib = _lib.load()
    ctx = ctypes.c_void_p()
    rc = self.lib.stk_init(int(device), ctypes.byref(ctx))
    if rc != 0:
      self.ctx = None
      raise _lib.StarksB200Error(
          "stk_init(device=%d) failed (rc=%d): a CUDA device is required; there is no CPU fallback" % (device, rc))
    self.ctx = ctx
    self.device = device
    self.p = P_STARK
    self._pool = {}
    self._flag = None   # one pinned word for asynchronous device-side checks

  def release_pool(self):
    """Returns pooled device buffers to the driver."""
    for ptrs in self._pool.values():
      for p in ptrs:
        self.lib.stk_dev_free(self.ctx, p)
    self._pool = {}

  def close(self):
    if self.ctx is not None:
      self.release_pool()
      if self._flag is not None:
        self._flag.free()
        self._flag = None
      self.lib.stk_destroy(self.ctx)
      self.ctx = None

  def _check(self, rc):
    if rc == 0:
      return
    msg = self.lib.stk_last_error(self.ctx).decode() if self.ctx else ""
    if rc == _lib.STK_EINDEX:
      raise IndexError(msg or "list index out of range")
    if rc == _lib.STK_EINVAL:
      raise ValueError(msg or "invalid argument")
    raise _lib.StarksB200Error("libstarks_b200 error %d: %s" % (rc, msg))

  # ---- context ---------------------------------------------------------------
  def set_field(self, p):
    p = int(p)
    if p != self.p:
      self._check(self.lib.stk_field_set(self.ctx, _u32(int_to_limbs(p))))
      self.p = p

  def set_stream(self, cuda_stream_handle):
    self._check(self.lib.stk_set_stream(self.ctx, ctypes.c_void_p(cuda_stream_handle or 0)))

  def sync(self):
    self._check(self.lib.stk_sync(self.ctx))

  def alloc(self, nbytes):
    return DevBuf(self, nbytes)

  def pinned(self, shape, dtype=np.uint32):
    return PinnedBuf(self, shape, dtype)

  # ---- NTT -------------------------------------------------------------------
  def ntt(self, d_in, n_in, in_stride, d_out, out_stride, n, batch, root, inverse=False):
    """Device pointers (ints); see stk_ntt."""
    self._check(self.lib.stk_ntt(self.ctx, d_in, n_in, in_stride, d_out, out_stride, n, batch,
                                 _u32(int_to_limbs(int(root) % self.p)), int(bool(inverse))))

  def dft_generic(self, d_in, n_in, in_stride, d_out, out_stride, n, batch, root, inverse=False):
    """Direct O(n^2) DFT (stk_dft_generic), any order <= 4096."""
    self._check(self.lib.stk_dft_generic(self.ctx, d_in, n_in, in_stride, d_out, out_stride, n, batch,
                                         _u32(int_to_limbs(int(root) % self.p)), int(bool(inverse))))

  def ntt_host(self, cols, n, root, inverse=False, out=None):
    """cols: (batch, n_in, 8) uint32 host array -> (batch, n, 8) uint32 (stk_ntt_host)."""
    cols = np.ascontiguousarray(cols, dtype=np.uint32)
    batch, n_in, _ = cols.shape
    if out is None:
      out = np.empty((batch, n, 8), dtype=np.uint32)
    self._check(self.lib.stk_ntt_host(self.ctx, cols.ctypes.data, n_in, n_in, out.ctypes.data, n, n, batch,
                                      _u32(int_to_limbs(int(root) % self.p)), int(bool(inverse))))
    return out

  def ntt_dist_phase(self, phase, d_in, d_out, local_n, batch, stride, root, nranks, rank, inverse=False):
    """One phase of the multi-GPU four-step transform (stk_ntt_dist_phase)."""
    self._check(self.lib.stk_ntt_dist_phase(self.ctx, int(phase), d_in, d_out, local_n, batch, stride,
                                            _u32(int_to_limbs(int(root) % self.p)), nranks, rank,
                                            int(bool(inverse))))

  def ntt_dist_phase0_p2p(self, d_inout, local_n, root, nranks, rank, peer_ptrs, inverse=False):
    """Phase 0 with the exchange fused into its last pass (stk_ntt_dist_phase0_p2p)."""
    arr = (ctypes.c_uint64 * nranks)(*[int(p) for p in peer_ptrs])
    self._check(self.lib.stk_ntt_dist_phase0_p2p(self.ctx, d_inout, local_n, _u32(int_to_limbs(int(root) % self.p)),
                                                 nranks, rank, int(bool(inverse)), arr))

  def mul_polys(self, a, b, n, root):
    a = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, 8)
    b = np.ascontiguousarray(b, dtype=np.uint32).reshape(-1, 8)
    da, db, do = self.alloc(max(a.nbytes, 32)), self.alloc(max(b.nbytes, 32)), self.alloc(n * 32)
    da.upload(a)
    db.upload(b)
    self._check(self.lib.stk_mul_polys(self.ctx, da.ptr, len(a), db.ptr, len(b), do.ptr, n,
                                       _u32(int_to_limbs(int(root) % self.p))))
    out = do.download((n, 8))
    for x in (da, db, do):
      x.free()
    return out

  def poly_mul(self, d_a, na, d_b, nb, d_out):
    """Linear product of two coefficient vectors on the device (stk_poly_mul): d_out receives
    na + nb - 1 coefficients."""
    self._check(self.lib.stk_poly_mul(self.ctx, d_a, na, d_b, nb, d_out))

  def poly_divmod(self, d_a, na, d_b, nb, d_q, d_r):
    """Long division a = b*q + r on the device (stk_poly_divmod): d_q receives max(na-nb+1, 0)
    coefficients, d_r receives nb-1.  Synchronises the stream."""
    self._check(self.lib.stk_poly_divmod(self.ctx, d_a, na, d_b, nb, d_q, d_r))

  def poly_compose(self, d_a, na, d_b, nb, d_out):
    """Composition a(b(X)) on the device (stk_poly_compose): d_out receives (na-1)(nb-1)+1
    coefficients; nb >= 2.  Synchronises the stream when nb == 2."""
    self._check(self.lib.stk_poly_compose(self.ctx, d_a, na, d_b, nb, d_out))

  def poly_eval_multivar(self, d_polys, lens, in_stride, monomials, nout, d_out, out_len):
    """Multivariate polynomials evaluated at polynomials on the device (stk_poly_eval_multivar).
    Argument k has lens[k] coefficients at d_polys + 32*k*in_stride; monomials is a list of
    (output index, int coefficient, exponent tuple of len(lens)); output j is written at
    d_out + 32*j*out_len, and out_len must be D + 1 (see the header)."""
    width, nmono = len(lens), len(monomials)
    h_lens = np.asarray(lens, dtype=np.uint64)
    h_out = np.asarray([m[0] for m in monomials] or [0], dtype=np.uint32)
    h_coeffs = ints_to_limbs([int(m[1]) % self.p for m in monomials] or [0])
    h_exps = np.asarray([e for m in monomials for e in m[2]] or [0], dtype=np.uint32)
    assert h_exps.size == max(nmono * width, 1), "every exponent tuple needs one entry per argument"
    self._check(self.lib.stk_poly_eval_multivar(self.ctx, d_polys, h_lens.ctypes.data, in_stride, width,
                                                h_out.ctypes.data, h_coeffs.ctypes.data, h_exps.ctypes.data, nmono,
                                                nout, d_out, out_len))

  def power_cycle(self, r, n):
    do = self.alloc(n * 32)
    self._check(self.lib.stk_power_cycle(self.ctx, _u32(int_to_limbs(int(r) % self.p)), n, do.ptr))
    out = do.download((n, 8))
    do.free()
    return out

  # ---- LDE / Merkle / FRI (device pointers) ------------------------------------
  def lde(self, d_trace, steps, trace_stride, ext, cols, g2, d_evals, eval_stride, d_coeffs=0, coeff_stride=0):
    self._check(self.lib.stk_lde(self.ctx, d_trace, steps, trace_stride, ext, cols,
                                 _u32(int_to_limbs(int(g2) % self.p)), d_coeffs or None, coeff_stride, d_evals,
                                 eval_stride))

  def lde_p2p(self, d_trace, steps, trace_stride, ext, cols, g2, nranks, col_base, peer_ptrs):
    """LDE of a column shard whose final pass scatters rows to their leaf owners (stk_lde_p2p)."""
    arr = (ctypes.c_uint64 * nranks)(*[int(p) for p in peer_ptrs])
    self._check(self.lib.stk_lde_p2p(self.ctx, d_trace, steps, trace_stride, ext, cols,
                                     _u32(int_to_limbs(int(g2) % self.p)), nranks, col_base, arr))

  def ntt_p2p(self, d_coeffs, n_in, in_stride, n, cols, root, nranks, col_base, peer_ptrs):
    """Forward transform of coefficient rows whose final pass scatters rows to their leaf owners
    (stk_ntt_p2p); cols may be 0."""
    arr = (ctypes.c_uint64 * nranks)(*[int(p) for p in peer_ptrs])
    self._check(self.lib.stk_ntt_p2p(self.ctx, d_coeffs, n_in, in_stride, n, cols,
                                     _u32(int_to_limbs(int(root) % self.p)), nranks, col_base, arr))

  def lincomb(self, d_cols, n, ncols, col_stride, weights, d_out):
    """out[i] = sum_c weights[c] * cols[c][i] (stk_lincomb); weights: list of ints."""
    from .limbs import ints_to_limbs
    wl = ints_to_limbs([int(x) % self.p for x in weights])
    self._check(self.lib.stk_lincomb(self.ctx, d_cols, n, ncols, col_stride, wl.ctypes.data, d_out))

  def fri_fold4_rows(self, d_rows, n, root, special_x, q_run, i0, d_out):
    """Fold of the quads i0 .. i0+q_run-1 of an n-point layer held as four runs (stk_fri_fold4_rows)."""
    self._check(self.lib.stk_fri_fold4_rows(self.ctx, d_rows, n, _u32(int_to_limbs(int(root) % self.p)),
                                            _u32(int_to_limbs(int(special_x))), q_run, i0, d_out))

  def lde_commit(self, d_trace, steps, trace_stride, ext, cols, g2, d_evals, eval_stride, d_nodes):
    root = (ctypes.c_uint8 * 32)()
    self._check(self.lib.stk_lde_commit(self.ctx, d_trace, steps, trace_stride, ext, cols,
                                        _u32(int_to_limbs(int(g2) % self.p)), d_evals, eval_stride, d_nodes, root))
    return bytes(root)

  def lde_commit_host(self, h_trace, ext, g2, d_evals, eval_stride, d_nodes):
    """stk_lde_commit_host: h_trace is a (cols, steps, 8) uint32 HOST array (pinned for overlap)."""
    cols, steps, _ = h_trace.shape
    assert h_trace.dtype == np.uint32 and h_trace.flags["C_CONTIGUOUS"]
    root = (ctypes.c_uint8 * 32)()
    self._check(self.lib.stk_lde_commit_host(self.ctx, h_trace.ctypes.data, steps, steps, ext, cols,
                                             _u32(int_to_limbs(int(g2) % self.p)), d_evals, eval_stride, d_nodes, root))
    return bytes(root)

  def merkle_commit(self, d_cols, n, ncols, col_stride, d_nodes, want_root=True):
    root = (ctypes.c_uint8 * 32)()
    self._check(self.lib.stk_merkle_commit(self.ctx, d_cols, n, ncols, col_stride, d_nodes,
                                           root if want_root else None))
    return bytes(root) if want_root else None

  def merkle_commit_raw(self, d_leaves, n, leaf_len, d_nodes):
    root = (ctypes.c_uint8 * 32)()
    self._check(self.lib.stk_merkle_commit_raw(self.ctx, d_leaves, n, leaf_len, d_nodes, root))
    return bytes(root)

  def merkle_paths(self, d_cols, n, ncols, col_stride, d_nodes, indices):
    """mk_branch for many indices at once -> list of branches (lists of bytes)."""
    k = len(indices)
    if k == 0:
      return []
    depth = (4 * (n // 4)).bit_length() - 1
    L = 32 * ncols
    rec = 2 * L + 32 * (depth - 1)
    idx = np.asarray(indices, dtype=np.uint64)
    out = np.empty((k, rec), dtype=np.uint8)
    self._check(self.lib.stk_merkle_paths(self.ctx, d_cols, n, ncols, col_stride, d_nodes, idx.ctypes.data, k,
                                          out.ctypes.data, rec))
    # one C call splits every record into its [leaf, sibling leaf, nodes...] bytes objects
    S = _path_struct(L, depth)
    res = [list(t) for t in S.iter_unpack(out.tobytes())]
    return res

  def verify_branches(self, root, indices, branches):
    """verify_branch (starks/merkle_tree.py:71-86) for many branches of one tree in one kernel.
    Returns the leaves (proof[0] of every branch); raises AssertionError like the reference
    when a branch does not hash up to `root`."""
    k = len(indices)
    if k == 0:
      return []
    depth = len(branches[0]) - 1
    assert depth >= 1, "malformed branch"
    n = 1 << depth
    L = len(branches[0][0])
    rec = 2 * L + 32 * (depth - 1)
    # The kernel hashes fixed offsets of the packed record ([0:L] leaf, [L:2L] sibling leaf, then
    # 32-byte nodes) and the caller computes with b[0]: every element must have exactly the width
    # the kernel assumes, otherwise a proof could shift bytes between elements and have a value
    # other than the committed leaf accepted (the reference hashes exactly the proof[0] it
    # returns, merkle_tree.py:71-86).
    assert L > 0 and L % 32 == 0, "malformed branch: leaf width"
    for b in branches:
      assert len(b) == depth + 1, "branches of one tree have one length"
      assert len(b[0]) == L and len(b[1]) == L, "malformed branch: leaf / sibling width"
      for x in b[2:]:
        assert len(x) == 32, "malformed branch: node width"
    buf = np.frombuffer(b"".join(b"".join(b) for b in branches), dtype=np.uint8)
    assert buf.size == k * rec, "malformed branch"
    idx = np.asarray(indices, dtype=np.uint64)
    ok = np.zeros(k, dtype=np.uint8)
    rb = (ctypes.c_uint8 * 32).from_buffer_copy(root)
    self._check(self.lib.stk_verify_branches(self.ctx, rb, n, L, idx.ctypes.data, k, buf.ctypes.data, rec,
                                             ok.ctypes.data))
    assert ok.all(), "Merkle branch does not match the root"
    return [b[0] for b in branches]

  def fri_fold4(self, d_vals, n, root, special_x, d_out):
    self._check(self.lib.stk_fri_fold4(self.ctx, d_vals, n, _u32(int_to_limbs(int(root) % self.p)),
                                       _u32(int_to_limbs(int(special_x))), d_out))

  def fri_prove(self, d_vals, n, d_nodes, root_bytes, root, maxdeg_plus_1, exclude_multiples_of, security):
    """stk_fri_prove -> the proof list of generate_proximity_proof (starks/fri.py:189-266):
    [[root2, [[branch(m2,y), branch(m,y), branch(m,y+q), branch(m,y+2q), branch(m,y+3q)], ...]], ...,
    [final values as 32-byte big-endian]]."""
    layers, nn, md, k, total = [], n, maxdeg_plus_1, security, 0
    while md > 16:
      q = nn // 4
      d1, d2 = nn.bit_length() - 1, q.bit_length() - 1
      layers.append((k, d1, d2))
      total += 32 + k * (64 + 32 * (d2 - 1)) + 4 * k * (64 + 32 * (d1 - 1))
      nn, md, k = q, md // 4, 40
    total += 32 * nn
    out = np.empty(total, dtype=np.uint8)
    need = ctypes.c_uint64(0)
    rb = (ctypes.c_uint8 * 32).from_buffer_copy(root_bytes) if d_nodes else None
    self._check(self.lib.stk_fri_prove(self.ctx, d_vals, n, d_nodes or None, rb, _u32(int_to_limbs(int(root) % self.p)),
                                       maxdeg_plus_1, exclude_multiples_of, security, out.ctypes.data, total,
                                       ctypes.byref(need)))
    assert need.value == total, (need.value, total)
    buf, off, proof = out.tobytes(), 0, []
    for k, d1, d2 in layers:
      root2 = buf[off:off + 32]
      off += 32
      r2, r1 = 64 + 32 * (d2 - 1), 64 + 32 * (d1 - 1)
      col = [list(t) for t in _path_struct(32, d2).iter_unpack(buf[off:off + k * r2])]
      off += k * r2
      rows = [list(t) for t in _path_struct(32, d1).iter_unpack(buf[off:off + 4 * k * r1])]
      off += 4 * k * r1
      proof.append([root2, [[col[i]] + rows[4 * i:4 * i + 4] for i in range(k)]])
    proof.append(list(struct.unpack("32s" * nn, buf[off:off + 32 * nn])))
    return proof

  def count_noncanonical(self, d_vals, n, wait=True):
    """How many of the n elements at d_vals are >= p (stk_count_noncanonical).  wait=False
    returns a zero-argument callable to be called after the stream has been synchronised."""
    if wait:
      bad = ctypes.c_uint32(0)
      self._check(self.lib.stk_count_noncanonical(self.ctx, d_vals, n, ctypes.addressof(bad), 1))
      return bad.value
    if self._flag is None:
      self._flag = self.pinned((16,))
    self._check(self.lib.stk_count_noncanonical(self.ctx, d_vals, n, self._flag.ptr, 0))
    return lambda: int(self._flag.array[0])

  def microbench_variant(self, variant, which, iters):
    ms, ops, bad = ctypes.c_float(), ctypes.c_double(), ctypes.c_uint64()
    self._check(self.lib.stk_microbench_variant(self.ctx, variant, which, iters, ctypes.byref(ms), ctypes.byref(ops),
                                                ctypes.byref(bad)))
    return ms.value, ops.value, bad.value

  def microbench(self, which, iters):
    ms, ops = ctypes.c_float(), ctypes.c_double()
    self._check(self.lib.stk_microbench(self.ctx, which, iters, ctypes.byref(ms), ctypes.byref(ops)))
    return ms.value, ops.value


@functools.lru_cache(maxsize=None)
def _path_struct(L, depth):
  return struct.Struct("%ds%ds" % (L, L) + "32s" * (depth - 1))


def _u32(arr):
  return arr.ctypes.data_as(_lib.u32p)


_default = None
_lock = threading.Lock()


def default_engine() -> Engine:
  """Process-wide engine on LOCAL_RANK's GPU (one process per GPU)."""
  global _default
  with _lock:
    if _default is None:
      import os
      _default = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default
