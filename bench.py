#!/usr/bin/env python
"""bench.py -- the reference's headline metric (BASELINE.json) on B200:
"NTT Melem/s at 2^20; LDE+Merkle-commit ms/proof at 1/2/4/8 B200".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line (rank 0).  `--dump-outputs DIR` also writes rank 0's output of the last timed step
(a fixed, seeded sample of its points; see dump_outputs) to DIR, so that two builds can be compared
output for output: the inputs are seeded and the same in every run.  What is in the line:

  value / ms_per_step   forward NTT of `--cols` (64) columns x 2^20 per GPU, inputs resident in
                        HBM (2 GiB in, 2 GiB out: larger than L2), CUDA events on the launching
                        stream, max over ranks.  N > 1: every rank transforms its own columns
                        (column sharding, no data-path collective) -> weak scaling.
  e2e                   the same step through the host-buffer API (stk_ntt_host): pinned host
                        buffers, H2D + transform + D2H inside the timed region.
  roofline              the dominant kernel (ntt_pass_kernel) against the INTEGER pipes (the
                        binding roofline of 256-bit modular butterflies; SURVEY.md 8d's frozen
                        264 int32 ops per butterfly against the K0 microbenchmark of this run),
                        HBM as the secondary figure.
  parity                the TIMED output checked against the CPU oracle (4 of the 64 columns,
                        element for element) and an on-device inverse round trip of all columns.
  lde_merkle_commit_ms  BASELINE config 3 (64 trace columns x 2^18 steps, 8x blowup, one Merkle
                        tree over all columns) on the N GPUs of this run: N = 1 one GPU; N > 1
                        columns sharded over the ranks with the leaf exchange as (a) an NCCL
                        all-to-all and (b) P2P stores fused into the transform's final pass.
                        Root compared with the single-GPU root computed in the same run.
  lde_merkle_commit_e2e_ms   the metric as BASELINE defines it end to end: trace in pinned HOST
                        memory -> H2D -> LDE + commit -> 32-byte root on the host.
  ntt_2^26_ms           BASELINE config 4: one 2^26-point transform; N = 1 one GPU; N > 1
                        four-step with (a) NCCL all-to-all + transpose, (b) the exchange fused
                        into the last phase-0 pass.  The TIMED output is compared with the
                        single-GPU transform of the same input.
  strong_scaling        both of the above are strong-scaling workloads: efficiency =
                        t(1 GPU, same run) / (N * t(N GPUs)).
  stark_proof_*         BASELINE config 5 shape (Fibonacci, 2^20 steps, 8x) on one GPU.
  cpu_baseline          N = 1 only: the pure-Python reference (baseline/_ref) timed on this host
                        (1 core: it is single-threaded) next to the C oracle port.

`--impl reference` is the CPU arm: the reference is pure Python (fft_1d at 2^20 = 74 s per
column), so the arm times the C oracle port of fft_1d (oracle/) on all the host threads this
process may use, on a bounded sample of the same workload."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P = 2**256 - 351 * 2**32 + 1
LOGN = 20
N = 1 << LOGN
INT_OPS_PER_BUTTERFLY = 264       # SURVEY.md 8(d), frozen
BYTES_PER_ELEM = 64               # read once + write once
# measured once per change with ncu (profiles/r02_ncu_ntt_pass_summary.txt): the two passes of
# one step move 4.44 GB and 4.24 GB; each pass reads and writes the whole 2 GiB batch
NCU_TRAFFIC_BYTES_PER_LAUNCH = 4.34e9
NCU_SOURCE = "profiles/r02_ncu_ntt_pass_summary.txt"
# per butterfly in the pass kernel's SASS: 64 (product) + 8 (fold by 351) half-rate wide multiply-adds
WIDE_MACS_PER_BUTTERFLY = 72
NCU_FMAHEAVY_ACTIVE_PCT = (72.3, 70.2)   # first pass, final pass
WORKLOAD = "forward NTT, %d columns x 2^20 per GPU, p = 2^256-351*2^32+1 (BASELINE configs[1] at its headline size)"


def bench_config(cols, world):
  """The `config` object of the line: identical for our arm and for the reference arm."""
  return {"workload": WORKLOAD % cols, "cols_per_gpu": cols, "log2_n": LOGN,
          "l2_policy": "inputs (2 GiB) exceed L2, no flush",
          "parallelism": "column-sharded x%d, no collective (configs 3 and 4 in the same line use the exchange paths)" % world}


def host_threads():
  """Threads this process may run on.  Not OMP_NUM_THREADS: torchrun exports it as 1."""
  try:
    return max(1, len(os.sched_getaffinity(0)))
  except AttributeError:
    return max(1, os.cpu_count() or 1)


def peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    d = json.load(open(path))
    return float(d["hbm_gbs"]), "measured"
  return 6650.0, "fallback"


class ClockSampler(threading.Thread):
  """Samples SM clock / throttle reasons through NVML every ~5 ms while the timed region runs
  (nvidia-smi as a fallback)."""

  def __init__(self, gpu_index):
    super().__init__(daemon=True)
    self.idx, self.samples, self.reasons, self.maxmhz = gpu_index, [], set(), None
    self._stop_evt = threading.Event()
    self.nvml = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nvml = pynvml
      self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu_index))
      self.maxmhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
    except Exception:
      self.nvml = None

  @staticmethod
  def _physical_index(i):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
      try:
        return int(vis.split(",")[i])
      except Exception:
        return i
    return i

  def _sample_nvml(self):
    n = self.nvml
    self.samples.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
    for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                      ("hw_thermal_slowdown", 0x40)):
      if r & bit:
        self.reasons.add(name)

  def _sample_smi(self):
    q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, timeout=5).stdout.strip().split(",")
    self.samples.append(float(out[0]))
    self.maxmhz = float(out[1])
    for nm, v in zip(names, out[2:]):
      if v.strip().lower() == "active":
        self.reasons.add(nm)

  def run(self):
    while not self._stop_evt.is_set():
      try:
        if self.nvml is not None:
          self._sample_nvml()
        else:
          self._sample_smi()
      except Exception:
        pass
      self._stop_evt.wait(0.005 if self.nvml is not None else 0.1)

  def stop(self):
    self._stop_evt.set()
    self.join(timeout=10)
    s = sorted(self.samples)
    return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxmhz, "reasons": sorted(self.reasons),
            "samples": len(s), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


class Watchdog(object):
  """A device-side barrier that never completes cannot be caught as an exception: if the
  multi-GPU section overruns, rank 0 still prints the line it has (with the overrun named) and
  every rank leaves."""

  def __init__(self, seconds, rank, line, label):
    self.t = threading.Timer(seconds, self._fire)
    self.t.daemon = True
    self.rank, self.line, self.label, self.seconds = rank, line, label, seconds

  def _fire(self):
    if self.rank == 0:
      self.line["watchdog"] = "%s did not finish within %d s; line printed by the watchdog" % (self.label, self.seconds)
      print(json.dumps(self.line), flush=True)
    os._exit(0 if self.rank == 0 else 3)

  def __enter__(self):
    self.t.start()
    return self

  def __exit__(self, *a):
    self.t.cancel()
    return False


def pcie_duplex_ceiling(torch, local):
  """Pinned H2D and D2H copies of 512 MiB at once on two streams: GB/s per direction."""
  nbytes = 1 << 29
  dev = "cuda:%d" % local
  h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
  h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
  d_a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
  d_b = torch.empty(nbytes, dtype=torch.uint8, device=dev)
  s1, s2 = torch.cuda.Stream(device=local), torch.cuda.Stream(device=local)
  best = 0.0
  for rep in range(3):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2):
      with torch.cuda.stream(s1):
        d_a.copy_(h_in, non_blocking=True)
      with torch.cuda.stream(s2):
        h_out.copy_(d_b, non_blocking=True)
    torch.cuda.synchronize()
    if rep:
      best = max(best, 2 * nbytes / (time.perf_counter() - t0) / 1e9)
  return best


def synth_columns(cols, n, seed):
  import numpy as np
  rng = np.random.default_rng(seed)
  a = rng.integers(0, 2**32, size=(cols, n, 8), dtype=np.uint64).astype(np.uint32)
  a[:, :, 7] &= 0x7FFFFFFF  # < 2^255 < p: canonical residues
  return a


DUMP_POINTS = 8192     # sampled points per column: 64 columns x 8192 x 8 limbs in float64 = 32 MiB
DUMP_SEED = 20        # fixed: every run and every build samples the same points


def dump_outputs(out_dir, torch, d_out):
  """Writes what the timed NTT handed back in its last step to out_dir as .npy files:
  ntt_out_limbs.npy (cols, DUMP_POINTS, 8): the eight little-endian 32-bit limbs of every column at
  a fixed, seeded sample of evaluation points, as float64 (exact for 32-bit values);
  ntt_out_points.npy (DUMP_POINTS,): the sampled point indices."""
  import numpy as np
  cols, n, _ = d_out.shape
  pts = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(DUMP_POINTS, n), replace=False))
  limbs = d_out[:, torch.from_numpy(pts).to(d_out.device), :].cpu().numpy().view(np.uint32)
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "ntt_out_limbs.npy"), limbs.astype(np.float64))
  np.save(os.path.join(out_dir, "ntt_out_points.npy"), pts.astype(np.float64))


def numa_note():
  """The NTT e2e is bound by the host side: name what the box exposes."""
  try:
    nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")]
    return "%d NUMA node(s) visible; pinned buffers come from cudaHostAlloc on the node of the allocating thread" % len(nodes)
  except Exception:
    return "NUMA layout not readable"


# ------------------------------------------------------------------ the per-config sections

class Ctx(object):
  def __init__(self, torch, dist, eng, stream, rank, world, local):
    self.torch, self.dist, self.eng, self.stream = torch, dist, eng, stream
    self.rank, self.world, self.local = rank, world, local
    self.dev = torch.device("cuda", local)

  def tmax(self, v):
    if self.world == 1:
      return float(v)
    t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
    self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
    return float(t[0])

  def all_true(self, ok):
    if self.world == 1:
      return bool(ok)
    t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int32, device=self.dev)
    self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
    return bool(int(t[0]))

  def barrier(self):
    if self.world > 1:
      self.dist.barrier()
    self.torch.cuda.synchronize()

  def same_everywhere(self, t):
    """A tensor made on rank 0 and broadcast over NVLink: every rank works on the same input."""
    if self.world > 1:
      self.dist.broadcast(t, src=0)
    return t

  def timed(self, fn, reps):
    """ms per call of fn (enqueued on torch's current stream), CUDA events, max over ranks."""
    torch = self.torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    self.barrier()
    e0.record()
    out = None
    for _ in range(reps):
      out = fn()
    e1.record()
    torch.cuda.synchronize()
    return self.tmax(e0.elapsed_time(e1) / reps), out


def section_config3(cx, line, reps=4):
  """LDE + Merkle commit of 64 x 2^18 -> 2^21 on the GPUs of this run."""
  torch, eng, world, rank, dev = cx.torch, cx.eng, cx.world, cx.rank, cx.dev
  from starks_b200 import dist as sd
  import numpy as np
  steps, ext, ncols = 1 << 18, 8, 64
  n = steps * ext
  g2 = pow(7, (P - 1) // n, P)
  out = {"workload": "64 trace columns x 2^18 steps, 8x blowup -> one Merkle tree over 2^21 leaves of 2048 B"}
  gen = torch.Generator(device=dev)
  gen.manual_seed(3)
  trace = cx.same_everywhere(torch.randint(0, 2**31 - 1, (ncols, steps, 8), dtype=torch.int32, device=dev, generator=gen))
  sd._adopt_stream(eng, trace)
  d_ev = torch.empty((ncols, n, 8), dtype=torch.int32, device=dev)
  d_nodes = torch.empty((n, 32), dtype=torch.uint8, device=dev)

  def one_gpu():
    return eng.lde_commit(trace.data_ptr(), steps, steps, ext, ncols, g2, d_ev.data_ptr(), n, d_nodes.data_ptr())
  for _ in range(2):
    want_root = one_gpu()
  # wall clock: the call returns with the root on the host
  cx.barrier()
  t0 = time.perf_counter()
  for _ in range(reps):
    one_gpu()
  t1 = cx.tmax((time.perf_counter() - t0) / reps * 1e3)
  out["one_gpu_ms"] = t1
  # split of the one-GPU call (CUDA events)
  e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
  e[0].record()
  eng.lde(trace.data_ptr(), steps, steps, ext, ncols, g2, d_ev.data_ptr(), n)
  e[1].record()
  eng.merkle_commit(d_ev.data_ptr(), n, ncols, n, d_nodes.data_ptr(), want_root=False)
  e[2].record()
  torch.cuda.synchronize()
  out["one_gpu_lde_ms"], out["one_gpu_merkle_ms"] = e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])
  compressions = (n // 2) * ncols + (n // 2 - 1)
  out["merkle_gcompress_per_s"] = compressions / (out["one_gpu_merkle_ms"] * 1e-3) / 1e9
  lde_bfly = ncols * ((steps // 2) * 18 + (n // 2) * 21)
  out["lde_gbutterflies_per_s"] = lde_bfly / (out["one_gpu_lde_ms"] * 1e-3) / 1e9
  if world == 1:
    # the fused LDE -> leaf-hash kernel of the north star (opt-in: see DESIGN.md section 4)
    os.environ["STK_FUSED_HASH"] = "1"
    try:
      root_f = one_gpu()
      cx.barrier()
      t0 = time.perf_counter()
      for _ in range(reps):
        one_gpu()
      out["one_gpu_fused_leaf_hash_ms"] = (time.perf_counter() - t0) / reps * 1e3
      out["fused_leaf_hash_root_ok"] = bool(root_f == want_root)
    finally:
      del os.environ["STK_FUSED_HASH"]
  del d_ev
  best, parity = t1, True
  # end to end as BASELINE defines it: trace on the HOST (pinned) -> root on the host
  cl = ncols // world
  h_tr = eng.pinned((cl, steps, 8))
  h_tr.array[...] = trace[rank * cl:(rank + 1) * cl].cpu().numpy().view(np.uint32)
  d_tr = torch.empty((cl, steps, 8), dtype=torch.int32, device=dev)
  h_t = torch.from_numpy(h_tr.array.view(np.int32))
  if world == 1:
    d_ev1 = torch.empty((ncols, n, 8), dtype=torch.int32, device=dev)

    def e2e():
      d_tr.copy_(h_t, non_blocking=True)
      return eng.lde_commit(d_tr.data_ptr(), steps, steps, ext, ncols, g2, d_ev1.data_ptr(), n, d_nodes.data_ptr())
    assert e2e() == want_root
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
      e2e()
    out["e2e_copy_then_commit_ms"] = (time.perf_counter() - t0) / reps * 1e3

    def e2e_api():   # the host-trace entry point: upload pipelined with the transforms
      return eng.lde_commit_host(h_tr.array, ext, g2, d_ev1.data_ptr(), n, d_nodes.data_ptr())
    assert e2e_api() == want_root
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
      e2e_api()
    out["e2e_ms"] = (time.perf_counter() - t0) / reps * 1e3
    del d_ev1
  else:
    del d_nodes
    torch.cuda.empty_cache()
    mine = trace[rank * cl:(rank + 1) * cl].contiguous()
    # this rank's LDE alone (column-sharded evaluations, no exchange), with and without the copied coset
    ev_loc = torch.empty((cl, n, 8), dtype=torch.int32, device=dev)
    for tag, env in (("lde_only_ms", None), ("lde_only_full_transform_ms", "0")):
      if env is not None:
        os.environ["STK_LDE_R0"] = env
      try:
        eng.lde(mine.data_ptr(), steps, steps, ext, cl, g2, ev_loc.data_ptr(), n)
        out[tag], _ = cx.timed(lambda: eng.lde(mine.data_ptr(), steps, steps, ext, cl, g2, ev_loc.data_ptr(), n), reps)
      finally:
        if env is not None:
          del os.environ["STK_LDE_R0"]
    del ev_loc
    torch.cuda.empty_cache()
    sc = sd.ShardedCommit(eng)
    for _ in range(2):
      r = sc.lde_commit(mine, ext, g2)
    ok_nccl = cx.all_true(r[0] == want_root)
    del r
    per_call = []
    for _ in range(reps + 1):
      cx.barrier()
      t0 = time.perf_counter()
      r = sc.lde_commit(mine, ext, g2)
      torch.cuda.synchronize()
      per_call.append((time.perf_counter() - t0) * 1e3)
      del r                                  # evaluations, rows and nodes of this call (6 GiB) go back first
    per_call = sorted(per_call[1:])
    out["nccl_all_to_all_ms"] = cx.tmax(per_call[len(per_call) // 2])      # median call, max over ranks
    out["nccl_all_to_all_ms_per_call"] = [round(x, 2) for x in per_call]
    out["nccl_root_equals_one_gpu_root"] = ok_nccl
    out["nccl_host_timeline_ms"] = getattr(sc, "timings", None)
    torch.cuda.empty_cache()
    parity = parity and ok_nccl
    best_n = out["nccl_all_to_all_ms"]
    try:
      scp = sd.ShardedCommitP2P(eng, ncols, n, dev)
      for _ in range(2):
        rp = scp.lde_commit(mine, ext, g2)
      ok_p2p = cx.all_true(rp[0] == want_root)
      cx.barrier()
      t0 = time.perf_counter()
      for _ in range(reps):
        scp.lde_commit(mine, ext, g2)
      torch.cuda.synchronize()
      out["fused_p2p_ms"] = cx.tmax((time.perf_counter() - t0) / reps * 1e3)
      out["fused_p2p_root_equals_one_gpu_root"] = ok_p2p
      parity = parity and ok_p2p
      if ok_p2p:
        best_n = min(best_n, out["fused_p2p_ms"])

      def e2e_serial():
        d_tr.copy_(h_t, non_blocking=True)
        return scp.lde_commit(d_tr, ext, g2)[0]

      def e2e():   # upload pipelined with the per-group transforms + scatter
        return scp.lde_commit_host(h_t, d_tr, ext, g2)[0]
      for name, fn in (("e2e_copy_then_commit_ms", e2e_serial), ("e2e_ms", e2e)):
        ok_e2e = cx.all_true(fn() == want_root)
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
          fn()
        torch.cuda.synchronize()
        out[name] = cx.tmax((time.perf_counter() - t0) / reps * 1e3)
        out["e2e_root_ok"] = bool(out.get("e2e_root_ok", True) and ok_e2e)
      del scp
    except Exception as ex:  # pragma: no cover
      out["fused_p2p_error"] = repr(ex)[:300]
    best = best_n
    out["strong_scaling_efficiency"] = t1 / (world * best)
    out["limiter"] = ("per-rank LDE of %d columns (integer pipes) + the leaf rows' trip over NVLink (%.0f MiB out per "
                      "rank) + one subtree per rank" % (cl, cl * n * 32 * (world - 1) / world / 2**20))
  out["e2e_h2d_bytes_per_rank"] = cl * steps * 32
  out["e2e_d2h_bytes"] = 32
  h_tr.free()
  line["lde_merkle_commit_ms"] = best
  line["lde_merkle_commit_e2e_ms"] = out.get("e2e_ms")
  line["lde_merkle_commit_parity_ok"] = bool(parity)
  line["lde_merkle_commit_strong_scaling_efficiency"] = out.get("strong_scaling_efficiency", 1.0)
  line["lde_merkle_commit"] = out
  torch.cuda.empty_cache()


def section_config4(cx, line, reps=4):
  """One 2^26-point transform on the GPUs of this run; the timed output is compared with the
  one-GPU transform of the same input."""
  torch, eng, world, rank, dev = cx.torch, cx.eng, cx.world, cx.rank, cx.dev
  from starks_b200 import dist as sd
  logn = 26
  n = 1 << logn
  w = pow(7, (P - 1) // n, P)
  out = {"workload": "one forward NTT of 2^26 points (2 GiB)"}
  gen = torch.Generator(device=dev)
  gen.manual_seed(4)
  x = cx.same_everywhere(torch.randint(0, 2**31 - 1, (n, 8), dtype=torch.int32, device=dev, generator=gen))
  ref = torch.empty_like(x)
  sd._adopt_stream(eng, x)

  def one_gpu():
    eng.ntt(x.data_ptr(), n, n, ref.data_ptr(), n, n, 1, w)
  for _ in range(2):
    one_gpu()
  t1, _ = cx.timed(one_gpu, reps)
  out["one_gpu_ms"] = t1
  best, parity = t1, True
  if world > 1:
    L = n // world
    g = world.bit_length() - 1
    rho = int(format(rank, "0%db" % g)[::-1], 2) if g else 0
    mine = x[rank::world].contiguous()            # cyclic shard: rank r holds x[r + G m]
    want = ref[rho::world].contiguous()           # dist output: rank r holds X[K], K mod G = bitrev(r)
    del x, ref
    torch.cuda.empty_cache()
    for _ in range(2):
      o = sd.dist_ntt(eng, mine, w)
    t_nccl, o = cx.timed(lambda: sd.dist_ntt(eng, mine, w), reps)
    ok_nccl = cx.all_true(torch.equal(o, want))
    out["nccl_all_to_all_ms"], out["nccl_timed_output_equals_one_gpu"] = t_nccl, ok_nccl
    parity = parity and ok_nccl
    best_n = t_nccl
    del o
    try:
      fs = sd.FourStepP2P(eng, L, dev)
      for _ in range(2):
        o = fs.ntt(mine, w)
      t_p2p, o = cx.timed(lambda: fs.ntt(mine, w), reps)
      ok_p2p = cx.all_true(torch.equal(o, want))
      out["fused_p2p_ms"], out["fused_p2p_timed_output_equals_one_gpu"] = t_p2p, ok_p2p
      parity = parity and ok_p2p
      if ok_p2p:
        best_n = min(best_n, t_p2p)
      # where the time goes: phase 0 alone (local), phase 0 with the fused exchange, phase 1
      y = mine.clone()
      t_p0, _ = cx.timed(lambda: eng.ntt_dist_phase(0, y.data_ptr(), y.data_ptr(), L, 1, L, w, world, rank, False), reps)

      def p0_p2p():
        fs.hdl.barrier(channel=0)
        eng.ntt_dist_phase0_p2p(y.data_ptr(), L, w, world, rank, fs.ptrs, False)
        fs.hdl.barrier(channel=1)
      t_p0x, _ = cx.timed(p0_p2p, reps)
      o2 = torch.empty_like(mine)
      t_p1, _ = cx.timed(lambda: eng.ntt_dist_phase(2, fs.recv.data_ptr(), o2.data_ptr(), L, 1, L, w, world, rank, False), reps)
      out["phase0_local_ms"], out["phase0_with_fused_exchange_ms"], out["phase1_ms"] = t_p0, t_p0x, t_p1
      out["exchange_bytes_out_per_rank"] = L * 32 * (world - 1) // world
      out["limiter"] = ("phase 0 compute (integer pipes); the exchange adds %.2f ms on top of it at %d GPUs "
                        "(%.0f MiB out per rank over NVLink)" % (max(0.0, t_p0x - t_p0), world,
                                                                 L * 32 * (world - 1) / world / 2**20))
      del fs, y, o, o2
    except Exception as ex:  # pragma: no cover
      out["fused_p2p_error"] = repr(ex)[:300]
    best = best_n
    out["strong_scaling_efficiency"] = t1 / (world * best)
  line["ntt_2^26_ms"] = best
  line["ntt_2^26_melem_per_s"] = n / (best * 1e-3) / 1e6
  line["ntt_2^26_parity_ok"] = bool(parity)
  line["ntt_2^26_strong_scaling_efficiency"] = out.get("strong_scaling_efficiency", 1.0)
  line["ntt_2^26"] = out
  torch.cuda.empty_cache()


def section_config5(cx, line):
  """Fibonacci AIR, 2^20 steps, 8x blowup, one GPU (rank 0's; other ranks idle): trace on the
  device, proof, verification."""
  torch, eng = cx.torch, cx.eng
  import numpy as np
  from starks_b200.limbs import ints_to_limbs
  from starks_b200.modp import IntegersModP
  from starks_b200.stark import STARK
  from starks_b200.air import witness_limbs, witness_device
  out = {}
  eng.set_stream(0)
  psteps = 1 << 20
  F = IntegersModP(P)
  fib = [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}]
  bnd = [(0, 0, 0), (0, 1, 1)]
  wpin = eng.pinned((2, psteps, 8))
  t0 = time.perf_counter()
  witness = witness_limbs(F, [0, 1], psteps, 2, fib, engine=eng, out=wpin.array)
  out["trace_generate_host_s"] = time.perf_counter() - t0
  a, b = 0, 1
  for _ in range(psteps - 1):
    a, b = b, (a + b) % P
  assert ints_to_limbs([a, b]).tolist() == witness[:, -1, :].tolist(), "generated trace differs from the plain recurrence"
  # the same trace generated on the device (chunk starts from powers of the companion matrix)
  d_w = witness_device(F, [0, 1], psteps, 2, fib, engine=eng)
  eng.sync()
  best = None
  for _ in range(3):   # the first repetition may pay a cudaMalloc of the 64 MiB witness buffer
    t0 = time.perf_counter()
    d_w2 = witness_device(F, [0, 1], psteps, 2, fib, engine=eng)
    eng.sync()
    dt = time.perf_counter() - t0
    best = dt if best is None else min(best, dt)
    if _ < 2:
      d_w2.free()
  out["trace_generate_device_s"] = best
  assert (d_w2.download((2, psteps, 8)) == witness).all(), "device trace differs from the host recurrence"
  d_w2.free()
  S = STARK(F, psteps, 8, 2, fib, engine=eng)
  for _ in range(2):  # warm-up: tables, buffer pool, first-use transients
    S.mk_proof(witness, bnd)
  t0 = time.perf_counter()
  for _ in range(3):
    proof = S.mk_proof(witness, bnd)
  out["proof_s"] = (time.perf_counter() - t0) / 3
  out["proof_phases_ms"] = {k: round(v, 2) for k, v in S.timings.items() if k.endswith("_ms")}
  t0 = time.perf_counter()
  d_w3 = witness_device(F, [0, 1], psteps, 2, fib, engine=eng)
  proof_dev = S.mk_proof(d_w3, bnd)
  out["trace_plus_proof_device_resident_s"] = time.perf_counter() - t0
  assert proof_dev == proof, "proof from the device-generated trace differs"
  t0 = time.perf_counter()
  assert S.verify_proof(proof, witness, bnd)
  out["verify_s"] = time.perf_counter() - t0
  out["fri_layers"] = len(proof[3])
  d_w.free()
  d_w3.free()
  wpin.free()
  line["stark_proof_s_fib_2^20_steps_x8"] = out["proof_s"]
  line["stark_proof"] = out


def section_config5_sharded(cx, line, reps=3):
  """ONE proof over the N GPUs of this run (dist.ShardedProver) next to the same proof on one GPU:
  the Fibonacci AIR of config 5 (w = 2: six committed columns, little to shard) and an 8-wide affine
  AIR (24 committed columns over a 2^21-point domain), where the column split has something to divide."""
  torch, eng, world, rank, dev = cx.torch, cx.eng, cx.world, cx.rank, cx.dev
  from starks_b200 import dist as sd
  from starks_b200.air import witness_device
  from starks_b200.modp import IntegersModP
  from starks_b200.stark import STARK
  F = IntegersModP(P)
  out = {"witness": "device-resident on every rank (air.witness_device), for the one-GPU and the sharded prover alike"}
  unit = lambda k, w: tuple(1 if i == k else 0 for i in range(w))
  cases = [("fib_w2_2^20", 1 << 20, 2, [{(0, 1): 1}, {(1, 0): 1, (0, 1): 1}], [0, 1]),
           ("affine_w8_2^18", 1 << 18, 8, [{unit(j, 8): 1, unit((j + 1) % 8, 8): 1} for j in range(8)],
            list(range(1, 9)))]
  for tag, steps, width, sp, inp in cases:
    res = {"steps": steps, "width": width, "committed_columns": 3 * width, "domain": steps * 8}
    eng.set_stream(0)
    wit = witness_device(F, inp, steps, width, sp, engine=eng)   # device-resident witness on every rank
    eng.sync()
    bnd = [(0, j, inp[j]) for j in range(width)]
    S = STARK(F, steps, 8, width, sp, engine=eng)
    for _ in range(2):
      want = S.mk_proof(wit, bnd)
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
      S.mk_proof(wit, bnd)
    res["one_gpu_ms"] = cx.tmax((time.perf_counter() - t0) / reps * 1e3)
    prover = sd.ShardedProver(eng, F, steps, 8, width, sp, dev)
    for _ in range(2):
      got = prover.mk_proof(wit, bnd)
    res["equals_one_gpu_proof"] = cx.all_true(got == want if rank == 0 else True)
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
      prover.mk_proof(wit, bnd)
    torch.cuda.synchronize()
    res["sharded_ms"] = cx.tmax((time.perf_counter() - t0) / reps * 1e3)
    res["speedup_vs_one_gpu"] = res["one_gpu_ms"] / res["sharded_ms"]
    res["rank0_phases_ms"] = {k: round(v, 2) for k, v in prover.timings.items() if k.endswith("_ms")}
    out[tag] = res
    del prover
    wit.free()
    torch.cuda.empty_cache()
  line["stark_proof_sharded"] = out
  line["stark_proof_sharded_ms_fib_2^20_steps_x8"] = out["fib_w2_2^20"]["sharded_ms"]
  line["stark_proof_sharded_parity_ok"] = all(v["equals_one_gpu_proof"] for v in out.values() if isinstance(v, dict))


# ------------------------------------------------------------------ CPU legs

def cpu_port_baseline(cols_sample, threads):
  """Times the oracle (C port of starks/fft.py:303-331) on `cols_sample` columns of 2^20."""
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import oracle as orc
  w = pow(7, (P - 1) // N, P)
  data = synth_columns(cols_sample, N, 1234)
  t0 = time.perf_counter()
  orc.fft_limbs(P, w, data, N, nthreads=threads)
  dt = time.perf_counter() - t0
  return cols_sample * N / dt / 1e6, dt


def cpu_python_reference(budget_s=150.0):
  """The pure-Python reference itself (staged under baseline/_ref, FRI restored in memory),
  one core: fft_1d 2^10..2^16, merkelize 2^16, mk_proof at 1024 steps (BASELINE config 1)."""
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import pyref
  if not pyref.available():
    return None
  out = {}
  with pyref.quiet():
    pyref.load()
    from starks.modp import IntegersModP
    from starks.fft import fft_1d
    from starks.merkle_tree import merkelize
    F = IntegersModP(P)
    t_start = time.perf_counter()
    for logn in (10, 12, 14, 16):
      n = 1 << logn
      w = F(7)**((P - 1) // n)
      vals = [F((i * 2654435761 + 12345) % P) for i in range(n)]
      t0 = time.perf_counter()
      ev = fft_1d(F, vals, P, w)
      dt = time.perf_counter() - t0
      out["fft_1d_2^%d_s" % logn] = dt
      out["fft_1d_2^%d_melem_per_s" % logn] = n / dt / 1e6
    t0 = time.perf_counter()
    merkelize(ev)
    out["merkelize_2^16_s"] = time.perf_counter() - t0
    if time.perf_counter() - t_start < budget_s:
      from starks.utils import generate_Xi_s
      from starks.air import get_computational_trace
      import starks.stark as us
      steps = 1024
      Xs = generate_Xi_s(F, 2)
      sp = [Xs[1], Xs[0] + Xs[1]]
      trace, _ = get_computational_trace([F(0), F(1)], steps, 2, sp)
      witness = [[trace[i][j] for i in range(steps)] for j in range(2)]
      bnd = [(0, 0, F(0)), (0, 1, F(1))]
      S = us.STARK(F, steps, 8, 2, sp)
      t0 = time.perf_counter()
      proof = S.mk_proof(witness, bnd)
      out["mk_proof_1024_steps_s"] = time.perf_counter() - t0
      t0 = time.perf_counter()
      assert S.verify_proof(proof, witness, bnd)
      out["verify_proof_1024_steps_s"] = time.perf_counter() - t0
  return out


def run_reference(args, rank, world):
  """The CPU arm.  Same metric / unit / workload name as ours; every step is a bounded sample of
  the 64-column step: one 2^20 column per host thread."""
  if rank != 0:
    return
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import oracle as orc
  orc.build()
  threads = host_threads()
  cols = max(1, min(threads, args.cols))
  w = pow(7, (P - 1) // N, P)
  data = synth_columns(cols, N, 99)
  steps, warm = max(1, args.steps), max(0, args.warmup)
  t0 = time.perf_counter()
  orc.fft_limbs(P, w, data, N, nthreads=threads)          # calibration step (untimed, counts as warm-up)
  per_step = time.perf_counter() - t0
  budget = 150.0
  if per_step * (steps + warm) > budget:                  # keep the whole arm within a few minutes
    cols = max(1, int(cols * budget / (per_step * (steps + warm))))
    data = data[:cols]
  for _ in range(max(0, warm - 1)):
    orc.fft_limbs(P, w, data, N, nthreads=threads)
  t0 = time.perf_counter()
  for _ in range(steps):
    orc.fft_limbs(P, w, data, N, nthreads=threads)
  dt = (time.perf_counter() - t0) / steps
  val = cols * N / dt / 1e6
  line = {
      "impl": "reference", "metric": "ntt_melem_per_s_2^20", "value": val, "unit": "Melem/s", "n_gpus": args.gpus,
      "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True,
      "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (256-bit modular integers)", "data": "synthetic",
      "config": bench_config(args.cols, max(1, args.gpus)),
      "reference_note": "the reference is pure Python and single-threaded (fft_1d at 2^20 = 74 s per column, "
                        "BASELINE.md); this arm is the C oracle port of fft_1d on %d host threads "
                        "(os.sched_getaffinity, not OMP_NUM_THREADS); each step is a bounded sample of the "
                        "workload: %d of its columns, one per thread" % (threads, cols),
      "cpu_baseline": {"value": val, "unit": "Melem/s", "cores": threads, "kind": "port",
                       "sample": "%d columns x 2^20 per step, %d steps after %d warm-up" % (cols, steps, warm)},
      "e2e": {"value": val, "unit": "Melem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ main

def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours")
  ap.add_argument("--cols", type=int, default=64)
  ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline legs")
  ap.add_argument("--no-e2e", action="store_true")
  ap.add_argument("--no-extras", action="store_true", help="skip configs 3, 4, 5 (LDE+commit, 2^26 NTT, full proof)")
  ap.add_argument("--no-pyref", action="store_true", help="skip the pure-Python reference timings (~80 s)")
  ap.add_argument("--dump-outputs", metavar="DIR",
                  help="write a fixed sample of the last timed step's NTT output to DIR/*.npy (rank 0)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl == "reference":
    ap.error("--dump-outputs applies to the GPU implementation only")
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if args.impl == "reference":
    run_reference(args, rank, world)
    return
  warmup = max(args.warmup, 3)

  import numpy as np
  import torch
  import torch.distributed as dist
  from starks_b200 import Engine

  torch.cuda.set_device(local)
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
  eng = Engine(local)
  stream = torch.cuda.Stream(device=local)
  eng.set_stream(stream.cuda_stream)
  cx = Ctx(torch, dist, eng, stream, rank, world, local)
  cols = args.cols
  w = pow(7, (P - 1) // N, P)

  host_in = eng.pinned((cols, N, 8))
  host_out = eng.pinned((cols, N, 8))
  host_in.array[...] = synth_columns(cols, N, 1000 + rank)
  d_in = torch.empty((cols, N, 8), dtype=torch.int32, device="cuda:%d" % local)
  d_out = torch.empty_like(d_in)
  with torch.cuda.stream(stream):
    d_in.copy_(torch.from_numpy(host_in.array.view(np.int32)), non_blocking=True)
  stream.synchronize()

  def step():
    eng.ntt(d_in.data_ptr(), N, N, d_out.data_ptr(), N, N, cols, w)

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for _ in range(warmup):
    step()
  barrier()
  sampler = ClockSampler(local)
  sampler.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  with torch.cuda.stream(stream):
    e0.record(stream)
    for _ in range(args.steps):
      step()
    e1.record(stream)
  barrier()
  ms = e0.elapsed_time(e1)
  clocks = sampler.stop()
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, torch, d_out)
  # e2e through the host-buffer API
  e2e_s, pcie_duplex = None, None
  if not args.no_e2e:
    e2e_steps = max(1, min(args.steps, 5))
    eng.ntt_host(host_in.array, N, w, out=host_out.array)  # warm
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
      eng.ntt_host(host_in.array, N, w, out=host_out.array)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    barrier()  # all ranks copy at once, like the e2e steps: the host side is shared
    pcie_duplex = pcie_duplex_ceiling(torch, local)
  if world > 1:
    t = torch.tensor([ms, e2e_s or 0.0], dtype=torch.float64, device="cuda:%d" % local)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_max = float(t[0]), float(t[1])
    e2e_s = e2e_max if e2e_s is not None else None
  # ---- parity of the TIMED output (not timed)
  parity = {}
  with torch.cuda.stream(stream):
    back = torch.empty_like(d_in)
    eng.ntt(d_out.data_ptr(), N, N, back.data_ptr(), N, N, cols, w, inverse=True)
    ok_rt = bool(torch.equal(back, d_in))
    del back
  parity["inverse_round_trip_all_columns"] = cx.all_true(ok_rt)
  assert parity["inverse_round_trip_all_columns"], "timed NTT output failed the inverse round trip"
  if e2e_s is not None:
    got_host = torch.from_numpy(host_out.array.view(np.int32))
    parity["e2e_output_equals_device_output"] = cx.all_true(bool(torch.equal(got_host, d_out.cpu())))
    assert parity["e2e_output_equals_device_output"]
  if rank == 0 and not args.no_cpu:
    # the oracle's fft_1d on 4 of the 64 timed columns, element for element
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    import hashlib
    pick = sorted(set([0, cols // 3, (2 * cols) // 3, cols - 1]))
    want = orc.fft_limbs(P, w, host_in.array[pick], N, nthreads=min(len(pick), host_threads()))
    got = d_out[pick].cpu().numpy().view(np.uint32)
    parity["oracle_columns_checked"] = pick
    parity["timed_output_equals_oracle"] = bool((got == want).all())
    parity["digest_all_output_columns"] = hashlib.blake2s(d_out.cpu().numpy().tobytes()).hexdigest()
    assert parity["timed_output_equals_oracle"], "timed NTT output differs from the oracle"
  torch.cuda.empty_cache()

  line = {}
  if rank == 0:
    ms_step = ms / args.steps
    elems = world * cols * N
    value = elems / (ms_step * 1e-3) / 1e6
    hbm_peak, peak_src = peaks()
    launches_per_step = 2  # 2^20 = two radix-2^10 passes of ntt_pass_kernel
    alg_bytes = BYTES_PER_ELEM * cols * N + 16 * N
    hbm_achieved = alg_bytes / (ms_step * 1e-3) / 1e9
    butterflies = cols * (N // 2) * LOGN
    int_ops = INT_OPS_PER_BUTTERFLY * butterflies
    mb = {}
    try:
      eng.set_stream(0)
      for which, name in ((7, "imad_iadd3_mixed_gops"), (0, "imad_gops"), (10, "imad_wide_carry_rows_gops"),
                          (6, "butterfly_gops"), (5, "field_mul_gops")):
        best = 0.0
        for _ in range(2):
          mms, ops = eng.microbench(which, 4000 if which not in (5, 6) else 1000)
          best = max(best, ops / (mms * 1e-3) / 1e9)
        mb[name] = best
      for variant in (1, 2, 3):   # experimental multiply (csrc/field_exp.cuh), A/B in registers
        for which, nm in ((5, "mul"), (6, "butterfly")):
          mms, ops, bad = eng.microbench_variant(variant, which, 1000)
          mb["exp_variant%d_%s_gops" % (variant, nm)] = ops / (mms * 1e-3) / 1e9
          mb["exp_variant%d_%s_mismatches" % (variant, nm)] = bad
    except Exception as ex:  # pragma: no cover
      mb["error"] = str(ex)
    int_peak = mb.get("imad_iadd3_mixed_gops")
    int_achieved = int_ops / (ms_step * 1e-3) / 1e9
    line.update({
        "metric": "ntt_melem_per_s_2^20", "value": value, "unit": "Melem/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32x8 (256-bit modular integers)", "data": "synthetic",
        "config": bench_config(cols, world),
        "clocks": clocks,
        "gpu_launches": args.steps * launches_per_step,
        "roofline": {"bound": "int32", "achieved": int_achieved / 1e3, "peak": (int_peak or 0) / 1e3, "unit": "Tops/s",
                     "frac": (int_achieved / int_peak) if int_peak else None,
                     "traffic": NCU_TRAFFIC_BYTES_PER_LAUNCH,
                     "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch, " + NCU_SOURCE,
                     "kernel": "ntt_pass_kernel<StarkField>", "launches_per_step": launches_per_step,
                     "alg_int32_ops_per_step": int_ops, "alg_int32_ops_per_launch": int_ops / launches_per_step,
                     "peak_source": "K0 microbenchmark of this run (IMAD + IADD3 on independent chains, dual issue); "
                                    "MEASURED_PEAKS.json carries no integer figure",
                     "butterflies_per_s_g": butterflies / (ms_step * 1e-3) / 1e9,
                     "in_register_butterfly_peak_g": mb.get("butterfly_gops"),
                     "frac_of_in_register_butterfly": (butterflies / (ms_step * 1e-3) / 1e9 / mb["butterfly_gops"]) if mb.get("butterfly_gops") else None,
                     "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                             "alg_bytes_per_launch": alg_bytes / launches_per_step, "alg_bytes_per_step": alg_bytes,
                             "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)"},
                     "binding_pipe": {
                         "name": "fmaheavy: IMAD.WIDE.U32(.X), the half-rate 32x32+64 multiply-add (4 clk per warp instruction)",
                         "wide_macs_per_butterfly": WIDE_MACS_PER_BUTTERFLY,
                         "achieved_wide_macs_tops": WIDE_MACS_PER_BUTTERFLY * butterflies / (ms_step * 1e-3) / 1e12,
                         "peak_wide_macs_tops": (mb.get("imad_wide_carry_rows_gops") or 0) / 1e3,
                         "frac": (WIDE_MACS_PER_BUTTERFLY * butterflies / (ms_step * 1e-3) / 1e9 / mb["imad_wide_carry_rows_gops"])
                         if mb.get("imad_wide_carry_rows_gops") else None,
                         "ncu_pipe_fmaheavy_cycles_active_pct": list(NCU_FMAHEAVY_ACTIVE_PCT),
                         "note": "ncu (" + NCU_SOURCE + "): the pipe is 72 % / 70 % active in the two passes -- the multiply-adds plus the "
                                 "moves ptxas places on the same pipe; ALU pipe 46 %, issue slots 49 %, DRAM 12 %"},
                     "microbench": mb,
                     "note": "256-bit modular butterflies: ~41 int32 op per byte against a machine balance of ~4.7, so "
                             "the integer pipes bind and HBM is ~12 % busy (ncu)"},
        "parity": parity,
    })
    if e2e_s is not None:
      line["e2e"] = {"value": elems / e2e_s / 1e6, "unit": "Melem/s", "h2d_bytes_per_step": cols * N * 32,
                     "d2h_bytes_per_step": cols * N * 32, "ms_per_step": e2e_s * 1e3,
                     "gb_per_s_each_way": cols * N * 32 / e2e_s / 1e9,
                     "pcie_duplex_plain_copies_gb_per_s_each_way": pcie_duplex,
                     "host_ceiling": "plain pinned copies both ways at once, measured in this run with all %d ranks "
                                     "copying together: %.1f GB/s each way per GPU; %s" % (world, pcie_duplex or 0.0, numa_note()),
                     "note": "host-buffer API (stk_ntt_host): three-slot H2D / transform / D2H pipeline; bound by the "
                             "host link, not by a kernel"}
  del d_in, d_out
  host_in.free()
  host_out.free()
  torch.cuda.empty_cache()
  eng.set_stream(0)
  if not args.no_extras:
    with Watchdog(480, rank, line, "the multi-GPU sections (configs 3, 4 and 5)"):
      secs = [("lde_merkle_commit", section_config3), ("ntt_2^26", section_config4)]
      if world > 1:
        secs.append(("stark_proof_sharded", section_config5_sharded))
      for name, fn in secs:
        try:
          fn(cx, line)
        except Exception as ex:  # pragma: no cover
          import traceback
          line[name + "_error"] = traceback.format_exc()[-500:]
    if rank == 0 and world == 1:
      try:
        section_config5(cx, line)
      except Exception as ex:  # pragma: no cover
        import traceback
        line["stark_proof_error"] = traceback.format_exc()[-500:]
  if rank == 0:
    if world == 1 and not args.no_cpu:
      v, dt = cpu_port_baseline(4, 1)
      cb = {"value": v, "unit": "Melem/s", "cores": 1, "kind": "port",
            "sample": "4 columns x 2^20, one pass, %.1f s" % dt,
            "note": "C oracle port of fft_1d (oracle/starks_oracle.c), one thread"}
      if not args.no_pyref:
        try:
          py = cpu_python_reference()
        except Exception as ex:  # pragma: no cover
          py = {"error": repr(ex)[:200]}
        if py and "fft_1d_2^16_melem_per_s" in py:
          cb = {"value": py["fft_1d_2^16_melem_per_s"], "unit": "Melem/s", "cores": 1, "kind": "reference",
                "sample": "the pure-Python reference (baseline/_ref, unmodified; FRI restored in memory): fft_1d at "
                          "2^10..2^16 (2^16 is the value; 2^20 takes 74 s), merkelize 2^16, mk_proof + verify_proof "
                          "at 1024 steps",
                "python_reference": py, "host_threads_available": host_threads(),
                "port": {"value": v, "unit": "Melem/s", "cores": 1,
                         "sample": "C oracle port, 4 columns x 2^20, one pass, %.1f s" % dt}}
        elif py:
          cb["python_reference"] = py
      line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
  main()
