"""Coefficient-form polynomial arithmetic on one GPU (stk_poly_mul, stk_poly_divmod,
stk_poly_compose, stk_poly_eval_multivar), STARK prime.

For n = 2^16 .. 2^22: the product of two polynomials of n coefficients and the division of 2n
coefficients by n; up to --compose-max-log (default 20) also a(b(X)) for a of n coefficients with
b = alpha X, b = alpha X + beta and a 65-coefficient b (n/64 coefficients of a, so that the output
has about n), a ** 8 with a of n/8 coefficients, and the Fibonacci step polynomials
{X2, X1 + X2} evaluated at two polynomials of n coefficients.  Each is timed with a host clock
around calls that end in a device synchronise (median of `--reps` calls after two warm-up calls)
and reported as a multiple of one forward transform of length n timed the same way.  The CPU
oracle's schoolbook routines at 2^14, and composition by Horner's rule through stk_poly_mul (what
Polynomial.__call__ did before it had a device path) at 2^10, are timed once for context.  Prints
one JSON object (card name and power limit included); --out also writes it to a file.

  python tools/gpu_poly_bench.py [--max-log 22] [--reps 5] [--out poly_bench.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

P = 2**256 - 351 * 2**32 + 1


def card():
  q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True)
  name, _, limit = q.stdout.strip().partition(", ")
  return {"name": name, "power_limit": limit}


def rand(rng, n):
  a = rng.integers(0, 2**32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
  a[:, 7] &= 0x7FFFFFFF   # below 2^255 < p
  a[-1, 0] |= 1           # non-zero leading coefficient
  return a


def timed(eng, fn, reps):
  for _ in range(2):
    fn()
  eng.sync()
  ts = []
  for _ in range(reps):
    t0 = time.perf_counter()
    fn()
    eng.sync()
    ts.append(time.perf_counter() - t0)
  return statistics.median(ts) * 1e3


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--min-log", type=int, default=16)
  ap.add_argument("--max-log", type=int, default=22)
  ap.add_argument("--reps", type=int, default=5)
  ap.add_argument("--oracle-log", type=int, default=14)
  ap.add_argument("--compose-max-log", type=int, default=20)
  ap.add_argument("--horner-log", type=int, default=10)
  ap.add_argument("--out")
  args = ap.parse_args()
  from starks_b200 import Engine
  eng = Engine(0)
  rng = np.random.default_rng(0)
  rows = []
  for logn in range(args.min_log, args.max_log + 1):
    n = 1 << logn
    a2, b = rand(rng, 2 * n), rand(rng, n)
    da, db = eng.alloc(a2.nbytes).upload(a2), eng.alloc(b.nbytes).upload(b)
    out, q, r, t = eng.alloc(2 * n * 32), eng.alloc((n + 1) * 32), eng.alloc(n * 32), eng.alloc(n * 32)
    w = pow(7, (P - 1) // n, P)
    ntt_ms = timed(eng, lambda: eng.ntt(db.ptr, n, n, t.ptr, n, n, 1, w), args.reps)
    mul_ms = timed(eng, lambda: eng.poly_mul(da.ptr, n, db.ptr, n, out.ptr), args.reps)
    div_ms = timed(eng, lambda: eng.poly_divmod(da.ptr, 2 * n, db.ptr, n, q.ptr, r.ptr), args.reps)
    row = {"log2n": logn, "ntt_fwd_ms": round(ntt_ms, 4),
           "mul_nxn_ms": round(mul_ms, 4), "mul_in_ntts": round(mul_ms / ntt_ms, 2),
           "divmod_2n_by_n_ms": round(div_ms, 4), "divmod_in_ntts": round(div_ms / ntt_ms, 2)}
    if logn <= args.compose_max_log:
      b2 = rand(rng, 2)
      ax, axb, b65 = eng.alloc(64), eng.alloc(64), eng.alloc(65 * 32).upload(rand(rng, 65))
      ax.upload(np.concatenate([np.zeros((1, 8), np.uint32), b2[1:]]))
      axb.upload(b2)
      na65 = n // 64
      for name, fn in (("compose_ax", lambda: eng.poly_compose(db.ptr, n, ax.ptr, 2, out.ptr)),
                       ("compose_ax_plus_b", lambda: eng.poly_compose(db.ptr, n, axb.ptr, 2, out.ptr)),
                       ("compose_b65_n_over_64", lambda: eng.poly_compose(db.ptr, na65, b65.ptr, 65, out.ptr)),
                       ("pow8_n_over_8", lambda: eng.poly_eval_multivar(db.ptr, [n // 8], n // 8, [(0, 1, (8,))], 1,
                                                                        out.ptr, n - 7)),
                       ("fibonacci_step_at_polys", lambda: eng.poly_eval_multivar(
                           da.ptr, [n, n], n, [(0, 1, (0, 1)), (1, 1, (1, 0)), (1, 1, (0, 1))], 2, out.ptr, n))):
        ms = timed(eng, fn, args.reps)
        row[name + "_ms"], row[name + "_in_ntts"] = round(ms, 4), round(ms / ntt_ms, 2)
      for x in (ax, axb, b65):
        x.free()
    rows.append(row)
    print(json.dumps(rows[-1]), flush=True)
    for x in (da, db, out, q, r, t):
      x.free()
  import oracle as orc
  n = 1 << args.oracle_log
  a2 = [int(x) for x in rng.integers(1, 2**62, size=2 * n)]
  bo = [int(x) for x in rng.integers(1, 2**62, size=n)]
  t0 = time.perf_counter()
  orc.poly_mul(P, a2[:n], bo)
  omul = time.perf_counter() - t0
  t0 = time.perf_counter()
  orc.poly_divmod(P, a2, bo)
  odiv = time.perf_counter() - t0
  # a(b(X)) by Horner's rule through device products, a of 2^horner_log coefficients, b of 2
  from starks_b200.modp import IntegersModP
  from starks_b200.polynomial import polynomials_over
  Poly = polynomials_over(IntegersModP(P))
  ha, hb = Poly(a2[:1 << args.horner_log]), Poly([3, 5])
  t0 = time.perf_counter()
  acc = Poly([])
  for c in reversed(ha.coefficients):
    acc = acc * hb + c
  horner_s = time.perf_counter() - t0
  t0 = time.perf_counter()
  assert ha(hb) == acc
  dev_s = time.perf_counter() - t0
  res = {"card": card(), "field": "stark", "timing": "host clock, median of %d synchronised calls" % args.reps,
         "rows": rows, "oracle_cpu_1thread": {"log2n": args.oracle_log, "mul_nxn_s": round(omul, 3),
                                              "divmod_2n_by_n_s": round(odiv, 3)},
         "compose_ax_plus_b_2_%d" % args.horner_log: {"horner_through_mul_s": round(horner_s, 3),
                                                      "polynomial_call_s": round(dev_s, 4)}}
  print(json.dumps(res))
  if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
      json.dump(res, fh, indent=1)
  eng.close()


if __name__ == "__main__":
  main()
