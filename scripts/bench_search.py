"""Exact flat search on one GPU: grafp_b200.search.FingerprintIndex against the exact torch path, and
evaluate_sequences end to end.

Databases of unit rows (d = 128) are generated on the device.  Per (n_db, n_q, k): the median of --reps timed searches
(CUDA events, after a warm-up) of ours and of the torch path - fp32 distances (TF32 off) |q|^2 - 2 q.x + |x|^2 over
row chunks, torch.topk per chunk and over the chunk winners - alternating in the same process, with:
  * algorithmic TFLOP/s: 2 n_q n_db d over our time;
  * tensor work issued: three fp16 MMAs per product (hi/lo split), queries padded to the 128-row MMA tile, and
    ceil(k / 16) passes over the database for k > 16;
  * database bytes per pass (fp16 hi + lo planes + |x|^2) x passes over our time, against HBM's 7.7 TB/s.
Every database is larger than the 126 MB L2.  The card's name and power limit are read in the same run.

  python scripts/bench_search.py --out bench_search.jsonl
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from grafp_b200.search import FingerprintIndex, evaluate_sequences  # noqa: E402

HBM_TBS = 7.7


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [v.strip() for v in out[0].split(",")] if out else ("unknown", "unknown", "unknown")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def build_index(n_db: int, d: int, seed: int, dev) -> FingerprintIndex:
    index = FingerprintIndex(d, dev)
    index._reserve(n_db)   # one allocation at the final size instead of geometric growth
    g = torch.Generator(device=dev).manual_seed(seed)
    step = 1 << 22
    for r0 in range(0, n_db, step):
        m = min(step, n_db - r0)
        index.add(torch.nn.functional.normalize(torch.randn(m, d, generator=g, device=dev), dim=1))
    return index


def torch_search(R: torch.Tensor, sq: torch.Tensor, q: torch.Tensor, k: int, budget: int = 1 << 33):
    """Exact fp32 search with cuBLAS (TF32 off) + torch.topk, chunked so a chunk's score matrix stays under budget."""
    n_q = q.shape[0]
    qq = (q * q).sum(1, keepdim=True)
    chunk = max(1 << 16, budget // (4 * n_q))
    best_d, best_i = None, None
    for r0 in range(0, R.shape[0], chunk):
        dist = torch.addmm(sq[None, r0:r0 + chunk], q, R[r0:r0 + chunk].T, alpha=-2.0).add_(qq)
        v, i = torch.topk(dist, min(k, dist.shape[1]), dim=1, largest=False)
        i += r0
        if best_d is None:
            best_d, best_i = v, i
        else:
            v, j = torch.topk(torch.cat([best_d, v], 1), k, dim=1, largest=False)
            best_i = torch.gather(torch.cat([best_i, i], 1), 1, j)
            best_d = v
    return best_d, best_i


def time_pair(fa, fb, reps: int, slow_ms: float = 2000.0, slow_reps: int = 3):
    """Alternating CUDA-event timings (ms) of fa and fb after one warm-up call each: medians of `reps` calls, except
    that fb (the torch path) takes `slow_reps` when one call of it exceeds `slow_ms` (seconds per call at the largest
    points; ours keeps `reps`).  Returns (median a, median b, calls of b)."""
    fa()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record(); fb(); e.record()
    e.synchronize()
    reps_b = slow_reps if s.elapsed_time(e) > slow_ms else reps
    ta, tb = [], []
    for r in range(reps):
        for f, acc in ((fa, ta), (fb, tb)):
            if f is fb and r >= reps_b:
                continue
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); f(); e.record()
            e.synchronize()
            acc.append(s.elapsed_time(e))
    return statistics.median(ta), statistics.median(tb), len(tb)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000,50000000")
    ap.add_argument("--nq", default="19,2048,32768")
    ap.add_argument("--k", default="1,20")
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--eval-ids", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_search.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    info = gpu_info()
    lines = []

    def emit(rec):
        rec = {**rec, **info}
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    d = args.d
    for n_db in [int(float(v)) for v in args.sizes.split(",")]:
        t0 = time.time()
        index = build_index(n_db, d, n_db, dev)
        torch.cuda.synchronize()
        emit({"what": "build", "n_db": n_db, "d": d, "add_s": round(time.time() - t0, 3)})
        R = index.rows
        sq = torch.cat([(R[r0:r0 + (1 << 22)] ** 2).sum(1) for r0 in range(0, n_db, 1 << 22)])
        g = torch.Generator(device=dev).manual_seed(1)
        for n_q in [int(v) for v in args.nq.split(",")]:
            q = torch.nn.functional.normalize(torch.randn(n_q, d, generator=g, device=dev), dim=1)
            for k in [int(v) for v in args.k.split(",")]:
                ours_ms, ref_ms, ref_reps = time_pair(lambda: index.search(q, k), lambda: torch_search(R, sq, q, k), args.reps)
                D, I = index.search(q, k)
                Dr, Ir = torch_search(R, sq, q, k)
                agree = float((I[:, 0] == Ir[:, 0]).float().mean())
                passes = 1 if k <= 16 else math.ceil(k / 16)
                flop = 2.0 * n_q * n_db * d
                issued = 3 * 2.0 * math.ceil(n_q / 128) * 128 * n_db * d * passes
                db_bytes = n_db * (2 * d * 2 + 4)
                emit({"what": "search", "n_db": n_db, "n_q": n_q, "k": k, "d": d, "ours_ms": round(ours_ms, 3),
                      "torch_ms": round(ref_ms, 3), "speedup": round(ref_ms / ours_ms, 2),
                      "alg_tflops": round(flop / ours_ms / 1e9, 1), "issued_tflops": round(issued / ours_ms / 1e9, 1),
                      "passes": passes, "db_bytes_per_pass": db_bytes,
                      "hbm_share": round(db_bytes * passes / (ours_ms * 1e-3) / (HBM_TBS * 1e12), 3),
                      "top1_agree_with_torch": agree, "reps": args.reps, "torch_reps": ref_reps})
        if args.eval_ids and n_db == 10_000_000:
            n_ids, L = args.eval_ids, 19
            base = 1234
            query = torch.nn.functional.normalize(R[base:base + n_ids + L] + 0.05 * torch.randn(n_ids + L, d, generator=g, device=dev), dim=1)
            evaluate_sequences(index, query, list(range(100)), gt_offset=base)   # warm-up
            torch.cuda.synchronize()
            t0 = time.time()
            res = evaluate_sequences(index, query, list(range(n_ids)), gt_offset=base)
            torch.cuda.synchronize()
            emit({"what": "evaluate_sequences", "n_db": n_db, "test_ids": n_ids, "seq_lens": res["seq_lens"],
                  "seconds": round(time.time() - t0, 3), "top1_exact": [round(float(v), 2) for v in res["top1_exact"]]})
        del index, R, sq
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
