"""Cost of the full-catalogue top-k as k grows, single GPU.

U = 16 384 users x N = 1 000 000 items x D = 64 (the whole table), and one 125 000-row shard (a rank's work at 8 GPUs),
for k in {10, 20, 50, 64}.  Per k: srfrd_catalogue_topk (both phases), the same call with SRFRD_TOPK_DEBUG=2 (phase 1
alone; phase 2 = the difference) and evaluation.local_topk end to end (bf16 split of the features + both phases + the
merge).  CUDA events around enough passes for a window of >= 1 s after a warm-up; the k values run alternately, in
`--rounds` rounds; median and range over the rounds.  Inputs are Gaussian; the table (128 MB) is larger than L2.

    python tools/bench_topk_k.py [--rounds 5] [--window 1.0] [--out profiles/r5_topk_k.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from srfrd_b200 import evaluation as EV, ops

KS = (10, 20, 50, 64)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


class Case:
    def __init__(self, feats, index, k):
        self.feats, self.index, self.k = feats, index, k
        U = feats.shape[0]
        L = EV.list_len(k)
        self.fb, self.u_pad = EV._split_feats(feats, index.Dp, 1)
        self.chunks = ops.catalogue_topk_plan(U, index.n_rows, index.row_lo, index.Dp, 1, k)
        self.ps = torch.empty(U, self.chunks, L, dtype=torch.float32, device="cuda")
        self.pi = torch.empty(U, self.chunks, L, dtype=torch.int32, device="cuda")

    def kernel(self):
        ops.catalogue_topk(self.fb, self.feats.shape[0], self.u_pad, 1, self.index.table, self.index.row_lo,
                           self.index.id_base, self.chunks, self.ps, self.pi, None, k=self.k)

    def phase1(self):
        os.environ["SRFRD_TOPK_DEBUG"] = "2"
        try:
            self.kernel()
        finally:
            del os.environ["SRFRD_TOPK_DEBUG"]

    def end_to_end(self):
        EV.local_topk(self.feats, self.index, 1, self.k)


def measure(cases, rounds, window_s):
    fns = {(k, name): getattr(c, name) for k, c in cases.items() for name in ("kernel", "phase1", "end_to_end")}
    passes = {}
    for key, fn in fns.items():                           # warm-up, then size each window to >= window_s
        for _ in range(3):
            fn()
        ms = timed(fn, 5)
        passes[key] = max(10, int(window_s * 1e3 / max(ms, 1e-3)) + 1)
    res = {key: [] for key in fns}
    for _ in range(rounds):
        for k in cases:                                   # k values alternate within every round
            for name in ("kernel", "phase1", "end_to_end"):
                res[(k, name)].append(timed(fns[(k, name)], passes[(k, name)]))
    out = {}
    for k in cases:
        row = {}
        for name in ("kernel", "phase1", "end_to_end"):
            v = res[(k, name)]
            row[name + "_ms"] = {"median": round(float(np.median(v)), 4), "min": round(min(v), 4), "max": round(max(v), 4),
                                 "passes": passes[(k, name)]}
        row["phase2_ms_median"] = round(row["kernel_ms"]["median"] - row["phase1_ms"]["median"], 4)
        out[str(k)] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--users", type=int, default=16384)
    ap.add_argument("--items", type=int, default=1_000_000)
    ap.add_argument("--out", default="profiles/r5_topk_k.json")
    a = ap.parse_args()
    D = 64
    g = torch.Generator().manual_seed(0)
    feats = torch.randn(a.users, D, generator=g).cuda()
    table = (torch.randn(a.items + 1, D, generator=g) * 0.05).cuda()
    shard_rows = (a.items + 1 + 7) // 8
    result = {"device": gpu_info(), "users": a.users, "items": a.items, "D": D, "rounds": a.rounds,
              "window_s": a.window, "timing": "CUDA events around back-to-back passes; median / min / max over rounds",
              "configs": {}}
    for name, index in (("full_table", EV.CatalogueIndex(table, 0)),
                        ("shard_125k", EV.CatalogueIndex(table[shard_rows:2 * shard_rows].contiguous(), shard_rows))):
        cases = {k: Case(feats, index, k) for k in KS}
        result["configs"][name] = {"rows": index.n_rows, "chunks": {str(k): c.chunks for k, c in cases.items()},
                                   "k": measure(cases, a.rounds, a.window)}
        print(name, json.dumps(result["configs"][name]["k"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
