"""Cost of the exact full-catalogue rank (srfrd_catalogue_rank) against the top-k it replaces for metrics, single GPU.

U = 16 384 users x N = 1 000 000 items x D = 64 (the whole table), and one 125 000-row shard (a rank's work at 8 GPUs).
The rank call's cost depends on how many ranking units reach the target's score, so it is timed for three targets:
  top1     each user's own top-1 item (rank 0)
  rank500  the item at rank ~500 of each user (a trained model's regime)
  random   a uniformly random item (an untrained model's regime: ranks around N / 2)
next to srfrd_catalogue_topk at k = 10 and k = 64, in the same rounds.  Per case: the library call alone (kernel; for the
rank: the zeroing of rank_out + the streaming kernel) and the Python entry point end to end (catalogue_ranks: target
validation, gather of the target rows, bf16 split of the features, the call; local_topk: split, both phases, merge).
CUDA events around enough passes for a window of >= 1 s after a warm-up; the cases run alternately, in `--rounds`
rounds; median and range over the rounds.  Inputs are Gaussian; the table (128 MB in bf16) is larger than L2.  The
targets of top1 / rank500 come from a chunked fp32 torch matmul of the bf16-rounded operands (setup only, not timed).

    python tools/bench_catalogue_rank.py [--rounds 5] [--window 1.0] [--out profiles/r6_catalogue_rank.json]
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

bf16 = torch.bfloat16


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


def pick_targets(feats, table, ranks=(0, 500), chunk=512):
    """per user, the item at each 0-based rank of `ranks` under the bf16-rounded operands (fp32 matmul, ties by id)"""
    f = feats.to(bf16).float()
    t = table[1:].to(bf16).float()
    out = {r: [] for r in ranks}
    for s in range(0, f.shape[0], chunk):
        sc = f[s:s + chunk] @ t.T
        _, idx = torch.topk(sc, max(ranks) + 1, dim=1, sorted=True)
        for r in ranks:
            out[r].append(idx[:, r] + 1)
        del sc
    return {r: torch.cat(v) for r, v in out.items()}


class RankCase:
    def __init__(self, feats, index, table, target):
        self.feats, self.index, self.table, self.target = feats, index, table, target
        U = feats.shape[0]
        self.fb, self.u_pad = EV._split_feats(feats, index.Dp, 1)
        self.rows = torch.zeros(U, index.Dp, dtype=bf16, device="cuda")
        ops.f32_to_bf16_split(table, self.rows[:, :index.D], None, row_index=target)
        self.rank = torch.empty(U, dtype=torch.int32, device="cuda")

    def kernel(self):
        ops.catalogue_rank(self.fb, self.feats.shape[0], self.u_pad, 1, self.index.table, self.index.row_lo,
                           self.index.id_base, self.rows, self.target, self.rank)

    def end_to_end(self):
        EV.catalogue_ranks(self.feats, self.index, self.table, self.target)


class TopkCase:
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

    def end_to_end(self):
        EV.local_topk(self.feats, self.index, 1, self.k)


def measure(cases, rounds, window_s):
    names = ("kernel", "end_to_end")
    fns = {(c, n): getattr(case, n) for c, case in cases.items() for n in names}
    passes = {}
    for key, fn in fns.items():                           # warm-up, then size each window to >= window_s
        for _ in range(3):
            fn()
        ms = timed(fn, 5)
        passes[key] = max(10, int(window_s * 1e3 / max(ms, 1e-3)) + 1)
    res = {key: [] for key in fns}
    for _ in range(rounds):
        for c in cases:                                   # cases alternate within every round
            for n in names:
                res[(c, n)].append(timed(fns[(c, n)], passes[(c, n)]))
    out = {}
    for c in cases:
        out[c] = {n + "_ms": {"median": round(float(np.median(res[(c, n)])), 4), "min": round(min(res[(c, n)]), 4),
                              "max": round(max(res[(c, n)]), 4), "passes": passes[(c, n)]} for n in names}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--users", type=int, default=16384)
    ap.add_argument("--items", type=int, default=1_000_000)
    ap.add_argument("--out", default="profiles/r6_catalogue_rank.json")
    a = ap.parse_args()
    D = 64
    g = torch.Generator().manual_seed(0)
    feats = torch.randn(a.users, D, generator=g).cuda()
    table = (torch.randn(a.items + 1, D, generator=g) * 0.05).cuda()
    picked = pick_targets(feats, table)
    targets = {"top1": picked[0], "rank500": picked[500],
               "random": torch.randint(1, a.items + 1, (a.users,), generator=g).cuda()}
    shard_rows = (a.items + 1 + 7) // 8
    result = {"device": gpu_info(), "users": a.users, "items": a.items, "D": D, "rounds": a.rounds,
              "window_s": a.window, "timing": "CUDA events around back-to-back passes; median / min / max over rounds",
              "targets": {}, "configs": {}}
    full = EV.CatalogueIndex(table, 0)
    for name, t in targets.items():                       # the ranks the three target choices actually have
        r = EV.catalogue_ranks(feats, full, table, t).double()
        result["targets"][name] = {"rank_median": float(r.median()), "rank_mean": round(float(r.mean()), 1),
                                   "rank_max": float(r.max())}
    print("targets", json.dumps(result["targets"]), flush=True)
    for name, index in (("full_table", full),
                        ("shard_125k", EV.CatalogueIndex(table[shard_rows:2 * shard_rows].contiguous(), shard_rows))):
        cases = {"rank_" + tn: RankCase(feats, index, table, t) for tn, t in targets.items()}
        cases.update({"topk_%d" % k: TopkCase(feats, index, k) for k in (10, 64)})
        result["configs"][name] = {"rows": index.n_rows, "cases": measure(cases, a.rounds, a.window)}
        print(name, json.dumps(result["configs"][name]["cases"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
