"""Cost of gSASRec's gBCE objective (FusedTrainer(loss="gbce"), csrc/gbce.cu) next to the BCE and the full-catalogue CE,
single GPU.

Two tables under the C2 workload (SRFR D = 64 + F = 16, 2 blocks, maxlen 50, batch 4096, Beauty-shaped users, soft
discriminator weights, batches drawn by the device sampler inside the step graph):
  C2   N = 12 101 items (the C2 catalogue)
  C5t  N = 150 000 items (the C5 catalogue size; the users and sequence shapes stay C2's)
Per table, the BCE step, the gBCE step at k = 64, 128 and 256 (t = 0.75) and the CE step (trainers from the same initial
parameters) run alternately for `--rounds` rounds of CUDA-event-timed windows of >= `--window` seconds after a warm-up;
median and range over the rounds.  Then the gBCE kernels alone at k = 256 on the last step's operands: the draw (ids,
bf16 rows, exclusion mask), the loss call without dE (the DH pass alone) and the full loss call (DH + DN + scatter).
Achieved TFLOP/s are from shape-derived counts over the M packed rows of the batch (S = h N^T is 2 M k Dp flops; DH adds
X N, DN recomputes S and adds X^T h, each of the same size), not from the padded tiles the kernels compute.

    python tools/bench_gbce.py [--rounds 5] [--window 1.0] [--out profiles/r8_gbce.json]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from srfrd_b200 import ops, synth
from srfrd_b200.losses import gbce_beta
from srfrd_b200.trainer import DeviceSampler, FusedTrainer
from tools.bench_ce import gpu_info, make_model, reps_for, timed

KS = (64, 128, 256)


def bench_table(name, N, rounds, window, B=4096, L=50):
    data = synth.make_interactions(1236, 22363, N, 5, 4.0, L)
    smp = DeviceSampler(data, L, "cuda", seed=1000)
    tr = {"bce": FusedTrainer(make_model(N), use_graph=True)}
    for k in KS:
        tr[f"gbce{k}"] = FusedTrainer(make_model(N), use_graph=True, loss="gbce", num_negatives=k, gbce_t=0.75)
    tr["ce"] = FusedTrainer(make_model(N), use_graph=True, loss="ce")
    steps = {name_: (lambda t=t: t.step_sampled(smp, B, "soft")) for name_, t in tr.items()}
    for f in steps.values():
        for _ in range(5):
            f()
    n = {name_: reps_for(f, window) for name_, f in steps.items()}
    step_ms = {name_: [] for name_ in tr}
    for _ in range(rounds):
        for name_ in tr:
            step_ms[name_].append(timed(steps[name_], n[name_]))
    losses = {name_: float(t.loss_dev) for name_, t in tr.items()}

    # the gBCE kernels alone at k = 256, on the operands the last step used
    t = tr["gbce256"]
    eng, gb, k = t.eng, t._gbce_ws, 256
    plan = eng._plans[(B, L)]
    cap = plan.cap
    M_rows = int(plan.rows[0])
    E = t.P.view(t.spec.item_key)
    pos, w, norm = t._static["pos"].view(-1), t._static["w_pos"].view(-1), t.scal[0:2]
    Dp, D = t.spec.Dp, t.spec.D
    beta = gbce_beta(k, N, 0.75)
    acc = torch.zeros(2, device="cuda")
    dh = torch.zeros(cap, eng._ws["dh"].shape[1], device="cuda")
    dE = torch.zeros(N + 1, D, device="cuda")
    hb = gb["h"][:cap]
    kern = {
        "draw": lambda: ops.gbce_draw(E, gb["ids"], gb["nb"], gb["excl"][:B], t._static["seq"], t._static["pos"],
                                      seed=eng.drop_seed, step=eng.step_state[3:4]),
        "dh_pass": lambda: ops.gbce_loss(hb, gb["nb"], gb["ids"], E, pos, w, norm, gb["excl"], L, beta, acc, dh[:cap], None,
                                         gb["part"], plan),
        "full_loss_call": lambda: ops.gbce_loss(hb, gb["nb"], gb["ids"], E, pos, w, norm, gb["excl"], L, beta, acc,
                                                dh[:cap], dE, gb["part"], plan),
    }
    for f in kern.values():
        f()
    kn = {kk: reps_for(f, window / 2) for kk, f in kern.items()}
    kern_ms = {kk: [] for kk in kern}
    for _ in range(rounds):
        for kk, f in kern.items():
            kern_ms[kk].append(timed(f, kn[kk]))
    med = lambda v: float(np.median(v))
    gemm = 2.0 * M_rows * k * Dp
    work = {"draw": 0.0, "dh_pass": 2 * gemm, "full_loss_call": 4 * gemm}
    out = {
        "table": name, "items": N, "batch": B, "maxlen": L, "packed_rows": M_rows, "Dp": Dp,
        "step_ms": {kk: {"median": med(v), "min": min(v), "max": max(v), "rounds": v} for kk, v in step_ms.items()},
        "minus_bce_ms": {kk: med(v) - med(step_ms["bce"]) for kk, v in step_ms.items() if kk != "bce"},
        "loss_after_warmup_and_timing": losses,
        "kernels_k256": {},
    }
    for kk, v in kern_ms.items():
        out["kernels_k256"][kk] = {"median_ms": med(v), "min_ms": min(v), "max_ms": max(v), "flop": work[kk],
                                   "tflops": work[kk] / (med(v) * 1e-3) / 1e12}
    out["kernels_k256"]["dn_and_scatter_ms"] = med(kern_ms["full_loss_call"]) - med(kern_ms["dh_pass"])
    del tr
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gbce: needs a CUDA device")
    res = {"gpu": gpu_info(), "rounds": args.rounds, "window_s": args.window,
           "workload": "C2 model and users (SRFR 64 + 16, 2 blocks, maxlen 50, batch 4096, soft weights, device sampler)",
           "tables": [bench_table("C2", 12101, args.rounds, args.window), bench_table("C5t", 150000, args.rounds, args.window)]}
    print(f"gpu: {res['gpu']}")
    for t in res["tables"]:
        s = t["step_ms"]
        print(f"{t['table']:4s} N={t['items']:6d} rows={t['packed_rows']}: " +
              "  ".join(f"{kk} {v['median']:.3f}" for kk, v in s.items()) + " ms")
        for kk, v in t["kernels_k256"].items():
            print(f"     {kk}: {v if isinstance(v, float) else v['median_ms']:.4f} ms")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"ok": True}))


if __name__ == "__main__":
    main()
