"""Cost of the lazy item-table Adam (FusedTrainer(lazy_item_adam=True)) next to the dense Adam sweep, single GPU.

Three tables under the C2 workload (SRFR D = 64 + F = 16, 2 blocks, maxlen 50, batch 4096, Beauty-shaped users, soft
discriminator weights, batches drawn by the device sampler inside the step graph):
  C2   N = 12 101 items (the C2 catalogue)
  C5t  N = 150 000 items
  C3t  N = 1 000 000 items (the users and sequence shapes stay C2's)
Per table, the BCE step and the gBCE step (k = 256, t = 0.75), each dense and lazy (four trainers from the same initial
parameters), run alternately for `--rounds` rounds of CUDA-event-timed windows of >= `--window` seconds after a warm-up;
median and range over the rounds.  Then the Adam tail alone on the lazy BCE trainer's last-step operands (parameters,
moments, stamps): srfrd_adam_step_fused against srfrd_adam_step_fused_rows.  Each timed call first restores the 32-byte
step state (so the gated kernel sees the last step's epoch every time); that copy is timed alone too and subtracted.
Rows touched per step = the stamps equal to the last step's epoch.  Algorithmic bytes: dense 32 B per parameter (read p,
g, m, v; write p, m, v and the zeroed g); gated 32 B per non-table parameter and per parameter of a touched row, plus
4 B per stamp read.

    python tools/bench_lazy_adam.py [--rounds 5] [--window 1.0] [--out profiles/r9_lazy_adam.json]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from srfrd_b200 import ops, synth
from srfrd_b200.trainer import DeviceSampler, FusedTrainer
from tools.bench_ce import gpu_info, make_model, reps_for, timed

TABLES = (("C2", 12101), ("C5t", 150000), ("C3t", 1000000))


def bench_table(name, N, rounds, window, B=4096, L=50):
    data = synth.make_interactions(1236, 22363, N, 5, 4.0, L)
    smp = DeviceSampler(data, L, "cuda", seed=1000)
    gb = dict(loss="gbce", num_negatives=256, gbce_t=0.75)
    tr = {"bce": FusedTrainer(make_model(N), use_graph=True),
          "bce_lazy": FusedTrainer(make_model(N), use_graph=True, lazy_item_adam=True),
          "gbce256": FusedTrainer(make_model(N), use_graph=True, **gb),
          "gbce256_lazy": FusedTrainer(make_model(N), use_graph=True, lazy_item_adam=True, **gb)}
    steps = {k: (lambda t=t: t.step_sampled(smp, B, "soft")) for k, t in tr.items()}
    for f in steps.values():
        for _ in range(5):
            f()
    n = {k: reps_for(f, window) for k, f in steps.items()}
    step_ms = {k: [] for k in tr}
    for _ in range(rounds):
        for k in tr:
            step_ms[k].append(timed(steps[k], n[k]))
    losses = {k: float(t.loss_dev) for k, t in tr.items()}
    torch.cuda.synchronize()
    bits = lambda t: int(t.eng.step_state.cpu().view(torch.int32)[3])
    touched = {k: int((t.stamp == bits(t)).sum()) for k, t in tr.items() if t.lazy}

    # the Adam tail alone, on the lazy BCE trainer's operands
    t = tr["bce_lazy"]
    P = t.P
    st = t.eng.step_state
    st0 = st.clone()
    st0.view(torch.int32)[3] = bits(t) - 1                # epoch = bits + 1 = the last step's
    norm, acc, loss = t.scal[0:2], P.grad_tail[0:2], t.scal[4:5]
    reset = lambda: st.copy_(st0)
    kern = {
        "reset_only": reset,
        "dense": lambda: (reset(), ops.adam_step_fused(P.data, P.grad, t.m, t.v, t.lr, t.betas[0], t.betas[1], t.eps, st,
                                                       acc2=acc, norm2=norm, loss=loss)),
        "gated": lambda: (reset(), ops.adam_step_fused_rows(P.data, P.grad, t.m, t.v, t.lr, t.betas[0], t.betas[1], t.eps,
                                                            st, *t._table, t.stamp, acc2=acc, norm2=norm, loss=loss)),
    }
    for f in kern.values():
        f()
    kn = {k: reps_for(f, window / 2) for k, f in kern.items()}
    kern_ms = {k: [] for k in kern}
    for _ in range(rounds):
        for k, f in kern.items():
            kern_ms[k].append(timed(f, kn[k]))
    med = lambda v: float(np.median(v))
    rows, D = t._table[1], t._table[2]
    n_par = P.numel
    n_tab = rows * D
    bytes_ = {"dense": 32.0 * n_par,
              "gated": 32.0 * (n_par - n_tab + touched["bce_lazy"] * D) + 4.0 * rows}
    out = {
        "table": name, "items": N, "batch": B, "maxlen": L, "flat_params": n_par, "table_params": n_tab,
        "step_ms": {k: {"median": med(v), "min": min(v), "max": max(v), "rounds": v} for k, v in step_ms.items()},
        "lazy_minus_dense_ms": {"bce": med(step_ms["bce_lazy"]) - med(step_ms["bce"]),
                                "gbce256": med(step_ms["gbce256_lazy"]) - med(step_ms["gbce256"])},
        "rows_touched_last_step": touched,
        "rows_touched_share": {k: v / N for k, v in touched.items()},
        "loss_after_warmup_and_timing": losses,
        "adam_tail": {},
    }
    for k, v in kern_ms.items():
        out["adam_tail"][k] = {"median_ms": med(v), "min_ms": min(v), "max_ms": max(v)}
    r = med(kern_ms["reset_only"])
    for k in ("dense", "gated"):
        ms = med(kern_ms[k]) - r
        out["adam_tail"][k].update(minus_reset_ms=ms, algorithmic_bytes=bytes_[k], tb_per_s=bytes_[k] / (ms * 1e-3) / 1e12)
    out["adam_tail"]["gated_over_dense"] = out["adam_tail"]["gated"]["minus_reset_ms"] / out["adam_tail"]["dense"]["minus_reset_ms"]
    del tr, t, P
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lazy_adam: needs a CUDA device")
    res = {"gpu": gpu_info(), "rounds": args.rounds, "window_s": args.window,
           "workload": "C2 model and users (SRFR 64 + 16, 2 blocks, maxlen 50, batch 4096, soft weights, device sampler)",
           "tables": [bench_table(name, N, args.rounds, args.window) for name, N in TABLES]}
    print(f"gpu: {res['gpu']}")
    for t in res["tables"]:
        s, a = t["step_ms"], t["adam_tail"]
        print(f"{t['table']:4s} N={t['items']:7d}: " + "  ".join(f"{k} {v['median']:.3f} [{v['min']:.3f}, {v['max']:.3f}]"
                                                                  for k, v in s.items()) + " ms")
        print(f"     rows touched {t['rows_touched_last_step']}; Adam tail dense {a['dense']['minus_reset_ms']:.4f} ms, "
              f"gated {a['gated']['minus_reset_ms']:.4f} ms ({a['gated_over_dense']:.3f} of dense)")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"ok": True}))


if __name__ == "__main__":
    main()
