"""Cost of the full-catalogue cross-entropy objective (FusedTrainer(loss="ce"), csrc/catalogue_ce.cu), single GPU.

Two tables under the C2 workload (SRFR D = 64 + F = 16, 2 blocks, maxlen 50, batch 4096, Beauty-shaped users, soft
discriminator weights, batches drawn by the device sampler inside the step graph):
  C2   N = 12 101 items (the C2 catalogue)
  C5t  N = 150 000 items (the C5 catalogue size; the users and sequence shapes stay C2's)
Per table, the BCE step and the CE step (two trainers from the same initial parameters) run alternately for `--rounds`
rounds of CUDA-event-timed windows of >= `--window` seconds after a warm-up; median and range over the rounds.  Then each
CE kernel alone on the last step's operands (packed rows, bf16 hidden rows and table, the step's targets and weights):
pass 1 (LSE + loss), pass 2 (dh) and pass 3 (dE).  For each kernel: achieved TFLOP/s and exp/s from shape-derived counts
over the M packed rows of the batch and the N items (S = h E^T is 2 M N Dp flops and M N exponentials per pass; passes
2 and 3 add a second product of the same size), not from the padded tiles the kernels actually compute.

    python tools/bench_ce.py [--rounds 5] [--window 1.0] [--out profiles/r7_catalogue_ce.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from srfrd_b200 import SRFR_model as M, ops, synth
from srfrd_b200.trainer import DeviceSampler, FusedTrainer


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


def reps_for(fn, window_s):
    t = timed(fn, 3)
    return max(5, int(window_s * 1e3 / max(t, 1e-3)))


def make_model(N, seed=1236):
    torch.manual_seed(seed)
    m = M.SRFR(N, 50, 64, 16, 0.0, 2, 1, "cuda")
    for _, p in m.named_parameters():          # trainer.py:364-369
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to("cuda")


def bench_table(name, N, rounds, window, B=4096, L=50):
    data = synth.make_interactions(1236, 22363, N, 5, 4.0, L)
    smp = DeviceSampler(data, L, "cuda", seed=1000)
    tr = {loss: FusedTrainer(make_model(N), use_graph=True, loss=loss) for loss in ("bce", "ce")}
    steps = {loss: (lambda t=t: t.step_sampled(smp, B, "soft")) for loss, t in tr.items()}
    for f in steps.values():
        for _ in range(5):
            f()
    n = {loss: reps_for(f, window) for loss, f in steps.items()}
    step_ms = {"bce": [], "ce": []}
    for _ in range(rounds):
        for loss in ("bce", "ce"):
            step_ms[loss].append(timed(steps[loss], n[loss]))
    losses = {loss: float(t.loss_dev) for loss, t in tr.items()}

    # each CE kernel alone, on the operands the last CE step used
    t = tr["ce"]
    eng = t.eng
    plan = eng._plans[(B, L)]
    cap = plan.cap
    M_rows = int(plan.rows[0])
    hb, lse, table = t._ce_ws["h"][:cap], t._ce_ws["lse"][:cap], eng.sh["ce_table"]
    pos, w, norm = t._static["pos"].view(-1), t._static["w_pos"].view(-1), t.scal[0:2]
    Dp, D = table.shape[1], t.spec.D
    acc = torch.zeros(2, device="cuda")
    dh = torch.zeros(cap, eng._ws["dh"].shape[1], device="cuda")
    dE = torch.zeros(N + 1, D, device="cuda")
    kern = {
        "lse": lambda: ops.catalogue_ce_fwd(hb, table, pos, w, lse, acc, plan),
        "dh": lambda: ops.catalogue_ce_bwd(hb, table, pos, w, norm, lse, dh, None, D, plan),
        "dE": lambda: ops.catalogue_ce_bwd(hb, table, pos, w, norm, lse, None, dE, D, plan),
    }
    for f in kern.values():
        f()
    kn = {k: reps_for(f, window / 2) for k, f in kern.items()}
    kern_ms = {k: [] for k in kern}
    for _ in range(rounds):
        for k, f in kern.items():
            kern_ms[k].append(timed(f, kn[k]))
    gemm = 2.0 * M_rows * N * Dp
    work = {"lse": (gemm, M_rows * N), "dh": (2 * gemm, M_rows * N), "dE": (2 * gemm, M_rows * N)}
    med = lambda v: float(np.median(v))
    out = {
        "table": name, "items": N, "batch": B, "maxlen": L, "packed_rows": M_rows, "Dp": Dp,
        "step_ms": {k: {"median": med(v), "min": min(v), "max": max(v), "rounds": v} for k, v in step_ms.items()},
        "ce_minus_bce_ms": med(step_ms["ce"]) - med(step_ms["bce"]),
        "loss_after_warmup_and_timing": losses,
        "kernels": {},
    }
    for k, v in kern_ms.items():
        fl, ex = work[k]
        out["kernels"][k] = {"median_ms": med(v), "min_ms": min(v), "max_ms": max(v), "flop": fl, "exp": ex,
                             "tflops": fl / (med(v) * 1e-3) / 1e12, "gexp_per_s": ex / (med(v) * 1e-3) / 1e9}
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
        raise SystemExit("bench_ce: needs a CUDA device")
    res = {"gpu": gpu_info(), "rounds": args.rounds, "window_s": args.window,
           "workload": "C2 model and users (SRFR 64 + 16, 2 blocks, maxlen 50, batch 4096, soft weights, device sampler)",
           "tables": [bench_table("C2", 12101, args.rounds, args.window), bench_table("C5t", 150000, args.rounds, args.window)]}
    print(f"gpu: {res['gpu']}")
    for t in res["tables"]:
        s = t["step_ms"]
        print(f"{t['table']:4s} N={t['items']:6d} rows={t['packed_rows']}: step bce {s['bce']['median']:.3f} ms  "
              f"ce {s['ce']['median']:.3f} ms  (+{t['ce_minus_bce_ms']:.3f})")
        for k, v in t["kernels"].items():
            print(f"     {k:3s} {v['median_ms']:.3f} ms  {v['tflops']:.0f} TFLOP/s  {v['gexp_per_s']:.0f} Gexp/s")
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"ok": True}))


if __name__ == "__main__":
    main()
