"""Cost of the l2_emb regulariser in the fused training step, single GPU.

C2 (device-resident host-built batches) and C5 (batches drawn on the device) ms/step at l2_emb = 0 and 1e-4, as alternating
runs of two trainers within one process (median and range over the rounds), plus the per-launch time of the norm kernel
(srfrd_param_l2) and of the fused Adam with and without the l2 term on the same flat buffers.

    python tools/bench_l2.py [--rounds 5] [--steps 50] [--out FILE]
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
from srfrd_b200.trainer import DeviceSampler, FusedTrainer, discriminator_weights

L2 = 1e-4


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def make_model(c, itemnum):
    torch.manual_seed(c["seed"])
    m = M.SRFR(itemnum, c["L"], c["D"], c["F"], 0.0, c["blocks"], c["heads"], "cuda")
    for _, p in m.named_parameters():
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to("cuda")


def timed(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def per_launch(fn, n=200):
    for _ in range(10):
        fn()
    return timed(lambda i: fn(), n)


def bench_config(name, rounds, steps):
    c = synth.CONFIGS[name]
    data = synth.make_interactions(c["seed"], c["usernum"], c["itemnum"], c["min_len"], c["mean_extra"], c["max_len"],
                                   fake_rate=c.get("fake_rate", 0.15), lognormal=c.get("lognormal", False))
    B = c["batch"]
    runs = {}
    for l2 in (0.0, L2):
        tr = FusedTrainer(make_model(c, data.itemnum), use_graph=True, l2_emb=l2)
        if name == "C5":
            smp = DeviceSampler(data, c["L"], "cuda", seed=1000)
            fn = (lambda tr, smp: lambda i: tr.step_sampled(smp, B, "soft"))(tr, smp)
        else:
            hs = synth.BatchSampler(data, c["L"], seed=200)
            packs = []
            for _ in range(4):
                nb = hs.next_batch(B)
                b = {k: torch.from_numpy(nb[k]).cuda() for k in ("seq", "rsq", "pos", "prs", "neg", "nrs", "p_fake")}
                packs.append(tr.pack_batch(b, w_pos=discriminator_weights(b["pos"], b["p_fake"], "soft")))
            fn = (lambda tr, packs: lambda i: tr.step_packed(packs[i % 4]))(tr, packs)
        timed(fn, 8)                                          # eager step, capture, replays
        runs[l2] = dict(tr=tr, fn=fn, ms=[])
    for _ in range(rounds):
        for l2 in (0.0, L2):
            runs[l2]["ms"].append(timed(runs[l2]["fn"], steps))
    out = {}
    for l2, r in runs.items():
        ms = np.array(r["ms"])
        out[f"l2={l2:g}"] = dict(median_ms=round(float(np.median(ms)), 4), min_ms=round(float(ms.min()), 4),
                                 max_ms=round(float(ms.max()), 4), loss=round(float(r["tr"].loss_dev), 5))
    # per-launch times on the l2 trainer's own flat buffers (copies: the trainers' state is left alone)
    tr = runs[L2]["tr"]
    P = tr.P
    p, g, mm, vv = (t.clone() for t in (P.data, P.grad, tr.m, tr.v))
    st = tr.eng.step_state.clone()
    acc, norm, loss = torch.zeros(2, device="cuda"), torch.ones(2, device="cuda"), torch.zeros(1, device="cuda")
    k = tr._l2
    out["param_l2_us"] = round(per_launch(lambda: k.launch(p)) * 1e3, 2)
    out["adam_fused_us"] = round(per_launch(lambda: ops.adam_step_fused(p, g, mm, vv, 1e-3, 0.9, 0.98, 1e-8, st, True, acc, norm,
                                                                          loss)) * 1e3, 2)
    out["adam_fused_l2_us"] = round(per_launch(lambda: ops.adam_step_fused(p, g, mm, vv, 1e-3, 0.9, 0.98, 1e-8, st, True, acc,
                                                                             norm, loss, l2=k)) * 1e3, 2)
    out["params"] = P.numel
    out["segments"] = k.n_seg
    out["rounds"], out["steps_per_round"], out["batch"] = rounds, steps, B
    for r in runs.values():
        r.pop("tr"), r.pop("fn")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = dict(gpu=gpu_info(), l2_emb=L2)
    for name in ("C2", "C5"):
        res[name] = bench_config(name, a.rounds, a.steps)
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
