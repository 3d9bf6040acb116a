#!/usr/bin/env python
"""Benchmark of the SRFRD hot path on B200 (contract: see the task statement / DESIGN.md section "Measurement").

  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches N ranks for N > 1)
  python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port) on host cores
  python bench.py --steps K --dump-outputs DIR              # also save what the timed steps computed (DIR/<name>.npy)

A "step" is one training step (forward + discriminator-weighted BCE + backward + gradient all-reduce +
Adam) of the reference SRFR model on Beauty-shaped synthetic data, config C2 of BASELINE.json:
22 363 users, 12 101 items, maxlen 50, D=64, F=16, 2 blocks, batch 4096 per GPU (weak scaling).
`value` = global sequences / second with the batch already resident in HBM; `e2e` = the same step driven
through FusedTrainer.step() from pinned HOST batches (H2D copies + a D2H read of the loss every step).
Further objects in the same line (every BASELINE.json config is driver-measured at every N): "catalogue" = full-catalogue
top-10 users/s (C3: 1 M items, row-sharded; score + top-k + all-gather + merge, and `with_encode` = the same plus the
sequence encoder), "c4" = the long-sequence variant (maxlen 200, D=256, 4 blocks, batch 1024/GPU, DP), "c5" = the
Yelp-shaped setting (~10 M interactions, 30 % fake, batches drawn ON THE DEVICE inside the step graph, soft and mask
discriminator policies, batch 4096/GPU), "dropout" = C2 at the reference's default dropout 0.5 (trainer.py:128),
"dp_parity" (N > 1) = first-step DP loss vs one rank on the concatenated batch + sharded vs unsharded top-10, "gather" =
K1 at catalogue scale against the HBM roofline.  `roofline` = the dominant kernel's algorithmic bytes per launch / its
event-timed launch duration, `roofline.traffic` = its DRAM bytes per launch from the committed ncu capture
(profiles/traffic.json); `clocks` = NVML samples taken every 2 ms DURING the timed region.  Baselines on rank 0 at N = 1
only: `cpu_baseline` (the reference's arithmetic, oracle port, on the host cores) and `gpu_eager_baseline` (the same as
stock PyTorch eager fp32 on this GPU).  Nothing of the product runs in either baseline.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "training seqs/sec; full-catalogue top-10 users/sec"
CFG = dict(kind="SRFR", usernum=22363, itemnum=12101, L=50, D=64, F=16, blocks=2, heads=1, batch=4096)
DUMP_LIMIT = 64 << 20          # bytes --dump-outputs may write in all


def write_outputs(out_dir, arrays):
    """--dump-outputs: save each array as out_dir/<name>.npy so that two builds can be compared output for output.
    Floating arrays become float32 (float64 stays float64), integer ids float64 (exact below 2**53).  Raises before writing
    anything if the arrays exceed DUMP_LIMIT bytes in all; returns the bytes written."""
    conv = {}
    for name, a in arrays.items():
        t = torch.as_tensor(a).detach()
        if t.dtype != torch.float64:
            t = t.float() if t.is_floating_point() else t.double()
        conv[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback (B200_PROFILING.md)")


def measured_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the committed `ncu --set full`
    capture (profiles/traffic.json, written by tools/profile_round.py); None if the capture is missing."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")) as f:
            return json.load(f).get(key)
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region: NVML in a thread every 2 ms (the timed region of a
    default run is a few hundred ms, shorter than `nvidia-smi -lms` needs to start); nvidia-smi as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.h, self.nv = index, [], None, None, None
        self.sm, self.reason_bits, self.mx, self._stop = [], 0, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: look the handle up by the CUDA device's PCI bus id
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.h = h
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self._stop:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._stop = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            nv, bits = self.nv, self.reason_bits
            table = [("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", 0x8), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", 0x20), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", 0x4)]
            reasons = sorted(name for name, attr, dflt in table if bits & int(getattr(nv, attr, dflt)))
            return dict(sm_mhz=float(np.median(self.sm)) if self.sm else None, sm_max_mhz=self.mx, reasons=reasons,
                        samples=len(self.sm), source="nvml")
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm), source="nvidia-smi")


# ---------------------------------------------------------------------------------------------
def algorithmic_bytes(name, a, valid_frac, packed=None):
    """Algorithmic (minimum) HBM bytes of one C-ABI call, from its arguments (DESIGN.md 'bytes per unit').
    packed = (capacity rows, actual rows M, sequences B, maxlen L) when the step ran on the packed token layout: the
    row-wise calls are then launched with the CAPACITY as their row argument and read the actual count on the device."""
    g = lambda i: a[i] or 0
    rows = (lambda r: packed[1] if (packed and r == packed[0]) else r)
    if packed:
        cap, Mp, Bp, Lp = packed
        if name == "srfrd_embed_ln_fwd_packed":
            D, F, mode = a[2], a[6], a[7]
            H = D + (F if mode == 1 else 0)
            return Mp * (4 + 16 + D * 4 + 2 * H * 2 + 8), 0.0
        if name in ("srfrd_attention_fwd_packed", "srfrd_attention_bwd_packed"):
            H = a[9] if name.endswith("fwd_packed") else a[14]
            n = 4 if name.endswith("fwd_packed") else 7
            avg = Mp / max(Bp, 1)                                     # rows per sequence incl. its pad representative
            return n * Mp * H * 2 + Mp * 16, (2.0 if n == 4 else 5.0) * Mp * avg * H
        if name == "srfrd_score_loss_fused_packed":
            D = a[11]
            return Mp * (4 + 16 + D * 4 + 2 * D * 4 + D * 4 + 2 * 2 * D * 4), 0.0
        if name == "srfrd_embed_bwd_packed":
            D, F, mode = a[8], a[9], a[10]
            return Mp * (4 + 8 + (D + (F if mode == 1 else 0)) * 2 + D * 8), 0.0
        if name == "srfrd_pack_plan":
            return Bp * Lp * (16 + 4) + Mp * (4 + 8 + 16), 0.0
    if name == "srfrd_gemm_tn":
        M, N, K = rows(a[4]), a[5], a[6]
        ep = a[7]._obj
        b = M * K * 2 + N * K * 2 + M * N * (2 if ep.out_bf16 else 4)
        b += (M * N * 2 if ep.residual else 0) + (M * N * 2 if ep.gate else 0) + (M * 8 if ep.row_ids else 0)
        if ep.ln_out_bf16:                       # fused LayerNorm: its output and (mean, rstd) are extra stores
            b += M * N * 2 + (M * 8 if ep.ln_stats else 0)
        return b, 2.0 * M * N * K
    if name == "srfrd_mlp2_tn":                      # A, mid, out (+ LayerNorm output), two square weights; residual = A
        M, N = rows(a[6]), a[7]
        ep = a[8]._obj
        b = 3 * M * N * 2 + 2 * N * N * 2 + (M * N * 2 if ep.gate else 0) + (M * N * 2 if ep.residual else 0)
        b += (M * N * 2 + M * 8) if ep.ln_out else 0
        return b, 4.0 * M * N * N
    if name == "srfrd_gemm_wgrad":
        T, Mo, No = rows(a[4]), a[5], a[6]
        return T * (Mo + No) * 2 + Mo * No * 4, 2.0 * T * Mo * No
    if name == "srfrd_attention_fwd":
        B, L, H = a[8], a[9], a[10]
        return 4 * B * L * H * 2, 2.0 * B * L * L * H           # causal half of 2 x (2 L^2 H)
    if name == "srfrd_attention_bwd":
        B, L, H = a[15], a[16], a[17]
        return 7 * B * L * H * 2, 5.0 * B * L * L * H
    if name == "srfrd_layernorm_fwd":
        T, H = rows(a[9]), a[10]
        return T * H * 2 + T * H * (2 if a[5] else 4) + T * 8, 0.0
    if name == "srfrd_layernorm_bwd":
        T, H = rows(a[14]), a[15]
        return T * H * (2 if a[0] else 4) + 2 * T * H * 2 + T * 8 + (T * H * 2 if a[7] else 0) + (T * 8 if a[9] else 0), 0.0
    if name == "srfrd_embed_ln_fwd":
        D, F, mode, T = a[2], a[6], a[7], a[10] * a[11]
        H = D + (F if mode == 1 else 0)
        return T * 16 + valid_frac * T * D * 4 + 2 * T * H * 2 + T * 8, 0.0
    if name == "srfrd_score_loss_fused":
        T, D, F = a[11], a[12], a[13]
        return T * 16 + valid_frac * T * (D * 4 + 2 * D * 4 + D * 4 + 2 * 2 * D * 4) + (1 - valid_frac) * T * D * 4, 0.0
    if name == "srfrd_colsum":
        return a[1] * a[2] * 2 + a[2] * 4, 0.0
    if name == "srfrd_adam_step":
        return a[4] * 32, 0.0
    if name == "srfrd_embed_bwd":
        T, D, F, mode = a[4] * a[5], a[6], a[7], a[8]
        return T * 16 + valid_frac * T * ((D + (F if mode == 1 else 0)) * 2 + D * 8), 0.0
    if name == "srfrd_dropout_apply":
        return rows(a[4]) * a[5] * 4, 0.0
    return 0, 0.0


def kernel_breakdown(tr, steps, valid_frac):
    """Eager, event-bracketed pass over `steps` steps: per entry point total ms, launches, algorithmic bytes."""
    from srfrd_b200 import _lib
    recs = []
    tr_graph, tr.use_graph = tr.use_graph, False
    ov, tr.eng.overlap = tr.eng.overlap, False      # one kernel at a time: clean per-kernel durations
    _lib.set_profile(recs)
    for _ in range(steps):
        # park the GPU behind a ~20 ms spin so the host has enqueued the whole step (kernels + bracketing events)
        # before the first kernel starts: the event deltas then hold GPU time only, not host launch gaps
        torch.cuda._sleep(40_000_000)
        tr.run_step()
    torch.cuda.synchronize()
    _lib.set_profile(None)
    tr.use_graph, tr.eng.overlap = tr_graph, ov
    packed = None
    plans = getattr(tr.eng, "_plans", {})
    st = tr._static["seq"].shape if tr._static is not None else None
    if tr.packed and st is not None and tuple(st) in plans:          # row count of the last batch (device -> host, after the run)
        pl = plans[tuple(st)]
        packed = (pl.cap, int(pl.rows[0].item()), int(st[0]), int(st[1]))
    agg = {}
    for name, args, e0, e1 in recs:
        if name == "srfrd_set_row_limit":                             # host-side state, no launch
            continue
        ms = e0.elapsed_time(e1)
        by, fl = algorithmic_bytes(name, args, valid_frac, packed)
        d = agg.setdefault(name, dict(ms=0.0, n=0, bytes=0.0, flops=0.0))
        d["ms"] += ms; d["n"] += 1; d["bytes"] += by; d["flops"] += fl
    n_launch = sum(1 for r in recs if r[0] != "srfrd_set_row_limit")
    return agg, n_launch // max(steps, 1), packed


# ---------------------------------------------------------------------------------------------
def make_model(device, itemnum, L, D, F, blocks, heads=1, dropout=0.0, seed=1236):
    from srfrd_b200 import SRFR_model as M
    torch.manual_seed(seed)
    m = M.SRFR(itemnum, L, D, F, dropout, blocks, heads, device)
    for _, p in m.named_parameters():          # trainer.py:364-369
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to(device)


def make_model_and_data(device, seed=1236, dropout=0.0):
    from srfrd_b200 import synth
    c = CFG
    data = synth.make_interactions(seed, c["usernum"], c["itemnum"], 5, 4.0, c["L"])
    return make_model(device, c["itemnum"], c["L"], c["D"], c["F"], c["blocks"], c["heads"], dropout, seed), data


class Timer:
    """barrier + synchronize on both sides, CUDA events on the launching stream, MAX over ranks."""

    def __init__(self, dev, world):
        self.dev, self.world = dev, world

    def sync_all(self):
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def __call__(self, fn, steps, warm):
        import torch.distributed as dist
        for i in range(warm):
            fn(i)
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warm + i)
        e1.record()
        self.sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)


def top_kernel_roofline(agg, nsteps, pk, traffic_key=None):
    tot = sum(d["ms"] for d in agg.values())
    tname, td = max(agg.items(), key=lambda kv: kv[1]["ms"])
    per_ms = td["ms"] / td["n"]
    ach = td["bytes"] / td["n"] / (per_ms * 1e-3) / 1e9
    return dict(bound="hbm", kernel=tname, achieved=round(ach, 1), peak=pk["hbm"], unit="GB/s", frac=round(ach / pk["hbm"], 4),
                traffic=measured_traffic(traffic_key or tname), algorithmic_bytes_per_launch=round(td["bytes"] / td["n"]),
                peak_source=pk["src"] + ", sustained figure not needed for HBM", avg_launch_ms=round(per_ms, 4),
                share_of_step=round(td["ms"] / tot, 3),
                note=("algorithmic bytes counted over the rows the launch actually processed; when a launch moves a few MB "
                      "(packed token layout: every operand is L2-resident, traffic << algorithmic) its duration is the fixed "
                      "cost of a launch, not HBM time -- DESIGN.md section 6; the HBM-bound kernels are measured beyond L2 in "
                      "`gather` and `scale_kernels`"),
                kernels={k: dict(ms_per_step=round(v["ms"] / nsteps, 4), launches_per_step=v["n"] // nsteps,
                                 gbs=round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] > 0 else None,
                                 tflops=round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2) if v["flops"] else None)
                         for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])})


def bench_train_config(name, dev, rank, world, pg, timed, pk, steps, model_kw, data_kw, B, L, dropout=0.0, policy="soft",
                       sampler="host", breakdown=True):
    """One training configuration: device-resident batches (or batches drawn on the device inside the step graph),
    CUDA-graph replay, max-over-ranks CUDA-event time.  Returns ms/step, global seqs/s and the dominant kernel's roofline."""
    import torch.distributed as dist
    from srfrd_b200 import synth
    from srfrd_b200.trainer import DeviceSampler, FusedTrainer, discriminator_weights
    data = synth.make_interactions(**data_kw)
    m = make_model(dev, data.itemnum, L, dropout=dropout, seed=data_kw["seed"], **model_kw)
    if world > 1:
        dist.broadcast(m.flat_parameters().data, 0)
    tr = FusedTrainer(m, lr=1e-3, betas=(0.9, 0.98), process_group=pg, use_graph=True)
    if sampler == "device":
        smp = DeviceSampler(data, L, dev, seed=1000 + rank)
        fn = lambda i: tr.step_sampled(smp, B, policy)
        valid_frac = float(np.minimum(np.maximum(data.train_len() - 1, 0), L)[data.train_len() > 1].mean() / L)
    else:
        hs = synth.BatchSampler(data, L, seed=200 + rank)
        packs, vf = [], []
        for _ in range(4):
            nb = hs.next_batch(B)
            b = {k: torch.from_numpy(nb[k]).to(dev) for k in ("seq", "rsq", "pos", "prs", "neg", "nrs", "p_fake")}
            vf.append(float((b["pos"] != 0).float().mean()))
            packs.append(tr.pack_batch(b, w_pos=discriminator_weights(b["pos"], b["p_fake"], policy)))
        valid_frac = float(np.mean(vf))
        fn = lambda i: tr.step_packed(packs[i % 4])
    W = 4
    timed(fn, 2, W)
    ms = timed(fn, steps, W)
    out = dict(value=round(world * B * steps / (ms / 1e3), 1), unit="seqs/s", ms_per_step=round(ms / steps, 4), steps=steps,
               warmup=W, batch_per_gpu=B, n_gpus=world, valid_slot_fraction=round(valid_frac, 4), policy=policy,
               dropout=dropout, loss=round(float(tr.loss_dev), 5))
    if breakdown:                                    # EVERY rank runs the eager pass (it steps through the all-reduce)
        if sampler == "device":                      # the eager pass needs the sampler attached for its step body
            tr._sampler, tr._sampler_policy = smp, policy
        agg, calls, packed_rows = kernel_breakdown(tr, 2, valid_frac)
        out["roofline"] = top_kernel_roofline(agg, 2, pk)
        if packed_rows:
            out["packed_rows"] = dict(capacity=packed_rows[0], rows=packed_rows[1], dense_tokens=packed_rows[2] * packed_rows[3])
        out["gpu_launches_per_step"] = calls
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        tr._graph = None                             # drop the captured NCCL work before the trainer goes away
        torch.cuda.synchronize()
    del tr, m
    torch.cuda.empty_cache()
    return out


def dp_parity_check(dev, rank, world, pg):
    """N > 1, before any timing: (1) the first DP step (batch rows sharded over the ranks, loss normalised by the
    all-reduced weight sums, gradients SUM-all-reduced) against ONE rank stepping the concatenated batch: loss and
    parameters after the step; (2) row-sharded catalogue top-10 (all-gather + merge) torch.equal the unsharded one on
    dyadic data, where every accumulation order is exact."""
    import torch.distributed as dist
    from srfrd_b200 import evaluation as EV, parallel as PL, synth
    from srfrd_b200.trainer import FusedTrainer, discriminator_weights
    c = CFG
    Bg, L = 512 * world, c["L"]
    data = synth.make_interactions(4321, 6000, 3000, 5, 4.0, L)
    nb = synth.BatchSampler(data, L, seed=9).next_batch(Bg)               # same global batch on every rank
    full = {k: torch.from_numpy(v).to(dev) for k, v in nb.items()}
    w = discriminator_weights(full["pos"], full["p_fake"], "soft")
    m_dp = make_model(dev, 3000, L, c["D"], c["F"], c["blocks"], seed=77)
    m_one = make_model(dev, 3000, L, c["D"], c["F"], c["blocks"], seed=77)
    dist.broadcast(m_dp.flat_parameters().data, 0)
    tr_dp = FusedTrainer(m_dp, process_group=pg, use_graph=False)
    sh = PL.shard_batch({**full, "w": w}, rank, world)
    l_dp = float(tr_dp.step(sh, w_pos=sh["w"]))
    tr_one = FusedTrainer(m_one, use_graph=False)
    l_one = float(tr_one.step(full, w_pos=w))
    a, b = m_one.flat_parameters().data, m_dp.flat_parameters().data
    drift = torch.tensor([float((a - b).abs().max())], device=dev)
    dist.all_reduce(drift, op=dist.ReduceOp.MAX)
    g = torch.Generator().manual_seed(3)
    feats = (torch.randint(-16, 17, (1000, 64), generator=g).float() / 8).to(dev)
    table = (torch.randint(-16, 17, (50001, 64), generator=g).float() / 8).to(dev)
    _, ref = EV.local_topk(feats, EV.CatalogueIndex(table, 0), 1)
    lo, hi = EV.CatalogueIndex.shard_bounds(table.shape[0], rank, world)
    _, ids = EV.sharded_topk(feats, EV.CatalogueIndex(table[lo:hi], lo), pg, 1)
    same = torch.tensor([1.0 if torch.equal(ids, ref) else 0.0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    # (3) user-sharded encode + all-gather (EV.encode_users) against every rank encoding everybody: the same sequences in
    # other attention tiles -- equal to a bf16 ulp of the activations (hidden-state tolerance of the golden tests: 4e-2)
    seq_e, rsq_e, _ = synth.eval_sequences(data, L, np.arange(1000))
    seq_e, rsq_e = torch.from_numpy(seq_e).to(dev), torch.from_numpy(rsq_e).to(dev)
    enc_diff = (EV.encode_users(m_one, seq_e, rsq_e, pg) - m_one.encode_last(seq_e, rsq_e)).abs().max().reshape(1)
    dist.all_reduce(enc_diff, op=dist.ReduceOp.MAX)
    torch.cuda.synchronize()
    del tr_dp, tr_one
    return dict(loss_dp=round(l_dp, 6), loss_single_rank_on_concatenated_batch=round(l_one, 6),
                loss_abs_diff=round(abs(l_dp - l_one), 7), param_max_abs_diff_after_step=float(drift),
                sharded_top10_equals_unsharded=bool(same.item() == 1.0), global_batch=Bg,
                user_sharded_encode_max_abs_diff=float(enc_diff),
                ok=bool(abs(l_dp - l_one) < 2e-3 and float(drift) < 2e-3 and same.item() == 1.0 and float(enc_diff) < 4e-2))


def run_ours(args):
    import torch.distributed as dist
    from srfrd_b200 import _lib, evaluation as EV, synth
    from srfrd_b200.trainer import FusedTrainer, discriminator_weights
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        import datetime
        # a collective mismatch must fail in minutes, not hold the GPUs for NCCL's default 10-minute watchdog
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=150))
        pg = dist.group.WORLD
    c = CFG
    B, L = c["batch"], c["L"]
    timed = Timer(dev, world)
    pk = peaks()

    def guarded(fn, *a, **kw):
        """Secondary objects must never take the headline line down: an exception becomes {"error": ...} (all ranks
        run the same code, so a deterministic failure fails everywhere and no rank is left waiting in a collective)."""
        try:
            return fn(*a, **kw)
        except Exception as ex:  # noqa: BLE001
            return dict(error=f"{type(ex).__name__}: {str(ex)[:300]}")

    # ---- N > 1: DP == single rank on the concatenated batch, sharded top-10 == unsharded, BEFORE any timing ----
    dp_parity = guarded(dp_parity_check, dev, rank, world, pg) if world > 1 else None

    m, data = make_model_and_data(dev)
    if world > 1:                               # identical replicas
        dist.broadcast(m.flat_parameters().data, 0)
    tr = FusedTrainer(m, lr=1e-3, betas=(0.9, 0.98), process_group=pg, use_graph=True)
    smp = synth.BatchSampler(data, L, seed=100 + rank)
    npool = 8
    host, packs = [], []
    for _ in range(npool):
        nb = smp.next_batch(B)
        hb = {k: torch.from_numpy(nb[k]).pin_memory() for k in ("seq", "rsq", "pos", "prs", "neg", "nrs", "p_fake")}
        host.append(hb)
        db = {k: v.to(dev) for k, v in hb.items()}
        # inputs resident in HBM, already in the layout of the step's static buffers: ONE device-to-device copy per step
        packs.append(tr.pack_batch(db, w_pos=discriminator_weights(db["pos"], db["p_fake"], "soft")))
    valid_frac = float(np.mean([float((hb["pos"] != 0).float().mean()) for hb in host]))
    h2d = sum(host[0][k].numel() * host[0][k].element_size() for k in ("seq", "rsq", "pos", "prs", "neg", "nrs")) + B * L * 4

    # ---- value: batch resident in HBM (weights 'soft') ----
    def dev_step(i):
        tr.step_packed(packs[i % npool])

    # ---- e2e: pinned host batch -> H2D -> step -> D2H loss ----
    wbuf = [discriminator_weights(hb["pos"], hb["p_fake"], "soft").pin_memory() for hb in host]

    # Every step's inputs start in pinned host memory and its loss is read back; the H2D copy of batch i+1 is issued
    # (copy stream, staging buffer) right after step i is launched, so it overlaps step i's compute.
    def host_step(i):
        if i == 0 or getattr(tr, "_stage_flat", None) is None:
            tr.prefetch(host[i % npool], w_pos=wbuf[i % npool])
        loss = tr.step_prefetched()
        tr.prefetch(host[(i + 1) % npool], w_pos=wbuf[(i + 1) % npool])
        return float(loss.item())

    clk = ClockSampler(local)
    W = max(args.warmup, 3)
    timed(dev_step, 2, W)                       # sizes workspaces, captures the graph
    clk.start()
    ms = timed(dev_step, args.steps, W)
    clocks = clk.stop()
    dump = {} if args.dump_outputs and rank == 0 else None
    if dump is not None:
        # what the last timed step returns to its caller: the loss (read now: the e2e run below keeps training).  The
        # parameters are not saved: gradients are summed with float atomics and Adam turns that rounding into +-lr steps
        # wherever a gradient is ~0 (the key bias of in_proj_bias is 0 analytically), so after a few steps two correct
        # runs differ there by far more than rounding while the loss agrees to ~1e-6.
        dump["train_loss"] = tr.loss_dev.reshape(1).cpu()
    ms_e2e = timed(host_step, args.steps, W)
    value = world * B * args.steps / (ms / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)

    # ---- per-kernel breakdown + roofline of the dominant kernel (rank 0) ----
    agg, calls_per_step, packed_rows = kernel_breakdown(tr, 3, valid_frac)
    roofline = top_kernel_roofline(agg, 3, pk)
    if packed_rows:
        roofline["packed_rows"] = dict(capacity=packed_rows[0], rows=packed_rows[1], dense_tokens=packed_rows[2] * packed_rows[3])
    roofline["how"] = ("event-bracketed pass of 3 eager steps right after the timed region (which replays a CUDA graph); the "
                       "GPU is parked behind a spin kernel while the host enqueues each step, so the deltas are GPU time")
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        tr._graph = None
        torch.cuda.synchronize()
    del tr, m, packs
    torch.cuda.empty_cache()

    extras = {}
    if not args.no_extras:
        ex_steps = max(5, min(args.steps, 40))
        c2_model = dict(D=c["D"], F=c["F"], blocks=c["blocks"])
        c2_data = dict(seed=1236, usernum=c["usernum"], itemnum=c["itemnum"], min_len=5, mean_extra=4.0, max_len=L)
        # C2 at the reference's default dropout 0.5 (trainer.py:128): in-kernel dropout in attention and twice in the FFN
        extras["dropout"] = guarded(bench_train_config, "C2-dropout0.5", dev, rank, world, pg, timed, pk, ex_steps, c2_model,
                                    c2_data, B, L, dropout=0.5)
        # C4: maxlen 200, D = 256, F = 16, 4 blocks, batch 1024 per GPU, data parallel at N
        c4 = synth.CONFIGS["C4"]
        extras["c4"] = guarded(bench_train_config, "C4", dev, rank, world, pg, timed, pk, max(4, ex_steps // 2),
                               dict(D=c4["D"], F=c4["F"], blocks=c4["blocks"]),
                               dict(seed=c4["seed"], usernum=c4["usernum"], itemnum=c4["itemnum"], min_len=c4["min_len"],
                                    mean_extra=c4["mean_extra"], max_len=c4["max_len"]), c4["batch"], c4["L"])
        if isinstance(extras["c4"], dict) and "value" in extras["c4"]:
            extras["c4"]["config"] = "C4: SRFR maxlen 200, D=256 F=16 (H=272), 4 blocks, 12101 items, batch 1024/GPU, soft weights, DP"
        # C5: Yelp-shaped, ~10 M interactions, 500 k users, 150 k items, 30 % fake; batches drawn on the device INSIDE the
        # step graph (no host batch at all), discriminator-in-the-loop weights under both policies
        c5 = synth.CONFIGS["C5"]
        c5_data = dict(seed=c5["seed"], usernum=c5["usernum"], itemnum=c5["itemnum"], min_len=c5["min_len"],
                       mean_extra=c5["mean_extra"], max_len=c5["max_len"], fake_rate=c5["fake_rate"], lognormal=True)
        c5_model = dict(D=c5["D"], F=c5["F"], blocks=c5["blocks"])
        c5o = {}
        for pol in ("soft", "mask"):
            c5o[pol] = guarded(bench_train_config, "C5-" + pol, dev, rank, world, pg, timed, pk, ex_steps, c5_model, c5_data,
                               c5["batch"], c5["L"], policy=pol, sampler="device", breakdown=(pol == "soft"))
        c5o["config"] = ("C5: Yelp-shaped synthetic, ~10.05 M interactions, 500 k users, 150 k items, 30 % fake-labelled, SRFR D=64 F=16 "
                         "L=50 2 blocks, batch 4096/GPU drawn by the on-device sampler inside the CUDA graph, weights per batch")
        extras["c5"] = c5o

    # ---- catalogue: C3, 1 M items row-sharded, U = 16384 users ----
    cat = None
    if not args.no_catalogue:
        cat = guarded(bench_catalogue, dev, rank, world, pg, args, pk, timed, dump)

    # ---- gather: K1 on the C3 item table (1 M rows x 64 fp32 = 256 MB > L2), 4 M tokens, every slot valid ----
    gat = None
    if not args.no_catalogue and rank == 0:
        gat = guarded(bench_gather, dev, pk)

    scale_k = None
    if not args.no_catalogue and rank == 0:
        scale_k = guarded(bench_scale_kernels, dev, pk)
        torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline(sample_steps=10)          # ~10 s of host work
    eager = None
    if rank == 0 and world == 1 and not args.no_cpu:
        eager = guarded(gpu_eager_baseline, dev)     # the same arithmetic as stock PyTorch eager on this GPU (informative)

    if rank == 0:
        line = dict(metric=METRIC, value=round(value, 1), unit="seqs/s", n_gpus=world, steps=args.steps, warmup=W,
                    ms_per_step=round(ms / args.steps, 4), higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="bf16", data="synthetic",
                    config=dict(workload="C2: SRFR D=64 F=16 L=50 2 blocks 1 head, 12101 items, 22363 users, batch 4096/GPU, "
                                         "discriminator-weighted (soft) BCE, dropout 0.0, Adam(1e-3,(0.9,0.98))",
                                global_batch=world * B, maxlen=L, parallelism=f"dp{world}", valid_slot_fraction=round(valid_frac, 4),
                                l2="per-step working set ~0.7 GB of activations > 126 MB L2; 8 distinct batches rotate"),
                    e2e=dict(value=round(e2e, 1), unit="seqs/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=4,
                             ms_per_step=round(ms_e2e / args.steps, 4)),
                    gpu_launches=int(calls_per_step * args.steps), clocks=clocks, roofline=roofline)
        if dp_parity is not None:
            line["dp_parity"] = dp_parity
        line.update(extras)
        if cat is not None:
            line["catalogue"] = cat
        if gat is not None:
            line["gather"] = gat
        if scale_k is not None:
            line["scale_kernels"] = scale_k
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if eager is not None:
            line["gpu_eager_baseline"] = eager
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear down without dist.destroy_process_group(): with the NCCL all-reduce captured inside live CUDA graphs the
        # communicator teardown can block for minutes.  All ranks meet and leave.
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def bench_gather(dev, pk):
    """K1 (gather + positional add + fake concat + pad mask + LayerNorm) at a size where the table cannot sit in L2:
    algorithmic bytes per token = 16 (ids) + 256 (fp32 row) + 2 x 160 (x0, LN out, bf16) + 8 (stats) = 600."""
    from srfrd_b200 import ops
    N, D, F, L, B = 1_000_000, 64, 16, 50, 81920
    T, H = B * L, D + F
    g = torch.Generator(device="cpu").manual_seed(1238)
    E = torch.randn(N + 1, D, generator=g).to(dev)
    P, Fe = torch.randn(L, D, generator=g).to(dev), torch.randn(3, F, generator=g).to(dev)
    w, b = torch.ones(H, device=dev), torch.zeros(H, device=dev)
    seq = torch.randint(1, N + 1, (B, L), generator=g).to(dev)
    rsq = torch.randint(1, 3, (B, L), generator=g).to(dev)
    x0 = [torch.empty(T, H, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    q = [torch.empty(T, H, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    st = torch.empty(T, 2, device=dev)
    run = lambda i: ops.embed_ln_fwd(E, P, Fe, 1, seq, rsq, 1.0, w, b, 1e-8, x0_bf16=x0[i % 2], q_bf16=q[i % 2], stats=st)
    for i in range(3):
        run(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(10):
        run(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    by = T * 600.0
    gbs = by / (ms * 1e-3) / 1e9
    return dict(kernel="srfrd_embed_ln_fwd", tokens=T, table_rows=N + 1, table_bytes=(N + 1) * D * 4, ms=round(ms, 4),
                roofline=dict(bound="hbm", achieved=round(gbs, 1), peak=pk["hbm"], unit="GB/s", frac=round(gbs / pk["hbm"], 4),
                              traffic=measured_traffic("srfrd_embed_ln_fwd@C3"), bytes_per_token=600, peak_source=pk["src"]),
                config="C3 table (1M x 64 fp32, 256 MB > L2), 81920 x 50 tokens, all slots valid, SRFR D=64 F=16")


def bench_scale_kernels(dev, pk):
    """K4 (fused gather-dot + weighted BCE fwd/bwd), K5 (sparse embedding-gradient scatter-add) and K7 (dense Adam) at
    catalogue scale -- 1 M x 64 fp32 item table and gradient (256 MB each, beyond L2), 2 M tokens with every slot valid --
    each against the HBM roofline (SURVEY 8d: at C2 the 3 MB table is L2-resident, so the HBM fraction must be shown here).
    K5's destination rows are random (uniform over 1 M rows): the bound there is the L2 atomic unit, not HBM."""
    from srfrd_b200 import ops
    N, D, F, L, B = 1_000_000, 64, 16, 50, 40960
    T, H = B * L, D + F
    g = torch.Generator(device="cpu").manual_seed(1240)
    E = torch.randn(N + 1, D, generator=g).to(dev)
    dE = torch.zeros(N + 1, D, device=dev)
    pos = torch.randint(1, N + 1, (T,), generator=g).to(dev)
    neg = torch.randint(1, N + 1, (T,), generator=g).to(dev)
    h = torch.randn(T, D, generator=g).to(dev) * 0.1
    dh = torch.empty(T, D, device=dev)
    norm, acc = torch.zeros(2, device=dev), torch.zeros(2, device=dev)
    ops.weight_sums(pos, None, None, norm)

    def timeit(fn):
        iters = int(os.environ.get("SRFRD_SCALE_ITERS", 5))          # (1 under ncu: one launch of each kernel)
        for _ in range(2 if iters > 1 else 0):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    def roof(ms, by, key, per):
        gbs = by / (ms * 1e-3) / 1e9
        return dict(ms=round(ms, 4), roofline=dict(bound="hbm", achieved=round(gbs, 1), peak=pk["hbm"], unit="GB/s",
                                                   frac=round(gbs / pk["hbm"], 4), traffic=measured_traffic(key),
                                                   algorithmic_bytes=int(by), bytes_per_unit=per, peak_source=pk["src"]))
    out = {}
    ms = timeit(lambda: ops.score_loss_fused(h, E, None, pos, neg, None, None, None, None, norm, acc, dh, dE, None))
    per = 16 + D * 4 + 2 * D * 4 + D * 4 + 2 * 2 * D * 4          # ids, h, two gathered rows, dh, two read-modify-write rows
    out["k4"] = dict(kernel="srfrd_score_loss_fused", tokens=T, **roof(ms, T * per, "srfrd_score_loss_fused@C3", f"{per} B/token"))
    del h, dh
    dx0 = (torch.randn(T, H, generator=g) * 0.1).to(torch.bfloat16).to(dev)
    seq = torch.randint(1, N + 1, (B, L), generator=g).to(dev)
    rsq = torch.randint(1, 3, (B, L), generator=g).to(dev)
    dF = torch.zeros(3, F, device=dev)
    ms = timeit(lambda: ops.embed_bwd(dx0, seq, rsq, D, F, 1, 1.0, dE, dF))
    per = 16 + H * 2 + D * 8
    out["k5"] = dict(kernel="srfrd_embed_bwd", tokens=T, **roof(ms, T * per, "srfrd_embed_bwd@C3", f"{per} B/token"),
                     note="uniform random destination rows over a 256 MB fp32 gradient table: bound by the L2 atomic units "
                          "(red.global.add.f32, one 4-byte reduction per element), see tools/microbench")
    del dx0
    n = (N + 1) * D
    p_, g_, m_, v_ = (torch.zeros(n, device=dev) for _ in range(4))
    g_.normal_(generator=None)
    st = torch.zeros(8, device=dev)
    ops.adam_tick(st, 0.9, 0.98)
    ms = timeit(lambda: ops.adam_step(p_, g_, m_, v_, 1e-3, 0.9, 0.98, 1e-8, st, zero_grad=True))
    out["k7"] = dict(kernel="srfrd_adam_step", params=n, **roof(ms, n * 32.0, "srfrd_adam_step@C3", "32 B/param (read p g m v, write p m v g)"))
    out["config"] = "C3-scale: 1M x 64 fp32 item table + gradient, 40960 x 50 tokens all valid, uniform random ids"
    return out


def bench_catalogue(dev, rank, world, pg, args, pk, timed, dump=None):
    """C3: (a) score + top-k + all-gather + merge on given user representations (the roofline-graded part), (b) the same
    preceded by the sequence encoder on 16 384 Beauty-shaped sequences over the 1 M-item catalogue (SURVEY 8d metric 2:
    encode + score + top-k + all-gather + merge).  The table is row-sharded; the users are split over the ranks for the encode
    and their representations all-gathered (EV.encode_users).  `dump` (a dict) receives the top-10 scores and global item
    ids of the last timed pass of (a) and (b)."""
    from srfrd_b200 import evaluation as EV, synth, _lib
    N, D, U = 1_000_000, 64, 16384
    lo, hi = EV.CatalogueIndex.shard_bounds(N + 1, rank, world)
    m = make_model(dev, N, 50, D, 16, 2, seed=1237)             # xavier_normal_ on the (N+1, D) table (trainer.py:364-369)
    table = m.flat_parameters().view(m.spec.item_key)
    table.copy_(table.to(torch.bfloat16).float())              # bf16-representable rows (SURVEY 8d C3)
    index = EV.CatalogueIndex(table[lo:hi], lo)
    g = torch.Generator(device="cpu").manual_seed(99173)      # NOT the model's seed: the same stream would reproduce table rows
    feats = torch.randn(U, D, generator=g).to(dev)
    data = synth.make_interactions(1237, U, N, 5, 4.0, 50)
    seq, rsq, _ = synth.eval_sequences(data, 50, np.arange(U))
    seq, rsq = torch.from_numpy(seq).to(dev), torch.from_numpy(rsq).to(dev)
    out = {}

    def step(i):
        out["r"] = EV.sharded_topk(feats, index, pg, 1)

    def step_enc(i):
        f = EV.encode_users(m, seq, rsq, pg)                 # users split over the ranks, one all-gather of (U, 80) fp32
        out["e"] = EV.sharded_topk(f[:, :D], index, pg, 1)

    steps = max(3, min(args.steps, 10))
    ms = timed(step, steps, 3)
    ms_enc = timed(step_enc, steps, 3)
    if dump is not None:
        dump["catalogue_scores"], dump["catalogue_ids"] = (t.cpu() for t in out["r"])
        dump["catalogue_encode_scores"], dump["catalogue_encode_ids"] = (t.cpu() for t in out["e"])
    users_s = U * steps / (ms / 1e3)
    flops = 2.0 * U * (hi - lo) * D
    # kernel-only time of the scoring kernel on this rank
    recs = []
    _lib.set_profile(recs)
    for i in range(3):
        torch.cuda._sleep(20_000_000)
        step(i)
    torch.cuda.synchronize()
    _lib.set_profile(None)
    kms = np.mean([e0.elapsed_time(e1) for n, a, e0, e1 in recs if n == "srfrd_catalogue_topk"])
    tf = flops / (kms * 1e-3) / 1e12
    res = dict(value=round(users_s, 1), unit="users/s", users=U, items=N, D=D, shards=world, ms_per_pass=round(ms / steps, 4),
               config="C3: 1M items x D=64 bf16 table row-sharded, 16384 users, top-10, all-gather merge",
               with_encode=dict(value=round(U * steps / (ms_enc / 1e3), 1), unit="users/s", ms_per_pass=round(ms_enc / steps, 4),
                                what="SRFR encoder (D=64 F=16 L=50 2 blocks) on 16384 sequences + score + top-10 + all-gather + merge"),
               roofline=dict(bound="tensor", kernel="srfrd_catalogue_topk", achieved=round(tf, 1), peak=pk["tf_burst"],
                             unit="TFLOP/s", frac=round(tf / pk["tf_burst"], 4), avg_launch_ms=round(float(kms), 4),
                             traffic=measured_traffic("srfrd_catalogue_topk"), peak_source=pk["src"] + ", burst figure (kernel timed alone)"))
    del m, index
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------
def cpu_baseline(sample_steps=2, batch=None):
    """The reference's CPU path on this box's host cores, on a bounded sample of the SAME workload (C2 batches of 4096,
    soft discriminator weights, dropout 0.0).  kind "reference": the UNMODIFIED reference module SRFR_model.SRFR staged
    under oracle/_ref/ by oracle/build_ref.py (the upstream checkout itself does not exist on the GPU box) driven by the
    step of trainer.py:27-41 (forward, BCE over pos != 0 -- here with the discriminator weights of row L --, backward,
    Adam(1e-3, (0.9, 0.98))); kind "port": the oracle restatement of the same arithmetic when oracle/_ref is absent."""
    from oracle import build_ref, srfrd_oracle as O
    from srfrd_b200 import synth                 # synthetic data generator only: no product kernel or model on this path
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = CFG
    B = batch or c["batch"]
    data = synth.make_interactions(1236, c["usernum"], c["itemnum"], 5, 4.0, c["L"])
    sd = O.init_state_dict("SRFR", c["itemnum"], c["L"], c["D"], c["F"], 0, c["blocks"], seed=1236)
    smp = synth.BatchSampler(data, c["L"], seed=100)
    batches = [{k: torch.from_numpy(v) for k, v in smp.next_batch(B).items()} for _ in range(sample_steps + 1)]
    ws = [O.discriminator_weights(b["pos"], b["p_fake"], "soft") for b in batches]
    SR = build_ref.load_ref()
    if SR is not None:
        model = SR.SRFR(c["itemnum"], c["L"], c["D"], c["F"], 0.0, c["blocks"], c["heads"], "cpu")
        model.load_state_dict(sd)
        model.train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, betas=(0.9, 0.98))      # trainer.py:390

        def step(b, w):
            _, zp, zn = model(None, b["seq"], b["rsq"], b["pos"], b["prs"], b["neg"], b["nrs"])   # trainer.py:30
            opt.zero_grad()
            loss = O.weighted_loss(zp, zn, w)                                                     # trainer.py:36-38 + row L
            loss.backward()                                                                       # trainer.py:40
            opt.step()                                                                            # trainer.py:41
            return float(loss.item())                                                             # trainer.py:42
        kind = "reference"
    else:
        orc = O.OracleTrainer(sd, "SRFR", 1)
        step = lambda b, w: orc.step(b, w)
        kind = "port"
    step(batches[0], ws[0])                     # warm-up
    t0 = time.perf_counter()
    for b, w in zip(batches[1:], ws[1:]):
        step(b, w)
    dt = time.perf_counter() - t0
    return dict(value=round(B * sample_steps / dt, 1), unit="seqs/s", cores=cores, kind=kind,
                sample=f"{sample_steps} steps of batch {B} (C2 workload, fp32, dropout 0.0, soft discriminator weights), "
                       f"torch {torch.__version__} CPU with {cores} threads"
                       + (", unmodified reference SRFR_model.SRFR (oracle/_ref)" if kind == "reference" else ", oracle port"),
                seconds=round(dt, 2))


def gpu_eager_baseline(dev, sample_steps=10):
    """SURVEY 8(d) / BASELINE.md 3.4 'the honest bar': the reference's arithmetic (oracle port) as stock PyTorch eager fp32
    on the SAME B200 (cuBLAS / cuDNN / ATen kernels; the reference ships no GPU kernel of its own), C2 batches resident on
    the device.  A reported baseline like cpu_baseline: nothing of the product runs here."""
    from oracle import srfrd_oracle as O
    from srfrd_b200 import synth
    c = CFG
    B = c["batch"]
    data = synth.make_interactions(1236, c["usernum"], c["itemnum"], 5, 4.0, c["L"])
    sd = {k: v.to(dev) for k, v in O.init_state_dict("SRFR", c["itemnum"], c["L"], c["D"], c["F"], 0, c["blocks"], seed=1236).items()}
    orc = O.OracleTrainer(sd, "SRFR", 1)
    smp = synth.BatchSampler(data, c["L"], seed=100)
    batches = [{k: torch.from_numpy(v).to(dev) for k, v in smp.next_batch(B).items()} for _ in range(4)]
    ws = [O.discriminator_weights(b["pos"], b["p_fake"], "soft") for b in batches]
    for i in range(3):
        orc.step(batches[i % 4], ws[i % 4])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(sample_steps):
        orc.step(batches[i % 4], ws[i % 4])      # float(loss) inside: one D2H sync per step, as trainer.py:39 does
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dict(value=round(B * sample_steps / dt, 1), unit="seqs/s", kind="oracle port, PyTorch eager fp32 on this GPU",
                sample=f"{sample_steps} steps of batch {B}, batches resident on the device", ms_per_step=round(dt / sample_steps * 1e3, 3))


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    steps = max(1, args.steps)
    W = 1
    from oracle import srfrd_oracle as O  # noqa: F401  (checker doubles as the timed CPU port here)
    t0 = time.perf_counter()
    cpu = cpu_baseline(sample_steps=max(4, min(steps, 12)))
    line = dict(impl="reference", metric=METRIC, value=cpu["value"], unit="seqs/s", n_gpus=args.gpus, steps=max(4, min(steps, 12)),
                warmup=W, ms_per_step=round(1e3 * CFG["batch"] / cpu["value"], 2), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload="C2: SRFR D=64 F=16 L=50 2 blocks 1 head, 12101 items, batch 4096, soft discriminator "
                                     "weights, dropout 0.0, Adam(1e-3,(0.9,0.98)) -- reference CPU path (" + cpu["kind"] + ")"),
                cpu_baseline=cpu, e2e=dict(value=cpu["value"], unit="seqs/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                wall_s=round(time.perf_counter() - t0, 1))
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-catalogue", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C4 / C5 / dropout objects")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, save the loss of the last training step and the top-10 scores / ids of "
                         "the last catalogue passes as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves what the product's timed path computed: use it with --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
