"""Host-order trace of every library call the encoder makes, in a form that does not depend on addresses.

For each configuration of a fixed matrix (model kind and widths, heads, maxlen, dropout, the SRFRD_* switches) and each
entry path (the autograd model call + backward, an eval forward, encode_last, eager FusedTrainer steps with loss "bce"
and "ce", each on the dense and the packed token layout where it has one), every call into libsrfrd_b200.so is written
as one line:
  - the entry point's name;
  - the stream it was enqueued on: "main", "side", "side2" (HotPath's branch streams) or "comm" (FusedTrainer's);
  - every scalar argument;
  - every pointer argument as "b<n>+<offset>": the caching-allocator block it falls in, numbered by first appearance in
    that entry path's trace, and the byte offset into the block; null for a null pointer;
  - the fields of by-reference structs (GemmEpilogue, Mlp2Epilogue, PackDesc, RepackPart arrays), resolved the same way.
Two trees that make the same calls with the same scalars on the same buffers give identical files, whatever the workspace
names or the addresses; a refactor of the host-side sequence is checked by diffing the files of the two trees.

    python tools/launch_trace.py --out trace.json
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from srfrd_b200 import SRFR_model as M, _lib, ops  # noqa: E402
from srfrd_b200.trainer import FusedTrainer  # noqa: E402

N_ITEMS, B = 500, 12


class _Resolver:
    """Maps device pointers to (block number, offset) against the caching allocator's live blocks."""

    def __init__(self, streams):
        self.streams = streams
        self.ids = {}
        self.blocks = []

    def _refresh(self):
        self.blocks = []
        for seg in torch.cuda.memory_snapshot():
            for b in seg["blocks"]:
                if b["state"].startswith("active"):
                    self.blocks.append((b["address"], b["size"]))

    def ptr(self, p):
        for _ in range(2):
            for a, n in self.blocks:
                if a <= p < a + n:
                    k = self.ids.setdefault((a, n), len(self.ids))
                    return f"b{k}+{p - a}"
            self._refresh()
        raise RuntimeError(f"launch_trace: pointer {p:#x} is in no live caching-allocator block")

    def value(self, v, t):
        if t is C.c_void_p:
            if v is None:
                return None
            if v in self.streams:
                return self.streams[v]
            return self.ptr(v)
        if t is C.c_float:
            return C.c_float(v).value
        if t in (C.c_int, C.c_int64, C.c_uint32, C.c_uint64):
            return int(v)
        if isinstance(t, type) and issubclass(t, C._Pointer):
            obj = getattr(v, "_obj", v)                 # C.byref(struct) or a ctypes array
            if isinstance(obj, C.Array):
                return [self.struct(e) for e in obj]
            if isinstance(obj, C.Structure):
                return self.struct(obj)
            return obj.value
        raise TypeError(f"launch_trace: unhandled argument type {t}")

    def struct(self, s):
        return {f: self.value(getattr(s, f), t) for f, t in s._fields_}


class _Trace(list):
    """The list _lib.set_profile appends to: resolves each call while its buffers are alive."""

    def __init__(self, resolver):
        super().__init__()
        self.res = resolver

    def append(self, rec):
        name, args = rec[0], rec[1]
        types = _lib.SIGNATURES[name]
        super().append([name] + [self.res.value(a, t) for a, t in zip(args, types)])


def _batch(L, seed):
    rng = np.random.default_rng(seed)
    z = lambda: np.zeros((B, L), np.int64)
    seq, pos, neg = z(), z(), z()
    for b in range(B):
        n = 0 if b % 5 == 0 else int(rng.integers(1, L + 1)) if b % 3 else L
        if n:
            seq[b, L - n:] = rng.integers(1, N_ITEMS + 1, n)
            pos[b, L - n:] = rng.integers(1, N_ITEMS + 1, n)
            neg[b, L - n:] = rng.integers(1, N_ITEMS + 1, n)
    lab = lambda a: (a != 0) * rng.integers(1, 3, (B, L))
    out = dict(seq=seq, rsq=lab(seq), pos=pos, prs=lab(pos), neg=neg, nrs=lab(neg))
    return {k: torch.from_numpy(v).cuda() for k, v in out.items()}


# name -> (model constructor (maxlen) , maxlen, environment)
CONFIGS = {
    "SRFR 64+16 L50": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 50, {}),
    "SRFR 64+16 L50 drop0.5": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.5, 2, 1, "cuda"), 50, {}),
    "SRFR 45+5 L50 (ragged)": (lambda L: M.SRFR(N_ITEMS, L, 45, 5, 0.0, 2, 1, "cuda"), 50, {}),
    "SRFR 45+5 L50 (ragged) drop0.5": (lambda L: M.SRFR(N_ITEMS, L, 45, 5, 0.5, 2, 1, "cuda"), 50, {}),
    "SASRec 256 L50": (lambda L: M.SASRec(N_ITEMS, L, 256, 0.0, 2, 1, "cuda"), 50, {}),
    "SASRec 128 h1 L50": (lambda L: M.SASRec(N_ITEMS, L, 128, 0.0, 2, 1, "cuda"), 50, {}),
    "SASRec 128 h2 L50": (lambda L: M.SASRec(N_ITEMS, L, 128, 0.0, 2, 2, "cuda"), 50, {}),
    "SASRec 128 h2 L50 drop0.5": (lambda L: M.SASRec(N_ITEMS, L, 128, 0.5, 2, 2, "cuda"), 50, {}),
    "SRFRN 64+16 L50 drop0.5": (lambda L: M.SRFRN(N_ITEMS, L, 64, 16, 0.5, 2, 1, "cuda"), 50, {}),
    "SRFU_F 64 L50 drop0.5": (lambda L: M.SRFU_F(N_ITEMS, L, 64, L + 1, 0.5, 2, 1, "cuda"), 50, {}),
    "SRFR 64+16 L160 live1": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 160, {"SRFRD_LIVE_TILES": "1"}),
    "SRFR 64+16 L160 live0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 160, {"SRFRD_LIVE_TILES": "0"}),
    "SRFR 64+16 L200 live1": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 200, {"SRFRD_LIVE_TILES": "1"}),
    "SRFR 64+16 L200 live0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 200, {"SRFRD_LIVE_TILES": "0"}),
    "SASRec 128 h2 L200 drop0.5": (lambda L: M.SASRec(N_ITEMS, L, 128, 0.5, 2, 2, "cuda"), 200, {}),
    "SRFR 64+16 L50 FUSE_LN=0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 50, {"SRFRD_FUSE_LN": "0"}),
    "SRFR 64+16 L50 FUSE_FFN=0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 50, {"SRFRD_FUSE_FFN": "0"}),
    "SRFR 64+16 L200 HYBRID=0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 200, {"SRFRD_HYBRID": "0"}),
    "SRFR 64+16 L50 OVERLAP=0": (lambda L: M.SRFR(N_ITEMS, L, 64, 16, 0.0, 2, 1, "cuda"), 50, {"SRFRD_OVERLAP": "0"}),
}


def run_config(make, L, seed):
    torch.manual_seed(seed)
    m = make(L).to("cuda")
    eng = m._sync_flat()
    s = eng.spec
    b = _batch(L, seed)
    w = (torch.rand(B, L, device="cuda") * (b["pos"] != 0)).contiguous()
    main = torch.cuda.current_stream()
    streams = {main.cuda_stream: "main", eng.side.cuda_stream: "side", eng.side2.cuda_stream: "side2"}
    meta = dict(kind=s.kind, H=s.H, Hp=s.Hp, heads=s.num_heads, L=L, dropout=s.dropout,
                packed_mode=eng.packed_mode(B, L), oproj_bits=ops.attention_packed_oproj_supported(L, s.H, s.num_heads))
    entries = {}

    def trace(name, fn, extra=None):
        st = {**streams, **(extra or {})}
        rec = _Trace(_Resolver(st))
        _lib.set_profile(rec)
        try:
            fn()
        finally:
            _lib.set_profile(None)
        torch.cuda.synchronize()
        entries[name] = list(rec)

    args = lambda: (None, b["seq"], b["rsq"], b["pos"], b["prs"], b["neg"], b["nrs"])

    def autograd():
        m.train()
        h, zp, zn = m(*args())
        (h.sum() * 1e-3 + zp.sum() - zn.sum()).backward()

    def eval_fwd():
        m.eval()
        with torch.no_grad():
            m(*args())
        m.train()

    def encode_last(packed):
        keep = eng.packed_default
        eng.packed_default = packed
        try:
            m.encode_last(b["seq"], b["rsq"])
        finally:
            eng.packed_default = keep

    trace("autograd", autograd)
    trace("eval forward", eval_fwd)
    trace("encode_last dense", lambda: encode_last(False))
    trace("encode_last packed", lambda: encode_last(True))
    for loss in ("bce", "ce"):
        if loss == "ce" and s.kind == "SRFRN":
            continue
        for packed in (False, True):
            tr = FusedTrainer(m, use_graph=False, packed=packed, loss=loss)
            trace(f"trainer {loss} {'packed' if packed else 'dense'}", lambda: tr.step(b, w_pos=w),
                  {tr.comm.cuda_stream: "comm"})
    return dict(meta=meta, entries=entries)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    lines = ["{"]
    names = list(CONFIGS)
    for ci, name in enumerate(names):
        make, L, env = CONFIGS[name]
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            res = run_config(make, L, 1000 + ci)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        lines.append(f"{json.dumps(name)}: {{\"meta\": {json.dumps(res['meta'])},")
        ents = list(res["entries"].items())
        for ei, (en, calls) in enumerate(ents):
            lines.append(f"  {json.dumps(en)}: [")
            lines += [f"    {json.dumps(c)}{',' if k + 1 < len(calls) else ''}" for k, c in enumerate(calls)]
            lines.append(f"  ]{',' if ei + 1 < len(ents) else ''}")
        lines.append("}" + ("," if ci + 1 < len(names) else ""))
        print(f"{name}: {res['meta']['packed_mode']}, "
              + ", ".join(f"{en} {len(c)}" for en, c in ents), flush=True)
    lines.append("}")
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
