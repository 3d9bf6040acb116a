"""Host-side orchestration of the hot path: parameter layout, workspaces and the kernel sequence
for forward, backward, the fused loss and Adam.  Pure plumbing: every arithmetic step is a call
into libsrfrd_b200.so (see ops.py); there is no eager-PyTorch fallback for any of them.

The block wiring reproduces the reference's non-standard encoder (SRFR_model.py:109-121):
  Q = LN1(x); q = Q Wq^T + bq;  [k, v] = x Wkv^T + bkv  (UN-normalised x);  o = causal_attn(q, k, v)
  r = Q + o Wo^T + bo;  y = LN2(r);  z = relu(y W1^T + b1) W2^T + b2 + y;  x' = z * (seq != 0)
"""
from __future__ import annotations

import math
import os
from contextlib import contextmanager, nullcontext
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from . import ops

bf16 = torch.bfloat16
LN_EPS = 1e-8  # SRFR_model.py:77,80,86

KINDS = ("SRFR", "SRFRN", "SRFU_B", "SRFU_F", "SRFU_R", "SASRec")


@dataclass
class ModelSpec:
    kind: str
    item_number: int
    max_len: int
    D: int                       # item_embedding_size / hidden_units
    F: int = 0                   # fake_embedding_size (SRFR / SRFRN)
    n_labels: int = 0            # SRFU_*: rows of user_label_embed
    num_blocks: int = 2
    num_heads: int = 1
    dropout: float = 0.0

    def __post_init__(self):
        if self.kind not in KINDS:
            raise ValueError(f"unknown model kind {self.kind}")
        if self.H % self.num_heads:
            raise ValueError("hidden size must be divisible by num_heads")
        if (self.H // self.num_heads) % 2:
            raise ValueError(f"srfrd_b200: head width {self.H // self.num_heads} must be even (bf16 pairs)")

    @property
    def H(self) -> int:
        return self.D + self.F if self.kind in ("SRFR", "SRFRN") else self.D

    @property
    def Dout(self) -> int:       # width of the hidden state the model returns
        return self.H if self.kind == "SRFRN" else self.D

    # Activations and GEMM operands are laid out with their widths padded to a multiple of 16 (tcgen05 N granularity,
    # 16-byte TMA pitch); the padding columns are zero everywhere, parameters and LayerNorm statistics keep their
    # true widths.  The reference's own sizes (45 + 5, trainer.py:129-130; constructor defaults 50 + 10) need this.
    @property
    def Hp(self) -> int:
        return (self.H + 15) // 16 * 16

    @property
    def Dp(self) -> int:
        return (self.D + 15) // 16 * 16

    @property
    def Doutp(self) -> int:
        return self.Hp if self.kind == "SRFRN" else self.Dp

    @property
    def padded(self) -> bool:
        return self.Hp != self.H or self.Dp != self.D

    @property
    def mode(self) -> int:       # K1 mode
        return 1 if self.kind in ("SRFR", "SRFRN") else (2 if self.kind.startswith("SRFU") else 0)

    @property
    def item_scale(self) -> float:   # SASRec scales embeddings by sqrt(d), SRFR_model.py:622
        return float(self.D ** 0.5) if self.kind == "SASRec" else 1.0

    @property
    def item_key(self) -> str:
        return "item_emb.weight" if self.kind == "SASRec" else "embedding_layer.item_embed.weight"

    @property
    def pos_key(self) -> str:
        return "pos_emb.weight" if self.kind == "SASRec" else "embedding_layer.pos_embed.weight"

    @property
    def aux_key(self) -> Optional[str]:
        if self.mode == 1:
            return "embedding_layer.fake_embed.weight"
        if self.mode == 2:
            return "embedding_layer.user_label_embed.weight"
        return None

    def param_shapes(self) -> List[Tuple[str, Tuple[int, ...]]]:
        """state_dict names and shapes in the reference's registration order (SURVEY.md 8b)."""
        H, D, L, N = self.H, self.D, self.max_len, self.item_number
        out: List[Tuple[str, Tuple[int, ...]]] = []
        if self.kind == "SASRec":
            out += [("item_emb.weight", (N + 1, D)), ("pos_emb.weight", (L, D))]
        elif self.mode == 1:
            out += [("embedding_layer.item_embed.weight", (N + 1, D)),
                    ("embedding_layer.fake_embed.weight", (3, self.F)),
                    ("embedding_layer.pos_embed.weight", (L, D))]
        else:
            out += [("embedding_layer.item_embed.weight", (N + 1, D)),
                    ("embedding_layer.user_label_embed.weight", (self.n_labels, D)),
                    ("embedding_layer.pos_embed.weight", (L, D))]
        for i in range(self.num_blocks):
            out += [(f"attention_layernorms.{i}.weight", (H,)), (f"attention_layernorms.{i}.bias", (H,))]
        for i in range(self.num_blocks):
            out += [(f"attention_layers.{i}.in_proj_weight", (3 * H, H)), (f"attention_layers.{i}.in_proj_bias", (3 * H,)),
                    (f"attention_layers.{i}.out_proj.weight", (H, H)), (f"attention_layers.{i}.out_proj.bias", (H,))]
        for i in range(self.num_blocks):
            out += [(f"forward_layernorms.{i}.weight", (H,)), (f"forward_layernorms.{i}.bias", (H,))]
        for i in range(self.num_blocks):
            out += [(f"forward_layers.{i}.conv1.weight", (H, H, 1)), (f"forward_layers.{i}.conv1.bias", (H,)),
                    (f"forward_layers.{i}.conv2.weight", (H, H, 1)), (f"forward_layers.{i}.conv2.bias", (H,))]
        if self.kind == "SRFR":
            out += [("last_conv.weight", (D, H, 1)), ("last_conv.bias", (D,))]
        out += [("last_layernorm.weight", (self.Dout,)), ("last_layernorm.bias", (self.Dout,))]
        return out


class FlatParams:
    """All parameters in ONE fp32 buffer (plus a same-shaped gradient buffer): the Adam kernel, the
    gradient all-reduce and the bf16 shadow refresh each touch it in a single launch."""

    def __init__(self, spec: ModelSpec, device, alloc=None):
        """alloc(numel) -> fp32 tensor: lets the data-parallel trainer place the parameter buffer and the gradient bucket
        in symmetric (peer-mapped) memory; default = ordinary device memory."""
        self.spec = spec
        self.offsets: Dict[str, Tuple[int, Tuple[int, ...]]] = {}
        off = 0
        for name, shape in spec.param_shapes():
            n = int(math.prod(shape))
            self.offsets[name] = (off, shape)
            off += (n + 3) // 4 * 4                      # keep every view 16-byte aligned
        self.numel = off
        zeros = (lambda n: alloc(n).zero_()) if alloc is not None else (lambda n: torch.zeros(n, dtype=torch.float32, device=device))
        # parameter buffer + a 4-float tail (the fused data-parallel optimizer writes the step's loss there on every rank)
        self.data_ext = zeros(off + 4)
        self.data = self.data_ext[:off]
        self.data_tail = self.data_ext[off:]
        # gradient bucket = every parameter gradient followed by a 4-float tail that carries the step's loss accumulators:
        # data-parallel training moves gradients AND loss with ONE all-reduce over `grad_bucket`
        self.grad_bucket = zeros(off + 4)
        self.grad = self.grad_bucket[:off]
        self.grad_tail = self.grad_bucket[off:]

    def segments(self) -> List[Tuple[int, int]]:
        """(offset, numel) of every parameter tensor, in the reference's registration order (= model.parameters());
        the zero padding between tensors belongs to none of them."""
        return [(off, int(math.prod(shape))) for off, shape in self.offsets.values()]

    def view(self, name: str, grad: bool = False) -> torch.Tensor:
        off, shape = self.offsets[name]
        buf = self.grad if grad else self.data
        return buf[off:off + int(math.prod(shape))].view(shape)

    def mat(self, name: str, grad: bool = False) -> torch.Tensor:
        """2-D view (conv weights (out, in, 1) -> (out, in))."""
        v = self.view(name, grad)
        return v.view(v.shape[0], -1)


@dataclass
class _Saved:
    """What a saving forward used; backward() takes every input and layout decision from here."""
    seq: torch.Tensor
    aux_ids: Optional[torch.Tensor]
    B: int
    L: int
    T: int                                # activation rows: B * L dense, plan.cap packed
    row_ids: torch.Tensor                 # item id of every row (0: a pad row, zeroed by the row_ids epilogues)
    plan: Optional[ops.PackedPlan]        # None: dense layout
    hyb: Optional[Dict[str, torch.Tensor]]    # hybrid mode's dense attention operands (None: dense or tile layout)
    live: Optional[ops.LiveTiles]         # hybrid mode's live query tiles (None: every tile walked)
    p_drop: float
    seed: int
    step: Optional[torch.Tensor]
    fuse_ln: bool
    oproj: int                            # bit 0 / 1: the packed attention forward / backward takes the out-projection
    mlp2: bool                            # FFN1 + FFN2 (and their backward pair) as one mlp2_tn launch
    version: int

    def __getitem__(self, key: str):
        """saved["plan"] etc.: callers that read the forward's record as the dict it used to be keep working."""
        return getattr(self, key)


class HotPath:
    """Forward / backward kernel sequences over a FlatParams store, one sequence for the dense and the packed layout."""

    def __init__(self, spec: ModelSpec, params: FlatParams):
        self.spec, self.P = spec, params
        self.device = params.data.device
        self._ws_tokens = 0
        self._ws: Dict[str, torch.Tensor] = {}
        # bumped whenever the workspace is re-allocated: a captured CUDA graph holds raw pointers into it, so
        # FusedTrainer keys its graph on this and re-captures after a larger forward (evaluation chunk, bigger batch)
        self.ws_generation = 0
        self.fwd_version = 0            # stamps every forward; backward() of anything but the latest forward raises
        self.host_drop_counter = 0      # mixed into the dropout seed on the autograd path (no device step counter there)
        self._build_shadows()
        self.step_state = torch.zeros(8, dtype=torch.float32, device=self.device)   # Adam {step, bc1, bc2, uint32 step bits}
        # Independent branches of the step (the k/v projection next to LN1 + the q projection; every weight-gradient
        # GEMM next to the data-gradient chain) are enqueued on a second stream: captured into the CUDA graph they
        # become parallel branches, so one kernel's launch latency, tail and CTA skew are filled by the other's CTAs.
        self.side = torch.cuda.Stream(device=self.device)
        self.side2 = torch.cuda.Stream(device=self.device)     # a second independent branch (backward: dx through k | v)
        self.overlap = os.environ.get("SRFRD_OVERLAP", "1") != "0"
        self.drop_seed = 0x5EED5EED
        self.saved: Optional[_Saved] = None
        self._plans: Dict[Tuple[int, int], ops.PackedPlan] = {}
        self._lives: Dict[Tuple[int, int], ops.LiveTiles] = {}
        # experiment switches (DESIGN.md section 8), fixed for the engine's lifetime
        self.packed_default = os.environ.get("SRFRD_PACKED", "1") != "0"
        self.fuse_ffn = os.environ.get("SRFRD_FUSE_FFN", "1") != "0"    # FFN1 + FFN2 (and their backward pair) in one launch
        self.fuse_ln = os.environ.get("SRFRD_FUSE_LN", "1") != "0"      # LayerNorms in the epilogues of the GEMMs before them
        self.hybrid = os.environ.get("SRFRD_HYBRID", "1") != "0"        # packed layout for maxlen > 127 (packed_mode)
        self.live_tiles = os.environ.get("SRFRD_LIVE_TILES", "1") != "0"  # hybrid attention skips all-pad query tiles

    # ------------------------------------------------------------------ bf16 operand shadows
    def _build_shadows(self):
        s, P, dev = self.spec, self.P, self.device
        H, D, Hp, Dp = s.H, s.D, s.Hp, s.Dp
        self.sh: Dict[str, torch.Tensor] = {}
        self.vsh: Dict[str, torch.Tensor] = {}       # zero-padded fp32 shadows of biases (only when widths are padded)
        entries = []
        zb = lambda r, c: torch.zeros(r, c, dtype=bf16, device=dev)

        def vec(name, src, n_pad, dst_off=0, dst=None):
            """bias vector `src` (true length) -> self.vsh[name][dst_off : dst_off + len]; identity when nothing is padded"""
            if not s.padded:
                return
            if dst is None:
                dst = self.vsh.setdefault(name, torch.zeros(n_pad, dtype=torch.float32, device=dev))
            entries.append((src.view(1, -1), dst[dst_off:dst_off + src.numel()].view(1, -1), None))

        for i in range(s.num_blocks):
            win = P.mat(f"attention_layers.{i}.in_proj_weight")
            bin_ = P.view(f"attention_layers.{i}.in_proj_bias")
            self.sh[f"wq{i}"] = zb(Hp, Hp)                          # rows = output features (padded), K-major
            self.sh[f"wkv{i}"] = zb(2 * Hp, Hp)                     # k rows at [0, H), v rows at [Hp, Hp + H)
            self.sh[f"wqT{i}"] = zb(Hp, Hp)
            self.sh[f"wkvT{i}"] = zb(Hp, 2 * Hp)
            entries.append((win[:H], self.sh[f"wq{i}"][:H, :H], self.sh[f"wqT{i}"][:H, :H]))
            entries.append((win[H:2 * H], self.sh[f"wkv{i}"][:H, :H], self.sh[f"wkvT{i}"][:H, :H]))
            entries.append((win[2 * H:], self.sh[f"wkv{i}"][Hp:Hp + H, :H], self.sh[f"wkvT{i}"][:H, Hp:Hp + H]))
            vec(f"bq{i}", bin_[:H], Hp)
            vec(f"bkv{i}", bin_[H:2 * H], 2 * Hp)
            vec(f"bkv{i}", bin_[2 * H:], 2 * Hp, dst_off=Hp)
            for tag, key in (("wo", f"attention_layers.{i}.out_proj"), ("w1", f"forward_layers.{i}.conv1"),
                             ("w2", f"forward_layers.{i}.conv2")):
                self.sh[f"{tag}{i}"] = zb(Hp, Hp)
                self.sh[f"{tag}T{i}"] = zb(Hp, Hp)
                entries.append((P.mat(key + ".weight"), self.sh[f"{tag}{i}"][:H, :H], self.sh[f"{tag}T{i}"][:H, :H]))
                vec(f"b{tag[1]}{i}", P.view(key + ".bias"), Hp)
        if s.kind == "SRFR":
            self.sh["wc"] = zb(Dp, Hp)
            self.sh["wcT"] = zb(Hp, Dp)
            entries.append((P.mat("last_conv.weight"), self.sh["wc"][:D, :H], self.sh["wcT"][:H, :D]))
            vec("bc", P.view("last_conv.bias"), Dp)
        self._cast_entries = entries
        self._cast_table, self._cast_n = ops.make_cast_table(entries, dev)
        self.shadows_version = -1

    def enable_ce_table(self) -> torch.Tensor:
        """The bf16 K-major copy of the item table the catalogue cross-entropy kernels read, (N + 1, Dp) with zero
        padding columns, refreshed by the same cast launch as every other shadow from then on.  The table is cast in
        blocks of rows so that a large catalogue spreads over many CTAs of that launch."""
        if "ce_table" not in self.sh:
            s = self.spec
            E = self.P.view(s.item_key)
            self.sh["ce_table"] = torch.zeros(E.shape[0], s.Dp, dtype=bf16, device=self.device)
            for r0 in range(0, E.shape[0], 4096):
                self._cast_entries.append((E[r0:r0 + 4096], self.sh["ce_table"][r0:r0 + 4096, :s.D], None))
            self._cast_table, self._cast_n = ops.make_cast_table(self._cast_entries, self.device)
            self.refresh_shadows()
        return self.sh["ce_table"]

    def bias(self, tag: str, i: Optional[int] = None) -> torch.Tensor:
        """Bias vector a GEMM epilogue reads (length = the GEMM's padded N)."""
        s, P = self.spec, self.P
        if s.padded:
            return self.vsh[tag if i is None else f"{tag}{i}"]
        if tag == "bq":
            return P.view(f"attention_layers.{i}.in_proj_bias")[:s.H]
        if tag == "bkv":
            return P.view(f"attention_layers.{i}.in_proj_bias")[s.H:]
        if tag == "bc":
            return P.view("last_conv.bias")
        key = {"bo": f"attention_layers.{i}.out_proj.bias", "b1": f"forward_layers.{i}.conv1.bias",
               "b2": f"forward_layers.{i}.conv2.bias"}[tag]
        return P.view(key)

    def refresh_shadows(self):
        """fp32 master weights -> bf16 GEMM operands (W and W^T); one launch."""
        ops.cast_weights(self._cast_table, self._cast_n)

    @contextmanager
    def _branch(self, second: bool = False):
        """Run the enclosed launches on a side stream, ordered after everything enqueued so far on the main one."""
        if not self.overlap:
            yield
            return
        main = torch.cuda.current_stream()
        st = self.side2 if second else self.side
        st.wait_stream(main)
        with torch.cuda.stream(st):
            yield

    def _join(self, second: bool = False):
        if self.overlap:
            torch.cuda.current_stream().wait_stream(self.side2 if second else self.side)

    # ------------------------------------------------------------------ workspaces
    def _workspace(self, T: int, L: int) -> Dict[str, torch.Tensor]:
        """Activation / gradient buffers for up to T tokens.  Everything whose size depends on the sequence length
        (pos_tmp, the long-sequence softmax statistics) is sized by spec.max_len, so reuse depends on T only."""
        if T <= self._ws_tokens:
            return self._ws
        s, dev = self.spec, self.device
        Lmax = max(L, s.max_len)
        H, nb = s.Hp, s.num_blocks               # padded widths; padding columns stay zero (buffers start zeroed and
        ws: Dict[str, torch.Tensor] = {}         # no kernel ever writes a non-zero value there)

        def act(name, w=H, dtype=bf16):
            ws[name] = torch.zeros(T, w, dtype=dtype, device=dev)

        for i in range(nb + 1):
            act(f"x{i}")
        for i in range(nb):
            for n in ("Q", "q", "o", "r", "y", "h1"):
                act(f"{n}{i}")
            act(f"kv{i}", 2 * H)
            act(f"st1_{i}", 2, torch.float32)
            act(f"st2_{i}", 2, torch.float32)
            if Lmax > 128:                           # softmax row statistics for the tile-pair backward (maxlen > 128)
                ws[f"ast{i}"] = torch.zeros(T * s.num_heads, 4, dtype=torch.float32, device=dev)
        if s.kind == "SRFR":
            act("c", s.Dp)
        act("stF", 2, torch.float32)
        act("hfin", s.Doutp, torch.float32)
        act("dh", s.Doutp, torch.float32)
        for n in ("gA", "gC", "gD", "gX"):          # data-gradient chain only (never read by a side-stream GEMM)
            act(n)
        for i in range(nb):                         # operands of weight-gradient GEMMs: one buffer each, so a later
            for n in ("gda1_", "gdr_", "gdq_"):     # kernel of the main chain never overwrites what a side-stream
                act(f"{n}{i}")                      # wgrad is still reading
            act(f"gdz_{i}")
            act(f"gdkv_{i}", 2 * H)
        if s.kind == "SRFR":
            act("gc", s.Dp)
        if s.dropout > 0:
            for i in range(nb):
                act(f"gE_{i}")
        ws["pos_tmp"] = torch.zeros(Lmax * H, dtype=torch.float32, device=dev)
        self._ws, self._ws_tokens = ws, T
        self.ws_generation += 1
        return ws

    # ------------------------------------------------------------------ packed token layout
    def packed_ok(self, B: int, L: int) -> bool:
        """Can this batch shape run on the packed token layout (csrc/pack.cu: no work on pad slots)?  Needs widths that
        are multiples of 16 (no ragged padding columns), tcgen05 attention with a whole sequence + its pad representative
        in one 128-row tile, and at most 16384 sequences per call."""
        return self.packed_mode(B, L) is not None

    def packed_mode(self, B: int, L: int) -> Optional[str]:
        """'tile': everything incl. attention on packed rows (a sequence + its pad representative fit one 128-row tile);
        'hybrid': row-wise kernels on packed rows, attention on the dense (B, L) layout with pack / unpack copies around it
        (128 <= maxlen: the tile-pair kernels of attention_long.cu); None: dense layout only."""
        s = self.spec
        if s.padded or s.H % 16 or s.D % 8 or B > 16384 or B < 1:
            return None
        if ops.attention_packed_supported(L, s.H, s.num_heads):
            return "tile"
        if self.hybrid and L <= 4096:
            return "hybrid"
        return None

    def _hybrid_ws(self, Td: int) -> Dict[str, torch.Tensor]:
        """Dense-layout attention operands of the hybrid mode: q, k|v, o per block (kept for backward) + gradient scratch."""
        hw = getattr(self, "_hws", None)
        if hw is not None and hw["_rows"] >= Td:
            return hw
        s, dev = self.spec, self.device
        Hp = s.Hp
        hw = {"_rows": Td}
        z = lambda w: torch.zeros(Td, w, dtype=bf16, device=dev)
        for i in range(s.num_blocks):
            hw[f"qd{i}"], hw[f"kvd{i}"], hw[f"od{i}"] = z(Hp), z(2 * Hp), z(Hp)
        hw["dod"], hw["dqd"], hw["dkvd"] = z(Hp), z(Hp), z(2 * Hp)
        self._hws = hw
        self.ws_generation += 1
        return hw

    def _cached(self, cache: dict, key, make):
        """cache[key], made on a miss.  A captured graph may hold pointers into the entries, so when a fifth key arrives the
        cache is cleared and ws_generation bumped (FusedTrainer then re-captures)."""
        if key not in cache:
            if len(cache) >= 4:
                cache.clear()
                self.ws_generation += 1
            cache[key] = make()
        return cache[key]

    # ------------------------------------------------------------------ forward
    def _aux_ids(self, fake_ids: Optional[torch.Tensor], B: int, L: int) -> Optional[torch.Tensor]:
        """The embedding's aux ids: the per-token fake labels (SRFR / SRFRN) or the per-user labels (SRFU_*)."""
        s = self.spec
        if s.mode == 1:
            return None if fake_ids is None else fake_ids.contiguous()
        if s.mode != 2:
            return None
        aux_ids = torch.empty(B, dtype=torch.int64, device=self.device)
        ops.srfu_labels(fake_ids.contiguous(), {"SRFU_B": 0, "SRFU_F": 1, "SRFU_R": 2}[s.kind], aux_ids)
        # label ranges are static per kind: B {1, 2}, F [0, L], R [0, 10] (SRFR_model.py:546-570; the reference's own
        # zoo passes 3 / maxlen + 1 / 11 rows, trainer.py:173-205).  A smaller table (e.g. the constructor default
        # number_of_labels = 2) makes the reference raise IndexError when such a label occurs; only in that
        # under-provisioned case the labels are checked here (one D2H sync) instead of reading past the table.
        need = {"SRFU_B": 3, "SRFU_F": L + 1, "SRFU_R": 11}[s.kind]
        if s.n_labels < need and B > 0 and int(aux_ids.max()) >= s.n_labels:
            raise IndexError(f"index out of range in self: {s.kind} user label {int(aux_ids.max())} needs "
                             f"number_of_labels >= {need}, got {s.n_labels}")
        return aux_ids

    def forward(self, seq: torch.Tensor, fake_ids: Optional[torch.Tensor], training: bool,
                last_only: bool = False, save: Optional[bool] = None, packed: bool = False,
                keep: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Encoder forward.  Returns hidden (B, L, Dout) fp32 -- or (B, Dout) for last_only (predict uses
        hidden[:, -1, :] only, SRFR_model.py:147).  Saves what backward needs when training.
        packed=True runs on the packed token layout (pad slots are not computed; `keep` (B, L) marks pad slots that must
        still get a row because they carry a loss term): the full hidden state is then left in PACKED rows in the
        workspace (ws["hfin"], row maps in the plan) and only last_only returns a dense result.  The packed row count M is
        data dependent and lives on the device: every row-wise kernel reads it through ops.row_limit, the packed kernels
        take the plan."""
        s, P = self.spec, self.P
        B, L = seq.shape
        if L > s.max_len:
            raise RuntimeError(f"sequence length {L} exceeds max_len {s.max_len} (pos_embed rows, SRFR_model.py:12)")
        H, Hp, nb = s.H, s.Hp, s.num_blocks
        plan = self._cached(self._plans, (B, L), lambda: ops.PackedPlan(B, L, self.device)) if packed else None
        T = plan.cap if packed else B * L
        ws = self._workspace(T, L)
        self.fwd_version += 1                   # EVERY forward overwrites the shared activations (saving or not)
        p_drop = s.dropout if training else 0.0
        step = self.step_state[3:4] if p_drop > 0 else None      # integer step counter bits (adam_tick), never stalls
        # FusedTrainer advances the device step counter (step_state[0]) once per step, which gives a captured graph a fresh
        # mask per replay; the autograd path (model.forward + a torch optimizer, trainer.simulate) has no such counter, so
        # _EncodeAndScore bumps host_drop_counter per training forward and it is folded into the seed here
        seed = (self.drop_seed + self.host_drop_counter * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        seq = seq.contiguous()
        aux_ids = self._aux_ids(fake_ids, B, L)
        hyb = live = None
        if packed:
            plan.build(seq, None if keep is None else keep.contiguous())
            if self.packed_mode(B, L) == "hybrid":
                hyb = self._hybrid_ws(B * L)
                if self.live_tiles:
                    # query tiles whose 128 positions are all dropped padding (C4: the first tile of 58 % of the sequences):
                    # the dense-layout attention kernels skip them -- nothing reads a pad query's o / dq and its dO is zero
                    live = self._cached(self._lives, (B, L), lambda: ops.LiveTiles(B, L, s.num_heads, self.device))
                    live.build(plan)
        # rows wider than the true width (ragged H, zero padded) keep the separate LayerNorm with true-width statistics
        fuse_ln = H == Hp and Hp <= 128 and self.fuse_ln
        # the packed tile attention takes the out-projection (bit 0 forward, bit 1 backward) with one head at the
        # fused-LayerNorm width when the kernel's shared-memory plan fits; otherwise the separate gemm_tn launches
        oproj = 0
        if packed and hyb is None and s.num_heads == 1 and fuse_ln:
            oproj = ops.attention_packed_oproj_supported(L, H, s.num_heads)
        sv = _Saved(seq=seq, aux_ids=aux_ids, B=B, L=L, T=T, row_ids=plan.row_ids if packed else seq.view(-1), plan=plan,
                    hyb=hyb, live=live, p_drop=p_drop, seed=seed, step=step, fuse_ln=fuse_ln, oproj=oproj,
                    mlp2=packed and self.fuse_ffn and Hp <= 128, version=self.fwd_version)
        x = [ws[f"x{i}"][:T] for i in range(nb + 1)]
        with ops.row_limit(plan.rows) if packed else nullcontext():
            emb = (P.view(s.item_key), P.view(s.pos_key), P.view(s.aux_key) if s.aux_key else None, s.mode, seq, aux_ids,
                   s.item_scale, P.view("attention_layernorms.0.weight"), P.view("attention_layernorms.0.bias"), LN_EPS)
            emb_drop = dict(drop_p=p_drop if s.kind == "SASRec" else 0.0, drop_seed=seed, drop_stream=1, drop_step=step)
            if packed:
                ops.embed_ln_fwd_packed(*emb, x[0], ws["Q0"][:T], ws["st1_0"][:T], plan, **emb_drop)
            else:
                ops.embed_ln_fwd(*emb, x0_bf16=x[0], q_bf16=ws["Q0"][:T], stats=ws["st1_0"][:T], **emb_drop)
            for i in range(nb):
                Q, q, kv, o, r, y, h1 = (ws[f"{n}{i}"][:T] for n in ("Q", "q", "kv", "o", "r", "y", "h1"))
                with self._branch():                                   # k | v need the un-normalised x only
                    ops.gemm_tn(x[i], self.sh[f"wkv{i}"], out_bf16=kv, bias=self.bias("bkv", i))
                if i > 0 and not fuse_ln:
                    ops.layernorm_fwd(x[i], P.view(f"attention_layernorms.{i}.weight"), P.view(f"attention_layernorms.{i}.bias"),
                                      LN_EPS, y_bf16=Q, stats=ws[f"st1_{i}"][:T], H=H)
                ops.gemm_tn(Q, self.sh[f"wq{i}"], out_bf16=q, bias=self.bias("bq", i))
                self._join()                                           # k | v (side stream) are ready
                ln2 = dict(ln_w=P.view(f"forward_layernorms.{i}.weight"), ln_b=P.view(f"forward_layernorms.{i}.bias"),
                           ln_eps=LN_EPS, ln_stats=ws[f"st2_{i}"][:T])
                fold = dict(wo=self.sh[f"wo{i}"], bias=self.bias("bo", i), residual=Q, r=r, y=y, **ln2) if oproj & 1 else {}
                self._attention_fwd(sv, i, q, kv, o, ws.get(f"ast{i}"), fold)
                if oproj & 1:
                    pass                    # r, y and their statistics came out of the attention kernel
                elif fuse_ln:                                          # LayerNorm computed in the GEMM's epilogue
                    ops.gemm_tn(o, self.sh[f"wo{i}"], out_bf16=r, bias=self.bias("bo", i), residual=Q, ln_out=y, **ln2)
                else:
                    ops.gemm_tn(o, self.sh[f"wo{i}"], out_bf16=r, bias=self.bias("bo", i), residual=Q)
                    ops.layernorm_fwd(r, ln2["ln_w"], ln2["ln_b"], LN_EPS, y_bf16=y, stats=ln2["ln_stats"], H=H)
                nxt = {}
                if fuse_ln and i + 1 < nb:                             # the next block's attention LayerNorm rides along
                    nxt = dict(ln_out=ws[f"Q{i + 1}"][:T], ln_w=P.view(f"attention_layernorms.{i + 1}.weight"),
                               ln_b=P.view(f"attention_layernorms.{i + 1}.bias"), ln_eps=LN_EPS,
                               ln_stats=ws[f"st1_{i + 1}"][:T])
                if sv.mlp2:                 # FFN1 + FFN2 (+ the next LayerNorm) in one launch, h1 through smem (packed only)
                    ops.mlp2_tn(y, self.sh[f"w1{i}"], self.sh[f"w2{i}"], h1, x[i + 1], bias1=self.bias("b1", i),
                                bias2=self.bias("b2", i), relu1=True, drop1_p=p_drop, drop2_p=p_drop, drop1_stream=11 + 4 * i,
                                drop2_stream=12 + 4 * i, drop_seed=seed, drop_step=step, residual_is_a=True,
                                row_ids=sv.row_ids, **nxt)
                else:
                    ops.gemm_tn(y, self.sh[f"w1{i}"], out_bf16=h1, bias=self.bias("b1", i), relu=True,
                                drop_p=p_drop, drop_seed=seed, drop_stream=11 + 4 * i, drop_step=step)
                    ops.gemm_tn(h1, self.sh[f"w2{i}"], out_bf16=x[i + 1], bias=self.bias("b2", i), residual=y,
                                row_ids=sv.row_ids, drop_p=p_drop, drop_seed=seed, drop_stream=12 + 4 * i, drop_step=step,
                                **nxt)
            fin_in = x[nb]
            if s.kind == "SRFR":      # last_conv H -> D (SRFR_model.py:123)
                ops.gemm_tn(x[nb], self.sh["wc"], out_bf16=ws["c"][:T], bias=self.bias("bc"))
                fin_in = ws["c"][:T]
            if not last_only:
                ops.layernorm_fwd(fin_in, P.view("last_layernorm.weight"), P.view("last_layernorm.bias"), LN_EPS,
                                  y_f32=ws["hfin"][:T], stats=ws["stF"][:T], H=s.Dout)
        if last_only:               # the final LayerNorm of each sequence's last position only
            out = ws["hfin"][:B]
            if packed:
                ops.layernorm_fwd_rows(fin_in, P.view("last_layernorm.weight"), P.view("last_layernorm.bias"), LN_EPS, out,
                                       plan.last_row, B, s.Dout)
            else:                   # row L - 1 of every sequence: a strided row walk
                ops.layernorm_fwd(fin_in, P.view("last_layernorm.weight"), P.view("last_layernorm.bias"), LN_EPS, y_f32=out,
                                  T=B, H=s.Dout, row_stride=L, row_offset=L - 1)
            return out[:, :s.Dout]
        if training if save is None else save:
            self.saved = sv
        return ws["hfin"][:T] if packed else ws["hfin"][:T].view(B, L, s.Doutp)[..., :s.Dout]

    def _attention_fwd(self, sv: "_Saved", i: int, q, kv, o, stats, fold: dict) -> None:
        """o = attention(q, k | v) of block i.  Packed tile layout: the packed kernel, which with `fold` (oproj bit 0) also
        writes r, y and y's statistics.  Dense layout: the dense kernel.  Hybrid: the dense kernel on dense copies of the
        packed rows, under the live-tile list when there is one."""
        s, Hp = self.spec, self.spec.Hp
        drop = (sv.p_drop, sv.seed, 10 + 4 * i, sv.step)
        if sv.plan is not None and sv.hyb is None:
            ops.attention_fwd_packed(q, kv[:, :Hp], kv[:, Hp:], o, sv.plan, sv.L, s.H, s.num_heads, *drop, **fold)
            return
        qd, kvd, od = q, kv, o
        if sv.hyb is not None:
            Td = sv.B * sv.L
            qd, kvd, od = sv.hyb[f"qd{i}"][:Td], sv.hyb[f"kvd{i}"][:Td], sv.hyb[f"od{i}"][:Td]
            ops.unpack_rows([(q, qd, Hp, 0), (kv, kvd, 2 * Hp, 0)], sv.plan)
        with sv.live.active() if sv.live is not None else nullcontext():
            ops.attention_fwd(qd, kvd[:, :Hp], kvd[:, Hp:], od, sv.B, sv.L, s.H, s.num_heads, *drop, stats=stats)
        if sv.hyb is not None:
            ops.pack_rows([(od, o, Hp, 0)], sv.plan)

    # ------------------------------------------------------------------ backward
    def check_saved(self, version: Optional[int] = None) -> "_Saved":
        """The record of the forward being back-propagated.  The activations live in the engine's shared workspace, so
        only the LATEST saving forward can be back-propagated: `version` (the stamp an autograd node took at forward
        time) is checked against it."""
        sv = self.saved
        if sv is None and version is None:
            raise RuntimeError("backward() without a training forward()")
        if sv is None or sv.version != self.fwd_version or (version is not None and version != sv.version):
            raise RuntimeError("srfrd_b200: backward() of a stale forward -- another forward() (training, validation or "
                               "predict) ran on this model after the one being back-propagated and overwrote the shared "
                               "activation workspace; run backward() before the next forward()")
        return sv

    def backward(self, dh: torch.Tensor, version: Optional[int] = None) -> None:
        """Given dL/dhidden (T, Dout) fp32 -- T rows of the forward's layout -- accumulate every parameter gradient into
        P.grad (the score kernels have already added the pos/neg rows of the item table).  Every layout decision is the
        saving forward's (check_saved)."""
        s, P = self.spec, self.P
        sv = self.check_saved(version)
        T, H, Hp, nb = sv.T, s.H, s.Hp, s.num_blocks
        ws = self._ws
        row_ids = sv.row_ids
        p_drop, seed, step = sv.p_drop, sv.seed, sv.step
        gA, gC, gD, gX = (ws[n][:T] for n in ("gA", "gC", "gD", "gX"))
        G = lambda name: P.view(name, grad=True)
        GM = lambda name: P.mat(name, grad=True)
        x = [ws[f"x{i}"][:T] for i in range(nb + 1)]
        dz_top = ws[f"gdz_{nb - 1}"][:T]
        with ops.row_limit(sv.plan.rows) if sv.plan is not None else nullcontext():
            # final LayerNorm (+ last_conv) -> dz = dL/dx[nb], pad rows zeroed
            if s.kind == "SRFR":
                gc = ws["gc"][:T]
                ops.layernorm_bwd(dh, ws["c"][:T], ws["stF"][:T], P.view("last_layernorm.weight"), gc,
                                  G("last_layernorm.weight"), G("last_layernorm.bias"), H=s.D)
                with self._branch():
                    ops.gemm_wgrad(gc, x[nb], GM("last_conv.weight"), G("last_conv.bias"), Mo=s.D, No=H)
                ops.gemm_tn(gc, self.sh["wcT"], out_bf16=dz_top, row_ids=row_ids)
            else:
                ops.layernorm_bwd(dh, x[nb], ws["stF"][:T], P.view("last_layernorm.weight"), dz_top,
                                  G("last_layernorm.weight"), G("last_layernorm.bias"), row_ids=row_ids, H=s.Dout)

            for i in reversed(range(nb)):
                Q, q, kv, o, r, y, h1 = (ws[f"{n}{i}"][:T] for n in ("Q", "q", "kv", "o", "r", "y", "h1"))
                dz, da1, dr, dq, dkv = (ws[f"{n}{i}"][:T] for n in ("gdz_", "gda1_", "gdr_", "gdq_", "gdkv_"))
                dx_out = ws[f"gdz_{i - 1}"][:T] if i > 0 else gA          # dL/dx[i]: the next (earlier) block's dz
                dz2 = dz
                if p_drop > 0:      # da2 = dz * mask2 (dropout2 sits between conv2 and the residual add)
                    dz2 = ws[f"gE_{i}"][:T]
                    ops.dropout_apply(dz, dz2, Hp, p_drop, seed, 12 + 4 * i, step)
                # FFN: z = drop2(h1 W2^T + b2) + y ; h1 = relu(drop1(y W1^T + b1))
                with self._branch():
                    ops.gemm_wgrad(dz2, h1, GM(f"forward_layers.{i}.conv2.weight"), G(f"forward_layers.{i}.conv2.bias"),
                                   Mo=H, No=H)
                if sv.mlp2:                 # da1 = (dz2 W2) * drop1 * (h1 > 0);  dy = da1 W1 + dz: one launch
                    ops.mlp2_tn(dz2, self.sh[f"w2T{i}"], self.sh[f"w1T{i}"], da1, gC, gate=h1, drop1_p=p_drop,
                                drop1_stream=11 + 4 * i, drop_seed=seed, drop_step=step, residual=dz)
                else:
                    ops.gemm_tn(dz2, self.sh[f"w2T{i}"], out_bf16=da1, gate=h1, drop_p=p_drop, drop_seed=seed,
                                drop_stream=11 + 4 * i, drop_step=step)                               # da1
                with self._branch():
                    ops.gemm_wgrad(da1, y, GM(f"forward_layers.{i}.conv1.weight"), G(f"forward_layers.{i}.conv1.bias"),
                                   Mo=H, No=H)
                if not sv.mlp2:
                    ops.gemm_tn(da1, self.sh[f"w1T{i}"], out_bf16=gC, residual=dz)                     # dy
                # LN2
                ops.layernorm_bwd(gC, r, ws[f"st2_{i}"][:T], P.view(f"forward_layernorms.{i}.weight"), dr,
                                  G(f"forward_layernorms.{i}.weight"), G(f"forward_layernorms.{i}.bias"), H=H)   # dr
                # r = Q + o Wo^T + bo
                with self._branch():
                    ops.gemm_wgrad(dr, o, GM(f"attention_layers.{i}.out_proj.weight"),
                                   G(f"attention_layers.{i}.out_proj.bias"), Mo=H, No=H)
                if not sv.oproj & 2:        # otherwise dO = dr Wo inside the attention kernel
                    ops.gemm_tn(dr, self.sh[f"woT{i}"], out_bf16=gC)                                   # do
                self._attention_bwd(sv, i, gC, q, kv, o, dq, dkv, dr, ws.get(f"ast{i}"))               # dq, dk|dv
                gin = GM(f"attention_layers.{i}.in_proj_weight")
                gbin = G(f"attention_layers.{i}.in_proj_bias")
                with self._branch():
                    ops.gemm_wgrad(dq, Q, gin[:H], gbin[:H], Mo=H, No=H)
                    if Hp == H:
                        ops.gemm_wgrad(dkv, x[i], gin[H:], gbin[H:], Mo=2 * H, No=H)
                    else:   # k and v gradients sit at column offsets 0 and Hp: two row blocks of in_proj_weight
                        ops.gemm_wgrad(dkv[:, :Hp], x[i], gin[H:2 * H], gbin[H:2 * H], Mo=H, No=H)
                        ops.gemm_wgrad(dkv[:, Hp:], x[i], gin[2 * H:], gbin[2 * H:], Mo=H, No=H)
                with self._branch(second=True):                                                        # independent of dQ
                    ops.gemm_tn(dkv, self.sh[f"wkvT{i}"], out_bf16=gX)                                 # dx via k, v
                ops.gemm_tn(dq, self.sh[f"wqT{i}"], out_bf16=gD, residual=dr)                          # dQ = dr + dq Wq
                self._join(second=True)
                # LN1 + the un-normalised k/v path; pad rows zeroed (x_i was masked, SRFR_model.py:99,121)
                ops.layernorm_bwd(gD, x[i], ws[f"st1_{i}"][:T], P.view(f"attention_layernorms.{i}.weight"), dx_out,
                                  G(f"attention_layernorms.{i}.weight"), G(f"attention_layernorms.{i}.bias"),
                                  add=gX, row_ids=row_ids, H=H)
            dx0 = gA
            if s.kind == "SASRec" and p_drop > 0:
                ops.dropout_apply(gA, gC, H, p_drop, seed, 1, step)
                dx0 = gC

        # embedding tables
        aux_grad = G(s.aux_key) if s.aux_key else None
        F = s.F if s.mode == 1 else 0
        if sv.plan is not None:
            ops.embed_bwd_packed(dx0, sv.seq, sv.aux_ids, sv.plan, s.D, F, s.mode, s.item_scale, G(s.item_key), aux_grad,
                                 G(s.pos_key))
        else:
            ops.embed_bwd(dx0, sv.seq, sv.aux_ids, s.D, F, s.mode, s.item_scale, G(s.item_key), aux_grad)
            LH = sv.L * Hp
            pos_tmp = ws["pos_tmp"][:LH]      # zero on entry: allocated zeroed, and add_segments consumes (re-zeroes) it
            ops.colsum(dx0, pos_tmp, M=sv.B, N=LH, ld=LH)
            ops.add_segments(pos_tmp, LH, Hp, s.D, G(s.pos_key))
        self._join()                                # every weight gradient has landed in P.grad
        self.saved = None

    def _attention_bwd(self, sv: "_Saved", i: int, do, q, kv, o, dq, dkv, dr, stats) -> None:
        """dq, dk | dv of block i's attention from dO = `do`.  Packed tile layout: the packed kernel, which with oproj
        bit 1 computes dO = dr Wo itself.  Dense layout: the dense kernel.  Hybrid: the dense kernel on dense copies,
        under the live-tile list when there is one."""
        s, Hp = self.spec, self.spec.Hp
        drop = (sv.p_drop, sv.seed, 10 + 4 * i, sv.step)
        if sv.plan is not None and sv.hyb is None:
            fold = dict(dr=dr, woT=self.sh[f"woT{i}"]) if sv.oproj & 2 else {}
            ops.attention_bwd_packed(None if fold else do, q, kv[:, :Hp], kv[:, Hp:], dq, dkv[:, :Hp], dkv[:, Hp:], sv.plan,
                                     sv.L, s.H, s.num_heads, *drop, **fold)
            return
        dqd, dkvd = dq, dkv
        if sv.hyb is not None:
            Td, hyb = sv.B * sv.L, sv.hyb
            q, kv, o = hyb[f"qd{i}"][:Td], hyb[f"kvd{i}"][:Td], hyb[f"od{i}"][:Td]
            dod, dqd, dkvd = hyb["dod"][:Td], hyb["dqd"][:Td], hyb["dkvd"][:Td]
            ops.unpack_rows([(do, dod, Hp, 1)], sv.plan)                   # a pad query's output is dead: dO = 0
            do = dod
        with sv.live.active() if sv.live is not None else nullcontext():
            ops.attention_bwd(do, q, kv[:, :Hp], kv[:, Hp:], dqd, dkvd[:, :Hp], dkvd[:, Hp:], sv.B, sv.L, s.H, s.num_heads,
                              *drop, o=o, stats=stats)
        if sv.hyb is not None:
            # dk, dv of the pad representative = the sum over its sequence's pad slots (every copy of the pad key)
            ops.pack_rows([(dqd, dq, Hp, 0), (dkvd, dkv, 2 * Hp, 1)], sv.plan)

    # ------------------------------------------------------------------ scoring helpers
    def fake_table(self) -> Optional[torch.Tensor]:
        return self.P.view("embedding_layer.fake_embed.weight") if self.spec.kind == "SRFRN" else None

    def fake_table_grad(self) -> Optional[torch.Tensor]:
        return self.P.view("embedding_layer.fake_embed.weight", grad=True) if self.spec.kind == "SRFRN" else None
