"""Drop-in replacements for the reference's ``SRFR_model.py`` classes, running on the sm_100a kernels.

Same constructor signatures, ``forward`` / ``predict`` signatures and ``state_dict`` keys as the
reference (SRFR_model.py:53-63, :154-164, :429-440, :572-581), so ``simulate`` (trainer.py:15),
``evaluation`` (utils.py:544) and reference checkpoints work unchanged.  Underneath, all
parameters live in one flat fp32 buffer and every arithmetic step is a hand-written CUDA kernel;
``forward`` is ONE autograd node so the user's own criterion / optimizer still work.  The fused
no-sync training step (weighted BCE + Adam + CUDA graph) is ``srfrd_b200.trainer.FusedTrainer``.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn

from . import ops
from .engine import FlatParams, HotPath, ModelSpec

bf16 = torch.bfloat16


class _Node(nn.Module):
    """Parameter container used to reproduce the reference's nested state_dict names."""


def _attach(root: nn.Module, dotted: str, param: nn.Parameter) -> None:
    parts = dotted.split(".")
    mod = root
    for p in parts[:-1]:
        if p.isdigit():
            while len(mod) <= int(p):
                mod.append(_Node())
            mod = mod[int(p)]
        else:
            if not hasattr(mod, p):
                nxt = nn.ModuleList() if p in ("attention_layernorms", "attention_layers", "forward_layernorms",
                                               "forward_layers") else _Node()
                setattr(mod, p, nxt)
            mod = getattr(mod, p)
    mod.register_parameter(parts[-1], param)


class _EncodeAndScore(torch.autograd.Function):
    """hidden, pos_logits, neg_logits = f(parameters; ids) as a single autograd node."""

    @staticmethod
    def forward(ctx, model, seq, rsq, pos, prs, neg, nrs, *params):
        eng: HotPath = model._engine
        train = any(ctx.needs_input_grad)    # (grad mode is always off inside Function.forward)
        if model.training and eng.spec.dropout > 0:
            eng.host_drop_counter += 1           # a fresh dropout mask per training forward (reference: torch's RNG stream)
        with torch.no_grad():
            hidden = eng.forward(seq, rsq, training=model.training, save=train)
            ctx.version = eng.fwd_version
            B, L = seq.shape
            zp = zn = None
            if pos is not None or neg is not None:
                # the reference allows either to be None (SRFR_model.py:127-136); score both, drop one
                pp = pos if pos is not None else neg
                nn_ = neg if neg is not None else pos
                zp = torch.empty(B, L, dtype=torch.float32, device=seq.device)
                zn = torch.empty(B, L, dtype=torch.float32, device=seq.device)
                h2 = eng._ws["hfin"][:B * L]            # (T, Doutp) fp32, padding columns zero; score reads W true columns
                ft = eng.fake_table()
                ops.score_fwd(h2, eng.P.view(eng.spec.item_key), ft, pp.contiguous(), nn_.contiguous(),
                              None if ft is None else (prs if prs is not None else nrs).contiguous(),
                              None if ft is None else (nrs if nrs is not None else prs).contiguous(), zp, zn)
            out_hidden = hidden.clone()
        ctx.model, ctx.ids = model, (seq, rsq, pos, prs, neg, nrs)
        ctx.train = train
        return out_hidden, zp if pos is not None else None, zn if neg is not None else None

    @staticmethod
    def backward(ctx, d_hidden, d_zp, d_zn):
        model = ctx.model
        eng: HotPath = model._engine
        seq, rsq, pos, prs, neg, nrs = ctx.ids
        B, L = seq.shape
        T = B * L
        eng.check_saved(ctx.version)                # raises before score_bwd writes anything
        ws = eng._ws
        dh = ws["dh"][:T]
        eng.P.grad.zero_()
        if pos is not None or neg is not None:
            pp = pos if pos is not None else neg
            nn_ = neg if neg is not None else pos
            zero = torch.zeros(T, dtype=torch.float32, device=seq.device)
            dzp = d_zp.contiguous().view(-1).float() if (d_zp is not None and pos is not None) else zero
            dzn = d_zn.contiguous().view(-1).float() if (d_zn is not None and neg is not None) else zero
            ft = eng.fake_table()
            ops.score_bwd(ws["hfin"][:T], eng.P.view(eng.spec.item_key), ft, pp.contiguous(), nn_.contiguous(),
                          None if ft is None else (prs if prs is not None else nrs).contiguous(),
                          None if ft is None else (nrs if nrs is not None else prs).contiguous(), dzp, dzn, dh,
                          eng.P.view(eng.spec.item_key, grad=True), eng.fake_table_grad())
        else:
            dh.zero_()
        if d_hidden is not None:
            dh[:, :eng.spec.Dout].add_(d_hidden.reshape(T, -1))
        eng.backward(dh, ctx.version)
        grads = tuple(eng.P.view(n, grad=True).clone() for n in model._param_names)
        return (None,) * 7 + grads


class _HotPathModule(nn.Module):
    def __init__(self, spec: ModelSpec, device):
        super().__init__()
        self.spec = spec
        self.device = device
        self.dev = device
        self._param_names = [n for n, _ in spec.param_shapes()]
        for name, shape in spec.param_shapes():
            _attach(self, name, nn.Parameter(torch.empty(shape)))
        self._default_init()
        self._engine: Optional[HotPath] = None
        self._flat: Optional[FlatParams] = None

    # ---- initialisation: same distributions torch.nn gives the reference's layers ----
    @torch.no_grad()
    def _default_init(self):
        for name, p in self.named_parameters():
            if name.endswith(("item_embed.weight", "item_emb.weight", "fake_embed.weight")):
                p.normal_(0, 1)
                p[0].zero_()                                   # padding_idx=0 (SRFR_model.py:10-11, :591)
            elif "embed" in name or "emb." in name:
                p.normal_(0, 1)
            elif "layernorm" in name:
                p.fill_(1.0) if name.endswith("weight") else p.zero_()
            elif name.endswith("in_proj_weight"):
                nn.init.xavier_uniform_(p)
            elif name.endswith(("in_proj_bias", "out_proj.bias")):
                p.zero_()
            elif name.endswith("weight"):                      # Linear / Conv1d default
                nn.init.kaiming_uniform_(p, a=math.sqrt(5))
            else:                                              # conv biases
                fan_in = self.spec.H
                p.uniform_(-1 / math.sqrt(fan_in), 1 / math.sqrt(fan_in))

    # ---- flat parameter store -------------------------------------------------------
    def _sync_flat(self) -> HotPath:
        """(Re)build the flat fp32 store if .to(device) / load_state_dict replaced the parameter tensors."""
        params = dict(self.named_parameters())
        dev = params[self._param_names[0]].device
        if dev.type != "cuda":
            raise RuntimeError("srfrd_b200 models run on a CUDA (sm_100a) device only; call .to('cuda') -- "
                               "there is no CPU fallback")
        ok = self._flat is not None and self._flat.data.device == dev
        if ok:
            for n in self._param_names:
                if params[n].data_ptr() != self._flat.view(n).data_ptr():
                    ok = False
                    break
        if not ok:
            flat = FlatParams(self.spec, dev)
            with torch.no_grad():
                for n in self._param_names:
                    flat.view(n).copy_(params[n].detach().to(torch.float32))
                    params[n].data = flat.view(n)
            self._flat = flat
            self._engine = HotPath(self.spec, flat)
        return self._engine

    def rehome(self, alloc) -> HotPath:
        """Move the flat parameter store into buffers from `alloc(numel)` (symmetric / peer-mapped memory for the fused
        data-parallel optimizer) and rebuild the engine around them; parameter values are preserved."""
        self._sync_flat()
        params = dict(self.named_parameters())
        dev = params[self._param_names[0]].device
        flat = FlatParams(self.spec, dev, alloc)
        with torch.no_grad():
            for n in self._param_names:
                flat.view(n).copy_(params[n].detach().to(torch.float32))
                params[n].data = flat.view(n)
        self._flat = flat
        self._engine = HotPath(self.spec, flat)
        return self._engine

    def flat_parameters(self) -> FlatParams:
        self._sync_flat()
        return self._flat

    # ---- reference API ----------------------------------------------------------------
    def forward(self, user_ids, input_ids, fake_ids, positive_ids=None, positive_fake_ids=None, negative_ids=None,
                negative_fake_ids=None):
        eng = self._sync_flat()
        eng.refresh_shadows()
        params = [dict(self.named_parameters())[n] for n in self._param_names]
        to = lambda t: None if t is None else torch.as_tensor(t, device=eng.device).long()
        return _EncodeAndScore.apply(self, to(input_ids), to(fake_ids), to(positive_ids), to(positive_fake_ids),
                                     to(negative_ids), to(negative_fake_ids), *params)

    @torch.no_grad()
    def encode_last(self, input_ids, fake_ids) -> torch.Tensor:
        """hidden[:, -1, :] of forward() without materialising the other positions' final LayerNorm."""
        eng = self._sync_flat()
        eng.refresh_shadows()
        to = lambda t: None if t is None else torch.as_tensor(t, device=eng.device).long()
        seq = to(input_ids)
        packed = eng.packed_default and eng.packed_ok(seq.shape[0], seq.shape[1])
        return eng.forward(seq, to(fake_ids), training=False, last_only=True, packed=packed).clone()

    @torch.no_grad()
    def predict(self, user_ids, input_ids, fake_ids, label):
        """logits (U, I) = hidden[:, -1, :] . E[label]^T  (SRFR_model.py:144-152), squeezed like the reference."""
        eng = self._engine if self._engine is not None else self._sync_flat()
        feats = self.encode_last(input_ids, fake_ids)                      # (U, Dout) fp32
        label = torch.as_tensor(label, device=eng.device).long().view(-1)
        logits = _split_gemm_logits(feats[:, :self.spec.D], eng.P.view(self.spec.item_key), label)
        if self.spec.kind == "SRFRN":       # rows are E[label] || Fe[user_label] (SRFR_model.py:244-257)
            fid = torch.as_tensor(fake_ids, device=eng.device).long()
            lab = torch.empty(fid.shape[0], dtype=torch.int64, device=eng.device)
            ops.srfu_labels(fid.contiguous(), 3, lab)
            logits = logits.contiguous()
            ops.add_user_term(logits, feats[:, self.spec.D:], eng.P.view("embedding_layer.fake_embed.weight"), lab)
        return logits.squeeze()


def _split_gemm_logits(feats: torch.Tensor, table: torch.Tensor, label: torch.Tensor) -> torch.Tensor:
    """feats (U, D) fp32 x table[label] (I, D) fp32 on the tensor cores at near-fp32 accuracy:
    A = [f_hi | f_lo | f_hi], B = [E_hi | E_hi | E_lo] (bf16 hi/lo splits, K = 3D)."""
    U, D = feats.shape
    I = label.numel()
    Ip = (I + 15) // 16 * 16
    Dp = (D + 7) // 8 * 8                    # K-segments padded to 16 bytes (zero columns add nothing)
    dev = feats.device
    A = torch.zeros(U, 3 * Dp, dtype=bf16, device=dev)
    Bm = torch.zeros(Ip, 3 * Dp, dtype=bf16, device=dev)
    f = feats.contiguous()
    ops.f32_to_bf16_split(f, A[:, :D], A[:, Dp:Dp + D])
    ops.f32_to_bf16_split(f, A[:, 2 * Dp:2 * Dp + D], None)
    ops.f32_to_bf16_split(table, Bm[:I, :D], Bm[:I, 2 * Dp:2 * Dp + D], row_index=label)
    ops.f32_to_bf16_split(table, Bm[:I, Dp:Dp + D], None, row_index=label)
    out = torch.empty(U, Ip, dtype=torch.float32, device=dev)
    ops.gemm_tn(A, Bm, out_f32=out)
    return out[:, :I]


class SRFR(_HotPathModule):
    """SRFR_model.py:53-152."""

    def __init__(self, item_number, max_len=20, item_embedding_size=50, fake_embedding_size=10, dropout_rate=0.5,
                 num_blocks=2, num_heads=1, device="cpu"):
        super().__init__(ModelSpec("SRFR", item_number, max_len, item_embedding_size, fake_embedding_size, 0,
                                   num_blocks, num_heads, dropout_rate), device)
        self.total_hidden_size = item_embedding_size + fake_embedding_size


class SRFRN(_HotPathModule):
    """SRFR_model.py:154-259."""

    def __init__(self, item_number, max_len=20, item_embedding_size=50, fake_embedding_size=10, dropout_rate=0.5,
                 num_blocks=2, num_heads=1, device="cpu"):
        super().__init__(ModelSpec("SRFRN", item_number, max_len, item_embedding_size, fake_embedding_size, 0,
                                   num_blocks, num_heads, dropout_rate), device)
        self.total_hidden_size = item_embedding_size + fake_embedding_size


class _SRFU(_HotPathModule):
    KIND = ""

    def __init__(self, item_number, max_len=20, item_embedding_size=50, number_of_labels=2, dropout_rate=0.5,
                 num_blocks=2, num_heads=1, device="cpu"):
        super().__init__(ModelSpec(self.KIND, item_number, max_len, item_embedding_size, 0, number_of_labels,
                                   num_blocks, num_heads, dropout_rate), device)
        self.maxlen = max_len

    @torch.no_grad()
    def get_Labels(self, fake_ids):
        """SRFR_model.py:546-570."""
        fid = torch.as_tensor(fake_ids).long().cuda().contiguous()
        out = torch.empty(fid.shape[0], dtype=torch.int64, device=fid.device)
        ops.srfu_labels(fid, {"SRFU_B": 0, "SRFU_F": 1, "SRFU_R": 2}[self.KIND], out)
        return out


class SRFU_B(_SRFU):
    KIND = "SRFU_B"


class SRFU_F(_SRFU):
    KIND = "SRFU_F"


class SRFU_R(_SRFU):
    KIND = "SRFU_R"


class SASRec(_HotPathModule):
    """SRFR_model.py:572-681 (tensor inputs; fake ids are accepted and ignored)."""

    def __init__(self, item_number, maxlen=20, hidden_units=50, dropout_rate=0.5, num_blocks=2, num_heads=1,
                 device="cpu"):
        super().__init__(ModelSpec("SASRec", item_number, maxlen, hidden_units, 0, 0, num_blocks, num_heads,
                                   dropout_rate), device)
        self.item_num = item_number

    def log2feats(self, log_seqs):
        return self.forward(None, log_seqs, None)[0]
