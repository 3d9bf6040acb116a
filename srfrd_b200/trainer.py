"""Training loops for the hot path.

``simulate``      -- drop-in for the reference's ``simulate(model, optimizer, criterion, sampler, config,
                     wandb, model_index=0)`` (trainer.py:15-68): same batches, same masked BCE, any torch
                     criterion / optimizer; the model's forward/backward run on the sm_100a kernels.
``FusedTrainer``  -- the B200-first step: ids and discriminator weights are copied to static device buffers,
                     then ONE captured CUDA graph runs forward -> fused weighted BCE (forward+backward, no
                     ``nonzero`` sync, trainer.py:36) -> backward -> [gradient all-reduce] -> flat Adam ->
                     bf16 shadow refresh; with l2_emb > 0 the per-tensor norms of the regulariser run on a side
                     stream next to the forward.  The loss stays on the device until the caller asks for it.
"""
from __future__ import annotations

import time
from typing import Dict, Optional

import numpy as np
import torch

from . import ops, parallel
from .engine import HotPath
from .losses import check_ce_width, check_gbce, gbce_beta

__all__ = ["simulate", "FusedTrainer", "DeviceSampler", "discriminator_weights"]

POLICIES = {"none": 0, "mask": 1, "soft": 2}


class DeviceSampler:
    """The training interactions resident on the device in CSR form plus the batch-building kernel
    (srfrd_sample_batch): the B200-side replacement of WarpSampler_fr (utils.py:67-90).  ``next_batch`` keeps the
    reference's 7-tuple order (u, seq, rsq, pos, prs, neg, nrs) as int64 device tensors; ``FusedTrainer.step_sampled``
    draws inside the captured CUDA graph so no batch ever crosses PCIe."""

    def __init__(self, data, maxlen: int, device, seed: int = 0):
        """data: srfrd_b200.synth.Interactions (or any object with offsets / items / labels / p_fake / itemnum)."""
        dev = torch.device(device)
        self.L, self.itemnum, self.seed = maxlen, int(data.itemnum), int(seed)
        self.offsets = torch.as_tensor(np.asarray(data.offsets, np.int64)).to(dev)
        self.items = torch.as_tensor(np.asarray(data.items, np.int32)).to(dev)
        self.labels = torch.as_tensor(np.asarray(data.labels, np.int8)).to(dev)
        pf = getattr(data, "p_fake", None)
        self.p_fake = None if pf is None else torch.as_tensor(np.asarray(pf, np.float32)).to(dev)
        lens = np.diff(np.asarray(data.offsets, np.int64))
        self.eligible = torch.as_tensor(np.nonzero(lens > 1)[0].astype(np.int32)).to(dev)      # utils.py:25
        if self.eligible.numel() == 0:
            raise ValueError("no user has more than one training interaction")
        self.device = dev
        self.draws = 0

    def alloc(self, B: int):
        z = lambda: torch.zeros(B, self.L, dtype=torch.int64, device=self.device)
        return dict(users=torch.zeros(B, dtype=torch.int64, device=self.device), seq=z(), rsq=z(), pos=z(), prs=z(),
                    neg=z(), nrs=z())

    def sample_into(self, out, w_pos=None, policy: str = "none", step=None):
        """Fill pre-allocated tensors; ``step`` = device fp32 counter mixed into the seed (graph replays)."""
        B = out["seq"].shape[0]
        ops.sample_batch(self.offsets, self.items, self.labels, self.p_fake, self.eligible, self.itemnum, B, self.L,
                         POLICIES[policy], self.seed + (0 if step is not None else self.draws), step, out, w_pos)
        self.draws += 1

    def next_batch(self, batch_size: int):
        out = self.alloc(batch_size)
        self.sample_into(out)
        return out["users"], out["seq"], out["rsq"], out["pos"], out["prs"], out["neg"], out["nrs"]



def discriminator_weights(pos: torch.Tensor, p_fake: Optional[torch.Tensor], policy: str = "none") -> torch.Tensor:
    """w = 1[pos != 0] * g(p_fake): 'none' g = 1 (the reference's loss, trainer.py:36-38), 'mask'
    g = 1[p_fake < 0.5] (== the hard label prs == 2 the BERT discriminator emits,
    data/userDiscriminator.py:68,117-122), 'soft' g = 1 - p_fake.  Tiny elementwise plumbing on the
    batch's (B, L) weights; the weighted loss itself is the fused CUDA kernel."""
    valid = (pos != 0).to(torch.float32)
    if policy == "none" or p_fake is None:
        return valid
    if policy == "mask":
        return valid * (p_fake < 0.5).to(torch.float32)
    if policy == "soft":
        return valid * (1.0 - p_fake.to(torch.float32))
    raise ValueError(f"unknown discriminator weighting policy {policy!r}")


class FusedTrainer:
    """One data-parallel replica of the fused training step.

    model        : a srfrd_b200.SRFR_model module already on the CUDA device
    lr, betas, eps: Adam hyper-parameters (reference: lr 1e-3, betas (0.9, 0.98), trainer.py:390)
    process_group: torch.distributed group for batch-sharded data parallelism (None = single GPU).
                   Gradients are SUM-all-reduced and the loss is normalised by the all-reduced weight
                   sums, so N ranks on B/N sequences each reproduce one rank on B sequences.
    use_graph    : capture the step in a CUDA graph after the first (eager) step.
    packed       : run the encoder on the packed token layout (csrc/pack.cu) -- pad slots, ~88 % of a Beauty-shaped batch,
                   are not computed; results equal the dense path (None = on when the shape supports it).
    l2_emb       : the reference's regulariser (trainer.py:31-39): the loss gains l2_emb * sum_p ||p||_2 over every tensor
                   of model.parameters() (plain norm, not squared) and each gradient l2_emb * p / ||p|| (0 for a zero
                   tensor), both from the parameters before the step's update.  The norm gradient reaches every row of the
                   embedding tables, the pad row included, so rows no batch touches drift under Adam as in the reference.
                   Fixed for the trainer's lifetime (a captured graph holds it).
    loss         : "bce" -- the reference's objective (one sampled negative per position, trainer.py:31-38);
                   "ce" -- full-catalogue softmax cross-entropy over predict's logits (every item 1..N a candidate, the
                   positive the target; losses.catalogue_cross_entropy) with the same discriminator weights and normaliser,
                   computed by the tcgen05 kernels of csrc/catalogue_ce.cu without materialising the logits.  The sampled
                   negatives are unused and w_neg is refused; SRFRN is refused (its logits need a fake label per candidate,
                   SRFR_model.py:225-233, which unobserved items do not have).
                   "gbce" -- gSASRec's gBCE (losses.sampled_gbce) over num_negatives (k, default 256) item ids drawn
                   uniformly on the device each step from (the engine's seed, the device step counter) and shared by
                   every position of the batch, with calibration gbce_t (t, default 0.75; t = 0 is BCE with k negatives).
                   A negative that occurs in a position's sequence (its seq or pos ids) is left out of that position's
                   loss.  Same discriminator weights and normaliser as the BCE; the kernels are csrc/gbce.cu.  Every
                   data-parallel rank draws the same negatives.  w_neg and SRFRN are refused as for "ce".
    lazy_item_adam: update only the item-table rows the step looks up (SparseAdam's rule; default False = dense Adam
                   over the whole flat buffer).  A step looks up the non-zero ids of the batch's seq, pos and neg for
                   "bce", of seq and pos plus the drawn negatives for "gbce", and data parallel the union over ranks.
                   Those rows get exactly the dense update (torch.optim.Adam's m_hat / (sqrt(v_hat) + eps), bias
                   corrections of the trainer's global step) even when their gradient is zero; every other row keeps
                   its parameters and moments bit for bit.  Every other parameter tensor stays dense.  When a step looks
                   up every row, the result is bit-identical to the dense step.  Refused with l2_emb != 0 (the
                   regulariser's gradient reaches every row) and with loss="ce" (every row is a candidate).
    """

    def __init__(self, model, lr: float = 1e-3, betas=(0.9, 0.98), eps: float = 1e-8, process_group=None,
                 use_graph: bool = True, l2_emb: float = 0.0, packed: Optional[bool] = None, loss: str = "bce",
                 num_negatives: Optional[int] = None, gbce_t: Optional[float] = None, lazy_item_adam: bool = False):
        if loss not in ("bce", "ce", "gbce"):
            raise ValueError(f"unknown loss {loss!r} (expected 'bce', 'ce' or 'gbce')")
        if loss != "gbce" and (num_negatives is not None or gbce_t is not None):
            raise ValueError(f"num_negatives / gbce_t configure loss='gbce', not loss={loss!r}")
        if lazy_item_adam and l2_emb != 0.0:
            raise ValueError("lazy_item_adam needs l2_emb == 0: the regulariser's gradient reaches every item row on every "
                             "step, so no row is left untouched")
        if lazy_item_adam and loss == "ce":
            raise ValueError("lazy_item_adam does not apply to loss='ce': every item is a candidate of every step, so every "
                             "row is updated and lazy equals dense")
        if loss in ("ce", "gbce") and model.spec.kind == "SRFRN":
            raise ValueError(f"loss={loss!r} does not support SRFRN: its logits need each candidate's fake label "
                             "(SRFR_model.py:225-233), which unobserved items do not have")
        if loss == "ce":
            check_ce_width(model.spec.D)
        if loss == "gbce":
            self.num_negatives = 256 if num_negatives is None else num_negatives
            self.gbce_t = 0.75 if gbce_t is None else gbce_t
            n_items = dict(model.named_parameters())[model.spec.item_key].shape[0] - 1
            check_gbce(self.num_negatives, self.gbce_t, n_items, model.spec.D)
        self.loss_kind = loss
        self.model = model
        self.lazy = bool(lazy_item_adam)
        item_rows = dict(model.named_parameters())[model.spec.item_key].shape[0]
        self._dp = None
        # the fused data-parallel kernel's lazy row walk moves whole float4 rows (D % 4 == 0); other widths take the NCCL
        # all-reduce + the single-GPU gated Adam, which handles any D
        if process_group is not None and torch.distributed.get_world_size(process_group) > 1 and \
                not (self.lazy and model.spec.D % 4):
            self._dp = self._setup_fused_dp(model, process_group, item_rows if self.lazy else 0)
        self.eng: HotPath = model._sync_flat()
        self.P = self.eng.P
        self.spec = self.eng.spec
        self.lr, self.betas, self.eps = lr, betas, eps
        self.pg = process_group
        self.use_graph = use_graph
        # packed token layout (no work on pad slots) whenever the shape supports it; SRFRD_PACKED=0 / packed=False = dense
        self.packed = self.eng.packed_default if packed is None else bool(packed)
        dev = self.eng.device
        self.m = torch.zeros_like(self.P.data)
        self.v = torch.zeros_like(self.P.data)
        self.scal = torch.zeros(8, dtype=torch.float32, device=dev)   # [0:2] norm (weight sums), [4] loss
        # the loss accumulators live in the tail of the gradient bucket (one all-reduce moves gradients and loss)
        self.comm = torch.cuda.Stream(device=dev)
        self._static: Optional[Dict[str, torch.Tensor]] = None
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._graph_key = None
        self._eager_key = None
        self._has_w = (False, False)
        self.l2_emb = float(l2_emb)
        self._l2 = self._setup_l2(model) if self.l2_emb != 0.0 else None
        self._ce_ws: Optional[Dict[str, torch.Tensor]] = None
        self._gbce_ws: Optional[Dict[str, torch.Tensor]] = None
        if loss == "ce":
            self.eng.enable_ce_table()
        # lazy item-table Adam: one uint32 epoch stamp per item row (srfrd_touch_rows); in symmetric memory under the fused
        # data-parallel optimizer, which ORs every rank's stamps
        self.stamp: Optional[torch.Tensor] = None
        if self.lazy:
            self.stamp = self._dp["stamp"] if self._dp is not None else torch.zeros(item_rows, dtype=torch.int32, device=dev)
            self._table = (self.P.offsets[self.spec.item_key][0], item_rows, self.spec.D)
        self.P.grad_bucket.zero_()
        self.eng.refresh_shadows()
        self.steps = 0

    def _ce_buffers(self, rows: int) -> Dict[str, torch.Tensor]:
        """bf16 copy of the final hidden rows and their log-sum-exp (loss="ce"); a larger batch re-allocates, which the
        graph key's workspace generation covers."""
        if self._ce_ws is None or self._ce_ws["lse"].numel() < rows:
            dev = self.eng.device
            self._ce_ws = dict(h=torch.zeros(rows, self.spec.Dp, dtype=torch.bfloat16, device=dev),
                               lse=torch.zeros(rows, dtype=torch.float32, device=dev))
            self.eng.ws_generation += 1
        return self._ce_ws

    def _gbce_buffers(self, rows: int, B: int) -> Dict[str, torch.Tensor]:
        """loss="gbce": the bf16 final hidden rows, the drawn ids, their bf16 rows, the exclusion words of the batch's
        sequences and the dN pass's partials; re-allocated (bumping the workspace generation) when a batch needs more."""
        ws = self._gbce_ws
        if ws is None or ws["h"].shape[0] < rows or ws["excl"].shape[0] < B:
            dev, Dp, k = self.eng.device, self.spec.Dp, self.num_negatives
            rows = max(rows, 0 if ws is None else ws["h"].shape[0])
            B = max(B, 0 if ws is None else ws["excl"].shape[0])
            Kp, n_split, _, _ = ops.gbce_plan(k, Dp, rows)
            self._gbce_ws = ws = dict(
                h=torch.zeros(rows, Dp, dtype=torch.bfloat16, device=dev),
                ids=torch.zeros(k, dtype=torch.int64, device=dev),
                nb=torch.zeros(Kp, Dp, dtype=torch.bfloat16, device=dev),
                excl=torch.zeros(B, (k + 31) // 32, dtype=torch.int32, device=dev),
                part=torch.zeros(n_split * Kp * Dp, dtype=torch.float32, device=dev))
            self.eng.ws_generation += 1
        return ws

    def _refuse_w_neg(self, w_neg):
        if w_neg is not None and self.loss_kind in ("ce", "gbce"):
            raise ValueError(f"w_neg weights the sampled negative of the BCE; loss={self.loss_kind!r} does not take it")

    def _setup_l2(self, model) -> ops.ParamL2:
        """The regulariser's segment table: every tensor of model.parameters() is one segment of the flat buffer."""
        segs = self.P.segments()
        base = self.P.data.data_ptr()
        mine = sorted((p.data_ptr(), p.numel()) for p in model.parameters())
        assert mine == [(base + 4 * off, n) for off, n in segs], \
            "srfrd_b200: l2_emb: the flat parameter segments do not cover exactly model.parameters()"
        return ops.ParamL2(segs, self.l2_emb, self.eng.device)

    # ------------------------------------------------------------------
    @staticmethod
    def _setup_fused_dp(model, pg, stamp_rows: int = 0):
        """Place the flat parameter buffer and the gradient bucket in symmetric memory (mapped into every rank of the
        node) so that ONE kernel per rank can do reduce-scatter -> Adam -> all-gather through NVLink peer pointers
        (csrc/dp_adam.cu).  Returns None -- the NCCL all-reduce path stays -- when symmetric memory is unavailable or
        SRFRD_FUSED_DP=0.  stamp_rows > 0 (lazy_item_adam): the item rows' epoch stamps are placed there too."""
        import os
        if os.environ.get("SRFRD_FUSED_DP", "1") == "0":
            return None
        try:
            import torch.distributed._symmetric_memory as symm
            dev = next(model.parameters()).device
            gname = pg.group_name
            try:
                symm.enable_symm_mem_for_group(gname)
            except Exception:  # noqa: BLE001  (newer torch: not needed / deprecated)
                pass
            eng = model.rehome(lambda n: symm.empty(n, dtype=torch.float32, device=dev))
            P = eng.P
            sig = symm.empty(64, dtype=torch.int32, device=dev).zero_()
            torch.cuda.synchronize()
            hg, hp, hs = (symm.rendezvous(t, gname) for t in (P.grad_bucket, P.data_ext, sig))
            dp = dict(g=int(hg.buffer_ptrs_dev), p=int(hp.buffer_ptrs_dev), s=int(hs.buffer_ptrs_dev), rank=int(hg.rank),
                      world=int(hg.world_size), keep=(hg, hp, hs, sig),
                      local=torch.zeros(4, dtype=torch.int32, device=dev))
            if stamp_rows > 0:
                stamp = symm.empty(stamp_rows, dtype=torch.int32, device=dev).zero_()
                torch.cuda.synchronize()
                hst = symm.rendezvous(stamp, gname)
                dp.update(stamp=stamp, st=int(hst.buffer_ptrs_dev), keep=dp["keep"] + (hst, stamp))
            torch.cuda.synchronize()
            torch.distributed.barrier(group=pg)
            return dp
        except Exception as ex:  # noqa: BLE001
            import warnings
            warnings.warn(f"srfrd_b200: fused data-parallel optimizer unavailable ({type(ex).__name__}: {ex}); "
                          "falling back to the NCCL all-reduce + replicated Adam")
            return None

    @property
    def loss_dev(self) -> torch.Tensor:
        """Device scalar holding the last step's loss."""
        return self.P.data_tail[0] if self._dp is not None else self.scal[4]

    _KEYS = ("seq", "rsq", "pos", "prs", "neg", "nrs")

    @staticmethod
    def _carve(flat: torch.Tensor, B: int, L: int):
        """views of one flat int64 buffer: six (B, L) int64 id arrays followed by two (B, L) fp32 weight arrays"""
        n = B * L
        out = {k: flat[i * n:(i + 1) * n].view(B, L) for i, k in enumerate(FusedTrainer._KEYS)}
        w = flat[6 * n:7 * n].view(torch.float32)            # n int64 words = 2 n fp32 words
        out["w_pos"], out["w_neg"] = w[:n].view(B, L), w[n:].view(B, L)
        return out

    def _alloc_static(self, B: int, L: int):
        dev = self.eng.device
        self._static_flat = torch.zeros(7 * B * L, dtype=torch.int64, device=dev)   # ONE buffer: one D2D copy fills it
        self._static = self._carve(self._static_flat, B, L)
        self._stage_flat = None
        self._graph = None

    def _step_body(self, has_wp: bool, has_wn: bool):
        """The kernel sequence of one step, on static buffers (captured once, replayed forever)."""
        st, eng, P, s = self._static, self.eng, self.P, self.spec
        B, L = st["seq"].shape
        pos, neg = st["pos"].view(-1), st["neg"].view(-1)
        w_pos = st["w_pos"].view(-1) if has_wp else None
        w_neg = st["w_neg"].view(-1) if has_wn else None
        norm, acc, loss = self.scal[0:2], P.grad_tail[0:2], self.scal[4:5]
        smp = getattr(self, "_sampler", None)
        if smp is not None:
            smp.sample_into(st, st["w_pos"] if has_wp else None, self._sampler_policy, step=eng.step_state[3:4])
        # The weight sums (loss normaliser: the reference's mean over ALL pos != 0 of the batch, trainer.py:36-38) and, data
        # parallel, their tiny all-reduce run on a side stream: the forward pass does not wait for them, only the loss
        # kernel does.
        self.comm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.comm):
            ops.weight_sums(pos, w_pos, w_neg, norm)
            if self.pg is not None:
                parallel.allreduce_sum_(norm, self.pg)
            if self.lazy:
                # the rows this step's forward and loss gather (gBCE leaves neg unused; its drawn ids are stamped below)
                ops.touch_rows(self.stamp, eng.step_state, self._table[1] - 1, st["seq"].view(-1), pos,
                               neg if self.loss_kind == "bce" else None)
            if self._l2 is not None:
                # the norms of the parameters the previous step left behind, next to the forward pass; the join below
                # orders them before Adam (in the fused data-parallel kernel, peers overwrite this buffer once this rank
                # reaches its entry barrier, which only stream order can delay)
                self._l2.launch(P.data)
        packed = self.packed and eng.packed_ok(B, L)
        # packed token layout: pad slots (88 % of a C2 batch) get no rows; slots whose POSITIVE id is set keep one even if
        # their input is a pad, because the loss reads their hidden state
        hidden = eng.forward(st["seq"], st["rsq"], training=True, packed=packed, keep=st["pos"] if packed else None)
        ws = eng._ws
        ft = eng.fake_table()
        torch.cuda.current_stream().wait_stream(self.comm)
        prs_ = st["prs"].view(-1) if ft is not None else None
        nrs_ = st["nrs"].view(-1) if ft is not None else None
        rows, plan = eng.saved.T, eng.saved.plan          # the forward's activation rows (B * L, or packed) and plan
        if self.loss_kind == "ce":
            ce = self._ce_buffers(rows)
            hb, lse, table = ce["h"][:rows], ce["lse"][:rows], eng.sh["ce_table"]
            ops.f32_to_bf16_split(ws["hfin"][:rows], hb)
            ops.catalogue_ce_fwd(hb, table, pos, w_pos, lse, acc, plan)
            ops.catalogue_ce_bwd(hb, table, pos, w_pos, norm, lse, ws["dh"][:rows], P.view(s.item_key, grad=True), s.D, plan)
        elif self.loss_kind == "gbce":
            gb = self._gbce_buffers(rows, B)
            hb, E = gb["h"][:rows], P.view(s.item_key)
            ops.f32_to_bf16_split(ws["hfin"][:rows], hb)
            # the same (seed, step) on every data-parallel rank: every rank draws the same negatives
            ops.gbce_draw(E, gb["ids"], gb["nb"], gb["excl"][:B], st["seq"], st["pos"], seed=eng.drop_seed,
                          step=eng.step_state[3:4])
            if self.lazy:
                self.comm.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(self.comm):
                    ops.touch_rows(self.stamp, eng.step_state, E.shape[0] - 1, ids=gb["ids"])
            ops.gbce_loss(hb, gb["nb"], gb["ids"], E, pos, w_pos, norm, gb["excl"], L,
                          gbce_beta(self.num_negatives, E.shape[0] - 1, self.gbce_t), acc, ws["dh"][:rows],
                          P.view(s.item_key, grad=True), gb["part"], plan)
        elif plan is not None:
            ops.score_loss_fused_packed(ws["hfin"][:rows], P.view(s.item_key), ft, pos, neg, prs_, nrs_, w_pos, w_neg, norm,
                                        acc, ws["dh"][:rows], P.view(s.item_key, grad=True), eng.fake_table_grad(), plan)
        else:
            ops.score_loss_fused(ws["hfin"][:rows], P.view(s.item_key), ft, pos, neg, prs_, nrs_, w_pos, w_neg, norm, acc,
                                 ws["dh"][:rows], P.view(s.item_key, grad=True), eng.fake_table_grad())
        eng.backward(ws["dh"][:rows])
        if self.lazy:
            torch.cuda.current_stream().wait_stream(self.comm)           # every stamp of the step is written
        if self._dp is not None and self.lazy:
            d = self._dp
            ops.dp_adam_step_rows(d["g"], d["p"], d["s"], d["rank"], d["world"], P.numel, self.m, self.v, self.lr,
                                  self.betas[0], self.betas[1], self.eps, eng.step_state, norm, d["local"], *self._table,
                                  d["st"])
        elif self._dp is not None:
            # reduce-scatter -> Adam on this rank's slice -> all-gather of the new parameters + loss, one kernel over NVLink
            # peer memory (csrc/dp_adam.cu) instead of an NCCL all-reduce followed by the same Adam on every rank
            d = self._dp
            ops.dp_adam_step(d["g"], d["p"], d["s"], d["rank"], d["world"], P.numel, self.m, self.v, self.lr, self.betas[0],
                             self.betas[1], self.eps, eng.step_state, norm, d["local"], l2=self._l2)
        else:
            if self.pg is not None:
                parallel.allreduce_sum_(P.grad_bucket, self.pg)           # ONE NCCL sum over NVLink: gradients + loss sums
                if self.lazy:
                    parallel.union_row_stamps_(self.stamp, self.pg)       # the rows of the global batch on every rank
            if self.lazy:
                ops.adam_step_fused_rows(P.data, P.grad, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps,
                                         eng.step_state, *self._table, self.stamp, zero_grad=True, acc2=acc, norm2=norm,
                                         loss=loss)
            else:
                # Adam tick + dense Adam + loss read-out (consumes acc: zero again for the next step) in one launch
                ops.adam_step_fused(P.data, P.grad, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps,
                                    eng.step_state, zero_grad=True, acc2=acc, norm2=norm, loss=loss, l2=self._l2)
        eng.refresh_shadows()

    # ------------------------------------------------------------------
    def load_batch(self, batch: Dict[str, torch.Tensor], w_pos=None, w_neg=None, non_blocking: bool = True):
        """Copy one batch (host pinned or device tensors, int64 (B, L)) into the static buffers."""
        self._refuse_w_neg(w_neg)
        B, L = batch["seq"].shape
        if self._static is None or self._static["seq"].shape != (B, L):
            self._alloc_static(B, L)
        st = self._static
        for k in ("seq", "rsq", "pos", "prs", "neg", "nrs"):
            src = batch.get(k)
            if src is None:
                st[k].zero_()
            else:
                st[k].copy_(torch.as_tensor(src), non_blocking=non_blocking)
        if w_pos is not None:
            st["w_pos"].copy_(torch.as_tensor(w_pos), non_blocking=non_blocking)
        if w_neg is not None:
            st["w_neg"].copy_(torch.as_tensor(w_neg), non_blocking=non_blocking)
        self._has_w = (w_pos is not None, w_neg is not None)

    def pack_batch(self, batch: Dict[str, torch.Tensor], w_pos=None, w_neg=None) -> torch.Tensor:
        """One flat device buffer holding a whole batch in the layout of the step's static inputs (six int64 (B, L) id
        arrays + two fp32 (B, L) weight arrays): ``step_packed`` then needs ONE device-to-device copy per step."""
        self._refuse_w_neg(w_neg)
        B, L = batch["seq"].shape
        flat = torch.zeros(7 * B * L, dtype=torch.int64, device=self.eng.device)
        v = self._carve(flat, B, L)
        for k in self._KEYS:
            if batch.get(k) is not None:
                v[k].copy_(torch.as_tensor(batch[k]))
        if w_pos is not None:
            v["w_pos"].copy_(torch.as_tensor(w_pos))
        if w_neg is not None:
            v["w_neg"].copy_(torch.as_tensor(w_neg))
        flat._srfrd_shape, flat._srfrd_w = (B, L), (w_pos is not None, w_neg is not None)
        return flat

    def step_packed(self, flat: torch.Tensor) -> torch.Tensor:
        """One step on a batch prepared by ``pack_batch`` (device resident)."""
        B, L = flat._srfrd_shape
        if self._static is None or self._static["seq"].shape != (B, L):
            self._alloc_static(B, L)
        self._static_flat.copy_(flat, non_blocking=True)
        self._has_w = flat._srfrd_w
        return self.run_step()

    # ---- host batches pipelined across steps: H2D of batch n+1 (copy stream) overlaps the compute of batch n ----------
    def prefetch(self, batch: Dict[str, torch.Tensor], w_pos=None, w_neg=None):
        """Start copying a (pinned) host batch into a device staging buffer on a separate copy stream.  The next
        ``step_prefetched()`` waits for it, moves it into the step's static buffers with ONE device-to-device copy and
        runs the step, so the PCIe transfer of the next batch hides behind the current step."""
        self._refuse_w_neg(w_neg)
        B, L = batch["seq"].shape
        if self._static is None or self._static["seq"].shape != (B, L):
            self._alloc_static(B, L)
        if self._stage_flat is None:
            self._stage_flat = torch.zeros_like(self._static_flat)
            self._stage = self._carve(self._stage_flat, B, L)
            self._copy_stream = torch.cuda.Stream(device=self.eng.device)
            self._stage_free = torch.cuda.Event()
            self._stage_full = torch.cuda.Event()
            self._stage_free.record()                             # (after the zero fill above, on the current stream)
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._stage_free)        # the previous staged batch has been consumed
            for k in self._KEYS:
                src = batch.get(k)
                if src is None:
                    self._stage[k].zero_()
                else:
                    self._stage[k].copy_(torch.as_tensor(src), non_blocking=True)
            if w_pos is not None:
                self._stage["w_pos"].copy_(torch.as_tensor(w_pos), non_blocking=True)
            if w_neg is not None:
                self._stage["w_neg"].copy_(torch.as_tensor(w_neg), non_blocking=True)
            self._stage_full.record()
        self._stage_w = (w_pos is not None, w_neg is not None)

    def step_prefetched(self) -> torch.Tensor:
        """Run one step on the batch handed to ``prefetch``; returns the device loss scalar (no sync)."""
        main = torch.cuda.current_stream()
        main.wait_event(self._stage_full)
        self._static_flat.copy_(self._stage_flat)                 # one D2D copy (10 MB at C2: a few microseconds)
        self._stage_free.record(main)
        self._has_w = self._stage_w
        return self.run_step()

    def run_step(self) -> torch.Tensor:
        """Run one step on the loaded batch; returns the device scalar holding the loss (no sync)."""
        # the graph holds raw pointers into the engine's workspace: a re-allocation (a larger evaluation / encode_last
        # forward between training steps) bumps ws_generation and forces a re-capture instead of a replay into freed memory
        key = (tuple(self._static["seq"].shape), self._has_w, id(getattr(self, "_sampler", None)), self.eng.ws_generation)
        if self.use_graph and self._graph is not None and self._graph_key == key:
            self._graph.replay()
        elif self.use_graph and self.steps >= 1 and self._eager_key == key[:3] + (self.eng.ws_generation,):
            # capture after one eager step has sized the workspaces, set kernel attributes and (data parallel) warmed
            # up the NCCL communicator; the gradient all-reduce is captured into the same graph
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                self._step_body(*self._has_w)
            self._graph, self._graph_key = g, key
            g.replay()
        else:
            self._step_body(*self._has_w)
            # an eager step may itself have re-allocated the workspace: remember the generation it LEFT behind
            self._eager_key = key[:3] + (self.eng.ws_generation,)
        self.steps += 1
        return self.loss_dev

    def step(self, batch, w_pos=None, w_neg=None) -> torch.Tensor:
        self.load_batch(batch, w_pos, w_neg)
        return self.run_step()

    def step_sampled(self, sampler: "DeviceSampler", batch_size: int, policy: str = "none") -> torch.Tensor:
        """One step on a batch drawn ON THE DEVICE by ``sampler`` (no host batch, no H2D copies): the sampling kernel
        is the first node of the captured graph and re-seeds itself from the device-resident step counter."""
        if self._static is None or self._static["seq"].shape != (batch_size, sampler.L):
            self._alloc_static(batch_size, sampler.L)
        self._sampler, self._sampler_policy = sampler, policy
        self._has_w = (policy != "none", False)
        out = self.run_step()
        self._sampler = None
        return out

    def state_dict(self):
        return {k: v.detach().clone() for k, v in self.model.state_dict().items()}


# ---------------------------------------------------------------------------------------------
def simulate(model, optimizer, criterion, sampler, config, wandb=None, model_index=0, num_batch=None, device=None,
             dataset=None, evaluation=None, log_every: int = 1):
    """The reference loop (trainer.py:15-68) with its module globals (num_batch, device, dataset) made
    explicit keyword arguments.  ``wandb`` is duck-typed (anything with .log(dict)) or None.
    ``log_every`` strides the per-step ``loss.item()`` sync the reference performs every step."""
    T, t0 = 0.0, time.time()
    metricsbyepoch = dict()
    device = device if device is not None else next(model.parameters()).device
    num_batch = num_batch if num_batch is not None else getattr(config, "num_batch")
    for epoch in range(config.num_epochs):
        if config.inference_only:
            break
        epoch_loss = 0.0
        model.train()
        for step in range(num_batch):
            u, seq, rsq, pos, prs, neg, nrs = sampler.next_batch()
            seq, rsq, pos, prs, neg, nrs = (torch.as_tensor(np.array(a)).long().to(device)
                                            for a in (seq, rsq, pos, prs, neg, nrs))
            hidden_state, pos_logits, neg_logits = model(user_ids=None, input_ids=seq, fake_ids=rsq, positive_ids=pos,
                                                         positive_fake_ids=prs, negative_ids=neg, negative_fake_ids=nrs)
            pos_labels = torch.ones(pos_logits.shape, device=device)
            neg_labels = torch.zeros(neg_logits.shape, device=device)
            optimizer.zero_grad()
            indices = torch.where(pos != 0)
            loss = criterion(pos_logits[indices], pos_labels[indices])
            loss += criterion(neg_logits[indices], neg_labels[indices])
            if getattr(config, "l2_emb", 0.0):
                for param in model.parameters():
                    loss += config.l2_emb * torch.norm(param)
            loss.backward()
            optimizer.step()
            if step % log_every == 0:
                li = loss.item()
                if wandb is not None:
                    wandb.log({"Training Loss by iteration": li})
                epoch_loss += li
        if wandb is not None:
            wandb.log({"Training Loss by Epoch": epoch_loss, "Epochs": epoch + 1})
        if (epoch + 1) % 10 == 0 and evaluation is not None and dataset is not None:
            model.eval()
            T += time.time() - t0
            t_test = evaluation(model, dataset, config.maxlen, device)
            if wandb is not None:
                wandb.log({"NDCG@10": t_test[0], "HT@10": t_test[1]})
            metricsbyepoch[epoch + 1] = {"NDCG@10": t_test[0], "HT@10": t_test[1]}
            t0 = time.time()
            model.train()
    return metricsbyepoch
