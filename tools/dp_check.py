"""Multi-GPU check (run under torchrun): G-rank data-parallel FusedTrainer == 1-rank on the concatenated batch,
and row-sharded catalogue top-10 (NCCL all-gather + merge) == unsharded top-10.
`--l2 X` trains both with l2_emb = X (the regulariser's gradient is added once, after the reduction over ranks).
`--topk-k K` checks the sharded top-K (1 <= K <= 64) instead of the top-10.
`--loss ce` trains both with the full-catalogue cross-entropy (FusedTrainer(loss="ce")) instead of the BCE.
`--loss gbce [--negatives K] [--t T]` trains both with gSASRec's gBCE (FusedTrainer(loss="gbce")); every rank draws the
same K negatives per step, so the check is the same.  Its loss is about K times the BCE's, so its bound is relative.
`--lazy` trains both with FusedTrainer(lazy_item_adam=True) (combinable with `--loss gbce`): the G ranks update the union
of their batches' item rows, so they still reproduce one rank on the concatenated batch."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from srfrd_b200 import SRFR_model as M, evaluation as EV, parallel as P, synth
from srfrd_b200.trainer import FusedTrainer, discriminator_weights

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)


def make_model():
    torch.manual_seed(11)
    m = M.SRFR(3000, 50, 64, 16, 0.0, 2, 1, dev)
    for _, p in m.named_parameters():
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to(dev)


data = synth.make_interactions(77, 4000, 3000, 5, 4.0, 50)
smp = synth.BatchSampler(data, 50, 5)
batches = [smp.next_batch(64 * world) for _ in range(6)]
m_dp, m_one = make_model(), make_model()
P.broadcast_parameters(m_dp.flat_parameters().data, 0)
use_graph = os.environ.get("DP_CHECK_GRAPH", "0") == "1"
l2_emb = float(sys.argv[sys.argv.index("--l2") + 1]) if "--l2" in sys.argv else 0.0
topk_k = int(sys.argv[sys.argv.index("--topk-k") + 1]) if "--topk-k" in sys.argv else 10
loss = sys.argv[sys.argv.index("--loss") + 1] if "--loss" in sys.argv else "bce"
gb = {}
if loss == "gbce":
    gb = dict(num_negatives=int(sys.argv[sys.argv.index("--negatives") + 1]) if "--negatives" in sys.argv else 256,
              gbce_t=float(sys.argv[sys.argv.index("--t") + 1]) if "--t" in sys.argv else 0.75)
if "--lazy" in sys.argv:
    gb["lazy_item_adam"] = True
tr_dp = FusedTrainer(m_dp, process_group=dist.group.WORLD, use_graph=use_graph, l2_emb=l2_emb, loss=loss, **gb)
if rank == 0:
    print("fused reduce-scatter/Adam/all-gather kernel:", tr_dp._dp is not None, "graph:", use_graph, "l2_emb:", l2_emb,
          "loss:", loss, gb)
tr_one = FusedTrainer(m_one, use_graph=False, l2_emb=l2_emb, loss=loss, **gb)
ok = True
for i, nb in enumerate(batches):
    full = {k: torch.from_numpy(v).to(dev) for k, v in nb.items()}
    w = discriminator_weights(full["pos"], full["p_fake"], "soft")
    l1 = float(tr_one.step(full, w_pos=w))
    sh = P.shard_batch({**full, "w": w}, rank, world)
    l2 = float(tr_dp.step(sh, w_pos=sh["w"]))
    if rank == 0:
        print(f"loss single {l1:.6f}  dp{world} {l2:.6f}")
    ok &= abs(l1 - l2) < 2e-3 * (max(1.0, abs(l1)) if loss == "gbce" else 1.0)
    if i == 0:                      # the first step's parameters, before Adam amplifies bf16 noise into sign flips
        d0 = float((m_one.flat_parameters().data - m_dp.flat_parameters().data).abs().max())
        if rank == 0:
            print(f"param drift after the first step {d0:.2e}")
        ok &= d0 < 2e-3
a, b = m_one.flat_parameters().data, m_dp.flat_parameters().data
drift = float((a - b).abs().max())
# replicas must be bit-identical (every element is computed by exactly one rank and written everywhere)
mine = m_dp.flat_parameters().data.clone()
other = mine.clone()
dist.broadcast(other, 0)
ok &= bool(torch.equal(mine, other))
if rank == 0:
    print("replicas bit-identical:", bool(torch.equal(mine, other)))
cos = float(torch.dot(a - 0, b - 0) / (a.norm() * b.norm()))
ok &= drift < 5e-3
# sharded catalogue top-k
g = torch.Generator().manual_seed(3)
feats = (torch.randint(-16, 17, (500, 64), generator=g).float() / 8).to(dev)
table = (torch.randint(-16, 17, (20001, 64), generator=g).float() / 8).to(dev)
ref_s, ref = EV.local_topk(feats, EV.CatalogueIndex(table, 0), 1, topk_k)
lo, hi = EV.CatalogueIndex.shard_bounds(table.shape[0], rank, world)
got_s, ids = EV.sharded_topk(feats, EV.CatalogueIndex(table[lo:hi], lo), dist.group.WORLD, 1, topk_k)
same = bool(torch.equal(ids, ref)) and bool(torch.equal(got_s, ref_s))
ok &= same
flag = torch.tensor([1.0 if ok else 0.0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print(f"param drift after 6 steps {drift:.2e}; sharded top-{topk_k} == unsharded: {same}; ALL OK: {bool(flag.item())}")
# (no destroy_process_group(): with NCCL work captured in live CUDA graphs the communicator teardown can block for minutes)
rc = 0 if flag.item() else 1
torch.cuda.synchronize()
dist.barrier()
tr_dp._graph = None
torch.cuda.synchronize()
sys.stdout.flush()
os._exit(rc)
