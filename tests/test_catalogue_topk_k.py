"""Full-catalogue top-k for 10 < k <= 64: the k-list variants of the catalogue kernels (srfrd_b200/csrc/topk.cu), the
k-list merge (K9), the 8k-byte wire row and HR@k / NDCG@k.

GPU tests: bit-exact against the oracle on dyadic inputs, the top-10 kernels' lists as a prefix, Gaussian precision,
row shards emulated on one GPU, the benchmark size, the metrics and the refusals.  CPU tests: the gloo all-gather of
2k-word rows, hr_ndcg_from_topk's width check and a model check of the unit form's ring refill at the short rings the
k-list variant runs (the machinery of test_pipeline_protocol.py)."""
import numpy as np
import pytest
import torch
import torch.distributed as dist

from oracle import srfrd_oracle as O
from tests.test_dp_protocol import _run
from tests.test_pipeline_protocol import MBar, Sim

bf16 = torch.bfloat16
gpu = pytest.mark.gpu


def _dyadic(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-16, 17, shape, generator=g).float() / 8.0


def _oracle_padded(feats, table, k, **kw):
    """oracle top-k with the kernel's tail for N < k: (-inf, -1)"""
    v, i = O.catalogue_topk(feats, table, k, **kw)
    if v.shape[1] < k:
        pad = k - v.shape[1]
        v = np.concatenate([v, np.full((v.shape[0], pad), -np.inf)], 1)
        i = np.concatenate([i, np.full((i.shape[0], pad), -1, np.int64)], 1)
    return v, i


# ------------------------------------------------------------------------------------------------------------ GPU
@gpu
@pytest.mark.parametrize("U,N,D,k", [(5, 300, 16, 64), (200, 5000, 64, 11), (130, 70000, 64, 50), (300, 20000, 64, 20),
                                     (100, 3000, 128, 64), (64, 1000, 256, 48), (40, 2000, 256, 20), (7, 30, 64, 64),
                                     (260, 9000, 64, 64)])
def test_topk_k_bit_exact_on_dyadic_inputs(U, N, D, k):
    """Entries j/8 with |j| <= 16: every partial sum is exact in fp32, so ids and scores must equal the oracle's, ties
    broken by lower id.  5000 / 9000 items leave a ragged last tile; N = 30 < k leaves an empty tail (-inf, -1);
    130 users x 70 000 items cut the one user group into many pieces; 260 users fill two groups."""
    from srfrd_b200 import evaluation as EV, ops
    feats, table = _dyadic((U, D), 190 + k), _dyadic((N + 1, D), 191 + D)
    table[5] = table[9]                                   # forced exact ties
    table[N] = table[7]
    v_ref, i_ref = _oracle_padded(feats, table, k)
    idx = EV.CatalogueIndex(table.cuda(), 0)
    if (U, N) == (130, 70000):
        assert ops.catalogue_topk_plan(U, idx.n_rows, idx.row_lo, idx.Dp, 1, k) > 2
    s, i = EV.local_topk(feats.cuda(), idx, 1, k)
    assert s.shape == (U, k) and i.shape == (U, k)
    assert np.array_equal(i.cpu().numpy(), i_ref)
    assert np.array_equal(s.cpu().numpy(), v_ref.astype(np.float32))


@gpu
@pytest.mark.parametrize("D", [64, 128])
def test_top10_is_the_prefix_of_top64_and_small_k_the_prefix_of_top10(D):
    from srfrd_b200 import evaluation as EV
    feats, table = _dyadic((500, D), 3 + D).cuda(), _dyadic((30001, D), 4 + D).cuda()
    idx = EV.CatalogueIndex(table, 0)
    s10, i10 = EV.local_topk(feats, idx, 1)
    s64, i64 = EV.local_topk(feats, idx, 1, 64)
    assert torch.equal(i64[:, :10], i10) and torch.equal(s64[:, :10], s10)
    for k in (1, 5, 10):
        sk, ik = EV.local_topk(feats, idx, 1, k)
        assert torch.equal(ik, i10[:, :k]) and torch.equal(sk, s10[:, :k])


@gpu
def test_topk_k_gaussian_and_split_precision():
    """Same bounds as the top-10 test: index mismatches only at near-ties (gap < 1e-5), < 1 % of entries."""
    from srfrd_b200 import evaluation as EV
    g = torch.Generator().manual_seed(92)
    U, N, D, k = 300, 40000, 64, 50
    feats = torch.randn(U, D, generator=g)
    table = (torch.randn(N + 1, D, generator=g) * 0.05).to(bf16).float()
    idx = EV.CatalogueIndex(table.cuda(), 0)
    v_ref, i_ref = O.catalogue_topk(feats, table, k, operand_dtype=bf16)
    s, i = EV.local_topk(feats.cuda(), idx, 1, k)
    got_i, got_s = i.cpu().numpy(), s.cpu().numpy()
    mism = got_i != i_ref
    assert np.all(np.abs(got_s - v_ref)[mism] < 1e-5) and mism.mean() < 0.01
    np.testing.assert_allclose(got_s, v_ref, rtol=1e-5, atol=1e-5)
    v32, i32 = O.catalogue_topk(feats, table, k)
    s3, i3 = EV.local_topk(feats.cuda(), idx, 3, k)
    m3 = i3.cpu().numpy() != i32
    assert m3.mean() < 0.01 and np.all(np.abs(s3.cpu().numpy() - v32)[m3] < 1e-5)
    np.testing.assert_allclose(s3.cpu().numpy(), v32, rtol=1e-4, atol=1e-5)


def _shards(n_rows, G):
    """G - 1 ceil-split row ranges followed by one empty shard"""
    from srfrd_b200.evaluation import CatalogueIndex
    return [CatalogueIndex.shard_bounds(n_rows, r, G - 1) for r in range(G - 1)] + [(n_rows, n_rows)]


def _sharded_both_ways(feats, table, G, k):
    """per-shard top-k merged (a) by merge_shards over the (U, G, k) lists and (b) by merge_topk_packed over a
    hand-built gathered wire buffer (G, U, 2k), as the all-gather would deliver it"""
    from srfrd_b200 import evaluation as EV, ops
    U = feats.shape[0]
    L = EV.list_len(k)
    ss, ii, wires = [], [], []
    for lo, hi in _shards(table.shape[0], G):
        index = EV.CatalogueIndex(table[lo:hi].cuda(), lo)
        s, i = EV.local_topk(feats.cuda(), index, 1, k)
        ss.append(s); ii.append(i)
        packed = torch.empty(U, 2 * L, dtype=torch.float32, device="cuda")
        if index.n_rows <= index.row_lo:
            packed.view(torch.int32).fill_(-1)
        else:
            EV._local_lists(feats.cuda(), index, 1, packed, k)
        wires.append(packed)
    ms, mi = EV.merge_shards(torch.stack(ss, 1), torch.stack(ii, 1), k)
    gathered = torch.stack(wires, 0).contiguous()
    ps = torch.empty(U, k, dtype=torch.float32, device="cuda")
    pi = torch.empty(U, k, dtype=torch.int64, device="cuda")
    ops.merge_topk_packed(gathered, U, G, k, ps, pi)
    return (ms, mi), (ps, pi)


@gpu
def test_row_shards_merge_to_the_unsharded_topk():
    """8 shards, the last one empty, k = 50: both merges equal the unsharded top-50 and the oracle, bit for bit."""
    from srfrd_b200 import evaluation as EV
    U, N, D, k = 150, 9000, 64, 50
    feats, table = _dyadic((U, D), 93), _dyadic((N + 1, D), 94)
    _, i_ref = O.catalogue_topk(feats, table, k)
    s_un, i_un = EV.local_topk(feats.cuda(), EV.CatalogueIndex(table.cuda(), 0), 1, k)
    assert np.array_equal(i_un.cpu().numpy(), i_ref)
    (ms, mi), (ps, pi) = _sharded_both_ways(feats, table, 8, k)
    for s, i in ((ms, mi), (ps, pi)):
        assert torch.equal(i, i_un) and torch.equal(s, s_un)


@gpu
def test_benchmark_size_top64():
    """1 M items x D = 64 x 768 users, k = 64, dyadic: unsharded and 8-shard results equal the oracle on a user subset."""
    from srfrd_b200 import evaluation as EV
    U, N, D, k = 768, 1_000_000, 64, 64
    feats, table = _dyadic((U, D), 95), _dyadic((N + 1, D), 96)
    sub = np.arange(0, U, 12)
    v_ref, i_ref = O.catalogue_topk(feats[sub], table, k, chunk=32)
    s, i = EV.local_topk(feats.cuda(), EV.CatalogueIndex(table.cuda(), 0), 1, k)
    assert np.array_equal(i.cpu().numpy()[sub], i_ref)
    assert np.array_equal(s.cpu().numpy()[sub], v_ref.astype(np.float32))
    (ms, mi), (ps, pi) = _sharded_both_ways(feats, table, 8, k)
    assert torch.equal(mi, i) and torch.equal(pi, i) and torch.equal(ms, s) and torch.equal(ps, s)


@gpu
def test_full_catalogue_metrics_at_20_match_oracle():
    """HR@20 / NDCG@20 from evaluate_full_catalogue(k=20) vs the oracle's exact ranking (same bound as the @10 test)."""
    from srfrd_b200 import SRFR_model as M, evaluation as EV, synth
    data = synth.make_interactions(21, 3000, 5000, 5, 4.0, 50)
    torch.manual_seed(1)
    m = M.SRFR(data.itemnum, 50, 64, 16, 0.0, 2, 1, "cuda")
    for _, p in m.named_parameters():
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    m = m.to("cuda").eval()
    users0 = np.nonzero(data.test_item > 0)[0][:2000]
    seq, rsq, tgt = synth.eval_sequences(data, 50, users0)
    ndcg, hr, ids = EV.evaluate_full_catalogue(m, torch.from_numpy(seq).cuda(), torch.from_numpy(rsq).cuda(),
                                               torch.from_numpy(tgt), n_split=3, k=20)
    assert ids.shape == (len(users0), 20)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    h = O.encode(sd, "SRFR", torch.from_numpy(seq), torch.from_numpy(rsq), 1)[:, -1, :]
    rank = O.full_catalogue_rank(h, sd["embedding_layer.item_embed.weight"], tgt)
    ndcg_ref, hr_ref = O.hr_ndcg_from_rank(rank, 20)
    assert abs(hr - hr_ref) <= 1e-3 and abs(ndcg - ndcg_ref) <= 1e-3, (hr, hr_ref, ndcg, ndcg_ref)
    n10, h10 = EV.hr_ndcg_from_topk(ids, torch.from_numpy(tgt), 10)
    assert h10 <= hr and n10 <= ndcg


@gpu
def test_k_limits_are_refused_before_any_launch():
    from srfrd_b200 import evaluation as EV, ops
    assert ops.catalogue_topk_kmax(64, 1) == 64
    assert ops.catalogue_topk_kmax(128, 1) == 64
    assert ops.catalogue_topk_kmax(256, 1) == 48
    assert ops.catalogue_topk_kmax(128, 3) == 10                         # tile form (n_split * D > 256)
    for k in (0, 65):
        with pytest.raises(RuntimeError, match="k must be in 1..64"):
            ops.catalogue_topk_plan(100, 1001, 1, 64, 1, k)
    with pytest.raises(RuntimeError, match="exceeds the limit 48"):
        ops.catalogue_topk_plan(100, 1001, 1, 256, 1, 49)
    with pytest.raises(RuntimeError, match="tile form"):
        ops.catalogue_topk_plan(100, 1001, 1, 128, 3, 11)
    ops.catalogue_topk_plan(100, 1001, 1, 128, 3, 10)                    # the tile form keeps k <= 10
    feats, table = _dyadic((10, 256), 1), _dyadic((101, 256), 2)
    idx = EV.CatalogueIndex(table.cuda(), 0)
    from srfrd_b200 import _lib
    n0 = _lib.launch_count
    for k in (0, 65, 49):
        with pytest.raises(RuntimeError):
            EV.local_topk(feats.cuda(), idx, 1, k)
    assert _lib.launch_count == n0                                      # no library call got through
    with pytest.raises(RuntimeError):
        EV.local_topk(feats[:, :128].cuda(), EV.CatalogueIndex(table[:, :128].cuda(), 0), 3, 11)


# ------------------------------------------------------------------------------------------------------------ CPU
def _topk50_job(rank, world):
    from srfrd_b200 import parallel as P
    k = 50
    g = torch.Generator().manual_seed(19)
    feats = torch.randint(-16, 17, (37, 32), generator=g).float() / 8
    table = torch.randint(-16, 17, (1001, 32), generator=g).float() / 8
    lo, hi = P.shard_rows(table.shape[0], rank, world)
    first = 1 if lo == 0 else 0
    sc = (feats @ table[lo + first:hi].T).numpy()
    v, i = O.topk_stable(sc, k, first_id=lo + first)
    # the k-list wire row: k fp32 scores + k int32 global ids per user (8k bytes), one all-gather
    packed = torch.from_numpy(np.concatenate([v.astype(np.float32), i.astype(np.int32).view(np.float32)], 1))
    gathered = P.allgather_packed_topk(packed, dist.group.WORLD)
    assert gathered.shape == (world, 37, 2 * k)
    mv, mi = P.merge_packed_topk_host(gathered, k)
    return mi


def test_gloo_allgather_of_top50_wire_rows_merges_to_the_unsharded_top50():
    g = torch.Generator().manual_seed(19)
    feats = torch.randint(-16, 17, (37, 32), generator=g).float() / 8
    table = torch.randint(-16, 17, (1001, 32), generator=g).float() / 8
    _, ref = O.catalogue_topk(feats, table, 50)
    outs = _run(_topk50_job, port=29631)
    for mi in outs:
        np.testing.assert_array_equal(mi, ref)


def test_hr_ndcg_refuses_k_wider_than_the_list():
    from srfrd_b200 import evaluation as EV
    ids = torch.arange(40).view(4, 10)
    with pytest.raises(ValueError, match="exceeds the 10 ids"):
        EV.hr_ndcg_from_topk(ids, torch.tensor([0, 11, 25, 99]), 20)
    ndcg, hr = EV.hr_ndcg_from_topk(ids, torch.tensor([0, 11, 25, 99]), 10)
    assert hr == 0.75 and abs(ndcg - (1 + 1 / np.log2(3) + 1 / np.log2(7)) / 4) < 1e-12


def test_list_length_rule():
    from srfrd_b200 import evaluation as EV
    assert [EV.list_len(k) for k in (1, 10, 11, 64)] == [10, 10, 11, 64] and EV.KMAX == 64
    for k in (0, 65):
        with pytest.raises(RuntimeError):
            EV.list_len(k)


# ---- model check of catalogue_unitmax_kernel's ring (no producer warp: the issuers refill the slots) ----------------
class UnitSim(Sim):
    """catalogue_unitmax_kernel's protocol.  Four issuers: w = user tile + 2 * tile parity; issuer 0 fills the ring of
    `ring` item tiles (kblocks stages each) up front.  After issuing tile n's MMAs, the SECOND of the two issuers of n's
    parity to get there (shared counter) re-fills tile n - 2's slot with tile n - 2 + ring: passing tempty[w] for tile n
    told each of them that its own MMAs on tile n - 2 are complete.  The epilogue groups of user tiles 0 / 1 read tfull[w]
    and hand the accumulator back on tempty[w]; afull / aempty hand the user tiles over per piece.  Asserted besides the
    parity rule: a slot is never re-filled while an MMA may still read it, an MMA reads the tile it was written for and an
    accumulator is never overwritten before the epilogue has read it."""

    def __init__(self, seed, pieces, kblocks, ring, max_delay=6):
        Sim.__init__(self, seed, sum(pieces), kblocks, ring * kblocks, 1, 4, 2, False, False, max_delay)
        self.pieces, self.ring_tiles = pieces, ring
        self.full = [MBar(1) for _ in range(self.stages)]
        self.tfull = [MBar(1) for _ in range(4)]
        self.tempty = [MBar(1) for _ in range(4)]          # (4 epilogue warp arrivals modelled as one)
        self.afull, self.aempty = MBar(2), MBar(4)
        self.rcnt = [0] * self.stages
        self.content = [None] * self.stages               # tile whose k-block a slot holds
        self.reads = [0] * self.stages                    # MMAs issued on a slot and not complete yet
        self.acc = [None] * 4                             # tile last written into accumulator stage w ...
        self.acc_read = [None] * 4                        # ... and last read back by the epilogue
        self.seen = {"mma": [], "epi": []}

    def load(self, slot_stage, tile, kb):
        st = slot_stage + kb
        assert self.reads[st] == 0, f"slot {st} re-filled while an MMA may still read it"
        self.full[st].arrive_expect_tx(1)

        def land():
            assert self.reads[st] == 0, f"slot {st} overwritten under a running MMA"
            self.content[st] = (tile, kb)
            self.full[st].complete_tx()
        self.later(land)

    def u_issuer(self, w):
        ub, par = w & 1, w >> 1
        queue = []                                        # this thread's MMAs and commits complete in order

        def push(fn):
            queue.append(fn)

            def fire():
                if queue[0] is not fn:
                    return self.later(fire, 1)
                queue.pop(0)
                fn()
            self.later(fire)

        T, R, kb_n = self.T, self.ring_tiles, self.kblocks
        if w == 0:
            for m in range(min(R, T)):
                for kb in range(kb_n):
                    self.load(m * kb_n, m, kb)
        stage, phase, uphase, aphase, own, n = 0, 0, 0, 0, 0, 0
        for pi, ntiles in enumerate(self.pieces):
            yield from self.wait(self.afull, uphase, pi)
            uphase ^= 1
            for _ in range(ntiles):
                if (n & 1) == par:
                    yield from self.wait(self.tempty[w], aphase ^ 1, own - 1)
                    aphase ^= 1
                    for kb in range(kb_n):
                        st, ph = stage + kb, phase
                        if st >= self.stages:
                            st, ph = st - self.stages, ph ^ 1
                        yield from self.wait(self.full[st], ph, n // R)
                        assert self.content[st] == (n, kb), f"MMA of tile {n} reads {self.content[st]}"
                        assert self.acc[w] is None or self.acc_read[w] == self.acc[w], "accumulator overwritten unread"
                        self.reads[st] += 1
                        push(lambda st=st: self.reads.__setitem__(st, self.reads[st] - 1))
                        yield
                    self.acc[w] = n
                    push(lambda w=w: self.tfull[w].arrive())
                    if n >= 2 and n - 2 + R < T:
                        ps = (stage - 2 * kb_n) % self.stages
                        self.rcnt[ps] += 1
                        if self.rcnt[ps] == 2:
                            self.rcnt[ps] = 0
                            for kb in range(kb_n):
                                self.load(ps, n - 2 + R, kb)
                    self.seen["mma"].append((n, ub))
                    own += 1
                    yield
                stage += kb_n
                if stage >= self.stages:
                    stage, phase = stage - self.stages, phase ^ 1
                n += 1
            push(lambda: self.aempty.arrive())

    def u_epilogue(self, ub):
        uphase, tph, n = 0, [0, 0], 0
        for pi, ntiles in enumerate(self.pieces):
            yield from self.wait(self.aempty, uphase ^ 1, pi - 1)
            uphase ^= 1
            yield                                         # stage this user tile into TMEM
            self.afull.arrive()
            for _ in range(ntiles):
                odd = n & 1
                w = ub + 2 * odd
                yield from self.wait(self.tfull[w], tph[odd], n // 2)
                tph[odd] ^= 1
                assert self.acc[w] == n
                yield                                     # tcgen05.ld
                self.acc_read[w] = n
                self.tempty[w].arrive()
                self.seen["epi"].append((n, ub))
                n += 1

    def run(self, max_steps=400000):
        procs = {"epi0": self.u_epilogue(0), "epi1": self.u_epilogue(1)}
        for w in range(4):
            procs["mma%d" % w] = self.u_issuer(w)
        while procs:
            self.step_no += 1
            assert self.step_no < max_steps, f"deadlock / livelock: {sorted(procs)} still running"
            due = [e for e in self.events if e[0] <= self.step_no]
            self.events = [e for e in self.events if e[0] > self.step_no]
            for _, _, fn in sorted(due, key=lambda e: (e[0], e[1])):
                fn()
            name = self.rng.choice(sorted(procs))
            try:
                next(procs[name])
            except StopIteration:
                del procs[name]
        want = sorted((n, ub) for n in range(self.T) for ub in (0, 1))
        assert sorted(self.seen["mma"]) == want and sorted(self.seen["epi"]) == want


@pytest.mark.parametrize("ring", [4, 6, 8])
@pytest.mark.parametrize("kblocks", [1, 2, 4])
def test_unit_form_ring_refill_protocol(ring, kblocks):
    """the k-list variant runs rings of 4 item tiles (D = 128, k = 64) where the top-10 form's shortest is 6"""
    for pieces in ([1], [2], [5], [3, 1, 4], [1, 1, 1, 1], [11, 6], [30]):
        for seed in range(3):
            UnitSim(seed + 7 * ring, pieces, kblocks, ring, max_delay=(2 if seed == 0 else 9)).run()


def test_unit_form_ring_refill_under_extreme_reordering():
    for seed in range(3):
        UnitSim(seed, [11, 6, 9], 2, 4, max_delay=300).run(max_steps=2000000)


def test_unit_model_flags_a_ring_of_two_tiles():
    """with 2 tiles, tile n - 2's slot IS tile n's: the refill comes after tile n's MMAs that need it"""
    flagged = 0
    for seed in range(8):
        try:
            UnitSim(seed, [9], 1, 2).run(max_steps=20000)
        except AssertionError:
            flagged += 1
    assert flagged == 8
