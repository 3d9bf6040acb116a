"""CPU model check of the packed attention kernels' protocol with the fused out-projection
(srfrd_b200/csrc/attention_tc.cu, attn_fwd_tc_kernel<*, true, true> and attn_bwd_tc_kernel<*, true, true>).

The fused kernels reuse shared-memory slots and TMEM columns within an item: forward, K's blocks hold K, then P, then Wo;
V's blocks hold V, then the residual, then r; Q's blocks hold Q, then O, then y; S's TMEM columns hold S, then the
out-projection accumulator.  Backward, P's blocks hold dr, then P; dO's blocks are written by the epilogue warps.  As in
test_pipeline_protocol.py, every warp role's loop is transcribed into a coroutine over simulated parity-wait mbarriers
and run under random interleavings and completion delays.  On top of "every wait passes on the phase it was written
for" and "no deadlock", each slot / column range carries the tag of what it holds, and every access asserts that
  * it reads the tag it was written for (no stale or early read),
  * no asynchronous write (TMA load, MMA result) is in flight on what it reads, and nothing in flight on what it writes.
tcgen05.commit arrives once every MMA issued before it has completed; MMAs complete in issue order.
No GPU, no product code is executed.
"""
import random

import pytest

from tests.test_pipeline_protocol import MBar


class AttnSim:
    def __init__(self, seed, items, max_delay=6):
        self.rng, self.items, self.max_delay = random.Random(seed), items, max_delay
        self.events, self.step_no, self.seq = [], 0, 0
        self.content, self.inflight = {}, {}          # resource -> tag; resource -> list of 'r' / 'w'
        self.mma_queue, self.commits, self.retired = [], [], 0
        self.done = {}

    # ---- time, barriers -------------------------------------------------------------------------------------------
    def later(self, fn, after=None):
        self.seq += 1
        self.events.append((self.step_no + (after if after is not None else self.rng.randint(1, self.max_delay)), self.seq, fn))

    def wait(self, bar, parity, intended):
        while not bar.passes(parity):
            yield
        assert bar.phase == intended + 1, f"wait meant phase {intended}, barrier has completed {bar.phase} phases"

    # ---- resource accesses ----------------------------------------------------------------------------------------
    def _start(self, res, kind, expect=None):
        fl = self.inflight.setdefault(res, [])
        if kind == "r":
            assert "w" not in fl, f"{res} read while a write to it is in flight"
            assert self.content.get(res) == expect, f"{res} holds {self.content.get(res)}, reader expected {expect}"
        else:
            assert not fl, f"{res} written while {fl} in flight on it"
        fl.append(kind)

    def _end(self, res, kind, tag=None):
        self.inflight[res].remove(kind)
        if kind == "w":
            self.content[res] = tag

    def read(self, res, expect):                       # thread (generic proxy) access: synchronous
        self._start(res, "r", expect)
        self._end(res, "r")

    def write(self, res, tag):
        self._start(res, "w")
        self._end(res, "w", tag)

    def tma(self, bar, loads):
        """loads: [(resource, tag)]; one expect_tx arrival, each load completes its bytes independently"""
        bar.arrive_expect_tx(len(loads))
        for res, tag in loads:
            self._start(res, "w")

            def land(res=res, tag=tag):
                self._end(res, "w", tag)
                bar.complete_tx()
            self.later(land)

    def mma(self, reads, writes):
        """reads: [(resource, expected tag)], writes: [(resource, tag)]"""
        for res, exp in reads:
            self._start(res, "r", exp)
        for res, _ in writes:
            self._start(res, "w")
        self.mma_queue.append((reads, writes))

    def commit(self, bar):
        """arrive on bar once every MMA issued so far has completed (commits fire in issue order)"""
        upto = len(self.mma_queue) + self.retired
        self.commits.append(bar)

        def fire():
            if self.commits[0] is not bar:
                return self.later(fire, 1)
            self.commits.pop(0)
            while self.retired < upto:
                reads, writes = self.mma_queue.pop(0)
                self.retired += 1
                for res, _ in reads:
                    self._end(res, "r")
                for res, tag in writes:
                    self._end(res, "w", tag)
            bar.arrive()
        self.later(fire)

    def run(self, procs, max_steps=400000):
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


class FwdSim(AttnSim):
    def __init__(self, seed, items, max_delay=6, kv_wait=True):
        AttnSim.__init__(self, seed, items, max_delay)
        self.kv_wait = kv_wait
        (self.qk_full, self.v_full, self.s_full, self.o_full, self.kv_free, self.q_free, self.w_full, self.o_staged,
         self.proj_full) = (MBar(1) for _ in range(9))
        self.p_full = MBar(8)

    def producer(self):
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.q_free, ph ^ 1, n - 1)
            self.tma(self.qk_full, [("Qs", ("Q", n)), ("Ks", ("K", n))])
            self.tma(self.v_full, [("Vs", ("V", n))])
            yield
            if self.kv_wait:
                yield from self.wait(self.kv_free, ph, n)
            self.tma(self.w_full, [("Ks", ("Wo", n)), ("Vs", ("res", n))])
            yield

    def mma_warp(self):
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.qk_full, ph, n)
            self.mma([("Qs", ("Q", n)), ("Ks", ("K", n))], [("tS", ("S", n))])
            self.commit(self.s_full)
            yield from self.wait(self.p_full, ph, n)
            yield from self.wait(self.v_full, ph, n)
            self.mma([("Ks", ("P", n)), ("Vs", ("V", n))], [("tO", ("O", n))])
            self.commit(self.kv_free)
            self.commit(self.o_full)
            yield from self.wait(self.o_staged, ph, n)
            yield from self.wait(self.w_full, ph, n)
            self.mma([("Qs", ("Ostaged", n)), ("Ks", ("Wo", n))], [("tS", ("R", n))])
            self.commit(self.proj_full)
        self.done["mma"] = self.items

    def epilogue(self):
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.s_full, ph, n)
            self.read("tS", ("S", n))
            yield
            self.write("Ks", ("P", n))
            self.p_full.arrive(8)
            yield from self.wait(self.o_full, ph, n)
            self.read("tO", ("O", n))
            self.write("Qs", ("Ostaged", n))
            self.o_staged.arrive()
            yield
            self.read("Qs", ("Ostaged", n))                      # o leaves
            yield from self.wait(self.proj_full, ph, n)
            yield from self.wait(self.w_full, ph, n)
            self.read("tS", ("R", n))
            self.read("Vs", ("res", n))
            self.write("Vs", ("r", n))
            yield
            self.write("Qs", ("y", n))
            yield
            self.read("Vs", ("r", n))
            self.read("Qs", ("y", n))
            self.q_free.arrive()
        self.done["epi"] = self.items

    def check(self, max_steps=400000):
        self.run({"producer": self.producer(), "mma": self.mma_warp(), "epi": self.epilogue()}, max_steps)
        assert self.done == {"mma": self.items, "epi": self.items}


class BwdSim(AttnSim):
    def __init__(self, seed, items, max_delay=6, staged_count=8):
        AttnSim.__init__(self, seed, items, max_delay)
        (self.in_full, self.in_free, self.sdp_full, self.out_full, self.w_full, self.do_full) = (MBar(1) for _ in range(6))
        self.ds_full, self.do_staged = MBar(8), MBar(staged_count)

    def producer(self):
        self.tma(self.w_full, [("Ws", "WoT")])
        yield
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.in_free, ph ^ 1, n - 1)
            self.tma(self.in_full, [("Qs", ("Q", n)), ("Ks", ("K", n)), ("Vs", ("V", n)), ("Ps", ("dr", n))])
            yield

    def mma_warp(self):
        yield from self.wait(self.w_full, 0, 0)
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.in_full, ph, n)
            self.mma([("Ps", ("dr", n)), ("Ws", "WoT")], [("tDO", ("dO", n))])
            self.commit(self.do_full)
            self.mma([("Qs", ("Q", n)), ("Ks", ("K", n))], [("tS", ("S", n))])
            yield from self.wait(self.do_staged, ph, n)
            self.mma([("Ds", ("dO", n)), ("Vs", ("V", n))], [("tDP", ("dP", n))])
            self.commit(self.sdp_full)
            yield from self.wait(self.ds_full, ph, n)
            self.mma([("Gs", ("dS", n)), ("Ks", ("K", n)), ("Qs", ("Q", n)), ("Ps", ("P", n)), ("Ds", ("dO", n))],
                     [("tDQ", ("dQ", n)), ("tS", ("dK", n)), ("tDP", ("dV", n))])
            self.commit(self.out_full)
        self.done["mma"] = self.items

    def epilogue(self, part):
        """the four warps of one `part` (two processes, so that they may drift apart)"""
        for n in range(self.items):
            ph = n & 1
            yield from self.wait(self.do_full, ph, n)
            self.read("tDO", ("dO", n))
            yield
            if part == 0:          # the tag of the whole slot flips once (the parts write disjoint columns)
                self.write("Ds", ("dO", n))
            self.do_staged.arrive(4)
            yield from self.wait(self.sdp_full, ph, n)
            self.read("tS", ("S", n))
            self.read("tDP", ("dP", n))
            yield
            if part == 0:
                self.write("Ps", ("P", n))
                self.write("Gs", ("dS", n))
            self.ds_full.arrive(4)
            yield from self.wait(self.out_full, ph, n)
            self.read("tDQ", ("dQ", n))
            yield
            self.done.setdefault("bar", {}).setdefault(n, set()).add(part)
            while len(self.done["bar"][n]) < 2:                    # named barrier of the 256 epilogue threads
                yield
            if part == 0:
                self.write("Ds", ("dQout", n))
                self.write("Ks", ("dKout", n))
                self.write("Qs", ("dVout", n))
                self.in_free.arrive()
        self.done["epi%d" % part] = self.items

    def check(self, max_steps=400000):
        self.run({"producer": self.producer(), "mma": self.mma_warp(), "e0": self.epilogue(0), "e1": self.epilogue(1)},
                 max_steps)
        assert self.done["mma"] == self.items and self.done["epi0"] == self.done["epi1"] == self.items


@pytest.mark.parametrize("items", [1, 2, 3, 6])
def test_fused_out_projection_forward_protocol(items):
    for seed in range(6):
        FwdSim(seed, items, max_delay=(2 if seed == 0 else 12)).check()
    FwdSim(7, items, max_delay=300).check(max_steps=3000000)


@pytest.mark.parametrize("items", [1, 2, 3, 6])
def test_fused_out_projection_backward_protocol(items):
    for seed in range(6):
        BwdSim(seed, items, max_delay=(2 if seed == 0 else 12)).check()
    BwdSim(7, items, max_delay=300).check(max_steps=3000000)


def test_forward_model_flags_wo_loaded_over_live_p():
    """Wo lands in K's blocks: loading it before the PV MMA has released P (kv_free) is a hazard the model must see"""
    hits = 0
    for seed in range(20):
        try:
            FwdSim(seed, 2, max_delay=12, kv_wait=False).check(max_steps=50000)
        except AssertionError:
            hits += 1
    assert hits > 0


def test_backward_model_flags_a_miscounted_staging_barrier():
    """do_staged collects all eight epilogue warps; with a count of 4 the dP MMA can start on a half-written dO"""
    with pytest.raises(AssertionError):
        for seed in range(20):
            BwdSim(seed, 3, max_delay=12, staged_count=4).check(max_steps=50000)
