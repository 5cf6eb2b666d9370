"""GPU: the tier residency policy (speckv_ext_policy_*, tier.TierPolicy) against the oracle
(oracle_policy_*, driven a batch at a time through oracle.PolicyOracle) where tests/test_policy_gpu.py
does not reach:

* page counts past the grid cap of the grid-stride loops, touch batches of a million ids with
  duplicates and stray ids, promotion batches that evict thousands of pages;
* logical clocks on every boundary of the 11-bit digits of the 44-bit stamps, so that each of the
  four passes of the radix select splits its candidates at a bucket edge;
* the select's edge cases, touches still in flight when a host-driven call runs, CUDA-graph capture,
  the hot threshold and the hit counters.

Every batch is compared as it happens (results, evicted ids in order, is_hot answers); the full
state (tiers, LRU order, statistics) at checkpoints.  Each assertion names the batch and the op.

The library stamps touch index i of a batch with clock + i + 1 and a successful promotion with
++clock; out-of-range ids advance the clock without touching a page.  The tests use that rule only
to aim (`Pair.jump`): what they assert is what the oracle, which has no clock, can see."""
import numpy as np
import pytest
import torch

from cxl_speckv_b200 import SPECKV_ERR_INVAL, SpeckvError, lib
from cxl_speckv_b200.tier import TierPolicy
from oracle.oracle import PolicyOracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BIG = 1 << 62                       # a capacity that is never reached
FILLER = 1 << 27                    # ids per clock-advancing touch (1 GiB)
SLEEP_CYCLES = 100_000_000          # torch.cuda._sleep: about 50 ms at B200 clocks


@pytest.fixture(scope="module")
def filler():
    t = torch.empty(FILLER, dtype=torch.int64, device=DEV)
    yield t
    del t
    torch.cuda.empty_cache()


class Pair:
    """The library's policy and the oracle's, fed the same batches and compared after each one."""

    def __init__(self, n_pages, l1, filler=None):
        self.n = n_pages
        self.gpu = TierPolicy(n_pages, l1, BIG, BIG)
        self.ref = PolicyOracle(n_pages, (l1, BIG, BIG))
        self.clock = 0                  # the library's logical clock, by its stamp rule
        self.batch = 0
        self.filler = filler

    def close(self):
        self.gpu.close()
        self.ref.close()

    def at(self, op):
        return f"batch {self.batch} ({op})"

    def place(self, ids, tier):
        ids = np.asarray(ids, dtype=np.int64)
        got = self.gpu.place(ids.astype(np.uint64), tier).astype(np.int32)
        want = self.ref.place(ids, tier)
        assert np.array_equal(got, np.where(want < 0, 255, want)), self.at(f"place tier {tier}")
        self.batch += 1
        return got

    def touch(self, ids, on_device=True):
        ids = np.asarray(ids, dtype=np.int64)
        if on_device:
            self.gpu.touch(torch.from_numpy(ids).to(DEV))
        else:
            self.gpu.touch(ids.astype(np.uint64))
        self.ref.touch(ids)
        self.clock += ids.size
        self.batch += 1

    def jump(self, to):
        """Advance the library's clock to `to` with out-of-range ids (value n_pages) the oracle never sees."""
        assert to >= self.clock
        self.filler.fill_(self.n)
        while self.clock < to:
            r = min(to - self.clock, FILLER)
            self.gpu.touch(self.filler[:r])
            self.clock += r

    def is_hot(self, ids, op="is_hot"):
        ids = np.asarray(ids, dtype=np.int64)
        got = self.gpu.is_hot(torch.from_numpy(ids).to(DEV)).cpu().numpy()
        want = self.ref.is_hot(ids)
        assert np.array_equal(got, want), self.at(op)
        self.batch += 1
        return got

    def promote(self, ids):
        ids = np.asarray(ids, dtype=np.int64)
        ok, ev = self.gpu.promote(ids.astype(np.uint64))
        want_ok, want_ev = self.ref.promote(ids)
        assert np.array_equal(ok, want_ok), self.at("promote: ok")
        assert np.array_equal(ev, want_ev), self.at(f"promote: evicted ({ev.size} vs {want_ev.size})")
        self.clock += int(want_ok.sum())
        self.batch += 1
        return ok, ev

    def demote(self, ids):
        ids = np.asarray(ids, dtype=np.int64)
        ok = self.gpu.demote(ids.astype(np.uint64))
        assert np.array_equal(ok, self.ref.demote(ids)), self.at("demote")
        self.batch += 1

    def release(self, ids):
        ids = np.asarray(ids, dtype=np.int64)
        self.gpu.release(ids.astype(np.uint64))
        self.ref.release(ids)
        self.batch += 1

    def check_lru(self, op="lru_order"):
        assert np.array_equal(self.gpu.lru_order(), self.ref.lru_order()), self.at(op)

    def check_stats(self, op="stats"):
        got, want = self.gpu.stats(), self.ref.stats()
        for k, v in want.items():
            assert got[k] == v, self.at(f"{op}: {k} {got[k]} vs {v}")

    def check_state(self, op="state"):
        assert np.array_equal(self.gpu.tiers(), self.ref.tiers()), self.at(f"{op}: tiers")
        self.check_lru(f"{op}: lru_order")
        self.check_stats(op)


def stray_ids(rng, n_pages, k, dup=True):
    """k page ids with duplicates and about 1 % stray ids (negative, n_pages and beyond)."""
    ids = rng.integers(0, n_pages, k, dtype=np.int64)
    if dup and k >= 8:
        ids[-(k // 8):] = ids[: k // 8]
    stray = rng.random(k) < 0.01
    ids[stray] = rng.choice(np.array([-1, -(1 << 40), n_pages, n_pages + 1, 1 << 62], dtype=np.int64), int(stray.sum()))
    rng.shuffle(ids)
    return ids


def place_mixed(p, rng):
    """Every page with probability 0.9, into tier 0 / 1 / 2 / 2 (an L1 preference falls back to L3 when full)."""
    tier = rng.choice(np.array([0, 1, 2, 2, 255]), p.n, p=[0.225, 0.225, 0.225, 0.225, 0.1])
    for t in (0, 1, 2):
        p.place(np.flatnonzero(tier == t), t)


# ---- 1 + 2: scale traces, with clock jumps onto the digit boundaries ----------------------------
EDGES = {0: 1 << 11, 2: 1 << 22, 10: 1 << 33}        # batch index -> the boundary its touch straddles
N_BATCHES = 18
CHECKPOINTS = (3, 11, N_BATCHES - 1)


@pytest.mark.parametrize("l1", [0, 1, 4096, 1 << 18, "all"])
@pytest.mark.parametrize("n_pages", [(1 << 20) + 37, 3 << 20])
def test_scale_trace_matches_oracle(filler, n_pages, l1):
    l1 = n_pages + 1 if l1 == "all" else l1
    rng = np.random.default_rng([n_pages, l1])
    p = Pair(n_pages, l1, filler)
    try:
        place_mixed(p, rng)
        p.check_state("after placement")
        probe = stray_ids(rng, n_pages, 1 << 16)
        for b in range(N_BATCHES):
            if b in EDGES:
                # a device touch whose stamps straddle the boundary, then a promotion batch that evicts thousands
                m = int(rng.integers(4096, (1 << 20) + 1))
                p.jump(max(p.clock, EDGES[b] - m // 2))
                assert p.clock < EDGES[b] <= p.clock + m
                p.touch(stray_ids(rng, n_pages, m))
            elif b - 1 in EDGES:
                p.promote(stray_ids(rng, n_pages, 8192))
            else:
                r = rng.random()
                if r < 0.3:
                    p.touch(stray_ids(rng, n_pages, int(rng.integers(1, (1 << 20) + 1))))
                elif r < 0.4:
                    p.touch(stray_ids(rng, n_pages, int(rng.integers(1, 1 << 16))), on_device=False)
                elif r < 0.5:
                    p.is_hot(stray_ids(rng, n_pages, int(rng.integers(1, 1 << 20))))
                elif r < 0.7:
                    p.promote(stray_ids(rng, n_pages, int(rng.integers(1, 8193))))
                elif r < 0.82:
                    p.demote(stray_ids(rng, n_pages, int(rng.integers(1, 4097))))
                elif r < 0.9:
                    p.release(stray_ids(rng, n_pages, int(rng.integers(1, 2049))))
                else:
                    free = np.flatnonzero(p.ref.tiers() == 255)
                    ids = np.concatenate([rng.choice(free, min(free.size, 1024), replace=False),
                                          stray_ids(rng, n_pages, 64)])
                    p.place(ids, int(rng.integers(0, 3)))
            p.is_hot(probe, op="is_hot probe")
            if b in CHECKPOINTS:
                p.check_state()
    finally:
        p.close()


# ---- 2 + 3: the k-th victim's stamp on each side of a bucket edge --------------------------------
@pytest.mark.parametrize("side", [-2, -1, 0, 1, "one_bucket"])
@pytest.mark.parametrize("edge", [1 << 11, 1 << 22, 1 << 33])
def test_kth_victim_at_a_digit_edge(filler, edge, side):
    """1024 full L1 pages touched (with 256 L3 pages among them) in one batch whose stamps straddle
    `edge`; a promotion batch then evicts exactly the k least recently used of them, where the k-th
    carries stamp edge + side: the last ones below the edge or the first ones at it, so the select
    splits its bucket at the edge in every pass from the edge's digit down.  "one_bucket": all the
    stamps share their three upper digits."""
    C, X = 1024, 256
    n = 4 * C
    rng = np.random.default_rng([edge, 7 if side == "one_bucket" else side + 3])
    p = Pair(n, C, filler)
    try:
        p.place(np.arange(C), 0)
        p.place(np.arange(C, n), 2)
        m = C + X
        start = edge if side == "one_bucket" else edge - m // 2 - 1      # the clock before the batch
        forced = [] if side == "one_bucket" else [edge + s - start - 1 for s in (-2, -1, 0, 1)]
        batch = np.empty(m, dtype=np.int64)
        others = np.setdiff1d(np.arange(m), forced)
        l3_at = rng.choice(others, X, replace=False)
        batch[l3_at] = rng.choice(np.arange(C, n), X, replace=False)
        batch[np.setdiff1d(np.arange(m), l3_at)] = rng.permutation(C)
        p.jump(start)
        p.touch(batch)
        stamps = start + 1 + np.flatnonzero(batch < C)                     # the L1 pages' stamps, ascending
        if side == "one_bucket":
            assert stamps[0] >> 11 == stamps[-1] >> 11
            k = C // 2 + 1
        else:
            k = int(np.searchsorted(stamps, edge + side)) + 1
            assert stamps[k - 1] == edge + side
        ok, ev = p.promote(np.arange(n - k, n))
        assert ok.all() and ev.size == k
        head = batch[: stamps[k - 1] - start]                               # the touches up to the k-th victim's
        assert np.array_equal(ev, head[head < C])
        p.check_state()
    finally:
        p.close()


# ---- 3: small hand-built selections -------------------------------------------------------------
def _k_one(p, rng):
    p.place(np.arange(8), 0); p.place(np.arange(8, 32), 2)
    p.touch(rng.permutation(16))
    p.promote([20])


def _k_equal_to_members(p, rng):
    p.place(np.arange(8), 0); p.place(np.arange(8, 32), 2)
    p.touch(rng.permutation(8))
    p.promote(np.arange(16, 24))                       # every L1 member leaves, in stamp order


def _k_past_members(p, rng):
    p.place(np.arange(8), 0); p.place(np.arange(8, 32), 2)
    p.touch(rng.permutation(4))                        # L1 pages 4..7 never enter the list
    p.promote(np.arange(16, 24))                       # 4 members for 8 evictions: then this batch's own pages


def _non_l1_in_front(p, rng):
    p.place(np.arange(8), 0); p.place(np.arange(8, 16), 1); p.place(np.arange(16, 32), 2)
    p.touch(np.concatenate([[20, 9, 30], rng.permutation(8), [21, 10]]))
    p.promote([25, 26, 9])                             # 20, 9, 30 dropped before the first victim
    p.check_lru("after promote")
    p.promote([20])


def _no_l1_in_list(p, rng):
    p.place(np.arange(4), 0); p.place(np.arange(4, 32), 2)
    p.touch(rng.permutation(np.arange(4, 20)))          # the list holds no L1 page
    p.promote([25, 26])                                # the list empties, nothing is evicted, L1 overfills
    p.check_stats("after promote")
    p.touch([4, 1, 5])
    p.promote([27, 28, 29])


def _duplicates_evicted_between(p, rng):
    p.place([0], 0); p.place(np.arange(1, 16), 2)
    p.touch([0, 3])
    p.promote([5, 6, 5, 7, 5, 5])                      # 5 leaves for 6, comes back, leaves for 7, comes back
    p.promote([6, 6, 0])


def _duplicates_no_l1(p, rng):
    p.place(np.arange(16), 2)
    p.touch(rng.permutation(16))
    p.promote([5, 6, 5, 5, 7])                         # L1 capacity 0: each promotion evicts the previous one


SELECT_CASES = {
    "k_one": (32, 8, _k_one),
    "k_equal_to_members": (32, 8, _k_equal_to_members),
    "k_past_members": (32, 8, _k_past_members),
    "non_l1_in_front": (32, 8, _non_l1_in_front),
    "no_l1_in_list": (32, 4, _no_l1_in_list),
    "duplicates_evicted_between": (16, 1, _duplicates_evicted_between),
    "duplicates_no_l1": (16, 0, _duplicates_no_l1),
}


@pytest.mark.parametrize("start", [0, (1 << 22) - 6, (1 << 33) - 6])
@pytest.mark.parametrize("case", list(SELECT_CASES))
def test_select_edge_cases(filler, case, start):
    n, l1, body = SELECT_CASES[case]
    p = Pair(n, l1, filler)
    try:
        p.jump(start)                                  # the cases' stamps straddle 2^22 and 2^33
        body(p, np.random.default_rng(len(case)))
        p.check_state()
    finally:
        p.close()


# ---- 4: host-driven calls while a touch is still queued -------------------------------------------
def _in_flight_setup(seed):
    rng = np.random.default_rng(seed)
    p = Pair(4096, 64)
    p.place(np.arange(64), 0); p.place(np.arange(64, 1024), 1); p.place(np.arange(1024, 3072), 2)
    p.touch(rng.permutation(3072)[:1500])
    p.check_state("before")
    batch = rng.permutation(np.concatenate([np.arange(64), np.arange(500, 600), np.arange(2000, 2100),
                                            np.arange(3072, 3200), [-1, 4096]]))
    return p, batch


@pytest.mark.parametrize("side_stream", [False, True], ids=["same_stream", "side_stream"])
@pytest.mark.parametrize("call", ["place", "release", "promote", "demote", "lru_order", "stats"])
def test_calls_wait_for_a_touch_in_flight(call, side_stream):
    """A device touch queued behind a ~50 ms spin, then a host-driven call: the answer and the state after
    it are the oracle's sequential ones, as if the touch had already run."""
    p, batch = _in_flight_setup(11)
    try:
        ids = torch.from_numpy(batch).to(DEV)
        s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP_CYCLES)
            p.gpu.touch(ids)
        p.ref.touch(batch)
        p.clock += batch.size
        p.batch += 1
        if call == "place":
            p.place(np.arange(3072, 3200), 1)          # pages the queued touch finds unallocated
        elif call == "release":
            p.release(np.concatenate([np.arange(0, 16), np.arange(500, 600), np.arange(2000, 2050)]))
        elif call == "promote":
            p.promote(np.arange(2000, 2040))           # the victims follow the queued touch's order
        elif call == "demote":
            p.demote(np.arange(0, 32))
        elif call == "lru_order":
            p.check_lru()
        else:
            p.check_stats()
        torch.cuda.synchronize()
        p.check_state(f"after {call}")
    finally:
        torch.cuda.synchronize()
        p.close()


def test_touches_on_two_streams_commute():
    """The first touch waits behind a spin on one stream while the second runs on another: the LRU order
    is still the order of the calls."""
    p, batch = _in_flight_setup(13)
    try:
        second = np.random.default_rng(1).permutation(batch)
        a, b = torch.from_numpy(batch).to(DEV), torch.from_numpy(second).to(DEV)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        for s in (s1, s2):
            s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s1):
            torch.cuda._sleep(SLEEP_CYCLES)
            p.gpu.touch(a)
        with torch.cuda.stream(s2):
            p.gpu.touch(b)
        p.ref.touch(batch)
        p.ref.touch(second)
        p.batch += 2
        torch.cuda.synchronize()
        p.check_state("after both touches")
    finally:
        torch.cuda.synchronize()
        p.close()


# ---- 6: the hot threshold and the hit counters -------------------------------------------------------
def test_hot_threshold_and_count_reset():
    p = Pair(64, 8)
    try:
        p.place(np.arange(8), 0); p.place(np.arange(8, 48), 2)        # 48.. unallocated
        # 10 against 11 touches of one page, by duplicates inside one device batch
        batch = np.concatenate([np.full(10, 3), np.full(11, 4), np.full(10, 20), np.full(11, 21),
                                np.full(12, 50), np.full(12, 64), np.full(12, -1)])
        p.touch(np.random.default_rng(0).permutation(batch))
        probe = np.array([3, 4, 20, 21, 50, 63, 64, 65, -1, 1 << 62], dtype=np.int64)
        hot = p.is_hot(probe)
        assert hot.tolist() == [0, 1, 0, 1, 0, 0, 0, 0, 0, 0], hot
        p.touch([3, 20])                                              # the 11th touch
        assert p.is_hot([3, 20]).tolist() == [1, 1]
        # release and place again: the count starts from zero
        p.release([4, 21])
        assert p.is_hot([4, 21]).tolist() == [0, 0]
        p.place([4], 0); p.place([21], 2)
        p.touch([4, 21])
        assert p.is_hot([4, 21]).tolist() == [0, 0]
        p.touch(np.tile([4, 21], 10))
        assert p.is_hot([4, 21]).tolist() == [1, 1]
        p.check_state()
    finally:
        p.close()


def test_hit_counters_on_a_large_batch():
    """One 2^24-id batch over pages of all three tiers, unallocated pages and stray ids: the per-CTA
    counters add up to exact numpy counts."""
    n = 1 << 20
    p = Pair(n, 1 << 18)
    try:
        rng = np.random.default_rng(5)
        place_mixed(p, rng)
        ids = torch.randint(-4, n + 4, (1 << 24,), device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
        p.gpu.touch(ids)
        tiers = p.gpu.tiers()
        h = ids.cpu().numpy()
        h = h[(h >= 0) & (h < n)]
        by_tier = np.bincount(tiers[h], minlength=256)
        st = p.gpu.stats()
        assert (st["l1_hits"], st["l2_hits"], st["l3_accesses"]) == (by_tier[0], by_tier[1], by_tier[2])
        assert by_tier[255] > 0 and min(by_tier[:3]) > 0
    finally:
        p.close()


# ---- 5: capture ---------------------------------------------------------------------------------
def test_touch_refuses_capture():
    """touch on a capturing stream returns SPECKV_ERR_INVAL in both forms and changes nothing; the capture
    stays valid; an is_hot captured alongside reports the counts current at each replay."""
    p, batch = _in_flight_setup(12)
    try:
        L = lib()
        ids = torch.from_numpy(batch).to(DEV)
        host = batch.astype(np.uint64)
        probe_np = np.arange(-2, p.n + 2, dtype=np.int64)
        probe = torch.from_numpy(probe_np).to(DEV)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            st = torch.cuda.current_stream().cuda_stream
            status = [L.speckv_ext_policy_touch(p.gpu._h, ids.data_ptr(), ids.numel(), 1, st),
                      L.speckv_ext_policy_touch(p.gpu._h, host.ctypes.data, host.size, 0, st)]
            with pytest.raises(SpeckvError):
                p.gpu.touch(ids)
            hot = p.gpu.is_hot(probe)
        assert status == [SPECKV_ERR_INVAL, SPECKV_ERR_INVAL]
        p.check_state("after the refused touches")
        p.touch(batch)                                 # touches made afterwards order as the oracle's
        p.check_state("touch after capture")
        for r in range(12):
            g.replay()
            torch.cuda.synchronize()
            assert np.array_equal(hot.cpu().numpy(), p.ref.is_hot(probe_np)), f"replay {r}"
            p.touch(np.tile(batch[r % 3::3], 3))        # counts cross the threshold between replays
        assert p.ref.is_hot(probe_np).any()
        p.check_state("after the replays")
    finally:
        p.close()
