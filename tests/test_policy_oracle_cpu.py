"""CPU: the oracle's batch forms of the residency policy (oracle_policy_*_n, oracle_policy_tiers, driven through
oracle.PolicyOracle) give exactly what the single-page calls give through run_policy_trace, on the traces of
tests/test_policy_gpu.py."""
import numpy as np
import pytest

from oracle.oracle import PolicyOracle
from tests.test_policy_gpu import make_trace, run_oracle


def run_batched(batches, n_pages, caps):
    """The same flattened results as run_oracle, one batch-form call per batch."""
    pol = PolicyOracle(n_pages, caps)
    results = []
    try:
        for op, pages, tier in batches:
            if op == "place_mixed":
                for t in (0, 1, 2):
                    results += pol.place([g for g, tt in pages if tt == t], t).tolist()
            elif op == "place":
                results += pol.place(pages, tier).tolist()
            elif op == "touch":
                pol.touch(pages)
                results += [0] * len(pages)
            elif op == "hot":
                results += pol.is_hot(pages).tolist()
            elif op == "promote":
                ok, ev = pol.promote(pages)
                results.append(("promote", ok.tolist(), ev.tolist()))
            elif op == "demote":
                results += pol.demote(pages).tolist()
            elif op == "release":
                pol.release(pages)
                results += [0] * len(pages)
        return {"results": results, "tiers": pol.tiers().tolist(), "lru": pol.lru_order().tolist(),
                "stats": pol.stats()}
    finally:
        pol.close()


@pytest.mark.parametrize("seed,n_pages,caps", [
    (0, 64, (1 << 40, 1 << 40, 1 << 40)),
    (1, 64, (8, 1 << 40, 1 << 40)),
    (3, 17, (1, 1 << 40, 1 << 40)),
    (4, 33, (0, 1 << 40, 1 << 40)),
    (5, 5000, (100, 1 << 40, 1 << 40)),
])
def test_batch_forms_match_single_page_calls(seed, n_pages, caps):
    batches = make_trace(seed, n_pages, n_batches=400, max_batch=min(64, 2 * n_pages))
    got = run_batched(batches, n_pages, caps)
    want = run_oracle(batches, n_pages, caps)
    assert got["results"] == want["results"]
    assert got["tiers"] == want["tiers"]
    assert got["lru"] == want["lru"]
    assert got["stats"] == want["stats"]


def test_batch_forms_take_ids_as_uint64():
    """A negative id is a page past the end, as the library reads a device int64 tensor."""
    pol = PolicyOracle(8, (2, 1 << 40, 1 << 40))
    try:
        assert pol.place(np.array([0, 1, 2, -1, 8], dtype=np.int64), 0).tolist() == [0, 0, 2, -1, -1]
        pol.touch(np.array([-1, 2, 1 << 62, 0, 8], dtype=np.int64))
        assert pol.lru_order().tolist() == [2, 0]
        assert pol.is_hot(np.array([-1, 0], dtype=np.int64)).tolist() == [0, 0]
        ok, ev = pol.promote(np.array([-5, 2], dtype=np.int64))
        assert ok.tolist() == [0, 1] and ev.tolist() == [0]      # L1 full: its least recently used page leaves
        assert pol.tiers().tolist() == [2, 0, 0] + [255] * 5
    finally:
        pol.close()
