"""GPU: the device-side tier fetch (speckv_ext_tier_fetch).  Every fetched block must equal, bit for bit, the host-driven
restore of the same id (HostTier.restore / restore_blocks, pinned to the oracle by tests/test_tier_gpu.py and
tests/test_ragged_gpu.py); requests the tier cannot serve report status 0 and leave their destination alone."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.oracle import Port

pytestmark = pytest.mark.gpu

import cxl_speckv_b200 as pkg  # noqa: E402
from cxl_speckv_b200 import SpeckvError, prefetch  # noqa: E402
from cxl_speckv_b200.tier import HostTier  # noqa: E402

DEV = "cuda:0"
SENT = {torch.float16: 0x7E01, torch.bfloat16: 0x7F81, torch.float32: 0x7FC00001}   # NaN payloads no decoder writes
INT_VIEW = {torch.float16: torch.int16, torch.bfloat16: torch.int16, torch.float32: torch.int32}


def _sentinel(shape, dtype):
    return torch.full(shape, SENT[dtype], dtype=INT_VIEW[dtype], device=DEV).view(dtype)


def _bits(t):
    return t.view(INT_VIEW[t.dtype])


def _tier(n_bytes):
    return HostTier(pool_bytes=int(n_bytes * 1.6) + (4 << 20))


def _ids(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(DEV)


def _check_same_as_restore(tier, ids, G, dtype, scheme, want_elems):
    out, oel, status = tier.fetch(_ids(ids), G, dtype, scheme=scheme, out=_sentinel((len(ids), G), dtype))
    ref = tier.restore(ids, G, dtype, out=_sentinel((len(ids), G), dtype))
    torch.cuda.synchronize()
    assert torch.equal(_bits(out), _bits(ref))
    assert status.cpu().numpy().tolist() == [1] * len(ids)
    assert np.array_equal(oel.cpu().numpy(), want_elems)
    return out


@pytest.mark.parametrize("G,n", [(2048, 96), (131072, 6), (1000, 40)])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("scheme", [1, 2, 3, 4])
def test_fetch_matches_restore(G, n, dtype, scheme):
    torch.manual_seed(G * 10 + scheme)
    rng = np.random.default_rng(G + scheme)
    x = torch.randn(n * G, device=DEV).to(dtype)
    x[2 * G:3 * G] = 0.25                                                     # long runs
    cache = torch.randn((n, G), device=DEV).to(dtype)
    lens = torch.from_numpy(rng.integers(0, G + 1, n).astype(np.int32)).to(DEV)
    lens[0] = 0
    lens[1] = G
    tier = _tier(3 * n * G * x.element_size())
    try:
        tier.set_scheme(scheme)
        dense = np.arange(n, dtype=np.uint64)
        paged = dense + np.uint64(1 << 40)
        ragged = dense + np.uint64(2 << 40)
        tier.offload(x, G, dense)                                             # stored before enable_fetch
        tier.enable_fetch()
        table = torch.from_numpy(rng.permutation(n).astype(np.int32)).to(DEV)
        tier.offload_blocks(cache, table, paged)
        tier.offload_ragged(cache, G, lens, ragged)                           # the tails behind lens are garbage
        for base, elems in ((dense, np.full(n, G)), (paged, np.full(n, G)), (ragged, lens.cpu().numpy())):
            sel = np.concatenate([rng.permutation(n), rng.integers(0, n, 9)])  # shuffled, with duplicate ids
            out = _check_same_as_restore(tier, base[sel], G, dtype, scheme, elems[sel].astype(np.int32))
        if scheme == 2 and dtype == torch.float16:                            # oracle, directly, on a seeded sample
            out = tier.fetch(_ids(dense[[2, 5]]), G, dtype)[0]
            for row, g in enumerate((2, 5)):
                s, p = Port.compress(x[g * G:(g + 1) * G].cpu().numpy().astype(np.float32))
                ref = Port.decompress(s, p, G).astype(np.float16)
                assert np.array_equal(out[row].cpu().numpy().view(np.uint16), ref.view(np.uint16))
    finally:
        tier.close()


def test_device_count_leaves_the_rest_untouched():
    G, n = 2048, 64
    x = torch.randn(n * G, device=DEV).half()
    tier = _tier(n * G * 2)
    try:
        ids = np.arange(n, dtype=np.uint64)
        tier.offload(x, G, ids)
        tier.enable_fetch()
        sel = np.random.default_rng(1).permutation(n)
        for c in (0, 5, 63, 64, 1000):
            out = _sentinel((n, G), torch.float16)
            oel = torch.full((n,), 0x5A5A5A5A, dtype=torch.int32, device=DEV)
            status = torch.full((n,), 77, dtype=torch.uint8, device=DEV)
            count = torch.tensor([c], dtype=torch.int32, device=DEV)
            tier.fetch(_ids(sel), G, torch.float16, out=out, count=count, out_elems=oel, status=status)
            live = min(c, n)
            if live:
                ref = tier.restore(sel[:live], G, torch.float16)
                assert torch.equal(_bits(out[:live]), _bits(ref))
            assert torch.equal(_bits(out[live:]), _bits(_sentinel((n - live, G), torch.float16)))
            assert (oel[:live] == G).all() and (oel[live:] == 0x5A5A5A5A).all()
            assert (status[:live] == 1).all() and (status[live:] == 77).all()
    finally:
        tier.close()


def test_unserved_requests():
    G = 2048
    tier = _tier(64 * G * 4)
    try:
        a = torch.randn(4 * G, device=DEV).half()
        tier.offload(a, G, np.arange(4, dtype=np.uint64))                          # 0..3 served
        tier.offload(torch.randn(4 * 1000, device=DEV).half(), 1000, np.arange(10, 14, dtype=np.uint64))  # geometry
        tier.offload(torch.randn(2 * G, device=DEV).bfloat16(), G, np.array([20, 21], dtype=np.uint64))    # dtype
        tier.set_scheme(0)
        tier.offload(torch.randn(2 * G, device=DEV).half(), G, np.array([30, 31], dtype=np.uint64))        # raw
        tier.set_scheme(1)
        tier.offload(torch.randn(2 * G, device=DEV).half(), G, np.array([40, 41], dtype=np.uint64))        # codes
        tier.enable_fetch()
        ids = np.array([0, 99, 10, 20, 30, 40, 3, 1 << 63, 2], dtype=np.uint64)
        ok = np.array([1, 0, 0, 0, 0, 0, 1, 0, 1], dtype=np.uint8)
        out, oel, status = tier.fetch(_ids(ids.view(np.int64)), G, torch.float16, scheme=2,
                                      out=_sentinel((len(ids), G), torch.float16))
        assert np.array_equal(status.cpu().numpy(), ok)
        assert np.array_equal(oel.cpu().numpy(), ok.astype(np.int32) * G)
        sent = _bits(_sentinel((G,), torch.float16))
        ref = tier.restore(ids[ok == 1], G, torch.float16)
        assert torch.equal(_bits(out[torch.from_numpy(ok == 1).to(DEV)]), _bits(ref))
        for i in np.flatnonzero(ok == 0):
            assert torch.equal(_bits(out[i]), sent)
        # the codes-only blocks are served by the codes decoder (scheme 1 or 4), the RLE ones are not
        out, oel, status = tier.fetch(_ids([40, 41, 0]), G, torch.float16, scheme=4)
        assert status.cpu().numpy().tolist() == [1, 1, 0]
        assert torch.equal(_bits(out[:2]), _bits(tier.restore(np.array([40, 41], dtype=np.uint64), G, torch.float16)))
    finally:
        tier.close()


@pytest.mark.parametrize("G", [2048, 131072])
def test_paged_scatter_writes_only_named_blocks(G):
    n, nb = 24, 64
    rng = np.random.default_rng(G)
    x = torch.randn(n * G, device=DEV).bfloat16()
    tier = _tier(n * G * 2)
    try:
        ids = np.arange(n, dtype=np.uint64) + np.uint64(500)
        tier.offload(x, G, ids)
        tier.enable_fetch()
        sel = rng.permutation(n)[:17]
        table = torch.from_numpy(rng.permutation(nb)[:17].astype(np.int32)).to(DEV)
        cache = torch.randn((nb, G), device=DEV).bfloat16()
        want = tier.restore_blocks(ids[sel], cache.clone(), table)
        _, oel, status = tier.fetch(_ids(ids[sel]), G, torch.bfloat16, out=cache, block_table=table)
        assert torch.equal(_bits(cache), _bits(want))
        assert (status == 1).all() and (oel == G).all()
    finally:
        tier.close()


def test_directory_upkeep_and_graph_across_growth():
    G, n0 = 2048, 64
    s = torch.cuda.Stream()
    tier = _tier(8192 * G * 2)
    try:
        ids = np.arange(n0, dtype=np.uint64) * np.uint64(7919)
        with torch.cuda.stream(s):
            tier.offload(torch.randn(n0 * G, device=DEV).half(), G, ids)
            tier.enable_fetch()
            # re-offloading an id with new data: the next fetch returns the new data
            tier.offload(torch.randn(2 * G, device=DEV).half(), G, ids[:2])
            _check_same_as_restore(tier, ids[:8], G, torch.float16, 2, np.full(8, G, np.int32))
            # a dropped id is no longer served (drop moves later entries of its probe run: the rest still is)
            tier.drop(ids[8:40])
            status = tier.fetch(_ids(ids[:48]), G, torch.float16)[2]
            assert status.cpu().numpy().tolist() == [1] * 8 + [0] * 32 + [1] * 8
            # capture a fetch graph, then grow the directory well past its first table
            sel = _ids(ids[[0, 3, 45, 60]])
            out = torch.empty((4, G), dtype=torch.float16, device=DEV)
            oel = torch.empty(4, dtype=torch.int32, device=DEV)
            st = torch.empty(4, dtype=torch.uint8, device=DEV)
            tier.fetch(sel, G, torch.float16, out=out, out_elems=oel, status=st)
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                tier.fetch(sel, G, torch.float16, out=out, out_elems=oel, status=st)
            more = np.arange(3000, dtype=np.uint64) + np.uint64(1 << 20)
            tier.offload(torch.randn(3000 * G, device=DEV).half(), G, more)
            tier.offload(torch.randn(4 * G, device=DEV).half(), G, ids[[0, 3, 45, 60]])   # new contents of the captured ids
            g.replay()
            s.synchronize()
            assert torch.equal(_bits(out), _bits(tier.restore(ids[[0, 3, 45, 60]], G, torch.float16)))
            assert (st == 1).all() and (oel == G).all()
            # ids added after the capture are found when the id tensor is rewritten before a replay
            sel.copy_(_ids(more[[0, 1234, 2999, 7]]))
            g.replay()
            s.synchronize()
            assert torch.equal(_bits(out), _bits(tier.restore(more[[0, 1234, 2999, 7]], G, torch.float16)))
            assert (st == 1).all()
    finally:
        tier.close()


def test_prefetch_chain_from_the_tier_in_one_graph():
    G, n_blocks, batch, k, base = 2048, 512, 32, 4, 1 << 32
    rng = np.random.default_rng(3)
    emb = ((rng.random((4096, 64), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    wout = ((rng.random((4096, 128), dtype=np.float32) - 0.5) * 0.1).astype(np.float32)
    prefetch.load_predictor(emb, wout)
    tier = _tier(n_blocks * G * 2)
    s = torch.cuda.Stream()
    try:
        with torch.cuda.stream(s):
            tier.offload(torch.randn(n_blocks * G, device=DEV).half(), G,
                         np.arange(n_blocks, dtype=np.uint64) + np.uint64(base))
            tier.enable_fetch()
            cap = batch * k
            toks = torch.from_numpy(rng.integers(0, 4096, (batch, 16)).astype(np.int32)).to(DEV)
            table = torch.zeros((prefetch.table_records(batch, k), prefetch.REQUEST_BYTES), dtype=torch.uint8, device=DEV)
            block_index = torch.zeros(cap, dtype=torch.int32, device=DEV)
            count = torch.zeros(1, dtype=torch.int32, device=DEV)
            ids = torch.zeros(cap, dtype=torch.int64, device=DEV)
            out = torch.empty((cap, G), dtype=torch.float16, device=DEV)
            oel = torch.empty(cap, dtype=torch.int32, device=DEV)
            st = torch.empty(cap, dtype=torch.uint8, device=DEV)

            def step():
                prefetch.emit(toks, k=k, layer_id=0, timestamp=1, table=table)
                prefetch.route(table, 1, cap, n_blocks, 1, 0, block_index=block_index, count=count)
                torch.add(block_index.long(), base, out=ids)
                tier.fetch(ids, G, torch.float16, out=out, count=count, out_elems=oel, status=st)

            step()
            s.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                step()
            for r in range(3):
                toks.copy_(torch.from_numpy(rng.integers(0, 4096, (batch, 16)).astype(np.int32)))
                g.replay()
                s.synchronize()
                n = int(count.item())
                assert 0 < n <= cap
                want = tier.restore(ids[:n].cpu().numpy().astype(np.uint64), G, torch.float16)
                assert torch.equal(_bits(out[:n]), _bits(want))
                assert (st[:n] == 1).all() and (oel[:n] == G).all()
    finally:
        tier.close()


def test_argument_checks():
    L = pkg.lib()
    G, n = 2048, 8
    tier = _tier(n * G * 2)
    try:
        tier.offload(torch.randn(n * G, device=DEV).half(), G, np.arange(n, dtype=np.uint64))
        ids = _ids(np.arange(n))
        with pytest.raises(SpeckvError) as e:
            tier.fetch(ids, G, torch.float16)                                # before enable_fetch
        assert e.value.status == pkg.SPECKV_ERR_INVAL
        tier.enable_fetch()
        tier.enable_fetch()                                                  # idempotent
        with pytest.raises(SpeckvError) as e:
            tier.fetch(ids, G, torch.float16, scheme=0)
        assert e.value.status == pkg.SPECKV_ERR_INVAL
        out = torch.empty((n, G), dtype=torch.float16, device=DEV)
        need = L.speckv_ext_tier_fetch_workspace_bytes(n, G)
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def call(n_req, ws_bytes, dev_ids=ids, dev_out=out, dev_ws=ws):
            return L.speckv_ext_tier_fetch(tier._h, dev_ids.data_ptr(), None, n_req, G, 0, 2, dev_out.data_ptr(), None,
                                           None, None, dev_ws.data_ptr(), ws_bytes, stream)

        assert call(n, need - 1) == pkg.SPECKV_ERR_INVAL
        assert call(0, 0) == pkg.SPECKV_OK
        assert call(n, need) == pkg.SPECKV_OK
        torch.cuda.synchronize()
        assert torch.equal(_bits(out), _bits(tier.restore(np.arange(n, dtype=np.uint64), G, torch.float16)))
        if torch.cuda.device_count() < 2:
            pytest.skip("one GPU: the other-device check needs two")
        with torch.cuda.device(1):
            ids1, out1 = ids.to("cuda:1"), out.to("cuda:1")
            ws1 = torch.empty(need, dtype=torch.uint8, device="cuda:1")
            stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert call(n, need, ids1, out1, ws1) == pkg.SPECKV_ERR_INVAL
    finally:
        tier.close()
