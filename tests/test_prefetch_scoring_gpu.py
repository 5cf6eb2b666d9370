"""GPU: prefetch scoring against the fp64 reference (tests/lstm_reference.py) for predictor weights and geometries
beyond the reference's srand(1) draw, on every kernel path: the default (rank-one candidate pass with its exact-pass
fallback, or the tiled kernel for k >= 15), SPECKV_SCORE_EXACT=1 (rank-one kernel, exact logits) and =2 (tiled kernel).
Every run is compared with the reference, not with the other runs.

Bar, the same for every path:
  ids          identical to the reference's top-k by (logit, lower id), except permutations among logits within
               2 fp32 ulps (covers a one-ulp difference of h between the device's and the host's fp64 tanh)
  confidences  |conf - p| <= 1e-7 + 2^-22 p, p the fp64 softmax of the fp32 logits; conf <= 1, non-increasing,
               sum <= 1 + 1e-6
  addresses    va = (req << 32) | (layer << 16) | (i + 1)"""
import numpy as np
import pytest
import torch

from oracle.oracle import Port
from tests import lstm_reference as R

pytestmark = pytest.mark.gpu

from cxl_speckv_b200 import prefetch  # noqa: E402
from cxl_speckv_b200._lib import SpeckvError, lib  # noqa: E402

DEV = "cuda:0"
MODES = ("0", "1", "2")
BASE = (32000, 64, 128, 2, 16)   # vocab, emb_dim, hidden, layers, history_len of the reference's predictor


class _Predictors:
    """Weights by (family, geometry), generated once; the device holds the last one installed."""

    def __init__(self):
        self.weights, self.refs, self.loaded = {}, {}, None

    def install(self, family, vocab, emb_dim, hidden, layers, hist_len):
        key = (family, vocab, emb_dim, hidden)
        if key not in self.weights:
            self.weights[key] = Port.lstm_weights(1, vocab, emb_dim, hidden) if family == "srand" else \
                R.weights(family, vocab, emb_dim, hidden, seed=vocab + hidden)
        emb, wout = self.weights[key]
        if self.loaded != key + (layers, hist_len):
            prefetch.load_predictor(emb, wout, layers=layers, history_len=hist_len)
            self.loaded = key + (layers, hist_len)
        return emb, wout

    def reference(self, emb, wout, layers, wins, rows):
        """R.predict for the checked rows, top min(16, vocab), cached across modes and k."""
        key = (id(wout), layers, wins.tobytes(), rows.tobytes())
        if key not in self.refs:
            if len(self.refs) >= 6:
                self.refs.clear()
            self.refs[key] = R.predict(emb, wout, wins[rows], layers, min(16, wout.shape[0]))
        return self.refs[key]


@pytest.fixture(scope="module")
def preds():
    p = _Predictors()
    yield p
    emb, wout = Port.lstm_weights(1)
    prefetch.load_predictor(emb, wout, layers=2, history_len=16)


def _rows(batch):
    """Every sequence up to 64, a fixed stride sample (and the last one) above that."""
    if batch <= 64:
        return np.arange(batch)
    return np.unique(np.r_[np.arange(0, batch, batch // 48), batch - 1])


def _windows(vocab, batch, hist_len, seed):
    rng = np.random.default_rng(seed)
    w = rng.integers(0, vocab, (batch, hist_len))
    if batch > 2:
        w[1, : (hist_len + 1) // 2] = vocab + 7           # partly out of the vocabulary (embeds to zeros)
    return w


def _score_and_check(preds, emb, wout, layers, wins, k, mode, monkeypatch, layer_id=3, req_id=5):
    """One scoring call on the device, every checked row against the reference -> (ref tuple, max |conf - p|)."""
    monkeypatch.setenv("SPECKV_SCORE_EXACT", mode)
    toks = torch.from_numpy(wins.astype(np.int32)).to(DEV)
    ids, conf, va = prefetch.score(toks, k=k, layer_id=layer_id, req_id=req_id)
    ids, conf, va = ids.cpu().numpy(), conf.cpu().numpy().astype(np.float64), va.cpu().numpy().view(np.uint64)
    want_va = np.array([(req_id << 32) | (layer_id << 16) | (i + 1) for i in range(k)], dtype=np.uint64)
    assert (va == want_va).all(), f"mode {mode}: request addresses"
    assert (conf <= 1.0).all() and (np.diff(conf, axis=1) <= 0).all() and (conf.sum(axis=1) <= 1 + 1e-6).all(), \
        f"mode {mode}: confidences above 1, not sorted, or summing above 1 (max {conf.max()!r})"
    rows = _rows(len(wins))
    ref = preds.reference(emb, wout, layers, wins, rows)
    _, rid, _, x, p = ref
    errs = np.zeros(len(rows))
    bad_ids = []
    for n, b in enumerate(rows):
        if not R.ids_match(ids[b], rid[n][:k], x[n]):
            bad_ids.append((int(b), ids[b].tolist(), rid[n][:k].tolist()))
        pc = p[n][ids[b]]
        errs[n] = (np.abs(conf[b] - pc) - R.conf_tolerance(pc)).max()
    worst = max(float(np.abs(conf[b] - p[n][ids[b]]).max()) for n, b in enumerate(rows))
    assert not bad_ids, f"mode {mode} k {k}: top-k ids differ from the reference in {len(bad_ids)} rows, first {bad_ids[0]}"
    n = int(np.argmax(errs))
    assert (errs <= 0).all(), f"mode {mode} k {k}: max |conf - p64| = {worst:.3g} (row {rows[n]}: conf " \
        f"{conf[rows[n]].tolist()}, p {p[n][ids[rows[n]]].tolist()})"
    return ref, worst


# ---- weight families at the reference's geometry -----------------------------------------------------------------
FAMILIES = ("srand", "normal0.1", "normal1", "dominant", "permuted", "large", "signs")


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", FAMILIES)
def test_weight_families(preds, family, mode, monkeypatch):
    vocab, emb_dim, hidden, layers, hist_len = BASE
    emb, wout = preds.install(family, *BASE)
    wins = _windows(vocab, 40, hist_len, seed=101)
    wins[2] = vocab + 100                                  # wholly out of the vocabulary: h = 0
    if family == "signs":
        wins[3:20] = np.random.default_rng(5).integers(0, vocab // 2, (17, hist_len))              # h > 0
        wins[20:] = np.random.default_rng(6).integers(vocab - vocab // 2, vocab, (20, hist_len))  # h < 0
    for k in (4, 14, 16):
        (h, _, conf, x, _), _ = _score_and_check(preds, emb, wout, layers, wins, k, mode, monkeypatch)
    assert h[2] == 0.0
    if family == "signs":
        assert (h > 0).any() and (h < 0).any() and (h == 0).any()
    if family == "dominant":
        assert conf[:, 0].max() > 0.999
    if family == "large":
        assert np.abs(x).max() > 50.0


# ---- every k, on the reference's predictor and on a peaked one ---------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", ("srand", "normal1"))
def test_every_k(preds, family, mode, monkeypatch):
    vocab, emb_dim, hidden, layers, hist_len = BASE if family == "srand" else (5003, 200, 130, 2, 16)
    emb, wout = preds.install(family, vocab, emb_dim, hidden, layers, hist_len)
    wins = _windows(vocab, 9, hist_len, seed=202)
    for k in range(1, 17):
        _score_and_check(preds, emb, wout, layers, wins, k, mode, monkeypatch)


# ---- batches on both sides of the tiled kernel's geometry thresholds ---------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("batch", (1, 7, 8, 9, 32, 33, 255, 256, 257, 1000, 4096))
def test_batches(preds, batch, mode, monkeypatch):
    vocab, emb_dim, hidden, layers, hist_len = BASE
    emb, wout = preds.install("normal1", *BASE)
    wins = _windows(vocab, batch, hist_len, seed=batch)
    for k in (4, 8, 16):
        _score_and_check(preds, emb, wout, layers, wins, k, mode, monkeypatch)


# ---- geometries ---------------------------------------------------------------------------------------------------
# (id, vocab, emb_dim, hidden, layers, history_len)
GEOMETRIES = [
    ("base", *BASE),
    ("h130-e200", 5003, 200, 130, 2, 16),       # hidden not a multiple of 4 (4-byte staging, scalar tail), emb > hidden
    ("h300-e16", 5003, 16, 300, 2, 16),         # two row chunks in the rank-one re-scoring
    ("t1", 4001, 64, 128, 2, 1),
    ("t33", 4001, 64, 128, 2, 33),              # windows over 32 tokens: two rounds of the hidden-state warp
    ("t40", 4001, 64, 128, 2, 40),
    ("t48", 4001, 64, 128, 2, 48),              # 4 warps x 48 x 64 floats = 48 KiB of staging, the last that fits
    ("t49", 4001, 64, 128, 2, 49),              # one thread per sequence
    ("L0", 4001, 64, 128, 0, 16),
    ("L1", 4001, 64, 128, 1, 16),
    ("L3", 4001, 64, 128, 3, 16),
    ("v1", 1, 64, 128, 2, 16),
    ("v5", 5, 64, 128, 2, 16),
    ("v17", 17, 64, 128, 2, 16),
    ("v100003", 100003, 64, 128, 2, 16),        # prime
    ("h448", 2003, 64, 448, 2, 16),             # the widest tile of 64 rows that fits 227 KB
    ("h450", 2003, 64, 450, 2, 16),             # rows padded to 452 words: 64 rows no longer fit
    ("h904", 2003, 64, 904, 2, 16),             # the widest tile of 32 rows that fits
    ("h1024", 2003, 64, 1024, 2, 16),           # no tile fits
    ("h4096", 2003, 64, 4096, 2, 16),           # the widest predictor that loads
]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("geom", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_geometries(preds, geom, mode, monkeypatch):
    _, vocab, emb_dim, hidden, layers, hist_len = geom
    emb, wout = preds.install("normal0.5", vocab, emb_dim, hidden, layers, hist_len)
    ks = sorted({min(k, vocab) for k in (1, 4, 15, 16)})
    for batch in (8, 40):                              # the tiled kernel's small-batch (64-row) and wide-batch tiles
        wins = _windows(vocab, batch, hist_len, seed=batch + hidden)
        for k in ks:
            (h, ids, _, _, _), _ = _score_and_check(preds, emb, wout, layers, wins, k, mode, monkeypatch)
        if layers == 0:
            assert not h.any() and (ids == np.arange(ids.shape[1])).all()


# ---- request emission: residency filter and compaction over several 256-sequence scan chunks ----------------------
def _page_table(req):
    """One speckv_page_t: the page at (req << 32), resident in L1."""
    rec = np.zeros(1, dtype=[("virt", "<u8"), ("phys", "<u8"), ("size", "<u4"), ("flags", "<u4")])
    rec["virt"], rec["phys"], rec["size"], rec["flags"] = req << 32, 0x4000000000, 4096, 1
    return torch.from_numpy(rec.view(np.uint8).copy()).to(DEV)


@pytest.mark.parametrize("kept", ("random", "none", "all"))
def test_emit_compaction(preds, kept, monkeypatch):
    """batch 1000, k 4, per-sequence request ids: a sequence with id R addresses the resident page at va_base = R << 32
    and is filtered, one with id R - 1 lies below the table and is kept.  The surviving records follow in sequence
    order, field by field equal to the same call's predictions; the outstanding queue holds the last 16."""
    monkeypatch.delenv("SPECKV_SCORE_EXACT", raising=False)
    vocab, emb_dim, hidden, layers, hist_len = BASE
    preds.install("normal1", *BASE)
    B, k, R_ID, ts = 1000, 4, 9, 77
    keep = {"random": np.random.default_rng(13).random(B) < 0.5, "none": np.zeros(B, bool), "all": np.ones(B, bool)}[kept]
    rid = np.where(keep, R_ID - 1, R_ID).astype(np.int32)
    toks = torch.from_numpy(_windows(vocab, B, hist_len, seed=303).astype(np.int32)).to(DEV)
    _, q_before = prefetch.outstanding()
    table, ids, conf = prefetch.emit(toks, k=k, layer_id=0, req_ids=torch.from_numpy(rid).to(DEV),
                                     page_table=_page_table(R_ID), va_base=R_ID << 32, timestamp=ts, want_predictions=True)
    n, va, lay, tok, cf, tss = prefetch.unpack_table(table)
    ids, conf = ids.cpu().numpy().view(np.uint32), conf.cpu().numpy()
    seqs = np.nonzero(keep)[0]
    assert n == k * seqs.size
    raw = table.cpu().numpy()
    assert int(raw[0, :8].view(np.uint64)[0]) == n and int(raw[0, 12:16].view(np.uint32)[0]) == B * k   # header
    want_va = ((rid[seqs].astype(np.uint64)[:, None] << np.uint64(32)) | np.arange(1, k + 1, dtype=np.uint64)).ravel()
    assert np.array_equal(va, want_va)
    assert (lay == 0).all() and (tss == ts).all()
    assert np.array_equal(tok, ids[seqs].ravel())
    assert np.array_equal(cf.view(np.uint32), conf[seqs].ravel().view(np.uint32))
    _, queue = prefetch.outstanding()
    if n >= 16:
        assert [q["virtual_addr"] for q in queue] == va[-16:].tolist()
        assert [q["predicted_token_id"] for q in queue] == tok[-16:].tolist()
        found, _ = prefetch.outstanding(va[-16:].tolist() + [int(R_ID) << 32 | 1])
        assert found[:16].all() and not found[16]          # a filtered request never enters the queue
    else:
        assert n == 0 and queue == q_before                # nothing emitted: the queue is untouched


# ---- arguments ----------------------------------------------------------------------------------------------------
def test_rejected_arguments(preds, monkeypatch):
    monkeypatch.delenv("SPECKV_SCORE_EXACT", raising=False)
    emb, wout = preds.install("normal1", 17, 64, 128, 2, 16)
    toks = torch.zeros((3, 16), dtype=torch.int32, device=DEV)
    for k in (0, 17, 18):
        with pytest.raises(SpeckvError):
            prefetch.score(toks, k=k)
    prefetch.score(toks, k=16)
    emb5, wout5 = emb[:5].copy(), wout[:5].copy()
    prefetch.load_predictor(emb5, wout5, layers=2, history_len=16)
    preds.loaded = None
    with pytest.raises(SpeckvError):
        prefetch.score(toks, k=6)                          # k > vocab
    prefetch.score(toks, k=5)
    with pytest.raises(SpeckvError):
        prefetch.load_predictor(emb5, np.zeros((5, 4097), np.float32), layers=2, history_len=16)
    lib().speckv_ext_predictor_unload()
    with pytest.raises(SpeckvError):
        prefetch.score(toks, k=4)                          # nothing loaded
    emb, wout = preds.install("normal1", 17, 64, 128, 2, 16)
    prefetch.score(toks, k=4)
