"""CPU: the fp64 prefetch reference (tests/lstm_reference.py) against the C restatement of the reference's predictor
(oracle/speckv_oracle.c, LSTMPredictor::predict_top_k), over geometries and weight families the GPU tests use.

Each stage is pinned on its own: h within 2^-24 + 2 ulps (the restatement takes tanhf, the reference fp64 tanh rounded
once; a one-ulp difference of tanh(g_t), at most 2^-24, moves c = 0.5 c + 0.5 tanh(g_t) by at most that much and h by
half of it, plus the rounding of tanh(c)), then the logits, softmax and order from the
restatement's own h: same top-k ids up to permutations inside exact fp32 confidence ties, and confidences within the
kernels' bar plus the restatement's fp32 summation error (a recursive sum over the vocabulary: gamma_vocab relative)."""
import numpy as np
import pytest

from oracle import oracle
from oracle.oracle import Port
from tests import lstm_reference as R
from tests.test_oracle_golden import same_topk

U = 2.0 ** -24

# (name, family, vocab, emb_dim, hidden, layers, hist_len, k)
CASES = [
    ("srand", "srand", 32000, 64, 128, 2, 16, 8),
    ("normal1", "normal1", 8000, 64, 128, 2, 16, 8),
    ("normal0.5-h512", "normal0.5", 3001, 64, 512, 2, 16, 16),
    ("dominant-h130-e200-L3-t33", "dominant", 3000, 200, 130, 3, 33, 8),
    ("permuted-h300-e16-L1-t49", "permuted", 5003, 16, 300, 1, 49, 16),
    ("large-t1", "large", 2003, 64, 128, 2, 1, 4),
    ("signs-t40", "signs", 4001, 64, 128, 2, 40, 4),
    ("layers0-v17", "normal1", 17, 64, 128, 0, 16, 16),
]


@pytest.fixture(scope="module", autouse=True)
def _port():
    oracle.build(ref=False)


def _weights(family, vocab, emb_dim, hidden):
    if family == "srand":
        return Port.lstm_weights(1, vocab, emb_dim, hidden)
    return R.weights(family, vocab, emb_dim, hidden, seed=3)


def _h_close(a, b) -> bool:
    return abs(float(a) - float(b)) <= U + 2.0 * float(np.spacing(np.abs(np.float32(b))))


@pytest.mark.parametrize("name,family,vocab,emb_dim,hidden,layers,hist_len,k", CASES, ids=[c[0] for c in CASES])
def test_reference_matches_restatement(name, family, vocab, emb_dim, hidden, layers, hist_len, k):
    emb, wout = _weights(family, vocab, emb_dim, hidden)
    rng = np.random.default_rng(17)
    wins = rng.integers(0, vocab, (8, hist_len))
    wins[1, : hist_len // 2] = vocab + 5                  # partly out of the vocabulary: those tokens embed to zeros
    wins[2, :] = vocab + 1000                             # wholly out of it: h = 0
    if family == "signs":
        wins[3:5] = rng.integers(0, vocab // 2, (2, hist_len))            # h > 0
        wins[5:7] = rng.integers(vocab - vocab // 2, vocab, (2, hist_len))   # h < 0
    h, ids, conf, x, p = R.predict(emb, wout, wins, layers, k)
    assert h[2] == 0.0
    if layers == 0:
        assert not h.any() and (conf == 1.0 / vocab).all() and (ids == np.arange(k)).all()
    if family == "signs":
        assert (h[3:5] > 0).all() and (h[5:7] < 0).all()
    worst = 0.0
    for b in range(len(wins)):
        oi, oc, oh = Port.lstm_predict(emb, wout, wins[b].astype(np.uint32), k=k, layers=layers, hist_len=hist_len)
        assert (oh == oh[0]).all()                        # every hidden unit carries the same value
        assert _h_close(oh[0], h[b]), (b, oh[0], h[b])
        # the rest of the pipeline from the restatement's own h
        xo = R.logits(wout, oh[:1])[0]
        po = R.softmax64(xo)
        ro = R.topk(xo, k)[0]
        assert same_topk(ro.tolist(), oi.tolist(), oc.view(np.uint32).tolist()), (b, ro, oi)
        err = np.abs(oc.astype(np.float64) - po[oi])
        bar = R.conf_tolerance(po[oi]) + (0.0 if family == "srand" else vocab * U * po[oi])
        assert (err <= bar).all(), (b, err.max())
        worst = max(worst, float(err.max()))
        # where h agrees bit for bit, so does everything downstream
        if oh[0] == h[b]:
            assert np.array_equal(xo, x[b]) and np.array_equal(ro, ids[b])
    print(name, "max |conf_restatement - p64| =", worst)


def test_order_and_tie_helpers():
    """topk breaks logit ties by the lower id; ids_match accepts permutations within 2 ulps and nothing wider."""
    x = np.array([1.0, 3.0, 3.0, 2.0, np.nextafter(np.float32(2.0), np.float32(0.0))], dtype=np.float32)
    assert R.topk(x, 4)[0].tolist() == [1, 2, 3, 4]
    assert R.ids_match([2, 1, 4, 3], [1, 2, 3, 4], x)
    assert not R.ids_match([1, 2, 3, 0], [1, 2, 3, 4], x)
    assert not R.ids_match([1, 1, 3, 4], [1, 2, 3, 4], x)
    p = R.softmax64(np.array([0.0, np.log(3.0)]))
    assert np.allclose(p, [0.25, 0.75], rtol=0, atol=1e-15)
