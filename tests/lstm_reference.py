"""fp64 reference of the prefetch predictor (test infrastructure only, plain numpy).

The predictor (lstm_predictor.cpp:116-188, restated in oracle/speckv_oracle.c) carries one value h in every hidden
unit; the kernels reproduce its fp32 arithmetic step for step:
    g_t = sum_{j < min(emb_dim, hidden)} fl(e_t[j] * 0.1f)        sequential fp32; out-of-vocabulary tokens embed to 0
    c   = fl(fl(0.5 c) + fl(0.5 fl32(tanh(g_t))))                  once per layer and token, in token order
    h   = fl(0.5 fl32(tanh(c)))                                    0 when layers or history_len is 0
    x_v = sum_j fl(h * W[v][j])                                    sequential fp32 over j
tanh is taken in fp64 and rounded once (the kernels do the same; glibc's tanhf is within 1 ulp of it).  Everything
after the logits -- softmax and the order -- is fp64 here: the confidences a kernel reports are compared with the exact
softmax of the fp32 logits, not with another fp32 evaluation of it."""
from __future__ import annotations

import numpy as np

f32 = np.float32


def hidden_values(emb: np.ndarray, windows: np.ndarray, hidden: int, layers: int) -> np.ndarray:
    """h for each window (rows of `windows`, history_len tokens each) -> float32 [batch]."""
    emb = np.asarray(emb, dtype=f32)
    windows = np.asarray(windows, dtype=np.int64).reshape(len(windows), -1)
    vocab, emb_dim = emb.shape
    batch, hist_len = windows.shape
    if layers == 0 or hist_len == 0:
        return np.zeros(batch, dtype=f32)
    inside = (windows >= 0) & (windows < vocab)
    rows = np.where(inside, windows, 0)
    g = np.zeros((batch, hist_len), dtype=f32)
    for j in range(min(emb_dim, hidden)):
        e = np.where(inside, emb[rows, j], f32(0.0))
        g = (g + (e * f32(0.1)).astype(f32)).astype(f32)
    tg = np.tanh(g.astype(np.float64)).astype(f32)
    half = f32(0.5)
    c = np.zeros(batch, dtype=f32)
    for t in range(hist_len):
        a = (half * tg[:, t]).astype(f32)
        for _ in range(layers):
            c = ((half * c).astype(f32) + a).astype(f32)
    return (half * np.tanh(c.astype(np.float64)).astype(f32)).astype(f32)


def logits(wout: np.ndarray, h: np.ndarray) -> np.ndarray:
    """Sequential fp32 sums fl(h * W[v][j]) over j for each h -> float32 [len(h), vocab]."""
    w = np.asarray(wout, dtype=f32)
    h = np.asarray(h, dtype=f32).reshape(-1, 1)
    x = np.zeros((h.shape[0], w.shape[0]), dtype=f32)
    for j in range(w.shape[1]):
        x = (x + (h * w[:, j][None, :]).astype(f32)).astype(f32)
    return x


def softmax64(x: np.ndarray) -> np.ndarray:
    xd = np.asarray(x, dtype=np.float64)
    p = np.exp(xd - xd.max(axis=-1, keepdims=True))
    return p / p.sum(axis=-1, keepdims=True)


def topk(x: np.ndarray, k: int) -> np.ndarray:
    """The k first ids of each row by (logit descending, id ascending)."""
    x = np.atleast_2d(x)
    ids = np.arange(x.shape[1])
    return np.stack([np.lexsort((ids, -row.astype(np.float64)))[:k] for row in x])


def predict(emb, wout, windows, layers: int, k: int):
    """-> (h [batch], ids [batch, k], conf64 [batch, k], logits [batch, vocab], p64 [batch, vocab])."""
    wout = np.asarray(wout, dtype=f32)
    h = hidden_values(emb, windows, wout.shape[1], layers)
    hu, inv = np.unique(h, return_inverse=True)   # the logits depend on h alone
    xu = logits(wout, hu)
    x, p = xu[inv], softmax64(xu)[inv]
    ids = topk(x, k)
    return h, ids, np.take_along_axis(p, ids, axis=1), x, p


def weights(family: str, vocab: int, emb_dim: int, hidden: int, seed: int = 0):
    """Predictor weights beyond the reference's near-uniform srand(1) draw (whose confidences are all ~1/vocab):
      normal<s>   embedding N(0, 1), W_out N(0, s): peaked softmaxes, top confidences up to ~0.5
      dominant    normal1 plus 3 on every element of one row: that row's confidence is ~1 when h > 0
      permuted    N(0, 0.1) plus groups of 3, 7, 15 and 40 copies of one row, its elements permuted: within a group
                  the row sums (the rank-one order) tie, the exact sequential fp32 sums differ in the last bits
      large       W_out N(0, 8): logits around +-80
      signs       embedding +0.5 on the lower half of the vocabulary, -0.5 on the upper: windows from either half
                  give h > 0 or h < 0, out-of-vocabulary windows h = 0; W_out N(0, 0.5)
    -> (emb float32 [vocab, emb_dim], wout float32 [vocab, hidden])."""
    rng = np.random.default_rng(seed)
    emb = rng.standard_normal((vocab, emb_dim)).astype(f32)
    if family.startswith("normal"):
        return emb, (rng.standard_normal((vocab, hidden)) * float(family[6:])).astype(f32)
    if family == "dominant":
        wout = rng.standard_normal((vocab, hidden)).astype(f32)
        wout[vocab // 3] += f32(3.0)
        return emb, wout
    if family == "permuted":
        wout = (rng.standard_normal((vocab, hidden)) * 0.1).astype(f32)
        rows = rng.permutation(vocab)
        at = 0
        for n, base in ((3, 0.6), (7, 0.5), (15, 0.4), (40, -0.6)):   # the 40 lead the reverse order (h < 0)
            row = (rng.standard_normal(hidden) * 0.3 + base).astype(f32)
            for r in rows[at:at + n]:
                wout[r] = rng.permutation(row)
            at += n
        return emb, wout
    if family == "large":
        return emb, (rng.standard_normal((vocab, hidden)) * 8.0).astype(f32)
    if family == "signs":
        emb = np.full((vocab, emb_dim), 0.5, dtype=f32)
        emb[vocab // 2:] = -0.5
        return emb, (rng.standard_normal((vocab, hidden)) * 0.5).astype(f32)
    raise ValueError(family)


def conf_tolerance(p):
    """|conf - p| allowed for a kernel's fp32 confidence: 1e-7 absolute (SURVEY.md section 8a A11) plus 2^-22 relative,
    about one ulp of 1.0 for confidences near 1."""
    return 1e-7 + 2.0 ** -22 * np.asarray(p, dtype=np.float64)


def ids_match(got, want, x, ulps: int = 2) -> bool:
    """got[i] is a distinct id whose reference logit lies within `ulps` fp32 ulps of the i-th best reference logit
    x[want[i]]: identical ids, except permutations inside groups of near-equal logits (the slack covers a one-ulp
    difference of h between the device's and the host's fp64 tanh)."""
    got = [int(v) for v in got]
    x = np.asarray(x, dtype=f32)
    if len(set(got)) != len(got) or any(v < 0 or v >= x.size for v in got):
        return False
    for g, w in zip(got, want):
        if g == int(w):
            continue
        a, b = x[g], x[int(w)]
        if abs(float(a) - float(b)) > ulps * float(np.spacing(np.abs(b))):
            return False
    return True
