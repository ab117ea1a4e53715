"""The tensor-core prefilters at their error bounds.

Every fast path of the library decides with an approximate tcgen05 contraction and keeps only the decisions that clear
a proven margin; the rest go to an exact fp32 arbiter.  Random test data almost never puts a decision near such a
margin, so a bound that is wrong by a small factor passes the other parity tests.  The generators below construct
inputs whose decisions sit at chosen distances from the bound, return the float64 quantities they produced (so a test
can assert it really covered the boundary), and the tests hold the kernels to bars that would fail if the bound did
not hold:
  * codes (RQ encode, k-means assignment, PQ): no hard mismatch against the float64 arbiter, the fix-up ran, and the
    fused / delta k-means steps assign exactly like the plain step;
  * power-of-two scale invariance: inputs scaled by 2^s give bit-identical codes and exactly 2^s-scaled scores;
  * top-k: ids are the float64 top-k up to pairs whose float64 scores lie within the rigorous fp32 dot-product bound
    gamma_d * sum |q_i d_i|, and every returned score is within that bound of float64;
  * mixed-norm query batches: a query 2^-30 ... 2^-36 times smaller than the rest of its batch (its fp16 image
    underflows) gets the answer of the unscaled query.

The generators need no GPU; tests/test_prefilter_generators.py checks them on the CPU.
"""
import numpy as np
import pytest
import torch

from oracle import oracle

TIE = oracle.TIE_EPS_DEFAULT
DELTAS_CODES = 2.0 ** np.linspace(-24, -8, 17)   # target relative gaps of the code generators
DELTAS_TOPK = 2.0 ** np.linspace(-24, -6, 19)    # target relative distances from the k-th score


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------
def rq_path64(X, cb, metric="l2"):
    """float64 decisions along the fp32 residual path (sequential fp32 subtraction, as oracle.classify_code_mismatches).
    -> codes [n,M] (first best wins), rel [n,M] = top-2 gap relative to the classifier's scale, runner-up [n,M]."""
    X = np.asarray(X, np.float32)
    cb = np.asarray(cb, np.float32)
    n, M = X.shape[0], cb.shape[0]
    codes = np.empty((n, M), np.int32)
    second = np.empty((n, M), np.int32)
    rel = np.empty((n, M), np.float64)
    res = X.copy()
    rows = np.arange(n)
    for j in range(M):
        r = res.astype(np.float64)
        c = cb[j].astype(np.float64)
        if metric == "l2":
            score = -((r * r).sum(1)[:, None] - 2.0 * r @ c.T + (c * c).sum(1)[None])
        else:
            score = r @ c.T
        a = np.argmax(score, 1)
        masked = score.copy()
        masked[rows, a] = -np.inf
        b = np.argmax(masked, 1)
        sa, sb = score[rows, a], score[rows, b]
        if metric == "l2":
            scale = np.maximum(-sa, -sb)
        else:
            cn = np.linalg.norm(c, axis=1)
            scale = np.maximum(np.maximum(np.abs(sa), np.abs(sb)), np.linalg.norm(r, axis=1) * np.maximum(cn[a], cn[b]))
        rel[:, j] = (sa - sb) / np.maximum(scale, 1e-300)
        codes[:, j], second[:, j] = a, b
        res = res - cb[j][a]
    return codes, rel, second


def _residual_at(X, cb, codes, j):
    res = np.asarray(X, np.float32).copy()
    for m in range(j):
        res = res - cb[m][codes[:, m]]
    return res.astype(np.float64)


def rq_gap_rows(X, cb, rs, metric="l2", levels=None, deltas=DELTAS_CODES, keep_eps=64 * TIE):
    """Move each row along c_b - c_a (L2; c_a - c_b for IP) of its best / runner-up centroid at one level so that the
    top-2 gap there becomes delta * scale, delta log-spaced over `deltas`.  The level of row i is levels[i % len] (all
    levels by default).  Rows whose earlier levels no longer clear `keep_eps` are dropped.
    -> (X' fp32, level [n'], target delta [n'], codes64 [n',M], rel [n',M])"""
    X = np.asarray(X, np.float32)
    cb = np.asarray(cb, np.float32)
    M = cb.shape[0]
    levels = list(range(M)) if levels is None else list(levels)
    n = X.shape[0]
    lev = np.array([levels[i % len(levels)] for i in range(n)])
    dl = np.asarray(deltas)[rs.permutation(n) % len(deltas)]
    codes, _, second = rq_path64(X, cb, metric)
    out = X.astype(np.float64).copy()
    for j in set(lev.tolist()):
        sel = np.nonzero(lev == j)[0]
        r = _residual_at(X[sel], cb, codes[sel], j)
        ca = cb[j][codes[sel, j]].astype(np.float64)
        cb_ = cb[j][second[sel, j]].astype(np.float64)
        if metric == "l2":
            dA, dB = ((r - ca) ** 2).sum(1), ((r - cb_) ** 2).sum(1)
            u = cb_ - ca
            # gap(t) = dB - dA - 2 t |u|^2 for r + t u; aim at delta * max(dA, dB) (dB moves little: solve once more)
            t = (dB - dA - dl[sel] * dB) / (2.0 * (u * u).sum(1))
            r2 = r + t[:, None] * u
            dA2, dB2 = ((r2 - ca) ** 2).sum(1), ((r2 - cb_) ** 2).sum(1)
            t = t + (dB2 - dA2 - dl[sel] * np.maximum(dA2, dB2)) / (2.0 * (u * u).sum(1))
        else:
            v = ca - cb_
            sA, sB = (r * ca).sum(1), (r * cb_).sum(1)
            scale = np.maximum(np.linalg.norm(r, axis=1) * np.maximum(np.linalg.norm(ca, axis=1), np.linalg.norm(cb_, axis=1)),
                               np.maximum(np.abs(sA), np.abs(sB)))
            t = (dl[sel] * scale - (sA - sB)) / (v * v).sum(1)  # gap(t) = sA - sB + t |v|^2 for r + t v
            u = v
        out[sel] += t[:, None] * u
    Xn = out.astype(np.float32)
    codes2, rel2, _ = rq_path64(Xn, cb, metric)
    keep = np.ones(n, bool)
    for i in range(n):
        if lev[i] > 0 and (rel2[i, : lev[i]] < keep_eps).any():
            keep[i] = False
    return Xn[keep], lev[keep], dl[keep], codes2[keep], rel2[keep]


def decided_gaps(rel, lev):
    """relative gap of every row at its constructed level"""
    return rel[np.arange(len(lev)), lev]


def pq_path64(X, cb, metric="l2"):
    """float64 best / runner-up per (row, sub-vector) and the gap relative to oracle.classify_pq_mismatches' scale."""
    M, K, ds = cb.shape
    n = X.shape[0]
    codes = np.empty((n, M), np.int32)
    second = np.empty((n, M), np.int32)
    rel = np.empty((n, M))
    rows = np.arange(n)
    for j in range(M):
        x = X[:, j * ds:(j + 1) * ds].astype(np.float64)
        c = cb[j].astype(np.float64)
        xx = (x * x).sum(1)
        if metric == "l2":
            score = -(xx[:, None] - 2.0 * x @ c.T + (c * c).sum(1)[None])
        else:
            score = x @ c.T
        a = np.argmax(score, 1)
        m2 = score.copy()
        m2[rows, a] = -np.inf
        b = np.argmax(m2, 1)
        sa, sb = score[rows, a], score[rows, b]
        if metric == "l2":
            scale = np.maximum(-sa, -sb) + xx
        else:
            ax = np.abs(x)
            scale = (ax * np.abs(c[a])).sum(1) + (ax * np.abs(c[b])).sum(1)
        rel[:, j] = (sa - sb) / np.maximum(scale, 1e-300)
        codes[:, j], second[:, j] = a, b
    return codes, rel, second


def pq_gap_rows(X, cb, rs, metric="l2", deltas=DELTAS_CODES):
    """Every (row, sub-vector) moved along its own best / runner-up direction to a gap of its own delta.
    -> (X' fp32, target delta [n,M], codes64 [n,M], rel [n,M])"""
    X = np.asarray(X, np.float32)
    M, K, ds = cb.shape
    n = X.shape[0]
    dl = np.asarray(deltas)[rs.randint(0, len(deltas), size=(n, M))]
    codes, _, second = pq_path64(X, cb, metric)
    out = X.astype(np.float64).copy()
    rows = np.arange(n)
    for j in range(M):
        x = out[:, j * ds:(j + 1) * ds]
        ca, cb_ = cb[j][codes[:, j]].astype(np.float64), cb[j][second[:, j]].astype(np.float64)
        if metric == "l2":
            u = cb_ - ca
            for _ in range(2):  # the scale moves with x: two Newton-like steps
                dA, dB = ((x - ca) ** 2).sum(1), ((x - cb_) ** 2).sum(1)
                scale = np.maximum(dA, dB) + (x * x).sum(1)
                x = x + ((dB - dA - dl[:, j] * scale) / (2.0 * (u * u).sum(1)))[:, None] * u
        else:
            v = ca - cb_
            for _ in range(2):
                scale = (np.abs(x) * np.abs(ca)).sum(1) + (np.abs(x) * np.abs(cb_)).sum(1)
                x = x + ((dl[:, j] * scale - ((x * ca).sum(1) - (x * cb_).sum(1))) / (v * v).sum(1))[:, None] * v
        out[:, j * ds:(j + 1) * ds] = x
    Xn = out.astype(np.float32)
    codes2, rel2, _ = pq_path64(Xn, cb, metric)
    return Xn, dl, codes2, rel2


def topk_boundary_docs(D, Q, k, rs, per_query=200, deltas=DELTAS_TOPK):
    """For each query move `per_query` documents along q so that their float64 scores sit at s_k +- delta |q| |d|
    (s_k = the query's k-th float64 score before the move, delta log-spaced over `deltas`, both signs).
    -> (D' fp32, rel [nq, per_query] = (score - s_k) / (|q||d|) achieved in float64, rows moved [nq, per_query])"""
    D = np.asarray(D, np.float32).copy()
    n = D.shape[0]
    nq = Q.shape[0]
    Q64 = Q.astype(np.float64)
    picks = rs.permutation(n)[: nq * per_query].reshape(nq, per_query)
    s_k = np.empty(nq)
    for q in range(nq):
        s = D.astype(np.float64) @ Q64[q]
        s_k[q] = np.sort(s)[-k]
    D64 = D.astype(np.float64)
    for q in range(nq):
        qq = Q64[q]
        qn2 = qq @ qq
        rows = picks[q]
        sgn = np.where(np.arange(per_query) % 2 == 0, 1.0, -1.0)
        dl = np.asarray(deltas)[(np.arange(per_query) // 2) % len(deltas)] * sgn
        d = D64[rows]
        for _ in range(2):  # |d| moves with d
            target = s_k[q] + dl * np.sqrt(qn2) * np.linalg.norm(d, axis=1)
            d = d + ((target - d @ qq) / qn2)[:, None] * qq[None]
        D64[rows] = d
    D2 = D64.astype(np.float32)
    rel = np.empty((nq, per_query))
    for q in range(nq):
        d = D2[picks[q]].astype(np.float64)
        rel[q] = (d @ Q64[q] - s_k[q]) / (np.linalg.norm(Q64[q]) * np.linalg.norm(d, axis=1))
    return D2, rel, picks


def adversarial_rounding_docs(n=20000, d=256, k=100, n_rivals=300, seed=0):
    """Documents whose fp16 rounding errors are as large as the bound allows and point the wrong way.
    With the query all ones and every element in [1, 2) the scales are 2^11 and the fp16 spacing of the scaled
    elements is 2.  The k true members hold odd-minus-2^-10 values (their images round DOWN by ~1 per element); the
    n_rivals rivals hold odd-plus-2^-10 values (rounded UP) and are 52 scaled units below the weakest members in
    exact arithmetic, far outside the fp32 bound.  Their approximate scores are ~460 units above those members, so the
    weakest members are only found with a margin of at least that much (the rigorous margin is ~1,560 units).
    -> (D fp32, q [1, d] fp32, member rows [k])"""
    rs = np.random.RandomState(seed)
    sd = 2048.0
    down, up = 1.0 - 2.0 ** -10, 1.0 + 2.0 ** -10
    D = (1.0 + 0.3 * rs.random_sample((n, d))).astype(np.float32)   # background, far below
    base = rs.randint(1100, 1900, size=d)
    rows = rs.permutation(n)[: k + n_rivals]
    members, rivals = rows[:k], rows[k:]
    weak = 10
    for j in range(k):
        m = base.copy()
        if j < weak:
            m[j] += 1              # the weakest members: exact scores base, base + 2 units, ...
        else:
            m += 1                 # the rest: 512 + 2 j units above
            m[j % d] += j
        D[members[j]] = ((2.0 * m + down) / sd).astype(np.float32)
    for i, r in enumerate(rivals):
        m = base.copy()
        m[rs.choice(d, 26, replace=False)] -= 1  # 52 units below the weakest member in exact arithmetic
        D[r] = ((2.0 * m + up) / sd).astype(np.float32)
    return D, np.ones((1, d), np.float32), members


def fp32_dot_bound(Q, D):
    """[nq, n] rigorous bound of any fp32 evaluation order of q.d: gamma_d * sum |q_i d_i|, gamma_d = d u / (1 - d u)"""
    d = Q.shape[1]
    u = 2.0 ** -24
    return (d * u / (1 - d * u)) * (np.abs(Q.astype(np.float64)) @ np.abs(D.astype(np.float64)).T)


def check_topk_float64(scores, ids, Q, D, k, allowed=None):
    """Ids are the float64 top-k up to pairs within the fp32 bound; scores within the bound of float64.
    At rank p the returned document g and the float64 document r satisfy |s(g) - s(r)| <= b(g) + max_U b, U = returned
    ids + float64 top-k (the p-th order statistics of two score vectors differ by at most the largest error on U)."""
    Q64, D64 = Q.astype(np.float64), D.astype(np.float64)
    S = Q64 @ D64.T
    B = fp32_dot_bound(Q, D)
    if allowed is not None:  # [nq, n] bool: the documents a query may return (its candidates)
        S = np.where(allowed, S, -np.inf)
    for q in range(Q.shape[0]):
        ref = np.argsort(-S[q], kind="stable")[:k]
        got = np.asarray(ids[q])
        assert (got >= 0).all() and len(set(got.tolist())) == k, f"query {q}: padded or repeated ids"
        err = np.abs(np.asarray(scores[q], np.float64) - S[q, got])
        bad = np.nonzero(err > B[q, got])[0]
        assert not len(bad), f"query {q}: score of rank {bad[0]} off float64 by {err[bad[0]]:.3e} > {B[q, got[bad[0]]]:.3e}"
        bmax = B[q, np.union1d(ref, got)].max()
        diff = np.nonzero(got != ref)[0]
        for p in diff:
            gap = abs(S[q, got[p]] - S[q, ref[p]])
            assert gap <= B[q, got[p]] + bmax, (f"query {q} rank {p}: returned doc {got[p]} vs float64 doc {ref[p]}, "
                                                f"float64 gap {gap:.3e} beyond the fp32 bound {B[q, got[p]] + bmax:.3e}")


# ---------------------------------------------------------------------------------------------------------------------
# input sets
# ---------------------------------------------------------------------------------------------------------------------
def reference_like_codebook(X, M, K, rs):
    """level means of random subsets of the residual (as in test_gpu_rq_encode.test_larger_random_against_oracle)"""
    n, d = X.shape
    cb = np.empty((M, K, d), np.float32)
    res = X.copy()
    for j in range(M):
        lab = rs.randint(0, K, size=n)
        for k in range(K):
            cb[j, k] = res[lab == k][:400].mean(0)
        res = res - cb[j][oracle.rq_encode(res, cb[j:j + 1], batch_size=1024)[:, 0]]
    return cb


def rq_boundary_set(regime, seed=0):
    """-> (X', codebook, metric, level [n'], codes64, rel) for one regime of the issue's list:
    gauss / gauss_ip: N(0,1) rows, reference-like codebook; offset: mu + noise with |mu| = 10 |noise|, level-0 centroids
    share mu; mixed_norms: IP decisions at level 0 on rows scaled by 2^-20 ... 2^10 (the rows of the 2,048-row scale
    sample keep scale 1, so the largest rows overflow the fp16 range and the smallest underflow it);
    clustered_M{M}_K{K}: clustered rows, every level moved."""
    rs = np.random.RandomState(seed)
    d = 256
    if regime.startswith("clustered"):
        M, K = (int(v[1:]) for v in regime.split("_")[1:])
        n = 6000
        centers = rs.standard_normal((K, d)).astype(np.float32)
        X = (centers[rs.randint(0, K, n)] + 0.7 * rs.standard_normal((n, d))).astype(np.float32)
        cb = np.empty((M, K, d), np.float32)
        res = X.copy()
        for j in range(M):
            cb[j] = res[rs.choice(n, K, replace=False)] * (0.9 if j == 0 else 0.5)
            res = res - cb[j][oracle.rq_encode(res, cb[j:j + 1], batch_size=1024)[:, 0]]
        Xn, lev, _, c64, rel = rq_gap_rows(X, cb, rs, "l2")
        return Xn, cb, "l2", lev, c64, rel
    n, M, K = 8000, 4, 32
    X = rs.standard_normal((n, d)).astype(np.float32)
    if regime == "offset":
        mu = (10.0 * rs.standard_normal(d)).astype(np.float32)
        noise = X
        cb = reference_like_codebook(noise, M, K, rs)
        cb[0] += mu
        X = (mu + noise).astype(np.float32)
        Xn, lev, _, c64, rel = rq_gap_rows(X, cb, rs, "l2")
        return Xn, cb, "l2", lev, c64, rel
    cb = reference_like_codebook(X, M, K, rs)
    if regime == "mixed_norms":
        Xn, lev, _, _, _ = rq_gap_rows(X, cb, rs, "ip", levels=[0])
        e = rs.randint(-20, 11, size=len(Xn))
        e[:: max(len(Xn) // 2048, 1)] = 0  # the scale sample
        Xn = (Xn * np.ldexp(1.0, e)[:, None]).astype(np.float32)  # powers of two: exact
        c64, rel, _ = rq_path64(Xn, cb, "ip")
        return Xn, cb, "ip", lev, c64, rel
    metric = "ip" if regime == "gauss_ip" else "l2"
    Xn, lev, _, c64, rel = rq_gap_rows(X, cb, rs, metric)
    return Xn, cb, metric, lev, c64, rel


def assert_boundary_coverage(gaps, near_frac=0.2, below_frac=0.05):
    """the generator really put decisions at the bound: a share in [tie_eps, 64 tie_eps], some in [2^-24, tie_eps)"""
    near = np.mean((gaps >= TIE) & (gaps <= 64 * TIE))
    below = np.mean((gaps >= 2.0 ** -24) & (gaps < TIE))
    assert near >= near_frac and below >= below_frac, f"generator drifted off the boundary: {near:.3f} near, {below:.3f} below"


# clustered shapes: the tensor path's shared-memory budget takes M K <= 128 at d = 256
RQ_REGIMES = ["gauss", "gauss_ip", "offset", "mixed_norms", "clustered_M1_K128", "clustered_M2_K64", "clustered_M3_K32",
              "clustered_M4_K32"]


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _ctx():
    import mevi_b200

    return mevi_b200.get_context(0)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda(0)


def _rq_modes(c, d, M, K, metric):
    from gpu_util import tensor_modes

    modes = tensor_modes(c, d, M, K, metric)
    assert "tensor" in modes, f"the tensor path must take d={d} M={M} K={K} {metric}"
    return modes + ["auto"]


@pytest.mark.gpu
@pytest.mark.parametrize("regime", RQ_REGIMES)
def test_rq_codes_on_the_bound(regime):
    X, cb, metric, lev, c64, rel = rq_boundary_set(regime)
    assert_boundary_coverage(decided_gaps(rel, lev), near_frac=0.15 if regime == "mixed_norms" else 0.2)
    c = _ctx()
    clear = (rel > TIE).all(1)  # every decision of the row outside the tie window
    for mode in _rq_modes(c, X.shape[1], cb.shape[0], cb.shape[1], metric):
        codes, stats = c.rq_encode(_dev(X), _dev(cb), metric=metric, mode=mode, return_stats=True)
        codes = codes.cpu().numpy()
        rep = oracle.classify_code_mismatches(X, cb, c64, codes, dist_mode=metric)
        assert rep["n_hard"] == 0, f"{mode}: {rep['n_hard']} hard mismatches, rows {rep['hard_rows'][:8]}"
        assert np.array_equal(codes[clear], c64[clear]), f"{mode}: {(codes[clear] != c64[clear]).any(1).sum()} clear rows differ"
        if mode == "tensor":
            assert int(stats[0]) > 0, "no row was sent to the exact kernel"


@pytest.mark.gpu
def test_kmeans_assignment_on_the_bound():
    """mevi_kmeans_step (tensor / auto), _fused and _delta on rows whose nearest / second-nearest gap sits at the bound."""
    rs = np.random.RandomState(5)
    n, d, K = 8000, 256, 32
    centers = rs.standard_normal((K, d)).astype(np.float32)
    X = (centers[rs.randint(0, K, n)] + 0.7 * rs.standard_normal((n, d))).astype(np.float32)
    C = X[rs.choice(n, K, replace=False)].copy()
    Xn, lev, _, c64, rel = rq_gap_rows(X, C[None], rs, "l2")
    assert_boundary_coverage(rel[:, 0])
    c = _ctx()
    Xd, Cd = _dev(Xn), _dev(C)
    n = len(Xn)
    got = {}
    for mode in ("tensor", "auto", "exact"):
        buf = torch.empty(K * d + K, device="cuda:0")
        a = torch.empty(n, dtype=torch.int32, device="cuda:0")
        c.kmeans_step(Xd, Cd, buf, assign=a, mode=mode)
        got[mode] = (a, buf)
        rep = oracle.classify_code_mismatches(Xn, C[None], c64, a.cpu().numpy()[:, None])
        assert rep["n_hard"] == 0, f"{mode}: {rep['n_hard']} hard mismatches"
    want, buf = got["tensor"]
    prev = got["exact"][0]  # any previous assignment will do; its sums come from the plain step
    cur = torch.empty(n, dtype=torch.int32, device="cuda:0")
    sums_prev = torch.empty(K * d + K, device="cuda:0")
    c.kmeans_step_fused(Xd, Cd, prev, cur, sums_prev)
    assert torch.equal(cur, want), f"fused: {(cur != want).sum().item()} assignments differ from mevi_kmeans_step"
    master = got["exact"][1].double()
    cur2 = torch.empty(n, dtype=torch.int32, device="cuda:0")
    buf2 = torch.empty(K * d + K, device="cuda:0")
    c.kmeans_step_delta(Xd, Cd, prev, cur2, master, buf2, mode="tensor")
    c.check()
    assert torch.equal(cur2, want), f"delta: {(cur2 != want).sum().item()} assignments differ from mevi_kmeans_step"


@pytest.mark.gpu
@pytest.mark.parametrize("M,K,ds,metric", [(4, 32, 64, "l2"), (4, 32, 64, "ip"), (32, 256, 24, "l2"), (24, 256, 32, "l2"),
                                           (24, 256, 32, "ip")])
def test_pq_codes_on_the_bound(M, K, ds, metric):
    """block-padded route (M K <= 128, the RQ tensor kernel on a block-diagonal codebook) and the 256-centroid kernel"""
    rs = np.random.RandomState(M + K + ds)
    n = 6000
    X = rs.standard_normal((n, M * ds)).astype(np.float32)
    cb = (rs.standard_normal((M, K, ds)) * 0.7).astype(np.float32)
    Xn, _, c64, rel = pq_gap_rows(X, cb, rs, metric)
    assert_boundary_coverage(rel.ravel())
    codes = _ctx().pq_encode(_dev(Xn), _dev(cb), metric=metric).cpu().numpy()
    ties, real = oracle.classify_pq_mismatches(Xn, cb, codes, c64, metric)
    assert real == 0, f"{real} hard mismatches ({ties} ties)"
    clear = rel > TIE
    assert np.array_equal(codes[clear], c64[clear])


@pytest.mark.gpu
def test_codes_power_of_two_scale_invariance():
    """X and the codebook times 2^s: fp16 images, bound constants and the fp32 direct form all scale exactly, so the
    codes of every mode (and of both PQ routes) are bit-identical across s."""
    X, cb, metric, _, _, _ = rq_boundary_set("gauss", seed=3)
    c = _ctx()
    for mode in _rq_modes(c, X.shape[1], cb.shape[0], cb.shape[1], metric):
        base = None
        for s in (-20, 0, 20):
            f = np.float32(2.0 ** s)
            codes = c.rq_encode(_dev(X * f), _dev(cb * f), metric=metric, mode=mode).cpu().numpy()
            if base is None:
                base = codes
            assert np.array_equal(codes, base), f"{mode} s={s}: {(codes != base).any(1).sum()} rows differ"
    rs = np.random.RandomState(7)
    for M, K, ds in ((4, 32, 64), (24, 256, 32)):
        Xp = rs.standard_normal((6000, M * ds)).astype(np.float32)
        cbp = (rs.standard_normal((M, K, ds)) * 0.7).astype(np.float32)
        Xp, _, _, _ = pq_gap_rows(Xp, cbp, rs)
        outs = [c.pq_encode(_dev(Xp * np.float32(2.0 ** s)), _dev(cbp * np.float32(2.0 ** s))).cpu().numpy() for s in (-20, 0, 20)]
        assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[1], outs[2]), f"PQ {M}x{K}x{ds}"


def _flat_searches(D, mode):
    """the flat entry points: one-shot flat_ip_topk and a persistent FlatIndex -> list of (name, search(Q, k))"""
    from mevi_b200 import faiss_search

    c = _ctx()
    Dd = _dev(D)
    index = faiss_search.FlatIndex(D.shape[1], mode=mode)
    index.add(D)
    return [(f"flat_ip_topk[{mode}]", lambda Q, k: tuple(t.cpu().numpy() for t in c.flat_ip_topk(_dev(Q), Dd, k, mode=mode))),
            (f"FlatIndex[{mode}]", lambda Q, k: index.search(Q, k))], index


def _reranker_set(seed=0, n=50000, d=256, nq=24, nb=8):
    """a corpus of n N(0,1) documents in 256 leaves (codes M = 2, K = 16) and nq queries choosing nb leaves each"""
    from mevi_b200.rerank import ClusterIndex

    rs = np.random.RandomState(seed)
    D = rs.standard_normal((n, d)).astype(np.float32)
    codes = rs.randint(0, 16, size=(n, 2)).astype(np.int32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    leaves = np.stack([rs.choice(256, nb, replace=False) for _ in range(nq)])
    dec = np.stack([leaves // 16, leaves % 16], axis=-1).astype(np.int64)  # [nq, nb, 2]
    allowed = np.zeros((nq, n), bool)
    leaf_of_doc = codes[:, 0] * 16 + codes[:, 1]
    for q in range(nq):
        allowed[q] = np.isin(leaf_of_doc, leaves[q])
    return D, codes, Q, dec, allowed, ClusterIndex.from_codes(codes, 16)


def _reranker(D, index, mode):
    from mevi_b200.rerank import ClusterReranker

    return ClusterReranker(_dev(D), index, mode=mode)


@pytest.mark.gpu
def test_topk_power_of_two_scale_invariance():
    """D times 2^s and Q times 2^t: ids identical and scores exactly 2^(s+t) times the unscaled scores, for the flat
    search in every mode, the persistent index, and the cluster re-rank in both paths."""
    rs = np.random.RandomState(9)
    n, d, nq, k = 20000, 256, 16, 100
    D = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    pairs = ((0, 0), (-20, 0), (0, 20), (20, -20))
    for mode in ("exact", "tensor", "auto"):
        base = {}
        for s, t in pairs:
            searches, index = _flat_searches(D * np.float32(2.0 ** s), mode)
            for name, search in searches:
                sc, ids = search(Q * np.float32(2.0 ** t), k)
                if name not in base:
                    base[name] = (sc, ids)
                assert np.array_equal(ids, base[name][1]), f"{name} s={s} t={t}: ids differ"
                assert np.array_equal(sc, base[name][0] * np.float32(2.0 ** (s + t))), f"{name} s={s} t={t}: scores not exact"
            index.close()
    D, _, Q, dec, _, index = _reranker_set()
    for mode in ("stream", "grouped"):
        base = None
        for s, t in pairs:
            rr = _reranker(D * np.float32(2.0 ** s), index, mode)
            sc, ids, _ = rr.rerank(Q * np.float32(2.0 ** t), dec, topk=k)
            assert rr.last_path.startswith(mode)
            sc, ids = sc.cpu().numpy(), ids.cpu().numpy()
            if base is None:
                base = (sc, ids)
            assert np.array_equal(ids, base[1]), f"rerank {mode} s={s} t={t}: ids differ"
            assert np.array_equal(sc, base[0] * np.float32(2.0 ** (s + t))), f"rerank {mode} s={s} t={t}: scores not exact"


@pytest.mark.gpu
@pytest.mark.parametrize("docs", ["gauss", "mixed_norms"])
def test_topk_boundary_documents(docs):
    """~200 documents per query at s_k +- delta |q||d| (delta 2^-24 ... 2^-6): the float64 top-k up to the fp32 bound.
    mixed_norms: 5 % of the other documents scaled by 2^-20 ... 2^10."""
    rs = np.random.RandomState(17)
    n, d, nq, k = 20000, 256, 8, 100
    D = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    if docs == "mixed_norms":
        sel = rs.choice(n, n // 20, replace=False)
        D[sel] *= np.ldexp(1.0, rs.randint(-20, 11, size=len(sel)))[:, None].astype(np.float32)
    D, rel, _ = topk_boundary_docs(D, Q, k, rs)
    assert (np.abs(rel) < 2.0 ** -5).mean() > 0.95 and (np.abs(rel) < TIE).mean() > 0.05
    for mode in ("exact", "tensor", "auto"):
        searches, index = _flat_searches(D, mode)
        for name, search in searches:
            sc, ids = search(Q, k)
            check_topk_float64(sc, ids, Q, D, k)
        index.close()


TINY = (-30, -33, -36)


def _mixed_batch(Q, exps=TINY, n_copies=4, zeros=2):
    """Q plus copies of its first queries scaled by 2^e for e in exps, and zero queries
    -> (batch, source row (-1: zero query), exponent (None: zero query))"""
    rows, src, ex = [Q], list(range(len(Q))), [0] * len(Q)
    for e in exps:
        rows.append(Q[:n_copies] * np.float32(2.0 ** e))
        src += list(range(n_copies))
        ex += [e] * n_copies
    rows.append(np.zeros((zeros, Q.shape[1]), np.float32))
    src += [-1] * zeros
    ex += [None] * zeros
    return np.concatenate(rows).astype(np.float32), np.array(src), ex


@pytest.mark.gpu
@pytest.mark.parametrize("scale", ["2^-30", "2^-33", "2^-36", "0", "all"])
def test_mixed_norm_query_batch_flat(scale):
    """Queries 2^-30 ... 2^-36 times smaller than the rest of their batch: their fp16 images are subnormal or zero, so
    the prefilter error is no longer relative to |q|.  Every mode must still return the float64 top-k up to the fp32
    bound, and the exact mode exactly 2^e times the unscaled query's answer.  One scale per batch: a zero query puts
    every document in its window, and the overflow sends the whole call to the fp32 search."""
    rs = np.random.RandomState(23)
    n, d, nq, k = 20000, 768, 8, 100
    D = rs.standard_normal((n, d)).astype(np.float32)
    Q = rs.standard_normal((nq, d)).astype(np.float32)
    exps = {"all": TINY, "0": ()}.get(scale, (int(scale[2:]),) if scale.startswith("2^") else ())
    B, src, ex = _mixed_batch(Q, exps, zeros=2 if scale in ("0", "all") else 0)
    c = _ctx()
    s_ref, i_ref = (t.cpu().numpy() for t in c.flat_ip_topk(_dev(Q), _dev(D), k, mode="exact"))
    s_zero, i_zero = (t.cpu().numpy() for t in c.flat_ip_topk(_dev(np.zeros((1, d), np.float32)), _dev(D), k, mode="exact"))
    for mode in ("exact", "tensor", "auto"):
        searches, index = _flat_searches(D, mode)
        for name, search in searches:
            sc, ids = search(B, k)
            check_topk_float64(sc, ids, B, D, k)
            if mode == "exact":
                for i, (j, e) in enumerate(zip(src, ex)):
                    want_s, want_i = (s_zero[0], i_zero[0]) if e is None else (s_ref[j] * np.float32(2.0 ** e), i_ref[j])
                    assert np.array_equal(ids[i], want_i) and np.array_equal(sc[i], want_s), f"{name} row {i}"
        index.close()


@pytest.mark.gpu
def test_topk_adversarial_rounding():
    """fp16 rounding errors near the bound, pointing the wrong way (adversarial_rounding_docs): the weakest true
    members are found only through the full margin, in every flat entry point."""
    D, q, members = adversarial_rounding_docs()
    k = len(members)
    Q = np.concatenate([q, q * np.float32(2.0 ** -7)])
    for mode in ("tensor", "auto"):
        searches, index = _flat_searches(D, mode)
        for name, search in searches:
            sc, ids = search(Q, k)
            for r in range(len(Q)):
                assert set(ids[r].tolist()) == set(members.tolist()), f"{name} query {r}: {len(set(members) - set(ids[r]))} members missing"
            check_topk_float64(sc, ids, Q, D, k)
        index.close()


@pytest.mark.gpu
def test_mixed_norm_query_batch_grouped_rerank():
    """The same batch through the leaf-grouped tensor re-rank: only the tiny queries may fail their guarantee (and are
    then re-run by the streaming kernel); every query gets the float64 top-k of its candidates up to the fp32 bound."""
    D, _, Q, dec, allowed, index = _reranker_set(seed=4)
    B, src, ex = _mixed_batch(Q)
    decB = dec[np.where(src >= 0, src, 0)]
    allowedB = allowed[np.where(src >= 0, src, 0)]
    k = 100
    stream = _reranker(D, index, "stream")
    s_ref, i_ref, _ = stream.rerank(Q, dec, topk=k)
    s_ref, i_ref = s_ref.cpu().numpy(), i_ref.cpu().numpy()
    rr = _reranker(D, index, "grouped")
    sc, ids, _ = rr.rerank(B, decB, topk=k)
    sc, ids = sc.cpu().numpy(), ids.cpu().numpy()
    n_small = int(sum(e is not None and e != 0 for e in ex)) + 2
    assert rr.last_path in ("grouped", "grouped+stream") and rr.last_failed_queries <= n_small, (rr.last_path, rr.last_failed_queries)
    check_topk_float64(sc, ids, B, D, k, allowed=allowedB)
    sc2, ids2, _ = stream.rerank(B, decB, topk=k)
    check_topk_float64(sc2.cpu().numpy(), ids2.cpu().numpy(), B, D, k, allowed=allowedB)
    for i, (j, e) in enumerate(zip(src, ex)):  # the streaming kernel: exactly 2^e times the unscaled answer
        if e is not None:
            assert np.array_equal(ids2[i].cpu().numpy(), i_ref[j])
            assert np.array_equal(sc2[i].cpu().numpy(), s_ref[j] * np.float32(2.0 ** e))
