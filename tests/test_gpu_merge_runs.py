"""mevi_merge_sorted_runs (the cross-rank merge of a sharded rerank_all) through the C ABI, against numpy: the runs
concatenated and lexsorted by (query, -score, id)."""
import numpy as np
import pytest
import torch

import mevi_b200
from gpu_util import ctx, dev

pytestmark = pytest.mark.gpu


def _runs(S, nq, lens, rs, tie_pool=None, pad=0):
    """S runs of nq queries with lens[r][q] elements each, sorted by (score desc, id asc); ids distinct across runs
    (a document lives on one rank).  -> (scores_in, ids_in, bases, run_offsets, expected scores, expected ids, out_offsets),
    the runs laid out one block per run, each block followed by `pad` garbage elements."""
    lens = np.asarray(lens, dtype=np.int64).reshape(S, nq)
    total = int(lens.sum())
    ids = rs.permutation(max(4 * total, 1))[:total].astype(np.int64) * 3 + 1
    if tie_pool is not None:
        scores = rs.choice(np.asarray(tie_pool, np.float32), total)
    else:
        scores = rs.standard_normal(total).astype(np.float32)
    run_off = np.zeros((S, nq + 1), np.int64)
    run_off[:, 1:] = np.cumsum(lens, axis=1)
    blocks_s, blocks_i, bases, ref = [], [], [], []
    at, base = 0, 0
    for r in range(S):
        bs, bi = [], []
        for q in range(nq):
            s_, i_ = scores[at : at + lens[r, q]], ids[at : at + lens[r, q]]
            at += lens[r, q]
            o = np.lexsort((i_, -s_))
            bs.append(s_[o])
            bi.append(i_[o])
            ref.append((np.full(lens[r, q], q), s_, i_))
        bases.append(base)
        blocks_s += bs + [np.full(pad, np.nan, np.float32)]
        blocks_i += bi + [np.full(pad, -7, np.int64)]
        base += int(lens[r].sum()) + pad
    qq, ss, ii = (np.concatenate([x[j] for x in ref]) if ref else np.zeros(0) for j in range(3))
    o = np.lexsort((ii, -ss, qq))
    out_off = np.zeros(nq + 1, np.int64)
    out_off[1:] = np.cumsum(lens.sum(0))
    return (np.concatenate(blocks_s).astype(np.float32), np.concatenate(blocks_i).astype(np.int64), np.asarray(bases, np.int64),
            run_off, ss[o].astype(np.float32), ii[o].astype(np.int64), out_off)


def _merge(scores_in, ids_in, bases, run_off, out_off):
    s, i = ctx().merge_sorted_runs(dev(scores_in), dev(ids_in), dev(bases), dev(run_off), dev(out_off))
    return s.cpu().numpy(), i.cpu().numpy()


def _check(case):
    scores_in, ids_in, bases, run_off, want_s, want_i, out_off = case
    s, i = _merge(scores_in, ids_in, bases, run_off, out_off)
    assert np.array_equal(i, want_i)
    assert np.array_equal(s.view(np.int32), want_s.view(np.int32))  # bit for bit: -0.0 stays -0.0


@pytest.mark.parametrize("S", [1, 2, 3, 4, 5, 6, 7, 8])
def test_random_runs(S):
    rs = np.random.RandomState(S)
    nq = 37
    lens = rs.randint(0, 3000, size=(S, nq))
    lens[:, 3] = 0  # an empty query
    lens[0, 5] = 0  # an empty run
    lens[:, 7] = rs.randint(0, 3, S)  # tiny queries: one tile spans many of them
    _check(_runs(S, nq, lens, rs, pad=13))


@pytest.mark.parametrize("S", [2, 3, 8])
def test_ties_and_signed_zeros(S):
    """Exact score ties across runs (ordered by id) and -0.0 / +0.0, which compare equal."""
    rs = np.random.RandomState(10 + S)
    lens = rs.randint(0, 5000, size=(S, 5))
    _check(_runs(S, 5, lens, rs, tie_pool=[1.5, 0.25, 0.0, -0.0, -1.0, np.float32(1e-38)]))


@pytest.mark.parametrize("S", [1, 4, 7])
def test_one_query_holds_everything(S):
    rs = np.random.RandomState(20 + S)
    lens = np.zeros((S, 6), np.int64)
    lens[:, 4] = rs.randint(20000, 70001, S)
    _check(_runs(S, 6, lens, rs))


def test_no_elements_and_no_queries():
    for nq in (0, 3):
        _check(_runs(3, nq, np.zeros((3, nq), np.int64), np.random.RandomState(0)))


def test_invalid_arguments():
    c = ctx()
    case = _runs(2, 4, np.full((2, 4), 5), np.random.RandomState(0))
    s_in, i_in, bases, run_off, _, _, out_off = (dev(a) for a in case)
    with pytest.raises(mevi_b200.MeviError, match="error -1"):
        c.merge_sorted_runs(s_in, i_in, bases, run_off, out_off + torch.arange(5, device=out_off.device))
    bad = run_off.clone()
    bad[1, 2] = bad[1, 3] + 1  # a run that shrinks
    with pytest.raises(mevi_b200.MeviError, match="error -1"):
        c.merge_sorted_runs(s_in, i_in, bases, bad, out_off)
    for S in (0, 9):
        ro = torch.zeros((S, 5), dtype=torch.int64, device=s_in.device)
        with pytest.raises(mevi_b200.MeviError, match="error -1"):
            c.merge_sorted_runs(s_in, i_in, torch.zeros(S, dtype=torch.int64, device=s_in.device), ro, torch.zeros_like(out_off))


def test_torch_device_sort_orders_signed_zeros_as_equal():
    """The order the merge reproduces: rerank_all's stable descending device sort keeps -0.0 and +0.0 in their input
    order, both on its small-sort path and on its radix-sort path."""
    for n in (1000, 1 << 20):
        x = torch.zeros(n, device="cuda:0")
        x[::2] = -0.0
        x[: n // 4] = 1.0
        order = torch.argsort(x, descending=True, stable=True)
        zeros = order[n // 4 :]
        assert torch.equal(zeros, torch.arange(n // 4, n, device="cuda:0")), f"n={n}: -0.0 and +0.0 are ordered apart"


def test_more_than_2_31_elements():
    """int64 offsets: three runs, 2^31 + 4,099 elements in three queries (one of them nearly all), through the scratch
    buffers.  Expected result built arithmetically: ids 0..total-1 ascending, score -(id >> 10)."""
    total = (1 << 31) + 4099
    need = total * 12 * 3 + (8 << 30)
    if torch.cuda.mem_get_info(0)[0] < need:
        pytest.skip(f"needs {need / 2**30:.0f} GiB free")
    d = torch.device("cuda", 0)
    qb = [0, 5, (1 << 31) - 7, total]
    S = 3
    ids_in = torch.empty(total, dtype=torch.int64, device=d)
    run_off = torch.zeros((S, 4), dtype=torch.int64)
    at = 0
    bases = []
    for r in range(S):
        bases.append(at)
        for q in range(3):
            first = qb[q] + (r - qb[q]) % S
            n = max(0, (qb[q + 1] - first + S - 1) // S)
            torch.arange(first, first + S * n, S, out=ids_in[at : at + n])
            at += n
            run_off[r, q + 1] = run_off[r, q] + n
    assert at == total
    scores_in = torch.empty(total, dtype=torch.float32, device=d)
    chunk = 1 << 28
    for a in range(0, total, chunk):
        scores_in[a : a + chunk] = -(ids_in[a : a + chunk] >> 10).to(torch.float32)
    out_off = torch.tensor(qb, dtype=torch.int64, device=d)
    s, i = ctx().merge_sorted_runs(scores_in, ids_in, torch.tensor(bases, dtype=torch.int64, device=d), run_off.to(d), out_off)
    del scores_in, ids_in
    for a in range(0, total, chunk):
        want = torch.arange(a, min(a + chunk, total), device=d)
        assert torch.equal(i[a : a + chunk], want), f"ids differ in [{a}, {a + chunk})"
        assert torch.equal(s[a : a + chunk], -(want >> 10).to(torch.float32))
