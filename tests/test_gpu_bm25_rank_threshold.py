"""K3's admission threshold from the commit-time rank table (Postings::rank_score).

rank_score[t][i] is the 2^i-th best posting score of term t, the stored fp32 value bit for bit (0 when df(t) < 2^i). The
query stage admits only documents scoring at or above the largest entry of rank 2^ceil(log2 P) over the query's terms;
results must stay bit-identical to the oracle. When the bitmap of a call admits fewer documents than the postings were
built from (a delete since the commit, a pushdown filter), the table's bound may not hold and the sampled threshold is
used instead."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RANKS = 11


def _expected_ranks(post, t):
    s = np.sort(post.score[post.off[t]:post.off[t + 1]])[::-1]
    return np.array([s[(1 << i) - 1] if len(s) >= (1 << i) else 0.0 for i in range(RANKS)], np.float32)


def _csr(n, triples):
    """(doc, term, tf) triples -> CSR by document, terms ascending inside a document"""
    doc, term, tf = (np.concatenate(a) for a in zip(*triples))
    o = np.lexsort((term, doc))
    off = np.concatenate([[0], np.cumsum(np.bincount(doc[o], minlength=n))]).astype(np.int64)
    return off, term[o].astype(np.uint32), tf[o].astype(np.uint16)


def _oracle_live(oracle, off, ids, tf, dl, vocab, dead):
    n = len(dl)
    live = np.ones(n, bool)
    live[list(dead)] = False
    keep = np.repeat(live, np.diff(off))
    off2 = np.concatenate([[0], np.cumsum(np.where(live, np.diff(off), 0))]).astype(np.int64)
    df = np.bincount(ids[keep], minlength=vocab).astype(np.uint32)
    return oracle.bm25_build(off2, ids[keep], tf[keep], dl, vocab, df, int(live.sum()), int(dl[live].astype(np.int64).sum()))


@pytest.mark.parametrize("chunk", [None, 1, 777, 20_000])
def test_rank_table_equals_order_statistics(ctx_scan, oracle, monkeypatch, chunk):
    """live df just below, at and above every 2^i (warp sort up to 1024 postings, radix select above), terms whose postings
    all tie, postings of documents tombstoned before the commit, and a build in several term ranges"""
    if chunk is not None:
        monkeypatch.setenv("KRAG_BM25_BUILD_CHUNK", str(chunk))
    g = np.random.default_rng(41)
    n = 6000
    dead = np.arange(0, n, 11)
    live_rows = np.setdiff1d(np.arange(n), dead)
    dl = g.integers(20, 300, n).astype(np.uint32)
    tie_rows = live_rows[:1500]
    dl[tie_rows] = 100
    dfs = sorted({max(1, (1 << i) + e) for i in range(12) for e in (-1, 0, 1)} | {3000, len(live_rows)})
    triples = []
    for t, df in enumerate(dfs):                                   # live postings exactly df, plus some on tombstoned rows
        rows = np.concatenate([g.choice(live_rows, df, replace=False), g.choice(dead, min(len(dead), df // 10 + 1), replace=False)])
        triples.append((rows, np.full(len(rows), t), g.integers(1, 6, len(rows))))
    t_tie_big, t_tie_small = len(dfs), len(dfs) + 1                # tf 1 on rows of one length: every score equal
    triples.append((tie_rows, np.full(1500, t_tie_big), np.ones(1500, np.int64)))
    triples.append((tie_rows[:700], np.full(700, t_tie_small), np.ones(700, np.int64)))
    vocab = len(dfs) + 3                                           # the last id has no postings
    off, ids, tf = _csr(n, triples)
    x = oracle.synth_dense(n, 8, 42)
    ix = ctx_scan.create_index(f"rank_{chunk}", 8)
    try:
        ix.add(np.arange(n, dtype=np.uint64), x, off, ids, tf, dl)
        ix.remove(dead.astype(np.uint64))
        ix.commit(vocab)
        post = _oracle_live(oracle, off, ids, tf, dl, vocab, dead)
        assert [int(post.off[t + 1] - post.off[t]) for t in range(len(dfs))] == dfs
        for t in range(vocab):
            got, want = ix.read_rank_scores(t), _expected_ranks(post, t)
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (t, got, want)
        assert np.all(ix.read_rank_scores(t_tie_big) == post.score[post.off[t_tie_big]])
    finally:
        ix.drop()


@pytest.fixture(scope="module")
def sparse_400k_tie(ctx_scan, oracle):
    """400k documents (98 sub-tiles, above the 32768-entry candidate lists: the thresholded path) plus one extra term on
    1500 documents of the same length with tf 1, so its top postings all tie"""
    n, vocab0 = 400_000, 60_000
    x = oracle.synth_dense(n, 32, 51)
    off, ids, tf, dl = oracle.synth_sparse(n, vocab0, 52)
    common = np.bincount(dl).argmax()
    rows = np.nonzero(dl == common)[0][:1500]
    assert len(rows) >= 1100
    t_tie, vocab = vocab0, vocab0 + 1
    ids = np.insert(ids, off[rows + 1], np.uint32(t_tie))          # appended to each chosen document's list
    tf = np.insert(tf, off[rows + 1], np.uint16(1))
    add = np.zeros(n, np.int64)
    add[rows] = 1
    off = off + np.concatenate([[0], np.cumsum(add)])
    ix = ctx_scan.create_index("rank_400k", 32)
    ix.add(np.arange(n, dtype=np.uint64), x, off, ids, tf, dl)
    ix.commit(vocab)
    post = oracle.bm25_build(off, ids, tf, dl, vocab)
    yield ix, post, x, n, vocab, t_tie
    ix.drop()


def _queries(oracle, vocab, t_tie):
    qs = oracle.synth_query_terms(vocab - 1, 24, seed=53, rank_offset=20)
    qs[0] = np.concatenate([qs[0], qs[0]])                         # every term twice
    qs[1] = np.concatenate([[vocab + 5], qs[1], [vocab + 1000]]).astype(np.uint32)   # out-of-vocabulary ids
    qs[2] = np.random.default_rng(54).integers(0, 2000, 45).astype(np.uint32)       # > 32 terms
    qs[3] = np.array([t_tie], np.uint32)
    qs[4] = np.array([t_tie, vocab - 2, t_tie], np.uint32)
    qs[5] = np.array([vocab + 3], np.uint32)                      # nothing in the vocabulary
    qs[6] = np.array([0, 1, 2, 3], np.uint32)                     # the most frequent terms: ~every document matches
    qs[7] = np.array([vocab - 2], np.uint32)                      # a rare term: fewer postings than P
    return qs


@pytest.mark.parametrize("P", [1, 30, 33, 1024])
def test_rank_threshold_results_bit_exact(sparse_400k_tie, oracle, monkeypatch, P):
    ix, post, x, n, vocab, t_tie = sparse_400k_tie
    monkeypatch.setenv("KRAG_BM25_KERNEL", "warp")
    qs = _queries(oracle, vocab, t_tie)
    score, ordn = ix.search_bm25(qs, P)
    for b, qt in enumerate(qs):
        rs, ro = oracle.bm25_query(post, qt[qt < vocab], P)
        assert np.array_equal(ordn[b], ro), (b, P)
        assert np.array_equal(score[b], rs), (b, P)


def test_pushdown_filter_takes_the_sampled_threshold(sparse_400k_tie, ctx_scan, oracle, monkeypatch):
    """eligible = allow & alive excludes documents the rank table counted: the sampled threshold (one more launch than
    the rank-table threshold) serves the call, results exact"""
    from kaito_b200 import _native
    ix, post, x, n, vocab, t_tie = sparse_400k_tie
    monkeypatch.setenv("KRAG_BM25_KERNEL", "warp")
    qs = _queries(oracle, vocab, t_tie)[:8]
    q = oracle.synth_queries(x, len(qs), 55)
    k = 10
    P = oracle.pool_size(k)
    allow = np.packbits(np.random.default_rng(56).random(((n + 31) // 32) * 32) < 0.3, bitorder="little").view(np.uint32)
    ix.retrieve(q, qs, k, keyword_allow_bitmap=allow)             # warm-up of both paths' workspaces
    ix.retrieve(q, qs, k, fusion_mode=_native.FILTER_PUSHDOWN, keyword_allow_bitmap=allow)
    l0 = ctx_scan.launch_count()
    ix.retrieve(q, qs, k, keyword_allow_bitmap=allow)
    l1 = ctx_scan.launch_count()
    got = ix.retrieve(q, qs, k, fusion_mode=_native.FILTER_PUSHDOWN, keyword_allow_bitmap=allow)
    l2 = ctx_scan.launch_count()
    assert (l2 - l1) - (l1 - l0) == 1                              # sample pass + its select instead of the threshold kernel
    for b, qt in enumerate(qs):
        dd, do = oracle.dense_topk(x, q[b:b + 1], P, allow)
        bs, bo = oracle.bm25_query(post, qt[qt < vocab], P, allow)
        fin, de, sp, rk, od = oracle.fuse(dd[0], do[0], bs, bo, k)
        cnt = int(got["count"][b])
        assert cnt == len(od) and np.array_equal(got["ordinal"][b, :cnt], od), b
        assert np.array_equal(got["final"][b, :cnt], fin), b


def test_delete_after_commit_takes_the_sampled_threshold(sparse_400k_tie, ctx_scan, oracle, monkeypatch):
    """documents deleted after the commit stay in the postings and in the rank table: the bound may not hold, so the
    sampled threshold serves the query until the next commit.  Deletes the best documents of every query (runs last:
    it changes the module's index)"""
    ix, post, x, n, vocab, t_tie = sparse_400k_tie
    monkeypatch.setenv("KRAG_BM25_KERNEL", "warp")
    qs = _queries(oracle, vocab, t_tie)
    P = 30
    ix.search_bm25(qs, P)
    l0 = ctx_scan.launch_count()
    _, ordn = ix.search_bm25(qs, P)
    l1 = ctx_scan.launch_count()
    dead = sorted(set(ordn[ordn >= 0].tolist()))
    assert ix.remove(np.array(dead, np.uint64)) == len(dead)
    score, ordn = ix.search_bm25(qs, P)
    l2 = ctx_scan.launch_count()
    assert (l2 - l1) - (l1 - l0) == 1
    alive = oracle.alive_bitmap(n, dead)
    for b, qt in enumerate(qs):
        rs, ro = oracle.bm25_query(post, qt[qt < vocab], P, alive)
        assert np.array_equal(ordn[b], ro), b
        assert np.array_equal(score[b], rs), b
