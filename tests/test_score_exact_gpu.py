"""Adversarial and headline-size parity tests for the score + top-k path: the cases where an approximate candidate
selection CAN differ from the exact order (VERDICT r01 "weak #2"), checked bit-exactly against oracle/score_oracle.c.

What makes the ids provable (score.cu header): the tensor-core key only selects candidates; after the exact fp64
re-score a per-query guard checks that nothing outside the candidate set can reach the k-th exact key, and queries that
fail it go through a threshold-collect pass.  These tests build inputs that fail the guard on purpose.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _unit_rows(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def _check(store, so, q, corpus, k, metric="prenormalized-angular", doc_of_row=None, **kw):
    doc, row, score = store.search(q, k, **kw)
    edoc, erow, escore = so.search(q, corpus, k, metric, doc_of_row)
    np.testing.assert_array_equal(doc, edoc)
    np.testing.assert_array_equal(row, erow)
    np.testing.assert_allclose(score, escore, rtol=0, atol=1e-12)
    return doc, row, score


def _ulp_family(base: np.ndarray, count: int, rng) -> np.ndarray:
    """`count` fp16 neighbours of `base` whose dot products with `base` differ by ~1e-9 .. 1e-7: one-ulp moves of
    SMALL components (a 1-ulp step of a 1e-3 component changes the dot by ~1e-9) — far below what an fp32 tensor-core
    accumulation can order."""
    h = base.astype(np.float16)
    small = np.argsort(np.abs(h.astype(np.float32)))[8:8 + 64]
    out = np.repeat(h[None, :], count, axis=0)
    for i in range(count):
        idx = rng.choice(small, size=1 + i % 3, replace=False)
        bits = out[i].view(np.uint16).copy()
        bits[idx] += np.uint16(1 + (i % 2))
        out[i] = bits.view(np.float16)
    return out.astype(np.float32)


def test_many_identical_rows_with_permuted_documents(gpu_required, score_oracle):
    """40 identical rows whose document numbers are NOT monotone in row order (routine after overwrites: the document
    keeps its number, its rows go to the end).  Exact order = doc asc; arrival order = row asc."""
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(1)
    n, d = 40000, 256
    corpus = _unit_rows(rng, n, d)
    dup_rows = rng.choice(n, size=40, replace=False)
    corpus[dup_rows] = corpus[dup_rows[0]]
    doc_of_row = rng.permutation(n).astype(np.int32)             # one chunk per document, shuffled numbering
    q = _unit_rows(rng, 9, d)
    q[0] = corpus[dup_rows[0]]
    store = RowStore(d)
    store.add(corpus, doc_of_row)
    doc, _, score = _check(store, score_oracle, q, corpus, 10, doc_of_row=doc_of_row)
    assert list(doc[0]) == sorted(doc_of_row[dup_rows])[:10]
    assert np.all(score[0] == score[0, 0])
    # 40 ties still fit the 64 candidates the merge re-scores exactly: answered in one pass, provably (guard held)
    assert store.search_stats()["flagged"] == 0
    for k in (1, 16, 39, 40, 41, 64):
        _check(store, score_oracle, q, corpus, k, doc_of_row=doc_of_row)
    # 150 ties do not: the guard must notice (exact k-th key == bound of the unexamined rows) and the collect pass answer
    more = rng.choice(n, size=150, replace=False)
    corpus2 = corpus.copy()
    corpus2[more] = corpus2[more[0]]
    q2 = q.copy()
    q2[0] = corpus2[more[0]]
    store2 = RowStore(d)
    store2.add(corpus2, doc_of_row)
    doc2, _, _ = _check(store2, score_oracle, q2, corpus2, 10, doc_of_row=doc_of_row)
    assert list(doc2[0]) == sorted(doc_of_row[more])[:10]
    st = store2.search_stats()
    assert st["flagged"] >= 1 and st["collect_passes"] >= 1
    for k in (64, 100, 149, 150, 151):
        _check(store2, score_oracle, q2, corpus2, k, doc_of_row=doc_of_row)


@pytest.mark.parametrize("spread", ["one_tile", "all_over"])
def test_near_ties_around_rank_k(gpu_required, score_oracle, spread):
    """30 rows whose exact scores differ by < 1e-7 straddle rank k: fp32 cannot order them, fp64 must."""
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(2)
    n, d = 60000, 768
    corpus = _unit_rows(rng, n, d)
    base = corpus[77].copy()
    fam = _ulp_family(base, 30, rng)
    rows = np.arange(5000, 5030) if spread == "one_tile" else rng.choice(n, size=30, replace=False)
    corpus[rows] = fam
    q = _unit_rows(rng, 5, d)
    q[0] = base
    store = RowStore(d)
    store.add(corpus)
    doc, _, score = _check(store, score_oracle, q, corpus, 10)
    top = score[0]
    assert set(doc[0]).issubset(set(rows.tolist()) | {77})
    assert np.all(np.diff(top) <= 0) and (top[0] - top[-1]) < 1e-6       # really a near-tie cluster
    for k in (3, 16, 25):
        _check(store, score_oracle, q, corpus, k)


def test_near_tied_chunks_of_one_document(gpu_required, score_oracle):
    """A document's best chunk is chosen on the EXACT score: chunks closer than the approximation error are all kept
    by the scan and decided by the fp64 pass (row = Vespa's closest(), the _highlights source)."""
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(3)
    n, d = 20000, 512
    corpus = _unit_rows(rng, n, d)
    doc_of_row = (np.arange(n) // 4).astype(np.int32)
    base = corpus[4000].copy()
    fam = _ulp_family(base, 24, rng)
    corpus[4000:4004] = fam[:4]                                  # doc 1000: four chunks within 1e-8
    corpus[8000:8020] = fam[4:]                                  # docs 2000..2004: twenty more
    q = _unit_rows(rng, 6, d)
    q[0] = base
    store = RowStore(d)
    store.add(corpus, doc_of_row)
    for k in (1, 5, 10, 30):
        _check(store, score_oracle, q, corpus, k, doc_of_row=doc_of_row)


def test_ties_across_a_shard_boundary(gpu_required, score_oracle):
    """The same family split over two row shards with document offsets, merged on the device."""
    import torch
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(4)
    n, d, nq, k = 30000, 256, 4, 10
    corpus = _unit_rows(rng, n, d)
    base = corpus[5].copy()
    rows = np.concatenate([np.arange(100, 112), np.arange(20000, 20012)])
    corpus[rows] = _ulp_family(base, 24, rng)
    corpus[25000:25004] = base                                   # exact duplicates in the second shard
    q = _unit_rows(rng, nq, d)
    q[0] = base
    cut = 15000
    shards = [RowStore(d), RowStore(d)]
    shards[0].add(corpus[:cut])
    shards[1].add(corpus[cut:])
    shards[1].set_doc_offset(cut)
    nk = nq * k
    qd = torch.from_numpy(q).cuda()
    gathered = torch.empty(2 * nk * 16, dtype=torch.uint8, device="cuda")
    for i, st in enumerate(shards):
        b = gathered.data_ptr() + i * nk * 16
        st.search_device(qd.data_ptr(), nq, k, b, b + nk * 4, b + nk * 8, sync=True)
    od = torch.empty(nq, k, dtype=torch.int32, device="cuda")
    orow = torch.empty_like(od)
    osc = torch.empty(nq, k, dtype=torch.float64, device="cuda")
    shards[0].merge_shards_device(gathered.data_ptr(), 2, nq, k, od.data_ptr(), orow.data_ptr(), osc.data_ptr())
    ed, _, es = score_oracle.search(q, corpus, k)
    np.testing.assert_array_equal(od.cpu().numpy(), ed)
    np.testing.assert_allclose(osc.cpu().numpy(), es, rtol=0, atol=1e-12)


def test_async_entry_point_runs_the_fallback_without_host_help(gpu_required, score_oracle):
    """b200_index_search_device(sync=0) enqueues one collect + finalize pass unconditionally: the tie case is answered
    with no host round trip in between."""
    import torch
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(5)
    n, d, nq, k = 30000, 128, 8, 10
    corpus = _unit_rows(rng, n, d)
    corpus[1000:1030] = corpus[3]
    q = _unit_rows(rng, nq, d)
    q[0] = corpus[3]
    store = RowStore(d)
    store.add(corpus)
    qd = torch.from_numpy(q).cuda()
    od = torch.empty(nq, k, dtype=torch.int32, device="cuda")
    orow = torch.empty_like(od)
    osc = torch.empty(nq, k, dtype=torch.float64, device="cuda")
    store.search_device(qd.data_ptr(), nq, k, od.data_ptr(), orow.data_ptr(), osc.data_ptr(), sync=False)
    torch.cuda.synchronize()
    ed, er, es = score_oracle.search(q, corpus, k)
    np.testing.assert_array_equal(od.cpu().numpy(), ed)
    np.testing.assert_array_equal(orow.cpu().numpy(), er)
    assert store.search_stats()["unresolved_async"] == 0


@pytest.mark.parametrize("k", [11, 100, 160, 161, 1000, 3000])
def test_large_k(gpu_required, score_oracle, k):
    """limit <= 1000, offset <= 10000 (api/configs.py:24-25): k <= 160 is one pass over random data; beyond that one
    collect pass (or more for deep pagination)."""
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(k)
    n, d = 100000, 128
    corpus = _unit_rows(rng, n, d)
    corpus[100:140] = corpus[5]                                   # a run of exact ties
    doc_of_row = (np.arange(n) // 2).astype(np.int32)            # 2 chunks per doc
    q = _unit_rows(rng, 7, d)
    q[0] = corpus[5]
    store = RowStore(d)
    store.add(corpus, doc_of_row)
    _check(store, score_oracle, q[1:], corpus, k, doc_of_row=doc_of_row)
    st = store.search_stats()
    if k <= 160:
        assert st["flagged"] == 0, st                             # single pass: nothing needed the fallback
    _check(store, score_oracle, q, corpus, k, doc_of_row=doc_of_row)
    small = RowStore(d)
    small.add(corpus[:30])                                        # fewer documents than k
    doc, _, _ = small.search(q[:2], k)
    assert (doc[:, :30] >= 0).all() and (doc[:, 30:] == -1).all()
    _check(small, score_oracle, q[:2], corpus[:30], k)


def test_document_filter_bitset(gpu_required, score_oracle):
    """A filtered query = the same scan with a document bitset next to the tombstone check."""
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(7)
    n, d = 50000, 256
    corpus = _unit_rows(rng, n, d)
    doc_of_row = (np.arange(n) // 2).astype(np.int32)
    ndocs = n // 2
    q = _unit_rows(rng, 12, d)
    for frac in (0.5, 0.01, 0.0002, 0.0):
        keep = rng.random(ndocs) < frac
        bits = np.packbits(keep, bitorder="little").view(np.uint8)
        bits = np.concatenate([bits, np.zeros((-len(bits)) % 4, np.uint8)]).view(np.uint32)
        masked = np.where(keep[doc_of_row], doc_of_row, -1).astype(np.int32)
        for store_docs in (doc_of_row, None):
            store = RowStore(d)
            if store_docs is None:                                # identity-mapped corpus: filter still applies
                store.add(corpus)
                keep_r = rng.random(n) < frac
                b2 = np.packbits(keep_r, bitorder="little")
                b2 = np.concatenate([b2, np.zeros((-len(b2)) % 4, np.uint8)]).view(np.uint32)
                m2 = np.where(keep_r, np.arange(n), -1).astype(np.int32)
                _check(store, score_oracle, q, corpus, 10, doc_of_row=m2, filter_bits=b2, filter_docs=n, filter_tag=11)
                _check(store, score_oracle, q, corpus, 10, doc_of_row=m2, filter_bits=b2, filter_docs=n, filter_tag=11)
            else:
                store.add(corpus, store_docs)
                _check(store, score_oracle, q, corpus, 10, doc_of_row=masked, filter_bits=bits, filter_docs=ndocs)
                _check(store, score_oracle, q, corpus, 200, doc_of_row=masked, filter_bits=bits, filter_docs=ndocs)
            _check(store, score_oracle, q, corpus, 10, doc_of_row=store_docs)   # and the filter is gone afterwards


def test_filter_with_modifiers(gpu_required, score_oracle):
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(8)
    n, d = 20000, 128
    corpus = _unit_rows(rng, n, d)
    q = _unit_rows(rng, 5, d)
    store = RowStore(d)
    store.add(corpus)
    vals = rng.uniform(0.5, 2.0, size=n)
    store.set_attributes_multi(np.zeros(n, np.int32), np.arange(n, dtype=np.int32), vals)
    keep = rng.random(n) < 0.1
    bits = np.packbits(keep, bitorder="little")
    bits = np.concatenate([bits, np.zeros((-len(bits)) % 4, np.uint8)]).view(np.uint32)
    mod = score_oracle.modifiers(vals[None, :], [(0, 1.5)], [(0, 0.01)])
    doc, row, score = store.search(q, 10, mult=[(0, 1.5)], add=[(0, 0.01)], filter_bits=bits, filter_docs=n)
    masked = np.where(keep, np.arange(n), -1).astype(np.int32)
    ed, er, es = score_oracle.search_modified(q, corpus, 10, mod, doc_of_row=masked)
    np.testing.assert_array_equal(doc, ed)
    np.testing.assert_array_equal(row, er)
    np.testing.assert_allclose(score, es, rtol=0, atol=1e-12)


def test_delete_rows_and_compact(gpu_required, score_oracle):
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(9)
    n, d = 12000, 128
    corpus = _unit_rows(rng, n, d)
    doc_of_row = (np.arange(n) // 3).astype(np.int32)
    q = _unit_rows(rng, 10, d)
    store = RowStore(d, metric="euclidean")
    store.add(corpus, doc_of_row)
    dead = rng.choice(n, size=5000, replace=False)
    store.delete_rows(dead)
    masked = doc_of_row.copy()
    masked[dead] = -1
    _check(store, score_oracle, q, corpus, 10, metric="euclidean", doc_of_row=masked)
    new_of_old = store.compact()
    assert len(store) == n - 5000 and (new_of_old[dead] == -1).all()
    live = np.flatnonzero(masked >= 0)
    assert np.array_equal(new_of_old[live], np.arange(len(live)))
    _check(store, score_oracle, q, corpus[live], 10, metric="euclidean", doc_of_row=masked[live])
    store.add(corpus[:10], np.arange(4000, 4010, dtype=np.int32))
    _check(store, score_oracle, q, np.concatenate([corpus[live], corpus[:10]]), 10, metric="euclidean",
           doc_of_row=np.concatenate([masked[live], np.arange(4000, 4010, dtype=np.int32)]))


def test_non_finite_and_out_of_range_rows_are_rejected(gpu_required):
    from marqo_b200.engine import RowStore
    from marqo_b200._native import NativeError
    store = RowStore(64, metric="dotproduct")
    good = np.ones((3, 64), np.float32)
    store.add(good)
    for bad_value in (np.nan, np.inf, 1.0e5):
        bad = good.copy()
        bad[1, 7] = bad_value
        with pytest.raises(NativeError):
            store.add(bad)
        assert len(store) == 3                                    # nothing of a rejected batch is kept
    with pytest.raises(NativeError):
        store.search(np.full((1, 64), np.nan, np.float32), 2)
    doc, _, _ = store.search(good[:1], 5)
    assert list(doc[0]) == [0, 1, 2, -1, -1]


@pytest.mark.parametrize("metric", ["angular", "dotproduct", "euclidean"])
def test_ties_other_metrics_and_modifiers(gpu_required, score_oracle, metric):
    from marqo_b200.engine import RowStore
    rng = np.random.default_rng(10)
    n, d = 30000, 256
    corpus = rng.standard_normal((n, d)).astype(np.float32) * (0.3 if metric != "angular" else 1.0)
    corpus[200:240] = corpus[17]
    q = rng.standard_normal((6, d)).astype(np.float32) * 0.3
    q[0] = corpus[17]
    store = RowStore(d, metric=metric)
    store.add(corpus)
    for k in (10, 45):
        _check(store, score_oracle, q, corpus, k, metric=metric)
    vals = rng.uniform(0.9, 1.1, size=n)
    vals[200:240] = 1.0
    vals[17] = 1.0
    store.set_attributes(0, np.arange(n, dtype=np.int32), vals)
    mod = score_oracle.modifiers(vals[None, :], [(0, 1.0)], [])
    doc, row, score = store.search(q, 10, mult=[(0, 1.0)])
    ed, er, es = score_oracle.search_modified(q, corpus, 10, mod, metric=metric)
    np.testing.assert_array_equal(doc, ed)
    np.testing.assert_array_equal(row, er)
    np.testing.assert_allclose(score, es, rtol=0, atol=1e-9)


def test_two_million_rows_768(gpu_required, score_oracle):
    """VERDICT r01 next #1: parity at a corpus size where the scan runs thousands of tiles per SM.  2 M x 768 fp16
    (3 GB), 16 queries incl. self-matches and duplicates, bit-exact ids vs the OpenMP oracle."""
    import torch
    from marqo_b200.engine import RowStore
    n, d, nq = 2_000_000, 768, 8
    g = torch.Generator(device="cuda").manual_seed(123)
    store = RowStore(d, capacity=n)
    host = np.empty((n, d), np.float16)
    for lo in range(0, n, 250_000):
        x = torch.nn.functional.normalize(torch.randn(250_000, d, device="cuda", generator=g), dim=1)
        if lo == 0:
            x[1000:1024] = x[7]                                   # duplicates
        torch.cuda.synchronize()
        store.add_device(x.data_ptr(), 250_000)
        host[lo:lo + 250_000] = x.half().cpu().numpy()
    q = torch.nn.functional.normalize(torch.randn(nq, d, device="cuda", generator=g), dim=1).cpu().numpy()
    q[0] = host[7].astype(np.float32)
    q[1] = host[1_999_999].astype(np.float32)
    doc, row, score = store.search(q, 10)
    qh = q.astype(np.float16).view(np.uint16)
    edoc, erow, escore = score_oracle.search_half(qh, host.view(np.uint16), 10)
    np.testing.assert_array_equal(doc, edoc)
    np.testing.assert_array_equal(row, erow)
    np.testing.assert_allclose(score, escore, rtol=0, atol=1e-12)
    assert doc[0, 0] == 7 and list(doc[0, 1:10]) == list(range(1000, 1009)) and doc[1, 0] == 1_999_999
    d100, _, _ = store.search(q[:2], 100)
    e100, _, _ = score_oracle.search_half(qh[:2], host.view(np.uint16), 100)
    np.testing.assert_array_equal(d100, e100)


def test_row_sharded_search_two_gpus(gpu_required):
    """N = 2 data path under torchrun: row shards, fused peer-store exchange (falls back to NCCL all-gather), identical
    merged result on both ranks, ids bit-exact vs the oracle (tests/dist_check_multigpu.py).  Needs 2 GPUs."""
    import os
    import subprocess
    import sys
    from marqo_b200 import _native
    if _native.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "tests", "dist_check_multigpu.py")]
    r = subprocess.run(cmd, cwd=root, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "ids bit-exact vs oracle: True" in r.stdout and "all ranks identical: True" in r.stdout
