"""GPU parity tests of the ft_fast merge (rxgpu_ft_merge) against the oracle -- the reference's own ft::Merger::Merge when
oracle/_ref is present, else the pinned C port -- and the committed golden fixtures.  Integer outputs (ids, order, uint8 ranks,
fields) must match exactly: the device evaluates BM25 in fp64 and the rank products in fp32 in the reference's operation order."""
import os

import numpy as np
import pytest
from ft_helpers import (add_random_synonyms, assert_same_merge, assert_same_merge_as_digest, corpus_problem, gpu_merge, load_golden_problem,
                        merge_digest, random_problem)

from oracle import ft_oracle as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_golden_fixtures():
    g = np.load(os.path.join(ROOT, "tests", "golden", "ft_golden.npz"))
    for name in g["names"]:
        p = load_golden_problem(g, str(name))
        for rst in (F.RANK_AND_ID, F.RANK_ONLY):
            res, st = gpu_merge(p, rst)
            assert_same_merge(g[f"{name}/result{rst}"], res, rst, ctx=f"{name} rst={rst}")
        if "preselect" in str(name):
            assert st["preselected"] == 1


def test_known_answer_values():
    p = F.FtProblem(6, np.array([0, 8, 3, 6, 12, 3], np.uint32))
    p.add_term([(p.add_list([1], [[(0, 0)]]), 100.0), (p.add_list([1], [[(6, 0)]]), 80.0)])
    assert gpu_merge(p)[0].tolist() == [(1, 97.0, 0, 97)]  # uint8(97.9844), FTGenericApi.DebugInfo ft_generic.cc:326
    p2 = F.FtProblem(6, np.array([0, 8, 3, 6, 12, 3], np.uint32))
    p2.add_term([(p2.add_list([1], [[(6, 0)]]), 80.0)])
    assert gpu_merge(p2)[0].tolist() == [(1, 77.0, 0, 77)]  # uint8(77.91719), ft_generic.cc:327


def test_random_problems_match_oracle():
    preselects = 0
    for seed in range(120):
        rng = np.random.default_rng(seed)
        kw = dict(total_docs=int(rng.integers(30, 3000)), nfields=1 + seed % 3, nterms=1 + seed % 4, removed_frac=0.05 * (seed % 2),
                  excluded_frac=0.05 * (seed % 3 == 0), field_boost_zero=(seed % 5 == 0))
        if seed % 4 == 1:
            kw["merge_limit"] = int(rng.integers(5, 60))
        p = random_problem(seed, **kw)
        for rst in (F.RANK_AND_ID, F.RANK_ONLY):
            a, _ = F.best_merge(p, rst)
            b, st = gpu_merge(p, rst)
            preselects += st["preselected"]
            assert_same_merge(a, b, rst, ctx=f"seed {seed} rst {rst}")
    assert preselects > 10


def test_config_knobs_and_bm25_variants():
    for seed in range(24):
        p = random_problem(1000 + seed, total_docs=400, nfields=2, nterms=2)
        p.cfg.update(bm25_type=seed % 3, bm25_k1=1.2 + 0.1 * (seed % 5), bm25_b=0.5 + 0.05 * (seed % 4), min_rank=seed % 40,
                     distance_weight=0.3, distance_boost=1.5, full_match_boost=1.3)
        p.field_cfg[0].update(bm25_weight=0.4, position_weight=0.3, term_len_weight=0.2, bm25_boost=1.2)
        assert_same_merge(F.best_merge(p)[0], gpu_merge(p)[0], F.RANK_AND_ID, ctx=f"seed {seed}")


def test_summation_of_ranks_by_fields():
    """FTConfig::summationRanksByFieldsRatio > 0 with needSumRank fields (phrasemergerimpl.h:21,58-78): the ranks of the other
    matching fields are added with geometric weights"""
    hit = 0
    for seed in range(40):
        rng = np.random.default_rng(5000 + seed)
        nfields = 2 + seed % 4
        p = random_problem(5000 + seed, total_docs=500, nfields=nfields, nterms=1 + seed % 3, max_pos=6)
        p.cfg["summation_ranks_by_fields_ratio"] = float(rng.choice([0.3, 0.5, 0.9, 1.0]))
        for t in p.terms:
            t["need_sum_rank"] = (rng.random(nfields) < 0.7).astype(np.uint8)
        a, _ = F.best_merge(p)
        b, _ = gpu_merge(p)
        assert_same_merge(a, b, F.RANK_AND_ID, ctx=f"seed {seed}")
        p.cfg["summation_ranks_by_fields_ratio"] = 0.0
        hit += int(len(a) != len(F.best_merge(p)[0]) or (a["normalized_proc"] != F.best_merge(p)[0]["normalized_proc"][:len(a)]).any())
    assert hit > 5  # the knob changes results


def test_multi_word_synonyms_match_reference(ref_tape):
    """Merger::Merge with QueryMergeData::synonyms (mergerimpl.h:510-560, restricting mask :352-363, preselect :392-396): documents
    reached only through a synonym stay iff they hold all of its terms; suppressed subterms only count."""
    kept_by_syn = preselects = 0
    for seed in range(60):
        rng = np.random.default_rng(7000 + seed)
        kw = dict(total_docs=int(rng.integers(60, 2500)), nfields=1 + seed % 3, nterms=1 + seed % 3, removed_frac=0.05 * (seed % 2),
                  excluded_frac=0.05 * (seed % 3 == 0))
        if seed % 4 == 1:
            kw["merge_limit"] = int(rng.integers(10, 80))
        p = add_random_synonyms(random_problem(7000 + seed, **kw), seed, nsyn=1 + seed % 2)
        plain = random_problem(7000 + seed, **kw)
        for rst in (F.RANK_AND_ID, F.RANK_ONLY):
            a = ref_tape(lambda: merge_digest(F.ref_merge(p, rst)[0], rst), p, rst)
            b, st = gpu_merge(p, rst)
            preselects += st["preselected"]
            assert_same_merge_as_digest(a, b, rst, ctx=f"seed {seed} rst {rst}")
        # documents the reference keeps only because of the synonym
        kept_by_syn += ref_tape(lambda: len(set(F.ref_merge(p, F.RANK_ONLY)[0]["id"].tolist()) - set(F.ref_merge(plain)[0]["id"].tolist())) > 0,
                                p, plain)
    assert kept_by_syn > 10 and preselects > 3


def test_phrases_match_reference(ref_tape):
    """PhraseMerger (phrasemerger.h:285-399, phrasemergerimpl.h:166-312) + Merger::mergePhrase (mergerimpl.h:41-90) on the device:
    phrases drawn from a token corpus, 2-3 terms with distances 1-3 and variant subterms in the caller's order, mixed with plain terms
    under OR / AND / NOT, with and without the merge-limit cut-off, removed / excluded documents, multi-word synonyms"""
    nonempty = preselects = 0
    for seed in range(70):
        p = corpus_problem(seed, total_docs=300 + 17 * seed, nfields=1 + seed % 3, merge_limit=(30 if seed % 4 == 1 else 20000),
                           removed_frac=0.05 * (seed % 2), excluded_frac=0.05 * (seed % 3 == 0), with_synonym=seed % 5 == 0)
        for rst in (F.RANK_AND_ID, F.RANK_ONLY):
            a = ref_tape(lambda: merge_digest(F.ref_merge(p, rst)[0], rst), p, rst)
            b, st = gpu_merge(p, rst)
            preselects += st["preselected"]
            assert_same_merge_as_digest(a, b, rst, ctx=f"seed {seed} rst {rst}")
        nonempty += len(b) > 0
    assert nonempty > 60 and preselects > 3
    import reindexer_b200 as rx
    q = corpus_problem(3)
    q.terms = [dict(q.terms[0], phrase_num=9)]  # a one-term phrase
    with pytest.raises(rx.RxGpuError):
        gpu_merge(q)


def test_empty_and_degenerate_queries():
    p = random_problem(5, total_docs=100, nterms=1)
    p.terms[0]["op"] = F.OP_NOT  # a lone NOT term: Empty()
    assert len(gpu_merge(p)[0]) == 0 and len(F.best_merge(p)[0]) == 0
    p = random_problem(6, total_docs=100, nterms=2, ops=[F.OP_AND, F.OP_AND])  # pure AND: never preselects (estimate 0)
    assert_same_merge(F.best_merge(p)[0], gpu_merge(p)[0], F.RANK_AND_ID)
    p = random_problem(7, total_docs=100, nterms=2, ops=[F.OP_OR, F.OP_NOT])
    assert_same_merge(F.best_merge(p)[0], gpu_merge(p)[0], F.RANK_AND_ID)


def test_larger_corpus_three_term_or_with_preselect():
    """BASELINE config 3 in miniature: 3-term OR with document frequencies 10% / 1% / 0.1%, more candidates than merge_limit,
    top-100 of the final (rank desc, id asc) order."""
    total, rng = 400_001, np.random.default_rng(3)
    words = rng.poisson(100, size=(total, 1)).astype(np.uint32) + 1
    words[0] = 0
    p = F.FtProblem(total, words)
    for df in (0.10, 0.01, 0.001):
        docs = np.sort(rng.choice(np.arange(1, total), size=int(df * (total - 1)), replace=False)).astype(np.uint32)
        npos = rng.integers(1, 4, size=len(docs))
        begin = np.concatenate([[0], np.cumsum(npos)]).astype(np.uint32)
        pos = np.zeros(begin[-1], np.uint32)
        for i in range(len(docs)):  # ascending distinct positions inside the document
            pos[begin[i]:begin[i + 1]] = np.sort(rng.choice(int(words[docs[i], 0]), size=min(int(npos[i]), int(words[docs[i], 0])),
                                                            replace=False))[:npos[i]] if words[docs[i], 0] >= npos[i] else np.arange(npos[i])
        p.add_term([(p.add_list_arrays(docs, begin, pos), 100.0)], op=F.OP_OR)
    a, ns = F.best_merge(p)
    b, st = gpu_merge(p)
    assert st["preselected"] == 1 and len(a) > 1000
    assert_same_merge(a, b, F.RANK_AND_ID)
    assert (F.after_select_order(a)[:100] == F.after_select_order(b)[:100]).all()


def test_packed_posting_lists_give_the_same_merge(ref_tape):
    """lists handed over in the reference's packed container format (PackedIdRelVec bytes from the reference's own encoder, committed
    in tests/golden/packed_golden.npz for one case and in tests/golden/ref_tapes/ for random problems)"""
    g = np.load(os.path.join(ROOT, "tests", "golden", "packed_golden.npz"))
    d, b, pp = (g[f"multi_field/{k}"] for k in ("doc_ids", "pos_begin", "positions"))
    total = int(d.max()) + 2
    rng = np.random.default_rng(3)
    words = rng.integers(3000, 4000, size=(total, 5)).astype(np.uint32)
    words[0] = 0
    p = F.FtProblem(total, words)
    p.add_term([(p.add_list_arrays(d, b, pp), 100.0)], field_boosts=np.ones(5, np.float32))
    a, _ = gpu_merge(p)
    c, _ = gpu_merge(p, packed=[g["multi_field/packed"]])
    assert_same_merge(a, c, F.RANK_AND_ID)
    assert len(a) > 100
    e, _ = gpu_merge(p, packed=[g["multi_field/packed"]], batch=True)  # decoded on the device
    assert_same_merge(a, e, F.RANK_AND_ID)
    for seed in range(10):
        q = random_problem(1000 + seed, total_docs=1500, nfields=1 + seed % 3, nterms=2 + seed % 2)
        packed = [ref_tape(lambda: F.ref_pack_list(*lst), *lst) for lst in q.lists]
        x, _ = F.best_merge(q)
        y, _ = gpu_merge(q, packed=packed)
        assert_same_merge(x, y, F.RANK_AND_ID, ctx=f"seed {seed}")
        z, _ = gpu_merge(q, packed=packed, batch=True)
        assert_same_merge(x, z, F.RANK_AND_ID, ctx=f"seed {seed} device decode")


def test_device_decode_of_packed_lists_batch(ref_tape):
    """rxgpu_ft_add_postings_packed_batch: many lists decoded by the device in one call give the lists the host decoder gives (checked
    through merges over every list), a list above the per-thread size limit takes the host decoder inside the same batch, and a
    malformed stream rejects the whole batch"""
    import reindexer_b200 as rx
    g = np.load(os.path.join(ROOT, "tests", "golden", "packed_golden.npz"))
    names = sorted({k.split("/")[0] for k in g.files if k.endswith("/packed")})
    total = max(max(int(g[f"{n}/doc_ids"].max()) for n in names) + 2, 60000)
    nfields = max(int((g[f"{n}/positions"] >> 24).max()) for n in names) + 1
    rng = np.random.default_rng(5)
    words = rng.integers(3000, 4000, size=(total, nfields)).astype(np.uint32)
    words[0] = 0
    avg = words[1:].mean(axis=0).astype(np.float32)
    # a long list (> 256 KiB of stream) next to the short golden ones, packed by the reference's own encoder
    big_docs = np.arange(1, min(total, 200_000), dtype=np.uint32)
    big_begin = np.arange(0, 3 * len(big_docs) + 1, 3, dtype=np.uint32)
    # strictly ascending within a document, field 0; the same in every document, so that the stored stream compresses
    big_pos = np.tile(np.array([0, 5, 11], np.uint32), len(big_docs))
    streams = [g[f"{n}/packed"] for n in names]
    counts = [len(g[f"{n}/doc_ids"]) for n in names]
    soa = [(g[f"{n}/doc_ids"], g[f"{n}/pos_begin"], g[f"{n}/positions"]) for n in names]
    big_stream = ref_tape(lambda: F.ref_pack_list(big_docs, big_begin, big_pos), big_docs, big_begin, big_pos)
    assert len(big_stream) > (256 << 10)
    streams.append(big_stream)
    counts.append(len(big_docs))
    soa.append((big_docs, big_begin, big_pos))
    a = rx.GpuFtIndex(total, words, avg)
    ids_a = a.add_postings_packed_batch(streams * 40, counts * 40)  # 40 copies: a few hundred lists in one call
    b = rx.GpuFtIndex(total, words, avg)
    ids_b = [b.add_postings(*t) for t in soa]
    p = F.FtProblem(total, words)
    for k in range(len(soa)):
        term = dict(op=F.OP_OR, boost=1.0, term_len_boost=1.0, field_boosts=np.ones(nfields, np.float32), procs=[100.0])
        for copy in (0, 17, 39):
            ra = a.merge(p.cfg, p.field_cfg, [dict(term, postings=[ids_a[copy * len(soa) + k]])])
            rb = b.merge(p.cfg, p.field_cfg, [dict(term, postings=[ids_b[k]])])
            assert_same_merge(ra, rb, F.RANK_AND_ID, ctx=f"list {k} copy {copy}")
            assert len(ra) > 0
    bad = [streams[0], streams[1][:-1] if len(streams) > 1 else streams[0][:-1]]
    c = rx.GpuFtIndex(total, words, avg)
    with pytest.raises(rx.RxGpuError):
        c.add_postings_packed_batch(bad, [counts[0], counts[1] if len(counts) > 1 else counts[0]])
    assert c.add_postings_packed_batch([streams[0]], [counts[0]]) == [0]  # nothing of the failed batch stayed


def test_select_after_merge_on_device():
    """rxgpu_ft_select = merge + postProcessResults + IndexText::afterSelect + sortAfterSelect on the device: the first `limit` rows in
    (rank desc, row id asc) order must equal the oracle's merge followed by the reference's ordering rule (indextext.cc:480-520), with
    a vdoc -> row ids expansion and external row statuses too"""
    import reindexer_b200 as rx

    for seed in range(30):
        rng = np.random.default_rng(7000 + seed)
        total = int(rng.integers(200, 4000))
        p = random_problem(7000 + seed, total_docs=total, nfields=1 + seed % 2, nterms=1 + seed % 3,
                           merge_limit=int(rng.integers(20, 200)) if seed % 3 == 0 else 20000)
        ref, _ = F.best_merge(p, F.RANK_AND_ID)
        ft = rx.GpuFtIndex(p.total_docs, p.words, p.avg, p.removed)
        ids = [ft.add_postings(d, b, q) for d, b, q in p.lists]
        terms = [dict(t, postings=[ids[int(x)] for x in t["postings"]]) for t in p.terms]
        # (a) identity rows: vdoc i = row i
        want = F.after_select_order(ref)
        for limit in (10, 100, len(ref) + 5):
            got_ids, got_ranks, n = ft.select(p.cfg, p.field_cfg, terms, limit, excluded=p.excluded)
            assert n == len(want)
            m = min(limit, len(want))
            assert (got_ids == want["id"][:m]).all() and (got_ranks == want["normalized_proc"][:m].astype(np.float32)).all(), (seed, limit)
        got_ids, got_ranks, n = ft.select(p.cfg, p.field_cfg, terms, len(ref) + 5, excluded=p.excluded, rank_sort_type=F.ID_ONLY)
        o = np.argsort(ref["id"], kind="stable")
        assert (got_ids == ref["id"][o]).all() and (got_ranks == ref["normalized_proc"][o].astype(np.float32)).all()
        # (b) vdocs that own several rows (duplicated documents share one vdoc) + external statuses on rows
        nrows_of = rng.integers(0, 4, size=total).astype(np.uint32)
        nrows_of[0] = 0
        row_begin = np.concatenate([[0], np.cumsum(nrows_of)]).astype(np.uint32)
        row_ids = rng.permutation(int(row_begin[-1])).astype(np.int32)
        status = (rng.random(int(row_begin[-1]) + 1) < 0.8).astype(np.uint8)
        ft.set_rows(row_begin, row_ids)
        exp = []
        for e in ref:
            for r in row_ids[row_begin[e["id"]]:row_begin[e["id"] + 1]]:
                if status[r]:
                    exp.append((int(r), int(e["normalized_proc"])))
        exp.sort(key=lambda x: (-x[1], x[0]))
        got_ids, got_ranks, n = ft.select(p.cfg, p.field_cfg, terms, 50, excluded=p.excluded, row_status=status)
        assert n == len(exp)
        assert got_ids.tolist() == [x[0] for x in exp[:50]] and got_ranks.tolist() == [float(x[1]) for x in exp[:50]], seed
        ft.close()
