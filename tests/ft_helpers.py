"""Random ft_fast merge problems for the oracle pin tests and the GPU parity tests (test infrastructure)."""
import numpy as np

from oracle import ft_oracle as F


def random_problem(seed, total_docs=400, nfields=1, nterms=3, max_sub=3, density=0.2, merge_limit=20000, ops=None, removed_frac=0.0,
                   excluded_frac=0.0, field_boost_zero=False, max_pos=3, doc_len=(3, 40)):
    rng = np.random.default_rng(seed)
    words = rng.integers(doc_len[0], doc_len[1], size=(total_docs, nfields)).astype(np.uint32)
    words[0] = 0
    removed = (rng.random(total_docs) < removed_frac).astype(np.uint8) if removed_frac else None
    excluded = (rng.random(total_docs) < excluded_frac).astype(np.uint8) if excluded_frac else None
    p = F.FtProblem(total_docs, words, removed=removed, excluded=excluded)
    p.cfg["merge_limit"] = merge_limit
    procs_pool = [100.0, 90.0, 85.0, 80.0, 72.0, 65.0, 57.0, 50.0, 43.0, 31.0]
    for t in range(nterms):
        nsub = int(rng.integers(1, max_sub + 1))
        subs = []
        procs = rng.choice(procs_pool, size=nsub, replace=False)  # distinct procs: SortSubterms is unstable for ties
        for s in range(nsub):
            dens = density * float(rng.uniform(0.3, 1.5)) / (1 + s)
            ndocs = max(1, int(dens * (total_docs - 1)))
            docs = np.sort(rng.choice(np.arange(1, total_docs), size=min(ndocs, total_docs - 1), replace=False))
            pos_lists = []
            for d in docs:
                npos = int(rng.integers(1, max_pos + 1))
                pp = []
                for _ in range(npos):
                    f = int(rng.integers(0, nfields))
                    pp.append((int(rng.integers(0, max(int(words[d, f]), 1))), f))
                pos_lists.append(pp)
            subs.append((p.add_list(docs, pos_lists), float(procs[s])))
        op = ops[t] if ops else int(rng.choice([F.OP_OR, F.OP_OR, F.OP_AND, F.OP_NOT])) if t else F.OP_OR
        fb = np.ones(nfields, np.float32)
        if nfields > 1:
            fb = rng.choice([1.0, 0.5, 2.0, 1.5], size=nfields).astype(np.float32)
            if field_boost_zero:
                fb[int(rng.integers(0, nfields))] = 0.0
        p.add_term(subs, op=op, boost=float(rng.choice([1.0, 1.0, 0.7, 1.3])), term_len_boost=float(rng.choice([1.0, 0.8, 0.5])),
                   field_boosts=fb)
    return p


def add_random_synonyms(p, seed, nsyn=2, density=0.25, suppress=True):
    """Multi-word synonyms on top of random_problem: every synonym has 2-3 terms of 1-2 subterms each, is attached to one or two
    OR / AND query parts (PhraseOrTerm::AddSynonymId), and may carry a suppressed subterm that re-uses a posting list of the query
    (what QueryMergeData::SupressDuplicatesInSynonyms marks)."""
    rng = np.random.default_rng(seed ^ 0x5A17)
    total_docs, nfields = p.total_docs, p.nfields
    hosts = [i for i, t in enumerate(p.terms) if t["op"] != F.OP_NOT]
    for y in range(nsyn):
        terms = []
        for _ in range(int(rng.integers(2, 4))):
            subs = []
            procs = rng.choice([60.0, 52.0, 45.0, 38.0, 33.0], size=2, replace=False)
            for s_ in range(int(rng.integers(1, 3))):
                ndocs = max(1, int(density * float(rng.uniform(0.4, 1.4)) * (total_docs - 1)))
                docs = np.sort(rng.choice(np.arange(1, total_docs), size=min(ndocs, total_docs - 1), replace=False))
                pos_lists = [[(int(rng.integers(0, max(int(p.words[d, f]), 1))), f) for f in [int(rng.integers(0, nfields))]
                              for _ in range(int(rng.integers(1, 3)))] for d in docs]
                subs.append((p.add_list(docs, pos_lists), float(procs[s_])))
            if suppress and rng.random() < 0.4:  # a word of the query repeated inside the synonym
                host = p.terms[int(rng.choice(hosts))]
                subs.append((int(host["postings"][0]), 29.0, True))
            terms.append(dict(subterms=subs, op=F.OP_OR, boost=float(rng.choice([1.0, 0.8])), term_len_boost=1.0,
                              field_boosts=np.ones(nfields, np.float32)))
        sid = p.add_synonym(terms)
        for h in rng.choice(hosts, size=min(len(hosts), int(rng.integers(1, 3))), replace=False):
            p.terms[int(h)]["synonym_ids"] = np.append(p.terms[int(h)]["synonym_ids"], np.uint32(sid)).astype(np.uint32)
    return p


def corpus_problem(seed, total_docs=600, nfields=2, vocab=24, merge_limit=20000, removed_frac=0.0, excluded_frac=0.0, with_synonym=False):
    """A problem built from an actual token corpus, so that PHRASES match: every document holds random words of a small vocabulary in
    every field; posting lists are derived from it.  The query mixes one or two phrases (2-3 terms, distances 1-3, 1-2 variant subterms
    per term, in the caller's -- unsorted -- order) with plain terms under OR / AND / NOT."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(4, 22, size=(total_docs, nfields))
    lens[0] = 0
    words = lens.astype(np.uint32)
    removed = (rng.random(total_docs) < removed_frac).astype(np.uint8) if removed_frac else None
    excluded = (rng.random(total_docs) < excluded_frac).astype(np.uint8) if excluded_frac else None
    p = F.FtProblem(total_docs, words, removed=removed, excluded=excluded)
    p.cfg["merge_limit"] = merge_limit
    tokens = [[rng.integers(0, vocab, size=lens[d, f]) for f in range(nfields)] for d in range(total_docs)]
    list_of_word = {}

    def postings(w):
        if w not in list_of_word:
            docs, pos_lists = [], []
            for d in range(1, total_docs):
                pp = [(int(i), f) for f in range(nfields) for i in np.nonzero(tokens[d][f] == w)[0]]
                if pp:
                    docs.append(d)
                    pos_lists.append(pp)
            list_of_word[w] = p.add_list(docs, pos_lists)
        return list_of_word[w]

    def subterms(primary):
        subs = [(postings(int(primary)), float(rng.choice([100.0, 90.0, 85.0])))]
        if rng.random() < 0.5:  # a variant (typo / stem) of lower relevancy, possibly listed FIRST
            v = (postings(int(rng.integers(0, vocab))), float(rng.choice([72.0, 65.0, 57.0])))
            subs = [v] + subs if rng.random() < 0.5 else subs + [v]
        return subs

    nparts = int(rng.integers(1, 4))
    phrase_num = 0
    for part in range(nparts):
        op = F.OP_OR if part == 0 else int(rng.choice([F.OP_OR, F.OP_OR, F.OP_AND, F.OP_NOT]))
        fb = rng.choice([1.0, 0.5, 2.0], size=nfields).astype(np.float32) if nfields > 1 else np.ones(1, np.float32)
        if part == 0 or rng.random() < 0.5:  # a phrase taken from a real document, so that it occurs
            phrase_num += 1
            d, f = int(rng.integers(1, total_docs)), int(rng.integers(0, nfields))
            n = int(rng.integers(2, 4))
            at = int(rng.integers(0, max(1, lens[d, f] - 2 * n)))
            step = int(rng.integers(1, 3))
            chosen = [int(tokens[d][f][min(at + k * step, lens[d, f] - 1)]) for k in range(n)]
            for k, w in enumerate(chosen):
                p.add_term(subterms(w), op=op, boost=float(rng.choice([1.0, 0.8])), term_len_boost=float(rng.choice([1.0, 0.9])),
                           field_boosts=fb, phrase_num=phrase_num, distance=int(rng.integers(1, 4)) if k else 0)
        else:
            syn = ()
            if with_synonym and op != F.OP_NOT:
                syn = (p.add_synonym([dict(subterms=[(postings(int(rng.integers(0, vocab))), 45.0)], field_boosts=np.ones(nfields, np.float32))
                                      for _ in range(2)]),)
            p.add_term(subterms(int(rng.integers(0, vocab))), op=op, boost=1.0, term_len_boost=1.0, field_boosts=fb, synonym_ids=syn)
    return p


def assert_same_merge(a, b, rank_sort_type, ctx=""):
    """a, b: MERGE_INFO arrays.  RankAndID / IDOnly keep the merge order (deterministic); RankOnly / IDAndPositions are sorted by an
    unstable sort, so equal ranks compare as sets."""
    assert len(a) == len(b), (ctx, len(a), len(b))
    if rank_sort_type in (F.RANK_AND_ID, F.ID_ONLY):
        assert (a["id"] == b["id"]).all(), ctx
        assert (a["normalized_proc"] == b["normalized_proc"]).all(), (ctx, a[:8], b[:8])
        assert (a["field"] == b["field"]).all(), ctx
        assert (a["proc"] == b["proc"]).all(), ctx
    else:
        assert (a["normalized_proc"] == b["normalized_proc"]).all(), ctx
        oa, ob = np.lexsort((a["id"], -a["normalized_proc"].astype(int))), np.lexsort((b["id"], -b["normalized_proc"].astype(int)))
        assert (a["id"][oa] == b["id"][ob]).all() and (a["field"][oa] == b["field"][ob]).all(), ctx


def merge_digest(res, rank_sort_type):
    """digest of what assert_same_merge compares: equal digests <=> assert_same_merge passes (stored reference answers stay small)"""
    from helpers import digest

    if rank_sort_type in (F.RANK_AND_ID, F.ID_ONLY):
        return digest(res["id"], res["normalized_proc"], res["field"], res["proc"])
    o = np.lexsort((res["id"], -res["normalized_proc"].astype(int)))
    return digest(res["normalized_proc"], res["id"][o], res["field"][o])


def assert_same_merge_as_digest(want, res, rank_sort_type, ctx=""):
    assert merge_digest(res, rank_sort_type) == want, (ctx, len(res), res[:8])


def load_golden_problem(g, name):
    """Rebuild an FtProblem from tests/golden/ft_golden.npz (inputs are stored, not regenerated)."""
    words = g[f"{name}/words"]
    rem, exc = g[f"{name}/removed"], g[f"{name}/excluded"]
    p = F.FtProblem(words.shape[0], words, avg=g[f"{name}/avg"], removed=rem if len(rem) else None, excluded=exc if len(exc) else None)
    for i in range(int(g[f"{name}/nlists"])):
        p.add_list_arrays(g[f"{name}/list{i}/docs"], g[f"{name}/list{i}/begin"], g[f"{name}/list{i}/pos"])
    for i in range(int(g[f"{name}/nterms"])):
        op, boost, tlb = g[f"{name}/term{i}/scalars"]
        p.terms.append(dict(op=int(op), boost=float(boost), term_len_boost=float(tlb), field_boosts=g[f"{name}/term{i}/field_boosts"],
                            postings=g[f"{name}/term{i}/postings"], procs=g[f"{name}/term{i}/procs"]))
    p.cfg["merge_limit"] = int(g[f"{name}/merge_limit"])
    return p


def gpu_merge(prob, rank_sort_type=F.RANK_AND_ID, packed=None, batch=False):
    """Run one problem through the product (rxgpu_ft_*); returns (result, stats).  packed: per-list byte streams of the reference's
    PackedIdRelVec -- the lists are then uploaded through rxgpu_ft_add_postings_packed."""
    import reindexer_b200 as rx

    ft = rx.GpuFtIndex(prob.total_docs, prob.words, prob.avg, prob.removed)
    if packed is not None and batch:  # the raw streams travel to the device and are decoded there (rxgpu_ft_add_postings_packed_batch)
        ids = ft.add_postings_packed_batch(packed, [len(l[0]) for l in prob.lists])
    elif packed is not None:
        ids = [ft.add_postings_packed(packed[i], len(prob.lists[i][0])) for i in range(len(prob.lists))]
    else:
        ids = [ft.add_postings(d, b, p) for d, b, p in prob.lists]
    terms = [dict(t, postings=[ids[int(x)] for x in t["postings"]]) for t in prob.terms]
    syns = [[dict(t, postings=[ids[int(x)] for x in t["postings"]]) for t in syn] for syn in prob.synonyms]
    res = ft.merge(prob.cfg, prob.field_cfg, terms, excluded=prob.excluded, rank_sort_type=rank_sort_type, synonyms=syns or None)
    st = ft.last_stats()
    ft.close()
    return res, st
