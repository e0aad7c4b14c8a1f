"""CPU tests: the oracle restatement (oracle/knn_port.c) is pinned against
 (a) the committed golden fixtures, which are outputs of the reference's own code (tests/golden/make_knn_golden.py), and
 (b) the reference's own translation units (oracle/_ref), through their outputs stored in tests/golden/ref_tapes/."""
import numpy as np
import pytest
from conftest import GOLDEN_SYNTH_CASES, GOLDEN_TIE_CASES
from helpers import ATOL, RTOL, prep_query

from oracle import oracle as O


def test_synth_twins_agree():
    a = O.synth(0x5EED0001, 12345, 4097)
    b = np.empty(4097, np.float32)
    O.port_lib().port_synth_fill(0x5EED0001, 12345, 4097, b.ctypes.data_as(O._f32p))
    assert (a == b).all()
    big = O.synth(7, 0, 1 << 18)
    assert abs(big.std() - 0.25) < 0.005 and abs(big.mean()) < 0.005


@pytest.mark.parametrize("name", GOLDEN_SYNTH_CASES)
def test_port_matches_golden_synth(golden, name):
    metric, n, dim, k, nq, seed = (int(x) for x in golden[f"{name}/meta"])
    vecs, queries, labels = O.synth_matrix(seed, n, dim), O.synth_matrix(seed + 1, nq, dim), O.row_labels(n)
    bf = O.PortBF(metric, dim, n)
    assert bf.add_batch(labels, vecs) == 0
    for i in range(nq):
        d, l = bf.search_knn(prep_query(metric, queries[i], use_ref=False), k)
        cnt = int(golden[f"{name}/count"][i])
        assert len(d) == cnt == min(k, n)
        assert (l == golden[f"{name}/label"][i, :cnt]).all()
        assert np.allclose(d, golden[f"{name}/dist"][i, :cnt], rtol=RTOL, atol=ATOL)
    rd, rl = bf.search_range(prep_query(metric, queries[0], use_ref=False), float(golden[f"{name}/range_radius"]))
    assert (rl == golden[f"{name}/range_label"]).all()
    assert np.allclose(rd, golden[f"{name}/range_dist"], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("name", GOLDEN_TIE_CASES)
def test_port_matches_golden_ties(golden, name):
    metric, n, dim, k, nq, _ = (int(x) for x in golden[f"{name}/meta"])
    bf = O.PortBF(metric, dim, n)
    assert bf.add_batch(golden[f"{name}/labels"], golden[f"{name}/vecs"]) == 0
    for l in golden[f"{name}/removes"]:
        bf.remove(int(l))
    for i in range(nq):
        d, l = bf.search_knn(prep_query(metric, golden[f"{name}/queries"][i], use_ref=False), k)
        assert (l == golden[f"{name}/label"][i]).all(), (name, i)
        assert np.allclose(d, golden[f"{name}/dist"][i], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("metric", [O.L2, O.IP, O.COS])
def test_port_matches_reference_build(ref_tape, metric):
    rng = np.random.default_rng(metric + 11)
    n, dim, k = 2500, 72, 12
    vecs, labels = O.synth_matrix(100 + metric, n, dim), O.row_labels(n)
    p = O.PortBF(metric, dim, n + 5)
    r = ref_tape.proxy(lambda: O.RefBF(metric, dim, n + 5), metric, dim, n + 5)  # the reference's map
    p.add_batch(labels, vecs)
    r.add_batch(labels, vecs)
    for l in labels[rng.choice(n, 200, replace=False)]:
        p.remove(int(l))
        r.remove(int(l))
    # upsert over existing labels and fresh ones
    newv = O.synth_matrix(900 + metric, 50, dim)
    newl = np.concatenate([labels[rng.choice(n, 25, replace=False)], O.row_labels(25, first_row=n + 100)])
    p.add_batch(newl, newv)
    r.add_batch(newl, newv)
    assert p.size() == r.size() and p.element_size() == r.element_size() == dim * 4 + 8
    for q in O.synth_matrix(200 + metric, 16, dim):
        qp = prep_query(metric, q, False)
        qr = ref_tape(lambda: prep_query(metric, q, True), q) if metric == O.COS else q  # the reference's own normalisation
        dp, lp = p.search_knn(qp, k)
        dr, lr = r.search_knn(qr, k)
        assert (lp == lr).all()
        assert np.allclose(dp, dr, rtol=RTOL, atol=ATOL)
        radius = float((dr[5] + dr[6]) / 2)
        dp, lp = p.search_range(qp, radius)
        dr2, lr2 = r.search_range(qr, radius)
        assert (lp == lr2).all() and len(lp) == 6
    # capacity / resize errors
    assert p.add(vecs[0], 1 << 50) == 0
    small_p, small_r = O.PortBF(metric, dim, 2), ref_tape.proxy(lambda: O.RefBF(metric, dim, 2), metric, dim, 2)
    for i in range(2):
        assert small_p.add(vecs[i], i) == 0 and small_r.add(vecs[i], i) == 0
    assert small_p.add(vecs[2], 2) == 1 and small_r.add(vecs[2], 2) == 1
    assert "exceeds the specified limit" in small_r._err()
    assert small_p.resize(1) == 1 and small_r.resize(1) == 1


def test_normalize_shortcut(ref_tape):
    # tools/normalize.cc:19: vectors whose squared norm is within 1e-5 of 1 (or zero) keep coefficient exactly 1.0
    x = np.zeros(8, np.float32)
    assert O.normalize_copy(x, False)[1] == 1.0
    x[0] = 1.0
    assert O.normalize_copy(x, False)[1] == 1.0
    x[0] = 3.0
    out, k = O.normalize_copy(x, False)
    assert abs(k - 1 / 3) < 1e-7 and abs(out[0] - 1.0) < 1e-6
    for v in (np.zeros(8, np.float32), x, O.synth(3, 0, 100)):
        a, ka = O.normalize_copy(v, False)
        b, kb = ref_tape(lambda: O.normalize_copy(v, True), v)
        assert np.allclose(a, b, rtol=1e-6) and abs(ka - kb) <= 1e-6 * abs(kb)


def test_select_postprocess_properties():
    """checkOrdering of the reference's own test (cpp_src/gtests/tests/unit/float_vector_index.cc:32-86): ranks monotone,
    equal ranks ordered by ascending row id; IP/Cosine ranks have flipped sign; array fields are de-duplicated by row."""
    d = np.array([1.0, 1.0, 1.0, 2.0, 3.0, 3.0], np.float32)
    lab = (np.array([9, 4, 7, 1, 8, 2], np.uint64) << np.uint64(32))
    # best-first as the heap drains: equal distances arrive in ascending label order
    order = np.lexsort((lab, d))
    ids, ranks = O.select_postprocess(O.L2, d[order], lab[order])
    assert ids.tolist() == [4, 7, 9, 1, 2, 8] and ranks.tolist() == sorted(d.tolist())
    ids, ranks = O.select_postprocess(O.IP, d[order], lab[order])
    assert ranks.tolist() == (-np.sort(d)).tolist()
    # array field: labels rowId<<32|arrayIdx, duplicates of a row keep the best
    lab2 = np.array([(5 << 32) | 1, (5 << 32) | 0, (3 << 32) | 2, (5 << 32) | 2], np.uint64)
    d2 = np.array([0.5, 0.6, 0.7, 0.8], np.float32)
    ids, ranks = O.select_postprocess(O.L2, d2, lab2, is_array=True)
    assert ids.tolist() == [5, 3] and np.allclose(ranks, [0.5, 0.7])
    # k + radius => trimmed to k
    ids, _ = O.select_postprocess(O.L2, d[order], lab[order], k=2, has_radius=True)
    assert len(ids) == 2


@pytest.mark.skipif(not O.ref_ivf_available(), reason="needs oracle/_ref (reference FAISS build)")
def test_reference_ivf_oracle_is_self_consistent():
    """the IVF oracle is the reference's own FAISS; pin the facade's export against its search: scanning the exported lists of the
    nprobe nearest exported centroids by brute force reproduces IndexIVFFlat::search"""
    n, dim, nlist, k, nprobe = 4000, 24, 16, 10, 3
    vecs, labels = O.synth_matrix(901, n, dim), O.row_labels(n)
    def coef(m):  # CalculateL2Module: 1/||v|| with the "already normalised" shortcut (tools/normalize.cc:10-23)
        s2 = (m.astype(np.float64) ** 2).sum(axis=1)
        return np.where(np.abs(1.0 - s2) > 1e-5, 1.0 / np.sqrt(np.maximum(s2, 1e-30)), 1.0).astype(np.float32)

    for metric in (O.L2, O.IP, O.COS):
        ref = O.RefIvf(metric, dim, nlist)
        ref.train_add(labels, vecs)
        st = ref.export()
        begin = np.concatenate([[0], np.cumsum(st["list_sizes"].astype(np.int64))])
        for q in O.synth_matrix(902, 12, dim):
            if metric == O.COS:
                q = O.normalize_copy(q)[0]  # the caller normalises the key (ivf_index.cc: NormalizeCopyVector)
            if metric == O.L2:
                cd = ((st["centroids"] - q) ** 2).sum(axis=1)
            else:
                cd = -(st["centroids"] @ q) * (coef(st["centroids"]) if metric == O.COS else 1.0)
            probe = np.argsort(cd, kind="stable")[:nprobe]
            rows = np.concatenate([np.arange(begin[c], begin[c + 1]) for c in probe])
            sub = st["vecs"][rows]
            dd = ((sub - q) ** 2).sum(axis=1) if metric == O.L2 else -(sub @ q) * (coef(sub) if metric == O.COS else 1.0)
            order = np.argsort(dd, kind="stable")[:k]
            dr, lr = ref.search(q, k, nprobe)
            assert (st["labels"][rows[order]] == lr).all()
            assert np.allclose(dd[order], dr if metric == O.L2 else -dr, rtol=1e-4, atol=1e-5)


@pytest.mark.skipif(not O.ref_knn_available(), reason="needs oracle/_ref (reference HNSW build)")
def test_reference_streaming_search_contract():
    """groundwork for the device streaming search (SURVEY §8 a10): the contract of the reference's Begin/ContinueStreamingSearch, pinned
    on its own code -- batches never repeat a label, every batch is sorted, the stream ends exhausted, and on a connected graph it
    eventually yields every row; the first batch is close to (not necessarily equal to) the k best of SearchKnn"""
    n, dim = 3000, 24
    vecs, labels = O.synth_matrix(1501, n, dim), O.row_labels(n)
    ref = O.RefHnsw(O.L2, dim, n, M=16, ef_construction=200, seed=100, multithread=False)
    ref.add_batch(labels, vecs)
    q = O.synth_matrix(1502, 1, dim)[0]
    seen, batches = [], 0
    for d, l in ref.stream(q, 64, ef=100):
        assert (np.diff(d) >= 0).all()
        seen += l.tolist()
        batches += 1
    assert len(seen) == len(set(seen)), "a label was streamed twice"
    assert len(seen) >= 0.99 * n and batches >= n // 64
    dk, lk = ref.search_knn(q, 10, 100)
    first = next(iter(ref.stream(q, 10, ef=100)))[1]
    assert len(set(first.tolist()) & set(lk.tolist())) >= 8


@pytest.mark.skipif(not O.ref_knn_available(), reason="needs oracle/_ref (reference HNSW build)")
@pytest.mark.parametrize("metric", [O.L2, O.IP])
def test_reference_sq8_distance_formula(metric):
    """groundwork for SQ8 on the device (SURVEY §8 f2): the reference's quantised distance is integer arithmetic plus stored
    corrections -- alpha^2 * int_dist(u8, u8) + offset(query) + offset(row) (hnswlib.h:192-197, quantizer.h:93-125) -- so a dp4a
    kernel can reproduce it exactly.  Pinned on the reference's own quantised graph: codes, offsets and the quantised query are
    read back through the facade, the formula is restated here, and it must give the distances SearchKnn returns."""
    n, dim, k = 3000, 32, 10
    vecs, labels = O.synth_matrix(1601, n, dim), O.row_labels(n)
    g = O.RefHnsw(metric, dim, n, M=16, ef_construction=200, seed=100, multithread=False)
    g.add_batch(labels, vecs)
    sq = g.quantize()
    p = sq.params()
    codes, offs = sq.export()
    assert codes.shape == (n, dim) and abs(p["alpha"] - (p["maxQ"] - p["minQ"]) / 255.0) < 1e-6 * abs(p["alpha"])
    # the codes are the documented clamp((x - minQ) / alpha, 0, 255) truncated to u8
    expect = np.clip((vecs - p["minQ"]) / p["alpha"], 0.0, 255.0).astype(np.uint8)
    assert (codes == expect).mean() > 0.999  # fp rounding at the bin edges only
    for q in O.synth_matrix(1602, 8, dim):
        d, l = sq.search_knn(q, k, 64)
        cq, oq = sq.prepare_query(q)
        rows = (l >> np.uint64(32)).astype(np.int64)  # single-threaded build: internal id = insertion order = row id
        a = codes[rows].astype(np.int64)
        b = cq.astype(np.int64)[None, :]
        if metric == O.L2:
            mine = np.float32(p["alpha_2"]) * ((a - b) ** 2).sum(axis=1).astype(np.float32) + np.float32(oq) + offs[rows]
        else:
            mine = -(np.float32(p["alpha_2"]) * (a * b).sum(axis=1).astype(np.float32) + np.float32(oq) + offs[rows])
        assert np.allclose(mine, d, rtol=1e-5, atol=1e-5), (mine, d)
        # and the quantised search still finds most of the true neighbours
        exact = np.argsort(((vecs - q) ** 2).sum(axis=1) if metric == O.L2 else -(vecs @ q), kind="stable")[:k]
        assert len(set(rows.tolist()) & set(exact.tolist())) >= 6
