"""GPU tests of the HNSW search kernel (SURVEY.md §8 a9): a graph built by the reference's own CPU code (oracle/_ref, or its graph and
answers stored in tests/golden/ref_tapes/ where they are small enough) is
imported and searched on the device; results are compared with the reference's HierarchicalNSW::SearchKnn on the same graph
and with exact brute force (recall).  Bit parity of HNSW is only attainable with bit-identical distances (SURVEY §8a rule 7),
so the acceptance criteria are: nearly all queries return the identical top-k, recall@10 equals the reference's, and the
work counters (distance computations / hops) match the reference's own counters."""
import numpy as np
import pytest
from helpers import ATOL, RTOL, prep_query

import reindexer_b200 as rx
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def build(ref_tape, metric, n, dim, seed, M=16, efc=200):
    vecs, labels = O.synth_matrix(seed, n, dim), O.row_labels(n)
    ref = ref_tape.proxy(lambda: O.RefHnsw(metric, dim, n, M=M, ef_construction=efc, seed=100, multithread=False), metric, dim, n, M, efc)
    ref.add_batch(labels, vecs)  # single-threaded => deterministic graph, internal id == insertion order
    g = ref.export(with_vectors=False)
    assert (g["labels"] == labels).all()
    gpu = rx.GpuBruteforceSearch(metric, dim, n)
    gpu.add_points(labels, vecs)
    gpu.hnsw_import(g)
    return ref, gpu, vecs, labels


@pytest.mark.parametrize("metric,dim", [(rx.L2, 64), (rx.IP, 96), (rx.COS, 128)])
def test_hnsw_search_matches_reference_graph_search(ref_tape, metric, dim):
    n, k, ef, nq = 20000, 10, 128, 200
    ref, gpu, vecs, labels = build(ref_tape, metric, n, dim, 700 + metric)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(800 + metric, nq, dim)])
    d, l, c, st = gpu.hnsw_search_knn(queries, k, ef, with_stats=True)
    dr, lr, cr = ref.search_knn_batch(queries, k, ef, threads=4)
    assert (c == cr).all() and (c == k).all()
    same = sum(int((l[i] == lr[i]).all()) for i in range(nq))
    assert same >= 0.97 * nq, f"only {same}/{nq} queries returned the reference's exact top-{k}"
    ok = [i for i in range(nq) if (l[i] == lr[i]).all()]
    assert np.allclose(d[ok], dr[ok], rtol=RTOL, atol=ATOL)
    # recall@k against exact brute force (device), equal to the reference's own recall
    db, lb, _ = gpu.search_knn(queries, k)
    rec_gpu = np.mean([len(set(l[i]) & set(lb[i])) / k for i in range(nq)])
    rec_ref = np.mean([len(set(lr[i]) & set(lb[i])) / k for i in range(nq)])
    # i.i.d. Gaussian vectors are the worst case for any graph index (no cluster structure): the absolute recall is what the
    # reference's own search achieves on its own graph; the device search must reproduce it
    assert abs(rec_gpu - rec_ref) <= 0.01 and rec_gpu > 0.5, (rec_gpu, rec_ref)
    # work counters: same traversal => same number of distance evaluations and hops as the reference counts
    agree = 0
    for i in range(40):
        dc, hops = ref.search_metrics(queries[i], ef)
        agree += int(st[i, 0] == dc and st[i, 1] == hops)
    assert agree >= 36, agree


def test_hnsw_default_ef_small_k_and_errors(ref_tape):
    metric, n, dim = rx.L2, 3000, 32
    ref, gpu, vecs, labels = build(ref_tape, metric, n, dim, 900, M=8, efc=100)
    queries = O.synth_matrix(901, 50, dim)
    for k, ef in [(1, 0), (5, 0), (10, 10), (20, 7), (10, 1000)]:
        d, l, c = gpu.hnsw_search_knn(queries, k, ef)
        dr, lr, cr = ref.search_knn_batch(queries, k, ef, threads=2)
        assert (c == cr).all(), (k, ef, c[:5], cr[:5])
        same = sum(int((l[i, :c[i]] == lr[i, :cr[i]]).all()) for i in range(len(queries)))
        assert same >= 46, (k, ef, same)
    with pytest.raises(rx.RxGpuError):
        gpu.hnsw_search_knn(queries, 10, 5000)  # ef above the device limit
    gpu.add_point(vecs[0], int(labels[5]))  # a row was overwritten: the imported graph is stale
    with pytest.raises(rx.RxGpuError) as e:
        gpu.hnsw_search_knn(queries, 10, 64)
    assert "changed after the HNSW graph was imported" in e.value.what
    fresh = rx.GpuBruteforceSearch(metric, dim, 10)
    d, l, c = fresh.hnsw_search_knn(queries, 10, 64)  # empty index: empty result like hnswalg.h:1989-1991
    assert (c == 0).all()
    fresh.add_point(vecs[0], 7)
    with pytest.raises(rx.RxGpuError) as e:
        fresh.hnsw_search_knn(queries, 10, 64)
    assert "no HNSW graph imported" in e.value.what


def test_hnsw_768_cosine_recall(ref_tape):
    """BASELINE config 2 shape (768-dim, Cosine, M=16, efC=200, ef=128, k=10) at a size the reference builds in seconds."""
    metric, n, dim, k, ef, nq = rx.COS, 6000, 768, 10, 128, 64
    ref, gpu, vecs, labels = build(ref_tape, metric, n, dim, 950)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(951, nq, dim)])
    d, l, c = gpu.hnsw_search_knn(queries, k, ef)
    dr, lr, cr = ref.search_knn_batch(queries, k, ef, threads=4)
    same = sum(int((l[i] == lr[i]).all()) for i in range(nq))
    assert same >= nq - 2
    db, lb, _ = gpu.search_knn(queries, k)
    rec = np.mean([len(set(l[i]) & set(lb[i])) / k for i in range(nq)])
    rec_ref = np.mean([len(set(lr[i]) & set(lb[i])) / k for i in range(nq)])
    assert abs(rec - rec_ref) <= 0.01, (rec, rec_ref)


def lowrank(seed, n, dim, latent=16, noise=0.02):
    """vectors with low intrinsic dimension (what learned embeddings look like), unlike i.i.d. Gaussian noise"""
    a = np.random.default_rng(99).normal(0, 1.0, size=(latent, dim)).astype(np.float32)
    rng = np.random.default_rng(seed)
    return (rng.normal(0, 1, size=(n, latent)).astype(np.float32) @ a + rng.normal(0, noise, size=(n, dim))).astype(np.float32)


def test_hnsw_recall_on_structured_data(ref_tape):
    """data with low intrinsic dimension: recall@10 >= 0.99 at ef=128 like the north star asks, identical
    to the reference's search on the same graph"""
    metric, n, dim, k, ef, nq = rx.COS, 20000, 96, 10, 128, 128
    vecs, labels = lowrank(1, n, dim), O.row_labels(n)
    ref = ref_tape.proxy(lambda: O.RefHnsw(metric, dim, n, M=16, ef_construction=200, seed=100, multithread=False), metric, dim, n)
    ref.add_batch(labels, vecs)
    gpu = rx.GpuBruteforceSearch(metric, dim, n)
    gpu.add_points(labels, vecs)
    gpu.hnsw_import(ref.export(with_vectors=False))
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in lowrank(2, nq, dim)])
    d, l, c = gpu.hnsw_search_knn(queries, k, ef)
    dr, lr, cr = ref.search_knn_batch(queries, k, ef, threads=4)
    db, lb, _ = gpu.search_knn(queries, k)
    rec = np.mean([len(set(l[i]) & set(lb[i])) / k for i in range(nq)])
    rec_ref = np.mean([len(set(lr[i]) & set(lb[i])) / k for i in range(nq)])
    assert rec >= 0.99 and abs(rec - rec_ref) <= 0.005, (rec, rec_ref)
    assert sum(int((l[i] == lr[i]).all()) for i in range(nq)) >= 0.95 * nq


@pytest.mark.parametrize("metric,dim", [(rx.L2, 48), (rx.IP, 64), (rx.COS, 96)])
def test_hnsw_search_range_matches_reference(ref_tape, metric, dim):
    """SearchRange (hnswalg.h:2015-2070): ef-search seeds + BFS closure under the radius.  The closure does not depend on the
    traversal order, so the device's level-synchronous expansion must return the reference's set whenever the seeds agree."""
    n, ef, nq = 15000, 64, 40
    ref, gpu, vecs, labels = build(ref_tape, metric, n, dim, 1300 + metric)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(1400 + metric, nq, dim)])
    same = 0
    sizes = []
    for i in range(nq):
        db, lb, _ = gpu.search_knn(queries[i:i + 1], 201)
        j = [3, 40, 120, 200][i % 4]
        radius = float((np.float64(db[0, j - 1]) + np.float64(db[0, j])) / 2)  # halfway between two neighbours: no fp coin flips
        d, l, total = gpu.hnsw_search_range(queries[i], radius, ef)
        dr, lr, tr = ref.search_range(queries[i], radius, ef)
        assert total == len(l) and tr == len(lr)
        assert (np.diff(d) >= 0).all() and (d < radius).all()
        sizes.append(total)
        if total == tr and (l == lr).all():
            same += 1
            assert np.allclose(d, dr, rtol=RTOL, atol=ATOL)
        assert set(l) <= set(lb[0, :j]), "a result outside the exact radius ball"
    assert same >= nq - 2, (same, nq)
    assert max(sizes) >= 20, sizes  # the expansion really found neighbourhoods, not just seeds
    # max_out truncation keeps the best, out_n still reports the total
    d2, l2, t2 = gpu.hnsw_search_range(queries[1], 1e9, ef, max_out=5)
    dr2, lr2, tr2 = ref.search_range(queries[1], 1e9, ef, max_out=5)
    assert len(l2) == 5 and t2 == tr2 and t2 > n * 0.99 and (l2 == lr2).all()  # an unbounded radius floods the reachable graph
    fresh = rx.GpuBruteforceSearch(metric, dim, 10)
    assert fresh.hnsw_search_range(queries[0], 1.0, ef)[2] == 0  # empty index: empty result (:2017-2019)


def test_sharded_hnsw_two_shards_on_one_gpu(ref_tape):
    """§8e for HNSW: two independent sub-graphs (one per row range), both searched on the device, merged like brute-force shards.
    world = 1 here, so the two shards are merged through rxgpu_merge_shards directly; the NCCL exchange itself is the one the
    brute-force path uses."""
    import torch
    from reindexer_b200 import binding as B

    metric, n, dim, k, ef, nq = rx.L2, 12000, 48, 10, 96, 64
    half = n // 2
    vecs, labels = O.synth_matrix(2100, n, dim), O.row_labels(n)
    queries = O.synth_matrix(2101, nq, dim)
    shards, refs = [], []
    for s in range(2):
        ref = ref_tape.proxy(lambda s=s: O.RefHnsw(metric, dim, half, M=16, ef_construction=200, seed=100 + s, multithread=False), metric, dim,
                             half, s)
        ref.add_batch(labels[s * half:(s + 1) * half], vecs[s * half:(s + 1) * half])
        g = ref.export(with_vectors=False)
        gpu = rx.GpuBruteforceSearch(metric, dim, half)
        gpu.add_points(labels[s * half:(s + 1) * half], vecs[s * half:(s + 1) * half])
        gpu.hnsw_import(g)
        shards.append(gpu)
        refs.append(ref)
    dq = torch.from_numpy(queries).cuda()
    D = np.zeros((2, nq, k), np.float32)
    I = np.zeros((2, nq, k), np.uint32)
    L = np.zeros((2, nq, k), np.uint64)
    Cn = np.zeros((2, nq), np.uint32)
    for s, gpu in enumerate(shards):
        od = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
        oi = torch.zeros((nq, k), dtype=torch.int32, device="cuda")
        ol = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
        oc = torch.zeros((nq,), dtype=torch.int32, device="cuda")
        gpu.hnsw_search_knn_device(nq, dq.data_ptr(), k, ef, od.data_ptr(), oi.data_ptr(), oc.data_ptr())
        gpu.gather_labels_device(nq * k, oi.data_ptr(), ol.data_ptr())
        torch.cuda.synchronize()
        D[s], I[s], L[s], Cn[s] = od.cpu().numpy(), oi.cpu().numpy().view(np.uint32), ol.cpu().numpy().view(np.uint64), oc.cpu().numpy()
    rd, rg, rl, rc, _ = B.merge_shards(k, D, I, L, Cn, np.array([0, half], np.uint64))
    # the same thing with the reference's CPU searches per shard, merged by (dist, label)
    same = 0
    for i in range(nq):
        cand = []
        for s in range(2):
            dr, lr = refs[s].search_knn(queries[i], k, ef)
            cand += list(zip(dr.tolist(), lr.tolist()))
        cand.sort()
        same += int([c[1] for c in cand[:k]] == rl[i].tolist())
    assert same >= nq - 2, same
    # recall of the sharded search against exact brute force over all rows
    full = rx.GpuBruteforceSearch(metric, dim, n)
    full.add_points(labels, vecs)
    db, lb, _ = full.search_knn(queries, k)
    recall = np.mean([len(set(rl[i]) & set(lb[i])) / k for i in range(nq)])
    assert recall > 0.6, recall


@pytest.mark.parametrize("metric,frac", [(rx.L2, 0.02), (rx.COS, 0.15), (rx.IP, 0.4)])
def test_hnsw_search_with_deleted_nodes_matches_reference(ref_tape, metric, frac):
    """MarkDelete leaves tombstones in the graph: the reference switches to searchBaseLayerST<bare_bone = false> -- deleted nodes are
    traversed, never returned, and the stop rule waits for a full result list.  Same graph, same deletions, same answers."""
    n, dim, k, ef, nq = 8000, 48, 10, 64, 120
    ref, gpu, vecs, labels = build(ref_tape, metric, n, dim, 4100 + metric)
    rng = np.random.default_rng(4200 + metric)
    dead = labels[rng.choice(n, int(frac * n), replace=False)]
    for lab in dead:
        ref.mark_delete(int(lab))
        gpu.hnsw_mark_deleted(int(lab))
    assert gpu.hnsw_deleted_count() == len(dead)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(4300 + metric, nq, dim)])
    d, l, c, st = gpu.hnsw_search_knn(queries, k, ef, with_stats=True)
    dr, lr, cr = ref.search_knn_batch(queries, k, ef, threads=4)
    assert (c == cr).all()
    dead_set = set(dead.tolist())
    assert not (set(l[c[:, None] > np.arange(k)[None, :]].tolist()) & dead_set), "a deleted row was returned"
    same = sum(int((l[i, :c[i]] == lr[i, :cr[i]]).all()) for i in range(nq))
    assert same >= 0.95 * nq, f"only {same}/{nq} queries returned the reference's exact top-{k}"
    agree = 0
    for i in range(30):
        dc, hops = ref.search_metrics(queries[i], ef)
        agree += int(st[i, 0] == dc and st[i, 1] == hops)
    assert agree >= 26, agree
    # range search skips tombstones too
    db, lb, _ = gpu.search_knn(queries[:1], 60)
    radius = float((np.float64(db[0, 39]) + np.float64(db[0, 40])) / 2)
    rd, rl, total = gpu.hnsw_search_range(queries[0], radius, ef)
    fr, fl, ft = ref.search_range(queries[0], radius, ef)
    assert not (set(rl.tolist()) & dead_set) and total == ft and (rl == fl).all()
    with pytest.raises(rx.RxGpuError) as e:
        gpu.hnsw_mark_deleted(int(dead[0]))
    assert "already deleted" in e.value.what
    with pytest.raises(rx.RxGpuError):
        gpu.hnsw_mark_deleted(0xDEAD << 40)


@pytest.mark.parametrize("metric", [rx.L2, rx.COS])
def test_streaming_search_matches_reference_batches(ref_tape, metric):
    """rxgpu_hnsw_stream_* vs HierarchicalNSWImpl::Begin/ContinueStreamingSearch (hnswalg.h:1864-1975) on the same graph: the
    device keeps the session state in HBM and must hand out the same batches (labels and order; the reference's heaps break exact
    distance ties by heap mechanics, which random float data does not produce), never repeat a label, end exhausted having returned
    every reachable row, and follow tombstones like the reference (expanded, never returned)."""
    n, dim = 4000, 40
    rng = np.random.default_rng(77 + metric)
    vecs = rng.normal(0, 0.3, size=(n, dim)).astype(np.float32)
    labels = O.row_labels(n)
    ref = ref_tape.proxy(lambda: O.RefHnsw(metric, dim, n, M=16, ef_construction=100, seed=100, multithread=False), metric, dim, n)
    ref.add_batch(labels, vecs)
    g = ref.export(with_vectors=False)
    gpu = rx.GpuBruteforceSearch(metric, dim, n)
    gpu.add_points(g["labels"], vecs[(g["labels"] >> np.uint64(32)).astype(np.int64)])
    gpu.hnsw_import(g)
    queries = [prep_query(metric, q, use_ref=False) for q in rng.normal(0, 0.3, size=(12, dim)).astype(np.float32)]

    def compare(batch, ef, max_batches, qs):
        same = total = 0
        for q in qs:
            it_ref = ref.stream(q, batch, ef=ef, max_batches=max_batches)
            it_gpu = gpu.hnsw_stream(q, batch, ef=ef, max_batches=max_batches)
            seen = set()
            for (dr, lr), (dg, lg) in zip(it_ref, it_gpu):
                total += 1
                assert (np.diff(dg) >= 0).all() and not (set(lg.tolist()) & seen)
                seen |= set(lg.tolist())
                if len(lr) == len(lg) and (lr == lg).all():
                    same += 1
                    assert np.allclose(dg, dr, rtol=RTOL, atol=ATOL)
        return same, total

    same, total = compare(20, 64, 8, queries)
    assert total == 8 * len(queries) and same >= 0.95 * total, (same, total)
    same, total = compare(150, 32, 4, queries[:4])  # batch larger than ef: ContinueStreamingSearch widens ef for the call
    assert same >= 0.9 * total, (same, total)
    # a whole stream: exhausted exactly when every row was returned once
    got = []
    nb = 0
    for d, l in gpu.hnsw_stream(queries[0], 256, ef=100):
        got += l.tolist()
        nb += 1
    assert len(got) == len(set(got)) and len(got) >= 0.99 * n and nb >= n // 256
    ref_all = []
    for d, l in ref.stream(queries[0], 256, ef=100):
        ref_all += l.tolist()
    assert set(got) == set(ref_all)
    # tombstones
    for lab in g["labels"][::7]:
        ref.mark_delete(int(lab))
        gpu.hnsw_mark_deleted(int(lab))
    dead = set(int(x) for x in g["labels"][::7])
    same, total = compare(25, 64, 6, queries[:6])
    assert same >= 0.9 * total, (same, total)
    for d, l in gpu.hnsw_stream(queries[1], 100, ef=64, max_batches=10):
        assert not (set(l.tolist()) & dead)


@pytest.mark.parametrize("metric", [O.L2, O.COS])
def test_incremental_update_equals_fresh_import(ref_tape, metric):
    """rxgpu_hnsw_update: after the reference's inserter added rows, patching the nodes whose lists differ between two exports gives
    the same device graph -- identical answers -- as importing the new graph from scratch (hnswalg.h:1695-1852, :1070-1180)."""
    n0, extra, dim, k, ef = 3000, 400, 24, 10, 48
    rng = np.random.default_rng(11)
    vecs = rng.normal(size=(n0 + extra, dim)).astype(np.float32)
    labels = O.row_labels(n0 + extra)
    ref = ref_tape.proxy(lambda: O.RefHnsw(metric, dim, n0 + extra, M=8, ef_construction=60, seed=100), metric, dim, n0 + extra)
    ref.add_batch(labels[:n0], vecs[:n0])
    g0 = ref.export(with_vectors=False)
    patched = rx.GpuBruteforceSearch(metric, dim, n0 + extra)
    patched.add_points(labels[:n0], vecs[:n0])
    patched.hnsw_import(g0)
    queries = rng.normal(size=(64, dim)).astype(np.float32)
    done = n0
    for step in (1, 7, 92, 300):  # single upserts and small bursts
        ref.add_batch(labels[done:done + step], vecs[done:done + step])
        g1 = ref.export(with_vectors=False)
        old_n = done
        done += step
        changed = [v for v in range(old_n) if g1["levels"][v] != g0["levels"][v] or (g1["level0"][v] != g0["level0"][v]).any()
                   or (g1["levels"][v] > 0 and (g1["upper"][g1["upper_offsets"][v]:g1["upper_offsets"][v] + g1["levels"][v]]
                                                != g0["upper"][g0["upper_offsets"][v]:g0["upper_offsets"][v] + g0["levels"][v]]).any())]
        # the reference's export packs upper lists densely by node id; the device keeps appended nodes at the end of its slab --
        # both are addressed through per-node offsets, so only the lists themselves travel
        patched.hnsw_update(g1, changed, new_rows={v: (int(labels[v]), vecs[v]) for v in range(old_n, done)})
        fresh = rx.GpuBruteforceSearch(metric, dim, done)
        fresh.add_points(labels[:done], vecs[:done])
        fresh.hnsw_import(g1)
        dp, lp, cp = patched.hnsw_search_knn(queries, k, ef)
        df, lf, cf = fresh.hnsw_search_knn(queries, k, ef)
        assert (cp == cf).all() and (lp == lf).all() and (dp == df).all(), f"after {done - n0} upserts"
        if metric == O.L2:
            dr, lr, cr = ref.search_knn_batch(queries, k, ef)
            assert np.mean([(lp[i] == lr[i]).all() for i in range(64)]) >= 0.97
        g0 = g1
    assert patched.hnsw_update_count() > 400
    with pytest.raises(rx.RxGpuError):  # malformed patch: nothing applied
        bad = dict(g0)
        bad["level0"] = g0["level0"].copy()
        bad["level0"][5, 1] = 10_000_000
        patched.hnsw_update(bad, [5])
    dp2, lp2, _ = patched.hnsw_search_knn(queries, k, ef)
    assert (lp2 == lp).all()
