"""GPU parity tests of the IVF search (SURVEY.md §8 a11 / f1): the index is trained and filled by the REFERENCE's own FAISS
(oracle/_ref/liboracle_ref_ivf.so: vendor_subdirs/faiss compiled in place, driven like reindexer::IvfIndex), its centroids and
inverted lists are imported into the device index, and every search is compared with faiss::IndexIVFFlat::search on the same state.
The reference's state and answers for the smaller index shapes are stored in tests/golden/ref_tapes/."""
import numpy as np
import pytest
from helpers import ATOL, RTOL, prep_query

import reindexer_b200 as rx
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def export(ref_tape, ref, vecs):
    """the reference's centroids and lists.  FAISS appends the rows of a fresh index to their lists in order (checked when recorded),
    and the rows are the inputs', so the list of every row is all there is to store."""
    def run():
        st = ref.real().export()
        rows = (st["labels"] >> np.uint64(32)).astype(np.int64)
        row_list = np.repeat(np.arange(len(st["list_sizes"]), dtype=np.uint32), st["list_sizes"].astype(np.int64))
        assert (np.argsort(row_list[np.argsort(rows)], kind="stable") == rows).all() and (st["vecs"] == vecs[rows]).all()
        out = np.zeros(len(rows), np.uint32)
        out[rows] = row_list
        return dict(centroids=st["centroids"], row_list=out)

    st = ref_tape(run, "export")
    rows = np.argsort(st["row_list"], kind="stable")
    return dict(centroids=st["centroids"], list_sizes=np.bincount(st["row_list"], minlength=len(st["centroids"])).astype(np.uint64),
                labels=O.row_labels(len(rows))[rows], vecs=vecs[rows])


def build(ref_tape, metric, n, dim, nlist, seed):
    vecs, labels = O.synth_matrix(seed, n, dim), O.row_labels(n)
    ref = ref_tape.proxy(lambda: O.RefIvf(metric, dim, nlist), metric, dim, nlist)
    ref.train_add(labels, vecs)
    st = export(ref_tape, ref, vecs)
    assert int(st["list_sizes"].sum()) == n and sorted(st["labels"].tolist()) == sorted(labels.tolist())
    gpu = rx.GpuBruteforceSearch(metric, dim, n)
    gpu.add_points(st["labels"], st["vecs"])  # rows grouped by list, label = FAISS id
    gpu.ivf_import(st["centroids"], st["list_sizes"])
    return ref, gpu, st


@pytest.mark.parametrize("metric,dim,nlist", [(rx.L2, 32, 16), (rx.L2, 96, 64), (rx.IP, 64, 32), (rx.L2, 768, 24), (rx.IP, 200, 50),
                                              (rx.COS, 48, 20), (rx.COS, 384, 32)])
def test_ivf_search_matches_reference_faiss(ref_tape, metric, dim, nlist):
    n = 12000 if dim < 500 else 4000
    ref, gpu, st = build(ref_tape, metric, n, dim, nlist, 3100 + dim)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(3200 + dim, 40, dim)])
    for k, nprobe in [(10, 1), (10, 4), (1, 8), (50, nlist // 2), (10, nlist), (10, nlist + 7)]:
        d, l, c = gpu.ivf_search_knn(queries, k, nprobe)
        for i in range(len(queries)):
            dr, lr = ref.search(queries[i], k, nprobe)
            assert c[i] == len(lr), (k, nprobe, i, c[i], len(lr))
            dr_map = dr if metric == rx.L2 else -dr  # FAISS reports +IP / +cos (descending); the map space is the negation (ascending)
            assert np.allclose(d[i, :c[i]], dr_map, rtol=RTOL, atol=ATOL), (k, nprobe, i)
            if not (l[i, :c[i]] == lr).all():  # ids may differ only where neighbouring distances are within fp noise
                bad = np.nonzero(l[i, :c[i]] != lr)[0]
                assert set(l[i, :c[i]]) == set(lr) or np.allclose(d[i, bad], dr_map[bad], rtol=1e-5), (k, nprobe, i, l[i, :c[i]], lr)
    # nprobe = nlist scans every list: the result is the exact brute-force answer
    d, l, c = gpu.ivf_search_knn(queries[:8], 10, nlist)
    db, lb, _ = gpu.search_knn(queries[:8], 10)
    assert (l == lb).all() and (d.view(np.uint32) == db.view(np.uint32)).all()  # same per-row arithmetic => same bits


def test_ivf_errors_and_staleness():
    # any valid partition does here: 8 rows as centroids, every row in the list of its nearest one
    vecs = O.synth_matrix(77, 3000, 16)
    centroids = vecs[::375].copy()
    nearest = ((vecs[:, None, :] - centroids[None]) ** 2).sum(-1).argmin(1)
    rows = np.argsort(nearest, kind="stable")
    st = dict(centroids=centroids, list_sizes=np.bincount(nearest, minlength=8).astype(np.uint64), labels=O.row_labels(3000)[rows],
              vecs=vecs[rows])
    gpu = rx.GpuBruteforceSearch(rx.L2, 16, 3000)
    gpu.add_points(st["labels"], st["vecs"])
    gpu.ivf_import(st["centroids"], st["list_sizes"])
    q = O.synth_matrix(78, 2, 16)
    with pytest.raises(rx.RxGpuError):
        gpu.ivf_search_knn(q, 0, 4)
    with pytest.raises(rx.RxGpuError):
        gpu.ivf_search_knn(q, 300, 4)
    gpu.add_point(st["vecs"][0], int(st["labels"][5]))  # a row was overwritten: the imported lists are stale
    with pytest.raises(rx.RxGpuError) as e:
        gpu.ivf_search_knn(q, 5, 4)
    assert "changed after the IVF lists were imported" in e.value.what
    fresh = rx.GpuBruteforceSearch(rx.L2, 16, 10)
    fresh.add_point(st["vecs"][0], 1)
    with pytest.raises(rx.RxGpuError) as e:
        fresh.ivf_search_knn(q, 5, 4)
    assert "no IVF lists imported" in e.value.what
    with pytest.raises(rx.RxGpuError):
        fresh.ivf_import(st["centroids"], st["list_sizes"])  # sizes do not add up to the rows of this index


@pytest.mark.parametrize("metric", [rx.L2, rx.IP, rx.COS])
def test_ivf_range_search_matches_reference_faiss(ref_tape, metric):
    n, dim, nlist, nprobe = 8000, 40, 16, 5
    ref, gpu, st = build(ref_tape, metric, n, dim, nlist, 3500 + metric)
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(3600 + metric, 12, dim)])
    for i, q in enumerate(queries):
        d, l, c = gpu.ivf_search_knn(q, 60, nprobe)
        j = [5, 20, 59][i % 3]
        radius = float((np.float64(d[0, j - 1]) + np.float64(d[0, j])) / 2)  # map space, halfway between two neighbours
        rd, rl, total = gpu.ivf_search_range(q, radius, nprobe)
        fd, fl = ref.range_search(q, radius if metric == rx.L2 else -radius, nprobe)
        assert total == len(rl) == len(fl) == j
        assert sorted(rl.tolist()) == sorted(fl.tolist())
        assert (np.diff(rd) >= 0).all() and (rl == l[0, :j]).all()
    rd, rl, total = gpu.ivf_search_range(queries[0], 1e30, nlist, max_out=7)  # everything, truncated output
    assert total == n and len(rl) == 7


@pytest.mark.parametrize("metric,dim,nlist", [(rx.L2, 40, 24), (rx.IP, 64, 16), (rx.COS, 96, 12)])
def test_mutable_lists_follow_reference_upserts_and_deletes(ref_tape, metric, dim, nlist):
    """rxgpu_ivf_create / _add / _remove against faiss::IndexIVFFlat driven like IvfIndex::upsert / del (ivf_index.cc:87-132): the device
    lists are never re-imported; after every burst of upserts and deletes the searches agree with the reference on the same state."""
    n0, seed = 6000, 4400 + dim
    vecs, labels = O.synth_matrix(seed, n0 + 3000, dim), O.row_labels(n0 + 3000)
    ref = ref_tape.proxy(lambda: O.RefIvf(metric, dim, nlist), metric, dim, nlist)
    ref.train_add(labels[:n0], vecs[:n0])
    st = export(ref_tape, ref, vecs[:n0])
    gpu = rx.GpuBruteforceSearch(metric, dim, 16)  # rows live in the lists, not in the flat index
    gpu.ivf_create(st["centroids"])
    gpu.ivf_add(ref.list_of(labels[:n0]), labels[:n0], vecs[:n0])
    queries = np.stack([prep_query(metric, q, use_ref=False) for q in O.synth_matrix(seed + 1, 24, dim)])
    rng = np.random.default_rng(seed)
    alive = set(labels[:n0].tolist())

    def check(ctx):
        assert gpu.ivf_size() == len(alive)
        for k, nprobe in [(10, 3), (20, nlist)]:
            d, l, c = gpu.ivf_search_knn(queries, k, nprobe)
            for i in range(len(queries)):
                dr, lr = ref.search(queries[i], k, nprobe)
                dr_map = dr if metric == rx.L2 else -dr
                assert c[i] == len(lr) and np.allclose(d[i, :c[i]], dr_map, rtol=RTOL, atol=ATOL), (ctx, k, nprobe, i)
                if not (l[i, :c[i]] == lr).all():
                    bad = np.nonzero(l[i, :c[i]] != lr)[0]
                    assert set(l[i, :c[i]]) == set(lr) or np.allclose(d[i, bad], dr_map[bad], rtol=1e-5), (ctx, k, nprobe, i)
        d31 = ref.search(queries[0], 31, nlist)[0]  # best first in FAISS' convention
        radius = float((d31[29] + d31[30]) / 2)  # between two neighbours: no boundary ambiguity
        dg, lg, _ = gpu.ivf_search_range(queries[0], radius if metric == rx.L2 else -radius, nlist)
        drr, lrr = ref.range_search(queries[0], radius, nlist)
        assert set(lg.tolist()) == set(lrr.tolist()), ctx

    check("initial fill")
    done = n0
    for burst in (1, 40, 900, 2059):
        new = slice(done, done + burst)
        ref.add(labels[new], vecs[new])
        gpu.ivf_add(ref.list_of(labels[new]), labels[new], vecs[new])
        alive |= set(labels[new].tolist())
        done += burst
        victims = rng.choice(sorted(alive), size=min(len(alive) // 10, 300), replace=False)
        for v in victims:
            ref.remove(int(v))
            gpu.ivf_remove(int(v))
            alive.discard(int(v))
        check(f"after {done - n0} upserts")
    stats = gpu.ivf_list_stats()
    assert stats["relocations"] > 0
    with pytest.raises(rx.RxGpuError):
        gpu.ivf_remove(int(victims[0]))  # already gone
    with pytest.raises(rx.RxGpuError):
        gpu.ivf_add([0], [int(next(iter(alive)))], vecs[:1])  # duplicate id
    # delete most rows, then keep inserting: dead space is compacted instead of growing the slab forever
    for v in sorted(alive)[: len(alive) * 3 // 4]:
        ref.remove(int(v))
        gpu.ivf_remove(int(v))
        alive.discard(int(v))
    check("after mass delete")
