"""GPU tests of the multi-GPU path behind the C ABI (reindexer_b200/csrc/shard.cu): rxgpu_sharded_search_knn = local scan + one
ncclAllGather + device merge + the reference's tie rule replayed from the filter's candidate lists.  On one GPU the communicator has a
single rank (no NCCL involved) and the answer must equal rxgpu_search_knn's and the oracle's; the device merge kernel is checked
against the host merge (rxgpu_merge_shards, itself pinned to the sequential reference algorithm by tests/test_host_logic.py); the
world-2 NCCL run is tests/mp_sharded_nccl.py, launched by test_two_ranks_nccl when the box has two GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import reindexer_b200 as rx
from reindexer_b200 import binding as B
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def tie_heavy(n, dim, seed):
    """integer-valued rows: every summation order gives the same fp32 sums, so bit-equal distances abound"""
    rng = np.random.default_rng(seed)
    return rng.integers(-2, 3, size=(n, dim)).astype(np.float32)


@pytest.mark.parametrize("metric", [rx.L2, rx.IP])
@pytest.mark.parametrize("nq,tc", [(3, 0), (96, 1)])
def test_single_rank_equals_search_knn_and_oracle(metric, nq, tc):
    n, dim, k = 20000, 32, 10
    vecs, labels = tie_heavy(n, dim, 7), O.row_labels(n)
    gpu = rx.GpuBruteforceSearch(metric, dim, n)
    gpu.add_points(labels, vecs)
    gpu.set_tensor_core_filter(tc)
    queries = tie_heavy(nq, dim, 8)
    comm = B.ShardComm(1, 0, None, 0)
    d1, l1, c1 = comm.search_knn(gpu, queries, k)
    st = rx.last_search_stats()
    d0, l0, c0 = gpu.search_knn(queries, k)
    assert (c0 == c1).all() and (l0 == l1).all() and (d0.view(np.uint32) == d1.view(np.uint32)).all()
    assert st["tie_replays"] > 0  # this data ties at the k-th place
    if tc:
        assert st["tc_used"] == 1 and st["tie_from_lists"] == st["tie_replays"]  # no second pass over the rows
    cpu = O.best_bf(metric, dim, n)
    cpu.add_batch(labels, vecs)
    for i in range(0, nq, max(1, nq // 5)):
        dr, lr = cpu.search_knn(queries[i], k)
        assert (l1[i] == lr).all() and (d1[i].view(np.uint32) == np.asarray(dr, np.float32).view(np.uint32)).all(), i
    comm.close()


def test_device_queries_and_random_data():
    import torch

    n, dim, k, nq = 50000, 96, 10, 256
    gpu = rx.GpuBruteforceSearch(rx.IP, dim, n)
    gpu.append_synth(0x51, 0, n)
    queries = O.synth_matrix(0x52, nq, dim)
    comm = B.ShardComm(1, 0, None, 0)
    dq = torch.from_numpy(queries).cuda()
    torch.cuda.synchronize()
    d1, l1, c1 = comm.search_knn(gpu, dq.data_ptr(), k, nq=nq)
    d0, l0, c0 = gpu.search_knn(queries, k)
    assert (l0 == l1).all() and (d0.view(np.uint32) == d1.view(np.uint32)).all() and (c1 == k).all()


def test_merge_kernel_equals_host_merge():
    import torch

    rng = np.random.default_rng(3)
    for shards, nq, k in ((2, 40, 10), (8, 300, 10), (5, 17, 1), (3, 9, 33)):
        k1 = k + 1
        sizes = rng.integers(k1 + 5, 5000, size=shards).astype(np.uint64)
        base = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64)
        D = np.zeros((shards, nq, k1), np.float32)
        I = np.zeros((shards, nq, k1), np.uint32)
        L = np.zeros((shards, nq, k1), np.uint64)
        Cn = np.zeros((shards, nq), np.uint32)
        for s in range(shards):
            for q in range(nq):
                c = int(rng.integers(0, k1 + 1)) if rng.random() < 0.2 else k1
                dist = np.sort(rng.integers(0, 6, size=c).astype(np.float32))  # few distinct values: ties within and across shards
                idx = np.zeros(c, np.uint32)
                for v in np.unique(dist):  # ascending internal index inside runs of equal distance, like the scan's total order
                    m = dist == v
                    idx[m] = np.sort(rng.choice(int(sizes[s]), size=int(m.sum()), replace=False)).astype(np.uint32)
                D[s, q, :c], I[s, q, :c], Cn[s, q] = dist, idx, c
                L[s, q, :c] = rng.integers(0, 1 << 40, size=c).astype(np.uint64)
        rd, rg, rl, rc, nt = B.merge_shards(k, D, I, L, Cn, base)
        nbytes = int(B.lib().rxgpu_shard_payload_bytes(nq, k1))
        up = lambda x: (x + 15) & ~15
        n = nq * k1
        off_idx = up(n * 4)
        off_label = up(off_idx + n * 4)
        off_count = up(off_label + n * 8)
        off_size = up(off_count + nq * 4)
        assert up(off_size + 16) == nbytes
        buf = np.zeros((shards, nbytes), np.uint8)
        for s in range(shards):
            buf[s, 0:n * 4] = D[s].reshape(-1).view(np.uint8)
            buf[s, off_idx:off_idx + n * 4] = I[s].reshape(-1).view(np.uint8)
            buf[s, off_label:off_label + n * 8] = L[s].reshape(-1).view(np.uint8)
            buf[s, off_count:off_count + nq * 4] = Cn[s].view(np.uint8)
            buf[s, off_size:off_size + 8] = np.array([sizes[s]], np.uint64).view(np.uint8)
        dbuf = torch.from_numpy(buf).cuda()
        od = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
        og = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
        ol = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
        oc = torch.zeros((nq,), dtype=torch.int32, device="cuda")
        ot = torch.zeros((nq,), dtype=torch.uint8, device="cuda")
        B._check(B.lib().rxgpu_merge_shards_device(shards, nq, k, k1, dbuf.data_ptr(), od.data_ptr(), og.data_ptr(), ol.data_ptr(),
                                                   oc.data_ptr(), ot.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert (oc.cpu().numpy().astype(np.uint32) == rc).all()
        assert (ot.cpu().numpy() == nt).all()
        gd, gg = od.cpu().numpy(), og.cpu().numpy().view(np.uint64)
        for q in range(nq):
            c = int(rc[q])
            # the kernel leaves runs of equal distance in (global row) order; the host merge orders them by label afterwards
            assert (gd[q, :c] == rd[q, :c]).all()
            assert sorted(gg[q, :c].tolist()) == sorted(rg[q, :c].tolist())


def test_two_ranks_nccl():
    if rx.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", os.path.join(ROOT, "tests", "mp_sharded_nccl.py")], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "mp_sharded_nccl ok" in r.stdout
