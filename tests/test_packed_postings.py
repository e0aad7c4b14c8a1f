"""CPU tests of the packed posting-list decoder (reindexer_b200/host/packed_postings.h through the C ABI, no device involved):
the byte streams come from the REFERENCE's own encoder (tests/golden/packed_golden.npz, tests/golden/ref_tapes/)."""
import os

import numpy as np
import pytest

import reindexer_b200 as rx
from reindexer_b200 import binding as B
from oracle import ft_oracle as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def packed_golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "packed_golden.npz"))


def test_decoder_inverts_the_reference_encoder_on_golden_streams(packed_golden):
    for name in packed_golden["names"]:
        d, b, p = (packed_golden[f"{name}/{k}"] for k in ("doc_ids", "pos_begin", "positions"))
        dd, bb, pp = B.ft_decode_packed(packed_golden[f"{name}/packed"], len(d))
        assert (dd == d).all() and (bb == b).all() and (pp == p).all(), name


def test_decoder_inverts_the_reference_encoder_live(ref_tape):
    rng = np.random.default_rng(5)
    for trial in range(30):
        ndocs = int(rng.integers(1, 400))
        docs = np.sort(rng.choice(np.arange(1, 100000), size=ndocs, replace=False)).astype(np.uint32)
        npos = rng.integers(1, 6, size=ndocs)
        begin = np.concatenate([[0], np.cumsum(npos)]).astype(np.uint32)
        nf = int(rng.integers(1, 9))
        f = rng.integers(0, nf, size=begin[-1])
        w = rng.integers(0, 1 << int(rng.integers(4, 24)), size=begin[-1])
        positions = np.zeros(begin[-1], np.uint32)
        for i in range(ndocs):
            s = slice(begin[i], begin[i + 1])
            order = np.lexsort((w[s], f[s]))
            positions[s] = (w[s][order] | (f[s][order] << 24)).astype(np.uint32)
        packed = ref_tape(lambda: F.ref_pack_list(docs, begin, positions), docs, begin, positions)
        dd, bb, pp = B.ft_decode_packed(packed, ndocs)
        assert (dd == docs).all() and (bb == begin).all() and (pp == positions).all(), trial


def test_decoder_rejects_malformed_streams(packed_golden):
    packed = packed_golden["multi_field/packed"]
    n = len(packed_golden["multi_field/doc_ids"])
    with pytest.raises(rx.RxGpuError):
        B.ft_decode_packed(packed[:-1], n)          # truncated inside the last record
    with pytest.raises(rx.RxGpuError):
        B.ft_decode_packed(packed, n + 1)           # record count mismatch
    with pytest.raises(rx.RxGpuError):
        B.ft_decode_packed(np.full(8, 0xFF, np.uint8), 1)  # varint longer than 5 bytes
    d, b, p = B.ft_decode_packed(np.zeros(0, np.uint8), 0)  # the empty list
    assert len(d) == 0 and b.tolist() == [0] and len(p) == 0
