"""CPU tests: the full-text oracle restatement (oracle/ft_port.c) pinned against
 (a) tests/golden/ft_golden.npz -- outputs of the reference's own ft::Merger::Merge (tests/golden/make_ft_golden.py), including the
     term-rank values the reference's own test FTGenericApi.DebugInfo pins, and
 (b) the reference's own merger (oracle/_ref/liboracle_ref_ft.so) on random problems, through its answers stored in
     tests/golden/ref_tapes/."""
import os

import numpy as np
import pytest
from ft_helpers import assert_same_merge, assert_same_merge_as_digest, load_golden_problem, merge_digest, random_problem

from oracle import ft_oracle as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ft_golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "ft_golden.npz"))


def test_known_answer_values_of_the_reference_test(ft_golden):
    # FTGenericApi.DebugInfo (cpp_src/gtests/tests/unit/ft/ft_generic.cc:326-327): term_rank 97.9844 and 77.91719
    assert f"{ft_golden['kat/term_rank'][0]:.4f}" == "97.9844" and f"{ft_golden['kat/term_rank'][1]:.5f}" == "77.91719"
    # the port reproduces them through a whole merge: one doc, rank = uint8(max(97.98.., 77.9..)) = 97 (mergeSimple keeps the max)
    p = F.FtProblem(6, np.array([0, 8, 3, 6, 12, 3], np.uint32))
    l0, l1 = p.add_list([1], [[(0, 0)]]), p.add_list([1], [[(6, 0)]])
    p.add_term([(l0, 100.0), (l1, 80.0)])
    res, _ = F.port_merge(p)
    assert res.tolist() == [(1, 97.0, 0, 97)]
    p2 = F.FtProblem(6, np.array([0, 8, 3, 6, 12, 3], np.uint32))
    p2.add_term([(p2.add_list([1], [[(6, 0)]]), 80.0)])
    assert F.port_merge(p2)[0].tolist() == [(1, 77.0, 0, 77)]


def test_port_matches_golden(ft_golden):
    for name in ft_golden["names"]:
        p = load_golden_problem(ft_golden, str(name))
        for rst in (F.RANK_AND_ID, F.RANK_ONLY):
            res, _ = F.port_merge(p, rst)
            assert_same_merge(ft_golden[f"{name}/result{rst}"], res, rst, ctx=f"{name} rst={rst}")


def test_port_matches_reference_merger_on_random_problems(ref_tape):
    preselected = 0
    for seed in range(160):
        rng = np.random.default_rng(seed)
        kw = dict(total_docs=int(rng.integers(30, 600)), nfields=1 + seed % 3, nterms=1 + seed % 4, removed_frac=0.05 * (seed % 2),
                  excluded_frac=0.05 * (seed % 3 == 0), field_boost_zero=(seed % 5 == 0))
        if seed % 4 == 1:
            kw["merge_limit"] = int(rng.integers(5, 60))
            preselected += 1
        p = random_problem(seed, **kw)
        for rst in (F.RANK_AND_ID, F.RANK_ONLY, F.ID_ONLY):
            a = ref_tape(lambda: merge_digest(F.ref_merge(p, rst)[0], rst), p, rst)
            b, _ = F.port_merge(p, rst)
            assert_same_merge_as_digest(a, b, rst, ctx=f"seed {seed} rst {rst}")
        # the default container (PackedIdRelVec, Optimization::Memory) gives the same merge as IdRelVec
        packed = ref_tape(lambda: merge_digest(F.ref_merge(p, F.RANK_AND_ID, packed=True)[0], F.RANK_AND_ID), p, "packed")
        assert_same_merge_as_digest(packed, F.port_merge(p, F.RANK_AND_ID)[0], F.RANK_AND_ID, ctx=f"seed {seed} packed")
    assert preselected > 20


def test_bm25_variants_and_config_knobs(ref_tape):
    for seed in range(30):
        p = random_problem(1000 + seed, total_docs=200, nfields=2, nterms=2)
        p.cfg.update(bm25_type=seed % 3, bm25_k1=1.2 + 0.1 * (seed % 5), bm25_b=0.5 + 0.05 * (seed % 4), min_rank=seed % 40,
                     distance_weight=0.3, distance_boost=1.5, full_match_boost=1.3)
        p.field_cfg[0].update(bm25_weight=0.4, position_weight=0.3, term_len_weight=0.2, bm25_boost=1.2)
        a = ref_tape(lambda: merge_digest(F.ref_merge(p)[0], F.RANK_AND_ID), p)
        b, _ = F.port_merge(p)
        assert_same_merge_as_digest(a, b, F.RANK_AND_ID, ctx=f"seed {seed}")


def test_port_summation_of_ranks_by_fields_matches_reference(ref_tape):
    for seed in range(40):
        rng = np.random.default_rng(5000 + seed)
        nfields = 2 + seed % 4
        p = random_problem(5000 + seed, total_docs=300, nfields=nfields, nterms=1 + seed % 3, max_pos=6)
        p.cfg["summation_ranks_by_fields_ratio"] = float(rng.choice([0.3, 0.5, 0.9, 1.0]))
        for t in p.terms:
            t["need_sum_rank"] = (rng.random(nfields) < 0.7).astype(np.uint8)
        want = ref_tape(lambda: merge_digest(F.ref_merge(p)[0], F.RANK_AND_ID), p)
        assert_same_merge_as_digest(want, F.port_merge(p)[0], F.RANK_AND_ID, ctx=f"seed {seed}")
