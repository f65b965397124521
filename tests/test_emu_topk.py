"""The device selection of a query's best subjects (csrc/kern_topk.cuh), stepped in CPU emulation: the kk rows it
writes are those of np.lexsort((ids, -score))[:kk], the rule of psb_batch_topk (score descending, then smaller id)."""
import numpy as np
import pytest

import emu_topk as emu


def expected(score, kk):
    return np.lexsort((np.arange(len(score)), -np.asarray(score, dtype=np.int64)))[:kk]


def check(score, k, nblocks=1, nwarps=1):
    score = np.asarray(score, dtype=np.int32)
    kk = min(k, len(score))
    ids, sc = emu.topk(score, kk, nblocks, nwarps)
    order = np.lexsort((ids, -sc.astype(np.int64)))
    assert np.array_equal(ids[order], expected(score, kk))
    assert np.array_equal(sc, score[ids])


@pytest.mark.parametrize("nblocks,nwarps", [(1, 1), (3, 4), (7, 9)])
def test_random_scores(nblocks, nwarps):
    rng = np.random.default_rng(11 + nwarps)
    score = rng.integers(-50, 400, 3000)
    for k in (1, 7, 100, 2999):
        check(score, k, nblocks, nwarps)


def test_full_int_range_and_negative_scores():
    rng = np.random.default_rng(3)
    check(rng.integers(-2**31, 2**31 - 1, 1500, dtype=np.int64), 40, 2, 5)
    check(rng.integers(-5000, -10, 1500), 60, 2, 5)   # all negative: global / semi-global scans
    check(np.array([-2**31, 2**31 - 1, 0, -1, 1] * 20), 33, 1, 3)


def test_all_equal():
    for k in (1, 64, 999, 1000, 5000):
        check(np.full(1000, 17), k, 2, 6)
    check(np.full(700, -3), 100, 3, 4)


def test_tie_group_at_threshold_spans_blocks():
    # 40 subjects above, then a group of 900 ties spread over every warp's chunk and cut in the middle by k
    rng = np.random.default_rng(5)
    score = rng.integers(0, 50, 2500)
    tie = rng.choice(2500, 900, replace=False)
    score[tie] = 60
    score[rng.choice(np.setdiff1d(np.arange(2500), tie), 40, replace=False)] = 80 + rng.integers(0, 5, 40)
    for k in (41, 500, 939, 940, 941):
        check(score, k, 4, 8)


def test_tiny():
    check([5], 1)
    check([5], 3)
    check([-5], 1, 2, 2)
    check([1, 1], 1)
    check([3, 9, 9, 1], 4, 1, 2)
    check([3, 9, 9, 1], 10, 1, 2)


def test_empty_warps():
    # more compaction warps than 32-id chunks: the last warps own no ids
    check(np.arange(70) % 7, 9, 2, 8)
