"""BFMatcher(NORM_L2, crossCheck=True).match is the mutual-nearest rule over knnMatch in both directions: the CPU oracle's
cvo_knn2 (query -> train and train -> query, first neighbours) reproduces every cv2 golden of golden_crosscheck.npz bit for
bit.  The GPU tests (test_gpu_cross_check.py) use the same goldens."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import crosscheck_cases  # noqa: E402


@pytest.fixture(scope="module")
def golden():
    return crosscheck_cases.load_golden()


@pytest.mark.parametrize("tag", ["real", "sat", "tie", "float", "small", "big"])
def test_mutual_rule_reproduces_cv2(oracle, golden, tag):
    sets, gi, gd, off = golden[tag]
    for k, (q, t) in enumerate(sets):
        idx, dist = crosscheck_cases.mutual(oracle, q, t)
        assert np.array_equal(idx, gi[off[k]:off[k + 1]]), (tag, k)
        assert np.array_equal(dist.view(np.uint32), gd[off[k]:off[k + 1]].view(np.uint32)), (tag, k)


def test_real_pairs_keep_more_than_the_ratio_test(golden):
    sets, gi, _, off = golden["real"]
    assert len(sets) == 890
    kept = np.array([(gi[off[k]:off[k + 1]] >= 0).sum() for k in range(len(sets))])
    assert kept.min() >= 4 and np.median(kept) == 82 and kept.max() == 183


def test_no_second_choice(golden):
    _, gi, _, off = golden["small"]
    assert list(gi[off[2]:off[3]]) == [-1, 0]          # query 0's nearest train row prefers query 1: no fallback
    assert list(gi[off[0]:off[1]]).count(0) == 1 and gi[off[0] + 6] == 0   # n_train = 1: lowest of the tied rows
