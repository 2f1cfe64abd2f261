"""Exact search and sequence evaluation: the oracle's rules on hand-built cases, test-id resolution and the C ABI's
workspace sizes (no GPU needed)."""
import numpy as np
import pytest

from grafp_b200 import _native, build
from grafp_b200.search import resolve_test_ids
from oracle import search_oracle as SO


def _unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def test_flat_search_orders_by_distance_then_lower_id():
    R = _unit([[1, 0, 0], [0, 1, 0], [1, 0, 0], [0, 0, 1]])
    D, I = SO.flat_search(R, _unit([[1, 0, 0], [0, 1, 1]]), 3)
    assert I[0].tolist() == [0, 2, 1]          # the duplicate rows 0 and 2 tie: lower id first
    assert I[1].tolist() == [1, 3, 0]
    assert float(D[0, 0]) == pytest.approx(0.0, abs=1e-12)


def _hand_index():
    # 6 database rows on a circle; query rows sit on rows 2, 3, 4 of it
    ang = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 2.5])
    R = np.stack([np.cos(ang), np.sin(ang), np.zeros(6)], 1)
    return R


def test_oracle_drops_negative_candidates_and_truncates_at_the_end():
    R = _hand_index()
    query = R[[2, 3, 4]]
    probe = np.array([[2, 1], [3, 2], [4, 5]])      # exact top-2 of each query row, fixed by hand
    out = SO.sequence_hit_rates(R, query, [0], [3], k_probe=2, gt_offset=2, probe_ids=probe)
    # candidates: {2, 1} u {2, 1} u {2, 3} = {1, 2, 3}; row 2 scores all three rows 1.0
    assert out["hits"]["top1_exact"][0, 0] and out["top1_exact"][0] == 100.0
    # a candidate near the end of the index averages over the rows that exist (numpy slice semantics)
    probe_end = np.array([[5, 4], [5, 4], [5, 4]])
    out = SO.sequence_hit_rates(R, query, [0], [3], k_probe=2, gt_offset=2, probe_ids=probe_end)
    # candidates 5, 4 (row 0), 4, 3 (row 1 minus 1), 3, 2 (row 2 minus 2): {2, 3, 4, 5}; 2 is exact, 5 scores one row
    assert out["hits"]["top1_exact"][0, 0]
    neg = np.array([[0, 1], [0, 1], [0, 1]])         # row 1 minus 1 -> -1, 0; row 2 minus 2 -> -2, -1: dropped
    out = SO.sequence_hit_rates(R, query, [0], [3], k_probe=2, gt_offset=2, probe_ids=neg)
    assert not out["hits"]["top1_exact"][0, 0] and not out["hits"]["top10_exact"][0, 0]


def test_oracle_near_hits_and_tie_rule():
    R = _hand_index()
    query = R[[3]]
    # gt = 2 (offset -1): the prediction 3 is one off: near but not exact
    out = SO.sequence_hit_rates(R, query, [0], [1], k_probe=2, gt_offset=2, probe_ids=np.array([[3, 2]]))
    assert out["hits"]["top1_near"][0, 0] and not out["hits"]["top1_exact"][0, 0] and out["hits"]["top3_exact"][0, 0]
    # two candidates with equal scores: the lower id ranks first
    R2 = np.vstack([R, R[3:4]])                      # row 6 duplicates row 3
    out = SO.sequence_hit_rates(R2, R2[[3]], [0], [1], k_probe=2, gt_offset=3, probe_ids=np.array([[6, 3]]))
    assert out["hits"]["top1_exact"][0, 0] and out["score_gap"][0, 0] == 0.0


def test_test_ids_resolve_from_all_and_npy(tmp_path):
    assert resolve_test_ids("all", 30, (1, 3, 19)).tolist() == list(range(11))
    p = tmp_path / "ids.npy"
    np.save(p, np.array([4, 1, 7]))
    assert resolve_test_ids(str(p), 30, (1,)).tolist() == [4, 1, 7]
    assert resolve_test_ids([2, 5], 30, (1,)).dtype == np.int64
    with pytest.raises(ValueError):
        resolve_test_ids("nope", 30, (1,))
    with pytest.raises(ValueError):
        resolve_test_ids([30], 30, (1,))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _native.load()


def test_search_workspace_sizes(lib):
    ws = lib.grafp_search_workspace_bytes
    # outside the envelope: 0
    for args in [(0, 100, 128, 1), (1, 100, 48, 1), (1, 100, 60, 1), (1, 100, 512, 1), (1, 100, 128, 129), (1, 3, 128, 4)]:
        assert ws(*args) == 0, args
    # the query planes and the per-slice lists at least
    for n_q, n_db, d, k in [(1, 1, 64, 1), (7, 129, 128, 17), (1000, 10 ** 7, 128, 20), (32768, 5 * 10 ** 7, 256, 128)]:
        need = ws(n_q, n_db, d, k)
        assert need >= 2 * n_q * d * 2 + n_q * 4 + n_q * k * 8, (n_q, n_db, d, k)
    # more key slices for few queries than for many: the per-query list space shrinks as the batch grows
    assert ws(19, 10 ** 7, 128, 20) / 19 > ws(32768, 10 ** 7, 128, 20) / 32768


def test_search_fails_loudly_without_a_device(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    rc = lib.grafp_search_fwd(None, 1, None, None, None, 128, 128, 1, None, None, None, 0, None)
    assert rc != 0
    assert lib.grafp_search_fwd(None, 1, None, None, None, 128, 48, 1, None, None, None, 0, None) == -2
