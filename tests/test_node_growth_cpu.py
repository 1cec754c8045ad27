"""Capacity logic of a growing node set, on the host only (numpy): the layout a regrow gives the live rows and the padded
tail, the room new rows take from the tail, when that forces a regrow, and the validation of new node ids and rows."""
import numpy as np
import pytest

from lstep_b200.sampler import (MIN_SLACK, NODE_ID_MAX, new_row_need, plan_capacity, plan_layout, rows_fit, tail_entries)


def test_layout_live_rows_then_empty_spare_rows_and_tail():
    need = np.array([0, 3, 20, 1], np.int64)
    indptr, total = plan_layout(need, 10, min_slack=4)
    cap = plan_capacity(need, 4)
    assert list(cap) == [4, 7, 40, 5]
    assert indptr.shape == (11,)
    assert list(indptr[:5]) == [0, 4, 11, 51, 56]
    assert (indptr[5:] == 56).all()  # rows that are not live yet are empty at the end of the live rows
    assert total == 56 + tail_entries(6, 4) == 56 + 6 * 2 * 4


def test_layout_without_spare_rows_is_the_plain_regrow():
    need = np.array([2, 0, 5], np.int64)
    indptr, total = plan_layout(need, 3)
    want = np.zeros(4, np.int64)
    np.cumsum(plan_capacity(need), out=want[1:])
    assert np.array_equal(indptr, want) and total == int(want[-1])


def test_new_rows_take_need_plus_slack_from_the_tail():
    indptr, total = plan_layout(np.array([1, 1], np.int64), 6, min_slack=MIN_SLACK)
    tail0 = int(indptr[2])
    cap = plan_capacity(np.array([0, 2, 60], np.int64))
    assert list(cap) == [MIN_SLACK, 2 + MIN_SLACK, 120]
    assert rows_fit(2, 6, tail0, total, plan_capacity(np.zeros(4, np.int64)))  # 4 spare rows, 2 * MIN_SLACK each
    assert not rows_fit(2, 6, tail0, total, plan_capacity(np.zeros(5, np.int64)))  # beyond the row capacity
    assert not rows_fit(2, 6, tail0, total, cap)  # a hub row needs more than the tail holds: regrow


def test_new_row_need_counts_endpoints_of_new_rows_only():
    src = np.array([1, 5, 6, 6], np.int64)
    dst = np.array([5, 2, 6, 7], np.int64)
    assert list(new_row_need(src, dst, 5, 3)) == [2, 3, 1]
    assert list(new_row_need(src, dst, 8, 2)) == [0, 0]


class _Rows:
    """The HostFed validation of new rows and ids, without a device."""

    def __init__(self, d=4, max_nodes=None, V1=10):
        from lstep_b200.hostfeed import HostFed
        self.h = HostFed.__new__(HostFed)
        self.h.d, self.h.max_nodes, self.h.V1 = d, max_nodes, V1
        self.h._growable_sampler = lambda: None


def test_rows_validation():
    h = _Rows().h
    assert h._rows_array([[1, 2, 3, 4]], 2).dtype == np.float32
    for bad in ([[1, 2, 3]], [1, 2, 3, 4], [["a", 1, 2, 3]], [[np.nan, 0, 0, 0]], [[np.inf, 0, 0, 0]]):
        with pytest.raises(ValueError):
            h._rows_array(bad, 2)
    assert h._rows_array([0, 0, 0, 1], 1).shape == (4,)
    with pytest.raises(ValueError):
        h._rows_array([[0, 0, 0, 1]], 1)


def test_id_limits():
    h = _Rows(max_nodes=50).h
    h._check_new_ids(49)
    with pytest.raises(IndexError):
        h._check_new_ids(50)
    h = _Rows().h
    h._check_new_ids(NODE_ID_MAX)
    with pytest.raises(IndexError):
        h._check_new_ids(NODE_ID_MAX + 1)


def test_new_nodes_for_batch():
    h = _Rows(V1=10).h
    a = np.array([3, 9], np.int64)
    assert h._new_nodes_for([a, a]) == 0
    assert h._new_nodes_for([a, np.array([12, 1], np.int64)]) == 3
    with pytest.raises(IndexError):
        h._new_nodes_for([a, np.array([-1], np.int64)])
    h.max_nodes = 12
    with pytest.raises(IndexError):
        h._new_nodes_for([np.array([12], np.int64)])
