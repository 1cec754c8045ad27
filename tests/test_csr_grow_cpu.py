"""Host side of the growable CSR (l-step_b200/sampler.py): batch validation and capacity planning are numpy functions, so
they are checked here without a device."""
import numpy as np
import pytest

from lstep_b200.sampler import MIN_SLACK, check_edges, overflow_rows, plan_capacity, row_counts


def _batch(n=6):
    src = np.array([1, 2, 3, 3, 4, 1][:n], dtype=np.int64)
    dst = np.array([2, 3, 3, 5, 1, 2][:n], dtype=np.int64)
    eid = np.arange(10, 10 + n, dtype=np.int64)
    t = np.array([1.0, 1.0, 2.0, 2.5, 2.5, 3.0][:n])
    return src, dst, eid, t


def test_check_edges_accepts_and_normalises():
    src, dst, eid, t = _batch()
    a = check_edges(list(src), dst.astype(np.int32), eid, t.astype(np.float32), num_rows=6, last_time=1.0)
    assert [x.dtype for x in a] == [np.int64, np.int64, np.int64, np.float64]
    assert all(x.flags.c_contiguous for x in a)
    assert np.array_equal(a[0], src) and np.array_equal(a[3], t)
    # ties with the last time ingested are allowed; an int stands for consecutive edge ids
    assert check_edges(src, dst, 5, t, num_rows=6, last_time=1.0)[2].tolist() == [5, 6, 7, 8, 9, 10]
    assert check_edges(src[:1], dst[:1], np.int64(7), t[:1], num_rows=6)[2].tolist() == [7]
    assert len(check_edges([], [], [], [], num_rows=1)[0]) == 0


@pytest.mark.parametrize("case", ["length", "length_eid", "id_high", "id_negative", "nan", "inf", "decreasing", "before_last",
                                  "eid_high", "eid_negative", "eid_base_high"])
def test_check_edges_rejections(case):
    src, dst, eid, t = _batch()
    last, eids, rows = 0.5, eid, 6
    err = ValueError
    if case == "length":
        dst = dst[:-1]
    elif case == "length_eid":
        eids = eid[:-1]
    elif case == "id_high":
        src = src.copy()
        src[3] = 6
        err = IndexError
    elif case == "id_negative":
        dst = dst.copy()
        dst[0] = -1
        err = IndexError
    elif case == "nan":
        t = t.copy()
        t[2] = np.nan
    elif case == "inf":
        t = t.copy()
        t[-1] = np.inf
    elif case == "decreasing":
        t = t.copy()
        t[4] = 2.4
    elif case == "before_last":
        last = 1.5
    elif case == "eid_high":
        eids = eid.copy()
        eids[1] = 2 ** 31
    elif case == "eid_negative":
        eids = eid.copy()
        eids[1] = -3
    elif case == "eid_base_high":
        eids = 2 ** 31 - 3  # ids 2^31-3 .. 2^31+2
    with pytest.raises(err):
        check_edges(src, dst, eids, t, num_rows=rows, last_time=last)


def test_row_counts_count_self_loops_twice():
    rows, cnt = row_counts(np.array([3, 1, 3]), np.array([3, 2, 1]))
    assert rows.tolist() == [1, 2, 3] and cnt.tolist() == [2, 1, 3]


def test_overflow_rows_looks_at_touched_rows_only():
    fill = np.array([0, 4, 1, 3, 9, 0], dtype=np.int64)
    cap = np.array([0, 5, 2, 4, 2, 1], dtype=np.int64)  # row 4 is over capacity already but the batch does not touch it
    src = np.array([1, 2, 5])
    dst = np.array([3, 1, 5])
    # row 1 gets 2 (4 + 2 > 5), row 2 gets 1 (fits), row 3 gets 1 (fits), row 5 gets 2 (self-loop: 0 + 2 > 1)
    assert overflow_rows(fill, cap, src, dst).tolist() == [1, 5]
    assert overflow_rows(fill, cap, np.array([2]), np.array([3])).size == 0


def test_plan_capacity_gives_every_row_room():
    need = np.array([0, 1, 5, MIN_SLACK, 3 * MIN_SLACK, 10 ** 6], dtype=np.int64)
    cap = plan_capacity(need)
    assert (cap - need >= MIN_SLACK).all()  # even rows no batch touched get the floor
    assert (cap >= 2 * need).all()  # rows can double before the next regrow
    assert cap.tolist() == (need + np.maximum(MIN_SLACK, need)).tolist()
    assert plan_capacity(np.zeros(3, np.int64), min_slack=0).tolist() == [0, 0, 0]


def test_planned_stream_regrows_rarely_and_never_overflows():
    """The host planner over a hub-heavy stream from empty: after each regrow nothing overflows, the batch fits, and the
    number of regrows stays logarithmic in the entry count."""
    rng = np.random.default_rng(0)
    rows, B, nb = 500, 200, 300
    fill = np.zeros(rows, np.int64)
    cap = plan_capacity(fill)
    regrows = 0
    for _ in range(nb):
        src = np.minimum(rng.zipf(1.2, B), rows - 1).astype(np.int64)
        dst = rng.integers(0, rows, B)
        if overflow_rows(fill, cap, src, dst).size:
            need = fill.copy()
            r, c = row_counts(src, dst)
            need[r] += c
            cap = plan_capacity(need)
            regrows += 1
        assert overflow_rows(fill, cap, src, dst).size == 0
        r, c = row_counts(src, dst)
        fill[r] += c
        assert (fill <= cap).all()
    assert fill.sum() == 2 * B * nb
    assert regrows <= 2 * np.log2(fill.max()) + 2, regrows
