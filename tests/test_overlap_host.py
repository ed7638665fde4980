"""The hazard predicate of the K1 / K3 launch-boundary overlap, without a device: two launches conflict on a
read-after-write, write-after-read or write-after-write of at least one byte."""
import ctypes

import pytest

R, W = 0, 1


def conflict(prev, nxt):
    from beast_tokenizer_b200 import _lib
    lib = _lib.load()

    def arr(ranges):
        flat = [v for r in ranges for v in r]
        return (ctypes.c_int64 * max(len(flat), 1))(*flat), len(ranges)

    a, na = arr(prev)
    b, nb = arr(nxt)
    rc = lib.beast_debug_ranges_conflict(a, na, b, nb)
    assert rc in (0, 1), rc
    return bool(rc)


@pytest.mark.parametrize("prev, nxt, expected", [
    ([(0, 100, W)], [(50, 150, R)], True),                  # read after write
    ([(0, 100, R)], [(50, 150, W)], True),                  # write after read
    ([(0, 100, W)], [(99, 100, W)], True),                  # write after write, last byte
    ([(0, 100, R)], [(0, 100, R)], False),                  # both only read
    ([(0, 100, W)], [(100, 200, R)], False),                # touching: next starts where prev ends
    ([(100, 200, W)], [(0, 100, W)], False),                # touching from below
    ([(0, 100, W)], [(50, 50, R)], False),                  # empty range inside a written one
    ([(50, 50, W)], [(0, 100, W)], False),
    ([(0, 100, W)], [(10, 20, R)], True),                   # contained
    ([(10, 20, R)], [(0, 100, W)], True),                   # containing
    ([(0, 10, R), (20, 30, W)], [(10, 20, W), (30, 40, R)], False),
    ([(0, 10, R), (20, 30, W)], [(10, 20, W), (29, 40, R)], True),
    ([], [(0, 100, W)], False),
    ([(0, 100, W)], [], False),
    ([(1 << 40, (1 << 40) + 8, W)], [((1 << 40) + 4, (1 << 40) + 12, R)], True),
])
def test_ranges_conflict(prev, nxt, expected):
    assert conflict(prev, nxt) == expected
    # the predicate is symmetric in which launch came first
    assert conflict(nxt, prev) == expected


def test_ranges_conflict_rejects_bad_arguments():
    from beast_tokenizer_b200 import _lib
    lib = _lib.load()
    one = (ctypes.c_int64 * 3)(0, 1, 1)
    assert lib.beast_debug_ranges_conflict(one, -1, one, 1) == -2
    assert lib.beast_debug_ranges_conflict(one, 9, one, 1) == -2
    assert lib.beast_debug_ranges_conflict(None, 1, one, 1) == -1


def test_overlap_switches_need_no_device():
    from beast_tokenizer_b200 import _lib
    lib = _lib.load()
    assert lib.beast_overlap_count() >= 0
    prev = lib.beast_debug_force_wait(1)
    assert lib.beast_debug_force_wait(prev) == 1
