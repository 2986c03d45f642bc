"""CPU tests of the occupancy bucket rule of StreamSampler steps: ``occupancy_slots`` (the library's ``fmt_occupancy_slots``, shared by
Python and C) against a restatement of the rule for every slot count and every ready count, its refusals, and the C declarations of
the two entry points."""
import ctypes as C
import os
import re
import sys

import pytest

from __graft_entry__ import load_package

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    p = load_package()
    sys.modules[p.__name__ + ".build"].build()
    return p


def bucket(S, k):
    """The smallest of {1, 2, 4, ..., the powers of two below S, S} that is >= k."""
    sizes = [1 << i for i in range(9) if (1 << i) < S] + [S]
    return min(b for b in sizes if b >= k)


def test_occupancy_slots_matches_the_rule(pkg):
    for S in range(1, 257):
        for k in range(1, S + 1):
            assert pkg.occupancy_slots(S, k) == bucket(S, k), (S, k)


def test_occupancy_slots_examples(pkg):
    assert [pkg.occupancy_slots(256, k) for k in (1, 2, 3, 5, 8, 9, 129, 256)] == [1, 2, 4, 8, 8, 16, 256, 256]
    assert [pkg.occupancy_slots(16, k) for k in (1, 2, 3, 5, 9, 16)] == [1, 2, 4, 8, 16, 16]
    assert [pkg.occupancy_slots(24, k) for k in (16, 17, 24)] == [16, 24, 24]     # no power of two between 16 and 24
    assert pkg.occupancy_slots(1, 1) == 1


@pytest.mark.parametrize("S,k", [(0, 1), (1, 0), (4, 5), (257, 1), (257, 257), (-1, -1), (8, -3)])
def test_occupancy_slots_refuses_bad_arguments(pkg, S, k):
    with pytest.raises(ValueError):
        pkg.occupancy_slots(S, k)
    assert sys.modules[pkg.__name__ + "._cabi"].load_library().fmt_occupancy_slots(S, k) < 0


@pytest.mark.parametrize("S,k", [(4.0, 1), (4, True), ("4", 1)])
def test_occupancy_slots_refuses_non_integers(pkg, S, k):
    with pytest.raises(ValueError):
        pkg.occupancy_slots(S, k)


def test_entry_points_are_declared(pkg):
    cabi = sys.modules[pkg.__name__ + "._cabi"]
    hdr = open(os.path.join(ROOT, "include", "fmt_b200.h")).read()
    assert re.search(r"FMT_API int32_t fmt_occupancy_slots\(int32_t plan_slots, int32_t n_ready\);", hdr)
    assert re.search(r"FMT_API int32_t fmt_last_window_slots\(const FmtHandle\* h\);", hdr)
    lib = cabi.load_library()
    assert lib.fmt_occupancy_slots.argtypes == [C.c_int32, C.c_int32] and lib.fmt_occupancy_slots.restype is C.c_int32
    assert lib.fmt_last_window_slots.argtypes == [C.c_void_p] and lib.fmt_last_window_slots.restype is C.c_int32
    assert lib.fmt_last_window_slots(None) == 0
