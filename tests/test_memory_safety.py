"""Memory-safety net for a GPU pool on which compute-sanitizer is closed (DESIGN.md section 3.8).

  * guard regions: every device array of an env between two 4 KiB regions of 0xA5 (GCB_GUARD_BYTES); after every kernel
    of the env API has run on awkward env counts the guards must be intact;
  * the CHECKED build of the same sources (libgymchess_b200_checked.so, -DGCB_CHECKED): every indexed global access of the
    env kernels verifies its index against the extent of its array; the exercise must report no violation;
  * the self-test build (-DGCB_CHECKED -DGCB_SELFTEST_OOB) re-introduces the round-1 bug -- the statistics row
    read-modify-write of warps that lie wholly past the env range (value-preserving, so guard bytes cannot see it) -- and
    the checks MUST flag it: the net catches that class of bug.
"""
import pytest

from tests import memsafety_exercise as mx

pytestmark = pytest.mark.gpu


def test_guard_regions_stay_intact_on_the_product_build():
    res = mx.run()["steps"]
    assert res["checked"] == 0 and res["guard_bad_bytes"] == 0 and res["violations"] == 0, res


def test_checked_build_reports_no_index_violation():
    res = mx.run("checked")["steps"]
    assert res["checked"] == 1 and res["violations"] == 0 and res["guard_bad_bytes"] == 0, res


def test_checked_build_catches_the_reintroduced_stat_row_bug():
    res = mx.run("checked_selftest")["steps_quick"]
    assert res["checked"] == 1 and res["violations"] & 1, res          # bit 0 = CHK_STAT_ROW
    assert res["guard_bad_bytes"] == 0                                 # ... which guard bytes alone cannot see (it adds 0)
