"""The drop-in server with ADB_INDEX_TIES=reference: every index is built on the GPU in the
reference quicksort's tie order, so the milestone-3 replies that list positions or values in
index order (tests 18-31) print the same bytes as the unmodified reference -- including 25 and
27, whose reference answers read wrong rows through the declaration-order quirk (SURVEY.md A2)
and so depend on that tie order."""
import tempfile

import pytest

import dsl_harness as H

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not (H.ServerPair.available("ref") and H.ServerPair.available("b200")),
                                 reason="oracle/_ref/dropin not built")]
TESTS = range(1, 32)
INDEX_ORDERED = range(18, 32)


@pytest.fixture(scope="module", params=["1", "3"], ids=["1gpu", "3gpus"])
def outputs(request):
    with tempfile.TemporaryDirectory(prefix="adb_ref_") as w1, tempfile.TemporaryDirectory(prefix="adb_b200_") as w2:
        ref = H.ServerPair("ref", w1).run_suite(TESTS)
        b200 = H.ServerPair("b200", w2, env={"ADB_GPUS": request.param, "ADB_INDEX_BUILD": "engine",
                                             "ADB_INDEX_TIES": "reference"}).run_suite(TESTS)
        log = open(H.ServerPair("b200", w2).server_log, errors="replace").read()
        yield ref, b200, log


def test_index_ordered_replies_are_byte_identical(outputs):
    ref, b200, log = outputs
    bad = [t for t in INDEX_ORDERED if b200[t] != ref[t]]
    assert not bad, (bad, b200[bad[0]][:300], ref[bad[0]][:300], log[-600:])
    assert not any("Failed" in b200[t] for t in INDEX_ORDERED)
