"""Pins the CPU side against the reference's own golden vectors: the reference's
project_tests generators produced tests/golden/dsl/*.dsl + *.exp (tests/golden/make_golden.py),
and the UNMODIFIED reference server/client (oracle/_ref/dropin/server_ref, compiled from
the reference's sources by oracle/Makefile) replays them.  CPU-only; the replay is skipped
where the reference was never built.

Expected verdicts (SURVEY.md section 4, re-established here at 2000 rows / seed 42): the
reference matches its .exp on every test except
  14  print of an empty result emits uninitialised bytes (query.c:253),
  25  clustered-index position-space bug (SURVEY.md A2),
  26, 27  avg over an empty fetch prints -nan where pandas prints 0.00 (A7),
and 21, 22, 29 match only order-insensitively (index selects return value order)."""
import os
import tempfile

import pytest

import dsl_harness as H

KNOWN_FAIL = {14, 25, 26, 27}
ORDER_INSENSITIVE = {21, 22, 29}


@pytest.fixture(scope="module")
def ref_outputs():
    if not H.ServerPair.available("ref"):
        pytest.skip("oracle/_ref/dropin not built (reference sources absent)")
    with tempfile.TemporaryDirectory(prefix="adb_ref_") as wd:
        yield H.ServerPair("ref", wd).run_suite(range(1, 38))


def test_fixtures_are_complete():
    for t in range(1, 38):
        assert os.path.exists(os.path.join(H.GOLDEN, f"test{t:02d}gen.dsl"))
        assert os.path.exists(os.path.join(H.GOLDEN, f"test{t:02d}gen.exp"))


def test_reference_reproduces_its_golden_vectors(ref_outputs):
    got = {t: H.verdict(o, H.exp_text(t)) for t, o in ref_outputs.items()}
    for t, v in got.items():
        if t in KNOWN_FAIL:
            continue
        assert v in (("exact", "sorted") if t in ORDER_INSENSITIVE else ("exact",)), (t, v)


def test_verifier_rules():
    assert H.clean("\x1b[32mabc\x1b[0m -- note\n\n 1.005,2 \n") == ["abc", "1.00,2"] or \
        H.clean("\x1b[32mabc\x1b[0m -- note\n\n 1.005,2 \n") == ["abc", "1.01,2"]
    assert H.verdict("3\n1\n2\n", "1\n2\n3\n") == "sorted"
    assert H.verdict("1\n2\n", "1\n3\n") == "fail"
    assert H.verdict("-- c\n4.0\n", "4.00\n") == "exact"
