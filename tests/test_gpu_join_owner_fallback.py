"""The sharded join's owner falls back to the direct probe when the keys routed to it do not fit the
partitioned probe's share of its scratch arena (engine.cu, adb_join_probe_received).

Four contexts, started afresh so that no earlier join has grown an arena, run one hash join with
ADB_JOIN_PROBE=partitioned.  Every one of the 8 Mi probe rows carries the same key, which appears
once on the build side, so all 8 Mi probe keys route to one owner.  Each context reserves its arena
for its own 2 Mi probe rows (adb_peer_exchange_reserve): the build (< 0.1 MiB), the routed rows
(2 Mi x 16 B = 32 MiB), the owner's partitioned probe of 2 Mi keys (~33 MiB), the direct probe's
sums (~0.1 MiB) and the finish (2 Mi x 8 B = 16 MiB), ~81.2 MiB, which grows to ~92.3 MiB with
the arena's slack.  After the build and the routed rows (~32.0 MiB) the hot owner has ~60.3 MiB
left, while the partitioned probe of 8 Mi keys and the finish after it take ~146.7 MiB: it must
probe directly.  The pairs must still be the reference's, in order."""
import ctypes as C

import numpy as np
import pytest

from query_api import Api

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    with pytest.MonkeyPatch.context() as mp:
        for var in ("ADB_SHIM_MIRROR", "ADB_SHIM_EAGER", "ADB_SHARD_MIN_ROWS", "ADB_REBALANCE_MIN", "ADB_TRACE"):
            mp.delenv(var, raising=False)
        a = Api()
        a.lib.adb_host_shutdown()                     # every context starts with an empty arena
        assert a.lib.adb_host_init_multi(4) == 0, a.lib.adb_host_last_error()
        yield a
        a.lib.adb_host_shutdown()


def test_hot_owner_takes_the_direct_probe(api, port, monkeypatch):
    monkeypatch.setenv("ADB_JOIN_PROBE", "partitioned")
    rng = np.random.default_rng(5)
    nb, n_probe, hot = 4096, 8 << 20, 7
    k1 = rng.permutation(np.arange(1, nb + 1)).astype(np.int32)       # the hot key appears once
    p1 = rng.permutation(10 * nb)[:nb].astype(np.int32)
    k2 = np.full(n_probe, hot, np.int32)
    p2 = rng.permutation(n_probe).astype(np.int32)
    R = [C.pointer(api.host_result(x)) for x in (k1, p1, k2, p2)]
    o1, o2 = api.join("hash_join", *R)
    e1, e2 = port.hash_join(k1, p1, k2, p2)
    assert e1.size == n_probe
    assert np.array_equal(api.tuples(o1), e1) and np.array_equal(api.tuples(o2), e2)
    api.drop(o1), api.drop(o2)
