"""The joins in numpy, exact and vectorised, and a Python mirror of the join's launch geometry on
one engine context (csrc/engine.cu, csrc/hash_join.cu).  Test plumbing.

hash_join / nested_loop_join give the oracle's pair lists (tests/test_gpu_join_geometry.py pins
them to it): probe-major over side two with side one's insertion order inside a key, and the
nested loop outer-major over side one.  A stable sort, two binary searches and a repeat take
seconds where the oracle's multimap takes minutes at 100 M rows."""
import numpy as np

I32MIN, I32MAX = -2**31, 2**31 - 1


def hash_join(k1, p1, k2, p2):
    """(side one positions, side two positions) of every pair with k1[i] == k2[j], j-major, then
    i in side one's order."""
    k1, p1, k2, p2 = (np.ascontiguousarray(x, np.int32) for x in (k1, p1, k2, p2))
    sk, order = stable_sort(k1)
    keys, rows = stable_sort(k2)                       # the searches walk sk in order
    lo, cnt = np.empty(k2.size, np.int64), np.empty(k2.size, np.int64)
    lo[rows] = np.searchsorted(sk, keys, "left")
    cnt[rows] = np.searchsorted(sk, keys, "right") - lo[rows]
    first = np.cumsum(cnt) - cnt                        # every probe row's first output slot
    idx = np.arange(int(cnt.sum()), dtype=np.int64) + np.repeat(lo - first, cnt)
    return p1[order[idx]], np.repeat(p2, cnt)


def stable_sort(k):
    """(sorted keys, their rows) with equal keys in row order: one sort of key * 2^32 + row."""
    c = np.sort((k.astype(np.int64) << 32) | np.arange(k.size, dtype=np.int64))
    return (c >> 32).astype(np.int32), c & 0xFFFFFFFF


def nested_loop_join(k1, p1, k2, p2):
    """The same pairs, i-major, then j in side two's order."""
    o2, o1 = hash_join(k2, p2, k1, p1)
    return o1, o2


# ---- the join's geometry ---------------------------------------------------------------------------
HASH_MUL = 0x9E3779B1                   # the join hash: h = key * HASH_MUL mod 2^32 (a bijection)
HASH_INV = pow(HASH_MUL, -1, 1 << 32)
ROUTE_MUL = 0x85EBCA6B                  # the owner hash of the sharded join (route_owner)
RADIX_TILE = 4096                       # kRadixTile: rows per tile of the probe's partition pass
SHARED_SLOTS = 2048                     # HJ_BUILD_SLOTS: the shared-memory table of hj_table_build_kernel
PIECE_PARTITIONED = 512                 # rows per warp piece of the partitioned probe (HJ_SUB / 8)
STEP_ROWS = 128                         # rows per step of the expansion: 32 lanes x HJ_EXP_STEPS


def join_hash(keys):
    return (np.asarray(keys).astype(np.int64).astype(np.uint64) * np.uint64(HASH_MUL)) & np.uint64(0xFFFFFFFF)


def keys_of_hashes(h):
    """The keys whose join hash is h (the inverse of the multiplier)."""
    h = np.asarray(h, np.uint64)
    return ((h * np.uint64(HASH_INV)) & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.int32)


def partition_of(keys, bits):
    """hj_pid: the top `bits` bits of the join hash."""
    return (join_hash(keys) >> np.uint64(32 - bits)).astype(np.int64)


def slice_of(keys):
    """The table slice a probe row is grouped by in the partitioned probe: the top 8 hash bits."""
    return partition_of(keys, 8)


def route_owner(keys, parts):
    h = (np.asarray(keys).astype(np.int64).astype(np.uint64) * np.uint64(ROUTE_MUL)) & np.uint64(0xFFFFFFFF)
    return ((h * np.uint64(parts)) >> np.uint64(32)).astype(np.int64)


def part_bits(nb):
    """join_part_bits: partitions of at most ~1024 rows on average, 1 to 20 bits."""
    bits = 1
    while bits < 20 and (nb >> bits) > 1024:
        bits += 1
    return bits


def table_slots(rows):
    """hj_geometry_local_kernel: a power of two >= 16 at <= 80 % load, 0 for an empty partition."""
    if rows == 0:
        return 0
    cap = 16
    while cap < rows + rows // 4 + 1:
        cap <<= 1
    return cap


def builds_in_shared_memory(rows):
    return 0 < table_slots(rows) <= SHARED_SLOTS


def probe_geom(n, sm_count):
    """hj_probe_geom, the direct probe: (CTAs, warps, rows per warp piece)."""
    blocks = min(-(-n // 256), sm_count * 8) or 1
    warps = blocks * 8
    rows = -(-(-(-n // warps)) // 32) * 32 or 32
    return blocks, warps, rows


def window_tiles(n):
    """probe_window_tiles: whole 4096-row tiles per window of the partitioned probe, <= 256 windows."""
    return (-(-n // RADIX_TILE) + 255) // 256


def windows(n):
    """radix_segments(n, window_tiles(n))."""
    tiles, wt = -(-n // RADIX_TILE), window_tiles(n)
    return 1 if wt >= tiles else -(-tiles // wt)


def row_scan_is_warp_wide(n):
    """launch_radix_pass_segmented scans a window's histogram rows with rx_row_scan_warp_kernel up
    to 512 tiles per window, with rx_row_scan_kernel beyond."""
    return window_tiles(n) <= 512


def partitioned_by_default(nb, n_probe):
    """join_count's size rule for the one-context join."""
    return nb >= 6 << 20 and n_probe >= 4 << 20


def owner_partitioned_by_default(n_recv, nb_owner):
    """adb_join_probe_received's size rule (given arena room) for an owner of the sharded join."""
    return n_recv >= 4 << 20 and nb_owner >= 24 << 20
