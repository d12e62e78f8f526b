"""ctypes binding of the engine's C-ABI (``include/adb_engine.h`` -> ``libadb_b200.so``).

Plumbing only: this module moves numpy arrays in and out of HBM and forwards every
operator to the CUDA library.  It never computes a result itself and has no fallback --
``Engine()`` raises ``EngineError`` when the library is missing or no device opens.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_I32P = C.POINTER(C.c_int32)
_I64P = C.POINTER(C.c_int64)


class EngineError(RuntimeError):
    pass


def lib_path() -> str:
    return os.path.join(_HERE, "libadb_b200.so")


def build_native(quiet: bool = True) -> str:
    """Compile every CUDA source for sm_100a into libadb_b200.so (nvcc cross-compiles)."""
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")] + (["-s"] if quiet else []),
                   check=True)
    host = os.path.join(_HERE, "host")
    if os.path.exists(os.path.join(host, "Makefile")):
        subprocess.run(["make", "-C", host] + (["-s"] if quiet else []), check=True)
    return lib_path()


class _AggStruct(C.Structure):
    _fields_ = [("sum", C.c_int64), ("count", C.c_int64), ("min", C.c_int32), ("max", C.c_int32)]


@dataclass
class Agg:
    sum: int
    count: int
    min: int
    max: int

    @property
    def avg(self) -> float:
        """(double)sum / (double)num_tuples, /root/reference/src/query.c:314."""
        return float(np.float64(self.sum) / np.float64(self.count)) if self.count else float("nan")


class DevBuf:
    """A device allocation owned by the engine's stream-ordered pool."""

    def __init__(self, eng: "Engine", nbytes: int):
        self.eng, self.nbytes = eng, int(nbytes)
        p = C.c_void_p()
        eng._ck(eng.lib.adb_alloc(C.byref(p), self.nbytes))
        self.ptr = p.value

    def free(self):
        if self.ptr:
            self.eng.lib.adb_free(C.c_void_p(self.ptr))
            self.ptr = None

    def i32(self, offset_elems: int = 0):
        return C.cast(C.c_void_p(self.ptr + 4 * offset_elems), _I32P)

    def i64(self, offset_elems: int = 0):
        return C.cast(C.c_void_p(self.ptr + 8 * offset_elems), _I64P)

    def void(self, offset_bytes: int = 0):
        return C.c_void_p(self.ptr + offset_bytes)

    def to_host(self, n: int, dtype=np.int32, offset_bytes: int = 0) -> np.ndarray:
        out = np.empty(int(n), dtype=dtype)
        if n:
            self.eng._ck(self.eng.lib.adb_download(out.ctypes.data_as(C.c_void_p),
                                                   self.void(offset_bytes), out.nbytes))
        return out


def _bound(x):
    if x is None:
        return None, None
    box = C.c_int32(int(x))
    return C.pointer(box), box


class Engine:
    """One engine per process (one process per GPU)."""

    _SIGS = {
        "adb_init": (C.c_int32, [C.c_int]),
        "adb_shutdown": (C.c_int32, []),
        "adb_last_error": (C.c_char_p, []),
        "adb_version": (C.c_char_p, []),
        "adb_sm_count": (C.c_int, []),
        "adb_alloc": (C.c_int32, [C.POINTER(C.c_void_p), C.c_size_t]),
        "adb_free": (C.c_int32, [C.c_void_p]),
        "adb_upload": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
        "adb_download": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
        "adb_upload_async": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
        "adb_download_async": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
        "adb_memset": (C.c_int32, [C.c_void_p, C.c_int, C.c_size_t]),
        "adb_sync": (C.c_int32, []),
        "adb_stream": (C.c_void_p, []),
        "adb_set_stream": (C.c_int32, [C.c_void_p]),
        "adb_host_alloc": (C.c_int32, [C.POINTER(C.c_void_p), C.c_size_t]),
        "adb_host_free": (C.c_int32, [C.c_void_p]),
        "adb_host_register": (C.c_int32, [C.c_void_p, C.c_size_t]),
        "adb_host_unregister": (C.c_int32, [C.c_void_p]),
        "adb_timer_start": (C.c_int32, []),
        "adb_timer_stop": (C.c_int32, [C.POINTER(C.c_float)]),
        "adb_launch_count": (C.c_int64, []),
        "adb_mark": (C.c_int32, [C.c_int32]),
        "adb_chain_marks": (C.c_int32, [C.c_int32]),
        "adb_mark_elapsed": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
        "adb_select_scan": (C.c_int32, [_I32P, C.c_int64, _I32P, _I32P, C.c_int32, _I32P, _I64P, _I64P]),
        "adb_select_count": (C.c_int32, [_I32P, C.c_int64, _I64P, _I32P, _I32P, _I64P, _I64P]),
        "adb_select_emit": (C.c_int32, [_I32P, C.c_int32, _I32P]),
        "adb_select_emit_fetch_agg": (C.c_int32, [_I32P, _I32P, _I32P, C.POINTER(_AggStruct), C.POINTER(_AggStruct)]),
        "adb_select_generation": (C.c_uint64, []),
        "adb_select_index_count": (C.c_int32, [C.c_void_p, C.c_int32, _I32P, _I32P, _I64P, _I64P]),
        "adb_select_index_emit": (C.c_int32, [C.c_void_p, _I32P]),
        "adb_fetch": (C.c_int32, [_I32P, _I32P, C.c_int64, _I64P, C.c_int32, _I32P]),
        "adb_aggregate": (C.c_int32, [_I32P, C.c_int64, _I64P, C.POINTER(_AggStruct), C.POINTER(_AggStruct)]),
        "adb_agg_combine": (C.c_int32, [C.POINTER(_AggStruct), C.c_int32, C.POINTER(_AggStruct), C.POINTER(_AggStruct)]),
        "adb_agg_export": (C.c_int32, [C.POINTER(_AggStruct), C.c_void_p, C.c_void_p]),
        "adb_agg_import": (C.c_int32, [C.c_void_p, C.c_void_p, C.POINTER(_AggStruct)]),
        "adb_format_i32_count": (C.c_int32, [_I32P, C.c_int64, _I64P]),
        "adb_format_i32_emit": (C.c_int32, [C.c_void_p]),
        "adb_csv_index": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, _I64P]),
        "adb_csv_parse": (C.c_int32, [C.c_int32, C.POINTER(C.c_void_p)]),
        "adb_csv_parse_piece": (C.c_int32, [C.c_int32, C.POINTER(C.c_void_p), _I32P, _I32P, _I32P]),
        "adb_csv_fill": (C.c_int32, [_I32P]),
        "adb_peer_create": (C.c_int32, [C.c_int32, C.c_int32, C.c_char_p]),
        "adb_peer_connect": (C.c_int32, [C.c_char_p]),
        "adb_agg_combine_allreduce": (C.c_int32, [C.POINTER(_AggStruct), C.c_int32, C.POINTER(_AggStruct), C.POINTER(_AggStruct)]),
        "adb_peer_destroy": (C.c_int32, []),
        "adb_peer_join_create": (C.c_int32, [C.c_int64, C.c_char_p]),
        "adb_peer_join_connect": (C.c_int32, [C.c_char_p]),
        "adb_peer_exchange_pairs": (C.c_int32, [C.c_int32, _I32P, _I32P, C.c_int64, _I64P,
                                                C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
        "adb_chain_select_fetch_agg_exchange": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P, _I32P, _I32P, _I64P,
                                                            C.POINTER(_AggStruct), C.c_int32, C.POINTER(_AggStruct)]),
        "adb_add": (C.c_int32, [_I32P, _I32P, C.c_int64, _I64P, _I32P]),
        "adb_sub": (C.c_int32, [_I32P, _I32P, C.c_int64, _I64P, _I32P]),
        "adb_chain_select_fetch_agg": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P, _I32P, _I32P, _I64P, C.POINTER(_AggStruct)]),
        "adb_shared_select_count": (C.c_int32, [_I32P, C.c_int64, _I32P, _I32P, C.c_int32, _I64P]),
        "adb_shared_select_emit": (C.c_int32, [C.POINTER(C.c_void_p), C.c_int64]),
        "adb_shared_select_plan": (C.c_int32, [_I32P, _I32P, C.c_int32, C.c_void_p, C.c_size_t, C.POINTER(C.c_uint32)]),
        "adb_index_create": (C.c_int32, [_I32P, _I32P, C.c_int64, C.c_int32, C.POINTER(C.c_void_p)]),
        "adb_index_destroy": (C.c_int32, [C.c_void_p]),
        "adb_index_sort": (C.c_int32, [_I32P, C.c_int64, _I32P, _I32P]),
        "adb_index_sort_ref_ties": (C.c_int32, [_I32P, C.c_int64, _I32P, _I32P]),
        "adb_hash_join_count": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P, C.c_int64, _I64P]),
        "adb_nested_loop_join_count": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P, C.c_int64, _I64P]),
        "adb_join_emit": (C.c_int32, [_I32P, _I32P]),
        "adb_route_pairs": (C.c_int32, [_I32P, _I32P, C.c_int64, C.c_int32, _I32P, _I32P, _I64P]),
        "adb_synth_uniform": (C.c_int32, [_I32P, C.c_int64, C.c_uint64, C.c_uint64, C.c_int32, C.c_uint32]),
        # several contexts in one process (one per GPU) + in-process peer exchange
        "adb_device_count": (C.c_int32, []),
        "adb_ctx_init": (C.c_int32, [C.c_int32, C.c_int]),
        "adb_ctx_select": (C.c_int32, [C.c_int32]),
        "adb_ctx_current": (C.c_int32, []),
        "adb_ctx_wait": (C.c_int32, [C.c_int32]),
        "adb_copy_from_ctx": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t]),
        "adb_launch_count_all": (C.c_int64, []),
        "adb_peer_connect_local": (C.c_int32, [C.c_int32]),
        "adb_peer_join_connect_local": (C.c_int32, [C.c_int64]),
        "adb_select_count_base": (C.c_int32, [_I32P, C.c_int64, _I32P, _I32P, C.c_int32, _I64P, _I64P]),
        "adb_select_emit_fetch_agg_exchange": (C.c_int32, [_I32P, _I32P, _I32P, C.POINTER(_AggStruct),
                                                           C.POINTER(_AggStruct), C.POINTER(_AggStruct)]),
        "adb_fetch_sharded": (C.c_int32, [C.POINTER(C.c_void_p), C.c_int32, C.c_int64, _I32P, C.c_int64, _I64P, _I32P]),
        "adb_shared_select_count_base": (C.c_int32, [_I32P, C.c_int64, C.c_int32, _I32P, _I32P, C.c_int32, _I64P]),
        "adb_index_set_slice": (C.c_int32, [C.c_void_p, C.c_int32]),
        "adb_narrow_u64_to_i32": (C.c_int32, [C.c_void_p, C.c_int64, _I32P]),
        "adb_widen_i32_to_u64": (C.c_int32, [_I32P, C.c_int64, C.c_void_p]),
        "adb_iota_i32": (C.c_int32, [_I32P, C.c_int64, C.c_int32]),
        "adb_update_rows": (C.c_int32, [_I32P, C.c_int64, _I32P, C.c_int64, C.c_int32, C.c_int32]),
        "adb_delete_rows_plan": (C.c_int32, [C.c_int64, _I32P, C.c_int64, C.c_int32, _I64P]),
        "adb_delete_rows_apply": (C.c_int32, [_I32P, _I32P]),
        "adb_join_build": (C.c_int32, [_I32P, _I32P, C.c_int64, C.c_int64]),
        "adb_peer_exchange_reserve": (C.c_int32, [C.c_int64, C.c_int64, C.c_int64]),
        "adb_copy_from_ctx_ready": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t]),
        "adb_route_rows": (C.c_int32, [C.c_int32, C.c_int64, _I32P, C.c_int64, _I64P, C.POINTER(_I32P),
                                       C.POINTER(C.c_void_p)]),
        "adb_route_finish32": (C.c_int32, [C.c_int32, _I32P, C.c_int64]),
        "adb_join_route_probe": (C.c_int32, [C.c_int32, _I32P, C.c_int64, _I64P, C.POINTER(_I32P),
                                             C.POINTER(C.c_void_p)]),
        "adb_join_recv_buffers": (C.c_int32, [C.c_int64, C.POINTER(_I32P), C.POINTER(C.c_void_p)]),
        "adb_join_probe_received": (C.c_int32, [C.c_int64]),
        "adb_join_finish_routed": (C.c_int32, [C.c_int32, _I32P, _I32P, C.c_int64, C.c_int32, _I64P]),
        "adb_alloc_cached_on": (C.c_int32, [C.c_int32, C.POINTER(C.c_void_p), C.c_size_t]),
        "adb_free_cached_on": (C.c_int32, [C.c_int32, C.c_void_p]),
        "adb_chain_select_agg": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P, _I64P, C.POINTER(_AggStruct),
                                             C.POINTER(_AggStruct)]),
        "adb_synth_affine": (C.c_int32, [_I32P, C.c_int64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64]),
        "adb_histogram_i32": (C.c_int32, [_I32P, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_uint64)]),
        "adb_rank_hist": (C.c_int32, [_I32P, C.c_int64, C.POINTER(C.c_uint32), C.c_int32, C.c_int32,
                                      C.POINTER(C.c_uint32)]),
        "adb_route_range": (C.c_int32, [_I32P, C.c_int64, C.c_int64, _I32P, C.c_int32, _I32P, _I32P, _I64P]),
        "adb_index_sort_pairs": (C.c_int32, [_I32P, _I32P, C.c_int64, _I32P, _I32P]),
    }

    def __init__(self, device: int = 0):
        path = lib_path()
        if not os.path.exists(path):
            raise EngineError(f"{path} is not built (run __graft_entry__.build()); "
                              "the engine has no CPU fallback")
        self.lib = C.CDLL(path)
        for name, (res, args) in self._SIGS.items():
            fn = getattr(self.lib, name)
            fn.restype, fn.argtypes = res, args
        self._ck(self.lib.adb_init(int(device)))
        self.device = device
        self.sm_count = self.lib.adb_sm_count()

    # ---- plumbing ------------------------------------------------------------------
    def _ck(self, status: int):
        if status != 0:
            raise EngineError(f"adb status {status}: {self.lib.adb_last_error().decode()}")

    def close(self):
        self.lib.adb_shutdown()

    def peer_setup(self, dist) -> None:
        """Map every rank's aggregate mailbox into this process (adb_peer_create ->
        all-gather of the 64-byte IPC handles over `dist` -> adb_peer_connect).  After this,
        adb_agg_combine_allreduce does the aggregate exchange inside one kernel over NVLink
        peer memory.  `dist` is torch.distributed (plumbing: it only carries the handles)."""
        import torch
        world, rank = dist.get_world_size(), dist.get_rank()
        mine = C.create_string_buffer(64)
        self._ck(self.lib.adb_peer_create(world, rank, mine))
        dev = torch.device("cuda", self.device)
        t = torch.frombuffer(bytearray(mine.raw), dtype=torch.uint8).to(dev)
        allh = torch.zeros(64 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, t)
        self._ck(self.lib.adb_peer_connect(bytes(allh.cpu().numpy().tobytes())))
        dist.barrier()                                   # every mailbox is mapped everywhere

    def peer_join_setup(self, dist, cap_pairs: int) -> None:
        """Reserve this rank's receive buffer for the join's pair exchange (cap_pairs pairs per
        side) and map every peer's (adb_peer_join_create -> all-gather of the handles ->
        adb_peer_join_connect).  Needs peer_setup first."""
        import torch
        world = dist.get_world_size()
        mine = C.create_string_buffer(64)
        self._ck(self.lib.adb_peer_join_create(int(cap_pairs), mine))
        dev = torch.device("cuda", self.device)
        t = torch.frombuffer(bytearray(mine.raw), dtype=torch.uint8).to(dev)
        allh = torch.zeros(64 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, t)
        self._ck(self.lib.adb_peer_join_connect(bytes(allh.cpu().numpy().tobytes())))
        dist.barrier()

    def alloc(self, nbytes: int) -> DevBuf:
        return DevBuf(self, nbytes)

    def alloc_i32(self, n: int) -> DevBuf:
        return DevBuf(self, 4 * max(int(n), 1))

    def upload(self, a: np.ndarray) -> DevBuf:
        a = np.ascontiguousarray(a)
        buf = DevBuf(self, max(a.nbytes, 16))
        if a.nbytes:
            self._ck(self.lib.adb_upload(buf.void(), a.ctypes.data_as(C.c_void_p), a.nbytes))
        return buf

    def csv_load(self, text, n_cols: int, skip_lines: int = 1, d_text: DevBuf | None = None):
        """Bulk load: the bytes of a CSV file -> n_cols device columns (adb_csv_index +
        adb_csv_parse; replaces load_db's ingest loop, db_manager.c:304-318).  `text` is
        bytes / a uint8 numpy array on the host, or pass the device copy as d_text together
        with the byte count as `text`.  Returns ([DevBuf per column], rows)."""
        own = d_text is None
        if own:
            a = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else text
            nbytes = int(a.size)
            d_text = self.upload(a) if nbytes else self.alloc(16)
        else:
            nbytes = int(text)
        rows = C.c_int64(0)
        try:
            self._ck(self.lib.adb_csv_index(d_text.void(), nbytes, skip_lines, C.byref(rows)))
            cols = [self.alloc_i32(rows.value) for _ in range(n_cols)]
            ptrs = (C.c_void_p * n_cols)(*[c.ptr for c in cols])
            try:
                self._ck(self.lib.adb_csv_parse(n_cols, ptrs))
            except EngineError:
                for c in cols:
                    c.free()
                raise
        finally:
            if own:
                self.sync()
                d_text.free()
        return cols, int(rows.value)

    def format_i32(self, val: DevBuf, n: int) -> bytes:
        """print's text for an INT result ("%d" joined by newlines, query.c:262-269), formatted
        on the device and downloaded as text."""
        nb = C.c_int64(0)
        self._ck(self.lib.adb_format_i32_count(val.i32(), n, C.byref(nb)))
        if nb.value == 0:
            self._ck(self.lib.adb_format_i32_emit(None))
            return b""
        d = self.alloc(nb.value)
        self._ck(self.lib.adb_format_i32_emit(d.void()))
        out = d.to_host(nb.value, np.uint8).tobytes()
        d.free()
        return out

    def sync(self):
        self._ck(self.lib.adb_sync())

    def timer_start(self):
        self._ck(self.lib.adb_timer_start())

    def timer_stop(self) -> float:
        ms = C.c_float(0)
        self._ck(self.lib.adb_timer_stop(C.byref(ms)))
        return float(ms.value)

    def mark(self, slot: int):
        self._ck(self.lib.adb_mark(slot))

    def mark_elapsed(self, a: int, b: int) -> float:
        ms = C.c_float(0)
        self._ck(self.lib.adb_mark_elapsed(a, b, C.byref(ms)))
        return float(ms.value)

    def launch_count(self) -> int:
        return int(self.lib.adb_launch_count())

    def set_stream(self, cuda_stream_ptr: int):
        self._ck(self.lib.adb_set_stream(C.c_void_p(cuda_stream_ptr)))

    # ---- operators (thin: arguments in, device buffers out) -------------------------------
    def select_scan(self, col: DevBuf, n: int, lo=None, hi=None, base: int = 0,
                    out: DevBuf | None = None, d_count: DevBuf | None = None, sync: bool = True,
                    col_offset: int = 0):
        """select_column_scan (query.c:92).  Returns (pos DevBuf, d_count DevBuf, count|None)."""
        out = out or self.alloc_i32(n)
        d_count = d_count or self.alloc(8)
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_scan(col.i32(col_offset), n, plo, phi, base, out.i32(),
                                          d_count.i64(), C.byref(h) if sync else None))
        return out, d_count, (int(h.value) if sync else None)

    def select_pairs(self, val: DevBuf, pos: DevBuf, n_max: int, lo=None, hi=None,
                     d_n: DevBuf | None = None, sync: bool = True):
        """select_result (query.c:38)."""
        out, d_count = self.alloc_i32(n_max), self.alloc(8)
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_count(val.i32(), n_max, d_n.i64() if d_n else None, plo, phi,
                                           d_count.i64(), C.byref(h) if sync else None))
        self._ck(self.lib.adb_select_emit(pos.i32(), 0, out.i32()))
        return out, d_count, (int(h.value) if sync else None)

    def select_exact(self, val: DevBuf, n: int, lo=None, hi=None, pos_in: DevBuf | None = None,
                     base: int = 0, d_n: DevBuf | None = None):
        """Two-phase select (count, then emit into an exactly sized list): (pos DevBuf, count)."""
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_count(val.i32(), n, d_n.i64() if d_n else None, plo, phi,
                                           None, C.byref(h)))
        out = self.alloc_i32(h.value)
        self._ck(self.lib.adb_select_emit(pos_in.i32() if pos_in else None, base, out.i32()))
        return out, int(h.value)

    def select_fetch_agg_deferred(self, sel_col: DevBuf, fetch_col: DevBuf, n: int, lo=None, hi=None):
        """adb_select_count, host reads the count, then positions + gather + aggregates in one
        kernel (adb_select_emit_fetch_agg): (pos DevBuf, val DevBuf, count, Agg)."""
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_count(sel_col.i32(), n, None, plo, phi, None, C.byref(h)))
        gen = int(self.lib.adb_select_generation())
        pos, val = self.alloc_i32(h.value), self.alloc_i32(h.value)
        d_out = self.alloc(C.sizeof(_AggStruct))
        a = _AggStruct()
        assert int(self.lib.adb_select_generation()) == gen
        self._ck(self.lib.adb_select_emit_fetch_agg(fetch_col.i32(), pos.i32(), val.i32(),
                                                    C.cast(d_out.void(), C.POINTER(_AggStruct)), C.byref(a)))
        d_out.free()
        return pos, val, int(h.value), Agg(a.sum, a.count, a.min, a.max)

    def fetch(self, col: DevBuf, pos: DevBuf, n_max: int, d_n: DevBuf | None = None, base: int = 0,
              out: DevBuf | None = None) -> DevBuf:
        """fetch_column (query.c:223)."""
        out = out or self.alloc_i32(n_max)
        self._ck(self.lib.adb_fetch(col.i32(), pos.i32(), n_max, d_n.i64() if d_n else None, base,
                                    out.i32()))
        return out

    def aggregate(self, val: DevBuf, n_max: int, d_n: DevBuf | None = None, offset: int = 0) -> Agg:
        """sum / average / min / max partials in one pass (query.c:306-437)."""
        d_out = self.alloc(C.sizeof(_AggStruct))
        h = _AggStruct()
        self._ck(self.lib.adb_aggregate(val.i32(offset), n_max, d_n.i64() if d_n else None,
                                        C.cast(d_out.void(), C.POINTER(_AggStruct)), C.byref(h)))
        d_out.free()
        return Agg(h.sum, h.count, h.min, h.max)

    def ewise(self, a: DevBuf, b: DevBuf, n_max: int, subtract: bool, d_n: DevBuf | None = None) -> DevBuf:
        """add / sub (query.c:356,374)."""
        out = self.alloc_i32(n_max)
        fn = self.lib.adb_sub if subtract else self.lib.adb_add
        self._ck(fn(a.i32(), b.i32(), n_max, d_n.i64() if d_n else None, out.i32()))
        return out

    def shared_select(self, col: DevBuf, n: int, lows, highs):
        """shared_select (query.c:496): count phase, exact-size outputs, emit phase.
        Returns a list of (pos DevBuf, count) per query."""
        lows = np.ascontiguousarray(lows, dtype=np.int32)
        highs = np.ascontiguousarray(highs, dtype=np.int32)
        q = lows.size
        counts = (C.c_int64 * q)()
        self._ck(self.lib.adb_shared_select_count(col.i32(), n, lows.ctypes.data_as(_I32P),
                                                  highs.ctypes.data_as(_I32P), q, counts))
        outs = [self.alloc_i32(counts[i]) for i in range(q)]
        ptrs = (C.c_void_p * q)(*[o.ptr for o in outs])
        cap = max(list(counts) + [1])
        self._ck(self.lib.adb_shared_select_emit(ptrs, cap))
        return [(outs[i], int(counts[i])) for i in range(q)]

    def index_sort(self, col: DevBuf, n: int):
        """build_unclustered_index's sort (index.c:140): (values DevBuf, positions DevBuf)."""
        values, positions = self.alloc_i32(n), self.alloc_i32(n)
        self._ck(self.lib.adb_index_sort(col.i32(), n, values.i32(), positions.i32()))
        return values, positions

    def index_sort_ref_ties(self, col: DevBuf, n: int):
        """index_sort with the reference quicksort's order of equal keys (index.c:25-46)."""
        values, positions = self.alloc_i32(n), self.alloc_i32(n)
        self._ck(self.lib.adb_index_sort_ref_ties(col.i32(), n, values.i32(), positions.i32()))
        return values, positions

    def rank_hist(self, col: DevBuf, n: int, prefixes, rnd: int) -> np.ndarray:
        """One multi-target radix-select round: a (len(prefixes), 256) uint32 histogram."""
        pre = np.ascontiguousarray(prefixes, dtype=np.uint32)
        hist = np.zeros((pre.size, 256), dtype=np.uint32)
        self._ck(self.lib.adb_rank_hist(col.i32(), n, pre.ctypes.data_as(C.POINTER(C.c_uint32)), pre.size, rnd,
                                        hist.ctypes.data_as(C.POINTER(C.c_uint32))))
        return hist

    def route_range(self, keys: DevBuf, n: int, row_base: int, splitters, parts: int):
        """Stable partition by index slice: (keys DevBuf, rows DevBuf, counts per slice)."""
        split = np.ascontiguousarray(splitters, dtype=np.int32)
        counts = (C.c_int64 * max(parts, 1))()
        keys_out, rows_out = self.alloc_i32(n), self.alloc_i32(n)
        self._ck(self.lib.adb_route_range(keys.i32(), n, row_base, split.ctypes.data_as(_I32P), parts,
                                          keys_out.i32(), rows_out.i32(), counts))
        return keys_out, rows_out, [int(counts[i]) for i in range(parts)]

    def index_sort_pairs(self, keys: DevBuf, payload: DevBuf, n: int):
        """index_sort carrying the given payload: (values DevBuf, payload DevBuf)."""
        values, pay = self.alloc_i32(n), self.alloc_i32(n)
        self._ck(self.lib.adb_index_sort_pairs(keys.i32(), payload.i32(), n, values.i32(), pay.i32()))
        return values, pay

    def join(self, v1: DevBuf, p1: DevBuf, n1: int, v2: DevBuf, p2: DevBuf, n2: int,
             nested_loop: bool = False):
        """hash_join / nested_loop_join (query.c:652,585): (out1 DevBuf, out2 DevBuf, pairs)."""
        m = C.c_int64(-1)
        fn = self.lib.adb_nested_loop_join_count if nested_loop else self.lib.adb_hash_join_count
        self._ck(fn(v1.i32(), p1.i32(), n1, v2.i32(), p2.i32(), n2, C.byref(m)))
        o1, o2 = self.alloc_i32(m.value), self.alloc_i32(m.value)
        self._ck(self.lib.adb_join_emit(o1.i32(), o2.i32()))
        return o1, o2, int(m.value)

    def index_create(self, values: DevBuf, positions: DevBuf, n: int, with_btree: bool = True):
        """Wrap device-resident (sorted values, int32 positions) as an index handle."""
        h = C.c_void_p()
        self._ck(self.lib.adb_index_create(values.i32(), positions.i32(), n, int(with_btree), C.byref(h)))
        return h

    def index_destroy(self, handle):
        self._ck(self.lib.adb_index_destroy(handle))

    def select_index(self, handle, n: int, lo=None, hi=None, use_btree: bool = False):
        """select_column_sorted_index (query.c:165).  Returns (pos DevBuf, count)."""
        out, d_count = self.alloc_i32(n), self.alloc(8)
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_index_count(handle, int(use_btree), plo, phi, d_count.i64(), C.byref(h)))
        self._ck(self.lib.adb_select_index_emit(handle, out.i32()))
        d_count.free()
        return out, int(h.value)

    def select_index_exact(self, handle, lo=None, hi=None, use_btree: bool = False):
        """Two-phase index select: (pos DevBuf, count)."""
        (plo, _a), (phi, _b) = _bound(lo), _bound(hi)
        h = C.c_int64(-1)
        self._ck(self.lib.adb_select_index_count(handle, int(use_btree), plo, phi, None, C.byref(h)))
        out = self.alloc_i32(h.value)
        self._ck(self.lib.adb_select_index_emit(handle, out.i32()))
        return out, int(h.value)

    def synth_uniform(self, n: int, seed: int, first_row: int = 0, lo: int = 0,
                      span: int = 1 << 31, out: DevBuf | None = None, out_offset: int = 0) -> DevBuf:
        out = out or self.alloc_i32(n)
        self._ck(self.lib.adb_synth_uniform(out.i32(out_offset), n, seed, first_row, lo, span))
        return out

    def agg_ptr(self, buf: DevBuf, index: int = 0):
        return C.cast(buf.void(index * C.sizeof(_AggStruct)), C.POINTER(_AggStruct))

    def read_agg(self, buf: DevBuf, index: int = 0) -> Agg:
        raw = buf.to_host(C.sizeof(_AggStruct), np.uint8, index * C.sizeof(_AggStruct))
        h = _AggStruct.from_buffer_copy(raw.tobytes())
        return Agg(h.sum, h.count, h.min, h.max)


AGG_BYTES = C.sizeof(_AggStruct)
