"""ReplayEngine: one sgr_engine handle behind a small Python surface.

Host arrays (numpy) go through the host-buffer entry points (H2D/D2H inside the call, what a
JNI caller with direct ByteBuffers would use); CUDA tensors go through the `_device`
entry points and are borrowed, not copied.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import native as N


def _is_cuda_tensor(x) -> bool:
    return hasattr(x, "is_cuda") and bool(getattr(x, "is_cuda"))


def _producer_done(*tensors) -> None:
    """The engine launches on its own non-blocking stream: a tensor torch is still writing on ITS current stream must be complete
    before the engine borrows it (the `_device` entry points take plain pointers, they cannot order against torch's stream)."""
    import torch

    for t in tensors:
        if _is_cuda_tensor(t):
            torch.cuda.current_stream(t.device).synchronize()
            return


class _DevView:
    """Exposes a raw device pointer through __cuda_array_interface__ (for torch.as_tensor)."""

    def __init__(self, ptr: int, nbytes: int, owner):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        self._owner = owner


class ReplayEngine:
    def __init__(self, device: int = 0):
        self._lib = N.load_library()
        self._h = C.c_void_p()
        cfg = N.sgr_config()
        cfg.device = device
        rc = self._lib.sgr_create(C.byref(cfg), C.byref(self._h))
        if rc != N.SGR_OK:
            self._h = C.c_void_p()
            N.check(self._lib, None, rc)
        self.device = device
        self.state_bytes = 0
        self._keep = []  # borrowed device tensors kept alive

    # -- lifecycle
    def close(self) -> None:
        if self._h:
            self._lib.sgr_destroy(self._h)
            self._h = C.c_void_p()
            self._keep = []

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc: int) -> None:
        N.check(self._lib, self._h, rc)

    # -- program
    def register_program(self, prog: N.sgr_fold_program) -> None:
        self._ck(self._lib.sgr_register_program(self._h, C.byref(prog)))
        self.state_bytes = int(prog.state_bytes)

    # -- loads
    def load_events(self, events, seg_offsets) -> None:
        """CSR event log. numpy -> copied to HBM; CUDA tensors -> borrowed."""
        if _is_cuda_tensor(events):
            assert _is_cuda_tensor(seg_offsets)
            ev = events.contiguous().view(-1)
            nbytes = ev.numel() * ev.element_size()
            n_agg = seg_offsets.numel() - 1
            _producer_done(ev)
            self._keep = [ev, seg_offsets]
            self._ck(self._lib.sgr_load_events_device(self._h, ev.data_ptr(), nbytes, seg_offsets.data_ptr(), n_agg))
            return
        ev = np.ascontiguousarray(events).view(np.uint8).reshape(-1)
        off = np.ascontiguousarray(seg_offsets, dtype=np.uint64)
        self._ck(self._lib.sgr_load_events(self._h, ev.ctypes.data, ev.size, off.ctypes.data, len(off) - 1))

    def load_events_indexed(self, events, seg_offsets, rec_offsets) -> None:
        """Variable records + record directory (rec_offsets[n_records+1]): enables the record-parallel kernel."""
        if _is_cuda_tensor(events):
            ev = events.contiguous().view(-1)
            _producer_done(ev)
            self._keep = [ev, seg_offsets, rec_offsets]
            self._ck(self._lib.sgr_load_events_indexed_device(self._h, ev.data_ptr(), ev.numel() * ev.element_size(), seg_offsets.data_ptr(),
                                                              seg_offsets.numel() - 1, rec_offsets.data_ptr(), rec_offsets.numel() - 1))
            return
        ev = np.ascontiguousarray(events).view(np.uint8).reshape(-1)
        off = np.ascontiguousarray(seg_offsets, dtype=np.uint64)
        ro = np.ascontiguousarray(rec_offsets, dtype=np.uint64)
        self._ck(self._lib.sgr_load_events_indexed(self._h, ev.ctypes.data, ev.size, off.ctypes.data, len(off) - 1, ro.ctypes.data, len(ro) - 1))

    def load_unsorted(self, records, n_agg: int) -> None:
        """Fixed 64-byte records in arrival order; grouped stably by aggregate on the device."""
        if _is_cuda_tensor(records):
            r = records.contiguous().view(-1)
            n = r.numel() * r.element_size() // 64
            _producer_done(r)
            self._keep = [r]
            self._ck(self._lib.sgr_load_unsorted_device(self._h, r.data_ptr(), n, n_agg))
            return
        r = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
        self._ck(self._lib.sgr_load_unsorted(self._h, r.ctypes.data, r.size // 64, n_agg))

    def fold_unsorted(self, records, n_agg: int) -> None:
        """Rebuild all states from an arrival-order log (Kafka partition order) in one call."""
        if _is_cuda_tensor(records):
            r = records.contiguous().view(-1)
            _producer_done(r)
            self._keep = [r]
            self._ck(self._lib.sgr_fold_unsorted_device(self._h, r.data_ptr(), r.numel() * r.element_size() // 64, n_agg))
            return
        r = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
        self._ck(self._lib.sgr_fold_unsorted(self._h, r.ctypes.data, r.size // 64, n_agg))

    def set_initial_states(self, states: Optional[np.ndarray]) -> None:
        if states is None:
            self._ck(self._lib.sgr_set_initial_states(self._h, None, 0))
            return
        s = np.ascontiguousarray(states).view(np.uint8).reshape(-1, self.state_bytes)
        self._ck(self._lib.sgr_set_initial_states(self._h, s.ctypes.data, s.shape[0]))

    # -- compute
    def fold(self) -> None:
        self._ck(self._lib.sgr_fold(self._h))

    def fold_async(self) -> None:
        """Enqueue the fold on the engine's stream without waiting (pair with wait())."""
        self._ck(self._lib.sgr_fold_async(self._h))

    def wait(self) -> None:
        self._ck(self._lib.sgr_wait(self._h))

    def fold_incremental(self, records) -> None:
        if _is_cuda_tensor(records):
            r = records.contiguous().view(-1)
            _producer_done(r)
            self._keep.append(r)
            self._ck(self._lib.sgr_fold_incremental_device(self._h, r.data_ptr(), r.numel() * r.element_size() // 64))
            self._keep.pop()
            return
        r = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
        self._ck(self._lib.sgr_fold_incremental(self._h, r.ctypes.data, r.size // 64))

    def grow_states(self, n_agg: int) -> None:
        """Resize the live table on the device, keeping its content (new slots are None)."""
        self._ck(self._lib.sgr_grow_states(self._h, n_agg))

    def fold_ingested(self, ingest) -> None:
        """Fold everything pending in an Ingest onto the live table and publish its id dictionary to get()."""
        self._ck(self._lib.sgr_fold_ingested(self._h, ingest.handle))

    # -- results
    def n_aggregates(self) -> int:
        p, n, sb = C.c_void_p(), C.c_uint64(), C.c_uint32()
        self._ck(self._lib.sgr_states_device(self._h, C.byref(p), C.byref(n), C.byref(sb)))
        return int(n.value)

    def export_states(self, out: Optional[np.ndarray] = None, bitmaps: bool = False):
        n = self.n_aggregates()
        if out is None:
            out = np.empty((n, self.state_bytes), dtype=np.uint8)
        if not bitmaps:
            self._ck(self._lib.sgr_export_states(self._h, out.ctypes.data, out.nbytes, None, None, None))
            return out
        nb = (n + 7) // 8
        ex, ch, er = (np.zeros(nb, dtype=np.uint8) for _ in range(3))
        self._ck(self._lib.sgr_export_states(self._h, out.ctypes.data, out.nbytes, ex.ctypes.data, ch.ctypes.data, er.ctypes.data))
        return out, ex, ch, er

    def states_tensor(self):
        """The live device state table as a torch uint8 tensor [n_agg, state_bytes] (borrowed)."""
        import torch

        p, n, sb = C.c_void_p(), C.c_uint64(), C.c_uint32()
        self._ck(self._lib.sgr_states_device(self._h, C.byref(p), C.byref(n), C.byref(sb)))
        view = _DevView(p.value, n.value * sb.value, self)
        return torch.as_tensor(view, device=f"cuda:{self.device}").view(n.value, sb.value)

    def events_tensors(self):
        """(events u8[nbytes], seg_offsets i64[n_agg+1]) device tensors of the engine's CSR log (borrowed)."""
        import torch

        p, nb, po = C.c_void_p(), C.c_uint64(), C.c_void_p()
        self._ck(self._lib.sgr_events_device(self._h, C.byref(p), C.byref(nb), C.byref(po)))
        ev = torch.as_tensor(_DevView(p.value, nb.value, self), device=f"cuda:{self.device}")
        return ev, po.value

    def load_keys(self, keys: Sequence[str]) -> None:
        enc = [k.encode("utf-8") for k in keys]
        offs = np.zeros(len(enc) + 1, dtype=np.uint32)
        np.cumsum([len(b) for b in enc], out=offs[1:])
        blob = np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8).copy()
        self._ck(self._lib.sgr_load_keys(self._h, blob.ctypes.data, offs.ctypes.data, len(enc)))

    def get(self, key: str) -> Optional[bytes]:
        """getAggregateBytes(aggregateId): Option[Array[Byte]] — None when the state does not exist."""
        kb = key.encode("utf-8")
        buf = C.create_string_buffer(N.MAX_STATE_BYTES)
        outlen, exists = C.c_uint32(), C.c_int32()
        kbuf = C.create_string_buffer(kb, len(kb)) if kb else None
        self._ck(self._lib.sgr_get(self._h, C.cast(kbuf, C.c_void_p) if kbuf else None, len(kb), buf, N.MAX_STATE_BYTES,
                                   C.byref(outlen), C.byref(exists)))
        return bytes(buf.raw[:outlen.value]) if exists.value else None

    def index_of(self, key: str) -> Optional[int]:
        """Dense aggregate index `get(key)` reads, or None for an unknown id."""
        kb = key.encode("utf-8")
        kbuf = C.create_string_buffer(kb, len(kb)) if kb else None
        agg = C.c_uint64()
        self._ck(self._lib.sgr_key_index(self._h, C.cast(kbuf, C.c_void_p) if kbuf else None, len(kb), C.byref(agg)))
        return None if agg.value == (1 << 64) - 1 else int(agg.value)

    def get_index(self, agg: int) -> Tuple[Optional[bytes], int, int]:
        """(program bytes or None, flags, err_idx) of one dense aggregate index."""
        buf = C.create_string_buffer(N.MAX_STATE_BYTES)
        outlen, exists, flags, err = C.c_uint32(), C.c_int32(), C.c_uint32(), C.c_uint32()
        self._ck(self._lib.sgr_get_index(self._h, agg, buf, N.MAX_STATE_BYTES, C.byref(outlen), C.byref(exists),
                                         C.byref(flags), C.byref(err)))
        return (bytes(buf.raw[:outlen.value]) if exists.value else None), int(flags.value), int(err.value)

    # -- multi-GPU (one process per GPU)
    def dist_init(self, rank: int, nranks: int, unique_id: Optional[bytes], recv_capacity_records: int) -> None:
        buf = C.create_string_buffer(unique_id, 128) if unique_id else None
        self._ck(self._lib.sgr_dist_init(self._h, rank, nranks, buf, recv_capacity_records))

    def dist_set_partitions(self, partition_of_agg: np.ndarray) -> None:
        p = np.ascontiguousarray(partition_of_agg, dtype=np.uint32)
        self._ck(self._lib.sgr_dist_set_partitions(self._h, p.ctypes.data, len(p)))

    def dist_ipc_export(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self._lib.sgr_dist_ipc_export(self._h, buf))
        return bytes(buf.raw)

    def dist_ipc_import(self, handles: Sequence[bytes]) -> None:
        blob = C.create_string_buffer(b"".join(handles), 64 * len(handles))
        self._ck(self._lib.sgr_dist_ipc_import(self._h, blob))

    def dist_route_and_fold(self, records, fused) -> None:
        """records: CUDA tensor of fixed 64-byte records in arrival order carrying GLOBAL aggregate indices.
        fused: 0 NCCL all-to-all, 1 peer scatter, 2 pipelined push + fold, 3 the same with projected records (see sgr.h)."""
        r = records.contiguous().view(-1)
        _producer_done(r)
        self._keep = [r]
        self._ck(self._lib.sgr_dist_route_and_fold(self._h, r.data_ptr(), r.numel() * r.element_size() // 64, int(fused)))

    def dist_recv_base(self) -> int:
        p = C.c_void_p()
        self._ck(self._lib.sgr_dist_recv_base(self._h, C.byref(p)))
        return int(p.value or 0)

    def dist_set_peers(self, bases: Sequence[int]) -> None:
        """Loopback ranks (one process, one device): the other ranks' receive allocations as raw device pointers."""
        arr = (C.c_void_p * len(bases))(*[C.c_void_p(b) for b in bases])
        self._ck(self._lib.sgr_dist_set_peers(self._h, arr))

    def dist_reserve(self, max_records: int) -> None:
        """Allocate everything the pipelined push needs up front (required for loopback ranks, see sgr.h)."""
        self._ck(self._lib.sgr_dist_reserve(self._h, int(max_records)))

    def states_hash(self) -> int:
        """Order-independent 64-bit hash of the live table (global aggregate indices on a routed engine)."""
        h = C.c_uint64()
        self._ck(self._lib.sgr_states_hash(self._h, C.byref(h)))
        return int(h.value)

    def dist_stats(self) -> N.sgr_dist_stats:
        s = N.sgr_dist_stats()
        self._ck(self._lib.sgr_dist_get_stats(self._h, C.byref(s)))
        return s

    def dist_local_aggregates(self) -> np.ndarray:
        n = C.c_uint64()
        self._ck(self._lib.sgr_dist_local_aggregates(self._h, None, 0, C.byref(n)))
        out = np.zeros(int(n.value), dtype=np.uint32)
        self._ck(self._lib.sgr_dist_local_aggregates(self._h, out.ctypes.data, len(out), C.byref(n)))
        return out

    def stats(self) -> N.sgr_stats:
        s = N.sgr_stats()
        self._ck(self._lib.sgr_get_stats(self._h, C.byref(s)))
        return s

    def set_option(self, name: str, value: int) -> None:
        self._ck(self._lib.sgr_set_option(self._h, name.encode(), int(value)))

    def stream_ptr(self) -> int:
        p = C.c_void_p()
        self._ck(self._lib.sgr_stream(self._h, C.byref(p)))
        return int(p.value or 0)
