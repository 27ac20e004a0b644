"""ctypes binding of ``liblwse.so`` (the C ABI of ``include/lwse.h``).

This is the only way Python reaches the engine, and it is the same set of
symbols a cgo shim binds (INTEGRATION.md).  There is no fallback: if the
library is missing or no sm_100 device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import records as R

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "liblwse.so")
_lib = None

# every symbol include/lwse.h declares: name → (argtypes, restype)
SYMBOLS = {
    "lwse_create": ([C.POINTER(R.Config), C.POINTER(C.c_void_p)], C.c_int),
    "lwse_destroy": ([C.c_void_p], None),
    "lwse_strerror": ([C.c_int], C.c_char_p),
    "lwse_last_cuda_error": ([C.c_void_p], C.c_int),
    "lwse_abi_version": ([], C.c_uint32),
    "lwse_stream": ([C.c_void_p], C.c_void_p),
    "lwse_launch_count": ([C.c_void_p], C.c_uint64),
    "lwse_graph_tick_count": ([C.c_void_p], C.c_uint64),
    "lwse_shard_of": ([C.c_uint64, C.c_uint32], C.c_uint32),
    "lwse_hash64": ([C.c_void_p, C.c_size_t], C.c_uint64),
    "lwse_upload_nodes": ([C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32], C.c_int),
    "lwse_sweep_lws_host": ([C.c_void_p, C.POINTER(R.LwsTables)], C.c_int),
    "lwse_sweep_lws_device": ([C.c_void_p, C.POINTER(R.LwsTables), C.c_void_p], C.c_int),
    "lwse_resident_load": ([C.c_void_p, C.POINTER(R.LwsTables)], C.c_int),
    "lwse_resident_patch": ([C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint32], C.c_int),
    "lwse_resident_sweep": ([C.c_void_p, C.c_uint32, C.POINTER(R.Changes)], C.c_int),
    "lwse_resident_outputs": ([C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "lwse_resident_arena": ([C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)], C.c_int),
    "lwse_resident_place_load": ([C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32], C.c_int),
    "lwse_resident_tick": ([C.c_void_p, C.POINTER(R.Tick)], C.c_int),
    "lwse_resident_tick_submit": ([C.c_void_p, C.POINTER(R.Tick)], C.c_int),
    "lwse_resident_tick_wait": ([C.c_void_p, C.POINTER(R.Tick)], C.c_int),
    "lwse_resident_place_outputs": ([C.c_void_p, C.c_void_p], C.c_int),
    "lwse_resident_occupancy": ([C.c_void_p, C.c_void_p], C.c_int),
    "lwse_place_host": (
        [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32)],
        C.c_int,
    ),
    "lwse_place_device": (
        [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p],
        C.c_int,
    ),
    "lwse_place_grouped_device": (
        [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
         C.POINTER(C.c_uint32), C.c_void_p],
        C.c_int,
    ),
    "lwse_place_gathered_device": (
        [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p,
         C.POINTER(C.c_uint32), C.c_void_p],
        C.c_int,
    ),
    "lwse_reconcile_device": (
        [C.c_void_p, C.POINTER(R.LwsTables), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p],
        C.c_int,
    ),
    "lwse_reconcile_host": (
        [C.c_void_p, C.POINTER(R.LwsTables), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p],
        C.c_int,
    ),
    "lwse_exchange_create": ([C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p], C.c_int),
    "lwse_exchange_connect": ([C.c_void_p, C.c_void_p], C.c_int),
    "lwse_exchange_part_bytes": ([C.c_void_p], C.c_uint64),
    "lwse_reconcile_exchanged_device": (
        [C.c_void_p, C.POINTER(R.LwsTables), C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p],
        C.c_int,
    ),
    "lwse_reconcile_shared_device": (
        [C.c_void_p, C.POINTER(R.LwsTables), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p],
        C.c_int,
    ),
    "lwse_exchange_status": ([C.c_void_p, C.POINTER(C.c_uint32)], C.c_int),
    "lwse_sweep_ds_host": ([C.c_void_p, C.POINTER(R.DsTables)], C.c_int),
    "lwse_sweep_ds_device": ([C.c_void_p, C.POINTER(R.DsTables), C.c_void_p], C.c_int),
    "lwse_ds_resident_load": ([C.c_void_p, C.POINTER(R.DsTables)], C.c_int),
    "lwse_ds_resident_tick": ([C.c_void_p, C.POINTER(R.DsTick)], C.c_int),
    "lwse_ds_resident_outputs": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "lwse_joint_tick": ([C.c_void_p, C.POINTER(R.Tick), C.POINTER(R.DsTick)], C.c_int),
    "lwse_joint_tick_submit": ([C.c_void_p, C.POINTER(R.Tick), C.POINTER(R.DsTick)], C.c_int),
    "lwse_joint_tick_wait": ([C.c_void_p, C.POINTER(R.Tick), C.POINTER(R.DsTick)], C.c_int),
    "lwse_group_keys_host": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p], C.c_int),
    "lwse_subgroup_keys_host": (
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "lwse_subgroup_keys_device": (
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
         C.c_void_p], C.c_int),
    "lwse_group_keys_device": (
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p],
        C.c_int,
    ),
}


class LwseError(RuntimeError):
    def __init__(self, status: int, cuda_error: int = 0):
        self.status, self.cuda_error = status, cuda_error
        msg = lib().lwse_strerror(status).decode()
        if cuda_error:
            msg += f" [cudaError {cuda_error}]"
        super().__init__(f"lwse: {msg} ({status})")


def lib_path() -> str:
    return _LIB_PATH


def lib() -> C.CDLL:
    """Load liblwse.so; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise FileNotFoundError(
                f"{_LIB_PATH} is missing: build it with `python -m lws_b200.build` "
                "(the engine has no CPU fallback)"
            )
        _lib = C.CDLL(_LIB_PATH)
        for name, (args, res) in SYMBOLS.items():
            fn = getattr(_lib, name)  # AttributeError = ABI drift, fail loudly
            fn.argtypes, fn.restype = args, res
    return _lib


def shard_of(uid_hash: int, n_shards: int) -> int:
    return lib().lwse_shard_of(uid_hash, n_shards)


class Engine:
    """One engine per GPU (``lwse_create``)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        cfg = R.Config(R.ABI_VERSION, device, 0, 0)
        rc = lib().lwse_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise LwseError(rc)
        self.device = device
        self.n_nodes = 0
        self.n_domains = 0

    def close(self):
        if self._h:
            lib().lwse_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise LwseError(rc, lib().lwse_last_cuda_error(self._h))

    @property
    def stream(self) -> int:
        return lib().lwse_stream(self._h) or 0

    @property
    def launch_count(self) -> int:
        return lib().lwse_launch_count(self._h)

    @property
    def graph_tick_count(self) -> int:
        """Resident ticks replayed as one CUDA graph since creation."""
        return lib().lwse_graph_tick_count(self._h)

    # ------------------------------------------------------------------ nodes
    def upload_nodes(self, nodes: np.ndarray, n_domains: int):
        assert nodes.dtype == R.NODE_REC
        self._check(lib().lwse_upload_nodes(self._h, R.ptr(nodes) if len(nodes) else None, len(nodes), n_domains))
        self.n_nodes, self.n_domains = len(nodes), n_domains

    # -------------------------------------------------------------- LWS sweep
    def sweep_lws_host(self, lws, groups, pod_state, pod_ident, flags=0, want_occupancy=False, out=None):
        """Host tables in → (lws_out, group_out, occupancy|None) host tables out."""
        assert lws.dtype == R.LWS_REC and groups.dtype == R.GROUP_REC
        assert pod_state.dtype == R.POD_STATE and pod_ident.dtype == R.POD_IDENT and len(pod_state) == len(pod_ident)
        if out is None:
            lws_out = R.aligned_empty(len(lws), R.LWS_OUT)
            group_out = R.aligned_empty(len(groups), R.GROUP_OUT)
        else:
            lws_out, group_out = out
        occ = np.zeros(max(self.n_nodes, 1), dtype=np.uint32) if want_occupancy else None
        t = R.LwsTables(
            R.ptr(lws), len(lws), R.ptr(groups), len(groups), R.ptr(pod_state), R.ptr(pod_ident), len(pod_state),
            R.ptr(lws_out), R.ptr(group_out), R.ptr(occ), flags,
        )
        self._check(lib().lwse_sweep_lws_host(self._h, C.byref(t)))
        return lws_out, group_out, (occ[: self.n_nodes] if occ is not None else None)

    def reconcile_host(self, lws, groups, pod_state, pod_ident, reqs, occupancy=None, n_namespaces=1, flags=0,
                       out=None, place_out=None):
        """Host tables + placement requests in → (lws_out, group_out, place_out): one tick, one call."""
        assert lws.dtype == R.LWS_REC and groups.dtype == R.GROUP_REC and reqs.dtype == R.PLACE_REQ
        assert pod_state.dtype == R.POD_STATE and pod_ident.dtype == R.POD_IDENT and len(pod_state) == len(pod_ident)
        lws_out, group_out = out if out is not None else (R.aligned_empty(len(lws), R.LWS_OUT),
                                                          R.aligned_empty(len(groups), R.GROUP_OUT))
        if place_out is None:
            place_out = R.aligned_empty(len(reqs), R.PLACE_OUT)
        if occupancy is not None:
            occupancy = np.ascontiguousarray(occupancy, dtype=np.uint32)
        t = R.LwsTables(
            R.ptr(lws), len(lws), R.ptr(groups), len(groups), R.ptr(pod_state), R.ptr(pod_ident), len(pod_state),
            R.ptr(lws_out), R.ptr(group_out), None, flags,
        )
        self._check(lib().lwse_reconcile_host(self._h, C.byref(t), R.ptr(reqs) if len(reqs) else None, len(reqs),
                                              R.ptr(occupancy), n_namespaces, R.ptr(place_out) if len(reqs) else None))
        return lws_out, group_out, place_out

    def sweep_lws_device(self, d_lws, n_lws, d_groups, n_groups, d_pod_state, d_pod_ident, n_pods, d_lws_out,
                         d_group_out, d_occupancy=None, flags=0, stream=None):
        """Device pointers (ints / tensors) in; kernels are enqueued, no synchronize."""
        t = R.LwsTables(
            R.ptr(d_lws), n_lws, R.ptr(d_groups), n_groups, R.ptr(d_pod_state), R.ptr(d_pod_ident), n_pods,
            R.ptr(d_lws_out), R.ptr(d_group_out), R.ptr(d_occupancy), flags,
        )
        self._check(lib().lwse_sweep_lws_device(self._h, C.byref(t), stream))

    @staticmethod
    def device_tables(d_lws, n_lws, d_groups, n_groups, d_pod_state, d_pod_ident, n_pods, d_lws_out, d_group_out,
                      d_occupancy=None, flags=0):
        """The ``lwse_lws_tables`` descriptor of device-resident tables (build once, reuse every tick)."""
        return R.LwsTables(
            R.ptr(d_lws), n_lws, R.ptr(d_groups), n_groups, R.ptr(d_pod_state), R.ptr(d_pod_ident), n_pods,
            R.ptr(d_lws_out), R.ptr(d_group_out), R.ptr(d_occupancy), flags,
        )

    def reconcile_device(self, tables, d_reqs, n_reqs, d_occupancy, n_namespaces, d_place_out, stream=None):
        """One reconcile tick: sweep on ``stream``, placement round concurrently on the engine's
        side stream, joined back into ``stream``.  Enqueue only, no synchronize."""
        self._check(lib().lwse_reconcile_device(self._h, C.byref(tables), R.ptr(d_reqs), n_reqs, R.ptr(d_occupancy),
                                                n_namespaces, R.ptr(d_place_out), stream))

    # --------------------------------------------------------- peer exchange
    def exchange_create(self, reqs_per_part: int, world: int, rank: int) -> bytes:
        """Allocate this rank's exchange buffer → its 64-byte IPC handle (all-gather these)."""
        h = (C.c_uint8 * 64)()
        self._check(lib().lwse_exchange_create(self._h, reqs_per_part, world, rank, h))
        return bytes(h)

    def exchange_connect(self, handles: bytes):
        """``handles``: every rank's handle, concatenated in rank order."""
        buf = (C.c_uint8 * len(handles)).from_buffer_copy(handles)
        self._check(lib().lwse_exchange_connect(self._h, buf))

    @property
    def exchange_part_bytes(self) -> int:
        return int(lib().lwse_exchange_part_bytes(self._h))

    def reconcile_exchanged_device(self, tables, d_local_part, n_namespaces, d_place_out, stream=None):
        """One tick of a shard: push this rank's [occupancy | requests] part to every peer over
        NVLink, wait for theirs, placement round over all parts — on the side stream, concurrently
        with the sweep of ``tables`` (None: placement step only).  Enqueue only."""
        self._check(lib().lwse_reconcile_exchanged_device(
            self._h, C.byref(tables) if tables is not None else None, R.ptr(d_local_part), n_namespaces,
            R.ptr(d_place_out), stream))

    def reconcile_shared_device(self, tables, d_reqs, n_reqs, d_local_occupancy, n_namespaces, d_place_out, flags=0, stream=None):
        """One tick of a shard with LOCAL requests and SHARED occupancy: the rank's occupancy counters go to
        every peer over NVLink, the local (namespace-grouped) requests are solved against the sum — on the
        side stream, concurrently with the sweep of ``tables`` (None: placement branch only)."""
        self._check(lib().lwse_reconcile_shared_device(
            self._h, C.byref(tables) if tables is not None else None, R.ptr(d_reqs), n_reqs, R.ptr(d_local_occupancy),
            n_namespaces, R.ptr(d_place_out), flags, stream))

    def exchange_status(self) -> int:
        err = C.c_uint32(0)
        self._check(lib().lwse_exchange_status(self._h, C.byref(err)))
        return err.value

    # ------------------------------------------------------- resident tables
    def resident_load(self, lws, groups, pod_state, pod_ident):
        """Make the four input tables resident on the device."""
        self._resident_shape = (len(lws), len(groups))
        self._resident_pods = len(pod_state)
        self._n_place = 0
        t = R.LwsTables(R.ptr(lws), len(lws), R.ptr(groups), len(groups), R.ptr(pod_state), R.ptr(pod_ident),
                        len(pod_state), None, None, None, 0)
        self._check(lib().lwse_resident_load(self._h, C.byref(t)))
        self._chg = None

    _DT = {R.TABLE_LWS: R.LWS_REC, R.TABLE_GROUPS: R.GROUP_REC, R.TABLE_POD_STATE: R.POD_STATE,
           R.TABLE_POD_IDENT: R.POD_IDENT, R.TABLE_PLACE_REQS: R.PLACE_REQ, R.TABLE_DS: R.DS_REC,
           R.TABLE_DS_ROLES: R.DS_ROLE_REC, R.TABLE_DS_REVROLES: R.DS_REVROLE_REC}

    # ----------------------------------------------------------- resident tick
    def resident_arena(self, min_bytes: int = 0) -> np.ndarray:
        """The engine's pinned, mapped patch arena as a uint8 array: patch rows / values written
        into it are read by the GPU in place (no staging copy)."""
        base, size = C.c_void_p(), C.c_uint64()
        self._check(lib().lwse_resident_arena(self._h, min_bytes, C.byref(base), C.byref(size)))
        buf = (C.c_uint8 * size.value).from_address(base.value)
        return np.frombuffer(buf, dtype=np.uint8)

    def resident_place_load(self, reqs: np.ndarray, n_namespaces: int = 1):
        assert reqs.dtype == R.PLACE_REQ
        self._n_place = len(reqs)
        self._check(lib().lwse_resident_place_load(self._h, R.ptr(reqs) if len(reqs) else None, len(reqs), n_namespaces))

    def make_tick(self, segments=(), flags=0) -> "R.Tick":
        """Build a reusable ``lwse_tick`` descriptor.  ``segments``: (table, rows, values) with
        numpy arrays (ideally views of the arena), or (table, first_row, values, True) for a range."""
        return self._fill_tick(R.Tick(), segments, flags)

    def make_ds_tick(self, segments=()) -> "R.DsTick":
        """A reusable ``lwse_ds_tick`` descriptor; ``segments`` as for ``make_tick`` (tables
        ``TABLE_DS`` / ``TABLE_DS_ROLES`` / ``TABLE_DS_REVROLES``)."""
        return self._fill_tick(R.DsTick(), segments, 0)

    def _fill_tick(self, t, segments, flags):
        segs = (R.PatchSeg * max(len(segments), 1))()
        keep = []
        for i, sg in enumerate(segments):
            if len(sg) == 4 and sg[3]:
                table, first, values = sg[0], sg[1], sg[2]
                segs[i] = R.PatchSeg(table, R.PATCH_RANGE, len(values), int(first), None, R.ptr(values))
                keep.append(values)
            else:
                table, rows, values = sg[0], sg[1], sg[2]
                assert rows.dtype == np.uint32 and len(rows) == len(values) and values.dtype == self._DT[table]
                segs[i] = R.PatchSeg(table, 0, len(rows), 0, R.ptr(rows) if len(rows) else None,
                                     R.ptr(values) if len(rows) else None)
                keep.append((rows, values))
        t.segs = segs
        t.n_segs = len(segments)
        t.flags = flags
        t._keep = (segs, keep)
        return t

    def resident_tick(self, tick: "R.Tick"):
        """One tick: patches in, changed result rows out (views of engine-owned pinned memory,
        valid until the next resident call).  → dict of numpy views."""
        self._check(lib().lwse_resident_tick(self._h, C.byref(tick)))
        return self._tick_views(tick)

    def resident_tick_submit(self, tick: "R.Tick"):
        """Enqueue a tick and return (at most two in flight); its patch segments stay untouched in the
        arena until the matching ``resident_tick_wait``."""
        self._check(lib().lwse_resident_tick_submit(self._h, C.byref(tick)))

    def resident_tick_wait(self, tick: "R.Tick" = None):
        """Wait for the OLDEST submitted tick → the same dict as ``resident_tick`` (views valid until
        the second submit after this call)."""
        tick = tick if tick is not None else R.Tick()
        self._check(lib().lwse_resident_tick_wait(self._h, C.byref(tick)))
        return self._tick_views(tick)

    def _tick_views(self, tick: "R.Tick"):
        def view(ptr, n, dtype):
            if not ptr or n == 0:
                return np.zeros(0, dtype=dtype)
            nbytes = n * np.dtype(dtype).itemsize
            return np.frombuffer((C.c_uint8 * nbytes).from_address(ptr), dtype=dtype)

        n_lws = min(tick.n_lws, self._resident_shape[0])
        n_grp = min(tick.n_groups, self._resident_shape[1])
        n_pl = min(tick.n_place, getattr(self, "_n_place", 0))
        return {
            "lws_rows": view(tick.lws_rows, n_lws, np.uint32), "lws_out": view(tick.lws_out, n_lws, R.LWS_OUT),
            "group_rows": view(tick.group_rows, n_grp, np.uint32), "group_out": view(tick.group_out, n_grp, R.GROUP_OUT),
            "place_rows": view(tick.place_rows, n_pl, np.uint32), "place_out": view(tick.place_out, n_pl, R.PLACE_OUT),
            "n_lws": tick.n_lws, "n_groups": tick.n_groups, "n_place": tick.n_place, "rounds": tick.place_rounds,
        }

    def resident_place_outputs(self) -> np.ndarray:
        out = R.aligned_empty(self._n_place, R.PLACE_OUT)
        self._check(lib().lwse_resident_place_outputs(self._h, R.ptr(out)))
        return out

    def resident_occupancy(self) -> np.ndarray:
        occ = np.zeros(max(self.n_nodes, 1), dtype=np.uint32)
        self._check(lib().lwse_resident_occupancy(self._h, R.ptr(occ)))
        return occ[: self.n_nodes]

    def resident_patch(self, which: int, rows, values):
        """Overwrite rows of a resident table (rows: uint32 indices, values: packed rows)."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        values = np.ascontiguousarray(values, dtype=self._DT[which])
        assert len(rows) == len(values)
        self._check(lib().lwse_resident_patch(self._h, which, R.ptr(rows) if len(rows) else None,
                                              R.ptr(values) if len(rows) else None, len(rows)))

    def resident_sweep(self, flags=0, lws_capacity=None, group_capacity=None):
        """Sweep the resident tables → (lws_rows, lws_out, group_rows, group_out, n_lws_changed,
        n_groups_changed): only result rows that changed since the previous resident sweep."""
        n_lws, n_grp = self._resident_shape
        lc = n_lws if lws_capacity is None else lws_capacity
        gc = n_grp if group_capacity is None else group_capacity
        if self._chg is None or self._chg[0] != (lc, gc):
            self._chg = ((lc, gc), np.zeros(max(lc, 1), np.uint32), R.aligned_empty(max(lc, 1), R.LWS_OUT),
                         np.zeros(max(gc, 1), np.uint32), R.aligned_empty(max(gc, 1), R.GROUP_OUT))
        _, lr, lo, gr, go = self._chg
        ch = R.Changes(R.ptr(lr), R.ptr(lo), lc, 0, R.ptr(gr), R.ptr(go), gc, 0)
        self._check(lib().lwse_resident_sweep(self._h, flags, C.byref(ch)))
        nl, ng = min(ch.n_lws, lc), min(ch.n_groups, gc)
        return lr[:nl], lo[:nl], gr[:ng], go[:ng], ch.n_lws, ch.n_groups

    def resident_outputs(self):
        n_lws, n_grp = self._resident_shape
        lo, go = R.aligned_empty(n_lws, R.LWS_OUT), R.aligned_empty(n_grp, R.GROUP_OUT)
        self._check(lib().lwse_resident_outputs(self._h, R.ptr(lo), R.ptr(go)))
        return lo, go

    # -------------------------------------------------------------- placement
    def place_host(self, reqs: np.ndarray, occupancy=None, n_namespaces=1):
        assert reqs.dtype == R.PLACE_REQ
        out = R.aligned_empty(len(reqs), R.PLACE_OUT)
        rounds = C.c_uint32(0)
        if occupancy is not None:
            occupancy = np.ascontiguousarray(occupancy, dtype=np.uint32)
        self._check(
            lib().lwse_place_host(self._h, R.ptr(reqs), len(reqs), R.ptr(occupancy), n_namespaces,
                                  R.ptr(out), C.byref(rounds))
        )
        return out, rounds.value

    def place_device(self, d_reqs, n_reqs, d_occupancy, n_namespaces, d_out, stream=None, want_rounds=False):
        """Enqueue a placement round; synchronizes only when ``want_rounds``."""
        rounds = C.c_uint32(0)
        self._check(
            lib().lwse_place_device(self._h, R.ptr(d_reqs), n_reqs, R.ptr(d_occupancy), n_namespaces,
                                    R.ptr(d_out), C.byref(rounds) if want_rounds else None, stream)
        )
        return rounds.value if want_rounds else None

    def place_grouped_device(self, d_reqs, n_reqs, d_occupancy, n_namespaces, d_out, flags=0, stream=None, want_rounds=False):
        """Placement round over a request table grouped by namespace (one CTA per namespace; flags:
        SWEEP_PLACE_SCAN = brute-force (request x node) form).  → (rounds, scans) when ``want_rounds``."""
        rounds, scans = C.c_uint32(0), C.c_uint32(0)
        self._check(lib().lwse_place_grouped_device(self._h, R.ptr(d_reqs), n_reqs, R.ptr(d_occupancy), n_namespaces,
                                                    R.ptr(d_out), flags, C.byref(rounds) if want_rounds else None,
                                                    C.byref(scans) if want_rounds else None, stream))
        return (rounds.value, scans.value) if want_rounds else None

    def place_gathered_device(self, d_parts, n_parts, part_stride_bytes, reqs_offset_bytes, reqs_per_part,
                              n_namespaces, d_out, stream=None, want_rounds=False):
        """Placement over the all-gathered [occupancy | requests] parts of every rank."""
        rounds = C.c_uint32(0)
        self._check(
            lib().lwse_place_gathered_device(self._h, R.ptr(d_parts), n_parts, part_stride_bytes, reqs_offset_bytes,
                                             reqs_per_part, n_namespaces, R.ptr(d_out),
                                             C.byref(rounds) if want_rounds else None, stream)
        )
        return rounds.value if want_rounds else None

    # --------------------------------------------------------------------- DS
    def sweep_ds_host(self, ds, roles, revroles, out=None):
        """lwse_sweep_ds_host: host tables in, host result rows out.  `out` = (ds_out, role_out, revrole_out)
        arrays to fill instead of fresh ones (page-locked tables and outputs copy at PCIe speed; pageable ones
        are staged by the driver)."""
        assert ds.dtype == R.DS_REC and roles.dtype == R.DS_ROLE_REC and revroles.dtype == R.DS_REVROLE_REC
        if out is None:
            ds_out = R.aligned_empty(len(ds), R.DS_OUT)
            role_out = R.aligned_empty(len(roles), R.DS_ROLE_OUT)
            revrole_out = R.aligned_empty(len(revroles), R.DS_REVROLE_OUT)
        else:
            ds_out, role_out, revrole_out = out
            assert ds_out.dtype == R.DS_OUT and role_out.dtype == R.DS_ROLE_OUT and revrole_out.dtype == R.DS_REVROLE_OUT
            assert len(ds_out) == len(ds) and len(role_out) == len(roles) and len(revrole_out) == len(revroles)
        t = R.DsTables(
            R.ptr(ds), len(ds), R.ptr(roles), len(roles), R.ptr(revroles), len(revroles),
            R.ptr(ds_out), R.ptr(role_out), R.ptr(revrole_out),
        )
        self._check(lib().lwse_sweep_ds_host(self._h, C.byref(t)))
        return ds_out, role_out, revrole_out

    def sweep_ds_device(self, d_ds, n_ds, d_roles, n_roles, d_revroles, n_revroles, d_ds_out, d_role_out,
                        d_revrole_out, stream=None):
        t = R.DsTables(
            R.ptr(d_ds), n_ds, R.ptr(d_roles), n_roles, R.ptr(d_revroles), n_revroles,
            R.ptr(d_ds_out), R.ptr(d_role_out), R.ptr(d_revrole_out),
        )
        self._check(lib().lwse_sweep_ds_device(self._h, C.byref(t), stream))

    def ds_resident_load(self, ds, roles, revroles):
        """Make the three DS input tables resident on the device (committed results start at zero)."""
        assert ds.dtype == R.DS_REC and roles.dtype == R.DS_ROLE_REC and revroles.dtype == R.DS_REVROLE_REC
        self._ds_shape = (len(ds), len(roles), len(revroles))
        t = R.DsTables(R.ptr(ds), len(ds), R.ptr(roles), len(roles), R.ptr(revroles), len(revroles), None, None, None)
        self._check(lib().lwse_ds_resident_load(self._h, C.byref(t)))

    def ds_resident_tick(self, tick: "R.DsTick"):
        """One DS tick: patches in, listed result rows out → dict of numpy views of engine-owned
        pinned memory (valid until the next resident call)."""
        self._check(lib().lwse_ds_resident_tick(self._h, C.byref(tick)))
        return self._ds_tick_views(tick)

    @staticmethod
    def _ds_tick_views(tick: "R.DsTick"):
        def view(ptr, n, dtype):
            if not ptr or n == 0:
                return np.zeros(0, dtype=dtype)
            nbytes = n * np.dtype(dtype).itemsize
            return np.frombuffer((C.c_uint8 * nbytes).from_address(ptr), dtype=dtype)

        return {
            "ds_rows": view(tick.ds_rows, tick.n_ds, np.uint32), "ds_out": view(tick.ds_out, tick.n_ds, R.DS_OUT),
            "role_rows": view(tick.role_rows, tick.n_roles, np.uint32),
            "role_out": view(tick.role_out, tick.n_roles, R.DS_ROLE_OUT),
            "revrole_rows": view(tick.revrole_rows, tick.n_revroles, np.uint32),
            "revrole_out": view(tick.revrole_out, tick.n_revroles, R.DS_REVROLE_OUT),
            "n_ds": tick.n_ds, "n_roles": tick.n_roles, "n_revroles": tick.n_revroles,
        }

    def ds_resident_outputs(self):
        """Every committed DS result row → (ds_out, role_out, revrole_out)."""
        n_ds, n_ro, n_rr = self._ds_shape
        o = (R.aligned_empty(n_ds, R.DS_OUT), R.aligned_empty(n_ro, R.DS_ROLE_OUT), R.aligned_empty(n_rr, R.DS_REVROLE_OUT))
        self._check(lib().lwse_ds_resident_outputs(self._h, *(R.ptr(x) for x in o)))
        return o

    # ------------------------------------------------------------- joint tick
    def joint_tick(self, tick, ds_tick):
        """One tick of both controllers (``tick`` may be None: DS only) → (lws_result, ds_result), the
        dicts of ``resident_tick`` and ``ds_resident_tick`` (lws_result None without ``tick``)."""
        self._check(lib().lwse_joint_tick(self._h, C.byref(tick) if tick is not None else None, C.byref(ds_tick)))
        return (self._tick_views(tick) if tick is not None else None), self._ds_tick_views(ds_tick)

    def joint_tick_submit(self, tick, ds_tick):
        """Enqueue a joint tick and return; it shares the two-slot ring of ``resident_tick_submit``."""
        self._check(lib().lwse_joint_tick_submit(self._h, C.byref(tick) if tick is not None else None, C.byref(ds_tick)))

    def joint_tick_wait(self):
        """Wait for the OLDEST tick in flight, joint or LWS-only → (lws_result, ds_result); an LWS-only
        tick reports no DS rows.  lws_result is None on an engine without resident LWS tables."""
        tick = R.Tick() if hasattr(self, "_resident_shape") else None
        ds_tick = R.DsTick()
        self._check(lib().lwse_joint_tick_wait(self._h, C.byref(tick) if tick is not None else None, C.byref(ds_tick)))
        return (self._tick_views(tick) if tick is not None else None), self._ds_tick_views(ds_tick)

    # ------------------------------------------------------------- group keys
    def group_keys_host(self, strings) -> np.ndarray:
        """SHA-1 of each string → (n, 20) uint8."""
        enc = [s.encode() if isinstance(s, str) else bytes(s) for s in strings]
        offsets = np.zeros(len(enc) + 1, dtype=np.uint32)
        offsets[1:] = np.cumsum([len(b) for b in enc], dtype=np.uint64).astype(np.uint32)
        blob = np.frombuffer(b"".join(enc) + b"\0", dtype=np.uint8)
        digests = np.zeros((len(enc), 20), dtype=np.uint8)
        self._check(
            lib().lwse_group_keys_host(self._h, R.ptr(blob), R.ptr(offsets), len(enc), R.ptr(digests))
        )
        return digests

    def subgroup_keys_host(self, leader_names, pod_count, subgroup_size, worker_index):
        """getSubGroupIndex + SHA-1("<leaderName>/<index>") for a batch of pods → (index int32[n], digests (n, 20))."""
        enc = [s.encode() if isinstance(s, str) else bytes(s) for s in leader_names]
        n = len(enc)
        offsets = np.zeros(n + 1, dtype=np.uint32)
        offsets[1:] = np.cumsum([len(b) for b in enc], dtype=np.uint64).astype(np.uint32)
        blob = np.frombuffer(b"".join(enc) + b"\0\0\0\0", dtype=np.uint8)
        pc, sg, wi = (np.ascontiguousarray(x, dtype=np.int32) for x in (pod_count, subgroup_size, worker_index))
        index = np.zeros(n, dtype=np.int32)
        digests = np.zeros((n, 20), dtype=np.uint8)
        self._check(lib().lwse_subgroup_keys_host(self._h, R.ptr(blob), R.ptr(offsets), n, R.ptr(pc), R.ptr(sg), R.ptr(wi),
                                                  R.ptr(index), R.ptr(digests)))
        return index, digests

    def group_keys_device(self, d_bytes, d_offsets, n, d_digests, stream=None):
        self._check(lib().lwse_group_keys_device(self._h, R.ptr(d_bytes), R.ptr(d_offsets), n, R.ptr(d_digests), stream))
