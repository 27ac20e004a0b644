"""Fixed-width record tables of the engine — numpy mirrors of ``include/lwse.h``.

Every dtype below has exactly the layout of the C struct of the same name; the
``tests/test_abi.py`` suite checks the sizes and field offsets against the
header through the compiled library.  Field meaning and the reference lines
each field comes from are documented once, in the header.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 2
NONE = 0xFFFFFFFF
NODE_NOT_FOUND = 0xFFFFFFFE

# --------------------------------------------------------------------------- #
# input records
# --------------------------------------------------------------------------- #
LWS_REC = np.dtype(
    [
        ("rev_hash", "<u8"),
        ("size", "<i4"),
        ("flags", "<u4"),
        ("replicas", "<i4"),
        ("partition", "<i4"),
        ("max_surge", "<i4"),
        ("max_unavailable", "<i4"),
        ("sts_replicas", "<i4"),
        ("sts_partition", "<i4"),
        ("sts_replicas_annotation", "<i4"),
        ("subgroup_size", "<i4"),
        ("uid_hash", "<u8"),
        ("group_base", "<u4"),
        ("group_count", "<u4"),
    ],
    align=False,
)
assert LWS_REC.itemsize == 64

LWS_SURGE_IS_PERCENT = 1 << 0
LWS_UNAVAIL_IS_PERCENT = 1 << 1
LWS_STS_EXISTS = 1 << 2
LWS_UPDATED = 1 << 3
LWS_ANNOT_VALID = 1 << 4
LWS_RESTART_SHIFT = 5
LWS_RESTART_MASK = 3 << 5
LWS_RECREATE_AFTER_START_ANNOT = 1 << 7
LWS_STARTUP_LEADER_READY = 1 << 8
LWS_EXCLUSIVE_TOPOLOGY = 1 << 9
LWS_SUBGROUP_LEADER_EXCLUDED = 1 << 10
LWS_GROUP_LABEL_INVALID = 1 << 11
LWS_INTSTR_INVALID = 1 << 12
LWS_IRREGULAR = 1 << 13

RESTART_NONE = 0
RESTART_ON_POD_RESTART = 1
RESTART_AFTER_START = 2

GROUP_REC = np.dtype(
    [
        ("leader_rev_hash", "<u8"),
        ("wsts_rev_hash", "<u8"),
        ("wsts_spec_replicas", "<i4"),
        ("wsts_avail_replicas", "<i4"),
        ("leader_uid_hash", "<u4"),
        ("wsts_uid_hash", "<u4"),
        ("wsts_owner_uid_hash", "<u4"),
        ("leader_node", "<u4"),
        ("pod_base", "<u4"),
        ("pod_count", "<u4"),
        ("lws_index", "<u4"),
        ("flags", "<u4"),
        ("reserved", "<u4", (2,)),
    ],
    align=False,
)
assert GROUP_REC.itemsize == 64

GRP_POD_PRESENT = 1 << 0
GRP_POD_NAME_MATCH = 1 << 1
GRP_POD_RUNNING = 1 << 2
GRP_POD_READY = 1 << 3
GRP_POD_DELETING = 1 << 4
GRP_WSTS_LABEL_NAME_MATCH = 1 << 5
GRP_WSTS_FOUND = 1 << 6
GRP_WSTS_REV_SETTLED = 1 << 7
GRP_WSTS_OWNER_IS_POD = 1 << 8
GRP_WSTS_OWNER_NAME_MATCH = 1 << 9
GRP_MISTAKEN_ANNOTATION = 1 << 10
GRP_REVISION_EXISTS = 1 << 11

POD_STATE = np.dtype("u1")  # lwse_pod_state: the hot byte column
POD_IDENT = np.dtype([("rev_hash", "<u8"), ("owner_uid_hash", "<u4"), ("place", "<u4")], align=False)
assert POD_IDENT.itemsize == 16


def pod_ident_table(rev_hash: np.ndarray, owner_uid_hash: np.ndarray, place: np.ndarray | int = 0) -> np.ndarray:
    """Build the identity column from 64-bit revision hashes, 32-bit owner uid hashes and the
    ``place`` words (PODID_NAME_OK | PODID_SCHEDULED | node << PODID_NODE_SHIFT)."""
    t = aligned_empty(len(rev_hash), POD_IDENT)
    t["rev_hash"] = np.asarray(rev_hash, dtype=np.uint64)
    t["owner_uid_hash"] = owner_uid_hash
    t["place"] = place
    return t


POD_PHASE_MASK = 3
POD_PHASE_PENDING = 1
POD_PHASE_RUNNING = 2
POD_ANY_RESTART = 1 << 2
POD_DELETING = 1 << 3
POD_OWNER_SHIFT = 4
POD_OWNER_MASK = 3 << 4
POD_OWNER_NONE, POD_OWNER_POD, POD_OWNER_STS, POD_OWNER_OTHER = 0, 1, 2, 3
POD_OWNER_NAME_MATCH = 1 << 6
POD_IS_LEADER = 1 << 7
PODID_NAME_OK = 1 << 0
PODID_SCHEDULED = 1 << 1
PODID_NODE_SHIFT = 10
POD_NODE_MAX = (1 << 22) - 1


def occupancy_of(pod_ident: np.ndarray, n_nodes: int) -> np.ndarray:
    """Scheduled pods per node of an identity column (what the engine counts at load)."""
    place = pod_ident["place"]
    sched = (place & PODID_SCHEDULED) != 0
    node = (place[sched] >> PODID_NODE_SHIFT).astype(np.int64)
    return np.bincount(node[node < n_nodes], minlength=n_nodes).astype(np.uint32)


NODE_REC = np.dtype(
    [("topo_value_hash", "<u8"), ("domain_id", "<u4"), ("capacity", "<u2"), ("flags", "<u2")],
    align=False,
)
assert NODE_REC.itemsize == 16
NODE_HAS_TOPOLOGY = 1 << 0
NODE_SCHEDULABLE = 1 << 1

# --------------------------------------------------------------------------- #
# output records
# --------------------------------------------------------------------------- #
LWS_OUT = np.dtype(
    [
        ("sts_partition", "<i4"),
        ("sts_replicas", "<i4"),
        ("sts_max_unavailable", "<i4"),
        ("ready_replicas", "<i4"),
        ("updated_replicas", "<i4"),
        ("min_member", "<i4"),
        ("flags", "<u4"),
        ("unready_replicas", "<i4"),
    ],
    align=False,
)
assert LWS_OUT.itemsize == 32

LOUT_RUP_ERROR = 1 << 0
LOUT_STATUS_ERROR = 1 << 1
LOUT_COND_SHIFT = 2
LOUT_COND_MASK = 3 << 2
LOUT_UPDATE_DONE = 1 << 4
LOUT_EVENT_SHIFT = 5
LOUT_EVENT_MASK = 3 << 5
LOUT_IRREGULAR = 1 << 7
LOUT_BAD_TABLE = 1 << 8
COND_PROGRESSING, COND_AVAILABLE, COND_UPDATE_IN_PROGRESS = 0, 1, 2
EVENT_NONE, EVENT_DELETE_ONE, EVENT_DELETE_RANGE = 0, 1, 2

GROUP_OUT = np.dtype(
    [("flags", "<u4"), ("first_trigger", "<u4"), ("worker_replicas", "<i4"), ("domain_id", "<u4")],
    align=False,
)
assert GROUP_OUT.itemsize == 16

GOUT_STATE_READY = 1 << 0
GOUT_STATE_UPDATED = 1 << 1
GOUT_COUNTED = 1 << 2
GOUT_COND_READY = 1 << 3
GOUT_COND_UPDATED = 1 << 4
GOUT_PENDING = 1 << 5
GOUT_DELETE_LEADER = 1 << 6
GOUT_LEADER_DELETING = 1 << 7
GOUT_RESTART_ERROR = 1 << 8
GOUT_CREATE_WSTS = 1 << 9
GOUT_WAIT_SCHEDULE = 1 << 10
GOUT_TOPOLOGY_ERROR = 1 << 11
GOUT_REQUEUE_REVISION = 1 << 12
GOUT_CREATE_PODGROUP = 1 << 13
GOUT_BAD_TABLE = 1 << 14

SWEEP_GANG = 1 << 0
SWEEP_SKIP_GROUP_PASS = 1 << 1
SWEEP_SKIP_LWS_PASS = 1 << 2
SWEEP_SKIP_POD_SCAN = 1 << 3
SWEEP_REUSE_POD_IDENT = 1 << 4
SWEEP_PLACE_GROUPED = 1 << 5
SWEEP_PLACE_SCAN = 1 << 6
EXCHANGE_LAGGED = 1 << 16

# --------------------------------------------------------------------------- #
# placement
# --------------------------------------------------------------------------- #
PLACE_REQ = np.dtype(
    [
        ("priority", "<u8"),
        ("group_key", "<u8"),
        ("group", "<u4"),
        ("ns", "<u4"),
        ("size", "<i4"),
        ("leader_node", "<u4"),
    ],
    align=False,
)
assert PLACE_REQ.itemsize == 32
PLACE_OUT = np.dtype(
    [("domain_id", "<u4"), ("leader_node", "<u4"), ("flags", "<u4"), ("score", "<u4")], align=False
)
assert PLACE_OUT.itemsize == 16
PLACE_PLACED = 1 << 0
PLACE_PINNED = 1 << 1
PLACE_CONFLICT = 1 << 2
PLACE_UNSCHEDULABLE = 1 << 3

# --------------------------------------------------------------------------- #
# DisaggregatedSet
# --------------------------------------------------------------------------- #
DS_MAX_ROLES = 10
DS_REC = np.dtype(
    [
        ("uid_hash", "<u8"),
        ("role_base", "<u4"),
        ("n_roles", "<u4"),
        ("n_spec_roles", "<u4"),
        ("rev_base", "<u4"),
        ("n_old_revs", "<u4"),
        ("flags", "<u4"),
    ],
    align=False,
)
assert DS_REC.itemsize == 32
DS_HAS_NEW_REVISION = 1 << 0

DS_ROLE_REC = np.dtype(
    [("target_replicas", "<i4"), ("max_surge", "<i4"), ("max_unavailable", "<i4"), ("flags", "<u4")],
    align=False,
)
assert DS_ROLE_REC.itemsize == 16
ROLE_SURGE_IS_PERCENT = 1 << 0
ROLE_UNAVAIL_IS_PERCENT = 1 << 1
ROLE_HAS_ROLLING_CONFIG = 1 << 2
ROLE_IN_SPEC = 1 << 3
ROLE_SURGE_INVALID = 1 << 4
ROLE_UNAVAIL_INVALID = 1 << 5

DS_REVROLE_REC = np.dtype(
    [("replicas", "<i4"), ("initial_replicas", "<i4"), ("ready_replicas", "<i4"), ("flags", "<u4")],
    align=False,
)
assert DS_REVROLE_REC.itemsize == 16
RR_EXISTS = 1 << 0
RR_REPLICAS_NIL = 1 << 1
RR_TS_SHIFT = 2

DS_OUT = np.dtype(
    [("flags", "<u4"), ("drained_revs", "<u4"), ("ready_revs", "<u4"), ("reserved", "<u4")], align=False
)
assert DS_OUT.itemsize == 16
DOUT_ROLLING = 1 << 0
DOUT_INIT = 1 << 1
DOUT_STABLE = 1 << 2
DOUT_STEP = 1 << 3
DOUT_COMPLETE = 1 << 4
DOUT_NEW_READY = 1 << 5
DOUT_BAD_TABLE = 1 << 6
DS_MAX_OLD_REVS = 32

DS_ROLE_OUT = np.dtype([("next_old", "<i4"), ("next_new", "<i4")], align=False)
assert DS_ROLE_OUT.itemsize == 8
DS_REVROLE_OUT = np.dtype("<i4")


# --------------------------------------------------------------------------- #
# ctypes bundles (lwse_lws_tables / lwse_ds_tables / lwse_config)
# --------------------------------------------------------------------------- #
class LwsTables(C.Structure):
    _fields_ = [
        ("lws", C.c_void_p),
        ("n_lws", C.c_uint32),
        ("groups", C.c_void_p),
        ("n_groups", C.c_uint32),
        ("pod_state", C.c_void_p),
        ("pod_ident", C.c_void_p),
        ("n_pods", C.c_uint64),
        ("lws_out", C.c_void_p),
        ("group_out", C.c_void_p),
        ("node_occupancy", C.c_void_p),
        ("flags", C.c_uint32),
    ]


class Changes(C.Structure):
    _fields_ = [
        ("lws_rows", C.c_void_p),
        ("lws_out", C.c_void_p),
        ("lws_capacity", C.c_uint32),
        ("n_lws", C.c_uint32),
        ("group_rows", C.c_void_p),
        ("group_out", C.c_void_p),
        ("group_capacity", C.c_uint32),
        ("n_groups", C.c_uint32),
    ]


TABLE_LWS, TABLE_GROUPS, TABLE_POD_STATE, TABLE_POD_IDENT, TABLE_PLACE_REQS = 0, 1, 2, 3, 4
TABLE_DS, TABLE_DS_ROLES, TABLE_DS_REVROLES = 5, 6, 7  # the DS tick's tables (lwse_ds_resident_tick)
PATCH_RANGE = 1 << 0
TICK_MAX_SEGS = 8
TICK_PLACE = 1 << 8
TICK_NO_SWEEP = 1 << 9
TICK_SHARED_OCCUPANCY = 1 << 10


class PatchSeg(C.Structure):
    _fields_ = [
        ("table", C.c_uint32),
        ("flags", C.c_uint32),
        ("n", C.c_uint32),
        ("first_row", C.c_uint32),
        ("rows", C.c_void_p),
        ("values", C.c_void_p),
    ]


class Tick(C.Structure):
    _fields_ = [
        ("segs", C.POINTER(PatchSeg)),
        ("n_segs", C.c_uint32),
        ("flags", C.c_uint32),
        ("lws_rows", C.c_void_p),
        ("lws_out", C.c_void_p),
        ("n_lws", C.c_uint32),
        ("n_groups", C.c_uint32),
        ("group_rows", C.c_void_p),
        ("group_out", C.c_void_p),
        ("place_rows", C.c_void_p),
        ("place_out", C.c_void_p),
        ("n_place", C.c_uint32),
        ("place_rounds", C.c_uint32),
    ]


class DsTick(C.Structure):
    _fields_ = [
        ("segs", C.POINTER(PatchSeg)),
        ("n_segs", C.c_uint32),
        ("flags", C.c_uint32),
        ("ds_rows", C.c_void_p),
        ("ds_out", C.c_void_p),
        ("n_ds", C.c_uint32),
        ("n_roles", C.c_uint32),
        ("role_rows", C.c_void_p),
        ("role_out", C.c_void_p),
        ("revrole_rows", C.c_void_p),
        ("revrole_out", C.c_void_p),
        ("n_revroles", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class DsTables(C.Structure):
    _fields_ = [
        ("ds", C.c_void_p),
        ("n_ds", C.c_uint32),
        ("roles", C.c_void_p),
        ("n_roles", C.c_uint32),
        ("revroles", C.c_void_p),
        ("n_revroles", C.c_uint32),
        ("ds_out", C.c_void_p),
        ("role_out", C.c_void_p),
        ("revrole_out", C.c_void_p),
    ]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32),
        ("device", C.c_int32),
        ("flags", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


def aligned_empty(n: int, dtype: np.dtype, align: int = 64) -> np.ndarray:
    """An ``n``-row table whose base address is ``align``-byte aligned."""
    dtype = np.dtype(dtype)
    raw = np.zeros(n * dtype.itemsize + align, dtype=np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off : off + n * dtype.itemsize].view(dtype)


def ptr(a) -> int | None:
    """Base address of a numpy array / torch tensor, or None."""
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return a.ctypes.data


FNV_OFFSET = 0xCBF29CE484222325
FNV_PRIME = 0x100000001B3


def hash64(s: str | bytes) -> int:
    """FNV-1a 64 — the string hash of the encoders (same as ``lwse_hash64``)."""
    if isinstance(s, str):
        s = s.encode()
    h = FNV_OFFSET
    for b in s:
        h = ((h ^ b) * FNV_PRIME) & 0xFFFFFFFFFFFFFFFF
    return h


def hash32(s: str | bytes) -> int:
    h = hash64(s)
    return (h ^ (h >> 32)) & 0xFFFFFFFF
