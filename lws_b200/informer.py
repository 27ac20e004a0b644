"""Watch events → row patches: the incremental encoder (SURVEY.md §8(f) rank 1).

The reference reads its world through informer-cache ``List`` calls on every reconcile
(pkg/controllers/leaderworkerset_controller.go:421, :584, :598; pod_controller.go:348).  The
engine keeps the same world as resident record tables; this module keeps them current from the
watch stream, so that a reconcile pass is ``lwse_resident_tick(patches)`` instead of a re-encode:

* the tables are laid out in **slots**: every LeaderWorkerSet owns a fixed range of group rows,
  pod rows and placement-request rows with some slack, so an event never moves another object;
* an event marks its object dirty; ``flush()`` re-encodes just the dirty objects with the very
  function the full encoder uses (``encoder.encode_lws`` on the object's slice of the cache — the
  incremental tables therefore mean exactly what a fresh encode means), compares the fresh rows
  with the resident ones and emits one patch segment per table holding only the rows that differ;
* an object that outgrows its slots is moved to the spare rows at the end of the tables; when
  those run out ``needs_reload`` is set and the caller re-encodes everything (``lwse_resident_load``).

Rows that no object references (slack, vacated slots) are never read by the engine: group rows are
reached through ``lws.group_base/count``, pod rows through ``groups.pod_base/count``; unused
placement-request rows are inert (unpinned, size 0).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Optional

import numpy as np

from . import api, encoder
from . import records as R


@dataclass
class Slots:
    lws_row: int
    group_base: int
    group_cap: int
    pod_base: int
    pod_cap: int
    req_base: int  # placement request rows = group rows of exclusive objects (same count as group_cap), or -1


@dataclass
class Patches:
    """One tick's row patches, ready for ``Engine.make_tick`` (rows sorted, distinct)."""

    segments: list = field(default_factory=list)  # (table id, rows uint32, values)

    def add(self, table: int, rows: list, values: np.ndarray):
        if rows:
            order = np.argsort(rows, kind="stable")
            r = np.asarray(rows, dtype=np.uint32)[order]
            v = R.aligned_empty(len(r), values.dtype)
            v[:] = values[order]
            self.segments.append((table, r, v))

    def n_rows(self) -> int:
        return sum(len(s[1]) for s in self.segments)


def _slack(n: int) -> int:
    return n + max(2, n // 4)


class IncrementalEncoder:
    """Resident tables + the slice of the informer cache they were encoded from."""

    def __init__(self, items: list, cluster: encoder.Cluster, topology_key: Optional[str] = None,
                 namespaces: Optional[dict] = None, spare: float = 0.25):
        self.topology_key = topology_key
        self.nodes = list(cluster.nodes)
        self._encoded_nodes = encoder.encode_nodes(self.nodes, topology_key)
        self.node_rec, self.domain_values, self.node_index = self._encoded_nodes
        self.ns_ids = dict(namespaces or {})  # namespace name → dense id (exclusivity scope)
        self.items: dict[tuple, encoder.LwsItem] = {(it.lws.namespace, it.lws.name): it for it in items}
        self.pods: dict[tuple, dict] = {}  # (ns, set name) → {pod name: Pod}
        self.sts: dict[tuple, dict] = {}   # (ns, set name) → {sts name: StatefulSet}  (the leader sts lives in the item)
        for p in cluster.pods:
            self.pods.setdefault((p.namespace, p.labels.get(api.SetNameLabelKey)), {})[p.name] = p
        for s in cluster.statefulsets:
            self.sts.setdefault((s.namespace, s.labels.get(api.SetNameLabelKey)), {})[s.name] = s
        self.needs_reload = False
        self.dirty: set = set()
        # ---- first layout: objects in (namespace id, name) order so that the request table is grouped by namespace
        keys = sorted(self.items, key=lambda k: (self._ns_id(k[0]), k))
        fresh = {k: self._encode_object(k) for k in keys}
        self.slots: dict[tuple, Slots] = {}
        g = p = r = 0
        for i, k in enumerate(keys):
            t = fresh[k]
            gcap = _slack(max(len(t.groups), self._wanted_groups(k)))
            size = max(1, self.items[k].lws.size)
            pcap = max(_slack(len(t.pod_state)), gcap * (size + 1))
            self.slots[k] = Slots(i, g, gcap, p, pcap, r)
            g, p, r = g + gcap, p + pcap, r + gcap
        self.order = keys
        n_lws = len(keys)
        self.lws = R.aligned_empty(n_lws + max(4, int(n_lws * spare)), R.LWS_REC)
        self.groups = R.aligned_empty(g + max(16, int(g * spare)), R.GROUP_REC)
        self.pod_state = R.aligned_empty(p + max(64, int(p * spare)), R.POD_STATE)
        self.pod_ident = R.aligned_empty(len(self.pod_state), R.POD_IDENT)
        self.reqs = R.aligned_empty(len(self.groups), R.PLACE_REQ)
        self.n_lws, self.g_end, self.p_end, self.r_end = n_lws, g, p, r
        last_ns = max([self._ns_id(k[0]) for k in keys], default=0)
        self.reqs["leader_node"] = R.NONE  # inert rows: unpinned, size 0 — never claim anything;
        self.reqs["ns"] = last_ns          # the spare tail keeps the table grouped by namespace
        for k in keys:
            self._write_object(k, fresh[k], None)
        self.n_namespaces = max(1, last_ns + 1, len(self.ns_ids))

    # ------------------------------------------------------------------ helpers
    def _ns_id(self, namespace: str) -> int:
        return self.ns_ids.setdefault(namespace, len(self.ns_ids))

    def _wanted_groups(self, key) -> int:
        it = self.items[key]
        want = it.lws.replicas
        surge, is_pct, ok = encoder.parse_int_or_percent(it.lws.rollingUpdate.maxSurge)
        if ok:
            want += -(-surge * it.lws.replicas // 100) if is_pct else surge
        if it.leader_sts is not None:
            want = max(want, it.leader_sts.replicas)
        return max(want, 0)

    def _encode_object(self, key) -> encoder.LwsTables:
        it = self.items[key]
        cl = encoder.Cluster(pods=list(self.pods.get(key, {}).values()),
                             statefulsets=list(self.sts.get(key, {}).values()), nodes=self.nodes)
        return encoder.encode_lws([it], cl, self.topology_key, encoded_nodes=self._encoded_nodes)

    def _object_requests(self, key, t: encoder.LwsTables, sl: Slots) -> np.ndarray:
        """The request rows of the object's slot range (inert where no exclusive group sits)."""
        out = R.aligned_empty(sl.group_cap, R.PLACE_REQ)
        out["leader_node"] = R.NONE
        out["ns"] = self._ns_id(key[0])
        if len(t.lws) and (int(t.lws["flags"][0]) & R.LWS_EXCLUSIVE_TOPOLOGY) and len(t.groups):
            rq = encoder.encode_place_requests(t.lws, t.groups)
            idx = rq["group"].astype(np.int64)  # group rows of this object start at 0 in its own encode
            rq["group"] = idx + sl.group_base
            rq["ns"] = self._ns_id(key[0])
            out[idx] = rq
        return out

    def _write_object(self, key, t: encoder.LwsTables, patches: Optional[Patches]):
        """Place the object's fresh rows into its slots; with `patches`, emit the rows that changed."""
        sl = self.slots[key]
        ng, npod = len(t.groups), len(t.pod_state)
        if ng > sl.group_cap or npod > sl.pod_cap:
            if not self._relocate(key, ng, npod):
                self.needs_reload = True
                return
            sl = self.slots[key]
        lws_row = t.lws.copy()
        lws_row["group_base"] = sl.group_base
        grp = t.groups.copy()
        grp["lws_index"] = sl.lws_row
        grp["pod_base"] = grp["pod_base"].astype(np.int64) + sl.pod_base
        reqs = self._object_requests(key, t, sl)

        def put(table_id, table, base, fresh_rows):
            n = len(fresh_rows)
            if n == 0:
                return
            cur = table[base: base + n]
            if patches is None:
                cur[:] = fresh_rows
                return
            a = np.ascontiguousarray(cur).view(np.uint8).reshape(n, -1)
            b = np.ascontiguousarray(fresh_rows).view(np.uint8).reshape(n, -1)
            diff = np.flatnonzero((a != b).any(axis=1))
            if len(diff):
                vals = R.aligned_empty(len(diff), table.dtype)
                vals[:] = fresh_rows[diff]
                cur[diff] = vals
                patches._pending.setdefault(table_id, ([], []))
                patches._pending[table_id][0].extend((diff + base).tolist())
                patches._pending[table_id][1].append(vals)

        put(R.TABLE_LWS, self.lws, sl.lws_row, lws_row)
        put(R.TABLE_GROUPS, self.groups, sl.group_base, grp)
        # the pod columns are written over the WHOLE slot range: rows a shrinking object no longer
        # references go back to zero (the engine counts node occupancy over every identity row)
        pst = R.aligned_empty(sl.pod_cap, R.POD_STATE)
        pst[:npod] = t.pod_state
        pid = R.aligned_empty(sl.pod_cap, R.POD_IDENT)
        pid[:npod] = t.pod_ident
        put(R.TABLE_POD_STATE, self.pod_state, sl.pod_base, pst)
        put(R.TABLE_POD_IDENT, self.pod_ident, sl.pod_base, pid)
        put(R.TABLE_PLACE_REQS, self.reqs, sl.req_base, reqs)

    def _relocate(self, key, ng: int, npod: int) -> bool:
        """Move an object that outgrew its slots to the spare rows at the end of the tables."""
        sl = self.slots[key]
        gcap = _slack(max(ng, self._wanted_groups(key)))
        size = max(1, self.items[key].lws.size)
        pcap = max(_slack(npod), gcap * (size + 1))
        if self.g_end + gcap > len(self.groups) or self.p_end + pcap > len(self.pod_state) or self.r_end + gcap > len(self.reqs):
            return False
        # the vacated request rows must stop claiming: they are rewritten as inert by the diff below
        self._vacated_reqs = (sl.req_base, sl.group_cap, self._ns_id(key[0]))
        self._vacated_pods = (sl.pod_base, sl.pod_cap)  # and the vacated pod rows must stop occupying nodes
        self.slots[key] = Slots(sl.lws_row, self.g_end, gcap, self.p_end, pcap, self.r_end)
        self.g_end, self.p_end, self.r_end = self.g_end + gcap, self.p_end + pcap, self.r_end + gcap
        return True

    # ------------------------------------------------------------------- events
    def _set_key(self, obj):
        return (obj.namespace, obj.labels.get(api.SetNameLabelKey))

    def pod_event(self, kind: str, pod: api.Pod):
        """kind: ADDED | MODIFIED | DELETED (a watch event of the pod informer)."""
        key = self._set_key(pod)
        if key not in self.items:
            return
        bucket = self.pods.setdefault(key, {})
        if kind == "DELETED":
            bucket.pop(pod.name, None)
        else:
            bucket[pod.name] = pod
        self.dirty.add(key)

    def statefulset_event(self, kind: str, sts: api.StatefulSet):
        key = self._set_key(sts)
        if key not in self.items:
            return
        it = self.items[key]
        if sts.name == it.lws.name and api.GroupIndexLabelKey not in sts.labels:  # the leader StatefulSet
            it.leader_sts = None if kind == "DELETED" else sts
        else:
            bucket = self.sts.setdefault(key, {})
            if kind == "DELETED":
                bucket.pop(sts.name, None)
            else:
                bucket[sts.name] = sts
        self.dirty.add(key)

    def lws_event(self, kind: str, item: encoder.LwsItem):
        """MODIFIED only: a new or deleted object changes the table shapes → reload."""
        key = (item.lws.namespace, item.lws.name)
        if kind != "MODIFIED" or key not in self.items:
            self.needs_reload = True
            return
        keep = self.items[key]
        item.leader_sts = item.leader_sts if item.leader_sts is not None else keep.leader_sts
        self.items[key] = item
        self.dirty.add(key)

    def flush(self) -> Patches:
        """Re-encode the dirty objects → the patch segments of one ``lwse_resident_tick``."""
        patches = Patches()
        patches._pending = {}
        for key in sorted(self.dirty):
            self._vacated_reqs = None
            self._vacated_pods = None
            self._write_object(key, self._encode_object(key), patches)
            if self._vacated_reqs is not None:
                base, cap, ns = self._vacated_reqs
                inert = R.aligned_empty(cap, R.PLACE_REQ)
                inert["leader_node"] = R.NONE
                inert["ns"] = ns
                cur = self.reqs[base: base + cap]
                diff = np.flatnonzero((np.ascontiguousarray(cur).view(np.uint8).reshape(cap, -1)
                                       != inert.view(np.uint8).reshape(cap, -1)).any(axis=1))
                if len(diff):
                    cur[diff] = inert[diff]
                    patches._pending.setdefault(R.TABLE_PLACE_REQS, ([], []))
                    patches._pending[R.TABLE_PLACE_REQS][0].extend((diff + base).tolist())
                    patches._pending[R.TABLE_PLACE_REQS][1].append(inert[diff].copy())
            if self._vacated_pods is not None:
                base, cap = self._vacated_pods
                for table_id, table in ((R.TABLE_POD_STATE, self.pod_state), (R.TABLE_POD_IDENT, self.pod_ident)):
                    cur = table[base: base + cap]
                    used = np.flatnonzero(np.ascontiguousarray(cur).view(np.uint8).reshape(cap, -1).any(axis=1))
                    if len(used):
                        zeros = R.aligned_empty(len(used), table.dtype)
                        cur[used] = zeros
                        patches._pending.setdefault(table_id, ([], []))
                        patches._pending[table_id][0].extend((used + base).tolist())
                        patches._pending[table_id][1].append(zeros)
        self.dirty.clear()
        for table_id in (R.TABLE_LWS, R.TABLE_GROUPS, R.TABLE_POD_STATE, R.TABLE_POD_IDENT, R.TABLE_PLACE_REQS):
            if table_id in patches._pending:
                rows, chunks = patches._pending[table_id]
                patches.add(table_id, rows, np.concatenate(chunks))
        del patches._pending
        return patches

    # ------------------------------------------------------------------ results
    def tables(self):
        """(lws, groups, pod_state, pod_ident, reqs) trimmed to the rows in use (+ spare already laid out)."""
        return (self.lws[: self.n_lws], self.groups[: self.g_end], self.pod_state[: self.p_end],
                self.pod_ident[: self.p_end], self.reqs[: self.r_end])

    def full_tables(self):
        """The whole allocation (what ``resident_load`` should take, so that relocations stay in range)."""
        return self.lws[: self.n_lws], self.groups, self.pod_state, self.pod_ident, self.reqs

    def group_row(self, namespace: str, name: str, group_index: int) -> int:
        return self.slots[(namespace, name)].group_base + group_index

    def lws_row(self, namespace: str, name: str) -> int:
        return self.slots[(namespace, name)].lws_row


# --------------------------------------------------------------------------- #
# DisaggregatedSet controller: For(DisaggregatedSet), Owns(LeaderWorkerSet)
# --------------------------------------------------------------------------- #
@dataclass
class DsSlots:
    ds_row: int
    role_base: int
    role_cap: int
    rev_base: int
    rev_cap: int


class DsIncrementalEncoder:
    """The DS tables of ``lwse_ds_resident_tick`` kept current from the DS controller's watches
    (disaggregatedset_controller.go:271-286: ``For(DisaggregatedSet)``, ``Owns(LeaderWorkerSet)``).

    Laid out like ``IncrementalEncoder``: every DS owns a slot of role rows and of (revision, role)
    rows with slack; ``flush()`` re-encodes the dirty DSes with ``encoder.encode_ds([item])`` and
    emits one patch segment per table holding the rows that differ (the DS row included, when
    ``n_roles`` / ``n_old_revs`` change); a DS that outgrows its slot moves to the spare rows at the
    end of the tables, and when those run out ``needs_reload`` is set.  A DS ADDED / DELETED event
    changes the DS table's shape: it sets ``needs_reload`` too.

    Creation-timestamp ranks are per DS here (each DS is encoded on its own), not global as in one
    ``encode_ds`` over every DS.  That is equivalent: ``sortByNewestTimestamp`` (executor.go:283-302)
    only compares the revisions of one DS, and a per-DS rank preserves their order and ties.
    """

    def __init__(self, items: list, spare: float = 0.25):
        self.items: dict[tuple, encoder.DsItem] = {(it.ds.namespace, it.ds.name): it for it in items}
        self.needs_reload = False
        self.dirty: set = set()
        keys = sorted(self.items)
        fresh = {k: encoder.encode_ds([self.items[k]]) for k in keys}
        self.slots: dict[tuple, DsSlots] = {}
        ro = rr = 0
        for i, k in enumerate(keys):
            t = fresh[k]
            rcap, vcap = _slack(len(t.roles)), _slack(len(t.revroles))
            self.slots[k] = DsSlots(i, ro, rcap, rr, vcap)
            ro, rr = ro + rcap, rr + vcap
        self.order = keys
        self.ds = R.aligned_empty(len(keys), R.DS_REC)
        self.roles = R.aligned_empty(ro + max(16, int(ro * spare)), R.DS_ROLE_REC)
        self.revroles = R.aligned_empty(rr + max(64, int(rr * spare)), R.DS_REVROLE_REC)
        self.role_end, self.rev_end = ro, rr
        self._names: dict[tuple, list] = {}
        self._old_revs: dict[tuple, list] = {}
        for k in keys:
            self._write(k, fresh[k], None)

    # ------------------------------------------------------------------ layout
    def _write(self, key, t: encoder.DsTablesHost, pending: Optional[dict]):
        sl = self.slots[key]
        if len(t.roles) > sl.role_cap or len(t.revroles) > sl.rev_cap:
            rcap, vcap = _slack(len(t.roles)), _slack(len(t.revroles))
            if self.role_end + rcap > len(self.roles) or self.rev_end + vcap > len(self.revroles):
                self.needs_reload = True
                return
            sl = self.slots[key] = DsSlots(sl.ds_row, self.role_end, rcap, self.rev_end, vcap)
            self.role_end, self.rev_end = self.role_end + rcap, self.rev_end + vcap
        self._names[key], self._old_revs[key] = t.role_names[0], t.old_revisions[0]
        row = t.ds.copy()
        row["role_base"], row["rev_base"] = sl.role_base, sl.rev_base
        for table_id, table, base, fresh_rows in ((R.TABLE_DS, self.ds, sl.ds_row, row),
                                                  (R.TABLE_DS_ROLES, self.roles, sl.role_base, t.roles),
                                                  (R.TABLE_DS_REVROLES, self.revroles, sl.rev_base, t.revroles)):
            n = len(fresh_rows)
            if n == 0:
                continue
            cur = table[base: base + n]
            if pending is None:
                cur[:] = fresh_rows
                continue
            a = np.ascontiguousarray(cur).view(np.uint8).reshape(n, -1)
            b = np.ascontiguousarray(fresh_rows).view(np.uint8).reshape(n, -1)
            diff = np.flatnonzero((a != b).any(axis=1))
            if len(diff):
                vals = R.aligned_empty(len(diff), table.dtype)
                vals[:] = fresh_rows[diff]
                cur[diff] = vals
                rows, chunks = pending.setdefault(table_id, ([], []))
                rows.extend((diff + base).tolist())
                chunks.append(vals)

    # ------------------------------------------------------------------ events
    def ds_event(self, kind: str, item: encoder.DsItem):
        """A watch event of the DisaggregatedSet informer.  MODIFIED (spec or target revision): the
        children stay those the child events delivered.  ADDED / DELETED: reload."""
        key = (item.ds.namespace, item.ds.name)
        if kind != "MODIFIED" or key not in self.items:
            self.needs_reload = True
            return
        self.items[key] = encoder.DsItem(item.ds, item.revision, self.items[key].children)
        self.dirty.add(key)

    def child_event(self, kind: str, ds_key: tuple, child: api.ChildLWS):
        """A watch event of an owned LeaderWorkerSet (ADDED | MODIFIED | DELETED): replicas,
        readyReplicas, annotations, or the child itself.  The List order (first seen) is kept."""
        it = self.items.get(ds_key)
        if it is None:
            return
        kids = it.children
        at = next((i for i, c in enumerate(kids) if c.role == child.role and c.revision == child.revision), None)
        if kind == "DELETED":
            if at is not None:
                kids.pop(at)
        elif at is None:
            kids.append(child)
        else:
            kids[at] = child
        self.dirty.add(ds_key)

    def flush(self) -> Patches:
        """Re-encode the dirty DSes → the patch segments of one ``lwse_ds_resident_tick``."""
        pending: dict = {}
        for key in sorted(self.dirty):
            self._write(key, encoder.encode_ds([self.items[key]]), pending)
        self.dirty.clear()
        patches = Patches()
        for table_id in (R.TABLE_DS, R.TABLE_DS_ROLES, R.TABLE_DS_REVROLES):
            if table_id in pending:
                rows, chunks = pending[table_id]
                patches.add(table_id, rows, np.concatenate(chunks))
        return patches

    # ------------------------------------------------------------------ results
    def full_tables(self):
        """(ds, roles, revroles): the whole allocation, spare rows included (what ``ds_resident_load``
        takes, so that relocations stay in range)."""
        return self.ds, self.roles, self.revroles

    def ds_row(self, key) -> int:
        return self.slots[key].ds_row

    def role_names(self, key) -> list:
        """allRoleNames of the DS: role i is row ``slots[key].role_base + i``."""
        return self._names[key]

    def old_revisions(self, key) -> list:
        """Old revisions in row order: revision r, role i is row ``rev_base + r * n_roles + i``; the
        target revision follows them (bit r of ``drained_revs`` / ``ready_revs`` is revision r)."""
        return self._old_revs[key]
