// Package lwse is the cgo binding of liblwse.so (include/lwse.h): the B200
// reconcile-and-placement engine behind the LeaderWorkerSet / DisaggregatedSet
// reconcilers.
//
// A SKETCH, NOT A BUILD ARTEFACT: this repository's image has no Go toolchain, so these two
// files (lwse.go, arena.go) have never been compiled.  They show the binding a maintainer adds
// to sigs.k8s.io/lws, kept next to the header it binds; what IS built and run here is the same
// calling pattern in C — C-malloc'd tables, several threads on one handle, the resident tick fed
// from the pinned arena — tests/host_c/cgo_pattern_check.c, driven by tests/test_cgo_pattern.py.
// Every exported function maps 1:1 to a C symbol; tables are passed as C-allocated
// (or pinned) memory because cgo forbids the C side to retain Go pointers.
package lwse

/*
#cgo CFLAGS: -I${SRCDIR}/../../include
#cgo LDFLAGS: -L${SRCDIR}/../../lws_b200 -llwse -Wl,-rpath,${SRCDIR}/../../lws_b200
#include <stdlib.h>
#include "lwse.h"
*/
import "C"

import (
	"fmt"
	"unsafe"
)

// Engine is one GPU's engine handle (lwse_create). One per device; a handle runs one
// sweep at a time.
type Engine struct{ h *C.lwse_engine }

// Error wraps a negative lwse_status.
type Error struct {
	Status int
	Cuda   int
}

func (e *Error) Error() string {
	return fmt.Sprintf("lwse: %s (status %d, cudaError %d)", C.GoString(C.lwse_strerror(C.int(e.Status))), e.Status, e.Cuda)
}

func (e *Engine) check(rc C.int) error {
	if rc == C.LWSE_OK {
		return nil
	}
	return &Error{Status: int(rc), Cuda: int(C.lwse_last_cuda_error(e.h))}
}

// New creates an engine on a CUDA device. There is no CPU fallback: without a usable
// sm_100 device this fails with LWSE_ERR_NO_DEVICE and the operator keeps its stock path.
func New(device int) (*Engine, error) {
	cfg := C.lwse_config{abi_version: C.LWSE_ABI_VERSION, device: C.int32_t(device)}
	var h *C.lwse_engine
	if rc := C.lwse_create(&cfg, &h); rc != C.LWSE_OK {
		return nil, &Error{Status: int(rc)}
	}
	return &Engine{h: h}, nil
}

func (e *Engine) Close() { C.lwse_destroy(e.h); e.h = nil }

// ShardOf: which of n engines owns an object (hash(LWS.UID) mod nGPU; DS-owned LWS pass
// the DS uid hash so a DS and its children co-reside).
func ShardOf(uidHash uint64, n uint32) uint32 { return uint32(C.lwse_shard_of(C.uint64_t(uidHash), C.uint32_t(n))) }

// Hash64 is the string hash of the encoders (revision keys, label values, UIDs).
func Hash64(s string) uint64 {
	if len(s) == 0 {
		return uint64(C.lwse_hash64(nil, 0))
	}
	b := []byte(s)
	return uint64(C.lwse_hash64(unsafe.Pointer(&b[0]), C.size_t(len(b))))
}

// Tables is a set of C-allocated record tables (see Arena in arena.go).
type LwsTables struct {
	Lws      *C.lwse_lws_rec
	NLws     uint32
	Groups   *C.lwse_group_rec
	NGroups  uint32
	PodState *C.lwse_pod_state
	PodIdent *C.lwse_pod_ident
	NPods    uint64
	LwsOut   *C.lwse_lws_out
	GroupOut *C.lwse_group_out
	Occ      *C.uint32_t // optional
	Flags    uint32
}

func (t *LwsTables) c() C.lwse_lws_tables {
	return C.lwse_lws_tables{
		lws: t.Lws, n_lws: C.uint32_t(t.NLws), groups: t.Groups, n_groups: C.uint32_t(t.NGroups),
		pod_state: t.PodState, pod_ident: t.PodIdent, n_pods: C.uint64_t(t.NPods),
		lws_out: t.LwsOut, group_out: t.GroupOut, node_occupancy: t.Occ, flags: C.uint32_t(t.Flags),
	}
}

// UploadNodes makes the node table resident (call on Node add/update/delete batches).
func (e *Engine) UploadNodes(nodes *C.lwse_node_rec, n, nDomains uint32) error {
	return e.check(C.lwse_upload_nodes(e.h, nodes, C.uint32_t(n), C.uint32_t(nDomains)))
}

// SweepLws: host tables in, host result tables out (H2D, two or three kernels, D2H, sync).  With
// pinned, mapped tables the 16-byte pod identity column is not uploaded: a prefetch kernel copies
// just the rows of pods with a restart / deletion event while the other tables cross PCIe.
func (e *Engine) SweepLws(t *LwsTables) error {
	ct := t.c()
	return e.check(C.lwse_sweep_lws_host(e.h, &ct))
}

// Place runs one placement round over host request rows.
func (e *Engine) Place(reqs *C.lwse_place_req, n uint32, occupancy *C.uint32_t, nNamespaces uint32, out *C.lwse_place_out) (rounds uint32, err error) {
	var r C.uint32_t
	err = e.check(C.lwse_place_host(e.h, reqs, C.uint32_t(n), occupancy, C.uint32_t(nNamespaces), out, &r))
	return uint32(r), err
}

// SweepDs advances every DisaggregatedSet by one reconcile.
func (e *Engine) SweepDs(t *C.lwse_ds_tables) error { return e.check(C.lwse_sweep_ds_host(e.h, t)) }

// DsResidentLoad copies the three DisaggregatedSet input tables to the device, where they stay
// (their own buffers: SweepDs and the LWS resident tables never touch them).  Committed results
// start at zero; the next DsTick lists every owned row.
func (e *Engine) DsResidentLoad(t *C.lwse_ds_tables) error { return e.check(C.lwse_ds_resident_load(e.h, t)) }

// DsTickResult: views of engine-owned pinned memory, valid until the next resident call.
type DsTickResult struct {
	DsRows      []uint32
	DsOut       []C.lwse_ds_out
	RoleRows    []uint32
	RoleOut     []C.lwse_ds_role_out
	RevroleRows []uint32
	RevroleOut  []C.lwse_ds_revrole_out
}

// DsTick is one pass of the DS controller's work queue (lwse_ds_resident_tick): the patch segments
// (tables LWSE_TABLE_DS .. LWSE_TABLE_DS_REVROLES, ideally in the arena) in, the listed rows out —
// the DS keys that need work with their current ds_out, and their role / (revision, role) rows
// whose decision changed.  Still uncompiled, like the rest of this file.
func (e *Engine) DsTick(segs []C.lwse_patch_seg) (DsTickResult, error) {
	var t C.lwse_ds_tick
	if len(segs) > 0 {
		t.segs = &segs[0]
		t.n_segs = C.uint32_t(len(segs))
	}
	if err := e.check(C.lwse_ds_resident_tick(e.h, &t)); err != nil {
		return DsTickResult{}, err
	}
	return DsTickResult{
		DsRows:      unsafe.Slice((*uint32)(unsafe.Pointer(t.ds_rows)), int(t.n_ds)),
		DsOut:       unsafe.Slice(t.ds_out, int(t.n_ds)),
		RoleRows:    unsafe.Slice((*uint32)(unsafe.Pointer(t.role_rows)), int(t.n_roles)),
		RoleOut:     unsafe.Slice(t.role_out, int(t.n_roles)),
		RevroleRows: unsafe.Slice((*uint32)(unsafe.Pointer(t.revrole_rows)), int(t.n_revroles)),
		RevroleOut:  unsafe.Slice(t.revrole_out, int(t.n_revroles)),
	}, nil
}

// JointSubmit enqueues one pass of both controllers (lwse_joint_tick_submit): the LWS part as Submit
// (lwsSegs / flags; hasLws = false for a DS-only tick) and the DS
// part as DsTick, one scatter, one publish.  It shares the two-slot ring of Submit; JointWait takes the
// oldest tick of either kind (an LWS-only tick reports no DS rows).  The patch bytes of a submitted tick
// stay untouched until its JointWait returned.  Uncompiled, like the rest of this file.
func (e *Engine) JointSubmit(hasLws bool, lwsSegs []C.lwse_patch_seg, flags uint32, dsSegs []C.lwse_patch_seg) error {
	var t C.lwse_tick
	var d C.lwse_ds_tick
	if len(lwsSegs) > 0 {
		t.segs = (*C.lwse_patch_seg)(unsafe.Pointer(&lwsSegs[0]))
		t.n_segs = C.uint32_t(len(lwsSegs))
	}
	t.flags = C.uint32_t(flags)
	if len(dsSegs) > 0 {
		d.segs = &dsSegs[0]
		d.n_segs = C.uint32_t(len(dsSegs))
	}
	tp := &t
	if !hasLws {
		tp = nil
	}
	return e.check(C.lwse_joint_tick_submit(e.h, tp, &d))
}

// JointWait blocks for the oldest tick in flight → both controllers' listed rows (views valid until
// the second submit after this call).
func (e *Engine) JointWait() (TickResult, DsTickResult, error) {
	var t C.lwse_tick
	var d C.lwse_ds_tick
	if err := e.check(C.lwse_joint_tick_wait(e.h, &t, &d)); err != nil {
		return TickResult{}, DsTickResult{}, err
	}
	return tickResult(&t), DsTickResult{
		DsRows:      unsafe.Slice((*uint32)(unsafe.Pointer(d.ds_rows)), int(d.n_ds)),
		DsOut:       unsafe.Slice(d.ds_out, int(d.n_ds)),
		RoleRows:    unsafe.Slice((*uint32)(unsafe.Pointer(d.role_rows)), int(d.n_roles)),
		RoleOut:     unsafe.Slice(d.role_out, int(d.n_roles)),
		RevroleRows: unsafe.Slice((*uint32)(unsafe.Pointer(d.revrole_rows)), int(d.n_revroles)),
		RevroleOut:  unsafe.Slice(d.revrole_out, int(d.n_revroles)),
	}, nil
}

// DsResidentOutputs copies every committed DS result row into the caller's tables (nil skips one).
func (e *Engine) DsResidentOutputs(ds *C.lwse_ds_out, roles *C.lwse_ds_role_out, revroles *C.lwse_ds_revrole_out) error {
	return e.check(C.lwse_ds_resident_outputs(e.h, ds, roles, revroles))
}

// GroupKeys computes SHA-1 digests (20 bytes each) of n strings laid out CSR-style.
func (e *Engine) GroupKeys(bytes *C.uint8_t, offsets *C.uint32_t, n uint32, digests *C.uint8_t) error {
	return e.check(C.lwse_group_keys_host(e.h, bytes, offsets, C.uint32_t(n), digests))
}

// --- incremental form: tables resident on the device, fed from watch events -----------------

// ResidentLoad copies the four input tables to the device, where they stay.
func (e *Engine) ResidentLoad(t *LwsTables) error {
	ct := t.c()
	return e.check(C.lwse_resident_load(e.h, &ct))
}

// ResidentPatch overwrites n rows of one resident table (rows[i] <- i-th packed row of values):
// what an informer delta (pod phase change, sts status update, spec edit) turns into.
func (e *Engine) ResidentPatch(which C.lwse_table, rows *C.uint32_t, values unsafe.Pointer, n uint32) error {
	return e.check(C.lwse_resident_patch(e.h, which, rows, values, C.uint32_t(n)))
}

// ResidentSweep sweeps the resident tables and returns only the result rows that changed since
// the previous sweep — the objects whose Reconcile() has something to do.
func (e *Engine) ResidentSweep(flags uint32, ch *C.lwse_changes) error {
	return e.check(C.lwse_resident_sweep(e.h, C.uint32_t(flags), ch))
}

// --- device-pointer form: one reconcile tick (sweep + placement round, concurrently) --------

// ReconcileDevice enqueues one tick on stream (nil = the engine's stream); no synchronize.
func (e *Engine) ReconcileDevice(t *LwsTables, reqs *C.lwse_place_req, n uint32, occupancy *C.uint32_t,
	nNamespaces uint32, placeOut *C.lwse_place_out, stream unsafe.Pointer) error {
	ct := t.c()
	return e.check(C.lwse_reconcile_device(e.h, &ct, reqs, C.uint32_t(n), occupancy, C.uint32_t(nNamespaces), placeOut, stream))
}

// --- one operator replica per GPU of a node: placement parts exchanged over NVLink -----------

// ExchangeCreate allocates this replica's exchange buffer and returns its 64-byte IPC handle;
// the replicas swap handles (any transport) and each calls ExchangeConnect with all of them.
func (e *Engine) ExchangeCreate(reqsPerPart, world, rank uint32) ([64]byte, error) {
	var h [64]byte
	err := e.check(C.lwse_exchange_create(e.h, C.uint32_t(reqsPerPart), C.uint32_t(world), C.uint32_t(rank), unsafe.Pointer(&h[0])))
	return h, err
}

func (e *Engine) ExchangeConnect(handles []byte) error {
	return e.check(C.lwse_exchange_connect(e.h, unsafe.Pointer(&handles[0])))
}

// ReconcileExchangedDevice: a tick of one shard; localPart = [occupancy | request rows] in device memory.
func (e *Engine) ReconcileExchangedDevice(t *LwsTables, localPart unsafe.Pointer, nNamespaces uint32,
	placeOut *C.lwse_place_out, stream unsafe.Pointer) error {
	ct := t.c()
	return e.check(C.lwse_reconcile_exchanged_device(e.h, &ct, localPart, C.uint32_t(nNamespaces), placeOut, stream))
}
