// LWS sweep kernels (sm_100a).  One sweep = two launches on one stream when groups are small —
// group_fused_kernel (the pod scan and the group pass of 256 consecutive groups in one CTA,
// bitmaps in shared memory) and lws_sweep_kernel — and three otherwise:
//
//   pod_scan_kernel<U>   pod-centric streaming pass over the 1-BYTE pod state column: every
//                        lane takes U x 16 pods with coalesced 128-bit loads (all U loads in
//                        flight before the first use), derives "Pending" (pod_controller.go:356)
//                        and "has a restart or deletion event" (pod_utils.go:29-50) for 4 pods
//                        per 32-bit SWAR step and packs them into two bitmaps (1 bit / pod).
//   group_sweep_kernel   one lane (or W-lane tile) per pod group.  Reads its 64-byte group row,
//                        the first 16 bytes of its owner row and the bitmap words of its pod
//                        range; only pods whose event bit is set are visited individually
//                        (state byte + 16-byte identity row: workerPodBelongsToLeader,
//                        pod_controller.go:268-295).  Emits the restart verdict
//                        (pod_controller.go:204-266), the leader pod's worker-sts gating
//                        (:100-198), and the per-replica state bits
//                        (leaderworkerset_controller.go:608-638, :433-476) — the latter also as
//                        one BYTE per group in a dense column for the LWS pass.
//   lws_sweep_kernel<W>  one lane (W lanes for objects with hundreds of groups) per
//                        LeaderWorkerSet over its groups' flag bytes, 8 groups per 64-bit SWAR
//                        step: counters are popcounts of masked byte lanes, the partition walk
//                        (:643-673) is three such reductions.  32 B out per object.
//
// All of them are integer/compare kernels bound by HBM traffic (DESIGN.md).
#include <cstdlib>
#include <cstring>

#include "lwse_device.cuh"

namespace lwse {

// --------------------------------------------------------------------------
// pod scan
// --------------------------------------------------------------------------
struct PodScanArgs {
  const uint8_t* state;
  uint32_t* pending_bits;  // ceil(n_pods / 32) words
  uint32_t* event_bits;
  uint64_t n_pods;
  uint32_t* event_count;  // nullable: += pods with an event bit (the host entry point sizes its
                          // identity-column transfer with it)
};

__device__ __forceinline__ bool pod_has_event(uint32_t bits) {
  const uint32_t phase = bits & LWSE_POD_PHASE_MASK;
  // ContainerRestarted (pod_utils.go:29-45) || PodDeleted (:48)
  return ((phase - 1u) < 2u && (bits & LWSE_POD_ANY_RESTART)) || (bits & LWSE_POD_DELETING);
}

// SWAR over the 16 pods of one 128-bit load: every byte is one pod's state (phase bits 0-1,
// any-restart bit 2, deleting bit 3).  Both predicates are evaluated on four bytes at once and
// the four bit-0s are gathered into a nibble with one multiply; 16 bits per predicate per lane.
__device__ __forceinline__ void pod16_predicates(const uint4 v, uint32_t& pend16, uint32_t& ev16) {
  const uint32_t x[4] = {v.x, v.y, v.z, v.w};
  pend16 = 0;
  ev16 = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t X = x[k], y = X >> 1, z = X >> 2, w3 = X >> 3;
    const uint32_t P = X & ~y & 0x01010101u;                // phase == Pending (bit0 ∧ ¬bit1)
    const uint32_t E = (((X ^ y) & z) | w3) & 0x01010101u;  // (phase ∈ {Pending,Running} ∧ restart) ∨ deleting
    pend16 |= ((P * 0x10204080u) >> 28) << (4 * k);
    ev16 |= ((E * 0x10204080u) >> 28) << (4 * k);
  }
}

// Two neighbouring lanes hold the 32 pods of one bitmap word: one shuffle moves both predicate
// halves; the even lane ends up with the two words.
__device__ __forceinline__ void pair_words(uint32_t pend16, uint32_t ev16, uint32_t& wp, uint32_t& we) {
  const uint32_t mine = pend16 | (ev16 << 16);
  const uint32_t other = __shfl_xor_sync(0xFFFFFFFFu, mine, 1);
  wp = (mine & 0xFFFFu) | (other << 16);
  we = (mine >> 16) | (other & 0xFFFF0000u);
}

// 16 state bytes at pod index idx (idx % 16 == 0); bytes past the end of the column read as 0
__device__ __forceinline__ uint4 load_pods16(const uint8_t* state, uint64_t idx, uint64_t n_pods) {
  if (idx + 15u < n_pods) return ldg_stream(state + idx);
  uint32_t w[4] = {0, 0, 0, 0};
  for (uint32_t k = 0; k < 16u; k++)
    if (idx + k < n_pods) w[k >> 2] |= (uint32_t)__ldg(state + idx + k) << (8u * (k & 3u));
  return make_uint4(w[0], w[1], w[2], w[3]);
}

template <int U>
__global__ void __launch_bounds__(256) pod_scan_kernel(const PodScanArgs a) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warp = (uint64_t)blockIdx.x * 8u + (threadIdx.x >> 5);
  const uint64_t n_warps = (uint64_t)gridDim.x * 8u;
  const uint64_t n_words = (a.n_pods + 31u) >> 5;
  constexpr uint64_t kPodsPerChunk = 512ull * U;  // 32 lanes x 16 pods x U
  pdl_launch_dependents();
  bool waited = false;
  uint32_t events = 0;
  for (uint64_t base = warp * kPodsPerChunk; base < a.n_pods; base += n_warps * kPodsPerChunk) {
    uint4 v[U];
#pragma unroll
    for (int j = 0; j < U; j++) {  // all U 128-bit loads in flight before the first use
      const uint64_t idx = base + (uint64_t)j * 512u + lane * 16u;
      v[j] = idx < a.n_pods ? load_pods16(a.state, idx, a.n_pods) : make_uint4(0, 0, 0, 0);
    }
    if (!waited) {  // the bitmaps (and counters) may still be read by the previous sweep's group pass
      pdl_wait_prior();
      waited = true;
    }
#pragma unroll
    for (int j = 0; j < U; j++) {
      uint32_t pend, ev, wp, we;
      pod16_predicates(v[j], pend, ev);
      pair_words(pend, ev, wp, we);
      const uint64_t w = ((base + (uint64_t)j * 512u) >> 5) + (lane >> 1);
      if ((lane & 1u) == 0u && w < n_words) {
        a.pending_bits[w] = wp;
        a.event_bits[w] = we;
        events += __popc(we);
      }
    }
  }
  if (a.event_count != nullptr) {
    events = __reduce_add_sync(0xFFFFFFFFu, events);
    if (lane == 0 && events) atomicAdd(a.event_count, events);
  }
}

// Scheduled pods per node (the placement occupancy): the node binding lives in the cold identity
// rows, so this optional count reads that column (16 B / pod).  The resident engine counts once
// at load and then follows the identity-row patches (scatter kernel below).
__global__ void __launch_bounds__(256) pod_occupancy_kernel(const lwse_pod_ident* __restrict__ ident, uint64_t n_pods,
                                                            uint32_t* __restrict__ occupancy, uint32_t n_nodes) {
  for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pods; p += (uint64_t)gridDim.x * blockDim.x) {
    const uint4 r = ldg_stream(ident + p);
    if (r.w & LWSE_PODID_SCHEDULED) {
      const uint32_t node = r.w >> LWSE_PODID_NODE_SHIFT;
      if (node < n_nodes) atomicAdd(occupancy + node, 1u);
    }
  }
}

// The host entry point with a pinned, mapped identity column: only pods with an event bit ever
// need their identity row.  This kernel streams the (already uploaded) state bytes and copies
// exactly those rows host -> device, on a side stream, WHILE the group and LWS tables are still
// crossing PCIe — the latency-bound gather hides behind the bandwidth-bound copies.
__global__ void __launch_bounds__(256) ident_prefetch_kernel(const uint8_t* __restrict__ state, uint64_t n_pods,
                                                             const lwse_pod_ident* __restrict__ host_ident,
                                                             lwse_pod_ident* __restrict__ dev_ident) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warp = (uint64_t)blockIdx.x * 8u + (threadIdx.x >> 5), n_warps = (uint64_t)gridDim.x * 8u;
  for (uint64_t base = warp * 512u; base < n_pods; base += n_warps * 512u) {
    const uint64_t idx = base + lane * 16u;
    if (idx >= n_pods) continue;
    uint32_t pend, ev;
    pod16_predicates(load_pods16(state, idx, n_pods), pend, ev);
    while (ev) {
      const uint64_t p = idx + (__ffs(ev) - 1u);
      ev &= ev - 1u;
      if (p < n_pods) stg_stream(dev_ident + p, ldg_stream(host_ident + p));
    }
  }
}

int launch_ident_prefetch(const uint8_t* d_state, uint64_t n_pods, const lwse_pod_ident* mapped_host_ident,
                          lwse_pod_ident* d_ident, int sm_count, cudaStream_t s, int* cuda_err) {
  *cuda_err = 0;
  if (n_pods == 0) return 0;
  const uint64_t want = (n_pods + 4095u) / 4096u;
  const uint32_t cap = (uint32_t)sm_count * 8u;
  ident_prefetch_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, s>>>(d_state, n_pods, mapped_host_ident, d_ident);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

// --------------------------------------------------------------------------
// group pass
// --------------------------------------------------------------------------
// Optional change list: result rows that differ from what the output table held before.  The
// lists live in device memory; a tick's publish kernel moves them to the host in one coalesced
// pass (a system-scope fence per changed row — the first version wrote rows straight into mapped
// host memory — cost 20 us per thousand rows).
struct ChangeList {
  uint32_t* rows;   // nullptr = off
  void* outs;       // packed result rows
  uint32_t* count;  // device counter
  uint32_t capacity;
};

template <int N>  // N = uint4 per result row
__device__ __forceinline__ void emit_if_changed(const ChangeList& c, uint4* slot, uint32_t row, const uint4 (&v)[N]) {
  if (c.rows != nullptr) {
    bool diff = false;
#pragma unroll
    for (int k = 0; k < N; k++) {
      const uint4 old = __ldcg(slot + k);
      diff |= old.x != v[k].x || old.y != v[k].y || old.z != v[k].z || old.w != v[k].w;
    }
    if (diff) {
      const uint32_t i = atomicAdd(c.count, 1u);
      if (i < c.capacity) {
        c.rows[i] = row;
#pragma unroll
        for (int k = 0; k < N; k++) reinterpret_cast<uint4*>(c.outs)[(size_t)i * N + k] = v[k];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < N; k++) stg_stream(slot + k, v[k]);
}

constexpr uint32_t kSweepWaitAtTop = 1u << 31;  // internal bit of GroupSweepArgs::sweep_flags

struct GroupSweepArgs {
  const lwse_lws_rec* lws;
  const lwse_group_rec* groups;
  const uint8_t* pod_state;
  const lwse_pod_ident* pod_ident;
  const uint32_t* pending_bits;
  const uint32_t* event_bits;
  const lwse_node_rec* nodes;
  lwse_group_out* out;
  uint8_t* gflag8;  // dense column: the low 5 bits of out.flags, one byte per group (for the LWS pass)
  uint64_t n_pods;
  uint32_t n_lws;
  uint32_t n_groups;
  uint32_t n_nodes;
  uint32_t sweep_flags;
  ChangeList changes;
  uint32_t* event_count;  // nullable (fused kernel): += (group, event pod) pairs visited — sizes the host
                          // entry point's identity-column transfer of the NEXT call
};

// bits [lo, hi) of a 32-bit word, 0 <= lo <= hi <= 32
__device__ __forceinline__ uint32_t bit_range(uint32_t lo, uint32_t hi) {
  const uint32_t upto_hi = hi >= 32u ? 0xFFFFFFFFu : ((1u << hi) - 1u);
  return upto_hi & ~((1u << lo) - 1u) & (lo >= 32u ? 0u : 0xFFFFFFFFu);
}

// Where a group's bitmap words come from: the scan kernel's global bitmaps (written by the
// previous kernel of the same sweep: read through L2, never the non-coherent path), or the
// shared-memory window of the fused kernel.
struct GlobalBits {
  const uint32_t* pending_bits;
  const uint32_t* event_bits;
  __device__ __forceinline__ uint32_t pending(uint32_t w) const { return __ldcg(pending_bits + w); }
  __device__ __forceinline__ uint32_t event(uint32_t w) const { return __ldcg(event_bits + w); }
};

// What deciding one event pod needs from its group (pod_controller.go:233-257).
struct VisitCtx {
  uint32_t rev_lo, rev_hi;  // leader pod's revision hash
  uint32_t leader_uid, wsts_uid;
  uint32_t pod_base;
  uint32_t bits;  // kLeaderFound | kChainOk | kLeaderDeleting
};
constexpr uint32_t kLeaderFound = 1u, kChainOk = 2u, kLeaderDeleting = 4u;
constexpr uint32_t kAccLeaderCand = 0x80000000u;

// handleRestartPolicy (:204-266) for ONE pod that has a restart / deletion event, policy checks
// already done: returns the verdict bits it contributes; *cand = it would recreate the group.
__device__ __forceinline__ uint32_t visit_pod(const VisitCtx& c, uint32_t state, const uint4 id, bool& cand) {
  uint32_t acc = 0;
  bool deleting;
  if (state & LWSE_POD_IS_LEADER) {
    cand = true;  // leader = pod (:251)
    deleting = state & LWSE_POD_DELETING;
    acc |= kAccLeaderCand;
  } else if (!(id.w & LWSE_PODID_NAME_OK)) {
    cand = false;
    return LWSE_GOUT_RESTART_ERROR;  // :230
  } else {
    const uint32_t kind = (state & LWSE_POD_OWNER_MASK) >> LWSE_POD_OWNER_SHIFT;
    // workerPodBelongsToLeader :268-295
    const bool belongs = (state & LWSE_POD_OWNER_NAME_MATCH) &&
                         ((kind == 1u && id.z == c.leader_uid) || (kind == 2u && id.z == c.wsts_uid && (c.bits & kChainOk)));
    cand = (c.bits & kLeaderFound) && id.x == c.rev_lo && id.y == c.rev_hi && belongs;  // :233, :239
    deleting = c.bits & kLeaderDeleting;
  }
  if (!cand) return 0;
  return acc | (deleting ? LWSE_GOUT_LEADER_DELETING : LWSE_GOUT_DELETE_LEADER);  // :255 / :259
}

// First part of the group pass for group g (row ca..cd, first 16 bytes of its owner L):
// pendingPodsInGroup (:338-362) from the pending bitmap and the decision whether the group's
// event pods have to be visited at all.
struct GroupPre {
  uint32_t oflags;
  uint32_t w_first, w_last, pod_end;
  bool visit;  // tile-uniform
  VisitCtx ctx;
};

template <int W, class Bits>
__device__ __forceinline__ GroupPre group_pre(const Bits& bits, uint32_t lane, const uint4 ca, const uint4 cb,
                                              const uint4 cc, const uint4 cd, const uint4 L) {
  GroupPre r;
  const uint32_t pod_base = cc.z, pod_count = cc.w, gflags = cd.y;
  const int32_t size = (int32_t)L.z;
  const uint32_t lflags = L.w;
  const uint32_t policy = (lflags & LWSE_LWS_RESTART_MASK) >> LWSE_LWS_RESTART_SHIFT;
  const bool policy_on = policy == LWSE_RESTART_ON_POD_RESTART || policy == LWSE_RESTART_AFTER_START;
  r.oflags = 0;
  r.pod_end = pod_base + pod_count;  // <= n_pods < 2^32 (checked by the entry points)
  r.w_first = pod_base >> 5;
  r.w_last = pod_count ? ((r.pod_end - 1u) >> 5) : r.w_first;
  uint32_t any_bits = 0;  // bit0 pending, bit1 event
  if (pod_count) {
    for (uint32_t w = r.w_first + lane; w <= r.w_last; w += W) {
      const uint32_t lo = w == r.w_first ? (pod_base & 31u) : 0u;
      const uint32_t hi = w == r.w_last ? (((r.pod_end - 1u) & 31u) + 1u) : 32u;
      const uint32_t m = bit_range(lo, hi);
      if (bits.pending(w) & m) any_bits |= 1u;
      if (bits.event(w) & m) any_bits |= 2u;
    }
  }
  any_bits = tile_or<W>(any_bits);
  const bool pending = (uint32_t)size != pod_count || (any_bits & 1u);
  if (pending) r.oflags |= LWSE_GOUT_PENDING;
  // :222 skip when pending ∧ (AfterStart ∨ annotation)
  const bool suppressed =
      pending && (policy == LWSE_RESTART_AFTER_START || (lflags & LWSE_LWS_RECREATE_AFTER_START_ANNOT));
  r.visit = (any_bits & 2u) && policy_on && !suppressed;
  constexpr uint32_t kChain = LWSE_GRP_WSTS_FOUND | LWSE_GRP_WSTS_OWNER_IS_POD | LWSE_GRP_WSTS_OWNER_NAME_MATCH;
  r.ctx.rev_lo = ca.x;
  r.ctx.rev_hi = ca.y;
  r.ctx.leader_uid = cb.z;
  r.ctx.wsts_uid = cb.w;
  r.ctx.pod_base = pod_base;
  r.ctx.bits = 0;
  if ((gflags & (LWSE_GRP_POD_PRESENT | LWSE_GRP_POD_NAME_MATCH)) == (LWSE_GRP_POD_PRESENT | LWSE_GRP_POD_NAME_MATCH))
    r.ctx.bits |= kLeaderFound;  // :233
  if ((gflags & kChain) == kChain && cc.x == cb.z) r.ctx.bits |= kChainOk;  // sts owner uid == leader uid
  if (gflags & LWSE_GRP_POD_DELETING) r.ctx.bits |= kLeaderDeleting;
  return r;
}

// The event pods of one group visited by the group's own lanes: collected four at a time so
// that their state and identity loads are all in flight together.
template <int W, class Bits>
__device__ __forceinline__ void group_visit_inline(const GroupSweepArgs& a, const Bits& bits, uint32_t lane,
                                                   const GroupPre& pre, uint32_t& acc_out, uint32_t& first_out) {
  uint32_t acc = 0, first = LWSE_NONE;
  auto visit = [&](const uint32_t* ev, int cnt) {
    uint32_t st[4];
    uint4 id[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (k < cnt) {
        st[k] = __ldg(a.pod_state + ev[k]);
        id[k] = ldg_cached(a.pod_ident + ev[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (k < cnt) {
        bool cand;
        acc |= visit_pod(pre.ctx, st[k], id[k], cand);
        if (cand) first = min(first, ev[k] - pre.ctx.pod_base);
      }
    }
  };
  uint32_t ev[4];
  int cnt = 0;
  for (uint32_t w = pre.w_first + lane; w <= pre.w_last; w += W) {
    const uint32_t lo = w == pre.w_first ? (pre.ctx.pod_base & 31u) : 0u;
    const uint32_t hi = w == pre.w_last ? (((pre.pod_end - 1u) & 31u) + 1u) : 32u;
    uint32_t m = bits.event(w) & bit_range(lo, hi);
    while (m) {
      const uint32_t p = (w << 5) + (__ffs(m) - 1u);
      m &= m - 1u;
      // fixed-slot insert keeps ev[] in registers
      if (cnt == 0) ev[0] = p;
      else if (cnt == 1) ev[1] = p;
      else if (cnt == 2) ev[2] = p;
      else ev[3] = p;
      if (++cnt == 4) {
        visit(ev, 4);
        cnt = 0;
      }
    }
  }
  if (cnt) visit(ev, cnt);
  acc_out = tile_or<W>(acc);
  first_out = tile_min<W>(first);
}

// Last part: the per-replica state bits, the leader pod's own Reconcile tail
// (pod_controller.go:95-198) and the 16-byte result row.
__device__ __forceinline__ uint4 group_finish(const GroupSweepArgs& a, const uint4 ca, const uint4 cb, const uint4 cc,
                                              const uint4 cd, const uint4 L, uint32_t oflags, uint32_t acc,
                                              uint32_t first_out) {
  const uint32_t gflags = cd.y;
  const int32_t size = (int32_t)L.z;
  const uint32_t lflags = L.w;
  uint32_t domain = LWSE_NONE;
  int32_t worker_replicas = 0;
  const bool leader_deleted = acc & kAccLeaderCand;
  oflags |= acc & ~kAccLeaderCand;

  // ---- per-replica state bits (consumed by lws_sweep_kernel) ----
  const bool no_wsts = size == 1;
  const uint64_t rev = u64_of(L.x, L.y);
  const bool leader_updated = u64_of(ca.x, ca.y) == rev;
  const bool wsts_updated = u64_of(ca.z, ca.w) == rev;
  const bool leader_ready = (gflags & (LWSE_GRP_POD_RUNNING | LWSE_GRP_POD_READY)) ==
                            (LWSE_GRP_POD_RUNNING | LWSE_GRP_POD_READY);  // PodRunningAndReady
  const bool wsts_ready = cb.x == cb.y && (gflags & LWSE_GRP_WSTS_REV_SETTLED);  // StatefulsetReady
  const bool ready = leader_ready && (no_wsts || wsts_ready);
  const bool updated = leader_updated && (no_wsts || wsts_updated);
  // getReplicaStates :609-617 — names decide whether the slot is live
  const bool named = (gflags & LWSE_GRP_POD_NAME_MATCH) && (no_wsts || (gflags & LWSE_GRP_WSTS_LABEL_NAME_MATCH));
  if (named && ready) oflags |= LWSE_GOUT_STATE_READY;
  if (named && updated) oflags |= LWSE_GOUT_STATE_UPDATED;
  // updateConditions :433-476 — existing leader pods whose worker sts is found
  const bool counted = (gflags & LWSE_GRP_POD_PRESENT) && (no_wsts || (gflags & LWSE_GRP_WSTS_FOUND));
  if (counted) {
    oflags |= LWSE_GOUT_COUNTED;
    if (ready) oflags |= LWSE_GOUT_COND_READY;
    if (updated) oflags |= LWSE_GOUT_COND_UPDATED;
  }

  // ---- the leader pod's own Reconcile tail, pod_controller.go:95-198 ----
  bool go_on = (gflags & LWSE_GRP_POD_PRESENT) && !leader_deleted &&
               !(gflags & (LWSE_GRP_MISTAKEN_ANNOTATION | LWSE_GRP_POD_DELETING));
  if (go_on) {
    if (a.sweep_flags & LWSE_SWEEP_GANG) oflags |= LWSE_GOUT_CREATE_PODGROUP;  // :130
    go_on = !no_wsts &&                                                          // :138
            !((lflags & LWSE_LWS_STARTUP_LEADER_READY) && !(gflags & LWSE_GRP_POD_READY));  // :143
  }
  if (go_on && !(gflags & LWSE_GRP_REVISION_EXISTS)) {  // :152
    oflags |= LWSE_GOUT_REQUEUE_REVISION;
    go_on = false;
  }
  if (go_on && (lflags & LWSE_LWS_EXCLUSIVE_TOPOLOGY)) {  // :162
    const uint32_t node = cc.y;
    if (node == LWSE_NONE) {  // :164
      oflags |= LWSE_GOUT_WAIT_SCHEDULE;
      go_on = false;
    } else if (node != LWSE_NODE_NOT_FOUND && node < a.n_nodes) {
      const uint4 nr = ldg_cached(reinterpret_cast<const uint4*>(a.nodes + node));
      const uint32_t nflags = nr.w >> 16;
      if (!(nflags & LWSE_NODE_HAS_TOPOLOGY)) {  // :330
        oflags |= LWSE_GOUT_TOPOLOGY_ERROR;
        go_on = false;
      } else {
        domain = nr.z;
      }
    }  // Node NotFound → empty value, nil error (:327)
  }
  if (go_on && !(gflags & LWSE_GRP_WSTS_FOUND)) {  // :188-192
    oflags |= LWSE_GOUT_CREATE_WSTS;
    worker_replicas = size - 1;  // :437; ordinals start at 1 (:440)
  }
  return make_uint4(oflags, first_out, (uint32_t)worker_replicas, domain);
}

__device__ __forceinline__ uint4 bad_group_row() { return make_uint4(LWSE_GOUT_BAD_TABLE, LWSE_NONE, 0u, LWSE_NONE); }
constexpr uint32_t kFlagByteMask = LWSE_GOUT_STATE_READY | LWSE_GOUT_STATE_UPDATED | LWSE_GOUT_COUNTED |
                                   LWSE_GOUT_COND_READY | LWSE_GOUT_COND_UPDATED;
static_assert(kFlagByteMask == 0x1Fu, "the LWS pass reads the low five bits of group_out.flags as one byte");

// 128-thread CTAs capped at 64 registers: a tick's placement round holds part of the register
// file of some SMs while this kernel runs, and the groups of a 100k-group table should still
// fit in one wave next to it.
constexpr uint32_t kGroupThreads = 128;
template <int W>
__global__ void __launch_bounds__(kGroupThreads, 8) group_sweep_kernel(const GroupSweepArgs a) {
  constexpr uint32_t kTilesPerBlock = kGroupThreads / W;
  const uint32_t lane = threadIdx.x & (W - 1);
  const uint32_t stride = gridDim.x * kTilesPerBlock;
  const GlobalBits bits{a.pending_bits, a.event_bits};
  pdl_launch_dependents();
  bool waited = false;
  for (uint32_t g = blockIdx.x * kTilesPerBlock + threadIdx.x / W; g < a.n_groups; g += stride) {
    const uint4* row = reinterpret_cast<const uint4*>(a.groups + g);
    const uint4 ca = ldg_cached(row + 0), cb = ldg_cached(row + 1), cc = ldg_cached(row + 2),
                cd = ldg_cached(row + 3);
    const uint32_t pod_base = cc.z, pod_count = cc.w, lws_index = cd.x;
    const bool bad = lws_index >= a.n_lws || (uint64_t)pod_base + pod_count > a.n_pods;
    // owner row: only its first 16 bytes (rev_hash, size, flags)
    uint4 L = make_uint4(0, 0, 0, 0);
    if (!bad) L = ldg_cached(reinterpret_cast<const uint4*>(a.lws + lws_index));
    if (!waited) {  // everything above is input; the scan's bitmaps and group_out come next
      pdl_wait_prior();
      waited = true;
    }
    uint4 v[1] = {bad_group_row()};
    if (!bad) {
      const GroupPre pre = group_pre<W>(bits, lane, ca, cb, cc, cd, L);
      uint32_t acc = 0, first = LWSE_NONE;
      if (pre.visit) group_visit_inline<W>(a, bits, lane, pre, acc, first);
      v[0] = group_finish(a, ca, cb, cc, cd, L, pre.oflags, acc, first);
    }
    if (lane == 0) {
      emit_if_changed<1>(a.changes, reinterpret_cast<uint4*>(a.out + g), g, v);
      a.gflag8[g] = (uint8_t)(v[0].x & kFlagByteMask);
    }
  }
}

// --------------------------------------------------------------------------
// fused pod scan + group pass
// --------------------------------------------------------------------------
// One CTA per 256 consecutive groups, one thread per group.
//   1. rows: the CTA loads its 256 group rows and the first 16 B of their owners, and reduces the
//      union of their pod ranges to a window of bitmap words (contiguous for tables the encoder
//      lays out: pods of group g right after those of g-1);
//   2. scan: the window's state BYTES are streamed with coalesced 128-bit loads (16 pods each,
//      4 in flight per lane) and the two predicate bitmaps are packed into SHARED memory;
//   3. pre: every thread derives pendingPodsInGroup of its group and counts the event pods it
//      has to visit (policy on, not suppressed);
//   4. visit, event-centric: the (group, pod) pairs of the whole CTA are compacted into shared
//      memory and taken by all 256 threads, one pair each — every identity-row load of the CTA
//      is in flight at once instead of per-group batches of four behind divergent loops; verdicts
//      meet in shared memory (atomicOr / atomicMin per group);
//   5. finish: state bits, worker-sts gating, one 16-byte store and one flag byte per group.
// Used when groups are small (the window of 256 groups fits 65 536 pods).  A window that does
// not fit (irregular tables: ranges far apart) falls back to deriving each bitmap word from the
// state column directly, and more pairs than the shared list holds to the per-group visit —
// slow, still exact.
constexpr uint32_t kFusedThreads = 256;
constexpr uint32_t kWinWords = 2048;  // 65 536 pods per CTA: 2 x 8 KB of shared memory
constexpr uint32_t kPairCap = 1280;   // (group, event pod) pairs visited cooperatively per CTA

struct WindowBits {
  const uint32_t* pend;  // word (w - w0)
  const uint32_t* ev;
  uint32_t w0;
  __device__ __forceinline__ uint32_t pending(uint32_t w) const { return pend[w - w0]; }
  __device__ __forceinline__ uint32_t event(uint32_t w) const { return ev[w - w0]; }
};

struct DirectBits {
  const uint8_t* state;
  uint64_t n_pods;
  __device__ __forceinline__ void word(uint32_t w, uint32_t& pend, uint32_t& ev) const {
    pend = ev = 0;
    for (uint32_t k = 0; k < 32u; k++) {
      const uint64_t p = ((uint64_t)w << 5) + k;
      if (p >= n_pods) break;
      const uint32_t b = __ldg(state + p);
      if ((b & LWSE_POD_PHASE_MASK) == LWSE_POD_PHASE_PENDING) pend |= 1u << k;
      if (pod_has_event(b)) ev |= 1u << k;
    }
  }
  __device__ __forceinline__ uint32_t pending(uint32_t w) const {
    uint32_t p, e;
    word(w, p, e);
    return p;
  }
  __device__ __forceinline__ uint32_t event(uint32_t w) const {
    uint32_t p, e;
    word(w, p, e);
    return e;
  }
};

#ifdef LWSE_FUSED_MAXNREG  // build-time experiment switch, see lwse_place_ns_kernels.cu
#define LWSE_FUSED_BOUNDS __maxnreg__(LWSE_FUSED_MAXNREG)
#else
#define LWSE_FUSED_BOUNDS __launch_bounds__(kFusedThreads, 3)
#endif
__global__ void LWSE_FUSED_BOUNDS group_fused_kernel(const GroupSweepArgs a) {
  __shared__ uint32_t s_pend[kWinWords], s_ev[kWinWords];
  __shared__ uint32_t s_pair[kPairCap];  // tid << 16 | pod index relative to the window start
  __shared__ uint4 s_ctx4[kFusedThreads];
  __shared__ uint2 s_ctx2[kFusedThreads];
  __shared__ uint32_t s_acc[kFusedThreads], s_first[kFusedThreads];
  __shared__ uint32_t s_lo[kFusedThreads / 32], s_hi[kFusedThreads / 32], s_cnt[kFusedThreads / 32];
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t g = blockIdx.x * kFusedThreads + tid;
  const bool valid = g < a.n_groups;
  // Behind a kernel that WRITES the input tables (a tick's patch scatter) the kernel is launched
  // programmatically dependent all the same — the launch latency overlaps the scatter — and waits
  // here, before its first read.  Its own dependent (the LWS pass reads LWS rows BEFORE its wait) may
  // only be released after that: it must not start while the scatter still writes.
  if (a.sweep_flags & kSweepWaitAtTop) pdl_wait_prior();
  pdl_launch_dependents();

  // ---- 1. rows ----
  uint4 ca = make_uint4(0, 0, 0, 0), cb = ca, cc = ca, cd = ca, L = ca;
  bool bad = true;
  if (valid) {
    const uint4* row = reinterpret_cast<const uint4*>(a.groups + g);
    ca = ldg_cached(row + 0), cb = ldg_cached(row + 1), cc = ldg_cached(row + 2), cd = ldg_cached(row + 3);
    bad = cd.x >= a.n_lws || (uint64_t)cc.z + cc.w > a.n_pods;
    if (!bad) L = ldg_cached(reinterpret_cast<const uint4*>(a.lws + cd.x));  // first 16 bytes of the owner row
  }
  // the CTA's window of bitmap words
  const bool has_pods = valid && !bad && cc.w != 0u;
  uint32_t lo = has_pods ? (cc.z >> 5) : 0xFFFFFFFFu;
  uint32_t hi = has_pods ? (((cc.z + cc.w - 1u) >> 5) + 1u) : 0u;
  lo = __reduce_min_sync(0xFFFFFFFFu, lo);
  hi = __reduce_max_sync(0xFFFFFFFFu, hi);
  if (lane == 0) {
    s_lo[warp] = lo;
    s_hi[warp] = hi;
  }
  __syncthreads();
  lo = s_lo[0], hi = s_hi[0];
#pragma unroll
  for (int k = 1; k < (int)(kFusedThreads / 32); k++) {
    lo = min(lo, s_lo[k]);
    hi = max(hi, s_hi[k]);
  }
  lo &= ~3u;  // 128-byte aligned window start: the scan's 128-bit loads stay aligned
  const uint32_t n_words = hi > lo ? hi - lo : 0u;
  const bool windowed = n_words <= kWinWords;  // CTA-uniform

  // ---- 2. scan ----
  if (windowed && n_words) {
    // 512 pods (16 bitmap words) per warp and chunk, U chunks in flight per warp
    constexpr int U = 4;
    const uint32_t n_chunks = (n_words + 15u) >> 4;
    for (uint32_t c0 = warp * U; c0 < n_chunks; c0 += (kFusedThreads / 32) * U) {
      uint4 v[U];
#pragma unroll
      for (int j = 0; j < U; j++) {
        const uint32_t c = c0 + (uint32_t)j;
        const uint64_t idx = ((uint64_t)lo << 5) + (uint64_t)c * 512u + lane * 16u;
        v[j] = (c < n_chunks && idx < a.n_pods) ? load_pods16(a.pod_state, idx, a.n_pods) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int j = 0; j < U; j++) {
        uint32_t pend, ev, wp, we;
        pod16_predicates(v[j], pend, ev);
        pair_words(pend, ev, wp, we);
        const uint32_t w = (c0 + (uint32_t)j) * 16u + (lane >> 1);
        if ((lane & 1u) == 0u && w < n_words) {
          s_pend[w] = wp;
          s_ev[w] = we;
        }
      }
    }
  }
  __syncthreads();

  uint4 v[1] = {bad_group_row()};
  if (windowed) {
    // ---- 3. pre ----
    const WindowBits bits{s_pend, s_ev, lo};
    GroupPre pre{};
    uint32_t my_pairs = 0;
    if (!bad) {
      pre = group_pre<1>(bits, 0u, ca, cb, cc, cd, L);
      if (pre.visit) {
        for (uint32_t w = pre.w_first; w <= pre.w_last; w++) {
          const uint32_t blo = w == pre.w_first ? (cc.z & 31u) : 0u;
          const uint32_t bhi = w == pre.w_last ? (((pre.pod_end - 1u) & 31u) + 1u) : 32u;
          my_pairs += __popc(bits.event(w) & bit_range(blo, bhi));
        }
      }
    }
    // exclusive scan of the pair counts over the CTA
    uint32_t incl = my_pairs;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, incl, off);
      if ((int)lane >= off) incl += up;
    }
    if (lane == 31u) s_cnt[warp] = incl;
    s_acc[tid] = 0u;
    s_first[tid] = LWSE_NONE;
    __syncthreads();
    uint32_t warp_base = 0, total = 0;
#pragma unroll
    for (int k = 0; k < (int)(kFusedThreads / 32); k++) {
      const uint32_t c = s_cnt[k];
      if (k < (int)warp) warp_base += c;
      total += c;
    }
    if (a.event_count != nullptr && tid == 0 && total) atomicAdd(a.event_count, total);
    uint32_t acc = 0, first = LWSE_NONE;
    if (total <= kPairCap) {  // CTA-uniform
      // ---- 4. visit, event-centric ----
      if (total) {
        if (my_pairs) {
          uint32_t at = warp_base + incl - my_pairs;
          for (uint32_t w = pre.w_first; w <= pre.w_last; w++) {
            const uint32_t blo = w == pre.w_first ? (cc.z & 31u) : 0u;
            const uint32_t bhi = w == pre.w_last ? (((pre.pod_end - 1u) & 31u) + 1u) : 32u;
            uint32_t m = bits.event(w) & bit_range(blo, bhi);
            while (m) {
              const uint32_t rel = ((w - lo) << 5) + (__ffs(m) - 1u);  // < 65 536
              m &= m - 1u;
              s_pair[at++] = (tid << 16) | rel;
            }
          }
          s_ctx4[tid] = make_uint4(pre.ctx.rev_lo, pre.ctx.rev_hi, pre.ctx.leader_uid, pre.ctx.wsts_uid);
          s_ctx2[tid] = make_uint2(pre.ctx.pod_base, pre.ctx.bits);
        }
        __syncthreads();
        for (uint32_t e = tid; e < total; e += kFusedThreads) {
          const uint32_t pr = s_pair[e], t = pr >> 16;
          const uint32_t p = (lo << 5) + (pr & 0xFFFFu);
          const uint32_t st = __ldg(a.pod_state + p);       // the SM loaded this line a moment ago
          const uint4 id = ldg_stream(a.pod_ident + p);     // the CTA's only gathers
          const uint4 c4 = s_ctx4[t];
          const uint2 c2 = s_ctx2[t];
          const VisitCtx ctx{c4.x, c4.y, c4.z, c4.w, c2.x, c2.y};
          bool cand;
          const uint32_t bitsv = visit_pod(ctx, st, id, cand);
          if (bitsv) atomicOr(&s_acc[t], bitsv);
          if (cand) atomicMin(&s_first[t], p - c2.x);
        }
        __syncthreads();
        acc = s_acc[tid];
        first = s_first[tid];
      }
    } else if (pre.visit) {
      group_visit_inline<1>(a, bits, 0u, pre, acc, first);
    }
    // ---- 5. finish ----
    if (!bad) v[0] = group_finish(a, ca, cb, cc, cd, L, pre.oflags, acc, first);
  } else if (!bad) {
    const DirectBits bits{a.pod_state, a.n_pods};
    const GroupPre pre = group_pre<1>(bits, 0u, ca, cb, cc, cd, L);
    uint32_t acc = 0, first = LWSE_NONE;
    if (pre.visit) group_visit_inline<1>(a, bits, 0u, pre, acc, first);
    v[0] = group_finish(a, ca, cb, cc, cd, L, pre.oflags, acc, first);
  }
  pdl_wait_prior();  // group_out / the flag column may still be read by the previous sweep's LWS pass
  if (valid) {
    emit_if_changed<1>(a.changes, reinterpret_cast<uint4*>(a.out + g), g, v);
    a.gflag8[g] = (uint8_t)(v[0].x & kFlagByteMask);
  }
}

// --------------------------------------------------------------------------
// LWS-level pass
// --------------------------------------------------------------------------
struct LwsSweepArgs {
  const lwse_lws_rec* lws;
  const uint8_t* gflag8;  // one flag byte per group (written by the group pass)
  lwse_lws_out* out;
  uint32_t n_lws;
  uint32_t n_groups;
  uint32_t sweep_flags;
  ChangeList changes;
};

__device__ __forceinline__ int32_t want_replicas(int32_t lws_replicas, int32_t surge, int32_t mu,
                                                 int32_t unready, int32_t sts_replicas,
                                                 uint32_t& event) {
  // calculateRollingUpdateReplicas :685-696
  int32_t fin;
  if (unready <= surge) {
    fin = lws_replicas + max(0, unready - mu);
  } else {
    fin = lws_replicas + surge;
  }
  if (fin == sts_replicas - 1)  // :313
    event = LWSE_EVENT_DELETE_ONE;
  else if (fin < sts_replicas)  // :315
    event = LWSE_EVENT_DELETE_RANGE;
  return fin;
}

// Byte-lane masks of one 64-bit word of the flag column.  Byte b of word j is group slot
// idx = off + b of the object (off = 8 j - group_base, negative in the object's first word).
constexpr uint64_t kLaneOnes = 0x0101010101010101ull;
__device__ __forceinline__ uint64_t lanes_upto(int64_t n) {  // bit 0 of bytes [0, n)
  if (n <= 0) return 0ull;
  if (n >= 8) return kLaneOnes;
  return kLaneOnes & ((1ull << (8 * (int)n)) - 1ull);
}
__device__ __forceinline__ uint64_t lanes_idx_range(int32_t off, int32_t lo, int32_t hi) {  // lo <= idx < hi
  return lanes_upto((int64_t)hi - off) & ~lanes_upto((int64_t)lo - off);
}
__device__ __forceinline__ int32_t highest_lane(uint64_t m) { return (63 - __clzll((long long)m)) >> 3; }  // m != 0

template <int W>
__global__ void __launch_bounds__(256) lws_sweep_kernel(const LwsSweepArgs a) {
  constexpr uint32_t kTilesPerBlock = 256 / W;
  const uint32_t lane = threadIdx.x & (W - 1);
  const uint32_t n_tiles = gridDim.x * kTilesPerBlock;
  const uint64_t* words = reinterpret_cast<const uint64_t*>(a.gflag8);
  pdl_launch_dependents();
  bool waited = false;
  for (uint32_t i = blockIdx.x * kTilesPerBlock + threadIdx.x / W; i < a.n_lws; i += n_tiles) {
    const uint4* row = reinterpret_cast<const uint4*>(a.lws + i);
    const uint4 r0 = ldg_stream(row + 0), r1 = ldg_stream(row + 1), r2 = ldg_stream(row + 2),
                r3 = ldg_stream(row + 3);
    if (!waited) {  // the object rows are input; the group pass's flag bytes come next
      pdl_wait_prior();
      waited = true;
    }
    const int32_t size = (int32_t)r0.z;
    const uint32_t lflags = r0.w;
    const int32_t R = (int32_t)r1.x, P = (int32_t)r1.y;
    const int32_t n = (int32_t)r2.x;  // sts replicas
    const int32_t cur_partition = (int32_t)r2.y, annot = (int32_t)r2.z;
    const uint32_t gbase = r3.z, gc = r3.w;

    uint32_t oflags = 0, event = LWSE_EVENT_NONE;
    int32_t o_partition = 0, o_replicas = 0, o_mu = 0, o_ready = 0, o_updated = 0, o_unready = 0,
            o_min_member = 0;

    if ((uint64_t)gbase + gc > a.n_groups) {
      oflags = LWSE_LOUT_BAD_TABLE;
    } else {
      const bool sts_exists = lflags & LWSE_LWS_STS_EXISTS;
      const bool intstr_bad = lflags & LWSE_LWS_INTSTR_INVALID;
      int32_t mu = scaled_value((int32_t)r1.w, lflags & LWSE_LWS_UNAVAIL_IS_PERCENT, R, false);
      int32_t surge = scaled_value((int32_t)r1.z, lflags & LWSE_LWS_SURGE_IS_PERCENT, R, true);
      if (surge > R) surge = R;  // :307
      const int32_t burst = R + surge;
      const int32_t gcs = (int32_t)min(gc, 0x7FFFFFFFu);
      const uint32_t j0 = gbase >> 3, j1 = gc ? ((gbase + gc - 1u) >> 3) : j0;  // words of the object's flag bytes

      // ---- pass A: counters over every group slot of the object ----
      // updateConditions counters (:450-475) and, for slots below the leader
      // sts's replica count, the getReplicaStates view.
      int32_t c_ready = 0, c_updated = 0, c_cur_nb = 0, c_upd_nb = 0, c_ready_nb = 0, c_upd_rdy = 0;
      int32_t c_ok_below_R = 0;  // slots < min(R, n) that are ready ∧ updated
      int32_t max_bad = -1;      // highest slot < n that is not (ready ∧ updated)
      const int32_t n_live = min(n, gcs);
      if (gc) {
        for (uint32_t j = j0 + lane; j <= j1; j += W) {
          const uint64_t w = __ldcg(words + j);
          const int32_t off = (int32_t)(j << 3) - (int32_t)gbase;  // |off| < 2^31: n_groups < 2^31 in practice
          const uint64_t valid = lanes_idx_range(off, 0, gcs);
          const uint64_t st_rd = w & kLaneOnes, st_up = (w >> 1) & kLaneOnes;
          const uint64_t cnt = (w >> 2) & valid, rd = (w >> 3) & kLaneOnes, up = (w >> 4) & kLaneOnes;
          const uint64_t in_R = lanes_idx_range(off, 0, R), in_nb = lanes_idx_range(off, P, R);
          c_ready += __popcll(cnt & rd);
          c_updated += __popcll(cnt & up);
          c_cur_nb += __popcll(cnt & in_nb);
          c_upd_nb += __popcll(cnt & in_nb & up);
          c_ready_nb += __popcll(cnt & in_R & rd);
          c_upd_rdy += __popcll(cnt & in_nb & rd & up);
          const uint64_t live = valid & lanes_idx_range(off, 0, n_live), ok = st_rd & st_up;
          c_ok_below_R += __popcll(ok & live & in_R);
          const uint64_t badm = live & ~ok;
          if (badm) max_bad = off + highest_lane(badm);  // j ascends per lane
        }
      }
      c_ready = tile_add<W>(c_ready);
      c_updated = tile_add<W>(c_updated);
      c_cur_nb = tile_add<W>(c_cur_nb);
      c_upd_nb = tile_add<W>(c_upd_nb);
      c_ready_nb = tile_add<W>(c_ready_nb);
      c_upd_rdy = tile_add<W>(c_upd_rdy);
      c_ok_below_R = tile_add<W>(c_ok_below_R);
      max_bad = tile_max<W>(max_bad);
      if (n > n_live) max_bad = n - 1;  // slots without any object are zero-valued states

      // ---- status / conditions (:478-501) ----
      if (lflags & LWSE_LWS_GROUP_LABEL_INVALID) {
        oflags |= LWSE_LOUT_STATUS_ERROR;  // :434-437
      } else {
        o_ready = c_ready;
        o_updated = c_updated;
        uint32_t cond;
        if (c_upd_nb < c_cur_nb)
          cond = LWSE_COND_UPDATE_IN_PROGRESS;
        else if (c_ready_nb == R && c_upd_rdy == c_cur_nb)
          cond = LWSE_COND_AVAILABLE;
        else
          cond = LWSE_COND_PROGRESSING;
        oflags |= cond << LWSE_LOUT_COND_SHIFT;
        if (P == 0 && c_upd_rdy == R) oflags |= LWSE_LOUT_UPDATE_DONE;
      }

      // ---- rollingUpdateParameters (:280-373) ----
      bool err = false;
      if (!sts_exists) {  // Case 1
        o_partition = 0;
        o_replicas = R;
      } else if (intstr_bad) {
        err = true;
      } else if (lflags & LWSE_LWS_UPDATED) {  // Case 2
        o_partition = min(R, n);
        o_replicas = n < R ? R : want_replicas(R, surge, mu, R, n, event);
      } else if (cur_partition == 0 && n == R) {  // Case 3
        o_partition = 0;
        o_replicas = R;
      } else if (n < R) {
        o_partition = cur_partition;
        o_replicas = R;
      } else {
        // calculateLWSUnreadyReplicas :675-683 (R >= 0 here because n >= R is not implied; clamp)
        const int32_t unready = max(R, 0) - c_ok_below_R;
        o_unready = unready;
        if (!(lflags & LWSE_LWS_ANNOT_VALID)) {
          err = true;  // :351-354
        } else if (annot != R) {  // Case 4
          o_partition = min(cur_partition, burst);
          o_replicas = want_replicas(R, surge, mu, unready, n, event);
        } else {  // Case 5
          const int32_t step = mu + surge - (burst - n);  // :366-369
          // rollingUpdatePartition :643-673
          const int32_t cont_ready = n - 1 - max_bad;  // calculateContinuousReadyReplicas
          const int32_t rsp = max(0, n - cont_ready - step);
          // pass B: unavailable = #{idx < rsp : !ready}
          int32_t unavail = 0;
          const int32_t rsp_live = min(rsp, n_live);
          if (rsp_live > 0) {
            const uint32_t jb = (gbase + (uint32_t)rsp_live - 1u) >> 3;
            for (uint32_t j = j0 + lane; j <= jb; j += W) {
              const int32_t off = (int32_t)(j << 3) - (int32_t)gbase;
              unavail += __popcll(~__ldcg(words + j) & lanes_idx_range(off, 0, rsp_live));
            }
          }
          unavail = tile_add<W>(unavail) + (rsp - rsp_live);
          int32_t part = rsp + unavail;
          const int32_t hi = min(part, n - 1);
          if (hi >= rsp) {
            // pass C: the walk stops at the highest idx in [rsp, hi] that is ready ∧ ¬updated
            int32_t blocker = -1;
            const int32_t hi_live = min(hi, n_live - 1);
            if (hi_live >= rsp) {
              const uint32_t ja = (gbase + (uint32_t)rsp) >> 3, jb = (gbase + (uint32_t)hi_live) >> 3;
              for (uint32_t j = ja + lane; j <= jb; j += W) {
                const uint64_t w = __ldcg(words + j);
                const int32_t off = (int32_t)(j << 3) - (int32_t)gbase;
                const uint64_t m = w & ~(w >> 1) & lanes_idx_range(off, rsp, hi_live + 1);
                if (m) blocker = off + highest_lane(m);
              }
            }
            blocker = tile_max<W>(blocker);
            if (blocker < 0)
              part = rsp;
            else if (blocker < hi)
              part = blocker + 1;
            // blocker == hi: the first probe breaks, partition keeps rsp + unavail
          }
          o_partition = min(part, cur_partition);
          o_replicas = want_replicas(R, surge, mu, unready, n, event);
        }
      }
      if (err) {
        oflags |= LWSE_LOUT_RUP_ERROR;
        o_partition = 0;
        o_replicas = 0;
        event = LWSE_EVENT_NONE;
      }
      o_partition = max(o_partition, P);  // deferred clamp :285-288
      oflags |= event << LWSE_LOUT_EVENT_SHIFT;

      // stsMaxUnavailable :811-830
      if (!intstr_bad) o_mu = max(1, mu + surge);
      // PodGroup MinMember, volcano_provider.go:72,81-83
      if (a.sweep_flags & LWSE_SWEEP_GANG)
        o_min_member = (lflags & LWSE_LWS_STARTUP_LEADER_READY) ? 1 : size;
      if (lflags & LWSE_LWS_IRREGULAR) oflags |= LWSE_LOUT_IRREGULAR;
    }
    if (lane == 0) {
      const uint4 v[2] = {make_uint4((uint32_t)o_partition, (uint32_t)o_replicas, (uint32_t)o_mu, (uint32_t)o_ready),
                          make_uint4((uint32_t)o_updated, (uint32_t)o_min_member, oflags, (uint32_t)o_unready)};
      emit_if_changed<2>(a.changes, reinterpret_cast<uint4*>(a.out + i), i, v);
    }
  }
}

// --------------------------------------------------------------------------
// launchers
// --------------------------------------------------------------------------
// LWSE_NO_PDL=1 turns programmatic dependent launch off (A/B measurements).
static const bool g_pdl = [] {
  const char* v = getenv("LWSE_NO_PDL");
  return !(v && v[0] == '1');
}();

static int pick_tile(uint64_t items, uint64_t owners) {
  // Lanes per object: a lane handles 8 groups per 64-bit word, and every lane of a tile runs the
  // object-level logic (the five cases, the walk) itself — one lane per object until objects
  // average more than 64 groups, then next power of two >= avg / 64, in [1, 32].
  static const uint64_t div = [] {
    const char* v = getenv("LWSE_LWS_TILE_DIV");
    const int d = v ? atoi(v) : 64;
    return (uint64_t)(d < 1 ? 1 : d);
  }();
  if (owners == 0) return 1;
  const uint64_t avg = ((items + owners - 1) / owners + div - 1) / div;
  int w = 1;
  while (w < 32 && (uint64_t)w < avg) w <<= 1;
  return w;
}

// Persistent-style grids: as many CTAs as are resident at once (SM count x
// occupancy), each thread/tile striding over its share of the rows.
template <typename K>
static uint32_t resident_ctas(K kernel, int sm_count) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1)
    per_sm = 4;
  return (uint32_t)sm_count * (uint32_t)per_sm;
}

template <int W>
static cudaError_t launch_group(const GroupSweepArgs& a, int sm_count, cudaStream_t s) {
  constexpr uint32_t kTilesPerBlock = kGroupThreads / W;
  (void)sm_count;
  const uint32_t want = (a.n_groups + kTilesPerBlock - 1) / kTilesPerBlock;
  return launch_pdl(group_sweep_kernel<W>, dim3(want < (1u << 20) ? want : (1u << 20)), dim3(kGroupThreads), 0, s,
                    g_pdl, a);
}

template <int W>
static cudaError_t launch_lws(const LwsSweepArgs& a, int sm_count, cudaStream_t s) {
  constexpr uint32_t kTilesPerBlock = 256 / W;
  static uint32_t resident = 0;
  if (resident == 0) resident = resident_ctas(lws_sweep_kernel<W>, sm_count);
  const uint32_t want = (a.n_lws + kTilesPerBlock - 1) / kTilesPerBlock;
  return launch_pdl(lws_sweep_kernel<W>, dim3(want < resident ? want : resident), dim3(256), 0, s, g_pdl, a);
}

constexpr int kScanUnroll = 4;  // 128-bit loads per lane per chunk: 4 x 512 B = 2 KB in flight per warp

// scratch: [pending bitmap | event bitmap | flag bytes (one per group, padded to 8)]
static uint64_t bitmap_words(uint64_t n_pods) { return ((n_pods + 31u) / 32u + 31u) & ~(uint64_t)31u; }
size_t lws_sweep_scratch_bytes(uint64_t n_pods, uint32_t n_groups) {
  return (size_t)(2 * bitmap_words(n_pods) * sizeof(uint32_t) + (((uint64_t)n_groups + 7u) & ~7ull) + 256);
}

// Returns the number of kernels launched (>=0) or -1 with *cuda_err set.
// scratch: lws_sweep_scratch_bytes(n_pods, n_groups) bytes of device memory.
struct SweepChangeLists {  // device (or mapped host) pointers; all null = off
  uint32_t* lws_rows = nullptr;
  lwse_lws_out* lws_out = nullptr;
  uint32_t lws_capacity = 0;
  uint32_t* group_rows = nullptr;
  lwse_group_out* group_out = nullptr;
  uint32_t group_capacity = 0;
  uint32_t* counts = nullptr;  // device: [0] lws, [1] groups; zeroed by the caller (a tick's publish kernel resets them)
};

// first_pdl: the sweep's first kernel may start before the previous kernel on the stream has
// finished (it reads only input tables before its griddepcontrol.wait) — false when that previous
// kernel WRITES the input tables (the patch scatter of a tick).
int launch_lws_sweep(const lwse_lws_tables* t, const lwse_node_rec* d_nodes, uint32_t n_nodes,
                     void* scratch, int sm_count, cudaStream_t s, int* cuda_err, const SweepChangeLists* cl,
                     uint32_t* d_event_count, int first_mode) {
  // first_mode — how the sweep's FIRST kernel is launched:
  //   0  an ordinary launch (its predecessor is a copy, a memset, an event: nothing to overlap with)
  //   1  programmatically dependent, input tables read before griddepcontrol.wait (the predecessor
  //      kernel does not write them)
  //   2  programmatically dependent, waits at its top (the predecessor kernel — a tick's patch
  //      scatter — WRITES the input tables)
  const bool first_pdl = first_mode == 1;
  *cuda_err = 0;
  int launches = 0;
  cudaError_t e = cudaSuccess;
  const uint64_t words = bitmap_words(t->n_pods);
  uint32_t* pending_bits = static_cast<uint32_t*>(scratch);
  uint32_t* event_bits = pending_bits + words;
  uint8_t* gflag8 = reinterpret_cast<uint8_t*>(event_bits + words);
  const bool group_pass = t->n_groups && !(t->flags & LWSE_SWEEP_SKIP_GROUP_PASS);

  // lanes per group: one per bitmap word of an average group, in {1, 2, 4, 8}
  const uint64_t avg_pods = t->n_groups ? (t->n_pods + t->n_groups - 1) / t->n_groups : 0;
  const int w = avg_pods > 2048 ? 8 : avg_pods > 1024 ? 4 : avg_pods > 512 ? 2 : 1;
  static const bool no_fuse = [] {
    const char* v = getenv("LWSE_NO_FUSE");
    return v && atoi(v) != 0;
  }();
  // scan + group pass in one kernel: mid-sized groups, both passes wanted.  Upper bound: the pod
  // window of 256 consecutive groups has to fit the CTA's bitmap window of 65 536 pods.  Lower bound:
  // with a handful of pods per group a CTA of 256 groups streams only 2-4 KB of state and the
  // kernel is all per-group work — on C5 (1.65 M groups x 8 pods) the fused kernel measured 86 us
  // against 4.7 + 47.8 us for the scan and the group pass as two kernels.
  static const uint64_t fuse_min_pods = [] {
    const char* v = getenv("LWSE_FUSE_MIN_PODS");
    return v ? (uint64_t)atol(v) : (uint64_t)16;
  }();
  const bool fused = group_pass && avg_pods <= 256 && avg_pods >= fuse_min_pods && !no_fuse && !(t->flags & LWSE_SWEEP_SKIP_POD_SCAN);
  if (t->node_occupancy && n_nodes && !(t->flags & LWSE_SWEEP_SKIP_POD_SCAN)) {
    e = cudaMemsetAsync(t->node_occupancy, 0, (size_t)n_nodes * sizeof(uint32_t), s);
    if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
    if (t->n_pods) {
      const uint64_t want = (t->n_pods + 255) / 256;
      const uint32_t cap = (uint32_t)sm_count * 16u;
      pod_occupancy_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, s>>>(t->pod_ident, t->n_pods, t->node_occupancy, n_nodes);
      e = cudaGetLastError();
      if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
      launches++;
    }
  }
  if (fused) {
    GroupSweepArgs a{t->lws,   t->groups, t->pod_state, t->pod_ident, nullptr, nullptr, d_nodes,
                     t->group_out, gflag8, t->n_pods, t->n_lws, t->n_groups, n_nodes, t->flags, ChangeList{}, d_event_count};
    if (cl && cl->group_rows) a.changes = ChangeList{cl->group_rows, cl->group_out, cl->counts + 1, cl->group_capacity};
    const uint32_t grid = (t->n_groups + kFusedThreads - 1) / kFusedThreads;
    // (a memset / occupancy kernel right before: an ordinary launch orders behind it)
    const bool pdl = g_pdl && !t->node_occupancy && first_mode != 0;
    if (pdl && first_mode == 2) a.sweep_flags |= kSweepWaitAtTop;
    e = launch_pdl(group_fused_kernel, dim3(grid), dim3(kFusedThreads), 0, s, pdl, a);
    if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
    launches++;
  }
  if (!fused && t->n_pods && t->n_groups && !(t->flags & LWSE_SWEEP_SKIP_POD_SCAN)) {
    PodScanArgs a{t->pod_state, pending_bits, event_bits, t->n_pods, d_event_count};
    // one chunk per warp: the kernel is a few microseconds long, so let the
    // hardware CTA scheduler balance it instead of a persistent grid-stride loop
    const uint64_t chunks = (t->n_pods + 512ull * kScanUnroll - 1) / (512ull * kScanUnroll);
    const uint64_t want = (chunks + 7) / 8;
    const uint32_t grid = (uint32_t)(want < (1u << 20) ? want : (1u << 20));
    e = launch_pdl(pod_scan_kernel<kScanUnroll>, dim3(grid), dim3(256), 0, s, g_pdl && first_pdl && !t->node_occupancy && !d_event_count, a);
    if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
    launches++;
  }
  if (group_pass && !fused) {
    GroupSweepArgs a{t->lws,   t->groups, t->pod_state, t->pod_ident, pending_bits, event_bits, d_nodes,
                     t->group_out, gflag8, t->n_pods, t->n_lws, t->n_groups, n_nodes, t->flags, ChangeList{}, nullptr};
    if (cl && cl->group_rows) a.changes = ChangeList{cl->group_rows, cl->group_out, cl->counts + 1, cl->group_capacity};
    switch (w) {
      case 8: e = launch_group<8>(a, sm_count, s); break;
      case 4: e = launch_group<4>(a, sm_count, s); break;
      case 2: e = launch_group<2>(a, sm_count, s); break;
      default: e = launch_group<1>(a, sm_count, s); break;
    }
    if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
    launches++;
  }
  if (t->n_lws && !(t->flags & LWSE_SWEEP_SKIP_LWS_PASS)) {
    LwsSweepArgs a{t->lws, gflag8, t->lws_out, t->n_lws, t->n_groups, t->flags, ChangeList{}};
    if (cl && cl->lws_rows) a.changes = ChangeList{cl->lws_rows, cl->lws_out, cl->counts + 0, cl->lws_capacity};
    switch (pick_tile(t->n_groups, t->n_lws)) {
      case 1: e = launch_lws<1>(a, sm_count, s); break;
      case 2: e = launch_lws<2>(a, sm_count, s); break;
      case 4: e = launch_lws<4>(a, sm_count, s); break;
      case 8: e = launch_lws<8>(a, sm_count, s); break;
      case 16: e = launch_lws<16>(a, sm_count, s); break;
      default: e = launch_lws<32>(a, sm_count, s); break;
    }
    if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
    launches++;
  }
  return launches;
}

// --------------------------------------------------------------------------
// tick: change lists to the host
// --------------------------------------------------------------------------
// The last kernel of a tick (lwse_resident_tick).  The sweep / placement kernels appended the
// changed rows to device-memory lists; this kernel copies the used part of up to three lists (six for
// a joint LWS + DS tick) into pinned, mapped host memory with coalesced stores and then raises the
// sequence word the host spins on — no stream synchronize, no copy-engine launch on the critical path.
// Ordering: a system-scope fence costs microseconds and fences from many threads queue up behind
// each other (one per writing thread measured 15-25 us for this kernel), so there is exactly ONE.
// Usual case, one CTA: bar.sync, then thread 0 writes the counts, fences at system scope (cumulative:
// it covers what happens-before it, the other threads' stores included) and stores the word.
// Several CTAs (many changed rows): every CTA orders its stores with bar.sync + a gpu-scope fence
// before it takes a ticket, the last CTA acquires with a gpu-scope fence and does the same.
struct PublishList {
  const uint32_t* src_rows;
  const uint4* src_outs;
  uint32_t* dst_rows;   // mapped host
  uint4* dst_outs;      // mapped host
  uint32_t* count;      // device counter (reset here); null = list not in this tick
  uint32_t capacity;
  uint32_t out_vec;     // uint4 per result row (rows of 16-byte multiples), else 0
  uint32_t out_words;   // 32-bit words per result row of rows narrower than 16 bytes, else 0
};
// kLists = 3: one controller's lists (an LWS tick: LWS, group, placement; a DS tick: DS, role,
// revision-role).  kLists = 6: a joint tick, the LWS tick's three lists then the DS tick's three.
template <int kLists>
struct PublishArgs {
  PublishList list[kLists];
  const uint32_t* extra;   // nullable: one more device word to publish (the placement round counter)
  uint32_t* host_words;    // mapped host: count of list k at [host_word(k)], [3] = extra, the sequence word at [seq_slot]
  uint32_t seq_slot;
  uint32_t seq;
  uint32_t* ticket;
  uint32_t fence_each;     // A/B: every CTA fences at system scope as well
  // clear: device words zeroed after `extra` was read (the tick slot's block of placement counters)
  uint32_t* clear;
  uint32_t n_clear;
};

constexpr uint32_t kPublishThreads = 1024;

// Host word of list k's count: lists 0-2 at [0..2] (then [3] extra, [4] the sequence word of a tick
// slot), lists 3-5 at [5..7].
__host__ __device__ constexpr uint32_t host_word(uint32_t k) { return k < 3u ? k : k + 2u; }

template <int kLists>
__global__ void __launch_bounds__(kPublishThreads) publish_lists_kernel(const PublishArgs<kLists> a) {
  __shared__ uint32_t s_last;
  pdl_wait_prior();  // every producer kernel of the tick has completed: lists and counters are final
  const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsize = gridDim.x * blockDim.x;
  // the counts and each thread's first elements are requested together (the lists' memory is valid
  // up to the capacity): one L2 round trip instead of two before the first store leaves
  uint32_t counts[kLists] = {}, row0[kLists] = {};
  uint4 out0[kLists];
#pragma unroll
  for (uint32_t k = 0; k < kLists; k++) {
    const PublishList& l = a.list[k];
    out0[k] = make_uint4(0, 0, 0, 0);
    if (l.count == nullptr) continue;
    counts[k] = __ldcg(l.count);
    if (gtid < l.capacity) row0[k] = __ldcg(l.src_rows + gtid);
    if (gtid < l.capacity * l.out_vec) out0[k] = __ldcg(l.src_outs + gtid);
  }
#pragma unroll
  for (uint32_t k = 0; k < kLists; k++) {
    const PublishList& l = a.list[k];
    if (l.count == nullptr) continue;
    const uint32_t n = min(counts[k], l.capacity);
    if (gtid < n) l.dst_rows[gtid] = row0[k];
    if (gtid < n * l.out_vec) l.dst_outs[gtid] = out0[k];
    for (uint32_t i = gtid + gsize; i < n; i += gsize) l.dst_rows[i] = __ldcg(l.src_rows + i);
#pragma unroll 4
    for (uint32_t i = gtid + gsize; i < n * l.out_vec; i += gsize) l.dst_outs[i] = __ldcg(l.src_outs + i);
    for (uint32_t i = gtid; i < n * l.out_words; i += gsize)  // (DS role / revision-role rows: 8 and 4 bytes)
      reinterpret_cast<uint32_t*>(l.dst_outs)[i] = __ldcg(reinterpret_cast<const uint32_t*>(l.src_outs) + i);
  }
  __syncthreads();
  bool last = true;
  if (gridDim.x > 1) {
    if (threadIdx.x == 0) {
      if (a.fence_each) __threadfence_system();
      uint32_t t;  // release at gpu scope: the CTA's stores (ordered before this by bar.sync) happen-before the ticket
      asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(t) : "l"(a.ticket) : "memory");
      s_last = t == gridDim.x - 1u ? 1u : 0u;
    }
    __syncthreads();
    last = s_last != 0u;
  }
  if (last && threadIdx.x == 0) {
    volatile uint32_t* hw = a.host_words;
#pragma unroll
    for (uint32_t k = 0; k < kLists; k++) {
      if (a.list[k].count == nullptr) continue;
      hw[host_word(k)] = counts[k];
      *a.list[k].count = 0u;  // ready for the next tick (stream-ordered)
    }
    if (a.extra != nullptr) hw[3] = __ldcg(a.extra);
    for (uint32_t k = 0; k < a.n_clear; k++) a.clear[k] = 0u;
    *a.ticket = 0u;
    // release at system scope (fence.acq_rel.sys + store; __threadfence_system() is the heavier
    // fence.sc.sys + L1 invalidate): everything that happens-before this store is visible to the
    // host thread that observes the word
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.host_words + a.seq_slot), "r"(a.seq) : "memory");
  }
}

struct PublishListHost {
  const uint32_t* src_rows;
  const void* src_outs;
  uint32_t* dst_rows;
  void* dst_outs;
  uint32_t* count;   // null = skip this slot
  uint32_t capacity;
  uint32_t out_bytes;
};

template <int kLists>
static int launch_publish_lists(const PublishListHost* lists, const uint32_t* d_extra, uint32_t* h_words, uint32_t seq_slot,
                                uint32_t seq, uint32_t* d_ticket, uint32_t expected_rows, cudaStream_t s, int* cuda_err,
                                uint32_t* d_clear, uint32_t n_clear, bool pdl) {
  *cuda_err = 0;
  PublishArgs<kLists> a{};
  for (int k = 0; k < kLists; k++) {
    const bool vec = lists[k].out_bytes % 16u == 0;
    a.list[k] = PublishList{lists[k].src_rows, static_cast<const uint4*>(lists[k].src_outs), lists[k].dst_rows,
                            static_cast<uint4*>(lists[k].dst_outs), lists[k].count, lists[k].capacity,
                            vec ? lists[k].out_bytes / 16u : 0u, vec ? 0u : lists[k].out_bytes / 4u};
  }
  a.extra = d_extra;
  a.host_words = h_words;
  a.seq_slot = seq_slot;
  a.seq = seq;
  a.ticket = d_ticket;
  a.clear = d_clear;
  a.n_clear = d_clear ? n_clear : 0u;
  static const bool fence_each = [] {
    const char* v = getenv("LWSE_PUBLISH_FENCE_EACH");
    return v && atoi(v) != 0;
  }();
  a.fence_each = fence_each ? 1u : 0u;
  // ONE CTA for the usual few thousand rows (no ticket stage then); more when the previous tick reported many
  unsigned grid = expected_rows / 8192u + 1u;
  if (grid > 32u) grid = 32u;
  const cudaError_t e = launch_pdl(publish_lists_kernel<kLists>, dim3(grid), dim3(kPublishThreads), 0, s, g_pdl && pdl, a);
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

// lists[0..2]: the three slots (host_words[k] receives the count of slot k).
int launch_publish(const PublishListHost* lists, const uint32_t* d_extra, uint32_t* h_words, uint32_t seq_slot,
                   uint32_t seq, uint32_t* d_ticket, uint32_t expected_rows, cudaStream_t s, int* cuda_err,
                   uint32_t* d_clear, uint32_t n_clear, bool pdl) {
  return launch_publish_lists<3>(lists, d_extra, h_words, seq_slot, seq, d_ticket, expected_rows, s, cuda_err, d_clear, n_clear,
                                 pdl);
}

// A joint tick: lists[0..5], counts to host_words[0..2] and [5..7] (host_word).
int launch_publish_joint(const PublishListHost* lists, const uint32_t* d_extra, uint32_t* h_words, uint32_t seq_slot,
                         uint32_t seq, uint32_t* d_ticket, uint32_t expected_rows, cudaStream_t s, int* cuda_err,
                         uint32_t* d_clear, uint32_t n_clear) {
  return launch_publish_lists<6>(lists, d_extra, h_words, seq_slot, seq, d_ticket, expected_rows, s, cuda_err, d_clear, n_clear,
                                 false);
}

// --------------------------------------------------------------------------
// row patches for the resident tables
// --------------------------------------------------------------------------
// One launch applies every scattered patch segment of a tick (lwse_resident_tick): row numbers
// and packed values are read where the host wrote them (mapped pinned memory, or a staged device
// copy).  Identity-row patches also move the pod's occupancy count from its old node to the new.
struct ScatterSeg {
  void* table;
  const uint32_t* rows;
  const void* values;
  uint64_t table_rows;
  uint32_t n;
  uint32_t row_bytes;   // 1, 16 (identity), 32 (placement request), 64
  uint32_t work_begin;  // first work item of this segment (16-byte pieces, or groups of four 1-byte rows)
  uint32_t is_ident;
};
constexpr int kMaxScatterSegs = 8;
struct ScatterArgs {
  ScatterSeg seg[kMaxScatterSegs];
  uint32_t n_segs;
  uint32_t total_work;
  uint32_t* occupancy;  // nullable
  uint32_t n_nodes;
};

__device__ __forceinline__ void scatter_body(const ScatterArgs& a) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < a.total_work; i += gridDim.x * blockDim.x) {
    int k = 0;
#pragma unroll
    for (int q = 1; q < kMaxScatterSegs; q++)
      if (q < (int)a.n_segs && i >= a.seg[q].work_begin) k = q;
    const ScatterSeg& sg = a.seg[k];
    const uint32_t j = i - sg.work_begin;
    if (sg.row_bytes == 1u) {
      // four patches per thread: one 16-byte read of row numbers and one 4-byte read of values —
      // over PCIe (the arena is host memory) the number of read requests is what costs, not the bytes
      const uint32_t k0 = j * 4u;
      uint8_t* tb = static_cast<uint8_t*>(sg.table);
      if (k0 + 3u < sg.n) {
        const uint4 r4 = *reinterpret_cast<const uint4*>(sg.rows + k0);
        const uint32_t v4 = *reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(sg.values) + k0);
        if (r4.x < sg.table_rows) tb[r4.x] = (uint8_t)v4;
        if (r4.y < sg.table_rows) tb[r4.y] = (uint8_t)(v4 >> 8);
        if (r4.z < sg.table_rows) tb[r4.z] = (uint8_t)(v4 >> 16);
        if (r4.w < sg.table_rows) tb[r4.w] = (uint8_t)(v4 >> 24);
      } else {
        for (uint32_t k = k0; k < sg.n; k++) {
          const uint32_t r = sg.rows[k];
          if (r < sg.table_rows) tb[r] = static_cast<const uint8_t*>(sg.values)[k];
        }
      }
    } else {
      const uint32_t pieces = sg.row_bytes >> 4;
      const uint32_t row_i = j / pieces, piece = j - row_i * pieces;
      const uint32_t r = sg.rows[row_i];
      if (r >= sg.table_rows) continue;
      const uint4 v = static_cast<const uint4*>(sg.values)[j];
      uint4* dst = static_cast<uint4*>(sg.table) + (uint64_t)r * pieces + piece;
      if (sg.is_ident && a.occupancy != nullptr) {
        // (through L2 only: a line of the table cached in this SM's L1 would be stale for the sweep
        // kernel, which may already be resident — programmatic dependent launch — and reads after us)
        const uint32_t old = __ldcg(&dst->w);
        if (old != v.w) {
          if ((old & LWSE_PODID_SCHEDULED) && (old >> LWSE_PODID_NODE_SHIFT) < a.n_nodes)
            atomicSub(a.occupancy + (old >> LWSE_PODID_NODE_SHIFT), 1u);
          if ((v.w & LWSE_PODID_SCHEDULED) && (v.w >> LWSE_PODID_NODE_SHIFT) < a.n_nodes)
            atomicAdd(a.occupancy + (v.w >> LWSE_PODID_NODE_SHIFT), 1u);
        }
      }
      *dst = v;
    }
  }
}

__global__ void __launch_bounds__(256) scatter_rows_kernel(const __grid_constant__ ScatterArgs a) {
  pdl_launch_dependents();
  pdl_wait_prior();  // the tables may still be read by the previous tick's kernels
  scatter_body(a);
}

// The same kernel for a tick replayed as a CUDA graph: kernel parameters are frozen in a graph, so
// the segment descriptors of THIS tick come from device memory (a 1 KB copy node at the root of the
// graph brings them from the pinned slot the host just wrote).
__global__ void __launch_bounds__(256) scatter_rows_desc_kernel(const ScatterArgs* __restrict__ desc) {
  __shared__ ScatterArgs s_a;
  pdl_launch_dependents();
  pdl_wait_prior();
  static_assert(sizeof(ScatterArgs) % 4 == 0, "copied word by word");
  for (uint32_t i = threadIdx.x; i < sizeof(ScatterArgs) / 4u; i += blockDim.x)
    reinterpret_cast<uint32_t*>(&s_a)[i] = __ldcg(reinterpret_cast<const uint32_t*>(desc) + i);
  __syncthreads();
  scatter_body(s_a);
}

struct ScatterSegHost {
  void* table;
  uint64_t table_rows;
  const uint32_t* rows;
  const void* values;
  uint32_t n;
  uint32_t row_bytes;
  bool is_ident;
};

// Segment list -> kernel arguments.  false: more than kMaxScatterSegs segments, a row width the kernel
// does not handle, or more than 2^32 work items.
static bool fill_scatter_args(const ScatterSegHost* segs, int n_segs, uint32_t* d_occupancy, uint32_t n_nodes, ScatterArgs* out) {
  ScatterArgs a{};
  uint64_t work = 0;
  int k = 0;
  for (int i = 0; i < n_segs; i++) {
    if (segs[i].n == 0) continue;
    if (k >= kMaxScatterSegs || (segs[i].row_bytes != 1u && (segs[i].row_bytes & 15u))) return false;
    a.seg[k] = ScatterSeg{segs[i].table, segs[i].rows, segs[i].values, segs[i].table_rows, segs[i].n,
                          segs[i].row_bytes, (uint32_t)work, segs[i].is_ident ? 1u : 0u};
    work += segs[i].row_bytes == 1u ? ((uint64_t)segs[i].n + 3u) / 4u : (uint64_t)segs[i].n * (segs[i].row_bytes >> 4);
    k++;
  }
  if (work > 0xFFFFFFFFull) return false;
  a.n_segs = (uint32_t)k;
  a.total_work = (uint32_t)work;
  a.occupancy = d_occupancy;
  a.n_nodes = n_nodes;
  *out = a;
  return true;
}

// Graph form: the descriptor block (scatter_desc_bytes() bytes, written by write_scatter_desc into a
// pinned slot and copied to d_desc by a node of the graph) and a fixed grid.
size_t scatter_desc_bytes() { return sizeof(ScatterArgs); }
bool write_scatter_desc(void* h_desc, const ScatterSegHost* segs, int n_segs, uint32_t* d_occupancy, uint32_t n_nodes) {
  ScatterArgs a{};
  if (!fill_scatter_args(segs, n_segs, d_occupancy, n_nodes, &a)) return false;
  memcpy(h_desc, &a, sizeof(a));
  return true;
}
int launch_scatter_desc(const void* d_desc, int sm_count, cudaStream_t s, bool pdl, int* cuda_err) {
  *cuda_err = 0;
  const cudaError_t e = launch_pdl(scatter_rows_desc_kernel, dim3((unsigned)sm_count * 4u), dim3(256), 0, s, pdl && g_pdl,
                                   static_cast<const ScatterArgs*>(d_desc));
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

int launch_scatter(const ScatterSegHost* segs, int n_segs, uint32_t* d_occupancy, uint32_t n_nodes, cudaStream_t s,
                   bool pdl, int* cuda_err) {
  *cuda_err = 0;
  ScatterArgs a{};
  if (!fill_scatter_args(segs, n_segs, d_occupancy, n_nodes, &a)) {
    *cuda_err = (int)cudaErrorInvalidValue;
    return -1;
  }
  if (a.n_segs == 0) return 0;
  const uint64_t work = a.total_work;
  uint64_t grid = (work + 255) / 256;
  if (grid > 148ull * 16ull) grid = 148ull * 16ull;
  const cudaError_t e = launch_pdl(scatter_rows_kernel, dim3((unsigned)grid), dim3(256), 0, s, pdl && g_pdl, a);
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

// Scheduled pods per node of a resident identity column (at load).
int launch_occupancy(const lwse_pod_ident* d_ident, uint64_t n_pods, uint32_t* d_occupancy, uint32_t n_nodes, int sm_count,
                     cudaStream_t s, int* cuda_err) {
  *cuda_err = 0;
  cudaError_t e = cudaMemsetAsync(d_occupancy, 0, (size_t)n_nodes * 4, s);
  if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
  if (n_pods == 0) return 0;
  const uint64_t want = (n_pods + 255) / 256;
  const uint32_t cap = (uint32_t)sm_count * 16u;
  pod_occupancy_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, s>>>(d_ident, n_pods, d_occupancy, n_nodes);
  e = cudaGetLastError();
  if (e != cudaSuccess) { *cuda_err = (int)e; return -1; }
  return 1;
}

// LWSE_SMEM_CARVEOUT (experiment switch, engine creation): one preferred shared-memory carveout (percent of the
// SM's maximum) for every kernel of a tick, so that CTAs of the sweep and of the placement round never ask the SM
// for different L1 / shared-memory splits.
cudaError_t set_sweep_carveout(int pct) {
  cudaError_t e = cudaSuccess;
  auto set = [&](const void* k) {
    const cudaError_t r = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    if (r != cudaSuccess) e = r;
  };
  set((const void*)group_fused_kernel);
  set((const void*)lws_sweep_kernel<1>);
  set((const void*)lws_sweep_kernel<2>);
  set((const void*)lws_sweep_kernel<4>);
  set((const void*)lws_sweep_kernel<8>);
  set((const void*)lws_sweep_kernel<16>);
  set((const void*)lws_sweep_kernel<32>);
  set((const void*)scatter_rows_kernel);
  set((const void*)scatter_rows_desc_kernel);
  set((const void*)publish_lists_kernel<3>);
  set((const void*)publish_lists_kernel<6>);
  return e;
}

}  // namespace lwse
