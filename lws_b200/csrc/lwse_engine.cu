// C-ABI implementation of include/lwse.h: engine lifecycle, device staging,
// host- and device-pointer entry points.  No CPU compute path exists in this
// library: every sweep is a CUDA kernel launch or the call fails.
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <unordered_map>
#include <vector>
#include <new>

#include "lwse_device.cuh"

namespace lwse {
// lwse_lws_kernels.cu
struct SweepChangeLists {
  uint32_t* lws_rows = nullptr;
  lwse_lws_out* lws_out = nullptr;
  uint32_t lws_capacity = 0;
  uint32_t* group_rows = nullptr;
  lwse_group_out* group_out = nullptr;
  uint32_t group_capacity = 0;
  uint32_t* counts = nullptr;
};
struct PublishListHost {
  const uint32_t* src_rows;
  const void* src_outs;
  uint32_t* dst_rows;
  void* dst_outs;
  uint32_t* count;
  uint32_t capacity;
  uint32_t out_bytes;
};
int launch_publish(const PublishListHost* lists, const uint32_t* d_extra, uint32_t* h_words, uint32_t seq_slot,
                   uint32_t seq, uint32_t* d_ticket, uint32_t expected_rows, cudaStream_t s, int* cuda_err,
                   uint32_t* d_clear, uint32_t n_clear, bool pdl);
int launch_publish_joint(const PublishListHost* lists, const uint32_t* d_extra, uint32_t* h_words, uint32_t seq_slot,
                         uint32_t seq, uint32_t* d_ticket, uint32_t expected_rows, cudaStream_t s, int* cuda_err,
                         uint32_t* d_clear, uint32_t n_clear);
cudaError_t set_sweep_carveout(int pct);
cudaError_t set_place_ns_carveout(int pct);
int launch_lws_sweep(const lwse_lws_tables* t, const lwse_node_rec* d_nodes, uint32_t n_nodes,
                     void* scratch, int sm_count, cudaStream_t s, int* cuda_err, const SweepChangeLists* cl,
                     uint32_t* d_event_count = nullptr, int first_mode = 1);
size_t lws_sweep_scratch_bytes(uint64_t n_pods, uint32_t n_groups);
struct ScatterSegHost {
  void* table;
  uint64_t table_rows;
  const uint32_t* rows;
  const void* values;
  uint32_t n;
  uint32_t row_bytes;
  bool is_ident;
};
int launch_scatter(const ScatterSegHost* segs, int n_segs, uint32_t* d_occupancy, uint32_t n_nodes, cudaStream_t s,
                   bool pdl, int* cuda_err);
size_t scatter_desc_bytes();
bool write_scatter_desc(void* h_desc, const ScatterSegHost* segs, int n_segs, uint32_t* d_occupancy, uint32_t n_nodes);
int launch_scatter_desc(const void* d_desc, int sm_count, cudaStream_t s, bool pdl, int* cuda_err);
int launch_ident_prefetch(const uint8_t* d_state, uint64_t n_pods, const lwse_pod_ident* mapped_host_ident,
                          lwse_pod_ident* d_ident, int sm_count, cudaStream_t s, int* cuda_err);
int launch_occupancy(const lwse_pod_ident* d_ident, uint64_t n_pods, uint32_t* d_occupancy, uint32_t n_nodes, int sm_count,
                     cudaStream_t s, int* cuda_err);
// lwse_place_kernels.cu
int launch_place(const lwse_node_rec* d_nodes, const uint32_t* d_dom_first, const uint32_t* d_node_order,
                 const uint32_t* d_node_pos, uint32_t n_nodes, uint32_t n_domains,
                 const lwse_place_req* d_reqs, uint32_t n_reqs, const uint32_t* d_occupancy,
                 uint32_t n_namespaces, lwse_place_out* d_out, void* d_scratch, size_t scratch_bytes,
                 uint32_t* h_rounds, int sm_count, cudaStream_t s, int* cuda_err, uint32_t call_index,
                 bool fresh, uint32_t n_parts, uint32_t reqs_per_part, uint64_t part_stride_bytes,
                 uint32_t* h_unpinned, const uint32_t** d_counters_out, const uint32_t** d_unpinned_out,
                 bool after_push);
size_t place_scratch_bytes(uint32_t n_nodes, uint32_t n_domains, uint32_t n_reqs, uint32_t n_namespaces);
size_t place_ns_scratch_bytes(uint32_t n_nodes, uint32_t n_domains, uint32_t n_reqs, uint32_t n_namespaces);
struct PlaceNsChanges {  // a tick's placement change list (device memory); prev == null: off
  lwse_place_out* prev;
  uint32_t* rows;
  lwse_place_out* outs;
  uint32_t* count;
  uint32_t capacity;
  int tick_slot;    // see lwse_place_ns_kernels.cu
  void* mid_event;
};
struct PlaceNsExchange {
  const unsigned long long* step_ctr;
  uint64_t half_bytes;
  bool lagged;
};
bool place_ns_supported(uint32_t n_nodes, uint32_t n_domains);
int launch_place_ns(const lwse_node_rec* d_nodes, const uint32_t* d_dom_first, const uint32_t* d_node_order, uint32_t n_nodes,
                    uint32_t n_usable, uint32_t n_domains, const lwse_place_req* d_reqs, uint32_t n_reqs,
                    const uint32_t* d_occupancy, uint32_t n_parts, uint64_t part_stride_bytes, uint32_t n_namespaces,
                    lwse_place_out* d_out, void* d_scratch, size_t scratch_bytes, bool fresh, uint32_t call_index, bool scan,
                    int sm_count, cudaStream_t s, int* cuda_err, const uint32_t** d_counters_out, bool first_pdl,
                    const PlaceNsChanges* changes, const PlaceNsExchange* xch);
int launch_place_diff(const lwse_place_out* d_cur, lwse_place_out* d_prev, uint32_t n, uint32_t* d_rows,
                      lwse_place_out* d_outs, uint32_t capacity, uint32_t* d_count, cudaStream_t s, int* cuda_err);
// lwse_ds_kernels.cu
int launch_ds_sweep(const lwse_ds_tables* t, int sm_count, cudaStream_t s, int* cuda_err);
struct DsResidentArgs {
  lwse_ds_out* ds_committed;
  lwse_ds_role_out* role_committed;
  lwse_ds_revrole_out* revrole_committed;
  lwse_ds_role_out* role_scratch;
  lwse_ds_revrole_out* revrole_scratch;
  uint32_t* ds_rows;
  lwse_ds_out* ds_outs;
  uint32_t* role_rows;
  lwse_ds_role_out* role_outs;
  uint32_t* revrole_rows;
  lwse_ds_revrole_out* revrole_outs;
  uint32_t* counts;
  uint32_t first;
};
int launch_ds_resident_sweep(const lwse_ds_tables* t, const DsResidentArgs* r, int sm_count, cudaStream_t s, bool pdl,
                             int* cuda_err);
// lwse_sha1_kernels.cu
int launch_sha1(const uint8_t* d_bytes, const uint32_t* d_offsets, uint32_t n, uint8_t* d_digests,
                int sm_count, cudaStream_t s, int* cuda_err);
int launch_subgroup_keys(const uint8_t* d_bytes, const uint32_t* d_offsets, uint32_t n, const int32_t* d_pod_count,
                         const int32_t* d_subgroup_size, const int32_t* d_worker_index, int32_t* d_index_out,
                         uint8_t* d_digests, int sm_count, cudaStream_t s, int* cuda_err);
// lwse_exchange_kernels.cu
int launch_exchange_push(const void* d_local_part, uint8_t* const* d_peer_base, void* d_local_base,
                         uint64_t part_bytes, uint64_t part_stride, uint64_t half_bytes, uint64_t flags_offset,
                         uint64_t step, uint64_t wait_step, uint32_t world, uint32_t rank, cudaStream_t s, int* cuda_err,
                         bool lagged);
}  // namespace lwse


namespace {

// A device buffer that only grows (sweeps reuse their staging memory).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

// Pinned, mapped host memory that only grows: the host writes / reads it in place and the GPU
// reaches it through `d` (patch arena, change lists, tick words).
struct PinBuf {
  void* h = nullptr;
  void* d = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (h) cudaFreeHost(h);
    h = d = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 8 + 4096;
    cudaError_t e = cudaHostAlloc(&h, want, cudaHostAllocMapped);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer(&d, h, 0);
    if (e == cudaSuccess) {
      cap = want;
      memset(h, 0, want);  // sequence words and counters start at zero
    } else if (h) {
      cudaFreeHost(h);
      h = d = nullptr;
    }
    return e;
  }
  void release() {
    if (h) cudaFreeHost(h);
    h = d = nullptr;
    cap = 0;
  }
  bool holds(const void* ptr, size_t bytes) const {
    const uintptr_t a = reinterpret_cast<uintptr_t>(ptr), b = reinterpret_cast<uintptr_t>(h);
    return h && a >= b && a + bytes <= b + cap;
  }
  template <typename T>
  T* dev_of(const T* host_ptr) const {
    return reinterpret_cast<T*>(static_cast<uint8_t*>(d) + (reinterpret_cast<const uint8_t*>(host_ptr) - static_cast<uint8_t*>(h)));
  }
};

}  // namespace

struct lwse_engine {
  int device = 0;
  int sm_count = lwse::kSmCount;
  cudaStream_t stream = nullptr;
  cudaStream_t side_stream = nullptr;  // placement round of lwse_reconcile_device
  cudaStream_t hist_stream = nullptr;  // copies the unpinned-request count of a round to the host, off the critical path
  cudaEvent_t ev_hist = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  std::mutex mu;
  int last_cuda_error = 0;
  uint64_t launches = 0;
  // resident node table
  DevBuf nodes;
  DevBuf dom_first, node_order, node_pos;  // static domain-sorted index of the node table (placement)
  uint32_t n_nodes = 0, n_domains = 0;
  // staging for the *_host entry points
  DevBuf lws, groups, pod_state, pod_ident, lws_out, group_out, occupancy, scan_scratch;
  DevBuf place_reqs, place_out, place_occ, place_scratch;
  uint64_t ident_rows = ~0ull;       // rows of the identity column resident from the last host sweep
  uint64_t ident_hint_pods = ~0ull;  // n_pods the hint below was measured on
  uint32_t ident_hint_events = 0;    // event pods the previous host sweep of that table visited
  // resident tables (lwse_resident_*)
  DevBuf r_lws, r_groups, r_pst, r_pid, r_lws_out, r_group_out, r_scan;
  DevBuf r_counts;                   // per tick slot (16 words): [0] lws changes, [1] group changes, [2] publish ticket, [4] place changes
  DevBuf r_occ;                      // scheduled pods per node of the resident identity column
  DevBuf r_preq, r_pout, r_pout_prev;  // resident placement requests / results of this and the previous tick
  PinBuf arena;                      // patch arena handed to the caller
  PinBuf stage;                      // staging for patch segments that lie outside the arena
  DevBuf arena_mirror, stage_mirror; // device copies of the two: a tick with many patches moves them with one DMA
                                     // copy per buffer (SM reads of host memory are latency-bound: ~6 GB/s measured)
  PinBuf chg;                        // change lists: [lws rows | lws out | group rows | group out | place rows | place out]
  DevBuf chg_dev;                    // the same layout in device memory: the kernels append here, a publish kernel copies out
  uint32_t last_changed[2] = {0, 0}; // rows the previous tick reported (sweep lists, placement list): sizes the publish grid
  PinBuf tickw;                      // per tick slot (16 words): [0] lws changes [1] group changes [2] place changes
                                     // [3] placement rounds [4] sequence word; a joint tick also [5] ds [6] role [7] revrole
  size_t chg_off[6] = {};
  uint32_t rn_lws = 0, rn_groups = 0, rn_reqs = 0, rn_namespaces = 0;
  uint64_t rn_pods = 0;
  bool r_loaded = false, r_place_loaded = false;
  uint32_t tick_seq = 0;
  // ticks in flight (lwse_resident_tick_submit / _wait): two slots of pinned change lists and words
  struct TickSlot {
    uint32_t seq = 0;
    bool do_sweep = false, do_place = false, published = false, wrote = false;
    bool joint = false;  // lwse_joint_tick_submit: the slot's DS lists are published too
  } tslot[2];
  uint64_t t_submitted = 0, t_waited = 0;
  size_t chg_bytes = 0;              // one slot of `chg`
  // a tick replayed as a CUDA graph (one cudaGraphLaunch instead of ~10 launches of 2-4 us each)
  struct TickGraph {
    cudaGraphExec_t exec = nullptr;
    uint32_t seen = 0;      // eager ticks with this key so far (the first one lets every buffer settle)
    uint32_t kernels = 0;   // kernel nodes (launch accounting)
    bool failed = false;    // capture or instantiation failed once: this key stays eager
    bool place_ns = false;  // its round runs the namespace kernels (counters in the slot's block)
    const uint32_t* rounds_ptr = nullptr;  // where its round counts
  };
  std::unordered_map<uint32_t, TickGraph> tick_graphs;
  PinBuf tdesc;                      // 2 slots x 512 B: the scatter's segment descriptors of the tick of that parity
  DevBuf tdesc_dev;                  // device copy (the copy node at the root of a tick graph fills it)
  cudaStream_t copy_stream = nullptr;  // the patch copy of a replayed tick: overlaps the previous tick's kernels
  cudaEvent_t ev_dma = nullptr;
  cudaStream_t pub_stream = nullptr;   // the publish kernels: tick k+1 starts while tick k's changed rows travel to the host
  cudaEvent_t ev_done = nullptr;       // behind the last kernel of a tick on the engine's stream (both branches joined)
  cudaEvent_t ev_mid = nullptr;        // (graph capture) between the condense and the namespace kernel
  bool tick_place_ns = false;          // the last enqueue_place() ran the namespace kernels (their counters are per slot)
  int use_graph = 1;                 // LWSE_TICK_GRAPH: 0 never, 1 when a tick is in flight (default), 2 always
  uint64_t graph_ticks = 0;
  cudaEvent_t ev_pub = nullptr;      // behind the previous tick's publish kernel: the next tick's side stream starts there
  cudaStream_t ds_stream = nullptr;   // a joint tick's DS sweep: forked behind the scatter, joined before the publish
  cudaEvent_t ev_ds_fork = nullptr, ev_ds_join = nullptr;
  int tick_order = 0;                // LWSE_TICK_ORDER (A/B of the tick's enqueue order, see tick_locked)
  uint32_t* h_counts = nullptr;      // pinned, 2 words
  DevBuf h_counts_dev;               // event-pod count of the host entry point's sweep
  bool no_zero_copy = false;         // LWSE_NO_ZERO_COPY=1: always upload the identity column
  uint32_t place_calls = 0;          // selects the scratch half
  uint32_t place_geometry[4] = {0, 0, 0, 0};  // (n_reqs, n_namespaces, nodes, domains) the scratch was laid out for
  cudaEvent_t ev_place = nullptr;    // end of the last placement call: the next one (any stream) orders behind it
  bool place_pending = false;
  DevBuf place_ns_scratch;           // namespace-parallel form (grouped request tables)
  uint32_t place_ns_calls = 0;
  uint32_t place_ns_geometry[4] = {0, 0, 0, 0};
  uint32_t n_usable = 0;             // nodes a request can use (schedulable, labelled): length of the sorted index
  const uint32_t* place_rounds_ptr = nullptr;  // device: the round counter of the last placement call
  const uint32_t* place_scans_ptr = nullptr;   // device: its (request, round) search counter (grouped form), or null
  bool r_place_grouped = false;      // the resident request table is grouped by namespace
  std::vector<uint32_t> r_req_ns;    // its namespace column (host copy: patches must not regroup it)
  const uint32_t* place_counters = nullptr;  // device: counters / phase stamps of the last placement call
  const uint32_t* place_unpinned = nullptr;  // device: its unpinned-request count
  DevBuf ds, ds_roles, ds_revroles, ds_out, ds_role_out, ds_revrole_out;
  // resident DS tables (lwse_ds_resident_*): inputs, committed outputs, scratch, change lists — none
  // shared with the stateless DS sweep's staging above or with the LWS resident state
  DevBuf rd_ds, rd_roles, rd_revroles, rd_ds_out, rd_role_out, rd_revrole_out, rd_role_scratch, rd_revrole_scratch;
  // Change lists and counters per tick slot: a joint tick uses the ring slot it takes, lwse_ds_resident_tick slot 0.
  DevBuf rd_chg_dev;                 // change lists: [ds rows | ds out | role rows | role out | revrole rows | revrole out]
  DevBuf rd_counts;                  // 16 words per slot: [0] ds [1] role [2] revrole rows listed, [3] publish ticket
  PinBuf rd_chg;                     // the same layout in pinned, mapped memory (the publish kernel copies into it)
  PinBuf rd_tickw;                   // lwse_ds_resident_tick: [0..2] the three counts, [4] sequence word
  size_t rd_chg_off[6] = {};
  size_t rd_chg_bytes = 0;           // one slot of rd_chg / rd_chg_dev
  uint32_t rdn_ds = 0, rdn_roles = 0, rdn_revroles = 0;
  uint32_t rd_seq = 0, rd_last_changed = 0;
  bool rd_loaded = false, rd_first = false;
  DevBuf sha_bytes, sha_offsets, sha_digests, sha_ints;
  uint32_t* h_rounds = nullptr;  // pinned
  // peer exchange of the multi-GPU placement step (lwse_exchange_*)
  DevBuf xch, xch_peers_dev;
  void* xch_peer[LWSE_MAX_RANKS] = {};
  uint32_t xch_world = 0, xch_rank = 0, xch_reqs_per_part = 0;
  uint64_t xch_stride = 0, xch_reqs_off = 0, xch_half = 0, xch_flags_off = 0, xch_step = 0;
  bool xch_connected = false;
};

namespace {

int fail_cuda(lwse_engine* e, cudaError_t err) {
  e->last_cuda_error = (int)err;
  (void)cudaGetLastError();  // clear the sticky-free error state
  return err == cudaErrorMemoryAllocation ? LWSE_ERR_OOM : LWSE_ERR_CUDA;
}

#define LWSE_CUDA(e, call)                                \
  do {                                                    \
    cudaError_t err__ = (call);                           \
    if (err__ != cudaSuccess) return fail_cuda(e, err__); \
  } while (0)

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Tick graphs freeze device pointers and sizes in their kernel nodes: whatever reallocates or
// resizes a resident buffer drops them (the next ticks re-capture).
void invalidate_tick_graphs(lwse_engine* e) {
  for (auto& kv : e->tick_graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  e->tick_graphs.clear();
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

int check_lws_tables(const lwse_lws_tables* t) {
  if (!t) return LWSE_ERR_INVALID_ARG;
  if (t->n_lws && (!t->lws || !t->lws_out)) return LWSE_ERR_INVALID_ARG;
  if (t->n_groups && (!t->groups || !t->group_out)) return LWSE_ERR_INVALID_ARG;
  if (t->n_pods && (!t->pod_state || !t->pod_ident)) return LWSE_ERR_INVALID_ARG;
  if (t->n_pods > 0xFFFFFFFFull) return LWSE_ERR_UNSUPPORTED;  // pod_base / pod_count are 32-bit
  if (!aligned16(t->lws) || !aligned16(t->groups) || !aligned16(t->lws_out) || !aligned16(t->group_out) ||
      !aligned16(t->pod_state) || !aligned16(t->pod_ident))
    return LWSE_ERR_INVALID_ARG;
  return LWSE_OK;
}

}  // namespace

extern "C" {

static int drain_ticks_locked(lwse_engine* e);  // waits for (and drops the results of) every tick in flight

LWSE_API uint32_t lwse_abi_version(void) { return LWSE_ABI_VERSION; }

LWSE_API const char* lwse_strerror(int status) {
  switch (status) {
    case LWSE_OK: return "ok";
    case LWSE_ERR_INVALID_ARG: return "invalid argument (NULL or misaligned table, bad count)";
    case LWSE_ERR_NO_DEVICE: return "no usable CUDA device (this engine has no CPU fallback)";
    case LWSE_ERR_CUDA: return "CUDA call failed (see lwse_last_cuda_error)";
    case LWSE_ERR_OOM: return "device or pinned memory allocation failed";
    case LWSE_ERR_BAD_TABLE: return "a base/count in a record points outside its table";
    case LWSE_ERR_NOT_READY: return "engine not ready for this call (upload the node table first)";
    case LWSE_ERR_UNSUPPORTED: return "unsupported input";
    default: return "unknown lwse status";
  }
}

LWSE_API uint64_t lwse_hash64(const void* bytes, size_t len) {
  const uint8_t* b = static_cast<const uint8_t*>(bytes);
  uint64_t h = 0xCBF29CE484222325ull;
  for (size_t i = 0; i < len; i++) h = (h ^ b[i]) * 0x100000001B3ull;
  return h;
}

LWSE_API uint32_t lwse_shard_of(uint64_t uid_hash, uint32_t n_shards) {
  if (n_shards <= 1) return 0;
  // finalizer of splitmix64 so that weak uid hashes still spread
  uint64_t x = uid_hash;
  x ^= x >> 30;
  x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27;
  x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (uint32_t)(x % n_shards);
}

// The placement round of a tick is short and latency-bound; at the highest priority its CTAs
// take the first SM slots the sweep kernels free instead of queueing behind their blocks.
static cudaError_t create_side_stream(cudaStream_t* s) {
  int least = 0, greatest = 0;
  cudaError_t e = cudaDeviceGetStreamPriorityRange(&least, &greatest);
  if (e != cudaSuccess) return e;
  return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, greatest);
}

LWSE_API int lwse_create(const lwse_config* cfg, lwse_engine** out) {
  if (!cfg || !out) return LWSE_ERR_INVALID_ARG;
  *out = nullptr;
  if (cfg->abi_version != LWSE_ABI_VERSION) return LWSE_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || cfg->device < 0 || cfg->device >= n) {
    (void)cudaGetLastError();
    return LWSE_ERR_NO_DEVICE;
  }
  lwse_engine* e = new (std::nothrow) lwse_engine();
  if (!e) return LWSE_ERR_OOM;
  e->device = cfg->device;
  DeviceGuard guard(e->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, e->device) != cudaSuccess) {
    delete e;
    return LWSE_ERR_NO_DEVICE;
  }
  if (prop.major < 10) {  // the kernels are built for sm_100a only
    delete e;
    return LWSE_ERR_NO_DEVICE;
  }
  e->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess ||
      create_side_stream(&e->side_stream) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_pub, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_dma, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->pub_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_done, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_mid, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->hist_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_hist, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_place, cudaEventDisableTiming) != cudaSuccess ||
      cudaMallocHost(reinterpret_cast<void**>(&e->h_rounds), 64) != cudaSuccess ||
      cudaMallocHost(reinterpret_cast<void**>(&e->h_counts), 64) != cudaSuccess) {
    (void)cudaGetLastError();
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_join) cudaEventDestroy(e->ev_join);
    if (e->ev_pub) cudaEventDestroy(e->ev_pub);
    if (e->ev_dma) cudaEventDestroy(e->ev_dma);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->ev_done) cudaEventDestroy(e->ev_done);
    if (e->ev_mid) cudaEventDestroy(e->ev_mid);
    if (e->pub_stream) cudaStreamDestroy(e->pub_stream);
    if (e->ev_hist) cudaEventDestroy(e->ev_hist);
    if (e->ev_place) cudaEventDestroy(e->ev_place);
    if (e->hist_stream) cudaStreamDestroy(e->hist_stream);
    if (e->side_stream) cudaStreamDestroy(e->side_stream);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return LWSE_ERR_CUDA;
  }
  if (e->h_counts_dev.reserve(64) != cudaSuccess) {
    (void)cudaGetLastError();
    lwse_destroy(e);
    return LWSE_ERR_OOM;
  }
  if (cudaStreamCreateWithFlags(&e->ds_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_ds_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_ds_join, cudaEventDisableTiming) != cudaSuccess) {
    (void)cudaGetLastError();
    lwse_destroy(e);
    return LWSE_ERR_CUDA;
  }
  {
    const char* v = getenv("LWSE_NO_ZERO_COPY");
    e->no_zero_copy = v && atoi(v) != 0;
    const char* o = getenv("LWSE_TICK_ORDER");
    e->tick_order = o ? atoi(o) : 0;
    if (e->tick_order < 0 || e->tick_order > 2) e->tick_order = 0;
    const char* g = getenv("LWSE_TICK_GRAPH");
    e->use_graph = g ? atoi(g) : 1;
    const char* c = getenv("LWSE_SMEM_CARVEOUT");  // percent of the maximum shared memory, every tick kernel alike
    if (c && atoi(c) >= 0 && atoi(c) <= 100) {
      (void)lwse::set_sweep_carveout(atoi(c));
      (void)lwse::set_place_ns_carveout(atoi(c));
      (void)cudaGetLastError();
    }
  }
  *out = e;
  return LWSE_OK;
}

LWSE_API void lwse_destroy(lwse_engine* e) {
  if (!e) return;
  {
    DeviceGuard guard(e->device);
    cudaStreamSynchronize(e->stream);
    cudaStreamSynchronize(e->side_stream);
    cudaStreamSynchronize(e->hist_stream);  // its copies target h_rounds, freed below
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    if (e->pub_stream) cudaStreamSynchronize(e->pub_stream);
    for (auto& kv : e->tick_graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    e->tick_graphs.clear();
    for (uint32_t p = 0; p < e->xch_world; p++)
      if (e->xch_connected && p != e->xch_rank && e->xch_peer[p]) cudaIpcCloseMemHandle(e->xch_peer[p]);
    e->xch.release();
    e->xch_peers_dev.release();
    DevBuf* bufs[] = {&e->nodes,      &e->dom_first, &e->node_order, &e->node_pos, &e->lws,         &e->groups,     &e->pod_state,   &e->pod_ident,
                      &e->scan_scratch, &e->lws_out,
                      &e->group_out,  &e->occupancy,   &e->place_reqs, &e->place_out,   &e->place_occ,
                      &e->place_scratch, &e->ds,       &e->ds_roles,   &e->ds_revroles, &e->ds_out,
                      &e->ds_role_out, &e->ds_revrole_out, &e->sha_bytes, &e->sha_offsets, &e->sha_digests, &e->sha_ints,
                      &e->r_lws, &e->r_groups, &e->r_pst, &e->r_pid, &e->r_lws_out, &e->r_group_out, &e->r_scan,
                      &e->r_counts, &e->r_occ, &e->r_preq, &e->r_pout, &e->r_pout_prev, &e->h_counts_dev, &e->place_ns_scratch,
                      &e->arena_mirror, &e->stage_mirror, &e->chg_dev, &e->tdesc_dev,
                      &e->rd_ds, &e->rd_roles, &e->rd_revroles, &e->rd_ds_out, &e->rd_role_out, &e->rd_revrole_out,
                      &e->rd_role_scratch, &e->rd_revrole_scratch, &e->rd_chg_dev, &e->rd_counts};
    for (DevBuf* b : bufs) b->release();
    PinBuf* pins[] = {&e->arena, &e->stage, &e->chg, &e->tickw, &e->tdesc, &e->rd_chg, &e->rd_tickw};
    for (PinBuf* b : pins) b->release();
    if (e->ev_place) cudaEventDestroy(e->ev_place);
    if (e->h_rounds) cudaFreeHost(e->h_rounds);
    if (e->h_counts) cudaFreeHost(e->h_counts);
    cudaEventDestroy(e->ev_hist);
    cudaStreamDestroy(e->hist_stream);
    cudaEventDestroy(e->ev_fork);
    cudaEventDestroy(e->ev_join);
    if (e->ev_pub) cudaEventDestroy(e->ev_pub);
    if (e->ev_dma) cudaEventDestroy(e->ev_dma);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->ev_done) cudaEventDestroy(e->ev_done);
    if (e->ev_mid) cudaEventDestroy(e->ev_mid);
    if (e->pub_stream) cudaStreamDestroy(e->pub_stream);
    if (e->ds_stream) {
      cudaStreamSynchronize(e->ds_stream);
      cudaStreamDestroy(e->ds_stream);
    }
    if (e->ev_ds_fork) cudaEventDestroy(e->ev_ds_fork);
    if (e->ev_ds_join) cudaEventDestroy(e->ev_ds_join);
    cudaStreamDestroy(e->side_stream);
    cudaStreamDestroy(e->stream);
  }
  delete e;
}

LWSE_API int lwse_last_cuda_error(const lwse_engine* e) { return e ? e->last_cuda_error : 0; }
LWSE_API void* lwse_stream(const lwse_engine* e) { return e ? (void*)e->stream : nullptr; }
LWSE_API uint64_t lwse_launch_count(const lwse_engine* e) { return e ? e->launches : 0; }
LWSE_API uint64_t lwse_graph_tick_count(const lwse_engine* e) { return e ? e->graph_ticks : 0; }

LWSE_API int lwse_upload_nodes(lwse_engine* e, const lwse_node_rec* nodes, uint32_t n_nodes,
                               uint32_t n_domains) {
  if (!e || (n_nodes && !nodes) || !aligned16(nodes)) return LWSE_ERR_INVALID_ARG;
  if (n_nodes > LWSE_POD_NODE_MAX) return LWSE_ERR_UNSUPPORTED;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  {
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
    invalidate_tick_graphs(e);
  }
  LWSE_CUDA(e, e->nodes.reserve((size_t)n_nodes * sizeof(lwse_node_rec) + 16));
  // Static index for the placement round: the usable nodes (schedulable, labelled with a
  // topology domain) in domain order — a counting sort, done once per node-table upload.
  // dom_first[d] .. dom_first[d + 1] is the run of domain d in node_order; node_pos is the
  // inverse (LWSE_NONE for nodes no request can use).
  std::vector<uint32_t> first((size_t)n_domains + 2, 0u), order, pos(n_nodes ? n_nodes : 1, LWSE_NONE);
  auto usable = [&](const lwse_node_rec& nd) {
    return (nd.flags & LWSE_NODE_SCHEDULABLE) && (nd.flags & LWSE_NODE_HAS_TOPOLOGY) && nd.domain_id < n_domains;
  };
  for (uint32_t n = 0; n < n_nodes; n++)
    if (usable(nodes[n])) first[(size_t)nodes[n].domain_id + 1]++;
  for (uint32_t d = 0; d < n_domains; d++) first[(size_t)d + 1] += first[d];
  order.resize(first[n_domains] ? first[n_domains] : 1, 0u);
  {
    std::vector<uint32_t> cursor(first.begin(), first.end() - 1);
    for (uint32_t n = 0; n < n_nodes; n++)
      if (usable(nodes[n])) {
        const uint32_t p = cursor[nodes[n].domain_id]++;
        order[p] = n;
        pos[n] = p;
      }
  }
  LWSE_CUDA(e, e->dom_first.reserve(((size_t)n_domains + 1) * 4 + 16));
  // (padded to whole rows of 256 entries: the namespace-parallel placement kernel stages the index
  // into shared memory with one bulk copy of that size)
  const size_t order_padded = ((size_t)(n_nodes + 255u) / 256u + 1u) * 1024u;
  LWSE_CUDA(e, e->node_order.reserve(order_padded + 16));
  LWSE_CUDA(e, cudaMemsetAsync(e->node_order.p, 0, order_padded, e->stream));
  LWSE_CUDA(e, e->node_pos.reserve(pos.size() * 4 + 16));
  if (n_nodes)
    LWSE_CUDA(e, cudaMemcpyAsync(e->nodes.p, nodes, (size_t)n_nodes * sizeof(lwse_node_rec),
                                 cudaMemcpyHostToDevice, e->stream));
  LWSE_CUDA(e, cudaMemcpyAsync(e->dom_first.p, first.data(), ((size_t)n_domains + 1) * 4, cudaMemcpyHostToDevice,
                               e->stream));
  LWSE_CUDA(e, cudaMemcpyAsync(e->node_order.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, e->stream));
  LWSE_CUDA(e, cudaMemcpyAsync(e->node_pos.p, pos.data(), pos.size() * 4, cudaMemcpyHostToDevice, e->stream));
  LWSE_CUDA(e, cudaStreamSynchronize(e->stream));  // the host vectors above go out of scope
  e->n_nodes = n_nodes;
  e->n_domains = n_domains;
  e->n_usable = (uint32_t)first[n_domains];
  e->place_ns_geometry[0] = e->place_ns_geometry[1] = e->place_ns_geometry[2] = e->place_ns_geometry[3] = 0;
  e->place_geometry[0] = e->place_geometry[1] = e->place_geometry[2] = e->place_geometry[3] = 0;  // re-initialise the scratch
  return LWSE_OK;
}

// ---------------------------------------------------------------------------
// LWS sweep
// ---------------------------------------------------------------------------
static int sweep_device_locked(lwse_engine* e, const lwse_lws_tables* t, cudaStream_t s) {
  // the scan bitmaps live in engine-owned scratch; it only grows (a growth is a
  // cudaMalloc, so size it with one warm-up call before capturing a graph)
  LWSE_CUDA(e, e->scan_scratch.reserve(lwse::lws_sweep_scratch_bytes(t->n_pods, t->n_groups)));
  int cuda_err = 0;
  int launched = lwse::launch_lws_sweep(t, (const lwse_node_rec*)e->nodes.p, e->n_nodes,
                                        e->scan_scratch.p, e->sm_count, s, &cuda_err, nullptr);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  return LWSE_OK;
}

LWSE_API int lwse_sweep_lws_device(lwse_engine* e, const lwse_lws_tables* t, void* stream) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  int rc = check_lws_tables(t);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return sweep_device_locked(e, t, stream ? (cudaStream_t)stream : e->stream);
}

// lwse_sweep_lws_host with the engine locked and its device current; returns after the results
// are in the caller's tables (stream synchronized — the only synchronize of the call).
// `after_uploads` (optional): called once the table uploads are enqueued and before the sweep is —
// lwse_reconcile_host enqueues its placement branch there, so that the copy engine starts on the
// big tables at once instead of behind the host-side preparation of the round.
static int sweep_host_locked(lwse_engine* e, const lwse_lws_tables* h, const std::function<int()>* after_uploads = nullptr) {
  cudaStream_t s = e->stream;
  const size_t b_lws = (size_t)h->n_lws * sizeof(lwse_lws_rec);
  const size_t b_grp = (size_t)h->n_groups * sizeof(lwse_group_rec);
  const size_t b_pst = (size_t)h->n_pods * sizeof(lwse_pod_state);
  const size_t b_pid = (size_t)h->n_pods * sizeof(lwse_pod_ident);
  const size_t b_lo = (size_t)h->n_lws * sizeof(lwse_lws_out);
  const size_t b_go = (size_t)h->n_groups * sizeof(lwse_group_out);
  LWSE_CUDA(e, e->lws.reserve(b_lws + 16));
  LWSE_CUDA(e, e->groups.reserve(b_grp + 16));
  LWSE_CUDA(e, e->pod_state.reserve(b_pst + 32));
  const void* ident_before = e->pod_ident.p;
  LWSE_CUDA(e, e->pod_ident.reserve(b_pid + 16));
  const bool ident_moved = ident_before != e->pod_ident.p;
  LWSE_CUDA(e, e->scan_scratch.reserve(lwse::lws_sweep_scratch_bytes(h->n_pods, h->n_groups)));
  LWSE_CUDA(e, e->lws_out.reserve(b_lo + 16));
  LWSE_CUDA(e, e->group_out.reserve(b_go + 16));
  const bool want_occ = h->node_occupancy != nullptr && e->n_nodes > 0;
  if (want_occ) {
    LWSE_CUDA(e, e->occupancy.reserve((size_t)e->n_nodes * 4 + 16));
  }
  // the hot byte column first: the identity prefetch below needs only it
  if (b_pst) LWSE_CUDA(e, cudaMemcpyAsync(e->pod_state.p, h->pod_state, b_pst, cudaMemcpyHostToDevice, s));
  lwse_lws_tables d = *h;
  d.lws = (const lwse_lws_rec*)e->lws.p;
  d.groups = (const lwse_group_rec*)e->groups.p;
  d.pod_state = (const lwse_pod_state*)e->pod_state.p;
  d.pod_ident = (const lwse_pod_ident*)e->pod_ident.p;
  d.lws_out = (lwse_lws_out*)e->lws_out.p;
  d.group_out = (lwse_group_out*)e->group_out.p;
  d.node_occupancy = want_occ ? (uint32_t*)e->occupancy.p : nullptr;
  int cuda_err = 0;
  bool counted = false, prefetching = false;
  if (b_pst) {
    // The identity column (16 B / pod, 16 of the 17 input bytes per pod) is only read for pods
    // with a restart / deletion event.  It is left out of the upload
    //  - when the caller says it did not change (LWSE_SWEEP_REUSE_POD_IDENT), or
    //  - when the caller's buffer is pinned, mapped host memory and few pods have an event: a
    //    prefetch kernel on the side stream copies just those rows over PCIe while the other
    //    tables are still being uploaded (a 64-byte read per event pod against 16 B / pod in
    //    bulk).  "Few" is what the PREVIOUS sweep of a table of this size visited (no mid-step
    //    synchronize; the first sweep of a table is optimistic).
    const bool reuse = (h->flags & LWSE_SWEEP_REUSE_POD_IDENT) && e->ident_rows == h->n_pods && !ident_moved;
    const void* mapped = nullptr;
    if (!reuse && !e->no_zero_copy && !want_occ) {
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, h->pod_ident) == cudaSuccess && attr.type == cudaMemoryTypeHost)
        mapped = attr.devicePointer;
      else
        (void)cudaGetLastError();
    }
    const bool few = e->ident_hint_pods != h->n_pods || (uint64_t)e->ident_hint_events * 64u <= b_pid / 2u;
    if (mapped && few && h->n_groups && !(h->flags & (LWSE_SWEEP_SKIP_POD_SCAN | LWSE_SWEEP_SKIP_GROUP_PASS))) {
      LWSE_CUDA(e, cudaEventRecord(e->ev_fork, s));
      LWSE_CUDA(e, cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
      int launched = lwse::launch_ident_prefetch((const uint8_t*)e->pod_state.p, h->n_pods, (const lwse_pod_ident*)mapped,
                                                 (lwse_pod_ident*)e->pod_ident.p, e->sm_count, e->side_stream, &cuda_err);
      if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
      e->launches += (uint64_t)launched;
      LWSE_CUDA(e, cudaEventRecord(e->ev_join, e->side_stream));
      prefetching = true;
      e->ident_rows = ~0ull;  // the device copy holds the event pods' rows only
    } else {
      if (!reuse) LWSE_CUDA(e, cudaMemcpyAsync(e->pod_ident.p, h->pod_ident, b_pid, cudaMemcpyHostToDevice, s));
      e->ident_rows = h->n_pods;
    }
    counted = h->n_groups && !(h->flags & (LWSE_SWEEP_SKIP_POD_SCAN | LWSE_SWEEP_SKIP_GROUP_PASS));
    if (counted) LWSE_CUDA(e, cudaMemsetAsync(e->h_counts_dev.p, 0, 4, s));
  }
  if (b_grp) LWSE_CUDA(e, cudaMemcpyAsync(e->groups.p, h->groups, b_grp, cudaMemcpyHostToDevice, s));
  if (b_lws) LWSE_CUDA(e, cudaMemcpyAsync(e->lws.p, h->lws, b_lws, cudaMemcpyHostToDevice, s));
  if (after_uploads) {
    const int arc = (*after_uploads)();
    if (arc != LWSE_OK) return arc;
  }
  if (prefetching) LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_join, 0));
  int launched = lwse::launch_lws_sweep(&d, (const lwse_node_rec*)e->nodes.p, e->n_nodes, e->scan_scratch.p, e->sm_count,
                                        s, &cuda_err, nullptr, counted ? (uint32_t*)e->h_counts_dev.p : nullptr,
                                        /*first_pdl=*/false);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;

  // group results first: they are complete while the LWS pass still runs
  if (b_go) LWSE_CUDA(e, cudaMemcpyAsync(h->group_out, e->group_out.p, b_go, cudaMemcpyDeviceToHost, s));
  if (b_lo) LWSE_CUDA(e, cudaMemcpyAsync(h->lws_out, e->lws_out.p, b_lo, cudaMemcpyDeviceToHost, s));
  if (want_occ)
    LWSE_CUDA(e, cudaMemcpyAsync(h->node_occupancy, e->occupancy.p, (size_t)e->n_nodes * 4,
                                 cudaMemcpyDeviceToHost, s));
  if (counted) LWSE_CUDA(e, cudaMemcpyAsync(e->h_counts, e->h_counts_dev.p, 4, cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  if (counted) {
    e->ident_hint_pods = h->n_pods;
    e->ident_hint_events = e->h_counts[0];
  }
  return LWSE_OK;
}

LWSE_API int lwse_sweep_lws_host(lwse_engine* e, const lwse_lws_tables* h) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  int rc = check_lws_tables(h);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return sweep_host_locked(e, h);
}

// ---------------------------------------------------------------------------
// Resident tables
// ---------------------------------------------------------------------------
static size_t align256(size_t v) { return (v + 255u) & ~(size_t)255u; }

// (re)allocate the pinned change lists for the resident tables' sizes
static int reserve_change_lists(lwse_engine* e) {
  invalidate_tick_graphs(e);  // called by both resident loads: table pointers and sizes change
  LWSE_CUDA(e, cudaStreamSynchronize(e->pub_stream));  // (a publish kernel may still be copying out of the lists)
  size_t off = 0;
  const size_t sizes[6] = {(size_t)e->rn_lws * 4,       (size_t)e->rn_lws * sizeof(lwse_lws_out),
                           (size_t)e->rn_groups * 4,    (size_t)e->rn_groups * sizeof(lwse_group_out),
                           (size_t)e->rn_reqs * 4,      (size_t)e->rn_reqs * sizeof(lwse_place_out)};
  for (int k = 0; k < 6; k++) {
    e->chg_off[k] = off;
    off += align256(sizes[k] + 16);
  }
  e->chg_bytes = off;
  LWSE_CUDA(e, e->chg.reserve(2 * off));  // two ticks may be in flight: the host reads one slot while the next tick fills the other
  LWSE_CUDA(e, e->chg_dev.reserve(2 * off));  // per tick slot: tick k+1 appends while tick k's lists are published
  LWSE_CUDA(e, e->tickw.reserve(256));
  return LWSE_OK;
}

LWSE_API int lwse_resident_load(lwse_engine* e, const lwse_lws_tables* h) {
  if (!e || !h) return LWSE_ERR_INVALID_ARG;
  if ((h->n_lws && !h->lws) || (h->n_groups && !h->groups) || (h->n_pods && (!h->pod_state || !h->pod_ident)))
    return LWSE_ERR_INVALID_ARG;
  if (h->n_pods > 0xFFFFFFFFull) return LWSE_ERR_UNSUPPORTED;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  {
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
  }
  cudaStream_t s = e->stream;
  const size_t b_lws = (size_t)h->n_lws * sizeof(lwse_lws_rec), b_grp = (size_t)h->n_groups * sizeof(lwse_group_rec);
  const size_t b_pst = (size_t)h->n_pods * sizeof(lwse_pod_state), b_pid = (size_t)h->n_pods * sizeof(lwse_pod_ident);
  const size_t b_lo = (size_t)h->n_lws * sizeof(lwse_lws_out), b_go = (size_t)h->n_groups * sizeof(lwse_group_out);
  LWSE_CUDA(e, e->r_lws.reserve(b_lws + 16));
  LWSE_CUDA(e, e->r_groups.reserve(b_grp + 16));
  LWSE_CUDA(e, e->r_pst.reserve(b_pst + 32));
  LWSE_CUDA(e, e->r_pid.reserve(b_pid + 16));
  LWSE_CUDA(e, e->r_lws_out.reserve(b_lo + 16));
  LWSE_CUDA(e, e->r_group_out.reserve(b_go + 16));
  LWSE_CUDA(e, e->r_scan.reserve(lwse::lws_sweep_scratch_bytes(h->n_pods, h->n_groups)));
  LWSE_CUDA(e, e->r_counts.reserve(128));  // 64 bytes per tick slot
  LWSE_CUDA(e, e->r_occ.reserve((size_t)e->n_nodes * 4 + 16));
  LWSE_CUDA(e, cudaMemsetAsync(e->r_counts.p, 0, 128, s));
  if (b_lws) LWSE_CUDA(e, cudaMemcpyAsync(e->r_lws.p, h->lws, b_lws, cudaMemcpyHostToDevice, s));
  if (b_grp) LWSE_CUDA(e, cudaMemcpyAsync(e->r_groups.p, h->groups, b_grp, cudaMemcpyHostToDevice, s));
  if (b_pst) LWSE_CUDA(e, cudaMemcpyAsync(e->r_pst.p, h->pod_state, b_pst, cudaMemcpyHostToDevice, s));
  if (b_pid) LWSE_CUDA(e, cudaMemcpyAsync(e->r_pid.p, h->pod_ident, b_pid, cudaMemcpyHostToDevice, s));
  // forget previous results: an all-ones row never equals a real result, so the first sweep reports every row
  if (b_lo) LWSE_CUDA(e, cudaMemsetAsync(e->r_lws_out.p, 0xFF, b_lo, s));
  if (b_go) LWSE_CUDA(e, cudaMemsetAsync(e->r_group_out.p, 0xFF, b_go, s));
  if (e->n_nodes) {  // scheduled pods per node; identity-row patches keep it current from here on
    int cuda_err = 0;
    int launched = lwse::launch_occupancy((const lwse_pod_ident*)e->r_pid.p, h->n_pods, (uint32_t*)e->r_occ.p, e->n_nodes,
                                          e->sm_count, s, &cuda_err);
    if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
    e->launches += (uint64_t)launched;
  }
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  e->rn_lws = h->n_lws;
  e->rn_groups = h->n_groups;
  e->rn_pods = h->n_pods;
  e->r_loaded = true;
  e->r_place_loaded = false;
  e->rn_reqs = 0;
  return reserve_change_lists(e);
}

LWSE_API int lwse_resident_arena(lwse_engine* e, uint64_t min_bytes, void** base_out, uint64_t* bytes_out) {
  if (!e || !base_out) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  const size_t want_arena = min_bytes ? (size_t)min_bytes : ((size_t)8 << 20);
  if (want_arena > e->arena.cap) {  // growing replaces the buffer: nothing may still be reading it
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
    LWSE_CUDA(e, cudaStreamSynchronize(e->stream));
    LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
  }
  LWSE_CUDA(e, e->arena.reserve(min_bytes ? (size_t)min_bytes : ((size_t)8 << 20)));
  *base_out = e->arena.h;
  if (bytes_out) *bytes_out = e->arena.cap;
  return LWSE_OK;
}

// Table-id sets a call resolves: the LWS tick takes ids 0-4, the DS tick 5-7, a joint tick both.
constexpr uint32_t kLwsTableIds = 0x1Fu, kDsTableIds = 0xE0u, kAllTableIds = kLwsTableIds | kDsTableIds;

// table → (device base, rows, bytes per row); false for an id outside `ids`.
static bool resident_table(lwse_engine* e, uint32_t which, void** base, uint64_t* rows, uint32_t* row_bytes,
                           uint32_t ids = kLwsTableIds) {
  if (which > LWSE_TABLE_DS_REVROLES || !((ids >> which) & 1u)) return false;
  switch (which) {
    case LWSE_TABLE_DS: *base = e->rd_ds.p; *rows = e->rdn_ds; *row_bytes = sizeof(lwse_ds_rec); return true;
    case LWSE_TABLE_DS_ROLES: *base = e->rd_roles.p; *rows = e->rdn_roles; *row_bytes = sizeof(lwse_ds_role_rec); return true;
    case LWSE_TABLE_DS_REVROLES:
      *base = e->rd_revroles.p; *rows = e->rdn_revroles; *row_bytes = sizeof(lwse_ds_revrole_rec); return true;
    case LWSE_TABLE_LWS: *base = e->r_lws.p; *rows = e->rn_lws; *row_bytes = sizeof(lwse_lws_rec); return true;
    case LWSE_TABLE_GROUPS: *base = e->r_groups.p; *rows = e->rn_groups; *row_bytes = sizeof(lwse_group_rec); return true;
    case LWSE_TABLE_POD_STATE: *base = e->r_pst.p; *rows = e->rn_pods; *row_bytes = sizeof(lwse_pod_state); return true;
    case LWSE_TABLE_POD_IDENT: *base = e->r_pid.p; *rows = e->rn_pods; *row_bytes = sizeof(lwse_pod_ident); return true;
    case LWSE_TABLE_PLACE_REQS:
      if (!e->r_place_loaded) return false;
      *base = e->r_preq.p; *rows = e->rn_reqs; *row_bytes = sizeof(lwse_place_req); return true;
    default: return false;
  }
}

// A segment's rows / values are read by the scatter kernel where the caller wrote them when they
// lie in the arena and are aligned for its vector loads (16-byte row-number reads; 16-byte value
// reads, 4-byte for the byte column); otherwise the call stages a copy.
static bool rows_in_place(const lwse_engine* e, const lwse_patch_seg& g) {
  return e->arena.holds(g.rows, (size_t)g.n * 4) && aligned16(g.rows);
}
static bool values_in_place(const lwse_engine* e, const lwse_patch_seg& g, uint32_t rb) {
  return e->arena.holds(g.values, (size_t)g.n * rb) &&
         (rb == 1 ? (reinterpret_cast<uintptr_t>(g.values) & 3u) == 0 : aligned16(g.values));
}

// Enqueue the patch segments of a tick on the engine's stream.  *wrote = some table changed
// (the sweep's first kernel then has to wait for the scatter kernel to finish).
// `tables`: bit t set = apply the segments of lwse_table t (a tick applies the placement request
// patches on the side stream, where the round that reads them runs, and the rest on the engine's
// stream); `stage_base`: where in the staging buffer this call may put copies.
struct ScatterPlan {  // a prepared scatter launch (apply_patches_locked with `defer`): the copy is enqueued, the kernel is not
  lwse::ScatterSegHost sc[2 * LWSE_TICK_MAX_SEGS];  // (both parts of a joint tick)
  int n = 0;
  bool recount = false;
  // with `plan_only`: nothing was enqueued at all; the arena span [lo, hi) still has to be copied
  // to the mirror (dma), or — staged segments, range segments — the plan cannot be replayed (eager_only)
  bool dma = false, eager_only = false;
  size_t lo = 0, hi = 0;
};

// One scatter launch per LWSE_TICK_MAX_SEGS segments (the kernel's limit): only a joint tick can need a
// second one, which follows programmatically and waits for the first at its top.
static int launch_scatter_plan(lwse_engine* e, const ScatterPlan& p, cudaStream_t s) {
  int cuda_err = 0;
  for (int k0 = 0; k0 < p.n; k0 += (int)LWSE_TICK_MAX_SEGS) {
    const int n = p.n - k0 < (int)LWSE_TICK_MAX_SEGS ? p.n - k0 : (int)LWSE_TICK_MAX_SEGS;
    int launched = lwse::launch_scatter(p.sc + k0, n, e->n_nodes ? (uint32_t*)e->r_occ.p : nullptr, e->n_nodes, s, true, &cuda_err);
    if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
    e->launches += (uint64_t)launched;
  }
  if (p.recount && e->n_nodes) {
    int launched = lwse::launch_occupancy((const lwse_pod_ident*)e->r_pid.p, e->rn_pods, (uint32_t*)e->r_occ.p, e->n_nodes,
                                          e->sm_count, s, &cuda_err);
    if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
    e->launches += (uint64_t)launched;
  }
  return LWSE_OK;
}

static int apply_patches_locked(lwse_engine* e, const lwse_patch_seg* segs, uint32_t n_segs, bool* wrote,
                                uint32_t tables = 0xFFFFFFFFu, cudaStream_t s = nullptr, size_t stage_base = 0,
                                size_t* stage_used = nullptr, long dma_min_bytes = 0, ScatterPlan* defer = nullptr,
                                bool plan_only = false, uint32_t ids = kLwsTableIds) {
  *wrote = false;
  if (stage_used) *stage_used = stage_base;
  if (n_segs == 0) return LWSE_OK;
  // (a joint tick hands both parts' segments in one call, each part at most LWSE_TICK_MAX_SEGS)
  if (!segs || n_segs > (ids == kAllTableIds ? 2u : 1u) * LWSE_TICK_MAX_SEGS) return LWSE_ERR_INVALID_ARG;
  if (!s) s = e->stream;
  // room for every segment that is not in the arena
  size_t need = 0;
  for (uint32_t i = 0; i < n_segs; i++) {
    void* base;
    uint64_t rows;
    uint32_t rb;
    if (!resident_table(e, segs[i].table, &base, &rows, &rb, ids)) return LWSE_ERR_INVALID_ARG;
    if (segs[i].n == 0 || !((tables >> segs[i].table) & 1u)) continue;
    if (!segs[i].values || (!(segs[i].flags & LWSE_PATCH_RANGE) && !segs[i].rows)) return LWSE_ERR_INVALID_ARG;
    if (segs[i].flags & LWSE_PATCH_RANGE) {
      if ((uint64_t)segs[i].first_row + segs[i].n > rows) return LWSE_ERR_BAD_TABLE;
      continue;
    }
    if (!rows_in_place(e, segs[i])) need += align256((size_t)segs[i].n * 4);
    if (!values_in_place(e, segs[i], rb)) need += align256((size_t)segs[i].n * rb);
  }
  if (stage_base + need > e->stage.cap) {
    if (stage_base) return LWSE_ERR_OOM;  // (the tick sizes the buffer for both of its calls up front)
    LWSE_CUDA(e, cudaStreamSynchronize(e->stream));
    LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
    LWSE_CUDA(e, e->stage.reserve(need));
  }
  ScatterPlan plan;
  lwse::ScatterSegHost* sc = plan.sc;
  int n_sc = 0;
  size_t cursor = stage_base;
  bool recount = false;
  for (uint32_t i = 0; i < n_segs; i++) {
    const lwse_patch_seg& g = segs[i];
    if (g.n == 0 || !((tables >> g.table) & 1u)) continue;
    void* base;
    uint64_t rows;
    uint32_t rb;
    resident_table(e, g.table, &base, &rows, &rb, ids);
    *wrote = true;
    if (g.table == LWSE_TABLE_PLACE_REQS && e->r_place_grouped) {
      // a request that moves to another namespace breaks the grouping the fast placement kernels rely on
      const lwse_place_req* v = static_cast<const lwse_place_req*>(g.values);
      for (uint32_t k = 0; k < g.n; k++) {
        const uint32_t row = (g.flags & LWSE_PATCH_RANGE) ? g.first_row + k : g.rows[k];
        if (row < e->rn_reqs && v[k].ns != e->r_req_ns[row]) {
          e->r_req_ns[row] = v[k].ns;
          e->r_place_grouped = false;
        }
      }
    } else if (g.table == LWSE_TABLE_PLACE_REQS) {
      const lwse_place_req* v = static_cast<const lwse_place_req*>(g.values);
      for (uint32_t k = 0; k < g.n; k++) {
        const uint32_t row = (g.flags & LWSE_PATCH_RANGE) ? g.first_row + k : g.rows[k];
        if (row < e->rn_reqs) e->r_req_ns[row] = v[k].ns;
      }
    }
    if (g.flags & LWSE_PATCH_RANGE) {  // one DMA copy straight into the table
      if (plan_only) {
        plan.eager_only = true;
        continue;
      }
      LWSE_CUDA(e, cudaMemcpyAsync(static_cast<uint8_t*>(base) + (size_t)g.first_row * rb, g.values, (size_t)g.n * rb,
                                   cudaMemcpyHostToDevice, s));
      if (g.table == LWSE_TABLE_POD_IDENT) recount = true;
      continue;
    }
    const uint32_t* d_rows;
    const void* d_vals;
    if (rows_in_place(e, g)) {
      d_rows = e->arena.dev_of(g.rows);
    } else {
      if (plan_only) plan.eager_only = true;
      uint8_t* dst = static_cast<uint8_t*>(e->stage.h) + cursor;
      memcpy(dst, g.rows, (size_t)g.n * 4);
      d_rows = reinterpret_cast<const uint32_t*>(static_cast<uint8_t*>(e->stage.d) + cursor);
      cursor += align256((size_t)g.n * 4);
    }
    if (values_in_place(e, g, rb)) {
      d_vals = e->arena.dev_of(static_cast<const uint8_t*>(g.values));
    } else {
      if (plan_only) plan.eager_only = true;
      uint8_t* dst = static_cast<uint8_t*>(e->stage.h) + cursor;
      memcpy(dst, g.values, (size_t)g.n * rb);
      d_vals = static_cast<uint8_t*>(e->stage.d) + cursor;
      cursor += align256((size_t)g.n * rb);
    }
    sc[n_sc++] = lwse::ScatterSegHost{base, rows, d_rows, d_vals, g.n, rb, g.table == LWSE_TABLE_POD_IDENT};
  }
  if (n_sc) {
    // Few patch bytes: the scatter kernel reads them in place over PCIe (one round trip, no copy
    // launch).  Many: one DMA copy per pinned buffer of the span this call uses, then the kernel
    // reads device memory — the copy engine moves 400 KB in ~10 us, SM reads of host memory need 60.
    static const long dma_threshold = [] {
      const char* v = getenv("LWSE_PATCH_DMA_BYTES");
      return v ? atol(v) : 16384L;
    }();
    size_t total = 0;
    for (int k = 0; k < n_sc; k++) total += (size_t)sc[k].n * (4u + sc[k].row_bytes);
    const long dma_from = dma_threshold < 0 ? -1 : (dma_min_bytes > dma_threshold ? dma_min_bytes : dma_threshold);
    if (dma_from >= 0 && total >= (size_t)dma_from) {
      struct Span { const PinBuf* pin; DevBuf* mirror; uintptr_t lo, hi; } spans[2] = {
          {&e->arena, &e->arena_mirror, UINTPTR_MAX, 0}, {&e->stage, &e->stage_mirror, UINTPTR_MAX, 0}};
      auto touch = [&](const void* dptr, size_t bytes) {
        for (Span& sp : spans) {
          const uintptr_t d0 = reinterpret_cast<uintptr_t>(sp.pin->d), a = reinterpret_cast<uintptr_t>(dptr);
          if (sp.pin->d && a >= d0 && a + bytes <= d0 + sp.pin->cap) {
            sp.lo = a - d0 < sp.lo ? a - d0 : sp.lo;
            sp.hi = a - d0 + bytes > sp.hi ? a - d0 + bytes : sp.hi;
          }
        }
      };
      for (int k = 0; k < n_sc; k++) {
        touch(sc[k].rows, (size_t)sc[k].n * 4);
        touch(sc[k].values, (size_t)sc[k].n * sc[k].row_bytes);
      }
      for (Span& sp : spans) {
        if (sp.hi <= sp.lo) continue;
        if (sp.mirror->cap < sp.pin->cap) {  // (first use, or the pinned buffer grew)
          LWSE_CUDA(e, cudaStreamSynchronize(e->stream));
          LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
          LWSE_CUDA(e, cudaStreamSynchronize(e->copy_stream));
          LWSE_CUDA(e, sp.mirror->reserve(sp.pin->cap));
        }
        if (plan_only) {
          if (sp.pin == &e->stage) {
            plan.eager_only = true;
          } else {
            plan.dma = true;
            plan.lo = sp.lo;
            plan.hi = sp.hi;
          }
        } else {
          LWSE_CUDA(e, cudaMemcpyAsync(static_cast<uint8_t*>(sp.mirror->p) + sp.lo, static_cast<const uint8_t*>(sp.pin->h) + sp.lo,
                                       sp.hi - sp.lo, cudaMemcpyHostToDevice, s));
        }
        const uintptr_t d0 = reinterpret_cast<uintptr_t>(sp.pin->d), m0 = reinterpret_cast<uintptr_t>(sp.mirror->p);
        for (int k = 0; k < n_sc; k++) {
          uintptr_t a = reinterpret_cast<uintptr_t>(sc[k].rows);
          if (a >= d0 && a < d0 + sp.pin->cap) sc[k].rows = reinterpret_cast<const uint32_t*>(m0 + (a - d0));
          a = reinterpret_cast<uintptr_t>(sc[k].values);
          if (a >= d0 && a < d0 + sp.pin->cap) sc[k].values = reinterpret_cast<const void*>(m0 + (a - d0));
        }
      }
    }
  }
  plan.n = n_sc;
  plan.recount = recount;
  if (stage_used) *stage_used = cursor;
  if (defer) {
    *defer = plan;
    return LWSE_OK;
  }
  return launch_scatter_plan(e, plan, s);
}

// bytes of staging the segments of a tick need in the worst case (nothing in the arena)
static size_t stage_bytes_upper_bound(const lwse_patch_seg* segs, uint32_t n_segs) {
  size_t need = 0;
  for (uint32_t i = 0; i < n_segs; i++)
    if (segs && !(segs[i].flags & LWSE_PATCH_RANGE)) need += align256((size_t)segs[i].n * 4) + align256((size_t)segs[i].n * 64);
  return need;
}

LWSE_API int lwse_resident_patch(lwse_engine* e, lwse_table which, const uint32_t* rows, const void* values,
                                 uint32_t n) {
  if (!e || (n && (!rows || !values))) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  if (n == 0) return LWSE_OK;
  DeviceGuard guard(e->device);
  {
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
  }
  lwse_patch_seg seg{};
  seg.table = (uint32_t)which;
  seg.n = n;
  seg.rows = rows;
  seg.values = values;
  bool wrote = false;
  const int rc = apply_patches_locked(e, &seg, 1, &wrote);
  if (rc != LWSE_OK) return rc;
  // the caller's buffers (and the staging copy) are free again once the scatter ran
  LWSE_CUDA(e, cudaStreamSynchronize(e->stream));
  return LWSE_OK;
}

LWSE_API int lwse_resident_outputs(lwse_engine* e, lwse_lws_out* lws_out, lwse_group_out* group_out) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaStream_t s = e->stream;
  if (lws_out && e->rn_lws)
    LWSE_CUDA(e, cudaMemcpyAsync(lws_out, e->r_lws_out.p, (size_t)e->rn_lws * sizeof(lwse_lws_out), cudaMemcpyDeviceToHost, s));
  if (group_out && e->rn_groups)
    LWSE_CUDA(e, cudaMemcpyAsync(group_out, e->r_group_out.p, (size_t)e->rn_groups * sizeof(lwse_group_out),
                                 cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

// ---------------------------------------------------------------------------
// Placement
// ---------------------------------------------------------------------------
constexpr uint32_t kFormGeneral = 0, kFormGrouped = 1, kFormScan = 2;
static const int g_place_form_env = [] {  // LWSE_PLACE_FORM=general|grouped|scan: A/B measurements
  const char* v = getenv("LWSE_PLACE_FORM");
  if (!v) return -1;
  return v[0] == 'g' && v[1] == 'e' ? 0 : v[0] == 's' ? 2 : 1;
}();

// The namespace-parallel form (request table grouped by namespace): condense kernel + one CTA per
// namespace.  `first_pdl`: nothing on the stream right before writes the request table.
static int place_grouped_locked(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs, const uint32_t* d_occupancy,
                                uint32_t n_parts, uint64_t part_stride_bytes, uint32_t n_namespaces, lwse_place_out* d_out,
                                bool scan, uint32_t* rounds_out, uint32_t* scans_out, cudaStream_t s, bool first_pdl,
                                const lwse::PlaceNsChanges* changes = nullptr, const lwse::PlaceNsExchange* xch = nullptr) {
  const size_t scratch = lwse::place_ns_scratch_bytes(e->n_nodes, e->n_domains, n_reqs, n_namespaces);
  const void* before = e->place_ns_scratch.p;
  LWSE_CUDA(e, e->place_ns_scratch.reserve(scratch));
  const uint32_t geometry[4] = {n_reqs, n_namespaces, e->n_nodes, e->n_domains};
  const bool fresh = before != e->place_ns_scratch.p || memcmp(geometry, e->place_ns_geometry, sizeof(geometry)) != 0;
  memcpy(e->place_ns_geometry, geometry, sizeof(geometry));
  cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
  const bool eager = cudaStreamIsCapturing(s, &capturing) == cudaSuccess && capturing == cudaStreamCaptureStatusNone;
  if (fresh && eager) invalidate_tick_graphs(e);  // (their kernel nodes hold the old scratch pointers)
  if (eager && e->place_pending) LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_place, 0));
  int cuda_err = 0;
  const uint32_t* counters = nullptr;
  int launched = lwse::launch_place_ns((const lwse_node_rec*)e->nodes.p, (const uint32_t*)e->dom_first.p,
                                       (const uint32_t*)e->node_order.p, e->n_nodes, e->n_usable, e->n_domains, d_reqs, n_reqs,
                                       d_occupancy, n_parts, part_stride_bytes, n_namespaces, d_out, e->place_ns_scratch.p,
                                       scratch, fresh, e->place_ns_calls++, scan, e->sm_count, s, &cuda_err, &counters,
                                       first_pdl && !fresh, changes, xch);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  e->place_rounds_ptr = counters;
  e->place_scans_ptr = counters + 3;
  if (eager && !changes) {  // (a tick — `changes` — returns only after the host has seen the round complete)
    LWSE_CUDA(e, cudaEventRecord(e->ev_place, s));
    e->place_pending = true;
  }
  if (rounds_out) {
    LWSE_CUDA(e, cudaMemcpyAsync(e->h_rounds + 4, counters, 16, cudaMemcpyDeviceToHost, s));
    LWSE_CUDA(e, cudaStreamSynchronize(s));
    *rounds_out = e->h_rounds[4];
    if (scans_out) *scans_out = e->h_rounds[7];
  }
  return LWSE_OK;
}

static int place_locked(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                        const uint32_t* d_occupancy, uint32_t n_namespaces, lwse_place_out* d_out,
                        uint32_t* rounds_out, cudaStream_t s, uint32_t n_parts, uint32_t reqs_per_part,
                        uint64_t part_stride_bytes, bool after_push = false, uint32_t form = kFormGeneral,
                        bool first_pdl = false, const lwse::PlaceNsChanges* changes = nullptr, bool* diffed = nullptr) {
  if ((n_reqs && (!d_reqs || !d_out)) || n_namespaces == 0) return LWSE_ERR_INVALID_ARG;
  if (e->n_nodes == 0 || e->n_domains == 0) return LWSE_ERR_NOT_READY;
  if (g_place_form_env == 0) form = kFormGeneral;
  if (g_place_form_env == 2 && form != kFormGeneral) form = kFormScan;
  if (diffed) *diffed = false;
  if (form != kFormGeneral && n_parts <= 1 && lwse::place_ns_supported(e->n_nodes, e->n_domains)) {
    if (diffed) *diffed = changes != nullptr;
    return place_grouped_locked(e, d_reqs, n_reqs, d_occupancy, 1, 0, n_namespaces, d_out, form == kFormScan, rounds_out, nullptr,
                                s, first_pdl, changes);
  }
  const size_t scratch = lwse::place_scratch_bytes(e->n_nodes, e->n_domains, n_reqs, n_namespaces);
  const void* before = e->place_scratch.p;
  LWSE_CUDA(e, e->place_scratch.reserve(scratch));
  // the two scratch halves are laid out for one geometry; any change re-initialises them
  const uint32_t geometry[4] = {n_reqs, n_namespaces, e->n_nodes, e->n_domains};
  const bool fresh = before != e->place_scratch.p || memcmp(geometry, e->place_geometry, sizeof(geometry)) != 0;
  if (fresh) e->h_rounds[2] = 0xFFFFFFFFu;  // no history for this geometry
  memcpy(e->place_geometry, geometry, sizeof(geometry));
  // placement calls of one engine share the scratch (a call resets the half the next one uses):
  // whatever streams they run on, each orders behind the previous one
  cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
  const bool eager = cudaStreamIsCapturing(s, &capturing) == cudaSuccess && capturing == cudaStreamCaptureStatusNone;
  if (eager && e->place_pending) LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_place, 0));
  int cuda_err = 0;
  int launched = lwse::launch_place((const lwse_node_rec*)e->nodes.p, (const uint32_t*)e->dom_first.p,
                                    (const uint32_t*)e->node_order.p, (const uint32_t*)e->node_pos.p, e->n_nodes,
                                    e->n_domains, d_reqs,
                                    n_reqs, d_occupancy, n_namespaces, d_out, e->place_scratch.p,
                                    scratch, rounds_out ? e->h_rounds : nullptr, e->sm_count, s, &cuda_err,
                                    e->place_calls++, fresh, n_parts, reqs_per_part, part_stride_bytes,
                                    e->h_rounds + 2, &e->place_counters, &e->place_unpinned, after_push);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  e->place_rounds_ptr = e->place_counters + 3;
  e->place_scans_ptr = nullptr;
  if (rounds_out) *rounds_out = e->h_rounds[0];
  if (eager) {
    LWSE_CUDA(e, cudaEventRecord(e->ev_place, s));
    e->place_pending = true;
  }
  // history for the next call's cluster-or-grid decision (only consulted beyond 1024 requests):
  // the round's unpinned-request count, copied on a third stream so that nothing waits for it
  if (n_reqs > 1024u && e->place_unpinned && eager) {
    LWSE_CUDA(e, cudaStreamWaitEvent(e->hist_stream, e->ev_place, 0));
    LWSE_CUDA(e, cudaMemcpyAsync(e->h_rounds + 2, e->place_unpinned, 4, cudaMemcpyDeviceToHost, e->hist_stream));
  }
  return LWSE_OK;
}

// ns non-decreasing over the table?  (host tables: a 4-byte read per 32-byte row)
static bool grouped_by_namespace(const lwse_place_req* reqs, uint32_t n) {
  for (uint32_t i = 1; i < n; i++)
    if (reqs[i].ns < reqs[i - 1].ns) return false;
  return true;
}

static uint32_t form_of_flags(uint32_t sweep_flags) {
  if (!(sweep_flags & LWSE_SWEEP_PLACE_GROUPED)) return kFormGeneral;
  return (sweep_flags & LWSE_SWEEP_PLACE_SCAN) ? kFormScan : kFormGrouped;
}

static int place_common(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                        const uint32_t* d_occupancy, uint32_t n_namespaces, lwse_place_out* d_out,
                        uint32_t* rounds_out, void* stream, uint32_t n_parts, uint32_t reqs_per_part,
                        uint64_t part_stride_bytes) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return place_locked(e, d_reqs, n_reqs, d_occupancy, n_namespaces, d_out, rounds_out,
                      stream ? (cudaStream_t)stream : e->stream, n_parts, reqs_per_part, part_stride_bytes);
}

// One reconcile tick on device tables: the placement round reads only inputs (requests, occupancy,
// node table), never the sweep's outputs, so it is enqueued on the engine's side stream and runs
// concurrently with the three sweep kernels; `stream` continues when both are done.
LWSE_API int lwse_reconcile_device(lwse_engine* e, const lwse_lws_tables* t, const lwse_place_req* d_reqs,
                                   uint32_t n_reqs, const uint32_t* d_occupancy, uint32_t n_namespaces,
                                   lwse_place_out* d_place_out, void* stream) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  int rc = check_lws_tables(t);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
  if (n_reqs == 0) return sweep_device_locked(e, t, s);
  LWSE_CUDA(e, cudaEventRecord(e->ev_fork, s));
  LWSE_CUDA(e, cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
  rc = place_locked(e, d_reqs, n_reqs, d_occupancy, n_namespaces, d_place_out, nullptr, e->side_stream, 1, n_reqs, 0, false,
                    form_of_flags(t->flags), /*first_pdl=*/false);
  if (rc == LWSE_OK) rc = sweep_device_locked(e, t, s);
  // join even after a failure, so that the side stream never runs ahead of `stream`
  cudaError_t je = cudaEventRecord(e->ev_join, e->side_stream);
  if (je == cudaSuccess) je = cudaStreamWaitEvent(s, e->ev_join, 0);
  if (rc != LWSE_OK) return rc;
  if (je != cudaSuccess) return fail_cuda(e, je);
  return LWSE_OK;
}

LWSE_API int lwse_place_device(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                               const uint32_t* d_occupancy, uint32_t n_namespaces,
                               lwse_place_out* d_out, uint32_t* rounds_out, void* stream) {
  return place_common(e, d_reqs, n_reqs, d_occupancy, n_namespaces, d_out, rounds_out, stream, 1, n_reqs, 0);
}

LWSE_API int lwse_place_grouped_device(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                                       const uint32_t* d_occupancy, uint32_t n_namespaces, lwse_place_out* d_out,
                                       uint32_t flags, uint32_t* rounds_out, uint32_t* pair_scans_out, void* stream) {
  if (!e || (n_reqs && (!d_reqs || !d_out)) || n_namespaces == 0) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (e->n_nodes == 0 || e->n_domains == 0) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
  if (!lwse::place_ns_supported(e->n_nodes, e->n_domains))  // too many domains for one CTA's shared memory
    return place_locked(e, d_reqs, n_reqs, d_occupancy, n_namespaces, d_out, rounds_out, s, 1, n_reqs, 0);
  return place_grouped_locked(e, d_reqs, n_reqs, d_occupancy, 1, 0, n_namespaces, d_out, (flags & LWSE_SWEEP_PLACE_SCAN) != 0,
                              rounds_out, pair_scans_out, s, /*first_pdl=*/false);
}

LWSE_API int lwse_place_gathered_device(lwse_engine* e, const void* d_parts, uint32_t n_parts,
                                        uint64_t part_stride_bytes, uint64_t reqs_offset_bytes,
                                        uint32_t reqs_per_part, uint32_t n_namespaces,
                                        lwse_place_out* d_out, uint32_t* rounds_out, void* stream) {
  if (!d_parts || n_parts == 0 || (part_stride_bytes & 15u) || (reqs_offset_bytes & 15u) ||
      (uint64_t)n_parts * reqs_per_part > 0xFFFFFFull)
    return LWSE_ERR_INVALID_ARG;
  const uint8_t* base = static_cast<const uint8_t*>(d_parts);
  return place_common(e, reinterpret_cast<const lwse_place_req*>(base + reqs_offset_bytes), n_parts * reqs_per_part,
                      reinterpret_cast<const uint32_t*>(base), n_namespaces, d_out, rounds_out, stream, n_parts,
                      reqs_per_part, part_stride_bytes);
}

// ---------------------------------------------------------------------------
// Peer exchange (multi-GPU placement step)
// ---------------------------------------------------------------------------
LWSE_API int lwse_exchange_create(lwse_engine* e, uint32_t reqs_per_part, uint32_t world, uint32_t rank,
                                  void* handle_out) {
  if (!e || !handle_out || world == 0 || world > LWSE_MAX_RANKS || rank >= world) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (e->n_nodes == 0 || e->n_domains == 0) return LWSE_ERR_NOT_READY;
  if (e->xch_world) return LWSE_ERR_UNSUPPORTED;  // one exchange per engine
  DeviceGuard guard(e->device);
  const uint64_t reqs_off = ((uint64_t)e->n_nodes * 4u + 15u) / 16u * 16u;
  const uint64_t stride = reqs_off + (uint64_t)reqs_per_part * sizeof(lwse_place_req);
  const uint64_t half = ((uint64_t)world * stride + 255u) / 256u * 256u;
  const uint64_t flags_off = 3u * half;  // three buffers: step s uses buffer s % 3 (lwse_exchange_kernels.cu)
  const uint64_t total = flags_off + (uint64_t)world * 8u + 64u;
  LWSE_CUDA(e, e->xch.reserve(total));
  LWSE_CUDA(e, cudaMemset(e->xch.p, 0, total));
  LWSE_CUDA(e, e->xch_peers_dev.reserve(sizeof(void*) * LWSE_MAX_RANKS));
  cudaIpcMemHandle_t h;
  LWSE_CUDA(e, cudaIpcGetMemHandle(&h, e->xch.p));
  static_assert(sizeof(h) == LWSE_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle_out, &h, sizeof(h));
  e->xch_world = world;
  e->xch_rank = rank;
  e->xch_reqs_per_part = reqs_per_part;
  e->xch_stride = stride;
  e->xch_reqs_off = reqs_off;
  e->xch_half = half;
  e->xch_flags_off = flags_off;
  e->xch_step = 0;
  e->xch_connected = false;
  return LWSE_OK;
}

LWSE_API int lwse_exchange_connect(lwse_engine* e, const void* handles) {
  if (!e || !handles) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->xch_world || e->xch_connected) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  for (uint32_t p = 0; p < e->xch_world; p++) {
    if (p == e->xch_rank) {
      e->xch_peer[p] = e->xch.p;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const uint8_t*>(handles) + (size_t)p * LWSE_IPC_HANDLE_BYTES, sizeof(h));
    LWSE_CUDA(e, cudaIpcOpenMemHandle(&e->xch_peer[p], h, cudaIpcMemLazyEnablePeerAccess));
  }
  LWSE_CUDA(e, cudaMemcpy(e->xch_peers_dev.p, e->xch_peer, sizeof(void*) * e->xch_world, cudaMemcpyHostToDevice));
  e->xch_connected = true;
  return LWSE_OK;
}

LWSE_API uint64_t lwse_exchange_part_bytes(const lwse_engine* e) { return e ? e->xch_stride : 0; }

// One reconcile tick of a multi-GPU shard: as lwse_reconcile_device, with the placement round
// solved over every rank's part — this rank's part is pushed to all peers first.
LWSE_API int lwse_reconcile_exchanged_device(lwse_engine* e, const lwse_lws_tables* t, const void* d_local_part,
                                             uint32_t n_namespaces, lwse_place_out* d_place_out, void* stream) {
  if (!e || !d_local_part || !aligned16(d_local_part)) return LWSE_ERR_INVALID_ARG;
  int rc = t ? check_lws_tables(t) : LWSE_OK;
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->xch_connected) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
  LWSE_CUDA(e, cudaEventRecord(e->ev_fork, s));
  LWSE_CUDA(e, cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
  const uint64_t step = ++e->xch_step;
  int cuda_err = 0;
  int launched = lwse::launch_exchange_push(d_local_part, (uint8_t* const*)e->xch_peers_dev.p, e->xch.p, e->xch_stride,
                                            e->xch_stride, e->xch_half, e->xch_flags_off, step, step, e->xch_world,
                                            e->xch_rank, e->side_stream, &cuda_err, false);
  if (launched < 0) {
    rc = fail_cuda(e, (cudaError_t)cuda_err);
  } else {
    e->launches += (uint64_t)launched;
    const uint8_t* half = static_cast<const uint8_t*>(e->xch.p) + (step % 3ull) * e->xch_half;
    rc = place_locked(e, reinterpret_cast<const lwse_place_req*>(half + e->xch_reqs_off),
                      e->xch_world * e->xch_reqs_per_part, reinterpret_cast<const uint32_t*>(half), n_namespaces,
                      d_place_out, nullptr, e->side_stream, e->xch_world, e->xch_reqs_per_part, e->xch_stride,
                      /*after_push=*/true);
  }
  if (rc == LWSE_OK && t) rc = sweep_device_locked(e, t, s);
  cudaError_t je = cudaEventRecord(e->ev_join, e->side_stream);
  if (je == cudaSuccess) je = cudaStreamWaitEvent(s, e->ev_join, 0);
  if (rc != LWSE_OK) return rc;
  if (je != cudaSuccess) return fail_cuda(e, je);
  return LWSE_OK;
}

// The placement branch of a tick whose requests are LOCAL and whose occupancy is shared: push this
// rank's occupancy counters to every peer, then solve the local requests against the sum of all
// ranks' counters.  Enqueued on `ps`.  lagged: read the previous step's snapshot (see the kernel file).
static int shared_occupancy_place_locked(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                                         const uint32_t* d_local_occ, uint32_t n_namespaces, lwse_place_out* d_out,
                                         uint32_t form, bool lagged, cudaStream_t ps,
                                         const lwse::PlaceNsChanges* changes = nullptr) {
  // While a tick graph is being captured the step is not a parameter: the push kernel takes it from
  // the device counter every push advances (and the condense kernel the blocks to sum from the same
  // counter), so that the replayed nodes follow the step; the replay itself advances e->xch_step.
  cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
  const bool eager = cudaStreamIsCapturing(ps, &capturing) == cudaSuccess && capturing == cudaStreamCaptureStatusNone;
  const uint64_t step = eager ? ++e->xch_step : 0ull;
  const uint64_t read_step = (lagged && step > 1) ? step - 1 : step;
  int cuda_err = 0;
  int launched = lwse::launch_exchange_push(d_local_occ, (uint8_t* const*)e->xch_peers_dev.p, e->xch.p,
                                            e->xch_reqs_off,  // the occupancy block of a part: n_nodes counters, 16-byte padded
                                            e->xch_stride, e->xch_half, e->xch_flags_off, step, read_step, e->xch_world,
                                            e->xch_rank, ps, &cuda_err, lagged);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  if (n_reqs == 0) return LWSE_OK;
  const lwse::PlaceNsExchange xch{reinterpret_cast<const unsigned long long*>(static_cast<const uint8_t*>(e->xch.p) + e->xch_flags_off +
                                                                              (uint64_t)e->xch_world * 8u + 16u),
                                  e->xch_half, lagged};
  if (form != kFormGeneral && lwse::place_ns_supported(e->n_nodes, e->n_domains))
    return place_grouped_locked(e, d_reqs, n_reqs, static_cast<const uint32_t*>(e->xch.p), e->xch_world, e->xch_stride, n_namespaces,
                                d_out, form == kFormScan, nullptr, nullptr, ps, /*first_pdl=*/true, changes, &xch);  // behind the push kernel
  return LWSE_ERR_UNSUPPORTED;  // the shared-occupancy form needs a request table grouped by namespace
}

LWSE_API int lwse_reconcile_shared_device(lwse_engine* e, const lwse_lws_tables* t, const lwse_place_req* d_reqs,
                                          uint32_t n_reqs, const uint32_t* d_local_occupancy, uint32_t n_namespaces,
                                          lwse_place_out* d_place_out, uint32_t flags, void* stream) {
  if (!e || !d_local_occupancy || !aligned16(d_local_occupancy) || (n_reqs && (!d_reqs || !d_place_out)) || n_namespaces == 0)
    return LWSE_ERR_INVALID_ARG;
  int rc = t ? check_lws_tables(t) : LWSE_OK;
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->xch_connected) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
  LWSE_CUDA(e, cudaEventRecord(e->ev_fork, s));
  LWSE_CUDA(e, cudaStreamWaitEvent(e->side_stream, e->ev_fork, 0));
  rc = shared_occupancy_place_locked(e, d_reqs, n_reqs, d_local_occupancy, n_namespaces, d_place_out,
                                     (flags & LWSE_SWEEP_PLACE_SCAN) ? kFormScan : kFormGrouped,
                                     (flags & LWSE_EXCHANGE_LAGGED) != 0, e->side_stream);
  if (rc == LWSE_OK && t) rc = sweep_device_locked(e, t, s);
  cudaError_t je = cudaEventRecord(e->ev_join, e->side_stream);
  if (je == cudaSuccess) je = cudaStreamWaitEvent(s, e->ev_join, 0);
  if (rc != LWSE_OK) return rc;
  if (je != cudaSuccess) return fail_cuda(e, je);
  return LWSE_OK;
}

// 0 = every wait so far saw all peers; 1 = a wait timed out (a peer is gone).  Synchronizes.
LWSE_API int lwse_exchange_status(lwse_engine* e, uint32_t* error_out) {
  if (!e || !error_out) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->xch_world) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  LWSE_CUDA(e, cudaDeviceSynchronize());
  LWSE_CUDA(e, cudaMemcpy(error_out, static_cast<const uint8_t*>(e->xch.p) + e->xch_flags_off + (uint64_t)e->xch_world * 8u + 4u,
                          4, cudaMemcpyDeviceToHost));
  return LWSE_OK;
}

// Tuning aid (not part of lwse.h): phase timestamps of the most recent placement kernel.
extern "C" __attribute__((visibility("default"))) int lwse_debug_place_trace(lwse_engine* e, uint64_t* out16) {
  if (!e || !out16 || !e->place_scratch.p || e->place_calls == 0) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaDeviceSynchronize();
  // the half used by the last call: layout [holder | counters …]; holder size is unknown here, so the
  // launcher recorded the counters pointer
  if (!e->place_counters) return LWSE_ERR_NOT_READY;
  uint32_t raw[32];
  if (cudaMemcpy(raw, e->place_counters + 16, sizeof(raw), cudaMemcpyDeviceToHost) != cudaSuccess)
    return LWSE_ERR_CUDA;
  for (int k = 0; k < 16; k++) out16[k] = (uint64_t)raw[2 * k] | ((uint64_t)raw[2 * k + 1] << 32);
  return LWSE_OK;
}

LWSE_API int lwse_place_host(lwse_engine* e, const lwse_place_req* reqs, uint32_t n_reqs,
                             const uint32_t* occupancy, uint32_t n_namespaces, lwse_place_out* out,
                             uint32_t* rounds_out) {
  if (!e || (n_reqs && (!reqs || !out)) || n_namespaces == 0) return LWSE_ERR_INVALID_ARG;
  // one lock for staging, launch and download: concurrent callers (Go reconcile workers) share
  // the staging buffers
  std::lock_guard<std::mutex> lock(e->mu);
  if (e->n_nodes == 0 || e->n_domains == 0) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  cudaStream_t s = e->stream;
  LWSE_CUDA(e, e->place_reqs.reserve((size_t)n_reqs * sizeof(lwse_place_req) + 16));
  LWSE_CUDA(e, e->place_out.reserve((size_t)n_reqs * sizeof(lwse_place_out) + 16));
  LWSE_CUDA(e, e->place_occ.reserve((size_t)e->n_nodes * 4 + 16));
  if (n_reqs)
    LWSE_CUDA(e, cudaMemcpyAsync(e->place_reqs.p, reqs, (size_t)n_reqs * sizeof(lwse_place_req), cudaMemcpyHostToDevice, s));
  if (occupancy)
    LWSE_CUDA(e, cudaMemcpyAsync(e->place_occ.p, occupancy, (size_t)e->n_nodes * 4, cudaMemcpyHostToDevice, s));
  else
    LWSE_CUDA(e, cudaMemsetAsync(e->place_occ.p, 0, (size_t)e->n_nodes * 4, s));
  // a table grouped by namespace (the encoder emits it that way) takes the namespace-parallel kernels
  const uint32_t form = n_reqs && grouped_by_namespace(reqs, n_reqs) ? kFormGrouped : kFormGeneral;
  const int rc = place_locked(e, (const lwse_place_req*)e->place_reqs.p, n_reqs, (const uint32_t*)e->place_occ.p, n_namespaces,
                              (lwse_place_out*)e->place_out.p, rounds_out, s, 1, n_reqs, 0, false, form);
  if (rc != LWSE_OK) return rc;
  if (n_reqs)
    LWSE_CUDA(e, cudaMemcpyAsync(out, e->place_out.p, (size_t)n_reqs * sizeof(lwse_place_out), cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

// One reconcile tick from host tables: lwse_sweep_lws_host and lwse_place_host in one call.  The
// placement round (its inputs are 70 KB) is uploaded, solved and read back on the side stream
// while the tables of the sweep are still crossing PCIe; one synchronize at the end.
LWSE_API int lwse_reconcile_host(lwse_engine* e, const lwse_lws_tables* h, const lwse_place_req* reqs,
                                 uint32_t n_reqs, const uint32_t* occupancy, uint32_t n_namespaces,
                                 lwse_place_out* place_out) {
  if (!e || (n_reqs && (!reqs || !place_out || n_namespaces == 0))) return LWSE_ERR_INVALID_ARG;
  int rc = check_lws_tables(h);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  if (n_reqs && (e->n_nodes == 0 || e->n_domains == 0)) return LWSE_ERR_NOT_READY;
  // LWSE_SWEEP_PLACE_GROUPED: the caller promises a request table grouped by namespace (the encoder
  // emits it that way) — no host pass over the table; the condense kernel counts order violations
  // and a broken promise comes back as LWSE_ERR_BAD_TABLE.
  const bool promised = n_reqs && (h->flags & LWSE_SWEEP_PLACE_GROUPED) && lwse::place_ns_supported(e->n_nodes, e->n_domains);
  bool check_order = false;
  const std::function<int()> place_branch = [&]() -> int {
    if (!n_reqs) return LWSE_OK;
    cudaStream_t ps = e->side_stream;
    LWSE_CUDA(e, e->place_reqs.reserve((size_t)n_reqs * sizeof(lwse_place_req) + 16));
    LWSE_CUDA(e, e->place_out.reserve((size_t)n_reqs * sizeof(lwse_place_out) + 16));
    LWSE_CUDA(e, e->place_occ.reserve((size_t)e->n_nodes * 4 + 16));
    // (the side stream only ever runs work enqueued under this lock and joined before it is released)
    LWSE_CUDA(e, cudaMemcpyAsync(e->place_reqs.p, reqs, (size_t)n_reqs * sizeof(lwse_place_req), cudaMemcpyHostToDevice, ps));
    if (occupancy)
      LWSE_CUDA(e, cudaMemcpyAsync(e->place_occ.p, occupancy, (size_t)e->n_nodes * 4, cudaMemcpyHostToDevice, ps));
    else
      LWSE_CUDA(e, cudaMemsetAsync(e->place_occ.p, 0, (size_t)e->n_nodes * 4, ps));
    const bool grouped = promised || grouped_by_namespace(reqs, n_reqs);
    const uint32_t form = grouped ? ((h->flags & LWSE_SWEEP_PLACE_SCAN) ? kFormScan : kFormGrouped) : kFormGeneral;
    const int prc = place_locked(e, (const lwse_place_req*)e->place_reqs.p, n_reqs, (const uint32_t*)e->place_occ.p, n_namespaces,
                                 (lwse_place_out*)e->place_out.p, nullptr, ps, 1, n_reqs, 0, false, form);
    if (prc != LWSE_OK) return prc;
    if (promised && g_place_form_env != 0 && e->place_scans_ptr != nullptr) {  // (the namespace kernels ran: their counter block)
      LWSE_CUDA(e, cudaMemcpyAsync(e->h_rounds + 8, e->place_rounds_ptr + 2, 4, cudaMemcpyDeviceToHost, ps));
      check_order = true;
    }
    LWSE_CUDA(e, cudaMemcpyAsync(place_out, e->place_out.p, (size_t)n_reqs * sizeof(lwse_place_out), cudaMemcpyDeviceToHost, ps));
    return LWSE_OK;
  };
  const int rc_sweep = sweep_host_locked(e, h, &place_branch);
  if (n_reqs) {
    const cudaError_t pe = cudaStreamSynchronize(e->side_stream);
    if (rc_sweep == LWSE_OK && pe != cudaSuccess) return fail_cuda(e, pe);
    if (rc_sweep == LWSE_OK && check_order && e->h_rounds[8] != 0u) return LWSE_ERR_BAD_TABLE;
  }
  return rc_sweep;
}

// ---------------------------------------------------------------------------
// The resident tick
// ---------------------------------------------------------------------------
LWSE_API int lwse_resident_place_load(lwse_engine* e, const lwse_place_req* reqs, uint32_t n_reqs,
                                      uint32_t n_namespaces) {
  if (!e || (n_reqs && !reqs) || n_namespaces == 0 || !aligned16(reqs)) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded || e->n_nodes == 0 || e->n_domains == 0) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  {
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
    LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
  }
  cudaStream_t s = e->stream;
  const size_t b_req = (size_t)n_reqs * sizeof(lwse_place_req), b_out = (size_t)n_reqs * sizeof(lwse_place_out);
  LWSE_CUDA(e, e->r_preq.reserve(b_req + 16));
  LWSE_CUDA(e, e->r_pout.reserve(b_out + 16));
  LWSE_CUDA(e, e->r_pout_prev.reserve(b_out + 16));
  if (b_req) LWSE_CUDA(e, cudaMemcpyAsync(e->r_preq.p, reqs, b_req, cudaMemcpyHostToDevice, s));
  if (b_out) LWSE_CUDA(e, cudaMemsetAsync(e->r_pout_prev.p, 0xFF, b_out, s));  // the first tick reports every row
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  e->rn_reqs = n_reqs;
  e->rn_namespaces = n_namespaces;
  e->r_place_loaded = true;
  e->r_place_grouped = grouped_by_namespace(reqs, n_reqs);
  e->r_req_ns.resize(n_reqs);
  for (uint32_t i = 0; i < n_reqs; i++) e->r_req_ns[i] = reqs[i].ns;
  return reserve_change_lists(e);
}

static inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
  __builtin_ia32_pause();
#endif
}

// Spin until the device has raised *w to `seq` (mapped host memory).  While waiting, look at the
// stream now and then: a faulted kernel never raises the word.  false = error or 10 s without news.
static bool wait_word(volatile uint32_t* w, uint32_t seq, cudaStream_t s, cudaError_t* err) {
  *err = cudaSuccess;
  const auto t0 = std::chrono::steady_clock::now();
  for (uint64_t it = 1;; it++) {
    if (*w == seq) {
      std::atomic_thread_fence(std::memory_order_acquire);
      return true;
    }
    cpu_relax();
    if ((it & 0x3FFFu) == 0) {
      const cudaError_t q = cudaStreamQuery(s);
      if (q != cudaSuccess && q != cudaErrorNotReady) {
        *err = q;
        return false;
      }
      if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 10.0) return *w == seq;
    }
  }
}

struct TickCounts {
  uint32_t n_lws = 0, n_groups = 0, n_place = 0, rounds = 0;
  uint32_t n_ds = 0, n_roles = 0, n_revroles = 0;  // a joint tick's DS lists
};

static int enqueue_ds_sweep(lwse_engine* e, uint32_t slot, bool first, cudaStream_t s, bool pdl, lwse::PublishListHost* pl,
                            int* launched_out);

static inline uint8_t* d_desc_of(lwse_engine* e, uint32_t slot, size_t desc_bytes) {
  return static_cast<uint8_t*>(e->tdesc_dev.p) + slot * desc_bytes;
}

// Enqueue one tick (nothing waits): slot = t_submitted & 1.  At most two ticks are in flight.
// `joint` (lwse_joint_tick_submit): segs holds both parts' segments (table ids 0-7, checked by the caller) and the
// resident DS sweep runs in the tick as well; its three lists are published with the tick's.
static int tick_submit_locked(lwse_engine* e, const lwse_patch_seg* segs, uint32_t n_segs, uint32_t flags, bool joint = false) {
  if (e->t_submitted - e->t_waited >= 2) return LWSE_ERR_NOT_READY;  // wait for the oldest tick first
  const bool in_flight = e->t_submitted != e->t_waited;
  const uint32_t slot = (uint32_t)(e->t_submitted & 1u);
  cudaStream_t s = e->stream;
  uint32_t* hw_dev = static_cast<uint32_t*>(e->tickw.d) + slot * 16u;
  uint8_t* chg_d = static_cast<uint8_t*>(e->chg.d) + slot * e->chg_bytes;  // the pinned lists of this slot, as the device sees them
  uint8_t* chg_v = static_cast<uint8_t*>(e->chg_dev.p) + slot * e->chg_bytes;  // the device-memory lists (of this slot) the kernels append to
  uint32_t* cnt = static_cast<uint32_t*>(e->r_counts.p) + slot * 16u;          // and their counters
  const bool do_place = (flags & LWSE_TICK_PLACE) && e->r_place_loaded && e->rn_reqs > 0;
  const bool do_sweep = !(flags & LWSE_TICK_NO_SWEEP) && (e->rn_lws || e->rn_groups);
  if (n_segs && !segs) return LWSE_ERR_INVALID_ARG;
  // sequence numbers count the ticks that end in a publish kernel (the device counts the same ones)
  const uint32_t ids = joint ? kAllTableIds : kLwsTableIds;
  const bool ds_first = joint && e->rd_first;  // the first DS tick after lwse_ds_resident_load lists every row
  uint32_t seq = 0;
  if (do_sweep || do_place || joint) {
    seq = ++e->tick_seq;
    if (seq == 0) seq = ++e->tick_seq;
  }
  {
    const size_t ub = stage_bytes_upper_bound(segs, n_segs);
    if (ub > e->stage.cap) {  // rare: only segments outside the arena are staged
      bool all_in_arena = true;
      for (uint32_t i = 0; i < n_segs; i++)
        if (segs[i].n && !(segs[i].flags & LWSE_PATCH_RANGE) &&
            (!rows_in_place(e, segs[i]) || !e->arena.holds(segs[i].values, 1)))
          all_in_arena = false;
      if (!all_in_arena) {
        LWSE_CUDA(e, cudaStreamSynchronize(s));
        LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
        LWSE_CUDA(e, e->stage.reserve(ub));
      }
    }
  }
  // Patches go where their readers run: the placement request table is read only by the round on
  // the side stream, everything else by the sweep on the engine's stream — the round then starts
  // behind its own few rows (read in place over PCIe: no copy-engine launch) while the copy engine
  // still moves the pod patches, and is mostly done when the sweep needs the SMs.  Identity-row
  // patches move occupancy counts, which the round reads: with those in the tick it forks behind
  // the main scatter.  ONE publish kernel behind the join copies all change lists out.
  constexpr uint32_t kSideTables = 1u << LWSE_TABLE_PLACE_REQS;
  bool has_ident = false, has_side = false;
  for (uint32_t i = 0; i < n_segs; i++) {
    if (segs[i].n && segs[i].table == LWSE_TABLE_POD_IDENT) has_ident = true;
    if (segs[i].n && segs[i].table == LWSE_TABLE_PLACE_REQS) has_side = true;
  }
  bool wrote = false, wrote_side = false;
  size_t stage_used = 0;
  int rc = LWSE_OK;
  int cuda_err = 0;
  cudaStream_t ps = e->side_stream;
  // Enqueue order (every call costs 1.5-3 us of host time, and the copy of the pod patches is the
  // head of the critical path):
  //   0 (default)  copy of the pod patches; the round's launches on the side stream while the copy
  //                engine works; then the scatter and the sweep behind the copy
  //   1            the round's launches first, then copy + scatter + sweep (segments in the arena only)
  //   2            copy + scatter, the round, the sweep
  // With identity patches the round forks behind the main scatter (it reads the occupancy counters).
  bool all_in_place = true;  // no segment needs the staging buffer
  for (uint32_t i = 0; i < n_segs; i++) {
    if (!segs[i].n || (segs[i].flags & LWSE_PATCH_RANGE)) continue;
    void* tb;
    uint64_t trows;
    uint32_t rb = 0;
    if (!resident_table(e, segs[i].table, &tb, &trows, &rb, ids)) return LWSE_ERR_INVALID_ARG;
    if (!rows_in_place(e, segs[i]) || !values_in_place(e, segs[i], rb)) all_in_place = false;
  }
  int order = has_ident ? 2 : e->tick_order;
  if (order == 1 && !all_in_place) order = 0;  // (the two calls share the staging buffer: main part first)
  if (in_flight) {
    // a tick is still running.  Its DMA may still read the staging buffer: segments outside the arena
    // wait for it.  Its publish kernel (the last thing on the engine's stream) still has to copy and
    // reset the placement change list the side stream appends to: the side stream starts behind it.
    if (!all_in_place) {
      LWSE_CUDA(e, cudaStreamSynchronize(s));
      LWSE_CUDA(e, cudaStreamSynchronize(ps));
    }
    // the general placement kernel keeps its counters in two alternating scratch halves (a call resets
    // the half the next one uses): its round may not start before the previous tick's publish kernel
    // has read them.  (The namespace kernels count in the tick slot's own block.)
    if (do_place && !(e->r_place_grouped && g_place_form_env != 0 && lwse::place_ns_supported(e->n_nodes, e->n_domains)))
      LWSE_CUDA(e, cudaStreamWaitEvent(ps, e->ev_pub, 0));
  }
  ScatterPlan main_plan;
  auto apply_main = [&](bool defer) -> int {
    return apply_patches_locked(e, segs, n_segs, &wrote, ~kSideTables, s, 0, &stage_used, 0, defer ? &main_plan : nullptr, false,
                                ids);
  };
  auto apply_side = [&]() -> int {
    if (has_ident && wrote && (has_side || do_place)) {
      LWSE_CUDA(e, cudaEventRecord(e->ev_fork, s));
      LWSE_CUDA(e, cudaStreamWaitEvent(ps, e->ev_fork, 0));
    }
    if (!has_side) return LWSE_OK;
    return apply_patches_locked(e, segs, n_segs, &wrote_side, kSideTables, ps, stage_used, nullptr, /*dma_min_bytes=*/65536, nullptr,
                                false, ids);
  };
  lwse::PublishListHost pl[6] = {};  // [0..2] the LWS tick's lists, [3..5] a joint tick's DS lists
  int sweep_first_mode = -1;      // -1: 2 behind this tick's scatter kernel, else 1 (see launch_lws_sweep)
  bool place_first_pdl = true;    // the round's first kernel follows a kernel on the side stream
  void* place_mid_event = nullptr;  // (graph capture) recorded between the condense and the namespace kernel
  auto enqueue_sweep = [&]() -> int {
    lwse_lws_tables d{};
    d.lws = (const lwse_lws_rec*)e->r_lws.p;
    d.n_lws = e->rn_lws;
    d.groups = (const lwse_group_rec*)e->r_groups.p;
    d.n_groups = e->rn_groups;
    d.pod_state = (const lwse_pod_state*)e->r_pst.p;
    d.pod_ident = (const lwse_pod_ident*)e->r_pid.p;
    d.n_pods = e->rn_pods;
    d.lws_out = (lwse_lws_out*)e->r_lws_out.p;
    d.group_out = (lwse_group_out*)e->r_group_out.p;
    d.flags = flags & LWSE_SWEEP_GANG;
    lwse::SweepChangeLists cl;
    cl.lws_rows = reinterpret_cast<uint32_t*>(chg_v + e->chg_off[0]);
    cl.lws_out = reinterpret_cast<lwse_lws_out*>(chg_v + e->chg_off[1]);
    cl.lws_capacity = e->rn_lws;
    cl.group_rows = reinterpret_cast<uint32_t*>(chg_v + e->chg_off[2]);
    cl.group_out = reinterpret_cast<lwse_group_out*>(chg_v + e->chg_off[3]);
    cl.group_capacity = e->rn_groups;
    cl.counts = cnt;
    int launched = lwse::launch_lws_sweep(&d, (const lwse_node_rec*)e->nodes.p, e->n_nodes, e->r_scan.p, e->sm_count, s,
                                          &cuda_err, &cl, nullptr, sweep_first_mode >= 0 ? sweep_first_mode : (wrote ? 2 : 1));
    if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
    e->launches += (uint64_t)launched;
    pl[0] = {cl.lws_rows, cl.lws_out, reinterpret_cast<uint32_t*>(chg_d + e->chg_off[0]), chg_d + e->chg_off[1],
             cnt + 0, e->rn_lws, (uint32_t)sizeof(lwse_lws_out)};
    pl[1] = {cl.group_rows, cl.group_out, reinterpret_cast<uint32_t*>(chg_d + e->chg_off[2]), chg_d + e->chg_off[3],
             cnt + 1, e->rn_groups, (uint32_t)sizeof(lwse_group_out)};
    return LWSE_OK;
  };
  auto enqueue_place = [&]() -> int {
    const uint32_t form = !e->r_place_grouped ? kFormGeneral : (flags & LWSE_SWEEP_PLACE_SCAN) ? kFormScan : kFormGrouped;
    // the namespace kernels append the changed rows themselves; the general form gets a diff kernel
    const lwse::PlaceNsChanges changes{(lwse_place_out*)e->r_pout_prev.p, reinterpret_cast<uint32_t*>(chg_v + e->chg_off[4]),
                                       reinterpret_cast<lwse_place_out*>(chg_v + e->chg_off[5]), cnt + 4, e->rn_reqs, (int)slot,
                                       place_mid_event};
    bool diffed = false;
    if (flags & LWSE_TICK_SHARED_OCCUPANCY) {  // multi-rank: this rank's counters go to the peers, the round sees the sum
      if (!e->xch_connected) return LWSE_ERR_NOT_READY;
      rc = shared_occupancy_place_locked(e, (const lwse_place_req*)e->r_preq.p, e->rn_reqs, (const uint32_t*)e->r_occ.p,
                                         e->rn_namespaces, (lwse_place_out*)e->r_pout.p, form,
                                         (flags & LWSE_EXCHANGE_LAGGED) != 0, ps, &changes);
      diffed = rc == LWSE_OK;
    } else {
      rc = place_locked(e, (const lwse_place_req*)e->r_preq.p, e->rn_reqs, (const uint32_t*)e->r_occ.p, e->rn_namespaces,
                        (lwse_place_out*)e->r_pout.p, nullptr, ps, 1, e->rn_reqs, 0, false, form, place_first_pdl, &changes,
                        &diffed);
    }
    if (rc != LWSE_OK) return rc;
    if (!diffed) {
      int launched = lwse::launch_place_diff((const lwse_place_out*)e->r_pout.p, changes.prev, e->rn_reqs, changes.rows,
                                             changes.outs, changes.capacity, changes.count, ps, &cuda_err);
      if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
      e->launches += (uint64_t)launched;
    }
    pl[2] = {changes.rows, changes.outs, reinterpret_cast<uint32_t*>(chg_d + e->chg_off[4]), chg_d + e->chg_off[5], changes.count,
             e->rn_reqs, (uint32_t)sizeof(lwse_place_out)};
    e->tick_place_ns = diffed;
    return LWSE_OK;
  };
  // The tick's last step, on the publish stream: behind everything the tick enqueued on the engine's
  // stream (both branches joined there), so the NEXT tick's kernels do not wait for the copy of this
  // tick's changed rows to the host.  Lists, counters and the round's counter block are per slot.
  auto enqueue_publish = [&]() -> int {
    LWSE_CUDA(e, cudaEventRecord(e->ev_done, s));
    LWSE_CUDA(e, cudaStreamWaitEvent(e->pub_stream, e->ev_done, 0));
    const bool ns_counters = do_place && e->tick_place_ns;
    int launched = joint ? lwse::launch_publish_joint(pl, do_place ? e->place_rounds_ptr : nullptr, hw_dev, 4, seq, cnt + 2,
                                                      e->last_changed[0] + e->last_changed[1], e->pub_stream, &cuda_err,
                                                      ns_counters ? const_cast<uint32_t*>(e->place_rounds_ptr) : nullptr, 8u)
                         : lwse::launch_publish(pl, do_place ? e->place_rounds_ptr : nullptr, hw_dev, 4, seq, cnt + 2,
                                                e->last_changed[0] + e->last_changed[1], e->pub_stream, &cuda_err,
                                                ns_counters ? const_cast<uint32_t*>(e->place_rounds_ptr) : nullptr, 8u, /*pdl=*/false);
    if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
    e->launches += (uint64_t)launched;
    LWSE_CUDA(e, cudaEventRecord(e->ev_pub, e->pub_stream));
    return LWSE_OK;
  };
  // ---- replay as a CUDA graph --------------------------------------------------------------
  // Enqueueing a tick kernel by kernel costs ~10 runtime calls of 2-4 us each (launches with
  // attributes and 200-400 bytes of parameters): more host time than the GPU needs for the tick.
  // A tick whose patches lie in the arena is therefore replayed as ONE graph per (shape of the
  // tick, slot):   scatter -> condense -> { fused -> LWS pass  ||  namespace kernel }.
  // What changes from tick to tick travels outside the graph, on the copy stream, so that the
  // copies of tick k+1 overlap the kernels of tick k: the patch bytes (arena span -> mirror) and
  // the scatter's segment descriptors (a 512-byte block, pinned slot -> device).  The publish
  // kernel follows on the publish stream, launched with the tick's sequence number.
  bool any_range = false;
  for (uint32_t i = 0; i < n_segs; i++)
    if (segs[i].n && (segs[i].flags & LWSE_PATCH_RANGE)) any_range = true;
  // (LWSE_TICK_GRAPH: 1 = replay when the previous tick is still in flight — the pipelined use, where the
  //  host's enqueue time is what limits the rate; a lone tick is faster kernel by kernel, because its
  //  round starts while the copy engine still moves the pod patches; 2 = always; 0 = never)
  const bool shared_occ = (flags & LWSE_TICK_SHARED_OCCUPANCY) != 0;
  const bool graph_ok = !joint && (e->use_graph >= 2 || (e->use_graph == 1 && in_flight)) && all_in_place && !any_range &&
                        (!shared_occ || (do_place && e->xch_connected)) &&
                        (do_sweep || do_place) && !(has_side && !do_place) &&
                        (!do_place || (e->r_place_grouped && g_place_form_env != 0 && lwse::place_ns_supported(e->n_nodes, e->n_domains)));
  if (graph_ok) {
    bool has_patches = false;
    for (uint32_t i = 0; i < n_segs; i++)
      if (segs[i].n) has_patches = true;
    const uint32_t key = (has_patches ? 1u : 0u) | (do_sweep ? 8u : 0u) | (do_place ? 16u : 0u) |
                         ((flags & LWSE_SWEEP_GANG) ? 32u : 0u) | ((flags & LWSE_SWEEP_PLACE_SCAN) ? 64u : 0u) | (slot << 8) |
                         (shared_occ ? 512u : 0u) | ((shared_occ && (flags & LWSE_EXCHANGE_LAGGED)) ? 1024u : 0u);
    lwse_engine::TickGraph& tg = e->tick_graphs[key];
    bool replay = !tg.failed && tg.seen >= 1;  // the first tick of a shape runs eagerly: every buffer settles
    tg.seen++;
    ScatterPlan gp;
    if (replay) {
      bool w = false;  // one plan for every table: one scatter launch behind one copy of the arena span
      rc = apply_patches_locked(e, segs, n_segs, &w, 0xFFFFFFFFu, s, 0, nullptr, 0, &gp, /*plan_only=*/true);
      if (rc != LWSE_OK) return rc;
      if (gp.eager_only || gp.recount) replay = false;
      if (do_place && !e->r_place_grouped) replay = false;  // (a patch moved a request to another namespace)
    }
    const size_t desc_bytes = 512;
    if (replay && (lwse::scatter_desc_bytes() > desc_bytes || e->tdesc.reserve(2 * desc_bytes) != cudaSuccess ||
                   e->tdesc_dev.reserve(2 * desc_bytes) != cudaSuccess)) {
      (void)cudaGetLastError();
      replay = false;
    }
    if (replay) {
      uint8_t* h_desc = static_cast<uint8_t*>(e->tdesc.h) + slot * desc_bytes;
      uint8_t* d_desc = static_cast<uint8_t*>(e->tdesc_dev.p) + slot * desc_bytes;
      if (has_patches && !lwse::write_scatter_desc(h_desc, gp.sc, gp.n, e->n_nodes ? (uint32_t*)e->r_occ.p : nullptr, e->n_nodes))
        replay = false;
      if (replay && !tg.exec) {
        // ---- capture: the same enqueue functions, on capturing streams ----
        cudaError_t ce = cudaStreamSynchronize(s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(ps);
        if (ce != cudaSuccess) return fail_cuda(e, ce);
        const uint64_t launches_before = e->launches;
        int crc = LWSE_OK;
        ce = cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed);
        if (ce == cudaSuccess) {
          auto cap = [&](cudaError_t x) { if (crc == LWSE_OK && x != cudaSuccess) { ce = x; crc = LWSE_ERR_CUDA; } };
          if (has_patches) {  // the graph's first node: an ordinary launch
            int err = 0;
            const int launched = lwse::launch_scatter_desc(d_desc, e->sm_count, s, /*pdl=*/false, &err);
            if (launched < 0) cap((cudaError_t)err); else e->launches += (uint64_t)launched;
          }
          if (do_place) {  // the round forks behind the scatter (it reads the request rows and the occupancy counters)
            cap(cudaEventRecord(e->ev_fork, s));
            cap(cudaStreamWaitEvent(ps, e->ev_fork, 0));
            place_first_pdl = false;  // (behind an event: an ordinary launch)
            // The fused sweep kernel fills every SM (3 CTAs of 256 x 77 registers) the moment it starts
            // and the namespace kernel's CTAs (512 x 53 registers) then wait for CTAs to retire: hold
            // the sweep back until the (short) condense kernel is done, so that both reach the SMs together.
            place_mid_event = do_sweep ? (void*)e->ev_mid : nullptr;
            if (crc == LWSE_OK) crc = enqueue_place();
            if (do_sweep && e->tick_place_ns) cap(cudaStreamWaitEvent(s, e->ev_mid, 0));
            place_mid_event = nullptr;
          }
          // behind the scatter kernel alone: programmatic, waits at its top; behind an event / first node: ordinary
          sweep_first_mode = (has_patches && !(do_place && e->tick_place_ns)) ? 2 : 0;
          if (crc == LWSE_OK && do_sweep) crc = enqueue_sweep();
          if (do_place) {
            cap(cudaEventRecord(e->ev_join, ps));
            cap(cudaStreamWaitEvent(s, e->ev_join, 0));
          }
          cudaGraph_t graph = nullptr;
          const cudaError_t ee = cudaStreamEndCapture(s, &graph);
          if (ee != cudaSuccess || graph == nullptr) cap(ee != cudaSuccess ? ee : cudaErrorUnknown);
          if (crc == LWSE_OK) cap(cudaGraphInstantiate(&tg.exec, graph, 0));
          if (graph) cudaGraphDestroy(graph);
        } else {
          crc = LWSE_ERR_CUDA;
        }
        tg.kernels = (uint32_t)(e->launches - launches_before);
        e->launches = launches_before;
        sweep_first_mode = -1;
        place_first_pdl = true;
        if (crc != LWSE_OK || !tg.exec) {  // this shape stays eager; the streams are usable again after EndCapture
          (void)cudaGetLastError();
          if (tg.exec) cudaGraphExecDestroy(tg.exec);
          tg.exec = nullptr;
          tg.failed = true;
          replay = false;
          pl[0] = pl[1] = pl[2] = lwse::PublishListHost{};
        } else {
          tg.place_ns = e->tick_place_ns;
          tg.rounds_ptr = e->place_rounds_ptr;
        }
      }
    }
    if (replay) {
      if (has_patches) {  // patch bytes (arena span -> mirror) and the descriptor block, on the copy stream
        if (gp.dma)
          LWSE_CUDA(e, cudaMemcpyAsync(static_cast<uint8_t*>(e->arena_mirror.p) + gp.lo, static_cast<const uint8_t*>(e->arena.h) + gp.lo,
                                       gp.hi - gp.lo, cudaMemcpyHostToDevice, e->copy_stream));
        LWSE_CUDA(e, cudaMemcpyAsync(d_desc_of(e, slot, desc_bytes), static_cast<uint8_t*>(e->tdesc.h) + slot * desc_bytes, desc_bytes,
                                     cudaMemcpyHostToDevice, e->copy_stream));
        LWSE_CUDA(e, cudaEventRecord(e->ev_dma, e->copy_stream));
        LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_dma, 0));
      }
      LWSE_CUDA(e, cudaGraphLaunch(tg.exec, s));
      e->launches += tg.kernels;
      e->graph_ticks++;
      if (shared_occ) e->xch_step++;  // (the replayed push kernel advanced the device counter by one)
      if (!pl[0].count && do_sweep) {  // (replayed without capturing: the lists the graph's kernels append to)
        pl[0] = {reinterpret_cast<uint32_t*>(chg_v + e->chg_off[0]), chg_v + e->chg_off[1], reinterpret_cast<uint32_t*>(chg_d + e->chg_off[0]),
                 chg_d + e->chg_off[1], cnt + 0, e->rn_lws, (uint32_t)sizeof(lwse_lws_out)};
        pl[1] = {reinterpret_cast<uint32_t*>(chg_v + e->chg_off[2]), chg_v + e->chg_off[3], reinterpret_cast<uint32_t*>(chg_d + e->chg_off[2]),
                 chg_d + e->chg_off[3], cnt + 1, e->rn_groups, (uint32_t)sizeof(lwse_group_out)};
      }
      if (!pl[2].count && do_place)
        pl[2] = {reinterpret_cast<uint32_t*>(chg_v + e->chg_off[4]), chg_v + e->chg_off[5], reinterpret_cast<uint32_t*>(chg_d + e->chg_off[4]),
                 chg_d + e->chg_off[5], cnt + 4, e->rn_reqs, (uint32_t)sizeof(lwse_place_out)};
      if (do_place) {
        e->tick_place_ns = tg.place_ns;
        e->place_rounds_ptr = tg.rounds_ptr;
      }
      rc = enqueue_publish();
      if (rc != LWSE_OK) return rc;
      lwse_engine::TickSlot& gts = e->tslot[slot];
      gts.seq = seq;
      gts.do_sweep = do_sweep;
      gts.do_place = do_place;
      gts.published = true;
      gts.wrote = has_patches;
      gts.joint = false;
      e->t_submitted++;
      return LWSE_OK;
    }
  }
  // A joint tick's DS sweep reads only the DS tables, which only the main scatter writes: it forks behind
  // the scatter onto its own stream and overlaps the LWS sweep; the publish waits for it.  (On its own
  // stream it measured 100 us per serial C3 + C4 pass against 114 us behind the LWS pass; DESIGN §4.)
  auto fork_ds = [&]() -> int {
    if (!joint) return LWSE_OK;
    LWSE_CUDA(e, cudaEventRecord(e->ev_ds_fork, s));
    LWSE_CUDA(e, cudaStreamWaitEvent(e->ds_stream, e->ev_ds_fork, 0));
    int n = 0;
    const int r = enqueue_ds_sweep(e, slot, ds_first, e->ds_stream, false, pl + 3, &n);
    if (r != LWSE_OK) return r;
    LWSE_CUDA(e, cudaEventRecord(e->ev_ds_join, e->ds_stream));
    return LWSE_OK;
  };
  if (order == 1) {
    rc = apply_side();
    if (rc == LWSE_OK && do_place) rc = enqueue_place();
    if (rc == LWSE_OK) rc = apply_main(false);
    if (rc == LWSE_OK) rc = fork_ds();
    if (rc == LWSE_OK && do_sweep) rc = enqueue_sweep();
  } else if (order == 0) {
    rc = apply_main(true);
    if (rc == LWSE_OK) rc = apply_side();
    if (rc == LWSE_OK && do_place && wrote) rc = enqueue_place();
    if (rc == LWSE_OK) rc = launch_scatter_plan(e, main_plan, s);
    if (rc == LWSE_OK) rc = fork_ds();
    if (rc == LWSE_OK && do_sweep) rc = enqueue_sweep();
    if (rc == LWSE_OK && do_place && !wrote) rc = enqueue_place();
  } else {
    rc = apply_main(false);
    if (rc == LWSE_OK) rc = fork_ds();
    if (rc == LWSE_OK) rc = apply_side();
    if (rc == LWSE_OK && do_place && wrote) rc = enqueue_place();
    if (rc == LWSE_OK && do_sweep) rc = enqueue_sweep();
    if (rc == LWSE_OK && do_place && !wrote) rc = enqueue_place();
  }
  if (rc == LWSE_OK && joint) LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_ds_join, 0));
  if (rc != LWSE_OK) return rc;
  if (do_place || wrote_side) {
    LWSE_CUDA(e, cudaEventRecord(e->ev_join, ps));
    LWSE_CUDA(e, cudaStreamWaitEvent(s, e->ev_join, 0));
  }
  const bool published = do_sweep || do_place || joint;
  if (published) {
    rc = enqueue_publish();
    if (rc != LWSE_OK) return rc;
  }
  lwse_engine::TickSlot& ts = e->tslot[slot];
  ts.seq = seq;
  ts.do_sweep = do_sweep;
  ts.do_place = do_place;
  ts.published = published;
  ts.wrote = wrote || wrote_side;
  ts.joint = joint;
  if (joint) e->rd_first = false;
  e->t_submitted++;
  return LWSE_OK;
}

// The oldest tick in flight: spin on its sequence word (the tick's only wait), report its counts.
static int tick_wait_locked(lwse_engine* e, TickCounts* out, uint32_t* slot_out) {
  if (e->t_submitted == e->t_waited) return LWSE_ERR_NOT_READY;
  const uint32_t slot = (uint32_t)(e->t_waited & 1u);
  const lwse_engine::TickSlot ts = e->tslot[slot];
  cudaStream_t s = e->stream;
  volatile uint32_t* hw = static_cast<volatile uint32_t*>(e->tickw.h) + slot * 16u;
  cudaError_t werr = cudaSuccess;
  bool ok = true;
  if (ts.published) {
    ok = wait_word(hw + 4, ts.seq, s, &werr);
  } else if (ts.wrote) {
    werr = cudaStreamSynchronize(s);
    ok = werr == cudaSuccess;
  }
  e->t_waited++;
  if (!ok) {
    const cudaError_t a = cudaStreamSynchronize(s), b = cudaStreamSynchronize(e->side_stream);
    e->t_waited = e->t_submitted;  // whatever else was in flight died with it
    return fail_cuda(e, werr != cudaSuccess ? werr : a != cudaSuccess ? a : b != cudaSuccess ? b : cudaErrorUnknown);
  }
  if (ts.do_place && e->t_submitted == e->t_waited) e->place_pending = false;  // the publish kernel ran behind the join: the round is complete
  out->n_lws = ts.do_sweep ? hw[0] : 0u;
  out->n_groups = ts.do_sweep ? hw[1] : 0u;
  out->n_place = ts.do_place ? hw[2] : 0u;
  out->rounds = ts.do_place ? hw[3] : 0u;
  out->n_ds = ts.joint ? hw[5] : 0u;
  out->n_roles = ts.joint ? hw[6] : 0u;
  out->n_revroles = ts.joint ? hw[7] : 0u;
  e->last_changed[0] = out->n_lws + out->n_groups + out->n_ds + out->n_roles + out->n_revroles;
  if (ts.joint) e->rd_last_changed = out->n_ds + out->n_roles + out->n_revroles;  // (sizes lwse_ds_resident_tick's publish grid)
  e->last_changed[1] = out->n_place;
  if (slot_out) *slot_out = slot;
  return LWSE_OK;
}

static void fill_tick_outputs(const lwse_engine* e, uint32_t slot, const TickCounts& c, lwse_tick* t) {
  const uint8_t* base = static_cast<const uint8_t*>(e->chg.h) + slot * e->chg_bytes;
  t->lws_rows = reinterpret_cast<const uint32_t*>(base + e->chg_off[0]);
  t->lws_out = reinterpret_cast<const lwse_lws_out*>(base + e->chg_off[1]);
  t->group_rows = reinterpret_cast<const uint32_t*>(base + e->chg_off[2]);
  t->group_out = reinterpret_cast<const lwse_group_out*>(base + e->chg_off[3]);
  t->place_rows = reinterpret_cast<const uint32_t*>(base + e->chg_off[4]);
  t->place_out = reinterpret_cast<const lwse_place_out*>(base + e->chg_off[5]);
  t->n_lws = c.n_lws;
  t->n_groups = c.n_groups;
  t->n_place = c.n_place;
  t->place_rounds = c.rounds;
}

// Every tick in flight is waited for (its results are dropped): the synchronous entry points call this first.
static int drain_ticks_locked(lwse_engine* e) {
  while (e->t_submitted != e->t_waited) {
    TickCounts c;
    const int rc = tick_wait_locked(e, &c, nullptr);
    if (rc != LWSE_OK) return rc;
  }
  return LWSE_OK;
}

LWSE_API int lwse_resident_tick(lwse_engine* e, lwse_tick* t) {
  if (!e || !t || (t->n_segs && !t->segs)) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  int rc = drain_ticks_locked(e);
  if (rc != LWSE_OK) return rc;
  rc = tick_submit_locked(e, t->segs, t->n_segs, t->flags);
  if (rc != LWSE_OK) return rc;
  TickCounts c;
  uint32_t slot = 0;
  rc = tick_wait_locked(e, &c, &slot);
  if (rc != LWSE_OK) return rc;
  fill_tick_outputs(e, slot, c, t);
  return LWSE_OK;
}

LWSE_API int lwse_resident_tick_submit(lwse_engine* e, const lwse_tick* t) {
  if (!e || !t || (t->n_segs && !t->segs)) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  return tick_submit_locked(e, t->segs, t->n_segs, t->flags);
}

LWSE_API int lwse_resident_tick_wait(lwse_engine* e, lwse_tick* t) {
  if (!e || !t) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  // a joint tick at the head of the ring stays in flight: only lwse_joint_tick_wait reports its DS lists
  if (e->t_submitted != e->t_waited && e->tslot[e->t_waited & 1u].joint) return LWSE_ERR_INVALID_ARG;
  DeviceGuard guard(e->device);
  TickCounts c;
  uint32_t slot = 0;
  const int rc = tick_wait_locked(e, &c, &slot);
  if (rc != LWSE_OK) return rc;
  fill_tick_outputs(e, slot, c, t);
  return LWSE_OK;
}

// The earlier form of the tick: no patches, no placement, results copied to the caller's arrays.
LWSE_API int lwse_resident_sweep(lwse_engine* e, uint32_t flags, lwse_changes* ch) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  if (ch && ((ch->lws_capacity && (!ch->lws_rows || !ch->lws_out)) || (ch->group_capacity && (!ch->group_rows || !ch->group_out))))
    return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  TickCounts c;
  uint32_t slot = 0;
  int rc = drain_ticks_locked(e);
  if (rc == LWSE_OK) rc = tick_submit_locked(e, nullptr, 0, flags & LWSE_SWEEP_GANG);
  if (rc == LWSE_OK) rc = tick_wait_locked(e, &c, &slot);
  if (rc != LWSE_OK || !ch) return rc;
  ch->n_lws = c.n_lws;
  ch->n_groups = c.n_groups;
  const uint32_t nl = c.n_lws < ch->lws_capacity ? c.n_lws : ch->lws_capacity;
  const uint32_t ng = c.n_groups < ch->group_capacity ? c.n_groups : ch->group_capacity;
  const uint8_t* base = static_cast<const uint8_t*>(e->chg.h) + slot * e->chg_bytes;
  if (nl) {
    memcpy(ch->lws_rows, base + e->chg_off[0], (size_t)nl * 4);
    memcpy(ch->lws_out, base + e->chg_off[1], (size_t)nl * sizeof(lwse_lws_out));
  }
  if (ng) {
    memcpy(ch->group_rows, base + e->chg_off[2], (size_t)ng * 4);
    memcpy(ch->group_out, base + e->chg_off[3], (size_t)ng * sizeof(lwse_group_out));
  }
  return LWSE_OK;
}

LWSE_API int lwse_resident_place_outputs(lwse_engine* e, lwse_place_out* out) {
  if (!e || !out) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_place_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  LWSE_CUDA(e, cudaStreamSynchronize(e->side_stream));
  if (e->rn_reqs)
    LWSE_CUDA(e, cudaMemcpy(out, e->r_pout.p, (size_t)e->rn_reqs * sizeof(lwse_place_out), cudaMemcpyDeviceToHost));
  return LWSE_OK;
}

LWSE_API int lwse_resident_occupancy(lwse_engine* e, uint32_t* occupancy_out) {
  if (!e || !occupancy_out) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->r_loaded || e->n_nodes == 0) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  LWSE_CUDA(e, cudaStreamSynchronize(e->stream));
  LWSE_CUDA(e, cudaMemcpy(occupancy_out, e->r_occ.p, (size_t)e->n_nodes * 4, cudaMemcpyDeviceToHost));
  return LWSE_OK;
}

// ---------------------------------------------------------------------------
// DisaggregatedSet sweep
// ---------------------------------------------------------------------------
static int check_ds_tables(const lwse_ds_tables* t) {
  if (!t) return LWSE_ERR_INVALID_ARG;
  if (t->n_ds && (!t->ds || !t->ds_out)) return LWSE_ERR_INVALID_ARG;
  if (t->n_roles && (!t->roles || !t->role_out)) return LWSE_ERR_INVALID_ARG;
  if (t->n_revroles && (!t->revroles || !t->revrole_out)) return LWSE_ERR_INVALID_ARG;
  if (!aligned16(t->ds) || !aligned16(t->roles) || !aligned16(t->revroles)) return LWSE_ERR_INVALID_ARG;
  return LWSE_OK;
}

LWSE_API int lwse_sweep_ds_device(lwse_engine* e, const lwse_ds_tables* t, void* stream) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  int rc = check_ds_tables(t);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
  int cuda_err = 0;
  int launched = lwse::launch_ds_sweep(t, e->sm_count, s, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  return LWSE_OK;
}

LWSE_API int lwse_sweep_ds_host(lwse_engine* e, const lwse_ds_tables* h) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  int rc = check_ds_tables(h);
  if (rc != LWSE_OK) return rc;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  cudaStream_t s = e->stream;
  const size_t b_ds = (size_t)h->n_ds * sizeof(lwse_ds_rec), b_ro = (size_t)h->n_roles * sizeof(lwse_ds_role_rec),
               b_rr = (size_t)h->n_revroles * sizeof(lwse_ds_revrole_rec);
  const size_t o_ds = (size_t)h->n_ds * sizeof(lwse_ds_out), o_ro = (size_t)h->n_roles * sizeof(lwse_ds_role_out),
               o_rr = (size_t)h->n_revroles * sizeof(lwse_ds_revrole_out);
  LWSE_CUDA(e, e->ds.reserve(b_ds + 16));
  LWSE_CUDA(e, e->ds_roles.reserve(b_ro + 16));
  LWSE_CUDA(e, e->ds_revroles.reserve(b_rr + 16));
  LWSE_CUDA(e, e->ds_out.reserve(o_ds + 16));
  LWSE_CUDA(e, e->ds_role_out.reserve(o_ro + 16));
  LWSE_CUDA(e, e->ds_revrole_out.reserve(o_rr + 16));
  if (b_ds) LWSE_CUDA(e, cudaMemcpyAsync(e->ds.p, h->ds, b_ds, cudaMemcpyHostToDevice, s));
  if (b_ro) LWSE_CUDA(e, cudaMemcpyAsync(e->ds_roles.p, h->roles, b_ro, cudaMemcpyHostToDevice, s));
  if (b_rr) LWSE_CUDA(e, cudaMemcpyAsync(e->ds_revroles.p, h->revroles, b_rr, cudaMemcpyHostToDevice, s));
  lwse_ds_tables d = *h;
  d.ds = (const lwse_ds_rec*)e->ds.p;
  d.roles = (const lwse_ds_role_rec*)e->ds_roles.p;
  d.revroles = (const lwse_ds_revrole_rec*)e->ds_revroles.p;
  d.ds_out = (lwse_ds_out*)e->ds_out.p;
  d.role_out = (lwse_ds_role_out*)e->ds_role_out.p;
  d.revrole_out = (lwse_ds_revrole_out*)e->ds_revrole_out.p;
  int cuda_err = 0;
  int launched = lwse::launch_ds_sweep(&d, e->sm_count, s, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  if (o_ds) LWSE_CUDA(e, cudaMemcpyAsync(h->ds_out, e->ds_out.p, o_ds, cudaMemcpyDeviceToHost, s));
  if (o_ro) LWSE_CUDA(e, cudaMemcpyAsync(h->role_out, e->ds_role_out.p, o_ro, cudaMemcpyDeviceToHost, s));
  if (o_rr) LWSE_CUDA(e, cudaMemcpyAsync(h->revrole_out, e->ds_revrole_out.p, o_rr, cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

// ---------------------------------------------------------------------------
// Resident DisaggregatedSet tables
// ---------------------------------------------------------------------------
// Enqueue the resident DS sweep of tick slot `slot` on `s` (pdl: programmatically dependent on the kernel
// before it, the patch scatter; the sweep waits at its top).  pl[0..2] receive the
// slot's three lists for the publish kernel; pl[0].count + 3 is the slot's publish ticket.
static int enqueue_ds_sweep(lwse_engine* e, uint32_t slot, bool first, cudaStream_t s, bool pdl, lwse::PublishListHost* pl,
                            int* launched_out) {
  uint8_t* chg_v = static_cast<uint8_t*>(e->rd_chg_dev.p) + slot * e->rd_chg_bytes;
  uint8_t* chg_d = static_cast<uint8_t*>(e->rd_chg.d) + slot * e->rd_chg_bytes;
  uint32_t* cnt = static_cast<uint32_t*>(e->rd_counts.p) + slot * 16u;
  lwse_ds_tables d{};
  d.ds = (const lwse_ds_rec*)e->rd_ds.p;
  d.n_ds = e->rdn_ds;
  d.roles = (const lwse_ds_role_rec*)e->rd_roles.p;
  d.n_roles = e->rdn_roles;
  d.revroles = (const lwse_ds_revrole_rec*)e->rd_revroles.p;
  d.n_revroles = e->rdn_revroles;
  lwse::DsResidentArgs r{};
  r.ds_committed = (lwse_ds_out*)e->rd_ds_out.p;
  r.role_committed = (lwse_ds_role_out*)e->rd_role_out.p;
  r.revrole_committed = (lwse_ds_revrole_out*)e->rd_revrole_out.p;
  r.role_scratch = (lwse_ds_role_out*)e->rd_role_scratch.p;
  r.revrole_scratch = (lwse_ds_revrole_out*)e->rd_revrole_scratch.p;
  r.ds_rows = reinterpret_cast<uint32_t*>(chg_v + e->rd_chg_off[0]);
  r.ds_outs = reinterpret_cast<lwse_ds_out*>(chg_v + e->rd_chg_off[1]);
  r.role_rows = reinterpret_cast<uint32_t*>(chg_v + e->rd_chg_off[2]);
  r.role_outs = reinterpret_cast<lwse_ds_role_out*>(chg_v + e->rd_chg_off[3]);
  r.revrole_rows = reinterpret_cast<uint32_t*>(chg_v + e->rd_chg_off[4]);
  r.revrole_outs = reinterpret_cast<lwse_ds_revrole_out*>(chg_v + e->rd_chg_off[5]);
  r.counts = cnt;
  r.first = first ? 1u : 0u;
  int cuda_err = 0;
  const int launched = lwse::launch_ds_resident_sweep(&d, &r, e->sm_count, s, pdl, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  *launched_out = launched;
  pl[0] = {r.ds_rows, r.ds_outs, reinterpret_cast<uint32_t*>(chg_d + e->rd_chg_off[0]), chg_d + e->rd_chg_off[1], cnt + 0, e->rdn_ds,
           (uint32_t)sizeof(lwse_ds_out)};
  pl[1] = {r.role_rows, r.role_outs, reinterpret_cast<uint32_t*>(chg_d + e->rd_chg_off[2]), chg_d + e->rd_chg_off[3], cnt + 1,
           e->rdn_roles, (uint32_t)sizeof(lwse_ds_role_out)};
  pl[2] = {r.revrole_rows, r.revrole_outs, reinterpret_cast<uint32_t*>(chg_d + e->rd_chg_off[4]), chg_d + e->rd_chg_off[5], cnt + 2,
           e->rdn_revroles, (uint32_t)sizeof(lwse_ds_revrole_out)};
  return LWSE_OK;
}

static void fill_ds_tick_outputs(const lwse_engine* e, uint32_t slot, uint32_t n_ds, uint32_t n_roles, uint32_t n_revroles,
                                 lwse_ds_tick* t) {
  const uint8_t* base = static_cast<const uint8_t*>(e->rd_chg.h) + slot * e->rd_chg_bytes;
  t->n_ds = n_ds < e->rdn_ds ? n_ds : e->rdn_ds;
  t->n_roles = n_roles < e->rdn_roles ? n_roles : e->rdn_roles;
  t->n_revroles = n_revroles < e->rdn_revroles ? n_revroles : e->rdn_revroles;
  t->ds_rows = reinterpret_cast<const uint32_t*>(base + e->rd_chg_off[0]);
  t->ds_out = reinterpret_cast<const lwse_ds_out*>(base + e->rd_chg_off[1]);
  t->role_rows = reinterpret_cast<const uint32_t*>(base + e->rd_chg_off[2]);
  t->role_out = reinterpret_cast<const lwse_ds_role_out*>(base + e->rd_chg_off[3]);
  t->revrole_rows = reinterpret_cast<const uint32_t*>(base + e->rd_chg_off[4]);
  t->revrole_out = reinterpret_cast<const lwse_ds_revrole_out*>(base + e->rd_chg_off[5]);
}

LWSE_API int lwse_ds_resident_load(lwse_engine* e, const lwse_ds_tables* h) {
  if (!e || !h) return LWSE_ERR_INVALID_ARG;
  if ((h->n_ds && !h->ds) || (h->n_roles && !h->roles) || (h->n_revroles && !h->revroles)) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  {
    const int drc = drain_ticks_locked(e);
    if (drc != LWSE_OK) return drc;
  }
  cudaStream_t s = e->stream;
  LWSE_CUDA(e, cudaStreamSynchronize(s));  // (the previous DS tick's publish kernel is done with the lists)
  LWSE_CUDA(e, cudaStreamSynchronize(e->pub_stream));  // (so is a joint tick's)
  e->rd_loaded = false;
  const size_t b_ds = (size_t)h->n_ds * sizeof(lwse_ds_rec), b_ro = (size_t)h->n_roles * sizeof(lwse_ds_role_rec),
               b_rr = (size_t)h->n_revroles * sizeof(lwse_ds_revrole_rec);
  const size_t o_ds = (size_t)h->n_ds * sizeof(lwse_ds_out), o_ro = (size_t)h->n_roles * sizeof(lwse_ds_role_out),
               o_rr = (size_t)h->n_revroles * sizeof(lwse_ds_revrole_out);
  LWSE_CUDA(e, e->rd_ds.reserve(b_ds + 16));
  LWSE_CUDA(e, e->rd_roles.reserve(b_ro + 16));
  LWSE_CUDA(e, e->rd_revroles.reserve(b_rr + 16));
  LWSE_CUDA(e, e->rd_ds_out.reserve(o_ds + 16));
  LWSE_CUDA(e, e->rd_role_out.reserve(o_ro + 16));
  LWSE_CUDA(e, e->rd_revrole_out.reserve(o_rr + 16));
  LWSE_CUDA(e, e->rd_role_scratch.reserve(o_ro + 16));
  LWSE_CUDA(e, e->rd_revrole_scratch.reserve(o_rr + 16));
  size_t off = 0;
  const size_t sizes[6] = {(size_t)h->n_ds * 4, o_ds, (size_t)h->n_roles * 4, o_ro, (size_t)h->n_revroles * 4, o_rr};
  for (int k = 0; k < 6; k++) {
    e->rd_chg_off[k] = off;
    off += align256(sizes[k] + 16);
  }
  e->rd_chg_bytes = off;
  LWSE_CUDA(e, e->rd_chg_dev.reserve(2 * off));  // two tick slots (joint ticks in flight)
  LWSE_CUDA(e, e->rd_chg.reserve(2 * off));
  LWSE_CUDA(e, e->rd_counts.reserve(128));
  LWSE_CUDA(e, e->rd_tickw.reserve(64));
  LWSE_CUDA(e, cudaMemsetAsync(e->rd_counts.p, 0, 128, s));
  // the ring's tick words and per-slot counters (publish ticket): a DS-only joint tick uses them on an
  // engine that never called lwse_resident_load (which resets the counters itself)
  if (!e->r_counts.p) {
    LWSE_CUDA(e, e->r_counts.reserve(128));
    LWSE_CUDA(e, cudaMemsetAsync(e->r_counts.p, 0, 128, s));
  }
  LWSE_CUDA(e, e->tickw.reserve(256));
  if (b_ds) LWSE_CUDA(e, cudaMemcpyAsync(e->rd_ds.p, h->ds, b_ds, cudaMemcpyHostToDevice, s));
  if (b_ro) LWSE_CUDA(e, cudaMemcpyAsync(e->rd_roles.p, h->roles, b_ro, cudaMemcpyHostToDevice, s));
  if (b_rr) LWSE_CUDA(e, cudaMemcpyAsync(e->rd_revroles.p, h->revroles, b_rr, cudaMemcpyHostToDevice, s));
  if (o_ds) LWSE_CUDA(e, cudaMemsetAsync(e->rd_ds_out.p, 0, o_ds, s));  // committed values start at zero bytes
  if (o_ro) LWSE_CUDA(e, cudaMemsetAsync(e->rd_role_out.p, 0, o_ro, s));
  if (o_rr) LWSE_CUDA(e, cudaMemsetAsync(e->rd_revrole_out.p, 0, o_rr, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  e->rdn_ds = h->n_ds;
  e->rdn_roles = h->n_roles;
  e->rdn_revroles = h->n_revroles;
  e->rd_last_changed = 0;
  e->rd_first = true;
  e->rd_loaded = true;
  return LWSE_OK;
}

LWSE_API int lwse_ds_resident_tick(lwse_engine* e, lwse_ds_tick* t) {
  if (!e || !t || (t->n_segs && !t->segs) || t->n_segs > LWSE_TICK_MAX_SEGS || t->flags != 0) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->rd_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  int rc = drain_ticks_locked(e);
  if (rc != LWSE_OK) return rc;
  cudaStream_t s = e->stream;
  bool wrote = false;
  rc = apply_patches_locked(e, t->segs, t->n_segs, &wrote, 0xFFFFFFFFu, s, 0, nullptr, 0, nullptr, false, kDsTableIds);
  if (rc != LWSE_OK) return rc;
  lwse::PublishListHost pl[3];
  // behind the scatter kernel: programmatically dependent, the sweep waits at its top
  int launched = 0;
  rc = enqueue_ds_sweep(e, 0, e->rd_first, s, wrote, pl, &launched);
  if (rc != LWSE_OK) return rc;
  uint32_t seq = ++e->rd_seq;
  if (seq == 0) seq = ++e->rd_seq;
  int cuda_err = 0;
  launched = lwse::launch_publish(pl, nullptr, static_cast<uint32_t*>(e->rd_tickw.d), 4, seq, pl[0].count + 3, e->rd_last_changed,
                                  s, &cuda_err, nullptr, 0, /*pdl=*/launched > 0);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  volatile uint32_t* hw = static_cast<volatile uint32_t*>(e->rd_tickw.h);
  cudaError_t werr = cudaSuccess;
  if (!wait_word(hw + 4, seq, s, &werr)) {
    const cudaError_t a = cudaStreamSynchronize(s);
    return fail_cuda(e, werr != cudaSuccess ? werr : a != cudaSuccess ? a : cudaErrorUnknown);
  }
  fill_ds_tick_outputs(e, 0, hw[0], hw[1], hw[2], t);
  e->rd_last_changed = t->n_ds + t->n_roles + t->n_revroles;
  e->rd_first = false;
  return LWSE_OK;
}

LWSE_API int lwse_ds_resident_outputs(lwse_engine* e, lwse_ds_out* ds_out, lwse_ds_role_out* role_out,
                                      lwse_ds_revrole_out* revrole_out) {
  if (!e) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  if (!e->rd_loaded) return LWSE_ERR_NOT_READY;
  DeviceGuard guard(e->device);
  int rc = drain_ticks_locked(e);
  if (rc != LWSE_OK) return rc;
  cudaStream_t s = e->stream;
  if (ds_out && e->rdn_ds)
    LWSE_CUDA(e, cudaMemcpyAsync(ds_out, e->rd_ds_out.p, (size_t)e->rdn_ds * sizeof(lwse_ds_out), cudaMemcpyDeviceToHost, s));
  if (role_out && e->rdn_roles)
    LWSE_CUDA(e, cudaMemcpyAsync(role_out, e->rd_role_out.p, (size_t)e->rdn_roles * sizeof(lwse_ds_role_out),
                                 cudaMemcpyDeviceToHost, s));
  if (revrole_out && e->rdn_revroles)
    LWSE_CUDA(e, cudaMemcpyAsync(revrole_out, e->rd_revrole_out.p, (size_t)e->rdn_revroles * sizeof(lwse_ds_revrole_out),
                                 cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

// ---------------------------------------------------------------------------
// Joint LWS + DS tick
// ---------------------------------------------------------------------------
// One part's segments, checked as the scatter would check them, before anything is enqueued: a refused
// joint tick changes nothing.
static int check_joint_part(lwse_engine* e, const lwse_patch_seg* segs, uint32_t n_segs, uint32_t ids) {
  if (n_segs > LWSE_TICK_MAX_SEGS || (n_segs && !segs)) return LWSE_ERR_INVALID_ARG;
  for (uint32_t i = 0; i < n_segs; i++) {
    const lwse_patch_seg& g = segs[i];
    void* base;
    uint64_t rows;
    uint32_t rb;
    if (!resident_table(e, g.table, &base, &rows, &rb, ids)) return LWSE_ERR_INVALID_ARG;
    if (g.n == 0) continue;
    if (!g.values || (!(g.flags & LWSE_PATCH_RANGE) && !g.rows)) return LWSE_ERR_INVALID_ARG;
    if ((g.flags & LWSE_PATCH_RANGE) && (uint64_t)g.first_row + g.n > rows) return LWSE_ERR_BAD_TABLE;
  }
  return LWSE_OK;
}

static int joint_submit_locked(lwse_engine* e, const lwse_tick* lws, const lwse_ds_tick* ds) {
  if (!e->rd_loaded || (lws && !e->r_loaded) || (lws && (lws->flags & LWSE_TICK_PLACE) && !e->r_place_loaded))
    return LWSE_ERR_NOT_READY;
  if (ds->flags != 0 || (lws && (lws->flags & LWSE_TICK_SHARED_OCCUPANCY))) return LWSE_ERR_INVALID_ARG;
  int rc = lws ? check_joint_part(e, lws->segs, lws->n_segs, kLwsTableIds) : LWSE_OK;
  if (rc == LWSE_OK) rc = check_joint_part(e, ds->segs, ds->n_segs, kDsTableIds);
  if (rc != LWSE_OK) return rc;
  if (e->t_submitted - e->t_waited >= 2) return LWSE_ERR_NOT_READY;
  lwse_patch_seg segs[2 * LWSE_TICK_MAX_SEGS];
  uint32_t n = 0;
  for (uint32_t i = 0; lws && i < lws->n_segs; i++) segs[n++] = lws->segs[i];
  for (uint32_t i = 0; i < ds->n_segs; i++) segs[n++] = ds->segs[i];
  return tick_submit_locked(e, segs, n, lws ? lws->flags : LWSE_TICK_NO_SWEEP, /*joint=*/true);
}

static int joint_wait_locked(lwse_engine* e, lwse_tick* lws, lwse_ds_tick* ds) {
  if (e->t_submitted == e->t_waited) return LWSE_ERR_NOT_READY;
  const bool joint = e->tslot[e->t_waited & 1u].joint;
  TickCounts c;
  uint32_t slot = 0;
  const int rc = tick_wait_locked(e, &c, &slot);
  if (rc != LWSE_OK) return rc;
  if (lws) fill_tick_outputs(e, slot, c, lws);
  if (joint) {
    fill_ds_tick_outputs(e, slot, c.n_ds, c.n_roles, c.n_revroles, ds);
  } else {  // an LWS tick: no DS lists
    ds->ds_rows = ds->role_rows = ds->revrole_rows = nullptr;
    ds->ds_out = nullptr;
    ds->role_out = nullptr;
    ds->revrole_out = nullptr;
    ds->n_ds = ds->n_roles = ds->n_revroles = 0;
  }
  return LWSE_OK;
}

LWSE_API int lwse_joint_tick_submit(lwse_engine* e, const lwse_tick* lws, const lwse_ds_tick* ds) {
  if (!e || !ds) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return joint_submit_locked(e, lws, ds);
}

LWSE_API int lwse_joint_tick_wait(lwse_engine* e, lwse_tick* lws, lwse_ds_tick* ds) {
  if (!e || !ds) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return joint_wait_locked(e, lws, ds);
}

LWSE_API int lwse_joint_tick(lwse_engine* e, lwse_tick* lws, lwse_ds_tick* ds) {
  if (!e || !ds) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  if (e->t_submitted != e->t_waited) return LWSE_ERR_NOT_READY;  // the ticks in flight keep their results for _wait
  int rc = joint_submit_locked(e, lws, ds);
  if (rc == LWSE_OK) rc = joint_wait_locked(e, lws, ds);
  return rc;
}

// ---------------------------------------------------------------------------
// SHA-1 group keys
// ---------------------------------------------------------------------------
static int group_keys_locked(lwse_engine* e, const uint8_t* d_bytes, const uint32_t* d_offsets, uint32_t n,
                             uint8_t* d_digests, cudaStream_t s) {
  int cuda_err = 0;
  int launched = lwse::launch_sha1(d_bytes, d_offsets, n, d_digests, e->sm_count, s, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  return LWSE_OK;
}

LWSE_API int lwse_group_keys_device(lwse_engine* e, const uint8_t* d_bytes, const uint32_t* d_offsets,
                                    uint32_t n, uint8_t* d_digests, void* stream) {
  if (!e || (n && (!d_offsets || !d_digests))) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  return group_keys_locked(e, d_bytes, d_offsets, n, d_digests, stream ? (cudaStream_t)stream : e->stream);
}

LWSE_API int lwse_group_keys_host(lwse_engine* e, const uint8_t* bytes, const uint32_t* offsets,
                                  uint32_t n, uint8_t* digests) {
  if (!e || (n && (!offsets || !digests))) return LWSE_ERR_INVALID_ARG;
  if (n == 0) return LWSE_OK;
  const size_t total = offsets[n];
  if (total && !bytes) return LWSE_ERR_INVALID_ARG;
  // one lock for staging, launch and download (concurrent webhook admissions share the buffers)
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  cudaStream_t s = e->stream;
  LWSE_CUDA(e, e->sha_bytes.reserve(total + 64));
  LWSE_CUDA(e, e->sha_offsets.reserve((size_t)(n + 1) * 4 + 16));
  LWSE_CUDA(e, e->sha_digests.reserve((size_t)n * 20 + 16));
  if (total) LWSE_CUDA(e, cudaMemcpyAsync(e->sha_bytes.p, bytes, total, cudaMemcpyHostToDevice, s));
  LWSE_CUDA(e, cudaMemcpyAsync(e->sha_offsets.p, offsets, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
  const int rc = group_keys_locked(e, (const uint8_t*)e->sha_bytes.p, (const uint32_t*)e->sha_offsets.p, n,
                                   (uint8_t*)e->sha_digests.p, s);
  if (rc != LWSE_OK) return rc;
  LWSE_CUDA(e, cudaMemcpyAsync(digests, e->sha_digests.p, (size_t)n * 20, cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

LWSE_API int lwse_subgroup_keys_device(lwse_engine* e, const uint8_t* d_bytes, const uint32_t* d_offsets, uint32_t n,
                                       const int32_t* d_pod_count, const int32_t* d_subgroup_size,
                                       const int32_t* d_worker_index, int32_t* d_index_out, uint8_t* d_digests,
                                       void* stream) {
  if (!e || (n && (!d_offsets || !d_digests || !d_pod_count || !d_subgroup_size || !d_worker_index || !d_index_out)))
    return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  int cuda_err = 0;
  int launched = lwse::launch_subgroup_keys(d_bytes, d_offsets, n, d_pod_count, d_subgroup_size, d_worker_index, d_index_out,
                                            d_digests, e->sm_count, stream ? (cudaStream_t)stream : e->stream, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  return LWSE_OK;
}

LWSE_API int lwse_subgroup_keys_host(lwse_engine* e, const uint8_t* bytes, const uint32_t* offsets, uint32_t n,
                                     const int32_t* pod_count, const int32_t* subgroup_size,
                                     const int32_t* worker_index, int32_t* index_out, uint8_t* digests) {
  if (!e || (n && (!offsets || !digests || !pod_count || !subgroup_size || !worker_index || !index_out)))
    return LWSE_ERR_INVALID_ARG;
  if (n == 0) return LWSE_OK;
  const size_t total = offsets[n];
  if (total && !bytes) return LWSE_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(e->mu);
  DeviceGuard guard(e->device);
  cudaStream_t s = e->stream;
  const size_t b_int = (size_t)n * 4;
  LWSE_CUDA(e, e->sha_bytes.reserve(total + 64));
  LWSE_CUDA(e, e->sha_offsets.reserve((size_t)(n + 1) * 4 + 16));
  LWSE_CUDA(e, e->sha_digests.reserve((size_t)n * 20 + 16));
  LWSE_CUDA(e, e->sha_ints.reserve(4 * b_int + 64));
  int32_t* d_int = static_cast<int32_t*>(e->sha_ints.p);
  if (total) LWSE_CUDA(e, cudaMemcpyAsync(e->sha_bytes.p, bytes, total, cudaMemcpyHostToDevice, s));
  LWSE_CUDA(e, cudaMemcpyAsync(e->sha_offsets.p, offsets, (size_t)(n + 1) * 4, cudaMemcpyHostToDevice, s));
  LWSE_CUDA(e, cudaMemcpyAsync(d_int, pod_count, b_int, cudaMemcpyHostToDevice, s));
  LWSE_CUDA(e, cudaMemcpyAsync(d_int + n, subgroup_size, b_int, cudaMemcpyHostToDevice, s));
  LWSE_CUDA(e, cudaMemcpyAsync(d_int + 2 * (size_t)n, worker_index, b_int, cudaMemcpyHostToDevice, s));
  int cuda_err = 0;
  int launched = lwse::launch_subgroup_keys((const uint8_t*)e->sha_bytes.p, (const uint32_t*)e->sha_offsets.p, n, d_int, d_int + n,
                                            d_int + 2 * (size_t)n, d_int + 3 * (size_t)n, (uint8_t*)e->sha_digests.p,
                                            e->sm_count, s, &cuda_err);
  if (launched < 0) return fail_cuda(e, (cudaError_t)cuda_err);
  e->launches += (uint64_t)launched;
  LWSE_CUDA(e, cudaMemcpyAsync(index_out, d_int + 3 * (size_t)n, b_int, cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaMemcpyAsync(digests, e->sha_digests.p, (size_t)n * 20, cudaMemcpyDeviceToHost, s));
  LWSE_CUDA(e, cudaStreamSynchronize(s));
  return LWSE_OK;
}

}  // extern "C"
