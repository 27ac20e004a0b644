/*
 * lwse.h — C ABI of the B200 reconcile-and-placement engine ("lwse") for the
 * LeaderWorkerSet / DisaggregatedSet controllers.
 *
 * This is the drop-in boundary for the hot path named in BASELINE.json:
 * a cgo (or any FFI) caller hands fixed-width record tables to the engine and
 * reads fixed-width result tables back.  Plain pointers and sizes only; no
 * CUDA, torch or C++ types cross this boundary.
 *
 * The reference (kubernetes-sigs/lws @ 1d9204a2) has no FFI for this path —
 * every hot function is package-private Go.  Each entry point below therefore
 * cites the reference function(s) whose arithmetic it replaces
 * (paths relative to the reference root):
 *
 *   lwse_sweep_lws_*   pkg/controllers/leaderworkerset_controller.go:280-373
 *                      (rollingUpdateParameters), :414-509 (updateConditions),
 *                      :576-641 (getReplicaStates), :643-708 (partition math),
 *                      :811-830 (stsMaxUnavailable);
 *                      pkg/controllers/pod_controller.go:100-172 (worker-sts
 *                      gating), :204-266 (handleRestartPolicy), :268-295
 *                      (workerPodBelongsToLeader), :315-336
 *                      (topologyValueFromPod), :338-362 (pendingPodsInGroup),
 *                      :434-443 (worker ordinals);
 *                      pkg/schedulerprovider/volcano_provider.go:72-83 (MinMember)
 *   lwse_place_*       build-defined placement spec over the constraints of
 *                      pkg/webhooks/pod_webhook.go:185-227 (exclusive affinity /
 *                      anti-affinity per topology domain) — the reference has no
 *                      node scoring; see DESIGN.md "Placement (parity unpinned)"
 *   lwse_sweep_ds_*    pkg/controllers/disaggregatedset/planner.go:61-352,
 *                      executor.go:199-302 (planner state / config / stability),
 *                      :330-398 (scaleDownOld), disaggregatedset_controller.go:
 *                      203-236 (cleanup predicate), service_manager.go:57-89
 *   lwse_group_keys_*  pkg/webhooks/pod_webhook.go:180-182 + pkg/utils/utils.go:39-43
 *                      (SHA-1 group / subgroup keys)
 *   lwse_subgroup_keys_*  pkg/webhooks/pod_webhook.go:249-255 (getSubGroupIndex) + :130,:151
 *                      (the subgroup key of that index)
 *
 * Conventions
 *   - All records are little-endian plain-old-data with explicit padding; every
 *     table base must be 16-byte aligned.
 *   - Every function returns LWSE_OK (0) or a negative lwse_status.  Nothing
 *     aborts.  lwse_last_cuda_error() returns the cudaError_t behind
 *     LWSE_ERR_CUDA.
 *   - The caller owns every host buffer (cgo: C.malloc / pinned pool — the
 *     engine never retains a host pointer past the call).  The engine owns its
 *     device staging memory.
 *   - An engine handle is bound to one CUDA device and runs one sweep at a time
 *     (internal mutex).  Create one per GPU.
 *   - There is no CPU fallback: if no CUDA device is usable lwse_create fails
 *     with LWSE_ERR_NO_DEVICE.
 */
#ifndef LWSE_H_
#define LWSE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LWSE_ABI_VERSION 2u

#if defined(__GNUC__)
#define LWSE_API __attribute__((visibility("default")))
#else
#define LWSE_API
#endif

/* ------------------------------------------------------------------------- */
/* Status codes                                                              */
/* ------------------------------------------------------------------------- */
typedef enum lwse_status {
  LWSE_OK = 0,
  LWSE_ERR_INVALID_ARG = -1, /* NULL / misaligned pointer, bad count            */
  LWSE_ERR_NO_DEVICE = -2,   /* no usable CUDA device (no CPU fallback exists)  */
  LWSE_ERR_CUDA = -3,        /* a CUDA call failed; see lwse_last_cuda_error    */
  LWSE_ERR_OOM = -4,         /* device or pinned allocation failed              */
  LWSE_ERR_BAD_TABLE = -5,   /* a base/count in a record points outside a table */
  LWSE_ERR_NOT_READY = -6,   /* e.g. lwse_place_* before lwse_upload_nodes      */
  LWSE_ERR_UNSUPPORTED = -7  /* e.g. more than LWSE_DS_MAX_ROLES roles          */
} lwse_status;

/* ------------------------------------------------------------------------- */
/* Input records                                                             */
/* ------------------------------------------------------------------------- */

#define LWSE_NONE 0xFFFFFFFFu           /* "no index" (unscheduled, no domain, …) */
#define LWSE_NODE_NOT_FOUND 0xFFFFFFFEu /* leader.spec.nodeName set, Node object missing */

/* One LeaderWorkerSet object (64 B).  The first 16 bytes are everything the
 * per-group kernel needs from its owner. */
typedef struct lwse_lws_rec {
  uint64_t rev_hash;  /* hash of the revisionKey handed to the reconciler
                         (leaderworkerset_controller.go:159,:196)                */
  int32_t size;       /* *spec.leaderWorkerTemplate.size                         */
  uint32_t flags;     /* LWSE_LWS_* */
  int32_t replicas;   /* *spec.replicas                                          */
  int32_t partition;  /* *spec.rolloutStrategy.rollingUpdateConfiguration.partition */
  int32_t max_surge;  /* IntVal, or the percent number when ..._IS_PERCENT       */
  int32_t max_unavailable;
  int32_t sts_replicas;            /* leader sts *spec.replicas                  */
  int32_t sts_partition;           /* leader sts rollingUpdate.partition         */
  int32_t sts_replicas_annotation; /* Atoi(leaderworkerset.sigs.k8s.io/replicas) */
  int32_t subgroup_size;           /* 0 = no subGroupPolicy                      */
  uint64_t uid_hash;  /* hash of metadata.uid: shard key, placement priority     */
  uint32_t group_base;             /* first row of this object in the group table */
  uint32_t group_count;            /* rows = group indices 0..group_count-1      */
} lwse_lws_rec;

#define LWSE_LWS_SURGE_IS_PERCENT (1u << 0)
#define LWSE_LWS_UNAVAIL_IS_PERCENT (1u << 1)
#define LWSE_LWS_STS_EXISTS (1u << 2)       /* leader StatefulSet found (:293)            */
#define LWSE_LWS_UPDATED (1u << 3)          /* leaderWorkerSetUpdated argument (:325)     */
#define LWSE_LWS_ANNOT_VALID (1u << 4)      /* strconv.Atoi of the annotation ok (:351)   */
#define LWSE_LWS_RESTART_SHIFT 5            /* 2 bits: lwse_restart_policy                */
#define LWSE_LWS_RESTART_MASK (3u << 5)
#define LWSE_LWS_RECREATE_AFTER_START_ANNOT (1u << 7) /* pod_controller.go:220            */
#define LWSE_LWS_STARTUP_LEADER_READY (1u << 8)       /* spec.startupPolicy == LeaderReady */
#define LWSE_LWS_EXCLUSIVE_TOPOLOGY (1u << 9) /* exclusive-topology annotation present    */
#define LWSE_LWS_SUBGROUP_LEADER_EXCLUDED (1u << 10)
#define LWSE_LWS_GROUP_LABEL_INVALID (1u << 11) /* a leader pod's group-index label fails
                                                   Atoi → updateConditions error (:434)   */
#define LWSE_LWS_INTSTR_INVALID (1u << 12)  /* maxSurge/maxUnavailable string not "N%"    */
#define LWSE_LWS_IRREGULAR (1u << 13)       /* encoder could not express the object
                                               (see DESIGN.md "Encoder invariants")       */

typedef enum lwse_restart_policy {
  LWSE_RESTART_NONE = 0,          /* "None", "Default", anything else            */
  LWSE_RESTART_ON_POD_RESTART = 1,/* RecreateGroupOnPodRestart                   */
  LWSE_RESTART_AFTER_START = 2    /* RecreateGroupAfterStart                     */
} lwse_restart_policy;

/* One pod group = leader pod slot + its worker StatefulSet (64 B).
 * Row r of an object describes group index r. */
typedef struct lwse_group_rec {
  uint64_t leader_rev_hash;   /* leader pod template-revision-hash label          */
  uint64_t wsts_rev_hash;     /* worker sts template-revision-hash label          */
  int32_t wsts_spec_replicas; /* worker sts *spec.replicas                        */
  int32_t wsts_avail_replicas;/* worker sts status.availableReplicas              */
  uint32_t leader_uid_hash;   /* leader pod metadata.uid                          */
  uint32_t wsts_uid_hash;     /* worker sts metadata.uid                          */
  uint32_t wsts_owner_uid_hash; /* controller ownerRef.uid of the worker sts      */
  uint32_t leader_node;       /* node-table row, LWSE_NONE, or LWSE_NODE_NOT_FOUND */
  uint32_t pod_base;          /* first row of this group in the pod columns       */
  uint32_t pod_count;         /* pods carrying (set name, group index) labels     */
  uint32_t lws_index;         /* row of the owning object in the LWS table        */
  uint32_t flags;             /* LWSE_GRP_* */
  uint32_t reserved[2];
} lwse_group_rec;

#define LWSE_GRP_POD_PRESENT (1u << 0)    /* a leader pod with this group-index label exists */
#define LWSE_GRP_POD_NAME_MATCH (1u << 1) /* its name == "<lws>-<idx>" (:609)                 */
#define LWSE_GRP_POD_RUNNING (1u << 2)    /* status.phase == Running                          */
#define LWSE_GRP_POD_READY (1u << 3)      /* Ready condition == True                          */
#define LWSE_GRP_POD_DELETING (1u << 4)   /* deletionTimestamp != nil                         */
#define LWSE_GRP_WSTS_LABEL_NAME_MATCH (1u << 5) /* sts with this group-index label is named
                                                    "<lws>-<idx>" (:611)                      */
#define LWSE_GRP_WSTS_FOUND (1u << 6)     /* Get(sts named like the leader pod) succeeded     */
#define LWSE_GRP_WSTS_REV_SETTLED (1u << 7) /* status.currentRevision == status.updateRevision */
#define LWSE_GRP_WSTS_OWNER_IS_POD (1u << 8)
#define LWSE_GRP_WSTS_OWNER_NAME_MATCH (1u << 9) /* sts ownerRef.name == leader pod name      */
#define LWSE_GRP_MISTAKEN_ANNOTATION (1u << 10)  /* leader carries leader-name annotation     */
#define LWSE_GRP_REVISION_EXISTS (1u << 11)      /* ControllerRevision for leader's key found */

/* Pods are stored column-split: the per-sweep-hot state BYTE (changes with every status
 * update; the only pod column a sweep streams) and the cold identity row (16 B, 16-byte
 * aligned; fixed at pod creation apart from the node binding; read only for pods that have a
 * restart / deletion event, and by the optional occupancy count). */
typedef uint8_t lwse_pod_state; /* LWSE_POD_* */

typedef struct lwse_pod_ident { /* 16 B */
  uint64_t rev_hash;       /* template-revision-hash label (hash64)                  */
  uint32_t owner_uid_hash; /* controller ownerRef.uid — a 32-bit hash: two different UIDs
                              compare equal with probability 2^-32 per comparison (only
                              pods that already have a restart event are ever compared;
                              DESIGN.md "hash widths")                                */
  uint32_t place;          /* LWSE_PODID_* | node << LWSE_PODID_NODE_SHIFT            */
} lwse_pod_ident;

#define LWSE_POD_PHASE_MASK 3u       /* 0 other, 1 Pending, 2 Running              */
#define LWSE_POD_PHASE_PENDING 1u
#define LWSE_POD_PHASE_RUNNING 2u
#define LWSE_POD_ANY_RESTART (1u << 2) /* some (init)containerStatus.restartCount > 0 */
#define LWSE_POD_DELETING (1u << 3)
#define LWSE_POD_OWNER_SHIFT 4       /* 2 bits: 0 none, 1 Pod, 2 StatefulSet, 3 other */
#define LWSE_POD_OWNER_MASK (3u << 4)
#define LWSE_POD_OWNER_NAME_MATCH (1u << 6) /* ownerRef.name == "<lws>-<group>"    */
#define LWSE_POD_IS_LEADER (1u << 7) /* worker-index label == "0"                  */

#define LWSE_PODID_NAME_OK (1u << 0)   /* GetParentNameAndOrdinal ordinal != -1    */
#define LWSE_PODID_SCHEDULED (1u << 1) /* node field below is valid                */
#define LWSE_PODID_NODE_SHIFT 10       /* 22-bit node-table row                    */
#define LWSE_POD_NODE_MAX ((1u << 22) - 1u)

/* One node (16 B). */
typedef struct lwse_node_rec {
  uint64_t topo_value_hash; /* hash of node.labels[topologyKey]                   */
  uint32_t domain_id;       /* dense id of that label value, or LWSE_NONE         */
  uint16_t capacity;        /* pod slots available to LWS pods                    */
  uint16_t flags;           /* LWSE_NODE_* */
} lwse_node_rec;

#define LWSE_NODE_HAS_TOPOLOGY (1u << 0) /* label present (pod_controller.go:330) */
#define LWSE_NODE_SCHEDULABLE (1u << 1)

/* ------------------------------------------------------------------------- */
/* Output records                                                            */
/* ------------------------------------------------------------------------- */

/* Per LeaderWorkerSet (32 B). */
typedef struct lwse_lws_out {
  int32_t sts_partition;      /* rollingUpdateParameters → stsPartition           */
  int32_t sts_replicas;       /* rollingUpdateParameters → replicas               */
  int32_t sts_max_unavailable;/* constructLeaderStatefulSetApplyConfiguration     */
  int32_t ready_replicas;     /* status.readyReplicas                             */
  int32_t updated_replicas;   /* status.updatedReplicas                           */
  int32_t min_member;         /* PodGroup spec.minMember                          */
  uint32_t flags;             /* LWSE_LOUT_* */
  int32_t unready_replicas;   /* calculateLWSUnreadyReplicas (diagnostic; 0 when
                                 the reference does not compute it)               */
} lwse_lws_out;

#define LWSE_LOUT_RUP_ERROR (1u << 0)     /* rollingUpdateParameters returned err  */
#define LWSE_LOUT_STATUS_ERROR (1u << 1)  /* updateConditions returned err         */
#define LWSE_LOUT_COND_SHIFT 2            /* 2 bits: lwse_condition                */
#define LWSE_LOUT_COND_MASK (3u << 2)
#define LWSE_LOUT_UPDATE_DONE (1u << 4)
#define LWSE_LOUT_EVENT_SHIFT 5           /* 2 bits: lwse_surge_event              */
#define LWSE_LOUT_EVENT_MASK (3u << 5)
#define LWSE_LOUT_IRREGULAR (1u << 7)
#define LWSE_LOUT_BAD_TABLE (1u << 8)     /* group_base/group_count outside the group table */

typedef enum lwse_condition {
  LWSE_COND_PROGRESSING = 0,
  LWSE_COND_AVAILABLE = 1,
  LWSE_COND_UPDATE_IN_PROGRESS = 2 /* UpdateInProgress + Progressing              */
} lwse_condition;

typedef enum lwse_surge_event {
  LWSE_EVENT_NONE = 0,
  LWSE_EVENT_DELETE_ONE = 1,  /* "deleting surge replica %s-%d" (:314)            */
  LWSE_EVENT_DELETE_RANGE = 2 /* "deleting surge replicas from … to …" (:316)     */
} lwse_surge_event;

/* Per pod group (16 B). */
typedef struct lwse_group_out {
  uint32_t flags;           /* LWSE_GOUT_* */
  uint32_t first_trigger;   /* pod row (relative to pod_base) of the first pod
                               whose reconcile would recreate the group, or NONE  */
  int32_t worker_replicas;  /* worker sts replicas (= size-1, ordinals start at 1)
                               when LWSE_GOUT_CREATE_WSTS, else 0                 */
  uint32_t domain_id;       /* nodeSelector topology domain of the workers
                               (topologyValueFromPod), or LWSE_NONE               */
} lwse_group_out;

#define LWSE_GOUT_STATE_READY (1u << 0)    /* getReplicaStates ready  (name-checked)   */
#define LWSE_GOUT_STATE_UPDATED (1u << 1)  /* getReplicaStates updated                 */
#define LWSE_GOUT_COUNTED (1u << 2)        /* leader pod visited by updateConditions   */
#define LWSE_GOUT_COND_READY (1u << 3)     /* updateConditions ready                   */
#define LWSE_GOUT_COND_UPDATED (1u << 4)   /* updateConditions updated                 */
#define LWSE_GOUT_PENDING (1u << 5)        /* pendingPodsInGroup                       */
#define LWSE_GOUT_DELETE_LEADER (1u << 6)  /* some pod's reconcile issues Delete(leader) */
#define LWSE_GOUT_LEADER_DELETING (1u << 7)/* …returns true because it is already going  */
#define LWSE_GOUT_RESTART_ERROR (1u << 8)  /* worker name failed to parse (:231)       */
#define LWSE_GOUT_CREATE_WSTS (1u << 9)    /* leader reconcile reaches Create(worker sts) */
#define LWSE_GOUT_WAIT_SCHEDULE (1u << 10) /* exclusive topology, leader unscheduled   */
#define LWSE_GOUT_TOPOLOGY_ERROR (1u << 11)/* node lacks the topology label (:331)     */
#define LWSE_GOUT_REQUEUE_REVISION (1u << 12) /* revision missing → requeue 1s (:152)  */
#define LWSE_GOUT_CREATE_PODGROUP (1u << 13)  /* SchedulerProvider.CreatePodGroupIfNotExists reached */
#define LWSE_GOUT_BAD_TABLE (1u << 14)     /* lws_index / pod_base+pod_count outside a table  */

/* ------------------------------------------------------------------------- */
/* Table bundles                                                             */
/* ------------------------------------------------------------------------- */

/* The same bundle is used with host pointers (lwse_sweep_lws_host) and with
 * device pointers (lwse_sweep_lws_device). */
typedef struct lwse_lws_tables {
  const lwse_lws_rec* lws;
  uint32_t n_lws;
  const lwse_group_rec* groups;
  uint32_t n_groups;
  const lwse_pod_state* pod_state; /* n_pods words  */
  const lwse_pod_ident* pod_ident; /* n_pods rows   */
  uint64_t n_pods;
  lwse_lws_out* lws_out;     /* n_lws rows   */
  lwse_group_out* group_out; /* n_groups rows */
  uint32_t* node_occupancy;  /* optional: n_nodes counters, scheduled pods per node
                                over the whole pod table (the call overwrites
                                them; it reads the identity column for it); NULL
                                to skip                                           */
  uint32_t flags;            /* LWSE_SWEEP_* */
} lwse_lws_tables;

#define LWSE_SWEEP_GANG (1u << 0) /* a SchedulerProvider is configured (min_member,
                                     CREATE_PODGROUP are meaningful)              */
#define LWSE_SWEEP_SKIP_GROUP_PASS (1u << 1) /* profiling: run only the LWS-level pass
                                                (group_out must hold a previous result) */
#define LWSE_SWEEP_SKIP_LWS_PASS (1u << 2)   /* profiling: skip the LWS-level pass       */
#define LWSE_SWEEP_REUSE_POD_IDENT (1u << 4) /* host entry point only: the pod identity column
                                                (revision hash, owner uid — fixed at pod creation)
                                                is unchanged since this engine's previous host
                                                sweep with the same n_pods; skip its upload     */
#define LWSE_SWEEP_PLACE_GROUPED (1u << 5)   /* lwse_reconcile_*_device: the placement requests are grouped by
                                                namespace (ns non-decreasing) — enables the namespace-parallel
                                                placement kernels (one CTA per namespace, state in shared memory).
                                                A promise: a violated order is counted, rows are then unspecified  */
#define LWSE_SWEEP_PLACE_SCAN (1u << 6)      /* with GROUPED: brute-force (request x node) scoring from the
                                                TMA-staged node table instead of the two-level search (same rows) */
#define LWSE_SWEEP_SKIP_POD_SCAN (1u << 3)   /* profiling: skip the pod-state scan (its
                                                bitmaps must hold a previous result)     */

typedef struct lwse_config {
  uint32_t abi_version; /* LWSE_ABI_VERSION */
  int32_t device;       /* CUDA device ordinal */
  uint32_t flags;       /* reserved, 0 */
  uint32_t reserved;
} lwse_config;

typedef struct lwse_engine lwse_engine;

/* ------------------------------------------------------------------------- */
/* Lifecycle                                                                 */
/* ------------------------------------------------------------------------- */
LWSE_API int lwse_create(const lwse_config* cfg, lwse_engine** out);
LWSE_API void lwse_destroy(lwse_engine* e);
LWSE_API const char* lwse_strerror(int status);
LWSE_API int lwse_last_cuda_error(const lwse_engine* e);
LWSE_API uint32_t lwse_abi_version(void);
/* The CUDA stream (cudaStream_t) all of this engine's work is issued on. */
LWSE_API void* lwse_stream(const lwse_engine* e);
/* Number of kernels this engine has launched since creation. */
LWSE_API uint64_t lwse_launch_count(const lwse_engine* e);
/* Number of resident ticks this engine has replayed as one CUDA graph (LWSE_TICK_GRAPH) since creation. */
LWSE_API uint64_t lwse_graph_tick_count(const lwse_engine* e);

/* Shard an object onto one of n engines (Go: hash(LWS.UID) mod nGPU; DS-owned
 * LWS pass the DS uid hash so a DS and its children co-reside). */
LWSE_API uint32_t lwse_shard_of(uint64_t uid_hash, uint32_t n_shards);
/* The 64-bit string hash the encoders use for revision keys / label values /
 * UIDs (FNV-1a 64; 32-bit fields take the low word xor the high word). */
LWSE_API uint64_t lwse_hash64(const void* bytes, size_t len);

/* ------------------------------------------------------------------------- */
/* Node table                                                                */
/* ------------------------------------------------------------------------- */
/* Copies n node rows to the device; they stay resident across sweeps. */
LWSE_API int lwse_upload_nodes(lwse_engine* e, const lwse_node_rec* nodes, uint32_t n_nodes,
                               uint32_t n_domains);

/* ------------------------------------------------------------------------- */
/* LWS sweep                                                                 */
/* ------------------------------------------------------------------------- */
/* Host buffers in, host buffers out: H2D of the three tables, the sweep
 * kernels, D2H of the two result tables, then a stream synchronize. */
LWSE_API int lwse_sweep_lws_host(lwse_engine* e, const lwse_lws_tables* host_tables);
/* All pointers are device pointers on the engine's device; kernels are
 * enqueued on `stream` (cudaStream_t; NULL = the engine's stream) and the call
 * returns without synchronizing. */
LWSE_API int lwse_sweep_lws_device(lwse_engine* e, const lwse_lws_tables* dev_tables, void* stream);

/* ------------------------------------------------------------------------- */
/* Resident tables: incremental operation                                    */
/* ------------------------------------------------------------------------- */
/* A controller sees watch events, not tables: between two sweeps only a few rows change.
 * The engine can keep the input tables resident in HBM; the host then sends row patches
 * (lwse_resident_patch) and reads back only the result rows that changed
 * (lwse_resident_sweep) — the actions the reconcilers have to take. */
typedef enum lwse_table {
  LWSE_TABLE_LWS = 0,       /* lwse_lws_rec    */
  LWSE_TABLE_GROUPS = 1,    /* lwse_group_rec  */
  LWSE_TABLE_POD_STATE = 2, /* lwse_pod_state  */
  LWSE_TABLE_POD_IDENT = 3, /* lwse_pod_ident  */
  LWSE_TABLE_PLACE_REQS = 4, /* lwse_place_req (lwse_resident_place_load)  */
  LWSE_TABLE_DS = 5,          /* lwse_ds_rec          (lwse_ds_resident_tick only) */
  LWSE_TABLE_DS_ROLES = 6,    /* lwse_ds_role_rec     (lwse_ds_resident_tick only) */
  LWSE_TABLE_DS_REVROLES = 7  /* lwse_ds_revrole_rec  (lwse_ds_resident_tick only) */
} lwse_table;

/* Result rows that differ from the previous resident sweep (all rows after a load).
 * n_* is the number of changed rows; if it exceeds the capacity the surplus rows are not
 * returned and the caller falls back to lwse_resident_outputs.  Order is unspecified. */
typedef struct lwse_changes {
  uint32_t* lws_rows;        /* [lws_capacity]   row numbers          */
  lwse_lws_out* lws_out;     /* [lws_capacity]   their new results    */
  uint32_t lws_capacity;
  uint32_t n_lws;            /* out */
  uint32_t* group_rows;      /* [group_capacity] */
  lwse_group_out* group_out; /* [group_capacity] */
  uint32_t group_capacity;
  uint32_t n_groups;         /* out */
} lwse_changes;

/* Copy the four input tables of `host` to the device; they stay resident (and the
 * previous results are forgotten).  Output pointers in `host` are ignored. */
LWSE_API int lwse_resident_load(lwse_engine* e, const lwse_lws_tables* host);
/* Overwrite n rows of a resident table: row rows[i] ← the i-th packed row of `values` (rows
 * distinct).  Synchronous convenience form of one patch segment of lwse_resident_tick. */
LWSE_API int lwse_resident_patch(lwse_engine* e, lwse_table which, const uint32_t* rows, const void* values,
                                 uint32_t n);
/* Sweep the resident tables (flags: LWSE_SWEEP_GANG).  `changes` may be NULL. */
LWSE_API int lwse_resident_sweep(lwse_engine* e, uint32_t flags, lwse_changes* changes);
/* Every result row of the last resident sweep. */
LWSE_API int lwse_resident_outputs(lwse_engine* e, lwse_lws_out* lws_out, lwse_group_out* group_out);

/* ---- the resident tick: what one pass of the controllers' work queues maps to ---------------
 * Watch events in (as row patches), actions out (the result rows that changed), ONE call:
 *   patches -> scatter kernel -> fused pod scan + group pass -> LWS pass     (engine stream)
 *           \-> placement round over the resident request table            (side stream)
 * The patch rows / values are consumed where the host wrote them when they lie in the engine's
 * arena (pinned, mapped memory: lwse_resident_arena) — no staging copy (large sets go to a device
 * mirror with one copy-engine transfer, small ones are read in place over PCIe); the kernels
 * append the changed result rows to device lists, a publish kernel copies them into pinned,
 * mapped result buffers and raises a sequence word the call spins on: no stream synchronize, no
 * device->host copy-engine launch on the path.  A tick that follows one still in flight is
 * replayed as one CUDA graph (LWSE_TICK_GRAPH=0 turns that off).  Replaces, per reconcile pass, the
 * informer-cache reads of
 * leaderworkerset_controller.go:421,584,598 and pod_controller.go:348 (List) for every object. */

typedef struct lwse_place_req lwse_place_req; /* defined below (Placement) */
typedef struct lwse_place_out lwse_place_out;

/* One patch segment. */
typedef struct lwse_patch_seg {
  uint32_t table;       /* lwse_table                                                      */
  uint32_t flags;       /* LWSE_PATCH_*                                                    */
  uint32_t n;           /* rows patched                                                    */
  uint32_t first_row;   /* LWSE_PATCH_RANGE: rows first_row .. first_row + n - 1           */
  const uint32_t* rows; /* n distinct row numbers (ignored for a range)                    */
  const void* values;   /* n packed rows of the table's record type                        */
} lwse_patch_seg;

#define LWSE_PATCH_RANGE (1u << 0) /* contiguous rows: one DMA copy instead of a scatter (use it
                                      when a large share of a column changed)              */
#define LWSE_TICK_MAX_SEGS 8u

typedef struct lwse_tick {
  /* in */
  const lwse_patch_seg* segs;
  uint32_t n_segs;
  uint32_t flags; /* LWSE_SWEEP_GANG | LWSE_TICK_* */
  /* out: views of engine-owned pinned memory, valid until the next lwse_resident_* call on this
   * engine.  n_* counts every changed row; rows beyond the capacity (= table size, so this
   * cannot happen for the sweep) are not listed.  Order is unspecified. */
  const uint32_t* lws_rows;
  const lwse_lws_out* lws_out;
  uint32_t n_lws;
  uint32_t n_groups;
  const uint32_t* group_rows;
  const lwse_group_out* group_out;
  const uint32_t* place_rows; /* request rows whose placement changed (LWSE_TICK_PLACE) */
  const lwse_place_out* place_out;
  uint32_t n_place;
  uint32_t place_rounds;
} lwse_tick;

#define LWSE_TICK_PLACE (1u << 8)     /* run the placement round over the resident request table */
#define LWSE_TICK_NO_SWEEP (1u << 9)  /* patches (+ placement) only */
#define LWSE_TICK_SHARED_OCCUPANCY (1u << 10) /* multi-rank: the round runs as lwse_reconcile_shared_device does
                                                 — the engine's occupancy counters are pushed to the peers
                                                 (lwse_exchange_*), the resident requests are solved against
                                                 the sum; combine with LWSE_EXCHANGE_LAGGED                    */
/* (LWSE_SWEEP_PLACE_SCAN selects the brute-force form of the round; the resident request table
 * is checked for namespace grouping when it is loaded) */

/* The engine's patch arena: at least min_bytes of pinned, mapped host memory (grown on demand;
 * growing invalidates the previous base).  Patch segments whose rows / values pointers lie inside
 * it are consumed in place; others are first copied into it by the call. */
LWSE_API int lwse_resident_arena(lwse_engine* e, uint64_t min_bytes, void** base_out, uint64_t* bytes_out);
/* Make the placement request table resident (rows are then patched with LWSE_TABLE_PLACE_REQS);
 * the per-node occupancy the rounds use is counted by the engine from the resident identity
 * column and follows its patches.  Needs lwse_upload_nodes and lwse_resident_load first. */
LWSE_API int lwse_resident_place_load(lwse_engine* e, const lwse_place_req* reqs, uint32_t n_reqs,
                                      uint32_t n_namespaces);
LWSE_API int lwse_resident_tick(lwse_engine* e, lwse_tick* t);
/* The same tick in two halves, for callers that keep the work queue flowing: _submit enqueues a
 * tick and returns at once, _wait blocks (spins on the tick's sequence word) for the OLDEST
 * submitted tick and fills t's outputs.  At most two ticks are in flight (a third _submit returns
 * LWSE_ERR_NOT_READY): while the GPU sweeps tick k the copy engine already moves the patches of
 * tick k+1.  Rules: the patch segments of a tick in flight stay untouched in the arena until its
 * _wait returned (use two arena regions alternately); a tick's output views stay valid until the
 * second _submit after its _wait; every other lwse_resident_* call first waits for (and drops the
 * results of) the ticks in flight.  lwse_resident_tick == _submit + _wait. */
LWSE_API int lwse_resident_tick_submit(lwse_engine* e, const lwse_tick* t);
LWSE_API int lwse_resident_tick_wait(lwse_engine* e, lwse_tick* t);
/* Every placement row of the last tick with LWSE_TICK_PLACE / the occupancy counters the engine
 * maintains (n_nodes words). */
LWSE_API int lwse_resident_place_outputs(lwse_engine* e, lwse_place_out* out);
LWSE_API int lwse_resident_occupancy(lwse_engine* e, uint32_t* occupancy_out);

/* ------------------------------------------------------------------------- */
/* Placement (build-defined spec — the reference has no node scoring)        */
/* ------------------------------------------------------------------------- */

/* One placement request per pod group of an exclusive-topology object (32 B). */
typedef struct lwse_place_req {
  uint64_t priority;    /* total order: smaller wins (uid_hash-derived)          */
  uint64_t group_key;   /* first 8 bytes of the SHA-1 group key: preference salt */
  uint32_t group;       /* caller's group id, echoed back                        */
  uint32_t ns;          /* dense namespace id: exclusivity is per namespace      */
  int32_t size;         /* pods that must fit in the domain                      */
  uint32_t leader_node; /* node row if the leader is scheduled, else LWSE_NONE   */
} lwse_place_req;

typedef struct lwse_place_out {
  uint32_t domain_id;   /* claimed domain or LWSE_NONE                           */
  uint32_t leader_node; /* chosen (or given) node for the leader, or LWSE_NONE   */
  uint32_t flags;       /* LWSE_PLACE_* */
  uint32_t score;       /* score of the winning (group, node) pair               */
} lwse_place_out;

#define LWSE_PLACE_PLACED (1u << 0)
#define LWSE_PLACE_PINNED (1u << 1)        /* domain came from a scheduled leader */
#define LWSE_PLACE_CONFLICT (1u << 2)      /* pinned domain already held by a
                                              higher-priority group              */
#define LWSE_PLACE_UNSCHEDULABLE (1u << 3) /* no feasible domain left            */

/* occupancy: pods per node (n_nodes counters, host memory) already summed over
 * every shard; NULL = all zero. */
LWSE_API int lwse_place_host(lwse_engine* e, const lwse_place_req* reqs, uint32_t n_reqs,
                             const uint32_t* occupancy, uint32_t n_namespaces,
                             lwse_place_out* out, uint32_t* rounds_out);
/* Device pointers; enqueued on `stream`.  rounds_out == NULL: no synchronize;
 * otherwise the call waits for the round count.  The placement rounds of one engine share
 * its scratch: they must not overlap in time — keep them on one stream (lwse_reconcile_*
 * use the engine's side stream for theirs) or order the streams with events. */
LWSE_API int lwse_place_device(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                               const uint32_t* d_occupancy, uint32_t n_namespaces,
                               lwse_place_out* d_out, uint32_t* rounds_out, void* stream);

/* As lwse_place_device for a request table the caller keeps GROUPED BY NAMESPACE (ns
 * non-decreasing): one CTA per namespace, holder table / capacities / node table in shared memory
 * (the latter staged by TMA).  flags: LWSE_SWEEP_PLACE_SCAN.  pair_scans_out (optional, with
 * rounds_out): number of (request, round) searches the call made — x usable nodes = (request x
 * node) pairs the scan form scored. */
LWSE_API int lwse_place_grouped_device(lwse_engine* e, const lwse_place_req* d_reqs, uint32_t n_reqs,
                                       const uint32_t* d_occupancy, uint32_t n_namespaces, lwse_place_out* d_out,
                                       uint32_t flags, uint32_t* rounds_out, uint32_t* pair_scans_out, void* stream);

/* Multi-GPU form: `d_parts` is the result of ONE all-gather over the ranks; part p
 * (rank p, at d_parts + p * part_stride_bytes) holds that shard's per-node occupancy
 * (n_nodes uint32 counters) followed, at reqs_offset_bytes, by reqs_per_part request
 * rows (unused rows: leader_node = LWSE_NONE, size = 0).  Node occupancy is summed over
 * the parts; request r = p * reqs_per_part + j; d_out has n_parts * reqs_per_part rows.
 * Every rank solves the same problem and keeps the rows of its own part. */
LWSE_API int lwse_place_gathered_device(lwse_engine* e, const void* d_parts, uint32_t n_parts,
                                        uint64_t part_stride_bytes, uint64_t reqs_offset_bytes,
                                        uint32_t reqs_per_part, uint32_t n_namespaces,
                                        lwse_place_out* d_out, uint32_t* rounds_out, void* stream);

/* One reconcile tick on device tables: lwse_sweep_lws_device(d) on `stream` and a
 * placement round (as lwse_place_device, rounds_out = NULL) on an engine-owned side
 * stream, forked from and joined back into `stream` with events — the placement
 * round reads only its own inputs, never the sweep's outputs, so the two overlap.
 * This is what one pass of the controller's work queue maps to: every
 * Reconcile() (leaderworkerset_controller.go:106-193, pod_controller.go:71-201)
 * plus the scheduler's share of the exclusive-topology contract.
 * n_reqs == 0: sweep only. */
LWSE_API int lwse_reconcile_device(lwse_engine* e, const lwse_lws_tables* d, const lwse_place_req* d_reqs,
                                   uint32_t n_reqs, const uint32_t* d_occupancy, uint32_t n_namespaces,
                                   lwse_place_out* d_place_out, void* stream);

/* The same tick from host tables: lwse_sweep_lws_host(host) and lwse_place_host(reqs, …) in one
 * call, the placement round solved on the side stream while the sweep's tables are uploaded;
 * returns when all results are in the caller's buffers.  n_reqs == 0: sweep only.
 * host->flags & LWSE_SWEEP_PLACE_GROUPED: the request table is grouped by namespace — the call then
 * skips its own pass over the table (it is checked on the device instead: LWSE_ERR_BAD_TABLE when
 * the promise does not hold; without the flag the call finds out itself). */
LWSE_API int lwse_reconcile_host(lwse_engine* e, const lwse_lws_tables* host, const lwse_place_req* reqs,
                                 uint32_t n_reqs, const uint32_t* occupancy, uint32_t n_namespaces,
                                 lwse_place_out* place_out);

/* ------------------------------------------------------------------------- */
/* Peer exchange: the multi-GPU placement step without a collective library  */
/* ------------------------------------------------------------------------- */
#define LWSE_MAX_RANKS 16u
#define LWSE_IPC_HANDLE_BYTES 64u /* sizeof(cudaIpcMemHandle_t) */

/* One process per GPU of one node.  Every rank creates its exchange buffer (room for
 * `world` parts of [n_nodes occupancy counters | reqs_per_part request rows], twice) and
 * gets an IPC handle for it; the caller all-gathers the handles (any transport — they are
 * 64 opaque bytes) and hands all of them to lwse_exchange_connect, which maps the peers'
 * buffers over NVLink.  lwse_upload_nodes must have been called (the layout depends on
 * n_nodes); one exchange per engine.  reqs_per_part = 0: the parts carry occupancy only
 * (lwse_reconcile_shared_device). */
LWSE_API int lwse_exchange_create(lwse_engine* e, uint32_t reqs_per_part, uint32_t world, uint32_t rank,
                                  void* handle_out /* LWSE_IPC_HANDLE_BYTES */);
LWSE_API int lwse_exchange_connect(lwse_engine* e, const void* handles /* world x LWSE_IPC_HANDLE_BYTES */);
/* bytes of one part: align16(n_nodes * 4) + reqs_per_part * sizeof(lwse_place_req) */
LWSE_API uint64_t lwse_exchange_part_bytes(const lwse_engine* e);

/* A reconcile tick of one shard (see lwse_reconcile_device): `d_local_part` — this rank's
 * [occupancy | request rows (unused rows: leader_node = LWSE_NONE, size = 0)] in device
 * memory — is pushed into every peer's buffer with peer stores and a per-source flag is
 * raised there; the same kernel waits for all sources' flags of this step; then the placement
 * round runs over the gathered parts exactly as lwse_place_gathered_device does (d_place_out:
 * world * reqs_per_part rows; every rank computes the same answer and keeps its own rows).
 * All of it on the engine's side stream, concurrently with the sweep of `d` on `stream`
 * (d == NULL: placement step only).  Every rank must call this the same number of times. */
LWSE_API int lwse_reconcile_exchanged_device(lwse_engine* e, const lwse_lws_tables* d, const void* d_local_part,
                                             uint32_t n_namespaces, lwse_place_out* d_place_out, void* stream);
/* The tick of a shard whose placement requests are LOCAL to the rank and whose node occupancy is
 * shared — the north star's "single all-gather of the per-node occupancy vector": ranks own disjoint
 * namespaces (exclusivity is per namespace, so their rounds are independent), every rank's pods load
 * the same nodes.  `d_local_occupancy` (n_nodes counters, this rank's pods) is pushed into every
 * peer's buffer with peer stores + flags (lwse_exchange_create with reqs_per_part = 0 is enough);
 * the round then solves the n_reqs local requests (grouped by namespace) against the SUM of all
 * ranks' counters, concurrently with the sweep of `d` (NULL: placement branch only).
 * flags: LWSE_SWEEP_PLACE_SCAN, LWSE_EXCHANGE_LAGGED.  Every rank must call it the same number of times. */
#define LWSE_EXCHANGE_LAGGED (1u << 16) /* solve against the snapshot every rank pushed in the PREVIOUS
                                           call (own part included): no rank waits for the slowest
                                           rank's launch of this tick; results lag remote occupancy
                                           changes by one tick (the first call is in step)           */
LWSE_API int lwse_reconcile_shared_device(lwse_engine* e, const lwse_lws_tables* d, const lwse_place_req* d_reqs,
                                          uint32_t n_reqs, const uint32_t* d_local_occupancy, uint32_t n_namespaces,
                                          lwse_place_out* d_place_out, uint32_t flags, void* stream);
/* *error_out = 1 if a wait for the peers ever timed out (2 s; a rank is gone).  Synchronizes. */
LWSE_API int lwse_exchange_status(lwse_engine* e, uint32_t* error_out);

/* ------------------------------------------------------------------------- */
/* DisaggregatedSet sweep                                                    */
/* ------------------------------------------------------------------------- */
#define LWSE_DS_MAX_ROLES 10u /* api/disaggregatedset/v1: 2..10 roles             */

/* One DisaggregatedSet (32 B). */
typedef struct lwse_ds_rec {
  uint64_t uid_hash;
  uint32_t role_base;  /* first row in the role table                            */
  uint32_t n_roles;    /* spec roles first, then removed roles (executor.go:140) */
  uint32_t n_spec_roles;
  uint32_t rev_base;   /* first row in the revision-role table                   */
  uint32_t n_old_revs; /* old revisions, each n_roles consecutive rows; the new
                          revision's n_roles rows follow them                    */
  uint32_t flags;      /* LWSE_DS_* */
} lwse_ds_rec;

#define LWSE_DS_HAS_NEW_REVISION (1u << 0) /* GetRevisionRolesList newRevision != nil */

/* One role of a DS (16 B). */
typedef struct lwse_ds_role_rec {
  int32_t target_replicas; /* getTargetReplicas (nil → 1)                        */
  int32_t max_surge;
  int32_t max_unavailable;
  uint32_t flags;          /* LWSE_ROLE_* */
} lwse_ds_role_rec;

#define LWSE_ROLE_SURGE_IS_PERCENT (1u << 0)
#define LWSE_ROLE_UNAVAIL_IS_PERCENT (1u << 1)
#define LWSE_ROLE_HAS_ROLLING_CONFIG (1u << 2) /* rollingUpdateConfiguration != nil */
#define LWSE_ROLE_IN_SPEC (1u << 3)
#define LWSE_ROLE_SURGE_INVALID (1u << 4)   /* intstr error (ignored → 0, executor.go:249) */
#define LWSE_ROLE_UNAVAIL_INVALID (1u << 5)

/* One (revision, role) LWS child of a DS (16 B).  Rows of one DS: for each old
 * revision (in List order) n_roles rows in role order, then n_roles rows for
 * the new (target) revision. */
typedef struct lwse_ds_revrole_rec {
  int32_t replicas;         /* getLWSReplicas: *spec.replicas, nil → 1            */
  int32_t initial_replicas; /* initial-replicas annotation, or -1 when absent/unparsable */
  int32_t ready_replicas;   /* status.readyReplicas                               */
  uint32_t flags;           /* LWSE_RR_* | creation rank << LWSE_RR_TS_SHIFT      */
} lwse_ds_revrole_rec;

#define LWSE_RR_EXISTS (1u << 0)       /* this revision has an LWS for this role   */
#define LWSE_RR_REPLICAS_NIL (1u << 1) /* spec.replicas == nil (cleanup counts it as 0,
                                          disaggregatedset_controller.go:222-225) */
#define LWSE_RR_TS_SHIFT 2             /* 30-bit order-preserving rank of
                                          metadata.creationTimestamp (executor.go:283-302) */

/* Per DS (16 B). */
typedef struct lwse_ds_out {
  uint32_t flags;        /* LWSE_DOUT_* */
  uint32_t drained_revs; /* bit r: old revision r has every role at 0 → delete its LWS */
  uint32_t ready_revs;   /* bit r: old revision r is ready on all spec roles (its
                            services are kept, service_manager.go:174-189)          */
  uint32_t reserved;
} lwse_ds_out;

#define LWSE_DOUT_ROLLING (1u << 0)   /* old revisions still hold replicas → rolling path */
#define LWSE_DOUT_INIT (1u << 1)      /* …but no new revision yet → initRollingUpdate     */
#define LWSE_DOUT_STABLE (1u << 2)    /* isRevisionStable(newRevision)                    */
#define LWSE_DOUT_STEP (1u << 3)      /* ComputeNextStep returned a step                  */
#define LWSE_DOUT_COMPLETE (1u << 4)  /* ComputeNextStep returned nil                     */
#define LWSE_DOUT_NEW_READY (1u << 5) /* target revision ready on all roles → ensure services */
#define LWSE_DOUT_BAD_TABLE (1u << 6)
#define LWSE_DS_MAX_OLD_REVS 32u

/* Per role (8 B): the planner step. */
typedef struct lwse_ds_role_out {
  int32_t next_old; /* UpdateStep.Past[i] */
  int32_t next_new; /* UpdateStep.New[i]  */
} lwse_ds_role_out;

/* Per (revision, role): spec.replicas after this reconcile — scaleUpNew /
 * scaleDownOld / reconcileSimple — or -1 where no LWS exists and none is
 * created (4 B). */
typedef int32_t lwse_ds_revrole_out;

typedef struct lwse_ds_tables {
  const lwse_ds_rec* ds;
  uint32_t n_ds;
  const lwse_ds_role_rec* roles;
  uint32_t n_roles;
  const lwse_ds_revrole_rec* revroles;
  uint32_t n_revroles;
  lwse_ds_out* ds_out;              /* n_ds       */
  lwse_ds_role_out* role_out;       /* n_roles    */
  lwse_ds_revrole_out* revrole_out; /* n_revroles */
} lwse_ds_tables;

LWSE_API int lwse_sweep_ds_host(lwse_engine* e, const lwse_ds_tables* host_tables);
LWSE_API int lwse_sweep_ds_device(lwse_engine* e, const lwse_ds_tables* dev_tables, void* stream);

/* ---- the resident DS tick: what one pass of the DisaggregatedSet controller's work queue maps to --
 * The three DS input tables stay resident in HBM (their own buffers: a stateless lwse_sweep_ds_* call
 * and the LWS resident tables / ticks never touch them).  Watch events arrive as row patches
 * (lwse_patch_seg with LWSE_TABLE_DS / _DS_ROLES / _DS_REVROLES, consumed in place when they lie in
 * the arena, staged otherwise; LWSE_PATCH_RANGE as for the LWS tick), one call returns the result rows
 * that changed:   patches -> scatter kernel -> resident DS sweep -> publish kernel   (engine stream)
 * and the host spins on a sequence word in pinned memory: no stream synchronize, no device->host
 * copy-engine transfer on the path.  The results equal lwse_sweep_ds_* on the same tables.  Replaces,
 * per reconcile pass, GetRevisionRolesList -> List (lws_manager.go:161-213) for every DS.
 *
 * Change lists.  A DS is VALID in a tick when the sweep does not flag it LWSE_DOUT_BAD_TABLE.  The
 * rows a valid DS OWNS are role rows [role_base, role_base + n_roles) and revision-role rows
 * [rev_base, rev_base + (n_old_revs + 1) * n_roles).  Every result row has a COMMITTED value: the last
 * value a tick wrote to it (zero bytes if none did since lwse_ds_resident_load).
 *   - a role / revision-role row is listed when a valid DS owns it and its new value differs from its
 *     committed value, or this is the first tick after lwse_ds_resident_load;
 *   - a DS row is listed when its ds_out differs from its committed value, or any of its role /
 *     revision-role rows is listed, or this is the first tick after a load: the list is the set of DS
 *     keys that need work, always with the current ds_out;
 *   - a DS flagged BAD_TABLE writes only its ds_out; the rows it used to own keep their committed
 *     values and are not listed.
 * Invariant: a zero mirror with every tick's lists applied in order equals lwse_ds_resident_outputs
 * on every row (and, on the rows valid DSes own, the stateless sweep of the same tables).
 * Like every other resident call, a DS resident call first waits for (and drops the results of) the
 * ticks in flight.  One DS tick runs at a time; to keep two in flight, use the joint tick below with
 * lws = NULL. */
typedef struct lwse_ds_tick {
  /* in */
  const lwse_patch_seg* segs; /* tables LWSE_TABLE_DS .. LWSE_TABLE_DS_REVROLES only */
  uint32_t n_segs;            /* <= LWSE_TICK_MAX_SEGS */
  uint32_t flags;             /* reserved, 0 */
  /* out: views of engine-owned pinned memory, valid until the next lwse_*resident* call on this
   * engine (joint ticks: see lwse_joint_tick).  n_* counts the listed rows (at most the table's rows).
   * Order is unspecified. */
  const uint32_t* ds_rows;
  const lwse_ds_out* ds_out;
  uint32_t n_ds;
  uint32_t n_roles;
  const uint32_t* role_rows;
  const lwse_ds_role_out* role_out;
  const uint32_t* revrole_rows;
  const lwse_ds_revrole_out* revrole_out;
  uint32_t n_revroles;
  uint32_t reserved;
} lwse_ds_tick;

/* Copy the three input tables of `host` to the device, where they stay resident; output pointers are
 * ignored.  Previous results are forgotten: committed outputs start at zero bytes. */
LWSE_API int lwse_ds_resident_load(lwse_engine* e, const lwse_ds_tables* host);
LWSE_API int lwse_ds_resident_tick(lwse_engine* e, lwse_ds_tick* t);
/* Every committed result row (n_ds / n_roles / n_revroles rows of the loaded tables; NULL skips). */
LWSE_API int lwse_ds_resident_outputs(lwse_engine* e, lwse_ds_out* ds_out, lwse_ds_role_out* role_out,
                                      lwse_ds_revrole_out* revrole_out);

/* ---- the joint tick: one pass of the LWS, pod and DS controllers' work queues, one call ----------
 * One tick of both controllers: the LWS part exactly as lwse_resident_tick_submit, the DS part with the
 * listing rules of lwse_ds_resident_tick, ONE scatter, ONE publish.  lws may be NULL (a DS-only tick,
 * which pipelines like an LWS tick); ds may not.
 *   patches of both parts -> scatter kernel -> fused pod scan + group pass -> LWS pass ---> publish
 *                                           \-> DS sweep (own stream) -------------------/
 *                         \-> placement round (side stream) --------------------------/
 * Rules:
 *   - Preconditions: lwse_ds_resident_load, else LWSE_ERR_NOT_READY; lwse_resident_load when lws != NULL,
 *     and lwse_resident_place_load when lws->flags has LWSE_TICK_PLACE (else LWSE_ERR_NOT_READY).  An
 *     engine with DS tables only runs DS-only joint ticks.
 *   - lws->segs name tables 0-4 only, ds->segs tables 5-7 only, at most LWSE_TICK_MAX_SEGS each;
 *     ds->flags must be 0; LWSE_TICK_SHARED_OCCUPANCY is refused (LWSE_ERR_INVALID_ARG): a joint tick
 *     runs on one rank.
 *   - A refused call does nothing: it enqueues nothing, takes no ring slot, moves no sequence number.
 *   - One ring: joint ticks share the two slots of lwse_resident_tick_submit.  At most two ticks of
 *     either kind are in flight; a third submit returns LWSE_ERR_NOT_READY.
 *   - lwse_joint_tick_wait takes the oldest tick of either kind (lws may be NULL: its LWS results are
 *     then not reported); for an LWS-only tick it fills ds with zero counts and NULL views.
 *     lwse_resident_tick_wait refuses a joint tick at the head of the ring (LWSE_ERR_INVALID_ARG) and
 *     leaves it in flight, so its DS lists are not lost.
 *   - lwse_joint_tick == _submit + _wait of one tick; with ticks in flight it returns LWSE_ERR_NOT_READY
 *     (their results stay with _wait).
 *   - Output views (both parts) and arena regions have the lifetime of lwse_resident_tick_submit's:
 *     views stay valid until the second submit after their wait, patch segments stay untouched until
 *     their wait returned.
 *   - Every other resident call (lwse_ds_resident_tick, lwse_ds_resident_load, lwse_resident_load, ...)
 *     still first waits for (and drops the results of) the ticks in flight.  Joint ticks and
 *     lwse_ds_resident_tick share the DS committed outputs: the committed-value model above applies
 *     across both.
 *   - The DS change lists follow committed values exactly as in lwse_ds_resident_tick, in stream order
 *     across pipelined ticks: a zero mirror with every tick's lists applied in order equals
 *     lwse_ds_resident_outputs.
 *   - A joint tick is enqueued kernel by kernel (LWSE_TICK_GRAPH does not apply to it). */
LWSE_API int lwse_joint_tick(lwse_engine* e, lwse_tick* lws, lwse_ds_tick* ds);
LWSE_API int lwse_joint_tick_submit(lwse_engine* e, const lwse_tick* lws, const lwse_ds_tick* ds);
LWSE_API int lwse_joint_tick_wait(lwse_engine* e, lwse_tick* lws, lwse_ds_tick* ds);

/* ------------------------------------------------------------------------- */
/* Group / subgroup keys (SHA-1) and subgroup indices                        */
/* ------------------------------------------------------------------------- */
/* keys: n strings, string i = bytes[offsets[i] .. offsets[i+1]) (the caller
 * formats "<ns>/<podName>" or "<leaderName>/<subIdx>"); digests: n x 20 bytes. */
LWSE_API int lwse_group_keys_host(lwse_engine* e, const uint8_t* bytes, const uint32_t* offsets,
                                  uint32_t n, uint8_t* digests);
LWSE_API int lwse_group_keys_device(lwse_engine* e, const uint8_t* d_bytes,
                                    const uint32_t* d_offsets, uint32_t n, uint8_t* d_digests,
                                    void* stream);

/* Subgroup indices and subgroup keys of n pods in one pass (pod_webhook.go:249-255
 * getSubGroupIndex, :130/:151 the subgroup key): pod i has leader-pod name
 * bytes[offsets[i] .. offsets[i+1]), group size pod_count[i], subgroup size subgroup_size[i] and
 * worker index worker_index[i].  index_out[i] = getSubGroupIndex(...) with Go's truncating
 * division (worker 0 of a "leader is extra" group with subgroup size 1 gives -1, as the Go
 * expression does); digests[i] = SHA-1("<leaderName>/<index>") — the "/<index>" suffix is formed on
 * the device.  subgroup_size[i] == 0 (a division by zero in Go): index_out[i] = INT32_MIN and a
 * zero digest. */
LWSE_API int lwse_subgroup_keys_host(lwse_engine* e, const uint8_t* bytes, const uint32_t* offsets, uint32_t n,
                                     const int32_t* pod_count, const int32_t* subgroup_size,
                                     const int32_t* worker_index, int32_t* index_out, uint8_t* digests);
LWSE_API int lwse_subgroup_keys_device(lwse_engine* e, const uint8_t* d_bytes, const uint32_t* d_offsets, uint32_t n,
                                       const int32_t* d_pod_count, const int32_t* d_subgroup_size,
                                       const int32_t* d_worker_index, int32_t* d_index_out, uint8_t* d_digests,
                                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LWSE_H_ */
