// DisaggregatedSet sweep (sm_100a): one thread per DisaggregatedSet, the ≤10
// roles of a DS in registers / local arrays.
//
// Follows pkg/controllers/disaggregatedset/{planner.go:61-352, executor.go:
// 199-302,306-398, disaggregatedset_controller.go:95-112,137-186,203-236,
// service_manager.go:57-89,174-189}.  The reference's float64 step arithmetic
// (planner.go:92,103-104,125,139-140) is evaluated in 64-bit integers: for
// non-negative a, b, c with a·b < 2^53 the IEEE quotient a·b/c lies on the same
// side of every integer as the exact one, so int(x), floor(x) and ceil(x) equal
// integer floor / ceil division (DESIGN.md "float vs int"); the CPU oracle keeps
// the float form, so parity tests compare the two formulations.
#include "lwse_device.cuh"

namespace lwse {

constexpr int MAXR = (int)LWSE_DS_MAX_ROLES;

struct RuConfig {
  int ms, mu;
};

__device__ __forceinline__ int batch_size(int ms, int mu) { return ms > 0 ? ms : max(1, mu); }  // :61-66

// floor(a*b/c) and ceil(a*b/c) for a,b >= 0, c > 0
__device__ __forceinline__ int floor_muldiv(int a, int b, int c) { return (int)(((long long)a * b) / c); }
__device__ __forceinline__ int ceil_muldiv(int a, int b, int c) {
  return (int)((((long long)a * b) + c - 1) / c);
}

// planner.go:264-294
__device__ void apply_orphan_prevention(int n, int* next_old, const int* cur_new, const int* initial_old,
                                        const int* target, const RuConfig* cfg) {
  bool any_zero = false, all_zero = true;
  for (int i = 0; i < n; i++) {
    if (initial_old[i] == 0) continue;
    if (next_old[i] == 0)
      any_zero = true;
    else
      all_zero = false;
  }
  if (!any_zero || all_zero) return;
  bool can_all = true;  // canDrainAllToZero :252-262
  for (int i = 0; i < n; i++)
    if (initial_old[i] >= target[i] && cur_new[i] < target[i] - cfg[i].mu) can_all = false;
  if (can_all) {
    for (int i = 0; i < n; i++) next_old[i] = 0;
    return;
  }
  for (int i = 0; i < n; i++)
    if (next_old[i] == 0 && initial_old[i] > 0) next_old[i] = 1;
}

// planner.go:320-352 ComputeNextStep → true when a step exists
__device__ bool compute_next_step(int n, const int* initial_old, const int* cur_old, const int* cur_new,
                                  const int* target, const RuConfig* cfg, int* past, int* new_) {
  bool complete = true;  // :173-180
  for (int i = 0; i < n; i++)
    if (cur_old[i] != 0 || cur_new[i] < target[i]) complete = false;
  if (complete) return false;
  int total_steps = 0;  // :68-78
  for (int i = 0; i < n; i++) {
    const int mx = max(max(initial_old[i], target[i]), 0);
    const int b = batch_size(cfg[i].ms, cfg[i].mu);
    total_steps = max(total_steps, (mx + b - 1) / b);
  }
  if (total_steps == 0) return false;
  {  // correctAbnormalState :151-171
    bool needs = false;
    for (int i = 0; i < n; i++) {
      past[i] = min(initial_old[i], cur_old[i]);
      if (cur_old[i] > past[i]) needs = true;
      new_[i] = cur_new[i];
    }
    if (needs) return true;
  }
  {  // isNewAtTarget :182-189
    bool at = true;
    for (int i = 0; i < n; i++)
      if (cur_new[i] < target[i]) at = false;
    if (at) {
      for (int i = 0; i < n; i++) {
        past[i] = 0;
        new_[i] = cur_new[i];
      }
      return true;
    }
  }
  int next_new[MAXR], min_old[MAXR];
  {  // computeNextNewReplicas :80-113
    int min_idx = total_steps;
    for (int i = 0; i < n; i++) {
      const int idx = target[i] == 0 ? total_steps : floor_muldiv(cur_new[i], total_steps, target[i]);
      min_idx = min(min_idx, idx);
    }
    const int next_idx = min_idx + 1;
    for (int i = 0; i < n; i++) {
      const int computed = min(ceil_muldiv(next_idx, target[i], total_steps), target[i]);
      next_new[i] = max(computed, cur_new[i]);
    }
  }
  for (int i = 0; i < n; i++) {  // computeMinOld :203-211
    min_old[i] = 0;
    if (initial_old[i] >= target[i]) min_old[i] = max(0, target[i] - cfg[i].mu - cur_new[i]);
  }
  {  // tryScaleUp :213-228, canScaleUp :191-201
    bool needs = false, can = true;
    for (int i = 0; i < n; i++) {
      if (next_new[i] > cur_new[i]) needs = true;
      if (target[i] != 0 && cur_old[i] + next_new[i] > target[i] + cfg[i].ms) can = false;
    }
    if (needs && can) {
      for (int i = 0; i < n; i++) {
        past[i] = cur_old[i];
        new_[i] = next_new[i];
      }
      return true;
    }
  }
  {  // tryProportionalDrain :230-250 (computeNextOldReplicas :115-149)
    int next_old[MAXR];
    int max_idx = 0;
    for (int i = 0; i < n; i++) {
      if (initial_old[i] == 0) continue;
      max_idx = max(max_idx, floor_muldiv(initial_old[i] - cur_old[i], total_steps, initial_old[i]));
    }
    const int next_idx = max_idx + 1;
    bool needs = false;
    for (int i = 0; i < n; i++) {
      const int computed = max(0, initial_old[i] - floor_muldiv(next_idx, initial_old[i], total_steps));
      next_old[i] = max(min(computed, cur_old[i]), min_old[i]);
    }
    apply_orphan_prevention(n, next_old, cur_new, initial_old, target, cfg);
    for (int i = 0; i < n; i++)
      if (next_old[i] < cur_old[i]) needs = true;
    if (needs) {
      for (int i = 0; i < n; i++) {
        past[i] = next_old[i];
        new_[i] = cur_new[i];
      }
      return true;
    }
  }
  {  // tryForceDrain :296-318
    int drained[MAXR];
    bool needs = false;
    for (int i = 0; i < n; i++) {
      const int max_old = target[i] + cfg[i].ms - next_new[i];
      drained[i] = max(0, min(cur_old[i], max_old));
      if (initial_old[i] >= target[i]) drained[i] = max(drained[i], max(0, target[i] - cfg[i].mu - next_new[i]));
      if (drained[i] < cur_old[i]) needs = true;
    }
    if (needs) {
      apply_orphan_prevention(n, drained, next_new, initial_old, target, cfg);
      for (int i = 0; i < n; i++) {
        past[i] = drained[i];
        new_[i] = next_new[i];
      }
      return true;
    }
  }
  return false;
}

// A DS record's row ranges lie inside the tables (else the DS is flagged LWSE_DOUT_BAD_TABLE).
__device__ __forceinline__ bool ds_in_tables(const lwse_ds_tables& t, const uint4 h0, const uint4 h1) {
  const uint32_t role_base = h0.z, n_roles = h0.w, n_spec = h1.x, rev_base = h1.y, n_old = h1.z;
  return !(n_roles > LWSE_DS_MAX_ROLES || n_spec > n_roles || n_old > LWSE_DS_MAX_OLD_REVS ||
           (uint64_t)role_base + n_roles > t.n_roles ||
           (uint64_t)rev_base + (uint64_t)(n_old + 1u) * n_roles > t.n_revroles);
}

// The decisions of one DS (record words h0, h1; its ranges checked by ds_in_tables): the role rows go
// to role_out, the (revision, role) rows to revrole_out — both indexed like the input tables.
// revrole_out is working storage as well: scaleDownOld reads back what scaleUpNew / reconcileSimple
// wrote.  Returns the ds_out row.
__device__ __forceinline__ uint4 ds_decide(const lwse_ds_tables& t, const uint4 h0, const uint4 h1,
                                           lwse_ds_role_out* role_out, lwse_ds_revrole_out* revrole_out) {
  {
    const uint32_t role_base = h0.z, n_roles = h0.w, n_spec = h1.x, rev_base = h1.y, n_old = h1.z, dflags = h1.w;
    uint32_t oflags = 0, drained = 0, ready_revs = 0;
    const int n = (int)n_roles, S = (int)n_spec, V = (int)n_old;
    const lwse_ds_role_rec* roles = t.roles + role_base;
    const uint4* rr = reinterpret_cast<const uint4*>(t.revroles + rev_base);  // {replicas, initial, ready, flags}
    lwse_ds_role_out* ro = role_out + role_base;
    lwse_ds_revrole_out* rro = revrole_out + rev_base;

    int initial_old[MAXR], cur_old[MAXR], cur_new[MAXR], target[MAXR];
    RuConfig cfg[MAXR];
    for (int i = 0; i < n; i++) initial_old[i] = cur_old[i] = cur_new[i] = target[i] = 0;

    // one pass over the old revisions: totals, cleanup predicate, service readiness, defaults
    int total_old_spec = 0;
    for (int r = 0; r < V; r++) {
      bool any = false, all_drained = true, ready = true;
      for (int i = 0; i < n; i++) {
        const uint4 x = ldg_stream(rr + r * n + i);
        const bool exists = x.w & LWSE_RR_EXISTS;
        rro[r * n + i] = exists ? (int)x.x : -1;
        if (i < S && (!exists || (int)x.z < 1)) ready = false;  // service_manager.go:62-67
        if (!exists) continue;
        any = true;
        if (((x.w & LWSE_RR_REPLICAS_NIL) ? 0 : (int)x.x) != 0) all_drained = false;  // :222-225
        cur_old[i] += (int)x.x;                                                        // utils.go:167-175
        initial_old[i] += (int)x.y >= 0 ? (int)x.y : (int)x.x;                         // utils.go:177-190
        if (i < S) total_old_spec += (int)x.x;
      }
      if (any && all_drained) drained |= 1u << r;
      if (ready) ready_revs |= 1u << r;
    }
    bool new_ready = true, stable = true;
    for (int i = 0; i < n; i++) {
      const uint4 x = ldg_stream(rr + V * n + i);
      const bool exists = x.w & LWSE_RR_EXISTS;
      rro[V * n + i] = exists ? (int)x.x : -1;
      const uint4 rl = ldg_cached(reinterpret_cast<const uint4*>(roles + i));  // {target, surge, unavail, flags}
      const bool in_spec = rl.w & LWSE_ROLE_IN_SPEC;
      if (i < S) {
        if (!exists || (int)x.z < 1) new_ready = false;
        if (!exists || (int)x.x != (int)x.z) stable = false;  // isRevisionStable executor.go:270-281
      }
      if (in_spec) {
        if (exists) cur_new[i] = (int)x.x;
        target[i] = (int)rl.x;
      }
      // extractRollingUpdateConfig executor.go:235-260
      cfg[i].ms = 1;
      cfg[i].mu = 0;
      if (in_spec && (rl.w & LWSE_ROLE_HAS_ROLLING_CONFIG)) {
        const int replicas = (int)rl.x;
        const int surge = (rl.w & LWSE_ROLE_SURGE_INVALID)
                              ? 0
                              : scaled_value((int)rl.y, rl.w & LWSE_ROLE_SURGE_IS_PERCENT, replicas, true);
        const int unav = (rl.w & LWSE_ROLE_UNAVAIL_INVALID)
                             ? 0
                             : scaled_value((int)rl.z, rl.w & LWSE_ROLE_UNAVAIL_IS_PERCENT, replicas, false);
        if (unav > 0) {
          cfg[i].mu = unav;
          cfg[i].ms = surge;
        } else if (surge > 0) {
          cfg[i].ms = surge;
        }
      }
      ro[i].next_old = -1;
      ro[i].next_new = -1;
    }
    if (new_ready) oflags |= LWSE_DOUT_NEW_READY;

    if (!(V > 0 && total_old_spec > 0)) {
      // reconcileSimple disaggregatedset_controller.go:137-186
      for (int i = 0; i < S; i++) rro[V * n + i] = target[i];
    } else {
      oflags |= LWSE_DOUT_ROLLING;
      if (!(dflags & LWSE_DS_HAS_NEW_REVISION)) {
        oflags |= LWSE_DOUT_INIT;  // initRollingUpdate executor.go:85-124
        for (int i = 0; i < S; i++) rro[V * n + i] = 0;
      } else if (stable) {
        oflags |= LWSE_DOUT_STABLE;
        int past[MAXR], new_[MAXR];
        if (!compute_next_step(n, initial_old, cur_old, cur_new, target, cfg, past, new_)) {
          oflags |= LWSE_DOUT_COMPLETE;
        } else {
          oflags |= LWSE_DOUT_STEP;
          for (int i = 0; i < n; i++) {
            ro[i].next_old = past[i];
            ro[i].next_new = new_[i];
            // scaleUpNew executor.go:306-328
            if ((__ldg(&roles[i].flags) & LWSE_ROLE_IN_SPEC) && cur_new[i] < new_[i]) rro[V * n + i] = new_[i];
          }
          // scaleDownOld executor.go:330-398, revisions newest-first (:283-302)
          int budget[MAXR];
          for (int i = 0; i < n; i++) budget[i] = cur_old[i] - past[i];
          uint32_t done_mask = 0;
          for (int k = 0; k < V; k++) {
            bool all_zero = true;
            for (int i = 0; i < n; i++)
              if (budget[i] > 0) all_zero = false;
            if (all_zero) break;
            // next newest revision not yet handled (stable: lowest row on equal stamps)
            int r = -1;
            uint32_t best_ts = 0;
            for (int c = 0; c < V; c++) {
              if (done_mask & (1u << c)) continue;
              uint32_t ts = 0;
              for (int i = 0; i < n; i++) {
                const uint32_t w = __ldg(&t.revroles[rev_base + c * n + i].flags);
                if (w & LWSE_RR_EXISTS) ts = max(ts, w >> LWSE_RR_TS_SHIFT);
              }
              if (r < 0 || ts > best_ts) {
                r = c;
                best_ts = ts;
              }
            }
            done_mask |= 1u << r;
            int new_rep[MAXR], planned[MAXR];
            uint32_t trig = 0;
            for (int i = 0; i < n; i++) {
              planned[i] = 0;
              new_rep[i] = 0;
              const int rep = rro[r * n + i];
              if (rep < 0) continue;
              const int drain = min(budget[i], rep);
              planned[i] = drain;
              new_rep[i] = rep - drain;
              if (new_rep[i] == 0) trig |= 1u << i;
            }
            for (int i = 0; i < n; i++) {
              const int rep = rro[r * n + i];
              if (rep < 0) continue;
              const int nr = trig ? 0 : new_rep[i];  // coordinated drain :366-373
              if (rep <= nr) continue;
              rro[r * n + i] = nr;
              if ((trig & (1u << i)) || !trig) budget[i] -= planned[i];  // :392-394
            }
          }
        }
      }
    }
    return make_uint4(oflags, drained, ready_revs, 0);
  }
}

// Resident form (lwse_ds_resident_tick): the tables are the engine's resident ones; the decisions go
// to scratch rows, and every row a valid DS owns is compared with its committed value — rows that
// differ (all rows on the first tick after a load) are written back and appended to the change lists.
struct DsResidentArgs {
  lwse_ds_out* ds_committed;
  lwse_ds_role_out* role_committed;
  lwse_ds_revrole_out* revrole_committed;
  lwse_ds_role_out* role_scratch;
  lwse_ds_revrole_out* revrole_scratch;
  uint32_t* ds_rows;  // change lists (device memory), capacity = table rows
  lwse_ds_out* ds_outs;
  uint32_t* role_rows;
  lwse_ds_role_out* role_outs;
  uint32_t* revrole_rows;
  lwse_ds_revrole_out* revrole_outs;
  uint32_t* counts;  // [0] ds, [1] role, [2] revrole rows listed
  uint32_t first;    // first tick after a load: list every row
};

// Warp-aggregated append: every lane of the warp calls this; lane i reserves n_i slots of *counter with
// one atomic for the whole warp.  Returns lane i's first slot.
__device__ __forceinline__ uint32_t warp_reserve(uint32_t* counter, uint32_t n) {
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t incl = n;
#pragma unroll
  for (uint32_t o = 1; o < 32u; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += v;
  }
  const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
  uint32_t base = 0;
  if (total) {
    if (lane == 31u) base = atomicAdd(counter, total);
    base = __shfl_sync(0xFFFFFFFFu, base, 31);
  }
  return base + incl - n;
}

__device__ __forceinline__ bool ne(const lwse_ds_role_out a, const lwse_ds_role_out b) {
  return a.next_old != b.next_old || a.next_new != b.next_new;
}
__device__ __forceinline__ bool ne(const uint4 a, const uint4 b) { return a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w; }

template <bool kResident>
__global__ void __launch_bounds__(128) ds_sweep_kernel(const lwse_ds_tables t, const DsResidentArgs r) {
  if constexpr (!kResident) {
    for (uint32_t d = blockIdx.x * blockDim.x + threadIdx.x; d < t.n_ds; d += gridDim.x * blockDim.x) {
      const uint4 h0 = ldg_stream(reinterpret_cast<const uint4*>(t.ds + d) + 0);
      const uint4 h1 = ldg_stream(reinterpret_cast<const uint4*>(t.ds + d) + 1);
      if (!ds_in_tables(t, h0, h1)) {
        stg_stream(t.ds_out + d, make_uint4(LWSE_DOUT_BAD_TABLE, 0, 0, 0));
        continue;
      }
      stg_stream(t.ds_out + d, ds_decide(t, h0, h1, t.role_out, t.revrole_out));
    }
  } else {
    pdl_launch_dependents();
    pdl_wait_prior();  // the kernel before this one (the tick's patch scatter) writes the input tables
    // whole warps iterate together: the list appends are warp-collective
    const uint32_t n_iter = (t.n_ds + 31u) & ~31u;
    for (uint32_t d = blockIdx.x * blockDim.x + threadIdx.x; d < n_iter; d += gridDim.x * blockDim.x) {
      const bool live = d < t.n_ds;
      uint4 h0 = make_uint4(0, 0, 0, 0), h1 = h0, o = h0;
      bool valid = false;
      if (live) {
        h0 = ldg_stream(reinterpret_cast<const uint4*>(t.ds + d) + 0);
        h1 = ldg_stream(reinterpret_cast<const uint4*>(t.ds + d) + 1);
        valid = ds_in_tables(t, h0, h1);
        o = valid ? ds_decide(t, h0, h1, r.role_scratch, r.revrole_scratch) : make_uint4(LWSE_DOUT_BAD_TABLE, 0, 0, 0);
      }
      const uint32_t role_base = h0.z, n = valid ? h0.w : 0u, rev_base = h1.y;
      const uint32_t n_rr = valid ? (h1.z + 1u) * n : 0u;
      const bool first = r.first != 0u;
      // pass 1: how many rows of each list this DS appends
      uint32_t c_role = 0, c_rr = 0;
      for (uint32_t i = 0; i < n; i++)
        c_role += (first || ne(r.role_scratch[role_base + i], r.role_committed[role_base + i])) ? 1u : 0u;
      for (uint32_t k = 0; k < n_rr; k++)
        c_rr += (first || r.revrole_scratch[rev_base + k] != r.revrole_committed[rev_base + k]) ? 1u : 0u;
      const uint4 committed = live ? *reinterpret_cast<const uint4*>(r.ds_committed + d) : o;
      const uint32_t c_ds = live && (first || ne(o, committed) || c_role || c_rr) ? 1u : 0u;
      uint32_t at_role = warp_reserve(r.counts + 1, c_role);
      uint32_t at_rr = warp_reserve(r.counts + 2, c_rr);
      const uint32_t at_ds = warp_reserve(r.counts + 0, c_ds);
      // pass 2: write back and list the rows that changed
      if (c_role)
        for (uint32_t i = 0; i < n; i++) {
          const uint32_t row = role_base + i;
          const lwse_ds_role_out v = r.role_scratch[row];
          if (!first && !ne(v, r.role_committed[row])) continue;
          r.role_committed[row] = v;
          if (at_role < t.n_roles) {
            r.role_rows[at_role] = row;
            r.role_outs[at_role] = v;
          }
          at_role++;
        }
      if (c_rr)
        for (uint32_t k = 0; k < n_rr; k++) {
          const uint32_t row = rev_base + k;
          const lwse_ds_revrole_out v = r.revrole_scratch[row];
          if (!first && v == r.revrole_committed[row]) continue;
          r.revrole_committed[row] = v;
          if (at_rr < t.n_revroles) {
            r.revrole_rows[at_rr] = row;
            r.revrole_outs[at_rr] = v;
          }
          at_rr++;
        }
      if (c_ds) {
        *reinterpret_cast<uint4*>(r.ds_committed + d) = o;
        if (at_ds < t.n_ds) {
          r.ds_rows[at_ds] = d;
          *reinterpret_cast<uint4*>(r.ds_outs + at_ds) = o;
        }
      }
    }
  }
}

int launch_ds_sweep(const lwse_ds_tables* t, int sm_count, cudaStream_t s, int* cuda_err) {
  *cuda_err = 0;
  if (t->n_ds == 0) return 0;
  const uint32_t want = (t->n_ds + 127u) / 128u;
  const uint32_t cap = (uint32_t)sm_count * 16u;
  ds_sweep_kernel<false><<<want < cap ? want : cap, 128, 0, s>>>(*t, DsResidentArgs{});
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

// pdl: launched programmatically dependent on the kernel before it (which may write the input tables:
// the resident kernel waits at its top either way).
int launch_ds_resident_sweep(const lwse_ds_tables* t, const DsResidentArgs* r, int sm_count, cudaStream_t s, bool pdl,
                             int* cuda_err) {
  *cuda_err = 0;
  if (t->n_ds == 0) return 0;
  const uint32_t want = (t->n_ds + 127u) / 128u;
  const uint32_t cap = (uint32_t)sm_count * 16u;
  const cudaError_t e = launch_pdl(ds_sweep_kernel<true>, dim3(want < cap ? want : cap), dim3(128), 0, s, pdl, *t, *r);
  if (e != cudaSuccess) {
    *cuda_err = (int)e;
    return -1;
  }
  return 1;
}

}  // namespace lwse
