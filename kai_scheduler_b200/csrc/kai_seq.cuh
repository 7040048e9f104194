// kai_seq.cuh — the sequencer: job-order tree, capacity policy, statement log and the allocate
// bookkeeping, written once and compiled for BOTH sides:
//   * device: lane 0 of warp 0 of CTA 0 of k_action (device-resident mode)
//   * host:   a CPU thread of libkaigpu.so driving the scan-server kernel (host-sequenced mode)
// Backend-specific pieces (publishing a decision record, gathering candidates, flushing the delta
// list) are supplied by kai_action.cuh (device) and kai_host_seq.cuh (host).
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "kai_device.cuh"

#define KAI_HD __host__ __device__

namespace kai {

// ---- arithmetic / memory wrappers: IEEE binary64, no contraction, on both sides ----
KAI_HD inline double kadd(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(a, b);
#else
  return a + b;  // host translation unit is built with -ffp-contract=off
#endif
}
KAI_HD inline double ksub(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
KAI_HD inline double kmul(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
KAI_HD inline double kdiv(double a, double b) {
#ifdef __CUDA_ARCH__
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
template <class T>
KAI_HD inline T kldg(const T *p) {
#ifdef __CUDA_ARCH__
  return __ldg(p);
#else
  return *p;
#endif
}
KAI_HD inline unsigned long long kbits(double x) {
  unsigned long long u;
  memcpy(&u, &x, 8);
  return u;
}
KAI_HD inline long long kclock() {
#ifdef __CUDA_ARCH__
  return clock64();
#else
  return 0;
#endif
}
// self-validating 128-bit word {data, tag}: device = one relaxed 128-bit store; host = data then tag (release)
KAI_HD inline void store_tagged(unsigned long long *p, unsigned long long data, unsigned long long tag) {
#ifdef __CUDA_ARCH__
  asm volatile("{ .reg .b128 q; mov.b128 q, {%1, %2}; st.relaxed.gpu.global.b128 [%0], q; }" ::"l"(p), "l"(data), "l"(tag)
               : "memory");
#else
  __atomic_store_n(p, data, __ATOMIC_RELAXED);
  __atomic_store_n(p + 1, tag, __ATOMIC_RELEASE);
#endif
}
KAI_HD inline double requestable_share(double max_allowed, double request) {
  if (max_allowed == KAI_UNLIMITED) return request;
  return fmin(max_allowed, request);
}
// resource_share.go:51-61
KAI_HD inline double allocatable_share(double deserved, double fair, double max_allowed) {
  if (deserved == KAI_UNLIMITED) return max_allowed;
  double a = fmax(deserved, fair);
  if (max_allowed != KAI_UNLIMITED) a = fmin(max_allowed, a);
  return a;
}
// resource_quantities.go:81-97
KAI_HD inline int compare_quantities(double q, double o) {
  if (q == KAI_UNLIMITED) return o == KAI_UNLIMITED ? 0 : 1;
  if (o == KAI_UNLIMITED) return -1;
  if (q > o) return 1;
  if (q < o) return -1;
  return 0;
}

constexpr unsigned long long kKeyNone = ~0ull;
constexpr uint32_t kRankNone = 0xFFFFFFu;  // 24-bit rank field
constexpr int kMaxRepeat = 10;             // 6 flag bits per repeat in one 64-bit word

KAI_HD inline unsigned long long make_job_key(int priority, int cls, int order_rank) {
  unsigned long long pinv = (unsigned long long)(unsigned int)(0x40000000 - priority) & 0x7fffffffull;
  return (pinv << 33) | ((unsigned long long)cls << 31) | (unsigned long long)(order_rank & 0x7fffffff);
}

// ---------------------------------------------------------------------------------------------
// action kernel state
// ---------------------------------------------------------------------------------------------
struct Track {  // global min/max of NonAllocated(res) over nodes with Allocatable(res) != 0 (pack.go:66-86)
  double mn, mx;
  int cnt_mn, cnt_mx;
  int dirty;
};

struct Decision {
  double req[KAI_MAX_RES];
  double mn, mx;
  int task, res, strategy, gpu_task, pipeline_only, nominated, pred_class, best_effort;
  int restricted;  // sweep only the rows of the current feasible-node set (solver simulations)
};

// tracker event bits per resource (gpu bits 0-2, cpu bits 3-5)
enum { WF_B_EQ_MX = 1, WF_A_EQ_MN = 2, WF_A_LT_MN = 4 };
enum { SLOT_TO_IDLE = 64, SLOT_HAS_REPEAT = 128 };

struct Winner {
  double score;
  uint32_t rank;
  uint32_t flags;
  int node;
};

struct Batch {  // same-node batching state
  int valid, node, to_idle, left, idx;
  unsigned long long fl;  // 6 tracker-event bits per repeat
};

enum { DK_SCAN = 1, DK_MINMAX = 2, DK_FLUSH = 3, DK_DONE = 4, DK_TOPK = 5 };
// extra record bits (word 0 bits 48..63).  XB_SNAP_*: after the deltas of the record, every scanner recomputes the
// feasible-set bit of its rows (common.FeasibleNodesForJob: all nodes / nodes with idle or releasing GPUs).
// XB_FUSED_MM: the scanners exchange their local binpack min/max among themselves (device slots) before scoring, so a
// sweep over a changed node set needs no separate MINMAX round trip through the host.
// XB_SINGLE: answer this SCAN with the single best row through the relay's reduction (cheaper sweep when the
// list would be used once: heterogeneous requests, solver simulations) instead of the top-M lists.
// XB_RESTRICT_DOM: sweep only the rows of the topology domain selected by the last EXT_SELECT entry.
enum { XB_RESTRICT = 1, XB_SNAP_ALL = 2, XB_SNAP_GPUFREE = 4, XB_FUSED_MM = 8, XB_SINGLE = 16, XB_RESTRICT_DOM = 32 };
constexpr uint32_t kTileDom = 1u << 29;  // tile flag bits 29, 28, 27, 26: row belongs to the domain selected in slot 0..3
constexpr int kDomSlots = 4;             // nesting depth of SubGroupSet / PodSet constraints the scanners can intersect
// XB_RESTRICT_DOM sweeps carry the number of active slots in xbits bits 8..10: a row must sit in all of them
KAI_HD inline uint32_t dom_need_mask(unsigned int xbits) {
  const unsigned int n = (xbits >> 8) & 7u;
  uint32_t m = 0;
  for (unsigned int i = 0; i < n && i < (unsigned int)kDomSlots; i++) m |= kTileDom >> i;
  return m;
}
// Extended delta entries (low word bit 31 set; every scanner applies them, they name no row):
//   [31]=1 [30:28]=kind [27:0]=a | b
enum {
  EXT_SELECT = 0,       // a = (level + 1) | slot << 8, b = domain id: slot bit = (dom[level][row] == b)
  EXT_SELECT_ROOT = 1,  // a = lb | le << 8 | slot << 16: slot bit = the row carries every level label of topology [lb, le)
  EXT_SCORE_BEGIN = 2,  // a = preferred level (global): clear the per-domain bucket table, scoring on
  EXT_SCORE = 3,        // a = domain id at the preferred level, b = bucket: node score = bucket * scores.Topology
  EXT_SCORE_END = 4     // scoring off
};
constexpr uint32_t kTileFeas = 1u << 30;  // tile flag bit: row belongs to the feasible-node set
enum { DB_GPU_TASK = 1, DB_BEST_EFFORT = 2, DB_PIPELINE_ONLY = 4, DB_BATCHING = 8, DB_DIRTY0 = 16, DB_DIRTY1 = 32 };

struct Ctl {  // sequencer control block (shared memory of CTA 0), written by lane 0
  int job, n_items, job_ok, item_ok, need_minmax, use_batch, stop;
  unsigned int seq;  // sequence number of the next decision record
  int n_delta;       // node deltas queued for the next record
  unsigned int xbits;  // XB_* bits of the next record
  unsigned int last_dkey;  // last queued delta: rank | code << 28, its first task and its repeat count
  int last_dtask, last_dcount;
  Decision dec;
  Winner win;
  Track trk[2];  // 0 gpu, 1 cpu
  Batch batch;
  unsigned long long dw[kDecWords];
  // context of the job being allocated: its podset counters stay here and are written back at the end
  int ctx_job, ctx_ps, ctx_fresh, ctx_queue, ctx_preempt, ctx_base;
  int ctx_cnt[3];
};

struct Tile {  // shared-memory node tile of this CTA
  double *I, *L;        // [R][npc]
  double *Agpu, *Acpu;  // [npc]
  double *gpu_count;    // [npc]
  int *rank;            // [npc]
  uint32_t *flags;      // [npc]
  int *node;            // [npc] node index of the row
  int *dom;             // [n_dom_levels][npc] topology domain per level
  int n_dom_levels;
  int npc, count, R;
  // Rows are striped by NAME RANK over the GPUs of the box and over the scanners of a GPU: row j of scanner `my`
  // of shard `shard` is the node of name rank (j * nscan + my) * nshard + shard.  Consecutive ranks land on
  // different scanners, so the global top-K rows of a sweep come from ~K different scanners.
  int nscan, my, nshard, shard;
  int nscan_log2;  // log2(nscan) when nscan is a power of two, else -1
};
KAI_HD inline int tile_row_rank(const Tile &tl, int ln) { return (ln * tl.nscan + tl.my) * tl.nshard + tl.shard; }
KAI_HD inline bool tile_owns(const Tile &tl, unsigned int rank, int &ln) {
  unsigned int q = rank;
  if (tl.nshard != 1) {  // one GPU: every rank is this shard's
    q = rank / (unsigned int)tl.nshard;
    if (rank - q * (unsigned int)tl.nshard != (unsigned int)tl.shard) return false;
  }
  unsigned int j;
  if (tl.nscan_log2 >= 0) {  // scanner count is a power of two (256 by default): no integer division on the device
    j = q >> tl.nscan_log2;
    if ((q & ((1u << tl.nscan_log2) - 1u)) != (unsigned int)tl.my) return false;
  } else {
    j = q / (unsigned int)tl.nscan;
    if (q - j * (unsigned int)tl.nscan != (unsigned int)tl.my) return false;
  }
  ln = (int)j;
  return true;
}

struct Seq {  // sequencer state (lane 0 of warp 0 of CTA 0)
  const DevSnap *s;
  const kai_config *cfg;
  const ActionParams *p;
  unsigned long long *delta_base;  // tagged node-delta words [2][kMaxDelta] (device memory or pinned host memory)
  void *host_backend;               // host-sequenced mode: HostBackend*
  double *mirror;                   // host-sequenced mode: Idle / Releasing of ALL nodes, node-major [N][2][R] (one cache
                                    // line per node), kept in step with the deltas (solver look-ups, topology domain
                                    // sums; identical on every rank)
  void *topology;                   // host-sequenced mode: TopologyHost* (or null)
  void (*on_node_changed)(void *topology, int node, const double *before, const double *after);  // Idle+Releasing per resource
  Replica rp;
  Tile *tile;
  Ctl *ctl;
  int n_ops, ops_cap;
  int root_len;
  int batching;
  bool is_cta0;
  long long pods_placed, pods_evicted, sweeps, nodes_scanned, n_visits, minmax_exchanges, batched;
  kai_job_visit *visits;
  int visits_cap;
  int error;
  long long t_pop, t_prep, t_scan, t_xchg, t_apply, t_finish, t_init;  // clock64 phase totals (thread 0)
  long long t_key, n_key, t_tta, t_heap;
  // host-sequenced mode, KAI_PROFILE only: rdtsc split of pop_next_job (null = off; never set on the device)
  unsigned long long *pop_split;  // [4]: fix root heap, fix child heaps, key recomputation, leaf pop + handle_pop
  unsigned long long pop_mark;
  long long pop_key_mark;
};

KAI_HD inline double &q_alloc(Seq &q, int r, int qi) { return q.rp.q_alloc[(size_t)r * q.s->Q + qi]; }
KAI_HD inline double &q_alloc_np(Seq &q, int r, int qi) {
  return q.rp.q_alloc_np[(size_t)r * q.s->Q + qi];
}
KAI_HD inline void invalidate_chain(Seq &q, int qi) {
  for (int c = qi; c >= 0; c = kldg(&q.s->q_parent[c])) q.rp.qkey[c].valid = 0;
}

KAI_HD inline bool job_touched(const Seq &q, int j) { return (q.rp.touched[j >> 5] >> (j & 31)) & 1u; }
KAI_HD inline void prefetch_l1(const void *ptr) {
#ifdef __CUDA_ARCH__
  asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr));
#else
  __builtin_prefetch(ptr);
#endif
}
// podset status counters: those of the job being allocated live in the control block
KAI_HD inline int ps_get(const Seq &q, int ps, int which) {
  if (ps == q.ctl->ctx_ps) return q.ctl->ctx_cnt[which];
  return q.rp.ps_active_alloc[(size_t)which * q.s->S + ps];
}
KAI_HD inline void ps_add(Seq &q, int ps, int which, int d) {
  if (ps == q.ctl->ctx_ps)
    q.ctl->ctx_cnt[which] += d;
  else
    q.rp.ps_active_alloc[(size_t)which * q.s->S + ps] += d;
}

// ---- PodInfo helpers ----
KAI_HD inline bool should_allocate(const Seq &q, int t, bool real) {  // pod_info.go:518-521
  int st = q.rp.t_status[t];
  return st == KAI_POD_PENDING || (!real && st == KAI_POD_RELEASING && q.rp.t_virtual[t]);
}

// ---- node mutations (node_info.go:457-551) are queued as deltas for the scanner that owns the node ----
enum { ND_ADD = 0, ND_ADD_PIPELINED = 1, ND_ADD_RELEASING = 2, ND_REM = 3, ND_REM_PIPELINED = 4, ND_REM_RELEASING = 5,
       ND_FEAS_SET = 6, ND_FEAS_CLR = 7 };  // 6, 7: feasible-set membership of the row (no task attached)
KAI_HD void seq_flush_deltas(Seq &q);  // FLUSH exchange when the delta list is full (backend specific)
// applied by the owning scanner to its tile row (lane r handles resource r)
KAI_HD inline void apply_delta_row(double &I, double &L, int code, double v) {
  switch (code) {
    case ND_ADD: I = ksub(I, v); break;
    case ND_ADD_PIPELINED: L = ksub(L, v); break;
    case ND_ADD_RELEASING: L = kadd(L, v); I = ksub(I, v); break;
    case ND_REM: I = kadd(I, v); break;
    case ND_REM_PIPELINED: L = kadd(L, v); break;
    case ND_REM_RELEASING: L = ksub(L, v); I = kadd(I, v); break;
  }
}

// Every delta word is written exactly once (readers validate it by its tag only): the newest entry stays pending in
// the control block, so that consecutive deltas of the same kind on the same row with bit-identical requests can be
// folded into it as a repeat count (tag word bits 32+; the owner applies the same subtraction `count` times, in
// order).  close_delta() writes the pending entry; the backends call it before a record is published.
KAI_HD void close_delta(Ctl &c, unsigned long long *delta_base) {
  if (c.n_delta > 0 && c.last_dcount > 0) {
    unsigned long long data = (unsigned long long)c.last_dkey | ((unsigned long long)(unsigned int)c.last_dtask << 32);
    store_tagged(delta_base + ((size_t)(c.seq & 1) * kMaxDelta + c.n_delta - 1) * 2, data,
                 (unsigned long long)c.seq | ((unsigned long long)(c.last_dcount - 1) << 32));
  }
  c.last_dcount = 0;
}
KAI_HD void emit_delta(Seq &q, int node, int code, int t) {
  Ctl &c = *q.ctl;
#ifndef __CUDA_ARCH__
  if (q.mirror && code < ND_FEAS_SET) {
    const int R_ = q.s->R;
    double *row = q.mirror + (size_t)node * 2 * R_;
    const double *rq = q.s->t_req + (size_t)t * R_;
    if (q.topology) {
      double before[KAI_MAX_RES], after[KAI_MAX_RES];
      for (int r = 0; r < R_; r++) {
        before[r] = row[r] + row[R_ + r];
        apply_delta_row(row[r], row[R_ + r], code, rq[r]);
        after[r] = row[r] + row[R_ + r];
      }
      q.on_node_changed(q.topology, node, before, after);
    } else {
      for (int r = 0; r < R_; r++) apply_delta_row(row[r], row[R_ + r], code, rq[r]);
    }
  }
#endif
  // the delta names the node by its NAME RANK: that is what decides which scanner owns the row
  const unsigned int key = (unsigned int)(kldg(&q.s->name_rank[node]) | (code << 28));
  if (code < ND_FEAS_SET && c.n_delta > 0 && c.last_dcount > 0 && c.last_dkey == key && c.last_dcount < 255) {
    const int R = q.s->R;
    const double *a = q.s->t_req + (size_t)c.last_dtask * R, *b = q.s->t_req + (size_t)t * R;
    bool same = true;
    for (int r = 0; r < R; r++) same = same && kbits(kldg(&a[r])) == kbits(kldg(&b[r]));
    if (same) {
      c.last_dcount++;
      return;
    }
  }
  close_delta(c, q.delta_base);
  if (c.n_delta >= kMaxDelta) seq_flush_deltas(q);
  c.n_delta++;
  c.last_dkey = key;
  c.last_dtask = t;
  c.last_dcount = 1;
}
// extended entry: applied by every scanner (topology domain selection / score table)
KAI_HD void emit_ext(Seq &q, int kind, unsigned int a, unsigned int b) {
  Ctl &c = *q.ctl;
  close_delta(c, q.delta_base);
  if (c.n_delta >= kMaxDelta) seq_flush_deltas(q);
  c.n_delta++;
  c.last_dkey = 0x80000000u | ((unsigned int)kind << 28) | (a & 0x0fffffffu);
  c.last_dtask = (int)b;
  c.last_dcount = 1;
  close_delta(c, q.delta_base);  // written at once; never folded
}
KAI_HD void node_add_task(Seq &q, int t, int n, int st) {  // n = task node, st = task status (just set)
  q.rp.t_node_status[t] = st;
  emit_delta(q, n, st == KAI_POD_RELEASING ? ND_ADD_RELEASING : (st == KAI_POD_PIPELINED ? ND_ADD_PIPELINED : ND_ADD), t);
}
KAI_HD void node_remove_task(Seq &q, int t, int n) {
  int st = q.rp.t_node_status[t];
  emit_delta(q, n, st == KAI_POD_RELEASING ? ND_REM_RELEASING : (st == KAI_POD_PIPELINED ? ND_REM_PIPELINED : ND_REM), t);
}
// ---- PodGroupInfo.UpdateTaskStatus (job_info.go:253-264) + podset counters ----
// job / old may be passed when the caller already knows them (saves dependent L2 loads)
KAI_HD void set_status(Seq &q, int t, int status, int job = -1, int old = -1) {
  Ctl &c = *q.ctl;
  if (old < 0) old = q.rp.t_status[t];
  int j = job >= 0 ? job : kldg(&q.s->t_job[t]);
  int ps = (j == c.ctx_job && c.ctx_ps >= 0) ? c.ctx_ps : kldg(&q.s->t_podset[t]);
  if (old & kActiveAllocated) ps_add(q, ps, 0, -1);
  if (status & kActiveAllocated) ps_add(q, ps, 0, +1);
  if (old == KAI_POD_PENDING) ps_add(q, ps, 1, -1);
  if (status == KAI_POD_PENDING) ps_add(q, ps, 1, +1);
  if (old == KAI_POD_PIPELINED) ps_add(q, ps, 2, -1);
  if (status == KAI_POD_PIPELINED) ps_add(q, ps, 2, +1);
  q.rp.t_status[t] = status;
  q.rp.j_req_valid[j] = 0;
  q.rp.touched[j >> 5] |= 1u << (j & 31);
  int qi = j == c.ctx_job ? c.ctx_queue : kldg(&q.s->j_queue[j]);
  invalidate_chain(q, qi);  // the job may be the best pending job of its queue chain
}

// ---- proportion event handlers (proportion.go:443-489) ----
KAI_HD void queue_allocate(Seq &q, int t, bool add, int job = -1) {
  const DevSnap &s = *q.s;
  Ctl &c = *q.ctl;
  int j = job >= 0 ? job : kldg(&s.t_job[t]);
  bool preemptible;
  int qi;
  if (j == c.ctx_job) {
    preemptible = c.ctx_preempt != 0;
    qi = c.ctx_queue;
  } else {
    preemptible = (kldg(&s.j_flags[j]) & KAI_JOB_PREEMPTIBLE) != 0;
    qi = kldg(&s.j_queue[j]);
  }
  double v[QR];
  if (t == c.dec.task)
    for (int r = 0; r < QR; r++) v[r] = c.dec.req[r];
  else
    for (int r = 0; r < QR; r++) v[r] = kldg(&s.t_req[(size_t)t * s.R + r]);
  for (; qi >= 0; qi = kldg(&s.q_parent[qi])) {
    for (int r = 0; r < QR; r++) {
      double &a = q_alloc(q, r, qi);
      a = add ? kadd(a, v[r]) : ksub(a, v[r]);
      if (!preemptible) {
        double &b = q_alloc_np(q, r, qi);
        b = add ? kadd(b, v[r]) : ksub(b, v[r]);
      }
    }
    q.rp.qkey[qi].valid = 0;
  }
}

// ---- Statement (framework/statement.go) ----
KAI_HD void push_op(Seq &q, const Op &op) {
  if (q.n_ops >= q.ops_cap) {
    q.error = 1;
    return;
  }
  q.rp.ops[q.n_ops++] = op;
}
// `fresh`: the task belongs to the context job and is known to be Pending / unplaced / not virtual
KAI_HD void stmt_place(Seq &q, int t, int n, int kind, bool fresh) {  // :297-358 Allocate, :197-295 Pipeline
  Op op;
  op.kind = kind;
  op.task = t;
  if (fresh) {
    op.prev_status = KAI_POD_PENDING;
    op.prev_node = -1;
    op.prev_virtual = 0;
  } else {
    op.prev_status = q.rp.t_status[t];
    op.prev_node = q.rp.t_node[t];
    op.prev_virtual = q.rp.t_virtual[t];
  }
  op.next_node = n;
  op.undo_index = -1;
  op.pad = 0;
  int job = fresh ? q.ctl->ctx_job : -1;
  int st = kind == OP_ALLOCATE ? KAI_POD_ALLOCATED : KAI_POD_PIPELINED;
  set_status(q, t, st, job, op.prev_status);
  q.rp.t_node[t] = n;
  node_add_task(q, t, n, st);
  queue_allocate(q, t, true, job);
  push_op(q, op);
  q.rp.t_virtual[t] = 1;
}
KAI_HD void stmt_allocate(Seq &q, int t, int n, bool fresh = false) { stmt_place(q, t, n, OP_ALLOCATE, fresh); }
KAI_HD void stmt_pipeline(Seq &q, int t, int n, bool fresh = false) { stmt_place(q, t, n, OP_PIPELINE, fresh); }
KAI_HD void unallocate(Seq &q, int t, int prev_virtual) {  // :392-427
  set_status(q, t, KAI_POD_PENDING);
  node_remove_task(q, t, q.rp.t_node[t]);
  q.rp.t_node[t] = -1;
  q.rp.t_virtual[t] = (unsigned char)prev_virtual;
  queue_allocate(q, t, false);
}
KAI_HD void unpipeline(Seq &q, const Op &op) {  // :432-476
  int t = op.task;
  set_status(q, t, op.prev_status);
  int host = q.rp.t_node[t];
  q.rp.t_node[t] = op.prev_node;
  q.rp.t_virtual[t] = (unsigned char)op.prev_virtual;
  node_remove_task(q, t, host);
  queue_allocate(q, t, false);
}
KAI_HD void node_state_disturbed(Seq &q) {  // a node changed outside a sweep: trackers and batch are stale
  q.ctl->trk[0].dirty = q.ctl->trk[1].dirty = 1;
  q.ctl->batch.valid = 0;
}
KAI_HD void undo_op(Seq &q, int i) {  // :597-643 (allocate-action subset: no undo chains survive)
  Op op = q.rp.ops[i];
  if (op.kind == OP_ALLOCATE)
    unallocate(q, op.task, op.prev_virtual);
  else if (op.kind == OP_PIPELINE)
    unpipeline(q, op);
  node_state_disturbed(q);
}
KAI_HD void stmt_rollback(Seq &q, int cp) {  // :48-61
  for (int i = q.n_ops - 1; i >= cp; i--) undo_op(q, i);
  q.n_ops = cp;
}
KAI_HD void stmt_convert_all_allocated_to_pipelined(Seq &q, int job) {  // :483-520
  int n0 = q.n_ops;
  for (int i = 0; i < n0; i++) {
    Op op = q.rp.ops[i];
    if (op.kind != OP_ALLOCATE || q.s->t_job[op.task] != job) continue;
    int node = q.rp.t_node[op.task];
    unallocate(q, op.task, 1);
    stmt_pipeline(q, op.task, node);
  }
  int k = 0;
  for (int i = 0; i < q.n_ops; i++) {
    Op op = q.rp.ops[i];
    if (op.kind == OP_ALLOCATE && q.s->t_job[op.task] == job) continue;
    q.rp.ops[k++] = op;
  }
  q.n_ops = k;
  node_state_disturbed(q);
}
KAI_HD void stmt_commit(Seq &q) {  // :536-571
  for (int i = 0; i < q.n_ops; i++) {
    Op op = q.rp.ops[i];
    if (op.kind == OP_ALLOCATE) {
      // BindPod -> updatePodOnSession(Binding) (session.go:111-125): active-allocated -> active-allocated
      q.rp.t_status[op.task] = KAI_POD_BINDING;
      q.rp.t_node_status[op.task] = KAI_POD_BINDING;
      q.rp.j_req_valid[q.s->t_job[op.task]] = 0;
      q.pods_placed++;
    } else if (op.kind == OP_PIPELINE) {
      q.pods_placed++;
    } else if (op.kind == OP_EVICT) {
      q.pods_evicted++;
    }
  }
  q.n_ops = 0;
}

// ---- podset / task selection (api/podgroup_info/allocation_info.go) ----
KAI_HD bool podset_less(const Seq &q, int a, int b) {  // subgroup_order.go:31-62, name order = index order
  int ln = ps_get(q, a, 0), rn = ps_get(q, b, 0);
  int lm = kldg(&q.s->ps_min[a]), rm = kldg(&q.s->ps_min[b]);
  bool lsat = ln >= lm, rsat = rn >= rm;
  if (!lsat && !rsat) return a < b;
  if (!lsat) return true;
  if (!rsat) return false;
  double lr = kdiv((double)ln, (double)lm);
  double rr = kdiv((double)rn, (double)rm);
  if (lr < rr) return true;
  if (rr < lr) return false;
  return a < b;
}
KAI_HD int sorted_podsets(const Seq &q, int job, int *out) {
  int b = kldg(&q.s->j_ps_begin[job]), e = kldg(&q.s->j_ps_begin[job + 1]);
  if (e - b == 1) {
    out[0] = b;
    return 1;
  }
  int n = 0;
  for (int ps = b; ps < e; ps++) {  // insertion sort with the PodSetOrderFn total order
    int i = n++;
    while (i > 0 && podset_less(q, ps, out[i - 1])) {
      out[i] = out[i - 1];
      i--;
    }
    out[i] = ps;
  }
  return n;
}
// :27-54 GetTasksToAllocate; result into q.rp.tta, returns count.  If sum != null only accumulates the
// request of the selected tasks (GetTasksToAllocateInitResource :87-113).
KAI_HD int tasks_to_allocate(Seq &q, int job, bool real, double *sum) {
  const DevSnap &s = *q.s;
  int *order = q.rp.ps_order;
  int nps = sorted_podsets(q, job, order);
  int unsat = 0;
  for (int k = 0; k < nps; k++)
    if (ps_get(q, order[k], 0) < kldg(&s.ps_min[order[k]])) unsat++;
  int max_sets = unsat > 0 ? unsat : 1;
  int n_sets = 0, n = 0;
  if (sum) sum[0] = sum[1] = sum[2] = 0.0;
  for (int k = 0; k < nps && n_sets < max_sets; k++) {
    int ps = order[k];
    int tb = kldg(&s.ps_task_begin[ps]), te = kldg(&s.ps_task_begin[ps + 1]);
    int n_alloc = ps_get(q, ps, 0);
    int m = kldg(&s.ps_min[ps]);
    int max_tasks = n_alloc >= m ? 1 : m - n_alloc;  // :144-153
    int taken = 0;
    for (int i = tb; i < te && taken < max_tasks; i++) {
      int t = i;  // tasks of a podset are stored in TaskOrderFn order
      if (!should_allocate(q, t, real)) continue;
      if (sum)
        for (int r = 0; r < QR; r++) sum[r] = kadd(sum[r], kldg(&s.t_req[(size_t)t * s.R + r]));
      else
        q.rp.tta[n] = t;
      n++;
      taken++;
    }
    if (taken > 0) n_sets++;
  }
  return n;
}
KAI_HD const double *job_init_resource(Seq &q, int job) {
  if (!job_touched(q, job)) {
    const JobRec *rec = q.s->jrec + job;
    if (rec->n_podsets == 1) return rec->req0;
  }
  double *c = q.rp.j_req + (size_t)job * QR;
  if (!q.rp.j_req_valid[job]) {
    tasks_to_allocate(q, job, false, c);
    q.rp.j_req_valid[job] = 1;
  }
  return c;
}
KAI_HD bool has_tasks_to_allocate(const Seq &q, int job) {  // :18-25 (isRealAllocation = true)
  for (int ps = kldg(&q.s->j_ps_begin[job]); ps < kldg(&q.s->j_ps_begin[job + 1]); ps++)
    if (ps_get(q, ps, 1) > 0) return true;
  return false;
}
// job_info.go:443-464 ShouldPipelineJob
KAI_HD bool should_pipeline_job(const Seq &q, int job) {
  for (int ps = kldg(&q.s->j_ps_begin[job]); ps < kldg(&q.s->j_ps_begin[job + 1]); ps++) {
    int pipe = ps_get(q, ps, 2);
    if (pipe > 0 && ps_get(q, ps, 0) - pipe < kldg(&q.s->ps_min[ps])) return true;
  }
  return false;
}

// ---- capacity policy (plugins/proportion/capacity_policy) ----
KAI_HD bool over_capacity(Seq &q, int job, const double *req) {
  const DevSnap &s = *q.s;
  bool preemptible = (kldg(&s.j_flags[job]) & KAI_JOB_PREEMPTIBLE) != 0;
  for (int qi = kldg(&s.j_queue[job]); qi >= 0; qi = kldg(&s.q_parent[qi]))
    for (int r = 0; r < QR; r++) {
      if (req[r] == 0) continue;
      double lim = kldg(&s.q_limit[(size_t)r * s.Q + qi]);
      if (lim != KAI_UNLIMITED && lim < kadd(q_alloc(q, r, qi), req[r])) return true;
    }
  if (preemptible) return false;
  for (int qi = kldg(&s.j_queue[job]); qi >= 0; qi = kldg(&s.q_parent[qi]))
    for (int r = 0; r < QR; r++) {
      if (req[r] == 0) continue;
      double d = kldg(&s.q_deserved[(size_t)r * s.Q + qi]);
      if (d != KAI_UNLIMITED && d < kadd(q_alloc_np(q, r, qi), req[r])) return true;
    }
  return false;
}

// ---- job-order tree (actions/utils/job_order_by_queue.go), one node per queue ----
KAI_HD inline bool qn_is_leaf(const Seq &q, int qi) { return kldg(&q.s->q_nchildren[qi]) == 0; }
KAI_HD inline int leaf_len(const Seq &q, int qi) {
  return (q.rp.leaf_end[qi] - q.rp.leaf_head[qi]) + q.rp.ovl_len[qi];
}
KAI_HD inline int qn_len(const Seq &q, int qi) {
  return qn_is_leaf(q, qi) ? leaf_len(q, qi) : q.rp.child_len[qi];
}
// the leaf priority queue: sorted run [head, end) + overflow heap for re-pushed jobs.  JobOrderFn
// (session_plugins.go:227-242: priority, elastic, creation, UID) is a strict total order on the packed key,
// so any exact priority queue pops in the same order as container/heap.
KAI_HD int leaf_peek(const Seq &q, int qi) {
  int h = q.rp.leaf_head[qi], e = q.rp.leaf_end[qi];
  int a = h < e ? q.rp.leaf_heap[h] : -1;
  int b = q.rp.ovl_len[qi] > 0 ? q.rp.leaf_heap[kldg(&q.s->q_job_begin[qi])] : -1;
  if (a < 0) return b;
  if (b < 0) return a;
  return q.rp.j_key[b] < q.rp.j_key[a] ? b : a;
}
KAI_HD int leaf_pop(Seq &q, int qi) {
  int h = q.rp.leaf_head[qi], e = q.rp.leaf_end[qi];
  int base = kldg(&q.s->q_job_begin[qi]);
  int a = h < e ? q.rp.leaf_heap[h] : -1;
  int n = q.rp.ovl_len[qi];
  int b = n > 0 ? q.rp.leaf_heap[base] : -1;
  bool from_ovl = a < 0 || (b >= 0 && q.rp.j_key[b] < q.rp.j_key[a]);
  if (!from_ovl) {
    q.rp.leaf_head[qi] = h + 1;
    return a;
  }
  // binary-heap pop on the overflow area
  int *it = q.rp.leaf_heap + base;
  n--;
  it[0] = it[n];
  int i = 0;
  for (;;) {
    int j1 = 2 * i + 1;
    if (j1 >= n) break;
    int j = j1;
    if (j1 + 1 < n && q.rp.j_key[it[j1 + 1]] < q.rp.j_key[it[j1]]) j = j1 + 1;
    if (!(q.rp.j_key[it[j]] < q.rp.j_key[it[i]])) break;
    int t = it[i];
    it[i] = it[j];
    it[j] = t;
    i = j;
  }
  q.rp.ovl_len[qi] = n;
  return b;
}
KAI_HD int elastic_class(const Seq &q, int job) {  // plugins/elastic/elastic.go:50-63
  bool exactly = true;
  for (int ps = kldg(&q.s->j_ps_begin[job]); ps < kldg(&q.s->j_ps_begin[job + 1]); ps++) {
    int n = ps_get(q, ps, 0), m = kldg(&q.s->ps_min[ps]);
    if (n < m) return 0;
    if (n > m) exactly = false;
  }
  return exactly ? 1 : 2;
}
KAI_HD void leaf_push(Seq &q, int qi, int job) {
  q.rp.j_key[job] = make_job_key(kldg(&q.s->j_priority[job]), elastic_class(q, job), kldg(&q.s->j_order_rank[job]));
  int base = kldg(&q.s->q_job_begin[qi]);
  int n = q.rp.ovl_len[qi];
  if (base + n >= q.rp.leaf_head[qi] && q.rp.leaf_head[qi] < q.rp.leaf_end[qi]) {
    q.error = 2;  // cannot happen while pushes follow pops
    return;
  }
  int *it = q.rp.leaf_heap + base;
  it[n] = job;
  int j = n;
  for (;;) {
    int i = (j - 1) / 2;
    if (i == j || !(q.rp.j_key[it[j]] < q.rp.j_key[it[i]])) break;
    int t = it[i];
    it[i] = it[j];
    it[j] = t;
    j = i;
  }
  q.rp.ovl_len[qi] = n + 1;
}
KAI_HD int best_job(Seq &q, int qi) {  // :283-292 getBestJobFromNode
  while (!qn_is_leaf(q, qi)) qi = q.rp.child_heap[kldg(&q.s->q_child_begin[qi])];
  return leaf_peek(q, qi);
}

// queue_order.go:19-73 on cached per-node keys.  A key is recomputed when the queue's Allocated or its
// best pending job changed since it was last used (invalidate_chain / queue_allocate).
// clock of the key-recomputation counter: clock64 on the device, rdtsc on the host while the pop is profiled
KAI_HD inline long long key_clock(const Seq &q) {
#ifdef __CUDA_ARCH__
  return clock64();
#else
  return q.pop_split ? (long long)__builtin_ia32_rdtsc() : 0;
#endif
}
// host pop profile: charge the time since the last mark to section i, less the key recomputations inside it
KAI_HD inline void pop_lap(Seq &q, int i) {
#ifndef __CUDA_ARCH__
  if (!q.pop_split) return;
  const unsigned long long t = __builtin_ia32_rdtsc();
  const long long keys = q.t_key - q.pop_key_mark;
  if (i >= 0) {
    q.pop_split[i] += (t - q.pop_mark) - (unsigned long long)keys;
    q.pop_split[2] += (unsigned long long)keys;
  }
  q.pop_mark = t;
  q.pop_key_mark = q.t_key;
#endif
}
KAI_HD const QKey &queue_key(Seq &q, int qi) {
  QKey &k = q.rp.qkey[qi];
  if (k.valid) return k;
  long long tkk = key_clock(q);
  q.n_key++;
  const DevSnap &s = *q.s;
  const double *req = job_init_resource(q, best_job(q, qi));
  bool over = true, starved = true, viol = false;
  double dj = 0.0, dr = 0.0;
  for (int r = 0; r < QR; r++) {
    size_t o = (size_t)r * s.Q + qi;
    double alloc = q.rp.q_alloc[o];
    double with_job = kadd(alloc, req[r]);
    if (kldg(&s.q_fair[o]) >= alloc) over = false;                                   // :87-100
    if (compare_quantities(with_job, kldg(&s.q_deserved[o])) > 0) starved = false;  // :102-128
    double la = kldg(&s.q_allocatable[o]);
    if (la == 0 && with_job > 0) viol = true;  // :130-180
    double denom = la == KAI_UNLIMITED ? s.total[r] : la;  // queue_resource_share.go:142-166
    double vj = denom == 0 ? kmul(with_job, 1000.0) : kdiv(with_job, denom);
    double vr = denom == 0 ? kmul(alloc, 1000.0) : kdiv(alloc, denom);
    dj = fmax(dj, vj);
    dr = fmax(dr, vr);
  }
  k.over = over;
  k.starved = starved;
  k.viol = viol;
  k.drf_job = dj;
  k.drf = dr;
  k.priority = kldg(&s.q_priority[qi]);
  k.w0 = ((unsigned long long)(over ? 1 : 0) << 44) | ((unsigned long long)(starved ? 0 : 1) << 43) |
         (((unsigned long long)(0x80000000LL - (long long)k.priority) & 0x1ffffffffull) << 10) | ((unsigned long long)(viol ? 1 : 0) << 9);
  k.valid = 1;
  q.t_key += key_clock(q) - tkk;
  return k;
}
KAI_HD bool node_less(Seq &q, int l, int r) {  // :256-278 buildNodeOrderFn (pending order)
  if (qn_len(q, l) == 0) return true;
  if (qn_len(q, r) == 0) return false;
  // over fair share last, starved first, higher priority first, limit violations last (packed: QKey::w0), then the
  // dominant shares with and without the best pending job
  const unsigned long long wl = queue_key(q, l).w0;
  const double jl = q.rp.qkey[l].drf_job, dl = q.rp.qkey[l].drf;
  const QKey &kr = queue_key(q, r);  // (a recomputation writes only the entry of r)
  if (wl != kr.w0) return wl < kr.w0;
  if (jl < kr.drf_job) return true;
  if (jl > kr.drf_job) return false;
  if (dl < kr.drf) return true;
  if (dl > kr.drf) return false;
  const DevSnap &s = *q.s;
  bool l_le_r = true, r_le_l = true;  // :221-233
  for (int i = 0; i < QR; i++) {
    double la = kldg(&s.q_allocatable[(size_t)i * s.Q + l]), ra = kldg(&s.q_allocatable[(size_t)i * s.Q + r]);
    if (compare_quantities(la, ra) > 0) l_le_r = false;
    if (compare_quantities(ra, la) > 0) r_le_l = false;
  }
  if (!r_le_l && l_le_r) return true;
  if (!l_le_r && r_le_l) return false;
  return kldg(&s.q_creation[l]) < kldg(&s.q_creation[r]);  // :235-240
}
// container/heap over queue nodes
KAI_HD void qheap_up(Seq &q, int *items, int j) {
  for (;;) {
    int i = (j - 1) / 2;
    if (i == j || !node_less(q, items[j], items[i])) break;
    int t = items[i];
    items[i] = items[j];
    items[j] = t;
    j = i;
  }
}
KAI_HD bool qheap_down(Seq &q, int *items, int i0, int n) {
  int i = i0;
  for (;;) {
    int j1 = 2 * i + 1;
    if (j1 >= n || j1 < 0) break;
    int j = j1;
    int j2 = j1 + 1;
    if (j2 < n && node_less(q, items[j2], items[j1])) j = j2;
    if (!node_less(q, items[j], items[i])) break;
    int t = items[i];
    items[i] = items[j];
    items[j] = t;
    i = j;
  }
  return i > i0;
}
KAI_HD void qheap_push(Seq &q, int *items, int &len, int x) {
  items[len++] = x;
  qheap_up(q, items, len - 1);
}
KAI_HD int qheap_pop(Seq &q, int *items, int &len) {
  int n = len - 1;
  int t = items[0];
  items[0] = items[n];
  items[n] = t;
  qheap_down(q, items, 0, n);
  len = n;
  return items[n];
}
KAI_HD void mark_ancestors(Seq &q, int qi) {  // :246-250 (+ key invalidation: best job / heap tops changed)
  for (int c = qi; c >= 0; c = kldg(&q.s->q_parent[c])) {
    q.rp.qn_flags[c] |= QN_REORDER;
    q.rp.qkey[c].valid = 0;
  }
}
KAI_HD void ensure_chain(Seq &q, int child) {  // :135-175
  for (;;) {
    int p = kldg(&q.s->q_parent[child]);
    if (p < 0) {
      if (!(q.rp.qn_flags[child] & QN_LINKED)) {
        qheap_push(q, q.rp.root_heap, q.root_len, child);
        q.rp.qn_flags[child] |= QN_LINKED;
      }
      return;
    }
    bool is_new = !(q.rp.qn_flags[p] & QN_EXISTS);
    if (is_new) {
      q.rp.qn_flags[p] = QN_EXISTS;
      q.rp.child_len[p] = 0;
    }
    if (!(q.rp.qn_flags[child] & QN_LINKED)) {
      qheap_push(q, q.rp.child_heap + kldg(&q.s->q_child_begin[p]), q.rp.child_len[p], child);
      q.rp.qn_flags[child] |= QN_LINKED;
      invalidate_chain(q, p);
    }
    if (!is_new) return;
    child = p;
  }
}
KAI_HD void push_job(Seq &q, int job) {  // :90-119
  int qi = kldg(&q.s->j_queue[job]);
  if (!qn_is_leaf(q, qi)) return;
  bool needs_linking = !(q.rp.qn_flags[qi] & QN_EXISTS);
  if (needs_linking) q.rp.qn_flags[qi] = QN_EXISTS;
  leaf_push(q, qi, job);
  invalidate_chain(q, qi);
  if (needs_linking) ensure_chain(q, qi);
  mark_ancestors(q, qi);
}
// owner = queue whose children heap `items` is (or -1 for the root heap)
KAI_HD int get_next_node(Seq &q, int *items, int &len, int owner) {  // :193-215
  for (;;) {
    if (len == 0) return -1;
    int ni = items[0];
    if (q.rp.qn_flags[ni] & QN_REORDER) {
      if (!qheap_down(q, items, 0, len)) qheap_up(q, items, 0);  // heap.Fix(0)
      q.rp.qn_flags[ni] &= ~QN_REORDER;
      if (owner >= 0) invalidate_chain(q, owner);
      continue;
    }
    if (qn_len(q, ni) == 0) return -1;
    return ni;
  }
}
KAI_HD void handle_pop(Seq &q, int qi) {  // :219-243
  for (;;) {
    if (qn_len(q, qi) == 0) {
      int p = kldg(&q.s->q_parent[qi]);
      if (p >= 0) {
        qheap_pop(q, q.rp.child_heap + kldg(&q.s->q_child_begin[p]), q.rp.child_len[p]);
        invalidate_chain(q, p);
      } else {
        qheap_pop(q, q.rp.root_heap, q.root_len);
      }
      q.rp.qn_flags[qi] = 0;
      q.rp.qkey[qi].valid = 0;
      if (p < 0) return;
      qi = p;
      continue;
    }
    mark_ancestors(q, qi);
    return;
  }
}
KAI_HD int pop_next_job(Seq &q) {  // :61-88
  if (q.root_len == 0) return -1;
  pop_lap(q, -1);
  int ni = get_next_node(q, q.rp.root_heap, q.root_len, -1);
  pop_lap(q, 0);
  while (ni >= 0 && !qn_is_leaf(q, ni))
    ni = get_next_node(q, q.rp.child_heap + kldg(&q.s->q_child_begin[ni]), q.rp.child_len[ni], ni);
  pop_lap(q, 1);
  if (ni < 0) return -1;
  int job = leaf_pop(q, ni);
  {  // warm L1 for the next pops of this queue
    int h = q.rp.leaf_head[ni], e = q.rp.leaf_end[ni];
    if (h < e) {
      const JobRec *r1 = q.s->jrec + q.rp.leaf_heap[h];
      prefetch_l1(r1);
      if (h + 1 < e) prefetch_l1(q.s->jrec + q.rp.leaf_heap[h + 1]);
    }
  }
  invalidate_chain(q, ni);
  handle_pop(q, ni);
  pop_lap(q, 3);
  return job;
}

// ---- min/max trackers ----
// update after a placement that lowered NonAllocated(res) of a node from b to a (a < b)
KAI_HD inline void track_decrease(Track &t, uint32_t f, double a) {
  if (t.dirty) return;
  if (f & WF_B_EQ_MX) {
    if (--t.cnt_mx == 0) {
      t.dirty = 1;
      return;
    }
  }
  if (f & WF_A_LT_MN) {
    t.mn = a;
    t.cnt_mn = 1;
  } else if (f & WF_A_EQ_MN) {
    t.cnt_mn++;
  }
}
KAI_HD inline uint32_t track_flags(const Track &t, double b, double a) {
  uint32_t f = 0;
  if (b == t.mx) f |= WF_B_EQ_MX;
  if (a < t.mn)
    f |= WF_A_LT_MN;
  else if (a == t.mn)
    f |= WF_A_EQ_MN;
  return f;
}

// decision record words (each stored as {data, tag}):
//   0  kind | res<<8 | strategy<<16 | bits<<24 | n_delta<<32      1  nominated | pred_class<<32
//   2..9 req[0..7]      10,11 gpu tracker mn,mx      12,13 cpu tracker mn,mx
//   14 gpu cnt_mn | cnt_mx<<32      15 cpu cnt_mn | cnt_mx<<32
KAI_HD void build_decision_words(Ctl &c, int kind, int batching) {
  const Decision &d = c.dec;
  unsigned long long bits = (d.gpu_task ? DB_GPU_TASK : 0) | (d.best_effort ? DB_BEST_EFFORT : 0) |
                            (d.pipeline_only ? DB_PIPELINE_ONLY : 0) | (batching ? DB_BATCHING : 0) |
                            (c.trk[0].dirty ? DB_DIRTY0 : 0) | (c.trk[1].dirty ? DB_DIRTY1 : 0);
  c.dw[0] = (unsigned long long)kind | ((unsigned long long)d.res << 8) | ((unsigned long long)d.strategy << 16) |
            (bits << 24) | ((unsigned long long)c.n_delta << 32) |
            ((unsigned long long)((c.xbits & 0xfffeu) | (d.restricted ? XB_RESTRICT : 0u)) << 48);
  c.dw[1] = (unsigned long long)(unsigned int)d.nominated | ((unsigned long long)(unsigned int)d.pred_class << 32);
  for (int r = 0; r < KAI_MAX_RES; r++) c.dw[2 + r] = kbits(d.req[r]);
  for (int k = 0; k < 2; k++) {
    c.dw[10 + 2 * k] = kbits(c.trk[k].mn);
    c.dw[11 + 2 * k] = kbits(c.trk[k].mx);
    c.dw[14 + k] = (unsigned long long)(unsigned int)c.trk[k].cnt_mn | ((unsigned long long)(unsigned int)c.trk[k].cnt_mx << 32);
  }
}

// =============================================================================================
// sequencer steps (lane 0)
// =============================================================================================
// InitializeWithJobs (input_jobs.go:21-68) in canonical order: leaf queues ascending, jobs of a queue in
// JobOrderFn order (the Go map order is unspecified; DESIGN.md §oracle).
KAI_HD void seq_init_job_order(Seq &q) {
  const DevSnap &s = *q.s;
  for (int qi = 0; qi < s.Q; qi++) {
    if (kldg(&s.q_nchildren[qi]) != 0) continue;
    if (leaf_len(q, qi) == 0) continue;
    q.rp.qn_flags[qi] = QN_EXISTS;
    ensure_chain(q, qi);
    mark_ancestors(q, qi);
  }
}

// builds ctl.dec for task t of `job`; returns false when the task cannot be placed at all
KAI_HD bool seq_prepare_task(Seq &q, int t, int job) {
  const DevSnap &s = *q.s;
  Ctl &c = *q.ctl;
  double rq[KAI_MAX_RES];
  for (int r = 0; r < KAI_MAX_RES; r++) rq[r] = r < s.R ? kldg(&s.t_req[(size_t)t * s.R + r]) : 0.0;
  int nominated = s.t_nominated ? kldg(&s.t_nominated[t]) : -1;
  int pred_class = s.t_pred_class ? kldg(&s.t_pred_class[t]) : -1;
  bool gpu_task = rq[KAI_RES_GPU] > 0;
  // predicates.go:196-200 -> capacity_policy.go:51-61 with node_info.go:734-744 (SURVEY Appendix C.1)
  double creq[QR] = {rq[KAI_RES_CPU], rq[KAI_RES_MEM], gpu_task ? 1.0 : 0.0};
  if (over_capacity(q, job, creq)) return false;
  bool empty = !(rq[KAI_RES_GPU] > 0.01) && !(rq[KAI_RES_CPU] >= 10) && !(rq[KAI_RES_MEM] >= 10.0 * 1024 * 1024);
  for (int r = 3; r < s.R; r++)
    if (rq[r] >= 10) empty = false;
  int strategy = gpu_task ? q.cfg->gpu_placement : q.cfg->cpu_placement;
  Decision &d = c.dec;
  // same request/flags as the previous sweep and the owner vouched for more placements on the same node?
  bool same = c.batch.valid && c.batch.left > 0 && d.gpu_task == (int)gpu_task && d.nominated == nominated &&
              d.pred_class == pred_class && d.best_effort == (int)empty && d.strategy == strategy &&
              d.pipeline_only == 0;
  if (same)
    for (int r = 0; r < KAI_MAX_RES; r++)
      if (d.req[r] != rq[r]) same = false;
  c.use_batch = same ? 1 : 0;
  c.need_minmax = 0;
  d.task = t;
  if (same) return true;
  c.batch.valid = 0;
  for (int r = 0; r < KAI_MAX_RES; r++) d.req[r] = rq[r];
  d.gpu_task = gpu_task;
  d.res = gpu_task ? KAI_RES_GPU : KAI_RES_CPU;
  d.strategy = strategy;
  d.pipeline_only = 0;
  d.nominated = nominated;
  d.pred_class = pred_class;
  d.best_effort = empty;
  c.need_minmax = (d.strategy == KAI_PLACEMENT_BINPACK) && c.trk[gpu_task ? 0 : 1].dirty;
  return true;
}

KAI_HD void seq_apply_winner(Seq &q, int t) {
  Ctl &c = *q.ctl;
  q.sweeps++;
  q.nodes_scanned += q.s->N;
  if (c.win.node < 0) {
    c.item_ok = 0;
    return;
  }
  if (c.win.flags & SLOT_TO_IDLE)
    stmt_allocate(q, t, c.win.node, c.ctx_fresh != 0);
  else
    stmt_pipeline(q, t, c.win.node, c.ctx_fresh != 0);
  c.item_ok = 1;
}
KAI_HD void seq_apply_batched(Seq &q, int t) {
  Ctl &c = *q.ctl;
  Batch &b = c.batch;
  uint32_t f6 = (uint32_t)((b.fl >> (6 * b.idx)) & 0x3fu);
  for (int k = 0; k < 2; k++) {
    uint32_t f = (f6 >> (3 * k)) & 7u;
    if (f) track_decrease(c.trk[k], f, 0.0);
  }
  b.idx++;
  b.left--;
  if (b.to_idle)
    stmt_allocate(q, t, b.node, c.ctx_fresh != 0);
  else
    stmt_pipeline(q, t, b.node, c.ctx_fresh != 0);
  q.batched++;
  c.item_ok = 1;
}

KAI_HD void record_visit(Seq &q, int job, int outcome) {
  if (q.n_visits < q.visits_cap) {
    q.visits[q.n_visits].job = job;
    q.visits[q.n_visits].outcome = outcome;
  }
  q.n_visits++;
}


}  // namespace kai
