// kai_host_seq.cuh — host backend of the sequencer (host-sequenced mode).
//
// The sequencer source (kai_seq.cuh) is compiled for the host as well.  A CPU thread of libkaigpu.so runs it against a
// host mirror of the session state and sends the GPU one decision record per node-table sweep:
//   * launch transport (default): publish() = one k_record launch carrying the record in its kernel parameters; list
//     answers come back as ONE merged, cut and sorted list per GPU (k_merge_cluster), single-row / min-max answers as one
//     line reduced by the last CTA; the host waits on a sequence tag in pinned host memory;
//   * persistent transport: the GPU runs k_action as a "scan server": CTA 0 relays the records the host writes into pinned
//     mapped memory to the scanners' device-side record buffer, the scanners keep their node tiles in shared memory and
//     answer every record with tagged 128-bit words written straight into pinned host memory.
//
// Why: measured on B200 (profiles/microbench, profiles/r01_sequencer_modes.md) one GPU lane needs ~20k
// cycles (10 us) of dependent L1/L2/shared-memory latencies per job for the pointer-chasing part of the
// cycle (heap pops, DRF keys, statement log); a host core does the same in a few hundred ns.  The O(N)
// work per allocateTask — the node sweep — stays on the GPU in both modes.
#pragma once
#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "kai_action.cuh"
#include "kai_job_order.cuh"
#include "kai_seq.cuh"
#include "kai_topology.cuh"

namespace kai {

struct HostBackend {
  // pinned, device-mapped buffers
  unsigned long long *h_rec = nullptr;    // [2][kDecWords][2]
  unsigned long long *h_delta = nullptr;  // [2][kMaxDelta][2]
  unsigned long long *h_slots = nullptr;  // [2][kMaxGrid][kSlotWords]
  unsigned long long *h_mm = nullptr;     // [2][kMaxGrid][kSlotWords]
  int n_scanners = 0;
  int batching = 1;
  double timeout_s = 20.0;
  bool failed = false;
  const int *rank_to_node = nullptr;  // host copy
  Ctl ctl;
  Seq seq;
  long long spins = 0;
  double t_exchange = 0, t_total = 0;  // seconds: waiting for the GPU / whole action
  // ---- top-M candidate lists ----
  unsigned long long *h_list = nullptr;  // [2][kListScanners][kListLines][kListLineWords]
  int topm = 0;
  int n_list_scanners = 0;  // scanners of all GPUs
  struct ListCand {
    double score;
    uint32_t rank, flags;
    int node, cap, used;
    double Ig, Lg, Ic, Lc;
    const unsigned long long *payload;
    bool loaded;
  };
  std::vector<ListCand> list;
  size_t list_pos = 0, list_valid = 0;
  long long listed = 0;

  static double now() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
  }
  // wait until the 64-bit word at p satisfies pred; false on timeout
  template <class Pred>
  bool wait_word(const unsigned long long *p, Pred pred, unsigned long long &out) {
    unsigned long long v = __atomic_load_n(p, __ATOMIC_ACQUIRE);
    if (pred(v)) {
      out = v;
      return true;
    }
    double t0 = now();
    for (unsigned long long it = 0;; it++) {
      v = __atomic_load_n(p, __ATOMIC_ACQUIRE);
      if (pred(v)) {
        out = v;
        return true;
      }
      __builtin_ia32_pause();
      if ((it & 0xffff) == 0xffff && now() - t0 > timeout_s) {
        failed = true;
        return false;
      }
    }
  }

  bool prof = false;
  // rdtsc: pop, admit, place (incl. sweeps), finish, loop, job-order eligibility check, job-order tree build
  unsigned long long t_sec[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  unsigned long long t_pop_split[4] = {0, 0, 0, 0};  // replica pop: fix root, fix children, keys, leaf pop + handle_pop
  // ---- job order of run_allocate: the keyed order (kai_job_order.cuh) when the snapshot allows it, else the replica ----
  bool keyed_order_allowed = true;  // false: KAI_JOB_ORDER=replica
  bool keyed_order_used = false;    // what the last run_allocate did
  KeyedJobOrder korder;
  int trace_kind[64];
  unsigned int trace_seq[64];
  int trace_nd[64];
  unsigned int trace_n = 0;
  // ---- launch transport: a record is a kernel launch (k_record), the answer one merged line / list per GPU ----
  bool launch_mode = false;
  void *launch_ctx = nullptr;
  bool (*launch_fn)(void *ctx, const LaunchRec &rec) = nullptr;  // kai_engine.cu: enqueues the launch(es) of one record
  unsigned long long *h_clist = nullptr;  // [ranks][2][kCListWords] merged candidate lists (pinned / shared host memory)
  int n_ranks = 1;
  LaunchRec lrec;
  long long launches = 0;
  double t_launch = 0;  // seconds inside the launch calls (KAI_PROFILE)
  void publish(int kind) {
    trace_kind[trace_n & 63] = kind;
    trace_seq[trace_n & 63] = ctl.seq;
    trace_nd[trace_n & 63] = ctl.n_delta;
    trace_n++;
    close_delta(ctl, seq.delta_base);
    build_decision_words(ctl, kind, batching);
    if (launch_mode) {
      for (int i = 0; i < kDecWords; i++) lrec.dw[i] = ctl.dw[i];
      lrec.seq = ctl.seq;
      lrec.n_delta = ctl.n_delta;
      const unsigned long long *dl = seq.delta_base + (size_t)(ctl.seq & 1) * kMaxDelta * 2;
      for (int e = 0; e < ctl.n_delta; e++) {
        lrec.dkey[e] = (unsigned int)(dl[2 * e] & 0xffffffffu);
        lrec.dtask[e] = (unsigned int)(dl[2 * e] >> 32);
        lrec.dcount[e] = (unsigned char)((dl[2 * e + 1] >> 32) & 0xffu);
      }
      launches++;
      const double tl = prof ? now() : 0.0;
      if (!launch_fn(launch_ctx, lrec)) failed = true;
      if (prof) t_launch += now() - tl;
      return;
    }
    unsigned long long *rec = h_rec + (size_t)(ctl.seq & 1) * kDecWords * 2;
    for (int i = kDecWords - 1; i >= 0; i--) store_tagged(rec + 2 * i, ctl.dw[i], (unsigned long long)ctl.seq);
  }

  // gather the candidate slots (written by the scanners over PCIe as single 16-byte stores)
  void gather_candidates() {
    const unsigned int seq_no = ctl.seq;
    const unsigned long long *buf = h_slots + (size_t)(seq_no & 1) * kMaxGrid * kSlotWords;
    const unsigned int tag = seq_no & 0xffffffu;
    double bs = -1.0;
    uint32_t brank = kRankNone, bmeta = 0;
    int bslot = -1;
    for (int c = 0; c < n_scanners; c++) {
      const unsigned long long *slot = buf + (size_t)c * kSlotWords;
      unsigned long long hi;
      if (!wait_word(slot + 1, [&](unsigned long long v) { return (unsigned int)(v >> 40) == tag; }, hi)) break;
      unsigned long long lo = __atomic_load_n(slot, __ATOMIC_RELAXED);
      double sc;
      memcpy(&sc, &lo, 8);
      uint32_t rk = (uint32_t)(hi & 0xffffffu);
      bool better_ = rk != kRankNone && (brank == kRankNone || sc > bs || (sc == bs && rk < brank));
      if (better_) {
        bs = sc;
        brank = rk;
        bmeta = (uint32_t)((hi >> 24) & 0xffffu);
        bslot = c;
      }
    }
    uint32_t bflags = bmeta >> 8, repeat = bmeta & 0xffu;
    ctl.win.score = bs;
    ctl.win.rank = brank;
    ctl.win.flags = bflags;
    ctl.win.node = brank == kRankNone ? -1 : rank_to_node[brank];
    ctl.batch.valid = 0;
    if (brank != kRankNone && !failed) {
      const unsigned long long *slot = buf + (size_t)bslot * kSlotWords;
      for (int k = 0; k < 2; k++) {
        uint32_t f = (bflags >> (3 * k)) & 7u;
        double a = 0;
        if (f & WF_A_LT_MN) {
          unsigned long long hi;
          if (!wait_word(slot + 2 + 2 * k + 1, [&](unsigned long long v) { return (unsigned int)v == tag; }, hi)) break;
          unsigned long long lo = __atomic_load_n(slot + 2 + 2 * k, __ATOMIC_RELAXED);
          memcpy(&a, &lo, 8);
        }
        if (f) track_decrease(ctl.trk[k], f, a);
      }
      if (repeat) {
        unsigned long long hi;
        if (wait_word(slot + 7, [&](unsigned long long v) { return (unsigned int)v == tag; }, hi)) {
          ctl.batch.valid = 1;
          ctl.batch.node = ctl.win.node;
          ctl.batch.to_idle = (bflags & SLOT_TO_IDLE) ? 1 : 0;
          ctl.batch.left = (int)repeat;
          ctl.batch.idx = 0;
          ctl.batch.fl = __atomic_load_n(slot + 6, __ATOMIC_RELAXED);
        }
      }
    }
    ctl.seq = seq_no + 1;
    ctl.n_delta = 0;
  }

  // Gather the top-M answers of every scanner, merge them into one list in key order and mark the prefix that
  // is provably the global order: entries strictly better than the last reported key of any scanner that has more
  // fitting rows than it reported.
  // launch transport: every GPU's last CTA has merged, cut and written its list; merge the lists of the ranks
  void gather_list_merged() {
    const unsigned int seq_no = ctl.seq;
    list.clear();
    bool have_cut = false;
    double cut_score = 0;
    uint32_t cut_rank = 0;
    for (int r = 0; r < n_ranks && !failed; r++) {
      const unsigned long long *cl = h_clist + ((size_t)r * 2 + (seq_no & 1)) * kCListWords;
      unsigned long long hi;
      if (!wait_word(cl + 1, [&](unsigned long long v) { return v == (unsigned long long)seq_no; }, hi)) break;
      const unsigned long long head = __atomic_load_n(cl, __ATOMIC_RELAXED);
      const int n = (int)(head & 0x7fffffffu);
      const bool more = ((head >> 31) & 1ull) != 0;
      for (int i = 0; i < n; i++) {
        const unsigned long long *e = cl + 2 + (size_t)i * kCEntryWords;
        ListCand lc;
        memcpy(&lc.score, &e[0], 8);
        const unsigned long long meta = e[1];
        lc.rank = (uint32_t)(meta & 0xffffffu);
        lc.flags = (uint32_t)((meta >> 32) & 0xffu);
        lc.node = rank_to_node[lc.rank];
        lc.cap = 1 + (int)((meta >> 24) & 0xffu);
        lc.used = 0;
        lc.payload = nullptr;
        lc.loaded = true;
        memcpy(&lc.Ig, &e[2], 8);
        memcpy(&lc.Lg, &e[3], 8);
        memcpy(&lc.Ic, &e[4], 8);
        memcpy(&lc.Lc, &e[5], 8);
        list.push_back(lc);
      }
      if (more && n > 0) {  // unseen rows of this GPU are worse than its last listed row
        const ListCand &last = list.back();
        if (!have_cut || last.score > cut_score || (last.score == cut_score && last.rank < cut_rank)) {
          have_cut = true;
          cut_score = last.score;
          cut_rank = last.rank;
        }
      }
    }
    if (n_ranks > 1)
      std::sort(list.begin(), list.end(), [](const ListCand &a, const ListCand &b) {
        return a.score > b.score || (a.score == b.score && a.rank < b.rank);
      });
    list_valid = list.size();
    if (have_cut && n_ranks > 1)
      for (size_t i = 0; i < list.size(); i++)
        if (!(list[i].score > cut_score || (list[i].score == cut_score && list[i].rank <= cut_rank))) {
          list_valid = i;
          break;
        }
    list_pos = 0;
    list_more = have_cut;
    list_tag = seq_no & 0xffffffu;
    ctl.seq = seq_no + 1;
    ctl.n_delta = 0;
    ctl.batch.valid = 0;
  }
  void gather_list() {
    if (launch_mode) return gather_list_merged();
    const unsigned int seq_no = ctl.seq;
    const unsigned int tag = seq_no & 0xffffffu;
    const unsigned long long *base = h_list + (size_t)(seq_no & 1) * kListScanners * kListLines * kListLineWords;
    list.clear();
    bool have_cut = false;
    double cut_score = 0;
    uint32_t cut_rank = 0;
    for (int c = 0; c < n_list_scanners && !failed; c++) {
      const unsigned long long *lines = base + (size_t)c * kListLines * kListLineWords;
      bool more = false;
      double last_score = 0;
      uint32_t last_rank = kRankNone;
      for (int m = 0; m < kTopM; m++) {
        unsigned long long hi;
        if (!wait_word(lines + 2 * m + 1, [&](unsigned long long v) { return (unsigned int)(v >> 40) == tag; }, hi)) break;
        unsigned long long lo = __atomic_load_n(lines + 2 * m, __ATOMIC_RELAXED);
        uint32_t rk = (uint32_t)(hi & 0xffffffu);
        uint32_t fl = (uint32_t)((hi >> 32) & 0xffu);
        if (fl & LF_MORE) more = true;
        if (rk == kRankNone) continue;
        ListCand lc;
        memcpy(&lc.score, &lo, 8);
        lc.rank = rk;
        lc.flags = fl;
        lc.node = rank_to_node[rk];
        lc.cap = 1 + (int)((hi >> 24) & 0xffu);
        lc.used = 0;
        lc.payload = lines + (size_t)(1 + m) * kListLineWords;
        lc.loaded = false;
        lc.Ig = lc.Lg = lc.Ic = lc.Lc = 0;
        list.push_back(lc);
        last_score = lc.score;
        last_rank = rk;
      }
      if (more && last_rank != kRankNone) {  // an unseen row of this scanner can be at most this good
        if (!have_cut || last_score > cut_score || (last_score == cut_score && last_rank < cut_rank)) {
          have_cut = true;
          cut_score = last_score;
          cut_rank = last_rank;
        }
      }
    }
    std::sort(list.begin(), list.end(), [](const ListCand &a, const ListCand &b) {
      return a.score > b.score || (a.score == b.score && a.rank < b.rank);
    });
    list_valid = list.size();
    if (have_cut)
      for (size_t i = 0; i < list.size(); i++)
        if (!(list[i].score > cut_score || (list[i].score == cut_score && list[i].rank <= cut_rank))) {
          list_valid = i;
          break;
        }
    // the cut row itself was reported (it IS the last reported row of that scanner): it may be used, rows after it not
    list_pos = 0;
    list_more = have_cut;
    list_tag = tag;
    ctl.seq = seq_no + 1;
    ctl.n_delta = 0;
    ctl.batch.valid = 0;
  }
  unsigned int list_tag = 0;
  bool list_more = false;
  bool batch_is_single = false;  // ctl.batch comes from a single-winner answer (same-node repeats), not from a list
  double list_yield_ema = 8.0;   // pods served per list, recent average
  long long list_served = -1;
  unsigned int single_streak = 0;
  long long single_sweeps = 0;
  void list_invalidate_keep_batch() {
    list_pos = list_valid = 0;
    list.clear();
    single_sweeps++;
  }  // some scanner has more qualifying rows than it reported
  bool list_available() const { return list_pos < list_valid && list[list_pos].used < list[list_pos].cap; }
  void list_invalidate() {
    list_pos = list_valid = 0;
    list.clear();
    ctl.batch.valid = 0;
  }
  // ---- fresh gangs: deferred bookkeeping ----
  // A gang whose tasks are untouched and interchangeable (JobRec::pad[0]) is placed task by task like any other job —
  // same sweeps, lists, capacity checks, node deltas and queue shares, in the same order — but the per-task writes of
  // Statement.Allocate / Pipeline that nothing reads before the gang is complete (task status / node / statement log,
  // PodSet counters) are made once at the end: in bulk when every task went to Idle resources (the job is committed
  // as it stands: statement.go:536-571), otherwise replayed in placement order so that the usual finish
  // (ShouldPipelineJob, ConvertAllAllocatedToPipelined, Commit) sees exactly the state the per-task path leaves.
  bool gang_mode = false, gang_fast = true;
  int gang_n = 0;
  std::vector<int> gang_node;
  std::vector<unsigned char> gang_idle;
  long long gang_bulk = 0, gang_replayed = 0, gang_failed = 0;
  void place(int t, int node, bool to_idle) {
    if (gang_mode) {
      gang_node[gang_n] = node;
      gang_idle[gang_n] = to_idle ? 1 : 0;
      gang_n++;
      emit_delta(seq, node, to_idle ? ND_ADD : ND_ADD_PIPELINED, t);  // node_info.go:457-493
      queue_allocate(seq, t, true, ctl.ctx_job);                      // proportion.go:443-466
      return;
    }
    if (to_idle)
      stmt_allocate(seq, t, node, ctl.ctx_fresh != 0);
    else
      stmt_pipeline(seq, t, node, ctl.ctx_fresh != 0);
  }
  bool place_fresh_gang(int job, int n, int base) {
    if ((int)gang_node.size() < n) {
      gang_node.resize(n);
      gang_idle.resize(n);
    }
    gang_n = 0;
    gang_mode = true;
    const bool ok = place_tasks(job, n);
    gang_mode = false;
    const DevSnap &s = *seq.s;
    if (!ok) {  // Discard (statement.go:522-534): undo in reverse order; the tasks' own fields were never written
      for (int k = gang_n - 1; k >= 0; k--) {
        emit_delta(seq, gang_node[k], gang_idle[k] ? ND_REM : ND_REM_PIPELINED, base + k);
        queue_allocate(seq, base + k, false, job);
      }
      if (gang_n > 0) {
        node_state_disturbed(seq);
        seq.rp.touched[job >> 5] |= 1u << (job & 31);
        seq.rp.j_req_valid[job] = 0;
        invalidate_chain(seq, ctl.ctx_queue);
      }
      gang_failed++;
      return false;
    }
    bool all_idle = gang_n == n;
    for (int k = 0; k < gang_n; k++) all_idle = all_idle && gang_idle[k];
    if (all_idle) {  // Allocate x n then Commit: Binding on the chosen nodes
      for (int k = 0; k < n; k++) {
        const int t = base + k;
        seq.rp.t_status[t] = KAI_POD_BINDING;
        seq.rp.t_node[t] = gang_node[k];
        seq.rp.t_node_status[t] = KAI_POD_BINDING;
        seq.rp.t_virtual[t] = 1;
      }
      ctl.ctx_cnt[0] += n;  // active allocated
      ctl.ctx_cnt[1] -= n;  // pending
      seq.rp.touched[job >> 5] |= 1u << (job & 31);
      seq.rp.j_req_valid[job] = 0;
      invalidate_chain(seq, ctl.ctx_queue);
      seq.pods_placed += n;
      gang_bulk++;
      return true;
    }
    for (int k = 0; k < gang_n; k++) {  // replay what stmt_place writes besides the node delta and the queue shares
      const int t = base + k;
      Op op;
      op.kind = gang_idle[k] ? OP_ALLOCATE : OP_PIPELINE;
      op.task = t;
      op.prev_status = KAI_POD_PENDING;
      op.prev_node = -1;
      op.prev_virtual = 0;
      op.next_node = gang_node[k];
      op.undo_index = -1;
      op.pad = 0;
      const int st = gang_idle[k] ? KAI_POD_ALLOCATED : KAI_POD_PIPELINED;
      set_status(seq, t, st, job, KAI_POD_PENDING);
      seq.rp.t_node[t] = gang_node[k];
      seq.rp.t_node_status[t] = st;
      push_op(seq, op);
      seq.rp.t_virtual[t] = 1;
    }
    (void)s;
    gang_replayed++;
    return true;
  }
  // seq_apply_winner / seq_apply_batched (kai_seq.cuh) with the placement routed through place()
  void apply_winner_host(int t) {
    seq.sweeps++;
    seq.nodes_scanned += seq.s->N;
    if (ctl.win.node < 0) {
      ctl.item_ok = 0;
      return;
    }
    place(t, ctl.win.node, (ctl.win.flags & SLOT_TO_IDLE) != 0);
    ctl.item_ok = 1;
  }
  void apply_batched_host(int t) {
    Batch &b = ctl.batch;
    uint32_t f6 = (uint32_t)((b.fl >> (6 * b.idx)) & 0x3fu);
    for (int k = 0; k < 2; k++) {
      uint32_t f = (f6 >> (3 * k)) & 7u;
      if (f) track_decrease(ctl.trk[k], f, 0.0);
    }
    b.idx++;
    b.left--;
    place(t, b.node, b.to_idle != 0);
    seq.batched++;
    ctl.item_ok = 1;
  }
  // Place task t on the current list candidate (pack.go / node_info.go arithmetic restated on the reported row
  // values), update the min/max trackers exactly and decide whether the list stays usable.
  bool apply_listed(int t) {
    if (!list_available()) return false;
    ListCand &lc = list[list_pos];
    const Decision &d = ctl.dec;
    if (!lc.loaded) {
      const unsigned int tag = list_tag;  // the sweep that produced the list (a FLUSH may have advanced ctl.seq since)
      double *dst[4] = {&lc.Ig, &lc.Lg, &lc.Ic, &lc.Lc};
      for (int w = 0; w < 4; w++) {
        unsigned long long hi;
        if (!wait_word(lc.payload + 2 * w + 1, [&](unsigned long long v) { return (unsigned int)v == tag; }, hi)) return false;
        unsigned long long lo = __atomic_load_n(lc.payload + 2 * w, __ATOMIC_RELAXED);
        memcpy(dst[w], &lo, 8);
      }
      lc.loaded = true;
    }
    const bool to_idle = (lc.flags & LF_TO_IDLE) != 0;
    bool scored_moved = false;
    for (int k = 0; k < 2; k++) {
      if (!(lc.flags & (k == 0 ? LF_HAS_GPU : LF_HAS_CPU))) continue;
      double &I = k == 0 ? lc.Ig : lc.Ic, &L = k == 0 ? lc.Lg : lc.Lc;
      const double rq = d.req[k == 0 ? KAI_RES_GPU : KAI_RES_CPU];
      const double b = kadd(I, L);
      if (to_idle)
        I = ksub(I, rq);
      else
        L = ksub(L, rq);
      const double a = kadd(I, L);
      Track &tr = ctl.trk[k];
      if (tr.dirty) continue;
      const Track before = tr;
      uint32_t f = track_flags(tr, b, a);
      if (f) track_decrease(tr, f, a);
      const bool scored = (k == 0) == (d.res == KAI_RES_GPU);
      if (scored && d.strategy == KAI_PLACEMENT_BINPACK && (tr.dirty || tr.mn != before.mn || tr.mx != before.mx))
        scored_moved = true;
    }
    place(t, lc.node, to_idle);
    lc.used++;
    listed++;
    list_served++;
    ctl.item_ok = 1;
    if (scored_moved) {  // every other key was computed under the old min/max
      list_invalidate();
      return true;
    }
    if (lc.used >= lc.cap) {
      if (lc.flags & LF_EXHAUSTED)
        list_pos++;  // the row no longer fits: the next entry is the reference's next pick
      else
        list_invalidate();  // the row could still take pods (cap / mode / score): sweep again
    }
    ctl.batch.valid = list_available() ? 1 : 0;
    ctl.batch.left = 1;
    return true;
  }

  void gather_minmax() {
    const unsigned int seq_no = ctl.seq;
    const unsigned long long *buf = h_mm + (size_t)(seq_no & 1) * kMaxGrid * kSlotWords;
    double gmn[2] = {DBL_MAX, DBL_MAX}, gmx[2] = {0, 0};
    long long cmn[2] = {0, 0}, cmx[2] = {0, 0};
    for (int c = 0; c < n_scanners && !failed; c++) {
      const unsigned long long *slot = buf + (size_t)c * kSlotWords;
      for (int k = 0; k < 2; k++) {
        unsigned long long hi, lo;
        double v;
        if (!wait_word(slot + 4 * k + 1, [&](unsigned long long x) { return (x >> 32) == (unsigned long long)seq_no; }, hi)) break;
        lo = __atomic_load_n(slot + 4 * k, __ATOMIC_RELAXED);
        memcpy(&v, &lo, 8);
        int cnt = (int)(hi & 0xffffffffu);
        if (cnt > 0) {
          if (cmn[k] == 0 || v < gmn[k]) {
            gmn[k] = v;
            cmn[k] = cnt;
          } else if (v == gmn[k])
            cmn[k] += cnt;
        }
        if (!wait_word(slot + 4 * k + 3, [&](unsigned long long x) { return (x >> 32) == (unsigned long long)seq_no; }, hi)) break;
        lo = __atomic_load_n(slot + 4 * k + 2, __ATOMIC_RELAXED);
        memcpy(&v, &lo, 8);
        cnt = (int)(hi & 0xffffffffu);
        if (cnt > 0) {
          if (cmx[k] == 0 || v > gmx[k]) {
            gmx[k] = v;
            cmx[k] = cnt;
          } else if (v == gmx[k])
            cmx[k] += cnt;
        }
      }
    }
    for (int k = 0; k < 2; k++) {  // pack.go:66-86: min starts at MaxFloat64, max at 0
      ctl.trk[k].mn = cmn[k] > 0 ? gmn[k] : DBL_MAX;
      ctl.trk[k].mx = (cmx[k] > 0 && gmx[k] > 0) ? gmx[k] : 0.0;
      ctl.trk[k].cnt_mn = (int)cmn[k];
      ctl.trk[k].cnt_mx = (int)cmx[k];
      ctl.trk[k].dirty = 0;
    }
    ctl.seq = seq_no + 1;
    ctl.n_delta = 0;
  }

  // One sweep answered with the single best row (ctl.dec prepared by the caller): binpack extremes over the row set
  // of THIS sweep (fused among the scanners on one GPU, through the host when sharded), then the scan.
  void sweep_single(unsigned int xb) {
    const bool one_gpu = seq.cfg->shard_count <= 1;
    const bool binpack = ctl.dec.strategy == KAI_PLACEMENT_BINPACK;
    ctl.batch.valid = 0;
    if (!one_gpu && binpack) {
      seq.minmax_exchanges++;
      ctl.xbits = xb & XB_RESTRICT_DOM;
      publish(DK_MINMAX);
      ctl.xbits = 0;
      gather_minmax();
      if (failed) return;
    }
    if (one_gpu) ctl.trk[0].dirty = ctl.trk[1].dirty = 1;
    ctl.xbits = xb | XB_SINGLE | ((one_gpu && binpack) ? XB_FUSED_MM : 0);
    const int keep = batching;
    batching = 0;
    publish(DK_SCAN);
    batching = keep;
    ctl.xbits = 0;
    gather_candidates();
    ctl.batch.valid = 0;
    seq.sweeps++;
    seq.nodes_scanned += seq.s->N;
  }

  // allocateTasksOnNodeSet (allocate.go:104-119) for the tasks of the context job: lists / same-node batches while
  // they apply, a sweep otherwise.  `tasks` = explicit list or null for the context's own range.
  unsigned int sweep_xbits = 0;  // XB_RESTRICT_DOM while a topology domain is the node set
  double t_topo[4] = {0, 0, 0, 0};
  long long n_topo_jobs = 0, n_topo_domains = 0, n_flush = 0;
  bool place_tasks(int job, int n, const int *tasks = nullptr) {
    bool job_success = true;
    for (int k = 0; k < n; k++) {
      int t = tasks ? tasks[k] : (ctl.ctx_base >= 0 ? ctl.ctx_base + k : seq.rp.tta[k]);
      if (!seq_prepare_task(seq, t, job)) {
        job_success = false;
        break;
      }
      if (ctl.use_batch) {
        if (topm && !batch_is_single) {
          if (apply_listed(t)) continue;
          ctl.batch.valid = 0;  // list ran dry between prepare and apply: fall through to a sweep
          ctl.use_batch = 0;
          if (!seq_prepare_task(seq, t, job)) {
            job_success = false;
            break;
          }
        } else {
          apply_batched_host(t);
          continue;
        }
      }
      if (ctl.need_minmax) {
        seq.minmax_exchanges++;
        ctl.xbits = sweep_xbits;
        publish(DK_MINMAX);
        ctl.xbits = 0;
        gather_minmax();
      }
      double tx = now();
      // Lists pay off when one sweep serves many pods.  When the recent lists served ~1 pod each (a different
      // request on almost every job) the sweep is asked to answer with the single best row instead (XB_SINGLE:
      // one scan round, one reduced line); every 128th sweep probes the list form again.
      bool as_list = topm != 0;
      if (as_list && list_yield_ema < 1.5 && (++single_streak & 127) != 0) as_list = false;
      ctl.xbits = ((topm && !as_list) ? XB_SINGLE : 0) | sweep_xbits;
      publish(DK_SCAN);
      ctl.xbits = 0;
      if (as_list) {
        if (list_served >= 0) list_yield_ema = 0.75 * list_yield_ema + 0.25 * (double)list_served;
        gather_list();
        list_served = 0;
        batch_is_single = false;
      } else {
        gather_candidates();
        batch_is_single = true;
        if (topm) list_invalidate_keep_batch();
      }
      t_exchange += now() - tx;
      if (failed) {
        job_success = false;
        break;
      }
      if (as_list) {
        seq.sweeps++;
        seq.nodes_scanned += seq.s->N;
        ctl.item_ok = 0;
        if (list_available()) apply_listed(t);
      } else {
        apply_winner_host(t);
      }
      if (!ctl.item_ok) {
        job_success = false;
        break;
      }
    }
    return job_success;
  }

  // AllocateJob for a job with nested SubGroupSets / topology constraints (allocate.go:36-83 with
  // topology.subSetNodesFn): the SubGroupSet tree is walked by TopoAllocator; this is the session side for the
  // allocate action (the live job; lists / batching inside a selected row set as usual).
  struct AllocOps {
    HostBackend &hb;
    int job;
    int active_alloc(int ps) { return ps_get(hb.seq, ps, 0); }
    void active_nodes(int ps, std::vector<int> &out) {
      const DevSnap &s = *hb.seq.s;
      for (int t = s.ps_task_begin[ps]; t < s.ps_task_begin[ps + 1]; t++)
        if (hb.seq.rp.t_status[t] & kActiveAllocated) out.push_back(hb.seq.rp.t_node[t]);
    }
    bool podset_less(int a, int b) { return kai::podset_less(hb.seq, a, b); }
    int checkpoint() { return hb.seq.n_ops; }
    void rollback(int cp) { stmt_rollback(hb.seq, cp); }
    bool place(const std::vector<int> &tasks, unsigned int xbits) {
      double tt0 = now();
      node_state_disturbed(hb.seq);  // another row set: the min/max trackers and any list belong to the previous one
      hb.list_invalidate();
      hb.sweep_xbits = xbits;
      bool ok = hb.place_tasks(job, (int)tasks.size(), tasks.data());
      hb.sweep_xbits = 0;
      hb.t_topo[2] += now() - tt0;
      hb.n_topo_domains++;
      return ok && !hb.failed;
    }
    bool extra_in_set(int) { return true; }
    bool all_nodes() { return true; }
  };
  bool allocate_constrained(TopologyHost &topo, int job, const std::vector<int> &tta) {
    double tt0 = now();
    AllocOps ops{*this, job};
    TopoAllocator<AllocOps> ta(topo, seq, ops, job);
    list_invalidate();
    n_topo_jobs++;
    bool placed = ta.alloc_set(topo.job_root_set[job], tta);
    if (ta.unsupported) seq.error = 2;
    list_invalidate();
    node_state_disturbed(seq);
    t_topo[0] += now() - tt0;
    return placed;
  }

  void flush_deltas() {
    n_flush++;
    publish(DK_FLUSH);
    if (launch_mode) {  // stream order: the next launch sees these deltas applied; nothing to wait for
      ctl.seq++;
      ctl.n_delta = 0;
      return;
    }
    const unsigned int seq_no = ctl.seq;
    const unsigned long long *buf = h_slots + (size_t)(seq_no & 1) * kMaxGrid * kSlotWords;
    const unsigned int tag = seq_no & 0xffffffu;
    for (int c = 0; c < n_scanners; c++) {
      unsigned long long hi;
      if (!wait_word(buf + (size_t)c * kSlotWords + 1, [&](unsigned long long v) { return (unsigned int)(v >> 40) == tag; }, hi)) break;
    }
    ctl.seq = seq_no + 1;
    ctl.n_delta = 0;
  }

  // actions/allocate/allocate.go:46-111 — same steps as sequencer_main of the device-resident mode
  void run_allocate() {
    const DevSnap &s = *seq.s;
    double t_begin = now();
    t_exchange = 0;
    unsigned long long tk = prof ? __builtin_ia32_rdtsc() : 0;
    auto lap = [&](int i) {
      if (!prof) return;
      unsigned long long t = __builtin_ia32_rdtsc();
      t_sec[i] += t - tk;
      tk = t;
    };
    korder.reason = "KAI_JOB_ORDER=replica";
    korder.reason_queue = -1;
    const bool keyed = keyed_order_allowed && korder.check(seq);
    keyed_order_used = keyed;
    lap(5);
    if (keyed)
      korder.build(seq);
    else
      seq_init_job_order(seq);
    lap(6);
    seq.pop_split = prof && !keyed ? t_pop_split : nullptr;
    for (;;) {
      lap(4);
      int job = keyed ? korder.pop(seq) : pop_next_job(seq);
      lap(0);
      if (job < 0 || failed) break;
      seq.n_ops = 0;
      const JobRec rec = s.jrec[job];
      ctl.job = job;
      ctl.ctx_job = job;
      ctl.ctx_queue = s.j_queue[job];
      ctl.ctx_preempt = (s.j_flags[job] & KAI_JOB_PREEMPTIBLE) ? 1 : 0;
      ctl.ctx_fresh = (!job_touched(seq, job) && rec.n_tta >= 0) ? 1 : 0;
      ctl.ctx_ps = -1;
      if (rec.n_podsets == 1) {
        if (!job_touched(seq, job)) {
          for (int w = 0; w < 3; w++) ctl.ctx_cnt[w] = rec.cnt[w];
        } else {
          for (int w = 0; w < 3; w++) ctl.ctx_cnt[w] = seq.rp.ps_active_alloc[(size_t)w * s.S + rec.ps0];
        }
        ctl.ctx_ps = rec.ps0;
      }
      int n;
      double req[QR] = {0, 0, 0};
      if (ctl.ctx_fresh) {
        n = rec.n_tta;
        ctl.ctx_base = rec.tb;
        for (int r = 0; r < QR; r++) req[r] = rec.req0[r];
      } else {
        n = tasks_to_allocate(seq, job, true, nullptr);
        ctl.ctx_base = -1;
        for (int k = 0; k < n; k++)
          for (int r = 0; r < QR; r++) req[r] = kadd(req[r], s.t_req[(size_t)seq.rp.tta[k] * s.R + r]);
      }
      bool job_success = !over_capacity(seq, job, req);
      lap(1);
      TopologyHost *topo = (TopologyHost *)seq.topology;
      if (job_success && topo && topo->constrained(job)) {
        std::vector<int> tta(n);
        for (int k = 0; k < n; k++) tta[k] = ctl.ctx_base >= 0 ? ctl.ctx_base + k : seq.rp.tta[k];
        job_success = allocate_constrained(*topo, job, tta);
      } else if (job_success) {
        if (topo) topo->scores_off(seq);  // no NodeOrderFn term from the previous job's topology scores
        if (gang_fast && ctl.ctx_fresh && rec.pad[0] && n == rec.n_tta)
          job_success = place_fresh_gang(job, n, rec.tb);
        else
          job_success = place_tasks(job, n);
      }
      lap(2);
      if (job_success) {
        if (should_pipeline_job(seq, job)) stmt_convert_all_allocated_to_pipelined(seq, job);
        stmt_commit(seq);
        record_visit(seq, job, 1);
        if (has_tasks_to_allocate(seq, job)) {
          if (keyed)
            seq.error = 3;  // KeyedJobOrder::check rules this out; the keyed heaps cannot take the job back
          else
            push_job(seq, job);
        }
      } else {
        stmt_rollback(seq, 0);
        record_visit(seq, job, 0);
      }
      if (ctl.ctx_ps >= 0)
        for (int w = 0; w < 3; w++) seq.rp.ps_active_alloc[(size_t)w * s.S + ctl.ctx_ps] = ctl.ctx_cnt[w];
      ctl.ctx_ps = -1;
      ctl.ctx_job = -1;
      ctl.ctx_fresh = 0;
      lap(3);
      if (seq.error || failed) break;
    }
    seq.pop_split = nullptr;
    publish(DK_DONE);  // carries the last node deltas; the scanners write their tiles back and exit
    t_total = now() - t_begin;
  }
};

inline void host_flush_deltas(Seq &q) { ((HostBackend *)q.host_backend)->flush_deltas(); }

}  // namespace kai
