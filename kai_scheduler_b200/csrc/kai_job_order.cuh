// kai_job_order.cuh — keyed job order of the allocate action (host-sequenced mode).
//
// The replica job-order tree (kai_seq.cuh: pop_next_job) copies container/heap move for move: a node's DRF key is
// recomputed lazily through best_job / job_init_resource, and every heap compare goes through items[j] -> qkey.  That
// matters only when the queue comparator can tie, or when a department's key depends on which child sits at the top
// of its (possibly stale) child heap.  When a snapshot rules both out, any exact priority queue over the same keys pops
// the same job sequence, and this one does it with the keys stored inline in the heaps.
//
// Why the order is the same.  Within one allocate action a queue's key changes only when its own Allocated changes or
// its best pending job changes; both happen only on the chain of the job just popped, whose nodes are all at the top of
// their heaps.  The replica fixes each of them with heap.Fix(0) before it reads it; every other entry keeps the key it
// was sifted with.  So if the comparator is a strict total order, every replica heap top is the unique minimum of its
// entries.  check() proves, per action:
//   P1  no ties: in every sibling group of queues that enter the tree, creation stamps are pairwise distinct and no
//       queue's allocatable share strictly dominates another's (queue_order.go:221-233 then always falls through), so
//       node_less is lexicographic on (w0, drf with the job, drf, creation);
//   P2  a department's key does not depend on its heap top: every pending job below a linked queue has a bit-identical
//       GetTasksToAllocateInitResource, and no job is pushed back during the action (the first GetTasksToAllocate set
//       of every pending job is all of its pending tasks: one podset, untouched, n_tta == pending).
// Keys are recomputed for the popped chain only, with the f64 operations of queue_key in the same order, from one
// packed record of per-queue constants and the queue's uniform request; best_job and the job records are not read.
#pragma once
#include <cstring>
#include <vector>

#include "kai_seq.cuh"

namespace kai {

struct KeyedJobOrder {
  struct Entry {  // one heap entry: the comparator inputs of queue_order.go:19-73 stored inline
    unsigned long long w0;
    double drf_job, drf;
    long long creation;
    int queue;
  };
  struct QConst {  // per-queue constants of a key
    double fair[QR], deserved[QR], la[QR], denom[QR], req[QR];
    unsigned long long w0_prio;  // inverted priority bits of QKey::w0
    long long creation;
    int parent;
    int heap;  // first entry of this queue's child heap in `arena` (internal nodes)
    int len;   // entries in this queue's child heap
    int leaf;
  };
  std::vector<QConst> qc;
  std::vector<Entry> arena;  // child heaps by q_child_begin, then the root heap
  int root_base = 0, root_len = 0;
  int chain[64];  // queues whose keys changed with the last pop (leaf first)
  int n_chain = 0;
  // what the last check() found
  const char *reason = "";
  int reason_queue = -1;
  // scratch of check()
  std::vector<unsigned char> linked;
  std::vector<int> group;

  static bool less(const Entry &a, const Entry &b) {  // node_less when P1 holds
    if (a.w0 != b.w0) return a.w0 < b.w0;
    if (a.drf_job < b.drf_job) return true;
    if (a.drf_job > b.drf_job) return false;
    if (a.drf < b.drf) return true;
    if (a.drf > b.drf) return false;
    return a.creation < b.creation;
  }
  static void sift_down(Entry *h, int n, int i) {
    const Entry x = h[i];
    for (;;) {
      const int j1 = 2 * i + 1;
      if (j1 >= n) break;
      const int j = j1 + (int)(j1 + 1 < n && less(h[j1 + 1], h[j1]));
      if (!less(h[j], x)) break;
      h[i] = h[j];
      i = j;
    }
    h[i] = x;
  }
  static void sift_up(Entry *h, int j) {
    const Entry x = h[j];
    while (j > 0) {
      const int i = (j - 1) / 2;
      if (!less(x, h[i])) break;
      h[j] = h[i];
      j = i;
    }
    h[j] = x;
  }
  Entry *heap_of(int parent, int *&len) {
    if (parent < 0) {
      len = &root_len;
      return arena.data() + root_base;
    }
    len = &qc[parent].len;
    return arena.data() + qc[parent].heap;
  }

  // queue_key (kai_seq.cuh) on the packed constants and the queue's uniform request
  void key(const Seq &q, int qi, Entry &e) const {
    const QConst &c = qc[qi];
    const double *alloc_r = q.rp.q_alloc + qi;
    const size_t Q = (size_t)q.s->Q;
    bool over = true, starved = true, viol = false;
    double dj = 0.0, dr = 0.0;
    for (int r = 0; r < QR; r++) {
      const double alloc = alloc_r[r * Q];
      const double with_job = kadd(alloc, c.req[r]);
      if (c.fair[r] >= alloc) over = false;
      if (compare_quantities(with_job, c.deserved[r]) > 0) starved = false;
      if (c.la[r] == 0 && with_job > 0) viol = true;
      const double denom = c.denom[r];
      const double vj = denom == 0 ? kmul(with_job, 1000.0) : kdiv(with_job, denom);
      const double vr = denom == 0 ? kmul(alloc, 1000.0) : kdiv(alloc, denom);
      dj = fmax(dj, vj);
      dr = fmax(dr, vr);
    }
    e.w0 = ((unsigned long long)(over ? 1 : 0) << 44) | ((unsigned long long)(starved ? 0 : 1) << 43) | c.w0_prio |
           ((unsigned long long)(viol ? 1 : 0) << 9);
    e.drf_job = dj;
    e.drf = dr;
    e.creation = c.creation;
    e.queue = qi;
  }

  bool fail(const char *why, int queue) {
    reason = why;
    reason_queue = queue;
    return false;
  }
  // P1 / P2 over the queues that enter the tree and their pending jobs, at action start (before any pop).
  // O(Q + J + sum of sibling-group sizes squared).  Fills the per-queue constants on success.
  bool check(const Seq &q) {
    const DevSnap &s = *q.s;
    const int Q = s.Q;
    reason = "";
    reason_queue = -1;
    qc.resize(Q);
    linked.assign(Q, 0);
    // P2: one request per linked queue, pushed up from the leaves
    for (int qi = 0; qi < Q; qi++) {
      if (s.q_nchildren[qi] != 0) continue;
      const int h = q.rp.leaf_head[qi], e = q.rp.leaf_end[qi];
      if (h == e && q.rp.ovl_len[qi] == 0) continue;
      if (q.rp.ovl_len[qi] != 0) return fail("a leaf queue holds re-pushed jobs", qi);
      const JobRec &r0 = s.jrec[q.rp.leaf_heap[h]];
      for (int k = h; k < e; k++) {
        const int j = q.rp.leaf_heap[k];
        const JobRec &rec = s.jrec[j];
        if (job_touched(q, j) || rec.n_podsets != 1 || rec.n_tta < 0)
          return fail("a pending job's first GetTasksToAllocate set is not a prefix of one untouched podset", qi);
        if (rec.n_tta != rec.cnt[1]) return fail("a pending job would be pushed back (elastic: n_tta below its pending tasks)", qi);
        if (memcmp(rec.req0, r0.req0, sizeof(rec.req0)) != 0) return fail("mixed init requests among the pending jobs of a queue", qi);
      }
      int depth = 0;
      for (int c = qi; c >= 0; c = s.q_parent[c]) {
        if (++depth > (int)(sizeof(chain) / sizeof(chain[0]))) return fail("queue tree deeper than the keyed order tracks", qi);
        if (!linked[c]) {
          linked[c] = 1;
          memcpy(qc[c].req, r0.req0, sizeof(r0.req0));
        } else if (memcmp(qc[c].req, r0.req0, sizeof(r0.req0)) != 0) {
          return fail("mixed init requests among the pending jobs below a department", c);
        }
      }
    }
    // P1: every sibling group (children of a linked queue, and the linked top queues)
    auto group_ok = [&](int parent) {
      for (size_t a = 0; a < group.size(); a++)
        for (size_t b = a + 1; b < group.size(); b++) {
          const int l = group[a], r = group[b];
          if (s.q_creation[l] == s.q_creation[r]) return fail("equal creation stamps among sibling queues", parent >= 0 ? parent : l);
          bool l_le_r = true, r_le_l = true;
          for (int i = 0; i < QR; i++) {
            const double la = s.q_allocatable[(size_t)i * Q + l], ra = s.q_allocatable[(size_t)i * Q + r];
            if (compare_quantities(la, ra) > 0) l_le_r = false;
            if (compare_quantities(ra, la) > 0) r_le_l = false;
          }
          if (l_le_r != r_le_l) return fail("a sibling queue's allocatable share strictly dominates another's", parent >= 0 ? parent : l);
        }
      return true;
    };
    group.clear();
    for (int i = 0; i < s.n_top; i++)
      if (linked[s.top_queues[i]]) group.push_back(s.top_queues[i]);
    if (!group_ok(-1)) return false;
    for (int p = 0; p < Q; p++) {
      if (!linked[p] || s.q_nchildren[p] == 0) continue;
      group.clear();
      const int cb = s.q_child_begin[p];
      for (int k = 0; k < s.q_nchildren[p]; k++)
        if (linked[s.q_children[cb + k]]) group.push_back(s.q_children[cb + k]);
      if (!group_ok(p)) return false;
    }
    return true;
  }

  // heaps of the linked queues with their keys at action start (replaces seq_init_job_order)
  void build(const Seq &q) {
    const DevSnap &s = *q.s;
    const int Q = s.Q;
    root_base = Q;
    root_len = 0;
    arena.resize((size_t)Q + s.n_top + 1);
    n_chain = 0;
    for (int qi = 0; qi < Q; qi++) {
      QConst &c = qc[qi];
      c.parent = s.q_parent[qi];
      c.leaf = s.q_nchildren[qi] == 0;
      c.heap = c.leaf ? 0 : s.q_child_begin[qi];
      c.len = 0;
      c.creation = s.q_creation[qi];
      c.w0_prio = ((unsigned long long)(0x80000000LL - (long long)s.q_priority[qi]) & 0x1ffffffffull) << 10;
      for (int r = 0; r < QR; r++) {
        const size_t o = (size_t)r * Q + qi;
        c.fair[r] = s.q_fair[o];
        c.deserved[r] = s.q_deserved[o];
        c.la[r] = s.q_allocatable[o];
        c.denom[r] = c.la[r] == KAI_UNLIMITED ? s.total[r] : c.la[r];
      }
    }
    for (int qi = 0; qi < Q; qi++) {
      if (!linked[qi]) continue;
      int *len;
      Entry *h = heap_of(qc[qi].parent, len);
      key(q, qi, h[*len]);
      sift_up(h, (*len)++);
    }
  }

  int pop(Seq &q) {
    // keys of the last popped chain: each of its queues is still the top of its parent's heap
    for (int i = 0; i < n_chain; i++) {
      const int c = chain[i];
      int *len;
      Entry *h = heap_of(qc[c].parent, len);
      key(q, c, h[0]);
      sift_down(h, *len, 0);
    }
    n_chain = 0;
    if (root_len == 0) return -1;
    int c = arena[root_base].queue;
    while (!qc[c].leaf) c = arena[qc[c].heap].queue;
    const int head = q.rp.leaf_head[c];
    const int job = q.rp.leaf_heap[head];
    q.rp.leaf_head[c] = head + 1;
    // handle_pop: queues that ran empty leave their parent's heap; the rest of the chain gets new keys at the next pop
    for (;;) {
      const QConst &x = qc[c];
      const bool empty = x.leaf ? q.rp.leaf_head[c] == q.rp.leaf_end[c] : x.len == 0;
      if (!empty) break;
      int *len;
      Entry *h = heap_of(x.parent, len);
      h[0] = h[--*len];
      sift_down(h, *len, 0);
      if (x.parent < 0) return job;
      c = x.parent;
    }
    for (; c >= 0; c = qc[c].parent) chain[n_chain++] = c;
    return job;
  }
};

}  // namespace kai
