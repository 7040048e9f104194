// Host-only check of the keyed job order of the allocate action (kai_job_order.cuh) against the replica job-order tree
// (kai_seq.cuh: seq_init_job_order / pop_next_job / push-free handle_pop):
//   (1) on seeded two- and three-level queue trees (up to 1 000 leaves, uniform gangs per department, random
//       priorities, fair shares, quotas and initial allocations), with queue_allocate of every popped job simulated
//       (commits, and discards that add and remove again), both orders pop the identical job sequence;
//   (2) the eligibility check rejects equal creation stamps among siblings, a strictly dominating allocatable share,
//       mixed requests within one department and an elastic job (fewer tasks to allocate than pending tasks).
// Built and run by tests/test_job_order_keyed.py (nvcc, no GPU needed: nothing is launched).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../kai_scheduler_b200/csrc/kai_host_seq.cuh"

using namespace kai;

static unsigned long long rng_state = 0x0C43ULL;
static unsigned int rnd() {
  rng_state = rng_state * 6364136223846793005ULL + 1442695040888963407ULL;
  return (unsigned int)(rng_state >> 33);
}
static unsigned int rnd(unsigned int n) { return rnd() % n; }

#define CHECK(cond, ...)                           \
  do {                                             \
    if (!(cond)) {                                 \
      printf("FAIL %s:%d ", __FILE__, __LINE__);   \
      printf(__VA_ARGS__);                         \
      printf("\n");                                \
      return 1;                                    \
    }                                              \
  } while (0)

// One synthetic cluster: the snapshot tables the job-order tree reads, and the replica state it starts from.
struct Cluster {
  int Q = 0, J = 0, T = 0, R = 4, n_top = 0;
  std::vector<int> parent, nchildren, child_begin, children, top, priority, job_begin, leaf_count;
  std::vector<long long> creation;
  std::vector<double> fair, deserved, allocatable, alloc0, total;  // [QR][Q], total [QR]
  std::vector<int> j_queue, leaf_sorted, t_job;
  std::vector<uint32_t> j_flags;
  std::vector<unsigned long long> j_key;
  std::vector<JobRec> jrec;
  std::vector<double> t_req;  // [T][R]
  std::vector<std::vector<int>> kids;
  DevSnap s;

  int add_queue(int p) {
    parent.push_back(p);
    kids.emplace_back();
    if (p >= 0) kids[p].push_back(Q);
    return Q++;
  }
  // levels = 2: departments -> leaves; levels = 3: departments -> sub-departments -> leaves
  void make(int levels, int n_leaves, bool uniform_params) {
    const int n_dept = 1 + (int)rnd(levels == 2 ? 60 : 12);
    std::vector<int> mids;
    for (int d = 0; d < n_dept; d++) mids.push_back(add_queue(-1));
    if (levels == 3) {
      std::vector<int> depts = mids;
      mids.clear();
      for (int d : depts)
        for (int k = 0, n = 1 + (int)rnd(6); k < n; k++) mids.push_back(add_queue(d));
    }
    for (int l = 0; l < n_leaves; l++) add_queue(mids[rnd((unsigned int)mids.size())]);
    if (rnd(3) == 0) add_queue(-1);  // a top-level leaf queue
    // a childless department has no jobs (only leaves hold jobs) and never enters the tree; that is fine
    nchildren.assign(Q, 0);
    child_begin.assign(Q + 1, 0);
    for (int q = 0; q < Q; q++) {
      nchildren[q] = (int)kids[q].size();
      child_begin[q + 1] = child_begin[q] + nchildren[q];
      for (int c : kids[q]) children.push_back(c);
      if (parent[q] < 0) top.push_back(q);
    }
    n_top = (int)top.size();
    // creation stamps: distinct within every sibling group (a permutation of the group, times 60)
    creation.assign(Q, 0);
    auto stamp = [&](const std::vector<int> &g) {
      std::vector<int> perm(g.size());
      for (size_t i = 0; i < g.size(); i++) perm[i] = (int)i;
      for (size_t i = g.size(); i > 1; i--) std::swap(perm[i - 1], perm[rnd((unsigned int)i)]);
      for (size_t i = 0; i < g.size(); i++) creation[g[i]] = (long long)perm[i] * 60;
    };
    stamp(top);
    for (int q = 0; q < Q; q++) stamp(kids[q]);
    priority.assign(Q, 100);
    fair.assign((size_t)QR * Q, 0);
    deserved.assign((size_t)QR * Q, 0);
    allocatable.assign((size_t)QR * Q, 0);
    alloc0.assign((size_t)QR * Q, 0);
    total = {2e7 * 1000, 2e10 * 1000, 8000};
    for (int q = 0; q < Q; q++) {
      if (!uniform_params && rnd(4) == 0) priority[q] = 100 + (int)rnd(3) * 50;
      // allocatable: the same GPU share for everyone; CPU / memory trade off against each other, so siblings are
      // equal or incomparable, never strictly dominated
      const int k = uniform_params ? 0 : (int)rnd(5);
      allocatable[0 * Q + q] = uniform_params ? KAI_UNLIMITED : 1e6 * (1 + k);
      allocatable[1 * Q + q] = uniform_params ? KAI_UNLIMITED : 1e12 * (5 - k);
      allocatable[2 * Q + q] = uniform_params ? 40.0 : (rnd(6) == 0 ? KAI_UNLIMITED : 10.0 + 10.0 * (rnd(4)));
      for (int r = 0; r < QR; r++) {
        fair[(size_t)r * Q + q] = uniform_params ? 20.0 * (r == 2) : (double)rnd(30) * (r == 2 ? 1.0 : 1e3);
        deserved[(size_t)r * Q + q] = uniform_params ? (r == 2 ? 20.0 : KAI_UNLIMITED) : (rnd(3) == 0 ? KAI_UNLIMITED : (double)rnd(25));
        alloc0[(size_t)r * Q + q] = uniform_params ? 0.0 : (double)rnd(8) * (r == 0 ? 1000.0 : r == 1 ? 1e9 : 1.0);
      }
    }
    if (!uniform_params) {  // a sibling group shares its GPU allocatable (CPU / memory then decide incomparability)
      auto share = [&](const std::vector<int> &g) {
        for (size_t i = 1; i < g.size(); i++) allocatable[2 * Q + g[i]] = allocatable[2 * Q + g[0]];
      };
      share(top);
      for (int q = 0; q < Q; q++) share(kids[q]);
    }
    // jobs: gangs with one request per department (top-level subtree)
    std::vector<int> dept_of(Q);
    for (int q = 0; q < Q; q++) {
      int d = q;
      while (parent[d] >= 0) d = parent[d];
      dept_of[q] = d;
    }
    std::vector<double> dreq((size_t)Q * R);
    std::vector<int> dgang(Q);
    for (int q = 0; q < Q; q++) {
      const double g = uniform_params ? 1.0 : (double)(1 << rnd(3));
      dreq[(size_t)q * R + 0] = 1000.0 * (1 + rnd(2));
      dreq[(size_t)q * R + 1] = 1e9;
      dreq[(size_t)q * R + 2] = g;
      dreq[(size_t)q * R + 3] = 1.0;
      dgang[q] = uniform_params ? 4 : 1 + (int)rnd(4);
    }
    job_begin.assign(Q + 1, 0);
    leaf_count.assign(Q, 0);
    for (int q = 0; q < Q; q++) {
      job_begin[q] = J;
      if (nchildren[q] != 0) continue;
      const int n = rnd(4) == 0 ? 0 : 1 + (int)rnd(uniform_params ? 60 : 12);
      const int d = dept_of[q];
      for (int i = 0; i < n; i++) {
        const int j = J++;
        j_queue.push_back(q);
        j_flags.push_back(rnd(3) == 0 ? 0u : (uint32_t)KAI_JOB_PREEMPTIBLE);
        j_key.push_back(make_job_key(50, 0, j));
        leaf_sorted.push_back(j);
        JobRec rec;
        memset(&rec, 0, sizeof(rec));
        rec.n_podsets = 1;
        rec.ps0 = j;
        rec.tb = T;
        rec.n_tta = dgang[d];
        rec.cnt[1] = dgang[d];
        for (int k = 0; k < dgang[d]; k++) {
          t_job.push_back(j);
          for (int r = 0; r < R; r++) t_req.push_back(dreq[(size_t)d * R + r]);
          for (int r = 0; r < QR; r++) rec.req0[r] = kadd(rec.req0[r], dreq[(size_t)d * R + r]);
          T++;
        }
        rec.pad[0] = 1;
        jrec.push_back(rec);
      }
      leaf_count[q] = n;
    }
    job_begin[Q] = J;
  }
  void snap() {
    memset(&s, 0, sizeof(s));
    s.R = R;
    s.Q = Q;
    s.J = J;
    s.T = T;
    s.S = J;
    s.n_top = n_top;
    s.q_parent = parent.data();
    s.q_priority = priority.data();
    s.q_nchildren = nchildren.data();
    s.q_creation = creation.data();
    s.q_deserved = deserved.data();
    s.q_fair = fair.data();
    s.q_allocatable = allocatable.data();
    s.q_child_begin = child_begin.data();
    s.q_children = children.data();
    s.top_queues = top.data();
    s.q_job_begin = job_begin.data();
    s.j_queue = j_queue.data();
    s.j_flags = j_flags.data();
    s.t_req = t_req.data();
    s.t_job = t_job.data();
    s.total = total.data();
    s.jrec = jrec.data();
  }
};

// The replica state of one action, as kai_engine.cu sets it up for the host sequencer.
struct State {
  std::vector<double> q_alloc, q_alloc_np;
  std::vector<QKey> qkey;
  std::vector<int> leaf_head, leaf_end, ovl_len, child_len, child_heap, root_heap, leaf_heap, j_req_valid_i;
  std::vector<unsigned char> qn_flags, j_req_valid;
  std::vector<unsigned int> touched;
  std::vector<double> j_req;
  std::vector<unsigned long long> j_key;
  Ctl ctl;
  Seq q;
  void init(Cluster &c) {
    const int Q = c.Q, J = c.J;
    q_alloc = c.alloc0;
    q_alloc_np = c.alloc0;
    qkey.assign(Q, QKey{});
    leaf_head.assign(Q, 0);
    leaf_end.assign(Q, 0);
    for (int i = 0; i < Q; i++) {
      leaf_head[i] = c.job_begin[i];
      leaf_end[i] = c.job_begin[i] + (c.nchildren[i] == 0 ? c.leaf_count[i] : 0);
    }
    ovl_len.assign(Q, 0);
    child_len.assign(Q, 0);
    child_heap.assign(Q + 1, 0);
    root_heap.assign(c.n_top + 1, 0);
    leaf_heap = c.leaf_sorted;
    qn_flags.assign(Q, 0);
    touched.assign((J + 31) / 32 + 1, 0);
    j_req.assign((size_t)J * QR + 1, 0);
    j_req_valid.assign(J + 1, 0);
    j_key = c.j_key;
    memset(&ctl, 0, sizeof(ctl));
    memset(&q, 0, sizeof(q));
    ctl.ctx_job = ctl.ctx_ps = -1;
    ctl.dec.task = -1;
    Replica &rp = q.rp;
    rp.q_alloc = q_alloc.data();
    rp.q_alloc_np = q_alloc_np.data();
    rp.qkey = qkey.data();
    rp.leaf_head = leaf_head.data();
    rp.leaf_end = leaf_end.data();
    rp.ovl_len = ovl_len.data();
    rp.child_len = child_len.data();
    rp.child_heap = child_heap.data();
    rp.root_heap = root_heap.data();
    rp.qn_flags = qn_flags.data();
    rp.touched = touched.data();
    rp.j_req = j_req.data();
    rp.j_req_valid = j_req_valid.data();
    rp.j_key = j_key.data();
    rp.leaf_heap = leaf_heap.data();
    q.s = &c.s;
    q.ctl = &ctl;
  }
};

// what run_allocate does to the queue shares of a popped job: commit (all tasks added) or discard (a prefix added and
// removed again, which need not restore the f64 sums bit for bit)
static void simulate(Cluster &c, Seq &q, int job) {
  const JobRec &rec = c.jrec[job];
  const unsigned int h = (unsigned int)job * 2654435761u;
  const bool commit = (h >> 7) % 5 != 0;
  const int n = commit ? rec.n_tta : (int)((h >> 11) % (rec.n_tta + 1));
  for (int k = 0; k < n; k++) queue_allocate(q, rec.tb + k, true, job);
  if (!commit)
    for (int k = n - 1; k >= 0; k--) queue_allocate(q, rec.tb + k, false, job);
  q.rp.touched[job >> 5] |= 1u << (job & 31);
  invalidate_chain(q, c.j_queue[job]);
}

static std::vector<int> run_replica(Cluster &c) {
  State st;
  st.init(c);
  seq_init_job_order(st.q);
  std::vector<int> seqn;
  for (int job; (job = pop_next_job(st.q)) >= 0;) {
    seqn.push_back(job);
    simulate(c, st.q, job);
  }
  return seqn;
}
static bool run_keyed(Cluster &c, std::vector<int> &seqn, std::string &why) {
  State st;
  st.init(c);
  KeyedJobOrder ko;
  if (!ko.check(st.q)) {
    why = ko.reason;
    return false;
  }
  ko.build(st.q);
  for (int job; (job = ko.pop(st.q)) >= 0;) {
    seqn.push_back(job);
    simulate(c, st.q, job);
  }
  return true;
}
static std::string rejection(Cluster &c) {
  State st;
  st.init(c);
  KeyedJobOrder ko;
  return ko.check(st.q) ? std::string() : std::string(ko.reason);
}

int main() {
  // ---------------------------------------------------------------- (1) identical pop sequences
  long long pops = 0;
  int trees = 0;
  for (int trial = 0; trial < 120; trial++) {
    Cluster c;
    const int levels = 2 + (trial & 1);
    const int leaves = trial < 8 ? 1000 : 1 + (int)rnd(300);
    c.make(levels, leaves, (trial % 3) == 0);
    c.snap();
    const std::vector<int> want = run_replica(c);
    std::vector<int> got;
    std::string why;
    CHECK(run_keyed(c, got, why), "trial %d (%d levels, %d leaves): eligibility check refused: %s", trial, levels, leaves, why.c_str());
    CHECK(got.size() == want.size(), "trial %d: keyed order popped %zu jobs, replica %zu", trial, got.size(), want.size());
    for (size_t i = 0; i < want.size(); i++)
      CHECK(got[i] == want[i], "trial %d (%d levels, %d leaves): pop %zu is job %d, replica pops job %d", trial, levels, leaves, i,
            got[i], want[i]);
    CHECK((int)want.size() == c.J, "trial %d: %zu pops of %d jobs", trial, want.size(), c.J);
    pops += (long long)want.size();
    trees++;
  }

  // ---------------------------------------------------------------- (2) rejected snapshots
  auto linked_siblings = [](Cluster &c, int &a, int &b) {  // two top-level queues that both hold pending jobs below them
    std::vector<int> live(c.Q, 0);
    for (int q = 0; q < c.Q; q++)
      if (c.nchildren[q] == 0 && c.leaf_count[q] > 0)
        for (int x = q; x >= 0; x = c.parent[x]) live[x] = 1;
    a = b = -1;
    for (int q : c.top)
      if (live[q]) {
        if (a < 0)
          a = q;
        else if (b < 0)
          b = q;
      }
    return b >= 0;
  };
  int rejected = 0;
  for (int trial = 0; trial < 40; trial++) {
    Cluster c;
    c.make(2 + (trial & 1), 40 + (int)rnd(200), (trial % 3) == 0);
    c.snap();
    CHECK(rejection(c).empty(), "rejection trial %d: the unmodified cluster is refused: %s", trial, rejection(c).c_str());
    int a, b;
    if (!linked_siblings(c, a, b)) continue;
    {  // equal creation stamps
      const long long keep = c.creation[b];
      c.creation[b] = c.creation[a];
      const std::string why = rejection(c);
      CHECK(why.find("creation") != std::string::npos, "trial %d: equal creation stamps accepted (%s)", trial, why.c_str());
      c.creation[b] = keep;
    }
    {  // strictly dominating allocatable share
      const double keep = c.allocatable[(size_t)0 * c.Q + b];
      c.allocatable[(size_t)0 * c.Q + b] = KAI_UNLIMITED;  // unlimited CPU: b >= a everywhere, > in CPU
      const double keep1 = c.allocatable[(size_t)1 * c.Q + b];
      c.allocatable[(size_t)1 * c.Q + b] = KAI_UNLIMITED;
      const double keep2 = c.allocatable[(size_t)2 * c.Q + b];
      c.allocatable[(size_t)2 * c.Q + b] = c.allocatable[(size_t)2 * c.Q + a];
      const bool dominated = c.allocatable[(size_t)0 * c.Q + a] != KAI_UNLIMITED || c.allocatable[(size_t)1 * c.Q + a] != KAI_UNLIMITED;
      const std::string why = rejection(c);
      if (dominated) CHECK(why.find("dominates") != std::string::npos, "trial %d: strict dominance accepted (%s)", trial, why.c_str());
      c.allocatable[(size_t)0 * c.Q + b] = keep;
      c.allocatable[(size_t)1 * c.Q + b] = keep1;
      c.allocatable[(size_t)2 * c.Q + b] = keep2;
    }
    // a pending job below department a, and another pending job in the same department
    std::vector<int> below;
    for (int j = 0; j < c.J; j++) {
      int x = c.j_queue[j];
      while (c.parent[x] >= 0) x = c.parent[x];
      if (x == a) below.push_back(j);
    }
    if (below.size() >= 2) {  // mixed requests within one department
      const int j = below[below.size() - 1];
      const double keep = c.jrec[j].req0[1];
      c.jrec[j].req0[1] = kadd(keep, 1e9);
      const std::string why = rejection(c);
      CHECK(why.find("mixed") != std::string::npos, "trial %d: mixed requests accepted (%s)", trial, why.c_str());
      c.jrec[j].req0[1] = keep;
    }
    {  // elastic job: GetTasksToAllocate takes fewer tasks than the job has pending
      const int j = below[0];
      c.jrec[j].cnt[1] = c.jrec[j].n_tta + 2;
      const std::string why = rejection(c);
      CHECK(why.find("pushed back") != std::string::npos, "trial %d: elastic job accepted (%s)", trial, why.c_str());
      c.jrec[j].cnt[1] = c.jrec[j].n_tta;
    }
    CHECK(rejection(c).empty(), "rejection trial %d: the restored cluster is refused", trial);
    rejected++;
  }
  CHECK(rejected >= 20, "only %d rejection trials had two linked top-level queues", rejected);
  printf("OK keyed order equals the replica on %d trees (%lld pops); %d clusters x 4 crafted rejections\n", trees, pops, rejected);
  return 0;
}
