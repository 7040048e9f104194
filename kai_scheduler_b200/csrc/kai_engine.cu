// kai_engine.cu — host side of libkaigpu.so: the C ABI declared in include/kai_engine.h.
//
// Validates the caller's SoA snapshot, derives the index structures the kernels need (queue
// children CSR, jobs grouped by leaf queue in JobOrderFn order, tasks per podset in TaskOrderFn
// order, name-rank inverse), stages everything through one pinned buffer into HBM (or, for a resident
// snapshot, refreshes the per-cycle columns only), runs the open-session kernels, drives the sweep
// kernels of an action from the host sequencer (one k_record launch per decision record; or the
// persistent k_action kernel), and copies results back.
//
// There is NO CPU fallback: without a usable CUDA device kai_engine_create fails.
#include <algorithm>
#include <array>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <numeric>
#include <type_traits>
#include <string>
#include <vector>

#include "kai_device.cuh"
#include "kai_kernels.cuh"  // single translation unit: kernels + host API
#include "kai_action.cuh"
#include "kai_host_seq.cuh"
#include "kai_solver.cuh"

using namespace kai;

namespace {

// Simple device bump arena: one cudaMalloc per snapshot generation.
struct DeviceArena {
  unsigned char *base = nullptr;
  size_t cap = 0, off = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) {
      off = 0;
      return cudaSuccess;
    }
    if (base) cudaFree(base);
    base = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&base, bytes);
    if (e == cudaSuccess) cap = bytes;
    off = 0;
    return e;
  }
  template <class T>
  T *take(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
    T *p = (T *)(base + off);
    off += bytes;
    return p;
  }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = off = 0;
  }
};

struct Staging {  // pinned host staging buffer mirrored 1:1 onto a device arena region
  unsigned char *host = nullptr;
  size_t cap = 0, off = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) {
      off = 0;
      return cudaSuccess;
    }
    if (host) cudaFreeHost(host);
    host = nullptr;
    cap = 0;
    cudaError_t e = cudaMallocHost(&host, bytes);
    if (e == cudaSuccess) cap = bytes;
    off = 0;
    return e;
  }
  void release() {
    if (host) cudaFreeHost(host);
    host = nullptr;
    cap = off = 0;
  }
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) & ~(a - 1); }

constexpr int kShmRanks = 16;  // GPUs of one box that can share the exchange segment
// layout of the shared exchange segment (u64 words): answer lines | min/max lines | top-M lines | merged lists per rank
size_t shm_clist_offset_words() {
  return (size_t)2 * 2 * kMaxGrid * kSlotWords + (size_t)2 * kListScanners * kListLines * kListLineWords;
}

}  // namespace

struct kai_engine {
  kai_config cfg;
  std::string err;
  int device = 0;
  int num_sms = 0;
  int max_smem_optin = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_mirror = nullptr;
  bool loaded = false;

  DeviceArena dsnap;     // snapshot + session state
  Staging stage;         // pinned mirror of the uploaded part of dsnap
  DeviceArena dreplica;  // replica arenas
  DeviceArena dmisc;     // exchange buffers, counters, visits, fair-share scratch
  DevSnap ds;
  int R = 4, N = 0, Q = 0, J = 0, S = 0, T = 0;
  int grid = 0, npc = 0;
  size_t smem_bytes = 0, replica_bytes = 0, tile_bytes = 0, hot_bytes = 0;
  bool hot_in_smem = false;
  int ops_cap = 0, visits_cap = 0;
  unsigned long long *xbuf = nullptr, *mmbuf = nullptr, *dbuf = nullptr;
  unsigned long long *delta = nullptr;
  // host-sequenced mode
  unsigned long long *h_pinned = nullptr;  // one pinned mapped allocation: rec | delta | slots | mm
  unsigned long long *h_rec = nullptr, *h_delta = nullptr, *h_slots = nullptr, *h_mm = nullptr, *h_list = nullptr;
  HostBackend hb;
  // launch transport (default): one k_record launch per decision record, node tiles resident in global memory
  DeviceArena dlaunch;
  int lgrid = 0, lnpc = 0;  // scanners (= CTAs of k_record) and rows per scanner
  size_t ltile_stride = 0, ltile_bytes = 0, lsmem_bytes = 0;
  unsigned char *g_tiles = nullptr, *g_scan_state = nullptr;
  unsigned long long *d_list = nullptr;
  unsigned int *ticket = nullptr;
  double *mm_result = nullptr;
  unsigned long long *h_clist = nullptr;  // pinned mapped: [2][kCListWords]
  ActionParams lp;                        // parameters of the running action (launch transport)
  long long record_launches = 0;
  bool merge_cluster = true;  // k_merge_cluster (4-CTA cluster) instead of the one-CTA k_merge (KAI_MERGE=single)
  // multi-GPU (one engine per process per GPU): the reduced answer lines of all GPUs live in one POSIX shm
  // segment that every process maps and registers with CUDA; each host sequencer reads all lines.
  unsigned long long *shm_base = nullptr;  // [slots | mm], each [2][kMaxGrid][kSlotWords]
  size_t shm_bytes = 0;
  char shm_name[48] = {0};
  bool shm_owner = false, shm_registered = false;
  unsigned long long *shm_dev = nullptr;  // device-side address of the registered segment
  DevSnap hs;  // DevSnap whose pointers address the host mirror (the pinned staging buffer)
  std::vector<unsigned char> hot_host;
  std::vector<int> rank_to_node_h;
  // solver actions: second NodeInfo.PodInfos entry of a task (evicted from A, pipelined to B), mirror of the GPU column
  std::vector<int> on_other_node, on_other_status;
  std::vector<std::array<int, 3>> on_extra;  // (task, node, status) node entries beyond two per task (kai_solver.cuh)
  std::vector<double> h_mirror;  // host mirror of Idle / Releasing, node-major [N][2][R]
  std::vector<double> h_tmp;     // staging for the re-read after a device-sequenced action
  int *d_node_domain = nullptr;
  TopologyHost topo;
  int n_dom_levels = 0;
  bool mirror_valid = false;  // h_ig / h_lg followed every delta since the load (host-sequenced actions only)
  std::vector<int> job_signature;
  std::vector<double> q_preempt_mrt, q_reclaim_mrt, j_last_start;  // plugins/minruntime inputs (host only)
  std::vector<double> j_stale_since;                               // stalegangeviction input (host only)
  double now_s = 0;
  size_t dev_only_begin = 0, dev_only_bytes = 0;
  // resident snapshot (kai_snapshot::structure_epoch): where the per-cycle columns live in the arena
  unsigned long long structure_epoch = 0;
  int shape[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // R, N, Q, J, S, T, pred classes, optional-array presence bits
  size_t off_idle = 0, off_rel = 0, off_nflags = 0, off_usage = 0, off_tst = 0, off_tnode = 0, off_tnst = 0;
  std::vector<int> task_perm;
  std::vector<int32_t> r_tmp_node, r_tmp_status;
  long long *counters = nullptr;
  kai_job_visit *d_visits = nullptr;
  double *fs_w = nullptr, *fs_rr = nullptr;
  unsigned int seq = 2;

  // host result buffers (pinned)
  Staging rstage;
  std::vector<int32_t> r_task_node, r_task_status;
  std::vector<kai_job_visit> r_visits;
  std::vector<double> r_fair, r_alloc, r_alloc_np, r_request, r_idle, r_rel;
  double r_total[3] = {0, 0, 0};
  kai_stats stats;

  int fail(int code, const std::string &m) {
    err = m;
    return code;
  }
  int cuda_fail(cudaError_t e, const char *what) {
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return KAI_ERR_CUDA;
  }
};

#define CK(call)                                   \
  do {                                             \
    cudaError_t _e = (call);                       \
    if (_e != cudaSuccess) return e->cuda_fail(_e, #call); \
  } while (0)

static int load_tail(kai_engine *e, const kai_snapshot *s, int n_dom_levels, bool resident) {
  const int N = e->N, T = e->T, Q = e->Q;
  const DevSnap &ds = e->ds;
  const size_t RN = (size_t)e->R * N, QN = (size_t)QR * Q;
  (void)RN;
  // ---------------- open session: totals, queue usage, fair share ----------------
  if (N > 0) {
    int blocks = std::min(e->num_sms * 4, (N + 255) / 256);
    k_node_totals<<<blocks, 256, 0, e->stream>>>(ds);
  }
  if (T > 0) {
    int blocks = std::min(e->num_sms * 8, (T + 255) / 256);
    k_queue_usage<<<blocks, 256, 0, e->stream>>>(ds);
  }
  if (Q > 0) k_fair_share<<<1, 1024, 0, e->stream>>>(ds, e->cfg.k_value, e->fs_w, e->fs_rr);
  cudaEventRecord(e->ev[2], e->stream);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]);
  e->stats.upload_ms = ms;
  cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]);
  e->stats.open_session_ms = ms;
  e->stats.kernel_launches = (N > 0) + (T > 0) + (Q > 0);
  e->stats.action_ms = 0;
  e->stats.download_ms = 0;
  e->stats.decisions = e->stats.nodes_scanned = e->stats.algorithmic_bytes = 0;

  // result buffers
  e->r_task_node.assign(T, -1);
  e->r_task_status.assign(T, 0);
  e->r_fair.assign(QN, 0);
  e->r_alloc.assign(QN, 0);
  e->r_alloc_np.assign(QN, 0);
  e->r_request.assign(QN, 0);
  e->r_idle.assign(RN, 0);
  e->r_rel.assign(RN, 0);
  e->r_visits.clear();
  e->on_other_node.clear();
  e->on_other_status.clear();
  e->on_extra.clear();
  e->job_signature.clear();
  e->h_mirror.resize((size_t)2 * s->n_res * s->n_nodes);
  for (int n = 0; n < s->n_nodes; n++)
    for (int r = 0; r < s->n_res; r++) {
      e->h_mirror[(size_t)n * 2 * s->n_res + r] = s->node_idle[(size_t)r * s->n_nodes + n];
      e->h_mirror[(size_t)n * 2 * s->n_res + s->n_res + r] = s->node_releasing[(size_t)r * s->n_nodes + n];
    }
  if (e->d_node_domain && !resident) {
    cudaFree(e->d_node_domain);
    e->d_node_domain = nullptr;
  }
  e->n_dom_levels = n_dom_levels;
  e->topo.build(s);
  if (n_dom_levels > 0 && s->n_nodes > 0 && !resident) {
    CK(cudaMalloc(&e->d_node_domain, sizeof(int) * (size_t)n_dom_levels * s->n_nodes));
    CK(cudaMemcpy(e->d_node_domain, s->node_domain, sizeof(int) * (size_t)n_dom_levels * s->n_nodes, cudaMemcpyHostToDevice));
  }
  e->mirror_valid = true;
  if (s->job_signature) e->job_signature.assign(s->job_signature, s->job_signature + s->n_jobs);
  e->q_preempt_mrt.clear();
  e->q_reclaim_mrt.clear();
  e->j_last_start.clear();
  e->j_stale_since.clear();
  e->now_s = s->now_s;
  if (s->queue_preempt_min_runtime_s) e->q_preempt_mrt.assign(s->queue_preempt_min_runtime_s, s->queue_preempt_min_runtime_s + s->n_queues);
  if (s->queue_reclaim_min_runtime_s) e->q_reclaim_mrt.assign(s->queue_reclaim_min_runtime_s, s->queue_reclaim_min_runtime_s + s->n_queues);
  if (s->job_last_start_s) e->j_last_start.assign(s->job_last_start_s, s->job_last_start_s + s->n_jobs);
  if (s->job_stale_since_s) e->j_stale_since.assign(s->job_stale_since_s, s->job_stale_since_s + s->n_jobs);
  e->loaded = true;
  return KAI_OK;
}


extern "C" {

int kai_abi_version(void) { return KAI_ABI_VERSION; }

int kai_engine_create(const kai_config *cfg, kai_engine **out) {
  if (!cfg || !out) return KAI_ERR_INVALID;
  if (cfg->abi_version != KAI_ABI_VERSION) return KAI_ERR_INVALID;
  int n_dev = 0;
  cudaError_t ce = cudaGetDeviceCount(&n_dev);
  if (ce != cudaSuccess || n_dev <= 0 || cfg->device < 0 || cfg->device >= n_dev) return KAI_ERR_NO_DEVICE;
  kai_engine *e = new kai_engine();
  e->cfg = *cfg;
  if (e->cfg.shard_count < 1) e->cfg.shard_count = 1;
  e->device = cfg->device;
  memset(&e->stats, 0, sizeof(e->stats));
  if (cudaSetDevice(e->device) != cudaSuccess) {
    delete e;
    return KAI_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, e->device) != cudaSuccess) {
    delete e;
    return KAI_ERR_NO_DEVICE;
  }
  if (prop.major < 10) {  // sm_100a cubin only
    delete e;
    return KAI_ERR_NO_DEVICE;
  }
  e->num_sms = prop.multiProcessorCount;
  e->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete e;
    return KAI_ERR_CUDA;
  }
  for (auto &ev : e->ev) cudaEventCreate(&ev);
  cudaEventCreateWithFlags(&e->ev_mirror, cudaEventDisableTiming);
  {  // pinned, device-mapped protocol buffers of the host-sequenced mode
    const size_t list_words = (size_t)2 * kListScanners * kListLines * kListLineWords;
    size_t words = (size_t)2 * kDecWords * 2 + (size_t)2 * kMaxDelta * 2 + (size_t)2 * 2 * kMaxGrid * kSlotWords + list_words;
    if (cudaHostAlloc((void **)&e->h_pinned, words * 8, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
      delete e;
      return KAI_ERR_CUDA;
    }
    memset(e->h_pinned, 0, words * 8);
    e->h_rec = e->h_pinned;
    e->h_delta = e->h_rec + (size_t)2 * kDecWords * 2;
    e->h_slots = e->h_delta + (size_t)2 * kMaxDelta * 2;
    e->h_mm = e->h_slots + (size_t)2 * kMaxGrid * kSlotWords;
    e->h_list = e->h_mm + (size_t)2 * kMaxGrid * kSlotWords;
    if (cudaHostAlloc((void **)&e->h_clist, (size_t)2 * kCListWords * 8, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
      delete e;
      return KAI_ERR_CUDA;
    }
    memset(e->h_clist, 0, (size_t)2 * kCListWords * 8);
  }
  *out = e;
  return KAI_OK;
}

void kai_engine_destroy(kai_engine *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  e->dsnap.release();
  e->dreplica.release();
  e->dmisc.release();
  e->stage.release();
  e->rstage.release();
  if (e->h_pinned) cudaFreeHost(e->h_pinned);
  if (e->h_clist) cudaFreeHost(e->h_clist);
  e->dlaunch.release();
  if (e->d_node_domain) cudaFree(e->d_node_domain);
  if (e->shm_base) {
    if (e->shm_registered) cudaHostUnregister(e->shm_base);
    munmap(e->shm_base, e->shm_bytes);
    if (e->shm_owner) shm_unlink(e->shm_name);
  }
  for (auto &ev : e->ev)
    if (ev) cudaEventDestroy(ev);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

const char *kai_last_error(const kai_engine *e) { return e ? e->err.c_str() : "null engine"; }

int kai_engine_load_snapshot(kai_engine *e, const kai_snapshot *s) {
  if (!e || !s) return KAI_ERR_INVALID;
  if (s->abi_version != KAI_ABI_VERSION) return e->fail(KAI_ERR_INVALID, "snapshot abi_version mismatch");
  if (s->n_res < 4 || s->n_res > KAI_MAX_RES) return e->fail(KAI_ERR_INVALID, "n_res out of range");
  if (s->n_nodes < 0 || s->n_queues < 0 || s->n_jobs < 0 || s->n_podsets < 0 || s->n_tasks < 0)
    return e->fail(KAI_ERR_INVALID, "negative count");
  if (!s->node_allocatable || !s->node_idle || !s->node_releasing || !s->node_name_rank || !s->node_flags)
    if (s->n_nodes > 0) return e->fail(KAI_ERR_INVALID, "null node table");
  CK(cudaSetDevice(e->device));
  {  // resident snapshot: same structure as the previous load -> only the per-cycle columns are refreshed
    const int opt = (s->queue_usage ? 1 : 0) | (s->node_foreign ? 2 : 0) | (s->task_nominated ? 4 : 0) | (s->task_pred_class ? 8 : 0) |
                    (s->pred_mask ? 16 : 0) | (s->node_gpu_count ? 32 : 0) | ((s->n_topologies > 0) ? 64 : 0);
    const int shape[8] = {s->n_res, s->n_nodes, s->n_queues, s->n_jobs, s->n_podsets, s->n_tasks, s->n_pred_classes, opt};
    const bool resident = e->loaded && s->structure_epoch != 0 && s->structure_epoch == e->structure_epoch &&
                          memcmp(shape, e->shape, sizeof(shape)) == 0 && !getenv("KAI_NO_RESIDENT");
    memcpy(e->shape, shape, sizeof(shape));
    e->structure_epoch = s->structure_epoch;
    if (resident) {
      const int R = s->n_res, N = s->n_nodes, Q = s->n_queues, T = s->n_tasks;
      const size_t RN = (size_t)R * N, QN = (size_t)QR * Q;
      e->loaded = false;
      for (int t = 0; t < T; t++) {
        int n = s->task_node[t];
        if (n >= N) return e->fail(KAI_ERR_INVALID, "bad task_node");
        if ((s->task_status[t] & kActiveUsed) && n < 0) return e->fail(KAI_ERR_INVALID, "active task without node");
      }
      cudaEventRecord(e->ev[0], e->stream);
      unsigned char *h = e->stage.host, *d = e->dsnap.base;
      memcpy(h + e->off_idle, s->node_idle, RN * 8);
      memcpy(h + e->off_rel, s->node_releasing, RN * 8);
      memcpy(h + e->off_nflags, s->node_flags, (size_t)N * 4);
      if (s->queue_usage) memcpy(h + e->off_usage, s->queue_usage, QN * 8);
      {
        const std::vector<int> &perm = e->task_perm;
        int *x = (int *)(h + e->off_tst), *y = (int *)(h + e->off_tnst), *tn = (int *)(h + e->off_tnode);
        for (int t = 0; t < T; t++) {
          const int st = s->task_status[perm[t]];
          x[t] = y[t] = st;
          tn[t] = (st & kActiveUsed) ? s->task_node[perm[t]] : -1;
        }
      }
      // idle | releasing and status | node | node status are adjacent regions of the arena: one copy each
      CK(cudaMemcpyAsync(d + e->off_idle, h + e->off_idle, (e->off_rel - e->off_idle) + RN * 8, cudaMemcpyHostToDevice, e->stream));
      CK(cudaMemcpyAsync(d + e->off_nflags, h + e->off_nflags, (size_t)N * 4, cudaMemcpyHostToDevice, e->stream));
      if (s->queue_usage) CK(cudaMemcpyAsync(d + e->off_usage, h + e->off_usage, QN * 8, cudaMemcpyHostToDevice, e->stream));
      CK(cudaMemcpyAsync(d + e->off_tst, h + e->off_tst, (e->off_tnst - e->off_tst) + (size_t)std::max(T, 1) * 4, cudaMemcpyHostToDevice, e->stream));
      CK(cudaMemsetAsync(d + e->dev_only_begin, 0, e->dev_only_bytes, e->stream));
      cudaEventRecord(e->ev[1], e->stream);
      return load_tail(e, s, e->n_dom_levels, true);
    }
  }
  e->loaded = false;
  const int R = s->n_res, N = s->n_nodes, Q = s->n_queues, J = s->n_jobs, S = s->n_podsets, T = s->n_tasks;
  e->R = R;
  e->N = N;
  e->Q = Q;
  e->J = J;
  e->S = S;
  e->T = T;
  const int NPC = s->n_pred_classes;
  const int mask_words = (N + 31) / 32;

  // ---------------- host-side derived index structures ----------------
  std::vector<int> rank_to_node(N, -1);
  for (int n = 0; n < N; n++) {
    int rk = s->node_name_rank[n];
    if (rk < 0 || rk >= N || rank_to_node[rk] != -1) return e->fail(KAI_ERR_INVALID, "node_name_rank is not a permutation");
    rank_to_node[rk] = n;
  }
  std::vector<int> q_nchildren(Q, 0), q_child_begin(Q + 1, 0), q_children(std::max(Q, 1), 0), top;
  for (int q = 0; q < Q; q++) {
    int p = s->queue_parent[q];
    if (p >= Q || p == q || p < -1) return e->fail(KAI_ERR_INVALID, "bad queue_parent");
    if (p >= 0)
      q_nchildren[p]++;
    else
      top.push_back(q);
  }
  for (int q = 0; q < Q; q++) q_child_begin[q + 1] = q_child_begin[q] + q_nchildren[q];
  {
    std::vector<int> fill(q_child_begin.begin(), q_child_begin.end() - 1);
    for (int q = 0; q < Q; q++) {
      int p = s->queue_parent[q];
      if (p >= 0) q_children[fill[p]++] = q;
    }
  }
  // levels for the fair-share recursion (proportion.go:410-423): level 0 = {top group}
  std::vector<int> level_group_begin{0}, level_groups;
  {
    std::vector<int> cur{-1};
    int depth = 0;
    while (!cur.empty()) {
      if (++depth > KAI_MAX_QUEUE_DEPTH + 1) return e->fail(KAI_ERR_INVALID, "queue hierarchy too deep or cyclic");
      std::vector<int> next;
      for (int g : cur) {
        level_groups.push_back(g);
        if (g < 0) {
          for (int q : top)
            if (q_nchildren[q] > 0) next.push_back(q);
        } else {
          for (int k = q_child_begin[g]; k < q_child_begin[g + 1]; k++)
            if (q_nchildren[q_children[k]] > 0) next.push_back(q_children[k]);
        }
      }
      level_group_begin.push_back((int)level_groups.size());
      cur.swap(next);
    }
  }
  const int n_levels = (int)level_group_begin.size() - 1;
  // jobs grouped by leaf queue, in (priority desc, order_rank) order
  std::vector<int> q_job_begin(Q + 1, 0), q_jobs_sorted(std::max(J, 1), 0);
  {
    std::vector<int> cnt(Q, 0);
    for (int j = 0; j < J; j++) {
      int q = s->job_queue[j];
      if (q >= Q) return e->fail(KAI_ERR_INVALID, "bad job_queue");
      if (q < 0 || q_nchildren[q] != 0) continue;  // input_jobs.go:47-63
      int p = s->queue_parent[q];
      (void)p;
      cnt[q]++;
    }
    for (int q = 0; q < Q; q++) q_job_begin[q + 1] = q_job_begin[q] + cnt[q];
    std::vector<int> fill(q_job_begin.begin(), q_job_begin.end() - 1);
    // job_order_rank is a rank (a permutation of 0..J-1) in every well-formed snapshot: walk the jobs in rank order so
    // that each queue's list is already ordered by rank, then only a stable pass on priority is left (a no-op when the
    // priorities of a queue are already non-increasing, the common case).  Anything else falls back to a full sort.
    std::vector<int> by_rank(std::max(J, 1), -1);
    bool ranks_are_a_permutation = true;
    for (int j = 0; j < J && ranks_are_a_permutation; j++) {
      int rk = s->job_order_rank[j];
      if (rk < 0 || rk >= J || by_rank[rk] != -1)
        ranks_are_a_permutation = false;
      else
        by_rank[rk] = j;
    }
    for (int k = 0; k < J; k++) {
      int j = ranks_are_a_permutation ? by_rank[k] : k;
      int q = s->job_queue[j];
      if (q < 0 || q_nchildren[q] != 0) continue;
      q_jobs_sorted[fill[q]++] = j;
    }
    auto by_priority = [&](int a, int b) { return s->job_priority[a] > s->job_priority[b]; };
    for (int q = 0; q < Q; q++) {
      auto b = q_jobs_sorted.begin() + q_job_begin[q], en = q_jobs_sorted.begin() + q_job_begin[q + 1];
      if (ranks_are_a_permutation) {
        if (!std::is_sorted(b, en, by_priority)) std::stable_sort(b, en, by_priority);
      } else {
        std::sort(b, en, [&](int a, int b2) {
          if (s->job_priority[a] != s->job_priority[b2]) return s->job_priority[a] > s->job_priority[b2];
          return s->job_order_rank[a] < s->job_order_rank[b2];
        });
      }
    }
  }
  // podsets / tasks
  // device task i = caller task perm[i]: the tasks of a podset are renumbered into TaskOrderFn order so that
  // the kernels never chase an index array (results are scattered back through perm on download)
  std::vector<int> ps_job(std::max(S, 1), 0), t_job(std::max(T, 1), 0), t_podset(std::max(T, 1), 0);
  std::vector<int> &perm = e->task_perm;
  perm.assign(std::max(T, 1), 0);
  int max_job_tasks = 1, max_job_podsets = 1;
  for (int j = 0; j < J; j++) {
    int b = s->job_podset_begin[j], en = s->job_podset_begin[j + 1];
    if (b < 0 || en < b || en > S) return e->fail(KAI_ERR_INVALID, "bad job_podset_begin");
    max_job_podsets = std::max(max_job_podsets, en - b);
    int nt = 0;
    for (int ps = b; ps < en; ps++) {
      ps_job[ps] = j;
      int tb = s->podset_task_begin[ps], te = s->podset_task_begin[ps + 1];
      if (tb < 0 || te < tb || te > T) return e->fail(KAI_ERR_INVALID, "bad podset_task_begin");
      nt += te - tb;
      for (int t = tb; t < te; t++) {
        t_job[t] = j;
        t_podset[t] = ps;
        perm[t] = t;
      }
      std::stable_sort(perm.begin() + tb, perm.begin() + te,
                       [&](int a, int b2) { return s->task_order_rank[a] < s->task_order_rank[b2]; });
    }
    max_job_tasks = std::max(max_job_tasks, nt);
  }
  if (J > 0 && (s->job_podset_begin[0] != 0 || s->job_podset_begin[J] != S))
    return e->fail(KAI_ERR_INVALID, "job_podset_begin must cover all podsets");
  if (S > 0 && (s->podset_task_begin[0] != 0 || s->podset_task_begin[S] != T))
    return e->fail(KAI_ERR_INVALID, "podset_task_begin must cover all tasks");
  for (int t = 0; t < T; t++) {
    int n = s->task_node[t];
    if (n >= N) return e->fail(KAI_ERR_INVALID, "bad task_node");
    if ((s->task_status[t] & kActiveUsed) && n < 0) return e->fail(KAI_ERR_INVALID, "active task without node");
  }

  // ---------------- layout of the device arena (upload region first, then device-only) ----------------
  cudaEventRecord(e->ev[0], e->stream);
  size_t up = 0;
  auto reserve_up = [&](size_t bytes) {
    size_t o = up;
    up += align_up(bytes, 256);
    return o;
  };
  const size_t RN = (size_t)R * N, QN = (size_t)QR * Q;
  size_t o_alloc = reserve_up(RN * 8), o_idle = reserve_up(RN * 8), o_rel = reserve_up(RN * 8);
  size_t o_rank = reserve_up((size_t)N * 4), o_r2n = reserve_up((size_t)N * 4), o_nflags = reserve_up((size_t)N * 4);
  size_t o_gpuc = reserve_up((size_t)N * 8);
  size_t o_foreign = s->node_foreign ? reserve_up((size_t)3 * N * 8) : 0;
  size_t o_qparent = reserve_up((size_t)Q * 4), o_qprio = reserve_up((size_t)Q * 4), o_quid = reserve_up((size_t)Q * 4);
  size_t o_qnch = reserve_up((size_t)Q * 4), o_qcreate = reserve_up((size_t)Q * 8);
  size_t o_qdes = reserve_up(QN * 8), o_qlim = reserve_up(QN * 8), o_qoqw = reserve_up(QN * 8);
  size_t o_quse = s->queue_usage ? reserve_up(QN * 8) : 0;
  size_t o_qcb = reserve_up((size_t)(Q + 1) * 4), o_qch = reserve_up((size_t)std::max(Q, 1) * 4);
  size_t o_top = reserve_up((size_t)std::max((int)top.size(), 1) * 4);
  size_t o_lgb = reserve_up(level_group_begin.size() * 4), o_lg = reserve_up(std::max<size_t>(level_groups.size(), 1) * 4);
  size_t o_qjb = reserve_up((size_t)(Q + 1) * 4), o_qjs = reserve_up((size_t)std::max(J, 1) * 4);
  size_t o_jq = reserve_up((size_t)std::max(J, 1) * 4), o_jp = reserve_up((size_t)std::max(J, 1) * 4);
  size_t o_jor = reserve_up((size_t)std::max(J, 1) * 4), o_jfl = reserve_up((size_t)std::max(J, 1) * 4);
  size_t o_jpb = reserve_up((size_t)(J + 1) * 4);
  size_t o_psmin = reserve_up((size_t)std::max(S, 1) * 4), o_pstb = reserve_up((size_t)(S + 1) * 4);
  size_t o_psjob = reserve_up((size_t)std::max(S, 1) * 4);
  size_t o_treq = reserve_up((size_t)std::max(T, 1) * R * 8);
  size_t o_tjob = reserve_up((size_t)std::max(T, 1) * 4), o_tps = reserve_up((size_t)std::max(T, 1) * 4);
  size_t o_tnom = s->task_nominated ? reserve_up((size_t)std::max(T, 1) * 4) : 0;
  size_t o_tpc = s->task_pred_class ? reserve_up((size_t)std::max(T, 1) * 4) : 0;
  size_t o_tst = reserve_up((size_t)std::max(T, 1) * 4), o_tnode = reserve_up((size_t)std::max(T, 1) * 4);
  size_t o_tnst = reserve_up((size_t)std::max(T, 1) * 4);
  size_t o_mask = (s->pred_mask && NPC > 0) ? reserve_up((size_t)NPC * mask_words * 4) : 0;
  const size_t upload_bytes = up;
  e->off_idle = o_idle;
  e->off_rel = o_rel;
  e->off_nflags = o_nflags;
  e->off_usage = o_quse;
  e->off_tst = o_tst;
  e->off_tnode = o_tnode;
  e->off_tnst = o_tnst;
  // device-only region
  size_t o_tvirt = reserve_up((size_t)std::max(T, 1));
  size_t o_qfair = reserve_up(QN * 8), o_qreq = reserve_up(QN * 8), o_qal = reserve_up(QN * 8), o_qalnp = reserve_up(QN * 8);
  size_t o_total = reserve_up(3 * 8);
  size_t o_qla = reserve_up(QN * 8);
  size_t o_jkey = reserve_up((size_t)std::max(J, 1) * 8), o_leafs = reserve_up((size_t)std::max(J, 1) * 4);
  size_t o_leafc = reserve_up((size_t)std::max(Q, 1) * 4), o_pscnt = reserve_up((size_t)3 * std::max(S, 1) * 4);
  size_t o_jreq = reserve_up((size_t)std::max(J, 1) * QR * 8), o_jreqv = reserve_up((size_t)std::max(J, 1));
  const int ops_cap = 4 * max_job_tasks + 64;
  size_t o_ops = reserve_up(sizeof(Op) * (size_t)ops_cap);
  size_t o_tta = reserve_up((size_t)(max_job_tasks + 1) * 4), o_psord = reserve_up((size_t)(max_job_podsets + 1) * 4);
  auto a16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
  // hot per-queue sequencer arrays — must match the carving in sequencer_main
  const size_t hot = 2 * a16(sizeof(double) * QR * Q) + a16(sizeof(QKey) * (size_t)Q) + 5 * a16(sizeof(int) * (size_t)Q) +
                     a16(sizeof(int) * (size_t)(top.size() + 1)) + a16((size_t)Q) +
                     a16(sizeof(unsigned int) * (size_t)((J + 31) / 32 + 1));
  size_t o_hot = reserve_up(hot + 16);
  size_t o_jrec = reserve_up(sizeof(JobRec) * (size_t)std::max(J, 1));
  const size_t zero_begin = o_tvirt, zero_bytes = up - o_tvirt;

  CK(e->dsnap.reserve(up + 256));
  CK(e->stage.reserve(up + 256));  // the staging buffer doubles as the host mirror of the whole arena
  e->dev_only_begin = zero_begin;
  e->dev_only_bytes = zero_bytes;
  e->rank_to_node_h = rank_to_node;
  unsigned char *h = e->stage.host;
  unsigned char *d = e->dsnap.base;
  auto put = [&](size_t off, const void *src, size_t bytes) {
    if (bytes) memcpy(h + off, src, bytes);
  };
  put(o_alloc, s->node_allocatable, RN * 8);
  put(o_idle, s->node_idle, RN * 8);
  put(o_rel, s->node_releasing, RN * 8);
  put(o_rank, s->node_name_rank, (size_t)N * 4);
  put(o_r2n, rank_to_node.data(), (size_t)N * 4);
  put(o_nflags, s->node_flags, (size_t)N * 4);
  if (s->node_gpu_count)
    put(o_gpuc, s->node_gpu_count, (size_t)N * 8);
  else
    put(o_gpuc, s->node_allocatable + (size_t)KAI_RES_GPU * N, (size_t)N * 8);
  if (s->node_foreign) put(o_foreign, s->node_foreign, (size_t)3 * N * 8);
  put(o_qparent, s->queue_parent, (size_t)Q * 4);
  put(o_qprio, s->queue_priority, (size_t)Q * 4);
  put(o_quid, s->queue_uid_rank, (size_t)Q * 4);
  put(o_qnch, q_nchildren.data(), (size_t)Q * 4);
  put(o_qcreate, s->queue_creation, (size_t)Q * 8);
  put(o_qdes, s->queue_deserved, QN * 8);
  put(o_qlim, s->queue_limit, QN * 8);
  put(o_qoqw, s->queue_oqw, QN * 8);
  if (s->queue_usage) put(o_quse, s->queue_usage, QN * 8);
  put(o_qcb, q_child_begin.data(), (size_t)(Q + 1) * 4);
  put(o_qch, q_children.data(), (size_t)Q * 4);
  put(o_top, top.data(), top.size() * 4);
  put(o_lgb, level_group_begin.data(), level_group_begin.size() * 4);
  put(o_lg, level_groups.data(), level_groups.size() * 4);
  put(o_qjb, q_job_begin.data(), (size_t)(Q + 1) * 4);
  put(o_qjs, q_jobs_sorted.data(), (size_t)J * 4);
  put(o_jq, s->job_queue, (size_t)J * 4);
  put(o_jp, s->job_priority, (size_t)J * 4);
  put(o_jor, s->job_order_rank, (size_t)J * 4);
  put(o_jfl, s->job_flags, (size_t)J * 4);
  put(o_jpb, s->job_podset_begin, (size_t)(J + 1) * 4);
  put(o_psmin, s->podset_min_available, (size_t)S * 4);
  put(o_pstb, s->podset_task_begin, (size_t)(S + 1) * 4);
  put(o_psjob, ps_job.data(), (size_t)S * 4);
  {
    double *tr = (double *)(h + o_treq);
    for (int t = 0; t < T; t++) memcpy(tr + (size_t)t * R, s->task_req + (size_t)perm[t] * R, (size_t)R * 8);
  }
  put(o_tjob, t_job.data(), (size_t)T * 4);
  put(o_tps, t_podset.data(), (size_t)T * 4);
  if (s->task_nominated) {
    int *x = (int *)(h + o_tnom);
    for (int t = 0; t < T; t++) x[t] = s->task_nominated[perm[t]];
  }
  if (s->task_pred_class) {
    int *x = (int *)(h + o_tpc);
    for (int t = 0; t < T; t++) x[t] = s->task_pred_class[perm[t]];
  }
  {
    int *x = (int *)(h + o_tst), *y = (int *)(h + o_tnst);
    for (int t = 0; t < T; t++) x[t] = y[t] = s->task_status[perm[t]];
  }
  {
    int *tn = (int *)(h + o_tnode);
    for (int t = 0; t < T; t++) tn[t] = (s->task_status[perm[t]] & kActiveUsed) ? s->task_node[perm[t]] : -1;
  }
  if (o_mask || (s->pred_mask && NPC > 0)) put(o_mask, s->pred_mask, (size_t)NPC * mask_words * 4);

  CK(cudaMemcpyAsync(d, h, upload_bytes, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemsetAsync(d + zero_begin, 0, zero_bytes, e->stream));
  cudaEventRecord(e->ev[1], e->stream);

  DevSnap &ds = e->ds;
  memset(&ds, 0, sizeof(ds));
  ds.R = R;
  ds.N = N;
  ds.Q = Q;
  ds.J = J;
  ds.S = S;
  ds.T = T;
  ds.NPC = NPC;
  ds.mask_words = mask_words;
  ds.n_top = (int)top.size();
  ds.max_job_tasks = max_job_tasks;
  ds.max_job_podsets = max_job_podsets;
  ds.n_levels = n_levels;
  ds.alloc = (const double *)(d + o_alloc);
  ds.idle = (double *)(d + o_idle);
  ds.rel = (double *)(d + o_rel);
  ds.name_rank = (const int *)(d + o_rank);
  ds.rank_to_node = (const int *)(d + o_r2n);
  ds.nflags = (const uint32_t *)(d + o_nflags);
  ds.gpu_count = (const double *)(d + o_gpuc);
  ds.foreign = s->node_foreign ? (const double *)(d + o_foreign) : nullptr;
  ds.q_parent = (const int *)(d + o_qparent);
  ds.q_priority = (const int *)(d + o_qprio);
  ds.q_uid_rank = (const int *)(d + o_quid);
  ds.q_nchildren = (const int *)(d + o_qnch);
  ds.q_creation = (const long long *)(d + o_qcreate);
  ds.q_deserved = (const double *)(d + o_qdes);
  ds.q_limit = (const double *)(d + o_qlim);
  ds.q_oqw = (const double *)(d + o_qoqw);
  ds.q_usage = s->queue_usage ? (const double *)(d + o_quse) : nullptr;
  ds.q_fair = (double *)(d + o_qfair);
  ds.q_request = (double *)(d + o_qreq);
  ds.q_alloc = (double *)(d + o_qal);
  ds.q_alloc_np = (double *)(d + o_qalnp);
  ds.q_child_begin = (const int *)(d + o_qcb);
  ds.q_children = (const int *)(d + o_qch);
  ds.top_queues = (const int *)(d + o_top);
  ds.level_group_begin = (const int *)(d + o_lgb);
  ds.level_groups = (const int *)(d + o_lg);
  ds.q_job_begin = (const int *)(d + o_qjb);
  ds.q_jobs_sorted = (const int *)(d + o_qjs);
  ds.j_queue = (const int *)(d + o_jq);
  ds.j_priority = (const int *)(d + o_jp);
  ds.j_order_rank = (const int *)(d + o_jor);
  ds.j_flags = (const uint32_t *)(d + o_jfl);
  ds.j_ps_begin = (const int *)(d + o_jpb);
  ds.ps_min = (const int *)(d + o_psmin);
  ds.ps_task_begin = (const int *)(d + o_pstb);
  ds.ps_job = (const int *)(d + o_psjob);
  ds.t_req = (const double *)(d + o_treq);
  ds.t_job = (const int *)(d + o_tjob);
  ds.t_podset = (const int *)(d + o_tps);
  ds.t_nominated = s->task_nominated ? (const int *)(d + o_tnom) : nullptr;
  ds.t_pred_class = s->task_pred_class ? (const int *)(d + o_tpc) : nullptr;
  ds.t_status = (int *)(d + o_tst);
  ds.t_node = (int *)(d + o_tnode);
  ds.t_node_status = (int *)(d + o_tnst);
  ds.t_virtual = (unsigned char *)(d + o_tvirt);
  ds.pred_mask = (s->pred_mask && NPC > 0) ? (const uint32_t *)(d + o_mask) : nullptr;
  ds.total = (double *)(d + o_total);
  ds.q_allocatable = (double *)(d + o_qla);
  ds.j_key0 = (unsigned long long *)(d + o_jkey);
  ds.leaf_sorted = (int *)(d + o_leafs);
  ds.leaf_count = (int *)(d + o_leafc);
  ds.ps_cnt0 = (int *)(d + o_pscnt);
  ds.j_req = (double *)(d + o_jreq);
  ds.j_req_valid = (unsigned char *)(d + o_jreqv);
  ds.ops = (Op *)(d + o_ops);
  ds.tta = (int *)(d + o_tta);
  ds.ps_order = (int *)(d + o_psord);
  ds.hot_global = d + o_hot;
  ds.jrec = (JobRec *)(d + o_jrec);
  {  // host view: every pointer of ds rebased onto the staging buffer (same offsets)
    static_assert(sizeof(void *) == 8, "64-bit only");
    e->hs = ds;
    unsigned char *hb_ = e->stage.host;
    auto rb = [&](auto &ptr) {
      if (ptr) {
        unsigned char *raw = (unsigned char *)ptr;
        ptr = (std::remove_reference_t<decltype(ptr)>)(hb_ + (raw - d));
      }
    };
    DevSnap &h_ = e->hs;
    rb(h_.alloc); rb(h_.idle); rb(h_.rel); rb(h_.name_rank); rb(h_.rank_to_node); rb(h_.nflags); rb(h_.gpu_count);
    rb(h_.foreign); rb(h_.q_parent); rb(h_.q_priority); rb(h_.q_uid_rank); rb(h_.q_nchildren); rb(h_.q_creation);
    rb(h_.q_deserved); rb(h_.q_limit); rb(h_.q_oqw); rb(h_.q_usage); rb(h_.q_fair); rb(h_.q_request); rb(h_.q_alloc);
    rb(h_.q_alloc_np); rb(h_.q_child_begin); rb(h_.q_children); rb(h_.top_queues); rb(h_.level_group_begin);
    rb(h_.level_groups); rb(h_.q_job_begin); rb(h_.q_jobs_sorted); rb(h_.j_queue); rb(h_.j_priority);
    rb(h_.j_order_rank); rb(h_.j_ps_begin); rb(h_.j_flags); rb(h_.ps_min); rb(h_.ps_task_begin); rb(h_.ps_job);
    rb(h_.t_req); rb(h_.t_job); rb(h_.t_podset); rb(h_.t_nominated); rb(h_.t_pred_class); rb(h_.t_status);
    rb(h_.t_node); rb(h_.t_node_status); rb(h_.t_virtual); rb(h_.pred_mask); rb(h_.total); rb(h_.q_allocatable);
    rb(h_.j_key0); rb(h_.leaf_sorted); rb(h_.leaf_count); rb(h_.ps_cnt0); rb(h_.j_req); rb(h_.j_req_valid);
    rb(h_.ops); rb(h_.tta); rb(h_.ps_order); rb(h_.hot_global); rb(h_.jrec);
  }

  // ---------------- launch geometry of the action kernel ----------------
  // CTA 0 = sequencer, CTAs 1..grid-1 = scanners that split the node rows
  int grid = std::min(e->num_sms, kMaxGrid);
  if (const char *g = getenv("KAI_GRID")) {
    int v = atoi(g);
    if (v >= 2) grid = std::min(v, grid);
  }
  const int n_shard_rows = (N + e->cfg.shard_count - 1) / e->cfg.shard_count;  // rows of the largest shard
  if (N > 0) grid = std::min(grid, n_shard_rows + 1);  // at least one node per scanner when possible
  grid = std::max(grid, 2);
  if (const char *g = getenv("KAI_GRID_EXACT")) {  // tests: force scanners without nodes as well
    int v = atoi(g);
    if (v >= 2) grid = std::min(std::min(v, e->num_sms), kMaxGrid);
  }
  int npc = std::max(1, (n_shard_rows + (grid - 1) - 1) / (grid - 1));
  npc = (npc + 1) & ~1;  // keep the int arrays 8-byte aligned
  const int n_dom_levels = (s->n_topologies > 0 && s->topology_level_begin && s->node_domain) ? s->topology_level_begin[s->n_topologies] : 0;
  if (n_dom_levels > kMaxDomLevels) return e->fail(KAI_ERR_UNSUPPORTED, "more topology levels than kMaxDomLevels");
  // a GPU request with a fractional part is a shared-GPU pod (gpu_resource_requirment.go:52-54,230-234): it needs the
  // per-GPU-group tables of gpu_sharing_node_info.go, which this ABI does not carry; refuse instead of treating the
  // fraction as a plain quantity
  for (int t = 0; t < s->n_tasks; t++) {
    const double g = s->task_req[(size_t)t * R + KAI_RES_GPU];
    if (g != (double)(long long)g) return e->fail(KAI_ERR_UNSUPPORTED, "fractional GPU request: GPU sharing is outside this engine's scope");
  }
  size_t tile_bytes = align_up((size_t)npc * ((size_t)2 * R * 8 + 3 * 8 + 4 + 4 + 4 + (size_t)4 * n_dom_levels), 16);
  const size_t smem_limit = (size_t)e->max_smem_optin - 28 * 1024;  // static shared memory of k_action
  if (tile_bytes > smem_limit)
    return e->fail(KAI_ERR_UNSUPPORTED, "node tile does not fit in shared memory (N too large for one GPU tile)");
  bool hot_in_smem = hot <= smem_limit;
  if (getenv("KAI_NO_SMEM_HOT")) hot_in_smem = false;
  e->grid = grid;
  e->npc = npc;
  e->tile_bytes = tile_bytes;
  e->hot_bytes = hot;
  e->hot_in_smem = hot_in_smem;
  e->smem_bytes = std::max(tile_bytes, hot_in_smem ? hot : (size_t)0);
  e->ops_cap = ops_cap;
  e->visits_cap = std::max(16, 2 * J + T + 16);
  {  // launch transport: scanners = CTAs of k_record; k_merge sorts scanners x kTopM candidates (<= kMergeThreads)
    int lg = 1;
    while (lg * 2 <= std::min(2 * e->num_sms, kMergeThreads / kTopM)) lg *= 2;  // 256 on B200: a power of two keeps the merge sort full
    if (const char *g = getenv("KAI_LAUNCH_GRID")) {
      int v = atoi(g);
      if (v >= 1) lg = std::min(v, kMergeThreads / kTopM);
    }
    if (N > 0) lg = std::min(lg, std::max(1, n_shard_rows));
    if (const char *g = getenv("KAI_GRID_EXACT")) {  // tests: the same forced geometries as the persistent kernel (grid - 1 scanners)
      int v = atoi(g);
      if (v >= 2) lg = std::min(v - 1, kMergeThreads / kTopM);
    }
    int lnpc = std::max(1, (n_shard_rows + lg - 1) / lg);
    lnpc = (lnpc + 1) & ~1;
    e->lgrid = lg;
    e->lnpc = lnpc;
    e->ltile_bytes = align_up((size_t)lnpc * ((size_t)2 * R * 8 + 3 * 8 + 4 + 4 + 4 + (size_t)4 * n_dom_levels), 16);
    e->ltile_stride = align_up(e->ltile_bytes, 256);
    // dynamic shared memory of k_record: the staged tile during a sweep (scanned from global memory when it does not fit)
    e->lsmem_bytes = e->ltile_bytes <= (size_t)e->max_smem_optin - 40 * 1024 ? e->ltile_bytes : 16;
    const size_t list_words = (size_t)2 * kListScanners * kListLines * kListLineWords;
    CK(e->dlaunch.reserve((size_t)lg * e->ltile_stride + (size_t)lg * align_up(kScanStateBytes, 256) + list_words * 8 + 4096));
    e->g_tiles = e->dlaunch.take<unsigned char>((size_t)lg * e->ltile_stride);
    e->g_scan_state = e->dlaunch.take<unsigned char>((size_t)lg * kScanStateBytes);
    e->d_list = e->dlaunch.take<unsigned long long>(list_words);
    e->ticket = e->dlaunch.take<unsigned int>(4);
    e->mm_result = e->dlaunch.take<double>(4);
    CK(cudaMemsetAsync(e->d_list, 0, list_words * 8, e->stream));
    CK(cudaMemsetAsync(e->ticket, 0, 16, e->stream));
    CK(cudaMemsetAsync(e->mm_result, 0, 32, e->stream));
  }
  {
    size_t xb = (size_t)2 * kMaxGrid * 8 * 8;
    size_t misc = 2 * xb + 256 + sizeof(long long) * 48 + sizeof(kai_job_visit) * (size_t)e->visits_cap + 2 * QN * 8 + 4096 +
                  sizeof(unsigned long long) * 2 * kDecWords * 2 + sizeof(unsigned long long) * 2 * kMaxDelta * 2 + 1024;
    CK(e->dmisc.reserve(misc));
    e->xbuf = e->dmisc.take<unsigned long long>(2 * kMaxGrid * 8);
    e->mmbuf = e->dmisc.take<unsigned long long>(2 * kMaxGrid * 8);
    e->counters = e->dmisc.take<long long>(48);
    e->d_visits = e->dmisc.take<kai_job_visit>(e->visits_cap);
    e->fs_w = e->dmisc.take<double>(QN + 1);
    e->fs_rr = e->dmisc.take<double>(QN + 1);
    e->dbuf = e->dmisc.take<unsigned long long>(2 * kDecWords * 2);
    e->delta = e->dmisc.take<unsigned long long>(2 * kMaxDelta * 2);
    CK(cudaMemsetAsync(e->delta, 0, sizeof(unsigned long long) * 2 * kMaxDelta * 2, e->stream));
    CK(cudaMemsetAsync(e->dbuf, 0, sizeof(unsigned long long) * 2 * kDecWords * 2, e->stream));
    CK(cudaMemsetAsync(e->xbuf, 0, xb, e->stream));
    CK(cudaMemsetAsync(e->mmbuf, 0, xb, e->stream));
    // sequence numbers stay monotone across snapshots (tags of older cycles can never match); a rare full reset
    // keeps the 24-bit slot tags unambiguous
    if (e->seq > (1u << 22) && e->cfg.shard_count == 1) {
      e->seq = 2;
      memset(e->h_pinned, 0, ((size_t)2 * kDecWords * 2 + (size_t)2 * kMaxDelta * 2 + (size_t)2 * 2 * kMaxGrid * kSlotWords +
                              (size_t)2 * kListScanners * kListLines * kListLineWords) * 8);
    }
  }

  return load_tail(e, s, n_dom_levels, false);
}

static int download(kai_engine *e, kai_result *out, long long n_visits, long long placed, long long evicted) {
  const DevSnap &ds = e->ds;
  const size_t QN = (size_t)QR * e->Q, RN = (size_t)e->R * e->N;
  cudaEventRecord(e->ev[4], e->stream);
  e->r_tmp_node.resize(std::max(e->T, 1));
  e->r_tmp_status.resize(std::max(e->T, 1));
  CK(cudaMemcpyAsync(e->r_tmp_node.data(), ds.t_node, (size_t)e->T * 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_tmp_status.data(), ds.t_status, (size_t)e->T * 4, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_fair.data(), ds.q_fair, QN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_alloc.data(), ds.q_alloc, QN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_alloc_np.data(), ds.q_alloc_np, QN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_request.data(), ds.q_request, QN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_idle.data(), ds.idle, RN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_rel.data(), ds.rel, RN * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemcpyAsync(e->r_total, ds.total, 3 * 8, cudaMemcpyDeviceToHost, e->stream));
  long long nv = std::min<long long>(n_visits, e->visits_cap);
  e->r_visits.resize((size_t)nv);
  if (nv > 0)
    CK(cudaMemcpyAsync(e->r_visits.data(), e->d_visits, (size_t)nv * sizeof(kai_job_visit), cudaMemcpyDeviceToHost,
                       e->stream));
  cudaEventRecord(e->ev[5], e->stream);
  CK(cudaStreamSynchronize(e->stream));
  for (int t = 0; t < e->T; t++) {  // device order -> caller order
    e->r_task_node[e->task_perm[t]] = e->r_tmp_node[t];
    e->r_task_status[e->task_perm[t]] = e->r_tmp_status[t];
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[4], e->ev[5]);
  e->stats.download_ms = ms;
  memset(out, 0, sizeof(*out));
  out->n_tasks = e->T;
  out->task_node = e->r_task_node.data();
  out->task_status = e->r_task_status.data();
  out->n_visits = (int)nv;
  out->visits = e->r_visits.data();
  out->n_queues = e->Q;
  out->queue_fair_share = e->r_fair.data();
  out->queue_allocated = e->r_alloc.data();
  out->queue_allocated_non_preemptible = e->r_alloc_np.data();
  out->queue_request = e->r_request.data();
  out->total_resource = e->r_total;
  out->n_nodes = e->N;
  out->node_idle = e->r_idle.data();
  out->node_releasing = e->r_rel.data();
  out->pods_placed = placed;
  out->pods_evicted = evicted;
  return KAI_OK;
}

int kai_engine_fair_share(kai_engine *e, kai_result *out) {
  if (!e || !out) return KAI_ERR_INVALID;
  if (!e->loaded) return e->fail(KAI_ERR_STATE, "no snapshot loaded");
  CK(cudaSetDevice(e->device));
  return download(e, out, 0, 0, 0);
}

// Launch transport: enqueue the kernel launch(es) of one decision record on the engine's stream.
static bool engine_launch_record(void *ctx, const LaunchRec &rec) {
  kai_engine *e = (kai_engine *)ctx;
  const int kind = (int)(rec.dw[0] & 0xff);
  const unsigned int xbits = (unsigned int)((rec.dw[0] >> 48) & 0xffff);
  const size_t dyn = e->lsmem_bytes;
  if (kind == DK_SCAN && (xbits & XB_FUSED_MM) && e->lp.fused_in_kernel) {
    // every CTA is resident (checked at load): the scanners exchange their binpack extremes among themselves
    // through tagged device slots inside this one launch
    void *args[] = {(void *)&e->lp, (void *)&rec};
    cudaLaunchCooperativeKernel((const void *)k_record, dim3(e->lgrid), dim3(kThreads), args, dyn, e->stream);
    e->record_launches++;
  } else if (kind == DK_SCAN && (xbits & XB_FUSED_MM)) {
    // pack.go:66-86 over the row set of this sweep: a MINMAX launch (applies the deltas and the feasible-set snapshot,
    // leaves the reduced extremes in device memory) followed by the sweep itself, back to back on the stream
    LaunchRec a = rec;
    a.dw[0] = (rec.dw[0] & ~0xffull) | (unsigned long long)DK_MINMAX;
    k_record<<<e->lgrid, kThreads, dyn, e->stream>>>(e->lp, a);
    LaunchRec b = rec;
    b.n_delta = 0;
    b.dw[0] = rec.dw[0] & ~(0xffffull << 32) & ~((unsigned long long)(XB_SNAP_ALL | XB_SNAP_GPUFREE) << 48);
    k_record<<<e->lgrid, kThreads, dyn, e->stream>>>(e->lp, b);
    e->record_launches += 2;
  } else {
    k_record<<<e->lgrid, kThreads, dyn, e->stream>>>(e->lp, rec);
    e->record_launches++;
    if (kind == DK_TOPK || (kind == DK_SCAN && e->lp.topm && !(xbits & XB_SINGLE))) {  // list answer: sort, cut, stream to the host
      if (e->merge_cluster)
        k_merge_cluster<<<kMergeCtas, kMergeCtaThreads, kMergeCtaSmemBytes, e->stream>>>(e->lp, rec.seq, kind == DK_SCAN ? 1 : 0);
      else
        k_merge<<<1, kMergeThreads, kMergeSmemBytes, e->stream>>>(e->lp, rec.seq, kind == DK_SCAN ? 1 : 0);
      e->record_launches++;
    }
  }
  return cudaPeekAtLastError() == cudaSuccess;
}

int kai_engine_run(kai_engine *e, kai_action action, kai_result *out) {
  if (!e || !out) return KAI_ERR_INVALID;
  if (!e->loaded) return e->fail(KAI_ERR_STATE, "no snapshot loaded");
  const bool solver_action = action == KAI_ACTION_RECLAIM || action == KAI_ACTION_CONSOLIDATION || action == KAI_ACTION_PREEMPT ||
                             action == KAI_ACTION_STALEGANGEVICTION;
  if (action != KAI_ACTION_ALLOCATE && !solver_action) return e->fail(KAI_ERR_UNSUPPORTED, "unknown action");
  if (e->cfg.shard_count > 1 && !e->shm_base) return e->fail(KAI_ERR_STATE, "multi-GPU: call kai_engine_wire_peers first");
  CK(cudaSetDevice(e->device));
  ActionParams p;
  memset(&p, 0, sizeof(p));
  p.s = e->ds;
  p.cfg = e->cfg;
  p.action = (int)action;
  p.grid = e->grid;
  p.nodes_per_cta = e->npc;
  p.dbuf = e->dbuf;
  p.delta = e->delta;
  p.ops_cap = e->ops_cap;
  p.xbuf = e->xbuf;
  p.mmbuf = e->mmbuf;
  p.visits = e->d_visits;
  p.visits_cap = e->visits_cap;
  p.counters = e->counters;
  p.node_domain = e->d_node_domain;
  p.n_dom_levels = e->n_dom_levels;
  p.seq0 = e->seq;
  p.hot_in_smem = e->hot_in_smem ? 1 : 0;
  p.tile_bytes = e->tile_bytes;
  p.hot_bytes = e->hot_bytes;
  p.batching = getenv("KAI_NO_BATCHING") ? 0 : 1;
  CK(cudaFuncSetAttribute(k_action, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->smem_bytes));
  int max_blocks = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks, k_action, kThreads, e->smem_bytes));
  if (max_blocks < 1 || max_blocks * e->num_sms < e->grid)
    return e->fail(KAI_ERR_CUDA, "action kernel cannot be made co-resident");
  const char *mode_env = getenv("KAI_SEQUENCER");
  const bool host_mode = !(mode_env && strcmp(mode_env, "device") == 0);
  if (!host_mode && e->cfg.shard_count > 1) return e->fail(KAI_ERR_UNSUPPORTED, "device-resident sequencer is single-GPU");
  if (solver_action && !host_mode) return e->fail(KAI_ERR_UNSUPPORTED, "reclaim / consolidation / preempt run host-sequenced");
  if (solver_action && e->cfg.shard_count > 1 && !e->mirror_valid)
    return e->fail(KAI_ERR_UNSUPPORTED, "multi-GPU solver actions need every earlier action of the cycle to be host-sequenced");
  if (!host_mode) e->mirror_valid = false;
  if (!host_mode && e->topo.any())
    for (int j = 0; j < e->J; j++)
      if (e->topo.constrained(j)) return e->fail(KAI_ERR_UNSUPPORTED, "topology constraints need the host-sequenced mode");
  // transport of the host-sequenced mode: "launch" (default) = one k_record launch per decision record, tiles in global
  // memory; "persistent" = the cooperative scan-server kernel polling records in pinned host memory
  const char *tr_env = getenv("KAI_TRANSPORT");
  const bool launch_mode = host_mode && !(tr_env && strcmp(tr_env, "persistent") == 0);
  p.mode = host_mode ? (launch_mode ? 2 : 1) : 0;
  p.spin_log2 = host_mode ? 26 : 22;
  if (host_mode) {
    p.h_rec = e->h_rec;
    p.h_delta = e->h_delta;
    // one reduced answer line per GPU; with several GPUs the lines live in the shared segment
    unsigned long long *lines = e->cfg.shard_count > 1 ? e->shm_dev : e->h_slots;
    unsigned long long *mm_lines = e->cfg.shard_count > 1 ? e->shm_dev + (size_t)2 * kMaxGrid * kSlotWords : e->h_mm;
    p.h_slot = lines + (size_t)e->cfg.shard_rank * kSlotWords;
    p.h_mmslot = mm_lines + (size_t)e->cfg.shard_rank * kSlotWords;
    p.topm = (p.batching && !getenv("KAI_NO_TOPM")) ? 1 : 0;
    p.h_list = e->cfg.shard_count > 1 ? e->shm_dev + (size_t)2 * 2 * kMaxGrid * kSlotWords : e->h_list;
    p.scanner_base = e->cfg.shard_rank * (e->grid - 1);
    if ((long long)e->cfg.shard_count * (e->grid - 1) > kListScanners) p.topm = 0;
    if (launch_mode) {
      if (e->cfg.shard_count > kShmRanks) return e->fail(KAI_ERR_UNSUPPORTED, "more GPUs than the exchange segment holds");
      p.grid = e->lgrid + 1;  // scanners = grid - 1, as in the persistent kernel
      p.nodes_per_cta = e->lnpc;
      p.topm = (p.batching && !getenv("KAI_NO_TOPM")) ? 1 : 0;
      p.h_list = e->d_list;  // the scanners' top-M lines stay on the device; the last CTA merges them
      p.scanner_base = 0;
      p.g_tiles = e->g_tiles;
      p.g_tile_stride = e->ltile_stride;
      p.g_scan_state = e->g_scan_state;
      p.ticket = e->ticket;
      p.mm_result = e->mm_result;
      p.h_clist = e->cfg.shard_count > 1 ? e->shm_dev + shm_clist_offset_words() + (size_t)e->cfg.shard_rank * 2 * kCListWords : e->h_clist;
      p.spin_log2 = 22;
      p.tile_bytes = e->ltile_bytes;
      p.hot_in_smem = e->ltile_bytes <= e->lsmem_bytes ? 1 : 0;  // the scanners stage their tile in shared memory for a sweep
      {
        int per_sm = 0;
        CK(cudaFuncSetAttribute(k_record, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->lsmem_bytes));
        CK(cudaFuncSetAttribute(k_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMergeSmemBytes));
        {
          const char *mk = getenv("KAI_MERGE");
          e->merge_cluster = !(mk && strcmp(mk, "single") == 0);
        }
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_record, kThreads, e->lsmem_bytes));
        p.fused_in_kernel = (per_sm * e->num_sms >= e->lgrid && !getenv("KAI_NO_FUSED_LAUNCH")) ? 1 : 0;
      }
    }
  }
  void *args[] = {(void *)&p};
  CK(cudaMemsetAsync(e->counters, 0, sizeof(long long) * 48, e->stream));
  cudaEventRecord(e->ev[2], e->stream);
  if (e->J > 0) k_prep_jobs<<<std::min(e->num_sms * 8, (e->J + 255) / 256), 256, 0, e->stream>>>(e->ds, 1, 1);
  if (e->Q > 0) k_prep_queues<<<e->Q, 256, 0, e->stream>>>(e->ds);
  long long c[48];
  memset(c, 0, sizeof(c));
  if (host_mode) {
    // host mirror of everything the open-session / prepare kernels produced
    CK(cudaMemcpyAsync(e->stage.host + e->dev_only_begin, e->dsnap.base + e->dev_only_begin, e->dev_only_bytes,
                       cudaMemcpyDeviceToHost, e->stream));
    const bool feed_mirror = solver_action || e->topo.any() || e->cfg.shard_count > 1;
    const bool refresh_mirror = feed_mirror && !e->mirror_valid;
    if (refresh_mirror) e->topo.live = false;  // the incremental per-domain state is rebuilt from the re-read tables
    if (refresh_mirror) {  // a device-sequenced action ran before: re-read the node tables (one GPU)
      e->h_tmp.resize((size_t)2 * e->R * e->N);
      if (e->N > 0) {
        CK(cudaMemcpyAsync(e->h_tmp.data(), e->ds.idle, sizeof(double) * (size_t)e->R * e->N, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaMemcpyAsync(e->h_tmp.data() + (size_t)e->R * e->N, e->ds.rel, sizeof(double) * (size_t)e->R * e->N, cudaMemcpyDeviceToHost, e->stream));
      }
    }
    cudaEventRecord(e->ev_mirror, e->stream);
    if (launch_mode) {
      CK(cudaFuncSetAttribute(k_record, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->lsmem_bytes));
      e->lp = p;
      e->record_launches = 0;
      LaunchRec load;
      memset(&load, 0, sizeof(load));
      load.dw[0] = (unsigned long long)DK_LOAD;
      load.seq = p.seq0;
      if (!engine_launch_record(e, load)) return e->cuda_fail(cudaGetLastError(), "k_record (tile load)");
    } else {
      CK(cudaLaunchCooperativeKernel((const void *)k_action, dim3(e->grid), dim3(kThreads), args, e->smem_bytes, e->stream));
      cudaEventRecord(e->ev[3], e->stream);
    }
    // wait for the mirror copy only (the kernel keeps running): event-free trick = query the D2H through an event
    cudaEvent_t mirror_done = e->ev[4];
    (void)mirror_done;
    // the D2H above precedes the kernel in stream order; its completion is observed by polling a sentinel
    // written last: simplest robust way is a second stream-ordered event recorded before the launch.
    // (see below: ev_mirror)
    HostBackend &hb = e->hb;
    hb.h_rec = e->h_rec;
    hb.h_delta = e->h_delta;
    hb.h_slots = e->cfg.shard_count > 1 ? e->shm_base : e->h_slots;
    hb.h_mm = e->cfg.shard_count > 1 ? e->shm_base + (size_t)2 * kMaxGrid * kSlotWords : e->h_mm;
    hb.n_scanners = e->cfg.shard_count;  // the relay CTA of every GPU reduces its scanners' answers: one line per GPU
    hb.topm = p.topm;
    hb.prof = getenv("KAI_PROFILE") != nullptr;
    for (int i = 0; i < 8; i++) hb.t_sec[i] = 0;
    for (int i = 0; i < 4; i++) hb.t_pop_split[i] = 0;
    {  // job order of the allocate action: "keyed" (default; used when the snapshot allows it) or "replica"
      const char *jo = getenv("KAI_JOB_ORDER");
      hb.keyed_order_allowed = !(jo && strcmp(jo, "replica") == 0);
      hb.keyed_order_used = false;
    }
    hb.h_list = e->cfg.shard_count > 1 ? e->shm_base + (size_t)2 * 2 * kMaxGrid * kSlotWords : e->h_list;
    hb.n_list_scanners = e->cfg.shard_count * (e->grid - 1);
    hb.launch_mode = launch_mode;
    hb.launch_fn = &engine_launch_record;
    hb.launch_ctx = e;
    hb.launches = 0;
    hb.t_launch = 0;
    hb.n_ranks = e->cfg.shard_count;
    hb.h_clist = e->cfg.shard_count > 1 ? e->shm_base + shm_clist_offset_words() : e->h_clist;
    hb.listed = 0;
    hb.batch_is_single = false;
    hb.list_yield_ema = 8.0;
    hb.list_served = -1;
    hb.single_streak = 0;
    hb.single_sweeps = 0;
    hb.n_flush = hb.n_topo_jobs = hb.n_topo_domains = 0;
    hb.t_topo[0] = hb.t_topo[1] = hb.t_topo[2] = 0;
    hb.list_invalidate();
    hb.batching = p.batching;
    hb.failed = false;
    hb.gang_fast = getenv("KAI_NO_GANG_FAST") == nullptr;
    hb.gang_bulk = hb.gang_replayed = hb.gang_failed = 0;
    hb.rank_to_node = e->rank_to_node_h.data();
    CK(cudaEventSynchronize(e->ev_mirror));
    if (refresh_mirror && !e->h_tmp.empty()) {  // re-read tables -> node-major mirror
      for (int n = 0; n < e->N; n++)
        for (int r = 0; r < e->R; r++) {
          e->h_mirror[(size_t)n * 2 * e->R + r] = e->h_tmp[(size_t)r * e->N + n];
          e->h_mirror[(size_t)n * 2 * e->R + e->R + r] = e->h_tmp[(size_t)(e->R + r) * e->N + n];
        }
    }
    if (feed_mirror) e->mirror_valid = true;  // from here on the host-sequenced deltas keep it in step
    // ---- sequencer state on the host ----
    const DevSnap &hs = e->hs;
    const int Q = e->Q, J = e->J;
    e->hot_host.assign(e->hot_bytes + 64, 0);
    Seq &seq = hb.seq;
    Ctl &ctl = hb.ctl;
    memset(&ctl, 0, sizeof(ctl));
    memset(&seq, 0, sizeof(seq));
    {
      unsigned char *h = e->hot_host.data();
      auto take_from = [](unsigned char *&base, size_t bytes) {
        unsigned char *r = base;
        base += (bytes + 15) & ~(size_t)15;
        return r;
      };
      Replica &rp = seq.rp;
      rp.q_alloc = (double *)take_from(h, sizeof(double) * QR * Q);
      rp.q_alloc_np = (double *)take_from(h, sizeof(double) * QR * Q);
      rp.qkey = (QKey *)take_from(h, sizeof(QKey) * Q);
      rp.leaf_head = (int *)take_from(h, sizeof(int) * Q);
      rp.leaf_end = (int *)take_from(h, sizeof(int) * Q);
      rp.ovl_len = (int *)take_from(h, sizeof(int) * Q);
      rp.child_len = (int *)take_from(h, sizeof(int) * Q);
      rp.child_heap = (int *)take_from(h, sizeof(int) * Q);
      rp.root_heap = (int *)take_from(h, sizeof(int) * (hs.n_top + 1));
      rp.qn_flags = (unsigned char *)take_from(h, Q);
      rp.touched = (unsigned int *)take_from(h, sizeof(unsigned int) * ((J + 31) / 32 + 1));
      rp.t_status = hs.t_status;
      rp.t_node = hs.t_node;
      rp.t_node_status = hs.t_node_status;
      rp.t_virtual = hs.t_virtual;
      rp.ps_active_alloc = hs.ps_cnt0;
      rp.ps_pending = hs.ps_cnt0 + hs.S;
      rp.ps_pipelined = hs.ps_cnt0 + 2 * hs.S;
      rp.j_req = hs.j_req;
      rp.j_req_valid = hs.j_req_valid;
      rp.j_key = hs.j_key0;
      rp.leaf_heap = hs.leaf_sorted;
      rp.ops = hs.ops;
      rp.tta = hs.tta;
      rp.ps_order = hs.ps_order;
      for (int i = 0; i < QR * Q; i++) {
        rp.q_alloc[i] = hs.q_alloc[i];
        rp.q_alloc_np[i] = hs.q_alloc_np[i];
      }
      for (int i = 0; i < Q; i++) {
        int b = hs.q_job_begin[i];
        rp.leaf_head[i] = b;
        rp.leaf_end[i] = b + (hs.q_nchildren[i] == 0 ? hs.leaf_count[i] : 0);
      }
    }
    seq.s = &e->hs;
    seq.cfg = &e->cfg;
    seq.p = &p;
    seq.delta_base = e->h_delta;
    seq.host_backend = &hb;
    // The mirror is fed by the delta stream whenever something will read it: solver actions, topology, several GPUs.
    // A plain single-GPU allocate skips that (one cache line per placement) and marks the mirror stale instead; a
    // later solver action of the cycle re-reads the node tables from the device.
    seq.mirror = feed_mirror ? e->h_mirror.data() : nullptr;
    if (!feed_mirror) e->mirror_valid = false;
    e->topo.mirror = e->h_mirror.data();
    e->topo.t_req = hs.t_req;
    e->topo.t_podset = hs.t_podset;
    seq.topology = e->topo.any() ? &e->topo : nullptr;
    seq.on_node_changed = &TopologyHost::node_changed_hook;
    e->topo.reset_gpu_state();
    seq.ctl = &ctl;
    seq.ops_cap = e->ops_cap;
    seq.batching = p.batching;
    seq.is_cta0 = true;
    e->r_visits.assign((size_t)e->visits_cap, kai_job_visit{0, 0});
    seq.visits = e->r_visits.data();
    seq.visits_cap = e->visits_cap;
    ctl.trk[0].dirty = ctl.trk[1].dirty = 1;
    ctl.trk[0].mn = ctl.trk[1].mn = DBL_MAX;
    ctl.dec.nominated = ctl.dec.pred_class = -1;
    ctl.dec.task = -1;
    ctl.ctx_job = ctl.ctx_ps = -1;
    ctl.seq = p.seq0;
    long long solver_scenarios = 0, solver_topk = 0;
    if (!solver_action) {
      hb.run_allocate();
    } else {
      const int T = e->T;
      if ((int)e->on_other_node.size() != T) {
        e->on_other_node.assign(T, -1);
        e->on_other_status.assign(T, 0);
      }
      std::vector<int> n0(T), s0(T);
      for (int t = 0; t < T; t++) {
        bool on = (hs.t_status[t] & kActiveUsed) && hs.t_node[t] >= 0;
        n0[t] = on ? hs.t_node[t] : -1;
        s0[t] = hs.t_node_status[t];
      }
      double t_begin = HostBackend::now();
      Solver solver(hb, n0, s0, e->on_other_node, e->on_other_status, e->on_extra);
      solver.use_signatures = e->cfg.use_scheduling_signatures != 0;
      solver.job_signature = e->job_signature.empty() ? nullptr : e->job_signature.data();
      solver.q_preempt_mrt = e->q_preempt_mrt.empty() ? nullptr : e->q_preempt_mrt.data();
      solver.q_reclaim_mrt = e->q_reclaim_mrt.empty() ? nullptr : e->q_reclaim_mrt.data();
      solver.j_last_start = e->j_last_start.empty() ? nullptr : e->j_last_start.data();
      solver.j_stale_since = e->j_stale_since.empty() ? nullptr : e->j_stale_since.data();
      solver.now_s = e->now_s;
      if (action == KAI_ACTION_RECLAIM)
        solver.run_reclaim();
      else if (action == KAI_ACTION_PREEMPT)
        solver.run_preempt();
      else if (action == KAI_ACTION_STALEGANGEVICTION)
        solver.run_stale_gang_eviction();
      else
        solver.run_consolidation();
      hb.publish(DK_DONE);
      hb.t_total = HostBackend::now() - t_begin;
      if (getenv("KAI_PROFILE"))
        fprintf(stderr, "[kai] solver host profile: %lld simulations; sweeps %.1f ms, simulation set-up %.1f ms, evicting recorded victims %.1f ms, victims queues %.1f ms\n",
                solver.simulations, solver.t_sweeps * 1e3, solver.t_sim_setup * 1e3, solver.t_evict * 1e3, solver.t_victims_queue * 1e3);
      if (getenv("KAI_PROFILE"))
        fprintf(stderr, "[kai] solver host profile: scenario loop: victims pop %.1f ms, tasks_to_evict %.1f, add potential %.1f, filter %.1f, filter init (top-k sweep) %.1f, by-pod solve %.1f\n",
                solver.t_vq_pop * 1e3, solver.t_tte * 1e3, solver.t_addp * 1e3, solver.t_filter * 1e3, solver.t_finit * 1e3, solver.t_bypod * 1e3);
      solver_scenarios = solver.scenarios;
      solver_topk = solver.topk_sweeps;
      // one status per task for the allocate path: the entry on the task's current node; the other entry persists
      for (auto &x : e->on_extra) {  // the entry on the task's current node belongs in slot 0
        const int t = x[0], cur = hs.t_node[t];
        if (x[1] == cur && n0[t] != cur && e->on_other_node[t] != cur) {
          if (n0[t] < 0) {
            n0[t] = x[1];
            s0[t] = x[2];
            x[0] = -1;
          } else {
            std::swap(n0[t], x[1]);
            std::swap(s0[t], x[2]);
          }
        }
      }
      e->on_extra.erase(std::remove_if(e->on_extra.begin(), e->on_extra.end(), [](const std::array<int, 3> &x) { return x[0] < 0; }),
                        e->on_extra.end());
      for (int t = 0; t < T; t++) {
        int cur = hs.t_node[t];
        if (n0[t] >= 0 && n0[t] != cur && e->on_other_node[t] == cur) {
          std::swap(n0[t], e->on_other_node[t]);
          std::swap(s0[t], e->on_other_status[t]);
        }
        if (n0[t] >= 0 && n0[t] == cur)
          hs.t_node_status[t] = s0[t];
        else if (n0[t] >= 0) {  // only a stale entry on another node: it persists as "other" (or beyond the two slots)
          if (e->on_other_node[t] < 0) {
            e->on_other_node[t] = n0[t];
            e->on_other_status[t] = s0[t];
          } else {
            e->on_extra.push_back({t, n0[t], s0[t]});
          }
        }
      }
    }
    if (launch_mode) cudaEventRecord(e->ev[3], e->stream);  // after the DONE launch: the action's span on the device
    CK(cudaStreamSynchronize(e->stream));
    if (launch_mode) CK(cudaGetLastError());
    if (solver_action && getenv("KAI_PROFILE"))
      fprintf(stderr, "[kai] solver: %lld scenarios simulated, %lld node sweeps, %lld top-k sweeps, %lld minmax exchanges\n",
              solver_scenarios, seq.sweeps, solver_topk, seq.minmax_exchanges);
    {
      long long cd[48];
      CK(cudaMemcpy(cd, e->counters, sizeof(cd), cudaMemcpyDeviceToHost));
      for (int i = 20; i < 32; i++) c[i] = cd[i];
      for (int i = 32; i < 48; i++) c[i] = cd[i];
    }
    c[0] = seq.n_visits;
    c[1] = seq.sweeps;
    c[2] = seq.nodes_scanned;
    c[3] = seq.pods_placed;
    c[4] = seq.pods_evicted;
    c[5] = seq.minmax_exchanges;
    c[6] = seq.error;
    c[7] = ctl.seq + 1;
    c[15] = seq.batched + hb.listed;
    if (hb.failed && c[24] == 0) c[24] = 99;
    // session state back to the device copies (later actions' prepare kernels and the result download read them)
    for (int i = 0; i < QR * Q; i++) {
      hs.q_alloc[i] = seq.rp.q_alloc[i];
      hs.q_alloc_np[i] = seq.rp.q_alloc_np[i];
    }
    auto up = [&](const void *hp, size_t bytes) {
      size_t off = (const unsigned char *)hp - e->stage.host;
      return cudaMemcpyAsync(e->dsnap.base + off, hp, bytes, cudaMemcpyHostToDevice, e->stream);
    };
    CK(up(hs.t_status, (size_t)e->T * 4));
    CK(up(hs.t_node, (size_t)e->T * 4));
    CK(up(hs.t_node_status, (size_t)e->T * 4));
    CK(up(hs.t_virtual, (size_t)e->T));
    CK(up(hs.q_alloc, (size_t)QR * Q * 8));
    CK(up(hs.q_alloc_np, (size_t)QR * Q * 8));
    if (e->visits_cap > 0 && seq.n_visits > 0)
      CK(cudaMemcpyAsync(e->d_visits, e->r_visits.data(), sizeof(kai_job_visit) * (size_t)std::min<long long>(seq.n_visits, e->visits_cap),
                         cudaMemcpyHostToDevice, e->stream));
  } else {
    CK(cudaLaunchCooperativeKernel((const void *)k_action, dim3(e->grid), dim3(kThreads), args, e->smem_bytes, e->stream));
    cudaEventRecord(e->ev[3], e->stream);
    CK(cudaMemcpyAsync(c, e->counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  }
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[2], e->ev[3]);
  e->stats.action_ms = ms;
  e->stats.decisions = c[1];
  e->stats.nodes_scanned = c[2];
  e->stats.algorithmic_bytes = c[2] * ((2 * e->R + 1) * 8 + 4);
  e->stats.kernel_launches += (launch_mode ? e->record_launches : 1) + (e->J > 0) + (e->Q > 0);
  e->seq = (unsigned int)c[7];
  if (getenv("KAI_PROFILE")) {
    const char *nm[] = {"init", "pop", "prepare", "keycalc", "exchange", "apply", "finish"};
    fprintf(stderr, "[kai] %s-sequenced action %.3f ms, %lld sweeps, %lld batched placements, %lld minmax exchanges, hot_in_smem=%d; CTA0 thread0 cycles:", host_mode ? "host" : "device", ms, c[1], c[15], c[5], (int)e->hot_in_smem);
    for (int i = 0; i < 7; i++) fprintf(stderr, " %s=%lld", nm[i], c[8 + i]);
    fprintf(stderr, " n_key=%lld tta=%lld popheap=%lld\n", c[16], c[17], c[18]);
    if (host_mode)
      fprintf(stderr, "[kai] host sequencer (%s transport, %lld record launches): total %.3f ms, of which waiting for sweeps %.3f ms (%.2f us per sweep)\n",
              launch_mode ? "launch" : "persistent", launch_mode ? e->record_launches : 0LL, e->hb.t_total * 1e3, e->hb.t_exchange * 1e3,
              c[1] ? e->hb.t_exchange * 1e6 / c[1] : 0.0);
    if (host_mode && launch_mode) fprintf(stderr, "[kai] launch calls: %.3f ms on the host thread (%.2f us per record)\n", e->hb.t_launch * 1e3, e->hb.launches ? e->hb.t_launch * 1e6 / e->hb.launches : 0.0);
    if (host_mode) fprintf(stderr, "[kai] sweeps answered with a single row (XB_SINGLE): %lld; FLUSH records %lld\n", e->hb.single_sweeps, e->hb.n_flush);
    if (host_mode) fprintf(stderr, "[kai] fresh gangs: %lld committed in bulk, %lld replayed per task, %lld discarded\n", e->hb.gang_bulk, e->hb.gang_replayed, e->hb.gang_failed);
    if (host_mode && e->hb.n_topo_jobs)
      fprintf(stderr, "[kai] topology: %lld constrained jobs with candidates, %lld domains tried; subSetNodesFn %.1f ms, score table %.1f ms, placing %.1f ms\n",
              e->hb.n_topo_jobs, e->hb.n_topo_domains, e->hb.t_topo[0] * 1e3, e->hb.t_topo[1] * 1e3, e->hb.t_topo[2] * 1e3);
    if (host_mode)
      fprintf(stderr, "[kai] host sequencer rdtsc Mcycles: pop %.2f admit %.2f place(+sweeps) %.2f finish %.2f loop %.2f\n",
              e->hb.t_sec[0] / 1e6, e->hb.t_sec[1] / 1e6, e->hb.t_sec[2] / 1e6, e->hb.t_sec[3] / 1e6, e->hb.t_sec[4] / 1e6);
    if (host_mode && !solver_action) {
      if (e->hb.keyed_order_used)
        fprintf(stderr, "[kai] job order: keyed; eligibility check %.3f Mcycles, tree build %.3f Mcycles\n", e->hb.t_sec[5] / 1e6,
                e->hb.t_sec[6] / 1e6);
      else
        fprintf(stderr, "[kai] job order: replica (%s, queue %d); eligibility check %.3f Mcycles, tree build %.3f Mcycles; pop Mcycles: fix root %.2f fix children %.2f keys %.2f leaf pop + handle_pop %.2f\n",
                e->hb.korder.reason, e->hb.korder.reason_queue,
                e->hb.t_sec[5] / 1e6, e->hb.t_sec[6] / 1e6, e->hb.t_pop_split[0] / 1e6, e->hb.t_pop_split[1] / 1e6,
                e->hb.t_pop_split[2] / 1e6, e->hb.t_pop_split[3] / 1e6);
    }
    if (host_mode && c[45] > 0)
      fprintf(stderr, "[kai] %s: %lld cycles per list (%lld lists): load %lld, sort %lld, prefix + payload %lld, stream out %lld, fence + header %lld\n",
              e->merge_cluster ? "k_merge_cluster" : "k_merge", c[44] / c[45], c[45], c[39] / c[45], c[46] / c[45], c[31] / c[45], c[47] / c[45], c[43] / c[45]);
    if (host_mode && c[22] > 0)
      fprintf(stderr, "[kai] relay CTA per record: forward %lld cycles, scanners+reduce %lld cycles (%lld records)\n",
              c[20] / c[22], c[21] / c[22], c[22]);
    if (host_mode && c[38] > 0)
      fprintf(stderr, "[kai] scanner 0 per record (cycles): wait-for-record %lld (of which word-0 poll %lld), decode %lld, deltas %lld, scan %lld, scan+publish %lld\n",
              c[33] / c[38], c[32] / c[38], c[34] / c[38], c[35] / c[38], c[36] / c[38], c[37] / c[38]);
    if (host_mode && c[38] > 0)
      fprintf(stderr, "[kai] publish_candidate of scanner 0 (cycles per record): row+advance %lld, key %lld, events+pack %lld\n",
              c[40] / c[38], c[41] / c[38], c[42] / c[38]);
  }
  if (c[24] != 0) {
    char msg[256];
    snprintf(msg, sizeof(msg), "device protocol watchdog: wait code %lld seq %lld who %lld cta %lld (seq0 %u, end seq %lld)",
             c[24], c[25], c[26], c[27], p.seq0, c[7]);
    e->loaded = false;
    std::string m2 = msg;
    if (host_mode) {
      char b2[96];
      snprintf(b2, sizeof(b2), "; relay last forwarded kind %lld seq %lld; host trace:", c[23] >> 32, c[23] & 0xffffffff);
      m2 += b2;
      unsigned int n0 = e->hb.trace_n > 16 ? e->hb.trace_n - 16 : 0;
      for (unsigned int i = n0; i < e->hb.trace_n; i++) {
        snprintf(b2, sizeof(b2), " (%u k%d nd%d)", e->hb.trace_seq[i & 63], e->hb.trace_kind[i & 63], e->hb.trace_nd[i & 63]);
        m2 += b2;
      }
    }
    return e->fail(KAI_ERR_CUDA, m2);
  }
  if (c[6] == 2) return e->fail(KAI_ERR_UNSUPPORTED, "topology: more preferred-level domains than the score table holds (kDomBuckets)");
  if (c[6] == 3) return e->fail(KAI_ERR_STATE, "keyed job order: a popped job still has pending tasks (KAI_JOB_ORDER=replica runs the replica order)");
  if (c[6] != 0) return e->fail(KAI_ERR_CUDA, "device sequencer overflow (statement log)");
  return download(e, out, c[0], c[3], c[4]);
}

int kai_engine_time_sweeps(kai_engine *e, int n_launches, double *elapsed_ms, double *merge_ms, int64_t *rows_per_launch) {
  if (!e || !elapsed_ms || !rows_per_launch || n_launches < 1) return KAI_ERR_INVALID;
  if (!e->loaded) return e->fail(KAI_ERR_STATE, "no snapshot loaded");
  CK(cudaSetDevice(e->device));
  ActionParams p;
  memset(&p, 0, sizeof(p));
  p.s = e->ds;
  p.cfg = e->cfg;
  p.action = KAI_ACTION_ALLOCATE;
  p.grid = e->lgrid + 1;
  p.nodes_per_cta = e->lnpc;
  p.xbuf = e->xbuf;
  p.mmbuf = e->mmbuf;
  p.counters = e->counters;
  p.node_domain = e->d_node_domain;
  p.n_dom_levels = e->n_dom_levels;
  p.mode = 2;
  p.spin_log2 = 22;
  p.topm = 1;
  p.batching = 1;
  p.h_list = e->d_list;
  p.g_tiles = e->g_tiles;
  p.g_tile_stride = e->ltile_stride;
  p.g_scan_state = e->g_scan_state;
  p.ticket = e->ticket;
  p.mm_result = e->mm_result;
  p.h_slot = e->h_slots;
  p.h_mmslot = e->h_mm;
  p.h_clist = e->h_clist;
  CK(cudaFuncSetAttribute(k_record, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->lsmem_bytes));
  CK(cudaFuncSetAttribute(k_merge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMergeSmemBytes));
  p.tile_bytes = e->ltile_bytes;
  p.hot_in_smem = e->ltile_bytes <= e->lsmem_bytes ? 1 : 0;
  e->lp = p;
  LaunchRec rec;
  memset(&rec, 0, sizeof(rec));
  rec.dw[0] = (unsigned long long)DK_LOAD;
  rec.seq = e->seq;
  if (!engine_launch_record(e, rec)) return e->cuda_fail(cudaGetLastError(), "k_record (tile load)");
  // one list sweep: the benchmark pod (jobs_fake/jobs.go:261-291), binpack on the GPU column with the extremes of an
  // empty-to-full cluster; no deltas, so every launch reads the same rows
  Ctl c;
  memset(&c, 0, sizeof(c));
  c.dec.req[KAI_RES_CPU] = 1000.0;
  c.dec.req[KAI_RES_MEM] = 1e9;
  c.dec.req[KAI_RES_GPU] = 1.0;
  if (e->R > 3) c.dec.req[3] = 1.0;
  c.dec.gpu_task = 1;
  c.dec.res = KAI_RES_GPU;
  c.dec.strategy = e->cfg.gpu_placement;
  c.dec.nominated = c.dec.pred_class = -1;
  c.trk[0].mn = 0.0;
  c.trk[0].mx = 8.0;
  c.trk[0].cnt_mn = c.trk[0].cnt_mx = 1;
  c.trk[1].dirty = 1;
  build_decision_words(c, DK_SCAN, 1);
  for (int i = 0; i < kDecWords; i++) rec.dw[i] = c.dw[i];
  rec.n_delta = 0;
  // the sweep kernel alone (its top-M lines stay in device memory), then the merge kernel alone on the last answer
  cudaEventRecord(e->ev[0], e->stream);
  for (int i = 0; i < n_launches; i++) {
    rec.seq = e->seq + 1 + (unsigned int)i;
    k_record<<<e->lgrid, kThreads, e->lsmem_bytes, e->stream>>>(e->lp, rec);
  }
  cudaEventRecord(e->ev[1], e->stream);
  {
    const char *mk = getenv("KAI_MERGE");
    e->merge_cluster = !(mk && strcmp(mk, "single") == 0);
  }
  for (int i = 0; i < n_launches; i++) {
    if (e->merge_cluster)
      k_merge_cluster<<<kMergeCtas, kMergeCtaThreads, kMergeCtaSmemBytes, e->stream>>>(e->lp, rec.seq, 1);
    else
      k_merge<<<1, kMergeThreads, kMergeSmemBytes, e->stream>>>(e->lp, rec.seq, 1);
  }
  cudaEventRecord(e->ev[2], e->stream);
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaGetLastError());
  float ms = 0;
  cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]);
  *elapsed_ms = ms;
  cudaEventElapsedTime(&ms, e->ev[1], e->ev[2]);
  if (merge_ms) *merge_ms = ms;
  const int n_shard_rows = e->N > e->cfg.shard_rank ? (e->N - e->cfg.shard_rank + e->cfg.shard_count - 1) / e->cfg.shard_count : 0;
  *rows_per_launch = n_shard_rows;
  e->seq += (unsigned int)n_launches + 4;
  return KAI_OK;
}

int kai_engine_stats(kai_engine *e, kai_stats *out) {
  if (!e || !out) return KAI_ERR_INVALID;
  *out = e->stats;
  return KAI_OK;
}

// Multi-GPU wiring.  Rank 0 creates the shared segment and exports its name; every rank (rank 0 included)
// passes the table of handles (only entry 0 is read) to kai_engine_wire_peers.
static int shm_map(kai_engine *e, bool create) {
  const size_t bytes = (shm_clist_offset_words() + (size_t)kShmRanks * 2 * kCListWords) * 8;
  int fd = shm_open(e->shm_name, create ? (O_CREAT | O_EXCL | O_RDWR) : O_RDWR, 0600);
  if (fd < 0) return e->fail(KAI_ERR_INVALID, std::string("shm_open failed for ") + e->shm_name);
  if (create && ftruncate(fd, (off_t)bytes) != 0) {
    close(fd);
    return e->fail(KAI_ERR_INVALID, "ftruncate failed");
  }
  void *ptr = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (ptr == MAP_FAILED) return e->fail(KAI_ERR_INVALID, "mmap failed");
  if (create) memset(ptr, 0, bytes);
  e->shm_base = (unsigned long long *)ptr;
  e->shm_bytes = bytes;
  return KAI_OK;
}

int kai_engine_export_peer_handle(kai_engine *e, uint8_t handle[KAI_PEER_HANDLE_BYTES]) {
  if (!e || !handle) return KAI_ERR_INVALID;
  memset(handle, 0, KAI_PEER_HANDLE_BYTES);
  if (e->cfg.shard_rank != 0) return KAI_OK;  // only rank 0 owns the segment
  if (!e->shm_base) {
    snprintf(e->shm_name, sizeof(e->shm_name), "/kai_b200_%d_%llx", (int)getpid(),
             (unsigned long long)std::chrono::steady_clock::now().time_since_epoch().count());
    int rc = shm_map(e, true);
    if (rc != KAI_OK) return rc;
    e->shm_owner = true;
  }
  memcpy(handle, e->shm_name, std::min(sizeof(e->shm_name), (size_t)KAI_PEER_HANDLE_BYTES - 1));
  return KAI_OK;
}

int kai_engine_wire_peers(kai_engine *e, const uint8_t *handles) {
  if (!e || !handles) return KAI_ERR_INVALID;
  if (e->cfg.shard_count <= 1) return KAI_OK;
  if (!e->shm_base) {
    memcpy(e->shm_name, handles, std::min(sizeof(e->shm_name) - 1, (size_t)KAI_PEER_HANDLE_BYTES));
    if (e->shm_name[0] != '/') return e->fail(KAI_ERR_INVALID, "peer handle 0 does not carry a segment name");
    int rc = shm_map(e, false);
    if (rc != KAI_OK) return rc;
  }
  if (!e->shm_registered) {
    CK(cudaSetDevice(e->device));
    CK(cudaHostRegister(e->shm_base, e->shm_bytes, cudaHostRegisterMapped | cudaHostRegisterPortable));
    CK(cudaHostGetDevicePointer((void **)&e->shm_dev, e->shm_base, 0));
    e->shm_registered = true;
  }
  return KAI_OK;
}

int kai_shard_range(int n_nodes, int shard_count, int shard_rank, int *first_rank, int *count) {
  if (n_nodes < 0 || shard_count < 1 || shard_rank < 0 || shard_rank >= shard_count || !first_rank || !count) return KAI_ERR_INVALID;
  // name-rank stripes: shard s owns the nodes of name rank s, s + S, s + 2S, ...
  *first_rank = shard_rank;
  *count = shard_rank < n_nodes ? (n_nodes - shard_rank + shard_count - 1) / shard_count : 0;
  return KAI_OK;
}

}  // extern "C"
