// vcalloc.cu — libvcalloc.so: C ABI (include/vcalloc.h) + host orchestration of the CUDA kernels.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false -std=c++17
//             -Xcompiler -fPIC -shared vcalloc.cu -o libvcalloc.so          (volcano_b200/build.py)
// There is no CPU path in this library: every entry point that computes needs a CUDA device.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vcalloc.h"
#include "vc_commit.cuh"
#include "vc_backfill.cuh"
#include "vc_commit_fast.cuh"
#include "vc_device.cuh"
#include "vc_evict.cuh"
#include "vc_evict.hpp"
#include "vc_host.hpp"
#include "vc_kernels.cuh"

namespace {

thread_local std::string g_err;
int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CUDA_TRY(x)                                                                     \
  do {                                                                                  \
    cudaError_t e_ = (x);                                                               \
    if (e_ != cudaSuccess) return fail(VC_ECUDA, "%s: %s", #x, cudaGetErrorString(e_)); \
  } while (0)

// mailbox: two parities x up to 2048 CTA slots (several ranks) of MBOX_STRIDE uint4; a second region of the same size serves
// the count all-gather of feasible-node sampling
constexpr size_t kMbox2Offset = (size_t)MBOX_STRIDE * 2 * 2048;                // in uint4
constexpr size_t kMboxBytes = sizeof(uint4) * MBOX_STRIDE * 2 * 2048 * 2;

// a launch whose grid.y runs over `count` groups / work items, in slices of at most 65535 (the limit of gridDim.y)
#define LAUNCH_Y_SLICED(kernel, gx, count, block, smem, stream, P, ...)                         \
  do {                                                                                           \
    for (size_t y0_ = 0; y0_ < (size_t)(count); y0_ += 65535) {                                   \
      (P).y_off = (int)y0_;                                                                      \
      dim3 g_((unsigned)(gx), (unsigned)std::min<size_t>(65535, (size_t)(count) - y0_));          \
      kernel<<<g_, block, smem, stream>>>((P), ##__VA_ARGS__);                                   \
    }                                                                                            \
    (P).y_off = 0;                                                                               \
  } while (0)

bool g_inited = false;
int g_device = -1;
int g_sm_count = 0;
int g_smem_optin = 0;  // cudaDevAttrMaxSharedMemoryPerBlockOptin of the bound device
int g_launches = 0;

// A forced or unusual launch geometry can ask for more shared memory per CTA than the device has: refuse it here, by
// name, instead of letting cudaFuncSetAttribute fail with a bare CUDA error.
int check_smem(const void *kfn, size_t smem, const char *what) {
  cudaFuncAttributes a;
  CUDA_TRY(cudaFuncGetAttributes(&a, kfn));
  if (smem + a.sharedSizeBytes > (size_t)g_smem_optin)
    return fail(VC_EUNSUPPORTED, "%s: %zu B of shared memory per CTA (+ %zu B static), the device allows %d B", what, smem,
                a.sharedSizeBytes, g_smem_optin);
  return VC_OK;
}

// Diagnostic switches: read from the environment ONCE, in vc_init (never on the per-cycle entry points), and
// overridable at run time through vc_debug_option (tests and tools/). None of them changes a result.
struct Tunables {
  int commit_ctas = 0;      // VC_COMMIT_CTAS: CTAs of the commit kernels (0 = one per SM)
  int commit_threads = 0;   // VC_COMMIT_THREADS: minimum block size
  int commit_generic = 0;   // VC_COMMIT_GENERIC: always the general commit kernel (k_commit)
  int commit_norun = 0;     // VC_COMMIT_NORUN: the incremental kernel without run-length placement batches
  int watchdog_ms = 0;      // VC_WATCHDOG_MS: exchange polls of the incremental kernel give up after this long (0 = 10 s)
  int run_max = 0;          // VC_RUN_MAX: placements per publication (0 = default: two node states per worker warp, 14)
  int prof = 0;             // VC_PROF: instrumented kernel instances (phase timers)
  int prof_owner = 0;       // VC_PROF_OWNER: owner-path statistics on stderr
  int prof_wait = 0;        // VC_PROF_WAIT: per-CTA all-gather wait of the general kernel on stderr
  int prof_upload = 0;      // VC_PROF_UPLOAD: host checkpoints of vc_snapshot_upload on stderr
  int backfill_depth1 = 0;  // VC_BACKFILL_DEPTH1: k_backfill run-ahead depth 1
  int expand_rows = 0;      // VC_EXPAND_ROWS: task rows per work item of the expand kernel
  int expand_plain = 0;     // VC_EXPAND_PLAIN: warp-store expand kernel
  int expand_chunk = 0;     // VC_EXPAND_CHUNK: nodes per staged piece
};
Tunables g_tun;
struct TunName { const char *name; int Tunables::*field; };
const TunName kTunNames[] = {
    {"VC_COMMIT_CTAS", &Tunables::commit_ctas}, {"VC_COMMIT_THREADS", &Tunables::commit_threads},
    {"VC_COMMIT_GENERIC", &Tunables::commit_generic}, {"VC_COMMIT_NORUN", &Tunables::commit_norun},
    {"VC_RUN_MAX", &Tunables::run_max}, {"VC_WATCHDOG_MS", &Tunables::watchdog_ms},
    {"VC_PROF", &Tunables::prof}, {"VC_PROF_OWNER", &Tunables::prof_owner}, {"VC_PROF_WAIT", &Tunables::prof_wait},
    {"VC_PROF_UPLOAD", &Tunables::prof_upload}, {"VC_BACKFILL_DEPTH1", &Tunables::backfill_depth1},
    {"VC_EXPAND_ROWS", &Tunables::expand_rows}, {"VC_EXPAND_PLAIN", &Tunables::expand_plain},
    {"VC_EXPAND_CHUNK", &Tunables::expand_chunk}};
void read_tunables() {
  for (const TunName &t : kTunNames)
    if (const char *e = getenv(t.name)) {
      const int v = atoi(e);
      g_tun.*(t.field) = (v == 0 && e[0] != '0') ? 1 : v;  // "VC_PROF=yes" counts as set
    }
}

double now_ms() {
  using namespace std::chrono;
  return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

// One device arena + one pinned staging arena per snapshot: the whole session goes up in a single
// cudaMemcpyAsync (SURVEY §8f-2 'upload once per cycle').
struct Arena {
  unsigned char *dev = nullptr, *pin = nullptr;
  size_t cap = 0, used = 0;
  size_t reserve(size_t bytes) {
    size_t off = (used + 255) & ~(size_t)255;
    used = off + bytes;
    return off;
  }
};

template <class T>
struct Slot {  // a typed region inside the arena
  size_t off = 0, count = 0;
  T *d(const Arena &a) const { return reinterpret_cast<T *>(a.dev + off); }
  T *h(const Arena &a) const { return reinterpret_cast<T *>(a.pin + off); }
};

}  // namespace

struct vc_result {
  std::vector<vc_decision> decisions;
  std::vector<vc_visit> visits;
  std::vector<int32_t> fit_errors;
  std::vector<int32_t> job_alloc;
  vc_stats stats{};
};

struct vc_snapshot {
  vc_dims dims{};
  DevDims dd{};
  DevConf dc{};
  vc_conf conf{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  bool uploaded = false;
  Arena in;  // uploaded inputs (H2D once per cycle)
  // ---- input slots ----
  Slot<double> n_alloc, n_idle, n_used, n_rel, n_pip, n_kalloc, n_kreq, n_knz;
  Slot<int32_t> n_max_tasks, n_pod_count, n_zone;
  Slot<uint64_t> n_labels, n_thard, n_tsoft;
  Slot<uint32_t> n_flags;
  Slot<uint8_t> zone_active;
  Slot<double> t_req, t_kreq, t_knz;
  Slot<uint32_t> t_has;
  Slot<int32_t> t_class, t_role, t_job;
  Slot<uint64_t> c_sel, c_aff, c_tolh, c_tols, c_pref;
  Slot<int32_t> c_naff, c_npref, c_prefw;
  Slot<uint32_t> c_flags;
  Slot<int32_t> j_queue, j_min, j_ntasks, j_pbe, j_taskmintotal, j_roleoff, j_prio, j_ready0, j_waiting0;
  Slot<uint32_t> j_flags, j_rank;
  Slot<double> j_alloc0, j_share0;
  Slot<int32_t> r_min, r_occ0, r_pip0, r_pending0;
  Slot<uint32_t> r_flags;
  Slot<int32_t> q_prio;
  Slot<uint32_t> q_rank, q_flags, q_alloc_has0, q_des_has, q_flags2;
  Slot<double> q_alloc0, q_des, q_share0;
  Slot<int32_t> qjobs_off, qjobs, task_order, job_task_off, tmeta;
  Slot<double> sg_req, sg_kreq, sg_knz;
  Slot<uint32_t> sg_has;
  Slot<int32_t> sg_class;
  std::vector<int32_t> group_rep, h_group_of;
  Slot<JobStatic> s_jstat;
  Slot<RoleStatic> s_rstat;
  Slot<QueueStatic> s_qstat;
  Slot<int32_t> s_heap_off;
  int fast_ready_word = 0, fast_ready_shift = 0, fast_share_on = 0, heap_total = 0, heap_in_smem = 0;
  bool fast = false;
  uint4 *ring = nullptr;
  uint4 *d_score_log = nullptr;   // [T] tagged chosen-node score per placement attempt of the run-length batches
  int last_full = 0, last_incr = 0;
  // ---- HyperNode tree (vc_snapshot_set_topology) ----
  bool has_topo = false;
  int hn_H = 1, hn_L = 1, hn_min_tier = 1, hn_cap = 1;
  std::vector<int32_t> h_member;  // [L][N]
  std::vector<int32_t> h_tier, h_parent, h_job_alloc, h_placed_off, h_placed_node;
  std::vector<uint8_t> h_job_soft;
  bool topo_any = false;  // the plugin scores pods of soft-mode topology jobs in this session
  Slot<int32_t> hn_up, hn_tier_s, hn_parent_s, job_soft_s, job_alloc0_s, placed_off_s, placed0_s, placed_n0_s;
  int32_t *rep_placed = nullptr, *d_job_alloc = nullptr;
  size_t rep_placed_count = 0, placed_total = 0;
  int topo_nval = 0;
  double topo_val[VC_MAX_TIERS + 2]{};
  Slot<int32_t> hn_member, hn_slot, cta_hn_off, cta_hn, node_chain, cta_chain_off, cta_chain;
  int chain_cap = 1, hn_smem = 0;
  Slot<double> hn_alloc, hn_used0;
  double *rep_hn_used = nullptr;
  size_t rep_hn_used_count = 0;
  double *hn_score = nullptr;  // dense pass [G][H]
  // ---- device-only buffers ----
  uint32_t *cstat = nullptr;
  double *w_idle = nullptr, *w_used = nullptr, *w_pip = nullptr, *w_kreq = nullptr, *w_knz = nullptr;  // working copies
  int32_t *w_pod_count = nullptr;
  int32_t *rep_i32 = nullptr;
  double *rep_f64 = nullptr;
  HeapEnt *rep_heap = nullptr;
  size_t rep_i32_stride = 0, rep_f64_stride = 0, rep_heap_stride = 0;
  int rep_ctas = 0;  // CTA count the replica buffers were sized for
  uint4 *mbox = nullptr;
  long long *d_prof = nullptr, *d_wait = nullptr;
  long long h_prof[16] = {0};
  vc_decision *d_decisions = nullptr;
  vc_visit *d_visits = nullptr;
  int32_t *d_fit = nullptr, *d_counters = nullptr;
  vc_decision *h_decisions = nullptr;  // pinned
  vc_visit *h_visits = nullptr;
  int32_t *h_fit = nullptr, *h_counters = nullptr;
  int max_job_tasks = 1;
  int n_cta = 0, block = 0, npc = 0;
  size_t smem_bytes = 0;
  double total[VC_MAX_DIMS]{};
  uint32_t total_has = 0;
  std::vector<vch::QAttr> qattr;
  double upload_ms = 0;
  int64_t h2d_bytes = 0;
  // ---- dense pass (K1) ----
  bool dense_ready = false;
  int n_groups = 0, n_work = 0;
  double *g_req = nullptr, *g_kreq = nullptr, *g_knz = nullptr, *g_order = nullptr, *g_best_score = nullptr;
  uint32_t *g_has = nullptr;
  int32_t *g_class = nullptr, *g_stats = nullptr, *g_best_node = nullptr;
  uint8_t *g_cat = nullptr;
  int32_t *work_group = nullptr, *work_begin = nullptr, *work_end = nullptr, *group_tasks = nullptr, *task_group = nullptr;
  double *part_score = nullptr;
  int32_t *part_node = nullptr;
  uint32_t *mask_out = nullptr;
  double *score_out = nullptr, *best_score = nullptr;
  int32_t *best_node = nullptr;
  int rows_per_item = 16;
  int mw32 = 0;        // 32-bit words per mask row on the device (16-byte pitch)
  int mw32_logical = 0;  // ... of the uint64 row the ABI hands out
  double *g_final = nullptr;   // [G][Nloc] final score of every (group, node)
  uint32_t *g_maskw = nullptr; // [G][mwg] feasibility words
  int mwg = 0;
  bool matrix_allocated = false;
  double last_expand_ms = 0, last_dense_ms = 0;
  // (the host copies of the task arrays the dense-pass grouping and the later actions read live in `ek`)
  // ---- backfill action (vc_snapshot_set_backfill / vc_backfill_run) ----
  vch::BackfillTasks bf;  // host copy of the BestEffort task list
  vch::BackfillKeep bk;   // session-open state pickUpPendingTasks needs, kept at upload when bf.n > 0
  std::vector<vc_decision> last_dec;  // operations of the last vc_allocate_run (kept visits only)
  bool alloc_ran = false, bf_ran = false;
  int last_idx_cur = 0;   // util.lastProcessedNodeIndex as the last action of the cycle left it
  int *d_dbg = nullptr;
  std::vector<int32_t> h_nominated;  // [T] node index per task or -1 (vc_snapshot_set_nominated); empty: none
  bool any_nominated = false;
  int32_t *d_nominated = nullptr;
  size_t d_nominated_cap = 0;
  bool fut_rows = false;  // Releasing / Pipelined resources present at open
  bool all_pure = true;  // every job's named roles map to one (class, request) group each: the role-keyed error cache is a no-op
  bool rows_integral = false;  // every quantity a placement adds to / subtracts from a node row is integer-valued
  void *d_bf = nullptr;   // device slab of the backfill inputs / outputs
  size_t d_bf_bytes = 0;
  // ---- preempt / reclaim actions (vc_snapshot_set_running / vc_preempt_run / vc_reclaim_run) ----
  vch::RunningTasks rt;            // host copy of node.Tasks
  std::vector<uint32_t> t_flags;   // VC_TASK_* per pending task
  vch::EvictKeep ek;               // session-open state, kept at every upload
  vch::EvictSession es;            // session state as the actions so far left it
  bool es_built = false;
  std::vector<vc_visit> last_vis;  // visits of the last vc_allocate_run
  double *w_rel = nullptr;         // working copy of Releasing (Statement.Evict adds to it)
  void *d_ev = nullptr;            // device slab: running-task table + per-preemptor scratch
  size_t d_ev_bytes = 0;
  int32_t *h_ev = nullptr;         // mapped pinned: [0..EV_PICK_K) picked nodes, [EV_CMD_OFF..] apply command
  // ---- one session across the GPUs of a node (vc_comm_create / vc_comm_attach) ----
  int world = 1, rank = 0;
  int n_cta_total = 0;             // CTAs of all ranks (the exchange); n_cta stays this rank's grid
  unsigned char *comm = nullptr;   // this rank's slab: mailbox | ring | score log (cudaMalloc, exported over CUDA IPC)
  size_t comm_bytes = 0, comm_mbox_bytes = 0, comm_ring_off = 0, comm_log_off = 0, comm_bytes_all = 0;
  unsigned char *peer_comm[8] = {nullptr};  // every rank's slab as mapped into this process (own one included)
  bool comm_attached = false;
  // ---- incremental upload (vc_snapshot_update_nodes) ----
  unsigned char *delta_pin = nullptr, *delta_dev = nullptr;
  size_t delta_cap = 0;
};

namespace {

template <class T>
void put(vc_snapshot *s, Slot<T> &slot, const T *src, size_t count, bool plan) {
  if (plan) {
    slot.count = count;
    slot.off = s->in.reserve(count * sizeof(T));
  } else if (count) {
    if (src) std::memcpy(slot.h(s->in), src, count * sizeof(T));
    else std::memset(slot.h(s->in), 0, count * sizeof(T));
  }
}

int build_devconf(vc_snapshot *s, const vc_nodes *nd) {
  const vc_conf &c = s->conf;
  DevConf &d = s->dc;
  std::memset(&d, 0, sizeof d);
  if (c.n_plugins < 0 || c.n_plugins > VC_MAX_PLUGINS) return fail(VC_EINVAL, "n_plugins out of range");
  d.n_plugins = c.n_plugins;
  for (int i = 0; i < c.n_plugins; ++i) {
    d.plugin[i] = c.plugins[i].plugin;
    d.tier[i] = c.plugins[i].tier;
    d.enabled[i] = c.plugins[i].enabled;
  }
  d.binpack_weight = c.binpack_weight;
  for (int i = 0; i < VC_MAX_DIMS; ++i) d.binpack_dim_weight[i] = c.binpack_dim_weight[i];
  d.w_least = c.w_least; d.w_most = c.w_most; d.w_balanced = c.w_balanced;
  d.w_node_affinity = c.w_node_affinity; d.w_taint = c.w_taint_toleration;
  d.predicates_enable = c.predicates_enable;
  d.enable_ecache = c.enable_predicate_error_cache;
  d.has_gang = vch::has_plugin(c, VC_PLUGIN_GANG);
  d.has_drf = vch::has_plugin(c, VC_PLUGIN_DRF);
  d.has_proportion = vch::has_plugin(c, VC_PLUGIN_PROPORTION);
  d.has_predicates = vch::has_plugin(c, VC_PLUGIN_PREDICATES);
  d.pred_predicates = vch::plugin_enabled(c, VC_PLUGIN_PREDICATES, VC_EN_PREDICATE);
  bool no = vch::plugin_enabled(c, VC_PLUGIN_NODEORDER, VC_EN_NODE_ORDER);
  d.taint_batch = no && c.w_taint_toleration != 0;
  d.nta_plugin = vch::plugin_enabled(c, VC_PLUGIN_NETWORK_TOPOLOGY_AWARE, VC_EN_NODE_ORDER);
  d.nta_on = d.nta_plugin && c.nta_normal_pod_enable;
  s->topo_any = false;
  if (d.nta_plugin)
    for (uint8_t f : s->h_job_soft) s->topo_any = s->topo_any || f;
  d.nta_tables = d.nta_on || s->topo_any;
  d.nta_weight = c.nta_weight;
  for (int i = 0; i < VC_MAX_DIMS; ++i) d.nta_dim_weight[i] = c.nta_dim_weight[i];
  d.nta_L = s->hn_L;
  d.tier_w_total = 0.0;
  for (int l = 0; l < s->hn_L; ++l) {  // tierWeights, network_topology_aware.go:469-476
    d.tier_w[l] = vch::go_pow_uint(c.nta_fading, (unsigned)(s->hn_min_tier + l - 1));
    d.tier_w_total += d.tier_w[l];
  }
  d.batch_any = no || vch::plugin_enabled(c, VC_PLUGIN_PREDICATES, VC_EN_NODE_ORDER) || d.nta_plugin;
  const size_t RN = (size_t)s->dims.n_dims * s->dims.n_nodes;
  int fut = 0;
  for (size_t i = 0; i < RN && !fut; ++i)
    if ((nd->releasing && nd->releasing[i] != 0.0) || (nd->pipelined && nd->pipelined[i] != 0.0)) fut = 1;
  {
    const int32_t n_all = s->dims.n_nodes;
    const int32_t tf = vch::num_feasible_nodes_to_find(n_all, c.percentage_nodes_to_find, c.min_nodes_to_find,
                                                       c.min_percentage_nodes_to_find);
    d.to_find = tf < n_all ? tf : 0;
    d.last_idx0 = n_all > 0 ? ((c.last_processed_node_index % n_all) + n_all) % n_all : 0;
  }
  // the topology and sampling variants of the commit kernel are <FUT, SOFT> instances
  d.has_future = fut || s->topo_any || d.to_find > 0;
  s->fut_rows = fut != 0;
  int soft = 0;
  const size_t WN = (size_t)s->dims.taint_words * s->dims.n_nodes;
  for (size_t i = 0; i < WN && !soft; ++i)
    if (nd->taint_soft && nd->taint_soft[i]) soft = 1;
  d.soft_active = d.taint_batch && soft;
  return VC_OK;
}

// smallest launch geometry that keeps one node per thread when possible
void choose_geometry(vc_snapshot *s) {
  const int nloc = s->dd.node_end - s->dd.node_begin;
  int ctas = g_sm_count > 0 ? g_sm_count : 148;
  if (g_tun.commit_ctas > 0) ctas = g_tun.commit_ctas;
  int block = 128;
  if (g_tun.commit_threads > 0) block = std::max(128, std::min(256, g_tun.commit_threads / 32 * 32));
  const int per_rank_max = ctas;
  ctas *= std::max(1, s->world);  // one session across `world` GPUs: the node axis is cut over all their CTAs
  ctas = std::max(1, std::min(ctas, (nloc + 31) / 32));  // at least a warp of nodes per CTA
  int npc = (nloc + ctas - 1) / ctas;
  npc = std::max(32, (npc + 31) / 32 * 32);
  // mid-sized clusters on one GPU: four full warps of nodes per CTA (one per SM sub-partition in a sweep) and fewer slots to
  // gather beat three warps on more CTAs (10k nodes: 79 x 128 instead of 105 x 96, +2.7 % at cfg2, +1.7 % at cfg3)
  // (the incremental kernel only: the general kernel keeps one node per thread at its 128-thread blocks)
  const int R0 = s->dims.n_dims, K0 = s->dims.n_kdims;
  const bool samp_ok0 = s->dc.to_find == 0 || (s->world <= 1 && !s->dc.soft_active && (s->all_pure || !s->dc.enable_ecache));
  const bool fast0 = !s->topo_any && !s->dc.nta_on && samp_ok0 && !s->any_nominated && R0 <= 8 && K0 <= VC_MAX_KDIMS && !g_tun.commit_generic;
  if (fast0 && g_tun.commit_ctas <= 0 && s->world <= 1 && npc < 128 && nloc >= 64 * 128) npc = 128;
  ctas = std::max(1, (nloc + npc - 1) / npc);
  if (npc > block) block = std::min(256, (npc + 31) / 32 * 32);
  s->n_cta_total = ctas;
  if (s->world > 1) {  // equal grids on every rank (trailing CTAs may own no node)
    ctas = std::min(per_rank_max, (ctas + s->world - 1) / s->world);
    s->n_cta_total = ctas * s->world;
  }
  s->n_cta = ctas;
  s->npc = npc;
  s->block = block;
  const int R = s->dims.n_dims, K = s->dims.n_kdims;
  // hypernode-level scores change for every node after every placement: per-step full sweeps (k_commit)
  // (Releasing / Pipelined resources alone keep the incremental kernel: its FUT instance)
  // and PreferNoSchedule taints under the TaintToleration batch scorer its SOFT instance
  // and feasible-node sampling its SAMP instance (one GPU, no normalising scorer, no job that needs the error cache)
  // (a session with nominated tasks takes the general kernel: allocate.go:624-634 is implemented there)
  s->fast = fast0;
  if (s->fast) {
    if (g_tun.commit_threads <= 0) s->block = 256;  // 7 worker warps: a run's node states are evaluated two per warp
    size_t rows = 3 * (size_t)R + (s->dc.has_future ? 2 * (size_t)R : 0) + 2 * (size_t)K + 2 + 1;
    s->smem_bytes = ((sizeof(Ctl) + 15) & ~(size_t)15) + ((sizeof(CtlFast) + 15) & ~(size_t)15) + rows * npc * 8 +
                    (size_t)npc * (8 + 4 * 5) + (size_t)s->n_cta_total * (8 + 4 + 4 + 4 + 4) + 64;
    const size_t heap_bytes = (size_t)s->heap_total * sizeof(HeapKey);
    s->heap_in_smem = (heap_bytes <= 96 * 1024 && s->smem_bytes + heap_bytes <= 200 * 1024) ? 1 : 0;
    if (s->heap_in_smem) s->smem_bytes += heap_bytes + 16;
  } else {
    size_t rows = 3 * (size_t)R + (s->dc.has_future ? 2 * (size_t)R : 0) + 2 * (size_t)K + 2;
    s->smem_bytes = ((sizeof(Ctl) + 15) & ~(size_t)15) + rows * npc * 8 + (size_t)npc * (8 + 4 + 4) + 64;
    s->smem_bytes += (size_t)npc * (8 + 4 + 1 + 1) + 32;  // verdict cache + sampling flags
    // hn_score (at most npc * L local hypernodes) + chain_val (at most npc chains); hn_cap is set after this call
    // ... + node -> chain (npc ints) + chain slots (at most npc chains x L)
    if (s->dc.nta_tables) s->smem_bytes += (size_t)npc * (s->hn_L + 1) * 8 + (size_t)npc * 4 + (size_t)npc * s->hn_L * 4 + 64;
  }
}

int free_dense(vc_snapshot *s) {
  if (s->g_final) cudaFree(s->g_final);
  if (s->g_maskw) cudaFree(s->g_maskw);
  s->g_final = nullptr; s->g_maskw = nullptr;
  void *ptrs[] = {s->g_req, s->g_kreq, s->g_knz, s->g_order, s->g_best_score, s->g_has, s->g_class, s->g_stats,
                  s->g_best_node, s->g_cat, s->work_group, s->work_begin, s->work_end, s->group_tasks, s->task_group,
                  s->part_score, s->part_node, s->mask_out, s->score_out, s->best_score, s->best_node};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  s->g_req = s->g_kreq = s->g_knz = s->g_order = s->g_best_score = nullptr;
  s->g_has = nullptr; s->g_class = s->g_stats = s->g_best_node = nullptr; s->g_cat = nullptr;
  s->work_group = s->work_begin = s->work_end = s->group_tasks = s->task_group = nullptr;
  s->part_score = nullptr; s->part_node = nullptr;
  s->mask_out = nullptr; s->score_out = s->best_score = nullptr; s->best_node = nullptr;
  s->dense_ready = false;
  s->matrix_allocated = false;
  return VC_OK;
}

}  // namespace

// =======================================================================================
extern "C" {

int vc_abi_version(void) { return VC_ABI_VERSION; }
const char *vc_last_error(void) { return g_err.c_str(); }

int vc_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return fail(VC_ENODEV, "no CUDA device (%s): libvcalloc has no CPU path", cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(VC_EINVAL, "device %d out of range (%d devices)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (!prop.cooperativeLaunch) return fail(VC_ENODEV, "device lacks cooperative launch");
  g_sm_count = prop.multiProcessorCount;
  g_smem_optin = (int)prop.sharedMemPerBlockOptin;
  g_device = device;
  if (!g_inited) read_tunables();
  g_inited = true;
  return VC_OK;
}

int vc_debug_option(const char *name, int value) {
  if (!name) return fail(VC_EINVAL, "null option name");
  for (const TunName &t : kTunNames)
    if (!std::strcmp(name, t.name)) { g_tun.*(t.field) = value; return VC_OK; }
  return fail(VC_EINVAL, "unknown diagnostic option %s", name);
}

int vc_snapshot_create(const vc_dims *dims, vc_snapshot **out) {
  if (!g_inited) return fail(VC_ENODEV, "vc_init was not called (or failed): no CUDA device bound");
  if (!dims || !out) return fail(VC_EINVAL, "null argument");
  if (dims->n_dims < 2 || dims->n_dims > VC_MAX_DIMS) return fail(VC_EINVAL, "n_dims must be in [2,%d]", VC_MAX_DIMS);
  if (dims->n_kdims < 2 || dims->n_kdims > VC_MAX_KDIMS) return fail(VC_EINVAL, "n_kdims must be in [2,%d]", VC_MAX_KDIMS);
  if (dims->label_words < 1 || dims->label_words > VC_MAX_WORDS || dims->taint_words < 1 || dims->taint_words > VC_MAX_WORDS)
    return fail(VC_EINVAL, "label_words / taint_words must be in [1,%d]", VC_MAX_WORDS);
  if (dims->n_nodes < 0 || dims->n_tasks < 0 || dims->n_jobs < 0 || dims->n_queues < 0 || dims->n_classes < 1)
    return fail(VC_EINVAL, "negative size");
  vc_snapshot *s = new vc_snapshot();
  s->dims = *dims;
  DevDims &d = s->dd;
  d.N = dims->n_nodes; d.T = dims->n_tasks; d.J = dims->n_jobs; d.Q = dims->n_queues; d.C = dims->n_classes;
  d.R = dims->n_dims; d.K = dims->n_kdims; d.Wl = dims->label_words; d.Wt = dims->taint_words; d.NR = dims->n_roles;
  d.Z = dims->n_zones; d.pods_dim = dims->pods_dim;
  d.node_begin = 0; d.node_end = d.N;
  cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
  if (e == cudaSuccess) e = cudaEventCreate(&s->ev2);
  if (e != cudaSuccess) { delete s; return fail(VC_ECUDA, "stream/event create: %s", cudaGetErrorString(e)); }
  *out = s;
  return VC_OK;
}

void vc_snapshot_destroy(vc_snapshot *s) {
  if (!s) return;
  free_dense(s);
  for (int r = 0; r < s->world; ++r)
    if (r != s->rank && s->peer_comm[r]) cudaIpcCloseMemHandle(s->peer_comm[r]);
  if (s->comm) cudaFree(s->comm);
  void *dptrs[] = {s->in.dev, s->cstat, s->w_idle, s->w_used, s->w_pip, s->w_kreq, s->w_knz, s->w_pod_count,
                   s->rep_i32, s->rep_f64, s->rep_heap, s->rep_hn_used, s->rep_placed, s->d_job_alloc, s->hn_score, s->mbox, s->ring, s->d_score_log, s->d_prof, s->d_wait, s->d_dbg, s->d_nominated, s->d_decisions, s->d_visits, s->d_fit, s->d_counters, s->d_bf, s->w_rel, s->d_ev};
  for (void *p : dptrs) if (p) cudaFree(p);
  void *hptrs[] = {s->in.pin, s->h_decisions, s->h_visits, s->h_fit, s->h_counters, s->h_ev, s->delta_pin};
  if (s->delta_dev) cudaFree(s->delta_dev);
  for (void *p : hptrs) if (p) cudaFreeHost(p);
  if (s->ev0) cudaEventDestroy(s->ev0);
  if (s->ev1) cudaEventDestroy(s->ev1);
  if (s->ev2) cudaEventDestroy(s->ev2);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int vc_snapshot_set_topology(vc_snapshot *s, const vc_hypernodes *topo) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  s->uploaded = false;
  if (!topo || !topo->member) {  // no HyperNode objects: the cluster top hypernode alone (tier 1)
    s->has_topo = false;
    s->hn_H = s->hn_L = s->hn_min_tier = 1;
    s->h_member.clear(); s->h_tier.clear(); s->h_parent.clear(); s->h_job_soft.clear();
    return VC_OK;
  }
  const int L = topo->max_tier - topo->min_tier + 1;
  if (topo->n_hypernodes < 1 || L < 1 || L > VC_MAX_TIERS || topo->min_tier < 1)
    return fail(VC_EINVAL, "hypernode table: %d hypernodes, tiers [%d,%d] (at most %d tiers, tier >= 1)", topo->n_hypernodes,
                topo->min_tier, topo->max_tier, VC_MAX_TIERS);
  const size_t N = s->dims.n_nodes;
  for (size_t i = 0; i < (size_t)L * N; ++i)
    if (topo->member[i] < -1 || topo->member[i] >= topo->n_hypernodes) return fail(VC_EINVAL, "hypernode index out of range");
  s->has_topo = true;
  s->hn_H = topo->n_hypernodes; s->hn_L = L; s->hn_min_tier = topo->min_tier;
  s->h_member.assign(topo->member, topo->member + (size_t)L * N);
  const size_t H = topo->n_hypernodes, J = s->dims.n_jobs;
  s->h_tier.clear(); s->h_parent.clear(); s->h_job_soft.clear(); s->h_job_alloc.clear();
  s->h_placed_off.clear(); s->h_placed_node.clear();
  if (topo->tier && topo->parent) {
    s->h_tier.assign(topo->tier, topo->tier + H);
    s->h_parent.assign(topo->parent, topo->parent + H);
    for (size_t h = 0; h < H; ++h) {
      if (s->h_tier[h] < topo->min_tier || s->h_tier[h] > topo->max_tier) return fail(VC_EINVAL, "hypernode %zu: tier outside [min_tier,max_tier]", h);
      if (s->h_parent[h] < -1 || s->h_parent[h] >= (int)H) return fail(VC_EINVAL, "hypernode %zu: bad parent", h);
    }
  }
  if (topo->job_soft) {
    if (!topo->tier || !topo->parent || !topo->job_allocated || !topo->job_placed_off || !topo->job_placed_node)
      return fail(VC_EINVAL, "soft-mode topology jobs need tier, parent, job_allocated and the placed-node lists");
    s->h_job_soft.assign(topo->job_soft, topo->job_soft + J);
    s->h_job_alloc.assign(topo->job_allocated, topo->job_allocated + J);
    s->h_placed_off.assign(topo->job_placed_off, topo->job_placed_off + J + 1);
    s->h_placed_node.assign(topo->job_placed_node, topo->job_placed_node + s->h_placed_off[J]);
    for (size_t j = 0; j < J; ++j)
      if (s->h_job_alloc[j] < -1 || s->h_job_alloc[j] >= (int)H) return fail(VC_EINVAL, "job %zu: bad allocated hypernode", j);
    for (int32_t n : s->h_placed_node)
      if (n < 0 || (size_t)n >= N) return fail(VC_EINVAL, "placed-node list: node index out of range");
  }
  return VC_OK;
}

// ---- one session across the GPUs of a node: CUDA IPC slabs, peer-mapped -----------------------------------------
int vc_comm_create(vc_snapshot *s, int world, int rank, void *handle_out) {
  if (!s || !handle_out) return fail(VC_EINVAL, "null argument");
  if (world < 1 || world > 8 || rank < 0 || rank >= world) return fail(VC_EINVAL, "world %d / rank %d out of range (1..8)", world, rank);
  s->uploaded = false;  // the launch geometry depends on the number of ranks
  s->world = world; s->rank = rank; s->comm_attached = false;
  const size_t T = s->dims.n_tasks;
  const size_t mbox = sizeof(uint4) * MBOX_STRIDE * 2 * 2048, ring = sizeof(uint4) * RING_STRIDE * RING_DEPTH;
  s->comm_mbox_bytes = mbox;
  s->comm_ring_off = (mbox + 255) & ~(size_t)255;
  s->comm_log_off = (s->comm_ring_off + ring + 255) & ~(size_t)255;
  const size_t bytes = s->comm_log_off + (T + 64) * sizeof(uint4);
  s->comm_bytes_all = bytes;
  if (!s->comm || s->comm_bytes < bytes) {
    if (s->comm) cudaFree(s->comm);
    s->comm = nullptr;
    CUDA_TRY(cudaMalloc(&s->comm, bytes));
    s->comm_bytes = bytes;
  }
  CUDA_TRY(cudaMemset(s->comm, 0, s->comm_bytes));
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, s->comm));
  static_assert(sizeof(cudaIpcMemHandle_t) == VC_COMM_HANDLE_BYTES, "IPC handle size");
  std::memcpy(handle_out, &h, sizeof h);
  return VC_OK;
}

int vc_comm_attach(vc_snapshot *s, const void *handles) {
  if (!s || !handles) return fail(VC_EINVAL, "null argument");
  if (!s->comm) return fail(VC_EINVAL, "vc_comm_create must precede vc_comm_attach");
  for (int r = 0; r < s->world; ++r) {
    if (r == s->rank) { s->peer_comm[r] = s->comm; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, reinterpret_cast<const unsigned char *>(handles) + (size_t)r * VC_COMM_HANDLE_BYTES, sizeof h);
    void *ptr = nullptr;
    CUDA_TRY(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    s->peer_comm[r] = reinterpret_cast<unsigned char *>(ptr);
  }
  s->comm_attached = true;
  return VC_OK;
}

int vc_comm_prepare(vc_snapshot *s) {
  if (!s || !s->comm) return fail(VC_EINVAL, "no communication slab (vc_comm_create)");
  CUDA_TRY(cudaMemsetAsync(s->comm, 0, s->comm_bytes_all, s->stream));  // mailbox + ring + score log (its entries are tagged by attempt index)
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return VC_OK;
}

int vc_snapshot_set_shard(vc_snapshot *s, int32_t node_begin, int32_t node_end) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  if (node_begin < 0 || node_end > s->dims.n_nodes || node_begin > node_end || (node_begin % 64) != 0)
    return fail(VC_EINVAL, "shard [%d,%d) invalid (begin must be a multiple of 64)", node_begin, node_end);
  if (s->dd.node_begin == node_begin && s->dd.node_end == node_end) return VC_OK;  // unchanged: the dense-pass tables stay
  s->dd.node_begin = node_begin;
  s->dd.node_end = node_end;
  s->dense_ready = false;
  return VC_OK;
}

int vc_snapshot_upload(vc_snapshot *s, const vc_nodes *nd, const vc_tasks *tk, const vc_classes *cl,
                       const vc_jobs *jb, const vc_queues *qu, const vc_conf *conf) {
  if (!s || !nd || !tk || !cl || !jb || !qu || !conf) return fail(VC_EINVAL, "null argument");
  s->uploaded = false;  // a failed upload must not leave a half-described session runnable
  const double t0 = now_ms();
  const vc_dims &D = s->dims;
  const size_t N = D.n_nodes, T = D.n_tasks, J = D.n_jobs, Q = D.n_queues, C = D.n_classes, R = D.n_dims,
               K = D.n_kdims, Wl = D.label_words, Wt = D.taint_words, NR = D.n_roles, Z = D.n_zones;
  s->conf = *conf;
  // ---- every caller-supplied index is range-checked here, before any session-open logic reads through it ----
  if (conf->n_plugins < 0 || conf->n_plugins > VC_MAX_PLUGINS) return fail(VC_EINVAL, "n_plugins out of range");
  if (J > 0 && jb->role_off[0] != 0) return fail(VC_EINVAL, "role_off[0] must be 0");
  for (size_t j = 0; j < J; ++j) {
    if (jb->role_off[j + 1] < jb->role_off[j] || (size_t)jb->role_off[j + 1] > NR)
      return fail(VC_EINVAL, "job %zu: role_off not monotone / beyond n_roles", j);
    if (jb->queue[j] < -1 || jb->queue[j] >= (int32_t)Q) return fail(VC_EINVAL, "job %zu: bad queue index", j);
  }
  for (size_t t = 0; t < T; ++t) {
    const int32_t j = tk->job[t];
    if (j < 0 || (size_t)j >= J) return fail(VC_EINVAL, "task %zu: bad job index", t);
    if (tk->klass[t] < 0 || (size_t)tk->klass[t] >= C) return fail(VC_EINVAL, "task %zu: bad class index", t);
    if (tk->role[t] < jb->role_off[j] || tk->role[t] >= jb->role_off[j + 1])
      return fail(VC_EINVAL, "task %zu: role row outside its job", t);
  }
  for (size_t j = 0; j < J; ++j) {
    if (jb->flags[j] & VC_JOB_UNSUPPORTED) return fail(VC_EUNSUPPORTED, "job %zu uses hard topology / subjob policy", j);
    if (jb->role_off[j + 1] - jb->role_off[j] > VC_MAX_JOB_ROLES) return fail(VC_EUNSUPPORTED, "job %zu has too many roles", j);
  }
  int rc = build_devconf(s, nd);
  if (rc) return rc;
  const bool tprof = g_tun.prof_upload != 0;
  double tlast = now_ms();
  auto tick = [&](const char *what) {
    if (!tprof) return;
    const double t = now_ms();
    fprintf(stderr, "upload: %-28s %.3f ms\n", what, t - tlast);
    tlast = t;
  };
  tick("devconf (scans node arrays)");

  // ---- host session-open logic ---------------------------------------------------------
  // ssn.TotalResource (framework/session.go:272-274)
  vch::HRes total;
  for (size_t d = 0; d < R; ++d) {
    double acc = 0;
    const double *col = nd->allocatable + d * N;
    for (size_t n = 0; n < N; ++n) acc += col[n];
    total.v[d] = acc;
    if (d >= 2 && N > 0) { total.has |= 1u << d; total.nil = false; }
  }
  for (int d = 0; d < VC_MAX_DIMS; ++d) s->total[d] = total.v[d];
  s->total_has = total.has;
  // drf job shares at open (plugins/drf/drf.go:186-214, :566-578)
  std::vector<double> j_share(J, 0.0);
  if (s->dc.has_drf)
    for (size_t j = 0; j < J; ++j) {
      double res = 0;
      for (size_t d = 0; d < R; ++d) {
        if (d >= 2 && !((total.has >> d) & 1u)) continue;
        if (!(total.v[d] >= vch::kMinRes)) continue;
        double sh = vch::share_of(jb->allocated[d * J + j], total.v[d]);
        if (sh > res) res = sh;
      }
      j_share[j] = res;
    }
  // proportion deserved / share (plugins/proportion/proportion.go:90-264)
  if (s->dc.has_proportion) vch::proportion_open(D, *jb, *qu, total, s->qattr);
  else s->qattr.assign(Q, vch::QAttr());
  // TaskOrderFn order inside each job
  std::vector<int32_t> job_task_off(J + 1, 0), task_order(T);
  for (size_t t = 0; t < T; ++t) {
    if (tk->job[t] < 0 || (size_t)tk->job[t] >= J) return fail(VC_EINVAL, "task %zu: bad job index", t);
    job_task_off[tk->job[t] + 1]++;
  }
  int max_job_tasks = 1;
  for (size_t j = 0; j < J; ++j) {
    max_job_tasks = std::max(max_job_tasks, job_task_off[j + 1]);
    job_task_off[j + 1] += job_task_off[j];
  }
  {
    std::vector<int32_t> fill(job_task_off.begin(), job_task_off.end() - 1);
    for (size_t t = 0; t < T; ++t) task_order[fill[tk->job[t]]++] = (int32_t)t;
    vch::TaskLess less{tk, vch::plugin_enabled(*conf, VC_PLUGIN_PRIORITY, VC_EN_TASK_ORDER)};
    std::vector<int> tmp;
    for (size_t j = 0; j < J; ++j) {
      int b = job_task_off[j], e = job_task_off[j + 1];
      // helpers.CompareTask is transitive only among pods that all carry a numeric name index or all lack one
      // (index order between indexed pods, creation time otherwise): the shortcut is taken for such jobs alone
      bool sorted = true, any_idx = false, any_noidx = false;
      for (int i = b; i < e; ++i) {
        const bool has_idx = tk->pod_index && tk->pod_index[task_order[i]] >= 0;
        any_idx |= has_idx; any_noidx |= !has_idx;
      }
      if (any_idx && any_noidx) sorted = false;
      for (int i = b + 1; i < e && sorted; ++i)
        if (!less(task_order[i - 1], task_order[i])) sorted = false;
      if (sorted) continue;  // a strictly increasing run under a transitive order is its own heap-pop order
      tmp.assign(task_order.begin() + b, task_order.begin() + e);
      vch::go_heap_order(tmp, less);
      std::copy(tmp.begin(), tmp.end(), task_order.begin() + b);
    }
  }
  s->max_job_tasks = max_job_tasks;
  tick("totals, shares, task order");
  // buildAllocateContext (allocate.go:142-206): jobs that enter the per-queue PQs, in JobOrderFn order
  std::vector<uint32_t> j_rank(J);
  {
    std::vector<int> idx(J);
    for (size_t j = 0; j < J; ++j) idx[j] = (int)j;
    std::sort(idx.begin(), idx.end(), [&](int a, int b) {
      if (jb->creation_ts[a] != jb->creation_ts[b]) return jb->creation_ts[a] < jb->creation_ts[b];
      return jb->uid_rank[a] < jb->uid_rank[b];
    });
    for (size_t r = 0; r < J; ++r) j_rank[idx[r]] = (uint32_t)r;
  }
  std::vector<uint32_t> q_rank(Q);
  {
    std::vector<int> idx(Q);
    for (size_t q = 0; q < Q; ++q) idx[q] = (int)q;
    std::sort(idx.begin(), idx.end(), [&](int a, int b) {
      if (qu->creation_ts[a] != qu->creation_ts[b]) return qu->creation_ts[a] < qu->creation_ts[b];
      return qu->uid_rank[a] < qu->uid_rank[b];
    });
    for (size_t r = 0; r < Q; ++r) q_rank[idx[r]] = (uint32_t)r;
  }
  std::vector<std::vector<int>> qlists(Q);
  for (size_t j = 0; j < J; ++j) {
    if ((jb->flags[j] & VC_JOB_PENDING_PHASE) && conf->enqueue_action_enabled) continue;
    if (!vch::job_valid(*conf, *jb, (int)j)) continue;
    int q = jb->queue[j];
    if (q < 0) continue;
    if ((size_t)q >= Q) return fail(VC_EINVAL, "job %zu: bad queue index", j);
    if (job_task_off[j + 1] == job_task_off[j]) continue;
    qlists[q].push_back((int)j);
  }
  auto job_less = [&](int l, int r) {  // ssn.JobOrderFn, session_plugins.go:660-683
    for (int i = 0; i < conf->n_plugins; ++i) {
      const vc_plugin_option &p = conf->plugins[i];
      if (!(p.enabled & VC_EN_JOB_ORDER)) continue;
      int c = 0;
      switch (p.plugin) {
        case VC_PLUGIN_PRIORITY: c = jb->priority[l] > jb->priority[r] ? -1 : (jb->priority[l] < jb->priority[r] ? 1 : 0); break;
        case VC_PLUGIN_GANG: {
          bool lr = jb->ready_num[l] + jb->pending_besteffort[l] >= jb->min_available[l];
          bool rr = jb->ready_num[r] + jb->pending_besteffort[r] >= jb->min_available[r];
          c = (lr && rr) ? 0 : (lr ? 1 : (rr ? -1 : 0));
          break;
        }
        case VC_PLUGIN_DRF: c = j_share[l] == j_share[r] ? 0 : (j_share[l] < j_share[r] ? -1 : 1); break;
        case VC_PLUGIN_TDM: {
          bool lp = jb->flags[l] & VC_JOB_PREEMPTABLE, rp = jb->flags[r] & VC_JOB_PREEMPTABLE;
          c = lp == rp ? 0 : (!lp ? -1 : 1);
          break;
        }
        default: break;
      }
      if (c != 0) return c < 0;
    }
    return j_rank[l] < j_rank[r];
  };
  std::vector<int32_t> qjobs_off(Q + 1, 0), qjobs;
  for (size_t q = 0; q < Q; ++q) {
    std::sort(qlists[q].begin(), qlists[q].end(), job_less);
    qjobs_off[q + 1] = qjobs_off[q] + (int32_t)qlists[q].size();
    qjobs.insert(qjobs.end(), qlists[q].begin(), qlists[q].end());
  }
  tick("job / queue order");
  // (class, request) groups: tasks of one pod template share their whole verdict / score row
  std::vector<int32_t> group_of(T);
  {
    // (1) one 64-bit hash per task, built in dimension-major passes (the inputs are dimension-major: sequential reads)
    auto mix = [](uint64_t h, uint64_t v) {
      h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
      h *= 0xff51afd7ed558ccdull;
      return h ^ (h >> 33);
    };
    auto bits = [](double x) { uint64_t u; std::memcpy(&u, &x, 8); return u; };
    std::vector<uint64_t> hsh(T, 0x243f6a8885a308d3ull);
    std::vector<uint32_t> has_x(T);
    for (size_t t = 0; t < T; ++t) {
      has_x[t] = tk->req_has[t] | ((s->topo_any && s->h_job_soft[tk->job[t]]) ? VC_HAS_TOPO_TASK : 0u);
      hsh[t] = mix(mix(hsh[t], (uint32_t)tk->klass[t]), has_x[t]);
    }
    for (size_t d = 0; d < R; ++d) { const double *col = tk->resreq + d * T; for (size_t t = 0; t < T; ++t) hsh[t] = mix(hsh[t], bits(col[t])); }
    for (size_t k = 0; k < K; ++k) { const double *col = tk->k8s_req + k * T; for (size_t t = 0; t < T; ++t) hsh[t] = mix(hsh[t], bits(col[t])); }
    for (size_t k = 0; k < 2; ++k) { const double *col = tk->k8s_nonzero_req + k * T; for (size_t t = 0; t < T; ++t) hsh[t] = mix(hsh[t], bits(col[t])); }
    // (2) tentative groups by hash (tasks of a job are adjacent and usually share their record)
    std::unordered_map<uint64_t, int> index;
    index.reserve(1024);
    s->group_rep.clear();
    for (size_t t = 0; t < T; ++t) {
      if (t > 0 && hsh[t] == hsh[t - 1]) { group_of[t] = group_of[t - 1]; continue; }
      auto it = index.find(hsh[t]);
      if (it == index.end()) {
        it = index.emplace(hsh[t], (int)s->group_rep.size()).first;
        s->group_rep.push_back((int32_t)t);
      }
      group_of[t] = it->second;
    }
    // (3) exact verification against the group representative, again in dimension-major passes; a hash collision
    //     (never observed) falls back to exact keys
    bool exact = true;
    const std::vector<int32_t> &rep = s->group_rep;
    for (size_t t = 0; t < T && exact; ++t) {
      const int r = rep[group_of[t]];
      if (tk->klass[t] != tk->klass[r] || has_x[t] != has_x[r]) exact = false;
    }
    auto verify = [&](const double *col) {
      for (size_t t = 0; t < T; ++t)
        if (bits(col[t]) != bits(col[rep[group_of[t]]])) return false;
      return true;
    };
    for (size_t d = 0; d < R && exact; ++d) exact = verify(tk->resreq + d * T);
    for (size_t k = 0; k < K && exact; ++k) exact = verify(tk->k8s_req + k * T);
    for (size_t k = 0; k < 2 && exact; ++k) exact = verify(tk->k8s_nonzero_req + k * T);
    if (!exact) {
      std::unordered_map<std::string, int> sindex;
      s->group_rep.clear();
      std::string key;
      for (size_t t = 0; t < T; ++t) {
        key.clear();
        key.append(reinterpret_cast<const char *>(&tk->klass[t]), 4);
        key.append(reinterpret_cast<const char *>(&has_x[t]), 4);
        for (size_t d = 0; d < R; ++d) key.append(reinterpret_cast<const char *>(&tk->resreq[d * T + t]), 8);
        for (size_t k = 0; k < K; ++k) key.append(reinterpret_cast<const char *>(&tk->k8s_req[k * T + t]), 8);
        for (size_t k = 0; k < 2; ++k) key.append(reinterpret_cast<const char *>(&tk->k8s_nonzero_req[k * T + t]), 8);
        auto it = sindex.find(key);
        if (it == sindex.end()) {
          it = sindex.emplace(key, (int)s->group_rep.size()).first;
          s->group_rep.push_back((int32_t)t);
        }
        group_of[t] = it->second;
      }
    }
  }
  tick("group dedup");
  const size_t NG = s->group_rep.size();
  s->n_groups = (int)NG;
  s->h_group_of = group_of;
  std::vector<double> g_req(R * NG), g_kreq(K * NG), g_knz(2 * NG);
  std::vector<uint32_t> g_has(NG);
  std::vector<int32_t> g_class(NG);
  for (size_t g = 0; g < NG; ++g) {
    const int t = s->group_rep[g];
    for (size_t d = 0; d < R; ++d) g_req[d * NG + g] = tk->resreq[d * T + t];
    for (size_t k = 0; k < K; ++k) g_kreq[k * NG + g] = tk->k8s_req[k * T + t];
    for (size_t k = 0; k < 2; ++k) g_knz[k * NG + g] = tk->k8s_nonzero_req[k * T + t];
    g_has[g] = tk->req_has[t] | ((s->topo_any && s->h_job_soft[tk->job[t]]) ? VC_HAS_TOPO_TASK : 0u);
    g_class[g] = tk->klass[t];
  }
  // per position of task_order: {task, group, role row}; a job is 'pure' when each named role maps to
  // one group (then the role-level predicate-error cache cannot change any verdict)
  std::vector<int32_t> tmeta(4 * T);
  std::vector<uint32_t> j_flags_x(jb->flags, jb->flags + J);
  {
    std::vector<int32_t> role_group(NR, -1);
    std::vector<uint8_t> impure(J, 0);
    for (size_t pos = 0; pos < T; ++pos) {
      const int t = task_order[pos];
      tmeta[4 * pos + 0] = t; tmeta[4 * pos + 1] = group_of[t]; tmeta[4 * pos + 2] = tk->role[t]; tmeta[4 * pos + 3] = 0;
    }
    for (size_t t = 0; t < T; ++t) {
      const int r = tk->role[t];
      if (r < 0 || (size_t)r >= NR) return fail(VC_EINVAL, "task %zu: bad role row", t);
      if (jb->role_flags[r] & VC_ROLE_EMPTY_NAME) continue;
      if (role_group[r] < 0) role_group[r] = group_of[t];
      else if (role_group[r] != group_of[t]) impure[tk->job[t]] = 1;
    }
    s->all_pure = true;
    for (size_t j = 0; j < J; ++j) {
      if (!impure[j]) j_flags_x[j] |= VC_JOBX_PURE;
      else s->all_pure = false;
    }
  }
  // role pending counts incl. the tasks in scope (job_info.go:936-939)
  std::vector<int32_t> r_pending(NR, 0);
  for (size_t r = 0; r < NR; ++r) r_pending[r] = jb->role_pending_other ? jb->role_pending_other[r] : 0;
  for (size_t t = 0; t < T; ++t) {
    int r = tk->role[t], j = tk->job[t];
    if (r < jb->role_off[j] || r >= jb->role_off[j + 1]) return fail(VC_EINVAL, "task %zu: role row outside its job", t);
    r_pending[r] += 1;
  }
  // queue arrays for the device
  std::vector<double> q_des(R * Q, 0.0), q_alloc(R * Q, 0.0), q_share(Q, 0.0);
  std::vector<uint32_t> q_des_has(Q, 0), q_alloc_has(Q, 0), q_flags2(Q, 0);
  for (size_t q = 0; q < Q; ++q) {
    const vch::QAttr &a = s->qattr[q];
    if (!a.exists) continue;
    for (size_t d = 0; d < R; ++d) { q_des[d * Q + q] = a.deserved.v[d]; q_alloc[d * Q + q] = a.allocated.v[d]; }
    q_des_has[q] = a.deserved.has;
    q_alloc_has[q] = a.allocated.has;
    q_flags2[q] = 1u | (a.allocated.nil ? 2u : 0u);
    q_share[q] = a.share;
  }

  // packed read-only records for the fast commit kernel (one coalesced access per record)
  std::vector<JobStatic> jstat(J);
  for (size_t j = 0; j < J; ++j) {
    JobStatic &r = jstat[j];
    std::memset(&r, 0, sizeof r);
    r.min_available = jb->min_available[j]; r.n_tasks_total = jb->n_tasks_total[j];
    r.pending_besteffort = jb->pending_besteffort[j]; r.task_min_total = jb->task_min_total[j];
    r.role_off = jb->role_off[j]; r.n_roles = jb->role_off[j + 1] - jb->role_off[j];
    r.priority = jb->priority[j]; r.flags = j_flags_x[j]; r.rank = j_rank[j];
    r.task_off = job_task_off[j]; r.task_end = job_task_off[j + 1]; r.queue = jb->queue[j];
  }
  // packed JobOrderFn keys (see HeapKey): comparators in plugin order, MSB first
  {
    std::vector<int> pre_c, post_c;  // 0 priority, 1 gang readiness, 2 tdm preemptable
    bool share_on = false;
    for (int i = 0; i < conf->n_plugins; ++i) {
      const vc_plugin_option &po = conf->plugins[i];
      if (!(po.enabled & VC_EN_JOB_ORDER)) continue;
      std::vector<int> &dst = share_on ? post_c : pre_c;
      if (po.plugin == VC_PLUGIN_PRIORITY) dst.push_back(0);
      else if (po.plugin == VC_PLUGIN_GANG) dst.push_back(1);
      else if (po.plugin == VC_PLUGIN_TDM) dst.push_back(2);
      else if (po.plugin == VC_PLUGIN_DRF) share_on = true;
    }
    std::vector<int32_t> prios(jb->priority, jb->priority + J);
    std::sort(prios.begin(), prios.end(), std::greater<int32_t>());
    prios.erase(std::unique(prios.begin(), prios.end()), prios.end());
    if (prios.size() >= (1u << 24)) return fail(VC_EUNSUPPORTED, "too many distinct job priorities");
    s->fast_ready_word = 0; s->fast_ready_shift = 0; s->fast_share_on = share_on ? 1 : 0;
    for (size_t j = 0; j < J; ++j) {
      const uint64_t prio_rank = (uint64_t)(std::lower_bound(prios.begin(), prios.end(), jb->priority[j], std::greater<int32_t>()) - prios.begin());
      auto pack = [&](const std::vector<int> &comps, uint64_t low, int low_bits, int word) {
        uint64_t v = low;
        int shift = low_bits;
        for (int k = (int)comps.size() - 1; k >= 0; --k) {
          const int kind = comps[k];
          if (kind == 0) { v |= prio_rank << shift; shift += 24; }
          else if (kind == 1) { s->fast_ready_word = word; s->fast_ready_shift = shift; shift += 1; }
          else { v |= (uint64_t)((jb->flags[j] & VC_JOB_PREEMPTABLE) ? 1 : 0) << shift; shift += 1; }
        }
        return v;
      };
      if (share_on) {
        jstat[j].key_pre = pack(pre_c, 0, 0, 1);
        jstat[j].key_post = pack(post_c, j_rank[j], 32, 2);
      } else {
        jstat[j].key_pre = pack(pre_c, j_rank[j], 32, 1);
        jstat[j].key_post = 0;
      }
    }
  }
  // per-queue heap capacity: only jobs that can be Ready with tasks left are ever re-pushed (allocate.go:334-336)
  std::vector<int32_t> heap_off(Q + 1, 0);
  const bool gang_ready = vch::plugin_enabled(*conf, VC_PLUGIN_GANG, VC_EN_JOB_READY);
  for (size_t q = 0; q < Q; ++q) {
    int cnt = 0;
    for (int k = qjobs_off[q]; k < qjobs_off[q + 1]; ++k) {
      const int j = qjobs[k];
      const int scope = job_task_off[j + 1] - job_task_off[j];
      // with gang's JobReadyFn: Ready with a task left needs ready + bestEffort + (scope - 1) >= minAvailable;
      // without it ssn.JobReady is always true and every job with a second task comes back
      if (gang_ready ? (jb->ready_num[j] + jb->pending_besteffort[j] + scope > jb->min_available[j]) : (scope >= 2)) ++cnt;
    }
    heap_off[q + 1] = heap_off[q] + cnt;
  }
  s->heap_total = heap_off[Q];
  std::vector<RoleStatic> rstat(NR);
  for (size_t r = 0; r < NR; ++r) { rstat[r].min = jb->role_min[r]; rstat[r].flags = jb->role_flags[r]; }
  std::vector<QueueStatic> qstat(Q);
  for (size_t q = 0; q < Q; ++q) {
    QueueStatic &r = qstat[q];
    std::memset(&r, 0, sizeof r);
    r.prio = qu->priority[q]; r.rank = q_rank[q]; r.flags = qu->flags[q]; r.des_has = q_des_has[q];
    for (size_t d = 0; d < R && d < FAST_R; ++d) r.des[d] = q_des[d * Q + q];
  }

  // nominated nodes of the pending tasks (vc_snapshot_set_nominated): range check, device copy
  s->any_nominated = false;
  if (!s->h_nominated.empty()) {
    if (s->h_nominated.size() != T) return fail(VC_EINVAL, "nominated-node list: %zu entries for %zu tasks", s->h_nominated.size(), T);
    for (size_t t = 0; t < T; ++t) {
      if (s->h_nominated[t] >= (int32_t)N) return fail(VC_EINVAL, "task %zu: nominated node %d out of range", t, s->h_nominated[t]);
      if (s->h_nominated[t] >= 0) s->any_nominated = true;
    }
    if (s->any_nominated) {
      if (T > s->d_nominated_cap) {
        if (s->d_nominated) cudaFree(s->d_nominated);
        s->d_nominated = nullptr;
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->d_nominated), T * 4));
        s->d_nominated_cap = T;
      }
      CUDA_TRY(cudaMemcpyAsync(s->d_nominated, s->h_nominated.data(), T * 4, cudaMemcpyHostToDevice, s->stream));
    }
  }
  // network-topology-aware: hyperNodeResourceCache at open (network_topology_aware.go:106-125) and, for the
  // commit kernel, the hypernodes each CTA's node slice belongs to
  choose_geometry(s);
  if (s->n_cta_total > 2048) return fail(VC_EUNSUPPORTED, "too many CTAs (%d)", s->n_cta_total);
  if (s->world > 1 && !s->fast)
    return fail(VC_EUNSUPPORTED, "one session across GPUs runs on the incremental commit kernel only (no topology plugin, "
                                 "no feasible-node sampling)");
  if (s->dc.to_find > 0 && (s->npc + s->block - 1) / s->block > 4)
    return fail(VC_EUNSUPPORTED, "feasible-node sampling: more than 4 node rows per CTA (%d nodes per CTA)", s->npc);
  std::vector<int32_t> hn_member, hn_slot, cta_hn_off, cta_hn, node_chain, cta_chain_off, cta_chain;
  std::vector<double> hn_alloc, hn_used0;
  s->hn_cap = 1;
  s->chain_cap = 1;
  std::vector<int32_t> hn_up, job_soft32, placed_off, placed0, placed_n0;
  s->placed_total = 0;
  if (s->topo_any) {
    // ancestor (Parent chain, the hypernode itself included) of every hypernode at every tier level
    const size_t L = s->hn_L, H = s->hn_H;
    hn_up.assign(L * H, -1);
    for (size_t h = 0; h < H; ++h) {
      int a = (int)h;
      for (int guard = 0; a >= 0 && guard < VC_MAX_TIERS + 2; ++guard) {
        const size_t l = (size_t)(s->h_tier[a] - s->hn_min_tier);
        if (hn_up[l * H + h] < 0) hn_up[l * H + h] = a;
        a = s->h_parent[a];
      }
    }
    // values networkTopologyAwareScore can return (network_topology_aware.go:716-756), ascending
    std::vector<double> vals{0.0, 1.0};
    const int min_t = s->hn_min_tier, max_t = s->hn_min_tier + s->hn_L - 1;
    for (int tier = min_t; tier <= max_t; ++tier)
      vals.push_back(min_t == max_t ? 1.0 : (double)(max_t - tier) / (double)(max_t - min_t));
    std::sort(vals.begin(), vals.end());
    vals.erase(std::unique(vals.begin(), vals.end()), vals.end());
    s->topo_nval = (int)vals.size();
    for (size_t i = 0; i < vals.size(); ++i) s->topo_val[i] = vals[i];
    // per-job lists of nodes that hold a task of the job: room for the tasks in scope on top of those at open
    job_soft32.assign(J, 0);
    placed_off.assign(J + 1, 0);
    placed_n0.assign(J, 0);
    for (size_t j = 0; j < J; ++j) {
      job_soft32[j] = s->h_job_soft[j];
      const int n0 = s->h_job_soft[j] ? s->h_placed_off[j + 1] - s->h_placed_off[j] : 0;
      placed_n0[j] = n0;
      placed_off[j + 1] = placed_off[j] + (s->h_job_soft[j] ? n0 + (job_task_off[j + 1] - job_task_off[j]) : 0);
    }
    s->placed_total = (size_t)placed_off[J];
    placed0.assign(std::max<size_t>(s->placed_total, 1), 0);
    for (size_t j = 0; j < J; ++j)
      for (int k = 0; k < placed_n0[j]; ++k) placed0[placed_off[j] + k] = s->h_placed_node[s->h_placed_off[j] + k];
  }
  if (s->dc.nta_tables) {
    const size_t L = s->hn_L, H = s->hn_H;
    if (s->has_topo) hn_member = s->h_member;
    else hn_member.assign(L * N, 0);
    hn_alloc.assign(R * H, 0.0);
    hn_used0.assign(R * H, 0.0);
    for (size_t l = 0; l < L; ++l)
      for (size_t n = 0; n < N; ++n) {
        const int h = hn_member[l * N + n];
        if (h < 0) continue;
        for (size_t d = 0; d < R; ++d) {
          hn_alloc[d * H + h] += nd->allocatable[d * N + n];
          hn_used0[d * H + h] += nd->used[d * N + n];
        }
      }
    hn_slot.assign(L * N, -1);
    cta_hn_off.assign(s->n_cta + 1, 0);
    std::unordered_map<int, int> local;
    for (int cta = 0; cta < s->n_cta; ++cta) {
      local.clear();
      const size_t nb = (size_t)cta * s->npc, ne = std::min(N, nb + (size_t)s->npc);
      for (size_t n = nb; n < ne; ++n)
        for (size_t l = 0; l < L; ++l) {
          const int h = hn_member[l * N + n];
          if (h < 0) continue;
          auto it = local.find(h);
          if (it == local.end()) {
            it = local.emplace(h, (int)local.size()).first;
            cta_hn.push_back(h);
          }
          hn_slot[l * N + n] = it->second;
        }
      cta_hn_off[cta + 1] = (int32_t)cta_hn.size();
      s->hn_cap = std::max<int>(s->hn_cap, (int)local.size());
    }
    // distinct per-tier slot tuples ("chains") among each CTA's nodes: the plugin's normal-pod score is one value
    // per chain and step
    node_chain.assign(N, 0);
    cta_chain_off.assign(s->n_cta + 1, 0);
    std::unordered_map<std::string, int> chains;
    std::string key;
    for (int cta = 0; cta < s->n_cta; ++cta) {
      chains.clear();
      const size_t nb = (size_t)cta * s->npc, ne = std::min(N, nb + (size_t)s->npc);
      for (size_t n = nb; n < ne; ++n) {
        key.clear();
        for (size_t l = 0; l < L; ++l) key.append(reinterpret_cast<const char *>(&hn_slot[l * N + n]), 4);
        auto it = chains.find(key);
        if (it == chains.end()) {
          it = chains.emplace(key, (int)chains.size()).first;
          for (size_t l = 0; l < L; ++l) cta_chain.push_back(hn_slot[l * N + n]);
        }
        node_chain[n] = it->second;
      }
      cta_chain_off[cta + 1] = cta_chain_off[cta] + (int32_t)chains.size();
      s->chain_cap = std::max<int>(s->chain_cap, (int)chains.size());
    }
    s->hn_smem = (!s->fast && s->hn_cap <= 96) ? 1 : 0;
    if (s->hn_smem) s->smem_bytes += 3 * R * (size_t)s->hn_cap * 8 + R * (size_t)s->hn_cap + (size_t)s->hn_cap * 4 + 64;
  }

  tick("records, heap sizes, topology");
  // ---- plan + stage + one H2D copy ------------------------------------------------------
  for (int pass = 0; pass < 2; ++pass) {
    const bool plan = pass == 0;
    if (plan) s->in.used = 0;
    put(s, s->n_alloc, nd->allocatable, R * N, plan); put(s, s->n_idle, nd->idle, R * N, plan);
    put(s, s->n_used, nd->used, R * N, plan); put(s, s->n_rel, nd->releasing, R * N, plan);
    put(s, s->n_pip, nd->pipelined, R * N, plan); put(s, s->n_kalloc, nd->k8s_allocatable, K * N, plan);
    put(s, s->n_kreq, nd->k8s_requested, K * N, plan); put(s, s->n_knz, nd->k8s_nonzero_requested, 2 * N, plan);
    put(s, s->n_max_tasks, nd->max_tasks, N, plan); put(s, s->n_pod_count, nd->pod_count, N, plan);
    put(s, s->n_zone, nd->revocable_zone, N, plan); put(s, s->n_labels, nd->label_bits, Wl * N, plan);
    put(s, s->n_thard, nd->taint_hard, Wt * N, plan); put(s, s->n_tsoft, nd->taint_soft, Wt * N, plan);
    put(s, s->n_flags, nd->flags, N, plan); put(s, s->zone_active, nd->zone_active, std::max<size_t>(Z, 1), plan);
    put(s, s->t_req, tk->resreq, R * T, plan); put(s, s->t_kreq, tk->k8s_req, K * T, plan);
    put(s, s->t_knz, tk->k8s_nonzero_req, 2 * T, plan); put(s, s->t_has, tk->req_has, T, plan);
    put(s, s->t_class, tk->klass, T, plan); put(s, s->t_role, tk->role, T, plan); put(s, s->t_job, tk->job, T, plan);
    put(s, s->c_sel, cl->selector, C * Wl, plan); put(s, s->c_aff, cl->affinity, C * VC_MAX_TERMS * Wl, plan);
    put(s, s->c_tolh, cl->tolerated_hard, C * Wt, plan); put(s, s->c_tols, cl->tolerated_soft, C * Wt, plan);
    put(s, s->c_pref, cl->preferred, C * VC_MAX_TERMS * Wl, plan); put(s, s->c_naff, cl->n_affinity, C, plan);
    put(s, s->c_npref, cl->n_preferred, C, plan); put(s, s->c_prefw, cl->preferred_weight, C * VC_MAX_TERMS, plan);
    put(s, s->c_flags, cl->flags, C, plan);
    put(s, s->j_queue, jb->queue, J, plan); put(s, s->j_min, jb->min_available, J, plan);
    put(s, s->j_ntasks, jb->n_tasks_total, J, plan); put(s, s->j_pbe, jb->pending_besteffort, J, plan);
    put(s, s->j_taskmintotal, jb->task_min_total, J, plan); put(s, s->j_roleoff, jb->role_off, J + 1, plan);
    put(s, s->j_prio, jb->priority, J, plan); put(s, s->j_ready0, jb->ready_num, J, plan);
    put(s, s->j_waiting0, jb->waiting_num, J, plan); put(s, s->j_flags, j_flags_x.data(), J, plan);
    put(s, s->j_rank, j_rank.data(), J, plan); put(s, s->j_alloc0, jb->allocated, R * J, plan);
    put(s, s->j_share0, j_share.data(), J, plan);
    put(s, s->r_min, jb->role_min, NR, plan); put(s, s->r_occ0, jb->role_occupied, NR, plan);
    put(s, s->r_pip0, jb->role_pipelined, NR, plan); put(s, s->r_pending0, r_pending.data(), NR, plan);
    put(s, s->r_flags, jb->role_flags, NR, plan);
    put(s, s->q_prio, qu->priority, Q, plan); put(s, s->q_rank, q_rank.data(), Q, plan);
    put(s, s->q_flags, qu->flags, Q, plan); put(s, s->q_alloc_has0, q_alloc_has.data(), Q, plan);
    put(s, s->q_des_has, q_des_has.data(), Q, plan); put(s, s->q_flags2, q_flags2.data(), Q, plan);
    put(s, s->q_alloc0, q_alloc.data(), R * Q, plan); put(s, s->q_des, q_des.data(), R * Q, plan);
    put(s, s->q_share0, q_share.data(), Q, plan);
    put(s, s->qjobs_off, qjobs_off.data(), Q + 1, plan); put(s, s->qjobs, qjobs.data(), qjobs.size(), plan);
    put(s, s->task_order, task_order.data(), T, plan); put(s, s->job_task_off, job_task_off.data(), J + 1, plan);
    put(s, s->tmeta, tmeta.data(), 4 * T, plan);
    put(s, s->sg_req, g_req.data(), R * NG, plan); put(s, s->sg_kreq, g_kreq.data(), K * NG, plan);
    put(s, s->sg_knz, g_knz.data(), 2 * NG, plan); put(s, s->sg_has, g_has.data(), NG, plan);
    put(s, s->sg_class, g_class.data(), NG, plan);
    put(s, s->s_jstat, jstat.data(), J, plan); put(s, s->s_rstat, rstat.data(), NR, plan);
    put(s, s->s_qstat, qstat.data(), Q, plan);
    put(s, s->s_heap_off, heap_off.data(), Q + 1, plan);
    put(s, s->hn_member, hn_member.data(), hn_member.size(), plan); put(s, s->hn_slot, hn_slot.data(), hn_slot.size(), plan);
    put(s, s->cta_hn_off, cta_hn_off.data(), cta_hn_off.size(), plan); put(s, s->cta_hn, cta_hn.data(), cta_hn.size(), plan);
    put(s, s->hn_alloc, hn_alloc.data(), hn_alloc.size(), plan); put(s, s->hn_used0, hn_used0.data(), hn_used0.size(), plan);
    put(s, s->node_chain, node_chain.data(), node_chain.size(), plan); put(s, s->cta_chain_off, cta_chain_off.data(), cta_chain_off.size(), plan);
    put(s, s->cta_chain, cta_chain.data(), cta_chain.size(), plan);
    put(s, s->hn_up, hn_up.data(), hn_up.size(), plan); put(s, s->hn_tier_s, s->h_tier.data(), s->topo_any ? s->h_tier.size() : 0, plan);
    put(s, s->hn_parent_s, s->h_parent.data(), s->topo_any ? s->h_parent.size() : 0, plan);
    put(s, s->job_soft_s, job_soft32.data(), job_soft32.size(), plan);
    put(s, s->job_alloc0_s, s->h_job_alloc.data(), s->topo_any ? s->h_job_alloc.size() : 0, plan);
    put(s, s->placed_off_s, placed_off.data(), placed_off.size(), plan); put(s, s->placed0_s, placed0.data(), placed0.size(), plan);
    put(s, s->placed_n0_s, placed_n0.data(), placed_n0.size(), plan);
    if (plan) {
      size_t need = (s->in.used + 255) & ~(size_t)255;
      if (need > s->in.cap) {
        if (s->in.dev) cudaFree(s->in.dev);
        if (s->in.pin) cudaFreeHost(s->in.pin);
        s->in.dev = s->in.pin = nullptr;
        CUDA_TRY(cudaMalloc(&s->in.dev, need));
        CUDA_TRY(cudaMallocHost(&s->in.pin, need));
        s->in.cap = need;
      }
    }
  }
  tick("staging memcpy");
  CUDA_TRY(cudaEventRecord(s->ev0, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->in.dev, s->in.pin, s->in.used, cudaMemcpyHostToDevice, s->stream));
  s->h2d_bytes = (int64_t)s->in.used;

  // ---- device-only buffers --------------------------------------------------------------
  auto ensure = [&](auto *&ptr, size_t bytes) -> int {
    if (ptr) return VC_OK;
    void *q = nullptr;
    CUDA_TRY(cudaMalloc(&q, std::max<size_t>(bytes, 16)));
    ptr = reinterpret_cast<std::remove_reference_t<decltype(ptr)>>(q);
    return VC_OK;
  };
  if ((rc = ensure(s->cstat, C * N * 4))) return rc;
  if ((rc = ensure(s->w_idle, R * N * 8)) || (rc = ensure(s->w_used, R * N * 8)) || (rc = ensure(s->w_pip, R * N * 8)) ||
      (rc = ensure(s->w_kreq, K * N * 8)) || (rc = ensure(s->w_knz, 2 * N * 8)) || (rc = ensure(s->w_pod_count, N * 4)))
    return rc;
  // K0
  K0Params k0;
  k0.d = s->dd; k0.c = s->dc;
  k0.labels = s->n_labels.d(s->in); k0.thard = s->n_thard.d(s->in); k0.tsoft = s->n_tsoft.d(s->in);
  k0.nflags = s->n_flags.d(s->in); k0.zone = s->n_zone.d(s->in); k0.zone_active = s->zone_active.d(s->in);
  k0.c_sel = s->c_sel.d(s->in); k0.c_aff = s->c_aff.d(s->in); k0.c_tolh = s->c_tolh.d(s->in);
  k0.c_tols = s->c_tols.d(s->in); k0.c_pref = s->c_pref.d(s->in); k0.c_naff = s->c_naff.d(s->in);
  k0.c_npref = s->c_npref.d(s->in); k0.c_prefw = s->c_prefw.d(s->in); k0.c_flags = s->c_flags.d(s->in);
  k0.cstat = s->cstat;
  if (N > 0) {
    dim3 grid((unsigned)((N + 255) / 256), (unsigned)C);
    k_class_static<<<grid, 256, 0, s->stream>>>(k0);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaEventRecord(s->ev1, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  tick("H2D + K0 + sync");
  s->uploaded = true;
  s->dense_ready = false;
  // milli-units / bytes / counts are integers by construction (Quantity.MilliValue / Value); when that holds for the
  // rows and every request, m placements leave exactly row -/+ m * request: the commit kernel may cover a run of
  // placements on one node with one publication and k_backfill may run ahead m steps
  s->rows_integral = vch::runs_exact(R, N, T, {nd->idle, nd->used}, {tk->resreq}) &&
                     vch::future_rows_exact(R, N, T, nd->idle, nd->releasing, nd->pipelined, tk->resreq) &&
                     vch::runs_exact(K, N, T, {nd->k8s_requested}, {tk->k8s_req}) &&
                     vch::runs_exact(2, N, T, {nd->k8s_nonzero_requested}, {tk->k8s_nonzero_req});
  tick("integrality scan");
  s->alloc_ran = false; s->bf_ran = false;
  s->last_idx_cur = s->dc.last_idx0;
  s->last_dec.clear(); s->last_vis.clear();
  s->es_built = false;
  {  // what the preempt / reclaim actions read of the opening session
    vch::EvictKeep &k = s->ek;
    k.j_queue.assign(jb->queue, jb->queue + J); k.j_min.assign(jb->min_available, jb->min_available + J);
    k.j_prio.assign(jb->priority, jb->priority + J); k.j_ntasks.assign(jb->n_tasks_total, jb->n_tasks_total + J);
    k.j_ready0.assign(jb->ready_num, jb->ready_num + J); k.j_waiting0.assign(jb->waiting_num, jb->waiting_num + J);
    k.j_pbe.assign(jb->pending_besteffort, jb->pending_besteffort + J);
    k.j_taskmintotal.assign(jb->task_min_total, jb->task_min_total + J);
    k.j_roleoff.assign(jb->role_off, jb->role_off + J + 1);
    k.j_flags.assign(jb->flags, jb->flags + J); k.j_rank = j_rank;
    k.j_valid.resize(J);
    for (size_t j = 0; j < J; ++j) k.j_valid[j] = vch::job_valid(*conf, *jb, (int)j) ? 1 : 0;
    k.j_alloc0.assign(jb->allocated, jb->allocated + R * J);
    k.r_min.assign(jb->role_min, jb->role_min + NR); k.r_occ0.assign(jb->role_occupied, jb->role_occupied + NR);
    k.r_pip0.assign(jb->role_pipelined, jb->role_pipelined + NR); k.r_flags.assign(jb->role_flags, jb->role_flags + NR);
    k.q_prio.assign(qu->priority, qu->priority + Q); k.q_rank = q_rank; k.q_flags.assign(qu->flags, qu->flags + Q);
    k.t_job.assign(tk->job, tk->job + T); k.t_role.assign(tk->role, tk->role + T);
    k.t_prio.assign(tk->priority, tk->priority + T); k.t_class.assign(tk->klass, tk->klass + T);
    if (tk->pod_index) k.t_podidx.assign(tk->pod_index, tk->pod_index + T); else k.t_podidx.assign(T, -1);
    if (tk->creation_ts) k.t_ts.assign(tk->creation_ts, tk->creation_ts + T); else k.t_ts.assign(T, 0);
    k.t_uid.assign(tk->uid_rank, tk->uid_rank + T); k.t_has.assign(tk->req_has, tk->req_has + T);
    k.t_req.assign(tk->resreq, tk->resreq + R * T); k.t_kreq.assign(tk->k8s_req, tk->k8s_req + K * T);
    k.t_knz.assign(tk->k8s_nonzero_req, tk->k8s_nonzero_req + 2 * T);
    k.n_idle.assign(nd->idle, nd->idle + R * N);
    if (nd->releasing) k.n_rel.assign(nd->releasing, nd->releasing + R * N); else k.n_rel.assign(R * N, 0.0);
    if (nd->pipelined) k.n_pip.assign(nd->pipelined, nd->pipelined + R * N); else k.n_pip.assign(R * N, 0.0);
    for (int r = 0; r < s->rt.n; ++r) {  // the table of vc_snapshot_set_running against this session's sizes
      if (s->rt.node[r] < 0 || (size_t)s->rt.node[r] >= N) return fail(VC_EINVAL, "running task %d: bad node index", r);
      const int j = s->rt.job[r];
      if (j < -1 || j >= (int)J) return fail(VC_EINVAL, "running task %d: bad job index", r);
      if (j >= 0 && (s->rt.role[r] < jb->role_off[j] || s->rt.role[r] >= jb->role_off[j + 1]))
        return fail(VC_EINVAL, "running task %d: role row outside its job", r);
    }
    if (!s->t_flags.empty() && s->t_flags.size() != T) return fail(VC_EINVAL, "task flags: %zu entries for %zu tasks", s->t_flags.size(), T);
  }
  tick("host copies for the later actions");
  if (s->bf.n > 0) {  // what pickUpPendingTasks (backfill.go:118-199) orders by, as of session open
    vch::BackfillKeep &k = s->bk;
    k.j_queue.assign(jb->queue, jb->queue + J); k.j_min.assign(jb->min_available, jb->min_available + J);
    k.j_prio.assign(jb->priority, jb->priority + J); k.j_ready0.assign(jb->ready_num, jb->ready_num + J);
    k.j_pbe.assign(jb->pending_besteffort, jb->pending_besteffort + J);
    k.j_taskmintotal.assign(jb->task_min_total, jb->task_min_total + J);
    k.j_roleoff.assign(jb->role_off, jb->role_off + J + 1);
    k.r_min.assign(jb->role_min, jb->role_min + NR); k.r_occ0.assign(jb->role_occupied, jb->role_occupied + NR);
    k.r_flags.assign(jb->role_flags, jb->role_flags + NR);
    k.q_prio.assign(qu->priority, qu->priority + Q);
    k.t_role.assign(tk->role, tk->role + T);
    k.j_flags.assign(jb->flags, jb->flags + J);
    k.j_rank = j_rank; k.q_rank = q_rank;
    k.j_valid.resize(J);
    for (size_t j = 0; j < J; ++j) k.j_valid[j] = vch::job_valid(*conf, *jb, (int)j) ? 1 : 0;
    k.j_alloc0.assign(jb->allocated, jb->allocated + R * J);
    const size_t Bn = (size_t)s->bf.n;
    s->rows_integral = s->rows_integral && vch::runs_exact(R, N, Bn, {nd->idle, nd->used}, {s->bf.req.data()}) &&
                       vch::runs_exact(K, N, Bn, {nd->k8s_requested}, {s->bf.kreq.data()}) &&
                       vch::runs_exact(2, N, Bn, {nd->k8s_nonzero_requested}, {s->bf.knz.data()});
    for (int t = 0; t < s->bf.n; ++t) {
      if (s->bf.job[t] < 0 || (size_t)s->bf.job[t] >= J) return fail(VC_EINVAL, "backfill task %d: bad job index", t);
      if (s->bf.klass[t] < 0 || (size_t)s->bf.klass[t] >= C) return fail(VC_EINVAL, "backfill task %d: bad class index", t);
      const int j = s->bf.job[t], r = s->bf.role[t];
      if (r < jb->role_off[j] || r >= jb->role_off[j + 1]) return fail(VC_EINVAL, "backfill task %d: role row outside its job", t);
    }
  }
  s->upload_ms = now_ms() - t0;
  return VC_OK;
}

int vc_snapshot_update_nodes(vc_snapshot *s, int32_t n_dirty, const int32_t *node_idx, const vc_nodes *rows) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  if (!s->uploaded) return fail(VC_EINVAL, "vc_snapshot_upload must precede vc_snapshot_update_nodes");
  if (n_dirty < 0 || (n_dirty > 0 && (!node_idx || !rows))) return fail(VC_EINVAL, "null argument");
  if (s->dc.nta_tables) return fail(VC_EUNSUPPORTED, "incremental upload: the session carries hypernode tables, upload it in full");
  const double t0 = now_ms();
  const size_t N = s->dims.n_nodes, R = s->dims.n_dims, K = s->dims.n_kdims, m = (size_t)n_dirty;
  if (m > 0 && (!rows->idle || !rows->used || !rows->k8s_requested || !rows->k8s_nonzero_requested || !rows->pod_count))
    return fail(VC_EINVAL, "incremental upload: idle, used, k8s_requested, k8s_nonzero_requested and pod_count are required");
  for (size_t i = 0; i < m; ++i)
    if (node_idx[i] < 0 || (size_t)node_idx[i] >= N) return fail(VC_EINVAL, "dirty node %zu: index out of range", i);
  bool fut = false;
  for (size_t i = 0; i < R * m && !fut; ++i)
    if ((rows->releasing && rows->releasing[i] != 0.0) || (rows->pipelined && rows->pipelined[i] != 0.0)) fut = true;
  if (fut && !s->dc.has_future)
    return fail(VC_EUNSUPPORTED, "incremental upload: first Releasing / Pipelined resource of the session, upload it in full");
  // every value the run-length batches rely on stays an integer of safe magnitude
  if (s->rows_integral) {
    double mx = 0.0;
    s->rows_integral = vch::max_abs_integral(rows->idle, R * m, mx) && vch::max_abs_integral(rows->used, R * m, mx) &&
                       vch::max_abs_integral(rows->releasing, R * m, mx) && vch::max_abs_integral(rows->pipelined, R * m, mx) &&
                       vch::max_abs_integral(rows->k8s_requested, K * m, mx) &&
                       vch::max_abs_integral(rows->k8s_nonzero_requested, 2 * m, mx) && mx < 8.0e15;
  }
  if (m > 0) {
    const size_t rows_n = 4 * R + 2 * K, bytes = rows_n * m * 8 + m * 4 + m * 4;
    if (bytes > s->delta_cap) {
      if (s->delta_pin) cudaFreeHost(s->delta_pin);
      if (s->delta_dev) cudaFree(s->delta_dev);
      s->delta_pin = s->delta_dev = nullptr;
      const size_t cap = std::max<size_t>(bytes * 2, 1 << 16);
      CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&s->delta_pin), cap));
      CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->delta_dev), cap));
      s->delta_cap = cap;
    }
    double *v = reinterpret_cast<double *>(s->delta_pin);
    auto put_rows = [&](size_t row0, const double *src, size_t nrows) {
      if (src) std::memcpy(v + row0 * m, src, nrows * m * 8);
      else std::memset(v + row0 * m, 0, nrows * m * 8);
    };
    put_rows(0, rows->idle, R); put_rows(R, rows->used, R); put_rows(2 * R, rows->releasing, R); put_rows(3 * R, rows->pipelined, R);
    put_rows(4 * R, rows->k8s_requested, K); put_rows(4 * R + K, rows->k8s_nonzero_requested, 2);
    int32_t *pi = reinterpret_cast<int32_t *>(s->delta_pin + rows_n * m * 8);
    std::memcpy(pi, rows->pod_count, m * 4);
    std::memcpy(pi + m, node_idx, m * 4);
    CUDA_TRY(cudaMemcpyAsync(s->delta_dev, s->delta_pin, bytes, cudaMemcpyHostToDevice, s->stream));
    NodeDeltaParams p;
    p.N = (int)N; p.R = (int)R; p.K = (int)K; p.n = (int)m;
    p.vals = reinterpret_cast<const double *>(s->delta_dev);
    p.pods = reinterpret_cast<const int32_t *>(s->delta_dev + rows_n * m * 8);
    p.idx = p.pods + m;
    p.idle = s->n_idle.d(s->in); p.used = s->n_used.d(s->in); p.rel = s->n_rel.d(s->in); p.pip = s->n_pip.d(s->in);
    p.kreq = s->n_kreq.d(s->in); p.knz = s->n_knz.d(s->in); p.pod_count = s->n_pod_count.d(s->in);
    k_node_delta<<<(unsigned)((m + 127) / 128), 128, 0, s->stream>>>(p);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    // host mirrors the later actions read (pinned staging copy of the inputs, the evicting actions' opening rows)
    double *h_idle = s->n_idle.h(s->in), *h_used = s->n_used.h(s->in), *h_rel = s->n_rel.h(s->in), *h_pip = s->n_pip.h(s->in);
    double *h_kreq = s->n_kreq.h(s->in), *h_knz = s->n_knz.h(s->in);
    int32_t *h_pods = s->n_pod_count.h(s->in);
    for (size_t i = 0; i < m; ++i) {
      const size_t n = (size_t)node_idx[i];
      for (size_t d = 0; d < R; ++d) {
        h_idle[d * N + n] = rows->idle[d * m + i]; h_used[d * N + n] = rows->used[d * m + i];
        h_rel[d * N + n] = rows->releasing ? rows->releasing[d * m + i] : 0.0;
        h_pip[d * N + n] = rows->pipelined ? rows->pipelined[d * m + i] : 0.0;
        s->ek.n_idle[d * N + n] = h_idle[d * N + n]; s->ek.n_rel[d * N + n] = h_rel[d * N + n]; s->ek.n_pip[d * N + n] = h_pip[d * N + n];
      }
      for (size_t kk = 0; kk < K; ++kk) h_kreq[kk * N + n] = rows->k8s_requested[kk * m + i];
      for (size_t kk = 0; kk < 2; ++kk) h_knz[kk * N + n] = rows->k8s_nonzero_requested[kk * m + i];
      h_pods[n] = rows->pod_count[i];
    }
    CUDA_TRY(cudaStreamSynchronize(s->stream));
  }
  // the session is at its (new) opening state
  s->alloc_ran = false; s->bf_ran = false; s->es_built = false; s->dense_ready = false;
  s->last_idx_cur = s->dc.last_idx0;
  s->last_dec.clear(); s->last_vis.clear();
  s->upload_ms = now_ms() - t0;
  s->h2d_bytes = (int64_t)((4 * R + 2 * K) * m * 8 + m * 8);
  return VC_OK;
}

int vc_queue_deserved(vc_snapshot *s, double *deserved_out, double *share_out) {
  if (!s || !s->uploaded) return fail(VC_EINVAL, "snapshot not uploaded");
  const int R = s->dims.n_dims, Q = s->dims.n_queues;
  for (int q = 0; q < Q; ++q) {
    const vch::QAttr &a = s->qattr[q];
    for (int d = 0; d < R; ++d)
      if (deserved_out) deserved_out[(size_t)d * Q + q] = (d < 2 || a.deserved.k(d)) ? a.deserved.v[d] : 0.0;
    if (share_out) share_out[q] = a.share;
  }
  return VC_OK;
}

// ---------------------------------------------------------------------------------------
// allocate
// ---------------------------------------------------------------------------------------
int vc_allocate_run(vc_snapshot *s, vc_result **out) {
  if (!s || !out) return fail(VC_EINVAL, "null argument");
  if (!s->uploaded) return fail(VC_EINVAL, "vc_snapshot_upload must precede vc_allocate_run");
  const double t0 = now_ms();
  const vc_dims &D = s->dims;
  const size_t N = D.n_nodes, T = D.n_tasks, J = D.n_jobs, Q = D.n_queues, R = D.n_dims, K = D.n_kdims, NR = D.n_roles;
  if (s->dd.node_begin != 0 || s->dd.node_end != (int)N)
    return fail(VC_EUNSUPPORTED, "the commit engine takes the full node axis (vc_comm_create cuts it over the ranks itself)");
  if (s->world > 1 && !s->comm_attached) return fail(VC_EINVAL, "vc_comm_attach must precede vc_allocate_run");
  const int G = s->n_cta;
  // replicas, mailbox, outputs
  const size_t i32_stride = ((5 * J + 4 * NR + 5 * Q + 3 * (size_t)s->max_job_tasks) + 63) & ~(size_t)63;
  const size_t f64_words_fast = (J * sizeof(JobDyn) + Q * sizeof(QueueDyn) + NR * sizeof(RoleDyn)) / 8 + (size_t)s->max_job_tasks;
  const size_t f64_stride = (std::max<size_t>(J + R * J + R * Q + Q + (size_t)s->max_job_tasks, f64_words_fast) + 31) & ~(size_t)31;
  // per-CTA heap replica: HeapEnt entries for k_commit, HeapKey (32 B) entries for k_commit_fast; stride in entries of
  // the kernel's own type, sized for the larger one
  const size_t heap_stride = (s->qjobs.count + 7) & ~(size_t)7;
  if (!s->rep_i32 || s->rep_i32_stride != i32_stride || s->rep_f64_stride != f64_stride || s->rep_heap_stride != heap_stride ||
      s->rep_ctas < G) {
    if (s->rep_i32) cudaFree(s->rep_i32);
    if (s->rep_f64) cudaFree(s->rep_f64);
    if (s->rep_heap) cudaFree(s->rep_heap);
    s->rep_i32 = nullptr; s->rep_f64 = nullptr; s->rep_heap = nullptr;
    CUDA_TRY(cudaMalloc(&s->rep_i32, std::max<size_t>(16, i32_stride * G * 4)));
    CUDA_TRY(cudaMalloc(&s->rep_f64, std::max<size_t>(16, f64_stride * G * 8)));
    CUDA_TRY(cudaMalloc(&s->rep_heap, std::max<size_t>(16, std::max<size_t>(heap_stride, 1) * G * sizeof(HeapKey))));
    s->rep_i32_stride = i32_stride; s->rep_f64_stride = f64_stride; s->rep_heap_stride = heap_stride;
    s->rep_ctas = G;
  }
  if (s->topo_any && !s->d_job_alloc) CUDA_TRY(cudaMalloc(&s->d_job_alloc, std::max<size_t>(16, J * 4)));
  if (s->topo_any) {
    const size_t cnt = (size_t)G * std::max<size_t>(s->placed_total, 1);
    if (!s->rep_placed || s->rep_placed_count < cnt) {
      if (s->rep_placed) cudaFree(s->rep_placed);
      s->rep_placed = nullptr;
      CUDA_TRY(cudaMalloc(&s->rep_placed, cnt * 4));
      s->rep_placed_count = cnt;
    }
  }
  if (s->dc.nta_tables) {
    const size_t cnt = (size_t)G * R * s->hn_cap;
    if (!s->rep_hn_used || s->rep_hn_used_count < cnt) {
      if (s->rep_hn_used) cudaFree(s->rep_hn_used);
      s->rep_hn_used = nullptr;
      CUDA_TRY(cudaMalloc(&s->rep_hn_used, std::max<size_t>(16, cnt * 8)));
      s->rep_hn_used_count = cnt;
    }
  }
  const size_t mbox_bytes = kMboxBytes;
  if (!s->mbox) CUDA_TRY(cudaMalloc(&s->mbox, mbox_bytes));
  if (!s->d_prof) CUDA_TRY(cudaMalloc(&s->d_prof, 16 * sizeof(long long)));
  const size_t ring_bytes = sizeof(uint4) * RING_STRIDE * RING_DEPTH;
  if (!s->ring) CUDA_TRY(cudaMalloc(&s->ring, ring_bytes));
  if (!s->d_score_log) CUDA_TRY(cudaMalloc(&s->d_score_log, (T + 64) * sizeof(uint4)));
  if (!s->d_decisions) {
    CUDA_TRY(cudaMalloc(&s->d_decisions, std::max<size_t>(1, T) * sizeof(vc_decision)));
    CUDA_TRY(cudaMalloc(&s->d_visits, (T + J + 1) * sizeof(vc_visit)));
    CUDA_TRY(cudaMalloc(&s->d_fit, std::max<size_t>(1, T) * 4));
    CUDA_TRY(cudaMalloc(&s->d_counters, 16 * 4));
    CUDA_TRY(cudaMallocHost(&s->h_decisions, std::max<size_t>(1, T) * sizeof(vc_decision)));
    CUDA_TRY(cudaMallocHost(&s->h_visits, (T + J + 1) * sizeof(vc_visit)));
    CUDA_TRY(cudaMallocHost(&s->h_fit, std::max<size_t>(1, T) * 4));
    CUDA_TRY(cudaMallocHost(&s->h_counters, 16 * 4));
  }
  K2Params p;
  std::memset(&p, 0, sizeof p);
  p.d = s->dd; p.c = s->dc; p.npc = s->npc; p.n_cta = s->world > 1 ? s->n_cta_total : G; p.max_job_tasks = s->max_job_tasks;
  p.n_ranks = s->world; p.cta_base = s->rank * G;
  p.wd_cycles = (long long)(g_tun.watchdog_ms > 0 ? g_tun.watchdog_ms : 10000) * 2000000ll;  // ~2 GHz SM clock
  p.dbg = nullptr;
  if (g_tun.watchdog_ms > 0 && g_tun.prof) {  // diagnostics (VC_PROF=1 VC_WATCHDOG_MS=n): per-CTA progress words the watchdog prints
    if (!s->d_dbg) CUDA_TRY(cudaMalloc(&s->d_dbg, 4096 * 32));
    CUDA_TRY(cudaMemsetAsync(s->d_dbg, 0, 4096 * 32, s->stream));
    p.dbg = s->d_dbg;
  }
  p.alloc = s->n_alloc.d(s->in); p.rel = s->n_rel.d(s->in); p.kalloc = s->n_kalloc.d(s->in);
  p.idle = s->w_idle; p.used = s->w_used; p.pip = s->w_pip; p.kreq = s->w_kreq; p.knz = s->w_knz;
  p.max_tasks = s->n_max_tasks.d(s->in); p.pod_count = s->w_pod_count; p.cstat = s->cstat;
  p.req = s->t_req.d(s->in); p.tkreq = s->t_kreq.d(s->in); p.tknz = s->t_knz.d(s->in); p.req_has = s->t_has.d(s->in);
  p.t_class = s->t_class.d(s->in); p.t_role = s->t_role.d(s->in);
  p.task_order = s->task_order.d(s->in); p.job_task_off = s->job_task_off.d(s->in);
  p.nominated = s->any_nominated ? s->d_nominated : nullptr;
  p.j_queue = s->j_queue.d(s->in); p.j_min = s->j_min.d(s->in); p.j_ntasks = s->j_ntasks.d(s->in);
  p.j_pbe = s->j_pbe.d(s->in); p.j_taskmintotal = s->j_taskmintotal.d(s->in); p.j_roleoff = s->j_roleoff.d(s->in);
  p.j_prio = s->j_prio.d(s->in); p.j_ready0 = s->j_ready0.d(s->in); p.j_waiting0 = s->j_waiting0.d(s->in);
  p.j_flags = s->j_flags.d(s->in); p.j_rank = s->j_rank.d(s->in); p.j_alloc0 = s->j_alloc0.d(s->in);
  p.j_share0 = s->j_share0.d(s->in);
  p.r_min = s->r_min.d(s->in); p.r_occ0 = s->r_occ0.d(s->in); p.r_pip0 = s->r_pip0.d(s->in);
  p.r_pending0 = s->r_pending0.d(s->in); p.r_flags = s->r_flags.d(s->in);
  p.q_prio = s->q_prio.d(s->in); p.q_rank = s->q_rank.d(s->in); p.q_flags = s->q_flags.d(s->in);
  p.q_alloc_has0 = s->q_alloc_has0.d(s->in); p.q_des_has = s->q_des_has.d(s->in); p.q_flags2 = s->q_flags2.d(s->in);
  p.q_alloc0 = s->q_alloc0.d(s->in); p.q_des = s->q_des.d(s->in); p.q_share0 = s->q_share0.d(s->in);
  p.qjobs_off = s->qjobs_off.d(s->in); p.qjobs = s->qjobs.d(s->in);
  for (int d = 0; d < VC_MAX_DIMS; ++d) p.total[d] = s->total[d];
  p.total_has = s->total_has;
  p.rep_i32 = s->rep_i32; p.rep_i32_stride = i32_stride; p.rep_f64 = s->rep_f64; p.rep_f64_stride = f64_stride;
  p.rep_heap = s->rep_heap; p.rep_heap_stride = std::max<size_t>(heap_stride, 1);
  p.mbox = s->mbox;
  p.mbox2 = s->mbox + kMbox2Offset;
  p.decisions = s->d_decisions; p.visits = s->d_visits; p.fit_errors = s->d_fit; p.counters = s->d_counters;
  p.prof = s->d_prof;
  p.tmeta = reinterpret_cast<const int4 *>(s->tmeta.d(s->in)); p.n_groups = s->n_groups;
  p.g_req = s->sg_req.d(s->in); p.g_kreq = s->sg_kreq.d(s->in); p.g_knz = s->sg_knz.d(s->in);
  p.g_has = s->sg_has.d(s->in); p.g_class = s->sg_class.d(s->in); p.ring = s->ring;

  p.hn_H = s->hn_H; p.hn_cap = s->hn_cap;
  p.hn_member = s->hn_member.d(s->in); p.hn_slot = s->hn_slot.d(s->in); p.cta_hn_off = s->cta_hn_off.d(s->in);
  p.cta_hn = s->cta_hn.d(s->in); p.hn_alloc = s->hn_alloc.d(s->in); p.hn_used0 = s->hn_used0.d(s->in);
  p.rep_hn_used = s->rep_hn_used;
  p.node_chain = s->node_chain.d(s->in); p.cta_chain_off = s->cta_chain_off.d(s->in); p.cta_chain = s->cta_chain.d(s->in);
  p.chain_cap = s->chain_cap;
  p.hn_smem = s->hn_smem;
  p.hn_min_tier = s->hn_min_tier; p.hn_up = s->hn_up.d(s->in); p.hn_tier = s->hn_tier_s.d(s->in);
  p.hn_parent = s->hn_parent_s.d(s->in); p.job_soft = s->job_soft_s.d(s->in); p.job_alloc0 = s->job_alloc0_s.d(s->in);
  p.placed_off = s->placed_off_s.d(s->in); p.placed0 = s->placed0_s.d(s->in); p.placed_n0 = s->placed_n0_s.d(s->in);
  p.rep_placed = s->rep_placed; p.placed_total = s->placed_total; p.job_alloc_out = s->d_job_alloc;
  p.topo_nval = s->topo_nval;
  for (int i = 0; i < VC_MAX_TIERS + 2; ++i) p.topo_val[i] = s->topo_val[i];

  long long *d_wait = nullptr;
  if (g_tun.prof_wait) {
    if (!s->d_wait) CUDA_TRY(cudaMalloc(&s->d_wait, 1024 * 8));
    d_wait = s->d_wait;
    CUDA_TRY(cudaMemsetAsync(d_wait, 0, 1024 * 8, s->stream));
  }
  p.cta_wait = d_wait;
  // (the instrumented instance exists for the plain and the FUT shape)
  const void *kfn = s->fast && s->dc.to_find > 0 ? (s->fut_rows ? (const void *)k_commit_fast<false, true, false, true>
                                                                 : g_tun.prof ? (const void *)k_commit_fast<true, false, false, true> : (const void *)k_commit_fast<false, false, false, true>)
                  : s->fast ? (s->dc.soft_active ? (s->dc.has_future ? (const void *)k_commit_fast<false, true, true> : (const void *)k_commit_fast<false, false, true>)
                               : s->dc.has_future ? (g_tun.prof ? (const void *)k_commit_fast<true, true> : (const void *)k_commit_fast<false, true>)
                                                  : (g_tun.prof ? (const void *)k_commit_fast<true, false> : (const void *)k_commit_fast<false, false>))
                  : s->dc.to_find > 0 ? (s->topo_any ? (const void *)k_commit<true, true, true, true> : (const void *)k_commit<true, true, false, true>)
                  : s->topo_any ? (const void *)k_commit<true, true, true> : s->dc.has_future ? (s->dc.soft_active ? (const void *)k_commit<true, true> : (const void *)k_commit<true, false>)
                                     : (s->dc.soft_active ? (const void *)k_commit<false, true> : (const void *)k_commit<false, false>);
  if (int rc = check_smem(kfn, s->smem_bytes, "commit kernel")) return rc;
  CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes));
  int max_blocks = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks, kfn, s->block, s->smem_bytes));
  if (max_blocks * g_sm_count < G)
    return fail(VC_EUNSUPPORTED, "commit kernel cannot be co-resident: %d CTAs x %zu B smem (max %d/SM)", G, s->smem_bytes, max_blocks);
  FastParams fp;
  fp.jstat = s->s_jstat.d(s->in); fp.rstat = s->s_rstat.d(s->in); fp.qstat = s->s_qstat.d(s->in);
  fp.q_share0 = s->q_share0.d(s->in);
  fp.heap_off = s->s_heap_off.d(s->in); fp.ready_word = s->fast_ready_word; fp.ready_shift = s->fast_ready_shift;
  fp.share_on = s->fast_share_on; fp.heap_in_smem = s->heap_in_smem; fp.heap_total = s->heap_total;
  fp.run_max = (s->rows_integral && !g_tun.commit_norun && s->dc.to_find == 0)
                   ? std::max(1, std::min(g_tun.run_max > 0 ? g_tun.run_max : RUN_MAX, std::min(RUN_MAX, 2 * (s->block / 32 - 1)))) : 1;
  fp.score_log = s->d_score_log;
  if (s->world > 1) {  // mailbox, ring and score log live in the exported slabs; the score log is rank 0's (it writes the decisions)
    p.mbox = reinterpret_cast<uint4 *>(s->comm);
    p.ring = reinterpret_cast<uint4 *>(s->comm + s->comm_ring_off);
    for (int r = 0; r < s->world; ++r) {
      p.peer_mbox[r] = reinterpret_cast<uint4 *>(s->peer_comm[r]);
      p.peer_ring[r] = reinterpret_cast<uint4 *>(s->peer_comm[r] + s->comm_ring_off);
    }
    fp.score_log = reinterpret_cast<uint4 *>(s->peer_comm[0] + s->comm_log_off);
  }
  // ---- the timed region (vc_stats.commit_ms) starts here: the per-cycle resets and working copies are work
  //      every cycle does, so they are inside it ----
  CUDA_TRY(cudaEventRecord(s->ev0, s->stream));
  CUDA_TRY(cudaMemsetAsync(s->d_prof, 0, 16 * sizeof(long long), s->stream));
  if (s->world <= 1) {  // with several ranks vc_comm_prepare cleared the exported slab before the ranks' barrier
    CUDA_TRY(cudaMemsetAsync(s->ring, 0, ring_bytes, s->stream));
    CUDA_TRY(cudaMemsetAsync(s->mbox, 0, mbox_bytes, s->stream));
    if (s->fast) CUDA_TRY(cudaMemsetAsync(s->d_score_log, 0, (T + 64) * sizeof(uint4), s->stream));
  }
  CUDA_TRY(cudaMemsetAsync(s->d_counters, 0, 16 * 4, s->stream));
  // working copies of the mutable node state (the uploaded snapshot stays intact for re-runs / K1)
  CUDA_TRY(cudaMemcpyAsync(s->w_idle, s->n_idle.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->w_used, s->n_used.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->w_pip, s->n_pip.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->w_kreq, s->n_kreq.d(s->in), K * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->w_knz, s->n_knz.d(s->in), 2 * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->w_pod_count, s->n_pod_count.d(s->in), N * 4, cudaMemcpyDeviceToDevice, s->stream));

  void *args[] = {&p, &fp};
  CUDA_TRY(cudaLaunchCooperativeKernel(kfn, dim3(G), dim3(s->block), args, s->smem_bytes, s->stream));
  g_launches++;
  CUDA_TRY(cudaEventRecord(s->ev1, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->h_counters, s->d_counters, 16 * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaMemcpyAsync(s->h_prof, s->d_prof, 16 * sizeof(long long), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (d_wait) {
    std::vector<long long> w(G);
    cudaMemcpy(w.data(), d_wait, G * 8, cudaMemcpyDeviceToHost);
    fprintf(stderr, "all-gather wait per CTA (Mcycles):");
    for (int i = 0; i < G; ++i) fprintf(stderr, " %.0f", w[i] / 1e6);
    fprintf(stderr, "\n");
  }
  const double t_k = now_ms();
  const int n_dec = s->h_counters[0], n_vis = s->h_counters[1], n_fit = s->h_counters[2];
  if (n_dec) CUDA_TRY(cudaMemcpyAsync(s->h_decisions, s->d_decisions, (size_t)n_dec * sizeof(vc_decision), cudaMemcpyDeviceToHost, s->stream));
  if (n_vis) CUDA_TRY(cudaMemcpyAsync(s->h_visits, s->d_visits, (size_t)n_vis * sizeof(vc_visit), cudaMemcpyDeviceToHost, s->stream));
  if (n_fit) CUDA_TRY(cudaMemcpyAsync(s->h_fit, s->d_fit, (size_t)n_fit * 4, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  vc_result *r = new vc_result();
  r->decisions.assign(s->h_decisions, s->h_decisions + n_dec);
  r->visits.assign(s->h_visits, s->h_visits + n_vis);
  r->fit_errors.assign(s->h_fit, s->h_fit + n_fit);
  s->alloc_ran = true; s->bf_ran = false;
  s->last_dec = r->decisions;  // discarded visits carry no operations
  s->last_vis = r->visits;
  s->es_built = false;  // the session state of the evicting actions is rebuilt from this run's operations
  if (s->topo_any) {
    r->job_alloc.resize(J);
    CUDA_TRY(cudaMemcpy(r->job_alloc.data(), s->d_job_alloc, J * 4, cudaMemcpyDeviceToHost));
  } else if (!s->h_job_soft.empty() && !s->h_member.empty()) {
    // soft-mode topology jobs without the plugin: allocate.go still tracks the allocated hypernode
    // (:572, :672-674, :681-686); nothing on the device reads it, so replay the visits on the host
    bool any = false;
    for (uint8_t f : s->h_job_soft) any = any || f;
    if (any) {
      r->job_alloc = s->h_job_alloc;
      const int H = s->hn_H;
      auto ancestor_of = [&](int a, int hn) {  // is `a` on the Parent chain of hn (hn included)?
        for (int x = hn, g = 0; x >= 0 && g < VC_MAX_TIERS + 2; x = s->h_parent[x], ++g)
          if (x == a) return true;
        return false;
      };
      for (const vc_visit &v : r->visits) {
        if (!s->h_job_soft[v.job] || v.n_ops == 0) continue;
        int a = r->job_alloc[v.job];
        for (int k = v.first_op; k < v.first_op + v.n_ops; ++k) {
          const int hn = s->h_member[r->decisions[k].node];  // util.FindHyperNodeForNode: lowest tier only
          if (hn < 0 || hn >= H) continue;
          if (a < 0) { a = hn; continue; }
          int lca = -1;  // GetLCAHyperNode(hn, a): first ancestor of `a` that is an ancestor of hn
          for (int x = a, g = 0; x >= 0 && g < VC_MAX_TIERS + 2; x = s->h_parent[x], ++g)
            if (ancestor_of(x, hn)) { lca = x; break; }
          a = lca;
        }
        if (v.outcome == VC_VISIT_COMMIT) r->job_alloc[v.job] = a;
      }
    }
  }
  float kms = 0;
  cudaEventElapsedTime(&kms, s->ev0, s->ev1);
  r->stats.upload_ms = s->upload_ms;
  r->stats.commit_ms = kms;
  r->stats.download_ms = now_ms() - t_k;
  r->stats.total_ms = now_ms() - t0;
  r->stats.h2d_bytes = s->h2d_bytes;
  r->stats.d2h_bytes = 32 + (int64_t)n_dec * sizeof(vc_decision) + (int64_t)n_vis * sizeof(vc_visit) + (int64_t)n_fit * 4;
  r->stats.kernel_launches = 2;  // k_class_static + k_commit
  r->stats.n_steps = s->h_counters[3];
  r->stats.last_processed_node_index = (s->dc.to_find > 0 || s->any_nominated) ? s->h_counters[4] : s->dc.last_idx0;
  r->stats.commit_kernel = s->fast ? VC_KERNEL_INCREMENTAL : VC_KERNEL_GENERAL;
  s->last_idx_cur = r->stats.last_processed_node_index;
  for (int k = 0; k < 8; ++k) r->stats.prof_cycles[k] = s->h_prof[k];
  r->stats.prof_cycles[6] = s->h_counters[5];  // full sweeps (fast kernel)
  r->stats.prof_cycles[7] = s->h_counters[6];  // incremental steps (fast kernel)
  r->stats.prof_cycles[5] = s->h_counters[7];  // owner changes between consecutive publications
  if (g_tun.prof_owner)
    fprintf(stderr, "runs: %d publications covering %d placements (%.2f per run), command -> publish %.0f cycles per run\n",
            s->h_counters[13], s->h_counters[14], (double)s->h_counters[14] / std::max(1, s->h_counters[13]),
            1024.0 * s->h_counters[15] / std::max(1, s->h_counters[13]));
  if (g_tun.prof_owner)
    fprintf(stderr, "evaluator (all CTAs): %d evaluations, %d speculation hits, %d cache rescans; command -> publish %.0f cycles, "
                    "speculative run-ahead %.0f cycles per evaluation (VC_PROF instance only)\n", s->h_counters[10], s->h_counters[8],
            s->h_counters[9], 1024.0 * s->h_counters[11] / std::max(1, s->h_counters[10]), 1024.0 * s->h_counters[12] / std::max(1, s->h_counters[10]));
  if (g_tun.prof_owner && s->h_prof[9]) fprintf(stderr, "owner steps=%lld: post->join-start %.0f, join wait %.0f, join->next post (same owner) %.0f cycles [join->a %.0f, a->b %.0f, b->c %.0f, c->post %.0f]\n",
      s->h_prof[9], (double)s->h_prof[8] / s->h_prof[9], (double)s->h_prof[10] / s->h_prof[9], (double)s->h_prof[11] / s->h_prof[9], (double)s->h_prof[12] / s->h_prof[9], (double)s->h_prof[13] / s->h_prof[9], (double)s->h_prof[14] / s->h_prof[9], (double)s->h_prof[15] / s->h_prof[9]);
  *out = r;
  return VC_OK;
}

size_t vc_result_num_decisions(const vc_result *r) { return r ? r->decisions.size() : 0; }
const vc_decision *vc_result_decisions(const vc_result *r) { return r ? r->decisions.data() : nullptr; }
size_t vc_result_num_visits(const vc_result *r) { return r ? r->visits.size() : 0; }
const vc_visit *vc_result_visits(const vc_result *r) { return r ? r->visits.data() : nullptr; }
size_t vc_result_num_fit_errors(const vc_result *r) { return r ? r->fit_errors.size() : 0; }
const int32_t *vc_result_fit_errors(const vc_result *r) { return r ? r->fit_errors.data() : nullptr; }
const vc_stats *vc_result_stats(const vc_result *r) { return r ? &r->stats : nullptr; }
const int32_t *vc_result_job_allocated_hypernodes(const vc_result *r, size_t *n_jobs) {
  if (n_jobs) *n_jobs = r ? r->job_alloc.size() : 0;
  return (r && !r->job_alloc.empty()) ? r->job_alloc.data() : nullptr;
}
void vc_result_free(vc_result *r) { delete r; }

// ---------------------------------------------------------------------------------------
// preempt / reclaim (actions/preempt/preempt.go, actions/reclaim/reclaim.go)
// ---------------------------------------------------------------------------------------
int vc_snapshot_set_running(vc_snapshot *s, const vc_running_tasks *rt, const uint32_t *task_flags) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  s->uploaded = false;  // validated against the job / role tables by the next upload
  const size_t T = s->dims.n_tasks, R = s->dims.n_dims, K = s->dims.n_kdims, N = s->dims.n_nodes;
  s->t_flags.clear();
  if (task_flags) s->t_flags.assign(task_flags, task_flags + T);
  vch::RunningTasks &b = s->rt;
  b = vch::RunningTasks();
  if (!rt || rt->n_tasks <= 0) return VC_OK;
  const size_t B = (size_t)rt->n_tasks;
  if (!rt->node || !rt->job || !rt->role || !rt->priority || !rt->uid_rank || !rt->resreq || !rt->req_has || !rt->k8s_req ||
      !rt->k8s_nonzero_req || !rt->flags)
    return fail(VC_EINVAL, "running task table: null array");
  b.n = (int)B;
  b.node.assign(rt->node, rt->node + B); b.job.assign(rt->job, rt->job + B); b.role.assign(rt->role, rt->role + B);
  b.prio.assign(rt->priority, rt->priority + B); b.uid.assign(rt->uid_rank, rt->uid_rank + B);
  if (rt->pod_index) b.podidx.assign(rt->pod_index, rt->pod_index + B); else b.podidx.assign(B, -1);
  if (rt->creation_ts) b.ts.assign(rt->creation_ts, rt->creation_ts + B); else b.ts.assign(B, 0);
  b.has.assign(rt->req_has, rt->req_has + B); b.flags.assign(rt->flags, rt->flags + B);
  b.req.assign(rt->resreq, rt->resreq + R * B); b.kreq.assign(rt->k8s_req, rt->k8s_req + K * B);
  b.knz.assign(rt->k8s_nonzero_req, rt->k8s_nonzero_req + K * B);
  // node.Tasks as CSR, ascending running-task id inside a node (the canonical walk order of the Go map)
  b.off.assign(N + 1, 0);
  for (size_t r = 0; r < B; ++r) {
    if (b.node[r] < 0 || (size_t)b.node[r] >= N) return fail(VC_EINVAL, "running task %zu: bad node index", r);
    b.off[b.node[r] + 1] += 1;
  }
  for (size_t n = 0; n < N; ++n) b.off[n + 1] += b.off[n];
  b.idx.resize(B);
  std::vector<int32_t> fill(b.off.begin(), b.off.end() - 1);
  for (size_t r = 0; r < B; ++r) b.idx[fill[b.node[r]]++] = (int32_t)r;
  return VC_OK;
}

namespace {

// session state of the evicting actions: the opening session plus whatever vc_allocate_run did
int ensure_evict_session(vc_snapshot *s) {
  const vc_dims &D = s->dims;
  const size_t N = D.n_nodes, T = D.n_tasks, J = D.n_jobs, Q = D.n_queues, R = D.n_dims, K = D.n_kdims, NR = D.n_roles;
  if (s->bf.n > 0 || s->bf_ran) return fail(VC_EUNSUPPORTED, "preempt / reclaim: BestEffort pending tasks in the session");
  if (s->dc.to_find > 0) return fail(VC_EUNSUPPORTED, "preempt / reclaim: feasible-node sampling");
  if (s->dc.soft_active || s->dc.nta_plugin || vch::has_plugin(s->conf, VC_PLUGIN_TDM))
    return fail(VC_EUNSUPPORTED, "preempt / reclaim: PreferNoSchedule taints, network-topology-aware and tdm are outside the path");
  for (uint8_t f : s->h_job_soft)
    if (f) return fail(VC_EUNSUPPORTED, "preempt / reclaim: jobs with a network topology (preempt.go:131-135)");
  if (s->es_built) return VC_OK;
  vch::EvictSession &e = s->es;
  e = vch::EvictSession();
  e.conf = &s->conf; e.k = &s->ek; e.rt = &s->rt; e.t_flags = &s->t_flags;
  if (s->t_flags.empty()) s->t_flags.assign(T, 0u);
  e.R = (int)R; e.K = (int)K; e.N = (int)N; e.T = (int)T; e.J = (int)J; e.Q = (int)Q; e.pods_dim = D.pods_dim;
  for (int d = 0; d < VC_MAX_DIMS; ++d) e.total[d] = s->total[d];
  e.total_has = s->total_has;
  const vch::EvictKeep &k = s->ek;
  e.t_status.assign(T, 0);
  e.j_ready = k.j_ready0; e.j_waiting = k.j_waiting0; e.r_occ = k.r_occ0; e.r_pip = k.r_pip0;
  e.j_alloc = k.j_alloc0; e.j_share.assign(J, 0.0);
  e.qattr = s->qattr;
  e.n_idle = k.n_idle; e.n_rel = k.n_rel; e.n_pip = k.n_pip;
  e.rt_evicted.assign((size_t)std::max(s->rt.n, 1), 0);
  e.phase_flipped = s->alloc_ran && !s->conf.enqueue_action_enabled;
  if (s->dc.has_drf)
    for (size_t j = 0; j < J; ++j) e.drf_share((int)j);
  // Statement.Allocate / Pipeline of every kept visit of the allocate action, in order
  std::vector<double> &idle = e.n_idle;  // the host mirror of Idle moves with allocate's placements
  for (const vc_decision &op : s->last_dec) {
    const int t = op.task, j = k.t_job[t], n = op.node;
    if (op.kind == VC_OP_ALLOCATE) {
      e.t_status[t] = 1; e.j_ready[j] += 1; e.r_occ[k.t_role[t]] += 1;
      for (size_t d = 0; d < R; ++d) idle[d * N + n] -= k.t_req[d * T + t];
    } else {
      e.t_status[t] = 2; e.j_waiting[j] += 1; e.r_pip[k.t_role[t]] += 1;
      for (size_t d = 0; d < R; ++d) e.n_pip[d * N + n] += k.t_req[d * T + t];
    }
    e.on_allocate(j, e.task_res(t), k.t_req.data(), (int)T, t);
  }
  s->last_dec.clear();  // applied (a second evicting action continues from e)
  // device: working rows (left by allocate, or the opening ones), Releasing, the running-task table, scratch
  cudaError_t ce;
  auto ensure = [&](auto *&ptr, size_t bytes) -> cudaError_t {
    if (ptr) return cudaSuccess;
    void *q = nullptr;
    cudaError_t x = cudaMalloc(&q, std::max<size_t>(bytes, 16));
    ptr = reinterpret_cast<std::remove_reference_t<decltype(ptr)>>(q);
    return x;
  };
  if ((ce = ensure(s->w_rel, R * N * 8)) != cudaSuccess) return fail(VC_ECUDA, "cudaMalloc: %s", cudaGetErrorString(ce));
  CUDA_TRY(cudaMemcpyAsync(s->w_rel, s->n_rel.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
  if (!s->alloc_ran) {
    CUDA_TRY(cudaMemcpyAsync(s->w_idle, s->n_idle.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->w_used, s->n_used.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->w_pip, s->n_pip.d(s->in), R * N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->w_kreq, s->n_kreq.d(s->in), K * N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->w_knz, s->n_knz.d(s->in), 2 * N * 8, cudaMemcpyDeviceToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(s->w_pod_count, s->n_pod_count.d(s->in), N * 4, cudaMemcpyDeviceToDevice, s->stream));
  }
  const size_t B = (size_t)std::max(s->rt.n, 1);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
  const size_t o_off = take((N + 1) * 4), o_idx = take(B * 4), o_req = take(R * B * 8), o_kreq = take(K * B * 8),
               o_knz = take(K * B * 8), o_flags = take(B * 4), o_job = take(B * 4), o_ev = take(B), o_key = take(N * 8),
               o_cand = take(N), o_prio = take(B * 4), o_jready = take(std::max<size_t>(J, 1) * 4), o_qover = take(std::max<size_t>(Q, 1)),
               o_key2 = take(N * 8), o_cand2 = take(N);  // second ranking scratch: the preemptor ranked one ahead
  if (off > s->d_ev_bytes) {
    if (s->d_ev) cudaFree(s->d_ev);
    s->d_ev = nullptr;
    CUDA_TRY(cudaMalloc(&s->d_ev, off));
    s->d_ev_bytes = off;
  }
  if (!s->h_ev) CUDA_TRY(cudaHostAlloc(reinterpret_cast<void **>(&s->h_ev), (EV_CMD_OFF + 2 + EV_MAX_VICTIMS) * 4, cudaHostAllocMapped));
  (void)o_key2; (void)o_cand2;
  unsigned char *base = reinterpret_cast<unsigned char *>(s->d_ev);
  CUDA_TRY(cudaMemsetAsync(base, 0, off, s->stream));
  if (s->rt.n > 0) {
    const vch::RunningTasks &b = s->rt;
    CUDA_TRY(cudaMemcpyAsync(base + o_off, b.off.data(), (N + 1) * 4, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_idx, b.idx.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_req, b.req.data(), R * B * 8, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_kreq, b.kreq.data(), K * B * 8, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_knz, b.knz.data(), K * B * 8, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_flags, b.flags.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_job, b.job.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
    CUDA_TRY(cudaMemcpyAsync(base + o_prio, b.prio.data(), B * 4, cudaMemcpyHostToDevice, s->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  s->es_built = true;
  (void)NR; (void)o_ev; (void)o_key; (void)o_cand; (void)o_jready; (void)o_qover;
  return VC_OK;
}

// Action.Execute of preempt (preempt.go:101-283) / reclaim (reclaim.go:56-168)
int run_evict_action(vc_snapshot *s, bool reclaim, vc_result **out) {
  if (!s || !out) return fail(VC_EINVAL, "null argument");
  if (!s->uploaded) return fail(VC_EINVAL, "vc_snapshot_upload must precede the action");
  if (s->any_nominated)
    return fail(VC_EUNSUPPORTED, "preempt / reclaim: a pending task carries a NominatedNodeName (taskEligibleToPreempt's rules are not modelled)");
  const double t0 = now_ms();
  int rc = ensure_evict_session(s);
  if (rc) return rc;
  const vc_dims &D = s->dims;
  const size_t N = D.n_nodes, T = D.n_tasks, J = D.n_jobs, Q = D.n_queues, R = D.n_dims, K = D.n_kdims;
  vch::EvictSession &e = s->es;
  const vch::EvictKeep &k = s->ek;
  const size_t B = (size_t)std::max(s->rt.n, 1);
  // device parameter block (same slab layout as ensure_evict_session)
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
  const size_t o_off = take((N + 1) * 4), o_idx = take(B * 4), o_req = take(R * B * 8), o_kreq = take(K * B * 8),
               o_knz = take(K * B * 8), o_flags = take(B * 4), o_job = take(B * 4), o_ev = take(B), o_key = take(N * 8),
               o_cand = take(N), o_prio = take(B * 4), o_jready = take(std::max<size_t>(J, 1) * 4), o_qover = take(std::max<size_t>(Q, 1)),
               o_key2 = take(N * 8), o_cand2 = take(N);  // second ranking scratch: the preemptor ranked one ahead
  unsigned char *base = reinterpret_cast<unsigned char *>(s->d_ev);
  EvictParams p;
  std::memset(&p, 0, sizeof p);
  p.d = s->dd; p.c = s->dc;
  p.alloc = s->n_alloc.d(s->in); p.kalloc = s->n_kalloc.d(s->in);
  p.idle = s->w_idle; p.used = s->w_used; p.rel = s->w_rel; p.pip = s->w_pip; p.kreq = s->w_kreq; p.knz = s->w_knz;
  p.pod_count = s->w_pod_count; p.cstat = s->cstat;
  p.rt_off = reinterpret_cast<const int32_t *>(base + o_off); p.rt_idx = reinterpret_cast<const int32_t *>(base + o_idx);
  p.rt_req = reinterpret_cast<const double *>(base + o_req); p.rt_kreq = reinterpret_cast<const double *>(base + o_kreq);
  p.rt_knz = reinterpret_cast<const double *>(base + o_knz); p.rt_flags = reinterpret_cast<const uint32_t *>(base + o_flags);
  p.rt_job = reinterpret_cast<const int32_t *>(base + o_job); p.rt_evicted = base + o_ev;
  p.j_queue = s->j_queue.d(s->in); p.q_flags = s->q_flags.d(s->in); p.RT = (int)B;
  p.rt_prio = reinterpret_cast<const int32_t *>(base + o_prio); p.j_prio = s->j_prio.d(s->in); p.j_min = s->j_min.d(s->in);
  p.j_ready = reinterpret_cast<const int32_t *>(base + o_jready); p.q_over = base + o_qover;
  {
    double m1 = 0, m2 = 0;  // sums of requests are exact when every request is an integer well below 2^53 / RT
    p.exact_sums = (s->rows_integral && vch::max_abs_integral(s->rt.req.data(), s->rt.req.size(), m1) &&
                    vch::max_abs_integral(k.t_req.data(), k.t_req.size(), m2) && m1 * 4096.0 < 9.0e15) ? 1 : 0;
  }
  // ReadyTaskNum per job and proportion's "queue above deserved" as the session stands; refreshed after every success
  std::vector<uint8_t> q_over(std::max<size_t>(Q, 1), 0);
  auto refresh_dynamic = [&]() -> int {
    for (size_t q = 0; q < Q; ++q)
      q_over[q] = (e.qattr[q].exists && !e.qattr[q].allocated.less_equal_zero(e.qattr[q].deserved, (int)R)) ? 1 : 0;
    if (J) CUDA_TRY(cudaMemcpyAsync(base + o_jready, e.j_ready.data(), J * 4, cudaMemcpyHostToDevice, s->stream));
    if (Q) CUDA_TRY(cudaMemcpyAsync(base + o_qover, q_over.data(), Q, cudaMemcpyHostToDevice, s->stream));
    return VC_OK;
  };
  if ((rc = refresh_dynamic())) return rc;
  p.key = reinterpret_cast<unsigned long long *>(base + o_key); p.cand = base + o_cand;
  int32_t *dev_h = nullptr;
  CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&dev_h), s->h_ev, 0));
  p.pick_node = dev_h; p.cmd = dev_h + EV_CMD_OFF;
  int32_t *h_cmd = s->h_ev + EV_CMD_OFF;
  int launches = 0, cur_mode = 0;
  EvictTask et;
  auto stage = [&](int t, int mode) {
    std::memset(&et, 0, sizeof et);
    for (size_t d = 0; d < R; ++d) et.rec.req[d] = k.t_req[d * T + t];
    for (size_t x = 0; x < K; ++x) et.rec.kreq[x] = k.t_kreq[x * T + t];
    for (size_t x = 0; x < 2; ++x) et.rec.knz[x] = k.t_knz[x * T + t];
    et.rec.has = k.t_has[t]; et.rec.klass = k.t_class[t];
    et.klass = k.t_class[t]; et.job = k.t_job[t]; et.queue = k.j_queue[k.t_job[t]]; et.mode = mode;
    et.job_prio = k.j_prio[et.job]; et.task_prio = k.t_prio[t];
    // ssn.Allocatable goes through proportion's queueAllocatable when the plugin has EnabledAllocatable
    et.quota_on = vch::plugin_enabled(s->conf, VC_PLUGIN_PROPORTION, VC_EN_ALLOCATABLE) ? 1 : 0;
    if (et.quota_on) {
      const vch::QAttr &a = e.qattr[et.queue];
      et.quota_open = (k.q_flags[et.queue] & VC_QUEUE_OPEN) ? 1 : 0;
      et.qalloc_has = a.allocated.has; et.qdes_has = a.deserved.has;
      for (size_t d = 0; d < R; ++d) { et.qalloc[d] = a.allocated.v[d]; et.qdes[d] = a.deserved.v[d]; }
    }
  };
  int pick_buf[EV_PICK_K], pick_pos = EV_PICK_K, pick_n = 0;
  // the pick kernel stages the candidates' keys in shared memory when they fit (N * 8 bytes)
  size_t pick_smem = N * 8 <= 200 * 1024 ? N * 8 : 0;
  if (pick_smem > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_evict_pick, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pick_smem));
  double t_launch = 0.0, t_sync = 0.0;  // host time inside kernel launches / waiting for a hand-out (vc_stats.prof_cycles, us)
  // Two ranking scratch sets (candidate flags, keys, hand-out slots): while the host walks the candidates of one
  // preemptor the device already ranks the one the control loop will most likely try next (rk.hint). Most preemptors fail,
  // and a failed one leaves the session untouched, so the ranking made ahead is still exact; any eviction / pipeline /
  // discard in between (`epoch`) voids it.
  struct RankSet { unsigned long long *key; uint8_t *cand; int32_t *d_pick; volatile int32_t *h_pick; int seq; };
  RankSet sets[2] = {{reinterpret_cast<unsigned long long *>(base + o_key), base + o_cand, dev_h, s->h_ev, 0},
                     {reinterpret_cast<unsigned long long *>(base + o_key2), base + o_cand2, dev_h + (EV_PICK_K + 1),
                      s->h_ev + (EV_PICK_K + 1), 0}};
  s->h_ev[EV_PICK_K] = 0; s->h_ev[2 * EV_PICK_K + 1] = 0;
  int cur = 0, hint_t = -1, hint_mode = 0, pref_t = -1, pref_mode = 0, n_ahead = 0, n_ahead_used = 0;
  unsigned epoch = 0, pref_epoch = 0;
  bool first_pending = false;  // the first hand-out of the preemptor under trial is launched but not consumed yet
  auto with_set = [&](int k) { EvictParams q = p; q.key = sets[k].key; q.cand = sets[k].cand; q.pick_node = sets[k].d_pick; return q; };
  auto launch_pick = [&](int k, int mode) -> int {
    sets[k].seq += 1;
    if (pick_smem) k_evict_pick<<<1, 1024, pick_smem, s->stream>>>(with_set(k), mode, sets[k].seq);
    else k_evict_pick_big<<<1, 1024, 0, s->stream>>>(with_set(k), mode, 0, sets[k].seq);
    launches++;
    CUDA_TRY(cudaGetLastError());
    return VC_OK;
  };
  auto launch_rank_pick = [&](int k, int t, int mode) -> int {
    stage(t, mode);
    const double tl0 = now_ms();
    if (R <= 8) k_evict_rank<16, 8><<<(unsigned)((N * 16 + 255) / 256), 256, 0, s->stream>>>(with_set(k), et);
    else k_evict_rank<16, VC_MAX_DIMS><<<(unsigned)((N * 16 + 255) / 256), 256, 0, s->stream>>>(with_set(k), et);
    launches++;
    CUDA_TRY(cudaGetLastError());
    const int rc2 = launch_pick(k, mode);
    t_launch += now_ms() - tl0;
    return rc2;
  };
  vch::Ranker rk;
  rk.hint = [&](int t, int mode) { hint_t = t; hint_mode = mode; };
  rk.begin = [&](int t, int mode) -> int {
    cur_mode = mode;
    pick_pos = pick_n = 0;
    if (N == 0) return VC_OK;
    int rc2 = VC_OK;
    if (pref_t == t && pref_mode == mode && pref_epoch == epoch) {
      cur = 1 - cur;  // ranked ahead on a session state that still stands
      n_ahead_used += 1;
    } else if ((rc2 = launch_rank_pick(cur, t, mode))) {
      return rc2;
    }
    pref_t = -1;
    first_pending = true;
    if (hint_t >= 0 && hint_t != t) {
      if ((rc2 = launch_rank_pick(1 - cur, hint_t, hint_mode))) return rc2;
      pref_t = hint_t; pref_mode = hint_mode; pref_epoch = epoch;
      n_ahead += 1;
    }
    hint_t = -1;
    stage(t, mode);  // `et` describes the preemptor under trial again
    return VC_OK;
  };
  rk.next = [&](int *node) -> int {
    *node = -1;
    if (N == 0) return VC_OK;
    if (pick_pos >= pick_n) {
      if (pick_n > 0 && pick_n < EV_PICK_K) return VC_OK;  // the last batch was short: no candidate is left
      if (!first_pending) {
        const double tl0 = now_ms();
        const int rc2 = launch_pick(cur, cur_mode);
        t_launch += now_ms() - tl0;
        if (rc2) return rc2;
      }
      first_pending = false;
      const double tl1 = now_ms();
      // the kernel's last store is its sequence number into the mapped buffer: poll it (a stream query every few thousand
      // spins turns a failed launch into an error instead of an endless wait)
      volatile int32_t *h_pick = sets[cur].h_pick;
      for (unsigned spins = 0; h_pick[EV_PICK_K] != sets[cur].seq; ++spins)
        if ((spins & 0xfffu) == 0xfffu) {
          const cudaError_t qe = cudaStreamQuery(s->stream);
          if (qe != cudaSuccess && qe != cudaErrorNotReady) return fail(VC_ECUDA, "evict pick: %s", cudaGetErrorString(qe));
          if (qe == cudaSuccess && h_pick[EV_PICK_K] != sets[cur].seq) return fail(VC_ECUDA, "evict pick: completion word missing");
        }
      t_sync += now_ms() - tl1;
      pick_n = 0;
      for (int i = 0; i < EV_PICK_K && h_pick[i] >= 0; ++i) pick_buf[pick_n++] = h_pick[i];
      pick_pos = 0;
      if (pick_n == 0) return VC_OK;
    }
    *node = pick_buf[pick_pos++];
    return VC_OK;
  };
  auto apply_cmd = [&](int t, int node, const std::vector<int> &victims, int undo) -> int {
    if (victims.size() > EV_MAX_VICTIMS) return fail(VC_EUNSUPPORTED, "more than %d victims on one node", EV_MAX_VICTIMS);
    epoch += 1;  // node rows, ReadyTaskNum, queue shares move: a ranking made ahead is void
    stage(t, cur_mode);
    CUDA_TRY(cudaStreamSynchronize(s->stream));  // the previous command has been consumed
    h_cmd[0] = node; h_cmd[1] = (int32_t)victims.size();
    for (size_t i = 0; i < victims.size(); ++i) h_cmd[2 + i] = victims[i];
    k_evict_apply<<<1, 64, 0, s->stream>>>(p, et, undo);
    launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    return refresh_dynamic();  // ReadyTaskNum / queue shares moved (the host state is already updated)
  };
  rk.apply = [&](int t, int node, const std::vector<int> &v) { return apply_cmd(t, node, v, 0); };
  rk.revert = [&](int t, int node, const std::vector<int> &v) { return apply_cmd(t, node, v, 1); };

  vc_result *r = new vc_result();
  auto emit = [&](int job, const std::vector<vch::EvictOp> &ops, bool commit) {
    vc_visit v;
    v.job = job; v.first_op = (int32_t)r->decisions.size();
    v.outcome = commit ? VC_VISIT_COMMIT : VC_VISIT_DISCARD;
    v.n_ops = commit ? (int32_t)ops.size() : 0;
    if (commit)
      for (const vch::EvictOp &op : ops) {
        vc_decision d;
        d.task = op.task; d.node = op.node; d.kind = op.kind; d.visit = (int32_t)r->visits.size(); d.score = 0.0;
        r->decisions.push_back(d);
      }
    r->visits.push_back(v);
  };
  auto bail = [&](int code) { delete r; return code; };
  auto job_pending = [&](int j) { return (k.j_flags[j] & VC_JOB_PENDING_PHASE) && !e.phase_flipped; };
  auto pending_tasks = [&](int j, vch::GoPQ &pq) {
    pq.less = [&e](int l, int x) { return e.task_less(l, x); };
    for (size_t t = 0; t < T; ++t)
      if (k.t_job[t] == j && e.t_status[t] == 0) pq.push((int)t);
  };
  std::vector<vch::GoPQ> preemptors(Q), ptasks(J);
  for (size_t q = 0; q < Q; ++q) preemptors[q].less = [&e](int l, int x) { return e.job_less(l, x); };
  vch::GoPQ queues;
  queues.less = [&e](int l, int x) { return e.queue_less(l, x); };
  if (!reclaim) {
    std::vector<std::vector<int>> under_request(Q);
    std::vector<uint8_t> has_q(Q, 0);
    for (size_t j = 0; j < J; ++j) {
      if (job_pending((int)j) || !k.j_valid[j]) continue;
      const int q = k.j_queue[j];
      if (q < 0 || !e.job_starving((int)j)) continue;
      has_q[q] = 1;
      preemptors[q].push((int)j);
      under_request[q].push_back((int)j);
      pending_tasks((int)j, ptasks[j]);
    }
    for (size_t q = 0; q < Q; ++q)
      if (has_q[q]) queues.push((int)q);
    while (!queues.empty()) {
      const int q = queues.pop();
      while (!preemptors[q].empty()) {  // preemption between jobs within the queue, preempt.go:163-243
        const int pj = preemptors[q].pop();
        std::vector<vch::EvictOp> stmt;
        bool assigned = false;
        for (;;) {
          if (!e.job_starving(pj) || ptasks[pj].empty()) break;
          const int t = ptasks[pj].pop();
          if (!ptasks[pj].empty()) rk.hint(ptasks[pj].h[0], EV_MODE_PREEMPT_INTER);  // tried next unless this one succeeds
          if ((rc = e.try_task(rk, stmt, t, EV_MODE_PREEMPT_INTER, &assigned))) return bail(rc);
        }
        if (e.job_pipelined(pj)) {
          emit(pj, stmt, true);
        } else {
          if ((rc = e.discard_applied(rk, stmt))) return bail(rc);
          emit(pj, stmt, false);
          continue;
        }
        if (assigned) preemptors[q].push(pj);
      }
      for (int j : under_request[q]) {  // preemption between tasks within a job, preempt.go:246-280
        vch::GoPQ intra;
        pending_tasks(j, intra);
        while (!intra.empty()) {
          const int t = intra.pop();
          std::vector<vch::EvictOp> stmt;
          bool assigned = false;
          if ((rc = e.try_task(rk, stmt, t, EV_MODE_PREEMPT_INTRA, &assigned))) return bail(rc);
          if (!assigned) {
            if ((rc = e.discard_applied(rk, stmt))) return bail(rc);
            emit(j, stmt, false);
            break;
          }
          emit(j, stmt, true);
        }
      }
    }
  } else {
    std::vector<uint8_t> q_seen(Q, 0), has_pre(Q, 0);
    for (size_t j = 0; j < J; ++j) {
      if (job_pending((int)j) || !k.j_valid[j]) continue;
      const int q = k.j_queue[j];
      if (q < 0) continue;
      if (!q_seen[q]) { q_seen[q] = 1; queues.push(q); }
      if (e.job_starving((int)j)) {
        has_pre[q] = 1;
        preemptors[q].push((int)j);
        pending_tasks((int)j, ptasks[j]);
      }
    }
    while (!queues.empty()) {
      const int q = queues.pop();
      if (e.overused(q)) continue;
      for (;;) {
        if (!has_pre[q] || preemptors[q].empty()) break;
        const int job = preemptors[q].pop();
        std::vector<vch::EvictOp> stmt;
        for (;;) {
          if (!e.job_starving(job) || ptasks[job].empty()) break;
          const int t = ptasks[job].pop();
          if (s->t_flags[t] & VC_TASK_PREEMPT_NEVER) continue;     // reclaim.go:140-143
          if (!e.gate(VC_EN_PREEMPTIVE, q, t)) continue;           // ssn.Preemptive, reclaim.go:145-148
          if (!ptasks[job].empty()) rk.hint(ptasks[job].h[0], EV_MODE_RECLAIM);
          bool assigned = false;
          if ((rc = e.try_task(rk, stmt, t, EV_MODE_RECLAIM, &assigned))) return bail(rc);
        }
        if (e.job_pipelined(job)) {
          emit(job, stmt, true);
        } else {
          if ((rc = e.discard_applied(rk, stmt))) return bail(rc);
          emit(job, stmt, false);
        }
        if (!preemptors[q].empty()) queues.push(q);
      }
    }
  }
  r->stats.total_ms = now_ms() - t0;
  r->stats.commit_ms = r->stats.total_ms;
  r->stats.kernel_launches = launches;
  r->stats.n_steps = launches;
  r->stats.prof_cycles[0] = (int64_t)(t_launch * 1e3);  // microseconds of host time in launches / in synchronisations
  r->stats.prof_cycles[1] = (int64_t)(t_sync * 1e3);
  r->stats.prof_cycles[2] = n_ahead;       // preemptors ranked one ahead / of those, how many rankings were used
  r->stats.prof_cycles[3] = n_ahead_used;
  *out = r;
  return VC_OK;
}

}  // namespace

int vc_preempt_run(vc_snapshot *s, vc_result **out) { return run_evict_action(s, false, out); }
int vc_reclaim_run(vc_snapshot *s, vc_result **out) { return run_evict_action(s, true, out); }

// ---------------------------------------------------------------------------------------
// backfill (actions/backfill/backfill.go)
// ---------------------------------------------------------------------------------------
int vc_snapshot_set_nominated(vc_snapshot *s, const int32_t *nominated_node) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  s->uploaded = false;  // validated against the node table and shipped by the next upload
  if (!nominated_node) { s->h_nominated.clear(); return VC_OK; }
  s->h_nominated.assign(nominated_node, nominated_node + s->dims.n_tasks);
  return VC_OK;
}

int vc_snapshot_set_backfill(vc_snapshot *s, int32_t n_tasks, const vc_tasks *bt) {
  if (!s) return fail(VC_EINVAL, "null snapshot");
  if (n_tasks < 0 || (n_tasks > 0 && !bt)) return fail(VC_EINVAL, "backfill task list: negative size / null pointer");
  s->uploaded = false;  // the list is validated against the job / class tables by the next upload
  vch::BackfillTasks &b = s->bf;
  const size_t B = (size_t)n_tasks, R = s->dims.n_dims, K = s->dims.n_kdims;
  b.n = n_tasks;
  if (B == 0) return VC_OK;
  if (!bt->resreq || !bt->req_has || !bt->k8s_req || !bt->k8s_nonzero_req || !bt->job || !bt->klass || !bt->role ||
      !bt->priority || !bt->uid_rank)
    return fail(VC_EINVAL, "backfill task list: null array");
  b.req.assign(bt->resreq, bt->resreq + R * B); b.kreq.assign(bt->k8s_req, bt->k8s_req + K * B);
  b.knz.assign(bt->k8s_nonzero_req, bt->k8s_nonzero_req + 2 * B);
  b.has.assign(bt->req_has, bt->req_has + B); b.uid.assign(bt->uid_rank, bt->uid_rank + B);
  b.job.assign(bt->job, bt->job + B); b.klass.assign(bt->klass, bt->klass + B); b.role.assign(bt->role, bt->role + B);
  b.prio.assign(bt->priority, bt->priority + B);
  if (bt->pod_index) b.podidx.assign(bt->pod_index, bt->pod_index + B); else b.podidx.assign(B, -1);
  if (bt->creation_ts) b.ts.assign(bt->creation_ts, bt->creation_ts + B); else b.ts.assign(B, 0);
  return VC_OK;
}

int vc_backfill_run(vc_snapshot *s, vc_result **out) {
  if (!s || !out) return fail(VC_EINVAL, "null argument");
  if (!s->uploaded) return fail(VC_EINVAL, "vc_snapshot_upload must precede vc_backfill_run");
  if (s->bf_ran) return fail(VC_EINVAL, "vc_backfill_run already ran on this session state (run vc_allocate_run or upload again)");
  const double t0 = now_ms();
  const vc_dims &D = s->dims;
  const size_t N = D.n_nodes, T = D.n_tasks, J = D.n_jobs, Q = D.n_queues, R = D.n_dims, K = D.n_kdims, NR = D.n_roles;
  const size_t B = (size_t)s->bf.n;
  vc_result *r = new vc_result();
  r->stats.upload_ms = s->upload_ms;
  if (B > 0 && s->dc.to_find > 0 && s->npc > 4 * s->block) { delete r; return fail(VC_EUNSUPPORTED, "feasible-node sampling: more than 4 x blockDim nodes per CTA"); }
  if (B > 0 && s->dc.nta_on) {
    // hypernode binpacking of a BestEffort pod: every term is skipped unless a weighted resource is requested
    // (network_topology_aware.go:507-520), i.e. unless "pods" is listed in hypernode.binpack.resources
    for (size_t t = 0; t < B; ++t)
      for (size_t d = 0; d < R; ++d)
        if ((d < 2 || ((s->bf.has[t] >> d) & 1u)) && s->bf.req[d * B + t] >= vch::kMinRes && s->dc.nta_dim_weight[d] >= 0) {
          delete r;
          return fail(VC_EUNSUPPORTED, "backfill: network-topology-aware weighs a resource (dimension %zu) BestEffort pods request", d);
        }
  }
  if (s->dd.node_begin != 0 || s->dd.node_end != (int)N) { delete r; return fail(VC_EUNSUPPORTED, "the backfill engine runs on the full node axis"); }
  if (B == 0) { *out = r; return VC_OK; }
  const vch::BackfillTasks &bf = s->bf;
  const vch::BackfillKeep &bk = s->bk;
  const vc_conf &conf = s->conf;

  // ---- 1 + 2. session state after allocate and pickUpPendingTasks (backfill.go:118-199): vc_host.hpp ----
  vch::BackfillPick pick = vch::backfill_pick(conf, s->alloc_ran, R, T, J, Q, B, s->dc.has_drf != 0, s->dc.has_proportion != 0, s->total,
                                              s->total_has, bf, bk, s->last_dec.data(), s->last_dec.size(), s->ek.t_job.data(),
                                              s->ek.t_req.data(), s->ek.t_has.data(), s->qattr);
  const std::vector<int32_t> &order = pick.order, &j_ready = pick.j_ready, &r_occ = pick.r_occ;
  const std::vector<int> &visit_job = pick.visit_job, &visit_begin = pick.visit_begin;
  auto is_ready = [&](int j) { return j_ready[j] + bk.j_pbe[j] >= bk.j_min[j]; };  // job_info.go:1169
  const size_t n = order.size();

  // ---- 3. (class, request) groups of the verdict cache; the plugin's state-independent entry per node ----
  std::vector<uint32_t> has_x(bf.has);
  if (s->dc.nta_plugin)
    for (size_t t = 0; t < B; ++t)
      if (!s->h_job_soft.empty() && s->h_job_soft[bf.job[t]]) has_x[t] |= VC_HAS_TOPO_TASK;
  std::vector<double> nta_static;
  if (s->dc.nta_on) {  // batchNodeOrderFnForNormalPods :462-496 with every hypernode score 0
    nta_static.resize(N);
    const int L = s->dc.nta_L;
    for (size_t nn = 0; nn < N; ++nn) {
      double total = 0.0;
      for (int l = 0; l < L; ++l) {
        const int h = s->has_topo ? s->h_member[(size_t)l * N + nn] : 0;
        total += s->dc.tier_w[l] * (h < 0 ? 1.0 : 0.0);
      }
      const double sc = total / s->dc.tier_w_total;
      nta_static[nn] = (double)VC_MAX_NODE_SCORE * (double)s->dc.nta_weight * sc;
    }
  }
  std::vector<int32_t> group(B, 0);
  {
    std::unordered_map<std::string, int> index;
    std::string key;
    for (size_t t = 0; t < B; ++t) {
      key.clear();
      key.append(reinterpret_cast<const char *>(&bf.klass[t]), 4);
      key.append(reinterpret_cast<const char *>(&has_x[t]), 4);
      for (size_t d = 0; d < R; ++d) key.append(reinterpret_cast<const char *>(&bf.req[d * B + t]), 8);
      for (size_t k = 0; k < K; ++k) key.append(reinterpret_cast<const char *>(&bf.kreq[k * B + t]), 8);
      for (size_t k = 0; k < 2; ++k) key.append(reinterpret_cast<const char *>(&bf.knz[k * B + t]), 8);
      group[t] = index.emplace(key, (int)index.size()).first->second;
    }
  }

  // ---- 4. device buffers: one slab ----
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t off = 0;
  const size_t o_req = off; off += al(R * B * 8);
  const size_t o_kreq = off; off += al(K * B * 8);
  const size_t o_knz = off; off += al(2 * B * 8);
  const size_t o_has = off; off += al(B * 4);
  const size_t o_klass = off; off += al(B * 4);
  const size_t o_group = off; off += al(B * 4);
  const size_t o_order = off; off += al(std::max<size_t>(n, 1) * 4);
  const size_t o_nta = off; off += al(nta_static.size() * 8);
  const size_t in_bytes = off;
  const size_t o_node = off; off += al(std::max<size_t>(n, 1) * 4);
  const size_t o_score = off; off += al(std::max<size_t>(n, 1) * 8);
  const size_t o_last = off; off += al(4);
  const size_t o_prof = off; off += al(10 * 8);
  if (s->d_bf_bytes < off) {
    if (s->d_bf) cudaFree(s->d_bf);
    s->d_bf = nullptr; s->d_bf_bytes = 0;
    if (cudaMalloc(&s->d_bf, off) != cudaSuccess) { delete r; return fail(VC_ENOMEM, "backfill buffers (%zu bytes)", off); }
    s->d_bf_bytes = off;
  }
  std::vector<unsigned char> stage(in_bytes, 0);
  std::memcpy(stage.data() + o_req, bf.req.data(), R * B * 8);
  std::memcpy(stage.data() + o_kreq, bf.kreq.data(), K * B * 8);
  std::memcpy(stage.data() + o_knz, bf.knz.data(), 2 * B * 8);
  std::memcpy(stage.data() + o_has, has_x.data(), B * 4);
  if (!nta_static.empty()) std::memcpy(stage.data() + o_nta, nta_static.data(), nta_static.size() * 8);
  std::memcpy(stage.data() + o_klass, bf.klass.data(), B * 4);
  std::memcpy(stage.data() + o_group, group.data(), B * 4);
  if (n) std::memcpy(stage.data() + o_order, order.data(), n * 4);
  auto bail = [&](cudaError_t e, const char *what) { delete r; return fail(VC_ECUDA, "%s: %s", what, cudaGetErrorString(e)); };
  cudaError_t e = cudaMemcpyAsync(s->d_bf, stage.data(), in_bytes, cudaMemcpyHostToDevice, s->stream);
  if (e != cudaSuccess) return bail(e, "backfill H2D");
  if (!s->alloc_ran) {  // no allocate action in this cycle: start from the opening node state
    const struct { void *dst; const void *src; size_t bytes; } cp[] = {
        {s->w_idle, s->n_idle.d(s->in), R * N * 8}, {s->w_used, s->n_used.d(s->in), R * N * 8},
        {s->w_pip, s->n_pip.d(s->in), R * N * 8},   {s->w_kreq, s->n_kreq.d(s->in), K * N * 8},
        {s->w_knz, s->n_knz.d(s->in), 2 * N * 8},   {s->w_pod_count, s->n_pod_count.d(s->in), N * 4}};
    for (const auto &c : cp)
      if ((e = cudaMemcpyAsync(c.dst, c.src, c.bytes, cudaMemcpyDeviceToDevice, s->stream)) != cudaSuccess) return bail(e, "node state copy");
  }
  float kms = 0;
  std::vector<int32_t> h_node(n, -1);
  std::vector<double> h_score(n, 0.0);
  int32_t h_last = s->last_idx_cur;
  long long h_prof[10] = {0};
  if (n > 0) {
    const int G = s->n_cta;
    const size_t mbox_bytes = kMboxBytes;
    if (!s->mbox && (e = cudaMalloc(&s->mbox, mbox_bytes)) != cudaSuccess) return bail(e, "mailbox");
    if ((e = cudaMemsetAsync(s->mbox, 0, mbox_bytes, s->stream)) != cudaSuccess) return bail(e, "mailbox reset");
    K2Params p;
    std::memset(&p, 0, sizeof p);
    p.d = s->dd; p.c = s->dc; p.npc = s->npc; p.n_cta = G;
    p.alloc = s->n_alloc.d(s->in); p.kalloc = s->n_kalloc.d(s->in);
    p.idle = s->w_idle; p.used = s->w_used; p.kreq = s->w_kreq; p.knz = s->w_knz;
    p.max_tasks = s->n_max_tasks.d(s->in); p.pod_count = s->w_pod_count; p.cstat = s->cstat;
    p.mbox = s->mbox;
    p.mbox2 = s->mbox + kMbox2Offset;
    BackfillParams bp;
    unsigned char *base = static_cast<unsigned char *>(s->d_bf);
    bp.n = (int)n; bp.B = (int)B;
    bp.order = reinterpret_cast<const int32_t *>(base + o_order);
    bp.req = reinterpret_cast<const double *>(base + o_req); bp.kreq = reinterpret_cast<const double *>(base + o_kreq);
    bp.knz = reinterpret_cast<const double *>(base + o_knz); bp.has = reinterpret_cast<const uint32_t *>(base + o_has);
    bp.klass = reinterpret_cast<const int32_t *>(base + o_klass); bp.group = reinterpret_cast<const int32_t *>(base + o_group);
    bp.out_node = reinterpret_cast<int32_t *>(base + o_node); bp.out_score = reinterpret_cast<double *>(base + o_score);
    bp.nta_static = nta_static.empty() ? nullptr : reinterpret_cast<const double *>(base + o_nta);
    bp.prof = g_tun.prof ? reinterpret_cast<long long *>(base + o_prof) : nullptr;
    bp.spec_depth = (s->rows_integral && !g_tun.backfill_depth1) ? 32 : 1;
    bp.last_idx0 = s->last_idx_cur; bp.out_last_idx = reinterpret_cast<int32_t *>(base + o_last);
    const void *kfn = s->dc.to_find > 0 ? (const void *)k_backfill<true, true>
                    : s->dc.soft_active ? (const void *)k_backfill<true> : (const void *)k_backfill<false>;
    const size_t smem = ((sizeof(BfCtl) + 15) & ~(size_t)15) + (3 * R + 2 * K + 2) * (size_t)s->npc * 8 +
                        (size_t)s->npc * (4 + 4) + 8 + (size_t)s->npc * (8 + 4 + 1 + 1) + 8 + (size_t)G * (8 + 4 + 4) + 64;
    if (int rc = check_smem(kfn, smem, "backfill kernel")) { delete r; return rc; }
    if ((e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return bail(e, "backfill smem");
    int max_blocks = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_blocks, kfn, s->block, smem)) != cudaSuccess) return bail(e, "occupancy");
    if (max_blocks * g_sm_count < G) { delete r; return fail(VC_EUNSUPPORTED, "backfill kernel cannot be co-resident: %d CTAs x %zu B smem", G, smem); }
    void *args[] = {&p, &bp};
    cudaEventRecord(s->ev0, s->stream);
    if ((e = cudaLaunchCooperativeKernel(kfn, dim3(G), dim3(s->block), args, smem, s->stream)) != cudaSuccess) return bail(e, "backfill launch");
    g_launches++;
    cudaEventRecord(s->ev1, s->stream);
    if ((e = cudaMemcpyAsync(h_node.data(), base + o_node, n * 4, cudaMemcpyDeviceToHost, s->stream)) != cudaSuccess) return bail(e, "backfill D2H");
    if ((e = cudaMemcpyAsync(h_score.data(), base + o_score, n * 8, cudaMemcpyDeviceToHost, s->stream)) != cudaSuccess) return bail(e, "backfill D2H");
    if ((e = cudaMemcpyAsync(&h_last, base + o_last, 4, cudaMemcpyDeviceToHost, s->stream)) != cudaSuccess) return bail(e, "backfill D2H");
    if (bp.prof && (e = cudaMemcpyAsync(h_prof, base + o_prof, 10 * 8, cudaMemcpyDeviceToHost, s->stream)) != cudaSuccess) return bail(e, "backfill D2H");
  }
  if ((e = cudaStreamSynchronize(s->stream)) != cudaSuccess) return bail(e, "backfill kernel");
  if (n > 0) cudaEventElapsedTime(&kms, s->ev0, s->ev1);
  for (int k = 0; k < 8; ++k) r->stats.prof_cycles[k] = h_prof[k];
  if (g_tun.prof && n > 0)
    fprintf(stderr, "k_backfill CTA 0: top barrier -> record seen (bystander, summed) %lld cycles, top barrier -> record sent "
                    "(republisher, summed) %lld cycles\n", h_prof[8], h_prof[9]);
  s->bf_ran = true;
  if (s->dc.to_find > 0) s->last_idx_cur = h_last;
  r->stats.last_processed_node_index = s->last_idx_cur;

  // ---- 5. the result: one visit per job in pick order ----
  const bool gang_ready = vch::plugin_enabled(conf, VC_PLUGIN_GANG, VC_EN_JOB_READY);
  for (size_t v = 0; v < visit_job.size(); ++v) {
    const int j = visit_job[v];
    bool ready = true;  // ssn.JobReady (session_plugins.go:428-446; gang.go:183-189): unchanged by backfill itself, a
    if (gang_ready) {   // placed BestEffort task moves from PendingBestEffortTaskNum to ReadyTaskNum
      bool task_ready = true;  // CheckTaskReady, job_info.go:1024-1036
      if (!(bk.j_min[j] < bk.j_taskmintotal[j]))
        for (int rr = bk.j_roleoff[j]; rr < bk.j_roleoff[j + 1] && task_ready; ++rr)
          if ((bk.r_flags[rr] & VC_ROLE_IN_MIN_MAP) && r_occ[rr] < bk.r_min[rr]) task_ready = false;
      ready = task_ready && is_ready(j);
    }
    vc_visit vis;
    vis.job = j; vis.outcome = ready ? VC_VISIT_COMMIT : VC_VISIT_KEEP;
    vis.first_op = (int32_t)r->decisions.size(); vis.n_ops = 0;
    for (int k = visit_begin[v]; k < visit_begin[v + 1]; ++k) {
      if (h_node[k] < 0) { r->fit_errors.push_back(order[k]); continue; }
      vc_decision dcs;
      dcs.task = order[k]; dcs.node = h_node[k]; dcs.kind = VC_OP_ALLOCATE; dcs.visit = (int32_t)r->visits.size(); dcs.score = h_score[k];
      r->decisions.push_back(dcs);
      vis.n_ops += 1;
    }
    r->visits.push_back(vis);
  }
  r->stats.commit_ms = kms;
  r->stats.total_ms = now_ms() - t0;
  r->stats.h2d_bytes = (int64_t)in_bytes;
  r->stats.d2h_bytes = (int64_t)n * 12;
  r->stats.kernel_launches = n > 0 ? 1 : 0;
  r->stats.n_steps = (int32_t)n;
  *out = r;
  (void)NR;
  return VC_OK;
}

// ---------------------------------------------------------------------------------------
// dense pass (K1)
// ---------------------------------------------------------------------------------------
__global__ void k_best_to_tasks(const int32_t *task_group, const double *g_best_score, const int32_t *g_best_node,
                                double *best_score, int32_t *best_node, int T);

static int dense_prepare(vc_snapshot *s) {
  if (s->dense_ready) return VC_OK;
  free_dense(s);
  const vc_dims &D = s->dims;
  const size_t T = D.n_tasks, R = D.n_dims, K = D.n_kdims, N = D.n_nodes;
  const int nloc = s->dd.node_end - s->dd.node_begin;
  const std::vector<int32_t> &group_of = s->h_group_of;
  const std::vector<int32_t> &rep = s->group_rep;
  const size_t G = rep.size();
  s->n_groups = (int)G;
  std::vector<double> g_req(R * G), g_kreq(K * G), g_knz(2 * G);
  std::vector<uint32_t> g_has(G);
  std::vector<int32_t> g_class(G), g_count(G + 1, 0);
  for (size_t g = 0; g < G; ++g) {
    int t = rep[g];
    for (size_t d = 0; d < R; ++d) g_req[d * G + g] = s->ek.t_req[d * T + t];
    for (size_t k = 0; k < K; ++k) g_kreq[k * G + g] = s->ek.t_kreq[k * T + t];
    for (size_t k = 0; k < 2; ++k) g_knz[k * G + g] = s->ek.t_knz[k * T + t];
    g_has[g] = s->ek.t_has[t] | ((s->topo_any && s->h_job_soft[s->ek.t_job[t]]) ? VC_HAS_TOPO_TASK : 0u);
    g_class[g] = s->ek.t_class[t];
  }
  for (size_t t = 0; t < T; ++t) g_count[group_of[t] + 1]++;
  for (size_t g = 0; g < G; ++g) g_count[g + 1] += g_count[g];
  std::vector<int32_t> group_tasks(T), fill(g_count.begin(), g_count.end() - 1);
  for (size_t t = 0; t < T; ++t) group_tasks[fill[group_of[t]]++] = (int32_t)t;
  // work items: a few rows of one group each
  int chunk = 16;  // rows per work item: more, smaller CTAs keep the copy engines of all SMs busy to the end
  if (g_tun.expand_rows > 0) chunk = g_tun.expand_rows;
  std::vector<int32_t> wg, wb, we;
  for (size_t g = 0; g < G; ++g)
    for (int b = g_count[g]; b < g_count[g + 1]; b += chunk) {
      wg.push_back((int32_t)g); wb.push_back(b); we.push_back(std::min(b + chunk, g_count[g + 1]));
    }
  // launch order = row order of the matrix: concurrent CTAs then write one contiguous band of task rows (tasks of a
  // job are consecutive and share their group), which keeps the HBM write stream and the TLB local
  {
    std::vector<int> ord(wg.size());
    for (size_t i = 0; i < ord.size(); ++i) ord[i] = (int)i;
    std::sort(ord.begin(), ord.end(), [&](int a, int b) { return group_tasks[wb[a]] < group_tasks[wb[b]]; });
    std::vector<int32_t> wg2(wg.size()), wb2(wg.size()), we2(wg.size());
    for (size_t i = 0; i < ord.size(); ++i) { wg2[i] = wg[ord[i]]; wb2[i] = wb[ord[i]]; we2[i] = we[ord[i]]; }
    wg.swap(wg2); wb.swap(wb2); we.swap(we2);
  }
  s->n_work = (int)wg.size();
  s->rows_per_item = chunk;
  auto up = [&](auto *&dptr, const auto &vec) -> int {
    using E = typename std::remove_reference_t<decltype(vec)>::value_type;
    void *q = nullptr;
    CUDA_TRY(cudaMalloc(&q, std::max<size_t>(16, vec.size() * sizeof(E))));
    if (!vec.empty()) CUDA_TRY(cudaMemcpyAsync(q, vec.data(), vec.size() * sizeof(E), cudaMemcpyHostToDevice, s->stream));
    dptr = reinterpret_cast<std::remove_reference_t<decltype(dptr)>>(q);
    return VC_OK;
  };
  int rc;
  if ((rc = up(s->g_req, g_req)) || (rc = up(s->g_kreq, g_kreq)) || (rc = up(s->g_knz, g_knz)) || (rc = up(s->g_has, g_has)) ||
      (rc = up(s->g_class, g_class)) || (rc = up(s->work_group, wg)) || (rc = up(s->work_begin, wb)) ||
      (rc = up(s->work_end, we)) || (rc = up(s->group_tasks, group_tasks)) || (rc = up(s->task_group, group_of)))
    return rc;
  CUDA_TRY(cudaStreamSynchronize(s->stream));  // the staging vectors die with this scope
  const int nparts = (nloc + 255) / 256;
  CUDA_TRY(cudaMalloc(&s->g_order, std::max<size_t>(16, G * (size_t)nloc * 8)));
  CUDA_TRY(cudaMalloc(&s->g_cat, std::max<size_t>(16, G * (size_t)nloc)));
  CUDA_TRY(cudaMalloc(&s->g_stats, std::max<size_t>(16, G * 4 * 4)));
  CUDA_TRY(cudaMalloc(&s->g_best_score, std::max<size_t>(16, G * 8)));
  CUDA_TRY(cudaMalloc(&s->g_best_node, std::max<size_t>(16, G * 4)));
  CUDA_TRY(cudaMalloc(&s->part_score, std::max<size_t>(16, G * (size_t)std::max(nparts, 1) * 8)));
  CUDA_TRY(cudaMalloc(&s->part_node, std::max<size_t>(16, G * (size_t)std::max(nparts, 1) * 4)));
  CUDA_TRY(cudaMalloc(&s->best_score, std::max<size_t>(16, T * 8)));
  CUDA_TRY(cudaMalloc(&s->best_node, std::max<size_t>(16, T * 4)));
  if (s->dc.nta_on) {
    if (s->hn_score) cudaFree(s->hn_score);
    s->hn_score = nullptr;
    CUDA_TRY(cudaMalloc(&s->hn_score, std::max<size_t>(16, G * (size_t)s->hn_H * 8)));
  }
  s->mw32_logical = (int)(2 * ((N + 63) / 64));
  s->mw32 = (s->mw32_logical + 3) & ~3;
  s->dense_ready = true;
  return VC_OK;
}

static K1Params dense_params(vc_snapshot *s) {
  K1Params p;
  std::memset(&p, 0, sizeof p);
  p.d = s->dd; p.c = s->dc;
  p.alloc = s->n_alloc.d(s->in); p.idle = s->n_idle.d(s->in); p.used = s->n_used.d(s->in);
  p.rel = s->n_rel.d(s->in); p.pip = s->n_pip.d(s->in); p.kalloc = s->n_kalloc.d(s->in);
  p.kreq = s->n_kreq.d(s->in); p.knz = s->n_knz.d(s->in);
  p.max_tasks = s->n_max_tasks.d(s->in); p.pod_count = s->n_pod_count.d(s->in); p.cstat = s->cstat;
  p.n_groups = s->n_groups; p.g_req = s->g_req; p.g_kreq = s->g_kreq; p.g_knz = s->g_knz; p.g_has = s->g_has;
  p.g_class = s->g_class; p.g_order = s->g_order; p.g_cat = s->g_cat; p.g_stats = s->g_stats;
  p.g_best_score = s->g_best_score; p.g_best_node = s->g_best_node;
  p.n_work = s->n_work; p.work_group = s->work_group; p.work_begin = s->work_begin; p.work_end = s->work_end;
  p.group_tasks = s->group_tasks; p.mask_out = s->mask_out; p.score_out = s->score_out;
  p.best_score = s->best_score; p.best_node = s->best_node; p.mw32 = s->mw32;
  p.hn_H = s->hn_H; p.hn_member = s->hn_member.d(s->in); p.hn_alloc = s->hn_alloc.d(s->in);
  p.hn_used = s->hn_used0.d(s->in); p.hn_score = s->hn_score;
  return p;
}

int vc_dense_begin(vc_snapshot *s) {
  if (!s || !s->uploaded) return fail(VC_EINVAL, "snapshot not uploaded");
  if (s->topo_any)
    for (size_t j = 0; j < s->h_job_soft.size(); ++j)
      if (s->h_job_soft[j] && s->h_job_alloc[j] >= 0)
        return fail(VC_EUNSUPPORTED, "dense pass: job %zu is a soft-mode topology job with an allocated hypernode; its pods are "
                                     "scored per job inside the commit kernel only", j);
  int rc = dense_prepare(s);
  if (rc) return rc;
  const int nloc = s->dd.node_end - s->dd.node_begin;
  CUDA_TRY(cudaMemsetAsync(s->g_stats, 0, std::max<size_t>(16, (size_t)s->n_groups * 16), s->stream));
  if (nloc > 0 && s->n_groups > 0) {
    K1Params p = dense_params(s);
    LAUNCH_Y_SLICED(k_group_eval, (nloc + 255) / 256, s->n_groups, 256, 0, s->stream, p);
    g_launches++;
    if (s->dc.nta_on) {
      LAUNCH_Y_SLICED(k_hn_scores, (s->hn_H + 127) / 128, s->n_groups, 128, 0, s->stream, p);
      g_launches++;
    }
    CUDA_TRY(cudaGetLastError());
  }
  return VC_OK;
}

int vc_dense_stats(vc_snapshot *s, int32_t **stats_dev_out, int32_t *count_out) {
  if (!s || !s->dense_ready) return fail(VC_EINVAL, "vc_dense_begin first");
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  *stats_dev_out = s->g_stats;
  *count_out = s->n_groups * 4;
  return VC_OK;
}

int vc_dense_finish(vc_snapshot *s, int materialize) {
  if (!s || !s->dense_ready) return fail(VC_EINVAL, "vc_dense_begin first");
  const vc_dims &D = s->dims;
  const size_t T = D.n_tasks, N = D.n_nodes;
  const int nloc = s->dd.node_end - s->dd.node_begin;
  if (materialize && !s->matrix_allocated) {
    CUDA_TRY(cudaMalloc(&s->score_out, std::max<size_t>(16, T * N * 8)));
    CUDA_TRY(cudaMalloc(&s->mask_out, std::max<size_t>(16, T * (size_t)s->mw32 * 4)));
    CUDA_TRY(cudaMemsetAsync(s->score_out, 0, std::max<size_t>(16, T * N * 8), s->stream));
    CUDA_TRY(cudaMemsetAsync(s->mask_out, 0, std::max<size_t>(16, T * (size_t)s->mw32 * 4), s->stream));
    s->matrix_allocated = true;
  }
  K1Params p = dense_params(s);
  const int nparts = std::max(1, (nloc + 255) / 256);
  if (s->n_groups > 0) {
    if (nloc > 0) {
      LAUNCH_Y_SLICED(k_group_best_partial, nparts, s->n_groups, 256, 0, s->stream, p, s->part_score, s->part_node);
      g_launches++;
    } else {
      CUDA_TRY(cudaMemsetAsync(s->part_node, 0xff, (size_t)s->n_groups * nparts * 4, s->stream));
    }
    k_group_best_final<<<(s->n_groups + 127) / 128, 128, 0, s->stream>>>(p, s->part_score, s->part_node, nparts);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
  }
  if (materialize && s->n_work > 0 && nloc > 0) {
    if ((N % 2) == 0 && (s->dd.node_begin % 128) == 0 && !g_tun.expand_plain) {
      // bulk-copy variant: final rows of the groups first (G x Nloc evaluations), then one streaming kernel
      s->mwg = ((nloc + 127) / 128) * 4;
      if (!s->g_final) {
        CUDA_TRY(cudaMalloc(&s->g_final, std::max<size_t>(16, (size_t)s->n_groups * nloc * 8)));
        CUDA_TRY(cudaMalloc(&s->g_maskw, std::max<size_t>(16, (size_t)s->n_groups * s->mwg * 4)));
      }
      CUDA_TRY(cudaMemsetAsync(s->g_maskw, 0, std::max<size_t>(16, (size_t)s->n_groups * s->mwg * 4), s->stream));
      LAUNCH_Y_SLICED(k_group_final, (nloc + 255) / 256, s->n_groups, 256, 0, s->stream, p, s->g_final, s->g_maskw, s->mwg);
      g_launches++;
      // node chunks of <= 8192 nodes (64 KB of scores) so several CTAs share an SM
      int max_chunk = 8192;
      if (g_tun.expand_chunk > 0) max_chunk = std::max(128, g_tun.expand_chunk / 128 * 128);
      const int nchunks = (nloc + max_chunk - 1) / max_chunk;
      const int chunk = (((nloc + nchunks - 1) / nchunks) + 127) & ~127;
      const size_t smem = (size_t)chunk * 8 + 16;
      CUDA_TRY(cudaFuncSetAttribute(k_group_expand_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int rows_cap = std::max(1, std::min(s->rows_per_item, (int)(96 * 1024 / std::max(16, s->mw32 * 4))));
      const size_t msmem = (size_t)rows_cap * s->mw32 * 4 + 16;
      CUDA_TRY(cudaFuncSetAttribute(k_mask_expand_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
      CUDA_TRY(cudaEventRecord(s->ev1, s->stream));
      LAUNCH_Y_SLICED(k_group_expand_bulk, (nloc + chunk - 1) / chunk, s->n_work, 256, smem, s->stream, p, chunk, s->g_final, s->g_maskw, s->mwg);
      k_mask_expand_bulk<<<(unsigned)s->n_work, 128, msmem, s->stream>>>(p, s->g_maskw, s->mwg, rows_cap);
      g_launches++;
    } else {
      CUDA_TRY(cudaEventRecord(s->ev1, s->stream));
      LAUNCH_Y_SLICED(k_group_expand, (nloc + 511) / 512, s->n_work, 256, 0, s->stream, p);
    }
    g_launches++;
    CUDA_TRY(cudaEventRecord(s->ev2, s->stream));
    CUDA_TRY(cudaGetLastError());
  }
  if (T > 0) {
    k_best_to_tasks<<<(unsigned)((T + 255) / 256), 256, 0, s->stream>>>(s->task_group, s->g_best_score, s->g_best_node,
                                                                       s->best_score, s->best_node, (int)T);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
  }
  return VC_OK;
}

// per-task best = best of the task's group
__global__ void k_best_to_tasks(const int32_t *task_group, const double *g_best_score, const int32_t *g_best_node,
                                double *best_score, int32_t *best_node, int T) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  int g = task_group[t];
  best_score[t] = g_best_score[g];
  best_node[t] = g_best_node[g];
}

int vc_dense_best(vc_snapshot *s, double **best_score_dev_out, int32_t **best_node_dev_out) {
  if (!s || !s->dense_ready) return fail(VC_EINVAL, "vc_dense_begin first");
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  *best_score_dev_out = s->best_score;
  *best_node_dev_out = s->best_node;
  return VC_OK;
}

int vc_dense_fetch(vc_snapshot *s, uint64_t *mask_out, double *score_out, double *best_score, int32_t *best_node) {
  if (!s || !s->dense_ready) return fail(VC_EINVAL, "vc_dense_begin first");
  const size_t T = s->dims.n_tasks, N = s->dims.n_nodes;
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if ((mask_out || score_out) && !s->matrix_allocated) return fail(VC_EINVAL, "matrix was not materialised");
  if (mask_out && T > 0)
    CUDA_TRY(cudaMemcpy2D(mask_out, (size_t)s->mw32_logical * 4, s->mask_out, (size_t)s->mw32 * 4, (size_t)s->mw32_logical * 4, T,
                          cudaMemcpyDeviceToHost));
  if (score_out) CUDA_TRY(cudaMemcpy(score_out, s->score_out, T * N * 8, cudaMemcpyDeviceToHost));
  if (best_score) CUDA_TRY(cudaMemcpy(best_score, s->best_score, T * 8, cudaMemcpyDeviceToHost));
  if (best_node) CUDA_TRY(cudaMemcpy(best_node, s->best_node, T * 4, cudaMemcpyDeviceToHost));
  return VC_OK;
}

int vc_score_matrix(vc_snapshot *s, uint64_t *mask_out, double *score_out, double *best_score, int32_t *best_node) {
  int rc = vc_dense_begin(s);
  if (rc) return rc;
  if ((rc = vc_dense_finish(s, 1))) return rc;
  return vc_dense_fetch(s, mask_out, score_out, best_score, best_node);
}

int vc_score_matrix_device(vc_snapshot *s, int repeats, double *kernel_ms_out, int64_t *algorithmic_bytes_out) {
  if (repeats < 1) repeats = 1;
  double tot = 0, exp_tot = 0;
  for (int i = 0; i < repeats; ++i) {
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaEventRecord(s->ev0, s->stream));
    int rc = vc_dense_begin(s);
    if (rc) return rc;
    if ((rc = vc_dense_finish(s, 1))) return rc;
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, s->ev0, s->ev2);
    cudaEventElapsedTime(&b, s->ev1, s->ev2);
    if (i == 0 && repeats > 1) continue;  // first pass allocates + zero-fills the matrix
    tot += a;
    exp_tot += b;
  }
  const int used = repeats > 1 ? repeats - 1 : 1;
  if (kernel_ms_out) { kernel_ms_out[0] = tot / used; kernel_ms_out[1] = exp_tot / used; }
  if (algorithmic_bytes_out) {
    const vc_dims &D = s->dims;
    const int64_t T = D.n_tasks, R = D.n_dims, Wl = D.label_words, Wt = D.taint_words;
    const int64_t nloc = s->dd.node_end - s->dd.node_begin;
    // SURVEY §8(d): T*N*(8 + 1/8) + T*(R*8 + 8*Wc) + N*(5*R*8 + 8*(Wl+Wt) + 16), Wc = 4 class words
    *algorithmic_bytes_out = T * nloc * 8 + T * nloc / 8 + T * (R * 8 + 8 * 4) + nloc * (5 * R * 8 + 8 * (Wl + Wt) + 16);
  }
  return VC_OK;
}

}  // extern "C"
