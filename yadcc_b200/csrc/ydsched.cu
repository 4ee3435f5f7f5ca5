// ydsched.cu -- host side of the B200-native scheduler hot path and its C ABI
// (include/ydsched.h).  This translation unit owns:
//
//   * the servant registry mirror (strings, digests, leases) -- the part of
//     TaskDispatcher that is string handling, not arithmetic
//     (KeepServantAlive cc:190-220, the expiry decision of OnExpirationTimer
//     cc:503-516, RunningTaskBookkeeper);
//   * the topology builder: digest<->servant components, per-component digest
//     membership bit tables, requestor-ip -> servant CSR;
//   * the launch sequences for the kernels in slots.cuh / solve_rowscan.cuh /
//     tasks.cuh.  All arithmetic of the hot path (eligibility, capacity,
//     utilisation, pick, task ids, leases, sweeps) runs on the GPU.
//
// There is no CPU fallback: yd_create fails without an sm_100 device.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "slots.cuh"
#include "radix.cuh"
#include "solve_rowscan.cuh"
#include "solve_stream.cuh"
#include "parallel.cuh"
#include "solve_merge.cuh"
#include "bloom.cuh"
#include "running_index.cuh"
#include "tasks.cuh"
#include "tiny.cuh"
#include "fused.cuh"
#include "filter.cuh"

namespace {

using yd::Counters;
using yd::kNone;

// ---- small helpers ---------------------------------------------------------

// Bumped whenever any device buffer moves: captured graphs hold raw pointers.
static unsigned long long g_buf_generation = 0;

struct DevBuf {  // grow-only device allocation
  void* p = nullptr;
  size_t cap = 0;
  template <class T> T* as() const { return static_cast<T*>(p); }
  void ensure(size_t bytes, bool keep = false, cudaStream_t st = nullptr) {
    if (bytes <= cap) return;
    size_t ncap = std::max(bytes, cap * 2);
    ncap = (ncap + 255) & ~size_t(255);
    void* np = nullptr;
    YD_CUDA_CHECK(cudaMalloc(&np, ncap));
    if (keep && p && cap) YD_CUDA_CHECK(cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, st));
    if (p) {
      YD_CUDA_CHECK(cudaStreamSynchronize(st));
      YD_CUDA_CHECK(cudaFree(p));
    }
    p = np;
    cap = ncap;
    ++g_buf_generation;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    ++g_buf_generation;
  }
};

struct PinBuf {  // grow-only pinned host staging
  void* p = nullptr;
  size_t cap = 0;
  template <class T> T* as() const { return static_cast<T*>(p); }
  void ensure(size_t bytes) {
    if (bytes <= cap) return;
    size_t ncap = std::max(bytes, cap * 2);
    if (p) YD_CUDA_CHECK(cudaFreeHost(p));
    YD_CUDA_CHECK(cudaHostAlloc(&p, ncap, cudaHostAllocDefault));
    cap = ncap;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
};

// yadcc::TryParseSize, yadcc/common/parse_size.cc:25-45.
bool ParseSize(const char* text, uint64_t* out) {
  if (!text) return false;
  size_t len = strlen(text);
  if (len == 0) return false;
  uint64_t scale = 1;
  switch (text[len - 1]) {
    case 'G': scale = 1ull << 30; --len; break;
    case 'M': scale = 1ull << 20; --len; break;
    case 'K': scale = 1ull << 10; --len; break;
    case 'B': --len; break;
    default: break;
  }
  if (len == 0) return false;
  uint64_t v = 0;
  for (size_t i = 0; i != len; ++i) {
    if (text[i] < '0' || text[i] > '9') return false;
    uint64_t nv = v * 10 + uint64_t(text[i] - '0');
    if (nv / 10 != v) return false;
    v = nv;
  }
  *out = v * scale;
  return true;
}

struct ServantHost {  // ServantPersonality + ServantDesc lease fields (h:80-116,184-193)
  int32_t version = 0;
  std::string observed, reported;
  std::vector<uint32_t> envs;  // interned digest ids, heartbeat order (duplicates kept)
  uint32_t nproc = 0, load = 0, max_tasks = 0;
  uint64_t total_mem = 0, avail_mem = 0;
  int32_t priority = 0, reason = 0;
  int64_t discovered_at = 0, expires_at = 0;
};

struct RunningRec {
  uint64_t servant_task_id, task_grant_id;
  std::string servant_location, task_digest;
};

}  // namespace

struct yd_shard_ctx;  // range-sharded queue over several GPUs (shard_host.inc)

struct yd_sched {
  int device = 0;
  yd_shard_ctx* shard = nullptr;
  cudaStream_t st = nullptr;
  uint64_t min_mem = 0;
  uint32_t solver_pref = 0;

  // interning
  std::vector<std::string> envs, ips;
  std::unordered_map<std::string, uint32_t> env_ids, ip_ids;

  // registry mirror
  std::vector<ServantHost> sv;
  std::unordered_map<std::string, uint32_t> loc2pos;
  bool topo_dirty = true, facts_dirty = true;
  // The sorted slot order depends on the heartbeat facts only (key(s, r) is static, slots.cuh): it is built when
  // a capacity fact, a priority or the servant set changes and kept across solves; a solve only filters out the
  // slots servants have filled meanwhile.  (Above kStaticSlotLimit slots the table is rebuilt per solve, clamped
  // to the batch size.)
  bool order_dirty = true, order_static = false;
  size_t order_slot_b = 0;
  unsigned long long order_rebuilds = 0;

  // device servant arrays; state (run/ever) is valid for positions < S_dev
  DevBuf d_nproc, d_load, d_maxt, d_flags, d_ver, d_run, d_ever;
  DevBuf d_run_tmp, d_ever_tmp, d_remap;
  uint32_t S_dev = 0;
  PinBuf h_facts;

  // topology on device
  DevBuf d_env_comp, d_env_local, d_comp_sv_off, d_comp_sv, d_comp_mask_off, d_comp_nwarps, d_envmask,
      d_sv_comp, d_sv_local, d_ip_off, d_ip_sv;
  uint32_t n_comps = 0, n_envs_dev = 0, n_ips_dev = 0, max_warps = 1, max_comp_servants = 0;
  bool wide = false;
  PinBuf h_topo;

  // slot-stream solver state
  DevBuf d_sv_env_off, d_sv_envs, d_comp_mode, d_sv_emask, d_slot_rec;
  bool emask_ok = false;  // every component holds <= 64 digests: d_sv_emask is valid
  DevBuf d_slot_owner, d_sort_k[2], d_sort_v[2];
  // one zero-filled scratch region per solve: radix histograms (one per pass), the class
  // table's u32 arrays, the per-(class, tile) list counts -- a single memset node
  DevBuf d_zero;
  size_t z_hist_off[10] = {}, z_cls_off = 0, z_listcnt_off = 0, z_bytes = 0;
  uint32_t sort_nb = 0;
  cudaStream_t st2 = nullptr, st_copy = nullptr;  // class/rank branch; request upload
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_h2d = nullptr, ev_fin = nullptr;
  uint32_t cls_bound = 16;  // classes the per-class grids are sized for; grows on demand (<= yd::kMaxClasses)
  DevBuf d_list, d_list_bal, d_rcls, d_rrank, d_rank_cnt, d_rq, d_rself;
  // merge solver (solve_merge.cuh): per-slot verdicts and the chunk boundary states
  DevBuf d_slot_pick, d_mst_in, d_mst_out, d_stream_scratch;
  size_t z_merge_off = 0, z_layout_off = 0, z_final_off = 0, z_scan_off = 0;
  uint32_t merge_chunk = 512, merge_rounds = 16, merge_max_chunks = 0, merge_grid = 0, merge_grid_kcap = 0;
  bool merge_chunk_auto = true;  // no YDSCHED_MERGE_CHUNK: 256 slots per chunk up to 262 144 requests, 512 above
  uint32_t stream_debug = 0;   // YDSCHED_STREAM_DEBUG, read once at yd_create
  uint32_t force_stream = 0;   // yd_config.reserved bit 1 / YDSCHED_FORCE_STREAM: no merge solver for self-requests
  bool dump_env = false, debug_env = false, tiny_ok = true;
  bool stream_attr_set = false;
  // fused front kernel (fused.cuh): one persistent launch for the class / rank / list phases and -- `solo` -- the grants
  bool fused_cfg = true;       // yd_config.reserved bit 3 / YDSCHED_NO_FUSED switch it off
  bool solo_hint = true;       // the last batch consisted of data-parallel components only
  uint32_t fused_grid = 0;     // blocks of the fused kernel: one per SM
  uint32_t fused_max_nb = 262144;  // largest batch size class that takes it (YDSCHED_FUSED_MAX_N)
  size_t z_fbar_off = 0;
  DevBuf d_reqs16, d_out8;     // packed upload / download (yd_task_req16, yd_grant8)
  yd::FusedHostIO* h_fio = nullptr;  // mapped pinned record: the solo kernel's result (no copy nodes after it)
  yd::FusedHostIO* d_fio = nullptr;  // its device-side address
  yd::FusedScalars fsc{};            // the call's scalars: kernel parameters of a solo launch ...
  PinBuf h_fsc;                      // ... or (graphed general sequence) copied into d_fsc by the graph's first node
  DevBuf d_fsc;
  // The solo kernel re-initialises the scratch it dirtied (class-table keys, zeroed region) before it ends; while this
  // signature matches the current buffers and layout the next solo solve needs no memset nodes either.
  struct CleanSig { unsigned long long gen = ~0ull; size_t z_cls_off = 0, z_bytes = 0, res_words = 0; const void* zero = nullptr; const void* res = nullptr;
    bool operator==(const CleanSig& o) const { return gen == o.gen && z_cls_off == o.z_cls_off && z_bytes == o.z_bytes && res_words == o.res_words && zero == o.zero && res == o.res; } };
  CleanSig clean_sig;
  bool clean_valid = false;
  bool fused_lite = true;      // YDSCHED_FUSED_NOLITE: the solo kernel's second barrier keeps its leader scans
  bool zero_copy = true;       // YDSCHED_NO_ZEROCOPY: page-locked caller arrays are copied like pageable ones
  bool fused_prof = false;     // YDSCHED_FUSED_PROF: phase stamps of the fused kernel, printed after every solve
  DevBuf d_fused_prof;
  size_t res_words = 0;  // u32 words of res[] in d_res (the class-table keys follow)
  size_t staged_n = 0;   // requests placed in d_reqs by yd_stage_requests

  // lease ring
  DevBuf d_t_exp, d_t_srv, d_t_flags;
  uint64_t ring_cap = 0;
  uint64_t lo = 0, next_id = 0;
  uint32_t id_stride = 1, id_offset = 0;
  uint64_t zombies_ub = 0;

  // per-solve buffers
  DevBuf d_reqs, d_res, d_out, d_blk, d_row_off, d_row_len, d_codes, d_ids, d_ok;
  DevBuf d_counters;
  PinBuf h_counters, h_small;

  // RunningTaskBookkeeper (running_task_bookkeeper.h:41-42): same container, same
  // operation sequence as the reference, hence the same iteration order.
  std::unordered_map<std::string, std::vector<RunningRec>> running;
  std::vector<RunningRec> running_cache;
  std::vector<const char*> personality_envs;  // backing store for yd_get_servant_personality

  // captured solve graphs, keyed by size class
  struct GraphKey {
    uint32_t Nb = 0, S = 0, n_comps = 0, max_comp = 0, cls_bound = 0, solver = 0, wide = 0, merge_rounds = 0, force_stream = 0,
             order_static = 0, variant = 0, packed = 0;
    size_t slot_b = 0;
    unsigned long long gen = 0, topo_gen = 0;  // buffer reallocations; topology rebuilds (n_envs, n_ips, ... are baked in)
    uint64_t ring_cap = 0;
    bool operator==(const GraphKey& o) const {
      return Nb == o.Nb && S == o.S && n_comps == o.n_comps && max_comp == o.max_comp && cls_bound == o.cls_bound &&
             merge_rounds == o.merge_rounds && force_stream == o.force_stream && order_static == o.order_static &&
             solver == o.solver && wide == o.wide && slot_b == o.slot_b && gen == o.gen && topo_gen == o.topo_gen &&
             ring_cap == o.ring_cap && variant == o.variant && packed == o.packed;
    }
  };
  struct GraphEntry {
    GraphKey key;
    cudaGraphExec_t exec = nullptr;
    uint32_t launches = 0;
    // solo graphs (one kernel node): the per-call scalars are kernel parameters, patched before every launch
    cudaGraph_t graph = nullptr;
    cudaGraphNode_t knode = nullptr;
    yd::FusedArgs fargs{};
    uint32_t fgrid = 0;
    size_t fdyn = 0;
  };
  yd::FusedArgs last_fused{};  // what LaunchFused passed last (picked up right after a capture)
  uint32_t last_fused_grid = 0;
  size_t last_fused_dyn = 0;
  bool report_dev = false;     // YDSCHED_REPORT_DEV: the solo kernel's report goes to HBM + a copy node (comparison)
  bool host_prof = false;      // YDSCHED_HOST_PROF: host-side timestamps of a solve, printed
  DevBuf d_report;
  std::vector<GraphEntry> graphs;
  unsigned long long topo_gen = 0;
  bool use_graphs = true;
  DevBuf d_dyn;
  PinBuf h_dyn, h_meta;

  // compilation-cache bloom pre-filter
  DevBuf d_bloom, d_bloom_keys, d_bloom_out;
  uint64_t bloom_bits = 0;
  uint32_t bloom_hashes = 0;

  // in-flight task index (running_index.cuh)
  std::vector<RunningRec> rt_snapshot;
  DevBuf d_rt_bytes, d_rt_off, d_rt_len, d_rt_ids, d_rt_slots, d_rt_keys, d_rt_out;
  DevBuf d_freqs, d_fverdict, d_ftile;  // pre-filtered solve (filter.cuh): the unfiltered queue, verdicts, tile counts
  PinBuf h_fcount;
  cudaEvent_t ev_f[2] = {};
  uint32_t rt_mask = 0;
  size_t rt_distinct = 0;

  cudaEvent_t ev[6] = {};
  yd_solve_stats stats{};
  bool have_stats = false;
  int stats_times_pending = 0;  // 1: events of an eager solve, 2: of a graphed one, not yet turned into milliseconds
  size_t static_bound_cache = 0;  // StaticSlotBound() of the current facts

  yd::ServantArrays arrays() const {
    return yd::ServantArrays{d_nproc.as<uint32_t>(), d_load.as<uint32_t>(), d_maxt.as<uint32_t>(),
                             d_flags.as<uint32_t>(), d_ver.as<int32_t>(), d_run.as<uint32_t>(),
                             d_ever.as<unsigned long long>()};
  }
  yd::TaskRing ring() const {
    return yd::TaskRing{d_t_exp.as<long long>(), d_t_srv.as<uint32_t>(), d_t_flags.as<uint32_t>(),
                        ring_cap - 1, lo, next_id, id_stride, id_offset};
  }

  uint32_t InternEnv(const std::string& k) {
    auto it = env_ids.find(k);
    if (it != env_ids.end()) return it->second;
    uint32_t id = (uint32_t)envs.size();
    envs.push_back(k);
    env_ids.emplace(k, id);
    return id;
  }
  uint32_t InternIp(const std::string& k) {
    auto it = ip_ids.find(k);
    if (it != ip_ids.end()) return it->second;
    uint32_t id = (uint32_t)ips.size();
    ips.push_back(k);
    ip_ids.emplace(k, id);
    return id;
  }

  uint32_t FactFlags(const ServantHost& s) const {
    uint32_t f = 0;
    if (s.priority == YD_PRIORITY_DEDICATED) f |= yd::kFlagDedicated;
    if (s.total_mem != 0 && s.avail_mem < min_mem) f |= yd::kFlagLowMem;  // cc:286-292
    return f;
  }

  void EnsureRing(uint64_t need_ids);
  void SyncServantState();
  void SyncFacts();
  void SyncTopology();
  void FetchCounters();
};

// ---- device state maintenance ------------------------------------------------

// Extend run[] / ever[] with zeros for servants appended since the last sync
// (a new ServantDesc starts with running_tasks = 0, cc:208).
void yd_sched::SyncServantState() {
  uint32_t S = (uint32_t)sv.size();
  if (S <= S_dev) return;
  d_run.ensure(size_t(S) * 4, true, st);
  d_ever.ensure(size_t(S) * 8, true, st);
  YD_CUDA_CHECK(cudaMemsetAsync(d_run.as<uint32_t>() + S_dev, 0, size_t(S - S_dev) * 4, st));
  YD_CUDA_CHECK(cudaMemsetAsync(d_ever.as<unsigned long long>() + S_dev, 0, size_t(S - S_dev) * 8, st));
  S_dev = S;
}

void yd_sched::SyncFacts() {
  if (!facts_dirty) return;
  uint32_t S = (uint32_t)sv.size();
  if (S) {
    h_facts.ensure(size_t(S) * 20);
    uint32_t* h = h_facts.as<uint32_t>();
    uint32_t maxcap = 0;
    for (uint32_t i = 0; i != S; ++i) {
      const ServantHost& s = sv[i];
      h[i] = s.nproc;
      h[S + i] = s.load;
      h[2 * S + i] = s.max_tasks;
      h[3 * S + i] = FactFlags(s);
      h[4 * S + i] = (uint32_t)s.version;
      maxcap = std::max(maxcap, std::min(s.nproc, s.max_tasks));
    }
    static_bound_cache = 0;
    for (uint32_t i = 0; i != S; ++i) static_bound_cache += size_t(std::min(sv[i].nproc, sv[i].max_tasks)) + 1;
    if (wide != (maxcap > yd::kNarrowCapLimit)) order_dirty = true;
    wide = maxcap > yd::kNarrowCapLimit;
    d_nproc.ensure(size_t(S) * 4); d_load.ensure(size_t(S) * 4); d_maxt.ensure(size_t(S) * 4);
    d_flags.ensure(size_t(S) * 4); d_ver.ensure(size_t(S) * 4);
    YD_CUDA_CHECK(cudaMemcpyAsync(d_nproc.p, h, size_t(S) * 4, cudaMemcpyHostToDevice, st));
    YD_CUDA_CHECK(cudaMemcpyAsync(d_load.p, h + S, size_t(S) * 4, cudaMemcpyHostToDevice, st));
    YD_CUDA_CHECK(cudaMemcpyAsync(d_maxt.p, h + 2 * S, size_t(S) * 4, cudaMemcpyHostToDevice, st));
    YD_CUDA_CHECK(cudaMemcpyAsync(d_flags.p, h + 3 * S, size_t(S) * 4, cudaMemcpyHostToDevice, st));
    YD_CUDA_CHECK(cudaMemcpyAsync(d_ver.p, h + 4 * S, size_t(S) * 4, cudaMemcpyHostToDevice, st));
    // h_facts is reused by the next SyncFacts: make sure the DMA has read it.
    YD_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  facts_dirty = false;
}

// Components of the digest<->servant graph, digest membership bit tables and the
// requestor-ip CSR.  Runs only when the servant set or a digest list changed.
void yd_sched::SyncTopology() {
  if (!topo_dirty) return;
  const uint32_t S = (uint32_t)sv.size();
  const uint32_t E = (uint32_t)envs.size();
  // union-find over servants, joined through shared digests
  std::vector<uint32_t> parent(S);
  std::iota(parent.begin(), parent.end(), 0u);
  auto find = [&](uint32_t x) {
    while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
    return x;
  };
  std::vector<uint32_t> env_first(E, kNone);
  for (uint32_t i = 0; i != S; ++i) {
    for (uint32_t e : sv[i].envs) {
      if (env_first[e] == kNone) { env_first[e] = i; continue; }
      uint32_t a = find(env_first[e]), b = find(i);
      if (a != b) parent[std::max(a, b)] = std::min(a, b);
    }
  }
  std::vector<uint32_t> comp_of_root(S, kNone), sv_comp(S, kNone), sv_local(S, kNone);
  std::vector<std::vector<uint32_t>> comp_sv, comp_envs;
  for (uint32_t i = 0; i != S; ++i) {
    if (sv[i].envs.empty()) continue;  // can never be eligible
    uint32_t r = find(i);
    if (comp_of_root[r] == kNone) {
      comp_of_root[r] = (uint32_t)comp_sv.size();
      comp_sv.emplace_back();
      comp_envs.emplace_back();
    }
    uint32_t c = comp_of_root[r];
    sv_comp[i] = c;
    sv_local[i] = (uint32_t)comp_sv[c].size();
    comp_sv[c].push_back(i);
  }
  std::vector<uint32_t> env_comp(E, kNone), env_local(E, kNone);
  for (uint32_t i = 0; i != S; ++i) {
    for (uint32_t e : sv[i].envs) {
      if (env_comp[e] != kNone) continue;
      uint32_t c = sv_comp[i];
      env_comp[e] = c;
      env_local[e] = (uint32_t)comp_envs[c].size();
      comp_envs[c].push_back(e);
    }
  }
  const uint32_t C = (uint32_t)comp_sv.size();
  std::vector<uint32_t> sv_off(C + 1, 0), mask_off(C, 0), nwarps(C, 1), flat_sv;
  size_t mask_bytes = 0;
  max_warps = 1;
  for (uint32_t c = 0; c != C; ++c) {
    sv_off[c] = (uint32_t)flat_sv.size();
    flat_sv.insert(flat_sv.end(), comp_sv[c].begin(), comp_sv[c].end());
    uint32_t w = (uint32_t)((comp_sv[c].size() + 32 * yd::kK - 1) / (32 * yd::kK));
    nwarps[c] = std::max(1u, std::min(w, 32u));  // > 32 warps: only the slot-stream solver applies
    max_warps = std::max(max_warps, nwarps[c]);
    mask_off[c] = (uint32_t)mask_bytes;
    mask_bytes += size_t(comp_envs[c].size()) * nwarps[c] * 32;
  }
  sv_off[C] = (uint32_t)flat_sv.size();
  std::vector<uint8_t> envmask(std::max<size_t>(mask_bytes, 1), 0);
  for (uint32_t i = 0; i != S; ++i) {
    uint32_t c = sv_comp[i];
    if (c == kNone) continue;
    uint32_t l = sv_local[i], T = nwarps[c] * 32;
    if (l / yd::kK >= T) continue;  // component beyond the row-scan solver's 8192 servants: it never reads these masks
    for (uint32_t e : sv[i].envs) {
      envmask[mask_off[c] + size_t(env_local[e]) * T + l / yd::kK] |= uint8_t(1u << (l % yd::kK));
    }
  }
  // requestor-ip CSR: IsNetworkAddressEqual(ip_port, ip) (cc:66-69) holds iff `ip`
  // is a prefix of the observed location that ends right before a ':'.
  std::vector<std::vector<uint32_t>> by_ip(ips.size());
  for (uint32_t i = 0; i != S; ++i) {
    const std::string& loc = sv[i].observed;
    for (size_t k = 0; k < loc.size(); ++k) {
      if (loc[k] != ':') continue;
      uint32_t id = InternIp(loc.substr(0, k));
      if (id >= by_ip.size()) by_ip.resize(id + 1);
      by_ip[id].push_back(i);
    }
  }
  const uint32_t NI = (uint32_t)by_ip.size();
  std::vector<uint32_t> ip_off(NI + 1, 0), ip_sv;
  for (uint32_t k = 0; k != NI; ++k) {
    ip_off[k] = (uint32_t)ip_sv.size();
    ip_sv.insert(ip_sv.end(), by_ip[k].begin(), by_ip[k].end());
  }
  ip_off[NI] = (uint32_t)ip_sv.size();

  auto up = [&](DevBuf& b, const void* src, size_t bytes) {
    b.ensure(std::max<size_t>(bytes, 4));
    if (bytes) YD_CUDA_CHECK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, st));
  };
  up(d_env_comp, env_comp.data(), size_t(E) * 4);
  up(d_env_local, env_local.data(), size_t(E) * 4);
  up(d_comp_sv_off, sv_off.data(), size_t(C + 1) * 4);
  up(d_comp_sv, flat_sv.data(), flat_sv.size() * 4);
  up(d_comp_mask_off, mask_off.data(), size_t(C) * 4);
  up(d_comp_nwarps, nwarps.data(), size_t(C) * 4);
  up(d_envmask, envmask.data(), envmask.size());
  up(d_sv_comp, sv_comp.data(), size_t(S) * 4);
  up(d_sv_local, sv_local.data(), size_t(S) * 4);
  up(d_ip_off, ip_off.data(), size_t(NI + 1) * 4);
  up(d_ip_sv, ip_sv.data(), ip_sv.size() * 4);
  // digest ids per servant (CSR) for class-eligibility tests on the device
  std::vector<uint32_t> env_off(S + 1, 0), env_flat;
  for (uint32_t i = 0; i != S; ++i) {
    env_off[i] = (uint32_t)env_flat.size();
    env_flat.insert(env_flat.end(), sv[i].envs.begin(), sv[i].envs.end());
  }
  env_off[S] = (uint32_t)env_flat.size();
  up(d_sv_env_off, env_off.data(), size_t(S + 1) * 4);
  up(d_sv_envs, env_flat.data(), env_flat.size() * 4);
  // digest membership as a 64-bit word per servant, when every component's digests fit
  emask_ok = true;
  for (uint32_t c = 0; c != C; ++c) emask_ok = emask_ok && comp_envs[c].size() <= 64;
  std::vector<unsigned long long> emask(std::max(S, 1u), 0ull);
  if (emask_ok) {
    for (uint32_t i = 0; i != S; ++i) for (uint32_t e : sv[i].envs) emask[i] |= 1ull << env_local[e];
  }
  up(d_sv_emask, emask.data(), emask.size() * 8);
  std::vector<uint32_t> comp_mode(std::max(C, 1u), 0);
  up(d_comp_mode, comp_mode.data(), comp_mode.size() * 4);
  max_comp_servants = 0;
  for (uint32_t c = 0; c != C; ++c) max_comp_servants = std::max<uint32_t>(max_comp_servants, (uint32_t)comp_sv[c].size());
  YD_CUDA_CHECK(cudaStreamSynchronize(st));  // sources are pageable temporaries
  n_comps = C;
  n_envs_dev = E;
  n_ips_dev = NI;
  topo_dirty = false;
  ++topo_gen;
}

void yd_sched::EnsureRing(uint64_t need_ids) {
  uint64_t need = (next_id - lo) + need_ids;
  if (ring_cap && need <= ring_cap) return;
  uint64_t ncap = ring_cap ? ring_cap : (1ull << 16);
  while (ncap < need * 2) ncap <<= 1;
  DevBuf ne, ns, nf;
  ne.ensure(ncap * 8); ns.ensure(ncap * 4); nf.ensure(ncap * 4);
  YD_CUDA_CHECK(cudaMemsetAsync(nf.p, 0, ncap * 4, st));
  if (ring_cap && next_id > lo) {
    yd::TaskRing nr{ne.as<long long>(), ns.as<uint32_t>(), nf.as<uint32_t>(), ncap - 1, lo, next_id, id_stride, id_offset};
    uint64_t cnt = next_id - lo;
    yd::k_ring_grow<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(ring(), nr);
    YD_CUDA_CHECK(cudaGetLastError());
  }
  YD_CUDA_CHECK(cudaStreamSynchronize(st));
  d_t_exp.release(); d_t_srv.release(); d_t_flags.release();
  d_t_exp = ne; d_t_srv = ns; d_t_flags = nf;
  ring_cap = ncap;
}

void yd_sched::FetchCounters() {
  YD_CUDA_CHECK(cudaMemcpyAsync(h_counters.p, d_counters.p, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  YD_CUDA_CHECK(cudaStreamSynchronize(st));
}

// ---- C ABI -------------------------------------------------------------------

extern "C" {

const char* yd_backend_name(void) { return "cuda-sm100a"; }

int yd_parse_size(const char* text, uint64_t* out_bytes) { return ParseSize(text, out_bytes) ? 1 : 0; }

yd_sched* yd_create(const yd_config* cfg) {
  if (!cfg || cfg->abi_version != YD_ABI_VERSION) return nullptr;
  uint64_t min_mem = 0;
  const char* mm = cfg->servant_min_memory_for_accepting_new_task;
  if (!ParseSize(mm ? mm : "10G", &min_mem)) return nullptr;  // cc:83-87
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) {
    fprintf(stderr, "ydsched: no CUDA device %d (found %d); this backend has no CPU fallback\n",
            cfg->device, ndev);
    return nullptr;
  }
  cudaDeviceProp prop{};
  YD_CUDA_CHECK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major < 10) {
    fprintf(stderr, "ydsched: device %d is sm_%d%d; kernels are built for sm_100a only\n", cfg->device,
            prop.major, prop.minor);
    return nullptr;
  }
  YD_CUDA_CHECK(cudaSetDevice(cfg->device));
  auto* s = new yd_sched;
  s->device = cfg->device;
  s->min_mem = min_mem;
  s->solver_pref = cfg->solver;
  s->id_stride = cfg->id_stride ? cfg->id_stride : 1;
  s->id_offset = cfg->id_stride ? cfg->id_offset : 0;
  s->use_graphs = !(cfg->reserved & 1u) && !getenv("YDSCHED_NO_GRAPH");
  s->force_stream = ((cfg->reserved & 2u) || getenv("YDSCHED_FORCE_STREAM")) ? 1u : 0u;
  if (const char* e = getenv("YDSCHED_STREAM_DEBUG")) s->stream_debug = (uint32_t)atoi(e);
  if (const char* e = getenv("YDSCHED_MERGE_CHUNK")) { s->merge_chunk = std::max(32u, (uint32_t)atoi(e) & ~31u); s->merge_chunk_auto = false; }
  if (const char* e = getenv("YDSCHED_MERGE_ROUNDS")) s->merge_rounds = std::max(2u, (uint32_t)atoi(e));
  s->tiny_ok = !(cfg->reserved & 4u) && !getenv("YDSCHED_NO_TINY");
  s->fused_cfg = !(cfg->reserved & 8u) && !getenv("YDSCHED_NO_FUSED");
  if (const char* e = getenv("YDSCHED_FUSED_MAX_N")) s->fused_max_nb = (uint32_t)std::max(1024, atoi(e));
  YD_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&s->h_fio), sizeof(yd::FusedHostIO), cudaHostAllocMapped));
  memset(s->h_fio, 0, sizeof(yd::FusedHostIO));
  YD_CUDA_CHECK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&s->d_fio), s->h_fio, 0));
  s->zero_copy = getenv("YDSCHED_NO_ZEROCOPY") == nullptr;
  s->fused_lite = getenv("YDSCHED_FUSED_NOLITE") == nullptr;
  s->report_dev = getenv("YDSCHED_REPORT_DEV") != nullptr;
  s->host_prof = getenv("YDSCHED_HOST_PROF") != nullptr;
  s->d_report.ensure(sizeof(yd::FusedHostIO));
  s->fused_prof = getenv("YDSCHED_FUSED_PROF") != nullptr;
  s->d_fused_prof.ensure(128);
  YD_CUDA_CHECK(cudaMemset(s->d_fused_prof.p, 0, 128));
  {
    int sms = 0, per_sm = 0;
    YD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device));
    YD_CUDA_CHECK(cudaFuncSetAttribute(yd::k_fused_front, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    YD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, yd::k_fused_front, 1024, 64 * 1024));
    s->fused_grid = per_sm >= 1 ? (uint32_t)sms : 0u;  // (0: the kernel does not fit an SM -- never on sm_100a; the pipeline is used)
  }
  s->dump_env = getenv("YDSCHED_DUMP") != nullptr;
  s->debug_env = getenv("YDSCHED_DEBUG") != nullptr;
  YD_CUDA_CHECK(cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking));
  YD_CUDA_CHECK(cudaStreamCreateWithFlags(&s->st2, cudaStreamNonBlocking));
  YD_CUDA_CHECK(cudaStreamCreateWithFlags(&s->st_copy, cudaStreamNonBlocking));
  for (auto& e : s->ev) YD_CUDA_CHECK(cudaEventCreate(&e));
  for (auto& e : s->ev_f) YD_CUDA_CHECK(cudaEventCreate(&e));
  YD_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming));
  YD_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
  YD_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_h2d, cudaEventDisableTiming));
  YD_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev_fin, cudaEventDisableTiming));
  s->ips.emplace_back();  // id 0 == YD_IP_NONE == the empty requestor string
  s->ip_ids.emplace("", 0);
  s->d_counters.ensure(sizeof(Counters));
  YD_CUDA_CHECK(cudaMemsetAsync(s->d_counters.p, 0, sizeof(Counters), s->st));
  s->h_counters.ensure(sizeof(Counters));
  s->h_small.ensure(1 << 16);
  s->d_dyn.ensure(sizeof(yd::DynParams));
  s->h_dyn.ensure(sizeof(yd::DynParams));
  s->h_fsc.ensure(sizeof(yd::FusedScalars));
  s->d_fsc.ensure(sizeof(yd::FusedScalars));
  s->h_meta.ensure(64);
  s->EnsureRing(0);
  return s;
}

extern "C" void yd_shard_finalize(yd_sched* s);

void yd_destroy(yd_sched* s) {
  if (!s) return;
  yd_shard_finalize(s);
  cudaSetDevice(s->device);
  cudaStreamSynchronize(s->st);
  for (DevBuf* b : {&s->d_nproc, &s->d_load, &s->d_maxt, &s->d_flags, &s->d_ver, &s->d_run, &s->d_ever,
                    &s->d_run_tmp, &s->d_ever_tmp, &s->d_remap, &s->d_env_comp, &s->d_env_local,
                    &s->d_comp_sv_off, &s->d_comp_sv, &s->d_comp_mask_off, &s->d_comp_nwarps, &s->d_envmask,
                    &s->d_sv_comp, &s->d_sv_local, &s->d_ip_off, &s->d_ip_sv, &s->d_t_exp, &s->d_t_srv,
                    &s->d_t_flags, &s->d_reqs, &s->d_res, &s->d_out, &s->d_blk, &s->d_row_off, &s->d_row_len,
                    &s->d_codes, &s->d_ids, &s->d_ok, &s->d_counters, &s->d_sv_env_off, &s->d_sv_envs,
                    &s->d_comp_mode, &s->d_sv_emask, &s->d_slot_rec, &s->d_slot_owner, &s->d_sort_k[0], &s->d_sort_k[1], &s->d_sort_v[0],
                    &s->d_sort_v[1], &s->d_zero, &s->d_list, &s->d_list_bal, &s->d_rcls, &s->d_rrank, &s->d_rank_cnt, &s->d_rq, &s->d_rself,
                    &s->d_slot_pick, &s->d_mst_in, &s->d_mst_out, &s->d_stream_scratch, &s->d_reqs16, &s->d_out8, &s->d_fused_prof, &s->d_report, &s->d_bloom,
                    &s->d_bloom_keys, &s->d_bloom_out, &s->d_rt_bytes, &s->d_rt_off, &s->d_rt_len, &s->d_rt_ids,
                    &s->d_rt_slots, &s->d_rt_keys, &s->d_rt_out}) {
    b->release();
  }
  for (auto& g : s->graphs) { if (g.exec) cudaGraphExecDestroy(g.exec); if (g.graph) cudaGraphDestroy(g.graph); }
  if (s->h_fio) cudaFreeHost(s->h_fio);
  s->d_dyn.release();
  s->d_fsc.release();
  for (PinBuf* b : {&s->h_facts, &s->h_topo, &s->h_counters, &s->h_small, &s->h_dyn, &s->h_meta, &s->h_fsc}) b->release();
  for (auto& e : s->ev) cudaEventDestroy(e);
  for (auto& e : s->ev_f) cudaEventDestroy(e);
  for (DevBuf* b : {&s->d_freqs, &s->d_fverdict, &s->d_ftile}) b->release();
  s->h_fcount.release();
  cudaEventDestroy(s->ev_fork); cudaEventDestroy(s->ev_join); cudaEventDestroy(s->ev_h2d); cudaEventDestroy(s->ev_fin);
  cudaStreamDestroy(s->st2); cudaStreamDestroy(s->st_copy);
  cudaStreamDestroy(s->st);
  delete s;
}

uint32_t yd_intern_env(yd_sched* s, const char* digest, size_t len) {
  return s->InternEnv(std::string(digest, len));
}
uint32_t yd_intern_ip(yd_sched* s, const char* ip, size_t len) { return s->InternIp(std::string(ip, len)); }

// KeepServantAlive, cc:190-220.  Pure registry work; the device copy of the facts
// is refreshed lazily before the next solve.
void yd_keep_servant_alive(yd_sched* s, int64_t now_ns, const yd_servant* v, int64_t expires_in_ns) {
  std::string loc = v->observed_location;
  auto it = s->loc2pos.find(loc);
  ServantHost* rec;
  std::vector<uint32_t> envs(v->num_envs);
  for (uint32_t i = 0; i != v->num_envs; ++i) envs[i] = s->InternEnv(v->env_digests[i]);
  if (it == s->loc2pos.end()) {
    s->loc2pos.emplace(loc, (uint32_t)s->sv.size());
    rec = &s->sv.emplace_back();
    rec->observed = loc;
    rec->discovered_at = now_ns;
    s->topo_dirty = true;
    s->order_dirty = true;
  } else {
    rec = &s->sv[it->second];
    if (rec->envs != envs) s->topo_dirty = true;
    uint32_t nf = 0;  // FactFlags of the new personality
    if (v->priority == YD_PRIORITY_DEDICATED) nf |= yd::kFlagDedicated;
    if (v->total_memory_in_bytes != 0 && v->memory_available_in_bytes < s->min_mem) nf |= yd::kFlagLowMem;
    if (rec->nproc != v->num_processors || rec->load != v->current_load || rec->max_tasks != v->max_tasks ||
        nf != s->FactFlags(*rec)) {
      s->order_dirty = true;  // a slot key or a free_end changed: the sorted slot order is rebuilt before the next solve
    }
  }
  rec->version = v->version;
  rec->reported = v->reported_location ? v->reported_location : "";
  rec->envs = std::move(envs);
  rec->nproc = v->num_processors;
  rec->load = v->current_load;
  rec->max_tasks = v->max_tasks;
  rec->total_mem = v->total_memory_in_bytes;
  rec->avail_mem = v->memory_available_in_bytes;
  rec->priority = v->priority;
  rec->reason = v->not_accepting_task_reason;
  rec->expires_at = now_ns + expires_in_ns;
  s->facts_dirty = true;
}

// ---- the two solvers' launch sequences -------------------------------------------

extern "C++" {
namespace {

constexpr size_t kRowscanMaxComponent = 32 * 32 * yd::kK;  // 8192 servants per component
constexpr size_t kStreamMaxComponent = 22000;              // 2 x u32 per servant of dynamic shared memory

yd::TopoView MakeTopo(yd_sched* s) {
  yd::TopoView t{};
  t.env_comp = s->d_env_comp.as<uint32_t>();
  t.n_envs = s->n_envs_dev;
  t.sv_comp = s->d_sv_comp.as<uint32_t>();
  t.sv_local = s->d_sv_local.as<uint32_t>();
  t.ip_off = s->d_ip_off.as<uint32_t>();
  t.ip_sv = s->d_ip_sv.as<uint32_t>();
  t.n_ips = s->n_ips_dev;
  t.sv_env_off = s->d_sv_env_off.as<uint32_t>();
  t.sv_envs = s->d_sv_envs.as<uint32_t>();
  t.comp_sv_off = s->d_comp_sv_off.as<uint32_t>();
  t.comp_sv = s->d_comp_sv.as<uint32_t>();
  t.sv_emask = s->emask_ok ? s->d_sv_emask.as<unsigned long long>() : nullptr;
  t.env_local = s->d_env_local.as<uint32_t>();
  return t;
}

yd::ClassTable MakeClassTable(yd_sched* s) {
  uint32_t* u = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_cls_off);
  yd::ClassTable ct{};
  // the 8-byte keys sit right behind res[] so one 0xFF memset initialises both
  ct.keys = reinterpret_cast<unsigned long long*>(s->d_res.as<uint32_t>() + s->res_words);
  ct.slot_cls = u;                       u += yd::kClsTableSize;
  ct.meta = u;                           u += 8;
  ct.cls_env = u;                        u += yd::kMaxClasses;
  ct.cls_mv = u;                         u += yd::kMaxClasses;
  ct.cls_comp = u;                       u += yd::kMaxClasses;
  ct.cls_nelig = u;                      u += yd::kMaxClasses;
  ct.cls_count = u;                      u += yd::kMaxClasses;
  ct.cls_lbit = u;                       u += yd::kMaxClasses;
  ct.comp_flags = u;                     u += s->n_comps;
  ct.comp_ncls = u;                      u += s->n_comps;
  ct.comp_midx = u;                      u += s->n_comps;
  ct.merge_comp = u;                     u += yd::kMaxClasses;
  ct.comp_cls = u;                       // [cls_bound * 32], the tail of the class region
  ct.cls_bound = s->cls_bound;
  ct.force_stream = s->force_stream;
  return ct;
}

yd::MergePlan MakeMergePlan(yd_sched* s) {
  uint32_t* u = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_merge_off);
  yd::MergePlan mp{};
  mp.bar = u;                            u += yd::kMaxClasses + 1;  // (only the first cell is used)
  mp.changed = u;                        u += 16;
  mp.viol = u;                           u += s->n_comps;
  mp.tau = u;                            // [S]
  return mp;
}

// Row-total mailboxes of the two row-parallel scans (k_scan_rows), in the zeroed scratch region.
unsigned long long* ScanPub(yd_sched* s, int which) {
  return reinterpret_cast<unsigned long long*>(static_cast<char*>(s->d_zero.p) + s->z_scan_off) + size_t(which) * (yd::kMaxClasses + 1);
}

yd::RqLayout MakeRqLayout(yd_sched* s, uint32_t q_base, uint32_t n_local, bool sharded) {
  uint32_t* u = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_layout_off);
  yd::RqLayout L{};
  L.goff = u;                            u += yd::kMaxClasses;
  L.gn = u;                              u += yd::kMaxClasses;
  L.win = u;                             u += yd::kMaxClasses;
  L.base = u;                            u += yd::kMaxClasses;
  L.total = u;
  L.q_base = q_base;
  L.n_local = n_local;
  L.sharded = sharded ? 1u : 0u;
  L.rank_off = s->d_rank_cnt.as<uint32_t>();
  L.nrt = (uint32_t)((s->res_words + yd::kRankTile - 1) / yd::kRankTile);
  return L;
}

// Slot table (both solvers).  For the slot-stream solver it also records slot owners.
// Returns the number of kernels launched.
uint32_t LaunchSlotTable(yd_sched* s, bool for_stream, bool static_rows = false) {
  const uint32_t S = (uint32_t)s->sv.size();
  cudaStream_t st = s->st;
  yd::ServantArrays arr = s->arrays();
  const uint32_t sentinel = for_stream ? 0u : 1u;
  const uint32_t sr = static_rows ? 1u : 0u;
  yd::k_slot_rows<<<1, 1024, 0, st>>>(S, s->d_dyn.as<yd::DynParams>(), arr, s->d_row_off.as<uint32_t>(),
                                      s->d_row_len.as<uint32_t>(), s->d_counters.as<Counters>(), sentinel, sr);
  uint32_t* owner = for_stream ? s->d_slot_owner.as<uint32_t>() : nullptr;
  if (s->wide) {
    yd::k_slot_fill<true><<<(S + 7) / 8, 256, 0, st>>>(S, arr, s->d_row_off.as<uint32_t>(),
                                                       s->d_row_len.as<uint32_t>(), nullptr,
                                                       s->d_codes.as<unsigned long long>(), owner, sentinel, sr);
  } else {
    yd::k_slot_fill<false><<<(S + 7) / 8, 256, 0, st>>>(S, arr, s->d_row_off.as<uint32_t>(),
                                                        s->d_row_len.as<uint32_t>(), s->d_codes.as<uint32_t>(),
                                                        nullptr, owner, sentinel, sr);
  }
  return 2;
}

// Solver 1: one (task x servant) row per decision.
uint32_t LaunchRowscan(yd_sched* s) {
  cudaStream_t st = s->st;
  yd::SolveArgs a{};
  a.reqs = s->d_reqs.as<yd_task_req>();
  a.dp = s->d_dyn.as<yd::DynParams>();
  a.res = s->d_res.as<uint32_t>();
  a.env_comp = s->d_env_comp.as<uint32_t>();
  a.env_local = s->d_env_local.as<uint32_t>();
  a.n_envs = s->n_envs_dev;
  a.comp_sv_off = s->d_comp_sv_off.as<uint32_t>();
  a.comp_sv = s->d_comp_sv.as<uint32_t>();
  a.comp_mask_off = s->d_comp_mask_off.as<uint32_t>();
  a.comp_nwarps = s->d_comp_nwarps.as<uint32_t>();
  a.envmask = s->d_envmask.as<uint8_t>();
  a.sv_comp = s->d_sv_comp.as<uint32_t>();
  a.sv_local = s->d_sv_local.as<uint32_t>();
  a.ip_off = s->d_ip_off.as<uint32_t>();
  a.ip_sv = s->d_ip_sv.as<uint32_t>();
  a.n_ips = s->n_ips_dev;
  a.sv = s->arrays();
  a.row_off = s->d_row_off.as<uint32_t>();
  a.codes = s->d_codes.p;
  // Two register budgets: up to 8 solver warps (2048 servants per component) plus
  // 8 producer warps run with <= 128 registers per thread; larger components are
  // capped at 64 registers.
  const unsigned threads = std::min(32u, s->max_warps + yd::kMaxProducers) * 32;
  if (threads <= 512) {
    if (s->wide) yd::k_solve_rowscan<unsigned long long, 512><<<s->n_comps, threads, 0, st>>>(a);
    else yd::k_solve_rowscan<uint32_t, 512><<<s->n_comps, threads, 0, st>>>(a);
  } else {
    if (s->wide) yd::k_solve_rowscan<unsigned long long, 1024><<<s->n_comps, threads, 0, st>>>(a);
    else yd::k_solve_rowscan<uint32_t, 1024><<<s->n_comps, threads, 0, st>>>(a);
  }
  return 1;
}

template <typename KeyT>
uint32_t LaunchSort(yd_sched* s, int first_bit, int last_bit) {
  cudaStream_t st = s->st;
  const uint32_t nb = s->sort_nb;
  const unsigned long long* n_ptr = &s->d_counters.as<Counters>()->slots;
  uint32_t* zbase = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_hist_off[0]);
  const size_t stride = yd::rs_pass_words(nb);
  const int passes = (last_bit - first_bit) / yd::kRsBits + 1;
  const KeyT* kin = s->d_codes.as<KeyT>();
  const uint32_t* vin = nullptr;
  int cur = (passes - 1) & 1;  // ping-pong so that the LAST pass writes buffer 0 (captured graphs keep its address)
  // digit histograms of all passes in one read, then one kernel per pass
  yd::k_rs_ghist<KeyT><<<nb, yd::kRsThreads, 0, st>>>(kin, n_ptr, first_bit, passes, nb, zbase);
  uint32_t launches = 1;
  for (int pass = 0; pass < passes; ++pass) {
    KeyT* kout = s->d_sort_k[cur].as<KeyT>();
    uint32_t* vout = s->d_sort_v[cur].as<uint32_t>();
    yd::k_rs_pass<KeyT><<<nb, yd::kRsThreads, 0, st>>>(kin, vin, n_ptr, first_bit + pass * yd::kRsBits, nb,
                                                       yd::rs_pass_scratch(zbase + pass * stride, nb), kout, vout);
    launches += 1;
    kin = kout;
    vin = vout;
    cur ^= 1;
  }
  return launches;
}

// Allocates everything the slot-stream sequence touches for size class (Nb, slot_b) and
// lays out the zero-initialised scratch region; called before a graph capture so that no
// allocation happens inside it.
void PrepareStreamBuffers(yd_sched* s, uint32_t Nb, size_t slot_b) {
  const size_t ksz = s->wide ? 8 : 4;
  for (int b = 0; b < 2; ++b) { s->d_sort_k[b].ensure(slot_b * ksz); s->d_sort_v[b].ensure(slot_b * 4); }
  s->d_slot_rec.ensure(slot_b * 8);
  s->sort_nb = (uint32_t)((slot_b + yd::kRsTile - 1) / yd::kRsTile);
  const int passes = s->wide ? 9 : 4;
  size_t off = 0;
  for (int p = 0; p < passes; ++p) { s->z_hist_off[p] = off; off += yd::rs_pass_words(s->sort_nb) * 4; }
  s->z_cls_off = off;
  off += (yd::kClsTableSize + 8 + 7 * yd::kMaxClasses + 3 * size_t(s->n_comps) + 32 * size_t(s->cls_bound) + 8) * 4;
  s->z_merge_off = off;
  off += (yd::kMaxClasses + 1 + 16 + size_t(s->n_comps) + s->sv.size() + 8) * 4;
  s->z_layout_off = off;
  off += (4 * yd::kMaxClasses + 8) * 4;
  off = (off + 7) & ~size_t(7);
  s->z_scan_off = off;
  off += 2 * (yd::kMaxClasses + 1) * 8;
  s->z_final_off = off;
  off += (size_t(Nb + 1023) / 1024 + 2) * 8;
  s->z_fbar_off = off;
  off += 8 * 4;
  const uint32_t n_tiles = (uint32_t)((slot_b + yd::kListTile - 1) / yd::kListTile);
  s->z_listcnt_off = off;
  off += (size_t(s->cls_bound) * n_tiles + 1) * 4;
  s->z_bytes = (off + 255) & ~size_t(255);
  s->d_zero.ensure(s->z_bytes);
  s->d_list.ensure(slot_b * 8 * 4);
  s->d_list_bal.ensure(size_t(n_tiles) * s->cls_bound * 32 * 4);  // membership ballots: (tile, list, warp)
  const uint32_t n_rtiles = (Nb + yd::kRankTile - 1) / yd::kRankTile;
  s->d_rcls.ensure(size_t(Nb) * 4); s->d_rrank.ensure(size_t(Nb) * 4); s->d_rq.ensure(size_t(Nb) * 8);
  s->d_rself.ensure(size_t(Nb) * 4);
  s->d_stream_scratch.ensure(std::max<size_t>(s->sv.size(), 1) * 8);
  s->d_slot_pick.ensure(slot_b * 4 * 4);  // one word per list entry
  // every slot is in at most one pseudo-class list: chunks <= slots / chunk + one partial chunk per list
  s->merge_max_chunks = (uint32_t)(slot_b / s->merge_chunk) + s->cls_bound + 1;
  s->d_mst_in.ensure(size_t(s->merge_max_chunks) * yd::kMergeStateWords * 4);
  s->d_mst_out.ensure(size_t(s->merge_max_chunks) * yd::kMergeStateWords * 4);
  s->d_rank_cnt.ensure((size_t(s->cls_bound) * n_rtiles + 1) * 4);
  if (!s->stream_attr_set) {
    YD_CUDA_CHECK(cudaFuncSetAttribute(yd::k_solve_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, 190 * 1024));
    s->stream_attr_set = true;
  }
}

// The merge solver: ONE persistent launch (rounds, scatter and check are phases behind grid barriers), so the
// grid must be co-resident: occupancy x SMs blocks at most, each looping over its chunks.
uint32_t LaunchMerge(yd_sched* s, yd::MergeArgs& m, cudaStream_t st) {
  m.kcap = std::min(32u, s->cls_bound);
  const size_t dyn = size_t(1 + m.kcap) * yd::kRingRecs * sizeof(uint2);
  if (s->merge_grid_kcap != m.kcap) {
    int per_sm = 0, sms = 0;
    YD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, yd::k_merge_solve, 32, dyn));
    YD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    s->merge_grid = (uint32_t)std::max(1, std::min(per_sm, 16) * sms);
    s->merge_grid_kcap = m.kcap;
  }
  m.chunk = s->merge_chunk;
  m.max_chunks = s->merge_max_chunks;
  m.diag = &s->d_counters.as<Counters>()->pad[0];
  m.rq_blocks = (uint32_t)(s->d_rq.cap / 256);
  m.ls_blocks = (uint32_t)(s->d_list.cap / 256);
  const uint32_t grid = std::min(s->merge_grid, s->merge_max_chunks);
  yd::k_merge_solve<<<grid, 32, dyn, st>>>(m);
  yd::k_merge_check<<<(std::max(m.L.n_local, 1u) + 255) / 256, 256, 0, st>>>(m);
  return 2;
}

constexpr size_t kStaticSlotLimit = size_t(1) << 26;

// (Re)builds the kept slot order: slot table over ALL running_tasks values + its sort, outside any graph.
// Buffers must exist (PrepareStreamBuffers).  Returns the number of kernels launched.
uint32_t RebuildSlotOrder(yd_sched* s, size_t slot_b) {
  cudaStream_t st = s->st;
  // the sort's digit histograms live in the zeroed scratch region
  YD_CUDA_CHECK(cudaMemsetAsync(static_cast<char*>(s->d_zero.p) + s->z_hist_off[0], 0, s->z_cls_off - s->z_hist_off[0], st));
  uint32_t l = LaunchSlotTable(s, true, true);
  if (s->wide) l += LaunchSort<unsigned long long>(s, 0, 62);
  else l += LaunchSort<uint32_t>(s, 3, 30);
  {
    yd::SlotDecode dec{s->d_sort_v[0].as<uint32_t>(), s->d_slot_owner.as<uint32_t>(), s->d_row_off.as<uint32_t>(),
                       s->d_row_len.as<uint32_t>(), s->d_run.as<uint32_t>(), 1u, nullptr};
    yd::k_slot_records<<<(unsigned)((slot_b + 255) / 256), 256, 0, st>>>(&s->d_counters.as<Counters>()->slots, dec,
                                                                          s->d_slot_rec.as<uint2>());
    l += 1;
  }
  YD_CUDA_CHECK(cudaGetLastError());
  s->order_dirty = false;
  s->order_static = true;
  s->order_slot_b = slot_b;
  s->order_rebuilds += 1;
  return l;
}

// The solvers for everything the data-parallel path does not decide: the merge solver (all components but those with
// several servants behind one requestor IP), then the sequential slot-stream walk for the rest.
uint32_t LaunchCoupledSolvers(yd_sched* s, uint32_t N, size_t slot_b, const yd::RqLayout& L) {
  cudaStream_t st = s->st;
  uint32_t launches = 0;
  yd::TopoView t = MakeTopo(s);
  yd::ClassTable ct = MakeClassTable(s);
  yd::ServantArrays arr = s->arrays();
  const yd::DynParams* dp = s->d_dyn.as<yd::DynParams>();
  uint32_t* list_cnt = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_listcnt_off);
  const uint32_t n_tiles = (uint32_t)((slot_b + yd::kListTile - 1) / yd::kListTile);
  const uint32_t n_rtiles = (N + yd::kRankTile - 1) / yd::kRankTile;
  // ---- merge solver: everything but components with several servants behind one requestor IP -------
  yd::MergePlan mp = MakeMergePlan(s);
  {
    yd::MergeArgs m{};
    m.t = t; m.ct = ct; m.mp = mp; m.sv = arr; m.dp = dp;
    m.comp_mode = s->d_comp_mode.as<uint32_t>();
    m.list_off = list_cnt; m.n_list_tiles = n_tiles; m.list = s->d_list.as<uint2>();
    m.rank_off = s->d_rank_cnt.as<uint32_t>(); m.n_rank_tiles = n_rtiles;
    m.rq = s->d_rq.as<uint2>(); m.rcls = s->d_rcls.as<uint32_t>(); m.rself = s->d_rself.as<uint32_t>();
    m.slot_pick = s->d_slot_pick.as<uint32_t>();
    m.st_in = s->d_mst_in.as<uint32_t>(); m.st_out = s->d_mst_out.as<uint32_t>();
    m.res = s->d_res.as<uint32_t>();
    m.L = L;
    launches += LaunchMerge(s, m, st);
  }

  // ---- sequential decisions for everything else ---------------------------------------------
  yd::StreamArgs a{};
  a.reqs = s->d_reqs.as<yd_task_req>();
  a.dp = dp;
  a.res = s->d_res.as<uint32_t>();
  a.t = t;
  a.ct = ct;
  a.sv = arr;
  a.row_len = s->d_row_len.as<uint32_t>();
  a.static_rows = s->order_static ? 1u : 0u;
  a.list_off = list_cnt;
  a.n_list_tiles = n_tiles;
  a.list = s->d_list.as<uint2>();
  a.max_comp_servants = (uint32_t)std::min<size_t>(s->max_comp_servants, kStreamMaxComponent);
  a.gscratch = s->d_stream_scratch.as<uint32_t>();
  a.n_servants = (uint32_t)s->sv.size();
  a.comp_mode = s->d_comp_mode.as<uint32_t>();
  a.viol = mp.viol;
  a.counters = s->d_counters.as<Counters>();
  a.debug = s->stream_debug;
  const size_t dyn = size_t(a.max_comp_servants) * 8;
  yd::k_solve_stream<<<s->n_comps, (yd::kStreamProducers + 1) * 32, dyn, st>>>(a);
  launches += 1;
  return launches;
}

// Solver 2: sorted slot streams.  Two concurrent branches:
//   st  : slot table (+ first histogram) -> radix passes
//   st2 : [wait for the request upload] class table -> finalize -> FIFO ranks -> scan
// joined before the per-class lists.  `capturing` selects the external-event flavour of
// the wait on the upload (the upload itself is never part of the graph).
uint32_t LaunchStream(yd_sched* s, uint32_t N, size_t slot_b, bool capturing) {
  cudaStream_t st = s->st, st2 = s->st2;
  uint32_t launches = 0;
  yd::TopoView t = MakeTopo(s);
  yd::ClassTable ct = MakeClassTable(s);
  yd::ServantArrays arr = s->arrays();
  const yd::DynParams* dp = s->d_dyn.as<yd::DynParams>();
  uint32_t* list_cnt = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_listcnt_off);
  const uint32_t n_tiles = (uint32_t)((slot_b + yd::kListTile - 1) / yd::kListTile);
  const uint32_t n_rtiles = (N + yd::kRankTile - 1) / yd::kRankTile;

  // ---- fork ---------------------------------------------------------------------
  YD_CUDA_CHECK(cudaEventRecord(s->ev_fork, st));
  YD_CUDA_CHECK(cudaStreamWaitEvent(st2, s->ev_fork, 0));
  // branch B: classes and FIFO ranks (needs the requests in HBM)
  YD_CUDA_CHECK(cudaStreamWaitEvent(st2, s->ev_h2d, capturing ? cudaEventWaitExternal : 0));
  yd::k_cls_insert<<<(N + 255) / 256, 256, 0, st2>>>(s->d_reqs.as<yd_task_req>(), dp, t, ct);
  yd::k_cls_finalize<<<1, 1024, 0, st2>>>(t, ct, arr, s->n_comps, s->d_comp_mode.as<uint32_t>());
  YD_CUDA_CHECK(cudaEventRecord(s->ev_fin, st2));  // the list kernels on `st` need the class table, not what follows
  yd::k_cls_elig<<<ct.cls_bound, 256, 0, st2>>>(t, ct, arr);
  yd::k_rank_count<<<n_rtiles, yd::kRankTile, 0, st2>>>(s->d_reqs.as<yd_task_req>(), dp, t, ct,
                                                         s->d_comp_mode.as<uint32_t>(), n_rtiles,
                                                         s->d_rcls.as<uint32_t>(), s->d_rrank.as<uint32_t>(),
                                                         s->d_rself.as<uint32_t>(), s->d_rank_cnt.as<uint32_t>());
  yd::k_scan_rows<<<ct.cls_bound, 1024, 0, st2>>>(s->d_rank_cnt.as<uint32_t>(), ct.meta, n_rtiles, ScanPub(s, 0));
  YD_CUDA_CHECK(cudaEventRecord(s->ev_join, st2));
  launches += 5;
  // branch A: slot table and its sort -- unless the kept (static) order is valid
  if (!s->order_static) {
    launches += LaunchSlotTable(s, true);
    if (s->wide) launches += LaunchSort<unsigned long long>(s, 0, 62);
    else launches += LaunchSort<uint32_t>(s, 3, 30);
  }
  YD_CUDA_CHECK(cudaStreamWaitEvent(st, s->ev_fin, 0));

  // ---- per-class sorted slot lists ----------------------------------------------------
  const unsigned long long* m_ptr = &s->d_counters.as<Counters>()->slots;
  yd::SlotDecode dec{s->d_sort_v[0].as<uint32_t>(), s->d_slot_owner.as<uint32_t>(), s->d_row_off.as<uint32_t>(),
                     s->d_row_len.as<uint32_t>(), s->d_run.as<uint32_t>(), s->order_static ? 1u : 0u,
                     s->order_static ? s->d_slot_rec.as<uint2>() : nullptr};
  yd::k_list_count<<<n_tiles, yd::kListTile, 0, st>>>(m_ptr, dec, t, ct, arr, n_tiles, list_cnt,
                                                      s->d_list_bal.as<uint32_t>());
  yd::k_scan_rows<<<ct.cls_bound, 1024, 0, st>>>(list_cnt, ct.meta + 3, n_tiles, ScanPub(s, 1));
  yd::k_list_fill<<<n_tiles, yd::kListTile, 0, st>>>(m_ptr, dec, t, ct, n_tiles, list_cnt, s->d_list_bal.as<uint32_t>(),
                                                     s->d_list.as<uint2>(), (uint32_t)(slot_b * 4));
  launches += 3;

  // ---- join: FIFO ranks and eligibility counts are needed from here on ---------------------------------------
  YD_CUDA_CHECK(cudaStreamWaitEvent(st, s->ev_join, 0));
  // ---- data-parallel path: single-class components without self-requests ----------------
  // (n_local = the grid bound: res[] has that many cells and only requests < dp->n are ever named)
  const yd::RqLayout L = MakeRqLayout(s, 0, N, false);
  yd::k_rank_assign<<<(N + 255) / 256, 256, 0, st>>>(dp, n_rtiles, t, ct, s->d_rcls.as<uint32_t>(),
                                                     s->d_rrank.as<uint32_t>(), s->d_rself.as<uint32_t>(),
                                                     s->d_rank_cnt.as<uint32_t>(), list_cnt,
                                                     n_tiles, s->d_list.as<uint2>(), arr, s->d_comp_mode.as<uint32_t>(),
                                                     s->d_rq.as<uint2>(), s->d_res.as<uint32_t>(), L);
  launches += 1;

  launches += LaunchCoupledSolvers(s, N, slot_b, L);
  return launches;
}

constexpr size_t kFusedLoffCacheWords = 16384;  // 64 KB of dynamic shared memory at most

// The fused front (fused.cuh): classes, ranks, lists and the data-parallel verdicts in ONE persistent launch on `st`;
// `solo`: grants, task ids and leases too (batches made of data-parallel components only), else the coupled solvers
// follow.  Needs the kept slot order.
uint32_t LaunchFused(yd_sched* s, uint32_t N, size_t slot_b, bool capturing, bool solo, bool packed_in, bool packed_out) {
  cudaStream_t st = s->st;
  uint32_t launches = 0;
  const uint32_t n_tiles = (uint32_t)((slot_b + yd::kListTile - 1) / yd::kListTile);
  const uint32_t n_rtiles = (N + yd::kRankTile - 1) / yd::kRankTile;
  yd::FusedArgs a{};
  a.sc = s->fsc;
  // graphed general sequence: the scalars come through a copy node; a solo graph gets them as (patched) kernel parameters
  a.sc_dev = (capturing && !solo) ? s->d_fsc.as<yd::FusedScalars>() : nullptr;
  if (a.sc_dev) YD_CUDA_CHECK(cudaMemcpyAsync(s->d_fsc.p, s->h_fsc.p, sizeof(yd::FusedScalars), cudaMemcpyHostToDevice, st));
  a.hio = s->report_dev ? s->d_report.as<yd::FusedHostIO>() : s->d_fio;
  a.dyn_out = solo ? nullptr : s->d_dyn.as<yd::DynParams>();
  a.clean_keys = reinterpret_cast<unsigned long long*>(s->d_res.as<uint32_t>() + s->res_words);
  a.clean_zero = reinterpret_cast<uint4*>(static_cast<char*>(s->d_zero.p) + s->z_cls_off);
  a.clean_zero_vec = (uint32_t)((s->z_bytes - s->z_cls_off) / 16);
  a.reqs = s->d_reqs.as<yd_task_req>();
  a.reqs16 = packed_in ? s->d_reqs16.as<uint4>() : nullptr;
  a.reqs16_w = packed_in ? s->d_reqs16.as<uint4>() : nullptr;
  a.reqs_w = (packed_in && !solo) ? s->d_reqs.as<yd_task_req>() : nullptr;
  a.t = MakeTopo(s);
  a.ct = MakeClassTable(s);
  a.sv = s->arrays();
  a.dec = yd::SlotDecode{s->d_sort_v[0].as<uint32_t>(), s->d_slot_owner.as<uint32_t>(), s->d_row_off.as<uint32_t>(),
                         s->d_row_len.as<uint32_t>(), s->d_run.as<uint32_t>(), 1u, s->d_slot_rec.as<uint2>()};
  a.m_ptr = &s->d_counters.as<Counters>()->slots;
  a.comp_mode = s->d_comp_mode.as<uint32_t>();
  a.n_comps = s->n_comps;
  a.n_rtiles = n_rtiles;
  a.n_ltiles = n_tiles;
  a.rcls = s->d_rcls.as<uint32_t>();
  a.rrank = s->d_rrank.as<uint32_t>();
  a.rself = s->d_rself.as<uint32_t>();
  a.rank_cnt = s->d_rank_cnt.as<uint32_t>();
  a.list_cnt = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_listcnt_off);
  a.list_bal = s->d_list_bal.as<uint32_t>();
  a.list = s->d_list.as<uint2>();
  a.list_cap = (uint32_t)(slot_b * 4);
  a.rq = s->d_rq.as<uint2>();
  a.res = s->d_res.as<uint32_t>();
  a.L = MakeRqLayout(s, 0, N, false);
  a.bar = reinterpret_cast<uint32_t*>(static_cast<char*>(s->d_zero.p) + s->z_fbar_off);
  a.solo = solo ? 1u : 0u;
  a.packed_out = packed_out ? 1u : 0u;
  a.look = reinterpret_cast<unsigned long long*>(static_cast<char*>(s->d_zero.p) + s->z_final_off);
  a.comp_sv = s->d_comp_sv.as<uint32_t>();
  a.ring = s->ring();
  a.out = packed_out ? s->d_out8.p : s->d_out.p;
  a.counters = s->d_counters.as<Counters>();
  a.n_servants = (uint32_t)s->sv.size();
  a.prof = s->fused_prof ? s->d_fused_prof.as<unsigned long long>() : nullptr;
  YD_CUDA_CHECK(cudaStreamWaitEvent(st, s->ev_h2d, capturing ? cudaEventWaitExternal : 0));
  const uint32_t grid = s->fused_grid;  // one block per SM, whatever the batch: the phases hand out tiles of two kinds
  // solo: the scanned list offsets are searched once per request -- from shared memory when they fit
  const size_t cells = size_t(s->cls_bound) * (n_tiles + 1) + 1;
  const size_t dyn = solo && cells <= kFusedLoffCacheWords ? cells * 4 : 0;
  a.loff_cache_words = (uint32_t)(dyn / 4);
  a.lite = s->fused_lite ? 1u : 0u;
  yd::k_fused_front<<<grid, 1024, dyn, st>>>(a);
  s->last_fused = a;
  s->last_fused_grid = grid;
  s->last_fused_dyn = dyn;
  if (solo && s->report_dev) {
    YD_CUDA_CHECK(cudaMemcpyAsync(s->h_fio, s->d_report.p, sizeof(yd::FusedHostIO), cudaMemcpyDeviceToHost, st));
  }
  launches += 1;
  if (!solo) launches += LaunchCoupledSolvers(s, N, slot_b, a.L);
  return launches;
}

}  // namespace
}  // extern "C++"

extern "C++" {
namespace {

uint64_t NextPow2(uint64_t v, uint64_t lo) {
  uint64_t r = lo;
  while (r < v) r <<= 1;
  return r;
}

// Largest grid (1024-request blocks) whose slot-stream final is the one-launch k_final_fused: beyond ~2 M requests the
// look-back chain of 1024-thread blocks is slower than three plain passes (count, scan, write).
constexpr uint32_t kFinalFusedMaxBlocks = 2048;

// Kernels that write the grants after the solver: 0 (the solo fused kernel wrote them), 1 (k_final_fused) or 3.
uint32_t FinalPasses(bool solo, uint32_t solver, bool have_work, uint32_t nb) {
  if (solo) return 0;
  return solver == 2 && have_work && nb <= kFinalFusedMaxBlocks ? 1 : 3;
}

// Everything between the request upload and the grant download, for size class
// (Nb, slot_b): the sequence that is captured into a CUDA graph.
// variant: 0 = the kernel-by-kernel pipeline, 1 = fused front + coupled solvers + final, 2 = fused front alone (solo).
// packed bit 0: the upload is 16-byte records in d_reqs16; bit 1: the download is 8-byte grants from d_out8.
uint32_t EnqueueSolve(yd_sched* s, uint32_t Nb, size_t slot_b, uint32_t solver, bool record_events, bool capturing,
                      uint32_t variant = 0, uint32_t packed = 0) {
  cudaStream_t st = s->st;
  const uint32_t S = (uint32_t)s->sv.size();
  const bool have_work = S && s->n_comps;
  const uint32_t nb = (Nb + 1023) / 1024;
  const bool packed_in = packed & 1u, packed_out = packed & 2u;
  uint32_t launches = 0;
  const yd::DynParams* dp = s->d_dyn.as<yd::DynParams>();
  const bool fused = variant && have_work && solver == 2;
  const bool solo = fused && variant >= 2;
  // (the fused kernel reads the call's scalars from the mapped host record and -- not solo -- stores them in d_dyn itself)
  if (!fused) YD_CUDA_CHECK(cudaMemcpyAsync(s->d_dyn.p, s->h_dyn.p, sizeof(yd::DynParams), cudaMemcpyHostToDevice, st));
  if (solo) {
    // the solo kernel keeps the verdicts in registers: only the class-table keys behind res[] are initialised -- and
    // not even those (variant 3) when the previous solo solve left the scratch clean
    if (variant == 2) {
      YD_CUDA_CHECK(cudaMemsetAsync(s->d_res.as<uint32_t>() + s->res_words, 0xFF, yd::kClsTableSize * 8, st));
      YD_CUDA_CHECK(cudaMemsetAsync(static_cast<char*>(s->d_zero.p) + s->z_cls_off, 0, s->z_bytes - s->z_cls_off, st));
    }
  } else {
    // res[] = kResEnvNotFound, and (slot-stream) the class-table keys behind it = empty
    YD_CUDA_CHECK(cudaMemsetAsync(s->d_res.p, 0xFF, size_t(Nb) * 4 + (solver == 2 ? yd::kClsTableSize * 8 : 0), st));
    if (solver == 2 && have_work) YD_CUDA_CHECK(cudaMemsetAsync(s->d_zero.p, 0, s->z_bytes, st));
  }
  if (record_events) YD_CUDA_CHECK(cudaEventRecord(s->ev[1], st));
  const uint32_t* abort_flag = nullptr;
  if (packed_in && !(variant && have_work && solver == 2)) {
    // 16-byte upload -> the 24-byte queue the pipeline kernels read
    YD_CUDA_CHECK(cudaStreamWaitEvent(st, s->ev_h2d, capturing ? cudaEventWaitExternal : 0));
    yd::k_unpack_reqs<<<(Nb + 255) / 256, 256, 0, st>>>(s->d_reqs16.as<uint4>(), dp, s->d_reqs.as<yd_task_req>());
    launches += 1;
  }
  if (have_work && solver == 2) {
    if (record_events) YD_CUDA_CHECK(cudaEventRecord(s->ev[2], st));
    if (variant) launches += LaunchFused(s, Nb, slot_b, capturing, variant >= 2, packed_in, packed_out);
    else launches += LaunchStream(s, Nb, slot_b, capturing);
    abort_flag = MakeClassTable(s).meta + 1;
  } else {
    if (have_work) launches += LaunchSlotTable(s, false);
    if (record_events) YD_CUDA_CHECK(cudaEventRecord(s->ev[2], st));
    // the row-scan kernels read the requests: they were uploaded on the copy stream
    YD_CUDA_CHECK(cudaStreamWaitEvent(st, s->ev_h2d, capturing ? cudaEventWaitExternal : 0));
    if (have_work) launches += LaunchRowscan(s);
  }
  if (record_events) YD_CUDA_CHECK(cudaEventRecord(s->ev[3], st));
  const uint32_t final_passes = FinalPasses(solo, solver, have_work, nb);
  if (final_passes == 0) {
    // grants, ids and leases were written by the fused kernel
  } else if (final_passes == 1) {
    // grants, task ids (single-pass scan with look-back), leases, ++running_tasks: one launch
    unsigned long long* look = reinterpret_cast<unsigned long long*>(static_cast<char*>(s->d_zero.p) + s->z_final_off);
    yd::k_final_fused<<<nb, 1024, 0, st>>>(s->d_res.as<uint32_t>(), s->d_reqs.as<yd_task_req>(), dp, look, nb,
                                           s->d_comp_sv.as<uint32_t>(), s->ring(), s->d_out.as<yd_grant>(),
                                           s->d_counters.as<Counters>(), abort_flag, s->d_run.as<uint32_t>(),
                                           s->d_ever.as<unsigned long long>());
    launches += 1;
  } else {
    yd::k_final_count<<<nb, 1024, 0, st>>>(s->d_res.as<uint32_t>(), dp, s->d_blk.as<uint32_t>(), abort_flag);
    yd::k_final_scan<<<1, 1024, 0, st>>>(s->d_blk.as<uint32_t>(), nb, s->d_counters.as<Counters>(), abort_flag);
    yd::k_final_write<<<nb, 1024, 0, st>>>(s->d_res.as<uint32_t>(), s->d_reqs.as<yd_task_req>(), dp,
                                           s->d_blk.as<uint32_t>(), s->d_comp_sv.as<uint32_t>(), s->ring(),
                                           s->d_out.as<yd_grant>(), abort_flag,
                                           // the row-scan solver writes running_tasks back itself
                                           solver == 2 ? s->d_run.as<uint32_t>() : nullptr,
                                           s->d_ever.as<unsigned long long>());
    launches += 3;
  }
  if (packed_out && !solo) {
    yd::k_pack_grants<<<(Nb + 255) / 256, 256, 0, st>>>(s->d_out.as<uint4>(), dp, s->ring(), s->d_out8.as<uint2>());
    launches += 1;
  }
  YD_CUDA_CHECK(cudaGetLastError());
  if (record_events) YD_CUDA_CHECK(cudaEventRecord(s->ev[4], st));
  if (solo) return launches;  // the kernel left grant count and flags in the mapped host record
  YD_CUDA_CHECK(cudaMemcpyAsync(s->h_counters.p, s->d_counters.p, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  if (abort_flag) {
    YD_CUDA_CHECK(cudaMemcpyAsync(s->h_meta.p, abort_flag - 1, 32, cudaMemcpyDeviceToHost, st));  // meta[0..7]
  }
  return launches;
}


// Debug aid (YDSCHED_DUMP=1): hashes of every intermediate of the slot-stream pipeline after a
// solve, to compare two runs stage by stage.
void DumpStreamState(yd_sched* s, uint32_t Nb, size_t slot_b) {
  static int solve_no = 0;
  ++solve_no;
  auto fetch = [&](const void* p, size_t bytes) {
    std::vector<unsigned char> h(bytes);
    if (bytes) YD_CUDA_CHECK(cudaMemcpy(h.data(), p, bytes, cudaMemcpyDeviceToHost));
    return h;
  };
  auto hash = [&](const char* name, const std::vector<unsigned char>& h) {
    unsigned long long x = 1469598103934665603ull;
    for (unsigned char c : h) { x ^= c; x *= 1099511628211ull; }
    fprintf(stderr, "YDDUMP %d %-12s %8zu %016llx\n", solve_no, name, h.size(), x);
  };
  Counters c;
  YD_CUDA_CHECK(cudaMemcpy(&c, s->d_counters.p, sizeof c, cudaMemcpyDeviceToHost));
  const size_t m = (size_t)c.slots, ksz = s->wide ? 8 : 4;
  const uint32_t S = (uint32_t)s->sv.size();
  fprintf(stderr, "YDDUMP %d slots %zu Nb %u slot_b %zu cls_bound %u\n", solve_no, m, Nb, slot_b, s->cls_bound);
  hash("row_off", fetch(s->d_row_off.p, size_t(S + 1) * 4));
  hash("row_len", fetch(s->d_row_len.p, size_t(S) * 4));
  hash("codes", fetch(s->d_codes.p, m * ksz));
  hash("owner", fetch(s->d_slot_owner.p, m * 4));
  hash("sorted_k", fetch(s->d_sort_k[0].p, m * ksz));
  hash("sorted_v", fetch(s->d_sort_v[0].p, m * 4));
  yd::ClassTable ct = MakeClassTable(s);
  auto meta = fetch(ct.meta, 32);
  const uint32_t* mt = reinterpret_cast<const uint32_t*>(meta.data());
  fprintf(stderr, "YDDUMP %d meta %u %u %u %u\n", solve_no, mt[0], mt[1], mt[2], mt[3]);
  const uint32_t ncls = std::min(mt[0], yd::kMaxClasses);
  hash("cls_env", fetch(ct.cls_env, ncls * 4));
  hash("cls_mv", fetch(ct.cls_mv, ncls * 4));
  hash("cls_nelig", fetch(ct.cls_nelig, ncls * 4));
  hash("comp_mode", fetch(s->d_comp_mode.p, size_t(s->n_comps) * 4));
  const uint32_t n_tiles = (uint32_t)((slot_b + yd::kListTile - 1) / yd::kListTile);
  auto lo = fetch(static_cast<char*>(s->d_zero.p) + s->z_listcnt_off, (size_t(mt[3]) * n_tiles + 1) * 4);
  hash("list_off", lo);
  const uint32_t total = reinterpret_cast<const uint32_t*>(lo.data())[size_t(mt[3]) * n_tiles];
  fprintf(stderr, "YDDUMP %d list_total %u\n", solve_no, total);
  hash("list", fetch(s->d_list.p, size_t(total) * 8));
  hash("res", fetch(s->d_res.p, size_t(s->h_dyn.as<yd::DynParams>()->n) * 4));
  hash("run_after", fetch(s->d_run.p, size_t(S) * 4));
  if (const char* dir = getenv("YDSCHED_DUMP_DIR")) {
    auto save = [&](const char* name, const std::vector<unsigned char>& h) {
      char path[512];
      snprintf(path, sizeof path, "%s/s%d_%s.bin", dir, solve_no, name);
      if (FILE* f = fopen(path, "wb")) { fwrite(h.data(), 1, h.size(), f); fclose(f); }
    };
    save("sorted_k", fetch(s->d_sort_k[0].p, m * ksz));
    save("sorted_v", fetch(s->d_sort_v[0].p, m * 4));
    save("owner", fetch(s->d_slot_owner.p, m * 4));
    save("row_off", fetch(s->d_row_off.p, size_t(S + 1) * 4));
    save("row_len", fetch(s->d_row_len.p, size_t(S) * 4));
    save("list_off", lo);
    save("list", fetch(s->d_list.p, size_t(total) * 8));
    save("cls_env", fetch(ct.cls_env, ncls * 4));
    save("cls_mv", fetch(ct.cls_mv, ncls * 4));
    save("res", fetch(s->d_res.p, size_t(s->h_dyn.as<yd::DynParams>()->n) * 4));
    save("run_after", fetch(s->d_run.p, size_t(S) * 4));
    save("reqs", fetch(s->d_reqs.p, size_t(s->h_dyn.as<yd::DynParams>()->n) * sizeof(yd_task_req)));
  }
}
}  // namespace
}  // extern "C++"

// THE HOT PATH: n sequential WaitForStartingNewTask decisions (cc:93-140).
// Queue staging: a front end can move the pending queue into HBM while RPCs are still
// arriving and start the solve when the batch closes.
void yd_stage_requests(yd_sched* s, const yd_task_req* reqs, size_t n) {
  if (n > 0x40000000ull) { fprintf(stderr, "ydsched: batch too large\n"); abort(); }
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->staged_n = 0;
  if (n == 0) return;
  s->d_reqs.ensure(size_t(NextPow2(n, 1024)) * sizeof(yd_task_req));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_reqs.p, reqs, n * sizeof(yd_task_req), cudaMemcpyHostToDevice, s->st_copy));
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st_copy));  // `reqs` may be reused by the caller right away
  s->staged_n = n;
}

void yd_wait_for_staged_tasks(yd_sched* s, int64_t now_ns, size_t n, yd_grant* out) {
  if (n == 0) return;
  if (n > s->staged_n) { fprintf(stderr, "ydsched: %zu requests asked for, %zu staged\n", n, s->staged_n); abort(); }
  yd_wait_for_starting_new_tasks(s, now_ns, nullptr, n, out);
}

extern "C++" {
namespace {
// The solve behind yd_wait_for_starting_new_tasks and its packed twin.  Requests: `reqs` (24-byte records), or `reqs16`
// (16-byte records), or neither = the first n staged requests (yd_stage_requests) are already in HBM.  Grants: `out`
// (16-byte records) or `out8` (8-byte records, ids = ids_out->first_task_id + ordinal * stride).
void WaitImpl(yd_sched* s, int64_t now_ns, const yd_task_req* reqs, const yd_task_req16* reqs16, size_t n, yd_grant* out,
              yd_grant8* out8, yd_packed_ids* ids_out) {
  if (ids_out) { ids_out->first_task_id = s->next_id * s->id_stride + s->id_offset; ids_out->stride = s->id_stride; }
  if (n == 0) return;
  double hp[8] = {};
  auto hp_now = [&]() { return s->host_prof ? std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count() : 0.0; };
  hp[0] = hp_now();
  if (!reqs && !reqs16 && n > s->staged_n) { fprintf(stderr, "ydsched: NULL request array and nothing staged\n"); abort(); }
  if (n > 0x40000000ull) { fprintf(stderr, "ydsched: batch too large\n"); abort(); }
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  cudaStream_t st = s->st;
  const uint32_t N = (uint32_t)n;
  const uint32_t S = (uint32_t)s->sv.size();
  const uint32_t packed = (reqs16 ? 1u : 0u) | (out8 ? 2u : 0u);
  s->SyncServantState();
  s->SyncFacts();
  s->SyncTopology();
  s->EnsureRing(N);

  // ---- a handful of requests: one launch, arguments in, pinned memory out (tiny.cuh) ------------------------------
  if ((reqs || reqs16) && N <= yd::kTinyMax && s->solver_pref == 0 && s->tiny_ok && S && s->n_comps) {
    s->h_small.ensure(256);
    yd::TinyArgs ta{};
    if (reqs) memcpy(ta.reqs, reqs, size_t(N) * sizeof(yd_task_req));
    else for (uint32_t i = 0; i != N; ++i) ta.reqs[i] = yd_unpack_req(reqs16[i]);
    ta.n = N;
    ta.now_ns = now_ns;
    ta.t = MakeTopo(s);
    ta.sv = s->arrays();
    ta.ring = s->ring();
    ta.out = s->h_small.as<yd_grant>();
    ta.granted_out = reinterpret_cast<unsigned long long*>(s->h_small.as<char>() + yd::kTinyMax * sizeof(yd_grant));
    ta.counters = s->d_counters.as<Counters>();
    YD_CUDA_CHECK(cudaEventRecord(s->ev[0], st));
    yd::k_solve_tiny<<<1, 1024, 0, st>>>(ta);
    YD_CUDA_CHECK(cudaGetLastError());
    YD_CUDA_CHECK(cudaEventRecord(s->ev[5], st));
    YD_CUDA_CHECK(cudaStreamSynchronize(st));
    if (out) memcpy(out, ta.out, size_t(N) * sizeof(yd_grant));
    else for (uint32_t i = 0; i != N; ++i) out8[i] = yd_pack_grant(ta.out[i], *ids_out);
    const unsigned long long granted = *ta.granted_out;
    s->next_id += granted;
    s->staged_n = 0;
    float ms = 0;
    cudaEventElapsedTime(&ms, s->ev[0], s->ev[5]);
    s->stats = yd_solve_stats{};
    s->stats_times_pending = 0;
    s->stats.total_ms = s->stats.solve_ms = ms;
    s->stats.decisions = N;
    s->stats.granted = granted;
    s->stats.kernel_launches = 1;
    s->stats.solver = 3;
    s->stats.h2d_bytes = 0;  // the requests are kernel arguments
    s->stats.d2h_bytes = size_t(N) * sizeof(yd_grant) + 8;  // written by the kernel into pinned host memory
    s->have_stats = true;
    return;
  }

  // Size classes: grids, scratch arrays and memsets are dimensioned for the next power of
  // two; kernels read the exact n from DynParams.
  const uint32_t Nb = (uint32_t)NextPow2(N, 1024);
  // The slot table: kept across solves (all running_tasks values of every servant) while it is small enough,
  // else rebuilt per solve and clamped to the batch size.
  // Merge-solver chunk: more, shorter chunks pay while the request-side passes are short (measured on a B200: cfg2-random
  // 306 vs 349 us, cfg-self 181 vs 199 us at 256 vs 512 slots; at 1 M requests 551 vs 515 us)
  if (s->merge_chunk_auto && !s->shard) s->merge_chunk = Nb <= 262144 ? 256u : 512u;
  const size_t static_bound = S ? s->static_bound_cache : 0;  // (= StaticSlotBound(s), kept by SyncFacts)
  const bool want_static = s->solver_pref != 1 && static_bound <= kStaticSlotLimit;
  size_t slot_bound = static_bound;
  if (!want_static) {
    slot_bound = 0;
    for (auto&& v : s->sv) slot_bound += size_t(std::min(std::min(v.nproc, v.max_tasks), N)) + 1;
  }
  if (slot_bound > 0x7ffffff0ull) { fprintf(stderr, "ydsched: slot table too large\n"); abort(); }
  const size_t slot_b = (size_t)NextPow2(std::max<size_t>(slot_bound, 1), 4096);
  if (!want_static) s->order_static = false;
  const uint32_t nb = (Nb + 1023) / 1024;
  s->d_reqs.ensure(size_t(Nb) * sizeof(yd_task_req));
  s->res_words = Nb;
  s->d_res.ensure(size_t(Nb) * 4 + yd::kClsTableSize * 8);
  s->d_out.ensure(size_t(Nb) * sizeof(yd_grant));
  if (reqs16) s->d_reqs16.ensure(size_t(Nb) * sizeof(yd_task_req16));
  if (out8) s->d_out8.ensure(size_t(Nb) * sizeof(yd_grant8));
  s->d_blk.ensure(size_t(nb) * 4);
  s->d_row_off.ensure(size_t(S + 1) * 4);
  s->d_row_len.ensure(size_t(S + 1) * 4);
  s->d_codes.ensure(slot_b * (s->wide ? 8 : 4));
  s->d_slot_owner.ensure(slot_b * 4);

  // solver choice: 2 (slot streams) unless asked otherwise or a component is too big for it
  // (the slot-stream solver takes components of any size: its sequential fallback keeps running_tasks of a
  // component beyond kStreamMaxComponent servants in HBM instead of shared memory)
  uint32_t solver = s->solver_pref == 1 ? 1 : 2;
  if (solver == 1 && s->max_comp_servants > kRowscanMaxComponent) solver = 2;  // the row-scan solver holds 8192 servants per component

  yd::DynParams* hd = s->h_dyn.as<yd::DynParams>();
  hd->n = N;
  hd->slot_clamp = N;
  hd->now_ns = now_ns;
  hd->ring_lo = s->lo;
  hd->ring_next = s->next_id;
  s->fsc.dyn = *hd;

  uint32_t launches = 0;
  hp[1] = hp_now();
  YD_CUDA_CHECK(cudaEventRecord(s->ev[0], st));
  // The request upload runs on its own stream so that the slot table and its sort (which
  // do not read the requests) overlap it; consumers wait on ev_h2d.
  // (Page-locked caller arrays -- yd_alloc_host -- are not copied at all when the fused kernel runs: its first phase
  // reads the requests over PCIe itself and, solo, its last phase writes the grants straight into the caller's array.)
  bool uploaded = false;
  auto upload = [&]() {
    if (uploaded) return;
    if (reqs) {
      YD_CUDA_CHECK(cudaMemcpyAsync(s->d_reqs.p, reqs, size_t(N) * sizeof(yd_task_req), cudaMemcpyHostToDevice, s->st_copy));
    } else if (reqs16) {
      YD_CUDA_CHECK(cudaMemcpyAsync(s->d_reqs16.p, reqs16, size_t(N) * sizeof(yd_task_req16), cudaMemcpyHostToDevice, s->st_copy));
    }
    uploaded = true;
  };
  auto mapped_address = [&](const void* p) -> void* {
    if (!p || !s->zero_copy || (reinterpret_cast<uintptr_t>(p) & 15u)) return nullptr;  // (16-byte vector accesses)
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
  };
  const void* in_host = reqs ? static_cast<const void*>(reqs) : static_cast<const void*>(reqs16);
  void* const in_dev = mapped_address(in_host);
  void* const out_dev = mapped_address(out ? static_cast<void*>(out) : static_cast<void*>(out8));
  if (in_host) s->staged_n = 0;  // the staging area now holds this batch
  bool graphed = false;
  size_t fused_dyn = 0;  // dynamic shared memory of the solo fused kernel (0: its list offsets are read from HBM)
  uint32_t variant_ran = 0;  // the fused variant of the pass that decided the batch
  const uint32_t merge_rounds_cfg = s->merge_rounds, force_stream_cfg = s->force_stream;
  int merge_retry = 0, grow_attempts = 0;
  for (;;) {
    memset(s->h_meta.p, 0, 32);
    graphed = false;
    // The fused front kernel takes batches in the latency-bound regime whose (class, tile) count matrices one block
    // scans in a few rounds; it needs the kept slot order.  solo = it also writes the grants (no coupled component
    // had requests last time; if one has now, the kernel raises flag 4 and the batch is replayed with variant 1).
    uint32_t variant = 0;
    if (s->fused_cfg && s->fused_grid && s->solver_pref == 0 && solver == 2 && want_static && S && s->n_comps && Nb <= s->fused_max_nb &&
        size_t(s->cls_bound) * ((Nb + yd::kRankTile - 1) / yd::kRankTile) <= 32768 &&
        size_t(s->cls_bound) * ((slot_b + yd::kListTile - 1) / yd::kListTile) <= 32768) {
      variant = s->solo_hint ? 2u : 1u;
    }
    yd_sched::CleanSig sig_now;
    if (variant == 2) {
      if (solver == 2) PrepareStreamBuffers(s, Nb, slot_b);  // (fixes the scratch layout the signature describes)
      sig_now = yd_sched::CleanSig{g_buf_generation, s->z_cls_off, s->z_bytes, s->res_words, s->d_zero.p, s->d_res.p};
      if (s->clean_valid && s->clean_sig == sig_now) variant = 3;  // no memset nodes: the graph is the kernel alone
    }
    s->clean_valid = false;  // (whatever runs now dirties the scratch; a completed solo solve says otherwise below)
    // (a staged solve -- no request array in this call -- leaves its grants in HBM and copies them afterwards, so that
    // the device-side events around it time the solve alone)
    const bool zc_in = variant >= 1 && in_dev, zc_out = variant >= 2 && out_dev && in_host;
    hp[2] = hp_now();
    if (!zc_in) upload();
    YD_CUDA_CHECK(cudaEventRecord(s->ev_h2d, s->st_copy));
    s->fsc.zc_in = zc_in ? in_dev : nullptr;
    s->fsc.zc_out = zc_out ? out_dev : nullptr;
    s->fsc.seq += 1;
    *s->h_fsc.as<yd::FusedScalars>() = s->fsc;
    s->h_fio->done_seq = 0;
    if (s->use_graphs) {
      // make sure every buffer the sequence touches exists BEFORE capturing (no allocation
      // inside a capture), then look the size class up
      if (solver == 2) PrepareStreamBuffers(s, Nb, slot_b);
      if (solver == 2 && want_static && S && s->n_comps && (s->order_dirty || !s->order_static || s->order_slot_b != slot_b)) {
        launches += RebuildSlotOrder(s, slot_b);
      }
      yd_sched::GraphKey key;
      key.Nb = Nb; key.S = S; key.n_comps = s->n_comps; key.max_comp = s->max_comp_servants;
      key.cls_bound = s->cls_bound; key.solver = solver; key.wide = s->wide; key.slot_b = slot_b;
      key.gen = g_buf_generation; key.topo_gen = s->topo_gen; key.ring_cap = s->ring_cap;
      key.merge_rounds = s->merge_rounds; key.force_stream = s->force_stream;
      key.order_static = (solver == 2 && s->order_static) ? 1u : 0u;
      key.variant = variant; key.packed = packed;
      yd_sched::GraphEntry* hit = nullptr;
      for (auto& g : s->graphs) if (g.key == key) { hit = &g; break; }
      if (!hit) {
        cudaGraph_t graph = nullptr;
        YD_CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        uint32_t l = EnqueueSolve(s, Nb, slot_b, solver, false, true, variant, packed);
        YD_CUDA_CHECK(cudaStreamEndCapture(st, &graph));
        cudaGraphExec_t exec = nullptr;
        YD_CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
        yd_sched::GraphEntry ge;
        ge.key = key; ge.exec = exec; ge.launches = l;
        if (variant >= 2) {
          // keep the graph: its kernel node is the handle through which the scalars are patched
          size_t nn = 0;
          YD_CUDA_CHECK(cudaGraphGetNodes(graph, nullptr, &nn));
          std::vector<cudaGraphNode_t> nodes(nn);
          YD_CUDA_CHECK(cudaGraphGetNodes(graph, nodes.data(), &nn));
          for (cudaGraphNode_t nd : nodes) {
            cudaGraphNodeType ty;
            YD_CUDA_CHECK(cudaGraphNodeGetType(nd, &ty));
            if (ty == cudaGraphNodeTypeKernel) ge.knode = nd;
          }
          if (!ge.knode) { fprintf(stderr, "ydsched: no kernel node in the solo graph\n"); abort(); }
          ge.graph = graph;
          ge.fargs = s->last_fused;
          ge.fgrid = s->last_fused_grid;
          ge.fdyn = s->last_fused_dyn;
        } else {
          YD_CUDA_CHECK(cudaGraphDestroy(graph));
        }
        if (s->graphs.size() >= 16) {  // drop the oldest size class
          cudaGraphExecDestroy(s->graphs.front().exec);
          if (s->graphs.front().graph) cudaGraphDestroy(s->graphs.front().graph);
          s->graphs.erase(s->graphs.begin());
        }
        s->graphs.push_back(ge);
        hit = &s->graphs.back();
      }
      if (variant >= 2) {  // this call's scalars -> the kernel node's parameters
        hit->fargs.sc = s->fsc;
        void* kp[1] = {&hit->fargs};
        cudaKernelNodeParams np{};
        np.func = reinterpret_cast<void*>(yd::k_fused_front);
        np.gridDim = dim3(hit->fgrid);
        np.blockDim = dim3(1024);
        np.sharedMemBytes = (unsigned)hit->fdyn;
        np.kernelParams = kp;
        np.extra = nullptr;
        YD_CUDA_CHECK(cudaGraphExecKernelNodeSetParams(hit->exec, hit->knode, &np));
      }
      fused_dyn = variant >= 2 ? hit->fdyn : 0;
      hp[3] = hp_now();
      YD_CUDA_CHECK(cudaEventRecord(s->ev[1], st));
      YD_CUDA_CHECK(cudaGraphLaunch(hit->exec, st));
      YD_CUDA_CHECK(cudaEventRecord(s->ev[4], st));
      hp[4] = hp_now();
      launches += hit->launches;
      graphed = true;
    } else {
      if (solver == 2) PrepareStreamBuffers(s, Nb, slot_b);
      if (solver == 2 && want_static && S && s->n_comps && (s->order_dirty || !s->order_static || s->order_slot_b != slot_b)) {
        launches += RebuildSlotOrder(s, slot_b);
      }
      launches += EnqueueSolve(s, Nb, slot_b, solver, true, false, variant, packed);
      fused_dyn = variant >= 2 ? s->last_fused_dyn : 0;
    }
    if (solver == 1) { s->order_dirty = true; s->order_static = false; }  // the row-scan solver's table overwrote the kept one
    if (zc_out) {}  // the kernel wrote the grants into the caller's page-locked array
    else if (out8) YD_CUDA_CHECK(cudaMemcpyAsync(out8, s->d_out8.p, size_t(N) * sizeof(yd_grant8), cudaMemcpyDeviceToHost, st));
    else YD_CUDA_CHECK(cudaMemcpyAsync(out, s->d_out.p, size_t(N) * sizeof(yd_grant), cudaMemcpyDeviceToHost, st));
    YD_CUDA_CHECK(cudaEventRecord(s->ev[5], st));
    hp[5] = hp_now();
    YD_CUDA_CHECK(cudaStreamSynchronize(st));
    hp[6] = hp_now();
    if (variant >= 2) {  // the solo kernel's report: flags and grant count (there are no copy nodes in its graph)
      if (s->h_fio->done_seq != s->fsc.seq) { fprintf(stderr, "ydsched: the fused kernel left no report\n"); abort(); }
      memcpy(s->h_meta.p, const_cast<const uint32_t*>(s->h_fio->meta), 32);
      s->h_counters.as<Counters>()->granted = s->h_fio->granted;
    }
    if (s->dump_env && solver == 2 && S && s->n_comps) DumpStreamState(s, Nb, slot_b);
    if (s->fused_prof && variant) {
      unsigned long long t[9];
      YD_CUDA_CHECK(cudaMemcpy(t, s->d_fused_prof.p, sizeof t, cudaMemcpyDeviceToHost));
      fprintf(stderr, "ydsched: fused variant %u n %u ns: P1 %llu E1 %llu P3 %llu E2 %llu P5 %llu B3 %llu P6 %llu total %llu (+report/clean %lld)\n", variant, N,
              t[1] - t[0], t[2] - t[1], t[3] - t[2], t[4] - t[3], t[5] - t[4], t[6] - t[5], t[7] - t[6], t[7] - t[0], (long long)(t[8] - t[7]));
    }
    if (solver == 2 && S && s->n_comps && s->h_meta.as<uint32_t>()[1] != 0) {
      // Nothing was decided (the stream solver and the final kernels all stood down).
      const uint32_t flag = s->h_meta.as<uint32_t>()[1], ncls = s->h_meta.as<uint32_t>()[0];
      if (flag == 4) {  // the solo kernel met a component it cannot decide: the general sequence, now and next time
        s->solo_hint = false;
      } else if (flag == 2 && grow_attempts++ < 3 && s->cls_bound < yd::kMaxClasses) {  // more lists than provisioned: grow and go again
        // one list per class plus one pseudo-class list per merge-mode component
        const uint32_t want = ncls + s->h_meta.as<uint32_t>()[2] + 1;
        s->cls_bound *= 2;
        while (s->cls_bound < want && s->cls_bound < yd::kMaxClasses) s->cls_bound *= 2;
      } else if (flag == 3 && merge_retry < 2) {
        // the merge solver's boundary states had not settled after the rounds in the graph: more
        // rounds first, then the sequential solver for everything it would have decided
        if (merge_retry == 0) s->merge_rounds = std::min(s->merge_rounds * 8, s->merge_max_chunks + 2);
        else s->force_stream = 2;
        ++merge_retry;
      } else {
        if (s->max_comp_servants > kRowscanMaxComponent) {
          // More classes than the class table holds AND a component beyond the row-scan solver's reach.  n sequential
          // decisions are the first half's followed by the second half's: decide the batch as two consecutive halves
          // (each with half the requests, hence -- eventually -- few enough classes).
          if (N < 2) { fprintf(stderr, "ydsched: class table overflow on a single request\n"); abort(); }
          s->merge_rounds = merge_rounds_cfg;
          s->force_stream = force_stream_cfg;
          std::vector<yd_task_req> r(N);
          if (reqs) memcpy(r.data(), reqs, size_t(N) * sizeof(yd_task_req));
          else if (reqs16) for (uint32_t i = 0; i != N; ++i) r[i] = yd_unpack_req(reqs16[i]);
          else YD_CUDA_CHECK(cudaMemcpy(r.data(), s->d_reqs.p, size_t(N) * sizeof(yd_task_req), cudaMemcpyDeviceToHost));
          std::vector<yd_grant> g(N);
          const uint32_t h = N / 2;
          WaitImpl(s, now_ns, r.data(), nullptr, h, g.data(), nullptr, nullptr);
          WaitImpl(s, now_ns, r.data() + h, nullptr, N - h, g.data() + h, nullptr, nullptr);
          if (out) memcpy(out, g.data(), size_t(N) * sizeof(yd_grant));
          else for (uint32_t i = 0; i != N; ++i) out8[i] = yd_pack_grant(g[i], *ids_out);
          s->stats.decisions = N;
          return;
        }
        solver = 1;
      }
      continue;
    }
    if (variant == 1) s->solo_hint = s->h_meta.as<uint32_t>()[4] == 0;  // back to one launch when nothing is coupled any more
    if (variant >= 2) {  // completed: the kernel's last block has re-initialised the scratch
      if (variant == 2) sig_now = yd_sched::CleanSig{g_buf_generation, s->z_cls_off, s->z_bytes, s->res_words, s->d_zero.p, s->d_res.p};
      s->clean_sig = sig_now;
      s->clean_valid = true;
    }
    variant_ran = variant;
    break;
  }
  const Counters* c = s->h_counters.as<Counters>();
  s->next_id += c->granted;
  s->merge_rounds = merge_rounds_cfg;
  s->force_stream = force_stream_cfg;

  yd_solve_stats& stt = s->stats;
  stt = yd_solve_stats{};
  // (the event arithmetic costs a driver call apiece: done when yd_last_solve_stats asks, the events stay valid until the next solve)
  s->stats_times_pending = graphed ? 2 : 1;
  stt.decisions = N;
  stt.granted = c->granted;
  stt.kernel_launches = launches;
  stt.solver = solver;
  stt.h2d_bytes = (reqs ? size_t(N) * sizeof(yd_task_req) : reqs16 ? size_t(N) * sizeof(yd_task_req16) : 0) + sizeof(yd::DynParams);
  stt.d2h_bytes = size_t(N) * (out8 ? sizeof(yd_grant8) : sizeof(yd_grant)) + sizeof(Counters) + 32;
  s->have_stats = true;
  if (s->host_prof) {
    hp[7] = hp_now();
    fprintf(stderr, "ydsched: host us: prep %.1f (attrs+variant %.1f) upload+event+setparams %.1f launch %.1f d2h-enqueue %.1f sync-wait %.1f stats %.1f total %.1f\n",
            hp[1] - hp[0], hp[2] - hp[1], hp[3] - hp[2], hp[4] - hp[3], hp[5] - hp[4], hp[6] - hp[5], hp[7] - hp[6], hp[7] - hp[0]);
  }
  if (s->debug_env) {
    // (which path decided the batch: fused variant (0 = pipeline, 1 = front + coupled solvers, 2/3 = solo), the solo
    // kernel's shared-memory offset table, the final's launches, 64-bit slot keys, the kept slot table)
    fprintf(stderr, "ydsched: solver %u graph %d merge_rounds %llu merge_chunks %llu walks %llu windows %llu solve_ms %.3f"
            " variant %u fused_dyn %zu lite %d final_passes %u wide %d static %d\n",
            solver, (int)graphed, c->pad[0], c->pad[1], c->pad[2], c->pad[3], stt.solve_ms, variant_ran, fused_dyn,
            (int)s->fused_lite, FinalPasses(variant_ran >= 2, solver, S && s->n_comps, nb), (int)s->wide, (int)want_static);
  }
}
}  // namespace
}  // extern "C++"

// `reqs` == NULL: the first n staged requests (yd_stage_requests) are already in HBM.
void yd_wait_for_starting_new_tasks(yd_sched* s, int64_t now_ns, const yd_task_req* reqs, size_t n,
                                    yd_grant* out) {
  WaitImpl(s, now_ns, reqs, nullptr, n, out, nullptr, nullptr);
}

// The same decisions with 16-byte requests up and 8-byte grants down (ydsched.h: yd_task_req16, yd_grant8).
void yd_wait_for_starting_new_tasks_packed(yd_sched* s, int64_t now_ns, const yd_task_req16* reqs, size_t n,
                                           yd_grant8* out, yd_packed_ids* ids) {
  yd_packed_ids local;
  WaitImpl(s, now_ns, nullptr, reqs, n, nullptr, out, ids ? ids : &local);
}

// KeepTaskAlive x n, cc:142-165.
void yd_keep_task_alive(yd_sched* s, int64_t now_ns, const uint64_t* ids, size_t n, int64_t new_expires_in_ns,
                        uint8_t* ok_out) {
  if (n == 0) return;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->d_ids.ensure(n * 8);
  s->d_ok.ensure(n);
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_ids.p, ids, n * 8, cudaMemcpyHostToDevice, s->st));
  yd::k_keep_alive<<<(unsigned)((n + 255) / 256), 256, 0, s->st>>>(
      s->d_ids.as<unsigned long long>(), (uint32_t)n, (long long)now_ns, (long long)new_expires_in_ns, s->ring(),
      s->d_ok.as<uint8_t>());
  YD_CUDA_CHECK(cudaGetLastError());
  YD_CUDA_CHECK(cudaMemcpyAsync(ok_out, s->d_ok.p, n, cudaMemcpyDeviceToHost, s->st));
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
}

// FreeTask x n, cc:167-188.  Fire and forget: ordered on the solve stream.
void yd_free_tasks(yd_sched* s, const uint64_t* ids, size_t n) {
  if (n == 0) return;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->SyncServantState();
  s->d_ids.ensure(n * 8);
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_ids.p, ids, n * 8, cudaMemcpyHostToDevice, s->st));
  yd::k_free<<<(unsigned)((n + 255) / 256), 256, 0, s->st>>>(s->d_ids.as<unsigned long long>(), (uint32_t)n,
                                                              s->ring(), s->d_run.as<uint32_t>(),
                                                              s->d_counters.as<Counters>());
  YD_CUDA_CHECK(cudaGetLastError());
  // `ids` may be pageable and reused by the caller: the copy above has already
  // staged it (pageable H2D returns after staging) or the memory is pinned and we
  // must wait for the DMA.
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
}

// OnExpirationTimer, cc:498-536.
void yd_on_expiration_timer(yd_sched* s, int64_t now_ns) {
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  cudaStream_t st = s->st;
  s->SyncServantState();
  const uint32_t S_old = (uint32_t)s->sv.size();
  std::vector<uint32_t> remap;
  uint32_t kept = 0;
  bool any_expired = false;
  for (auto&& v : s->sv) any_expired |= v.expires_at < now_ns;
  if (any_expired) {
    remap.resize(S_old);
    std::vector<ServantHost> alive;
    alive.reserve(S_old);
    for (uint32_t i = 0; i != S_old; ++i) {
      if (s->sv[i].expires_at < now_ns) {
        remap[i] = kNone;
        s->running.erase(s->sv[i].observed);  // RunningTaskBookkeeper::DropServant, cc:510-511
      } else {
        remap[i] = kept++;
        alive.push_back(std::move(s->sv[i]));
      }
    }
    s->sv.swap(alive);
    s->loc2pos.clear();
    for (uint32_t i = 0; i != s->sv.size(); ++i) s->loc2pos.emplace(s->sv[i].observed, i);
    s->topo_dirty = s->facts_dirty = s->order_dirty = true;
    s->d_remap.ensure(size_t(S_old) * 4);
    YD_CUDA_CHECK(cudaMemcpyAsync(s->d_remap.p, remap.data(), size_t(S_old) * 4, cudaMemcpyHostToDevice, st));
  }
  // min_live = ~0 before the pass
  YD_CUDA_CHECK(cudaMemsetAsync(&s->d_counters.as<Counters>()->min_live, 0xFF, 8, st));
  if (s->next_id > s->lo) {
    uint64_t cnt = s->next_id - s->lo;
    yd::k_tick<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(
        s->ring(), (long long)now_ns, any_expired ? s->d_remap.as<uint32_t>() : nullptr,
        s->d_counters.as<Counters>());
    YD_CUDA_CHECK(cudaGetLastError());
  }
  if (any_expired) {
    s->d_run_tmp.ensure(std::max<size_t>(size_t(S_old) * 4, 4));
    s->d_ever_tmp.ensure(std::max<size_t>(size_t(S_old) * 8, 8));
    yd::k_compact_servants<<<(S_old + 255) / 256, 256, 0, st>>>(
        S_old, s->d_remap.as<uint32_t>(), s->d_run.as<uint32_t>(), s->d_ever.as<unsigned long long>(),
        s->d_run_tmp.as<uint32_t>(), s->d_ever_tmp.as<unsigned long long>());
    YD_CUDA_CHECK(cudaGetLastError());
    std::swap(s->d_run, s->d_run_tmp);
    std::swap(s->d_ever, s->d_ever_tmp);
    s->S_dev = kept;
  }
  s->FetchCounters();  // also makes `remap` (pageable) safe to drop
  const Counters* c = s->h_counters.as<Counters>();
  s->zombies_ub = c->zombies;
  s->lo = (c->min_live == ~0ull) ? s->next_id : c->min_live;
}

// KeepServantAlive x n (cc:190-220): registry work only, the facts go up before the next solve.
void yd_keep_servants_alive(yd_sched* s, int64_t now_ns, const yd_servant* servants, const int64_t* expires_in_ns, size_t n) {
  for (size_t i = 0; i != n; ++i) yd_keep_servant_alive(s, now_ns, &servants[i], expires_in_ns[i]);
}

extern "C++" {
namespace {
// NotifyServantRunningTasks (cc:222-277) for heartbeats of DISTINCT known servants: one upload, one
// sweep + one check kernel, one synchronisation, whatever the number of servants or reported tasks.
// `idx` = the items of the caller's array handled here, `pos` their registry positions.
void NotifyDistinct(yd_sched* s, const yd_heartbeat_item* items, const std::vector<uint32_t>& idx,
                    const std::vector<uint32_t>& pos, std::vector<std::vector<uint8_t>>& permitted) {
  const uint32_t m = (uint32_t)idx.size();
  std::vector<uint32_t> order(m);
  std::iota(order.begin(), order.end(), 0u);
  std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return pos[a] < pos[b]; });
  size_t total = 0;
  for (uint32_t k = 0; k != m; ++k) total += items[idx[k]].n_tasks;
  if (total > 0xfffffff0ull) { fprintf(stderr, "ydsched: heartbeat batch reports too many tasks\n"); abort(); }
  const bool window = s->next_id > s->lo;
  if (!window || (total == 0 && s->zombies_ub == 0)) return;  // nothing can be permitted, nothing to sweep
  // staging layout: ids[total] (u64) | item_off[m + 1] | item_pos[m] | (device only) permitted[total]
  const size_t b_ids = total * 8, b_off = (size_t(m) + 1) * 4, b_pos = size_t(m) * 4;
  s->h_small.ensure(b_ids + b_off + b_pos + total + 64);
  char* hb = s->h_small.as<char>();
  unsigned long long* h_ids = reinterpret_cast<unsigned long long*>(hb);
  uint32_t* h_off = reinterpret_cast<uint32_t*>(hb + b_ids);
  uint32_t* h_pos = h_off + m + 1;
  uint8_t* h_ok = reinterpret_cast<uint8_t*>(hb + b_ids + b_off + b_pos);
  size_t at = 0;
  for (uint32_t k = 0; k != m; ++k) {
    const yd_heartbeat_item& it = items[idx[order[k]]];
    h_off[k] = (uint32_t)at;
    h_pos[k] = pos[order[k]];
    for (size_t i = 0; i != it.n_tasks; ++i) h_ids[at++] = it.tasks[i].task_grant_id;
  }
  h_off[m] = (uint32_t)at;
  cudaStream_t st = s->st;
  s->d_ids.ensure(b_ids + b_off + b_pos + 8);
  s->d_ok.ensure(std::max<size_t>(total, 1));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_ids.p, hb, b_ids + b_off + b_pos, cudaMemcpyHostToDevice, st));
  yd::NotifyBatch nb{};
  nb.ids = s->d_ids.as<unsigned long long>();
  nb.item_off = reinterpret_cast<const uint32_t*>(s->d_ids.as<char>() + b_ids);
  nb.item_pos = nb.item_off + m + 1;
  nb.n_items = m;
  if (s->zombies_ub) {
    const uint64_t cnt = s->next_id - s->lo;
    yd::k_notify_sweep<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(s->ring(), nb, s->d_run.as<uint32_t>(),
                                                                       s->d_counters.as<Counters>());
    YD_CUDA_CHECK(cudaGetLastError());
  }
  if (total) {
    yd::k_notify_check<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(s->ring(), nb, (uint32_t)total, s->d_ok.as<uint8_t>());
    YD_CUDA_CHECK(cudaGetLastError());
    YD_CUDA_CHECK(cudaMemcpyAsync(h_ok, s->d_ok.p, total, cudaMemcpyDeviceToHost, st));
  }
  s->FetchCounters();  // the one synchronisation
  s->zombies_ub = s->h_counters.as<Counters>()->zombies;
  for (uint32_t k = 0; k != m; ++k) {
    std::vector<uint8_t>& p = permitted[idx[order[k]]];
    if (total) memcpy(p.data(), h_ok + h_off[k], p.size());
  }
}
}  // namespace
}  // extern "C++"

// NotifyServantRunningTasks x n, in array order (cc:222-277).
size_t yd_notify_servants_running_tasks(yd_sched* s, const yd_heartbeat_item* items, size_t n, uint64_t* unknown_out,
                                        size_t* unknown_counts) {
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->SyncServantState();
  std::vector<std::vector<uint8_t>> permitted(n);
  for (size_t i = 0; i != n; ++i) permitted[i].assign(items[i].n_tasks, 0);
  // Heartbeats of different servants touch disjoint leases, so any number of them is one device pass.
  // A servant that appears twice must see its first heartbeat's sweep: the batch is cut there.
  std::vector<uint32_t> idx, pos;
  std::unordered_map<uint32_t, char> seen;
  std::vector<uint32_t> item_pos(n, kNone);
  for (size_t i = 0; i != n; ++i) {
    auto it = s->loc2pos.find(items[i].servant_location ? items[i].servant_location : "");
    if (it == s->loc2pos.end()) continue;  // the servant itself expired: every id is unknown (cc:243-245)
    item_pos[i] = it->second;
    if (seen.count(it->second)) {
      NotifyDistinct(s, items, idx, pos, permitted);
      idx.clear(); pos.clear(); seen.clear();
    }
    seen.emplace(it->second, 1);
    idx.push_back((uint32_t)i);
    pos.push_back(it->second);
  }
  if (!idx.empty()) NotifyDistinct(s, items, idx, pos, permitted);
  size_t total = 0;
  for (size_t i = 0; i != n; ++i) {
    const yd_heartbeat_item& it = items[i];
    size_t k = 0;
    if (item_pos[i] == kNone) {
      for (size_t t = 0; t != it.n_tasks; ++t) unknown_out[total + k++] = it.tasks[t].task_grant_id;
    } else {
      std::vector<RunningRec> kept;
      for (size_t t = 0; t != it.n_tasks; ++t) {
        if (!permitted[i][t]) {
          unknown_out[total + k++] = it.tasks[t].task_grant_id;
        } else {
          kept.push_back(RunningRec{it.tasks[t].servant_task_id, it.tasks[t].task_grant_id,
                                    it.tasks[t].servant_location ? it.tasks[t].servant_location : "",
                                    it.tasks[t].task_digest ? it.tasks[t].task_digest : ""});
        }
      }
      // RunningTaskBookkeeper::SetServantRunningTasks, running_task_bookkeeper.cc:24-29
      s->running.erase(it.servant_location);
      s->running.emplace(it.servant_location, std::move(kept));
    }
    if (unknown_counts) unknown_counts[i] = k;
    total += k;
  }
  return total;
}

// NotifyServantRunningTasks, cc:222-277: a batch of one.
size_t yd_notify_servant_running_tasks(yd_sched* s, const char* servant_location, const yd_running_task* tasks,
                                       size_t n, uint64_t* unknown_out) {
  const yd_heartbeat_item item{servant_location, tasks, n};
  return yd_notify_servants_running_tasks(s, &item, 1, unknown_out, nullptr);
}

// RunningTaskBookkeeper::GetRunningTasks, running_task_bookkeeper.cc:36-43.
size_t yd_get_running_tasks(yd_sched* s, yd_running_task* out, size_t cap) {
  s->running_cache.clear();
  for (auto&& [k, v] : s->running) s->running_cache.insert(s->running_cache.begin(), v.begin(), v.end());
  for (size_t i = 0; i < s->running_cache.size() && i < cap; ++i) {
    auto&& t = s->running_cache[i];
    out[i] = yd_running_task{t.servant_task_id, t.task_grant_id, t.servant_location.c_str(), t.task_digest.c_str()};
  }
  return s->running_cache.size();
}

size_t yd_num_servants(yd_sched* s) { return s->sv.size(); }

uint64_t yd_grant_capacity_bound(yd_sched* s) {
  uint64_t b = 0;
  for (auto&& v : s->sv) b += std::min(v.nproc, v.max_tasks);
  return b;
}

const char* yd_servant_location(yd_sched* s, uint32_t idx) {
  return idx < s->sv.size() ? s->sv[idx].observed.c_str() : nullptr;
}

size_t yd_get_servant_state(yd_sched* s, yd_servant_state* out, size_t cap) {
  const size_t S = s->sv.size();
  if (!S || !cap) return S;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->SyncServantState();
  std::vector<uint32_t> run(S);
  std::vector<unsigned long long> ever(S);
  YD_CUDA_CHECK(cudaMemcpyAsync(run.data(), s->d_run.p, S * 4, cudaMemcpyDeviceToHost, s->st));
  YD_CUDA_CHECK(cudaMemcpyAsync(ever.data(), s->d_ever.p, S * 8, cudaMemcpyDeviceToHost, s->st));
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
  for (size_t i = 0; i < S && i < cap; ++i) {
    const ServantHost& v = s->sv[i];
    uint64_t capav = (s->FactFlags(v) & yd::kFlagLowMem)
                         ? run[i]
                         : (uint64_t)yd::capacity_at(v.max_tasks, v.nproc, v.load, run[i]);
    out[i] = yd_servant_state{run[i], ever[i], capav, v.expires_at};
  }
  return S;
}

int yd_get_servant_personality(yd_sched* s, uint32_t idx, yd_servant* out) {
  if (idx >= s->sv.size()) return 0;
  const ServantHost& v = s->sv[idx];
  s->personality_envs.clear();
  for (uint32_t e : v.envs) s->personality_envs.push_back(s->envs[e].c_str());
  if (out) {
    *out = yd_servant{v.version, v.priority, v.reason, (uint32_t)v.envs.size(), v.observed.c_str(), v.reported.c_str(),
                      s->personality_envs.data(), v.nproc, v.load, v.max_tasks, 0, v.total_mem, v.avail_mem};
  }
  return 1;
}

uint64_t yd_next_task_id(yd_sched* s) { return s->next_id * s->id_stride + s->id_offset; }

uint64_t yd_num_tasks(yd_sched* s) {
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->FetchCounters();
  return s->h_counters.as<Counters>()->alive;
}

int yd_last_solve_stats(yd_sched* s, yd_solve_stats* out) {
  if (!s->have_stats) return 0;
  if (s->stats_times_pending) {
    float ms = 0;
    yd_solve_stats& stt = s->stats;
    cudaEventElapsedTime(&ms, s->ev[0], s->ev[5]); stt.total_ms = ms;
    if (s->stats_times_pending == 2) {
      // inside a graph the phases are not separable: solve_ms is the whole device pipeline
      cudaEventElapsedTime(&ms, s->ev[1], s->ev[4]); stt.solve_ms = ms;
    } else {
      cudaEventElapsedTime(&ms, s->ev[1], s->ev[2]); stt.prep_ms = ms;
      cudaEventElapsedTime(&ms, s->ev[2], s->ev[3]); stt.solve_ms = ms;
      cudaEventElapsedTime(&ms, s->ev[3], s->ev[4]); stt.final_ms = ms;
    }
    s->stats_times_pending = 0;
  }
  *out = s->stats;
  return 1;
}

void* yd_alloc_host(size_t bytes) {
  void* p = nullptr;
  // Mapped + portable up to 32 MB: the fused kernel reads requests from / writes grants to such arrays directly (batches
  // up to 262 144 requests).  Bigger arrays only ever go through the copy engines and are allocated as before (plain
  // page-locked memory: the 240 MB + 160 MB arrays of a 10 M-request batch copied at 16 GB/s when mapped, 45 GB/s when not).
  const unsigned flags = bytes <= (32u << 20) ? (cudaHostAllocMapped | cudaHostAllocPortable) : cudaHostAllocDefault;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, flags) != cudaSuccess) return nullptr;
  return p;
}
void yd_free_host(void* p) {
  if (p) cudaFreeHost(p);
}

}  // extern "C"
#include "ydsched_rpc_impl.inc"
#include "yddump_impl.inc"
#include "ydservice_impl.inc"
#include "ydwire_impl.inc"

// ---- compilation-cache bloom pre-filter (bloom.cuh) ------------------------------------------
extern "C" {

int yd_bloom_reset(yd_sched* s, uint64_t size_in_bits, uint32_t num_hashes) {
  if (size_in_bits == 0 || size_in_bits > (1ull << 30) || num_hashes == 0) return 1;
  uint64_t bits = 8;  // max(8, next_pow2(m)) (bloom_filter.h:214-219)
  while (bits < size_in_bits) bits <<= 1;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  const size_t alloc = std::max<size_t>(bits / 8, 4);  // the kernels address the table as le32 words
  s->d_bloom.ensure(alloc);
  YD_CUDA_CHECK(cudaMemsetAsync(s->d_bloom.p, 0, alloc, s->st));
  s->bloom_bits = bits;
  s->bloom_hashes = num_hashes;
  return 0;
}

int yd_bloom_load(yd_sched* s, const uint8_t* bytes, size_t n_bytes, uint32_t num_hashes) {
  if (n_bytes == 0 || ((n_bytes * 8) & (n_bytes * 8 - 1)) || num_hashes == 0) return 1;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  s->d_bloom.ensure(std::max<size_t>(n_bytes, 4));
  YD_CUDA_CHECK(cudaMemsetAsync(s->d_bloom.p, 0, 4, s->st));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_bloom.p, bytes, n_bytes, cudaMemcpyHostToDevice, s->st));
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
  s->bloom_bits = n_bytes * 8;
  s->bloom_hashes = num_hashes;
  return 0;
}

static void BloomRun(yd_sched* s, const char* keys, size_t n, size_t key_len, size_t stride, uint8_t* out) {
  if (!s->bloom_bits) { fprintf(stderr, "ydsched: bloom filter used before yd_bloom_reset / yd_bloom_load\n"); abort(); }
  if (key_len > yd::kBloomMaxKey) { fprintf(stderr, "ydsched: bloom keys longer than %d bytes\n", yd::kBloomMaxKey); abort(); }
  if (n == 0) return;
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  const size_t span = (n - 1) * stride + key_len;
  s->d_bloom_keys.ensure(span ? span : 1);
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_bloom_keys.p, keys, span, cudaMemcpyHostToDevice, s->st));
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (out) {
    s->d_bloom_out.ensure(n);
    yd::k_bloom<false><<<grid, 128, 0, s->st>>>(s->d_bloom_keys.as<unsigned char>(), (uint32_t)n, (uint32_t)key_len, stride,
                                                s->bloom_hashes, s->bloom_bits - 1, s->d_bloom.as<uint32_t>(),
                                                s->d_bloom_out.as<uint8_t>());
    YD_CUDA_CHECK(cudaGetLastError());
    YD_CUDA_CHECK(cudaMemcpyAsync(out, s->d_bloom_out.p, n, cudaMemcpyDeviceToHost, s->st));
  } else {
    yd::k_bloom<true><<<grid, 128, 0, s->st>>>(s->d_bloom_keys.as<unsigned char>(), (uint32_t)n, (uint32_t)key_len, stride,
                                               s->bloom_hashes, s->bloom_bits - 1, s->d_bloom.as<uint32_t>(), nullptr);
    YD_CUDA_CHECK(cudaGetLastError());
  }
  YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
}

void yd_bloom_add(yd_sched* s, const char* keys, size_t n, size_t key_len, size_t stride) {
  BloomRun(s, keys, n, key_len, stride, nullptr);
}

void yd_bloom_possibly_contains(yd_sched* s, const char* keys, size_t n, size_t key_len, size_t stride, uint8_t* out) {
  if (!out) return;
  BloomRun(s, keys, n, key_len, stride, out);
}

size_t yd_bloom_get_bytes(yd_sched* s, uint8_t* out, size_t cap) {
  const size_t nbytes = s->bloom_bits / 8;
  if (out && cap && nbytes) {
    YD_CUDA_CHECK(cudaSetDevice(s->device));
    YD_CUDA_CHECK(cudaMemcpyAsync(out, s->d_bloom.p, std::min(cap, nbytes), cudaMemcpyDeviceToHost, s->st));
    YD_CUDA_CHECK(cudaStreamSynchronize(s->st));
  }
  return nbytes;
}

// ---- in-flight task index (running_index.cuh) ---------------------------------------------------

static yd::RtIndex MakeRtIndex(yd_sched* s) {
  yd::RtIndex ix{};
  ix.bytes = s->d_rt_bytes.as<unsigned char>();
  ix.off = s->d_rt_off.as<uint32_t>();
  ix.len = s->d_rt_len.as<uint32_t>();
  ix.slots = s->rt_snapshot.empty() ? nullptr : s->d_rt_slots.as<uint32_t>();
  ix.mask = s->rt_mask;
  return ix;
}

// RunningTaskKeeper::Refresh, running_task_keeper.cc:40-65.
size_t yd_running_index_refresh(yd_sched* s) {
  // the snapshot: what GetRunningTasks answers now (running_task_bookkeeper.cc:36-43)
  // (each servant's list goes to the FRONT there: same order, built back to front in O(n))
  s->rt_snapshot.clear();
  {
    std::vector<const std::vector<RunningRec>*> groups;
    for (auto&& [k, v] : s->running) groups.push_back(&v);
    for (auto it = groups.rbegin(); it != groups.rend(); ++it) {
      s->rt_snapshot.insert(s->rt_snapshot.end(), (*it)->begin(), (*it)->end());
    }
  }
  const size_t n = s->rt_snapshot.size();
  s->rt_distinct = 0;
  if (n == 0) return 0;
  if (n > 0x7fffffffull) { fprintf(stderr, "ydsched: running-task snapshot too large\n"); abort(); }
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  // digests packed on 8-byte boundaries so the kernels can use word loads
  std::vector<uint32_t> off(n), len(n);
  std::vector<unsigned long long> ids(n);
  size_t total = 0;
  for (size_t i = 0; i < n; ++i) {
    off[i] = (uint32_t)total;
    len[i] = (uint32_t)s->rt_snapshot[i].task_digest.size();
    ids[i] = s->rt_snapshot[i].servant_task_id;
    total += (len[i] + 7) & ~size_t(7);
    if (total > 0xfffffff0ull) { fprintf(stderr, "ydsched: running-task digests exceed 4 GiB\n"); abort(); }
  }
  std::vector<unsigned char> bytes(total ? total : 8, 0);
  for (size_t i = 0; i < n; ++i) memcpy(bytes.data() + off[i], s->rt_snapshot[i].task_digest.data(), len[i]);
  uint64_t cap = 1024;
  while (cap < 2 * n) cap <<= 1;  // load factor <= 0.5
  s->rt_mask = (uint32_t)(cap - 1);
  s->d_rt_bytes.ensure(bytes.size());
  s->d_rt_off.ensure(n * 4);
  s->d_rt_len.ensure(n * 4);
  s->d_rt_ids.ensure(n * 8);
  s->d_rt_slots.ensure(cap * 4 + 4);  // + the distinct-digest counter
  cudaStream_t st = s->st;
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_bytes.p, bytes.data(), bytes.size(), cudaMemcpyHostToDevice, st));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_off.p, off.data(), n * 4, cudaMemcpyHostToDevice, st));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_len.p, len.data(), n * 4, cudaMemcpyHostToDevice, st));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_ids.p, ids.data(), n * 8, cudaMemcpyHostToDevice, st));
  YD_CUDA_CHECK(cudaMemsetAsync(s->d_rt_slots.p, 0, cap * 4 + 4, st));
  uint32_t* distinct = s->d_rt_slots.as<uint32_t>() + cap;
  yd::k_rt_build<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(MakeRtIndex(s), (uint32_t)n, distinct);
  YD_CUDA_CHECK(cudaGetLastError());
  uint32_t h_distinct = 0;
  YD_CUDA_CHECK(cudaMemcpyAsync(&h_distinct, distinct, 4, cudaMemcpyDeviceToHost, st));
  YD_CUDA_CHECK(cudaStreamSynchronize(st));  // also keeps the pageable staging vectors alive long enough
  s->rt_distinct = h_distinct;
  return n;
}

size_t yd_running_index_size(yd_sched* s) { return s->rt_distinct; }

// RunningTaskKeeper::TryFindTask x n, running_task_keeper.cc:67-75.
void yd_running_index_find(yd_sched* s, const char* keys, size_t n, size_t key_len, size_t stride,
                           yd_running_hit* out) {
  if (n == 0 || !out) return;
  if (n > 0x7fffffffull || key_len > 0x7fffffffull) { fprintf(stderr, "ydsched: running-index query too large\n"); abort(); }
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  cudaStream_t st = s->st;
  const size_t span = (n - 1) * stride + key_len;
  s->d_rt_keys.ensure(span ? span : 1);
  s->d_rt_out.ensure(n * sizeof(yd_running_hit));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_keys.p, keys, span, cudaMemcpyHostToDevice, st));
  yd::k_rt_find<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(MakeRtIndex(s), s->d_rt_keys.as<unsigned char>(), (uint32_t)n,
                                                              (uint32_t)key_len, stride,
                                                              s->d_rt_ids.as<unsigned long long>(), s->d_rt_out.as<uint4>());
  YD_CUDA_CHECK(cudaGetLastError());
  YD_CUDA_CHECK(cudaMemcpyAsync(out, s->d_rt_out.p, n * sizeof(yd_running_hit), cudaMemcpyDeviceToHost, st));
  YD_CUDA_CHECK(cudaStreamSynchronize(st));
}

int yd_running_index_entry(yd_sched* s, uint32_t i, yd_running_task* out) {
  if (i >= s->rt_snapshot.size()) return 0;
  auto&& t = s->rt_snapshot[i];
  if (out) *out = yd_running_task{t.servant_task_id, t.task_grant_id, t.servant_location.c_str(), t.task_digest.c_str()};
  return 1;
}

// BASELINE configs[3] in one call: bloom probes, in-flight index probes, order-preserving compaction and the solve,
// with the queue resident in HBM from the first stage to the last (filter.cuh).
size_t yd_filter_and_wait_for_starting_new_tasks(yd_sched* s, int64_t now_ns, const yd_task_req* reqs, size_t n,
                                                 const yd_prefilter* f, uint8_t* verdict_out, yd_running_hit* hits_out,
                                                 yd_grant* grants_out) {
  if (n == 0) return 0;
  if (n > 0x40000000ull) { fprintf(stderr, "ydsched: batch too large\n"); abort(); }
  YD_CUDA_CHECK(cudaSetDevice(s->device));
  cudaStream_t st = s->st;
  const uint32_t N = (uint32_t)n;
  const uint32_t nt = (N + 1023) / 1024;
  const bool bloom = f && f->cache_keys, dedupe = f && f->task_digests;
  if (bloom) {
    if (!s->bloom_bits) { fprintf(stderr, "ydsched: bloom filter used before yd_bloom_reset / yd_bloom_load\n"); abort(); }
    if (f->cache_key_len > yd::kBloomMaxKey) { fprintf(stderr, "ydsched: bloom keys longer than %d bytes\n", yd::kBloomMaxKey); abort(); }
  }
  s->d_freqs.ensure(size_t(N) * sizeof(yd_task_req));
  s->d_fverdict.ensure(N);
  s->d_ftile.ensure(size_t(nt + 1) * 4);
  s->d_reqs.ensure(size_t(NextPow2(N, 1024)) * sizeof(yd_task_req));
  s->h_fcount.ensure(16);
  s->staged_n = 0;
  // uploads: the queue, the cache keys, the task digests (one stream: each stage starts when its input has landed)
  YD_CUDA_CHECK(cudaMemcpyAsync(s->d_freqs.p, reqs, size_t(N) * sizeof(yd_task_req), cudaMemcpyHostToDevice, st));
  if (bloom) {
    const size_t span = (n - 1) * f->cache_key_stride + f->cache_key_len;
    s->d_bloom_keys.ensure(span ? span : 1);
    s->d_bloom_out.ensure(n);
    YD_CUDA_CHECK(cudaMemcpyAsync(s->d_bloom_keys.p, f->cache_keys, span, cudaMemcpyHostToDevice, st));
  }
  if (dedupe) {
    const size_t span = (n - 1) * f->task_digest_stride + f->task_digest_len;
    s->d_rt_keys.ensure(span ? span : 1);
    s->d_rt_out.ensure(n * sizeof(yd_running_hit));
    YD_CUDA_CHECK(cudaMemcpyAsync(s->d_rt_keys.p, f->task_digests, span, cudaMemcpyHostToDevice, st));
  }
  YD_CUDA_CHECK(cudaEventRecord(s->ev_f[0], st));
  if (bloom) {
    yd::k_bloom<false><<<(N + 127) / 128, 128, 0, st>>>(s->d_bloom_keys.as<unsigned char>(), N, (uint32_t)f->cache_key_len,
                                                        f->cache_key_stride, s->bloom_hashes, s->bloom_bits - 1,
                                                        s->d_bloom.as<uint32_t>(), s->d_bloom_out.as<uint8_t>());
  }
  if (dedupe) {
    yd::k_rt_find<<<(N + 255) / 256, 256, 0, st>>>(MakeRtIndex(s), s->d_rt_keys.as<unsigned char>(), N,
                                                   (uint32_t)f->task_digest_len, f->task_digest_stride,
                                                   s->d_rt_ids.as<unsigned long long>(), s->d_rt_out.as<uint4>());
  }
  yd::k_keep_count<<<nt, 1024, 0, st>>>(bloom ? s->d_bloom_out.as<uint8_t>() : nullptr, dedupe ? s->d_rt_out.as<uint4>() : nullptr, N,
                                        s->d_fverdict.as<uint8_t>(), s->d_ftile.as<uint32_t>());
  yd::k_scan_u32<<<1, 1024, 0, st>>>(s->d_ftile.as<uint32_t>(), nt + 1, nullptr, 0, nullptr, 0);
  yd::k_keep_scatter<<<nt, 1024, 0, st>>>(s->d_freqs.as<yd_task_req>(), s->d_fverdict.as<uint8_t>(), s->d_ftile.as<uint32_t>(), N,
                                          s->d_reqs.as<yd_task_req>());
  YD_CUDA_CHECK(cudaGetLastError());
  YD_CUDA_CHECK(cudaEventRecord(s->ev_f[1], st));
  YD_CUDA_CHECK(cudaMemcpyAsync(s->h_fcount.p, s->d_ftile.as<uint32_t>() + nt, 4, cudaMemcpyDeviceToHost, st));
  YD_CUDA_CHECK(cudaMemcpyAsync(verdict_out, s->d_fverdict.p, N, cudaMemcpyDeviceToHost, st));
  if (hits_out) {
    if (dedupe) YD_CUDA_CHECK(cudaMemcpyAsync(hits_out, s->d_rt_out.p, n * sizeof(yd_running_hit), cudaMemcpyDeviceToHost, st));
    else for (size_t i = 0; i != n; ++i) hits_out[i] = yd_running_hit{0, YD_NO_SERVANT, 0};
  }
  YD_CUDA_CHECK(cudaStreamSynchronize(st));
  const uint32_t kept = *s->h_fcount.as<uint32_t>();
  float filter_ms = 0;
  cudaEventElapsedTime(&filter_ms, s->ev_f[0], s->ev_f[1]);
  if (kept) {
    s->staged_n = kept;  // the compaction wrote the solver's queue
    WaitImpl(s, now_ns, nullptr, nullptr, kept, grants_out, nullptr, nullptr);
    yd_solve_stats st2;
    yd_last_solve_stats(s, &st2);  // (turns the solve's events into milliseconds before they are reused)
  } else {
    s->stats = yd_solve_stats{};
    s->stats_times_pending = 0;
    s->have_stats = true;
  }
  // stats of the whole call: prep = the filter stages + compaction (device), solve / final = the solve's, decisions = n
  s->stats.prep_ms += filter_ms;
  s->stats.decisions = N;
  s->stats.kernel_launches += 3 + (bloom ? 1 : 0) + (dedupe ? 1 : 0);
  s->stats.h2d_bytes += size_t(N) * sizeof(yd_task_req) + (bloom ? (n - 1) * f->cache_key_stride + f->cache_key_len : 0) +
                        (dedupe ? (n - 1) * f->task_digest_stride + f->task_digest_len : 0);
  s->stats.d2h_bytes += N + 4 + (hits_out && dedupe ? n * sizeof(yd_running_hit) : 0);
  return kept;
}

}  // extern "C"

// ---- range-sharded queue over the GPUs of a node (include/ydshard.h) ------------------------------------
#include "shard_host.inc"
