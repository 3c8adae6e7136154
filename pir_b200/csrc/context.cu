// context.cu — host side of the C ABI (include/pir_b200.h): context, HBM-resident database shard, Galois key
// handles, expansion plans, workspaces and the orchestration of the kernels in kernels_*.cu.
//
// Reference call stack this file replaces (SURVEY §3.1):
//   PIRServer::processQuery (server.cpp:173-195) -> oblivious_expansion (server.cpp:105-171)
//   -> PIRDatabase::multiply / DatabaseMultiplier::multiply (database.cpp:170-258, 290-316)
//   -> CiphertextReencoder::Encode (ct_reencoder.cpp:40-71)
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <optional>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/pir_b200.h"
#include "behz_host.h"
#include "host_math.h"
#include "kernels.cuh"

using namespace pirb;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(x)                                                                                     \
  do {                                                                                            \
    cudaError_t e_ = (x);                                                                         \
    if (e_ != cudaSuccess) return fail(PIRB_INTERNAL, std::string(#x) + ": " + cudaGetErrorString(e_)); \
  } while (0)
#define RC(x)             \
  do {                    \
    int rc_ = (x);        \
    if (rc_) return rc_;  \
  } while (0)

// Captured graphs hold raw workspace pointers, so every context counts the moves of ITS buffers (alloc_epoch) and a
// graph is replayed only while that count is unchanged.  Buffers that no graph of a context depends on (plan offset
// tables, key handles: a new one never replaces a captured one) count into a process-wide dummy.
unsigned long long g_unowned_epoch = 0;
std::atomic<unsigned long long> g_next_key_id{1};

struct DevBuf {
  u64* p = nullptr;
  size_t bytes = 0;
  unsigned long long* epoch = &g_unowned_epoch;  // the owning context's alloc_epoch
  ~DevBuf() { if (p) cudaFree(p); }
  int ensure(size_t b) {
    if (b <= bytes) return 0;
    ++*epoch;
    if (p) { cudaFree(p); p = nullptr; bytes = 0; }
    cudaError_t e = cudaMalloc(&p, b);
    if (e != cudaSuccess) {
      return fail(PIRB_INTERNAL, "cudaMalloc(" + std::to_string(b) + " bytes): " + cudaGetErrorString(e));
    }
    bytes = b;
    return 0;
  }
};

// One oblivious-expansion job: every query ciphertext is the root of a binary tree (server.cpp:105-146);
// trees of all ciphertexts (server.cpp:148-171) and of all queries of a batch run level by level.
struct ExpandPlan {
  u64 total_items = 0;
  int n_trees = 0;               // trees of this plan (a sub-range of the query's ciphertexts for a d=1 shard)
  int t_first = 0;               // first query ciphertext expanded by this plan
  int n_ct_in = 0;               // ciphertexts per query in the input array
  std::vector<u64> items, base;  // per tree: outputs kept, first ct index in S
  std::vector<int> logm;
  u64 cap = 0;  // ciphertext slots in S (and in T)
  int max_logm = 0;
  u64 max_nodes = 0;  // per query, max over levels
  DevBuf d_off;       // [root_off | per level: src_off, dst_off]
  std::vector<int> lvl_ntrees;
  std::vector<size_t> lvl_src, lvl_dst;  // element positions inside d_off
};

}  // namespace

struct pirb_keys {
  unsigned long long id = g_next_key_id.fetch_add(1);  // never reused: captured graphs are keyed on it, not on the pointer
  std::vector<u32> elts;
  DevBuf d;  // [n][k][2][k+1][N]
  u64 key_limbs = 0;
  int device = 0;
  const u64* find(u32 g) const {
    for (size_t i = 0; i < elts.size(); ++i)
      if (elts[i] == g) return d.p + i * key_limbs;
    return nullptr;
  }
};

struct pirb_ctx {
  pirb_params prm;
  DevParams P;
  int device = 0, sm_count = 148;
  u32 N = 0;
  int k = 0, logn = 0, d = 0;
  u64 ctL = 0, ptL = 0;
  u32 two_er = 0;
  std::vector<u32> dims;
  u64 dim_sum = 0, reply_cts = 1, rest = 1;  // rest = prod dims[1..]
  u32 top_lo = 0, top_hi = 0;                // owned slice of dims[0]
  u64 pt_begin = 0, pt_count = 0;            // owned plaintexts (global indices)
  // which of the owned plaintexts have been loaded (re-loading a range is idempotent); `loaded` = how many
  std::vector<u8> have;
  u64 loaded = 0;
  void mark_loaded(u64 first_local, u64 n) {
    if (have.size() < pt_count) have.resize(pt_count, 0);
    for (u64 i = first_local; i < first_local + n; ++i)
      if (!have[i]) { have[i] = 1; ++loaded; }
    tc.built = false;  // the byte-planar copy follows the database
    // A captured answer graph scans the byte-planar copy as it was at capture time and never rebuilds it.  Drop them
    // all: the next call of each shape runs eagerly (rebuilding the copy), the one after captures without the repack.
    for (auto& kv : graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    graphs.clear();
  }
  u64 loaded_prefix() const {  // plaintexts loaded contiguously from the start of the shard
    if (loaded == pt_count) return pt_count;
    u64 i = 0;
    while (i < have.size() && have[i]) ++i;
    return i;
  }
  unsigned long long alloc_epoch = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;          // second branch of the answer graph (work off the critical path)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // end of the last *_dev call: the next one (possibly on another caller stream) waits on it, because all calls share
  // the context's workspaces
  cudaEvent_t ev_last = nullptr;
  bool ev_last_valid = false;
  std::vector<DevBuf> tables;
  DevBuf db, stage, work, dig, acc, xch, part, bufA[2], pts, qbuf, rbuf, svbuf;
  // key pointers of the calls with per-query Galois keys (pirb_answer_multi*): [tree level][query], uploaded before the
  // call's first launch; captured graphs read it at its fixed address, so one graph serves every mix of clients
  DevBuf ktab;
  std::map<std::tuple<u64, int, int, int>, std::unique_ptr<ExpandPlan>> plans;  // (items, single, first tree, trees)
  bool profiling = false;
  cudaEvent_t ev[PIRB_N_STAGES + 1] = {};
  bool ev_valid = false;
  u64 launches = 0;
  int scan_split = 1;
  // CUDA graphs of the whole answer path (expansion + multiply), one per (batch size, key handle, partial flag);
  // they read c->qbuf and write c->rbuf, so they stay valid as long as no workspace buffer moves.
  struct GraphEntry { cudaGraphExec_t exec = nullptr; unsigned long long epoch = 0; u64 launches = 0; };
  std::map<std::tuple<int, u32, unsigned long long, const void*, const void*>, GraphEntry> graphs;  // (op, Q, key id, in, out)
  bool use_graphs = true;
  // Multi-GPU exchange over NVLink peer memory (pirb_dist_*): one block per rank that every peer maps:
  //   [ flags: err | sv[n_sub][n_ranks] | part[n_sub][n_ranks] ] [ sv slot 0 | sv slot 1 ] [ partial slot 0 | slot 1 ]
  struct Dist {
    bool ready = false, ipc = false;
    u32 n_ranks = 0, rank = 0, max_local = 0, n_sub = 0, sub_q = 0;  // sub_q = local queries per sub-batch
    u32 rows_per_rank = 0;
    u64 sv_qstride = 0;                       // limbs per query in a selection-vector slot (compact layout)
    // tensor-core mode: the last-dimension entries travel repacked into the scan's operand layout (svT region of the
    // slot, [coefficient][slot rows][Kp] bytes) instead of as u64 limbs in the per-query part
    bool tc_mode = false;
    TcGeom g = {};
    u32 sub_rows = 0;                         // svT rows per coefficient of ONE sub-batch: n_ranks * sub_q * 2 * nb
    u64 sub_bytes = 0;                        // bytes of one sub-batch's svT region [coefficient][sub_rows][Kp]
    u64 svt_off = 0;                          // limb offset of the svT region inside a slot
    DevBuf stage;                             // local repacking of the rank's own queries before the push
    u64 flag_limbs = 0, sv_slot_limbs = 0, part_slot_limbs = 0;
    u64* base = nullptr;
    size_t bytes = 0;
    std::vector<void*> opened;                // IPC mappings to close
    DevBuf peer_table;
    DevBuf self_table;                        // every entry = own block: the solo warm-up step exchanges with itself
    u64 step = 0;
    u32 warmed_for = 0;
    cudaStream_t prod = nullptr, xfer = nullptr, cons = nullptr;
    cudaEvent_t ev_in = nullptr, ev_prod = nullptr, ev_xfer = nullptr, ev_done[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> ev_exp;          // per sub-batch: expansion finished (prod -> xfer)
    bool done_valid[2] = {false, false}, xfer_valid = false;
    cudaEvent_t prof[6] = {};                 // step start, expansion end, exchange end, multiply start/end, step end
    cudaEvent_t xprof[5] = {};                // transfer stream, last sub-batch: start, NTT, head push, repack, row push
    bool prof_valid = false;
    u64 timeout_ns = 20ull * 1000 * 1000 * 1000;
    u64 launches = 0;
    u32 sized_for = 0;                        // largest local batch the workspaces have been sized for
  } dist;
  DevBuf dbg;            // PIRB_DEBUG_STAMPS=<level>: clock64 phase stamps of that expansion level
  int dbg_level = -1;
  bool use_cluster = false;  // one-launch-per-level key switch on thread-block clusters
  bool dry = false;          // see LAUNCH
  // batched scan on the tensor cores (kernels_tc.cu): byte-planar copy of the shard, built on first use
  struct Tc {
    int min_queries = 4;     // batches of at least this many queries take the tensor-core scan (0 = never)
    u64 min_pt = 1024;       // ... on shards of at least this many plaintexts
    bool built = false;
    TcGeom g = {};
    u32 dimL = 0, n_rows = 0;
    u64 npt = 0;
    DevBuf dbT, svT;
    int* err = nullptr;      // mapped host memory: raised by the kernel if its pipeline times out
  } tc;
  // ciphertext-multiplication mode (PIRParameters.use_ciphertext_multiplication, database.cpp:202-211)
  struct CtMul {
    bool on = false;
    BehzC B;                     // SEAL RNSTool constants of the first data level
    DevParams PB;                // NTT tables of the auxiliary base Bsk for kernels_ntt.cu (integer engine): m[i] = bsk_i
    int nbsk = 0;                // |Bsk| = |B| + 1
    std::vector<DevBuf> tables;
    // selection entries of the scanned / of the current upper dimension (NTT form, bases q and Bsk), lower results in
    // both bases, tensor products, scaled products, relinearization scratch, level results
    DevBuf svq, sq, sb, aq, ab, dq, db, prod, dig, acc, x, low[2];
    u64 work_bytes = 4ull << 30;  // products of a level are formed for as many queries at a time as fit this budget
  } ct;
  pirb_ctx() {
    for (DevBuf* b : {&db, &stage, &work, &dig, &acc, &xch, &part, &bufA[0], &bufA[1], &pts, &qbuf, &rbuf, &svbuf, &ktab, &dbg,
                      &dist.peer_table, &dist.self_table, &dist.stage, &tc.dbT, &tc.svT})
      b->epoch = &alloc_epoch;
  }
};

namespace {

// (ctx)->dry: sizing pass — walk the same code path, grow every workspace it needs, launch nothing
#define LAUNCH(ctx, call)                                                                            \
  do {                                                                                               \
    if (!(ctx)->dry) {                                                                               \
      cudaError_t e_ = (call);                                                                       \
      ++(ctx)->launches;                                                                             \
      if (e_ != cudaSuccess) return fail(PIRB_INTERNAL, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    }                                                                                                \
  } while (0)

// uint64_t (unsigned long) <-> u64 (unsigned long long): same representation on LP64
inline u64* U(uint64_t* p) { return reinterpret_cast<u64*>(p); }
inline const u64* U(const uint64_t* p) { return reinterpret_cast<const u64*>(p); }
static_assert(sizeof(u64) == sizeof(uint64_t), "u64 must be 64 bits");

u32 inv_mod_2n(u32 g, u32 N) {
  // g odd; inverse modulo 2N (power of two) by Newton iteration
  u32 x = g;
  for (int i = 0; i < 5; ++i) x *= 2 - g * x;
  return x & (2 * N - 1);
}

// t_first / t_count select a sub-range of the query's ciphertexts (t_count < 0: all of them).  A row shard of a
// d=1 database only multiplies the selection entries of its own plaintexts, so it expands only the trees that
// cover them; their outputs are stored compactly from slot 0.
ExpandPlan* get_plan(pirb_ctx* c, u64 total_items, int single, int* rc, int t_first = 0, int t_count = -1) {
  *rc = 0;
  const u64 N = c->N;
  const int n_all = single ? 1 : (int)(total_items / N + 1);
  if (t_count < 0) { t_first = 0; t_count = n_all; }
  auto key = std::make_tuple(total_items, single, t_first, t_count);
  auto it = c->plans.find(key);
  if (it != c->plans.end()) return it->second.get();
  auto pl = std::make_unique<ExpandPlan>();
  pl->total_items = total_items;
  pl->n_trees = t_count;
  pl->t_first = t_first;
  pl->n_ct_in = n_all;
  for (int t = t_first; t < t_first + t_count; ++t) {
    const u64 before = (u64)t * N;
    u64 it_ = single ? total_items : (total_items > before ? std::min<u64>(N, total_items - before) : 0);
    pl->items.push_back(it_);
    pl->logm.push_back((int)hm::ceil_log2((uint32_t)it_));
    pl->base.push_back((u64)(t - t_first) * N);
    pl->max_logm = std::max(pl->max_logm, pl->logm.back());
  }
  pl->cap = pl->base.back() + hm::next_power_two(pl->items.back());
  const u64 Soff = 0, Toff = pl->cap * c->ctL;
  std::vector<u64> h;
  for (int t = 0; t < pl->n_trees; ++t) h.push_back(((pl->logm[t] & 1) ? Toff : Soff) + pl->base[t] * c->ctL);
  for (int j = 0; j < pl->max_logm; ++j) {
    std::vector<u64> src, dst;
    for (int t = 0; t < pl->n_trees; ++t) {
      if (pl->logm[t] <= j) continue;
      const bool src_in_S = ((pl->logm[t] - j) % 2) == 0;
      src.push_back((src_in_S ? Soff : Toff) + pl->base[t] * c->ctL);
      dst.push_back((src_in_S ? Toff : Soff) + pl->base[t] * c->ctL);
    }
    pl->lvl_ntrees.push_back((int)src.size());
    pl->lvl_src.push_back(h.size());
    h.insert(h.end(), src.begin(), src.end());
    pl->lvl_dst.push_back(h.size());
    h.insert(h.end(), dst.begin(), dst.end());
    pl->max_nodes = std::max(pl->max_nodes, (u64)src.size() << j);
  }
  if (pl->d_off.ensure(h.size() * sizeof(u64))) { *rc = PIRB_INTERNAL; return nullptr; }
  if (cudaMemcpy(pl->d_off.p, h.data(), h.size() * sizeof(u64), cudaMemcpyHostToDevice) != cudaSuccess) {
    *rc = fail(PIRB_INTERNAL, "plan upload failed");
    return nullptr;
  }
  ExpandPlan* raw = pl.get();
  c->plans[key] = std::move(pl);
  return raw;
}

// Expansion of n_queries x n_trees root ciphertexts (contiguous at d_query) into c->work.
// Result: work[qi*q_stride + i*ctL] for i < total_items (S region), coefficient form.
// lvl_lo / lvl_hi and q_first / q_count restrict the call to tree levels [lvl_lo, lvl_hi) of queries
// [q_first, q_first + q_count) of the batch (the workspaces are always sized for the whole batch): the multi-GPU flow
// runs the small top levels for all queries at once and the wide bottom levels per sub-batch.
// key_table: every query has its own Galois keys, whose pointers c->ktab holds ([level][n_queries], see
// multi_key_table); `keys` is unused.
int run_expand(pirb_ctx* c, const pirb_keys* keys, ExpandPlan* pl, const u64* d_query, int n_queries,
               cudaStream_t st, int lvl_lo = 0, int lvl_hi = -1, int q_first = 0, int q_count = -1,
               bool key_table = false) {
  const u64 q_stride = 2 * pl->cap * c->ctL;
  if (lvl_hi < 0) lvl_hi = pl->max_logm;
  if (q_count < 0) q_count = n_queries - q_first;
  RC(c->work.ensure((size_t)n_queries * q_stride * sizeof(u64)));
  const u64 nodes = pl->max_nodes * n_queries;
  if (c->use_cluster) {
    RC(c->xch.ensure((size_t)std::max<u64>(nodes, 1) * 2 * c->N * sizeof(u64)));
  } else {  // the cluster kernel keeps digits and accumulators in shared memory
    RC(c->dig.ensure((size_t)std::max<u64>(nodes, 1) * (c->k + 1) * c->k * c->N * sizeof(u64)));
    RC(c->acc.ensure((size_t)std::max<u64>(nodes, 1) * 2 * (c->k + 1) * c->N * sizeof(u64)));
  }
  u64* work = c->work.p + (u64)q_first * q_stride;
  if (lvl_lo == 0)
    LAUNCH(c, launch_place_roots(c->P, d_query + ((u64)q_first * pl->n_ct_in + pl->t_first) * c->ctL,
                                 (u64)pl->n_ct_in * c->ctL, work, pl->d_off.p, pl->n_trees, q_count, q_stride, st));
  for (int j = lvl_lo; j < lvl_hi; ++j) {
    const u32 g = (c->N >> j) + 1;
    const u64* key = nullptr;
    if (!key_table) {
      if (!keys) return fail(PIRB_INTERNAL, "Galois keys required");
      key = keys->find(g);
      if (!key) return fail(PIRB_INTERNAL, "Galois key not present for element " + std::to_string(g));
    }
    LevelArgs L;
    L.src_off = pl->d_off.p + pl->lvl_src[j];
    L.dst_off = pl->d_off.p + pl->lvl_dst[j];
    L.n_trees = pl->lvl_ntrees[j];
    L.j = j;
    L.ginv = inv_mod_2n(g, c->N);
    L.g = g;
    L.q_stride = q_stride;
    L.n_queries = q_count;
    L.key_tab = key_table ? reinterpret_cast<const u64* const*>(c->ktab.p) + (size_t)j * n_queries + q_first : nullptr;
    L.xch = c->xch.p;
    L.dbg = !c->dbg.p ? nullptr : (c->dbg_level == -2 ? c->dbg.p + (size_t)j * 65536 : (j == c->dbg_level ? c->dbg.p : nullptr));
    L.dbg_clock = (c->dbg_level >= 0 && getenv("PIRB_STAMP_CLOCK")) ? atoi(getenv("PIRB_STAMP_CLOCK")) : 0;
    const int n_nodes = (q_count * L.n_trees) << j;
    if (c->use_cluster) {
      LAUNCH(c, launch_ks_level_cluster(c->P, work, L, key, 0, st));
    } else {
      LAUNCH(c, launch_ks_digits(c->P, work, L, c->dig.p, st));
      LAUNCH(c, launch_ks_mac_intt(c->P, c->dig.p, key, c->acc.p, n_nodes, st, L.key_tab, (u32)L.n_trees << j));
      LAUNCH(c, launch_ks_combine(c->P, work, L, c->acc.p, 0, st));
    }
  }
  return 0;
}

// Last-dimension scan of n_queries selection vectors against the shard into c->part ([q][split][row][2][k][N]):
// the HBM-bound streaming kernel for single queries, the tensor-core contraction for batches.
// svt != nullptr: the last-dimension selection entries arrive already repacked into the tensor-core scan's operand
// layout (rows [row0, ...) of an svT array with rows_total rows per coefficient: the exchange slots of the multi-GPU
// flow) — tensor-core scan only, no repacking here.
struct SvtRef {
  const u8* p;
  u32 rows_total, row0;
};
int run_scan(pirb_ctx* c, const u64* sv_last, u64 sv_qstride, int n_queries, u32 dimL, u32 n_rows, u64 npt, bool allow_tc,
             int* n_split_out, cudaStream_t st, const SvtRef* svt = nullptr) {
  const DevParams& P = c->P;
  const u64 ctL = c->ctL;
  int n_split;
  // small shards are launch-latency territory: the CUDA-core batched scan is as fast there; so is it for a last
  // dimension too long for any tensor-core plan
  TcPlan plan = {};
  const bool want_tc = svt || (allow_tc && c->tc.min_queries > 0 && n_queries >= c->tc.min_queries && npt >= c->tc.min_pt);
  const bool use_tc = want_tc && tc_launch_plan(P, dimL, (u32)n_queries, &plan);
  // dist_layout chose the repacked exchange because a plan exists for the sub-batch, so one exists for these queries
  if (svt && !use_tc) return fail(PIRB_INTERNAL, "tensor-core scan: no launch plan for the exchanged operand layout");
  if (use_tc) {
    // batch of queries: dense u8 contraction per coefficient slot on the tensor cores
    pirb_ctx::Tc& T = c->tc;
    if (T.err && *T.err) return fail(PIRB_INTERNAL, "tensor-core scan: pipeline timed out in an earlier call");
    if (!T.built || T.dimL != dimL || T.n_rows != n_rows || T.npt != npt) {
      tc_geometry(P, dimL, n_rows, &T.g);
      RC(T.dbT.ensure(T.g.db_bytes));
      if (!c->dry) {
        cudaError_t e_ = launch_tc_pack_db(P, c->db.p, npt, dimL, n_rows, T.g, reinterpret_cast<u8*>(T.dbT.p), st);
        if (e_ != cudaSuccess) return fail(PIRB_INTERNAL, std::string("launch_tc_pack_db: ") + cudaGetErrorString(e_));
        T.built = true;
        T.dimL = dimL;
        T.n_rows = n_rows;
        T.npt = npt;
      }
    }
    n_split = 1;
    c->scan_split = 1;
    RC(c->part.ensure((size_t)n_queries * n_rows * ctL * sizeof(u64)));
    if (svt) {
      LAUNCH(c, launch_tc_scan_packed(P, T.g, plan, reinterpret_cast<const u8*>(T.dbT.p), n_rows, svt->p, svt->rows_total,
                                      svt->row0, (u32)n_queries, T.err, c->sm_count, c->part.p, st));
    } else {
      const u64 sv_bytes = tc_sv_bytes(P, T.g, plan);
      if (sv_bytes > T.svT.bytes) {
        RC(T.svT.ensure(sv_bytes));
        CU(cudaMemsetAsync(T.svT.p, 0, sv_bytes, st));  // the K padding is never written afterwards
      }
      LAUNCH(c, launch_tc_scan(P, T.g, plan, reinterpret_cast<const u8*>(T.dbT.p), dimL, n_rows, sv_last, sv_qstride,
                               (u32)n_queries, reinterpret_cast<u8*>(T.svT.p), T.err, c->sm_count, c->part.p, st));
    }
  } else {
    scan_config(P, dimL, n_rows, n_queries, c->sm_count, &n_split);
    c->scan_split = n_split;
    RC(c->part.ensure((size_t)n_queries * n_split * n_rows * ctL * sizeof(u64)));
    LAUNCH(c, launch_scan(P, c->db.p, npt, dimL, n_rows, sv_last, sv_qstride, n_queries, n_split, c->part.p, st));
  }
  *n_split_out = n_split;
  return 0;
}

// DatabaseMultiplier::multiply on the device.  d_sv: [n_queries] x (sv_qstride limbs apart) x [dim_sum][2][k][N]
// coefficient form; transformed to NTT form in place.  d_out: [n_queries][reply_cts][2][k][N]; coefficient form,
// or (partial != 0) the NTT-form sum over this shard's rows, to be reduced across shards.
// sv_item0 / sv_items: index of the first selection ciphertext stored at d_sv and how many are stored (a d=1 shard
// only holds the expansion of its own trees).
// compact_rows != 0: the per-query selection vector holds only this shard's rows of the first dimension (compact_rows
// slots, own row r at slot r - top_lo) followed by the other dimensions — the layout of the multi-GPU exchange slots.
int run_multiply(pirb_ctx* c, u64* d_sv, u64 sv_qstride, int n_queries, u64* d_out, int partial, cudaStream_t st,
                 bool sv_is_ntt = false, u64 sv_item0 = 0, u64 sv_items = ~0ull, u32 compact_rows = 0,
                 const SvtRef* svt = nullptr) {
  if (c->ct.on)
    return fail(PIRB_INVALID_ARGUMENT,
                "context is in ciphertext-multiplication mode: use pirb_answer_ct / pirb_db_multiply_ct");
  if (sv_items == ~0ull) sv_items = c->dim_sum;
  const int d = c->d, k = c->k;
  const u64 ctL = c->ctL;
  const DevParams& P = c->P;
  const bool prof = c->profiling && !c->dry;
  if (prof) cudaEventRecord(c->ev[1], st);
  // database.cpp:190,222: the selection vector goes to NTT form.  Only the last dimension's entries are needed by the
  // scan; for d >= 2 the others are transformed on a side branch (a second stream, captured as a parallel branch of the
  // answer graph) that joins the main one before the first upper-dimension multiply.
  bool forked = false;
  if (!sv_is_ntt) {
    u64 head = 0;
    for (int e = 0; e < d - 1; ++e) head += c->dims[e];
    if (d >= 2 && sv_item0 == 0 && sv_items == c->dim_sum && head > 0 && c->side && !c->dry) {
      CU(cudaEventRecord(c->ev_fork, st));
      CU(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
      LAUNCH(c, launch_ntt_fwd(P, d_sv, d_sv, (int)(head * 2 * k), k, 0, n_queries, sv_qstride, sv_qstride, c->side));
      CU(cudaEventRecord(c->ev_join, c->side));
      forked = true;
      LAUNCH(c, launch_ntt_fwd(P, d_sv + head * ctL, d_sv + head * ctL, (int)((sv_items - head) * 2 * k), k, 0, n_queries,
                               sv_qstride, sv_qstride, st));
    } else {
      LAUNCH(c, launch_ntt_fwd(P, d_sv, d_sv, (int)(sv_items * 2 * k), k, 0, n_queries, sv_qstride, sv_qstride, st));
    }
  }
  if (prof) cudaEventRecord(c->ev[2], st);

  const u64 out_cts = c->reply_cts;
  // the reference multiplies whatever the database holds (database.cpp:183 stops at db_.end()); here that is the
  // contiguously loaded prefix of the shard — a database with unloaded gaps is an error, not uninitialised memory
  const u64 npt = c->loaded_prefix();
  if (npt != c->loaded) return fail(PIRB_INVALID_ARGUMENT, "database has unloaded gaps");
  if (npt == 0) {
    if (forked) CU(cudaStreamWaitEvent(st, c->ev_join, 0));
    // empty shard: contributes the additive identity
    if (!c->dry) CU(cudaMemsetAsync(d_out, 0, (size_t)n_queries * out_cts * ctL * sizeof(u64), st));
    if (prof) { cudaEventRecord(c->ev[3], st); cudaEventRecord(c->ev[4], st); cudaEventRecord(c->ev[5], st); }
    return 0;
  }
  // ---- last dimension: scan against the database ----
  u32 dimL, n_rows;
  const u64* sv_last;
  if (d == 1) {
    dimL = c->top_hi - c->top_lo;
    n_rows = 1;
    sv_last = d_sv + ((u64)c->top_lo - sv_item0) * ctL;
  } else {
    dimL = c->dims[d - 1];
    n_rows = (u32)((npt + dimL - 1) / dimL);
    u64 off = compact_rows ? compact_rows : c->dims[0];
    for (int e = 1; e < d - 1; ++e) off += c->dims[e];
    sv_last = d_sv + off * ctL;  // (not present in the exchange slots when svt is given)
  }
  int n_split;
  RC(run_scan(c, sv_last, sv_qstride, n_queries, dimL, n_rows, npt, d >= 2, &n_split, st, svt));
  if (prof) cudaEventRecord(c->ev[3], st);
  if (d == 1) {
    if (partial) {
      LAUNCH(c, launch_modadd_reduce(P, c->part.p, ctL, n_split, d_out, 1, st, n_queries, (u64)n_split * ctL, ctL));
    } else {
      LAUNCH(c, launch_ntt_inv(P, c->part.p, d_out, 2 * k, k, 0, n_split, (u64)n_rows * ctL, n_queries,
                               (u64)n_split * n_rows * ctL, ctL, st));
    }
    if (prof) { cudaEventRecord(c->ev[4], st); cudaEventRecord(c->ev[5], st); }
    return 0;
  }
  // rows -> coefficient form (database.cpp:250-254)
  RC(c->bufA[0].ensure((size_t)n_queries * n_rows * ctL * sizeof(u64)));
  LAUNCH(c, launch_ntt_inv(P, c->part.p, c->bufA[0].p, (int)(n_rows * 2 * k), k, 0, n_split, (u64)n_rows * ctL,
                           n_queries, (u64)n_split * n_rows * ctL, (u64)n_rows * ctL, st));
  if (prof) cudaEventRecord(c->ev[4], st);
  if (forked) CU(cudaStreamWaitEvent(st, c->ev_join, 0));
  // ---- upper dimensions (database.cpp:196-235) ----
  u32 n_entries = n_rows;
  u32 w = 1;
  int cur = 0;
  for (int l = d - 2; l >= 0; --l) {
    const u32 dim = (l == 0) ? (c->top_hi - c->top_lo) : c->dims[l];
    const u32 n_groups = (n_entries + dim - 1) / dim;
    const u32 w_out = w * c->two_er;
    u64 sv_off = (l == 0) ? (compact_rows ? 0 : c->top_lo) : (compact_rows ? compact_rows : c->dims[0]);
    for (int e = 1; e < l; ++e) sv_off += c->dims[e];
    const u64 n_cts_in = (u64)n_entries * w;  // per query, contiguous
    RC(c->pts.ensure((size_t)n_queries * n_cts_in * c->two_er * c->ptL * sizeof(u64)));
    LAUNCH(c, launch_reencode_ntt(P, c->bufA[cur].p, c->pts.p, (int)(n_queries * n_cts_in), st));
    const u32 slices = (u32)(c->ptL / 256);
    const int ns = dim_mac_config(P, (u64)slices * w_out * n_groups * n_queries, dim, c->sm_count);
    RC(c->part.ensure((size_t)n_queries * ns * n_groups * w_out * ctL * sizeof(u64)));
    LAUNCH(c, launch_dim_mac(P, c->pts.p, n_cts_in * c->two_er * c->ptL, d_sv + sv_off * ctL, sv_qstride, n_queries, dim,
                             n_entries, n_groups, w_out, ns, c->part.p, st));
    const u64 lvl_cts = (u64)n_groups * w_out;  // per query
    if (l == 0 && partial) {
      LAUNCH(c, launch_modadd_reduce(P, c->part.p, lvl_cts * ctL, ns, d_out, lvl_cts, st, n_queries, (u64)ns * lvl_cts * ctL,
                                     lvl_cts * ctL));
    } else {
      u64* dst = d_out;
      if (l != 0) {
        RC(c->bufA[cur ^ 1].ensure((size_t)n_queries * lvl_cts * ctL * sizeof(u64)));
        dst = c->bufA[cur ^ 1].p;
      }
      LAUNCH(c, launch_ntt_inv(P, c->part.p, dst, (int)(lvl_cts * 2 * k), k, 0, ns, lvl_cts * ctL, n_queries,
                               (u64)ns * lvl_cts * ctL, lvl_cts * ctL, st));
    }
    n_entries = n_groups;
    w = w_out;
    cur ^= 1;
  }
  if (prof) cudaEventRecord(c->ev[5], st);
  return 0;
}

// One upper dimension in ciphertext-multiplication mode (database.cpp:196-211, 240-247), for every query of the batch:
//   out[g] = sum_{i} relinearize( multiply( A[g*dim + i], S[i] ) )
// A: [Q][n_entries][s1][k][N] lower results, S: [Q] x (s_bstride apart) [dim][2][k][N] selection entries, both in
// coefficient form; key: relinearization key or nullptr; out: [Q][n_groups][so][k][N], so = 2 with a key, else s1 + 1.
int ct_level(pirb_ctx* c, const u64* key, const u64* A, u64 a_bstride, int s1, const u64* S, u64 s_bstride, u32 dim,
             u32 n_entries, int n_queries, u64* out, u64 out_bstride, cudaStream_t st) {
  pirb_ctx::CtMul& M = c->ct;
  const DevParams& P = c->P;
  const BehzC& B = M.B;
  const int k = c->k, nb = M.nbsk, sp = s1 + 1;
  const u64 N = c->N;
  const u64 ctL = c->ctL;
  // selection entries of this dimension in both bases, NTT form
  const u64 sq_stride = (u64)dim * ctL, sb_stride = (u64)dim * 2 * nb * N;
  RC(M.sq.ensure((size_t)n_queries * sq_stride * sizeof(u64)));
  RC(M.sb.ensure((size_t)n_queries * sb_stride * sizeof(u64)));
  LAUNCH(c, launch_ntt_fwd(P, S, M.sq.p, (int)(dim * 2 * k), k, 0, n_queries, s_bstride, sq_stride, st));
  LAUNCH(c, launch_behz_extend(B, S, s_bstride, dim * 2, M.sb.p, sb_stride, n_queries, st));
  LAUNCH(c, launch_ntt_fwd(M.PB, M.sb.p, M.sb.p, (int)(dim * 2 * nb), nb, 0, n_queries, sb_stride, sb_stride, st));
  // per-query strides of the product workspaces
  const u64 aq_s = (u64)n_entries * s1 * k * N, ab_s = (u64)n_entries * s1 * nb * N;
  const u64 dq_s = (u64)n_entries * sp * k * N, db_s = (u64)n_entries * sp * nb * N;
  const u64 dig_s = (u64)n_entries * k * (k + 1) * N, acc_s = (u64)n_entries * 2 * (k + 1) * N, x_s = (u64)n_entries * ctL;
  u64 per_q = aq_s + ab_s + 2 * dq_s + db_s;
  if (key) per_q += dig_s + acc_s + x_s;
  int qc = (int)std::max<u64>(1, std::min<u64>((u64)n_queries, M.work_bytes / (per_q * sizeof(u64))));
  qc = (n_queries + (n_queries + qc - 1) / qc - 1) / ((n_queries + qc - 1) / qc);  // equal chunks
  RC(M.aq.ensure((size_t)qc * aq_s * sizeof(u64)));
  RC(M.ab.ensure((size_t)qc * ab_s * sizeof(u64)));
  RC(M.dq.ensure((size_t)qc * dq_s * sizeof(u64)));
  RC(M.db.ensure((size_t)qc * db_s * sizeof(u64)));
  RC(M.prod.ensure((size_t)qc * dq_s * sizeof(u64)));
  if (key) {
    if (sp != 3) return fail(PIRB_INTERNAL, "not enough relinearization keys");  // SEAL: relinearize_internal throws
    RC(M.dig.ensure((size_t)qc * dig_s * sizeof(u64)));
    RC(M.acc.ensure((size_t)qc * acc_s * sizeof(u64)));
    RC(M.x.ensure((size_t)qc * x_s * sizeof(u64)));
  }
  for (int q0 = 0; q0 < n_queries; q0 += qc) {
    const int nq = std::min(qc, n_queries - q0);
    const u64* A0 = A + (u64)q0 * a_bstride;
    // bfv_multiply (1)-(3): both operands to base q u Bsk, NTT form
    LAUNCH(c, launch_ntt_fwd(P, A0, M.aq.p, (int)(n_entries * s1 * k), k, 0, nq, a_bstride, aq_s, st));
    LAUNCH(c, launch_behz_extend(B, A0, a_bstride, n_entries * s1, M.ab.p, ab_s, nq, st));
    LAUNCH(c, launch_ntt_fwd(M.PB, M.ab.p, M.ab.p, (int)(n_entries * s1 * nb), nb, 0, nq, ab_s, ab_s, st));
    // (4) tensor product, (5) back to coefficient form
    LAUNCH(c, launch_behz_tensor(B, 0, M.aq.p, aq_s, M.sq.p + (u64)q0 * sq_stride, sq_stride, M.dq.p, dq_s, n_entries, dim, s1,
                                 nq, st));
    LAUNCH(c, launch_behz_tensor(B, 1, M.ab.p, ab_s, M.sb.p + (u64)q0 * sb_stride, sb_stride, M.db.p, db_s, n_entries, dim, s1,
                                 nq, st));
    LAUNCH(c, launch_ntt_inv(P, M.dq.p, M.dq.p, (int)(n_entries * sp * k), k, 0, 1, 0, nq, dq_s, dq_s, st));
    LAUNCH(c, launch_ntt_inv(M.PB, M.db.p, M.db.p, (int)(n_entries * sp * nb), nb, 0, 1, 0, nq, db_s, db_s, st));
    // (6)-(8) scale by t/Q, round, back to base q
    LAUNCH(c, launch_behz_floor(B, M.dq.p, dq_s, M.db.p, db_s, M.prod.p, dq_s, n_entries * sp, nq, st));
    u64* dst = out + (u64)q0 * out_bstride;
    if (key) {  // relinearize_inplace: switch_key_inplace on the third polynomial
      LAUNCH(c, launch_relin_digits(B, M.prod.p, dq_s, M.dig.p, dig_s, n_entries, nq, st));
      LAUNCH(c, launch_ntt_fwd(P, M.dig.p, M.dig.p, (int)(n_entries * k * (k + 1)), k + 1, 0, nq, dig_s, dig_s, st));
      LAUNCH(c, launch_relin_mac(B, M.dig.p, dig_s, key, M.acc.p, acc_s, n_entries, nq, st));
      LAUNCH(c, launch_ntt_inv(P, M.acc.p, M.acc.p, (int)(n_entries * 2 * (k + 1)), k + 1, 0, 1, 0, nq, acc_s, acc_s, st));
      LAUNCH(c, launch_relin_finish(B, M.prod.p, dq_s, M.acc.p, acc_s, M.x.p, x_s, n_entries, nq, st));
      LAUNCH(c, launch_ct_reduce(B, M.x.p, x_s, dst, out_bstride, n_entries, dim, 2, nq, st));
    } else {
      LAUNCH(c, launch_ct_reduce(B, M.prod.p, dq_s, dst, out_bstride, n_entries, dim, (u32)sp, nq, st));
    }
  }
  return 0;
}

// DatabaseMultiplier::multiply with ct_reencoder_ == nullptr (database.cpp:170-258) on the device.
// d_sv: [n_queries] x (sv_qstride limbs apart) x [dim_sum][2][k][N], coefficient form, NOT modified (database.cpp:188
// transforms the selection vector only on the re-encoder path).  The plaintexts are held in NTT form as always: the
// reference keeps them in coefficient form in this mode and multiply_plain transforms both operands per call
// [SEAL multiply_plain_normal] — the product is the same canonical polynomial.
// d_out: [n_queries][polys][k][N] coefficient form, polys = 2 with a relinearization key (or d = 1), else d + 1.
int run_multiply_ct(pirb_ctx* c, const pirb_keys* relin, const u64* d_sv, u64 sv_qstride, int n_queries, u64* d_out,
                    cudaStream_t st) {
  const int d = c->d, k = c->k;
  const u64 ctL = c->ctL, ptL = c->ptL;
  const DevParams& P = c->P;
  pirb_ctx::CtMul& M = c->ct;
  const u64* key = nullptr;
  if (relin) {
    key = relin->find(0);
    if (!key) return fail(PIRB_INVALID_ARGUMENT, "not a relinearization key handle (pirb_relin_keys_load)");
  }
  const u32 out_polys = (d == 1 || key) ? 2u : (u32)d + 1;
  const u64 npt = c->loaded_prefix();
  if (npt != c->loaded) return fail(PIRB_INVALID_ARGUMENT, "database has unloaded gaps");
  if (npt == 0) {
    if (!c->dry) CU(cudaMemsetAsync(d_out, 0, (size_t)n_queries * out_polys * ptL * sizeof(u64), st));
    return 0;
  }
  // ---- last dimension: scan against the database, on an NTT-form COPY of its selection entries ----
  const u32 dimL = c->dims[d - 1];
  const u32 n_rows = d == 1 ? 1u : (u32)((npt + dimL - 1) / dimL);
  const u64 off = c->dim_sum - dimL;
  const u64 svq_stride = (u64)dimL * ctL;
  RC(M.svq.ensure((size_t)n_queries * svq_stride * sizeof(u64)));
  LAUNCH(c, launch_ntt_fwd(P, d_sv + off * ctL, M.svq.p, (int)(dimL * 2 * k), k, 0, n_queries, sv_qstride, svq_stride, st));
  int n_split;
  RC(run_scan(c, M.svq.p, svq_stride, n_queries, dimL, n_rows, npt, d >= 2, &n_split, st));
  if (d == 1) {
    LAUNCH(c, launch_ntt_inv(P, c->part.p, d_out, 2 * k, k, 0, n_split, (u64)n_rows * ctL, n_queries,
                             (u64)n_split * n_rows * ctL, ctL, st));
    return 0;
  }
  RC(M.low[0].ensure((size_t)n_queries * n_rows * ctL * sizeof(u64)));
  LAUNCH(c, launch_ntt_inv(P, c->part.p, M.low[0].p, (int)(n_rows * 2 * k), k, 0, n_split, (u64)n_rows * ctL, n_queries,
                           (u64)n_split * n_rows * ctL, (u64)n_rows * ctL, st));
  // ---- upper dimensions: Evaluator::multiply (+ relinearize_inplace) per entry, summed per group ----
  u32 n_entries = n_rows;
  int s1 = 2, cur = 0;
  for (int l = d - 2; l >= 0; --l) {
    const u32 dim = c->dims[l];
    const u32 n_groups = (n_entries + dim - 1) / dim;
    u64 sv_off = 0;
    for (int e = 0; e < l; ++e) sv_off += c->dims[e];
    const int so = key ? 2 : s1 + 1;
    const u64 out_bstride = (u64)n_groups * so * ptL;
    u64* dst = d_out;
    if (l != 0) {
      RC(M.low[cur ^ 1].ensure((size_t)n_queries * out_bstride * sizeof(u64)));
      dst = M.low[cur ^ 1].p;
    }
    RC(ct_level(c, key, M.low[cur].p, (u64)n_entries * s1 * ptL, s1, d_sv + sv_off * ctL, sv_qstride, dim, n_entries,
                n_queries, dst, out_bstride, st));
    n_entries = n_groups;
    s1 = so;
    cur ^= 1;
  }
  return 0;
}

int run_answer(pirb_ctx* c, const pirb_keys* keys, const u64* d_queries, u32 n_queries, u64 n_ct, u64* d_out,
               int partial, cudaStream_t st, bool key_table = false) {
  if (!n_queries) return 0;
  if (n_ct != c->dim_sum / c->N + 1) {  // server.cpp:154-158
    return fail(PIRB_INVALID_ARGUMENT,
                "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  }
  if (c->loaded != c->pt_count) return fail(PIRB_INVALID_ARGUMENT, "database size mismatch");  // server.cpp:37-39
  int rc;
  // a row shard of a one-dimensional database expands only the query ciphertexts that cover its plaintexts
  int t_first = 0, t_count = -1;
  if (c->d == 1 && partial && c->top_hi > c->top_lo && (c->top_lo > 0 || c->top_hi < c->dims[0])) {
    t_first = (int)(c->top_lo / c->N);
    t_count = (int)((c->top_hi - 1) / c->N) - t_first + 1;
  }
  ExpandPlan* pl = get_plan(c, c->dim_sum, 0, &rc, t_first, t_count);
  if (!pl) return rc;
  c->launches = 0;
  if (c->profiling) cudaEventRecord(c->ev[0], st);
  RC(run_expand(c, keys, pl, d_queries, (int)n_queries, st, 0, -1, 0, -1, key_table));
  u64 sv_items = 0;
  for (size_t t = 0; t < pl->items.size(); ++t) sv_items = std::max(sv_items, pl->base[t] + pl->items[t]);
  RC(run_multiply(c, c->work.p, 2 * pl->cap * c->ctL, (int)n_queries, d_out, partial, st, false, (u64)pl->t_first * c->N,
                  t_count < 0 ? c->dim_sum : sv_items));
  c->ev_valid = c->profiling;
  return 0;
}

// Run `body(stream)` (a fixed sequence of kernel launches for fixed pointers and shapes), replaying a captured CUDA
// graph when one is valid for `key`.  The first call with a key runs eagerly (it sizes every workspace), the second
// one captures, later ones replay.  Any workspace reallocation bumps the context's alloc_epoch and invalidates the
// cache; key handles enter the cache key by their never-reused id.
template <typename Body>
int run_graphed(pirb_ctx* c, const std::tuple<int, u32, unsigned long long, const void*, const void*>& key, cudaStream_t st,
                Body&& body) {
  if (!c->use_graphs || c->profiling || c->dbg.p) return body(st);
  auto it = c->graphs.find(key);
  if (it != c->graphs.end() && it->second.exec && it->second.epoch == c->alloc_epoch) {
    c->launches = it->second.launches;
    CU(cudaGraphLaunch(it->second.exec, st));
    return 0;
  }
  if (it == c->graphs.end()) {  // first sight of this shape: eager run, remember that we have seen it
    if (c->graphs.size() > 64) {  // callers that keep changing pointers: do not grow without bound
      for (auto& kv : c->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
      c->graphs.clear();
    }
    c->graphs[key] = pirb_ctx::GraphEntry();
    return body(st);
  }
  if (it->second.exec) { cudaGraphExecDestroy(it->second.exec); it->second.exec = nullptr; }
  const unsigned long long epoch_before = c->alloc_epoch;
  CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
  const int rc = body(st);
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(st, &graph);
  if (rc || e != cudaSuccess || epoch_before != c->alloc_epoch) {
    // argument error, or a workspace had to grow during capture: fall back to an eager run (and try again next time)
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    if (rc) return rc;
    return body(st);
  }
  cudaGraphExec_t exec = nullptr;
  e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) {
    cudaGetLastError();
    c->use_graphs = false;
    return body(st);
  }
  it->second.exec = exec;
  it->second.epoch = c->alloc_epoch;
  it->second.launches = c->launches;
  CU(cudaGraphLaunch(exec, st));
  return 0;
}

// Answer n_queries queries held at d_in (device-accessible) into d_out (device-accessible).  tab: per-query Galois keys
// (multi_key_table; `keys` is unused), uploaded into c->ktab on st here: after the caller's DevCallOrder wait, so that
// no earlier call still reads the table, and outside any capture.  The source is pageable, so the copy has taken it
// when cudaMemcpyAsync returns.  These calls have graphs of their own (op 3) that are not keyed on any handle.
int answer_buffers(pirb_ctx* c, const pirb_keys* keys, const std::vector<const u64*>* tab, u32 n_queries, u64 n_ct,
                   int partial, cudaStream_t st, const u64* d_in = nullptr, u64* d_out = nullptr) {
  if (!d_in) d_in = c->qbuf.p;
  if (!d_out) d_out = c->rbuf.p;
  if (tab) {
    RC(c->ktab.ensure(std::max<size_t>(tab->size() * sizeof(const u64*), 256)));
    if (!tab->empty()) CU(cudaMemcpyAsync(c->ktab.p, tab->data(), tab->size() * sizeof(const u64*), cudaMemcpyHostToDevice, st));
  }
  const int op = tab ? 3 : partial;
  const unsigned long long key_id = (!tab && keys) ? keys->id : 0ull;
  return run_graphed(c, std::make_tuple(op, n_queries, key_id, (const void*)d_in, (const void*)d_out), st,
                     [&](cudaStream_t s_) { return run_answer(c, keys, d_in, n_queries, n_ct, d_out, partial, s_, tab != nullptr); });
}

// All *_dev entry points work on the context's single set of workspaces, whatever stream the caller passes: each call
// first makes its stream wait for the end of the previous call and records its own end.
struct DevCallOrder {
  pirb_ctx* c;
  cudaStream_t st;
  DevCallOrder(pirb_ctx* c_, cudaStream_t st_) : c(c_), st(st_) {
    if (c->ev_last_valid) cudaStreamWaitEvent(st, c->ev_last, 0);
  }
  ~DevCallOrder() {
    if (cudaEventRecord(c->ev_last, st) == cudaSuccess) c->ev_last_valid = true;
  }
};

// Page-locked host memory is addressable from kernels under unified addressing: the first kernel of the answer path
// can read the queries from it and the last one can write the replies into it, so a caller that passes pinned buffers
// pays no staging copies (and no extra launch latencies) on either side.
bool host_buffer_is_device_accessible(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost && a.devicePointer == p;
}

}  // namespace

// =================================================================================================
extern "C" {

const char* pirb_last_error(void) { return g_err.c_str(); }

int pirb_ctx_create(const pirb_params* prm, pirb_ctx** out) {
  if (!prm || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  const u32 N = prm->poly_modulus_degree;
  int logn = 0;
  while ((1u << logn) < N) ++logn;
  if ((1u << logn) != N || logn < 11 || logn > 14)
    return fail(PIRB_INVALID_ARGUMENT, "poly_modulus_degree must be a power of two in [2048, 16384]");
  if (prm->n_moduli < 2 || prm->n_moduli > PIRB_MAX_MODULI)
    return fail(PIRB_INVALID_ARGUMENT, "need 1..8 data moduli plus the special prime");
  if (prm->n_dims < 1 || prm->n_dims > PIRB_MAX_DIMS) return fail(PIRB_INVALID_ARGUMENT, "bad number of dimensions");
  for (u32 i = 0; i < prm->n_moduli; ++i) {
    const u64 q = prm->coeff_modulus[i];
    if (q >> 61) return fail(PIRB_INVALID_ARGUMENT, "coefficient moduli must be below 2^61");
    if (!hm::is_prime(q) || (q - 1) % (2ull * N)) return fail(PIRB_INVALID_ARGUMENT, "coefficient modulus is not an NTT prime");
    for (u32 j = 0; j < i; ++j)
      if (prm->coeff_modulus[j] == q) return fail(PIRB_INVALID_ARGUMENT, "coefficient moduli must be distinct");
  }
  const u64 t = prm->plain_modulus;
  const bool ct_mode = prm->use_ciphertext_multiplication != 0;
  // the re-encoder splits residues into chunks of log2(t) bits through 32-bit arithmetic (ct_reencoder.cpp:45); the
  // ciphertext-multiplication mode has no such limit (the reference tests a 42-bit t, correctness_test.cpp:100)
  if (t < 2 || (!ct_mode && (t >> 32))) return fail(PIRB_INVALID_ARGUMENT, "plain modulus out of range");
  if (ct_mode && prm->shard_count != 1)
    return fail(PIRB_INVALID_ARGUMENT, "ciphertext-multiplication mode runs on one GPU (shard_count must be 1)");
  for (u32 i = 0; i + 1 < prm->n_moduli; ++i)
    if (t >= prm->coeff_modulus[i]) return fail(PIRB_INVALID_ARGUMENT, "plain modulus must be below every data modulus");
  for (u32 i = 0; i < prm->n_dims; ++i)
    if (!prm->dims[i]) return fail(PIRB_INVALID_ARGUMENT, "zero dimension");
  if (prm->shard_count == 0 || prm->shard_index >= prm->shard_count)
    return fail(PIRB_INVALID_ARGUMENT, "bad shard index/count");

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(PIRB_INTERNAL, "no CUDA device available (this library has no CPU fallback)");
  if (prm->device < 0 || prm->device >= ndev) return fail(PIRB_INVALID_ARGUMENT, "bad device ordinal");
  CU(cudaSetDevice(prm->device));

  std::unique_ptr<pirb_ctx> c(new pirb_ctx());
  c->prm = *prm;
  c->device = prm->device;
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, prm->device);
  c->N = N;
  c->logn = logn;
  c->k = (int)prm->n_moduli - 1;
  c->d = (int)prm->n_dims;
  c->ctL = 2ull * c->k * N;
  c->ptL = (u64)c->k * N;
  c->dims.assign(prm->dims, prm->dims + prm->n_dims);
  for (u32 v : c->dims) c->dim_sum += v;
  for (int i = 1; i < c->d; ++i) c->rest *= c->dims[i];

  DevParams& P = c->P;
  memset(&P, 0, sizeof(P));
  P.logn = logn;
  P.k = c->k;
  P.N = N;
  P.t = t;
  P.thr = (t + 1) >> 1;
  P.ptb = hm::trunc_log2((uint32_t)t);  // pir::log2 takes a uint32_t (utils.h:43): a wider t is truncated first
  if (P.ptb == 0) return fail(PIRB_INVALID_ARGUMENT, "plain modulus too small");
  const u64 Pq = prm->coeff_modulus[c->k];
  P.half_P = Pq >> 1;
  c->tables.resize(prm->n_moduli);
  for (auto& tb : c->tables) tb.epoch = &c->alloc_epoch;
  for (u32 i = 0; i < prm->n_moduli; ++i) {
    const u64 q = prm->coeff_modulus[i];
    hm::Tables T = hm::build_tables(q, logn);
    RC(c->tables[i].ensure(12ull * N * sizeof(u64)));
    u64* base = c->tables[i].p;
    CU(cudaMemcpy(base, T.rp.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(base + N, T.rps.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(base + 2ull * N, T.irp.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(base + 3ull * N, T.irps.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
    ModC& m = P.m[i];
    m.q = q;
    hm::barrett_ratio(q, &m.ratio_hi, &m.ratio_lo);
    m.inv_n = T.inv_n;
    m.inv_n_s = T.inv_n_s;
    m.rp = base;
    m.rps = base + N;
    m.irp = base + 2ull * N;
    m.irps = base + 3ull * N;
    m.qd = (double)q;
    m.qinv = 1.0 / (double)q;
    if (!T.fw.empty()) {
      // interleave (w, w/q) pairs: [fw | iw | fin], N double2 each
      std::vector<double> packed(6ull * N);
      const std::vector<double>* a3[3] = {&T.fw, &T.iw, &T.fin};
      const std::vector<double>* b3[3] = {&T.fwi, &T.iwi, &T.fini};
      for (int t3 = 0; t3 < 3; ++t3)
        for (u64 n = 0; n < N; ++n) {
          packed[(t3 * (u64)N + n) * 2] = (*a3[t3])[n];
          packed[(t3 * (u64)N + n) * 2 + 1] = (*b3[t3])[n];
        }
      double* dbase = reinterpret_cast<double*>(base + 4ull * N);
      CU(cudaMemcpy(dbase, packed.data(), packed.size() * sizeof(double), cudaMemcpyHostToDevice));
      m.fw = reinterpret_cast<const double2*>(dbase);
      m.iw = reinterpret_cast<const double2*>(dbase + 2ull * N);
      m.fin = reinterpret_cast<const double2*>(dbase + 4ull * N);
      CU(cudaMemcpy(dbase + 6ull * N, T.fw.data(), N * sizeof(double), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(dbase + 7ull * N, T.iw.data(), N * sizeof(double), cudaMemcpyHostToDevice));
      m.fw1 = dbase + 6ull * N;
      m.iw1 = dbase + 7ull * N;
    }
    if ((int)i < c->k) {
      P.inv_P[i] = hm::invmod_prime(Pq % q, q);
      P.inv_P_s[i] = hm::shoup(P.inv_P[i], q);
      P.half_P_mod[i] = P.half_P % q;
      P.inv_P_d[i] = (double)P.inv_P[i];
      P.inv_P_di[i] = (double)P.inv_P[i] / (double)q;
      P.half_P_mod_d[i] = (double)P.half_P_mod[i];
    }
  }
  // re-encode chunk table (ct_reencoder.cpp:29-71: double log2, ceil)
  u32 e = 0;
  for (int poly = 0; poly < 2 && !ct_mode; ++poly)  // (no re-encoder in ciphertext-multiplication mode, database.cpp:302-305)
    for (int j = 0; j < c->k; ++j) {
      const u32 le = (u32)std::ceil(std::log2((double)prm->coeff_modulus[j]) / P.ptb);
      for (u32 i = 0; i < le; ++i, ++e) {
        if (e >= PIRB_MAX_REENC) return fail(PIRB_INVALID_ARGUMENT, "expansion ratio too large");
        P.re_poly[e] = (u8)poly;
        P.re_mod[e] = (u8)j;
        P.re_shift[e] = (u8)(i * P.ptb);
      }
    }
  P.two_er = (int)e;
  int max_bits = 0;
  for (u32 i = 0; i < prm->n_moduli; ++i) max_bits = std::max(max_bits, 64 - __builtin_clzll(prm->coeff_modulus[i]));
  P.lazy_ntt = (max_bits <= 62 - logn - 1) ? 1 : 0;
  P.ntt_engine = max_bits <= 44 ? 2 : (P.lazy_ntt ? 1 : 0);
  if (const char* e = getenv("PIRB_NTT_ENGINE")) {  // testing: force a slower-but-more-general engine
    const int want = atoi(e);
    if (want == 0) P.ntt_engine = 0;
    if (want == 1 && P.lazy_ntt) P.ntt_engine = 1;
  }
  P.half_bits = (max_bits + 1) / 2;
  P.half_P_d = (double)P.half_P;
  for (u32 i = 0; i < prm->n_moduli; ++i) {
    const u64 q = prm->coeff_modulus[i];
    const u64 ph = hm::powmod(2, (u64)P.half_bits, q), p2h = hm::powmod(2, 2ull * P.half_bits, q);
    P.m[i].pow_h = (double)ph;
    P.m[i].pow_h_i = (double)ph / (double)q;
    P.m[i].pow_2h = (double)p2h;
    P.m[i].pow_2h_i = (double)p2h / (double)q;
  }
  if (max_bits <= 44) {
    P.mac_mode = 2;  // Karatsuba middle term < 2^(2h+2): chains of 2^(53-2h-2) terms stay below 2^53
    P.mac_max_terms = 1u << std::min(14, 51 - 2 * P.half_bits);
  } else if (max_bits <= 48) {
    P.mac_mode = 1;
    P.half_bits = 24;
    P.mac_max_terms = 1u << 14;
  } else {
    P.mac_mode = 0;
    P.mac_max_terms = 1u << 30;
  }
  // 128-bit accumulation of products below q_max^2 wraps after 2^(128 - 2*bits) terms (64 terms for 61-bit moduli)
  P.wide_max_terms = 1u << std::min(30, 128 - 2 * max_bits);
  if (P.mac_mode == 0) P.mac_max_terms = P.wide_max_terms;
  c->two_er = e;
  for (int i = 1; i < c->d && !ct_mode; ++i) c->reply_cts *= e;  // ciphertext-multiplication mode: always one ciphertext

  if (ct_mode) {
    // SEAL RNSTool of the first data level + NTT tables of the auxiliary base Bsk (61-bit primes: integer engine)
    pirb_ctx::CtMul& M = c->ct;
    std::vector<u64> bsk;
    std::vector<u64> qv(prm->coeff_modulus, prm->coeff_modulus + c->k);
    if (c->k > PIRB_MAX_DATA || !hm::build_behz(qv.data(), c->k, Pq, N, logn, t, &M.B, &bsk))
      return fail(PIRB_INVALID_ARGUMENT, "cannot set up the auxiliary bases for ciphertext multiplication");
    M.nbsk = (int)bsk.size();
    if (M.nbsk > PIRB_MAX_MODULI) return fail(PIRB_INVALID_ARGUMENT, "too many auxiliary primes for this parameter set");
    memset(&M.PB, 0, sizeof(M.PB));
    M.PB.logn = logn;
    M.PB.k = M.nbsk;
    M.PB.N = N;
    M.PB.ntt_engine = 0;
    M.PB.lazy_ntt = 0;
    M.tables.resize(bsk.size());
    for (size_t i = 0; i < bsk.size(); ++i) {
      const hm::Tables T = hm::build_tables(bsk[i], logn);
      RC(M.tables[i].ensure(4ull * N * sizeof(u64)));
      u64* base = M.tables[i].p;
      CU(cudaMemcpy(base, T.rp.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(base + N, T.rps.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(base + 2ull * N, T.irp.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(base + 3ull * N, T.irps.data(), N * sizeof(u64), cudaMemcpyHostToDevice));
      ModC& m = M.PB.m[i];
      m.q = bsk[i];
      hm::barrett_ratio(bsk[i], &m.ratio_hi, &m.ratio_lo);
      m.inv_n = T.inv_n;
      m.inv_n_s = T.inv_n_s;
      m.rp = base;
      m.rps = base + N;
      m.irp = base + 2ull * N;
      m.irps = base + 3ull * N;
      m.qd = (double)bsk[i];
      m.qinv = 1.0 / (double)bsk[i];
    }
    if (const char* e2 = getenv("PIRB_CT_WORK_MB")) M.work_bytes = std::max<u64>(1, (u64)atoll(e2)) << 20;
    M.on = true;
  }

  // row shard of the first dimension (SURVEY §8e)
  const u32 d0 = c->dims[0];
  const u32 per = (d0 + prm->shard_count - 1) / prm->shard_count;
  c->top_lo = std::min<u64>(d0, (u64)per * prm->shard_index);
  c->top_hi = std::min<u64>(d0, (u64)c->top_lo + per);
  const u64 lo = std::min<u64>(prm->num_pt, (u64)c->top_lo * c->rest);
  const u64 hi = std::min<u64>(prm->num_pt, (u64)c->top_hi * c->rest);
  c->pt_begin = lo;
  c->pt_count = hi - lo;
  RC(c->db.ensure(std::max<size_t>(c->pt_count * c->ptL * sizeof(u64), 256)));

  {
    const char* e = getenv("PIRB_KS_CLUSTER");
    c->use_cluster = ks_cluster_supported(c->P) && !(e && *e == '0');
  }
  if (const char* e = getenv("PIRB_GRAPHS")) c->use_graphs = atoi(e) != 0;
  if (const char* e = getenv("PIRB_TC_MIN")) c->tc.min_queries = atoi(e);  // 0 disables the tensor-core scan
  if (const char* e = getenv("PIRB_TC_MIN_PT")) c->tc.min_pt = (u64)atoll(e);
  {
    int* herr = nullptr;
    if (cudaHostAlloc(&herr, sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
      *herr = 0;
      c->tc.err = herr;
    } else {
      cudaGetLastError();
      c->tc.min_queries = 0;
    }
  }
  if (const char* e = getenv("PIRB_DEBUG_STAMPS")) {
    c->dbg_level = atoi(e);
    RC(c->dbg.ensure(8 << 20));
    CU(cudaMemset(c->dbg.p, 0, 8 << 20));
  }
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_last, cudaEventDisableTiming));
  for (auto& ev : c->ev) CU(cudaEventCreate(&ev));
  *out = c.release();
  return 0;
}

void pirb_ctx_destroy(pirb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& ev : c->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto& kv : c->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  if (c->tc.err) cudaFreeHost(c->tc.err);
  {
    pirb_ctx::Dist& D = c->dist;
    for (void* pm : D.opened) cudaIpcCloseMemHandle(pm);
    if (D.base) cudaFree(D.base);
    for (cudaStream_t s_ : {D.prod, D.xfer, D.cons})
      if (s_) cudaStreamDestroy(s_);
    for (cudaEvent_t e_ : {D.ev_in, D.ev_prod, D.ev_xfer, D.ev_done[0], D.ev_done[1]})
      if (e_) cudaEventDestroy(e_);
    for (cudaEvent_t e_ : D.ev_exp) cudaEventDestroy(e_);
    for (cudaEvent_t e_ : D.prof)
      if (e_) cudaEventDestroy(e_);
    for (cudaEvent_t e_ : D.xprof)
      if (e_) cudaEventDestroy(e_);
  }
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->side) cudaStreamDestroy(c->side);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->ev_last) cudaEventDestroy(c->ev_last);
  delete c;
}

uint64_t pirb_ct_limbs(const pirb_ctx* c) { return c->ctL; }
uint64_t pirb_pt_limbs(const pirb_ctx* c) { return c->ptL; }
uint64_t pirb_key_limbs(const pirb_ctx* c) { return (u64)c->k * 2 * (c->k + 1) * c->N; }
uint32_t pirb_expansion_ratio(const pirb_ctx* c) { return c->two_er / 2; }
uint64_t pirb_reply_cts(const pirb_ctx* c) { return c->reply_cts; }
uint64_t pirb_dim_sum(const pirb_ctx* c) { return c->dim_sum; }
uint64_t pirb_query_cts(const pirb_ctx* c) { return c->dim_sum / c->N + 1; }
uint64_t pirb_shard_pt_begin(const pirb_ctx* c) { return c->pt_begin; }
uint64_t pirb_shard_pt_count(const pirb_ctx* c) { return c->pt_count; }
uint64_t pirb_db_size(const pirb_ctx* c) { return c->loaded; }

static int clip_to_shard(const pirb_ctx* c, uint64_t first, uint64_t count, u64* lo, u64* hi) {
  if (first + count > c->prm.num_pt) return fail(PIRB_INVALID_ARGUMENT, "plaintext index beyond num_pt");
  *lo = std::max<u64>(first, c->pt_begin);
  *hi = std::min<u64>(first + count, c->pt_begin + c->pt_count);
  return 0;
}

int pirb_db_load_coeff(pirb_ctx* c, const uint64_t* coeffs, uint64_t first, uint64_t count) {
  if (!c || !coeffs) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  u64 lo, hi;
  RC(clip_to_shard(c, first, count, &lo, &hi));
  const u64 chunk_max = std::max<u64>(1, (64ull << 20) / (c->N * sizeof(u64)));
  for (u64 p = lo; p < hi;) {
    const u64 n = std::min(chunk_max, hi - p);
    RC(c->stage.ensure(n * c->N * sizeof(u64)));
    CU(cudaMemcpyAsync(c->stage.p, coeffs + (p - first) * c->N, n * c->N * sizeof(u64), cudaMemcpyHostToDevice,
                       c->stream));
    LAUNCH(c, launch_db_preprocess(c->P, c->stage.p, c->db.p + (p - c->pt_begin) * c->ptL, n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->mark_loaded(p - c->pt_begin, n);
    p += n;
  }
  return 0;
}

int pirb_db_load_items(pirb_ctx* c, const uint8_t* items, uint64_t first_item, uint64_t n_items,
                       uint32_t bytes_per_item, uint32_t items_per_plaintext, uint32_t bits_per_coeff) {
  if (!c || !items || !bytes_per_item || !items_per_plaintext) return fail(PIRB_INVALID_ARGUMENT, "bad argument");
  CU(cudaSetDevice(c->device));
  if (bits_per_coeff == 0) bits_per_coeff = c->P.ptb;
  if (bits_per_coeff > c->P.ptb || bits_per_coeff > 32) return fail(PIRB_INVALID_ARGUMENT, "Bits per coefficient greater than max");
  if (first_item % items_per_plaintext) return fail(PIRB_INVALID_ARGUMENT, "first_item must start a plaintext");
  const u64 bytes_per_pt = (u64)bytes_per_item * items_per_plaintext;
  if ((bytes_per_pt * 8 + bits_per_coeff - 1) / bits_per_coeff > c->N)  // string_encoder.cpp:86-93
    return fail(PIRB_INVALID_ARGUMENT, "Number of coefficients needed greater than poly modulus degree");
  const u64 first_pt = first_item / items_per_plaintext;
  const u64 n_pt = (n_items + items_per_plaintext - 1) / items_per_plaintext;
  u64 lo, hi;
  RC(clip_to_shard(c, first_pt, n_pt, &lo, &hi));
  const u64 chunk_max = std::max<u64>(1, (64ull << 20) / (c->N * sizeof(u64)));
  DevBuf raw;
  for (u64 p = lo; p < hi;) {
    const u64 n = std::min(chunk_max, hi - p);
    const u64 byte_lo = (p - first_pt) * bytes_per_pt;
    const u64 byte_hi = std::min<u64>(n_items * (u64)bytes_per_item, (p - first_pt + n) * bytes_per_pt);
    RC(raw.ensure(std::max<u64>(byte_hi - byte_lo, 16)));
    RC(c->stage.ensure(n * c->N * sizeof(u64)));
    CU(cudaMemcpyAsync(raw.p, items + byte_lo, byte_hi - byte_lo, cudaMemcpyHostToDevice, c->stream));
    LAUNCH(c, launch_pack_items(reinterpret_cast<const u8*>(raw.p), c->stage.p, c->N, bits_per_coeff, bytes_per_pt,
                                byte_hi - byte_lo, n, c->stream));
    LAUNCH(c, launch_db_preprocess(c->P, c->stage.p, c->db.p + (p - c->pt_begin) * c->ptL, n, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->mark_loaded(p - c->pt_begin, n);
    p += n;
  }
  return 0;
}

int pirb_db_load_ntt(pirb_ctx* c, const uint64_t* limbs, uint64_t first, uint64_t count) {
  if (!c || !limbs) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  u64 lo, hi;
  RC(clip_to_shard(c, first, count, &lo, &hi));
  if (hi > lo) {
    CU(cudaMemcpy(c->db.p + (lo - c->pt_begin) * c->ptL, limbs + (lo - first) * c->ptL, (hi - lo) * c->ptL * sizeof(u64),
                  cudaMemcpyHostToDevice));
    c->mark_loaded(lo - c->pt_begin, hi - lo);
  }
  return 0;
}

int pirb_db_read_ntt(const pirb_ctx* c, uint64_t* out, uint64_t first, uint64_t count) {
  if (!c || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (first < c->pt_begin || first + count > c->pt_begin + c->pt_count)
    return fail(PIRB_INVALID_ARGUMENT, "range outside this shard");
  CU(cudaMemcpy(out, c->db.p + (first - c->pt_begin) * c->ptL, count * c->ptL * sizeof(u64), cudaMemcpyDeviceToHost));
  return 0;
}

int pirb_db_fill_random(pirb_ctx* c, uint64_t seed) {
  if (!c) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  // keyed by the GLOBAL plaintext index: the shards of a database are slices of the unsharded fill with the same seed
  LAUNCH(c, launch_fill_random(c->P, c->db.p, c->pt_count * (u64)c->k, c->k, 0, seed, c->pt_begin * (u64)c->k, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->mark_loaded(0, c->pt_count);
  return 0;
}

int pirb_keys_load(pirb_ctx* c, const uint32_t* elts, uint32_t n, const uint64_t* limbs, pirb_keys** out) {
  if (!c || !out || (n && (!elts || !limbs))) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  std::unique_ptr<pirb_keys> kz(new pirb_keys());
  kz->elts.assign(elts, elts + n);
  kz->key_limbs = pirb_key_limbs(c);
  kz->device = c->device;
  for (u32 i = 0; i < n; ++i)
    if (!(elts[i] & 1) || elts[i] >= 2 * c->N) return fail(PIRB_INVALID_ARGUMENT, "Galois element must be odd and < 2N");
  RC(kz->d.ensure(std::max<size_t>((size_t)n * kz->key_limbs * sizeof(u64), 256)));
  if (n) CU(cudaMemcpy(kz->d.p, limbs, (size_t)n * kz->key_limbs * sizeof(u64), cudaMemcpyHostToDevice));
  *out = kz.release();
  return 0;
}
void pirb_keys_destroy(pirb_keys* kz) {
  if (!kz) return;
  cudaSetDevice(kz->device);
  delete kz;  // graphs captured with this handle are keyed on its id, which is never handed out again
}

int pirb_substitute(pirb_ctx* c, const pirb_keys* keys, uint64_t* ct, uint32_t power) {
  if (!c || !keys || !ct) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  const u64* key = keys->find(power);
  if (!key) return fail(PIRB_INTERNAL, "Galois key not present");  // SEAL throws; server.cpp:72-74 -> InternalError
  cudaStream_t st = c->stream;
  RC(c->work.ensure(2 * c->ctL * sizeof(u64)));
  RC(c->dig.ensure((size_t)(c->k + 1) * c->k * c->N * sizeof(u64)));
  RC(c->acc.ensure((size_t)2 * (c->k + 1) * c->N * sizeof(u64)));
  RC(c->stage.ensure(2 * sizeof(u64)));
  const u64 offs[2] = {0, c->ctL};
  CU(cudaMemcpyAsync(c->stage.p, offs, sizeof(offs), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(c->work.p, ct, c->ctL * sizeof(u64), cudaMemcpyHostToDevice, st));
  LevelArgs L;
  L.src_off = c->stage.p;
  L.dst_off = c->stage.p + 1;
  L.n_trees = 1;
  L.j = 0;
  L.ginv = inv_mod_2n(power, c->N);
  L.g = power;
  L.q_stride = 0;
  L.n_queries = 1;
  L.dbg = nullptr;
  L.dbg_clock = 0;
  L.key_tab = nullptr;
  L.xch = nullptr;
  if (c->use_cluster) {
    RC(c->xch.ensure((size_t)2 * c->N * sizeof(u64)));
    L.xch = c->xch.p;
    LAUNCH(c, launch_ks_level_cluster(c->P, c->work.p, L, key, 1, st));
  } else {
    LAUNCH(c, launch_ks_digits(c->P, c->work.p, L, c->dig.p, st));
    LAUNCH(c, launch_ks_mac_intt(c->P, c->dig.p, key, c->acc.p, 1, st));
    LAUNCH(c, launch_ks_combine(c->P, c->work.p, L, c->acc.p, 1, st));
  }
  CU(cudaMemcpyAsync(ct, c->work.p + c->ctL, c->ctL * sizeof(u64), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

int pirb_mul_inv_pow_x(pirb_ctx* c, const uint64_t* in, uint32_t kpow, uint64_t* out) {
  if (!c || !in || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  RC(c->work.ensure(2 * c->ctL * sizeof(u64)));
  CU(cudaMemcpyAsync(c->work.p, in, c->ctL * sizeof(u64), cudaMemcpyHostToDevice, st));
  LAUNCH(c, launch_mul_inv_pow_x(c->P, c->work.p, c->work.p + c->ctL, kpow, 1, st));
  CU(cudaMemcpyAsync(out, c->work.p + c->ctL, c->ctL * sizeof(u64), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

int pirb_expand(pirb_ctx* c, const pirb_keys* keys, const uint64_t* cts, uint64_t n_ct, uint64_t total_items,
                int single, uint64_t* out) {
  if (!c || !cts || (!out && total_items)) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (single) {
    if (total_items > c->N)  // server.cpp:111-114
      return fail(PIRB_INVALID_ARGUMENT, "Cannot expand more items from a CT than poly modulus degree");
    n_ct = 1;
  } else if (n_ct != total_items / c->N + 1) {  // server.cpp:154-158
    return fail(PIRB_INVALID_ARGUMENT,
                "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  }
  int rc;
  ExpandPlan* pl = get_plan(c, total_items, single ? 1 : 0, &rc);
  if (!pl) return rc;
  cudaStream_t st = c->stream;
  RC(c->qbuf.ensure(n_ct * c->ctL * sizeof(u64)));
  CU(cudaMemcpyAsync(c->qbuf.p, cts, n_ct * c->ctL * sizeof(u64), cudaMemcpyHostToDevice, st));
  RC(run_expand(c, keys, pl, c->qbuf.p, 1, st));
  if (total_items)
    CU(cudaMemcpyAsync(out, c->work.p, total_items * c->ctL * sizeof(u64), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

int pirb_db_multiply(pirb_ctx* c, uint64_t* sv, uint64_t n_sv, uint64_t* out, uint64_t out_cap, uint64_t* out_count) {
  if (!c || !sv || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (n_sv != c->dim_sum)  // database.cpp:297-300
    return fail(PIRB_INVALID_ARGUMENT, "Selection vector size does not match dimensions");
  if (c->prm.shard_count != 1) return fail(PIRB_INVALID_ARGUMENT, "pirb_db_multiply needs an unsharded context");
  if (out_cap < c->reply_cts) return fail(PIRB_INVALID_ARGUMENT, "output buffer too small");
  cudaStream_t st = c->stream;
  RC(c->svbuf.ensure(n_sv * c->ctL * sizeof(u64)));
  RC(c->rbuf.ensure(c->reply_cts * c->ctL * sizeof(u64)));
  CU(cudaMemcpyAsync(c->svbuf.p, sv, n_sv * c->ctL * sizeof(u64), cudaMemcpyHostToDevice, st));
  c->launches = 0;
  RC(run_multiply(c, c->svbuf.p, n_sv * c->ctL, 1, c->rbuf.p, 0, st));
  if (c->loaded == 0) {
    // empty database: the reference returns an empty result vector (database.cpp:181-183)
    CU(cudaStreamSynchronize(st));
    if (out_count) *out_count = 0;
    return 0;
  }
  CU(cudaMemcpyAsync(out, c->rbuf.p, c->reply_cts * c->ctL * sizeof(u64), cudaMemcpyDeviceToHost, st));
  // mirror the in-place NTT of the selection vector entries the reference touches (database.cpp:190,222)
  u64 off = 0;
  u64 entries_below = 0;  // entries produced by the level below (n_rows for the level above the scan)
  std::vector<u64> used(c->d);
  for (int l = c->d - 1; l >= 0; --l) {
    if (l == c->d - 1) {
      used[l] = std::min<u64>(c->dims[l], c->loaded);
      entries_below = (c->loaded + c->dims[l] - 1) / c->dims[l];
    } else {
      used[l] = std::min<u64>(c->dims[l], entries_below);
      entries_below = (entries_below + c->dims[l] - 1) / c->dims[l];
    }
  }
  for (int l = 0; l < c->d; ++l) {
    if (used[l])
      CU(cudaMemcpyAsync(sv + off * c->ctL, c->svbuf.p + off * c->ctL, used[l] * c->ctL * sizeof(u64),
                         cudaMemcpyDeviceToHost, st));
    off += c->dims[l];
  }
  CU(cudaStreamSynchronize(st));
  if (out_count) *out_count = c->reply_cts;
  return 0;
}

// pirb_answer and pirb_answer_multi on host buffers (tab: see answer_buffers)
static int answer_host_common(pirb_ctx* c, const pirb_keys* keys, const std::vector<const u64*>* tab,
                              const uint64_t* queries, uint32_t n_queries, uint64_t n_ct, uint64_t* replies) {
  cudaStream_t st = c->stream;
  std::optional<DevCallOrder> order;  // the key table must not change under a *_dev call still in flight
  if (tab) order.emplace(c, st);
  const size_t qbytes = (size_t)n_queries * n_ct * c->ctL * sizeof(u64);
  const size_t rbytes = (size_t)n_queries * c->reply_cts * c->ctL * sizeof(u64);
  const char* zc = getenv("PIRB_ZERO_COPY");  // read per call so that a caller can compare both paths in one process
  const bool zero_copy = !(zc && zc[0] == '0');
  const bool q_direct = zero_copy && host_buffer_is_device_accessible(queries);
  const bool r_direct = zero_copy && host_buffer_is_device_accessible(replies);
  if (!q_direct) {
    RC(c->qbuf.ensure(std::max<size_t>(qbytes, 256)));
    CU(cudaMemcpyAsync(c->qbuf.p, queries, qbytes, cudaMemcpyHostToDevice, st));
  }
  if (!r_direct) RC(c->rbuf.ensure(std::max<size_t>(rbytes, 256)));
  RC(answer_buffers(c, keys, tab, n_queries, n_ct, 0, st, q_direct ? U(queries) : nullptr, r_direct ? U(replies) : nullptr));
  if (!r_direct) CU(cudaMemcpyAsync(replies, c->rbuf.p, rbytes, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

int pirb_answer(pirb_ctx* c, const pirb_keys* keys, const uint64_t* queries, uint32_t n_queries, uint64_t n_ct,
                uint64_t* replies) {
  if (!c || !queries || !replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (c->prm.shard_count != 1) return fail(PIRB_INVALID_ARGUMENT, "pirb_answer needs an unsharded context");
  return answer_host_common(c, keys, nullptr, queries, n_queries, n_ct, replies);
}

// ---- ciphertext-multiplication mode (PIRParameters.use_ciphertext_multiplication; database.cpp:202-211) ----
int pirb_relin_keys_load(pirb_ctx* c, const uint64_t* limbs, pirb_keys** out) {
  if (!c || !out || !limbs) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  std::unique_ptr<pirb_keys> kz(new pirb_keys());
  kz->elts.assign(1, 0u);  // not a Galois element: marks the handle as the relinearization key (RelinKeys::get_index(2) == 0)
  kz->key_limbs = pirb_key_limbs(c);
  kz->device = c->device;
  RC(kz->d.ensure(kz->key_limbs * sizeof(u64)));
  CU(cudaMemcpy(kz->d.p, limbs, kz->key_limbs * sizeof(u64), cudaMemcpyHostToDevice));
  *out = kz.release();
  return 0;
}

uint32_t pirb_reply_polys(const pirb_ctx* c, int with_relin_keys) {
  if (!c || !c->ct.on) return 2;
  return (c->d == 1 || with_relin_keys) ? 2u : (uint32_t)c->d + 1;
}

int pirb_db_multiply_ct(pirb_ctx* c, const uint64_t* sv, uint64_t n_sv, const pirb_keys* relin, uint64_t* out,
                        uint64_t out_cap_limbs, uint32_t* out_polys) {
  if (!c || !sv || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (!c->ct.on) return fail(PIRB_INVALID_ARGUMENT, "context was not created with use_ciphertext_multiplication");
  if (n_sv != c->dim_sum)  // database.cpp:297-300
    return fail(PIRB_INVALID_ARGUMENT, "Selection vector size does not match dimensions");
  const u32 polys = pirb_reply_polys(c, relin != nullptr);
  if (out_cap_limbs < (u64)polys * c->ptL) return fail(PIRB_INVALID_ARGUMENT, "output buffer too small");
  cudaStream_t st = c->stream;
  RC(c->svbuf.ensure(n_sv * c->ctL * sizeof(u64)));
  RC(c->rbuf.ensure((size_t)polys * c->ptL * sizeof(u64)));
  CU(cudaMemcpyAsync(c->svbuf.p, sv, n_sv * c->ctL * sizeof(u64), cudaMemcpyHostToDevice, st));
  c->launches = 0;
  RC(run_multiply_ct(c, relin, c->svbuf.p, n_sv * c->ctL, 1, c->rbuf.p, st));
  CU(cudaMemcpyAsync(out, c->rbuf.p, (size_t)polys * c->ptL * sizeof(u64), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (out_polys) *out_polys = c->loaded ? polys : 0;  // empty database: the reference returns no ciphertext at all
  return 0;
}

int pirb_answer_ct(pirb_ctx* c, const pirb_keys* keys, const pirb_keys* relin, const uint64_t* queries, uint32_t n_queries,
                   uint64_t n_ct, uint64_t* replies) {
  if (!c || !queries || !replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (!c->ct.on) return fail(PIRB_INVALID_ARGUMENT, "context was not created with use_ciphertext_multiplication");
  if (!n_queries) return 0;
  if (n_ct != c->dim_sum / c->N + 1)  // server.cpp:154-158
    return fail(PIRB_INVALID_ARGUMENT, "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  if (c->loaded != c->pt_count) return fail(PIRB_INVALID_ARGUMENT, "database size mismatch");  // server.cpp:37-39
  cudaStream_t st = c->stream;
  const u32 polys = pirb_reply_polys(c, relin != nullptr);
  const size_t qbytes = (size_t)n_queries * n_ct * c->ctL * sizeof(u64);
  const size_t rbytes = (size_t)n_queries * polys * c->ptL * sizeof(u64);
  RC(c->qbuf.ensure(qbytes));
  RC(c->rbuf.ensure(rbytes));
  CU(cudaMemcpyAsync(c->qbuf.p, queries, qbytes, cudaMemcpyHostToDevice, st));
  int rc;
  ExpandPlan* pl = get_plan(c, c->dim_sum, 0, &rc);
  if (!pl) return rc;
  c->launches = 0;
  RC(run_expand(c, keys, pl, c->qbuf.p, (int)n_queries, st));
  RC(run_multiply_ct(c, relin, c->work.p, 2 * pl->cap * c->ctL, (int)n_queries, c->rbuf.p, st));
  CU(cudaMemcpyAsync(replies, c->rbuf.p, rbytes, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return 0;
}

static int answer_dev_common(pirb_ctx* c, const pirb_keys* keys, const std::vector<const u64*>* tab,
                             const u64* d_queries, u32 n_queries, u64 n_ct, u64* d_out, int partial, cudaStream_t st) {
  if (!n_queries) return 0;
  if (n_ct != c->dim_sum / c->N + 1)
    return fail(PIRB_INVALID_ARGUMENT, "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  const size_t qbytes = (size_t)n_queries * n_ct * c->ctL * sizeof(u64);
  const size_t rbytes = (size_t)n_queries * c->reply_cts * c->ctL * sizeof(u64);
  RC(c->qbuf.ensure(std::max<size_t>(qbytes, 256)));
  RC(c->rbuf.ensure(std::max<size_t>(rbytes, 256)));
  DevCallOrder order(c, st);
  // the captured graph works on the context's own buffers; the caller's tensors are copied in and out
  CU(cudaMemcpyAsync(c->qbuf.p, d_queries, qbytes, cudaMemcpyDeviceToDevice, st));
  RC(answer_buffers(c, keys, tab, n_queries, n_ct, partial, st));
  CU(cudaMemcpyAsync(d_out, c->rbuf.p, rbytes, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int pirb_answer_dev(pirb_ctx* c, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries, uint64_t n_ct,
                    uint64_t* d_replies, void* stream) {
  if (!c || !d_queries || !d_replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (c->prm.shard_count != 1) return fail(PIRB_INVALID_ARGUMENT, "use pirb_answer_partial_dev on a sharded context");
  return answer_dev_common(c, keys, nullptr, U(d_queries), n_queries, n_ct, U(d_replies), 0,
                           stream ? (cudaStream_t)stream : c->stream);
}

// Checks of pirb_answer_multi*, all before anything is staged, uploaded or launched, and the key table they pass on:
// tab[j * n_queries + q] = query q's key of tree level j (Galois element N/2^j + 1).
static int multi_key_table(pirb_ctx* c, const pirb_keys* const* keys, uint32_t n_queries, uint64_t n_ct,
                           std::vector<const u64*>* tab) {
  if (c->prm.shard_count != 1) return fail(PIRB_INVALID_ARGUMENT, "pirb_answer_multi needs an unsharded context");
  if (c->ct.on) return fail(PIRB_INVALID_ARGUMENT, "pirb_answer_multi needs a re-encoder context");
  if (!n_queries) return 0;
  if (n_ct != c->dim_sum / c->N + 1)
    return fail(PIRB_INVALID_ARGUMENT, "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  if (c->loaded != c->pt_count) return fail(PIRB_INVALID_ARGUMENT, "database size mismatch");
  int rc;
  ExpandPlan* pl = get_plan(c, c->dim_sum, 0, &rc);
  if (!pl) return rc;
  const u64 key_limbs = pirb_key_limbs(c);
  tab->assign((size_t)pl->max_logm * n_queries, nullptr);
  for (u32 q = 0; q < n_queries; ++q) {
    const pirb_keys* kz = keys[q];
    const std::string where = " (query " + std::to_string(q) + ")";
    if (!kz) return fail(PIRB_INVALID_ARGUMENT, "null Galois key handle" + where);
    if (kz->key_limbs != key_limbs || kz->device != c->device)
      return fail(PIRB_INVALID_ARGUMENT, "Galois keys were loaded for a context of another shape" + where);
    for (int j = 0; j < pl->max_logm; ++j) {
      const u32 g = (c->N >> j) + 1;
      const u64* key = kz->find(g);
      if (!key) return fail(PIRB_INTERNAL, "Galois key not present for element " + std::to_string(g) + where);
      (*tab)[(size_t)j * n_queries + q] = key;
    }
  }
  return 0;
}

int pirb_answer_multi(pirb_ctx* c, const pirb_keys* const* keys, const uint64_t* queries, uint32_t n_queries,
                      uint64_t n_ct, uint64_t* replies) {
  if (!c || !keys || !queries || !replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  std::vector<const u64*> tab;
  RC(multi_key_table(c, keys, n_queries, n_ct, &tab));
  if (!n_queries) return 0;
  return answer_host_common(c, nullptr, &tab, queries, n_queries, n_ct, replies);
}

int pirb_answer_multi_dev(pirb_ctx* c, const pirb_keys* const* keys, const uint64_t* d_queries, uint32_t n_queries,
                          uint64_t n_ct, uint64_t* d_replies, void* stream) {
  if (!c || !keys || !d_queries || !d_replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  std::vector<const u64*> tab;
  RC(multi_key_table(c, keys, n_queries, n_ct, &tab));
  return answer_dev_common(c, nullptr, &tab, U(d_queries), n_queries, n_ct, U(d_replies), 0,
                           stream ? (cudaStream_t)stream : c->stream);
}

int pirb_answer_partial_dev(pirb_ctx* c, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries,
                            uint64_t n_ct, uint64_t* d_partial, void* stream) {
  if (!c || !d_queries || !d_partial) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  return answer_dev_common(c, keys, nullptr, U(d_queries), n_queries, n_ct, U(d_partial), 1,
                           stream ? (cudaStream_t)stream : c->stream);
}

int pirb_expand_ntt_dev(pirb_ctx* c, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_queries,
                        uint64_t n_ct, uint64_t* d_sv_ntt, void* stream) {
  if (!c || !d_queries || !d_sv_ntt) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (!n_queries) return 0;
  if (n_ct != c->dim_sum / c->N + 1)
    return fail(PIRB_INVALID_ARGUMENT, "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  int rc;
  ExpandPlan* pl = get_plan(c, c->dim_sum, 0, &rc);
  if (!pl) return rc;
  DevCallOrder order(c, st);
  return run_graphed(c, std::make_tuple(2, n_queries, keys ? keys->id : 0ull, (const void*)d_queries, (const void*)d_sv_ntt), st,
                     [&](cudaStream_t s_) -> int {
                       c->launches = 0;
                       if (c->profiling) cudaEventRecord(c->ev[0], s_);
                       RC(run_expand(c, keys, pl, U(d_queries), (int)n_queries, s_));
                       LAUNCH(c, launch_ntt_fwd(c->P, c->work.p, U(d_sv_ntt), (int)(c->dim_sum * 2 * c->k), c->k, 0,
                                                (int)n_queries, 2 * pl->cap * c->ctL, c->dim_sum * c->ctL, s_));
                       return 0;
                     });
}

int pirb_multiply_partial_dev(pirb_ctx* c, const uint64_t* d_sv_ntt, uint32_t n_queries, uint64_t* d_partial,
                              void* stream) {
  if (!c || !d_sv_ntt || !d_partial) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  if (!n_queries) return 0;
  if (c->loaded != c->pt_count) return fail(PIRB_INVALID_ARGUMENT, "database size mismatch");
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  DevCallOrder order(c, st);
  const int rc = run_graphed(c, std::make_tuple(3, n_queries, 0ull, (const void*)d_sv_ntt, (const void*)d_partial),
                             st, [&](cudaStream_t s_) -> int {
                               c->launches = 0;
                               if (c->profiling) cudaEventRecord(c->ev[0], s_);
                               return run_multiply(c, const_cast<u64*>(U(d_sv_ntt)), c->dim_sum * c->ctL, (int)n_queries,
                                                   U(d_partial), 1, s_, true);
                             });
  c->ev_valid = c->profiling && rc == 0;
  return rc;
}

int pirb_reduce_finish_dev(pirb_ctx* c, const uint64_t* d_partials, uint32_t n_parts, uint64_t part_stride,
                           uint32_t n_queries, uint64_t* d_replies, void* stream) {
  if (!c || !d_partials || !d_replies || !n_parts) return fail(PIRB_INVALID_ARGUMENT, "bad argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  const u64 cts = (u64)n_queries * c->reply_cts;
  DevCallOrder order(c, st);
  // the mod-q add of the partials is fused into the load side of the final inverse NTT
  LAUNCH(c, launch_ntt_inv(c->P, U(d_partials), U(d_replies), (int)(cts * 2 * c->k), c->k, 0, (int)n_parts, part_stride, 1, 0,
                           0, st));
  return 0;
}

// ---- row-sharded serving with the exchange done by the kernels over NVLink peer memory (SURVEY §8e) ----------------
// Per step and rank (all ranks run the same number of local queries in lockstep):
//   producer stream  oblivious expansion of the rank's own queries: top levels for all of them at once, the wide
//                    bottom levels per sub-batch;
//   transfer stream  per sub-batch: selection-vector NTT whose stores land in every peer's slot (first-dimension
//                    entries only at the row's owner), then a flag in every peer's block;
//   consumer stream  per sub-batch: wait for all ranks' flags, scan + re-encode + upper dimensions of the shard's rows
//                    for the n_ranks * sub_q queries of the sub-batch, partial replies into the own partial slot, flag;
//                    finally, per sub-batch: wait for all ranks' partial flags, mod-q add of the peers' partials for
//                    the own queries (loads over NVLink inside the kernel) and the final inverse NTT.
// Two slots alternate between steps; a rank reuses a slot only after its own consumer has finished the step that last
// used it, which (through the partial flags) implies every peer has finished reading that slot too.
static int dist_layout(pirb_ctx* c, u32 max_local, u32 sub_q) {
  pirb_ctx::Dist& D = c->dist;
  D.n_ranks = c->prm.shard_count;
  D.rank = c->prm.shard_index;
  D.max_local = max_local;
  D.sub_q = sub_q;
  D.n_sub = (max_local + sub_q - 1) / sub_q;
  D.rows_per_rank = (c->dims[0] + D.n_ranks - 1) / D.n_ranks;
  u64 mid = 0;
  for (int e = 1; e < c->d - 1; ++e) mid += c->dims[e];
  const u32 last = c->dims[c->d - 1];
  // Tensor-core mode whenever the consumers' scans can run on the tensor cores: a launch plan exists for a whole
  // sub-batch (n_ranks * sub_q queries; a ragged last sub-batch has fewer, and a plan that fits more queries fits
  // fewer).  The choice uses only quantities every rank agrees on: whether a plan exists does not depend on the
  // requested query tile (PIRB_TC_QT).  Otherwise the last-dimension entries travel as u64 limbs.
  const char* pk = getenv("PIRB_DIST_TC");
  TcPlan plan;
  D.tc_mode = !(pk && pk[0] == '0') && c->tc.min_queries > 0 && c->prm.num_pt / D.n_ranks >= c->tc.min_pt &&
              tc_launch_plan(c->P, last, D.n_ranks * D.sub_q, &plan);
  const u64 slot_queries = (u64)D.n_sub * D.sub_q * D.n_ranks;
  const u64 head = ((u64)D.rows_per_rank + mid) * c->ctL;
  if (D.tc_mode) {
    tc_geometry(c->P, last, 1, &D.g);
    D.sv_qstride = head;
    // one svT region per sub-batch, [coefficient][rows of the sub-batch's n_ranks * sub_q queries][Kp]: what one push
    // writes at a peer (and one scan reads) stays within a few hundred MB — peer-memory TLB reach matters for the
    // push throughput — and the scan's B tiles are dense
    D.sub_rows = (u32)(D.n_ranks * D.sub_q * 2 * D.g.nb);
    D.sub_bytes = (u64)c->k * c->N * D.sub_rows * D.g.Kp;
    D.svt_off = slot_queries * head;
    D.sv_slot_limbs = (D.svt_off + (D.n_sub * D.sub_bytes + 7) / 8 + 15) / 16 * 16;
  } else {
    D.sv_qstride = head + (u64)last * c->ctL;
    D.sv_slot_limbs = slot_queries * D.sv_qstride;
  }
  D.flag_limbs = ((1 + 2ull * D.n_sub * D.n_ranks) + 15) / 16 * 16;
  D.part_slot_limbs = slot_queries * c->reply_cts * c->ctL;
  D.bytes = (D.flag_limbs + 2 * D.sv_slot_limbs + 2 * D.part_slot_limbs) * sizeof(u64);
  return 0;
}
static u64 dist_flag_off(const pirb_ctx::Dist& D, int kind, u32 sub, u32 src) {  // kind 0: selection vectors, 1: partials
  return 1 + ((u64)kind * D.n_sub + sub) * D.n_ranks + src;
}
static u64 dist_sv_off(const pirb_ctx::Dist& D, int slot) { return D.flag_limbs + (u64)slot * D.sv_slot_limbs; }
static u64 dist_part_off(const pirb_ctx::Dist& D, int slot) {
  return D.flag_limbs + 2 * D.sv_slot_limbs + (u64)slot * D.part_slot_limbs;
}

int pirb_dist_create(pirb_ctx* c, uint32_t max_local_queries, uint32_t sub_batch, uint8_t* ipc_handle_out,
                     void** base_out) {
  if (!c || !max_local_queries) return fail(PIRB_INVALID_ARGUMENT, "bad argument");
  if (c->d < 2) return fail(PIRB_INVALID_ARGUMENT, "the peer-memory exchange serves databases of two or more dimensions");
  CU(cudaSetDevice(c->device));
  pirb_ctx::Dist& D = c->dist;
  if (D.base) return fail(PIRB_INVALID_ARGUMENT, "exchange block already created");
  if (!sub_batch && getenv("PIRB_DIST_SUB")) sub_batch = (u32)atoi(getenv("PIRB_DIST_SUB"));
  if (!sub_batch) {
    // default: sub-batches of two local queries, more while ranks x sub-batch < 8 (each multiply should see >= 8
    // queries): the exchange of one sub-batch hides behind the expansion of the next, so small sub-batches leave a
    // short exposed tail, while larger ones push longer contiguous rows (measured on 8 B200s: 2 beats 1 and 4)
    sub_batch = std::max<u32>(2, (8 + c->prm.shard_count - 1) / c->prm.shard_count);
    sub_batch = std::min<u32>(sub_batch, max_local_queries);
  }
  RC(dist_layout(c, max_local_queries, std::min(sub_batch, max_local_queries)));
  CU(cudaMalloc(&D.base, D.bytes));
  CU(cudaMemset(D.base, 0, D.flag_limbs * sizeof(u64)));
  int lo = 0, hi = 0;
  CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = numerically lowest = highest priority
  // transfer > expansion > multiply: the peers wait for what the transfer stream sends, and its narrow kernels must get
  // an SM slot as soon as any expansion CTA retires instead of queueing behind the whole level
  CU(cudaStreamCreateWithPriority(&D.xfer, cudaStreamNonBlocking, hi));
  CU(cudaStreamCreateWithPriority(&D.prod, cudaStreamNonBlocking, std::min(lo, hi + 1)));
  CU(cudaStreamCreateWithPriority(&D.cons, cudaStreamNonBlocking, lo));
  for (cudaEvent_t* e : {&D.ev_in, &D.ev_prod, &D.ev_xfer, &D.ev_done[0], &D.ev_done[1]})
    CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  D.ev_exp.resize(D.n_sub);
  for (auto& e : D.ev_exp) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto& e : D.prof) CU(cudaEventCreate(&e));
  for (auto& e : D.xprof) CU(cudaEventCreate(&e));
  if (const char* e = getenv("PIRB_DIST_TIMEOUT_MS")) D.timeout_ns = (u64)atoll(e) * 1000000ull;
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, D.base));
    memcpy(ipc_handle_out, &h, 64);
  }
  if (base_out) *base_out = D.base;
  return 0;
}

static int dist_finish_attach(pirb_ctx* c, const std::vector<u64*>& table) {
  pirb_ctx::Dist& D = c->dist;
  RC(D.peer_table.ensure(table.size() * sizeof(u64*)));
  CU(cudaMemcpy(D.peer_table.p, table.data(), table.size() * sizeof(u64*), cudaMemcpyHostToDevice));
  std::vector<u64*> self(table.size(), D.base);
  RC(D.self_table.ensure(self.size() * sizeof(u64*)));
  CU(cudaMemcpy(D.self_table.p, self.data(), self.size() * sizeof(u64*), cudaMemcpyHostToDevice));
  D.ready = true;
  return 0;
}

int pirb_dist_open_ipc(pirb_ctx* c, const uint8_t* handles, uint32_t n_ranks, uint32_t self_rank) {
  if (!c || !handles || !c->dist.base) return fail(PIRB_INVALID_ARGUMENT, "exchange block not created");
  if (n_ranks != c->prm.shard_count || self_rank != c->prm.shard_index)
    return fail(PIRB_INVALID_ARGUMENT, "ranks must match the context's shard index/count");
  CU(cudaSetDevice(c->device));
  std::vector<u64*> table(n_ranks);
  for (u32 r = 0; r < n_ranks; ++r) {
    if (r == self_rank) { table[r] = c->dist.base; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * 64, 64);
    void* pm = nullptr;
    CU(cudaIpcOpenMemHandle(&pm, h, cudaIpcMemLazyEnablePeerAccess));
    c->dist.opened.push_back(pm);
    table[r] = (u64*)pm;
  }
  c->dist.ipc = true;
  return dist_finish_attach(c, table);
}

int pirb_dist_attach(pirb_ctx* c, void* const* peer_bases, uint32_t n_ranks, uint32_t self_rank) {
  if (!c || !peer_bases || !c->dist.base) return fail(PIRB_INVALID_ARGUMENT, "exchange block not created");
  if (n_ranks != c->prm.shard_count || self_rank != c->prm.shard_index)
    return fail(PIRB_INVALID_ARGUMENT, "ranks must match the context's shard index/count");
  if (peer_bases[self_rank] != c->dist.base) return fail(PIRB_INVALID_ARGUMENT, "own entry must be this context's block");
  CU(cudaSetDevice(c->device));
  std::vector<u64*> table(n_ranks);
  for (u32 r = 0; r < n_ranks; ++r) {
    table[r] = (u64*)peer_bases[r];
    cudaPointerAttributes a;
    CU(cudaPointerGetAttributes(&a, peer_bases[r]));
    if (a.type != cudaMemoryTypeDevice) return fail(PIRB_INVALID_ARGUMENT, "peer block is not device memory");
    if (a.device != c->device) {  // same process, another GPU: direct peer access over NVLink
      int can = 0;
      CU(cudaDeviceCanAccessPeer(&can, c->device, a.device));
      if (!can) return fail(PIRB_INTERNAL, "no peer access between devices " + std::to_string(c->device) + " and " + std::to_string(a.device));
      cudaError_t e = cudaDeviceEnablePeerAccess(a.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU(e);
      cudaGetLastError();
    }
  }
  return dist_finish_attach(c, table);
}

// one step of the flow above; d_queries / d_replies are device-accessible (device memory or page-locked host memory)
// solo: the warm-up form of a step — the rank exchanges only with itself (every table entry is its own block) and the
// flags keep their value (sequence number 0 is always "arrived"), so it needs no peer to make progress: it loads every
// kernel of the flow and sets their attributes before the first real step.
static int dist_step(pirb_ctx* c, const pirb_keys* keys, const u64* d_queries, u32 n_local, u64 n_ct, u64* d_replies,
                     cudaStream_t user, bool solo = false) {
  pirb_ctx::Dist& D = c->dist;
  if (!D.ready) return fail(PIRB_INVALID_ARGUMENT, "exchange block not attached (pirb_dist_open_ipc / pirb_dist_attach)");
  if (!n_local || n_local > D.max_local) return fail(PIRB_INVALID_ARGUMENT, "local batch size out of range");
  if (n_ct != c->dim_sum / c->N + 1)
    return fail(PIRB_INVALID_ARGUMENT, "Number of ciphertexts doesn't match number of items for oblivious expansion.");
  if (c->loaded != c->pt_count) return fail(PIRB_INVALID_ARGUMENT, "database size mismatch");
  int rc;
  ExpandPlan* pl = get_plan(c, c->dim_sum, 0, &rc);
  if (!pl) return rc;
  const u32 W = D.n_ranks, SB = D.sub_q;
  if (!c->dry && D.sized_for < n_local) {
    // first step of this size: grow every workspace NOW (cudaMalloc synchronises the device, which must not happen
    // between a wait kernel and the launches of the peers it waits for when several ranks share one host thread)
    c->dry = true;
    const int rc_dry = dist_step(c, keys, d_queries, n_local, n_ct, d_replies, user);
    c->dry = false;
    if (rc_dry) return rc_dry;
    D.sized_for = n_local;
  }
  const bool dry = c->dry;
  const u64 seq = solo ? 0 : (dry ? D.step + 1 : ++D.step);
  const int slot = (int)((solo ? D.step + 1 : seq) & 1);
  const u32 n_sub = (n_local + SB - 1) / SB;
  const u64 q_stride = 2 * pl->cap * c->ctL;
  u64* const* peers = reinterpret_cast<u64* const*>(solo ? D.self_table.p : D.peer_table.p);
  u64* err = D.base;  // flag word 0
  c->launches = 0;
  const bool prof = c->profiling && !dry;

  // order: behind the caller's stream, behind the previous user of this slot, behind the last read of c->work
  if (!dry) CU(cudaEventRecord(D.ev_in, user));
  if (!dry) CU(cudaStreamWaitEvent(D.prod, D.ev_in, 0));
  if (!dry) CU(cudaStreamWaitEvent(D.cons, D.ev_in, 0));
  if (!dry && D.done_valid[slot]) CU(cudaStreamWaitEvent(D.prod, D.ev_done[slot], 0));
  if (!dry && D.xfer_valid) CU(cudaStreamWaitEvent(D.prod, D.ev_xfer, 0));
  if (prof) cudaEventRecord(D.prof[0], D.prod);

  // top levels for the whole local batch while they are too narrow to fill the GPU per sub-batch
  int split = 0;
  while (split < pl->max_logm && ((u64)SB * pl->n_trees << split) * 2 * (c->k + 1) < 2ull * c->sm_count) ++split;
  if (n_sub == 1) split = pl->max_logm;
  RC(run_expand(c, keys, pl, d_queries, (int)n_local, D.prod, 0, split, 0, (int)n_local));
  for (u32 sb = 0; sb < n_sub; ++sb) {
    const u32 q0 = sb * SB, qn = std::min(SB, n_local - q0);
    if (split < pl->max_logm) RC(run_expand(c, keys, pl, d_queries, (int)n_local, D.prod, split, pl->max_logm, (int)q0, (int)qn));
    if (!dry) CU(cudaEventRecord(D.ev_exp[sb], D.prod));
    if (!dry) CU(cudaStreamWaitEvent(D.xfer, D.ev_exp[sb], 0));
    PushArgs A;
    A.peers = peers;
    A.n_ranks = W;
    A.d0 = c->dims[0];
    A.rows_per_rank = D.rows_per_rank;
    A.slot_off = dist_sv_off(D, slot);
    A.g_first = ((u64)sb * W + D.rank) * SB;
    A.dst_qstride = D.sv_qstride;
    const u32 last = c->dims[c->d - 1], last_first = (u32)(c->dim_sum - last);
    const u64* sub_work = c->work.p + (u64)q0 * q_stride;
    const bool xp = prof && sb + 1 == n_sub;
    if (xp) cudaEventRecord(D.xprof[0], D.xfer);
    if (!D.tc_mode) {
      LAUNCH(c, launch_ntt_fwd_push(c->P, sub_work, q_stride, (u32)c->dim_sum, qn, A, D.xfer));
    } else {
      // one full-width NTT of the whole selection vector in place (database.cpp:190,222), then copy kernels narrow
      // enough to leave the SMs to the expansion: first / middle dimensions as u64 limbs to the owning rank / to everybody
      u64* sv_all = c->work.p + (u64)q0 * q_stride;
      u64* last_sv = sv_all + (u64)last_first * c->ctL;
      LAUNCH(c, launch_ntt_fwd(c->P, sv_all, sv_all, (int)(c->dim_sum * 2 * c->k), c->k, 0, (int)qn, q_stride, q_stride, D.xfer));
      if (xp) cudaEventRecord(D.xprof[1], D.xfer);
      LAUNCH(c, launch_push_head(c->P, sv_all, q_stride, last_first, qn, A, D.xfer));
      // last dimension: repacked ONCE here into the tensor-core scan's operand layout, then every coefficient's rows are
      // copied into every rank's svT region — no rank repacks another rank's queries
      if (xp) cudaEventRecord(D.xprof[2], D.xfer);
      const u32 stage_rows = SB * 2 * D.g.nb;
      RC(D.stage.ensure((size_t)c->k * c->N * stage_rows * D.g.Kp));
      LAUNCH(c, launch_tc_pack_sv(c->P, D.g, last_sv, q_stride, last, qn, reinterpret_cast<u8*>(D.stage.p), stage_rows, 0,
                                  D.xfer));
      if (xp) cudaEventRecord(D.xprof[3], D.xfer);
      const u64 row0 = (u64)D.rank * SB * 2 * D.g.nb;  // this rank's rows inside the sub-batch's region
      const u64 dst_off = (dist_sv_off(D, slot) + D.svt_off) * sizeof(u64) + sb * D.sub_bytes + row0 * D.g.Kp;
      LAUNCH(c, launch_push_rows(peers, W, reinterpret_cast<const u8*>(D.stage.p), (u64)stage_rows * D.g.Kp,
                                 qn * 2 * D.g.nb * D.g.Kp, (u32)c->k * c->N, dst_off, (u64)D.sub_rows * D.g.Kp, D.xfer));
      if (xp) cudaEventRecord(D.xprof[4], D.xfer);
    }
    LAUNCH(c, launch_signal(peers, W, dist_flag_off(D, 0, sb, D.rank), seq, D.xfer));
  }
  if (prof) cudaEventRecord(D.prof[1], D.prod);
  if (!dry) CU(cudaEventRecord(D.ev_xfer, D.xfer));
  if (!dry) D.xfer_valid = true;
  if (prof) cudaEventRecord(D.prof[2], D.xfer);

  // consumer: every sub-batch holds W * SB queries (rank-major), contiguous in the slot
  for (u32 sb = 0; sb < n_sub; ++sb) {
    const u32 qn = std::min(SB, n_local - sb * SB);
    LAUNCH(c, launch_wait(D.base + dist_flag_off(D, 0, sb, 0), W, seq, D.timeout_ns, err, D.cons));
    if (prof && sb == 0) cudaEventRecord(D.prof[3], D.cons);
    const u64 g0 = (u64)sb * W * SB;
    const u8* svt_base = reinterpret_cast<const u8*>(D.base + dist_sv_off(D, slot) + D.svt_off) + sb * D.sub_bytes;
    if (qn == SB) {
      SvtRef ref{svt_base, D.sub_rows, 0};
      RC(run_multiply(c, D.base + dist_sv_off(D, slot) + g0 * D.sv_qstride, D.sv_qstride, (int)(W * SB),
                      D.base + dist_part_off(D, slot) + g0 * c->reply_cts * c->ctL, 1, D.cons, true, 0, ~0ull,
                      D.rows_per_rank, D.tc_mode ? &ref : nullptr));
    } else {  // ragged last sub-batch: the ranks' queries are not contiguous, one multiply per rank
      for (u32 r = 0; r < W; ++r) {
        SvtRef ref{svt_base, D.sub_rows, (u32)(r * SB * 2 * D.g.nb)};
        RC(run_multiply(c, D.base + dist_sv_off(D, slot) + (g0 + (u64)r * SB) * D.sv_qstride, D.sv_qstride, (int)qn,
                        D.base + dist_part_off(D, slot) + (g0 + (u64)r * SB) * c->reply_cts * c->ctL, 1, D.cons, true, 0,
                        ~0ull, D.rows_per_rank, D.tc_mode ? &ref : nullptr));
      }
    }
    LAUNCH(c, launch_signal(peers, W, dist_flag_off(D, 1, sb, D.rank), seq, D.cons));
  }
  if (prof) cudaEventRecord(D.prof[4], D.cons);
  for (u32 sb = 0; sb < n_sub; ++sb) {
    const u32 q0 = sb * SB, qn = std::min(SB, n_local - q0);
    LAUNCH(c, launch_wait(D.base + dist_flag_off(D, 1, sb, 0), W, seq, D.timeout_ns, err, D.cons));
    const u64 cts = (u64)qn * c->reply_cts;
    RC(c->rbuf.ensure((size_t)D.max_local * c->reply_cts * c->ctL * sizeof(u64)));
    const u64 off = dist_part_off(D, slot) + (((u64)sb * W + D.rank) * SB) * c->reply_cts * c->ctL;
    LAUNCH(c, launch_modadd_reduce_ptrs(c->P, reinterpret_cast<const u64* const*>(peers), (int)W, off,
                                        c->rbuf.p + (u64)q0 * c->reply_cts * c->ctL, cts, D.cons));
    LAUNCH(c, launch_ntt_inv(c->P, c->rbuf.p + (u64)q0 * c->reply_cts * c->ctL, d_replies + (u64)q0 * c->reply_cts * c->ctL,
                             (int)(cts * 2 * c->k), c->k, 0, 1, 0, 1, 0, 0, D.cons));
  }
  if (prof) cudaEventRecord(D.prof[5], D.cons);
  if (!dry) D.prof_valid = prof;
  if (!dry) CU(cudaEventRecord(D.ev_done[slot], D.cons));
  if (!dry) D.done_valid[slot] = true;
  if (!dry) CU(cudaStreamWaitEvent(user, D.ev_done[slot], 0));
  if (!dry) CU(cudaStreamWaitEvent(user, D.ev_xfer, 0));
  if (!dry) D.launches = c->launches;
  return 0;
}

int pirb_dist_prepare(pirb_ctx* c, const pirb_keys* keys, uint32_t n_local) {
  if (!c || !keys) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  pirb_ctx::Dist& D = c->dist;
  if (!D.ready) return fail(PIRB_INVALID_ARGUMENT, "exchange block not attached");
  if (D.warmed_for >= n_local && D.sized_for >= n_local) return 0;
  const u64 n_ct = c->dim_sum / c->N + 1;
  // scratch queries (zeros are valid residues) and scratch replies
  RC(c->qbuf.ensure(std::max<size_t>((size_t)n_local * n_ct * c->ctL * sizeof(u64), 256)));
  RC(c->svbuf.ensure(std::max<size_t>((size_t)n_local * c->reply_cts * c->ctL * sizeof(u64), 256)));
  CU(cudaMemsetAsync(c->qbuf.p, 0, (size_t)n_local * n_ct * c->ctL * sizeof(u64), c->stream));
  RC(dist_step(c, keys, c->qbuf.p, n_local, n_ct, c->svbuf.p, c->stream, true));
  CU(cudaStreamSynchronize(c->stream));
  D.warmed_for = n_local;
  return pirb_dist_status(c);
}

int pirb_dist_answer_dev(pirb_ctx* c, const pirb_keys* keys, const uint64_t* d_queries, uint32_t n_local, uint64_t n_ct,
                         uint64_t* d_replies, void* stream) {
  if (!c || !d_queries || !d_replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  DevCallOrder order(c, st);
  return dist_step(c, keys, U(d_queries), n_local, n_ct, U(d_replies), st);
}

int pirb_dist_answer(pirb_ctx* c, const pirb_keys* keys, const uint64_t* queries, uint32_t n_local, uint64_t n_ct,
                     uint64_t* replies) {
  if (!c || !queries || !replies) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  const size_t qbytes = (size_t)n_local * n_ct * c->ctL * sizeof(u64);
  const size_t rbytes = (size_t)n_local * c->reply_cts * c->ctL * sizeof(u64);
  // page-locked buffers are read / written in place by the first / last kernels, pageable ones are staged
  const bool q_direct = host_buffer_is_device_accessible(queries);
  const bool r_direct = host_buffer_is_device_accessible(replies);
  DevCallOrder order(c, st);
  if (!q_direct) {
    RC(c->qbuf.ensure(std::max<size_t>(qbytes, 256)));
    CU(cudaMemcpyAsync(c->qbuf.p, queries, qbytes, cudaMemcpyHostToDevice, st));
  }
  if (!r_direct) RC(c->svbuf.ensure(std::max<size_t>(rbytes, 256)));
  RC(dist_step(c, keys, q_direct ? U(queries) : c->qbuf.p, n_local, n_ct, r_direct ? U(replies) : c->svbuf.p, st));
  if (!r_direct) CU(cudaMemcpyAsync(replies, c->svbuf.p, rbytes, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return pirb_dist_status(c);
}

int pirb_dist_status(pirb_ctx* c) {
  if (!c || !c->dist.base) return fail(PIRB_INVALID_ARGUMENT, "exchange block not created");
  CU(cudaSetDevice(c->device));
  u64 e = 0;
  CU(cudaMemcpy(&e, c->dist.base, sizeof(u64), cudaMemcpyDeviceToHost));
  if (e) return fail(PIRB_INTERNAL, "peer exchange timed out waiting for a rank's flag at step " + std::to_string(e));
  return 0;
}

// stage: 0 expansion (producer stream), 1 tail of the exchange after the expansion, 2 wait for the first sub-batch of
// all ranks, 3 multiplies, 4 partial-reply reduce + inverse NTT, 5 whole step
int pirb_dist_stage_ms(pirb_ctx* c, float* out) {
  if (!c || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  pirb_ctx::Dist& D = c->dist;
  if (!D.prof_valid) return fail(PIRB_INVALID_ARGUMENT, "no profiled distributed step recorded");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(D.prof[5]));
  CU(cudaEventSynchronize(D.prof[2]));
  CU(cudaEventElapsedTime(out + 0, D.prof[0], D.prof[1]));
  CU(cudaEventElapsedTime(out + 1, D.prof[1], D.prof[2]));
  CU(cudaEventElapsedTime(out + 2, D.prof[0], D.prof[3]));
  CU(cudaEventElapsedTime(out + 3, D.prof[3], D.prof[4]));
  CU(cudaEventElapsedTime(out + 4, D.prof[4], D.prof[5]));
  CU(cudaEventElapsedTime(out + 5, D.prof[0], D.prof[5]));
  for (int i = 0; i < 4; ++i) {
    out[6 + i] = 0.f;
    if (D.tc_mode && cudaEventElapsedTime(out + 6 + i, D.xprof[i], D.xprof[i + 1]) != cudaSuccess) cudaGetLastError();
  }
  return 0;
}

int pirb_scan_dev(pirb_ctx* c, const uint64_t* d_sv_ntt, uint32_t n_queries, uint64_t* d_rows, void* stream) {
  if (!c || !d_sv_ntt) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
  if (!c->pt_count) return 0;
  const u32 dimL = c->d == 1 ? (c->top_hi - c->top_lo) : c->dims[c->d - 1];
  const u32 n_rows = c->d == 1 ? 1 : (u32)((c->pt_count + dimL - 1) / dimL);
  DevCallOrder order(c, st);
  if (c->profiling) cudaEventRecord(c->ev[2], st);
  int n_split;
  c->launches = 0;
  RC(run_scan(c, U(d_sv_ntt), (u64)dimL * c->ctL, (int)n_queries, dimL, n_rows, c->pt_count, c->d >= 2, &n_split, st));
  if (c->profiling) cudaEventRecord(c->ev[3], st);
  if (d_rows && n_split == 1)
    CU(cudaMemcpyAsync(d_rows, c->part.p, (size_t)n_queries * n_rows * c->ctL * sizeof(u64), cudaMemcpyDeviceToDevice, st));
  if (d_rows && n_split != 1) {
    LAUNCH(c, launch_modadd_reduce(c->P, c->part.p, (u64)n_rows * c->ctL, n_split, U(d_rows), n_rows, st, (int)n_queries,
                                   (u64)n_split * n_rows * c->ctL, (u64)n_rows * c->ctL));
  }
  return 0;
}

int pirb_debug_stamps(pirb_ctx* c, uint64_t* out, uint64_t n) {
  if (!c || !out || !c->dbg.p) return fail(PIRB_INVALID_ARGUMENT, "debug stamps are off (PIRB_DEBUG_STAMPS)");
  CU(cudaSetDevice(c->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(out, c->dbg.p, std::min<size_t>(n * sizeof(u64), 8 << 20), cudaMemcpyDeviceToHost));
  return 0;
}
int pirb_sync(pirb_ctx* c) {
  if (!c) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream));
  if (c->tc.err && *c->tc.err) return fail(PIRB_INTERNAL, "tensor-core scan: pipeline timed out");
  return 0;
}

int pirb_set_profiling(pirb_ctx* c, int enabled) {
  if (!c) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  c->profiling = enabled != 0;
  c->ev_valid = false;
  return 0;
}
int pirb_get_stage_ms(pirb_ctx* c, float* out) {
  if (!c || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  if (!c->ev_valid) return fail(PIRB_INVALID_ARGUMENT, "no profiled call recorded");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ev[5]));
  for (int i = 0; i < 5; ++i) CU(cudaEventElapsedTime(out + i, c->ev[i], c->ev[i + 1]));
  CU(cudaEventElapsedTime(out + 5, c->ev[0], c->ev[5]));
  return 0;
}
int pirb_last_scan_ms(pirb_ctx* c, float* out) {
  if (!c || !out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  if (!c->profiling) return fail(PIRB_INVALID_ARGUMENT, "profiling is off");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ev[3]));
  CU(cudaEventElapsedTime(out, c->ev[2], c->ev[3]));
  return 0;
}
uint64_t pirb_last_launch_count(const pirb_ctx* c) { return c ? c->launches : 0; }
uint64_t pirb_scan_bytes(const pirb_ctx* c, uint32_t n_queries) {
  // SURVEY §8d: DB read once + last-dimension selection cts read once + row results written once
  if (!c || !c->pt_count) return 0;
  const u32 dimL = c->d == 1 ? (c->top_hi - c->top_lo) : c->dims[c->d - 1];
  const u64 n_rows = c->d == 1 ? 1 : (c->pt_count + dimL - 1) / dimL;
  return (c->pt_count * c->ptL + (u64)n_queries * dimL * c->ctL + (u64)n_queries * n_rows * c->ctL) * sizeof(u64);
}

int pirb_host_alloc(uint64_t bytes, void** out) {
  if (!out) return fail(PIRB_INVALID_ARGUMENT, "null argument");
  *out = nullptr;
  CU(cudaHostAlloc(out, std::max<uint64_t>(bytes, 16), cudaHostAllocPortable | cudaHostAllocMapped));
  return 0;
}
void pirb_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

void pirb_calculate_dimensions(uint32_t db_size, uint32_t nd, uint32_t* out) {
  auto v = hm::calculate_dimensions(db_size, nd);
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
}
uint64_t pirb_next_power_two(uint64_t v) { return hm::next_power_two(v); }
uint32_t pirb_ceil_log2(uint32_t v) { return hm::ceil_log2(v); }
uint32_t pirb_log2(uint32_t v) { return hm::trunc_log2(v); }
uint64_t pirb_plain_modulus_batching(uint32_t N, uint32_t bits) {
  if (bits < 2 || bits > 60) return 0;
  const u64 factor = 2ull * N;
  u64 value = (1ull << bits) - factor + 1;
  const u64 lower = 1ull << (bits - 1);
  while (value > lower) {
    if (hm::is_prime(value)) return value;
    value -= factor;
  }
  return 0;
}
int pirb_bfv_default_coeff_modulus(uint32_t N, uint64_t* out, uint32_t cap) {
  // SEAL CoeffModulus::BFVDefault (128-bit security) tables for the degrees this library supports
  static const u64 m4096[] = {0xffffee001ULL, 0xffffc4001ULL, 0x1ffffe0001ULL};
  static const u64 m8192[] = {0x7fffffd8001ULL, 0x7fffffc8001ULL, 0xfffffffc001ULL, 0xffffff6c001ULL, 0xfffffebc001ULL};
  static const u64 m16384[] = {0xfffffffd8001ULL, 0xfffffffa0001ULL, 0xfffffff00001ULL, 0x1fffffff68001ULL,
                               0x1fffffff50001ULL, 0x1ffffffee8001ULL, 0x1ffffffea0001ULL, 0x1ffffffe88001ULL,
                               0x1ffffffe48001ULL};
  const u64* src;
  u32 n;
  switch (N) {
    case 4096: src = m4096; n = 3; break;
    case 8192: src = m8192; n = 5; break;
    case 16384: src = m16384; n = 9; break;
    default: return -1;
  }
  if (n > cap) return -1;
  for (u32 i = 0; i < n; ++i) out[i] = src[i];
  return (int)n;
}

}  // extern "C"
