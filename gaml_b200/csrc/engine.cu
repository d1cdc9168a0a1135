// Host engine + C ABI (include/gaml_b200.h) of the B200 GAML likelihood path.
//
// Host side responsibilities, all O(#nodes in the touched walks), never O(records):
//   * mirror of aligment_cache_ (graph.h:427, 587): key -> id map, per-key arena range / max position;
//   * GetChanges (graph.cc:1745-1764) on the same container + hash as the reference so erased walks
//     come out in the same order;
//   * flattening of walks into per-key occurrence tables following the reference's three lookup
//     rules (graph.cc:547-597, 613-646, 2438-2500) — see flatten_*();
//   * host-computed constant tables (pow tables graph.cc:1448-1453, insert pdf graph.cc:1593-1598,
//     floor thresholds graph.cc:1506-1507/1528) so that those values are bit-identical to the
//     reference's on the same host.
// Everything that touches an alignment record runs in kernels.cu.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <limits>
#include <cmath>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <memory>
#include <memory_resource>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../include/gaml_b200.h"
#include "kernels.h"
#include "walk_set.h"

namespace gaml {
namespace {

constexpr int kWindowLen = 300;   // kMinSubpathLength, graph.cc:27

// graph.h:21-45: the reference's hash for vector<int> (walk_set.h: hash_nodes)
struct WalkHash {
  size_t operator()(const Walk& v) const { return hash_nodes(v.data(), (int)v.size()); }
};

inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
  __builtin_ia32_pause();
#elif defined(__aarch64__)
  asm volatile("yield");
#endif
}

thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  ~DevBuf() { if (p) cudaFree(p); }
  // grows (contents preserved when keep > 0); new space zeroed when zero_new
  cudaError_t reserve(size_t bytes, size_t keep, bool zero_new, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    size_t ncap = std::max(bytes, cap + cap / 2);
    ncap = (ncap + 255) & ~size_t(255);
    void* np = nullptr;
    cudaError_t e = cudaMalloc(&np, ncap);
    if (e != cudaSuccess) return e;
    if (zero_new) {
      e = cudaMemsetAsync(np, 0, ncap, st);
      if (e != cudaSuccess) return e;
    }
    if (p && keep) {
      e = cudaMemcpyAsync(np, p, keep, cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) return e;
    }
    if (p) {
      cudaStreamSynchronize(st);
      cudaFree(p);
    }
    p = np;
    cap = ncap;
    return cudaSuccess;
  }
  template <class T> T* as() const { return static_cast<T*>(p); }
};

struct KeyMeta {
  uint32_t arena_off = 0;   // into the store's arena (shard-local records)
  uint32_t count = 0;       // shard-local records
  int32_t max_pos = 0;      // over ALL reads' records
  bool any = false;         // the key has at least one record (any read)
};

// Walk-relative lookups of one walk in one paired set (build_walk_flat) and their cache.
struct FlatEntry { int32_t key, cur, skip; uint32_t count, arena_off; };
struct WalkFlat {
  std::vector<FlatEntry> e[2];
  std::vector<int> contig_starts;
  int64_t records = 0, records1 = 0;
  // validity across cache growth: keys are immutable once inserted, so a walk's lookups change only when a window that
  // was NOT in the cache when they were built is inserted later — gen = the store's key count at build time, missing =
  // the hashes of the windows that were looked up and not found
  size_t gen[2] = {0, 0};
  std::vector<size_t> missing[2];
};
struct FlatCache {   // chained hash table keyed by walk content; the caller supplies the (already computed) hash
  struct Node { size_t h; Walk w; WalkFlat f; int next; };
  std::vector<Node> nodes;
  std::vector<int> buckets;
  void clear() { nodes.clear(); buckets.clear(); }
  WalkFlat* find(const int* p, int n, size_t h) {
    if (buckets.empty()) return nullptr;
    for (int i = buckets[h & (buckets.size() - 1)]; i >= 0; i = nodes[i].next)
      if (nodes[i].h == h && (int)nodes[i].w.size() == n && (n == 0 || memcmp(nodes[i].w.data(), p, sizeof(int) * (size_t)n) == 0))
        return &nodes[i].f;
    return nullptr;
  }
  WalkFlat& insert(const Walk& w, size_t h) {
    if (nodes.size() >= buckets.size()) {
      buckets.assign(std::max<size_t>(1024, buckets.size() * 2), -1);
      for (size_t i = 0; i < nodes.size(); i++) {
        int& b = buckets[nodes[i].h & (buckets.size() - 1)];
        nodes[i].next = b;
        b = (int)i;
      }
    }
    int& b = buckets[h & (buckets.size() - 1)];
    nodes.push_back(Node{h, w, WalkFlat(), b});
    b = (int)nodes.size() - 1;
    return nodes.back().f;
  }
};

// Per-store accumulation of the occurrences of one evaluation.
struct OccBuilder {
  std::vector<std::pair<int, Occ>> items;   // (key id, occurrence) in enumeration order
  uint32_t next_seg = 0;                    // (the kernels order placements by seg as an unsigned number)
  void reset() { items.clear(); next_seg = 0; }
  void add(int key, int walk, int cur_pos, int skip_below) {
    items.push_back({key, Occ{walk, (int)next_seg++, cur_pos, skip_below}});
  }
};

struct MateStore {
  bool is_long = false;
  std::unordered_map<Walk, int, WalkHash> key_ids;
  std::vector<KeyMeta> keys;
  std::vector<int4> pending;          // staged arena records (ArenaShort / ArenaLong bit patterns)
  std::vector<Int2> pending_pos;      // long stores: {position, position_end} of the staged records (coverage penalty)
  DevBuf arena_pos;                   // long stores: Int2 per arena record
  size_t arena_n = 0;                 // records on the device
  DevBuf arena, rows, first, rowptr, cursor, slots_a, slots_b, crows, cptr;
  bool dirty = true;
  std::vector<double> pow_match, pow_mismatch;
  DevBuf d_pow_match, d_pow_mismatch;
  int table_index = -1;               // position in ctx->d_tables
  std::vector<uint32_t> key_stamp;    // group_occurrences scratch: epoch that last saw the key / its SlotUpdate index
  std::vector<int> key_slot, fill_cursor;
  std::vector<int> base_slot;         // patched full evaluations: the key's SlotUpdate index in the resident base blob, -1 = none
  // cache append (kernels.cu "cache append"): the row array has slack behind the rows of the last full build, rows_tail is
  // the next free row; h_count = every read's record count (internal read index), kept in step by the host
  size_t rows_cap = 0, rows_tail = 0;
  std::vector<uint16_t> h_count;
  std::vector<size_t> key_hash_log;   // hash of every key, in insertion order (WalkFlat validation)
  std::vector<const Walk*> key_by_id; // the key's node sequence (points into key_ids: stable)
  size_t built_keys = 0;              // keys the device tables / key maps know about
  size_t total_records() const { return arena_n + pending.size(); }
};

struct ReadSetState {
  gaml_readset_config cfg{};
  int64_t n_total = 0, lo = 0, hi = 0;
  int n_local = 0;
  int n_mates = 1;
  int max_len[2] = {0, 0};
  std::vector<int32_t> len[2];
  MateStore mate[2];
  DevBuf d_lens, d_values, d_stamp, d_ins, d_ovf_list, d_complex, d_clens, d_cdesc;
  DevBuf d_pairs;               // paired: PackedPair per pair (kernels.cu), valid when pairs_ok
  DevBuf d_uni_prob[2];           // paired, uniform lengths: alignment probability by edit distance, per mate (kernels.cu)
  // internal read order (kernels.cu "internal read order"): fixed at the first commit of a set with fast records
  // cache append: reads that gained records since the last full build are flagged (device) and listed for the appendix
  // phase; base_built = the static lists exist and appends may be applied on top of them
  bool base_built = false;
  DevBuf d_dirty, d_appx, d_append_blob;
  std::vector<uint8_t> h_dirty;
  int n_appx = 0;
  std::vector<int32_t> h_p12, h_p21;   // key maps between the mates' stores (same node sequence), -1 = no partner
  int64_t appends = 0, rebuilds = 0;
  bool perm_valid = false;
  std::vector<uint32_t> h_inv;    // caller's local read id -> internal index (cache inserts, gaml_read_values)
  std::vector<uint32_t> h_perm;   // internal index -> caller's local read id (gaml_cache_save)
  int n_fast = 0;                 // reads [0, n_fast) of the internal order are tier 1's
  DevBuf d_fast, d_xlist;         // with a term table: FastPair per pair + the cross list (kernels.cu), valid when fast_ok
  bool fast_ok = false;
  int n_cross = 0;
  DevBuf d_tq;                    // paired, uniform lengths: term table (pair term + its fixed-point logarithm), kernels.cu
  int tq_shift = 0;               //   edit distances below 1 << tq_shift are tabulated (0 = no table)
  // the per-read log term (kernels.cu acc_term): thresholds exp(mps + mppb*len) by length index (paired: len1 + len2), the
  // fixed-point log of each (device table), the length indices that occur, and the floor test of the last total length
  std::vector<double> h_thr;
  std::vector<long long> h_qthr;
  std::vector<int> len_classes;
  std::vector<double> h_pstar;
  int pstar_two_len = 0;
  bool pstar_valid = false;
  DevBuf d_qthr;
  DevBuf d_comb, d_partner12, d_partner21;   // paired: combined first slot words by mate-1 key id + the key maps (kernels.cu)
  bool comb_ok = false;
  DevBuf d_t2pack;              // paired: packed tier-2 entries (kernels.cu), valid when t2pack_ok
  bool t2pack_ok = false;
  uint32_t t2base[3] = {0, 0, 0};
  bool pairs_ok = false;
  bool lens_uniform = false;    // every pair of the set has the same packed lengths
  uint32_t uniform_ll = 0;
  int32_t class_begin[17] = {0};
  uint32_t cbase[2][5] = {{0}};  // first compact row of the five tier-2 classes, per mate
  int n_complex = 0;
  bool complex_dirty = true;
  int ins_n = 0;
  double floor_a = 0, floor_b = 0;
  // ScoringState (graph.h:612-619): probs live in d_values, old_paths here
  // running total of the per-read log terms, kept exactly on the device (finish_set): valid for two_len == total_two_len
  DevBuf d_state_acc;
  bool total_valid = false;
  int total_two_len = 0;
  bool has_state = false;       // old_paths = the context's last evaluated walk set (gaml_ctx::prev)
  FlatCache flat_cache;         // per distinct walk: its lookups in this set (cleared when the set's cache grows)
  int bad_bases = 0;            // ScoringState::bad_bases (graph.h:614)
  bool penalty = false;         // paired set with penalty_constant != 0: coverage events are collected
  // a penalised set on a read-id shard: a walk's coverage events live on all shards, so an evaluation leaves this
  // shard's events on the device (no sweep), the caller gathers every shard's (gaml_penalty_export), hands the union
  // back (gaml_penalty_import: sort + sweep + bad_bases bookkeeping) and only then combines the partials
  bool sharded = false;
  bool penalty_pending = false;
  std::vector<unsigned long long> h_type1;   // the host's contig-start events of the pending evaluation (paired)
  DevBuf d_cov_thr, d_ev, d_ev_sorted, d_ev_temp, d_bad;
  // PacBio coverage penalty (graph.cc:3197-3250)
  bool pb_penalty = false;
  DevBuf d_pb_ikey, d_pb_iend, d_pb_pkey, d_pb_packed, d_pb_runmax, d_pb_temp, d_pb_count;
  std::vector<int4> h_pb_seeds, h_pb_occ;
  std::vector<uint32_t> h_pb_prefix;
  std::vector<int> h_pb_walk_len;
  std::vector<int> h_bad;
  // paired full evaluations replayed as a graph end with the streaming kernel unless the set's previous full evaluation
  // listed reads for the many-placement pass (keep_tail). Without the pass in the chain, a pending line makes finish()
  // run it on demand with the parameters kept here.
  bool keep_tail = false;
  bool tail_on_demand = false;  // the pending evaluation's chain has no many-placement pass
  ScoreParams tail_params{};
  int tail_grid = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // around this set's streaming kernel(s)
  ~ReadSetState() {
    for (cudaEvent_t e : {ev0, ev1})
      if (e) cudaEventDestroy(e);
  }
};

struct SetPlan {
  bool full = true;
  bool delta_only = false;      // incremental evaluation at the running total's length: no O(R) pass
  int n_erased = 0;
  int total_len = 0;
  int64_t records = 0;          // A: live (record, occurrence) pairs in this shard
  int64_t touch_records = 0;
  int64_t records1 = 0;         // live mate-1 records (bounds the number of pair terms for the coverage events)
  // coverage-gap penalty (paired sets with penalty_constant != 0)
  int n_cov_walks = 0, n_type1 = 0;
  uint32_t ev_cap = 0;
  size_t type1_off = 0, csbegin_off = 0, cs_off = 0, evcount_off = 0;
  int grid = 0;                 // blocks of the reducing kernel
  int cgrid = 0;                // blocks of the tier-2 (several records per read) kernel
  size_t occ_off[2] = {0, 0};   // byte offsets inside the staging blob
  size_t touch_off = 0, prefix_off = 0;
  size_t pstar_off = 0;         // floor tests of this evaluation's total length, by length index (short-read sets)
  int n_touch = 0;
  // full paired evaluations: arena ranges of the keys that occur several times (the multi pass)
  size_t pb_seeds_off = 0, pb_occ_off = 0, pb_prefix_off = 0, pb_len_off = 0;   // PacBio coverage penalty inputs
  uint32_t pb_cap = 0;
  size_t mtouch_off = 0, mprefix_off = 0;
  int n_mtouch = 0, n_mtouch1 = 0;
  int64_t multi_records = 0;
};

}  // namespace
}  // namespace gaml

using namespace gaml;

struct gaml_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool timed = false;             // gaml_set_profiling >= 1: events around the whole evaluation (gaml_stats.last_device_ms)
  bool profile = false;           // gaml_set_profiling 2: + per-set events around the streaming kernels (direct launches)
  bool timeline = false;          // gaml_set_profiling 3: device-side globaltimer stamps per kernel instead (no events)
  DevBuf d_timeline;
  unsigned long long h_timeline[kTimelineWords] = {0};
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  std::string error;
  std::vector<int32_t> node_len, nmap;
  std::vector<std::unique_ptr<ReadSetState>> sets;
  std::vector<MateStore*> stores;
  StoreTables h_tables{};         // the same pointers by value, valid when stores.size() <= kInlineStores
  DevBuf d_tables;                // SlotA* per store, then SlotB* per store
  bool tables_dirty = true;
  DevBuf d_blob;                  // per-evaluation staging (updates, occurrences, touch ranges, set_begin)
  // A FULL evaluation's staging blob is a function of the walk list and the cache alone (the epoch is a kernel parameter).
  // It is kept on the device in its own buffer: a full re-score of the walk list that was evaluated last — a fresh
  // ScoringState over unchanged walks, gaml_reset_state — needs no flattening and no upload at all.
  DevBuf d_full_blob;
  char* blob_dev = nullptr;       // the blob of the pending evaluation (d_blob or d_full_blob)
  bool full_blob_valid = false;
  uint64_t list_gen = 0, cache_gen = 0, full_list_gen = 0, full_cache_gen = 0;
  std::vector<SetPlan> full_plan;
  int full_n_updates = 0;
  size_t full_upd_off = 0, full_blob_bytes = 0;
  int64_t full_blob_reuses = 0;
  // Patched full evaluation: a full re-score of a walk list a few walks away from the BASE list (the one the resident
  // blob was built for) uploads only the slot updates of the keys those walks look up. Walks carry order-preserving labels
  // with gaps ((base index + 1) << base_g; a walk that is not in the base list gets a label between its neighbours'), and
  // a lookup's enumeration number is label << base_s | index inside the walk, so patched lists keep the reference's
  // placement order without renumbering the resident entries. track[i] follows wsets[i].
  gaml::ListTrack track[2];          // labels of wsets[i] (walk_set.h)
  bool patch_enabled = true;       // GAML_B200_NO_FULL_PATCH=1: every full evaluation of a changed list flattens all walks (tests)
  bool base_valid = false;
  uint64_t base_gen = 0;
  int base_g = 3, base_s = 0;
  WalkSet base_ws;                 // nodes / offs / hash of the base list
  std::vector<SlotUpdate> full_updates;
  std::vector<std::vector<Occ>> full_occs;
  std::vector<std::vector<std::pair<int, int>>> base_mkeys;   // per set: (mate, key) of the base's keys with several occurrences
  size_t patch_upd_off = 0, patch_skip_off = 0;               // the pending evaluation's patch inside d_full_blob
  int n_patch = 0, n_skip = 0;
  void* h_blob = nullptr;         // pinned
  size_t h_blob_cap = 0;
  DevBuf d_flags, d_scratch, d_csr_temp, d_logtab;
  DevBuf d_batch_blob, d_batch_acc, d_batch_out;   // gaml_calc_prob_batch
  DevBuf d_aln[8];                                  // gaml_pacbio_alignment_logprob
  std::vector<double> h_batch_out;
  void* h_append_pinned = nullptr;                  // pinned staging of a cache append (arena records, rows, groups, lists, key-map patches)
  size_t h_append_cap = 0;
  cudaEvent_t ev_append = nullptr;                  // recorded behind the append's copy: the staging is reused only after it
  bool append_copy_pending = false;
  double* h_out = nullptr;        // pinned + mapped: kResultStride doubles per set, written by the last kernel of each set
  double* d_out_mapped = nullptr; // device-side address of h_out
  std::vector<double> h_res;      // validated copy of h_out taken by finish()
  // result exchange between the ranks of a multi-GPU job (gaml_set_result_exchange): a host shared-memory segment
  // mapped into every rank's GPU; each rank's publishing block writes its 64-byte line there, every host reads all
  double* exch_host = nullptr;
  double* exch_dev = nullptr;
  int exch_rank = 0, exch_world = 1;
  bool exch_owned = false;        // this context registered the segment with CUDA (and unregisters it)
  // (b) peer memory over NVLink (gaml_peer_exchange_*): every rank owns a small device buffer of result lines
  // [2 generations][world][GAML_EXCHANGE_MAX_SETS][64 B]; the publishing block of an evaluation stores its line into the
  // buffer of EVERY rank (peer_ptrs, IPC-mapped), and the chain's last kernel (exchange_gather_kernel) waits for all lines
  // in its own buffer and hands them to the host in one piece (h_gather: world x n_sets lines + one flag line)
  DevBuf d_peer_lines, d_peer_table;
  std::vector<void*> peer_ptrs;
  std::vector<char> peer_opened;  // entries of peer_ptrs that came from cudaIpcOpenMemHandle
  int peer_rank = 0, peer_world = 0;
  bool peer_on = false;
  unsigned long long* h_gather = nullptr;   // pinned + mapped
  unsigned long long* d_gather_mapped = nullptr;
  // (c) a collective library (gaml_nccl_exchange_init): all-reduce of the ranks' lines on the evaluation's stream
  void* nccl_lib = nullptr;
  void* nccl_comm = nullptr;
  int nccl_rank = 0, nccl_world = 0;
  bool nccl_on = false;
  DevBuf d_part, d_part_sum;
  unsigned long long exchange_timeout_ns = 20ull * 1000 * 1000 * 1000;   // a peer's line missing for this long fails the evaluation
  // CUDA graphs of the evaluations' kernel chains, keyed by the sequence of kernels (GAML_B200_NO_GRAPHS=1 disables)
  struct GraphEntry { cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr; std::vector<cudaGraphNode_t> nodes; };
  std::unordered_map<uint64_t, GraphEntry> graphs;
  bool use_graphs = true;
  bool running_total = true;      // GAML_B200_NO_RUNNING_TOTAL=1 forces the O(R) pass on every incremental evaluation (tests)
  bool timing_pending = false;    // events of the last evaluation not yet turned into gaml_stats times
  bool tail_timed = false;        // finish() ran many-placement passes on demand between ev[1] and ev[2] (timed)
  size_t h_out_cap = 0;
  unsigned long long scratch_entries = 1ull << 22;   // 4 Mi placements (96 MiB) for many-placement reads
  uint32_t ovf_cap = 1u << 20;
  uint32_t epoch = 0;             // device epoch: advanced by every successfully prepared evaluation
  uint32_t stamp_gen = 0;         // host generation of the stores' key_stamp tables: advanced by every prepare()
  bool capacity_grew = false;     // the last evaluation failed for capacity and the buffers it overran have been enlarged
  // pending evaluation
  bool prepared = false, launched = false;
  std::vector<SetPlan> plan;
  // walk sets: cur = the evaluation being prepared, prev = the last FINISHED evaluation (ScoringState::old_paths of
  // every paired set that has state, graph.cc:1986); ping-pong so that steady-state evaluations allocate nothing
  WalkSet wsets[2];
  int cur_set = 0;
  WalkSet& cur() { return wsets[cur_set]; }
  WalkSet& prev() { return wsets[cur_set ^ 1]; }
  // per-evaluation host staging, reused
  std::vector<SlotUpdate> h_updates;
  std::vector<std::vector<Occ>> h_occs;
  std::vector<std::vector<TouchRange>> h_touches, h_mtouches;
  std::vector<OccBuilder> h_ob;   // one per store
  std::vector<WalkView> h_refs;
  std::vector<Walk> h_walks;
  bool fast_changes = true;       // GAML_B200_NO_FAST_CHANGES=1: always build the reference's container (tests)
  bool permute_reads = true;      // GAML_B200_NO_PERMUTE=1: keep the caller's read order on the device (tests, measurements)
  bool append_enabled = true;     // GAML_B200_NO_APPEND=1: every cache growth rebuilds the device index (tests, measurements)
  HashCounts prev_counts;         // multiplicity of every walk hash in prev() (kept in step by finish())
  bool have_prev = false;         // prev() holds a finished evaluation's walks
  WalkDiff cur_diff;              // cur() against prev(), from prepare()
  int prev_total_len = 0, cur_total_len = 0;
  Changes h_changes;
  alignas(16) char pool_buf[1 << 18];   // nodes + buckets of the GetChanges multiset (bump-allocated, released per use;
  std::pmr::monotonic_buffer_resource pool{pool_buf, sizeof(pool_buf)};   // larger walk sets spill to the heap)
  int n_updates = 0;
  size_t upd_off = 0, blob_bytes = 0;
  gaml_stats stats{};
};

namespace gaml {
namespace {

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      ctx->error = std::string(#call) + ": " + cudaGetErrorString(e__);                            \
      return GAML_ERR_CUDA;                                                                        \
    }                                                                                              \
  } while (0)

int fail(gaml_ctx* ctx, int code, const std::string& msg) {
  ctx->error = msg;
  return code;
}

// d_flags layout (u64 words, zeroed at the start of every evaluation): [0] scratch cursor | [1] error flag (u32) |
// [2, 2+n) per-set overflow counters (u32 in u64 slots) | [2+n, 2+2n) tickets of the last streaming kernel |
// [2+2n, 2+3n) tickets of the last kernel | [2+3n, 2+4n) "published early" marks | [2+4n, 2+8n) tile counters (eight
// u32 per set: tier 1, rare shapes, tier 2, cross list, appendix) | then per set kAccumStride words of exact accumulators
size_t flags_words(size_t n_sets) { return 2 + std::max<size_t>(n_sets, 1) * (8 + kAccumStride); }

double insert_pdf(double d, double mean, double sd) {   // graph.cc:1593-1598, same expression order
  double z = (d - mean) / sd;
  double e = exp(-z * z / 2.0);
  double c = sqrt(2 * M_PI) * sd;
  return e / c;
}

// The floor test of GetTotalProb (graph.cc:1505-1512, 1527-1532) as a test on the read's value itself: the smallest
// double p whose IEEE quotient p / d (d = 2 * total_len) is not below thr. RN(p / d) is monotone in p, so
// "RN(p / d) < thr" is exactly "p < floor_pstar(thr, d)".
double floor_pstar(double thr, double d) {
  if (!(thr > 0.0)) return 0.0;   // nothing is below a zero threshold
  double p = thr * d;
  while (p > 0.0 && p / d >= thr) p = std::nextafter(p, 0.0);
  while (p / d < thr) p = std::nextafter(p, std::numeric_limits<double>::infinity());
  return p;
}

constexpr double kFixScaleHost = 1099511627776.0;   // 2^40 (kernels.cu kFixScale)
long long fix_log_host(double v) {                   // FIX(log v) for the host-side constants of the term (thr, 2L)
  if (!(v > 0.0)) return 0;
  return std::llrint(std::log(v) * kFixScaleHost);
}

int two_len_of(int total_len) {   // the reference's int expression 2*total_len with total_len == 0 -> 1 (graph.cc:1500-1505)
  const int tl = total_len == 0 ? 1 : total_len;
  return (int)(2u * (unsigned)tl);
}

// ---- walk helpers -------------------------------------------------------------------------
int walk_length(const gaml_ctx* ctx, const Walk& w) {   // graph.cc:1766-1773
  int t = 0;
  for (int x : w) t += x < 0 ? -x : ctx->node_len[x];
  return t;
}

void split_at_gaps(const Walk& w, std::vector<Walk>& ctgs, std::vector<int>& gaps) {   // graph.cc:1813-1824
  ctgs.assign(1, Walk());
  gaps.clear();
  for (int x : w) {
    if (x < 0) {
      gaps.push_back(-x);
      ctgs.emplace_back();
    } else {
      ctgs.back().push_back(x);
    }
  }
}

void window_key(const gaml_ctx* ctx, const Walk& ctg, size_t i, Walk& key) {   // graph.cc:552-561, 618-627
  key.assign(1, ctg[i]);
  int beyond = 0;
  for (size_t j = i + 1; j < ctg.size(); j++) {
    beyond += ctx->node_len[ctg[j]];
    key.push_back(ctg[j]);
    if (beyond > kWindowLen) break;
  }
}

int find_key(const MateStore& st, const Walk& key) {
  auto it = st.key_ids.find(key);
  return it == st.key_ids.end() ? -1 : it->second;
}

// Paired lookup rule (ReadSet::GetPositionsOnlyPath, graph.cc:535-598) for one walk, both mates: the keys the
// walk looks up, in the reference's order, with walk-relative offsets. It depends only on the walk and on the
// set's key metadata, so it is computed once per distinct walk and cached until the set's cache grows — an
// annealing step re-submits ~all walks unchanged.
void build_walk_flat(const gaml_ctx* ctx, ReadSetState& rs, const Walk& walk, WalkFlat& out) {
  std::vector<Walk> ctgs;
  std::vector<int> gaps;
  split_at_gaps(walk, ctgs, gaps);
  Walk key;
  int cur_len = 0;
  out.e[0].clear();
  out.e[1].clear();
  out.records = out.records1 = 0;
  for (int m = 0; m < 2; m++) {
    out.gen[m] = rs.mate[m].keys.size();
    out.missing[m].clear();
  }
  out.contig_starts.assign(1, 0);   // events (0,1) and (cur_len,1) per later contig, graph.cc:1826, 1835
  for (size_t c = 0; c < ctgs.size(); c++) {
    if (c > 0) {
      cur_len += gaps[c - 1];
      out.contig_starts.push_back(cur_len);
    }
    const Walk& ctg = ctgs[c];
    int ctg_len = 0;
    for (int m = 0; m < 2; m++) {
      MateStore& st = rs.mate[m];
      int cur = cur_len, seen_max = 0;
      for (size_t i = 0; i < ctg.size(); i++) {
        int node_max = 0;
        window_key(ctx, ctg, i, key);
        int kid[2] = {find_key(st, key), -1};
        if (kid[0] < 0) out.missing[m].push_back(hash_nodes(key.data(), (int)key.size()));
        if (ctx->node_len[ctg[i]] > kWindowLen) {
          if (key.size() == 1) kid[1] = -1;   // window key IS the single-node key: the second lookup re-visits
                                              // the same list at the same offset, a no-op under the de-dup rule
          else {
            Walk one(1, ctg[i]);
            kid[1] = find_key(st, one);
            if (kid[1] < 0) out.missing[m].push_back(hash_nodes(one.data(), 1));
          }
        }
        for (int t = 0; t < 2; t++) {
          if (kid[t] < 0) continue;
          const KeyMeta& km = st.keys[kid[t]];
          const int skip = seen_max - 5;   // graph.cc:577
          if (km.count) {
            out.e[m].push_back(FlatEntry{kid[t], cur, skip, km.count, km.arena_off});
            out.records += km.count;
            if (m == 0) out.records1 += km.count;
          }
          if (km.any) {
            const int gp = (int)((unsigned)km.max_pos + (unsigned)cur);
            if (gp >= skip) node_max = std::max(node_max, gp);   // graph.cc:580
          }
        }
        cur += ctx->node_len[ctg[i]];
        seen_max = std::max(seen_max, node_max);   // graph.cc:596
      }
      ctg_len = cur - cur_len;
    }
    cur_len += ctg_len;
  }
}

size_t hash_walk(const Walk& w) { return WalkHash()(w); }

const WalkFlat& cached_walk_flat(const gaml_ctx* ctx, ReadSetState& rs, const WalkView& v) {
  FlatCache& fc = rs.flat_cache;
  if (WalkFlat* f = fc.find(v.p, v.n, v.h)) {
    bool stale = false;
    for (int m = 0; m < 2; m++) {
      const MateStore& st = rs.mate[m];
      if (f->gen[m] == st.keys.size()) continue;
      if (!f->missing[m].empty())
        for (size_t g = f->gen[m]; g < st.key_hash_log.size() && !stale; g++)
          stale = std::find(f->missing[m].begin(), f->missing[m].end(), st.key_hash_log[g]) != f->missing[m].end();
      f->gen[m] = st.keys.size();
    }
    if (!stale) return *f;
    build_walk_flat(ctx, rs, Walk(v.p, v.p + v.n), *f);   // a window this walk looks up has been inserted since
    return *f;
  }
  if (fc.nodes.size() >= (1u << 17)) fc.clear();   // bound the memory of a very long annealing run
  const Walk walk(v.p, v.p + v.n);
  WalkFlat& f = fc.insert(walk, v.h);
  build_walk_flat(ctx, rs, walk, f);
  return f;
}

// Appends one walk's lookups to the evaluation (walk ordinal `ord`): occurrences per mate store, record counts,
// and — for incremental evaluations — the mate-1 arena ranges the delta kernel enumerates.
void flatten_paired_walk(const gaml_ctx* ctx, ReadSetState& rs, const WalkView& walk, int ord, OccBuilder* ob[2],
                         SetPlan& sp, std::vector<TouchRange>* touch, std::vector<int>* contig_starts = nullptr) {
  const WalkFlat& f = cached_walk_flat(ctx, rs, walk);
  for (int m = 0; m < 2; m++)
    for (const FlatEntry& e : f.e[m]) {
      ob[m]->add(e.key, ord, e.cur, e.skip);
      if (m == 0 && touch) touch->push_back(TouchRange{e.arena_off, e.count});
    }
  sp.records += f.records;
  sp.records1 += f.records1;
  if (contig_starts) *contig_starts = f.contig_starts;
}

// Single lookup rule (CalcScoreForPaths + ReadSet::AddPositions, graph.cc:1665-1686, 600-649).
void flatten_single(const gaml_ctx* ctx, ReadSetState& rs, const Walk* walks, int n_walks, OccBuilder& ob, SetPlan& sp) {
  std::vector<Walk> ctgs;
  std::vector<int> gaps;
  Walk key;
  unsigned stride = 0, tl = 0;
  for (int wi = 0; wi < n_walks; wi++) {
    const Walk& w = walks[wi];
    split_at_gaps(w, ctgs, gaps);
    for (size_t c = 0; c < ctgs.size(); c++) {
      if (c > 0) tl += (unsigned)gaps[c - 1];
      unsigned cur = stride + tl;
      for (size_t i = 0; i < ctgs[c].size(); i++) {
        tl += (unsigned)ctx->node_len[ctgs[c][i]];
        window_key(ctx, ctgs[c], i, key);
        int kid = find_key(rs.mate[0], key);
        if (kid >= 0 && rs.mate[0].keys[kid].count) {
          ob.add(kid, 0, (int)cur, INT_MIN);
          sp.records += rs.mate[0].keys[kid].count;
        }
        cur += (unsigned)ctx->node_len[ctgs[c][i]];
      }
    }
    stride += 1000000u;   // graph.cc:1685
  }
  sp.total_len = (int)tl;
}

// PacBio lookup rule (PacbioReadSet::GetReadProbabilities, graph.cc:2410-2503) on normalised walks.
void flatten_pacbio(const gaml_ctx* ctx, ReadSetState& rs, const Walk* walks, int n_walks, OccBuilder& ob, SetPlan& sp) {
  unsigned tl = 0;
  Walk key;
  std::vector<int> begin, end;
  rs.h_pb_seeds.clear();
  rs.h_pb_occ.clear();
  rs.h_pb_prefix.clear();
  rs.h_pb_walk_len.clear();
  for (int wi = 0; wi < n_walks; wi++) {
    Walk w = walks[wi];
    for (int& x : w)
      if (x >= 0) x = ctx->nmap[x];   // graph.h:268-273
    const size_t n = w.size();
    begin.resize(n);
    end.resize(n);
    int off = 0;
    for (size_t i = 0; i < n; i++) {
      begin[i] = off;
      off += w[i] < 0 ? -w[i] : ctx->node_len[w[i]];
      end[i] = off;
    }
    tl += (unsigned)off;
    if (rs.pb_penalty) {   // coverage sweep inputs of this walk: its length, the artificial interval, one interval per node
      rs.h_pb_walk_len.push_back(off);
      rs.h_pb_seeds.push_back(make_int4(wi, -1000, 2000, 0));   // events (-1000, 1), (2000, -3000), graph.cc:3199-3200
      for (size_t i = 0; i < n; i++)
        if (w[i] >= 0) rs.h_pb_seeds.push_back(make_int4(wi, begin[i], end[i], 0));
    }
    for (size_t i = 0; i < n; i++) {
      key.clear();
      for (size_t j = i; j < n; j++) {
        key.push_back(w[j]);
        int kid = find_key(rs.mate[0], key);
        if (kid >= 0 && rs.mate[0].keys[kid].count) {
          ob.add(kid, 0, begin[i], INT_MIN);
          sp.records += rs.mate[0].keys[kid].count;
          if (rs.pb_penalty) {
            const KeyMeta& km = rs.mate[0].keys[kid];
            rs.h_pb_occ.push_back(make_int4(wi, begin[i], (int)km.arena_off, (int)km.count));
          }
        }
        if ((end[j] - begin[i]) - (end[i] - begin[i]) > rs.max_len[0]) break;   // graph.cc:2450
      }
    }
  }
  sp.total_len = (int)tl;
}

// Groups a store's occurrences by key: one SlotUpdate per live key (carrying its first occurrence) and, for the
// keys that occur several times (repeat nodes), their occurrences contiguous in enumeration order in the Occ array
// — the kernels read occ[occ_begin + t] only for t >= 1, so single-occurrence keys need no Occ entry.
// Counting pass over a per-key stamp table, no sort.
void group_occurrences(OccBuilder& ob, MateStore& st, uint32_t epoch, std::vector<SlotUpdate>& updates, std::vector<Occ>& occ,
                       bool record_base = false) {
  occ.clear();
  if (st.key_stamp.size() < st.keys.size()) {
    st.key_stamp.resize(st.keys.size(), 0u);
    st.key_slot.resize(st.keys.size(), 0);
  }
  const size_t first_update = updates.size();
  for (const std::pair<int, Occ>& it : ob.items) {
    const int k = it.first;
    if (st.key_stamp[k] != epoch) {
      st.key_stamp[k] = epoch;
      st.key_slot[k] = (int)updates.size();
      if (record_base) st.base_slot[k] = (int)updates.size();
      SlotUpdate u;
      u.key = k;
      u.n_occ = 1;
      u.occ_begin = 0;
      u.store = st.table_index;
      u.first = it.second;
      updates.push_back(u);
    } else {
      updates[st.key_slot[k]].n_occ++;
    }
  }
  int total = 0;
  for (size_t i = first_update; i < updates.size(); i++)
    if (updates[i].n_occ > 1) {
      updates[i].occ_begin = total;
      total += updates[i].n_occ;
    }
  if (total == 0) return;
  occ.resize(total);
  st.fill_cursor.assign(updates.size() - first_update, 0);
  for (const std::pair<int, Occ>& it : ob.items) {
    const size_t slot = (size_t)st.key_slot[it.first];
    const SlotUpdate& u = updates[slot];
    if (u.n_occ > 1) occ[u.occ_begin + st.fill_cursor[slot - first_update]++] = it.second;
  }
}

int ensure_pinned(gaml_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->h_blob_cap) return GAML_OK;
  if (ctx->h_blob) cudaFreeHost(ctx->h_blob);
  ctx->h_blob = nullptr;
  size_t cap = std::max<size_t>(bytes * 2, 1 << 16);
  CU(cudaMallocHost(&ctx->h_blob, cap));
  ctx->h_blob_cap = cap;
  return GAML_OK;
}

// Cache append (SURVEY §7.3 "the arena must support append"; kernels.cu "cache append"): keys inserted since the last
// full build — typically the windows of one new join, a few hundred records — are applied in O(new records): records to
// the arena tail, one relocated row block per read that gained records, the read flagged for the appendix phase, the
// new keys added to the key maps. Returns 1 = applied, 0 = not applicable (the caller rebuilds), < 0 = error.
int try_append(gaml_ctx* ctx, ReadSetState& rs) {
  if (!ctx->append_enabled || rs.cfg.kind != GAML_KIND_PAIRED || rs.n_mates != 2 || !rs.base_built || !rs.pairs_ok || rs.penalty) return 0;
  cudaStream_t st_ = ctx->stream;
  struct MatePlan {
    std::vector<int4> new_rows;             // {key, pos, edor, seq}, grouped by read
    std::vector<AppendGroupHost> groups;
    size_t tail_after = 0;
  } plan[2];
  size_t newly_dirty = 0;
  std::vector<uint32_t> dirty_now;
  for (int m = 0; m < 2; m++) {
    MateStore& st = rs.mate[m];
    plan[m].tail_after = st.rows_tail;
    if (!st.dirty || st.pending.empty()) continue;
    if (st.total_records() > 0xfffffff0ull) return 0;
    const size_t n = st.pending.size();
    // group the new records by read, arena order inside a group. Grouping by the CALLER's read id is the same grouping
    // (the internal order is a bijection) and needs no lookups while sorting; one key's records usually arrive in
    // ascending read order already.
    std::vector<uint64_t> order(n);
    bool sorted = true;
    for (size_t i = 0; i < n; i++) {
      order[i] = ((uint64_t)(uint32_t)st.pending[i].x << 32) | (uint64_t)i;
      sorted &= i == 0 || order[i - 1] < order[i];
    }
    if (!sorted) std::sort(order.begin(), order.end());
    plan[m].new_rows.resize(n);
    size_t tail = st.rows_tail;
    for (size_t i = 0; i < n;) {
      const uint32_t caller_read = (uint32_t)(order[i] >> 32);
      const uint32_t r = rs.perm_valid ? rs.h_inv[(size_t)caller_read] : caller_read;
      size_t j = i;
      for (; j < n && (uint32_t)(order[j] >> 32) == caller_read; j++) {
        const uint32_t src = (uint32_t)order[j];
        const int4& a = st.pending[src];   // {read, pos, edor, key}
        plan[m].new_rows[j] = make_int4(a.w, a.y, a.z, (int)(uint32_t)(st.arena_n + src));
      }
      const size_t cnt_old = st.h_count[r], need = cnt_old + (j - i);
      if (need >= 0x3fff || cnt_old == 0xffff) return 0;
      plan[m].groups.push_back(AppendGroupHost{r, (uint32_t)i, (uint32_t)(j - i), (uint32_t)tail});
      tail += need;
      if (!rs.h_dirty[r]) {
        rs.h_dirty[r] = 2;   // provisional: counted once over both mates, confirmed or rolled back below
        dirty_now.push_back(r);
        newly_dirty++;
      }
      i = j;
    }
    plan[m].tail_after = tail;
  }
  const size_t limit = std::max<size_t>(4096, (size_t)rs.n_local / 16);
  const bool fits = plan[0].tail_after <= rs.mate[0].rows_cap && plan[1].tail_after <= rs.mate[1].rows_cap &&
                    (size_t)rs.n_appx + newly_dirty <= limit;
  if (!fits) {
    for (uint32_t r : dirty_now) rs.h_dirty[r] = 0;
    return 0;
  }
  for (uint32_t r : dirty_now) rs.h_dirty[r] = 1;
  // ---- key maps between the mates' stores (and the combined slot table): entries that change, as (index, value) patches ----
  std::vector<int2> p12_patch, p21_patch;
  size_t old1 = 0, old2 = 0;
  {
    MateStore &s1 = rs.mate[0], &s2 = rs.mate[1];
    const size_t k1 = s1.keys.size(), k2 = s2.keys.size();
    old1 = rs.h_p12.size();
    old2 = rs.h_p21.size();
    rs.h_p12.resize(std::max<size_t>(k1, 1), -1);
    rs.h_p21.resize(std::max<size_t>(k2, 1), -1);
    for (size_t k = s1.built_keys; k < k1; k++) {
      auto it = s2.key_ids.find(*s1.key_by_id[k]);
      if (it != s2.key_ids.end()) {
        rs.h_p12[k] = it->second;
        rs.h_p21[(size_t)it->second] = (int32_t)k;
        if ((size_t)it->second < std::min(old2, s2.built_keys)) p21_patch.push_back(make_int2(it->second, (int)k));   // an OLD key of the other store
      }
    }
    for (size_t k = s2.built_keys; k < k2; k++) {
      auto it = s1.key_ids.find(*s2.key_by_id[k]);
      if (it != s1.key_ids.end()) {
        rs.h_p21[k] = it->second;
        rs.h_p12[(size_t)it->second] = (int32_t)k;
        if ((size_t)it->second < std::min(old1, s1.built_keys)) p12_patch.push_back(make_int2(it->second, (int)k));
      }
    }
    for (size_t k = std::min(old1, s1.built_keys); k < rs.h_p12.size(); k++) p12_patch.push_back(make_int2((int)k, rs.h_p12[k]));
    for (size_t k = std::min(old2, s2.built_keys); k < rs.h_p21.size(); k++) p21_patch.push_back(make_int2((int)k, rs.h_p21[k]));
  }
  // ---- ONE staged blob (pinned), ONE copy, ONE launch ----
  auto align16 = [](size_t x) { return (x + 15) & ~size_t(15); };
  size_t off = 0, arena_off[2], rows_off[2], grp_off[2];
  for (int m = 0; m < 2; m++) {
    MateStore& st = rs.mate[m];
    const bool has = st.dirty && !st.pending.empty();
    arena_off[m] = off;
    off = align16(off + (has ? st.pending.size() * 16 : 0));
    rows_off[m] = off;
    off = align16(off + (has ? plan[m].new_rows.size() * 16 : 0));
    grp_off[m] = off;
    off = align16(off + (has ? plan[m].groups.size() * sizeof(AppendGroupHost) : 0));
  }
  const size_t appx_off = off;
  off = align16(off + dirty_now.size() * 4);
  const size_t p12_off = off;
  off = align16(off + p12_patch.size() * sizeof(int2));
  const size_t p21_off = off;
  off = align16(off + p21_patch.size() * sizeof(int2));
  const size_t blob_bytes = off;
  if (ctx->append_copy_pending) {   // the previous append's copy reads the pinned staging
    CU(cudaEventSynchronize(ctx->ev_append));
    ctx->append_copy_pending = false;
  }
  if (blob_bytes > ctx->h_append_cap) {
    if (ctx->h_append_pinned) cudaFreeHost(ctx->h_append_pinned);
    ctx->h_append_pinned = nullptr;
    ctx->h_append_cap = 0;
    const size_t cap = std::max<size_t>(blob_bytes * 2, (size_t)1 << 18);
    CU(cudaMallocHost(&ctx->h_append_pinned, cap));
    ctx->h_append_cap = cap;
  }
  char* hb = static_cast<char*>(ctx->h_append_pinned);
  CU(rs.d_append_blob.reserve(std::max<size_t>(blob_bytes, (size_t)1 << 18), 0, false, st_));
  char* db = rs.d_append_blob.as<char>();
  AppendJob J{};
  for (int m = 0; m < 2; m++) {
    MateStore& st = rs.mate[m];
    const bool has = st.dirty && !st.pending.empty();
    AppendMate& am = J.m[m];
    if (has) {
      const size_t total = st.total_records();
      if (rs.perm_valid)
        for (int4& v : st.pending) v.x = (int)rs.h_inv[(size_t)v.x];
      CU(st.arena.reserve(total * 16, st.arena_n * 16, false, st_));
      memcpy(hb + arena_off[m], st.pending.data(), st.pending.size() * 16);
      memcpy(hb + rows_off[m], plan[m].new_rows.data(), plan[m].new_rows.size() * 16);
      memcpy(hb + grp_off[m], plan[m].groups.data(), plan[m].groups.size() * sizeof(AppendGroupHost));
      am.arena_src = db + arena_off[m];
      am.arena_dst = st.arena.as<char>() + st.arena_n * 16;
      am.n_rec = (uint32_t)st.pending.size();
      am.groups = db + grp_off[m];
      am.n_groups = (int)plan[m].groups.size();
      am.new_rows = db + rows_off[m];
      am.rows = st.rows.p;
      am.first = st.first.p;
      for (const AppendGroupHost& g : plan[m].groups) st.h_count[g.read] = (uint16_t)(st.h_count[g.read] + g.n_new);
      st.rows_tail = plan[m].tail_after;
      st.arena_n = total;
      st.pending.clear();
    }
    if (st.dirty) {
      const size_t old_slots = st.slots_a.cap;
      CU(st.slots_a.reserve(std::max<size_t>(st.keys.size(), 1) * sizeof(SlotA), 0, true, st_));
      CU(st.slots_b.reserve(std::max<size_t>(st.keys.size(), 1) * sizeof(SlotB), 0, true, st_));
      if (st.slots_a.cap != old_slots) ctx->tables_dirty = true;
      st.dirty = false;
    }
  }
  J.dirty = rs.d_dirty.as<uint32_t>();
  J.pairs = rs.d_pairs.p;
  J.fast = rs.fast_ok ? rs.d_fast.p : nullptr;
  if (!dirty_now.empty()) {
    CU(rs.d_appx.reserve(((size_t)rs.n_appx + dirty_now.size()) * 4, (size_t)rs.n_appx * 4, false, st_));
    memcpy(hb + appx_off, dirty_now.data(), dirty_now.size() * 4);
    J.appx_src = reinterpret_cast<const uint32_t*>(db + appx_off);
    J.appx_dst = rs.d_appx.as<uint32_t>() + rs.n_appx;
    J.n_appx_new = (int)dirty_now.size();
    rs.n_appx += (int)dirty_now.size();
  }
  {
    MateStore &s1 = rs.mate[0], &s2 = rs.mate[1];
    const void* old_comb = rs.d_comb.p;
    const void* old_p21 = rs.d_partner21.p;
    CU(rs.d_partner12.reserve(rs.h_p12.size() * 4, old1 * 4, false, st_));
    CU(rs.d_partner21.reserve(rs.h_p21.size() * 4, old2 * 4, false, st_));
    if (!p12_patch.empty()) memcpy(hb + p12_off, p12_patch.data(), p12_patch.size() * sizeof(int2));
    if (!p21_patch.empty()) memcpy(hb + p21_off, p21_patch.data(), p21_patch.size() * sizeof(int2));
    J.p12_patch = reinterpret_cast<const int2*>(db + p12_off);
    J.n_p12 = (int)p12_patch.size();
    J.p12 = rs.d_partner12.as<int32_t>();
    J.p21_patch = reinterpret_cast<const int2*>(db + p21_off);
    J.n_p21 = (int)p21_patch.size();
    J.p21 = rs.d_partner21.as<int32_t>();
    CU(rs.d_comb.reserve(rs.h_p12.size() * 4 * sizeof(SlotA), 0, true, st_));   // per-evaluation contents: nothing to keep
    if (rs.d_comb.p != old_comb || rs.d_partner21.p != old_p21) ctx->tables_dirty = true;
    s1.built_keys = s1.keys.size();
    s2.built_keys = s2.keys.size();
  }
  int launches = 0;
  if (blob_bytes) {
    CU(cudaMemcpyAsync(db, hb, blob_bytes, cudaMemcpyHostToDevice, st_));
    CU(cudaEventRecord(ctx->ev_append, st_));
    ctx->append_copy_pending = true;
    launch_append_apply(J, st_);
    CU(cudaGetLastError());
    launches++;
  }
  ctx->stats.kernel_launches += launches;
  rs.appends++;
  return 1;
}

// Upload staged cache inserts and rebuild the read-major CSR of every dirty store.
int commit(gaml_ctx* ctx) {
  bool rebuilt = false;
  for (auto& rsp : ctx->sets) {
    ReadSetState& rs = *rsp;
    bool any_dirty = false;
    for (int m = 0; m < rs.n_mates; m++) any_dirty |= rs.mate[m].dirty;
    if (any_dirty) {
      ctx->cache_gen++;
      const int ar = try_append(ctx, rs);
      if (ar < 0) return ar;
      if (ar == 1) continue;
      for (int m = 0; m < rs.n_mates; m++) rs.mate[m].dirty = true;   // full rebuild of the set: both mates' lists and the shared ones
      rs.rebuilds++;
      rebuilt = true;
    }
   for (int pass = 0; pass < 2; pass++) {   // (a second pass only right after the internal read order has been fixed)
    for (int m = 0; m < rs.n_mates; m++) {
      MateStore& st = rs.mate[m];
      if (!st.dirty) continue;
      const size_t total = st.total_records();
      if (rs.perm_valid)   // the arena speaks internal read indices
        for (int4& v : st.pending) v.x = (int)rs.h_inv[(size_t)v.x];
      if (total > 0xfffffff0ull) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^32 alignment records in one mate store");
      CU(st.arena.reserve(std::max<size_t>(total, 1) * 16, st.arena_n * 16, false, ctx->stream));
      if (st.is_long) CU(st.arena_pos.reserve(std::max<size_t>(total, 1) * 8, st.arena_n * 8, false, ctx->stream));
      if (!st.pending.empty()) {
        CU(cudaMemcpyAsync(st.arena.as<char>() + st.arena_n * 16, st.pending.data(), st.pending.size() * 16,
                           cudaMemcpyHostToDevice, ctx->stream));
        if (st.is_long)
          CU(cudaMemcpyAsync(st.arena_pos.as<char>() + st.arena_n * 8, st.pending_pos.data(), st.pending_pos.size() * 8,
                             cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        st.arena_n = total;
        st.pending.clear();
        st.pending.shrink_to_fit();
        st.pending_pos.clear();
        st.pending_pos.shrink_to_fit();
      }
      st.rows_cap = st.is_long ? std::max<size_t>(total, 1) : total + std::max<size_t>(total / 4, (size_t)1 << 16);   // slack for appends
      st.rows_tail = total;
      CU(st.rows.reserve(st.rows_cap * 16, 0, false, ctx->stream));
      st.rows_cap = std::max(st.rows_cap, st.rows.cap / 16);
      if (!st.is_long) CU(st.first.reserve(std::max<size_t>(rs.n_local, 1) * 16, 0, false, ctx->stream));
      CU(st.rowptr.reserve(((size_t)rs.n_local + 1) * 4, 0, false, ctx->stream));
      CU(st.cursor.reserve(((size_t)rs.n_local + 1) * 4, 0, false, ctx->stream));
      const size_t old_slots = st.slots_a.cap;
      CU(st.slots_a.reserve(std::max<size_t>(st.keys.size(), 1) * sizeof(SlotA), 0, true, ctx->stream));
      CU(st.slots_b.reserve(std::max<size_t>(st.keys.size(), 1) * sizeof(SlotB), 0, true, ctx->stream));
      if (st.slots_a.cap != old_slots) ctx->tables_dirty = true;
      const size_t temp = csr_temp_bytes(rs.n_local);
      CU(ctx->d_csr_temp.reserve(std::max<size_t>(temp, 256), 0, false, ctx->stream));
      int launches = 0;
      CU(build_csr(st.arena.p, st.arena_n, rs.n_local, st.is_long, st.rowptr.as<uint32_t>(), st.cursor.as<uint32_t>(),
                   st.rows.p, st.first.p, ctx->d_csr_temp.p, ctx->d_csr_temp.cap, ctx->sm_count, ctx->stream, &launches));
      ctx->stats.kernel_launches += launches;
      st.dirty = false;
      rs.complex_dirty = true;
      // (the per-walk lookup cache stays: keys are immutable, cached_walk_flat re-checks the windows a walk missed)
    }
    if (rs.complex_dirty && rs.cfg.kind != GAML_KIND_PACBIO) {
      // static tier-2 list: reads that own more than one record on some mate
      CU(rs.d_complex.reserve(std::max<size_t>(rs.n_local, 1) * 4, 0, false, ctx->stream));
      uint32_t* flags = rs.mate[0].cursor.as<uint32_t>();   // scratch, free after build_csr
      int launches = 0;
      uint32_t n_complex = 0;
      CU(build_complex_list(rs.mate[0].first.p, rs.n_mates == 2 ? rs.mate[1].first.p : nullptr, rs.n_local, flags,
                            rs.d_complex.as<uint32_t>(), ctx->d_csr_temp.p, ctx->d_csr_temp.cap, ctx->stream, &launches,
                            &n_complex, rs.class_begin));
      ctx->stats.kernel_launches += launches;
      launches = 0;
      rs.n_complex = (int)n_complex;
      // compact copy of the listed reads' rows, per mate, + their packed lengths
      CU(rs.d_clens.reserve(std::max<size_t>(n_complex, 1) * 4, 0, false, ctx->stream));
      for (int m = 0; m < rs.n_mates; m++) {
        MateStore& st = rs.mate[m];
        CU(st.cptr.reserve(((size_t)n_complex + 1) * 4, 0, false, ctx->stream));
        CU(compact_offsets(rs.d_complex.as<uint32_t>(), rs.n_complex, st.rowptr.as<uint32_t>(), st.cptr.as<uint32_t>(),
                           rs.d_lens.as<uint32_t>(), m == 0 ? rs.d_clens.as<uint32_t>() : nullptr, ctx->d_csr_temp.p,
                           ctx->d_csr_temp.cap, ctx->stream, &launches));
        uint32_t total_rows = 0;
        CU(cudaMemcpyAsync(&total_rows, st.cptr.as<uint32_t>() + n_complex, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(st.crows.reserve(std::max<size_t>(total_rows, 1) * 16, 0, false, ctx->stream));
        CU(compact_copy(rs.d_complex.as<uint32_t>(), rs.n_complex, st.rowptr.as<uint32_t>(), st.cptr.as<uint32_t>(), st.rows.p,
                        st.crows.p, ctx->stream, &launches));
      }
      memset(rs.cbase, 0, sizeof(rs.cbase));
      for (int m = 0; m < rs.n_mates; m++)
        for (int c = 0; c < 5; c++)   // class_begin[c] <= n_complex, cptr has n_complex + 1 entries
          CU(cudaMemcpyAsync(&rs.cbase[m][c], rs.mate[m].cptr.as<uint32_t>() + rs.class_begin[c], 4, cudaMemcpyDeviceToHost, ctx->stream));
      CU(rs.d_cdesc.reserve(std::max<size_t>(n_complex, 1) * 16, 0, false, ctx->stream));
      launch_cdesc_fill(rs.d_complex.as<uint32_t>(), rs.n_complex, rs.d_lens.as<uint32_t>(), rs.mate[0].cptr.as<uint32_t>(),
                        rs.n_mates == 2 ? rs.mate[1].cptr.as<uint32_t>() : nullptr, rs.d_cdesc.p, ctx->stream);
      launches++;
      rs.pairs_ok = false;
      uint32_t pack_bad = 0;
      if (rs.cfg.kind == GAML_KIND_PAIRED && rs.n_mates == 2 && rs.n_local > 0) {
        // key maps between the two mates' stores (same node sequence) and the combined slot table
        {
          MateStore &s1 = rs.mate[0], &s2 = rs.mate[1];
          std::vector<int32_t>& p12 = rs.h_p12;
          std::vector<int32_t>& p21 = rs.h_p21;
          p12.assign(std::max<size_t>(s1.keys.size(), 1), -1);
          p21.assign(std::max<size_t>(s2.keys.size(), 1), -1);
          s1.built_keys = s1.keys.size();
          s2.built_keys = s2.keys.size();
          for (const auto& kv : s1.key_ids) {
            auto it = s2.key_ids.find(kv.first);
            if (it != s2.key_ids.end()) {
              p12[kv.second] = it->second;
              p21[it->second] = kv.second;
            }
          }
          const void* old_comb = rs.d_comb.p;
          const void* old_p21 = rs.d_partner21.p;
          CU(rs.d_partner12.reserve(p12.size() * 4, 0, false, ctx->stream));
          CU(rs.d_partner21.reserve(p21.size() * 4, 0, false, ctx->stream));
          CU(cudaMemcpyAsync(rs.d_partner12.p, p12.data(), p12.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
          CU(cudaMemcpyAsync(rs.d_partner21.p, p21.data(), p21.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
          CU(rs.d_comb.reserve(p12.size() * 4 * sizeof(SlotA), 0, true, ctx->stream));
          CU(cudaStreamSynchronize(ctx->stream));
          if (rs.d_comb.p != old_comb || rs.d_partner21.p != old_p21 || !rs.comb_ok) ctx->tables_dirty = true;
          rs.comb_ok = true;
        }
        // tier 1's packed copy of both mates' first records (16 B per pair instead of 2 x 16 B + lengths)
        CU(rs.d_pairs.reserve((size_t)rs.n_local * 16, 0, false, ctx->stream));
        uint32_t* bad = static_cast<uint32_t*>(ctx->d_csr_temp.p);   // scratch, free after build_csr / the list build
        CU(cudaMemsetAsync(bad, 0, 4, ctx->stream));
        launch_pack_pairs(rs.mate[0].first.p, rs.mate[1].first.p, rs.n_local, rs.d_partner12.as<int32_t>(), rs.d_pairs.p, bad, ctx->stream);
        launches++;
        pack_bad = 1;
        CU(cudaMemcpyAsync(&pack_bad, bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
      }
      CU(cudaStreamSynchronize(ctx->stream));   // cbase (copied above) and pack_bad are on the host now
      if (rs.cfg.kind == GAML_KIND_PAIRED && rs.n_mates == 2 && rs.n_local > 0) rs.pairs_ok = pack_bad == 0;
      rs.fast_ok = false;
      if (rs.pairs_ok && rs.comb_ok && rs.lens_uniform && rs.tq_shift > 0) {
        // tier 1's fast records: everything about a same-key pair that does not depend on the walks, resolved into a
        // term-table index; the remaining tier-1 reads go on the cross list
        CU(rs.d_fast.reserve((size_t)rs.n_local * 16, 0, false, ctx->stream));
        CU(rs.d_xlist.reserve((size_t)rs.n_local * 4, 0, false, ctx->stream));
        uint32_t* flags = rs.mate[0].cursor.as<uint32_t>();   // scratch (n_local + 1), free after the list build above
        CU(build_fast_pairs(rs.d_pairs.p, rs.n_local, rs.tq_shift, rs.ins_n, rs.uniform_ll, rs.d_fast.p, flags, rs.d_xlist.as<uint32_t>(),
                            ctx->d_csr_temp.p, ctx->d_csr_temp.cap, ctx->stream, &launches));
        uint32_t n_cross = 0;
        CU(cudaMemcpyAsync(&n_cross, flags + rs.n_local, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        rs.n_cross = (int)n_cross;
        rs.fast_ok = true;
      }
      rs.t2pack_ok = false;
      if (rs.pairs_ok && rs.class_begin[3] > 0) {
        // tier 2's packed entries: classes (1,2), (2,1) two units per read, (2,2) three, unit major per class
        const size_t n0 = (size_t)(rs.class_begin[1] - rs.class_begin[0]), n1 = (size_t)(rs.class_begin[2] - rs.class_begin[1]),
                     n2 = (size_t)(rs.class_begin[3] - rs.class_begin[2]);
        rs.t2base[0] = 0;
        rs.t2base[1] = (uint32_t)(2 * n0);
        rs.t2base[2] = (uint32_t)(2 * n0 + 2 * n1);
        CU(rs.d_t2pack.reserve((2 * n0 + 2 * n1 + 3 * n2) * 16, 0, false, ctx->stream));
        uint32_t* bad = static_cast<uint32_t*>(ctx->d_csr_temp.p);
        CU(cudaMemsetAsync(bad, 0, 4, ctx->stream));
        launch_pack_tier2(rs.d_cdesc.p, rs.mate[0].crows.p, rs.mate[1].crows.p, rs.class_begin, rs.cbase, rs.t2base, rs.d_t2pack.p,
                          bad, ctx->stream);
        launches++;
        uint32_t t2_bad = 1;
        CU(cudaMemcpyAsync(&t2_bad, bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        rs.t2pack_ok = t2_bad == 0;
      }
      ctx->stats.kernel_launches += launches;
      rs.complex_dirty = false;
      // the state appends build on: every read's record count per mate on the host, no read dirty, an empty appendix
      rs.base_built = false;
      if (rs.cfg.kind == GAML_KIND_PAIRED && rs.n_mates == 2 && rs.n_local > 0 && rs.pairs_ok) {
        DevBuf counts;
        CU(counts.reserve((size_t)rs.n_local * 2, 0, false, ctx->stream));
        for (int m = 0; m < 2; m++) {
          MateStore& st = rs.mate[m];
          launch_extract_counts(st.first.p, st.rowptr.as<uint32_t>(), rs.n_local, counts.as<uint16_t>(), ctx->stream);
          st.h_count.resize((size_t)rs.n_local);
          CU(cudaMemcpyAsync(st.h_count.data(), counts.p, (size_t)rs.n_local * 2, cudaMemcpyDeviceToHost, ctx->stream));
          CU(cudaStreamSynchronize(ctx->stream));
          ctx->stats.kernel_launches++;
        }
        CU(rs.d_dirty.reserve((size_t)rs.n_local * 4, 0, false, ctx->stream));
        CU(cudaMemsetAsync(rs.d_dirty.p, 0, (size_t)rs.n_local * 4, ctx->stream));
        rs.h_dirty.assign((size_t)rs.n_local, 0);
        rs.n_appx = 0;
        rs.base_built = true;
      }
    }
    if (pass == 1 || !rs.fast_ok || rs.perm_valid || !ctx->permute_reads) break;
    {
      // First commit of a set with fast records: fix the internal read order (fast reads by key and term-table index,
      // everything else behind them), rewrite the arenas' read field and build everything again in that order.
      const int n = rs.n_local;
      DevBuf keys, ids, inv, temp, nf;
      CU(keys.reserve((size_t)n * 2 * 8, 0, false, ctx->stream));
      CU(ids.reserve((size_t)n * 2 * 4, 0, false, ctx->stream));
      CU(inv.reserve((size_t)n * 4, 0, false, ctx->stream));
      CU(temp.reserve(std::max<size_t>(perm_temp_bytes(n), 256), 0, false, ctx->stream));
      CU(nf.reserve(256, 0, true, ctx->stream));
      int launches = 0;
      CU(build_read_permutation(rs.d_fast.p, n, keys.as<unsigned long long>(), ids.as<uint32_t>(), inv.as<uint32_t>(), nf.as<uint32_t>(),
                                temp.p, temp.cap, ctx->stream, &launches));
      rs.h_inv.resize((size_t)n);
      rs.h_perm.resize((size_t)n);
      uint32_t n_fast = 0;
      CU(cudaMemcpyAsync(rs.h_inv.data(), inv.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(rs.h_perm.data(), ids.as<uint32_t>() + n, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(&n_fast, nf.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
      for (int m = 0; m < rs.n_mates; m++) {
        launch_remap_arena(rs.mate[m].arena.p, rs.mate[m].arena_n, inv.as<uint32_t>(), ctx->sm_count, ctx->stream);
        launches++;
        rs.mate[m].dirty = true;
      }
      CU(cudaStreamSynchronize(ctx->stream));
      ctx->stats.kernel_launches += launches;
      rs.n_fast = (int)n_fast;
      rs.perm_valid = true;
      rs.has_state = false;      // (no evaluation can have happened on records of this set yet; a state of zeros stays zeros)
      rs.total_valid = false;
    }
   }
  }
  if (ctx->tables_dirty) {
    std::vector<void*> tabs;   // [SlotA* per store][SlotB* per store][combined-table base per store][its key map per store]
    for (MateStore* s : ctx->stores) tabs.push_back(s->slots_a.p);
    for (MateStore* s : ctx->stores) tabs.push_back(s->slots_b.p);
    std::vector<void*> cbase(ctx->stores.size(), nullptr), cmap(ctx->stores.size(), nullptr);
    for (auto& rsp2 : ctx->sets) {
      ReadSetState& r2 = *rsp2;
      if (!r2.comb_ok || r2.n_mates != 2) continue;
      for (size_t i = 0; i < ctx->stores.size(); i++) {
        if (ctx->stores[i] == &r2.mate[0]) cbase[i] = r2.d_comb.p;
        if (ctx->stores[i] == &r2.mate[1]) {
          cbase[i] = r2.d_comb.as<SlotA>() + 1;
          cmap[i] = r2.d_partner21.p;
        }
      }
    }
    for (void* q : cbase) tabs.push_back(q);
    for (void* q : cmap) tabs.push_back(q);
    ctx->h_tables = StoreTables{};
    for (size_t i = 0; i < ctx->stores.size() && i < (size_t)kInlineStores; i++) {
      ctx->h_tables.a[i] = ctx->stores[i]->slots_a.as<SlotA>();
      ctx->h_tables.b[i] = ctx->stores[i]->slots_b.as<SlotB>();
      ctx->h_tables.cb[i] = static_cast<SlotA*>(cbase[i]);
      ctx->h_tables.cm[i] = static_cast<const int32_t*>(cmap[i]);
    }
    CU(ctx->d_tables.reserve(std::max<size_t>(tabs.size(), 1) * sizeof(void*), 0, false, ctx->stream));
    if (!tabs.empty())
      CU(cudaMemcpyAsync(ctx->d_tables.p, tabs.data(), tabs.size() * sizeof(void*), cudaMemcpyHostToDevice, ctx->stream));
    ctx->tables_dirty = false;
  }
  if (rebuilt) CU(cudaStreamSynchronize(ctx->stream));   // (appends and table uploads are ordered on the stream: nothing to wait for)
  return GAML_OK;
}

// ---- patched full evaluation ------------------------------------------------------------------------------------------
constexpr int kMaxPatchWalks = 64;
constexpr size_t kPatchReserve = (size_t)1 << 18;   // room behind the base blob in d_full_blob
bool patch_debug() {
  static const bool on = getenv("GAML_B200_PATCH_DEBUG") != nullptr;
  return on;
}

// Prepares a full evaluation of cur() as the resident base blob plus a patch. Returns 1 = prepared, 0 = not applicable
// (the caller flattens every walk), < 0 = error.
int prepare_full_patch(gaml_ctx* ctx, int total_len) {
  const ListTrack& tc = ctx->track[ctx->cur_set];
  const WalkSet& ws = ctx->cur();
  const int g = ctx->base_g, S = ctx->base_s;
  const uint32_t gmask = (1u << g) - 1u;
  std::vector<int> added;
  for (int y = 0; y < ws.n; y++)
    if (tc.label[(size_t)y] & gmask) added.push_back(y);
  std::vector<uint32_t> gone;   // labels of the missing base walks, ascending
  for (int b : tc.removed) gone.push_back((uint32_t)(b + 1) << g);
  auto is_gone = [&](int walk) { return std::binary_search(gone.begin(), gone.end(), (uint32_t)walk); };
  if (++ctx->stamp_gen == 0) {
    for (MateStore* st : ctx->stores) std::fill(st->key_stamp.begin(), st->key_stamp.end(), 0u);
    ctx->stamp_gen = 1;
  }
  const uint32_t stamp = ctx->stamp_gen;
  const size_t n_sets = ctx->sets.size(), n_stores = ctx->stores.size();
  ctx->plan = ctx->full_plan;
  std::vector<int32_t> skip;
  std::vector<SlotUpdate> pupd;
  std::vector<std::vector<Occ>> pocc(n_stores);
  std::vector<std::vector<TouchRange>> pmt(n_sets);
  std::vector<char> mt_changed(n_sets, 0);
  struct AddOcc { int key; Occ o; };
  std::vector<Occ> tmp;
  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    SetPlan& sp = ctx->plan[s];
    std::vector<AddOcc> adds[2];
    std::vector<int> akeys[2];
    auto touch_key = [&](int m, int k) {
      MateStore& st = rs.mate[m];
      if (st.key_stamp.size() < st.keys.size()) {
        st.key_stamp.resize(st.keys.size(), 0u);
        st.key_slot.resize(st.keys.size(), 0);
      }
      if (st.key_stamp[k] == stamp) return;
      st.key_stamp[k] = stamp;
      akeys[m].push_back(k);
    };
    for (int b : tc.removed) {
      const WalkFlat& f = cached_walk_flat(ctx, rs, ctx->base_ws.view(b));
      sp.records -= f.records;
      sp.records1 -= f.records1;
      for (int m = 0; m < 2; m++)
        for (const FlatEntry& e : f.e[m]) touch_key(m, e.key);
    }
    for (int y : added) {
      const WalkFlat& f = cached_walk_flat(ctx, rs, ws.view(y));
      sp.records += f.records;
      sp.records1 += f.records1;
      const uint32_t lab = tc.label[(size_t)y];
      for (int m = 0; m < 2; m++) {
        if (f.e[m].size() >= ((size_t)1 << S)) return 0;   // more lookups than a label's enumeration range holds
        uint32_t seg = lab << S;
        for (const FlatEntry& e : f.e[m]) {
          adds[m].push_back(AddOcc{e.key, Occ{(int)lab, (int)seg++, e.cur, e.skip}});
          touch_key(m, e.key);
        }
      }
    }
    std::vector<std::pair<int, int>> new_multi;   // (mate, key)
    for (int m = 0; m < 2; m++) {
      MateStore& st = rs.mate[m];
      std::stable_sort(adds[m].begin(), adds[m].end(), [](const AddOcc& a, const AddOcc& b) { return a.key < b.key; });
      for (int k : akeys[m]) {
        tmp.clear();
        const int bi = (size_t)k < st.base_slot.size() ? st.base_slot[k] : -1;
        bool base_multi = false;
        if (bi >= 0) {
          skip.push_back(bi);
          const SlotUpdate& bu = ctx->full_updates[(size_t)bi];
          base_multi = bu.n_occ > 1;
          if (bu.n_occ == 1) {
            if (!is_gone(bu.first.walk)) tmp.push_back(bu.first);
          } else {
            const std::vector<Occ>& fo = ctx->full_occs[st.table_index];
            for (int t = 0; t < bu.n_occ; t++)
              if (!is_gone(fo[(size_t)bu.occ_begin + t].walk)) tmp.push_back(fo[(size_t)bu.occ_begin + t]);
          }
        }
        auto lo = std::lower_bound(adds[m].begin(), adds[m].end(), k, [](const AddOcc& a, int key) { return a.key < key; });
        for (; lo != adds[m].end() && lo->key == k; ++lo) tmp.push_back(lo->o);
        std::sort(tmp.begin(), tmp.end(), [](const Occ& a, const Occ& b) { return (uint32_t)a.seg < (uint32_t)b.seg; });
        if (base_multi || tmp.size() > 1) mt_changed[s] = 1;
        if (tmp.empty()) continue;   // the key is not live in this evaluation: its slot keeps a stale epoch
        SlotUpdate u;
        u.key = k;
        u.n_occ = (int)tmp.size();
        u.occ_begin = 0;
        u.store = st.table_index;
        u.first = tmp[0];
        if (tmp.size() > 1) {
          u.occ_begin = (int)pocc[st.table_index].size();   // rebased below, once the patch has its place in the blob
          pocc[st.table_index].insert(pocc[st.table_index].end(), tmp.begin(), tmp.end());
          new_multi.push_back({m, k});
        }
        pupd.push_back(u);
      }
    }
    if (mt_changed[s]) {
      sp.multi_records = 0;
      for (int m = 0; m < 2; m++) {
        const MateStore& st = rs.mate[m];
        auto push = [&](int k) {
          const KeyMeta& km = st.keys[k];
          if (!km.count) return;
          pmt[s].push_back(TouchRange{km.arena_off, km.count});
          sp.multi_records += km.count;
        };
        for (const std::pair<int, int>& mk : ctx->base_mkeys[s])
          if (mk.first == m && st.key_stamp[mk.second] != stamp) push(mk.second);
        for (const std::pair<int, int>& mk : new_multi)
          if (mk.first == m) push(mk.second);
        if (m == 0) sp.n_mtouch1 = (int)pmt[s].size();
      }
      sp.n_mtouch = (int)pmt[s].size();
    }
    sp.total_len = total_len;
    sp.full = true;
    sp.delta_only = false;
  }
  std::sort(skip.begin(), skip.end());

  // ---- the patch's place behind the base blob ----
  auto align16 = [](size_t x) { return (x + 15) & ~size_t(15); };
  const size_t p0 = align16(ctx->full_blob_bytes);
  size_t off = p0;
  ctx->patch_skip_off = off;
  off = align16(off + skip.size() * sizeof(int32_t));
  ctx->patch_upd_off = off;
  off = align16(off + pupd.size() * sizeof(SlotUpdate));
  std::vector<size_t> pocc_off(n_stores);
  for (size_t i = 0; i < n_stores; i++) {
    pocc_off[i] = off;
    off = align16(off + pocc[i].size() * sizeof(Occ));
  }
  for (size_t s = 0; s < n_sets; s++) {
    SetPlan& sp = ctx->plan[s];
    ReadSetState& rs = *ctx->sets[s];
    if (mt_changed[s]) {
      sp.mtouch_off = off;
      off = align16(off + pmt[s].size() * sizeof(TouchRange));
      sp.mprefix_off = off;
      off = align16(off + (pmt[s].size() + 1) * sizeof(uint32_t));
    }
    sp.pstar_off = off;
    off = align16(off + std::max<size_t>(rs.h_thr.size(), 1) * sizeof(double));
  }
  if (off > ctx->d_full_blob.cap) return 0;
  // occurrence lists of the patch are addressed relative to the base's per-store arrays (same buffer)
  for (SlotUpdate& u : pupd)
    if (u.n_occ > 1) {
      size_t base_occ = 0;
      for (size_t s = 0; s < n_sets; s++)
        for (int m = 0; m < 2; m++)
          if (ctx->sets[s]->mate[m].table_index == u.store) base_occ = ctx->plan[s].occ_off[m];
      u.occ_begin += (int)((pocc_off[(size_t)u.store] - base_occ) / sizeof(Occ));
    }
  const size_t bytes = off - p0;
  int rc = ensure_pinned(ctx, bytes);
  if (rc != GAML_OK) return rc;
  char* hb = static_cast<char*>(ctx->h_blob) - p0;   // (offsets below are blob offsets)
  if (!skip.empty()) memcpy(hb + ctx->patch_skip_off, skip.data(), skip.size() * sizeof(int32_t));
  if (!pupd.empty()) memcpy(hb + ctx->patch_upd_off, pupd.data(), pupd.size() * sizeof(SlotUpdate));
  for (size_t i = 0; i < n_stores; i++)
    if (!pocc[i].empty()) memcpy(hb + pocc_off[i], pocc[i].data(), pocc[i].size() * sizeof(Occ));
  for (size_t s = 0; s < n_sets; s++) {
    SetPlan& sp = ctx->plan[s];
    ReadSetState& rt = *ctx->sets[s];
    if (mt_changed[s]) {
      if (!pmt[s].empty()) memcpy(hb + sp.mtouch_off, pmt[s].data(), pmt[s].size() * sizeof(TouchRange));
      uint32_t* mpre = reinterpret_cast<uint32_t*>(hb + sp.mprefix_off);
      uint64_t macc = 0;
      for (size_t t = 0; t < pmt[s].size(); t++) {
        mpre[t] = (uint32_t)macc;
        macc += pmt[s][t].count;
      }
      if (macc > 0xffffffffull) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^32 records under repeated keys in one evaluation");
      mpre[pmt[s].size()] = (uint32_t)macc;
    }
    const int two_len = two_len_of(sp.total_len);
    if (!rt.pstar_valid || rt.pstar_two_len != two_len) {
      rt.h_pstar.assign(rt.h_thr.size(), 0.0);
      for (int li : rt.len_classes) rt.h_pstar[li] = floor_pstar(rt.h_thr[li], (double)two_len);
      rt.pstar_two_len = two_len;
      rt.pstar_valid = true;
    }
    if (!rt.h_pstar.empty()) memcpy(hb + sp.pstar_off, rt.h_pstar.data(), rt.h_pstar.size() * sizeof(double));
  }
  ctx->n_updates = ctx->full_n_updates;
  ctx->upd_off = ctx->full_upd_off;
  ctx->n_patch = (int)pupd.size();
  ctx->n_skip = (int)skip.size();
  ctx->blob_bytes = off;
  ctx->blob_dev = ctx->d_full_blob.as<char>();
  CU(ctx->d_flags.reserve(flags_words(n_sets) * sizeof(unsigned long long), 0, true, ctx->stream));
  for (auto& rsp : ctx->sets) CU(rsp->d_ovf_list.reserve((size_t)ctx->ovf_cap * 4, 0, false, ctx->stream));
  CU(ctx->d_scratch.reserve(ctx->scratch_entries * sizeof(Plc), 0, false, ctx->stream));
  if (bytes) CU(cudaMemcpyAsync(ctx->blob_dev + p0, ctx->h_blob, bytes, cudaMemcpyHostToDevice, ctx->stream));
  ctx->stats.last_h2d_bytes = (int64_t)bytes;
  return 1;
}

// GAML_B200_PREP_TIMING=1: mean host microseconds of prepare()'s phases, printed to stderr every 100 evaluations
struct PrepTimer {
  bool on;
  std::chrono::steady_clock::time_point t;
  static constexpr int kPhases = 8;
  static double acc[kPhases];
  static long calls;
  PrepTimer() : on(getenv("GAML_B200_PREP_TIMING") != nullptr) { if (on) t = std::chrono::steady_clock::now(); }
  void lap(int phase) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    acc[phase] += std::chrono::duration<double, std::micro>(n - t).count();
    t = n;
  }
  void done() {
    if (!on || ++calls % 100) return;
    fprintf(stderr, "[gaml_b200] prepare us/call: load %.1f len+commit %.1f track %.1f patch/reuse %.1f flatten %.1f pack %.1f enqueue %.1f\n",
            acc[0] / 100, acc[1] / 100, acc[2] / 100, acc[3] / 100, acc[4] / 100, acc[5] / 100, acc[6] / 100);
    for (double& a : acc) a = 0;
  }
};
double PrepTimer::acc[PrepTimer::kPhases] = {0};
long PrepTimer::calls = 0;

int prepare(gaml_ctx* ctx, const int32_t* nodes, const int64_t* offs, int n_walks) {
  PrepTimer pt;
  if (n_walks < 0 || (n_walks > 0 && (!nodes || !offs))) return fail(ctx, GAML_ERR_ARG, "bad walk arrays");
  if (ctx->node_len.empty()) return fail(ctx, GAML_ERR_STATE, "gaml_set_graph has not been called");
  // an evaluation in flight updates the read state and the walk bookkeeping when it is finished: preparing another one
  // underneath it would score deltas against the wrong old walks
  if (ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is in flight: call gaml_eval_finish before preparing the next one");
  if (ctx->prepared) CU(cudaStreamSynchronize(ctx->stream));   // a prepared-but-abandoned evaluation: its staging copy may still read h_blob
  ctx->prepared = false;
  if (ctx->epoch + 1 >= 0x7fffffffu) return fail(ctx, GAML_ERR_STATE, "epoch counter exhausted (2^31 evaluations): recreate the context");
  WalkSet& ws = ctx->cur();
  const WalkSet* old_set = ctx->have_prev ? &ctx->prev() : nullptr;
  WalkDiff& diff = ctx->cur_diff;
  load_walks(ws, old_set, nodes, offs, n_walks, diff);   // aligns with the previous list, hashes only the walks that changed
  pt.lap(0);
  const int n_nodes = (int)ctx->node_len.size();
  // node ids and GetTotalLen (graph.cc:1966, int arithmetic like the reference): over the changed walks when the rest is
  // the previous evaluation's, else over all of them
  auto walk_len = [&](const WalkSet& w, int i, bool check, bool& bad) {
    unsigned t = 0;
    for (int64_t k = w.offs[i]; k < w.offs[i + 1]; k++) {
      const int x = w.nodes[(size_t)k];
      if (check && x >= n_nodes) { bad = true; return 0u; }
      t += (unsigned)(x < 0 ? -x : ctx->node_len[x]);
    }
    return t;
  };
  bool bad = false;
  unsigned tl_u = 0;
  if (diff.valid) {
    tl_u = (unsigned)ctx->prev_total_len;
    for (int i : diff.old_changed) tl_u -= walk_len(*old_set, i, false, bad);
    for (int i : diff.new_changed) tl_u += walk_len(ws, i, true, bad);
  } else {
    for (int i = 0; i < ws.n && !bad; i++) tl_u += walk_len(ws, i, true, bad);
  }
  const int total_len = (int)tl_u;
  if (bad) return fail(ctx, GAML_ERR_ARG, "walk references a node outside the graph");
  ctx->cur_total_len = total_len;
  int rc = commit(ctx);
  if (rc != GAML_OK) return rc;
  const bool list_same = old_set && diff.valid && diff.old_changed.empty() && diff.new_changed.empty() && ws.n == old_set->n;
  if (!list_same) ctx->list_gen++;
  bool all_full = true;
  for (auto& rsp : ctx->sets) all_full &= !(rsp->cfg.kind == GAML_KIND_PAIRED && rsp->has_state);
  ctx->n_patch = ctx->n_skip = 0;
  pt.lap(1);
  // labels of this list relative to the resident base blob's list (patched full evaluation): followed through every
  // evaluation, full or incremental, for as long as the lists align and stay within a few walks of the base
  if (ctx->full_cache_gen != ctx->cache_gen || !ctx->full_blob_valid) ctx->base_valid = false;
  ListTrack& track = ctx->track[ctx->cur_set];
  track.valid = false;
  if (ctx->base_valid && old_set && diff.valid) {
    const ListTrack& tp = ctx->track[ctx->cur_set ^ 1];
    if (tp.valid && tp.base_gen == ctx->base_gen) {
      const char* why = nullptr;
      track.valid = derive_track(ctx->base_ws, ctx->base_g, ctx->base_s, kMaxPatchWalks, *old_set, ws, diff, tp, track, &why);
      if (!track.valid && patch_debug()) fprintf(stderr, "[gaml_b200] full patch: %s\n", why ? why : "?");
    }
    else if (patch_debug()) fprintf(stderr, "[gaml_b200] full patch: previous list not tracked (valid %d)\n", (int)tp.valid);
  } else if (patch_debug()) {
    fprintf(stderr, "[gaml_b200] full patch: no tracking (base %d, prev %d, diff %d)\n", (int)ctx->base_valid, old_set != nullptr, (int)diff.valid);
  }
  pt.lap(2);
  if (all_full && ctx->full_blob_valid && ctx->full_list_gen == ctx->list_gen && ctx->full_cache_gen == ctx->cache_gen &&
      ctx->full_plan.size() == ctx->sets.size()) {
    // the same walks, the same cache, every paired set from scratch: the blob of the last such evaluation is still on the device
    ctx->plan = ctx->full_plan;
    ctx->n_updates = ctx->full_n_updates;
    ctx->upd_off = ctx->full_upd_off;
    ctx->blob_bytes = ctx->full_blob_bytes;
    ctx->blob_dev = ctx->d_full_blob.as<char>();
    for (size_t s = 0; s < ctx->sets.size(); s++) {
      ReadSetState& rt = *ctx->sets[s];
      if (rt.cfg.kind == GAML_KIND_PACBIO) continue;
      const int two_len = two_len_of(ctx->plan[s].total_len);
      if (!rt.pstar_valid || rt.pstar_two_len != two_len) {
        rt.h_pstar.assign(rt.h_thr.size(), 0.0);
        for (int li : rt.len_classes) rt.h_pstar[li] = floor_pstar(rt.h_thr[li], (double)two_len);
        rt.pstar_two_len = two_len;
        rt.pstar_valid = true;
      }
    }
    CU(ctx->d_flags.reserve(flags_words(ctx->sets.size()) * sizeof(unsigned long long), 0, true, ctx->stream));
    for (auto& rsp : ctx->sets) CU(rsp->d_ovf_list.reserve((size_t)ctx->ovf_cap * 4, 0, false, ctx->stream));
    CU(ctx->d_scratch.reserve(ctx->scratch_entries * sizeof(Plc), 0, false, ctx->stream));
    ctx->stats.last_h2d_bytes = 0;
    ctx->full_blob_reuses++;
    ctx->stats.full_reuse_evals++;
    ctx->epoch++;
    ctx->prepared = true;
    ctx->launched = false;
    pt.lap(3);
    pt.done();
    return GAML_OK;
  }
  if (all_full && ctx->patch_enabled && ctx->base_valid && track.valid && track.base_gen == ctx->base_gen &&
      ctx->full_plan.size() == ctx->sets.size()) {
    // a full evaluation of a list a few walks away from the base list: the resident blob + the updates of those walks' keys
    rc = prepare_full_patch(ctx, total_len);
    if (rc < 0) return rc;
    if (rc == 1) {
      ctx->stats.full_patch_evals++;
      ctx->epoch++;
      ctx->prepared = true;
      ctx->launched = false;
      pt.lap(3);
      pt.done();
      return GAML_OK;
    }
    ctx->n_patch = ctx->n_skip = 0;
  }
  const size_t n_sets = ctx->sets.size();
  // Full evaluations of paired sets number their walks with gaps (labels) when the context allows patched re-scores later.
  bool spaced = all_full && ctx->patch_enabled && n_sets > 0 && ws.n > 0;
  for (auto& rsp : ctx->sets) spaced &= rsp->cfg.kind == GAML_KIND_PAIRED && !rsp->penalty && rsp->n_mates == 2;
  int lab_g = 3, lab_s = 0;
  if (spaced) {
    int bits = 0;
    while (((uint64_t)(ws.n + 2) << lab_g) >> bits) bits++;
    if (32 - (bits + 1) >= 12) bits++;   // (room for walks appended behind the base list's labels)
    lab_s = std::min(32 - bits, 20);
    if (lab_s < 6) spaced = false;
  }
  bool seg_overflow = false;
  std::vector<SlotUpdate>& updates = ctx->h_updates;
  std::vector<std::vector<Occ>>& occs = ctx->h_occs;
  std::vector<std::vector<TouchRange>>& touches = ctx->h_touches;
  std::vector<std::vector<TouchRange>>& mtouches = ctx->h_mtouches;
  std::vector<std::vector<std::vector<int>>> cov_cs;   // per penalty set: contig starts of every touched walk
 for (;;) {   // (a second round only when a walk has more lookups than a label's enumeration range: dense numbers then)
  // host-side generation of the per-key stamp tables (group_occurrences). The device epoch (slot liveness, result lines)
  // advances only at the end, once this function can no longer fail: the ranks of a multi-GPU job stay in step even when
  // one of them rejects a walk set.
  if (++ctx->stamp_gen == 0) {
    for (MateStore* st : ctx->stores) std::fill(st->key_stamp.begin(), st->key_stamp.end(), 0u);
    ctx->stamp_gen = 1;
  }

  ctx->plan.assign(n_sets, SetPlan());
  updates.clear();
  occs.resize(ctx->stores.size());
  ctx->h_ob.resize(ctx->stores.size());
  touches.resize(n_sets);
  for (auto& t : touches) t.clear();
  mtouches.resize(n_sets);
  for (auto& t : mtouches) t.clear();
  for (auto& o : ctx->h_ob) o.reset();
  ctx->h_walks.clear();
  cov_cs.assign(n_sets, {});
  seg_overflow = false;
  if (spaced) {
    ctx->base_mkeys.assign(n_sets, {});
    for (MateStore* st : ctx->stores) st->base_slot.assign(st->keys.size(), -1);
  }

  // GetChanges (graph.cc:1745-1764) is the same for every paired set with state (they all follow the last evaluated
  // walks). Fast path: the difference is confined to the region where the new walk list departs from the previous one
  // and the erased walks are ordered by the container's rule; otherwise the reference's own container is built
  // (walk_set.h; tests/cpp/test_walk_changes.cc checks the one against the other).
  std::vector<WalkView>& erased = ctx->h_changes.erased;
  std::vector<WalkView>& added = ctx->h_changes.added;
  bool changes_done = false;
  auto get_changes = [&]() {
    if (changes_done) return;
    changes_done = true;
    const WalkSet& old = ctx->prev();
    if (ctx->fast_changes && get_changes_fast(old, ws, diff, ctx->prev_counts, ctx->h_changes)) {
      ctx->stats.fast_change_evals++;
      return;
    }
    ctx->pool.release();
    get_changes_reference(old, ws, ctx->h_changes, ctx->h_refs, &ctx->pool);
  };

  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    SetPlan& sp = ctx->plan[s];
    sp.grid = 0;
    if (rs.cfg.kind == GAML_KIND_PAIRED) {
      OccBuilder* ob[2] = {&ctx->h_ob[rs.mate[0].table_index], &ctx->h_ob[rs.mate[1].table_index]};
      sp.full = !rs.has_state;
      if (!sp.full) get_changes();
      sp.grid = score_grid(sp.full ? kGridPairedFull : kGridPairedTotal, rs.n_local, ctx->sm_count);
      sp.n_erased = sp.full ? 0 : (int)erased.size();
      int ord = 0;
      std::vector<TouchRange>* tp = sp.full ? nullptr : &touches[s];
      std::vector<int> cs;
      if (sp.full) {
        for (int i = 0; i < ws.n; i++) {
          int lab = ord++;
          uint32_t seg0 = 0;
          if (spaced) {
            lab = (i + 1) << lab_g;
            seg0 = (uint32_t)lab << lab_s;
            ob[0]->next_seg = ob[1]->next_seg = seg0;
          }
          flatten_paired_walk(ctx, rs, ws.view(i), lab, ob, sp, tp, rs.penalty ? &cs : nullptr);
          if (spaced && (ob[0]->next_seg - seg0 >= (1u << lab_s) || ob[1]->next_seg - seg0 >= (1u << lab_s))) seg_overflow = true;
          if (rs.penalty) cov_cs[s].push_back(cs);
        }
      } else {
        for (const WalkView& c : erased) {
          flatten_paired_walk(ctx, rs, c, ord++, ob, sp, tp, rs.penalty ? &cs : nullptr);
          if (rs.penalty) cov_cs[s].push_back(cs);
        }
        for (const WalkView& c : added) {
          flatten_paired_walk(ctx, rs, c, ord++, ob, sp, tp, rs.penalty ? &cs : nullptr);
          if (rs.penalty) cov_cs[s].push_back(cs);
        }
      }
      sp.total_len = total_len;
      {
        const int tl1 = total_len == 0 ? 1 : total_len;
        sp.delta_only = ctx->running_total && !sp.full && rs.total_valid && rs.total_two_len == (int)(2u * (unsigned)tl1);
      }
      const size_t u0 = updates.size();
      for (int m = 0; m < 2; m++)
        group_occurrences(*ob[m], rs.mate[m], ctx->stamp_gen, updates, occs[rs.mate[m].table_index], spaced);
      if (sp.full) {   // records under keys that occur several times: enumerated by the multi pass, mate 1's ranges first
        std::vector<TouchRange>& mt = mtouches[s];
        for (int m = 0; m < 2; m++) {
          for (size_t u = u0; u < updates.size(); u++) {
            if (updates[u].n_occ < 2 || updates[u].store != rs.mate[m].table_index) continue;
            if (spaced) ctx->base_mkeys[s].push_back({m, updates[u].key});
            const KeyMeta& km = rs.mate[m].keys[updates[u].key];
            if (km.count) {
              mt.push_back(TouchRange{km.arena_off, km.count});
              sp.multi_records += km.count;
            }
          }
          if (m == 0) sp.n_mtouch1 = (int)mt.size();
        }
        sp.n_mtouch = (int)mt.size();
      }
      for (const TouchRange& t : touches[s]) sp.touch_records += t.count;
      sp.n_touch = (int)touches[s].size();
      sp.cgrid = sp.full && rs.class_begin[5] > 0 ? score_grid(kGridPairedComplex, rs.class_begin[5], ctx->sm_count) : 0;
    } else {
      OccBuilder& ob = ctx->h_ob[rs.mate[0].table_index];
      sp.full = true;
      if (ctx->h_walks.empty() && ws.n > 0)   // single / pacbio sets re-read every walk: materialise them once per evaluation
        for (int i = 0; i < ws.n; i++) ctx->h_walks.push_back(ws.walk(i));
      if (rs.cfg.kind == GAML_KIND_SINGLE) flatten_single(ctx, rs, ctx->h_walks.data(), ws.n, ob, sp);
      else flatten_pacbio(ctx, rs, ctx->h_walks.data(), ws.n, ob, sp);
      group_occurrences(ob, rs.mate[0], ctx->stamp_gen, updates, occs[rs.mate[0].table_index]);
      sp.grid = score_grid(rs.cfg.kind == GAML_KIND_SINGLE ? kGridSingleFull : kGridPacbioFull, rs.n_local, ctx->sm_count);
      sp.cgrid = rs.cfg.kind == GAML_KIND_SINGLE && rs.n_complex > 0 ? score_grid(kGridSingleComplex, rs.n_complex, ctx->sm_count) : 0;
    }
  }

  if (!(spaced && seg_overflow)) break;
  spaced = false;
 }
  pt.lap(4);

  // ---- pack the staging blob: [updates][occ per store][touch + prefix per set][set_begin] -----
  auto align16 = [](size_t x) { return (x + 15) & ~size_t(15); };
  size_t off = 0;
  ctx->upd_off = off;
  off = align16(off + updates.size() * sizeof(SlotUpdate));
  std::vector<size_t> occ_off(ctx->stores.size());
  for (size_t i = 0; i < ctx->stores.size(); i++) {
    occ_off[i] = off;
    off = align16(off + occs[i].size() * sizeof(Occ));
  }
  for (size_t s = 0; s < n_sets; s++) {
    SetPlan& sp = ctx->plan[s];
    ReadSetState& rs = *ctx->sets[s];
    for (int m = 0; m < rs.n_mates; m++) sp.occ_off[m] = occ_off[rs.mate[m].table_index];
    sp.touch_off = off;
    off = align16(off + touches[s].size() * sizeof(TouchRange));
    sp.prefix_off = off;
    off = align16(off + (touches[s].size() + 1) * sizeof(uint32_t));
    sp.mtouch_off = off;
    off = align16(off + mtouches[s].size() * sizeof(TouchRange));
    sp.mprefix_off = off;
    off = align16(off + (mtouches[s].size() + 1) * sizeof(uint32_t));
    if (rs.cfg.kind != GAML_KIND_PACBIO) {
      sp.pstar_off = off;
      off = align16(off + std::max<size_t>(rs.h_thr.size(), 1) * sizeof(double));
    }
    if (rs.pb_penalty) {
      sp.pb_seeds_off = off;
      off = align16(off + rs.h_pb_seeds.size() * 16);
      sp.pb_occ_off = off;
      off = align16(off + rs.h_pb_occ.size() * 16);
      sp.pb_prefix_off = off;
      off = align16(off + (rs.h_pb_occ.size() + 1) * 4);
      sp.pb_len_off = off;
      off = align16(off + std::max<size_t>(rs.h_pb_walk_len.size(), 1) * 4);
      uint64_t recs = 0;
      for (const int4& o : rs.h_pb_occ) recs += (uint32_t)o.w;
      const uint64_t cap = rs.h_pb_seeds.size() + recs + 16;
      if (cap > 0x3fffffffull) return fail(ctx, GAML_ERR_CAPACITY, "too many PacBio coverage intervals for one evaluation");
      sp.pb_cap = (uint32_t)cap;
    }
    if (rs.penalty) {
      sp.n_cov_walks = (int)cov_cs[s].size();
      sp.n_type1 = 0;
      for (auto& v : cov_cs[s]) sp.n_type1 += (int)v.size();
      sp.type1_off = off;
      off = align16(off + (size_t)sp.n_type1 * 8);
      sp.csbegin_off = off;
      off = align16(off + ((size_t)sp.n_cov_walks + 1) * 4);
      sp.cs_off = off;
      off = align16(off + (size_t)sp.n_type1 * 4);
      sp.evcount_off = off;
      off = align16(off + 4);
      const uint64_t cap = (uint64_t)sp.n_type1 + 4ull * (uint64_t)sp.records1 + 4096ull;
      if (cap > 0x7fffffffull) return fail(ctx, GAML_ERR_CAPACITY, "too many coverage events for one evaluation");
      sp.ev_cap = (uint32_t)cap;
    }
  }
  ctx->blob_bytes = off;
  rc = ensure_pinned(ctx, off);
  if (rc != GAML_OK) return rc;
  char* hb = static_cast<char*>(ctx->h_blob);
  if (!updates.empty()) memcpy(hb + ctx->upd_off, updates.data(), updates.size() * sizeof(SlotUpdate));
  for (size_t i = 0; i < ctx->stores.size(); i++)
    if (!occs[i].empty()) memcpy(hb + occ_off[i], occs[i].data(), occs[i].size() * sizeof(Occ));
  for (size_t s = 0; s < n_sets; s++) {
    SetPlan& sp = ctx->plan[s];
    if (!touches[s].empty()) memcpy(hb + sp.touch_off, touches[s].data(), touches[s].size() * sizeof(TouchRange));
    uint32_t* pre = reinterpret_cast<uint32_t*>(hb + sp.prefix_off);
    uint64_t acc = 0;
    for (size_t t = 0; t < touches[s].size(); t++) {
      pre[t] = (uint32_t)acc;
      acc += touches[s][t].count;
    }
    if (acc > 0xffffffffull) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^32 touched records in one evaluation");
    pre[touches[s].size()] = (uint32_t)acc;
    if (!mtouches[s].empty()) memcpy(hb + sp.mtouch_off, mtouches[s].data(), mtouches[s].size() * sizeof(TouchRange));
    uint32_t* mpre = reinterpret_cast<uint32_t*>(hb + sp.mprefix_off);
    uint64_t macc = 0;
    for (size_t t = 0; t < mtouches[s].size(); t++) {
      mpre[t] = (uint32_t)macc;
      macc += mtouches[s][t].count;
    }
    if (macc > 0xffffffffull) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^32 records under repeated keys in one evaluation");
    mpre[mtouches[s].size()] = (uint32_t)macc;
    if (ctx->sets[s]->cfg.kind != GAML_KIND_PACBIO) {   // floor tests at this evaluation's total length (acc_term, kernels.cu)
      ReadSetState& rt = *ctx->sets[s];
      const int two_len = two_len_of(sp.total_len);
      if (!rt.pstar_valid || rt.pstar_two_len != two_len) {
        rt.h_pstar.assign(rt.h_thr.size(), 0.0);
        for (int li : rt.len_classes) rt.h_pstar[li] = floor_pstar(rt.h_thr[li], (double)two_len);
        rt.pstar_two_len = two_len;
        rt.pstar_valid = true;
      }
      if (!rt.h_pstar.empty()) memcpy(hb + sp.pstar_off, rt.h_pstar.data(), rt.h_pstar.size() * sizeof(double));
    }
    if (ctx->sets[s]->pb_penalty) {
      ReadSetState& rp = *ctx->sets[s];
      if (!rp.h_pb_seeds.empty()) memcpy(hb + sp.pb_seeds_off, rp.h_pb_seeds.data(), rp.h_pb_seeds.size() * 16);
      if (!rp.h_pb_occ.empty()) memcpy(hb + sp.pb_occ_off, rp.h_pb_occ.data(), rp.h_pb_occ.size() * 16);
      uint32_t* pp = reinterpret_cast<uint32_t*>(hb + sp.pb_prefix_off);
      uint32_t run = 0;
      for (size_t t = 0; t < rp.h_pb_occ.size(); t++) {
        pp[t] = run;
        run += (uint32_t)rp.h_pb_occ[t].w;
      }
      pp[rp.h_pb_occ.size()] = run;
      if (!rp.h_pb_walk_len.empty()) memcpy(hb + sp.pb_len_off, rp.h_pb_walk_len.data(), rp.h_pb_walk_len.size() * 4);
    }
    if (ctx->sets[s]->penalty) {
      unsigned long long* keys = reinterpret_cast<unsigned long long*>(hb + sp.type1_off);
      int* csb = reinterpret_cast<int*>(hb + sp.csbegin_off);
      int* csv = reinterpret_cast<int*>(hb + sp.cs_off);
      int k = 0;
      for (size_t w = 0; w < cov_cs[s].size(); w++) {
        csb[w] = k;
        for (int p : cov_cs[s][w]) {
          keys[k] = ((unsigned long long)(uint32_t)w << 33) | ((unsigned long long)((uint32_t)p ^ 0x80000000u) << 1);
          csv[k] = p;
          k++;
        }
      }
      csb[cov_cs[s].size()] = k;
      *reinterpret_cast<uint32_t*>(hb + sp.evcount_off) = (uint32_t)k;
      ctx->sets[s]->h_type1.assign(keys, keys + k);
    }
  }
  ctx->n_updates = (int)updates.size();

  pt.lap(5);
  DevBuf& dst_blob = all_full ? ctx->d_full_blob : ctx->d_blob;
  CU(dst_blob.reserve(std::max<size_t>(off + (all_full ? kPatchReserve : 0), (size_t)1 << 18), 0, false, ctx->stream));   // (generous: growing a device buffer frees the old
                                                                                         //  one, which waits for the whole device)
  ctx->blob_dev = dst_blob.as<char>();
  CU(ctx->d_flags.reserve(flags_words(n_sets) * sizeof(unsigned long long), 0, true, ctx->stream));
  CU(ctx->d_scratch.reserve(ctx->scratch_entries * sizeof(Plc), 0, false, ctx->stream));
  if (ctx->h_out_cap < (n_sets + 1) * kResultStride) {
    if (ctx->h_out) {
      CU(cudaStreamSynchronize(ctx->stream));
      cudaFreeHost(ctx->h_out);
    }
    ctx->h_out = nullptr;
    const size_t cap = (n_sets + 1) * kResultStride;
    CU(cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_out), cap * sizeof(double), cudaHostAllocMapped));
    memset(ctx->h_out, 0, cap * sizeof(double));
    CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->d_out_mapped), ctx->h_out, 0));
    ctx->h_out_cap = cap;
  }
  for (auto& rsp : ctx->sets) CU(rsp->d_ovf_list.reserve((size_t)ctx->ovf_cap * 4, 0, false, ctx->stream));   // grows after a capacity error
  CU(cudaMemcpyAsync(ctx->blob_dev, ctx->h_blob, off, cudaMemcpyHostToDevice, ctx->stream));
  ctx->stats.last_h2d_bytes = (int64_t)off;
  if (all_full) {   // (an incremental evaluation stages into d_blob: the resident full blob stays as it is)
    ctx->full_blob_valid = true;
    ctx->full_plan = ctx->plan;
    ctx->full_n_updates = ctx->n_updates;
    ctx->full_upd_off = ctx->upd_off;
    ctx->full_blob_bytes = ctx->blob_bytes;
    ctx->full_list_gen = ctx->list_gen;
    ctx->full_cache_gen = ctx->cache_gen;
    ctx->base_valid = spaced;
    if (spaced) {   // this list is the base of later patched evaluations: keep its walks and its updates on the host
      ctx->base_gen++;
      ctx->base_g = lab_g;
      ctx->base_s = lab_s;
      ctx->base_ws.n = ws.n;
      ctx->base_ws.nodes = ws.nodes;
      ctx->base_ws.offs = ws.offs;
      ctx->base_ws.hash = ws.hash;
      ctx->full_updates.swap(updates);
      ctx->full_occs.swap(occs);
      track.valid = true;
      track.base_gen = ctx->base_gen;
      track.removed.clear();
      track.n_added = 0;
      track.label.resize((size_t)ws.n);
      for (int i = 0; i < ws.n; i++) track.label[(size_t)i] = (uint32_t)(i + 1) << lab_g;
    }
  }
  ctx->epoch++;
  ctx->prepared = true;
  ctx->launched = false;
  pt.lap(6);
  pt.done();
  return GAML_OK;
}


// Result line of (rank, set) for the evaluation with this epoch: two generations (epoch parity) so that a rank that is
// one evaluation ahead does not overwrite a line a slower rank has yet to read.
size_t exch_line(const gaml_ctx* ctx, int rank, size_t s) {
  return ((size_t)(ctx->epoch & 1u) * (size_t)ctx->exch_world + (size_t)rank) * GAML_EXCHANGE_MAX_SETS + s;
}

// The per-evaluation result lines go through NCCL only when no kernel-fused exchange is attached; the communicator also
// serves the candidate batches (gaml_calc_prob_batch_gathered) next to either of those.
bool nccl_lines(const gaml_ctx* ctx) { return ctx->nccl_on && !ctx->peer_on && !ctx->exch_host; }

ScoreParams make_params(gaml_ctx* ctx, size_t s) {
  ReadSetState& rs = *ctx->sets[s];
  const SetPlan& sp = ctx->plan[s];
  char* blob = ctx->blob_dev;
  ScoreParams P{};
  for (int m = 0; m < rs.n_mates; m++) {
    MateStore& st = rs.mate[m];
    P.m[m].first = st.first.p;
    P.m[m].rows = st.rows.p;
    P.m[m].rowptr = st.rowptr.as<uint32_t>();
    P.m[m].crows = st.crows.p;
    P.m[m].cptr = st.cptr.as<uint32_t>();
    P.m[m].slots_a = st.slots_a.as<SlotA>();
    P.m[m].slots_b = st.slots_b.as<SlotB>();
    P.m[m].n_keys = (int)st.keys.size();
    P.m[m].occ = reinterpret_cast<const Occ*>(blob + sp.occ_off[m]);
    P.m[m].pow_match = st.d_pow_match.as<double>();
    P.m[m].pow_mismatch = st.d_pow_mismatch.as<double>();
  }
  P.lens = rs.d_lens.as<uint32_t>();
  P.pairs = rs.pairs_ok ? rs.d_pairs.p : nullptr;
  P.comb = rs.pairs_ok && rs.comb_ok ? rs.d_comb.p : nullptr;
  P.lens_uniform = rs.lens_uniform ? 1 : 0;
  P.uniform_ll = rs.uniform_ll;
  for (int m = 0; m < 2; m++) P.uni_prob[m] = rs.lens_uniform && rs.d_uni_prob[m].p ? rs.d_uni_prob[m].as<double>() : nullptr;
  P.tq = rs.lens_uniform && rs.tq_shift > 0 ? rs.d_tq.p : nullptr;
  P.tq_shift = rs.tq_shift;
  P.fast = rs.fast_ok && rs.pairs_ok && rs.comb_ok ? rs.d_fast.p : nullptr;
  P.xlist = rs.d_xlist.as<uint32_t>();
  P.n_cross = rs.fast_ok ? rs.n_cross : 0;
  P.n_tier1 = rs.perm_valid ? rs.n_fast : rs.n_local;
  P.dirty = rs.n_appx > 0 ? rs.d_dirty.as<uint32_t>() : nullptr;
  P.appx_list = rs.d_appx.as<uint32_t>();
  P.n_appx = rs.n_appx;
  P.ins_tab = rs.d_ins.as<double>();
  P.ins_n = rs.ins_n;
  P.pstar_tab = reinterpret_cast<const double*>(blob + sp.pstar_off);
  P.qthr_tab = rs.d_qthr.as<long long>();
  if (rs.lens_uniform && rs.pstar_valid) {
    const size_t li = (size_t)(rs.uniform_ll & 0xffff) + (size_t)(rs.uniform_ll >> 16);
    P.uni_pstar = rs.h_pstar[li];
    P.uni_qthr = rs.h_qthr[li];
  }
  P.floor_a = rs.floor_a;
  P.floor_b = rs.floor_b;
  P.values = rs.d_values.as<double>();
  P.epoch = ctx->epoch;
  P.n_erased = sp.n_erased;
  P.n_reads = rs.n_local;
  P.two_len = two_len_of(sp.total_len);                   // the reference's int expression 2*total_len, graph.cc:1500-1505
  P.ql = rs.cfg.kind == GAML_KIND_PACBIO ? 0 : fix_log_host((double)P.two_len);   // PacBio: - log 2L is the host's, graph.cc:3087
  unsigned long long* fl = ctx->d_flags.as<unsigned long long>();
  P.scratch_cursor = fl;
  P.error_flag = reinterpret_cast<uint32_t*>(fl + 1);
  P.ovf_count = reinterpret_cast<uint32_t*>(fl + 2 + s);
  P.ovf_list = rs.d_ovf_list.as<uint32_t>();
  P.ovf_cap = ctx->ovf_cap;
  P.scratch = ctx->d_scratch.as<Plc>();
  P.scratch_cap = ctx->scratch_entries;
  P.complex_list = rs.d_complex.as<uint32_t>();
  P.clens = rs.d_clens.as<uint32_t>();
  P.cdesc = rs.d_cdesc.p;
  memcpy(P.class_begin, rs.class_begin, sizeof(P.class_begin));
  P.n_complex = rs.n_complex;
  P.n_main = rs.class_begin[5];
  memcpy(P.cbase, rs.cbase, sizeof(P.cbase));
  P.t2pack = rs.t2pack_ok ? rs.d_t2pack.p : nullptr;
  memcpy(P.t2base, rs.t2base, sizeof(P.t2base));
  P.arena2 = rs.n_mates == 2 ? rs.mate[1].arena.as<ArenaShort>() : nullptr;
  P.mtouch = reinterpret_cast<const TouchRange*>(blob + sp.mtouch_off);
  P.mtouch_prefix = reinterpret_cast<const uint32_t*>(blob + sp.mprefix_off);
  P.n_mtouch = sp.n_mtouch;
  P.n_mtouch1 = sp.n_mtouch1;
  const size_t ns = std::max<size_t>(ctx->sets.size(), 1);
  P.ticket = reinterpret_cast<uint32_t*>(fl + 2 + ns + s);
  P.ticket2 = reinterpret_cast<uint32_t*>(fl + 2 + 2 * ns + s);
  P.done = reinterpret_cast<uint32_t*>(fl + 2 + 3 * ns + s);
  P.tile_counter = reinterpret_cast<uint32_t*>(fl + 2 + 4 * ns + 4 * s);
  P.accum = fl + 2 + 8 * ns + s * kAccumStride;
  P.chain_first = 1;
  P.finish_here = 0;
  P.out = ctx->exch_dev ? ctx->exch_dev + exch_line(ctx, ctx->exch_rank, s) * kResultStride : ctx->d_out_mapped + s * kResultStride;
  if (ctx->peer_on) {
    P.peer_bufs = ctx->d_peer_table.as<unsigned long long*>();
    P.peer_world = ctx->peer_world;
    P.peer_line = (uint32_t)(((size_t)(ctx->epoch & 1u) * (size_t)ctx->peer_world + (size_t)ctx->peer_rank) * GAML_EXCHANGE_MAX_SETS + s);
  }
  if (nccl_lines(ctx)) P.part_out = ctx->d_part.as<double>() + s * kResultStride;
  P.timeline = ctx->timeline ? ctx->d_timeline.as<unsigned long long>() : nullptr;
  P.state_acc = rs.cfg.kind == GAML_KIND_PAIRED ? rs.d_state_acc.as<unsigned long long>() : nullptr;
  P.state_add = sp.delta_only ? 1 : 0;
  P.delta_only = sp.delta_only ? 1 : 0;
  P.log_tab = ctx->d_logtab.p;
  if (rs.penalty) {
    P.ev_keys = rs.d_ev.as<unsigned long long>();
    P.ev_count = reinterpret_cast<uint32_t*>(P.accum + 7);   // spare accumulator word of the set
    P.ev_cap = sp.ev_cap;
    P.cov_thr = rs.d_cov_thr.as<double>();
  }
  P.arena1 = rs.mate[0].arena.as<ArenaShort>();
  P.touch = reinterpret_cast<const TouchRange*>(blob + sp.touch_off);
  P.touch_prefix = reinterpret_cast<const uint32_t*>(blob + sp.prefix_off);
  P.n_touch = sp.n_touch;
  P.stamp = rs.d_stamp.as<uint32_t>();
  return P;
}

// Submits the recorded kernel chain of one evaluation. Steady state: the chain's CUDA graph exists (same kernels in
// the same order, with their programmatic-dependent-launch edges) — its kernel nodes get this evaluation's grids and
// parameter blocks and the graph goes to the device in one submission, instead of one driver call per kernel with the
// device idling in between. First time a chain shape is seen: captured from the stream while it is issued.
int replay_chain(gaml_ctx* ctx, LaunchList& list) {
  cudaStream_t st = ctx->stream;
  const bool timed = ctx->timed;   // the evaluation's two events become nodes of the graph: pure device time
  uint64_t key = 1469598103934665603ull ^ (timed ? 0x9e3779b97f4a7c15ull : 0ull);
  for (int i = 0; i < list.n; i++) {
    const uint64_t v[3] = {(uint64_t)(uintptr_t)list.item[i].func, (uint64_t)list.item[i].pdl, (uint64_t)list.item[i].block};
    for (uint64_t x : v) key = (key ^ x) * 1099511628211ull;
  }
  auto it = ctx->graphs.find(key);
  if (it == ctx->graphs.end()) {
    gaml_ctx::GraphEntry ge;
    CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    // (cudaEventRecordExternal: a real event-record node; a plain record inside a capture is only a dependency marker)
    cudaError_t err = timed ? cudaEventRecordWithFlags(ctx->ev[0], st, cudaEventRecordExternal) : cudaSuccess;
    for (int i = 0; i < list.n && err == cudaSuccess; i++) {
      err = issue_launch(list.item[i], st);
      if (err != cudaSuccess) break;
      cudaStreamCaptureStatus status;
      const cudaGraphNode_t* deps = nullptr;
      size_t n_deps = 0;
      err = cudaStreamGetCaptureInfo_v3(st, &status, nullptr, nullptr, &deps, nullptr, &n_deps);
      if (err == cudaSuccess && (status != cudaStreamCaptureStatusActive || n_deps != 1)) err = cudaErrorUnknown;
      if (err == cudaSuccess) ge.nodes.push_back(deps[0]);
    }
    if (err == cudaSuccess && timed) err = cudaEventRecordWithFlags(ctx->ev[3], st, cudaEventRecordExternal);
    cudaGraph_t graph = nullptr;
    const cudaError_t end_err = cudaStreamEndCapture(st, &graph);
    if (err == cudaSuccess) err = end_err;
    if (err == cudaSuccess) err = cudaGraphInstantiate(&ge.exec, graph, 0);
    ge.graph = graph;   // kept: the node handles used for the per-evaluation parameter updates belong to it
    if (err != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      // graphs unavailable for this chain: issue it directly from now on
      cudaGetLastError();
      ctx->use_graphs = false;
      if (timed) CU(cudaEventRecord(ctx->ev[0], st));
      for (int i = 0; i < list.n; i++) CU(issue_launch(list.item[i], st));
      if (timed) CU(cudaEventRecord(ctx->ev[3], st));
      return GAML_OK;
    }
    it = ctx->graphs.emplace(key, std::move(ge)).first;
  } else {
    for (int i = 0; i < list.n; i++) {
      const PendingLaunch& pl = list.item[i];
      cudaKernelNodeParams np{};
      np.func = const_cast<void*>(pl.func);
      np.gridDim = dim3(pl.grid);
      np.blockDim = dim3(pl.block);
      np.sharedMemBytes = 0;
      np.kernelParams = const_cast<void**>(pl.arg_ptrs);
      np.extra = nullptr;
      CU(cudaGraphExecKernelNodeSetParams(it->second.exec, it->second.nodes[i], &np));
    }
  }
  CU(cudaGraphLaunch(it->second.exec, st));
  return GAML_OK;
}

// ---- a collective library as the exchange (gaml_nccl_exchange_init) -------------------------------------------------
// NCCL is bound at run time (dlopen: the copy the host program has loaded already, else libnccl.so.2), so the library
// has no link-time dependency on it.
struct NcclId { char bytes[128]; };
struct NcclApi {
  int (*get_unique_id)(NcclId*) = nullptr;
  int (*comm_init_rank)(void**, int, NcclId, int) = nullptr;
  int (*all_reduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*comm_destroy)(void*) = nullptr;
  const char* (*get_error_string)(int) = nullptr;
  void* lib = nullptr;
};
NcclApi* nccl_api(std::string* why) {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW);
    if (lib) {
      api.get_unique_id = reinterpret_cast<int (*)(NcclId*)>(dlsym(lib, "ncclGetUniqueId"));
      api.comm_init_rank = reinterpret_cast<int (*)(void**, int, NcclId, int)>(dlsym(lib, "ncclCommInitRank"));
      api.all_reduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(dlsym(lib, "ncclAllReduce"));
      api.comm_destroy = reinterpret_cast<int (*)(void*)>(dlsym(lib, "ncclCommDestroy"));
      api.get_error_string = reinterpret_cast<const char* (*)(int)>(dlsym(lib, "ncclGetErrorString"));
      if (api.get_unique_id && api.comm_init_rank && api.all_reduce && api.comm_destroy) api.lib = lib;
    }
  }
  if (!api.lib && why) *why = "NCCL (libnccl.so.2) is not available in this process";
  return api.lib ? &api : nullptr;
}

// One ncclAllReduce(sum, fp64) over the ranks' result lines of this evaluation (SURVEY §8e) on the evaluation's stream,
// then a one-thread-per-set kernel that re-seals the summed lines into host-mapped memory. Every field of a line is an
// integer far below 2^53 (integer part and 2^-40 units of the exact sum, counts), so the sums of doubles are exact.
int nccl_reduce_lines(gaml_ctx* ctx, int n_sets) {
  NcclApi* api = nccl_api(&ctx->error);
  if (!api) return GAML_ERR_STATE;
  const int rc = api->all_reduce(ctx->d_part.p, ctx->d_part_sum.p, (size_t)n_sets * kResultStride, /*ncclDouble*/ 8, /*ncclSum*/ 0,
                                 ctx->nccl_comm, ctx->stream);
  if (rc != 0) return fail(ctx, GAML_ERR_CUDA, std::string("ncclAllReduce: ") + (api->get_error_string ? api->get_error_string(rc) : "error"));
  launch_reduced_publish(ctx->d_part_sum.as<double>(), n_sets, ctx->epoch, ctx->d_gather_mapped, ctx->stream);
  CU(cudaGetLastError());
  return GAML_OK;
}

int nccl_all_reduce_doubles(gaml_ctx* ctx, double* buf, size_t count) {   // in place, on the context's stream
  NcclApi* api = nccl_api(&ctx->error);
  if (!api || !ctx->nccl_comm) return fail(ctx, GAML_ERR_STATE, "no NCCL communicator: gaml_nccl_exchange_init first");
  const int rc = api->all_reduce(buf, buf, count, /*ncclDouble*/ 8, /*ncclSum*/ 0, ctx->nccl_comm, ctx->stream);
  if (rc != 0) return fail(ctx, GAML_ERR_CUDA, std::string("ncclAllReduce: ") + (api->get_error_string ? api->get_error_string(rc) : "error"));
  return GAML_OK;
}

int ensure_gather_area(gaml_ctx* ctx, int world) {
  if (ctx->h_gather) return GAML_OK;
  (void)world;
  const size_t words = ((size_t)64 * GAML_EXCHANGE_MAX_SETS + 1) * kResultStride;   // up to 64 ranks + the flag line
  CU(cudaHostAlloc(reinterpret_cast<void**>(&ctx->h_gather), words * 8, cudaHostAllocMapped));
  memset(ctx->h_gather, 0, words * 8);
  CU(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ctx->d_gather_mapped), ctx->h_gather, 0));
  return GAML_OK;
}

int launch(gaml_ctx* ctx) {
  if (!ctx->prepared) return fail(ctx, GAML_ERR_STATE, "gaml_eval_launch without gaml_eval_prepare");
  cudaStream_t st = ctx->stream;
  const size_t n_sets = ctx->sets.size();
  if (ctx->timeline) {
    CU(ctx->d_timeline.reserve(kTimelineWords * 8, 0, true, st));
    CU(cudaMemsetAsync(ctx->d_timeline.p, 0, kTimelineWords * 8, st));
  }
  char* blob = ctx->blob_dev;
  int launches = 0;
  bool any_penalty = false;
  for (auto& rs : ctx->sets) {
    any_penalty |= rs->penalty || rs->pb_penalty;
    rs->tail_on_demand = false;
  }
  ctx->tail_timed = false;
  LaunchList chain;
  const bool record = ctx->use_graphs && !ctx->profile && !any_penalty && ctx->sets.size() <= 3;
  struct RecorderGuard { ~RecorderGuard() { set_launch_recorder(nullptr); } } recorder_guard;
  if (record) set_launch_recorder(&chain);
  else if (ctx->timed) CU(cudaEventRecord(ctx->ev[0], st));
  launch_apply_slots(reinterpret_cast<const SlotUpdate*>(blob + ctx->upd_off), ctx->n_updates,
                     reinterpret_cast<const SlotUpdate*>(blob + ctx->patch_upd_off), ctx->n_patch,
                     reinterpret_cast<const int32_t*>(blob + ctx->patch_skip_off), ctx->n_skip, ctx->d_tables.as<SlotA*>(),
                     ctx->d_tables.as<SlotB*>() + ctx->stores.size(), ctx->d_tables.as<SlotA*>() + 2 * ctx->stores.size(),
                     ctx->d_tables.as<const int32_t*>() + 3 * ctx->stores.size(),
                     ctx->stores.size() <= (size_t)kInlineStores ? &ctx->h_tables : nullptr, ctx->epoch, ctx->d_flags.as<unsigned long long>(),
                     (int)flags_words(n_sets), ctx->timeline ? ctx->d_timeline.as<unsigned long long>() : nullptr, st);
  launches++;
  int64_t records = 0, reads = 0, bytes = 0;
  bool any_full = false;
  const bool profile = ctx->profile;
  bool chained = true;   // the operation before the next kernel on `st` is a kernel of this evaluation's chain
  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    const SetPlan& sp = ctx->plan[s];
    ScoreParams P = make_params(ctx, s);
    const int og = overflow_grid(ctx->sm_count);
    records += sp.records;
    reads += rs.n_local;
    if (rs.penalty) {
      // event buffer: padding keys, then the host's contig-start events, then the running count
      CU(rs.d_ev.reserve((size_t)sp.ev_cap * 8, 0, false, st));
      CU(rs.d_ev_sorted.reserve((size_t)sp.ev_cap * 8, 0, false, st));
      CU(rs.d_ev_temp.reserve(std::max<size_t>(coverage_sort_temp_bytes(sp.ev_cap), 256), 0, false, st));
      CU(rs.d_bad.reserve(std::max<size_t>(sp.n_cov_walks, 1) * 4, 0, false, st));
      P.ev_keys = rs.d_ev.as<unsigned long long>();
      CU(cudaMemsetAsync(rs.d_ev.p, 0xff, (size_t)sp.ev_cap * 8, st));
      CU(cudaMemsetAsync(rs.d_bad.p, 0, std::max<size_t>(sp.n_cov_walks, 1) * 4, st));
      if (sp.n_type1) CU(cudaMemcpyAsync(rs.d_ev.p, blob + sp.type1_off, (size_t)sp.n_type1 * 8, cudaMemcpyDeviceToDevice, st));
      CU(cudaMemcpyAsync(P.ev_count, blob + sp.evcount_off, 4, cudaMemcpyDeviceToDevice, st));
      chained = false;
    }
    if (rs.cfg.kind == GAML_KIND_PAIRED) {
      if (sp.full) {
        const uint32_t n_multi = (uint32_t)sp.multi_records;
        // the streaming kernel ends a graph-replayed chain whose line only this host waits for first: the host segment
        // exchange (or none) — the peer and collective exchanges consume the line on the device
        rs.tail_on_demand = record && !ctx->peer_on && !nccl_lines(ctx) && !rs.keep_tail;
        if (rs.tail_on_demand) {
          rs.tail_params = P;
          rs.tail_grid = og;
        }
        launches += launch_paired_full(P, sp.grid, sp.cgrid, n_multi, og, ctx->sm_count, st, chained, profile, rs.ev0, rs.ev1,
                                       !rs.tail_on_demand);
        any_full = true;
        // DESIGN.md §4: 16 B per live record + packed lengths (4) + probs write (8) per pair (no probs read: fused)
        bytes += 16 * sp.records + 12 * (int64_t)rs.n_local;
      } else {
        launch_paired_delta(P, (uint32_t)sp.touch_records, sp.grid, og, ctx->sm_count, st, chained, profile, rs.ev0, rs.ev1);
        launches += sp.delta_only ? (sp.touch_records > 0 ? 2 : 1) : (sp.touch_records > 0 ? 3 : 1);
        // touched records (+ the O(R) pass when the total length changed: probs read (8) + packed lengths (4) per pair)
        bytes += 16 * sp.records + (sp.delta_only ? 0 : 12 * (int64_t)rs.n_local);
      }
      if (rs.penalty && rs.sharded) {
        chained = false;   // the sweep waits for every shard's events: gaml_penalty_import
      } else if (rs.penalty) {
        CU(launch_coverage(rs.d_ev.as<unsigned long long>(), rs.d_ev_sorted.as<unsigned long long>(), sp.ev_cap, rs.d_ev_temp.p,
                           rs.d_ev_temp.cap, reinterpret_cast<const int*>(blob + sp.csbegin_off),
                           reinterpret_cast<const int*>(blob + sp.cs_off), rs.cfg.step,
                           rs.cfg.insert_mean + 5 * rs.cfg.insert_std, rs.d_bad.as<int>(), ctx->sm_count, st));
        launches += 3;
        chained = false;
      } else {
        chained = !(profile && !sp.full);   // the delta wrapper ends with its e1 record when profiling
      }
    } else if (rs.cfg.kind == GAML_KIND_SINGLE) {
      launch_single_full(P, sp.grid, sp.cgrid, og, st, chained, profile, rs.ev0, rs.ev1);
      chained = true;
      launches += 2 + (sp.cgrid > 0);
      bytes += 16 * sp.records + 12 * (int64_t)rs.n_local;
    } else {
      launch_pacbio_full(P, sp.grid, og, st, chained, profile, rs.ev0, rs.ev1);
      chained = true;
      launches += 2;
      if (rs.pb_penalty) {
        const size_t cap = sp.pb_cap;
        CU(rs.d_pb_ikey.reserve(cap * 2 * 8, 0, false, st));
        CU(rs.d_pb_iend.reserve(cap * 2 * 4, 0, false, st));
        CU(rs.d_pb_pkey.reserve(cap * 4 * 8, 0, false, st));
        CU(rs.d_pb_packed.reserve(cap * 8, 0, false, st));
        CU(rs.d_pb_runmax.reserve(cap * 8, 0, false, st));
        CU(rs.d_pb_temp.reserve(std::max<size_t>(pacbio_coverage_temp_bytes(sp.pb_cap), 256), 0, false, st));
        CU(rs.d_pb_count.reserve(256, 0, true, st));
        CU(rs.d_bad.reserve(256, 0, true, st));
        PbCovParams C{};
        C.seeds = blob + sp.pb_seeds_off;
        C.n_seed = rs.sharded ? 0 : (int)rs.h_pb_seeds.size();   // (a shard emits its own alignments' intervals only)
        C.occ = blob + sp.pb_occ_off;
        C.occ_prefix = reinterpret_cast<const uint32_t*>(blob + sp.pb_prefix_off);
        C.n_occ = (int)rs.h_pb_occ.size();
        C.arena = rs.mate[0].arena.as<ArenaLong>();
        C.arena_pos = rs.mate[0].arena_pos.p;
        C.lens = rs.d_lens.as<uint32_t>();
        C.log_mismatch = log(rs.cfg.mismatch_prob);   // logdouble(double) = log, graph.h:448, logdouble.hpp:18
        C.log_match = log(rs.cfg.match_prob);
        C.ikey = rs.d_pb_ikey.as<unsigned long long>();
        C.iend = rs.d_pb_iend.as<int32_t>();
        C.pkey = rs.d_pb_pkey.as<unsigned long long>();
        C.count = rs.d_pb_count.as<uint32_t>();
        C.cap = sp.pb_cap;
        C.error_flag = P.error_flag;
        CU(launch_pacbio_coverage(C, rs.d_pb_packed.as<unsigned long long>(), rs.d_pb_runmax.as<unsigned long long>(),
                                  rs.d_pb_temp.p, rs.d_pb_temp.cap, reinterpret_cast<const int*>(blob + sp.pb_len_off),
                                  rs.cfg.step, rs.d_bad.as<int>(), ctx->sm_count, st, rs.sharded ? 1 : 0));
        launches += rs.sharded ? 1 : 6;
        chained = false;
      }
      bytes += 16 * sp.records + 16 * (int64_t)rs.n_local;
    }
  }
  if (ctx->peer_on && n_sets > 0) {
    // last kernel of the chain: wait for every rank's line of this evaluation in this rank's exchange buffer
    const unsigned long long* gen = ctx->d_peer_lines.as<unsigned long long>() +
                                    (size_t)(ctx->epoch & 1u) * (size_t)ctx->peer_world * GAML_EXCHANGE_MAX_SETS * kResultStride;
    launch_exchange_gather(gen, ctx->peer_world, (int)n_sets, GAML_EXCHANGE_MAX_SETS, ctx->epoch, ctx->d_gather_mapped,
                           ctx->d_gather_mapped + (size_t)ctx->peer_world * GAML_EXCHANGE_MAX_SETS * kResultStride,
                           ctx->exchange_timeout_ns, st);
    launches++;
  }
  if (record) {
    set_launch_recorder(nullptr);
    const int rc = replay_chain(ctx, chain);
    if (rc != GAML_OK) return rc;
  }
  if (!record && ctx->timed) CU(cudaEventRecord(ctx->ev[3], st));
  if (nccl_lines(ctx) && n_sets > 0) {
    const int rc = nccl_reduce_lines(ctx, (int)n_sets);
    if (rc != GAML_OK) return rc;
    launches++;
  }
  CU(cudaGetLastError());
  ctx->stats.kernel_launches += launches;
  ctx->stats.last_records_gathered = records;
  ctx->stats.last_reads_scanned = reads;
  ctx->stats.last_algorithmic_bytes = bytes;
  ctx->stats.last_was_full = any_full ? 1 : 0;
  for (size_t s = 0; s < n_sets; s++)
    if (ctx->plan[s].delta_only) ctx->stats.delta_only_evals++;
  ctx->launched = true;
  return GAML_OK;
}

// Waits for one 64-byte result line of this evaluation (flag word = epoch, checksum intact) and copies it out. With
// `pending`, a line whose flag word is pend_bits is accepted too, and *pending tells which of the two arrived.
int wait_line(gaml_ctx* ctx, const volatile uint64_t* line, uint64_t want_bits, double* dst, bool own, bool* pending = nullptr,
              uint64_t pend_bits = 0) {
  unsigned spins = 0;
  const auto t0 = std::chrono::steady_clock::now();
  for (;;) {
    uint64_t w[8];
    for (int j = 0; j < 8; j++) w[j] = line[j];
    uint64_t sum = kResultSeal;
    for (int j = 0; j < 7; j++) sum ^= w[j];
    const bool alt = pending && w[6] == pend_bits;
    if ((w[6] == want_bits || alt) && w[7] == sum) {
      memcpy(dst, w, sizeof(w));
      if (pending) *pending = alt;
      return GAML_OK;
    }
    cpu_relax();
    if ((++spins & 0x3fffu) == 0) {
      const cudaError_t q = cudaStreamQuery(ctx->stream);
      if (q != cudaSuccess && q != cudaErrorNotReady) {
        ctx->error = std::string("evaluation failed on the device: ") + cudaGetErrorString(q);
        return GAML_ERR_CUDA;
      }
      const double waited = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      if (own && q == cudaSuccess && waited > 1.0) return fail(ctx, GAML_ERR_CUDA, "evaluation finished without publishing its result");
      if (!own && waited > 60.0) return fail(ctx, GAML_ERR_STATE, "a peer rank did not publish its result within 60 s");
    }
  }
}

int finish(gaml_ctx* ctx, double* partials, int32_t* total_len, double* gathered = nullptr) {
  if (!ctx->launched) return fail(ctx, GAML_ERR_STATE, "gaml_eval_finish without gaml_eval_launch");
  const size_t n_sets = ctx->sets.size();
  if (gathered && !ctx->exch_host && !ctx->peer_on && !ctx->nccl_on)
    return fail(ctx, GAML_ERR_STATE, "gaml_eval_finish_gathered needs a result exchange (gaml_set_result_exchange, gaml_peer_exchange_open "
                                     "or gaml_nccl_exchange_init)");
  const double want_d = (double)ctx->epoch;
  uint64_t want_bits;
  memcpy(&want_bits, &want_d, 8);
  const int gather_world = ctx->peer_on ? ctx->peer_world : (ctx->nccl_on ? ctx->nccl_world : ctx->exch_world);
  const bool peer_gather = gathered && ctx->peer_on;
  if (peer_gather) {
    // the chain's last kernel has collected every rank's lines in this rank's own pinned memory: ONE flag line to wait for
    const size_t flag_at = (size_t)ctx->peer_world * GAML_EXCHANGE_MAX_SETS * kResultStride;
    double flag[kResultStride];
    const int rc = wait_line(ctx, reinterpret_cast<const volatile uint64_t*>(ctx->h_gather + flag_at), want_bits, flag, true);
    if (rc != GAML_OK) return rc;
    std::atomic_thread_fence(std::memory_order_acquire);
    uint64_t status;
    memcpy(&status, &flag[0], 8);
    if (status != 0) {
      ctx->prepared = ctx->launched = false;
      for (auto& rsp : ctx->sets) rsp->has_state = rsp->total_valid = false;
      return fail(ctx, GAML_ERR_STATE, "a peer rank did not publish its result in time (ranks out of lockstep?)");
    }
  }
  const double* own_lines = peer_gather ? reinterpret_cast<const double*>(ctx->h_gather) + (size_t)ctx->peer_rank * n_sets * kResultStride
                            : (ctx->exch_host ? ctx->exch_host + exch_line(ctx, ctx->exch_rank, 0) * kResultStride : ctx->h_out);
  bool need_sync = false;
  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    if ((rs.pb_penalty || rs.penalty) && rs.sharded) {   // swept later, over all shards' events (gaml_penalty_import)
      rs.penalty_pending = true;
      need_sync = true;
      continue;
    }
    if (rs.pb_penalty) {   // one int: this evaluation's bad bases over all walks (a local in CalcScoreForPacbio)
      rs.h_bad.assign(1, 0);
      CU(cudaMemcpyAsync(rs.h_bad.data(), rs.d_bad.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
      need_sync = true;
      continue;
    }
    if (!rs.penalty) continue;
    rs.h_bad.assign(std::max(ctx->plan[s].n_cov_walks, 1), 0);
    if (ctx->plan[s].n_cov_walks)
      CU(cudaMemcpyAsync(rs.h_bad.data(), rs.d_bad.p, (size_t)ctx->plan[s].n_cov_walks * 4, cudaMemcpyDeviceToHost, ctx->stream));
    need_sync = true;
  }
  ctx->h_res.resize(std::max<size_t>(n_sets, 1) * kResultStride);
  if (need_sync) {
    CU(cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->h_res.data(), own_lines, n_sets * kResultStride * sizeof(double));
  } else if (peer_gather) {
    memcpy(ctx->h_res.data(), own_lines, n_sets * kResultStride * sizeof(double));   // complete: the flag line was written after them
  } else {
    // The last block of every set's last kernel wrote the set's result and then this evaluation's epoch into the
    // host-mapped buffer: spin on the flags instead of paying a copy and a stream synchronisation. The stream is
    // polled now and then so that a failed launch surfaces as an error instead of a hang.
    // A line counts only when its flag word carries this evaluation's epoch AND its checksum matches: the device
    // writes all eight words with one store and no fence, so a partially arrived line must be told from a whole one.
    // A set whose chain ended with its streaming kernel may instead publish a pending line (flag word -epoch): it listed
    // reads for the many-placement pass, which runs now, on demand, and publishes the final line.
    const volatile uint64_t* ho = reinterpret_cast<const volatile uint64_t*>(own_lines);
    const double pend_d = -(double)ctx->epoch;
    uint64_t pend_bits;
    memcpy(&pend_bits, &pend_d, 8);
    bool any_pending = false;
    for (size_t s = 0; s < n_sets; s++) {
      ReadSetState& rs = *ctx->sets[s];
      bool pending = false;
      const int rc = wait_line(ctx, ho + s * kResultStride, want_bits, ctx->h_res.data() + s * kResultStride, true,
                               rs.tail_on_demand ? &pending : nullptr, pend_bits);
      if (rc != GAML_OK) return rc;
      if (!pending) continue;
      if (!any_pending && ctx->timed) CU(cudaEventRecord(ctx->ev[1], ctx->stream));
      any_pending = true;
      launch_paired_tail(rs.tail_params, rs.tail_grid, ctx->stream);
      CU(cudaGetLastError());
      ctx->stats.kernel_launches++;
    }
    if (any_pending) {
      if (ctx->timed) {
        CU(cudaEventRecord(ctx->ev[2], ctx->stream));
        ctx->tail_timed = true;
      }
      for (size_t s = 0; s < n_sets; s++) {
        uint64_t flag;
        memcpy(&flag, ctx->h_res.data() + s * kResultStride + 6, 8);
        if (!ctx->sets[s]->tail_on_demand || flag != pend_bits) continue;
        const int rc = wait_line(ctx, ho + s * kResultStride, want_bits, ctx->h_res.data() + s * kResultStride, true);
        if (rc != GAML_OK) return rc;
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
  }
  if (gathered) {   // every rank's partials of this evaluation (the ranks evaluate in lockstep: same epoch everywhere)
    for (int rk = 0; rk < gather_world; rk++)
      for (size_t s = 0; s < n_sets; s++) {
        double line[kResultStride];
        if (nccl_lines(ctx)) {
          // the all-reduce left the SUM over ranks: reported as shard 0's partials, the other shards' as zeros — the
          // combine step adds the shards, so the result is the same double
          if (rk == 0) {
            const int rc = wait_line(ctx, reinterpret_cast<const volatile uint64_t*>(ctx->h_gather + s * kResultStride), want_bits, line, true);
            if (rc != GAML_OK) return rc;
            if (((uint64_t)line[5]) & 15) {   // (flags are summed too: any rank's error bits make the sum non-zero mod 16 or beyond)
              for (auto& rsp : ctx->sets) rsp->has_state = rsp->total_valid = false;
            }
          } else {
            memset(line, 0, sizeof(line));
          }
        } else if (peer_gather) {
          memcpy(line, reinterpret_cast<const double*>(ctx->h_gather) + ((size_t)rk * n_sets + s) * kResultStride, sizeof(line));
          if (rk != ctx->peer_rank && (((uint64_t)line[5]) & 15)) return fail(ctx, GAML_ERR_CAPACITY, "a peer rank reported a capacity error");
        } else if (rk == ctx->exch_rank) {
          memcpy(line, ctx->h_res.data() + s * kResultStride, sizeof(line));
        } else {
          const volatile uint64_t* src = reinterpret_cast<const volatile uint64_t*>(ctx->exch_host + exch_line(ctx, rk, s) * kResultStride);
          const int rc = wait_line(ctx, src, want_bits, line, false);
          if (rc != GAML_OK) return rc;
          if (((uint64_t)line[5]) & 15) return fail(ctx, GAML_ERR_CAPACITY, "a peer rank reported a capacity error");
        }
        for (int k = 0; k < GAML_PARTIAL_DOUBLES; k++) gathered[((size_t)rk * n_sets + s) * GAML_PARTIAL_DOUBLES + k] = line[k];
      }
  }
  ctx->stats.last_d2h_bytes = (int64_t)(n_sets * kResultStride * sizeof(double));
  ctx->timing_pending = ctx->timed;
  if (!ctx->timed) ctx->stats.last_device_ms = ctx->stats.last_score_kernel_ms = 0;
  ctx->stats.evals++;
  ctx->prepared = ctx->launched = false;
  int tl = 0;
  uint32_t flags = 0, ovf = 0;
  int64_t scratch_placements = 0;
  bool any_paired = false;
  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    const double* o = ctx->h_res.data() + s * kResultStride;   // the validated copy
    if (partials)
      for (int k = 0; k < GAML_PARTIAL_DOUBLES; k++) partials[s * GAML_PARTIAL_DOUBLES + k] = o[k];
    const uint64_t f = (uint64_t)o[5];
    flags |= (uint32_t)(f & 15);
    ovf += (uint32_t)((f >> 4) & 0xffffff);
    scratch_placements = std::max<int64_t>(scratch_placements, (int64_t)(f >> 28));
    if (rs.pb_penalty && !rs.sharded) rs.bad_bases = rs.h_bad[0];
    if (rs.cfg.kind == GAML_KIND_PAIRED) {
      if (ctx->plan[s].full) rs.keep_tail = ((f >> 4) & 0xffffff) != 0;   // expected to list reads again next time
      if (rs.penalty && !rs.sharded) {   // EraseFromScoringState / AddToScoringState, graph.cc:1938, 1946
        if (ctx->plan[s].full) rs.bad_bases = 0;
        for (int w = 0; w < ctx->plan[s].n_cov_walks; w++)
          rs.bad_bases += w < ctx->plan[s].n_erased ? -rs.h_bad[w] : rs.h_bad[w];
      }
      {
        const int tl1 = ctx->plan[s].total_len == 0 ? 1 : ctx->plan[s].total_len;
        rs.total_two_len = (int)(2u * (unsigned)tl1);
        rs.total_valid = true;   // (cleared again below when the evaluation reported a capacity error)
      }
      rs.has_state = true;   // graph.cc:1986: state follows the last EVALUATED walks (ctx->prev() after the swap below)
      any_paired = true;
    }
  }
  if (any_paired) {   // the evaluated walks become old_paths; the other buffer is reused next time
    const WalkSet& now = ctx->cur();
    const WalkDiff& d = ctx->cur_diff;
    if (ctx->have_prev && d.valid && ctx->prev_counts.valid && !ctx->prev_counts.crowded()) {
      const WalkSet& was = ctx->prev();
      for (int i : d.old_changed) ctx->prev_counts.add(was.hash[i], -1);
      for (int i : d.new_changed) ctx->prev_counts.add(now.hash[i], +1);
    } else {
      ctx->prev_counts.rebuild(now);
    }
    ctx->prev_total_len = ctx->cur_total_len;
    ctx->cur_set ^= 1;
    ctx->have_prev = true;
    ctx->cur_diff.valid = false;
  }
  // CalcProb leaves the value of the last set it ran: single sets, then paired, then pacbio (prob_calculator.h:70-107)
  for (int kind = 0; kind < 3; kind++)
    for (size_t s = 0; s < n_sets; s++)
      if (ctx->sets[s]->cfg.kind == kind) tl = ctx->plan[s].total_len;
  if (total_len) *total_len = tl;
  ctx->stats.last_overflow_reads = (int32_t)ovf;
  ctx->stats.last_scratch_placements = scratch_placements;
  {
    int64_t mi = 0;
    for (size_t s = 0; s < n_sets; s++)
      if (ctx->plan[s].full && ctx->sets[s]->cfg.kind == GAML_KIND_PAIRED)
        mi += ctx->plan[s].multi_records;
    ctx->stats.last_multi_items = mi;
  }
  ctx->capacity_grew = false;
  if (flags & 15) {
    // the kernels skipped the reads they had no room for: their per-read state (ScoringState::probs) was not updated, so
    // nothing incremental may build on this evaluation — the next one re-scores every read. The buffer that overflowed is
    // enlarged for it (the one-shot entry points retry by themselves).
    for (auto& rsp : ctx->sets) {
      rsp->has_state = false;
      rsp->total_valid = false;
    }
    if ((flags & 1) && ctx->ovf_cap < (1u << 30)) {
      ctx->ovf_cap *= 4;
      ctx->capacity_grew = true;
    }
    if ((flags & 2) && ctx->scratch_entries < (1ull << 27)) {
      ctx->scratch_entries *= 4;
      ctx->capacity_grew = true;
    }
  }
  if (flags & 1) return fail(ctx, GAML_ERR_CAPACITY, "too many many-placement reads for the overflow list");
  if (flags & 2) return fail(ctx, GAML_ERR_CAPACITY, "placement scratch exhausted (GAML_B200_SCRATCH_ENTRIES)");
  if (flags & 4) return fail(ctx, GAML_ERR_CAPACITY, "coverage-event buffer exhausted");
  return GAML_OK;
}

int combine_raw(const double* gathered, int n_shards, int n_sets, const int32_t* kinds, const int64_t* n_reads_total,
                const double* weights, int total_len, gaml_result* result, int32_t* zeros,
                const double* penalty_terms = nullptr) {
  if (!gathered || n_shards < 1 || n_sets < 0 || !result || (n_sets > 0 && (!kinds || !n_reads_total || !weights)))
    return GAML_ERR_ARG;
  std::vector<double> score(n_sets);
  for (int s = 0; s < n_sets; s++) {
    // shard totals are exact integers in units of 2^-40 (integer part, fraction units): add them exactly
    __int128 ip = 0, fr = 0;
    double fl = 0, neginf = 0, nan = 0;
    for (int k = 0; k < n_shards; k++) {
      const double* p = gathered + ((size_t)k * n_sets + s) * GAML_PARTIAL_DOUBLES;
      ip += (__int128)(long long)p[0];
      fr += (__int128)(long long)p[1];
      fl += p[2];
      neginf += p[3];
      nan += p[4];
    }
    const __int128 x = ip * ((__int128)1 << 40) + fr;
    double total = (double)x * (1.0 / 1099511627776.0);   // one rounding: int128 -> double, then an exact scaling
    if (nan > 0) total = std::numeric_limits<double>::quiet_NaN();
    else if (neginf > 0) total = -std::numeric_limits<double>::infinity();
    double sc = total / (double)n_reads_total[s];   // total_prob / total_c, graph.cc:1515, 1536, 3087
    if (kinds[s] == GAML_KIND_PACBIO) {
      const int tl = total_len == 0 ? 1 : total_len;
      sc -= log((double)(int)(2u * (unsigned)tl));   // graph.cc:3087
    }
    if (penalty_terms) sc = sc - penalty_terms[s];   // tp - bad_bases*no_cov_penalty, graph.cc:1742, 1988
    score[s] = sc;
    if (zeros) {
      zeros[2 * s] = (int32_t)fl;
      zeros[2 * s + 1] = (int32_t)n_reads_total[s];
    }
  }
  double prob = 0;
  for (int kind = 0; kind < 3; kind++)   // prob_calculator.h:70-107: single, paired, pacbio
    for (int s = 0; s < n_sets; s++)
      if (kinds[s] == kind) prob += score[s] * weights[s];
  result->prob = prob;
  result->total_len = total_len;
  result->n_sets = n_sets;
  return GAML_OK;
}

int combine(gaml_ctx* ctx, const double* gathered, int n_shards, int total_len, gaml_result* result, int32_t* zeros) {
  const size_t n_sets = ctx->sets.size();
  for (auto& rs : ctx->sets)
    if (rs->penalty_pending)
      return fail(ctx, GAML_ERR_STATE, "a penalised read set on a read-id shard: gather the shards' coverage events "
                                       "(gaml_penalty_export) and hand them to gaml_penalty_import before combining");
  std::vector<int32_t> kinds(n_sets);
  std::vector<int64_t> counts(n_sets);
  std::vector<double> weights(n_sets), pen(n_sets);
  for (size_t s = 0; s < n_sets; s++) {
    kinds[s] = ctx->sets[s]->cfg.kind;
    counts[s] = ctx->sets[s]->n_total;
    weights[s] = ctx->sets[s]->cfg.weight;
    pen[s] = ctx->sets[s]->bad_bases * ctx->sets[s]->cfg.penalty_constant;   // int * double like the reference
  }
  int rc = combine_raw(gathered, n_shards, (int)n_sets, kinds.data(), counts.data(), weights.data(), total_len, result, zeros,
                       pen.data());
  if (rc) return fail(ctx, rc, "bad combine arguments");
  return GAML_OK;
}

// ---- batched candidate evaluation (BASELINE config 5) ------------------------------------------------------
// Candidate c = the last evaluated walk set with walks erased_idx[c] removed and its added walks appended. Host
// work is O(#nodes of the touched walks) per candidate plus O(#base walks) once per batch.
int calc_prob_batch_partial(gaml_ctx* ctx, int n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                            const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                            double* partials, int32_t* total_lens, bool reduce_over_ranks = false) {
  if (n_cand <= 0 || !erased_off || !cand_added_off || !added_walk_off || !partials)
    return fail(ctx, GAML_ERR_ARG, "bad batch arguments");
  const auto t_batch0 = std::chrono::steady_clock::now();
  double batch_device_ms = 0.0;
  if (ctx->prepared || ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is pending");
  const size_t n_sets = ctx->sets.size();
  if (n_sets == 0) return fail(ctx, GAML_ERR_STATE, "no read sets");
  for (auto& rs : ctx->sets) {
    if (rs->cfg.kind != GAML_KIND_PAIRED)
      return fail(ctx, GAML_ERR_UNSUPPORTED, "gaml_calc_prob_batch supports paired read sets only (single / pacbio sets keep no "
                                             "incremental state: every candidate would be a full evaluation)");
    if (!rs->has_state) return fail(ctx, GAML_ERR_STATE, "gaml_calc_prob_batch needs a base state: call gaml_calc_prob first");
    if (rs->penalty) return fail(ctx, GAML_ERR_UNSUPPORTED, "gaml_calc_prob_batch with penalty_constant != 0 is not supported yet");
  }
  int rc = commit(ctx);
  if (rc != GAML_OK) return rc;
  const WalkSet& base_set = ctx->prev();   // old_paths of every set
  const int n_base = base_set.n;
  // Rank of every base walk in the iteration order of the reference's multiset (GetChanges, graph.cc:1747-1763): erasing
  // the kept walks leaves the others in place, so a candidate's erased walks come out in rank order. With no equal walks
  // in the base set the order is the container's rule (walk_set.h): buckets by the index of their first element,
  // descending, then index descending — found from the cached bucket numbers in one pass; with equal walks the
  // container itself is built.
  std::vector<int64_t> rank((size_t)n_base, 0);
  {
    bool unique = ctx->prev_counts.valid && base_set.bkt_count == bucket_count_for((size_t)std::max(n_base, 1)) &&
                  (int)base_set.bkt.size() == n_base;
    if (unique)
      for (int i = 0; i < n_base && unique; i++) unique = ctx->prev_counts.get(base_set.hash[i]) == 1;
    if (unique) {
      std::vector<int> first(base_set.bkt_count, -1);
      for (int i = 0; i < n_base; i++)
        if (first[base_set.bkt[i]] < 0) first[base_set.bkt[i]] = i;
      // ascending rank = earlier in the iteration: larger first-of-bucket first, then larger index first
      for (int i = 0; i < n_base; i++) rank[i] = -((int64_t)first[base_set.bkt[i]] * ((int64_t)n_base + 1) + (int64_t)i);
    } else {
      std::vector<Walk> base((size_t)n_base);
      for (int i = 0; i < n_base; i++) base[i] = base_set.walk(i);
      std::unordered_multiset<Walk, WalkHash> idx(base.begin(), base.begin() + n_base);
      std::unordered_map<Walk, std::vector<int>, WalkHash> where;
      for (int i = n_base - 1; i >= 0; i--) where[base[i]].push_back(i);
      int64_t k = 0;
      for (const Walk& w : idx) {
        std::vector<int>& v = where[w];
        rank[v.back()] = k++;
        v.pop_back();
      }
    }
  }
  long long base_len = 0;
  std::vector<int> base_walk_len(n_base);
  for (int i = 0; i < n_base; i++) {
    int t = 0;
    for (int64_t k = base_set.offs[i]; k < base_set.offs[i + 1]; k++) {
      const int x = base_set.nodes[(size_t)k];
      t += x < 0 ? -x : ctx->node_len[x];
    }
    base_walk_len[i] = t;
    base_len += t;
  }
  // distinct total lengths, ascending (the base pass relies on the floor test growing with the index)
  std::vector<int> cand_len(n_cand);
  std::vector<int> cand_two(n_cand);
  std::vector<int> two_lens;
  std::vector<int> cand_len_index(n_cand);
  std::vector<std::vector<Walk>> cand_added(n_cand);
  std::vector<std::vector<int>> cand_erased(n_cand);
  for (int c = 0; c < n_cand; c++) {
    long long tl = base_len;
    for (int64_t k = erased_off[c]; k < erased_off[c + 1]; k++) {
      const int bi = erased_idx[k];
      if (bi < 0 || bi >= n_base) return fail(ctx, GAML_ERR_ARG, "erased walk index outside the base walk set");
      cand_erased[c].push_back(bi);
      tl -= base_walk_len[bi];
    }
    std::sort(cand_erased[c].begin(), cand_erased[c].end(), [&](int a, int b) { return rank[a] < rank[b]; });
    for (size_t k = 1; k < cand_erased[c].size(); k++)
      if (cand_erased[c][k] == cand_erased[c][k - 1]) return fail(ctx, GAML_ERR_ARG, "erased walk listed twice");
    for (int64_t w = cand_added_off[c]; w < cand_added_off[c + 1]; w++) {
      Walk wk(added_nodes + added_walk_off[w], added_nodes + added_walk_off[w + 1]);
      for (int x : wk)
        if (x >= (int)ctx->node_len.size()) return fail(ctx, GAML_ERR_ARG, "walk references a node outside the graph");
      tl += walk_length(ctx, wk);
      cand_added[c].push_back(std::move(wk));
    }
    cand_len[c] = (int)tl;
    if (total_lens) total_lens[c] = (int)tl;
    cand_two[c] = two_len_of(cand_len[c]);
    two_lens.push_back(cand_two[c]);
  }
  std::sort(two_lens.begin(), two_lens.end());
  two_lens.erase(std::unique(two_lens.begin(), two_lens.end()), two_lens.end());
  for (int c = 0; c < n_cand; c++)
    cand_len_index[c] = (int)(std::lower_bound(two_lens.begin(), two_lens.end(), cand_two[c]) - two_lens.begin());
  std::vector<long long> ql(two_lens.size());
  for (size_t j = 0; j < two_lens.size(); j++) ql[j] = fix_log_host((double)two_lens[j]);
  const int n_len = (int)two_lens.size();
  ctx->h_batch_out.assign((size_t)n_cand * kOutStride, 0.0);
  cudaStream_t st = ctx->stream;

  for (size_t s = 0; s < n_sets; s++) {
    ReadSetState& rs = *ctx->sets[s];
    std::vector<BatchCand> cands(n_cand);
    std::vector<int32_t> keys[2];
    std::vector<SlotA> sa[2];
    std::vector<SlotB> sb[2];
    std::vector<Occ> occ[2];
    std::vector<TouchRange> ranges;
    std::vector<uint32_t> range_prefix(1, 0);
    std::vector<int32_t> range_cand;
    uint64_t touch_total = 0;
    for (int c = 0; c < n_cand; c++) {
      OccBuilder obs[2];
      OccBuilder* ob[2] = {&obs[0], &obs[1]};
      SetPlan sp;
      std::vector<TouchRange> touch;
      int ord = 0;
      for (int bi : cand_erased[c]) flatten_paired_walk(ctx, rs, base_set.view(bi), ord++, ob, sp, &touch);
      for (const Walk& w : cand_added[c])
        flatten_paired_walk(ctx, rs, WalkView{w.data(), (int)w.size(), hash_walk(w), -1}, ord++, ob, sp, &touch);
      BatchCand& cd = cands[c];
      cd.n_erased = (int)cand_erased[c].size();
      cd.len_index = cand_len_index[c];
      for (int m = 0; m < 2; m++) {
        std::vector<std::pair<int, Occ>>& items = obs[m].items;
        std::stable_sort(items.begin(), items.end(),
                         [](const std::pair<int, Occ>& a, const std::pair<int, Occ>& b) { return a.first < b.first; });
        cd.key_begin[m] = (int)keys[m].size();
        size_t i = 0;
        while (i < items.size()) {
          size_t j = i;
          while (j < items.size() && items[j].first == items[i].first) j++;
          const Occ& f = items[i].second;
          keys[m].push_back(items[i].first);
          sa[m].push_back(SlotA{(uint32_t)(j - i > 1 ? 0x80000000u : 0u), f.walk, f.cur_pos, f.skip_below});
          sb[m].push_back(SlotB{f.seg, (int)(j - i), (int)occ[m].size(), 0});
          for (size_t t = i; t < j; t++) occ[m].push_back(items[t].second);
          i = j;
        }
        cd.key_count[m] = (int)keys[m].size() - cd.key_begin[m];
      }
      cd.range_begin = (int32_t)ranges.size();
      // each touched mate-1 key once (a key of an erased walk often reappears in the added walk)
      std::sort(touch.begin(), touch.end(), [](const TouchRange& a, const TouchRange& b) { return a.begin < b.begin; });
      for (size_t t = 0; t < touch.size(); t++) {
        if (t > 0 && touch[t].begin == touch[t - 1].begin) continue;
        ranges.push_back(touch[t]);
        range_cand.push_back(c);
        touch_total += touch[t].count;
        if (touch_total > 0xffffffffull) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^32 touched records in one batch");
        range_prefix.push_back((uint32_t)touch_total);
      }
      cd.range_count = (int32_t)ranges.size() - cd.range_begin;
    }
    // ---- blob ----
    auto align16 = [](size_t x) { return (x + 15) & ~size_t(15); };
    size_t off = 0;
    auto place = [&](size_t bytes) { size_t o = off; off = align16(off + bytes); return o; };
    const size_t o_cands = place(cands.size() * sizeof(BatchCand));
    size_t o_keys[2], o_sa[2], o_sb[2], o_occ[2];
    for (int m = 0; m < 2; m++) {
      o_keys[m] = place(keys[m].size() * 4);
      o_sa[m] = place(sa[m].size() * 16);
      o_sb[m] = place(sb[m].size() * 16);
      o_occ[m] = place(occ[m].size() * 16);
    }
    const size_t o_ranges = place(ranges.size() * sizeof(TouchRange));
    const size_t o_prefix = place(range_prefix.size() * 4);
    const size_t o_rcand = place(range_cand.size() * 4);
    // the touched-record pass: one block per slice of kBatchSlice records of a candidate
    std::vector<Int2> blocks;
    for (int c = 0; c < n_cand; c++) {
      const uint32_t tot = range_prefix[(size_t)cands[c].range_begin + cands[c].range_count] - range_prefix[(size_t)cands[c].range_begin];
      for (uint32_t at = 0; at < tot; at += (uint32_t)kBatchSlice) blocks.push_back(Int2{c, (int32_t)at});
    }
    const size_t o_blocks = place(blocks.size() * sizeof(Int2));
    // floor tests: per length class of the set (distinct len1 + len2) and distinct total length
    std::vector<int32_t> len_class(std::max<size_t>(rs.h_thr.size(), 1), 0);
    std::vector<long long> qthr_cls(std::max<size_t>(rs.len_classes.size(), 1), 0);
    std::vector<double> pstar(std::max<size_t>(rs.len_classes.size(), 1) * (size_t)n_len, 0.0);
    for (size_t k = 0; k < rs.len_classes.size(); k++) {
      const int li = rs.len_classes[k];
      len_class[li] = (int32_t)k;
      qthr_cls[k] = rs.h_qthr[li];
      for (int j = 0; j < n_len; j++) pstar[k * (size_t)n_len + j] = floor_pstar(rs.h_thr[li], (double)two_lens[j]);
    }
    const size_t o_pstar = place(pstar.size() * 8);
    const size_t o_qcls = place(qthr_cls.size() * 8);
    const size_t o_lcls = place(len_class.size() * 4);
    const size_t o_ql = place(ql.size() * 8);
    std::vector<char> blob(std::max<size_t>(off, 16));
    auto put = [&](size_t o, const void* p, size_t bytes) { if (bytes) memcpy(blob.data() + o, p, bytes); };
    put(o_cands, cands.data(), cands.size() * sizeof(BatchCand));
    for (int m = 0; m < 2; m++) {
      put(o_keys[m], keys[m].data(), keys[m].size() * 4);
      put(o_sa[m], sa[m].data(), sa[m].size() * 16);
      put(o_sb[m], sb[m].data(), sb[m].size() * 16);
      put(o_occ[m], occ[m].data(), occ[m].size() * 16);
    }
    put(o_ranges, ranges.data(), ranges.size() * sizeof(TouchRange));
    put(o_prefix, range_prefix.data(), range_prefix.size() * 4);
    put(o_rcand, range_cand.data(), range_cand.size() * 4);
    put(o_blocks, blocks.data(), blocks.size() * sizeof(Int2));
    put(o_pstar, pstar.data(), pstar.size() * 8);
    put(o_qcls, qthr_cls.data(), qthr_cls.size() * 8);
    put(o_lcls, len_class.data(), len_class.size() * 4);
    put(o_ql, ql.data(), ql.size() * 8);
    CU(ctx->d_batch_blob.reserve(blob.size(), 0, false, st));
    CU(cudaMemcpyAsync(ctx->d_batch_blob.p, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));
    const size_t hist_words = (size_t)batch_hist_bins(n_len) * kBatchBin;
    const size_t acc_bytes = (((size_t)n_len + 1) * kAccumStride + (size_t)n_cand * 4 + hist_words) * 8;
    CU(ctx->d_batch_acc.reserve(acc_bytes, 0, false, st));
    CU(cudaMemsetAsync(ctx->d_batch_acc.p, 0, acc_bytes, st));
    CU(ctx->d_batch_out.reserve((size_t)n_cand * kOutStride * 8, 0, false, st));
    CU(ctx->d_flags.reserve(flags_words(n_sets) * sizeof(unsigned long long), 0, true, st));
    CU(cudaMemsetAsync(ctx->d_flags.p, 0, 2 * sizeof(unsigned long long), st));
    CU(ctx->d_scratch.reserve(ctx->scratch_entries * sizeof(Plc), 0, false, st));
    // ---- params ----
    ctx->plan.assign(n_sets, SetPlan());
    ScoreParams P = make_params(ctx, s);
    char* db = ctx->d_batch_blob.as<char>();
    BatchParams B{};
    B.cands = reinterpret_cast<const BatchCand*>(db + o_cands);
    B.n_cand = n_cand;
    for (int m = 0; m < 2; m++) {
      B.keys[m] = reinterpret_cast<const int32_t*>(db + o_keys[m]);
      B.slot_a[m] = db + o_sa[m];
      B.slot_b[m] = db + o_sb[m];
      B.occ[m] = reinterpret_cast<const Occ*>(db + o_occ[m]);
    }
    B.ranges = reinterpret_cast<const TouchRange*>(db + o_ranges);
    B.range_prefix = reinterpret_cast<const uint32_t*>(db + o_prefix);
    B.range_cand = reinterpret_cast<const int32_t*>(db + o_rcand);
    B.partner12 = rs.comb_ok ? rs.d_partner12.as<int32_t>() : nullptr;
    B.blocks = reinterpret_cast<const Int2*>(db + o_blocks);
    B.n_blocks = (int)blocks.size();
    B.n_ranges = (int)ranges.size();
    B.pstar = reinterpret_cast<const double*>(db + o_pstar);
    B.qthr_cls = reinterpret_cast<const long long*>(db + o_qcls);
    B.len_class = reinterpret_cast<const int32_t*>(db + o_lcls);
    B.ql = reinterpret_cast<const long long*>(db + o_ql);
    B.n_len = n_len;
    B.accum_len = ctx->d_batch_acc.as<unsigned long long>();
    B.accum_cand = reinterpret_cast<long long*>(B.accum_len + ((size_t)n_len + 1) * kAccumStride);
    B.hist = B.accum_len + ((size_t)n_len + 1) * kAccumStride + (size_t)n_cand * 4;
    CU(cudaEventRecord(ctx->ev[1], st));
    launch_batch(P, B, (uint32_t)touch_total, ctx->d_batch_out.as<double>(),
                 reinterpret_cast<const uint32_t*>(ctx->d_flags.as<unsigned long long>() + 1), ctx->sm_count, st);
    CU(cudaEventRecord(ctx->ev[2], st));
    CU(cudaGetLastError());
    ctx->stats.kernel_launches += batch_launches(n_len, touch_total > 0);
    if (reduce_over_ranks) {
      // all shards' partials of every candidate, summed by one all-reduce on the stream (exact: integers in doubles)
      const int rc2 = nccl_all_reduce_doubles(ctx, ctx->d_batch_out.as<double>(), (size_t)n_cand * kOutStride);
      if (rc2 != GAML_OK) return rc2;
      ctx->stats.kernel_launches++;
    }
    CU(cudaMemcpyAsync(ctx->h_batch_out.data(), ctx->d_batch_out.p, (size_t)n_cand * kOutStride * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]) == cudaSuccess) batch_device_ms += ms;
    }
    ctx->stats.last_records_gathered = (int64_t)touch_total;
    for (int c = 0; c < n_cand; c++) {
      const double* o = ctx->h_batch_out.data() + (size_t)c * kOutStride;
      if (((uint64_t)o[5]) & 2) return fail(ctx, GAML_ERR_CAPACITY, "placement scratch exhausted (GAML_B200_SCRATCH_ENTRIES)");
      for (int k = 0; k < GAML_PARTIAL_DOUBLES; k++) partials[((size_t)c * n_sets + s) * GAML_PARTIAL_DOUBLES + k] = o[k];
    }
  }
  // (measurement: the batch kernels' device time, and the whole call's wall time, in the fields of a normal evaluation)
  ctx->stats.last_device_ms = batch_device_ms;
  ctx->stats.last_prepare_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_batch0).count();
  ctx->timing_pending = false;
  return GAML_OK;
}

int check_ctx(gaml_ctx* ctx) { return ctx ? GAML_OK : GAML_ERR_ARG; }

}  // namespace
}  // namespace gaml

// ===========================================================================================
// C ABI
// ===========================================================================================
extern "C" {

int gaml_ctx_create(int device, gaml_ctx** out) {
  if (!out) return GAML_ERR_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (there is no CPU fallback)";
    return GAML_ERR_CUDA;
  }
  if (device < 0 || device >= n) {
    g_create_error = "device index out of range";
    return GAML_ERR_ARG;
  }
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_create_error = cudaGetErrorString(e);
    return GAML_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_create_error = "gaml_b200 is built for sm_100a only; found sm_" + std::to_string(prop.major * 10 + prop.minor);
    return GAML_ERR_CUDA;
  }
  gaml_ctx* ctx = new gaml_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* s = getenv("GAML_B200_SCRATCH_ENTRIES")) ctx->scratch_entries = strtoull(s, nullptr, 10);
  if (const char* s = getenv("GAML_B200_NO_RUNNING_TOTAL")) ctx->running_total = !(s[0] && s[0] != '0');
  if (const char* s = getenv("GAML_B200_NO_GRAPHS")) ctx->use_graphs = !(s[0] && s[0] != '0');
  if (const char* s = getenv("GAML_B200_NO_FAST_CHANGES")) ctx->fast_changes = !(s[0] && s[0] != '0');
  if (const char* s = getenv("GAML_B200_NO_PERMUTE")) ctx->permute_reads = !(s[0] && s[0] != '0');
  if (const char* s = getenv("GAML_B200_NO_APPEND")) ctx->append_enabled = !(s[0] && s[0] != '0');
  if (const char* s = getenv("GAML_B200_NO_FULL_PATCH")) ctx->patch_enabled = !(s[0] && s[0] != '0');
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_error = cudaGetErrorString(e);
    delete ctx;
    return GAML_ERR_CUDA;
  }
  for (auto& ev : ctx->ev) cudaEventCreate(&ev);
  cudaEventCreateWithFlags(&ctx->ev_append, cudaEventDisableTiming);
  {
    // log table for table_log (kernels.cu): interval i of z in [0.6875, 1.375) -> {invc = RN(1/centre), -log(invc)}
    // with the logarithm of the ROUNDED reciprocal taken in long double, so log z = log1p(z*invc - 1) + logc exactly.
    std::vector<double> tab(256);
    for (int i = 0; i < 128; i++) {
      const uint64_t lo = 0x3fe6000000000000ull + ((uint64_t)i << 45), hi = lo + ((uint64_t)1 << 45);
      double zlo, zhi;
      memcpy(&zlo, &lo, 8);
      memcpy(&zhi, &hi, 8);
      const double invc = (double)(2.0L / ((long double)zlo + (long double)zhi));
      tab[2 * i] = invc;
      tab[2 * i + 1] = (double)(-logl((long double)invc));
    }
    if (ctx->d_logtab.reserve(tab.size() * 8, 0, false, ctx->stream) != cudaSuccess ||
        cudaMemcpyAsync(ctx->d_logtab.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      g_create_error = "cannot upload the log table";
      gaml_ctx_destroy(ctx);
      return GAML_ERR_CUDA;
    }
  }
  *out = ctx;
  return GAML_OK;
}

void gaml_ctx_destroy(gaml_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  ctx->sets.clear();
  if (ctx->h_blob) cudaFreeHost(ctx->h_blob);
  if (ctx->h_out) cudaFreeHost(ctx->h_out);
  if (ctx->exch_host && ctx->exch_owned) cudaHostUnregister(ctx->exch_host);
  for (size_t p = 0; p < ctx->peer_ptrs.size(); p++)
    if (ctx->peer_opened[p] && ctx->peer_ptrs[p]) cudaIpcCloseMemHandle(ctx->peer_ptrs[p]);
  if (ctx->h_gather) cudaFreeHost(ctx->h_gather);
  if (ctx->nccl_comm)
    if (NcclApi* api = nccl_api(nullptr)) api->comm_destroy(ctx->nccl_comm);
  for (auto& ev : ctx->ev)
    if (ev) cudaEventDestroy(ev);
  if (ctx->ev_append) cudaEventDestroy(ctx->ev_append);
  if (ctx->h_append_pinned) cudaFreeHost(ctx->h_append_pinned);
  cudaStream_t st = ctx->stream;
  for (auto& g : ctx->graphs) {
    if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
    if (g.second.graph) cudaGraphDestroy(g.second.graph);
  }
  delete ctx;
  if (st) cudaStreamDestroy(st);
}

const char* gaml_last_error(gaml_ctx* ctx) { return ctx ? ctx->error.c_str() : g_create_error.c_str(); }

void* gaml_ctx_stream(gaml_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int gaml_set_graph(gaml_ctx* ctx, int32_t n_nodes, const int32_t* node_len, const int32_t* normalize_map) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (n_nodes <= 0 || !node_len) return fail(ctx, GAML_ERR_ARG, "bad graph");
  ctx->node_len.assign(node_len, node_len + n_nodes);
  ctx->nmap.resize(n_nodes);
  for (int i = 0; i < n_nodes; i++) {
    ctx->nmap[i] = normalize_map ? normalize_map[i] : i;
    if (ctx->nmap[i] < 0 || ctx->nmap[i] >= n_nodes) return fail(ctx, GAML_ERR_ARG, "normalize_map out of range");
    if (node_len[i] < 0) return fail(ctx, GAML_ERR_ARG, "negative node length");
  }
  ctx->have_prev = false;   // lengths and lookups of remembered walks refer to the old graph
  ctx->full_blob_valid = false;
  ctx->cache_gen++;
  for (auto& rs : ctx->sets) {
    rs->flat_cache.clear();
    rs->has_state = false;
    rs->total_valid = false;
  }
  return GAML_OK;
}

int gaml_add_readset(gaml_ctx* ctx, const gaml_readset_config* cfg, int64_t n_reads_total, int64_t shard_lo,
                     int64_t shard_hi, const int32_t* read_len1, const int32_t* read_len2, int32_t max_read_len1,
                     int32_t max_read_len2) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (!cfg || n_reads_total < 0 || shard_lo < 0 || shard_hi < shard_lo || shard_hi > n_reads_total)
    return fail(ctx, GAML_ERR_ARG, "bad read set shape");
  if (cfg->kind < 0 || cfg->kind > 2) return fail(ctx, GAML_ERR_ARG, "bad read set kind");
  if (cfg->penalty_constant != 0.0 && cfg->kind == GAML_KIND_PACBIO && !(cfg->match_prob > 0.0 && cfg->mismatch_prob > 0.0))
    return fail(ctx, GAML_ERR_ARG, "a pacbio set with penalty_constant != 0 needs match_prob and mismatch_prob (GetMinReadProb, graph.h:478)");
  // single sets: the reference's sweep never counts a gap (graph.cc:1710-1733: last_event_type is never >= 3), so
  // bad_bases is identically 0 and the penalty term vanishes whatever penalty_constant is
  const int64_t n_local = shard_hi - shard_lo;
  if (n_local > 0x7fffffff) return fail(ctx, GAML_ERR_CAPACITY, "more than 2^31 reads in one shard");
  if (n_local > 0 && !read_len1) return fail(ctx, GAML_ERR_ARG, "read_len1 is NULL");
  const bool paired = cfg->kind == GAML_KIND_PAIRED;
  if (paired && n_local > 0 && !read_len2) return fail(ctx, GAML_ERR_ARG, "read_len2 is NULL");
  if (paired && !(cfg->insert_std > 0)) return fail(ctx, GAML_ERR_ARG, "insert_std must be positive");
  cudaSetDevice(ctx->device);
  std::unique_ptr<ReadSetState> rsp(new ReadSetState());
  ReadSetState& rs = *rsp;
  rs.cfg = *cfg;
  rs.n_total = n_reads_total;
  rs.lo = shard_lo;
  rs.hi = shard_hi;
  rs.n_local = (int)n_local;
  rs.sharded = shard_lo != 0 || shard_hi != n_reads_total;
  rs.n_mates = paired ? 2 : 1;
  const int32_t* lens[2] = {read_len1, read_len2};
  const int32_t maxes[2] = {max_read_len1, max_read_len2};
  for (int m = 0; m < rs.n_mates; m++) {
    rs.len[m].assign(lens[m], lens[m] + n_local);
    int mx = 0;
    for (int v : rs.len[m]) {
      if (v < 0) return fail(ctx, GAML_ERR_ARG, "negative read length");
      mx = std::max(mx, v);
    }
    if (maxes[m] >= 0) {
      if (maxes[m] < mx) return fail(ctx, GAML_ERR_ARG, "max_read_len smaller than a given read length");
      mx = maxes[m];
    }
    rs.max_len[m] = mx;
    if (paired && mx > 0xffff) return fail(ctx, GAML_ERR_CAPACITY, "paired read longer than 65535");
    MateStore& st = rs.mate[m];
    st.is_long = cfg->kind == GAML_KIND_PACBIO;
    if (!st.is_long) {   // ReadSet::CalcMaxReadLen, graph.cc:1448-1453
      st.pow_match.resize(mx + 7);
      st.pow_mismatch.resize(mx + 7);
      for (size_t i = 0; i < st.pow_match.size(); i++) {
        st.pow_match[i] = pow(cfg->match_prob, (double)i);
        st.pow_mismatch[i] = pow(cfg->mismatch_prob, (double)i);
      }
      CU(st.d_pow_match.reserve(st.pow_match.size() * 8, 0, false, ctx->stream));
      CU(st.d_pow_mismatch.reserve(st.pow_match.size() * 8, 0, false, ctx->stream));
      CU(cudaMemcpyAsync(st.d_pow_match.p, st.pow_match.data(), st.pow_match.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
      CU(cudaMemcpyAsync(st.d_pow_mismatch.p, st.pow_mismatch.data(), st.pow_match.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    }
  }
  // lengths
  std::vector<uint32_t> packed(std::max<int64_t>(n_local, 1));
  for (int64_t i = 0; i < n_local; i++)
    packed[i] = paired ? ((uint32_t)rs.len[0][i] | ((uint32_t)rs.len[1][i] << 16)) : (uint32_t)rs.len[0][i];
  rs.lens_uniform = paired && n_local > 0;
  for (int64_t i = 1; i < n_local && rs.lens_uniform; i++) rs.lens_uniform = packed[i] == packed[0];
  rs.uniform_ll = rs.lens_uniform ? packed[0] : 0u;
  CU(rs.d_lens.reserve(packed.size() * 4, 0, false, ctx->stream));
  CU(cudaMemcpyAsync(rs.d_lens.p, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CU(rs.d_values.reserve(std::max<int64_t>(n_local, 1) * 8, 0, true, ctx->stream));
  CU(rs.d_ovf_list.reserve((size_t)ctx->ovf_cap * 4, 0, false, ctx->stream));
  if (paired) CU(rs.d_stamp.reserve(std::max<int64_t>(n_local, 1) * 4, 0, true, ctx->stream));
  if (paired) CU(rs.d_state_acc.reserve(kAccumStride * sizeof(unsigned long long), 0, true, ctx->stream));
  // floor thresholds by length index (paired: len1 + len2), their fixed-point logs, and the length indices that occur
  if (cfg->kind != GAML_KIND_PACBIO) {
    const int top = rs.max_len[0] + (paired ? rs.max_len[1] : 0);
    rs.h_thr.resize(top + 1);
    rs.h_qthr.resize(top + 1);
    for (int l = 0; l <= top; l++) {
      rs.h_thr[l] = exp(cfg->min_prob_start + cfg->min_prob_per_base * (l));   // graph.cc:1506-1507, 1528
      rs.h_qthr[l] = fix_log_host(rs.h_thr[l]);                                // log of the reference's own threshold
    }
    std::vector<char> seen(top + 1, 0);
    for (int64_t i = 0; i < n_local; i++) seen[rs.len[0][i] + (paired ? rs.len[1][i] : 0)] = 1;
    for (int l = 0; l <= top; l++)
      if (seen[l]) rs.len_classes.push_back(l);
    CU(rs.d_qthr.reserve(rs.h_qthr.size() * 8, 0, false, ctx->stream));
    CU(cudaMemcpyAsync(rs.d_qthr.p, rs.h_qthr.data(), rs.h_qthr.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (paired && rs.lens_uniform) {
      // every pair has the same lengths: tabulate mismatch^e * match^(len-e) (graph.cc:1859-1863; one IEEE product, the
      // same double the device forms with __dmul_rn) for the edit distances the packed records can hold
      const int l[2] = {(int)(rs.uniform_ll & 0xffff), (int)(rs.uniform_ll >> 16)};
      for (int m = 0; m < 2; m++) {
        const MateStore& st = rs.mate[m];
        std::vector<double> tab(128, 0.0);
        for (int e = 0; e < 128; e++)
          if (e <= l[m] && (size_t)e < st.pow_mismatch.size() && (size_t)(l[m] - e) < st.pow_match.size())
            tab[e] = st.pow_mismatch[e] * st.pow_match[l[m] - e];
        CU(rs.d_uni_prob[m].reserve(tab.size() * 8, 0, false, ctx->stream));
        CU(cudaMemcpyAsync(rs.d_uni_prob[m].p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));   // tab is a local
      }
    }
  } else {
    rs.floor_a = log(exp(cfg->min_prob_start));      // logdouble(exp(mps)), graph.cc:3075
    rs.floor_b = log(exp(cfg->min_prob_per_base));   // logdouble(exp(mppb)), graph.cc:3076
  }
  // insert-size pdf: the reference tabulates [0,(int)(mean+5 std)) and evaluates the closed form beyond
  // (graph.cc:1801-1804, 1877-1882). The same closed form is tabulated here on the HOST out to mean+40 std,
  // where exp(-z*z/2) has underflowed to exactly 0, so the device never evaluates exp for a pair term.
  std::vector<double> ins;
  if (paired) {
    const double top = cfg->insert_mean + 40.0 * cfg->insert_std + 2.0;
    if (!(top < 64.0 * 1024 * 1024)) return fail(ctx, GAML_ERR_CAPACITY, "insert distribution too wide for the pdf table");
    rs.ins_n = std::max((int)top, (int)(cfg->insert_mean + 5 * cfg->insert_std));
    ins.resize(std::max(rs.ins_n, 1));
    for (int d = 0; d < rs.ins_n; d++) ins[d] = insert_pdf((double)d, cfg->insert_mean, cfg->insert_std);
    CU(rs.d_ins.reserve(ins.size() * 8, 0, false, ctx->stream));
    CU(cudaMemcpyAsync(rs.d_ins.p, ins.data(), ins.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (rs.lens_uniform && rs.ins_n > 0 && !getenv("GAML_B200_NO_TERM_TABLE")) {
      // term table: (edit 1, edit 2, insert distance) -> pair term + its fixed-point logarithm, for the edit distances
      // below 2^shift — as many as fit 16 MiB (L2 resident; the entries a data set really uses are a few KB)
      int shift = 5;
      while (shift >= 2 && ((size_t)1 << (2 * shift)) * (size_t)rs.ins_n * sizeof(TermEntry) > (size_t)16 << 20) shift--;
      if (shift >= 2) {
        CU(rs.d_tq.reserve((1 + ((size_t)1 << (2 * shift)) * (size_t)rs.ins_n) * sizeof(TermEntry), 0, false, ctx->stream));
        launch_build_term_table(rs.d_uni_prob[0].as<double>(), rs.d_uni_prob[1].as<double>(), rs.d_ins.as<double>(), rs.ins_n, shift,
                                ctx->d_logtab.p, rs.d_tq.p, ctx->sm_count, ctx->stream);
        CU(cudaGetLastError());
        ctx->stats.kernel_launches++;
        rs.tq_shift = shift;
      }
    }
  }
  if (cfg->kind == GAML_KIND_PACBIO && cfg->penalty_constant != 0.0) rs.pb_penalty = true;
  if (paired && cfg->penalty_constant != 0.0) {
    rs.penalty = true;
    std::vector<double> cthr(rs.max_len[1] + 1);
    for (int l = 0; l <= rs.max_len[1]; l++) cthr[l] = exp(cfg->min_prob_start + cfg->min_prob_per_base * (l + l));   // graph.cc:1855-1857
    CU(rs.d_cov_thr.reserve(cthr.size() * 8, 0, false, ctx->stream));
    CU(cudaMemcpyAsync(rs.d_cov_thr.p, cthr.data(), cthr.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaEventCreate(&rs.ev0));
  CU(cudaEventCreate(&rs.ev1));
  for (int m = 0; m < rs.n_mates; m++) {
    rs.mate[m].table_index = (int)ctx->stores.size();
    ctx->stores.push_back(&rs.mate[m]);
  }
  ctx->tables_dirty = true;
  ctx->sets.push_back(std::move(rsp));
  return (int)ctx->sets.size() - 1;
}

static int insert_common(gaml_ctx* ctx, int set, int mate, const int32_t* key, int32_t key_len, MateStore** out_store,
                         ReadSetState** out_rs) {
  if (set < 0 || set >= (int)ctx->sets.size()) return fail(ctx, GAML_ERR_ARG, "bad read set index");
  ReadSetState& rs = *ctx->sets[set];
  if (mate < 0 || mate >= rs.n_mates) return fail(ctx, GAML_ERR_ARG, "bad mate index");
  if (!key || key_len <= 0) return fail(ctx, GAML_ERR_ARG, "empty key");
  *out_store = &rs.mate[mate];
  *out_rs = &rs;
  return GAML_OK;
}

int gaml_cache_insert(gaml_ctx* ctx, int set, int mate, const int32_t* key, int32_t key_len,
                      const gaml_alignment* records, int64_t n_records, int32_t key_max_position) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  MateStore* st;
  ReadSetState* rs;
  int rc = insert_common(ctx, set, mate, key, key_len, &st, &rs);
  if (rc) return rc;
  if (st->is_long) return fail(ctx, GAML_ERR_ARG, "use gaml_cache_insert_pacbio for pacbio sets");
  if (n_records < 0 || (n_records > 0 && !records)) return fail(ctx, GAML_ERR_ARG, "bad records");
  Walk k(key, key + key_len);
  if (st->key_ids.count(k)) return fail(ctx, GAML_ERR_KEY_EXISTS, "cache key inserted twice");
  KeyMeta km;
  km.arena_off = (uint32_t)st->total_records();
  int mx = INT_MIN;
  // every record is checked BEFORE anything is staged: a rejected call leaves the store untouched (records of reads
  // outside this shard are only checked for what does not need their length)
  for (int64_t i = 0; i < n_records; i++) {
    const gaml_alignment& a = records[i];
    if (a.read_id < 0 || a.read_id >= rs->n_total) return fail(ctx, GAML_ERR_ARG, "record read_id out of range");
    if (a.orientation != 0 && a.orientation != 1) return fail(ctx, GAML_ERR_ARG, "record orientation must be 0 or 1");
    if (a.edit_dist < 0 || a.edit_dist > 0xffff) return fail(ctx, GAML_ERR_ARG, "record edit_dist outside the pow tables");
    if (a.read_id < rs->lo || a.read_id >= rs->hi) continue;
    if (a.edit_dist > rs->len[mate][(size_t)(a.read_id - rs->lo)]) return fail(ctx, GAML_ERR_ARG, "edit_dist larger than the read length");
  }
  for (int64_t i = 0; i < n_records; i++) {
    const gaml_alignment& a = records[i];
    mx = std::max(mx, a.position);
    if (a.read_id < rs->lo || a.read_id >= rs->hi) continue;
    const int local = (int)(a.read_id - rs->lo);
    int4 v;
    v.x = local;
    v.y = a.position;
    v.z = a.edit_dist | (a.orientation << 30);
    v.w = (int)st->keys.size();
    st->pending.push_back(v);
    km.count++;
  }
  if (key_max_position != INT_MIN) {
    km.any = true;
    km.max_pos = key_max_position;
  } else {
    km.any = n_records > 0;
    km.max_pos = n_records > 0 ? mx : 0;
  }
  st->key_hash_log.push_back(hash_nodes(k.data(), (int)k.size()));
  auto ins = st->key_ids.emplace(std::move(k), (int)st->keys.size());
  st->key_by_id.push_back(&ins.first->first);
  st->keys.push_back(km);
  st->dirty = true;
  return GAML_OK;
}

int gaml_cache_insert_pacbio(gaml_ctx* ctx, int set, const int32_t* key, int32_t key_len,
                             const gaml_pacbio_alignment* records, int64_t n_records) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  MateStore* st;
  ReadSetState* rs;
  int rc = insert_common(ctx, set, 0, key, key_len, &st, &rs);
  if (rc) return rc;
  if (!st->is_long) return fail(ctx, GAML_ERR_ARG, "not a pacbio set");
  if (n_records < 0 || (n_records > 0 && !records)) return fail(ctx, GAML_ERR_ARG, "bad records");
  Walk k(key, key + key_len);
  if (st->key_ids.count(k)) return fail(ctx, GAML_ERR_KEY_EXISTS, "cache key inserted twice");
  KeyMeta km;
  km.arena_off = (uint32_t)st->total_records();
  for (int64_t i = 0; i < n_records; i++)   // checked before anything is staged
    if (records[i].read_id < 0 || records[i].read_id >= rs->n_total) return fail(ctx, GAML_ERR_ARG, "record read_id out of range");
  for (int64_t i = 0; i < n_records; i++) {
    const gaml_pacbio_alignment& a = records[i];
    if (a.read_id < rs->lo || a.read_id >= rs->hi) continue;
    ArenaLong al;
    al.read = (int)(a.read_id - rs->lo);
    al.key = (int)st->keys.size();
    al.logprob = a.logprob;
    int4 v;
    memcpy(&v, &al, 16);
    st->pending.push_back(v);
    st->pending_pos.push_back(Int2{a.position, a.position_end});
    km.count++;
  }
  km.any = n_records > 0;
  st->key_ids.emplace(std::move(k), (int)st->keys.size());
  st->keys.push_back(km);
  st->dirty = true;
  return GAML_OK;
}

// ---- flat on-disk cache (SURVEY §8f rank 4): the stores of one read set exactly as they sit in memory ---------------
// File: "GAMLCC01", {int32 kind, int32 n_mates, int64 n_total, int64 lo, int64 hi}; per mate {int64 n_keys, int64
// n_records}, per key {int32 key_len, key_len x int32 node ids, uint32 count, int32 max_pos, int32 any}, then the
// key-major arena, 16 bytes per record (PacBio stores: then {position, position_end}, 8 bytes per record) — which is what
// the device holds, so loading is one read + one upload.
namespace {
struct CacheFileHeader { char magic[8]; int32_t kind, n_mates; int64_t n_total, lo, hi; };
struct FileCloser { FILE* f; ~FileCloser() { if (f) fclose(f); } };
}  // namespace

int gaml_cache_save(gaml_ctx* ctx, int set, const char* path) {
  if (check_ctx(ctx) || !path) return GAML_ERR_ARG;
  if (set < 0 || set >= (int)ctx->sets.size()) return fail(ctx, GAML_ERR_ARG, "no such read set");
  cudaSetDevice(ctx->device);
  int rc = commit(ctx);
  if (rc != GAML_OK) return rc;
  ReadSetState& rs = *ctx->sets[set];
  FileCloser fc{fopen(path, "wb")};
  if (!fc.f) return fail(ctx, GAML_ERR_ARG, std::string("cannot open ") + path + " for writing");
  CacheFileHeader h{};
  memcpy(h.magic, "GAMLCC01", 8);
  h.kind = rs.cfg.kind;
  h.n_mates = rs.n_mates;
  h.n_total = rs.n_total;
  h.lo = rs.lo;
  h.hi = rs.hi;
  bool ok = fwrite(&h, sizeof(h), 1, fc.f) == 1;
  std::vector<int4> host;
  for (int m = 0; m < rs.n_mates && ok; m++) {
    MateStore& st = rs.mate[m];
    const int64_t counts[2] = {(int64_t)st.keys.size(), (int64_t)st.arena_n};
    ok = fwrite(counts, sizeof(counts), 1, fc.f) == 1;
    std::vector<const Walk*> by_id(st.keys.size(), nullptr);
    for (const auto& kv : st.key_ids) by_id[kv.second] = &kv.first;
    for (size_t k = 0; k < st.keys.size() && ok; k++) {
      const Walk& w = *by_id[k];
      const int32_t len = (int32_t)w.size();
      const int32_t meta[3] = {(int32_t)st.keys[k].count, st.keys[k].max_pos, st.keys[k].any ? 1 : 0};
      ok = fwrite(&len, 4, 1, fc.f) == 1 && (len == 0 || fwrite(w.data(), 4, (size_t)len, fc.f) == (size_t)len) &&
           fwrite(meta, sizeof(meta), 1, fc.f) == 1;
    }
    host.resize(st.arena_n);
    if (st.arena_n) {
      CU(cudaMemcpyAsync(host.data(), st.arena.p, st.arena_n * 16, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
      if (rs.perm_valid)   // the file speaks the caller's read ids
        for (int4& v : host) v.x = (int)rs.h_perm[(size_t)v.x];
      ok = ok && fwrite(host.data(), 16, st.arena_n, fc.f) == st.arena_n;
      if (st.is_long) {   // {position, position_end} of every record, after the arena
        std::vector<Int2> pos(st.arena_n);
        CU(cudaMemcpyAsync(pos.data(), st.arena_pos.p, st.arena_n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        ok = ok && fwrite(pos.data(), 8, st.arena_n, fc.f) == st.arena_n;
      }
    }
  }
  if (!ok) return fail(ctx, GAML_ERR_ARG, std::string("short write to ") + path);
  return GAML_OK;
}

int gaml_cache_load(gaml_ctx* ctx, int set, const char* path) {
  if (check_ctx(ctx) || !path) return GAML_ERR_ARG;
  if (set < 0 || set >= (int)ctx->sets.size()) return fail(ctx, GAML_ERR_ARG, "no such read set");
  ReadSetState& rs = *ctx->sets[set];
  for (int m = 0; m < rs.n_mates; m++)
    if (!rs.mate[m].keys.empty()) return fail(ctx, GAML_ERR_STATE, "gaml_cache_load needs an empty read set");
  FileCloser fc{fopen(path, "rb")};
  if (!fc.f) return fail(ctx, GAML_ERR_ARG, std::string("cannot open ") + path);
  CacheFileHeader h{};
  if (fread(&h, sizeof(h), 1, fc.f) != 1 || memcmp(h.magic, "GAMLCC01", 8) != 0) return fail(ctx, GAML_ERR_ARG, "not a gaml_b200 cache file");
  if (h.kind != rs.cfg.kind || h.n_mates != rs.n_mates || h.n_total != rs.n_total || h.lo != rs.lo || h.hi != rs.hi)
    return fail(ctx, GAML_ERR_ARG, "cache file was written for a different read set (kind, read count or shard)");
  const int n_nodes = (int)ctx->node_len.size();
  // The whole file is parsed and checked into temporaries first — with the checks gaml_cache_insert applies to every
  // record — and moved into the stores only when all of it is sound: a corrupt or stale file leaves the read set empty
  // (so that loading can be retried) and can never plant an out-of-table edit distance on the device.
  struct Loaded {
    std::unordered_map<Walk, int, WalkHash> key_ids;
    std::vector<KeyMeta> keys;
    std::vector<int4> pending;
    std::vector<Int2> pending_pos;
  } tmp[2];
  for (int m = 0; m < rs.n_mates; m++) {
    const bool is_long = rs.mate[m].is_long;
    Loaded& ld = tmp[m];
    int64_t counts[2];
    if (fread(counts, sizeof(counts), 1, fc.f) != 1 || counts[0] < 0 || counts[1] < 0 || counts[1] > 0xfffffff0ll)
      return fail(ctx, GAML_ERR_ARG, "corrupt cache file (store header)");
    uint64_t off = 0;
    Walk w;
    for (int64_t k = 0; k < counts[0]; k++) {
      int32_t len, meta[3];
      if (fread(&len, 4, 1, fc.f) != 1 || len <= 0 || len > (1 << 20)) return fail(ctx, GAML_ERR_ARG, "corrupt cache file (key length)");
      w.resize((size_t)len);
      if (fread(w.data(), 4, (size_t)len, fc.f) != (size_t)len || fread(meta, sizeof(meta), 1, fc.f) != 1)
        return fail(ctx, GAML_ERR_ARG, "corrupt cache file (key)");
      for (int x : w)
        if (x >= n_nodes && n_nodes > 0) return fail(ctx, GAML_ERR_ARG, "cache key references a node outside the graph");
      if (meta[0] < 0) return fail(ctx, GAML_ERR_ARG, "corrupt cache file (key record count)");
      KeyMeta km;
      km.arena_off = (uint32_t)off;
      km.count = (uint32_t)meta[0];
      km.max_pos = meta[1];
      km.any = meta[2] != 0;
      off += km.count;
      if (!ld.key_ids.emplace(w, (int)ld.keys.size()).second) return fail(ctx, GAML_ERR_ARG, "corrupt cache file (duplicate key)");
      ld.keys.push_back(km);
    }
    if (off != (uint64_t)counts[1]) return fail(ctx, GAML_ERR_ARG, "corrupt cache file (record count)");
    ld.pending.resize((size_t)counts[1]);
    if (counts[1] && fread(ld.pending.data(), 16, (size_t)counts[1], fc.f) != (size_t)counts[1])
      return fail(ctx, GAML_ERR_ARG, "corrupt cache file (records)");
    if (is_long) {
      ld.pending_pos.resize((size_t)counts[1]);
      if (counts[1] && fread(ld.pending_pos.data(), 8, (size_t)counts[1], fc.f) != (size_t)counts[1])
        return fail(ctx, GAML_ERR_ARG, "corrupt cache file (record positions)");
    }
    size_t at = 0;
    for (size_t k = 0; k < ld.keys.size(); k++) {   // records are key-major: record `at` must carry key k
      for (uint32_t t = 0; t < ld.keys[k].count; t++, at++) {
        const int4& v = ld.pending[at];   // {read, pos, edor, key} / {read, key, logprob}
        const int key = is_long ? v.y : v.w;
        if (v.x < 0 || v.x >= rs.n_local || key != (int)k) return fail(ctx, GAML_ERR_ARG, "corrupt cache file (record)");
        if (!is_long) {
          const int ed = v.z & 0xffff;
          if ((v.z & ~(0xffff | (1 << 30))) != 0 || ed > rs.len[m][(size_t)v.x])
            return fail(ctx, GAML_ERR_ARG, "corrupt cache file (record edit distance / orientation)");
        }   // (PacBio {position, position_end} are only ever used arithmetically, never as indices)
      }
    }
  }
  for (int m = 0; m < rs.n_mates; m++) {
    MateStore& st = rs.mate[m];
    st.key_ids = std::move(tmp[m].key_ids);
    st.keys = std::move(tmp[m].keys);
    st.key_hash_log.assign(st.keys.size(), 0);
    st.key_by_id.assign(st.keys.size(), nullptr);
    for (const auto& kv : st.key_ids) {
      st.key_hash_log[(size_t)kv.second] = hash_nodes(kv.first.data(), (int)kv.first.size());
      st.key_by_id[(size_t)kv.second] = &kv.first;
    }
    st.pending = std::move(tmp[m].pending);
    st.pending_pos = std::move(tmp[m].pending_pos);
    st.dirty = true;
  }
  return GAML_OK;
}

// ---- PacBio alignment probability (SURVEY §8f rank 3) ---------------------------------------------------------------
// The host only summarises each CIGAR (O(#operations)): the leading / trailing insertion runs (GetCigarEnds,
// graph.cc:2136-2149), where the path ends, and a bound on a row's width for the scratch strips. The cells themselves
// are derived on the device while the DP runs (kernels.cu).
int gaml_pacbio_alignment_logprob(gaml_ctx* ctx, double match_prob, double mismatch_prob, int32_t band, int64_t n,
                                  const uint8_t* s1, const int64_t* s1_off, const uint8_t* s2, const int64_t* s2_off,
                                  const int32_t* posstart, const int32_t* op_len, const uint8_t* op_chr, const int64_t* op_off,
                                  double* logprob_out) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (n < 0 || band < 0 || !(match_prob > 0.0) || !(mismatch_prob > 0.0))
    return fail(ctx, GAML_ERR_ARG, "bad alignment-probability arguments");
  if (band > kAlnMaxBand) return fail(ctx, GAML_ERR_UNSUPPORTED, "band larger than 8 (the reference uses 2, graph.cc:2755)");
  if (n == 0) return GAML_OK;
  if (!s1 || !s1_off || !s2 || !s2_off || !posstart || !op_len || !op_chr || !op_off || !logprob_out)
    return fail(ctx, GAML_ERR_ARG, "NULL array");
  cudaSetDevice(ctx->device);
  const auto t_host0 = std::chrono::steady_clock::now();
  std::vector<AlnMeta> meta((size_t)n);
  int64_t scratch = 0;
  for (int64_t a = 0; a < n; a++) {
    const int64_t k0 = op_off[a], k1 = op_off[a + 1];
    if (k1 < k0 || k1 - k0 > 0x7fffffff) return fail(ctx, GAML_ERR_ARG, "cigar offsets not ascending");
    int64_t rows = 0, cols = 0, lead = 0, trail = 0, run = 0, max_run = 0;
    bool seen = false;
    for (int64_t k = k0; k < k1; k++) {
      const int64_t len = op_len[k];
      const uint8_t c = op_chr[k];
      if (len < 0 || (c != 'M' && c != 'I' && c != 'D')) return fail(ctx, GAML_ERR_ARG, "cigar operations must be M, I or D with non-negative lengths");
      if (len == 0) continue;
      if (c == 'I') {
        cols += len;
        run += len;
        trail += len;
        if (!seen) lead += len;
      } else {
        rows += len;
        if (c == 'M') cols += len;
        seen = true;
        run = 0;
        trail = 0;
      }
      max_run = std::max(max_run, run);
    }
    if (rows > 0x3fffffff || cols > 0x3fffffff) return fail(ctx, GAML_ERR_CAPACITY, "alignment too long");
    AlnMeta& m = meta[(size_t)a];
    m.s1_off = s1_off[a];
    m.s1_len = (int32_t)(s1_off[a + 1] - s1_off[a]);
    m.s2_off = s2_off[a];
    m.s2_len = (int32_t)(s2_off[a + 1] - s2_off[a]);
    m.op_off = k0;
    m.n_ops = (int32_t)(k1 - k0);
    m.posstart = posstart[a];
    m.bl = seen ? (int32_t)std::min<int64_t>(lead, 200) : 0;
    m.el = seen ? (int32_t)std::min<int64_t>(trail + 1, 200) : 0;
    m.row_end = (int32_t)rows;
    m.col_end = (int32_t)cols;
    // a row's cells span at most 2*band+1 path rows (2*band diagonal steps and their insertion runs), the band on both
    // sides, and one of the two blocks
    const int64_t w = 4 * (int64_t)band + 3 + (2 * (int64_t)band + 1) * max_run + std::max<int64_t>(m.bl, m.el + 1);
    if (w > 0x0fffffff) return fail(ctx, GAML_ERR_CAPACITY, "insertion run too long");
    m.width = (int32_t)w;
    m.scratch_off = scratch;
    scratch += 2 * w;
    m.pad[0] = m.pad[1] = m.pad[2] = 0;
  }
  cudaStream_t st = ctx->stream;
  const size_t n1 = (size_t)s1_off[n], n2 = (size_t)s2_off[n], n_ops = (size_t)op_off[n];
  DevBuf &d_meta = ctx->d_aln[0], &d_s1 = ctx->d_aln[1], &d_s2 = ctx->d_aln[2], &d_len = ctx->d_aln[3], &d_chr = ctx->d_aln[4],
         &d_scratch = ctx->d_aln[5], &d_out = ctx->d_aln[6], &d_flag = ctx->d_aln[7];   // kept between calls
  CU(d_meta.reserve(meta.size() * sizeof(AlnMeta), 0, false, st));
  CU(d_s1.reserve(std::max<size_t>(n1, 1), 0, false, st));
  CU(d_s2.reserve(std::max<size_t>(n2, 1), 0, false, st));
  CU(d_len.reserve(std::max<size_t>(n_ops, 1) * 4, 0, false, st));
  CU(d_chr.reserve(std::max<size_t>(n_ops, 1), 0, false, st));
  CU(d_scratch.reserve(std::max<int64_t>(scratch, 1) * 8, 0, false, st));
  CU(d_out.reserve((size_t)n * 8, 0, false, st));
  CU(d_flag.reserve(256, 0, true, st));
  CU(cudaMemsetAsync(d_flag.p, 0, 4, st));
  CU(cudaMemcpyAsync(d_meta.p, meta.data(), meta.size() * sizeof(AlnMeta), cudaMemcpyHostToDevice, st));
  if (n1) CU(cudaMemcpyAsync(d_s1.p, s1, n1, cudaMemcpyHostToDevice, st));
  if (n2) CU(cudaMemcpyAsync(d_s2.p, s2, n2, cudaMemcpyHostToDevice, st));
  if (n_ops) {
    CU(cudaMemcpyAsync(d_len.p, op_len, n_ops * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_chr.p, op_chr, n_ops, cudaMemcpyHostToDevice, st));
  }
  AlnProbParams A{};
  A.meta = d_meta.as<AlnMeta>();
  A.n = n;
  A.s1 = d_s1.as<unsigned char>();
  A.s2 = d_s2.as<unsigned char>();
  A.op_len = d_len.as<int32_t>();
  A.op_chr = d_chr.as<unsigned char>();
  A.band = band;
  A.scratch = d_scratch.as<double>();
  A.log_match = log(match_prob);
  A.log_mismatch = log(mismatch_prob);
  A.out = d_out.as<double>();
  A.error_flag = d_flag.as<uint32_t>();
  ctx->stats.last_prepare_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_host0).count();
  CU(cudaEventRecord(ctx->ev[0], st));
  launch_pacbio_alnprob(A, ctx->sm_count, st);
  CU(cudaEventRecord(ctx->ev[3], st));
  CU(cudaGetLastError());
  ctx->stats.kernel_launches += 1;
  uint32_t flag = 0;
  CU(cudaMemcpyAsync(logprob_out, d_out.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(&flag, d_flag.p, 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  float ms = 0;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[3]);
  ctx->stats.last_device_ms = ms;   // the DP kernel alone
  ctx->timing_pending = false;
  if (flag & 1u) return fail(ctx, GAML_ERR_CAPACITY, "an alignment's row was wider than the scratch strip bound");
  return GAML_OK;
}

int gaml_cache_contains(gaml_ctx* ctx, int set, int mate, const int32_t* key, int32_t key_len) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  MateStore* st;
  ReadSetState* rs;
  int rc = insert_common(ctx, set, mate, key, key_len, &st, &rs);
  if (rc) return rc;
  return st->key_ids.count(Walk(key, key + key_len)) ? 1 : 0;
}

int gaml_cache_commit(gaml_ctx* ctx) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  return commit(ctx);
}

int gaml_eval_prepare(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = prepare(ctx, walk_nodes, walk_offsets, n_walks);
  ctx->stats.last_prepare_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int gaml_eval_launch(gaml_ctx* ctx) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = launch(ctx);
  ctx->stats.last_launch_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int gaml_eval_finish(gaml_ctx* ctx, double* partials, int32_t* total_len) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = finish(ctx, partials, total_len);
  ctx->stats.last_finish_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int gaml_eval_finish_gathered(gaml_ctx* ctx, double* gathered, int32_t* total_len) {
  if (check_ctx(ctx) || !gathered) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = finish(ctx, nullptr, total_len, gathered);
  ctx->stats.last_finish_host_us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int gaml_calc_prob_gathered(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks,
                            double* gathered, int32_t* total_len) {
  int rc = gaml_eval_prepare(ctx, walk_nodes, walk_offsets, n_walks);
  if (rc) return rc;
  rc = gaml_eval_launch(ctx);
  if (rc) return rc;
  return gaml_eval_finish_gathered(ctx, gathered, total_len);
}

int gaml_set_result_exchange(gaml_ctx* ctx, void* shared_base, int64_t bytes, int32_t rank, int32_t world) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->prepared || ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is pending");
  if (ctx->exch_host) {
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->exch_owned) cudaHostUnregister(ctx->exch_host);
    ctx->exch_host = ctx->exch_dev = nullptr;
    ctx->exch_world = 1;
    ctx->exch_rank = 0;
  }
  if (!shared_base) return GAML_OK;
  const int64_t need = 2ll * world * GAML_EXCHANGE_MAX_SETS * kResultStride * (int64_t)sizeof(double);
  if (world < 1 || rank < 0 || rank >= world || bytes < need)
    return fail(ctx, GAML_ERR_ARG, "result exchange: need 2 * world * GAML_EXCHANGE_MAX_SETS * 64 bytes and 0 <= rank < world");
  if (ctx->sets.size() > GAML_EXCHANGE_MAX_SETS) return fail(ctx, GAML_ERR_CAPACITY, "more read sets than GAML_EXCHANGE_MAX_SETS");
  {
    // (two contexts of ONE process may share a segment — the tests do: the second registration finds it mapped already)
    const cudaError_t e = cudaHostRegister(shared_base, (size_t)need, cudaHostRegisterMapped | cudaHostRegisterPortable);
    ctx->exch_owned = e == cudaSuccess;
    if (e == cudaErrorHostMemoryAlreadyRegistered) cudaGetLastError();
    else CU(e);
  }
  void* dev = nullptr;
  CU(cudaHostGetDevicePointer(&dev, shared_base, 0));
  ctx->exch_host = static_cast<double*>(shared_base);
  ctx->exch_dev = static_cast<double*>(dev);
  ctx->exch_rank = rank;
  ctx->exch_world = world;
  return GAML_OK;
}

// ---- result exchange over peer memory (NVLink) -------------------------------------------------------------------
static void peer_exchange_release(gaml_ctx* ctx) {
  for (size_t p = 0; p < ctx->peer_ptrs.size(); p++)
    if (ctx->peer_opened[p] && ctx->peer_ptrs[p]) cudaIpcCloseMemHandle(ctx->peer_ptrs[p]);
  ctx->peer_ptrs.clear();
  ctx->peer_opened.clear();
  ctx->peer_on = false;
}

int gaml_peer_exchange_create(gaml_ctx* ctx, int32_t rank, int32_t world, void* ipc_handle_out, void** buffer_out) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->prepared || ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is pending");
  if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(ctx, GAML_ERR_ARG, "peer exchange: 0 <= rank < world <= 64");
  if (ctx->sets.size() > GAML_EXCHANGE_MAX_SETS) return fail(ctx, GAML_ERR_CAPACITY, "more read sets than GAML_EXCHANGE_MAX_SETS");
  CU(cudaStreamSynchronize(ctx->stream));
  peer_exchange_release(ctx);
  const size_t bytes = 2 * (size_t)world * GAML_EXCHANGE_MAX_SETS * kResultStride * sizeof(double);
  if (!ctx->d_peer_lines.p) {   // allocated once per context: an exported buffer is never moved
    CU(ctx->d_peer_lines.reserve(2 * (size_t)64 * GAML_EXCHANGE_MAX_SETS * kResultStride * sizeof(double), 0, true, ctx->stream));
  }
  CU(cudaMemsetAsync(ctx->d_peer_lines.p, 0, bytes, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ctx->d_peer_lines.p));
    static_assert(sizeof(h) == GAML_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(ipc_handle_out, &h, sizeof(h));
  }
  if (buffer_out) *buffer_out = ctx->d_peer_lines.p;
  ctx->peer_rank = rank;
  ctx->peer_world = world;
  return GAML_OK;
}

int gaml_peer_exchange_open(gaml_ctx* ctx, const void* ipc_handles, void* const* local_buffers) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->prepared || ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is pending");
  if (ctx->peer_world < 1 || !ctx->d_peer_lines.p) return fail(ctx, GAML_ERR_STATE, "gaml_peer_exchange_create first");
  peer_exchange_release(ctx);
  const int world = ctx->peer_world;
  ctx->peer_ptrs.assign(world, nullptr);
  ctx->peer_opened.assign(world, 0);
  for (int p = 0; p < world; p++) {
    if (p == ctx->peer_rank) {
      ctx->peer_ptrs[p] = ctx->d_peer_lines.p;
    } else if (local_buffers && local_buffers[p]) {
      // another context of this process, on ANOTHER GPU (IPC handles cannot be opened by their creator; a kernel that
      // waits for a line must not share its GPU with the kernel that writes it)
      cudaPointerAttributes attr{};
      CU(cudaPointerGetAttributes(&attr, local_buffers[p]));
      if (attr.device == ctx->device) {
        peer_exchange_release(ctx);
        return fail(ctx, GAML_ERR_ARG, "peer exchange: two ranks on one GPU (their kernels would wait on one another)");
      }
      const cudaError_t pe = cudaDeviceEnablePeerAccess(attr.device, 0);
      if (pe == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (pe != cudaSuccess) {
        peer_exchange_release(ctx);
        return fail(ctx, GAML_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(pe));
      }
      ctx->peer_ptrs[p] = local_buffers[p];
    } else if (ipc_handles) {
      cudaIpcMemHandle_t h;
      memcpy(&h, static_cast<const char*>(ipc_handles) + (size_t)p * GAML_IPC_HANDLE_BYTES, sizeof(h));
      void* ptr = nullptr;
      const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        peer_exchange_release(ctx);
        return fail(ctx, GAML_ERR_CUDA, std::string("cudaIpcOpenMemHandle (peer access between the GPUs is required): ") + cudaGetErrorString(e));
      }
      ctx->peer_ptrs[p] = ptr;
      ctx->peer_opened[p] = 1;
    } else {
      peer_exchange_release(ctx);
      return fail(ctx, GAML_ERR_ARG, "peer exchange: no handle or buffer for a rank");
    }
  }
  CU(ctx->d_peer_table.reserve(64 * sizeof(void*), 0, false, ctx->stream));
  CU(cudaMemcpyAsync(ctx->d_peer_table.p, ctx->peer_ptrs.data(), (size_t)world * sizeof(void*), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  int rc = ensure_gather_area(ctx, world);
  if (rc != GAML_OK) return rc;
  ctx->peer_on = true;
  return GAML_OK;
}

int gaml_peer_exchange_close(gaml_ctx* ctx) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  peer_exchange_release(ctx);
  return GAML_OK;
}

// ---- result exchange through NCCL --------------------------------------------------------------------------------
int gaml_nccl_unique_id(void* out128) {
  if (!out128) return GAML_ERR_ARG;
  NcclApi* api = nccl_api(&g_create_error);
  if (!api) return GAML_ERR_STATE;
  NcclId id;
  if (api->get_unique_id(&id) != 0) {
    g_create_error = "ncclGetUniqueId failed";
    return GAML_ERR_CUDA;
  }
  memcpy(out128, &id, sizeof(id));
  return GAML_OK;
}

int gaml_nccl_exchange_init(gaml_ctx* ctx, const void* unique_id128, int32_t rank, int32_t world) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->prepared || ctx->launched) return fail(ctx, GAML_ERR_STATE, "an evaluation is pending");
  NcclApi* api = nccl_api(&ctx->error);
  if (!api) return GAML_ERR_STATE;
  if (ctx->nccl_comm) {
    cudaStreamSynchronize(ctx->stream);
    api->comm_destroy(ctx->nccl_comm);
    ctx->nccl_comm = nullptr;
    ctx->nccl_on = false;
  }
  if (!unique_id128) return GAML_OK;   // detach
  if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(ctx, GAML_ERR_ARG, "nccl exchange: 0 <= rank < world <= 64");
  NcclId id;
  memcpy(&id, unique_id128, sizeof(id));
  const int rc = api->comm_init_rank(&ctx->nccl_comm, world, id, rank);
  if (rc != 0) return fail(ctx, GAML_ERR_CUDA, std::string("ncclCommInitRank: ") + (api->get_error_string ? api->get_error_string(rc) : "error"));
  const size_t bytes = (size_t)GAML_EXCHANGE_MAX_SETS * kResultStride * sizeof(double);
  CU(ctx->d_part.reserve(bytes, 0, true, ctx->stream));
  CU(ctx->d_part_sum.reserve(bytes, 0, true, ctx->stream));
  int rc2 = ensure_gather_area(ctx, world);
  if (rc2 != GAML_OK) return rc2;
  ctx->nccl_rank = rank;
  ctx->nccl_world = world;
  ctx->nccl_on = true;
  return GAML_OK;
}

int gaml_calc_prob_partial(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks,
                           double* partials, int32_t* total_len) {
  // A capacity error (scratch arena / overflow list too small for this walk set) enlarges the buffer and invalidates the
  // incremental state; the reference never fails here, so the call repeats the evaluation — a full re-score — itself.
  // (Not with a result exchange attached: the ranks count evaluations in lockstep.)
  for (int attempt = 0;; attempt++) {
    int rc = gaml_eval_prepare(ctx, walk_nodes, walk_offsets, n_walks);
    if (rc) return rc;
    rc = gaml_eval_launch(ctx);
    if (rc) return rc;
    rc = gaml_eval_finish(ctx, partials, total_len);
    if (rc != GAML_ERR_CAPACITY || !ctx->capacity_grew || ctx->exch_host || ctx->peer_on || ctx->nccl_on || attempt >= 6) return rc;
  }
}

int gaml_combine_partials(gaml_ctx* ctx, const double* gathered, int32_t n_shards, int32_t total_len, gaml_result* result,
                          int32_t* zeros) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  return combine(ctx, gathered, n_shards, total_len, result, zeros);
}

int gaml_combine_partials_raw(const double* gathered, int32_t n_shards, int32_t n_sets, const int32_t* kinds,
                              const int64_t* n_reads_total, const double* weights, int32_t total_len,
                              gaml_result* result, int32_t* zeros) {
  return combine_raw(gathered, n_shards, n_sets, kinds, n_reads_total, weights, total_len, result, zeros);
}

int gaml_calc_prob(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks,
                   gaml_result* result, int32_t* zeros) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (!result) return fail(ctx, GAML_ERR_ARG, "result is NULL");
  for (auto& rs : ctx->sets)
    if (rs->lo != 0 || rs->hi != rs->n_total)
      return fail(ctx, GAML_ERR_STATE, "gaml_calc_prob on a sharded context: use gaml_calc_prob_partial + gaml_combine_partials");
  std::vector<double> partials(std::max<size_t>(ctx->sets.size(), 1) * GAML_PARTIAL_DOUBLES);
  int32_t tl = 0;
  int rc = gaml_calc_prob_partial(ctx, walk_nodes, walk_offsets, n_walks, partials.data(), &tl);
  if (rc) return rc;
  return combine(ctx, partials.data(), 1, tl, result, zeros);
}

int gaml_calc_prob_batch_partial(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                                 const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                                 double* partials, int32_t* total_lens) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  cudaSetDevice(ctx->device);
  return calc_prob_batch_partial(ctx, n_cand, erased_idx, erased_off, added_nodes, added_walk_off, cand_added_off, partials,
                                 total_lens);
}

int gaml_calc_prob_batch(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                         const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off, double* probs,
                         int32_t* total_lens, int32_t* zeros) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (!probs || n_cand <= 0) return fail(ctx, GAML_ERR_ARG, "bad batch arguments");
  for (auto& rs : ctx->sets)
    if (rs->lo != 0 || rs->hi != rs->n_total)
      return fail(ctx, GAML_ERR_STATE, "gaml_calc_prob_batch on a sharded context: use gaml_calc_prob_batch_partial + gaml_combine_partials");
  const size_t n_sets = ctx->sets.size();
  std::vector<double> partials((size_t)n_cand * std::max<size_t>(n_sets, 1) * GAML_PARTIAL_DOUBLES);
  std::vector<int32_t> tls(n_cand);
  int rc = gaml_calc_prob_batch_partial(ctx, n_cand, erased_idx, erased_off, added_nodes, added_walk_off, cand_added_off,
                                        partials.data(), tls.data());
  if (rc) return rc;
  for (int c = 0; c < n_cand; c++) {
    gaml_result res;
    rc = combine(ctx, partials.data() + (size_t)c * n_sets * GAML_PARTIAL_DOUBLES, 1, tls[c], &res,
                 zeros ? zeros + (size_t)c * 2 * n_sets : nullptr);
    if (rc) return rc;
    probs[c] = res.prob;
    if (total_lens) total_lens[c] = tls[c];
  }
  return GAML_OK;
}

int gaml_calc_prob_batch_gathered(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                                  const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off, double* probs,
                                  int32_t* total_lens, int32_t* zeros) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (!probs || n_cand <= 0) return fail(ctx, GAML_ERR_ARG, "bad batch arguments");
  if (!ctx->nccl_comm) return fail(ctx, GAML_ERR_STATE, "gaml_calc_prob_batch_gathered needs gaml_nccl_exchange_init");
  cudaSetDevice(ctx->device);
  const size_t n_sets = ctx->sets.size();
  std::vector<double> partials((size_t)n_cand * std::max<size_t>(n_sets, 1) * GAML_PARTIAL_DOUBLES);
  std::vector<int32_t> tls(n_cand);
  int rc = calc_prob_batch_partial(ctx, n_cand, erased_idx, erased_off, added_nodes, added_walk_off, cand_added_off, partials.data(),
                                   tls.data(), true);
  if (rc) return rc;
  for (int c = 0; c < n_cand; c++) {   // the partials are the sums over all shards already: one "shard" to combine
    gaml_result res;
    rc = combine(ctx, partials.data() + (size_t)c * n_sets * GAML_PARTIAL_DOUBLES, 1, tls[c], &res,
                 zeros ? zeros + (size_t)c * 2 * n_sets : nullptr);
    if (rc) return rc;
    probs[c] = res.prob;
    if (total_lens) total_lens[c] = tls[c];
  }
  return GAML_OK;
}

// ---- coverage penalty of a read set on a read-id shard (SURVEY §8f rank 1) --------------------------------------------
// Paired sets: one 64-bit event key per covered position (walk << 33 | position << 1 | 1, kernels.cu cov_key).
// PacBio sets: two words per interval {(walk << 32 | start), end}.
int gaml_penalty_export(gaml_ctx* ctx, int set, uint64_t* out, int64_t cap, int64_t* n_out) {
  if (check_ctx(ctx) || !n_out) return GAML_ERR_ARG;
  if (set < 0 || set >= (int)ctx->sets.size()) return fail(ctx, GAML_ERR_ARG, "no such read set");
  ReadSetState& rs = *ctx->sets[set];
  if (!rs.penalty_pending) return fail(ctx, GAML_ERR_STATE, "no pending coverage events: the set is not a penalised shard, or no evaluation has finished");
  cudaSetDevice(ctx->device);
  const SetPlan& sp = ctx->plan[set];
  CU(cudaStreamSynchronize(ctx->stream));
  if (rs.penalty) {
    uint32_t count = 0;
    const size_t ns = std::max<size_t>(ctx->sets.size(), 1);
    const unsigned long long* accum = ctx->d_flags.as<unsigned long long>() + 2 + 8 * ns + (size_t)set * kAccumStride;
    CU(cudaMemcpy(&count, accum + 7, 4, cudaMemcpyDeviceToHost));
    if (count > sp.ev_cap) return fail(ctx, GAML_ERR_CAPACITY, "coverage-event buffer exhausted");
    const int64_t n = (int64_t)count - sp.n_type1;   // the host's contig-start events lead the buffer: every rank has them
    *n_out = n;
    if (n > cap) return fail(ctx, GAML_ERR_CAPACITY, "gaml_penalty_export: output buffer too small (n_out holds the count)");
    if (n > 0) CU(cudaMemcpy(out, rs.d_ev.as<unsigned long long>() + sp.n_type1, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return GAML_OK;
  }
  uint32_t count = 0;
  CU(cudaMemcpy(&count, rs.d_pb_count.p, 4, cudaMemcpyDeviceToHost));
  if (count > sp.pb_cap) return fail(ctx, GAML_ERR_CAPACITY, "coverage-interval buffer exhausted");
  *n_out = 2 * (int64_t)count;
  if (2 * (int64_t)count > cap) return fail(ctx, GAML_ERR_CAPACITY, "gaml_penalty_export: output buffer too small (n_out holds the count)");
  std::vector<unsigned long long> ik(count);
  std::vector<int32_t> ie(count);
  if (count) {
    CU(cudaMemcpy(ik.data(), rs.d_pb_ikey.p, (size_t)count * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ie.data(), rs.d_pb_iend.p, (size_t)count * 4, cudaMemcpyDeviceToHost));
  }
  for (uint32_t i = 0; i < count; i++) {
    out[2 * (size_t)i] = ik[i];
    out[2 * (size_t)i + 1] = (uint64_t)(uint32_t)ie[i];
  }
  return GAML_OK;
}

int gaml_penalty_import(gaml_ctx* ctx, int set, const uint64_t* all, int64_t n_all) {
  if (check_ctx(ctx) || n_all < 0 || (n_all > 0 && !all)) return GAML_ERR_ARG;
  if (set < 0 || set >= (int)ctx->sets.size()) return fail(ctx, GAML_ERR_ARG, "no such read set");
  ReadSetState& rs = *ctx->sets[set];
  if (!rs.penalty_pending) return fail(ctx, GAML_ERR_STATE, "no pending coverage events for this read set");
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const SetPlan& sp = ctx->plan[set];
  char* blob = ctx->blob_dev;
  if (rs.penalty) {
    // [contig starts | every shard's covered positions | padding] -> sort -> one thread per event (graph.cc:1893-1919)
    const uint64_t total = (uint64_t)rs.h_type1.size() + (uint64_t)n_all;
    if (total > 0x7fffffffull) return fail(ctx, GAML_ERR_CAPACITY, "too many coverage events");
    const uint32_t cap = (uint32_t)total + 16;
    std::vector<unsigned long long> keys(cap, ~0ull);
    std::copy(rs.h_type1.begin(), rs.h_type1.end(), keys.begin());
    if (n_all) memcpy(keys.data() + rs.h_type1.size(), all, (size_t)n_all * 8);
    CU(rs.d_ev.reserve((size_t)cap * 8, 0, false, st));
    CU(rs.d_ev_sorted.reserve((size_t)cap * 8, 0, false, st));
    CU(rs.d_ev_temp.reserve(std::max<size_t>(coverage_sort_temp_bytes(cap), 256), 0, false, st));
    CU(rs.d_bad.reserve(std::max<size_t>(sp.n_cov_walks, 1) * 4, 0, false, st));
    CU(cudaMemcpyAsync(rs.d_ev.p, keys.data(), (size_t)cap * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(rs.d_bad.p, 0, std::max<size_t>(sp.n_cov_walks, 1) * 4, st));
    CU(launch_coverage(rs.d_ev.as<unsigned long long>(), rs.d_ev_sorted.as<unsigned long long>(), cap, rs.d_ev_temp.p, rs.d_ev_temp.cap,
                       reinterpret_cast<const int*>(blob + sp.csbegin_off), reinterpret_cast<const int*>(blob + sp.cs_off), rs.cfg.step,
                       rs.cfg.insert_mean + 5 * rs.cfg.insert_std, rs.d_bad.as<int>(), ctx->sm_count, st));
    ctx->stats.kernel_launches += 3;
    rs.h_bad.assign(std::max(sp.n_cov_walks, 1), 0);
    if (sp.n_cov_walks) CU(cudaMemcpyAsync(rs.h_bad.data(), rs.d_bad.p, (size_t)sp.n_cov_walks * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (sp.full) rs.bad_bases = 0;   // EraseFromScoringState / AddToScoringState, graph.cc:1938, 1946
    for (int w = 0; w < sp.n_cov_walks; w++) rs.bad_bases += w < sp.n_erased ? -rs.h_bad[w] : rs.h_bad[w];
    rs.penalty_pending = false;
    return GAML_OK;
  }
  // PacBio: the union of the shards' alignment intervals + the artificial and per-node intervals of every walk
  if (n_all & 1) return fail(ctx, GAML_ERR_ARG, "PacBio intervals come as pairs of words");
  const size_t n_int = (size_t)n_all / 2 + rs.h_pb_seeds.size();
  if (n_int > 0x3ffffff0ull) return fail(ctx, GAML_ERR_CAPACITY, "too many PacBio coverage intervals");
  const uint32_t cap = (uint32_t)n_int + 16;
  std::vector<unsigned long long> ikey(cap, ~0ull), pkey(2 * (size_t)cap, ~0ull);
  std::vector<int32_t> iend(cap, -1);
  size_t k = 0;
  auto put = [&](unsigned long long key, int32_t end) {
    ikey[k] = key;
    iend[k] = end;
    pkey[2 * k] = key;
    pkey[2 * k + 1] = (key & 0xffffffff00000000ull) | (unsigned long long)((uint32_t)end ^ 0x80000000u);
    k++;
  };
  for (const int4& sd : rs.h_pb_seeds)   // {walk, start, end, -}
    put(((unsigned long long)(uint32_t)sd.x << 32) | (unsigned long long)((uint32_t)sd.y ^ 0x80000000u), sd.z);
  for (int64_t i = 0; i < n_all; i += 2) put(all[i], (int32_t)(uint32_t)all[i + 1]);
  CU(rs.d_pb_ikey.reserve((size_t)cap * 2 * 8, 0, false, st));
  CU(rs.d_pb_iend.reserve((size_t)cap * 2 * 4, 0, false, st));
  CU(rs.d_pb_pkey.reserve((size_t)cap * 4 * 8, 0, false, st));
  CU(rs.d_pb_packed.reserve((size_t)cap * 8, 0, false, st));
  CU(rs.d_pb_runmax.reserve((size_t)cap * 8, 0, false, st));
  CU(rs.d_pb_temp.reserve(std::max<size_t>(pacbio_coverage_temp_bytes(cap), 256), 0, false, st));
  CU(rs.d_pb_count.reserve(256, 0, true, st));
  CU(rs.d_bad.reserve(256, 0, true, st));
  const uint32_t count = (uint32_t)n_int;
  CU(cudaMemcpyAsync(rs.d_pb_ikey.p, ikey.data(), (size_t)cap * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(rs.d_pb_iend.p, iend.data(), (size_t)cap * 4, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(rs.d_pb_pkey.p, pkey.data(), (size_t)cap * 2 * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(rs.d_pb_count.p, &count, 4, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(rs.d_bad.p, 0, 4, st));
  PbCovParams C{};
  C.ikey = rs.d_pb_ikey.as<unsigned long long>();
  C.iend = rs.d_pb_iend.as<int32_t>();
  C.pkey = rs.d_pb_pkey.as<unsigned long long>();
  C.count = rs.d_pb_count.as<uint32_t>();
  C.cap = cap;
  CU(launch_pacbio_coverage(C, rs.d_pb_packed.as<unsigned long long>(), rs.d_pb_runmax.as<unsigned long long>(), rs.d_pb_temp.p,
                            rs.d_pb_temp.cap, reinterpret_cast<const int*>(blob + sp.pb_len_off), rs.cfg.step, rs.d_bad.as<int>(),
                            ctx->sm_count, st, 2));
  ctx->stats.kernel_launches += 5;
  rs.h_bad.assign(1, 0);
  CU(cudaMemcpyAsync(rs.h_bad.data(), rs.d_bad.p, 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  rs.bad_bases = rs.h_bad[0];
  rs.penalty_pending = false;
  return GAML_OK;
}

int gaml_reset_state(gaml_ctx* ctx) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  for (auto& rs : ctx->sets) {
    rs->has_state = false;
    rs->total_valid = false;
    rs->bad_bases = 0;
  }
  return GAML_OK;
}

int gaml_read_values(gaml_ctx* ctx, int set, double* out, int64_t n) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  if (set < 0 || set >= (int)ctx->sets.size() || !out) return fail(ctx, GAML_ERR_ARG, "bad arguments");
  ReadSetState& rs = *ctx->sets[set];
  if (n != rs.n_local) return fail(ctx, GAML_ERR_ARG, "n must equal the shard's read count");
  cudaSetDevice(ctx->device);
  if (!rs.perm_valid) {
    if (n > 0) CU(cudaMemcpyAsync(out, rs.d_values.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return GAML_OK;
  }
  std::vector<double> tmp((size_t)n);   // the device holds the internal read order
  if (n > 0) CU(cudaMemcpyAsync(tmp.data(), rs.d_values.p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int64_t r = 0; r < n; r++) out[r] = tmp[rs.h_inv[(size_t)r]];
  return GAML_OK;
}

int gaml_set_profiling(gaml_ctx* ctx, int32_t level) {
  if (check_ctx(ctx)) return GAML_ERR_ARG;
  ctx->timed = level == 1 || level == 2;
  ctx->profile = level == 2;
  ctx->timeline = level == 3;
  return GAML_OK;
}

int gaml_read_timeline(gaml_ctx* ctx, double* out_us, int32_t n) {
  if (check_ctx(ctx) || !out_us || n < kTimelineWords) return GAML_ERR_ARG;
  if (!ctx->timeline || !ctx->d_timeline.p) return fail(ctx, GAML_ERR_STATE, "gaml_set_profiling(ctx, 3) and one evaluation first");
  cudaSetDevice(ctx->device);
  CU(cudaMemcpyAsync(ctx->h_timeline, ctx->d_timeline.p, kTimelineWords * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  unsigned long long t0 = ~0ull;
  for (int k = 0; k < kTimelineWords; k += 2)
    if (ctx->h_timeline[k]) t0 = std::min(t0, ~ctx->h_timeline[k]);
  for (int k = 0; k < kTimelineWords; k += 2) {
    const bool ran = ctx->h_timeline[k] != 0;
    out_us[k] = ran ? (double)(~ctx->h_timeline[k] - t0) * 1e-3 : -1.0;
    out_us[k + 1] = ran ? (double)(ctx->h_timeline[k + 1] - t0) * 1e-3 : -1.0;
  }
  return GAML_OK;
}

int gaml_get_stats(gaml_ctx* ctx, gaml_stats* out) {
  if (check_ctx(ctx) || !out) return GAML_ERR_ARG;
  if (ctx->timing_pending) {   // finish() returns on the result flag, possibly before the stream's closing event
    cudaSetDevice(ctx->device);
    float ms = 0, ms2 = 0;
    if (cudaEventSynchronize(ctx->ev[3]) == cudaSuccess) cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[3]);
    if (ctx->tail_timed) {   // + the many-placement passes finish() ran on demand after the chain
      float t = 0;
      if (cudaEventSynchronize(ctx->ev[2]) == cudaSuccess && cudaEventElapsedTime(&t, ctx->ev[1], ctx->ev[2]) == cudaSuccess) ms += t;
      ctx->tail_timed = false;
    }
    if (ctx->profile)
      for (auto& rs : ctx->sets) {
        float t = 0;
        if (cudaEventElapsedTime(&t, rs->ev0, rs->ev1) == cudaSuccess) ms2 += t;
      }
    ctx->stats.last_device_ms = ms;
    ctx->stats.last_score_kernel_ms = ms2;
    ctx->timing_pending = false;
  }
  ctx->stats.cache_appends = ctx->stats.cache_rebuilds = 0;
  for (auto& rs : ctx->sets) {
    ctx->stats.cache_appends += rs->appends;
    ctx->stats.cache_rebuilds += rs->rebuilds;
  }
  *out = ctx->stats;
  return GAML_OK;
}

}  // extern "C"
