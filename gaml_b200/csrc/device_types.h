// Plain structs shared by the host engine and the sm_100a kernels. Layout in HBM is documented in
// DESIGN.md §3; every struct is 16 or 32 bytes so one record is one (or two) 128-bit transactions.
#pragma once
#include <cstdint>

namespace gaml {

// One occurrence of a cache key in the walks of the current evaluation ("segment"): produced on the
// host by walking the reference's lookup loops (graph.cc:547-597 paired, 613-646 single,
// 2438-2500 pacbio) without touching any record.
struct Occ {
  int32_t walk;        // ordinal of the walk in this evaluation (erased walks first, then added)
  int32_t seg;         // global enumeration index of the lookup (walk-major) — the reference's order
  int32_t cur_pos;     // offset added to every record position (graph.cc:575, 636, 2497)
  int32_t skip_below;  // records with position+cur_pos below this are skipped (max_pos-5, graph.cc:577)
};

// Device-resident tables indexed by key id, two 16-byte words per key in two arrays. A key is live iff the epoch in
// word A matches the evaluation's epoch, so an evaluation only writes the slots of the keys it touches. Word A is
// all the streaming kernels need; word B (enumeration order, further occurrences) is read by the general paths.
struct SlotA {
  uint32_t epoch_flag;  // epoch (31 bits) | (n_occ > 1) << 31
  int32_t walk;         // first occurrence: walk ordinal
  int32_t cur_pos;
  int32_t skip_below;
};
struct SlotB {
  int32_t seg;          // first occurrence: enumeration index
  int32_t n_occ;
  int32_t occ_begin;    // into the evaluation's Occ array (all n_occ occurrences, first included)
  int32_t pad;
};
static_assert(sizeof(SlotA) == 16 && sizeof(SlotB) == 16, "slot words are 128-bit");

struct SlotUpdate {    // host -> device, scattered into KeySlot[key] by apply_slots_kernel
  int32_t key;
  int32_t n_occ;
  int32_t occ_begin;
  int32_t store;       // which mate store's slot table
  Occ first;
};
static_assert(sizeof(SlotUpdate) == 32, "");

// Key-major arena (mirror of aligment_cache_: keys in insertion order, records in list order).
struct ArenaShort { int32_t read; int32_t pos; int32_t edor; int32_t key; };   // edor = edit_dist | orientation<<30
struct ArenaLong { int32_t read; int32_t key; double logprob; };
// Read-major CSR rows built from the arena on the device; seq = arena index = reference list order.
struct RowShort { int32_t key; int32_t pos; int32_t edor; uint32_t seq; };
struct RowLong { int32_t key; uint32_t seq; double logprob; };
static_assert(sizeof(ArenaShort) == 16 && sizeof(ArenaLong) == 16 && sizeof(RowShort) == 16 && sizeof(RowLong) == 16, "");

// A record placed on a walk of the current evaluation.
struct Plc {
  unsigned long long ord;   // (seg << 32) | seq : the reference's enumeration order
  int32_t walk;
  int32_t pos;
  int32_t edor;
  int32_t pad;
};
struct PlcLong {
  unsigned long long ord;
  double logprob;
};

struct TouchRange { uint32_t begin; uint32_t count; };   // arena range of one touched mate-1 key

constexpr int kAccumStride = 8;   // per set, u64: four 32-bit limbs of the exact 128-bit sum, floored, -inf terms, nan terms, spare
constexpr int kBatchSlice = 4096;   // touched records of one candidate a block of the batch touch kernel takes
constexpr int kBatchBin = 5;      // batch base pass, per bin, u64: low / high 32-bit lanes of sum(Q - qthr), reads, -inf, nan
constexpr int kOutStride = 6;     // per set, f64: integer part, 2^-40 units, floored, -inf terms, nan terms, flags
constexpr unsigned long long kResultSeal = 0x5eed5eed5eed5eedull;   // word 7 = seal ^ xor of words 0..6
constexpr int kResultStride = 8;  // per set in the host-mapped result buffer (one 64-byte line): the kOutStride values,
                                  // the epoch of the evaluation that wrote them (the host's completion flag), a checksum
struct Int2 { int32_t x, y; };
struct Double2 { double x, y; };  // {1/c, -log(1/c)} entries of the log table
// One entry of a uniform-length paired set's term table: the pair term (p1*p2)*ins for (edit 1, edit 2, insert distance)
// and its fixed-point logarithm (kTermOdd when the logarithm is not finite).
struct TermEntry { double t; long long q; };
constexpr long long kTermOdd = (long long)0x8000000000000000ull;

struct MateView {
  const void* first;         // short stores: dense int4 per read {key, pos, edor | count<<16, row offset}; key<0 = none
  const void* rows;          // RowShort* / RowLong* (read-major CSR; a read's rows in reference list order)
  const uint32_t* rowptr;    // n_reads + 1
  const void* crows;         // compact copy of the rows of the tier-2 reads (list order), RowShort*
  const uint32_t* cptr;      // n_complex + 1 offsets into crows
  const SlotA* slots_a;
  const SlotB* slots_b;
  int32_t n_keys;
  const Occ* occ;
  const double* pow_match;   // match^k     (graph.cc:1451)
  const double* pow_mismatch;// mismatch^k  (graph.cc:1452)
};

struct ScoreParams {
  MateView m[2];
  const uint32_t* lens;      // single/pacbio: read length; paired: len1 | len2<<16
  const void* comb;          // paired: per mate-1 key {SlotA of that key, SlotA of the SAME key in mate 2's store} (32 B), or null
  const void* pairs;         // paired: one PackedPair (16 B) per pair for the streaming kernel's tier 1, or null (kernels.cu)
  const double* uni_prob[2]; // paired, lens_uniform: per mate mismatch^e * match^(len-e) for e in [0,128), host-computed (same rounding), or null
  double uni_pstar;          //   and the floor test / floored term of every pair (see pstar_tab / qthr_tab)
  long long uni_qthr;
  const void* tq;            // paired, lens_uniform: TermEntry[1 + (e1 << tq_shift | e2) * ins_n + dist] for e1, e2 < 1 << tq_shift
  int32_t tq_shift;          //   (entry 0: no pair term), or null
  const void* fast;          // with a term table: one FastPair (16 B) per pair for tier 1 (kernels.cu), or null
  const uint32_t* xlist;     //   and the cross list: tier-1 reads the fast records leave to the general body (ascending read ids)
  int32_t n_cross;
  int32_t n_tier1;           //   and the number of reads tier 1 streams ([0, n_tier1) of the internal order; n_reads without one)
  // reads that gained records since the static lists were built (cache appends, kernels.cu append_apply_kernel): flagged
  // in `dirty` (and in their packed / fast records), skipped by every list-driven phase and scored from their rows by the
  // appendix phase instead
  const uint32_t* dirty;     // per read, or null when no append has happened since the last rebuild
  const uint32_t* appx_list;
  int32_t n_appx;
  uint32_t uniform_ll;       // paired: the packed lengths when every pair of the set has the same ones (lens_uniform)
  int32_t lens_uniform;
  const double* ins_tab;     // insert pdf for dist in [0, ins_n), host-computed; 0 beyond (exp underflow)
  int32_t ins_n;
  // The per-read log term (GetTotalProb, graph.cc:1495-1537: log max(p / 2L, thr)), indexed by len (paired: len1+len2):
  //   floored <=> RN(p / 2L) < thr <=> p < pstar_tab[len]   (the smallest double whose IEEE quotient by 2L reaches thr: host, exact)
  //   floored: qthr_tab[len] = FIX(log thr);  otherwise FIX(LOG p) - FIX(log 2L), the second part applied once per set (ql)
  const double* pstar_tab;   // per evaluation (depends on L), in the staging blob
  const long long* qthr_tab; // per set
  long long ql;              // FIX(log 2L), host-computed
  double floor_a, floor_b;   // pacbio: log(exp(mps)), log(exp(mppb)) (graph.cc:3075-3076)
  double* values;            // paired: ScoringState::probs; single: sum p1; pacbio: LSE
  uint32_t epoch;
  int32_t n_erased;          // walks with ordinal < n_erased are subtracted (paired)
  int32_t n_reads;           // reads in this shard
  int32_t two_len;           // 2*total_len as the reference's int expression (total_len==0 -> 1)
  // many-placement reads
  uint32_t* ovf_count;
  uint32_t* ovf_list;
  uint32_t ovf_cap;
  Plc* scratch;              // also used as PlcLong (same size)
  unsigned long long* scratch_cursor;
  unsigned long long scratch_cap;
  uint32_t* error_flag;
  // static tier-2 list (reads owning several records on a mate), built at cache commit
  const uint32_t* complex_list;
  const uint32_t* clens;     // lens[] gathered in list order
  const void* cdesc;         // int4 per listed read {read, packed lengths, first compact row mate 1, mate 2}
  int32_t class_begin[17];   // first list index of every record-count class, in list order (complex_class ranks)
  int32_t n_complex;
  int32_t n_main;            // list entries tier 2 streams (ranks 0..4); the rest is the multi pass's static part
  const void* t2pack;        // packed tier-2 entries of classes (1,2) (2,1) (2,2), unit-major per class (kernels.cu), or null
  uint32_t t2base[3];        // first uint4 of each class in t2pack
  uint32_t cbase[2][5];      // per mate: first compact row of classes 0..4 (rows per read are uniform within a class)
  // multi pass: arena ranges (both mates) of the keys that occur several times in this evaluation
  const ArenaShort* arena2;
  const TouchRange* mtouch;        // n_mtouch ranges, the first n_mtouch1 in mate 1's arena
  const uint32_t* mtouch_prefix;   // n_mtouch + 1
  int32_t n_mtouch, n_mtouch1;
  // chain discipline of the streaming kernels (set per launch)
  int32_t chain_first;       // 1: first kernel after apply_slots in its group: waits at its top; 0: waits at its end
  int32_t finish_here;       // 1: this kernel's last block publishes the set when nothing was listed for the pass after it;
                             // 2: no pass follows: it publishes the set, as a pending line when reads were listed
  uint32_t* tile_counter;    // next tile of [0] tier 1, [1] the rare shapes, [2] tier 2, [3] the cross list, then the appendix (zeroed by apply_slots)
  uint32_t* ticket2;         // blocks-finished counter of the set's last kernel (finish_set)
  uint32_t* done;            // set by finish_set_if_complete
  // reduction: exact 128-bit fixed-point sum of the log terms of this set (kAccumStride u64)
  unsigned long long* accum;
  uint32_t* ticket;          // blocks-finished counter of the set's last streaming kernel (finish_set_if_complete)
  unsigned long long* timeline;    // profiling level 2: per kernel {first block start, last block end} in globaltimer ns; else null
  unsigned long long* state_acc;   // paired sets: running total on the device {low, high, floored, -inf, nan} (finish_set)
  int32_t state_add;         // 1: this evaluation accumulated a delta to add to state_acc; 0: it replaces it
  int32_t delta_only;        // 1: incremental evaluation at an unchanged total length (no O(R) pass)
  double* out;               // kResultStride doubles in HOST-MAPPED pinned memory, written by the last block (finish_set)
  // multi-GPU result exchange over peer memory (NVLink): the publishing block also stores the set's 64-byte line into
  // line `peer_line` of every rank's exchange buffer (peer_bufs[0 .. peer_world), this rank's own included)
  unsigned long long* const* peer_bufs;
  int32_t peer_world;
  uint32_t peer_line;
  double* part_out;          // device copy of the line for a collective library (NCCL all-reduce), or null
  const void* log_tab;       // 128 x {1/c, -log(1/c)} (double2)
  // coverage-gap penalty events (null when the set has penalty_constant == 0)
  unsigned long long* ev_keys;
  uint32_t* ev_count;
  uint32_t ev_cap;
  const double* cov_thr;     // exp(mps + mppb * 2*len2) indexed by len2 (graph.cc:1855-1857)
  // delta discovery
  const ArenaShort* arena1;
  const TouchRange* touch;
  const uint32_t* touch_prefix;   // n_touch + 1
  int32_t n_touch;
  uint32_t* stamp;           // per read: epoch of the evaluation that last claimed it
};

// ---- PacBio coverage penalty (graph.cc:3197-3250) -----------------------------------------------------------------
struct PbCovParams {
  const void* seeds;            // int4 {walk, start, end, -}: the artificial interval and one interval per node of every walk
  int32_t n_seed;
  const void* occ;              // int4 {walk, offset of the key's first node, arena range begin, count} per live key occurrence
  const uint32_t* occ_prefix;   // n_occ + 1 prefix sums of the counts
  int32_t n_occ;
  const ArenaLong* arena;
  const void* arena_pos;        // int2 {position, position_end} per arena record
  const uint32_t* lens;
  double log_mismatch, log_match;   // GetMinReadProb, graph.h:478-481
  unsigned long long* ikey;     // intervals: (walk, start) keys, 2 x cap (unsorted, sorted)
  int32_t* iend;                // their ends, 2 x cap
  unsigned long long* pkey;     // event positions (walk, pos), 4 x cap
  uint32_t* count;              // intervals emitted
  uint32_t cap;
  uint32_t* error_flag;
};

// ---- PacBio alignment probability (graph.cc:2175-2297) --------------------------------------------------------------
struct AlnMeta {
  int64_t s1_off, s2_off, op_off, scratch_off;
  int32_t s1_len, s2_len, posstart, n_ops;
  int32_t bl, el;              // leading / trailing insertion runs (GetCigarEnds, capped at 200)
  int32_t row_end, col_end;    // where the CIGAR path ends
  int32_t width;               // upper bound of a row's cells (scratch strip: 2 x width doubles)
  int32_t pad[3];
};
constexpr int kAlnMaxBand = 8;
struct AlnProbParams {
  const AlnMeta* meta;
  long long n;
  const unsigned char* s1;
  const unsigned char* s2;
  const int32_t* op_len;    // CIGAR operations of all alignments
  const unsigned char* op_chr;
  int32_t band;
  double* scratch;
  double log_match, log_mismatch;
  double* out;
  uint32_t* error_flag;     // bit 0: a row was wider than the host's bound (result NaN)
};

// ---- batched candidate evaluation (gaml_calc_prob_batch, BASELINE config 5) ------------------------------
struct BatchCand {             // one candidate move, one paired read set
  int32_t key_begin[2];        // this candidate's slice of the batch key/slot arrays, per mate (keys sorted)
  int32_t key_count[2];
  int32_t n_erased;            // walk ordinals < n_erased are subtracted
  int32_t len_index;           // index of this candidate's total length among the batch's distinct values
  int32_t range_begin;         // this candidate's slice of the batch's touched-key ranges
  int32_t range_count;
};
struct BatchParams {
  const BatchCand* cands;
  int32_t n_cand;
  const int32_t* keys[2];      // per mate: candidate-local sorted key ids
  const void* slot_a[2];       // parallel SlotA / SlotB words (epoch field unused)
  const void* slot_b[2];
  const Occ* occ[2];
  const TouchRange* ranges;    // mate-1 arena ranges of the touched keys, all candidates back to back
  const uint32_t* range_prefix;// n_ranges + 1 prefix sums of the range lengths
  const int32_t* range_cand;   // owning candidate of each range
  const int32_t* partner12;    // mate-1 key id -> the same node sequence's key id in mate 2's store (-1: none), or null
  const Int2* blocks;          // touched-record pass: {candidate, first record of the slice} per block (kBatchSlice records each)
  int32_t n_blocks;
  int32_t n_ranges;
  // The batch's distinct total lengths, ASCENDING (so that a read's floor test pstar grows with the index), for every
  // length class (distinct len1+len2) of the set: pstar[cls * n_len + j]; len_class maps len1+len2 -> cls.
  const double* pstar;
  const long long* qthr_cls;   // per class: FIX(log thr)
  const int32_t* len_class;
  const long long* ql;         // n_len: FIX(log 2L)
  int32_t n_len;
  unsigned long long* hist;         // (n_len + 1) x kBatchBin: per "first floored length index" bin of the base pass (kernels.cu)
  unsigned long long* accum_len;    // n_len x kAccumStride: {low, high 64 bits of the exact sum of all reads' FIX terms at that
                                    // length (before the - n FIX(log 2L) part), floored, -inf, nan}
  long long* accum_cand;            // n_cand x 4: {sum of low 32 bits, sum of high 32 bits (signed) of the term deltas, floored delta, bad}
  // penalised sets: each candidate's first coverage segment (one segment per erased or added walk of a candidate, batch-wide
  // ids: the candidate's walk ordinal k emits its events under seg_begin[c] + k), or null
  const int32_t* seg_begin;
};

}  // namespace gaml
