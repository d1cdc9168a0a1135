// Launch wrappers of kernels.cu (host-callable; all asynchronous on the given stream).
#pragma once
#include <cuda_runtime.h>

#include "device_types.h"

namespace gaml {

// One kernel launch of an evaluation, recorded instead of issued: the engine replays the list either directly or —
// the steady state — by updating the kernel nodes of a CUDA graph captured from the same sequence and launching that
// (one submission instead of one per kernel; the programmatic dependent launch edges are captured with it).
struct PendingLaunch {
  const void* func = nullptr;
  unsigned grid = 1, block = 1;
  bool pdl = false;
  int n_args = 0;
  void* arg_ptrs[16];
  alignas(16) unsigned char arg_buf[1536];
};
struct LaunchList {
  PendingLaunch item[16];
  int n = 0;
};
// While a list is set (per thread), launch_chain-based wrappers append to it instead of launching.
void set_launch_recorder(LaunchList* list);
cudaError_t issue_launch(const PendingLaunch& pl, cudaStream_t st);

enum { kGridPairedFull = 0, kGridPairedComplex, kGridPairedTotal, kGridSingleFull, kGridSingleComplex, kGridPacbioFull };
int score_grid(int which, int n_items, int sm_count);
int overflow_grid(int sm_count);

// Per-store table pointers passed BY VALUE (kernel parameter space) when a context has at most kInlineStores mate stores:
// apply_slots then needs no dependent load to find a store's tables. a/b: first/second slot words; cb/cm: the combined
// table of a paired set and the mate-2 -> mate-1 key map (see apply_slots_kernel).
constexpr int kInlineStores = 8;
struct StoreTables {
  SlotA* a[kInlineStores];
  SlotB* b[kInlineStores];
  SlotA* cb[kInlineStores];
  const int32_t* cm[kInlineStores];
};
void launch_apply_slots(const SlotUpdate* upd, int n, const SlotUpdate* patch, int n_patch, const int32_t* skip, int n_skip,
                        SlotA* const* tab_a, SlotB* const* tab_b, SlotA* const* comb_base,
                        const int32_t* const* comb_map, const StoreTables* inline_tabs, uint32_t epoch, unsigned long long* flags,
                        int n_flag_words, unsigned long long* timeline, cudaStream_t st);
constexpr int kTimelineWords = 12;   // profiling level 2: {start, end} ns of apply, tier 1, tier 2, many-placement, delta, total
// Each wrapper appends the kernels of one read set to the evaluation's chain on `st` (programmatic dependent
// launches, kernels.cu): streaming pass (tier 1, tier 2), many-placement pass, per-set finalize in the last block.
// chained: the operation before it on `st` is a kernel of the chain. profile: record e0 / e1 around the streaming
// kernel(s) of the set (the roofline timing) — which serialises those two boundaries in the ordinary way.
// tail: append the many-placement pass (always when profiling). Without it the streaming kernel publishes a pending
// line (word 6 = -epoch, running total not committed) when it listed reads, and the host calls launch_paired_tail.
int launch_paired_full(const ScoreParams& P, int grid, int cgrid, uint32_t n_multi_items, int ovf_grid, int sm_count,
                       cudaStream_t st, bool chained, bool profile, cudaEvent_t e0, cudaEvent_t e1,
                       bool tail);   // returns the kernels launched
// The many-placement pass of a full evaluation whose chain ended with a pending line: publishes the final line.
void launch_paired_tail(const ScoreParams& P, int ovf_grid, cudaStream_t st);
void launch_paired_delta(const ScoreParams& P, uint32_t n_touch_records, int grid_total, int ovf_grid, int sm_count, cudaStream_t st,
                         bool chained, bool profile, cudaEvent_t e0, cudaEvent_t e1);
void launch_single_full(const ScoreParams& P, int grid, int cgrid, int ovf_grid, cudaStream_t st, bool chained, bool profile,
                        cudaEvent_t e0, cudaEvent_t e1);
void launch_pacbio_full(const ScoreParams& P, int grid, int ovf_grid, cudaStream_t st, bool chained, bool profile, cudaEvent_t e0,
                        cudaEvent_t e1);

cudaError_t build_csr(const void* arena, size_t n_records, int n_reads, bool is_long, uint32_t* rowptr, uint32_t* cursor,
                      void* rows, void* first, void* temp, size_t temp_bytes, int sm_count, cudaStream_t st, int* launches);
cudaError_t build_complex_list(const void* first1, const void* first2, int n_reads, uint32_t* flags, uint32_t* list,
                               void* temp, size_t temp_bytes, cudaStream_t st, int* launches, uint32_t* n_complex_out,
                               int32_t* class_begin);
void launch_pack_tier2(const void* cdesc, const void* rows1, const void* rows2, const int32_t* class_begin, const uint32_t cbase[2][5],
                       const uint32_t tbase[3], void* out, uint32_t* bad, cudaStream_t st);
void launch_pack_pairs(const void* first1, const void* first2, int n, const int32_t* partner12, void* out, uint32_t* bad, cudaStream_t st);
void launch_cdesc_fill(const uint32_t* list, int n_complex, const uint32_t* lens, const uint32_t* cptr1, const uint32_t* cptr2,
                       void* desc, cudaStream_t st);
cudaError_t compact_offsets(const uint32_t* list, int n_complex, const uint32_t* rowptr, uint32_t* cptr, const uint32_t* lens,
                            uint32_t* clens, void* temp, size_t temp_bytes, cudaStream_t st, int* launches);
cudaError_t compact_copy(const uint32_t* list, int n_complex, const uint32_t* rowptr, const uint32_t* cptr, const void* rows,
                         void* crows, cudaStream_t st, int* launches);
// Batched candidate evaluation of one paired set: base pass per distinct total length, touched-read pass, finalize.
void launch_batch(const ScoreParams& P, const BatchParams& B, uint32_t n_touch_records, double* out, const uint32_t* error_flag,
                  int sm_count, cudaStream_t st);
int batch_hist_bins(int n_len);            // bins of BatchParams::hist for n_len distinct total lengths
int batch_launches(int n_len, bool touch);  // kernels launch_batch issues
// Term table of a uniform-length paired set: 1 + (1 << shift)^2 * ins_n TermEntry (entry 0 = "no pair term").
void launch_build_term_table(const double* p1, const double* p2, const double* ins, int ins_n, int shift, const void* log_tab, void* out,
                             int sm_count, cudaStream_t st);
// FastPair array + cross list of a paired set with a term table (kernels.cu); flags: n + 1 uint32 of scratch whose last
// entry holds the number of listed reads afterwards.
cudaError_t build_fast_pairs(const void* pairs, int n, int shift, int ins_n, uint32_t uniform_ll, void* fast, uint32_t* flags, uint32_t* list,
                             void* temp, size_t temp_bytes, cudaStream_t st, int* launches);
// Cache append (kernels.cu "cache append"): AppendGroup = {read, first new row, new rows, destination row} per affected read.
struct AppendGroupHost { uint32_t read, new_begin, n_new, dst; };
// One cache append of a paired set (append_apply_kernel): per mate the staged arena records and their place at the arena
// tail, the groups + new rows of the reads that gained records; the reads newly on the appendix list; key-map patches.
struct AppendMate {
  const void* arena_src; void* arena_dst; uint32_t n_rec;
  const void* groups; int n_groups; const void* new_rows; void* rows; void* first;
};
struct AppendJob {
  AppendMate m[2];
  uint32_t* dirty; void* pairs; void* fast;
  const uint32_t* appx_src; uint32_t* appx_dst; int n_appx_new;
  const int2* p12_patch; int n_p12; int32_t* p12;
  const int2* p21_patch; int n_p21; int32_t* p21;
};
void launch_append_apply(const AppendJob& J, cudaStream_t st);
void launch_extract_counts(const void* first, const uint32_t* rowptr, int n, uint16_t* out, cudaStream_t st);
// Internal read order of a paired set with fast records (kernels.cu): sort keys from the FastPair array, radix sort,
// inverse permutation (caller's local read id -> internal index) and the length of the fast region.
size_t perm_temp_bytes(int n);
cudaError_t build_read_permutation(const void* fast, int n, unsigned long long* keys, uint32_t* ids, uint32_t* inv, uint32_t* n_fast,
                                   void* temp, size_t temp_bytes, cudaStream_t st, int* launches);
void launch_remap_arena(void* arena, size_t n_records, const uint32_t* inv, int sm_count, cudaStream_t st);
// Coverage-gap penalty of one paired set: radix sort of the event keys, then the one-thread-per-event sweep.
size_t coverage_sort_temp_bytes(unsigned n);
cudaError_t launch_coverage(const unsigned long long* keys_in, unsigned long long* keys_sorted, unsigned n, void* temp,
                            size_t temp_bytes, const int* cs_begin, const int* cs, double step, double min_from_start, int* bad,
                            int sm_count, cudaStream_t st);
// PacBio coverage penalty of one set: emit intervals, sort by (walk, start), running max of ends, sort positions, sweep.
size_t pacbio_coverage_temp_bytes(uint32_t cap);
cudaError_t launch_pacbio_coverage(const PbCovParams& C, unsigned long long* packed, unsigned long long* run_max, void* temp,
                                   size_t temp_bytes, const int* walk_len, double step, int* bad, int sm_count, cudaStream_t st,
                                   int phase = 0);   // 1: emit only, 2: sort + sweep only (read-id shards, kernels.cu)
// PacBio alignment probability: one thread per alignment over host-prepared row ranges.
void launch_pacbio_alnprob(const AlnProbParams& A, int sm_count, cudaStream_t st);
// Multi-GPU result exchange: last kernel of an evaluation's chain (appended to it: recorded like the scoring kernels).
void launch_exchange_gather(const unsigned long long* lines, int world, int n_sets, int max_sets, uint32_t epoch,
                            unsigned long long* host_lines, unsigned long long* host_flag, unsigned long long timeout_ns, cudaStream_t st);
void launch_reduced_publish(const double* reduced, int n_sets, uint32_t epoch, unsigned long long* host_lines, cudaStream_t st);
size_t csr_temp_bytes(int n_reads);

}  // namespace gaml
