/* gaml_b200 — C ABI of the B200-native GAML assembly-likelihood path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): everything the reference's
 * `ProbCalculator::CalcProb` (prob_calculator.h:63-118) and the three per-read-set scorers it
 * forwards to (`CalcScoreForPaths` graph.cc:1650, `CalcScoreForPathsNew` graph.cc:1952,
 * `CalcScoreForPacbio` graph.cc:3171) need, as plain C: opaque context, plain pointers and sizes,
 * int return codes (0 = ok, <0 = error, text via gaml_last_error), never an exception.
 * Host buffers are borrowed for the duration of a call only. One context per host thread.
 * All device work is ordered on one context-owned CUDA stream; results are valid on return.
 * There is NO CPU fallback: every scoring entry point fails with GAML_ERR_CUDA when no sm_100 device
 * is usable.
 */
#ifndef GAML_B200_H_
#define GAML_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gaml_ctx gaml_ctx;

enum {
  GAML_OK = 0,
  GAML_ERR_CUDA = -1,          /* CUDA runtime / no device */
  GAML_ERR_ARG = -2,           /* bad argument */
  GAML_ERR_KEY_EXISTS = -3,    /* cache key inserted twice */
  GAML_ERR_UNSUPPORTED = -4,   /* e.g. a batch over non-paired sets, or a penalised set in a _partial / _gathered batch */
  GAML_ERR_CAPACITY = -5,      /* a read needs more placement scratch than configured */
  GAML_ERR_STATE = -6          /* call order (e.g. finalize without a pending evaluation) */
};

enum { GAML_KIND_SINGLE = 0, GAML_KIND_PAIRED = 1, GAML_KIND_PACBIO = 2 };

/* Per-read-set scoring parameters: SingleReadConfig / PairedReadConfig (prob_calculator.h:7-35)
 * plus the ReadSet constructor's probabilities (graph.h:347-351, 446-449; match = 1 - 4*mismatch is the
 * caller's business, gaml.cc:813,854). insert_* are ignored for single / pacbio sets. */
typedef struct {
  int32_t kind;                /* GAML_KIND_* */
  int32_t reserved;
  double mismatch_prob;
  double match_prob;
  double insert_mean;
  double insert_std;
  double min_prob_per_base;
  double min_prob_start;
  double weight;
  double penalty_constant;     /* coverage-gap penalty (SURVEY §8 A8), scored on the device; 0 = off (the reference's default) */
  double step;
} gaml_readset_config;

/* `Aligment` (graph.h:211-215): one cached short-read alignment under a subpath key. */
typedef struct {
  int32_t position;
  int32_t edit_dist;
  int32_t read_id;             /* GLOBAL read id; records outside this context's shard are dropped */
  int32_t orientation;
} gaml_alignment;

/* `PacbioReadSet::PacbioAligment` (graph.h:516-520). */
typedef struct {
  int32_t position;
  int32_t position_end;
  int32_t read_id;
  int32_t pad;
  double logprob;
} gaml_pacbio_alignment;

/* Result of one CalcProb (prob_calculator.h:63): zeros[i] = (floored reads, n_reads) per read set in
 * the order the sets were added; total_len as the reference leaves it (last set's value). */
typedef struct {
  double prob;
  int32_t total_len;
  int32_t n_sets;
} gaml_result;

/* Partial sums of one read-id shard, per set: {integer part, fraction in 2^-40 units, floored reads, -inf terms,
 * nan terms}. The first two are an EXACT integer sum of the shard's per-read log terms (each rounded once to
 * 2^-40), so adding shards is exact and the combined total does not depend on the number of shards or on any
 * summation order. Combine with gaml_combine_partials after an all-gather (SURVEY §8e). */
#define GAML_PARTIAL_DOUBLES 5

typedef struct {
  int64_t kernel_launches;         /* kernels of THIS library launched since context creation */
  int64_t evals;                   /* CalcProb evaluations */
  int64_t last_records_gathered;   /* alignment records whose key was live in the last evaluation (A) */
  int64_t last_reads_scanned;      /* reads streamed by the last evaluation (R of the shard, all sets) */
  int64_t last_algorithmic_bytes;  /* DESIGN.md §bytes: 16*A + per-read bytes of the pass that ran */
  int64_t last_h2d_bytes;          /* bytes copied host->device by the last evaluation */
  int64_t last_d2h_bytes;
  double last_device_ms;           /* CUDA-event time of the last evaluation's kernels (gaml_set_profiling >= 1; else 0) */
  double last_score_kernel_ms;     /* CUDA-event time of the streaming kernel(s) only (gaml_set_profiling 2; else 0) */
  int32_t last_was_full;           /* 1 if the paired sets were re-scored from scratch */
  int32_t last_overflow_reads;     /* reads a streaming/delta kernel handed to the many-placement pass (they need the order) */
  double last_prepare_host_us;     /* host wall time inside gaml_eval_prepare / launch / finish of the last evaluation */
  double last_launch_host_us;      /*   (prepare = walk flattening + H2D enqueue, launch = kernel enqueue, */
  double last_finish_host_us;      /*    finish = wait for the device's result flag (+ D2H of penalty counters)) */
  int64_t last_scratch_placements; /* placements the last evaluation parked in the scratch arena (reads with more than four
                                      live placements on a mate) */
  int64_t last_multi_items;        /* full evaluations: items of the multi pass = reads with 3+ records on a mate + records under
                                      keys that occur several times in the evaluation (repeat nodes) */
  int64_t fast_change_evals;       /* incremental evaluations whose erased/added walks came from the diff against the previous
                                      walk list (walk_set.h) instead of the reference's container */
  int64_t delta_only_evals;        /* paired-set evaluations that updated the running total in O(touched reads): incremental,
                                      total length unchanged, so no O(R) pass (GetTotalProb's sum is kept exactly on the device) */
  int64_t cache_appends;           /* cache growths applied in O(new records): rows of the affected reads relocated, reads handed to
                                      the appendix phase */
  int64_t cache_rebuilds;          /* cache growths that rebuilt a read set's device index (first build, appendix full, no slack) */
  int64_t full_reuse_evals;        /* full evaluations of the walk list evaluated last: slot tables already on the device, no upload */
  int64_t full_patch_evals;        /* full evaluations of a list a few walks away from the resident one: only the slot updates of
                                      those walks' keys were built and uploaded (O(changed walks) host work) */
  int64_t last_batch_cov_events;   /* coverage-gap events (contig starts + covered positions) the last candidate batch sorted and
                                      swept, over its penalised paired sets; 0 without such a set */
  int64_t last_batch_cov_segments; /* coverage segments of that batch: one per (candidate, erased or added walk, penalised set) */
  int64_t last_batch_cov_exported; /* gaml_calc_prob_batch_shard: the thinned keys it kept for gaml_batch_penalty_export over the
                                      penalised sets (its last_batch_cov_events count this shard's emitted events); else 0 */
} gaml_stats;

/* ---- context ---------------------------------------------------------------------------- */
int gaml_ctx_create(int device, gaml_ctx** out);
void gaml_ctx_destroy(gaml_ctx* ctx);
const char* gaml_last_error(gaml_ctx* ctx);          /* ctx may be NULL: last creation error */
void* gaml_ctx_stream(gaml_ctx* ctx);                /* the cudaStream_t all work is ordered on */

/* Graph (graph.h:74-77, 233-273): the path only needs Node::s.length() per node id (2k forward,
 * 2k+1 twin) and normalize_map (NULL = identity). */
int gaml_set_graph(gaml_ctx* ctx, int32_t n_nodes, const int32_t* node_len, const int32_t* normalize_map);

/* ---- read sets -------------------------------------------------------------------------- */
/* Adds a read set; returns its index (>= 0) or an error. The context holds reads
 * [shard_lo, shard_hi) of n_reads_total (read-id sharding, SURVEY §8e); read_len1/2 point at the
 * SHARD's lengths (shard_hi - shard_lo entries; read_len2 only for paired sets). max_read_len1/2 are
 * the maxima over ALL reads (ReadSet::max_read_len_, graph.cc:1443-1447); pass -1 to take them from
 * the given arrays (correct when the shard is the whole set). */
int gaml_add_readset(gaml_ctx* ctx, const gaml_readset_config* cfg, int64_t n_reads_total, int64_t shard_lo,
                     int64_t shard_hi, const int32_t* read_len1, const int32_t* read_len2, int32_t max_read_len1,
                     int32_t max_read_len2);

/* ---- alignment cache mirror (aligment_cache_, graph.h:427 / 587) -------------------------- */
/* aligment_cache_[key] = records. mate is 0/1 (paired: ReadSet 1 / 2), 0 otherwise.
 * key_max_position: largest `position` over the key's records of ALL reads (it drives the
 * `max_pos - 5` skip rule, graph.cc:577-596); pass INT32_MIN to compute it from `records`
 * (correct whenever `records` holds the whole list, not just this shard's). */
int gaml_cache_insert(gaml_ctx* ctx, int set, int mate, const int32_t* key, int32_t key_len,
                      const gaml_alignment* records, int64_t n_records, int32_t key_max_position);
int gaml_cache_insert_pacbio(gaml_ctx* ctx, int set, const int32_t* key, int32_t key_len,
                             const gaml_pacbio_alignment* records, int64_t n_records);
/* 1 if the key is present (aligment_cache_.count(key)), 0 if not, <0 on error. */
int gaml_cache_contains(gaml_ctx* ctx, int set, int mate, const int32_t* key, int32_t key_len);
/* Uploads staged inserts (also done lazily by CalcProb). The first commit of a set builds its device index (read-major
 * rows, packed pair records, term table, internal read order); later ones — the annealing loop inserts the windows of a
 * new join — are applied in O(new records): records appended to the arena, the affected reads' rows relocated, the reads
 * handed to an appendix phase (gaml_stats.cache_appends); the index is rebuilt only when the appendix or the row slack
 * is full (gaml_stats.cache_rebuilds). */
int gaml_cache_commit(gaml_ctx* ctx);

/* PacBio alignment probability on the device (PacbioReadSet::AligmentProbability, graph.cc:2175-2297; the value
 * ProcessBlasrOutput stores as PacbioAligment::prob, graph.cc:2756, 2902 — the dominant cost while a PacBio cache is
 * cold): the forward probability, in log space, of read s2 given walk sequence s1 over the band around the aligner's
 * CIGAR path. Alignment a uses s1[s1_off[a] .. s1_off[a+1]) (the walk's sequence or a window of it; '\n' separates
 * contigs), s2[s2_off[a] .. s2_off[a+1]), posstart[a] (offset of the alignment in its s1) and the CIGAR operations
 * op_off[a] .. op_off[a+1) as (op_len, op_chr in "MID"). match_prob / mismatch_prob are the set's
 * (PacbioReadSet::match_prob_ / mismatch_prob_, graph.h:576-577); band is 2 in the reference. logprob_out[a] = logval. */
int gaml_pacbio_alignment_logprob(gaml_ctx* ctx, double match_prob, double mismatch_prob, int32_t band, int64_t n,
                                  const uint8_t* s1, const int64_t* s1_off, const uint8_t* s2, const int64_t* s2_off,
                                  const int32_t* posstart, const int32_t* op_len, const uint8_t* op_chr, const int64_t* op_off,
                                  double* logprob_out);

/* Flat on-disk form of one read set's cache (replaces ReadSet::SaveAligments / LoadAligments, graph.cc:1035-1100, whose
 * Boost archive the reference has switched off): keys with their metadata, then the key-major record arena exactly as
 * the device holds it. gaml_cache_load wants the read set created (gaml_add_readset with the same kind, read count and
 * shard) and still empty; the device index is built at the next commit as usual. */
int gaml_cache_save(gaml_ctx* ctx, int set, const char* path);
int gaml_cache_load(gaml_ctx* ctx, int set, const char* path);

/* ---- scoring ---------------------------------------------------------------------------- */
/* ProbCalculator::CalcProb(paths, zeros, total_len) (prob_calculator.h:63-109). Walks are concatenated
 * node ids (negative = gap of that many N's) with n_walks+1 offsets. STATEFUL exactly like the
 * reference: every call commits old_paths := paths for the paired sets (graph.cc:1986).
 * zeros: 2*n_sets int32 (floored, n_reads) pairs; may be NULL. */
int gaml_calc_prob(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks,
                   gaml_result* result, int32_t* zeros);

/* Same evaluation split for sharded (one process per GPU) use: `partials` receives
 * GAML_PARTIAL_DOUBLES doubles per set for THIS shard; all-gather them over ranks, then every rank calls
 * gaml_combine_partials with the n_shards x n_sets x GAML_PARTIAL_DOUBLES array (rank-major) to get the identical result. */
int gaml_calc_prob_partial(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets,
                           int32_t n_walks, double* partials, int32_t* total_len);
int gaml_combine_partials(gaml_ctx* ctx, const double* gathered, int32_t n_shards, int32_t total_len,
                          gaml_result* result, int32_t* zeros);

/* Context-free form of the combine step (pure host arithmetic, usable on ranks that only reduce):
 * kinds / n_reads_total / weights describe the n_sets read sets in the order they were added. */
int gaml_combine_partials_raw(const double* gathered, int32_t n_shards, int32_t n_sets, const int32_t* kinds,
                              const int64_t* n_reads_total, const double* weights, int32_t total_len,
                              gaml_result* result, int32_t* zeros);

/* Three-phase form of gaml_calc_prob_partial for measurement: prepare = host side (the walk list is diffed against the
 * previous evaluation's, the lookups of the CHANGED walks are flattened, the per-evaluation tables go to the device with
 * one copy; a full evaluation of a list a few walks away from the one whose tables are resident uploads only a patch,
 * gaml_stats.full_patch_evals); launch = the kernels (one CUDA-graph submission on gaml_ctx_stream); finish = wait for the
 * 64-byte result line the last block writes into host-mapped memory. GAML_ERR_STATE if an evaluation is still in flight. */
int gaml_eval_prepare(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks);
int gaml_eval_launch(gaml_ctx* ctx);
int gaml_eval_finish(gaml_ctx* ctx, double* partials, int32_t* total_len);

/* Multi-GPU jobs (one process and one context per GPU, read-id shards; no reference counterpart): the only exchange of
 * an evaluation is each rank's 64-byte result line per read set. shared_base is a host shared-memory segment that
 * every rank has mapped (e.g. POSIX shm; page aligned; at least 2 * world * GAML_EXCHANGE_MAX_SETS * 64 bytes; zeroed
 * once by its creator). The library maps it into the GPU, and from then on the block that completes a read set writes
 * its line straight into the segment — the collective is fused into the kernel: no copy, no NCCL call, no stream
 * synchronisation on the evaluation's path. gaml_eval_finish_gathered = gaml_eval_finish, then waits for the lines of
 * ALL ranks: gathered[world][n_sets][GAML_PARTIAL_DOUBLES], ready for gaml_combine_partials. The ranks must evaluate
 * in lockstep (the same sequence of evaluations), which an SPMD annealing driver does by construction.
 * shared_base == NULL detaches. */
#define GAML_EXCHANGE_MAX_SETS 8
int gaml_set_result_exchange(gaml_ctx* ctx, void* shared_base, int64_t bytes, int32_t rank, int32_t world);
int gaml_eval_finish_gathered(gaml_ctx* ctx, double* gathered, int32_t* total_len);
/* The same exchange over PEER MEMORY (NVLink / NVSwitch) instead of host memory: every rank owns a small device buffer of
 * result lines; the block that completes a read set stores its 64-byte line into the buffer of EVERY rank (peer stores),
 * and the last kernel of the evaluation's chain waits until all ranks' lines of this evaluation have arrived in its own
 * buffer, then hands them to the host in one piece — the all-gather is part of the evaluation's kernels, and the host
 * waits for one flag in its own pinned memory. gaml_peer_exchange_create allocates this rank's buffer and returns its
 * cudaIpcMemHandle_t (GAML_IPC_HANDLE_BYTES) for the caller's plumbing to all-gather (and the raw device pointer, for
 * contexts of the same process); gaml_peer_exchange_open takes all ranks' handles (rank-major) and/or local pointers and
 * switches the exchange on. gaml_eval_finish_gathered / gaml_calc_prob_gathered then work as above. Every rank needs its OWN
 * GPU: a kernel that waits for a line must never share a GPU with the kernel that writes it (refused with GAML_ERR_ARG). */
#define GAML_IPC_HANDLE_BYTES 64
int gaml_peer_exchange_create(gaml_ctx* ctx, int32_t rank, int32_t world, void* ipc_handle_out, void** buffer_out);
int gaml_peer_exchange_open(gaml_ctx* ctx, const void* ipc_handles, void* const* local_buffers);
int gaml_peer_exchange_close(gaml_ctx* ctx);
/* ... or through NCCL (SURVEY §8e "one ncclAllReduce(sum, fp64)"): the lines are all-reduced on the evaluation's stream
 * (every field is an integer far below 2^53, so the sums of doubles are exact); gaml_eval_finish_gathered reports the sum
 * as shard 0's partials and zeros for the others, which gaml_combine_partials adds to the same result. NCCL is bound at
 * run time (the copy the process has loaded, else libnccl.so.2). unique_id: 128 bytes from gaml_nccl_unique_id on one
 * rank, handed to all; NULL detaches. */
int gaml_nccl_unique_id(void* out128);
int gaml_nccl_exchange_init(gaml_ctx* ctx, const void* unique_id128, int32_t rank, int32_t world);
/* prepare + launch + finish_gathered in one call (the multi-GPU form of gaml_calc_prob_partial) */
int gaml_calc_prob_gathered(gaml_ctx* ctx, const int32_t* walk_nodes, const int64_t* walk_offsets, int32_t n_walks,
                            double* gathered, int32_t* total_len);

/* Batched, STATELESS evaluation of candidate moves (BASELINE config 5; SURVEY §8b gaml_gpu_eval_batch): candidate c
 * is the last evaluated walk set with the base walks erased_idx[erased_off[c] .. erased_off[c+1]) removed and the
 * walks added_walk_off[cand_added_off[c] .. cand_added_off[c+1]) appended (added_nodes / added_walk_off in the
 * layout of gaml_calc_prob). probs[c] is exactly the double gaml_calc_prob would return for that walk set if it were
 * called now — the same per-read subtract/add replay from the current ScoringState and the same exact sum — but
 * nothing is committed, so a move (LocalChange2, FixRepForNode2, FixGapLength: moves.cc:107-113, 715-726, 1158-1203)
 * can score all its candidates in one launch and then commit the winner with gaml_calc_prob. Paired sets only. A set
 * with penalty_constant != 0 is scored with the candidate's own bad bases (the state's, minus the erased walks', plus the
 * added walks', each swept over the current cache: graph.cc:1938, 1946, 1988) on an unsharded context.
 * zeros (optional): n_cand x 2 n_sets. The _partial form returns n_cand x n_sets x GAML_PARTIAL_DOUBLES for shards; it
 * refuses a penalised set (GAML_ERR_UNSUPPORTED): partials carry no bad bases, gaml_combine_partials would apply the
 * base state's. On read-id shards with a penalised set use gaml_calc_prob_batch_shard (below). */
int gaml_calc_prob_batch(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                         const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                         double* probs, int32_t* total_lens, int32_t* zeros);
int gaml_calc_prob_batch_partial(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                                 const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                                 double* partials, int32_t* total_lens);

/* The multi-GPU form (read-id shards, one context per GPU, every rank calls it with the same candidates): the shards'
 * partials of all candidates are summed by ONE all-reduce on the library's stream (needs gaml_nccl_exchange_init) and
 * combined exactly, so every rank receives the same probs — bit-identical to the unsharded gaml_calc_prob_batch.
 * A penalised set is refused (GAML_ERR_UNSUPPORTED): every candidate's coverage events would have to be all-gathered;
 * gaml_calc_prob_batch_shard does that with the caller's collective. */
int gaml_calc_prob_batch_gathered(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                                  const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                                  double* probs, int32_t* total_lens, int32_t* zeros);

/* Candidate batch on read-id shards with penalised paired sets (also unsharded, and without a penalty). A candidate's
 * bad bases are a sweep over the coverage events of ALL reads, so every rank, with the same candidates:
 * (1) gaml_calc_prob_batch_shard: the same arguments and outputs as gaml_calc_prob_batch_partial (bit-identical partials
 *     for an unpenalised set). Per penalised set this shard's events are sorted and thinned on the device: of each
 *     step-wide bucket of a candidate walk's positions only the first and last distinct position is kept, which leaves
 *     every walk's sweep unchanged (kernels.cu, coverage_thin_kernel) and the exchange small. Nothing is committed.
 * (2) per penalised set: gaml_batch_penalty_export (n_out = keys written, or needed when cap is too small), all-gather,
 *     and gaml_batch_penalty_import with the concatenation of every shard's keys, its own included: the sort and sweep of
 *     the unsharded batch, giving each candidate bad_bases_c = the state's - the erased walks' + the added walks';
 * (3) all-gather the partials and gaml_combine_batch_partials(gathered = n_shards x n_cand x n_sets x
 *     GAML_PARTIAL_DOUBLES, rank-major): probs (and zeros, n_cand x 2 n_sets, optional) bit-identical to an unsharded
 *     gaml_calc_prob_batch.
 * The batch stays pending until the next evaluation, batch or gaml_reset_state, which drop it; export, import and combine
 * then return GAML_ERR_STATE, as do export / import on a set without a penalty and combine before every import or with
 * another n_cand. gaml_calc_prob_batch_shard returns GAML_ERR_STATE while an evaluation's shard penalty awaits
 * gaml_penalty_import. */
int gaml_calc_prob_batch_shard(gaml_ctx* ctx, int32_t n_cand, const int32_t* erased_idx, const int64_t* erased_off,
                               const int32_t* added_nodes, const int64_t* added_walk_off, const int64_t* cand_added_off,
                               double* partials, int32_t* total_lens);
int gaml_batch_penalty_export(gaml_ctx* ctx, int set, uint64_t* out, int64_t cap, int64_t* n_out);
int gaml_batch_penalty_import(gaml_ctx* ctx, int set, const uint64_t* all, int64_t n_all);
int gaml_combine_batch_partials(gaml_ctx* ctx, const double* gathered, int32_t n_shards, int32_t n_cand, double* probs,
                                int32_t* zeros);

/* Coverage-gap penalty (penalty_constant != 0) of a paired or PacBio set on a READ-ID SHARD (SURVEY §8f rank 1): the sweep of
 * graph.cc:1893-1919 / 3197-3250 runs over a walk's events from ALL reads, so after gaml_eval_finish[_gathered] every rank
 * (1) takes its shard's events with gaml_penalty_export (paired: one 64-bit key per covered position; PacBio: two words per
 * alignment interval; n_out = words written, or needed when cap is too small), (2) all-gathers them with whatever it has
 * (MPI, torch.distributed, ...), (3) hands the concatenation of all shards' events, its own included, to
 * gaml_penalty_import, which sorts and sweeps them on the device and updates the set's bad_bases — the same integer on
 * every rank — and only then (4) calls gaml_combine_partials (refused with GAML_ERR_STATE while events are pending). */
int gaml_penalty_export(gaml_ctx* ctx, int set, uint64_t* out, int64_t cap, int64_t* n_out);
int gaml_penalty_import(gaml_ctx* ctx, int set, const uint64_t* all, int64_t n_all);

/* Forget the paired ScoringState (== constructing a fresh ProbCalculator, prob_calculator.h:45-47): the
 * next evaluation re-scores every read from scratch ("full logL"). */
int gaml_reset_state(gaml_ctx* ctx);

/* Per-read values of the last evaluation for parity dumps, shard-local order: single = sum of p1
 * (graph.cc:1697), paired = ScoringState::probs (graph.h:615), pacbio = log-sum-exp (graph.cc:3057). */
int gaml_read_values(gaml_ctx* ctx, int set, double* out, int64_t n);

int gaml_get_stats(gaml_ctx* ctx, gaml_stats* out);
/* Measurement aids, no reference counterpart. level 0 (default): nothing is timed. 1: two CUDA events around the
 * whole evaluation (gaml_stats.last_device_ms) — recorded as nodes of the evaluation's CUDA graph, i.e. pure device
 * time. 2: also events around each set's streaming kernel(s) (gaml_stats.last_score_kernel_ms, the roofline timing);
 * an event between two kernels makes the second wait for the first in the ordinary way, so the graph and the
 * programmatic dependent launches that chain an evaluation's kernels are given up. 3: no events; instead the device's
 * globaltimer is stamped at the start of each kernel's first block and the end of its last block (chain intact):
 * gaml_read_timeline -> out_us[12] = {start, end} in microseconds since the first stamp for {apply_slots, tier 1 phase,
 * tier 2 phase, many-placement pass, delta / multi pass, total pass} of the last evaluation's paired set; -1 = not run. */
int gaml_set_profiling(gaml_ctx* ctx, int32_t level);
int gaml_read_timeline(gaml_ctx* ctx, double* out_us, int32_t n);

#ifdef __cplusplus
}
#endif
#endif /* GAML_B200_H_ */
