// Drop-in replacement for the reference's prob_calculator.h (usamec/GAML): same class, same constructor,
// same three CalcProb overloads, same public members — the bodies forward to the gaml_b200 CUDA library
// through its C ABI (include/gaml_b200.h). gaml.cc (Optimize, main) and moves.cc compile against this file
// UNCHANGED; graph.h / graph.cc stay the reference's (the ReadSet objects remain the host-side cache owners
// that the moves use, moves.cc:831-856, 948-964, and their aligners keep filling the caches).
//
// Build (see oracle/build_ref.sh, target gaml_gpu): put this directory BEFORE the reference on the include
// path and compile gaml.cc / moves.cc with -Dprivate=public so the adapter can read ReadSet::aligment_cache_
// (graph.h:427) — access specifiers do not change object layout, graph.o is the reference's own object file.
// A maintainer would instead add two accessors to ReadSet; INTEGRATION.md shows that patch.
//
// What stays on the host, exactly as the reference does it, is everything that FILLS the caches: for every walk the
// adapter has not seen yet it runs the reference's own precompute routines where CalcScoreForPathsNew /
// GetPositionsOnlyPath / AddPositions / PacbioReadSet::GetReadProbabilities run them (graph.cc:1967-1968, 538-542,
// 605-609, 2455-2486), so the same keys are aligned in the same order; it then mirrors the keys the device does not hold
// yet and calls gaml_calc_prob. A walk seen before costs a share of a block compare (or one hash probe): its keys are all in the
// cache already — the cache never shrinks — so it can contribute nothing to either step. No score is ever computed on the
// CPU; if the CUDA context cannot be created the program aborts like the reference's asserts do.
#ifndef PROB_CALCULATOR_H__
#define PROB_CALCULATOR_H__

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <unordered_map>
#include <unordered_set>

#include "flat_paths.h"
#include "gaml_b200.h"
#include "graph.h"
#include "utility.h"

struct SingleReadConfig {   // reference prob_calculator.h:7-18
  SingleReadConfig() {}
  SingleReadConfig(double pc, double s, double mp, double mps, double w, bool a)
      : penalty_constant(pc), step(s), min_prob_per_base(mp), min_prob_start(mps), weight(w), advice(a) {}
  double penalty_constant;
  double step;
  double min_prob_per_base;
  double min_prob_start;
  double weight;
  bool advice;
};

struct PairedReadConfig {   // reference prob_calculator.h:20-35
  PairedReadConfig() {}
  PairedReadConfig(double pc, double s, double im, double is, double mp, double mps, double w, bool a)
      : penalty_constant(pc), step(s), insert_mean(im), insert_std(is), min_prob_per_base(mp), min_prob_start(mps),
        weight(w), advice(a) {}
  double penalty_constant;
  double step;
  double insert_mean;
  double insert_std;
  double min_prob_per_base;
  double min_prob_start;
  double weight;
  bool advice;
};

class ProbCalculator {
 public:
  ProbCalculator(const vector<pair<SingleReadConfig, ReadSet*>>& single_reads,
                 const vector<pair<PairedReadConfig, pair<ReadSet*, ReadSet*>>>& paired_reads,
                 const vector<pair<SingleReadConfig, PacbioReadSet*>>& pacbio_reads, Graph& gr)
      : single_reads(single_reads), paired_reads(paired_reads), pacbio_reads(pacbio_reads), gr(gr), ctx_(NULL) {
    paired_scoring_states.resize(paired_reads.size());   // kept for source compatibility; the state lives on the device
  }
  ~ProbCalculator() { gaml_ctx_destroy(ctx_); }

  double CalcProb(vector<vector<int>>& paths, vector<pair<int, int>>& zeros, int& total_len) {
    if (!ctx_) Init();   // lazy: gaml.cc constructs the calculator before PrepareReads fills the read sets
    // ONE pass over the caller's vector-of-vectors: the flat arrays the C ABI takes. Everything else the adapter does per
    // call (which walks are new, FinalEnd bookkeeping) works on these arrays against the previous call's.
    gaml_flat::Flatten(paths, cur_);
    FillAndMirrorCaches(paths, cur_, prev_, prev_final_end_, cur_final_end_, NULL);
    z_.assign(2 * (n_sets_ ? n_sets_ : 1), 0);
    gaml_result res;
    Check(gaml_calc_prob(ctx_, cur_.nodes.data(), cur_.offs.data(), (int)paths.size(), &res, z_.data()));
    zeros.clear();
    for (size_t s = 0; s < n_sets_; s++) zeros.push_back(make_pair(z_[2 * s], z_[2 * s + 1]));
    total_len = res.total_len;
    had_calc_ = true;
    cur_.swap(prev_);   // the evaluated walks become the list the next call is compared with (no copy)
    prev_final_end_.swap(cur_final_end_);
    have_prev_ = true;
    return res.prob;
  }
  double CalcProb(vector<vector<int>>& paths, int& total_len) {
    vector<pair<int, int>> zeros;
    return CalcProb(paths, zeros, total_len);
  }
  double CalcProb(vector<vector<int>>& paths) {
    int tl;
    return CalcProb(paths, tl);
  }

  // NOT in the reference: scores every candidate walk set against the CURRENT state (the walk set of the last CalcProb)
  // in one device batch (gaml_calc_prob_batch) and changes no state. scores[c] is the double a CalcProb(candidates[c])
  // issued right now would return. The moves that try several alternatives one CalcProb at a time (LocalChange2
  // moves.cc:107-113, FixGapLength 715-726, FixRepForNode2 1158-1305) submit them here when built with
  // oracle/build_ref.sh's moves.cc patch (target gaml_gpu_batched, GamlBatchReplay below). Paired sets with a
  // coverage-gap penalty are batched too (each candidate gets its own bad bases). With single or PacBio sets
  // configured — they keep no incremental state to evaluate candidates against — the candidates are scored one by one.
  vector<double> CalcProbBatch(vector<vector<vector<int>>>& candidates) {
    vector<double> scores(candidates.size(), 0.0);
    if (candidates.empty()) return scores;
    if (!ctx_) Init();
    if (!single_reads.empty() || !pacbio_reads.empty() || paired_reads.empty() || !have_prev_ || prev_.n() == 0 || !had_calc_) {
      for (size_t c = 0; c < candidates.size(); c++) scores[c] = CalcProb(candidates[c]);
      return scores;
    }
    vector<int32_t> erased_idx, added_nodes;
    vector<int64_t> erased_off(1, 0), added_walk_off(1, 0), cand_added_off(1, 0);
    gaml_flat::FlatPaths cand;
    vector<int> fe, match;
    vector<int> un_base, un_cand;   // walks without an equal partner at the aligned position
    for (size_t c = 0; c < candidates.size(); c++) {
      gaml_flat::Flatten(candidates[c], cand);
      // aligns the candidate with the CURRENT walk list (which stays what it is) and mirrors the windows of walks seen
      // for the first time
      FillAndMirrorCaches(candidates[c], cand, prev_, prev_final_end_, fe, &match);
      // multiset difference against the current list: aligned equal walks drop out; what is left on either side (a
      // handful of walks) is matched by content
      gaml_flat::Difference(prev_, cand, match, un_base, un_cand, erased_idx, added_nodes, added_walk_off);
      erased_off.push_back((int64_t)erased_idx.size());
      cand_added_off.push_back((int64_t)added_walk_off.size() - 1);
    }
    if (erased_idx.empty()) erased_idx.push_back(0);
    if (added_nodes.empty()) added_nodes.push_back(0);
    vector<int32_t> tls(candidates.size());
    Check(gaml_calc_prob_batch(ctx_, (int32_t)candidates.size(), erased_idx.data(), erased_off.data(), added_nodes.data(),
                               added_walk_off.data(), cand_added_off.data(), scores.data(), tls.data(), NULL));
    return scores;
  }

  vector<pair<SingleReadConfig, ReadSet*>> single_reads;
  vector<pair<PairedReadConfig, pair<ReadSet*, ReadSet*>>> paired_reads;
  vector<pair<SingleReadConfig, PacbioReadSet*>> pacbio_reads;
  vector<ScoringState> paired_scoring_states;
  Graph& gr;

 private:
  typedef gaml_flat::FlatPaths FlatPaths;
  struct Mirror {   // one ReadSet <-> one (set, mate) store of the library
    ReadSet* rs;
    int set, mate;
    bool paired;
    unordered_set<vector<int>> sent;
  };

  struct PbMirror {
    PacbioReadSet* rs;
    int set;
    unordered_set<vector<int>> sent;
  };
  static const int kNoNode = -1000000;   // FinalEnd of a walk without any node: it leaves `last_end` alone

  void Check(int rc) {
    if (rc < 0) {
      fprintf(stderr, "gaml_b200: %s\n", gaml_last_error(ctx_));
      abort();
    }
  }

  static gaml_readset_config Cfg(int kind, double pc, double step, double mppb, double mps, double w, double match,
                                 double mismatch) {
    gaml_readset_config c;
    c.kind = kind;
    c.reserved = 0;
    c.mismatch_prob = mismatch;
    c.match_prob = match;
    c.insert_mean = 0;
    c.insert_std = 1;
    c.min_prob_per_base = mppb;
    c.min_prob_start = mps;
    c.weight = w;
    c.penalty_constant = pc;
    c.step = step;
    return c;
  }

  static vector<int32_t> Lens(const ReadSet& rs) {
    vector<int32_t> l(rs.GetNumberOfReads());
    for (size_t i = 0; i < l.size(); i++) l[i] = rs.GetReadLen((int)i);
    return l;
  }

  void Init() {
    Check(gaml_ctx_create(getenv("GAML_GPU_DEVICE") ? atoi(getenv("GAML_GPU_DEVICE")) : 0, &ctx_));
    vector<int32_t> node_len(gr.nodes.size());
    for (size_t i = 0; i < gr.nodes.size(); i++) node_len[i] = (int32_t)gr.nodes[i]->s.length();
    vector<int32_t> nmap(gr.normalize_map.begin(), gr.normalize_map.end());
    Check(gaml_set_graph(ctx_, (int)node_len.size(), node_len.data(), nmap.size() == node_len.size() ? nmap.data() : NULL));
    // CalcProb reports single sets, then paired, then pacbio (reference prob_calculator.h:70-107)
    for (auto& e : single_reads) {
      gaml_readset_config c = Cfg(GAML_KIND_SINGLE, e.first.penalty_constant, e.first.step, e.first.min_prob_per_base,
                                  e.first.min_prob_start, e.first.weight, e.second->match_prob_, e.second->mismatch_prob_);
      vector<int32_t> l = Lens(*e.second);
      int id = gaml_add_readset(ctx_, &c, (int64_t)l.size(), 0, (int64_t)l.size(), l.data(), NULL, -1, -1);
      Check(id);
      mirrors_.push_back(Mirror{e.second, id, 0, false, {}});
    }
    for (auto& e : paired_reads) {
      gaml_readset_config c = Cfg(GAML_KIND_PAIRED, e.first.penalty_constant, e.first.step, e.first.min_prob_per_base,
                                  e.first.min_prob_start, e.first.weight, e.second.first->match_prob_,
                                  e.second.first->mismatch_prob_);
      c.insert_mean = e.first.insert_mean;
      c.insert_std = e.first.insert_std;
      vector<int32_t> l1 = Lens(*e.second.first), l2 = Lens(*e.second.second);
      assert(l1.size() == l2.size());   // reference graph.cc:1962
      int id = gaml_add_readset(ctx_, &c, (int64_t)l1.size(), 0, (int64_t)l1.size(), l1.data(), l2.data(), -1, -1);
      Check(id);
      mirrors_.push_back(Mirror{e.second.first, id, 0, true, {}});
      mirrors_.push_back(Mirror{e.second.second, id, 1, true, {}});
    }
    for (auto& e : pacbio_reads) {
      // logdouble(double) = log (logdouble.hpp:18): the library's pacbio config wants the probabilities themselves
      gaml_readset_config c = Cfg(GAML_KIND_PACBIO, e.first.penalty_constant, e.first.step, e.first.min_prob_per_base,
                                  e.first.min_prob_start, e.first.weight, exp(e.second->match_prob_.logval),
                                  exp(e.second->mismatch_prob_.logval));
      vector<int32_t> l(e.second->GetNumberOfReads());
      for (size_t i = 0; i < l.size(); i++) l[i] = e.second->GetReadLen((int)i);
      int id = gaml_add_readset(ctx_, &c, (int64_t)l.size(), 0, (int64_t)l.size(), l.data(), NULL, -1, -1);
      Check(id);
      pb_mirrors_.push_back(PbMirror{e.second, id, {}});
    }
    n_sets_ = single_reads.size() + paired_reads.size() + pacbio_reads.size();
  }

  // Window key of node i inside a contig (reference graph.cc:552-561 / 618-627).
  vector<int> WindowKey(const vector<int>& ctg, size_t i) {
    vector<int> key(1, ctg[i]);
    int beyond = 0;
    for (size_t j = i + 1; j < ctg.size(); j++) {
      beyond += gr.nodes[ctg[j]]->s.length();
      key.push_back(ctg[j]);
      if (beyond > 300) break;   // kMinSubpathLength, graph.cc:27
    }
    return key;
  }

  void MirrorKey(Mirror& m, const vector<int>& key) {
    if (m.sent.count(key)) return;
    auto it = m.rs->aligment_cache_.find(key);
    if (it == m.rs->aligment_cache_.end()) return;   // never aligned: the reference treats it as an empty list
    m.sent.insert(key);
    static_assert(sizeof(Aligment) == sizeof(gaml_alignment), "Aligment is the ABI record");
    Check(gaml_cache_insert(ctx_, m.set, m.mate, key.data(), (int)key.size(),
                            reinterpret_cast<const gaml_alignment*>(it->second.data()), (int64_t)it->second.size(),
                            INT32_MIN));
  }

  // ReadSet::PrecomputeAlignmentForPaths (graph.cc:447-493) for the walks not seen before. The reference's loop carries
  // `last_end` from one walk into the next (it only decides whether the FIRST window of a walk joins the mass
  // precompute); a seen walk contributes its remembered final value and nothing else — every key it could add is in the
  // cache since its first evaluation.
  void PrecomputeNewWalks(ReadSet& rs, const vector<vector<int>>& paths, const vector<char>& is_new, vector<int>& final_end) {
    unordered_set<vector<int>> subpaths_precomp;
    int last_end = -1;
    for (size_t p = 0; p < paths.size(); p++) {
      const vector<int>& path = paths[p];
      if (!is_new[p]) {
        if (final_end[p] != kNoNode) last_end = final_end[p];
        continue;
      }
      for (int i = 0; i < (int)path.size(); i++) {
        if (path[i] < 0) continue;
        int cur_seq_len = 0;
        vector<int> cur_seq(1, path[i]);
        int cur_end = i;
        for (int j = i + 1; j < (int)path.size(); j++) {
          if (path[j] < 0) break;
          cur_seq_len += gr.nodes[path[j]]->s.length();
          cur_seq.push_back(path[j]);
          cur_end = j;
          if (cur_seq_len > 300) break;
        }
        if (rs.aligment_cache_.count(cur_seq) == 0 &&
            (last_end != cur_end || (cur_seq.size() == 1 && gr.nodes[cur_seq[0]]->s.length() > 150))) {
          subpaths_precomp.insert(cur_seq);
          subpaths_precomp.insert(InvertPath(cur_seq));
        }
        if (gr.nodes[path[i]]->s.length() > 300) {
          if (rs.aligment_cache_.count(vector<int>({path[i]})) == 0) {
            subpaths_precomp.insert(vector<int>({path[i]}));
            subpaths_precomp.insert(vector<int>({path[i] ^ 1}));
          }
        }
        last_end = cur_end;
      }
    }
    if (!subpaths_precomp.empty()) rs.PrecomputeAligmentForSubpaths(gr, USetToVector(subpaths_precomp));
  }

  static int FinalEnd(const vector<int>& path, const Graph& g) {   // last_end after the reference's loop over this walk
    int last = kNoNode;
    for (int i = 0; i < (int)path.size(); i++) {
      if (path[i] < 0) continue;
      int cur_seq_len = 0, cur_end = i;
      for (int j = i + 1; j < (int)path.size(); j++) {
        if (path[j] < 0) break;
        cur_seq_len += g.nodes[path[j]]->s.length();
        cur_end = j;
        if (cur_seq_len > 300) break;
      }
      last = cur_end;
    }
    return last;
  }

  // PacbioReadSet::GetReadProbabilities' cache fill (graph.cc:2438-2486) + mirroring for one NEW normalised walk.
  void FillAndMirrorPacbio(PbMirror& m, const vector<int>& path) {
    PacbioReadSet& rs = *m.rs;
    const size_t n = path.size();
    if (n == 0) return;
    vector<int> begin(n), end(n);
    int off = 0;
    for (size_t i = 0; i < n; i++) {
      begin[i] = off;
      off += path[i] < 0 ? -path[i] : (int)gr.nodes[path[i]]->s.length();
      end[i] = off;
    }
    vector<vector<int>> keys;
    vector<pair<int, int>> missing;
    for (size_t i = 0; i < n; i++) {
      vector<int> sub;
      for (size_t j = i; j < n; j++) {
        sub.push_back(path[j]);
        if (rs.aligment_cache_.count(sub) == 0) missing.push_back(make_pair((int)i, (int)j));
        keys.push_back(sub);
        if ((end[j] - begin[i]) - (end[i] - begin[i]) > rs.max_read_len_) break;   // graph.cc:2450
      }
    }
    if (!missing.empty()) {   // merged runs of missing windows go to the aligner, graph.cc:2455-2486
      int lastmissend = -47, lastmissbegin = -47;
      sort(missing.begin(), missing.end());
      for (size_t i = 0; i < missing.size(); i++) {
        if (missing[i].first > lastmissend) {
          if (lastmissend != -47) {
            int tl;
            rs.GetReadProbabilitiesSlow(gr, vector<int>(path.begin() + lastmissbegin, path.begin() + lastmissend + 1), tl);
          }
          lastmissbegin = missing[i].first;
          lastmissend = missing[i].second;
        }
        lastmissend = max(lastmissend, missing[i].second);
      }
      if (lastmissend != -47) {
        int tl;
        rs.GetReadProbabilitiesSlow(gr, vector<int>(path.begin() + lastmissbegin, path.begin() + lastmissend + 1), tl);
      }
    }
    vector<gaml_pacbio_alignment> recs;
    for (auto& key : keys) {
      if (m.sent.count(key)) continue;
      auto it = rs.aligment_cache_.find(key);
      if (it == rs.aligment_cache_.end()) continue;   // the reference asserts it is there by now (graph.cc:2497)
      m.sent.insert(key);
      recs.resize(it->second.size());
      for (size_t k = 0; k < recs.size(); k++) {
        recs[k].position = it->second[k].position;
        recs[k].position_end = it->second[k].position_end;
        recs[k].read_id = it->second[k].read_id;
        recs[k].pad = 0;
        recs[k].logprob = it->second[k].prob.logval;
      }
      Check(gaml_cache_insert_pacbio(ctx_, m.set, key.data(), (int)key.size(), recs.data(), (int64_t)recs.size()));
    }
  }

  // `paths` = the caller's walks, `cur` = the same flattened, `old` / `old_final_end` = the list to compare with.
  // Fills final_end (per walk of `cur`) and, when asked, the alignment.
  void FillAndMirrorCaches(const vector<vector<int>>& paths, const FlatPaths& cur, const FlatPaths& old,
                           const vector<int>& old_final_end, vector<int>& final_end, vector<int>* match_out) {
    // which walks are new to the adapter: aligned with an equal walk of the previous list (block compares on the flat
    // arrays), else the set of all walks ever evaluated (one hash probe)
    vector<int>& match = match_out ? *match_out : match_;
    if (have_prev_) gaml_flat::Align(old, cur, match);
    else match.assign(paths.size(), -1);
    is_new_.assign(paths.size(), 0);
    vector<char>& is_new = is_new_;
    final_end.resize(paths.size());
    bool any_new = false;
    for (size_t p = 0; p < paths.size(); p++) {
      if (match[p] >= 0) {
        final_end[p] = old_final_end[(size_t)match[p]];
        continue;
      }
      auto it = seen_.find(paths[p]);
      if (it != seen_.end()) {
        final_end[p] = it->second;
      } else {
        is_new[p] = 1;
        any_new = true;
        final_end[p] = FinalEnd(paths[p], gr);
      }
    }
    if (any_new) {
      // (1) the reference's own cache-filling calls where CalcScoreForPathsNew / GetPositionsOnlyPath / AddPositions run
      //     them, so the same keys get aligned (internal min-hash aligner or bowtie2)
      for (auto& e : paired_reads) {
        PrecomputeNewWalks(*e.second.first, paths, is_new, final_end);    // graph.cc:1967
        PrecomputeNewWalks(*e.second.second, paths, is_new, final_end);   // graph.cc:1968
      }
      for (auto& m : mirrors_) {
        for (size_t p = 0; p < paths.size(); p++) {
          if (!is_new[p]) continue;
          const vector<int>& path = paths[p];
          vector<int> ctg;
          for (size_t i = 0; i <= path.size(); i++) {
            if (i == path.size() || path[i] < 0) {
              unordered_set<vector<int>> missing;
              m.rs->GetSubpathsFromPath(ctg, gr, missing);          // graph.cc:538-542, 605-609
              if (!missing.empty()) m.rs->PrecomputeAligmentForSubpaths(gr, USetToVector(missing));
              // (2) mirror every key this contig looks up and the device does not hold yet
              for (size_t k = 0; k < ctg.size(); k++) {
                MirrorKey(m, WindowKey(ctg, k));
                if (m.paired && gr.nodes[ctg[k]]->s.length() > 300) MirrorKey(m, vector<int>(1, ctg[k]));   // graph.cc:563-566
              }
              ctg.clear();
            } else {
              ctg.push_back(path[i]);
            }
          }
        }
      }
      for (auto& m : pb_mirrors_) {
        for (size_t p = 0; p < paths.size(); p++) {
          if (!is_new[p]) continue;
          vector<int> path = paths[p];
          gr.NormalizePath(path);                                    // graph.cc:3184
          FillAndMirrorPacbio(m, path);
        }
      }
      for (size_t p = 0; p < paths.size(); p++)
        if (is_new[p]) seen_.emplace(paths[p], final_end[p]);
    }
  }

  gaml_ctx* ctx_;
  size_t n_sets_ = 0;
  vector<Mirror> mirrors_;
  vector<PbMirror> pb_mirrors_;
  unordered_map<vector<int>, int> seen_;   // every walk evaluated so far -> its FinalEnd
  FlatPaths cur_, prev_;                   // this call's walks / the last evaluated ones, in the C ABI's layout
  vector<int> prev_final_end_, cur_final_end_;
  vector<int> match_;
  vector<char> is_new_;
  vector<int32_t> z_;
  bool have_prev_ = false;
  bool had_calc_ = false;
};

// Two-pass replay for a move that scores a LIST of alternatives and acts on them in order (first improvement wins,
// similar scores are remembered, ...): pass 0 runs the move's own loop unchanged except that Score() records the
// candidate and answers NaN — every comparison the loops make on a score is false for NaN, so pass 0 has no effect
// besides building the candidates; End() scores them in ONE batch; pass 1 runs the loop again with the real scores, in
// the same order. oracle/build_ref.sh wraps the loops of moves.cc with it (in the compiler's input stream).
struct GamlBatchReplay {
  explicit GamlBatchReplay(ProbCalculator& pc) : pc_(pc), pass_(0), next_(0) {}
  void Begin(int pass) {
    pass_ = pass;
    next_ = 0;
    if (pass == 0) sets_.clear();
  }
  double Score(vector<vector<int>>& paths) {
    if (pass_ == 0) {
      sets_.push_back(paths);
      return std::numeric_limits<double>::quiet_NaN();
    }
    return scores_[next_++];
  }
  void End() {
    if (pass_ == 0) scores_ = pc_.CalcProbBatch(sets_);
  }
  ProbCalculator& pc_;
  int pass_;
  size_t next_;
  vector<vector<vector<int>>> sets_;
  vector<double> scores_;
};

#endif
