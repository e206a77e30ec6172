// train.cpp -- EM outer loop (host) driving the CUDA library through the C ABI.
//
// Mirrors WFST::train (carmel/src/train.cc:503-678): convergence tests, best-perplexity bookkeeping,
// over-relaxation schedule and the exact log lines, with forward_backward::estimate / maximize
// (train.cc:763-773,893-923) replaced by cml_estimate / cml_maximize.  All per-arc state the reference
// keeps in arcs_table<arc_counts> (weights, counts, scratch, em_weight, best_weight) lives on the GPU.
#include <algorithm>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>

#include "carmel_host.hpp"

namespace cb {

TrainOpts::TrainOpts() : ln_converge_delta(std::log(1e-4)), ln_converge_ratio(std::log(.999)) {}

void add_model_member(Wfst const& w, NormalizeMethod const& m, ModelArrays& M) {
  // normalisation groups: all arcs leaving a state (JOINT) or leaving a state with the same input
  // symbol (CONDITIONAL); NONE keeps weights (carmel/src/fst.h:1362-1446, cascade.h:339-350)
  std::unordered_map<uint32_t, uint32_t> tie_ids;  // '!N' ids are local to a transducer
  for (auto const& st : w.states) {
    std::unordered_map<uint32_t, uint32_t> by_input;
    uint32_t joint_group = kNoGroup;
    for (Arc const& a : st) {
      uint32_t g = kNoGroup;
      if (m.group == JOINT) {
        if (joint_group == kNoGroup) {
          joint_group = M.n_groups++;
          M.group_add.push_back(m.ln_add_count);
        }
        g = joint_group;
      } else if (m.group == CONDITIONAL) {
        auto it = by_input.find(a.in);
        if (it == by_input.end()) {
          it = by_input.emplace(a.in, M.n_groups++).first;
          M.group_add.push_back(m.ln_add_count);
        }
        g = it->second;
      }
      M.param_group.push_back(g);
      uint32_t t = a.group;
      if (t != kNoGroup && t != kLocked) {
        auto it = tie_ids.find(t);
        if (it == tie_ids.end()) it = tie_ids.emplace(t, ++M.n_ties).first;
        t = it->second;
      }
      M.param_tie.push_back(t);
      M.ln_w.push_back(a.ln_w);
    }
  }
}

namespace {

// logweight::root / ppxper keep a zero weight zero (weight.h:435-440, WEIGHT_CORRECT_ZERO): a corpus with a
// zero-probability example therefore has "perplexity 0", which the reference then treats as the best
inline bool w_is_zero(double ln) { return !(ln > kNegInf); }
inline double w_root(double ln, double n) { return w_is_zero(ln) ? ln : ln / n; }

void print_ppx(std::ostream& log, double ln_corpus_p, Corpus const& c) {  // weight.h:311-329
  log << "probability=" << format_base2(ln_corpus_p);
  const double n_symbol = std::max(c.n_output, c.n_input);
  if (n_symbol) log << " per-output-symbol-perplexity(N=" << n_symbol << ")=" << format_base2(w_root(ln_corpus_p, -n_symbol));
  if (c.n_pairs) log << " per-example-perplexity(N=" << c.n_pairs << ")=" << format_base2(w_root(ln_corpus_p, -(double)c.n_pairs));
}

}  // namespace

void TrainJob::ok(int rc) const {
  if (rc != CML_OK) throw std::runtime_error(std::string("carmel_b200: ") + cml_last_error(ctx));
}

TrainJob::~TrainJob() {
  if (ctx) cml_destroy(ctx);
}

void shard_range(Corpus const& corpus, int rank, int count, size_t& e0, size_t& e1) {
  const size_t n = corpus.examples.size();
  e0 = 0;
  e1 = n;
  if (count <= 1) return;
  std::vector<double> cost(n + 1, 0.);
  for (size_t e = 0; e < n; ++e) cost[e + 1] = cost[e] + 1. + corpus.examples[e].in.size() + corpus.examples[e].out.size();
  auto cut = [&](int r) {
    const double target = cost.back() * r / count;
    return std::min(n, (size_t)(std::lower_bound(cost.begin(), cost.end(), target) - cost.begin()));
  };
  e0 = rank == 0 ? 0 : cut(rank);
  e1 = rank == count - 1 ? n : cut(rank + 1);
  if (e1 < e0) e1 = e0;
}

// The dense-state view of this shard: symbol sequences + the arc table's (source, destination, symbol) triples.
// Examples without a derivation are found by a reachability pass over the supports (bit masks, S <= 32) and
// dropped like the lattice builder drops them; the same pass counts the states and arcs the reference's pruned
// lattices would have (derivations.h:572-629), which is what the throughput figures are quoted in.
// Returns false (nothing changed) when the library finds no transition x emission factorisation.
bool TrainJob::try_dense(int tape, Corpus const& local, std::vector<uint32_t>& kept, std::vector<uint32_t>& dropped) {
  const uint32_t S = x->num_states();
  std::unordered_map<uint32_t, uint32_t> sym_id;
  std::vector<uint32_t> a_src, a_dst, a_sym;
  const uint32_t fin = x->final_state;
  uint64_t phi_mask = 0;  // states with an epsilon arc into the final state (final weights)
  for (uint32_t s = 0; s < S; ++s)
    for (Arc const& a : x->states[s]) {
      const uint32_t sy = tape ? a.out : a.in;
      uint32_t id = CML_DENSE_EPS;
      if (sy != kEps) {
        auto it = sym_id.find(sy);
        if (it == sym_id.end()) it = sym_id.emplace(sy, (uint32_t)sym_id.size()).first;
        id = it->second;
      } else
        phi_mask |= 1ull << s;
      a_src.push_back(s);
      a_dst.push_back(a.dest);
      a_sym.push_back(id);
    }
  const uint32_t V = (uint32_t)sym_id.size();
  if (V == 0 || V > 65535) return false;
  std::vector<uint64_t> adj((size_t)V * S, 0), radj((size_t)V * S, 0);  // [symbol][state] -> successor / predecessor masks
  for (size_t a = 0; a < a_src.size(); ++a) {
    if (a_sym[a] == CML_DENSE_EPS) continue;
    adj[(size_t)a_sym[a] * S + a_src[a]] |= 1ull << a_dst[a];
    radj[(size_t)a_sym[a] * S + a_dst[a]] |= 1ull << a_src[a];
  }
  const uint64_t goal_mask = phi_mask ? phi_mask : (1ull << fin);  // lattice states of the last position that reach the goal
  std::vector<uint64_t> seq_off{0};
  std::vector<uint32_t> syms;
  std::vector<double> wts;
  std::vector<uint64_t> fwd;
  std::vector<uint32_t> cur;
  uint64_t n_states = 0, n_arcs = 0;
  for (uint32_t e = 0; e < local.examples.size(); ++e) {
    std::vector<uint32_t> const& str = tape ? local.examples[e].out : local.examples[e].in;
    const size_t n = str.size();
    cur.resize(n);
    bool known = true;
    for (size_t t = 0; t < n && known; ++t) {
      auto it = sym_id.find(str[t]);
      known = it != sym_id.end();
      if (known) cur[t] = it->second;
    }
    bool alive = known;
    if (alive) {
      fwd.assign(n + 1, 0);
      fwd[0] = 1ull;
      for (size_t t = 0; t < n; ++t) {
        uint64_t m = fwd[t], nx = 0;
        const uint64_t* row = &adj[(size_t)cur[t] * S];
        while (m) {
          const int i = __builtin_ctzll(m);
          m &= m - 1;
          nx |= row[i];
        }
        fwd[t + 1] = nx;
      }
      alive = (fwd[n] & goal_mask) != 0;
    }
    if (!alive) {
      dropped.push_back(e);
      continue;
    }
    // co-reachability; live_t = fwd_t & bwd_t, arcs between consecutive live sets
    uint64_t live_next = fwd[n] & goal_mask;
    uint64_t st = __builtin_popcountll(live_next), ar = 0;
    if (phi_mask) {  // the epsilon arcs of the last position and the final state itself
      ar += st;
      st += 1;
    }
    for (size_t t = n; t-- > 0;) {
      uint64_t m = live_next, pv = 0;
      const uint64_t* rrow = &radj[(size_t)cur[t] * S];
      while (m) {
        const int j = __builtin_ctzll(m);
        m &= m - 1;
        pv |= rrow[j];
      }
      const uint64_t live = pv & fwd[t];
      const uint64_t* row = &adj[(size_t)cur[t] * S];
      m = live;
      while (m) {
        const int i = __builtin_ctzll(m);
        m &= m - 1;
        ar += __builtin_popcountll(row[i] & live_next);
      }
      st += __builtin_popcountll(live);
      live_next = live;
    }
    n_states += st;
    n_arcs += ar;
    kept.push_back(e);
    syms.insert(syms.end(), cur.begin(), cur.end());
    seq_off.push_back(syms.size());
    wts.push_back(local.examples[e].weight);
  }
  cml_dense_view v{};
  v.n_states = S;
  v.n_symbols = V;
  v.start = 0;
  v.final_state = fin;
  v.arc_src = a_src.data();
  v.arc_dst = a_dst.data();
  v.arc_sym = a_sym.data();
  cml_sequence_batch b{};
  b.n_seq = wts.size();
  b.seq_off = seq_off.data();
  b.sym = syms.data();
  b.seq_weight = wts.data();
  const int rc = cml_add_sequences(ctx, &v, &b);
  if (rc == CML_ERR_NOT_DENSE) {
    if (!opt.quiet && !flags[(unsigned)'q']) std::cerr << "dense-state view not applicable (" << cml_last_error(ctx) << "); using lattices\n";
    kept.clear();
    dropped.clear();
    return false;
  }
  ok(rc);
  uint32_t nt = 0, ne = 0, kk = 0;
  int sparse = 0;
  ok(cml_dense_stats(ctx, nullptr, nullptr, &nt, &ne));
  ok(cml_dense_kernel(ctx, &sparse, &kk, nullptr));
  if (!opt.quiet && !flags[(unsigned)'q']) {
    std::cerr << "dense-state path: " << S << " states x " << V << " symbols, " << nt << " trainable transition cells, "
              << ne << " trainable emission cells";
    if (sparse == 1) std::cerr << " (sparse emission rows of " << kk << ", one sequence per lane)";
    if (sparse == 2) std::cerr << " (3xTF32 tensor-core sweeps, 16 sequences per warp)";
    std::cerr << "\n";
  }
  res.trellis_arcs = n_arcs;
  res.trellis_states = n_states;
  res.examples = wts.size();
  res.dense = true;
  return true;
}

// The model on the GPU: context, model tables, parameters after the initial normalisation, prior counts.
void TrainJob::prepare_model() {
  build_model();
  if (cml_create(&ctx, opt.device, opt.precision, opt.space) != CML_OK)
    throw std::runtime_error(std::string("carmel_b200: ") + cml_last_error(nullptr));
  if (opt.max_iter == 0) ok(cml_set_option(ctx, CML_OPT_ARC_COUNTS, 1));  // -M 0 writes per-arc fractional counts
  if (opt.no_ell) ok(cml_set_option(ctx, CML_OPT_NO_ELL, 1));
  if (opt.lane_min >= 0) ok(cml_set_option(ctx, CML_OPT_LANE_MIN, opt.lane_min));
  if (opt.shard_count > 1) {
    ok(cml_set_option(ctx, CML_OPT_ALLOW_EMPTY, 1));  // a rank whose block has no usable example still joins every collective
    if (have_comm_id) ok(cml_comm_init_rank(ctx, (int)opt.shard_count, (int)opt.shard_rank, comm_id));
  }
  if (opt.no_factor) ok(cml_set_option(ctx, CML_OPT_NO_FACTOR, 1));
  if (opt.no_wide) ok(cml_set_option(ctx, CML_OPT_NO_WIDE, 1));
  // locality keys: arcs with the same output symbol, then source state, are laid out together on the GPU,
  // so the weight gathers of one lattice level (one output position) fall into few cache sectors
  {
    uint32_t src = 0;
    for (auto const& st : x->states) {
      for (Arc const& a : st)
        M.arc_key.push_back(((uint64_t)(a.out & 0xFFFFF) << 44) | ((uint64_t)(a.in & 0xFFFFF) << 24) |
                            ((uint64_t)(src & 0xFFF) << 12) | (uint64_t)(a.dest & 0xFFF));
      ++src;
    }
  }
  cml_model mm{};
  mm.arc_locality_key = M.arc_key.data();
  mm.n_arcs = M.n_arcs;
  mm.chain_off = using_cascade ? M.chain_off.data() : nullptr;
  mm.chain_param = using_cascade ? M.chain_param.data() : nullptr;
  mm.arc_prior = nullptr;
  mm.n_params = M.n_params;
  mm.param_group = M.param_group.data();
  mm.param_tie = M.param_tie.data();
  mm.n_groups = M.n_groups;
  mm.group_add = M.group_add.data();
  mm.n_ties = M.n_ties;
  ok(cml_set_model(ctx, &mm));
  ok(cml_set_params(ctx, M.ln_w.data()));
  ok(cml_normalize_params(ctx));  // train.cc:509 cascade.normalize(methods)

  // prior counts per arc-table entry (train.cc:134-153; derivations.h:96-101): the -f floor, plus
  // the (normalised) arc weight itself with -U
  if (opt.ln_smooth_floor > kNegInf || opt.weight_is_prior) {
    std::vector<double> w(M.n_params);
    ok(cml_get_params(ctx, w.data()));
    M.arc_prior.assign(M.n_arcs, opt.ln_smooth_floor > kNegInf ? std::exp(opt.ln_smooth_floor) : 0.);
    if (opt.weight_is_prior)
      for (uint32_t a = 0; a < M.n_arcs; ++a) {
        double lw = 0;
        if (using_cascade)
          for (uint32_t k = M.chain_off[a]; k < M.chain_off[a + 1]; ++k) lw += w[M.chain_param[k]];
        else
          lw = w[a];
        M.arc_prior[a] += std::exp(lw);
      }
    mm.arc_prior = M.arc_prior.data();
    ok(cml_set_model(ctx, &mm));  // (no lattices are resident yet)
    ok(cml_set_params(ctx, w.data()));
  }
}

// Everything up to the first E-step: the model (prepare_model), derivation lattices (this rank's shard) flattened and
// resident on the GPU.
void TrainJob::prepare() {
  if (prepared) return;
  prepare_model();

  // ---- derivation lattices: built once, resident on the GPU (carmel's -: cache semantics) ----
  // With --shard=r/N only a contiguous block of the corpus (balanced by string length) is built and
  // kept on this GPU; corpus statistics are then made global through the all-reduce hook.
  // Dense-state view (cml_add_sequences): every arc consumes one symbol of one tape and the other tape of
  // every pair is empty -> lattice states are (position, state) and nothing needs to be materialised.  The
  // decision is made on the WHOLE corpus and the model, so every rank of a sharded run takes the same path.
  int dense_tape = -1;  // 0: symbols on the input tape, 1: on the output tape
  if (opt.dense >= 0 && opt.space == CML_SPACE_SCALED && opt.max_iter != 0 && opt.dump_trellis_file.empty() &&
      x->num_states() <= 64) {
    // every arc consumes one symbol of one tape; *e*:*e* arcs are candidates for final weights (the library checks)
    bool in_only = true, out_only = true;
    for (auto const& st : x->states)
      for (Arc const& a : st) {
        const bool eps = a.in == kEps && a.out == kEps;
        in_only = in_only && (eps || (a.in != kEps && a.out == kEps));
        out_only = out_only && (eps || (a.out != kEps && a.in == kEps));
      }
    for (Example const& ex : corpus.examples) {
      in_only = in_only && ex.out.empty();
      out_only = out_only && ex.in.empty();
    }
    dense_tape = out_only ? 1 : in_only ? 0 : -1;
  }
  size_t e0, e1;
  shard_range(corpus, opt.shard_rank, opt.shard_count, e0, e1);
  {
    Corpus local;
    local.examples.assign(std::make_move_iterator(corpus.examples.begin() + e0),
                          std::make_move_iterator(corpus.examples.begin() + e1));
    TrellisBatch tb;
    std::vector<uint32_t> dropped, kept;
    bool dense_done = false;
    if (dense_tape >= 0) dense_done = try_dense(dense_tape, local, kept, dropped);
    if (opt.dense > 0 && !dense_done)
      throw std::runtime_error(std::string("--dense: no dense-state view of this model / corpus") +
                               (ctx ? std::string(": ") + cml_last_error(ctx) : std::string()));
    if (!dense_done) {
      if (opt.device_build > 0) {  // (measured: not faster than 16 host threads at 1M sentences -- DESIGN.md; opt-in)
        double secs = 0;
        build_trellises_device(ctx, *x, local, tb, dropped, &secs);
        res.device_build_s = secs;
      } else
        build_trellises(*x, local, tb, dropped);
      kept = tb.kept_example;
    }
    corpus_size = e1 - e0;
    kept_example.clear();
    for (uint32_t e : kept) kept_example.push_back((uint32_t)(e0 + e));
    for (uint32_t e : dropped)  // cached_derivs.h:53-57,87-93
      std::cerr << "No derivations in transducer for input/output #" << e0 + e + 1 << ":\n";
    std::vector<Example> keep;
    keep.reserve(kept.size());
    for (uint32_t e : kept) keep.push_back(std::move(local.examples[e]));
    corpus.examples.swap(keep);
    corpus.count();
    if (opt.shard_count > 1) {  // global corpus statistics: one small all-reduce
      double h[4] = {(double)corpus.n_pairs, corpus.total_weight, corpus.n_input, corpus.n_output};
      if (have_comm_id) {
        ok(cml_allreduce_host(ctx, h, 4));
      } else {
        if (!allreduce) throw std::runtime_error("--shard needs a communicator (cml_job_set_comm / --gpus) or an all-reduce hook");
        void* buf;
        uint64_t nbuf;
        ok(cml_reduce_buffer(ctx, &buf, &nbuf));
        ok(cml_reduce_buffer_write(ctx, h, 4));  // (synchronises the context's stream)
        // hook contract: the sum is complete in device memory when the hook returns
        allreduce(allreduce_user, buf, nbuf);
        ok(cml_reduce_buffer_read(ctx, h, 4));
      }
      corpus.n_pairs = (uint32_t)(h[0] + .5);
      corpus.total_weight = h[1];
      corpus.n_input = h[2];
      corpus.n_output = h[3];
    }
    if (corpus.n_pairs == 0) {
      std::cerr << "No training example had a derivation - check your models, quotes, manually compose with -i, etc.\n";
      throw std::runtime_error("No training example had a derivation - aborting training.");
    }
    if (!opt.dump_trellis_file.empty()) {
      std::ofstream o(opt.dump_trellis_file, std::ios::binary);
      tb.dump(o, M.n_arcs);
    }
    if (lopt.count("fem-forest") && opt.shard_rank == 0) export_fem_forest(tb, std::cerr);
    if (!dense_done) {
      if (!tb.ex_states.empty()) {
        cml_trellis_batch b{};
        b.n_ex = tb.ex_states.size();
        b.ex_states = tb.ex_states.data();
        b.ex_fin = tb.ex_fin.data();
        b.ex_weight = tb.ex_weight.data();
        b.arc_off = tb.arc_off.data();
        b.arc_dst = tb.arc_dst.data();
        b.arc_id = tb.arc_id.data();
        ok(cml_add_trellises(ctx, &b));
        uint64_t cyc = 0, back = 0;
        ok(cml_cyclic_stats(ctx, &cyc, &back));
        if (cyc)  // derivations.h:726-728 (the reference prints this once per example)
          std::cerr << "Warning: at least one cycle in derivations for " << cyc << " example(s) (" << back
                    << " back edges).  Forward/backward will miss some paths.\n";
      }
      res.trellis_arcs = tb.arc_dst.size();
      res.examples = tb.ex_states.size();
      for (uint32_t n : tb.ex_states) res.trellis_states += n;
    }
  }
  prepared = true;
}

// one E-step over all resident lattices (+ the per-iteration all-reduce when sharded)
double TrainJob::estimate(double& ln_unweighted) {
  cml_estimate_result r;
  ok(cml_estimate_launch(ctx));
  if (opt.shard_count > 1) {
    if (have_comm_id) {
      ok(cml_allreduce_counts(ctx));  // NCCL, stream-ordered behind the E-step kernels
    } else if (allreduce) {
      // hook contract: the E-step has finished before the hook runs (it may use any stream), and the sum is
      // complete in device memory when it returns
      void* buf;
      uint64_t nbuf;
      ok(cml_reduce_buffer(ctx, &buf, &nbuf));
      ok(cml_synchronize(ctx));
      allreduce(allreduce_user, buf, nbuf);
    }
  }
  ok(cml_estimate_finish(ctx, &r));
  if (r.n_zero) {  // some example has probability zero: the corpus probability is zero
    ln_unweighted = kNegInf;
    return kNegInf;
  }
  ln_unweighted = r.sum_ln_p;
  return r.sum_w_ln_p;
}

void TrainJob::write_back() {  // device parameters -> transducer arcs
  std::vector<double> w(M.n_params);
  ok(cml_get_params(ctx, w.data()));
  size_t p = 0;
  for (Wfst* m : members)
    for (auto& st : m->states)
      for (Arc& a : st) a.ln_w = w[p++];
  if (using_cascade) {  // cascade.update(): composed weights = chain products
    size_t a_id = 0;
    for (auto& st : x->states)
      for (Arc& a : st) {
        double lw = 0;
        for (uint32_t k = M.chain_off[a_id]; k < M.chain_off[a_id + 1]; ++k) lw += w[M.chain_param[k]];
        a.ln_w = lw;
        ++a_id;
      }
  }
}

// cascade.random_restart (cascade.h:398-411): WFST::randomSet on every member that is normalised (state.h:84-102:
// locked arcs keep their weight, the arcs of a tie group share one draw), then normalize
void TrainJob::random_restart(std::mt19937_64& rng) {
  std::vector<double> w(M.n_params);
  ok(cml_get_params(ctx, w.data()));
  std::unordered_map<uint32_t, double> tied;
  std::uniform_real_distribution<double> u01(0., 1.);
  for (uint32_t p = 0; p < M.n_params; ++p) {
    if (M.param_group[p] == kNoGroup || M.param_tie[p] == kLocked) continue;
    if (M.param_tie[p] == kNoGroup) {
      w[p] = std::log(1. - u01(rng));  // (0,1]
      continue;
    }
    auto it = tied.find(M.param_tie[p]);
    if (it == tied.end()) it = tied.emplace(M.param_tie[p], std::log(1. - u01(rng))).first;
    w[p] = it->second;
  }
  ok(cml_set_params(ctx, w.data()));
  ok(cml_normalize_params(ctx));
}

// WFST::random_restart_acceptor (fst.h:999-1044).  All quantities are natural logs; +inf = accept anything.
RestartAcceptor::RestartAcceptor(double final_at_n, double ln_tol, double ln_final_tol)
    : ln_tolerance(ln_tol), ln_final_tolerance(ln_final_tol), n(final_at_n) {
  const double inf = std::numeric_limits<double>::infinity();
  if (!(ln_tolerance > kNegInf)) ln_tolerance = inf;  // a zero tolerance means none was given
  if (!(ln_final_tolerance > kNegInf)) ln_final_tolerance = ln_tolerance;
}
double RestartAcceptor::ln_likelihood_ratio(uint32_t i) const {
  if (i >= n) return ln_final_tolerance;
  if (std::isinf(ln_tolerance)) return ln_tolerance;
  return ln_tolerance + (ln_final_tolerance - ln_tolerance) * ((i - 1) / (n - 1));
}
bool RestartAcceptor::accept(double ln_this_start, uint32_t restart_i, std::ostream& o) {
  if (restart_i == 0) {
    ln_best_start = ln_this_start;
    o << "Initial best start point ppx=" << format_base2(ln_this_start) << std::endl;
    return true;
  }
  const double lr = ln_likelihood_ratio(restart_i);
  const double ppr = w_root(ln_this_start - ln_best_start, std::fabs(ln_this_start));  // relative_perplexity_ratio
  const bool r = lr > ppr;
  o << "For restart " << restart_i << ", " << (r ? "accepting" : "rejecting") << " worse random start of "
    << format_base2(ln_this_start) << " compared to " << format_base2(ln_best_start) << " with relative ppx ratio="
    << format_weight(ppr) << " compared to target of " << format_weight(lr) << std::endl;
  return r;
}

void TrainJob::finish() {
  if (!opt.history_file.empty()) {
    std::ofstream o(opt.history_file);
    o.precision(17);
    for (auto const& h : res.history) o << h.iter << ' ' << h.ln_prob << ' ' << h.ln_weighted_prob << ' ' << h.max_change << '\n';
  }
}

TrainResult const& TrainJob::run(std::ostream& log) {
  prepare();
  double ln_corpus_p = 0;
  if (opt.max_iter + 1 == 0) {  // -M -1: the likelihood of the (normalised) input weights, nothing else (train.cc:516-517)
    const double p = estimate(ln_corpus_p);
    res.history.push_back({1, ln_corpus_p, p, 0});
    res.ln_best_ppx = w_root(p, -corpus.total_weight);
    write_back();
    finish();
    return res;
  }
  // ---- -M 0 / -M 1: fractional counts only / a single iteration (train.cc:520-538) ----
  if (opt.max_iter == 0 || (opt.max_iter == 1 && opt.ran_restarts == 0)) {  // (train.cc:520)
    const double p = estimate(ln_corpus_p);
    res.history.push_back({1, ln_corpus_p, p, 0});
    log << "Corpus ";
    print_ppx(log, ln_corpus_p, corpus);
    if (opt.max_iter == 0) {
      log << "0 iterations specified for training; output weights will be unnormalized fractional counts (except locked arcs).\n";
      std::vector<double> counts(M.n_arcs);
      ok(cml_get_arc_counts(ctx, counts.data()));
      size_t a_id = 0;
      for (auto& st : x->states)
        for (Arc& a : st) {
          const double c = counts[a_id] + (M.arc_prior.empty() ? 0. : M.arc_prior[a_id]);
          if (a.group != kLocked || using_cascade) a.ln_w = c > 0 ? std::log(c) : kNegInf;
          ++a_id;
        }
      if (using_cascade) {
        // cascade.distribute_counts (cascade.h:286-325): unlocked member arcs are zeroed, then every composed arc's
        // count + prior is added to each unlocked arc of its chain; locked member arcs keep their weights
        std::vector<double> acc(M.n_params, 0.);
        for (uint32_t a = 0; a < M.n_arcs; ++a) {
          const double c = counts[a] + (M.arc_prior.empty() ? 0. : M.arc_prior[a]);
          for (uint32_t k = M.chain_off[a]; k < M.chain_off[a + 1]; ++k) acc[M.chain_param[k]] += c;
        }
        size_t p = 0;
        for (Wfst* m : members)
          for (auto& st : m->states)
            for (Arc& a : st) {
              if (M.param_tie[p] != kLocked) a.ln_w = acc[p] > 0 ? std::log(acc[p]) : kNegInf;
              ++p;
            }
      }
    } else {
      double d;
      ok(cml_maximize(ctx, 1., &d));
      write_back();
    }
    log << "\n";
    res.ln_best_ppx = w_root(p, -corpus.total_weight);
    finish();
    return res;
  }

  // ---- main loop (train.cc:540-667, single start) ----
  const double kInf = std::numeric_limits<double>::infinity();
  double ln_best_ppx = kInf;
  double growth = opt.rate_growth;
  if (using_cascade && growth != 1) {
    std::cerr << "Overrelaxed EM not supported for --train-cascade.  Disabling (growth factor=1)." << std::endl;
    growth = 1;
  }
  bool have_good_weights = false;
  const int SLOT_BEST = 0, SLOT_EM = 1;
  // random restarts (-! n, train.cc:553-667 outer loop): every further start draws the unlocked parameters
  // uniformly on (0,1], renormalises, and trains again; the best iteration of any start is kept
  uint32_t ran_restarts = opt.ran_restarts;
  RestartAcceptor ra(opt.final_restart ? opt.final_restart : opt.ran_restarts, opt.ln_restart_tolerance,
                     opt.ln_final_restart_tolerance);
  std::mt19937_64 restart_rng(opt.seed);
  for (uint32_t restart_no = 0;; ++restart_no) {
  uint32_t train_iter = 0;
  double ln_last_change = std::log(10.);
  double ln_last_ppx = kInf;
  double learning_rate = 1;
  bool last_was_reset = false;
  for (;;) {
    const bool first_time = train_iter == 0;
    ++train_iter;
    const bool cascade_counts = using_cascade && !first_time;
    if (~opt.max_iter && train_iter > opt.max_iter && have_good_weights) {
      log << "Maximum number of iterations (" << opt.max_iter
          << ") reached before convergence criteria was met - greatest arc weight change was "
          << format_weight(ln_last_change) << "\n";
      break;
    }
    if (~opt.max_iter && train_iter > opt.max_iter + 1) {
      // the reference would iterate forever here (no iteration was ever accepted as "best"); stop instead
      std::cerr << "Warning: no iteration produced usable weights after " << opt.max_iter << " iterations; stopping.\n";
      ok(cml_snapshot_params(ctx, SLOT_BEST));
      break;
    }
    const double p = estimate(ln_corpus_p);
    const double ln_new_ppx = w_root(p, -corpus.total_weight);  // ppxper(totalEmpiricalWeight)
    res.history.push_back({train_iter, ln_corpus_p, p, std::exp(ln_last_change)});
    log << "i=" << train_iter << " (rate=" << learning_rate << "): ";
    print_ppx(log, ln_corpus_p, corpus);
    if (ln_new_ppx < ln_best_ppx && (!using_cascade || cascade_counts)) {
      log << " (new best)";
      ln_best_ppx = ln_new_ppx;
      have_good_weights = true;
      ok(cml_snapshot_params(ctx, SLOT_BEST));  // save_best
    }
    double ln_ratio;
    if (first_time) {
      log << std::endl;
      if (!ra.accept(ln_new_ppx, restart_no, log)) {
        log << "Random start was insufficiently promising; trying another." << std::endl;
        break;  // to the next random restart
      }
      ln_ratio = kNegInf;
    } else {
      // relative_perplexity_ratio (weight.h:247-249): (new/old)^(1/|ln new|)
      ln_ratio = w_root(ln_new_ppx - ln_last_ppx, std::fabs(ln_new_ppx));
      log << " (relative-perplexity-ratio=" << format_weight(ln_ratio) << ")";
      if (ln_last_change < 0) log << ", max {d(weight)}=" << format_weight(ln_last_change);
      log << std::endl;
    }
    if (!last_was_reset) {
      if (ln_ratio >= opt.ln_converge_ratio) {
        if (learning_rate > 1) {
          log << "Failed to improve (relaxation rate too high); starting again at learning rate 1" << std::endl;
          learning_rate = 1;
          ok(cml_restore_params(ctx, SLOT_EM));  // keep_em_weight
          last_was_reset = true;
          continue;
        }
        log << "Converged - per-example perplexity ratio exceeds " << format_weight(opt.ln_converge_ratio) << " after "
            << train_iter << " iterations.\n";
        if (!have_good_weights)
          log << "Because of the --train-cascade implementation, we need another iteration even though we've converged.\n";
        else
          break;
      } else {
        if (learning_rate < 20) learning_rate *= growth;  // MAX_LEARNING_RATE_EXP, config.h:145
      }
    } else
      last_was_reset = false;
    double max_delta = 10;
    if (learning_rate > 1.) {
      // the raw EM weights (rate 1) are needed if the relaxed step fails: compute them first
      ok(cml_snapshot_params(ctx, 2));
      ok(cml_maximize(ctx, 1., &max_delta));
      ok(cml_snapshot_params(ctx, SLOT_EM));
      ok(cml_restore_params(ctx, 2));
    }
    ok(cml_maximize(ctx, learning_rate, &max_delta));
    if (using_cascade) max_delta = 10;  // train.cc:921-922
    ln_last_change = max_delta > 0 ? std::log(max_delta) : kNegInf;
    if (ln_last_change <= opt.ln_converge_delta && have_good_weights) {
      log << "Converged - maximum weight change less than " << format_weight(opt.ln_converge_delta) << " after "
          << train_iter << " iterations.\n";
      break;
    }
    ln_last_ppx = ln_new_ppx;
  }
  if (ran_restarts == 0) break;
  --ran_restarts;
  random_restart(restart_rng);
  log << "\nRandom restart - " << ran_restarts << " remaining.\n";
  }
  log << "Setting weights to model with lowest per-example-perplexity ( = "
         "prod[modelprob(example)]^(-1/num_examples) = 2^(-log_2(p_model(corpus))/N) = "
      << format_base2(ln_best_ppx) << std::endl;
  ok(cml_restore_params(ctx, SLOT_BEST));  // load_best (+ use_counts_final for cascades)
  write_back();
  res.ln_best_ppx = ln_best_ppx;
  finish();
  return res;
}

}  // namespace cb
