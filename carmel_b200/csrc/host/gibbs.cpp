// gibbs.cpp -- `carmel --crp`: collapsed Gibbs sampling of derivations (host driver).
//
// Mirrors WFST::train_gibbs / carmel_gibbs (carmel/src/gibbs.cc:12-430) and gibbs_base::run /
// iteration / finalize_cumulative_counts (graehl/shared/gibbs.hpp:626-644,803-877): CRP parameters per
// normalisation group with pseudo-counts alpha*p0*N, one sweep = every block (training example) resampled,
// time-averaged counts after burn-in become the trained weights.  Sampling itself (backward filter,
// forward sample, count updates) runs on the GPU through cml_gibbs_*; the cache-model probability of a
// sweep (gibbs.hpp:712-742) is a strictly sequential product over the corpus and is computed here from
// the downloaded sample paths.
#include <algorithm>
#include <fstream>
#include <iostream>
#include <stdexcept>

#include "carmel_host.hpp"

namespace cb {

namespace {

// CRP parameters of one transducer (gibbs.cc:114-186); parameter ids = arc-table order
void add_gibbs_params(Wfst const& w, NormalizeMethod const& nm, bool uniform_p0, bool dirichlet_p0, uint32_t& next_norm,
                      std::vector<uint32_t>& norm, std::vector<double>& prior) {
  const double alpha = std::exp(nm.ln_add_count);
  for (auto const& st : w.states) {
    const size_t base = norm.size();
    for (Arc const& a : st) {  // default: fixed probability (locked arc or NONE-normalised transducer)
      norm.push_back(kNoGroup);
      prior.push_back(std::exp(a.ln_w));
    }
    if (nm.group == NONE) continue;
    // groups of this state: JOINT = all arcs, CONDITIONAL = arcs sharing an input symbol
    std::vector<std::pair<uint32_t, std::vector<size_t>>> groups;
    for (size_t k = 0; k < st.size(); ++k) {
      const uint32_t key = nm.group == JOINT ? 0u : st[k].in;
      auto it = std::find_if(groups.begin(), groups.end(), [&](auto const& g) { return g.first == key; });
      if (it == groups.end()) {
        groups.push_back({key, {}});
        it = groups.end() - 1;
      }
      it->second.push_back(k);
    }
    for (auto const& g : groups) {
      double ln_sum = kNegInf;
      uint32_t n_unlocked = 0;
      for (size_t k : g.second)
        if (st[k].group != kLocked) {
          ln_sum = ln_add(ln_sum, st[k].ln_w);
          ++n_unlocked;
        }
      if (dirichlet_p0) ln_sum = 0;
      const uint32_t id = next_norm++;
      for (size_t k : g.second)
        if (st[k].group != kLocked) {
          norm[base + k] = id;
          prior[base + k] = uniform_p0 ? alpha : alpha * std::exp(st[k].ln_w - ln_sum) * n_unlocked;
        }
    }
  }
}

}  // namespace

// everything up to the first sweep: lattices resident, CRP parameters defined, counts = priors
void TrainJob::prepare_gibbs() {
  if (gibbs_prepared) return;
  GibbsOpts& g = gopt;
  for (auto& m : methods)  // gibbs.cc:390-397
    if (!(m.ln_add_count > kNegInf)) {
      std::cerr << "Gibbs sampling requires positive --priors for base model / initial sample.  Setting to 0.01\n";
      m.ln_add_count = std::log(1e-2);
    }
  if (g.final_counts) g.burnin = g.iter;  // gibbs_opts.hpp:253-267 validate
  if (g.burnin > g.iter) g.burnin = g.iter;
  opt.precision = 64;
  opt.space = CML_SPACE_LOG;  // layered-CSR lattices keep the reference's per-state arc order
  opt.no_ell = true;
  prepare();

  std::vector<uint32_t>& norm = g_norm;
  std::vector<double>& prior = g_prior;
  uint32_t& n_norms = g_n_norms;
  norm.clear();
  prior.clear();
  n_norms = 0;
  for (size_t i = 0; i < members.size(); ++i)
    add_gibbs_params(*members[i], i < methods.size() ? methods[i] : NormalizeMethod(), g.uniform_p0, g.dirichlet_p0, n_norms,
                     norm, prior);
  if (norm.size() != M.n_params) throw std::runtime_error("internal: gibbs parameter count mismatch");
  cml_gibbs_model gm{};
  gm.n_params = M.n_params;
  gm.param_norm = norm.data();
  gm.param_prior = prior.data();
  gm.n_norms = n_norms;
  ok(cml_gibbs_init(ctx, &gm));
  // sample slot bases (= prefix sums of lattice level counts) are recomputed from the layout
  g_base.assign(res.examples + 1, 0);
  for (uint64_t e = 0; e < res.examples; ++e) {
    uint32_t nl = 0;
    ok(cml_get_example_layout(ctx, e, &nl, nullptr, nullptr));
    g_base[e + 1] = g_base[e] + nl;
  }
  if (g.batched && opt.dense >= 0) attach_dense_sampler();
  gibbs_prepared = true;
}

// Batched sweeps on position-synchronous lattices (every arc consumes one symbol of one tape, the other tape of every
// pair empty) can use the dense-state sampler: hand the library the arc triples and the strings of the resident
// examples.  Anything else (or CML_ERR_NOT_DENSE) keeps the lattice sampler.
void TrainJob::attach_dense_sampler() {
  const uint32_t S = x->num_states();
  if (S > 32 || corpus.examples.size() != res.examples) return;
  bool in_only = true, out_only = true;
  for (auto const& st : x->states)
    for (Arc const& a : st) {
      in_only = in_only && a.in != kEps && a.out == kEps;
      out_only = out_only && a.out != kEps && a.in == kEps;
    }
  for (Example const& ex : corpus.examples) {
    in_only = in_only && ex.out.empty();
    out_only = out_only && ex.in.empty();
  }
  if (!in_only && !out_only) return;
  const int tape = out_only ? 1 : 0;
  std::unordered_map<uint32_t, uint32_t> sym_id;
  std::vector<uint32_t> a_src, a_dst, a_sym;
  for (uint32_t s = 0; s < S; ++s)
    for (Arc const& a : x->states[s]) {
      const uint32_t sy = tape ? a.out : a.in;
      auto it = sym_id.find(sy);
      if (it == sym_id.end()) it = sym_id.emplace(sy, (uint32_t)sym_id.size()).first;
      a_src.push_back(s);
      a_dst.push_back(a.dest);
      a_sym.push_back(it->second);
    }
  std::vector<uint64_t> seq_off{0};
  std::vector<uint32_t> syms;
  for (Example const& ex : corpus.examples) {
    for (uint32_t sy : (tape ? ex.out : ex.in)) {
      auto it = sym_id.find(sy);
      if (it == sym_id.end()) return;  // (cannot happen: the example has a derivation)
      syms.push_back(it->second);
    }
    seq_off.push_back(syms.size());
  }
  cml_dense_view v{};
  v.n_states = S;
  v.n_symbols = (uint32_t)sym_id.size();
  v.start = 0;
  v.final_state = x->final_state;
  v.arc_src = a_src.data();
  v.arc_dst = a_dst.data();
  v.arc_sym = a_sym.data();
  cml_sequence_batch b{};
  b.n_seq = corpus.examples.size();
  b.seq_off = seq_off.data();
  b.sym = syms.data();
  b.seq_weight = nullptr;
  const int rc = cml_gibbs_attach_dense(ctx, &v, &b);
  if (rc == CML_ERR_NOT_DENSE) {
    if (!flags[(unsigned)'q']) std::cerr << "dense-state sampler not applicable (" << cml_last_error(ctx) << "); sampling on lattices\n";
    return;
  }
  ok(rc);
  res.dense = true;
  if (!flags[(unsigned)'q']) std::cerr << "dense-state sampler: " << S << " states x " << v.n_symbols << " symbols\n";
}

TrainResult const& TrainJob::run_gibbs(std::ostream& log) {
  // Sharded sampling (SURVEY 8(e)): only batched sweeps shard -- every rank samples its blocks against the counts the
  // previous sweep left, the ranks' count deltas are summed by one all-reduce per sweep (cml_gibbs_sweep).  The exact
  // sampler visits the blocks one after another, so it stays on one GPU; results of a sharded run are reported as
  // perplexity agreement, not sample identity.
  const bool sharded = opt.shard_count > 1;
  if (sharded && (!gopt.batched || gopt.expectation || gopt.sample_prob))
    throw std::runtime_error("--shard / --gpus with --crp needs --crp-batched (and neither --expectation nor --sample-prob): "
                             "the exact sampler is sequential over the corpus");
  prepare_gibbs();
  if (sharded && !have_comm_id)
    throw std::runtime_error("sharded --crp-batched needs the library's communicator (cml_job_set_comm / --gpus)");
  GibbsOpts& g = gopt;
  std::vector<uint32_t> const& norm = g_norm;
  std::vector<double> const& prior = g_prior;
  const uint32_t n_norms = g_n_norms;
  std::vector<uint64_t> const& base = g_base;
  const uint64_t cap = cml_gibbs_sample_capacity(ctx);
  std::vector<uint32_t> path_len(res.examples), path_arcs(cap);
  auto time_of = [&](uint32_t it) { return it > g.burnin ? (double)it - (double)g.burnin : 0.; };
  std::vector<double> ccount(M.n_params), csum(std::max<uint32_t>(1, n_norms));
  const double n_sym = corpus.n_output;
  // --sample-prob: host mirror of the sampler's counts (prior + the current sample of every block) and the previous
  // sweep's sample, to evaluate each new path against the counts without its own block
  std::vector<double> sp_count, sp_sum;
  std::vector<uint32_t> prev_len, prev_arcs;
  if (g.sample_prob) {
    sp_count.assign(prior.begin(), prior.end());
    sp_sum.assign(std::max<uint32_t>(1, n_norms), 0.);
    for (uint32_t p = 0; p < M.n_params; ++p)
      if (norm[p] != kNoGroup) sp_sum[norm[p]] += prior[p];
    prev_len.assign(res.examples, 0);
    prev_arcs.assign(cap, 0);
  }
  auto for_params = [&](uint32_t a, auto&& f) {
    const uint32_t k0 = using_cascade ? M.chain_off[a] : a, k1 = using_cascade ? M.chain_off[a + 1] : a + 1;
    for (uint32_t c = k0; c < k1; ++c) f(using_cascade ? M.chain_param[c] : c);
  };
  for (uint32_t it = 0; it <= g.iter; ++it) {
    double temperature = g.high_temp;
    if (g.iter > 0 && g.high_temp != g.low_temp)
      temperature = g.high_temp + (g.low_temp - g.high_temp) * std::min(1.0, (double)it / g.iter);
    cml_gibbs_sweep_opts so{};
    so.mode = g.expectation ? CML_GIBBS_EXPECTATION : g.batched ? CML_GIBBS_BATCHED : CML_GIBBS_SEQUENTIAL;
    so.power = temperature > 0 ? 1. / temperature : 1.;
    so.seed = g.seed + (sharded ? 0x9E3779B97F4A7C15ull * (uint64_t)(opt.shard_rank + 1) : 0ull);  // (draws are keyed by local block number)
    so.sweep = it;
    so.init_from_params = 0;
    so.accumulate_dt = it == g.iter ? 1. : time_of(it + 1) - time_of(it);
    ok(cml_gibbs_sweep(ctx, &so));
    if (g.expectation) {  // record_iteration with probname "sum-all-derivations" (gibbs.hpp:930-945)
      std::vector<double> blk(res.examples);
      ok(cml_gibbs_get_block_logprob(ctx, blk.data(), blk.size()));
      double ln_p = 0;
      for (double v : blk) ln_p += v;
      res.history.push_back({it, ln_p, ln_p, 0});
      if (!opt.quiet) {
        log << "Gibbs i=" << it << " sum-all-derivations prob=" << format_base2(ln_p);
        if (n_sym) log << " per-point-ppx(N=" << n_sym << ")=" << format_base2(-ln_p / n_sym);
        log << " per-block-ppx(N=" << res.examples << ")=" << format_base2(-ln_p / (double)res.examples) << "\n";
      }
      continue;
    }
    ok(cml_gibbs_get_samples(ctx, path_len.data(), path_arcs.data(), cap));
    // cache-model probability of the sweep's sample (gibbs.hpp:137-140,700-742)
    std::fill(csum.begin(), csum.end(), 0.);
    for (uint32_t p = 0; p < M.n_params; ++p) {
      ccount[p] = prior[p];
      if (norm[p] != kNoGroup) csum[norm[p]] += prior[p];
    }
    double ln_p = 0;
    if (g.sample_prob) {
      // gibbs.hpp:851-871 in block order: remove the block's old sample, add the new one, score it
      for (uint64_t e = 0; e < res.examples; ++e) {
        const double wt = corpus.examples[e].weight;
        for (uint32_t k = 0; k < prev_len[e]; ++k)
          for_params(prev_arcs[base[e] + k], [&](uint32_t p) {
            if (norm[p] != kNoGroup) {
              sp_count[p] -= wt;
              sp_sum[norm[p]] -= wt;
            }
          });
        for (uint32_t k = 0; k < path_len[e]; ++k)
          for_params(path_arcs[base[e] + k], [&](uint32_t p) {
            if (norm[p] != kNoGroup) {
              sp_count[p] += wt;
              sp_sum[norm[p]] += wt;
            }
          });
        // scored with the new sample's counts back in (gibbs.hpp:866: "do it after to get overestimate"): the only
        // reading under which the golden log is possible (its i=0 sample, 2^-207028, beats the EM optimum 2^-212071)
        for (uint32_t k = 0; k < path_len[e]; ++k)
          for_params(path_arcs[base[e] + k], [&](uint32_t p) {
            ln_p += norm[p] != kNoGroup ? std::log(sp_count[p] / sp_sum[norm[p]]) : std::log(prior[p]);
          });
      }
      prev_len = path_len;
      prev_arcs = path_arcs;
    } else
    for (uint64_t e = 0; e < res.examples; ++e)
      for (uint32_t k = 0; k < path_len[e]; ++k) {
        const uint32_t a = path_arcs[base[e] + k];
        const uint32_t k0 = using_cascade ? M.chain_off[a] : a, k1 = using_cascade ? M.chain_off[a + 1] : a + 1;
        for (uint32_t c = k0; c < k1; ++c) {
          const uint32_t p = using_cascade ? M.chain_param[c] : c;
          ln_p += norm[p] != kNoGroup ? std::log(ccount[p]++ / csum[norm[p]]++) : std::log(prior[p]);
        }
      }
    if (sharded) ok(cml_allreduce_host(ctx, &ln_p, 1));  // (every rank scores its blocks with a cache of its own)
    const double n_blocks = sharded ? (double)corpus.n_pairs : (double)res.examples;
    res.history.push_back({it, ln_p, ln_p, 0});
    if (!opt.quiet) {
      log << "Gibbs i=" << it << (g.sample_prob ? " sample prob=" : " cache-model prob=") << format_base2(ln_p);
      if (n_sym) log << " per-point-ppx(N=" << n_sym << ")=" << format_base2(-ln_p / n_sym);
      log << " per-block-ppx(N=" << n_blocks << ")=" << format_base2(-ln_p / n_blocks) << "\n";
    }
  }
  if (!gopt.dump_samples_file.empty()) {
    std::ofstream o(gopt.dump_samples_file);
    for (uint64_t e = 0; e < res.examples; ++e) {
      for (uint32_t k = 0; k < path_len[e]; ++k) o << (k ? " " : "") << path_arcs[base[e] + k];
      o << "\n";
    }
  }
  // finalize_cumulative_counts + probs_to_cascade (gibbs.hpp:626-644, gibbs.cc:66-76)
  std::vector<double> count(M.n_params), cum(M.n_params), normsum(std::max<uint32_t>(1, n_norms), 0.);
  ok(cml_gibbs_get_state(ctx, count.data(), cum.data(), nullptr));
  const double tmax1 = ((double)g.iter - (double)g.burnin) + 1;
  std::vector<double> v(M.n_params);
  for (uint32_t p = 0; p < M.n_params; ++p) {
    if (g.final_counts && !g.exclude_prior)
      v[p] = count[p];
    else if (g.final_counts)
      v[p] = count[p] - prior[p];
    else
      v[p] = cum[p] - (g.exclude_prior ? prior[p] * tmax1 : 0.);
    if (norm[p] != kNoGroup) normsum[norm[p]] += v[p];
  }
  size_t p = 0;
  for (Wfst* m : members)
    for (auto& st : m->states)
      for (Arc& a : st) {
        const double fp = norm[p] != kNoGroup ? (v[p] > 0 ? v[p] / normsum[norm[p]] : 0.) : prior[p];
        a.ln_w = fp > 0 ? std::log(fp) : kNegInf;
        a.group = kNoGroup;  // cascade.clear_groups() (gibbs.cc:428)
        ++p;
      }
  finish();
  return res;
}

}  // namespace cb
