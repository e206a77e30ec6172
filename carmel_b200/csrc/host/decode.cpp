// decode.cpp -- `carmel --viterbi` / `--decode` (host driver): the best, k best or sampled derivations and the total
// weights of the training pairs, or of new strings with the other tape free, under the model as given.  The decoders
// themselves run on the GPU (cml_viterbi, cml_kbest, cml_sample).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <fstream>
#include <functional>
#include <memory>
#include <stdexcept>

#include "carmel_host.hpp"

namespace cb {

namespace {

// labels of every parameter's member arc (parameters are numbered member by member, state by state, arc by arc)
std::vector<std::string> param_labels(std::vector<Wfst*> const& members) {
  std::vector<std::string> plabel;
  for (Wfst* m : members)
    for (auto& st : m->states)
      for (Arc& a : st) plabel.push_back(m->alph[0]->names[a.in] + ":" + m->alph[1]->names[a.out]);
  return plabel;
}

// one decode line without its newline: ln weight, number of arcs, arc-table ids, "|", then per arc the (input:output)
// labels of the cascade members' arcs it stands for
void write_derivation(std::ostream& o, double lnw, const uint32_t* arcs, uint32_t len, std::vector<std::string> const& plabel,
                      bool using_cascade, ModelArrays const& M) {
  o << lnw << " " << len;
  for (uint32_t k = 0; k < len; ++k) o << " " << arcs[k];
  o << " |";
  for (uint32_t k = 0; k < len; ++k) {
    const uint32_t a = arcs[k];
    const uint32_t k0 = using_cascade ? M.chain_off[a] : a, k1 = using_cascade ? M.chain_off[a + 1] : a + 1;
    o << " (";
    for (uint32_t c = k0; c < k1; ++c) o << (c > k0 ? " " : "") << plabel[using_cascade ? M.chain_param[c] : c];
    o << ")";
  }
}

// --viterbi / --decode: one GPU, fp64 log space, layered-CSR lattices (they keep the reference's per-state arc order)
void force_decode_options(TrainOpts& opt, const char* what) {
  opt.precision = 64;
  opt.space = CML_SPACE_LOG;
  opt.no_ell = true;
  opt.dense = -1;
  if (opt.shard_count > 1) throw std::runtime_error(std::string(what) + " decodes on one GPU");
}

// n derivations of every resident lattice in cml_kbest's layout, ln of every lattice's total weight (--sample / --sum),
// the host time of the decoder call and its kernel time
struct Decoded {
  uint64_t n_ex = 0, n = 0;
  std::vector<uint32_t> len, arcs;
  std::vector<uint64_t> base;
  std::vector<double> lnw, total;
  double seconds = 0;
  float kernel_ms = 0;
};

// --sample=n draws n derivations per lattice (cml_sample, which also gives the totals); otherwise the -k n best
// (cml_viterbi for n = 1, cml_kbest otherwise), after a totals-only cml_sample call (n = 0) when --sum asks for them.
// The uniforms of lattice i are keyed by key[i].  `seconds` covers the decoder call, not the totals-only call.
Decoded decode_resident(TrainJob const& job, std::vector<uint64_t> const& key) {
  TrainOpts const& opt = job.opt;
  cml_ctx* ctx = job.ctx;
  Decoded d;
  d.n = opt.sample ? opt.sample : opt.kbest;
  uint64_t n_levels = 0;
  job.ok(cml_trellis_totals(ctx, &d.n_ex, nullptr, nullptr, &n_levels));
  const uint64_t m = d.n_ex * d.n;
  d.len.assign(m, 0);
  d.arcs.assign(std::max<uint64_t>(1, n_levels * d.n), 0);
  d.base.assign(m + 1, 0);
  d.lnw.assign(m, 0.);
  d.total.assign(d.n_ex, 0.);
  if (d.n_ex && !opt.sample && !opt.sum_file.empty())
    job.ok(cml_sample(ctx, 0, opt.seed, key.data(), nullptr, nullptr, nullptr, 0, nullptr, d.total.data()));
  const auto t0 = std::chrono::steady_clock::now();
  if (d.n_ex && opt.sample)
    job.ok(cml_sample(ctx, (uint32_t)d.n, opt.seed, key.data(), d.len.data(), d.base.data(), d.arcs.data(), d.arcs.size(),
                      d.lnw.data(), d.total.data()));
  else if (d.n_ex && d.n == 1)
    job.ok(cml_viterbi(ctx, d.len.data(), d.base.data(), d.arcs.data(), d.arcs.size(), d.lnw.data()));
  else if (d.n_ex && d.n > 1)
    job.ok(cml_kbest(ctx, (uint32_t)d.n, d.len.data(), d.base.data(), d.arcs.data(), d.arcs.size(), d.lnw.data()));
  d.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  job.ok(opt.sample ? cml_sample_stats(ctx, nullptr, nullptr, &d.kernel_ms) : cml_kbest_stats(ctx, nullptr, nullptr, &d.kernel_ms));
  return d;
}

// Writes d's derivation lines to path, d.n per lattice: per corpus line through lat_of when given (a line without a
// lattice, lat_of < 0, gets d.n empty derivations, "-inf 0 |"), else per resident lattice.  suffix, when given, ends
// every line.  Returns the sum of the rank-0 weights and the number of derivations found.
std::pair<double, uint64_t> write_derivations(TrainJob const& job, std::string const& path, Decoded const& d,
                                              std::vector<int64_t> const* lat_of,
                                              std::function<void(std::ostream&, const uint32_t*, uint32_t)> const& suffix) {
  const std::vector<std::string> plabel = param_labels(job.members);
  std::ofstream o(path);
  if (!o) throw std::runtime_error("cannot write " + path);
  o.precision(17);
  double total = 0;
  uint64_t found = 0;
  auto lines = [&](int64_t i) {
    for (uint64_t r = 0; r < d.n; ++r) {
      const uint64_t j = i < 0 ? 0 : (uint64_t)i * d.n + r;
      const uint32_t* p = i < 0 ? nullptr : d.arcs.data() + d.base[j];
      const uint32_t len = i < 0 ? 0 : d.len[j];
      write_derivation(o, i < 0 ? kNegInf : d.lnw[j], p, len, plabel, job.using_cascade, job.M);
      if (suffix) suffix(o, p, len);
      o << "\n";
      if (i < 0) continue;
      if (r == 0) total += d.lnw[j];
      if (d.lnw[j] > kNegInf) ++found;
    }
  };
  if (lat_of)
    for (int64_t i : *lat_of) lines(i);
  else
    for (uint64_t i = 0; i < d.n_ex; ++i) lines((int64_t)i);
  return {total, found};
}

// --sum=FILE: one line per example (lat_of[e] < 0: no lattice), ln of its total weight as %.17g, or -inf; the log line
// gives the product of the totals of the examples with a derivation
void write_sums(std::ostream& log, bool quiet, std::string const& path, std::vector<int64_t> const& lat_of,
                std::vector<double> const& total, const char* what) {
  std::ofstream o(path);
  if (!o) throw std::runtime_error("cannot write " + path);
  double prod = 0;
  uint64_t none = 0;
  char buf[64];
  for (int64_t i : lat_of) {
    const double t = i < 0 ? kNegInf : total[i];
    std::snprintf(buf, sizeof buf, "%.17g", t);
    o << buf << "\n";
    if (t > kNegInf)
      prod += t;
    else
      ++none;
  }
  if (!quiet)
    log << "Sum: total weights of " << lat_of.size() << " " << what << ", " << none
        << " without a derivation; product of the others=" << format_base2(prod) << "\n";
}

}  // namespace

// Decode: the -k n best derivations per training pair (cml_viterbi for n = 1, cml_kbest otherwise), n lines per resident
// lattice (an example without a derivation gets none) in corpus order, best first; ranks past the number of derivations
// read "-inf 0 |".  With --sample=n, n drawn derivations per example instead, examples without a derivation included.
// The weights are the model's as read, after the same normalisation a training run starts from (train.cc:509); no
// training happens.
void TrainJob::run_viterbi(std::ostream& log, std::string const& path) {
  force_decode_options(opt, "--viterbi");
  prepare();
  std::vector<int64_t> lat_of(corpus_size, -1);
  for (size_t i = 0; i < kept_example.size(); ++i) lat_of[kept_example[i]] = (int64_t)i;
  // --sample / --sum: keyed by the example's index in the corpus
  const Decoded d = decode_resident(*this, std::vector<uint64_t>(kept_example.begin(), kept_example.end()));
  if (!opt.sum_file.empty()) write_sums(log, opt.quiet, opt.sum_file, lat_of, d.total, "examples");
  if (opt.sample) {
    write_derivations(*this, path, d, &lat_of, nullptr);
    if (!opt.quiet)
      log << "Sample: " << d.n << " derivations drawn per example (seed " << opt.seed << ") from " << kept_example.size()
          << " of " << corpus_size << " examples (kernels " << d.kernel_ms << " ms)\n";
    return;
  }
  const std::pair<double, uint64_t> tf = write_derivations(*this, path, d, nullptr, nullptr);
  if (!opt.quiet) {
    log << "Viterbi: best derivations of " << d.n_ex << " examples, product of their weights=" << format_base2(tf.first)
        << "\n";
    if (d.n > 1) log << "Viterbi: " << d.n << "-best lists, " << tf.second << " derivations found\n";
  }
}

// Decode new strings: the lattice of every string on the given tape x the composed machine, the other tape free, built on
// the GPU (cml_build_free_trellises), then the same decoders and line format as run_viterbi.  The model is set up as for
// --viterbi (prepare_model: the weights as read, normalised as a training run starts from them).
void TrainJob::run_decode(std::ostream& log, std::string const& path) {
  force_decode_options(opt, "--decode");
  prepare_model();
  const int g = opt.given_tape;
  std::vector<uint32_t> soff, ain, aout, adest;
  x->arc_offsets(soff);
  for (auto const& st : x->states)
    for (Arc const& a : st) {
      ain.push_back(a.in);
      aout.push_back(a.out);
      adest.push_back(a.dest);
    }
  const size_t n = corpus.examples.size();
  std::vector<uint64_t> off(n + 1, 0);
  std::vector<uint32_t> sym;
  for (size_t e = 0; e < n; ++e) {
    auto const& v = g ? corpus.examples[e].out : corpus.examples[e].in;
    sym.insert(sym.end(), v.begin(), v.end());
    off[e + 1] = sym.size();
  }
  cml_wfst_view xv{};
  xv.n_states = x->num_states();
  xv.final_state = x->final_state;
  xv.n_arcs = ain.size();
  xv.state_arc_off = soff.data();
  xv.arc_in = ain.data();
  xv.arc_out = aout.data();
  xv.arc_dest = adest.data();
  cml_string_batch sb{n, off.data(), sym.data()};
  cml_built_trellises* b = nullptr;
  ok(cml_build_free_trellises(ctx, &xv, &sb, g, &b));
  std::unique_ptr<cml_built_trellises, void (*)(cml_built_trellises*)> hold(b, cml_free_built_trellises);
  const auto t0 = std::chrono::steady_clock::now();
  if (b->batch.n_ex) ok(cml_add_trellises(ctx, &b->batch));
  const double add_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  uint64_t n_states = 0, n_arcs = 0;
  ok(cml_trellis_totals(ctx, nullptr, &n_states, &n_arcs, nullptr));
  std::vector<int64_t> lat_of(n, -1);
  for (uint64_t i = 0; i < b->batch.n_ex; ++i) lat_of[b->kept_example[i]] = (int64_t)i;
  // --sample / --sum: keyed by the string's line, so a string's draws do not depend on the other lines
  const Decoded d = decode_resident(*this, std::vector<uint64_t>(b->kept_example, b->kept_example + b->batch.n_ex));
  if (!opt.sum_file.empty()) write_sums(log, opt.quiet || flags[(unsigned)'q'], opt.sum_file, lat_of, d.total, "strings");
  const std::vector<uint32_t>& free_label = g ? ain : aout;
  const std::vector<std::string>& free_name = x->alph[1 - g]->names;
  const std::pair<double, uint64_t> tf =
      write_derivations(*this, path, d, &lat_of, [&](std::ostream& o, const uint32_t* p, uint32_t len) {
        o << " ||";
        for (uint32_t k = 0; k < len; ++k)
          if (free_label[p[k]] != kEps) o << " " << free_name[free_label[p[k]]];
      });
  if (!opt.quiet && !flags[(unsigned)'q']) {
    log << "Decode: " << n << " strings on the " << (g ? "output" : "input") << " tape, " << b->n_dropped
        << " without a derivation";
    if (opt.sample)
      log << "; " << d.n << " derivations drawn per string (seed " << opt.seed << ")\n";
    else
      log << "; product of the best weights of the others=" << format_base2(tf.first) << "\n";
    if (d.n > 1 && !opt.sample) log << "Decode: " << d.n << "-best lists, " << tf.second << " derivations found\n";
    log << "Decode: lattices built on the GPU in " << b->seconds << " s (k_build_free " << b->kernel_ms << " ms, "
        << b->chunks << " chunk(s); " << n_states << " states, " << n_arcs << " arcs), cml_add_trellises " << add_s
        << " s, decode " << d.seconds << " s (kernels " << d.kernel_ms << " ms)\n";
  }
}

}  // namespace cb
