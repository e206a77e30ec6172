// forest.cpp -- forest-em on the GPU: readers/writers, option parsing and the EM driver (host side).
// See forest_host.hpp for the reference file:line each part mirrors.
#include "forest_host.hpp"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>
#include <unordered_map>

#include "carmel_host.hpp"

namespace cb {

namespace {

const double kNegInfD = -std::numeric_limits<double>::infinity();

inline const char* skip_ws(const char* p, const char* e) {
  while (p < e && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r' || *p == '\f' || *p == '\v')) ++p;
  return p;
}
inline bool read_uint(const char*& p, const char* e, uint64_t& v) {
  if (p >= e || *p < '0' || *p > '9') return false;
  v = 0;
  while (p < e && *p >= '0' && *p <= '9') v = v * 10 + (uint64_t)(*p++ - '0');
  return true;
}
std::string slurp(std::string const& path) {
  std::ifstream in(path, std::ios::binary);
  if (!in) throw std::runtime_error("can't open " + path);
  std::ostringstream o;
  o << in.rdbuf();
  return o.str();
}
// weight.h:463-490 with forest-em's ALWAYS_LOG / EXP base defaults (forest-em-params.cpp:75-84)
std::string fmt_forest_weight(double ln, bool dbl, bool human) {
  if (!(ln > kNegInfD)) return "0";
  std::ostringstream o;
  o.precision(dbl ? 15 : 7);
  if (human) {
    if (dbl)
      o << std::exp(ln);
    else
      o << (float)std::exp(ln);
  } else {
    o << "e^";
    if (dbl)
      o << ln;
    else
      o << (float)ln;
  }
  return o.str();
}

}  // namespace

// ---- forests (forest.hpp:135-242) --------------------------------------------------------------------
void ForestSet::read(const char* p, const char* end) {
  std::vector<uint64_t> open_parens;  // absolute node indices whose `next` the matching ')' sets
  std::unordered_map<uint64_t, uint32_t> backrefs;
  for (;;) {
    p = skip_ws(p, end);
    if (p >= end) return;
    const uint64_t base = next.size();
    auto fail = [&](std::string const& what) {
      throw std::runtime_error("forest #" + std::to_string(size() + 1) + ": " + what);
    };
    open_parens.clear();
    backrefs.clear();
    bool follows_paren = false;
    uint64_t n_done = 0;  // nodes completed or open (the reference's `stop - nodes`)
    auto at_stop = [&]() {
      if (next.size() <= base + n_done) {
        next.resize(base + n_done + 1, 0);
        label.resize(base + n_done + 1, 0);
        backref.resize(base + n_done + 1, 0);
      }
      return base + n_done;
    };
    while (n_done == 0 || !open_parens.empty()) {
      p = skip_ws(p, end);
      if (p >= end) fail("unexpected end of input");
      const char c = *p++;
      if (c == '#') {
        if (follows_paren) fail("Bad # following paren in Forest");
        uint64_t id;
        if (!read_uint(p, end, id)) fail("expected a back reference id after #");
        if (p >= end) fail("unexpected end of input after #id");
        if (*p == '(') {
          backrefs[id] = (uint32_t)n_done;
        } else {
          auto it = backrefs.find(id);
          if (it == backrefs.end()) fail("back reference to undefined #" + std::to_string(id));
          const uint64_t s = at_stop();
          label[s] = it->second;
          backref[s] = 1;
          next[s] = (uint32_t)(n_done + 1);
          ++n_done;
        }
      } else if (c == '(') {
        follows_paren = true;
        open_parens.push_back(at_stop());
      } else if (c >= '1' && c <= '9') {
        --p;
        uint64_t rule;
        read_uint(p, end, rule);
        if (rule >= 0x7fffffffull) fail("rule id too large");
        max_ruleid = std::max(max_ruleid, rule);
        const uint64_t s = at_stop();
        label[s] = (uint32_t)rule;
        backref[s] = 0;
        if (!follows_paren) next[s] = (uint32_t)(n_done + 1);
        follows_paren = false;
        ++n_done;
      } else if (c == 'O') {
        if (p >= end || *p != 'R') fail("expected OR");
        ++p;
        if (!follows_paren) fail("OR not following paren in Forest");
        follows_paren = false;
        const uint64_t s = at_stop();
        label[s] = 0;
        backref[s] = 0;
        ++n_done;
      } else if (c == ')') {
        if (open_parens.empty()) fail("unbalanced )");
        next[open_parens.back()] = (uint32_t)n_done;
        open_parens.pop_back();
      } else
        fail(std::string("unexpected char ") + c);
    }
    next.resize(base + n_done);
    label.resize(base + n_done);
    backref.resize(base + n_done);
    node_off.push_back(next.size());
    max_nodes = std::max(max_nodes, n_done);
  }
}

// forest.hpp:245-320 (back reference ids renumbered in order of first reference)
void ForestSet::print(std::ostream& o, uint64_t f) const {
  const uint64_t b = node_off[f];
  const uint32_t n = (uint32_t)(node_off[f + 1] - b);
  std::vector<uint32_t> ids(n, 0);
  uint32_t lastid = 0;
  for (uint32_t p = 0; p < n; ++p)
    if (backref[b + p] && !ids[label[b + p]]) ids[label[b + p]] = ++lastid;
  std::vector<uint32_t> ends{n};
  for (uint32_t p = 0; p < n; ++p) {
    while (p == ends.back() && ends.size() > 1) {
      o << ')';
      ends.pop_back();
    }
    if (p) o << ' ';
    if (ids[p]) o << '#' << ids[p];
    if (backref[b + p]) {
      o << '#' << ids[label[b + p]];
    } else if (next[b + p] == p + 1) {
      if (ids[p]) o << '(';
      o << label[b + p];
      if (ids[p]) o << ')';
    } else {
      o << '(';
      ends.push_back(next[b + p]);
      if (label[b + p])
        o << label[b + p];
      else
        o << "OR";
    }
  }
  while (ends.size() > 1) {
    o << ')';
    ends.pop_back();
  }
}

// ---- normalization groups (normalize.hpp:58-65) ---------------------------------------------------------
const char* NormGroupsHost::read(const char* p, const char* end) {
  p = skip_ws(p, end);
  if (p >= end || *p != '(') throw std::runtime_error("normalization groups: expected (");
  ++p;
  for (;;) {
    p = skip_ws(p, end);
    if (p >= end) throw std::runtime_error("normalization groups: unexpected end of input");
    if (*p == ')') return p + 1;
    if (*p != '(') throw std::runtime_error("normalization group #" + std::to_string(size() + 1) + ": expected ( or )");
    ++p;
    for (;;) {
      p = skip_ws(p, end);
      if (p >= end) throw std::runtime_error("normalization group: unexpected end of input");
      if (*p == ')') {
        ++p;
        break;
      }
      uint64_t v;
      if (!read_uint(p, end, v)) throw std::runtime_error("normalization group #" + std::to_string(size() + 1) + ": expected a parameter index");
      members.push_back(v);
      max_index = std::max(max_index, v);
    }
    off.push_back(members.size());
  }
}

// ---- job ------------------------------------------------------------------------------------------------
ForestJob::~ForestJob() {
  if (ctx) cml_forests_destroy(ctx);
}
void ForestJob::ok(int rc) const {
  if (rc != CML_OK) throw std::runtime_error(std::string("GPU library: ") + cml_forests_last_error(ctx));
}

// forest-em-params.cpp:62-112 (the reading part of perform_forest_em)
void ForestJob::load() {
  if (!opt.initparam_file.empty()) {  // forest-em.hpp:228-250 read_params
    const std::string s = slurp(opt.initparam_file);
    ln_w.assign(1, kNegInfD);
    std::istringstream in(s);
    std::string tok;
    while (in >> tok) {
      if (tok == "(" || tok == ")") continue;
      if (tok[0] == '(') tok = tok.substr(1);
      if (!tok.empty() && tok.back() == ')') tok.pop_back();
      if (tok.empty()) continue;
      double w;
      if (!parse_weight(tok.c_str(), w))
        throw std::runtime_error("Couldn't read vector of initial weights: bad weight " + tok +
                                 "\n - expected vector of weights e.g. (1 .5 0) with the first weight being for parameter #1.");
      ln_w.push_back(w);
    }
    have_init_params = true;
  }
  std::string norm_text;
  const char* after_norm = nullptr;
  if (!opt.normgroups_file.empty()) {  // forest-em.hpp:133-149
    norm_text = slurp(opt.normgroups_file);
    after_norm = groups.read(norm_text.data(), norm_text.data() + norm_text.size());
    if (have_init_params && ln_w.size() <= groups.max_index)
      throw std::runtime_error("Initial rule weights file not big enough - normalization used rule (" +
                               std::to_string(groups.max_index) + " expected)");
  }
  if (!opt.forests_file.empty()) {  // forest-em.hpp:150-168
    if (opt.forests_file == opt.normgroups_file)
      forests.read(after_norm, norm_text.data() + norm_text.size());
    else {
      const std::string s = slurp(opt.forests_file);
      forests.read(s.data(), s.data() + s.size());
    }
  }
  total_forests = forests.size();
}

// this process's block of the corpus: contiguous, balanced by node count, blocks cover the corpus without overlap
void ForestJob::compute_shard() {
  shard_begin = 0;
  shard_end = forests.size();
  if (opt.shard_count > 1) {
    const uint64_t total = forests.n_nodes();
    auto cut = [&](int r) -> uint64_t {
      if (r <= 0) return 0;
      if (r >= opt.shard_count) return forests.size();
      const uint64_t target = total / (uint64_t)opt.shard_count * (uint64_t)r;
      return (uint64_t)(std::lower_bound(forests.node_off.begin(), forests.node_off.end(), target) - forests.node_off.begin());
    };
    shard_begin = std::min(cut(opt.shard_rank), forests.size());
    shard_end = std::max(shard_begin, std::min(cut(opt.shard_rank + 1), forests.size()));
  }
}

// forest-em.hpp:335-381 prepare, :282-306 init_rule_weights
void ForestJob::prepare() {
  if (prepared) return;
  count_space = std::max(forests.max_ruleid, groups.max_index) + 1;
  rulespace = count_space;
  if (have_init_params) {
    if (rulespace > ln_w.size()) throw std::runtime_error("Initial params file wasn't large enough for forests/norms.");
    if (rulespace < ln_w.size())
      std::cerr << "Warning: more initial rule weights were provided (" << ln_w.size() << ") than used in norms or forests: " << rulespace
                << std::endl;
    rulespace = ln_w.size();
  } else if (opt.initial_1_params) {
    ln_w.assign(rulespace, 0.);
  } else {  // uniform within each group, zero elsewhere (normalize.hpp:229-246 init_uniform)
    ln_w.assign(rulespace, kNegInfD);
    for (uint64_t g = 0; g < groups.size(); ++g) {
      const uint64_t n = groups.off[g + 1] - groups.off[g];
      for (uint64_t k = groups.off[g]; k < groups.off[g + 1]; ++k) ln_w[groups.members[k]] = -std::log((double)n);
    }
  }
  if (cml_forests_create(&ctx, opt.device, opt.double_precision ? 64 : 32) != CML_OK)
    throw std::runtime_error(std::string("GPU library: ") + cml_forests_last_error(nullptr));
  if (opt.shard_count > 1 && have_comm_id) ok(cml_forests_comm_init_rank(ctx, opt.shard_count, opt.shard_rank, comm_id));
  ok(cml_forests_set_layout(ctx, opt.layout));
  ok(cml_forests_set_rules(ctx, rulespace, groups.size(), groups.off.data(), groups.members.data()));
  ok(cml_forests_set_params(ctx, ln_w.data()));
  if (have_init_params && opt.normalize_initial && groups.size()) ok(cml_forests_normalize_params(ctx));
  compute_shard();
  if (shard_end > shard_begin) {
    std::vector<uint64_t> off(forests.node_off.begin() + shard_begin, forests.node_off.begin() + shard_end + 1);
    const uint64_t o = off[0];
    for (auto& v : off) v -= o;
    cml_forest_batch b{};
    b.n_forests = shard_end - shard_begin;
    b.node_off = off.data();
    b.next = forests.next.data() + o;
    b.label = forests.label.data() + o;
    b.backref = forests.backref.data() + o;
    ok(cml_forests_add(ctx, &b));
  }
  firsttime = true;
  prepared = true;
}

// forest-em.hpp:556-572 estimate: average log prob over the non-zero forests; counts stay on the GPU
double ForestJob::estimate(bool first_time, std::ostream& log, uint64_t* n_used) {
  ok(cml_forests_estimate_launch(ctx));
  if (opt.shard_count > 1) {
    if (have_comm_id) {
      ok(cml_forests_allreduce_counts(ctx));  // NCCL, stream-ordered behind the E-step kernels
    } else if (allreduce) {
      // hook contract: the E-step has finished before the hook runs, the sum is complete when it returns
      void* p = nullptr;
      uint64_t n = 0;
      ok(cml_forests_reduce_buffer(ctx, &p, &n));
      ok(cml_forests_synchronize(ctx));
      allreduce(allreduce_user, p, n);
    }
  }
  cml_forest_estimate_result r{};
  ok(cml_forests_estimate_finish(ctx, &r));
  if (first_time && r.n_zero && opt.shard_count <= 1) {
    std::vector<double> in(shard_end - shard_begin);
    ok(cml_forests_get_inside(ctx, in.data(), in.size()));
    for (uint64_t i = 0; i < in.size(); ++i)
      if (!(in[i] > kNegInfD)) log << "Warning: 0 probability for forest #" << (i + 1) << std::endl;
  }
  last_n_zero = r.n_zero;
  const uint64_t N = r.n_forests - r.n_zero;
  log << "\nN=" << N << ' ';
  if (r.n_zero) log << '(' << r.n_zero << " 0 prob removed) ";
  if (n_used) *n_used = N;
  return r.sum_ln_p / (double)N;
}

// forest-em.hpp:626-655 maximize
void ForestJob::maximize(std::ostream& log, double& max_delta, uint64_t& max_index) {
  firsttime = false;
  cml_forest_norm_opts o{};
  o.prior_total = opt.prior_counts * (double)total_forests;
  o.add_k = opt.add_k_smoothing;
  o.zero_mode = opt.zero_zerocounts ? CML_FOREST_ZERO : CML_FOREST_UNIFORM;
  ok(cml_forests_maximize(ctx, &o, &max_delta, &max_index));
  // on_watch_iteration (forest-em.hpp:621-624) -> dump_params (:172-189)
  const bool watch = iteration <= opt.watch_period || (opt.watch_period && iteration % opt.watch_period == 0);
  if (watch && opt.checkpoint_parameters && opt.shard_rank == 0) {
    const std::string suffix = ".restart." + std::to_string(restart + 1) + ".iteration." + std::to_string(iteration + 1);
    const std::string wf = opt.checkpoint_prefix + ".params" + suffix, cf = opt.checkpoint_prefix + ".counts" + suffix;
    log << '\n';
    {
      log << "Writing trained parameters to " << wf << "\n";
      std::ofstream o(wf);
      write_params_to(o);
    }
    {
      log << "Writing trained counts to " << cf << "\n";
      std::ofstream o(cf);
      write_counts_to(o);
    }
  }
  ++iteration;
}

// forest-em.hpp:190-201 write_params / write_counts (one weight per line, 1-based rule ids)
void ForestJob::write_params_to(std::ostream& o) {
  if (ctx) ok(cml_forests_get_params(ctx, ln_w.data()));
  for (uint64_t i = 1; i < ln_w.size(); ++i) o << ' ' << fmt_forest_weight(ln_w[i], opt.double_precision, opt.human_probs) << "\n";
  o << std::endl;
}
void ForestJob::write_counts_to(std::ostream& o) {
  std::vector<double> c(rulespace, 0.);
  if (ctx && (!history.empty() || iteration)) ok(cml_forests_get_counts(ctx, c.data(), c.size()));
  const double prior = (history.empty() && !iteration) ? 0. : opt.prior_counts * (double)total_forests;
  for (uint64_t i = 1; i < count_space; ++i) {
    const double v = c[i] + prior;
    o << ' ' << fmt_forest_weight(v > 0 ? std::log(v) : kNegInfD, opt.double_precision, opt.human_probs) << "\n";
  }
  o << std::endl;
}

namespace {
void print_alp(std::ostream& logs, double N, double alp) {  // em.hpp:101-105, weight.h:331-337
  const double ln_prob = alp * N;
  logs << "probability=" << format_base2(ln_prob);
  if (N > 0) logs << " per-example-perplexity(N=" << N << ")=" << format_base2(-ln_prob / N);
}
std::string fmt_delta(double d, uint64_t idx) {  // em.hpp:60-67
  std::ostringstream o;
  if (d > 0)
    o << "delta_weight[" << idx << "]=" << d;
  else
    o << "unchanged";
  return o.str();
}
}  // namespace

// forests::randomize (forest-em.hpp:393-399) = NormalizeGroups::init_random (normalize.hpp:212-238): every member of
// a normalisation group gets a uniform draw on (0,1], divided by the group's sum; rules in no group keep their weight
void ForestJob::randomize(std::mt19937_64& rng) {
  ok(cml_forests_get_params(ctx, ln_w.data()));
  std::uniform_real_distribution<double> u01(0., 1.);
  for (uint64_t g = 0; g < groups.size(); ++g) {
    double sum = 0;
    for (uint64_t k = groups.off[g]; k < groups.off[g + 1]; ++k) {
      const double v = 1. - u01(rng);
      ln_w[groups.members[k]] = v;
      sum += v;
    }
    for (uint64_t k = groups.off[g]; k < groups.off[g + 1]; ++k) ln_w[groups.members[k]] = std::log(ln_w[groups.members[k]] / sum);
  }
  ok(cml_forests_set_params(ctx, ln_w.data()));
}

// graehl/shared/em.hpp:107-216 overrelaxed_em as forest-em calls it (growth factor 1)
double ForestJob::run(std::ostream& logs) {
  if (opt.parse_only) return 0;
  prepare();
  best_alp = -HUGE_VAL;
  if (opt.max_iter == 0) return best_alp;
  const double rel_eps = opt.converge_ratio;
  bool very_first_time = true;
  const double N = (double)total_forests;
  // random restarts (-r n): best-weights bookkeeping exists only then (forest-em.hpp:363-365,660-672)
  unsigned ran_restarts = opt.random_restarts;
  const bool save_best_enable = ran_restarts > 0;
  std::vector<double> best_w;
  std::mt19937_64 rng(opt.random_seed);
  for (;;) {
  bool first_time = true;
  unsigned train_iter = 0;
  double max_delta = 0, last_alp = -HUGE_VAL;
  uint64_t max_index = 0;
  for (;;) {
    ++train_iter;
    if (train_iter > opt.max_iter) {
      logs << "Maximum number of iterations (" << opt.max_iter
           << ") reached before convergence criteria was met - greatest param weight change was " << fmt_delta(max_delta, max_index) << "\n";
      break;
    }
    uint64_t n_used = 0;
    const double new_alp = estimate(very_first_time, logs, &n_used);
    logs << "i=" << train_iter << ": ";
    print_alp(logs, N, new_alp);
    if (new_alp > best_alp || very_first_time) {
      logs << " (new best)";
      best_alp = new_alp;
      if (save_best_enable) {  // save_best: the parameters this estimate was made with
        best_w.resize(ln_w.size());
        ok(cml_forests_get_params(ctx, best_w.data()));
      }
    }
    very_first_time = false;
    const double dpp = new_alp - last_alp;
    double last_abs = std::fabs(last_alp);
    if (last_abs < 1e-10) last_abs = 1e-10;  // LOGPROB_EPSILON
    double rel_dpp = dpp / last_abs;
    if (first_time) {
      rel_dpp = HUGE_VAL;
      logs << std::endl;
      first_time = false;
    } else
      logs << " (relative-d-avg-logprob=" << rel_dpp << "), max " << fmt_delta(max_delta, max_index) << std::endl;
    history.push_back({train_iter, new_alp, max_delta, max_index, n_used});
    if (rel_dpp < rel_eps) {
      logs << "\nConverged - relative per-example avg-logprob change less than " << rel_eps << " after " << train_iter << " iterations.\n";
      break;
    }
    maximize(logs, max_delta, max_index);
    if (max_delta <= opt.converge_delta) {
      logs << "\nConverged - all weights changed no more than " << opt.converge_delta << " after " << train_iter << " iterations.\n";
      break;
    }
    last_alp = new_alp;
  }
  if (ran_restarts == 0) break;
  --ran_restarts;
  logs << "\nRandom restart - " << ran_restarts << " remaining.\n";
  ++restart;
  iteration = 0;
  randomize(rng);
  }
  logs << "\nSetting weights to model with best ";
  print_alp(logs, N, best_alp);
  logs << std::endl;
  if (save_best_enable && !best_w.empty()) {  // restore_best
    ok(cml_forests_set_params(ctx, best_w.data()));
    logs << std::endl;
  }
  return best_alp;
}

// forest-em --crp (FForests::run_gibbs, forest-em/forest-em.hpp:711-750; gibbs_base::run / iteration,
// graehl/shared/gibbs.hpp:803-877): parameters from the normalised rule weights, one sweep per iteration on the GPU,
// the cache-model (or --sample-prob) probability of every sweep's sample on the host, final weights = time-averaged
// counts normalised per group (finalize_cumulative_counts + from_gibbs).
void ForestJob::run_gibbs(std::ostream& log) {
  prepare();
  if (opt.shard_count > 1) throw std::runtime_error("--crp samples the forests in corpus order: one GPU (no --shard / --gpus)");
  ok(cml_forests_normalize_params(ctx));  // to_gibbs -> define_gibbs(true): normalize() first
  ok(cml_forests_get_params(ctx, ln_w.data()));
  std::vector<uint32_t> norm(rulespace, 0xFFFFFFFFu);
  std::vector<double> prior(rulespace, 0.);
  for (uint64_t g = 0; g < groups.size(); ++g) {  // visit_norm_param (normalize.hpp:194-210); group ids 1.. as there
    const uint64_t n = groups.off[g + 1] - groups.off[g];
    for (uint64_t k = groups.off[g]; k < groups.off[g + 1]; ++k) {
      const uint64_t p = groups.members[k];
      norm[p] = (uint32_t)g + 1;
      prior[p] = opt.crp_uniform_p0 ? opt.crp_alpha : opt.crp_alpha * std::exp(ln_w[p]) * (double)n;
    }
  }
  for (uint64_t p = 0; p < rulespace; ++p)
    if (norm[p] == 0xFFFFFFFFu) prior[p] = std::exp(ln_w[p]);  // no group: fixed probability
  const uint32_t n_norms = (uint32_t)groups.size() + 1;
  const uint64_t nf = shard_end - shard_begin;
  std::vector<uint64_t> off(forests.node_off.begin() + shard_begin, forests.node_off.begin() + shard_end + 1);
  const uint64_t o0 = off.empty() ? 0 : off[0];
  for (auto& v : off) v -= o0;
  cml_forest_batch b{};
  b.n_forests = nf;
  b.node_off = off.data();
  b.next = forests.next.data() + o0;
  b.label = forests.label.data() + o0;
  b.backref = forests.backref.data() + o0;
  cml_forest_gibbs_model gm{norm.data(), prior.data(), n_norms};
  ok(cml_forests_gibbs_init(ctx, &b, &gm));
  const uint64_t cap = cml_forests_gibbs_sample_capacity(ctx);
  std::vector<uint32_t> len(nf), ids(cap), prev_len(nf, 0), prev_ids;
  std::vector<uint64_t> base(nf + 1);
  const unsigned Ni = opt.crp_iter;
  unsigned burnin = std::min(opt.crp_burnin, Ni);
  if (opt.crp_final_counts) burnin = Ni;  // gibbs_opts.hpp:259
  auto time_of = [&](unsigned it) { return it > burnin ? (double)it - (double)burnin : 0.; };
  const double n_sym = opt.crp_n_sym ? opt.crp_n_sym : (double)(off.empty() ? 0 : off[nf]);  // forest-em.hpp:733: n_nodes
  std::vector<double> ccount(rulespace), csum(n_norms), sp_count, sp_sum;
  if (opt.crp_sample_prob) {
    sp_count = prior;
    sp_sum.assign(n_norms, 0.);
    for (uint64_t p = 0; p < rulespace; ++p)
      if (norm[p] != 0xFFFFFFFFu) sp_sum[norm[p]] += prior[p];
    prev_ids.assign(cap, 0);
  }
  for (unsigned it = 0; it <= Ni; ++it) {
    double temperature = opt.crp_high_temp;
    if (Ni > 0 && opt.crp_high_temp != opt.crp_low_temp)
      temperature = opt.crp_high_temp + (opt.crp_low_temp - opt.crp_high_temp) * std::min(1.0, (double)it / Ni);
    cml_gibbs_sweep_opts so{};
    so.mode = opt.crp_batched ? CML_GIBBS_BATCHED : CML_GIBBS_SEQUENTIAL;
    so.power = temperature > 0 ? 1. / temperature : 1.;
    so.seed = opt.crp_seed;
    so.sweep = it;
    so.init_from_params = 0;
    so.accumulate_dt = it == Ni ? 1. : time_of(it + 1) - time_of(it);
    ok(cml_forests_gibbs_sweep(ctx, &so));
    ok(cml_forests_gibbs_get_samples(ctx, len.data(), ids.data(), cap, base.data()));
    double ln_p = 0;
    if (opt.crp_sample_prob) {  // as carmel-b200 --sample-prob: scored with the new sample's counts back in
      for (uint64_t f = 0; f < nf; ++f) {
        for (uint32_t k = 0; k < prev_len[f]; ++k) {
          const uint32_t p = prev_ids[base[f] + k];
          if (norm[p] != 0xFFFFFFFFu) sp_count[p] -= 1., sp_sum[norm[p]] -= 1.;
        }
        for (uint32_t k = 0; k < len[f]; ++k) {
          const uint32_t p = ids[base[f] + k];
          if (norm[p] != 0xFFFFFFFFu) sp_count[p] += 1., sp_sum[norm[p]] += 1.;
        }
        for (uint32_t k = 0; k < len[f]; ++k) {
          const uint32_t p = ids[base[f] + k];
          ln_p += norm[p] != 0xFFFFFFFFu ? std::log(sp_count[p] / sp_sum[norm[p]]) : std::log(prior[p]);
        }
      }
      prev_len = len;
      prev_ids = ids;
    } else {  // cache model (gibbs.hpp:137-140,700-742): reset every sweep
      std::fill(csum.begin(), csum.end(), 0.);
      for (uint64_t p = 0; p < rulespace; ++p) {
        ccount[p] = prior[p];
        if (norm[p] != 0xFFFFFFFFu) csum[norm[p]] += prior[p];
      }
      for (uint64_t f = 0; f < nf; ++f)
        for (uint32_t k = 0; k < len[f]; ++k) {
          const uint32_t p = ids[base[f] + k];
          ln_p += norm[p] != 0xFFFFFFFFu ? std::log(ccount[p]++ / csum[norm[p]]++) : std::log(prior[p]);
        }
    }
    history.push_back({it, ln_p, 0., 0, nf});
    log << "Gibbs i=" << it << (opt.crp_sample_prob ? " sample prob=" : " cache-model prob=") << format_base2(ln_p);
    if (n_sym) log << " per-point-ppx(N=" << n_sym << ")=" << format_base2(-ln_p / n_sym);
    log << " per-block-ppx(N=" << nf << ")=" << format_base2(-ln_p / (double)nf) << "\n";
  }
  if (!opt.outsample_file.empty()) {  // print_sample (forest-em.hpp:775-784)
    std::ofstream o(opt.outsample_file);
    for (uint64_t f = 0; f < nf; ++f) {
      for (uint32_t k = 0; k < len[f]; ++k) o << (k ? " " : "") << ids[base[f] + k];
      o << "\n";
    }
  }
  // finalize_cumulative_counts (gibbs.hpp:626-644) + from_gibbs (forest-em.hpp:743-750)
  std::vector<double> count(rulespace), cum(rulespace), normsum(n_norms, 0.), v(rulespace);
  ok(cml_forests_gibbs_get_state(ctx, count.data(), cum.data(), nullptr));
  const double tmax1 = ((double)Ni - (double)burnin) + 1;
  for (uint64_t p = 0; p < rulespace; ++p) {
    if (opt.crp_final_counts && !opt.crp_exclude_prior)
      v[p] = count[p];
    else if (opt.crp_final_counts)
      v[p] = count[p] - prior[p];
    else
      v[p] = cum[p] - (opt.crp_exclude_prior ? prior[p] * tmax1 : 0.);
    if (norm[p] != 0xFFFFFFFFu) normsum[norm[p]] += v[p];
  }
  for (uint64_t p = 0; p < rulespace; ++p) {
    const double fp = norm[p] != 0xFFFFFFFFu ? (v[p] > 0 ? v[p] / normsum[norm[p]] : 0.) : prior[p];
    ln_w[p] = fp > 0 ? std::log(fp) : kNegInfD;
  }
  ok(cml_forests_set_params(ctx, ln_w.data()));
  gibbs_done = true;
}

// forest-em-params.cpp:116-136 outputs; forest-em.hpp:190-201 write_params / write_counts
void ForestJob::write_outputs(std::ostream& log) {
  const bool dbl = opt.double_precision;
  if (ctx) ok(cml_forests_get_params(ctx, ln_w.data()));
  if (!opt.outparam_file.empty()) {
    log << "Writing trained parameters to " << opt.outparam_file << "\n";
    std::ofstream o(opt.outparam_file);
    write_params_to(o);
  }
  if (!opt.outcounts_file.empty()) {
    log << "Writing trained counts to " << opt.outcounts_file << "\n";
    std::ofstream o(opt.outcounts_file);
    write_counts_to(o);
  }
  if (!opt.outinside_file.empty() && ctx) {  // final_iteration (forest-em.hpp:500-509) with the final weights
    log << "Running final per-forest inside score printing.\n";
    ok(cml_forests_estimate(ctx, nullptr));
    std::vector<double> in(shard_end - shard_begin);
    ok(cml_forests_get_inside(ctx, in.data(), in.size()));
    std::ofstream o(opt.outinside_file);
    for (double v : in) o << fmt_forest_weight(v, dbl, opt.human_probs) << "\n";
  }
  if (!opt.outviterbi_file.empty() && ctx) {  // forest-em-params.cpp:125-131, forest-em.hpp:490-495,535-550
    log << "Running final viterbi forests decoding.\n";
    ok(cml_forests_estimate(ctx, nullptr));
    const uint64_t nf = shard_end - shard_begin;
    std::vector<double> sum(nf), best(nf);
    ok(cml_forests_get_inside(ctx, sum.data(), nf));
    std::vector<uint64_t> off(forests.node_off.begin() + shard_begin, forests.node_off.begin() + shard_end + 1);
    const uint64_t o0 = off.empty() ? 0 : off[0];
    for (auto& v : off) v -= o0;
    cml_forest_batch b{};
    b.n_forests = nf;
    b.node_off = off.data();
    b.next = forests.next.data() + o0;
    b.label = forests.label.data() + o0;
    b.backref = forests.backref.data() + o0;
    std::ofstream o(opt.outviterbi_file);
    // write_viterbi_rec (forest.hpp:590-631) without recursion: a stack of (node, next child) for the AND nodes;
    // and_of(slot) is the AND node a child slot (AND node, OR node or shared node) stands for in the derivation
    auto write_tree = [&](uint64_t f, auto&& and_of) {
      const uint32_t* nx = b.next + off[f];
      const uint32_t* lb = b.label + off[f];
      std::vector<std::pair<uint32_t, uint32_t>> st;
      uint32_t cur = 0;
      bool have = true;
      while (have || !st.empty()) {
        if (have) {
          cur = and_of(cur);
          if (nx[cur] == cur + 1) {
            o << lb[cur];
            have = false;
          } else {
            o << '(' << lb[cur];
            st.emplace_back(cur, cur + 1);
            have = false;
          }
        }
        if (st.empty()) break;
        auto& top = st.back();
        if (top.second == nx[top.first]) {
          o << ')';
          st.pop_back();
          continue;
        }
        o << ' ';
        cur = top.second;
        top.second = nx[cur];
        have = true;
      }
      o << '\n';
    };
    const uint32_t K = opt.sample ? opt.sample : opt.kbest;
    if (opt.sample) {  // n drawn derivations per forest, seed --seed, key = the forest's index in the file
      std::vector<double> lnw(nf * K), total(nf);
      std::vector<uint32_t> len(nf * K), nodes(std::max<uint64_t>(1, (nf ? off[nf] : 0) * K));
      std::vector<uint64_t> base(nf * K + 1);
      int rc = cml_forests_sample(ctx, &b, K, opt.crp_seed, nullptr, lnw.data(), len.data(), base.data(), nodes.data(),
                                  nodes.size(), total.data());
      if (rc == CML_ERR_ARG && base[nf * K] > nodes.size()) {
        nodes.resize(base[nf * K]);
        rc = cml_forests_sample(ctx, &b, K, opt.crp_seed, nullptr, lnw.data(), len.data(), base.data(), nodes.data(),
                                nodes.size(), total.data());
      }
      ok(rc);
      uint64_t found = 0;
      for (uint64_t f = 0; f < nf; ++f) {
        found += total[f] > kNegInfD;
        for (uint32_t r = 0; r < K; ++r) {
          const uint64_t i = f * K + r;
          o << fmt_forest_weight(lnw[i], dbl, opt.human_probs) << '/' << fmt_forest_weight(sum[f], dbl, opt.human_probs);
          if (!(lnw[i] > kNegInfD)) {
            o << "=0% \n";
            continue;
          }
          o << '=' << 100 * std::exp(lnw[i] - sum[f]) << "% ";
          const uint32_t* next_and = nodes.data() + base[i];
          write_tree(f, [&](uint32_t) { return *next_and++; });
        }
      }
      log << "Viterbi: " << K << " samples per forest, " << found << " forests with a derivation\n";
    } else if (K == 1) {
      std::vector<uint32_t> choice(nf ? off[nf] : 0);
      ok(cml_forests_viterbi(ctx, &b, best.data(), choice.data()));
      for (uint64_t f = 0; f < nf; ++f) {
        const uint32_t* lb = b.label + off[f];
        const uint8_t* br = b.backref + off[f];
        const uint32_t* ch = choice.data() + off[f];
        o << fmt_forest_weight(best[f], dbl, opt.human_probs) << '/' << fmt_forest_weight(sum[f], dbl, opt.human_probs) << '='
          << 100 * std::exp(best[f] - sum[f]) << "% ";
        write_tree(f, [&](uint32_t c) {
          while (br[c] || lb[c] == 0) c = br[c] ? lb[c] : ch[c];  // shared node / OR node: follow
          return c;
        });
      }
    } else {  // n lines per forest, best first; a rank past the last derivation reads "0/<sum>=0% " with no tree
      std::vector<double> score(nf * K);
      std::vector<uint32_t> len(nf * K), nodes(std::max<uint64_t>(1, (nf ? off[nf] : 0) * K));
      std::vector<uint64_t> base(nf * K + 1);
      // a derivation without shared nodes has at most one AND node per forest node; shared nodes can need more
      int rc = cml_forests_kbest(ctx, &b, K, score.data(), len.data(), base.data(), nodes.data(), nodes.size());
      if (rc == CML_ERR_ARG && base[nf * K] > nodes.size()) {
        nodes.resize(base[nf * K]);
        rc = cml_forests_kbest(ctx, &b, K, score.data(), len.data(), base.data(), nodes.data(), nodes.size());
      }
      ok(rc);
      uint64_t found = 0;
      for (uint64_t f = 0; f < nf; ++f)
        for (uint32_t r = 0; r < K; ++r) {
          const uint64_t i = f * K + r;
          if (!(score[i] > kNegInfD)) {
            o << fmt_forest_weight(score[i], dbl, opt.human_probs) << '/' << fmt_forest_weight(sum[f], dbl, opt.human_probs)
              << "=0% \n";
            continue;
          }
          ++found;
          o << fmt_forest_weight(score[i], dbl, opt.human_probs) << '/' << fmt_forest_weight(sum[f], dbl, opt.human_probs)
            << '=' << 100 * std::exp(score[i] - sum[f]) << "% ";
          const uint32_t* next_and = nodes.data() + base[i];
          write_tree(f, [&](uint32_t) { return *next_and++; });
        }
      log << "Viterbi: " << K << "-best lists, " << found << " derivations found\n";
    }
  }
  if (!opt.history_file.empty()) {
    std::ofstream o(opt.history_file);
    o.precision(17);
    for (auto const& h : history) o << h.iter << ' ' << h.avg_logprob << ' ' << h.max_delta << ' ' << h.max_index << ' ' << h.n << "\n";
  }
  if (!opt.print_forests_file.empty()) {
    std::ofstream o(opt.print_forests_file);
    if (!prepared) compute_shard();
    for (uint64_t f = shard_begin; f < shard_end; ++f) {  // with --shard=r/N: this rank's block only
      forests.print(o, f);
      o << "\n";
    }
  }
}

// forest-em-params.hpp:69-176 (training subset) + validate_parameters (forest-em-params.cpp:21-60)
int open_forest_job(int argc, const char* const* argv, ForestJob& job, std::ostream& err) {
  static const std::map<std::string, char> longs = {
      {"forests-file", 'f'},      {"normgroups-file", 'n'},      {"initparam-file", 'I'},  {"outparam-file", 'o'},
      {"outcounts-file", 'O'},    {"max-iter", 'i'},             {"converge", 'e'},        {"deltaparam-epsilon", 'd'},
      {"prior-counts-per", 'p'},  {"add-k-smoothing", 'k'},      {"zero-zerocounts", 'z'}, {"initial-1-params", 'u'},
      {"normalize-initial", 'N'}, {"use-double-precision", 'U'}, {"human-probs", 'H'},     {"log-level", 'L'},
      {"out-per-forest-inside-sum", 'S'}, {"max-forest-nodes", 'm'}, {"max-normgroup-size", 'M'}, {"prealloc-params", 'P'},
      {"tempfile-prefix", 't'},   {"forest-tick-period", 'T'},   {"watch-period", 'W'},    {"random-seed", 's'},
      {"random-restarts", 'r'},   {"checkpoint-prefix", 'x'},    {"checkpoint-parameters", 'c'}, {"outviterbi-file", 'v'}};
  ForestOpts& a = job.opt;
  bool have_kbest = false;
  try {
    for (int i = 1; i < argc; ++i) {
      const std::string s = argv[i];
      char c = 0;
      std::string val;
      bool have_val = false;
      if (s.rfind("--", 0) == 0) {
        const size_t eq = s.find('=');
        const std::string key = s.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
        if (eq != std::string::npos) {
          val = s.substr(eq + 1);
          have_val = true;
        }
        if (key == "history") { a.history_file = val; continue; }
        if (key == "print-forests") { a.print_forests_file = val; continue; }
        if (key == "parse-only") { a.parse_only = true; continue; }
        if (key == "layout") {
          if (val != "auto" && val != "group" && val != "thread" && val != "level") throw std::runtime_error("--layout=auto|group|thread|level");
          a.layout = val == "group" ? CML_FOREST_LAYOUT_GROUP : val == "thread" ? CML_FOREST_LAYOUT_THREAD : val == "level" ? CML_FOREST_LAYOUT_LEVEL : CML_FOREST_LAYOUT_AUTO;
          continue;
        }
        if (key == "gpu") { a.device = std::atoi(val.c_str()); continue; }
        if (key == "kbest") {
          char* end = nullptr;
          const unsigned long long n = val.empty() || val[0] < '0' || val[0] > '9' ? 0 : std::strtoull(val.c_str(), &end, 10);
          if (!n || *end || n > 0xFFFFFFFFull) throw std::runtime_error("--kbest=n needs a whole number of derivations >= 1 (got \"" + val + "\")");
          a.kbest = (uint32_t)n;
          have_kbest = true;
          continue;
        }
        if (key == "sample") {
          char* end = nullptr;
          const unsigned long long n = val.empty() || val[0] < '0' || val[0] > '9' ? 0 : std::strtoull(val.c_str(), &end, 10);
          if (!n || *end || n > 0xFFFFFFFFull) throw std::runtime_error("--sample=n needs a whole number of samples >= 1 (got \"" + val + "\")");
          a.sample = (uint32_t)n;
          continue;
        }
        if (key == "crp") { a.crp_iter = (unsigned)std::atol(val.c_str()); continue; }
        if (key == "burnin") { a.crp_burnin = (unsigned)std::atol(val.c_str()); continue; }
        if (key == "const-alpha") { a.crp_alpha = std::atof(val.c_str()); continue; }
        if (key == "high-temp") { a.crp_high_temp = std::atof(val.c_str()); continue; }
        if (key == "low-temp") { a.crp_low_temp = std::atof(val.c_str()); continue; }
        if (key == "n-symbols") { a.crp_n_sym = std::atof(val.c_str()); continue; }
        if (key == "seed") { a.crp_seed = std::strtoull(val.c_str(), nullptr, 10); continue; }
        if (key == "outsample-file") { a.outsample_file = val; continue; }
        if (key == "uniform-p0") { a.crp_uniform_p0 = true; continue; }
        if (key == "final-counts") { a.crp_final_counts = true; continue; }
        if (key == "crp-exclude-prior") { a.crp_exclude_prior = true; continue; }
        if (key == "sample-prob") { a.crp_sample_prob = true; continue; }
        if (key == "crp-batched") { a.crp_batched = true; continue; }
        if (key == "alpha" || key == "include-self" || key == "expectation" || key == "crp-restarts" || key == "init-em" ||
            key == "prior-inference-stddev")  // sampler variants this path does not build: refuse, do not ignore
          throw std::runtime_error("--" + key + " is not supported by forest-em-b200");
        if (key == "shard") {
          const size_t sl = val.find('/');
          if (sl == std::string::npos) throw std::runtime_error("--shard=r/N needs 0 <= r < N");
          a.shard_rank = std::atoi(val.substr(0, sl).c_str());
          a.shard_count = std::atoi(val.substr(sl + 1).c_str());
          if (a.shard_count < 1 || a.shard_rank < 0 || a.shard_rank >= a.shard_count) throw std::runtime_error("--shard=r/N needs 0 <= r < N");
          continue;
        }
        auto it = longs.find(key);
        if (it == longs.end()) throw std::runtime_error("unknown option --" + key);
        c = it->second;
      } else if (s.size() >= 2 && s[0] == '-') {
        c = s[1];
        if (s.size() > 2) {
          val = s.substr(2);
          have_val = true;
        }
      } else
        throw std::runtime_error("unexpected argument " + s);
      auto need = [&]() -> std::string {
        if (have_val) return val;
        if (i + 1 >= argc) throw std::runtime_error(std::string("option -") + c + " needs a value");
        return argv[++i];
      };
      switch (c) {
        case 'f': a.forests_file = need(); break;
        case 'n': a.normgroups_file = need(); break;
        case 'I': a.initparam_file = need(); break;
        case 'o': a.outparam_file = need(); break;
        case 'O': a.outcounts_file = need(); break;
        case 'S': a.outinside_file = need(); break;
        case 'v': a.outviterbi_file = need(); break;
        case 'i': a.max_iter = (unsigned)std::atol(need().c_str()); break;
        case 'e': a.converge_ratio = std::atof(need().c_str()); break;
        case 'd': a.converge_delta = std::atof(need().c_str()); break;
        case 'p': a.prior_counts = std::atof(need().c_str()); break;
        case 'k': a.add_k_smoothing = std::atof(need().c_str()); break;
        case 'L': a.log_level = (unsigned)std::atol(need().c_str()); break;
        case 'r': a.random_restarts = (unsigned)std::atol(need().c_str()); break;
        case 's': a.random_seed = std::strtoull(need().c_str(), nullptr, 10); break;
        case 'W': a.watch_period = (unsigned)std::atol(need().c_str()); break;
        case 'x': a.checkpoint_prefix = need(); break;
        case 'c': a.checkpoint_parameters = true; break;
        case 'm': case 'M': case 'P': case 't': case 'T': need(); break;  // sizing / cosmetic: accepted, unused
        case 'z': a.zero_zerocounts = true; break;
        case 'u': a.initial_1_params = true; break;
        case 'N': a.normalize_initial = true; break;
        case 'U': a.double_precision = true; break;
        case 'H': a.human_probs = true; break;
        default: throw std::runtime_error(std::string("unknown option -") + c);
      }
    }
    if (have_kbest && a.outviterbi_file.empty()) throw std::runtime_error("--kbest=n needs -v (outviterbi-file)");
    if (have_kbest && a.shard_count > 1) throw std::runtime_error("--kbest decodes on one GPU (no --gpus / --shard)");
    if (a.sample && a.outviterbi_file.empty()) throw std::runtime_error("--sample=n needs -v (outviterbi-file)");
    if (a.sample && have_kbest) throw std::runtime_error("--sample=n draws derivations in place of --kbest: give one of them");
    if (a.sample && a.shard_count > 1) throw std::runtime_error("--sample draws on one GPU (no --gpus / --shard)");
    if (a.max_iter && a.forests_file.empty()) throw std::runtime_error("Missing forests-file.");
    if (a.normgroups_file.empty() && (a.max_iter || a.normalize_initial)) throw std::runtime_error("Missing normgroups-file.\n");
    job.load();
  } catch (std::exception& e) {
    err << "ERROR: " << e.what() << "\n\nTry 'forest-em -h' for documentation\n";
    return 1;
  }
  return 0;
}

}  // namespace cb

// ---- C ABI: a whole forest-em run ---------------------------------------------------------------------------
struct cml_forest_job {
  cb::ForestJob job;
  std::string err;
  bool quiet = false;
};
namespace {
template <class F>
int fguarded(cml_forest_job* j, F&& f) {
  if (!j) return CML_ERR_ARG;
  try {
    return f();
  } catch (std::exception& e) {
    j->err = e.what();
    return CML_ERR_STATE;
  }
}
}  // namespace
extern "C" int cml_forest_job_open(cml_forest_job** out, int argc, const char* const* argv) {
  if (!out) return CML_ERR_ARG;
  *out = new cml_forest_job();
  cml_forest_job* j = *out;
  return fguarded(j, [&]() {
    std::ostringstream msg;
    const int rc = cb::open_forest_job(argc, argv, j->job, msg);
    if (rc != 0) {
      j->err = msg.str();
      std::cerr << j->err;
      return (int)CML_ERR_ARG;
    }
    return (int)CML_OK;
  });
}
extern "C" void cml_forest_job_close(cml_forest_job* j) { delete j; }
extern "C" const char* cml_forest_job_error(cml_forest_job* j) { return j ? j->err.c_str() : "null job"; }
extern "C" int cml_forest_job_set_comm(cml_forest_job* j, const unsigned char id[128]) {
  if (!j || !id) return CML_ERR_ARG;
  std::memcpy(j->job.comm_id, id, 128);
  j->job.have_comm_id = true;
  return CML_OK;
}
extern "C" int cml_forest_job_set_allreduce(cml_forest_job* j, cml_allreduce_fn fn, void* user) {
  if (!j) return CML_ERR_ARG;
  j->job.allreduce = fn;
  j->job.allreduce_user = user;
  return CML_OK;
}
extern "C" int cml_forest_job_prepare(cml_forest_job* j) {
  return fguarded(j, [&]() {
    j->job.prepare();
    return (int)CML_OK;
  });
}
extern "C" cml_forests* cml_forest_job_context(cml_forest_job* j) { return j ? j->job.ctx : nullptr; }
extern "C" int cml_forest_job_set_quiet(cml_forest_job* j, int quiet) {  // ranks > 0 of a multi-GPU run do not log
  if (!j) return CML_ERR_ARG;
  j->quiet = quiet != 0;
  return CML_OK;
}
extern "C" int cml_forest_job_train(cml_forest_job* j) {
  return fguarded(j, [&]() {
    std::ostringstream sink;
    std::ostream& lg = j->quiet ? (std::ostream&)sink : (std::ostream&)std::cerr;
    if (j->job.opt.crp_iter)
      j->job.run_gibbs(lg);  // forest-em-params.cpp:112-113: gibbs replaces EM
    else
      j->job.run(lg);
    return (int)CML_OK;
  });
}
extern "C" int cml_forest_job_write(cml_forest_job* j) {
  return fguarded(j, [&]() {
    j->job.write_outputs(std::cerr);
    return (int)CML_OK;
  });
}
extern "C" int cml_forest_job_stats(cml_forest_job* j, cml_forest_job_info* info) {
  if (!j || !info) return CML_ERR_ARG;
  std::memset(info, 0, sizeof(*info));
  if (j->job.ctx) cml_forests_totals(j->job.ctx, &info->forests, &info->nodes, &info->hyperedges, &info->links);
  info->rulespace = j->job.rulespace;
  info->iterations = j->job.history.size();
  info->best_avg_logprob = j->job.best_alp;
  return CML_OK;
}
