// job.cpp -- a training run as an object: carmel's argv grammar, transducer / corpus loading,
// composition, output writing, and the cml_job_* C entry points the command line, the Python
// multi-GPU driver and bench.py share.
//
// argv grammar kept from the reference (carmel/src/carmel.cc:929-1066): bundled single-character
// flags, value flags that consume the NEXT argument, --key[=value] long options (unknown keys are
// accepted silently, as in the reference), first file = training corpus, the rest = transducers
// composed left to right (carmel.cc:1286-1355).
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "carmel_host.hpp"

namespace cb {

static std::vector<std::string> split(std::string const& s, char c) {
  std::vector<std::string> r;
  std::stringstream ss(s);
  std::string t;
  while (std::getline(ss, t, c)) r.push_back(t);
  if (r.empty()) r.push_back("");
  return r;
}

int open_job(int argc, const char* const* argv, TrainJob& job, std::ostream& err) {
  std::vector<std::string> files;
  std::vector<char> pending;  // value flags waiting for their argument
  TrainOpts& topt = job.opt;
  NormGroupBy default_group = CONDITIONAL;
  bool* flags = job.flags;
  auto& lopt = job.lopt;
  for (int i = 1; i < argc; ++i) {
    const std::string arg = argv[i];
    if (!pending.empty()) {
      // carmel binds pending value flags by a FIXED priority chain, not in the order they were written
      // (carmel.cc:930-990: = N X o ! R w z k g M L T e f p F +); 'G' shares -g's argument (carmel.cc:1043)
      static const char kPriority[] = "=NXo!RwzkgMLTefpF+";
      size_t best = 0;
      for (size_t q = 1; q < pending.size(); ++q)
        if (std::strchr(kPriority, pending[q]) < std::strchr(kPriority, pending[best])) best = q;
      const char p = pending[best];
      pending.erase(pending.begin() + best);
      double w = 0;
      switch (p) {
        case 'M': topt.max_iter = (uint32_t)std::atol(arg.c_str()); break;
        case 'e':
          if (parse_weight(arg.c_str(), w)) topt.ln_converge_delta = w;
          break;
        case 'X':
          if (parse_weight(arg.c_str(), w)) topt.ln_converge_ratio = w;
          break;
        case 'f':
          if (parse_weight(arg.c_str(), w)) topt.ln_smooth_floor = w;
          break;
        case 'o': topt.rate_growth = std::max(1., std::atof(arg.c_str())); break;
        case 'F': job.outfile = arg; break;
        case '!': topt.ran_restarts = (uint32_t)std::atol(arg.c_str()); break;
        case 'R': topt.seed = std::strtoull(arg.c_str(), nullptr, 10); break;
        case 'k': topt.kbest_arg = arg; break;
        default: break;  // accepted, unused on this path
      }
      continue;
    }
    if (arg.size() > 1 && arg[0] == '-') {
      if (arg[1] == '-') {
        const size_t eq = arg.find('=');
        const std::string key = arg.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
        const std::string val = eq == std::string::npos ? "" : arg.substr(eq + 1);
        lopt[key] = val;
        err << "option " << key << " = " << val << std::endl;
      } else {
        for (size_t k = 1; k < arg.size(); ++k) {
          const char c = arg[k];
          flags[(unsigned char)c] = true;
          if (std::strchr("MeXfoFR!kTpwzgLN=+", c)) pending.push_back(c);
          if (c == 'G') pending.push_back('g');
          if (c == 'j') default_group = JOINT;
          if (c == 'u') default_group = NONE;
        }
      }
    } else
      files.push_back(arg);
  }
  // flags that change WHAT is computed and that this path does not build are refused, not ignored:
  // -r (right-to-left composition), -a (mediate-state composition: different composed arc ids), -+ (digamma)
  for (const char c : {'r', 'a', '+'})
    if (flags[(unsigned char)c]) {
      err << "carmel-b200: -" << c << " is not implemented on the training path\n";
      return -11;
    }
  // --decode=FILE --given=input|output: decode the strings of the first file with the other tape free (in place of -t)
  const bool decode = lopt.count("decode") > 0;
  if (decode) {
    const std::string g = lopt.count("given") ? lopt["given"] : "";
    if (g != "input" && g != "output") {
      err << "carmel-b200: --decode needs --given=input or --given=output (the tape the strings are on)\n";
      return -9;
    }
    if (lopt.count("viterbi") || lopt.count("crp")) {
      err << "carmel-b200: --decode cannot be combined with --viterbi or --crp\n";
      return -9;
    }
    // --decode decodes instead of training: switches that train, or write what only training writes, are refused
    // rather than ignored
    for (const char c : {'t', 'F', 'M', '!'})
      if (flags[(unsigned char)c]) {
        err << "carmel-b200: --decode cannot be combined with -" << c << " (it decodes instead of training)\n";
        return -9;
      }
    for (const char* k : {"trellis-only", "dump-trellis", "history", "fem-forest", "fem-norm", "fem-param", "dump-samples"})
      if (lopt.count(k)) {
        err << "carmel-b200: --decode cannot be combined with --" << k << "\n";
        return -9;
      }
    topt.given_tape = g == "input" ? 0 : 1;
  }
  // --crp forces -t and --train-cascade (carmel.cc:255-304 parse_gibbs_opts)
  const bool crp = lopt.count("crp") > 0;
  const bool trainc = lopt.count("train-cascade") > 0 || crp;
  job.train_cascade = trainc;
  if (trainc) flags[(unsigned)'t'] = true;
  if (crp) {
    // Options of carmel's sampler (carmel.cc:268-302) that change what is sampled and that this path does not
    // build: refuse them instead of training something else under the same command line.
    static const char* const not_built[] = {"random-start", "include-self", "crp-restarts",
                                            "crp-argmax-final", "crp-argmax-sum", "init-em", "em-p0",
                                            "init-from-p0", "prior-inference-stddev", "prior-inference-global",
                                            "prior-inference-restart-fresh"};
    for (const char* k : not_built)
      if (lopt.count(k)) {
        err << "carmel-b200: --" << k << " is not implemented on the --crp path\n";
        return -11;
      }
    GibbsOpts& g = job.gopt;
    g.enabled = true;
    g.iter = lopt["crp"].empty() ? topt.max_iter : (uint32_t)std::atol(lopt["crp"].c_str());
    if (lopt.count("burnin")) g.burnin = (uint32_t)std::atol(lopt["burnin"].c_str());
    g.uniform_p0 = lopt.count("uniform-p0") > 0;
    g.dirichlet_p0 = lopt.count("dirichlet-p0") > 0;
    g.final_counts = lopt.count("final-counts") > 0;
    g.exclude_prior = lopt.count("crp-exclude-prior") > 0;
    if (lopt.count("high-temp")) g.high_temp = std::atof(lopt["high-temp"].c_str());
    if (lopt.count("low-temp")) g.low_temp = std::atof(lopt["low-temp"].c_str());
    if (lopt.count("seed")) g.seed = std::strtoull(lopt["seed"].c_str(), nullptr, 10);
    g.batched = lopt.count("crp-batched") > 0;
    g.sample_prob = lopt.count("sample-prob") > 0;
    g.expectation = lopt.count("expectation") > 0;
    if (lopt.count("dump-samples")) g.dump_samples_file = lopt["dump-samples"];
  }
  if (!flags[(unsigned)'t'] && !decode) {
    err << "carmel-b200 implements carmel's training path only: use -t (or --train-cascade)\n";
    return -11;
  }
  if (files.size() < 2) return -9;
  topt.weight_is_prior = flags[(unsigned)'U'];
  {
    double w = 0;
    if (lopt.count("restart-tolerance") && parse_weight(lopt["restart-tolerance"].c_str(), w)) topt.ln_restart_tolerance = w;
    if (lopt.count("final-restart-tolerance") && parse_weight(lopt["final-restart-tolerance"].c_str(), w))
      topt.ln_final_restart_tolerance = w;
    if (lopt.count("final-restart")) topt.final_restart = (uint32_t)std::atol(lopt["final-restart"].c_str());
  }
  if (lopt.count("float")) topt.precision = 32;
  if (lopt.count("scaled")) topt.space = CML_SPACE_SCALED;
  if (lopt.count("no-ell")) topt.no_ell = true;
  if (lopt.count("no-dense")) topt.dense = -1;
  if (lopt.count("fem-forest")) topt.dense = -1;  // the forests are the derivation lattices (carmel.cc:764-767 force_cascade_derivs)
  if (lopt.count("lane-min")) topt.lane_min = std::atoi(lopt["lane-min"].c_str());
  if (lopt.count("no-lane")) topt.lane_min = 0;
  if (lopt.count("no-factor")) topt.no_factor = true;
  if (lopt.count("no-wide")) topt.no_wide = true;
  if (lopt.count("dense")) topt.dense = 1;
  if (lopt.count("device-build")) topt.device_build = 1;
  if (lopt.count("host-build")) topt.device_build = -1;
  if (lopt.count("gpu")) topt.device = std::atoi(lopt["gpu"].c_str());
  if (lopt.count("history")) topt.history_file = lopt["history"];
  if (lopt.count("dump-trellis")) topt.dump_trellis_file = lopt["dump-trellis"];
  if (lopt.count("shard")) {
    const auto v = split(lopt["shard"], '/');
    if (v.size() != 2 || std::atoi(v[1].c_str()) < 1 || std::atoi(v[0].c_str()) < 0 ||
        std::atoi(v[0].c_str()) >= std::atoi(v[1].c_str())) {
      err << "--shard=r/N needs 0 <= r < N\n";
      return -9;
    }
    topt.shard_rank = std::atoi(v[0].c_str());
    topt.shard_count = std::atoi(v[1].c_str());
  }

  job.corpus_file = files[0];
  job.fst_files.assign(files.begin() + 1, files.end());
  // --sample=n / --sum=FILE with --viterbi / --decode: draw n derivations per example instead of the best ones / write
  // ln of every example's total weight (without --viterbi / --decode they are unknown long options, accepted and unused)
  if ((lopt.count("viterbi") || decode) && lopt.count("sample")) {
    if (flags[(unsigned)'k']) {
      err << "carmel-b200: --sample cannot be combined with -k (it draws derivations instead of listing the best)\n";
      return -9;
    }
    const std::string v = lopt["sample"];
    char* end = nullptr;
    const unsigned long long n = std::strtoull(v.c_str(), &end, 10);
    if (v.empty() || *end || v[0] == '-' || n < 1 || n > 0xFFFFFFFFull) {
      err << "carmel-b200: --sample needs a whole number of derivations >= 1 (got \"" << v << "\")\n";
      return -9;
    }
    topt.sample = (uint32_t)n;
  }
  if ((lopt.count("viterbi") || decode) && lopt.count("sum")) {
    if (lopt["sum"].empty()) {
      err << "carmel-b200: --sum needs a file name (--sum=FILE)\n";
      return -9;
    }
    topt.sum_file = lopt["sum"];
  }
  if ((lopt.count("viterbi") || decode) && flags[(unsigned)'k']) {  // -k n with --viterbi / --decode: n derivations each
    char* end = nullptr;
    const unsigned long long n = std::strtoull(topt.kbest_arg.c_str(), &end, 10);
    if (topt.kbest_arg.empty() || *end || topt.kbest_arg[0] == '-' || n < 1 || n > 0xFFFFFFFFull) {
      err << "carmel-b200: -k needs a whole number of derivations >= 1 (got \"" << topt.kbest_arg << "\")\n";
      return -9;
    }
    topt.kbest = (uint32_t)n;
  }
  const uint32_t n_chain = (uint32_t)job.fst_files.size();
  for (auto const& f : job.fst_files) {
    std::ifstream in(f);
    if (!in) {
      err << "File " << f << " could not be opened for input.\n";
      return -9;
    }
    std::unique_ptr<Wfst> w(new Wfst());
    if (!w->read(in, !flags[(unsigned)'K'])) {
      err << "Bad format of transducer file: " << f << "\n";
      return -2;
    }
    if (n_chain > 1 && !flags[(unsigned)'m']) w->named = false;  // carmel.cc:1197
    job.chain.push_back(std::move(w));
  }
  job.methods.assign(n_chain, NormalizeMethod());
  for (auto& m : job.methods) m.group = default_group;
  if (lopt.count("normby")) {
    const std::string s = lopt["normby"];
    for (uint32_t i = 0; i < n_chain && !s.empty(); ++i) {
      const char c = i < s.size() ? s[i] : s.back();
      job.methods[i].group = (c == 'j' || c == 'J') ? JOINT : (c == 'c' || c == 'C') ? CONDITIONAL : NONE;
    }
  }
  if (lopt.count("priors")) {
    const auto v = split(lopt["priors"], ',');
    for (uint32_t i = 0; i < n_chain; ++i) {
      double w;
      if (parse_weight((i < v.size() ? v[i] : v.back()).c_str(), w)) job.methods[i].ln_add_count = w;
    }
  }

  Cascade& cascade = job.cascade;
  cascade.trivial = !(trainc && n_chain >= 2);
  if (!cascade.trivial) cascade.chains.emplace_back();  // chain 0 = nil (cascade.h:366-383)
  Wfst* result = job.chain[0].get();
  if (!flags[(unsigned)'d']) result->reduce();  // carmel.cc:1286 cm.minimize(result)
  for (auto& w : job.chain) cascade.members.push_back(w.get());
  cascade.number_members();  // after reducing the first member: parameter ids = final arc order
  for (uint32_t i = 1; i < n_chain && result->valid; ++i) {
    std::unique_ptr<Wfst> next = compose(cascade, *result, *job.chain[i], i > 1, 0, i);
    if (!flags[(unsigned)'q']) err << "\n\t(" << next->num_states() << " states / " << next->num_arcs() << " arcs";
    if (!next->valid) {
      err << ")\nEmpty or invalid result of composition with transducer \"" << job.fst_files[i] << "\".\n";
      return -3;
    }
    const uint32_t st = next->num_states();
    const size_t na = next->num_arcs();
    if (!flags[(unsigned)'d']) next->reduce();
    if (!flags[(unsigned)'q']) {
      if (next->num_states() != st || next->num_arcs() != na)
        err << " reduce-> " << next->num_states() << "/" << next->num_arcs();
      err << ")";
    }
    job.composed_keep.push_back(std::move(next));
    result = job.composed_keep.back().get();
  }
  if (!flags[(unsigned)'q']) err << std::endl;
  if (!result->valid) {
    err << "Empty or invalid transducer.\n";
    return -3;
  }
  cascade.composed = result;
  job.x = result;
  if (cascade.trivial) job.methods.resize(1);
  if (lopt.count("write-composed")) {
    std::ofstream o(lopt["write-composed"]);
    result->write(o, true, true, true, WeightFormat());
  }
  std::ifstream cf(job.corpus_file);
  if (!cf) {
    err << "File " << job.corpus_file << " could not be opened for input.\n";
    return -9;
  }
  if (decode)
    job.corpus.read_strings(cf, *result, topt.given_tape);
  else
    job.corpus.read(cf, *result);
  return 0;
}

void TrainJob::write_outputs(std::ostream& out) {
  WeightFormat wf;
  if (flags[(unsigned)'B'])
    wf.base = WeightFormat::LOG10;
  else if (flags[(unsigned)'2'])
    wf.base = WeightFormat::LN;
  if (flags[(unsigned)'Z']) wf.thresh = WeightFormat::ALWAYS;
  if (flags[(unsigned)'D']) wf.thresh = WeightFormat::NEVER;
  const bool full = flags[(unsigned)'J'], onearc = flags[(unsigned)'H'];
  if (train_cascade) {  // cascade.h:23-32 write_trained
    for (size_t i = 0; i < fst_files.size(); ++i) {
      const std::string ft = fst_files[i] + ".trained";
      std::cerr << "Writing trained " << fst_files[i] << " to " << ft << std::endl;
      std::ofstream of(ft);
      (cascade.trivial ? x : chain[i].get())->write(of, full, onearc, false, wf);
    }
  } else if (!outfile.empty()) {
    std::ofstream of(outfile);
    if (!of) throw std::runtime_error("Could not create file " + outfile);
    x->write(of, full, onearc, false, wf);
  } else
    x->write(out, full, onearc, false, wf);
}

}  // namespace cb

// -----------------------------------------------------------------------------------------------------
// C entry points (declared in include/carmel_b200.h)
// -----------------------------------------------------------------------------------------------------
struct cml_job {
  cb::TrainJob job;
  std::string err;
  std::ostringstream open_log;
};

namespace {
template <class F>
int guarded(cml_job* j, F&& f) {
  if (!j) return CML_ERR_ARG;
  try {
    return f();
  } catch (std::exception& e) {
    j->err = e.what();
    return j->err.find("No training example had a derivation") != std::string::npos ? CML_ERR_NODERIV : CML_ERR_STATE;
  }
}
}  // namespace

extern "C" int cml_job_open(cml_job** out, int argc, const char* const* argv) {
  if (!out) return CML_ERR_ARG;
  *out = new cml_job();
  cml_job* j = *out;
  return guarded(j, [&]() {
    const int rc = cb::open_job(argc, argv, j->job, std::cerr);
    if (rc != 0) {
      j->err = "carmel exit code " + std::to_string(rc);
      return (int)CML_ERR_ARG;
    }
    return (int)CML_OK;
  });
}
extern "C" void cml_job_close(cml_job* j) { delete j; }
extern "C" const char* cml_job_error(cml_job* j) { return j ? j->err.c_str() : "null job"; }
extern "C" int cml_job_set_comm(cml_job* j, const unsigned char id[128]) {
  if (!j || !id) return CML_ERR_ARG;
  std::memcpy(j->job.comm_id, id, 128);
  j->job.have_comm_id = true;
  return CML_OK;
}

extern "C" int cml_job_set_allreduce(cml_job* j, cml_allreduce_fn fn, void* user) {
  if (!j) return CML_ERR_ARG;
  j->job.allreduce = fn;
  j->job.allreduce_user = user;
  return CML_OK;
}
extern "C" int cml_job_prepare(cml_job* j) {
  return guarded(j, [&]() {
    if (j->job.gopt.enabled)
      j->job.prepare_gibbs();  // --crp: also defines the CRP parameters (counts = priors)
    else
      j->job.prepare();
    return (int)CML_OK;
  });
}
extern "C" cml_ctx* cml_job_context(cml_job* j) { return j ? j->job.ctx : nullptr; }
extern "C" int cml_job_stats(cml_job* j, cml_job_info* info) {
  if (!j || !info) return CML_ERR_ARG;
  info->examples = j->job.res.examples;
  info->trellis_states = j->job.res.trellis_states;
  info->trellis_arcs = j->job.res.trellis_arcs;
  info->device_build_s = j->job.res.device_build_s;
  info->n_params = j->job.M.n_params;
  info->n_arcs = j->job.M.n_arcs;
  info->corpus_pairs = j->job.corpus.n_pairs;
  info->iterations = j->job.res.history.size();
  info->ln_best_ppx = j->job.res.ln_best_ppx;
  info->last_ln_prob = j->job.res.history.empty() ? 0. : j->job.res.history.back().ln_prob;
  info->dense = j->job.res.dense ? 1 : 0;
  return CML_OK;
}
extern "C" int cml_job_train(cml_job* j) {
  return guarded(j, [&]() {
    if (j->job.gopt.enabled)
      j->job.run_gibbs(std::cerr);
    else
      j->job.run(std::cerr);
    return (int)CML_OK;
  });
}
extern "C" int cml_job_write(cml_job* j) {
  return guarded(j, [&]() {
    j->job.write_outputs(std::cout);
    std::cout.flush();
    return (int)CML_OK;
  });
}
