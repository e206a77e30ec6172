// main.cpp -- carmel-b200: carmel's training command line on the B200.
//
// A thin shell over the job object (job.cpp): same argv grammar, log lines and outputs as
// `carmel -t ...` / `carmel --train-cascade ...` (carmel/src/carmel.cc:868-1561).  Exit codes
// follow the reference: 0 ok, -11 on an exception (carmel.cc:1558-1561), -2/-3/-8/-9 input errors.
//
//   carmel-b200 -t [-HJ] [-M n] [-e w] [-X w] [-f w] [-U] [-o g] [-j|-u] [-d] [-K] [-F out]
//               [--train-cascade] [--normby=JCN] [--priors=w,w] [--float] [--scaled] [--gpu=n]
//               [--dump-trellis=file] [--history=file] [--trellis-only] corpus wfst [wfst ...]
//   carmel-b200 --decode=out --given=input|output [-k n | --sample=n [-R seed]] [--sum=file] [--train-cascade] strings wfst ...
#include <cstring>
#include <fstream>
#include <iostream>
#include <memory>
#include <sstream>
#include <thread>

#include "carmel_host.hpp"

using namespace cb;

static void usage() {
  std::cerr << "carmel-b200 (" << cml_version() << "): B200-native carmel training path\n"
               "usage: carmel-b200 -t [options] corpus wfst [wfst ...]\n"
               "  -t            train (EM forward-backward) on the pair corpus\n"
               "  -M n          maximum iterations (default 500)     -e w  converge on max weight change (1e-4)\n"
               "  -X w          converge on perplexity ratio (.999)  -f w  add floor count w to every arc\n"
               "  -U            initial weights are prior counts     -o g  over-relaxation growth factor\n"
               "  -j / -u       joint / no normalisation (default conditional on input)\n"
               "  -d            do not reduce    -K  state names are indices    -F file  output file\n"
               "  -H -J -B -2 -Z -D   output formatting as in carmel\n"
               "  --train-cascade     train the cascade members, write <file>.trained\n"
               "  --normby=JCN --priors=w,w   per-transducer normalisation / additive priors\n"
               "  --float  fp32 state scores (default fp64)   --scaled  scaled linear space (default log)\n"
               "  --gpu=n  CUDA device   --history=file  --dump-trellis=file  --write-composed=file\n"
               "  --gpus=N examples sharded over GPUs 0..N-1 of this box, one host thread per GPU; the count table is\n"
               "           all-reduced with NCCL every iteration (EM only)\n"
               "  --trellis-only  build (and dump) the derivation lattices on the host, then stop\n"
               "  --fem-forest=f --fem-norm=f --fem-param=f   export the cascade for forest-em(-b200): one derivation forest\n"
               "           per example, normalisation groups, parameters after training (-M -1: the normalised input weights)\n"
               "  --load-fem-param=f  read cascade weights written by --fem-param\n"
               "  --viterbi=file [-k n]  decode only: the n best derivations (default 1) of every training pair, n lines per\n"
               "           example, best first (\"-inf 0 |\" past the last derivation)\n"
               "  --decode=file --given=input|output [-k n]  in place of -t: the corpus file holds one string per line on the\n"
               "           given tape; the n best derivations (default 1) with the other tape free, n lines per string, best\n"
               "           first: the --viterbi line, \" ||\" and the decoded free-tape string (\"-inf 0 | ||\" when there is none)\n"
               "  --sum=file    with --viterbi / --decode: ln of every example's total weight, one line per example or string\n"
               "  --sample=n    with --viterbi / --decode (not -k): n derivations drawn per example or string in proportion to\n"
               "           their weight, seed -R (default 1), in place of the best ones\n";
}

// carmel-b200 --gpus=N ...: N jobs in one process, job r keeps block r of the corpus on GPU r (--shard=r/N --gpu=r); the
// contexts share one NCCL communicator and every iteration all-reduces the count table on the GPUs' own streams.  All
// ranks take the same decisions (the reduced table and likelihood are identical everywhere); rank 0 logs and writes.
static int run_multi_gpu(int argc, char** argv, int n_gpus) {
  for (int i = 1; i < argc; ++i)
    for (const char* d : {"--viterbi", "--decode"})
      if (std::strncmp(argv[i], d, std::strlen(d)) == 0) {
        std::cerr << "ERROR: " << d << " decodes on one GPU (no --gpus)\n";
        return -11;
      }
  unsigned char id[CML_COMM_ID_BYTES];
  if (cml_comm_unique_id(id) != CML_OK) {
    std::cerr << "ERROR: --gpus needs NCCL (libnccl.so.2 could not be loaded)\n";
    return -11;
  }
  std::vector<std::unique_ptr<TrainJob>> jobs;
  std::vector<std::vector<std::string>> args(n_gpus);
  std::ostringstream quiet;
  for (int r = 0; r < n_gpus; ++r) {  // parse / read / compose once per rank (sequentially: the readers share nothing,
    for (int i = 0; i < argc; ++i)     //  but their messages should appear once)
      if (std::strncmp(argv[i], "--gpus", 6) != 0 && std::strncmp(argv[i], "--gpu=", 6) != 0 &&
          !(r > 0 && (std::strncmp(argv[i], "--history", 9) == 0 || std::strncmp(argv[i], "--dump-trellis", 14) == 0)))
        args[r].push_back(argv[i]);
    args[r].push_back("--shard=" + std::to_string(r) + "/" + std::to_string(n_gpus));
    args[r].push_back("--gpu=" + std::to_string(r));
    std::vector<const char*> av;
    for (auto const& a : args[r]) av.push_back(a.c_str());
    jobs.emplace_back(new TrainJob());
    const int rc = open_job((int)av.size(), av.data(), *jobs.back(), r == 0 ? (std::ostream&)std::cerr : (std::ostream&)quiet);
    if (rc != 0) return rc;
    if (jobs.back()->gopt.enabled && !jobs.back()->gopt.batched) {
      std::cerr << "ERROR: --gpus shards EM training and --crp-batched sweeps; the exact --crp sampler is sequential over the "
                   "corpus (one GPU)\n";
      return -11;
    }
    std::memcpy(jobs.back()->comm_id, id, sizeof(id));
    jobs.back()->have_comm_id = true;
  }
  std::vector<std::string> errs(n_gpus);
  std::vector<std::thread> th;
  for (int r = 0; r < n_gpus; ++r)
    th.emplace_back([&, r]() {
      try {
        std::ostringstream sink;
        if (jobs[r]->gopt.enabled)
          jobs[r]->run_gibbs(r == 0 ? (std::ostream&)std::cerr : (std::ostream&)sink);
        else
          jobs[r]->run(r == 0 ? (std::ostream&)std::cerr : (std::ostream&)sink);
      } catch (std::exception& e) {
        errs[r] = e.what();
        if (errs[r].empty()) errs[r] = "failed";
      }
    });
  for (auto& t : th) t.join();
  for (int r = 0; r < n_gpus; ++r)
    if (!errs[r].empty()) {
      std::cerr << "ERROR (GPU " << r << "): " << errs[r] << std::endl;
      return -11;
    }
  jobs[0]->write_outputs(std::cout);
  return 0;
}

int main(int argc, char** argv) {
  try {
    if (argc == 1) {
      usage();
      return 0;
    }
    for (int i = 1; i < argc; ++i)
      if (std::strncmp(argv[i], "--gpus=", 7) == 0 && std::atoi(argv[i] + 7) > 1)
        return run_multi_gpu(argc, argv, std::atoi(argv[i] + 7));
    TrainJob job;
    const int rc = open_job(argc, argv, job, std::cerr);
    if (job.lopt.count("help")) {
      usage();
      return 0;
    }
    if (rc == -9 && job.fst_files.empty()) usage();
    if (rc != 0) return rc;
    if (job.lopt.count("load-fem-param")) {  // carmel.cc:792-800
      std::cerr << "Reading cascade weights from --load-fem-param=" << job.lopt["load-fem-param"] << std::endl;
      job.load_fem_param(job.lopt["load-fem-param"]);
    }
    if (job.lopt.count("decode")) {  // decode new strings, the other tape free
      job.run_decode(std::cerr, job.lopt["decode"]);
      return 0;
    }
    if (job.lopt.count("trellis-only")) {  // host-side lattice construction only (no GPU work): parity tests
      TrellisBatch tb;
      std::vector<uint32_t> dropped;
      size_t e0, e1;  // with --shard=r/N: this rank's block only (what TrainJob::prepare keeps on its GPU)
      shard_range(job.corpus, job.opt.shard_rank, job.opt.shard_count, e0, e1);
      if (job.opt.shard_count > 1) {
        Corpus local;
        local.examples.assign(job.corpus.examples.begin() + e0, job.corpus.examples.begin() + e1);
        job.corpus.examples.swap(local.examples);
        std::cerr << "Shard " << job.opt.shard_rank << "/" << job.opt.shard_count << ": examples [" << e0 << ", " << e1 << ")\n";
      }
      if (job.opt.device_build > 0) {  // --device-build: the same lattices from the GPU builder (cml_build_trellises)
        cml_ctx* bctx = nullptr;
        if (cml_create(&bctx, job.opt.device, 64, CML_SPACE_LOG) != CML_OK)
          throw std::runtime_error(std::string("carmel-b200: ") + cml_last_error(nullptr));
        double secs = 0;
        try {
          build_trellises_device(bctx, *job.x, job.corpus, tb, dropped, &secs);
        } catch (...) {
          cml_destroy(bctx);
          throw;
        }
        cml_destroy(bctx);
        std::cerr << "Device-side lattice construction took " << secs << " s\n";
      } else
        build_trellises(*job.x, job.corpus, tb, dropped);
      uint64_t ns = 0;
      for (uint32_t n : tb.ex_states) ns += n;
      std::cerr << "Built " << tb.ex_states.size() << " derivation lattices (" << ns << " states, " << tb.arc_dst.size()
                << " arcs; " << dropped.size() << " examples without derivations; " << tb.pre_arcs
                << " arcs examined)\n";
      if (!job.opt.dump_trellis_file.empty()) {
        std::ofstream o(job.opt.dump_trellis_file, std::ios::binary);
        tb.dump(o, (uint32_t)job.x->num_arcs());
      }
      return 0;
    }
    if (job.lopt.count("viterbi")) {  // decode only: best derivation of every training pair
      job.run_viterbi(std::cerr, job.lopt["viterbi"]);
      return 0;
    }
    if (job.gopt.enabled)
      job.run_gibbs(std::cerr);
    else
      job.run(std::cerr);
    job.write_outputs(std::cout);
    if (job.lopt.count("fem-norm") || job.lopt.count("fem-param")) job.export_fem_tables(std::cerr);  // carmel.cc:1528 fem_out
    return 0;
  } catch (std::exception& e) {
    std::cerr << "ERROR: " << e.what() << std::endl;
    return -11;
  }
}
