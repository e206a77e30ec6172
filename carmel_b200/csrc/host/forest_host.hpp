// forest_host.hpp -- host side of the forest-em path: file formats, options and the EM driver
// (overrelaxed_em), with everything numeric handed to the CUDA library through the C ABI
// (include/carmel_b200.h, cml_forests_*).  Mirrors, without sharing data structures:
//   forests  "(OR #1(1 2) #1 (3 4))"     forest-em/forest.hpp:39-46,135-242 (reader), :245-320 (printer)
//   normalization groups "((1 2) (3 4))"  graehl/shared/normalize.hpp:58-65
//   parameters, one weight per line       forest-em/forest-em.hpp:190-201,228-250
//   options                               forest-em/forest-em-params.hpp:69-176
//   EM driver                             graehl/shared/em.hpp:107-216 ; forest-em/forest-em.hpp:556-655
#pragma once
#include <cstdint>
#include <iosfwd>
#include <map>
#include <random>
#include <string>
#include <vector>

#include "carmel_b200.h"

namespace cb {

// all forests of a corpus in the C ABI's layout (cml_forest_batch): pre-order node arrays, back to back
struct ForestSet {
  std::vector<uint64_t> node_off{0};
  std::vector<uint32_t> next, label;
  std::vector<uint8_t> backref;
  uint64_t max_ruleid = 0, max_nodes = 0;
  uint64_t size() const { return node_off.size() - 1; }
  uint64_t n_nodes() const { return next.size(); }
  // parses forests until the end of the buffer; throws std::runtime_error with the forest number on errors
  void read(const char* begin, const char* end);
  void print(std::ostream& o, uint64_t f) const;
};

struct NormGroupsHost {
  std::vector<uint64_t> off{0}, members;
  uint64_t max_index = 0;
  uint64_t size() const { return off.size() - 1; }
  // parses "((1 2) (3))" and returns the position after the closing paren
  const char* read(const char* begin, const char* end);
};

struct ForestOpts {
  std::string forests_file, normgroups_file, initparam_file, outparam_file, outcounts_file, outinside_file, history_file,
      print_forests_file, outviterbi_file;  // -v : 'best/sum=pct% <viterbi derivation>' per forest (forest-em-params.hpp:115)
  unsigned max_iter = 1000;            // -i  (forest-em-params.hpp:185)
  double converge_ratio = 1. / 65536;  // -e  (:186)
  double converge_delta = 0;           // -d  (:187)
  double prior_counts = 0;             // -p
  double add_k_smoothing = 0;          // -k
  bool zero_zerocounts = false;        // -z
  bool initial_1_params = false;       // -u
  bool normalize_initial = false;      // -N
  bool double_precision = false;       // -U
  bool human_probs = false;            // -H
  unsigned log_level = 1;              // -L
  unsigned random_restarts = 0;        // -r  (forest-em-params.hpp:103): further starts from random parameters
  uint64_t random_seed = 1;            // -s  : the restarts' generator (draws differ from the reference's)
  int device = 0;                      // --gpu=n
  int shard_rank = 0, shard_count = 1;  // --shard=r/N
  int layout = CML_FOREST_LAYOUT_AUTO;  // --layout=auto|group|thread|level (device layout family, see cml_forests_set_layout)
  uint32_t kbest = 1;                  // --kbest=n : -v writes the n best derivations per forest (cml_forests_kbest)
  uint32_t sample = 0;                 // --sample=n : -v writes n drawn derivations per forest instead (cml_forests_sample)
  bool parse_only = false;            // --parse-only : read (and --print-forests) without touching the GPU
  // checkpoints (forest-em.hpp:166-201,621-641; forest-em-params.hpp:138-145): on every "watch" iteration (the first
  // watch_period iterations, then every watch_period-th) write <prefix>.params / <prefix>.counts
  // .restart.R.iteration.I; a run is resumed by passing a params checkpoint as -I
  // --crp=n Gibbs sampling instead of EM (gibbs_opts.hpp:34-130 via forest-em-params.hpp:172-175)
  unsigned crp_iter = 0, crp_burnin = 0;
  double crp_alpha = .1;               // --const-alpha (gibbs_opts.hpp:229): prior = alpha * p0 * |group|
  bool crp_uniform_p0 = false, crp_final_counts = false, crp_exclude_prior = false, crp_sample_prob = false, crp_batched = false;
  double crp_high_temp = 1, crp_low_temp = 1, crp_n_sym = 0;
  uint64_t crp_seed = 1;               // --seed : seed of the counter-based uniforms (--crp, --sample)
  std::string outsample_file;          // --outsample-file : the final sample, rule ids in record order, one forest per line
  unsigned watch_period = 10;          // -W
  std::string checkpoint_prefix;       // -x
  bool checkpoint_parameters = false;  // -c
};

struct ForestIter {
  unsigned iter;
  double avg_logprob, max_delta;
  uint64_t max_index, n;
};

typedef void (*ForestAllReduceFn)(void* user, void* device_ptr, uint64_t n_doubles);

struct ForestJob {
  ForestOpts opt;
  ForestSet forests;
  NormGroupsHost groups;
  std::vector<double> ln_w;  // [rulespace]; index 0 unused
  bool have_init_params = false;
  uint64_t rulespace = 0, count_space = 0;
  uint64_t total_forests = 0;  // whole corpus (all shards)
  uint64_t shard_begin = 0, shard_end = 0;
  ForestAllReduceFn allreduce = nullptr;
  void* allreduce_user = nullptr;
  bool have_comm_id = false;          // NCCL rendezvous token (cml_forest_job_set_comm / forest-em-b200 --gpus=N): the
  unsigned char comm_id[128] = {0};   // library issues the per-iteration all-reduce itself
  cml_forests* ctx = nullptr;
  bool prepared = false, firsttime = true, gibbs_done = false;
  unsigned iteration = 0, restart = 0;  // maximize() calls so far / current random restart (checkpoint names)
  void write_params_to(std::ostream& o);
  void write_counts_to(std::ostream& o);
  std::vector<ForestIter> history;
  double best_alp = 0;
  uint64_t last_n_zero = 0;

  ~ForestJob();
  void load();     // read the files named in opt
  void compute_shard();  // [shard_begin, shard_end) from opt.shard_rank / opt.shard_count
  void prepare();  // rules, parameters and this shard's forests onto the GPU
  double estimate(bool first_time, std::ostream& log, uint64_t* n_used = nullptr);
  void maximize(std::ostream& log, double& max_delta, uint64_t& max_index);
  double run(std::ostream& log);  // overrelaxed_em
  void run_gibbs(std::ostream& log);  // --crp (forest-em.hpp:694-797)
  void randomize(std::mt19937_64& rng);
  void write_outputs(std::ostream& log);
  void ok(int rc) const;
};
// forest-em's argv (the training subset); returns 0 or forest-em's exit code 1 with the message on `err`
int open_forest_job(int argc, const char* const* argv, ForestJob& job, std::ostream& err);

}  // namespace cb
