// carmel_host.hpp -- host-side C++ of carmel_b200: the pieces of carmel that stay on the CPU
// (file formats, composition, cascade bookkeeping, per-example lattice construction, the EM
// outer loop) re-designed around flat arrays so that everything numeric is handed to the CUDA
// library through the C ABI (include/carmel_b200.h).  It mirrors the reference's interfaces for
// this path (names, argument meaning, log lines) without sharing its data structures:
//   WFST text format        carmel/src/wfstio.cc:341-506,594-625 ; carmel/doc/FORMATS
//   corpus format           carmel/src/train.cc:985-1025
//   reduce                  carmel/src/fst.cc:468-545
//   composition + chains    carmel/src/compose.cc:163-531 ; carmel/src/cascade.h:489-599
//   lattice construction    carmel/src/derivations.h:479-704
//   EM outer loop           carmel/src/train.cc:503-678
#pragma once
#include <cmath>
#include <cstdint>
#include <iosfwd>
#include <limits>
#include <map>
#include <memory>
#include <random>
#include <string>
#include <unordered_map>
#include <vector>

#include "carmel_b200.h"

namespace cb {

static const double kNegInf = -std::numeric_limits<double>::infinity();
static const uint32_t kNoGroup = CML_NO_GROUP, kLocked = CML_LOCKED_GROUP, kEps = 0;

// ---- weights as natural logs (graehl/shared/weight.h) -------------------------------------------
struct WeightFormat {
  enum Base { EXP, LN, LOG10 } base = EXP;
  enum Thresh { SOMETIMES, ALWAYS, NEVER } thresh = SOMETIMES;
};
bool parse_weight(const char* s, double& ln_out);               // weight.h:503-528
std::string format_weight(double ln_w, WeightFormat const& f = WeightFormat());  // weight.h:467-490
std::string format_base2(double ln_w);                           // Weight::as_base(2), 6 digits
double ln_add(double a, double b);                               // weight.h:765-801 (cutoff 36 nats)
double ln_sub(double a, double b);                               // weight.h:803-830

// ---- alphabet / transducer ----------------------------------------------------------------------
struct Alphabet {
  std::vector<std::string> names;
  std::unordered_map<std::string, uint32_t> idx;
  Alphabet();
  uint32_t index_of(std::string const& s);
  int find(std::string const& s) const;
};

struct Arc {
  uint32_t in, out, dest;
  double ln_w;
  uint32_t group;  // kNoGroup normal, kLocked '!', else tie id '!N'  (cascade composed arcs: chain id)
};

enum NormGroupBy { CONDITIONAL = 0, JOINT = 1, NONE = 2 };
struct NormalizeMethod {
  NormGroupBy group = CONDITIONAL;
  double ln_add_count = kNegInf;  // --priors
};

struct Wfst {
  std::vector<std::vector<Arc>> states;  // arc order within a state = the reference's list order
  std::vector<std::string> state_names;
  std::unordered_map<std::string, uint32_t> state_idx;
  bool named = true;
  uint32_t final_state = 0;
  bool valid = false;
  std::shared_ptr<Alphabet> alph[2];
  Wfst();
  uint32_t num_states() const { return (uint32_t)states.size(); }
  size_t num_arcs() const;
  std::string state_name(uint32_t i) const;
  bool read(std::istream& in, bool always_named = true);
  bool read_file(std::string const& path, bool always_named = true);
  void write(std::ostream& os, bool full, bool one_arc_per_line, bool include_zero, WeightFormat const& wf) const;
  void reduce();
  // arc table: id = visit order (state 0..n, list order) -- carmel/src/fst.h:1330-1334
  void arc_offsets(std::vector<uint32_t>& off) const;
};

struct Example {
  std::vector<uint32_t> in, out;
  double weight = 1;
};
struct Corpus {
  std::vector<Example> examples;
  uint32_t n_pairs = 0;
  double total_weight = 0, n_input = 0, n_output = 0;
  void count();
  void read(std::istream& in, Wfst& x);
  // one string per line (an empty line is the empty string) on tape 0 (input) or 1 (output) of x: the strings
  // --decode reads, kept as examples whose other side is empty
  void read_strings(std::istream& in, Wfst& x, int tape);
};

// ---- cascade: composed arc -> chain of original parameters (cascade.h) --------------------------
struct Cascade {
  bool trivial = true;
  std::vector<Wfst*> members;               // original transducers, in chain order
  std::vector<uint32_t> member_param_base;  // first parameter id of each member
  std::vector<std::vector<uint32_t>> chains;  // chain id -> parameter ids (chain 0 = nil)
  Wfst* composed = nullptr;
  uint32_t n_params = 0;
  // parameter id of (member m, state s, k-th arc)
  std::vector<std::vector<uint32_t>> member_state_base;
  void number_members();
};
// 3-state epsilon-filter composition (compose.cc:316-498).  With a non-trivial cascade the
// composed arcs' group field holds the chain id (cascade.h:588-599).
std::unique_ptr<Wfst> compose(Cascade& c, Wfst& a, Wfst& b, bool a_is_composed, uint32_t a_member, uint32_t b_member,
                              uint32_t index_threshold = 32);

// ---- per-example derivation lattices (derivations.h) --------------------------------------------
struct TrellisBatch {  // the C ABI's cml_trellis_batch, owning its storage; reference state order
  std::vector<uint32_t> ex_states, ex_fin;
  std::vector<double> ex_weight;
  std::vector<uint32_t> arc_off, arc_dst, arc_id;
  std::vector<uint32_t> kept_example;  // index into the corpus of each kept example
  uint64_t pre_arcs = 0;
  void clear();
  void dump(std::ostream& o, uint32_t n_arcs_table) const;
};
// Builds the pruned lattice of every example (string x WFST x string), multi-threaded over
// examples; examples without a derivation are reported in `dropped` and left out.
void build_trellises(Wfst const& x, Corpus const& corpus, TrellisBatch& out, std::vector<uint32_t>& dropped,
                     unsigned n_threads = 0);

// The same, on the GPU (cml_build_trellises): one persistent thread per example walks the reference's DFS.  Chosen by
// --device-build (--host-build, the default, keeps the multi-threaded host builder).
void build_trellises_device(cml_ctx* ctx, Wfst const& x, Corpus const& corpus, TrellisBatch& out, std::vector<uint32_t>& dropped,
                            double* seconds = nullptr);

// Multi-GPU sharding of the E-step (examples are independent given the weights: cached_derivs.h:69-75):
// rank r of n keeps the contiguous block [e0, e1) of the corpus; blocks are balanced by string length
// (1 + |in| + |out| per example), cover the corpus and do not overlap.
void shard_range(Corpus const& corpus, int rank, int count, size_t& e0, size_t& e1);

// ---- training -------------------------------------------------------------------------------------
struct TrainOpts {
  uint32_t max_iter = 500;          // -M   (fst.h:1089)
  double ln_converge_delta;         // -e   (carmel.cc:896) ln(1e-4)
  double ln_converge_ratio;         // -X   (carmel.cc:897) ln(.999)
  double ln_smooth_floor = kNegInf; // -f
  bool weight_is_prior = false;     // -U
  double rate_growth = 1.;          // -o
  int precision = 64;               // --float => 32
  int space = CML_SPACE_LOG;        // --scaled => CML_SPACE_SCALED
  int device = 0;                   // --gpu=n
  int shard_rank = 0, shard_count = 1;  // --shard=r/N : this process trains on block r of N of the corpus
  bool quiet = false;
  bool no_ell = false;              // --no-ell : general (layered CSR) kernels only
  int lane_min = -1;                // --lane-min=n / --no-lane : CML_OPT_LANE_MIN (-1 = library default)
  bool no_factor = false;           // --no-factor : one weight-table entry per arc (CML_OPT_NO_FACTOR)
  bool no_wide = false;             // --no-wide : wide lattices stay on the k_fb_ell classes (CML_OPT_NO_WIDE)
  int device_build = 0;             // lattice construction: 0 / --host-build -1: host threads; --device-build 1: cml_build_trellises
  int dense = 0;                    // dense-state path: 0 auto (when the model has the view), --no-dense -1, --dense 1 (required)
  std::string history_file, dump_trellis_file;
  uint32_t ran_restarts = 0;        // -! n : additional random starts (train.cc:553-667)
  uint32_t final_restart = 0;       // --final-restart=N : restart index at which the tolerance reaches its final value
  double ln_restart_tolerance = kNegInf, ln_final_restart_tolerance = kNegInf;  // --restart-tolerance= --final-restart-tolerance= (none: accept all)
  uint64_t seed = 1;                // -R seed : the restarts' generator (the reference seeds boost's lagged Fibonacci; draws differ)
  std::string kbest_arg;            // -k n : derivations per example written by --viterbi (unused when training)
  uint32_t kbest = 1;
  int given_tape = -1;              // --given=input|output : the tape --decode reads its strings on (0 / 1)
  uint32_t sample = 0;              // --sample=n : with --viterbi / --decode, n derivations drawn per example (seed -R)
  std::string sum_file;             // --sum=FILE : with --viterbi / --decode, ln of every example's total weight
  TrainOpts();
};
// WFST::random_restart_acceptor (fst.h:999-1044): a further start must be, after its first iteration, within a
// tolerance of the first start's first iteration
struct RestartAcceptor {
  double ln_best_start = 0, ln_tolerance, ln_final_tolerance, n;
  RestartAcceptor(double final_at_n, double ln_tol, double ln_final_tol);
  double ln_likelihood_ratio(uint32_t i) const;
  bool accept(double ln_this_start, uint32_t restart_i, std::ostream& o);
};
struct IterRecord {
  uint32_t iter;
  double ln_prob, ln_weighted_prob, max_change;
};
struct TrainResult {
  double ln_best_ppx = 0;
  std::vector<IterRecord> history;
  uint64_t trellis_arcs = 0, trellis_states = 0, examples = 0;  // resident on this GPU
  double device_build_s = 0;  // > 0: lattices built by cml_build_trellises in this many seconds
  bool dense = false;  // the E-step runs on the dense-state view (no lattices materialised)
};
// The device model: parameters = all arcs of the cascade members (or of x) in arc-table order.
struct ModelArrays {
  std::vector<uint32_t> chain_off, chain_param, param_group, param_tie;
  std::vector<double> group_add, ln_w, arc_prior;
  std::vector<uint64_t> arc_key;
  uint32_t n_groups = 0, n_ties = 0, n_arcs = 0, n_params = 0;
};
// --crp options (graehl/shared/gibbs_opts.hpp:34-130, defaults :213-252)
struct GibbsOpts {
  bool enabled = false;
  uint32_t iter = 0, burnin = 0;     // --crp[=n] / -M n ; --burnin=n
  bool uniform_p0 = false, dirichlet_p0 = false, final_counts = false, exclude_prior = false;
  double high_temp = 1, low_temp = 1;  // --high-temp= --low-temp=
  uint64_t seed = 1;                 // --seed= : key of the counter-based uniforms
  bool batched = false;              // --crp-batched : all blocks in parallel against the previous sweep's counts
  bool expectation = false;          // --expectation (gibbs.cc:311-316): blocks carry posteriors of all their arcs (incremental EM)
  bool sample_prob = false;          // --sample-prob (carmel.cc:1869): log the proposal probability of each new sample given
                                     // the counts without its block (gibbs.hpp:866 with cache_prob off) instead of the cache
                                     // model's -- the quantity in the golden log commands.trace:6976-12996
  std::string dump_samples_file;     // --dump-samples=file : final sample, arc-table ids per block
};
// sum-all-reduce of n doubles at device_ptr across the ranks of a multi-GPU run (NCCL, supplied by the driver)
typedef void (*AllReduceFn)(void* user, void* device_ptr, uint64_t n_doubles);

// One training run = the reference's `carmel -t ...` invocation: WFST::train (train.cc:503-678) with the
// E- and M-steps on the GPU.  After run() the cascade members (or x for a trivial cascade) hold the
// trained weights.  Methods throw std::runtime_error.
struct TrainJob {
  // inputs (filled by open_job or by the caller)
  std::vector<std::string> fst_files;
  std::string corpus_file, outfile;
  std::vector<std::unique_ptr<Wfst>> chain, composed_keep;
  Wfst* x = nullptr;  // the (composed) transducer being trained
  Cascade cascade;
  Corpus corpus;
  std::vector<NormalizeMethod> methods;
  TrainOpts opt;
  GibbsOpts gopt;
  bool flags[256] = {false};
  std::map<std::string, std::string> lopt;
  bool train_cascade = false;
  AllReduceFn allreduce = nullptr;
  void* allreduce_user = nullptr;
  // NCCL rendezvous token of a sharded run (cml_job_set_comm): the context joins the communicator in prepare() and
  // the per-iteration all-reduce is issued by the library on its own stream (no callback)
  bool have_comm_id = false;
  unsigned char comm_id[128] = {0};
  // state
  cml_ctx* ctx = nullptr;
  ModelArrays M;
  std::vector<Wfst*> members;
  bool using_cascade = false, prepared = false;
  TrainResult res;
  std::vector<uint32_t> kept_example;  // prepare(): corpus index of each resident lattice
  uint64_t corpus_size = 0;            // prepare(): examples read, with or without a derivation

  ~TrainJob();
  void build_model();  // parameters, chains, normalisation groups (host only; fem.cpp)
  void export_fem_tables(std::ostream& log);        // --fem-norm / --fem-param, after training (fem.cpp)
  void export_fem_forest(TrellisBatch const& tb, std::ostream& log);  // --fem-forest, from prepare()
  void load_fem_param(std::string const& file);     // --load-fem-param
  void prepare_model();  // context, model, parameters after the initial normalisation (the first part of prepare)
  void prepare();
  bool try_dense(int tape, Corpus const& local, std::vector<uint32_t>& kept, std::vector<uint32_t>& dropped);
  double estimate(double& ln_unweighted);
  TrainResult const& run(std::ostream& log);        // EM (WFST::train)
  TrainResult const& run_gibbs(std::ostream& log);  // --crp (WFST::train_gibbs)
  void prepare_gibbs();
  // --viterbi=FILE (decode.cpp): the best derivation of every training pair under the (normalised) model as given, one
  // line per kept example: ln weight, number of arcs, arc-table ids; then, per arc, the (input:output) labels of the
  // cascade members' arcs it stands for (decode side: carmel -k 1 on the composed machine, fst.h:769-800).  With -k n,
  // n lines per kept example.  With --sample=n the file holds n derivations drawn per example instead, in corpus order
  // (examples without a derivation included); with --sum=FILE that file gets ln of every example's total weight.
  void run_viterbi(std::ostream& log, std::string const& path);
  // --decode=FILE --given=input|output (decode.cpp): the -k n best derivations of every string of the corpus file on the
  // given tape with the other tape free (carmel -sri / -sli ... -k n), n lines per string in file order: the --viterbi
  // line, then " ||" and the free-tape labels of the path; "-inf 0 | ||" past the last derivation or for a string
  // without one
  void run_decode(std::ostream& log, std::string const& path);
  void attach_dense_sampler();  // batched --crp on position-synchronous lattices: cml_gibbs_attach_dense  // lattices + CRP parameters on the GPU, counts = priors; no sweep yet
  bool gibbs_prepared = false;
  std::vector<uint32_t> g_norm;  // CRP normalisation group of every parameter (kNoGroup = fixed probability)
  std::vector<double> g_prior;   // pseudo-count (or the fixed probability)
  std::vector<uint64_t> g_base;  // sample slot base of every resident example
  uint32_t g_n_norms = 0;
  void write_back();
  void random_restart(std::mt19937_64& rng);
  void write_outputs(std::ostream& out);  // trained transducer(s) as carmel writes them
  void finish();
  void ok(int rc) const;
};
void add_model_member(Wfst const& w, NormalizeMethod const& m, ModelArrays& M);  // train.cpp
// Parse carmel's argv grammar (carmel.cc:929-1066), read the transducers, reduce / compose them and read the
// corpus.  Returns carmel's exit code (0 = ready to train); messages go to `err`.
int open_job(int argc, const char* const* argv, TrainJob& job, std::ostream& err);

}  // namespace cb
