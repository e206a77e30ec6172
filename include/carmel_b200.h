/* carmel_b200.h -- C ABI of the B200-native training hot path for graehl/carmel.
 *
 * The reference (graehl/carmel) has no plugin / FFI surface: carmel and forest-em are single
 * binaries.  This header is the seam a maintainer would bind if the reference's executor concepts
 * were moved behind a library: each entry point names the reference interface it replaces
 * (file:line relative to the reference root).  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions
 *   - every function returns 0 on success, a negative cml_status on failure; cml_last_error()
 *     gives the message.  No exception crosses the boundary.
 *   - host buffers belong to the caller; device memory belongs to the context.
 *   - one context per GPU; a context is not thread-safe, different contexts are independent
 *     (the reference itself is single threaded with static state, forest-em/forest.hpp:86-107).
 *   - weights cross the boundary as natural logs of non-negative reals (the reference's
 *     logweight<Real>::weight, graehl/shared/weight.h:131-137); -INFINITY is the zero weight.
 *   - there is NO CPU fallback: every compute entry point fails with CML_ERR_CUDA when no
 *     sm_100 device is usable.
 */
#ifndef CARMEL_B200_H
#define CARMEL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cml_ctx cml_ctx;

enum cml_status {
  CML_OK = 0,
  CML_ERR_ARG = -1,    /* bad argument / inconsistent sizes */
  CML_ERR_CUDA = -2,   /* CUDA runtime error or no usable device */
  CML_ERR_STATE = -3,  /* call order violated (e.g. estimate before set_model) */
  CML_ERR_CYCLE = -4,  /* a forest's back references form a cycle; Gibbs sampling over a lattice with a cycle */
  CML_ERR_NODERIV = -5, /* no training example had a derivation (train.cc:249-252) */
  CML_ERR_NOT_DENSE = -6 /* cml_add_sequences: the arc table has no transition x emission factorisation
                            (or too many states); nothing was changed, use cml_add_trellises instead */
};

enum cml_space { CML_SPACE_LOG = 0, CML_SPACE_SCALED = 1 };
enum cml_norm_group { CML_NORM_CONDITIONAL = 0, CML_NORM_JOINT = 1, CML_NORM_NONE = 2 };

#define CML_NO_GROUP 0xFFFFFFFFu /* graehl/shared/arc.h:43 FSTArc::no_group  */
#define CML_LOCKED_GROUP 0u      /* graehl/shared/arc.h:44 FSTArc::locked_group */

/* ---- library / context ------------------------------------------------------------------- */
const char* cml_version(void);
/* precision: 32 or 64 = sizeof(Real)*8 of the forward/backward state scores (carmel FLOAT_TYPE,
 * graehl/shared/config.h:98-104; forest-em -U, forest-em-params.cpp:9-19).  Counts, likelihood sums
 * and the M-step are always fp64. */
int cml_create(cml_ctx** out, int device, int precision, int space);
void cml_destroy(cml_ctx* ctx);
const char* cml_last_error(cml_ctx* ctx); /* ctx may be NULL: error of the last failed cml_create */
/* run all subsequent work of this context on an existing CUDA stream (cudaStream_t as void*). */
int cml_set_stream(cml_ctx* ctx, void* cuda_stream);
int cml_synchronize(cml_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t cml_launch_count(cml_ctx* ctx);

/* options (cml_set_option) */
enum cml_option {
  CML_OPT_ARC_COUNTS = 1, /* keep one expected-count accumulator per arc-table entry (needed by
                             cml_get_arc_counts on real cascades); default 0: arcs whose chains have the same
                             unlocked parameters share an accumulator.  Set before cml_set_model. */
  CML_OPT_NO_ELL = 2,     /* force the layered-CSR kernels (tests).  Set before cml_add_trellises. */
  CML_OPT_LANE_MIN = 3,   /* the lane-per-lattice kernel (narrow lattices, tiles of 32) is used when a batch has at
                             least this many eligible lattices; default 16384, 0 = never.  Before cml_add_trellises. */
  CML_OPT_NO_COUNTS = 4,  /* profiling only: the wide / lane kernels skip their expected-count REDs */
  CML_OPT_NO_FACTOR = 5,  /* keep one weight-table entry per arc: no arc classes / state parts (see DESIGN.md 3.2).
                             Set before cml_set_model. */
  CML_OPT_NO_WIDE = 6,    /* lattices with levels of 9..32 states stay on the k_fb_ell classes instead of the
                             warp-per-lattice kernel (tests).  Set before cml_add_trellises. */
  CML_OPT_ALLOW_EMPTY = 7, /* a rank of a sharded job whose block holds no usable example still takes part in every
                             collective: its E-step contributes zeros instead of failing with CML_ERR_NODERIV */
  CML_OPT_NO_GRAPH = 8,   /* cml_em_step enqueues its launches one by one instead of replaying a CUDA graph */
  CML_OPT_KBEST_SCRATCH_MB = 9, /* device scratch budget (MiB) of one cml_kbest or cml_sample chunk; default 4096 */
  CML_OPT_FREE_BUILD_SCRATCH_MB = 10 /* device scratch budget (MiB) of one cml_build_free_trellises chunk; default 4096 */
};
int cml_set_option(cml_ctx* ctx, int option, int value);

/* ---- model: parameters, cascade chains, normalisation groups ------------------------------ *
 * Replaces arcs_table<arc_counts> (carmel/src/derivations.h:79-140, train.h:28-40),
 * cascade_parameters::chains (carmel/src/cascade.h:222-262) and the group structure walked by
 * WFST::normalize / NormGroupIter (carmel/src/fst.cc:86-244, fst.h:1362-1446).
 *
 *   n_arcs      size of the arc table the trellis arc ids index (composed transducer arcs).
 *   chain_off   [n_arcs+1] CSR into chain_param: the parameters whose product is the arc's weight
 *               (cascade.h:426-433).  NULL = trivial cascade: arc i is parameter i (n_params==n_arcs).
 *   arc_prior   [n_arcs] linear prior count added to the arc's expected count before the M-step
 *               (train.cc:134-153 prior_counts; -f floor, + weight with -U).  NULL = all 0.
 *   n_params    number of original (cascade member) arcs = trainable or locked parameters.
 *   param_group [n_params] normalisation group id in [0,n_groups) or CML_NO_GROUP for members of a
 *               NONE-normalised transducer (weights kept, cascade.h:339-350).
 *   param_tie   [n_params] CML_NO_GROUP (normal), CML_LOCKED_GROUP (locked '!'), else tie id in
 *               [1,n_ties] ('!N', wfstio.cc:453-464; ids are made dense and unique per cascade by the caller).
 *   group_add   [n_groups] ln of the per-group additive prior (--priors, fst.cc:124-125); NULL = zero.
 */
typedef struct cml_model {
  uint32_t n_arcs;
  const uint32_t* chain_off;
  const uint32_t* chain_param;
  const double* arc_prior;
  uint32_t n_params;
  const uint32_t* param_group;
  const uint32_t* param_tie;
  uint32_t n_groups;
  const double* group_add;
  uint32_t n_ties;
  /* optional [n_arcs]: arcs with nearby keys are used together (e.g. output symbol, then destination, then
   * source state); the library lays its weight tables out in key order so gathers of one lattice level share
   * cache sectors.  Must be the same on every rank of a multi-GPU job.  NULL = arc-table order. */
  const uint64_t* arc_locality_key;
} cml_model;
int cml_set_model(cml_ctx* ctx, const cml_model* m);
/* ln weights of the n_params parameters: FSTArc::weight (arc.h:37) */
int cml_set_params(cml_ctx* ctx, const double* ln_w);
int cml_get_params(cml_ctx* ctx, double* ln_w);
/* device-side copies used for save_best / load_best (train.cc:449-457, for_arcs::save_best :184-197) */
int cml_snapshot_params(cml_ctx* ctx, int slot /*0..3*/);
int cml_restore_params(cml_ctx* ctx, int slot);

/* ---- trellises ------------------------------------------------------------------------------ *
 * Replaces derivations::g (carmel/src/derivations.h:170-171) = dynamic_array<GraphState> of
 * List<GraphArc{src,dest,weight,data=arc id}> (graehl/shared/graph.h:37-121) together with the
 * per-example DFS order and reversed graph (derivations.h:706-736, graph.cc:41-57).
 * The caller hands over each example's pruned derivation lattice exactly as the reference holds
 * it: states in reference id order (DFS pre-order after prune, start = 0), per state its arc list in
 * stored order (derivations.h:698 push_front => reverse discovery order).  The library flattens
 * the batch into topologically layered CSR arrays in HBM (states renumbered by (level, id), level =
 * longest-path depth from the start; incoming- and outgoing-arc CSR per example) and keeps it
 * resident across iterations like carmel's in-memory derivation cache (-: , cached_derivs.h:104-138).
 *
 *   n_ex       examples in this batch (appended to those already resident)
 *   ex_states  [n_ex] states per example        ex_fin [n_ex] goal state id
 *   ex_weight  [n_ex] example weight (train.h IOSymSeq::weight)
 *   arc_off    [sum(ex_states) + n_ex] per example a CSR row-offset array of ex_states+1 entries,
 *              offsets local to the example's first arc
 *   arc_dst, arc_id [total arcs] destination state id and arc-table id (GraphArc.dest / .data)
 * A lattice with a cycle (an *e*:*e* loop in the transducer) is accepted like the reference accepts it
 * (derivations.h:722-729 "Warning: at least one cycle in derivations ... Forward/backward will miss some paths"):
 * it is walked in the reference's DFS order by a sequential kernel, back-edge contributions arriving after their
 * destination has been propagated, so likelihood and counts equal the reference's; cml_cyclic_stats reports how many
 * such lattices / back edges are resident (the caller prints the warning).  Only the Gibbs sampler refuses them. */
typedef struct cml_trellis_batch {
  uint64_t n_ex;
  const uint32_t* ex_states;
  const uint32_t* ex_fin;
  const double* ex_weight;
  const uint32_t* arc_off;
  const uint32_t* arc_dst;
  const uint32_t* arc_id;
} cml_trellis_batch;
int cml_add_trellises(cml_ctx* ctx, const cml_trellis_batch* b);
int cml_clear_trellises(cml_ctx* ctx);

/* ---- device-side lattice construction ------------------------------------------------------------- *
 * Replaces derivations::compute (carmel/src/derivations.h:479-513: derive :640-676, add_arcs :678-704, prune
 * :572-629) for a whole corpus: the intersection  input string x transducer x output string  of every example,
 * built on the GPU (one persistent thread per example walks the reference's DFS with an explicit stack; cml_build.cu)
 * and returned in HOST memory in exactly the form cml_add_trellises takes -- reference state ids (DFS pre-order after
 * pruning), stored arc order, arc-table ids -- so the result is interchangeable with a host-built batch, byte for byte.
 * Examples without a derivation are left out and listed in `dropped` (cached_derivs.h:87-93).
 *   transducer: arc table in arc-table order (fst.h:1330-1334), state s owns arcs [state_arc_off[s], state_arc_off[s+1]);
 *               symbol 0 = *e* on either tape
 *   corpus:     example e = (in_sym[in_off[e] .. in_off[e+1]), out_sym[out_off[e] .. out_off[e+1])), weight[e] (NULL = 1) */
typedef struct cml_wfst_view {
  uint32_t n_states, final_state;
  uint64_t n_arcs;
  const uint32_t* state_arc_off; /* [n_states + 1] */
  const uint32_t* arc_in;        /* [n_arcs] */
  const uint32_t* arc_out;
  const uint32_t* arc_dest;
} cml_wfst_view;
typedef struct cml_corpus_view {
  uint64_t n_ex;
  const uint64_t* in_off;  /* [n_ex + 1] */
  const uint32_t* in_sym;
  const uint64_t* out_off; /* [n_ex + 1] */
  const uint32_t* out_sym;
  const double* weight;    /* [n_ex] or NULL */
} cml_corpus_view;
typedef struct cml_built_trellises {
  cml_trellis_batch batch;       /* the kept examples, corpus order; pointers owned by this object */
  const uint32_t* kept_example;  /* [batch.n_ex] corpus index of each kept example */
  uint64_t n_dropped;
  const uint32_t* dropped;       /* corpus indices of the examples without a derivation */
  uint64_t pre_arcs;             /* transducer arcs examined (the reference's "derivations pre-prune" figure) */
  uint32_t launches;             /* kernel launches (capacity rounds of the sizing pass + the fill pass) */
  uint32_t peak_states, peak_kept_arcs, peak_depth; /* largest walk: states / kept arcs before pruning, DFS depth */
  double seconds;                /* wall time of the call (index, upload, both passes, download) */
  uint64_t chunks;               /* cml_build_free_trellises: chunks of strings processed (0 for cml_build_trellises) */
  double kernel_ms;              /* cml_build_free_trellises: time of its k_build_free launches, CUDA events (0 otherwise) */
  void* owner;
} cml_built_trellises;
int cml_build_trellises(cml_ctx* ctx, const cml_wfst_view* x, const cml_corpus_view* c, cml_built_trellises** out);
void cml_free_built_trellises(cml_built_trellises* b);
/* ---- lattices of one given string, the other tape free (carmel -sri / -sli ... -k n: decode new strings) ---------- *
 * The lattice of  string s on tape g  x  transducer x, with the other tape free:
 *   x        the composed machine's arc table as a cml_wfst_view (arc-table order, symbol 0 = *e*, start = state 0)
 *   g        the given tape: 0 = input, 1 = output
 *   s        symbol ids on tape g
 * States     pairs (q, t) of a machine state q and a position t in [0, |s|], kept when reachable from (0, 0) and
 *            co-reachable to (final_state, |s|).
 * Arcs       machine arc a of q leads from (q, t) to (dest, t) when its tape-g label is *e*, and to (dest, t + 1) when
 *            that label equals s[t] (a symbol 0 in s matches no arc).  Its label on the free tape is not looked at.
 * eps-level  of a machine state: its longest-path depth in the subgraph of the arcs with *e* on tape g.  When that
 *            subgraph has a cycle the call fails with CML_ERR_CYCLE before any device work (such a model has strings
 *            with unboundedly many derivations, and the decoders need acyclic lattices).
 * Numbering  kept states are numbered in the order (t, eps-level(q), q): (0, 0) is state 0 and (final, |s|) the last
 *            state (ex_fin = ex_states - 1); each state's out-arcs are its kept arcs in arc-table order; arc_id is the
 *            machine arc id, as cml_add_trellises and the weights expect.
 * Strings without a derivation (the empty lattice, symbols the tape never uses, ids out of range) are left out and
 * listed in `dropped`; kept_example gives the string index of each kept lattice.  ex_weight is 1.
 * The result is host memory in the form cml_add_trellises takes (release it with cml_free_built_trellises).  Of the
 * statistics, `launches`, `peak_states` / `peak_kept_arcs` (the largest kept lattice), `seconds`, `chunks` and
 * `kernel_ms` are filled in; `pre_arcs` and `peak_depth` are 0.
 * GPU work: kernel k_build_free, one warp per string: reachability forward and co-reachability backward over the
 * positions, the eps-levels of one position in order and the states of one eps-level across the lanes; then a counting
 * pass, an exclusive scan on the host and a fill pass.  Device scratch is 6 B per (position, machine state) cell;
 * strings are processed in chunks of consecutive strings whose scratch fits CML_OPT_FREE_BUILD_SCRATCH_MB (a string
 * larger than that gets a chunk of its own).  Results do not depend on the chunking.
 * Errors: CML_ERR_ARG for a null pointer, a tape other than 0 / 1, an incomplete or inconsistent transducer view,
 * string offsets that do not start at 0 or decrease, or a string s with (|s| + 1) * n_states or (|s| + 1) * n_arcs of
 * 2^32 or more (the bounds of its lattice's states and arcs, which are counted in 32 bits); CML_ERR_CYCLE as above. */
typedef struct cml_string_batch {
  uint64_t n;           /* strings */
  const uint64_t* off;  /* [n + 1] string i is sym[off[i] .. off[i + 1]) */
  const uint32_t* sym;
} cml_string_batch;
int cml_build_free_trellises(cml_ctx* ctx, const cml_wfst_view* x, const cml_string_batch* s, int given_tape,
                             cml_built_trellises** out);
int cml_trellis_totals(cml_ctx* ctx, uint64_t* n_ex, uint64_t* n_states, uint64_t* n_arcs, uint64_t* n_levels);
int cml_cyclic_stats(cml_ctx* ctx, uint64_t* n_examples, uint64_t* n_back_edges);
/* Best derivation of every resident lattice at the current parameters -- the decode carmel does with `-k 1` on the
 * composed  string x transducer x string  machine (fst.h:769-800 bestPaths, graehl/shared/kbest.h): max-plus forward
 * pass over the layered CSR (states in topological order, out-arcs in the reference's stored order, a destination takes
 * a new best only on a strict improvement), then the walk back from the goal.  Among derivations of exactly equal
 * weight (the same arcs in another order) the one found first in that order is reported.  Needs an fp64 CML_SPACE_LOG context
 * whose lattices are all in the layered-CSR layout (CML_OPT_NO_ELL), like the samplers.  cml_viterbi and cml_kbest are
 * in cml_decode.cu, cml_sample in cml_sample.cu.
 *   path_len[n_ex]       arcs of example e's best derivation (0: none)
 *   path_base[n_ex + 1]  example e's arcs are path_arcs[path_base[e] .. path_base[e] + path_len[e])
 *   path_arcs[cap]       arc-table ids in path order; cap >= the total number of lattice levels (cml_trellis_totals)
 *   ln_weight[n_ex]      ln of the derivation's weight (-inf: none) */
int cml_viterbi(cml_ctx* ctx, uint32_t* path_len, uint64_t* path_base, uint32_t* path_arcs, uint64_t cap, double* ln_weight);
/* The k best derivations of every resident lattice, best first -- carmel's `-k n` on the composed
 * string x transducer x string machine (graehl/shared/kbest.h).  Same preconditions and errors as cml_viterbi, and
 * CML_ERR_ARG for k == 0 or a path_arcs buffer that is too small.
 *   path_len[n_ex * k]       arcs of derivation (e, r) at [e * k + r]; 0 = no such derivation
 *   path_base[n_ex * k + 1]  derivation (e, r) is path_arcs[path_base[e * k + r] .. + path_len[e * k + r])
 *   path_arcs[cap]           arc-table ids in path order, or NULL for weights only; cap >= k * the total number of
 *                            lattice levels (cml_trellis_totals)
 *   ln_weight[n_ex * k]      ln weight of derivation (e, r); -inf where example e has fewer than r + 1 derivations
 * Contract:
 *   order       example e's derivations come in non-increasing ln weight
 *   distinct    they are distinct lattice paths (in a string x transducer x string lattice: distinct arc-id sequences)
 *   zero weight derivations of weight zero (ln -inf) are never listed; a -inf entry has path_len 0
 *   ties        a state's list is the top k of (source list entry + arc weight) over its in-arcs; among candidates of
 *               exactly equal score the one earlier in the state's in-list (sorted by source layered index, then the
 *               source's stored out-arc order) comes first, then the lower source rank
 *   rank 0      is bit-identical to cml_viterbi: same double, same arc ids
 *   determinism the same inputs give the same bytes on every run
 *   memory      device scratch of about 16 B * k per lattice state plus 4 B per state and per lattice arc; the
 *               lattices are processed in chunks of consecutive lattices whose scratch fits CML_OPT_KBEST_SCRATCH_MB
 *               (a lattice larger than that gets a chunk of its own).  Results do not depend on the chunking. */
int cml_kbest(cml_ctx* ctx, uint32_t k, uint32_t* path_len, uint64_t* path_base, uint32_t* path_arcs, uint64_t cap,
              double* ln_weight);
/* the last cml_kbest / cml_viterbi call: device scratch bytes of its largest chunk, number of chunks, and the time of
 * its derivation kernels from CUDA events (ms) */
int cml_kbest_stats(cml_ctx* ctx, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms);
/* The total weight of every resident lattice, and n derivations of each drawn in proportion to their weight,
 * P(d | lattice) = w(d) / sum of w over its derivations.  Same preconditions and errors as cml_kbest (an fp64
 * CML_SPACE_LOG context whose lattices are all in the layered-CSR layout; CML_ERR_CYCLE for a lattice with a cycle), and
 * CML_ERR_ARG for a cap below n * the total number of lattice levels, a null ln_total, or n > 0 with a null output.
 *   ln_total[n_ex]          beta(start) of lattice e, where beta(s) = ln of the sum over the paths s -> goal of the
 *                           product of their arc weights: fp64, a max-shifted log-sum-exp over each state's out-arcs;
 *                           -inf when the lattice has no derivation of non-zero weight
 *   n = 0                   computes ln_total only; ex_key and the path arrays may then be null
 *   ex_key[n_ex]            the key of lattice e's uniforms, or null for key = e
 *   path_len, path_base, path_arcs, cap
 *                           as in cml_kbest with k = n: sample r of lattice e is path_arcs[path_base[e * n + r] ..
 *                           + path_len[e * n + r]), arc-table ids in path order
 *   ln_weight[n_ex * n]     the sum of the sample's arc ln weights, in path order
 * Sample r of lattice e walks from the start state to the goal.  At step t (0, 1, ...) it draws
 *   u = sample_uniform(seed, key, r, t):  h = mix64(seed ^ mix64(key)); h = mix64(h + ((uint64_t)r << 32 | t));
 *                                          u = (h >> 11) * 2^-53
 * (mix64 = the splitmix64 finaliser: x += 0x9E3779B97F4A7C15; x = (x ^ x >> 30) * 0xBF58476D1CE4E5B9;
 *  x = (x ^ x >> 27) * 0x94D049BB133111EB; x ^ x >> 31), sets c = u, and goes through state s's out-arcs in the order
 * cml_add_trellises received them: arc j has p_j = exp(lnw_j + beta(dst_j) - beta(s)), c -= p_j, and the first arc after
 * which c < 0 is taken.  When rounding leaves c >= 0 after the last arc, the last arc with p_j > 0 is taken.  An arc of
 * weight zero, or whose destination has beta = -inf, is never taken.  A lattice with ln_total = -inf gives n entries
 * with path_len 0 and ln_weight -inf.
 *   determinism the same inputs give the same bytes on every run; results do not depend on the chunking or the launch
 *               shape, and a lattice's samples do not depend on the other lattices
 *   memory      device scratch of 8 B per lattice state (beta); the lattices are processed in chunks of consecutive
 *               lattices whose scratch fits CML_OPT_KBEST_SCRATCH_MB (a lattice larger than that gets a chunk of its own)
 * GPU work: kernel k_sample, one warp per lattice: a backward pass over the levels from the top, the states of one
 * level across the lanes, then lane j draws samples j, j + 32, ... */
int cml_sample(cml_ctx* ctx, uint32_t n, uint64_t seed, const uint64_t* ex_key, uint32_t* path_len, uint64_t* path_base,
               uint32_t* path_arcs, uint64_t cap, double* ln_weight, double* ln_total);
/* the last cml_sample call: device scratch bytes of its largest chunk, number of chunks, and the time of its k_sample
 * launches from CUDA events (ms) */
int cml_sample_stats(cml_ctx* ctx, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms);
/* how the resident lattices are stored: examples / arcs / padded records in the level-sliced ELL layout
 * (throughput kernel) and examples in the layered-CSR layout (general kernels) */
int cml_layout_stats(cml_ctx* ctx, uint64_t* ell_examples, uint64_t* ell_arcs, uint64_t* ell_records,
                     uint64_t* csr_examples);
/* lattices / arcs / padded records (both sweeps) resident in the lane-per-lattice layout, and its tiles */
int cml_lane_stats(cml_ctx* ctx, uint64_t* lane_examples, uint64_t* lane_arcs, uint64_t* lane_records, uint64_t* tiles);
/* lattices on the warp-per-lattice kernel (levels of 9..32 states), their arcs and stored records (with padding), and
 * the number of arc classes / state classes the resident wide and lane lattices reference (factored arc weights) */
int cml_wide_stats(cml_ctx* ctx, uint64_t* wide_examples, uint64_t* wide_arcs, uint64_t* wide_records,
                   uint64_t* arc_classes, uint64_t* state_classes);
/* introspection for parity tests: the layered layout of resident example e.
 *   level_of[ex_states]  level of each reference state id;  local_of[ex_states] its layered index. */
int cml_get_example_layout(cml_ctx* ctx, uint64_t e, uint32_t* n_levels, uint32_t* level_of, uint32_t* local_of);

/* ---- dense-state sequences (position-synchronous lattices) ------------------------------------ *
 * The same derivations::g lattices (carmel/src/derivations.h:479-513,640-704) for the special case where
 * every arc of the trained transducer consumes exactly one symbol of ONE tape and nothing of the other
 * (e.g. a letter-bigram LM composed with a substitution channel, trained on (empty input, ciphertext)
 * pairs): lattice state (t, s) exists for every position t and transducer state s, so the lattice is never
 * materialised.  The caller gives the arc table's (source, destination, symbol) triples and the observed
 * symbol sequences; the library checks that the cascade chains factor as
 *     w(i -> j, o) = T[i][j] * E[j][o]      (chain = parameters depending on (i,j) + parameters depending on (j,o))
 * and then runs forward/backward as one S x S transition product per position followed by the emission
 * column of the observed symbol (each position step of a batch of sequences is a dense [batch x S] * [S x S]
 * product).  Expected counts are accumulated per T cell (xi) and per E cell (gamma) and handed to the same
 * M-step; likelihoods and learned weights equal the lattice path's (unreachable / dead lattice states carry
 * alpha = 0 or beta = 0).  Needs a CML_SPACE_SCALED context and no lattices resident.  Two kernels:
 *   dense   one warp per sequence, all n_states <= 32 states live at every position (cipher: 27 x 27 per letter);
 *           fp32 contexts with >= 16,384 sequences run the position step of 16 sequences at a time as 3xTF32
 *           tensor-core products (k_dense_tc), the transition counts included
 *   sparse  one lane per sequence, every symbol emitted by <= 8 states, n_states <= 64, optional final weights
 *           (HMM tagging: a word has a handful of tags); chosen for batches of >= 4096 sequences.
 * After success the count slots (cml_count_slots, cml_get_counts, the reduce buffer) are the trainable T / E
 * cells and stay so until the next cml_set_model; per-arc counts are not available.
 * Returns CML_ERR_NOT_DENSE (context unchanged) when the arc table does not factor. */
#define CML_DENSE_EPS 0xFFFFFFFFu /* arc_sym of an arc that consumes nothing: allowed only as a FINAL WEIGHT, i.e. into a
                                     final state that nothing else reaches and that has no outgoing arcs (tagging.fsa) */
typedef struct cml_dense_view {
  uint32_t n_states;        /* states of the trained transducer */
  uint32_t n_symbols;       /* observed alphabet: sequence symbols are ids in [0, n_symbols) */
  uint32_t start, final_state;
  const uint32_t* arc_src;  /* [n_arcs] per arc-table id */
  const uint32_t* arc_dst;
  const uint32_t* arc_sym;  /* the symbol the arc consumes */
} cml_dense_view;
typedef struct cml_sequence_batch {
  uint64_t n_seq;
  const uint64_t* seq_off;  /* [n_seq+1] sequence e owns sym[seq_off[e] .. seq_off[e+1]) */
  const uint32_t* sym;
  const double* seq_weight; /* [n_seq] example weight */
} cml_sequence_batch;
int cml_add_sequences(cml_ctx* ctx, const cml_dense_view* v, const cml_sequence_batch* b);
/* which kernel the resident sequences use: *sparse = 1 sparse-emission, 0 dense (FMA), 2 dense on the tensor cores
 * (3xTF32, fp32 contexts with >= 16,384 sequences), -1 none; *k = emission row width;
 * *n_states = states of the dense view */
int cml_dense_kernel(cml_ctx* ctx, int* sparse, uint32_t* k, uint32_t* n_states);
/* resident dense sequences: count, positions (sum of lengths), and whether T cells are trainable (xi kept) */
int cml_dense_stats(cml_ctx* ctx, uint64_t* n_seq, uint64_t* n_positions, uint32_t* n_t_slots, uint32_t* n_e_slots);

/* ---- E-step ----------------------------------------------------------------------------------- *
 * Replaces forward_backward::estimate (carmel/src/train.cc:763-773) = cascade.update (cascade.h:466-479),
 * clear counts, then for every example derivations::collect_counts (derivations.h:432-449:
 * compute_fb :400-417 + the count loop) and the corpus probability products (train.cc:326-332).
 *   sum_ln_p    Σ_e ln P_e           (ln of "unweighted_corpus_prob")
 *   sum_w_ln_p  Σ_e w_e ln P_e       (ln of "weighted_corpus_prob")
 *   n_zero      examples with P_e == 0 (excluded from both sums)
 * Expected counts stay on the device (per arc-table id, linear domain). */
typedef struct cml_estimate_result {
  double sum_ln_p;
  double sum_w_ln_p;
  uint64_t n_zero;
} cml_estimate_result;
int cml_estimate(cml_ctx* ctx, cml_estimate_result* out);
/* asynchronous halves of cml_estimate for multi-GPU use: launch, (all-reduce the reduce buffer), finish */
int cml_estimate_launch(cml_ctx* ctx);
int cml_estimate_finish(cml_ctx* ctx, cml_estimate_result* out);
/* device time (CUDA events on the context's stream) spent in the forward-backward-count kernels of the
 * last cml_estimate_launch, and how many such kernels ran (one per resident example class). */
int cml_last_fb_time_ms(cml_ctx* ctx, float* ms, uint32_t* n_kernels);
/* per-example ln P_e of the last estimate (order of insertion), for parity tests */
int cml_get_example_logprob(cml_ctx* ctx, double* ln_p, uint64_t n);
/* expected counts per arc-table id (linear) of the last estimate.  On a real cascade this needs
 * CML_OPT_ARC_COUNTS (otherwise counts are kept per unlocked-parameter slot: cml_get_counts). */
int cml_get_arc_counts(cml_ctx* ctx, double* counts);
uint64_t cml_count_slots(cml_ctx* ctx);
int cml_get_counts(cml_ctx* ctx, double* counts, uint64_t n);
/* The per-iteration reduce buffer: [count slots | sum_ln_p | sum_w_ln_p | n_zero] as fp64 on the
 * device.  A multi-GPU driver all-reduces (sum) it between cml_estimate_launch and
 * cml_estimate_finish (one collective per iteration).  cml_use_reduce_buffer lets the caller own the
 * memory (e.g. a torch tensor registered with NCCL); pass NULL to go back to the internal one. */
int cml_reduce_buffer(cml_ctx* ctx, void** device_ptr, uint64_t* n_doubles);
int cml_use_reduce_buffer(cml_ctx* ctx, void* device_ptr, uint64_t n_doubles);

/* ---- M-step ----------------------------------------------------------------------------------- *
 * Replaces forward_backward::maximize (carmel/src/train.cc:893-923): prep_new_weights (:134-153),
 * cascade.distribute_counts (cascade.h:286-325), WFST::normalize per cascade member (fst.cc:86-244),
 * overrelax (:157-171, rate > 1) + renormalise, max_change (:173-182).
 *   max_delta  max |w_new - w_old| over unlocked parameters (linear domain), as Weight absdiff. */
int cml_maximize(cml_ctx* ctx, double rate, double* max_delta);
/* WFST::normalize of the current parameters only (train.cc:509 initial cascade.normalize) */
int cml_normalize_params(cml_ctx* ctx);

/* ---- --crp Gibbs sampling --------------------------------------------------------------------- *
 * Replaces gibbs_base / gibbs_param (graehl/shared/gibbs.hpp:106-227,229-1079) and carmel_gibbs::
 * resample_block + derivations::random_path (carmel/src/gibbs.cc:306-371, derivations.h:345-375).
 * Parameters are the model's n_params (cml_set_model supplies the chains); lattices must be resident in
 * one batch in the layered-CSR layout (fp64 log-space context), which keeps the reference's per-state arc
 * order -- the order the sampler walks when it turns a uniform draw into an arc.
 *   param_norm  [n_params] CRP normalisation group, or CML_NO_GROUP for a fixed probability (locked arc /
 *               NONE-normalised transducer): then param_prior IS the probability (gibbs.cc:105-120)
 *   param_prior [n_params] pseudo-count alpha*p0*N (gibbs.hpp:589-597)
 * Uniform draws are counter based, u(seed, sweep, block, draw): one per visited non-final lattice state in
 * path order (random.ipp:118), so sequential mode reproduces the CPU restatement derivation by derivation. */
typedef struct cml_gibbs_model {
  uint32_t n_params;
  const uint32_t* param_norm;
  const double* param_prior;
  uint32_t n_norms;
} cml_gibbs_model;
enum cml_gibbs_mode {
  CML_GIBBS_SEQUENTIAL = 0, /* exact collapsed sampler: blocks in corpus order, counts updated between blocks */
  CML_GIBBS_BATCHED = 1,    /* all blocks in parallel against the previous sweep's counts */
  CML_GIBBS_EXPECTATION = 2 /* --expectation (gibbs.cc:311-316, derivations.h:381-398): blocks in corpus order, a block's
                               "sample" is every arc of its lattice weighted by its posterior under the current counts */
};
typedef struct cml_gibbs_sweep_opts {
  int mode;
  double power;          /* 1/temperature (gibbs.hpp:838-839) */
  uint64_t seed;
  uint32_t sweep;        /* iteration number: part of the uniform counter */
  int init_from_params;  /* sample from the current cml_set_params weights (--init-em first sample, gibbs.cc:317-322) */
  double accumulate_dt;  /* after the sweep add dt * count to the time-averaged counts (delta_sum.hpp:60-84) */
} cml_gibbs_sweep_opts;
int cml_gibbs_init(cml_ctx* ctx, const cml_gibbs_model* g); /* counts := priors (restore_p0, gibbs.hpp:618-623) */
/* Optional dense-state sampler for CML_GIBBS_BATCHED sweeps (after cml_gibbs_init): the same view / sequences as
 * cml_add_sequences (n_states <= 32, no epsilon arcs), one sequence per resident lattice in the same order.  The
 * backward filter then runs as one S x S product per position over a per-sweep dense table of arc probabilities
 * and the forward sample picks the successor state with one warp-wide scan -- the lattices are only used by the
 * sequential mode.  Samples have the same format (arc-table ids) and the same distribution; they are not the
 * lattice sampler's derivations for equal uniforms (arcs are visited in destination-state order).
 * Returns CML_ERR_NOT_DENSE (nothing changed) when an arc's CRP parameters depend on its source state. */
int cml_gibbs_attach_dense(cml_ctx* ctx, const cml_dense_view* v, const cml_sequence_batch* b);
int cml_gibbs_sweep(cml_ctx* ctx, const cml_gibbs_sweep_opts* o);
uint64_t cml_gibbs_sample_capacity(cml_ctx* ctx);
/* current sample: path_len[example], and the arc-table ids of example e's path at path_arcs[base_e ..],
 * base_e = sum of the lattice level counts of the examples before e */
int cml_gibbs_get_samples(cml_ctx* ctx, uint32_t* path_len, uint32_t* path_arcs, uint64_t cap);
int cml_gibbs_get_state(cml_ctx* ctx, double* count, double* cum, double* normsum);
/* CML_GIBBS_EXPECTATION: ln P(block) (sum over all its derivations, derivations.h:386) of the n first blocks, last sweep */
int cml_gibbs_get_block_logprob(cml_ctx* ctx, double* ln_p, uint64_t n);

/* ---- collective: the per-iteration all-reduce of the count table (SURVEY 8(e); north_star (4)) -------------- *
 * The reference is single process; the sharded E-step relies on "examples are independent given the weights"
 * (carmel/src/cached_derivs.h:69-75, forest-em/forest-em.hpp:573-578).  One ncclAllReduce(sum, fp64) of the reduce
 * buffer [count slots | sum ln P | sum w ln P | n_zero] per iteration, enqueued on the context's stream after the E-step
 * kernels; the M-step then runs redundantly on every rank (no broadcast).  NCCL is bound at run time (libnccl.so.2).
 *   one process per GPU:      rank 0 calls cml_comm_unique_id, the launcher ships the 128 bytes to every rank, every
 *                             rank calls cml_comm_init_rank on its context;
 *   one process, n contexts:  cml_comm_init_all (ncclCommInitAll), one host thread per context afterwards;
 *   existing communicator:    cml_set_comm(ctx, ncclComm_t, rank, n_ranks). */
#define CML_COMM_ID_BYTES 128
int cml_comm_unique_id(unsigned char out[CML_COMM_ID_BYTES]);
int cml_comm_init_rank(cml_ctx* ctx, int n_ranks, int rank, const unsigned char id[CML_COMM_ID_BYTES]);
int cml_comm_init_all(cml_ctx** ctxs, int n);
int cml_set_comm(cml_ctx* ctx, void* nccl_comm, int rank, int n_ranks);
int cml_comm_info(cml_ctx* ctx, int* rank, int* n_ranks);
int cml_allreduce_counts(cml_ctx* ctx);                      /* between cml_estimate_launch and cml_estimate_finish */
int cml_allreduce_buffer(cml_ctx* ctx, void* device_ptr, uint64_t n_doubles); /* in place, on the context's stream */
int cml_allreduce_host(cml_ctx* ctx, double* inout, uint64_t n /* <= 64 */);  /* small host-side sums (corpus totals) */
uint64_t cml_collective_count(cml_ctx* ctx);

/* ---- one whole EM iteration in one call ------------------------------------------------------------------------- *
 * forward_backward::estimate + maximize (carmel/src/train.cc:763-773,893-923) of one iteration of WFST::train's loop
 * (train.cc:576-657): arc weights from the parameters, E-step, all-reduce (when a communicator is set), M-step at the
 * given over-relaxation rate, and ONE host synchronisation that returns the corpus likelihood of the weights the
 * iteration started from and the largest weight change.  The parameters the iteration started from stay available to
 * cml_snapshot_previous (save_best, train.cc:592-600, after the fact).  Launches are replayed from a CUDA graph
 * captured on first use (the iteration of a small model is launch bound: ~10 launches around a 60 us kernel). */
int cml_em_step(cml_ctx* ctx, double rate, cml_estimate_result* out, double* max_delta);
int cml_snapshot_previous(cml_ctx* ctx, int slot); /* parameters before the last cml_em_step -> snapshot slot */

/* host access to the first n doubles of the reduce buffer (small control all-reduces) */
int cml_reduce_buffer_write(cml_ctx* ctx, const double* src, uint64_t n);
int cml_reduce_buffer_read(cml_ctx* ctx, double* dst, uint64_t n);

/* ---- a whole training run: the `carmel -t ...` / `--train-cascade` invocation ------------------ *
 * Replaces main()'s -t branch (carmel/src/carmel.cc:1155-1173,1286-1355,1415-1437) and WFST::train
 * (carmel/src/train.cc:503-678).  argv follows carmel's grammar (carmel.cc:929-1066): bundled flags,
 * value flags taking the next argument, --key[=value]; first file = pair corpus, then the
 * transducers (composed left to right).  Extra long options of this implementation: --float
 * (fp32 scores), --scaled (scaled linear space), --gpu=n, --shard=r/N (this process keeps block r of
 * N of the corpus on its GPU; needs an all-reduce hook), --history=file, --dump-trellis=file,
 * --device-build / --host-build (where the derivation lattices are constructed; default: host threads).
 * Log lines go to stderr in the reference's format (train.cc:587-627). */
typedef struct cml_job cml_job;
typedef void (*cml_allreduce_fn)(void* user, void* device_ptr, uint64_t n_doubles); /* in-place fp64 sum */
typedef struct cml_job_info {
  uint64_t examples, trellis_states, trellis_arcs; /* resident on this GPU */
  uint64_t n_params, n_arcs, corpus_pairs, iterations;
  double ln_best_ppx, last_ln_prob;
  uint64_t dense; /* 1: the E-step / batched sampler runs on the dense-state view (no lattice walked) */
  double device_build_s; /* > 0: the lattices were built on the GPU (cml_build_trellises) in this many seconds */
} cml_job_info;
int cml_job_open(cml_job** out, int argc, const char* const* argv); /* parse, read, reduce, compose */
void cml_job_close(cml_job* job);
const char* cml_job_error(cml_job* job);
/* sharded runs (--shard=r/N): either the NCCL rendezvous token of cml_comm_unique_id (the job's context joins the
 * communicator in cml_job_prepare and the library issues the all-reduces itself), or a host hook that sums a device
 * buffer in place; the hook is called after the context's stream has been synchronised and must have completed the
 * sum when it returns. */
int cml_job_set_comm(cml_job* job, const unsigned char id[CML_COMM_ID_BYTES]);
int cml_job_set_allreduce(cml_job* job, cml_allreduce_fn fn, void* user);
int cml_job_prepare(cml_job* job); /* model + lattices onto the GPU; no iteration yet */
cml_ctx* cml_job_context(cml_job* job); /* valid after cml_job_prepare; owned by the job */
int cml_job_train(cml_job* job);   /* the EM loop to convergence; trained weights end up in the job */
int cml_job_write(cml_job* job);   /* stdout / -F file / <input>.trained, as carmel writes them */
int cml_job_stats(cml_job* job, cml_job_info* info);

/* ---- forest-em: inside-outside EM over derivation forests -------------------------------------- *
 * Replaces FForest::compute_inside / compute_norm_outside / visit_inside_norm_outside
 * (forest-em/forest.hpp:326-491,636-697), FForests::estimate / maximize (forest-em/forest-em.hpp:
 * 511-572,626-655) and NormalizeGroups::normalize (graehl/shared/normalize.hpp:123-164,254-267).
 * Forests cross the boundary in the reference's own representation (forest.hpp:60-76): a pre-order node
 * array per forest; the library resolves back references, levelises by height and lays the hyperedges
 * out for the GPU itself.  Rule ids are the reference's 1-based parameter ids (0 is reserved for OR).
 * Scores are fp32 (forest-em's default) or fp64 (-U) natural logs; expected counts are accumulated
 * linearly in fp64.  One handle per GPU, not thread-safe per handle. */
typedef struct cml_forests cml_forests;
typedef struct cml_forest_batch {
  uint64_t n_forests;
  const uint64_t* node_off; /* [n_forests+1] forest f owns nodes [node_off[f], node_off[f+1]) */
  const uint32_t* next;     /* per node: in-forest index one past its last descendant (ForestNode::next) */
  const uint32_t* label;    /* rule id (>0), 0 = OR, or the in-forest index of the shared node (back reference) */
  const uint8_t* backref;   /* per node: 1 = label is a back reference (ForestNode::is_backref) */
} cml_forest_batch;
typedef struct cml_forest_estimate_result {
  double sum_ln_p;     /* sum over non-zero forests of ln inside[root]   (forest-em.hpp:519-527) */
  uint64_t n_zero;     /* forests with inside[root] == 0 */
  uint64_t n_forests;  /* forests visited (this GPU) */
} cml_forest_estimate_result;
enum cml_forest_zero_mode { CML_FOREST_ZERO = 0, CML_FOREST_SKIP = 1, CML_FOREST_UNIFORM = 2 }; /* normalize.hpp:113 */
typedef struct cml_forest_norm_opts {
  double prior_total;   /* added to every rule's count: prior_counts * total_forests (forest-em.hpp:448-449) */
  double add_k;         /* added to the denominator of non-empty groups (normalize.hpp:133) */
  int zero_mode;        /* groups whose counts sum to 0 */
} cml_forest_norm_opts;

int cml_forests_create(cml_forests** out, int device, int precision /* 32 | 64 */);
void cml_forests_destroy(cml_forests* f);
const char* cml_forests_last_error(cml_forests* f);
int cml_forests_set_stream(cml_forests* f, void* cuda_stream);
/* Device layout of the forests added afterwards.  AUTO: corpora of >= 256 forests that fit in a CTA's shared memory
 * use LEVEL tiles (a CTA owns a run of forests and walks their nodes height-major, all values in shared memory);
 * few or large forests use one warp / one CTA per forest with height-levelised CSRs (GROUP).  THREAD = one forest per
 * lane (32 forests per warp, transposed streams; round 1's throughput layout, efficient only when the forests of a
 * warp share a shape).  The explicit values force one family (tests, measurements). */
enum cml_forest_layout { CML_FOREST_LAYOUT_AUTO = 0, CML_FOREST_LAYOUT_GROUP = 1, CML_FOREST_LAYOUT_THREAD = 2, CML_FOREST_LAYOUT_LEVEL = 3 };
int cml_forests_set_layout(cml_forests* f, int layout);
/* level-synchronous tiles resident (CML_FOREST_LAYOUT_LEVEL, the AUTO choice for >= 256 forests that fit in shared
 * memory): forests, tiles (= CTAs per E-step), nodes, links, nodes of the largest tile, and how many of the tiles are
 * SMALL tiles (<= 12 KB of values: 128-thread CTAs, 16 per SM; the others are 512-thread CTAs with up to 100 KB) */
int cml_forests_level_stats(cml_forests* f, uint64_t* forests, uint64_t* tiles, uint64_t* nodes, uint64_t* links,
                            uint64_t* max_tile_nodes, uint64_t* small_tiles);
/* thread-per-forest tiles resident: forests in tiles, tiles, real steps, padded steps, padded value rows x 32 */
int cml_forests_layout_stats(cml_forests* f, uint64_t* tile_forests, uint64_t* tiles, uint64_t* steps, uint64_t* padded_steps,
                             uint64_t* padded_rows);
uint64_t cml_forests_launch_count(cml_forests* f);
/* rulespace = 1 + largest rule id; groups = the normalization groups file ((1 2 3) (4 5)) as CSR of rule ids */
int cml_forests_set_rules(cml_forests* f, uint64_t rulespace, uint64_t n_groups, const uint64_t* group_off,
                          const uint64_t* group_members);
int cml_forests_set_params(cml_forests* f, const double* ln_w /* [rulespace] */);
int cml_forests_get_params(cml_forests* f, double* ln_w);
int cml_forests_add(cml_forests* f, const cml_forest_batch* b);
int cml_forests_totals(cml_forests* f, uint64_t* n_forests, uint64_t* n_nodes, uint64_t* n_hyperedges, uint64_t* n_links);
/* E-step over all resident forests.  Afterwards the reduce buffer holds
 * [rulespace linear counts (no prior) | sum_ln_p | n_zero | n_forests] for an optional all-reduce. */
int cml_forests_estimate(cml_forests* f, cml_forest_estimate_result* out);
int cml_forests_estimate_launch(cml_forests* f);                               /* asynchronous half */
int cml_forests_estimate_finish(cml_forests* f, cml_forest_estimate_result* out); /* reads the (reduced) buffer */
int cml_forests_last_time_ms(cml_forests* f, float* ms, uint32_t* n_kernels);  /* inside-outside kernels only */
int cml_forests_get_inside(cml_forests* f, double* ln_inside, uint64_t n);     /* per forest, in the order added */
int cml_forests_get_counts(cml_forests* f, double* counts, uint64_t n);        /* linear, [rulespace] */
int cml_forests_reduce_buffer(cml_forests* f, void** device_ptr, uint64_t* n_doubles);
/* multi-GPU: join an NCCL communicator (token from cml_comm_unique_id) and sum the reduce buffer over the ranks on the
 * context's stream, between cml_forests_estimate_launch and cml_forests_estimate_finish */
/* ---- forest-em --crp: Gibbs sampling over forests (SURVEY 8 row a24) ------------------------------------------ *
 * Replaces FForests::run_gibbs / to_gibbs / resample_block (forest-em/forest-em.hpp:694-797), FForest::compute_inside(W)
 * and choose_random (forest-em/forest.hpp:726-816) under gibbs_base (graehl/shared/gibbs.hpp:803-877).  One parameter
 * per rule: param_norm[rule] = normalisation group (or 0xFFFFFFFF: fixed probability = param_prior[rule]),
 * param_prior[rule] = alpha * p0 * |group| (gibbs.hpp:589-597).  `b` is the batch as given to cml_forests_add.  Sweeps
 * take the same options as cml_gibbs_sweep; uniforms are u(seed, sweep, forest, draw), one per OR node visited, so
 * CML_GIBBS_SEQUENTIAL reproduces the CPU restatement derivation by derivation.  CML_GIBBS_BATCHED samples every
 * forest against the previous sweep's counts, its own previous sample included (gibbs --include-self semantics). */
typedef struct cml_forest_gibbs_model {
  const uint32_t* param_norm;  /* [rulespace] */
  const double* param_prior;   /* [rulespace] */
  uint32_t n_norms;
} cml_forest_gibbs_model;
int cml_forests_gibbs_init(cml_forests* f, const cml_forest_batch* b, const cml_forest_gibbs_model* g);
int cml_forests_gibbs_sweep(cml_forests* f, const cml_gibbs_sweep_opts* o);
uint64_t cml_forests_gibbs_sample_capacity(cml_forests* f);
/* current sample: len[forest] rule ids at ids[bases[forest] ..] in record order; bases has n_forests + 1 entries */
int cml_forests_gibbs_get_samples(cml_forests* f, uint32_t* len, uint32_t* ids, uint64_t cap, uint64_t* bases);
int cml_forests_gibbs_get_state(cml_forests* f, double* count, double* cum, double* normsum);

/* Viterbi (best derivation, FForest::viterbi_rec, forest-em/forest.hpp:507-574; forest-em -v): ln score of every
 * forest's best derivation and, per node of `b` (the batch as given to cml_forests_add), the chosen child of OR nodes
 * (in-forest pre-order index, the first child that attains the maximum; 0xFFFFFFFF elsewhere), at the current weights */
int cml_forests_viterbi(cml_forests* f, const cml_forest_batch* b, double* root_ln, uint32_t* best_child);
/* The k best derivations of every forest of `b` (the batch as given to cml_forests_add) at the current weights, best
 * first (forest-em -v FILE --kbest=n).  A derivation is returned as the AND nodes (rule applications) it uses, in
 * derivation pre-order; the tree is rebuilt from the forest alone: each child slot of an AND node (its direct pre-order
 * child: an AND node, an OR node or a back reference) takes the next listed node, the AND node the slot resolves to.
 *   ln_score[n_forests * k]   ln score of derivation (i, r) at [i * k + r]; -inf where forest i has fewer than r + 1
 *   n_and[n_forests * k]      AND nodes of derivation (i, r); 0 with -inf
 *   base[n_forests * k + 1]   derivation (i, r) is nodes[base[i * k + r] .. + n_and[i * k + r])
 *   nodes[cap]                in-forest pre-order indices of its AND nodes, or NULL for scores and sizes only
 * Contract:
 *   order        each forest's derivations come in non-increasing score
 *   distinct     they are distinct choice sets (one child per OR node reached), so k counts derivations, not unique
 *                trees; a back-referenced shared node is expanded independently at each use
 *   zero weight  derivations of weight zero (ln -inf) are never listed; a forest of probability zero is all padding
 *   scores       fp64, from the handle's fp64 weights whatever its precision (as cml_forests_viterbi)
 *   ties         an OR node's list is the top k over its children's entries by score (descending), then child
 *                pre-order position, then child rank; an AND node with rule weight w and slots s1..sm is the left fold
 *                L0 = [w], Lj = top k { L(j-1)[a] + sj[b] } (ties by a, then b), summed in that order; a back reference
 *                has its shared node's list
 *   rank 0       for every forest with a finite Viterbi score it is bit-identical to cml_forests_viterbi: the same
 *                double and the same OR choices
 *   determinism  the same inputs give the same bytes on every run
 *   nesting      no depth limit: a forest nested deeper than cml_forests_viterbi's 96 levels decodes
 *   memory       device scratch of 40 B * k + 16 B per pre-order node (a node's list and the fold through a child slot,
 *                each 20 B per entry: score, back pointer, subtree size) plus 8 B * max(k, largest OR fan-out) per lane
 *                group; forests are processed in chunks of consecutive forests whose scratch fits the budget of
 *                cml_forests_set_kbest_scratch_mb (a forest larger than that gets a chunk of its own).  Results do not
 *                depend on the chunking.
 * Errors: CML_ERR_STATE before cml_forests_set_params; CML_ERR_ARG for k == 0, for a malformed forest, or for a non-NULL
 * `nodes` with cap < base[n_forests * k] -- then ln_score, n_and and base are still filled, so the caller can size the
 * buffer and call again. */
int cml_forests_kbest(cml_forests* f, const cml_forest_batch* b, uint32_t k, double* ln_score, uint32_t* n_and,
                      uint64_t* base, uint32_t* nodes, uint64_t cap);
int cml_forests_set_kbest_scratch_mb(cml_forests* f, uint64_t mb); /* scratch budget of one chunk (MiB); default 4096 */
/* the last cml_forests_kbest call: device scratch bytes of its largest chunk, chunks, and the time of its derivation
 * kernels from CUDA events (ms) */
int cml_forests_kbest_stats(cml_forests* f, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms);
/* The total weight of every forest of `b` (the batch as given to cml_forests_add) at the current weights, and n
 * derivations of each drawn in proportion to their weight, P(d | forest) = w(d) / sum of w over its derivations
 * (forest-em -v FILE --sample=n).  Scores are fp64, from the handle's fp64 weights whatever its precision.
 *   ln_total[n_forests]       the inside weight of forest i's root, in fp64:
 *                               AND node, rule r, slots s1..sm   ln_w[r] + in(s1) + ... + in(sm), summed in slot order
 *                               OR node                          a max-shifted log-sum-exp over its children, in order;
 *                                                                -inf when every child is -inf
 *                               back reference                   its shared node's value
 *                             This is not the E-step's pairwise log-add with its cutoff (cml_forests_get_inside): the
 *                             two agree to rounding, not bit for bit.
 *   n = 0                     computes ln_total only; key and the other outputs may then be null
 *   key[n_forests]            the key of forest i's uniforms, or null for key = i
 *   ln_weight[n_forests * n]  ln weight of sample (i, r) at [i * n + r]: the sum of its rules' ln weights, added in
 *                             the order of its nodes
 *   n_and, base, nodes, cap   as in cml_forests_kbest with k = n: sample r of forest i is nodes[base[i * n + r] ..
 *                             + n_and[i * n + r]), the in-forest pre-order indices of its AND nodes in derivation
 *                             pre-order; nodes = NULL for weights and sizes only
 * A forest with ln_total = -inf gives n entries with n_and 0 and ln_weight -inf.
 * Sample r of forest i walks the derivation in pre-order from the root, as FForest::choose_random does
 * (forest-em/forest.hpp:726-758): depth first, children in order.  A back reference stands for its shared node.  An AND
 * node is recorded, then its slots are visited first to last, each slot's whole sub-derivation before the next.  At the
 * t-th OR decision of the sample (t = 0, 1, ... in visiting order) it draws u = sample_uniform(seed, key_i, r, t) (as
 * defined at cml_sample), sets c = u and goes through the OR node's children in pre-order: child j has
 * p_j = exp(in(child_j) - in(or)); children with p_j = 0 are skipped, otherwise c -= p_j, and the first child after
 * which c < 0 is taken.  When rounding leaves c >= 0 after the last child, the last child with p_j > 0 is taken.
 *   determinism  the same inputs give the same bytes on every run; results do not depend on the chunking or the launch
 *                shape, and a forest's samples depend only on that forest, the weights, seed and its key
 *   nesting      no depth limit: a forest nested deeper than cml_forests_viterbi's 96 levels samples
 *   size         with n > 0, a forest whose largest derivation of non-zero weight has more than 2^32 - 2 AND nodes is
 *                refused with CML_ERR_ARG and none of its samples is drawn (a saturating max-size pass runs next to
 *                the inside pass)
 *   memory       device scratch of 12 B per pre-order node (inside value, largest derivation size) and 8 B + 20 B * n
 *                per forest (total; per sample its weight, size and output offset); forests are processed in chunks of
 *                consecutive forests whose scratch fits the budget of cml_forests_set_kbest_scratch_mb (a forest
 *                larger than that gets a chunk of its own).  The walk adds 8 B * (levels of the tallest forest) per
 *                walker, with 32 walkers per warp of up to min(chunk forests / 4, 16 * SMs) blocks of 4 warps, and the
 *                drawn nodes of a chunk take 4 B each.
 * Errors: CML_ERR_STATE before cml_forests_set_params; CML_ERR_CYCLE for a cyclic back reference; CML_ERR_ARG for a
 * malformed forest, a rule id beyond rulespace, a null ln_total, n > 0 with a null ln_weight, n_and or base, a forest
 * too large (above), or a non-NULL `nodes` with cap < base[n_forests * n] -- then ln_weight, n_and, base and ln_total
 * are still filled, so the caller can size the buffer and call again.
 * GPU work: k_forest_sample, one warp per forest: an inside pass by height, the nodes of one height across the lanes,
 * then lane j draws samples j, j + 32, ...; k_forest_sample_paths, one thread per sample, walks it again with the
 * same uniforms and writes its nodes. */
int cml_forests_sample(cml_forests* f, const cml_forest_batch* b, uint32_t n, uint64_t seed, const uint64_t* key,
                       double* ln_weight, uint32_t* n_and, uint64_t* base, uint32_t* nodes, uint64_t cap,
                       double* ln_total);
/* the last cml_forests_sample call: device scratch bytes of its largest chunk, chunks, and the time of its kernels
 * from CUDA events (ms) */
int cml_forests_sample_stats(cml_forests* f, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms);
int cml_forests_synchronize(cml_forests* f);
int cml_forests_comm_init_rank(cml_forests* f, int n_ranks, int rank, const unsigned char id[CML_COMM_ID_BYTES]);
int cml_forests_allreduce_counts(cml_forests* f);
/* M-step: rule_weights <- normalised (counts + prior_total).  max_delta / max_index as NormalizeGroups
 * reports them (largest absolute change of a probability and the rule it belongs to). */
int cml_forests_maximize(cml_forests* f, const cml_forest_norm_opts* o, double* max_delta, uint64_t* max_index);
int cml_forests_normalize_params(cml_forests* f); /* --normalize-initial: weights normalised in place */

/* A whole forest-em run (forest-em/forest-em-params.cpp:62-148): argv follows forest-em's options
 * (forest-em-params.hpp:69-176; the training subset, see INTEGRATION.md).  Extra: --gpu=n, --shard=r/N,
 * --history=file. */
typedef struct cml_forest_job cml_forest_job;
typedef struct cml_forest_job_info {
  uint64_t forests, nodes, hyperedges, links, rulespace, iterations;
  double best_avg_logprob;
} cml_forest_job_info;
int cml_forest_job_open(cml_forest_job** out, int argc, const char* const* argv);
void cml_forest_job_close(cml_forest_job* job);
const char* cml_forest_job_error(cml_forest_job* job);
int cml_forest_job_set_quiet(cml_forest_job* job, int quiet); /* no log lines from this job (ranks > 0 of --gpus=N) */
int cml_forest_job_set_comm(cml_forest_job* job, const unsigned char id[CML_COMM_ID_BYTES]); /* as cml_job_set_comm */
int cml_forest_job_set_allreduce(cml_forest_job* job, cml_allreduce_fn fn, void* user);
int cml_forest_job_prepare(cml_forest_job* job);
cml_forests* cml_forest_job_context(cml_forest_job* job);
int cml_forest_job_train(cml_forest_job* job);
int cml_forest_job_write(cml_forest_job* job);
int cml_forest_job_stats(cml_forest_job* job, cml_forest_job_info* info);

/* ---- host-side helpers exported for bindings and tests (no GPU needed) ------------------------ */
/* Every symbol this header declares, for the loader test. */
const char* const* cml_exported_symbols(size_t* n);

#ifdef __cplusplus
}
#endif
#endif /* CARMEL_B200_H */
