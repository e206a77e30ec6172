// cml_ctx.cuh -- the context object behind the C ABI (shared by cml_device.cu and cml_gibbs.cu).
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "cml_common.cuh"
#include "cml_kernels_ell.cuh"
#include "cml_kernels_fb.cuh"
#include "cml_kernels_lane.cuh"
#include "cml_kernels_wide.cuh"

// ---- example classes ------------------------------------------------------------------------------
// ELL classes (scaled space only): one example per group of 4/8/16/32 lanes, level-sliced ELL layout.
// CSR classes (everything else): one example per warp (shared-memory capacity classes), per CTA, or
// per CTA with alpha/beta in an HBM scratch.
enum { NELL = 7 };
struct EllClass {
  int R, C;  // row-lanes x column-lanes per example: level width <= R, max degree <= C * kEllSlots
  bool cta;  // R*C == 256: one example per block
};
// ordered by group size: an example takes the first class it fits
static const EllClass kEllCls[NELL] = {{4, 1, false},  {8, 1, false},  {4, 4, false}, {8, 4, false},
                                       {16, 2, false}, {32, 1, false}, {32, 8, true}};
// CLS_CYCLIC: lattices with a cycle, walked in the reference's DFS order by k_fb_cyclic (one thread per lattice)
enum ExClass { CLS_WARP0 = 0, NWARPCLS = 6, CLS_CTA = 6, CLS_GLOBAL = 7, CLS_CYCLIC = 8, NCLS = 9 };
static const uint32_t kWarpCaps[NWARPCLS] = {64, 128, 256, 512, 1024, 2048};
static const uint32_t kPadNone = 0xFFFFFFFFu;

struct Batch {
  uint64_t n_ex = 0, n_states = 0, n_arcs = 0, n_levels = 0;
  DevArray<double> ex_lnp;
  DevArray<double> ex_weight;  // for k_reduce_lnp
  // --- CSR part (v1 kernels)
  uint64_t csr_ex = 0;
  DevArray<CmlExDesc> desc;
  DevArray<uint32_t> lvl_off, in_off, out_off;
  DevArray<uint2> in_arc, out_arc;
  DevArray<uint32_t> ex_list;  // all CSR classes concatenated (indices into desc)
  uint32_t cls_begin[NCLS + 1] = {0};
  uint32_t cta_cap = 0;
  DevArray<unsigned char> scratch;
  DevArray<int> scratch_lvl;
  DevArray<double> cyc_scratch;  // CLS_CYCLIC: ln alpha / ln beta, 2 per state
  uint64_t cyc_ex = 0, cyc_back_edges = 0;
  // --- ELL part (v2 kernel)
  uint64_t ell_ex = 0, ell_arcs = 0, ell_pad_records = 0;
  DevArray<cmlk::EllDesc> edesc;
  DevArray<uint4> lvl_meta;
  DevArray<uint2> ell_in, ell_out;
  DevArray<uint32_t> ell_list;
  uint32_t ell_begin[NELL + 1] = {0};
  uint32_t ell_ring[NELL] = {0};
  DevArray<unsigned char> alpha_g;
  DevArray<int> lvl_exp;
  // --- wide part (k_fb_wide: one lattice per warp, lane = state of the level; shares edesc / lvl_meta / ell_in /
  //     ell_out / alpha_g / lvl_exp with the ELL part, records carry arc-CLASS ids, states carry a state class)
  uint64_t wide_ex = 0, wide_arcs = 0, wide_records = 0;
  DevArray<uint32_t> wide_list;      // indices into edesc, longest first
  DevArray<uint32_t> ell_vcls;       // [ELL state slot] state class (v id) of the wide examples' states
  uint32_t wide_ring = 0;
  // --- lane part (k_fb_lane: one lattice per lane, tiles of 32)
  uint64_t lane_ex = 0, lane_arcs = 0, lane_records = 0;
  uint32_t lane_tiles = 0, lane_ring = 16;
  DevArray<cmlk::LaneTile> ltile;
  DevArray<uint2> lane_fw, lane_bw;
  DevArray<uint32_t> lane_exidx, lane_fin, lane_nlev;
  DevArray<double> lane_weight;
  DevArray<unsigned char> lane_alpha;
  DevArray<int> lane_lvle;
  DevArray<uint32_t> lane_vcls;      // [state ordinal][lane] state class (v id), same indexing as lane_alpha
  cudaEvent_t ev_fb0 = nullptr, ev_fb1 = nullptr;  // bracket this batch's forward-backward kernels
  uint32_t n_fb_kernels = 0;
  ~Batch() {
    if (ev_fb0) cudaEventDestroy(ev_fb0);
    if (ev_fb1) cudaEventDestroy(ev_fb1);
  }
  // host copies kept for introspection (cml_get_example_layout)
  std::vector<uint64_t> h_state_base;
  std::vector<uint32_t> h_level_of, h_local_of, h_nlevels;
};

// Dense-state sequences (cml_add_sequences, cml_dense.cu): w(i -> j, o) = T[i][j] * E[j][o].
struct SparseTile {     // sparse-emission kernel: 32 sequences of similar length
  uint64_t sym_base;    // symbol t of lane l at sym[sym_base + t*32 + l]
  uint64_t row_base;    // alpha rows: alpha[((row_base + t) * K + c) * 32 + l], exps[(row_base + t) * 32 + l]
  uint32_t n_max, pad;
};
struct DenseState {
  uint32_t S = 0, n_sym = 0, start = 0, fin = 0;
  uint32_t SP = 32, nT = 1024, K = 0;  // padded state count (row stride of T); sparse kernel: emission row width (4 / 8)
  bool sparse = false;      // lane-per-sequence sparse-emission kernel instead of the warp-per-sequence dense one
  int has_phi = 0;          // epsilon arcs into the final state = final weights
  uint32_t n_tiles = 0;
  uint64_t n_seq = 0, n_pos = 0;
  uint32_t n_t_slots = 0, n_e_slots = 0;
  uint32_t n_cells = 0;  // 32*32 T cells then n_sym*32 E cells (symbol major)
  DevArray<uint32_t> cell_off, cell_param, cell_slot;
  DevArray<unsigned char> cell_exists;
  DevArray<unsigned char> tables;  // Real T[32][32] then Real Et[n_sym][32]
  DevArray<uint64_t> seq_off;
  DevArray<uint16_t> sym;
  DevArray<double> seq_weight, ex_lnp;
  DevArray<unsigned char> alpha_g;  // Real[(n_pos + n_seq)][32]
  DevArray<int> exp_g;              // cumulative power-of-two exponent of every alpha row
  // tensor-core sweeps (k_dense_tc): groups of 16 sequences, beta rows, per-sequence alpha_n[final]
  bool tc = false;
  uint32_t tc_groups = 0;
  DevArray<uint32_t> tc_order;
  DevArray<unsigned char> beta_g;
  DevArray<int> bexp_g, tc_ean;
  DevArray<double> tc_afin;
  // sparse kernel: tiles of 32 sequences, per-lane facts, emission rows
  DevArray<SparseTile> stile;
  DevArray<uint32_t> lane_len, lane_seq, e_code;
  DevArray<double> lane_weight;
  DevArray<unsigned char> e_state;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  ~DenseState() {
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
  }
};

// what cml_kbest_stats / cml_sample_stats report: device scratch bytes of the largest chunk, chunks, kernel time
struct DecodeStats {
  uint64_t scratch = 0, chunks = 0;
  float ms = 0;
  int get(uint64_t* scratch_bytes, uint64_t* n_chunks, float* kernel_ms) const {
    if (scratch_bytes) *scratch_bytes = scratch;
    if (n_chunks) *n_chunks = chunks;
    if (kernel_ms) *kernel_ms = ms;
    return CML_OK;
  }
};

struct cml_ctx {
  int device = 0;
  int precision = 64;
  int space = CML_SPACE_LOG;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = CML_SM_COUNT_FALLBACK;
  uint32_t hot_copies = cmlk::kHotCopies;  // replicas of a hot count slot (power of two; CML_HOT_COPIES)
  size_t smem_optin = 0;
  std::string err;
  uint64_t launches = 0;
  int opt_arc_counts = 0;  // CML_OPT_ARC_COUNTS: keep one count slot per arc-table entry
  int opt_no_ell = 0;      // CML_OPT_NO_ELL: force the CSR kernels (tests)
  int opt_lane_min = 16384;  // CML_OPT_LANE_MIN: eligible lattices needed before the lane kernel is used (0 = never)
  int opt_no_counts = 0;     // CML_OPT_NO_COUNTS: profiling only, the sweeps skip their count REDs (lane kernel)
  int opt_no_factor = 0;     // CML_OPT_NO_FACTOR: keep per-arc weight records (no arc classes; round-1 kernels)
  int opt_no_wide = 0;       // CML_OPT_NO_WIDE: wide lattices stay on the k_fb_ell classes
  int opt_kbest_scratch_mb = 4096;  // CML_OPT_KBEST_SCRATCH_MB: scratch of one cml_kbest / cml_sample chunk
  int opt_free_build_scratch_mb = 4096;  // CML_OPT_FREE_BUILD_SCRATCH_MB: cell scratch of one cml_build_free_trellises chunk
  DecodeStats kbest, sample;  // last cml_kbest / cml_viterbi call; last cml_sample call

  // model
  bool have_model = false, trivial = true;
  uint32_t n_arcs = 0, n_params = 0, n_groups = 0, n_ties = 0, n_slots = 0, max_group_size = 0;
  bool slots_are_arcs = true;
  std::vector<uint32_t> h_arc_slot;  // host copy: slot of every arc (kPadNone = contributes to no parameter)
  // internal arc numbering (locality order): weight tables and lattice records use perm[arc id]
  std::vector<uint32_t> h_perm, h_slot_internal;
  DevArray<uint32_t> arc_perm;
  // hot count slots (see CountSink in cml_kernels_fb.cuh): occurrence statistics of the resident lattices
  std::vector<uint64_t> slot_occ;    // arcs per slot over all resident batches
  bool hot_dirty = true;             // slot codes must be rebuilt before the next E-step
  uint32_t n_hot = 0;
  DevArray<uint32_t> arc_slot_code, hot_slot;
  DevArray<double> hot_counts;
  DevArray<uint32_t> chain_off, chain_param, param_group, param_tie, group_off, group_members, tie_off, tie_members;
  DevArray<uint32_t> arc_slot, slot_off, slot_param;
  DevArray<double> slot_prior, group_add;
  bool have_prior = false, have_add = false;
  DevArray<double> ln_w, snap[4], arc_lnw, acc, u, old, gsum, glocked, tie_arc, tie_state, tie_maxl;
  DevArray<unsigned char> arc_w_real, arc_ws;
  DevArray<unsigned long long> maxchg;
  bool have_params = false;

  // reduce buffer: [n_slots counts | sum_ln_p | sum_w_ln_p | n_zero]
  DevArray<double> reduce_own;
  double* reduce = nullptr;
  uint64_t reduce_n = 0;

  std::vector<std::unique_ptr<Batch>> batches;
  bool estimate_pending = false;
  int opt_allow_empty = 0;   // CML_OPT_ALLOW_EMPTY: an E-step over no resident examples contributes zeros (empty shard)

  // collective (cml_comm.cu): ncclComm_t of this rank, or null for a single-GPU context
  void* comm = nullptr;
  bool own_comm = false;
  int comm_rank = 0, comm_size = 1;
  uint64_t collectives = 0;
  DevArray<double> host_scratch;  // 64 doubles: small host-side all-reduces (corpus statistics)
  // fused EM step (cml_em_step): pinned result block, CUDA graph of the whole iteration
  double* h_step = nullptr;       // pinned: sum ln P, sum w ln P, n_zero, max change (bits)
  cudaGraphExec_t graph = nullptr, graph_b = nullptr;  // graph_b: the part after the all-reduce (multi-GPU)
  bool graph_dirty = true, capturing = false;
  uint64_t graph_launches = 0, graph_collectives = 0;  // kernels / collectives one replay stands for
  int opt_no_graph = 0;           // CML_OPT_NO_GRAPH: cml_em_step enqueues its launches one by one
  // host copies of the chains (the dense-state factorisation needs them)
  std::vector<uint32_t> h_chain_off, h_chain_param, h_param_tie;
  std::vector<double> h_arc_prior;
  std::unique_ptr<DenseState> dense;  // non-null: the E-step runs over dense-state sequences

  // ---- factored arc weights (wide / lane kernels; see "arc classes" in cml_device.cu) ----------------------
  // model level (same on every rank): class = a multiset of parameters; every arc has a full class (its chain),
  // and, when its chain has >= 2 parameters, a state part (the last parameter) and a rest part.
  bool factored = false;
  std::vector<uint32_t> cls_off, cls_param;     // class -> parameters (CSR)
  std::vector<uint32_t> cls_slot;               // class -> count slot (kPadNone: nothing trainable)
  std::vector<uint32_t> arc_fcls, arc_ucls, arc_vcls;  // per arc-table entry (arc_vcls = kPadNone: no state part)
  // context level (append-only as batches arrive): classes referenced by lattice ARC records (a ids) and by
  // lattice STATES (v ids)
  std::vector<uint32_t> a_of_cls, v_of_cls, a_list, v_list;
  std::vector<uint64_t> a_occ, v_occ;           // occurrences in the resident lattices (hot-slot statistics)
  bool cls_dirty = true;                        // device tables must be rebuilt
  int any_a_slot = 0;                           // some arc class has a count slot
  DevArray<uint32_t> a_off, a_param, a_slot, v_off, v_param, v_slot;
  DevArray<unsigned char> a_w, v_w;             // Real[n + 1] linear weights (last = 0 / 1 padding entry)

  // --crp Gibbs sampling state (cml_gibbs.cu)
  bool have_gibbs = false;
  uint32_t g_norms = 0;
  DevArray<uint32_t> g_param_norm, g_arc_orig, g_sample[2], g_sample_len[2], g_au_off, g_au_param;
  DevArray<double> g_prior, g_count, g_cum, g_normsum, g_lnp, g_beta, g_tbl, g_delta;
  DevArray<uint64_t> g_sample_base, g_beta_base;
  DevArray<double> g_post[2], g_alpha, g_blk_lnp;  // --expectation: per-lattice-arc posteriors (two generations), alpha, ln P per block
  DevArray<uint2> g_arc_pg;
  std::vector<uint64_t> h_sample_base;
  uint64_t g_sample_cap = 0;
  int g_cur = 0;  // which sample buffer holds the current sample
  // dense-state batched sampler (cml_gibbs_attach_dense)
  bool gd_attached = false;
  uint32_t gd_S = 0, gd_V = 0, gd_start = 0, gd_fin = 0;
  DevArray<uint32_t> gd_arc, gd_rep;   // [(o*S+j)*32+i] internal arc id; [o*S+j] an arc that carries the (j,o) CRP parameters
  DevArray<uint64_t> gd_seq_off;
  DevArray<uint16_t> gd_sym;
  DevArray<double> gd_W, gd_beta;      // per-sweep dense probability table; beta rows [(positions + sequences)][32]
};

int cml_dense_estimate_launch(cml_ctx* ctx);  // cml_dense.cu

// Host code shared by the per-lattice decoders over the layered CSR (cml_decode.cu: cml_viterbi, cml_kbest;
// cml_sample.cu: cml_sample).
int cml_decode_batch(cml_ctx* ctx, const char* name, const char* cycle_msg, Batch** bt);
std::vector<uint64_t> cml_path_slots(Batch const& bt, uint32_t n, uint64_t* path_base);
int cml_arc_weights_f64(cml_ctx* ctx, const double* lnp);  // also cml_gibbs_sweep's per-arc table
int cml_upload_arc_orig(cml_ctx* ctx, DevArray<uint32_t>& orig);
// the chunks of desc slots one cml_kbest / cml_sample call walks
struct DecodeChunks {
  std::vector<uint64_t> st_base, cur_base;  // [desc slot] first state / in-arc of the lattice in its chunk's scratch
  std::vector<uint32_t> list;               // chunk c = list[begin[c] .. begin[c + 1]); in-degree > 8 from mid[c] on
  std::vector<uint64_t> begin, mid;
  uint64_t max_states = 0, max_arcs = 0;    // of the largest chunk
};
int cml_decode_chunks(cml_ctx* ctx, Batch& bt, uint64_t state_bytes, uint64_t arc_bytes, DecodeChunks& C);
int cml_decode_download(cml_ctx* ctx, uint64_t m, uint32_t* path_len, const uint32_t* d_len, double* ln_weight,
                        const double* d_lnw, uint64_t n_path, uint32_t* path_arcs, const uint32_t* d_path,
                        EventPair const& ev, float* ms);

#define CML_REQUIRE(cond, code, msg) \
  do {                               \
    if (!(cond)) {                   \
      ctx->err = (msg);              \
      return (code);                 \
    }                                \
  } while (0)

static inline unsigned cdiv(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

