// cml_decode.cu -- the best (cml_viterbi) and the k best (cml_kbest) derivations of every resident lattice (carmel -k n
// on the composed string x transducer x string machine, graehl/shared/kbest.h via fst.h:769-800), and the host code
// every per-lattice decoder over the layered CSR shares (cml_sample.cu's too).
//
// k_viterbi: a max-plus forward pass over the layered CSR -- states in layered (topological) order, each state's
// out-arcs in the reference's stored order, a destination takes a new best only on a STRICT improvement -- then a walk
// back from the goal.  One thread per lattice (a decode runs once after training).
//
// k-best: an eager per-state k-way merge in layered (topological) order.  A state's list is the top k of
//   { (score(src, r) + w(arc), in-list position p, r) }
// over its in-arcs, ordered by score (descending), then p, then r (ascending).  Every source list is already
// sorted that way, so the merge only ever looks at one head per in-arc.  Rank 0 of a state is then the FIRST
// maximum over its in-list, which is what a max-plus pass over sources in layered order with strict improvement
// finds (the in-list is sorted by source layered index, then stored out-arc order): rank 0 is bit-identical to the
// best derivation of that pass.
//
// k_kbest: one warp per lattice.  States of one level never feed each other (every arc goes up at least one level),
// so a level's states are merged in parallel by lane groups of G lanes; levels are separated by __syncwarp.  Source
// lists stay in global memory (epsilon arcs can skip levels).  Lane g of a group owns in-list positions g, g + G, ...;
// it keeps the best head among them in registers, the cursor of position g in a register and the cursors of the
// other positions (in-degree > G only) in a per-arc scratch.  Each round is a shuffle arg-max over the group; the
// owner of the winner appends it, advances its cursor and rescans its positions.
#include <algorithm>
#include <cmath>

#include "cml_ctx.cuh"
#include "cml_kernels_model.cuh"

namespace {

__global__ void k_viterbi(const CmlExDesc* __restrict__ desc, uint32_t n_ex, const uint32_t* __restrict__ out_off,
                          const uint2* __restrict__ out_arc, const double* __restrict__ arc_lnw,
                          const uint32_t* __restrict__ arc_orig, const uint64_t* __restrict__ state_base,
                          const uint64_t* __restrict__ path_base, double* __restrict__ best, uint32_t* __restrict__ bp_src,
                          uint32_t* __restrict__ bp_arc, uint32_t* __restrict__ path_len, uint32_t* __restrict__ path_arcs,
                          double* __restrict__ ln_weight) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_ex) return;
  const CmlExDesc d = desc[t];
  const uint32_t e = d.ex_index, n = d.n_states;
  const uint32_t* __restrict__ ooff = out_off + d.row_base;
  const uint2* __restrict__ oarc = out_arc + d.arc_base;
  double* __restrict__ b = best + state_base[e];
  uint32_t* __restrict__ ps = bp_src + state_base[e];
  uint32_t* __restrict__ pa = bp_arc + state_base[e];
  for (uint32_t j = 0; j < n; ++j) b[j] = -CUDART_INF;
  b[0] = 0.;  // the start state has layered index 0
  for (uint32_t j = 0; j < n; ++j) {
    const double bj = b[j];
    if (!(bj > -CUDART_INF)) continue;
    for (uint32_t k = ooff[j]; k < ooff[j + 1]; ++k) {
      const uint2 a = oarc[k];
      const double c = bj + arc_lnw[a.y];
      if (c > b[a.x]) {
        b[a.x] = c;
        ps[a.x] = j;
        pa[a.x] = a.y;
      }
    }
  }
  ln_weight[e] = b[d.fin];
  uint32_t len = 0;
  if (b[d.fin] > -CUDART_INF)
    for (uint32_t s = d.fin; s != 0; s = ps[s]) ++len;
  path_len[e] = len;
  uint32_t* __restrict__ out = path_arcs + path_base[e];
  uint32_t i = len;
  if (len)
    for (uint32_t s = d.fin; s != 0; s = ps[s]) out[--i] = arc_orig[pa[s]];
}

constexpr int kKbestWarps = 4;  // warps per block

struct KbestArgs {
  const CmlExDesc* desc;
  const uint32_t* list;      // desc slots handled by this launch
  uint32_t n_list;
  uint32_t k;
  const uint32_t* lvl_off;
  const uint32_t* in_off;
  const uint2* in_arc;
  const double* arc_lnw;     // ln weight per internal arc id
  const uint32_t* arc_orig;  // internal arc id -> arc-table id
  const uint64_t* st_base;   // [desc slot] first state of the lattice in the chunk's list scratch
  const uint64_t* cur_base;  // [desc slot] first in-arc of the lattice in the chunk's cursor scratch
  const uint64_t* lvl_pre;   // [example] sum of the levels of the examples before it
  double* sc;                // [chunk states * k] list scores
  uint2* bp;                 // [chunk states * k] (in-list position, source rank)
  uint32_t* len;             // [chunk states] list lengths
  uint32_t* cur;             // [chunk in-arcs] cursors of the positions >= G
  uint32_t* path_len;        // [n_ex * k]
  uint32_t* path_arcs;       // [k * total levels] or null
  double* ln_weight;         // [n_ex * k]
};

// head of an in-arc at cursor c: score of the source's rank c plus the arc's weight (-inf: the source has no rank c)
__device__ __forceinline__ double kbest_head(uint2 a, uint32_t c, uint32_t k, const double* __restrict__ S,
                                             const uint32_t* __restrict__ L, const double* __restrict__ arc_lnw) {
  return c < L[a.x] ? S[(uint64_t)a.x * k + c] + arc_lnw[a.y] : -CUDART_INF;
}

template <int G>
__global__ void k_kbest(KbestArgs A) {
  const uint32_t lane = threadIdx.x & 31, g = lane % G, grp = lane / G;
  const unsigned gmask = G == 32 ? 0xFFFFFFFFu : (((1u << G) - 1u) << (grp * G));
  const uint32_t k = A.k;
  for (uint32_t w = blockIdx.x * kKbestWarps + threadIdx.x / 32; w < A.n_list; w += gridDim.x * kKbestWarps) {
    const uint32_t slot = A.list[w];
    const CmlExDesc d = A.desc[slot];
    const uint32_t* __restrict__ lv = A.lvl_off + d.lvl_base;
    const uint32_t* __restrict__ ioff = A.in_off + d.row_base;
    const uint2* __restrict__ ia = A.in_arc + d.arc_base;
    double* __restrict__ S = A.sc + A.st_base[slot] * k;
    uint2* __restrict__ B = A.bp + A.st_base[slot] * k;
    uint32_t* __restrict__ L = A.len + A.st_base[slot];
    uint32_t* __restrict__ C = A.cur + A.cur_base[slot];
    for (uint32_t l = 0; l < d.n_levels; ++l) {
      const uint32_t j1 = lv[l + 1];
      for (uint32_t j = lv[l] + grp; j < j1; j += 32 / G) {  // group-uniform
        if (j == 0) {        // the start state: one empty derivation
          if (g == 0) {
            S[0] = 0.;
            B[0] = make_uint2(0, 0);
            L[0] = 1;
          }
          continue;
        }
        const uint32_t a0 = ioff[j], deg = ioff[j + 1] - a0;
        uint32_t c0 = 0;  // cursor of position g
        double bv = -CUDART_INF;
        uint32_t bq = 0xFFFFFFFFu;
        for (uint32_t q = g; q < deg; q += G) {
          if (q != g) C[a0 + q] = 0;
          const double v = kbest_head(ia[a0 + q], 0, k, S, L, A.arc_lnw);
          if (v > bv) {
            bv = v;
            bq = q;
          }
        }
        uint32_t r = 0;
        for (; r < k; ++r) {
          double v = bv;
          uint32_t q = bq;
#pragma unroll
          for (int o = G / 2; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(gmask, v, o, G);
            const uint32_t oq = __shfl_xor_sync(gmask, q, o, G);
            if (ov > v || (ov == v && oq < q)) {
              v = ov;
              q = oq;
            }
          }
          if (!(v > -CUDART_INF)) break;  // group-uniform: no candidate left
          if (q % G == g) {               // the owner appends the winner and advances its cursor
            const uint32_t c = q == g ? c0 : C[a0 + q];
            S[(uint64_t)j * k + r] = v;
            B[(uint64_t)j * k + r] = make_uint2(q, c);
            if (q == g)
              c0 = c + 1;
            else
              C[a0 + q] = c + 1;
            bv = -CUDART_INF;
            bq = 0xFFFFFFFFu;
            for (uint32_t p = g; p < deg; p += G) {
              const double hv = kbest_head(ia[a0 + p], p == g ? c0 : C[a0 + p], k, S, L, A.arc_lnw);
              if (hv > bv) {
                bv = hv;
                bq = p;
              }
            }
          }
        }
        if (g == 0) L[j] = r;
      }
      __syncwarp();
    }
    // walk back: one lane per final rank
    const uint32_t e = d.ex_index, fin = d.fin, nf = L[fin];
    for (uint32_t r = lane; r < k; r += 32) {
      const uint64_t o = (uint64_t)e * k + r;
      if (r >= nf) {
        A.ln_weight[o] = -CUDART_INF;
        A.path_len[o] = 0;
        continue;
      }
      A.ln_weight[o] = S[(uint64_t)fin * k + r];
      uint32_t n = 0;
      for (uint32_t s = fin, rr = r; s != 0; ++n) {
        const uint2 b = B[(uint64_t)s * k + rr];
        s = ia[ioff[s] + b.x].x;
        rr = b.y;
      }
      A.path_len[o] = n;
      if (!A.path_arcs) continue;
      uint32_t* __restrict__ out = A.path_arcs + A.lvl_pre[e] * k + (uint64_t)r * d.n_levels;
      for (uint32_t s = fin, rr = r, i = n; s != 0;) {
        const uint2 b = B[(uint64_t)s * k + rr];
        const uint2 a = ia[ioff[s] + b.x];
        out[--i] = A.arc_orig[a.y];
        s = a.x;
        rr = b.y;
      }
    }
  }
}

// per desc slot: (largest in-degree, number of in-arcs) -- sizes the lane groups and the chunks
__global__ void k_kbest_shape(const CmlExDesc* __restrict__ desc, uint32_t n, const uint32_t* __restrict__ in_off,
                              uint2* __restrict__ shape) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const CmlExDesc d = desc[t];
  const uint32_t* ioff = in_off + d.row_base;
  uint32_t m = 0;
  for (uint32_t j = 0; j < d.n_states; ++j) m = max(m, ioff[j + 1] - ioff[j]);
  shape[t] = make_uint2(m, ioff[d.n_states]);
}

}  // namespace

// The entry checks of a per-lattice decoder: model and parameters set, fp64 log space, the lattices in one batch in the
// layered-CSR layout, none with a cycle.  `name` starts the space and layout messages, cycle_msg is the cycle message.
int cml_decode_batch(cml_ctx* ctx, const char* name, const char* cycle_msg, Batch** bt) {
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  CML_REQUIRE(ctx->precision == 64 && ctx->space == CML_SPACE_LOG, CML_ERR_STATE,
              std::string(name) + " runs in fp64 log space (create the context with precision 64, CML_SPACE_LOG)");
  CML_REQUIRE(ctx->batches.size() == 1 && ctx->batches[0]->ell_ex == 0 && ctx->batches[0]->lane_ex == 0, CML_ERR_STATE,
              std::string(name) + " needs the lattices in ONE batch in the layered-CSR layout");
  CML_REQUIRE(ctx->batches[0]->cyc_ex == 0, CML_ERR_CYCLE, cycle_msg);
  *bt = ctx->batches[0].get();
  return CML_OK;
}

// the path slots of n derivations per lattice: a derivation has at most (levels - 1) arcs; example e's derivation r
// starts at n * lvl_pre[e] + r * levels(e).  Fills path_base[n_ex * n + 1] when non-null and returns lvl_pre[n_ex + 1].
std::vector<uint64_t> cml_path_slots(Batch const& bt, uint32_t n, uint64_t* path_base) {
  const uint64_t n_ex = bt.n_ex;
  std::vector<uint64_t> lvl_pre(n_ex + 1, 0);
  for (uint64_t e = 0; e < n_ex; ++e) lvl_pre[e + 1] = lvl_pre[e] + bt.h_nlevels[e];
  if (path_base) {
    for (uint64_t e = 0; e < n_ex; ++e)
      for (uint32_t r = 0; r < n; ++r) path_base[e * n + r] = lvl_pre[e] * n + (uint64_t)r * bt.h_nlevels[e];
    path_base[n_ex * n] = lvl_pre[n_ex] * n;
  }
  return lvl_pre;
}

// the fp64 ln weight of every arc, in internal order, at the ln parameters lnp (arc_w_real, the table the log-space
// sweeps use): ctx->ln_w for the decoders, the Gibbs sampler's own table for its sweeps
int cml_arc_weights_f64(cml_ctx* ctx, const double* lnp) {
  cudaStream_t s = ctx->stream;
  if (ctx->arc_slot_code.n < (size_t)ctx->n_arcs + 1) {
    CML_CUDA(ctx->arc_slot_code.alloc((size_t)ctx->n_arcs + 1));
    CML_CUDA(cudaMemsetAsync(ctx->arc_slot_code.p, 0xFF, ((size_t)ctx->n_arcs + 1) * sizeof(uint32_t), s));
  }
  cmlk::k_arc_weights<double, false, cmlk::WS<double>><<<cdiv(ctx->n_arcs + 1, 256), 256, 0, s>>>(
      ctx->n_arcs, ctx->trivial ? nullptr : ctx->chain_off.p, ctx->chain_param.p, lnp, ctx->arc_slot_code.p,
      ctx->arc_perm.p, ctx->arc_lnw.p, (double*)ctx->arc_w_real.p, (cmlk::WS<double>*)ctx->arc_ws.p);
  ++ctx->launches;
  return CML_OK;
}

// the way back from internal arc ids to arc-table ids, on the device
int cml_upload_arc_orig(cml_ctx* ctx, DevArray<uint32_t>& orig) {
  std::vector<uint32_t> h((size_t)ctx->n_arcs + 1, 0);
  for (uint32_t a = 0; a < ctx->n_arcs; ++a) h[ctx->h_perm[a]] = a;
  CML_CUDA(orig.upload(h.data(), h.size(), ctx->stream));
  return CML_OK;
}

// Chunks of consecutive desc slots whose scratch (state_bytes per state, arc_bytes per in-arc) fits
// CML_OPT_KBEST_SCRATCH_MB; a lattice larger than the budget gets a chunk of its own.  Within a chunk the slots whose
// largest in-degree is <= 8 come first (k_kbest's G = 8 part).
int cml_decode_chunks(cml_ctx* ctx, Batch& bt, uint64_t state_bytes, uint64_t arc_bytes, DecodeChunks& C) {
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  // lattice shapes (by desc slot) decide the lane-group width and the chunks
  DevArray<uint2> d_shape;
  CML_CUDA(d_shape.alloc(n_ex));
  k_kbest_shape<<<cdiv(n_ex, 128), 128, 0, s>>>(bt.desc.p, (uint32_t)n_ex, bt.in_off.p, d_shape.p);
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  std::vector<uint2> shape(n_ex);
  std::vector<CmlExDesc> desc(n_ex);
  CML_CUDA(cudaMemcpyAsync(shape.data(), d_shape.p, n_ex * sizeof(uint2), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaMemcpyAsync(desc.data(), bt.desc.p, n_ex * sizeof(CmlExDesc), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  const uint64_t budget = (uint64_t)ctx->opt_kbest_scratch_mb << 20;
  C.st_base.assign(n_ex, 0);
  C.cur_base.assign(n_ex, 0);
  C.list.clear();
  C.begin.assign(1, 0);
  C.mid.clear();
  C.max_states = C.max_arcs = 0;
  uint64_t ns = 0, na = 0;
  std::vector<uint32_t> wide;
  auto close_chunk = [&]() {
    C.mid.push_back(C.list.size());
    C.list.insert(C.list.end(), wide.begin(), wide.end());
    wide.clear();
    C.begin.push_back(C.list.size());
    C.max_states = std::max(C.max_states, ns);
    C.max_arcs = std::max(C.max_arcs, na);
    ns = na = 0;
  };
  for (uint64_t t = 0; t < n_ex; ++t) {
    const uint64_t st = desc[t].n_states, ar = shape[t].y;
    if ((ns || na) && ((ns + st) * state_bytes + (na + ar) * arc_bytes > budget)) close_chunk();
    C.st_base[t] = ns;
    C.cur_base[t] = na;
    ns += st;
    na += ar;
    if (shape[t].x <= 8)
      C.list.push_back((uint32_t)t);
    else
      wide.push_back((uint32_t)t);
  }
  close_chunk();
  return CML_OK;
}

// The end of a decoder call, once ev.b is recorded behind its kernels: copies the m path lengths and ln weights and the
// n_path path arcs back (each when its host pointer is non-null and its count non-zero), waits for the stream and
// stores the kernel time between the two events in *ms.
int cml_decode_download(cml_ctx* ctx, uint64_t m, uint32_t* path_len, const uint32_t* d_len, double* ln_weight,
                        const double* d_lnw, uint64_t n_path, uint32_t* path_arcs, const uint32_t* d_path,
                        EventPair const& ev, float* ms) {
  cudaStream_t s = ctx->stream;
  if (path_len && m) CML_CUDA(cudaMemcpyAsync(path_len, d_len, m * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  if (ln_weight && m) CML_CUDA(cudaMemcpyAsync(ln_weight, d_lnw, m * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (path_arcs && n_path)
    CML_CUDA(cudaMemcpyAsync(path_arcs, d_path, n_path * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  CML_CUDA(cudaEventElapsedTime(ms, ev.a, ev.b));
  return CML_OK;
}

extern "C" int cml_viterbi(cml_ctx* ctx, uint32_t* path_len, uint64_t* path_base, uint32_t* path_arcs, uint64_t cap, double* ln_weight) {
  if (!ctx || !path_len || !path_base || !ln_weight) return CML_ERR_ARG;
  Batch* b = nullptr;
  if (const int rc = cml_decode_batch(ctx, "cml_viterbi", "best derivation of a lattice with a cycle is not built", &b))
    return rc;
  Batch& bt = *b;
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  const std::vector<uint64_t> pbase = cml_path_slots(bt, 1, path_base);
  CML_REQUIRE(!path_arcs || cap >= pbase[n_ex], CML_ERR_ARG, "path_arcs too small (need the total number of lattice levels)");
  if (const int rc = cml_arc_weights_f64(ctx, ctx->ln_w.p)) return rc;
  DevArray<uint32_t> d_orig, d_src, d_arc, d_len, d_path;
  DevArray<uint64_t> d_sbase, d_pbase;
  DevArray<double> d_best, d_lnw;
  if (const int rc = cml_upload_arc_orig(ctx, d_orig)) return rc;
  CML_CUDA(d_sbase.upload(bt.h_state_base.data(), bt.h_state_base.size(), s));
  CML_CUDA(d_pbase.upload(pbase.data(), pbase.size(), s));
  CML_CUDA(d_best.alloc(std::max<uint64_t>(1, bt.n_states)));
  CML_CUDA(d_src.alloc(std::max<uint64_t>(1, bt.n_states)));
  CML_CUDA(d_arc.alloc(std::max<uint64_t>(1, bt.n_states)));
  CML_CUDA(d_len.alloc(std::max<uint64_t>(1, n_ex)));
  CML_CUDA(d_lnw.alloc(std::max<uint64_t>(1, n_ex)));
  CML_CUDA(d_path.alloc(std::max<uint64_t>(1, pbase[n_ex])));
  EventPair ev;
  CML_CUDA(ev.create());
  CML_CUDA(cudaEventRecord(ev.a, s));
  k_viterbi<<<cdiv(n_ex, 64), 64, 0, s>>>(bt.desc.p, (uint32_t)n_ex, bt.out_off.p, bt.out_arc.p, (const double*)ctx->arc_w_real.p,
                                         d_orig.p, d_sbase.p, d_pbase.p, d_best.p, d_src.p, d_arc.p, d_len.p, d_path.p, d_lnw.p);
  CML_CUDA(cudaEventRecord(ev.b, s));
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  if (const int rc = cml_decode_download(ctx, n_ex, path_len, d_len.p, ln_weight, d_lnw.p, pbase[n_ex], path_arcs, d_path.p,
                                         ev, &ctx->kbest.ms))
    return rc;
  ctx->kbest.chunks = 1;
  ctx->kbest.scratch = bt.n_states * (sizeof(double) + 2 * sizeof(uint32_t));
  return CML_OK;
}

extern "C" int cml_kbest(cml_ctx* ctx, uint32_t k, uint32_t* path_len, uint64_t* path_base, uint32_t* path_arcs,
                         uint64_t cap, double* ln_weight) {
  if (!ctx || !path_len || !path_base || !ln_weight) return CML_ERR_ARG;
  Batch* b = nullptr;
  if (const int rc = cml_decode_batch(ctx, "cml_kbest", "derivations of a lattice with a cycle are not built", &b)) return rc;
  Batch& bt = *b;
  CML_REQUIRE(k > 0, CML_ERR_ARG, "cml_kbest: k must be at least 1");
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  const std::vector<uint64_t> lvl_pre = cml_path_slots(bt, k, path_base);
  CML_REQUIRE(!path_arcs || cap >= lvl_pre[n_ex] * k, CML_ERR_ARG,
              "path_arcs too small (need k times the total number of lattice levels)");
  ctx->kbest = DecodeStats();
  if (!n_ex) return CML_OK;
  if (const int rc = cml_arc_weights_f64(ctx, ctx->ln_w.p)) return rc;
  DevArray<uint32_t> d_orig;
  if (const int rc = cml_upload_arc_orig(ctx, d_orig)) return rc;
  // chunk scratch: k list entries of 16 B and a length per state, a cursor per in-arc
  DecodeChunks P;
  if (const int rc = cml_decode_chunks(ctx, bt, 16ull * k + 4, 4, P)) return rc;
  const uint64_t n_chunks = P.mid.size(), max_states = P.max_states, max_arcs = P.max_arcs;
  DevArray<uint32_t> d_list, d_len, d_plen, d_path, d_cur;
  DevArray<uint64_t> d_stb, d_curb, d_pre;
  DevArray<double> d_sc, d_lnw;
  DevArray<uint2> d_bp;
  CML_CUDA(d_list.upload(P.list.data(), P.list.size(), s));
  CML_CUDA(d_stb.upload(P.st_base.data(), n_ex, s));
  CML_CUDA(d_curb.upload(P.cur_base.data(), n_ex, s));
  CML_CUDA(d_pre.upload(lvl_pre.data(), lvl_pre.size(), s));
  CML_CUDA(d_sc.alloc(std::max<uint64_t>(1, max_states * k)));
  CML_CUDA(d_bp.alloc(std::max<uint64_t>(1, max_states * k)));
  CML_CUDA(d_len.alloc(std::max<uint64_t>(1, max_states)));
  CML_CUDA(d_cur.alloc(std::max<uint64_t>(1, max_arcs)));
  CML_CUDA(d_plen.alloc(n_ex * k));
  CML_CUDA(d_lnw.alloc(n_ex * k));
  if (path_arcs) CML_CUDA(d_path.alloc(std::max<uint64_t>(1, lvl_pre[n_ex] * k)));
  ctx->kbest.chunks = n_chunks;
  ctx->kbest.scratch = max_states * (16ull * k + 4) + max_arcs * 4;
  KbestArgs A{bt.desc.p, nullptr, 0, k, bt.lvl_off.p, bt.in_off.p, bt.in_arc.p, (const double*)ctx->arc_w_real.p,
              d_orig.p, d_stb.p, d_curb.p, d_pre.p, d_sc.p, d_bp.p, d_len.p, d_cur.p, d_plen.p,
              path_arcs ? d_path.p : nullptr, d_lnw.p};
  EventPair ev;
  CML_CUDA(ev.create());
  CML_CUDA(cudaEventRecord(ev.a, s));
  const unsigned max_blocks = (unsigned)ctx->sm_count * 16u;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    for (int wide_part = 0; wide_part < 2; ++wide_part) {
      const uint64_t b0 = wide_part ? P.mid[c] : P.begin[c], b1 = wide_part ? P.begin[c + 1] : P.mid[c];
      if (b1 == b0) continue;
      A.list = d_list.p + b0;
      A.n_list = (uint32_t)(b1 - b0);
      const unsigned grid = std::max(1u, std::min(cdiv(b1 - b0, kKbestWarps), max_blocks));
      if (wide_part)
        k_kbest<32><<<grid, kKbestWarps * 32, 0, s>>>(A);
      else
        k_kbest<8><<<grid, kKbestWarps * 32, 0, s>>>(A);
      ++ctx->launches;
      CML_CUDA(cudaGetLastError());
    }
  }
  CML_CUDA(cudaEventRecord(ev.b, s));
  return cml_decode_download(ctx, n_ex * k, path_len, d_plen.p, ln_weight, d_lnw.p, lvl_pre[n_ex] * k, path_arcs, d_path.p,
                             ev, &ctx->kbest.ms);
}

extern "C" int cml_kbest_stats(cml_ctx* ctx, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms) {
  return ctx ? ctx->kbest.get(scratch_bytes, chunks, kernel_ms) : CML_ERR_ARG;
}
