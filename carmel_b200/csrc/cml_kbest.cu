// cml_kbest.cu -- the k best derivations of every resident lattice (carmel -k n on the composed
// string x transducer x string machine, graehl/shared/kbest.h via fst.h:769-800).
//
// An eager per-state k-way merge in layered (topological) order.  A state's list is the top k of
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

// What every per-lattice decoder needs before its launches: the ln arc weights at the current parameters (arc_w_real),
// the way back from internal arc ids to arc-table ids (C.orig), and chunks of consecutive desc slots whose scratch
// (state_bytes per state, arc_bytes per in-arc) fits CML_OPT_KBEST_SCRATCH_MB; a lattice larger than the budget gets a
// chunk of its own.  Within a chunk the slots whose largest in-degree is <= 8 come first (k_kbest's G = 8 part).
int cml_decode_setup(cml_ctx* ctx, Batch& bt, uint64_t state_bytes, uint64_t arc_bytes, DecodeChunks& C) {
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  if (ctx->arc_slot_code.n < (size_t)ctx->n_arcs + 1) {
    CML_CUDA(ctx->arc_slot_code.alloc((size_t)ctx->n_arcs + 1));
    CML_CUDA(cudaMemsetAsync(ctx->arc_slot_code.p, 0xFF, ((size_t)ctx->n_arcs + 1) * sizeof(uint32_t), s));
  }
  cmlk::k_arc_weights<double, false, cmlk::WS<double>><<<cdiv(ctx->n_arcs + 1, 256), 256, 0, s>>>(
      ctx->n_arcs, ctx->trivial ? nullptr : ctx->chain_off.p, ctx->chain_param.p, ctx->ln_w.p, ctx->arc_slot_code.p,
      ctx->arc_perm.p, ctx->arc_lnw.p, (double*)ctx->arc_w_real.p, (cmlk::WS<double>*)ctx->arc_ws.p);
  ++ctx->launches;
  std::vector<uint32_t> orig((size_t)ctx->n_arcs + 1, 0);
  for (uint32_t a = 0; a < ctx->n_arcs; ++a) orig[ctx->h_perm[a]] = a;
  CML_CUDA(C.orig.upload(orig.data(), orig.size(), s));
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

extern "C" int cml_kbest(cml_ctx* ctx, uint32_t k, uint32_t* path_len, uint64_t* path_base, uint32_t* path_arcs,
                         uint64_t cap, double* ln_weight) {
  if (!ctx || !path_len || !path_base || !ln_weight) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  CML_REQUIRE(ctx->precision == 64 && ctx->space == CML_SPACE_LOG, CML_ERR_STATE,
              "cml_kbest runs in fp64 log space (create the context with precision 64, CML_SPACE_LOG)");
  CML_REQUIRE(ctx->batches.size() == 1 && ctx->batches[0]->ell_ex == 0 && ctx->batches[0]->lane_ex == 0, CML_ERR_STATE,
              "cml_kbest needs the lattices in ONE batch in the layered-CSR layout");
  Batch& bt = *ctx->batches[0];
  CML_REQUIRE(bt.cyc_ex == 0, CML_ERR_CYCLE, "derivations of a lattice with a cycle are not built");
  CML_REQUIRE(k > 0, CML_ERR_ARG, "cml_kbest: k must be at least 1");
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  const std::vector<uint64_t> lvl_pre = cml_path_slots(bt, k, path_base);
  CML_REQUIRE(!path_arcs || cap >= lvl_pre[n_ex] * k, CML_ERR_ARG,
              "path_arcs too small (need k times the total number of lattice levels)");
  ctx->kbest_ms = 0;
  ctx->kbest_chunks = 0;
  ctx->kbest_scratch = 0;
  if (!n_ex) return CML_OK;
  // chunk scratch: k list entries of 16 B and a length per state, a cursor per in-arc
  DecodeChunks P;
  const int rc = cml_decode_setup(ctx, bt, 16ull * k + 4, 4, P);
  if (rc != CML_OK) return rc;
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
  ctx->kbest_chunks = n_chunks;
  ctx->kbest_scratch = max_states * (16ull * k + 4) + max_arcs * 4;
  KbestArgs A{bt.desc.p, nullptr, 0, k, bt.lvl_off.p, bt.in_off.p, bt.in_arc.p, (const double*)ctx->arc_w_real.p,
              P.orig.p, d_stb.p, d_curb.p, d_pre.p, d_sc.p, d_bp.p, d_len.p, d_cur.p, d_plen.p,
              path_arcs ? d_path.p : nullptr, d_lnw.p};
  struct Events {
    cudaEvent_t a = nullptr, b = nullptr;
    ~Events() {
      if (a) cudaEventDestroy(a);
      if (b) cudaEventDestroy(b);
    }
  } ev;
  CML_CUDA(cudaEventCreate(&ev.a));
  CML_CUDA(cudaEventCreate(&ev.b));
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
  CML_CUDA(cudaMemcpyAsync(path_len, d_plen.p, n_ex * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaMemcpyAsync(ln_weight, d_lnw.p, n_ex * k * sizeof(double), cudaMemcpyDeviceToHost, s));
  if (path_arcs && lvl_pre[n_ex])
    CML_CUDA(cudaMemcpyAsync(path_arcs, d_path.p, lvl_pre[n_ex] * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CML_CUDA(cudaStreamSynchronize(s));
  CML_CUDA(cudaEventElapsedTime(&ctx->kbest_ms, ev.a, ev.b));
  return CML_OK;
}

extern "C" int cml_kbest_stats(cml_ctx* ctx, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms) {
  if (!ctx) return CML_ERR_ARG;
  if (scratch_bytes) *scratch_bytes = ctx->kbest_scratch;
  if (chunks) *chunks = ctx->kbest_chunks;
  if (kernel_ms) *kernel_ms = ctx->kbest_ms;
  return CML_OK;
}
