// cml_sample.cu -- the total weight of every resident lattice, and derivations drawn from it in proportion to their
// weight (the backward filter, forward sample of carmel/src/derivations.h:345-375 random_path, at fixed weights).
//
// k_sample: one warp per lattice.  The backward pass walks the levels from the top down; the states of one level never
// feed each other (every arc goes up at least one level), so they are spread over the lanes, and levels are separated
// by __syncwarp.  beta(s) = ln sum over out-arcs of w(arc) * exp(beta(dst)), a max-shifted log-sum-exp in fp64, with
// beta(goal) = 0.  Then lane j draws samples j, j + 32, ...: each walks forward from the start, taking at state s the
// first out-arc (stored order) at which u - p_1 - ... - p_j drops below 0, p_j = exp(lnw_j + beta(dst_j) - beta(s)), and
// writes arc-table ids straight into its path slot.  The uniforms are counter based (seed, key, sample, step), so a
// draw does not depend on the launch shape, the chunking or the other lattices.
#include <algorithm>
#include <cmath>

#include "cml_ctx.cuh"

namespace {

constexpr int kSampleWarps = 4;  // warps per block

struct SampleArgs {
  const CmlExDesc* desc;
  const uint32_t* list;      // desc slots handled by this launch
  uint32_t n_list;
  uint32_t n;                // samples per lattice
  uint64_t seed;
  const uint64_t* key;       // [n_ex] key of every lattice's uniforms, or null (key = lattice index)
  const uint32_t* lvl_off;
  const uint32_t* out_off;
  const uint2* out_arc;      // {dst layered index, internal arc id}
  const double* arc_lnw;     // ln weight per internal arc id
  const uint32_t* arc_orig;  // internal arc id -> arc-table id
  const uint64_t* st_base;   // [desc slot] first state of the lattice in the chunk's beta scratch
  const uint64_t* lvl_pre;   // [example] sum of the levels of the examples before it
  double* beta;              // [chunk states]
  double* ln_total;          // [n_ex]
  uint32_t* path_len;        // [n_ex * n]
  uint32_t* path_arcs;       // [n * total levels]
  double* ln_weight;         // [n_ex * n]
};

__global__ void __launch_bounds__(kSampleWarps * 32) k_sample(SampleArgs A) {
  const uint32_t lane = threadIdx.x & 31;
  for (uint32_t w = blockIdx.x * kSampleWarps + threadIdx.x / 32; w < A.n_list; w += gridDim.x * kSampleWarps) {
    const uint32_t slot = A.list[w];
    const CmlExDesc d = A.desc[slot];
    const uint32_t* __restrict__ lv = A.lvl_off + d.lvl_base;
    const uint32_t* __restrict__ ooff = A.out_off + d.row_base;
    const uint2* __restrict__ oa = A.out_arc + d.arc_base;
    const double* __restrict__ lnw = A.arc_lnw;
    double* B = A.beta + A.st_base[slot];
    for (uint32_t l = d.n_levels; l-- > 0;) {
      for (uint32_t j = lv[l] + lane; j < lv[l + 1]; j += 32) {
        double b = 0.;
        if (j != d.fin) {
          const uint32_t a0 = ooff[j], a1 = ooff[j + 1];
          double m = -CUDART_INF;
          for (uint32_t a = a0; a < a1; ++a) {
            const uint2 x = oa[a];
            m = fmax(m, lnw[x.y] + B[x.x]);
          }
          if (m > -CUDART_INF) {
            double sum = 0.;
            for (uint32_t a = a0; a < a1; ++a) {
              const uint2 x = oa[a];
              sum += exp(lnw[x.y] + B[x.x] - m);
            }
            b = m + log(sum);
          } else {
            b = -CUDART_INF;
          }
        }
        B[j] = b;
      }
      __syncwarp();
    }
    const uint32_t e = d.ex_index;
    const double total = B[0];
    if (lane == 0) A.ln_total[e] = total;
    const uint64_t h0 = mix64(A.seed ^ mix64(A.key ? A.key[e] : (uint64_t)e));
    for (uint32_t r = lane; r < A.n; r += 32) {
      const uint64_t o = (uint64_t)e * A.n + r;
      if (!(total > -CUDART_INF)) {
        A.ln_weight[o] = -CUDART_INF;
        A.path_len[o] = 0;
        continue;
      }
      uint32_t* __restrict__ out = A.path_arcs + A.lvl_pre[e] * A.n + (uint64_t)r * d.n_levels;
      double wsum = 0.;
      uint32_t s = 0, t = 0;
      while (s != d.fin) {  // beta(s) > -inf on the way: some out-arc has p > 0
        double c = sample_uniform(h0, r, t);
        const double bs = B[s];
        uint32_t pick = 0xFFFFFFFFu, last = 0xFFFFFFFFu;
        for (uint32_t a = ooff[s]; a < ooff[s + 1]; ++a) {
          const uint2 x = oa[a];
          const double p = exp(lnw[x.y] + B[x.x] - bs);
          if (p > 0.) {
            last = a;
            c -= p;
            if (c < 0.) {
              pick = a;
              break;
            }
          }
        }
        if (pick == 0xFFFFFFFFu) pick = last;  // rounding left c >= 0: the last arc that can be taken
        const uint2 x = oa[pick];
        out[t++] = A.arc_orig[x.y];
        wsum += lnw[x.y];
        s = x.x;
      }
      A.path_len[o] = t;
      A.ln_weight[o] = wsum;
    }
  }
}

}  // namespace

extern "C" int cml_sample(cml_ctx* ctx, uint32_t n, uint64_t seed, const uint64_t* ex_key, uint32_t* path_len,
                          uint64_t* path_base, uint32_t* path_arcs, uint64_t cap, double* ln_weight, double* ln_total) {
  if (!ctx || !ln_total || (n && (!path_len || !path_base || !path_arcs || !ln_weight))) return CML_ERR_ARG;
  Batch* b = nullptr;
  if (const int rc = cml_decode_batch(ctx, "cml_sample", "derivations of a lattice with a cycle are not sampled", &b))
    return rc;
  Batch& bt = *b;
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  const uint64_t n_ex = bt.n_ex;
  const std::vector<uint64_t> lvl_pre = cml_path_slots(bt, n, path_base);
  CML_REQUIRE(!n || cap >= lvl_pre[n_ex] * n, CML_ERR_ARG,
              "path_arcs too small (need n times the total number of lattice levels)");
  ctx->sample = DecodeStats();
  if (!n_ex) return CML_OK;
  if (const int rc = cml_arc_weights_f64(ctx, ctx->ln_w.p)) return rc;
  DevArray<uint32_t> d_orig;
  if (const int rc = cml_upload_arc_orig(ctx, d_orig)) return rc;
  DecodeChunks P;  // chunk scratch: beta, 8 B per state
  if (const int rc = cml_decode_chunks(ctx, bt, sizeof(double), 0, P)) return rc;
  const uint64_t n_chunks = P.mid.size();
  DevArray<uint32_t> d_list, d_plen, d_path;
  DevArray<uint64_t> d_stb, d_pre, d_key;
  DevArray<double> d_beta, d_lnw, d_tot;
  CML_CUDA(d_list.upload(P.list.data(), P.list.size(), s));
  CML_CUDA(d_stb.upload(P.st_base.data(), n_ex, s));
  CML_CUDA(d_pre.upload(lvl_pre.data(), lvl_pre.size(), s));
  if (ex_key) CML_CUDA(d_key.upload(ex_key, n_ex, s));
  CML_CUDA(d_beta.alloc(std::max<uint64_t>(1, P.max_states)));
  CML_CUDA(d_tot.alloc(n_ex));
  CML_CUDA(d_plen.alloc(std::max<uint64_t>(1, n_ex * n)));
  CML_CUDA(d_lnw.alloc(std::max<uint64_t>(1, n_ex * n)));
  CML_CUDA(d_path.alloc(std::max<uint64_t>(1, lvl_pre[n_ex] * n)));
  ctx->sample.chunks = n_chunks;
  ctx->sample.scratch = P.max_states * sizeof(double);
  SampleArgs A{bt.desc.p, nullptr, 0, n, seed, ex_key ? d_key.p : nullptr, bt.lvl_off.p, bt.out_off.p, bt.out_arc.p,
               (const double*)ctx->arc_w_real.p, d_orig.p, d_stb.p, d_pre.p, d_beta.p, d_tot.p, d_plen.p, d_path.p,
               d_lnw.p};
  EventPair ev;
  CML_CUDA(ev.create());
  CML_CUDA(cudaEventRecord(ev.a, s));
  const unsigned max_blocks = (unsigned)ctx->sm_count * 16u;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const uint64_t b0 = P.begin[c], b1 = P.begin[c + 1];
    A.list = d_list.p + b0;
    A.n_list = (uint32_t)(b1 - b0);
    const unsigned grid = std::max(1u, std::min(cdiv(b1 - b0, kSampleWarps), max_blocks));
    k_sample<<<grid, kSampleWarps * 32, 0, s>>>(A);
    ++ctx->launches;
    CML_CUDA(cudaGetLastError());
  }
  CML_CUDA(cudaEventRecord(ev.b, s));
  CML_CUDA(cudaMemcpyAsync(ln_total, d_tot.p, n_ex * sizeof(double), cudaMemcpyDeviceToHost, s));
  // n = 0: the totals only (the counts below are 0, nothing else is copied)
  return cml_decode_download(ctx, n_ex * n, path_len, d_plen.p, ln_weight, d_lnw.p, lvl_pre[n_ex] * n, path_arcs, d_path.p,
                             ev, &ctx->sample.ms);
}

extern "C" int cml_sample_stats(cml_ctx* ctx, uint64_t* scratch_bytes, uint64_t* chunks, float* kernel_ms) {
  return ctx ? ctx->sample.get(scratch_bytes, chunks, kernel_ms) : CML_ERR_ARG;
}
