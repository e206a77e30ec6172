// cml_device.cu -- C ABI (include/carmel_b200.h) of the B200-native carmel training hot path:
// context, model tables, trellis flattening (layered CSR + level-sliced ELL), E-step and M-step
// launches.  sm_100a only; there is no CPU fallback (every compute entry point needs the device).
#include <algorithm>
#include <atomic>
#include <climits>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>

#include "cml_ctx.cuh"
#include "cml_kernels_model.cuh"

static thread_local std::string g_create_err;
void cml_comm_release(cml_ctx* ctx);  // cml_comm.cu

// -------------------------------------------------------------------------------------------------
// context
// -------------------------------------------------------------------------------------------------
extern "C" const char* cml_version(void) { return "carmel_b200 0.2 (sm_100a)"; }

extern "C" int cml_create(cml_ctx** out, int device, int precision, int space) {
  if (!out) return CML_ERR_ARG;
  *out = nullptr;
  if (precision != 32 && precision != 64) {
    g_create_err = "precision must be 32 or 64";
    return CML_ERR_ARG;
  }
  if (space != CML_SPACE_LOG && space != CML_SPACE_SCALED) {
    g_create_err = "space must be CML_SPACE_LOG or CML_SPACE_SCALED";
    return CML_ERR_ARG;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (carmel_b200 has no CPU fallback)";
    return CML_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) {
    g_create_err = "device index out of range";
    return CML_ERR_ARG;
  }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_create_err = cudaGetErrorString(e);
    return CML_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_create_err = "carmel_b200 is built for sm_100a (Blackwell B200) only; found sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor);
    return CML_ERR_CUDA;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    g_create_err = cudaGetErrorString(e);
    return CML_ERR_CUDA;
  }
  cml_ctx* ctx = new cml_ctx();
  ctx->device = device;
  ctx->precision = precision;
  ctx->space = space;
  ctx->sm_count = prop.multiProcessorCount;
  if (const char* e = getenv("CML_HOT_COPIES")) {  // tuning knob: replicas per hot count slot (power of two, 1..1024)
    uint32_t c = (uint32_t)std::max(1, atoi(e)), p2 = 1;
    while (p2 * 2 <= c && p2 < 1024) p2 *= 2;
    ctx->hot_copies = p2;
  }
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_err = cudaGetErrorString(e);
    delete ctx;
    return CML_ERR_CUDA;
  }
  ctx->own_stream = true;
  *out = ctx;
  return CML_OK;
}

extern "C" void cml_destroy(cml_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  cml_comm_release(ctx);
  if (ctx->graph) cudaGraphExecDestroy(ctx->graph);
  if (ctx->graph_b) cudaGraphExecDestroy(ctx->graph_b);
  if (ctx->h_step) cudaFreeHost(ctx->h_step);
  ctx->batches.clear();
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" const char* cml_last_error(cml_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int cml_set_stream(cml_ctx* ctx, void* s) {
  if (!ctx) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)s;
  ctx->own_stream = false;
  ctx->graph_dirty = true;
  return CML_OK;
}

extern "C" int cml_synchronize(cml_ctx* ctx) {
  if (!ctx) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" uint64_t cml_launch_count(cml_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int cml_set_option(cml_ctx* ctx, int option, int value) {
  if (!ctx) return CML_ERR_ARG;
  switch (option) {
    case CML_OPT_ARC_COUNTS:
      CML_REQUIRE(!ctx->have_model, CML_ERR_STATE, "CML_OPT_ARC_COUNTS must be set before cml_set_model");
      ctx->opt_arc_counts = value;
      return CML_OK;
    case CML_OPT_NO_ELL:
      CML_REQUIRE(ctx->batches.empty(), CML_ERR_STATE, "CML_OPT_NO_ELL must be set before cml_add_trellises");
      ctx->opt_no_ell = value;
      return CML_OK;
    case CML_OPT_LANE_MIN:
      CML_REQUIRE(ctx->batches.empty(), CML_ERR_STATE, "CML_OPT_LANE_MIN must be set before cml_add_trellises");
      ctx->opt_lane_min = value;
      return CML_OK;
    case CML_OPT_NO_COUNTS:
      ctx->opt_no_counts = value;
      ctx->graph_dirty = true;
      return CML_OK;
    case CML_OPT_NO_FACTOR:
      CML_REQUIRE(!ctx->have_model, CML_ERR_STATE, "CML_OPT_NO_FACTOR must be set before cml_set_model");
      ctx->opt_no_factor = value;
      return CML_OK;
    case CML_OPT_ALLOW_EMPTY:
      ctx->opt_allow_empty = value;
      return CML_OK;
    case CML_OPT_NO_GRAPH:
      ctx->opt_no_graph = value;
      ctx->graph_dirty = true;
      return CML_OK;
    case CML_OPT_NO_WIDE:
      CML_REQUIRE(ctx->batches.empty(), CML_ERR_STATE, "CML_OPT_NO_WIDE must be set before cml_add_trellises");
      ctx->opt_no_wide = value;
      return CML_OK;
    case CML_OPT_KBEST_SCRATCH_MB:
      CML_REQUIRE(value > 0, CML_ERR_ARG, "CML_OPT_KBEST_SCRATCH_MB must be positive");
      ctx->opt_kbest_scratch_mb = value;
      return CML_OK;
    case CML_OPT_FREE_BUILD_SCRATCH_MB:
      CML_REQUIRE(value > 0, CML_ERR_ARG, "CML_OPT_FREE_BUILD_SCRATCH_MB must be positive");
      ctx->opt_free_build_scratch_mb = value;
      return CML_OK;
    default: ctx->err = "unknown option"; return CML_ERR_ARG;
  }
}

// -------------------------------------------------------------------------------------------------
// model
// -------------------------------------------------------------------------------------------------
static void build_csr(uint32_t n_keys, const std::vector<uint32_t>& key_of, std::vector<uint32_t>& off,
                      std::vector<uint32_t>& members) {
  off.assign(n_keys + 1, 0);
  for (uint32_t k : key_of)
    if (k != CML_NO_GROUP) ++off[k + 1];
  for (uint32_t i = 0; i < n_keys; ++i) off[i + 1] += off[i];
  members.resize(off[n_keys]);
  std::vector<uint32_t> cur(off.begin(), off.end() - 1);
  for (uint32_t p = 0; p < key_of.size(); ++p)
    if (key_of[p] != CML_NO_GROUP) members[cur[key_of[p]]++] = p;
}

extern "C" int cml_set_model(cml_ctx* ctx, const cml_model* m) {
  if (!ctx || !m) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  CML_REQUIRE(ctx->batches.empty(), CML_ERR_STATE, "cml_set_model after cml_add_trellises: clear the trellises first");
  CML_REQUIRE(m->n_arcs > 0 && m->n_params > 0, CML_ERR_ARG, "empty model");
  CML_REQUIRE(m->param_group && m->param_tie, CML_ERR_ARG, "param_group / param_tie are required");
  const bool trivial = (m->chain_off == nullptr);
  CML_REQUIRE(!trivial || m->n_arcs == m->n_params, CML_ERR_ARG, "trivial cascade needs n_arcs == n_params");
  std::vector<uint32_t> pg(m->param_group, m->param_group + m->n_params), tie_key(m->n_params);
  for (uint32_t p = 0; p < m->n_params; ++p) {
    CML_REQUIRE(pg[p] == CML_NO_GROUP || pg[p] < m->n_groups, CML_ERR_ARG, "param_group out of range");
    const uint32_t t = m->param_tie[p];
    CML_REQUIRE(t == CML_NO_GROUP || t <= m->n_ties, CML_ERR_ARG, "param_tie out of range");
    tie_key[p] = (t == CML_NO_GROUP || t == CML_LOCKED_GROUP) ? CML_NO_GROUP : t - 1;
  }
  if (!trivial) {
    CML_REQUIRE(m->chain_param != nullptr, CML_ERR_ARG, "chain_param missing");
    CML_REQUIRE(m->chain_off[0] == 0, CML_ERR_ARG, "chain_off[0] must be 0");
    for (uint32_t a = 0; a < m->n_arcs; ++a)
      CML_REQUIRE(m->chain_off[a] <= m->chain_off[a + 1], CML_ERR_ARG, "chain_off not monotone");
    for (uint32_t k = 0; k < m->chain_off[m->n_arcs]; ++k)
      CML_REQUIRE(m->chain_param[k] < m->n_params, CML_ERR_ARG, "chain_param out of range");
  }
  std::vector<uint32_t> goff, gmem, toff, tmem;
  build_csr(m->n_groups, pg, goff, gmem);
  build_csr(m->n_ties, tie_key, toff, tmem);
  ctx->max_group_size = 0;
  for (uint32_t g = 0; g < m->n_groups; ++g) ctx->max_group_size = std::max(ctx->max_group_size, goff[g + 1] - goff[g]);

  // Count slots.  The expected count of an arc is only ever used through the UNLOCKED parameters of
  // its chain (cascade.h:286-325 distribute_counts skips locked arcs), so arcs whose chains have the
  // same unlocked parameters can share one accumulator: the cipher's 19,683 composed arcs collapse onto
  // its 729 channel parameters, and arcs with fully locked chains need no accumulator at all.
  std::vector<uint32_t> arc_slot(m->n_arcs), slot_off, slot_param;
  std::vector<double> slot_prior;
  uint32_t n_slots = 0;
  const bool merge = !trivial && !ctx->opt_arc_counts;
  if (!merge) {
    n_slots = m->n_arcs;
    for (uint32_t a = 0; a < m->n_arcs; ++a) arc_slot[a] = a;
    if (!trivial) {
      slot_off.assign(m->chain_off, m->chain_off + m->n_arcs + 1);
      slot_param.assign(m->chain_param, m->chain_param + m->chain_off[m->n_arcs]);
    }
    if (m->arc_prior) slot_prior.assign(m->arc_prior, m->arc_prior + m->n_arcs);
  } else {
    std::map<std::vector<uint32_t>, uint32_t> ids;
    slot_off.push_back(0);
    std::vector<uint32_t> key;
    for (uint32_t a = 0; a < m->n_arcs; ++a) {
      key.clear();
      for (uint32_t k = m->chain_off[a]; k < m->chain_off[a + 1]; ++k)
        if (m->param_tie[m->chain_param[k]] != CML_LOCKED_GROUP) key.push_back(m->chain_param[k]);
      if (key.empty()) {
        arc_slot[a] = kPadNone;
        continue;
      }
      auto ins = ids.emplace(key, n_slots);
      if (ins.second) {
        ++n_slots;
        slot_param.insert(slot_param.end(), key.begin(), key.end());
        slot_off.push_back((uint32_t)slot_param.size());
        slot_prior.push_back(0.);
      }
      arc_slot[a] = ins.first->second;
      if (m->arc_prior) slot_prior[arc_slot[a]] += m->arc_prior[a];
    }
    if (n_slots == 0) {  // nothing trainable: keep one dummy slot so buffers are non-empty
      n_slots = 1;
      slot_off.push_back(0);
      slot_prior.push_back(0.);
    }
    if (!m->arc_prior) slot_prior.clear();
  }

  // Arc classes (factored arc weights, SCALED-space wide / lane kernels).  A class is a multiset of parameters;
  // its weight is their product and its count slot is the slot of its unlocked parameters.  Every arc gets a FULL
  // class (its whole chain) and, when the chain has two or more parameters, a STATE part (the chain's last
  // parameter: for LM o channel cascades the channel arc) and a REST part.  When all arcs entering a lattice state
  // have the same state part, the flattener stores it once per state and the arc records carry the rest part:
  // alpha[dst] = V[state part] * sum alpha[src] * U[rest part], and the expected count of the state part is the
  // state posterior (one accumulation per state instead of one per arc; cascade.h:286-325 adds an arc's count
  // to every parameter of its chain, so the per-parameter totals are unchanged).  Class ids and slots depend on
  // the model only, so every rank of a multi-GPU job builds the same reduce buffer.
  {
    ctx->factored = !ctx->opt_no_factor;
    ctx->cls_off.assign(1, 0);
    ctx->cls_param.clear();
    ctx->cls_slot.clear();
    ctx->arc_fcls.assign(m->n_arcs, kPadNone);
    ctx->arc_ucls.assign(m->n_arcs, kPadNone);
    ctx->arc_vcls.assign(m->n_arcs, kPadNone);
    {
      if (!merge || !ctx->factored) {  // class a = arc a with the arc's own slot, no state parts
        ctx->factored = false;
        for (uint32_t a = 0; a < m->n_arcs; ++a) {
          if (trivial)
            ctx->cls_param.push_back(a);
          else
            ctx->cls_param.insert(ctx->cls_param.end(), m->chain_param + m->chain_off[a],
                                  m->chain_param + m->chain_off[a + 1]);
          ctx->cls_off.push_back((uint32_t)ctx->cls_param.size());
          ctx->cls_slot.push_back(arc_slot[a]);
          ctx->arc_fcls[a] = ctx->arc_ucls[a] = a;
        }
      } else {
        std::unordered_map<std::string, uint32_t> cls_ids;
        std::map<std::vector<uint32_t>, uint32_t> slot_ids;  // unlocked parameter set -> slot (existing slots first)
        for (uint32_t sl = 0; sl + 1 < slot_off.size(); ++sl)
          if (slot_off[sl + 1] > slot_off[sl]) {
            std::vector<uint32_t> k(slot_param.begin() + slot_off[sl], slot_param.begin() + slot_off[sl + 1]);
            std::sort(k.begin(), k.end());
            slot_ids.emplace(std::move(k), sl);
          }
        std::vector<uint32_t> key, ukey;
        auto intern = [&](const uint32_t* p, size_t n) -> uint32_t {
          key.assign(p, p + n);
          std::sort(key.begin(), key.end());
          std::string k((const char*)key.data(), key.size() * sizeof(uint32_t));
          auto ins = cls_ids.emplace(std::move(k), (uint32_t)ctx->cls_slot.size());
          if (!ins.second) return ins.first->second;
          ctx->cls_param.insert(ctx->cls_param.end(), key.begin(), key.end());
          ctx->cls_off.push_back((uint32_t)ctx->cls_param.size());
          ukey.clear();
          for (uint32_t q : key)
            if (m->param_tie[q] != CML_LOCKED_GROUP) ukey.push_back(q);
          uint32_t sl = kPadNone;
          if (!ukey.empty()) {
            auto it = slot_ids.find(ukey);  // (keys: sorted unlocked parameter sets)
            if (it == slot_ids.end()) {
              sl = n_slots++;
              slot_ids.emplace(ukey, sl);
              slot_param.insert(slot_param.end(), ukey.begin(), ukey.end());
              slot_off.push_back((uint32_t)slot_param.size());
              if (!slot_prior.empty()) slot_prior.push_back(0.);
            } else
              sl = it->second;
          }
          ctx->cls_slot.push_back(sl);
          return ins.first->second;
        };
        for (uint32_t a = 0; a < m->n_arcs; ++a) {
          const uint32_t* c = m->chain_param + m->chain_off[a];
          const size_t n = m->chain_off[a + 1] - m->chain_off[a];
          ctx->arc_fcls[a] = intern(c, n);
          if (n >= 2) {
            ctx->arc_vcls[a] = intern(c + n - 1, 1);
            ctx->arc_ucls[a] = intern(c, n - 1);
          } else
            ctx->arc_ucls[a] = ctx->arc_fcls[a];
        }
      }
    }
    ctx->a_of_cls.assign(ctx->cls_slot.size(), kPadNone);
    ctx->v_of_cls.assign(ctx->cls_slot.size(), kPadNone);
    ctx->a_list.clear();
    ctx->v_list.clear();
    ctx->a_occ.clear();
    ctx->v_occ.clear();
    ctx->cls_dirty = true;
  }

  cudaStream_t s = ctx->stream;
  ctx->dense.reset();
  ctx->h_param_tie.assign(m->param_tie, m->param_tie + m->n_params);
  if (!trivial) {
    ctx->h_chain_off.assign(m->chain_off, m->chain_off + m->n_arcs + 1);
    ctx->h_chain_param.assign(m->chain_param, m->chain_param + m->chain_off[m->n_arcs]);
  } else {
    ctx->h_chain_off.clear();
    ctx->h_chain_param.clear();
  }
  if (m->arc_prior)
    ctx->h_arc_prior.assign(m->arc_prior, m->arc_prior + m->n_arcs);
  else
    ctx->h_arc_prior.clear();
  ctx->trivial = trivial;
  ctx->n_arcs = m->n_arcs;
  ctx->n_params = m->n_params;
  ctx->n_groups = m->n_groups;
  ctx->n_ties = m->n_ties;
  ctx->n_slots = n_slots;
  ctx->slots_are_arcs = !merge;
  ctx->h_arc_slot = arc_slot;
  ctx->h_perm.resize((size_t)m->n_arcs + 1);
  {
    std::vector<uint32_t> order(m->n_arcs);
    for (uint32_t a = 0; a < m->n_arcs; ++a) order[a] = a;
    if (m->arc_locality_key)
      std::stable_sort(order.begin(), order.end(),
                       [&](uint32_t x, uint32_t y) { return m->arc_locality_key[x] < m->arc_locality_key[y]; });
    for (uint32_t i = 0; i < m->n_arcs; ++i) ctx->h_perm[order[i]] = i;
    ctx->h_perm[m->n_arcs] = m->n_arcs;  // the padding arc
    ctx->h_slot_internal.assign((size_t)m->n_arcs + 1, kPadNone);
    for (uint32_t a = 0; a < m->n_arcs; ++a) ctx->h_slot_internal[ctx->h_perm[a]] = arc_slot[a];
  }
  ctx->slot_occ.assign(n_slots, 0);
  ctx->hot_dirty = true;
  if (!trivial) {
    CML_CUDA(ctx->chain_off.upload(m->chain_off, m->n_arcs + 1, s));
    CML_CUDA(ctx->chain_param.upload(m->chain_param, m->chain_off[m->n_arcs], s));
    CML_CUDA(ctx->slot_off.upload(slot_off.data(), slot_off.size(), s));
    CML_CUDA(ctx->slot_param.upload(slot_param.data(), slot_param.size(), s));
  } else {
    ctx->chain_off.release();
    ctx->chain_param.release();
    ctx->slot_off.release();
    ctx->slot_param.release();
  }
  CML_CUDA(ctx->arc_slot.upload(arc_slot.data(), arc_slot.size(), s));
  CML_CUDA(ctx->arc_perm.upload(ctx->h_perm.data(), ctx->h_perm.size(), s));
  ctx->have_prior = !slot_prior.empty();
  if (ctx->have_prior) CML_CUDA(ctx->slot_prior.upload(slot_prior.data(), slot_prior.size(), s));
  ctx->have_add = m->group_add != nullptr && m->n_groups > 0;
  if (ctx->have_add) CML_CUDA(ctx->group_add.upload(m->group_add, m->n_groups, s));
  CML_CUDA(ctx->param_group.upload(pg.data(), m->n_params, s));
  CML_CUDA(ctx->param_tie.upload(m->param_tie, m->n_params, s));
  CML_CUDA(ctx->group_off.upload(goff.data(), goff.size(), s));
  CML_CUDA(ctx->group_members.upload(gmem.data(), gmem.size(), s));
  CML_CUDA(ctx->tie_off.upload(toff.data(), toff.size(), s));
  CML_CUDA(ctx->tie_members.upload(tmem.data(), tmem.size(), s));
  CML_CUDA(ctx->ln_w.alloc(m->n_params));
  for (auto& sn : ctx->snap) CML_CUDA(sn.alloc(m->n_params));
  CML_CUDA(ctx->acc.alloc(m->n_params));
  CML_CUDA(ctx->u.alloc(m->n_params));
  CML_CUDA(ctx->old.alloc(m->n_params));
  CML_CUDA(ctx->arc_lnw.alloc(m->n_arcs));
  CML_CUDA(ctx->arc_w_real.alloc(((size_t)m->n_arcs + 1) * (ctx->precision / 8)));
  CML_CUDA(ctx->arc_ws.alloc(((size_t)m->n_arcs + 1) * (ctx->precision == 64 ? 16 : 8)));
  CML_CUDA(ctx->gsum.alloc(std::max<uint32_t>(1, m->n_groups)));
  CML_CUDA(ctx->glocked.alloc(std::max<uint32_t>(1, m->n_groups)));
  CML_CUDA(ctx->tie_arc.alloc(std::max<uint32_t>(1, m->n_ties)));
  CML_CUDA(ctx->tie_state.alloc(std::max<uint32_t>(1, m->n_ties)));
  CML_CUDA(ctx->tie_maxl.alloc(std::max<uint32_t>(1, m->n_ties)));
  CML_CUDA(ctx->maxchg.alloc(1));
  CML_CUDA(ctx->reduce_own.alloc((size_t)n_slots + 3));
  ctx->reduce = ctx->reduce_own.p;
  ctx->reduce_n = (uint64_t)n_slots + 3;
  CML_CUDA(cudaMemsetAsync(ctx->reduce, 0, ctx->reduce_n * sizeof(double), s));
  CML_CUDA(cudaStreamSynchronize(s));  // the host staging vectors go out of scope
  ctx->have_model = true;
  ctx->have_params = false;
  ctx->graph_dirty = true;
  return CML_OK;
}

extern "C" int cml_set_params(cml_ctx* ctx, const double* ln_w) {
  if (!ctx || !ln_w) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ctx->ln_w.p, ln_w, ctx->n_params * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->have_params = true;
  return CML_OK;
}

extern "C" int cml_get_params(cml_ctx* ctx, double* ln_w) {
  if (!ctx || !ln_w) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_params, CML_ERR_STATE, "no parameters set");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ln_w, ctx->ln_w.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" int cml_snapshot_params(cml_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot > 3) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_params, CML_ERR_STATE, "no parameters set");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ctx->snap[slot].p, ctx->ln_w.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice,
                           ctx->stream));
  return CML_OK;
}

extern "C" int cml_restore_params(cml_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot > 3) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_params, CML_ERR_STATE, "no parameters set");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ctx->ln_w.p, ctx->snap[slot].p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice,
                           ctx->stream));
  return CML_OK;
}

// -------------------------------------------------------------------------------------------------
// trellis flattening: reference-order adjacency lists -> layered CSR / level-sliced ELL
// -------------------------------------------------------------------------------------------------
namespace {

struct FlatEx {  // per-example facts discovered in pass 1
  uint32_t n_levels = 0;
  bool cycle = false;      // the lattice has a cycle: laid out in the reference's DFS order (CLS_CYCLIC)
  uint32_t back_edges = 0;
  bool ell = false;        // eligible for the ELL kernel
  uint32_t g_class = 0;    // index into kEllG
  uint32_t ring_need = 0;  // max index distance of an arc + max level width + 1
  uint64_t in_pad = 0, out_pad = 0;  // ELL record counts (with padding)
  uint32_t width = 0;
  bool lane_ok = false;    // narrow, every arc spans exactly one level: eligible for the lane-per-lattice kernel
  bool lane = false;       // ... and chosen for it
  bool wide_ok = false;    // levels of 9..32 states, degrees <= 255: eligible for the warp-per-lattice kernel
  bool wide = false;       // ... and chosen for it (laid out like an ELL example, records carry arc classes)
};

inline uint32_t pow2ceil(uint32_t v) {
  uint32_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct Scratch {  // per-thread temporaries
  std::vector<uint64_t> occ;
  std::vector<uint32_t> indeg, queue, cnt, lvl_first, lvl_width, lvl_d, lvl_o, lvl_min, lvl_max, ref_of, icur, ocur, order;
  std::vector<uint32_t> vstate, occ_a, occ_v;  // factored records: state part per state; class occurrence counts
};

// pass 1: longest-path levels via Kahn's algorithm; level_of[] / local_of[]; ELL eligibility
void levelize(uint32_t n, const uint32_t* off, const uint32_t* dst, uint32_t* level_of, uint32_t* local_of, FlatEx& fx,
              Scratch& S, bool want_ell) {
  auto &indeg = S.indeg, &queue = S.queue, &cnt = S.cnt;
  indeg.assign(n, 0);
  for (uint32_t k = 0, e = off[n]; k < e; ++k) ++indeg[dst[k]];
  S.icur.assign(indeg.begin(), indeg.end());  // keep the in-degrees (indeg is consumed below)
  queue.clear();
  for (uint32_t s = 0; s < n; ++s) {
    level_of[s] = 0;
    if (indeg[s] == 0) queue.push_back(s);
  }
  uint32_t maxl = 0;
  for (size_t h = 0; h < queue.size(); ++h) {
    const uint32_t s = queue[h];
    const uint32_t l1 = level_of[s] + 1;
    for (uint32_t k = off[s]; k < off[s + 1]; ++k) {
      const uint32_t d = dst[k];
      if (level_of[d] < l1) level_of[d] = l1;
      if (--indeg[d] == 0) {
        queue.push_back(d);
        if (level_of[d] > maxl) maxl = level_of[d];
      }
    }
  }
  if (queue.size() != n) {
    // A cycle.  The reference warns and carries on (derivations.h:722-729): forward and backward both walk the states in
    // the reverse post-order of a DFS from the start over the stored arc lists (graph.h:241-288), so a back edge's
    // contribution reaches its destination after that state has been propagated.  Same order here: local_of[] = rank in
    // that order, one state per "level"; k_fb_cyclic walks it sequentially.
    fx.cycle = true;
    fx.ell = fx.lane_ok = fx.wide_ok = false;
    auto& begun = S.indeg;   // 0 new, 1 begun, 2 done
    auto& it = S.icur;       // next arc to follow
    begun.assign(n, 0);
    it.assign(n, 0);
    queue.clear();           // DFS stack
    uint32_t rank = n, nback = 0;
    begun[0] = 1;
    it[0] = off[0];
    queue.push_back(0);
    while (!queue.empty()) {
      const uint32_t s = queue.back();
      if (it[s] == off[s + 1]) {
        begun[s] = 2;
        local_of[s] = --rank;  // post-order position, reversed
        queue.pop_back();
        continue;
      }
      const uint32_t d = dst[it[s]++];
      if (begun[d] == 2) continue;
      if (begun[d] == 1) {
        ++nback;
        continue;
      }
      begun[d] = 1;
      it[d] = off[d];
      queue.push_back(d);
    }
    // (every state of a pruned lattice is reachable from the start; anything else keeps the lowest ranks, unreached)
    for (uint32_t s = 0; s < n; ++s)
      if (begun[s] != 2) local_of[s] = --rank;
    for (uint32_t s = 0; s < n; ++s) level_of[s] = local_of[s];
    fx.n_levels = n;
    fx.width = 1;
    fx.back_edges = nback;
    return;
  }
  const uint32_t nl = fx.n_levels = maxl + 1;
  cnt.assign(nl + 1, 0);
  for (uint32_t s = 0; s < n; ++s) ++cnt[level_of[s] + 1];
  uint32_t width = 0;
  for (uint32_t l = 0; l < nl; ++l) {
    width = std::max(width, cnt[l + 1]);
    cnt[l + 1] += cnt[l];
  }
  fx.width = width;
  S.lvl_first.assign(cnt.begin(), cnt.end());
  for (uint32_t s = 0; s < n; ++s) local_of[s] = cnt[level_of[s]]++;  // stable: (level, reference id)
  if (!want_ell) return;
  // ELL eligibility: bounded width / degrees / level spans / ring, modest padding
  auto &ld = S.lvl_d, &lo = S.lvl_o, &lmin = S.lvl_min, &lmax = S.lvl_max;
  ld.assign(nl, 0);
  lo.assign(nl, 0);
  lmin.assign(nl, 0);
  lmax.assign(nl, 0);
  uint32_t maxdist = 0, maxspan = 0;
  for (uint32_t s = 0; s < n; ++s) {
    const uint32_t l = level_of[s];
    ld[l] = std::max(ld[l], S.icur[s]);
    lo[l] = std::max(lo[l], off[s + 1] - off[s]);
    for (uint32_t k = off[s]; k < off[s + 1]; ++k) {
      const uint32_t d = dst[k];
      maxdist = std::max(maxdist, local_of[d] - local_of[s]);
      maxspan = std::max(maxspan, level_of[d] - l);
    }
  }
  uint64_t in_pad = 0, out_pad = 0;
  uint32_t maxdeg = 0;
  for (uint32_t l = 0; l < nl; ++l) {
    const uint32_t w = S.lvl_first[l + 1] - S.lvl_first[l];
    in_pad += (uint64_t)w * ld[l];
    out_pad += (uint64_t)w * lo[l];
    maxdeg = std::max(maxdeg, std::max(ld[l], lo[l]));
  }
  const uint64_t arcs = off[n];
  fx.in_pad = in_pad;
  fx.out_pad = out_pad;
  fx.ring_need = maxdist + width + 1;
  // smallest lane group (R x C) whose per-lane record slots hold every level of the example
  int gc = -1;
  for (int k = 0; k < NELL && gc < 0; ++k) {
    bool fits = true;
    for (uint32_t l = 0; l < nl && fits; ++l) {
      const uint32_t w = S.lvl_first[l + 1] - S.lvl_first[l], deg = std::max(ld[l], lo[l]);
      fits = w <= (uint32_t)kEllCls[k].R && deg <= (uint32_t)(kEllCls[k].C * cmlk::kEllSlots);
    }
    if (fits) gc = k;
  }
  fx.g_class = gc < 0 ? 0 : (uint32_t)gc;
  fx.lane_ok = maxspan <= 1 && 2 * width <= (uint32_t)cmlk::kLaneRing && n < (1u << 30);
  fx.ell = gc >= 0 && width <= 255 && maxdeg <= 255 && maxspan <= 15 && fx.ring_need <= 4096 &&
           in_pad <= arcs + arcs / 2 + 64 && out_pad <= arcs + arcs / 2 + 64;
  fx.wide_ok = width > 8 && width <= 32 && maxdeg <= 255 && maxspan <= 15 && fx.ring_need <= 4096 &&
               in_pad <= arcs + arcs / 2 + 64 && out_pad <= arcs + arcs / 2 + 64;
}

// State part of every lattice state (factored records): the common arc_vcls of its incoming arcs, or kPadNone.
// vs[] is indexed by the caller's state ids.
void state_parts(uint32_t n, const uint32_t* off, const uint32_t* dst, const uint32_t* id,
                 const std::vector<uint32_t>& arc_vcls, std::vector<uint32_t>& vs) {
  constexpr uint32_t kUnset = 0xFFFFFFFEu;
  vs.assign(n, kUnset);
  for (uint32_t k = 0, e = off[n]; k < e; ++k) {
    const uint32_t d = dst[k], v = arc_vcls[id[k]];
    if (vs[d] == kUnset)
      vs[d] = v;
    else if (vs[d] != v)
      vs[d] = kPadNone;
  }
  for (uint32_t s = 0; s < n; ++s)
    if (vs[s] == kUnset) vs[s] = kPadNone;
}

}  // namespace

extern "C" int cml_add_trellises(cml_ctx* ctx, const cml_trellis_batch* b) {
  if (ctx && ctx->dense) {
    ctx->err = "dense-state sequences are resident (cml_add_sequences): call cml_set_model before adding lattices";
    return CML_ERR_STATE;
  }
  if (!ctx || !b) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  CML_REQUIRE(b->n_ex > 0, CML_ERR_ARG, "empty batch");
  CML_REQUIRE(b->ex_states && b->ex_fin && b->arc_off && b->arc_dst && b->arc_id, CML_ERR_ARG, "null array in batch");
  CML_REQUIRE(b->n_ex < 0xFFFFFFFFull, CML_ERR_ARG, "too many examples in one batch");
  cudaSetDevice(ctx->device);
  const uint64_t n_ex = b->n_ex;
  const int rs = ctx->precision / 8;
  const bool scaled = ctx->space == CML_SPACE_SCALED;
  const bool want_ell = scaled && !ctx->opt_no_ell;

  // prefix sums over the caller's arrays
  std::vector<uint64_t> state_base(n_ex + 1), arc_base(n_ex + 1);
  state_base[0] = arc_base[0] = 0;
  for (uint64_t e = 0; e < n_ex; ++e) {
    const uint32_t n = b->ex_states[e];
    CML_REQUIRE(n > 0, CML_ERR_ARG, "example with no states");
    CML_REQUIRE(b->ex_fin[e] < n, CML_ERR_ARG, "ex_fin out of range");
    state_base[e + 1] = state_base[e] + n;
    const uint32_t* off = b->arc_off + state_base[e] + e;
    CML_REQUIRE(off[0] == 0, CML_ERR_ARG, "arc_off must start at 0 for every example");
    arc_base[e + 1] = arc_base[e] + off[n];
  }
  const uint64_t tot_states = state_base[n_ex], tot_arcs = arc_base[n_ex];

  std::unique_ptr<Batch> bt(new Batch());
  bt->n_ex = n_ex;
  bt->n_states = tot_states;
  bt->n_arcs = tot_arcs;
  bt->h_state_base = state_base;
  bt->h_level_of.resize(tot_states);
  bt->h_local_of.resize(tot_states);
  bt->h_nlevels.resize(n_ex);
  std::vector<FlatEx> fx(n_ex);

  // ---- pass 1 (parallel over examples): levels + ELL eligibility
  const unsigned nthr = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  std::atomic<int> bad_cycle{0}, bad_range{0};
  std::vector<uint64_t> batch_occ(ctx->n_slots, 0);  // arcs per count slot in this batch
  const size_t n_cls = ctx->cls_slot.size();
  std::vector<uint64_t> batch_occ_a(n_cls, 0), batch_occ_v(n_cls, 0);  // class occurrences (wide / lane examples)
  std::mutex occ_mutex;
  auto parallel_for = [&](auto&& body) {
    std::atomic<uint64_t> next{0};
    auto work = [&]() {
      Scratch S;
      for (;;) {
        const uint64_t e0 = next.fetch_add(256);
        if (e0 >= n_ex) break;
        for (uint64_t e = e0; e < std::min(n_ex, e0 + 256); ++e) body(e, S);
      }
      if (!S.occ.empty() || !S.occ_a.empty()) {  // merge this thread's occurrence counts
        std::lock_guard<std::mutex> lk(occ_mutex);
        for (size_t i = 0; i < S.occ.size(); ++i) batch_occ[i] += S.occ[i];
        for (size_t i = 0; i < S.occ_a.size(); ++i) batch_occ_a[i] += S.occ_a[i];
        for (size_t i = 0; i < S.occ_v.size(); ++i) batch_occ_v[i] += S.occ_v[i];
      }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nthr; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
  };
  parallel_for([&](uint64_t e, Scratch& S) {
    const uint32_t n = b->ex_states[e];
    const uint32_t* off = b->arc_off + state_base[e] + e;
    const uint32_t* dst = b->arc_dst + arc_base[e];
    const uint32_t* id = b->arc_id + arc_base[e];
    bool ok = true;
    for (uint32_t s = 0; s < n && ok; ++s) ok = off[s] <= off[s + 1];
    for (uint32_t k = 0; k < off[n] && ok; ++k) ok = dst[k] < n && id[k] < ctx->n_arcs;
    if (!ok) {
      bad_range = 1;
      return;
    }
    levelize(n, off, dst, &bt->h_level_of[state_base[e]], &bt->h_local_of[state_base[e]], fx[e], S, want_ell);
    if (fx[e].cycle) bad_cycle = 1;
    bt->h_nlevels[e] = fx[e].n_levels;
  });
  CML_REQUIRE(!bad_range, CML_ERR_ARG, "trellis arc destination or arc id out of range");
  if (bad_cycle)  // cyclic lattices take the reference's sequential order (k_fb_cyclic); the sampler has no such order
    for (uint64_t e = 0; e < n_ex; ++e)
      if (fx[e].cycle) {
        ++bt->cyc_ex;
        bt->cyc_back_edges += fx[e].back_edges;
      }

  // ---- lane-per-lattice layout for corpora of many narrow lattices (cml_kernels_lane.cuh)
  std::vector<uint32_t> lane_list;
  if (want_ell && ctx->opt_lane_min > 0) {
    for (uint64_t e = 0; e < n_ex; ++e)
      if (fx[e].lane_ok) lane_list.push_back((uint32_t)e);
    if (lane_list.size() >= (size_t)ctx->opt_lane_min)
      for (uint32_t e : lane_list) {
        fx[e].lane = true;
        fx[e].ell = false;
      }
    else
      lane_list.clear();
  }

  // ---- warp-per-lattice layout for wide lattices (cml_kernels_wide.cuh): laid out like ELL examples
  if (want_ell && !ctx->opt_no_wide)
    for (uint64_t e = 0; e < n_ex; ++e)
      if (!fx[e].lane && fx[e].wide_ok) {
        fx[e].wide = true;
        fx[e].ell = true;
      }

  // ---- pass 1b (parallel): occurrence counts -- per arc slot for the arc-id layouts, per arc class / state part for
  //      the class layouts (wide, lane)
  parallel_for([&](uint64_t e, Scratch& S) {
    const uint32_t n = b->ex_states[e];
    const uint32_t* off = b->arc_off + state_base[e] + e;
    const uint32_t* dst = b->arc_dst + arc_base[e];
    const uint32_t* id = b->arc_id + arc_base[e];
    if (!(fx[e].wide || fx[e].lane)) {
      if (S.occ.empty()) S.occ.assign(ctx->n_slots, 0);
      for (uint32_t k = 0; k < off[n]; ++k) {
        const uint32_t sl = ctx->h_arc_slot[id[k]];
        if (sl != kPadNone) ++S.occ[sl];
      }
      return;
    }
    if (S.occ_a.empty()) {
      S.occ_a.assign(n_cls, 0);
      S.occ_v.assign(n_cls, 0);
    }
    state_parts(n, off, dst, id, ctx->arc_vcls, S.vstate);
    for (uint32_t k = 0; k < off[n]; ++k)
      ++S.occ_a[S.vstate[dst[k]] != kPadNone ? ctx->arc_ucls[id[k]] : ctx->arc_fcls[id[k]]];
    for (uint32_t st = 0; st < n; ++st)
      if (S.vstate[st] != kPadNone) ++S.occ_v[S.vstate[st]];
  });
  // new classes get the next arc-class / state-class ids (id 0 of either table is the padding / "no class" entry)
  if (ctx->a_list.empty()) {
    ctx->a_list.push_back(kPadNone);
    ctx->v_list.push_back(kPadNone);
    ctx->a_occ.push_back(0);
    ctx->v_occ.push_back(0);
  }
  for (size_t c = 0; c < n_cls; ++c) {
    if (batch_occ_a[c]) {
      if (ctx->a_of_cls[c] == kPadNone) {
        ctx->a_of_cls[c] = (uint32_t)ctx->a_list.size();
        ctx->a_list.push_back((uint32_t)c);
        ctx->a_occ.push_back(0);
        ctx->cls_dirty = true;
      }
      ctx->a_occ[ctx->a_of_cls[c]] += batch_occ_a[c];
      if (ctx->cls_slot[c] != kPadNone) batch_occ[ctx->cls_slot[c]] += batch_occ_a[c];
    }
    if (batch_occ_v[c]) {
      if (ctx->v_of_cls[c] == kPadNone) {
        ctx->v_of_cls[c] = (uint32_t)ctx->v_list.size();
        ctx->v_list.push_back((uint32_t)c);
        ctx->v_occ.push_back(0);
        ctx->cls_dirty = true;
      }
      ctx->v_occ[ctx->v_of_cls[c]] += batch_occ_v[c];
      if (ctx->cls_slot[c] != kPadNone) batch_occ[ctx->cls_slot[c]] += batch_occ_v[c];
    }
  }

  // ---- layout offsets (serial prefix sums), separately for the CSR and the ELL examples
  std::vector<uint64_t> c_lvl(n_ex), c_row(n_ex), c_arc(n_ex), e_in(n_ex), e_out(n_ex), e_meta(n_ex), e_state(n_ex);
  std::vector<uint32_t> slot_of(n_ex);  // index of the example inside its part's descriptor array
  uint64_t n_c = 0, n_e = 0, cl = 0, cr = 0, ca = 0, ei = 0, eo = 0, em = 0, es = 0;
  bt->n_levels = 0;
  for (uint64_t e = 0; e < n_ex; ++e) {
    const uint32_t n = b->ex_states[e], nl = fx[e].n_levels;
    bt->n_levels += nl;
    if (fx[e].lane) continue;
    if (fx[e].ell) {
      slot_of[e] = (uint32_t)n_e++;
      if (fx[e].wide) {  // 16-byte aligned streams (bulk copies), padded to a whole number of 16-byte units
        ei = (ei + 1) & ~1ull;
        eo = (eo + 1) & ~1ull;
        fx[e].in_pad = (fx[e].in_pad + 1) & ~1ull;
        fx[e].out_pad = (fx[e].out_pad + 1) & ~1ull;
      }
      e_in[e] = ei;
      e_out[e] = eo;
      e_meta[e] = em;
      e_state[e] = es;
      ei += fx[e].in_pad;
      eo += fx[e].out_pad;
      em += nl;
      es += n;
    } else {
      slot_of[e] = (uint32_t)n_c++;
      c_lvl[e] = cl;
      c_row[e] = cr;
      c_arc[e] = ca;
      cl += 3ull * nl + 1;
      cr += n + 1;
      ca += arc_base[e + 1] - arc_base[e];
    }
  }
  bt->csr_ex = n_c;
  bt->ell_ex = n_e;
  bt->ell_pad_records = ei + eo;

  std::vector<CmlExDesc> desc(n_c);
  std::vector<uint32_t> h_lvl(cl), h_in_off(cr), h_out_off(cr);
  std::vector<uint2> h_in(ca), h_out(ca);
  std::vector<cmlk::EllDesc> edesc(n_e);
  std::vector<uint4> h_meta(em);
  std::vector<uint2> h_ein(ei), h_eout(eo);
  std::vector<uint32_t> h_evcls;
  {
    bool any_wide = false;
    for (uint64_t e = 0; e < n_ex && !any_wide; ++e) any_wide = fx[e].wide;
    if (any_wide) h_evcls.assign(es, 0u);
  }
  std::vector<double> h_weight(n_ex);
  const uint32_t pad_id = ctx->n_arcs;  // zero-weight padding arc
  const std::vector<uint32_t>& arc_slot = ctx->h_slot_internal;  // indexed by internal arc id
  const std::vector<uint32_t>& perm = ctx->h_perm;

  // ---- pass 2 (parallel): fill
  parallel_for([&](uint64_t e, Scratch& S) {
    const uint32_t n = b->ex_states[e], nl = fx[e].n_levels;
    const uint32_t* off = b->arc_off + state_base[e] + e;
    const uint32_t* dst = b->arc_dst + arc_base[e];
    const uint32_t* id = b->arc_id + arc_base[e];
    const uint32_t* level_of = &bt->h_level_of[state_base[e]];
    const uint32_t* local_of = &bt->h_local_of[state_base[e]];
    const double weight = b->ex_weight ? b->ex_weight[e] : 1.0;
    h_weight[e] = weight;
    if (fx[e].lane) return;  // laid out per tile below
    auto &lfirst = S.lvl_first, &ref_of = S.ref_of;
    lfirst.assign(nl + 1, 0);
    for (uint32_t s = 0; s < n; ++s) ++lfirst[level_of[s] + 1];
    for (uint32_t l = 0; l < nl; ++l) lfirst[l + 1] += lfirst[l];
    ref_of.resize(n);
    for (uint32_t s = 0; s < n; ++s) ref_of[local_of[s]] = s;
    auto &lmin = S.lvl_min, &lmax = S.lvl_max;
    lmin.resize(nl);
    lmax.resize(nl);
    for (uint32_t l = 0; l < nl; ++l) {
      lmin[l] = l ? l - 1 : 0;
      lmax[l] = std::min(nl - 1, l + 1);
    }
    for (uint32_t s = 0; s < n; ++s)
      for (uint32_t k = off[s]; k < off[s + 1]; ++k) {
        const uint32_t ls = level_of[s], ld = level_of[dst[k]];
        if (ls < lmin[ld]) lmin[ld] = ls;
        if (ld > lmax[ls]) lmax[ls] = ld;
      }
    if (!fx[e].ell) {
      // ------------------------------------------------ layered CSR
      uint32_t* lv = &h_lvl[c_lvl[e]];
      for (uint32_t l = 0; l <= nl; ++l) lv[l] = lfirst[l];
      for (uint32_t l = 0; l < nl; ++l) {
        lv[nl + 1 + l] = lmin[l];
        lv[2 * nl + 1 + l] = lmax[l];
      }
      uint32_t* ioff = &h_in_off[c_row[e]];
      uint32_t* ooff = &h_out_off[c_row[e]];
      uint2* ia = &h_in[c_arc[e]];
      uint2* oa = &h_out[c_arc[e]];
      for (uint32_t s = 0; s <= n; ++s) ioff[s] = ooff[s] = 0;
      for (uint32_t s = 0; s < n; ++s) {
        ooff[local_of[s] + 1] = off[s + 1] - off[s];
        for (uint32_t k = off[s]; k < off[s + 1]; ++k) ++ioff[local_of[dst[k]] + 1];
      }
      for (uint32_t s = 0; s < n; ++s) {
        ioff[s + 1] += ioff[s];
        ooff[s + 1] += ooff[s];
      }
      S.icur.assign(ioff, ioff + n);
      for (uint32_t j = 0; j < n; ++j) {  // sources in layered order => in-lists sorted by source (stable)
        const uint32_t s = ref_of[j];
        uint32_t o = ooff[j];
        for (uint32_t k = off[s]; k < off[s + 1]; ++k) {
          const uint32_t dj = local_of[dst[k]];
          oa[o++] = make_uint2(dj, perm[id[k]]);
          ia[S.icur[dj]++] = make_uint2(j, perm[id[k]]);
        }
      }
      CmlExDesc& d = desc[slot_of[e]];
      d.arc_base = c_arc[e];
      d.row_base = c_row[e];
      d.lvl_base = c_lvl[e];
      d.scratch_base = 0;
      d.n_states = n;
      d.n_levels = nl;
      d.fin = local_of[b->ex_fin[e]];
      d.ex_index = (uint32_t)e;
      d.weight = weight;
      d.ln_weight = weight > 0 ? std::log(weight) : -INFINITY;
      return;
    }
    // -------------------------------------------------- level-sliced ELL (wide examples: records carry arc classes)
    const bool wide = fx[e].wide;
    const uint32_t pad_rec = wide ? 0u : pad_id;
    if (wide) {
      state_parts(n, off, dst, id, ctx->arc_vcls, S.vstate);
      uint32_t* vc = &h_evcls[e_state[e]];
      for (uint32_t sr = 0; sr < n; ++sr) vc[local_of[sr]] = S.vstate[sr] == kPadNone ? 0u : ctx->v_of_cls[S.vstate[sr]];
    }
    auto rec_id = [&](uint32_t k) -> uint32_t {  // second word of arc k's record
      if (!wide) return perm[id[k]];
      return ctx->a_of_cls[S.vstate[dst[k]] != kPadNone ? ctx->arc_ucls[id[k]] : ctx->arc_fcls[id[k]]];
    };
    auto &ld = S.lvl_d, &lo = S.lvl_o;
    ld.assign(nl, 0);
    lo.assign(nl, 0);
    S.indeg.assign(n, 0);  // in-degree by layered index
    for (uint32_t s = 0; s < n; ++s) {
      lo[level_of[s]] = std::max(lo[level_of[s]], off[s + 1] - off[s]);
      for (uint32_t k = off[s]; k < off[s + 1]; ++k) ++S.indeg[local_of[dst[k]]];
    }
    for (uint32_t j = 0; j < n; ++j) {
      const uint32_t l = level_of[ref_of[j]];
      ld[l] = std::max(ld[l], S.indeg[j]);
    }
    uint4* meta = &h_meta[e_meta[e]];
    uint2* ein = &h_ein[e_in[e]];
    uint2* eout = &h_eout[e_out[e]];
    uint32_t in_off = 0, out_off = 0;
    for (uint32_t l = 0; l < nl; ++l) {
      const uint32_t w = lfirst[l + 1] - lfirst[l];
      meta[l].x = in_off;
      meta[l].y = out_off;
      meta[l].z = lfirst[l];
      meta[l].w = w | (ld[l] << 8) | (lo[l] << 16) | ((l - lmin[l]) << 24) | ((lmax[l] - l) << 28);
      // padding: zero-weight arc from/to a state that is certainly inside the ring window
      const uint2 pin = make_uint2(l ? lfirst[l - 1] : 0, pad_rec);
      const uint2 pout = make_uint2(l + 1 < nl ? lfirst[l + 1] : lfirst[l], pad_rec);
      for (uint64_t k = 0; k < (uint64_t)w * ld[l]; ++k) ein[in_off + k] = pin;
      for (uint64_t k = 0; k < (uint64_t)w * lo[l]; ++k) eout[out_off + k] = pout;
      in_off += w * ld[l];
      out_off += w * lo[l];
    }
    // outgoing blocks: row = source, columns sorted by destination index
    S.icur.assign(n, 0);  // next free in-column per destination (layered index)
    auto& order = S.order;
    for (uint32_t j = 0; j < n; ++j) {  // sources in layered order => in-columns sorted by source
      const uint32_t s = ref_of[j], l = level_of[s];
      const uint32_t w = lfirst[l + 1] - lfirst[l], r = j - lfirst[l];
      const uint32_t deg = off[s + 1] - off[s];
      order.resize(deg);
      for (uint32_t k = 0; k < deg; ++k) order[k] = off[s] + k;
      std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return local_of[dst[x]] < local_of[dst[y]]; });
      for (uint32_t c = 0; c < deg; ++c) {
        const uint32_t k = order[c];
        const uint32_t dj = local_of[dst[k]], dl = level_of[dst[k]];
        const uint32_t rid = rec_id(k);
        eout[meta[l].y + (uint64_t)c * w + r] = make_uint2(dj, rid);
        const uint32_t dw = lfirst[dl + 1] - lfirst[dl], dr = dj - lfirst[dl];
        ein[meta[dl].x + (uint64_t)(S.icur[dj]++) * dw + dr] = make_uint2(j, rid);
      }
    }
    // aggregate flag: no padding in the level's outgoing block and every column feeds one slot
    for (uint32_t l = 0; l < nl && !wide; ++l) {
      const uint32_t w = lfirst[l + 1] - lfirst[l], O = lo[l];
      bool agg = O > 0 && w > 1;
      for (uint32_t c = 0; c < O && agg; ++c) {
        const uint2* col = eout + meta[l].y + (uint64_t)c * w;
        if (col[0].y == pad_id) agg = false;
        const uint32_t s0 = col[0].y == pad_id ? kPadNone : arc_slot[col[0].y];
        for (uint32_t r = 1; r < w && agg; ++r) agg = col[r].y != pad_id && arc_slot[col[r].y] == s0;
      }
      if (agg) meta[l].z |= 0x80000000u;
    }
    cmlk::EllDesc& d = edesc[slot_of[e]];
    d.in_base = e_in[e];
    d.out_base = e_out[e];
    d.meta_base = e_meta[e];
    d.state_base = e_state[e];
    d.level_base = e_meta[e];
    d.n_states = n;
    d.n_levels = nl;
    d.fin = local_of[b->ex_fin[e]];
    d.ex_index = (uint32_t)e;
    d.weight = weight;
    d.fin_level = level_of[b->ex_fin[e]];
    d.pad = 0;
    d.in_len = (uint32_t)fx[e].in_pad;
    d.out_len = (uint32_t)fx[e].out_pad;
  });

  // ---- classes (serial; cheap)
  const size_t per_state = 2 * (size_t)rs + (scaled ? 8 : 0);
  const size_t smem_budget = std::min<size_t>(ctx->smem_optin ? ctx->smem_optin : 48 * 1024, 220 * 1024);
  const uint32_t cta_max_states = (uint32_t)((smem_budget - 64) / per_state);
  std::vector<std::vector<uint32_t>> cls(NCLS), ecls(NELL);
  std::vector<uint32_t> wide_list;
  uint64_t scratch_states = 0, cyc_states = 0;
  for (uint64_t e = 0; e < n_ex; ++e) {
    if (fx[e].lane) continue;
    if (fx[e].wide) {
      wide_list.push_back(slot_of[e]);
      bt->wide_ring = std::max(bt->wide_ring, pow2ceil(fx[e].ring_need));
      bt->wide_arcs += arc_base[e + 1] - arc_base[e];
      bt->wide_records += fx[e].in_pad + fx[e].out_pad;
      continue;
    }
    if (fx[e].ell) {
      ecls[fx[e].g_class].push_back(slot_of[e]);
      bt->ell_ring[fx[e].g_class] = std::max(bt->ell_ring[fx[e].g_class], pow2ceil(fx[e].ring_need));
      bt->ell_arcs += arc_base[e + 1] - arc_base[e];
      continue;
    }
    const uint32_t n = b->ex_states[e];
    int c = -1;
    if (fx[e].cycle) {
      c = CLS_CYCLIC;
      desc[slot_of[e]].scratch_base = cyc_states;
      cyc_states += n;
    } else if (fx[e].width <= 96) {
      for (int i = 0; i < NWARPCLS; ++i)
        if (n <= kWarpCaps[i]) {
          c = CLS_WARP0 + i;
          break;
        }
    }
    if (c < 0) {
      if (n <= cta_max_states) {
        c = CLS_CTA;
        bt->cta_cap = std::max(bt->cta_cap, n);
      } else {
        c = CLS_GLOBAL;
        desc[slot_of[e]].scratch_base = scratch_states;
        scratch_states += n;
      }
    }
    cls[c].push_back(slot_of[e]);
  }
  std::vector<uint32_t> ex_list, ell_list;
  for (int c = 0; c < NCLS; ++c) {
    bt->cls_begin[c] = (uint32_t)ex_list.size();
    std::stable_sort(cls[c].begin(), cls[c].end(), [&](uint32_t x, uint32_t y) { return desc[x].n_levels > desc[y].n_levels; });
    ex_list.insert(ex_list.end(), cls[c].begin(), cls[c].end());
  }
  bt->cls_begin[NCLS] = (uint32_t)ex_list.size();
  for (int c = 0; c < NELL; ++c) {
    bt->ell_begin[c] = (uint32_t)ell_list.size();
    // longest first; neighbours in a warp then have similar level counts (less sub-warp divergence)
    std::stable_sort(ecls[c].begin(), ecls[c].end(), [&](uint32_t x, uint32_t y) { return edesc[x].n_levels > edesc[y].n_levels; });
    ell_list.insert(ell_list.end(), ecls[c].begin(), ecls[c].end());
  }
  bt->ell_begin[NELL] = (uint32_t)ell_list.size();
  // wide examples: most records first (a persistent warp takes every n-th entry of the list)
  std::stable_sort(wide_list.begin(), wide_list.end(), [&](uint32_t x, uint32_t y) { return edesc[x].n_states > edesc[y].n_states; });
  bt->wide_ex = wide_list.size();

  // ---- lane tiles: 32 lattices of similar size per tile, streams aligned by state ordinal
  std::vector<cmlk::LaneTile> h_tile;
  std::vector<uint2> h_lfw, h_lbw;
  std::vector<uint32_t> h_lex, h_lfin, h_lnlev, h_lvcls;
  std::vector<double> h_lweight;
  uint64_t lane_states = 0, lane_levels = 0;
  if (!lane_list.empty()) {
    constexpr uint32_t U = cmlk::kLaneU;
    std::stable_sort(lane_list.begin(), lane_list.end(), [&](uint32_t x, uint32_t y) {
      return b->ex_states[x] != b->ex_states[y] ? b->ex_states[x] > b->ex_states[y]
                                                 : arc_base[x + 1] - arc_base[x] > arc_base[y + 1] - arc_base[y];
    });
    const uint32_t n_tiles = (uint32_t)((lane_list.size() + 31) / 32);
    h_tile.resize(n_tiles);
    h_lex.assign((size_t)n_tiles * 32, 0xFFFFFFFFu);
    h_lfin.assign((size_t)n_tiles * 32, 0xFFFFFFFFu);
    h_lnlev.assign((size_t)n_tiles * 32, 1);
    h_lweight.assign((size_t)n_tiles * 32, 0.);
    std::vector<std::vector<uint32_t>> rin(n_tiles), rout(n_tiles);  // rows per state ordinal (tile maxima)
    auto tile_for = [&](auto&& body) {
      std::atomic<uint32_t> next{0};
      auto work = [&]() {
        for (;;) {
          const uint32_t t = next.fetch_add(1);
          if (t >= n_tiles) break;
          body(t);
        }
      };
      std::vector<std::thread> th;
      for (unsigned k = 1; k < nthr; ++k) th.emplace_back(work);
      work();
      for (auto& k : th) k.join();
    };
    // phase A: per-ordinal maxima of the in / out degrees
    tile_for([&](uint32_t t) {
      uint32_t nmax = 0, nlmax = 0;
      for (uint32_t l = 0; l < 32 && (size_t)t * 32 + l < lane_list.size(); ++l) {
        const uint32_t e = lane_list[(size_t)t * 32 + l];
        nmax = std::max(nmax, b->ex_states[e]);
        nlmax = std::max(nlmax, fx[e].n_levels);
      }
      auto &ri = rin[t], &ro = rout[t];
      ri.assign(nmax, 0);
      ro.assign(nmax, 0);
      std::vector<uint32_t> ind;
      for (uint32_t l = 0; l < 32 && (size_t)t * 32 + l < lane_list.size(); ++l) {
        const uint32_t e = lane_list[(size_t)t * 32 + l], n = b->ex_states[e];
        const uint32_t* off = b->arc_off + state_base[e] + e;
        const uint32_t* dst = b->arc_dst + arc_base[e];
        const uint32_t* local_of = &bt->h_local_of[state_base[e]];
        ind.assign(n, 0);
        for (uint32_t sr = 0; sr < n; ++sr) {
          ro[local_of[sr]] = std::max(ro[local_of[sr]], off[sr + 1] - off[sr]);
          for (uint32_t k = off[sr]; k < off[sr + 1]; ++k) ++ind[local_of[dst[k]]];
        }
        for (uint32_t j = 0; j < n; ++j) ri[j] = std::max(ri[j], ind[j]);
      }
      uint64_t rf = 0, rb = 0;
      for (uint32_t j = 0; j < nmax; ++j) {
        if (j) rf += (ri[j] = std::max(1u, ri[j]));
        rb += (ro[j] = std::max(1u, ro[j]));
      }
      cmlk::LaneTile& T = h_tile[t];
      T.rows_f = (uint32_t)((rf + U - 1) / U * U);
      T.rows_b = (uint32_t)((rb + U - 1) / U * U);
      T.n_states = nmax;
      T.n_levels = nlmax;
    });
    uint64_t fo = 0, bo = 0;
    for (uint32_t t = 0; t < n_tiles; ++t) {
      cmlk::LaneTile& T = h_tile[t];
      T.fw_base = fo * 32;
      T.bw_base = bo * 32;
      T.st_base = lane_states * 32;
      T.lv_base = lane_levels * 32;
      fo += T.rows_f;
      bo += T.rows_b;
      lane_states += T.n_states;
      lane_levels += T.n_levels;
    }
    const uint2 padrec = make_uint2(0u, 0u);  // arc class 0: the zero-weight padding class
    h_lfw.assign((size_t)(fo + 2 * U) * 32, padrec);  // + the prefetch tail
    h_lbw.assign((size_t)(bo + 2 * U) * 32, padrec);
    h_lvcls.assign((size_t)(lane_states + 2) * 32, 0u);  // state class 0: no state part (+ the prefetch tail)
    // phase B: fill
    tile_for([&](uint32_t t) {
      const cmlk::LaneTile& T = h_tile[t];
      const auto &ri = rin[t], &ro = rout[t];
      std::vector<uint32_t> rowf(T.n_states + 1, 0), rowb(T.n_states + 1, 0);  // first row of every ordinal
      for (uint32_t j = 1; j < T.n_states; ++j) rowf[j + 1] = rowf[j] + ri[j];
      {
        uint32_t r = 0;
        for (uint32_t j = T.n_states; j-- > 0;) {
          rowb[j] = r;
          r += ro[j];
        }
      }
      uint2* fwp = &h_lfw[T.fw_base];
      uint2* bwp = &h_lbw[T.bw_base];
      // the LAST flag closes every ordinal in every lane (also in padding / empty lanes)
      for (uint32_t l = 0; l < 32; ++l) {
        for (uint32_t j = 1; j < T.n_states; ++j) fwp[(size_t)(rowf[j] + ri[j] - 1) * 32 + l].x |= cmlk::kLaneLast;
        for (uint32_t j = 0; j < T.n_states; ++j) bwp[(size_t)(rowb[j] + ro[j] - 1) * 32 + l].x |= cmlk::kLaneLast;
      }
      std::vector<uint32_t> cur, lfirst, vstate;
      for (uint32_t l = 0; l < 32 && (size_t)t * 32 + l < lane_list.size(); ++l) {
        const uint32_t e = lane_list[(size_t)t * 32 + l], n = b->ex_states[e], nl = fx[e].n_levels;
        const uint32_t* off = b->arc_off + state_base[e] + e;
        const uint32_t* dst = b->arc_dst + arc_base[e];
        const uint32_t* id = b->arc_id + arc_base[e];
        const uint32_t* level_of = &bt->h_level_of[state_base[e]];
        const uint32_t* local_of = &bt->h_local_of[state_base[e]];
        const size_t li = (size_t)t * 32 + l;
        h_lex[li] = e;
        h_lfin[li] = local_of[b->ex_fin[e]];
        h_lnlev[li] = nl;
        h_lweight[li] = b->ex_weight ? b->ex_weight[e] : 1.0;
        lfirst.assign(nl + 1, 0);
        for (uint32_t sr = 0; sr < n; ++sr) ++lfirst[level_of[sr] + 1];
        for (uint32_t L = 0; L < nl; ++L) lfirst[L + 1] += lfirst[L];
        cur.assign(n, 0);
        state_parts(n, off, dst, id, ctx->arc_vcls, vstate);
        for (uint32_t sr = 0; sr < n; ++sr)
          h_lvcls[T.st_base + (size_t)local_of[sr] * 32 + l] = vstate[sr] == kPadNone ? 0u : ctx->v_of_cls[vstate[sr]];
        for (uint32_t sr = 0; sr < n; ++sr) {
          const uint32_t j = local_of[sr];
          for (uint32_t k = off[sr]; k < off[sr + 1]; ++k) {
            const uint32_t dj = local_of[dst[k]];
            const uint32_t ia = ctx->a_of_cls[vstate[dst[k]] != kPadNone ? ctx->arc_ucls[id[k]] : ctx->arc_fcls[id[k]]];
            uint2& f = fwp[(size_t)(rowf[dj] + cur[dj]++) * 32 + l];
            f.x = (f.x & cmlk::kLaneLast) | j;
            f.y = ia;
            uint2& g = bwp[(size_t)(rowb[j] + (k - off[sr])) * 32 + l];
            g.x = (g.x & cmlk::kLaneLast) | dj;
            g.y = ia;
          }
        }
        for (uint32_t L = 0; L < nl; ++L) {
          const uint32_t hi = lfirst[L + 1] - 1, lo = lfirst[L];  // last / first state of the level
          if (hi >= 1) fwp[(size_t)(rowf[hi] + ri[hi] - 1) * 32 + l].x |= cmlk::kLaneLevelEnd;
          bwp[(size_t)(rowb[lo] + ro[lo] - 1) * 32 + l].x |= cmlk::kLaneLevelEnd;
        }
      }
    });
    {
      uint32_t wmax = 0;
      for (uint32_t e : lane_list) wmax = std::max(wmax, fx[e].width);
      bt->lane_ring = 2 * wmax <= 8 ? 8 : (uint32_t)cmlk::kLaneRing;
    }
    bt->lane_ex = lane_list.size();
    bt->lane_tiles = n_tiles;
    bt->lane_records = (fo + bo) * 32;
    for (uint32_t e : lane_list) bt->lane_arcs += arc_base[e + 1] - arc_base[e];
  }

  cudaStream_t s = ctx->stream;
  CML_CUDA(bt->ex_lnp.alloc(n_ex));
  CML_CUDA(bt->ex_weight.upload(h_weight.data(), n_ex, s));
  if (n_c) {
    CML_CUDA(bt->desc.upload(desc.data(), n_c, s));
    CML_CUDA(bt->lvl_off.upload(h_lvl.data(), h_lvl.size(), s));
    CML_CUDA(bt->in_off.upload(h_in_off.data(), h_in_off.size(), s));
    CML_CUDA(bt->out_off.upload(h_out_off.data(), h_out_off.size(), s));
    CML_CUDA(bt->in_arc.upload(h_in.data(), h_in.size(), s));
    CML_CUDA(bt->out_arc.upload(h_out.data(), h_out.size(), s));
    CML_CUDA(bt->ex_list.upload(ex_list.data(), ex_list.size(), s));
    if (scratch_states) {
      CML_CUDA(bt->scratch.alloc(scratch_states * 2 * rs));
      if (scaled) CML_CUDA(bt->scratch_lvl.alloc(scratch_states * 2));
    }
    if (cyc_states) CML_CUDA(bt->cyc_scratch.alloc(cyc_states * 2));
  }
  if (n_e) {
    CML_CUDA(bt->edesc.upload(edesc.data(), n_e, s));
    CML_CUDA(bt->lvl_meta.upload(h_meta.data(), h_meta.size(), s));
    CML_CUDA(bt->ell_in.upload(h_ein.data(), h_ein.size(), s));
    CML_CUDA(bt->ell_out.upload(h_eout.data(), h_eout.size(), s));
    CML_CUDA(bt->ell_list.upload(ell_list.data(), ell_list.size(), s));
    if (bt->wide_ex) {
      CML_CUDA(bt->wide_list.upload(wide_list.data(), wide_list.size(), s));
      CML_CUDA(bt->ell_vcls.upload(h_evcls.data(), h_evcls.size(), s));
    }
    CML_CUDA(bt->alpha_g.alloc(es * rs));
    CML_CUDA(bt->lvl_exp.alloc(em * 2));
  }
  if (bt->lane_tiles) {
    CML_CUDA(bt->ltile.upload(h_tile.data(), h_tile.size(), s));
    CML_CUDA(bt->lane_fw.upload(h_lfw.data(), h_lfw.size(), s));
    CML_CUDA(bt->lane_bw.upload(h_lbw.data(), h_lbw.size(), s));
    CML_CUDA(bt->lane_exidx.upload(h_lex.data(), h_lex.size(), s));
    CML_CUDA(bt->lane_fin.upload(h_lfin.data(), h_lfin.size(), s));
    CML_CUDA(bt->lane_nlev.upload(h_lnlev.data(), h_lnlev.size(), s));
    CML_CUDA(bt->lane_weight.upload(h_lweight.data(), h_lweight.size(), s));
    CML_CUDA(bt->lane_vcls.upload(h_lvcls.data(), h_lvcls.size(), s));
    CML_CUDA(bt->lane_alpha.alloc(lane_states * 32 * rs));
    CML_CUDA(bt->lane_lvle.alloc(lane_levels * 32));
  }
  CML_CUDA(cudaStreamSynchronize(s));
  ctx->batches.push_back(std::move(bt));
  ctx->graph_dirty = true;
  if (ctx->slot_occ.size() != ctx->n_slots) ctx->slot_occ.assign(ctx->n_slots, 0);
  for (size_t i = 0; i < batch_occ.size(); ++i) ctx->slot_occ[i] += batch_occ[i];
  ctx->hot_dirty = true;
  return CML_OK;
}

extern "C" int cml_clear_trellises(cml_ctx* ctx) {
  if (!ctx) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->batches.clear();
  ctx->graph_dirty = true;
  ctx->slot_occ.assign(ctx->n_slots, 0);
  ctx->hot_dirty = true;
  return CML_OK;
}

extern "C" int cml_cyclic_stats(cml_ctx* ctx, uint64_t* n_examples, uint64_t* n_back_edges) {
  if (!ctx) return CML_ERR_ARG;
  uint64_t a = 0, b = 0;
  for (auto& bt : ctx->batches) {
    a += bt->cyc_ex;
    b += bt->cyc_back_edges;
  }
  if (n_examples) *n_examples = a;
  if (n_back_edges) *n_back_edges = b;
  return CML_OK;
}
extern "C" int cml_trellis_totals(cml_ctx* ctx, uint64_t* n_ex, uint64_t* n_states, uint64_t* n_arcs,
                                  uint64_t* n_levels) {
  if (!ctx) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0;
  for (auto& bt : ctx->batches) {
    a += bt->n_ex;
    b += bt->n_states;
    c += bt->n_arcs;
    d += bt->n_levels;
  }
  if (n_ex) *n_ex = a;
  if (n_states) *n_states = b;
  if (n_arcs) *n_arcs = c;
  if (n_levels) *n_levels = d;
  return CML_OK;
}

extern "C" int cml_lane_stats(cml_ctx* ctx, uint64_t* lane_examples, uint64_t* lane_arcs, uint64_t* lane_records,
                              uint64_t* tiles) {
  if (!ctx) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0;
  for (auto& bt : ctx->batches) {
    a += bt->lane_ex;
    b += bt->lane_arcs;
    c += bt->lane_records;
    d += bt->lane_tiles;
  }
  if (lane_examples) *lane_examples = a;
  if (lane_arcs) *lane_arcs = b;
  if (lane_records) *lane_records = c;
  if (tiles) *tiles = d;
  return CML_OK;
}

extern "C" int cml_wide_stats(cml_ctx* ctx, uint64_t* wide_examples, uint64_t* wide_arcs, uint64_t* wide_records,
                              uint64_t* arc_classes, uint64_t* state_classes) {
  if (!ctx) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0;
  for (auto& bt : ctx->batches) {
    a += bt->wide_ex;
    b += bt->wide_arcs;
    c += bt->wide_records;
  }
  if (wide_examples) *wide_examples = a;
  if (wide_arcs) *wide_arcs = b;
  if (wide_records) *wide_records = c;
  if (arc_classes) *arc_classes = ctx->a_list.empty() ? 0 : ctx->a_list.size() - 1;
  if (state_classes) *state_classes = ctx->v_list.empty() ? 0 : ctx->v_list.size() - 1;
  return CML_OK;
}

extern "C" int cml_layout_stats(cml_ctx* ctx, uint64_t* ell_examples, uint64_t* ell_arcs, uint64_t* ell_records,
                                uint64_t* csr_examples) {
  if (!ctx) return CML_ERR_ARG;
  uint64_t a = 0, b = 0, c = 0, d = 0;
  for (auto& bt : ctx->batches) {
    a += bt->ell_ex - bt->wide_ex;
    b += bt->ell_arcs;
    c += bt->ell_pad_records - bt->wide_records;
    d += bt->csr_ex;
  }
  if (ell_examples) *ell_examples = a;
  if (ell_arcs) *ell_arcs = b;
  if (ell_records) *ell_records = c;
  if (csr_examples) *csr_examples = d;
  return CML_OK;
}

extern "C" int cml_get_example_layout(cml_ctx* ctx, uint64_t e, uint32_t* n_levels, uint32_t* level_of,
                                      uint32_t* local_of) {
  if (!ctx) return CML_ERR_ARG;
  for (auto& bt : ctx->batches) {
    if (e < bt->n_ex) {
      const uint64_t s0 = bt->h_state_base[e], s1 = bt->h_state_base[e + 1];
      if (n_levels) *n_levels = bt->h_nlevels[e];
      if (level_of) std::memcpy(level_of, &bt->h_level_of[s0], (s1 - s0) * 4);
      if (local_of) std::memcpy(local_of, &bt->h_local_of[s0], (s1 - s0) * 4);
      return CML_OK;
    }
    e -= bt->n_ex;
  }
  ctx->err = "example index out of range";
  return CML_ERR_ARG;
}

// -------------------------------------------------------------------------------------------------
// E-step
// -------------------------------------------------------------------------------------------------
template <typename Real, int R, int C, bool CTA>
static int launch_ell_class(cml_ctx* ctx, Batch& bt, cmlk::EllArgs& A, int c) {
  const uint32_t n = bt.ell_begin[c + 1] - bt.ell_begin[c];
  if (!n) return CML_OK;
  A.ex_list = bt.ell_list.p + bt.ell_begin[c];
  A.n_list = n;
  A.ring = bt.ell_ring[c];
  constexpr int GPB = CTA ? 1 : cmlk::kEllThreads / (R * C);
  const size_t smem = (size_t)cmlk::kEllStages * cmlk::kEllSlots * cmlk::kEllThreads * sizeof(uint2) +
                      (size_t)GPB * A.ring * sizeof(Real);
  auto kern = cmlk::k_fb_ell<Real, R, C, CTA>;
  if (smem > 48 * 1024) CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<cdiv(n, GPB), cmlk::kEllThreads, smem, ctx->stream>>>(A);
  ++ctx->launches;
  ++bt.n_fb_kernels;
  return CML_OK;
}

template <typename Real, bool SCALED>
static int launch_fb(cml_ctx* ctx, Batch& bt) {
  using namespace cmlk;
  if (!bt.ev_fb0) {
    CML_CUDA(cudaEventCreate(&bt.ev_fb0));
    CML_CUDA(cudaEventCreate(&bt.ev_fb1));
  }
  bt.n_fb_kernels = 0;
  if (!ctx->capturing) CML_CUDA(cudaEventRecord(bt.ev_fb0, ctx->stream));
  if (SCALED && bt.ell_ex) {
    EllArgs E;
    E.desc = bt.edesc.p;
    E.lvl_meta = bt.lvl_meta.p;
    E.ell_in = bt.ell_in.p;
    E.ell_out = bt.ell_out.p;
    E.arc_w = ctx->arc_w_real.p;
    E.arc_ws = ctx->arc_ws.p;
    E.sink = cmlk::CountSink{ctx->reduce, ctx->hot_counts.p, ctx->n_hot, ctx->hot_copies - 1};
    E.ex_lnp = bt.ex_lnp.p;
    E.alpha_g = bt.alpha_g.p;
    E.lvl_exp = bt.lvl_exp.p;
    int r;
    if ((r = launch_ell_class<Real, 4, 1, false>(ctx, bt, E, 0))) return r;   // kEllCls[0]
    if ((r = launch_ell_class<Real, 8, 1, false>(ctx, bt, E, 1))) return r;   // kEllCls[1]
    if ((r = launch_ell_class<Real, 4, 4, false>(ctx, bt, E, 2))) return r;   // kEllCls[2]
    if ((r = launch_ell_class<Real, 8, 4, false>(ctx, bt, E, 3))) return r;   // kEllCls[3]
    if ((r = launch_ell_class<Real, 16, 2, false>(ctx, bt, E, 4))) return r;  // kEllCls[4]
    if ((r = launch_ell_class<Real, 32, 1, false>(ctx, bt, E, 5))) return r;  // kEllCls[5]
    if ((r = launch_ell_class<Real, 32, 8, true>(ctx, bt, E, 6))) return r;   // kEllCls[6]
  }
  if (SCALED && bt.wide_ex) {
    WideArgs Wd;
    Wd.desc = bt.edesc.p;
    Wd.ex_list = bt.wide_list.p;
    Wd.n_list = (uint32_t)bt.wide_ex;
    Wd.lvl_meta = bt.lvl_meta.p;
    Wd.ell_in = bt.ell_in.p;
    Wd.ell_out = bt.ell_out.p;
    Wd.st_vcls = bt.ell_vcls.p;
    Wd.a_w = ctx->a_w.p;
    Wd.a_slot = ctx->a_slot.p;
    Wd.v_w = ctx->v_w.p;
    Wd.v_slot = ctx->v_slot.p;
    Wd.n_a = (uint32_t)ctx->a_list.size();
    Wd.n_v = (uint32_t)ctx->v_list.size();
    Wd.any_a_slot = ctx->any_a_slot;
    Wd.sink = cmlk::CountSink{ctx->reduce, ctx->hot_counts.p, ctx->n_hot, ctx->hot_copies - 1};
    Wd.ex_lnp = bt.ex_lnp.p;
    Wd.alpha_g = bt.alpha_g.p;
    Wd.lvl_exp = bt.lvl_exp.p;
    Wd.ring = std::max<uint32_t>(16, bt.wide_ring);
    Wd.no_counts = ctx->opt_no_counts;
    Wd.l2_prefetch = 0;
    Wd.generic_addr = 0;
    if (const char* e = getenv("CML_WIDE_PF")) Wd.l2_prefetch = atoi(e);      // tuning knobs (profiling)
    if (const char* e = getenv("CML_WIDE_GA")) Wd.generic_addr = atoi(e);
    // persistent warps, one CTA per SM: as many warps as shared memory allows (<= 16), trimmed so that the lattices
    // divide evenly over the warps (2,000 cipher lines on 148 SMs: 14 warps per CTA, one lattice per warp)
    const size_t budget = std::min<size_t>(ctx->smem_optin ? ctx->smem_optin : 48 * 1024, 220 * 1024);
    // layout (cml_kernels_wide.cuh): 8 KB alignment slack | chunk buffers | mbarriers | ring alignment slack | rings | tables
    size_t tbl = (((size_t)(Wd.n_a + Wd.n_v) * (sizeof(Real) + 4)) + 127) & ~(size_t)127;
    const size_t ring_bytes = (size_t)Wd.ring * sizeof(Real);
    const size_t per_warp = 64 + (size_t)kWideStages * kWideChunkBytes + ring_bytes;
    const size_t slack = (size_t)kWideStages * kWideChunkBytes + ring_bytes;
    const bool tblsm = tbl + slack + 4 * per_warp <= budget && tbl <= 96 * 1024;
    if (!tblsm) tbl = 0;
    int wmax = (int)std::min<size_t>(16, (budget - tbl - slack) / per_warp);
    CML_REQUIRE(wmax >= 1, CML_ERR_ARG, "wide lattice ring does not fit in shared memory");
    const uint64_t sm = (uint64_t)ctx->sm_count;
    int wpc = wmax;
    {
      double best = -1;
      for (int w = wmax; w >= std::max(1, wmax / 2); --w) {
        const uint64_t slots = sm * (uint64_t)w, waves = (Wd.n_list + slots - 1) / slots;
        const double util = (double)Wd.n_list / (double)(waves * slots) * (0.75 + 0.25 * w / wmax);
        if (util > best) {
          best = util;
          wpc = w;
        }
      }
    }
    if (const char* e = getenv("CML_WIDE_WPC")) wpc = std::max(1, std::min(wmax, atoi(e)));
    Wd.warps_per_cta = (uint32_t)wpc;
    const unsigned grid = (unsigned)std::min<uint64_t>(sm, (Wd.n_list + wpc - 1) / wpc);
    const size_t smem = tbl + slack + (size_t)wpc * per_warp;
    auto kern = tblsm ? k_fb_wide<Real, true> : k_fb_wide<Real, false>;
    if (smem > 48 * 1024) CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    kern<<<grid, wpc * 32, smem, ctx->stream>>>(Wd);
    ++ctx->launches;
    ++bt.n_fb_kernels;
  }
  if (SCALED && bt.lane_tiles) {
    LaneArgs L;
    L.tile = bt.ltile.p;
    L.n_tiles = bt.lane_tiles;
    L.fw = bt.lane_fw.p;
    L.bw = bt.lane_bw.p;
    L.ex = bt.lane_exidx.p;
    L.fin = bt.lane_fin.p;
    L.nlev = bt.lane_nlev.p;
    L.weight = bt.lane_weight.p;
    L.vcls = bt.lane_vcls.p;
    L.a_w = ctx->a_w.p;
    L.a_slot = ctx->a_slot.p;
    L.v_w = ctx->v_w.p;
    L.v_slot = ctx->v_slot.p;
    L.n_a = (uint32_t)ctx->a_list.size();
    L.n_v = (uint32_t)ctx->v_list.size();
    L.sink = cmlk::CountSink{ctx->reduce, ctx->hot_counts.p, ctx->n_hot, ctx->hot_copies - 1};
    L.ex_lnp = bt.ex_lnp.p;
    L.alpha = bt.lane_alpha.p;
    L.lvle = bt.lane_lvle.p;
    L.no_counts = ctx->opt_no_counts;
    // class tables in shared memory when they are small (HMM: the 1k transition classes yes, the 20k emission
    // classes no: those are gathered once per state)
    const size_t tbl_a = (((size_t)L.n_a * (sizeof(Real) + 4)) + 15) & ~(size_t)15;
    const size_t tbl_v = (size_t)L.n_v * (sizeof(Real) + 4);
    const bool ta = tbl_a <= 40 * 1024, tv = tbl_v <= 24 * 1024;
    int minb = 2;
    if (const char* e = getenv("CML_LANE_MINB")) minb = atoi(e);  // tuning knob: 3 = register cap for three resident blocks (measured slower: profiles/round2_D)
    const size_t smem = (size_t)kLaneWarps * kLaneRing * 32 * sizeof(Real) + (ta ? tbl_a : 0) + (tv ? tbl_v : 0);
    auto kern = minb >= 3 ? (ta ? (tv ? k_fb_lane<Real, true, true, 3> : k_fb_lane<Real, true, false, 3>)
                                : (tv ? k_fb_lane<Real, false, true, 3> : k_fb_lane<Real, false, false, 3>))
                          : (ta ? (tv ? k_fb_lane<Real, true, true, 2> : k_fb_lane<Real, true, false, 2>)
                                : (tv ? k_fb_lane<Real, false, true, 2> : k_fb_lane<Real, false, false, 2>));
    if (smem > 48 * 1024) CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    kern<<<cdiv(bt.lane_tiles, kLaneWarps), kLaneWarps * 32, smem, ctx->stream>>>(L);
    ++ctx->launches;
    ++bt.n_fb_kernels;
  }
  if (bt.csr_ex) {
    FbArgs A;
    A.desc = bt.desc.p;
    A.lvl_off = bt.lvl_off.p;
    A.in_off = bt.in_off.p;
    A.in_arc = bt.in_arc.p;
    A.out_off = bt.out_off.p;
    A.out_arc = bt.out_arc.p;
    A.arc_w = ctx->arc_w_real.p;
    A.arc_slot = ctx->arc_slot_code.p;
    A.sink = cmlk::CountSink{ctx->reduce, ctx->hot_counts.p, ctx->n_hot, ctx->hot_copies - 1};
    A.ex_lnp = bt.ex_lnp.p;
    A.scratch = bt.scratch.p;
    A.scratch_lvl = bt.scratch_lvl.p;
    const size_t per_state = 2 * sizeof(Real) + (SCALED ? 2 * sizeof(int) : 0);
    for (int c = 0; c < NWARPCLS; ++c) {
      const uint32_t n = bt.cls_begin[c + 1] - bt.cls_begin[c];
      if (!n) continue;
      A.ex_list = bt.ex_list.p + bt.cls_begin[c];
      A.n_list = n;
      A.cap_states = kWarpCaps[c];
      const size_t smem = 4 * per_state * kWarpCaps[c];
      auto kern = k_fb_warp<Real, SCALED>;
      if (smem > 48 * 1024) CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kern<<<cdiv(n, 4), 128, smem, ctx->stream>>>(A);
      ++ctx->launches;
      ++bt.n_fb_kernels;
    }
    {
      const uint32_t n = bt.cls_begin[CLS_CTA + 1] - bt.cls_begin[CLS_CTA];
      if (n) {
        A.ex_list = bt.ex_list.p + bt.cls_begin[CLS_CTA];
        A.n_list = n;
        A.cap_states = bt.cta_cap;
        const size_t smem = per_state * bt.cta_cap;
        auto kern = k_fb_cta<Real, SCALED, false>;
        if (smem > 48 * 1024)
          CML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<n, 256, smem, ctx->stream>>>(A);
        ++ctx->launches;
        ++bt.n_fb_kernels;
      }
    }
    {
      const uint32_t n = bt.cls_begin[CLS_GLOBAL + 1] - bt.cls_begin[CLS_GLOBAL];
      if (n) {
        A.ex_list = bt.ex_list.p + bt.cls_begin[CLS_GLOBAL];
        A.n_list = n;
        A.cap_states = 0;
        k_fb_cta<Real, SCALED, true><<<n, 256, 0, ctx->stream>>>(A);
        ++ctx->launches;
        ++bt.n_fb_kernels;
      }
    }
    {
      const uint32_t n = bt.cls_begin[CLS_CYCLIC + 1] - bt.cls_begin[CLS_CYCLIC];
      if (n) {  // lattices with a cycle: the reference's sequential walk, one thread per lattice
        A.ex_list = bt.ex_list.p + bt.cls_begin[CLS_CYCLIC];
        A.n_list = n;
        k_fb_cyclic<Real, SCALED><<<cdiv(n, 64), 64, 0, ctx->stream>>>(A, bt.cyc_scratch.p);
        ++ctx->launches;
        ++bt.n_fb_kernels;
      }
    }
  }
  if (!ctx->capturing) CML_CUDA(cudaEventRecord(bt.ev_fb1, ctx->stream));
  k_reduce_lnp<<<std::min<unsigned>(cdiv(bt.n_ex, 256), 4 * ctx->sm_count), 256, 0, ctx->stream>>>(
      bt.ex_lnp.p, bt.ex_weight.p, bt.n_ex, ctx->reduce + ctx->n_slots);
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  return CML_OK;
}

template <typename Real, bool SCALED>
static int launch_arc_weights(cml_ctx* ctx) {
  cmlk::k_arc_weights<Real, SCALED, cmlk::WS<Real>><<<cdiv(ctx->n_arcs + 1, 256), 256, 0, ctx->stream>>>(
      ctx->n_arcs, ctx->trivial ? nullptr : ctx->chain_off.p, ctx->chain_param.p, ctx->ln_w.p, ctx->arc_slot_code.p,
      ctx->arc_perm.p, ctx->arc_lnw.p, (Real*)ctx->arc_w_real.p, (cmlk::WS<Real>*)ctx->arc_ws.p);
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  return CML_OK;
}

// Slot codes: slots that occur at least kHotMinOcc times in the resident lattices become HOT (replicated
// accumulators, see CountSink); at most kHotMaxSlots of them, most frequent first.
static int rebuild_slot_codes(cml_ctx* ctx) {
  uint64_t kHotMinOcc = 4096;
  size_t kHotMaxSlots = 32768;
  if (const char* e = getenv("CML_HOT_MIN_OCC")) kHotMinOcc = (uint64_t)atoll(e);  // tuning knobs (profiling)
  if (const char* e = getenv("CML_HOT_MAX_SLOTS")) kHotMaxSlots = (size_t)atoll(e);
  std::vector<uint32_t> hot;
  for (uint32_t sl = 0; sl < ctx->n_slots && sl < ctx->slot_occ.size(); ++sl)
    if (ctx->slot_occ[sl] >= kHotMinOcc) hot.push_back(sl);
  std::sort(hot.begin(), hot.end(), [&](uint32_t a, uint32_t b) {
    return ctx->slot_occ[a] != ctx->slot_occ[b] ? ctx->slot_occ[a] > ctx->slot_occ[b] : a < b;
  });
  if (hot.size() > kHotMaxSlots) hot.resize(kHotMaxSlots);
  std::vector<uint32_t> hot_index(ctx->n_slots, kPadNone);
  for (uint32_t h = 0; h < hot.size(); ++h) hot_index[hot[h]] = h;
  std::vector<uint32_t> code((size_t)ctx->n_arcs + 1, kPadNone);  // indexed by internal arc id
  for (uint32_t a = 0; a < ctx->n_arcs; ++a) {
    const uint32_t sl = ctx->h_arc_slot[a];
    code[ctx->h_perm[a]] = (sl == kPadNone) ? kPadNone : (hot_index[sl] != kPadNone ? (cmlk::kSlotHot | hot_index[sl]) : sl);
  }
  ctx->n_hot = (uint32_t)hot.size();
  // arc-class / state-class tables of the wide and lane kernels (ids are append-only; entry 0 = padding / no class)
  if (ctx->a_list.size() > 1 || ctx->v_list.size() > 1) {
    auto build = [&](const std::vector<uint32_t>& list, std::vector<uint32_t>& off, std::vector<uint32_t>& par,
                     std::vector<uint32_t>& slc) {
      off.assign(1, 0);
      par.clear();
      slc.clear();
      for (uint32_t i = 0; i < list.size(); ++i) {
        uint32_t sl = kPadNone;
        if (i) {
          const uint32_t c = list[i];
          par.insert(par.end(), ctx->cls_param.begin() + ctx->cls_off[c], ctx->cls_param.begin() + ctx->cls_off[c + 1]);
          sl = ctx->cls_slot[c];
        }
        off.push_back((uint32_t)par.size());
        slc.push_back(sl == kPadNone ? kPadNone : (hot_index[sl] != kPadNone ? (cmlk::kSlotHot | hot_index[sl]) : sl));
      }
    };
    std::vector<uint32_t> off, par, slc;
    build(ctx->a_list, off, par, slc);
    CML_CUDA(ctx->a_off.upload(off.data(), off.size(), ctx->stream));
    CML_CUDA(ctx->a_param.upload(par.data(), par.size(), ctx->stream));
    CML_CUDA(ctx->a_slot.upload(slc.data(), slc.size(), ctx->stream));
    ctx->any_a_slot = 0;
    for (uint32_t c : slc) ctx->any_a_slot |= (c != kPadNone);
    CML_CUDA(cudaStreamSynchronize(ctx->stream));
    build(ctx->v_list, off, par, slc);
    CML_CUDA(ctx->v_off.upload(off.data(), off.size(), ctx->stream));
    CML_CUDA(ctx->v_param.upload(par.data(), par.size(), ctx->stream));
    CML_CUDA(ctx->v_slot.upload(slc.data(), slc.size(), ctx->stream));
    CML_CUDA(cudaStreamSynchronize(ctx->stream));
    CML_CUDA(ctx->a_w.alloc(ctx->a_list.size() * (ctx->precision / 8)));
    CML_CUDA(ctx->v_w.alloc(ctx->v_list.size() * (ctx->precision / 8)));
  }
  ctx->cls_dirty = false;
  CML_CUDA(ctx->arc_slot_code.upload(code.data(), code.size(), ctx->stream));
  CML_CUDA(ctx->hot_slot.upload(hot.data(), hot.size(), ctx->stream));
  if (!getenv("CML_HOT_COPIES")) {
    // many narrow lattices (k_fb_lane) put one fp64 RED per arc on ~1 k arc-class slots: 1,024 replicas instead of 64
    // are worth 12 % of the kernel there (profiles/round2_J); small corpora keep 64 (the fold and the memset scale with it)
    uint64_t lane_arcs = 0;
    for (auto& bt : ctx->batches) lane_arcs += bt->lane_arcs;
    ctx->hot_copies = lane_arcs >= (16ull << 20) ? 1024u : cmlk::kHotCopies;
  }
  CML_CUDA(ctx->hot_counts.alloc(std::max<size_t>(1, (size_t)ctx->n_hot * ctx->hot_copies)));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->hot_dirty = false;
  return CML_OK;
}

extern "C" int cml_estimate_launch(cml_ctx* ctx) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  cudaSetDevice(ctx->device);
  if (ctx->batches.empty() && !ctx->dense && ctx->opt_allow_empty) {
    // an empty shard of a multi-GPU job: zero counts and likelihood terms, the rank still joins the all-reduce
    CML_CUDA(cudaMemsetAsync(ctx->reduce, 0, ctx->reduce_n * sizeof(double), ctx->stream));
    ctx->estimate_pending = true;
    return CML_OK;
  }
  CML_REQUIRE(!ctx->batches.empty() || ctx->dense, CML_ERR_NODERIV,
              "no trellises resident (no training example had a derivation)");
  if (ctx->dense) {
    const int rc = cml_dense_estimate_launch(ctx);
    if (rc) return rc;
    ctx->estimate_pending = true;
    return CML_OK;
  }
  if (ctx->hot_dirty || ctx->cls_dirty) {
    const int rc = rebuild_slot_codes(ctx);
    if (rc) return rc;
  }
  const bool sc = ctx->space == CML_SPACE_SCALED;
  int r;
  if (ctx->precision == 64)
    r = sc ? launch_arc_weights<double, true>(ctx) : launch_arc_weights<double, false>(ctx);
  else
    r = sc ? launch_arc_weights<float, true>(ctx) : launch_arc_weights<float, false>(ctx);
  if (r) return r;
  if (ctx->a_list.size() > 1 || ctx->v_list.size() > 1) {
    const uint32_t na = (uint32_t)ctx->a_list.size(), nv = (uint32_t)ctx->v_list.size();
    if (ctx->precision == 64) {
      cmlk::k_class_weights<double><<<cdiv(na, 256), 256, 0, ctx->stream>>>(na, ctx->a_off.p, ctx->a_param.p, ctx->ln_w.p, 0.,
                                                                            (double*)ctx->a_w.p);
      cmlk::k_class_weights<double><<<cdiv(nv, 256), 256, 0, ctx->stream>>>(nv, ctx->v_off.p, ctx->v_param.p, ctx->ln_w.p, 1.,
                                                                            (double*)ctx->v_w.p);
    } else {
      cmlk::k_class_weights<float><<<cdiv(na, 256), 256, 0, ctx->stream>>>(na, ctx->a_off.p, ctx->a_param.p, ctx->ln_w.p, 0.f,
                                                                           (float*)ctx->a_w.p);
      cmlk::k_class_weights<float><<<cdiv(nv, 256), 256, 0, ctx->stream>>>(nv, ctx->v_off.p, ctx->v_param.p, ctx->ln_w.p, 1.f,
                                                                           (float*)ctx->v_w.p);
    }
    ctx->launches += 2;
    CML_CUDA(cudaGetLastError());
  }
  CML_CUDA(cudaMemsetAsync(ctx->reduce, 0, ctx->reduce_n * sizeof(double), ctx->stream));
  if (ctx->n_hot)
    CML_CUDA(cudaMemsetAsync(ctx->hot_counts.p, 0, (size_t)ctx->n_hot * ctx->hot_copies * sizeof(double), ctx->stream));
  for (auto& bt : ctx->batches) {
    if (ctx->precision == 64)
      r = sc ? launch_fb<double, true>(ctx, *bt) : launch_fb<double, false>(ctx, *bt);
    else
      r = sc ? launch_fb<float, true>(ctx, *bt) : launch_fb<float, false>(ctx, *bt);
    if (r) return r;
  }
  if (ctx->n_hot) {
    cmlk::k_fold_hot<<<cdiv(ctx->n_hot, 256), 256, 0, ctx->stream>>>(ctx->n_hot, ctx->hot_slot.p, ctx->hot_counts.p,
                                                                   ctx->reduce, ctx->hot_copies);
    ++ctx->launches;
    CML_CUDA(cudaGetLastError());
  }
  ctx->estimate_pending = true;
  return CML_OK;
}

extern "C" int cml_estimate_finish(cml_ctx* ctx, cml_estimate_result* out) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->estimate_pending, CML_ERR_STATE, "cml_estimate_launch first");
  cudaSetDevice(ctx->device);
  double h[3];
  CML_CUDA(cudaMemcpyAsync(h, ctx->reduce + ctx->n_slots, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->estimate_pending = false;
  if (out) {
    out->sum_ln_p = h[0];
    out->sum_w_ln_p = h[1];
    out->n_zero = (uint64_t)(h[2] + 0.5);
  }
  return CML_OK;
}

extern "C" int cml_estimate(cml_ctx* ctx, cml_estimate_result* out) {
  int r = cml_estimate_launch(ctx);
  if (r) return r;
  return cml_estimate_finish(ctx, out);
}

extern "C" int cml_last_fb_time_ms(cml_ctx* ctx, float* ms, uint32_t* n_kernels) {
  if (!ctx || !ms) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  float tot = 0;
  uint32_t nk = 0;
  if (ctx->dense && ctx->dense->ev0) {
    CML_CUDA(cudaEventElapsedTime(&tot, ctx->dense->ev0, ctx->dense->ev1));
    nk = 1;
  }
  for (auto& bt : ctx->batches) {
    if (!bt->ev_fb0) continue;
    float t = 0;
    CML_CUDA(cudaEventElapsedTime(&t, bt->ev_fb0, bt->ev_fb1));
    tot += t;
    nk += bt->n_fb_kernels;
  }
  *ms = tot;
  if (n_kernels) *n_kernels = nk;
  return CML_OK;
}

extern "C" int cml_get_example_logprob(cml_ctx* ctx, double* ln_p, uint64_t n) {
  if (!ctx || !ln_p) return CML_ERR_ARG;
  cudaSetDevice(ctx->device);
  uint64_t done = 0;
  if (ctx->dense) {
    const uint64_t k = std::min<uint64_t>(ctx->dense->n_seq, n);
    CML_CUDA(cudaMemcpyAsync(ln_p, ctx->dense->ex_lnp.p, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    done = k;
  }
  for (auto& bt : ctx->batches) {
    if (done >= n) break;
    const uint64_t k = std::min<uint64_t>(bt->n_ex, n - done);
    CML_CUDA(cudaMemcpyAsync(ln_p + done, bt->ex_lnp.p, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    done += k;
  }
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  CML_REQUIRE(done == n, CML_ERR_ARG, "fewer examples resident than requested");
  return CML_OK;
}

extern "C" int cml_get_arc_counts(cml_ctx* ctx, double* counts) {
  if (!ctx || !counts) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  CML_REQUIRE(ctx->slots_are_arcs && !ctx->dense, CML_ERR_STATE,
              "per-arc counts are not kept: counts are accumulated per unlocked-parameter slot "
              "(set CML_OPT_ARC_COUNTS before cml_set_model, or use cml_get_counts)");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(counts, ctx->reduce, ctx->n_arcs * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" int cml_get_counts(cml_ctx* ctx, double* counts, uint64_t n) {
  if (!ctx || !counts) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && n <= ctx->n_slots, CML_ERR_ARG, "more counts requested than count slots");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(counts, ctx->reduce, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" uint64_t cml_count_slots(cml_ctx* ctx) { return ctx ? ctx->n_slots : 0; }

extern "C" int cml_reduce_buffer(cml_ctx* ctx, void** p, uint64_t* n) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  if (p) *p = ctx->reduce;
  if (n) *n = ctx->reduce_n;
  return CML_OK;
}

extern "C" int cml_reduce_buffer_write(cml_ctx* ctx, const double* src, uint64_t n) {
  if (!ctx || !src) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && n <= ctx->reduce_n, CML_ERR_ARG, "reduce buffer smaller than requested");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemsetAsync(ctx->reduce, 0, ctx->reduce_n * sizeof(double), ctx->stream));
  CML_CUDA(cudaMemcpyAsync(ctx->reduce, src, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" int cml_reduce_buffer_read(cml_ctx* ctx, double* dst, uint64_t n) {
  if (!ctx || !dst) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && n <= ctx->reduce_n, CML_ERR_ARG, "reduce buffer smaller than requested");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(dst, ctx->reduce, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

extern "C" int cml_use_reduce_buffer(cml_ctx* ctx, void* p, uint64_t n) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model, CML_ERR_STATE, "cml_set_model first");
  if (!p) {
    ctx->reduce = ctx->reduce_own.p;
    return CML_OK;
  }
  CML_REQUIRE(n >= ctx->reduce_n, CML_ERR_ARG, "reduce buffer too small (need count slots + 3 doubles)");
  ctx->reduce = (double*)p;
  ctx->graph_dirty = true;
  return CML_OK;
}

// -------------------------------------------------------------------------------------------------
// M-step
// -------------------------------------------------------------------------------------------------
static int run_normalize(cml_ctx* ctx) {  // u -> ln_w
  using namespace cmlk;
  cudaStream_t s = ctx->stream;
  if (ctx->n_groups) {
    // a warp per group, or a block per group when some group is large (its members are summed serially per thread)
    const bool big = ctx->max_group_size > 512;
    const unsigned grid = big ? ctx->n_groups : cdiv((uint64_t)ctx->n_groups * 32, 256);
    auto sums = big ? k_norm_sums<256> : k_norm_sums<32>;
    auto assign = big ? k_norm_assign<256> : k_norm_assign<32>;
    sums<<<grid, 256, 0, s>>>(ctx->n_groups, ctx->group_off.p, ctx->group_members.p,
                              ctx->have_add ? ctx->group_add.p : nullptr, ctx->param_tie.p, ctx->u.p, ctx->gsum.p,
                              ctx->glocked.p);
    ++ctx->launches;
    if (ctx->n_ties) {
      k_tie_totals<<<cdiv((uint64_t)ctx->n_ties * 32, 256), 256, 0, s>>>(
          ctx->n_ties, ctx->tie_off.p, ctx->tie_members.p, ctx->param_group.p, ctx->u.p, ctx->gsum.p, ctx->glocked.p,
          ctx->tie_arc.p, ctx->tie_state.p, ctx->tie_maxl.p);
      ++ctx->launches;
    }
    assign<<<grid, 256, 0, s>>>(ctx->n_groups, ctx->group_off.p, ctx->group_members.p, ctx->param_tie.p, ctx->u.p,
                                ctx->tie_arc.p, ctx->tie_state.p, ctx->tie_maxl.p, ctx->ln_w.p);
    ++ctx->launches;
  }
  k_copy_ungrouped<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, ctx->param_group.p, ctx->u.p, ctx->ln_w.p);
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  return CML_OK;
}

extern "C" int cml_normalize_params(cml_ctx* ctx) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ctx->u.p, ctx->ln_w.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice,
                           ctx->stream));
  return run_normalize(ctx);
}

// M-step launches on the context's stream; the largest weight change ends up in ctx->maxchg (device).  No host
// synchronisation: cml_maximize and cml_em_step read it back.
static int enqueue_maximize(cml_ctx* ctx, double rate) {
  using namespace cmlk;
  cudaStream_t s = ctx->stream;
  const bool slots_are_params = ctx->trivial && !ctx->dense;  // dense mode: slots are T / E cells with chains
  if (rate <= 1. && ctx->n_ties == 0 && ctx->n_params <= 8192 && ctx->n_slots <= 16384 && ctx->max_group_size <= 256 &&
      !getenv("CML_NO_FUSED_MSTEP")) {
    // small model: the whole M-step in one launch (see k_mstep_fused)
    MstepArgs M;
    M.n_slots = ctx->n_slots;
    M.n_params = ctx->n_params;
    M.n_groups = ctx->n_groups;
    M.slot_off = slots_are_params ? nullptr : ctx->slot_off.p;
    M.slot_param = ctx->slot_param.p;
    M.counts = ctx->reduce;
    M.prior = ctx->have_prior ? ctx->slot_prior.p : nullptr;
    M.param_tie = ctx->param_tie.p;
    M.param_group = ctx->param_group.p;
    M.group_off = ctx->group_off.p;
    M.group_members = ctx->group_members.p;
    M.group_add = ctx->have_add ? ctx->group_add.p : nullptr;
    M.acc = ctx->acc.p;
    M.u = ctx->u.p;
    M.old = ctx->old.p;
    M.ln_w = ctx->ln_w.p;
    M.gsum = ctx->gsum.p;
    M.glocked = ctx->glocked.p;
    M.maxchg = ctx->maxchg.p;
    k_mstep_fused<<<1, 1024, 0, s>>>(M);
    ++ctx->launches;
    CML_CUDA(cudaGetLastError());
    return CML_OK;
  }
  if (!slots_are_params) CML_CUDA(cudaMemsetAsync(ctx->acc.p, 0, ctx->n_params * sizeof(double), s));
  k_param_acc<<<cdiv(ctx->n_slots, 256), 256, 0, s>>>(ctx->n_slots, slots_are_params ? nullptr : ctx->slot_off.p,
                                                      ctx->slot_param.p, ctx->reduce,
                                                      ctx->have_prior ? ctx->slot_prior.p : nullptr, ctx->param_tie.p,
                                                      ctx->acc.p);
  k_unnorm<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, ctx->acc.p, ctx->ln_w.p, ctx->param_tie.p,
                                                   ctx->param_group.p, ctx->u.p, ctx->old.p);
  ctx->launches += 2;
  int r = run_normalize(ctx);
  if (r) return r;
  if (rate > 1. && ctx->trivial) {  // over-relaxation is disabled for real cascades (train.cc:543-549)
    k_overrelax<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, rate, ctx->param_tie.p, ctx->old.p,
                                                        ctx->ln_w.p, ctx->u.p);
    ++ctx->launches;
    if ((r = run_normalize(ctx))) return r;
  }
  CML_CUDA(cudaMemsetAsync(ctx->maxchg.p, 0, sizeof(unsigned long long), s));
  k_max_change<<<cdiv(ctx->n_params, 256), 256, 0, s>>>(ctx->n_params, ctx->param_tie.p, ctx->old.p, ctx->ln_w.p,
                                                       ctx->maxchg.p);
  ++ctx->launches;
  CML_CUDA(cudaGetLastError());
  return CML_OK;
}

extern "C" int cml_maximize(cml_ctx* ctx, double rate, double* max_delta) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  cudaSetDevice(ctx->device);
  const int r = enqueue_maximize(ctx, rate);
  if (r) return r;
  unsigned long long bits = 0;
  CML_CUDA(cudaMemcpyAsync(&bits, ctx->maxchg.p, sizeof(bits), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  if (max_delta) std::memcpy(max_delta, &bits, sizeof(double));
  return CML_OK;
}

// One EM iteration, one host synchronisation (include/carmel_b200.h).  The sequence
//   parameters -> snapshot slot 3, arc / class weights, E-step kernels, all-reduce, likelihood scalars -> pinned host,
//   M-step kernels, max change -> pinned host
// is the same every iteration, so it is captured into a CUDA graph once and replayed (NCCL all-reduces are
// capturable); anything that changes the sequence marks the graph dirty.
static int enqueue_em_step_a(cml_ctx* ctx) {  // everything before the all-reduce
  cudaStream_t s = ctx->stream;
  CML_CUDA(cudaMemcpyAsync(ctx->snap[3].p, ctx->ln_w.p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice, s));
  const int r = cml_estimate_launch(ctx);
  if (r) return r;
  ctx->estimate_pending = false;
  return CML_OK;
}
static int enqueue_em_step_b(cml_ctx* ctx, double rate) {  // everything after it
  cudaStream_t s = ctx->stream;
  CML_CUDA(cudaMemcpyAsync(ctx->h_step, ctx->reduce + ctx->n_slots, 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
  const int r = enqueue_maximize(ctx, rate);
  if (r) return r;
  CML_CUDA(cudaMemcpyAsync(ctx->h_step + 3, ctx->maxchg.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  return CML_OK;
}
static int enqueue_em_step(cml_ctx* ctx, double rate) {
  int r = enqueue_em_step_a(ctx);
  if (r) return r;
  if ((r = cml_allreduce_counts(ctx))) return r;
  return enqueue_em_step_b(ctx, rate);
}
// capture fn() on the context's stream into an executable graph; launches / collectives counted once per replay
template <class F>
static int capture_graph(cml_ctx* ctx, cudaGraphExec_t* exec, F&& fn) {
  cudaGraph_t g = nullptr;
  CML_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  ctx->capturing = true;
  const int r = fn();
  ctx->capturing = false;
  const cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
  if (r) {
    if (g) cudaGraphDestroy(g);
    return r;
  }
  CML_CUDA(e);
  CML_CUDA(cudaGraphInstantiate(exec, g, 0));
  cudaGraphDestroy(g);
  return CML_OK;
}

extern "C" int cml_em_step(cml_ctx* ctx, double rate, cml_estimate_result* out, double* max_delta) {
  if (!ctx) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_model && ctx->have_params, CML_ERR_STATE, "cml_set_model and cml_set_params first");
  CML_REQUIRE(!ctx->batches.empty() || ctx->dense || ctx->opt_allow_empty, CML_ERR_NODERIV,
              "no trellises resident (no training example had a derivation)");
  cudaSetDevice(ctx->device);
  if (!ctx->h_step) CML_CUDA(cudaMallocHost((void**)&ctx->h_step, 8 * sizeof(double)));
  if (!ctx->dense && (ctx->hot_dirty || ctx->cls_dirty) && !ctx->batches.empty()) {  // host-side table rebuilds
    const int rc = rebuild_slot_codes(ctx);
    if (rc) return rc;
    ctx->graph_dirty = true;
  }
  const bool use_graph = !ctx->opt_no_graph && rate == 1. && !getenv("CML_NO_GRAPH");
  // With a communicator the iteration is two graphs around an eagerly enqueued ncclAllReduce (the collective itself
  // is not captured: one launch, and no dependence on NCCL's graph-capture support across processes).
  const bool split = ctx->comm && ctx->comm_size > 1;
  if (use_graph) {
    if (ctx->graph_dirty || !ctx->graph) {
      if (ctx->graph) cudaGraphExecDestroy(ctx->graph);
      if (ctx->graph_b) cudaGraphExecDestroy(ctx->graph_b);
      ctx->graph = ctx->graph_b = nullptr;
      // one plain pass first: kernels set their attributes / lazily created events outside the capture
      int r = enqueue_em_step(ctx, rate);
      if (r) return r;
      CML_CUDA(cudaStreamSynchronize(ctx->stream));
      CML_CUDA(cudaMemcpyAsync(ctx->ln_w.p, ctx->snap[3].p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice,
                               ctx->stream));  // undo: the captured pass below is the one that counts
      const uint64_t launches0 = ctx->launches, coll0 = ctx->collectives;
      if (!split) {
        if ((r = capture_graph(ctx, &ctx->graph, [&]() { return enqueue_em_step(ctx, rate); }))) return r;
      } else {
        if ((r = capture_graph(ctx, &ctx->graph, [&]() { return enqueue_em_step_a(ctx); }))) return r;
        if ((r = capture_graph(ctx, &ctx->graph_b, [&]() { return enqueue_em_step_b(ctx, rate); }))) return r;
      }
      ctx->graph_launches = ctx->launches - launches0;
      ctx->graph_collectives = ctx->collectives - coll0;
      ctx->launches = launches0;
      ctx->collectives = coll0;
      ctx->graph_dirty = false;
    }
    CML_CUDA(cudaGraphLaunch(ctx->graph, ctx->stream));
    if (split) {
      const int r = cml_allreduce_counts(ctx);
      if (r) return r;
      CML_CUDA(cudaGraphLaunch(ctx->graph_b, ctx->stream));
    }
    ctx->launches += ctx->graph_launches;
    ctx->collectives += ctx->graph_collectives;
  } else {
    const int r = enqueue_em_step(ctx, rate);
    if (r) return r;
  }
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  if (out) {
    out->sum_ln_p = ctx->h_step[0];
    out->sum_w_ln_p = ctx->h_step[1];
    out->n_zero = (uint64_t)(ctx->h_step[2] + 0.5);
  }
  if (max_delta) *max_delta = ctx->h_step[3];
  return CML_OK;
}

extern "C" int cml_snapshot_previous(cml_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot > 2) return CML_ERR_ARG;
  CML_REQUIRE(ctx->have_params, CML_ERR_STATE, "no parameters set");
  cudaSetDevice(ctx->device);
  CML_CUDA(cudaMemcpyAsync(ctx->snap[slot].p, ctx->snap[3].p, ctx->n_params * sizeof(double), cudaMemcpyDeviceToDevice,
                           ctx->stream));
  return CML_OK;
}

// small host-side sums over the ranks (corpus totals before training): through a 64-double device scratch
extern "C" int cml_allreduce_host(cml_ctx* ctx, double* inout, uint64_t n) {
  if (!ctx || !inout || n > 64) return CML_ERR_ARG;
  if (!ctx->comm || ctx->comm_size <= 1) return CML_OK;
  cudaSetDevice(ctx->device);
  if (!ctx->host_scratch.p) CML_CUDA(ctx->host_scratch.alloc(64));
  CML_CUDA(cudaMemcpyAsync(ctx->host_scratch.p, inout, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  const int r = cml_allreduce_buffer(ctx, ctx->host_scratch.p, n);
  if (r) return r;
  CML_CUDA(cudaMemcpyAsync(inout, ctx->host_scratch.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CML_CUDA(cudaStreamSynchronize(ctx->stream));
  return CML_OK;
}

// -------------------------------------------------------------------------------------------------
extern "C" const char* const* cml_exported_symbols(size_t* n) {
  static const char* const syms[] = {
      "cml_version", "cml_create", "cml_destroy", "cml_last_error", "cml_set_stream", "cml_synchronize",
      "cml_launch_count", "cml_set_option", "cml_set_model", "cml_set_params", "cml_get_params", "cml_snapshot_params",
      "cml_restore_params", "cml_add_sequences", "cml_dense_stats", "cml_dense_kernel", "cml_add_trellises", "cml_clear_trellises", "cml_trellis_totals", "cml_layout_stats",
      "cml_lane_stats", "cml_wide_stats", "cml_get_example_layout", "cml_estimate", "cml_estimate_launch", "cml_estimate_finish", "cml_last_fb_time_ms",
      "cml_get_example_logprob", "cml_get_arc_counts", "cml_get_counts", "cml_count_slots", "cml_reduce_buffer",
      "cml_use_reduce_buffer", "cml_reduce_buffer_write", "cml_reduce_buffer_read", "cml_maximize", "cml_em_step", "cml_snapshot_previous", "cml_comm_unique_id", "cml_comm_init_rank",
      "cml_comm_init_all", "cml_set_comm", "cml_comm_info", "cml_allreduce_counts", "cml_allreduce_buffer",
      "cml_allreduce_host", "cml_collective_count",
      "cml_normalize_params", "cml_exported_symbols", "cml_job_open", "cml_job_close", "cml_job_error",
      "cml_job_set_comm", "cml_job_set_allreduce", "cml_job_prepare", "cml_job_context", "cml_job_train", "cml_job_write", "cml_job_stats", "cml_gibbs_init", "cml_gibbs_attach_dense", "cml_gibbs_sweep",
      "cml_gibbs_sample_capacity", "cml_gibbs_get_samples", "cml_gibbs_get_state", "cml_gibbs_get_block_logprob", "cml_forests_create", "cml_forests_destroy",
      "cml_forests_last_error", "cml_forests_set_stream", "cml_forests_set_layout", "cml_forests_layout_stats", "cml_forests_level_stats", "cml_build_trellises", "cml_build_free_trellises", "cml_free_built_trellises", "cml_cyclic_stats", "cml_viterbi", "cml_kbest", "cml_kbest_stats", "cml_sample", "cml_sample_stats",
      "cml_forests_launch_count", "cml_forests_set_rules",
      "cml_forests_set_params", "cml_forests_get_params", "cml_forests_add", "cml_forests_totals", "cml_forests_estimate",
      "cml_forests_estimate_launch", "cml_forests_estimate_finish", "cml_forests_last_time_ms", "cml_forests_get_inside",
      "cml_forests_get_counts", "cml_forests_reduce_buffer", "cml_forests_comm_init_rank", "cml_forests_allreduce_counts", "cml_forests_maximize", "cml_forests_normalize_params",
      "cml_forest_job_open", "cml_forest_job_close", "cml_forest_job_error", "cml_forest_job_set_comm", "cml_forest_job_set_quiet", "cml_forest_job_set_allreduce", "cml_forests_synchronize", "cml_forests_viterbi", "cml_forests_kbest", "cml_forests_set_kbest_scratch_mb",
      "cml_forests_kbest_stats", "cml_forests_sample", "cml_forests_sample_stats", "cml_forests_gibbs_init", "cml_forests_gibbs_sweep", "cml_forests_gibbs_sample_capacity",
      "cml_forests_gibbs_get_samples", "cml_forests_gibbs_get_state",
      "cml_forest_job_prepare", "cml_forest_job_context", "cml_forest_job_train", "cml_forest_job_write",
      "cml_forest_job_stats"};
  if (n) *n = sizeof(syms) / sizeof(syms[0]);
  return syms;
}
