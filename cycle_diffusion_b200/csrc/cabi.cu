// cabi.cu -- the extern "C" surface declared in include/cdx.h, plus the in-library loop drivers
// (DPM-Encoder inversion and decode-with-recovered-noise) so that a whole chain is enqueued without
// returning to the host language between steps.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "nets.cuh"

struct cdx_engine { cdx::Engine e; };
struct cdx_net { cdx::Net* n; cdx_engine* owner; };

namespace cdx {
const std::string& last_error();

namespace {

template <class F>
int guard(F&& f) {
  try {
    f();
    return CDX_OK;
  } catch (const Error& err) {
    set_last_error(err.what());
    return err.code;
  } catch (const std::exception& err) {
    set_last_error(std::string("internal error: ") + err.what());
    return CDX_E_INVALID;
  }
}

// run `f` once in sizing mode, grow the arena, then for real
// The arena, the context K/V cache and the weight planes are reused from call to call with no synchronisation of their own,
// which is only safe in stream order.  A caller that switches streams between calls is handed over explicitly: every call
// records an event at its end, and a call arriving on a different stream first waits for it.
// `e2` (optional): a second engine whose networks `f` also runs (the two-model loops); both arenas are sized by the same sizing
// pass and both engines' hand-over events are honoured.
template <class F>
void with_arenas(Engine& e, Engine* e2, cudaStream_t s, F&& f) {
  Engine* es[2] = {&e, (e2 && e2 != &e) ? e2 : nullptr};
  const int ne = es[1] ? 2 : 1;
  if (es[1]) CDX_CHECK(es[1]->device == e.device, "two engines on different devices (%d, %d)", e.device, es[1]->device);
  CDX_CUDA(cudaSetDevice(e.device));
  for (int k = 0; k < ne; ++k) es[k]->arena.begin_dry();
  try {
    f();
  } catch (...) {
    for (int k = 0; k < ne; ++k) { es[k]->arena.dry = false; es[k]->arena.off = 0; }
    throw;
  }
  for (int k = 0; k < ne; ++k) {
    Engine& x = *es[k];
    x.arena.end_dry();
    if (!x.done_ev) CDX_CUDA(cudaEventCreateWithFlags(&x.done_ev, cudaEventDisableTiming));
    if (x.ev_recorded && x.last_stream != s) CDX_CUDA(cudaStreamWaitEvent(s, x.done_ev, 0));
  }
  f();
  for (int k = 0; k < ne; ++k) {
    Engine& x = *es[k];
    x.arena.off = 0;
    CDX_CUDA(cudaEventRecord(x.done_ev, s));
    x.ev_recorded = true;
    x.last_stream = s;
  }
}
template <class F>
void with_arena(Engine& e, cudaStream_t s, F&& f) { with_arenas(e, nullptr, s, f); }

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// fill a device float vector with one value per row, repeated `rep` times (timestep vector for [x;x] CFG batches)
void upload_timesteps(Engine& e, const float* t_host, int n_steps, int reps, float* dev, cudaStream_t s) {
  if (e.dry()) return;
  std::vector<float> h((size_t)n_steps * reps);
  for (int i = 0; i < n_steps; ++i)
    for (int r = 0; r < reps; ++r) h[(size_t)i * reps + r] = t_host[i];
  // pageable source: the runtime stages the copy before returning, so `h` may die afterwards
  CDX_CUDA(cudaMemcpyAsync(dev, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice, s));
}

// dst[b, slot, :] = src[b, :]  for a [B, n_slots, chw] tensor
void scatter_slot(Engine& e, const float* src, float* dst, int B, int chw, int n_slots, int slot, cudaStream_t s) {
  if (e.dry()) return;
  CDX_CUDA(cudaMemcpy2DAsync(dst + (size_t)slot * chw, (size_t)n_slots * chw * sizeof(float), src, (size_t)chw * sizeof(float),
                             (size_t)chw * sizeof(float), B, cudaMemcpyDeviceToDevice, s));
}
void gather_slot(Engine& e, const float* src, float* dst, int B, int chw, int n_slots, int slot, cudaStream_t s) {
  if (e.dry()) return;
  CDX_CUDA(cudaMemcpy2DAsync(dst, (size_t)chw * sizeof(float), src + (size_t)slot * chw, (size_t)n_slots * chw * sizeof(float),
                             (size_t)chw * sizeof(float), B, cudaMemcpyDeviceToDevice, s));
}
void copy_dd(Engine& e, const float* src, float* dst, size_t n, cudaStream_t s) {
  if (e.dry()) return;
  CDX_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
}

// test hooks: build the fp16-split planes of an ad-hoc weight matrix on the fly (networks do this once at finalize)
void hook_h16_planes(Engine& e, const float* w, size_t n, GemmArgs& g, cudaStream_t s) {
  if (e.tc_kind < 1 || (n & 7)) return;
  void* hi = e.arena.alloc(n * 2);
  void* lo = e.arena.alloc(n * 2);
  if (e.dry()) { g.Bw_h_hi = hi; g.Bw_h_lo = lo; return; }
  float* slot = e.amax_slot();
  amax_rows(e, w, 1, (int)n, (long long)n, slot, s);
  float wmax = 0.f;
  CDX_CUDA(cudaMemcpyAsync(&wmax, slot, sizeof(float), cudaMemcpyDeviceToHost, s));
  CDX_CUDA(cudaStreamSynchronize(s));
  g.b_exp = h16_exp_host(wmax);
  split_planes_h16(e, w, hi, lo, n, g.b_exp, s);
  g.Bw_h_hi = hi; g.Bw_h_lo = lo;
}

// ---------------------------------------------------------------------------------------------------------------------
// The latent sampling loops (DDIMSampler._ddpm_ddim_encoding ddim.py:450-501, ddim_sampling_with_eps ddim.py:395-448) as ONE
// driver with three modes: DPM-Encoder only, decode only, or both chains in lock-step (the source chain under the source
// condition and the target chain under the target condition share one U-Net call per step; the noise recovered at step i is
// consumed by the target chain in registers, so no z buffer is needed -- the Diffusers CycleDiffusionPipeline loop shape).
// Per step: one U-Net call on the batch [src segments | tgt segments] (a chain contributes [uncond, cond] when it runs with
// classifier-free guidance, ddim.py:550-559, else one segment) and ONE fused elementwise launch (latent_step).
// With a target network `tgt` (two-model lock-step, latentdiff_stochastic_wrapper.py:253-311 run as one loop) the source segments
// go through `unet` and the target segments through `tgt`: two U-Net calls on the same contiguous xin / eout slices, each chain at
// the batch it has in the two-phase loops.
// ---------------------------------------------------------------------------------------------------------------------
enum { LOOP_ENC = 1, LOOP_DEC = 2, LOOP_LOCK = 3 };
struct LatentLoopArgs {
  int mode = 0;
  const float* x0 = nullptr;                       // ENC / LOCK
  const float* c_src = nullptr; const float* c_tgt = nullptr; const float* uc = nullptr; int L = 0;
  float s_scale = 1.f, t_scale = 1.f;
  const float* s_scale_v = nullptr; const float* t_scale_v = nullptr;     // per-sample scales (device, [B]): ensemble members along B
  const cdx_ddim_coef* coef = nullptr; const float* t_host = nullptr; int n_steps = 0;
  int n_rec = 0; const float* noise = nullptr; float sa = 0.f, s1 = 0.f;      // ENC / LOCK: noise [n_rec+1, B, chw]
  float* z_out = nullptr;                           // ENC: [B, n_rec+1, chw]; LOCK: optional
  const float* z_in = nullptr; int n_eps = 0; const float* extra = nullptr;   // DEC
  float* x_out = nullptr;                           // DEC / LOCK
  int B = 0, C = 0, h = 0, w = 0;
};

void run_latent_loop(Net& unet, const LatentLoopArgs& a, cudaStream_t s, Net* tgt = nullptr) {
  Engine& e = *unet.eng;
  const int B = a.B, chw = a.C * a.h * a.w;
  const size_t n = (size_t)B * chw;
  const bool enc = a.mode & LOOP_ENC, dec = a.mode & LOOP_DEC;
  // (with per-sample scales both segments always run; samples whose scale is 0 / 1 pick their segment's output unchanged)
  const bool cfg_s = enc && a.uc && (a.s_scale_v || (a.s_scale != 1.0f && a.s_scale != 0.0f));
  const bool cfg_t = dec && a.uc && (a.t_scale_v || (a.t_scale != 1.0f && a.t_scale != 0.0f));
  const int nseg_src = enc ? (cfg_s ? 2 : 1) : 0, nseg_tgt = dec ? (cfg_t ? 2 : 1) : 0, nseg = nseg_src + nseg_tgt;
  const int nb = nseg * B;
  const int D = unet.ucfg.context_dim;
  const size_t ctx_n = (size_t)B * a.L * D;
  Scope sc(e.arena);
  unet.ctxkv.valid = false;                    // the conditioning is fixed for this loop: its K / V are computed by the first step only
  struct Invalidate { Net& u; ~Invalidate() { u.ctxkv.valid = false; } } inval{unet};
  if (tgt) tgt->ctxkv.valid = false;
  struct InvalidateTgt { Net* u; ~InvalidateTgt() { if (u) u->ctxkv.valid = false; } } inval_tgt{tgt};
  float* xin = (float*)e.arena.alloc((size_t)nseg * n * sizeof(float));
  float* eout = (float*)e.arena.alloc((size_t)nseg * n * sizeof(float));
  float* ctx_in = (float*)e.arena.alloc((size_t)nseg * ctx_n * sizeof(float));
  float* xb[3] = {nullptr, nullptr, nullptr};
  float* yb[2] = {nullptr, nullptr};
  if (enc) for (int k = 0; k < 3; ++k) xb[k] = (float*)e.arena.alloc(n * sizeof(float));
  if (dec) for (int k = 0; k < 2; ++k) yb[k] = (float*)e.arena.alloc(n * sizeof(float));
  const int loop_steps = enc && !dec ? a.n_rec : a.n_steps;
  float* tdev = (float*)e.arena.alloc((size_t)std::max(loop_steps, 1) * nb * sizeof(float));
  upload_timesteps(e, a.t_host, loop_steps, nb, tdev, s);
  if (ctx_n) {   // cat([uc, c]) per chain: uncond first (ddim.py:555-557); unconditional models (L == 0) carry no context
    int sg = 0;
    if (enc) {
      if (cfg_s) copy_dd(e, a.uc, ctx_in + (size_t)(sg++) * ctx_n, ctx_n, s);
      copy_dd(e, (a.uc && !a.s_scale_v && a.s_scale == 0.0f) ? a.uc : a.c_src, ctx_in + (size_t)(sg++) * ctx_n, ctx_n, s);
    }
    if (dec) {
      if (cfg_t) copy_dd(e, a.uc, ctx_in + (size_t)(sg++) * ctx_n, ctx_n, s);
      copy_dd(e, (a.uc && !a.t_scale_v && a.t_scale == 0.0f) ? a.uc : a.c_tgt, ctx_in + (size_t)(sg++) * ctx_n, ctx_n, s);
    }
  }
  const float* es_uc = cfg_s ? eout : nullptr;
  const float* es_c = eout + (cfg_s ? n : 0);
  const float* et_uc = cfg_t ? eout + (size_t)nseg_src * n : nullptr;
  const float* et_c = eout + (size_t)nseg_src * n + (cfg_t ? n : 0);
  auto next_kind = [&](int i_next) {             // how x_{t-1} of iteration i_next is obtained (0: that iteration does not exist)
    if (i_next >= a.n_rec) return 0;
    return (a.n_steps - 1 - i_next) == 0 ? 2 : 1;                               // ddim.py:583-584
  };
  if (enc) {
    LatentInit in;
    in.n = n; in.chw = chw;
    in.x0 = a.x0; in.noise0 = a.noise; in.sa = a.sa; in.s1 = a.s1;
    in.z_out = a.z_out; in.z_stride = (long long)(a.n_rec + 1) * chw;
    in.xt = xb[0]; in.yt = dec ? yb[0] : nullptr;
    in.next = next_kind(0);
    if (in.next) { in.noise_next = a.noise + n; in.cnext = a.coef[0]; }
    in.xn = xb[1];
    in.xin = xin; in.nseg_src = nseg_src; in.nseg_tgt = nseg_tgt;
    latent_init(e, in, s);
  } else {
    gather_slot(e, a.z_in, yb[0], B, chw, a.n_eps + 1, 0, s);                   // x_T = eps_list[:, 0], SDW:153
    for (int sg = 0; sg < nseg_tgt; ++sg) copy_dd(e, yb[0], xin + (size_t)sg * n, n, s);
  }
  const int iters = e.dry() ? std::min(loop_steps, 1) : loop_steps;
  for (int i = 0; i < iters; ++i) {
    if (!tgt) {
      unet_forward(unet, xin, tdev + (size_t)i * nb, ctx_in, a.L, eout, nb, a.h, a.w, s, true);
    } else {
      const size_t ns = (size_t)nseg_src * B;
      unet_forward(unet, xin, tdev + (size_t)i * nb, ctx_in, a.L, eout, (int)ns, a.h, a.w, s, true);
      unet_forward(*tgt, xin + ns * chw, tdev + (size_t)i * nb + ns, ctx_in + (size_t)nseg_src * ctx_n, a.L, eout + ns * chw,
                   nseg_tgt * B, a.h, a.w, s, true);
    }
    LatentStep st;
    st.n = n; st.chw = chw;
    if (enc) {
      st.enc = 1;
      st.x0 = a.x0; st.xt = xb[0]; st.xn = xb[1];
      st.es_c = es_c; st.es_uc = es_uc; st.s_scale = a.s_scale; st.s_scale_v = a.s_scale_v; st.cs = a.coef[i];
      if (a.z_out) { st.z_out = a.z_out + (size_t)(1 + i) * chw; st.z_stride = (long long)(a.n_rec + 1) * chw; }
      st.next = next_kind(i + 1);
      if (st.next) { st.noise_next = a.noise + (size_t)(2 + i) * n; st.cnext = a.coef[i + 1]; }
      st.xn2 = xb[2];
    }
    if (dec) {
      st.dec = 1;
      st.yt = yb[0]; st.et_c = et_c; st.et_uc = et_uc; st.t_scale = a.t_scale; st.t_scale_v = a.t_scale_v; st.ct = a.coef[i];
      if (!enc) {
        if (i < a.n_eps) { st.eps_in = a.z_in + (size_t)(1 + i) * chw; st.eps_stride = (long long)(a.n_eps + 1) * chw; }
        else { st.eps_in = a.extra + (size_t)(i - a.n_eps) * n; st.eps_stride = chw; }
      }
      st.y_out = (i == loop_steps - 1) ? a.x_out : yb[1];
    }
    st.xin = xin; st.nseg_src = nseg_src; st.nseg_tgt = nseg_tgt;
    latent_step(e, st, s);
    if (enc) { float* t0 = xb[0]; xb[0] = xb[1]; xb[1] = xb[2]; xb[2] = t0; }
    if (dec) std::swap(yb[0], yb[1]);
  }
}

}  // namespace
}  // namespace cdx

using namespace cdx;

static inline cdx::Engine& engine_of(cdx_engine* h) { return h->e; }

extern "C" {

int cdx_abi_version(void) { return CDX_ABI_VERSION; }
const char* cdx_last_error(void) { return cdx::last_error().c_str(); }

int cdx_engine_create(int device, cdx_engine** out) {
  return guard([&] {
    CDX_CHECK(out != nullptr, "engine_create: null out");
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count <= 0)
      throw Error(CDX_E_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(err));
    CDX_CHECK(device >= 0 && device < count, "engine_create: device %d out of range (count %d)", device, count);
    CDX_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    CDX_CUDA(cudaGetDeviceProperties(&prop, device));
    cdx_engine* eng = new cdx_engine();
    eng->e.device = device;
    eng->e.num_sms = prop.multiProcessorCount;
    *out = eng;
  });
}
void cdx_engine_destroy(cdx_engine* e) {
  if (!e) return;
  cudaSetDevice(e->e.device);
  cudaDeviceSynchronize();
  e->e.arena.destroy();
  if (e->e.done_ev) cudaEventDestroy(e->e.done_ev);
  if (e->e.amax_pool) cudaFree(e->e.amax_pool);
  delete e;
}
size_t cdx_engine_workspace_bytes(const cdx_engine* e) { return e ? e->e.arena.cap : 0; }
uint64_t cdx_engine_launch_count(const cdx_engine* e) { return e ? e->e.launches : 0; }
int cdx_engine_set_mma_mode(cdx_engine* e, int mode) {
  return guard([&] {
    CDX_CHECK(e != nullptr && mode >= 0 && mode <= 5, "set_mma_mode: bad arguments");
    e->e.mma_mode = mode == 0 ? 0 : 1;       // 2 = tcgen05 contractions but unfused attention (A/B comparisons)
    e->e.flash_attn = mode != 2 && mode != 0;
    e->e.tc_kind = mode == 3 ? 0 : mode == 4 ? 2 : 1;    // 3 = 3xTF32 contractions, 4 = single-term fp16 (fast path), else fp16 split
  });
}

int cdx_engine_profile(cdx_engine* e, int enable) {
  return guard([&] {
    CDX_CHECK(e != nullptr, "profile: null engine");
    CDX_CUDA(cudaSetDevice(e->e.device));
    CDX_CUDA(cudaDeviceSynchronize());
    for (ProfRec& r : e->e.prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    e->e.prof.recs.clear();
    e->e.prof.on = enable != 0;
  });
}
int cdx_engine_profile_read(cdx_engine* e, int tag, double* ms, double* flops, double* bytes, uint64_t* launches) {
  return guard([&] {
    CDX_CHECK(e && ms && flops && bytes && launches && tag >= 0 && tag < PROF_NTAGS, "profile_read: bad arguments");
    CDX_CUDA(cudaSetDevice(e->e.device));
    CDX_CUDA(cudaDeviceSynchronize());
    *ms = 0; *flops = 0; *bytes = 0; *launches = 0;
    const bool dump = getenv("CDX_PROF_DUMP") != nullptr;
    for (const ProfRec& r : e->e.prof.recs) {
      if (r.tag != tag) continue;
      float t = 0.f;
      CDX_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
      if (dump) fprintf(stderr, "[cdx prof] tag %d  %8.3f ms  %8.1f GFLOP  %7.1f TF/s  %s\n", tag, t, r.flops * 1e-9, t > 0 ? r.flops / (t * 1e9) : 0.0, r.note);
      *ms += t; *flops += r.flops; *bytes += r.bytes; *launches += (uint64_t)r.launches;
    }
  });
}

// ---------------------------------------------------------------- networks
int cdx_unet_create(cdx_engine* e, const cdx_unet_config* cfg, cdx_net** out) {
  return guard([&] {
    CDX_CHECK(cfg && out, "unet_create: null argument");
    cdx_net* h = new cdx_net();
    h->owner = e;
    static Engine host_only;   // inventory-only nets (e == NULL) can be built without a GPU
    h->n = make_unet(e ? &e->e : &host_only, *cfg);
    *out = h;
  });
}
int cdx_vae_create(cdx_engine* e, const cdx_vae_config* cfg, cdx_net** out) {
  return guard([&] {
    CDX_CHECK(cfg && out, "vae_create: null argument");
    cdx_net* h = new cdx_net();
    h->owner = e;
    static Engine host_only;
    h->n = make_vae(e ? &e->e : &host_only, *cfg);
    *out = h;
  });
}
int cdx_text_create(cdx_engine* e, const cdx_text_config* cfg, cdx_net** out) {
  return guard([&] {
    CDX_CHECK(cfg && out, "text_create: null argument");
    cdx_net* h = new cdx_net();
    h->owner = e;
    static Engine host_only;
    h->n = make_text(e ? &e->e : &host_only, *cfg);
    *out = h;
  });
}
void cdx_net_destroy(cdx_net* n) {
  if (!n) return;
  destroy_net(n->n);
  delete n;
}
int cdx_net_num_params(const cdx_net* n) { return n ? (int)n->n->params.size() : 0; }
const char* cdx_net_param_name(const cdx_net* n, int i) {
  if (!n || i < 0 || i >= (int)n->n->params.size()) return nullptr;
  return n->n->params[i].name.c_str();
}
int cdx_net_param_shape(const cdx_net* n, int i, int64_t dims[4]) {
  if (!n || i < 0 || i >= (int)n->n->params.size()) return CDX_E_INVALID;
  const Param& p = n->n->params[i];
  for (int k = 0; k < 4; ++k) dims[k] = k < p.rank ? p.dims[k] : 1;
  return p.rank;
}
int cdx_net_load_param(cdx_net* n, const char* name, const float* data, int on_device, const int64_t* dims, int rank) {
  return guard([&] {
    CDX_CHECK(n && n->owner && name && data && dims, "load_param: null argument (nets created without an engine are inventory-only)");
    net_load_param(*n->n, name, data, on_device != 0, dims, rank);
  });
}
int cdx_net_finalize(cdx_net* n) {
  return guard([&] {
    CDX_CHECK(n && n->owner, "finalize: null / inventory-only net");
    net_finalize(*n->n);
  });
}
int cdx_net_weight_blob(cdx_net* n, void** dev_ptr, size_t* bytes) {
  return guard([&] {
    CDX_CHECK(n && n->owner && dev_ptr && bytes, "weight_blob: null argument");
    net_ensure_blob(*n->n);
    *dev_ptr = n->n->blob;
    *bytes = n->n->blob_floats * sizeof(float);
  });
}
int cdx_net_adopt_blob(cdx_net* n) {
  return guard([&] {
    CDX_CHECK(n && n->owner, "adopt_blob: null / inventory-only net");
    net_ensure_blob(*n->n);
    for (Param& p : n->n->params) p.loaded = true;
    // the blob contents changed under us: everything derived from it (operand planes, cached context K/V) is stale
    n->n->planes_valid = false;
    n->n->ctxkv.valid = false;
    n->n->finalized = false;
    net_finalize(*n->n);
  });
}
int cdx_unet_set_time_freqs(cdx_net* n, const float* freqs, int half) {
  return guard([&] {
    CDX_CHECK(n && freqs, "set_time_freqs: null argument");
    CDX_CHECK(n->n->kind != NET_VAE, "set_time_freqs on a VAE");
    CDX_CHECK(half == n->n->ucfg.model_channels / 2, "set_time_freqs: half=%d, expected %d", half, n->n->ucfg.model_channels / 2);
    n->n->freqs_host.assign(freqs, freqs + half);
    if (n->n->finalized) net_finalize(*n->n);
  });
}

int cdx_unet_forward(cdx_net* n, const float* x, const float* t_dev, const float* ctx, int ctx_len, float* out, int B, int H, int W,
                     void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && x && t_dev && out && B > 0, "unet_forward: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { unet_forward(*n->n, x, t_dev, ctx, ctx_len, out, B, H, W, S(stream)); });
  });
}
int cdx_vae_encode(cdx_net* n, const float* img, float* moments, int B, int R, void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && img && moments && B > 0, "vae_encode: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { vae_encode(*n->n, img, moments, B, R, S(stream)); });
  });
}
int cdx_text_encode(cdx_net* n, const int* ids, int B, int L, float* out, void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && ids && out && B > 0, "text_encode: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { text_encode(*n->n, ids, out, B, L, S(stream)); });
  });
}
#define ENG_CALL_(EH_, ...)                                \
  return guard([&] {                                       \
    CDX_CHECK((EH_) != nullptr, "null engine");            \
    CDX_CUDA(cudaSetDevice(engine_of(EH_).device));        \
    __VA_ARGS__;                                           \
  })
int cdx_text_features(cdx_net* n, const int* ids, int B, int L, float* out, void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && ids && out && B > 0, "text_features: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { text_features(*n->n, ids, out, B, L, S(stream)); });
  });
}
int cdx_clip_image_features(cdx_net* n, const float* pixels, int B, float* out, void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && pixels && out && B > 0, "clip_image_features: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { clip_image_features(*n->n, pixels, out, B, S(stream)); });
  });
}
int cdx_clip_preprocess(cdx_engine* e, const float* img, int B, int R, int size, float* out, void* s) {
  ENG_CALL_(e, CDX_CHECK(img && out && B > 0 && R > 0 && size > 0, "clip_preprocess: bad arguments"); clip_preprocess(e->e, img, B, R, size, out, S(s)));
}
int cdx_dclip_scores(cdx_engine* e, const float* img_f, const float* orig_f, const float* enc_f, const float* dec_f, int B, int D, float* clip_out,
                     float* dclip_out, void* s) {
  ENG_CALL_(e, CDX_CHECK(img_f && orig_f && enc_f && dec_f && clip_out && dclip_out && B > 0 && D > 0, "dclip_scores: bad arguments");
            dclip_scores(e->e, img_f, orig_f, enc_f, dec_f, B, D, clip_out, dclip_out, S(s)));
}
int cdx_image_metrics(cdx_engine* eh, const float* a, const float* b, int B, int H, int W, float* out, void* stream) {
  return guard([&] {
    CDX_CHECK(eh && a && b && out && B > 0, "image_metrics: bad arguments");
    with_arena(eh->e, S(stream), [&] { image_metrics(eh->e, a, b, B, H, W, out, S(stream)); });
  });
}
int cdx_vae_decode(cdx_net* n, const float* z, float* img, int B, int h, void* stream) {
  return guard([&] {
    CDX_CHECK(n && n->owner && z && img && B > 0, "vae_decode: bad arguments");
    with_arena(n->owner->e, S(stream), [&] { vae_decode(*n->n, z, img, B, h, S(stream)); });
  });
}

// ---------------------------------------------------------------- per-step kernels
#define ENG_CALL(EH_, ...)                                 \
  return guard([&] {                                       \
    CDX_CHECK((EH_) != nullptr, "null engine");            \
    CDX_CUDA(cudaSetDevice(engine_of(EH_).device));        \
    __VA_ARGS__;                                           \
  })

int cdx_affine(cdx_engine* e, const float* x, float a, float b, float* out, size_t n, void* s) { ENG_CALL(e, affine(e->e, x, a, b, out, n, S(s))); }
int cdx_shift_scale(cdx_engine* e, const float* x, float b, float a, float* out, size_t n, void* s) { ENG_CALL(e, shift_scale(e->e, x, b, a, out, n, S(s))); }
int cdx_q_sample(cdx_engine* e, const float* x0, const float* nz, float sa, float s1, float* out, size_t n, void* s) {
  ENG_CALL(e, q_sample(e->e, x0, nz, sa, s1, out, n, S(s)));
}
int cdx_vae_posterior(cdx_engine* e, const float* mom, const float* nz, float sf, float* out, int B, int C, int hw, void* s) {
  ENG_CALL(e, vae_posterior(e->e, mom, nz, sf, out, B, C, hw, S(s)));
}
int cdx_ddim_posterior_sample(cdx_engine* e, const float* x0, const float* xt, const float* nz, const cdx_ddim_coef* c, float* o, size_t n, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); ddim_posterior_sample(e->e, x0, xt, nz, *c, o, n, S(s)));
}
int cdx_ddim_compute_eps(cdx_engine* e, const float* xt, const float* xn, const float* e_c, const float* e_uc, float scale, const cdx_ddim_coef* c,
                         float* o, size_t n, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); ddim_compute_eps(e->e, xt, xn, e_c, e_uc, scale, *c, o, n, S(s)));
}
int cdx_ddim_step_with_eps(cdx_engine* e, const float* x, const float* e_c, const float* e_uc, float scale, const float* eps, const cdx_ddim_coef* c,
                           float* o, size_t n, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); ddim_step_with_eps(e->e, x, e_c, e_uc, scale, eps, *c, o, n, S(s)));
}
int cdx_pixel_posterior_sample(cdx_engine* e, const float* x0, const float* xt, const float* nz, const cdx_pixel_coef* c, float* o, size_t n, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); pixel_posterior_sample(e->e, x0, xt, nz, *c, o, n, S(s)));
}
int cdx_pixel_compute_eps(cdx_engine* e, const float* xt, const float* xn, const float* et, const cdx_pixel_coef* c, float* o, int B, int chw,
                          int net_chw, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); pixel_compute_eps(e->e, xt, xn, et, *c, o, B, chw, net_chw, S(s)));
}
int cdx_pixel_step_with_eps(cdx_engine* e, const float* xt, const float* et, const float* eps, const cdx_pixel_coef* c, float* o, int B, int chw,
                            int net_chw, void* s) {
  ENG_CALL(e, CDX_CHECK(c, "null coef"); pixel_step_with_eps(e->e, xt, et, eps, *c, o, B, chw, net_chw, S(s)));
}

// ---------------------------------------------------------------- loop drivers
int cdx_latent_encode(cdx_net* un, const float* x0, const float* c, const float* uc, int L, float scale, const cdx_ddim_coef* coef,
                      const float* t_host, int n_steps, int n_rec, const float* noise, float sqrt_a_T, float sqrt_1ma_T, float* z_out, int B,
                      int C, int h, int w, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && x0 && (c || L == 0) && coef && t_host && noise && z_out, "latent_encode: null argument");
    CDX_CHECK(n_steps >= 1 && n_rec >= 0 && n_rec <= n_steps, "latent_encode: n_steps=%d n_rec=%d", n_steps, n_rec);
    for (int i = 0; i < n_rec; ++i) CDX_CHECK(coef[i].sigma > 0.f, "latent_encode: eta must be > 0 (sigma[%d] == 0), ddim.py:268", i);
    LatentLoopArgs a;
    a.mode = LOOP_ENC;
    a.x0 = x0; a.c_src = c; a.uc = uc; a.L = L; a.s_scale = scale;
    a.coef = coef; a.t_host = t_host; a.n_steps = n_steps; a.n_rec = n_rec; a.noise = noise; a.sa = sqrt_a_T; a.s1 = sqrt_1ma_T;
    a.z_out = z_out; a.B = B; a.C = C; a.h = h; a.w = w;
    with_arena(un->owner->e, S(stream), [&] { run_latent_loop(*un->n, a, S(stream)); });
  });
}

int cdx_latent_decode(cdx_net* un, const float* z, int n_eps, const float* c, const float* uc, int L, float scale, const cdx_ddim_coef* coef,
                      const float* t_host, int n_steps, const float* extra_noise, float* x_out, int B, int C, int h, int w, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && z && (c || L == 0) && coef && t_host && x_out, "latent_decode: null argument");
    CDX_CHECK(n_steps >= 1 && n_eps >= 0, "latent_decode: n_steps=%d n_eps=%d", n_steps, n_eps);
    CDX_CHECK(n_eps >= n_steps || extra_noise != nullptr, "latent_decode: %d steps but only %d recovered noises and no extra noise", n_steps, n_eps);
    LatentLoopArgs a;
    a.mode = LOOP_DEC;
    a.c_tgt = c; a.uc = uc; a.L = L; a.t_scale = scale;
    a.coef = coef; a.t_host = t_host; a.n_steps = n_steps;
    a.z_in = z; a.n_eps = n_eps; a.extra = extra_noise; a.x_out = x_out;
    a.B = B; a.C = C; a.h = h; a.w = w;
    with_arena(un->owner->e, S(stream), [&] { run_latent_loop(*un->n, a, S(stream)); });
  });
}

int cdx_cycle_lockstep(cdx_net* un, const float* x0, const float* c_src, const float* c_tgt, const float* uc, int L, float src_scale,
                       float tgt_scale, const cdx_ddim_coef* coef, const float* t_host, int n_steps, const float* noise, float sqrt_a_T,
                       float sqrt_1ma_T, float* x_out, float* z_out, int B, int C, int h, int w, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && x0 && c_src && c_tgt && coef && t_host && noise && x_out, "cycle_lockstep: null argument");
    CDX_CHECK(n_steps >= 1, "cycle_lockstep: n_steps=%d", n_steps);
    for (int i = 0; i < n_steps; ++i) CDX_CHECK(coef[i].sigma > 0.f, "cycle_lockstep: eta must be > 0 (sigma[%d] == 0), ddim.py:268", i);
    LatentLoopArgs a;
    a.mode = LOOP_LOCK;
    a.x0 = x0; a.c_src = c_src; a.c_tgt = c_tgt; a.uc = uc; a.L = L; a.s_scale = src_scale; a.t_scale = tgt_scale;
    a.coef = coef; a.t_host = t_host; a.n_steps = n_steps; a.n_rec = n_steps; a.noise = noise; a.sa = sqrt_a_T; a.s1 = sqrt_1ma_T;
    a.z_out = z_out; a.x_out = x_out; a.B = B; a.C = C; a.h = h; a.w = w;
    with_arena(un->owner->e, S(stream), [&] { run_latent_loop(*un->n, a, S(stream)); });
  });
}

int cdx_cycle_lockstep_pair(cdx_net* src, cdx_net* tgt, const float* x0, const float* c_src, const float* c_tgt, const float* uc, int L,
                            float src_scale, float tgt_scale, const cdx_ddim_coef* coef, const float* t_host, int n_steps, const float* noise,
                            float sqrt_a_T, float sqrt_1ma_T, float* x_out, float* z_out, int B, int C, int h, int w, void* stream) {
  return guard([&] {
    CDX_CHECK(src && src->owner && tgt && tgt->owner && x0 && ((c_src && c_tgt) || L == 0) && coef && t_host && noise && x_out,
              "cycle_lockstep_pair: null argument");
    CDX_CHECK(n_steps >= 1 && B > 0, "cycle_lockstep_pair: n_steps=%d B=%d", n_steps, B);
    CDX_CHECK(src->n->ucfg.context_dim == tgt->n->ucfg.context_dim, "cycle_lockstep_pair: context widths differ (%d, %d)",
              src->n->ucfg.context_dim, tgt->n->ucfg.context_dim);
    for (int i = 0; i < n_steps; ++i) CDX_CHECK(coef[i].sigma > 0.f, "cycle_lockstep_pair: eta must be > 0 (sigma[%d] == 0), ddim.py:268", i);
    LatentLoopArgs a;
    a.mode = LOOP_LOCK;
    a.x0 = x0; a.c_src = c_src; a.c_tgt = c_tgt; a.uc = uc; a.L = L; a.s_scale = src_scale; a.t_scale = tgt_scale;
    a.coef = coef; a.t_host = t_host; a.n_steps = n_steps; a.n_rec = n_steps; a.noise = noise; a.sa = sqrt_a_T; a.s1 = sqrt_1ma_T;
    a.z_out = z_out; a.x_out = x_out; a.B = B; a.C = C; a.h = h; a.w = w;
    with_arenas(src->owner->e, &tgt->owner->e, S(stream), [&] { run_latent_loop(*src->n, a, S(stream), tgt->n); });
  });
}

int cdx_latent_loop_ens(cdx_net* un, int mode, const float* x0, const float* c_src, const float* c_tgt, const float* uc, int L,
                        const float* src_scales, const float* tgt_scales, const cdx_ddim_coef* coef, const float* t_host, int n_steps, int n_rec,
                        const float* noise, float sqrt_a_T, float sqrt_1ma_T, const float* z_in, int n_eps, const float* extra_noise,
                        float* z_out, float* x_out, int B, int C, int h, int w, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && coef && t_host && mode >= LOOP_ENC && mode <= LOOP_LOCK, "latent_loop_ens: bad arguments (mode %d)", mode);
    const bool enc = mode & LOOP_ENC, dec = mode & LOOP_DEC;
    CDX_CHECK(n_steps >= 1, "latent_loop_ens: n_steps=%d", n_steps);
    LatentLoopArgs a;
    a.mode = mode;
    a.uc = uc; a.L = L; a.coef = coef; a.t_host = t_host; a.n_steps = n_steps;
    a.B = B; a.C = C; a.h = h; a.w = w;
    if (enc) {
      CDX_CHECK(x0 && c_src && noise && src_scales && uc, "latent_loop_ens: the encode chain needs x0, c_src, uc, noise and per-sample scales");
      if (mode == LOOP_LOCK) n_rec = n_steps;
      CDX_CHECK(n_rec >= 0 && n_rec <= n_steps, "latent_loop_ens: n_rec=%d", n_rec);
      for (int i = 0; i < n_rec; ++i) CDX_CHECK(coef[i].sigma > 0.f, "latent_loop_ens: eta must be > 0 (sigma[%d] == 0), ddim.py:268", i);
      CDX_CHECK(mode == LOOP_LOCK || z_out, "latent_loop_ens: encode needs z_out");
      a.x0 = x0; a.c_src = c_src; a.s_scale_v = src_scales; a.n_rec = n_rec; a.noise = noise; a.sa = sqrt_a_T; a.s1 = sqrt_1ma_T; a.z_out = z_out;
    }
    if (dec) {
      CDX_CHECK(c_tgt && tgt_scales && uc && x_out, "latent_loop_ens: the decode chain needs c_tgt, uc, per-sample scales and x_out");
      a.c_tgt = c_tgt; a.t_scale_v = tgt_scales; a.x_out = x_out;
      if (!enc) {
        CDX_CHECK(z_in && n_eps >= 0 && (n_eps >= n_steps || extra_noise), "latent_loop_ens: decode needs z (%d noises for %d steps) or extra noise", n_eps, n_steps);
        a.z_in = z_in; a.n_eps = n_eps; a.extra = extra_noise;
      }
    }
    with_arena(un->owner->e, S(stream), [&] { run_latent_loop(*un->n, a, S(stream)); });
  });
}

int cdx_pixel_encode(cdx_net* un, const float* x0, const cdx_pixel_coef* coef, const float* t_host, int n_rec, const float* noise,
                     float sqrt_a_T, float sqrt_1ma_T, float* z_out, int B, int C, int R, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && x0 && noise && z_out, "pixel_encode: null argument");
    CDX_CHECK(n_rec >= 0 && (n_rec == 0 || (coef && t_host)), "pixel_encode: n_rec=%d", n_rec);
    Engine& e = un->owner->e;
    Net& unet = *un->n;
    cudaStream_t s = S(stream);
    const int chw = C * R * R;
    const int net_chw = unet.ucfg.out_channels * R * R;
    const size_t n = (size_t)B * chw;
    with_arena(e, s, [&] {
      Scope sc(e.arena);
      float* xt = (float*)e.arena.alloc(n * sizeof(float));
      float* xn = (float*)e.arena.alloc(n * sizeof(float));
      float* eps = (float*)e.arena.alloc(n * sizeof(float));
      float* et = (float*)e.arena.alloc((size_t)B * net_chw * sizeof(float));
      float* tdev = (float*)e.arena.alloc((size_t)std::max(n_rec, 1) * B * sizeof(float));
      upload_timesteps(e, t_host, n_rec, B, tdev, s);
      q_sample(e, x0, noise, sqrt_a_T, sqrt_1ma_T, xt, n, s);                          // sample_xt, DW:310-314 (incl. the DW:483 index quirk)
      scatter_slot(e, xt, z_out, B, chw, n_rec + 1, 0, s);
      const int iters = e.dry() ? std::min(n_rec, 1) : n_rec;
      for (int i = 0; i < iters; ++i) {
        pixel_posterior_sample(e, x0, xt, noise + (size_t)(1 + i) * n, coef[i], xn, n, s);
        unet_forward(unet, xt, tdev + (size_t)i * B, nullptr, 0, et, B, R, R, s);
        pixel_compute_eps(e, xt, xn, et, coef[i], eps, B, chw, net_chw, s);
        scatter_slot(e, eps, z_out, B, chw, n_rec + 1, 1 + i, s);
        std::swap(xt, xn);
      }
    });
  });
}

int cdx_pixel_decode(cdx_net* un, const float* z, int n_eps, const cdx_pixel_coef* coef, const float* t_host, int n_steps,
                     const float* last_noise, float* x_out, int B, int C, int R, void* stream) {
  return guard([&] {
    CDX_CHECK(un && un->owner && z && coef && t_host && x_out, "pixel_decode: null argument");
    CDX_CHECK(n_steps >= 1 && n_eps >= 0 && n_eps <= n_steps, "pixel_decode: n_steps=%d n_eps=%d", n_steps, n_eps);
    Engine& e = un->owner->e;
    Net& unet = *un->n;
    cudaStream_t s = S(stream);
    const int chw = C * R * R;
    const int net_chw = unet.ucfg.out_channels * R * R;
    const size_t n = (size_t)B * chw;
    with_arena(e, s, [&] {
      Scope sc(e.arena);
      float* xa = (float*)e.arena.alloc(n * sizeof(float));
      float* xb = (float*)e.arena.alloc(n * sizeof(float));
      float* eps = (float*)e.arena.alloc(n * sizeof(float));
      float* et = (float*)e.arena.alloc((size_t)B * net_chw * sizeof(float));
      float* tdev = (float*)e.arena.alloc((size_t)n_steps * B * sizeof(float));
      upload_timesteps(e, t_host, n_steps, B, tdev, s);
      gather_slot(e, z, xa, B, chw, n_eps + 1, 0, s);
      const int iters = e.dry() ? 1 : n_steps;
      for (int i = 0; i < iters; ++i) {
        unet_forward(unet, xa, tdev + (size_t)i * B, nullptr, 0, et, B, R, R, s);
        const float* nz = nullptr;
        if (i < n_eps) { gather_slot(e, z, eps, B, chw, n_eps + 1, 1 + i, s); nz = eps; }
        else if (last_noise) nz = last_noise + (size_t)(i - n_eps) * n;
        float* dst = (i == n_steps - 1) ? x_out : xb;
        pixel_step_with_eps(e, xa, et, nz, coef[i], dst, B, chw, net_chw, s);
        std::swap(xa, xb);
      }
    });
  });
}

int cdx_pixel_cycle_lockstep(cdx_net* src, cdx_net* tgt, const float* x0, const cdx_pixel_coef* coef, const float* t_host, int n_steps,
                             const float* noise, float sqrt_a_T, float sqrt_1ma_T, const float* last_noise, float* x_out, float* z_out, int B,
                             int C, int R, void* stream) {
  return guard([&] {
    CDX_CHECK(src && src->owner && tgt && tgt->owner && x0 && coef && t_host && noise && x_out, "pixel_cycle_lockstep: null argument");
    CDX_CHECK(n_steps >= 1 && B > 0, "pixel_cycle_lockstep: n_steps=%d B=%d", n_steps, B);
    Engine& e = src->owner->e;
    Net& su = *src->n;
    Net& tu = *tgt->n;
    CDX_CHECK(su.ucfg.out_channels >= C && tu.ucfg.out_channels >= C, "pixel_cycle_lockstep: U-Nets with %d / %d output channels for C=%d",
              su.ucfg.out_channels, tu.ucfg.out_channels, C);
    cudaStream_t s = S(stream);
    const int chw = C * R * R;
    const int net_chw_s = su.ucfg.out_channels * R * R, net_chw_t = tu.ucfg.out_channels * R * R;
    const size_t n = (size_t)B * chw;
    const int n_rec = n_steps - 1;
    with_arenas(e, &tgt->owner->e, s, [&] {
      Scope sc(e.arena);
      float* xa = (float*)e.arena.alloc(n * sizeof(float));
      float* xb = (float*)e.arena.alloc(n * sizeof(float));
      float* ya = (float*)e.arena.alloc(n * sizeof(float));
      float* yb = (float*)e.arena.alloc(n * sizeof(float));
      float* es = (float*)e.arena.alloc((size_t)B * net_chw_s * sizeof(float));
      float* et = (float*)e.arena.alloc((size_t)B * net_chw_t * sizeof(float));
      float* tdev = (float*)e.arena.alloc((size_t)n_steps * B * sizeof(float));
      upload_timesteps(e, t_host, n_steps, B, tdev, s);
      q_sample(e, x0, noise, sqrt_a_T, sqrt_1ma_T, xa, n, s);                          // sample_xt, DW:310-314 (incl. the DW:483 index quirk)
      if (z_out) scatter_slot(e, xa, z_out, B, chw, n_steps, 0, s);
      const float* y = xa;                                                           // the target chain starts from the same x_T
      float* yn = ya;
      const int iters = e.dry() ? std::min(n_rec, 1) : n_rec;
      for (int i = 0; i < iters; ++i) {
        unet_forward(su, xa, tdev + (size_t)i * B, nullptr, 0, es, B, R, R, s);
        unet_forward(tu, y, tdev + (size_t)i * B, nullptr, 0, et, B, R, R, s);
        PixelLockStep st;
        st.n = n; st.chw = chw;
        st.cs = coef[i]; st.ct = coef[i];
        st.x0 = x0; st.xt = xa; st.noise = noise + (size_t)(1 + i) * n; st.x_next = xb;
        st.et_src = es; st.net_chw_src = net_chw_s;
        st.y = y; st.et_tgt = et; st.net_chw_tgt = net_chw_t; st.y_next = yn;
        if (z_out) { st.z_out = z_out + (size_t)(1 + i) * chw; st.z_stride = (long long)n_steps * chw; }
        pixel_lock_step(e, st, s);
        std::swap(xa, xb);
        y = yn;
        yn = (yn == ya) ? yb : ya;
      }
      // the last target step (0, -1) has no recovered noise: its draw is multiplied by 0 (DU:115,131)
      unet_forward(tu, y, tdev + (size_t)n_rec * B, nullptr, 0, et, B, R, R, s);
      pixel_step_with_eps(e, y, et, last_noise, coef[n_rec], x_out, B, chw, net_chw_t, s);
    });
  });
}

// ---------------------------------------------------------------- unit-test hooks
int cdx_op_gemm(cdx_engine* eh, const cdx_gemm_test* t, void* stream) {
  return guard([&] {
    CDX_CHECK(eh && t && t->A && t->w && t->C && t->N > 0 && t->C1 > 0, "op_gemm: null argument / empty problem");
    CDX_CHECK(!t->A2 || (!t->conv && t->C2 > 0), "op_gemm: a second source needs dense mode and C2 > 0");
    CDX_CHECK(!t->geglu || (!t->conv && (t->N % 128) == 0 && !t->c_stats), "op_gemm: GEGLU needs dense mode, N %% 128 == 0 and no statistics");
    Engine& e = eh->e;
    cudaStream_t s = S(stream);
    const int C2 = t->A2 ? t->C2 : 0;
    GemmArgs g;
    g.N = t->N;
    if (t->conv) {
      CDX_CHECK(t->B > 0 && t->H > 0 && t->W > 0 && (t->stride == 1 || t->stride == 2) && t->up >= 1, "op_gemm: bad conv geometry");
      const int Hl = t->H * t->up, Wl = t->W * t->up;
      g.mode = 1;
      g.Hout = t->stride == 1 ? Hl : Hl / 2;
      g.Wout = t->stride == 1 ? Wl : Wl / 2;
      g.M = t->B * g.Hout * g.Wout; g.K = 9 * t->C1;
      g.Hin = t->H; g.Win = t->W; g.stride = t->stride; g.pad = t->pad; g.up = t->up;
    } else {
      CDX_CHECK(t->M > 0, "op_gemm: M = %d", t->M);
      g.M = t->M; g.K = t->C1 + C2;
    }
    const int rows_img = t->conv ? g.Hout * g.Wout : g.M;
    g.A = t->A; g.lda = t->C1; g.C1 = t->C1;
    g.A2 = t->A2; g.lda2 = C2; g.C2 = C2;
    g.a_amax = t->a_amax; g.a2_amax = t->a2_amax;
    g.ldb = g.K;
    g.rowvec = t->rowvec; g.ld_rowvec = t->ld_rowvec;
    g.rows_per_batch = t->rows_per_batch > 0 ? t->rows_per_batch : rows_img;
    g.residual = t->residual; g.ldr = t->ldr > 0 ? t->ldr : t->N;
    g.alpha = t->alpha;
    g.geglu = t->geglu;
    g.Cout = t->C; g.ldc = t->ldc > 0 ? t->ldc : (t->geglu ? t->N / 2 : t->N);
    g.out_nchw = t->out_nchw; g.rows_per_img = t->rows_per_img > 0 ? t->rows_per_img : rows_img;
    g.Cout_lo = t->C_lo;
    g.Ct_hi = t->Ct_hi; g.Ct_lo = t->Ct_lo; g.t_col0 = t->t_col0; g.ldt = t->ldt > 0 ? t->ldt : g.M;
    g.c_amax = t->c_amax; g.c_stats = t->c_stats;
    CDX_CHECK(!t->c_stats || g.M % g.rows_per_batch == 0, "op_gemm: statistics need whole images (M=%d, rows_per_batch=%d)", g.M, g.rows_per_batch);
    with_arena(e, s, [&] {
      Scope sc(e.arena);
      e.pools_reset(s);
      e.last_gemm = cdx_gemm_plan{-1, 0, 0, 0, 0, 0, 0};
      const size_t nw = (size_t)g.N * g.K;
      // the weight as the networks store it: conv3x3 repacked O,kh,kw,I; GEGLU rows as [32 value | 32 gate] blocks (bias too)
      const float* w = t->w;
      if (t->conv) {
        float* wr = (float*)e.arena.alloc(nw * sizeof(float));
        repack_conv3x3(e, t->w, wr, g.N, t->C1, s);
        w = wr;
      } else if (t->geglu) {
        float* wi = (float*)e.arena.alloc(nw * sizeof(float));
        interleave_geglu_rows(e, t->w, wi, g.N, g.K, s);
        w = wi;
      }
      g.Bw = w;
      g.bias = t->bias;
      if (t->geglu && t->bias) {
        float* bi = (float*)e.arena.alloc((size_t)g.N * sizeof(float));
        interleave_geglu_rows(e, t->bias, bi, g.N, 1, s);
        g.bias = bi;
      }
      if (e.mma_mode == 1) {   // the operand planes the networks build at finalize: TF32 (TS kernel) and fp16-split
        float* hi = (float*)e.arena.alloc(nw * sizeof(float));
        float* lo = (float*)e.arena.alloc(nw * sizeof(float));
        split_planes(e, w, hi, lo, nw, s);
        g.Bw_hi = hi; g.Bw_lo = lo;
        hook_h16_planes(e, w, nw, g, s);
      }
      if (!e.dry()) {
        if (t->c_amax) CDX_CUDA(cudaMemsetAsync(t->c_amax, 0, sizeof(float), s));
        if (t->c_stats) CDX_CUDA(cudaMemsetAsync(t->c_stats, 0, (size_t)(g.M / g.rows_per_batch) * g.N * 2 * sizeof(double), s));
      }
      gemm(e, g, s);
    });
    if (t->plan) *t->plan = e.last_gemm;
  });
}
int cdx_op_groupnorm(cdx_engine* eh, const float* x, int C1, const float* x2, int C2, const float* gamma, const float* beta, float eps, int silu_,
                     const float* scale, const float* shift, int ld_ss, const double* st1, const double* st2, float* amax, float* y, int B, int HW,
                     void* stream) {
  return guard([&] {
    CDX_CHECK(eh && x && gamma && beta && y && (!x2 || C2 > 0), "op_groupnorm: null argument");
    Engine& e = eh->e;
    cudaStream_t s = S(stream);
    with_arena(e, s, [&] {
      e.pools_reset(s);
      if (amax && !e.dry()) CDX_CUDA(cudaMemsetAsync(amax, 0, sizeof(float), s));
      groupnorm(e, x, C1, x2, x2 ? C2 : 0, gamma, beta, eps, silu_ != 0, scale, shift, ld_ss, y, B, HW, s, st1, st2, amax);
    });
  });
}
int cdx_op_layernorm(cdx_engine* eh, const float* x, const float* gamma, const float* beta, float* y, int M, int C, void* stream) {
  ENG_CALL(eh, layernorm(eh->e, x, gamma, beta, y, M, C, S(stream)));
}
int cdx_op_attention(cdx_engine* eh, const float* q, const float* k, const float* v, float* out, int B, int Nq, int Nk, int heads, int d, float scale,
                     void* stream) {
  return guard([&] {
    CDX_CHECK(eh && q && k && v && out, "op_attention: null argument");
    const int C = heads * d;
    Engine& e = eh->e;
    cudaStream_t s = S(stream);
    with_arena(e, s, [&] {
      Scope sc(e.arena);
      bool done = false;
      if (e.mma_mode == 1 && e.flash_attn && e.tc_kind >= 1 && (Nq % 128) == 0 && (C % 8) == 0 && (d == 16 || d == 32 || d == 40 || d == 64 || d == 80)) {
        // the SpatialTransformer's fp16-split path on loose q / k / v: ranges measured here, keys padded to a multiple of 8 per image
        e.pools_reset(s);
        const int Nks = (Nk + 7) & ~7, M = B * Nq, Mk = B * Nks;
        float *qa = e.amax_slot(), *ka = e.amax_slot(), *va = e.amax_slot();
        amax_rows(e, q, M, C, C, qa, s);
        amax_rows(e, k, (long long)B * Nk, C, C, ka, s);
        amax_rows(e, v, (long long)B * Nk, C, C, va, s);
        const float *kp = k, *vp = v;
        if (Nks != Nk) {
          float* kb = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
          float* vb = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
          if (!e.dry()) {
            CDX_CUDA(cudaMemsetAsync(kb, 0, (size_t)Mk * C * 4, s));
            CDX_CUDA(cudaMemsetAsync(vb, 0, (size_t)Mk * C * 4, s));
            CDX_CUDA(cudaMemcpy2DAsync(kb, (size_t)Nks * C * 4, k, (size_t)Nk * C * 4, (size_t)Nk * C * 4, B, cudaMemcpyDeviceToDevice, s));
            CDX_CUDA(cudaMemcpy2DAsync(vb, (size_t)Nks * C * 4, v, (size_t)Nk * C * 4, (size_t)Nk * C * 4, B, cudaMemcpyDeviceToDevice, s));
          }
          kp = kb; vp = vb;
        }
        void* qh = e.arena.alloc((size_t)M * C * 2);
        void* ql = e.arena.alloc((size_t)M * C * 2);
        void* kh = e.arena.alloc((size_t)Mk * C * 2);
        void* kl = e.arena.alloc((size_t)Mk * C * 2);
        void* vh = e.arena.alloc((size_t)Mk * C * 2);
        void* vl = e.arena.alloc((size_t)Mk * C * 2);
        split_rows_h16(e, q, M, C, C, qh, ql, C, qa, s);
        split_rows_h16(e, kp, Mk, C, C, kh, kl, C, ka, s);
        split_transpose_h16(e, vp, Mk, C, C, vh, vl, va, s);
        done = flash_attention_h16(e, qh, ql, C, kh, kl, C, vh, vl, qa, ka, va, out, C, B, Nq, Nk, Nks, heads, d, scale, s);
      }
      if (!done && e.mma_mode == 1 && Nq == Nk && (Nq % 32) == 0 && Nq >= 128 && (d % 4) == 0) {
        // same operand preparation as the SpatialTransformer: q|k side by side, V transposed, TF32 planes
        const int M = B * Nq;
        float* qk = (float*)e.arena.alloc((size_t)M * 2 * C * sizeof(float));
        float* vt = (float*)e.arena.alloc((size_t)C * M * sizeof(float));
        if (!e.dry()) {
          CDX_CUDA(cudaMemcpy2DAsync(qk, (size_t)2 * C * 4, q, (size_t)C * 4, (size_t)C * 4, M, cudaMemcpyDeviceToDevice, s));
          CDX_CUDA(cudaMemcpy2DAsync(qk + C, (size_t)2 * C * 4, k, (size_t)C * 4, (size_t)C * 4, M, cudaMemcpyDeviceToDevice, s));
        }
        nhwc_to_nchw(e, v, vt, 1, C, M, s);
        if (e.flash_attn && (Nq % 128) == 0) {
          float* qh = (float*)e.arena.alloc((size_t)M * 2 * C * sizeof(float));
          float* ql = (float*)e.arena.alloc((size_t)M * 2 * C * sizeof(float));
          float* vh = (float*)e.arena.alloc((size_t)C * M * sizeof(float));
          float* vl = (float*)e.arena.alloc((size_t)C * M * sizeof(float));
          split_planes(e, qk, qh, ql, (size_t)M * 2 * C, s);
          split_planes(e, vt, vh, vl, (size_t)C * M, s);
          done = flash_attention_tc(e, qh, ql, 2 * C, qh + C, ql + C, 2 * C, vh, vl, out, C, B, Nq, Nq, Nq, heads, d, scale, s);
        }
        if (!done) done = attention_tc(e, qk, 2 * C, qk + C, 2 * C, d, vt, out, C, B, Nq, Nk, heads, d, scale, s);
      }
      if (!done && e.mma_mode == 1 && e.flash_attn && Nq != Nk && (Nq % 128) == 0) {
        // cross-attention shape: keys padded to a multiple of 4 per image (TMA strides), masked inside the kernel
        const int Nks = (Nk + 3) & ~3, M = B * Nq, Mk = B * Nks;
        float* kp = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
        float* vp = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
        float* vt = (float*)e.arena.alloc((size_t)C * Mk * sizeof(float));
        float* qh = (float*)e.arena.alloc((size_t)M * C * sizeof(float));
        float* ql = (float*)e.arena.alloc((size_t)M * C * sizeof(float));
        float* kh = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
        float* kl = (float*)e.arena.alloc((size_t)Mk * C * sizeof(float));
        float* vh = (float*)e.arena.alloc((size_t)C * Mk * sizeof(float));
        float* vl = (float*)e.arena.alloc((size_t)C * Mk * sizeof(float));
        if (!e.dry()) {
          CDX_CUDA(cudaMemsetAsync(kp, 0, (size_t)Mk * C * 4, s));
          CDX_CUDA(cudaMemsetAsync(vp, 0, (size_t)Mk * C * 4, s));
          CDX_CUDA(cudaMemcpy2DAsync(kp, (size_t)Nks * C * 4, k, (size_t)Nk * C * 4, (size_t)Nk * C * 4, B, cudaMemcpyDeviceToDevice, s));
          CDX_CUDA(cudaMemcpy2DAsync(vp, (size_t)Nks * C * 4, v, (size_t)Nk * C * 4, (size_t)Nk * C * 4, B, cudaMemcpyDeviceToDevice, s));
        }
        nhwc_to_nchw(e, vp, vt, 1, C, Mk, s);
        split_planes(e, q, qh, ql, (size_t)M * C, s);
        split_planes(e, kp, kh, kl, (size_t)Mk * C, s);
        split_planes(e, vt, vh, vl, (size_t)C * Mk, s);
        done = flash_attention_tc(e, qh, ql, C, kh, kl, C, vh, vl, out, C, B, Nq, Nk, Nks, heads, d, scale, s);
      }
      if (!done) attention(e, q, C, k, C, v, C, out, C, B, Nq, Nk, heads, d, d, scale, s);
    });
  });
}
int cdx_op_nchw_to_nhwc(cdx_engine* eh, const float* x, float* y, int B, int C, int HW, void* stream) { ENG_CALL(eh, nchw_to_nhwc(eh->e, x, y, B, C, HW, S(stream))); }
int cdx_op_nhwc_to_nchw(cdx_engine* eh, const float* x, float* y, int B, int C, int HW, void* stream) { ENG_CALL(eh, nhwc_to_nchw(eh->e, x, y, B, C, HW, S(stream))); }

}  // extern "C"
