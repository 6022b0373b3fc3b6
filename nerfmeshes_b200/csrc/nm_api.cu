// C ABI of libnerfmeshes_b200.so (include/nerfmeshes_b200.h): handle lifecycle, weight loading, and the orchestration
// of the hot path — the body of NeRFModel.forward / BuFFModel.forward (src/models/model_nerf.py:37-78,
// model_buff.py:34-69) and extract_radiance (src/mesh_nerf.py:27-53) as stream-ordered kernel sequences.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "nm_common.h"

namespace nm {
const char* last_error();
}

using namespace nm;

namespace {

struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); return -2; }
    cap = want;
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

}  // namespace

struct NmHandle_t {
  int device = 0;
  int num_sms = 0;
  NmRenderCfg cfg{};
  NetDev nets[2];
  bool has_fine = false;
  NmNetDesc desc[2]{};
  Buf s_table, u_table, voxels;
  int V = 0;
  // workspace
  Buf t_c, raw_c, w_c, t_f, raw_f, t_u, dirs, origins, lin[3], small, stage_in[3], stage_out[12];
  int lin_n[3] = {0, 0, 0};
  int* d_err = nullptr;       // [0] tcgen05 watchdog code, [1] aabb hit-list overflow (device alias of h_err)
  int* h_err = nullptr;       // mapped pinned host memory: still readable after a device-side trap
  double* d_stats = nullptr;
  cudaStream_t own_stream = nullptr;
  int64_t launches = 0;
  // timing of the fused-MLP launches
  bool timing = false;
  std::vector<cudaEvent_t> ev;
  size_t ev_used = 0;
  int64_t mlp_points = 0, mlp_launches = 0;
  size_t mc_ws_bytes = 0;
  void* mc_ws_ptr = nullptr;
  size_t mc_ws2_bytes = 0;
  void* mc_ws2_ptr = nullptr;
  int64_t mc_counts[2] = {0, 0};   // {vertices, triangles} of the last count step: sizes of the emit step
  // training (nm_train.cu): gradient accumulators per network + scratch
  Buf g_wt[2], g_bias[2], g_head[2], train_ws, dout, trans, tr_rgb[2], tr_drgb[2];
  bool grads_ready = false;
  Buf metric_ws;                   // nearest-neighbour merge keys / area CDF of the surface sampler (nm_metrics.cu)
};

namespace {

// rays per internal chunk (bounds the per-sample workspace: 20 B x 192 samples x 1 Mi rays = 4 GB); NM_CHUNK_RAYS overrides (tests)
long long chunk_rays() {
  static long long v = [] { const char* e = getenv("NM_CHUNK_RAYS"); long long x = e ? atoll(e) : 0; return x > 0 ? x : (1ll << 20); }();
  return v;
}

int check_kernel_flags(NmHandle h);

int bind_device(NmHandle h) {
  NM_CHECK(h != nullptr, "null handle");
  NM_CUDA(cudaSetDevice(h->device));
  return 0;
}

// device-pointer (asynchronous) entry points cannot wait for their own kernels; they report the device-side error flags
// raised by EARLIER work on this handle (mapped host memory, no synchronisation) and callers that need the answer for
// the current call use nm_check_flags(h, stream), which synchronises first.
int bind_checked(NmHandle h) {
  if (int e = bind_device(h)) return e;
  return check_kernel_flags(h);
}

void linspace_host(int n, std::vector<float>* out) {  // torch.linspace(0,1,n) fp32 (ATen's two-sided formula)
  out->resize(n);
  if (n == 1) { (*out)[0] = 0.f; return; }
  const float step = 1.0f / (float)(n - 1);
  for (int i = 0; i < n; ++i) (*out)[i] = (i < n / 2) ? 0.f + step * (float)i : 1.0f - step * (float)(n - 1 - i);
}

int upload(Buf* b, const void* src, size_t bytes) {
  if (int e = b->ensure(bytes)) return e;
  NM_CUDA(cudaMemcpy(b->p, src, bytes, cudaMemcpyHostToDevice));
  return 0;
}

int check_kernel_flags(NmHandle h) {
  const volatile int* flags = h->h_err;
  NM_CHECK(flags[0] == 0, "tcgen05 pipeline watchdog fired (code %d)", flags[0]);
  NM_CHECK(flags[1] == 0, "AABB sampler: more than 512 voxel hits on one ray (samples / voxel indices of that ray are truncated)");
  return 0;
}

// one fused-MLP launch in the configured arithmetic
int run_mlp(NmHandle h, int which, bool sigma_only, const MlpInput& in, float* out, cudaStream_t st, const MlpEmit* emit = nullptr,
            const CompositeArgs* comp = nullptr) {
  const NetDev& net = h->nets[which];
  NM_CHECK(net.loaded, "weights of network %d not loaded", which);
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (h->timing) {
    while (h->ev.size() < h->ev_used + 2) {
      cudaEvent_t e;
      NM_CUDA(cudaEventCreate(&e));
      h->ev.push_back(e);
    }
    e0 = h->ev[h->ev_used++]; e1 = h->ev[h->ev_used++];
    NM_CUDA(cudaEventRecord(e0, st));
  }
  int rc;
  if (h->cfg.precision == NM_PREC_FP32) rc = launch_mlp_simt(net, sigma_only, in, out, st, &h->launches);
  else rc = launch_mlp_tc(net, sigma_only, h->cfg.precision == NM_PREC_FAST ? 1 : 3, h->cfg.act_scale_log2, in, out,
                          h->num_sms, h->d_err, st, &h->launches, emit, comp);
  if (rc) return rc;
  if (h->timing) {
    NM_CUDA(cudaEventRecord(e1, st));
    h->mlp_points += in.M;
    h->mlp_launches += 1;
  }
  return 0;
}

constexpr uint64_t kNoiseSaltMain = 0x5bd1e995ull, kNoiseSaltCoarse = 0x7f4a7c15a3c59ac3ull;

struct RayBatch {
  const float* origins; int o_stride; const float* dirs; long long R;
  float nf[2]; const float* near_dev; const float* far_dev;
};

float* off(float* p, long long n) { return p ? p + n : nullptr; }

// NeRFModel.forward / BuFFModel.forward for one chunk of rays; `o` already offset to the chunk.
// emit_c / emit_f: training only — the coarse (or only) / fine network's forward also leaves the backward's operands (MlpEmit)
// need_raw: the caller reads h->raw_c / h->raw_f afterwards (the training backward) — otherwise the compositor runs inside the
// MLP kernel and the per-sample network outputs never reach HBM (NM_FUSED_COMPOSITE=0 keeps the two-kernel path for A/B tests).
int render_chunk(NmHandle h, const RayBatch& rb, int flags, uint64_t seed, const NmRenderOut& o, cudaStream_t st,
                 const MlpEmit* emit_c = nullptr, const MlpEmit* emit_f = nullptr, bool need_raw = false) {
  const NmRenderCfg& c = h->cfg;
  const long long R = rb.R;
  const int Nc = c.num_coarse;
  const bool buff = flags & NM_FLAG_BUFF;
  const bool teacher = flags & NM_FLAG_TEACHER_T;
  const bool training = flags & NM_FLAG_TRAINING;
  const int Nf = (h->has_fine && !buff) ? c.num_fine : 0;
  const int S = Nc + Nf;
  // the coarse and the fine compositor draw independent sigma noise (two torch.randn calls in the reference): distinct salts
  auto rays_input = [&](const float* t, int s) {
    MlpInput in{};
    in.mode = IN_RAYS; in.dirs = rb.dirs; in.ray_o = rb.origins; in.o_stride = rb.o_stride; in.t = t; in.S = s;
    in.M = R * s;
    return in;
  };
  const char* fe = getenv("NM_FUSED_COMPOSITE");       // read per call: the tests flip it to compare the two paths
  const bool fused_env = !fe || atoi(fe) != 0;
  // network `which` on the samples t (R,s) + VolumeRenderer: one launch when eligible, else raw (R,s,4) through `raw_buf`
  auto mlp_composite = [&](int which, Buf& raw_buf, const MlpEmit* emit, const float* t, int s, float* rgb, float* depth,
                           float* depth_raw, float* acc, float* disp, float* w, float* mw, uint64_t salt = kNoiseSaltMain) -> int {
    CompositeArgs a{};
    a.t = t; a.dirs = rb.dirs; a.R = R; a.S = s; a.noise_std = c.noise_std; a.seed = seed ^ salt;
    a.white_bg = c.white_background; a.training = training ? 1 : 0; a.thr = c.attenuation_threshold;
    a.rgb = rgb; a.depth = depth; a.depth_raw = depth_raw; a.acc = acc; a.disp = disp; a.weights = w; a.mask_weights = mw;
    const bool fuse = fused_env && !need_raw && !emit && c.precision != NM_PREC_FP32 && mlp_tc_composite_group(s) > 0;
    if (fuse) return run_mlp(h, which, false, rays_input(t, s), nullptr, st, nullptr, &a);
    if (int e = raw_buf.ensure((size_t)R * s * 16)) return e;
    if (int e = run_mlp(h, which, false, rays_input(t, s), raw_buf.as<float>(), st, emit)) return e;
    a.raw = raw_buf.as<float>();
    return launch_composite(a, st, &h->launches);
  };

  if (teacher) {
    NM_CHECK(o.t_vals != nullptr, "NM_FLAG_TEACHER_T needs out.t_vals as input");
    const int which = (h->has_fine && !buff) ? NM_NET_FINE : NM_NET_COARSE;
    return mlp_composite(which, h->raw_f, nullptr, o.t_vals, S, o.rgb, o.depth, o.depth_raw, o.acc, o.disp, o.weights, o.mask_weights);
  }

  // coarse / uniform samples (a3)
  if (int e = h->t_c.ensure((size_t)R * Nc * 4)) return e;
  float* t_c = h->t_c.as<float>();
  if (int e = launch_stratified(h->s_table.as<float>(), Nc, R, rb.nf, rb.near_dev, rb.far_dev, c.lindisp, c.perturb,
                                seed, t_c, st, &h->launches)) return e;
  if (buff) {
    NM_CHECK(h->V > 0, "BuFF render without a voxel list (nm_set_tree)");
    NM_CHECK(rb.near_dev == nullptr, "BuFF path takes scalar near/far");
    if (int e = h->t_u.ensure((size_t)R * Nc * 4)) return e;
    float* z = h->t_u.as<float>();
    if (int e = launch_aabb(h->voxels.as<float>(), h->V, rb.origins, rb.o_stride, rb.dirs, R, rb.nf[0], rb.nf[1], Nc,
                            h->s_table.as<float>(), t_c, z, nullptr, h->d_err + 1, st, &h->launches,
                            (flags & NM_FLAG_RANDOM_VOXELS) ? 1 : 0, seed)) return e;
    if (o.t_vals) NM_CUDA(cudaMemcpyAsync(o.t_vals, z, (size_t)R * Nc * 4, cudaMemcpyDeviceToDevice, st));
    return mlp_composite(NM_NET_COARSE, h->raw_c, emit_c, z, Nc, o.rgb, o.depth, o.depth_raw, o.acc, o.disp, o.weights, o.mask_weights);
  }
  if (Nf == 0) {
    if (o.t_vals) NM_CUDA(cudaMemcpyAsync(o.t_vals, t_c, (size_t)R * Nc * 4, cudaMemcpyDeviceToDevice, st));
    return mlp_composite(NM_NET_COARSE, h->raw_c, emit_c, t_c, Nc, o.rgb, o.depth, o.depth_raw, o.acc, o.disp, o.weights, o.mask_weights);
  }
  float* w_c = o.coarse_weights;
  if (!w_c) { if (int e = h->w_c.ensure((size_t)R * Nc * 4)) return e; w_c = h->w_c.as<float>(); }
  if (int e = mlp_composite(NM_NET_COARSE, h->raw_c, emit_c, t_c, Nc, o.coarse_rgb, nullptr, nullptr, o.coarse_acc, o.coarse_disp, w_c,
                            nullptr, kNoiseSaltCoarse)) return e;
  // inverse-CDF resampling + merge (a8)
  float* t_f = o.t_vals;
  if (!t_f) { if (int e = h->t_f.ensure((size_t)R * S * 4)) return e; t_f = h->t_f.as<float>(); }
  if (int e = launch_invcdf(t_c, w_c, h->u_table.as<float>(), Nc, Nf, R, c.perturb, seed ^ 0x9e3779b9u, t_f, st, &h->launches)) return e;
  return mlp_composite(NM_NET_FINE, h->raw_f, emit_f, t_f, S, o.rgb, o.depth, o.depth_raw, o.acc, o.disp, o.weights, o.mask_weights);
}

NmRenderOut offset_out(const NmRenderOut& o, long long r0, int S, int Nc) {
  NmRenderOut q = o;
  q.rgb = off(o.rgb, 3 * r0); q.depth = off(o.depth, r0); q.depth_raw = off(o.depth_raw, r0); q.acc = off(o.acc, r0);
  q.disp = off(o.disp, r0); q.weights = off(o.weights, r0 * S); q.mask_weights = off(o.mask_weights, r0 * S);
  q.t_vals = off(o.t_vals, r0 * S); q.coarse_rgb = off(o.coarse_rgb, 3 * r0); q.coarse_acc = off(o.coarse_acc, r0);
  q.coarse_disp = off(o.coarse_disp, r0); q.coarse_weights = off(o.coarse_weights, r0 * Nc);
  return q;
}

int out_samples(NmHandle h, int flags) {
  const bool buff = flags & NM_FLAG_BUFF;
  return h->cfg.num_coarse + ((h->has_fine && !buff) ? h->cfg.num_fine : 0);
}

int render_rays_impl(NmHandle h, const float* origins, int o_stride, const float* dirs, long long R, const float* nf_host,
                     const float* near_dev, const float* far_dev, int flags, uint64_t seed, const NmRenderOut& out,
                     cudaStream_t st) {
  NM_CHECK(o_stride == 0 || o_stride == 3, "o_stride must be 0 or 3");
  NM_CHECK(dirs && origins, "null ray pointers");
  NM_CHECK((near_dev == nullptr) == (far_dev == nullptr), "near_dev / far_dev must be given together");
  NM_CHECK(near_dev || nf_host, "no near/far bounds given");
  NM_CHECK(h->s_table.p != nullptr, "sampler tables missing");
  const int S = out_samples(h, flags);
  const long long kChunk = chunk_rays();
  for (long long r0 = 0; r0 < R; r0 += kChunk) {
    RayBatch rb{};
    rb.R = (R - r0 < kChunk) ? R - r0 : kChunk;
    rb.origins = origins + (long long)o_stride * r0; rb.o_stride = o_stride; rb.dirs = dirs + 3 * r0;
    if (nf_host) { rb.nf[0] = nf_host[0]; rb.nf[1] = nf_host[1]; }
    rb.near_dev = near_dev ? near_dev + r0 : nullptr; rb.far_dev = far_dev ? far_dev + r0 : nullptr;
    if (int e = render_chunk(h, rb, flags, seed + (uint64_t)r0, offset_out(out, r0, S, h->cfg.num_coarse), st)) return e;
  }
  return 0;
}

// host-buffer calls: a device-side NmRenderOut whose non-null fields mirror the caller's host block
int stage_outputs(NmHandle h, const NmRenderOut& host, long long R, int S, int Nc, NmRenderOut* dev, size_t sizes[12]) {
  float* const* hp = reinterpret_cast<float* const*>(&host);
  float** dp = reinterpret_cast<float**>(dev);
  const size_t per[12] = {3, 1, 1, 1, 1, (size_t)S, (size_t)S, (size_t)S, 3, 1, 1, (size_t)Nc};
  for (int i = 0; i < 12; ++i) {
    sizes[i] = (size_t)R * per[i] * sizeof(float);
    if (hp[i]) { if (int e = h->stage_out[i].ensure(sizes[i])) return e; dp[i] = h->stage_out[i].as<float>(); }
    else dp[i] = nullptr;
  }
  return 0;
}

int copy_outputs(const NmRenderOut& host, const NmRenderOut& dev, const size_t sizes[12], cudaStream_t st) {
  float* const* hp = reinterpret_cast<float* const*>(&host);
  float* const* dp = reinterpret_cast<float* const*>(&dev);
  for (int i = 0; i < 12; ++i)
    if (hp[i]) NM_CUDA(cudaMemcpyAsync(hp[i], dp[i], sizes[i], cudaMemcpyDeviceToHost, st));
  return 0;
}

// ---------------------------------------------------------------------------------------------- training backward
int ensure_grads(NmHandle h, cudaStream_t st, bool zero) {
  for (int w = 0; w < 2; ++w) {
    const NetDev& net = h->nets[w];
    if (!net.loaded) continue;
    size_t go[kMaxLayers]; int gl[kMaxLayers];
    const size_t nb[3] = {grad_layout(net.full, go, gl) * 4, (size_t)net.full.n_bias * 4, (size_t)(net.full.n_head > 0 ? net.full.n_head : 1) * 4};
    Buf* bufs[3] = {&h->g_wt[w], &h->g_bias[w], &h->g_head[w]};
    for (int i = 0; i < 3; ++i) {
      const bool fresh = bufs[i]->p == nullptr || bufs[i]->cap < nb[i];
      if (int e = bufs[i]->ensure(nb[i])) return e;
      if (fresh || zero) NM_CUDA(cudaMemsetAsync(bufs[i]->p, 0, bufs[i]->cap, st));
    }
  }
  h->grads_ready = true;
  return 0;
}

// One chunk of rays: forward (fills the per-sample workspaces), then for each bundle that carries a gradient the
// compositor adjoint and the network backward over sub-chunks of points.
int train_chunk(NmHandle h, const RayBatch& rb, int flags, uint64_t seed, const float* d_rgb, const float* d_rgb_coarse,
                const float* target, long long R_total, float* loss_dev, cudaStream_t st) {
  const NmRenderCfg& c = h->cfg;
  const long long R = rb.R;
  const bool buff = flags & NM_FLAG_BUFF;
  const bool two = h->has_fine && !buff && c.num_fine > 0;
  const int Nc = c.num_coarse, S = Nc + (two ? c.num_fine : 0);
  NmRenderOut o{};
  if (int e = h->tr_rgb[0].ensure((size_t)R * 12)) return e;
  o.rgb = h->tr_rgb[0].as<float>();
  if (two) { if (int e = h->tr_rgb[1].ensure((size_t)R * 12)) return e; o.coarse_rgb = h->tr_rgb[1].as<float>(); }
  // Direct mode: when the backward's workspace for ALL points of the chunk fits the budget (NM_TRAIN_DIRECT_GB, default 48),
  // the training forward itself emits the masks / activation packs and the backward skips its recompute launch; larger
  // chunks are walked in sub-chunks with a recompute each (below).
  const bool use_tc = c.precision != NM_PREC_FP32;
  const char* dg_env = getenv("NM_TRAIN_DIRECT_GB");      // read per call: the tests flip it to cover both walks
  const double direct_gb = dg_env ? atof(dg_env) : 48.0;
  const size_t ws_main = train_fused(use_tc) && c.act_scale_log2 == 0 ? train_ws_bytes(h->nets[two ? NM_NET_FINE : NM_NET_COARSE].full, R * S, true) + 1024 : 0;
  const size_t ws_coarse = (ws_main && two) ? train_ws_bytes(h->nets[NM_NET_COARSE].full, R * Nc, true) + 1024 : 0;
  const bool direct = ws_main > 0 && (double)(ws_main + ws_coarse) <= direct_gb * 1e9 && (d_rgb || target) && (!two || d_rgb_coarse || target);
  float *ws_m = nullptr, *ws_c = nullptr;
  MlpEmit em_main{}, em_coarse{};
  if (direct) {
    if (int e = h->train_ws.ensure(ws_main + ws_coarse + 2048)) return e;
    ws_m = reinterpret_cast<float*>(((uintptr_t)h->train_ws.p + 1023) & ~(uintptr_t)1023);
    train_emit_setup(h->nets[two ? NM_NET_FINE : NM_NET_COARSE].full, R * S, ws_m, &em_main);
    if (two) {
      ws_c = reinterpret_cast<float*>(((uintptr_t)ws_m + ws_main + 1023) & ~(uintptr_t)1023);
      train_emit_setup(h->nets[NM_NET_COARSE].full, R * Nc, ws_c, &em_coarse);
    }
    if (int e = render_chunk(h, rb, flags, seed, o, st, two ? &em_coarse : &em_main, two ? &em_main : nullptr, true)) return e;
  } else {
    if (int e = render_chunk(h, rb, flags, seed, o, st, nullptr, nullptr, true)) return e;
  }
  if (target) {
    for (int i = 0; i < (two ? 2 : 1); ++i) {
      if (int e = h->tr_drgb[i].ensure((size_t)R * 12)) return e;
      // loss_dev[0] = coarse (or only) bundle, loss_dev[1] = fine bundle — the two terms of model_nerf.py:118-126
      float* slot = loss_dev ? loss_dev + ((two && i == 0) ? 1 : 0) : nullptr;
      if (int e = launch_mse_grad(h->tr_rgb[i].as<float>(), target, 3 * R, 3 * R_total, h->tr_drgb[i].as<float>(), slot, st, &h->launches)) return e;
    }
    d_rgb = h->tr_drgb[0].as<float>();
    d_rgb_coarse = two ? h->tr_drgb[1].as<float>() : nullptr;
  }
  struct Pass { int which; const float* raw; const float* t; int s; const float* g; uint64_t salt; };
  Pass passes[2];
  int np = 0;
  if (two) {
    if (d_rgb) passes[np++] = {NM_NET_FINE, h->raw_f.as<float>(), h->t_f.as<float>(), S, d_rgb, kNoiseSaltMain};
    if (d_rgb_coarse) passes[np++] = {NM_NET_COARSE, h->raw_c.as<float>(), h->t_c.as<float>(), Nc, d_rgb_coarse, kNoiseSaltCoarse};
  } else if (d_rgb) {
    passes[np++] = {NM_NET_COARSE, h->raw_c.as<float>(), buff ? h->t_u.as<float>() : h->t_c.as<float>(), Nc, d_rgb, kNoiseSaltMain};
  }
  for (int pi = 0; pi < np; ++pi) {
    const Pass& P = passes[pi];
    NetDev& net = h->nets[P.which];
    if (int e = h->dout.ensure((size_t)R * P.s * 16)) return e;
    if (int e = h->trans.ensure((size_t)R * P.s * 4)) return e;
    if (int e = launch_composite_backward(P.raw, P.t, rb.dirs, P.g, R, P.s, c.noise_std, seed ^ P.salt,
                                          c.white_background, h->trans.as<float>(), h->dout.as<float>(), st, &h->launches)) return e;
    NetGrads gd{h->g_wt[P.which].as<float>(), h->g_bias[P.which].as<float>(), h->g_head[P.which].as<float>()};
    TrainMode md{use_tc ? 1 : 0, c.precision == NM_PREC_FAST ? 1 : 3, h->d_err};
    if (direct) {
      MlpInput in{};
      in.mode = IN_RAYS; in.dirs = rb.dirs; in.ray_o = rb.origins; in.o_stride = rb.o_stride; in.t = P.t; in.S = P.s; in.M = R * P.s;
      float* wsp = (two && P.which == NM_NET_COARSE) ? ws_c : ws_m;
      if (int e = mlp_backward(h->nets[P.which], in, h->dout.as<float>(), wsp, &gd, h->num_sms, md, st, &h->launches, 1)) return e;
      continue;
    }
    // sub-chunks of `waves` full waves of 128-point row blocks (148 SMs): bounds the activation workspace (~20 KB per point)
    static const int waves = [] { const char* e = getenv("NM_TRAIN_WAVES"); int v = e ? atoi(e) : 0; return v > 0 ? v : 16; }();
    long long rays_sub = ((long long)h->num_sms * 128 * waves) / P.s;
    if (rays_sub < 1) rays_sub = 1;
    if (rays_sub > R) rays_sub = R;
    if (int e = h->train_ws.ensure(train_ws_bytes(net.full, rays_sub * P.s, use_tc) + 1024)) return e;
    float* ws = reinterpret_cast<float*>(((uintptr_t)h->train_ws.p + 1023) & ~(uintptr_t)1023);
    NetGrads g{h->g_wt[P.which].as<float>(), h->g_bias[P.which].as<float>(), h->g_head[P.which].as<float>()};
    TrainMode mode{use_tc ? 1 : 0, c.precision == NM_PREC_FAST ? 1 : 3, h->d_err};
    for (long long r0 = 0; r0 < R; r0 += rays_sub) {
      const long long n = (R - r0 < rays_sub) ? R - r0 : rays_sub;
      MlpInput in{};
      in.mode = IN_RAYS; in.dirs = rb.dirs + 3 * r0; in.ray_o = rb.origins + (long long)rb.o_stride * r0;
      in.o_stride = rb.o_stride; in.t = P.t + r0 * P.s; in.S = P.s; in.M = n * P.s;
      if (int e = mlp_backward(h->nets[P.which], in, h->dout.as<float>() + r0 * P.s * 4, ws, &g, h->num_sms, mode, st, &h->launches)) return e;
    }
  }
  return 0;
}

int train_impl(NmHandle h, const float* origins, int o_stride, const float* dirs, long long R, const float* nf_host,
               const float* near_dev, const float* far_dev, int flags, uint64_t seed, const float* d_rgb,
               const float* d_rgb_coarse, const float* target, float* loss_dev, cudaStream_t st) {
  NM_CHECK(o_stride == 0 || o_stride == 3, "o_stride must be 0 or 3");
  NM_CHECK(dirs && origins, "null ray pointers");
  NM_CHECK((near_dev == nullptr) == (far_dev == nullptr), "near_dev / far_dev must be given together");
  NM_CHECK(near_dev || nf_host, "no near/far bounds given");
  NM_CHECK(!(flags & NM_FLAG_TEACHER_T), "NM_FLAG_TEACHER_T is not supported by the backward pass");
  NM_CHECK(target || d_rgb || d_rgb_coarse, "no gradient source (target or d_rgb)");
  NM_CHECK(h->s_table.p != nullptr, "sampler tables missing");
  if (!h->grads_ready) if (int e = ensure_grads(h, st, true)) return e;
  if (int e = ensure_grads(h, st, false)) return e;
  const long long kChunk = chunk_rays();
  for (long long r0 = 0; r0 < R; r0 += kChunk) {
    RayBatch rb{};
    rb.R = (R - r0 < kChunk) ? R - r0 : kChunk;
    rb.origins = origins + (long long)o_stride * r0; rb.o_stride = o_stride; rb.dirs = dirs + 3 * r0;
    if (nf_host) { rb.nf[0] = nf_host[0]; rb.nf[1] = nf_host[1]; }
    rb.near_dev = near_dev ? near_dev + r0 : nullptr; rb.far_dev = far_dev ? far_dev + r0 : nullptr;
    if (int e = train_chunk(h, rb, flags, seed + (uint64_t)r0, d_rgb ? d_rgb + 3 * r0 : nullptr,
                            d_rgb_coarse ? d_rgb_coarse + 3 * r0 : nullptr, target ? target + 3 * r0 : nullptr, R,
                            loss_dev, st)) return e;
  }
  return 0;
}

}  // namespace

extern "C" {

int nm_version(void) { return NM_VERSION; }
const char* nm_last_error(void) { return nm::last_error(); }

int nm_device_check(int device) {
  int n = 0;
  NM_CUDA(cudaGetDeviceCount(&n));
  NM_CHECK(device >= 0 && device < n, "device %d out of range (%d visible)", device, n);
  cudaDeviceProp p;
  NM_CUDA(cudaGetDeviceProperties(&p, device));
  NM_CHECK(p.major == 10, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, p.major, p.minor);
  return 0;
}

int nm_create(int device, const NmNetDesc* coarse, const NmNetDesc* fine, const NmRenderCfg* cfg, NmHandle* out) {
  NM_CHECK(coarse && cfg && out, "null argument");
  if (int e = nm_device_check(device)) return e;
  NetProgram a, b;
  if (int e = build_programs(*coarse, &a, &b)) return e;
  if (fine) if (int e = build_programs(*fine, &a, &b)) return e;
  NM_CUDA(cudaSetDevice(device));
  NmHandle h = new NmHandle_t();
  h->device = device;
  h->desc[0] = *coarse;
  h->has_fine = fine != nullptr;
  if (fine) h->desc[1] = *fine;
  auto init = [&]() -> int {
    cudaDeviceProp p;
    NM_CUDA(cudaGetDeviceProperties(&p, device));
    h->num_sms = p.multiProcessorCount;
    NM_CUDA(cudaHostAlloc(&h->h_err, 2 * sizeof(int), cudaHostAllocMapped));
    h->h_err[0] = h->h_err[1] = 0;
    NM_CUDA(cudaHostGetDevicePointer(&h->d_err, h->h_err, 0));
    NM_CUDA(cudaMalloc(&h->d_stats, 4 * sizeof(double)));
    NM_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    if (int e = nm_set_render_cfg(h, cfg)) return e;
    return nm_set_tables(h, nullptr, nullptr);
  };
  if (int e = init()) { nm_destroy(h); *out = nullptr; return e; }
  *out = h;
  return 0;
}

int nm_destroy(NmHandle h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  free_network(&h->nets[0]); free_network(&h->nets[1]);
  Buf* bufs[] = {&h->s_table, &h->u_table, &h->voxels, &h->t_c, &h->raw_c, &h->w_c, &h->t_f, &h->raw_f, &h->t_u,
                 &h->dirs, &h->origins, &h->lin[0], &h->lin[1], &h->lin[2], &h->small};
  for (Buf* b : bufs) b->release();
  for (Buf& b : h->stage_in) b.release();
  for (Buf& b : h->stage_out) b.release();
  for (int i = 0; i < 2; ++i) { h->g_wt[i].release(); h->g_bias[i].release(); h->g_head[i].release(); h->tr_rgb[i].release(); h->tr_drgb[i].release(); }
  h->train_ws.release(); h->dout.release(); h->trans.release(); h->metric_ws.release();
  if (h->mc_ws_ptr) cudaFree(h->mc_ws_ptr);
  if (h->mc_ws2_ptr) cudaFree(h->mc_ws2_ptr);
  if (h->h_err) cudaFreeHost(h->h_err);
  cudaFree(h->d_stats);
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return 0;
}

int nm_set_render_cfg(NmHandle h, const NmRenderCfg* cfg) {
  NM_CHECK(h && cfg, "null argument");
  NM_CHECK(cfg->num_coarse >= 3 && cfg->num_coarse <= 256, "num_coarse %d outside [3,256]", cfg->num_coarse);
  NM_CHECK(cfg->num_fine >= 0 && cfg->num_coarse + cfg->num_fine <= 512, "num_coarse+num_fine exceeds 512");
  NM_CHECK(cfg->precision >= NM_PREC_EXACT && cfg->precision <= NM_PREC_FP32, "unknown precision %d", cfg->precision);
  NM_CHECK(cfg->act_scale_log2 >= 0 && cfg->act_scale_log2 <= 12, "act_scale_log2 outside [0,12]");
  const bool resize = cfg->num_coarse != h->cfg.num_coarse || cfg->num_fine != h->cfg.num_fine;
  h->cfg = *cfg;
  if (resize && h->s_table.p) return nm_set_tables(h, nullptr, nullptr);
  return 0;
}

int nm_load_weights(NmHandle h, int which, int n_tensors, const char* const* names, const float* const* tensors_host,
                    const int64_t* numel) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(which == NM_NET_COARSE || (which == NM_NET_FINE && h->has_fine), "network slot %d not present", which);
  WeightSource src;
  src.n = n_tensors; src.names = names; src.ptrs = tensors_host; src.numel = numel;
  return pack_network(h->desc[which], src, &h->nets[which]);
}

int nm_load_weights_dev(NmHandle h, int which, int n_tensors, const char* const* names, const float* const* tensors_dev,
                        const int64_t* numel, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(which == NM_NET_COARSE || (which == NM_NET_FINE && h->has_fine), "network slot %d not present", which);
  WeightSource src;
  src.n = n_tensors; src.names = names; src.ptrs = tensors_dev; src.numel = numel;
  return load_network_dev(h->desc[which], src, &h->nets[which], (cudaStream_t)stream, &h->launches);
}

int nm_set_tables(NmHandle h, const float* coarse_s_host, const float* fine_u_host) {
  if (int e = bind_device(h)) return e;
  std::vector<float> tmp;
  if (!coarse_s_host) { linspace_host(h->cfg.num_coarse, &tmp); coarse_s_host = tmp.data(); }
  if (int e = upload(&h->s_table, coarse_s_host, sizeof(float) * h->cfg.num_coarse)) return e;
  if (h->cfg.num_fine > 0) {
    std::vector<float> tmp2;
    if (!fine_u_host) { linspace_host(h->cfg.num_fine, &tmp2); fine_u_host = tmp2.data(); }
    if (int e = upload(&h->u_table, fine_u_host, sizeof(float) * h->cfg.num_fine)) return e;
  }
  return 0;
}

int nm_set_tree(NmHandle h, const float* voxels_host, int32_t V) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(voxels_host && V > 0, "empty voxel list");
  h->V = V;
  return upload(&h->voxels, voxels_host, sizeof(float) * 6 * (size_t)V);
}

int nm_point_mlp(NmHandle h, int which, const float* pts_dev, const float* dirs_dev, int64_t M, float* out_dev,
                 int sigma_only, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(which == NM_NET_COARSE || (which == NM_NET_FINE && h->has_fine), "network slot %d not present", which);
  NM_CHECK(pts_dev && out_dev && M >= 0, "bad arguments");
  MlpInput in{};
  in.mode = IN_POINTS; in.pts = pts_dev; in.dirs = dirs_dev; in.M = M;
  return run_mlp(h, which, sigma_only != 0, in, out_dev, (cudaStream_t)stream);
}

int nm_render_rays(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                   const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                   const NmRenderOut* out_dev, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(out_dev, "null output block");
  return render_rays_impl(h, origins_dev, o_stride, dirs_dev, R, near_far_host, near_dev, far_dev, flags, seed, *out_dev,
                          (cudaStream_t)stream);
}

int nm_ray_bundle(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, float ndc_near, int row0,
                  int row1, float* origins_dev, float* dirs_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(pose_host && dirs_dev, "null argument");
  NM_CHECK(0 <= row0 && row0 <= row1 && row1 <= H && W > 0, "bad row range");
  NM_CHECK(!ndc || origins_dev, "ndc rays need an origins buffer");
  RayGenArgs a{};
  memcpy(a.pose, pose_host, sizeof(a.pose));
  a.H = H; a.W = W; a.focal = focal; a.ndc = ndc; a.ndc_near = ndc_near; a.row0 = row0; a.row1 = row1;
  return launch_raygen(a, origins_dev, dirs_dev, (cudaStream_t)stream, &h->launches);
}

int nm_render_image(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, int row0, int row1,
                    const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_dev, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(out_dev && pose_host && near_far_host, "null argument");
  const long long R = (long long)(row1 - row0) * W;
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = h->dirs.ensure((size_t)R * 12)) return e;
  float* origins = nullptr;
  int o_stride = 0;
  if (ndc) {
    if (int e = h->origins.ensure((size_t)R * 12)) return e;
    origins = h->origins.as<float>();
    o_stride = 3;
  }
  if (int e = nm_ray_bundle(h, pose_host, H, W, focal, ndc, 1.0f, row0, row1, origins, h->dirs.as<float>(), stream)) return e;
  if (!ndc) {
    if (int e = h->small.ensure(64)) return e;
    const float o3[3] = {pose_host[3], pose_host[7], pose_host[11]};
    NM_CUDA(cudaMemcpyAsync(h->small.p, o3, sizeof(o3), cudaMemcpyHostToDevice, st));
    origins = h->small.as<float>();
  }
  return render_rays_impl(h, origins, o_stride, h->dirs.as<float>(), R, near_far_host, nullptr, nullptr, flags, seed,
                          *out_dev, st);
}

// ---------------------------------------------------------------------------------------------- training entry points
int nm_zero_grad(NmHandle h, void* stream) {
  if (int e = bind_device(h)) return e;
  return ensure_grads(h, (cudaStream_t)stream, true);
}

int nm_backward_rays(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                     const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                     const float* d_rgb_dev, const float* d_coarse_rgb_dev, void* stream) {
  if (int e = bind_checked(h)) return e;
  return train_impl(h, origins_dev, o_stride, dirs_dev, R, near_far_host, near_dev, far_dev, flags, seed, d_rgb_dev,
                    d_coarse_rgb_dev, nullptr, nullptr, (cudaStream_t)stream);
}

int nm_loss_backward(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                     const float* near_far_host, const float* near_dev, const float* far_dev, int flags, uint64_t seed,
                     const float* target_rgb_dev, float* loss_dev, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(target_rgb_dev, "null target");
  return train_impl(h, origins_dev, o_stride, dirs_dev, R, near_far_host, near_dev, far_dev, flags, seed, nullptr, nullptr,
                    target_rgb_dev, loss_dev, (cudaStream_t)stream);
}

int nm_get_grad(NmHandle h, int which, const char* name, float* out_dev, int64_t numel, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(which == NM_NET_COARSE || (which == NM_NET_FINE && h->has_fine), "network slot %d not present", which);
  NM_CHECK(name && out_dev, "null argument");
  const NetDev& net = h->nets[which];
  NM_CHECK(net.loaded && h->grads_ready && h->g_wt[which].p, "no gradients accumulated for network %d", which);
  cudaStream_t st = (cudaStream_t)stream;
  for (int l = 0; l < net.full.n_layers; ++l) {
    const LayerProg& L = net.full.layers[l];
    const int K = L.k_act + L.k_pe, N = L.n_out;
    const int heads = L.kind == KIND_SIGMA ? 1 : (L.kind == KIND_RGB ? 3 : (L.kind == KIND_OUT4 ? 4 : 0));
    const std::string* nm4 = &net.names[4 * l];
    if (nm4[0] == name) {
      NM_CHECK(numel == (int64_t)K * N, "'%s' has %lld elements, expected %lld", name, (long long)numel, (long long)K * N);
      size_t go[kMaxLayers]; int gl[kMaxLayers];
      grad_layout(net.full, go, gl);
      NM_CUDA(cudaMemcpy2DAsync(out_dev, (size_t)K * 4, h->g_wt[which].as<float>() + go[l], (size_t)gl[l] * 4, (size_t)K * 4, N,
                                cudaMemcpyDeviceToDevice, st));
      return 0;
    }
    const float* src = nullptr;
    int64_t n = 0;
    if (nm4[1] == name) { src = h->g_bias[which].as<float>() + L.bias_off; n = N; }
    else if (heads && nm4[2] == name) { src = h->g_head[which].as<float>() + L.head_off; n = (int64_t)heads * N; }
    else if (heads && nm4[3] == name) { src = h->g_head[which].as<float>() + L.head_off + heads * N; n = heads; }
    if (src) {
      NM_CHECK(numel == n, "'%s' has %lld elements, expected %lld", name, (long long)numel, (long long)n);
      NM_CUDA(cudaMemcpyAsync(out_dev, src, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
      return 0;
    }
  }
  NM_CHECK(false, "no parameter named '%s'", name);
  return -1;
}

int nm_debug_gemm(NmHandle h, const float* a_dev, const float* b_dev, int M, int N, int K, int a_cols, int b_cols,
                  int k_split, int n_passes, int fp16, int atomic, float* d_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(a_dev && b_dev && d_dev && M > 0 && N > 0 && K > 0, "bad arguments");
  const size_t need = 3 * ((size_t)((M > N ? M : N) + 127) / 128 * ((K + 63) / 64) * 32768 + 1024) + 1024;
  if (int e = h->train_ws.ensure(need)) return e;
  uint8_t* ws = reinterpret_cast<uint8_t*>(((uintptr_t)h->train_ws.p + 1023) & ~(uintptr_t)1023);
  return debug_tc_gemm(a_dev, b_dev, M, N, K, a_cols, b_cols, k_split, n_passes, fp16, atomic, d_dev, ws, need - 1024, h->num_sms,
                       h->d_err, (cudaStream_t)stream, &h->launches);
}

// ---------------------------------------------------------------------------------------------- BuFF tree maintenance
int nm_ray_voxel_indices(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                         const float* near_far_host, float* z_out_dev, int32_t* idx_out_dev, void* stream) {
  return nm_ray_voxel_indices_ex(h, origins_dev, o_stride, dirs_dev, R, near_far_host, 0, 0, z_out_dev, idx_out_dev, stream);
}

int nm_ray_voxel_indices_ex(NmHandle h, const float* origins_dev, int o_stride, const float* dirs_dev, int64_t R,
                            const float* near_far_host, int flags, uint64_t seed, float* z_out_dev, int32_t* idx_out_dev,
                            void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(origins_dev && dirs_dev && near_far_host && idx_out_dev, "null argument");
  NM_CHECK(o_stride == 0 || o_stride == 3, "o_stride must be 0 or 3");
  NM_CHECK(h->V > 0, "no voxel list (nm_set_tree)");
  cudaStream_t st = (cudaStream_t)stream;
  const int S = h->cfg.num_coarse;
  float* t_u = nullptr;
  if (z_out_dev) {     // rays without a hit fall back to the uniform samples (src/models/model_buff.py:53)
    if (int e = h->t_c.ensure((size_t)R * S * 4)) return e;
    t_u = h->t_c.as<float>();
    if (int e = launch_stratified(h->s_table.as<float>(), S, R, near_far_host, nullptr, nullptr, h->cfg.lindisp, 0, 0, t_u, st,
                                  &h->launches)) return e;
  }
  // walked in the render calls' ray chunks with their per-chunk seeds, so that a random draw repeats the render's own
  const long long kChunk = chunk_rays();
  for (long long r0 = 0; r0 < R; r0 += kChunk) {
    const long long n = (R - r0 < kChunk) ? R - r0 : kChunk;
    if (int e = launch_aabb(h->voxels.as<float>(), h->V, origins_dev + (long long)o_stride * r0, o_stride, dirs_dev + 3 * r0, n,
                            near_far_host[0], near_far_host[1], S, h->s_table.as<float>(), t_u ? t_u + r0 * S : nullptr,
                            z_out_dev ? z_out_dev + r0 * S : nullptr, idx_out_dev + r0 * S, h->d_err + 1, st, &h->launches,
                            (flags & NM_FLAG_RANDOM_VOXELS) ? 1 : 0, seed + (uint64_t)r0)) return e;
  }
  return 0;
}

int nm_tree_integrate(NmHandle h, const int32_t* idx_dev, const float* weights_dev, const float* mask_weights_dev, int64_t n,
                      float* memm_dev, int32_t V, int32_t counter, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(idx_dev && weights_dev && mask_weights_dev && memm_dev && V > 0 && n >= 0, "bad arguments");
  if (int e = h->small.ensure(sizeof(float) * 2 * (size_t)V + 64)) return e;
  return launch_tree_integrate(idx_dev, weights_dev, mask_weights_dev, n, memm_dev, V, counter, h->small.as<float>(),
                               (cudaStream_t)stream, &h->launches);
}

int nm_grid_sigma(NmHandle h, const float* lin0_host, const float* lin1_host, const float* lin2_host, int n0, int n1,
                  int n2, int x0, int x1, float* sigma_dev, float* rgb_dev, void* stream) {
  if (int e = bind_checked(h)) return e;
  NM_CHECK(lin0_host && lin1_host && lin2_host && sigma_dev, "null argument");
  NM_CHECK(0 <= x0 && x0 <= x1 && x1 <= n0 && n1 > 0 && n2 > 0, "bad slab range");
  const int which = h->has_fine ? NM_NET_FINE : NM_NET_COARSE;     // BaseModel.get_model(): finest net
  const float* hs[3] = {lin0_host, lin1_host, lin2_host};
  const int ns[3] = {n0, n1, n2};
  for (int i = 0; i < 3; ++i) { if (int e = upload(&h->lin[i], hs[i], sizeof(float) * ns[i])) return e; h->lin_n[i] = ns[i]; }
  cudaStream_t st = (cudaStream_t)stream;
  MlpInput in{};
  in.mode = IN_GRID;
  in.lin0 = h->lin[0].as<float>(); in.lin1 = h->lin[1].as<float>(); in.lin2 = h->lin[2].as<float>();
  in.n1 = n1; in.n2 = n2;
  in.grid_base = (long long)x0 * n1 * n2;
  in.M = (long long)(x1 - x0) * n1 * n2;
  if (!rgb_dev) return run_mlp(h, which, true, in, sigma_dev, st);
  // reference-faithful rgb+sigma: run the full net into a scratch (M,4) and split
  if (int e = h->raw_f.ensure((size_t)in.M * 16)) return e;
  if (int e = run_mlp(h, which, false, in, h->raw_f.as<float>(), st)) return e;
  NM_CUDA(cudaMemcpy2DAsync(sigma_dev, 4, h->raw_f.as<float>() + 3, 16, 4, (size_t)in.M, cudaMemcpyDeviceToDevice, st));
  NM_CUDA(cudaMemcpy2DAsync(rgb_dev, 12, h->raw_f.as<float>(), 16, 12, (size_t)in.M, cudaMemcpyDeviceToDevice, st));
  return 0;
}

int nm_volume_stats(NmHandle h, const float* vol_dev, int64_t n, float* out_host) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(vol_dev && out_host, "null argument");
  return launch_volume_stats(vol_dev, n, h->d_stats, out_host, h->own_stream, &h->launches);
}

int nm_volume_stats_dev(NmHandle h, const float* vol_dev, int64_t n, int pass, const double* mean_dev, double* out_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(vol_dev && out_dev, "null argument");
  return launch_volume_stats_pass(vol_dev, n, pass, mean_dev, out_dev, (cudaStream_t)stream, &h->launches);
}

int nm_mc_count(NmHandle h, const float* vol_dev, int nb, int ny, int nz, float iso, int g_x0, int g_nx, int p_lo, int p_hi,
                int64_t* counts_host, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(vol_dev && counts_host, "null argument");
  const McShard s{vol_dev, nb, ny, nz, iso, g_x0, g_nx, p_lo, p_hi, 0};
  if (int e = mc_count(s, &h->mc_ws_ptr, &h->mc_ws_bytes, counts_host, (cudaStream_t)stream, &h->launches)) return e;
  h->mc_counts[0] = counts_host[0]; h->mc_counts[1] = counts_host[1];
  return 0;
}

int nm_mc_emit(NmHandle h, const float* vol_dev, int nb, int ny, int nz, float iso, int g_x0, int g_nx, int p_lo, int p_hi,
               int64_t v_base, float* verts_dev, float* normals_dev, int32_t* faces_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(vol_dev && verts_dev && faces_dev && h->mc_ws_ptr, "bad arguments (call nm_mc_count first)");
  const McShard s{vol_dev, nb, ny, nz, iso, g_x0, g_nx, p_lo, p_hi, 0};
  return mc_emit(s, h->mc_ws_ptr, h->mc_ws_bytes, &h->mc_ws2_ptr, &h->mc_ws2_bytes, v_base, h->mc_counts[0], h->mc_counts[1],
                 verts_dev, normals_dev, faces_dev, (cudaStream_t)stream, &h->launches);
}

int nm_marching_cubes_count(NmHandle h, const float* vol_dev, int nx, int ny, int nz, float iso, int64_t* counts_host,
                            void* stream) {
  return nm_mc_count(h, vol_dev, nx, ny, nz, iso, 0, nx, 0, nx, counts_host, stream);
}

int nm_marching_cubes_emit(NmHandle h, const float* vol_dev, int nx, int ny, int nz, float iso, float x_off,
                           float* verts_dev, float* normals_dev, int32_t* faces_dev, void* stream) {
  NM_CHECK(x_off >= 0.f && x_off == (float)(int)x_off, "x_off must be a non-negative integer number of planes");
  // a stand-alone volume whose axis-0 vertex coordinates start at x_off (a pure coordinate shift)
  if (int e = bind_device(h)) return e;
  NM_CHECK(vol_dev && verts_dev && faces_dev && h->mc_ws_ptr, "bad arguments (call nm_marching_cubes_count first)");
  const McShard s{vol_dev, nx, ny, nz, iso, 0, nx, 0, nx, (int)x_off};
  return mc_emit(s, h->mc_ws_ptr, h->mc_ws_bytes, &h->mc_ws2_ptr, &h->mc_ws2_bytes, 0, h->mc_counts[0], h->mc_counts[1], verts_dev,
                 normals_dev, faces_dev, (cudaStream_t)stream, &h->launches);
}

int nm_nearest(NmHandle h, const float* x_dev, int64_t N, const float* y_dev, int64_t M, float* dist_dev, int32_t* idx_dev,
               void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(N >= 0 && M >= 1 && M < (1ll << 31), "nearest: need N >= 0 and 1 <= M < 2^31 (got N=%lld, M=%lld)", (long long)N,
           (long long)M);
  NM_CHECK(N == 0 || (x_dev && y_dev && dist_dev && idx_dev), "null argument");
  if (int e = h->metric_ws.ensure(nearest_ws_bytes(N, M, h->num_sms))) return e;
  return launch_nearest(x_dev, N, y_dev, M, dist_dev, idx_dev, h->metric_ws.p, h->num_sms, (cudaStream_t)stream, &h->launches);
}

int nm_mesh_sample(NmHandle h, const float* verts_dev, int64_t V, const int32_t* faces_dev, int64_t F, int64_t n, uint64_t seed,
                   float* points_dev, int32_t* face_idx_dev, float* normals_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(V >= 0 && F >= 0 && n >= 0 && F < (1ll << 31), "mesh sample: bad sizes (V=%lld, F=%lld, n=%lld)", (long long)V,
           (long long)F, (long long)n);
  NM_CHECK(F == 0 || V > 0, "mesh sample: faces without vertices");
  NM_CHECK(n == 0 || points_dev, "null output");
  NM_CHECK(F == 0 || (verts_dev && faces_dev), "null mesh");
  if (int e = h->metric_ws.ensure(mesh_sample_ws_bytes(F))) return e;
  return launch_mesh_sample(verts_dev, faces_dev, F, n, seed, points_dev, face_idx_dev, normals_dev, h->metric_ws.p,
                            (cudaStream_t)stream, &h->launches);
}

int nm_query_host(NmHandle h, const float* origins_host, int o_stride, const float* dirs_host, int64_t R,
                  const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_host) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(origins_host && dirs_host && near_far_host && out_host && R > 0, "bad arguments");
  NM_CHECK(!(flags & NM_FLAG_TEACHER_T), "NM_FLAG_TEACHER_T is a device-pointer feature");
  cudaStream_t st = h->own_stream;
  const size_t ob = o_stride ? (size_t)R * 12 : 12;
  if (int e = h->stage_in[0].ensure(ob)) return e;
  if (int e = h->stage_in[1].ensure((size_t)R * 12)) return e;
  NM_CUDA(cudaMemcpyAsync(h->stage_in[0].p, origins_host, ob, cudaMemcpyHostToDevice, st));
  NM_CUDA(cudaMemcpyAsync(h->stage_in[1].p, dirs_host, (size_t)R * 12, cudaMemcpyHostToDevice, st));
  NmRenderOut dev{};
  size_t sizes[12];
  if (int e = stage_outputs(h, *out_host, R, out_samples(h, flags), h->cfg.num_coarse, &dev, sizes)) return e;
  if (int e = render_rays_impl(h, h->stage_in[0].as<float>(), o_stride, h->stage_in[1].as<float>(), R, near_far_host,
                               nullptr, nullptr, flags, seed, dev, st)) return e;
  if (int e = copy_outputs(*out_host, dev, sizes, st)) return e;
  NM_CUDA(cudaStreamSynchronize(st));
  return check_kernel_flags(h);
}

int nm_render_image_host(NmHandle h, const float* pose_host, int H, int W, float focal, int ndc, int row0, int row1,
                         const float* near_far_host, int flags, uint64_t seed, const NmRenderOut* out_host) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(out_host, "null output block");
  const long long R = (long long)(row1 - row0) * W;
  cudaStream_t st = h->own_stream;
  NmRenderOut dev{};
  size_t sizes[12];
  if (int e = stage_outputs(h, *out_host, R, out_samples(h, flags), h->cfg.num_coarse, &dev, sizes)) return e;
  if (int e = nm_render_image(h, pose_host, H, W, focal, ndc, row0, row1, near_far_host, flags, seed, &dev, st)) return e;
  if (int e = copy_outputs(*out_host, dev, sizes, st)) return e;
  NM_CUDA(cudaStreamSynchronize(st));
  return check_kernel_flags(h);
}

int nm_point_mlp_host(NmHandle h, int which, const float* pts_host, const float* dirs_host, int64_t M, float* out_host,
                      int sigma_only) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(pts_host && out_host && M > 0, "bad arguments");
  cudaStream_t st = h->own_stream;
  const size_t outb = (size_t)M * (sigma_only ? 4 : 16);
  if (int e = h->stage_in[0].ensure((size_t)M * 12)) return e;
  if (int e = h->stage_in[1].ensure((size_t)M * 12)) return e;
  if (int e = h->stage_out[0].ensure(outb)) return e;
  NM_CUDA(cudaMemcpyAsync(h->stage_in[0].p, pts_host, (size_t)M * 12, cudaMemcpyHostToDevice, st));
  if (dirs_host) NM_CUDA(cudaMemcpyAsync(h->stage_in[1].p, dirs_host, (size_t)M * 12, cudaMemcpyHostToDevice, st));
  if (int e = nm_point_mlp(h, which, h->stage_in[0].as<float>(), dirs_host ? h->stage_in[1].as<float>() : nullptr, M,
                           h->stage_out[0].as<float>(), sigma_only, st)) return e;
  NM_CUDA(cudaMemcpyAsync(out_host, h->stage_out[0].p, outb, cudaMemcpyDeviceToHost, st));
  NM_CUDA(cudaStreamSynchronize(st));
  return check_kernel_flags(h);
}

int nm_debug_pack(const NmNetDesc* desc, int n_tensors, const char* const* names, const float* const* tensors_host,
                  const int64_t* numel, int sigma_only, void* program_out, size_t program_cap, uint8_t* pack_out,
                  size_t pack_cap, size_t* pack_need) {
  NM_CHECK(desc && program_out && pack_need, "null argument");
  NM_CHECK(program_cap >= sizeof(NetProgram), "program buffer too small (%zu needed)", sizeof(NetProgram));
  WeightSource src;
  src.n = n_tensors; src.names = names; src.ptrs = tensors_host; src.numel = numel;
  return debug_pack(*desc, src, sigma_only != 0, reinterpret_cast<NetProgram*>(program_out), pack_out, pack_cap, pack_need);
}

int nm_check_flags(NmHandle h, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return check_kernel_flags(h);
}

int nm_ndc_rays(NmHandle h, int H, int W, float focal, float near, const float* origins_dev, int o_stride,
                const float* dirs_dev, int64_t n, float* origins_out_dev, float* dirs_out_dev, void* stream) {
  if (int e = bind_device(h)) return e;
  NM_CHECK(origins_dev && dirs_dev && origins_out_dev && dirs_out_dev && n >= 0, "bad arguments");
  NM_CHECK(o_stride == 0 || o_stride == 3, "o_stride must be 0 or 3");
  return launch_ndc(H, W, focal, near, origins_dev, o_stride, dirs_dev, n, origins_out_dev, dirs_out_dev, (cudaStream_t)stream,
                    &h->launches);
}

int nm_kernel_flags(NmHandle h, int32_t* out2) {
  NM_CHECK(h && out2, "null argument");
  out2[0] = h->h_err[0];
  out2[1] = h->h_err[1];
  return 0;
}

int64_t nm_launch_count(NmHandle h) { return h ? h->launches : -1; }

int nm_debug_tile_schedule(int samples_per_ray, int64_t n_tiles, int grid, int cta, int64_t* tiles_out, int64_t cap, int64_t* n_out) {
  const int g = mlp_tc_composite_group(samples_per_ray);
  if (tiles_out && n_out) {
    const int64_t gt = g > 0 ? g : 1;       // the kernel's tile_of(): groups of gt consecutive tiles dealt round-robin
    int64_t n = 0;
    for (int64_t i = 0;; ++i) {
      const int64_t grp = cta + (i / gt) * grid, t = grp * gt + (i % gt);
      if (t >= n_tiles) break;
      if (n < cap) tiles_out[n] = t;
      ++n;
    }
    *n_out = n;
  }
  return g;
}

int nm_set_timing(NmHandle h, int enable) {
  NM_CHECK(h, "null handle");
  h->timing = enable != 0;
  h->ev_used = 0; h->mlp_points = 0; h->mlp_launches = 0;
  return 0;
}

double nm_mlp_time_ms(NmHandle h, int64_t* points_out, int64_t* launches_out) {
  if (!h || !h->timing) return -1.0;
  cudaSetDevice(h->device);
  double total = 0.0;
  for (size_t i = 0; i + 1 < h->ev_used; i += 2) {
    if (cudaEventSynchronize(h->ev[i + 1]) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]) != cudaSuccess) return -1.0;
    total += ms;
  }
  if (points_out) *points_out = h->mlp_points;
  if (launches_out) *launches_out = h->mlp_launches;
  h->ev_used = 0; h->mlp_points = 0; h->mlp_launches = 0;
  return total;
}

}  // extern "C"
