// Internal declarations shared by the translation units of libnerfmeshes_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/nerfmeshes_b200.h"
#include "nm_program.h"

namespace nm {

void set_error(const char* fmt, ...);
#define NM_CUDA(expr)                                                                             \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      nm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -2;                                                                                  \
    }                                                                                             \
  } while (0)
#define NM_CHECK(cond, ...)       \
  do {                            \
    if (!(cond)) {                \
      nm::set_error(__VA_ARGS__); \
      return -1;                  \
    }                             \
  } while (0)

// One network's device-resident data.
struct NetDev {
  bool loaded = false;
  NmNetDesc desc{};
  NetProgram full{};        // rgb + sigma
  NetProgram sigma{};       // trunk + sigma head only (grid fast path)
  // device arrays
  NetProgram* d_full = nullptr;
  NetProgram* d_sigma = nullptr;
  uint8_t* d_wpack_full = nullptr;   // tensor-core weight stages, issue order of `full`
  uint8_t* d_wpack_sigma = nullptr;
  float* d_bias = nullptr;
  float* d_head = nullptr;
  float* d_wt = nullptr;             // transposed fp32 weights (CUDA-core kernel)
  float* d_w = nullptr;              // the same weights in the reference's (out,in) layout, same per-layer offsets
  size_t n_wt = 0;                   // floats in d_wt
  // training backward on the tensor cores (nm_gemm_tc.cu): bf16 hi/lo operand packs of W (forward) and W^T (data
  // gradient) per layer, rebuilt lazily after every weight load
  uint8_t* d_tcw = nullptr;
  size_t tcw_bytes = 0;
  size_t tcw_fwd_off[kMaxLayers] = {}, tcw_bwd_off[kMaxLayers] = {};
  bool tcw_valid = false;
  // fused data-gradient chain (nm_mlp_tc.cu, mode 2): backward program + W^T stages (bf16 hi/lo), rebuilt lazily
  NetProgram bwd{};
  NetProgram* d_bwd = nullptr;
  uint8_t* d_wpack_bwd = nullptr;
  bool bwd_valid = false;
  std::vector<std::string> names;    // per layer of `full`: weight, bias, head weight, head bias ("" if none)
};

// Weight-gradient buffer layout: per layer (n_out, ld) row-major in the reference's (out,in) orientation, ld = in
// features rounded up to 4 floats so that rows stay 16-byte aligned (vector atomics).  Returns the total float count.
inline size_t grad_layout(const NetProgram& G, size_t off[kMaxLayers], int ld[kMaxLayers]) {
  size_t total = 0;
  for (int l = 0; l < G.n_layers; ++l) {
    const int K = G.layers[l].k_act + G.layers[l].k_pe;
    ld[l] = (K + 3) & ~3;
    off[l] = total;
    total += (size_t)G.layers[l].n_out * ld[l];
  }
  return total;
}

// Gradient accumulators of one network: weights per grad_layout(), biases / heads like NetDev.d_bias / d_head.
struct NetGrads {
  float* w = nullptr;
  float* bias = nullptr;
  float* head = nullptr;
};

// Inputs of one fused-MLP launch (three front-end modes).
enum : int { IN_POINTS = 0, IN_RAYS = 1, IN_GRID = 2 };
struct MlpInput {
  int mode = IN_POINTS;
  const float* pts = nullptr;    // IN_POINTS (M,3)
  const float* dirs = nullptr;   // IN_POINTS (M,3);  IN_RAYS (R,3)
  const float* ray_o = nullptr;  // IN_RAYS
  int o_stride = 0;              //   0: shared origin, 3: per ray
  const float* t = nullptr;      // IN_RAYS (R,S)
  int S = 0;
  const float* lin0 = nullptr;   // IN_GRID: device linspace tables
  const float* lin1 = nullptr;
  const float* lin2 = nullptr;
  int n1 = 0, n2 = 0;
  long long grid_base = 0;       //   flat index of the first point
  long long M = 0;               // number of points
};

// Optional by-products of a fused-MLP launch for the training backward (nm_train.cu): per layer (nullptr = not wanted)
//   packT  the layer's output as the point-major bf16 hi/lo operand pack of the weight-gradient GEMM (nm_gemm.h: tiles of
//          128 features x 64 points, [feature block][point block], `kbt` point blocks per feature block; rows >= M zero)
//   bits   its relu mask, one bit per element (halfword [m * n_out/16 + n/16], bit n%16)
//   act    its fp32 value (M, n_out) row-major (the layers the SIMT head kernels read)
struct MlpEmit {
  uint8_t* packT[kMaxLayers];
  uint32_t* bits[kMaxLayers];
  float* act[kMaxLayers];
  int kbt;
  int mn;      // packT as MN-major tiles (bulk stores from a shared-memory staging block) instead of K-major ones
};

int build_programs(const NmNetDesc& d, NetProgram* full, NetProgram* sigma);
int build_backward_program(const NetProgram& full, NetProgram* bwd);
int build_backward_stream(NetDev* net, cudaStream_t st, int64_t* launches);
// Packs host fp32 reference tensors into the device layouts.  `get(name, &numel)` returns the host tensor.
struct WeightSource {
  int n = 0;
  const char* const* names = nullptr;
  const float* const* ptrs = nullptr;
  const int64_t* numel = nullptr;
  const float* find(const std::string& name, int64_t expect) const;
};
int pack_network(const NmNetDesc& d, const WeightSource& src, NetDev* net);
int load_network_dev(const NmNetDesc& d, const WeightSource& src_device, NetDev* net, cudaStream_t st, int64_t* launches);
void free_network(NetDev* net);
int debug_pack(const NmNetDesc& d, const WeightSource& src, bool sigma_only, NetProgram* prog, uint8_t* out, size_t cap,
               size_t* need);

// kernel launchers (return 0 / <0; count launches via *launches)
struct CompositeArgs;
// comp != nullptr (inference on ray inputs): the compositor runs inside the kernel on the staged outputs of every tile and
// writes the per-ray maps (and weights, if asked); `out` is not written.  mlp_tc_composite_group(S) == 0: not eligible.
int mlp_tc_composite_group(int samples_per_ray);
int launch_mlp_tc(const NetDev& net, bool sigma_only, int n_passes, int act_scale_log2, const MlpInput& in, float* out,
                  int num_sms, int* d_err, cudaStream_t st, int64_t* launches, const MlpEmit* emit = nullptr,
                  const CompositeArgs* comp = nullptr);
int launch_mlp_tc_bwd(const NetDev& net, long long M, const float* dz_in, int dz_ld, const float* dout,
                      const MlpEmit& io, int n_passes, int num_sms, int* d_err, cudaStream_t st, int64_t* launches, int emit_mn = 0);
int launch_mlp_simt(const NetDev& net, bool sigma_only, const MlpInput& in, float* out, cudaStream_t st,
                    int64_t* launches);

struct RayGenArgs {
  float pose[12];
  int H, W;
  float focal;
  int ndc;
  float ndc_near;
  int row0, row1;
};
int launch_raygen(const RayGenArgs& a, float* origins_or_null, float* dirs, cudaStream_t st, int64_t* launches);
int launch_ndc(int H, int W, float focal, float near, const float* origins, int o_stride, const float* dirs, long long n,
               float* out_o, float* out_d, cudaStream_t st, int64_t* launches);
int launch_stratified(const float* s_table, int Nc, long long R, const float* near_far2, const float* near_dev,
                      const float* far_dev, int lindisp, int perturb, uint64_t seed, float* t_out, cudaStream_t st,
                      int64_t* launches);
struct CompositeArgs {
  const float* raw;    // (R,S,4)
  const float* t;      // (R,S)
  const float* dirs;   // (R,3)
  long long R;
  int S;
  float noise_std;
  uint64_t seed;
  int white_bg, training;
  float thr;
  float *rgb, *depth, *depth_raw, *acc, *disp, *weights, *mask_weights;
};
int launch_composite(const CompositeArgs& a, cudaStream_t st, int64_t* launches);
int launch_invcdf(const float* t_c, const float* w_c, const float* u_table, int Nc, int Nf, long long R, int perturb,
                  uint64_t seed, float* t_f, cudaStream_t st, int64_t* launches);
int launch_aabb(const float* voxels, int V, const float* origins, int o_stride, const float* dirs, long long R,
                float near, float far, int S, const float* s_table, const float* t_uniform, float* z_out, int* idx_out,
                int* d_overflow, cudaStream_t st, int64_t* launches, int random = 0, uint64_t seed = 0);
int launch_tree_integrate(const int* idx, const float* w, const float* mw, long long n, float* memm, int V, int counter,
                          float* scratch2v, cudaStream_t st, int64_t* launches);
int launch_volume_stats(const float* vol, long long n, double* d_scratch, float* out_host, cudaStream_t st,
                        int64_t* launches);
int launch_volume_stats_pass(const float* vol, long long n, int pass, const double* mean_dev, double* out_dev, cudaStream_t st,
                             int64_t* launches);
// training backward (nm_train.cu)
size_t train_ws_bytes(const NetProgram& full, long long points, bool use_tc);
struct TrainMode { int use_tc; int n_passes; int* d_err; };
int mlp_backward(NetDev& net, const MlpInput& in, const float* dout, float* ws, NetGrads* g, int num_sms,
                 const TrainMode& mode, cudaStream_t st, int64_t* launches, int have_acts = 0);
bool train_fused(bool use_tc);
void train_emit_setup(const NetProgram& full, long long points, float* ws, MlpEmit* emit);
int debug_tc_gemm(const float* A, const float* B, int M, int N, int K, int a_cols, int b_cols, int k_split, int n_passes,
                  int fp16, int atomic, float* D, uint8_t* scratch, size_t scratch_bytes, int num_sms, int* d_err, cudaStream_t st,
                  int64_t* launches);
int launch_composite_backward(const float* raw, const float* t, const float* dirs, const float* d_rgb, long long R, int S,
                              float noise_std, uint64_t seed, int white_bg, float* scratch, float* dout,
                              cudaStream_t st, int64_t* launches);
int launch_mse_grad(const float* rgb, const float* target, long long n, long long count, float* d_rgb, float* loss,
                    cudaStream_t st, int64_t* launches);
// marching cubes (nm_mc.cu): one shard of a global grid — buffer planes [0,nb) are global planes [g_x0, g_x0+nb) of g_nx;
// the call owns the points (vertices, cells) of buffer planes [p_lo,p_hi)
struct McShard {
  const float* vol;
  int nb, ny, nz;
  float iso;
  int g_x0, g_nx, p_lo, p_hi;
  int x_shift;       // added to the axis-0 vertex coordinates only (stand-alone volumes that are a window of a larger one)
};
// counts_host[2]: {vertices owned, triangles}; ws2 is a second grow-only workspace (8 bytes per output vertex / triangle)
int mc_count(const McShard& s, void** ws, size_t* ws_bytes, int64_t* counts_host, cudaStream_t st, int64_t* launches);
int mc_emit(const McShard& s, void* ws, size_t ws_bytes, void** ws2, size_t* ws2_bytes, long long v_base, int64_t nv, int64_t nt,
            float* verts, float* normals, int32_t* faces, cudaStream_t st, int64_t* launches);
// metrics (nm_metrics.cu): exact nearest neighbour and area-weighted surface sampling; callers size `ws` with the *_ws_bytes
size_t nearest_ws_bytes(long long N, long long M, int num_sms);
int launch_nearest(const float* x, long long N, const float* y, long long M, float* d, int* j, void* ws, int num_sms,
                   cudaStream_t st, int64_t* launches);
size_t mesh_sample_ws_bytes(long long F);
int launch_mesh_sample(const float* verts, const int* faces, long long F, long long n, uint64_t seed, float* points, int* face_idx,
                       float* normals, void* ws, cudaStream_t st, int64_t* launches);

}  // namespace nm
