// NeRF field variant (SURVEY 8(f) item 3): the reference's vanilla NeRF MLP as persistent CUDA-core kernels - the
// forward (neddf_nerf_*) and the training backward (neddf_nerf_train_*), two instantiations of the tile program of
// nerf_train_kernel.cuh (which is also compiled by g++ into a host emulation for the CPU tests).  This file supplies the
// kernels, the weight packing and the C ABI.  The backward leaves the operands of the weight-gradient GEMMs (layer
// inputs X, pre-activation gradients G) in global memory for neddf_wgrad.
#include "nerf_train_kernel.cuh"

#include <algorithm>
#include <cstring>
#include <type_traits>

namespace neddf {
namespace nerft {

__global__ void __launch_bounds__(kThreads, 1) nerf_forward_kernel(const __grid_constant__ Params P) {
  extern __shared__ __align__(16) float smem[];
  CudaCtx cx{(int)threadIdx.x, (int)blockIdx.x, (int)gridDim.x};
  tile_program<false>(cx, P, smem);
}

__global__ void __launch_bounds__(kThreads, 1) nerf_train_kernel(const __grid_constant__ Params P) {
  extern __shared__ __align__(16) float smem[];
  CudaCtx cx{(int)threadIdx.x, (int)blockIdx.x, (int)gridDim.x};
  tile_program<true>(cx, P, smem);
}

// small heads: density [256] + bias, colour [3][128] + 3 biases, as stored by torch
__global__ void nerf_pack_heads_kernel(const float* __restrict__ wd, const float* __restrict__ bd, const float* __restrict__ wc,
                                       const float* __restrict__ bc, float* __restrict__ dst_d, float* __restrict__ dst_c) {
  for (int i = threadIdx.x; i < kW; i += blockDim.x) dst_d[i] = wd[i];
  if (threadIdx.x == 0) dst_d[kW] = bd[0];
  for (int i = threadIdx.x; i < 3 * (kW / 2); i += blockDim.x) dst_c[i] = wc[i];
  if (threadIdx.x < 3) dst_c[3 * (kW / 2) + threadIdx.x] = bc[threadIdx.x];
}

}  // namespace nerft
}  // namespace neddf

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace neddf;

struct neddf_nerf {
  neddf_nerf_config_t cfg;
  int shape_in[nerft::kMaxLayers + 3];
  int shape_out[nerft::kMaxLayers + 3];
  nerft::Params proto;  // network part filled at creation
  float* d_w = nullptr;
  bool packed = false;
};
// the training handle is the same; its weight buffer also holds the transposed packs of the backward
struct neddf_nerf_train : neddf_nerf {};

extern "C" int32_t neddf_nerf_layer_shapes(const neddf_nerf_config_t* cfg, int32_t* shapes_out, int32_t max_layers) {
  if (!cfg || cfg->layer_count < 2 || cfg->layer_count > nerft::kMaxLayers) return fail(NEDDF_E_INVALID, "neddf_nerf_layer_shapes: bad config");
  int sin[nerft::kMaxLayers + 3], sout[nerft::kMaxLayers + 3];
  const int n = nerft::layer_shapes(cfg, sin, sout);
  if (shapes_out) {
    if (max_layers < n) return fail(NEDDF_E_INVALID, "neddf_nerf_layer_shapes: buffer too small");
    for (int i = 0; i < n; ++i) {
      shapes_out[2 * i] = sin[i];
      shapes_out[2 * i + 1] = sout[i];
    }
  }
  return n;
}

template <class Handle>
static int32_t nerf_create(const neddf_nerf_config_t* cfg, Handle** out, const char* who) {
  if (!cfg || !out) return fail(NEDDF_E_INVALID, std::string(who) + ": null argument");
  int32_t code;
  if (const char* why = nerft::unsupported(cfg, &code)) return fail(code, std::string(who) + ": " + why);
  Handle* h = new Handle();
  h->cfg = *cfg;
  nerft::layer_shapes(cfg, h->shape_in, h->shape_out);
  std::memset(&h->proto, 0, sizeof(h->proto));
  const size_t w_floats = nerft::build_program(cfg, h->proto, std::is_same<Handle, neddf_nerf_train>::value);
  if (cudaMalloc(&h->d_w, w_floats * sizeof(float)) != cudaSuccess) {
    delete h;
    return fail(NEDDF_E_CUDA, std::string(who) + ": cudaMalloc failed");
  }
  *out = h;
  return NEDDF_OK;
}

template <class Handle>
static void nerf_destroy(Handle* h) {
  if (!h) return;
  cudaFree(h->d_w);
  delete h;
}

static int32_t nerf_set_weights(neddf_nerf* h, const float* const* d_w, const float* const* d_b, int32_t n_layers, void* stream,
                                 const char* who) {
  if (!h || !d_w || !d_b) return fail(NEDDF_E_INVALID, std::string(who) + ": null argument");
  const int L = h->cfg.layer_count;
  if (n_layers != L + 3) return fail(NEDDF_E_INVALID, std::string(who) + ": expected layer_count + 3 layers");
  cudaStream_t s = (cudaStream_t)stream;
  // hidden layers 0..L-1 are tensors 0..L-1; the colour branch's first layer (kernel layer L) is tensor L + 1
  for (int l = 0; l <= L; ++l) {
    const int t = (l < L) ? l : L + 1;
    simt::pack_layer_kernel<<<64, 256, 0, s>>>(d_w[t], d_b[t], h->shape_in[t], h->shape_out[t], h->proto.layer[l], h->d_w);
    NEDDF_LAUNCH_CHECK();
  }
  nerft::nerf_pack_heads_kernel<<<1, 256, 0, s>>>(d_w[L], d_b[L], d_w[L + 2], d_b[L + 2], h->d_w + h->proto.w_density_off,
                                                 h->d_w + h->proto.w_col2_off);
  NEDDF_LAUNCH_CHECK();
  h->packed = true;
  return NEDDF_OK;
}

static int32_t nerf_launch(const neddf_nerf* h, void (*kernel)(nerft::Params), nerft::Params& P, const float* lowpass, void* stream,
                           const char* who) {
  if (!h->packed) return fail(NEDDF_E_INVALID, std::string(who) + ": weights were never set");
  if (!lowpass) return fail(NEDDF_E_INVALID, std::string(who) + ": lowpass is null");
  if (P.n <= 0) return NEDDF_OK;
  for (int e = 0; e < h->cfg.embed_pos_rank; ++e) P.lowpass[e] = lowpass[e];
  P.w = h->d_w;
  const int64_t n_tiles = (P.n + nerft::kT - 1) / nerft::kT;
  const int grid = (int)std::min<int64_t>(n_tiles, sm_count());
  NEDDF_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)nerft::kSmemBytes));
  kernel<<<grid, nerft::kThreads, nerft::kSmemBytes, (cudaStream_t)stream>>>(P);
  NEDDF_LAUNCH_CHECK();
  return NEDDF_OK;
}

static int32_t nerf_rays(nerft::Params& P, const float* d_ray_dir, const float* d_ray_orig, const float* d_dists, int64_t n_rays,
                         int32_t n_edges, int32_t sampling_type, float ray_radius, const char* who) {
  if (n_edges < 1 || (sampling_type != NEDDF_SAMPLING_POINT && sampling_type != NEDDF_SAMPLING_CONE))
    return fail(NEDDF_E_INVALID, std::string(who) + ": bad n_edges / sampling_type");
  P.n = n_rays * n_edges;
  P.ray_dir = d_ray_dir; P.ray_orig = d_ray_orig; P.dists = d_dists;
  P.n_edges = n_edges; P.sampling_type = sampling_type; P.ray_radius = ray_radius;
  return NEDDF_OK;
}

// ---- forward ----
extern "C" int32_t neddf_nerf_create(const neddf_nerf_config_t* cfg, neddf_nerf_t** out) { return nerf_create(cfg, out, "neddf_nerf_create"); }

extern "C" void neddf_nerf_destroy(neddf_nerf_t* h) { nerf_destroy(h); }

extern "C" int32_t neddf_nerf_set_weights(neddf_nerf_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                                          void* stream) {
  return nerf_set_weights(h, d_w, d_b, n_layers, stream, "neddf_nerf_set_weights");
}

extern "C" int32_t neddf_nerf_forward(const neddf_nerf_t* h, const float* lowpass, const float* d_pos, const float* d_dir,
                                      const float* d_var, int64_t n, float* d_density, float* d_color, void* stream) {
  if (!h || !d_pos || !d_dir || !d_var || !d_density || !d_color) return fail(NEDDF_E_INVALID, "neddf_nerf_forward: null argument");
  nerft::Params P = h->proto;
  P.n = n;
  P.pos = d_pos; P.dir = d_dir; P.var = d_var;
  P.density = d_density; P.color = d_color;
  return nerf_launch(h, nerft::nerf_forward_kernel, P, lowpass, stream, "neddf_nerf_forward");
}

extern "C" int32_t neddf_nerf_forward_rays(const neddf_nerf_t* h, const float* lowpass, const float* d_ray_dir, const float* d_ray_orig,
                                           const float* d_dists, int64_t n_rays, int32_t n_edges, int32_t sampling_type,
                                           float ray_radius, float* d_density, float* d_color, void* stream) {
  const char* who = "neddf_nerf_forward_rays";
  if (!h || !d_ray_dir || !d_ray_orig || !d_dists || !d_density || !d_color) return fail(NEDDF_E_INVALID, std::string(who) + ": null argument");
  nerft::Params P = h->proto;
  if (int32_t rc = nerf_rays(P, d_ray_dir, d_ray_orig, d_dists, n_rays, n_edges, sampling_type, ray_radius, who)) return rc;
  P.density = d_density; P.color = d_color;
  return nerf_launch(h, nerft::nerf_forward_kernel, P, lowpass, stream, who);
}

// ---- training backward ----
extern "C" int32_t neddf_nerf_train_create(const neddf_nerf_config_t* cfg, neddf_nerf_train_t** out) {
  return nerf_create(cfg, out, "neddf_nerf_train_create");
}

extern "C" void neddf_nerf_train_destroy(neddf_nerf_train_t* h) { nerf_destroy(h); }

extern "C" int32_t neddf_nerf_train_set_weights(neddf_nerf_train_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                                                void* stream) {
  return nerf_set_weights(h, d_w, d_b, n_layers, stream, "neddf_nerf_train_set_weights");
}

static int32_t nerf_train_launch(const neddf_nerf_train_t* h, nerft::Params& P, const float* lowpass, const float* g_density,
                                 const float* g_color, float* X, float* G, float* E, float* D, float* C1, float* GC1, float* GZD,
                                 void* stream) {
  if (!g_density || !g_color || !X || !G || !E || !D || !C1 || !GC1 || !GZD)
    return fail(NEDDF_E_INVALID, "neddf_nerf_train_backward: null argument");
  P.g_density = g_density; P.g_color = g_color;
  P.X = X; P.G = G; P.Eo = E; P.Do = D; P.C1 = C1; P.GC1 = GC1; P.GZD = GZD;
  return nerf_launch(h, nerft::nerf_train_kernel, P, lowpass, stream, "neddf_nerf_train_backward");
}

extern "C" int32_t neddf_nerf_train_backward(const neddf_nerf_train_t* h, const float* lowpass, const float* d_pos, const float* d_dir,
                                             const float* d_var, int64_t n, const float* d_g_density, const float* d_g_color, float* d_x,
                                             float* d_g, float* d_e, float* d_d, float* d_c1, float* d_gc1, float* d_gzd, void* stream) {
  if (!h || !d_pos || !d_dir || !d_var) return fail(NEDDF_E_INVALID, "neddf_nerf_train_backward: null argument");
  nerft::Params P = h->proto;
  P.n = n;
  P.pos = d_pos; P.dir = d_dir; P.var = d_var;
  return nerf_train_launch(h, P, lowpass, d_g_density, d_g_color, d_x, d_g, d_e, d_d, d_c1, d_gc1, d_gzd, stream);
}

extern "C" int32_t neddf_nerf_train_backward_rays(const neddf_nerf_train_t* h, const float* lowpass, const float* d_ray_dir,
                                                  const float* d_ray_orig, const float* d_dists, int64_t n_rays, int32_t n_edges,
                                                  int32_t sampling_type, float ray_radius, const float* d_g_density,
                                                  const float* d_g_color, float* d_x, float* d_g, float* d_e, float* d_d, float* d_c1,
                                                  float* d_gc1, float* d_gzd, void* stream) {
  const char* who = "neddf_nerf_train_backward_rays";
  if (!h || !d_ray_dir || !d_ray_orig || !d_dists) return fail(NEDDF_E_INVALID, std::string(who) + ": null argument");
  nerft::Params P = h->proto;
  if (int32_t rc = nerf_rays(P, d_ray_dir, d_ray_orig, d_dists, n_rays, n_edges, sampling_type, ray_radius, who)) return rc;
  return nerf_train_launch(h, P, lowpass, d_g_density, d_g_color, d_x, d_g, d_e, d_d, d_c1, d_gc1, d_gzd, stream);
}
