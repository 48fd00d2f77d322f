// NeuS field variant (SURVEY 8(f) item 3): the reference's NeuS network as one persistent CUDA-core kernel.
// The tile program (index arithmetic, activations, density) lives in neus_kernel.cuh, which is also compiled by
// g++ into a host emulation for the CPU tests; this file supplies the kernel, the weight packing and the C ABI
// (neddf_neus_*).  Forward only, fp32 FMA (parity class of the fp32 NeDDF engine).
#include "neus_kernel.cuh"

#include <algorithm>
#include <cstring>

namespace neddf {
namespace neus {

__global__ void __launch_bounds__(kThreads, 1) neus_forward_kernel(const __grid_constant__ Params P) {
  extern __shared__ __align__(16) float smem[];
  CudaCtx cx{(int)threadIdx.x, (int)blockIdx.x, (int)gridDim.x};
  tile_program(cx, P, smem);
}

// colour output layer [3][256] + 3 biases as stored by torch, and the variance parameter
__global__ void neus_pack_head_kernel(const float* __restrict__ wc, const float* __restrict__ bc, const float* __restrict__ variance,
                                      float* __restrict__ dst_head, float* __restrict__ dst_var) {
  for (int i = threadIdx.x; i < 3 * kW; i += blockDim.x) dst_head[i] = wc[i];
  if (threadIdx.x < 3) dst_head[3 * kW + threadIdx.x] = bc[threadIdx.x];
  if (threadIdx.x == 0) dst_var[0] = variance[0];
}

}  // namespace neus
}  // namespace neddf

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
using namespace neddf;

struct neddf_neus {
  neddf_neus_config_t cfg;
  int n_layers = 0;
  int shape_in[neus::kMaxSdf + neus::kMaxCol + 2];
  int shape_out[neus::kMaxSdf + neus::kMaxCol + 2];
  neus::Params proto;  // network part filled at creation
  float* d_w = nullptr;
  size_t w_floats = 0;
  bool packed = false;
};

static int32_t neus_check(const neddf_neus_config_t* cfg, const char* who) {
  if (!cfg) return fail(NEDDF_E_INVALID, std::string(who) + ": null config");
  if (const char* why = neus::unsupported(cfg)) return fail(NEDDF_E_UNSUPPORTED, std::string(who) + ": " + why);
  return NEDDF_OK;
}

extern "C" int32_t neddf_neus_layer_shapes(const neddf_neus_config_t* cfg, int32_t* shapes_out, int32_t max_layers) {
  if (int32_t rc = neus_check(cfg, "neddf_neus_layer_shapes")) return rc;
  int sin[neus::kMaxSdf + neus::kMaxCol + 2], sout[neus::kMaxSdf + neus::kMaxCol + 2];
  const int n = neus::layer_shapes(cfg, sin, sout);
  if (shapes_out) {
    if (max_layers < n) return fail(NEDDF_E_INVALID, "neddf_neus_layer_shapes: buffer too small");
    for (int i = 0; i < n; ++i) {
      shapes_out[2 * i] = sin[i];
      shapes_out[2 * i + 1] = sout[i];
    }
  }
  return n;
}

extern "C" int32_t neddf_neus_create(const neddf_neus_config_t* cfg, neddf_neus_t** out) {
  if (!out) return fail(NEDDF_E_INVALID, "neddf_neus_create: null argument");
  if (int32_t rc = neus_check(cfg, "neddf_neus_create")) return rc;
  neddf_neus* h = new neddf_neus();
  h->cfg = *cfg;
  h->n_layers = neus::layer_shapes(cfg, h->shape_in, h->shape_out);
  std::memset(&h->proto, 0, sizeof(h->proto));
  h->w_floats = neus::build_program(cfg, h->proto);
  if (cudaMalloc(&h->d_w, h->w_floats * sizeof(float)) != cudaSuccess) {
    delete h;
    return fail(NEDDF_E_CUDA, "neddf_neus_create: cudaMalloc failed");
  }
  *out = h;
  return NEDDF_OK;
}

extern "C" void neddf_neus_destroy(neddf_neus_t* h) {
  if (!h) return;
  cudaFree(h->d_w);
  delete h;
}

extern "C" int32_t neddf_neus_set_weights(neddf_neus_t* h, const float* const* d_w, const float* const* d_b, int32_t n_layers,
                                          const float* d_variance, void* stream) {
  if (!h || !d_w || !d_b || !d_variance) return fail(NEDDF_E_INVALID, "neddf_neus_set_weights: null argument");
  if (n_layers != h->n_layers) return fail(NEDDF_E_INVALID, "neddf_neus_set_weights: expected sdf_layer_count + col_layer_count + 1 layers");
  cudaStream_t s = (cudaStream_t)stream;
  const neus::Params& P = h->proto;
  for (int t = 0; t < n_layers - 1; ++t) {
    const neus::Layer& ly = (t < P.n_sdf) ? P.lsdf[t] : P.lcol[t - P.n_sdf];
    simt::pack_layer_kernel<<<64, 256, 0, s>>>(d_w[t], d_b[t], h->shape_in[t], h->shape_out[t], ly, h->d_w);
    NEDDF_LAUNCH_CHECK();
  }
  neus::neus_pack_head_kernel<<<1, 256, 0, s>>>(d_w[n_layers - 1], d_b[n_layers - 1], d_variance, h->d_w + P.head_off, h->d_w + P.var_off);
  NEDDF_LAUNCH_CHECK();
  h->packed = true;
  return NEDDF_OK;
}

static int32_t neus_launch(const neddf_neus_t* h, neus::Params& P, void* stream) {
  if (!h->packed) return fail(NEDDF_E_INVALID, "neddf_neus_forward: weights were never set");
  if (P.n <= 0) return NEDDF_OK;
  P.w = h->d_w;
  const int64_t n_tiles = (P.n + neus::kT - 1) / neus::kT;
  const int grid = (int)std::min<int64_t>(n_tiles, sm_count());
  NEDDF_CUDA_CHECK(cudaFuncSetAttribute(neus::neus_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)neus::kSmemBytes));
  neus::neus_forward_kernel<<<grid, neus::kThreads, neus::kSmemBytes, (cudaStream_t)stream>>>(P);
  NEDDF_LAUNCH_CHECK();
  return NEDDF_OK;
}

extern "C" int32_t neddf_neus_forward(const neddf_neus_t* h, const float* d_pos, const float* d_dir, int64_t n, float* d_sdf,
                                      float* d_density, float* d_color, float* d_normal, void* stream) {
  if (!h || !d_pos || !d_dir || !d_sdf || !d_density || !d_color) return fail(NEDDF_E_INVALID, "neddf_neus_forward: null argument");
  neus::Params P = h->proto;
  P.n = n;
  P.pos = d_pos; P.dir = d_dir;
  P.sdf = d_sdf; P.density = d_density; P.color = d_color; P.normal = d_normal;
  return neus_launch(h, P, stream);
}

extern "C" int32_t neddf_neus_forward_rays(const neddf_neus_t* h, const float* d_ray_dir, const float* d_ray_orig, const float* d_dists,
                                           int64_t n_rays, int32_t n_edges, int32_t sampling_type, float ray_radius, float* d_sdf,
                                           float* d_density, float* d_color, float* d_normal, void* stream) {
  if (!h || !d_ray_dir || !d_ray_orig || !d_dists || !d_sdf || !d_density || !d_color)
    return fail(NEDDF_E_INVALID, "neddf_neus_forward_rays: null argument");
  if (n_edges < 1 || (sampling_type != NEDDF_SAMPLING_POINT && sampling_type != NEDDF_SAMPLING_CONE))
    return fail(NEDDF_E_INVALID, "neddf_neus_forward_rays: bad n_edges / sampling_type");
  neus::Params P = h->proto;
  P.n = n_rays * n_edges;
  P.ray_dir = d_ray_dir; P.ray_orig = d_ray_orig; P.dists = d_dists;
  P.n_edges = n_edges; P.sampling_type = sampling_type; P.ray_radius = ray_radius;
  P.sdf = d_sdf; P.density = d_density; P.color = d_color; P.normal = d_normal;
  return neus_launch(h, P, stream);
}
