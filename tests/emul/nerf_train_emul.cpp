// Host emulation of the NeRF kernels (TEST INFRASTRUCTURE; built and loaded only by tests/test_nerf_train_emul.py):
// neddf_b200/csrc/nerf_train_kernel.cuh - the tile program of csrc/nerf.cu, forward and training backward - compiled by g++
// and run on 256 OS threads per CTA (emul_common.h).
#include "emul_common.h"

#include "../../neddf_b200/csrc/nerf_train_kernel.cuh"

using namespace neddf;

// Weights as torch stores them (w[i] = [out][in], b[i] = [out], order of neddf_nerf_layer_shapes) packed as
// neddf_nerf[_train]_set_weights packs them; explicit samples (pos / dir / var, n = samples) or rays (n = rays).
// Returns 0, -1 for an unsupported configuration (same rule as neddf_nerf_create), -2 for a wrong layer count.
static int setup(const neddf_nerf_config_t* cfg, bool train, const float* const* w, const float* const* b, int n_layers,
                 const float* lowpass, const float* pos, const float* dir, const float* var, const float* ray_dir,
                 const float* ray_orig, const float* dists, long long n, int n_edges, int sampling_type, float ray_radius,
                 nerft::Params& P, std::vector<float>& packed) {
  if (nerft::unsupported(cfg)) return -1;
  memset(&P, 0, sizeof(P));
  packed.assign(nerft::build_program(cfg, P, train), 0.f);
  int sin[nerft::kMaxLayers + 3], sout[nerft::kMaxLayers + 3];
  if (nerft::layer_shapes(cfg, sin, sout) != n_layers) return -2;
  const int L = cfg->layer_count;
  // simt::pack_layer_kernel per layer, nerf_pack_heads_kernel
  for (int l = 0; l <= L; ++l) {
    const int t = (l < L) ? l : L + 1;
    const simt::Layer& ly = P.layer[l];
    for (int idx = 0; idx < ly.k_pad * simt::kW; ++idx)
      packed[ly.w_off + idx] = simt::pack_fwd(w[t], sin[t], sout[t], idx / simt::kW, idx % simt::kW);
    for (int idx = 0; idx < ly.kt_pad * simt::kW; ++idx)
      packed[ly.wt_off + idx] = simt::pack_bwd(w[t], sin[t], sout[t], idx / simt::kW, idx % simt::kW);
    for (int c = 0; c < simt::kW; ++c) packed[ly.b_off + c] = c < sout[t] ? b[t][c] : 0.f;
  }
  for (int i = 0; i < simt::kW; ++i) packed[P.w_density_off + i] = w[L][i];
  packed[P.w_density_off + simt::kW] = b[L][0];
  for (int i = 0; i < 3 * (simt::kW / 2); ++i) packed[P.w_col2_off + i] = w[L + 2][i];
  for (int i = 0; i < 3; ++i) packed[P.w_col2_off + 3 * (simt::kW / 2) + i] = b[L + 2][i];
  P.w = packed.data();
  for (int e = 0; e < cfg->embed_pos_rank; ++e) P.lowpass[e] = lowpass[e];
  if (dists) {
    P.n = n * n_edges;
    P.ray_dir = ray_dir; P.ray_orig = ray_orig; P.dists = dists;
    P.n_edges = n_edges; P.sampling_type = sampling_type; P.ray_radius = ray_radius;
  } else {
    P.n = n;
    P.pos = pos; P.dir = dir; P.var = var;
  }
  return 0;
}

template <bool kTrain>
static void run(const nerft::Params& P, int nblocks) {
  if (P.n <= 0) return;
#ifdef NEUS_EMUL_MISALIGN
  const int shift = 1;
#else
  const int shift = 0;
#endif
  emul::run_grid(nblocks, simt::kThreads, nerft::kSmemFloats, shift,
                 [&](emul::HostCtx& cx, float* smem) { nerft::tile_program<kTrain>(cx, P, smem); });
}

// neddf_nerf_forward[_rays]: density [n], colour [n, 3]
extern "C" int nerf_forward_emul(const neddf_nerf_config_t* cfg, const float* const* w, const float* const* b, int n_layers,
                                 const float* lowpass, const float* pos, const float* dir, const float* var, const float* ray_dir,
                                 const float* ray_orig, const float* dists, long long n, int n_edges, int sampling_type,
                                 float ray_radius, float* density, float* color, int nblocks) {
  nerft::Params P;
  std::vector<float> packed;
  if (int rc = setup(cfg, false, w, b, n_layers, lowpass, pos, dir, var, ray_dir, ray_orig, dists, n, n_edges, sampling_type,
                     ray_radius, P, packed))
    return rc;
  P.density = density; P.color = color;
  run<false>(P, nblocks);
  return 0;
}

// neddf_nerf_train_backward[_rays]: buffers as documented there
extern "C" int nerf_train_emul(const neddf_nerf_config_t* cfg, const float* const* w, const float* const* b, int n_layers,
                               const float* lowpass, const float* pos, const float* dir, const float* var, const float* ray_dir,
                               const float* ray_orig, const float* dists, long long n, int n_edges, int sampling_type,
                               float ray_radius, const float* g_density, const float* g_color, float* X, float* G, float* E,
                               float* D, float* C1, float* GC1, float* GZD, int nblocks) {
  nerft::Params P;
  std::vector<float> packed;
  if (int rc = setup(cfg, true, w, b, n_layers, lowpass, pos, dir, var, ray_dir, ray_orig, dists, n, n_edges, sampling_type,
                     ray_radius, P, packed))
    return rc;
  P.g_density = g_density; P.g_color = g_color;
  P.X = X; P.G = G; P.Eo = E; P.Do = D; P.C1 = C1; P.GC1 = GC1; P.GZD = GZD;
  run<true>(P, nblocks);
  return 0;
}
