// Sanitizer driver for the emulated NeRF kernels, forward and training backward (TEST INFRASTRUCTURE): see
// neus_emul_main.cpp.  Exact-size buffers (a store past sample n - 1 is a heap overflow), full + ragged tiles, two CTAs,
// explicit samples and fused ray geometry.  Exit code 0 = clean.
#include "nerf_train_emul.cpp"

#include <stdio.h>

#include <random>

static int run(const neddf_nerf_config_t& cfg, int n, bool rays, unsigned seed) {
  int sin[nerft::kMaxLayers + 3], sout[nerft::kMaxLayers + 3];
  const int nl = nerft::layer_shapes(&cfg, sin, sout);
  const int L = cfg.layer_count, n_e = 6 * cfg.embed_pos_rank, n_d = 6 * cfg.embed_dir_rank;
  std::mt19937 g(seed);
  std::normal_distribution<float> nd(0.f, 1.f);
  std::vector<std::vector<float>> W(nl), B(nl);
  std::vector<const float*> wp(nl), bp(nl);
  for (int t = 0; t < nl; ++t) {
    W[t].resize((size_t)sin[t] * sout[t]);
    B[t].resize(sout[t]);
    const float s = sqrtf(2.f / (sin[t] + sout[t]));
    for (auto& v : W[t]) v = s * nd(g);
    for (auto& v : B[t]) v = 0.05f * nd(g);
    wp[t] = W[t].data();
    bp[t] = B[t].data();
  }
  float lowpass[16];
  for (int e = 0; e < 16; ++e) lowpass[e] = e < 3 ? 1.f : 0.3f;
  const int n_edges = rays ? 7 : 0;
  const long long total = rays ? (long long)n * n_edges : n;
  std::vector<float> pos(3 * total), dir(3 * total), var(3 * total), rd(3 * n), ro(3 * n), dists((size_t)n * (rays ? n_edges : 1));
  for (auto& v : pos) v = 0.8f * nd(g);
  for (auto& v : var) v = 1e-4f * fabsf(nd(g));
  for (long long i = 0; i < total; ++i) {
    float a = nd(g), b = nd(g), c = nd(g), r = sqrtf(a * a + b * b + c * c) + 1e-6f;
    dir[3 * i] = a / r; dir[3 * i + 1] = b / r; dir[3 * i + 2] = c / r;
  }
  for (int i = 0; i < n; ++i) {
    float a = nd(g), b = nd(g), c = nd(g), r = sqrtf(a * a + b * b + c * c) + 1e-6f;
    rd[3 * i] = a / r; rd[3 * i + 1] = b / r; rd[3 * i + 2] = c / r;
    ro[3 * i] = 0.1f * nd(g); ro[3 * i + 1] = 0.1f * nd(g); ro[3 * i + 2] = 0.1f * nd(g);
    for (int j = 0; j < n_edges; ++j) dists[(size_t)i * n_edges + j] = 2.f + 0.5f * j + 0.1f * fabsf(nd(g));
  }
  std::vector<float> gd(total), gc(3 * total);
  for (auto& v : gd) v = nd(g);
  for (auto& v : gc) v = nd(g);
  std::vector<float> X((size_t)L * total * 256), G((size_t)L * total * 256), E((size_t)total * n_e), D((size_t)total * n_d), C1((size_t)total * 256),
      GC1((size_t)total * 256), GZD(total);
  const int rc = nerf_train_emul(&cfg, wp.data(), bp.data(), nl, lowpass, rays ? nullptr : pos.data(), rays ? nullptr : dir.data(),
                                 rays ? nullptr : var.data(), rays ? rd.data() : nullptr, rays ? ro.data() : nullptr,
                                 rays ? dists.data() : nullptr, n, n_edges, NEDDF_SAMPLING_CONE, 2.6e-4f, gd.data(), gc.data(), X.data(),
                                 G.data(), E.data(), D.data(), C1.data(), GC1.data(), GZD.data(), 2);
  double sum = 0;
  for (float v : G) sum += v;
  for (float v : GC1) sum += v;
  for (float v : GZD) sum += v;
  printf("rc %d checksum %.6f (%lld samples)\n", rc, sum, total);
  std::vector<float> den(total), col(3 * total);
  const int rc_f = nerf_forward_emul(&cfg, wp.data(), bp.data(), nl, lowpass, rays ? nullptr : pos.data(), rays ? nullptr : dir.data(),
                                     rays ? nullptr : var.data(), rays ? rd.data() : nullptr, rays ? ro.data() : nullptr,
                                     rays ? dists.data() : nullptr, n, n_edges, NEDDF_SAMPLING_CONE, 2.6e-4f, den.data(), col.data(), 2);
  double sum_f = 0;
  for (long long i = 0; i < total; ++i) sum_f += den[i] + col[3 * i] + col[3 * i + 2];
  printf("forward rc %d checksum %.6f (%lld samples)\n", rc_f, sum_f, total);
  return (rc == 0 && sum == sum && rc_f == 0 && sum_f == sum_f) ? 0 : 1;
}

int main() {
  neddf_nerf_config_t a = {10, 4, 8, 256, NEDDF_ACT_RELU, NEDDF_ACT_RELU, 1, {4}};               // config/network/nerf.yaml
  neddf_nerf_config_t b = {3, 2, 3, 256, NEDDF_ACT_TANHEXP, NEDDF_ACT_LEAKYRELU, 2, {0, 1}};  // shallow, skips after layers 0 and 1
  int bad = 0;
  bad |= run(a, 70, false, 1);  // one full tile + a ragged one, two CTAs
  bad |= run(b, 19, true, 2);   // fused ray geometry, 133 samples: three tiles (CTA 0 runs two of them)
  return bad;
}
