// NeRF field variant (SURVEY 8(f) item 3): the tile program of csrc/nerf.cu, forward and training backward.
//
// Reference: NeRF.forward (neddf/network/nerf.py:107-165): position embedding with low-pass x sample-size weights
// (:133-141), `layer_count` hidden layers with the skip concat [h | E] after the layers named in `skips` (:144-148),
// density head + density activation (:149), colour branch Linear(width + dir embedding -> width/2), ReLU,
// Linear(-> 3) (:96-103, :151-153).  Sample geometry optionally fused like the NeDDF kernels
// (Ray.get_sampling_points / get_sampling_cones, neddf/ray/ray.py:88-194).  Every multiply-add is an fp32 FMA (parity
// class of the fp32 NeDDF engine) on the CUDA-core skeleton of simt_mlp.cuh.
//
// One tile program, two kernels (compile-time kTrain):
//  - forward (kTrain = false): density and colour per sample.
//  - training backward (kTrain = true), the autograd graph of the forward with respect to the network parameters
//    (what nerf_trainer.py:38-42 hands to Adam; sample positions carry no gradient).  Per 64-sample tile: (1) recompute
//    the forward, parking every layer's pre-activation z_l in the slot of the gradient buffer G[l] and its activation
//    h_l in X[l] (both [n][256], global, L2 resident while the tile is alive); (2) walk back: g_zc1 = (Wc2^T g_color)
//    relu'(z_c1), g_h = Wc1[:, :256]^T g_zc1 + w_density g_zd, and per hidden layer g_z_l = g_h_l act'(z_l)
//    (overwrites z_l in G[l]), g_h_{l-1} = W_l[:, :256]^T g_z_l.  The backward GEMMs are the skeleton's loop over
//    TRANSPOSED packs WT_l[k = output channel][c = input channel < 256].  The weight gradients are sums over ALL
//    samples, gW_l = X_{l-1}^T G_l: tensor-core split-K GEMMs of this library (neddf_wgrad, csrc/wgrad.cu) on the
//    buffers this kernel leaves behind; bias gradients are column sums of G_l.
#pragma once

#include "simt_mlp.cuh"

namespace neddf {
namespace nerft {

using namespace simt;

constexpr int kMaxE = 64;       // rows reserved for the position embedding (6 * embed_pos_rank <= 64)
constexpr int kMaxD = 32;       // direction embedding (6 * embed_dir_rank <= 32)
constexpr int kMaxLayers = 12;  // hidden layers

enum Seg { kSegNone = 0, kSegE = 1, kSegH = 2, kSegD = 3 };

struct Params : Samples {  // the samples, then:
  // network
  int n_layers;  // hidden layers; layer[n_layers] = first layer of the colour branch (128 outputs)
  Layer layer[kMaxLayers + 1];
  const float* w;  // packed weights + biases (+ transposed packs for the backward)
  int embed_pos, embed_dir, n_e, n_d;
  int act, density_act;
  int w_density_off;  // [256] + bias
  int w_col2_off;     // [3][128] + 3 biases
  float lowpass[16];
  // forward outputs
  float* density;  // [n]
  float* color;    // [n, 3]
  // backward: upstream gradients and the operands of the weight-gradient GEMMs
  const float* g_density;  // [n]    d loss / d density
  const float* g_color;    // [n, 3] d loss / d colour
  float* X;    // [n_layers][n][256] activations h_l
  float* G;    // [n_layers][n][256] pre-activation gradients g_z_l (z_l between the two phases)
  float* Eo;   // [n][n_e] position embedding
  float* Do;   // [n][n_d] direction embedding
  float* C1;   // [n][256] colour hidden activations (columns >= 128 are zero)
  float* GC1;  // [n][256] their pre-activation gradients (columns >= 128 are zero)
  float* GZD;  // [n]      gradient of the density pre-activation
};

// shared-memory map (floats)
constexpr int kOffE = 0;
constexpr int kOffD = kOffE + kMaxE * kT;
constexpr int kOffH = kOffD + kMaxD * kT;
constexpr int kOffW = kOffH + kW * kT;
constexpr int kOffGeo = kOffW + 2 * kChunk * kW;  // [kT][9] pos, dir, var
constexpr int kOffUp = kOffGeo + kT * 9;          // [kT][4] g_color (3), g_zd (backward only)
constexpr int kSmemFloats = kOffUp + kT * 4;
constexpr size_t kSmemBytes = (size_t)kSmemFloats * sizeof(float);

__device__ __forceinline__ float* seg_ptr(float* smem, int seg) {
  return smem + (seg == kSegE ? kOffE : (seg == kSegD ? kOffD : kOffH));
}

template <class Ctx>
__device__ __forceinline__ void gemm(Ctx& cx, const float* w, const Layer& Ly, float* smem, float (&acc)[4][4][4]) {
  layer_gemm(cx, w + Ly.w_off, Ly.k_pad, seg_ptr(smem, Ly.seg_a), Ly.n_a, seg_ptr(smem, Ly.seg_b), Ly.n_b, smem + kOffW, acc);
}

// One CTA: tiles cx.block, cx.block + cx.nblocks, ...
template <bool kTrain = true, class Ctx>
__device__ __forceinline__ void tile_program(Ctx& cx, const Params& P, float* smem) {
  float* E = smem + kOffE;
  float* D = smem + kOffD;
  float* H = smem + kOffH;
  float* geo = smem + kOffGeo;
  float* up = smem + kOffUp;
  const int tid = cx.tid;
  const int cg = tid & 15, sg = tid >> 4;
  const int64_t N = P.n;
  const int64_t n_tiles = (N + kT - 1) / kT;
  const int L = P.n_layers;
  float acc[4][4][4];

  for (int64_t tile = cx.block; tile < n_tiles; tile += cx.nblocks) {
    const int64_t n0 = tile * kT;
    // ---- geometry (+ upstream gradients) of the tile's samples (one thread per sample) ----
    if (tid < kT) {
      float pos[3], dir[3], var[3];
      const int64_t n = n0 + tid;
      load_sample(P, n, pos, dir, var);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        geo[tid * 9 + i] = pos[i];
        geo[tid * 9 + 3 + i] = dir[i];
        geo[tid * 9 + 6 + i] = var[i];
      }
      if constexpr (kTrain) {
#pragma unroll
        for (int i = 0; i < 3; ++i) up[tid * 4 + i] = (n < N) ? P.g_color[3 * n + i] : 0.f;
        up[tid * 4 + 3] = (n < N) ? P.g_density[n] : 0.f;  // g_density for now; becomes g_zd after the density head
      }
    }
    cx.sync();
    // ---- embeddings (nerf.py:133-142): four threads per sample ----
    {
      const int s = tid >> 2, sub = tid & 3;
      const int half3 = 3 * P.embed_pos;
      for (int idx = sub; idx < half3; idx += 4) {
        const int e = idx / 3, d = idx - 3 * e;
        const float f = (float)(1u << e);
        float sn, cs;
        sincosf(f * geo[s * 9 + d], &sn, &cs);
        const float scale = P.lowpass[e] * expf(-0.5f * (f * f) * geo[s * 9 + 6 + d]);  // sampling.py:58-71 x low-pass
        E[idx * kT + s] = scale * sn;
        E[(half3 + idx) * kT + s] = scale * cs;
      }
      const int dhalf = 3 * P.embed_dir;
      for (int idx = sub; idx < dhalf; idx += 4) {
        const int e = idx / 3, d = idx - 3 * e;
        float sn, cs;
        sincosf((float)(1u << e) * geo[s * 9 + 3 + d], &sn, &cs);
        D[idx * kT + s] = sn;
        D[(dhalf + idx) * kT + s] = cs;
      }
    }
    cx.sync();
    if constexpr (kTrain) {  // embeddings as GEMM operands of the weight gradients: [n][n_e], [n][n_d]
      for (int idx = tid; idx < kT * P.n_e; idx += kThreads) {
        const int s = idx / P.n_e, k = idx - s * P.n_e;
        if (n0 + s < N) P.Eo[(n0 + s) * P.n_e + k] = E[k * kT + s];
      }
      for (int idx = tid; idx < kT * P.n_d; idx += kThreads) {
        const int s = idx / P.n_d, k = idx - s * P.n_d;
        if (n0 + s < N) P.Do[(n0 + s) * P.n_d + k] = D[k * kT + s];
      }
    }

    // ---- hidden layers (nerf.py:144-148), then the colour branch's first layer (nerf.py:96-100, :151-152) ----
    for (int l = 0; l <= L; ++l) {
      if (l == L && tid < kT) {
        // density head (nerf.py:149) on the trunk's features, before the colour layer overwrites H;
        // the backward's g_zd = g_density * act'(z_d)
        const float* wd = P.w + P.w_density_off;
        const int64_t n = n0 + tid;
        float zd = LDG(wd + kW);
        for (int c = 0; c < kW; ++c) zd = fmaf(LDG(wd + c), H[c * kT + tid], zd);
        if constexpr (kTrain) {
          float y, d1;
          act_fd(P.density_act, zd, y, d1);
          const float gzd = up[tid * 4 + 3] * d1;
          up[tid * 4 + 3] = gzd;
          if (n < N) P.GZD[n] = gzd;
        } else {
          if (n < N) P.density[n] = density_act(P.density_act, zd);
        }
        // (no barrier: the layer below starts by reading H, writes it and reads `up` only after its own barriers)
      }
      const Layer& Ly = P.layer[l];
      gemm(cx, P.w, Ly, smem, acc);
      const int act = (l < L) ? P.act : NEDDF_ACT_RELU;  // outL_color's nn.ReLU (nerf.py:99)
      const float* bl = P.w + Ly.b_off;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ch0 = 4 * cg + 64 * i;
        float z[4][4], h[4][4];  // [j][s]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float b = LDG(bl + ch0 + j);
#pragma unroll
          for (int s = 0; s < 4; ++s) {
            float d1;
            z[j][s] = acc[i][j][s] + b;
            act_fd(act, z[j][s], h[j][s], d1);
          }
        }
        if constexpr (kTrain) {
          if (l < L) {  // park z_l and h_l
            float* Xl = P.X + (size_t)l * N * kW;
            float* Gl = P.G + (size_t)l * N * kW;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
              const int64_t n = n0 + 4 * sg + s;
              if (n < N) {
                *reinterpret_cast<float4*>(Gl + n * kW + ch0) = make_float4(z[0][s], z[1][s], z[2][s], z[3][s]);
                *reinterpret_cast<float4*>(Xl + n * kW + ch0) = make_float4(h[0][s], h[1][s], h[2][s], h[3][s]);
              }
            }
          } else {  // z becomes g_zc1 = (Wc2^T g_color) relu'(z_c1), which H carries into the backward
            const float* wc2 = P.w + P.w_col2_off;  // [3][128]
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int ch = ch0 + j;
              const bool live = ch < kW / 2;  // the colour branch is 128 wide; the padded half stays zero
              const float w0 = live ? LDG(wc2 + ch) : 0.f;
              const float w1 = live ? LDG(wc2 + kW / 2 + ch) : 0.f;
              const float w2 = live ? LDG(wc2 + kW + ch) : 0.f;
#pragma unroll
              for (int s = 0; s < 4; ++s) {
                const float* g = up + (4 * sg + s) * 4;
                z[j][s] = (z[j][s] > 0.f) ? fmaf(w2, g[2], fmaf(w1, g[1], w0 * g[0])) : 0.f;
              }
            }
#pragma unroll
            for (int s = 0; s < 4; ++s) {
              const int64_t n = n0 + 4 * sg + s;
              if (n < N) {
                *reinterpret_cast<float4*>(P.C1 + n * kW + ch0) = make_float4(h[0][s], h[1][s], h[2][s], h[3][s]);
                *reinterpret_cast<float4*>(P.GC1 + n * kW + ch0) = make_float4(z[0][s], z[1][s], z[2][s], z[3][s]);
              }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
              for (int s = 0; s < 4; ++s) h[j][s] = z[j][s];
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(H + (ch0 + j) * kT + 4 * sg) = make_float4(h[j][0], h[j][1], h[j][2], h[j][3]);
      }
      cx.sync();
    }

    if constexpr (!kTrain) {
      // ---- colour output (nerf.py:101-102): 3 x (width / 2) ----
      if (tid < kT) {
        const float* wc2 = P.w + P.w_col2_off;
        const int64_t n = n0 + tid;
        float o[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          float a = wc2[3 * (kW / 2) + c];
          for (int k = 0; k < kW / 2; ++k) a = fmaf(LDG(wc2 + c * (kW / 2) + k), H[k * kT + tid], a);
          o[c] = a;
        }
        if (n < N) {
          P.color[3 * n + 0] = o[0];
          P.color[3 * n + 1] = o[1];
          P.color[3 * n + 2] = o[2];
        }
      }
      cx.sync();  // H, E, D, geo are rewritten by the next tile
    } else {
      // ---- backward through the trunk ----
      // H holds the gradient of the pre-activation of the layer ABOVE (k = its output channel); step l turns it into
      // g_z_l = (W_above[:, :256]^T g_z_above [+ w_density g_zd for the last hidden layer]) act'(z_l).
      for (int l = L - 1; l >= 0; --l) {
        const Layer& Up = P.layer[l + 1];  // l + 1 == L: the colour branch's first layer (128 outputs)
        layer_gemm(cx, P.w + Up.wt_off, Up.kt_pad, H, Up.kt_pad, H, 0, smem + kOffW, acc);
        float* Gl = P.G + (size_t)l * N * kW;
        const float* wd = P.w + P.w_density_off;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ch0 = 4 * cg + 64 * i;
          float gz[4][4];  // [j][s]
          float wdj[4] = {0.f, 0.f, 0.f, 0.f};
          if (l == L - 1) {
#pragma unroll
            for (int j = 0; j < 4; ++j) wdj[j] = LDG(wd + ch0 + j);
          }
#pragma unroll
          for (int s = 0; s < 4; ++s) {
            const int64_t n = n0 + 4 * sg + s;
            float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < N) z4 = *reinterpret_cast<const float4*>(Gl + n * kW + ch0);  // z_l parked by the forward
            const float zz[4] = {z4.x, z4.y, z4.z, z4.w};
            const float gzd = up[(4 * sg + s) * 4 + 3];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float y, d1;
              act_fd(P.act, zz[j], y, d1);
              gz[j][s] = fmaf(wdj[j], gzd, acc[i][j][s]) * d1;
            }
            if (n < N) *reinterpret_cast<float4*>(Gl + n * kW + ch0) = make_float4(gz[0][s], gz[1][s], gz[2][s], gz[3][s]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(H + (ch0 + j) * kT + 4 * sg) = make_float4(gz[j][0], gz[j][1], gz[j][2], gz[j][3]);
        }
        cx.sync();
      }
      // (the trailing barrier of the last step also protects E, D, H, geo, up against the next tile)
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host: layer table (nerf.py:86-103)
// ---------------------------------------------------------------------------------------------

// layers.0 .. layers.{L-1}, outL_density, outL_color.0, outL_color.2; returns the count
inline int layer_shapes(const neddf_nerf_config_t* c, int* sin, int* sout) {
  const int in_pos = 6 * c->embed_pos_rank, in_dir = 6 * c->embed_dir_rank, W = c->layer_width;
  int n = 0;
  sin[n] = in_pos; sout[n++] = W;
  for (int lid = 0; lid < c->layer_count - 1; ++lid) {
    sin[n] = W + (is_skip(c, lid) ? in_pos : 0);
    sout[n++] = W;
  }
  sin[n] = W; sout[n++] = 1;
  sin[n] = W + in_dir; sout[n++] = W / 2;
  sin[n] = W / 2; sout[n++] = 3;
  return n;
}

// NULL = supported, else the reason and in *code (if given) NEDDF_E_INVALID (malformed) or NEDDF_E_UNSUPPORTED (not covered)
inline const char* unsupported(const neddf_nerf_config_t* c, int32_t* code = nullptr) {
  int32_t unused;
  if (!code) code = &unused;
  *code = NEDDF_E_INVALID;
  if (c->n_skips < 0 || c->n_skips > 8) return "bad skips";
  for (int a : {c->activation_type, c->density_activation_type})
    if (a != NEDDF_ACT_TANHEXP && a != NEDDF_ACT_RELU && a != NEDDF_ACT_LEAKYRELU) return "bad activation";
  *code = NEDDF_E_UNSUPPORTED;
  if (c->layer_width != kW) return "layer_width must be 256";
  if (c->layer_count < 2 || c->layer_count > kMaxLayers) return "layer_count must be 2..12";
  if (c->embed_pos_rank < 1 || 6 * c->embed_pos_rank > kMaxE || c->embed_dir_rank < 1 || 6 * c->embed_dir_rank > kMaxD)
    return "embedding ranks must satisfy 6 pos <= 64, 6 dir <= 32";
  if (is_skip(c, c->layer_count - 1)) return "a skip after the last hidden layer widens the heads (not covered)";
  return nullptr;
}

// fills the network part of P; `backward` adds the transposed packs the training kernel reads.  Returns the floats of
// weight buffer.
inline size_t build_program(const neddf_nerf_config_t* c, Params& P, bool backward = true) {
  const int L = c->layer_count;
  P.n_layers = L;
  P.embed_pos = c->embed_pos_rank;
  P.embed_dir = c->embed_dir_rank;
  P.n_e = 6 * c->embed_pos_rank;
  P.n_d = 6 * c->embed_dir_rank;
  P.act = c->activation_type;
  P.density_act = c->density_activation_type;
  size_t off = 0;
  for (int l = 0; l <= L; ++l) {
    Layer& Ly = P.layer[l];
    if (l == 0) { Ly.seg_a = kSegE; Ly.n_a = P.n_e; Ly.seg_b = kSegNone; Ly.n_b = 0; }
    else if (l < L) { Ly.seg_a = kSegH; Ly.n_a = kW; Ly.seg_b = is_skip(c, l - 1) ? kSegE : kSegNone; Ly.n_b = Ly.seg_b ? P.n_e : 0; }
    else { Ly.seg_a = kSegH; Ly.n_a = kW; Ly.seg_b = kSegD; Ly.n_b = P.n_d; }
    Ly.k_pad = (Ly.n_a + Ly.n_b + kChunk - 1) / kChunk * kChunk;
    Ly.w_off = (int)off; off += (size_t)Ly.k_pad * kW;
    Ly.b_off = (int)off; off += kW;
    // layer 0 has nothing below it to propagate to
    Ly.kt_pad = (!backward || l == 0) ? 0 : ((l < L) ? kW : kW / 2);
    Ly.wt_off = (int)off; off += (size_t)Ly.kt_pad * kW;
  }
  P.w_density_off = (int)off; off += kW + 4;
  P.w_col2_off = (int)off; off += 3 * (kW / 2) + 4;
  return off;
}

}  // namespace nerft
}  // namespace neddf
