// NeuS field variant (SURVEY 8(f) item 3): the tile program of csrc/neus_simt.cu.
//
// Reference: NeuS.forward (neddf/network/neus.py:101-162): plain position / direction embeddings (:119-120,
// nn_module/positional_encoding.py:37-65), `sdf_layer_count` layers with the activation after EVERY layer and the
// skip concat [h | E] after the layers named in `skips` (:122-126), sdf = channel 0 of the trunk's output (:127),
// normal = d sdf / d position (:133-142, torch.autograd.grad in the reference), colour trunk on
// [position | direction embedding | normal | trunk features] with the activation after every layer including the
// 3-channel output (:144-149), density = 10 v e / (1 + e)^2 with e = exp(-10 v sdf) (:150-153).
//
// The normal is carried FORWARD instead of taken in reverse: every sample has four columns in the SDF trunk
// (value, d/dx, d/dy, d/dz; the layout of the NeDDF kernels), G = f'(x) (J W) - the same number as the reference's
// reverse-mode gradient up to rounding (oracle.neus_forward_jac against oracle.neus_forward, tests/test_neus_oracle.py).
//
// Work decomposition (the fp32 CUDA-core skeleton of simt_mlp.cuh)
//   CTA (256 threads) = tile of 64 samples, persistent over tiles.  Activations K-major in shared memory
//   (row = channel, 64 columns).  SDF trunk: four passes over sub-tiles of 16 samples, column = 4 sample + row type;
//   the last SDF layer parks its value rows in F (column = sample) and the normal in the colour input head X.
//   Colour trunk: one pass over the 64 samples (value rows only), input rows "X then F", hidden rows in H.
//   Thread (cg = tid % 16, sg = tid / 16) owns columns 4 sg .. 4 sg + 3 (SDF trunk: the four row types of sample
//   sg; colour trunk: four samples) and the 16 output channels {4 cg + 64 i + j}.
//
// Compiled twice like simt_mlp.cuh: by nvcc into the kernel and by g++ into tests/emul/libneus_emul.so, where it is
// checked against the goldens.
#pragma once

#include "simt_mlp.cuh"

namespace neddf {
namespace neus {

using namespace simt;

constexpr int kSub = 16;     // samples per SDF sub-tile (4 columns each)
constexpr int kMaxE = 64;    // rows reserved for the position embedding (6 * rank <= 64)
constexpr int kMaxX = 32;    // colour input head [pos 3 | dir embedding 6 * rank | normal 3] (<= 32 rows)
constexpr int kMaxSdf = 12;  // SDF layers
constexpr int kMaxCol = 12;  // colour layers of width 256 (the 3-channel output layer is a per-sample head)

enum Seg { kSegNone = 0, kSegE = 1, kSegH = 2, kSegX = 3, kSegF = 4 };

struct Params : Samples {  // the samples (var unused: the NeuS embeddings are plain), then:
  // network
  int n_sdf, n_col;
  Layer lsdf[kMaxSdf];
  Layer lcol[kMaxCol];
  int head_off;  // colour output layer: [3][256] + 3 biases
  int var_off;   // the variance parameter (one float)
  int embed_pos, embed_dir;
  int act;       // NEDDF_ACT_RELU | NEDDF_ACT_TANHEXP
  const float* w;
  // outputs ([n], [n], [n,3], optional [n,3])
  float* sdf;
  float* density;
  float* color;
  float* normal;
};

// shared-memory map (floats)
constexpr int kOffE = 0;
constexpr int kOffX = kOffE + kMaxE * kT;
constexpr int kOffH = kOffX + kMaxX * kT;
constexpr int kOffF = kOffH + kW * kT;
constexpr int kOffW = kOffF + kW * kT;
constexpr int kOffGeo = kOffW + 2 * kChunk * kW;  // [kT][6] position, direction
constexpr int kOffSdf = kOffGeo + kT * 6;         // [kT] sdf of the tile's samples
constexpr int kSmemFloats = kOffSdf + kT;
constexpr size_t kSmemBytes = (size_t)kSmemFloats * sizeof(float);

// neus.py:150-153, one rounding per torch op
__device__ __forceinline__ float sdf_density(float sdf, float variance) {
  const float v10 = __fmul_rn(variance, 10.0f);
  const float ex = expf(__fmul_rn(-v10, sdf));
  const float onep = __fadd_rn(1.0f, ex);
  return __fmul_rn(__fmul_rn(v10, ex), __frcp_rn(__fmul_rn(onep, onep)));
}

__device__ __forceinline__ float* seg_ptr(float* smem, int seg) {
  return smem + (seg == kSegE ? kOffE : (seg == kSegX ? kOffX : (seg == kSegF ? kOffF : kOffH)));
}

template <class Ctx>
__device__ __forceinline__ void gemm(Ctx& cx, const Params& P, const Layer& L, float* smem, float (&acc)[4][4][4]) {
  layer_gemm(cx, P.w + L.w_off, L.k_pad, seg_ptr(smem, L.seg_a), L.n_a, seg_ptr(smem, L.seg_b), L.n_b, smem + kOffW, acc);
}

// One CTA: tiles cx.block, cx.block + cx.nblocks, ...
template <class Ctx>
__device__ __forceinline__ void tile_program(Ctx& cx, const Params& P, float* smem) {
  float* E = smem + kOffE;
  float* X = smem + kOffX;
  float* H = smem + kOffH;
  float* F = smem + kOffF;
  float* geo = smem + kOffGeo;
  float* sdfv = smem + kOffSdf;
  const int tid = cx.tid;
  const int cg = tid & 15, sg = tid >> 4;
  const int64_t n_tiles = (P.n + kT - 1) / kT;
  const int ehalf = 3 * P.embed_pos;  // rows of the sine block of the position embedding
  const int dhalf = 3 * P.embed_dir;
  const int x_normal = 3 + 2 * dhalf;  // first normal row of X
  float acc[4][4][4];

  for (int64_t tile = cx.block; tile < n_tiles; tile += cx.nblocks) {
    const int64_t n0 = tile * kT;
    // ---- geometry of the tile's samples (one thread per sample); rows 0..2 of X = position (neus.py:145) ----
    if (tid < kT) {
      float pos[3], dir[3], var[3];
      load_sample(P, n0 + tid, pos, dir, var);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        geo[tid * 6 + i] = pos[i];
        geo[tid * 6 + 3 + i] = dir[i];
        X[i * kT + tid] = pos[i];
      }
    }
    cx.sync();
    // ---- direction embedding into X (neus.py:120): four threads per sample ----
    {
      const int s = tid >> 2, sub4 = tid & 3;
      for (int idx = sub4; idx < dhalf; idx += 4) {
        const int e = idx / 3, d = idx - 3 * e;
        float sn, cs;
        sincosf((float)(1u << e) * geo[s * 6 + 3 + d], &sn, &cs);
        X[(3 + idx) * kT + s] = sn;
        X[(3 + dhalf + idx) * kT + s] = cs;
      }
    }
    // (no barrier: X is first read by the colour trunk, behind the barriers of the SDF trunk)

    // ---- SDF trunk on four sub-tiles of 16 samples (value + three Jacobian columns per sample) ----
    for (int sub = 0; sub < kT / kSub; ++sub) {
      // position embedding with its Jacobian (neus.py:119): sixteen threads per sample
      {
        const int s = tid >> 4, lane16 = tid & 15;
        const float* p3 = geo + (kSub * sub + s) * 6;
        for (int idx = lane16; idx < ehalf; idx += 16) {
          const int e = idx / 3, d = idx - 3 * e;
          const float f = (float)(1u << e);
          float sn, cs;
          sincosf(f * p3[d], &sn, &cs);
          float4 vs = make_float4(sn, 0.f, 0.f, 0.f), vc = make_float4(cs, 0.f, 0.f, 0.f);
          const float js = f * cs, jc = -(f * sn);
          if (d == 0) { vs.y = js; vc.y = jc; }
          else if (d == 1) { vs.z = js; vc.z = jc; }
          else { vs.w = js; vc.w = jc; }
          *reinterpret_cast<float4*>(E + idx * kT + 4 * s) = vs;
          *reinterpret_cast<float4*>(E + (ehalf + idx) * kT + 4 * s) = vc;
        }
      }
      cx.sync();
      for (int l = 0; l < P.n_sdf; ++l) {
        const Layer& L = P.lsdf[l];
        gemm(cx, P, L, smem, acc);
        const float* bl = P.w + L.b_off;
        const bool last = (l == P.n_sdf - 1);
        const int col = kSub * sub + sg;  // the sample's column in the colour trunk
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int ch = 4 * cg + 64 * i + j;
            float y, d1;
            act_fd(P.act, acc[i][j][0] + LDG(bl + ch), y, d1);
            const float4 o = make_float4(y, d1 * acc[i][j][1], d1 * acc[i][j][2], d1 * acc[i][j][3]);
            if (!last) {
              *reinterpret_cast<float4*>(H + ch * kT + 4 * sg) = o;
            } else {
              F[ch * kT + col] = y;  // trunk features of the colour input (neus.py:128,145)
              if (ch == 0) {         // sdf = channel 0 (neus.py:127), normal = its Jacobian column (neus.py:133-142)
                sdfv[col] = y;
                X[(x_normal + 0) * kT + col] = o.y;
                X[(x_normal + 1) * kT + col] = o.z;
                X[(x_normal + 2) * kT + col] = o.w;
              }
            }
          }
        cx.sync();
      }
    }

    // ---- sdf, density, normal of the tile (neus.py:150-159) ----
    if (tid < kT) {
      const int64_t n = n0 + tid;
      if (n < P.n) {
        const float s = sdfv[tid];
        P.sdf[n] = s;
        P.density[n] = sdf_density(s, LDG(P.w + P.var_off));
        if (P.normal) {
#pragma unroll
          for (int i = 0; i < 3; ++i) P.normal[3 * n + i] = X[(x_normal + i) * kT + tid];
        }
      }
    }

    // ---- colour trunk on the 64 samples (neus.py:144-149) ----
    for (int l = 0; l < P.n_col; ++l) {
      const Layer& L = P.lcol[l];
      gemm(cx, P, L, smem, acc);
      const float* bl = P.w + L.b_off;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = 4 * cg + 64 * i + j;
          const float b = LDG(bl + ch);
          float4 o;
          float d1;
          act_fd(P.act, acc[i][j][0] + b, o.x, d1);
          act_fd(P.act, acc[i][j][1] + b, o.y, d1);
          act_fd(P.act, acc[i][j][2] + b, o.z, d1);
          act_fd(P.act, acc[i][j][3] + b, o.w, d1);
          *reinterpret_cast<float4*>(H + ch * kT + 4 * sg) = o;
        }
      cx.sync();
    }
    // ---- colour output layer + activation (neus.py:148-149: the activation follows the last layer too) ----
    if (tid < kT) {
      const float* wh = P.w + P.head_off;
      const int64_t n = n0 + tid;
      float o[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float a = LDG(wh + 3 * kW + c);
        for (int k = 0; k < kW; ++k) a = fmaf(LDG(wh + c * kW + k), H[k * kT + tid], a);
        float d1;
        act_fd(P.act, a, o[c], d1);
      }
      if (n < P.n) {
        P.color[3 * n + 0] = o[0];
        P.color[3 * n + 1] = o[1];
        P.color[3 * n + 2] = o[2];
      }
    }
    cx.sync();  // X, H, F, geo, sdfv are rewritten by the next tile
  }
}

// entry (k, c) of a layer's packed [in padded][256] block
__device__ __forceinline__ float pack_entry(const float* w, int n_in, int n_out, int k, int c) { return pack_fwd(w, n_in, n_out, k, c); }

// ---------------------------------------------------------------------------------------------
// host: layer table from the constructor arguments (neus.py:83-98)
// ---------------------------------------------------------------------------------------------
// layers_sdf.0 .. layers_sdf.{Ls-1}, layers_col.0 .. layers_col.{Lc}; returns the count
inline int layer_shapes(const neddf_neus_config_t* c, int* sin, int* sout) {
  const int in_sdf = 6 * c->embed_pos_rank, W = c->sdf_layer_width;
  int n = 0;
  sin[n] = in_sdf; sout[n++] = W;
  for (int lid = 0; lid < c->sdf_layer_count - 1; ++lid) {
    sin[n] = W + (is_skip(c, lid) ? in_sdf : 0);
    sout[n++] = W;
  }
  sin[n] = 6 + 6 * c->embed_dir_rank + W; sout[n++] = c->col_layer_width;
  for (int i = 0; i < c->col_layer_count - 1; ++i) { sin[n] = c->col_layer_width; sout[n++] = c->col_layer_width; }
  sin[n] = c->col_layer_width; sout[n++] = 3;
  return n;
}

// NULL = supported, else the reason
inline const char* unsupported(const neddf_neus_config_t* c) {
  if (c->sdf_layer_width != kW || c->col_layer_width != kW) return "sdf_layer_width and col_layer_width must be 256";
  if (c->sdf_layer_count < 1 || c->sdf_layer_count > kMaxSdf) return "sdf_layer_count must be 1..12";
  if (c->col_layer_count < 1 || c->col_layer_count > kMaxCol) return "col_layer_count must be 1..12";
  if (c->embed_pos_rank < 1 || 6 * c->embed_pos_rank > kMaxE) return "6 * embed_pos_rank must be <= 64";
  if (c->embed_dir_rank < 1 || 6 + 6 * c->embed_dir_rank > kMaxX) return "6 + 6 * embed_dir_rank must be <= 32";
  if (c->n_skips < 0 || c->n_skips > 8) return "at most 8 skips";
  if (c->activation_type != NEDDF_ACT_RELU && c->activation_type != NEDDF_ACT_TANHEXP) return "activation_type must be ReLU or tanhExp (neus.py:70-73)";
  if (is_skip(c, c->sdf_layer_count - 1)) return "a skip after the last SDF layer widens the colour input (the reference's layer shapes do not allow it either)";
  return nullptr;
}

// fills the network part of P; returns the floats of the packed weight buffer
inline size_t build_program(const neddf_neus_config_t* c, Params& P) {
  P.n_sdf = c->sdf_layer_count;
  P.n_col = c->col_layer_count;
  P.embed_pos = c->embed_pos_rank;
  P.embed_dir = c->embed_dir_rank;
  P.act = c->activation_type;
  const int n_e = 6 * c->embed_pos_rank, n_x = 6 + 6 * c->embed_dir_rank;
  size_t off = 0;
  auto place = [&](Layer& L) {
    L.k_pad = (L.n_a + L.n_b + kChunk - 1) / kChunk * kChunk;
    L.w_off = (int)off; off += (size_t)L.k_pad * kW;
    L.b_off = (int)off; off += kW;
  };
  for (int l = 0; l < P.n_sdf; ++l) {
    Layer& L = P.lsdf[l];
    if (l == 0) { L.seg_a = kSegE; L.n_a = n_e; L.seg_b = kSegNone; L.n_b = 0; }
    else { L.seg_a = kSegH; L.n_a = kW; L.seg_b = is_skip(c, l - 1) ? kSegE : kSegNone; L.n_b = L.seg_b ? n_e : 0; }
    place(L);
  }
  for (int l = 0; l < P.n_col; ++l) {
    Layer& L = P.lcol[l];
    if (l == 0) { L.seg_a = kSegX; L.n_a = n_x; L.seg_b = kSegF; L.n_b = kW; }
    else { L.seg_a = kSegH; L.n_a = kW; L.seg_b = kSegNone; L.n_b = 0; }
    place(L);
  }
  P.head_off = (int)off; off += 3 * kW + 4;
  P.var_off = (int)off; off += 4;
  return off;
}

}  // namespace neus
}  // namespace neddf
